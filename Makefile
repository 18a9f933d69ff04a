# Builds the C-ABI shared library of the engine (include/sipoc.h) for sm_100a,
# in-tree, plus the CPU oracle used by the tests.  No CMake / Bazel needed.
NVCC ?= /usr/local/cuda/bin/nvcc
HOSTCXX ?= /usr/bin/g++
ARCH := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -std=c++17 -O3 -lineinfo $(ARCH) -ccbin $(HOSTCXX) -Xcompiler -fPIC \
             -Xcompiler -Wall -cudart static --expt-relaxed-constexpr
CSRC := sip_optimal_control_b200/csrc
LIBDIR := sip_optimal_control_b200/lib
OBJDIR := build/obj
SRCS := $(CSRC)/api.cu $(CSRC)/generic_kernels.cu $(CSRC)/riccati_fast.cu $(CSRC)/riccati_cta.cu $(CSRC)/riccati_strict.cu $(CSRC)/kkt_fast.cu $(CSRC)/kkt_theta.cu $(CSRC)/comm.cu $(CSRC)/scan.cu $(CSRC)/model_scatter.cu $(CSRC)/riccati_f32.cu \
        $(CSRC)/lqr_vjp.cu $(CSRC)/kkt_vjp.cu $(CSRC)/jvp.cu $(CSRC)/workload.cu $(CSRC)/structure.cpp
OBJS := $(patsubst $(CSRC)/%,$(OBJDIR)/%.o,$(SRCS)) $(OBJDIR)/riccati_fast_part1.cu.o \
        $(OBJDIR)/riccati_fast_part2.cu.o $(OBJDIR)/riccati_fast_part3.cu.o
HDRS := $(wildcard $(CSRC)/*.cuh $(CSRC)/*.hpp) include/sipoc.h

HOSTDIR := sip_optimal_control_b200/host
HOSTSRC := $(HOSTDIR)/lqr.cpp $(HOSTDIR)/types.cpp $(HOSTDIR)/helpers.cpp $(HOSTDIR)/sip_optimal_control.cpp
HOSTHDR := $(HOSTDIR)/lqr.hpp $(HOSTDIR)/types.hpp $(HOSTDIR)/helpers.hpp $(HOSTDIR)/sip_optimal_control.hpp $(HOSTDIR)/device_state.hpp include/sipoc.h
HOSTFLAGS := -std=c++17 -O2 -Wall -Wextra -fPIC

all: $(LIBDIR)/libsipoc.so $(LIBDIR)/libsipoc_host.so build/host_tests oracle

# C++ host side (the reference's Topology / Dimensions / LQR / CallbackProvider classes
# over the C ABI) and the restated reference tests that run against it.
$(LIBDIR)/libsipoc_host.so: $(HOSTSRC) $(HOSTHDR) $(LIBDIR)/libsipoc.so
	$(HOSTCXX) $(HOSTFLAGS) -shared -o $@ $(HOSTSRC) -L$(LIBDIR) -lsipoc -Wl,-rpath,'$$ORIGIN'

build/host_tests: $(HOSTDIR)/host_tests.cpp $(LIBDIR)/libsipoc_host.so
	@mkdir -p build
	$(HOSTCXX) $(HOSTFLAGS) -o $@ $< -L$(LIBDIR) -lsipoc_host -lsipoc \
	    -Wl,-rpath,'$$ORIGIN/../$(LIBDIR)'

$(OBJDIR)/%.cu.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVCCFLAGS) $(EXTRA) -c $< -o $@

# riccati_fast.cu instantiates its shapes in four parts (-DSIPOC_FAST_PART) so they build in
# parallel; part 0 is the plain object above.
$(OBJDIR)/riccati_fast_part%.cu.o: $(CSRC)/riccati_fast.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVCCFLAGS) $(EXTRA) -DSIPOC_FAST_PART=$* -c $< -o $@

$(OBJDIR)/%.cpp.o: $(CSRC)/%.cpp $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVCCFLAGS) -x cu -c $< -o $@

$(LIBDIR)/libsipoc.so: $(OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -ccbin $(HOSTCXX) -shared -cudart static -o $@ $(OBJS) -ldl

oracle:
	$(MAKE) -C oracle liboracle.so

# FP64 issue / latency microbenchmark (DFMA, DMMA.8x8x4, rsqrt) behind profiles/r01/microbench_fp64.txt
microbench: build/microbench_fp64
build/microbench_fp64: tools/microbench_fp64.cu
	@mkdir -p build
	$(NVCC) -O3 $(ARCH) -ccbin $(HOSTCXX) -o $@ $<

clean:
	rm -rf build $(LIBDIR)/libsipoc.so $(LIBDIR)/libsipoc_host.so oracle/liboracle.so

.PHONY: all oracle clean microbench
