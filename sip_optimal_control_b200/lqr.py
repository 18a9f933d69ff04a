"""Host-side mirror of the reference's ``lqr.hpp`` for the batched engine.

``Topology``, ``Dimensions`` and ``LQR`` keep the reference's names, argument
meaning and error behaviour (lqr.hpp:5-64, 66-200); the one change is that an
``LQR`` object owns a *batch* of numerically independent problems of one
structure, so ``factor_with_status`` returns one ``FactorStatus`` per problem.

Device arrays are ``torch`` CUDA tensors of dtype float64 and shape
``[size, batch_stride]`` (the engine layout of include/sipoc.h: flat
per-problem index major, batch innermost).  PyTorch is used for device memory
and streams only; every computation goes through the C ABI in libsipoc.so.
"""
from __future__ import annotations

import ctypes
import enum
from typing import Dict, Optional

import numpy as np

from . import _capi
from ._capi import lib


class FactorStatus(enum.IntEnum):
    """LQR::FactorStatus (lqr.hpp:68-74)."""

    SUCCESS = 0
    INVALID_DELTA = 1
    F_FACTORIZATION_FAILURE = 2
    G_FACTORIZATION_FAILURE = 3
    INVALID_TOPOLOGY = 4


class SipocError(RuntimeError):
    def __init__(self, code: int, message: str = ""):
        self.code = code
        super().__init__(f"{_capi.ERROR_NAMES.get(code, code)}: {message}")


def _i32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32))


class Topology:
    """Rooted tree with one edge per non-root node (lqr.hpp:5-22)."""

    def __init__(self, num_edges: int = 0, root: int = 0, edge_parents=None, edge_children=None):
        self.num_edges = int(num_edges)
        self.root = int(root)
        self.edge_parents = None if edge_parents is None else _i32(edge_parents)
        self.edge_children = None if edge_children is None else _i32(edge_children)

    def num_nodes(self) -> int:
        return self.num_edges + 1

    def set_chain(self) -> None:  # lqr.cpp:32-40
        self.root = 0
        self.edge_parents = np.arange(self.num_edges, dtype=np.int32)
        self.edge_children = self.edge_parents + 1

    def set_tree(self, root: int, edge_parents, edge_children) -> None:  # lqr.cpp:42-47
        self.root = int(root)
        self.edge_parents = _i32(edge_parents)[: self.num_edges]
        self.edge_children = _i32(edge_children)[: self.num_edges]

    @staticmethod
    def chain(num_edges: int) -> "Topology":
        t = Topology(num_edges)
        t.set_chain()
        return t


class Dimensions:
    """Per-node / per-edge dimensions (lqr.hpp:24-64).  ``None`` = all zero."""

    def __init__(self, theta_dim: int = 0, state_dims=None, control_dims=None,
                 node_c_dims=None, node_g_dims=None, edge_c_dims=None, edge_g_dims=None):
        self.theta_dim = int(theta_dim)
        self.state_dims = None if state_dims is None else _i32(state_dims)
        self.control_dims = None if control_dims is None else _i32(control_dims)
        self.node_c_dims = None if node_c_dims is None else _i32(node_c_dims)
        self.node_g_dims = None if node_g_dims is None else _i32(node_g_dims)
        self.edge_c_dims = None if edge_c_dims is None else _i32(edge_c_dims)
        self.edge_g_dims = None if edge_g_dims is None else _i32(edge_g_dims)

    def set_uniform(self, num_edges, state_dim, control_dim, node_c_dim=0, node_g_dim=0,
                    edge_c_dim=0, edge_g_dim=0, theta_dim=0) -> None:  # lqr.cpp:77-88
        self.theta_dim = int(theta_dim)
        self.state_dims = np.full(num_edges + 1, state_dim, np.int32)
        self.control_dims = np.full(num_edges, control_dim, np.int32)
        self.node_c_dims = np.full(num_edges + 1, node_c_dim, np.int32)
        self.node_g_dims = np.full(num_edges + 1, node_g_dim, np.int32)
        self.edge_c_dims = np.full(num_edges, edge_c_dim, np.int32)
        self.edge_g_dims = np.full(num_edges, edge_g_dim, np.int32)

    @staticmethod
    def uniform(num_edges, state_dim, control_dim, **kw) -> "Dimensions":
        d = Dimensions()
        d.set_uniform(num_edges, state_dim, control_dim, **kw)
        return d

    def get_schur_dim(self) -> int:
        return self.theta_dim

    def get_state_dim(self, node) -> int:
        return int(self.state_dims[node])

    def get_control_dim(self, edge) -> int:
        return int(self.control_dims[edge])

    def _opt(self, arr, i) -> int:  # lqr.cpp:98-112
        return 0 if arr is None else int(arr[i])

    def get_node_c_dim(self, node) -> int:
        return self._opt(self.node_c_dims, node)

    def get_node_g_dim(self, node) -> int:
        return self._opt(self.node_g_dims, node)

    def get_edge_c_dim(self, edge) -> int:
        return self._opt(self.edge_c_dims, edge)

    def get_edge_g_dim(self, edge) -> int:
        return self._opt(self.edge_g_dims, edge)

    def get_stagewise_x_dim(self, num_edges) -> int:  # lqr.cpp:146-151
        return int(self.state_dims[num_edges] +
                   sum(int(self.state_dims[e]) + int(self.control_dims[e])
                       for e in range(num_edges)))

    def get_x_dim(self, num_edges) -> int:
        return self.get_stagewise_x_dim(num_edges) + self.theta_dim

    def get_y_dim(self, num_edges) -> int:  # lqr.cpp:157-165
        return int(sum(int(self.state_dims[i]) + self.get_node_c_dim(i)
                       for i in range(num_edges + 1)) +
                   sum(self.get_edge_c_dim(e) for e in range(num_edges)))

    def get_z_dim(self, num_edges) -> int:  # lqr.cpp:167-175
        return int(sum(self.get_node_g_dim(i) for i in range(num_edges + 1)) +
                   sum(self.get_edge_g_dim(e) for e in range(num_edges)))

    def get_stagewise_kkt_dim(self, num_edges) -> int:
        return (self.get_stagewise_x_dim(num_edges) + self.get_y_dim(num_edges) +
                self.get_z_dim(num_edges))


def _ip(a):
    return None if a is None else a.ctypes.data_as(_capi.c_int_p)


class Engine:
    """Owns one ``sipoc_engine`` handle (one structure, one batch, one device)."""

    def __init__(self, dimensions: Dimensions, topology: Topology, batch: int,
                 device: Optional[int] = None, force_generic: bool = False,
                 pad_variable_dims: bool = False, parallel_in_time: Optional[bool] = None):
        self.dimensions = dimensions
        self.topology = topology
        self.batch = int(batch)
        self._handle = ctypes.c_void_p()
        self._keep = (topology.edge_parents, topology.edge_children, dimensions.state_dims,
                      dimensions.control_dims, dimensions.node_c_dims, dimensions.node_g_dims,
                      dimensions.edge_c_dims, dimensions.edge_g_dims)
        s = _capi.Structure(
            topology.num_edges, topology.root, _ip(topology.edge_parents),
            _ip(topology.edge_children), _ip(dimensions.state_dims),
            _ip(dimensions.control_dims), _ip(dimensions.node_c_dims),
            _ip(dimensions.node_g_dims), _ip(dimensions.edge_c_dims),
            _ip(dimensions.edge_g_dims), dimensions.theta_dim, self.batch,
            -1 if device is None else int(device),
            (_capi.SIPOC_FLAG_FORCE_GENERIC if force_generic else 0)
            | (_capi.SIPOC_FLAG_PAD_VARIABLE_DIMS if pad_variable_dims else 0)
            # None: the engine decides (long horizon, small batch); True / False: forced
            | (_capi.SIPOC_FLAG_PARALLEL_IN_TIME if parallel_in_time is True else 0)
            | (_capi.SIPOC_FLAG_SERIAL_IN_TIME if parallel_in_time is False else 0))
        self.create_status = int(lib.sipoc_create(ctypes.byref(s), ctypes.byref(self._handle)))
        if self.create_status != _capi.SIPOC_OK:
            self._handle = ctypes.c_void_p()
            return
        self.batch_stride = int(lib.sipoc_batch_stride(self._handle))
        sz = _capi.LqrSizes()
        self._check(lib.sipoc_lqr_get_sizes(self._handle, ctypes.byref(sz)))
        self.lqr_sizes: Dict[str, int] = {k: int(getattr(sz, k)) for k, _ in sz._fields_}
        ks = _capi.KktSizes()
        self._check(lib.sipoc_kkt_get_sizes(self._handle, ctypes.byref(ks)))
        self.kkt_sizes: Dict[str, int] = {k: int(getattr(ks, k)) for k, _ in ks._fields_}
        self.device_index = device

    # -- plumbing -----------------------------------------------------------
    @property
    def ok(self) -> bool:
        return bool(self._handle)

    def _check(self, rc: int) -> None:
        if rc != _capi.SIPOC_OK:
            msg = lib.sipoc_last_error(self._handle) if self._handle else b""
            raise SipocError(int(rc), (msg or b"").decode())

    def close(self) -> None:
        if getattr(self, "_handle", None):
            lib.sipoc_destroy(self._handle)
            self._handle = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def kernel_variant(self) -> str:
        return lib.sipoc_kernel_variant(self._handle).decode()

    @property
    def launch_count(self) -> int:
        return int(lib.sipoc_launch_count(self._handle))

    def compiled_topology(self):
        E = self.topology.num_edges
        co = np.zeros(E + 2, np.int32)
        ce = np.zeros(max(E, 1), np.int32)
        pre = np.zeros(E + 1, np.int32)
        post = np.zeros(E + 1, np.int32)
        self._check(lib.sipoc_get_topology(self._handle, _ip(co), _ip(ce), _ip(pre), _ip(post)))
        return co, ce[:E], pre, post

    # -- torch helpers (device memory + streams only) -------------------------
    def _torch(self):
        import torch

        return torch

    def torch_device(self):
        torch = self._torch()
        idx = torch.cuda.current_device() if self.device_index is None else self.device_index
        return torch.device("cuda", idx)

    def empty(self, size: int, dtype=None):
        torch = self._torch()
        return torch.empty((max(int(size), 1), self.batch_stride),
                           dtype=dtype or torch.float64, device=self.torch_device())

    def zeros(self, size: int):
        t = self.empty(size)
        t.zero_()
        return t

    def empty_int(self):
        torch = self._torch()
        return torch.zeros((self.batch_stride,), dtype=torch.int32, device=self.torch_device())

    def stream_ptr(self, stream=None) -> int:
        torch = self._torch()
        s = stream if stream is not None else torch.cuda.current_stream(self.torch_device())
        return int(s.cuda_stream)

    def pack(self, host_array: np.ndarray, stream=None):
        """Problem-major host array [batch, size] -> engine-layout device tensor.  The copy,
        the transpose and the wait all happen on ``stream`` (default: torch's current)."""
        torch = self._torch()
        a = np.ascontiguousarray(host_array, dtype=np.float64)
        assert a.shape[0] == self.batch, (a.shape, self.batch)
        size = a.shape[1]
        st = stream if stream is not None else torch.cuda.current_stream(self.torch_device())
        with torch.cuda.stream(st):
            dst = self.zeros(size)
            if size == 0:
                return dst
            src = torch.from_numpy(a).to(self.torch_device())
            self._check(lib.sipoc_pack(self._handle, src.data_ptr(), dst.data_ptr(), size,
                                       int(st.cuda_stream)))
        st.synchronize()  # src may be recycled once this returns
        return dst

    def unpack(self, dev_tensor, size: int, stream=None) -> np.ndarray:
        """Engine-layout device tensor -> problem-major host array [batch, size]."""
        torch = self._torch()
        st = stream if stream is not None else torch.cuda.current_stream(self.torch_device())
        with torch.cuda.stream(st):
            out = torch.empty((self.batch, max(size, 1)), dtype=torch.float64,
                              device=self.torch_device())
            if size > 0:
                self._check(lib.sipoc_unpack(self._handle, dev_tensor.data_ptr(), out.data_ptr(),
                                             size, int(st.cuda_stream)))
            host = out.cpu()  # on `st`: ordered after the transpose
        st.synchronize()
        return host.numpy()[:, :size]


def _lqr_input_struct(inp: dict) -> _capi.LqrInput:
    s = _capi.LqrInput()
    for k in _capi.LQR_INPUT_FIELDS:
        t = inp.get(k)
        setattr(s, k, None if t is None else t.data_ptr())
    return s


def _lqr_output_struct(out: dict) -> _capi.LqrOutput:
    s = _capi.LqrOutput()
    for k in _capi.LQR_OUTPUT_FIELDS:
        setattr(s, k, out[k].data_ptr())
    return s


def _host_ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class LQR:
    """Batched regularized tree-LQR (reference ``LQR``, lqr.hpp:66-200).

    ``LQR(dimensions, topology, batch)`` compiles the topology like the
    reference constructor (lqr.cpp:635-643); an invalid tree is latched and
    reported by every later factor as ``INVALID_TOPOLOGY`` (lqr.cpp:646-648).
    """

    FactorStatus = FactorStatus

    def __init__(self, dimensions: Dimensions, topology: Topology, batch: int = 1,
                 device: Optional[int] = None, force_generic: bool = False,
                 pad_variable_dims: bool = False, parallel_in_time: Optional[bool] = None):
        self.engine = Engine(dimensions, topology, batch, device, force_generic,
                             pad_variable_dims, parallel_in_time)
        self.batch = int(batch)
        self.traversal_status_ = self.compile_topology()

    def compile_topology(self) -> FactorStatus:
        rc = self.engine.create_status
        if rc == _capi.SIPOC_OK:
            return FactorStatus.SUCCESS
        if rc in (_capi.SIPOC_INVALID_TOPOLOGY,):
            return FactorStatus.INVALID_TOPOLOGY
        raise SipocError(rc, "sipoc_create failed")

    # -- device path ------------------------------------------------------------
    def alloc_input(self) -> dict:
        return {k: self.engine.zeros(self.engine.lqr_sizes[k]) for k in _capi.LQR_INPUT_FIELDS}

    def alloc_output(self) -> dict:
        return {k: self.engine.zeros(self.engine.lqr_sizes[k]) for k in _capi.LQR_OUTPUT_FIELDS}

    def pack_input(self, host: dict) -> dict:
        """dict of problem-major numpy arrays -> dict of engine-layout tensors."""
        return {k: self.engine.pack(host[k]) for k in _capi.LQR_INPUT_FIELDS}

    def unpack_output(self, out: dict) -> dict:
        return {k: self.engine.unpack(out[k], self.engine.lqr_sizes[k])
                for k in _capi.LQR_OUTPUT_FIELDS}

    def _invalid(self):
        return np.full(self.batch, int(FactorStatus.INVALID_TOPOLOGY), np.int32)

    def factor_with_status(self, inp: dict, status=None, stream=None):
        """Returns a device int32 tensor [batch_stride] of FactorStatus values."""
        if self.traversal_status_ != FactorStatus.SUCCESS:
            return self._invalid()
        e = self.engine
        status = e.empty_int() if status is None else status
        s = _lqr_input_struct(inp)
        e._check(lib.sipoc_lqr_factor(e._handle, ctypes.byref(s), status.data_ptr(),
                                      e.stream_ptr(stream)))
        return status

    def factor(self, inp: dict, stream=None):
        """Per-problem ``factor_with_status() == SUCCESS`` (lqr.cpp:733)."""
        st = self.factor_with_status(inp, stream=stream)
        if isinstance(st, np.ndarray):
            return st == 0
        return (st[: self.batch] == 0)

    def solve(self, inp: dict, out: dict, stream=None) -> None:
        e = self.engine
        si, so = _lqr_input_struct(inp), _lqr_output_struct(out)
        e._check(lib.sipoc_lqr_solve(e._handle, ctypes.byref(si), ctypes.byref(so),
                                     e.stream_ptr(stream)))

    def factor_solve(self, inp: dict, out: dict, status=None, stream=None):
        if self.traversal_status_ != FactorStatus.SUCCESS:
            return self._invalid()
        e = self.engine
        status = e.empty_int() if status is None else status
        si, so = _lqr_input_struct(inp), _lqr_output_struct(out)
        e._check(lib.sipoc_lqr_factor_solve(e._handle, ctypes.byref(si), ctypes.byref(so),
                                            status.data_ptr(), e.stream_ptr(stream)))
        return status

    def vjp(self, inp: dict, out: dict, cot: dict, want=None, adjoint=None, status=None,
            stream=None) -> dict:
        """Reverse-mode derivative of ``factor_solve`` (sipoc_lqr_vjp; include/sipoc.h).

        ``inp`` and ``out`` are the forward's inputs and solution, ``cot`` holds dL/dx, dL/du,
        dL/dy (engine layout, keys x, u, y).  ``want`` is the set of input names to
        differentiate (default: all nine); the others are neither computed nor written.
        Returns a dict with one engine-layout gradient tensor per wanted name, ``adjoint``
        (dict x, u, y) and ``status`` (the adjoint factorization's FactorStatus per problem).
        Q and R get the symmetric gradient; failed problems and padding lanes get zeros."""
        e = self.engine
        want = set(_capi.LQR_INPUT_FIELDS if want is None else want)
        unknown = want - set(_capi.LQR_INPUT_FIELDS)
        if unknown:
            raise ValueError(f"not an LQR input: {sorted(unknown)}")
        adjoint = self.alloc_output() if adjoint is None else adjoint
        status = e.empty_int() if status is None else status
        grads = {k: e.empty(e.lqr_sizes[k]) for k in _capi.LQR_INPUT_FIELDS if k in want}
        si, ss, sa = _lqr_input_struct(inp), _lqr_output_struct(out), _lqr_output_struct(adjoint)
        sc = _capi.LqrCotangent()
        for k in _capi.LQR_OUTPUT_FIELDS:
            setattr(sc, k, cot[k].data_ptr())
        sg = _capi.LqrGrad()
        for k in _capi.LQR_INPUT_FIELDS:
            setattr(sg, k, grads[k].data_ptr() if k in grads else None)
        e._check(lib.sipoc_lqr_vjp(e._handle, ctypes.byref(si), ctypes.byref(ss),
                                   ctypes.byref(sc), ctypes.byref(sa), ctypes.byref(sg),
                                   status.data_ptr(), e.stream_ptr(stream)))
        grads["adjoint"] = adjoint
        grads["status"] = status
        return grads

    def jvp(self, inp: dict, out: dict, tan: dict, dsol=None, rhs=None, status=None,
            stream=None) -> dict:
        """Forward-mode derivative of ``factor_solve`` (sipoc_lqr_jvp; include/sipoc.h).

        ``inp`` and ``out`` are the forward's inputs and solution, ``tan`` holds the tangents
        of any subset of the nine input names (engine layout); an absent name is a zero
        tangent and is not read.  Returns a dict with the tangent of the solution ``x``,
        ``u``, ``y``, ``rhs`` (dict q, r, c: the right-hand side t = dK z + dh the tangent
        solve used) and ``status``.  Q and R enter through their symmetric parts; failed
        problems and padding lanes get zero x, u, y."""
        e = self.engine
        unknown = set(tan) - set(_capi.LQR_INPUT_FIELDS)
        if unknown:
            raise ValueError(f"not an LQR input: {sorted(unknown)}")
        dsol = self.alloc_output() if dsol is None else dsol
        if rhs is None:
            rhs = {k: e.empty(e.lqr_sizes[k]) for k in ("q", "r", "c")}
        status = e.empty_int() if status is None else status
        si, ss, st = _lqr_input_struct(inp), _lqr_output_struct(out), _lqr_input_struct(tan)
        sr = _lqr_output_struct(dict(x=rhs["q"], u=rhs["r"], y=rhs["c"]))
        sd = _lqr_output_struct(dsol)
        e._check(lib.sipoc_lqr_jvp(e._handle, ctypes.byref(si), ctypes.byref(ss),
                                   ctypes.byref(st), ctypes.byref(sr), ctypes.byref(sd),
                                   status.data_ptr(), e.stream_ptr(stream)))
        return dict(dsol, rhs=rhs, status=status)

    # -- optional FP32 mode (sipoc_lqr_factor_solve_f32; include/sipoc.h) -------------------
    @property
    def f32_supported(self) -> bool:
        return bool(lib.sipoc_f32_supported(self.engine._handle))

    def narrow_f32(self, arrays: dict) -> dict:
        """Engine-layout float64 device tensors -> float32 copies (plumbing, not timed)."""
        torch = self.engine._torch()
        return {k: v.to(torch.float32).contiguous() for k, v in arrays.items()}

    def alloc_output_f32(self) -> dict:
        e, sz = self.engine, self.engine.lqr_sizes
        torch = e._torch()
        return {k: e.empty(sz[k], dtype=torch.float32) for k in _capi.LQR_OUTPUT_FIELDS}

    def factor_solve_f32(self, inp32: dict, out32: dict, status=None, stream=None):
        """Factor + solve in single precision; every tensor float32 in the engine layout."""
        e = self.engine
        status = e.empty_int() if status is None else status
        si, so = _lqr_input_struct(inp32), _lqr_output_struct(out32)
        e._check(lib.sipoc_lqr_factor_solve_f32(e._handle, ctypes.byref(si), ctypes.byref(so),
                                                status.data_ptr(), e.stream_ptr(stream)))
        return status

    def factor_solve_thread_f64(self, inp: dict, out: dict, status=None, stream=None):
        """The FP32 mode's kernels instantiated on double (their numerical control)."""
        e = self.engine
        status = e.empty_int() if status is None else status
        si, so = _lqr_input_struct(inp), _lqr_output_struct(out)
        e._check(lib.sipoc_lqr_factor_solve_thread_f64(
            e._handle, ctypes.byref(si), ctypes.byref(so), status.data_ptr(),
            e.stream_ptr(stream)))
        return status

    # Problem-major device inputs (sipoc_lqr_*_pm): ``inp`` holds CUDA tensors laid out
    # [problem][flat] -- `problem_major_input` uploads host arrays that way.  Outputs stay
    # in the engine layout.
    def problem_major_input(self, host: dict) -> dict:
        e = self.engine
        torch = e._torch()
        return {k: torch.from_numpy(np.ascontiguousarray(host[k], dtype=np.float64)
                                    .reshape(self.batch, -1)).to(e.torch_device())
                for k in _capi.LQR_INPUT_FIELDS}

    def factor_with_status_pm(self, inp: dict, status=None, stream=None):
        if self.traversal_status_ != FactorStatus.SUCCESS:
            return self._invalid()
        e = self.engine
        status = e.empty_int() if status is None else status
        s = _lqr_input_struct(inp)
        e._check(lib.sipoc_lqr_factor_pm(e._handle, ctypes.byref(s), status.data_ptr(),
                                         e.stream_ptr(stream)))
        return status

    def solve_pm(self, inp: dict, out: dict, stream=None) -> None:
        e = self.engine
        si, so = _lqr_input_struct(inp), _lqr_output_struct(out)
        e._check(lib.sipoc_lqr_solve_pm(e._handle, ctypes.byref(si), ctypes.byref(so),
                                        e.stream_ptr(stream)))

    def factor_solve_pm(self, inp: dict, out: dict, status=None, stream=None):
        if self.traversal_status_ != FactorStatus.SUCCESS:
            return self._invalid()
        e = self.engine
        status = e.empty_int() if status is None else status
        si, so = _lqr_input_struct(inp), _lqr_output_struct(out)
        e._check(lib.sipoc_lqr_factor_solve_pm(e._handle, ctypes.byref(si), ctypes.byref(so),
                                               status.data_ptr(), e.stream_ptr(stream)))
        return status

    def residual(self, inp: dict, out: dict, status=None, stream=None):
        """Returns (per-problem KKT residual norms, 4 all-reducible statistics)."""
        e = self.engine
        torch = e._torch()
        norms = torch.zeros((e.batch_stride,), dtype=torch.float64, device=e.torch_device())
        stats = torch.zeros((4,), dtype=torch.float64, device=e.torch_device())
        si, so = _lqr_input_struct(inp), _lqr_output_struct(out)
        e._check(lib.sipoc_lqr_residual(e._handle, ctypes.byref(si), ctypes.byref(so),
                                        None if status is None else status.data_ptr(),
                                        norms.data_ptr(), stats.data_ptr(),
                                        e.stream_ptr(stream)))
        return norms, stats

    def generate_benchmark(self, seed: int, problem_offset: int = 0, inp=None, stream=None):
        """Fill ``inp`` with the reference benchmark distribution (uniform chains)."""
        e = self.engine
        inp = self.alloc_input() if inp is None else inp
        e._check(lib.sipoc_generate_lqr_benchmark(
            e._handle, int(seed), int(problem_offset),
            *[inp[k].data_ptr() for k in _capi.LQR_INPUT_FIELDS], e.stream_ptr(stream)))
        return inp

    # -- host path (reference-facing: host buffers, problem-major) --------------
    @staticmethod
    def _host_in(host: dict, keep: list) -> _capi.LqrInput:
        s = _capi.LqrInput()
        for k in _capi.LQR_INPUT_FIELDS:
            a = host.get(k)
            if a is not None:
                a = np.ascontiguousarray(a, dtype=np.float64)
                keep.append(a)
            setattr(s, k, _host_ptr(a))
        return s

    def _host_out(self, keep: list):
        out = {k: np.zeros((self.batch, self.engine.lqr_sizes[k])) for k in
               _capi.LQR_OUTPUT_FIELDS}
        s = _capi.LqrOutput()
        for k in _capi.LQR_OUTPUT_FIELDS:
            setattr(s, k, _host_ptr(out[k]))
        keep.append(out)
        return out, s

    def factor_solve_host(self, host: dict, out: Optional[dict] = None) -> dict:
        """factor + solve on host arrays; returns dict(x, u, y, status)."""
        if self.traversal_status_ != FactorStatus.SUCCESS:
            return dict(status=self._invalid())
        e, keep = self.engine, []
        si = self._host_in(host, keep)
        if out is None:
            out, so = self._host_out(keep)
        else:
            so = _capi.LqrOutput()
            for k in _capi.LQR_OUTPUT_FIELDS:
                setattr(so, k, _host_ptr(out[k]))
        status = np.zeros(self.batch, np.int32)
        e._check(lib.sipoc_lqr_factor_solve_host(e._handle, ctypes.byref(si), ctypes.byref(so),
                                                 _host_ptr(status)))
        return dict(x=out["x"], u=out["u"], y=out["y"], status=status)

    @staticmethod
    def pack_symmetric(blocks: np.ndarray, n: int) -> np.ndarray:
        """[batch, count n n] dense column-major symmetric blocks -> [batch, count n (n+1)/2]
        packed lower triangles (the layout sipoc_lqr_factor_solve_host_packed takes)."""
        if n == 0:
            return np.zeros((blocks.shape[0], 0))
        count = blocks.shape[1] // (n * n)
        idx = np.array([j * n + i for j in range(n) for i in range(j, n)])
        return np.ascontiguousarray(blocks.reshape(blocks.shape[0], count, n * n)[:, :, idx]
                                    .reshape(blocks.shape[0], -1))

    def factor_solve_host_packed(self, host: dict, out: Optional[dict] = None) -> dict:
        """factor + solve on host arrays with Q, R as packed lower triangles and M optional
        (None = zero): fewer bytes over the bus than the reference's dense blocks."""
        e, keep = self.engine, []
        si = _capi.LqrInput()
        for k in _capi.LQR_INPUT_FIELDS:
            a = host.get(k)
            if a is None:
                setattr(si, k, None)
                continue
            a = np.ascontiguousarray(a, dtype=np.float64)
            if not a.size:
                a = np.zeros(1)
            keep.append(a)
            setattr(si, k, _host_ptr(a))
        if out is None:
            out, so = self._host_out(keep)
        else:
            so = _capi.LqrOutput()
            for k in _capi.LQR_OUTPUT_FIELDS:
                setattr(so, k, _host_ptr(out[k]))
        status = np.zeros(self.batch, np.int32)
        e._check(lib.sipoc_lqr_factor_solve_host_packed(e._handle, ctypes.byref(si),
                                                        ctypes.byref(so), _host_ptr(status)))
        return dict(x=out["x"], u=out["u"], y=out["y"], status=status)

    def factor_host(self, host: dict) -> np.ndarray:
        if self.traversal_status_ != FactorStatus.SUCCESS:
            return self._invalid()
        e, keep = self.engine, []
        si = self._host_in(host, keep)
        status = np.zeros(self.batch, np.int32)
        e._check(lib.sipoc_lqr_factor_host(e._handle, ctypes.byref(si), _host_ptr(status)))
        return status

    def solve_host(self, host: dict) -> dict:
        e, keep = self.engine, []
        si = self._host_in(host, keep)
        out, so = self._host_out(keep)
        e._check(lib.sipoc_lqr_solve_host(e._handle, ctypes.byref(si), ctypes.byref(so)))
        return out
