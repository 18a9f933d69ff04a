"""ctypes binding of include/sipoc.h.

Loads sip_optimal_control_b200/lib/libsipoc.so (built in-tree by ``make`` /
``__graft_entry__.build()``).  There is no fallback of any kind: if the shared
library is missing, or a symbol declared in sipoc.h is not exported, importing
this module raises.
"""
from __future__ import annotations

import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
# SIPOC_LIB_PATH: development override (tools/build_variant.sh), another build of the same library
LIB_PATH = os.environ.get("SIPOC_LIB_PATH") or os.path.join(_HERE, "lib", "libsipoc.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "sipoc.h")

c_int_p = ctypes.POINTER(ctypes.c_int)
c_dbl_p = ctypes.POINTER(ctypes.c_double)
c_void_p = ctypes.c_void_p

SIPOC_OK = 0
ERROR_NAMES = {
    0: "SIPOC_OK", 1: "SIPOC_INVALID_ARGUMENT", 2: "SIPOC_CUDA_ERROR",
    3: "SIPOC_OUT_OF_MEMORY", 4: "SIPOC_INVALID_TOPOLOGY", 5: "SIPOC_INVALID_DIMENSIONS",
    6: "SIPOC_UNSUPPORTED", 7: "SIPOC_NOT_FACTORED",
}
SIPOC_INVALID_TOPOLOGY = 4
SIPOC_INVALID_DIMENSIONS = 5
SIPOC_COMM_ID_BYTES = 128
SIPOC_FLAG_FORCE_GENERIC = 1
SIPOC_FLAG_PAD_VARIABLE_DIMS = 2
SIPOC_FLAG_PARALLEL_IN_TIME = 4
SIPOC_FLAG_SERIAL_IN_TIME = 8
# sipoc_kkt_block
KKT_BLOCK_H, KKT_BLOCK_C, KKT_BLOCK_CT, KKT_BLOCK_G, KKT_BLOCK_GT = range(5)


class Structure(ctypes.Structure):
    _fields_ = [
        ("num_edges", ctypes.c_int), ("root", ctypes.c_int),
        ("edge_parents", c_int_p), ("edge_children", c_int_p),
        ("state_dims", c_int_p), ("control_dims", c_int_p),
        ("node_c_dims", c_int_p), ("node_g_dims", c_int_p),
        ("edge_c_dims", c_int_p), ("edge_g_dims", c_int_p),
        ("theta_dim", ctypes.c_int), ("batch", ctypes.c_int64),
        ("device", ctypes.c_int), ("flags", ctypes.c_int),
    ]


LQR_INPUT_FIELDS = ("Q", "M", "R", "q", "r", "A", "B", "c", "delta")
LQR_OUTPUT_FIELDS = ("x", "u", "y")
KKT_MODEL_FIELDS = ("node_hxx", "node_jc", "node_jg", "edge_hxx", "edge_hxu", "edge_huu",
                    "edge_A", "edge_B", "edge_jcx", "edge_jcu", "edge_jgx", "edge_jgu")


class LqrSizes(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int64) for k in LQR_INPUT_FIELDS + LQR_OUTPUT_FIELDS]


class LqrInput(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in LQR_INPUT_FIELDS]


class LqrOutput(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in LQR_OUTPUT_FIELDS]


class LqrCotangent(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in LQR_OUTPUT_FIELDS]


class LqrGrad(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in LQR_INPUT_FIELDS]


# sipoc_lqr_policy: feedback gains K, k and cost-to-go V, v; the element counts of M, r, Q, q
LQR_POLICY_FIELDS = ("K", "k", "V", "v")
LQR_POLICY_SIZE_OF = dict(K="M", k="r", V="Q", v="q")


class LqrPolicy(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in LQR_POLICY_FIELDS]


# sipoc_lqr_policy_cotangent: dL/d(K, k, V, v); any may be NULL (zeros)
class LqrPolicyCotangent(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in LQR_POLICY_FIELDS]


KKT_THETA_FIELDS = ("node_hxt", "node_jct", "node_jgt", "node_htt", "edge_hxt", "edge_hut",
                    "edge_dynt", "edge_jct", "edge_jgt", "edge_htt")


class KktSizes(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int64) for k in ("x_dim", "y_dim", "z_dim", "kkt_dim") +
                KKT_MODEL_FIELDS + ("theta_dim", "stagewise_x_dim") + KKT_THETA_FIELDS]


class KktThetaModel(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in KKT_THETA_FIELDS]


class KktModel(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in KKT_MODEL_FIELDS] + \
        [("theta", ctypes.POINTER(KktThetaModel))]


KKT_VECTOR_GRAD_FIELDS = ("b", "w", "r1", "r2", "r3")
# every array sipoc_kkt_vjp can differentiate (sipoc_kkt_grad and its theta part)
KKT_GRAD_FIELDS = KKT_MODEL_FIELDS + KKT_THETA_FIELDS + KKT_VECTOR_GRAD_FIELDS


class KktThetaGrad(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in KKT_THETA_FIELDS]


class KktGrad(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in KKT_MODEL_FIELDS] + \
        [("theta", ctypes.POINTER(KktThetaGrad))] + [(k, c_void_p) for k in KKT_VECTOR_GRAD_FIELDS]


# sipoc_kkt_tangent: a tangent of every array of KKT_GRAD_FIELDS
class KktTangent(ctypes.Structure):
    _fields_ = [("model", KktModel)] + [(k, c_void_p) for k in KKT_VECTOR_GRAD_FIELDS]


MODEL_VALUE_FIELDS = ("node_f", "node_df_dx", "node_df_dtheta", "node_c", "node_g", "edge_f",
                      "edge_df_dx", "edge_df_du", "edge_df_dtheta", "edge_dyn_res", "edge_c",
                      "edge_g")


class ModelValueSizes(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int64) for k in MODEL_VALUE_FIELDS]


class ModelValues(ctypes.Structure):
    _fields_ = [(k, c_void_p) for k in MODEL_VALUE_FIELDS]


def declared_symbols() -> list[str]:
    """Every function name include/sipoc.h declares."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sipoc_[a-z_0-9]+)\s*\(", text)))


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
            "The engine has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    if missing:
        raise ImportError(f"libsipoc.so does not export {missing}")

    E = c_void_p  # sipoc_engine*
    P = c_void_p  # any device / host data pointer
    lib.sipoc_validate.argtypes = [ctypes.POINTER(Structure)]
    lib.sipoc_create.argtypes = [ctypes.POINTER(Structure), ctypes.POINTER(E)]
    lib.sipoc_destroy.argtypes = [E]
    lib.sipoc_destroy.restype = None
    lib.sipoc_version.restype = ctypes.c_int
    lib.sipoc_last_error.argtypes = [E]
    lib.sipoc_last_error.restype = ctypes.c_char_p
    lib.sipoc_kernel_variant.argtypes = [E]
    lib.sipoc_kernel_variant.restype = ctypes.c_char_p
    lib.sipoc_get_topology.argtypes = [E, c_int_p, c_int_p, c_int_p, c_int_p]
    lib.sipoc_launch_count.argtypes = [E]
    lib.sipoc_launch_count.restype = ctypes.c_int64
    lib.sipoc_graph_begin.argtypes = [E, ctypes.c_void_p]
    lib.sipoc_graph_end.argtypes = [E, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]
    lib.sipoc_graph_launch.argtypes = [E, ctypes.c_void_p, ctypes.c_void_p]
    lib.sipoc_graph_kernel_count.argtypes = [ctypes.c_void_p]
    lib.sipoc_graph_kernel_count.restype = ctypes.c_int64
    lib.sipoc_graph_destroy.argtypes = [ctypes.c_void_p]
    lib.sipoc_graph_destroy.restype = None
    lib.sipoc_profile_enable.argtypes = [E, ctypes.c_int]
    lib.sipoc_profile_collect.argtypes = [E]
    lib.sipoc_profile_collect.restype = ctypes.c_int
    lib.sipoc_profile_get.argtypes = [E, ctypes.c_int, ctypes.POINTER(ctypes.c_char_p),
                                      ctypes.POINTER(ctypes.c_double),
                                      ctypes.POINTER(ctypes.c_int64)]
    lib.sipoc_lqr_get_sizes.argtypes = [E, ctypes.POINTER(LqrSizes)]
    lib.sipoc_batch.argtypes = [E]
    lib.sipoc_batch.restype = ctypes.c_int64
    lib.sipoc_batch_stride.argtypes = [E]
    lib.sipoc_batch_stride.restype = ctypes.c_int64
    LI, LO = ctypes.POINTER(LqrInput), ctypes.POINTER(LqrOutput)
    lib.sipoc_lqr_factor.argtypes = [E, LI, P, P]
    lib.sipoc_lqr_solve.argtypes = [E, LI, LO, P]
    lib.sipoc_lqr_factor_solve.argtypes = [E, LI, LO, P, P]
    lib.sipoc_lqr_factor_pm.argtypes = [E, LI, P, P]
    lib.sipoc_lqr_solve_pm.argtypes = [E, LI, LO, P]
    lib.sipoc_lqr_factor_solve_pm.argtypes = [E, LI, LO, P, P]
    lib.sipoc_lqr_residual.argtypes = [E, LI, LO, P, P, P, P]
    lib.sipoc_lqr_vjp.argtypes = [E, LI, LO, ctypes.POINTER(LqrCotangent), LO,
                                  ctypes.POINTER(LqrGrad), P, P]
    lib.sipoc_lqr_jvp.argtypes = [E, LI, LO, LI, LO, LO, P, P]
    lib.sipoc_lqr_factor_solve_policy.argtypes = [E, LI, LO, ctypes.POINTER(LqrPolicy), P, P]
    lib.sipoc_lqr_policy_vjp.argtypes = [E, LI, P, P, P, ctypes.POINTER(LqrPolicyCotangent),
                                         ctypes.POINTER(LqrGrad), P]
    lib.sipoc_lqr_policy_jvp.argtypes = [E, LI, P, P, P, LI, ctypes.POINTER(LqrPolicy), P]
    lib.sipoc_status_stats.argtypes = [E, P, P, P]
    lib.sipoc_pack.argtypes = [E, P, P, ctypes.c_int64, P]
    lib.sipoc_unpack.argtypes = [E, P, P, ctypes.c_int64, P]
    lib.sipoc_lqr_factor_solve_host.argtypes = [E, LI, LO, P]
    lib.sipoc_lqr_factor_host.argtypes = [E, LI, P]
    lib.sipoc_lqr_solve_host.argtypes = [E, LI, LO]
    lib.sipoc_kkt_get_sizes.argtypes = [E, ctypes.POINTER(KktSizes)]
    lib.sipoc_kkt_offsets.argtypes = [E] + [c_int_p] * 7
    KM = ctypes.POINTER(KktModel)
    lib.sipoc_kkt_factor.argtypes = [E, KM, P, P, P, P, P, P]
    lib.sipoc_kkt_solve.argtypes = [E, KM, P, P, P]
    lib.sipoc_kkt_apply.argtypes = [E, KM, P, P, P, P, P, P, P]
    lib.sipoc_kkt_apply_block.argtypes = [E, KM, ctypes.c_int, P, P, P]
    lib.sipoc_kkt_vjp.argtypes = [E, KM, P, P, P, P, P, P, P, ctypes.POINTER(KktGrad), P, P]
    lib.sipoc_kkt_jvp.argtypes = [E, KM, P, P, P, P, P, ctypes.POINTER(KktTangent), P, P, P, P]
    lib.sipoc_kkt_apply_block_host.argtypes = [E, ctypes.c_int, P, P]
    lib.sipoc_lqr_factor_solve_host_packed.argtypes = [E, LI, LO, P]
    lib.sipoc_f32_supported.argtypes = [E]
    lib.sipoc_f32_supported.restype = ctypes.c_int
    lib.sipoc_lqr_factor_solve_f32.argtypes = [E, LI, LO, P, P]
    lib.sipoc_lqr_factor_solve_thread_f64.argtypes = [E, LI, LO, P, P]
    MV = ctypes.POINTER(ModelValues)
    lib.sipoc_model_value_sizes.argtypes = [E, ctypes.POINTER(ModelValueSizes)]
    lib.sipoc_model_scatter.argtypes = [E, MV, P, P, ctypes.c_int, P, P, P, P, P]
    lib.sipoc_model_scatter_host.argtypes = [E, MV, P, P, ctypes.c_int, P, P, P, P]
    lib.sipoc_kkt_residual.argtypes = [E, KM, P, P, P, P, P, P, P, P, P, P]
    lib.sipoc_kkt_factor_host.argtypes = [E, KM, P, P, P, P, P]
    lib.sipoc_kkt_solve_host.argtypes = [E, P, P]
    lib.sipoc_kkt_set_model_host.argtypes = [E, KM]
    lib.sipoc_kkt_apply_host.argtypes = [E, P, P, P, P, P, P]
    C = c_void_p  # sipoc_comm*
    lib.sipoc_shard_range.argtypes = [ctypes.c_int64, ctypes.c_int, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]
    lib.sipoc_comm_unique_id.argtypes = [P]
    lib.sipoc_comm_create.argtypes = [P, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.POINTER(C)]
    lib.sipoc_comm_create_all.argtypes = [c_int_p, ctypes.c_int, ctypes.POINTER(C)]
    lib.sipoc_comm_destroy.argtypes = [C]
    lib.sipoc_comm_destroy.restype = None
    lib.sipoc_comm_rank.argtypes = [C]
    lib.sipoc_comm_size.argtypes = [C]
    lib.sipoc_comm_group_begin.argtypes = []
    lib.sipoc_comm_group_end.argtypes = []
    lib.sipoc_comm_allreduce_stats.argtypes = [C, P, P]
    lib.sipoc_comm_allgather_stats.argtypes = [C, P, P]
    lib.sipoc_comm_fold_stats.argtypes = [C, P, P]
    lib.sipoc_attach_comm.argtypes = [E, C]
    lib.sipoc_generate_lqr_benchmark.argtypes = [E, ctypes.c_uint64, ctypes.c_int64] + [P] * 9 + [P]
    for name in declared_symbols():
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int and name not in ("sipoc_version",):
            fn.restype = ctypes.c_int
    return lib


lib = _load()
