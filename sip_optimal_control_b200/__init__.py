"""B200-native batched regularized-LQR / Newton-KKT linear-solve engine.

Drop-in for the Newton-KKT linear-solve path of joaospinto/sip_optimal_control
(``LQR::factor/solve`` and ``CallbackProvider::factor/solve/add_Kx_to_y``),
one optimal-control problem per batch element, computed by hand-written
sm_100a CUDA kernels behind the C ABI of ``include/sipoc.h``.

Importing the package loads ``lib/libsipoc.so`` and fails loudly if it has not
been built; there is no CPU or PyTorch fallback.
"""
from ._capi import LIB_PATH, declared_symbols  # noqa: F401
from .kkt import CallbackProvider  # noqa: F401
from .lqr import LQR, Dimensions, Engine, FactorStatus, SipocError, Topology  # noqa: F401

__all__ = ["LQR", "CallbackProvider", "Dimensions", "Topology", "Engine", "FactorStatus",
           "SipocError", "LIB_PATH", "declared_symbols", "autograd"]


def __getattr__(name):
    # ``autograd`` (torch.autograd bindings of the LQR and KKT solves) imports torch, which the rest of
    # the package loads only when it first touches a device: import it on first use.
    if name == "autograd":
        import importlib

        return importlib.import_module(".autograd", __name__)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
