"""Host-side mirror of the reference's ``CallbackProvider`` (helpers.hpp:7-33).

Batched: ``factor`` / ``solve`` / ``add_Kx_to_y`` keep the reference's argument
meaning; flat vectors use the reference wire format ``[x | y | z]`` with
``x = [x_0, u_0, ..., x_E, theta]`` (types.cpp:24-64) and every array gains a
batch axis.  With ``theta_dim > 0`` the model dict also carries the ten theta
block arrays (``_capi.KKT_THETA_FIELDS``).  All computation goes through the C
ABI (sipoc_kkt_*).
"""
from __future__ import annotations

import ctypes
from typing import Optional

import numpy as np

from . import _capi
from ._capi import lib
from .lqr import Dimensions, Engine, SipocError, Topology, _host_ptr, _ip


def _fill(struct, fields, model: dict, host: bool, keep: list) -> None:
    for k in fields:
        a = model[k]
        if host:
            a = np.ascontiguousarray(a, dtype=np.float64)
            if not a.size:  # ctypes needs a non-NULL pointer even for empty blocks
                a = np.zeros(1)
            keep.append(a)
            setattr(struct, k, _host_ptr(a))
        else:
            setattr(struct, k, a.data_ptr())


def _model_struct(model: dict, host: bool, keep: list) -> _capi.KktModel:
    """sipoc_kkt_model over device tensors (or host arrays); the theta blocks ride along when
    the dict has them.  Everything the struct points at is appended to ``keep``."""
    s = _capi.KktModel()
    _fill(s, _capi.KKT_MODEL_FIELDS, model, host, keep)
    if all(k in model for k in _capi.KKT_THETA_FIELDS):
        t = _capi.KktThetaModel()
        _fill(t, _capi.KKT_THETA_FIELDS, model, host, keep)
        keep.append(t)
        s.theta = ctypes.pointer(t)
    return s


class CapturedKktStep:
    """A recorded factor + solve + residual sequence (CallbackProvider.capture_step;
    sipoc_graph_* in include/sipoc.h).

    ``ok`` / ``norms`` / ``stats`` are the step's outputs, rewritten by every replay;
    ``launches`` is the number of engine kernels one replay runs."""

    def __init__(self, engine: Engine, handle, ok, norms, stats, keep=()):
        self._engine, self._graph = engine, handle
        self.ok, self.norms, self.stats = ok, norms, stats
        self.launches = int(lib.sipoc_graph_kernel_count(handle))
        self._keep = keep  # the graph holds raw device pointers into these tensors

    def replay(self, stream=None):
        """Enqueue the whole step on ``stream`` (default: torch's current, which must not be
        the legacy default stream's capture); returns (norms, stats)."""
        e = self._engine
        e._check(lib.sipoc_graph_launch(e._handle, self._graph, e.stream_ptr(stream)))
        return self.norms, self.stats

    def __del__(self):
        if getattr(self, "_graph", None):
            lib.sipoc_graph_destroy(self._graph)
            self._graph = None


class CallbackProvider:
    """Batched Newton-KKT linear solve behind the reference's callback names."""

    def __init__(self, dimensions: Dimensions, topology: Topology, batch: int = 1,
                 device: Optional[int] = None, force_generic: bool = False,
                 pad_variable_dims: bool = False):
        self.engine = Engine(dimensions, topology, batch, device, force_generic,
                             pad_variable_dims)
        self.batch = int(batch)
        # validate_input(...) == SUCCESS  (helpers.cpp:25-26)
        self.input_is_valid_ = self.engine.create_status == _capi.SIPOC_OK
        if not self.input_is_valid_ and self.engine.create_status not in (
                _capi.SIPOC_INVALID_TOPOLOGY, _capi.SIPOC_INVALID_DIMENSIONS):
            raise SipocError(self.engine.create_status, "sipoc_create failed")

    @property
    def sizes(self) -> dict:
        return self.engine.kkt_sizes

    def offsets(self) -> dict:
        E = self.engine.topology.num_edges
        names_n = ("x_state", "y_dyn", "y_node_c", "z_node")
        names_e = ("x_control", "y_edge_c", "z_edge")
        o = {k: np.zeros(E + 1, np.int32) for k in names_n}
        o.update({k: np.zeros(max(E, 1), np.int32) for k in names_e})
        self.engine._check(lib.sipoc_kkt_offsets(
            self.engine._handle, _ip(o["x_state"]), _ip(o["x_control"]), _ip(o["y_dyn"]),
            _ip(o["y_node_c"]), _ip(o["y_edge_c"]), _ip(o["z_node"]), _ip(o["z_edge"])))
        for k in names_e:
            o[k] = o[k][:E]
        return o

    # -- device path ------------------------------------------------------------
    def pack_model(self, host_model: dict) -> dict:
        fields = _capi.KKT_MODEL_FIELDS
        if self.engine.kkt_sizes["theta_dim"] > 0:
            fields = fields + _capi.KKT_THETA_FIELDS
        return {k: self.engine.pack(host_model[k]) for k in fields}

    def factor(self, model: dict, w, r1, r2, r3, ok=None, stream=None):
        """Returns a device int32 tensor: 1 where the reference's factor returns true."""
        e = self.engine
        if not self.input_is_valid_:
            return np.zeros(self.batch, np.int32)  # helpers.cpp:244-246
        ok = e.empty_int() if ok is None else ok
        keep = []
        m = _model_struct(model, False, keep)
        e._check(lib.sipoc_kkt_factor(e._handle, ctypes.byref(m), w.data_ptr(), r1.data_ptr(),
                                      r2.data_ptr(), r3.data_ptr(), ok.data_ptr(),
                                      e.stream_ptr(stream)))
        return ok

    def solve(self, model: dict, b, sol, stream=None) -> None:
        e = self.engine
        keep = []
        m = _model_struct(model, False, keep)
        e._check(lib.sipoc_kkt_solve(e._handle, ctypes.byref(m), b.data_ptr(), sol.data_ptr(),
                                     e.stream_ptr(stream)))

    def add_Kx_to_y(self, model: dict, w, r1, r2, r3, x, y, stream=None) -> None:
        """y += K(w, r1, r2, r3) x on [x|y|z] vectors (helpers.cpp:953-977)."""
        e = self.engine
        keep = []
        m = _model_struct(model, False, keep)
        e._check(lib.sipoc_kkt_apply(e._handle, ctypes.byref(m), w.data_ptr(), r1.data_ptr(),
                                     r2.data_ptr(), r3.data_ptr(), x.data_ptr(), y.data_ptr(),
                                     e.stream_ptr(stream)))

    # The five blocks of the operator on their own (helpers.hpp:17-21): y += B x on device
    # vectors of the block's own lengths (H: x -> x, C: x -> y, CT: y -> x, G: x -> z, GT: z -> x).
    def _apply_block(self, block: int, model: dict, x, y, stream=None) -> None:
        e = self.engine
        keep = []
        m = _model_struct(model, False, keep)
        e._check(lib.sipoc_kkt_apply_block(e._handle, ctypes.byref(m), block, x.data_ptr(),
                                           y.data_ptr(), e.stream_ptr(stream)))

    def add_Hx_to_y(self, model: dict, x, y, stream=None) -> None:
        self._apply_block(_capi.KKT_BLOCK_H, model, x, y, stream)

    def add_Cx_to_y(self, model: dict, x, y, stream=None) -> None:
        self._apply_block(_capi.KKT_BLOCK_C, model, x, y, stream)

    def add_CTx_to_y(self, model: dict, x, y, stream=None) -> None:
        self._apply_block(_capi.KKT_BLOCK_CT, model, x, y, stream)

    def add_Gx_to_y(self, model: dict, x, y, stream=None) -> None:
        self._apply_block(_capi.KKT_BLOCK_G, model, x, y, stream)

    def add_GTx_to_y(self, model: dict, x, y, stream=None) -> None:
        self._apply_block(_capi.KKT_BLOCK_GT, model, x, y, stream)

    def residual(self, model: dict, w, r1, r2, r3, sol, b, ok=None, stream=None, out=None):
        """(||K sol - b||_2 per problem, 4 all-reducible statistics); ``out`` = zeroed
        (norms, stats) tensors to write into instead of new ones."""
        e = self.engine
        torch = e._torch()
        if out is None:
            norms = torch.zeros((e.batch_stride,), dtype=torch.float64, device=e.torch_device())
            stats = torch.zeros((4,), dtype=torch.float64, device=e.torch_device())
        else:
            norms, stats = out
        keep = []
        m = _model_struct(model, False, keep)
        e._check(lib.sipoc_kkt_residual(
            e._handle, ctypes.byref(m), w.data_ptr(), r1.data_ptr(), r2.data_ptr(),
            r3.data_ptr(), sol.data_ptr(), b.data_ptr(),
            None if ok is None else ok.data_ptr(), norms.data_ptr(), stats.data_ptr(),
            e.stream_ptr(stream)))
        return norms, stats

    def vjp(self, model: dict, w, r1, r2, r3, sol, cot, want=None, ok=None, stream=None) -> dict:
        """Reverse-mode derivative of ``factor`` + ``solve`` (sipoc_kkt_vjp; include/sipoc.h).

        ``model``, ``w``, ``r1``, ``r2``, ``r3`` are the forward's inputs and ``sol`` its
        solution, ``cot`` is dL/dsol (engine layout).  ``want`` is the set of names to
        differentiate among ``_capi.KKT_GRAD_FIELDS`` (default: all of them, the theta blocks
        when theta_dim > 0); the others are neither computed nor written.  Returns a dict with
        one engine-layout gradient tensor per wanted name, ``adjoint`` (lam = K^-1 cot) and
        ``ok`` (the factorization's per-problem flags).  Symmetric Hessian blocks get the
        symmetric gradient; problems with ok == 0 and padding lanes get zeros."""
        e = self.engine
        if not self.input_is_valid_:
            raise SipocError(self.engine.create_status, "vjp on an invalid structure")
        sizes = self.sizes
        theta = sizes["theta_dim"] > 0
        fields = _capi.KKT_MODEL_FIELDS + (_capi.KKT_THETA_FIELDS if theta else ()) + \
            _capi.KKT_VECTOR_GRAD_FIELDS
        want = set(fields if want is None else want)
        unknown = want - set(fields)
        if unknown:
            raise ValueError(f"not a differentiable KKT input: {sorted(unknown)}")
        vec_size = dict(b=sizes["kkt_dim"], w=sizes["z_dim"], r1=sizes["x_dim"],
                        r2=sizes["y_dim"], r3=sizes["z_dim"])
        size = {k: vec_size.get(k, sizes.get(k, 0)) for k in fields}
        # an empty array is one row of zeros, as Engine.pack makes it
        grads = {k: e.empty(size[k]) if size[k] else e.zeros(0) for k in fields if k in want}
        adjoint = e.empty(sizes["kkt_dim"])
        ok = e.empty_int() if ok is None else ok
        keep = []
        m = _model_struct(model, False, keep)
        sg = _capi.KktGrad()
        for k in _capi.KKT_MODEL_FIELDS + _capi.KKT_VECTOR_GRAD_FIELDS:
            setattr(sg, k, grads[k].data_ptr() if k in grads else None)
        if theta and want & set(_capi.KKT_THETA_FIELDS):
            st = _capi.KktThetaGrad()
            for k in _capi.KKT_THETA_FIELDS:
                setattr(st, k, grads[k].data_ptr() if k in grads else None)
            keep.append(st)
            sg.theta = ctypes.pointer(st)
        e._check(lib.sipoc_kkt_vjp(e._handle, ctypes.byref(m), w.data_ptr(), r1.data_ptr(),
                                   r2.data_ptr(), r3.data_ptr(), sol.data_ptr(), cot.data_ptr(),
                                   adjoint.data_ptr(), ctypes.byref(sg), ok.data_ptr(),
                                   e.stream_ptr(stream)))
        grads["adjoint"] = adjoint
        grads["ok"] = ok
        return grads

    def jvp(self, model: dict, w, r1, r2, r3, sol, tan: dict, dsol=None, rhs=None, ok=None,
            stream=None) -> dict:
        """Forward-mode derivative of ``factor`` + ``solve`` (sipoc_kkt_jvp; include/sipoc.h).

        ``model``, ``w``, ``r1``, ``r2``, ``r3`` are the forward's inputs and ``sol`` its
        solution; ``tan`` holds the tangents of any subset of ``_capi.KKT_GRAD_FIELDS`` (the
        theta blocks when theta_dim > 0; engine layout).  An absent name is a zero tangent and
        is not read.  Returns a dict with ``sol`` (the tangent of the solution), ``rhs`` (the
        right-hand side t = db - dK sol the tangent solve used) and ``ok``.  Symmetric Hessian
        blocks enter through their symmetric parts; problems with ok == 0 and padding lanes
        get a zero tangent."""
        e = self.engine
        if not self.input_is_valid_:
            raise SipocError(self.engine.create_status, "jvp on an invalid structure")
        sizes = self.sizes
        theta = sizes["theta_dim"] > 0
        fields = _capi.KKT_MODEL_FIELDS + (_capi.KKT_THETA_FIELDS if theta else ()) + \
            _capi.KKT_VECTOR_GRAD_FIELDS
        unknown = set(tan) - set(fields)
        if unknown:
            raise ValueError(f"not a differentiable KKT input: {sorted(unknown)}")
        dsol = e.empty(sizes["kkt_dim"]) if dsol is None else dsol
        rhs = e.empty(sizes["kkt_dim"]) if rhs is None else rhs
        ok = e.empty_int() if ok is None else ok
        keep = []
        m = _model_struct(model, False, keep)
        st = _capi.KktTangent()
        for k in _capi.KKT_MODEL_FIELDS:
            setattr(st.model, k, tan[k].data_ptr() if k in tan else None)
        for k in _capi.KKT_VECTOR_GRAD_FIELDS:
            setattr(st, k, tan[k].data_ptr() if k in tan else None)
        if theta and set(tan) & set(_capi.KKT_THETA_FIELDS):
            tt = _capi.KktThetaModel()
            for k in _capi.KKT_THETA_FIELDS:
                setattr(tt, k, tan[k].data_ptr() if k in tan else None)
            keep.append(tt)
            st.model.theta = ctypes.pointer(tt)
        e._check(lib.sipoc_kkt_jvp(e._handle, ctypes.byref(m), w.data_ptr(), r1.data_ptr(),
                                   r2.data_ptr(), r3.data_ptr(), sol.data_ptr(),
                                   ctypes.byref(st), rhs.data_ptr(), dsol.data_ptr(),
                                   ok.data_ptr(), e.stream_ptr(stream)))
        return dict(sol=dsol, rhs=rhs, ok=ok)

    def capture_step(self, model: dict, w, r1, r2, r3, b, sol, ok=None) -> "CapturedKktStep":
        """factor + solve + residual (one Newton-KKT iteration's linear algebra,
        sip_optimal_control.cpp:129-145) recorded once as a CUDA graph over the given device
        tensors.  ``replay()`` relaunches the whole kernel sequence with one driver call;
        the caller refreshes the tensors' contents in place between replays."""
        e = self.engine
        if not self.input_is_valid_:
            raise SipocError(self.engine.create_status, "capture_step on an invalid structure")
        torch = e._torch()
        dev = e.torch_device()
        ok = e.empty_int() if ok is None else ok

        norms = torch.zeros((e.batch_stride,), dtype=torch.float64, device=dev)
        stats = torch.zeros((4,), dtype=torch.float64, device=dev)

        def step(stream):
            self.factor(model, w, r1, r2, r3, ok=ok, stream=stream)
            self.solve(model, b, sol, stream=stream)
            with torch.cuda.stream(stream):
                norms.zero_()
                stats.zero_()
            self.residual(model, w, r1, r2, r3, sol, b, ok=ok, stream=stream,
                          out=(norms, stats))

        # One eager pass on the capture stream first: the engine sizes its workspaces and
        # sets kernel attributes on first use, neither of which may happen under capture.
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        step(side)
        side.synchronize()
        handle = ctypes.c_void_p()
        e._check(lib.sipoc_graph_begin(e._handle, int(side.cuda_stream)))
        try:
            step(side)
        finally:
            rc = lib.sipoc_graph_end(e._handle, int(side.cuda_stream), ctypes.byref(handle))
        e._check(rc)
        return CapturedKktStep(e, handle, ok, norms, stats, keep=(model, w, r1, r2, r3, b, sol))

    # -- host path ----------------------------------------------------------------
    def factor_host(self, model: dict, w, r1, r2, r3) -> np.ndarray:
        e, keep = self.engine, []
        if not self.input_is_valid_:
            return np.zeros(self.batch, np.int32)
        m = _model_struct(model, True, keep)
        regs = [np.ascontiguousarray(a, dtype=np.float64) for a in (w, r1, r2, r3)]
        ok = np.zeros(self.batch, np.int32)
        e._check(lib.sipoc_kkt_factor_host(e._handle, ctypes.byref(m),
                                           *[_host_ptr(a) for a in regs], _host_ptr(ok)))
        return ok

    def set_model_host(self, model: dict) -> None:
        """Uploads the model alone (sipoc_kkt_set_model_host): what the host operator entry
        points read, e.g. after the model callback has run again."""
        e, keep = self.engine, []
        m = _model_struct(model, True, keep)
        e._check(lib.sipoc_kkt_set_model_host(e._handle, ctypes.byref(m)))

    def solve_host(self, b: np.ndarray) -> np.ndarray:
        e = self.engine
        b = np.ascontiguousarray(b, dtype=np.float64)
        sol = np.zeros_like(b)
        e._check(lib.sipoc_kkt_solve_host(e._handle, _host_ptr(b), _host_ptr(sol)))
        return sol

    def apply_block_host(self, block: int, x, y) -> np.ndarray:
        """y += B x for one block against the model of the last ``factor_host``."""
        e = self.engine
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.array(y, dtype=np.float64, order="C")
        e._check(lib.sipoc_kkt_apply_block_host(e._handle, block, _host_ptr(x), _host_ptr(y)))
        return y

    def add_Kx_to_y_host(self, w, r1, r2, r3, x, y=None) -> np.ndarray:
        e = self.engine
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (w, r1, r2, r3, x)]
        y = np.zeros_like(arrs[4]) if y is None else np.array(y, dtype=np.float64, order="C")
        e._check(lib.sipoc_kkt_apply_host(e._handle, *[_host_ptr(a) for a in arrs],
                                          _host_ptr(y)))
        return y

    # -- model-callback scatter (sip_optimal_control.cpp:13-127) -----------------------
    @property
    def model_value_sizes(self) -> dict:
        z = _capi.ModelValueSizes()
        self.engine._check(lib.sipoc_model_value_sizes(self.engine._handle, ctypes.byref(z)))
        return {k: int(getattr(z, k)) for k in _capi.MODEL_VALUE_FIELDS}

    def model_callback_scatter(self, values: dict, x, initial_state, new_x: bool = True,
                               stream=None) -> dict:
        """f, gradient_f, c, g of one model evaluation from its node / edge values (device
        tensors in the engine layout, ``engine.pack`` of [batch, size] arrays)."""
        e, keep = self.engine, []
        v = _capi.ModelValues()
        _fill(v, _capi.MODEL_VALUE_FIELDS, values, False, keep)
        sz = self.sizes
        out = dict(f=e.empty(1), gradient_f=e.empty(sz["x_dim"]), c=e.empty(sz["y_dim"]),
                   g=e.empty(sz["z_dim"]))
        e._check(lib.sipoc_model_scatter(
            e._handle, ctypes.byref(v), x.data_ptr(), initial_state.data_ptr(), int(new_x),
            out["f"].data_ptr(), out["gradient_f"].data_ptr(), out["c"].data_ptr(),
            out["g"].data_ptr(), e.stream_ptr(stream)))
        return out

    def model_callback_scatter_host(self, values: dict, x, initial_state,
                                    new_x: bool = True) -> dict:
        """The same through host buffers ([batch, size] numpy arrays), synchronous."""
        e, keep = self.engine, []
        v = _capi.ModelValues()
        _fill(v, _capi.MODEL_VALUE_FIELDS, values, True, keep)
        sz = self.sizes
        x = np.ascontiguousarray(x, dtype=np.float64)
        x0 = np.ascontiguousarray(initial_state, dtype=np.float64)
        out = dict(f=np.zeros(self.batch), gradient_f=np.zeros((self.batch, sz["x_dim"])),
                   c=np.zeros((self.batch, sz["y_dim"])), g=np.zeros((self.batch, sz["z_dim"])))
        ptr = lambda a: _host_ptr(a if a.size else np.zeros(1))
        e._check(lib.sipoc_model_scatter_host(
            e._handle, ctypes.byref(v), _host_ptr(x), _host_ptr(x0), int(new_x),
            _host_ptr(out["f"]), ptr(out["gradient_f"]), ptr(out["c"]), ptr(out["g"])))
        return out
