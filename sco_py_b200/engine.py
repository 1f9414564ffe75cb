"""Engine: one compiled problem structure bound to one GPU (wraps sco_handle).

PyTorch is used only to own device memory and streams; every numerical step is a
kernel of libsco_b200.so reached through ctypes.
"""
import contextlib
import ctypes

import numpy as np
import torch

from . import _lib
from .structure import CNT_EQ, Structure

SETTING_NAMES = [f[0] for f in _lib.CSettings._fields_ if f[0] != "pad_"]


def make_settings(solver=None, osqp=None, **extra):
    """CSettings from Solver attributes (solver.py:17-28) and OSQP keywords (osqp_utils.py:10-15)."""
    lib = _lib.load()
    s = _lib.CSettings()
    lib.sco_default_settings(ctypes.byref(s))
    for k, v in (solver or {}).items():
        if k == "max_iter":  # Solver.max_iter is never read by the reference (solver.py:21)
            continue
        if not hasattr(s, k):
            raise KeyError("unknown solver setting %r" % k)
        setattr(s, k, v)
    osqp_map = {"eps_abs": "osqp_eps_abs", "eps_rel": "osqp_eps_rel", "max_iter": "osqp_max_iter",
                "rho": "osqp_rho", "sigma": "osqp_sigma", "adaptive_rho": "osqp_adaptive_rho",
                "alpha": "osqp_alpha", "scaling": "osqp_scaling",
                "adaptive_rho_interval": "osqp_adaptive_rho_interval"}
    for k, v in (osqp or {}).items():
        setattr(s, osqp_map.get(k, k), int(v) if isinstance(v, bool) else v)
    for k, v in extra.items():
        setattr(s, k, v)
    return s


def _field(f):
    return _lib.CField(int(f.off), int(bool(f.shared)), 0)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


class Engine(object):
    def __init__(self, st: Structure, device=0):
        if not torch.cuda.is_available():
            raise RuntimeError("sco_py_b200.Engine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.st = st
        self.device = torch.device("cuda", device)
        cs = _lib.CStructure()
        cs.n, cs.m_lin, cs.n_blocks, cs.n_groups = st.n, st.m_lin, len(st.blocks), st.n_groups
        cs.stride = st.stride
        self._keep = []

        def hold(a, dt):
            a = np.ascontiguousarray(a, dtype=dt)
            self._keep.append(a)
            return a.ctypes.data

        cs.shared_len = 0 if st.shared is None else int(np.asarray(st.shared).size)
        cs.shared = hold(st.shared, np.float64) if st.shared is not None else None
        cs.Q, cs.q, cs.c = _field(st.Q), _field(st.q), _field(st.c)
        cs.lin_l, cs.lin_u = _field(st.lin_l), _field(st.lin_u)
        cs.obj_prog, cs.obj_prog_len = _field(st.obj_prog), int(st.obj_prog_len)
        cs.obj_prog_flags = int(getattr(st, "obj_prog_flags", 0))
        cs.qa, cs.lb0, cs.ub0 = _field(st.qa), _field(st.lb0), _field(st.ub0)
        if st.m_lin:
            cs.lin_rowptr = hold(st.lin_rowptr, np.int32)
            cs.lin_col = hold(st.lin_col, np.int32)
            cs.lin_val = hold(st.lin_val, np.float64)
        if st.group_overlap is not None:
            cs.group_overlap = hold(st.group_overlap, np.int32)
        for i, b in enumerate(st.blocks):
            cb = cs.blocks[i]
            cb.family, cb.cnt_type, cb.m, cb.group_mask, cb.jw = b.family, b.cnt_type, b.m, b.group_mask, b.jw
            for k in range(8):
                cb.ipar[k] = int(b.ipar[k])
            cb.par, cb.val = _field(b.par), _field(b.val)
            if b.cols is not None:
                cb.n_in = int(np.shape(b.cols)[1])
                cb.cols = hold(b.cols, np.int32)
        cs.n_obj_blocks = len(st.obj_blocks)
        for i, ob in enumerate(st.obj_blocks):
            co = cs.obj_blocks[i]
            co.m, co.n_in, co.n_instr, co.flags = ob.m, ob.n_in, ob.n_instr, ob.flags
            co.prog = _field(ob.prog)
            co.cols = hold(ob.cols, np.int32)
        h = ctypes.c_void_p()
        _lib.check(self.lib.sco_create(ctypes.byref(cs), device, ctypes.byref(h)))
        self.h = h
        q = (ctypes.c_int64 * 8)()
        _lib.check(self.lib.sco_query(self.h, q))
        (self.n, self.m_nl, self.n_slack, self.jnnz, self.n_q, self.smem_bytes, self.team,
         self.occupancy) = [int(v) for v in q]
        # 32-bit words per penalty row of the frozen-sparsity mask passed to qp_solve (include/sco_b200.h)
        self.mask_words = max(1, max([(b.jw + 31) // 32 for b in st.blocks], default=1))

    def close(self):
        if getattr(self, "h", None):
            self.lib.sco_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _dev(self, a, dtype=torch.float64):
        if a is None:
            return None
        if isinstance(a, torch.Tensor):
            return a.to(self.device, dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(self.device)

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ hot path
    def solve_batch(self, params, x0, settings, stream=None, order=None):
        """Device-resident solve, enqueued on `stream` (default: torch's current stream).
        `order`: optional int32 device tensor, a permutation of range(B): the order in which the work
        queue hands problems out (longest first hides the tail).
        Returns dict of torch tensors (x, verdict, merit, objective, max_vio, stats)."""
        with (torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()):
            params, x0 = self._dev(params), self._dev(x0)
            B = x0.shape[0]
            x = torch.empty_like(x0)
            verdict = torch.empty(B, dtype=torch.int32, device=self.device)
            merit = torch.empty(B, dtype=torch.float64, device=self.device)
            obj = torch.empty_like(merit)
            vio = torch.empty_like(merit)
            stats = torch.empty((B, 4), dtype=torch.int32, device=self.device)
            nonconv = torch.empty(B, dtype=torch.int32, device=self.device)
            if order is not None:
                order = order.to(self.device, torch.int32).contiguous()
                assert order.numel() == B
            io = _lib.CBatchIO(params.data_ptr(), x0.data_ptr(), x.data_ptr(), verdict.data_ptr(), merit.data_ptr(),
                               obj.data_ptr(), vio.data_ptr(), stats.data_ptr(), nonconv.data_ptr(),
                               order.data_ptr() if order is not None else None, None, None)
            _lib.check(self.lib.sco_solve_batch_io(self.h, B, ctypes.byref(io), ctypes.byref(settings), self._stream()))
        return dict(x=x, verdict=verdict, merit=merit, objective=obj, max_vio=vio, stats=stats, nonconverged=nonconv)

    def solve_batch_host(self, params, x0, settings, out=None, stream=None):
        """Host buffers in, host buffers out (copies inside): the end-to-end entry.  With `stream`
        (a torch.cuda.Stream) everything is only enqueued there -- pinned buffers, caller synchronises."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        B = x0.shape[0]
        if out is None:
            out = dict(x=np.empty_like(x0), verdict=np.empty(B, np.int32), merit=np.empty(B),
                       objective=np.empty(B), max_vio=np.empty(B), stats=np.empty((B, 4), np.int32),
                       nonconverged=np.empty(B, np.int32))
        vp = lambda a: ctypes.c_void_p(a.ctypes.data) if a is not None else ctypes.c_void_p(0)
        cs = ctypes.c_void_p(stream.cuda_stream) if stream is not None else ctypes.c_void_p(0)
        _lib.check(self.lib.sco_solve_batch_host_groups(
            self.h, B, vp(params), vp(x0), ctypes.byref(settings), vp(out["x"]), vp(out["verdict"]),
            vp(out["merit"]), vp(out["objective"]), vp(out["max_vio"]), vp(out["stats"]),
            vp(out.get("nonconverged")), cs))
        if stream is None:  # the legacy stream: wait for it, like sco_solve_batch_host
            torch.cuda.default_stream(self.device).synchronize()
        return out

    # ------------------------------------------------------------------ stages
    def convexify(self, params, x):
        params, x = self._dev(params), self._dev(x)
        B = x.shape[0]
        f = torch.empty((B, self.m_nl), dtype=torch.float64, device=self.device)
        J = torch.empty((B, self.jnnz), dtype=torch.float64, device=self.device)
        b = torch.empty((B, self.m_nl), dtype=torch.float64, device=self.device)
        obj = torch.empty(B, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.sco_convexify(self.h, B, _ptr(params), _ptr(x), _ptr(f), _ptr(J), _ptr(b),
                                          _ptr(obj), self._stream()))
        return f, J, b, obj

    def convexify_model(self, params, x):
        """Convex model of the non-quadratic objective terms at x, each term convexified on its own and the models
        summed (expr.py:143-153): (sum_t H_t+ [B,n,n], sum_t A_t [B,n], sum_t b_t [B])."""
        params, x = self._dev(params), self._dev(x)
        B = x.shape[0]
        H = torch.empty((B, self.n, self.n), dtype=torch.float64, device=self.device)
        g = torch.empty((B, self.n), dtype=torch.float64, device=self.device)
        c = torch.empty(B, dtype=torch.float64, device=self.device)
        _lib.check(self.lib.sco_convexify_model(self.h, B, _ptr(params), _ptr(x), None, None, None, None, _ptr(H),
                                                _ptr(g), _ptr(c), self._stream()))
        return H, g, c

    def qp_solve(self, params, settings, J=None, b=None, mask=None, lbx=None, ubx=None, pi=None,
                 kdup=None, xref=None, use_penalty=True, closest_point=False, wa=None):
        params = self._dev(params)
        B = params.shape[0]
        J, b, lbx, ubx, pi, xref, wa = [self._dev(a) for a in (J, b, lbx, ubx, pi, xref, wa)]
        mask = self._dev(mask, torch.int32) if mask is not None else None
        if mask is not None and mask.numel() != B * self.m_nl * self.mask_words:
            raise ValueError("mask must hold %d x %d x %d 32-bit words" % (B, self.m_nl, self.mask_words))
        kdup = self._dev(kdup, torch.int32) if kdup is not None else None
        nq = self.n_q if use_penalty else self.n
        xq = torch.empty((B, nq), dtype=torch.float64, device=self.device)
        status = torch.empty(B, dtype=torch.int32, device=self.device)
        iters = torch.empty(B, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.sco_qp_solve_w(self.h, B, _ptr(params), _ptr(J), _ptr(b), _ptr(mask), _ptr(lbx),
                                           _ptr(ubx), _ptr(pi), _ptr(kdup), _ptr(wa), _ptr(xref), int(use_penalty),
                                           int(closest_point), ctypes.byref(settings), _ptr(xq),
                                           _ptr(status), _ptr(iters), self._stream()))
        return xq, status, iters

    def merit(self, params, x, mu, J=None, b=None):
        params, x, mu, J, b = [self._dev(a) for a in (params, x, mu, J, b)]
        B = x.shape[0]
        ng = self.st.n_groups
        merit = torch.empty(B, dtype=torch.float64, device=self.device)
        model = torch.full((B,), float("nan"), dtype=torch.float64, device=self.device)
        vio = torch.empty_like(merit)
        gv = torch.empty((B, ng), dtype=torch.float64, device=self.device)
        gm = torch.full((B, ng), float("nan"), dtype=torch.float64, device=self.device)
        _lib.check(self.lib.sco_merit(self.h, B, _ptr(params), _ptr(x), _ptr(J), _ptr(b), _ptr(mu),
                                      _ptr(merit), _ptr(model), _ptr(vio), _ptr(gv), _ptr(gm),
                                      self._stream()))
        return merit, model, vio, gv, gm
