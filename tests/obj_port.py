"""The oracle port (oracle/sqp_port.py) with non-quadratic objective terms bound to any Variable
(Structure.obj_blocks, include/sco_b200.h sco_obj_block_desc).

Every term is convexified on its own, as Prob.convexify calls BoundExpr.convexify(degree=2) per term
(prob.py:522-544; expr.py:143-153, 431-437): numerical Hessian of f_t on x[c_t], shift -min(lambda_min, 0) I,
A_t = g_t - x_t'H_t, b_t = 0.5 x_t'H_t x_t - g_t.x_t + f_t.  The QP gets P += sum_t scatter(H_t), q += sum_t
scatter(A_t) (prob.py:348-367); the merits sum f_t (prob.py:573-574) and the terms' models (prob.py:624-626).

`with obj_port(): ...` makes sqp_port.PortProblem (and so sqp_port.solve) take objective blocks this way; it composes
with bound_port.mapped_port().  `terms_of(st, row)` lists the terms as (f(xloc), grad(xloc) or None, cols).
"""
import contextlib

import numpy as np

import families as fam  # oracle/families.py
import numdifftools as nd  # oracle/shims/numdifftools
import sqp_port  # oracle/sqp_port.py

_PortProblem = sqp_port.PortProblem


def terms_of(st, row):
    """[(f(xloc) -> float, analytic gradient (xloc) -> (n_in,) or None, cols)] in block order, terms in their order."""
    terms = []
    for ob in st.obj_blocks:
        prog = sqp_port._field(st, ob.prog, row, ob.m + 2 * ob.n_instr)
        for r in range(ob.m):
            pr = np.concatenate([prog[r:r + 1], prog[ob.m:]])  # term r alone: its offset, every instruction
            f = lambda v, pr=pr: float(fam.vm_f(np.asarray(v, dtype=float).reshape(-1, 1), pr, 1)[0, 0])
            g = None
            if ob.flags & 1:
                g = lambda v, pr=pr: np.asarray(fam.vm_grad(np.asarray(v, dtype=float).reshape(-1, 1), pr, 1)).ravel()
            terms.append((f, g, np.asarray(ob.cols[r], dtype=np.int64)))
    return terms


def term_model(f, g, xl):
    """Expr.convexify(degree=2) of one term at its inputs xl (expr.py:143-153): (H+, A, b)."""
    H = nd.Hessian(f)(xl.copy())
    H = np.atleast_2d(H)
    lam = float(np.min(np.linalg.eigvalsh(H)))
    if lam < 0:
        H = H - np.eye(xl.size) * lam
    gv = g(xl) if g is not None else np.asarray(nd.Jacobian(f)(xl.copy()), dtype=float).ravel()
    A = gv - xl @ H
    b = float(0.5 * xl @ (H @ xl) - gv @ xl + f(xl))
    return H, A, b


class ObjPortProblem(_PortProblem):
    def __init__(self, st, row, x0):
        _PortProblem.__init__(self, st, row, x0)
        self.terms = terms_of(st, row) if getattr(st, "obj_blocks", None) else []
        self.models = None

    def objective(self, x):
        v = _PortProblem.objective(self, x)
        for f, _, c in self.terms:
            v += f(x[c, 0])
        return v

    def objective_model(self, x):
        v = _PortProblem.objective_model(self, x)
        for (H, A, b), (_, _, c) in zip(self.models or [], self.terms):
            xl = x[c, 0]
            v += float(0.5 * xl @ (H @ xl) + A @ xl + b)
        return v

    def convexify(self):
        _PortProblem.convexify(self)
        if self.terms:
            self.models = [term_model(f, g, self.x[c, 0]) for f, g, c in self.terms]
            self.Hq, self.aq, self.bq = assemble(self.n, self.models, [c for _, _, c in self.terms])

    def solve_qp(self, *args, **kw):
        if not self.terms:
            return _PortProblem.solve_qp(self, *args, **kw)
        self.obj_prog = ()  # the port adds the assembled model (Hq, aq) to P and q when obj_prog is set
        try:
            return _PortProblem.solve_qp(self, *args, **kw)
        finally:
            self.obj_prog = None


def assemble(n, models, cols):
    """sum_t scatter(H_t), sum_t scatter(A_t), sum_t b_t."""
    H, a, b = np.zeros((n, n)), np.zeros(n), 0.0
    for (Ht, At, bt), c in zip(models, cols):
        H[np.ix_(c, c)] += Ht
        a[c] += At
        b += bt
    return H, a, b


@contextlib.contextmanager
def obj_port():
    sqp_port.PortProblem = ObjPortProblem
    try:
        yield
    finally:
        sqp_port.PortProblem = _PortProblem


def model_at(st, row, x):
    """The assembled convex model of the objective terms at x: (H, A, c) as sco_convexify_model returns them."""
    terms = terms_of(st, row)
    models = [term_model(f, g, np.asarray(x, dtype=float)[c]) for f, g, c in terms]
    return assemble(st.n, models, [c for _, _, c in terms])


def solve(st, row, x0, **kw):
    """sqp_port.solve on a structure that may have objective blocks and column maps."""
    import bound_port
    with bound_port.mapped_port(), obj_port():
        return sqp_port.solve(st, row, x0, **kw)
