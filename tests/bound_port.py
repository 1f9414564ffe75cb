"""The oracle port (oracle/sqp_port.py) on blocks with a column map (Block.cols, include/sco_b200.h).

A mapped block evaluates each row -- each FK7 instance -- on x[cols_r] with the port's own family functions, as the
reference evaluates a BoundExpr on its Variable's value (expr.py:413-437), and scatters the local Jacobian into an
(m, n) matrix, so the rest of the port runs unchanged.  The finite differences of FK7 and of VM programs without an
analytic gradient run on the local inputs, as Expr._num_grad does on the bound Variable (expr.py:61-69).

`with mapped_port(): ...` makes sqp_port.PortProblem (and so sqp_port.solve and helpers.expand_qp) build mapped
blocks this way; blocks without a map keep the port's own class.
"""
import contextlib

import numpy as np

import families as fam  # oracle/families.py
import numdifftools as nd  # oracle/shims/numdifftools
import sqp_port  # oracle/sqp_port.py

_PortBlockFn = sqp_port._BlockFn


class MappedBlockFn(object):
    def __init__(self, st, blk, row):
        self.blk = blk
        self.n = st.n
        m, cols = blk.m, np.asarray(blk.cols)
        self.val = sqp_port._field(st, blk.val, row, m)[:, None]
        k = cols.shape[1]
        units = []  # (rows, columns, f(xloc) -> (len(rows), 1), grad(xloc) -> (len(rows), k))
        if blk.family == sqp_port.FAM_QUADFORM:
            ntri = k * (k + 1) // 2
            par = sqp_port._field(st, blk.par, row, m * ntri + m * k)
            Pm = fam.unpack_sym(par[:m * ntri].reshape(m, ntri), k)
            a = par[m * ntri:].reshape(m, k)
            for r in range(m):
                P, ar = Pm[r:r + 1], a[r:r + 1]
                units.append(([r], cols[r], lambda x, P=P, ar=ar: fam.quadform_f(x, P, ar),
                              lambda x, P=P, ar=ar: fam.quadform_grad(x, P, ar)))
        elif blk.family == sqp_port.FAM_CIRCLE2D:
            K = blk.ipar[1]
            par = sqp_port._field(st, blk.par, row, 3 * K)
            cen, rad = par[:2 * K].reshape(K, 2), par[2 * K:]
            for r in range(m):
                c, R = cen[r % K:r % K + 1], rad[r % K:r % K + 1]
                units.append(([r], cols[r], lambda x, c=c, R=R: fam.circle_f(x, c, R, 1),
                              lambda x, c=c, R=R: fam.circle_grad(x, c, R, 1)))
        elif blk.family == sqp_port.FAM_FK7:
            for i in range(m // 3):
                units.append(([3 * i, 3 * i + 1, 3 * i + 2], cols[3 * i], fam.fk7_f,
                              lambda x: nd.Jacobian(lambda v: fam.fk7_f(v.reshape(7, 1)).ravel())(x)))
        elif blk.family == sqp_port.FAM_VM:
            n_instr = blk.ipar[2]
            prog = sqp_port._field(st, blk.par, row, m + 2 * n_instr)
            for r in range(m):
                pr = np.concatenate([prog[r:r + 1], prog[m:]])  # row r alone: its offset, every instruction
                f = lambda x, pr=pr: fam.vm_f(x, pr, 1)
                if blk.ipar[3]:
                    g = lambda x, pr=pr: fam.vm_grad(x, pr, 1)
                else:
                    g = lambda x, pr=pr: nd.Jacobian(lambda v: fam.vm_f(v, pr, 1).ravel())(x)
                units.append(([r], cols[r], f, g))
        else:
            raise NotImplementedError(blk.family)
        self.units = units

    def f(self, x):
        out = np.zeros((self.blk.m, 1))
        for rows, c, f, _ in self.units:
            out[rows] = np.asarray(f(x[c]), dtype=float).reshape(len(rows), 1)
        return out

    def grad(self, x):
        J = np.zeros((self.blk.m, self.n))
        for rows, c, _, g in self.units:
            J[np.ix_(rows, c)] = np.asarray(g(x[c]), dtype=float).reshape(len(rows), len(c))
        return J

    violation = _PortBlockFn.violation


def _block_fn(st, blk, row):
    if getattr(blk, "cols", None) is None:
        return _PortBlockFn(st, blk, row)
    return MappedBlockFn(st, blk, row)


@contextlib.contextmanager
def mapped_port():
    sqp_port._BlockFn = _block_fn
    try:
        yield
    finally:
        sqp_port._BlockFn = _PortBlockFn


def solve(st, row, x0, **kw):
    """sqp_port.solve on a structure that may have column maps."""
    with mapped_port():
        return sqp_port.solve(st, row, x0, **kw)
