"""Structure compiler: reference-style `Prob` objects -> (Structure, params[B, stride], x0[B, n]).

Does on the host, once per batch, what the reference redoes for every QP: the variable ordering of
osqp_utils.optimize (stable sort of the scalar variables by `var_name`, osqp_utils.py:136-143), the
classification of objective terms and constraints of Prob.add_obj_expr / add_cnt_expr
(prob.py:88-144) and the row bounds of linear constraints, [val - b, val - b] for Eq and
[-inf, val - b] for LEq (prob.py:317-346).  The result is the shared-structure description the
kernels run on (structure.py / include/sco_b200.h) plus one parameter row per problem.
"""
import numpy as np

from . import expr as E
from .structure import (CNT_EQ, CNT_LEQ, MAX_BLOCKS, MAX_GROUPS, MAX_OBJ_BLOCKS, MAX_OBJ_INPUTS, Block, Field,
                        ObjBlock, Structure)


class UnsupportedProblem(Exception):
    """The problem uses something the device engine has no kernel for.  There is no CPU fallback."""


class Compiled(object):
    """One problem reduced to numbers, in the QP's variable order."""

    def __init__(self):
        self.ovars = []          # scalar variables, sorted
        self.slots = []          # (Variable, flat index inside it, global column)
        self.x0 = None
        self.Q = self.q = None
        self.qa = None           # summed A rows of AffExpr objective terms (quirk C-4)
        self.lb0 = self.ub0 = None  # user bounds of the scalar variables
        self.c = 0.0
        self.lin_A = self.lin_l = self.lin_u = None
        self.blocks = []         # device blocks: (family expr, cnt_type, val[m], group ids, column map [m, n_in] or None)
        self.obj_blocks = []     # non-quadratic objective: (PackedRows of scalar SymExpr terms, column map [m, n_in])
        self.gids = []


def _columns(var, col_of):
    cols = []
    for ov in var.get_osqp_vars().ravel():
        if id(ov) not in col_of:
            raise UnsupportedProblem("a bound expression uses scalar variable %r that was never added with "
                                     "Prob.add_osqp_var" % (ov.var_name,))
        cols.append(col_of[id(ov)])
    return np.asarray(cols, dtype=np.int64)


class PackedRows(object):
    """Bound QUADFORM or VM constraints of one kind (family, Eq / LEq, groups, inputs per row; for VM also the
    derivative mode) packed into one device block, rows in add order: per-row P and a concatenated (QUADFORM), or
    programs concatenated with re-offset row tables (VM).  Has the attributes of a family expression that
    compile_batch reads."""

    shared_params = False

    def __init__(self, parts):
        f0 = parts[0]
        self.parts = parts
        self.family = f0.family
        self.n = self.jw = f0.n
        self.m = sum(p.m for p in parts)
        if self.family == E.FAM_VM:
            self.n_instr = sum(p.n_instr for p in parts)
            self.ipar = [self.n, self.m, self.n_instr, int(f0.analytic), 0, 0, 0, 0]
        else:
            self.ipar = [self.n, self.m, 0, 0, 0, 0, 0, 0]

    def params(self):
        if self.family == E.FAM_QUADFORM:
            ntri = self.n * (self.n + 1) // 2
            ps = [p.params() for p in self.parts]
            return np.concatenate([q[:p.m * ntri] for p, q in zip(self.parts, ps)] +
                                  [q[p.m * ntri:] for p, q in zip(self.parts, ps)])
        offsets, code, base = [], [], 0
        for p in self.parts:
            offsets.append(p.program[:p.m] + base)
            code.append(p.program[p.m:])
            base += p.n_instr
        return np.concatenate(offsets + code)


def _row_map(fam, cols, n):
    """Column map [m, n_in] of a family constraint bound to the Variable whose columns (in the Variable's own
    order, the order expr.py evaluates it in) are `cols`."""
    name = type(fam).__name__
    if isinstance(fam, E.CircleDistExpr):
        if 2 * fam.T > cols.size:
            raise UnsupportedProblem("CircleDistExpr: %d way-points need %d variables, its Variable has %d"
                                     % (fam.T, 2 * fam.T, cols.size))
        return np.repeat(cols[:2 * fam.T].reshape(fam.T, 2), fam.K, axis=0)
    if fam.n != cols.size:
        raise UnsupportedProblem("a %s over %d variables is bound to a Variable of %d" % (name, fam.n, cols.size))
    if isinstance(fam, E.FK7Expr):
        return np.tile(cols[-7:], (3, 1))
    return np.tile(cols, (fam.m, 1))


def compile_problem(prob):
    cp = Compiled()
    cp.ovars = sorted(prob._osqp_vars, key=lambda v: v.var_name)  # stable, osqp_utils.py:137-142
    n = len(cp.ovars)
    if n == 0:
        raise UnsupportedProblem("the problem has no variables")
    col_of = {id(ov): j for j, ov in enumerate(cp.ovars)}
    x0 = np.full(n, np.nan)
    for var in prob._vars:
        val = var.get_value()
        cols = _columns(var, col_of)
        for k, j in enumerate(cols):
            cp.slots.append((var, k, int(j)))
            if val is not None:
                x0[j] = val.ravel()[k]
    if np.isnan(x0).any():
        raise UnsupportedProblem("every variable needs an initial value (Variable(osqp_vars, value))")
    cp.x0 = x0
    lb = np.array([float(ov.get_lower_bound()) for ov in cp.ovars])
    ub = np.array([float(ov.get_upper_bound()) for ov in cp.ovars])
    if np.isfinite(lb).any() or np.isfinite(ub).any():
        cp.lb0, cp.ub0 = lb, ub
    # ---- objective: QuadExpr terms summed (prob.py:97-103, 348-367)
    cp.Q = np.zeros((n, n))
    cp.q = np.zeros(n)
    for b in prob._quad_obj_exprs:
        cols = _columns(b.var, col_of)
        e = b.expr
        if isinstance(e, E.QuadExpr):
            cp.Q[np.ix_(cols, cols)] += e.Q
            cp.q[cols] += np.asarray(e.A).ravel()
            cp.c += float(np.asarray(e.b).ravel()[0])
        else:
            # AffExpr objective: exact value a'x + b in the merits (expr.py:173-174); in the QP the reference's OSQP
            # backend files the coefficients under the PENALTY terms, re-appended and re-scaled by the penalty
            # coefficient at every update_obj (prob.py:220-221,240-249,424-426; SURVEY.md quirk C-4) -- kept
            # apart here so the device can apply that weight (or weight 1 with sco_settings.aff_obj_quirk = 0)
            A = np.asarray(e.A, dtype=float)
            if cp.qa is None:
                cp.qa = np.zeros(n)
            np.add.at(cp.qa, cols, A.sum(axis=0))  # eval() sums the rows (prob.py:573-574)
            cp.c += float(np.asarray(e.b, dtype=float).sum())
    if prob._nonquad_obj_exprs:  # each term convexified to degree 2 on its own, on the device (expr.py:143-153)
        terms = []
        for b in prob._nonquad_obj_exprs:
            cols = _columns(b.var, col_of)
            e = b.expr
            if not (isinstance(e, E.SymExpr) and e.m == 1):
                raise UnsupportedProblem("a non-quadratic objective term must be a scalar SymExpr (sco_py_b200.sym) "
                                         "bound to a Variable; black-box callables cannot run on the device and there "
                                         "is no CPU fallback")
            if e.n != cols.size:
                raise UnsupportedProblem("an objective SymExpr over %d variables is bound to a Variable of %d"
                                         % (e.n, cols.size))
            uniq, counts = np.unique(cols, return_counts=True)
            if (counts > 1).any():
                raise UnsupportedProblem("an objective term's Variable lists scalar variable %r more than once"
                                         % (cp.ovars[int(uniq[counts > 1][0])].var_name,))
            if cols.size > MAX_OBJ_INPUTS:
                raise UnsupportedProblem("an objective term over %d variables: the limit is %d inputs per term "
                                         "(n_in x n_in Hessian model per term in shared memory, n_in^2 / 2 program "
                                         "evaluations per convexification)" % (cols.size, MAX_OBJ_INPUTS))
            terms.append((e, cols))
        packs = {}  # terms of one input count and derivative mode -> index into cp.obj_blocks
        for e, cols in terms:
            key = (e.n, bool(e.analytic))
            if key not in packs:
                packs[key] = len(cp.obj_blocks)
                cp.obj_blocks.append(([], []))
            cp.obj_blocks[packs[key]][0].append(e)
            cp.obj_blocks[packs[key]][1].append(cols)
        if len(cp.obj_blocks) > MAX_OBJ_BLOCKS:
            raise UnsupportedProblem("%d objective blocks (scalar SymExpr terms of one input count and derivative "
                                     "mode share one): the limit is %d" % (len(cp.obj_blocks), MAX_OBJ_BLOCKS))
        cp.obj_blocks = [(PackedRows(parts), np.vstack(maps)) for parts, maps in cp.obj_blocks]
    # ---- linear constraints
    rows_A, rows_l, rows_u = [], [], []
    for b, kind in prob._lin_cnt_exprs:
        cols = _columns(b.var, col_of)
        A = np.asarray(b.expr.expr.A, dtype=float)
        rhs = (np.asarray(b.expr.val, dtype=float) - np.asarray(b.expr.expr.b, dtype=float)).ravel()
        full = np.zeros((A.shape[0], n))
        np.add.at(full, (slice(None), cols), A)
        rows_A.append(full)
        rows_u.append(rhs)
        rows_l.append(rhs if kind == "eq" else np.full(rhs.shape, -np.inf))
    if rows_A:
        cp.lin_A = np.vstack(rows_A)
        cp.lin_l = np.concatenate(rows_l)
        cp.lin_u = np.concatenate(rows_u)
    # ---- nonlinear constraints -> family blocks
    cp.gids = sorted(prob._cnt_groups.keys())
    packs = {}  # bound QUADFORM / VM constraints of one kind -> index of their device block
    for b in prob._nonlin_cnt_exprs:
        comp = b.expr
        fam = comp.expr
        if not isinstance(fam, E.DeviceFamilyExpr):
            raise UnsupportedProblem(
                "constraint on a black-box Expr: the device engine evaluates closed families only "
                "(QuadFormExpr, CircleDistExpr, FK7Expr in sco_py_b200.expr); there is no CPU fallback")
        cols = _columns(b.var, col_of)
        uniq, counts = np.unique(cols, return_counts=True)
        if (counts > 1).any():
            raise UnsupportedProblem("a constraint's Variable lists scalar variable %r more than once"
                                     % (cp.ovars[int(uniq[counts > 1][0])].var_name,))
        ctype = CNT_EQ if isinstance(comp, E.EqExpr) else CNT_LEQ
        val = np.asarray(comp.val, dtype=float).ravel()
        if val.size != fam.m:
            raise UnsupportedProblem("comparison value has %d entries, the expression %d rows" % (val.size, fam.m))
        gids = [g for g in cp.gids if b in prob._cnt_groups[g]]
        if cols.size == n and np.array_equal(cols, np.arange(n)):
            # bound to every variable in QP order: the implied columns, no map (the structure of earlier versions)
            if getattr(fam, "n", n) != n:
                raise UnsupportedProblem("a %s over %d variables is bound to a problem of %d variables"
                                         % (type(fam).__name__, fam.n, n))
            if isinstance(fam, E.CircleDistExpr) and 2 * fam.T > n:
                raise UnsupportedProblem("CircleDistExpr: %d way-points need %d variables, the problem has %d" % (fam.T, 2 * fam.T, n))
            cp.blocks.append((fam, ctype, val, gids, None))
            continue
        rows = _row_map(fam, cols, n)
        if fam.family not in (E.FAM_QUADFORM, E.FAM_VM):
            cp.blocks.append((fam, ctype, val, gids, rows))
            continue
        key = (fam.family, ctype, tuple(gids), fam.n, getattr(fam, "analytic", None))
        if key not in packs:
            packs[key] = len(cp.blocks)
            cp.blocks.append(([], ctype, [], gids, []))
        parts, _, vals, _, maps = cp.blocks[packs[key]]
        parts.append(fam)
        vals.append(val)
        maps.append(rows)
    for k in packs.values():
        parts, ctype, vals, gids, maps = cp.blocks[k]
        cp.blocks[k] = (PackedRows(parts), ctype, np.concatenate(vals), gids, np.vstack(maps))
    if len(cp.blocks) > MAX_BLOCKS or len(cp.gids) > MAX_GROUPS:
        raise UnsupportedProblem("%d device constraint blocks (bound QUADFORM / VM constraints of one family, Eq / "
                                 "LEq kind, group set and input count share one) and %d groups: the limits are %d "
                                 "and %d" % (len(cp.blocks), len(cp.gids), MAX_BLOCKS, MAX_GROUPS))
    return cp


def _csr(A):
    rowptr, col, val = [0], [], []
    for r in range(A.shape[0]):
        (idx,) = np.nonzero(A[r])
        col.extend(idx.tolist())
        val.extend(A[r, idx].tolist())
        rowptr.append(len(col))
    return np.asarray(rowptr, np.int32), np.asarray(col, np.int32), np.asarray(val, np.float64)


def group_key(cp):
    """What two compiled problems must have in common to go into one launch."""
    return (cp.x0.size, cp.qa is not None, cp.lb0 is not None,
            None if cp.lin_A is None else (cp.lin_A.shape, cp.lin_A.tobytes()), tuple(cp.gids),
            tuple((b[0].family, b[0].m, b[1], tuple(b[0].ipar), tuple(b[3])) +
                  (() if b[4] is None else (b[4].shape, b[4].tobytes())) for b in cp.blocks),
            tuple((pk.m, pk.n, pk.n_instr, int(pk.ipar[3]), cols.tobytes()) for pk, cols in cp.obj_blocks))


def compile_batch(probs, compiled=None):
    """-> (Structure, params[B, stride], x0[B, n], compiled list).  All problems must share the
    structure: variable count, linear-row coefficients, constraint block families / sizes / groups."""
    cps = compiled if compiled is not None else [compile_problem(p) for p in probs]
    c0 = cps[0]
    n = c0.x0.size
    B = len(cps)
    key0 = group_key(c0)
    for i, c in enumerate(cps[1:], 1):
        if group_key(c) != key0:
            raise UnsupportedProblem("problem %d of the batch does not share the structure of problem 0" % i)
    shared_parts, shared_off = [], 0

    def shared_field(arr):
        nonlocal shared_off
        f = Field(shared_off, True)
        shared_parts.append(np.asarray(arr, dtype=float).ravel())
        shared_off += shared_parts[-1].size
        return f

    off = 0

    def own_field(size):
        nonlocal off
        f = Field(off, False)
        off += size
        return f

    fills = []  # (field, getter(compiled) -> flat array)
    q_shared = all(np.array_equal(c.Q, c0.Q) for c in cps[1:]) and B > 1
    if not c0.Q.any() and all(not c.Q.any() for c in cps):
        Qf = Field(-1, False)
    elif q_shared:
        Qf = shared_field(c0.Q)
    else:
        Qf = own_field(n * n)
        fills.append((Qf, lambda c: c.Q.ravel()))
    qf = own_field(n)
    fills.append((qf, lambda c: c.q))
    cf = own_field(1)
    fills.append((cf, lambda c: np.array([c.c])))
    kw = {}
    if c0.qa is not None:
        qaf = own_field(n)
        fills.append((qaf, lambda c: c.qa))
        kw["qa"] = qaf
    if c0.lb0 is not None:
        lf0, uf0 = own_field(n), own_field(n)
        fills.append((lf0, lambda c: c.lb0))
        fills.append((uf0, lambda c: c.ub0))
        kw.update(lb0=lf0, ub0=uf0)
    if c0.lin_A is not None:
        m_lin = c0.lin_A.shape[0]
        rp, ci, cv = _csr(c0.lin_A)
        lf, uf = own_field(m_lin), own_field(m_lin)
        fills.append((lf, lambda c: c.lin_l))
        fills.append((uf, lambda c: c.lin_u))
        kw.update(m_lin=m_lin, lin_rowptr=rp, lin_col=ci, lin_val=cv, lin_l=lf, lin_u=uf)
    obj_blocks = []
    for oi, (pk, cols) in enumerate(c0.obj_blocks):
        p0 = pk.params()
        if B > 1 and all(np.array_equal(c.obj_blocks[oi][0].params(), p0) for c in cps[1:]):
            of = shared_field(p0)
        else:
            of = own_field(p0.size)
            fills.append((of, lambda c, oi=oi: c.obj_blocks[oi][0].params()))
        obj_blocks.append(ObjBlock(of, pk.m, pk.n, pk.n_instr, int(pk.ipar[3]),
                                   np.ascontiguousarray(cols, dtype=np.int32)))
    if len(obj_blocks) == 1 and obj_blocks[0].m == 1 and np.array_equal(obj_blocks[0].cols[0], np.arange(n)):
        # one term over every variable in QP order: the obj_prog structure of earlier versions
        ob = obj_blocks.pop()
        kw.update(obj_prog=ob.prog, obj_prog_len=ob.n_instr, obj_prog_flags=ob.flags)
    blocks = []
    for bi, (fam, ctype, val, gids, cols) in enumerate(c0.blocks):
        p0 = fam.params()
        if fam.shared_params or (B > 1 and all(np.array_equal(c.blocks[bi][0].params(), p0) for c in cps[1:])):
            pf = shared_field(p0)
        else:
            pf = own_field(p0.size)
            fills.append((pf, lambda c, bi=bi: c.blocks[bi][0].params()))
        vf = own_field(fam.m)
        fills.append((vf, lambda c, bi=bi: c.blocks[bi][2]))
        mask = 0
        for g in gids:
            mask |= 1 << c0.gids.index(g)
        # group_ids=[] puts a constraint in NO group (prob.py:135-142): mask 0, and a problem without any group
        # has n_groups = 0 -- the reference then skips the per-group test (solver.py:209)
        blocks.append(Block(fam.family, ctype, fam.m, pf, vf, ipar=list(fam.ipar), group_mask=mask, jw=fam.jw,
                            cols=None if cols is None else np.ascontiguousarray(cols, dtype=np.int32)))
    ng = len(c0.gids)
    overlap = np.zeros((ng, ng), dtype=np.int32)
    ov = getattr(probs[0], "_cnt_groups_overlap", {}) if probs else {}
    for g, others in ov.items():
        for o in others:
            if g in c0.gids and o in c0.gids:
                overlap[c0.gids.index(g), c0.gids.index(o)] = 1
    st = Structure(n=n, stride=max(off, 1), Q=Qf, q=qf, c=cf, blocks=blocks, n_groups=ng,
                   group_overlap=overlap if ng > 1 else None,
                   shared=np.concatenate(shared_parts) if shared_parts else None, obj_blocks=obj_blocks, **kw)
    params = np.zeros((B, st.stride))
    x0 = np.empty((B, n))
    for i, c in enumerate(cps):
        x0[i] = c.x0
        for f, get in fills:
            a = np.asarray(get(c), dtype=float).ravel()
            params[i, f.off:f.off + a.size] = a
    return st, params, x0, cps


def signature(st):
    """Hashable identity of a structure (engines are cached per signature)."""
    def fld(f):
        return (f.off, bool(f.shared))
    lin = None
    if st.m_lin:
        lin = (st.lin_rowptr.tobytes(), st.lin_col.tobytes(), st.lin_val.tobytes(), fld(st.lin_l), fld(st.lin_u))
    sig = (st.n, st.stride, fld(st.Q), fld(st.q), fld(st.c), fld(st.qa), fld(st.lb0), fld(st.ub0), fld(st.obj_prog),
            st.obj_prog_len, st.obj_prog_flags, st.m_lin, lin, st.n_groups,
            None if st.group_overlap is None else st.group_overlap.tobytes(),
            None if st.shared is None else st.shared.tobytes(),
            tuple((b.family, b.cnt_type, b.m, fld(b.par), fld(b.val), tuple(b.ipar), b.group_mask, b.jw) +
                  (() if b.cols is None else (b.cols.shape, np.ascontiguousarray(b.cols, dtype=np.int32).tobytes()))
                  for b in st.blocks))
    if st.obj_blocks:  # appended only when present: the signatures of other structures stay as they were
        sig += (tuple((fld(o.prog), o.m, o.n_in, o.n_instr, o.flags,
                       np.ascontiguousarray(o.cols, dtype=np.int32).tobytes()) for o in st.obj_blocks),)
    return sig


def scatter_solution(cp, x):
    """Writes a solution (QP order) into the problem's scalar variables and Variables, in place, the
    way osqp_utils.update_osqp_vars + Variable.update deliver results (osqp_utils.py:224-229,
    variable.py:47-60)."""
    for j, ov in enumerate(cp.ovars):
        ov.val = float(x[j])
    touched = {}
    for var, k, j in cp.slots:
        if id(var) not in touched:
            touched[id(var)] = (var, np.zeros(var.get_osqp_vars().shape))
        touched[id(var)][1].ravel()[k] = x[j]
    for var, val in touched.values():
        var._value = val
