"""Shared-structure description of a batch of sco_py problems.

A *structure* is everything the B problems of a batch have in common: the
number of variables, the sparsity of the linear constraint rows, the list of
nonlinear constraint blocks (family, row count, Eq/LEq) and where each numeric
field of a problem lives inside its parameter block.  It is the host-side mirror
of `sco_structure_desc` in include/sco_b200.h and is what the structure compiler
(sco_py_b200/batch.py) extracts from a reference-style `Prob`
(sco_py/sco_osqp/prob.py:88-144).

Numeric fields are addressed as (offset, shared): `shared` fields live once in
the shared block, the others once per problem in `params[b, offset:...]`.
"""
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

FAM_QUADFORM = 1   # f_j = 0.5 x'P_j x + a_j'x        (packed-upper P_j, then a_j)
FAM_CIRCLE2D = 2   # f_{t,k} = R_k - ||p_t - c_k||    (centres K x 2, radii K)
FAM_FK7 = 3        # flange position of a 7-link DH chain on x[-7:], FD Jacobian
FAM_VM = 4         # stack program of sco_py_b200.sym, finite-difference Jacobian (dense rows)
# A block with a column map (Block.cols, include/sco_b200.h) reads the inputs of row r from x[cols[r]] instead:
# QUADFORM / VM rows are functions of their cols.shape[1] inputs, CIRCLE2D reads one point per row, FK7 one
# seven-joint instance per three rows.

CNT_LEQ = 0        # LEqExpr  -> hinge penalty, 1 slack per row   (expr.py:353-371)
CNT_EQ = 1         # EqExpr   -> abs penalty,   2 slacks per row  (expr.py:314-332)

MAX_BLOCKS = 16
MAX_GROUPS = 8
MAX_OBJ_BLOCKS = 4
MAX_OBJ_INPUTS = 64


@dataclass
class Field:
    off: int = -1          # offset in doubles; -1 = absent (treated as zeros)
    shared: bool = False


@dataclass
class Block:
    family: int
    cnt_type: int
    m: int
    par: Field                       # family parameters
    val: Field                       # comparison value, m doubles (CompExpr.val)
    ipar: List[int] = field(default_factory=lambda: [0] * 8)
    group_mask: int = 1              # bit g <=> member of constraint group g
    jw: int = 0                      # Jacobian entries stored per row (ELL width)
    cols: Optional[np.ndarray] = None  # (m, n_in) int32 column map, or None: the family's implied columns

    @property
    def n_in(self):
        """Inputs per row of a block with a column map (None without one)."""
        return None if self.cols is None else int(self.cols.shape[1])


@dataclass
class ObjBlock:
    """Non-quadratic objective terms of one input count and derivative mode (include/sco_b200.h
    sco_obj_block_desc): one scalar program row per term, term r reads x[cols[r]]."""
    prog: Field                      # m row offsets, then 2 * n_instr (like a VM constraint block)
    m: int
    n_in: int
    n_instr: int
    flags: int                       # bit 0: forward-mode gradient (SymExpr analytic=True)
    cols: np.ndarray                 # (m, n_in) int32


@dataclass
class Structure:
    n: int
    stride: int                      # doubles per problem block
    Q: Field                         # n*n dense row-major (QuadExpr.Q, not symmetrised)
    q: Field                         # n             (QuadExpr.A)
    c: Field                         # 1             (QuadExpr.b)
    m_lin: int = 0
    lin_rowptr: Optional[np.ndarray] = None   # CSR of the linear rows (shared pattern + values)
    lin_col: Optional[np.ndarray] = None
    lin_val: Optional[np.ndarray] = None
    lin_l: Field = field(default_factory=Field)   # m_lin
    lin_u: Field = field(default_factory=Field)   # m_lin
    blocks: List[Block] = field(default_factory=list)
    n_groups: int = 1                             # 0 = no constraint is in any group (add_cnt_expr(..., group_ids=[]))
    group_overlap: Optional[np.ndarray] = None    # n_groups x n_groups 0/1 (prob.py:139-142)
    shared: Optional[np.ndarray] = None           # shared block
    obj_prog: Field = field(default_factory=Field)  # non-quadratic objective: stack program (sym.py), 1 row
    obj_prog_len: int = 0                           # its instruction count (0 = none)
    obj_prog_flags: int = 0                         # bit 0: gradient by forward-mode differentiation (SymExpr analytic=True)
    qa: Field = field(default_factory=Field)        # n: summed A rows of AffExpr objective terms (quirk C-4 weight in the QP)
    lb0: Field = field(default_factory=Field)       # n: user lower bounds of the scalar variables (closest-point QP)
    ub0: Field = field(default_factory=Field)       # n: user upper bounds
    obj_blocks: List[ObjBlock] = field(default_factory=list)  # objective terms bound to Variables (or obj_prog)

    @property
    def m_nl(self):
        return sum(b.m for b in self.blocks)

    @property
    def n_slack(self):
        return sum(b.m * (2 if b.cnt_type == CNT_EQ else 1) for b in self.blocks)

    def jac_cols(self, bi):
        """Column index of every stored Jacobian slot of block bi: (m, jw) int32."""
        b = self.blocks[bi]
        n = self.n
        if b.cols is not None:
            return np.asarray(b.cols, dtype=np.int32)
        if b.family == FAM_QUADFORM:
            return np.tile(np.arange(n, dtype=np.int32), (b.m, 1))
        if b.family == FAM_CIRCLE2D:
            T, K = b.ipar[0], b.ipar[1]
            t = np.repeat(np.arange(T), K)
            return np.stack([2 * t, 2 * t + 1], axis=1).astype(np.int32)
        if b.family == FAM_FK7:
            return np.tile(np.arange(n - 7, n, dtype=np.int32), (3, 1))
        if b.family == FAM_VM:
            return np.tile(np.arange(n, dtype=np.int32), (b.m, 1))
        raise NotImplementedError(b.family)

    def get(self, f: Field, params_row, size):
        if f.off < 0:
            return np.zeros(size)
        src = self.shared if f.shared else params_row
        return src[f.off:f.off + size]
