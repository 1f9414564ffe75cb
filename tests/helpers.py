"""Test helpers: oracle access and expansion of a structured penalty QP into the full
(P, q, A, l, u) the reference hands to OSQP (osqp_utils.py:136-193)."""
import numpy as np
import scipy.sparse as sp

import osqp as osqp_oracle  # oracle/shims/osqp
import sqp_port  # oracle/sqp_port.py

CNT_EQ = 1


def expand_qp(st, row, J_list, b_list, masks, lbx, ubx, pi, kdup, closest_xref=None, use_penalty=True):
    """J_list/b_list/masks: per block dense (m, n) J, (m,) b, (m, n) bool mask."""
    pp = sqp_port.PortProblem(st, row, np.zeros(st.n))
    n = st.n
    ns = st.n_slack if use_penalty else 0
    nq = n + ns
    P = np.zeros((nq, nq))
    q = np.zeros(nq)
    if closest_xref is not None:
        P[:n, :n] = 2.0 * np.eye(n)
        q[:n] = -2.0 * closest_xref
    else:
        P[:n, :n] = 0.5 * (pp.Q + pp.Q.T)
        q[:n] = pp.q
    rows, lo, hi = [], [], []
    if st.m_lin:
        rows.append(sp.hstack([pp.A_lin, sp.csr_matrix((st.m_lin, ns))], format="csr"))
        lo.append(pp.l_lin)
        hi.append(pp.u_lin)
    if use_penalty:
        q[n:] = pi
        so = n
        prow, plo, phi = [], [], []
        for blk, J, b, M in zip(st.blocks, J_list, b_list, masks):
            m = blk.m
            A = np.zeros((m, nq))
            A[:, :n] = J * M
            A[np.arange(m), so + np.arange(m)] = -1.0
            if blk.cnt_type == CNT_EQ:
                A[np.arange(m), so + m + np.arange(m)] = 1.0
                plo.append(-b)
                so += 2 * m
            else:
                plo.append(np.full(m, -np.inf))
                so += m
            phi.append(-b)
            prow.append(sp.csr_matrix(A))
        for _ in range(int(kdup)):
            rows.extend(prow)
            lo.extend(plo)
            hi.extend(phi)
    rows.append(sp.identity(nq, format="csr"))
    lo.append(np.concatenate([lbx, np.zeros(ns)]))
    hi.append(np.concatenate([ubx, np.full(ns, np.inf)]))
    return P, q, sp.vstack(rows, format="csc"), np.concatenate(lo), np.concatenate(hi)


def oracle_qp(P, q, A, l, u, **settings):
    kw = dict(rho=0.1, sigma=5e-10, eps_abs=1e-6, eps_rel=1e-9, adaptive_rho=False, max_iter=100000)
    kw.update(settings)
    m = osqp_oracle.OSQP()
    m.setup(P=sp.csc_matrix(np.triu(P)), q=q, A=A, l=l, u=u, delta=1e-7, polish=False, warm_start=True,
            verbose=False, **kw)
    return m.solve()


def dense_J(st, bi, Jflat_block):
    """stored (m, jw) entries -> dense (m, n)."""
    blk = st.blocks[bi]
    cols = st.jac_cols(bi)
    J = np.zeros((blk.m, st.n))
    vals = np.asarray(Jflat_block).reshape(blk.m, blk.jw)
    for r in range(blk.m):
        J[r, cols[r]] = vals[r]
    return J


def split_J(st, Jflat):
    out = []
    off = 0
    for bi, blk in enumerate(st.blocks):
        cnt = blk.m * blk.jw
        out.append(dense_J(st, bi, Jflat[off:off + cnt]))
        off += cnt
    return out


def split_b(st, bflat):
    """stored (m_nl,) offsets -> per block (m,)."""
    out, r0 = [], 0
    for blk in st.blocks:
        out.append(np.asarray(bflat[r0:r0 + blk.m]))
        r0 += blk.m
    return out


def masks_from_bits(st, bits):
    """Frozen-sparsity mask words of one problem -> per block dense (m, n) bool masks.  `bits`: (m_nl,) or
    (m_nl, words) 32-bit words, bit s of word s // 32 of row r <=> stored slot s of that row participates;
    None switches every slot on."""
    out, r0 = [], 0
    for bi, blk in enumerate(st.blocks):
        M = np.zeros((blk.m, st.n), dtype=bool)
        cols = st.jac_cols(bi)
        for r in range(blk.m):
            for s in range(blk.jw):
                if bits is None:
                    M[r, cols[r, s]] = True
                else:
                    w = np.atleast_1d(np.asarray(bits[r0 + r]).astype(np.uint32))
                    if (int(w[s // 32]) >> (s % 32)) & 1:
                        M[r, cols[r, s]] = True
        out.append(M)
        r0 += blk.m
    return out


def stage_qp(st, row, Jflat, bflat, lbx, ubx, pi, kdup, bits=None):
    """The penalty QP the device stage (Engine.qp_solve) solves for one problem, from the stored J / b and mask words
    it is given, expanded to the (P, q, A, l, u) the reference hands to OSQP."""
    return expand_qp(st, row, split_J(st, Jflat), split_b(st, bflat), masks_from_bits(st, bits), lbx, ubx, pi, kdup)


def _port_job(job):
    name, index, solver, quirks, gen_kw, osqp_kw = job
    from sco_py_b200 import workloads as W
    st, params, x0 = W.GENERATORS[name](1, first=index, **gen_kw)
    r = sqp_port.solve(st, params[0], x0[0], solver=solver, quirks=quirks, osqp_kw=osqp_kw)
    r.pop("trace", None)
    return index, r


def port_solve_many(name, indices, solver, quirks=None, workers=None, gen_kw=None, osqp_kw=None):
    """The oracle port on problems `indices` of config `name` (generator keywords `gen_kw`, e.g. a QCQP's n and m;
    OSQP settings `osqp_kw`), one process per core (the port is single-threaded and a heavy-tailed problem can take
    a minute).  -> {index: result}"""
    import multiprocessing as mp
    import os
    jobs = [(name, int(i), solver, quirks, dict(gen_kw or {}), osqp_kw) for i in indices]
    workers = workers or min(len(jobs), os.cpu_count() or 1)
    if workers <= 1:
        return dict(_port_job(j) for j in jobs)
    with mp.get_context("fork").Pool(workers) as pool:
        return dict(pool.imap_unordered(_port_job, jobs, chunksize=1))
