// sco_abi.cu -- host side of the C ABI declared in include/sco_b200.h: the structure compiler
// (index arrays, shared-memory layout, team size) and the launch wrappers.  The kernels live in
// sco_kernels.cuh and are instantiated per team size by sco_team.cu.
// Build: python -m sco_py_b200.build  (nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3).
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <memory>
#include <vector>

#include "sco_b200.h"
#include "sco_device.cuh"
#include "sco_launch.h"

// ------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess)                                                                      \
      return fail(SCO_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                                    \
  } while (0)

extern "C" const char *sco_last_error(void) { return g_err; }

// ------------------------------------------------------------------------------------ handle
struct sco_handle {
  int device = 0;
  int team = 32;
  const TeamOps *ops = nullptr;    // solve / qp (dense variant when the structure qualifies)
  const TeamOps *gen_ops = nullptr; // convexify / merit (generic team kernels)
  int carve_ops = 100, carve_gen = 100;  // shared-memory carve-out of this handle (kernel attributes are shared)
  int sm_count = 0;
  int occupancy = 1;
  size_t smem_bytes = 0;
  DevStruct S;
  std::vector<void *> dev_allocs;
  // Launch slots: every launch owns a work-queue counter and a Jacobian scratch area until it ends,
  // so launches of one handle may be in flight on several streams at once (batches pipelined over
  // streams hide the tail of a launch, where a few long problems keep a handful of SMs busy).
  static const int NSLOT = SCO_LAUNCH_SLOTS;
  double *Jscr[NSLOT] = {};
  size_t Jscr_ctas = 0;
  unsigned long long *counter = nullptr;  // NSLOT counters
  int *order_err = nullptr;               // NSLOT flags (sco_solve_batch_ordered)
  unsigned *seen[NSLOT] = {};             // bitmap of the order check, grow-only
  long long seen_cap[NSLOT] = {};
  cudaEvent_t slot_done[NSLOT] = {};
  unsigned next_slot = 0;
  // host-entry staging buffers, one set per staging slot (grow-only)
  static const int NSTG = SCO_STAGING_SETS;
  struct Staging {
    double *params = nullptr, *x0 = nullptr, *x = nullptr, *merit = nullptr, *obj = nullptr, *vio = nullptr;
    int *verdict = nullptr, *stats = nullptr, *nonconv = nullptr;
    long long cap_B = 0;
    cudaEvent_t done = nullptr;
  } stg[NSTG];
  unsigned next_stg = 0;
};

template <typename T>
static int upload(sco_handle *h, const std::vector<T> &v, const T **out) {
  T *d = nullptr;
  size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
  CUDA_TRY(cudaMalloc(&d, bytes));
  h->dev_allocs.push_back(d);
  if (!v.empty()) CUDA_TRY(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  *out = d;
  return 0;
}

static DevField cvt(const sco_field &f) {
  DevField d;
  d.off = f.off;
  d.shared = f.shared;
  d.pad_ = 0;
  return d;
}

static void build_layout(DevStruct &S, int team) {
  Layout &L = S.L;
  // dense kinds: the two-warp solve owns a compile-time region at the start of dynamic shared memory
  static const int dense_words[5] = {0, DenseL<8, 6>::total, DenseL<12, 16>::total, DenseL<20, 30>::total,
                                     DenseL<32, 32>::total};
  int off = dense_words[S.dense_kind];
  auto take = [&](int cnt) {
    int o = off;
    off += (cnt + 1) & ~1;
    return o;
  };
  const int n = S.n, ml = S.m_lin, mp = S.m_nl, sl = S.nsl * S.m_nl;
  L.Js = take(S.sjnnz); L.S = take(S.sws ? 0 : n * n); L.Als = take(S.nnz_lin);
  L.x = take(n); L.xt = take(n); L.xt2 = take(n + 4); L.qh = take(n); L.D = take(n); L.bx = take(n);  // xt2, wp: + 4 = zero padding
  L.rb = take(n); L.lb = take(n); L.ub = take(n); L.zb = take(n); L.yb = take(n); L.Eb = take(n);
  L.dxv = take(n); L.dyb = take(n); L.xs = take(n);
  L.El = take(ml); L.rl = take(ml); L.ll = take(ml); L.ul = take(ml); L.zl = take(ml); L.yl = take(ml);
  L.wl = take(ml); L.dyl = take(ml);
  L.Ep = take(mp); L.rp = take(mp); L.lp = take(mp); L.up = take(mp); L.zp = take(mp); L.yp = take(mp);
  L.wp = take(mp + 4); L.bb = take(mp); L.fv = take(mp); L.dyp = take(mp);
  L.s = take(sl); L.Ds = take(sl); L.sl = take(sl); L.bs = take(sl); L.zs = take(sl); L.ys = take(sl);
  L.Es = take(sl); L.gs = take(sl); L.hs = take(sl); L.rs = take(sl); L.dss = take(sl); L.dys = take(sl);
  L.Minv = take(3 * mp);
  L.red = take((std::max(team / 32, 8) + 1) * 16);  // one 16-double slot per warp + one for the combined results
  L.msk = take((mp * S.mw + 1) / 2);
  L.stage = take(std::max((team / 32) * S.stage_per_warp, 100));
  // objective terms: the eigenvalue shift runs one term per warp, on at most 4,096 doubles of scratch in all
  S.nwj = S.n_ob ? std::max(1, std::min(std::min(S.n_terms, team / 32), 4096 / (S.n_in_max * S.n_in_max))) : 0;
  int ot_len = 0;
  for (int b = 0; b < S.n_ob; b++) ot_len += S.ob[b].m * (S.ob[b].n_in * (S.ob[b].n_in + 1) / 2 + S.ob[b].n_in + 1);
  L.ot = take(ot_len); L.jac = take(S.nwj * S.n_in_max * S.n_in_max);
  L.Hv = take(S.n_ob ? S.nnz_p : 0); L.gq = take(S.n_ob ? n : 0); L.oc = take(S.n_ob ? 1 : 0);
  L.ps = take(4 * n);
  L.total = off;
}

extern "C" void sco_default_settings(sco_settings *s) {
  memset(s, 0, sizeof(*s));
  s->improve_ratio_threshold = 0.25;  // solver.py:17-28
  s->min_trust_region_size = 1e-4;
  s->min_approx_improve = 1e-8;
  s->trust_shrink_ratio = 0.1;
  s->trust_expand_ratio = 1.5;
  s->cnt_tolerance = 1e-4;
  s->merit_coeff_increase_ratio = 10.0;
  s->initial_trust_region_size = 1.0;
  s->initial_penalty_coeff = 1e3;
  s->max_merit_coeff_increases = 1;
  s->max_sqp_iters = 100000;
  s->osqp_eps_abs = 1e-6;  // osqp_utils.py:10-15
  s->osqp_eps_rel = 1e-9;
  s->osqp_rho = 0.1;
  s->osqp_sigma = 5e-10;
  s->osqp_alpha = 1.6;  // OSQP defaults, SURVEY.md Appendix B
  s->osqp_eps_prim_inf = 1e-4;
  s->osqp_eps_dual_inf = 1e-4;
  s->osqp_max_iter = 100000;
  s->osqp_scaling = 10;
  s->osqp_check_termination = 25;
  s->osqp_adaptive_rho = 0;
  s->osqp_adaptive_rho_interval = 0;
  s->compound_penalty = 1;
  s->freeze_sparsity = 1;
  s->duplicate_rows = 1;
  s->threads_per_problem = 0;
  s->force_generic = 0;
  s->aff_obj_quirk = 1;
  s->warm_start = 0;
}

static DevSettings to_dev(const sco_settings *s) {
  DevSettings d;
  d.improve_ratio_threshold = s->improve_ratio_threshold;
  d.min_trust_region_size = s->min_trust_region_size;
  d.min_approx_improve = s->min_approx_improve;
  d.trust_shrink_ratio = s->trust_shrink_ratio;
  d.trust_expand_ratio = s->trust_expand_ratio;
  d.cnt_tolerance = s->cnt_tolerance;
  d.merit_coeff_increase_ratio = s->merit_coeff_increase_ratio;
  d.initial_trust_region_size = s->initial_trust_region_size;
  d.initial_penalty_coeff = s->initial_penalty_coeff;
  d.max_merit_coeff_increases = s->max_merit_coeff_increases;
  d.max_sqp_iters = s->max_sqp_iters;
  d.eps_abs = s->osqp_eps_abs;
  d.eps_rel = s->osqp_eps_rel;
  d.rho = s->osqp_rho;
  d.sigma = s->osqp_sigma;
  d.alpha = s->osqp_alpha;
  d.eps_prim_inf = s->osqp_eps_prim_inf;
  d.eps_dual_inf = s->osqp_eps_dual_inf;
  d.max_iter = s->osqp_max_iter;
  d.scaling = s->osqp_scaling;
  d.check_termination = s->osqp_check_termination;
  d.adaptive_rho = s->osqp_adaptive_rho;
  d.adaptive_rho_interval = s->osqp_adaptive_rho_interval;
  d.compound_penalty = s->compound_penalty;
  d.freeze_sparsity = s->freeze_sparsity;
  d.duplicate_rows = s->duplicate_rows;
  d.force_generic = s->force_generic;
  d.aff_obj_quirk = s->aff_obj_quirk;
  d.warm_start = s->warm_start;
  return d;
}

// ------------------------------------------------------------------------------------ structure compiler
// sco_create runs in stages: check_desc refuses a bad descriptor, build_index builds the index arrays on the host,
// choose_paths picks the ADMM loop, team and layout, setup_device uploads and configures.  Nothing is allocated on
// the device before the last stage.

static bool has_obj_prog(const sco_structure_desc *desc) { return desc->obj_prog_len > 0 && desc->obj_prog.off >= 0; }

// A column map: m rows of n_in indices in [0, n), none repeated within a row.  The messages name row r of block blk
// "<what> <blk> <row> <r>": "block 2 row 5", "objective block 0 term 3".
static int check_map(const int32_t *cols, int m, int n_in, int n, const char *what, int blk, const char *row) {
  for (int r = 0; r < m; r++) {
    const int32_t *c = cols + (size_t)r * n_in;
    for (int i = 0; i < n_in; i++) {
      if (c[i] < 0 || c[i] >= n) return fail(SCO_ERR_ARG, "%s %d %s %d: column %d outside [0, %d)", what, blk, row, r, c[i], n);
      if (std::find(c, c + i, c[i]) != c + i) return fail(SCO_ERR_ARG, "%s %d %s %d: column %d repeats", what, blk, row, r, c[i]);
    }
  }
  return 0;
}

// Every refusal of a descriptor, before anything is built or allocated.
static int check_desc(const sco_structure_desc *desc) {
  if (desc->n <= 0 || desc->n_blocks < 0 || desc->n_blocks > SCO_MAX_BLOCKS)
    return fail(SCO_ERR_ARG, "bad n / n_blocks");
  // n_groups = 0: no constraint belongs to a group -- the reference then skips the per-group test (solver.py:209)
  if (desc->n_groups < 0 || desc->n_groups > SCO_MAX_GROUPS) return fail(SCO_ERR_ARG, "bad n_groups");
  if (desc->m_lin < 0 || desc->stride <= 0 || desc->shared_len < 0) return fail(SCO_ERR_ARG, "negative m_lin / stride / shared_len");
  if (desc->shared_len > 0 && !desc->shared) return fail(SCO_ERR_ARG, "shared_len > 0 but shared is null");
  // every field must lie inside the block it lives in (out-of-range offsets would be device reads out of bounds)
  const int n = desc->n;
  auto field_ok = [&](const sco_field &f, long long len) {
    if (f.off < 0) return true;
    const long long lim = f.shared ? (long long)desc->shared_len : (long long)desc->stride;
    return f.off + len <= lim;
  };
  static const char outside[] = "a field lies outside its parameter block (offset + length > stride / shared_len)";
  if (desc->n_obj_blocks < 0 || desc->n_obj_blocks > SCO_MAX_OBJ_BLOCKS)
    return fail(SCO_ERR_ARG, "n_obj_blocks = %d outside [0, %d]", desc->n_obj_blocks, SCO_MAX_OBJ_BLOCKS);
  if (desc->obj_prog_len > 0 && desc->n_obj_blocks > 0)
    return fail(SCO_ERR_ARG, "obj_prog and objective blocks are both set: a structure has one or the other");
  if (!(field_ok(desc->Q, (long long)n * n) && field_ok(desc->q, n) && field_ok(desc->c, 1) &&
        field_ok(desc->lin_l, desc->m_lin) && field_ok(desc->lin_u, desc->m_lin) && field_ok(desc->qa, n) &&
        field_ok(desc->lb0, n) && field_ok(desc->ub0, n) &&
        (desc->obj_prog_len <= 0 || field_ok(desc->obj_prog, 1 + 2LL * desc->obj_prog_len))))
    return fail(SCO_ERR_ARG, "%s", outside);
  for (int oi = 0; oi < desc->n_obj_blocks; oi++) {
    const sco_obj_block_desc &o = desc->obj_blocks[oi];
    if (o.m <= 0 || o.n_instr <= 0) return fail(SCO_ERR_ARG, "objective block %d: m and n_instr must be positive", oi);
    if (o.n_in < 1 || o.n_in > 64)
      return fail(SCO_ERR_ARG, "objective block %d: n_in = %d outside [1, 64] (inputs per term)", oi, o.n_in);
    if (!o.cols) return fail(SCO_ERR_ARG, "objective block %d: cols is null", oi);
    if (int rc = check_map(o.cols, o.m, o.n_in, n, "objective block", oi, "term")) return rc;
    if (o.prog.off < 0) return fail(SCO_ERR_ARG, "objective block %d: the program is missing", oi);
    if (!field_ok(o.prog, o.m + 2LL * o.n_instr))
      return fail(SCO_ERR_ARG, "objective block %d: the program field lies outside its parameter block", oi);
  }
  for (int bi = 0; bi < desc->n_blocks; bi++) {
    const sco_block_desc &b = desc->blocks[bi];
    if (b.m <= 0) return fail(SCO_ERR_ARG, "block %d: m must be positive", bi);
    if (desc->n_groups < 32 && (b.group_mask >> desc->n_groups) != 0)
      return fail(SCO_ERR_ARG, "block %d: group_mask names a group >= n_groups", bi);
    const bool mapped = b.cols != nullptr;
    if (mapped) {
      const int want = b.family == SCO_FAM_CIRCLE2D ? 2 : b.family == SCO_FAM_FK7 ? 7 : b.n_in;
      if (b.n_in <= 0 || b.n_in > n || b.n_in != want)
        return fail(SCO_ERR_ARG, "block %d: n_in = %d is wrong for family %d (CIRCLE2D 2, FK7 7, else 1..n)", bi, b.n_in, b.family);
      if (b.family == SCO_FAM_FK7 && b.m % 3 != 0) return fail(SCO_ERR_ARG, "block %d: FK7 with a map needs m %% 3 == 0", bi);
      if (int rc = check_map(b.cols, b.m, b.n_in, n, "block", bi, "row")) return rc;
      for (int r = 0; b.family == SCO_FAM_FK7 && r < b.m; r++)  // the three rows of an instance are one position
        if (r % 3 != 0 && memcmp(b.cols + (size_t)r * 7, b.cols + (size_t)(r - r % 3) * 7, 7 * sizeof(int32_t)) != 0)
          return fail(SCO_ERR_ARG, "block %d: rows of FK7 instance %d have different maps", bi, r / 3);
    }
    const long long nb = mapped ? b.n_in : n;  // inputs of a row
    long long plen = 0;
    if (b.family == SCO_FAM_QUADFORM) plen = (long long)b.m * (nb * (nb + 1) / 2 + nb);
    else if (b.family == SCO_FAM_CIRCLE2D) plen = 3LL * b.ipar[1];
    else if (b.family == SCO_FAM_FK7) plen = 30;
    else if (b.family == SCO_FAM_VM) plen = b.m + 2LL * b.ipar[2];
    else return fail(SCO_ERR_UNSUPPORTED, "unknown constraint family %d", b.family);
    if (b.par.off < 0) return fail(SCO_ERR_ARG, "block %d: parameters are missing", bi);
    if (!field_ok(b.par, plen) || !field_ok(b.val, b.m)) return fail(SCO_ERR_ARG, "%s", outside);
    if (b.family == SCO_FAM_CIRCLE2D && (b.ipar[1] <= 0 || b.ipar[0] * b.ipar[1] != b.m || (!mapped && 2 * b.ipar[0] > n)))
      return fail(SCO_ERR_ARG, "CIRCLE2D: m != T*K or 2T > n");
    if (b.family == SCO_FAM_FK7 && ((!mapped && b.m != 3) || n < 7))
      return fail(SCO_ERR_ARG, "FK7: m must be 3 (without a map) and n >= 7");
    if (b.family == SCO_FAM_VM && (b.ipar[0] != nb || b.ipar[1] != b.m || b.ipar[2] <= 0))
      return fail(SCO_ERR_ARG, "VM: ipar must be {n (n_in with a map), m, instructions}");
  }
  if (desc->m_lin > 0 && (desc->lin_l.off < 0 || desc->lin_u.off < 0)) return fail(SCO_ERR_ARG, "m_lin > 0 needs lin_l and lin_u");
  if (has_obj_prog(desc) && n > 64) return fail(SCO_ERR_UNSUPPORTED, "non-quadratic objectives are limited to 64 variables");
  if (desc->m_lin > 0) {
    if (!desc->lin_rowptr || !desc->lin_col || !desc->lin_val) return fail(SCO_ERR_ARG, "m_lin > 0 but CSR arrays are null");
    for (int r = 0; r < desc->m_lin; r++)
      for (int p = desc->lin_rowptr[r]; p < desc->lin_rowptr[r + 1]; p++)
        if (desc->lin_col[p] < 0 || desc->lin_col[p] >= n) return fail(SCO_ERR_ARG, "linear row column out of range");
  }
  return 0;
}

// What sco_create hands to the device, built on the host: DevStruct's sizes and tables, the index arrays, the team
// and the shared memory per problem.  The device sums along pc_*, lin_c*, hv_src and gq_src in list order, so the
// order of every list is part of the results: rows ascending, and within a row its stored entries ascending.
struct HostStruct {
  DevStruct S;  // device pointers unset
  std::vector<int> row_goff, row_soff, row_w, row_eq, row_gmask, jcol, pc_ptr, pc_e, pc_r;  // penalty rows
  std::vector<int> lrp, lcol, lin_w, lcptr, lcentry, lcrow;                                 // linear rows
  std::vector<double> lval, shared;
  std::vector<int> ob_cols, P_cptr, P_row, hv_ptr, hv_src, gq_ptr, gq_src;                  // objective
  bool any_map = false;
  int team = 0; size_t smem_bytes = 0;  // choose_paths
};

// lists[i] -> ptr (ptr[i + 1] - ptr[i] = lists[i].size()) and src, the lists concatenated in order
static void flatten(const std::vector<std::vector<int>> &lists, std::vector<int> &ptr, std::vector<int> &src) {
  ptr.assign(lists.size() + 1, 0);
  for (size_t i = 0; i < lists.size(); i++) {
    ptr[i + 1] = ptr[i] + (int)lists[i].size();
    src.insert(src.end(), lists[i].begin(), lists[i].end());
  }
}

// CSC over the n user variables of a row pattern whose row r holds w[r] entries, entry e0[r] + k in column
// col[c0[r] + k]: per column its (entry, row) pairs, rows ascending and a row's entries ascending
static void to_csc(int n, const std::vector<int> &col, const std::vector<int> &c0, const std::vector<int> &e0,
                   const std::vector<int> &w, std::vector<int> &ptr, std::vector<int> &ent, std::vector<int> &row) {
  std::vector<std::vector<int>> ents(n), rows(n);
  for (size_t r = 0; r < w.size(); r++)
    for (int k = 0; k < w[r]; k++) {
      ents[col[c0[r] + k]].push_back(e0[r] + k);
      rows[col[c0[r] + k]].push_back((int)r);
    }
  flatten(ents, ptr, ent);
  flatten(rows, ptr, row);
}

// max - min of the w columns col[c0 ..]: the band a row adds to S = P + A'RA (0 for an empty row)
static int col_span(const std::vector<int> &col, int c0, int w) {
  if (w <= 0) return 0;
  const auto mm = std::minmax_element(col.begin() + c0, col.begin() + c0 + w);
  return *mm.second - *mm.first;
}

static void build_index(const sco_structure_desc *desc, HostStruct &ix) {
  DevStruct &S = ix.S;
  memset(&S, 0, sizeof(S));
  const int n = desc->n;
  S.n = n; S.m_lin = desc->m_lin; S.n_blocks = desc->n_blocks; S.n_groups = desc->n_groups; S.stride = desc->stride;
  S.Q = cvt(desc->Q); S.q = cvt(desc->q); S.c = cvt(desc->c);
  S.lin_l = cvt(desc->lin_l); S.lin_u = cvt(desc->lin_u);
  S.qa = cvt(desc->qa); S.lb0 = cvt(desc->lb0); S.ub0 = cvt(desc->ub0);
  // objective terms: the one-term obj_prog becomes a block of one term over all n variables in QP order
  std::vector<int32_t> all(n);
  for (int j = 0; j < n; j++) all[j] = j;
  const sco_obj_block_desc prog = {1, n, desc->obj_prog_len, desc->obj_prog_flags, desc->obj_prog, all.data()};
  std::vector<int> pidx((size_t)n * n, -1);  // (i, j) -> entry of the pattern of P (below)
  S.n_ob = has_obj_prog(desc) ? 1 : desc->n_obj_blocks;
  for (int oi = 0, toff = 0; oi < S.n_ob; oi++) {
    const sco_obj_block_desc &o = has_obj_prog(desc) ? prog : desc->obj_blocks[oi];
    DevObjBlock &d = S.ob[oi];
    d.m = o.m; d.n_in = o.n_in; d.flags = o.flags; d.prog = cvt(o.prog);
    d.t0 = S.n_terms; d.toff = toff; d.coff = (int)ix.ob_cols.size();
    ix.ob_cols.insert(ix.ob_cols.end(), o.cols, o.cols + (size_t)o.m * o.n_in);
    for (int r = 0; r < o.m; r++)  // the term's n_in x n_in block is in the pattern of P
      for (int a = 0; a < o.n_in; a++)
        for (int b = 0; b < o.n_in; b++) pidx[(size_t)o.cols[r * o.n_in + a] * n + o.cols[r * o.n_in + b]] = 0;
    S.n_terms += d.m;
    toff += d.m * (d.n_in * (d.n_in + 1) / 2 + d.n_in + 1);
    S.n_in_max = std::max(S.n_in_max, d.n_in);
  }
  for (int g = 0; g < desc->n_groups; g++) {
    int bits = 0;
    if (desc->group_overlap)
      for (int g2 = 0; g2 < desc->n_groups; g2++)
        if (desc->group_overlap[g * desc->n_groups + g2]) bits |= 1 << g2;
    S.overlap[g] = bits;
  }
  // ---- penalty rows
  int m_nl = 0, jnnz = 0, sj = 0, n_slack = 0, max_stage = 0, max_jw = 1;
  for (int bi = 0; bi < desc->n_blocks; bi++) {
    const sco_block_desc &b = desc->blocks[bi];
    DevBlock &d = S.blocks[bi];
    d.family = b.family; d.cnt_type = b.cnt_type; d.m = b.m; d.group_mask = b.group_mask;
    d.row0 = m_nl; d.joff = jnnz;
    memcpy(d.ipar, b.ipar, sizeof(d.ipar));
    d.par = cvt(b.par); d.val = cvt(b.val);
    const bool mapped = b.cols != nullptr;
    const int nb = mapped ? b.n_in : n;  // inputs of a row
    ix.any_map = ix.any_map || mapped;
    d.n_in = mapped ? b.n_in : 0;
    const int jw = b.family == SCO_FAM_CIRCLE2D ? 2 : b.family == SCO_FAM_FK7 ? 7 : nb;  // QUADFORM, VM: every input
    if (b.family == SCO_FAM_QUADFORM)  // a map's inputs are gathered into the staging buffer behind P_r
      max_stage = std::max(max_stage, nb * (nb + 1) / 2 + (mapped ? nb : 0));
    if (b.family == SCO_FAM_FK7 && mapped)  // 98 doubles of finite differences + the gathered joints
      max_stage = std::max(max_stage, 106);
    max_jw = std::max(max_jw, jw);
    d.jw = jw;
    const int ldj = (jw % 2 == 0) ? jw + 1 : jw;
    for (int r = 0; r < b.m; r++) {
      ix.row_goff.push_back(jnnz + r * jw);
      ix.row_soff.push_back(sj + r * ldj);
      ix.row_w.push_back(jw);
      ix.row_eq.push_back(b.cnt_type == SCO_CNT_EQ ? 1 : 0);
      ix.row_gmask.push_back(b.group_mask);
      for (int k = 0; k < jw; k++) {
        int col = 0;
        if (mapped) col = b.cols[(size_t)r * b.n_in + k];
        else if (b.family == SCO_FAM_QUADFORM || b.family == SCO_FAM_VM) col = k;
        else if (b.family == SCO_FAM_CIRCLE2D) col = 2 * (r / b.ipar[1]) + k;
        else col = n - 7 + k;
        ix.jcol.push_back(col);
      }
    }
    n_slack += b.m * (b.cnt_type == SCO_CNT_EQ ? 2 : 1);
    m_nl += b.m;
    jnnz += b.m * jw;
    sj += b.m * ldj;
  }
  S.m_nl = m_nl; S.jnnz = jnnz; S.sjnnz = sj; S.n_slack = n_slack; S.n_q = n + n_slack;
  S.nsl = n_slack > m_nl ? 2 : 1;  // an equality row has two slacks
  S.stage_per_warp = (max_stage + 1) & ~1;
  S.mw = (max_jw + 31) / 32;
  to_csc(n, ix.jcol, ix.row_goff, ix.row_soff, ix.row_w, ix.pc_ptr, ix.pc_e, ix.pc_r);
  // ---- linear rows
  ix.lrp.assign(1, 0);  // without linear rows the CSR arrays may be null
  if (desc->m_lin > 0) ix.lrp.assign(desc->lin_rowptr, desc->lin_rowptr + desc->m_lin + 1);
  S.nnz_lin = ix.lrp[desc->m_lin];
  ix.lcol.assign(desc->lin_col, desc->lin_col + S.nnz_lin);
  ix.lval.assign(desc->lin_val, desc->lin_val + S.nnz_lin);
  for (int r = 0; r < desc->m_lin; r++) ix.lin_w.push_back(ix.lrp[r + 1] - ix.lrp[r]);
  to_csc(n, ix.lcol, ix.lrp, ix.lrp, ix.lin_w, ix.lcptr, ix.lcentry, ix.lcrow);
  if (desc->shared_len > 0 && desc->shared) ix.shared.assign(desc->shared, desc->shared + desc->shared_len);
  // ---- pattern of Psym = (Q + Q') / 2 by column: exact for a shared Q, dense for a per-problem Q, empty without Q;
  // united with the n_in x n_in block of every objective term (marked above)
  ix.P_cptr.assign(n + 1, 0);
  if (desc->Q.off >= 0)
    for (int j = 0; j < n; j++)
      for (int i = 0; i < n; i++)
        if (!desc->Q.shared || ix.shared[desc->Q.off + (size_t)i * n + j] != 0.0 || ix.shared[desc->Q.off + (size_t)j * n + i] != 0.0)
          pidx[(size_t)i * n + j] = 0;
  for (int j = 0; j < n; j++) {
    for (int i = 0; i < n; i++)
      if (pidx[(size_t)i * n + j] >= 0) {
        pidx[(size_t)i * n + j] = (int)ix.P_row.size();
        ix.P_row.push_back(i);
      }
    ix.P_cptr[j + 1] = (int)ix.P_row.size();
  }
  S.nnz_p = (int)ix.P_row.size();
  // the term-model entries summed into each pattern entry of P and each entry of q, in term order
  std::vector<std::vector<int>> hv(ix.P_row.size()), gv(n);
  for (int oi = 0; oi < S.n_ob; oi++) {
    const DevObjBlock &d = S.ob[oi];
    const int nn = d.n_in, ntri = nn * (nn + 1) / 2;
    for (int r = 0; r < d.m; r++) {
      const int *c = ix.ob_cols.data() + d.coff + (size_t)r * nn;
      const int base = d.toff + r * (ntri + nn + 1);
      for (int a = 0; a < nn; a++) {
        for (int b = 0; b < nn; b++) {
          const int lo = std::min(a, b), hi = std::max(a, b);
          hv[pidx[(size_t)c[a] * n + c[b]]].push_back(base + lo * nn - lo * (lo - 1) / 2 + (hi - lo));
        }
        gv[c[a]].push_back(base + ntri + a);
      }
    }
  }
  flatten(hv, ix.hv_ptr, ix.hv_src);
  flatten(gv, ix.gq_ptr, ix.gq_src);
  // ---- structural half-bandwidth of S = P + A'RA
  int bw = 0;
  for (int j = 0; j < n; j++)
    for (int p = ix.P_cptr[j]; p < ix.P_cptr[j + 1]; p++) bw = std::max(bw, std::abs(ix.P_row[p] - j));
  for (int r = 0; r < desc->m_lin; r++) bw = std::max(bw, col_span(ix.lcol, ix.lrp[r], ix.lin_w[r]));
  for (int i = 0; i < m_nl; i++) bw = std::max(bw, col_span(ix.jcol, ix.row_goff[i], ix.row_w[i]));
  S.s_bw = std::min(bw, n - 1);
}

// The ADMM loop a structure takes (fast_ok, p_narrow, fast_dense, dense_kind), its team size and its shared-memory
// layout (sws when S has to move out).  Refuses a structure whose working set does not fit shared memory.
static int choose_paths(const sco_structure_desc *desc, HostStruct &ix, size_t smem_optin) {
  DevStruct &S = ix.S;
  const int n = S.n, m_nl = S.m_nl;
  // thread-per-entity ADMM loop (sco_qp.cuh: fast_role keeps SCO_EN = 8 row entries / SCO_EH = 4 + 4 column entries
  // in registers and has no path for more)
  bool ok = true;
  for (int w : ix.lin_w) ok = ok && w <= 8;
  for (int w : ix.row_w) ok = ok && w <= 8;
  for (int j = 0; j < n; j++) ok = ok && ix.lcptr[j + 1] - ix.lcptr[j] <= 4 && ix.pc_ptr[j + 1] - ix.pc_ptr[j] <= 4;
  S.fast_ok = ok ? 1 : 0;
  bool narrow = true;
  for (int j = 0; j < n; j++) narrow = narrow && ix.P_cptr[j + 1] - ix.P_cptr[j] <= 4;
  S.p_narrow = narrow ? 1 : 0;
  bool dense = desc->m_lin == 0 && n <= 32 && m_nl > 0 && m_nl <= 48;
  for (int w : ix.row_w) dense = dense && w == n;
  dense = dense && !ix.any_map;  // its kernels assume rows over all n variables in column order
  S.fast_dense = dense && !ok ? 1 : 0;
  // ---- dense fast path: one dense hinge block over all variables, no linear rows, sizes within the instantiated table
  if (desc->m_lin == 0 && S.n_ob == 0 && desc->n_blocks == 1 && desc->blocks[0].family == SCO_FAM_QUADFORM &&
      desc->blocks[0].cnt_type == SCO_CNT_LEQ && !ix.any_map) {
    static const int table[][2] = {{8, 6}, {12, 16}, {20, 30}, {32, 32}};  // keep in sync with QPSolver::solve in sco_qp.cuh
    for (int k = 0; k < 4; k++)
      if (n <= table[k][0] && m_nl <= table[k][1]) { S.dense_kind = k + 1; break; }
  }
  // ---- team size and shared-memory layout
  const int work = std::max(std::max(n, m_nl), desc->m_lin);
  int team = work <= 40 ? 32 : work <= 96 ? 64 : work <= 192 ? 128 : 256;
  // one thread per entity (variable / linear row / penalty row) is what the fast ADMM loop wants (sco_qp.cuh:
  // fast_loop); structures with more than 512 entities stay on the strided shared-memory loop
  // (every role starts on a warp boundary)
  const int entities = ((n + 31) & ~31) + ((desc->m_lin + 31) & ~31) + ((m_nl + 31) & ~31);
  if (entities <= 512) team = entities <= 32 ? 32 : entities <= 64 ? 64 : entities <= 128 ? 128 : entities <= 256 ? 256 : 512;
  if (S.dense_kind) team = 64;  // two warps per problem: rows | variables (sco_dense.cuh)
  ix.team = team;
  for (;;) {
    build_layout(S, team);
    ix.smem_bytes = (size_t)(S.L.total + ((n + 1) & ~1)) * sizeof(double);
    if (ix.smem_bytes <= smem_optin) return 0;
    if (S.sws || S.dense_kind || S.n_ob)  // objective terms stay in the resident regime
      return fail(SCO_ERR_UNSUPPORTED, "problem working set (%zu B) exceeds shared memory per block (%zu B)",
                  ix.smem_bytes, smem_optin);
    // the n x n matrix S (and its inverse) moves to a global workspace per resident team: the ADMM loop streams it
    // from L2 / HBM in every iteration (strided loop only); everything else stays in shared memory
    S.sws = n * n;
  }
}

// Uploads, kernel selection and configuration, launch-slot and staging scratch.  On failure the caller destroys h.
static int setup_device(sco_handle *h, const HostStruct &ix) {
  DevStruct &S = h->S = ix.S;
  h->team = ix.team;
  h->smem_bytes = ix.smem_bytes;
  int rc = 0;
  rc |= upload(h, ix.row_goff, &S.row_goff); rc |= upload(h, ix.row_soff, &S.row_soff);
  rc |= upload(h, ix.row_w, &S.row_w); rc |= upload(h, ix.row_eq, &S.row_eq);
  rc |= upload(h, ix.row_gmask, &S.row_gmask); rc |= upload(h, ix.jcol, &S.jcol_g);
  rc |= upload(h, ix.pc_ptr, &S.pc_ptr); rc |= upload(h, ix.pc_e, &S.pc_e); rc |= upload(h, ix.pc_r, &S.pc_r);
  rc |= upload(h, ix.lrp, &S.lin_rowptr); rc |= upload(h, ix.lcol, &S.lin_col); rc |= upload(h, ix.lval, &S.lin_val);
  rc |= upload(h, ix.lcptr, &S.lin_cptr); rc |= upload(h, ix.lcentry, &S.lin_centry); rc |= upload(h, ix.lcrow, &S.lin_crow);
  rc |= upload(h, ix.shared, &S.shared);
  rc |= upload(h, ix.P_cptr, &S.P_cptr); rc |= upload(h, ix.P_row, &S.P_row);
  rc |= upload(h, ix.ob_cols, &S.ob_cols); rc |= upload(h, ix.hv_ptr, &S.hv_ptr); rc |= upload(h, ix.hv_src, &S.hv_src);
  rc |= upload(h, ix.gq_ptr, &S.gq_ptr); rc |= upload(h, ix.gq_src, &S.gq_src);
  if (rc) return SCO_ERR_CUDA;
  const int team = ix.team;
  h->gen_ops = team == 32 ? sco_team_ops_32() : team == 64 ? sco_team_ops_64() : team == 128 ? sco_team_ops_128()
               : team == 256 ? sco_team_ops_256() : sco_team_ops_512();
  h->ops = h->gen_ops;
  if (S.dense_kind)
    h->ops = S.dense_kind == 1 ? sco_dense_ops_1() : S.dense_kind == 2 ? sco_dense_ops_2() : S.dense_kind == 3 ? sco_dense_ops_3() : sco_dense_ops_4();
  int occ = 0;
  cudaError_t ce = h->gen_ops->configure(h->smem_bytes, &occ, &h->carve_gen);
  h->carve_ops = h->carve_gen;
  if (ce == cudaSuccess && h->ops != h->gen_ops) ce = h->ops->configure(h->smem_bytes, &occ, &h->carve_ops);
  if (ce != cudaSuccess) return fail(SCO_ERR_CUDA, "kernel configuration failed: %s", cudaGetErrorString(ce));
  h->occupancy = std::max(occ, 1);
  h->Jscr_ctas = (size_t)h->sm_count * h->occupancy;
  bool ok = cudaMalloc(&h->counter, sco_handle::NSLOT * sizeof(unsigned long long)) == cudaSuccess &&
            cudaMalloc(&h->order_err, sco_handle::NSLOT * sizeof(int)) == cudaSuccess;
  for (int k = 0; k < sco_handle::NSLOT && ok; k++)
    ok = cudaMalloc(&h->Jscr[k], std::max<size_t>(h->Jscr_ctas * (size_t)std::max(S.jnnz + S.sws, 1), 1) * sizeof(double)) == cudaSuccess &&
         cudaEventCreateWithFlags(&h->slot_done[k], cudaEventDisableTiming) == cudaSuccess;
  for (int k = 0; k < sco_handle::NSTG && ok; k++)
    ok = cudaEventCreateWithFlags(&h->stg[k].done, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) return fail(SCO_ERR_CUDA, "cudaMalloc of scratch failed");
  return SCO_OK;
}

extern "C" int sco_create(const sco_structure_desc *desc, int device, sco_handle **out) {
  if (!desc || !out) return fail(SCO_ERR_ARG, "null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(SCO_ERR_CUDA, "no CUDA device: the engine has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SCO_ERR_ARG, "device %d out of range", device);
  if (int rc = check_desc(desc)) return rc;
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(SCO_ERR_CUDA, "device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor);
  HostStruct ix;
  build_index(desc, ix);
  if (int rc = choose_paths(desc, ix, (size_t)prop.sharedMemPerBlockOptin)) return rc;
  std::unique_ptr<sco_handle, decltype(&sco_destroy)> h(new sco_handle(), &sco_destroy);  // released on success
  h->device = device; h->sm_count = prop.multiProcessorCount;
  if (int rc = setup_device(h.get(), ix)) return rc;
  *out = h.release();
  return SCO_OK;
}

extern "C" int sco_destroy(sco_handle *h) {
  if (!h) return SCO_OK;
  cudaSetDevice(h->device);
  for (void *p : h->dev_allocs) cudaFree(p);
  cudaFree(h->counter);
  cudaFree(h->order_err);
  for (int k = 0; k < sco_handle::NSLOT; k++) {
    cudaFree(h->Jscr[k]);
    cudaFree(h->seen[k]);
    if (h->slot_done[k]) cudaEventDestroy(h->slot_done[k]);
  }
  for (int k = 0; k < sco_handle::NSTG; k++) {
    sco_handle::Staging &g = h->stg[k];
    cudaFree(g.params); cudaFree(g.x0); cudaFree(g.x); cudaFree(g.merit); cudaFree(g.obj); cudaFree(g.vio);
    cudaFree(g.verdict); cudaFree(g.stats); cudaFree(g.nonconv);
    if (g.done) cudaEventDestroy(g.done);
  }
  delete h;
  return SCO_OK;
}

extern "C" int sco_query(sco_handle *h, int64_t *out8) {
  if (!h || !out8) return fail(SCO_ERR_ARG, "null argument");
  out8[0] = h->S.n; out8[1] = h->S.m_nl; out8[2] = h->S.n_slack; out8[3] = h->S.jnnz;
  out8[4] = h->S.n_q; out8[5] = (int64_t)h->smem_bytes; out8[6] = h->team; out8[7] = h->occupancy;
  return SCO_OK;
}

// d_order must be a permutation of 0..B-1: every entry in range and seen once.  Violations are counted in *err;
// k_solve reads it and refuses the batch (verdict -3 everywhere) -- stream-ordered, no host synchronisation.
__global__ void k_check_order(const int *__restrict__ order, long long B, unsigned *seen, int *err) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < B; i += (long long)gridDim.x * blockDim.x) {
    const int v = order[i];
    if (v < 0 || v >= B) { atomicAdd(err, 1); continue; }
    const unsigned bit = 1u << (v & 31);
    if (atomicOr(seen + (v >> 5), bit) & bit) atomicAdd(err, 1);
  }
}

extern "C" int sco_solve_batch(sco_handle *h, int64_t B, const double *d_params, const double *d_x0,
                               const sco_settings *s, double *d_x_out, int32_t *d_verdict,
                               double *d_merit, double *d_objective, double *d_max_vio,
                               int32_t *d_stats, void *stream) {
  return sco_solve_batch_ordered(h, B, d_params, d_x0, s, d_x_out, d_verdict, d_merit, d_objective, d_max_vio,
                                 d_stats, nullptr, stream);
}

extern "C" int sco_solve_batch_ordered(sco_handle *h, int64_t B, const double *d_params, const double *d_x0,
                                       const sco_settings *s, double *d_x_out, int32_t *d_verdict,
                                       double *d_merit, double *d_objective, double *d_max_vio,
                                       int32_t *d_stats, const int32_t *d_order, void *stream) {
  sco_batch_io io;
  memset(&io, 0, sizeof(io));
  io.d_params = d_params; io.d_x0 = d_x0; io.d_x_out = d_x_out; io.d_verdict = d_verdict; io.d_merit = d_merit;
  io.d_objective = d_objective; io.d_max_vio = d_max_vio; io.d_stats = d_stats; io.d_order = d_order;
  return sco_solve_batch_io(h, B, &io, s, stream);
}

extern "C" int sco_solve_batch_io(sco_handle *h, int64_t B, const sco_batch_io *io, const sco_settings *s, void *stream) {
  if (!h || !s || !io) return fail(SCO_ERR_ARG, "null argument");
  if (B <= 0) return SCO_OK;  // an empty batch is valid and touches nothing
  if (!io->d_params || !io->d_x0 || !io->d_x_out || !io->d_verdict) return fail(SCO_ERR_ARG, "null argument");
  if (io->d_x_warm || io->d_y_warm) return fail(SCO_ERR_UNSUPPORTED, "x_warm / y_warm are reserved");
  if (B > 0x7fffffffLL) return fail(SCO_ERR_ARG, "batch too large");
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  DevSettings d = to_dev(s);
  const int slot = (int)(h->next_slot++ % sco_handle::NSLOT);
  CUDA_TRY(cudaStreamWaitEvent(st, h->slot_done[slot], 0));  // the slot's previous launch (any stream)
  CUDA_TRY(cudaMemsetAsync(h->counter + slot, 0, sizeof(unsigned long long), st));
  const int *order_err = nullptr;
  if (io->d_order) {
    const long long words = (B + 31) / 32;
    if (words > h->seen_cap[slot]) {
      CUDA_TRY(cudaEventSynchronize(h->slot_done[slot]));
      if (h->seen[slot]) cudaFree(h->seen[slot]);
      h->seen[slot] = nullptr;
      h->seen_cap[slot] = 0;
      CUDA_TRY(cudaMalloc(&h->seen[slot], (size_t)words * sizeof(unsigned)));
      h->seen_cap[slot] = words;
    }
    CUDA_TRY(cudaMemsetAsync(h->seen[slot], 0, (size_t)words * sizeof(unsigned), st));
    CUDA_TRY(cudaMemsetAsync(h->order_err + slot, 0, sizeof(int), st));
    const int blocks = (int)std::min<long long>((B + 255) / 256, 4096);
    k_check_order<<<blocks, 256, 0, st>>>(io->d_order, (long long)B, h->seen[slot], h->order_err + slot);
    CUDA_TRY(cudaGetLastError());
    order_err = h->order_err + slot;
  }
  const long long grid = std::min<long long>(B, (long long)h->Jscr_ctas);
  SolveArgs a = {(long long)B, io->d_params, io->d_x0, io->d_x_out, io->d_verdict, io->d_merit, io->d_objective,
                 io->d_max_vio, io->d_stats, h->Jscr[slot], h->counter + slot, io->d_order, io->d_nonconverged, order_err};
  CUDA_TRY(h->ops->prepare(h->carve_ops));
  h->ops->solve((unsigned)grid, h->smem_bytes, st, h->S, d, a);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaEventRecord(h->slot_done[slot], st));
  return SCO_OK;
}

template <typename T>
static int grow(T **p, size_t count) {
  if (*p) cudaFree(*p);
  *p = nullptr;
  CUDA_TRY(cudaMalloc(p, std::max<size_t>(count, 1) * sizeof(T)));
  return 0;
}

extern "C" int sco_solve_batch_host_async(sco_handle *h, int64_t B, const double *params, const double *x0,
                                          const sco_settings *s, double *x_out, int32_t *verdict,
                                          double *merit, double *objective, double *max_vio,
                                          int32_t *stats, void *stream) {
  return sco_solve_batch_host_groups(h, B, params, x0, s, x_out, verdict, merit, objective, max_vio, stats, nullptr,
                                     stream);
}

extern "C" int sco_solve_batch_host_groups(sco_handle *h, int64_t B, const double *params, const double *x0,
                                           const sco_settings *s, double *x_out, int32_t *verdict,
                                           double *merit, double *objective, double *max_vio,
                                           int32_t *stats, int32_t *nonconverged, void *stream) {
  if (!h || !s) return fail(SCO_ERR_ARG, "null argument");
  if (B <= 0) return SCO_OK;
  if (!params || !x0 || !x_out || !verdict) return fail(SCO_ERR_ARG, "null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  const int n = h->S.n;
  cudaStream_t st = (cudaStream_t)stream;
  sco_handle::Staging &g = h->stg[h->next_stg++ % sco_handle::NSTG];
  if (B > g.cap_B) {
    CUDA_TRY(cudaEventSynchronize(g.done));  // nothing in flight may still use the old buffers
    int rc = 0;
    rc |= grow(&g.params, (size_t)B * h->S.stride); rc |= grow(&g.x0, (size_t)B * n);
    rc |= grow(&g.x, (size_t)B * n); rc |= grow(&g.merit, (size_t)B); rc |= grow(&g.obj, (size_t)B);
    rc |= grow(&g.vio, (size_t)B); rc |= grow(&g.verdict, (size_t)B); rc |= grow(&g.stats, (size_t)4 * B);
    rc |= grow(&g.nonconv, (size_t)B);
    if (rc) { g.cap_B = 0; return SCO_ERR_CUDA; }
    g.cap_B = B;
  }
  CUDA_TRY(cudaStreamWaitEvent(st, g.done, 0));
  CUDA_TRY(cudaMemcpyAsync(g.params, params, (size_t)B * h->S.stride * sizeof(double), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(g.x0, x0, (size_t)B * n * sizeof(double), cudaMemcpyHostToDevice, st));
  sco_batch_io io;
  memset(&io, 0, sizeof(io));
  io.d_params = g.params; io.d_x0 = g.x0; io.d_x_out = g.x; io.d_verdict = g.verdict; io.d_merit = g.merit;
  io.d_objective = g.obj; io.d_max_vio = g.vio; io.d_stats = g.stats; io.d_nonconverged = nonconverged ? g.nonconv : nullptr;
  int rc = sco_solve_batch_io(h, B, &io, s, st);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(x_out, g.x, (size_t)B * n * sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(verdict, g.verdict, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (merit) CUDA_TRY(cudaMemcpyAsync(merit, g.merit, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (objective) CUDA_TRY(cudaMemcpyAsync(objective, g.obj, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (max_vio) CUDA_TRY(cudaMemcpyAsync(max_vio, g.vio, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (stats) CUDA_TRY(cudaMemcpyAsync(stats, g.stats, (size_t)4 * B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (nonconverged) CUDA_TRY(cudaMemcpyAsync(nonconverged, g.nonconv, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaEventRecord(g.done, st));
  return SCO_OK;
}

extern "C" int sco_solve_batch_host(sco_handle *h, int64_t B, const double *params, const double *x0,
                                    const sco_settings *s, double *x_out, int32_t *verdict,
                                    double *merit, double *objective, double *max_vio,
                                    int32_t *stats) {
  int rc = sco_solve_batch_host_async(h, B, params, x0, s, x_out, verdict, merit, objective, max_vio, stats, nullptr);
  if (rc) return rc;
  CUDA_TRY(cudaStreamSynchronize(0));
  return SCO_OK;
}

static unsigned stage_grid(sco_handle *h, int64_t B) {
  return (unsigned)std::min<long long>(B, (long long)h->Jscr_ctas);
}

extern "C" int sco_convexify(sco_handle *h, int64_t B, const double *d_params, const double *d_x,
                             double *d_f, double *d_J, double *d_b, double *d_obj, void *stream) {
  return sco_convexify_model(h, B, d_params, d_x, d_f, d_J, d_b, d_obj, nullptr, nullptr, nullptr, stream);
}

extern "C" int sco_convexify_model(sco_handle *h, int64_t B, const double *d_params, const double *d_x,
                                   double *d_f, double *d_J, double *d_b, double *d_obj, double *d_H, double *d_g,
                                   double *d_c, void *stream) {
  if (!h || !d_params || !d_x) return fail(SCO_ERR_ARG, "null argument");
  if ((d_H || d_g || d_c) && !h->S.n_ob) return fail(SCO_ERR_ARG, "the structure has no non-quadratic objective term");
  if (B <= 0) return SCO_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  // without d_J the kernel parks the Jacobian in a launch slot's scratch: take the slot like a solve does
  double *scratch = nullptr;
  int slot = -1;
  if (!d_J) {
    slot = (int)(h->next_slot++ % sco_handle::NSLOT);
    CUDA_TRY(cudaStreamWaitEvent(st, h->slot_done[slot], 0));
    scratch = h->Jscr[slot];
  }
  ConvexifyArgs a = {(long long)B, d_params, d_x, d_f, d_J, d_b, d_obj, scratch, d_H, d_g, d_c};
  CUDA_TRY(h->gen_ops->prepare(h->carve_gen));
  h->gen_ops->convexify(stage_grid(h, B), h->smem_bytes, st, h->S, a);
  CUDA_TRY(cudaGetLastError());
  if (slot >= 0) CUDA_TRY(cudaEventRecord(h->slot_done[slot], st));
  return SCO_OK;
}

extern "C" int sco_qp_solve(sco_handle *h, int64_t B, const double *d_params, const double *d_J,
                            const double *d_b, const uint32_t *d_mask, const double *d_lbx,
                            const double *d_ubx, const double *d_pi, const int32_t *d_kdup,
                            const double *d_xref, int use_penalty, int closest_point,
                            const sco_settings *s, double *d_xq, int32_t *d_status, int32_t *d_iters,
                            void *stream) {
  return sco_qp_solve_w(h, B, d_params, d_J, d_b, d_mask, d_lbx, d_ubx, d_pi, d_kdup, nullptr, d_xref, use_penalty,
                        closest_point, s, d_xq, d_status, d_iters, stream);
}

extern "C" int sco_qp_solve_w(sco_handle *h, int64_t B, const double *d_params, const double *d_J,
                              const double *d_b, const uint32_t *d_mask, const double *d_lbx,
                              const double *d_ubx, const double *d_pi, const int32_t *d_kdup,
                              const double *d_wa, const double *d_xref, int use_penalty, int closest_point,
                              const sco_settings *s, double *d_xq, int32_t *d_status, int32_t *d_iters,
                              void *stream) {
  if (!h || !s || !d_params || !d_xq || !d_status || !d_iters) return fail(SCO_ERR_ARG, "null argument");
  if (use_penalty && h->S.m_nl > 0 && (!d_J || !d_b)) return fail(SCO_ERR_ARG, "penalty rows need J and b");
  if (closest_point && !d_xref) return fail(SCO_ERR_ARG, "closest_point needs xref");
  if (B <= 0) return SCO_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  DevSettings d = to_dev(s);
  QpStageArgs a = {(long long)B, d_params, d_J, d_b, d_mask, d_lbx, d_ubx, d_pi, d_kdup, d_wa, d_xref,
                   use_penalty, closest_point, d_xq, d_status, d_iters, nullptr};
  int slot = -1;
  if (h->S.sws) {  // S lives in a launch slot's scratch: take the slot like a solve does
    slot = (int)(h->next_slot++ % sco_handle::NSLOT);
    CUDA_TRY(cudaStreamWaitEvent(st, h->slot_done[slot], 0));
    a.scr = h->Jscr[slot];
  }
  CUDA_TRY(h->ops->prepare(h->carve_ops));
  h->ops->qp(stage_grid(h, B), h->smem_bytes, st, h->S, d, a);
  CUDA_TRY(cudaGetLastError());
  if (slot >= 0) CUDA_TRY(cudaEventRecord(h->slot_done[slot], st));
  return SCO_OK;
}

extern "C" int sco_merit(sco_handle *h, int64_t B, const double *d_params, const double *d_x,
                         const double *d_J, const double *d_b, const double *d_mu, double *d_merit,
                         double *d_model, double *d_max_vio, double *d_gv, double *d_gm, void *stream) {
  if (!h || !d_params || !d_x) return fail(SCO_ERR_ARG, "null argument");
  if (B <= 0) return SCO_OK;
  CUDA_TRY(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  MeritArgs a = {(long long)B, d_params, d_x, d_J, d_b, d_mu, d_merit, d_model, d_max_vio, d_gv, d_gm};
  CUDA_TRY(h->gen_ops->prepare(h->carve_gen));
  h->gen_ops->merit(stage_grid(h, B), h->smem_bytes, st, h->S, a);
  CUDA_TRY(cudaGetLastError());
  return SCO_OK;
}
