// sco_device.cuh -- device-side data model shared by every kernel of the engine.
//
// One thread TEAM (a warp, or a CTA of 2..8 warps) owns one problem at a time and keeps the
// whole working set of its current penalty QP in shared memory for the duration of the ADMM
// solve ("resident regime", DESIGN.md section 4).  For generic structures all sizes are run-time
// values and the shared-memory carve-up (Layout) is computed once on the host; dense hinge-only
// structures use the compile-time layout DenseL below (sco_dense.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define SCO_DEV_MAX_BLOCKS 16
#define SCO_DEV_MAX_GROUPS 8
#define SCO_DEV_MAX_OBJ_BLOCKS 4

#define OSQP_INFTY 1e30
#define OSQP_MIN_SCALING 1e-4
#define OSQP_MAX_SCALING 1e4
#define OSQP_RHO_MIN 1e-6
#define OSQP_RHO_MAX 1e6
#define OSQP_RHO_EQ_OVER_RHO_INEQ 1e3
#define OSQP_RHO_TOL 1e-4


struct DevField {
  long long off;
  int shared;
  int pad_;
};

struct DevBlock {
  int family, cnt_type, m, group_mask;
  int jw;    // stored Jacobian entries per row
  int row0;  // first penalty row of the block
  int joff;  // offset of the block inside the per-problem J array (global layout, unpadded)
  int n_in;  // != 0: the block has a column map (include/sco_b200.h) with n_in inputs per row; row r reads
             // x[jcol_g[joff + r * n_in + i]] as its input i (the map is the block's stored-entry columns)
  int ipar[8];
  DevField par, val;
};

// Non-quadratic objective terms of one input count and derivative mode (include/sco_b200.h sco_obj_block_desc; a
// structure's obj_prog is turned into one such block over all n variables).  Term r of the block reads
// x[ob_cols[coff + r * n_in + i]] as its input i; its convex model lives at toff + r * (n_in (n_in + 1) / 2 + n_in + 1)
// in the term-model area (Layout::ot): the upper triangle of H_t+ (row-major), then A_t (n_in), then f_t.
struct DevObjBlock {
  int m, n_in, flags;  // flags bit 0: forward-mode gradient
  int t0;              // index of its first term among all terms
  int coff, toff;
  DevField prog;       // m row offsets, then the code
};

// shared-memory carve-up, offsets in doubles
struct Layout {
  int Js, S, Als;
  // per user variable (n)
  int x, xt, xt2, qh, D, bx, rb, lb, ub, zb, yb, Eb, dxv, dyb, xs;
  // per linear row (m_lin)
  int El, rl, ll, ul, zl, yl, wl, dyl;
  // per penalty row (m_nl)
  int Ep, rp, lp, up, zp, yp, wp, bb, fv, dyp;
  // per slack (nsl*m_nl, slot a*m_nl + i)
  int s, Ds, sl, bs, zs, ys, Es, gs, hs, rs, dss, dys;
  int Minv;   // 3*m_nl
  int red;    // reduction scratch: 8 warps * 8 values
  int msk;    // m_nl * mw uint32 (counted in doubles, rounded up)
  int stage;  // per-warp staging buffers for family evaluation
  // convex model of the non-quadratic objective terms: per-term models (DevObjBlock), the Jacobi scratch of the
  // eigenvalue shift (n_in_max^2 per warp), the assembled model on the pattern of P (nnz(P)), its linear term (n) and
  // its constant (1)
  int ot, jac, Hv, gq, oc;
  int ps;     // partial sums of S^-1 rhs: 4 column segments x n (fast_loop, sco_qp.cuh)
  int total;  // doubles
};

// compile-time shared-memory layout (offsets in doubles, from the start of dynamic shared memory) of
// the dense two-warp QP solve, sco_dense.cuh
template <int NP, int MP>
struct DenseL {
  static constexpr int ev(int x) { return (x + 1) & ~1; }
  static constexpr int LDJ = NP | 1;  // odd row stride: lane i reading J[i][k] is conflict-free
  static constexpr int NV = NP + MP;
  static constexpr int VLD = ev(NV) + 2;  // last slot = dump for the lanes that own no entry
  static constexpr int NE = ev(NP), ME = ev(MP);
  // matrices
  static constexpr int Js = 0;                      // scaled, masked Jacobian  MP x LDJ
  static constexpr int Si = Js + ev(MP * LDJ);      // Psym -> S -> S^-1        NP x NP
  static constexpr int Ph = Si + ev(NP * NP);       // c D Psym D               NP x NP
  static constexpr int Ks = Ph + ev(NP * NP);       // K = S^-1 J'              NP x MP
  // exchange buffers
  static constexpr int Vb = Ks + ev(NP * MP);       // (c, wp), double-buffered  2 x VLD
  static constexpr int Xs = Vb + 2 * VLD;           // x of every variable (termination test)  32
  static constexpr int Ys = Xs + 32;                // kd*y of every penalty row                32
  static constexpr int Red = Ys + 32;               // two warps x 16 partial results
  static constexpr int D = Red + 32;                // column scaling of the variables (32)
  static constexpr int t1 = D + 32;                 // scratch per variable (32)
  static constexpr int dg = t1 + 32;                // sigma + rho_j bx_j^2 (32)
  static constexpr int cf = dg + 32;                // Schur coefficient per row (32)
  // lane constants, [warp][k][lane]: 0 u0, 1 u1, 2 u2, 3 lo, 4 hi, 5 r0, 6 r1, 7 r2, 8 e0, 9 e1, 10 e2, 11 rho_j
  static constexpr int LA = cf + 32;
  static constexpr int NLA = 12;
  // iterates handed to the rare paths (certificates, max_iter epilogue): 5 per variable, 8 per row
  static constexpr int Sp = LA + 2 * NLA * 32;
  // scalars: 0 eps_abs, 1 eps_rel, 2 eps_prim_inf, 3 eps_dual_inf, 4 c, 5 1/c, 6 c*pi, 7 rho, 8 kd
  static constexpr int Sc = Sp + 13 * 32;
  static constexpr int total = Sc + 16;
};

struct DevStruct {
  int n, m_lin, nnz_lin, n_blocks, n_groups, m_nl, n_slack, jnnz, n_q, nsl;
  int sjnnz;           // padded Jacobian entries in shared memory
  int dense_kind;      // != 0: two-warp dense solve (sco_dense.cuh), index into its size table
  int fast_ok;         // rows of A with <= 8 entries, columns with <= 4 + 4: the thread-per-entity loop applies
  int p_narrow;        // every column of the objective matrix's pattern has <= 4 entries (in-loop termination test)
  int fast_dense;      // dense penalty rows over n <= 32 variables (no column map), m_nl <= 48, no linear rows: its
                       // dense variant applies
  int s_bw;            // structural half-bandwidth of S = P + A'RA (max |i - j| over its pattern): the Gauss-Jordan
                       // sweep of pivot k only touches the leading (k + s_bw + 1)^2 block
  int stage_per_warp;  // doubles
  int sws;             // != 0: n * n doubles of S live in the team's global workspace (behind its Jacobian scratch),
                       // not in shared memory: structures too large for one SM's shared memory otherwise
  int mw;              // 32-bit words of a row's frozen-sparsity mask: ceil(widest row / 32), >= 1
  long long stride;
  DevField Q, q, c, lin_l, lin_u;
  DevField qa;         // AffExpr objective terms, summed (n): enters the QP with the weight of quirk C-4
  DevField lb0, ub0;   // user bounds of the scalar variables (n each): the closest-point QP honours them
  int n_ob, n_terms;   // objective blocks (0 = no non-quadratic objective term) and their terms
  int n_in_max, nwj;   // widest term; warps that run the eigenvalue shift (each with n_in_max^2 doubles of scratch)
  int nnz_p;           // entries of the pattern of P (P_cptr[n])
  DevObjBlock ob[SCO_DEV_MAX_OBJ_BLOCKS];
  const int *ob_cols;          // column maps of the objective blocks
  const int *hv_ptr, *hv_src;  // nnz_p + 1 / per pattern entry of P: the term-model entries (H_t+) summed into it
  const int *gq_ptr, *gq_src;  // n + 1 / per variable: the term-model entries (A_t) summed into q
  // linear rows: CSR + CSC (entry index into lin_val / Als)
  const int *lin_rowptr, *lin_col, *lin_cptr, *lin_centry, *lin_crow;
  const double *lin_val;
  // penalty rows
  const int *row_goff;   // m_nl: offset of the row in the global J layout
  const int *row_soff;   // m_nl: offset of the row in the shared-memory (padded) layout
  const int *row_w;      // m_nl: entries in the row
  const int *row_eq;     // m_nl: 1 = equality (abs penalty, two slacks)
  const int *row_gmask;  // m_nl: constraint-group membership
  const int *jcol_g;     // jnnz: column of every stored entry (global layout)
  const int *pc_ptr, *pc_e, *pc_r;  // CSC over user variables: shared-memory entry index, row
  // sparsity pattern of the symmetrised objective matrix, by column (exact when Q is shared by the batch -- the
  // smoothness matrices of the trajectory configurations are block tridiagonal -- and dense otherwise; empty when
  // there is no Q), united with the n_in x n_in block of every objective term.  Column norms, P x and the assembly
  // of S walk this instead of n entries per column.
  const int *P_cptr, *P_row;
  const double *shared;
  int overlap[SCO_DEV_MAX_GROUPS];  // bit g2 of overlap[g] <=> groups overlap (prob.py:139-142)
  DevBlock blocks[SCO_DEV_MAX_BLOCKS];
  Layout L;
};

extern __shared__ __align__(16) double sco_smem[];
extern __shared__ __align__(16) double2 sco_smem2[];  // same storage, viewed as 16-byte words

// By-value view of the index arrays and sizes a QP needs.  Device functions copy it (and QPW,
// DevSettings) into locals on entry: anything read through a reference lives behind a generic pointer,
// and since a shared-memory store may alias a generic address the compiler re-loads it after every
// store -- measured as chains of LD.E in front of every shared access.
struct DevIdx {
  int n, m_lin, nnz_lin, m_nl, n_slack;
  const int *lin_rowptr, *lin_col, *lin_cptr, *lin_centry, *lin_crow;
  const double *lin_val;
  const int *row_goff, *row_soff, *row_w, *row_eq, *row_gmask, *jcol_g, *pc_ptr, *pc_e, *pc_r;
  const int *P_cptr, *P_row;
  __device__ __forceinline__ explicit DevIdx(const DevStruct &S)
      : n(S.n), m_lin(S.m_lin), nnz_lin(S.nnz_lin), m_nl(S.m_nl), n_slack(S.n_slack), lin_rowptr(S.lin_rowptr),
        lin_col(S.lin_col), lin_cptr(S.lin_cptr), lin_centry(S.lin_centry), lin_crow(S.lin_crow), lin_val(S.lin_val),
        row_goff(S.row_goff), row_soff(S.row_soff), row_w(S.row_w), row_eq(S.row_eq), row_gmask(S.row_gmask),
        jcol_g(S.jcol_g), pc_ptr(S.pc_ptr), pc_e(S.pc_e), pc_r(S.pc_r), P_cptr(S.P_cptr), P_row(S.P_row) {}
};

struct DevSettings {
  double improve_ratio_threshold, min_trust_region_size, min_approx_improve;
  double trust_shrink_ratio, trust_expand_ratio, cnt_tolerance, merit_coeff_increase_ratio;
  double initial_trust_region_size, initial_penalty_coeff;
  int max_merit_coeff_increases, max_sqp_iters;
  double eps_abs, eps_rel, rho, sigma, alpha, eps_prim_inf, eps_dual_inf;
  int max_iter, scaling, check_termination, adaptive_rho, adaptive_rho_interval;
  int compound_penalty, freeze_sparsity, duplicate_rows, force_generic;
  int aff_obj_quirk, warm_start;
};

__device__ __forceinline__ const double *field_ptr(const DevStruct &S, const DevField &f,
                                                   const double *prm) {
  return f.off < 0 ? nullptr : ((f.shared ? S.shared : prm) + f.off);
}


struct Sh {
  int off;
  __device__ __forceinline__ double &operator[](int i) const { return sco_smem[off + i]; }
  __device__ __forceinline__ Sh operator+(int k) const { return Sh{off + k}; }
  __device__ __forceinline__ double *ptr() const { return sco_smem + off; }
  // 16-byte word i of the array (off must be even): a shared-space access, no generic pointer
  __device__ __forceinline__ const double2 &v2(int i) const { return sco_smem2[(off >> 1) + i]; }
};
struct ShU32 {
  int off;  // in doubles
  __device__ __forceinline__ uint32_t &operator[](int i) const {
    return reinterpret_cast<uint32_t *>(sco_smem + off)[i];
  }
};


// ------------------------------------------------------------------------------------
// team primitives
template <int TEAM>
struct Team {
  static __device__ __forceinline__ void sync() {
    if (TEAM == 32) __syncwarp();
    else __syncthreads();
  }

  template <int K, bool IS_MAX>
  static __device__ __forceinline__ void reduce(double (&v)[K], Sh red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < K; k++) {
        double t = __shfl_xor_sync(0xffffffffu, v[k], o);
        v[k] = IS_MAX ? fmax(v[k], t) : v[k] + t;
      }
    }
    if (TEAM > 32) {
      const int wi = threadIdx.x >> 5, l = threadIdx.x & 31;
      __syncthreads();
      if (l == 0) {
#pragma unroll
        for (int k = 0; k < K; k++) red[wi * 16 + k] = v[k];
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < K; k++) {
        double acc = red[k];
        for (int ww = 1; ww < TEAM / 32; ww++)
          acc = IS_MAX ? fmax(acc, red[ww * 16 + k]) : acc + red[ww * 16 + k];
        v[k] = acc;
      }
    }
  }
  // KM maxima and KS sums in one pass (KM + KS <= 16).  The warps' partial results are combined by KM + KS threads
  // (in warp order, like `reduce`) and read back by everybody: three barriers, but no thread walks all the warps'
  // partials for every value (with 16 warps that walk was 16 shared loads per value per thread).
  template <int KM, int KS>
  static __device__ __forceinline__ void reduce_mixed(double (&vm)[KM], double (&vs)[KS], Sh red) {
    static_assert(KM + KS <= 16, "one 16-double slot per warp");
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int k = 0; k < KM; k++) vm[k] = fmax(vm[k], __shfl_xor_sync(0xffffffffu, vm[k], o));
#pragma unroll
      for (int k = 0; k < KS; k++) vs[k] += __shfl_xor_sync(0xffffffffu, vs[k], o);
    }
    if (TEAM > 32) {
      constexpr int NW = TEAM / 32;
      const int wi = threadIdx.x >> 5, l = threadIdx.x & 31;
      __syncthreads();
      if (l == 0) {
#pragma unroll
        for (int k = 0; k < KM; k++) red[wi * 16 + k] = vm[k];
#pragma unroll
        for (int k = 0; k < KS; k++) red[wi * 16 + KM + k] = vs[k];
      }
      __syncthreads();
      if (threadIdx.x < KM + KS) {
        const int k = threadIdx.x;
        double acc = red[k];
        for (int ww = 1; ww < NW; ww++) acc = k < KM ? fmax(acc, red[ww * 16 + k]) : acc + red[ww * 16 + k];
        red[NW * 16 + k] = acc;
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < KM; k++) vm[k] = red[NW * 16 + k];
#pragma unroll
      for (int k = 0; k < KS; k++) vs[k] = red[NW * 16 + KM + k];
    }
  }
  template <int K>
  static __device__ __forceinline__ void reduce_max(double (&v)[K], Sh red) {
    reduce<K, true>(v, red);
  }
  template <int K>
  static __device__ __forceinline__ void reduce_sum(double (&v)[K], Sh red) {
    reduce<K, false>(v, red);
  }
};

// explicit shared-window accesses (32-bit addresses from __cvta_generic_to_shared)
__device__ __forceinline__ double2 lds_v2(uint32_t addr) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
  asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
// warp-wide maximum of non-negative doubles: their bit patterns order like unsigned integers, so
// two redux.sync (high word, then low word among the lanes that hold the maximal high word) replace
// the five shuffle rounds of a butterfly
__device__ __forceinline__ double warp_max_nonneg(double v) {
  const unsigned hi = (unsigned)__double2hiint(v), lo = (unsigned)__double2loint(v);
  const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
  const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
  return __hiloint2double((int)mh, (int)ml);
}

__device__ __forceinline__ double limit_scaling(double v) {
  v = v < OSQP_MIN_SCALING ? 1.0 : v;
  v = v > OSQP_MAX_SCALING ? OSQP_MAX_SCALING : v;
  return v;
}

// ------------------------------------------------------------------------------------
// shared-memory views.  Every array of the working set is addressed as an offset into the ONE
// dynamic shared-memory array below, so the compiler can prove the address space and emits
// LDS/STS (raw double* members made every access a generic LD/ST).
struct QPW {
  Sh Js, Sm, Als;
  Sh x, xt, xt2, qh, D, bx, rb, lb, ub, zb, yb, Eb, dxv, dyb, xs;
  Sh El, rl, ll, ul, zl, yl, wl, dyl;
  Sh Ep, rp, lp, up, zp, yp, wp, bb, fv, dyp;
  Sh s, Ds, sl, bs, zs, ys, Es, gs, hs, rs, dss, dys, Minv;
  Sh red;
  ShU32 msk;
  Sh stage;
  Sh ot, jac, Hv, gq, oc;
  Sh ps;
  Sh xc;  // current SQP iterate, n doubles appended after the layout
  double *Sg;  // S in global memory (DevStruct::sws), else null; set by the kernel after bind()

  __device__ __forceinline__ void bind(const Layout &L) {
    Js = Sh{L.Js}; Sm = Sh{L.S}; Als = Sh{L.Als};
    x = Sh{L.x}; xt = Sh{L.xt}; xt2 = Sh{L.xt2}; qh = Sh{L.qh}; D = Sh{L.D}; bx = Sh{L.bx};
    rb = Sh{L.rb}; lb = Sh{L.lb}; ub = Sh{L.ub}; zb = Sh{L.zb}; yb = Sh{L.yb}; Eb = Sh{L.Eb};
    dxv = Sh{L.dxv}; dyb = Sh{L.dyb}; xs = Sh{L.xs};
    El = Sh{L.El}; rl = Sh{L.rl}; ll = Sh{L.ll}; ul = Sh{L.ul}; zl = Sh{L.zl}; yl = Sh{L.yl};
    wl = Sh{L.wl}; dyl = Sh{L.dyl};
    Ep = Sh{L.Ep}; rp = Sh{L.rp}; lp = Sh{L.lp}; up = Sh{L.up}; zp = Sh{L.zp}; yp = Sh{L.yp};
    wp = Sh{L.wp}; bb = Sh{L.bb}; fv = Sh{L.fv}; dyp = Sh{L.dyp};
    s = Sh{L.s}; Ds = Sh{L.Ds}; sl = Sh{L.sl}; bs = Sh{L.bs}; zs = Sh{L.zs}; ys = Sh{L.ys};
    Es = Sh{L.Es}; gs = Sh{L.gs}; hs = Sh{L.hs}; rs = Sh{L.rs}; dss = Sh{L.dss}; dys = Sh{L.dys};
    Minv = Sh{L.Minv};
    red = Sh{L.red};
    msk = ShU32{L.msk};
    stage = Sh{L.stage};
    ot = Sh{L.ot}; jac = Sh{L.jac}; Hv = Sh{L.Hv}; gq = Sh{L.gq}; oc = Sh{L.oc};
    ps = Sh{L.ps};
    xc = Sh{L.total};
    Sg = nullptr;
  }
};
