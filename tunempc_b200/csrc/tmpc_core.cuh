// tmpc_core.cuh -- per-instance device routines of the batched tuned-MPC feedback solve (fp64).
//
// Everything here is written from scratch for this repository; the reference (jdeschut/tunempc) has no native
// or GPU code on this path.  What each routine replaces in the reference's Python:
//   tm_lin_pair      jacg_fun / H_fun evaluations through the RK4 integrator   tunempc/sqp_method.py:152,159,330
//   tm_qp_solve      conic('qpoases') QP solve                                 tunempc/sqp_method.py:158-168
//   tm_post          __linesearch (filter) + w/lam update                      tunempc/sqp_method.py:171-177,289-325
//   tm_conv          __check_convergence + __postprocessing stats              tunempc/sqp_method.py:240-287,185-221
//   tm_init          k = 0 bookkeeping of __check_convergence, __prefilter_lam_g   :223-238,248-261
//   tm_shift         Pmpc.__shift_initial_guess                                tunempc/pmpc.py:867-906
//
// Execution model: one WARP per instance for the sequential parts (QP, line search, convergence), one THREAD per
// (instance, stage, sensitivity pair) for the linearisation.  The warp routines are written against
// TM_LANE / TM_NL / TM_SYNC so that the same source compiles as a 1-lane sequential program with g++ for the
// CPU twin used by the CPU-only tests (tests/twin); that twin is test infrastructure, not a product path.
#pragma once
#include <stdint.h>
#include <math.h>
#include TMPC_MODEL_HEADER

#ifdef __CUDACC__
#define TM_HD __host__ __device__ __forceinline__
#define TM_HDN static __host__ __device__ __noinline__
#define TM_HDM __host__ __device__ __forceinline__
#else
#define TM_HDM inline
#define TM_HD static inline
#define TM_HDN static
#endif

#if defined(__CUDA_ARCH__) && !defined(TM_THREAD_MODE)
#define TM_WARP_MODE 1
#define TM_LANE ((int)(threadIdx.x & 31))
#define TM_NL 32
#define TM_SYNC() __syncwarp()
__device__ __forceinline__ double tm_wsum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double tm_wmax(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int tm_wsumi(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// arg-min over the warp: returns the smallest value and its payload (ties: smallest payload)
__device__ __forceinline__ void tm_wargmin(double& v, int& id) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, v, o);
    int oi = __shfl_xor_sync(0xffffffffu, id, o);
    if (ov < v || (ov == v && oi < id)) { v = ov; id = oi; }
  }
}
__device__ __forceinline__ int tm_wany(int p) { return __any_sync(0xffffffffu, p); }
#else
#define TM_LANE 0
#define TM_NL 1
#define TM_SYNC() ((void)0)
TM_HD double tm_wsum(double v) { return v; }
TM_HD double tm_wmax(double v) { return v; }
TM_HD int tm_wsumi(int v) { return v; }
TM_HD void tm_wargmin(double&, int&) {}
TM_HD int tm_wany(int p) { return p; }
#endif

// workspace accessor: plain pointer (shared memory, warp-per-instance; host twin) or a lane-interleaved view of global
// memory (thread-per-instance mode: element e of lane l lives at base[e*TM_WS_STRIDE + l], so a warp touching the same
// element of its 32 instances issues one coalesced 256-byte transaction)
#ifdef TM_WS_STRIDE
struct TmP {
  double* p;
  TM_HDM double& operator[](int i) const { return p[(size_t)i * TM_WS_STRIDE]; }
  TM_HDM double& operator[](size_t i) const { return p[i * TM_WS_STRIDE]; }
  TM_HDM TmP operator+(size_t o) const { TmP r; r.p = p + o * TM_WS_STRIDE; return r; }
  TM_HDM TmP operator+(int o) const { TmP r; r.p = p + (size_t)o * TM_WS_STRIDE; return r; }
};
TM_HD TmP tm_mkp(double* base, size_t off) { TmP r; r.p = base + off * TM_WS_STRIDE; return r; }
#else
typedef double* TmP;
TM_HD TmP tm_mkp(double* base, size_t off) { return base + off; }
#endif
typedef double* TmL;    // plain pointer in every mode (shared memory / host memory / thread-local scratch)

// Stage variables z_k = (x, u, us, usc) (tunempc/pmpc.py:217-235).  NU / NZ count every free variable of a stage block; the
// dynamics and the slacked nonlinear constraints depend on (x, u) only: NUM model inputs, NZM = NX + NUM.  Without slacks
// (NS = NSC = 0) the two coincide.  The linearisation code below is written against the model dimensions (NZ, NU are
// re-defined to NZM, NUM inside that region); TM_NZS is the stride of a stage block in W / D everywhere.
#ifndef TMPC_NUM
#define TMPC_NUM TMPC_NU
#define TMPC_NZM TMPC_NZ
#define TMPC_NS 0
#define TMPC_NSC 0
#endif
#define NX TMPC_NX
#define NU TMPC_NU
#define NZ TMPC_NZ
#define NUM TMPC_NUM
#define NZM TMPC_NZM
#define NS TMPC_NS
#define NSC TMPC_NSC
#define TM_NZS TMPC_NZ
#define TM_NPAIR (NZM * (NZM + 1) / 2)
#define TM_LSZ (NX + NX * NZM + TM_NPAIR)   /* per-stage linearisation record: xf | S row-major nx*nzm | W packed i<=j (model variables) */
#define TM_INF 1e300
#define TM_NCNT 24
#define TM_ALW 12  /* words of the augmented-Lagrangian row mask: supports N*nh <= 384 */

// ---------------------------------------------------------------------------------------------------------------
// problem constants and per-batch state (plain pointers; device memory in the product, malloc in the twin)
// ---------------------------------------------------------------------------------------------------------------
struct TmProb {
  int N, nh, nxt, p, n_w, n_g;
  int hessian_exact, max_iter, max_ls, filter_cap, maxact;
  int reg_mode;           // 8: primal active-set continuation of non-convex QPs for instances past TM_NONCONVEX_AFTER iterations (default); 24: for every instance; 0: Gauss-Newton re-solve only
  int lin_adjoint;        // 1: stage linearisation by the forward / adjoint sweep (tmpc_lin3.cuh), one task per stage
  int nonconvex_after;    // SQP iteration from which reg_mode 8 applies (default TM_NONCONVEX_AFTER)
  int economic;           // 1: stage cost = the model card's l(x,u) (economic MPC, pmpc.py:97-107), 0: tuned tracking cost (mtools.py:43-57)
  double tol, lam_tresh, beta, reg_tol, rho_rel;
  const double *wref, *H, *q, *ref_du, *C, *c;   // wref p*nz | H p*nz*nz (symmetric) | q p*nz | ref_du p*n_g | C nh*nz | c nh
  const int *term_idx, *relax0;
  const int* rowpin;      // nh: input index j if row i of C has its only non-zero on input j (a bound on one input), else -1
  unsigned long long* prof_counters;   // profiling builds (-DTM_PROF_W): [0] cycles of the Riccati block products inside the factorisation
};

struct TmState {
  int64_t B;
  int phase;              // index mod p of this step
  const double* X0;       // B*nx
  double *W, *LAM;        // B*n_w, B*n_g   current iterate (warm start before the step, solution after)
  double *D, *LAMQ;       // QP step and QP multipliers
  double* LIN;            // B*N*TM_LSZ
  double* G;              // B*n_g constraint values at the last evaluated point
  double* FILT;           // B*filter_cap*2
  double* fval;           // B
  int *nfilt, *iter, *status, *flags, *nAS, *nACtot, *nAC;
  int* qpstat;            // B: result of the last QP (0 ok)
  int* qpmode;            // B: 0 fresh, 1..3 retry with the stored row mask, 100 Gauss-Newton fallback
  int* qpwork;            // B: active-set iterations of the instance's last QP (scheduling key: the thread-per-instance
                          //    kernel is fed instances of similar cost so that the lanes of a warp stay in step)
  unsigned* almask;       // B*TM_ALW: augmented-Lagrangian row mask carried between retries
  int *list_retry, *cnt_retry;   // instances whose QP must be re-solved (filled by tm_qp)
  int pd_check;           // 1: the QP kernels run tm_pd_check instead of a QP (same workspace, same dispatch)
  unsigned* asinit;       // B*aswords bitmask of initially active inequality rows
  int aswords;
  int *list_next, *cnt_next, *list_relin, *cnt_relin;
  unsigned long long* counters;   // TM_NCNT: [0] iterations [4] ls dynamics evals [5] QP attempts [6] active-set iterations [7] Riccati solves [8..19] attempt histogram
};

// g = [init(nx) | k < N: dyn_k(nx), g_k(ns), h_k(nh) | term(nx_term)]   (tunempc/pmpc.py:242-256,279-287)
#define TM_GS(P) (NX + NS + (P).nh)     /* rows per stage */
TM_HD int tm_gdyn(const TmProb& P, int k) { return NX + k * TM_GS(P); }
TM_HD int tm_gg(const TmProb& P, int k) { return NX + k * TM_GS(P) + NX; }
TM_HD int tm_gh(const TmProb& P, int k) { return NX + k * TM_GS(P) + NX + NS; }
TM_HD int tm_gterm(const TmProb& P) { return NX + P.N * TM_GS(P); }

// ---- model-dimension region: NZ, NU mean NZM, NUM down to the matching pop_macro ------------------------------------
#pragma push_macro("NZ")
#pragma push_macro("NU")
#undef NZ
#undef NU
#define NZ TMPC_NZM
#define NU TMPC_NUM

TM_HD void tm_pair_ij(int pr, int& i, int& j) {   // packed upper-triangular index -> (i<=j), row-major
  int r = 0, rem = pr;
  while (rem >= NZ - r) { rem -= NZ - r; ++r; }
  i = r; j = r + rem;
}
TM_HD int tm_pair_idx(int i, int j) {             // requires i<=j
  return i * NZ - i * (i - 1) / 2 + (j - i);
}

// ---------------------------------------------------------------------------------------------------------------
// K1: stage linearisation.  One call = one (stage, pair (i,j)) task: integrates x, s_i = dx/dz_i, s_j, t_ij = d2x/dz_i dz_j
// through RK4 (or one map evaluation for a discrete model).  ORDER 0: value; 1: + s_i; 2: + s_j and t_ij.
// ---------------------------------------------------------------------------------------------------------------
template <int ORDER>
TM_HD void tm_rhs(const double* X, const double* u, const double* Si, const double* Sj, const double* T, int i, int j,
                  double* k, double* dki, double* dkj, double* ddk) {
  if (ORDER == 0) { tmpc_ode(X, u, k); return; }
  double J[NX * NZ];
  double Hn[TMPC_NHESS > 0 ? TMPC_NHESS : 1];
  if (ORDER == 1) tmpc_ode_jac(X, u, k, J); else tmpc_ode_d2(X, u, k, J, Hn);
  double vi[NZ], vj[NZ];
#pragma unroll
  for (int a = 0; a < NX; ++a) { vi[a] = Si[a]; vj[a] = (ORDER == 2) ? Sj[a] : 0.0; }
#pragma unroll
  for (int b = 0; b < NU; ++b) { vi[NX + b] = (i == NX + b) ? 1.0 : 0.0; vj[NX + b] = (j == NX + b) ? 1.0 : 0.0; }
#pragma unroll
  for (int a = 0; a < NX; ++a) {
    double s = 0.0;
#pragma unroll
    for (int b = 0; b < NZ; ++b) s += J[a * NZ + b] * vi[b];
    dki[a] = s;
  }
  if (ORDER == 2) {
#pragma unroll
    for (int a = 0; a < NX; ++a) {
      double s = 0.0;
#pragma unroll
      for (int b = 0; b < NZ; ++b) s += J[a * NZ + b] * vj[b];
      dkj[a] = s;
    }
    tmpc_ode_bilin(Hn, vi, vj, ddk);
#pragma unroll
    for (int a = 0; a < NX; ++a) {
      double s = ddk[a];
#pragma unroll
      for (int b = 0; b < NX; ++b) s += J[a * NZ + b] * T[b];
      ddk[a] = s;
    }
  }
}


#ifndef TMPC_COLLOCATION
#define TMPC_COLLOCATION 0
#endif
#define TMPC_RK4 (!TMPC_DISCRETE && !TMPC_COLLOCATION)

#if TMPC_COLLOCATION
// ---------------------------------------------------------------------------------------------------------------
// CasADi integrator('F','collocation',ode,{'tf':..}) (reference: examples/evaporation_process/main.py:103): TMPC_RK_STEPS
// finite elements, Radau points of interpolation order 3 per element = the 3-stage Radau IIA method, solved to
// convergence by Newton.  Stage derivatives K_j = f(x + h sum_l a_jl K_l, u).  Sensitivities by the implicit function
// theorem with the converged iteration matrix M = I - h (a_jl J_j):  M dK_i = J_j v_i,  M ddK = f_zz[v_i, v_j] + J_x,j T.
// ---------------------------------------------------------------------------------------------------------------
#define TM_CN (3 * NX)
TM_HD void tm_lu_factor(double* M, int* piv) {          // row-major TM_CN x TM_CN, partial pivoting, in place
  for (int c = 0; c < TM_CN; ++c) {
    int p = c;
    double best = fabs(M[c * TM_CN + c]);
    for (int r = c + 1; r < TM_CN; ++r) { const double v = fabs(M[r * TM_CN + c]); if (v > best) { best = v; p = r; } }
    piv[c] = p;
    if (p != c) for (int k = 0; k < TM_CN; ++k) { const double t = M[c * TM_CN + k]; M[c * TM_CN + k] = M[p * TM_CN + k]; M[p * TM_CN + k] = t; }
    const double d = 1.0 / M[c * TM_CN + c];
    for (int r = c + 1; r < TM_CN; ++r) {
      const double f = M[r * TM_CN + c] * d;
      M[r * TM_CN + c] = f;
      for (int k = c + 1; k < TM_CN; ++k) M[r * TM_CN + k] -= f * M[c * TM_CN + k];
    }
  }
}
TM_HD void tm_lu_solve(const double* M, const int* piv, double* b) {
  for (int c = 0; c < TM_CN; ++c) {
    const int p = piv[c];
    if (p != c) { const double t = b[c]; b[c] = b[p]; b[p] = t; }
    for (int r = c + 1; r < TM_CN; ++r) b[r] -= M[r * TM_CN + c] * b[c];
  }
  for (int r = TM_CN - 1; r >= 0; --r) {
    double v = b[r];
    for (int k = r + 1; k < TM_CN; ++k) v -= M[r * TM_CN + k] * b[k];
    b[r] = v / M[r * TM_CN + r];
  }
}

template <int ORDER>
TM_HD void tm_integrate_colloc(const double* u, int i, int j, double* X, double* Si, double* Sj, double* T) {
  const double sq6 = 2.449489742783178;
  const double A[3][3] = {{(88.0 - 7.0 * sq6) / 360.0, (296.0 - 169.0 * sq6) / 1800.0, (-2.0 + 3.0 * sq6) / 225.0},
                          {(296.0 + 169.0 * sq6) / 1800.0, (88.0 + 7.0 * sq6) / 360.0, (-2.0 - 3.0 * sq6) / 225.0},
                          {(16.0 - sq6) / 36.0, (16.0 + sq6) / 36.0, 1.0 / 9.0}};
  const double h = TMPC_RK_DT;
  for (int s = 0; s < TMPC_RK_STEPS; ++s) {
    double K[3][NX], Jst[3][NX * NZ], M[TM_CN * TM_CN], rhs[TM_CN];
    double Hst[3][TMPC_NHESS > 0 ? TMPC_NHESS : 1];
    int piv[TM_CN];
    {
      double f0[NX];
      tmpc_ode(X, u, f0);
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) K[q][a] = f0[a];
    }
    // Newton to convergence; the last pass (done = 1) re-evaluates J (and d2f) at the converged stage points
    int done = 0;
    for (int it = 0; it < 40; ++it) {
      for (int q = 0; q < 3; ++q) {
        double Xq[NX], fq[NX];
        for (int a = 0; a < NX; ++a) {
          double v = X[a];
          for (int l = 0; l < 3; ++l) v += h * A[q][l] * K[l][a];
          Xq[a] = v;
        }
        if (done && ORDER == 2) tmpc_ode_d2(Xq, u, fq, Jst[q], Hst[q]); else tmpc_ode_jac(Xq, u, fq, Jst[q]);
        for (int a = 0; a < NX; ++a) rhs[q * NX + a] = -(K[q][a] - fq[a]);
      }
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) for (int l = 0; l < 3; ++l) for (int b = 0; b < NX; ++b)
        M[(q * NX + a) * TM_CN + l * NX + b] = ((q == l && a == b) ? 1.0 : 0.0) - h * A[q][l] * Jst[q][a * NZ + b];
      tm_lu_factor(M, piv);
      if (done) break;
      tm_lu_solve(M, piv, rhs);
      double dmax = 0.0, kmax = 1.0;
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) {
        K[q][a] += rhs[q * NX + a];
        dmax = fmax(dmax, fabs(rhs[q * NX + a]));
        kmax = fmax(kmax, fabs(K[q][a]));
      }
      if (!(dmax > 1e-14 * kmax)) done = 1;
      if (it == 38) done = 1;
    }
    double dKi[TM_CN], dKj[TM_CN], ddK[TM_CN];
    if (ORDER >= 1) {
      // stage-argument directions need dK, so solve first, then form v
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) {
        double t = 0.0;
        for (int b = 0; b < NX; ++b) t += Jst[q][a * NZ + b] * Si[b];
        if (i >= NX) t += Jst[q][a * NZ + i];
        dKi[q * NX + a] = t;
      }
      tm_lu_solve(M, piv, dKi);
    }
    if (ORDER >= 2) {
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) {
        double t = 0.0;
        for (int b = 0; b < NX; ++b) t += Jst[q][a * NZ + b] * Sj[b];
        if (j >= NX) t += Jst[q][a * NZ + j];
        dKj[q * NX + a] = t;
      }
      tm_lu_solve(M, piv, dKj);
      for (int q = 0; q < 3; ++q) {
        double vi[NZ], vj[NZ], dd[NX];
        for (int a = 0; a < NX; ++a) {
          double ti = Si[a], tj = Sj[a];
          for (int l = 0; l < 3; ++l) { ti += h * A[q][l] * dKi[l * NX + a]; tj += h * A[q][l] * dKj[l * NX + a]; }
          vi[a] = ti; vj[a] = tj;
        }
        for (int b = 0; b < NU; ++b) { vi[NX + b] = (i == NX + b) ? 1.0 : 0.0; vj[NX + b] = (j == NX + b) ? 1.0 : 0.0; }
        tmpc_ode_bilin(Hst[q], vi, vj, dd);
        for (int a = 0; a < NX; ++a) {
          double t = dd[a];
          for (int b = 0; b < NX; ++b) t += Jst[q][a * NZ + b] * T[b];
          ddK[q * NX + a] = t;
        }
      }
      tm_lu_solve(M, piv, ddK);
    }
    for (int a = 0; a < NX; ++a) {
      for (int q = 0; q < 3; ++q) {
        X[a] += h * A[2][q] * K[q][a];
        if (ORDER >= 1) Si[a] += h * A[2][q] * dKi[q * NX + a];
        if (ORDER >= 2) { Sj[a] += h * A[2][q] * dKj[q * NX + a]; T[a] += h * A[2][q] * ddK[q * NX + a]; }
      }
    }
  }
}
#endif

#if TMPC_COLLOCATION
// Whole linearisation record of one stage in ONE task: the Newton solve and the LU factorisation of an element are done
// once and shared by all NZ first-order and NZ(NZ+1)/2 second-order right-hand sides (the pair-per-task route repeats
// them for every pair).  order 1: xf, S;  order 2: + W = lam' d2F/dz2.  rec layout as everywhere: xf | S row-major | W.
TM_HD void tm_colloc_stage(const double* x0, const double* u, int order, const double* lam, double* rec) {
  const double sq6 = 2.449489742783178;
  const double A[3][3] = {{(88.0 - 7.0 * sq6) / 360.0, (296.0 - 169.0 * sq6) / 1800.0, (-2.0 + 3.0 * sq6) / 225.0},
                          {(296.0 + 169.0 * sq6) / 1800.0, (88.0 + 7.0 * sq6) / 360.0, (-2.0 - 3.0 * sq6) / 225.0},
                          {(16.0 - sq6) / 36.0, (16.0 + sq6) / 36.0, 1.0 / 9.0}};
  const double h = TMPC_RK_DT;
  double X[NX], Sm[NZ][NX], Tm[TM_NPAIR][NX];
  for (int a = 0; a < NX; ++a) X[a] = x0[a];
  for (int i = 0; i < NZ; ++i) for (int a = 0; a < NX; ++a) Sm[i][a] = (a == i) ? 1.0 : 0.0;
  for (int p = 0; p < TM_NPAIR; ++p) for (int a = 0; a < NX; ++a) Tm[p][a] = 0.0;
  for (int s = 0; s < TMPC_RK_STEPS; ++s) {
    double K[3][NX], Jst[3][NX * NZ], M[TM_CN * TM_CN], rhs[TM_CN];
    double Hst[3][TMPC_NHESS > 0 ? TMPC_NHESS : 1];
    int piv[TM_CN];
    {
      double f0[NX];
      tmpc_ode(X, u, f0);
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) K[q][a] = f0[a];
    }
    int done = 0;
    for (int it = 0; it < 40; ++it) {                  // same Newton iteration as tm_integrate_colloc
      for (int q = 0; q < 3; ++q) {
        double Xq[NX], fq[NX];
        for (int a = 0; a < NX; ++a) {
          double v = X[a];
          for (int l = 0; l < 3; ++l) v += h * A[q][l] * K[l][a];
          Xq[a] = v;
        }
        if (done && order == 2) tmpc_ode_d2(Xq, u, fq, Jst[q], Hst[q]); else tmpc_ode_jac(Xq, u, fq, Jst[q]);
        for (int a = 0; a < NX; ++a) rhs[q * NX + a] = -(K[q][a] - fq[a]);
      }
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) for (int l = 0; l < 3; ++l) for (int b = 0; b < NX; ++b)
        M[(q * NX + a) * TM_CN + l * NX + b] = ((q == l && a == b) ? 1.0 : 0.0) - h * A[q][l] * Jst[q][a * NZ + b];
      tm_lu_factor(M, piv);
      if (done) break;
      tm_lu_solve(M, piv, rhs);
      double dmax = 0.0, kmax = 1.0;
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) {
        K[q][a] += rhs[q * NX + a];
        dmax = fmax(dmax, fabs(rhs[q * NX + a]));
        kmax = fmax(kmax, fabs(K[q][a]));
      }
      if (!(dmax > 1e-14 * kmax)) done = 1;
      if (it == 38) done = 1;
    }
    // first order: all NZ directions against the same factorisation; V[i][q] = stage-argument direction
    double dK[NZ][TM_CN], V[NZ][3][NZ];
    for (int i = 0; i < NZ; ++i) {
      for (int q = 0; q < 3; ++q) for (int a = 0; a < NX; ++a) {
        double t = 0.0;
        for (int b = 0; b < NX; ++b) t += Jst[q][a * NZ + b] * Sm[i][b];
        if (i >= NX) t += Jst[q][a * NZ + i];
        dK[i][q * NX + a] = t;
      }
      tm_lu_solve(M, piv, dK[i]);
      for (int q = 0; q < 3; ++q) {
        for (int a = 0; a < NX; ++a) {
          double t = Sm[i][a];
          for (int l = 0; l < 3; ++l) t += h * A[q][l] * dK[i][l * NX + a];
          V[i][q][a] = t;
        }
        for (int b = 0; b < NU; ++b) V[i][q][NX + b] = (i == NX + b) ? 1.0 : 0.0;
      }
    }
    if (order == 2) {
      for (int i = 0; i < NZ; ++i)
        for (int j = i; j < NZ; ++j) {
          const int p = tm_pair_idx(i, j);
          double ddK[TM_CN];
          for (int q = 0; q < 3; ++q) {
            double dd[NX];
            tmpc_ode_bilin(Hst[q], V[i][q], V[j][q], dd);
            for (int a = 0; a < NX; ++a) {
              double t = dd[a];
              for (int b = 0; b < NX; ++b) t += Jst[q][a * NZ + b] * Tm[p][b];
              ddK[q * NX + a] = t;
            }
          }
          tm_lu_solve(M, piv, ddK);
          for (int a = 0; a < NX; ++a) for (int q = 0; q < 3; ++q) Tm[p][a] += h * A[2][q] * ddK[q * NX + a];
        }
    }
    for (int a = 0; a < NX; ++a)
      for (int q = 0; q < 3; ++q) {
        X[a] += h * A[2][q] * K[q][a];
        for (int i = 0; i < NZ; ++i) Sm[i][a] += h * A[2][q] * dK[i][q * NX + a];
      }
  }
  for (int a = 0; a < NX; ++a) rec[a] = X[a];
  for (int a = 0; a < NX; ++a) for (int i = 0; i < NZ; ++i) rec[NX + a * NZ + i] = Sm[i][a];
  if (order == 2)
    for (int p = 0; p < TM_NPAIR; ++p) {
      double wij = 0.0;
      for (int a = 0; a < NX; ++a) wij += lam[a] * Tm[p][a];
      rec[NX + NX * NZ + p] = wij;
    }
}
#endif

template <int ORDER>
TM_HD void tm_integrate(const double* x0, const double* u, int i, int j, double* X, double* Si, double* Sj, double* T) {
#pragma unroll
  for (int a = 0; a < NX; ++a) { X[a] = x0[a]; Si[a] = (a == i) ? 1.0 : 0.0; Sj[a] = (a == j) ? 1.0 : 0.0; T[a] = 0.0; }
#if TMPC_DISCRETE
  {
    double k[NX], di[NX], dj[NX], dd[NX];
    tm_rhs<ORDER>(X, u, Si, Sj, T, i, j, k, di, dj, dd);
#pragma unroll
    for (int a = 0; a < NX; ++a) {
      X[a] = k[a];
      if (ORDER >= 1) Si[a] = di[a];
      if (ORDER >= 2) { Sj[a] = dj[a]; T[a] = dd[a]; }
    }
  }
#elif TMPC_COLLOCATION
  tm_integrate_colloc<ORDER>(u, i, j, X, Si, Sj, T);
#else
  const double h = TMPC_RK_DT;
  for (int s = 0; s < TMPC_RK_STEPS; ++s) {
    double aX[NX], aI[NX], aJ[NX], aT[NX];      // accumulated increment (k1 + 2k2 + 2k3 + k4)
    double k[NX], di[NX], dj[NX], dd[NX];       // current stage derivative
    double Xs[NX], Is[NX], Js[NX], Ts[NX];      // stage argument
#pragma unroll
    for (int a = 0; a < NX; ++a) { Xs[a] = X[a]; Is[a] = Si[a]; Js[a] = Sj[a]; Ts[a] = T[a]; di[a] = dj[a] = dd[a] = 0.0; }
#pragma unroll
    for (int st = 0; st < 4; ++st) {
      tm_rhs<ORDER>(Xs, u, Is, Js, Ts, i, j, k, di, dj, dd);
      const double wgt = (st == 0 || st == 3) ? 1.0 : 2.0;
      const double cn = (st == 2) ? 1.0 : 0.5;  // coefficient of the NEXT stage argument
#pragma unroll
      for (int a = 0; a < NX; ++a) {
        if (st == 0) { aX[a] = k[a]; aI[a] = di[a]; aJ[a] = dj[a]; aT[a] = dd[a]; }
        else { aX[a] += wgt * k[a]; aI[a] += wgt * di[a]; aJ[a] += wgt * dj[a]; aT[a] += wgt * dd[a]; }
        if (st < 3) {
          Xs[a] = X[a] + cn * h * k[a];
          if (ORDER >= 1) Is[a] = Si[a] + cn * h * di[a];
          if (ORDER >= 2) { Js[a] = Sj[a] + cn * h * dj[a]; Ts[a] = T[a] + cn * h * dd[a]; }
        }
      }
    }
#pragma unroll
    for (int a = 0; a < NX; ++a) {
      X[a] += h / 6.0 * aX[a];
      if (ORDER >= 1) Si[a] += h / 6.0 * aI[a];
      if (ORDER >= 2) { Sj[a] += h / 6.0 * aJ[a]; T[a] += h / 6.0 * aT[a]; }
    }
  }
#endif
}

// ---- grouped linearisation: one task integrates x, up to TMPC_LIN_D first-order directions and up to TMPC_LIN_PP
// second-order pairs among them, so the ODE, its Jacobian and its second derivatives are evaluated once per group
// (TMPC_LIN_NG groups cover all NZ(NZ+1)/2 pairs; tables generated by modelgen.lin_groups).
#define TM_LD TMPC_LIN_D
#define TM_LP TMPC_LIN_PP
TM_HD constexpr int tm_g_nd(int g) { constexpr int t[] = TMPC_LIN_GND; return t[g]; }
TM_HD constexpr int tm_g_np(int g) { constexpr int t[] = TMPC_LIN_GNP; return t[g]; }
TM_HD constexpr int tm_g_dir(int g, int a) { constexpr int t[] = TMPC_LIN_GD; return t[g * TM_LD + a]; }
TM_HD constexpr int tm_g_own(int g, int a) { constexpr int t[] = TMPC_LIN_GOWN; return t[g * TM_LD + a]; }
TM_HD constexpr int tm_g_pa(int g, int p) { constexpr int t[] = TMPC_LIN_GPA; return t[g * TM_LP + p]; }
TM_HD constexpr int tm_g_pb(int g, int p) { constexpr int t[] = TMPC_LIN_GPB; return t[g * TM_LP + p]; }
TM_HD constexpr int tm_g_pi(int g, int p) { constexpr int t[] = TMPC_LIN_GPI; return t[g * TM_LP + p]; }

// derivative of the group state at stage argument (Xs, Ss, Ts).  ND directions with global ids dir[a]
template <int ND, int NP, class DirF, class PaF, class PbF>
TM_HD void tm_rhs_group(const double* Xs, const double* u, const double (*Ss)[NX], const double (*Ts)[NX], DirF dir, PaF pa,
                        PbF pb, double* k, double (*dS)[NX], double (*dT)[NX]) {
  double J[NX * NZ];
  double Hn[TMPC_NHESS > 0 ? TMPC_NHESS : 1];
  if (NP > 0) tmpc_ode_d2(Xs, u, k, J, Hn); else tmpc_ode_jac(Xs, u, k, J);
  double v[ND > 0 ? ND : 1][NZ];
#pragma unroll
  for (int a = 0; a < ND; ++a) {
#pragma unroll
    for (int i = 0; i < NX; ++i) v[a][i] = Ss[a][i];
#pragma unroll
    for (int b = 0; b < NU; ++b) v[a][NX + b] = (dir(a) == NX + b) ? 1.0 : 0.0;
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      double t = 0.0;
#pragma unroll
      for (int b = 0; b < NZ; ++b) t += J[i * NZ + b] * v[a][b];
      dS[a][i] = t;
    }
  }
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    double dd[NX];
    tmpc_ode_bilin(Hn, v[pa(p)], v[pb(p)], dd);
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      double t = dd[i];
#pragma unroll
      for (int b = 0; b < NX; ++b) t += J[i * NZ + b] * Ts[p][b];
      dT[p][i] = t;
    }
  }
}

template <int ND, int NP, class DirF, class PaF, class PbF>
TM_HD void tm_integrate_group(const double* x0, const double* u, DirF dir, PaF pa, PbF pb, double* X, double (*S)[NX],
                              double (*T)[NX]) {
#pragma unroll
  for (int i = 0; i < NX; ++i) X[i] = x0[i];
#pragma unroll
  for (int a = 0; a < ND; ++a)
#pragma unroll
    for (int i = 0; i < NX; ++i) S[a][i] = (dir(a) == i) ? 1.0 : 0.0;
#pragma unroll
  for (int p = 0; p < NP; ++p)
#pragma unroll
    for (int i = 0; i < NX; ++i) T[p][i] = 0.0;
#if TMPC_DISCRETE
  {
    double k[NX], dS[ND > 0 ? ND : 1][NX], dT[NP > 0 ? NP : 1][NX];
    tm_rhs_group<ND, NP>(X, u, S, T, dir, pa, pb, k, dS, dT);
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      X[i] = k[i];
#pragma unroll
      for (int a = 0; a < ND; ++a) S[a][i] = dS[a][i];
#pragma unroll
      for (int p = 0; p < NP; ++p) T[p][i] = dT[p][i];
    }
  }
#else
  const double h = TMPC_RK_DT;
  for (int s = 0; s < TMPC_RK_STEPS; ++s) {
    double aX[NX], aS[ND > 0 ? ND : 1][NX], aT[NP > 0 ? NP : 1][NX];
    double k[NX], dS[ND > 0 ? ND : 1][NX], dT[NP > 0 ? NP : 1][NX];
    double Xs[NX], Ss[ND > 0 ? ND : 1][NX], Ts[NP > 0 ? NP : 1][NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      Xs[i] = X[i];
#pragma unroll
      for (int a = 0; a < ND; ++a) Ss[a][i] = S[a][i];
#pragma unroll
      for (int p = 0; p < NP; ++p) Ts[p][i] = T[p][i];
    }
#pragma unroll
    for (int st = 0; st < 4; ++st) {
      tm_rhs_group<ND, NP>(Xs, u, Ss, Ts, dir, pa, pb, k, dS, dT);
      const double wgt = (st == 0 || st == 3) ? 1.0 : 2.0;
      const double cn = (st == 2) ? 1.0 : 0.5;
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        aX[i] = (st == 0) ? k[i] : aX[i] + wgt * k[i];
        if (st < 3) Xs[i] = X[i] + cn * h * k[i];
#pragma unroll
        for (int a = 0; a < ND; ++a) {
          aS[a][i] = (st == 0) ? dS[a][i] : aS[a][i] + wgt * dS[a][i];
          if (st < 3) Ss[a][i] = S[a][i] + cn * h * dS[a][i];
        }
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          aT[p][i] = (st == 0) ? dT[p][i] : aT[p][i] + wgt * dT[p][i];
          if (st < 3) Ts[p][i] = T[p][i] + cn * h * dT[p][i];
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      X[i] += h / 6.0 * aX[i];
#pragma unroll
      for (int a = 0; a < ND; ++a) S[a][i] += h / 6.0 * aS[a][i];
#pragma unroll
      for (int p = 0; p < NP; ++p) T[p][i] += h / 6.0 * aT[p][i];
    }
  }
#endif
}

// exact-Hessian group G: writes its owned S columns, its W entries and (group 0) xf
template <int G>
TM_HD void tm_lin_group_exact(const double* x, const double* u, const double* lam, double* rec) {
  constexpr int ND = tm_g_nd(G), NP = tm_g_np(G);
  double X[NX], S[ND][NX], T[NP][NX];
  tm_integrate_group<ND, NP>(x, u, [](int a) { return tm_g_dir(G, a); }, [](int p) { return tm_g_pa(G, p); },
                             [](int p) { return tm_g_pb(G, p); }, X, S, T);
#pragma unroll
  for (int p = 0; p < NP; ++p) {
    double wij = 0.0;
#pragma unroll
    for (int i = 0; i < NX; ++i) wij += lam[i] * T[p][i];
    rec[NX + NX * NZ + tm_g_pi(G, p)] = wij;
  }
#pragma unroll
  for (int a = 0; a < ND; ++a)
    if (tm_g_own(G, a)) {
#pragma unroll
      for (int i = 0; i < NX; ++i) rec[NX + i * NZ + tm_g_dir(G, a)] = S[a][i];
    }
  if (G == 0) {
#pragma unroll
    for (int i = 0; i < NX; ++i) rec[i] = X[i];
  }
}

// Gauss-Newton group g: directions 3g .. 3g+2 (first order only)
#define TM_GN_NG ((NZ + 2) / 3)
template <int G>
TM_HD void tm_lin_group_gn(const double* x, const double* u, double* rec) {
  constexpr int ND = (NZ - 3 * G) < 3 ? (NZ - 3 * G) : 3;
#if TMPC_COLLOCATION
  for (int a = 0; a < ND; ++a) {                     // implicit integrator: one direction at a time
    double Xc[NX], Sc[NX], t1[NX], t2[NX];
    tm_integrate<1>(x, u, 3 * G + a, 3 * G + a, Xc, Sc, t1, t2);
    for (int i = 0; i < NX; ++i) rec[NX + i * NZ + 3 * G + a] = Sc[i];
    if (G == 0 && a == 0) for (int i = 0; i < NX; ++i) rec[i] = Xc[i];
  }
  return;
#endif
  double X[NX], S[ND][NX], T[1][NX];
  tm_integrate_group<ND, 0>(x, u, [](int a) { return 3 * G + a; }, [](int) { return 0; }, [](int) { return 0; }, X, S, T);
#pragma unroll
  for (int a = 0; a < ND; ++a)
#pragma unroll
    for (int i = 0; i < NX; ++i) rec[NX + i * NZ + 3 * G + a] = S[a][i];
  if (G == 0) {
#pragma unroll
    for (int i = 0; i < NX; ++i) rec[i] = X[i];
  }
}

#if TMPC_COLLOCATION
TM_HD int tm_lin_tasks_per_stage(int) { return 1; }     // tm_colloc_stage: the whole record in one task
#elif defined(TMPC_LIN_GROUPED)
TM_HD int tm_lin_tasks_per_stage(int hessian_exact) { return hessian_exact ? TMPC_LIN_NG : TM_GN_NG; }
#else
TM_HD int tm_lin_tasks_per_stage(int hessian_exact) { return hessian_exact ? TM_NPAIR : TM_GN_NG; }
#endif

#include "tmpc_lin3.cuh"

// one linearisation task.  trial = 1: evaluate at (W + D, LAMQ), else at (W, LAM).  g = group id.
TM_HD void tm_lin_task(const TmProb& P, const TmState& S, int64_t inst, int k, int g, int trial) {
  const double* w = S.W + inst * P.n_w + (int64_t)k * TM_NZS;
  double x[NX], u[NU];
#pragma unroll
  for (int a = 0; a < NX; ++a) x[a] = w[a];
#pragma unroll
  for (int b = 0; b < NU; ++b) u[b] = w[NX + b];
  if (trial && S.qpstat[inst] != 0) return;   // failed QP: keep LIN at W for the final statistics
  if (trial) {
    const double* d = S.D + inst * P.n_w + (int64_t)k * TM_NZS;
#pragma unroll
    for (int a = 0; a < NX; ++a) x[a] += d[a];
#pragma unroll
    for (int b = 0; b < NU; ++b) u[b] += d[NX + b];
  }
  double* rec = S.LIN + (inst * P.N + k) * (int64_t)TM_LSZ;
#if TMPC_RK4
  if (P.lin_adjoint) {
    if (g != 0) return;
    double lamv[NX];
    const double* lamq = (trial ? S.LAMQ : S.LAM) + inst * P.n_g + tm_gdyn(P, k);
#pragma unroll
    for (int a = 0; a < NX; ++a) lamv[a] = P.hessian_exact ? lamq[a] : 0.0;
    tm_lin_adjoint(x, u, P.hessian_exact ? 2 : 1, lamv, rec);
    return;
  }
#endif
#if TMPC_COLLOCATION
  {
    double lamc[NX];
    const double* lamq = (trial ? S.LAMQ : S.LAM) + inst * P.n_g + tm_gdyn(P, k);
    for (int a = 0; a < NX; ++a) lamc[a] = P.hessian_exact ? lamq[a] : 0.0;
    tm_colloc_stage(x, u, P.hessian_exact ? 2 : 1, lamc, rec);
    (void)g;
    return;
  }
#endif
  if (P.hessian_exact) {
    const double* lamp = (trial ? S.LAMQ : S.LAM) + inst * P.n_g + tm_gdyn(P, k);
    double lam[NX];
#pragma unroll
    for (int a = 0; a < NX; ++a) lam[a] = lamp[a];
    // one (i,j) pair per thread: 164 registers, no spills, FP64 pipe 82 % busy.  The grouped variant
    // (tm_lin_group_exact: 3 directions + 3-4 pairs per thread, half the flops) needs 255 registers, spills, and ran
    // 3.5x slower on B200 (profiles/r01b_summary.md) -- kept for models with a cheaper right-hand side.
#ifdef TMPC_LIN_GROUPED
    switch (g) {
      case 0: tm_lin_group_exact<0>(x, u, lam, rec); break;
#if TMPC_LIN_NG > 1
      case 1: tm_lin_group_exact<1>(x, u, lam, rec); break;
#endif
#if TMPC_LIN_NG > 2
      case 2: tm_lin_group_exact<2>(x, u, lam, rec); break;
#endif
#if TMPC_LIN_NG > 3
      case 3: tm_lin_group_exact<3>(x, u, lam, rec); break;
#endif
#if TMPC_LIN_NG > 4
      case 4: tm_lin_group_exact<4>(x, u, lam, rec); break;
#endif
#if TMPC_LIN_NG > 5
      case 5: tm_lin_group_exact<5>(x, u, lam, rec); break;
#endif
#if TMPC_LIN_NG > 6
      case 6: tm_lin_group_exact<6>(x, u, lam, rec); break;
#endif
#if TMPC_LIN_NG > 7
      case 7: tm_lin_group_exact<7>(x, u, lam, rec); break;
#endif
      default: break;
    }
#else
    {
      int i, j;
      tm_pair_ij(g, i, j);
      double X[NX], Si[NX], Sj[NX], T[NX];
      tm_integrate<2>(x, u, i, j, X, Si, Sj, T);
      double wij = 0.0;
#pragma unroll
      for (int a = 0; a < NX; ++a) wij += lam[a] * T[a];
      rec[NX + NX * NZ + g] = wij;
      if (i == j) {
#pragma unroll
        for (int a = 0; a < NX; ++a) rec[NX + a * NZ + i] = Si[a];
      }
      if (g == 0) {
#pragma unroll
        for (int a = 0; a < NX; ++a) rec[a] = X[a];
      }
    }
#endif
  } else {
    switch (g) {
      case 0: tm_lin_group_gn<0>(x, u, rec); break;
#if (TMPC_NZM > 3)
      case 1: tm_lin_group_gn<1>(x, u, rec); break;
#endif
#if (TMPC_NZM > 6)
      case 2: tm_lin_group_gn<2>(x, u, rec); break;
#endif
#if (TMPC_NZM > 9)
      case 3: tm_lin_group_gn<3>(x, u, rec); break;
#endif
#if (TMPC_NZM > 12)
#error "more than 4 Gauss-Newton groups: extend the dispatch in tm_lin_task"
#endif
      default: break;
    }
  }
}

#pragma pop_macro("NU")
#pragma pop_macro("NZ")
// ---- end of the model-dimension region ----------------------------------------------------------------------------

#include "tmpc_qp.cuh"

// ---------------------------------------------------------------------------------------------------------------
// objective and infeasibility of a point w_t = W + alpha*D.  xf_from_lin: take F(x_k,u_k) from LIN (valid for the
// point LIN was evaluated at), else integrate (lane <-> stage).  Writes g (n_g) when gout != nullptr.
// ---------------------------------------------------------------------------------------------------------------
TM_HD void tm_eval_point(const TmProb& P, const TmState& S, int64_t inst, double alpha, int xf_from_lin,
                         double* gout, double& f_out, double& viol_out) {
  const int N = P.N, nh = P.nh;
  const int lane = TM_LANE;
  const double* w = S.W + inst * P.n_w;
  const double* d = S.D + inst * P.n_w;
  const double* lin = S.LIN + inst * P.N * (int64_t)TM_LSZ;
  double f = 0.0, viol = 0.0;
  for (int k = lane; k < N; k += TM_NL) {
    double z[NZ], xn[NX], xf[NX];
#pragma unroll
    for (int b = 0; b < NZ; ++b) z[b] = w[k * NZ + b] + (alpha != 0.0 ? alpha * d[k * NZ + b] : 0.0);
#pragma unroll
    for (int a = 0; a < NX; ++a) xn[a] = w[(k + 1) * NZ + a] + (alpha != 0.0 ? alpha * d[(k + 1) * NZ + a] : 0.0);
    if (xf_from_lin) {
#pragma unroll
      for (int a = 0; a < NX; ++a) xf[a] = lin[(size_t)k * TM_LSZ + a];
    } else {
      double t1[NX], t2[NX], t3[NX];
      tm_integrate<0>(z, z + NX, 0, 0, xf, t1, t2, t3);
    }
    const int ph = (S.phase + k) % P.p;
    const double* Hk = P.H + (size_t)ph * NZ * NZ;
    const double* wr = P.wref + (size_t)ph * NZ;
    const double* qk = P.q + (size_t)ph * NZ;
    double dz[NZ];
#pragma unroll
    for (int b = 0; b < NZ; ++b) dz[b] = z[b] - wr[b];
    double fk = 0.0;
    if (P.economic) {
      fk = tmpc_stage_cost(z, z + NX);
#pragma unroll
      for (int b = NZM + NS; b < NZ; ++b) fk += qk[b] * z[b];    // scost'usc (pmpc.py:338-339)
    } else {
#pragma unroll
      for (int a = 0; a < NZ; ++a) {
        double t = 0.0;
#pragma unroll
        for (int b = 0; b < NZ; ++b) t += Hk[a * NZ + b] * dz[b];
        fk += dz[a] * (0.5 * t + qk[a]);
      }
    }
    f += fk;
#pragma unroll
    for (int a = 0; a < NX; ++a) {
      const double rdy = xf[a] - xn[a];
      viol = fmax(viol, fabs(rdy));
      if (gout) gout[tm_gdyn(P, k) + a] = rdy;
    }
#if NS > 0
    {                                                     // g_k = h_nl(x_k, u_k) - us_k = 0   (preprocessing.py:107-108, pmpc.py:270-271)
      double gv[NS];
      tmpc_gnl(z, z + NX, gv);
#pragma unroll
      for (int i = 0; i < NS; ++i) {
        const double v = gv[i] - z[NZM + i];
        viol = fmax(viol, fabs(v));
        if (gout) gout[tm_gg(P, k) + i] = v;
      }
    }
#endif
    for (int i = 0; i < nh; ++i) {
      double v = P.c[i];
#pragma unroll
      for (int b = 0; b < NZ; ++b) v += P.C[(size_t)i * NZ + b] * z[b];
      if (gout) gout[tm_gh(P, k) + i] = v;
      if (!(k == 0 && P.relax0[i]) && v < 0.0) viol = fmax(viol, -v);
    }
    if (k == 0) {
#pragma unroll
      for (int a = 0; a < NX; ++a) {
        const double r0 = z[a] - S.X0[inst * NX + a];
        viol = fmax(viol, fabs(r0));
        if (gout) gout[a] = r0;
      }
    }
    if (k == N - 1) {
      const double* xrN = P.wref + (size_t)((S.phase + N) % P.p) * NZ;
      for (int t = 0; t < P.nxt; ++t) {
        const double rt = xn[P.term_idx[t]] - xrN[P.term_idx[t]];
        viol = fmax(viol, fabs(rt));
        if (gout) gout[tm_gterm(P) + t] = rt;
      }
    }
  }
  f_out = tm_wsum(f);
  viol_out = tm_wmax(viol);
}

// |grad_w L|_inf at (W, LAM) using the linearisation stored in LIN (must be valid at W)      sqp_method.py:246
TM_HD double tm_dual_infeas(const TmProb& P, const TmState& S, int64_t inst) {
  const int N = P.N, nh = P.nh;
  const int lane = TM_LANE;
  const double* w = S.W + inst * P.n_w;
  const double* lam = S.LAM + inst * P.n_g;
  const double* lin = S.LIN + inst * P.N * (int64_t)TM_LSZ;
  double mx = 0.0;
  for (int k = lane; k < N; k += TM_NL) {
    const int ph = (S.phase + k) % P.p;
    const double* Hk = P.H + (size_t)ph * NZ * NZ;
    const double* wr = P.wref + (size_t)ph * NZ;
    const double* qk = P.q + (size_t)ph * NZ;
    const double* AB = lin + (size_t)k * TM_LSZ + NX;
    const double* ld = lam + tm_gdyn(P, k);
    const double* lh = lam + tm_gh(P, k);
    double dz[NZ], gl[NZ];
#pragma unroll
    for (int b = 0; b < NZ; ++b) dz[b] = w[k * NZ + b] - wr[b];
    if (P.economic) {
      double z[NZ];
#pragma unroll
      for (int b = 0; b < NZ; ++b) { z[b] = w[k * NZ + b]; gl[b] = 0.0; }
      tmpc_cost_grad(z, z + NX, gl);                              // dl/d(x,u); 0 on us
#pragma unroll
      for (int b = NZM + NS; b < NZ; ++b) gl[b] = qk[b];          // scost on usc
    }
#if NS > 0
    double Jg[NS * NZM];
    const double* lg = lam + tm_gg(P, k);
    {
      double z[NZ], gv[NS];
#pragma unroll
      for (int b = 0; b < NZ; ++b) z[b] = w[k * NZ + b];
      tmpc_gnl_jac(z, z + NX, gv, Jg);
    }
#endif
#pragma unroll
    for (int a = 0; a < NZ; ++a) {
      double v = P.economic ? gl[a] : qk[a];
      if (!P.economic) {
#pragma unroll
        for (int b = 0; b < NZ; ++b) v += Hk[a * NZ + b] * dz[b];
      }
      if (a < NZM) {
#pragma unroll
        for (int i = 0; i < NX; ++i) v += AB[i * NZM + a] * ld[i];
      }
#if NS > 0
      if (a < NZM) {
#pragma unroll
        for (int i = 0; i < NS; ++i) v += Jg[i * NZM + a] * lg[i];
      } else if (a < NZM + NS) v -= lg[a - NZM];
#endif
      for (int i = 0; i < nh; ++i) v += P.C[(size_t)i * NZ + a] * lh[i];
      if (a < NX) v += (k == 0) ? lam[a] : -lam[tm_gdyn(P, k - 1) + a];
      mx = fmax(mx, fabs(v));
    }
    if (k == N - 1) {
#pragma unroll
      for (int a = 0; a < NX; ++a) {
        double v = -ld[a];
        for (int t = 0; t < P.nxt; ++t) if (P.term_idx[t] == a) v += lam[tm_gterm(P) + t];
        mx = fmax(mx, fabs(v));
      }
    }
  }
  return tm_wmax(mx);
}

TM_HD int tm_is_ineq_active(const TmProb& P, const double* lam, int e) {   // e = k*nh + i
  return lam[tm_gh(P, e / P.nh) + e % P.nh] != 0.0;
}

// k = 0 bookkeeping (sqp_method.py:248-261): filter <- [(f0, infeas0)], as_idx_init.  LIN valid at (W, LAM).
TM_HD void tm_init(const TmProb& P, const TmState& S, int64_t inst) {
  double f, v;
  tm_eval_point(P, S, inst, 0.0, 1, nullptr, f, v);
  const int lane = TM_LANE;
  if (lane == 0) {
    S.FILT[inst * P.filter_cap * 2 + 0] = f;
    S.FILT[inst * P.filter_cap * 2 + 1] = v;
    S.nfilt[inst] = 1;
    S.iter[inst] = 0;
    S.status[inst] = -1;
    S.flags[inst] = 0;
    S.qpmode[inst] = 0;
    S.qpstat[inst] = 0;
    const double* lam = S.LAM + inst * P.n_g;
    for (int wd = 0; wd < S.aswords; ++wd) {
      unsigned bits = 0;
      for (int bt = 0; bt < 32; ++bt) {
        int e = wd * 32 + bt;
        if (e < P.N * P.nh && tm_is_ineq_active(P, lam, e)) bits |= (1u << bt);
      }
      S.asinit[inst * S.aswords + wd] = bits;
    }
  }
  TM_SYNC();
}

// finalise an instance: stats of __postprocessing (sqp_method.py:203-219) and __detect_AC (pmpc.py:840-856)
TM_HD void tm_finalize(const TmProb& P, const TmState& S, int64_t inst, int status) {
  double f, v;
  tm_eval_point(P, S, inst, 0.0, 1, S.G + inst * P.n_g, f, v);
  if (TM_LANE == 0) {
    const double* lam = S.LAM + inst * P.n_g;
    int nAS = 0, nACt = 0, nAC0 = 0;
    for (int e = 0; e < P.N * P.nh; ++e) {
      const int a = tm_is_ineq_active(P, lam, e);
      const int a0 = (S.asinit[inst * S.aswords + e / 32] >> (e % 32)) & 1u;
      nAS += a;
      nACt += (a != a0);
    }
    const double* lref = P.ref_du + (size_t)S.phase * P.n_g;
    for (int i = 0; i < P.nh; ++i) nAC0 += ((lam[tm_gh(P, 0) + i] != 0.0) != (lref[tm_gh(P, 0) + i] != 0.0));
    S.fval[inst] = f;
    S.nAS[inst] = nAS;
    S.nACtot[inst] = nACt;
    S.nAC[inst] = nAC0;
    S.status[inst] = status;
  }
  TM_SYNC();
}

// convergence test at the accepted point (LIN valid at W, LAM):  sqp_method.py:276-283
TM_HD void tm_conv(const TmProb& P, const TmState& S, int64_t inst) {
  const double dual = tm_dual_infeas(P, S, inst);
  const int nf = S.nfilt[inst];
  const double viol = S.FILT[(inst * P.filter_cap + nf - 1) * 2 + 1];
  const int it = S.iter[inst];
  int done = -1;
  if (!(dual == dual) || !(viol == viol)) done = 4;
  else if (viol < P.tol && dual < P.tol) done = 0;
  else if (it >= P.max_iter || nf >= P.filter_cap) done = 1;
  if (done >= 0) {
    tm_finalize(P, S, inst, done);
  } else if (TM_LANE == 0) {
#ifdef __CUDA_ARCH__
    int pos = atomicAdd(S.cnt_next, 1);
#else
    int pos = (*S.cnt_next)++;
#endif
    S.list_next[pos] = (int)inst;
  }
  TM_SYNC();
}

// after the QP and the trial linearisation at (W + D, LAMQ): filter line search, update, convergence
TM_HD void tm_post(const TmProb& P, const TmState& S, int64_t inst) {
  const int lane = TM_LANE;
  const int qp_status = S.qpstat[inst];
  if (qp_status != 0) { tm_finalize(P, S, inst, qp_status); return; }
  double alpha = 1.0, f, v;
  tm_eval_point(P, S, inst, alpha, 1, nullptr, f, v);
  const int nf = S.nfilt[inst];
  const double* F = S.FILT + inst * P.filter_cap * 2;
  int relin = 0;
  unsigned long long ndyn = 0;
  for (int ls = 0; ls < P.max_ls; ++ls) {                       // sqp_method.py:304-320
    int cnt = 0;
    for (int e = lane; e < nf; e += TM_NL) cnt += (f > F[2 * e] && v > F[2 * e + 1]) ? 1 : 0;
    cnt = tm_wsumi(cnt);
    if (cnt > 1) {
      alpha *= P.beta;
      tm_eval_point(P, S, inst, alpha, 0, nullptr, f, v);
      relin = 1;
      ndyn += (unsigned long long)P.N;
    } else break;
  }
  if (!(f == f) || !(v == v)) { tm_finalize(P, S, inst, 4); return; }
  double* w = S.W + inst * P.n_w;
  const double* d = S.D + inst * P.n_w;
  double* lam = S.LAM + inst * P.n_g;
  const double* lq = S.LAMQ + inst * P.n_g;
  for (int e = lane; e < P.n_w; e += TM_NL) w[e] += alpha * d[e];        // :174
  for (int e = lane; e < P.n_g; e += TM_NL) lam[e] = lq[e];              // :175 full dual step
  if (lane == 0) {
    // The reference's filter grows by one row per iteration (:323) and is only ever asked "do more than one of the
    // stored rows dominate the trial point" (:305-311).  A stored row that is itself weakly dominated by two other
    // stored rows can never change that answer (whenever it counts, both of them count as well), so such rows are
    // dropped and the filter stays small however many iterations max_iter allows.  The newest row is kept: its
    // infeasibility is the one the convergence test reads (:271,276).
    double* Fw = S.FILT + inst * P.filter_cap * 2;
    int n = nf;
    for (int e = 0; e < n;) {
      int dom = 0;
      for (int o = 0; o < n; ++o) dom += (o != e && Fw[2 * o] <= Fw[2 * e] && Fw[2 * o + 1] <= Fw[2 * e + 1]) ? 1 : 0;
      dom += (f <= Fw[2 * e] && v <= Fw[2 * e + 1]) ? 1 : 0;
      if (dom >= 2) {
        for (int o = e; o < n - 1; ++o) { Fw[2 * o] = Fw[2 * o + 2]; Fw[2 * o + 1] = Fw[2 * o + 3]; }
        --n;
      } else ++e;
    }
    Fw[2 * n + 0] = f;                                                    // :323
    Fw[2 * n + 1] = v;
    S.nfilt[inst] = n + 1;
    S.iter[inst] += 1;
    if (relin) S.flags[inst] |= 2;
#ifdef __CUDA_ARCH__
    atomicAdd(S.counters + 0, 1ull);
    if (ndyn) atomicAdd(S.counters + 4, ndyn);
#else
    S.counters[0] += 1; S.counters[4] += ndyn;
#endif
  }
  TM_SYNC();
  if (relin) {
    if (lane == 0) {
#ifdef __CUDA_ARCH__
      int pos = atomicAdd(S.cnt_relin, 1);
#else
      int pos = (*S.cnt_relin)++;
#endif
      S.list_relin[pos] = (int)inst;
    }
    TM_SYNC();
    return;
  }
  tm_conv(P, S, inst);
}

// warm-start shift (pmpc.py:867-906): (W, LAM) -> (Ws, Ls); one warp per instance
TM_HD void tm_shift(const TmProb& P, const double* w, const double* lam, double* ws, double* ls) {
  const int N = P.N;
  const int lane = TM_LANE;
  for (int e = lane; e < P.n_w; e += TM_NL) {
    int k = e / NZ, o = e % NZ;
    double v;
    if (k >= N) v = w[N * NZ + o];                                   // x_N <- x_N
    else if (o < NX) v = w[(k + 1) * NZ + o];                        // x_i <- x_{i+1}  (x_{N-1} <- x_N)
    else v = (k < N - 1) ? w[(k + 1) * NZ + o] : w[(N - 1) * NZ + o];  // u_{N-1} <- u_{N-2}^{shifted} = u_{N-1}
    ws[e] = v;
  }
  for (int e = lane; e < P.n_g; e += TM_NL) {
    double v;
    if (e < NX) v = lam[tm_gdyn(P, 0) + e];                          // init <- dyn_0
    else if (e >= tm_gterm(P)) v = lam[e];                           // term kept
    else {
      int k = (e - NX) / TM_GS(P), o = (e - NX) % TM_GS(P);
      int ksrc = (k < N - 1) ? k + 1 : N - 1;                        // last stage duplicated
      v = lam[NX + ksrc * TM_GS(P) + o];
    }
    ls[e] = v;
  }
  TM_SYNC();
}

// __prefilter_lam_g (sqp_method.py:223-238): zero every multiplier below lam_tresh, equality rows included
TM_HD void tm_prefilter(const TmProb& P, const TmState& S, int64_t inst) {
  double* lam = S.LAM + inst * P.n_g;
  for (int e = TM_LANE; e < P.n_g; e += TM_NL) if (fabs(lam[e]) < P.lam_tresh) lam[e] = 0.0;
  TM_SYNC();
}

// ---------------------------------------------------------------------------------------------------------------
// First QP after reset(): every instance starts from the same (w0, lam0) (pmpc.py:930-942), so all B QPs share the
// Hessian, the constraint Jacobian and every offset except the x_0 residual e0 = x0 - w0[0:nx]: ONE parametric QP.
// Its equality-constrained solution map is tabulated once (tm_qp_solve with TmQpPert, one warp per table row):
//     TAB[0]          (d, lam) for e0 = 0                 TAB[1+a]       response to e0 = unit_a
//     TAB[1+NX+e]     response to a unit multiplier on inequality row e (terminal rows stay enforced)
//     SL0 / SLPHI     row values n_e'd of TAB[0] (+ h(w0)) / of TAB[1+a];     MCOL[e][e'] = n_e' G' n_e
// and each instance runs only the Goldfarb-Idnani working-set iteration on these tables (thread per instance, state in
// registers / local memory, no Riccati sweep, no per-instance workspace), then one table combination for (d, lam).
// Same exact active-set solution as tm_qp_solve (unique: strictly convex on the feasible null space).
// ---------------------------------------------------------------------------------------------------------------
#define TM_Q0_MAXM 20      /* working-set capacity (inequality rows); overflow -> generic path */
struct TmQp0Tab {
  int EI, EIs, n_out, nT;  // inequality rows N*nh, padded row stride of MCOL (odd), n_w + n_g, 1 + NX + EI
  double *TAB, *SL0, *SLPHI, *MCOL;
  int* bad;                // != 0: the tabulation failed (base factorisation not PD ...) -> every instance takes the generic path
};

// returns 0 ok / 2 not solved here (overflow, dependent rows, breakdown): the caller queues the instance for tm_qp
TM_HD int tm_qp0_gi(const TmProb& P, const TmQp0Tab& T, const double* e0, int* acte, double* nu, int& m_out, int& ngi_out) {
  const int EI = T.EI, EIs = T.EIs, nh = P.nh;
  double Lf[TM_Q0_MAXM * (TM_Q0_MAXM + 1) / 2], cA[TM_Q0_MAXM], rv[TM_Q0_MAXM];   // Lf: packed lower triangle
#define TM_LF(i, j) Lf[(i) * ((i) + 1) / 2 + (j)]
  int m = 0, ngi = 0;
  m_out = 0; ngi_out = 0;
  const int maxit = 4 * EI + 8;
  for (int it = 0; it < maxit; ++it) {
    double best = TM_INF, bval = 0.0;
    int bid = -1;
    for (int e = 0; e < EI; ++e) {
      const int k = e / nh, i = e - k * nh;
      if (k == 0 && P.relax0[i]) continue;
      double v = T.SL0[e];
#pragma unroll
      for (int a = 0; a < NX; ++a) v += e0[a] * T.SLPHI[a * EI + e];
      for (int j = 0; j < m; ++j) v += nu[j] * T.MCOL[(size_t)acte[j] * EIs + e];
      const double sc = v / fmax(1.0, fabs(P.c[i]));
      if (sc < best) { best = sc; bid = e; bval = v; }
    }
    if (!(best < -1e-10)) break;                 // primal feasible: optimal
    int dup = 0;
    for (int j = 0; j < m; ++j) if (acte[j] == bid) dup = 1;
    if (dup) break;
    if (m >= TM_Q0_MAXM) return 2;
    const int qe = bid;
    double sval = bval;
    const double yq = T.MCOL[(size_t)qe * EIs + qe];
    double nq = 0.0;
    int added = 0;
    ++ngi;
    for (int inner = 0; inner < TM_Q0_MAXM + 2; ++inner) {
      double ll = 0.0;
      for (int i = 0; i < m; ++i) {
        double v = T.MCOL[(size_t)qe * EIs + acte[i]];
        for (int l = 0; l < i; ++l) v -= TM_LF(i, l) * cA[l];
        v /= TM_LF(i, i);
        cA[i] = v;
        ll += v * v;
      }
      for (int i = m - 1; i >= 0; --i) {
        double v = cA[i];
        for (int l = i + 1; l < m; ++l) v -= TM_LF(l, i) * rv[l];
        rv[i] = v / TM_LF(i, i);
      }
      const double zn = yq - ll;
      double t1 = TM_INF;
      int jd = -1;
      for (int j = 0; j < m; ++j) {
        if (rv[j] > 1e-14) { const double tj = nu[j] / rv[j]; if (tj < t1) { t1 = tj; jd = j; } }
      }
      const int dependent = !(zn > 1e-11 * fmax(yq, 1e-300));
      double t;
      int do_add = 0;
      if (dependent) {
        if (jd < 0) return 2;
        t = t1;
      } else {
        const double t2 = -sval / zn;
        if (t2 <= t1) { t = t2; do_add = 1; } else t = t1;
        sval += t * zn;
      }
      for (int j = 0; j < m; ++j) nu[j] -= t * rv[j];
      nq += t;
      if (do_add) {
        for (int l = 0; l < m; ++l) TM_LF(m, l) = cA[l];
        TM_LF(m, m) = sqrt(zn);
        acte[m] = qe; nu[m] = nq;
        ++m;
        added = 1;
        break;
      }
      for (int a = jd; a < m - 1; ++a) { acte[a] = acte[a + 1]; nu[a] = nu[a + 1]; }
      --m;
      for (int i = 0; i < m; ++i)
        for (int j = 0; j <= i; ++j) TM_LF(i, j) = T.MCOL[(size_t)acte[j] * EIs + acte[i]];
      for (int c = 0; c < m; ++c) {
        double dg = TM_LF(c, c);
        for (int l = 0; l < c; ++l) dg -= TM_LF(c, l) * TM_LF(c, l);
        if (!(dg > 0.0)) return 2;
        const double ld = sqrt(dg);
        TM_LF(c, c) = ld;
        for (int i = c + 1; i < m; ++i) {
          double v = TM_LF(i, c);
          for (int l = 0; l < c; ++l) v -= TM_LF(i, l) * TM_LF(c, l);
          TM_LF(i, c) = v / ld;
        }
      }
    }
    if (!added) return 2;
    if (it == maxit - 1) return 2;
  }
  m_out = m; ngi_out = ngi;
  return 0;
}
#undef TM_LF

// (d, lam)[i] of one instance from the tables: element i of  TAB[0] + sum_a e0_a TAB[1+a] + sum_j nu_j TAB[1+NX+acte_j]
TM_HD double tm_qp0_combine(const TmQp0Tab& T, int i, const double* e0, const int* acte, const double* nu, int m) {
  double v = T.TAB[i];
#pragma unroll
  for (int a = 0; a < NX; ++a) v += e0[a] * T.TAB[(size_t)(1 + a) * T.n_out + i];
  for (int j = 0; j < m; ++j) v += nu[j] * T.TAB[(size_t)(1 + NX + acte[j]) * T.n_out + i];
  return v;
}

// table row t of the tabulation (one warp / one twin call per row); inst = any instance (all identical)
TM_HD void tm_qp0_build_row(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& ws, const TmQp0Tab& T, int t) {
  TmQpPert pt;
  pt.homog = t > 0;
  pt.e0_unit = (t >= 1 && t <= NX) ? t - 1 : -1;
  pt.row = t > NX ? t - 1 - NX : -1;
  pt.dout = T.TAB + (size_t)t * T.n_out;
  pt.lout = pt.dout + P.n_w;
  unsigned none[TM_ALW], nxt[TM_ALW];
  for (int wd = 0; wd < TM_ALW; ++wd) none[wd] = 0u;
  int nwrong = 0, ngi = 0;
  tm_qp_setup(P, S, inst, ws, P.hessian_exact);
  const int ret = tm_qp_solve(P, S, inst, ws, none, nxt, nwrong, ngi, &pt);
  if (TM_LANE == 0) {
    if (ret != 0) {
#ifdef __CUDA_ARCH__
      atomicExch(T.bad, 1);
#else
      *T.bad = 1;
#endif
    } else if (pt.row >= 0) {
      pt.lout[tm_gh(P, pt.row / P.nh) + pt.row % P.nh] = -1.0;       // the unit multiplier itself (lam_h = -nu)
    }
  }
  TM_SYNC();
}

// derived tables: entry (t, e) = n_e' TAB[t].d  (+ h_e(w0) for t = 0)
TM_HD void tm_qp0_derive(const TmProb& P, const TmState& S, int64_t inst, const TmQp0Tab& T, int t, int e) {
  const int k = e / P.nh, i = e % P.nh;
  const double* Ci = P.C + (size_t)i * NZ;
  const double* d = T.TAB + (size_t)t * T.n_out + (size_t)k * NZ;
  double v = 0.0;
#pragma unroll
  for (int b = 0; b < NZ; ++b) v += Ci[b] * d[b];
  if (t == 0) {
    const double* w = S.W + inst * P.n_w + (size_t)k * NZ;
    double hv = P.c[i];
#pragma unroll
    for (int b = 0; b < NZ; ++b) hv += Ci[b] * w[b];
    T.SL0[e] = hv + v;
  } else if (t <= NX) {
    T.SLPHI[(size_t)(t - 1) * T.EI + e] = v;
  } else {
    T.MCOL[(size_t)(t - 1 - NX) * T.EIs + e] = v;
  }
}

// bookkeeping of one instance solved (ret == 0) or not (ret != 0 -> queued for the generic path) by the table route
TM_HD void tm_qp0_finish(const TmProb& P, const TmState& S, int64_t inst, int ret, int ngi) {
  if (ret == 0) {
    S.qpmode[inst] = 0;
    S.qpstat[inst] = 0;
    S.qpwork[inst] = ngi;
#ifdef __CUDA_ARCH__
    atomicAdd(S.counters + 5, 1ull); atomicAdd(S.counters + 6, (unsigned long long)ngi); atomicAdd(S.counters + 8, 1ull);
#else
    S.counters[5] += 1; S.counters[6] += ngi; S.counters[8] += 1;
#endif
  } else {
    S.qpmode[inst] = 0;
#ifdef __CUDA_ARCH__
    const int pos = atomicAdd(S.cnt_retry, 1);
#else
    const int pos = (*S.cnt_retry)++;
#endif
    S.list_retry[pos] = (int)inst;
  }
}

// __postprocessing's sanity check (sqp_method.py:190-201): at the returned point the Hessian (exact or Gauss-Newton, as
// configured) must be positive definite on the null space of [equality rows; inequality rows with a non-zero multiplier],
// else the reference raises AssertionError -> status TMPC_NOT_PD here.  Test = the constraint-to-go factorisation with those
// rows held (its projected-block Cholesky pivots), terminal rows weighted 100x so the test space is the reference's.
// LIN must be valid at (W, LAM) -- it is for every finished instance (tm_finalize).
TM_HD void tm_pd_check(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& ws) {
  const int st = S.status[inst];
  if (st != 0 && st != 1) return;
  unsigned mask[TM_ALW];
  for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = 0u;
  const double* lam = S.LAM + inst * P.n_g;
  for (int e = 0; e < P.N * P.nh; ++e) {
    const int k = e / P.nh, i = e % P.nh;
    if (k == 0 && P.relax0[i]) continue;
    if (lam[tm_gh(P, k) + i] != 0.0) tm_mask_set(mask, e);
  }
  tm_pin_soft_slacks(P, mask);
  tm_qp_setup(P, S, inst, ws, P.hessian_exact);
  double qmax = 0.0;
  for (int e = TM_LANE; e < P.N * NZ; e += TM_NL) { const int k = e / NZ, i = e % NZ; qmax = fmax(qmax, fabs(ws.Q[(size_t)k * NZ * NZ + i * NZ + i])); }
  const double rho = 100.0 * P.rho_rel * fmax(tm_wmax(qmax), 1e-300);
  const int ret = tm_qp_factor(P, ws, mask, ws.pv + 2 * NX, rho);
  if (ret == 3 && TM_LANE == 0) S.status[inst] = 3;
  TM_SYNC();
}

#define TMPC_JAC_OK 0                   /* the jstatus values of include/tmpc.h (the CPU twin compiles this file without it) */
#define TMPC_JAC_WEAK 1
#define TMPC_JAC_NOT_SOLVED 2
#define TMPC_JAC_SINGULAR 3

// The prelude of the sensitivities of a converged instance (tm_feedback_jacobian, tm_solution_vjp).  Held set A = the equality
// rows + the inequality rows with a non-zero multiplier (stage-0 rows of relax0 excluded), as in tm_pd_check.  Returns
// TMPC_JAC_NOT_SOLVED when the step's status is not 0 (nothing set up); else TMPC_JAC_OK or TMPC_JAC_WEAK (strict complementarity
// fails), with A in `mask` and ws the base QP at (W, LAM) with the exact Hessian, the residuals of the held and of the nonlinear
// rows zeroed: they are O(tol) at a solution and would enter every perturbed solve.  LIN must be valid at (W, LAM).
TM_HD int tm_jac_prelude(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& ws, unsigned* mask) {
  const int lane = TM_LANE;
  const int NI = P.N * P.nh;
  if (S.status[inst] != 0) return TMPC_JAC_NOT_SOLVED;
  for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = 0u;
  const double* lam = S.LAM + inst * P.n_g;
  for (int e = 0; e < NI; ++e) {
    const int k = e / P.nh, i = e % P.nh;
    if (k == 0 && P.relax0[i]) continue;
    if (lam[tm_gh(P, k) + i] != 0.0) tm_mask_set(mask, e);
  }
  tm_pin_soft_slacks(P, mask);
  tm_qp_setup(P, S, inst, ws, 1);
  // strict complementarity: every held row with a multiplier above lam_tresh, every other row strictly inactive
  int weak = 0;
  for (int e = lane; e < NI; e += TM_NL) {
    const int k = e / P.nh, i = e % P.nh;
    if (k == 0 && P.relax0[i]) continue;
    if (tm_mask_get(mask, e)) weak |= fabs(lam[tm_gh(P, k) + i]) < P.lam_tresh;
    else weak |= ws.hv[e] < 10.0 * P.tol;
  }
  weak = tm_wany(weak);
  TM_SYNC();
  for (int e = lane; e < NI; e += TM_NL) ws.hv[e] = 0.0;
#if NS > 0
  for (int e = lane; e < P.N * NS; e += TM_NL) ws.gv[e] = 0.0;
#endif
  TM_SYNC();
  return weak ? TMPC_JAC_WEAK : TMPC_JAC_OK;
}

// Feedback Jacobian du0*/dx0 of a converged instance (tmpc_feedback_jacobian, include/tmpc.h).  Column j is the u_0 block of the
// linear response of the base QP at the solution (exact Hessian, rows of A held, every offset zero) to the x_0 offset e_j: the
// KKT system [H J_A'; J_A 0] [dw; dlam] = [0; e_j on the init rows], i.e. the implicit-function derivative of the solution map
// under strict complementarity.  Same perturbed solve as the tabulation of the first QP (tm_qp0_build_row).  LIN must be valid at
// (W, LAM); S.D / S.LAMQ of the instance are used as scratch.  J: B*NUM*NX, row-major (nu, nx) per instance; jst: B.
TM_HD void tm_feedback_jacobian(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& ws, double* J, int* jst) {
  const int lane = TM_LANE;
  double* Ji = J + inst * (int64_t)(NUM * NX);
  unsigned mask[TM_ALW];
  int res = tm_jac_prelude(P, S, inst, ws, mask);
  if (res != TMPC_JAC_NOT_SOLVED) {
    // the perturbed solve zeroes the gradient, the dynamics defects and the terminal residuals
    TmQpPert pt;
    pt.homog = 1;
    pt.row = -1;
    pt.dout = S.D + inst * P.n_w;
    pt.lout = S.LAMQ + inst * P.n_g;
    unsigned nxtm[TM_ALW];
    for (int j = 0; j < NX; ++j) {
      pt.e0_unit = j;
      int nwrong = 0, ngi = 0;
      if (tm_qp_solve(P, S, inst, ws, mask, nxtm, nwrong, ngi, &pt) != 0) { res = TMPC_JAC_SINGULAR; break; }
      for (int i = lane; i < NUM; i += TM_NL) Ji[i * NX + j] = pt.dout[NX + i];
    }
  }
  if (res >= TMPC_JAC_NOT_SOLVED)
    for (int e = lane; e < NUM * NX; e += TM_NL) Ji[e] = NAN;
  if (lane == 0) jst[inst] = res;
  TM_SYNC();
}

// Vector-Jacobian product of the solution map of a converged instance (tmpc_solution_vjp, include/tmpc.h): for the cotangents
// v_u0 on u_0 and v_w on w, G = v_u0' du0/dx0 + v_w' dw/dx0, with the held set, weak test and statuses of tm_feedback_jacobian.
// K = [H J_A'; J_A 0] is symmetric, so with v = v_w + v_u0 on the u_0 block, v' dw/dx0 = [v; 0]' K^-1 [0; E] is the init-row
// block of the solution of K [y; mu] = [v; 0]: the base QP at the solution with the gradient -v and every other offset zero
// (x_0 offset, dynamics defects, terminal residuals, held-row residuals), one solve whatever nx; G = mu (its sign checked against
// v' J with tm_feedback_jacobian's J).  Vu0: B*NUM or nullptr,
// Vw: B*n_w or nullptr; dscr / lscr: B*n_w / B*n_g scratch for the step and multipliers of the solve; G: B*NX; jst: B.
TM_HD void tm_solution_vjp(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& ws, const double* Vu0, const double* Vw,
                           double* dscr, double* lscr, double* G, int* jst) {
  const int lane = TM_LANE;
  double* Gi = G + inst * NX;
  unsigned mask[TM_ALW];
  int res = tm_jac_prelude(P, S, inst, ws, mask);
  if (res != TMPC_JAC_NOT_SOLVED) {
    const double* vw = Vw ? Vw + inst * P.n_w : nullptr;
    const double* vu = Vu0 ? Vu0 + inst * NUM : nullptr;
    // The QP's stage recursion has no gradient on x_N (the NLP has no terminal cost): the cotangent on x_N enters through the
    // held last dynamics row, d_N = [A B]_{N-1} d_{N-1}, as [A B]_{N-1}' v_N on stage N-1.  The objective is unchanged on the
    // feasible set, so is the optimal value and with it the init-row multipliers.
    for (int e = lane; e < (P.N + 1) * NZ; e += TM_NL) {
      double v = 0.0;
      if (e < P.N * NZ) {
        if (vw) v = vw[e];
        if (vu && e >= NX && e < NX + NUM) v += vu[e - NX];
        if (vw && e >= (P.N - 1) * NZ) {
          const int c = e - (P.N - 1) * NZ;
          for (int a = 0; a < NX; ++a) v += ws.AB[(size_t)(P.N - 1) * NX * NZ + a * NZ + c] * vw[P.N * NZ + a];
        }
      }
      ws.r[e] = -v;
    }
    for (int e = lane; e < P.N * NX; e += TM_NL) ws.b[e] = 0.0;
    for (int t = lane; t < P.nxt; t += TM_NL) ws.tr[t] = 0.0;
    TM_SYNC();
    TmQpPert pt;
    pt.homog = 0;                                            // keep the gradient -v; the x_0 offset is zeroed by the solve
    pt.e0_unit = -1;
    pt.row = -1;
    pt.dout = dscr + inst * P.n_w;
    pt.lout = lscr + inst * P.n_g;
    unsigned nxtm[TM_ALW];
    int nwrong = 0, ngi = 0;
    if (tm_qp_solve(P, S, inst, ws, mask, nxtm, nwrong, ngi, &pt) != 0) res = TMPC_JAC_SINGULAR;
    else for (int j = lane; j < NX; j += TM_NL) Gi[j] = pt.lout[j];
  }
  if (res >= TMPC_JAC_NOT_SOLVED)
    for (int j = lane; j < NX; j += TM_NL) Gi[j] = NAN;
  if (lane == 0) jst[inst] = res;
  TM_SYNC();
}

// The QP of one SQP iteration for one instance.  Base rows = the inequality rows active in the current multipliers
// (the reference's reduced space, sqp_method.py:338-341,417-423).  Outcomes of the base factorisation:
//   positive definite                      -> solve; base rows that come back with a wrong-signed multiplier are released
//                                             (and the rows the dual active set added are held) and the QP is re-solved
//   not positive definite, exact Hessian   -> the reference eigen-clips its reduced Hessian here (sqp_method.py:345-376);
//                                             this solver re-solves with the Gauss-Newton Hessian, instance flagged
//   base rows inconsistent / infeasible    -> re-solve from the empty working set
#ifndef TM_MAX_ATTEMPTS
#define TM_MAX_ATTEMPTS 6
#endif
#ifndef TM_NONCONVEX_AFTER
#define TM_NONCONVEX_AFTER 3
#endif
TM_HD void tm_qp(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& ws) {
  if (S.pd_check) { tm_pd_check(P, S, inst, ws); return; }
  unsigned mask[TM_ALW], next[TM_ALW];
  const int NI = P.N * P.nh;
  int use_exact = P.hessian_exact;
  int flag = 0, work = 0, ret = 0, emptied = 0, attempts = 0, have_held = 0, nflip = 0, rel_stage = 0, we = -1;
  unsigned held[TM_ALW], wrongm[TM_ALW];
  for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = 0u;
  {
    const double* lam = S.LAM + inst * P.n_g;
    for (int e = 0; e < NI; ++e) {
      const int k = e / P.nh, i = e % P.nh;
      if (k == 0 && P.relax0[i]) continue;
      if (lam[tm_gh(P, k) + i] != 0.0) tm_mask_set(mask, e);
    }
  }
  tm_qp_setup(P, S, inst, ws, use_exact);
  // Instances that are still iterating after TM_NONCONVEX_AFTER SQP iterations sit on non-convex QPs where the Gauss-Newton
  // re-solve converges slowly or cycles (measured on the CSTR sweep: 20 of 2^20 never converge, the reference needs 5-7
  // iterations): from then on a QP that turns non-convex is continued by primal active-set steps on the exact Hessian, and the
  // terminal rows' augmented-Lagrangian weight is raised so that the positive-definiteness test is the one on the reference's space.
  const int late = (P.reg_mode & 8) && (P.reg_mode >= 16 || S.iter[inst] >= P.nonconvex_after);
  const double rho_scale = late ? 100.0 : 1.0;
  for (int guard = 0; guard < 4 * TM_MAX_ATTEMPTS + 12; ++guard) {
    int nwrong = 0, ngi = 0;
    ret = tm_qp_solve(P, S, inst, ws, mask, next, nwrong, ngi, nullptr, 0, rho_scale);
    work += 1 + ngi;
    int hr = ret == 0 ? (nwrong ? 3 : 0) : (ret == 3 ? 2 : 1);
    if (TM_LANE == 0) {   // attempt histogram: [8 + 4*(0 exact first | 1 exact re-solve | 2 Gauss-Newton) + (0 ok | 1 infeasible | 2 not PD | 3 wrong-signed base rows)]
      const int hm = use_exact ? (guard == 0 ? 0 : 1) : 2;
#ifdef __CUDA_ARCH__
      atomicAdd(S.counters + 8 + 4 * hm + hr, 1ull);
#else
      S.counters[8 + 4 * hm + hr] += 1;
#endif
    }
#if defined(TM_DEBUG_QP) && !defined(__CUDA_ARCH__)
    if (ret == 0) {   // stationarity and feasibility residuals of the returned (d, lam)
      const double* lq = S.LAMQ + inst * P.n_g;
      const TmP d = ws.d;
      double rs = 0.0, rf = 0.0;
      for (int k = 0; k < P.N; ++k) {
        for (int c = 0; c < NZ; ++c) {
          double v = ws.r[k * NZ + c];
          for (int e = 0; e < NZ; ++e) v += 0.5 * (ws.Q[(size_t)k * NZ * NZ + c * NZ + e] + ws.Q[(size_t)k * NZ * NZ + e * NZ + c]) * d[k * NZ + e];
          for (int i = 0; i < NX; ++i) v += ws.AB[(size_t)k * NX * NZ + i * NZ + c] * lq[tm_gdyn(P, k) + i];
          for (int i = 0; i < P.nh; ++i) v += P.C[(size_t)i * NZ + c] * lq[tm_gh(P, k) + i];
          if (c < NX) v += (k == 0) ? lq[c] : -lq[tm_gdyn(P, k - 1) + c];
          rs = fmax(rs, fabs(v));
        }
        for (int i = 0; i < NX; ++i) {
          double v = ws.b[k * NX + i] - d[(k + 1) * NZ + i];
          for (int c = 0; c < NZ; ++c) v += ws.AB[(size_t)k * NX * NZ + i * NZ + c] * d[k * NZ + c];
          rf = fmax(rf, fabs(v));
        }
      }
      for (int a = 0; a < NX; ++a) {
        double v = -lq[tm_gdyn(P, P.N - 1) + a];
        for (int t = 0; t < P.nxt; ++t) if (P.term_idx[t] == a) v += lq[tm_gterm(P) + t];
        rs = fmax(rs, fabs(v));
      }
      for (int t = 0; t < P.nxt; ++t) rf = fmax(rf, fabs(ws.tr[t] + d[P.N * NZ + P.term_idx[t]]));
      double qv = 0.0;
      for (int k = 0; k < P.N; ++k) for (int c = 0; c < NZ; ++c) {
        double v = ws.r[k * NZ + c];
        for (int e = 0; e < NZ; ++e) v += 0.25 * (ws.Q[(size_t)k * NZ * NZ + c * NZ + e] + ws.Q[(size_t)k * NZ * NZ + e * NZ + c]) * d[k * NZ + e];
        qv += v * d[k * NZ + c];
      }
      double smin = 1e300; int nact = 0;
      for (int e = 0; e < NI; ++e) { double sl = ws.hv[e] + tm_erow_dot(P, e, ws.d); if (sl < smin) smin = sl; if (fabs(sl) < 1e-9) ++nact; }
      fprintf(stderr, "[qp] inst %lld guard %d exact %d nwrong %d ngi %d: stationarity %.2e feasibility %.2e  q %.10e  min slack %.2e  rows at bound %d\n", (long long)inst, guard, use_exact, nwrong, ngi, rs, rf, qv, smin, nact);
    }
#endif
    if (ret == 0 && nwrong == 0) break;
    int any = 0;
    for (int wd = 0; wd < TM_ALW; ++wd) any |= (mask[wd] != 0u);
    if (ret == 0) {                                  // wrong-signed base rows
      for (int wd = 0; wd < TM_ALW; ++wd) { held[wd] = mask[wd] | next[wd]; wrongm[wd] = mask[wd] & ~next[wd]; }   // the working set this solution sits on
      have_held = 1; rel_stage = 1;
      ++attempts;
      if (attempts < TM_MAX_ATTEMPTS) { for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = next[wd]; continue; }
      ret = 3;                                       // cycling: treat like a failed factorisation
    }
    if (ret == 3 && use_exact && have_held && late && nflip < 3 * TM_MAX_ATTEMPTS) {
      // Releasing the wrong-signed rows exposes negative curvature: the QP is not convex.  The reference's QP solver then
      // follows its homotopy until the next constraint blocks ("flipping bounds", external/acados/external/qpoases/
      // src/QProblem.c:5037-5060).  Here: one inertia-controlling primal active-set step from the held solution.  The
      // worst wrong-signed row r is moved off its bound along d(t) = argmin over {held rows active, row r at value t},
      // which is linear in t and descends (multiplier sign) without a minimiser (negative curvature), until the first
      // row outside the working set blocks; that row takes r's place, which keeps the reduced Hessian positive definite.
      int jblock = -1, tzero = 0;
      if (rel_stage == 1) {
        const double* lqh = S.LAMQ + inst * P.n_g;       // multipliers of the held solution (a failed solve leaves them)
        double worst = 0.0;
        we = -1;
        for (int e = 0; e < NI; ++e) {
          if (!tm_mask_get(wrongm, e)) continue;
          const double l = lqh[tm_gh(P, e / P.nh) + e % P.nh];
          if (l > worst) { worst = l; we = e; }
        }
        if (we >= 0) {                                   // first release the worst row alone: positive definite -> ordinary re-solve
          for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = held[wd];
          tm_mask_clr(mask, we);
          rel_stage = 2; ++nflip;
          continue;
        }
      }
      if (we >= 0 && rel_stage == 2) {
        int nw2 = 0, ngi2 = 0, r0, r1 = 1;
        r0 = tm_qp_solve(P, S, inst, ws, held, next, nw2, ngi2, nullptr, 1, rho_scale);
        if (r0 == 0) {
          for (int e = TM_LANE; e < NI; e += TM_NL) ws.sl0[e] = ws.hv[e] + tm_erow_dot(P, e, ws.d);
          TM_SYNC();
          if (TM_LANE == 0) ws.hv[we] -= 1.0;
          TM_SYNC();
          r1 = tm_qp_solve(P, S, inst, ws, held, next, nw2, ngi2, nullptr, 1, rho_scale);
          if (TM_LANE == 0) ws.hv[we] += 1.0;
          TM_SYNC();
        }
        work += 2;
        if (r0 == 0 && r1 == 0) {
          double tb = TM_INF;
          int jb = 0x7fffffff;
          for (int e = TM_LANE; e < NI; e += TM_NL) {
            const int k = e / P.nh, i = e % P.nh;
            if ((k == 0 && P.relax0[i]) || tm_mask_get(held, e)) continue;
            const double s0 = fmax(ws.sl0[e], 0.0), ds = ws.hv[e] + tm_erow_dot(P, e, ws.d) - ws.sl0[e];
            if (ds < -1e-12 * fmax(1.0, fabs(P.c[i]))) { const double te = s0 / (-ds); if (te < tb) { tb = te; jb = e; } }
          }
          tm_wargmin(tb, jb);
          if (tb < TM_INF) { jblock = jb; tzero = !(tb > 1e-9); }
        }
      }
#if defined(TM_DEBUG_QP) && !defined(__CUDA_ARCH__)
      fprintf(stderr, "[qp] primal step: release row %d (stage %d row %d, lam %.3e), blocking row %d (stage %d row %d) tzero %d\n", we, we / P.nh, we % P.nh,
              we >= 0 ? S.LAMQ[inst * P.n_g + tm_gh(P, we / P.nh) + we % P.nh] : 0.0, jblock, jblock / P.nh, jblock % P.nh, tzero);
#endif
      if (jblock >= 0) {
        for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = held[wd];
        if (!tzero) tm_mask_clr(mask, we);       // degenerate (zero-length) step: the blocking row joins, r stays
        tm_mask_set(mask, jblock);
        have_held = 0; rel_stage = 0; ++nflip; attempts = 0; flag |= 8;
        continue;
      }
    }
    if (ret == 3 && use_exact) {
      use_exact = 0; flag |= (guard == 0 ? 1 : 4); attempts = 0;
      tm_qp_setup(P, S, inst, ws, 0);
      continue;
    }
    if ((ret == 2 || ret == 6 || ret == 3) && any && !emptied) {
      emptied = 1; attempts = 0;
      for (int wd = 0; wd < TM_ALW; ++wd) mask[wd] = 0u;
      continue;
    }
    break;
  }
  if (TM_LANE == 0) {
    S.qpmode[inst] = 0;
    S.qpstat[inst] = ret == 0 ? 0 : (ret == 3 ? 3 : (ret == 7 ? 5 : 2));
    S.qpwork[inst] = work;
    if (flag) S.flags[inst] |= flag;
  }
  TM_SYNC();
}
