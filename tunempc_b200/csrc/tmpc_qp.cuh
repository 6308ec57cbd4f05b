// tmpc_qp.cuh -- K3/K4: the QP of one SQP iteration (included by tmpc_core.cuh).
//
// Replaces in the reference:  __regularize_hessian's positive-definiteness test (tunempc/sqp_method.py:335-347),
// __active_constraints_jacobian (:405-425) and the conic('qpoases') solve (:158-168).
//
// Method.  The reference tests (and, if needed, clips) its Hessian on the null space of
//        [ equality rows ; inequality rows with a non-zero multiplier ]                    (sqp_method.py:338-341)
// and the benchmark problems need exactly that space: with the exact Lagrangian Hessian the stage blocks are
// indefinite and the reduced Hessian is positive definite only once the rows active in the multipliers are held
// (measured on the CSTR sweep: min eig 1e-3 on that space, -1 on the null space of the equalities alone).  So the
// BASE problem of this solver is the equality-constrained QP on exactly that space:
//     min 1/2 d'Hd + r'd   s.t.  d_x0 = e0,  dynamics,  terminal rows T d_N + t = 0,  rows in A as equalities,
// factorised by a Riccati recursion with CONSTRAINT-TO-GO: going backwards, stage k holds a cost-to-go (P, p) and a
// set of linear constraints Gc x + gc = 0 on x_k inherited from later stages; together with the stage's own active
// rows they are eliminated against the stage inputs by Gauss-Jordan with full pivoting (u = Ku x + ku + Zu v), rows
// without an input pivot become the constraint-to-go of stage k-1, and the Cholesky factor of the projected block
// Zu'(R + B'PB)Zu is the positive-definiteness test: all pivots > reg_tol  <=>  the reduced Hessian on the
// reference's space is positive definite (block elimination of that matrix).  No penalty parameter anywhere.
// Every other inequality row enters a Goldfarb-Idnani dual active-set iteration carried in a small Schur complement
// over the base inverse (one Riccati sweep per added row).  Multipliers of the base rows come from a forward sweep
// over the stage-wise stationarity conditions; base rows whose multiplier has the wrong sign are released and the
// QP re-solved.  Exact active-set solution: inactive multipliers are exact zeros (sqp_method.py:421 relies on it).
#pragma once

#if TM_NL == 1
#define TM_UNROLL_T _Pragma("unroll")   /* one thread per instance: element loops have constant trip counts; unrolled, the staged blocks index statically */
#else
#define TM_UNROLL_T
#endif
#define NV NU               /* free variables of a stage block (inputs; + slacks in the slack formulation) */
#define TM_LFI(i, l) ((i) * ((i) + 1) / 2 + (l))   /* packed lower triangle of the Schur factor, l <= i */
#define TM_ES (NZ + 2)      /* row stride of the elimination scratch: coefficients | offset | state */

struct TmQpWs {
  TmP AB, Q, r, b, hv;                    // stage data: [A B] nx*nz | Hessian nz*nz | gradient | dynamics defect | row values
  TmP K, Wm, kkm;                         // per stage: feedback nv*nx, projected inverse Zu (Zu'Fuu Zu)^-1 Zu' nv*nv, main feed-forward
  TmP Pk, pm, py;                         // cost-to-go Hessian (N+1)*nx*nx, gradient of the main solve / of the correction solve
  TmP Gc, gc, ncs;                        // constraint-to-go rows (N+1)*nx*nx, offsets (N+1)*nx, row counts (N+1)
  TmP kk, d, y, rhs;                      // feed-forward of the current sweep; step, correction, right-hand side
  TmP sl, Mc, Lf, cA, rv, nu, acts, acte, sc;   // dual active set: row values, dual-Hessian columns, Schur factor, members
  TmP Ew, tr, lh, sl0;                    // scratch: elimination rows; terminal residual; row multipliers; row values of a held solution
  TmP Cg, gv;                             // slacked nonlinear rows g_k = h_nl(x,u) - us = 0: Jacobian w.r.t. (x,u) N*NS*NZM, values N*NS
  TmL F, f, PAB, pv;                      // per-stage scratch of the factorisation: KKT block, gradient, products, vectors (thread mode: thread-local)
};

// the large array of the dual active set (dual-Hessian columns Mc, swept with independent loads): the warp-per-instance
// kernels keep it in global memory (L2-resident: only the resident CTAs own a slot) so that several instances fit one SM
TM_HD size_t tm_qpws_cold_doubles(int N, int nh, int nxt, int M) {
  const size_t NI = (size_t)N * nh + nxt + 1;
  return (size_t)(M + 1) * NI;
}
TM_HD size_t tm_qpws_doubles(int N, int nh, int nxt, int M) {
  const size_t NI = (size_t)N * nh + nxt + 1;        // row universe of the dual active set: inequality rows, then terminal rows
  size_t n = 0;
  n += (size_t)N * NX * NZ + (size_t)N * NZ * NZ + (size_t)(N + 1) * NZ + (size_t)N * NX + NI;        // AB Q r b hv
  n += (size_t)N * NV * NX + (size_t)N * NV * NV + (size_t)N * NV;                                     // K Wm kkm
  n += (size_t)(N + 1) * NX * NX + 2 * (size_t)(N + 1) * NX;                                           // Pk pm py
  n += (size_t)(N + 1) * NX * NX + (size_t)(N + 1) * NX + (size_t)(N + 1);                             // Gc gc ncs
  n += (size_t)N * NV + 3 * (size_t)(N + 1) * NZ;                                                      // kk d y rhs
  n += NI + (size_t)(M + 1) * NI + (size_t)M * (M + 1) / 2 + 5 * (size_t)M + 8;                                  // sl Mc Lf cA rv nu acts acte sc
  n += (size_t)(NX + NS + nh) * TM_ES + NZ * NZ + NZ + NX * NZ + 4 * NX + (nxt > 0 ? nxt : 1) + 2 * NI;     // Ew F f PAB pv tr lh sl0
  n += (size_t)N * NS * NZM + (size_t)N * NS;                                                         // Cg gv
  return n;
}

#define TM_QP_LSCR (4 * NX)               /* thread mode: only pv (the x_0 offset lives in pv[2nx..3nx)) is addressed through the
                                             workspace struct; F, f, PAB are arrays local to tm_qp_factor */
TM_HD void tm_qpws_local(double* l, TmQpWs& s) { s.F = nullptr; s.f = nullptr; s.PAB = nullptr; s.pv = l; }
TM_HD void tm_qpws_carve(double* base, int N, int nh, int nxt, int M, TmQpWs& s, double* cold = nullptr) {
  const size_t NI = (size_t)N * nh + nxt + 1;
  size_t o = 0;
#define TM_CARVE(member, n) s.member = tm_mkp(base, o); o += (size_t)(n)
  TM_CARVE(AB, (size_t)N * NX * NZ);
  TM_CARVE(Q, (size_t)N * NZ * NZ);
  TM_CARVE(r, (size_t)(N + 1) * NZ);
  TM_CARVE(b, (size_t)N * NX);
  TM_CARVE(hv, NI);
  TM_CARVE(K, (size_t)N * NV * NX);
  TM_CARVE(Wm, (size_t)N * NV * NV);
  TM_CARVE(kkm, (size_t)N * NV);
  TM_CARVE(Pk, (size_t)(N + 1) * NX * NX);
  TM_CARVE(pm, (size_t)(N + 1) * NX);
  TM_CARVE(py, (size_t)(N + 1) * NX);
  TM_CARVE(Gc, (size_t)(N + 1) * NX * NX);
  TM_CARVE(gc, (size_t)(N + 1) * NX);
  TM_CARVE(ncs, (size_t)(N + 1));
  TM_CARVE(kk, (size_t)N * NV);
  TM_CARVE(d, (size_t)(N + 1) * NZ);
  TM_CARVE(y, (size_t)(N + 1) * NZ);
  TM_CARVE(rhs, (size_t)(N + 1) * NZ);
  TM_CARVE(sl, NI);
  if (cold) s.Mc = tm_mkp(cold, 0);           // Mc outside the (shared-memory) block: base then spans tm_qpws_doubles - tm_qpws_cold_doubles
  else { TM_CARVE(Mc, (size_t)(M + 1) * NI); }
  TM_CARVE(Lf, (size_t)M * (M + 1) / 2);
  TM_CARVE(cA, M);
  TM_CARVE(rv, M);
  TM_CARVE(nu, M);
  TM_CARVE(acts, M);
  TM_CARVE(acte, M);
  TM_CARVE(sc, 8);
  TM_CARVE(Ew, (size_t)(NX + NS + nh) * TM_ES);
#ifndef TM_WS_STRIDE
  TM_CARVE(F, NZ * NZ);
  TM_CARVE(f, NZ);
  TM_CARVE(PAB, NX * NZ);
  TM_CARVE(pv, 4 * NX);
#else
  o += NZ * NZ + NZ + NX * NZ + 4 * NX;     // thread mode: the caller points F, f, PAB, pv at a thread-local array (TM_QP_LSCR doubles)
#endif
  TM_CARVE(tr, (nxt > 0 ? nxt : 1));
  TM_CARVE(lh, NI);
  TM_CARVE(sl0, NI);
  TM_CARVE(Cg, (size_t)N * NS * NZM);
  TM_CARVE(gv, (size_t)N * NS);
#undef TM_CARVE
}

TM_HD int tm_mask_get(const unsigned* m, int e) { return (m[e >> 5] >> (e & 31)) & 1u; }
TM_HD void tm_mask_set(unsigned* m, int e) { m[e >> 5] |= (1u << (e & 31)); }
TM_HD void tm_mask_clr(unsigned* m, int e) { m[e >> 5] &= ~(1u << (e & 31)); }

// ---- one stage of the constrained factorisation (single lane) --------------------------------------------------
// in:  s.F (nz*nz stage block Q + [A B]'P[A B]), s.f (gradient r + [A B]'(P b + p)), nr candidate rows in s.Ew
//      ([coefficients nz | offset | state]: constraint-to-go of stage k+1 pulled back through the dynamics, then the
//      stage's own active rows)
// out: K, Wm, kkm of stage k; constraint-to-go (Gc, gc, ncs) of stage k; s.f <- f + F[:,u] ku
// returns 0 ok, 3 projected block not positive definite, 6 rows inconsistent
// Fast path of the stage elimination -- most stages of most QPs: no constraint-to-go from later stages, and the held rows of
// the stage (if any) each bound ONE input (P.rowpin), distinct inputs.  Those inputs are pinned (u_j = ku_j), the others are
// free: the plain Riccati step on the free inputs,  W = Zu (Zu'Fuu Zu)^-1 Zu',  K = -W Fux,  kk = ku - W (f_u + Fuu ku).
// Written with constant trip counts over all NV inputs (a pinned input is an identity row / column of the projected block), so
// everything stays in registers; per entry the same operations in the same order as the general routine below, whose
// elimination loops in this case only move zeros and unit vectors around: equal results.
TM_HD int tm_stage_factor_pinned(const TmProb& P, TmQpWs& s, int k, unsigned pinmask, const double* ku, const double* F, double* fv) {
  constexpr int NVV = NV > 0 ? NV : 1;
  double Rt[NVV * NVV], Y[NVV * NVV], Wl[NVV * NVV];
#pragma unroll
  for (int c = 0; c < NV; ++c)
#pragma unroll
    for (int e = 0; e <= c; ++e) {
      const bool pc = (pinmask >> c) & 1u, pe = (pinmask >> e) & 1u;
      Rt[c * NVV + e] = (pc || pe) ? ((c == e) ? 1.0 : 0.0) : 0.5 * (F[(NX + c) * NZ + NX + e] + F[(NX + e) * NZ + NX + c]);
    }
#pragma unroll
  for (int c = 0; c < NV; ++c) {
    double dg = Rt[c * NVV + c];
#pragma unroll
    for (int l = 0; l < c; ++l) dg -= Rt[c * NVV + l] * Rt[c * NVV + l];
    if (!((pinmask >> c) & 1u) && !(dg > P.reg_tol)) return 3;
    const double ld = sqrt(dg);
    Rt[c * NVV + c] = ld;
#pragma unroll
    for (int i = c + 1; i < NV; ++i) {
      double v = Rt[i * NVV + c];
#pragma unroll
      for (int l = 0; l < c; ++l) v -= Rt[i * NVV + l] * Rt[c * NVV + l];
      Rt[i * NVV + c] = v / ld;
    }
  }
#pragma unroll
  for (int a = 0; a < NV; ++a)
#pragma unroll
    for (int c = 0; c < NV; ++c) {
      double v = (a == c && !((pinmask >> a) & 1u)) ? 1.0 : 0.0;
#pragma unroll
      for (int l = 0; l < c; ++l) v -= Rt[c * NVV + l] * Y[l * NVV + a];
      Y[c * NVV + a] = ((pinmask >> c) & 1u) ? 0.0 : v / Rt[c * NVV + c];
    }
  const TmP Wk = s.Wm + (size_t)k * NV * NV;
#pragma unroll
  for (int a = 0; a < NV; ++a)
#pragma unroll
    for (int b2 = 0; b2 < NV; ++b2) {
      double v = 0.0;
#pragma unroll
      for (int c = 0; c < NV; ++c) v += Y[c * NVV + a] * Y[c * NVV + b2];
      Wl[a * NVV + b2] = v;
      Wk[a * NV + b2] = v;
    }
  const TmP Kk = s.K + (size_t)k * NV * NX;
#pragma unroll
  for (int j = 0; j < NX; ++j) {
    double t[NVV];
#pragma unroll
    for (int a = 0; a < NV; ++a) t[a] = 0.5 * (F[(NX + a) * NZ + j] + F[j * NZ + NX + a]);
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      double v = 0.0;
#pragma unroll
      for (int b2 = 0; b2 < NV; ++b2) v -= Wl[a * NVV + b2] * t[b2];
      Kk[a * NX + j] = v;
    }
  }
#pragma unroll
  for (int c = 0; c < NZ; ++c) {                      // ftil = f + F[:,u] ku
    double v = fv[c];
#pragma unroll
    for (int b2 = 0; b2 < NV; ++b2) v += 0.5 * (F[c * NZ + NX + b2] + F[(NX + b2) * NZ + c]) * ku[b2];
    fv[c] = v;
  }
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double v = ku[a];
#pragma unroll
    for (int b2 = 0; b2 < NV; ++b2) v -= Wl[a * NVV + b2] * fv[NX + b2];
    s.kkm[k * NV + a] = v;
  }
  s.ncs[k] = 0.0;
  return 0;
}

#if defined(TM_COUNT_STAGES) && !defined(__CUDA_ARCH__)
static long long tm_stage_counts[4] = {0, 0, 0, 0};   // twin diagnostics: stages without rows / with rows / total rows / with constraint-to-go
#endif
TM_HD int tm_stage_factor(const TmProb& P, TmQpWs& s, int k, int nr, double* F, double* fv) {
#if defined(TM_COUNT_STAGES) && !defined(__CUDA_ARCH__)
  tm_stage_counts[nr == 0 ? 0 : 1] += 1; tm_stage_counts[2] += nr; tm_stage_counts[3] += ((int)s.ncs[k + 1] > 0);
  if ((tm_stage_counts[0] + tm_stage_counts[1]) % 20000 == 0)
    fprintf(stderr, "[stages] free %lld with-rows %lld rows %lld ctg-stages %lld\n", tm_stage_counts[0], tm_stage_counts[1], tm_stage_counts[2], tm_stage_counts[3]);
#endif
#if NV > 0 && NV <= 4 && !defined(TM_NO_FREE_STAGE)
  if (nr == 0) { double ku0[NV]; for (int a = 0; a < NV; ++a) ku0[a] = 0.0; return tm_stage_factor_pinned(P, s, k, 0u, ku0, F, fv); }
#endif
  const TmP E = s.Ew;
  const double tolp = 1e-9, tolc = 1e-7;
  int colrow[NV > 0 ? NV : 1];
#pragma unroll
  for (int j = 0; j < NV; ++j) colrow[j] = -1;
  // normalise rows (max-abs 1); zero rows are dropped or flagged inconsistent
  for (int i = 0; i < nr; ++i) {
    double mx = 0.0;
    for (int c = 0; c < NZ; ++c) mx = fmax(mx, fabs(E[i * TM_ES + c]));
    if (!(mx > 1e-300)) {
      if (fabs(E[i * TM_ES + NZ]) > tolc) return 6;
      E[i * TM_ES + NZ + 1] = 3.0;
      continue;
    }
    const double inv = 1.0 / mx;
    for (int c = 0; c <= NZ; ++c) E[i * TM_ES + c] *= inv;
    E[i * TM_ES + NZ + 1] = 0.0;
  }
  // Gauss-Jordan on the input columns, full pivoting
  for (int step = 0; step < NV; ++step) {
    double best = 0.0;
    int bi = -1, bj = -1;
    for (int i = 0; i < nr; ++i) {
      if (E[i * TM_ES + NZ + 1] != 0.0) continue;
      for (int j = 0; j < NV; ++j) {
        if (colrow[j] >= 0) continue;
        const double v = fabs(E[i * TM_ES + NX + j]);
        if (v > best) { best = v; bi = i; bj = j; }
      }
    }
    if (!(best > tolp)) break;
    const double ip = 1.0 / E[bi * TM_ES + NX + bj];
    for (int c = 0; c <= NZ; ++c) E[bi * TM_ES + c] *= ip;
    E[bi * TM_ES + NX + bj] = 1.0;
    for (int i = 0; i < nr; ++i) {
      if (i == bi || E[i * TM_ES + NZ + 1] >= 2.0) continue;
      const double fc = E[i * TM_ES + NX + bj];
      if (fc == 0.0) continue;
      for (int c = 0; c <= NZ; ++c) E[i * TM_ES + c] -= fc * E[bi * TM_ES + c];
      E[i * TM_ES + NX + bj] = 0.0;
    }
    colrow[bj] = bi;
    E[bi * TM_ES + NZ + 1] = 1.0;
  }
  // rows without an input pivot constrain x_k alone: reduce them to independent rows = constraint-to-go of this stage
  int nck = 0;
  {
    int xrow[NX], xcol[NX];
    for (int step = 0; step < NX; ++step) {
      double best = 0.0;
      int bi = -1, bj = -1;
      for (int i = 0; i < nr; ++i) {
        if (E[i * TM_ES + NZ + 1] != 0.0) continue;
        for (int j = 0; j < NX; ++j) {
          int used = 0;
          for (int q = 0; q < nck; ++q) used |= (xcol[q] == j);
          if (used) continue;
          const double v = fabs(E[i * TM_ES + j]);
          if (v > best) { best = v; bi = i; bj = j; }
        }
      }
      if (!(best > tolp)) break;
      const double ip = 1.0 / E[bi * TM_ES + bj];
      for (int c = 0; c < NX; ++c) E[bi * TM_ES + c] *= ip;
      E[bi * TM_ES + NZ] *= ip;
      E[bi * TM_ES + bj] = 1.0;
      for (int i = 0; i < nr; ++i) {
        const double stt = E[i * TM_ES + NZ + 1];
        if (i == bi || stt == 1.0 || stt == 3.0) continue;
        const double fc = E[i * TM_ES + bj];
        if (fc == 0.0) continue;
        for (int c = 0; c < NX; ++c) E[i * TM_ES + c] -= fc * E[bi * TM_ES + c];
        E[i * TM_ES + NZ] -= fc * E[bi * TM_ES + NZ];
        E[i * TM_ES + bj] = 0.0;
      }
      E[bi * TM_ES + NZ + 1] = 2.0;
      xrow[nck] = bi; xcol[nck] = bj;
      ++nck;
    }
    for (int i = 0; i < nr; ++i)
      if (E[i * TM_ES + NZ + 1] == 0.0) {            // numerically zero row: redundant if its offset vanishes too
        if (fabs(E[i * TM_ES + NZ]) > tolc) return 6;
        E[i * TM_ES + NZ + 1] = 3.0;
      }
    const TmP Gk = s.Gc + (size_t)k * NX * NX;
    for (int q = 0; q < nck; ++q) {
      for (int c = 0; c < NX; ++c) Gk[q * NX + c] = E[xrow[q] * TM_ES + c];
      s.gc[k * NX + q] = E[xrow[q] * TM_ES + NZ];
    }
    s.ncs[k] = (double)nck;
  }
  // u = Ku x + ku + Zu v
  double Ku[(NV > 0 ? NV : 1) * NX], ku[NV > 0 ? NV : 1], Zu[(NV > 0 ? NV : 1) * (NV > 0 ? NV : 1)];
  int fl[NV > 0 ? NV : 1], nf = 0;
  for (int j = 0; j < NV; ++j) if (colrow[j] < 0) fl[nf++] = j;
  for (int j = 0; j < NV; ++j) {
    const int ri = colrow[j];
    for (int c = 0; c < NX; ++c) Ku[j * NX + c] = ri >= 0 ? -E[ri * TM_ES + c] : 0.0;
    ku[j] = ri >= 0 ? -E[ri * TM_ES + NZ] : 0.0;
    for (int c = 0; c < nf; ++c) Zu[j * NV + c] = ri >= 0 ? -E[ri * TM_ES + NX + fl[c]] : (fl[c] == j ? 1.0 : 0.0);
  }
  // projected block Rt = Zu' Fuu Zu and its Cholesky factor (lower, in place)
  double Rt[(NV > 0 ? NV : 1) * (NV > 0 ? NV : 1)], FZ[(NV > 0 ? NV : 1) * (NV > 0 ? NV : 1)];
  for (int a = 0; a < NV; ++a)
    for (int c = 0; c < nf; ++c) {
      double v = 0.0;
      for (int b2 = 0; b2 < NV; ++b2) v += 0.5 * (F[(NX + a) * NZ + NX + b2] + F[(NX + b2) * NZ + NX + a]) * Zu[b2 * NV + c];
      FZ[a * NV + c] = v;
    }
  for (int c = 0; c < nf; ++c)
    for (int e = 0; e <= c; ++e) {
      double v = 0.0;
      for (int a = 0; a < NV; ++a) v += Zu[a * NV + c] * FZ[a * NV + e];
      Rt[c * NV + e] = v;
    }
  for (int c = 0; c < nf; ++c) {
    double dg = Rt[c * NV + c];
    for (int l = 0; l < c; ++l) dg -= Rt[c * NV + l] * Rt[c * NV + l];
    if (!(dg > P.reg_tol)) {
#if defined(TM_DEBUG_QP) && !defined(__CUDA_ARCH__)
      fprintf(stderr, "[qp] stage %d not PD: pivot %d = %.3e (nf %d, nr %d, nck %d)\n", k, c, dg, nf, nr, nck);
#endif
      return 3;
    }
    const double ld = sqrt(dg);
    Rt[c * NV + c] = ld;
    for (int i = c + 1; i < nf; ++i) {
      double v = Rt[i * NV + c];
      for (int l = 0; l < c; ++l) v -= Rt[i * NV + l] * Rt[c * NV + l];
      Rt[i * NV + c] = v / ld;
    }
  }
  // Y = L^-1 Zu' (nf x nv);  Wm = Y'Y
  double Y[(NV > 0 ? NV : 1) * (NV > 0 ? NV : 1)];
  for (int a = 0; a < NV; ++a)
    for (int c = 0; c < nf; ++c) {
      double v = Zu[a * NV + c];
      for (int l = 0; l < c; ++l) v -= Rt[c * NV + l] * Y[l * NV + a];
      Y[c * NV + a] = v / Rt[c * NV + c];
    }
  const TmP Wk = s.Wm + (size_t)k * NV * NV;
  for (int a = 0; a < NV; ++a)
    for (int b2 = 0; b2 < NV; ++b2) {
      double v = 0.0;
      for (int c = 0; c < nf; ++c) v += Y[c * NV + a] * Y[c * NV + b2];
      Wk[a * NV + b2] = v;
    }
  // K = Ku - Wm (Fux + Fuu Ku)
  const TmP Kk = s.K + (size_t)k * NV * NX;
  for (int j = 0; j < NX; ++j) {
    double t[NV > 0 ? NV : 1];
    for (int a = 0; a < NV; ++a) {
      double v = 0.5 * (F[(NX + a) * NZ + j] + F[j * NZ + NX + a]);
      for (int b2 = 0; b2 < NV; ++b2) v += 0.5 * (F[(NX + a) * NZ + NX + b2] + F[(NX + b2) * NZ + NX + a]) * Ku[b2 * NX + j];
      t[a] = v;
    }
    for (int a = 0; a < NV; ++a) {
      double v = Ku[a * NX + j];
      for (int b2 = 0; b2 < NV; ++b2) v -= Wk[a * NV + b2] * t[b2];
      Kk[a * NX + j] = v;
    }
  }
  // main solve: ftil = f + F[:,u] ku ;  kk = ku - Wm ftil_u
  for (int c = 0; c < NZ; ++c) {
    double v = fv[c];
    for (int b2 = 0; b2 < NV; ++b2) v += 0.5 * (F[c * NZ + NX + b2] + F[(NX + b2) * NZ + c]) * ku[b2];
    fv[c] = v;
  }
  for (int a = 0; a < NV; ++a) {
    double v = ku[a];
    for (int b2 = 0; b2 < NV; ++b2) v -= Wk[a * NV + b2] * fv[NX + b2];
    s.kkm[k * NV + a] = v;
  }
  return 0;
}

#if TM_NL > 1
// ---- lane <-> stage sweeps (warp per instance, N <= 32) -----------------------------------------------------------
// The Riccati sweeps are chains over the stages with a handful of small mat-vecs per link.  Every lane keeps the blocks of
// "its" stage (A, B, K, W) in registers and the NX-vector travels from lane to lane by shuffle, so a sweep costs N links of
// register arithmetic instead of N rounds of shared-memory traffic and warp barriers.  Each scalar is computed by the same
// sequence of operations as in the sequential form below (one thread per instance, host twin): results are bitwise equal.
__device__ __forceinline__ double tm_shfl(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

struct TmLaneStage { double AB[NX * NZ], K[(NV > 0 ? NV : 1) * NX], W[(NV > 0 ? NV : 1) * (NV > 0 ? NV : 1)]; };
__device__ __forceinline__ void tm_lane_stage_load(const TmQpWs& s, int k, bool mine, TmLaneStage& L) {
#pragma unroll
  for (int e = 0; e < NX * NZ; ++e) L.AB[e] = mine ? s.AB[(size_t)k * NX * NZ + e] : 0.0;
#pragma unroll
  for (int e = 0; e < NV * NX; ++e) L.K[e] = mine ? s.K[(size_t)k * NV * NX + e] : 0.0;
#pragma unroll
  for (int e = 0; e < NV * NV; ++e) L.W[e] = mine ? s.Wm[(size_t)k * NV * NV + e] : 0.0;
}

// forward link: du = kk + K dx;  xo = [bk +] A dx + B du
__device__ __forceinline__ void tm_lane_fwd(const TmLaneStage& L, const double* kk, const double* dx, const double* bk, double* du, double* xo) {
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double v = kk[a];
#pragma unroll
    for (int j = 0; j < NX; ++j) v += L.K[a * NX + j] * dx[j];
    du[a] = v;
  }
#pragma unroll
  for (int i = 0; i < NX; ++i) {
    double v = bk ? bk[i] : 0.0;
#pragma unroll
    for (int j = 0; j < NX; ++j) v += L.AB[i * NZ + j] * dx[j];
#pragma unroll
    for (int a = 0; a < NV; ++a) v += L.AB[i * NZ + NX + a] * du[a];
    xo[i] = v;
  }
}

// backward link: fu = ru + B'p;  pn = rx + A'p + K'fu;  kk = -W fu
__device__ __forceinline__ void tm_lane_bwd(const TmLaneStage& L, const double* rk, const double* pin, double* pn, double* kk) {
  double fu[NV > 0 ? NV : 1];
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double v = rk[NX + a];
#pragma unroll
    for (int i = 0; i < NX; ++i) v += L.AB[i * NZ + NX + a] * pin[i];
    fu[a] = v;
  }
#pragma unroll
  for (int j = 0; j < NX; ++j) {
    double v = rk[j];
#pragma unroll
    for (int i = 0; i < NX; ++i) v += L.AB[i * NZ + j] * pin[i];
#pragma unroll
    for (int a = 0; a < NV; ++a) v += L.K[a * NX + j] * fu[a];
    pn[j] = v;
  }
#pragma unroll
  for (int a = 0; a < NV; ++a) {
    double v = 0.0;
#pragma unroll
    for (int b2 = 0; b2 < NV; ++b2) v -= L.W[a * NV + b2] * fu[b2];
    kk[a] = v;
  }
}

#endif  // TM_NL > 1 (lane <-> stage helpers)

// ---- base factorisation + main solve ----------------------------------------------------------------------------
// amask: inequality rows (k*nh + i) held as equalities.  Fills K, Wm, Pk, pm, Gc, gc, ncs and the step s.d of the base
// problem.  returns 0 ok, 3 not positive definite on the null space of the base rows, 6 base rows inconsistent.
TM_HD int tm_qp_factor(const TmProb& P, TmQpWs& s, const unsigned* amask, const double* e0, double rho) {
  const int N = P.N, nh = P.nh, nxt = P.nxt;
  const int lane = TM_LANE;
#if TM_NL == 1
  double Fl[NZ * NZ], fl[NZ], PABl[NX * NZ], pvl[NX];     // per-stage scratch: thread-local, statically indexed once the loops are unrolled
  double *const sF = Fl, *const sf = fl, *const sPAB = PABl, *const spv = pvl;
#else
  double *const sF = s.F, *const sf = s.f, *const sPAB = s.PAB, *const spv = s.pv;
#endif
#ifdef TM_TERM_ELIM
  // validation mode: terminal rows eliminated like base rows (exact null space; ill-conditioned when the inputs couple weakly)
  TM_UNROLL_T
  for (int e = lane; e < NX * NX; e += TM_NL) s.Pk[(size_t)N * NX * NX + e] = 0.0;
  for (int a = lane; a < NX; a += TM_NL) s.pm[N * NX + a] = 0.0;
  TM_UNROLL_T
  for (int e = lane; e < nxt * NX; e += TM_NL) s.Gc[(size_t)N * NX * NX + e] = (P.term_idx[e / NX] == e % NX) ? 1.0 : 0.0;
  for (int t = lane; t < nxt; t += TM_NL) s.gc[N * NX + t] = s.tr[t];
  if (lane == 0) s.ncs[N] = (double)nxt;
#else
  // terminal rows live in the dual active set (always-active equality members of the Schur complement); the base carries
  // their augmented-Lagrangian term rho/2 |T d_N + t|^2, which vanishes -- value and gradient -- at the QP solution
  TM_UNROLL_T
  for (int e = lane; e < NX * NX; e += TM_NL) {
    const int i = e / NX, j = e % NX;
    double v = 0.0;
    for (int t = 0; t < nxt; ++t) if (P.term_idx[t] == i && i == j) v += rho;
    s.Pk[(size_t)N * NX * NX + e] = v;
  }
  for (int a = lane; a < NX; a += TM_NL) {
    double v = 0.0;
    for (int t = 0; t < nxt; ++t) if (P.term_idx[t] == a) v += rho * s.tr[t];
    s.pm[N * NX + a] = v;
  }
  if (lane == 0) s.ncs[N] = 0.0;
#endif
  TM_SYNC();
  for (int k = N - 1; k >= 0; --k) {
    const TmP ABw = s.AB + (size_t)k * NX * NZ;
    const TmP Qk = s.Q + (size_t)k * NZ * NZ;
    const TmP Pnw = s.Pk + (size_t)(k + 1) * NX * NX;
    const TmP Gn = s.Gc + (size_t)(k + 1) * NX * NX;
    const int ncn = (int)s.ncs[k + 1];
#if TM_NL == 1
    // one thread per instance: the blocks every product below re-reads are staged once (registers / thread-local memory)
    double AB[NX * NZ], Pn[NX * NX], bk[NX];
#pragma unroll
    for (int e = 0; e < NX * NZ; ++e) AB[e] = ABw[e];
#pragma unroll
    for (int e = 0; e < NX * NX; ++e) Pn[e] = Pnw[e];
#pragma unroll
    for (int e = 0; e < NX; ++e) bk[e] = s.b[k * NX + e];
#else
    const TmP AB = ABw, Pn = Pnw;
    const TmP bk = s.b + k * NX;
#endif
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
    long long tq0 = clock64(), tq1 = 0;       // profiling build: cycles of the two block products P [A B] and Q + [A B]'(P [A B])
#endif
    TM_UNROLL_T
    for (int e = lane; e < NX * NZ; e += TM_NL) {
      const int i = e / NZ, c = e % NZ;
      double v = 0.0;
#pragma unroll
      for (int l = 0; l < NX; ++l) v += Pn[i * NX + l] * AB[l * NZ + c];
      sPAB[e] = v;
    }
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
    tq1 = clock64() - tq0;
#endif
    TM_UNROLL_T
    for (int i = lane; i < NX; i += TM_NL) {           // vv = P b + p
      double v = s.pm[(k + 1) * NX + i];
#pragma unroll
      for (int l = 0; l < NX; ++l) v += Pn[i * NX + l] * bk[l];
      spv[i] = v;
    }
    // candidate rows: constraint-to-go of stage k+1 through the dynamics, then the stage's own base rows
    TM_UNROLL_T
    for (int e = lane; e < ncn * (NZ + 1); e += TM_NL) {
      const int i = e / (NZ + 1), c = e % (NZ + 1);
      double v = (c == NZ) ? s.gc[(k + 1) * NX + i] : 0.0;
#pragma unroll
      for (int l = 0; l < NX; ++l) v += Gn[i * NX + l] * (c == NZ ? bk[l] : AB[l * NZ + c]);
      s.Ew[i * TM_ES + c] = v;
    }
    int nr = ncn;
#if NS > 0
    for (int i = 0; i < NS; ++i) {                    // equality rows  Jg_k,i (dx,du) - dus_i + g_k,i = 0: always held
      TM_UNROLL_T
      for (int c = lane; c <= NZ; c += TM_NL)
        s.Ew[nr * TM_ES + c] = (c == NZ) ? s.gv[k * NS + i] : (c < NZM ? s.Cg[((size_t)k * NS + i) * NZM + c] : (c == NZM + i ? -1.0 : 0.0));
      ++nr;
    }
#endif
#if NV > 0 && NV <= 4 && NS == 0 && !defined(TM_NO_FREE_STAGE)
    int simple = (ncn == 0);                          // every held row of the stage bounds one input of its own: fast path
    unsigned pinmask = 0u;
    double kuv[NV];
#pragma unroll
    for (int a = 0; a < NV; ++a) kuv[a] = 0.0;
#endif
    for (int i = 0; i < nh; ++i) {
      if (!tm_mask_get(amask, k * nh + i)) continue;
#if NV > 0 && NV <= 4 && NS == 0 && !defined(TM_NO_FREE_STAGE)
      {
        const int rp = P.rowpin[i];
        if (simple && rp >= 0 && !((pinmask >> rp) & 1u)) {
          // the general elimination's arithmetic on this row: scale to max-abs 1, divide by the pivot, ku = -offset
          const double cf = P.C[(size_t)i * NZ + NX + rp];
          const double inv = 1.0 / fabs(cf);
          const double ip = 1.0 / (cf * inv);
          const double kv = -((s.hv[k * nh + i] * inv) * ip);
          pinmask |= (1u << rp);
#pragma unroll
          for (int a = 0; a < NV; ++a) if (a == rp) kuv[a] = kv;
        } else simple = 0;
      }
#endif
      TM_UNROLL_T
      for (int c = lane; c <= NZ; c += TM_NL) s.Ew[nr * TM_ES + c] = (c == NZ) ? s.hv[k * nh + i] : P.C[(size_t)i * NZ + c];
      ++nr;
    }
    TM_SYNC();
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
    tq0 = clock64();
#endif
    TM_UNROLL_T
    for (int e = lane; e < NZ * NZ; e += TM_NL) {
      const int a = e / NZ, c = e % NZ;
      double v = Qk[e];
#pragma unroll
      for (int i = 0; i < NX; ++i) v += AB[i * NZ + a] * sPAB[i * NZ + c];
      sF[e] = v;
    }
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
    tq1 += clock64() - tq0;
    if (lane == 0) atomicAdd(P.prof_counters + 0, (unsigned long long)tq1);
#endif
    TM_UNROLL_T
    for (int c = lane; c < NZ; c += TM_NL) {
      double v = s.r[k * NZ + c];
#pragma unroll
      for (int i = 0; i < NX; ++i) v += AB[i * NZ + c] * spv[i];
      sf[c] = v;
    }
    TM_SYNC();
#if NV > 0 && NV <= 4 && NS == 0 && !defined(TM_NO_FREE_STAGE)
    if (lane == 0) s.sc[2] = (double)(simple ? tm_stage_factor_pinned(P, s, k, pinmask, kuv, sF, sf) : tm_stage_factor(P, s, k, nr, sF, sf));
#else
    if (lane == 0) s.sc[2] = (double)tm_stage_factor(P, s, k, nr, sF, sf);
#endif
    TM_SYNC();
    if (s.sc[2] != 0.0) return (int)s.sc[2];
    // P_k = [I;K]' F [I;K] (symmetrised), p_k = ftil_x + K' ftil_u
#if TM_NL == 1
    double Kk[(NV > 0 ? NV : 1) * NX];
#pragma unroll
    for (int e = 0; e < NV * NX; ++e) Kk[e] = s.K[(size_t)k * NV * NX + e];
#else
    const TmP Kk = s.K + (size_t)k * NV * NX;
#endif
    TM_UNROLL_T
    for (int e = lane; e < NX * NZ; e += TM_NL) {      // X = F_x. + K' F_u.
      const int i = e / NZ, c = e % NZ;
      double v = 0.5 * (sF[i * NZ + c] + sF[c * NZ + i]);
#pragma unroll
      for (int a = 0; a < NV; ++a) v += Kk[a * NX + i] * 0.5 * (sF[(NX + a) * NZ + c] + sF[c * NZ + NX + a]);
      sPAB[e] = v;
    }
    TM_SYNC();
    const TmP Pc = s.Pk + (size_t)k * NX * NX;
    TM_UNROLL_T
    for (int e = lane; e < NX * NX; e += TM_NL) {
      const int i = e / NX, j = e % NX;
      double vij = sPAB[i * NZ + j], vji = sPAB[j * NZ + i];
#pragma unroll
      for (int a = 0; a < NV; ++a) { vij += sPAB[i * NZ + NX + a] * Kk[a * NX + j]; vji += sPAB[j * NZ + NX + a] * Kk[a * NX + i]; }
      Pc[e] = 0.5 * (vij + vji);
    }
    TM_UNROLL_T
    for (int i = lane; i < NX; i += TM_NL) {
      double v = sf[i];
#pragma unroll
      for (int a = 0; a < NV; ++a) v += Kk[a * NX + i] * sf[NX + a];
      s.pm[k * NX + i] = v;
    }
    TM_SYNC();
  }
  // the constraint-to-go that reaches stage 0 must hold at the fixed x_0
  {
    const int nc0 = (int)s.ncs[0];
    int bad = 0;
    for (int i = 0; i < nc0; ++i) {
      double v = s.gc[i];
#pragma unroll
      for (int c = 0; c < NX; ++c) v += s.Gc[i * NX + c] * e0[c];
      if (fabs(v) > 1e-7) bad = 1;
    }
    if (bad) return 6;
  }
  // forward sweep of the main solve
#if TM_NL > 1
  if (N <= TM_NL) {                                    // lane <-> stage (tm_lane_fwd): same operations per scalar as the loop below
    const bool mine = lane < N;
    TmLaneStage L;
    tm_lane_stage_load(s, lane, mine, L);
    double dx[NX], du[NV > 0 ? NV : 1], xo[NX], kz[NV > 0 ? NV : 1], bk[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) { dx[i] = (lane == 0) ? e0[i] : 0.0; xo[i] = 0.0; bk[i] = mine ? s.b[lane * NX + i] : 0.0; }
#pragma unroll
    for (int a = 0; a < NV; ++a) { kz[a] = mine ? s.kkm[lane * NV + a] : 0.0; du[a] = 0.0; }
    for (int step = 0; step < N; ++step) {
      if (lane == step) tm_lane_fwd(L, kz, dx, bk, du, xo);
#pragma unroll
      for (int i = 0; i < NX; ++i) { const double t = tm_shfl(xo[i], step); if (lane == step + 1) dx[i] = t; }
    }
    if (mine) {
#pragma unroll
      for (int j = 0; j < NX; ++j) s.d[lane * NZ + j] = dx[j];
#pragma unroll
      for (int a = 0; a < NV; ++a) s.d[lane * NZ + NX + a] = du[a];
      if (lane == N - 1) {
#pragma unroll
        for (int i = 0; i < NX; ++i) s.d[N * NZ + i] = xo[i];
      }
    }
    for (int a = lane; a < NV; a += TM_NL) s.d[N * NZ + NX + a] = 0.0;
    TM_SYNC();
    return 0;
  }
#endif
  for (int a = lane; a < NX; a += TM_NL) s.d[a] = e0[a];
  TM_SYNC();
  for (int k = 0; k < N; ++k) {
    const TmP AB = s.AB + (size_t)k * NX * NZ;
    const TmP Kk = s.K + (size_t)k * NV * NX;
    const TmP dx = s.d + k * NZ;
    double du[NV > 0 ? NV : 1];
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      double v = s.kkm[k * NV + a];
#pragma unroll
      for (int j = 0; j < NX; ++j) v += Kk[a * NX + j] * dx[j];
      du[a] = v;
    }
    for (int a = lane; a < NV; a += TM_NL) s.d[k * NZ + NX + a] = du[a];
    for (int i = lane; i < NX; i += TM_NL) {
      double v = s.b[k * NX + i];
#pragma unroll
      for (int j = 0; j < NX; ++j) v += AB[i * NZ + j] * dx[j];
#pragma unroll
      for (int a = 0; a < NV; ++a) v += AB[i * NZ + NX + a] * du[a];
      s.d[(k + 1) * NZ + i] = v;
    }
    TM_SYNC();
  }
  for (int a = lane; a < NV; a += TM_NL) s.d[N * NZ + NX + a] = 0.0;
  TM_SYNC();
  return 0;
}

#if TM_NL > 1
__device__ __forceinline__ void tm_ricc_solve_lanes(const TmProb& P, TmQpWs& s, TmP rhs, TmP out, int kfrom) {
  const int N = P.N, lane = TM_LANE;
  const int kb = (kfrom >= N) ? N - 1 : kfrom;
  const bool mine = lane < N;
  TmLaneStage L;
  tm_lane_stage_load(s, lane, mine, L);
  double rk[NZ], pin[NX], pn[NX], kk[NV > 0 ? NV : 1];
#pragma unroll
  for (int c = 0; c < NZ; ++c) rk[c] = mine ? rhs[lane * NZ + c] : 0.0;
#pragma unroll
  for (int i = 0; i < NX; ++i) { pin[i] = (lane == kb && kfrom >= N) ? rhs[N * NZ + i] : 0.0; pn[i] = 0.0; }
#pragma unroll
  for (int a = 0; a < NV; ++a) kk[a] = 0.0;
  for (int step = kb; step >= 0; --step) {
    if (lane == step) tm_lane_bwd(L, rk, pin, pn, kk);
#pragma unroll
    for (int j = 0; j < NX; ++j) { const double t = tm_shfl(pn[j], step); if (lane == step - 1) pin[j] = t; }
  }
  // cost-to-go gradients of this solve (multiplier recovery): py_k = pn of lane k <= kb, the terminal right-hand side at N, else 0
  if (mine) {
#pragma unroll
    for (int j = 0; j < NX; ++j) s.py[lane * NX + j] = (lane <= kb) ? pn[j] : 0.0;
  }
  for (int a = lane; a < NX; a += TM_NL) s.py[N * NX + a] = (kfrom >= N) ? rhs[N * NZ + a] : 0.0;
  double dx[NX], du[NV > 0 ? NV : 1], xo[NX], kz[NV > 0 ? NV : 1];
#pragma unroll
  for (int i = 0; i < NX; ++i) { dx[i] = 0.0; xo[i] = 0.0; }
#pragma unroll
  for (int a = 0; a < NV; ++a) { kz[a] = (lane <= kb) ? kk[a] : 0.0; du[a] = 0.0; }
  for (int step = 0; step < N; ++step) {
    if (lane == step) tm_lane_fwd(L, kz, dx, nullptr, du, xo);
#pragma unroll
    for (int i = 0; i < NX; ++i) { const double t = tm_shfl(xo[i], step); if (lane == step + 1) dx[i] = t; }
  }
  if (mine) {
#pragma unroll
    for (int j = 0; j < NX; ++j) out[lane * NZ + j] = dx[j];
#pragma unroll
    for (int a = 0; a < NV; ++a) out[lane * NZ + NX + a] = du[a];
    if (lane == N - 1) {
#pragma unroll
      for (int i = 0; i < NX; ++i) out[N * NZ + i] = xo[i];
    }
  }
  for (int a = lane; a < NV; a += TM_NL) out[N * NZ + NX + a] = 0.0;
  TM_SYNC();
}

__device__ __forceinline__ void tm_ricc_col_lanes(const TmProb& P, TmQpWs& s, int qe, TmP mq) {
  const int N = P.N, nh = P.nh, NI = N * nh, lane = TM_LANE;
  const bool mine = lane < N;
  TmLaneStage L;
  tm_lane_stage_load(s, lane, mine, L);
  double rk[NZ], pin[NX], pn[NX], kk[NV > 0 ? NV : 1];
#pragma unroll
  for (int c = 0; c < NZ; ++c) rk[c] = 0.0;
#pragma unroll
  for (int i = 0; i < NX; ++i) { pin[i] = 0.0; pn[i] = 0.0; }
#pragma unroll
  for (int a = 0; a < NV; ++a) kk[a] = 0.0;
  int kb;
  if (qe >= NI) {
    const int ti = P.term_idx[qe - NI];
    kb = N - 1;
#pragma unroll
    for (int a = 0; a < NX; ++a) if (a == ti && lane == kb) pin[a] = -1.0;
  } else {
    kb = qe / nh;
    const double* Ci = P.C + (size_t)(qe % nh) * NZ;
#pragma unroll
    for (int b = 0; b < NZ; ++b) if (lane == kb) rk[b] = -Ci[b];
  }
  for (int step = kb; step >= 0; --step) {
    if (lane == step) tm_lane_bwd(L, rk, pin, pn, kk);
#pragma unroll
    for (int j = 0; j < NX; ++j) { const double t = tm_shfl(pn[j], step); if (lane == step - 1) pin[j] = t; }
  }
  double z[NZ], xo[NX], kz[NV > 0 ? NV : 1];
#pragma unroll
  for (int b = 0; b < NZ; ++b) z[b] = 0.0;
#pragma unroll
  for (int i = 0; i < NX; ++i) xo[i] = 0.0;
#pragma unroll
  for (int a = 0; a < NV; ++a) kz[a] = (lane <= kb) ? kk[a] : 0.0;
  for (int step = 0; step < N; ++step) {
    if (lane == step) tm_lane_fwd(L, kz, z, nullptr, z + NX, xo);
#pragma unroll
    for (int i = 0; i < NX; ++i) { const double t = tm_shfl(xo[i], step); if (lane == step + 1) z[i] = t; }
  }
  // row values of every stage, all lanes at once
  if (mine) {
    for (int i = 0; i < nh; ++i) {
      const double* Ci = P.C + (size_t)i * NZ;
      double t = 0.0;
#pragma unroll
      for (int b = 0; b < NZ; ++b) t += Ci[b] * z[b];
      mq[lane * nh + i] = t;
    }
  }
  for (int t = 0; t < P.nxt; ++t) {
    const int ti = P.term_idx[t];
    double v = 0.0;
#pragma unroll
    for (int a = 0; a < NX; ++a) if (a == ti) v = xo[a];
    v = tm_shfl(v, N - 1);
    if (lane == 0) mq[NI + t] = v;
  }
  TM_SYNC();
}
#endif  // TM_NL > 1

// homogeneous base solve:  out = argmin 1/2 d'Hd + rhs'd  over the null space of the base rows ( = -G rhs ).
// kfrom: last stage with a non-zero right-hand side.  The cost-to-go gradients go to s.py (multiplier recovery).
TM_HD void tm_ricc_solve(const TmProb& P, TmQpWs& s, TmP rhs, TmP out, int kfrom) {
  const int N = P.N;
  const int lane = TM_LANE;
#if TM_NL > 1
  if (N <= TM_NL) { tm_ricc_solve_lanes(P, s, rhs, out, kfrom); return; }
#endif
  const int kb = (kfrom >= N) ? N - 1 : kfrom;
  for (int e = lane; e < (N + 1) * NX; e += TM_NL) s.py[e] = (kfrom >= N && e >= N * NX) ? rhs[N * NZ + (e - N * NX)] : 0.0;
  TM_SYNC();
  for (int k = kb; k >= 0; --k) {
    const TmP AB = s.AB + (size_t)k * NX * NZ;
    const TmP Kk = s.K + (size_t)k * NV * NX;
    const TmP Wk = s.Wm + (size_t)k * NV * NV;
    const TmP rk = rhs + k * NZ;
    double pvr[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) pvr[i] = s.py[(k + 1) * NX + i];
    double fu[NV > 0 ? NV : 1];
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      double v = rk[NX + a];
#pragma unroll
      for (int i = 0; i < NX; ++i) v += AB[i * NZ + NX + a] * pvr[i];
      fu[a] = v;
    }
    for (int j = lane; j < NX; j += TM_NL) {
      double v = rk[j];
#pragma unroll
      for (int i = 0; i < NX; ++i) v += AB[i * NZ + j] * pvr[i];
#pragma unroll
      for (int a = 0; a < NV; ++a) v += Kk[a * NX + j] * fu[a];
      s.py[k * NX + j] = v;
    }
    for (int a = lane; a < NV; a += TM_NL) {
      double v = 0.0;
#pragma unroll
      for (int b2 = 0; b2 < NV; ++b2) v -= Wk[a * NV + b2] * fu[b2];
      s.kk[k * NV + a] = v;
    }
    TM_SYNC();
  }
  for (int a = lane; a < NX; a += TM_NL) out[a] = 0.0;
  TM_SYNC();
  for (int k = 0; k < N; ++k) {
    const TmP AB = s.AB + (size_t)k * NX * NZ;
    const TmP Kk = s.K + (size_t)k * NV * NX;
    const TmP dx = out + k * NZ;
    double dxr[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) dxr[j] = dx[j];
    double du[NV > 0 ? NV : 1];
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      double v = (k <= kb) ? s.kk[k * NV + a] : 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) v += Kk[a * NX + j] * dxr[j];
      du[a] = v;
    }
    for (int a = lane; a < NV; a += TM_NL) out[k * NZ + NX + a] = du[a];
    for (int i = lane; i < NX; i += TM_NL) {
      double v = 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) v += AB[i * NZ + j] * dxr[j];
#pragma unroll
      for (int a = 0; a < NV; ++a) v += AB[i * NZ + NX + a] * du[a];
      out[(k + 1) * NZ + i] = v;
    }
    TM_SYNC();
  }
  for (int a = lane; a < NV; a += TM_NL) out[N * NZ + NX + a] = 0.0;
  TM_SYNC();
}

// Dual-Hessian column of inequality row qe:  y = G n_qe is swept stage by stage and never stored; mq[e] = n_e' y for
// every inequality row e.  The NX-wide recursions are carried in registers by every lane (no synchronisation inside).
TM_HD void tm_ricc_col(const TmProb& P, TmQpWs& s, int qe, TmP mq) {
  const int N = P.N, nh = P.nh, NI = N * nh;
  const int lane = TM_LANE;
#if TM_NL > 1
  if (N <= TM_NL) { tm_ricc_col_lanes(P, s, qe, mq); return; }
#endif
  double pv[NX], rz[NZ];
#pragma unroll
  for (int a = 0; a < NX; ++a) pv[a] = 0.0;
#pragma unroll
  for (int b = 0; b < NZ; ++b) rz[b] = 0.0;
  int kb;
  if (qe >= NI) {
    const int ti = P.term_idx[qe - NI];
#pragma unroll
    for (int a = 0; a < NX; ++a) if (a == ti) pv[a] = -1.0;
    kb = N - 1;
  } else {
    kb = qe / nh;
    const double* Ci = P.C + (size_t)(qe % nh) * NZ;
#pragma unroll
    for (int b = 0; b < NZ; ++b) rz[b] = -Ci[b];
  }
  for (int k = kb; k >= 0; --k) {
    const TmP AB = s.AB + (size_t)k * NX * NZ;
    const TmP Kk = s.K + (size_t)k * NV * NX;
    const TmP Wk = s.Wm + (size_t)k * NV * NV;
    double fu[NV > 0 ? NV : 1], pn[NX];
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      double v = (k == kb) ? rz[NX + a] : 0.0;
#pragma unroll
      for (int i = 0; i < NX; ++i) v += AB[i * NZ + NX + a] * pv[i];
      fu[a] = v;
    }
#pragma unroll
    for (int j = 0; j < NX; ++j) {
      double v = (k == kb) ? rz[j] : 0.0;
#pragma unroll
      for (int i = 0; i < NX; ++i) v += AB[i * NZ + j] * pv[i];
#pragma unroll
      for (int a = 0; a < NV; ++a) v += Kk[a * NX + j] * fu[a];
      pn[j] = v;
    }
    for (int a = lane; a < NV; a += TM_NL) {
      double v = 0.0;
#pragma unroll
      for (int b2 = 0; b2 < NV; ++b2) v -= Wk[a * NV + b2] * fu[b2];
      s.kk[k * NV + a] = v;
    }
#pragma unroll
    for (int j = 0; j < NX; ++j) pv[j] = pn[j];
  }
  TM_SYNC();
  double z[NZ];
#pragma unroll
  for (int b = 0; b < NZ; ++b) z[b] = 0.0;
  for (int k = 0; k < N; ++k) {
    const TmP AB = s.AB + (size_t)k * NX * NZ;
    const TmP Kk = s.K + (size_t)k * NV * NX;
#pragma unroll
    for (int a = 0; a < NV; ++a) {
      double v = (k <= kb) ? s.kk[k * NV + a] : 0.0;
#pragma unroll
      for (int j = 0; j < NX; ++j) v += Kk[a * NX + j] * z[j];
      z[NX + a] = v;
    }
    for (int i = lane; i < nh; i += TM_NL) {
      const double* Ci = P.C + (size_t)i * NZ;
      double t = 0.0;
#pragma unroll
      for (int b = 0; b < NZ; ++b) t += Ci[b] * z[b];
      mq[k * nh + i] = t;
    }
    double xn[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) {
      double v = 0.0;
#pragma unroll
      for (int b = 0; b < NZ; ++b) v += AB[i * NZ + b] * z[b];
      xn[i] = v;
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) z[i] = xn[i];
  }
  for (int t = lane; t < P.nxt; t += TM_NL) {
    const int ti = P.term_idx[t];
    double v = 0.0;
#pragma unroll
    for (int a = 0; a < NX; ++a) if (a == ti) v = z[a];
    mq[NI + t] = v;
  }
  TM_SYNC();
}

// Dual-Hessian columns of ALL terminal rows (they enter the working set first, unconditionally): TM_TG columns share one pass
// over the stage blocks (A, B, K, W are read once per group instead of once per column, and the independent recursions
// overlap their memory latency).  Column of terminal row t goes to slot t of Mc.  Per column the same operations in the same
// order as tm_ricc_col: bitwise identical results.
#ifndef TM_TG
#if TMPC_NZ <= 8
#define TM_TG 2
#else
#define TM_TG 1            /* wide stages: the second set of recursion vectors would only spill */
#endif
#endif
TM_HD void tm_ricc_cols_term(const TmProb& P, TmQpWs& s, int E) {
  const int N = P.N, nh = P.nh, NI = N * nh, nxt = P.nxt;
  const int lane = TM_LANE;
#if TM_NL > 1
#ifdef TM_NO_FUSED_LANES
  if (N <= TM_NL) {
    for (int t = 0; t < nxt; ++t) tm_ricc_col_lanes(P, s, NI + t, s.Mc + (size_t)t * E);
    return;
  }
#endif
  if (N <= TM_NL) {                                   // lane <-> stage: one load of the stage blocks, TM_TG chains per pass
    const bool mine = lane < N;
    TmLaneStage L;
    tm_lane_stage_load(s, lane, mine, L);
    for (int t0 = 0; t0 < nxt; t0 += TM_TG) {
      const int ng = (nxt - t0 < TM_TG) ? nxt - t0 : TM_TG;
      double rk[NZ], pin[TM_TG][NX], pn[TM_TG][NX], kk[TM_TG][NV > 0 ? NV : 1];
#pragma unroll
      for (int c = 0; c < NZ; ++c) rk[c] = 0.0;
#pragma unroll
      for (int g = 0; g < TM_TG; ++g) {
        const int ti = g < ng ? P.term_idx[t0 + g] : -1;
#pragma unroll
        for (int i = 0; i < NX; ++i) { pin[g][i] = (i == ti && lane == N - 1) ? -1.0 : 0.0; pn[g][i] = 0.0; }
#pragma unroll
        for (int a = 0; a < NV; ++a) kk[g][a] = 0.0;
      }
      for (int step = N - 1; step >= 0; --step) {
        if (lane == step) {
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) tm_lane_bwd(L, rk, pin[g], pn[g], kk[g]);
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g)
#pragma unroll
          for (int j = 0; j < NX; ++j) { const double t = tm_shfl(pn[g][j], step); if (lane == step - 1) pin[g][j] = t; }
      }
      double z[TM_TG][NZ], xo[TM_TG][NX];
#pragma unroll
      for (int g = 0; g < TM_TG; ++g) {
#pragma unroll
        for (int b = 0; b < NZ; ++b) z[g][b] = 0.0;
#pragma unroll
        for (int i = 0; i < NX; ++i) xo[g][i] = 0.0;
      }
      for (int step = 0; step < N; ++step) {
        if (lane == step) {
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) tm_lane_fwd(L, kk[g], z[g], nullptr, z[g] + NX, xo[g]);
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g)
#pragma unroll
          for (int i = 0; i < NX; ++i) { const double t = tm_shfl(xo[g][i], step); if (lane == step + 1) z[g][i] = t; }
      }
#pragma unroll
      for (int g = 0; g < TM_TG; ++g) {               // static g: the recursion vectors stay in registers
        if (g >= ng) continue;
        const TmP mq = s.Mc + (size_t)(t0 + g) * E;
        if (mine) {
          for (int i = 0; i < nh; ++i) {
            const double* Ci = P.C + (size_t)i * NZ;
            double t = 0.0;
#pragma unroll
            for (int b = 0; b < NZ; ++b) t += Ci[b] * z[g][b];
            mq[lane * nh + i] = t;
          }
        }
        for (int t = 0; t < nxt; ++t) {
          const int ti = P.term_idx[t];
          double v = 0.0;
#pragma unroll
          for (int a = 0; a < NX; ++a) if (a == ti) v = xo[g][a];
          v = tm_shfl(v, N - 1);
          if (lane == 0) mq[NI + t] = v;
        }
      }
      TM_SYNC();
    }
    return;
  }
#endif
  for (int t0 = 0; t0 < nxt; t0 += TM_TG) {
    const int ng = (nxt - t0 < TM_TG) ? nxt - t0 : TM_TG;
    double pv[TM_TG][NX];
#pragma unroll
    for (int g = 0; g < TM_TG; ++g) {
      const int ti = g < ng ? P.term_idx[t0 + g] : -1;
#pragma unroll
      for (int a = 0; a < NX; ++a) pv[g][a] = (a == ti) ? -1.0 : 0.0;
    }
    for (int k = N - 1; k >= 0; --k) {
      const TmP AB = s.AB + (size_t)k * NX * NZ;
      const TmP Kk = s.K + (size_t)k * NV * NX;
      const TmP Wk = s.Wm + (size_t)k * NV * NV;
      double fu[TM_TG][NV > 0 ? NV : 1], pn[TM_TG][NX];
#pragma unroll
      for (int a = 0; a < NV; ++a) {
        double v[TM_TG];
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) v[g] = 0.0;
#pragma unroll
        for (int i = 0; i < NX; ++i) {
          const double ab = AB[i * NZ + NX + a];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) v[g] += ab * pv[g][i];
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) fu[g][a] = v[g];
      }
#pragma unroll
      for (int j = 0; j < NX; ++j) {
        double v[TM_TG];
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) v[g] = 0.0;
#pragma unroll
        for (int i = 0; i < NX; ++i) {
          const double ab = AB[i * NZ + j];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) v[g] += ab * pv[g][i];
        }
#pragma unroll
        for (int a = 0; a < NV; ++a) {
          const double kv = Kk[a * NX + j];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) v[g] += kv * fu[g][a];
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) pn[g][j] = v[g];
      }
      for (int a = lane; a < NV; a += TM_NL) {
        double v[TM_TG];
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) v[g] = 0.0;
#pragma unroll
        for (int b2 = 0; b2 < NV; ++b2) {
          const double wv = Wk[a * NV + b2];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) v[g] -= wv * fu[g][b2];
        }
        s.kk[k * NV + a] = v[0];                       // feed-forward of column g: kk (g = 0), y (g = 1; free until the correction solve)
#if TM_TG > 1
        s.y[k * NV + a] = v[1];
#endif
      }
#pragma unroll
      for (int g = 0; g < TM_TG; ++g)
#pragma unroll
        for (int j = 0; j < NX; ++j) pv[g][j] = pn[g][j];
    }
    TM_SYNC();
    double z[TM_TG][NZ];
#pragma unroll
    for (int g = 0; g < TM_TG; ++g)
#pragma unroll
      for (int b = 0; b < NZ; ++b) z[g][b] = 0.0;
    for (int k = 0; k < N; ++k) {
      const TmP AB = s.AB + (size_t)k * NX * NZ;
      const TmP Kk = s.K + (size_t)k * NV * NX;
#pragma unroll
      for (int a = 0; a < NV; ++a) {
        double v[TM_TG];
        v[0] = s.kk[k * NV + a];
#if TM_TG > 1
        v[1] = s.y[k * NV + a];
#endif
#pragma unroll
        for (int j = 0; j < NX; ++j) {
          const double kv = Kk[a * NX + j];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) v[g] += kv * z[g][j];
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) z[g][NX + a] = v[g];
      }
      for (int i = lane; i < nh; i += TM_NL) {
        const double* Ci = P.C + (size_t)i * NZ;
        double t[TM_TG];
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) t[g] = 0.0;
#pragma unroll
        for (int b = 0; b < NZ; ++b) {
          const double cv = Ci[b];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) t[g] += cv * z[g][b];
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) if (g < ng) s.Mc[(size_t)(t0 + g) * E + k * nh + i] = t[g];
      }
      double xn[TM_TG][NX];
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        double v[TM_TG];
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) v[g] = 0.0;
#pragma unroll
        for (int b = 0; b < NZ; ++b) {
          const double ab = AB[i * NZ + b];
#pragma unroll
          for (int g = 0; g < TM_TG; ++g) v[g] += ab * z[g][b];
        }
#pragma unroll
        for (int g = 0; g < TM_TG; ++g) xn[g][i] = v[g];
      }
#pragma unroll
      for (int g = 0; g < TM_TG; ++g)
#pragma unroll
        for (int i = 0; i < NX; ++i) z[g][i] = xn[g][i];
    }
#pragma unroll
    for (int g = 0; g < TM_TG; ++g) {
      if (g >= ng) continue;
      for (int t = lane; t < nxt; t += TM_NL) {
        const int ti = P.term_idx[t];
        double v = 0.0;
#pragma unroll
        for (int a = 0; a < NX; ++a) if (a == ti) v = z[g][a];
        s.Mc[(size_t)(t0 + g) * E + NI + t] = v;
      }
    }
    TM_SYNC();
  }
}

TM_HD double tm_erow_dot(const TmProb& P, int e, TmP v) {       // n_e' v: e < N*nh inequality row k*nh + i, else terminal row
  if (e >= P.N * P.nh) return v[P.N * NZ + P.term_idx[e - P.N * P.nh]];
  const int k = e / P.nh, i = e % P.nh;
  double t = 0.0;
  const double* Ci = P.C + (size_t)i * NZ;
  const TmP vk = v + k * NZ;
#pragma unroll
  for (int b = 0; b < NZ; ++b) t += Ci[b] * vk[b];
  return t;
}

// rebuild the Cholesky factor Lf of S_ij = Mc[j][acte_i] (i, j < m) after a deletion (single lane)
TM_HD int tm_schur_refactor(TmQpWs& s, int m, int M, int E) {
  for (int i = 0; i < m; ++i)
    for (int j = 0; j <= i; ++j) s.Lf[TM_LFI(i, j)] = s.Mc[(size_t)j * E + (int)s.acte[i]];
  for (int c = 0; c < m; ++c) {
    double dg = s.Lf[TM_LFI(c, c)];
    for (int l = 0; l < c; ++l) dg -= s.Lf[TM_LFI(c, l)] * s.Lf[TM_LFI(c, l)];
    if (!(dg > 0.0)) return 0;
    const double ld = sqrt(dg);
    s.Lf[TM_LFI(c, c)] = ld;
    for (int i = c + 1; i < m; ++i) {
      double v = s.Lf[TM_LFI(i, c)];
      for (int l = 0; l < c; ++l) v -= s.Lf[TM_LFI(i, l)] * s.Lf[TM_LFI(c, l)];
      s.Lf[TM_LFI(i, c)] = v / ld;
    }
  }
  return 1;
}

// ---- Goldfarb-Idnani dual active set over the factorised base ---------------------------------------------------
// Row universe e: e < N*nh inequality row (k = e / nh, i = e % nh), e >= N*nh terminal row.  The terminal rows enter
// first as equality members (full step, sign-free multiplier, never dropped); then the rows outside the base mask that
// are violated enter one at a time.  The primal iterate is never updated inside the loop (one correction solve at the
// end).  returns 0 ok, 2 infeasible, 7 working-set overflow.
TM_HD int tm_qp_gi(const TmProb& P, TmQpWs& s, const unsigned* amask, int& m_out, int& n_gi, int& n_ricc) {
  const int N = P.N, nh = P.nh, M = P.maxact;
  const int lane = TM_LANE;
  const int NI = N * nh;
#ifdef TM_TERM_ELIM
  const int neq = 0;
#else
  const int neq = P.nxt;
#endif
  const int E = NI + P.nxt;
  for (int k = lane; k < N; k += TM_NL) {       // row values at the base solution, one stage's step loaded once
    double z[NZ];
#pragma unroll
    for (int b = 0; b < NZ; ++b) z[b] = s.d[k * NZ + b];
    for (int i = 0; i < nh; ++i) {
      const int e = k * nh + i;
      double v = 0.0;
      if (!tm_mask_get(amask, e)) {
        const double* Ci = P.C + (size_t)i * NZ;
        double t = 0.0;
#pragma unroll
        for (int b = 0; b < NZ; ++b) t += Ci[b] * z[b];
        v = s.hv[e] + t;
      }
      s.sl[e] = v;
    }
  }
  for (int t = lane; t < P.nxt; t += TM_NL) s.sl[NI + t] = s.tr[t] + s.d[N * NZ + P.term_idx[t]];
  TM_SYNC();
  int m = 0, ret = 0, eq_next = 0;
  const int maxit = 4 * NI + 8 + neq;
  if (neq > 0) { tm_ricc_cols_term(P, s, E); n_ricc += neq; }   // the terminal rows' columns, slot t = row t
  for (int it = 0; it < maxit && !ret; ++it) {
    int qe, is_eq = 0;
    double sval;
    if (eq_next < neq) {
      qe = NI + eq_next;
      ++eq_next;
      is_eq = 1;
      sval = s.sl[qe];
    } else {
      double best = TM_INF;
      int bid = 0x7fffffff;
#if TM_NL == 1
      for (int k = 0, e = 0; k < N; ++k)
        for (int i = 0; i < nh; ++i, ++e) {
          if ((k == 0 && P.relax0[i]) || tm_mask_get(amask, e)) continue;
          const double v = s.sl[e] / fmax(1.0, fabs(P.c[i]));
          if (v < best) { best = v; bid = e; }
        }
#else
      for (int e = lane; e < NI; e += TM_NL) {
        const int k = e / nh, i = e % nh;
        if ((k == 0 && P.relax0[i]) || tm_mask_get(amask, e)) continue;
        const double v = s.sl[e] / fmax(1.0, fabs(P.c[i]));
        if (v < best) { best = v; bid = e; }
      }
#endif
      tm_wargmin(best, bid);
      if (!(best < -1e-10)) break;            // primal feasible: optimal
      int dup = 0;                            // a working-set row can only show up here through round-off
      for (int j2 = 0; j2 < m; ++j2) if ((int)s.acte[j2] == bid) dup = 1;
      if (dup) break;
      qe = bid;
      sval = s.sl[qe];
    }
    if (m >= M) { ret = 7; break; }
    TmP mq = s.Mc + (size_t)m * E;            // candidate column, becomes member m when added
    if (is_eq) {                              // precomputed (slot qe - NI); an earlier terminal row was skipped as redundant: move it down
      const int q = qe - NI;
      if (q != m) {
        for (int e = lane; e < E; e += TM_NL) mq[e] = s.Mc[(size_t)q * E + e];
        TM_SYNC();
      }
    } else {
      tm_ricc_col(P, s, qe, mq);
      ++n_gi;
      ++n_ricc;
    }
    const double yq = mq[qe];
    double nq = 0.0;
    int added = 0;
    for (int inner = 0; inner < M + 2; ++inner) {
      if (lane == 0) {                        // l = L^-1 S_Aq (cA), r = L^-T l (rv)
        double ll = 0.0;
        for (int i = 0; i < m; ++i) {
          double v = mq[(int)s.acte[i]];
          for (int l = 0; l < i; ++l) v -= s.Lf[TM_LFI(i, l)] * s.cA[l];
          v /= s.Lf[TM_LFI(i, i)];
          s.cA[i] = v;
          ll += v * v;
        }
        for (int i = m - 1; i >= 0; --i) {
          double v = s.cA[i];
          for (int l = i + 1; l < m; ++l) v -= s.Lf[TM_LFI(l, i)] * s.rv[l];
          s.rv[i] = v / s.Lf[TM_LFI(i, i)];
        }
        s.sc[0] = ll;
      }
      TM_SYNC();
      const double zn = yq - s.sc[0];
      double t1 = TM_INF;
      int jd = -1;
      for (int j2 = 0; j2 < m; ++j2) {
        if ((int)s.acte[j2] >= NI) continue;           // equality members are never dropped
        const double rj = s.rv[j2];
        if (rj > 1e-14) { const double tj = s.nu[j2] / rj; if (tj < t1) { t1 = tj; jd = j2; } }
      }
      const int dependent = !(zn > 1e-11 * fmax(yq, 1e-300));
      double t;
      int do_add = 0;
      if (dependent) {
        if (is_eq) {                                   // redundant terminal row: skip it if it already holds
          if (fabs(sval) > 1e-7) ret = 2;
          added = 2;
          break;
        }
        if (jd < 0) { ret = 2; break; }
        t = t1;
      } else {
        const double t2 = -sval / zn;
        if (is_eq || t2 <= t1) { t = t2; do_add = 1; } else t = t1;
        // row values along the step: four rows at a time (independent chains); base rows are never candidates
        for (int e0 = lane; e0 < E; e0 += 4 * TM_NL) {
          int ee[4];
          double acc[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            ee[q] = e0 + q * TM_NL;
            if (ee[q] >= E || (ee[q] < NI && tm_mask_get(amask, ee[q]))) ee[q] = -1;
            acc[q] = ee[q] >= 0 ? mq[ee[q]] : 0.0;
          }
          for (int j2 = 0; j2 < m; ++j2) {
            const double rj = s.rv[j2];
            const TmP col = s.Mc + (size_t)j2 * E;
#pragma unroll
            for (int q = 0; q < 4; ++q) if (ee[q] >= 0) acc[q] -= rj * col[ee[q]];
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) if (ee[q] >= 0) s.sl[ee[q]] += t * acc[q];
        }
        sval += t * zn;
      }
      TM_SYNC();
      for (int j2 = lane; j2 < m; j2 += TM_NL) s.nu[j2] -= t * s.rv[j2];
      nq += t;
      TM_SYNC();
      if (do_add) {
        if (lane == 0) {
          for (int l = 0; l < m; ++l) s.Lf[TM_LFI(m, l)] = s.cA[l];
          s.Lf[TM_LFI(m, m)] = sqrt(zn);
          s.acte[m] = (double)qe; s.nu[m] = nq;
        }
        TM_SYNC();
        ++m;
        added = 1;
        break;
      }
      // drop member jd: shift members jd+1..m-1 and the candidate column down by one slot, rebuild the factor
      for (int a = jd; a < m; ++a) {
        for (int e = lane; e < E; e += TM_NL) s.Mc[(size_t)a * E + e] = s.Mc[(size_t)(a + 1) * E + e];
        TM_SYNC();
      }
      if (lane == 0) {
        for (int a = jd; a < m - 1; ++a) { s.acte[a] = s.acte[a + 1]; s.nu[a] = s.nu[a + 1]; }
      }
      --m;
      TM_SYNC();
      mq = s.Mc + (size_t)m * E;
      if (lane == 0) s.sc[1] = (double)tm_schur_refactor(s, m, M, E);
      TM_SYNC();
      if (s.sc[1] == 0.0) { ret = 2; break; }
    }
    if (ret) break;
    if (!added) { ret = 2; break; }
    if (it == maxit - 1) ret = 2;
  }
  m_out = m;
  return ret;
}

// ---- multipliers of the base rows -------------------------------------------------------------------------------
// Stage-wise stationarity with the final step d and gradient r' (r plus the dual active-set rows' terms):
//     Q z_k + r'_k + [A B]' lam_{k+1} + sum_{i in A_k} C_i' mu_i = [lam_k ; 0],   lam_k = P_k x_k + p_k + Gc_k' nu_k
// solved forwards for (nu_{k+1}, mu) by least squares on the (consistent) nz equations of every stage.  Stages whose
// neighbours carry no constraint-to-go are independent of each other (lane <-> stage); the others chain through nu.
// Writes lq (n_g, CasADi sign) completely.  lamh: multipliers of the dual active-set rows, already in lq.
TM_HD void tm_qp_recover_stage(const TmProb& P, TmQpWs& s, const unsigned* amask, int k, const double* nu_k, double* nu_next,
                               double* lq) {
  const int nh = P.nh;
  const TmP AB = s.AB + (size_t)k * NX * NZ;
  const TmP Qk = s.Q + (size_t)k * NZ * NZ;
  const int nck = (int)s.ncs[k], ncn = (int)s.ncs[k + 1];
  double z[NZ], xn[NX], lin[NX], cst[NX], rh[NZ];
#pragma unroll
  for (int c = 0; c < NZ; ++c) z[c] = s.d[k * NZ + c];
#pragma unroll
  for (int i = 0; i < NX; ++i) xn[i] = s.d[(k + 1) * NZ + i];
  for (int i = 0; i < NX; ++i) {                      // lam_k and the cost-to-go part of lam_{k+1}
    double a = s.pm[k * NX + i] + s.py[k * NX + i], b2 = s.pm[(k + 1) * NX + i] + s.py[(k + 1) * NX + i];
    for (int l = 0; l < NX; ++l) {
      a += s.Pk[(size_t)k * NX * NX + i * NX + l] * z[l];
      b2 += s.Pk[(size_t)(k + 1) * NX * NX + i * NX + l] * xn[l];
    }
    for (int q = 0; q < nck; ++q) a += s.Gc[(size_t)k * NX * NX + q * NX + i] * nu_k[q];
    lin[i] = a; cst[i] = b2;
  }
  for (int c = 0; c < NZ; ++c) {                      // rh = [lam_k;0] - (Q z + r') - [A B]' cst
    double v = (c < NX ? lin[c] : 0.0) - s.rhs[k * NZ + c];
    for (int e = 0; e < NZ; ++e) v -= 0.5 * (Qk[c * NZ + e] + Qk[e * NZ + c]) * z[e];
    for (int i = 0; i < NX; ++i) v -= AB[i * NZ + c] * cst[i];
    rh[c] = v;
  }
  // rows: Gc_{k+1} [A B]  |  C_i, i in A_k        (at most NZ independent ones)
  double Er[NZ * NZ], Gm[NZ * NZ], et[NZ];
  int rid[NZ];
  int nr = 0;
  for (int q = 0; q < ncn && nr < NZ; ++q) {
    for (int c = 0; c < NZ; ++c) {
      double v = 0.0;
      for (int l = 0; l < NX; ++l) v += s.Gc[(size_t)(k + 1) * NX * NX + q * NX + l] * AB[l * NZ + c];
      Er[nr * NZ + c] = v;
    }
    rid[nr++] = -1 - q;
  }
#if NS > 0
  for (int i = 0; i < NS && nr < NZ; ++i) {
    for (int c = 0; c < NZ; ++c) Er[nr * NZ + c] = c < NZM ? s.Cg[((size_t)k * NS + i) * NZM + c] : (c == NZM + i ? -1.0 : 0.0);
    rid[nr++] = 100000 + i;
  }
#endif
  for (int i = 0; i < nh && nr < NZ; ++i) {
    if (!tm_mask_get(amask, k * nh + i)) continue;
    for (int c = 0; c < NZ; ++c) Er[nr * NZ + c] = P.C[(size_t)i * NZ + c];
    rid[nr++] = i;
  }
  for (int i = 0; i < nr; ++i) {
    double v = 0.0;
    for (int c = 0; c < NZ; ++c) v += Er[i * NZ + c] * rh[c];
    et[i] = v;
    for (int j = 0; j <= i; ++j) {
      double g = 0.0;
      for (int c = 0; c < NZ; ++c) g += Er[i * NZ + c] * Er[j * NZ + c];
      Gm[i * NZ + j] = g;
    }
  }
  // Cholesky of E E' with dependent rows skipped (their multiplier is set to zero)
  int skip[NZ];
  for (int c = 0; c < nr; ++c) {
    double dg = Gm[c * NZ + c];
    const double dg0 = dg;
    for (int l = 0; l < c; ++l) if (!skip[l]) dg -= Gm[c * NZ + l] * Gm[c * NZ + l];
    skip[c] = !(dg > 1e-12 * fmax(dg0, 1e-300));
    if (skip[c]) continue;
    const double ld = sqrt(dg);
    Gm[c * NZ + c] = ld;
    for (int i = c + 1; i < nr; ++i) {
      double v = Gm[i * NZ + c];
      for (int l = 0; l < c; ++l) if (!skip[l]) v -= Gm[i * NZ + l] * Gm[c * NZ + l];
      Gm[i * NZ + c] = v / ld;
    }
  }
  for (int i = 0; i < nr; ++i) {
    if (skip[i]) { et[i] = 0.0; continue; }
    double v = et[i];
    for (int l = 0; l < i; ++l) if (!skip[l]) v -= Gm[i * NZ + l] * et[l];
    et[i] = v / Gm[i * NZ + i];
  }
  for (int i = nr - 1; i >= 0; --i) {
    if (skip[i]) continue;
    double v = et[i];
    for (int l = i + 1; l < nr; ++l) if (!skip[l]) v -= Gm[l * NZ + i] * et[l];
    et[i] = v / Gm[i * NZ + i];
  }
#if defined(TM_DEBUG_QP) && !defined(__CUDA_ARCH__)
  {
    double res = 0.0, rmax = 0.0;
    for (int c = 0; c < NZ; ++c) {
      double v = rh[c];
      for (int i = 0; i < nr; ++i) v -= Er[i * NZ + c] * et[i];
      res = fmax(res, fabs(v)); rmax = fmax(rmax, fabs(rh[c]));
    }
    if (res > 1e-9 * fmax(1.0, rmax)) {
      fprintf(stderr, "[qp] recover stage %d: LS residual %.2e (rhs %.2e, nr %d, ncn %d, nck %d) rh:", k, res, rmax, nr, ncn, nck);
      for (int c = 0; c < NZ; ++c) fprintf(stderr, " %.2e", rh[c]);
      fprintf(stderr, " | lin:"); for (int c = 0; c < NX; ++c) fprintf(stderr, " %.2e", lin[c]);
      fprintf(stderr, " | cst:"); for (int c = 0; c < NX; ++c) fprintf(stderr, " %.2e", cst[c]);
      { double pn = 0, qn = 0, xnn = 0, yn = 0; for (int e = 0; e < NX * NX; ++e) pn = fmax(pn, fabs(s.Pk[(size_t)(k + 1) * NX * NX + e]));
        for (int e = 0; e < NX; ++e) { qn = fmax(qn, fabs(s.pm[(k + 1) * NX + e])); yn = fmax(yn, fabs(s.py[(k + 1) * NX + e])); xnn = fmax(xnn, fabs(xn[e])); }
        fprintf(stderr, " | |P+|=%.2e |pm+|=%.2e |py+|=%.2e |x+|=%.2e", pn, qn, yn, xnn); }
      fprintf(stderr, "\n");
    }
  }
#endif
  for (int q = 0; q < NX; ++q) nu_next[q] = 0.0;
  for (int i = 0; i < nr; ++i) {
    if (rid[i] < 0) nu_next[-1 - rid[i]] = et[i];
    else if (rid[i] >= 100000) lq[tm_gg(P, k) + rid[i] - 100000] = et[i];
    else lq[tm_gh(P, k) + rid[i]] = et[i];
  }
  for (int i = 0; i < NX; ++i) {                      // lam_{k+1} = multiplier of dynamics row k
    double v = cst[i];
    for (int q = 0; q < ncn; ++q) v += s.Gc[(size_t)(k + 1) * NX * NX + q * NX + i] * nu_next[q];
    lq[tm_gdyn(P, k) + i] = v;
  }
  if (k == 0) for (int i = 0; i < NX; ++i) lq[i] = -lin[i];
}

TM_HD void tm_qp_recover(const TmProb& P, TmQpWs& s, const unsigned* amask, double* lq) {
  const int N = P.N;
  const int lane = TM_LANE;
  int kseq = N;                                       // first stage of the sequential tail
  for (int k = 0; k <= N; ++k) if ((int)s.ncs[k] > 0) { kseq = k > 0 ? k - 1 : 0; break; }
  if (kseq > N - 1) kseq = N - 1;
  double nu0[NX], nu1[NX];
#pragma unroll
  for (int q = 0; q < NX; ++q) nu0[q] = 0.0;
  for (int k = lane; k < kseq; k += TM_NL) tm_qp_recover_stage(P, s, amask, k, nu0, nu1, lq);
  TM_SYNC();
  if (lane == 0) {
    for (int k = kseq; k < N; ++k) {
      tm_qp_recover_stage(P, s, amask, k, nu0, nu1, lq);
#pragma unroll
      for (int q = 0; q < NX; ++q) nu0[q] = nu1[q];
    }
#ifdef TM_TERM_ELIM
    for (int t = 0; t < P.nxt; ++t) lq[tm_gterm(P) + t] = nu0[t];    // Gc_N = the terminal rows themselves
#endif
  }
  TM_SYNC();
}

// Perturbed solve used to tabulate the solution map of the first QP after reset() (tm_qp0_*, tmpc_core.cuh): the base
// problem (no dual active set) is solved for modified data and the result goes to (dout, lout).
struct TmQpPert {
  int homog;      // 1: zero all offsets (gradient r, dynamics defect b, terminal residual): pure linear response; the x_0 offset is always zeroed
  int e0_unit;    // >= 0: x_0 offset = unit vector e0_unit
  int row;        // >= 0: gradient -= n_row (response to a unit multiplier on inequality row `row` = k*nh + i)
  double *dout, *lout;
};

// stage data of the QP at the iterate (W, LAM) with the linearisation in LIN
TM_HD void tm_qp_setup(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& s, int use_exact) {
  const int N = P.N, nh = P.nh, nxt = P.nxt;
  const int lane = TM_LANE;
  const double* w = S.W + inst * P.n_w;
  const double* lin = S.LIN + inst * P.N * (int64_t)TM_LSZ;
  for (int e = lane; e < N * NX * NZ; e += TM_NL) {   // [A B 0]: the slack columns of the dynamics are zero
    int k = e / (NX * NZ), o = e % (NX * NZ), i = o / NZ, c = o % NZ;
    s.AB[e] = c < NZM ? lin[(size_t)k * TM_LSZ + NX + i * NZM + c] : 0.0;
  }
  for (int e = lane; e < N * NX; e += TM_NL) { int k = e / NX, a = e % NX; s.b[e] = lin[(size_t)k * TM_LSZ + a] - w[(k + 1) * NZ + a]; }
  if (P.economic) {
    // economic stage cost l(x,u) + scost'usc (pmpc.py:299-301,338-339): Q_k = d2l/d(x,u)2 (+ lam' d2F) on the (x,u) block and
    // zero on the slacks, r_k = (dl/d(x,u), 0_ns, scost) at the iterate.  l lives on (x,u) only: tmpc_cost_grad / _hess write
    // NZM / NZM x NZM values.  scost comes from the usc entries of q (MpcProblem.device_tables).
    for (int k = lane; k < N; k += TM_NL) {
      const double* qk = P.q + (size_t)((S.phase + k) % P.p) * NZ;
      double z[NZ], gl[NZM], Hl[NZM * NZM];
#pragma unroll
      for (int b = 0; b < NZ; ++b) z[b] = w[k * NZ + b];
      tmpc_cost_grad(z, z + NX, gl);
      tmpc_cost_hess(z, z + NX, Hl);
      for (int i = 0; i < NZ; ++i) {
        for (int j = 0; j < NZ; ++j) {
          double v = 0.0;
          if (i < NZM && j < NZM) {
            v = 0.5 * (Hl[i * NZM + j] + Hl[j * NZM + i]);
            if (use_exact) v += lin[(size_t)k * TM_LSZ + NX + NX * NZM + (i <= j ? tm_pair_idx(i, j) : tm_pair_idx(j, i))];
          }
          s.Q[(size_t)k * NZ * NZ + i * NZ + j] = v;
        }
        s.r[k * NZ + i] = i < NZM ? gl[i] : (i < NZM + NS ? 0.0 : qk[i]);
      }
    }
  } else {
    for (int e = lane; e < N * NZ * NZ; e += TM_NL) {
      int k = e / (NZ * NZ), o = e % (NZ * NZ), i = o / NZ, j = o % NZ;
      int ph = (S.phase + k) % P.p;
      double v = P.H[(size_t)ph * NZ * NZ + o];
      if (use_exact && i < NZM && j < NZM) v += lin[(size_t)k * TM_LSZ + NX + NX * NZM + (i <= j ? tm_pair_idx(i, j) : tm_pair_idx(j, i))];
      s.Q[e] = v;
    }
    for (int e = lane; e < N * NZ; e += TM_NL) {
      int k = e / NZ, i = e % NZ;
      int ph = (S.phase + k) % P.p;
      const double* Hk = P.H + (size_t)ph * NZ * NZ + (size_t)i * NZ;
      const double* wr = P.wref + (size_t)ph * NZ;
      double v = P.q[(size_t)ph * NZ + i];
#pragma unroll
      for (int j = 0; j < NZ; ++j) v += Hk[j] * (w[k * NZ + j] - wr[j]);
      s.r[e] = v;
    }
  }
  for (int a = lane; a < NZ; a += TM_NL) s.r[N * NZ + a] = 0.0;
#if NS > 0
  // slacked nonlinear rows at the iterate: value h_nl(x_k,u_k) - us_k, Jacobian, and (exact Hessian) lam_g' d2 h_nl added to Q
  TM_SYNC();
  for (int k = lane; k < N; k += TM_NL) {
    double z[NZ], gvl[NS], Jg[NS * NZM];
#pragma unroll
    for (int b = 0; b < NZ; ++b) z[b] = w[k * NZ + b];
    tmpc_gnl_jac(z, z + NX, gvl, Jg);
    for (int i = 0; i < NS; ++i) s.gv[k * NS + i] = gvl[i] - z[NZM + i];
    for (int e = 0; e < NS * NZM; ++e) s.Cg[(size_t)k * NS * NZM + e] = Jg[e];
    if (use_exact) {
      double Hg[NZM * NZM];
      tmpc_gnl_hess(z, z + NX, S.LAM + inst * P.n_g + tm_gg(P, k), Hg);
      for (int i = 0; i < NZM; ++i)
        for (int j = 0; j < NZM; ++j) s.Q[(size_t)k * NZ * NZ + i * NZ + j] += 0.5 * (Hg[i * NZM + j] + Hg[j * NZM + i]);
    }
  }
#endif
  for (int e = lane; e < N * nh; e += TM_NL) {
    int k = e / nh, i = e % nh;
    double v = P.c[i];
#pragma unroll
    for (int j = 0; j < NZ; ++j) v += P.C[(size_t)i * NZ + j] * w[k * NZ + j];
    s.hv[e] = v;
  }
  TmL e0 = s.pv + 2 * NX;
  for (int a = lane; a < NX; a += TM_NL) e0[a] = S.X0[inst * NX + a] - w[a];
  {
    const double* xrN = P.wref + (size_t)((S.phase + N) % P.p) * NZ;
    for (int t = lane; t < nxt; t += TM_NL) s.tr[t] = w[N * NZ + P.term_idx[t]] - xrN[P.term_idx[t]];
  }
  TM_SYNC();
}

// Soft-constraint slacks have no curvature (pmpc.py:327-339: zero Hessian block, linear cost scost > 0), so every QP solution
// has, per stage and slack j, the row usc_j >= 0 or the softened row h_i + usc_j >= 0 active.  The base problem must be
// strictly convex on its null space: where the multipliers hold neither of the two (the dual reference after the stage-0
// relaxation pmpc.py:293-294 with its h_us_idx pointing into the usc rows, the shifted warm start, an emptied working set),
// one of them is added to the base -- usc_j >= 0, or the softened row where usc_j >= 0 is relaxed.  Its multiplier comes
// back with the right sign (-scost), or the usual release / re-solve logic takes over.
TM_HD void tm_pin_soft_slacks(const TmProb& P, unsigned* mask) {
#if NSC > 0
  const int nh = P.nh;
  for (int j = 0; j < NSC; ++j) {
    const int es = nh - NSC + j;
    int er = -1;
    for (int i = 0; i < nh - NSC; ++i) if (P.C[(size_t)i * NZ + NZM + NS + j] != 0.0) { er = i; break; }
    for (int k = 0; k < P.N; ++k) {
      const int rel_s = (k == 0 && P.relax0[es]), rel_r = (er < 0) || (k == 0 && P.relax0[er]);
      const int has_s = !rel_s && tm_mask_get(mask, k * nh + es), has_r = !rel_r && tm_mask_get(mask, k * nh + er);
      if (has_s || has_r) continue;
      if (!rel_s) tm_mask_set(mask, k * nh + es);
      else if (!rel_r) tm_mask_set(mask, k * nh + er);
    }
  }
#else
  (void)P; (void)mask;
#endif
}

// Stage 0 of a softened row that depends on the state only: x_0 is fixed, so the row's value v = h_i(x0) + usc_j(iterate) is known
// before the solve and decides which of the two rows is active there -- the softened row (usc_j = -h_i(x0) > 0) when the state
// violates the bound, else usc_j >= 0.  Holding both (what the shifted multipliers may ask for) is inconsistent.  w: the iterate.
TM_HD void tm_soft_stage0(const TmProb& P, const TmQpWs& s, const double* e0, const double* w, unsigned* mask) {
#if NSC > 0
  const int nh = P.nh;
  for (int j = 0; j < NSC; ++j) {
    const int es = nh - NSC + j;
    int er = -1;
    for (int i = 0; i < nh - NSC; ++i) if (P.C[(size_t)i * NZ + NZM + NS + j] != 0.0) { er = i; break; }
    if (er < 0 || P.relax0[er]) continue;
    int state_only = 1;
    for (int c = NX; c < NZ; ++c) if (c != NZM + NS + j && P.C[(size_t)er * NZ + c] != 0.0) state_only = 0;
    if (!state_only) continue;
    double v = s.hv[er] - P.C[(size_t)er * NZ + NZM + NS + j] * w[NZM + NS + j];   // the row at the new x_0 with its slack at zero
    for (int c = 0; c < NX; ++c) v += P.C[(size_t)er * NZ + c] * e0[c];
    if (v < -1e-12 || P.relax0[es]) { tm_mask_set(mask, er); tm_mask_clr(mask, es); }
    else { tm_mask_clr(mask, er); tm_mask_set(mask, es); }
  }
#else
  (void)P; (void)s; (void)e0; (void)mask;
#endif
}

// One QP with the base rows in amask.  returns 0 ok (step and multipliers in dout / lq, wrong-sign base rows reported
// in nwrong / amask_next), 2 infeasible, 3 base not positive definite, 6 base rows inconsistent, 7 working-set overflow.
// amask_next = base rows with a correctly signed multiplier + the rows the dual active set added: the working set a
// re-solve starts from.
TM_HDN int tm_qp_solve(const TmProb& P, const TmState& S, int64_t inst, TmQpWs& s, const unsigned* amask_in,
                       unsigned* amask_next, int& nwrong, int& n_gi_out, const TmQpPert* pert = nullptr, int eq_only = 0,
                       double rho_scale = 1.0) {
  const int N = P.N, nh = P.nh, nxt = P.nxt;
  const int lane = TM_LANE;
  const int NI = N * nh;
#if NSC > 0
  unsigned amask[TM_ALW];
  for (int wd = 0; wd < TM_ALW; ++wd) amask[wd] = amask_in[wd];
  tm_pin_soft_slacks(P, amask);
  if (!pert) tm_soft_stage0(P, s, s.pv + 2 * NX, S.W + inst * P.n_w, amask);
#else
  const unsigned* amask = amask_in;
#endif
  TmL e0 = s.pv + 2 * NX;
  if (pert) {
    if (pert->homog) {
      for (int e = lane; e < (N + 1) * NZ; e += TM_NL) s.r[e] = 0.0;
      for (int e = lane; e < N * NX; e += TM_NL) s.b[e] = 0.0;
      for (int t = lane; t < nxt; t += TM_NL) s.tr[t] = 0.0;
    }
    for (int a = lane; a < NX; a += TM_NL) e0[a] = 0.0;     // the x_0 offset always enters through the table
    TM_SYNC();
    if (pert->e0_unit >= 0) for (int a = lane; a < NX; a += TM_NL) e0[a] = (a == pert->e0_unit) ? 1.0 : 0.0;
    if (pert->row >= 0) {
      const int k = pert->row / nh, i = pert->row % nh;
      for (int b2 = lane; b2 < NZ; b2 += TM_NL) s.r[k * NZ + b2] -= P.C[(size_t)i * NZ + b2];
    }
    TM_SYNC();
  }
  // weight of the terminal rows' augmented-Lagrangian term: relative to the largest Hessian diagonal entry of the horizon
  double rho = 0.0;
  {
    double qmax = 0.0;
    for (int e = lane; e < N * NZ; e += TM_NL) { const int k = e / NZ, i = e % NZ; qmax = fmax(qmax, fabs(s.Q[(size_t)k * NZ * NZ + i * NZ + i])); }
    rho = rho_scale * P.rho_rel * fmax(tm_wmax(qmax), 1e-300);
  }
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
  long long tp0 = clock64();
#endif
  int ret = tm_qp_factor(P, s, amask, e0, rho);
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
  long long tp1 = clock64();
#endif
  int m = 0, n_gi = 0, n_ricc = 1;
  if (!ret && (NI > 0 || nxt > 0)) {
    if (pert || eq_only) {                        // tabulation / parametric line (tm_qp): equality rows only
      unsigned all[TM_ALW];
      for (int wd = 0; wd < TM_ALW; ++wd) all[wd] = 0xffffffffu;
      ret = tm_qp_gi(P, s, all, m, n_gi, n_ricc);
    } else {
      ret = tm_qp_gi(P, s, amask, m, n_gi, n_ricc);
    }
  }
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
  long long tp2 = clock64();
#endif
  n_gi_out = n_gi;
  if (!ret) {
    // gradient including the dual active-set rows (kept in s.rhs for the multiplier recovery), correction solve
    for (int e = lane; e < (N + 1) * NZ; e += TM_NL) s.rhs[e] = 0.0;
    for (int e = lane; e < NI + nxt; e += TM_NL) s.lh[e] = 0.0;
    TM_SYNC();
    int kfrom = -1;
    if (lane == 0)
      for (int j2 = 0; j2 < m; ++j2) {
        const int e = (int)s.acte[j2];
        s.lh[e] = -s.nu[j2];
        if (e >= NI) { s.rhs[N * NZ + P.term_idx[e - NI]] -= s.nu[j2]; continue; }
        const int k = e / nh, i = e % nh;
        const double* Ci = P.C + (size_t)i * NZ;
        for (int b2 = 0; b2 < NZ; ++b2) s.rhs[k * NZ + b2] -= s.nu[j2] * Ci[b2];
      }
    for (int j2 = 0; j2 < m; ++j2) { const int e = (int)s.acte[j2]; const int k = e < NI ? e / nh : N; if (k > kfrom) kfrom = k; }
    TM_SYNC();
    if (m > 0) {
      tm_ricc_solve(P, s, s.rhs, s.y, kfrom);
      ++n_ricc;
      for (int e = lane; e < (N + 1) * NZ; e += TM_NL) s.d[e] += s.y[e];
    } else {
      for (int e = lane; e < (N + 1) * NX; e += TM_NL) s.py[e] = 0.0;
    }
    TM_SYNC();
    for (int e = lane; e < (N + 1) * NZ; e += TM_NL) s.rhs[e] += s.r[e];
    TM_SYNC();
  }
  if (lane == 0 && !pert) {
#ifdef __CUDA_ARCH__
    atomicAdd(S.counters + 5, 1ull); atomicAdd(S.counters + 6, (unsigned long long)n_gi); atomicAdd(S.counters + 7, (unsigned long long)n_ricc);
#else
    S.counters[5] += 1; S.counters[6] += n_gi; S.counters[7] += n_ricc;
#endif
  }
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
  long long tp3 = clock64();
  if (lane == 0 && !pert) { atomicAdd(S.counters + 20, (unsigned long long)(tp1 - tp0)); atomicAdd(S.counters + 21, (unsigned long long)(tp2 - tp1)); atomicAdd(S.counters + 22, (unsigned long long)(tp3 - tp2)); }
#endif
  if (ret) return ret;
  if (eq_only) { nwrong = 0; return 0; }            // the step of the equality-constrained problem is in s.d
  double* dout = pert ? pert->dout : S.D + inst * P.n_w;
  double* lq = pert ? pert->lout : S.LAMQ + inst * P.n_g;
  for (int e = lane; e < P.n_g; e += TM_NL) lq[e] = 0.0;
  TM_SYNC();
  tm_qp_recover(P, s, amask, lq);
  for (int e = lane; e < NI; e += TM_NL) if (s.lh[e] != 0.0) lq[tm_gh(P, e / nh) + e % nh] = s.lh[e];
#ifndef TM_TERM_ELIM
  for (int t = lane; t < nxt; t += TM_NL) lq[tm_gterm(P) + t] = s.lh[NI + t];
#endif
  TM_SYNC();
  // base rows must carry the multiplier sign of an active lower bound (CasADi convention: lam < 0)
  int nw = 0;
  for (int wd = 0; wd < TM_ALW; ++wd) amask_next[wd] = amask[wd];
  if (!pert) {
    double lmax = 0.0;
    for (int e = 0; e < NI; ++e) if (tm_mask_get(amask, e)) lmax = fmax(lmax, fabs(lq[tm_gh(P, e / nh) + e % nh]));
#ifdef TM_RELEASE_ONE
    {
      double worst = 1e-12 * lmax; int we = -1;
      for (int e = 0; e < NI; ++e) {
        if (!tm_mask_get(amask, e)) continue;
        const double l = lq[tm_gh(P, e / nh) + e % nh];
        if (l > worst) { worst = l; we = e; }
      }
      if (we >= 0) { tm_mask_clr(amask_next, we); ++nw; }
    }
#else
    for (int e = 0; e < NI; ++e) {
      if (!tm_mask_get(amask, e)) continue;
      if (lq[tm_gh(P, e / nh) + e % nh] > 1e-12 * lmax) { tm_mask_clr(amask_next, e); ++nw; }
    }
#endif
    for (int j2 = 0; j2 < m; ++j2) if ((int)s.acte[j2] < NI) tm_mask_set(amask_next, (int)s.acte[j2]);
  }
#if defined(TM_PROF_W) && defined(__CUDA_ARCH__)
  if (lane == 0 && !pert) atomicAdd(S.counters + 23, (unsigned long long)(clock64() - tp3));
#endif
  nwrong = nw;
  if (nw == 0) {
    for (int e = lane; e < P.n_w; e += TM_NL) dout[e] = s.d[e];
    TM_SYNC();
  }
  return 0;
}
