// CPU twin of the solution VJP (tm_solution_vjp) -- TEST INFRASTRUCTURE ONLY (never loaded by the product package).
// Compiles tunempc_b200/csrc/tmpc_core.cuh with g++ as a 1-lane sequential program (TM_NL = 1), like twin_fbjac.cpp, into a
// library of its own (libtwin_vjp_<model>.so, built by tests/solution_vjp_support.py).
#include <string.h>
#include <vector>
#include "tmpc_core.cuh"

extern "C" {

// G = v_u0' du0/dx0 + v_w' dw/dx0 (tm_solution_vjp) at B solutions (W, LAM) with their step status: the stage records are
// linearised again at (W, LAM) here (tm_lin_task), as tmpc_solution_vjp does on the device.  Problem arguments as
// twin_feedback_jacobian; Vu0: B*nu or NULL, Vw: B*n_w or NULL; G: B*nx, jst: B.
int twin_solution_vjp(const int* dims, const int* iopts, const double* dopts, const double* wref, const double* H,
                      const double* q, const double* ref_du, const double* C, const double* c, const int* term_idx,
                      const int* relax0, int phase, long long B, const double* W, const double* LAM, const int* status,
                      const double* Vu0, const double* Vw, double* G, int* jst) {
  TmProb P;
  P.N = dims[0]; P.nh = dims[1]; P.nxt = dims[2]; P.p = dims[3];
  P.n_w = P.N * NZ + NX;
  P.n_g = NX + P.N * (NX + NS + P.nh) + P.nxt;
  P.hessian_exact = iopts[0];
  P.filter_cap = 64;
  P.max_iter = iopts[1];
  P.max_ls = iopts[2];
  P.maxact = (iopts[3] < P.N * P.nh ? iopts[3] : P.N * P.nh) + P.nxt; if (P.maxact < 1) P.maxact = 1;
  P.economic = iopts[4];
  P.reg_mode = iopts[5];
  P.nonconvex_after = iopts[6];
  P.lin_adjoint = 0;
  if (P.economic) P.hessian_exact = 1;
  if (!P.hessian_exact) return 1;
  P.tol = dopts[0]; P.lam_tresh = dopts[1]; P.beta = dopts[2]; P.reg_tol = dopts[3]; P.rho_rel = dopts[4];
  P.wref = wref; P.H = H; P.q = q; P.ref_du = ref_du; P.C = C; P.c = c; P.term_idx = term_idx; P.relax0 = relax0;
  std::vector<int> rowpin((size_t)(P.nh > 0 ? P.nh : 1), -1);
  for (int i = 0; i < P.nh; ++i) {
    int cnt = 0, jc = -1;
    for (int cidx = 0; cidx < NZ; ++cidx) if (C[(size_t)i * NZ + cidx] != 0.0) { ++cnt; jc = cidx; }
    if (cnt == 1 && jc >= NX) rowpin[i] = jc - NX;
  }
  P.rowpin = rowpin.data();
  P.prof_counters = nullptr;
  std::vector<double> Wc(W, W + (size_t)B * P.n_w), Lc(LAM, LAM + (size_t)B * P.n_g);
  std::vector<double> LIN((size_t)B * P.N * TM_LSZ), dscr((size_t)B * P.n_w), lscr((size_t)B * P.n_g);
  std::vector<int> st(status, status + B);
  TmState S;
  memset(&S, 0, sizeof S);
  // X0 only has to be readable: the solve replaces the x_0 offset that tm_qp_setup forms from it
  S.B = B; S.phase = phase; S.X0 = Wc.data(); S.W = Wc.data(); S.LAM = Lc.data(); S.LIN = LIN.data();
  S.status = st.data();
  const int per = tm_lin_tasks_per_stage(1);
  for (long long i = 0; i < B; ++i)
    if (st[i] == 0) for (int k = 0; k < P.N; ++k) for (int pr = 0; pr < per; ++pr) tm_lin_task(P, S, i, k, pr, 0);
  std::vector<double> wsbuf(tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact));
  TmQpWs ws;
  tm_qpws_carve(wsbuf.data(), P.N, P.nh, P.nxt, P.maxact, ws);
  for (long long i = 0; i < B; ++i) tm_solution_vjp(P, S, i, ws, Vu0, Vw, dscr.data(), lscr.data(), G, jst);
  return 0;
}

}  // extern "C"
