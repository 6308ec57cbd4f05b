// tmpc.cu -- kernels, SQP host loop and the C ABI (include/tmpc.h) of libtmpc_<model>.so.   sm_100a, fp64.
//
// Build (see __graft_entry__.build):
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC \
//        -DTMPC_MODEL_HEADER='"gen/model_cstr.h"' -Iinclude -Itunempc_b200/csrc tmpc.cu -o libtmpc_cstr.so
//
// Kernel inventory (SURVEY.md section 2.4 K1-K7):
//   k_lin      K1  one thread per (instance, stage, sensitivity pair): RK4 + 1st/2nd-order sensitivities, exact
//                  Lagrangian-Hessian block lam' d2F contracted in registers; FP64-FMA bound
//   k_qp       K3+K4  one warp per instance: Riccati base factorisation in shared memory + dual active set
//   k_post     K5+K2  one warp per instance: filter line search, primal/dual update, KKT residual, convergence
//   k_conv     K2  convergence for instances that were re-linearised after a damped step
//   k_prefilter, k_init, k_shift, k_gather, k_plant   K6 bookkeeping
// There is no CPU solve path in this library: if the device is unusable every entry point returns an error.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "tmpc.h"
#include "tmpc_core.cuh"
// model-dimension region (see tmpc_core.cuh): NZ, NU = NZM, NUM for the linearisation kernels
#pragma push_macro("NZ")
#pragma push_macro("NU")
#undef NZ
#undef NU
#define NZ TMPC_NZM
#define NU TMPC_NUM
#include "tmpc_lin2.cuh"

// thread-per-instance QP kernel (tmpc_qp_thread.cu), feedback Jacobian (tmpc_fbjac_thread.cu) and solution VJP (tmpc_vjp_thread.cu)
cudaError_t tm_launch_qp_thread(const TmProb& P, const TmState& S, const int* list, int cnt, const int* cnt_dev,
                                double* wsbase, size_t ws_per_inst, int nblocks, int* work_counter, cudaStream_t st);
cudaError_t tm_launch_fbjac_thread(const TmProb& P, const TmState& S, int cnt, double* wsbase, size_t ws_per_inst, int nblocks,
                                   int* work_counter, double* J, int* jst, cudaStream_t st);
cudaError_t tm_launch_vjp_thread(const TmProb& P, const TmState& S, int cnt, double* wsbase, size_t ws_per_inst, int nblocks,
                                 int* work_counter, const double* Vu0, const double* Vw, double* dscr, double* lscr, double* G,
                                 int* jst, cudaStream_t st);
int tm_qp_thread_block();

#define QP_WARPS 2          /* warps (instances) per CTA in the warp-per-instance kernels */
#define LIN_THREADS 128

struct tmpc_handle {
  int device = 0;
  tmpc_dims dims{};
  tmpc_opts opts{};
  TmProb P{};
  TmState S{};
  int64_t cap = 0;           // allocated instance capacity
  int64_t index = 0;         // Pmpc.__index
  bool tables_set = false;
  std::string err;
  std::vector<void*> tab_allocs, ws_allocs;
  int *list_a = nullptr, *list_b = nullptr, *cnts = nullptr;   // cnts[0] next, cnts[1] relin, cnts[2..3] retry ping-pong
  int *retry_a = nullptr, *retry_b = nullptr;
  int *list_s = nullptr, *sort_bins = nullptr;                 // sorted copy of the active list, 2*SORT_BINS counters
  bool sort_lists = true;
  double *Wsh = nullptr, *Lsh = nullptr;                       // shift targets
  double* X0buf = nullptr;                                     // device staging for tmpc_step_host
  int64_t counters_host[8] = {0};
  double timing_ms[4] = {0};
  cudaEvent_t ev[8];
  bool ev_ok = false;
  size_t qp_smem = 0;
  int qp_warps = QP_WARPS;     // instances per CTA of the warp-per-instance QP kernels: 2, 1, or 0 (workspace exceeds shared memory)
  int qp_mode = 2;             // 2: hybrid (thread per instance for big launches, warp per instance for the tail), 1: thread, 0: warp
  int qp_thread_min = 16384;   // hybrid: launches with fewer candidate instances use the low-latency warp kernel
  bool trace = false;
  bool pd_check = true;        // run the reference's post-solve reduced-Hessian test (status 3); TMPC_PD_CHECK=0 skips it
  int lin_mode = 3;             // 3: forward / adjoint sweep k_lin3 (RK4 models, default), 2: warp-specialised pair-wise k_lin2, 1: thread per (instance, stage, pair) k_lin
  bool uniform_ws = false;     // warm start identical for every instance (right after tmpc_reset)
  int qp_blocks = 0;           // resident CTAs of the thread-per-instance kernel
  double* qp_ws = nullptr;     // its workspace
  double* qp_cold = nullptr;   // warp-per-instance kernels: dual-Hessian columns + Schur factor of every resident warp
  int qp_wgrid = 0;            // resident CTAs of the warp-per-instance kernels
  size_t qp_ws_per_inst = 0;
  int* qp_counter = nullptr;
  TmQp0Tab q0{};               // tables of the shared first QP after reset (tm_qp0_*)
  bool q0_ok = false;          // allocated and applicable (nh > 0, smem fits)
  int64_t q0_min = 1024;       // smallest batch for which tabulating (1 + nx + N*nh warp-level QP solves) pays off
  std::vector<char> phase_clean;   // per phase: no reference multiplier on an inequality row (empty convexification mask)
  // ---- asynchronous step (tmpc_step_async / tmpc_wait): a host worker thread drives the SQP loop on an internal stream
  struct AsyncJob { const double* X0; int64_t B; double *U0, *W, *LAM, *G; int32_t *status, *iter, *flags; } job{};
  std::thread worker;
  std::mutex mu;
  std::condition_variable cv;
  bool has_job = false, busy = false, quit = false, async_ready = false;
  int job_rc = 0;
  void* host_pinned = nullptr;      // 4 + TM_NCNT words: per-iteration counts and the counters of the step
  cudaStream_t istream = nullptr;
  cudaEvent_t ev_in = nullptr;
  // ---- feedback Jacobian (tmpc_feedback_jacobian)
  bool solved = false;              // a step has finished since tmpc_create / tmpc_reset: its solutions are in Wsh / Lsh, LIN
  bool fbjac_smem = false;          // k_fbjac's dynamic shared-memory limit raised
  double* jac_buf = nullptr;        // device staging of J and jstatus for host destinations
  int* jst_buf = nullptr;
  int64_t jac_cap = 0;
  // ---- solution VJP (tmpc_solution_vjp): a stored solution, its linearisation records and the solve's scratch, grown with B
  bool vjp_smem = false;            // k_vjp's dynamic shared-memory limit raised
  int64_t vjp_cap = 0;
  double *vjp_W = nullptr, *vjp_L = nullptr, *vjp_LIN = nullptr, *vjp_D = nullptr, *vjp_LQ = nullptr;
  int* vjp_st = nullptr;
  int64_t vjp_io_cap = 0;           // device staging of the cotangents and results for host buffers
  double *vjp_Vu = nullptr, *vjp_Vw = nullptr, *vjp_G = nullptr;
  int* vjp_js = nullptr;
};

static int fail(tmpc_handle* h, const char* what, cudaError_t e) {
  if (h) h->err = std::string(what) + ": " + cudaGetErrorString(e);
  return 1;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(h, #call, e_); } while (0)

// ------------------------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LIN_THREADS) k_lin(TmProb P, TmState S, const int* list, const int* cnt_dev, int cnt,
                                                     int trial, int per) {
  if (cnt_dev) cnt = *cnt_dev;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)cnt * P.N * per;
  if (t >= total) return;
  const int pr = (int)(t % per);
  const int k = (int)((t / per) % P.N);
  const int64_t slot = t / ((int64_t)per * P.N);
  const int64_t inst = list ? list[slot] : slot;
  tm_lin_task(P, S, inst, k, pr, trial);
}

#if TMPC_RK4
// K1 by the forward / adjoint sweep (tmpc_lin3.cuh): one thread per (instance, stage) task, state in registers, the M stored
// states of the forward pass in local memory
#ifndef LIN3_THREADS
#define LIN3_THREADS 128
#endif
#ifndef LIN3_MINB
#define LIN3_MINB 1
#endif
template <bool EXACT>
__global__ void __launch_bounds__(LIN3_THREADS, LIN3_MINB) k_lin3(TmProb P, TmState S, const int* list, int cnt, int trial) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)cnt * P.N) return;
  const int k = (int)(t % P.N);
  const int64_t slot = t / P.N;
  const int64_t inst = list ? list[slot] : slot;
  if (trial && S.qpstat[inst] != 0) return;          // failed QP: keep LIN at W for the final statistics
  const double* w = S.W + inst * P.n_w + (int64_t)k * TM_NZS;
  double x[NX], u[NU], lam[NX];
#pragma unroll
  for (int a = 0; a < NX; ++a) x[a] = w[a];
#pragma unroll
  for (int b = 0; b < NU; ++b) u[b] = w[NX + b];
  if (trial) {
    const double* d = S.D + inst * P.n_w + (int64_t)k * TM_NZS;
#pragma unroll
    for (int a = 0; a < NX; ++a) x[a] += d[a];
#pragma unroll
    for (int b = 0; b < NU; ++b) u[b] += d[NX + b];
  }
  const double* lamp = (trial ? S.LAMQ : S.LAM) + inst * P.n_g + tm_gdyn(P, k);
#pragma unroll
  for (int a = 0; a < NX; ++a) lam[a] = EXACT ? lamp[a] : 0.0;
  tm_lin_adjoint(x, u, EXACT ? 2 : 1, lam, S.LIN + (inst * P.N + k) * (int64_t)TM_LSZ);
}
#endif

#pragma pop_macro("NU")
#pragma pop_macro("NZ")

__global__ void k_prefilter(TmProb P, TmState S) {
  const int64_t inst = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  if (inst >= S.B) return;
  tm_prefilter(P, S, inst);
}

__global__ void k_init(TmProb P, TmState S) {
  const int64_t inst = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  if (inst >= S.B) return;
  tm_init(P, S, inst);
}

// warp per instance, resident CTAs striding over the list: the hot part of the workspace in shared memory, the dual-Hessian
// columns and the Schur factor in this warp's slot of a small global buffer (cold)
__global__ void __launch_bounds__(QP_WARPS * 32) k_qp(TmProb P, TmState S, const int* list, int cnt, const int* cnt_dev, double* cold) {
  extern __shared__ double smem[];
  if (cnt_dev) cnt = *cnt_dev;
  const int wid = threadIdx.x / 32, W = blockDim.x / 32;
  const size_t cper = tm_qpws_cold_doubles(P.N, P.nh, P.nxt, P.maxact);
  const size_t per = tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact) - cper;
  TmQpWs ws;
  tm_qpws_carve(smem + (size_t)wid * per, P.N, P.nh, P.nxt, P.maxact, ws, cold + ((size_t)blockIdx.x * W + wid) * cper);
  for (int64_t slot = (int64_t)blockIdx.x * W + wid; slot < cnt; slot += (int64_t)gridDim.x * W) {   // 1 or QP_WARPS instances per CTA
    const int64_t inst = list ? list[slot] : slot;
    tm_qp(P, S, inst, ws);
    __syncwarp();
  }
}

// feedback Jacobian du0/dx0 at the solutions of the last step (tm_feedback_jacobian): warp per instance on the k_qp workspace
__global__ void __launch_bounds__(QP_WARPS * 32) k_fbjac(TmProb P, TmState S, int cnt, double* cold, double* J, int* jst) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x / 32, W = blockDim.x / 32;
  const size_t cper = tm_qpws_cold_doubles(P.N, P.nh, P.nxt, P.maxact);
  const size_t per = tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact) - cper;
  TmQpWs ws;
  tm_qpws_carve(smem + (size_t)wid * per, P.N, P.nh, P.nxt, P.maxact, ws, cold + ((size_t)blockIdx.x * W + wid) * cper);
  for (int64_t inst = (int64_t)blockIdx.x * W + wid; inst < cnt; inst += (int64_t)gridDim.x * W) {
    tm_feedback_jacobian(P, S, inst, ws, J, jst);
    __syncwarp();
  }
}

// solution VJP (tm_solution_vjp): warp per instance on the k_qp workspace
__global__ void __launch_bounds__(QP_WARPS * 32) k_vjp(TmProb P, TmState S, int cnt, double* cold, const double* Vu0,
                                                     const double* Vw, double* dscr, double* lscr, double* G, int* jst) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x / 32, W = blockDim.x / 32;
  const size_t cper = tm_qpws_cold_doubles(P.N, P.nh, P.nxt, P.maxact);
  const size_t per = tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact) - cper;
  TmQpWs ws;
  tm_qpws_carve(smem + (size_t)wid * per, P.N, P.nh, P.nxt, P.maxact, ws, cold + ((size_t)blockIdx.x * W + wid) * cper);
  for (int64_t inst = (int64_t)blockIdx.x * W + wid; inst < cnt; inst += (int64_t)gridDim.x * W) {
    tm_solution_vjp(P, S, inst, ws, Vu0, Vw, dscr, lscr, G, jst);
    __syncwarp();
  }
}

// ---- first QP after reset(): tabulate the shared parametric QP, then one thread per instance on the tables ----------
__global__ void __launch_bounds__(QP_WARPS * 32) k_qp0_build(TmProb P, TmState S, TmQp0Tab T, double* cold) {
  extern __shared__ double smem[];
  const int wid = threadIdx.x / 32, W = blockDim.x / 32;
  const size_t cper = tm_qpws_cold_doubles(P.N, P.nh, P.nxt, P.maxact);
  const size_t per = tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact) - cper;
  TmQpWs ws;
  tm_qpws_carve(smem + (size_t)wid * per, P.N, P.nh, P.nxt, P.maxact, ws, cold + ((size_t)blockIdx.x * W + wid) * cper);
  for (int t = blockIdx.x * W + wid; t < T.nT; t += gridDim.x * W) {
    tm_qp0_build_row(P, S, 0, ws, T, t);
    __syncwarp();
  }
}

__global__ void k_qp0_derive(TmProb P, TmState S, TmQp0Tab T) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= T.nT * T.EI) return;
  tm_qp0_derive(P, S, 0, T, idx / T.EI, idx % T.EI);
}

#define Q0_THREADS 128
#define Q0_CH 8            /* outputs per lane per chunk of the table combination */
__global__ void __launch_bounds__(Q0_THREADS) k_qp0(TmProb P, TmState S, TmQp0Tab T, int cnt) {
  const int64_t inst = (int64_t)blockIdx.x * Q0_THREADS + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool valid = inst < cnt;
  if (*T.bad) {                                   // tabulation failed: everybody takes the generic path
    if (valid) tm_qp0_finish(P, S, inst, 2, 0);
    return;
  }
  double e0[NX], nu[TM_Q0_MAXM];
  int acte[TM_Q0_MAXM];
  int m = 0, ngi = 0, ret = 2;
  if (valid) {
#pragma unroll
    for (int a = 0; a < NX; ++a) e0[a] = S.X0[inst * NX + a] - S.W[inst * P.n_w + a];
    ret = tm_qp0_gi(P, T, e0, acte, nu, m, ngi);
    tm_qp0_finish(P, S, inst, ret, ngi);
  } else {
#pragma unroll
    for (int a = 0; a < NX; ++a) e0[a] = 0.0;
  }
  // (d, lam) of the warp's 32 instances, one after the other, lanes across the n_w + n_g outputs (coalesced)
  const int n_out = T.n_out;
  for (int src = 0; src < 32; ++src) {
    const int r = __shfl_sync(0xffffffffu, ret, src);
    if (r != 0) continue;
    const int mm = __shfl_sync(0xffffffffu, m, src);
    const long long is = __shfl_sync(0xffffffffu, (long long)inst, src);
    double es[NX];
#pragma unroll
    for (int a = 0; a < NX; ++a) es[a] = __shfl_sync(0xffffffffu, e0[a], src);
    double* dout = S.D + is * P.n_w;
    double* lout = S.LAMQ + is * P.n_g;
    for (int base = 0; base < n_out; base += 32 * Q0_CH) {
      double acc[Q0_CH];
#pragma unroll
      for (int q = 0; q < Q0_CH; ++q) {
        const int i = base + q * 32 + lane;
        double v = 0.0;
        if (i < n_out) {
          v = T.TAB[i];
#pragma unroll
          for (int a = 0; a < NX; ++a) v += es[a] * T.TAB[(size_t)(1 + a) * n_out + i];
        }
        acc[q] = v;
      }
      for (int j = 0; j < mm; ++j) {
        const int aj = __shfl_sync(0xffffffffu, acte[j], src);
        const double nj = __shfl_sync(0xffffffffu, nu[j], src);
        const double* row = T.TAB + (size_t)(1 + NX + aj) * n_out;
#pragma unroll
        for (int q = 0; q < Q0_CH; ++q) {
          const int i = base + q * 32 + lane;
          if (i < n_out) acc[q] += nj * row[i];
        }
      }
#pragma unroll
      for (int q = 0; q < Q0_CH; ++q) {
        const int i = base + q * 32 + lane;
        if (i < n_out) { if (i < P.n_w) dout[i] = acc[q]; else lout[i - P.n_w] = acc[q]; }
      }
    }
  }
}

__global__ void __launch_bounds__(QP_WARPS * 32) k_post(TmProb P, TmState S, const int* list, int cnt) {
  const int64_t slot = (int64_t)blockIdx.x * QP_WARPS + threadIdx.x / 32;
  if (slot >= cnt) return;
  const int64_t inst = list ? list[slot] : slot;
  tm_post(P, S, inst);
}

__global__ void __launch_bounds__(QP_WARPS * 32) k_conv(TmProb P, TmState S, const int* list, const int* cnt_dev) {
  const int64_t slot = (int64_t)blockIdx.x * QP_WARPS + threadIdx.x / 32;
  if (slot >= *cnt_dev) return;
  tm_conv(P, S, list[slot]);
}

__global__ void k_shift(TmProb P, TmState S, double* Ws, double* Ls) {
  const int64_t inst = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  if (inst >= S.B) return;
  tm_shift(P, S.W + inst * P.n_w, S.LAM + inst * P.n_g, Ws + inst * P.n_w, Ls + inst * P.n_g);
}

__global__ void k_gather_u0(TmProb P, TmState S, double* U0) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= S.B * NUM) return;
  U0[t] = S.W[(t / NUM) * P.n_w + NX + (t % NUM)];
}

__global__ void k_bcast(double* dst, const double* row, int64_t B, int n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * n) return;
  dst[t] = row[t % n];
}

__global__ void k_plant(const double* X, const double* U, int64_t B, double* Xn) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double x[NX], u[NUM], xf[NX], t1[NX], t2[NX], t3[NX];
#pragma unroll
  for (int a = 0; a < NX; ++a) x[a] = X[b * NX + a];
#pragma unroll
  for (int a = 0; a < NUM; ++a) u[a] = U[b * NUM + a];
  tm_integrate<0>(x, u, 0, 0, xf, t1, t2, t3);
#pragma unroll
  for (int a = 0; a < NX; ++a) Xn[b * NX + a] = xf[a];
}

// plant Jacobian JF[b] = [dF/dx | dF/du] (nx x (nx+nu), row-major) at (X[b], U[b]): first-order sensitivities of the same
// integrator as k_plant, one direction per tm_integrate<1> call (RK4, discrete) or one tm_colloc_stage for all directions
__global__ void k_plant_jac(const double* X, const double* U, int64_t B, double* JF) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double x[NX], u[NUM];
#pragma unroll
  for (int a = 0; a < NX; ++a) x[a] = X[b * NX + a];
#pragma unroll
  for (int a = 0; a < NUM; ++a) u[a] = U[b * NUM + a];
  double* J = JF + b * (int64_t)(NX * NZM);
#if TMPC_COLLOCATION
  double rec[NX + NX * NZM];
  tm_colloc_stage(x, u, 1, nullptr, rec);
  for (int e = 0; e < NX * NZM; ++e) J[e] = rec[NX + e];
#else
  for (int i = 0; i < NZM; ++i) {
    double xf[NX], si[NX], sj[NX], t[NX];
    tm_integrate<1>(x, u, i, i, xf, si, sj, t);
#pragma unroll
    for (int a = 0; a < NX; ++a) J[a * NZM + i] = si[a];
  }
#endif
}

// closed-loop log of one (x,u) sample per instance: economic stage cost l(x,u) and the path constraint values h = C z + c
// (tunempc/closed_loop_tools.py:64-65, 98-99)
__global__ void k_stage_log(const double* X, const double* U, int64_t B, const double* C, const double* c, int nh,
                            double* l_out, double* h_out) {
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double z[NZ];
#pragma unroll
  for (int a = 0; a < NZ; ++a) z[a] = 0.0;
#pragma unroll
  for (int a = 0; a < NX; ++a) z[a] = X[b * NX + a];
#pragma unroll
  for (int a = 0; a < NUM; ++a) z[NX + a] = U[b * NUM + a];
#if NS > 0
  tmpc_gnl(z, z + NX, z + NZM);                     // us = h_nl(x,u): the logged rows us >= 0 are the nonlinear constraints themselves
#endif
  if (l_out) l_out[b] = tmpc_stage_cost(z, z + NX);
  if (h_out) {
    for (int i = 0; i < nh; ++i) {
      double v = c[i];
#pragma unroll
      for (int j = 0; j < NZ; ++j) v += C[(size_t)i * NZ + j] * z[j];
      h_out[b * nh + i] = v;
    }
  }
}

// ---- scheduling: counting sort of the active list by the cost of each instance's previous QP (heaviest first) -------
// Results do not depend on the order (instances are independent); the order only decides which instances share a warp
// of the thread-per-instance QP kernel, i.e. how long lanes idle while the longest active-set loop of the warp finishes.
#define SORT_BINS 64
__global__ void k_sort_hist(const int* list, int cnt, const int* key, int* bins) {
  __shared__ int sb[SORT_BINS];
  if (threadIdx.x < SORT_BINS) sb[threadIdx.x] = 0;
  __syncthreads();
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot < cnt) {
    const int inst = list ? list[slot] : slot;
    int k = key[inst];
    k = k < 0 ? 0 : (k >= SORT_BINS ? SORT_BINS - 1 : k);
    atomicAdd(&sb[k], 1);
  }
  __syncthreads();
  if (threadIdx.x < SORT_BINS && sb[threadIdx.x]) atomicAdd(&bins[threadIdx.x], sb[threadIdx.x]);
}
__global__ void k_sort_scan(int* bins) {   // bins[SORT_BINS + b] = first output slot of bin b, descending key order
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int b = SORT_BINS - 1; b >= 0; --b) { bins[SORT_BINS + b] = acc; acc += bins[b]; }
  }
}
__global__ void k_sort_scatter(const int* list, int cnt, const int* key, int* bins, int* out) {
  const int slot = blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= cnt) return;
  const int inst = list ? list[slot] : slot;
  int k = key[inst];
  k = k < 0 ? 0 : (k >= SORT_BINS ? SORT_BINS - 1 : k);
  out[atomicAdd(&bins[SORT_BINS + k], 1)] = inst;
}

// linearise `cnt` instances of S (list == nullptr: identity) at the iterate (trial = 0) or at the trial point (trial = 1)
static cudaError_t launch_lin(tmpc_handle* h, const TmState& S, const int* list, int64_t cnt, int trial, cudaStream_t st) {
  const TmProb& P = h->P;
#if TMPC_RK4
  if (h->lin_mode == 3) {
    const unsigned grid = (unsigned)((cnt * P.N + LIN3_THREADS - 1) / LIN3_THREADS);
    if (P.hessian_exact) k_lin3<true><<<grid, LIN3_THREADS, 0, st>>>(P, S, list, (int)cnt, trial);
    else k_lin3<false><<<grid, LIN3_THREADS, 0, st>>>(P, S, list, (int)cnt, trial);
    return cudaGetLastError();
  }
  if (h->lin_mode == 2) {
    const unsigned grid = (unsigned)((cnt * P.N + 31) / 32);
    if (P.hessian_exact) k_lin2<true><<<grid, L2_THREADS, tm_lin2_smem_bytes(), st>>>(P, S, list, nullptr, (int)cnt, trial);
    else k_lin2<false><<<grid, L2_THREADS, tm_lin2_smem_bytes(), st>>>(P, S, list, nullptr, (int)cnt, trial);
    return cudaGetLastError();
  }
#endif
  const int per = tm_lin_tasks_per_stage(P.hessian_exact);
  k_lin<<<(unsigned)((cnt * P.N * per + LIN_THREADS - 1) / LIN_THREADS), LIN_THREADS, 0, st>>>(P, S, list, nullptr, (int)cnt, trial, per);
  return cudaGetLastError();
}

// dependent-chain-free DFMA loop: 8 independent accumulators per thread
__global__ void k_fp64_peak(double* out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------------
extern "C" {

void tmpc_default_opts(tmpc_opts* o) {
  o->hessian_exact = 1;
  o->max_iter = 2000;
  o->max_ls_iter = 300;
  o->tol = 1e-6;
  o->lam_tresh = 1e-8;
  o->ls_step_factor = 0.8;
  o->reg_tol = 1e-8;
  o->max_working_set = 32;
  o->term_weight = 1e4;
  o->economic = 0;
}

const char* tmpc_model_info(int32_t* nx, int32_t* nu, int32_t* rk_steps, double* dt) {
  if (nx) *nx = NX;
  if (nu) *nu = NUM;
  if (rk_steps) *rk_steps = TMPC_DISCRETE ? 0 : TMPC_RK_STEPS;
  if (dt) *dt = TMPC_RK_DT;
  return TMPC_MODEL_NAME;
}

void tmpc_model_slacks(int32_t* ns, int32_t* nsc) {
  if (ns) *ns = NS;
  if (nsc) *nsc = NSC;
}

const char* tmpc_last_error(const tmpc_handle* h) { return h ? h->err.c_str() : "null handle"; }

int tmpc_create(tmpc_handle** out, const tmpc_dims* dims, const tmpc_opts* opts, int device) {
  if (!out || !dims) return 1;
  *out = nullptr;
  tmpc_handle* h = new tmpc_handle();
  h->device = device;
  h->dims = *dims;
  if (opts) h->opts = *opts; else tmpc_default_opts(&h->opts);
  if (dims->nx != NX || dims->nu != NUM || dims->ns != NS || dims->nsc != NSC) {
    fprintf(stderr, "tmpc_create: dims (nx %d, nu %d, ns %d, nsc %d) do not match compiled model %s (%d, %d, %d, %d)\n", dims->nx,
            dims->nu, dims->ns, dims->nsc, TMPC_MODEL_NAME, NX, NUM, NS, NSC);
    delete h;
    return 2;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || device >= ndev) {
    fprintf(stderr, "tmpc_create: no usable CUDA device %d (%s) -- this library has no CPU path\n", device,
            e != cudaSuccess ? cudaGetErrorString(e) : "index out of range");
    delete h;
    return 3;
  }
  cudaSetDevice(device);
  TmProb& P = h->P;
  P.N = dims->N; P.nh = dims->nh; P.nxt = dims->nx_term; P.p = dims->p;
  P.n_w = dims->N * NZ + NX;
  P.n_g = NX + dims->N * (NX + NS + dims->nh) + dims->nx_term;
  P.economic = h->opts.economic ? 1 : 0;
  P.hessian_exact = (h->opts.hessian_exact || P.economic) ? 1 : 0;   // economic MPC: exact Hessian forced (pmpc.py:97-107)
  P.filter_cap = 64;                      // rows of the pruned filter (tm_post): bounds memory, not the iteration count
  P.max_iter = h->opts.max_iter;           // pmpc.py:155 (2000), honoured as given
  P.max_ls = h->opts.max_ls_iter;
  // capacity of the dual active set's working set (rows ADDED to the base rows of one QP; the base rows -- terminal rows and
  // the rows active in the multipliers -- live in the factorisation and do not count): every inequality row if that is small
  P.maxact = h->opts.max_working_set > 0 ? h->opts.max_working_set : 32;
  if (P.maxact > P.N * P.nh) P.maxact = P.N * P.nh;
  P.maxact += P.nxt;                       // the terminal rows are permanent members of the Schur complement
  if (P.maxact < 1) P.maxact = 1;
  if (P.N * P.nh > 32 * TM_ALW) {
    h->err = "tmpc_create: N*nh exceeds the row-mask capacity";
    fprintf(stderr, "tmpc_create: N*nh = %d exceeds the %d-row capacity of the working-set masks (TM_ALW)\n", P.N * P.nh, 32 * TM_ALW);
    delete h;
    return 6;
  }
  P.tol = h->opts.tol; P.lam_tresh = h->opts.lam_tresh; P.beta = h->opts.ls_step_factor;
  P.reg_tol = h->opts.reg_tol; P.rho_rel = h->opts.term_weight;
  P.reg_mode = 8; P.nonconvex_after = TM_NONCONVEX_AFTER;
  { const char* na = getenv("TMPC_NONCONVEX_AFTER"); if (na) P.nonconvex_after = atoi(na); }
  { const char* rm = getenv("TMPC_REG_MODE"); if (rm) P.reg_mode = atoi(rm); }
  {
    // warp-per-instance QP kernels keep the workspace of their instances in shared memory: 2 per CTA if that fits, else
    // 1, else those kernels are not used at all (thread-per-instance kernel for every launch, no shared first QP)
    const size_t cold = tm_qpws_cold_doubles(P.N, P.nh, P.nxt, P.maxact);
    const size_t per = (tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact) - cold) * sizeof(double);
    h->qp_warps = (QP_WARPS * per <= 227 * 1024) ? QP_WARPS : (per <= 227 * 1024 ? 1 : 0);
    h->qp_smem = (size_t)h->qp_warps * per;
    if (h->qp_warps > 0 &&
        cudaFuncSetAttribute(k_qp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->qp_smem) != cudaSuccess) {
      cudaGetLastError();
      h->qp_warps = 0;
    }
    if (h->qp_warps > 0) {
      // resident CTAs of the warp kernels (they stride over their list): every resident warp owns one slot of the cold buffer
      int nb = 0, nsm = 148;
      cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device);
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_qp, h->qp_warps * 32, h->qp_smem) != cudaSuccess || nb < 1) { nb = 1; cudaGetLastError(); }
      h->qp_wgrid = nsm * nb;
      if (cudaMalloc(&h->qp_cold, (size_t)h->qp_wgrid * h->qp_warps * cold * sizeof(double)) != cudaSuccess) { cudaGetLastError(); h->qp_warps = 0; }
    }
    if (h->qp_warps == 0) h->qp_mode = 1;
  }
  {
    const char* m = getenv("TMPC_QP_MODE");
    if (m && m[0] == 'w' && h->qp_warps > 0) h->qp_mode = 0;
    if (m && m[0] == 't') h->qp_mode = 1;
    h->trace = getenv("TMPC_TRACE") != nullptr;
    { const char* pc = getenv("TMPC_PD_CHECK"); if (pc) h->pd_check = atoi(pc) != 0; }
    const char* lm = getenv("TMPC_LIN_MODE");
    if (lm) h->lin_mode = atoi(lm);
#if !TMPC_RK4
    h->lin_mode = 1;
#else
    if (tm_lin2_smem_bytes() > 48 * 1024) {
      cudaFuncSetAttribute(k_lin2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tm_lin2_smem_bytes());
      cudaFuncSetAttribute(k_lin2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tm_lin2_smem_bytes());
    }
    {
      // the warp-specialised kernel needs one warp per role: for larger models a CTA no longer fits the register file
      // or the thread limit -> pair-per-thread kernel
      int nb = 0;
      cudaError_t oe = (L2_THREADS <= 1024 && tm_lin2_smem_bytes() <= 227 * 1024)
                           ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_lin2<true>, L2_THREADS, tm_lin2_smem_bytes())
                           : cudaErrorInvalidConfiguration;
      if (h->lin_mode == 2 && (oe != cudaSuccess || nb < 1)) { h->lin_mode = 1; cudaGetLastError(); }
      // ... or only with the registers capped so low that the state spills (dims9, 27 warps: 1.4 KB of stack per thread, 3.3x
      // slower than the pair-per-thread kernel; chain, 13 warps: 0.4 KB, on par; the reference configs: none)
      cudaFuncAttributes fa;
      if (h->lin_mode == 2 && !lm && cudaFuncGetAttributes(&fa, k_lin2<true>) == cudaSuccess && fa.localSizeBytes > 1024) h->lin_mode = 1;
    }
#endif
    const char* so = getenv("TMPC_SORT");
    if (so) h->sort_lists = atoi(so) != 0;
    const char* tm = getenv("TMPC_QP_THREAD_MIN");
    if (tm) h->qp_thread_min = atoi(tm);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    h->qp_ws_per_inst = tm_qpws_doubles(P.N, P.nh, P.nxt, P.maxact);
    int tps = 1024;                        // resident threads per SM of the thread-per-instance kernel (its register budget: QT_MINB)
    // the workspace is sized by the resident grid: keep it below 24 GB for models with many rows
    while (tps > 256 && (double)prop.multiProcessorCount * tps * h->qp_ws_per_inst * sizeof(double) > 24e9) tps /= 2;
    const char* t = getenv("TMPC_QP_THREADS_PER_SM");
    if (t) tps = atoi(t);
    if (tps < 32) tps = 32;
    h->qp_blocks = prop.multiProcessorCount * (tps / tm_qp_thread_block() > 0 ? tps / tm_qp_thread_block() : 1);
    if (h->qp_mode >= 1) {
      const size_t nthreads = (size_t)h->qp_blocks * tm_qp_thread_block();
      if (cudaMalloc(&h->qp_ws, nthreads * h->qp_ws_per_inst * sizeof(double)) != cudaSuccess ||
          cudaMalloc(&h->qp_counter, sizeof(int)) != cudaSuccess) {
        fprintf(stderr, "tmpc_create: cannot allocate the QP workspace\n");
        delete h;
        return 5;
      }
    }
  }
  if (P.nh > 0) {
    TmQp0Tab& T = h->q0;
    T.EI = P.N * P.nh; T.EIs = T.EI | 1; T.n_out = P.n_w + P.n_g; T.nT = 1 + NX + T.EI;
    const char* qm = getenv("TMPC_QP0_MIN");
    if (qm) h->q0_min = atoll(qm);
    if (cudaMalloc(&T.TAB, (size_t)T.nT * T.n_out * sizeof(double)) == cudaSuccess &&
        cudaMalloc(&T.SL0, (size_t)T.EI * sizeof(double)) == cudaSuccess &&
        cudaMalloc(&T.SLPHI, (size_t)NX * T.EI * sizeof(double)) == cudaSuccess &&
        cudaMalloc(&T.MCOL, (size_t)T.EI * T.EIs * sizeof(double)) == cudaSuccess &&
        cudaMalloc(&T.bad, sizeof(int)) == cudaSuccess &&
        h->qp_warps > 0 &&
        cudaFuncSetAttribute(k_qp0_build, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->qp_smem) == cudaSuccess)
      h->q0_ok = h->q0_min >= 0;
    cudaMemset(T.MCOL, 0, (size_t)T.EI * T.EIs * sizeof(double));
  }
  for (int i = 0; i < 8; ++i) cudaEventCreate(&h->ev[i]);
  h->ev_ok = true;
  if (cudaHostAlloc(&h->host_pinned, (4 + TM_NCNT) * sizeof(unsigned long long), cudaHostAllocDefault) != cudaSuccess) {
    fprintf(stderr, "tmpc_create: cannot allocate pinned host memory\n");
    delete h;
    return 5;
  }
  if (cudaMalloc(&P.prof_counters, 4 * sizeof(unsigned long long)) == cudaSuccess) cudaMemset(P.prof_counters, 0, 4 * sizeof(unsigned long long));
  *out = h;
  return 0;
}

static void free_list(std::vector<void*>& v) {
  for (void* p : v) cudaFree(p);
  v.clear();
}

void tmpc_destroy(tmpc_handle* h) {
  if (!h) return;
  if (h->worker.joinable()) {
    { std::lock_guard<std::mutex> lk(h->mu); h->quit = true; }
    h->cv.notify_all();
    h->worker.join();
  }
  cudaSetDevice(h->device);
  if (h->host_pinned) cudaFreeHost(h->host_pinned);
  if (h->istream) cudaStreamDestroy(h->istream);
  if (h->ev_in) cudaEventDestroy(h->ev_in);

  free_list(h->tab_allocs);
  free_list(h->ws_allocs);
  if (h->qp_ws) cudaFree(h->qp_ws);
  if (h->qp_counter) cudaFree(h->qp_counter);
  if (h->qp_cold) cudaFree(h->qp_cold);
  if (h->q0.TAB) cudaFree(h->q0.TAB);
  if (h->q0.SL0) cudaFree(h->q0.SL0);
  if (h->q0.SLPHI) cudaFree(h->q0.SLPHI);
  if (h->q0.MCOL) cudaFree(h->q0.MCOL);
  if (h->q0.bad) cudaFree(h->q0.bad);
  if (h->P.prof_counters) cudaFree(h->P.prof_counters);
  if (h->jac_buf) cudaFree(h->jac_buf);
  if (h->jst_buf) cudaFree(h->jst_buf);
  for (void* q : {(void*)h->vjp_W, (void*)h->vjp_L, (void*)h->vjp_LIN, (void*)h->vjp_D, (void*)h->vjp_LQ, (void*)h->vjp_st,
                  (void*)h->vjp_Vu, (void*)h->vjp_Vw, (void*)h->vjp_G, (void*)h->vjp_js})
    if (q) cudaFree(q);
  if (h->ev_ok) for (int i = 0; i < 8; ++i) cudaEventDestroy(h->ev[i]);
  delete h;
}

}  // extern C (templates need C++ linkage)
template <typename T>
static int upload(tmpc_handle* h, std::vector<void*>& owner, const T* src, size_t n, const T** dst) {
  T* d = nullptr;
  CK(cudaMalloc(&d, (n ? n : 1) * sizeof(T)));
  owner.push_back(d);
  if (n) CK(cudaMemcpy(d, src, n * sizeof(T), cudaMemcpyHostToDevice));
  *dst = d;
  return 0;
}

extern "C" {
int tmpc_set_tables(tmpc_handle* h, const double* wref, const double* H, const double* q, const double* ref_du,
                    const double* C, const double* c, const int32_t* term_idx, const int32_t* relax0) {
  if (!h) return 1;
  cudaSetDevice(h->device);
  free_list(h->tab_allocs);
  TmProb& P = h->P;
  // symmetrise H on the way in (the reference's H blocks are symmetric, convexifier.py:206)
  std::vector<double> Hs((size_t)P.p * NZ * NZ);
  for (int ph = 0; ph < P.p; ++ph)
    for (int i = 0; i < NZ; ++i)
      for (int j = 0; j < NZ; ++j)
        Hs[((size_t)ph * NZ + i) * NZ + j] = 0.5 * (H[((size_t)ph * NZ + i) * NZ + j] + H[((size_t)ph * NZ + j) * NZ + i]);
  if (upload(h, h->tab_allocs, wref, (size_t)P.p * NZ, &P.wref)) return 1;
  if (upload(h, h->tab_allocs, Hs.data(), Hs.size(), &P.H)) return 1;
  if (upload(h, h->tab_allocs, q, (size_t)P.p * NZ, &P.q)) return 1;
  if (upload(h, h->tab_allocs, ref_du, (size_t)P.p * P.n_g, &P.ref_du)) return 1;
  if (upload(h, h->tab_allocs, C, (size_t)P.nh * NZ, &P.C)) return 1;
  if (upload(h, h->tab_allocs, c, (size_t)P.nh, &P.c)) return 1;
  if (upload(h, h->tab_allocs, (const int*)term_idx, (size_t)P.nxt, &P.term_idx)) return 1;
  if (upload(h, h->tab_allocs, (const int*)relax0, (size_t)P.nh, &P.relax0)) return 1;
  {
    std::vector<int> rowpin((size_t)(P.nh > 0 ? P.nh : 1), -1);    // rows that bound a single input (fast path of the stage elimination)
    for (int i = 0; i < P.nh; ++i) {
      int cnt = 0, jc = -1;
      for (int cidx = 0; cidx < NZ; ++cidx) if (C[(size_t)i * NZ + cidx] != 0.0) { ++cnt; jc = cidx; }
      if (cnt == 1 && jc >= NX) rowpin[i] = jc - NX;
    }
    if (upload(h, h->tab_allocs, rowpin.data(), rowpin.size(), &P.rowpin)) return 1;
  }
  h->phase_clean.assign(P.p, 1);
  for (int ph = 0; ph < P.p; ++ph)
    for (int k = 0; k < P.N; ++k)
      for (int i = 0; i < P.nh; ++i) {
        if (k == 0 && relax0[i]) continue;
        if (fabs(ref_du[(size_t)ph * P.n_g + tm_gh(P, k) + i]) >= h->opts.lam_tresh) h->phase_clean[ph] = 0;
      }
  h->tables_set = true;
  return 0;
}

}  // extern C
template <typename T>
static int dalloc(tmpc_handle* h, T** p, size_t n) {
  CK(cudaMalloc(p, (n ? n : 1) * sizeof(T)));
  h->ws_allocs.push_back(*p);
  return 0;
}

static int ensure_capacity(tmpc_handle* h, int64_t B) {
  if (B <= h->cap) return 0;
  free_list(h->ws_allocs);
  h->cap = 0;
  TmProb& P = h->P;
  TmState& S = h->S;
  S.aswords = (P.N * P.nh + 31) / 32;
  if (S.aswords < 1) S.aswords = 1;
  const size_t b = (size_t)B;
  if (dalloc(h, &S.W, b * P.n_w) || dalloc(h, &S.LAM, b * P.n_g) || dalloc(h, &S.D, b * P.n_w) ||
      dalloc(h, &S.LAMQ, b * P.n_g) || dalloc(h, &S.LIN, b * P.N * TM_LSZ) || dalloc(h, &S.G, b * P.n_g) ||
      dalloc(h, &S.FILT, b * P.filter_cap * 2) || dalloc(h, &S.fval, b) || dalloc(h, &S.nfilt, b) ||
      dalloc(h, &S.iter, b) || dalloc(h, &S.status, b) || dalloc(h, &S.flags, b) || dalloc(h, &S.nAS, b) ||
      dalloc(h, &S.nACtot, b) || dalloc(h, &S.nAC, b) || dalloc(h, &S.qpstat, b) || dalloc(h, &S.qpmode, b) || dalloc(h, &S.qpwork, b) || dalloc(h, &h->list_s, b) || dalloc(h, &h->sort_bins, 2 * SORT_BINS) || dalloc(h, &S.almask, b * TM_ALW) ||
      dalloc(h, &h->retry_a, b) || dalloc(h, &h->retry_b, b) ||
      dalloc(h, &S.asinit, b * S.aswords) || dalloc(h, &h->list_a, b) || dalloc(h, &h->list_b, b) ||
      dalloc(h, &S.list_relin, b) || dalloc(h, &h->cnts, 8) || dalloc(h, &S.counters, TM_NCNT) ||
      dalloc(h, &h->Wsh, b * P.n_w) || dalloc(h, &h->Lsh, b * P.n_g) || dalloc(h, &h->X0buf, b * NX))
    return 1;
  h->cap = B;
  return 0;
}

extern "C" {
static bool step_in_flight(tmpc_handle* h) {
  std::lock_guard<std::mutex> lk(h->mu);
  return h->busy;
}

int tmpc_reset(tmpc_handle* h, int64_t B) {
  if (!h) return 1;
  if (step_in_flight(h)) { h->err = "tmpc_reset: a step started by tmpc_step_async is still in flight (call tmpc_wait first)"; return 1; }
  if (!h->tables_set) { h->err = "tmpc_reset: tables not set"; return 1; }
  if (B < 0) { h->err = "tmpc_reset: negative batch size"; return 1; }
  cudaSetDevice(h->device);
  h->solved = false;
  if (B == 0) { h->index = 0; h->S.B = 0; h->uniform_ws = true; return 0; }
  if (ensure_capacity(h, B)) return 1;
  h->index = 0;
  h->S.B = B;
  h->uniform_ws = true;
  TmProb& P = h->P;
  // w0 <- reference window at phase 0, lam0 <- ref_du[0]   (pmpc.py:930-942)
  std::vector<double> w0(P.n_w);
  std::vector<double> wr((size_t)P.p * NZ);
  CK(cudaMemcpy(wr.data(), P.wref, wr.size() * sizeof(double), cudaMemcpyDeviceToHost));
  for (int k = 0; k < P.N; ++k)
    for (int i = 0; i < NZ; ++i) w0[k * NZ + i] = wr[(size_t)(k % P.p) * NZ + i];
  for (int i = 0; i < NX; ++i) w0[P.N * NZ + i] = wr[(size_t)(P.N % P.p) * NZ + i];
  CK(cudaMemcpy(h->Wsh, w0.data(), P.n_w * sizeof(double), cudaMemcpyHostToDevice));
  const int64_t nw = B * P.n_w, ng = B * P.n_g;
  k_bcast<<<(unsigned)((nw + 255) / 256), 256>>>(h->S.W, h->Wsh, B, P.n_w);
  CK(cudaDeviceSynchronize());   // Wsh row is overwritten below only by later steps; keep ordering simple
  k_bcast<<<(unsigned)((ng + 255) / 256), 256>>>(h->S.LAM, P.ref_du, B, P.n_g);
  CK(cudaMemset(h->S.qpwork, 0, (size_t)B * sizeof(int)));
  CK(cudaGetLastError());
  CK(cudaDeviceSynchronize());
  return 0;
}

int tmpc_get_index(const tmpc_handle* h, int64_t* index) {
  if (!h || !index) return 1;
  *index = h->index;
  return 0;
}

int tmpc_step(tmpc_handle* h, const double* X0_dev, int64_t B, double* U0_dev, double* W_dev, double* LAM_dev,
              double* G_dev, int32_t* status_dev, int32_t* iter_dev, int32_t* flags_dev, void* cuda_stream) {
  if (!h) return 1;
  if (B < 0) { h->err = "tmpc_step: negative batch size"; return 1; }
  if (!h->tables_set || h->cap < B || h->S.B != B) { h->err = "tmpc_step: call tmpc_reset(B) first"; return 1; }
  if (B == 0) { h->index += 1; h->solved = true; return 0; }   // empty batch: nothing to solve, the phase still advances
  cudaSetDevice(h->device);
  h->solved = false;                                         // set again once this step has finished
  cudaStream_t st = (cudaStream_t)cuda_stream;
  TmProb& P = h->P;
  TmState& S = h->S;
  S.X0 = X0_dev;
  S.phase = (int)(h->index % P.p);                           // pmpc.py:377
  S.list_next = h->list_a;
  S.cnt_next = h->cnts;
  S.cnt_relin = h->cnts + 1;
  int64_t launches = 0, n_qp = 0, n_lin = 0;
  float ms_lin = 0, ms_qp = 0, ms_post = 0, ms;
  const unsigned wblocks = (unsigned)((B + QP_WARPS - 1) / QP_WARPS);

  CK(cudaMemsetAsync(S.counters, 0, TM_NCNT * sizeof(unsigned long long), st));
  CK(cudaEventRecord(h->ev[6], st));
  k_prefilter<<<wblocks, QP_WARPS * 32, 0, st>>>(P, S);
  CK(cudaEventRecord(h->ev[0], st));
  const bool was_uniform = h->uniform_ws;   // first step after reset: no per-instance QP cost history yet
  if (h->uniform_ws && B > 1) {
    // right after reset every instance starts from the same (w0, lam0): linearise one and replicate the record
    CK(launch_lin(h, S, nullptr, 1, 0, st));
    const int64_t nrec = (int64_t)P.N * TM_LSZ;
    k_bcast<<<(unsigned)(((B - 1) * nrec + 255) / 256), 256, 0, st>>>(S.LIN + nrec, S.LIN, B - 1, (int)nrec);
    ++launches; n_lin -= (B - 1) * P.N;
  } else {
    CK(launch_lin(h, S, nullptr, B, 0, st));
  }
  h->uniform_ws = false;
  CK(cudaEventRecord(h->ev[1], st));
  k_init<<<wblocks, QP_WARPS * 32, 0, st>>>(P, S);
  CK(cudaGetLastError());
  launches += 3; n_lin += B * P.N;
  CK(cudaEventSynchronize(h->ev[1]));
  CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1])); ms_lin += ms;

  const int* cur = nullptr;   // nullptr = identity list (all instances)
  const int* src = nullptr;   // the list the previous iteration produced (list_a / list_b), before sorting
  int64_t nact = B;
  // pinned host words for the per-iteration counters: a D2H copy into pageable memory is not truly asynchronous (it may
  // synchronise with the legacy default stream, which tmpc_step_async holds on its ticket)
  int* hc = (int*)h->host_pinned;
  int iter_guard = 0;
  while (nact > 0) {
    const unsigned wb = (unsigned)((nact + QP_WARPS - 1) / QP_WARPS);
    S.list_next = (src == h->list_a) ? h->list_b : h->list_a;
    cur = src;
    if (h->sort_lists && h->qp_mode >= 1 && nact >= h->qp_thread_min && !(was_uniform && iter_guard == 0)) {
      const unsigned sb = (unsigned)((nact + 255) / 256);
      CK(cudaMemsetAsync(h->sort_bins, 0, 2 * SORT_BINS * sizeof(int), st));
      k_sort_hist<<<sb, 256, 0, st>>>(src, (int)nact, S.qpwork, h->sort_bins);
      k_sort_scan<<<1, 32, 0, st>>>(h->sort_bins);
      k_sort_scatter<<<sb, 256, 0, st>>>(src, (int)nact, S.qpwork, h->sort_bins, h->list_s);
      launches += 3;
      cur = h->list_s;
    }
    CK(cudaMemsetAsync(h->cnts, 0, 4 * sizeof(int), st));
    CK(cudaEventRecord(h->ev[0], st));
    for (int pass = 0; pass < 2; ++pass) {
      // pass 0: the active list (host-known count); pass 1: instances the shared-table route of the first QP handed
      // back (device count).  Re-solves of one instance's QP (released base rows, Gauss-Newton fallback) happen inside tm_qp.
      const int* plist = pass == 0 ? cur : h->retry_a;
      const int* pcnt = pass == 0 ? nullptr : h->cnts + 2;
      S.list_retry = h->retry_a;
      S.cnt_retry = h->cnts + 2;
      const bool use_thread = h->qp_mode == 1 || (h->qp_mode == 2 && nact >= h->qp_thread_min);
      bool q0 = false;
      if (pass == 0 && iter_guard == 0 && was_uniform && h->q0_ok && B >= h->q0_min && B > 1 && h->phase_clean[S.phase]) {
        // every instance shares (w0, lam0): tabulate the parametric QP once, then one thread per instance on the tables
        const TmQp0Tab& T = h->q0;
        CK(cudaMemsetAsync(T.bad, 0, sizeof(int), st));
        k_qp0_build<<<std::min((T.nT + h->qp_warps - 1) / h->qp_warps, h->qp_wgrid), h->qp_warps * 32, h->qp_smem, st>>>(P, S, T, h->qp_cold);
        k_qp0_derive<<<(T.nT * T.EI + 127) / 128, 128, 0, st>>>(P, S, T);
        k_qp0<<<(unsigned)((B + Q0_THREADS - 1) / Q0_THREADS), Q0_THREADS, 0, st>>>(P, S, T, (int)B);
        launches += 2;
        q0 = true;
      } else if (pass == 1 && !(iter_guard == 0 && was_uniform)) {
        break;                                     // nothing can be queued outside the shared-table route
      } else if (use_thread)
        CK(tm_launch_qp_thread(P, S, plist, (int)nact, pcnt, h->qp_ws, h->qp_ws_per_inst, h->qp_blocks, h->qp_counter, st));
      else
        k_qp<<<(unsigned)std::min<int64_t>((nact + h->qp_warps - 1) / h->qp_warps, h->qp_wgrid), h->qp_warps * 32, h->qp_smem, st>>>(P, S, plist, (int)nact, pcnt, h->qp_cold);
      ++launches;
      if (pass == 0 && !q0) break;
    }
    CK(cudaEventRecord(h->ev[1], st));
    CK(launch_lin(h, S, cur, nact, 1, st));
    CK(cudaEventRecord(h->ev[2], st));
    k_post<<<wb, QP_WARPS * 32, 0, st>>>(P, S, cur, (int)nact);
    CK(cudaEventRecord(h->ev[3], st));
    CK(cudaGetLastError());
    launches += 2; n_qp += nact; n_lin += nact * P.N;
    CK(cudaMemcpyAsync(hc, h->cnts, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    {
      float a, b2, c2;
      CK(cudaEventElapsedTime(&a, h->ev[0], h->ev[1])); ms_qp += a;
      CK(cudaEventElapsedTime(&b2, h->ev[1], h->ev[2])); ms_lin += b2;
      CK(cudaEventElapsedTime(&c2, h->ev[2], h->ev[3])); ms_post += c2;
      if (h->trace) fprintf(stderr, "[tmpc] it %3d nact %8lld  qp %9.3f ms  lin %9.3f ms  post %8.3f ms  next %d relin %d\n",
                            iter_guard, (long long)nact, a, b2, c2, hc[0], hc[1]);
    }
    if (hc[1] > 0) {   // damped steps: re-linearise at the accepted point, then test convergence
      CK(cudaEventRecord(h->ev[0], st));
      CK(launch_lin(h, S, S.list_relin, hc[1], 0, st));
      CK(cudaEventRecord(h->ev[1], st));
      k_conv<<<(unsigned)((hc[1] + QP_WARPS - 1) / QP_WARPS), QP_WARPS * 32, 0, st>>>(P, S, S.list_relin, S.cnt_relin);
      CK(cudaEventRecord(h->ev[2], st));
      CK(cudaGetLastError());
      launches += 2; n_lin += (int64_t)hc[1] * P.N;
      CK(cudaMemcpyAsync(hc, h->cnts, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1])); ms_lin += ms;
      CK(cudaEventElapsedTime(&ms, h->ev[1], h->ev[2])); ms_post += ms;
    }
    src = S.list_next;
    nact = hc[0];
    if (++iter_guard > P.max_iter + 2) { h->err = "tmpc_step: iteration guard tripped"; return 1; }
  }
  // post-solve sanity check of the reference (sqp_method.py:190-201): reduced Hessian positive definite at the solution
  if (h->pd_check) {
    TmState Sc = S;
    Sc.pd_check = 1;
    const bool use_thread = h->qp_mode == 1 || (h->qp_mode == 2 && B >= h->qp_thread_min);
    if (use_thread)
      CK(tm_launch_qp_thread(P, Sc, nullptr, (int)B, nullptr, h->qp_ws, h->qp_ws_per_inst, h->qp_blocks, h->qp_counter, st));
    else
      k_qp<<<(unsigned)std::min<int64_t>((B + h->qp_warps - 1) / h->qp_warps, h->qp_wgrid), h->qp_warps * 32, h->qp_smem, st>>>(P, Sc, nullptr, (int)B, nullptr, h->qp_cold);
    CK(cudaGetLastError());
    ++launches;
  }
  // outputs, then the warm-start shift (pmpc.py:410-423)
  const size_t b = (size_t)B;
  if (U0_dev) { k_gather_u0<<<(unsigned)((B * NUM + 255) / 256), 256, 0, st>>>(P, S, U0_dev); ++launches; }
  if (W_dev) CK(cudaMemcpyAsync(W_dev, S.W, b * P.n_w * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (LAM_dev) CK(cudaMemcpyAsync(LAM_dev, S.LAM, b * P.n_g * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (G_dev) CK(cudaMemcpyAsync(G_dev, S.G, b * P.n_g * sizeof(double), cudaMemcpyDeviceToDevice, st));
  if (status_dev) CK(cudaMemcpyAsync(status_dev, S.status, b * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (iter_dev) CK(cudaMemcpyAsync(iter_dev, S.iter, b * sizeof(int), cudaMemcpyDeviceToDevice, st));
  if (flags_dev) CK(cudaMemcpyAsync(flags_dev, S.flags, b * sizeof(int), cudaMemcpyDeviceToDevice, st));
  k_shift<<<wblocks, QP_WARPS * 32, 0, st>>>(P, S, h->Wsh, h->Lsh);
  ++launches;
  CK(cudaGetLastError());
  CK(cudaEventRecord(h->ev[7], st));
  unsigned long long* cnt_host = (unsigned long long*)h->host_pinned + 4;
  CK(cudaMemcpyAsync(cnt_host, S.counters, TM_NCNT * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  { double* t = S.W; S.W = h->Wsh; h->Wsh = t; }
  { double* t = S.LAM; S.LAM = h->Lsh; h->Lsh = t; }
  h->solved = true;
  h->index += 1;                                             // pmpc.py:415
  CK(cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]));
  h->timing_ms[0] = ms_lin; h->timing_ms[1] = ms_qp; h->timing_ms[2] = ms_post; h->timing_ms[3] = ms;
  h->counters_host[0] = (int64_t)cnt_host[0];
  h->counters_host[1] = launches;
  h->counters_host[2] = n_qp;
  h->counters_host[3] = n_lin;
  h->counters_host[4] = (int64_t)cnt_host[4];
  h->counters_host[5] = (int64_t)cnt_host[5];
  h->counters_host[6] = (int64_t)cnt_host[6];
  h->counters_host[7] = (int64_t)cnt_host[7];
  if (h->trace) {
    fprintf(stderr, "[tmpc] qp attempts %llu gi %llu ricc %llu | fresh ok/inf/npd/mask %llu %llu %llu %llu | retry %llu %llu %llu %llu | gn %llu %llu %llu %llu\n",
            cnt_host[5], cnt_host[6], cnt_host[7], cnt_host[8], cnt_host[9], cnt_host[10], cnt_host[11], cnt_host[12],
            cnt_host[13], cnt_host[14], cnt_host[15], cnt_host[16], cnt_host[17], cnt_host[18], cnt_host[19]);
    if (cnt_host[20]) {
      unsigned long long pc[4] = {0, 0, 0, 0};
      if (P.prof_counters) { cudaMemcpy(pc, P.prof_counters, sizeof pc, cudaMemcpyDeviceToHost); cudaMemset(P.prof_counters, 0, sizeof pc); }
      fprintf(stderr, "[tmpc] warp-kernel cycles per attempt: factor %.0f (of which the block products P[A B], Q + [A B]'P[A B]: %.0f)  dual active set %.0f  correction solve %.0f  multiplier recovery %.0f\n",
              (double)cnt_host[20] / cnt_host[5], (double)pc[0] / cnt_host[5], (double)cnt_host[21] / cnt_host[5], (double)cnt_host[22] / cnt_host[5], (double)cnt_host[23] / cnt_host[5]);
    }
  }
  return 0;
}

// ---- asynchronous call -------------------------------------------------------------------------------------------------------
static void async_worker(tmpc_handle* h) {
  cudaSetDevice(h->device);
  for (;;) {
    tmpc_handle::AsyncJob j;
    {
      std::unique_lock<std::mutex> lk(h->mu);
      h->cv.wait(lk, [h] { return h->has_job || h->quit; });
      if (h->quit) return;
      j = h->job;
      h->has_job = false;
    }
    cudaStreamWaitEvent(h->istream, h->ev_in, 0);                  // inputs enqueued on the caller's stream before the call
    const int rc = tmpc_step(h, j.X0, j.B, j.U0, j.W, j.LAM, j.G, j.status, j.iter, j.flags, (void*)h->istream);
    cudaStreamSynchronize(h->istream);                             // every output is complete before the step reports done
    {
      std::lock_guard<std::mutex> lk(h->mu);
      h->job_rc = rc;
      h->busy = false;
    }
    h->cv.notify_all();
  }
}

int tmpc_step_async(tmpc_handle* h, const double* X0_dev, int64_t B, double* U0_dev, double* W_dev, double* LAM_dev,
                    double* G_dev, int32_t* status_dev, int32_t* iter_dev, int32_t* flags_dev, void* cuda_stream) {
  if (!h) return 1;
  cudaSetDevice(h->device);
  {
    std::lock_guard<std::mutex> lk(h->mu);
    if (h->busy) { h->err = "tmpc_step_async: a step is still in flight on this handle (call tmpc_wait first)"; return 1; }
  }
  if (!h->async_ready) {
    CK(cudaStreamCreateWithFlags(&h->istream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
    h->worker = std::thread(async_worker, h);
    h->async_ready = true;
  }
  CK(cudaEventRecord(h->ev_in, (cudaStream_t)cuda_stream));       // the worker's stream waits for what the caller enqueued so far
  {
    std::lock_guard<std::mutex> lk(h->mu);
    h->job = {X0_dev, B, U0_dev, W_dev, LAM_dev, G_dev, status_dev, iter_dev, flags_dev};
    h->has_job = true;
    h->busy = true;
  }
  h->cv.notify_all();
  return 0;
}

int tmpc_wait(tmpc_handle* h) {
  if (!h) return 1;
  std::unique_lock<std::mutex> lk(h->mu);
  h->cv.wait(lk, [h] { return !h->busy; });
  return h->job_rc;
}

int tmpc_busy(tmpc_handle* h, int32_t* busy) {
  if (!h || !busy) return 1;
  std::lock_guard<std::mutex> lk(h->mu);
  *busy = h->busy ? 1 : 0;
  return 0;
}

int tmpc_step_host(tmpc_handle* h, const double* X0_host, int64_t B, double* U0_host, double* W_host,
                   double* LAM_host, double* G_host, int32_t* status_host, int32_t* iter_host, int32_t* flags_host) {
  if (!h) return 1;
  if (step_in_flight(h)) { h->err = "tmpc_step_host: a step started by tmpc_step_async is still in flight (call tmpc_wait first)"; return 1; }
  if (h->cap < B) { h->err = "tmpc_step_host: call tmpc_reset(B) first"; return 1; }
  if (B == 0) return tmpc_step(h, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
  cudaSetDevice(h->device);
  TmProb& P = h->P;
  const size_t b = (size_t)B;
  CK(cudaMemcpy(h->X0buf, X0_host, b * NX * sizeof(double), cudaMemcpyHostToDevice));
  // the solution lives in S.W / S.LAM until the shift swaps buffers: copy out of the pre-swap buffers
  double *Wsol = h->S.W, *Lsol = h->S.LAM;
  if (tmpc_step(h, h->X0buf, B, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr)) return 1;
  // after the swap the solution buffers are h->Wsh / h->Lsh (== Wsol / Lsol)
  if (U0_host) CK(cudaMemcpy2D(U0_host, NUM * sizeof(double), Wsol + NX, P.n_w * sizeof(double), NUM * sizeof(double), b,
                               cudaMemcpyDeviceToHost));
  if (W_host) CK(cudaMemcpy(W_host, Wsol, b * P.n_w * sizeof(double), cudaMemcpyDeviceToHost));
  if (LAM_host) CK(cudaMemcpy(LAM_host, Lsol, b * P.n_g * sizeof(double), cudaMemcpyDeviceToHost));
  if (G_host) CK(cudaMemcpy(G_host, h->S.G, b * P.n_g * sizeof(double), cudaMemcpyDeviceToHost));
  if (status_host) CK(cudaMemcpy(status_host, h->S.status, b * sizeof(int), cudaMemcpyDeviceToHost));
  if (iter_host) CK(cudaMemcpy(iter_host, h->S.iter, b * sizeof(int), cudaMemcpyDeviceToHost));
  if (flags_host) CK(cudaMemcpy(flags_host, h->S.flags, b * sizeof(int), cudaMemcpyDeviceToHost));
  return 0;
}

int tmpc_feedback_jacobian(tmpc_handle* h, double* J, int32_t* jstatus, int dst_is_host, void* cuda_stream) {
  if (!h) return 1;
  if (step_in_flight(h)) { h->err = "tmpc_feedback_jacobian: a step started by tmpc_step_async is still in flight (call tmpc_wait first)"; return 1; }
  if (!h->P.hessian_exact) { h->err = "tmpc_feedback_jacobian: needs the exact Hessian (a Gauss-Newton controller's linearisation has no second-order term)"; return 1; }
  if (!h->solved) { h->err = "tmpc_feedback_jacobian: no step has finished since tmpc_create / tmpc_reset"; return 1; }
  const int64_t B = h->S.B;
  if (B == 0) return 0;
  if (!J || !jstatus) { h->err = "tmpc_feedback_jacobian: J and jstatus are required"; return 1; }
  cudaSetDevice(h->device);
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const TmProb& P = h->P;
  double* Jd = J;
  int* jsd = (int*)jstatus;
  if (dst_is_host) {
    if (h->jac_cap < B) {
      if (h->jac_buf) cudaFree(h->jac_buf);
      if (h->jst_buf) cudaFree(h->jst_buf);
      h->jac_buf = nullptr; h->jst_buf = nullptr; h->jac_cap = 0;
      CK(cudaMalloc(&h->jac_buf, (size_t)B * NUM * NX * sizeof(double)));
      CK(cudaMalloc(&h->jst_buf, (size_t)B * sizeof(int)));
      h->jac_cap = B;
    }
    Jd = h->jac_buf;
    jsd = h->jst_buf;
  }
  // the solutions of the last step: after its warm-start shift they live in Wsh / Lsh; LIN still holds the linearisation at
  // them (nothing after a step's convergence test writes LIN, D or LAMQ before the next step).  X0 only has to be a valid
  // buffer (the perturbed solves replace the x_0 offset): the staging buffer, never the caller's pointer of the last step.
  TmState Sc = h->S;
  Sc.W = h->Wsh;
  Sc.LAM = h->Lsh;
  Sc.X0 = h->X0buf;
  const bool use_thread = h->qp_mode == 1 || (h->qp_mode == 2 && B >= h->qp_thread_min);
  if (use_thread) {
    CK(tm_launch_fbjac_thread(P, Sc, (int)B, h->qp_ws, h->qp_ws_per_inst, h->qp_blocks, h->qp_counter, Jd, jsd, st));
  } else {
    if (!h->fbjac_smem) {
      CK(cudaFuncSetAttribute(k_fbjac, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->qp_smem));
      h->fbjac_smem = true;
    }
    k_fbjac<<<(unsigned)std::min<int64_t>((B + h->qp_warps - 1) / h->qp_warps, h->qp_wgrid), h->qp_warps * 32, h->qp_smem, st>>>(P, Sc, (int)B, h->qp_cold, Jd, jsd);
    CK(cudaGetLastError());
  }
  if (dst_is_host) {
    CK(cudaMemcpyAsync(J, Jd, (size_t)B * NUM * NX * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(jstatus, jsd, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  return 0;
}

static int vjp_capacity(tmpc_handle* h, int64_t B, bool io) {
  const TmProb& P = h->P;
  const size_t b = (size_t)B;
  if (h->vjp_cap < B) {
    for (void** q : {(void**)&h->vjp_W, (void**)&h->vjp_L, (void**)&h->vjp_LIN, (void**)&h->vjp_D, (void**)&h->vjp_LQ,
                     (void**)&h->vjp_st}) {
      if (*q) cudaFree(*q);
      *q = nullptr;
    }
    h->vjp_cap = 0;
    CK(cudaMalloc(&h->vjp_W, b * P.n_w * sizeof(double)));
    CK(cudaMalloc(&h->vjp_L, b * P.n_g * sizeof(double)));
    CK(cudaMalloc(&h->vjp_LIN, b * P.N * TM_LSZ * sizeof(double)));
    CK(cudaMalloc(&h->vjp_D, b * P.n_w * sizeof(double)));
    CK(cudaMalloc(&h->vjp_LQ, b * P.n_g * sizeof(double)));
    CK(cudaMalloc(&h->vjp_st, b * sizeof(int)));
    h->vjp_cap = B;
  }
  if (io && h->vjp_io_cap < B) {
    for (void** q : {(void**)&h->vjp_Vu, (void**)&h->vjp_Vw, (void**)&h->vjp_G, (void**)&h->vjp_js}) {
      if (*q) cudaFree(*q);
      *q = nullptr;
    }
    h->vjp_io_cap = 0;
    CK(cudaMalloc(&h->vjp_Vu, b * NUM * sizeof(double)));
    CK(cudaMalloc(&h->vjp_Vw, b * P.n_w * sizeof(double)));
    CK(cudaMalloc(&h->vjp_G, b * NX * sizeof(double)));
    CK(cudaMalloc(&h->vjp_js, b * sizeof(int)));
    h->vjp_io_cap = B;
  }
  return 0;
}

int tmpc_solution_vjp(tmpc_handle* h, int64_t B, const double* W, const double* LAM, const int32_t* status, int32_t phase,
                      const double* V_u0, const double* V_w, double* G_x0, int32_t* jstatus, int is_host, void* cuda_stream) {
  if (!h) return 1;
  if (step_in_flight(h)) { h->err = "tmpc_solution_vjp: a step started by tmpc_step_async is still in flight (call tmpc_wait first)"; return 1; }
  if (!h->P.hessian_exact) { h->err = "tmpc_solution_vjp: needs the exact Hessian (a Gauss-Newton controller's linearisation has no second-order term)"; return 1; }
  if (B < 0) { h->err = "tmpc_solution_vjp: negative batch size"; return 1; }
  const TmProb& P = h->P;
  const bool stored = W == nullptr;
  if (stored) {
    if (LAM || status) { h->err = "tmpc_solution_vjp: W == NULL selects the last step's solutions: LAM and status must be NULL too"; return 1; }
    if (!h->solved) { h->err = "tmpc_solution_vjp: W == NULL and no step has finished since tmpc_create / tmpc_reset"; return 1; }
    if (B != h->S.B) { h->err = "tmpc_solution_vjp: W == NULL needs B equal to the last step's batch size"; return 1; }
  } else {
    if (!LAM || !status) { h->err = "tmpc_solution_vjp: W, LAM and status are given together"; return 1; }
    if (phase < 0 || phase >= P.p) { h->err = "tmpc_solution_vjp: phase outside [0, p)"; return 1; }
  }
  if (!V_u0 && !V_w) { h->err = "tmpc_solution_vjp: both cotangents are NULL"; return 1; }
  if (B == 0) return 0;
  if (!G_x0 || !jstatus) { h->err = "tmpc_solution_vjp: G_x0 and jstatus are required"; return 1; }
  cudaSetDevice(h->device);
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (vjp_capacity(h, B, is_host != 0)) return 1;
  const size_t b = (size_t)B;
  const cudaMemcpyKind kin = is_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const double* Vu = V_u0;
  const double* Vw = V_w;
  double* Gd = G_x0;
  int* jsd = (int*)jstatus;
  if (is_host) {
    if (V_u0) CK(cudaMemcpyAsync(h->vjp_Vu, V_u0, b * NUM * sizeof(double), kin, st));
    if (V_w) CK(cudaMemcpyAsync(h->vjp_Vw, V_w, b * P.n_w * sizeof(double), kin, st));
    Vu = V_u0 ? h->vjp_Vu : nullptr;
    Vw = V_w ? h->vjp_Vw : nullptr;
    Gd = h->vjp_G;
    jsd = h->vjp_js;
  }
  // The solution, its status and its linearisation records.  W == NULL: the last step's, read in place (after its warm-start
  // shift the solutions live in Wsh / Lsh and LIN holds the linearisation at them, as for tmpc_feedback_jacobian).  Otherwise a
  // copy in the VJP's own buffers, linearised again there with the step's dispatch: the handle's W, LAM, LIN, D and LAMQ stay
  // untouched.  X0 only has to be readable (the solve replaces the x_0 offset that tm_qp_setup forms from it).
  TmState Sv = h->S;
  Sv.B = B;
  if (stored) {
    Sv.W = h->Wsh;
    Sv.LAM = h->Lsh;
  } else {
    CK(cudaMemcpyAsync(h->vjp_W, W, b * P.n_w * sizeof(double), kin, st));
    CK(cudaMemcpyAsync(h->vjp_L, LAM, b * P.n_g * sizeof(double), kin, st));
    CK(cudaMemcpyAsync(h->vjp_st, status, b * sizeof(int), kin, st));
    Sv.W = h->vjp_W;
    Sv.LAM = h->vjp_L;
    Sv.LIN = h->vjp_LIN;
    Sv.status = h->vjp_st;
    Sv.phase = phase;
    CK(launch_lin(h, Sv, nullptr, B, 0, st));
  }
  Sv.X0 = Sv.W;
  const bool use_thread = h->qp_mode == 1 || (h->qp_mode == 2 && B >= h->qp_thread_min);
  if (use_thread) {
    CK(tm_launch_vjp_thread(P, Sv, (int)B, h->qp_ws, h->qp_ws_per_inst, h->qp_blocks, h->qp_counter, Vu, Vw, h->vjp_D, h->vjp_LQ,
                            Gd, jsd, st));
  } else {
    if (!h->vjp_smem) {
      CK(cudaFuncSetAttribute(k_vjp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->qp_smem));
      h->vjp_smem = true;
    }
    k_vjp<<<(unsigned)std::min<int64_t>((B + h->qp_warps - 1) / h->qp_warps, h->qp_wgrid), h->qp_warps * 32, h->qp_smem, st>>>(
        P, Sv, (int)B, h->qp_cold, Vu, Vw, h->vjp_D, h->vjp_LQ, Gd, jsd);
    CK(cudaGetLastError());
  }
  if (is_host) {
    CK(cudaMemcpyAsync(G_x0, Gd, b * NX * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(jstatus, jsd, b * sizeof(int), cudaMemcpyDeviceToHost, st));
  }
  CK(cudaStreamSynchronize(st));
  return 0;
}

int tmpc_plant_jacobian(tmpc_handle* h, const double* X_dev, const double* U_dev, int64_t B, double* JF_dev, void* cuda_stream) {
  if (!h) return 1;
  if (B < 0) { h->err = "tmpc_plant_jacobian: negative batch size"; return 1; }
  if (B == 0) return 0;
  cudaSetDevice(h->device);
  k_plant_jac<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(X_dev, U_dev, B, JF_dev);
  CK(cudaGetLastError());
  return 0;
}

int tmpc_plant_step(tmpc_handle* h, const double* X_dev, const double* U_dev, int64_t B, double* Xn_dev,
                    void* cuda_stream) {
  if (!h) return 1;
  cudaSetDevice(h->device);
  k_plant<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(X_dev, U_dev, B, Xn_dev);
  CK(cudaGetLastError());
  return 0;
}

int tmpc_stage_log(tmpc_handle* h, const double* X_dev, const double* U_dev, int64_t B, double* l_dev, double* h_dev,
                   void* cuda_stream) {
  if (!h) return 1;
  if (!h->tables_set) { h->err = "tmpc_stage_log: tables not set"; return 1; }
  cudaSetDevice(h->device);
  k_stage_log<<<(unsigned)((B + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(X_dev, U_dev, B, h->P.C, h->P.c, h->P.nh,
                                                                                 l_dev, h->P.nh > 0 ? h_dev : nullptr);
  CK(cudaGetLastError());
  return 0;
}

int tmpc_get_log(tmpc_handle* h, double* f, int32_t* nAS, int32_t* nACtot, int32_t* nAC, int dst_is_host) {
  if (!h) return 1;
  cudaSetDevice(h->device);
  const cudaMemcpyKind kd = dst_is_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  const size_t b = (size_t)h->S.B;
  if (f) CK(cudaMemcpy(f, h->S.fval, b * sizeof(double), kd));
  if (nAS) CK(cudaMemcpy(nAS, h->S.nAS, b * sizeof(int), kd));
  if (nACtot) CK(cudaMemcpy(nACtot, h->S.nACtot, b * sizeof(int), kd));
  if (nAC) CK(cudaMemcpy(nAC, h->S.nAC, b * sizeof(int), kd));
  return 0;
}

int tmpc_get_counters(const tmpc_handle* h, int64_t out[8]) {
  if (!h) return 1;
  memcpy(out, h->counters_host, sizeof h->counters_host);
  return 0;
}

int tmpc_get_timing(const tmpc_handle* h, double out_ms[4]) {
  if (!h) return 1;
  memcpy(out_ms, h->timing_ms, sizeof h->timing_ms);
  return 0;
}

int tmpc_stage_eval_host(int32_t n, const double* x, const double* u, int32_t order, double* xf, double* S, double* T) {
  for (int s = 0; s < n; ++s) {
    const double* xs = x + (size_t)s * NX;
    const double* us = u + (size_t)s * NUM;
    if (order == 0) {
      double t1[NX], t2[NX], t3[NX];
      tm_integrate<0>(xs, us, 0, 0, xf + (size_t)s * NX, t1, t2, t3);
      continue;
    }
#pragma push_macro("NZ")
#undef NZ
#define NZ TMPC_NZM
    for (int i = 0; i < NZ; ++i)
      for (int j = i; j < NZ; ++j) {
        if (order == 1 && j != i) continue;
        double X[NX], Si[NX], Sj[NX], Tt[NX];
        if (order == 1) tm_integrate<1>(xs, us, i, j, X, Si, Sj, Tt);
        else tm_integrate<2>(xs, us, i, j, X, Si, Sj, Tt);
        for (int a = 0; a < NX; ++a) {
          xf[(size_t)s * NX + a] = X[a];
          if (i == j) S[((size_t)s * NX + a) * NZ + i] = Si[a];
          if (order == 2) {
            T[(((size_t)s * NX + a) * NZ + i) * NZ + j] = Tt[a];
            T[(((size_t)s * NX + a) * NZ + j) * NZ + i] = Tt[a];
          }
        }
      }
#pragma pop_macro("NZ")
  }
  return 0;
}

int tmpc_fp64_peak(tmpc_handle* h, double* tflops) {
  if (!h || !tflops) return 1;
  cudaSetDevice(h->device);
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, h->device));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
  double* out = nullptr;
  CK(cudaMalloc(&out, (size_t)blocks * threads * sizeof(double)));
  k_fp64_peak<<<blocks, threads>>>(out, 1024);
  CK(cudaDeviceSynchronize());
  double best = 0.0;
  for (int rep = 0; rep < 3; ++rep) {
    CK(cudaEventRecord(h->ev[4]));
    k_fp64_peak<<<blocks, threads>>>(out, iters);
    CK(cudaEventRecord(h->ev[5]));
    CK(cudaEventSynchronize(h->ev[5]));
    float ms;
    CK(cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]));
    const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
    const double tf = fl / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  cudaFree(out);
  *tflops = best;
  return 0;
}

}  // extern "C"
