// tmpc_vjp_thread.cu -- the solution VJP (tm_solution_vjp) as one thread per instance, on the workspace of the thread-per-instance
// QP kernel.  A translation unit of its own for the reason tmpc_fbjac_thread.cu is one: tm_qp_solve is __noinline__, and another
// perturbed caller in an existing file would change the code of that file's copy.
#include "tmpc_qp_thread.cuh"

// solution VJP at a stored or the last step's solutions (tm_solution_vjp), thread per instance on the QP kernel's workspace:
// the same CTA size and register budget, at most `nblocks` CTAs (the workspace is sized by that grid)
__global__ void __launch_bounds__(QT_THREADS, QT_MINB) k_vjp_thread(TmProb P, TmState S, int cnt, double* wsbase, size_t ws_per_inst,
                                                           int* work_counter, const double* Vu0, const double* Vw, double* dscr,
                                                           double* lscr, double* G, int* jst) {
  const int lane = threadIdx.x & 31;
  const size_t gwarp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  double* base = wsbase + gwarp * ws_per_inst * 32 + lane;
  TmQpWs ws;
  tm_qpws_carve(base, P.N, P.nh, P.nxt, P.maxact, ws);
  double lscr_local[TM_QP_LSCR];
  tm_qpws_local(lscr_local, ws);
  for (;;) {
    int start = 0;
    if (lane == 0) start = atomicAdd(work_counter, 32);
    start = __shfl_sync(0xffffffffu, start, 0);
    if (start >= cnt) break;
    const int slot = start + lane;
    if (slot < cnt) tm_solution_vjp(P, S, slot, ws, Vu0, Vw, dscr, lscr, G, jst);
    __syncwarp();
  }
}

cudaError_t tm_launch_vjp_thread(const TmProb& P, const TmState& S, int cnt, double* wsbase, size_t ws_per_inst, int nblocks,
                                 int* work_counter, const double* Vu0, const double* Vw, double* dscr, double* lscr, double* G,
                                 int* jst, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  const int need = (cnt + QT_THREADS - 1) / QT_THREADS;
  k_vjp_thread<<<need < nblocks ? need : nblocks, QT_THREADS, 0, st>>>(P, S, cnt, wsbase, ws_per_inst, work_counter, Vu0, Vw, dscr,
                                                                       lscr, G, jst);
  return cudaGetLastError();
}
