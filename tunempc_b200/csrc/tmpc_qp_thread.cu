// tmpc_qp_thread.cu -- K3/K4 as ONE THREAD PER INSTANCE (the production QP kernel).
//
// Why: ncu on the warp-per-instance kernel (profiles/r01a_summary.md) showed it latency bound -- 36.7 KB of shared
// memory per instance leaves 4 resident warps per SM, 4 of 32 lanes busy, FP64 pipe 4 % active.  The per-instance QP
// is a long chain of tiny dependent operations; the parallelism that exists is ACROSS instances.  Here every lane owns
// an instance, the workspace lives in global memory in a lane-interleaved layout (element e of lane l at
// base[e*32 + l]: a warp reading "its" element e issues one coalesced 256-byte transaction), and the number of
// instances in flight is bounded by the grid, not by shared memory.  The routine itself is the same source as the
// warp version (tmpc_core.cuh compiled with TM_THREAD_MODE: TM_NL = 1, no warp collectives, no __syncwarp).
#include "tmpc_qp_thread.cuh"

__global__ void __launch_bounds__(QT_THREADS, QT_MINB) k_qp_thread(TmProb P, TmState S, const int* list, int cnt, const int* cnt_dev,
                                                          double* wsbase, size_t ws_per_inst, int* work_counter) {
  if (cnt_dev) cnt = *cnt_dev;
  const int lane = threadIdx.x & 31;
  const size_t gwarp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  double* base = wsbase + gwarp * ws_per_inst * 32 + lane;
  TmQpWs ws;
  tm_qpws_carve(base, P.N, P.nh, P.nxt, P.maxact, ws);
  double lscr[TM_QP_LSCR];                      // per-stage scratch of the factorisation: thread-local (registers / L1)
  tm_qpws_local(lscr, ws);
  for (;;) {
    int start = 0;
    if (lane == 0) start = atomicAdd(work_counter, 32);
    start = __shfl_sync(0xffffffffu, start, 0);
    if (start >= cnt) break;
    const int slot = start + lane;
    if (slot < cnt) {
      const int64_t inst = list ? list[slot] : slot;
      tm_qp(P, S, inst, ws);
    }
    __syncwarp();
  }
}

// host launcher used by tmpc.cu
cudaError_t tm_launch_qp_thread(const TmProb& P, const TmState& S, const int* list, int cnt, const int* cnt_dev,
                                double* wsbase, size_t ws_per_inst, int nblocks, int* work_counter, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(work_counter, 0, sizeof(int), st);
  if (e != cudaSuccess) return e;
  const int need = cnt_dev ? nblocks : (cnt + QT_THREADS - 1) / QT_THREADS;
  k_qp_thread<<<need < nblocks ? need : nblocks, QT_THREADS, 0, st>>>(P, S, list, cnt, cnt_dev, wsbase, ws_per_inst, work_counter);
  return cudaGetLastError();
}

int tm_qp_thread_block() { return QT_THREADS; }
