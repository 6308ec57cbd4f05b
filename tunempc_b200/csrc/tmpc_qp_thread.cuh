// tmpc_qp_thread.cuh -- the thread-per-instance configuration shared by tmpc_qp_thread.cu (QP) and tmpc_fbjac_thread.cu
// (feedback Jacobian): tmpc_core.cuh compiled with TM_THREAD_MODE on the lane-interleaved workspace, CTA size and register budget.
#pragma once
#define TM_THREAD_MODE 1
#define TM_WS_STRIDE 32
#include <cuda_runtime.h>
#include "tmpc_core.cuh"

#define QT_THREADS 128
#if !defined(QT_MINB) && TMPC_NZ > 12
#define QT_MINB 2          /* wide stages (config #5: nz = 18): the per-stage blocks no longer fit 64 registers by far (32 KB of stack,
                              75 KB of spill loads); with 255 registers the 2^14-instance closed loop runs 25 % faster
                              (profiles/r02_summary.md, capture Q) -- at that batch the grid is one CTA per SM anyway */
#endif
#ifndef QT_MINB
#define QT_MINB 8          /* resident CTAs / SM the register allocation aims for: 64 registers, 1024 threads / SM.  The kernel
                              waits on its workspace (DRAM latency), so resident warps matter more than spills: measured
                              QP time per 2^20-instance step 991 / 894 / 818 / 860 / 894 ms at 4 / 6 / 8 / 12 / 16 CTAs
                              (profiles/r02g_summary.md) */
#endif
