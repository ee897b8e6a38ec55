// Internal (non-exported) helpers shared between the translation units of libomc.
#pragma once
int omc_sm_count();

// Prior / generic precision-matrix kinds understood by the small-matrix kernels.
//   0: scaled identity  (ptr may be null => 1.0, else ptr[0] is the diagonal value)
//   1: diagonal vector  (p entries)
//   2: dense row-major  (p x p)
enum OmcMatKind { OMC_MAT_EYE = 0, OMC_MAT_DIAG = 1, OMC_MAT_DENSE = 2 };

// dense_blocked.cu: blocked Cholesky (DMMA trailing update) form of omc_nn_dense_draw, p <= 512
#include "../../include/omc.h"
#include <cuda_runtime.h>
int omc_launch_blocked_draw(const omc_nn_dense_t& a, cudaStream_t st);
long long omc_blocked_workspace_doubles(int p);
// dense_warp.cu: one warp per chain (p <= 64, no probes); Q in registers, or left-looking with L in shared memory
// (32 < p <= 64)
int omc_launch_warp_draw(const omc_nn_dense_t& a, cudaStream_t st);
int omc_launch_left_draw(const omc_nn_dense_t& a, cudaStream_t st);
// trunc_scan.cu: truncated-prior Gibbs scan for 64 < p <= 512, one warp per chain, rows of G / P0 streamed
int omc_launch_trunc_stream(const omc_nn_dense_t& a, cudaStream_t st);
