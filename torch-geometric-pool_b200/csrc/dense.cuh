// Shared declarations of the dense (MinCut / DiffPool) path.
#pragma once
#include <limits.h>

#include "common.cuh"

namespace tgp {
namespace tc {
// dense_fused.cu: one pass over A, X, S per graph -> Tt = A^T S, X_pool = S^T X, M = S^T S and the row statistics.
int dense_fwd_fused(const void* A, const void* S, const void* X, int B, int N, int K, int F, bool bf16, float eps,
                    void* Tt, void* Xp, float* Mm, float* d, float* ss, float* a2, float* ent, cudaStream_t stream);
// dense_fused_ts.cu: the fp32 form with the M-side MMA operand staged in tensor memory (less shared-memory traffic).
int dense_fwd_fused_ts(const float* A, const float* S, const float* X, int B, int N, int K, int F, float eps, float* Tt,
                       float* Xp, float* Mm, float* d, float* ss, float* a2, float* ent, cudaStream_t stream);
// dense_bwd_fused.cu: fp32 backward in one launch -- W = A S stays in tensor memory and feeds dS; dX from the same pass.
int dense_bwd_fused(const float* A, const float* S, const float* X, const float* Tt, const float* Gx, const float* Graw,
                    const float* Pm, int B, int N, int K, int F, const float* ew_S, const float* ew_d, const float* ew_coef,
                    const float* ew_uv, float eps, float* dS, float* dX, cudaStream_t stream);
}  // namespace tc

// A GEMM operand as stored in memory (per batch item, cols contiguous):
//   K-major : [MN extent rows][K extent cols];   MN-major: [K extent rows][MN extent cols]
struct Mat {
  const void* ptr;
  int64_t bs, rs;
  int mn;
};

struct EwHook {  // fused element-wise terms of dS (tc::GemmProblem::ew_*); *applied is set when the engine took it
  const void* S = nullptr;
  const float* d = nullptr;
  const float* coef = nullptr;
  float eps = 0.f;
  bool* applied = nullptr;
};

// dense_pool.cu: D[b] (M x N) = sum_p A_p B_p (+ D[b] when accumulate), written with (row, col) strides: the tcgen05
// engine (3xTF32 for fp32 operands, one bf16 pass) when the layout satisfies the TMA constraints, the FP32-pipe
// batched GEMM otherwise.  Instantiated for <float, float>, <bf16, float> and <bf16, bf16>.
template <typename T, typename TC>
int mm(int batch, int M, int N, int npairs, const int* kd, const Mat* A, const Mat* Bm, TC* out, int64_t obs,
       int64_t ors, int64_t ocs, cudaStream_t st, EwHook hook = EwHook(), const char* tag = nullptr,
       bool accumulate = false);
}  // namespace tgp
