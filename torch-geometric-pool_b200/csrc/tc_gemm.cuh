// tcgen05 / TMEM / TMA batched GEMM engine for sm_100a.
//
//   D[b] (M x N)  =  alpha * sum_{p < P}  A_p[b] (M x Kp) * B_p[b] (Kp x N)     (+ C[b] when accumulate)
//
// * operands arrive by TMA (cp.async.bulk.tensor, 128B swizzle) into a multi-stage shared-memory ring,
// * one elected thread issues tcgen05.mma (cta_group::1, M = 128) with the accumulator in TMEM
//   (double-buffered so the epilogue of tile t overlaps the main loop of tile t+1),
// * bf16 inputs are a single kind::f16 pass with both operands in shared memory (k_tc_gemm, 320 threads: warp 0 =
//   TMA producer, warp 1 = MMA issuer + TMEM allocator, warps 2-9 = epilogue),
// * fp32 inputs use the error-compensated 3xTF32 scheme (hi*hi + hi*lo + lo*hi, kind::tf32) with the A operand in
//   tensor memory (k_tc_gemm_ts): "split" warps write hi = rna_tf32(x) and lo = x - hi of the A tile into TMEM and of
//   the B tile into shared memory,
// * either operand may be K-major or MN-major in global memory (no transposes are materialised),
// * the epilogue reads TMEM with tcgen05.ld and writes fp32 or bf16 through swizzled shared-memory tiles and TMA
//   stores when the output is row-contiguous and 16-byte aligned (per-thread stores with arbitrary strides otherwise).
//
// One elected thread of the MMA warp runs the whole issuing loop.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace tgp {
namespace tc {

constexpr int kMaxPairs = 4;
constexpr int BM = 128;
constexpr int kStageRowBytes = 128;  // every smem tile row is one 128-byte swizzle line

struct OperandDesc {
  // how the MMA operand is stored in global memory, per batch item:
  //   K-major : rows = M (or N) extent, cols = K extent, cols contiguous
  //   MN-major: rows = K extent, cols = M (or N) extent, cols contiguous
  const void* ptr;
  int64_t batch_stride;  // elements
  int64_t row_stride;    // elements (cols are contiguous)
  int mn_major;          // 0 = K-major, 1 = MN-major
};

struct GemmProblem {
  int batch, M, N;
  int num_pairs;
  int kd[kMaxPairs];
  OperandDesc a[kMaxPairs], b[kMaxPairs];
  void* out;             // fp32 or bf16
  int64_t out_batch_stride, out_row_stride, out_col_stride;  // elements
  float alpha;
  int accumulate;        // D += existing out
  int out_bf16;
  int in_bf16;           // operand element type: 0 = fp32 (3xTF32), 1 = bf16
  int skip_lo_b_mask;    // bit p set: B_p is exactly representable in tf32 (lo pass skipped) -- optional hint
  // Optional fused epilogue of the dense backward (out must be [M, N] row-major, M = nodes, N = clusters):
  //   out[b, i, k] += c_den[b] * 2 * d[b, i] * S[b, i, k]  +  c_ent[b] * (-log(S + eps) - S / (S + eps))
  // with coef[b*4 + 0] = c_den, coef[b*4 + 2] = c_ent (the mincut-denominator and entropy-loss gradients).
  const void* ew_S;      // operand dtype, [batch, M, N]; nullptr = no element-wise term
  const float* ew_d;     // [batch, M]
  const float* ew_coef;  // [batch, 4]
  float ew_eps;
  const char* tag;       // optional launch name (string literal) shown by the per-kernel timing of bench.py
};

// Enqueue on `stream`.  Returns TGPB200_ERR_UNSUPPORTED when the shape violates the TMA / UMMA constraints
// (the caller then uses the shape-general FP32-pipe path).
int gemm(const GemmProblem& p, cudaStream_t stream);

// cuTensorMapEncodeTiled resolved through the runtime (no link-time dependency on libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn();
// 3-D tensor map over an operand stored [batch][rows][cols] (cols contiguous); box = {128 bytes of cols, box_rows, 1}.
// swizzle32 selects CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B (fp32 MN-major operands), else SWIZZLE_128B.
bool make_map_3d(CUtensorMap* map, const void* ptr, bool bf16, int64_t batch, int64_t rows, int64_t cols,
                 int64_t row_stride, int64_t batch_stride, int box_rows, bool swizzle32);
// 4-D "blocked" map of the same operand for MN-major tiles: dims {128 B of cols, rows, column blocks, batch};
// box {128 B, box_rows, box_blocks, 1} lands in shared memory block after block ([block][row][128 B]), i.e. the
// canonical UMMA MN-major layout, with ONE TMA instruction per tile.  cols must be a multiple of the block width.
bool make_map_blocked(CUtensorMap* map, const void* ptr, bool bf16, int64_t batch, int64_t rows, int64_t cols,
                      int64_t row_stride, int64_t batch_stride, int box_rows, int box_blocks, bool swizzle32);
// Operand [batch][rows][cols] (cols contiguous) of the engine.  K-major: rows = MN extent, cols = K extent, box
// {128 B of K, box_mn, 1}, 128B swizzle.  MN-major: rows = K extent, cols = MN extent, box {128 B of MN, 32 k-rows, 1}
// (one load per 128-byte block of the MN extent; fp32 uses the 32-byte-atom swizzle).
bool make_operand_map(CUtensorMap* map, const OperandDesc& op, bool bf16, int batch, int mn_extent, int k_extent,
                      int box_mn);
// fp32 MN-major operand as ONE unswizzled box [32 k-rows][128 MN columns] (read by the split warps only)
bool make_operand_map_mn_plain(CUtensorMap* map, const OperandDesc& op, int batch, int mn_extent, int k_extent);
int device_sm_count();
bool gemm_supported(const GemmProblem& p);

}  // namespace tc
}  // namespace tgp
