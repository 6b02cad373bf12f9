// Fused dense-pooling forward, fp32 (3xTF32), with the MMA A operand in TENSOR MEMORY.
//
// Same contraction as dense_fused.cu ([A | X | S]^T S per graph, one pass over A, X, S, row statistics on the way),
// but the hi / lo halves of the M-side operand never go back to shared memory: the split warps read the TMA tile
// once, round / subtract in registers and store both halves with tcgen05.st into a ring of TMEM operand stages (one
// per split group); tcgen05.mma then takes A from TMEM and only the small N-side operand (S, hi / lo) from shared
// memory.
// The 3xTF32 kernels are bound by the shared-memory pipe (dense_fused.cu moves ~260 KB through it per 28 KB of
// HBM data: TMA write, split read, hi + lo write back, three operand fetches); this form moves ~110 KB.
//
//   shared-memory stage (per 16-node k-block): [16][N] A | [16][F] X | [16][K] S  (row-major, NOT swizzled: nobody
//     but the split warps reads them)  |  S again as 128-byte column blocks with the 32-byte-atom swizzle (the MN-major
//     B operand, hi in place) | its lo half
//   tensor memory: [0, G*BN) accumulators of the G = t_a + t_x + t_s M-tiles (single buffered),
//     then 2 stages x G tiles x 2 k-steps x (8 hi + 8 lo) columns of A operand (lane = M row, column = k)
//
// Roles: warp 0 TMA producer, warp 1 MMA issuer (one elected thread) + TMEM allocator, then kSplitGroups groups of
// kSplitWarps split / TMEM staging warps (warp w owns TMEM lanes 32 (w & 3) .., the warps of a quadrant take the
// M-tiles round robin; group g takes every kSplitGroups-th k-block), then kEpiWarps epilogue warps, which also
// accumulate the row statistics from the stage's row-major tiles while the main loop runs and drain the accumulators
// through transposed shared-memory tiles + TMA stores.
#include <stdlib.h>
#include <string.h>

#include "dense.cuh"
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace tgp {
namespace tc {

namespace {

constexpr int TBK = 16;                              // nodes per k-block
constexpr int kSBlock = TBK * kStageRowBytes;        // one swizzled 128-byte column block of S: 2 KB
#ifndef TGPB200_TS_SPLIT_WARPS
#define TGPB200_TS_SPLIT_WARPS 8
#endif
#ifndef TGPB200_TS_SPLIT_GROUPS
#define TGPB200_TS_SPLIT_GROUPS 2
#endif
// The split of one k-block is a latency chain (barrier wait, shared-memory reads, shuffles, proxy fence, TMEM stores
// and their wait): kSplitGroups groups of kSplitWarps warps each take every kSplitGroups-th k-block, so consecutive
// k-blocks are split concurrently (group g always fills TMEM operand stage g).
constexpr int kSplitGroups = TGPB200_TS_SPLIT_GROUPS;   // 1 or 2 (= TMEM operand stages)
constexpr int kSplitWarps = TGPB200_TS_SPLIT_WARPS;     // per group; multiple of 4: kSplitWarps / 4 warps per lane quadrant
constexpr int kSplitThreads = kSplitWarps * 32;         // per group
constexpr int kEpiWarps = 8;                            // two per TMEM lane quadrant, alternate 32-column chunks
constexpr int kTsThreads = 64 + kSplitGroups * kSplitThreads + kEpiWarps * 32;  // TMA, MMA, split groups, epilogue
constexpr int kTpr = kEpiWarps * 32 / 16;               // statistics (epilogue warps): threads per node row
constexpr int kACols = 32;                           // TMEM columns per (tile, k-block): 2 k-steps x (8 hi + 8 lo)

struct TsParams {
  CUtensorMap map_a, map_x, map_s;  // row-major boxes {extent, 16, 1}, no swizzle
  CUtensorMap map_sb;               // S as swizzled 128-byte column blocks (B operand)
  CUtensorMap map_ot, map_ox, map_om;  // outputs Tt / Xp / Mm as [B][K rows][extent], box {32, 32, 1} (TMA stores)
  int B, N, K, F;
  int BN;                  // MMA N (K rounded up to 16)
  int t_a, t_x, t_s, nb_s;
  int stages;
  uint32_t tmem_cols, stage_bytes, off_sb;
  float eps;
  float* Tt;               // [B, K, N]
  float* Xp;               // [B, K, F]
  float* Mm;               // [B, K, K]
  float *d, *ss, *a2, *ent;
};

__global__ void __launch_bounds__(kTsThreads, 1) k_dense_fwd_fused_ts(const __grid_constant__ TsParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int stages = P.stages;
  const uint32_t stage_bytes = P.stage_bytes;
  // barriers: full[stages] (TMA landed), ready[stages] (split done: B operand in smem + A operand in TMEM),
  // empty[stages] (MMAs of the stage retired), tfree[2] (TMEM A stage retired), tfull, tempty (accumulators)
  // [stages][stage_bytes] | epilogue staging: kEpiWarps x 4 KB | barriers | lo flags
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stage_bytes * stages + kEpiWarps * 4096);
  const uint32_t bar_base = smem_u32(bars);
  auto bar_full = [&](int s) { return bar_base + 8u * s; };
  auto bar_ready = [&](int s) { return bar_base + 8u * (stages + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto bar_tfree = [&](int t) { return bar_base + 8u * (3 * stages + t); };
  const uint32_t bar_tfull = bar_base + 8u * (3 * stages + 2), bar_tempty = bar_base + 8u * (3 * stages + 3);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * stages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);
  const int G = P.t_a + P.t_x + P.t_s;
  const int BN = P.BN;
  const int kblocks = (P.N + TBK - 1) / TBK;
  const uint32_t off_x = (uint32_t)TBK * P.N * 4, off_s = off_x + (uint32_t)TBK * P.F * 4, off_sb = P.off_sb;
  const uint32_t sb_bytes = (uint32_t)P.nb_s * kSBlock;
  const uint32_t a_cols0 = (uint32_t)(G * BN);  // first TMEM column of the A-operand ring

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_ready(s), kSplitThreads);
      mbar_init(bar_empty(s), 1 + kEpiWarps * 32);  // MMAs retired (commit) + statistics read (epilogue threads)
    }
    mbar_init(bar_tfree(0), 1);
    mbar_init(bar_tfree(1), 1);
    mbar_init(bar_tfull, 1);
    mbar_init(bar_tempty, kEpiWarps * 32);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), P.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer (whole warp; one elected lane issues) =====================
    {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx = (uint32_t)TBK * (P.N + P.F + P.K) * 4 + sb_bytes;
      for (int b = blockIdx.x; b < P.B; b += gridDim.x) {
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(bar_empty(s), ph ^ 1);
          const uint32_t dst = smem_base + (uint32_t)s * stage_bytes;
          const int k0 = kb * TBK;
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_full(s), tx);
            tma_load_3d(dst, &P.map_a, bar_full(s), 0, k0, b);
            tma_load_3d(dst + off_x, &P.map_x, bar_full(s), 0, k0, b);
            tma_load_3d(dst + off_s, &P.map_s, bar_full(s), 0, k0, b);
            for (int j = 0; j < P.nb_s; ++j) tma_load_3d(dst + off_sb + j * kSBlock, &P.map_sb, bar_full(s), j * 32, k0, b);
          }
          __syncwarp();
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: ONE elected thread runs the whole loop =====================
    // (electing per k-block and reconverging the warp afterwards costs ~150 cycles per iteration: mma_rate.cu, k_loop)
    // tf32 x tf32 -> f32, A from TMEM (K-major by construction), B MN-major, N = BN, M = 128
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) |
                           ((uint32_t)(BM >> 4) << 24);
    const uint64_t desc0 = make_desc(smem_base, kSBlock, 512, 1);  // 32-byte-atom swizzle, 4-row atoms
    const uint32_t tm = __shfl_sync(kFull, tmem_base, 0);
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      uint32_t kc = 0;
      int it = 0;
      for (int b = blockIdx.x; b < P.B; b += gridDim.x, ++it) {
        mbar_wait(bar_tempty, ((uint32_t)it & 1u) ^ 1u);
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++kc) {
          mbar_wait(bar_ready(s), ph);
          tc_fence_after();
          const uint32_t ts = kc & 1u;
          const uint32_t a_stage = tm + a_cols0 + ts * (uint32_t)(G * kACols);
          const uint64_t db0 = desc0 + (uint64_t)(((uint32_t)s * stage_bytes + off_sb) >> 4);
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            const uint64_t db = db0 + (uint64_t)(kk * ((8 * kStageRowBytes) >> 4)), db_lo = db + (sb_bytes >> 4);
            const uint32_t acc0 = (kb > 0 || kk > 0) ? 1u : 0u;
            for (int g = 0; g < G; ++g) {
              const uint32_t a_hi = a_stage + (uint32_t)(g * kACols + kk * 16), a_lo = a_hi + 8;
              const uint32_t dt = tm + (uint32_t)(g * BN);
              umma_ts_tf32(dt, a_lo, db, idesc, acc0);
              umma_ts_tf32(dt, a_hi, db_lo, idesc, 1u);
              umma_ts_tf32(dt, a_hi, db, idesc, 1u);
            }
          }
          umma_commit(bar_empty(s));    // the TMA producer may refill the shared-memory stage
          umma_commit(bar_tfree(ts));   // the split warps may overwrite the TMEM operand stage
          if (++s == stages) { s = 0; ph ^= 1; }
        }
        umma_commit(bar_tfull);
      }
    }
    __syncwarp();
  } else if (warp < 2 + kSplitGroups * kSplitWarps) {
    // ===================== split: statistics, B operand (smem), A operand (TMEM) =====================
    const int grp = (warp - 2) / kSplitWarps;              // which k-blocks this warp's group takes
    const int t = (threadIdx.x - 64) % kSplitThreads;      // thread index inside the group
    const int q = warp & 3;                                // TMEM lane quadrant of this warp
    const int half = ((warp - 2) % kSplitWarps) >> 2;      // which of the quadrant's warps inside the group
    int s = 0;
    uint32_t ph = 0, kc = 0;
    for (int b = blockIdx.x; b < P.B; b += gridDim.x) {
      for (int kb = 0; kb < kblocks; ++kb, ++kc) {
        if (kSplitGroups > 1 && (int)(kc % kSplitGroups) != grp) {  // another group's k-block
          // The group still OBSERVES the phase of a k-block it skips: with an odd number of stages a stage alternates
          // between the groups, and a parity wait that has missed one completed phase of its barrier passes at once --
          // before the data of the awaited phase has landed (seen as a hang with 3 stages).
          mbar_wait(bar_full(s), ph);
          if (++s == stages) { s = 0; ph ^= 1; }
          continue;
        }
        mbar_wait(bar_full(s), ph);
        const uint32_t base = smem_base + (uint32_t)s * stage_bytes;
        // ---- pass 1b: hi / lo of the B operand (swizzled S blocks), in place + next to it
        for (uint32_t ch = t; ch < (uint32_t)P.nb_s * 128; ch += kSplitThreads) {
          const uint32_t a = base + off_sb + ch * 16;
          const float4 v = lds128(a);
          float4 h, l;
          h.x = rna_tf32(v.x), h.y = rna_tf32(v.y), h.z = rna_tf32(v.z), h.w = rna_tf32(v.w);
          l.x = v.x - h.x, l.y = v.y - h.y, l.z = v.z - h.z, l.w = v.w - h.w;
          sts128(a, h);
          sts128(a + sb_bytes, l);
        }
        fence_proxy_async();
        // ---- pass 2: hi / lo of the M-side operand into the TMEM ring (lane = M row, 8 columns = 8 nodes)
        const uint32_t ts = kc & 1u;
        mbar_wait(bar_tfree(ts), ((kc >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t a_stage = tmem_base + ((uint32_t)(q * 32) << 16) + a_cols0 + ts * (uint32_t)(G * kACols);
        for (int g = half; g < G; g += kSplitWarps / 4) {
          const int seg = g < P.t_a ? 0 : (g < P.t_a + P.t_x ? 1 : 2);
          const int m = (seg == 0 ? g : (seg == 1 ? g - P.t_a : g - P.t_a - P.t_x)) * BM + q * 32 + lane;
          const int ext = seg == 0 ? P.N : (seg == 1 ? P.F : P.K);
          const uint32_t col0 = base + (seg == 0 ? 0u : (seg == 1 ? off_x : off_s)) + (uint32_t)m * 4;
          const uint32_t pitch = (uint32_t)ext * 4;
          const bool on = m < ext;
#pragma unroll
          for (int kk = 0; kk < 2; ++kk) {
            float x[8], hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = on ? lds32(col0 + (uint32_t)(kk * 8 + i) * pitch) : 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              hi[i] = rna_tf32(x[i]);
              lo[i] = x[i] - hi[i];
            }
            tmem_st16(a_stage + (uint32_t)(g * kACols + kk * 16), hi, lo);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(bar_ready(s));
        if (++s == stages) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (accumulators single-buffered) =====================
    const int quad = warp & 3;
    const int ew = warp - 2 - kSplitGroups * kSplitWarps;  // 0 .. kEpiWarps - 1
    const int e2 = (ew >> 2) & 1;                          // which of the quadrant's two epilogue warps
    const uint32_t stg = smem_base + (uint32_t)stage_bytes * stages + (uint32_t)ew * 4096u;  // this warp's staging tile
    const int t = threadIdx.x - (kTsThreads - kEpiWarps * 32);  // 0 .. 255
    const int r = t / kTpr, c16 = t % kTpr;
    int s = 0;
    uint32_t ph = 0;
    int it = 0;
    for (int b = blockIdx.x; b < P.B; b += gridDim.x, ++it) {
      // ---- row statistics of every k-block of the graph (these warps are otherwise idle during the main loop; on the
      //      split warps this pass was ~35 % of the work of the role that bounds the kernel)
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(bar_full(s), ph);
        const uint32_t base = smem_base + (uint32_t)s * stage_bytes;
        float sd = 0.f, sa2 = 0.f, s2 = 0.f, se = 0.f;
        const uint32_t ra = base + (uint32_t)r * P.N * 4;
        for (int col = c16 * 4; col < P.N; col += 4 * kTpr) {
          const float4 v = lds128(ra + col * 4);
          sd += (v.x + v.y) + (v.z + v.w);
          sa2 += fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
        }
        const uint32_t rs = base + off_s + (uint32_t)r * P.K * 4;
        for (int col = c16 * 4; col < P.K; col += 4 * kTpr) {
          const float4 v = lds128(rs + col * 4);
          s2 += fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
          se -= fmaf(v.x, __logf(v.x + P.eps),
                     fmaf(v.y, __logf(v.y + P.eps), fmaf(v.z, __logf(v.z + P.eps), v.w * __logf(v.w + P.eps))));
        }
#pragma unroll
        for (int o = 1; o < kTpr; o <<= 1) {
          sd += __shfl_xor_sync(kFull, sd, o);
          sa2 += __shfl_xor_sync(kFull, sa2, o);
          s2 += __shfl_xor_sync(kFull, s2, o);
          se += __shfl_xor_sync(kFull, se, o);
        }
        const int node = kb * TBK + r;
        if (c16 == 0 && node < P.N) {
          const int64_t o = (int64_t)b * P.N + node;
          P.d[o] = sd, P.a2[o] = sa2, P.ss[o] = s2, P.ent[o] = se;
        }
        mbar_arrive(bar_empty(s));  // this thread has read its share of the stage
        if (++s == stages) { s = 0; ph ^= 1; }
      }
      mbar_wait(bar_tfull, (uint32_t)it & 1u);
      tc_fence_after();
      int chunk = 0;
      for (int g = 0; g < G; ++g) {
        const int seg = g < P.t_a ? 0 : (g < P.t_a + P.t_x ? 1 : 2);
        const int m0 = (seg == 0 ? g : (seg == 1 ? g - P.t_a : g - P.t_a - P.t_x)) * BM + quad * 32;  // warp-uniform
        const int m_ext = seg == 0 ? P.N : (seg == 1 ? P.F : P.K);
        for (int c0 = 0; c0 < BN; c0 += 32, ++chunk) {
          if ((chunk & 1) != e2) continue;
          float v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(g * BN + c0), v);
          if (m0 >= m_ext || c0 >= P.K) continue;
          // Transposed tile through shared memory: accumulator column j becomes row c0 + j of the destination, the 32
          // lanes (rows of the MMA tile) its 32 contiguous elements -> conflict-free 128-byte rows, ONE TMA store per
          // chunk (1024 scalar global stores per graph kept the LSU busy for most of the 7 k-cycle epilogue bubble).
          if (lane == 0) tma_store_wait_read<0>();  // the previous store of this warp has read the staging tile
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 32; ++j) sts32(stg + (uint32_t)(j * 128 + lane * 4), __float_as_uint(v[j]));
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(seg == 0 ? &P.map_ot : (seg == 1 ? &P.map_ox : &P.map_om), stg, m0, c0, b);
            tma_store_commit();
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_tempty);
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, P.tmem_cols);
}

// row-major box {cols, 16 rows, 1 batch item}, fp32, no swizzle
bool make_map_rows(CUtensorMap* map, const void* ptr, int64_t batch, int64_t rows, int64_t cols) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)rows * cols * 4};
  cuuint32_t box[3] = {(cuuint32_t)cols, (cuuint32_t)TBK, 1}, estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// output [batch][rows][cols] fp32, box {32 cols, 32 rows, 1}, no swizzle (TMA stores of the transposed chunks)
bool make_map_out(CUtensorMap* map, const void* ptr, int64_t batch, int64_t rows, int64_t cols) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || ((uintptr_t)ptr & 15)) return false;
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)rows * cols * 4};
  cuuint32_t box[3] = {32, 32, 1}, estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

}  // namespace

// fp32 only.  Returns TGPB200_ERR_UNSUPPORTED when the shape does not fit (the caller then uses dense_fused.cu).
int dense_fwd_fused_ts(const float* A, const float* S, const float* X, int B, int N, int K, int F, float eps, float* Tt,
                       float* Xp, float* Mm, float* d, float* ss, float* a2, float* ent, cudaStream_t stream) {
  if (!A || !S || !X || B <= 0 || N <= 0 || K <= 0 || F <= 0) return TGPB200_ERR_UNSUPPORTED;
  if (N > 256 || F > 256 || K > 256 || (N % 4) || (K % 4) || (F % 4)) return TGPB200_ERR_UNSUPPORTED;  // one TMA box per row tile
  if (((uintptr_t)A | (uintptr_t)S | (uintptr_t)X) & 15) return TGPB200_ERR_UNSUPPORTED;
  TsParams P;
  memset(&P, 0, sizeof(P));
  P.B = B, P.N = N, P.K = K, P.F = F;
  P.BN = (K + 15) / 16 * 16;
  P.t_a = (N + BM - 1) / BM, P.t_x = (F + BM - 1) / BM, P.t_s = (K + BM - 1) / BM;
  P.nb_s = (K + 31) / 32;
  const int G = P.t_a + P.t_x + P.t_s;
  const int cols_needed = G * P.BN + 2 * G * kACols;
  if (cols_needed > 512 || P.nb_s * 32 < P.BN) return TGPB200_ERR_UNSUPPORTED;
  uint32_t cols = 32;
  while (cols < (uint32_t)cols_needed) cols <<= 1;
  P.tmem_cols = cols;
  const size_t rows_bytes = (size_t)TBK * (N + F + K) * 4;
  P.off_sb = (uint32_t)((rows_bytes + 1023) / 1024 * 1024);
  P.stage_bytes = P.off_sb + 2u * (uint32_t)P.nb_s * kSBlock;
  int stages = (int)((size_t)(216 * 1024 - kEpiWarps * 4096) / P.stage_bytes);
  if (stages > 8) stages = 8;
  if (stages < 2) return TGPB200_ERR_UNSUPPORTED;
  P.stages = stages;
  P.eps = eps;
  P.Tt = Tt, P.Xp = Xp, P.Mm = Mm, P.d = d, P.ss = ss, P.a2 = a2, P.ent = ent;
  if (!make_map_rows(&P.map_a, A, B, N, N) || !make_map_rows(&P.map_x, X, B, N, F) || !make_map_rows(&P.map_s, S, B, N, K))
    return TGPB200_ERR_UNSUPPORTED;
  if (!make_map_3d(&P.map_sb, S, false, B, N, K, K, (int64_t)N * K, TBK, true)) return TGPB200_ERR_UNSUPPORTED;
  if (!make_map_out(&P.map_ot, Tt, B, K, N) || !make_map_out(&P.map_ox, Xp, B, K, F) || !make_map_out(&P.map_om, Mm, B, K, K))
    return TGPB200_ERR_UNSUPPORTED;
  static bool attr_set = false;
  if (!attr_set) {
    attr_set = true;
    cudaFuncSetAttribute(k_dense_fwd_fused_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  }
  const size_t smem = (size_t)P.stage_bytes * stages + kEpiWarps * 4096 + (3 * stages + 4) * 8 + 16 + 1024;
  if (smem > 227 * 1024) return TGPB200_ERR_UNSUPPORTED;
  const int sms = device_sm_count();
  const int grid = B < sms ? B : sms;
  launch("k_dense_fwd_fused_ts", k_dense_fwd_fused_ts, grid, kTsThreads, smem, stream, P);
  return launch_status();
}

}  // namespace tc
}  // namespace tgp
