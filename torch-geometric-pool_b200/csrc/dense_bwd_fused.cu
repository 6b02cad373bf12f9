// Fused dense-pooling backward, fp32 (3xTF32): ONE launch per batch instead of three engine launches.
//
//   W  = A S                                              (never leaves the SM: accumulated in TMEM, split into hi / lo
//                                                          in registers and fed back as the A operand of the next MMA)
//   dS = X Gx^T + T^T Graw + S P + W Graw^T (+ element-wise loss terms)          [N, K]
//   dX = S Gx                                                                    [N, F]
//
// (math: SURVEY Appendix B; reference autograd of tgp/connect/dense_conn.py:112-122 and tgp/utils/losses.py:39-123;
//  Graw = d loss / d (S^T A S), P = d loss / d (S^T S) and the per-graph coefficients come from k_graph_bwd.)
//
// Work item = (graph, 128-row block of nodes).  Per item the MMA warp runs a fixed chain of "pairs" (A_p, B_p), each a
// run of 32-wide k-blocks through the same shared-memory stage ring / TMEM operand ring as the fp32 engine
// (tc_gemm.cu, k_tc_gemm_ts):
//   pair 0          A rows x S                -> W accumulator          (contraction over all N nodes)
//   pair 1          X rows x Gx^T             -> dS accumulator (first)
//   pair 2          T^T rows x Graw           -> dS
//   pair 3          S rows x P                -> dS                     (only with auxiliary losses)
//   pair 4          W (from TMEM) x Graw^T    -> dS
//   pair 5, 6       S rows x Gx[:, 64 j ..]   -> dX accumulators (one per 64 feature columns)
// The dS / dX accumulators are single-buffered: the epilogue of item i drains them while pair 0 of item i+1 (40 % of an
// item's MMA work) only touches the W accumulator.
//
// Tensor memory (512 columns): W [0, 64) | dS [64, 128) | dX [128, 256) | operand ring: FOUR slots of 64 columns
// (two split groups: a slot is only reused after the MMAs that read it have retired, a round trip the split warps
// must not wait for).  Shared memory: 5 stages x 32 KB | epilogue staging 32 KB | S rows of the element-wise terms 32 KB.
// Warp roles (448 threads): 0 TMA, 1 MMA (one elected thread runs the issue loop), 2-9 two split groups of four
// warps, 10-13 epilogue (element-wise terms prefetched with cp.async, double-buffered TMA stores).
#include <stdlib.h>
#include <string.h>

#include "dense.cuh"
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace tgp {
namespace tc {

namespace {

constexpr int kPairs = 7;
constexpr int kGroups = 2;                 // split groups (k-block kc goes to group kc % kGroups)
// TMEM operand ring: the slot of k-block kc is kc % kSlots.  A slot is recycled when the MMAs that read it have
// RETIRED (tcgen05.commit -> mbarrier -> the split warps' wait): with as many slots as split groups that round trip
// (~1.8 k cycles, measured with every stage of the pipeline emptied) bounds the kernel at one k-block per
// ~900 cycles whatever the k-block contains.  With more slots than groups the split warps never wait for it.
constexpr int kSlots = 4;
static_assert(kSlots % kGroups == 0, "every operand slot must belong to ONE split group (its waiters see every phase)");
// 4 epilogue warps (one per TMEM lane quadrant) keep the CTA at 448 threads: registers are allocated per 128 threads, so
// 576 threads are budgeted as 640 (96 registers per thread, spills inside the pipeline loops) while 448 get 128
// registers and no spill.
constexpr int kEpiW = 4;
constexpr int kThreadsBwd = 64 + kGroups * 128 + kEpiW * 32;
constexpr int BK = 32, KSTEPS = 4;
constexpr int BNB = 64;                    // MMA N of every pair
constexpr uint32_t kAccW = 64;             // width of the W and dS accumulators
constexpr uint32_t kColW = 0, kColS = kAccW, kColX = 2 * kAccW, kColRing = 2 * kAccW + 128, kRing = 64;
static_assert(kColRing + kSlots * kRing <= 512, "tensor memory budget");
constexpr uint32_t kABytes = BM * kStageRowBytes, kBBytes = BNB * kStageRowBytes;
constexpr uint32_t kStage = kABytes + 2 * kBBytes;  // [A raw | B hi | B lo] = 32 KB
constexpr uint32_t kEpiBufs = 2;          // staging tiles per epilogue warp (32 KB in total)
constexpr uint32_t kEpiBytes = kEpiW * kEpiBufs * 4096;
// rows of S for the element-wise terms of dS: 128 rows x 64 columns fp32, prefetched with cp.async while the item's MMAs run
constexpr uint32_t kHookBytes = BM * BNB * 4;

enum ASrc { kAKMajor = 0, kAMnPlain = 1, kATmem = 2 };

struct BwdParams {
  CUtensorMap map_a[kPairs], map_b[kPairs];
  int kd[kPairs], a_src[kPairs], b_mn[kPairs], b_n0[kPairs], first[kPairs];
  uint32_t acc_col[kPairs];
  int num_pairs;
  int batch, N, K, F;
  int m_tiles, num_items, stages;
  CUtensorMap map_ds, map_dx;
  const float* S;      // element-wise terms (nullptr: none)
  const float* d;
  const float* coef;
  const float* uv;     // [B, 2, K]: DMoN term d_i u_k + v_k of dS (nullptr: none)
  float eps;
};

__global__ void __launch_bounds__(kThreadsBwd, 1) k_dense_bwd_fused(const __grid_constant__ BwdParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int stages = P.stages;
  // [stages][kStage] | epilogue staging | S rows of the element-wise terms | barriers
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)kStage * stages + kEpiBytes + kHookBytes);
  const uint32_t bar_base = smem_u32(bars);
  auto bar_full = [&](int s) { return bar_base + 8u * s; };
  auto bar_lo = [&](int s) { return bar_base + 8u * (stages + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto bar_tfree = [&](int g) { return bar_base + 8u * (3 * stages + g); };
  const uint32_t bar_wfull = bar_base + 8u * (3 * stages + kSlots), bar_tfull = bar_wfull + 8u, bar_tempty = bar_wfull + 16u;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * stages + kSlots + 3);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_lo(s), 4);  // one arrival per split warp of the group (after __syncwarp), not one per thread
      mbar_init(bar_empty(s), 1);
    }
    for (int g = 0; g < kSlots; ++g) mbar_init(bar_tfree(g), 1);
    mbar_init(bar_wfull, 1);
    mbar_init(bar_tfull, 1);
    mbar_init(bar_tempty, kEpiW);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // (k-block counts come from the kernel parameters each time: a dynamically indexed local array lives in local
  //  memory, and with 227 KB of the L1 carved out as shared memory those loads miss to L2 inside the hot loops)

  if (warp == 0) {
    // ===================== TMA producer =====================
    int s = 0;
    uint32_t ph = 0;
    for (int item = blockIdx.x; item < P.num_items; item += gridDim.x) {
      const int mt = item % P.m_tiles, b = item / P.m_tiles;
      const int m0 = mt * BM;
      for (int p = 0; p < P.num_pairs; ++p) {
        const int src = P.a_src[p];
        for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb) {
          mbar_wait(bar_empty(s), ph ^ 1);
          const uint32_t sa = smem_base + (uint32_t)s * kStage, sb = sa + kABytes;
          const int k0 = kb * BK;
          if (elect_one()) {
            mbar_arrive_expect_tx(bar_full(s), (src != kATmem ? kABytes : 0u) + kBBytes);
            if (src == kAMnPlain) tma_load_3d(sa, &P.map_a[p], bar_full(s), m0, k0, b);      // [32 k][128 m], no swizzle
            else if (src == kAKMajor) tma_load_3d(sa, &P.map_a[p], bar_full(s), k0, m0, b);  // [128 m][32 k], 128B swizzle
            if (P.b_mn[p]) {
              for (int blk = 0; blk < BNB / 32; ++blk)
                tma_load_3d(sb + blk * (BK * kStageRowBytes), &P.map_b[p], bar_full(s), P.b_n0[p] + blk * 32, k0, b);
            } else {
              tma_load_3d(sb, &P.map_b[p], bar_full(s), k0, P.b_n0[p], b);
            }
          }
          __syncwarp();
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: ONE elected thread runs the whole loop =====================
    // (electing per k-block and reconverging the warp afterwards costs ~150 cycles per iteration of the issue loop:
    //  benchmarks/mma_rate.cu, k_loop modes 0 / 1)
    const uint32_t tm = __shfl_sync(kFull, tmem_base, 0);
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0, kc = 0;
      int it = 0;
      for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
        for (int p = 0; p < P.num_pairs; ++p) {
          if (p == 1) {  // first pair that writes the dS / dX accumulators: the previous item's epilogue has drained them
            mbar_wait(bar_tempty, ((uint32_t)it & 1u) ^ 1u);
            tc_fence_after();
          }
          const uint32_t d_tmem = tm + P.acc_col[p];
          const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)P.b_mn[p] << 16) |
                                 ((uint32_t)(BNB >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
          const uint32_t b_lbo = P.b_mn[p] ? BK * kStageRowBytes : 16;
          const uint32_t b_step = P.b_mn[p] ? 8 * kStageRowBytes : 32;
          const uint64_t desc_b0 = make_desc(smem_base, b_lbo, P.b_mn[p] ? 512 : 1024, P.b_mn[p] ? 1 : 2);
          uint32_t accum = P.first[p] ? 0u : 1u;
          for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb, ++kc) {
            mbar_wait(bar_lo(s), ph);
            tc_fence_after();
            const uint32_t ts = kc % (uint32_t)kSlots;
            const uint32_t a_stage = tm + kColRing + ts * kRing;
            const uint64_t db0 = desc_b0 + (uint64_t)(((uint32_t)s * kStage + kABytes) >> 4);
#pragma unroll
            for (int kk = 0; kk < KSTEPS; ++kk) {
              const uint64_t db = db0 + (uint64_t)(kk * (b_step >> 4)), db_lo = db + (kBBytes >> 4);
              const uint32_t a_hi = a_stage + (uint32_t)(kk * 16), a_lo = a_hi + 8;
              umma_ts_tf32(d_tmem, a_lo, db, idesc, kk == 0 ? accum : 1u);
              umma_ts_tf32(d_tmem, a_hi, db_lo, idesc, 1u);
              umma_ts_tf32(d_tmem, a_hi, db, idesc, 1u);
            }
            umma_commit(bar_empty(s));
            umma_commit(bar_tfree(ts));
            accum = 1;
            if (++s == stages) { s = 0; ph ^= 1; }
          }
          if (p == 0) umma_commit(bar_wfull);  // W complete: the split warps may read it back
        }
        umma_commit(bar_tfull);
      }
    }
    __syncwarp();
  } else if (warp < 2 + kGroups * 4) {
    // ===================== split: B hi / lo in shared memory, A hi / lo into the TMEM ring =====================
    const int grp = (warp - 2) >> 2;
    const int t = (threadIdx.x - 64) & 127;
    const int q = warp & 3;             // TMEM lane quadrant of this warp
    const int m_local = q * 32 + lane;  // row of the tile this thread stages
    int s = 0;
    uint32_t ph = 0, kc = 0;
    int it = 0;
    for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
      for (int p = 0; p < P.num_pairs; ++p) {
        const int src = P.a_src[p];
        for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb, ++kc) {
          if ((int)(kc % (uint32_t)kGroups) != grp) {  // another group's k-block
            // The group still OBSERVES the phase of a k-block it skips: with an odd number of stages a stage alternates
            // between the groups, and a parity wait that has missed one completed phase of its barrier passes at once --
            // before the data of the awaited phase has landed (seen as a hang with 3 stages).
            mbar_wait(bar_full(s), ph);
            if (++s == stages) { s = 0; ph ^= 1; }
            continue;
          }
          mbar_wait(bar_full(s), ph);
          const uint32_t sa = smem_base + (uint32_t)s * kStage, sb = sa + kABytes;
          // B: hi in place, lo behind it
          for (uint32_t ch = t; ch < kBBytes / 16; ch += 128) {
            const float4 v = lds128(sb + ch * 16);
            float4 h, l;
            h.x = rna_tf32(v.x), h.y = rna_tf32(v.y), h.z = rna_tf32(v.z), h.w = rna_tf32(v.w);
            l.x = v.x - h.x, l.y = v.y - h.y, l.z = v.z - h.z, l.w = v.w - h.w;
            sts128(sb + ch * 16, h);
            sts128(sb + kBBytes + ch * 16, l);
          }
          fence_proxy_async();
          // A: this thread's row, 32 k values
          float x[32];
          if (src == kATmem) {
            mbar_wait(bar_wfull, (uint32_t)it & 1u);
            tc_fence_after();
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + kColW + (uint32_t)(kb * BK), x);
          } else if (src == kAMnPlain) {
#pragma unroll
            for (int k = 0; k < 32; ++k) x[k] = lds32(sa + (uint32_t)k * (BM * 4) + (uint32_t)m_local * 4);
          } else {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float4 v = lds128(sa + (uint32_t)m_local * kStageRowBytes + (uint32_t)((c ^ (m_local & 7)) << 4));
              x[4 * c] = v.x, x[4 * c + 1] = v.y, x[4 * c + 2] = v.z, x[4 * c + 3] = v.w;
            }
          }
          const uint32_t slot = kc % (uint32_t)kSlots;
          mbar_wait(bar_tfree(slot), ((kc / (uint32_t)kSlots) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t a_stage = tmem_base + ((uint32_t)(q * 32) << 16) + kColRing + slot * kRing;
#pragma unroll
          for (int kk = 0; kk < KSTEPS; ++kk) {
            float hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              hi[i] = rna_tf32(x[kk * 8 + i]);
              lo[i] = x[kk * 8 + i] - hi[i];
            }
            tmem_st16(a_stage + (uint32_t)(kk * 16), hi, lo);
          }
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_lo(s));  // 128 per-thread arrivals on one barrier word serialise
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue: dS (+ element-wise terms) and dX through TMA stores =====================
    const int quad = warp & 3;
    const int ew = warp - 2 - kGroups * 4;   // 0 .. 3
    const uint32_t stg0 = smem_base + (uint32_t)kStage * stages + (uint32_t)ew * kEpiBufs * 4096u;
    uint32_t n_stored = 0;
    const uint32_t hook0 = smem_base + (uint32_t)kStage * stages + kEpiBytes;
    const int n_chunks = 2 + (P.F + 31) / 32;
    int it = 0;
    for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
      const int mt = item % P.m_tiles, b = item / P.m_tiles;
      const int m_base = mt * BM + quad * 32;
      const int m = m_base + lane;
      // Element-wise gradient terms of dS (mincut denominator 2 c_den d_i S, entropy loss): this thread's row of S is
      // fetched NOW, asynchronously into shared memory, so that its latency sits behind the item's MMAs instead of in
      // the drain (loading it per chunk after the accumulators were ready cost 21 us of the 115 us kernel).
      float dd = 0.f, c_ent = 0.f, di = 0.f;
      bool hook = false;
      const uint32_t hrow = hook0 + (uint32_t)(quad * 32 + lane) * (BNB * 4);
      if (P.S != nullptr && m < P.N) {
        const float c_den = P.coef[b * 4 + 0];
        c_ent = P.coef[b * 4 + 2];
        hook = c_den != 0.f || c_ent != 0.f;
        if (hook) {
          dd = 2.f * c_den * P.d[(int64_t)b * P.N + m];
          const float* srow = P.S + ((int64_t)b * P.N + m) * P.K;
          for (int j = 0; j * 4 < P.K; ++j) cp_async16(hrow + (uint32_t)((j ^ (lane & 7)) << 4), srow + j * 4);
        }
        if (P.uv != nullptr) di = P.d[(int64_t)b * P.N + m];
      }
      cp_async_commit();
      mbar_wait(bar_tfull, (uint32_t)it & 1u);
      tc_fence_after();
      cp_async_wait_all();
      __syncwarp();
      for (int c = 0; c < n_chunks; ++c) {
        const bool is_ds = c < 2;
        const int n0 = is_ds ? c * 32 : (c - 2) * 32;
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (is_ds ? kColS : kColX) + (uint32_t)n0, v);
        if (m_base >= P.N || n0 >= (is_ds ? P.K : P.F)) continue;  // warp-uniform
        if (is_ds && hook) {
#pragma unroll
          for (int c4 = 0; c4 < 8; ++c4) {
            if (n0 + c4 * 4 < P.K) {  // K is a multiple of 4: whole 16-byte chunks
              const float4 t4 = lds128(hrow + (uint32_t)((((n0 >> 2) + c4) ^ (lane & 7)) << 4));
              const float sv[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                float add = dd * sv[j];
                if (c_ent != 0.f) add += c_ent * (-__logf(sv[j] + P.eps) - __fdividef(sv[j], sv[j] + P.eps));
                v[c4 * 4 + j] += add;
              }
            }
          }
        }
        if (is_ds && P.uv != nullptr) {  // DMoN: d_i u_k + v_k (per-graph vectors: every lane loads the same word)
          const float* ub = P.uv + (int64_t)b * 2 * P.K + n0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (n0 + j < P.K) v[j] += fmaf(di, __ldg(ub + j), __ldg(ub + P.K + j));
        }
        // two staging tiles per warp: the store of the previous chunk may still be reading the other one
        const uint32_t stg = stg0 + (n_stored % kEpiBufs) * 4096u;
        ++n_stored;
        if (lane == 0) tma_store_wait_read<kEpiBufs - 1>();
        __syncwarp();
        const uint32_t row = stg + (uint32_t)lane * 128u;
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4)
          sts128(row + (uint32_t)((c4 ^ (lane & 7)) << 4), make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]));
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(is_ds ? &P.map_ds : &P.map_dx, stg, n0, m_base, b);
          tma_store_commit();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty);
    }
    if (lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// row-major fp32 output [batch][rows][cols], box {32, 32, 1}, 128B swizzle (staged one row per lane)
bool make_out_map(CUtensorMap* map, float* ptr, int64_t batch, int64_t rows, int64_t cols) {
  EncodeTiledFn fn = encode_fn();
  if (!fn || ((uintptr_t)ptr & 15) || (cols % 4)) return false;
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)rows * cols * 4};
  cuuint32_t box[3] = {32, 32, 1}, estr[3] = {1, 1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

// fp32 only.  Graw / Pm: [B, K, K] from k_graph_bwd (Pm nullptr: no S P term); ew_*: element-wise terms (ew_S nullptr: none).
// Returns TGPB200_ERR_UNSUPPORTED outside the envelope (K <= 64, F <= 128, 16-byte aligned rows): the caller then runs
// the one-product-per-launch chain.
int dense_bwd_fused(const float* A, const float* S, const float* X, const float* Tt, const float* Gx, const float* Graw,
                    const float* Pm, int B, int N, int K, int F, const float* ew_S, const float* ew_d, const float* ew_coef,
                    const float* ew_uv, float eps, float* dS, float* dX, cudaStream_t stream) {
  {
    const char* e = getenv("TGPB200_BWD_FUSED");
    if (e && e[0] == '0') return TGPB200_ERR_UNSUPPORTED;
  }
  if (!A || !S || !X || !Tt || !Gx || !Graw || !dS || !dX || B <= 0) return TGPB200_ERR_UNSUPPORTED;
  if (K > BNB || F > 128 || (N % 4) || (K % 4) || (F % 4) || N < 1) return TGPB200_ERR_UNSUPPORTED;
  const uintptr_t al = (uintptr_t)A | (uintptr_t)S | (uintptr_t)X | (uintptr_t)Tt | (uintptr_t)Gx | (uintptr_t)Graw |
                       (uintptr_t)(Pm ? Pm : Graw);
  if (al & 15) return TGPB200_ERR_UNSUPPORTED;
  BwdParams P;
  memset(&P, 0, sizeof(P));
  P.batch = B, P.N = N, P.K = K, P.F = F;
  P.m_tiles = (N + BM - 1) / BM;
  P.num_items = B * P.m_tiles;
  const int64_t NN = (int64_t)N * N, NK = (int64_t)N * K, NF = (int64_t)N * F, KK = (int64_t)K * K, KF = (int64_t)K * F;
  int n = 0;
  bool ok = true;
  auto add = [&](int kd, int a_src, OperandDesc a, OperandDesc b, int b_n0, uint32_t acc, int first) {
    P.kd[n] = kd, P.a_src[n] = a_src, P.b_mn[n] = b.mn_major, P.b_n0[n] = b_n0, P.acc_col[n] = acc, P.first[n] = first;
    if (a_src == kAKMajor) ok = ok && make_operand_map(&P.map_a[n], a, false, B, N, kd, BM);
    else if (a_src == kAMnPlain) ok = ok && make_operand_map_mn_plain(&P.map_a[n], a, B, N, kd);
    // the N extent of a B operand is its full column / row count (b_n0 selects the 64-wide slice)
    ok = ok && make_operand_map(&P.map_b[n], b, false, B, b.mn_major ? (int)b.row_stride : (int)(b.batch_stride / b.row_stride), kd, BNB);
    ++n;
  };
  // pair 0: W = A S
  add(N, kAKMajor, OperandDesc{A, NN, N, 0}, OperandDesc{S, NK, K, 1}, 0, kColW, 1);
  // pair 1: dS = X Gx^T   (B = Gx [K rows][F], contraction over F: K-major)
  add(F, kAKMajor, OperandDesc{X, NF, F, 0}, OperandDesc{Gx, KF, F, 0}, 0, kColS, 1);
  // pair 2: dS += T^T Graw  (A = T [K][N]: node index contiguous -> MN-major; B = Graw [k1][k2]: MN-major)
  add(K, kAMnPlain, OperandDesc{Tt, NK, N, 1}, OperandDesc{Graw, KK, K, 1}, 0, kColS, 0);
  // pair 3: dS += S P
  if (Pm) add(K, kAKMajor, OperandDesc{S, NK, K, 0}, OperandDesc{Pm, KK, K, 1}, 0, kColS, 0);
  // pair 4: dS += W Graw^T  (A from the W accumulator; B = Graw [k2 rows][k1]: K-major)
  add(K, kATmem, OperandDesc{nullptr, 0, 0, 0}, OperandDesc{Graw, KK, K, 0}, 0, kColS, 0);
  // pairs 5..: dX[:, 64 j .. 64 j + 64) = S Gx[:, 64 j ..]   (B = Gx [K][F]: MN-major)
  for (int j = 0; j * BNB < F; ++j)
    add(K, kAKMajor, OperandDesc{S, NK, K, 0}, OperandDesc{Gx, KF, F, 1}, j * BNB, kColX + (uint32_t)(j * BNB), 1);
  if (!ok) return TGPB200_ERR_UNSUPPORTED;
  P.num_pairs = n;
  if (!make_out_map(&P.map_ds, dS, B, N, K) || !make_out_map(&P.map_dx, dX, B, N, F)) return TGPB200_ERR_UNSUPPORTED;
  P.S = ew_S, P.d = ew_d, P.coef = ew_coef, P.uv = ew_S ? ew_uv : nullptr, P.eps = eps;
  P.stages = 5;
  static bool attr_set = false;
  if (!attr_set) {
    attr_set = true;
    cudaFuncSetAttribute(k_dense_bwd_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  }
  const size_t smem = (size_t)kStage * P.stages + kEpiBytes + kHookBytes + (3 * P.stages + kSlots + 4) * 8 + 16 + 1024;
  const int sms = device_sm_count();
  const int grid = P.num_items < sms ? P.num_items : sms;
  launch("k_dense_bwd_fused", k_dense_bwd_fused, grid, kThreadsBwd, smem, stream, P);
  return launch_status();
}

}  // namespace tc
}  // namespace tgp
