// Fused dense-pooling forward main kernel (tcgen05 / TMEM / TMA):  one pass over A, X and S per graph.
//
//   For every graph b, with the node index i as the contraction dimension, the concatenation
//   C[i, :] = [ A[i, :] | X[i, :] | S[i, :] ]  (N + F + K columns) is contracted against S:
//        T    = S^T A   [K, N]     (computed as A^T S, stored transposed; kept for S^T A S and the backward)
//        Xp^T = X^T S   [F, K]  -> written transposed as X_pool [K, F]      (tgp/reduce/base_reduce.py:158-161)
//        M    = S^T S   [K, K]                                              (tgp/utils/losses.py:118)
//   while the tiles are in shared memory the "split" warps also produce the row statistics
//        d_i = sum_j A_ij,  a2_i = sum_j A_ij^2,  ss_i = sum_k S_ik^2,  ent_i = -sum_k S_ik log(S_ik + eps)
//   (mincut denominator, link-loss norm, entropy loss), so A, X and S are read from HBM exactly once.
//
// Every operand is MN-major (the contraction index i is the row of all three tensors): tiles are [BK = 16 nodes]
// x [128-byte column blocks]; fp32 runs as 3xTF32 (hi/lo split in place, 32-byte-atom swizzle), bf16 as one pass.
// Roles (320 threads): warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 split + statistics, warps 6-9 epilogue.
#include <string.h>

#include "dense.cuh"
#include <type_traits>

#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace tgp {
namespace tc {

constexpr int FBK = 16;  // nodes per k-block
constexpr int kBlockBytes = FBK * kStageRowBytes;  // one 128-byte column block of a k-block: 2 KB

struct FusedParams {
  CUtensorMap map_a, map_x, map_s;
  int B, N, K, F;
  int BN;                 // MMA N (K rounded up to 16)
  int nb_a, nb_x, nb_s;   // 128-byte column blocks per segment
  int t_a, t_x, t_s;      // 128-row MMA tiles per segment
  int stages, acc_bufs, blocked;
  int concat;             // fp32: accumulators 2 BN wide, hi_a x [hi_s | lo_s] as ONE MMA (lo of S right behind S)
  uint32_t tmem_cols;
  float eps;
  // 16-byte aligned: the output pointers are fetched in 16-byte-aligned pairs (ss / a2 with one 128-bit load)
  alignas(16) void* Tt;   // [B, K, N]  operand dtype: T = S^T A
  void* Xp;               // [B, K, F]  operand dtype
  float* Mm;              // [B, K, K]
  float *d, *ss, *a2, *ent;  // [B, N]
};

template <bool kF32>
__global__ void __launch_bounds__(320, 1) k_dense_fwd_fused(const __grid_constant__ FusedParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int ES = kF32 ? 4 : 2;
  constexpr int EPB = kStageRowBytes / ES;  // columns per 128-byte block
  constexpr int UMMA_K = 32 / ES;
  constexpr int KSTEPS = FBK / UMMA_K;      // 2 (tf32) or 1 (bf16)
  using T = typename std::conditional<kF32, float, __nv_bfloat16>::type;

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int nb = P.nb_a + P.nb_x + P.nb_s;
  const uint32_t raw_bytes = (uint32_t)nb * kBlockBytes;
  const uint32_t stage_bytes = raw_bytes * (kF32 ? 2 : 1);
  const int stages = P.stages;
  // +4 blocks of slack: a partial last MMA tile reads (and ignores) up to 3 blocks past its segment
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stage_bytes * stages + 4 * kBlockBytes);
  const uint32_t bar_base = smem_u32(bars);
  auto bar_full = [&](int s) { return bar_base + 8u * s; };
  auto bar_lo = [&](int s) { return bar_base + 8u * (stages + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto bar_tfull = [&](int i) { return bar_base + 8u * (3 * stages + i); };
  auto bar_tempty = [&](int i) { return bar_base + 8u * (3 * stages + 2 + i); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * stages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);
  const int G = P.t_a + P.t_x + P.t_s;  // accumulator tiles of one graph
  const int BN = P.BN;
  const int kblocks = (P.N + FBK - 1) / FBK;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_lo(s), 128);
      mbar_init(bar_empty(s), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull(i), 1);
      mbar_init(bar_tempty(i), 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), P.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int b = blockIdx.x; b < P.B; b += gridDim.x) {
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(bar_empty(s), ph ^ 1);
          uint32_t dst = smem_base + (uint32_t)s * stage_bytes;
          mbar_arrive_expect_tx(bar_full(s), raw_bytes);
          const int k0 = kb * FBK;
          if (P.blocked) {  // one TMA instruction per segment (4-D blocked maps)
            tma_load_4d(dst, &P.map_a, bar_full(s), 0, k0, 0, b);
            tma_load_4d(dst + P.nb_a * kBlockBytes, &P.map_x, bar_full(s), 0, k0, 0, b);
            tma_load_4d(dst + (P.nb_a + P.nb_x) * kBlockBytes, &P.map_s, bar_full(s), 0, k0, 0, b);
          } else {
            for (int j = 0; j < P.nb_a; ++j, dst += kBlockBytes) tma_load_3d(dst, &P.map_a, bar_full(s), j * EPB, k0, b);
            for (int j = 0; j < P.nb_x; ++j, dst += kBlockBytes) tma_load_3d(dst, &P.map_x, bar_full(s), j * EPB, k0, b);
            for (int j = 0; j < P.nb_s; ++j, dst += kBlockBytes) tma_load_3d(dst, &P.map_s, bar_full(s), j * EPB, k0, b);
          }
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp; tcgen05 instructions on one elected lane) =====================
    {
      const uint32_t tm = __shfl_sync(kFull, tmem_base, 0);
      const uint32_t fmt = kF32 ? 2u : 1u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)(BM >> 4) << 24);
      const uint32_t sbo = kF32 ? 512 : 1024, lt = kF32 ? 1 : 2;
      // The issuing thread is the serial bottleneck of this kernel, so descriptors are built once: only the
      // 14-bit start-address field (16-byte units) changes, and it never carries out of its field (smem < 256 KB).
      const uint64_t desc0 = make_desc(smem_base, kBlockBytes, sbo, lt);
      uint32_t tile_off[8];  // first column block of MMA tile g, in 16-byte units
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        int blk = g < P.t_a ? g * (BM / EPB)
                            : (g < P.t_a + P.t_x ? P.nb_a + (g - P.t_a) * (BM / EPB)
                                                 : P.nb_a + P.nb_x + (g - P.t_a - P.t_x) * (BM / EPB));
        tile_off[g] = (uint32_t)blk * (kBlockBytes >> 4);
      }
      const uint32_t b_off = (uint32_t)(P.nb_a + P.nb_x) * (kBlockBytes >> 4);
      const uint32_t lo_off = raw_bytes >> 4, stage_off = stage_bytes >> 4;
      // concat mode: stage = [A | X | S | S lo | A lo | X lo]
      const uint32_t s_lo_off = (uint32_t)P.nb_s * (kBlockBytes >> 4), ax_lo_off = lo_off + s_lo_off;
      const uint32_t idesc2 = (idesc & ~(0x3fu << 17)) | ((uint32_t)((2 * BN) >> 3) << 17);
      const int accw = P.concat ? 2 * BN : BN;  // accumulator columns per tile
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int b = blockIdx.x; b < P.B; b += gridDim.x, ++it) {
        const int ab = P.acc_bufs == 2 ? (it & 1) : 0;
        const uint32_t aph = P.acc_bufs == 2 ? ((uint32_t)(it >> 1) & 1u) : ((uint32_t)it & 1u);
        mbar_wait(bar_tempty(ab), aph ^ 1);
        tc_fence_after();
        const uint32_t d0 = tm + (uint32_t)(ab * G * accw);
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(bar_full(s), ph);
          mbar_wait(bar_lo(s), ph);
          tc_fence_after();
          const uint64_t dst = desc0 + (uint64_t)((uint32_t)s * stage_off);
          if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < KSTEPS; ++kk) {
            const uint64_t dk = dst + (uint64_t)(kk * ((UMMA_K * kStageRowBytes) >> 4));
            const uint64_t db = dk + b_off, db_lo = db + lo_off;
            const uint32_t acc0 = (kb > 0 || kk > 0) ? 1u : 0u;
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              if (g < G) {
                const uint64_t da = dk + tile_off[g];
                const uint32_t dt = d0 + (uint32_t)(g * accw);
                if (kF32 && P.concat) {
                  // two instructions per k-step: an MMA costs ~43 + N/2 cycles (benchmarks/mma_rate.cu), so one
                  // N = 2 BN instruction is cheaper than two N = BN ones
                  umma<true>(dt, da, db, idesc2, acc0);  // hi x [hi_s | lo_s]
                  umma<true>(dt, da + (g >= P.t_a + P.t_x ? s_lo_off : ax_lo_off), db, idesc, 1u);  // lo x hi_s
                } else if (kF32) {
                  umma<true>(dt, da + lo_off, db, idesc, acc0);
                  umma<true>(dt, da, db_lo, idesc, 1u);
                  umma<true>(dt, da, db, idesc, 1u);
                } else {
                  umma<false>(dt, da, db, idesc, acc0);
                }
              }
            }
          }
          umma_commit(bar_empty(s));
          }
          __syncwarp();
          if (++s == stages) { s = 0; ph ^= 1; }
        }
        if (elect_one()) umma_commit(bar_tfull(ab));
        __syncwarp();
      }
    }
  } else if (warp < 6) {
    // ===================== split (fp32) + row statistics =====================
    const int t = threadIdx.x - 64;   // 0..127
    const int r = t >> 3;             // node row inside the k-block (16 rows x 8 chunks = one 2 KB block)
    int s = 0;
    uint32_t ph = 0;
    for (int b = blockIdx.x; b < P.B; b += gridDim.x) {
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(bar_full(s), ph);
        const uint32_t st = smem_base + (uint32_t)s * stage_bytes + (uint32_t)t * 16;
        float sd = 0.f, sa2 = 0.f, s2 = 0.f, se = 0.f;
        constexpr int NV = 16 / ES;  // values per 16-byte chunk
        // One batch = UU blocks of one segment with no branch inside, so the compiler interleaves the UU
        // independent load -> round -> subtract -> store chains (the split warps run one warp per scheduler and are
        // latency-bound: `ncu` showed fixed-latency waits spread over a loop that was serialised by per-chunk
        // segment branches).  SEG: 0 = A (d, a2), 1 = X (no statistics), 2 = S (ss, ent).
        // byte distance from a block to its lo copy: [A/X blocks, S blocks]
        const uint32_t lo_delta[2] = {P.concat ? raw_bytes + (uint32_t)P.nb_s * kBlockBytes : raw_bytes,
                                      P.concat ? (uint32_t)P.nb_s * kBlockBytes : raw_bytes};
        auto batch = [&](auto seg_tag, auto uu_tag, int blk0) {
          constexpr int SEG = decltype(seg_tag)::value;
          constexpr int UU = decltype(uu_tag)::value;
          float v[UU][NV];
#pragma unroll
          for (int u = 0; u < UU; ++u) {
            const uint32_t a = st + (uint32_t)(blk0 + u) * kBlockBytes;
            if (kF32) {
              float4 x4 = lds128(a);
              v[u][0] = x4.x, v[u][1] = x4.y, v[u][2] = x4.z, v[u][3] = x4.w;
            } else {
              uint4 w4 = lds128u(a);
              const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&w4);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                float2 f = __bfloat1622float2(h2[q]);
                v[u][2 * q] = f.x, v[u][2 * q + 1] = f.y;
              }
            }
          }
#pragma unroll
          for (int u = 0; u < UU; ++u) {
            if (kF32) {
              const uint32_t a = st + (uint32_t)(blk0 + u) * kBlockBytes;
              float4 h, l;
              h.x = rna_tf32(v[u][0]), h.y = rna_tf32(v[u][1]), h.z = rna_tf32(v[u][2]), h.w = rna_tf32(v[u][3]);
              l.x = v[u][0] - h.x, l.y = v[u][1] - h.y, l.z = v[u][2] - h.z, l.w = v[u][3] - h.w;
              sts128(a, h);
              sts128(a + lo_delta[SEG == 2 ? 1 : 0], l);
            }
            if (SEG == 0) {  // per-chunk partial sums keep the accumulator chains one add deep per chunk
              float ps = 0.f, pq = 0.f;
#pragma unroll
              for (int q = 0; q < NV; ++q) { ps += v[u][q]; pq = fmaf(v[u][q], v[u][q], pq); }
              sd += ps, sa2 += pq;
            } else if (SEG == 2) {
              float pq = 0.f, pe = 0.f;
#pragma unroll
              for (int q = 0; q < NV; ++q) { pq = fmaf(v[u][q], v[u][q], pq); pe = fmaf(v[u][q], __logf(v[u][q] + P.eps), pe); }
              s2 += pq, se -= pe;
            }
          }
        };
        auto segment = [&](auto seg_tag, int b0, int b1) {
          int blk = b0;
          for (; blk + 4 <= b1; blk += 4) batch(seg_tag, std::integral_constant<int, 4>{}, blk);
          if (blk + 2 <= b1) { batch(seg_tag, std::integral_constant<int, 2>{}, blk); blk += 2; }
          if (blk < b1) batch(seg_tag, std::integral_constant<int, 1>{}, blk);
        };
        segment(std::integral_constant<int, 0>{}, 0, P.nb_a);
        segment(std::integral_constant<int, 1>{}, P.nb_a, P.nb_a + P.nb_x);
        segment(std::integral_constant<int, 2>{}, P.nb_a + P.nb_x, nb);
        // the 8 lanes of a row (fixed lane group, fixed block order -> deterministic)
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
          sd += __shfl_xor_sync(kFull, sd, o);
          sa2 += __shfl_xor_sync(kFull, sa2, o);
          s2 += __shfl_xor_sync(kFull, s2, o);
          se += __shfl_xor_sync(kFull, se, o);
        }
        const int node = kb * FBK + r;
        if ((t & 7) == 0 && node < P.N) {
          const int64_t o = (int64_t)b * P.N + node;
          P.d[o] = sd, P.a2[o] = sa2, P.ss[o] = s2, P.ent[o] = se;
        }
        if (kF32) fence_proxy_async();
        mbar_arrive(bar_lo(s));
        if (++s == stages) { s = 0; ph ^= 1; }
      }
    }
  } else {
    // ===================== epilogue =====================
    const int quad = warp & 3;
    int it = 0;
    for (int b = blockIdx.x; b < P.B; b += gridDim.x, ++it) {
      const int ab = P.acc_bufs == 2 ? (it & 1) : 0;
      const uint32_t aph = P.acc_bufs == 2 ? ((uint32_t)(it >> 1) & 1u) : ((uint32_t)it & 1u);
      mbar_wait(bar_tfull(ab), aph);
      tc_fence_after();
      const int row = quad * 32 + lane;
      for (int g = 0; g < G; ++g) {
        const int seg = g < P.t_a ? 0 : (g < P.t_a + P.t_x ? 1 : 2);
        const int m = (seg == 0 ? g : (seg == 1 ? g - P.t_a : g - P.t_a - P.t_x)) * BM + row;
        const int m_ext = seg == 0 ? P.N : (seg == 1 ? P.F : P.K);
        for (int c0 = 0; c0 < BN; c0 += 32) {
          float v[32];
          const int accw = P.concat ? 2 * BN : BN;
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * G * accw + g * accw + c0), v);
          if (P.concat) {  // + hi x lo_s
            float v2[32];
            tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * G * accw + g * accw + BN + c0), v2);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += v2[j];
          }
          if (m >= m_ext || c0 >= P.K) continue;
          // All three results are written "transposed": for a fixed accumulator column the 32 lanes of a warp
          // hold 32 consecutive rows, which are made the contiguous index of the destination (128-byte stores).
          if (seg == 0) {  // T[b, c, m] = (S^T A)[c, m]   row-major [K, N]
            T* o = reinterpret_cast<T*>(P.Tt) + (int64_t)b * P.K * P.N + m;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < P.K) o[(int64_t)(c0 + j) * P.N] = from_f32<T>(v[j]);
          } else if (seg == 1) {  // X_pool[b, c, m]
            T* o = reinterpret_cast<T*>(P.Xp) + (int64_t)b * P.K * P.F + m;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < P.K) o[(int64_t)(c0 + j) * P.F] = from_f32<T>(v[j]);
          } else {  // M[b, c, m]  (S^T S is symmetric)
            float* o = P.Mm + (int64_t)b * P.K * P.K + m;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < P.K) o[(int64_t)(c0 + j) * P.K] = v[j];
          }
        }
      }
      tc_fence_before();
      mbar_arrive(bar_tempty(ab));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, P.tmem_cols);
}

// Returns TGPB200_ERR_UNSUPPORTED when the shape does not fit (the caller then uses the per-product path).
int dense_fwd_fused(const void* A, const void* S, const void* X, int B, int N, int K, int F, bool bf16, float eps,
                    void* Tt, void* Xp, float* Mm, float* d, float* ss, float* a2, float* ent, cudaStream_t stream) {
  const int es = bf16 ? 2 : 4, epb = kStageRowBytes / es;
  if (!A || !S || !X || B <= 0 || N <= 0 || K <= 0 || F <= 0 || K > 256) return TGPB200_ERR_UNSUPPORTED;
  if ((N * es) % 16 || (K * es) % 16 || (F * es) % 16) return TGPB200_ERR_UNSUPPORTED;
  if (((uintptr_t)A | (uintptr_t)S | (uintptr_t)X) & 15) return TGPB200_ERR_UNSUPPORTED;
  FusedParams P;
  memset(&P, 0, sizeof(P));
  P.B = B, P.N = N, P.K = K, P.F = F;
  P.BN = (K + 15) / 16 * 16;
  P.nb_a = (N + epb - 1) / epb, P.nb_x = (F + epb - 1) / epb, P.nb_s = (K + epb - 1) / epb;
  P.t_a = (N + BM - 1) / BM, P.t_x = (F + BM - 1) / BM, P.t_s = (K + BM - 1) / BM;
  // every segment must start on an MMA-tile boundary of its own blocks: tiles are 128 columns = BM/epb blocks
  const int G = P.t_a + P.t_x + P.t_s;
  // the accumulators of a graph must fit the 512 TMEM columns (K = 256 never does): otherwise the caller runs the
  // per-product launches
  if (G * P.BN > 512 || G > 8) return TGPB200_ERR_UNSUPPORTED;
  P.concat = (!bf16 && K % 32 == 0 && P.BN == K && 2 * G * P.BN <= 512) ? 1 : 0;
  const int accw = P.concat ? 2 * P.BN : P.BN;
  P.acc_bufs = (2 * G * accw <= 512) ? 2 : 1;
  uint32_t cols = 32;
  while (cols < (uint32_t)(P.acc_bufs * G * accw)) cols <<= 1;
  P.tmem_cols = cols;
  const size_t stage_bytes = (size_t)(P.nb_a + P.nb_x + P.nb_s) * kBlockBytes * (bf16 ? 1 : 2);
  int stages = (int)((size_t)(210 * 1024) / stage_bytes);
  if (stages > 8) stages = 8;
  if (stages < 2) return TGPB200_ERR_UNSUPPORTED;
  P.stages = stages;
  P.eps = eps;
  P.Tt = Tt, P.Xp = Xp, P.Mm = Mm, P.d = d, P.ss = ss, P.a2 = a2, P.ent = ent;
  const bool sw32 = !bf16;
  P.blocked = (N % epb == 0 && F % epb == 0 && K % epb == 0 && P.nb_a <= 256) ? 1 : 0;
  if (P.blocked) {
    if (!make_map_blocked(&P.map_a, A, bf16, B, N, N, N, (int64_t)N * N, FBK, P.nb_a, sw32) ||
        !make_map_blocked(&P.map_x, X, bf16, B, N, F, F, (int64_t)N * F, FBK, P.nb_x, sw32) ||
        !make_map_blocked(&P.map_s, S, bf16, B, N, K, K, (int64_t)N * K, FBK, P.nb_s, sw32))
      P.blocked = 0;
  }
  if (!P.blocked) {
    if (!make_map_3d(&P.map_a, A, bf16, B, N, N, N, (int64_t)N * N, FBK, sw32)) return TGPB200_ERR_UNSUPPORTED;
    if (!make_map_3d(&P.map_x, X, bf16, B, N, F, F, (int64_t)N * F, FBK, sw32)) return TGPB200_ERR_UNSUPPORTED;
    if (!make_map_3d(&P.map_s, S, bf16, B, N, K, K, (int64_t)N * K, FBK, sw32)) return TGPB200_ERR_UNSUPPORTED;
  }
  static bool attr_set = false;
  if (!attr_set) {
    attr_set = true;
    cudaFuncSetAttribute(k_dense_fwd_fused<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(k_dense_fwd_fused<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  }
  const size_t smem = stage_bytes * stages + 4 * kBlockBytes + (3 * stages + 4) * 8 + 16 + 1024;
  if (smem > 227 * 1024) return TGPB200_ERR_UNSUPPORTED;
  const int sms = device_sm_count();
  const int grid = B < sms ? B : sms;
  if (bf16)
    launch("k_dense_fwd_fused_bf16", k_dense_fwd_fused<false>, grid, 320, smem, stream, P);
  else
    launch("k_dense_fwd_fused_3xtf32", k_dense_fwd_fused<true>, grid, 320, smem, stream, P);
  return launch_status();
}

}  // namespace tc
}  // namespace tgp
