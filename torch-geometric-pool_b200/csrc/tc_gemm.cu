// tcgen05 / TMEM / TMA batched GEMM engine (see tc_gemm.cuh for the contract).
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace tgp {
namespace tc {

// ------------------------------------------------------------------------------------------
// Kernel
// ------------------------------------------------------------------------------------------
struct KernelParams {
  CUtensorMap map_a[kMaxPairs];
  CUtensorMap map_b[kMaxPairs];
  int kd[kMaxPairs];
  int a_mn[kMaxPairs], b_mn[kMaxPairs];
  int num_pairs;
  int batch, M, N, BN;
  int m_tiles, n_tiles, num_items;
  int stages;
  uint32_t tmem_cols;
  void* out;
  int64_t out_bs, out_rs, out_cs;
  float alpha;
  int accumulate, out_bf16;
  int skip_lo_b_mask;
  const void* ew_S;
  const float* ew_d;
  const float* ew_coef;
  float ew_eps;
  // Row-major destinations leave through TMA stores: every epilogue warp stages its 32 x 32 chunk in shared memory
  // (swizzled, one row per lane) and one lane issues cp.async.bulk.tensor.  Writing the rows straight from the
  // registers costs 32 separate 128-byte lines per store instruction and kept the LSU busy for ~3 k cycles per
  // 128 x 64 tile (measured with a cycle-counter timeline of the fp32 engine), stalling the split warps that share it.
  CUtensorMap map_out;
  int tma_out;       // 1: use map_out
  int out_vec;       // 1: `out` is 16-byte aligned (the register-store epilogue may write 128-bit pieces)
  int epi_bufs;      // staging buffers per epilogue warp (1 or 2)
  int pack2;         // fp32 TMEM-operand engine: one 128 x 128 tile holds the products of TWO batch items with M, N <= 64
};

// Staging state of one epilogue warp for the TMA-store path
struct EpiStage {
  uint32_t smem;  // first staging buffer of this warp (1024-byte aligned, 4 KB per buffer)
  int n;          // chunks staged so far
};

// Element-wise gradient terms of the dense backward (GemmProblem::ew_*), software-pipelined: the per-row coefficients
// are loaded once per item BEFORE the wait for the accumulators, and the values of S that chunk c needs are loaded
// while chunk c - 1 is processed.  Loaded per chunk after the accumulators were ready, the four dependent global
// round trips (two coefficients, the degree, the row of S) made the epilogue of `dS` the bottleneck of that product
// (C3: 553 -> 354 us for that product with the terms skipped).
template <bool kF32>
struct EwPre {
  float dd = 0.f, c_ent = 0.f;
  bool on = false;      // this row has element-wise terms
  bool vec = false;     // raw[] holds the 32 values of the chunk (else: scalar loads at apply time)
  uint4 raw[kF32 ? 8 : 4];
};
template <bool kF32>
__device__ __forceinline__ void ew_item(const KernelParams& P, EwPre<kF32>& e, int b, int m) {
  e.on = false;
  if (P.ew_S == nullptr || m >= P.M || P.out_cs != 1) return;
  const float c_den = P.ew_coef[b * 4 + 0];
  e.c_ent = P.ew_coef[b * 4 + 2];
  if (c_den == 0.f && e.c_ent == 0.f) return;
  e.on = true;
  e.dd = 2.f * c_den * P.ew_d[(int64_t)b * P.M + m];
}
template <bool kF32>
__device__ __forceinline__ void ew_load(const KernelParams& P, EwPre<kF32>& e, int b, int m, int n0) {
  e.vec = false;
  if (!e.on || n0 >= P.N) return;
  const int64_t si = ((int64_t)b * P.M + m) * P.N + n0;
  if (n0 + 32 <= P.N && (si & (kF32 ? 3 : 7)) == 0) {
    const uint4* s4 = kF32 ? reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(P.ew_S) + si)
                           : reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(P.ew_S) + si);
#pragma unroll
    for (int j = 0; j < (kF32 ? 8 : 4); ++j) e.raw[j] = __ldg(s4 + j);
    e.vec = true;
  }
}
// Called by ALL lanes of the warp (it votes): rows without terms (e.on false) take no part in the arithmetic.
template <bool kF32>
__device__ __forceinline__ void ew_apply(const KernelParams& P, const EwPre<kF32>& e, float (&v)[32], int b, int m, int n0) {
  if (!__any_sync(0xffffffffu, e.on)) return;  // warp-uniform
  float sv[32];
  if (e.on && e.vec) {
    if (kF32) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sv[4 * j] = __uint_as_float(e.raw[j].x), sv[4 * j + 1] = __uint_as_float(e.raw[j].y);
        sv[4 * j + 2] = __uint_as_float(e.raw[j].z), sv[4 * j + 3] = __uint_as_float(e.raw[j].w);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&e.raw[j]);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 f2 = __bfloat1622float2(h2[q]);
          sv[8 * j + 2 * q] = f2.x, sv[8 * j + 2 * q + 1] = f2.y;
        }
      }
    }
  } else if (e.on) {
    const int64_t si = ((int64_t)b * P.M + m) * P.N + n0;
#pragma unroll
    for (int j = 0; j < 32; ++j)
      sv[j] = (n0 + j < P.N) ? (kF32 ? reinterpret_cast<const float*>(P.ew_S)[si + j]
                                     : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(P.ew_S)[si + j]))
                             : 0.f;
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) sv[j] = 1.f;  // inert row: keeps the vote below and the logarithm well defined
  }
  const float dd = e.on ? e.dd : 0.f, c_ent = e.on ? e.c_ent : 0.f;
  if (!__any_sync(0xffffffffu, c_ent != 0.f)) {  // warp-uniform
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaf(dd, sv[j], v[j]);
    return;
  }
  // entropy term -log(s + eps) - s / (s + eps).  With the reference's eps (1e-15) s + eps rounds to s for every s above
  // ~1e-8, where the quotient is EXACTLY 1 (as the reference's IEEE division gives): the reciprocal is only evaluated
  // when some element of the warp's chunk really needs it (the epilogue of dS is bound by the MUFU pipe: two
  // transcendental operations per element).
  bool need_div = false;
#pragma unroll
  for (int j = 0; j < 32; ++j) need_div |= (sv[j] + P.ew_eps) != sv[j];
  if (__any_sync(0xffffffffu, need_div)) {  // warp-uniform
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float se = sv[j] + P.ew_eps;
      v[j] += dd * sv[j] + c_ent * (-__logf(se) - (se == sv[j] ? 1.f : __fdividef(sv[j], se)));
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] += dd * sv[j] + c_ent * (-__logf(sv[j]) - 1.f);
  }
}

// Epilogue of one 32-column chunk: thread `lane` of a quadrant holds row m of the tile, v[0..32) = columns n0..n0+31.
template <bool kF32>
__device__ __forceinline__ void store_chunk(const KernelParams& P, float (&v)[32], int b, int m_base, int m, int n0,
                                            int64_t obase, EpiStage& es, const EwPre<kF32>& ew) {
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] *= P.alpha;
  if (P.out_cs == 1) {
    const bool full = n0 + 32 <= P.N;
    ew_apply<kF32>(P, ew, v, b, m, n0);
    if (P.tma_out) {
      // stage (lane = row of the chunk) with the swizzle of the output map, then one TMA store; rows >= M and
      // columns >= N are clipped by the map
      const int lane = threadIdx.x & 31;
      const int nb = P.epi_bufs;
      const uint32_t buf = es.smem + (uint32_t)(es.n % nb) * (P.out_bf16 ? 2048u : 4096u);  // a bf16 chunk is 2 KB
      if (lane == 0) {
        if (nb == 2) tma_store_wait_read<1>();
        else tma_store_wait_read<0>();
      }
      __syncwarp();
      if (!P.out_bf16) {
        const uint32_t row = buf + (uint32_t)lane * 128u;
#pragma unroll
        for (int c = 0; c < 8; ++c)
          sts128(row + (uint32_t)((c ^ (lane & 7)) << 4), make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]));
      } else {
        const uint32_t row = buf + (uint32_t)lane * 64u;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint4 pk;
          __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
          for (int q = 0; q < 4; ++q) h2[q] = __floats2bfloat162_rn(v[8 * c + 2 * q], v[8 * c + 2 * q + 1]);
          sts128u(row + (uint32_t)((c ^ ((lane >> 1) & 3)) << 4), pk);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        tma_store_3d(&P.map_out, buf, n0, m_base, b);
        tma_store_commit();
      }
      ++es.n;
      return;
    }
    // every thread owns one row and moves its 32 values as 8 x 128-bit accesses
    if (m < P.M) {
      if (P.out_vec && !P.out_bf16 && full && (((obase + n0) & 3) == 0)) {
        float4* o4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(P.out) + obase + n0);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 r4 = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          if (P.accumulate) {
            float4 c4 = o4[j];
            r4.x += c4.x, r4.y += c4.y, r4.z += c4.z, r4.w += c4.w;
          }
          o4[j] = r4;
        }
      } else if (P.out_vec && P.out_bf16 && full && (((obase + n0) & 7) == 0)) {
        uint4* o4 = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(P.out) + obase + n0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4 pk;
          __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&pk);
          if (P.accumulate) {
            uint4 c4 = o4[j];
            const __nv_bfloat162* c2 = reinterpret_cast<const __nv_bfloat162*>(&c4);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float2 f = __bfloat1622float2(c2[q]);
              v[8 * j + 2 * q] += f.x, v[8 * j + 2 * q + 1] += f.y;
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) h2[q] = __floats2bfloat162_rn(v[8 * j + 2 * q], v[8 * j + 2 * q + 1]);
          o4[j] = pk;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (n0 + j < P.N) {
            const int64_t idx = obase + n0 + j;
            float val = v[j];
            if (P.out_bf16) {
              __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(P.out);
              if (P.accumulate) val += __bfloat162float(o[idx]);
              o[idx] = __float2bfloat16_rn(val);
            } else {
              float* o = reinterpret_cast<float*>(P.out);
              if (P.accumulate) val += o[idx];
              o[idx] = val;
            }
          }
        }
      }
    }
  } else if (m < P.M) {
    // strided destination (e.g. transposed output, out_rs == 1): lanes already walk the contiguous index
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (n0 + j < P.N) {
        const int64_t idx = obase + (int64_t)(n0 + j) * P.out_cs;
        float val = v[j];
        if (P.out_bf16) {
          __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(P.out);
          if (P.accumulate) val += __bfloat162float(o[idx]);
          o[idx] = __float2bfloat16_rn(val);
        } else {
          float* o = reinterpret_cast<float*>(P.out);
          if (P.accumulate) val += o[idx];
          o[idx] = val;
        }
      }
    }
  }
}

constexpr int kThreads = 320;
constexpr uint32_t kEpiStageBytes = 32 * 1024;  // 8 x 4 KB staging buffers of the TMA-store epilogue

// bf16 engine: both operands in shared memory, one kind::f16 pass.
__global__ void __launch_bounds__(kThreads, 1) k_tc_gemm(const __grid_constant__ KernelParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int EPB = kStageRowBytes / 2;    // bf16 elements per 128-byte line (= BK)
  constexpr int BK = EPB;
  constexpr int UMMA_K = 16;                 // 32 bytes of K per instruction
  constexpr int KSTEPS = BK / UMMA_K;        // 4

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = P.BN;
  const uint32_t a_bytes = BM * kStageRowBytes, b_bytes = (uint32_t)BN * kStageRowBytes;
  const uint32_t stage_bytes = a_bytes + b_bytes;
  const int stages = P.stages;
  // [stages][stage_bytes] | epilogue staging (kEpiStageBytes, TMA stores) | barriers
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stage_bytes * stages + kEpiStageBytes);
  // barrier layout: full[stages], lo[stages], empty[stages], tmem_full[2], tmem_empty[2] -- the layout of
  // k_tc_gemm_ts, which gemm() sizes the shared memory for; nothing here waits on lo[]
  const uint32_t bar_base = smem_u32(bars);
  auto bar_full = [&](int s) { return bar_base + 8u * s; };
  auto bar_lo = [&](int s) { return bar_base + 8u * (stages + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto bar_tfull = [&](int i) { return bar_base + 8u * (3 * stages + i); };
  auto bar_tempty = [&](int i) { return bar_base + 8u * (3 * stages + 2 + i); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * stages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(bar_full(s), 1);
      mbar_init(bar_lo(s), 128);
      mbar_init(bar_empty(s), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_tfull(i), 1);
      mbar_init(bar_tempty(i), 256);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), P.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // total k-blocks per item (same for every item)
  // (k-block counts come from the kernel parameters each time: a dynamically indexed local array lives in local
  //  memory, and with 227 KB of the L1 carved out as shared memory those loads miss to L2 inside the hot loops)

  if (warp == 0) {
    // ===================== TMA producer (whole warp; one elected lane issues) =====================
    {
      int s = 0;
      uint32_t ph = 0;
      for (int item = blockIdx.x; item < P.num_items; item += gridDim.x) {
        int nt = item % P.n_tiles, mt = (item / P.n_tiles) % P.m_tiles, b = item / (P.n_tiles * P.m_tiles);
        int m0 = mt * BM, n0 = nt * BN;
        for (int p = 0; p < P.num_pairs; ++p) {
          for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb) {
            mbar_wait(bar_empty(s), ph ^ 1);
            uint32_t sa = smem_base + (uint32_t)s * stage_bytes, sb = sa + a_bytes;
            int k0 = kb * BK;
            if (elect_one()) {
              mbar_arrive_expect_tx(bar_full(s), a_bytes + b_bytes);
              // K-major: one box [rows x 128 B].  MN-major: one box [BK k-rows x 128 B] per 128-byte block of
              // the MN extent, laid out block after block (the canonical UMMA MN-major SW128 layout, LBO = BK*128 B).
              if (P.a_mn[p]) {
                for (int blk = 0; blk < BM / EPB; ++blk)
                  tma_load_3d(sa + blk * (BK * kStageRowBytes), &P.map_a[p], bar_full(s), m0 + blk * EPB, k0, b);
              } else {
                tma_load_3d(sa, &P.map_a[p], bar_full(s), k0, m0, b);
              }
              if (P.b_mn[p]) {
                for (int blk = 0; blk < BN / EPB; ++blk)
                  tma_load_3d(sb + blk * (BK * kStageRowBytes), &P.map_b[p], bar_full(s), n0 + blk * EPB, k0, b);
              } else {
                tma_load_3d(sb, &P.map_b[p], bar_full(s), k0, n0, b);
              }
            }
            __syncwarp();
            if (++s == stages) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: ONE elected thread runs the whole loop =====================
    // (electing per k-block and reconverging the warp afterwards costs ~150 cycles per iteration: mma_rate.cu, k_loop)
    // instruction descriptor: c=F32 (1<<4), a/b format BF16 (1), a/b major, N>>3 at [17,23), M>>4 at [24,29)
    const uint32_t tm = __shfl_sync(kFull, tmem_base, 0);
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      int it = 0;
      for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
        int ab = it & 1;
        uint32_t aph = (uint32_t)(it >> 1) & 1u;
        mbar_wait(bar_tempty(ab), aph ^ 1);
        tc_fence_after();
        uint32_t d_tmem = tm + (uint32_t)(ab * BN);
        uint32_t accum = 0;
        for (int p = 0; p < P.num_pairs; ++p) {
          const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)P.a_mn[p] << 15) |
                                 ((uint32_t)P.b_mn[p] << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
          const uint32_t a_lbo = P.a_mn[p] ? BK * kStageRowBytes : 16, b_lbo = P.b_mn[p] ? BK * kStageRowBytes : 16;
          const uint32_t a_step = P.a_mn[p] ? UMMA_K * kStageRowBytes : 32, b_step = P.b_mn[p] ? UMMA_K * kStageRowBytes : 32;
          const uint64_t desc_a0 = make_desc(smem_base, a_lbo, 1024, 2);
          const uint64_t desc_b0 = make_desc(smem_base, b_lbo, 1024, 2);
          for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb) {
            mbar_wait(bar_full(s), ph);
            tc_fence_after();
            // descriptors differ only in the 14-bit start-address field: build once per pair, then add offsets
            const uint32_t so = ((uint32_t)s * stage_bytes) >> 4;
            const uint64_t da0 = desc_a0 + so, db0 = desc_b0 + so + (a_bytes >> 4);
#pragma unroll
            for (int kk = 0; kk < KSTEPS; ++kk) {
              const uint64_t da = da0 + (uint64_t)(kk * (a_step >> 4)), db = db0 + (uint64_t)(kk * (b_step >> 4));
              umma<false>(d_tmem, da, db, idesc, kk == 0 ? accum : 1u);
            }
            umma_commit(bar_empty(s));
            accum = 1;
            if (++s == stages) { s = 0; ph ^= 1; }
          }
        }
        umma_commit(bar_tfull(ab));
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2-9): TMEM -> registers -> global =====================
    // Each quadrant's two warps take alternate 32-column chunks (the fused element-wise epilogue of the backward is
    // instruction-bound with four warps); every warp owns one 4 KB staging buffer.
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int c_first = warp < 6 ? 32 : 0, c_step = 64;
    EpiStage es{smem_base + (uint32_t)stage_bytes * stages + (uint32_t)(warp - 2) * 4096u, 0};
    int it = 0;
    for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
      int nt = item % P.n_tiles, mt = (item / P.n_tiles) % P.m_tiles, b = item / (P.n_tiles * P.m_tiles);
      int ab = it & 1;
      uint32_t aph = (uint32_t)(it >> 1) & 1u;
      const int m_base = mt * BM + quad * 32;
      const int m = m_base + lane;
      const int64_t obase = (int64_t)b * P.out_bs + (int64_t)m * P.out_rs;
      // element-wise terms: coefficients of this row and the S values of the first chunk before the accumulators are
      // waited for, the values of chunk c + 1 while chunk c is processed
      EwPre<false> ew, ew_next;
      ew_item<false>(P, ew, b, m);
      ew_load<false>(P, ew, b, m, nt * BN + c_first);
      mbar_wait(bar_tfull(ab), aph);
      tc_fence_after();
      for (int c0 = c_first; c0 < BN; c0 += c_step) {
        ew_next = ew;
        if (c0 + c_step < BN) ew_load<false>(P, ew_next, b, m, nt * BN + c0 + c_step);
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * BN + c0), v);
        const int n0 = nt * BN + c0;
        if (n0 < P.N && m_base < P.M) store_chunk<false>(P, v, b, m_base, m, n0, obase, es, ew);  // warp-uniform test
        ew = ew_next;
      }
      tc_fence_before();
      mbar_arrive(bar_tempty(ab));
    }
    if (P.tma_out && lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, P.tmem_cols);
}

// ------------------------------------------------------------------------------------------
// fp32 engine with the A operand in TENSOR MEMORY (3xTF32).  With both operands in shared memory the fp32 engine sits
// on the shared-memory pipe (TMA write + split read + hi/lo write back + three operand fetches per k-step); here
// the split warps read the A tile once, round / subtract in registers and tcgen05.st hi and lo into a ring of
// kTsSlots TMEM operand slots (lane = output row, 8 columns = 8 k); only B (hi, lo) stays in shared memory.
//   * two groups of four split warps take alternate k-blocks (the split of a stage is a latency chain); k-block kc
//     goes to group kc % kTsGroups and to operand slot kc % kTsSlots,
//   * K-major A tiles are read row-wise (128-bit, un-doing the 128B swizzle: conflict-free), MN-major A tiles are
//     loaded UNswizzled ([k][128 m]) and read column-wise (32-bit, conflict-free),
//   * three MMAs per k-step (lo_a hi_b, hi_a lo_b, hi_a hi_b), accumulators BN wide, double-buffered.
// Warp roles (448 threads): 0 TMA, 1 MMA, 2-5 split group 0, 6-9 epilogue, 10-13 split group 1.
// ------------------------------------------------------------------------------------------
#ifndef TGPB200_TS_GROUPS
#define TGPB200_TS_GROUPS 2
#endif
constexpr int kTsGroups = TGPB200_TS_GROUPS;  // split groups = TMEM operand stages (k-block kc goes to group kc % G)
constexpr int kThreadsTs = 320 + 128 * (kTsGroups - 1);  // TMA, MMA, split group 0, epilogue, split groups 1..
constexpr int kRingCols = 64;  // TMEM columns per operand stage: 4 k-steps x (8 hi + 8 lo)
// TMEM operand slots: k-block kc uses slot kc % kTsSlots.  More slots than split groups, so that the split warps do not
// wait for the retirement of the MMAs that read a slot two k-blocks ago (commit -> mbarrier -> wait is a long round trip).
constexpr int kTsSlots = 4;  // 2 BN + 4 x 64 columns <= 512 for BN <= 128
static_assert(kTsSlots % kTsGroups == 0, "every operand slot must belong to ONE split group (its waiters see every phase)");

__global__ void __launch_bounds__(kThreadsTs, 1) k_tc_gemm_ts(const __grid_constant__ KernelParams P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr int BK = 32, KSTEPS = 4;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = P.BN;
  const uint32_t a_bytes = BM * kStageRowBytes, b_bytes = (uint32_t)BN * kStageRowBytes;
  const uint32_t stage_bytes = a_bytes + 2 * b_bytes;  // [A raw | B hi | B lo]
  const int stages = P.stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stage_bytes * stages + kEpiStageBytes);
  const uint32_t bar_base = smem_u32(bars);
  auto bar_full = [&](int s) { return bar_base + 8u * s; };
  auto bar_lo = [&](int s) { return bar_base + 8u * (stages + s); };
  auto bar_empty = [&](int s) { return bar_base + 8u * (2 * stages + s); };
  auto bar_tfull = [&](int i) { return bar_base + 8u * (3 * stages + i); };
  auto bar_tempty = [&](int i) { return bar_base + 8u * (3 * stages + 2 + i); };
  auto bar_tfree = [&](int i) { return bar_base + 8u * (3 * stages + 4 + i); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * stages + 4 + kTsSlots);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t ring0 = (uint32_t)(2 * BN);  // first TMEM column of the operand ring

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
    for (int i = 0; i < kTsSlots; ++i) mbar_init(bar_tfree(i), 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(tmem_slot), P.tmem_cols);
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
      int nt = item % P.n_tiles, mt = (item / P.n_tiles) % P.m_tiles, b = item / (P.n_tiles * P.m_tiles);
      int m0 = mt * BM, n0 = nt * BN;
      for (int p = 0; p < P.num_pairs; ++p) {
        for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb) {
          mbar_wait(bar_empty(s), ph ^ 1);
          const uint32_t sa = smem_base + (uint32_t)s * stage_bytes, sb = sa + a_bytes;
          const int k0 = kb * BK;
          if (P.pack2) {
            // item = batch items (2 item, 2 item + 1): rows 0-63 / 64-127 of the A tile and columns 0-63 / 64-127 of the
            // B tile come from the two items (a batch index past the end arrives as zeros)
            if (elect_one()) {
              mbar_arrive_expect_tx(bar_full(s), a_bytes + b_bytes);
              for (int h = 0; h < 2; ++h) {
                tma_load_3d(sa + h * (64 * kStageRowBytes), &P.map_a[p], bar_full(s), k0, 0, 2 * item + h);
                for (int blk = 0; blk < 2; ++blk)
                  tma_load_3d(sb + (2 * h + blk) * (BK * kStageRowBytes), &P.map_b[p], bar_full(s), blk * 32, k0, 2 * item + h);
              }
            }
          } else if (elect_one()) {
            mbar_arrive_expect_tx(bar_full(s), a_bytes + b_bytes);
            if (P.a_mn[p]) tma_load_3d(sa, &P.map_a[p], bar_full(s), m0, k0, b);  // [32 k][128 m], no swizzle
            else tma_load_3d(sa, &P.map_a[p], bar_full(s), k0, m0, b);            // [128 m][32 k], 128B swizzle
            if (P.b_mn[p]) {
              for (int blk = 0; blk < BN / 32; ++blk)
                tma_load_3d(sb + blk * (BK * kStageRowBytes), &P.map_b[p], bar_full(s), n0 + blk * 32, k0, b);
            } else {
              tma_load_3d(sb, &P.map_b[p], bar_full(s), k0, n0, b);
            }
          }
          __syncwarp();
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer: ONE elected thread runs the whole loop =====================
    // (electing per k-block and reconverging the warp afterwards costs ~150 cycles per iteration: mma_rate.cu, k_loop)
    const uint32_t tm = __shfl_sync(kFull, tmem_base, 0);
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0, kc = 0;
      int it = 0;
      for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
        const int ab = it & 1;
        const uint32_t aph = (uint32_t)(it >> 1) & 1u;
        mbar_wait(bar_tempty(ab), aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tm + (uint32_t)(ab * BN);
        uint32_t accum = 0;
        for (int p = 0; p < P.num_pairs; ++p) {
          // tf32 x tf32 -> f32; A from TMEM (K-major by construction), B as stored
          const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)P.b_mn[p] << 16) |
                                 ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
          const uint32_t b_lbo = P.b_mn[p] ? BK * kStageRowBytes : 16;
          const uint32_t b_step = P.b_mn[p] ? 8 * kStageRowBytes : 32;
          const uint64_t desc_b0 = make_desc(smem_base, b_lbo, P.b_mn[p] ? 512 : 1024, P.b_mn[p] ? 1 : 2);
          for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb, ++kc) {
            mbar_wait(bar_lo(s), ph);
            tc_fence_after();
            const uint32_t ts = kc % (uint32_t)kTsSlots;
            const uint32_t a_stage = tm + ring0 + ts * kRingCols;
            const uint64_t db0 = desc_b0 + (uint64_t)(((uint32_t)s * stage_bytes + a_bytes) >> 4);
#pragma unroll
            for (int kk = 0; kk < KSTEPS; ++kk) {
              const uint64_t db = db0 + (uint64_t)(kk * (b_step >> 4)), db_lo = db + (b_bytes >> 4);
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
        }
        umma_commit(bar_tfull(ab));
      }
    }
    __syncwarp();
  } else if (warp < 6 || warp >= 10) {
    // ===================== split: B hi/lo in shared memory, A hi/lo into the TMEM ring =====================
    const int grp = warp >= 10 ? 1 + ((warp - 10) >> 2) : 0;
    const int t = (threadIdx.x - 64) & 127;
    const int q = warp & 3;            // TMEM lane quadrant of this warp
    const int m_local = q * 32 + lane; // output row of the tile this thread stages
    int s = 0;
    uint32_t ph = 0, kc = 0;
    for (int item = blockIdx.x; item < P.num_items; item += gridDim.x) {
      for (int p = 0; p < P.num_pairs; ++p) {
        for (int kb = 0, nkb = (P.kd[p] + BK - 1) / BK; kb < nkb; ++kb, ++kc) {
          if ((int)(kc % (uint32_t)kTsGroups) != grp) {  // another group's k-block
            // The group still OBSERVES the phase of a k-block it skips: with an odd number of stages a stage alternates
            // between the groups, and a parity wait that has missed one completed phase of its barrier passes at once --
            // before the data of the awaited phase has landed (seen as a hang with 3 stages).
            mbar_wait(bar_full(s), ph);
            if (++s == stages) { s = 0; ph ^= 1; }
            continue;
          }
          mbar_wait(bar_full(s), ph);
          const uint32_t sa = smem_base + (uint32_t)s * stage_bytes, sb = sa + a_bytes;
          // B: hi in place, lo behind it
          for (uint32_t ch = t; ch < b_bytes / 16; ch += 128) {
            const float4 v = lds128(sb + ch * 16);
            float4 h, l;
            h.x = rna_tf32(v.x), h.y = rna_tf32(v.y), h.z = rna_tf32(v.z), h.w = rna_tf32(v.w);
            l.x = v.x - h.x, l.y = v.y - h.y, l.z = v.z - h.z, l.w = v.w - h.w;
            sts128(sb + ch * 16, h);
            sts128(sb + b_bytes + ch * 16, l);
          }
          fence_proxy_async();
          // A: this thread's row, 32 k values
          float x[32];
          if (P.a_mn[p]) {
#pragma unroll
            for (int k = 0; k < 32; ++k) x[k] = lds32(sa + (uint32_t)k * (BM * 4) + (uint32_t)m_local * 4);
          } else {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float4 v = lds128(sa + (uint32_t)m_local * kStageRowBytes + (uint32_t)((c ^ (m_local & 7)) << 4));
              x[4 * c] = v.x, x[4 * c + 1] = v.y, x[4 * c + 2] = v.z, x[4 * c + 3] = v.w;
            }
          }
          const uint32_t slot = kc % (uint32_t)kTsSlots;
          mbar_wait(bar_tfree(slot), ((kc / (uint32_t)kTsSlots) & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t a_stage = tmem_base + ((uint32_t)(q * 32) << 16) + ring0 + slot * kRingCols;
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
          mbar_arrive(bar_lo(s));
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue (warps 6-9) =====================
    const int quad = warp & 3;
    EpiStage es{smem_base + (uint32_t)stage_bytes * stages + (uint32_t)(warp - 6) * 2u * 4096u, 0};
    int it = 0;
    for (int item = blockIdx.x; item < P.num_items; item += gridDim.x, ++it) {
      int nt = item % P.n_tiles, mt = (item / P.n_tiles) % P.m_tiles, b = item / (P.n_tiles * P.m_tiles);
      const int ab = it & 1;
      const uint32_t aph = (uint32_t)(it >> 1) & 1u;
      if (P.pack2) {
        // quadrants 0, 1 hold rows 0-63 of batch item 2 item (columns 0-63 of the accumulator), quadrants 2, 3 the
        // rows of item 2 item + 1 (columns 64-127): the off-diagonal blocks of the 128 x 128 tile are not read
        mbar_wait(bar_tfull(ab), aph);
        tc_fence_after();
        const int bb = 2 * item + (quad >> 1), mb = (quad & 1) * 32;
        EwPre<true> none;
        for (int c0 = 0; c0 < 64; c0 += 32) {
          float v[32];
          tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * BN + (quad >> 1) * 64 + c0), v);
          if (bb < P.batch && c0 < P.N && mb < P.M)  // warp-uniform
            store_chunk<true>(P, v, bb, mb, mb + lane, c0, (int64_t)bb * P.out_bs + (int64_t)(mb + lane) * P.out_rs, es, none);
        }
        tc_fence_before();
        mbar_arrive(bar_tempty(ab));
        continue;
      }
      const int m_base = mt * BM + quad * 32;
      const int m = m_base + lane;
      const int64_t obase = (int64_t)b * P.out_bs + (int64_t)m * P.out_rs;
      // element-wise terms (see EwPre): coefficients + the first chunk's S values before the accumulators are waited
      // for, every later chunk's values issued before its TMEM read (one prefetch buffer: 128 registers per thread here)
      EwPre<true> ew;
      ew_item<true>(P, ew, b, m);
      ew_load<true>(P, ew, b, m, nt * BN);
      mbar_wait(bar_tfull(ab), aph);
      tc_fence_after();
      for (int c0 = 0; c0 < BN; c0 += 32) {
        const int n0 = nt * BN + c0;
        if (c0 > 0) ew_load<true>(P, ew, b, m, n0);
        float v[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(ab * BN + c0), v);
        if (n0 < P.N && m_base < P.M) store_chunk<true>(P, v, b, m_base, m, n0, obase, es, ew);  // warp-uniform test
      }
      tc_fence_before();
      mbar_arrive(bar_tempty(ab));
    }
    if (P.tma_out && lane == 0) tma_store_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, P.tmem_cols);
}

// ------------------------------------------------------------------------------------------
// Host side: tensor maps and launch
// ------------------------------------------------------------------------------------------
EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

bool make_map_3d(CUtensorMap* map, const void* ptr, bool bf16, int64_t batch, int64_t rows, int64_t cols,
                 int64_t row_stride, int64_t batch_stride, int box_rows, bool swizzle32) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const int es = bf16 ? 2 : 4, epb = kStageRowBytes / es;
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t bs = (cuuint64_t)(batch_stride > 0 ? batch_stride : row_stride * rows) * es;
  cuuint64_t strides[2] = {(cuuint64_t)row_stride * es, bs};
  cuuint32_t box[3] = {(cuuint32_t)epb, (cuuint32_t)box_rows, 1}, estr[3] = {1, 1, 1};
  CUresult r = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3,
                  const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

bool make_map_blocked(CUtensorMap* map, const void* ptr, bool bf16, int64_t batch, int64_t rows, int64_t cols,
                      int64_t row_stride, int64_t batch_stride, int box_rows, int box_blocks, bool swizzle32) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const int es = bf16 ? 2 : 4, epb = kStageRowBytes / es;
  if (cols % epb) return false;
  cuuint64_t dims[4] = {(cuuint64_t)epb, (cuuint64_t)rows, (cuuint64_t)(cols / epb), (cuuint64_t)batch};
  cuuint64_t bs = (cuuint64_t)(batch_stride > 0 ? batch_stride : row_stride * rows) * es;
  cuuint64_t strides[3] = {(cuuint64_t)row_stride * es, (cuuint64_t)kStageRowBytes, bs};
  cuuint32_t box[4] = {(cuuint32_t)epb, (cuuint32_t)box_rows, (cuuint32_t)box_blocks, 1}, estr[4] = {1, 1, 1, 1};
  CUresult r = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4,
                  const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swizzle32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

int device_sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// Operand [batch][rows][cols] (cols contiguous).  K-major: rows = MN extent, cols = K extent, box {BK, box_mn, 1}.
// MN-major: rows = K extent, cols = MN extent, box {EPB, BK, 1} (one load per 128-byte block of the MN extent).
bool make_operand_map(CUtensorMap* map, const OperandDesc& op, bool bf16, int batch, int mn_extent, int k_extent,
                      int box_mn) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  const int es = bf16 ? 2 : 4, epb = kStageRowBytes / es;
  CUtensorMapDataType dt = bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  cuuint64_t dims[4], strides[3];
  cuuint32_t box[4], estr[4] = {1, 1, 1, 1};
  cuuint32_t rank;
  // a stride of 0 is not encodable: a single batch item gets a dummy (never used) batch stride
  cuuint64_t bstride = (cuuint64_t)(op.batch_stride > 0 ? op.batch_stride : (int64_t)op.row_stride * (op.mn_major ? k_extent : mn_extent)) * es;
  if (!op.mn_major) {
    rank = 3;
    dims[0] = (cuuint64_t)k_extent, dims[1] = (cuuint64_t)mn_extent, dims[2] = (cuuint64_t)batch;
    strides[0] = (cuuint64_t)op.row_stride * es, strides[1] = bstride;
    box[0] = epb, box[1] = box_mn, box[2] = 1;
  } else {
    rank = 3;
    dims[0] = (cuuint64_t)mn_extent, dims[1] = (cuuint64_t)k_extent, dims[2] = (cuuint64_t)batch;
    strides[0] = (cuuint64_t)op.row_stride * es, strides[1] = bstride;
    box[0] = epb, box[1] = epb /* BK rows */, box[2] = 1;
    (void)box_mn;
  }
  CUtensorMapSwizzle sw = (!bf16 && op.mn_major) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = fn(map, dt, rank, const_cast<void*>(op.ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// MN-major operand as ONE unswizzled box [BK k-rows][128 MN columns] (TMEM-operand engine: only the split warps read it)
bool make_operand_map_mn_plain(CUtensorMap* map, const OperandDesc& op, int batch, int mn_extent, int k_extent) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {(cuuint64_t)mn_extent, (cuuint64_t)k_extent, (cuuint64_t)batch};
  cuuint64_t bstride = (cuuint64_t)(op.batch_stride > 0 ? op.batch_stride : (int64_t)op.row_stride * k_extent) * 4;
  cuuint64_t strides[2] = {(cuuint64_t)op.row_stride * 4, bstride};
  cuuint32_t box[3] = {(cuuint32_t)BM, 32, 1}, estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(op.ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

static int pick_bn(const GemmProblem& p) {
  int cap = p.in_bf16 ? 256 : 128;
  int bn = 64;
  while (bn < cap && bn < p.N) bn <<= 1;
  return bn;
}

bool gemm_supported(const GemmProblem& p) {
  if (p.batch <= 0 || p.M <= 0 || p.N <= 0 || p.num_pairs < 1 || p.num_pairs > kMaxPairs) return false;
  const int es = p.in_bf16 ? 2 : 4;
  for (int i = 0; i < p.num_pairs; ++i) {
    if (p.kd[i] <= 0) return false;
    const OperandDesc* ops[2] = {&p.a[i], &p.b[i]};
    const int mn[2] = {p.M, p.N};
    for (int j = 0; j < 2; ++j) {
      const OperandDesc& o = *ops[j];
      if (((uintptr_t)o.ptr & 15) != 0) return false;
      if ((o.row_stride * es) % 16 != 0 || (o.batch_stride * es) % 16 != 0) return false;
      (void)mn;
    }
  }
  return encode_fn() != nullptr;
}

int gemm(const GemmProblem& p, cudaStream_t stream) {
  if (!gemm_supported(p)) return TGPB200_ERR_UNSUPPORTED;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (num_sms <= 0) num_sms = 148;
    cudaFuncSetAttribute(k_tc_gemm, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(k_tc_gemm_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  }
  KernelParams P;
  memset(&P, 0, sizeof(P));
  const bool bf16 = p.in_bf16 != 0;
  P.BN = pick_bn(p);
  const bool ts = !bf16;  // fp32: A operand staged in tensor memory (k_tc_gemm_ts)
  P.num_pairs = p.num_pairs;
  P.batch = p.batch, P.M = p.M, P.N = p.N;
  // Small per-item products (M, N <= 64: the [K, K] products of the pooled graphs) leave three quarters of a 128 x 128
  // tile empty and pay the per-k-block cost of the pipeline for it: TWO batch items share one tile -- A rows 0-63 /
  // 64-127 and B columns 0-63 / 64-127 come from the two items, the diagonal 64 x 64 blocks of the accumulator are
  // their products (the off-diagonal blocks are computed and dropped: the MMA costs N/2 cycles either way).
  {
    const char* e = getenv("TGPB200_GEMM_PACK2");
    P.pack2 = ts && !(e && e[0] == '0') && p.num_pairs == 1 && p.M <= 64 && p.N <= 64 && p.batch >= 2 &&
              !p.a[0].mn_major && p.b[0].mn_major && p.ew_S == nullptr && p.out_col_stride == 1;
  }
  if (P.pack2) P.BN = 128;
  P.m_tiles = (p.M + BM - 1) / BM, P.n_tiles = (p.N + P.BN - 1) / P.BN;
  P.num_items = P.pack2 ? (p.batch + 1) / 2 : p.batch * P.m_tiles * P.n_tiles;
  for (int i = 0; i < p.num_pairs; ++i) {
    P.kd[i] = p.kd[i];
    P.a_mn[i] = p.a[i].mn_major, P.b_mn[i] = p.b[i].mn_major;
    if (ts && p.a[i].mn_major) {
      if (!make_operand_map_mn_plain(&P.map_a[i], p.a[i], p.batch, p.M, p.kd[i])) return TGPB200_ERR_UNSUPPORTED;
    } else if (!make_operand_map(&P.map_a[i], p.a[i], bf16, p.batch, p.M, p.kd[i], P.pack2 ? 64 : BM)) {
      return TGPB200_ERR_UNSUPPORTED;
    }
    if (!make_operand_map(&P.map_b[i], p.b[i], bf16, p.batch, p.N, p.kd[i], P.BN)) return TGPB200_ERR_UNSUPPORTED;
  }
  const size_t stage_bytes = (size_t)(BM + (ts ? 2 : 1) * P.BN) * kStageRowBytes;
  const size_t budget = 192 * 1024;  // + 32 KB of epilogue staging + barriers + alignment slack <= 227 KB
  int stages = (int)(budget / stage_bytes);
  if (stages > 6) stages = 6;
  if (stages < 2) return TGPB200_ERR_UNSUPPORTED;
  P.stages = stages;
  uint32_t cols = 32;
  // two BN-wide accumulators; the TMEM-operand engine adds its ring of operand slots
  while (cols < (uint32_t)(2 * P.BN + (ts ? kTsSlots * kRingCols : 0))) cols <<= 1;
  P.tmem_cols = cols;
  P.out = p.out, P.out_bs = p.out_batch_stride, P.out_rs = p.out_row_stride, P.out_cs = p.out_col_stride;
  P.alpha = p.alpha, P.accumulate = p.accumulate, P.out_bf16 = p.out_bf16;
  P.skip_lo_b_mask = p.skip_lo_b_mask;
  P.ew_S = p.ew_S, P.ew_d = p.ew_d, P.ew_coef = p.ew_coef, P.ew_eps = p.ew_eps;
  // TMA-store epilogue: row-major destination, no read-modify-write, 16-byte aligned rows
  {
    const int oes = p.out_bf16 ? 2 : 4;
    // staging tiles per epilogue warp: the fp32 engine's four warps own 8 KB each, the bf16 engine's eight warps 4 KB
    // each -- room for two 2 KB bf16 chunks, so a store can still read one while the next chunk is staged
    P.epi_bufs = bf16 ? (p.out_bf16 ? 2 : 1) : 2;
    P.tma_out = 0;
    P.out_vec = ((uintptr_t)p.out & 15) == 0;
    if (p.out_col_stride == 1 && !p.accumulate && ((uintptr_t)p.out & 15) == 0 &&
        (p.out_row_stride * oes) % 16 == 0 && (p.out_batch_stride * oes) % 16 == 0 && p.out_row_stride >= p.N) {
      EncodeTiledFn fn = encode_fn();
      cuuint64_t dims[3] = {(cuuint64_t)p.N, (cuuint64_t)p.M, (cuuint64_t)p.batch};
      cuuint64_t bs = (cuuint64_t)(p.out_batch_stride > 0 ? p.out_batch_stride : p.out_row_stride * p.M) * oes;
      cuuint64_t strides[2] = {(cuuint64_t)p.out_row_stride * oes, bs};
      cuuint32_t box[3] = {32, 32, 1}, estr[3] = {1, 1, 1};
      if (fn && fn(&P.map_out, p.out_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, p.out,
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   p.out_bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
        P.tma_out = 1;
    }
  }
  const size_t smem = stage_bytes * stages + kEpiStageBytes + (3 * stages + 4) * 8 + 16 + 1024;
  int grid = P.num_items < num_sms ? P.num_items : num_sms;
  if (ts) {
    launch(p.tag ? p.tag : "k_tc_gemm_ts_3xtf32", k_tc_gemm_ts, grid, kThreadsTs, smem + 64, stream, P);
    return launch_status();
  }
  launch(p.tag ? p.tag : "k_tc_gemm_bf16", k_tc_gemm, grid, kThreads, smem, stream, P);
  return launch_status();
}

}  // namespace tc
}  // namespace tgp

// Test / integration entry point: one batched product with explicit operand layouts.
extern "C" int tgpb200_tc_gemm(const void* a, const void* b, void* out, int64_t batch, int64_t M, int64_t N, int64_t Kd,
                               int64_t a_batch_stride, int64_t a_row_stride, int a_mn_major, int64_t b_batch_stride,
                               int64_t b_row_stride, int b_mn_major, int64_t out_batch_stride, int64_t out_row_stride,
                               int64_t out_col_stride, int in_dtype, int out_dtype, float alpha, int accumulate,
                               tgpb200_stream_t stream) {
  tgp::tc::GemmProblem p;
  memset(&p, 0, sizeof(p));
  p.batch = (int)batch, p.M = (int)M, p.N = (int)N, p.num_pairs = 1, p.kd[0] = (int)Kd;
  p.a[0] = {a, a_batch_stride, a_row_stride, a_mn_major};
  p.b[0] = {b, b_batch_stride, b_row_stride, b_mn_major};
  p.out = out, p.out_batch_stride = out_batch_stride, p.out_row_stride = out_row_stride, p.out_col_stride = out_col_stride;
  p.alpha = alpha, p.accumulate = accumulate, p.out_bf16 = out_dtype == TGPB200_BF16, p.in_bf16 = in_dtype == TGPB200_BF16;
  return tgp::tc::gemm(p, (cudaStream_t)stream);
}
