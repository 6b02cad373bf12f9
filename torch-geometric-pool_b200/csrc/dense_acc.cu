// Asymmetric Cheeger Cut (TVGNN) losses of batched dense assignments, next to the fused dense chain:
//   totvar_b  = sum_ij A_ij ||S_i - S_j||_1 / (2 nnz(A_b))
//   balance_b = 1 - sum_ik f(S_ik - q_bk) / (N (K - 1)),  f(d) = (K - 1) d for d >= 0, -d otherwise,
//   q_bk      = entry of rank N // K of column k of S_b in a stable descending sort (padded N).
// Neither loss is a matrix product: the total variation is pairwise L1 work on the CUDA cores (64 x 64 node-pair
// tiles, S staged in 32-wide column chunks), the quantile a radix select per column.  Nothing of size B N^2 K is
// formed; the only N^2 buffer is dA itself.  Every sum has a fixed order (no float atomics): per-tile partials, then
// one finalize block.
#include "common.cuh"

namespace tgp {
namespace {

constexpr int kPT = 64;  // node-pair tile side of the pairwise kernel
constexpr int kPK = 32;  // columns of S staged per step
constexpr int kDI = 64;  // rows of dS per CTA
constexpr int kDK = 64;  // columns of dS per CTA (two per lane)
constexpr int kDJ = 32;  // neighbours j staged per step
constexpr int kMaxGridY = 65535;

int pair_tiles(int64_t N) { return (int)(ceil_div(N, kPT) * ceil_div(N, kPT)); }

// dL/d(numerator of graph b) = g_tv / (2 nnz_b B); a zero upstream gradient contributes nothing, even for an edgeless
// graph (whose loss is NaN)
__device__ __forceinline__ float tv_coef(const float* gl, long long nnz, int B) {
  const float g = gl ? gl[0] : 0.f;
  return g == 0.f ? 0.f : g / (2.f * (float)nnz * (float)B);
}

// order-preserving key of a float (ascending); -0.0 is folded onto +0.0 so that the two compare equal, as in a sort
__device__ __forceinline__ unsigned order_key(float x) {
  const unsigned u = __float_as_uint(x == 0.f ? 0.f : x);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// One 64 x 64 tile (i-block, j-block) of graph b = blockIdx.y of D_ij = ||S_i - S_j||_1.
//   kGradA = false: tv_part[b][tile] = sum_tile A_ij D_ij and cnt_part[b][tile] = nnz of A over the tile;
//   kGradA = true:  dA_ij = c_b D_ij.
// Thread (tx, ty) owns rows ty*4 .. +3 and columns tx*4 .. +3 of the tile.
template <typename T, bool kGradA>
__global__ void __launch_bounds__(256)
    k_acc_pair_l1(const T* __restrict__ A, const T* __restrict__ S, int N, int K, int B, const float* __restrict__ gl,
                  const long long* __restrict__ nnz, float* __restrict__ tv_part,
                  unsigned long long* __restrict__ cnt_part, T* __restrict__ dA) {
  __shared__ __align__(16) float si[kPK][kPT + 4];
  __shared__ __align__(16) float sj[kPK][kPT + 4];
  __shared__ float red[32];
  __shared__ unsigned long long cred[8];
  const int b = blockIdx.y, tile = blockIdx.x, side = (N + kPT - 1) / kPT;
  const int i0 = (tile / side) * kPT, j0 = (tile % side) * kPT;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const T* Sb = S + (int64_t)b * N * K;
  float acc[4][4];
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) acc[u][v] = 0.f;
  for (int k0 = 0; k0 < K; k0 += kPK) {
    for (int e = t; e < kPT * kPK; e += 256) {  // lanes along k: coalesced row segments of S
      const int r = e / kPK, k = e % kPK;
      const bool kin = k0 + k < K;
      si[k][r] = (kin && i0 + r < N) ? to_f32<T>(Sb[(int64_t)(i0 + r) * K + k0 + k]) : 0.f;
      sj[k][r] = (kin && j0 + r < N) ? to_f32<T>(Sb[(int64_t)(j0 + r) * K + k0 + k]) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < kPK; ++k) {  // zero-padded rows / columns add |0 - 0| = 0
      const float4 a = *reinterpret_cast<const float4*>(&si[k][ty * 4]);
      const float4 c = *reinterpret_cast<const float4*>(&sj[k][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, cv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] += fabsf(av[u] - cv[v]);
    }
    __syncthreads();
  }
  const T* Ab = A + (int64_t)b * N * N;
  if constexpr (kGradA) {
    const float c = tv_coef(gl, nnz[b], B);
    T* dAb = dA + (int64_t)b * N * N;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + ty * 4 + u;
      if (i >= N) break;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int j = j0 + tx * 4 + v;
        if (j < N) dAb[(int64_t)i * N + j] = from_f32<T>(c * acc[u][v]);
      }
    }
  } else {
    float part = 0.f;
    unsigned cnt = 0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + ty * 4 + u;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int j = j0 + tx * 4 + v;
        if (i < N && j < N) {
          const float a = to_f32<T>(Ab[(int64_t)i * N + j]);
          part = fmaf(a, acc[u][v], part);
          cnt += (a != 0.f);  // count_nonzero: NaN counts
        }
      }
    }
    part = block_sum(part, red);
    const int c32 = warp_sum_i((int)cnt);
    if ((t & 31) == 0) cred[t >> 5] = (unsigned long long)c32;
    __syncthreads();
    if (t == 0) {
      unsigned long long ct = 0;
      for (int q = 0; q < 8; ++q) ct += cred[q];
      tv_part[(int64_t)b * gridDim.x + tile] = part;
      cnt_part[(int64_t)b * gridDim.x + tile] = ct;
    }
  }
}

// Quantile of 32 columns k0 .. k0+31 of graph b = blockIdx.y: lane = column, warp w = contiguous row segment.
// A 4-pass radix select (8-bit digits of order_key, most significant first) finds the key of descending rank N // K
// and its rank r among equal keys; a last pass over the segments in row order picks the r-th such row, which is the
// row a stable descending sort puts at N // K.  Then per column: quant = S[i*, k], n_ge = #{i : S_ik >= q} and the
// balance sum sum_i f(S_ik - q); bal_part[b][chunk] = the chunk's balance sum.
template <typename T>
__global__ void __launch_bounds__(256)
    k_acc_quantile(const T* __restrict__ S, int N, int K, T* __restrict__ quant, int32_t* __restrict__ qidx,
                   int32_t* __restrict__ n_ge, float* __restrict__ bal_part) {
  __shared__ unsigned hist[32][257];
  __shared__ unsigned s_prefix[32];
  __shared__ int s_rem[32], s_idx[32];
  __shared__ int cseg[8][32];
  __shared__ float fseg[8][32];
  const int b = blockIdx.y, t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int k0 = blockIdx.x * 32, k = k0 + lane;
  const bool kin = k < K;
  const int seg = (N + 7) / 8, r0 = min(N, w * seg), r1 = min(N, r0 + seg);
  const T* col = S + (int64_t)b * N * K + (kin ? k : 0);
  if (t < 32) s_prefix[t] = 0u, s_rem[t] = N / K;
  unsigned mask = 0u;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int e = t; e < 32 * 257; e += 256) (&hist[0][0])[e] = 0u;
    __syncthreads();
    if (kin) {
      const unsigned pre = s_prefix[lane];
      for (int i = r0; i < r1; ++i) {
        const unsigned key = order_key(to_f32<T>(col[(int64_t)i * K]));
        if ((key & mask) == pre) atomicAdd(&hist[lane][(key >> shift) & 255u], 1u);
      }
    }
    __syncthreads();
    for (int c = w; c < 32; c += 8) {  // warp w picks the digit of columns w, w + 8, ...: lane l owns 8 bins, top down
      if (k0 + c >= K) break;
      const unsigned rem = (unsigned)s_rem[c];
      unsigned loc = 0u;
#pragma unroll
      for (int q = 0; q < 8; ++q) loc += hist[c][255 - 8 * lane - q];
      unsigned incl = loc;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(kFull, incl, o);
        if (lane >= o) incl += y;
      }
      const unsigned excl = incl - loc;
      if (rem >= excl && rem < incl) {  // exactly one lane: the matching count always exceeds rem
        unsigned r = rem - excl;
        int d = 255 - 8 * lane;
        for (int q = 0; q < 8; ++q, --d) {
          const unsigned h = hist[c][d];
          if (r < h) break;
          r -= h;
        }
        s_prefix[c] |= (unsigned)d << shift;
        s_rem[c] = (int)r;
      }
    }
    mask |= 0xffu << shift;
    __syncthreads();
  }
  // the r-th row (in row order) whose key equals the selected one
  const unsigned v = s_prefix[lane];
  int mine = 0;
  if (kin)
    for (int i = r0; i < r1; ++i) mine += order_key(to_f32<T>(col[(int64_t)i * K])) == v;
  cseg[w][lane] = mine;
  __syncthreads();
  if (kin) {
    int before = 0;
    for (int q = 0; q < w; ++q) before += cseg[q][lane];
    const int r = s_rem[lane];
    if (r >= before && r < before + mine) {
      int rr = r - before;
      for (int i = r0; i < r1; ++i)
        if (order_key(to_f32<T>(col[(int64_t)i * K])) == v && rr-- == 0) {
          s_idx[lane] = i;
          break;
        }
    }
  }
  __syncthreads();
  float fs = 0.f;
  int ge = 0;
  if (kin) {
    const float q = to_f32<T>(col[(int64_t)s_idx[lane] * K]), km1 = (float)(K - 1);
    for (int i = r0; i < r1; ++i) {
      const float d = to_f32<T>(col[(int64_t)i * K]) - q;
      if (d >= 0.f) {
        fs = fmaf(km1, d, fs);
        ++ge;
      } else {
        fs -= d;
      }
    }
  }
  fseg[w][lane] = fs;
  cseg[w][lane] = ge;
  __syncthreads();
  if (w == 0) {
    float cs = 0.f;
    if (kin) {
      int cg = 0;
      for (int q = 0; q < 8; ++q) cs += fseg[q][lane], cg += cseg[q][lane];
      const int i = s_idx[lane];
      quant[(int64_t)b * K + k] = col[(int64_t)i * K];
      qidx[(int64_t)b * K + k] = i;
      n_ge[(int64_t)b * K + k] = cg;
    }
    cs = warp_sum(cs);
    if (lane == 0) bal_part[(int64_t)b * gridDim.x + blockIdx.x] = cs;
  }
}

// losses = {mean_b totvar_b, mean_b balance_b}; nnz[b] = nnz(A_b) is saved for the backward.  One block, fixed order.
__global__ void k_acc_finalize(const float* __restrict__ tv_part, const unsigned long long* __restrict__ cnt_part,
                               int tiles, const float* __restrict__ bal_part, int chunks, int B, int N, int K,
                               long long* __restrict__ nnz, float* __restrict__ losses) {
  __shared__ float red[32];
  float tv = 0.f, bal = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float num = 0.f, bs = 0.f;
    unsigned long long ne = 0;
    for (int p = 0; p < tiles; ++p) num += tv_part[(int64_t)b * tiles + p], ne += cnt_part[(int64_t)b * tiles + p];
    for (int p = 0; p < chunks; ++p) bs += bal_part[(int64_t)b * chunks + p];
    nnz[b] = (long long)ne;
    tv += num / (2.f * (float)ne);  // an edgeless graph gives NaN, as the restated formula does
    bal += 1.f - bs / ((float)N * (float)(K - 1));
  }
  tv = block_sum(tv, red);
  bal = block_sum(bal, red);
  if (threadIdx.x == 0) losses[0] = tv / (float)B, losses[1] = bal / (float)B;
}

// dS of rows i0 .. i0+63, columns k0 .. k0+63 of graph b = blockIdx.y (lane = columns lane and lane + 32, warp w =
// rows w*8 .. +7):
//   dS_ik = c_b sum_j (A_ij + A_ji) sign(S_ik - S_jk) - e f'(S_ik - q_k) + [i = i*_k] e sum_i' f'(S_i'k - q_k)
// with e = g_bal / (N (K - 1) B), f' = K - 1 on d >= 0 and -1 below, sum_i' f' = K n_ge - N.  Each CTA streams the row
// panel A[I, J] and the column panel A[J, I] (runs of 64 contiguous entries per row j), so no atomics are needed.
template <typename T>
__global__ void __launch_bounds__(256)
    k_acc_ds(const T* __restrict__ A, const T* __restrict__ S, int N, int K, int B, const float* __restrict__ gl,
             const long long* __restrict__ nnz, const int32_t* __restrict__ qidx, const int32_t* __restrict__ n_ge,
             int kchunks, T* __restrict__ dS) {
  __shared__ __align__(16) float wt[kDJ][kDI + 4];  // wt[j][i] = A_ij + A_ji
  __shared__ float sj[kDJ][kDK];
  const int b = blockIdx.y, i0 = (blockIdx.x / kchunks) * kDI, k0 = (blockIdx.x % kchunks) * kDK;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const T* Sb = S + (int64_t)b * N * K;
  const T* Ab = A + (int64_t)b * N * N;
  float s[8][2], acc[8][2];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = i0 + w * 8 + r, k = k0 + lane + 32 * h;
      s[r][h] = (i < N && k < K) ? to_f32<T>(Sb[(int64_t)i * K + k]) : 0.f;
      acc[r][h] = 0.f;
    }
  for (int j0 = 0; j0 < N; j0 += kDJ) {
    for (int e = t; e < kDI * kDJ; e += 256) {  // row panel, lanes along j
      const int i = e / kDJ, j = e % kDJ;
      wt[j][i] = (i0 + i < N && j0 + j < N) ? to_f32<T>(Ab[(int64_t)(i0 + i) * N + j0 + j]) : 0.f;
    }
    for (int e = t; e < kDJ * kDK; e += 256) {
      const int j = e / kDK, k = e % kDK;
      sj[j][k] = (j0 + j < N && k0 + k < K) ? to_f32<T>(Sb[(int64_t)(j0 + j) * K + k0 + k]) : 0.f;
    }
    __syncthreads();
    for (int e = t; e < kDI * kDJ; e += 256) {  // column panel, lanes along i
      const int j = e / kDI, i = e % kDI;
      if (i0 + i < N && j0 + j < N) wt[j][i] += to_f32<T>(Ab[(int64_t)(j0 + j) * N + i0 + i]);
    }
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < kDJ; ++j) {  // padded neighbours have zero weight
      const float4 wa = *reinterpret_cast<const float4*>(&wt[j][w * 8]);
      const float4 wb = *reinterpret_cast<const float4*>(&wt[j][w * 8 + 4]);
      const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
      const float sv[2] = {sj[j][lane], sj[j][lane + 32]};
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (s[r][h] > sv[h]) acc[r][h] += wv[r];
          if (s[r][h] < sv[h]) acc[r][h] -= wv[r];
        }
    }
    __syncthreads();
  }
  const float c = tv_coef(gl, nnz[b], B);
  const float e = (gl ? gl[1] : 0.f) / ((float)N * (float)(K - 1) * (float)B);
  T* dSb = dS + (int64_t)b * N * K;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int k = k0 + lane + 32 * h;
    if (k >= K) continue;
    const int qi = qidx[(int64_t)b * K + k];
    const float q = to_f32<T>(Sb[(int64_t)qi * K + k]);
    const float tot = (float)K * (float)n_ge[(int64_t)b * K + k] - (float)N;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int i = i0 + w * 8 + r;
      if (i >= N) break;
      float g = c * acc[r][h] - e * (s[r][h] >= q ? (float)(K - 1) : -1.f);
      if (i == qi) g = fmaf(e, tot, g);
      dSb[(int64_t)i * K + k] = from_f32<T>(g);
    }
  }
}

// The saved buffer, shared by the forward and the backward.
struct AccSaved {
  long long* nnz;  // [B]
  int32_t* qidx;   // [B, K]
  int32_t* n_ge;   // [B, K]
  AccSaved(Workspace& ws, int64_t B, int64_t K) {
    nnz = ws.take<long long>((size_t)B);
    qidx = ws.take<int32_t>((size_t)(B * K));
    n_ge = ws.take<int32_t>((size_t)(B * K));
  }
};

// The forward workspace: per-tile partial sums of the total variation, their pair counts, per-chunk balance sums.
struct AccFwdLayout {
  float* tv_part;
  unsigned long long* cnt_part;
  float* bal_part;
  AccFwdLayout(Workspace& ws, int64_t B, int64_t N, int64_t K) {
    const size_t tiles = (size_t)pair_tiles(N);
    tv_part = ws.take<float>((size_t)B * tiles);
    cnt_part = ws.take<unsigned long long>((size_t)B * tiles);
    bal_part = ws.take<float>((size_t)B * ceil_div(K, 32));
  }
};

int acc_check(const void* adj, const void* s, int64_t B, int64_t N, int64_t K, int dtype) {
  if (!adj || !s || B < 0 || N < 1 || K < 2) return TGPB200_ERR_INVALID;
  if (dtype != TGPB200_F32 && dtype != TGPB200_BF16) return TGPB200_ERR_UNSUPPORTED;
  if (B > kMaxGridY || pair_tiles(N) >= INT32_MAX || N * K >= INT32_MAX) return TGPB200_ERR_UNSUPPORTED;
  return TGPB200_OK;
}

template <typename T>
int acc_fwd(const T* A, const T* S, int B, int N, int K, float* losses, T* quant, const AccSaved& sv,
            const AccFwdLayout& l, cudaStream_t st) {
  const int tiles = pair_tiles(N), chunks = (int)ceil_div(K, 32);
  float* tv_part = l.tv_part;
  unsigned long long* cnt_part = l.cnt_part;
  float* bal_part = l.bal_part;
  if (B > 0) {
    launch("k_acc_pair_l1", k_acc_pair_l1<T, false>, dim3(tiles, B), dim3(256), 0, st, A, S, N, K, B,
           (const float*)nullptr, (const long long*)nullptr, tv_part, cnt_part, (T*)nullptr);
    launch("k_acc_quantile", k_acc_quantile<T>, dim3(chunks, B), dim3(256), 0, st, S, N, K, quant, sv.qidx, sv.n_ge,
           bal_part);
  }
  launch("k_acc_finalize", k_acc_finalize, dim3(1), dim3(256), 0, st, (const float*)tv_part,
         (const unsigned long long*)cnt_part, tiles, (const float*)bal_part, chunks, B, N, K, sv.nnz, losses);
  return launch_status();
}

template <typename T>
int acc_bwd(const T* A, const T* S, const float* gl, int B, int N, int K, const AccSaved& sv, T* dS, T* dA,
            cudaStream_t st) {
  if (B == 0) return TGPB200_OK;
  const int kchunks = (int)ceil_div(K, kDK);
  launch("k_acc_ds", k_acc_ds<T>, dim3((unsigned)(ceil_div(N, kDI) * kchunks), B), dim3(256), 0, st, A, S, N, K, B,
         gl, (const long long*)sv.nnz, (const int32_t*)sv.qidx, (const int32_t*)sv.n_ge, kchunks, dS);
  if (dA)
    launch("k_acc_pair_l1:dA", k_acc_pair_l1<T, true>, dim3(pair_tiles(N), B), dim3(256), 0, st, A, S, N, K, B, gl,
           (const long long*)sv.nnz, (float*)nullptr, (unsigned long long*)nullptr, dA);
  return launch_status();
}

}  // namespace
}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_acc_loss_saved_bytes(int64_t B, int64_t K) {
  if (B < 0 || K < 0) return 0;
  return layout_bytes<AccSaved>(B, K);
}

size_t tgpb200_acc_loss_fwd_workspace_bytes(int64_t B, int64_t N, int64_t K) {
  if (B < 0 || N < 1 || K < 1) return 0;
  return layout_bytes<AccFwdLayout>(B, N, K);
}

int tgpb200_acc_loss_fwd(const void* adj, const void* s, int64_t B, int64_t N, int64_t K, int dtype, float* losses,
                         void* quant, void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                         tgpb200_stream_t stream) {
  int rc = acc_check(adj, s, B, N, K, dtype);
  if (rc != TGPB200_OK) return rc;
  if (!losses || !quant) return TGPB200_ERR_INVALID;
  Workspace sw(saved, saved_bytes), ws(workspace, workspace_bytes);
  const AccSaved sv(sw, B, K);
  const AccFwdLayout l(ws, B, N, K);
  if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TGPB200_F32)
    return acc_fwd<float>((const float*)adj, (const float*)s, (int)B, (int)N, (int)K, losses, (float*)quant, sv, l,
                          st);
  return acc_fwd<__nv_bfloat16>((const __nv_bfloat16*)adj, (const __nv_bfloat16*)s, (int)B, (int)N, (int)K, losses,
                                (__nv_bfloat16*)quant, sv, l, st);
}

int tgpb200_acc_loss_bwd(const void* adj, const void* s, const void* saved, size_t saved_bytes,
                         const float* grad_losses, int64_t B, int64_t N, int64_t K, int dtype, void* grad_s,
                         void* grad_adj, tgpb200_stream_t stream) {
  int rc = acc_check(adj, s, B, N, K, dtype);
  if (rc != TGPB200_OK) return rc;
  if (!grad_s) return TGPB200_ERR_INVALID;
  Workspace sw(const_cast<void*>(saved), saved_bytes);
  const AccSaved sv(sw, B, K);
  if (!sw.ok) return TGPB200_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TGPB200_F32)
    return acc_bwd<float>((const float*)adj, (const float*)s, grad_losses, (int)B, (int)N, (int)K, sv,
                          (float*)grad_s, (float*)grad_adj, st);
  return acc_bwd<__nv_bfloat16>((const __nv_bfloat16*)adj, (const __nv_bfloat16*)s, grad_losses, (int)B, (int)N,
                                (int)K, sv, (__nv_bfloat16*)grad_s, (__nv_bfloat16*)grad_adj, st);
}

}  // extern "C"
