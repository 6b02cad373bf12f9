// HOSC kernels shared by the batched dense losses (dense_hosc.cu) and the sparse-adjacency losses (hosc_sparse.cu):
// the padding of S to S1 = [S | 1 | 0 ..], the column statistics, the loss reduction and the elementwise pieces of
// the backward.  Both paths run them on the same padded [B, N, .] layouts, so their results agree bit for bit.
#pragma once
#include "common.cuh"

namespace tgp {
namespace {

constexpr int kFirst = 1, kMotif = 2, kOrtho = 4;  // term mask bits
constexpr int kPad = 8;                            // S1 width granule: 16 bytes of bf16 (TMA row-stride rule)
constexpr int kMaxGridY = 65535;

int s1_width(int K) { return (int)ceil_div(K + 1, kPad) * kPad; }

// S1[b, i, :] = [S[b, i, :] | 1 | 0 ..]
template <typename T>
__global__ void k_hosc_pad(const T* __restrict__ S, int64_t rows, int K, int K1, T* __restrict__ S1) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= rows * K1) return;
  const int64_t r = e / K1;
  const int c = (int)(e - r * K1);
  S1[e] = c < K ? S[r * K + c] : from_f32<T>(c == K ? 1.f : 0.f);
}

// Column statistics of 32 columns k0 .. k0+31 of graph b = blockIdx.y: lane = column, warp w = contiguous row segment;
// the 8 segment partials are added in segment order.  AS1 / AMS1 are [B, N, K1] fp32 (column K = the degree).
//   n1 = sum_i S_ik (A S)_ik, m1 = sum_i d_i S_ik^2 + eps, nM / mM the same of A_M, sq = sum_i S_ik^2.
// Chunk 0 also copies the degrees d, d^M [B, N] for the backward.
template <typename T>
__global__ void __launch_bounds__(256)
    k_hosc_stats(const T* __restrict__ S, const float* __restrict__ AS1, const float* __restrict__ AMS1, int N, int K,
                 int K1, int terms, float eps, float* __restrict__ d, float* __restrict__ dM, float* __restrict__ n1,
                 float* __restrict__ m1, float* __restrict__ nM, float* __restrict__ mM, float* __restrict__ sq) {
  __shared__ float part[5][8][32];
  const int b = blockIdx.y, t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int k = blockIdx.x * 32 + lane;
  const bool kin = k < K;
  const bool first = terms & kFirst, motif = terms & kMotif;
  const int seg = (N + 7) / 8, r0 = min(N, w * seg), r1 = min(N, r0 + seg);
  const T* Sb = S + (int64_t)b * N * K;
  const float* Ab = first ? AS1 + (int64_t)b * N * K1 : nullptr;
  const float* Mb = motif ? AMS1 + (int64_t)b * N * K1 : nullptr;
  float a[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  if (kin)
    for (int i = r0; i < r1; ++i) {
      const float s = to_f32<T>(Sb[(int64_t)i * K + k]), s2 = s * s;
      a[4] = fmaf(s, s, a[4]);
      if (first) {
        a[0] = fmaf(s, Ab[(int64_t)i * K1 + k], a[0]);
        a[1] = fmaf(Ab[(int64_t)i * K1 + K], s2, a[1]);
      }
      if (motif) {
        a[2] = fmaf(s, Mb[(int64_t)i * K1 + k], a[2]);
        a[3] = fmaf(Mb[(int64_t)i * K1 + K], s2, a[3]);
      }
    }
#pragma unroll
  for (int q = 0; q < 5; ++q) part[q][w][lane] = a[q];
  if (blockIdx.x == 0)
    for (int i = t; i < N; i += blockDim.x) {
      if (first) d[(int64_t)b * N + i] = Ab[(int64_t)i * K1 + K];
      if (motif) dM[(int64_t)b * N + i] = Mb[(int64_t)i * K1 + K];
    }
  __syncthreads();
  if (w == 0 && kin) {
    float r[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int p = 0; p < 8; ++p)
#pragma unroll
      for (int q = 0; q < 5; ++q) r[q] += part[q][p][lane];
    const int64_t o = (int64_t)b * K + k;
    n1[o] = r[0], m1[o] = r[1] + eps, nM[o] = r[2], mM[o] = r[3] + eps, sq[o] = r[4];
  }
}

// losses = {L1, L2, O} (zero for a term outside the mask).  One block, fixed order.
__global__ void k_hosc_finalize(const float* __restrict__ n1, const float* __restrict__ m1,
                                const float* __restrict__ nM, const float* __restrict__ mM,
                                const float* __restrict__ sq, const float* __restrict__ graph_nodes, int B, int N,
                                int K, int terms, float* __restrict__ losses) {
  __shared__ float red[32];
  float l1 = 0.f, l2 = 0.f, o = 0.f;
  const float rk = sqrtf((float)K);
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float c1 = 0.f, c2 = 0.f, cn = 0.f;
    for (int k = 0; k < K; ++k) {
      const int64_t e = (int64_t)b * K + k;
      if (terms & kFirst) c1 += n1[e] / m1[e];
      if (terms & kMotif) c2 += nM[e] / mM[e];
      if (terms & kOrtho) cn += sqrtf(sq[e]);
    }
    l1 -= c1 / (float)K;
    l2 -= c2 / (float)K;
    const float n = graph_nodes ? graph_nodes[b] : (float)N;
    if (terms & kOrtho) o += (rk - cn / sqrtf(n)) / (rk - 1.f);
  }
  l1 = block_sum(l1, red);
  l2 = block_sum(l2, red);
  o = block_sum(o, red);
  if (threadIdx.x == 0) losses[0] = l1 / (float)B, losses[1] = l2 / (float)B, losses[2] = o / (float)B;
}

// dL/dn_k of each order: alpha = -g / (K B m_k)
__device__ __forceinline__ float hosc_alpha(float g, float m, int K, int B) { return -g / ((float)K * (float)B * m); }
// dL/dm_k of each order: beta = g n_k / (K B m_k^2)
__device__ __forceinline__ float hosc_beta(float g, float n, float m, int K, int B) {
  return g * n / ((float)K * (float)B * m * m);
}

// Sa = S diag(alpha1), Sm = S diag(alpha2) in the operand dtype (either may be NULL)
template <typename T>
__global__ void k_hosc_scale(const T* __restrict__ S, const float* __restrict__ m1, const float* __restrict__ mM,
                             const float* __restrict__ gl, int64_t total, int B, int N, int K, T* __restrict__ Sa,
                             T* __restrict__ Sm) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int64_t row = e / K;
  const int64_t bk = (row / N) * K + (e - row * K);
  const float s = to_f32<T>(S[e]);
  if (Sa) Sa[e] = from_f32<T>(s * hosc_alpha(gl[0], m1[bk], K, B));
  if (Sm) Sm[e] = from_f32<T>(s * hosc_alpha(gl[1], mM[bk], K, B));
}

// dS += 2 d_i S_ik beta1_k + 2 d^M_i S_ik beta2_k - g2 S_ik / (B sqrt(n_b) (sqrt(K) - 1) ||S_:k||)  (the last term is
// zero for a zero column, as torch's norm backward gives)
template <typename T>
__global__ void k_hosc_ds_elementwise(const T* __restrict__ S, const float* __restrict__ d,
                                      const float* __restrict__ dM, const float* __restrict__ n1,
                                      const float* __restrict__ m1, const float* __restrict__ nM,
                                      const float* __restrict__ mM, const float* __restrict__ sq,
                                      const float* __restrict__ graph_nodes, const float* __restrict__ gl,
                                      int64_t total, int B, int N, int K, int terms, T* __restrict__ dS) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int64_t row = e / K;
  const int b = (int)(row / N);
  const int64_t bk = (int64_t)b * K + (e - row * K);
  const float s = to_f32<T>(S[e]);
  float v = to_f32<T>(dS[e]);
  if (terms & kFirst) v = fmaf(2.f * d[row] * s, hosc_beta(gl[0], n1[bk], m1[bk], K, B), v);
  if (terms & kMotif) v = fmaf(2.f * dM[row] * s, hosc_beta(gl[1], nM[bk], mM[bk], K, B), v);
  if ((terms & kOrtho) && sq[bk] > 0.f) {
    const float n = graph_nodes ? graph_nodes[b] : (float)N;
    v -= gl[2] * s / ((float)B * sqrtf(n) * (sqrtf((float)K) - 1.f) * sqrtf(sq[bk]));
  }
  dS[e] = from_f32<T>(v);
}

// Row terms of dA, one warp per row (b, i): r_i = sum_k beta1_k S_ik^2, rM_i = sum_k beta2_k S_ik^2
template <typename T>
__global__ void k_hosc_rows(const T* __restrict__ S, const float* __restrict__ n1, const float* __restrict__ m1,
                            const float* __restrict__ nM, const float* __restrict__ mM, const float* __restrict__ gl,
                            int64_t rows, int B, int N, int K, int terms, float* __restrict__ r,
                            float* __restrict__ rM) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int64_t b = row / N;
  float a = 0.f, am = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float s = to_f32<T>(S[row * K + k]), s2 = s * s;
    const int64_t bk = b * K + k;
    if (terms & kFirst) a = fmaf(hosc_beta(gl[0], n1[bk], m1[bk], K, B), s2, a);
    if (terms & kMotif) am = fmaf(hosc_beta(gl[1], nM[bk], mM[bk], K, B), s2, am);
  }
  a = warp_sum(a);
  am = warp_sum(am);
  if (lane == 0) r[row] = a, rM[row] = am;
}

}  // namespace
}  // namespace tgp
