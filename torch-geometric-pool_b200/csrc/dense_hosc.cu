// HOSC (higher-order spectral clustering) losses of batched dense assignments, next to the fused dense chain:
//   d = A 1,  n_k = (S^T A S)_kk,  m_k = sum_i d_i S_ik^2 + eps                    (first order)
//   A_M = (A A) . A,  d^M = A_M 1,  n^M_k = (S^T A_M S)_kk,  m^M_k = sum_i d^M_i S_ik^2 + eps   (triangle motif)
//   L1 = mean_b -(1/K) sum_k n_k / m_k,  L2 = the same of the motif terms,
//   O  = mean_b (sqrt(K) - sum_k ||S_:k|| / sqrt(n_b)) / (sqrt(K) - 1)             (HOSC's own orthogonality term)
// The products run through mm() (dense.cuh): P = A A, then [A S | A 1] and [A_M S | A_M 1] as ONE product each with
// S1 = [S | 1 | 0 ..] (multiplying by one is exact in 3xTF32 and bf16), so the degrees need no kernel of their own.
// The backward's dS is one four-pair product A Sa + A^T Sa + A_M Sm + A_M^T Sm (Sa = S diag(alpha1), Sm = S
// diag(alpha2), transposes read MN-major) plus k_hosc_ds_elementwise.  Every sum has a fixed order (no float atomics).
#include <type_traits>

#include "dense.cuh"
#include "hosc.cuh"

namespace tgp {
namespace {

// A_M = P . A in the operand dtype (P fp32; the fp32 form writes in place over P, so no __restrict__ on P / AM)
template <typename T>
__global__ void k_hosc_motif(const float* P, const T* __restrict__ A, int64_t total, T* AM) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < total) AM[e] = from_f32<T>(P[e] * to_f32<T>(A[e]));
}

// dA = r_i (+ G_ij P_ij) and H = G . A with G = E2 + rM_i, E2 = S diag(alpha2) S^T (motif term only)
template <typename T>
__global__ void k_hosc_da_prep(const T* __restrict__ A, const float* __restrict__ P, const float* __restrict__ E2,
                               const float* __restrict__ r, const float* __restrict__ rM, int64_t total, int N,
                               T* __restrict__ H, T* __restrict__ dA) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int64_t row = e / N;
  float v = r[row];
  if (P) {
    const float g = E2[e] + rM[row];
    v = fmaf(g, P[e], v);
    H[e] = from_f32<T>(g * to_f32<T>(A[e]));
  }
  dA[e] = from_f32<T>(v);
}

// The saved buffer, shared by the forward and the backward.
template <typename T>
struct HoscSaved {
  T* AM;       // [B, N, N] (motif term only)
  float* d;    // [B, N]
  float* dM;   // [B, N]
  float *n1, *m1, *nM, *mM, *sq;  // [B, K]
  HoscSaved(Workspace& ws, int64_t B, int64_t N, int64_t K, int terms) {
    AM = (terms & kMotif) ? ws.take<T>((size_t)(B * N * N)) : nullptr;
    d = ws.take<float>((size_t)(B * N));
    dM = ws.take<float>((size_t)(B * N));
    n1 = ws.take<float>((size_t)(B * K));
    m1 = ws.take<float>((size_t)(B * K));
    nM = ws.take<float>((size_t)(B * K));
    mM = ws.take<float>((size_t)(B * K));
    sq = ws.take<float>((size_t)(B * K));
  }
};

// The forward workspace: S padded to K1 columns, the products A S1 and A_M S1, and the fp32 A A of bf16 runs (fp32
// runs build it in the saved A_M).
template <typename T>
struct HoscFwdLayout {
  T* S1;
  float *AS1, *AMS1, *P;
  HoscFwdLayout(Workspace& ws, int64_t B, int64_t N, int64_t K, int terms) {
    const size_t NK1 = (size_t)N * s1_width((int)K);
    S1 = ws.take<T>((size_t)B * NK1);
    AS1 = ws.take<float>((size_t)B * NK1);
    AMS1 = ws.take<float>((size_t)B * NK1);
    P = ((terms & kMotif) && !std::is_same<T, float>::value) ? ws.take<float>((size_t)(B * N * N)) : nullptr;
  }
};

// The backward workspace: the scaled assignments, and the terms of the adjacency gradient when it is asked for.
template <typename T>
struct HoscBwdLayout {
  T *Sa, *Sm, *H;
  float *P, *E2, *r, *rM;
  HoscBwdLayout(Workspace& ws, int64_t B, int64_t N, int64_t K, bool need_grad_adj) {
    Sa = ws.take<T>((size_t)(B * N * K));
    Sm = ws.take<T>((size_t)(B * N * K));
    P = need_grad_adj ? ws.take<float>((size_t)(B * N * N)) : nullptr;
    E2 = need_grad_adj ? ws.take<float>((size_t)(B * N * N)) : nullptr;
    H = need_grad_adj ? ws.take<T>((size_t)(B * N * N)) : nullptr;
    r = need_grad_adj ? ws.take<float>((size_t)(B * N)) : nullptr;
    rM = need_grad_adj ? ws.take<float>((size_t)(B * N)) : nullptr;
  }
};

// Bytes of a HOSC layout for the operand dtype.
template <template <typename> class Layout, typename... Args>
size_t hosc_layout_bytes(int dtype, Args... args) {
  return dtype == TGPB200_F32 ? layout_bytes<Layout<float>>(args...) : layout_bytes<Layout<__nv_bfloat16>>(args...);
}

int hosc_check(const void* adj, const void* s, int64_t B, int64_t N, int64_t K, int dtype, int terms) {
  if (!adj || !s || B < 0 || N < 1 || K < 2 || terms <= 0 || terms > 7) return TGPB200_ERR_INVALID;
  if (dtype != TGPB200_F32 && dtype != TGPB200_BF16) return TGPB200_ERR_UNSUPPORTED;
  if (B > kMaxGridY || N >= 65536 || K >= 32768) return TGPB200_ERR_UNSUPPORTED;
  return TGPB200_OK;
}

unsigned blocks(int64_t total, int threads = 256) { return (unsigned)ceil_div(total, threads); }

template <typename T>
int hosc_fwd(const T* A, const T* S, const float* graph_nodes, int B, int N, int K, int terms, float eps,
             float* losses, const HoscSaved<T>& sv, const HoscFwdLayout<T>& l, cudaStream_t st) {
  constexpr bool f32 = std::is_same<T, float>::value;
  const int K1 = s1_width(K);
  const int64_t NN = (int64_t)N * N, NK1 = (int64_t)N * K1;
  const bool first = terms & kFirst, motif = terms & kMotif;
  T* S1 = l.S1;
  float *AS1 = l.AS1, *AMS1 = l.AMS1;
  float* P = (motif && !f32) ? l.P : reinterpret_cast<float*>(sv.AM);
  int rc;
  if (B > 0) {
    const int64_t rows = (int64_t)B * N;
    if (first || motif) launch("k_hosc_pad", k_hosc_pad<T>, blocks(rows * K1), 256, 0, st, S, rows, K, K1, S1);
    const Mat s1{S1, NK1, K1, 1};
    if (motif) {  // P = A A (fp32), A_M = P . A, [A_M S | d^M] = A_M S1
      const int kd = N;
      const Mat a{A, NN, N, 0}, at{A, NN, N, 1};
      rc = mm<T, float>(B, N, N, 1, &kd, &a, &at, P, NN, N, 1, st, EwHook(), "k_tc_gemm:hosc:P=AA");
      if (rc) return rc;
      launch("k_hosc_motif", k_hosc_motif<T>, blocks((int64_t)B * NN), 256, 0, st, (const float*)P, A,
             (int64_t)B * NN, sv.AM);
      const Mat am{sv.AM, NN, N, 0};
      rc = mm<T, float>(B, N, K1, 1, &kd, &am, &s1, AMS1, NK1, K1, 1, st, EwHook(), "k_tc_gemm:hosc:AMS1");
      if (rc) return rc;
    }
    if (first) {  // [A S | d] = A S1
      const int kd = N;
      const Mat a{A, NN, N, 0};
      rc = mm<T, float>(B, N, K1, 1, &kd, &a, &s1, AS1, NK1, K1, 1, st, EwHook(), "k_tc_gemm:hosc:AS1");
      if (rc) return rc;
    }
    launch("k_hosc_stats", k_hosc_stats<T>, dim3((unsigned)ceil_div(K, 32), (unsigned)B), 256, 0, st, S,
           (const float*)AS1, (const float*)AMS1, N, K, K1, terms, eps, sv.d, sv.dM, sv.n1, sv.m1, sv.nM, sv.mM,
           sv.sq);
  }
  launch("k_hosc_finalize", k_hosc_finalize, 1, 256, 0, st, (const float*)sv.n1, (const float*)sv.m1,
         (const float*)sv.nM, (const float*)sv.mM, (const float*)sv.sq, graph_nodes, B, N, K, terms, losses);
  return launch_status();
}

template <typename T>
int hosc_bwd(const T* A, const T* S, const float* graph_nodes, const float* gl, int B, int N, int K, int terms,
             const HoscSaved<T>& sv, T* dS, T* dA, const HoscBwdLayout<T>& l, cudaStream_t st) {
  const int64_t NN = (int64_t)N * N, NK = (int64_t)N * K;
  const bool first = terms & kFirst, motif = terms & kMotif;
  T *Sa = l.Sa, *Sm = l.Sm, *H = l.H;
  float *P = l.P, *E2 = l.E2, *r = l.r, *rM = l.rM;
  if (B == 0) return TGPB200_OK;
  if (!gl) {  // no upstream gradient: zero
    cudaMemsetAsync(dS, 0, (size_t)B * NK * sizeof(T), st);
    if (dA) cudaMemsetAsync(dA, 0, (size_t)B * NN * sizeof(T), st);
    return launch_status();
  }
  int rc;
  const int64_t total = (int64_t)B * NK;
  if (first || motif)
    launch("k_hosc_scale", k_hosc_scale<T>, blocks(total), 256, 0, st, S, (const float*)sv.m1, (const float*)sv.mM,
           gl, total, B, N, K, first ? Sa : (T*)nullptr, motif ? Sm : (T*)nullptr);
  {  // dS = A Sa + A^T Sa + A_M Sm + A_M^T Sm
    int kd[4];
    Mat a[4], b[4];
    int n = 0;
    if (first) {
      kd[n] = N, a[n] = Mat{A, NN, N, 0}, b[n] = Mat{Sa, NK, K, 1}, ++n;
      kd[n] = N, a[n] = Mat{A, NN, N, 1}, b[n] = Mat{Sa, NK, K, 1}, ++n;
    }
    if (motif) {
      kd[n] = N, a[n] = Mat{sv.AM, NN, N, 0}, b[n] = Mat{Sm, NK, K, 1}, ++n;
      kd[n] = N, a[n] = Mat{sv.AM, NN, N, 1}, b[n] = Mat{Sm, NK, K, 1}, ++n;
    }
    if (n > 0) {
      rc = mm<T, T>(B, N, K, n, kd, a, b, dS, NK, K, 1, st, EwHook(), "k_tc_gemm:hosc:dS");
      if (rc) return rc;
    } else {
      cudaMemsetAsync(dS, 0, (size_t)B * NK * sizeof(T), st);
    }
  }
  launch("k_hosc_ds_elementwise", k_hosc_ds_elementwise<T>, blocks(total), 256, 0, st, S, (const float*)sv.d,
         (const float*)sv.dM, (const float*)sv.n1, (const float*)sv.m1, (const float*)sv.nM, (const float*)sv.mM,
         (const float*)sv.sq, graph_nodes, gl, total, B, N, K, terms, dS);
  if (!dA) return launch_status();
  // dA = S diag(alpha1) S^T + r 1^T + G . P + H A^T + A^T H,  G = S diag(alpha2) S^T + rM 1^T,  H = G . A
  const int64_t rows = (int64_t)B * N;
  launch("k_hosc_rows", k_hosc_rows<T>, blocks(rows * 32), 256, 0, st, S, (const float*)sv.n1, (const float*)sv.m1,
         (const float*)sv.nM, (const float*)sv.mM, gl, rows, B, N, K, terms, r, rM);
  if (motif) {
    const int kn = N, kk = K;
    const Mat a{A, NN, N, 0}, at{A, NN, N, 1}, sm{Sm, NK, K, 0}, s{S, NK, K, 0};
    rc = mm<T, float>(B, N, N, 1, &kn, &a, &at, P, NN, N, 1, st, EwHook(), "k_tc_gemm:hosc:P=AA");
    if (rc) return rc;
    rc = mm<T, float>(B, N, N, 1, &kk, &sm, &s, E2, NN, N, 1, st, EwHook(), "k_tc_gemm:hosc:E2=SmSt");
    if (rc) return rc;
  }
  launch("k_hosc_da_prep", k_hosc_da_prep<T>, blocks((int64_t)B * NN), 256, 0, st, A,
         motif ? (const float*)P : (const float*)nullptr, (const float*)E2, (const float*)r, (const float*)rM,
         (int64_t)B * NN, N, H, dA);
  {  // dA += Sa S^T + H A^T + A^T H  (one accumulating call)
    int kd[3];
    Mat a[3], b[3];
    int n = 0;
    if (first) kd[n] = K, a[n] = Mat{Sa, NK, K, 0}, b[n] = Mat{S, NK, K, 0}, ++n;
    if (motif) {
      kd[n] = N, a[n] = Mat{H, NN, N, 0}, b[n] = Mat{A, NN, N, 0}, ++n;
      kd[n] = N, a[n] = Mat{A, NN, N, 1}, b[n] = Mat{H, NN, N, 1}, ++n;
    }
    if (n > 0) {
      rc = mm<T, T>(B, N, N, n, kd, a, b, dA, NN, N, 1, st, EwHook(), "k_tc_gemm:hosc:dA", true);
      if (rc) return rc;
    }
  }
  return launch_status();
}

}  // namespace
}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_hosc_loss_saved_bytes(int64_t B, int64_t N, int64_t K, int terms, int dtype) {
  if (B < 0 || N < 1 || K < 1) return 0;
  return hosc_layout_bytes<HoscSaved>(dtype, B, N, K, terms);
}

size_t tgpb200_hosc_loss_fwd_workspace_bytes(int64_t B, int64_t N, int64_t K, int terms, int dtype) {
  if (B < 0 || N < 1 || K < 1) return 0;
  return hosc_layout_bytes<HoscFwdLayout>(dtype, B, N, K, terms);
}

size_t tgpb200_hosc_loss_bwd_workspace_bytes(int64_t B, int64_t N, int64_t K, int dtype, int need_grad_adj) {
  if (B < 0 || N < 1 || K < 1) return 0;
  return hosc_layout_bytes<HoscBwdLayout>(dtype, B, N, K, need_grad_adj != 0);
}

int tgpb200_hosc_loss_fwd(const void* adj, const void* s, const float* graph_nodes, int64_t B, int64_t N, int64_t K,
                          int dtype, int terms, float eps, float* losses, void* saved, size_t saved_bytes,
                          void* workspace, size_t workspace_bytes, tgpb200_stream_t stream) {
  int rc = hosc_check(adj, s, B, N, K, dtype, terms);
  if (rc != TGPB200_OK) return rc;
  if (!losses) return TGPB200_ERR_INVALID;
  Workspace sw(saved, saved_bytes), ws(workspace, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TGPB200_F32) {
    const HoscSaved<float> sv(sw, B, N, K, terms);
    const HoscFwdLayout<float> l(ws, B, N, K, terms);
    if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
    return hosc_fwd<float>((const float*)adj, (const float*)s, graph_nodes, (int)B, (int)N, (int)K, terms, eps, losses,
                           sv, l, st);
  }
  const HoscSaved<__nv_bfloat16> sv(sw, B, N, K, terms);
  const HoscFwdLayout<__nv_bfloat16> l(ws, B, N, K, terms);
  if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
  return hosc_fwd<__nv_bfloat16>((const __nv_bfloat16*)adj, (const __nv_bfloat16*)s, graph_nodes, (int)B, (int)N,
                                 (int)K, terms, eps, losses, sv, l, st);
}

int tgpb200_hosc_loss_bwd(const void* adj, const void* s, const float* graph_nodes, const void* saved,
                          size_t saved_bytes, const float* grad_losses, int64_t B, int64_t N, int64_t K, int dtype,
                          int terms, void* grad_s, void* grad_adj, void* workspace, size_t workspace_bytes,
                          tgpb200_stream_t stream) {
  int rc = hosc_check(adj, s, B, N, K, dtype, terms);
  if (rc != TGPB200_OK) return rc;
  if (!grad_s) return TGPB200_ERR_INVALID;
  Workspace sw(const_cast<void*>(saved), saved_bytes), ws(workspace, workspace_bytes);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TGPB200_F32) {
    const HoscSaved<float> sv(sw, B, N, K, terms);
    const HoscBwdLayout<float> l(ws, B, N, K, grad_adj != nullptr);
    if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
    return hosc_bwd<float>((const float*)adj, (const float*)s, graph_nodes, grad_losses, (int)B, (int)N, (int)K, terms,
                           sv, (float*)grad_s, (float*)grad_adj, l, st);
  }
  const HoscSaved<__nv_bfloat16> sv(sw, B, N, K, terms);
  const HoscBwdLayout<__nv_bfloat16> l(ws, B, N, K, grad_adj != nullptr);
  if (!sw.ok || !ws.ok) return TGPB200_ERR_WORKSPACE;
  return hosc_bwd<__nv_bfloat16>((const __nv_bfloat16*)adj, (const __nv_bfloat16*)s, graph_nodes, grad_losses, (int)B,
                                 (int)N, (int)K, terms, sv, (__nv_bfloat16*)grad_s, (__nv_bfloat16*)grad_adj, l, st);
}

}  // extern "C"
