// TopK selection (the producer of the kept-node SelectOutput): per-graph top ceil(ratio * n_g) nodes by descending
// score, ties broken by lower node id.  Reference: tgp/select/topk_select.py:163-203 -> PyG topk (restated in
// oracle/pyg_shim.py: sort by score descending, stable sort by graph, keep the first k_g of every graph), then
// cluster_to_s (tgp/select/base_select.py:56-71) sorts the kept node ids ascending and permutes the cluster ids.
//
// One stable LSD radix sort on the composite key (graph id << 32 | ~orderable(score)) gives the (graph asc, score
// desc, node id asc) order directly; two order-preserving compactions produce the rank list and the node-sorted view.
#include "prims.cuh"

namespace tgp {

static __global__ void k_topk_count(const int64_t* __restrict__ batch, int64_t N, int64_t G, int* __restrict__ cnt) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int64_t g = batch ? batch[i] : 0;
  if (g >= 0 && g < G) atomicAdd(&cnt[g], 1);
}

static __global__ void k_topk_keys(const float* __restrict__ score, const int64_t* __restrict__ batch, int64_t N,
                                   int64_t G, uint64_t* __restrict__ keys) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float s = score[i];
  if (s == 0.f) s = 0.f;  // -0.0 and +0.0 compare equal in torch.sort
  uint32_t u = __float_as_uint(s);
  u ^= (u >> 31) ? 0xffffffffu : 0x80000000u;  // monotone float -> uint
  int64_t g = batch ? batch[i] : 0;
  if (g < 0 || g >= G) g = G - 1;
  keys[i] = ((uint64_t)g << 32) | (uint64_t)(~u);  // descending score inside a graph
}

// k_g = ceil(ratio * n_g) evaluated in fp32 like the reference ((float(ratio) * n.to(x.dtype)).ceil()), or
// int(ratio) when ratio >= 1.
__device__ __forceinline__ int topk_k(float ratio, int n) {
  if (ratio >= 1.f) return (int)ratio;
  return (int)ceilf(__fmul_rn(ratio, (float)n));
}

struct RankPred {
  struct Payload {
    int node;
  };
  const uint64_t* keys;     // sorted
  const uint32_t* perm;     // sorted payload = node id
  const int* ptr;           // graph offsets (exclusive scan of counts)
  float ratio;
  __device__ bool operator()(int64_t p, Payload& out) const {
    int g = (int)(keys[p] >> 32);
    int r = (int)p - ptr[g];
    int n = ptr[g + 1] - ptr[g];
    out.node = (int)perm[p];
    return r < topk_k(ratio, n);
  }
};
struct RankEmit {
  int* sel_rank;  // [N] rank (= cluster id) of a selected node, -1 otherwise (pre-filled)
  __device__ void operator()(int64_t, int pos, const RankPred::Payload& p) const { sel_rank[p.node] = pos; }
};

struct NodePred {
  struct Payload {
    int rank;
  };
  const int* sel_rank;
  __device__ bool operator()(int64_t n, Payload& out) const {
    out.rank = sel_rank[n];
    return out.rank >= 0;
  }
};
struct NodeEmit {
  int64_t* node_index;
  int64_t* cluster_index;
  __device__ void operator()(int64_t n, int pos, const NodePred::Payload& p) const {
    node_index[pos] = n;
    cluster_index[pos] = p.rank;
  }
};

// Workspace of tgpb200_topk_select: the (graph, score) sort, the selection ranks, the graph offsets with their scan,
// and the two compactions (rank -> selected, selected -> outputs).
struct TopkLayout {
  uint64_t *keys0, *keys1;
  uint32_t *vals0, *vals1;
  int* sel_rank;
  int* ptr;
  Workspace sort, scan, tiles1, tiles2;
  TopkLayout(Workspace& ws, int64_t N, int64_t G) {
    const size_t n = (size_t)(N > 0 ? N : 1);
    keys0 = ws.take<uint64_t>(n);
    keys1 = ws.take<uint64_t>(n);
    vals0 = ws.take<uint32_t>(n);
    vals1 = ws.take<uint32_t>(n);
    sel_rank = ws.take<int>(n);
    ptr = ws.take<int>((size_t)(G > 0 ? G : 0) + 2);
    sort = ws.sub(radix_sort_workspace_bytes(N));
    scan = ws.sub(scan_workspace_bytes(G + 1));
    tiles1 = ws.sub(compact_workspace_bytes(N));
    tiles2 = ws.sub(compact_workspace_bytes(N));
  }
};

}  // namespace tgp

using namespace tgp;

extern "C" {

size_t tgpb200_topk_select_workspace_bytes(int64_t N, int64_t G) { return layout_bytes<TopkLayout>(N, G); }

int tgpb200_topk_select(const float* score, const int64_t* batch, int64_t N, int64_t G, float ratio,
                        int64_t* node_index, int64_t* cluster_index, int64_t* count_out, void* workspace,
                        size_t workspace_bytes, tgpb200_stream_t stream) {
  if (N < 0 || G <= 0 || N >= INT32_MAX || G >= INT32_MAX || !count_out || !(ratio > 0.f)) return TGPB200_ERR_INVALID;
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) {
    cudaMemsetAsync(count_out, 0, sizeof(int64_t), st);
    return launch_status();
  }
  if (!score || !node_index || !cluster_index) return TGPB200_ERR_INVALID;
  Workspace ws(workspace, workspace_bytes);
  const TopkLayout l(ws, N, G);
  if (!ws.ok) return TGPB200_ERR_WORKSPACE;
  const size_t n = (size_t)N;
  uint64_t *keys0 = l.keys0, *keys1 = l.keys1;
  uint32_t *vals0 = l.vals0, *vals1 = l.vals1;
  int* sel_rank = l.sel_rank;
  int* ptr = l.ptr;
  unsigned grid = (unsigned)ceil_div(N, 256);
  cudaMemsetAsync(ptr, 0, (size_t)(G + 1) * sizeof(int), st);
  launch("k_topk_count", k_topk_count, grid, 256, 0, st, batch, N, G, ptr);
  int rc = exclusive_scan_i32(ptr, ptr, G + 1, nullptr, nullptr, l.scan, st);
  if (rc) return rc;
  launch("k_topk_keys", k_topk_keys, grid, 256, 0, st, score, batch, N, G, keys0);
  int gbits = 0;
  while (((int64_t)1 << gbits) < G) ++gbits;
  bool in1 = false;
  rc = radix_sort_pairs<uint64_t>(keys0, nullptr, vals0, keys1, vals1, N, 32 + gbits, &in1, l.sort, st);
  if (rc) return rc;
  cudaMemsetAsync(sel_rank, 0xff, n * sizeof(int), st);
  RankPred rp{in1 ? keys1 : keys0, in1 ? vals1 : vals0, ptr, ratio};
  RankEmit re{sel_rank};
  rc = compact_count(rp, N, l.tiles1, nullptr, nullptr, st);
  if (rc) return rc;
  rc = compact_emit(rp, re, N, l.tiles1, st);
  if (rc) return rc;
  NodePred np{sel_rank};
  NodeEmit ne{node_index, cluster_index};
  rc = compact_count(np, N, l.tiles2, nullptr, count_out, st);
  if (rc) return rc;
  return compact_emit(np, ne, N, l.tiles2, st);
}

}  // extern "C"
