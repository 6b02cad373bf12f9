"""CPU: the C-ABI library loads, exports every symbol include/tgp_b200.h declares, and the host
layer fails loudly on CPU tensors (no fallback).  No kernels are launched here."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "tgp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tgpb200_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    from tgp_b200 import _lib as L

    lib = L.load()
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/tgp_b200.h but not exported"
        assert name in L.SIGNATURES, f"{name} has no ctypes signature"
    assert sorted(L.SIGNATURES) == declared
    assert lib.tgpb200_abi_version() == 2


def test_workspace_queries_are_pure_host_functions():
    from tgp_b200 import _lib as L

    lib = L.load()
    assert lib.tgpb200_build_csr_workspace_bytes(1000, 10) > 0
    assert lib.tgpb200_remap_coalesce_workspace_bytes(10**6, 10**5) > 20 * 10**6
    assert lib.tgpb200_dense_pool_saved_bytes(2, 16, 4) > 0
    assert lib.tgpb200_graph_ptr_workspace_bytes(128) > 0


def test_cpu_tensors_raise_no_fallback():
    import tgp_b200 as T

    so = T.SelectOutput(cluster_index=torch.tensor([0, 1, 0]))
    x = torch.randn(3, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        T.B200Reduce()(x, so)
    with pytest.raises(RuntimeError, match="CUDA"):
        T.B200SparseConnect()(torch.tensor([[0, 1], [1, 2]]), so)
    with pytest.raises(RuntimeError, match="CUDA"):
        T.mincut_pool(torch.randn(1, 4, 2), torch.rand(1, 4, 4), torch.rand(1, 4, 2))


def test_host_side_errors_match_reference():
    import tgp_b200 as T

    so = T.SelectOutput(cluster_index=torch.tensor([0, 1, 0]))
    with pytest.raises(ValueError, match="return_batched"):
        T.B200Reduce()(torch.randn(3, 4), so, return_batched=True)
    with pytest.raises(AssertionError, match="batch_pooled"):
        T.B200SparseConnect(edge_weight_norm=True)(torch.zeros(2, 3, dtype=torch.long), so)
    with pytest.raises(TypeError):
        T.B200DenseConnect(sparse_output="yes")
    with pytest.raises(ValueError, match="batch sizes do not match"):
        T.B200DenseConnect._prepare_batched_dense_inputs(torch.randn(2, 4, 2), torch.randn(3, 4, 4))
    with pytest.raises(ValueError, match="Unknown aggregator"):
        T.B200Reduce("invalid")


def test_select_output_mirror_matches_oracle():
    import tgp_b200 as T
    from oracle import ref_path as R

    torch.manual_seed(0)
    node = torch.tensor([7, 2, 9, 4])
    w = torch.rand(4)
    a = T.SelectOutput(node_index=node, num_nodes=12, cluster_index=torch.arange(4), num_supernodes=4, weight=w)
    b = R.OracleSelectOutput(node_index=node, num_nodes=12, cluster_index=torch.arange(4), num_supernodes=4, weight=w)
    assert torch.equal(a.node_index, b.node_index) and torch.equal(a.cluster_index, b.cluster_index)
    assert torch.equal(a.weight, b.weight) and a.num_nodes == 12 and a.num_supernodes == 4
    assert repr(T.B200Reduce()) == "B200Reduce(reduce_op=sum)"


def test_torch_custom_ops_registered_with_fake_kernels():
    """SURVEY 8b: the path's operators are torch custom ops (dispatcher schemas, fake kernels, autograd)."""
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode

    from tgp_b200 import ops

    for name in ops.OP_NAMES:
        assert hasattr(torch.ops.tgp_b200, name), name
    schema = str(torch.ops.tgp_b200.stas_fused.default._schema)
    assert "Tensor? x" in schema and "Tensor? adj" in schema and "int loss_kind" in schema
    with FakeTensorMode():  # shape propagation without a device (what torch.compile / export trace through)
        s = torch.empty(4, 32, 8, device="cuda")
        x = torch.empty(4, 32, 16, device="cuda")
        a = torch.empty(4, 32, 32, device="cuda")
        xp, ap, losses, saved = torch.ops.tgp_b200.stas_fused(x, a, s, 3, 1, 1.0, 1.0)
        assert xp.shape == (4, 8, 16) and ap.shape == (4, 8, 8) and losses.shape == (4,) and saved.dtype == torch.uint8
        xp, ap, _, _ = torch.ops.tgp_b200.stas_fused(None, a, s, 0, 0, 1.0, 1.0)
        assert xp.numel() == 0 and ap.shape == (4, 8, 8)
        idx = torch.empty(100, dtype=torch.long, device="cuda")
        order, ptr = torch.ops.tgp_b200.build_csr(idx, 7)
        assert order.dtype == torch.int32 and ptr.shape == (8,)
        feats = torch.empty(100, 12, device="cuda")
        assert torch.ops.tgp_b200.segment_reduce(feats, idx, idx, None, order, ptr, 7, 0).shape == (7, 12)
        ei, w, src, cnt = torch.ops.tgp_b200.filter_relabel_edges(idx, idx, None, idx, 50, 1, 1e-8, True, False)
        assert ei.shape == (2, 100) and w.numel() == 0 and cnt.shape == (1,)
        wts = torch.empty(100, device="cuda")
        out = torch.ops.tgp_b200.remap_coalesce(idx, idx, wts, idx, None, None, 100, 7, 0, 1, 1e-8, True, True)
        assert out[0].shape == (2, 100) and out[1].shape == (100,) and out[2].shape == (100,)
        assert torch.ops.tgp_b200.degree_norm(wts, idx, idx, 7, 1e-8, True, None)[0].shape == (100,)
    with pytest.raises(NotImplementedError):  # no CPU kernel by design
        torch.ops.tgp_b200.stas_fused(None, None, torch.zeros(1, 2, 2), 0, 0, 1.0, 1.0)
