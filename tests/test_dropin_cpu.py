"""CPU: ``patch_pooler`` on stand-ins of the reference pooler classes (tests/dropin_harness.py): operator swap,
preserved ctor attributes, reduce op derived from the existing reducer, unsupported aggregators left alone, and a
dense pooler lacking an attribute its fused forward reads keeps the reference forward."""
import pytest

import dropin_harness as H
import tgp_b200 as T


def test_patch_pooler_swaps_and_preserves_attributes():
    p = H.TopkPooling(reducer=H.BaseReduce(), connector=H.SparseConnect("mean", False, True, True))
    p.preconnector = H.SparseConnect("max", True, False, False)
    T.patch_pooler(p)
    assert isinstance(p.reducer, T.B200Reduce) and p.reducer.reduce_op == "sum"
    c = p.connector
    assert isinstance(c, T.B200SparseConnect)
    assert (c.reduce_op, c.remove_self_loops, c.edge_weight_norm, c.degree_norm) == ("mean", False, True, True)
    assert isinstance(p.preconnector, T.B200SparseConnect) and p.preconnector.reduce_op == "max"
    assert "reduce_op=mean" in repr(c)


def test_patch_pooler_derives_reduce_op_and_leaves_unknown_aggregators():
    p = H.TopkPooling(reducer=H.AggrReduce(H.MeanAggregation()), connector=H.SparseConnect())
    T.patch_pooler(p)
    assert isinstance(p.reducer, T.B200Reduce) and p.reducer.reduce_op == "mean"
    q = H.TopkPooling(reducer=H.AggrReduce(H.LSTMAggregation()), connector=H.SparseConnect())
    T.patch_pooler(q)
    assert isinstance(q.reducer, H.AggrReduce) and q.reduce() == "reference AggrReduce ran"
    r = H.TopkPooling(reducer=H.AggrReduce(H.LSTMAggregation()), connector=H.SparseConnect())
    T.patch_pooler(r, reduce_op="max")  # explicit override
    assert r.reducer.reduce_op == "max"


def test_patch_pooler_dense_gets_fused_forward():
    p = H.MinCutPooling(reducer=H.BaseReduce(), connector=H.DenseConnect(True, False, True, True, False))
    ref_forward = p.forward
    T.patch_pooler(p)
    c = p.connector
    assert isinstance(c, T.B200DenseConnect)
    assert (c.remove_self_loops, c.degree_norm, c.adj_transpose, c.edge_weight_norm, c.sparse_output) == (
        True, False, True, True, False)
    assert p.forward is not ref_forward
    q = H.MinCutPooling(reducer=H.BaseReduce(), connector=H.DenseConnect())
    T.patch_pooler(q, fuse_dense=False)
    with pytest.raises(AssertionError):
        q.forward()
    with pytest.raises(TypeError):
        T.B200DenseConnect(sparse_output="yes")


@pytest.mark.parametrize("name, attrs", [
    ("DMoNPooling", {}),                                   # no loss coefficient
    ("AsymCheegerCutPooling", {"totvar_coeff": 1.0}),      # balance_coeff missing
    ("HOSCPooling", {"mu": 0.1, "alpha": 0.5}),            # hosc_ortho missing
], ids=["dmon", "acc", "hosc"])
def test_pooler_without_attributes_keeps_reference_forward(name, attrs):
    pooler = type(name, (H._DenseBase,), attrs)(selector=None, reducer=H.BaseReduce(), connector=H.DenseConnect())
    ref = pooler.forward
    T.patch_pooler(pooler)
    assert pooler.forward == ref


def test_select_output_rejects_inverse_and_keeps_extras_on_to():
    import torch

    so = T.SelectOutput(cluster_index=torch.tensor([0, 1, 0]), num_supernodes=2, theta=torch.ones(2), tag="x")
    moved = so.to("cpu")
    assert moved.tag == "x" and torch.equal(moved.theta, torch.ones(2)) and moved.num_supernodes == 2
    with pytest.raises(ValueError):
        T.SelectOutput(cluster_index=torch.tensor([0, 1, 0]), num_supernodes=2, s_inv_op="inverse")
    s = torch.sparse_coo_tensor(torch.tensor([[0, 1, 2], [0, 1, 0]]), torch.ones(3), (3, 2)).coalesce()
    so2 = T.SelectOutput(s=s, weight=torch.tensor([1.0, 2.0, 3.0]), num_supernodes=5)
    assert so2.num_supernodes == 5 and torch.equal(so2.weight, torch.tensor([1.0, 2.0, 3.0]))
