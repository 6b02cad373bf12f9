"""GPU: the tcgen05 batched GEMM engine against float64 matmul, for every operand-major combination."""
import pytest
import torch

from tgp_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _run(a_store, b_store, a_mn, b_mn, M, N, Kd, out_dtype=torch.float32, alpha=1.0, acc=None, transposed_out=False):
    """a_store: [B, M, Kd] (K-major) or [B, Kd, M] (MN-major); likewise b_store [B, N, Kd] / [B, Kd, N]."""
    B = a_store.size(0)
    if transposed_out:
        out = torch.zeros(B, N, M, dtype=out_dtype, device=DEV)
        obs, ors, ocs = N * M, 1, M
    else:
        out = torch.zeros(B, M, N, dtype=out_dtype, device=DEV) if acc is None else acc.clone()
        obs, ors, ocs = M * N, N, 1
    L.call("tgpb200_tc_gemm", L.ptr(a_store), L.ptr(b_store), L.ptr(out), B, M, N, Kd,
           a_store.stride(0), a_store.stride(1), int(a_mn), b_store.stride(0), b_store.stride(1), int(b_mn),
           obs, ors, ocs, L.dtype_code(a_store.dtype), L.dtype_code(out_dtype), alpha, int(acc is not None), L.stream())
    torch.cuda.synchronize()
    return out


def _ref(a_store, b_store, a_mn, b_mn):
    a = a_store.double().transpose(1, 2) if a_mn else a_store.double()   # [B, M, Kd]
    b = b_store.double() if b_mn else b_store.double().transpose(1, 2)   # [B, Kd, N]
    return a @ b


@pytest.mark.parametrize("a_mn", [False, True])
@pytest.mark.parametrize("b_mn", [False, True])
@pytest.mark.parametrize("B,M,N,Kd", [(1, 128, 64, 32), (3, 256, 64, 256), (2, 64, 128, 96), (5, 128, 256, 72),
                                      (2, 384, 32, 8)])
def test_tc_gemm_fp32_3xtf32(a_mn, b_mn, B, M, N, Kd):
    g = torch.Generator().manual_seed(M + N + Kd)
    a = torch.randn((B, Kd, M) if a_mn else (B, M, Kd), generator=g).to(DEV)
    b = torch.randn((B, Kd, N) if b_mn else (B, N, Kd), generator=g).to(DEV)
    out = _run(a, b, a_mn, b_mn, M, N, Kd)
    ref = _ref(a, b, a_mn, b_mn)
    err = (out.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-6 * scale * max(1.0, (Kd / 64) ** 0.5), f"3xTF32 error {err} vs scale {scale}"


@pytest.mark.parametrize("tma_store", ["1", "0"])
@pytest.mark.parametrize("a_mn", [False, True])
@pytest.mark.parametrize("b_mn", [False, True])
@pytest.mark.parametrize("B,M,N,Kd", [(2, 200, 40, 100), (3, 132, 72, 36), (1, 640, 320, 260), (300, 128, 64, 64)])
def test_tc_gemm_fp32_ragged_shapes_both_engines(tma_store, a_mn, b_mn, B, M, N, Kd):
    """fp32 products with ragged M / N / K (partial tiles, zero-filled TMA tails, several n-tiles, more tiles than
    SMs) on the TMEM-operand engine, through both of its epilogues: a plain row-major output leaves through the
    TMA-store epilogue (tma_store "1"), an accumulated one through the register-store epilogue (tma_store "0")."""
    g = torch.Generator().manual_seed(5 * M + N + Kd)
    a = torch.randn((B, Kd, M) if a_mn else (B, M, Kd), generator=g).to(DEV)
    b = torch.randn((B, Kd, N) if b_mn else (B, N, Kd), generator=g).to(DEV)
    ref = _ref(a, b, a_mn, b_mn)
    scale = ref.abs().max().item()
    if tma_store == "1":
        out = _run(a, b, a_mn, b_mn, M, N, Kd)
    else:
        acc = torch.randn(B, M, N, generator=g).to(DEV)
        out = _run(a, b, a_mn, b_mn, M, N, Kd, alpha=0.5, acc=acc)
        ref = 0.5 * ref + acc.double()
    torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5 * scale)


@pytest.mark.parametrize("pack", ["1", "0"])
@pytest.mark.parametrize("B,M,N,Kd", [(2, 64, 64, 256), (5, 64, 64, 96), (7, 48, 40, 100), (3, 16, 16, 64), (1, 64, 64, 32),
                                      (301, 64, 64, 64)])
def test_tc_gemm_fp32_two_items_per_tile(monkeypatch, pack, B, M, N, Kd):
    """Products with M, N <= 64 (K-major A, MN-major B: the A_raw = T S layout) share a 128 x 128 tile pairwise: odd
    batch counts, ragged M / N / K, a single item (no packing), more tiles than SMs; against the unpacked engine's bound."""
    monkeypatch.setenv("TGPB200_GEMM_PACK2", pack)
    g = torch.Generator().manual_seed(3 * M + N + Kd + B)
    a = torch.randn((B, M, Kd), generator=g).to(DEV)
    b = torch.randn((B, Kd, N), generator=g).to(DEV)
    out = _run(a, b, False, True, M, N, Kd)
    ref = _ref(a, b, False, True)
    scale = ref.abs().max().item()
    torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5 * scale)


@pytest.mark.parametrize("a_mn", [False, True])
@pytest.mark.parametrize("b_mn", [False, True])
def test_tc_gemm_bf16(a_mn, b_mn):
    B, M, N, Kd = 3, 256, 256, 192
    g = torch.Generator().manual_seed(7)
    a = torch.randn((B, Kd, M) if a_mn else (B, M, Kd), generator=g).bfloat16().to(DEV)
    b = torch.randn((B, Kd, N) if b_mn else (B, N, Kd), generator=g).bfloat16().to(DEV)
    out = _run(a, b, a_mn, b_mn, M, N, Kd)
    ref = _ref(a, b, a_mn, b_mn)
    torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-4)  # bf16 inputs are exact, fp32 accumulate
    outb = _run(a, b, a_mn, b_mn, M, N, Kd, out_dtype=torch.bfloat16)
    torch.testing.assert_close(outb.double(), ref, rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("out_bf16", ["1", "0"])
@pytest.mark.parametrize("a_mn", [False, True])
@pytest.mark.parametrize("b_mn", [False, True])
@pytest.mark.parametrize("B,M,N,Kd", [(1, 256, 64, 64), (7, 512, 256, 128), (3, 384, 128, 200), (2, 200, 192, 64),
                                      (160, 256, 128, 64), (2, 1024, 512, 320)])
def test_tc_gemm_bf16_cta_pairs(out_bf16, a_mn, b_mn, B, M, N, Kd):
    """bf16 products with more than one 128-row tile on the bf16 engine: ragged M / N, several n-tiles, more tiles
    than SMs, with and without alpha / accumulation, into a bf16 (out_bf16 "1") or an fp32 output."""
    if (a_mn and M % 8) or (b_mn and N % 8):
        pytest.skip("MN-major rows must be 16-byte multiples")
    odt = torch.bfloat16 if out_bf16 == "1" else torch.float32
    tol = dict(rtol=2e-2, atol=2e-2) if out_bf16 == "1" else dict(rtol=1e-5, atol=2e-4)
    g = torch.Generator().manual_seed(M + 3 * N + Kd)
    a = torch.randn((B, Kd, M) if a_mn else (B, M, Kd), generator=g).bfloat16().to(DEV)
    b = torch.randn((B, Kd, N) if b_mn else (B, N, Kd), generator=g).bfloat16().to(DEV)
    out = _run(a, b, a_mn, b_mn, M, N, Kd, out_dtype=odt)
    ref = _ref(a, b, a_mn, b_mn)
    torch.testing.assert_close(out.double(), ref, **tol)
    acc = torch.randn(B, M, N, generator=g).to(DEV, odt)
    out2 = _run(a, b, a_mn, b_mn, M, N, Kd, out_dtype=odt, alpha=0.5, acc=acc)
    torch.testing.assert_close(out2.double(), 0.5 * ref + acc.double(), **tol)


def test_tc_gemm_alpha_accumulate_and_transposed_output():
    B, M, N, Kd = 2, 128, 64, 64
    g = torch.Generator().manual_seed(9)
    a = torch.randn(B, M, Kd, generator=g).to(DEV)
    b = torch.randn(B, Kd, N, generator=g).to(DEV)
    c = torch.randn(B, M, N, generator=g).to(DEV)
    out = _run(a, b, False, True, M, N, Kd, alpha=0.5, acc=c)
    ref = 0.5 * (a.double() @ b.double()) + c.double()
    torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5)
    outt = _run(a, b, False, True, M, N, Kd, transposed_out=True)
    torch.testing.assert_close(outt.double(), (a.double() @ b.double()).transpose(1, 2), rtol=1e-5, atol=1e-5)


def test_tc_gemm_rejects_unsupported_layout():
    a = torch.randn(1, 8, 101, device=DEV)  # row stride 101 floats: not a multiple of 16 bytes
    b = torch.randn(1, 8, 64, device=DEV)
    out = torch.zeros(1, 101, 64, device=DEV)
    rc = L.load().tgpb200_tc_gemm(L.ptr(a), L.ptr(b), L.ptr(out), 1, 101, 64, 8, 808, 101, 1, 512, 64, 1, 6464, 64, 1,
                                  0, 0, 1.0, 0, L.stream())
    assert rc == -4
