"""Split-precision tcgen05 GEMM against a float64 product."""
import numpy as np
import pytest
import torch

from checkers import matmul_route
from mclstexp_b200 import ops

pytestmark = pytest.mark.gpu
ROUTES = ["tf32", "packed"]


def misaligned(t):
    """A copy of the row-major matrix t whose base and rows are not 16-byte aligned: keeps a product
    off the 3xTF32 kernel, which loads plain operands 16 bytes at a time."""
    v = torch.empty(t.shape[0], t.shape[1] + 1, device="cuda")[:, 1:]
    return v.copy_(t)


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (1, 1, 1), (37, 300, 171), (1024, 1536, 785),
                                   (129, 257, 1000), (1024, 256, 2048), (300, 1000, 512)])
def test_matmul_nt_precise(M, N, K):
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g)
    want = a.double() @ b.double().T
    got = ops.matmul_nt(a.cuda(), b.cuda()).cpu().double()
    err = (got - want).abs().max().item()
    scale = want.abs().max().item()
    assert err <= 3e-5 * scale + 1e-6, (err, scale)     # fp32-GEMM-level: far inside the 1e-3 budget
    fast = ops.matmul_nt(a.cuda(), b.cuda(), precise=False).cpu().double()
    assert (fast - want).abs().max().item() <= 2e-3 * scale + 1e-3


def test_matmul_nt_epilogue():
    """Bias, GELU and residual on both routes: the aligned operands take the 3xTF32 kernel, a
    misaligned copy of A the packed one."""
    g = torch.Generator().manual_seed(5)
    M, N, K = 200, 333, 96
    a, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) * 0.2
    bias, res = torch.randn(N, generator=g), torch.randn(M, N, generator=g)
    want = torch.nn.functional.gelu(0.5 * a.double() @ b.double().T + bias.double()) + res.double()
    for route in ROUTES:
        a_dev = a.cuda() if route == "tf32" else misaligned(a.cuda())
        taken, got = matmul_route(lambda: ops.matmul_nt(a_dev, b.cuda(), alpha=0.5, bias=bias.cuda(), act="gelu",
                                                        residual=res.cuda()))
        assert taken == route
        got = got.cpu().double()
        assert (got - want).abs().max().item() <= 5e-6 * want.abs().max().item(), route


def test_matmul_nt_strided_views():
    g = torch.Generator().manual_seed(6)
    big_a, big_b = torch.randn(70, 300, generator=g).cuda(), torch.randn(90, 300, generator=g).cuda()
    a, b = big_a[:, 10:138], big_b[:, 20:148]
    out = torch.zeros(70, 128, device="cuda")[:, :90]
    ops.matmul_nt(a, b, out=out)
    want = a.double() @ b.double().T
    assert (out.double() - want).abs().max().item() <= 1e-5 * want.abs().max().item()


@pytest.mark.parametrize("a_trans,b_trans", [(False, True), (True, False), (True, True)])
def test_matmul_transposes(a_trans, b_trans):
    g = torch.Generator().manual_seed(11)
    M, N, K = 150, 200, 333
    a = torch.randn((K, M) if a_trans else (M, K), generator=g).cuda()
    b = torch.randn((K, N) if b_trans else (N, K), generator=g).cuda()
    opa = a.T if a_trans else a
    opb = b.T if b_trans else b
    want = opa.double() @ opb.double().T
    got = ops.matmul(a, b, a_trans, b_trans)
    assert (got.double() - want).abs().max().item() <= 3e-5 * want.abs().max().item()


def test_matmul_batched_head_slices():
    """The attention pattern: per-head [B,64] slices of a [B,1536] qkv matrix."""
    g = torch.Generator().manual_seed(12)
    Bt, H, dh = 300, 8, 64
    qkv = torch.randn(Bt, 3 * H * dh, generator=g).cuda()
    q = qkv[:, :H * dh].view(Bt, H, dh).permute(1, 0, 2)          # [H, B, dh] strided view
    k = qkv[:, H * dh:2 * H * dh].view(Bt, H, dh).permute(1, 0, 2)
    v = qkv[:, 2 * H * dh:].view(Bt, H, dh).permute(1, 0, 2)
    dots = ops.matmul(q, k, alpha=0.125)
    want = torch.einsum("hid,hjd->hij", q.double(), k.double()) * 0.125
    assert (dots.double() - want).abs().max().item() <= 3e-5 * want.abs().max().item()
    p = torch.softmax(dots, -1)
    out = torch.empty(Bt, H * dh, device="cuda")
    ov = out.view(Bt, H, dh).permute(1, 0, 2)
    ops.matmul(p, v, b_trans=True, out=ov)                        # [H,B,B] x [H,B(K),dh(N)]
    want = torch.einsum("hij,hjd->hid", p.double(), v.double()).permute(1, 0, 2).reshape(Bt, H * dh)
    assert (out.double() - want).abs().max().item() <= 3e-5 * want.abs().max().item()


@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("sa,sb", [(1e-5, 1.0), (1e-5, 1e-5), (1e4, 1e4), (1e-30, 1e20), (3e30, 1e-12)])
@pytest.mark.parametrize("a_trans,b_trans", [(False, False), (True, True)])
def test_matmul_operand_magnitudes(sa, sb, a_trans, b_trans, route):
    """fp16 hi/lo halves have a 5-bit exponent: operands are brought into range with exact
    power-of-two row factors (gemm.cu), so gradients of magnitude 1e-5 and activations of 1e4
    keep fp32-level accuracy (VERDICT r1 weak 6).  The 3xTF32 kernel needs no factors (8-bit
    exponent) and must hold the same accuracy; K % 4 != 0 sends the product to the packed route."""
    g = torch.Generator().manual_seed(21)
    M, N, K = 130, 270, 200 if route == "tf32" else 201
    a = (torch.randn((K, M) if a_trans else (M, K), generator=g) * sa).cuda()
    b = (torch.randn((K, N) if b_trans else (N, K), generator=g) * sb).cuda()
    opa, opb = (a.T if a_trans else a), (b.T if b_trans else b)
    want = opa.double() @ opb.double().T
    taken, got = matmul_route(lambda: ops.matmul(a, b, a_trans, b_trans))
    assert taken == route
    got = got.double()
    assert torch.isfinite(got).all()
    assert (got - want).abs().max().item() <= 3e-5 * want.abs().max().item()


def test_matmul_rows_of_very_different_scale_and_outliers():
    """Row-wise factors: a 1e5 outlier (beyond fp16's 65504) in one row must neither saturate nor
    cost the other rows their precision; rows 1e-6 apart in scale are each accurate on their own
    scale."""
    g = torch.Generator().manual_seed(22)
    M, N, K = 96, 140, 300
    a = torch.randn(M, K, generator=g)
    b = torch.randn(N, K, generator=g)
    a[3, 17] = 1e5
    a[10] *= 1e-6
    b[5] *= 1e6
    b[7, :] = 0.0
    want = a.double() @ b.double().T
    got = ops.matmul_nt(a.cuda(), b.cuda()).cpu().double()
    # every output element against the scale of ITS row and column
    ref = a.double().abs().max(1).values[:, None] * b.double().abs().max(1).values[None, :] * K ** 0.5
    assert ((got - want).abs() <= 3e-5 * ref + 1e-30).all()
    assert (got[:, 7] == 0).all()


def test_matmul_non_finite_inputs_propagate():
    """On both routes: the aligned operands take the 3xTF32 kernel, a misaligned copy of A the packed one."""
    a = torch.randn(40, 64).cuda()
    b = torch.randn(50, 64).cuda()
    a[2, 3] = float("inf")
    b[4, 5] = float("nan")
    for route in ROUTES:
        a_op = a if route == "tf32" else misaligned(a)
        taken, got = matmul_route(lambda: ops.matmul_nt(a_op, b))
        assert taken == route
        assert not torch.isfinite(got[2]).any(), route      # inf * finite sums: inf or NaN, never a finite lie
        assert torch.isnan(got[:, 4]).all(), route
        assert torch.isfinite(got[[0, 1, 3]][:, [0, 1, 2, 3]]).all(), route


@pytest.mark.parametrize("a_trans,b_trans", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("M,N,K,nb", [(1024, 256, 256, 1), (130, 70, 36, 1), (3, 5, 4, 1), (257, 129, 200, 1),
                                      (300, 64, 520, 8), (128, 40, 1024, 3)])
def test_matmul_in_kernel_split_route(M, N, K, nb, a_trans, b_trans):
    """Shapes mclst_matmul sends to the 3xTF32 kernel that splits inside the K loop (gemm_tf32.cu):
    short contractions and large batched operands, every storage order, ragged tile edges, K not a
    multiple of the 32-wide K block, with the full epilogue."""
    g = torch.Generator().manual_seed(M + 3 * N + 5 * K + 7 * nb)
    lead = (nb,) if nb > 1 else ()
    a = torch.randn(lead + ((K, M) if a_trans else (M, K)), generator=g).cuda()
    b = torch.randn(lead + ((K, N) if b_trans else (N, K)), generator=g).cuda()
    bias = torch.randn(N, generator=g).cuda()
    res = torch.randn(lead + (M, N), generator=g).cuda()
    opa = a.transpose(-1, -2) if a_trans else a
    opb = b.transpose(-1, -2) if b_trans else b
    want = torch.nn.functional.gelu(0.25 * opa.double() @ opb.double().transpose(-1, -2) + bias.double()) + res.double()
    got = ops.matmul(a, b, a_trans, b_trans, alpha=0.25, bias=bias, act="gelu", residual=res)
    scale = (0.25 * opa.double() @ opb.double().transpose(-1, -2)).abs().max().item() + 1.0
    # (K / 8 accumulating MMAs per pass, each rounding toward zero: 1.1e-3 absolute at K = 1024 on
    # sums of magnitude 130 -- twice the packed fp16 route, whose MMAs take 16 K at a time)
    assert (got.double() - want).abs().max().item() <= 6e-5 * scale
    # in place: out aliases the residual (gradient accumulation into .grad)
    acc = res.clone()
    ops.matmul(a, b, a_trans, b_trans, out=acc, residual=acc)
    want2 = opa.double() @ opb.double().transpose(-1, -2) + res.double()
    assert (acc.double() - want2).abs().max().item() <= 6e-5 * 4 * scale
