"""mclst_matmul (ops.matmul) on every kernel it chooses between, against exact and float64 references.

A product takes the 3xTF32 kernel (csrc/gemm_tf32.cu) or is packed into fp16 hi/lo images and run on
one of four tile kernels (csrc/gemm.cu): CTA pairs at 128 x 256 tiles, or one CTA at 128 x 256,
128 x 128 or 128 x 64.  Shapes are picked through mclst_debug_gemm_variant, so every kernel stays
covered on a part with another SM count, and each call checks the route it took in the kernel trace.

  * exact: small-integer operands, bias and residual and alpha in {1, 0.5, -2} make every product,
    partial sum and power-of-two operand factor exact in fp16, TF32 and fp32, so the result must
    equal the float64 product bit for bit -- a wrong tile, batch offset, missing K block or stale
    accumulator shows as a wrong integer;
  * canaries: operands are views into NaN-filled buffers (a read past K, M, N or the batch poisons
    the result) and out / residual are views into sentinel-filled buffers that must stay bit-unchanged;
  * random data: the element-wise bound |C - C64| <= TAU |alpha| (|A| |B|^T) + epilogue rounding, which
    the fp16 product without the lo terms and a result missing one K block both violate by 10x.
"""
import functools
import os
import subprocess
import sys
import zlib

import pytest
import torch

from checkers import gemm_variant, matmul_route
from mclstexp_b200 import ops

pytestmark = pytest.mark.gpu

TILES = {"pair": (2, 256), "w256": (1, 256), "w128": (1, 128), "w64": (1, 64)}
KERNELS = list(TILES) + ["tf32"]
ORDERS = [(False, False), (False, True), (True, False), (True, True)]
SENTINEL = 0x7FC0BEEF                    # a NaN payload no kernel writes
# Worst ratio |C - C64| / (|alpha| |A| |B|^T), epilogue rounding taken off, over every case of
# test_random_operands_within_float64_bound on one B200 (1000 W power limit): 2.03e-6 on the packed
# route (the 128 x 256 kernels at K = 1097; 1.3e-6 on the 128 x 128 and 128 x 64 kernels), 2.29e-6 on
# the 3xTF32 route.  TAU is 1.75x the larger; the fp16-only product must still exceed it by 10x.
TAU = 4e-6
EPS32 = 2.0 ** -24


@functools.lru_cache(None)
def shape(kernel, batched):
    """(M, N, batch) of a product that runs on `kernel`.  Batched: M = 300 (three row tiles: the last
    pair of a 2-CTA grid has a ghost partner), N = 700 (ragged at 64, 128 and 256), the smallest batch
    > 1 that gives the kernel.  Unbatched: M = 300, or M = 2100 (17 row tiles) for the 256-wide kernels,
    and the smallest N from 700 up in steps of 100."""
    if kernel == "tf32":
        return (300, 700, 3) if batched else (300, 700, 1)
    want = TILES[kernel]
    if batched:
        return 300, 700, next(b for b in range(2, 1 << 16) if gemm_variant(300, 700, b) == want)
    M = 2100 if want[1] == 256 else 300
    return M, next(n for n in range(700, 1 << 20, 100) if gemm_variant(M, n, 1) == want), 1


def contraction_lengths(kernel, batched):
    """K values for the kernel: 333 and 1097 pack through the register fast path (K <= 1024) and the
    two-pass slow path, neither a multiple of the 64-wide K block, and K % 4 != 0 keeps even a short
    or batched-long contraction off the 3xTF32 kernel.  That kernel itself takes K = 252 (short) or
    a batched K = 1100."""
    if kernel == "tf32":
        return (1100,) if batched else (252,)
    return (333, 1097)


CASES = [(k, bt, K) for k in KERNELS for bt in (False, True) for K in contraction_lengths(k, bt)]


def seed_of(*key):
    return zlib.crc32(repr(key).encode()) & 0x7FFFFFFF


def _ids(case):
    return f"{case[0]}-{'batched' if case[1] else 'single'}-K{case[2]}"


def fenced(values):
    """values [nb, r, c] as a view into a NaN-filled buffer with one more batch entry, a row above,
    two rows below and at least five columns to the right (row stride a multiple of 4)."""
    nb, r, c = values.shape
    ld = (c + 5 + 3) // 4 * 4
    buf = torch.full((nb + 1, r + 3, ld), float("nan"), device="cuda")
    view = buf[:nb, 1:r + 1, :c]
    view.copy_(values)
    return view


def canvas(nb, M, N, layout):
    """(buffer, view): an [nb, M, N] view into a sentinel-filled buffer with one more batch entry, a
    row above and two below, and extra columns on both sides.  layout "aligned": 16-byte aligned base
    and row stride; "ldc_odd": row stride % 4 == 1; "base_off": base 4 bytes past a 16-byte boundary."""
    c0 = 1 if layout == "base_off" else 4
    ldc = (N + 8 + 3) // 4 * 4 + (1 if layout == "ldc_odd" else 0)
    buf = torch.full((nb + 1, M + 3, ldc), SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)
    return buf, buf[:nb, 1:M + 1, c0:c0 + N]


def assert_canvas_intact(buf, view, name):
    bits = buf.view(torch.int32)
    outside = torch.ones_like(bits, dtype=torch.bool)
    nb, M, N = view.shape
    r0, c0 = divmod(view.storage_offset(), buf.stride(1))
    outside[:nb, r0:r0 + M, c0:c0 + N] = False
    changed = int((bits[outside] != SENTINEL).sum())
    assert changed == 0, f"{name}: {changed} elements outside the [{nb}, {M}, {N}] view were written"


def operands(M, N, K, nb, a_trans, b_trans, seed, integer=True):
    """NaN-fenced A and B in the requested storage orders and the float64 op(A), op(B) ([nb, M, K],
    [nb, N, K]).  Integer data: |x| <= 4, with whole rows of op(A) scaled by 1, 2 or 4 and rows of op(B)
    by 1, 1/2 or 1/4 (different per-row operand factors), and one zero row in each."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    if integer:
        a = torch.randint(-4, 5, (nb, M, K), generator=g, device="cuda").float()
        b = torch.randint(-4, 5, (nb, N, K), generator=g, device="cuda").float()
        a *= torch.pow(2.0, torch.randint(0, 3, (nb, M, 1), generator=g, device="cuda").float())
        b *= torch.pow(2.0, -torch.randint(0, 3, (nb, N, 1), generator=g, device="cuda").float())
        a[:, M // 2] = 0
        b[:, N // 3] = 0
    else:
        a = torch.randn(nb, M, K, generator=g, device="cuda")
        b = torch.randn(nb, N, K, generator=g, device="cuda")
    A = fenced(a.transpose(1, 2).contiguous() if a_trans else a)
    B = fenced(b.transpose(1, 2).contiguous() if b_trans else b)
    if nb == 1:
        A, B = A[0], B[0]
    return A, B, a.double(), b.double()


def run(kernel, A, B, a_trans, b_trans, **kw):
    """ops.matmul, asserting the route it took: the 3xTF32 kernel for "tf32", pack + tile kernel otherwise."""
    route, out = matmul_route(lambda: ops.matmul(A, B, a_trans, b_trans, **kw))
    assert route == ("tf32" if kernel == "tf32" else "packed"), (kernel, route)
    return out


def as3(t):
    return t if t.dim() == 3 else t[None]


@pytest.mark.parametrize("a_trans,b_trans", ORDERS)
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_exact_products_and_canaries(case, a_trans, b_trans):
    kernel, batched, K = case
    M, N, nb = shape(kernel, batched)
    if kernel != "tf32":
        assert gemm_variant(M, N, nb) == TILES[kernel]
    seed = seed_of(kernel, batched, K, a_trans, b_trans)
    A, B, a64, b64 = operands(M, N, K, nb, a_trans, b_trans, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    alpha = (1.0, 0.5, -2.0)[seed % 3]
    bias = torch.randint(-8, 9, (N,), generator=g, device="cuda").float()
    res = torch.randint(-8, 9, (nb, M, N), generator=g, device="cuda").float()
    prod = torch.bmm(a64, b64.transpose(1, 2))
    squeeze = (lambda t: t) if batched else (lambda t: t[0])

    obuf, out = canvas(nb, M, N, "aligned")
    rbuf, r = canvas(nb, M, N, "aligned")
    r.copy_(res)
    run(kernel, A, B, a_trans, b_trans, alpha=alpha, bias=bias, residual=squeeze(r), out=squeeze(out))
    want = alpha * prod + bias.double() + res.double()
    bad = int((out.double() != want).sum())
    assert bad == 0, f"{bad} of {want.numel()} elements differ from the exact product"
    assert_canvas_intact(obuf, out, "out")
    assert_canvas_intact(rbuf, r, "residual")
    assert torch.equal(r, res), "the residual was written"

    # in place, the dK / dV and .grad accumulation pattern: out is residual
    run(kernel, A, B, a_trans, b_trans, alpha=alpha, residual=squeeze(r), out=squeeze(r))
    bad = int((r.double() != alpha * prod + res.double()).sum())
    assert bad == 0, f"in place: {bad} elements differ from the exact product"
    assert_canvas_intact(rbuf, r, "in-place out")

    if K <= 333:
        # GELU: exact pre-activation, then the float32 erf against float64
        got = as3(run(kernel, A, B, a_trans, b_trans, alpha=alpha, bias=bias, act="gelu",
                      residual=squeeze(res)))
        pre = alpha * prod + bias.double()
        want = torch.nn.functional.gelu(pre) + res.double()
        err = (got.double() - want).abs()
        assert (err <= 2e-6 * (pre.abs() + res.abs().double() + 1)).all(), float(err.max())


@pytest.mark.parametrize("batched", [False, True], ids=["single", "batched"])
@pytest.mark.parametrize("layout", ["ldc_odd", "base_off"])
@pytest.mark.parametrize("kernel", KERNELS)
def test_exact_products_scalar_stores(kernel, layout, batched):
    """Outputs the epilogues cannot store 16 bytes at a time: row stride % 4 != 0, or a base that is
    not 16-byte aligned (then the residual, with the same strides, is misaligned too)."""
    M, N, nb = shape(kernel, batched)
    K = contraction_lengths(kernel, batched)[0]
    seed = seed_of(kernel, layout, batched)
    A, B, a64, b64 = operands(M, N, K, nb, False, True, seed)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    bias = torch.randint(-8, 9, (N,), generator=g, device="cuda").float()
    res = torch.randint(-8, 9, (nb, M, N), generator=g, device="cuda").float()
    squeeze = (lambda t: t) if batched else (lambda t: t[0])
    obuf, out = canvas(nb, M, N, layout)
    rbuf, r = canvas(nb, M, N, layout)
    r.copy_(res)
    run(kernel, A, B, False, True, alpha=-2.0, bias=bias, residual=squeeze(r), out=squeeze(out))
    want = -2.0 * torch.bmm(a64, b64.transpose(1, 2)) + bias.double() + res.double()
    assert int((out.double() != want).sum()) == 0
    assert_canvas_intact(obuf, out, "out")
    assert_canvas_intact(rbuf, r, "residual")
    run(kernel, A, B, False, True, alpha=0.5, residual=squeeze(r), out=squeeze(r))
    assert int((r.double() != 0.5 * torch.bmm(a64, b64.transpose(1, 2)) + res.double()).sum()) == 0
    assert_canvas_intact(rbuf, r, "in-place out")


def bound_ratio(got, want, absprod, alpha, extra):
    """Worst |got - want| / (|alpha| |A| |B|^T) once the epilogue's own rounding (two float32
    roundings of values no larger than |alpha A B^T| + |bias| + |residual|) is taken off."""
    err = (got.double() - want).abs() - 2 * EPS32 * extra
    return float((err.clamp(min=0) / (abs(alpha) * absprod)).max())


@pytest.mark.parametrize("a_trans,b_trans", [(False, False), (True, True)], ids=["nn", "tt"])
@pytest.mark.parametrize("case", CASES, ids=_ids)
def test_random_operands_within_float64_bound(case, a_trans, b_trans):
    kernel, batched, K = case
    M, N, nb = shape(kernel, batched)
    seed = seed_of("random", kernel, batched, K, a_trans)
    A, B, a64, b64 = operands(M, N, K, nb, a_trans, b_trans, seed, integer=False)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    bias = torch.randn(N, generator=g, device="cuda")
    res = torch.randn(nb, M, N, generator=g, device="cuda")
    squeeze = (lambda t: t) if batched else (lambda t: t[0])
    alpha = 0.75
    prod = torch.bmm(a64, b64.transpose(1, 2))
    absprod = torch.bmm(a64.abs(), b64.abs().transpose(1, 2))
    want = alpha * prod + bias.double() + res.double()
    extra = (alpha * prod).abs() + bias.double().abs() + res.double().abs()
    got = as3(run(kernel, A, B, a_trans, b_trans, alpha=alpha, bias=bias, residual=squeeze(res)))
    ratio = bound_ratio(got, want, absprod, alpha, extra)
    assert ratio <= TAU, (ratio, TAU)
    # the bound rejects a result that lost one K block ...
    kb = slice(64, 128)
    dropped = want - alpha * torch.bmm(a64[..., kb], b64[..., kb].transpose(1, 2))
    assert bound_ratio(dropped, want, absprod, alpha, extra) >= 10 * TAU
    if kernel != "tf32":
        # ... and the packed product without its lo terms (fp16 operands, hi x hi only)
        fast = as3(run(kernel, A, B, a_trans, b_trans, alpha=alpha, bias=bias, residual=squeeze(res),
                       precise=False))
        fast_ratio = bound_ratio(fast, want, absprod, alpha, extra)
        assert fast_ratio >= 10 * TAU, (ratio, fast_ratio)


def test_parameter_set_reaches_all_five_kernels():
    """On this device the shapes above reach the 3xTF32 kernel and all four packed tile kernels."""
    reached = set()
    for kernel, batched, K in CASES:
        M, N, nb = shape(kernel, batched)
        lead = (nb,) if batched else ()
        a = torch.randn(lead + (M, K), device="cuda")
        b = torch.randn(lead + (N, K), device="cuda")
        route, _ = matmul_route(lambda: ops.matmul(a, b))
        reached.add("tf32" if route == "tf32" else "packed cluster=%d width=%d" % gemm_variant(M, N, nb))
    print("kernels reached:", sorted(reached))
    assert reached == {"tf32", "packed cluster=2 width=256", "packed cluster=1 width=256",
                       "packed cluster=1 width=128", "packed cluster=1 width=64"}, reached


FORCED_PAIRS = """
import sys
sys.path.insert(0, 'tests')
from checkers import gemm_variant
import test_matmul_routes_gpu as t
for M, N, nb, K in [(100, 700, 1, 333), (64, 300, 3, 1097), (300, 700, 1, 1097), (300, 700, 2, 333),
                    (2100, 700, 1, 333)]:
    assert gemm_variant(M, N, nb) == (2, 256), (M, N, nb)
    t.check_exact_forced(M, N, nb, K)
print('ok')
"""


def check_exact_forced(M, N, nb, K):
    """Exact answer and canaries of one product on whatever kernel this process is forced to."""
    for a_trans, b_trans in ORDERS:
        seed = seed_of("forced", M, N, nb, K, a_trans, b_trans)
        A, B, a64, b64 = operands(M, N, K, nb, a_trans, b_trans, seed)
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        res = torch.randint(-8, 9, (nb, M, N), generator=g, device="cuda").float()
        squeeze = (lambda t: t) if nb > 1 else (lambda t: t[0])
        obuf, out = canvas(nb, M, N, "aligned")
        rbuf, r = canvas(nb, M, N, "aligned")
        r.copy_(res)
        run("pair", A, B, a_trans, b_trans, alpha=0.5, residual=squeeze(r), out=squeeze(out))
        want = 0.5 * torch.bmm(a64, b64.transpose(1, 2)) + res.double()
        assert int((out.double() != want).sum()) == 0, (M, N, nb, K, a_trans, b_trans)
        assert_canvas_intact(obuf, out, "out")
        assert_canvas_intact(rbuf, r, "residual")


def test_forced_pairs_exact():
    """MCLST_GEMM_CLUSTER=2 sends every packed product to the 2-CTA kernel: single row tiles (every
    partner a ghost), odd row-tile counts, batches."""
    env = dict(os.environ, MCLST_GEMM_CLUSTER="2")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", FORCED_PAIRS], env=env, cwd=root, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr
