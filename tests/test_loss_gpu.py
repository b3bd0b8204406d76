"""Contrastive loss fwd+bwd through the C-ABI against the reference's golden outputs and the
oracle (literal autograd restatement + float64 closed form)."""
import numpy as np
import pytest
import torch

from mclstexp_b200 import loss as mloss, synth
from oracle import oracle
from conftest import golden_checksum, golden_cpu_threads, golden_sha256
from checkers import assert_grad_close, loss_closed_form_f64

pytestmark = pytest.mark.gpu

RTOL = 1e-3      # north star: loss and gradients within 1e-3 relative error under FP32


def _check(S, I, T, targets, scale, ref=None, env=None):
    St = torch.tensor(S, device="cuda", requires_grad=True)
    It = torch.tensor(I, device="cuda", requires_grad=True)
    l = mloss.contrastive_loss(St, It, T, targets, scale)
    assert l.dim() == 0 and l.dtype == torch.float32
    (l * 1.0).backward()
    l64, dS64, dI64 = oracle.contrastive_loss_closed_form(S, I, T, targets, scale)
    np.testing.assert_allclose(l.item(), l64, rtol=RTOL)
    for name, got, want in (("dS", St.grad, dS64), ("dI", It.grad, dI64)):
        # norm-wise, max-normalised AND element-wise relative on every entry above 1e-3 max
        assert_grad_close(got, want, RTOL, name=name)
    if ref is not None:
        np.testing.assert_allclose(l.item(), ref[0], rtol=RTOL)
        np.testing.assert_allclose(St.grad.cpu().numpy(), ref[1], rtol=RTOL, atol=RTOL * np.abs(ref[1]).max())
        np.testing.assert_allclose(It.grad.cpu().numpy(), ref[2], rtol=RTOL, atol=RTOL * np.abs(ref[2]).max())


@pytest.mark.parametrize("case", ["loss_b48", "loss_b65_t07", "loss_b16_t2"])
@pytest.mark.parametrize("tag", ["eye", "soft_div", "soft_mul"])
def test_loss_vs_reference_golden(golden_model, case, tag):
    z, meta = golden_model
    m = meta[case]
    S = synth.embeddings(m["B"], m["D"], m["seed"], "clustered", centres=5)
    I = synth.embeddings(m["B"], m["D"], m["seed"] + 1, "clustered", centres=5)
    if m["scaled"]:
        S *= 0.25
        I *= 0.25
    assert golden_checksum(S, I) == m["checksum"]
    targets = "eye" if tag == "eye" else "soft"
    scale = "mul" if tag.endswith("mul") else "div"
    # the oracle's literal restatement is bit-equal to the reference's gradients (stored as digests)
    with golden_cpu_threads():
        _, dS, dI = oracle.contrastive_loss_ref(S, I, m["T"], targets, scale)
    dS, dI = dS.numpy(), dI.numpy()
    assert golden_sha256(dS) == str(z[f"{case}/{tag}/dS/sha256"])
    assert golden_sha256(dI) == str(z[f"{case}/{tag}/dI/sha256"])
    _check(S, I, m["T"], targets, scale, ref=(z[f"{case}/{tag}/loss"], dS, dI))


@pytest.mark.parametrize("B,D,T,scale_in", [(256, 256, 1.0, 1.0), (1024, 256, 1.0, 1.0), (130, 256, 0.5, 0.3),
                                            (257, 100, 2.0, 1.0), (1, 256, 1.0, 1.0), (2, 8, 1.0, 1.0)])
@pytest.mark.parametrize("targets", ["eye", "soft"])
def test_loss_shapes(B, D, T, scale_in, targets):
    # LayerNorm-like rows (norm 16): logits reach +-256 -- the regime the reference trains in
    S = synth.embeddings(B, D, 50 + B, "clustered", centres=7) * scale_in
    I = synth.embeddings(B, D, 51 + B, "clustered", centres=7) * scale_in
    _check(S, I, T, targets, "div")


@pytest.mark.parametrize("B,mb", [(700, 3), (4096, 64)])
@pytest.mark.parametrize("targets", ["eye", "soft"])
def test_loss_row_blocked_equals_single_block(targets, B, mb):
    """The general pipeline (what a rank of a row-sharded batch runs) with several row blocks forced
    by a small scratch budget (3 MiB -> 128-row blocks at B=700; 64 MiB -> 512-row blocks at B=4096),
    against the float64 closed form.  test_loss_phases_gpu.py drives the same pipeline through the
    row-sharded phases."""
    import subprocess, sys, os
    code = f"""
import sys, torch
sys.path.insert(0, 'tests')
from checkers import assert_grad_close, loss_closed_form_f64
from mclstexp_b200 import loss as mloss, synth
B, D = {B}, 256
S = torch.tensor(synth.embeddings(B, D, 1, 'clustered', centres=9) * 0.5, device='cuda')
I = torch.tensor(synth.embeddings(B, D, 2, 'clustered', centres=9) * 0.5, device='cuda')
St = S.clone().requires_grad_(True); It = I.clone().requires_grad_(True)
l = mloss.contrastive_loss(St, It, 1.0, '{targets}'); l.backward()
l64, dS64, dI64 = loss_closed_form_f64(S, I, 1.0, '{targets}')
assert abs(l.item() - l64) <= 1e-3 * abs(l64), (l.item(), l64)
assert_grad_close(St.grad, dS64, 1e-3, name='dS')
assert_grad_close(It.grad, dI64, 1e-3, name='dI')
print('ok')
"""
    env = dict(os.environ, MCLST_LOSS_SCRATCH_MB=str(mb))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_loss_no_grad_path():
    S = torch.tensor(synth.embeddings(64, 256, 3), device="cuda")
    I = torch.tensor(synth.embeddings(64, 256, 4), device="cuda")
    l = mloss.contrastive_loss(S, I, 1.0, "soft")
    l64, _, _ = oracle.contrastive_loss_closed_form(S.cpu().numpy(), I.cpu().numpy(), 1.0, "soft")
    np.testing.assert_allclose(l.item(), l64, rtol=RTOL)


def test_gpu_checker_equals_cpu_oracle():
    """Pins tests/checkers.py (float64 on the GPU, row-chunked) against the CPU oracle's closed form."""
    S = synth.embeddings(300, 64, 1, "clustered", centres=5) * 0.5
    I = synth.embeddings(300, 64, 2, "clustered", centres=5) * 0.5
    for targets, scale in (("eye", "div"), ("soft", "div"), ("soft", "mul")):
        l, dS, dI = loss_closed_form_f64(torch.tensor(S, device="cuda"), torch.tensor(I, device="cuda"),
                                         0.7, targets, scale, chunk=128)
        l64, dS64, dI64 = oracle.contrastive_loss_closed_form(S, I, 0.7, targets, scale)
        assert abs(l - l64) <= 1e-12 * abs(l64)
        assert_grad_close(dS, dS64, rtol=1e-9, elem_rtol=1e-9, name="dS")
        assert_grad_close(dI, dI64, rtol=1e-9, elem_rtol=1e-9, name="dI")


def _big_inputs(B, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    c = 4.0 * torch.randn(64, 256, generator=g, device="cuda")

    def emb():
        x = c[torch.randint(0, 64, (B,), generator=g, device="cuda")] + torch.randn(B, 256, generator=g, device="cuda")
        x = x - x.mean(1, keepdim=True)
        return x / x.std(1, keepdim=True, unbiased=False)      # LayerNorm-like rows: norm 16, logits to +-256
    return emb(), emb()


@pytest.mark.parametrize("B", [4096, 8192, 32768])
@pytest.mark.parametrize("targets", ["eye", "soft"])
def test_loss_at_size_vs_f64(B, targets):
    """The sizes BASELINE cfg5 is quoted on (VERDICT r1 weak 2): loss, dS, dI against the float64
    closed form evaluated on the GPU in row chunks."""
    S, I = _big_inputs(B, 100 + B)
    St, It = S.clone().requires_grad_(True), I.clone().requires_grad_(True)
    l = mloss.contrastive_loss(St, It, 1.0, targets)
    l.backward()
    l64, dS64, dI64 = loss_closed_form_f64(S, I, 1.0, targets, chunk=2048)
    assert abs(l.item() - l64) <= RTOL * abs(l64), (l.item(), l64)
    assert_grad_close(St.grad, dS64, RTOL, name=f"dS B={B}")
    assert_grad_close(It.grad, dI64, RTOL, name=f"dI B={B}")


def test_loss_operand_scale_extremes():
    """Embeddings far from the LayerNorm scale (1e-4 x and 30 x): the split-precision operands must
    not lose the small ones or saturate the large ones (VERDICT r1 weak 6)."""
    for mult, T in ((1e-4, 1e-8), (3000.0, 9e6), (1e5, 1e10), (1.0, 1.0)):
        S = synth.embeddings(384, 256, 5, "clustered", centres=7) * np.float32(mult)
        I = synth.embeddings(384, 256, 6, "clustered", centres=7) * np.float32(mult)
        for targets in ("eye", "soft"):
            _check(S, I, T, targets, "div")
