"""Float64 checkers that run ON THE GPU for sizes the CPU oracle cannot finish in seconds.

Test infrastructure only (like ``oracle/``): plain ``torch.float64`` tensor algebra, row-chunked
so that no more than ``chunk x B`` doubles exist at a time.  ``loss_closed_form_f64`` restates
``oracle.contrastive_loss_closed_form`` (SURVEY.md section 8a; reference model.py:242-247 and
baselines/Bleep/models.py:34-43,228-234) and is pinned against it at small B by
``tests/test_loss_gpu.py::test_gpu_checker_equals_cpu_oracle``.
"""
from __future__ import annotations

import numpy as np
import torch


def _lse_merge(m, s, x, dim):
    """Running log-sum-exp state (m, s) merged with the block x along ``dim``."""
    bm = x.max(dim=dim).values
    nm = torch.maximum(m, bm)
    s = s * torch.exp(m - nm) + torch.exp(x - nm.unsqueeze(dim)).sum(dim=dim)
    return nm, s


@torch.no_grad()
def loss_closed_form_f64(S, I, temperature, targets="eye", soft_scale="div", chunk=2048):
    """(loss float, dS float64 [B,D], dI float64 [B,D]) on the device of S, float64 throughout."""
    S = torch.as_tensor(S).double()
    I = torch.as_tensor(I).double()
    dev = S.device
    B = S.shape[0]
    T = float(temperature)
    soft = targets != "eye"
    a = 0.0 if not soft else (1.0 / (2 * T) if soft_scale == "div" else T / 2.0)
    ninf = torch.full((B,), -float("inf"), dtype=torch.float64, device=dev)
    rl = torch.empty(B, dtype=torch.float64, device=dev)
    za = torch.empty(B, dtype=torch.float64, device=dev)
    cm, cs_ = ninf.clone(), torch.zeros(B, dtype=torch.float64, device=dev)
    blocks = [(r0, min(B, r0 + chunk)) for r0 in range(0, B, chunk)]
    for r0, r1 in blocks:                                    # pass 1: rl, cl, za
        Lg = S[r0:r1] @ I.T / T
        rl[r0:r1] = torch.logsumexp(Lg, 1)
        cm, cs_ = _lse_merge(cm, cs_, Lg, 0)
        if soft:
            A = (I[r0:r1] @ I.T + S[r0:r1] @ S.T) * a
            za[r0:r1] = torch.logsumexp(A, 1)
    cl = cm + torch.log(cs_)
    wbar = torch.empty(B, dtype=torch.float64, device=dev)
    csum = torch.zeros(B, dtype=torch.float64, device=dev)
    diag = (S * I).sum(1) / T
    if soft:
        for r0, r1 in blocks:                                # pass 2: wbar, cs
            Lg = S[r0:r1] @ I.T / T
            A = (I[r0:r1] @ I.T + S[r0:r1] @ S.T) * a
            Pt = torch.exp(A - za[r0:r1, None])
            W = rl[r0:r1, None] + cl[None, :] - 2 * Lg
            wbar[r0:r1] = (Pt * W).sum(1)
            csum += Pt.sum(0)
    else:
        wbar = rl + cl - 2 * diag
        csum.fill_(1.0)
    loss = float(wbar.sum() / (2 * B))
    dS = torch.zeros_like(S)
    dI = torch.zeros_like(I)
    ar = torch.arange(B, device=dev)
    for r0, r1 in blocks:                                    # pass 3: gradients
        Lg = S[r0:r1] @ I.T / T
        dLg = torch.exp(Lg - rl[r0:r1, None]) + csum[None, :] * torch.exp(Lg - cl[None, :])
        if soft:
            A = (I[r0:r1] @ I.T + S[r0:r1] @ S.T) * a
            Pt = torch.exp(A - za[r0:r1, None])
            dLg -= 2 * Pt
            W = rl[r0:r1, None] + cl[None, :] - 2 * Lg
            dA = Pt * (W - wbar[r0:r1, None]) / (2 * B)
            dS[r0:r1] += dA @ S * a
            dS += dA.T @ S[r0:r1] * a
            dI[r0:r1] += dA @ I * a
            dI += dA.T @ I[r0:r1] * a
        else:
            dLg[ar[r0:r1] - r0, ar[r0:r1]] -= 2.0
        dLg /= 2 * B
        dS[r0:r1] += dLg @ I / T
        dI += dLg.T @ S[r0:r1] / T
    return loss, dS, dI


def assert_grad_close(got, want, rtol=1e-3, rel_floor=2e-2, abs_cap=1e-4, elem_rtol=2e-3, name=""):
    """Checks of a gradient matrix against its float64 statement (numpy or torch inputs):
      * norm-wise:      ||got - want|| <= rtol ||want||
      * max-normalised: |got - want| <= min(rtol, abs_cap) max|want| EVERYWHERE.  abs_cap = 1e-4 is
        10 x tighter than the north star's 1e-3, so every entry -- however small -- is pinned on the
        scale float32 arithmetic allows: against float64 the reference's own float32 formulation
        (stock PyTorch on the same GPU) measures 0.5e-5 .. 2e-5 here and this library 2.4e-5 .. 7e-5
        at B = 1024 .. 16384 (profiles/r2_loss_accuracy.md, tools/loss_accuracy.py);
      * element-wise RELATIVE: |got - want| <= elem_rtol |want| on every entry with
        |want| > rel_floor max|want|.  Floor and tolerance are where float32 arithmetic can deliver:
        with logits of +-256 every exponent carries ~1.5e-5 of float32 rounding, and at a floor of
        1e-3 the reference's own float32 result already reads 1.2e-3 .. 7.7e-3 (this library
        4.8e-3 .. 1.1e-2); at 1e-2 they read 1.6e-4 .. 9.6e-4 and 6.1e-4 .. 1.04e-3.
    """
    g = torch.as_tensor(got).double().cpu()
    w = torch.as_tensor(want).double().cpu()
    assert g.shape == w.shape, (name, g.shape, w.shape)
    err = (g - w).abs()
    wmax = float(w.abs().max())
    assert float((g - w).norm()) <= rtol * float(w.norm()) + 1e-300, \
        f"{name}: norm-wise {float((g - w).norm() / w.norm()):.3e}"
    assert float(err.max()) <= min(rtol, abs_cap) * wmax + 1e-300, \
        f"{name}: max-normalised {float(err.max() / wmax):.3e}"
    big = w.abs() > rel_floor * wmax
    rel = (err[big] / w.abs()[big])
    assert rel.numel() == 0 or float(rel.max()) <= max(rtol, elem_rtol), \
        f"{name}: element-wise relative {float(rel.max()):.3e} over {int(big.sum())} entries"


def gemm_variant(M, N, batch=1):
    """(cluster, tile width) of the tile kernel mclst_matmul's packed route runs for an M x N x batch
    output on this device (mclst_debug_gemm_variant): (2, 256), (1, 256), (1, 128) or (1, 64)."""
    import ctypes
    from mclstexp_b200 import _lib
    cl, w = ctypes.c_int(), ctypes.c_int()
    _lib.check(_lib.load().mclst_debug_gemm_variant(M, N, batch, ctypes.byref(cl), ctypes.byref(w)),
               "gemm_variant")
    return cl.value, w.value


def matmul_route(call):
    """Runs call() -- one ops.matmul -- under the library's kernel trace and returns the route it took:
    "tf32" (the 3xTF32 kernel that splits inside the K loop) or "packed" (pack_split, then gemm_tn)."""
    from mclstexp_b200 import _lib
    _lib.profile_enable(True)
    try:
        out = call()
        names = [n for n, _ in _lib.profile_collect()]
    finally:
        _lib.profile_enable(False)
    route = {("gemm_tf32",): "tf32", ("pack_split", "gemm_tn"): "packed"}.get(tuple(names))
    assert route is not None, names
    return route, out


from oracle.oracle import find_matches_spec_rows  # noqa: E402,F401  (bank-chunked spec for a few rows)
