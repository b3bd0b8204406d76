"""The row-sharded contrastive loss (mclst_contrastive_loss_phase: what each rank of
distributed.contrastive_loss_sharded runs on a global batch above REPLICATE_LOSS_BELOW) replayed on
one GPU.  Every emulated rank owns its workspace (its products survive there between the phases);
the ranks share one statistics block, and since each rank writes its own rows of it the all-gathers
between the phases are no-ops.  Checked against the float64 closed form, and for bit-identical
statistics across decompositions of the same batch."""
import ctypes as C

import pytest
import torch

from mclstexp_b200 import _lib, synth
from mclstexp_b200.loss import TARGET_MODES
from checkers import assert_grad_close, loss_closed_form_f64

pytestmark = pytest.mark.gpu

RTOL = 1e-3
LEAN_SAFE_ROWS = (0, 2, 5, 6, 8)     # rl, za, diag, rl_lo, za_lo: the lean path computes these the same way

# per batch size: (rows per emulated rank, scratch budget in MiB or None for the default).  A single
# rank at the default budget is the lean whole-batch path; 64 MiB at B = 4096 makes every rank of
# 1024 rows run two row blocks (512 rows, soft targets; 768 + 256, eye) and one rank eight (six).
SPLITS = {
    1024: [([1024], None), ([512, 512], None), ([256] * 4, None)],
    640: [([640], None), ([128] * 5, None)],
    700: [([700], None), ([384, 316], None)],
    4096: [([4096], None), ([1024] * 4, None), ([1024] * 4, 64), ([4096], 64)],
}
TARGETS = [("eye", "div"), ("soft", "div"), ("soft", "mul")]


def _inputs(B, D=256):
    S = torch.tensor(synth.embeddings(B, D, 1, "clustered", centres=9) * 0.5, device="cuda")
    I = torch.tensor(synth.embeddings(B, D, 2, "clustered", centres=9) * 0.5, device="cuda")
    return S, I


def replay(S, I, T, mode, split, budget_mb, monkeypatch):
    """(loss, dS, dI, stats) of the batch with its rows split over len(split) emulated ranks."""
    if budget_mb is None:
        monkeypatch.delenv("MCLST_LOSS_SCRATCH_MB", raising=False)
    else:
        monkeypatch.setenv("MCLST_LOSS_SCRATCH_MB", str(budget_mb))
    lib = _lib.load()
    B, D = S.shape
    assert sum(split) == B
    stats = torch.zeros((_lib.LOSS_STAT_ROWS, B), dtype=torch.float32, device="cuda")
    dS, dI = torch.empty_like(S), torch.empty_like(I)
    ranks, row0 = [], 0
    for rows in split:
        n = C.c_size_t()
        _lib.check(lib.mclst_contrastive_loss_workspace_bytes(B, D, mode, rows, C.byref(n)), "workspace")
        ranks.append((row0, rows, torch.empty(n.value, dtype=torch.uint8, device="cuda"),
                      torch.zeros((), dtype=torch.float32, device="cuda")))
        row0 += rows
    for phase in ((1, 3) if mode == _lib.T_EYE else (1, 2, 3)):
        for row0, rows, ws, loss in ranks:
            dSr, dIr = dS[row0:row0 + rows], dI[row0:row0 + rows]
            _lib.check(lib.mclst_contrastive_loss_phase(
                _lib.ptr(S), S.stride(0), _lib.ptr(I), I.stride(0), B, D, float(T), mode, row0, rows, phase,
                _lib.ptr(stats), _lib.ptr(loss), _lib.ptr(dSr), dSr.stride(0), _lib.ptr(dIr), dIr.stride(0),
                _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), f"contrastive_loss_phase {phase}")
    torch.cuda.synchronize()
    return sum(float(loss.item()) for *_, loss in ranks), dS, dI, stats


def _name(B, split, budget_mb):
    return f"B={B} rows={split[0]}x{len(split)}" + (f" last={split[-1]}" if split[-1] != split[0] else "") + \
        (f" {budget_mb} MiB" if budget_mb else "")


@pytest.mark.parametrize("T", [1.0, 0.5])
@pytest.mark.parametrize("targets,scale", TARGETS)
@pytest.mark.parametrize("B", sorted(SPLITS))
def test_loss_phases_replay_vs_f64(B, targets, scale, T, monkeypatch):
    S, I = _inputs(B)
    l64, dS64, dI64 = loss_closed_form_f64(S, I, T, targets, scale)
    for split, mb in SPLITS[B]:
        name = _name(B, split, mb)
        loss, dS, dI, _ = replay(S, I, T, TARGET_MODES[(targets, scale)], split, mb, monkeypatch)
        assert abs(loss - l64) <= RTOL * abs(l64), (name, loss, l64)
        assert_grad_close(dS, dS64, RTOL, name=f"dS {name}")
        assert_grad_close(dI, dI64, RTOL, name=f"dI {name}")


@pytest.mark.parametrize("T", [1.0, 0.5])
@pytest.mark.parametrize("targets,scale", TARGETS)
@pytest.mark.parametrize("B", sorted(SPLITS))
def test_loss_phases_decomposition_invariant(B, targets, scale, T, monkeypatch):
    """Every row's statistics come from the epilogue partials of the same 256-wide product tiles and
    the same merge, whatever the number of ranks and row blocks: the stats block and the gradients
    are bit-identical across decompositions.  The lean whole-batch path (one rank, default budget)
    takes the column statistics (and so wbar, cs) from a column sweep instead; its row statistics
    must still match bit for bit."""
    S, I = _inputs(B)
    mode = TARGET_MODES[(targets, scale)]
    runs = [(_name(B, split, mb), len(split) == 1 and mb is None, replay(S, I, T, mode, split, mb, monkeypatch))
            for split, mb in SPLITS[B]]
    general = [(n, r) for n, lean, r in runs if not lean]
    n0, (_, dS0, dI0, st0) = general[0]
    for n, (_, dS, dI, st) in general[1:]:
        for k in range(_lib.LOSS_STAT_ROWS):
            assert torch.equal(st[k], st0[k]), (f"stats row {k}", n, n0)
        assert torch.equal(dS, dS0), ("dS", n, n0)
        assert torch.equal(dI, dI0), ("dI", n, n0)
    for n, lean, (_, _, _, st) in runs:
        if lean:
            for k in LEAN_SAFE_ROWS:
                assert torch.equal(st[k], st0[k]), (f"stats row {k}", n, n0)
