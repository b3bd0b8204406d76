"""Multi-GPU forms of the two shardable pieces of the path (SURVEY.md section 8e).

One process per GPU, ``torch.distributed`` (NCCL over NVLink/NVSwitch) for the exchanges.
The reference is single-process (train.py:107) -- these are new capabilities, specified by
the north star, whose results must equal the single-GPU results on the concatenated inputs.

Retrieval -- the bank (spot embeddings AND expression rows) is split into contiguous row
ranges, queries are replicated:
    local   : find_matches on the shard (+ index offset) and the distances of its own winners
    exchange: all-gather of (similarity, global index, distance) candidate lists  [R, Q, k]
    merge   : global top-k by (value desc, index asc) -- identical on every rank
    average : each rank accumulates w_j * expression[idx_j] for the winners it owns,
              all-reduce of the [Q, G] partial sums
Contrastive loss -- rank r owns batch rows [r*B/R, (r+1)*B/R):
    all-gather of the embeddings, three phases on the local rows separated by all-gathers of
    the per-row statistics (5 floats per row); gradients of the local rows need no exchange.

The host logic is backend-agnostic: ``CudaBackend`` drives libmclst_b200.so; the CPU test
suite injects an oracle-backed backend to exercise the sharding / gather / merge plumbing
under ``gloo`` with world_size 2 (tests/test_distributed_cpu.py).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib
from ._lib import WEIGHT_MODES, check, load, ptr, stream_ptr

__all__ = ["shard_bounds", "bind_to_gpu_cpus", "BankShard", "CudaBackend", "retrieve_sharded", "contrastive_loss_sharded",
           "RetrievalGrid", "make_retrieval_grid"]


def bind_to_gpu_cpus(device_index: int) -> bool:
    """Pin this process to the CPU cores next to its GPU (NVML's ideal affinity), so that the pinned
    host buffers it allocates afterwards live on that GPU's NUMA node.  One process per GPU under
    torchrun starts unbound; with all ranks' upload buffers on one socket the aggregate host-to-device
    rate of an 8-GPU box stalled near 100-140 GB/s however many links were used.  Returns False when
    NVML is not available (nothing changes)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(device_index))
        return True
    except Exception:
        return False


def shard_bounds(n: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous, balanced row ranges [(start, end)] by global index."""
    return [(n * r // world, n * (r + 1) // world) for r in range(world)]


@dataclass
class BankShard:
    spot_key: torch.Tensor          # [n_local, D] float32
    expression_key: torch.Tensor    # [n_local, G] float32 / float64
    index_offset: int               # global index of local row 0
    n_total: int
    expr_ready: Optional["torch.cuda.Event"] = None   # set when expression_key is still uploading
    _ws: Optional[dict] = None       # (slot, top_k) -> (workspace holding this shard's packed image, query capacity)

    def workspace(self, slot: int, n_query: int, top_k: int):
        """(workspace, already_packed) for one of the query blocks in flight: the shard's packed image
        (normalised fp16 tiles, norms, residuals) is written on first use and stays resident."""
        from .retrieval import fm_workspace
        if self._ws is None:
            self._ws = {}
        ent = self._ws.get((slot, top_k))
        if ent is None or ent[1] < n_query:
            ws = fm_workspace(self.spot_key.shape[0], n_query, self.spot_key.shape[1], top_k, self.spot_key.device)
            self._ws[(slot, top_k)] = (ws, n_query)
            return ws, False
        return ent[0], True

    @classmethod
    def from_full(cls, spot_key, expression_key, rank: int, world: int) -> "BankShard":
        lo, hi = shard_bounds(spot_key.shape[0], world)[rank]
        return cls(spot_key[lo:hi].contiguous(), expression_key[lo:hi].contiguous(), lo,
                   spot_key.shape[0])

    @classmethod
    def from_host(cls, spot_key: torch.Tensor, expression_key: torch.Tensor, index_offset: int,
                  n_total: int, device) -> "BankShard":
        """Upload one shard from (pinned) host tensors.  The expression rows -- most of the bytes,
        not needed before the average -- go on a side stream so that the copy runs underneath the
        shard's top-k kernels; ``retrieve_sharded`` waits for ``expr_ready``."""
        from .retrieval import _side_stream
        device = torch.device(device)
        sk = spot_key.to(device, non_blocking=True)
        side = _side_stream(device)
        with torch.cuda.stream(side):
            ek = expression_key.to(device, non_blocking=True)
            ready = side.record_event()
        ek.record_stream(torch.cuda.current_stream(device))
        return cls(sk, ek, index_offset, n_total, ready)


class CudaBackend:
    """libmclst_b200.so on the local device."""

    def local_topk(self, shard: BankShard, query: torch.Tensor, k: int, p: int, need_dist: bool):
        from .retrieval import find_matches_device
        n_loc = shard.spot_key.shape[0]
        kk = min(k, n_loc)
        Q = query.shape[0]
        dev = query.device
        val = torch.full((Q, k), float("-inf"), dtype=torch.float32, device=dev)
        idx = torch.full((Q, k), 2 ** 31 - 1, dtype=torch.int64, device=dev)
        dst = torch.full((Q, k), float("inf"), dtype=torch.float32, device=dev) if need_dist else None
        if kk == k:
            r = find_matches_device(shard.spot_key, query, k, index_offset=shard.index_offset,
                                    dist_p=p if need_dist else None)
            return (r[0], r[1], r[2]) if need_dist else (r[0], r[1], None)
        if kk > 0:
            r = find_matches_device(shard.spot_key, query, kk, index_offset=shard.index_offset,
                                    dist_p=p if need_dist else None)
            val[:, :kk], idx[:, :kk] = r[0], r[1]
            if need_dist:
                dst[:, :kk] = r[2]
        return val, idx, dst

    def merge(self, vals, idx, dst, k: int):
        R, Q, _ = vals.shape
        dev = vals.device
        ov = torch.empty((Q, k), dtype=torch.float32, device=dev)
        oi = torch.empty((Q, k), dtype=torch.int64, device=dev)
        od = torch.empty((Q, k), dtype=torch.float32, device=dev) if dst is not None else None
        with torch.cuda.device(dev):
            check(load().mclst_merge_topk(ptr(vals), ptr(idx), ptr(dst), R, Q, k, ptr(ov), ptr(oi), ptr(od),
                                          stream_ptr()), "merge_topk")
        return ov, oi, od

    def weights(self, dst, val, mode: str):
        Q, k = val.shape
        w = torch.empty((Q, k), dtype=torch.float32, device=val.device)
        with torch.cuda.device(val.device):
            check(load().mclst_neighbor_weights(ptr(dst), ptr(val), Q, k, WEIGHT_MODES[mode], ptr(w),
                                                stream_ptr()), "neighbor_weights")
        return w

    def partial_average(self, rows: torch.Tensor, index_offset: int, idx, w):
        n_loc, G = rows.shape
        Q, k = idx.shape
        out = torch.empty((Q, G), dtype=torch.float32, device=idx.device)
        with torch.cuda.device(idx.device):
            check(load().mclst_weighted_gather(ptr(rows), n_loc, rows.stride(0), G,
                                               int(rows.dtype == torch.float64), ptr(idx), ptr(w), Q, k,
                                               index_offset, ptr(out), stream_ptr()), "weighted_gather")
        return out


def _all_gather_cat(t: torch.Tensor, group, async_op: bool = False):
    """[R * rows, ...] = the ranks' tensors concatenated along dim 0, written by ONE collective
    straight into its final place (no per-rank list, no stack copy)."""
    world = dist.get_world_size(group)
    t = t.contiguous()
    out = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    work = dist.all_gather_into_tensor(out, t, group=group, async_op=async_op)
    return out, work


def _tc_eligible(shard: BankShard, k: int) -> bool:
    from .retrieval import tc_eligible
    n, d = shard.spot_key.shape
    return tc_eligible(n, d, k)


class _Block:
    """One query block of a sharded retrieval on its way through the pipeline."""
    __slots__ = ("q", "ws", "packed", "bounds", "w_bounds", "val", "idx", "dst", "g", "w_g", "expr", "emb",
                 "w_out", "rows", "a2a")


def retrieve_sharded(shard: BankShard, query: torch.Tensor, top_k: int = 50, mode: str = "inv_sq_l2",
                     group=None, backend=None, want_emb: bool = False, scatter_output: bool = False,
                     query_blocks: Optional[int] = None):
    """(indices int64 [Q,k], values f32 [Q,k], emb_pred | None, expr_pred f32 [Q,G]) -- identical on
    every rank and equal to the single-GPU ``retrieve_device`` on the concatenated bank.

    With ``scatter_output`` the partial sums are reduce-scattered instead of all-reduced: every rank
    keeps only its share of the finished rows and the call returns a fifth value ``rows`` (int64 row
    numbers into the query batch) -- expr_pred / emb_pred then hold exactly those rows.

    Bank shards (CUDA backend): per query block  seed pass -> all-reduce of per-query bounds of the
    GLOBAL k-th best score (2 floats per query) -> candidate pass against that bound -> all-reduce
    (MAX) of the bounds the converged thresholds give -> exact re-rank of only the candidates that
    can still win globally (short, padded lists) -> all-to-all of the lists (every rank merges only
    its own Q/R queries) -> all-gather of the merged lists -> owner-only partial sums ->
    reduce-scatter / all-reduce.  The queries
    go in ``query_blocks`` blocks (default 2 when large) so that the collectives of one block run
    under the top-k kernels of the next."""
    backend = backend or CudaBackend()
    need_dist = mode in ("inv_sq_l1", "inv_sq_l2", "bleep_exp")
    p = 1 if mode == "inv_sq_l1" else 2
    world = dist.get_world_size(group) if (dist.is_initialized() and shard.n_total != shard.spot_key.shape[0]) else 1
    Q = query.shape[0]
    if world == 1:
        val, idx, dst = backend.local_topk(shard, query, top_k, p, need_dist)
        w = backend.weights(dst, val, mode)
        if shard.expr_ready is not None:
            torch.cuda.current_stream(shard.expression_key.device).wait_event(shard.expr_ready)
        expr = backend.partial_average(shard.expression_key, shard.index_offset, idx, w)
        emb = backend.partial_average(shard.spot_key, shard.index_offset, idx, w) if want_emb else None
        if scatter_output:
            return idx, val, emb, expr, torch.arange(Q, device=query.device)
        return idx, val, emb, expr
    rank = dist.get_rank(group)
    staged = isinstance(backend, CudaBackend) and _tc_eligible(shard, top_k) and Q > 0
    nb = query_blocks if query_blocks else (2 if Q >= 32768 else 1)
    nb = max(1, min(nb, Q)) if Q else 1
    nccl = dist.get_backend(group) == "nccl"
    scatter = scatter_output and nccl
    a2a = nccl and isinstance(backend, CudaBackend)
    cuts = [Q * b // nb for b in range(nb + 1)]
    blocks: List[_Block] = []
    for b in range(nb):
        blk = _Block()
        blk.q = query[cuts[b]:cuts[b + 1]]
        blk.rows = None
        blocks.append(blk)
    # -- stage 1: seed pass of every block, bounds exchange in flight
    if staged:
        from .retrieval import fm_seed
        k_part = -(-top_k // world)
        for b, blk in enumerate(blocks):
            blk.ws, blk.packed = shard.workspace(b, blk.q.shape[0], top_k)
            bounds = fm_seed(shard.spot_key, blk.q, top_k, blk.ws, k_part, want_bounds=True, bank_packed=blk.packed)
            # one MAX all-reduce carries both: row 0 = bound_k (max over shards is valid), row 1 = minus
            # bound_part (min over shards of the ceil(k/R)-th best: every shard then has that many rows)
            bounds[1].neg_()
            blk.bounds = bounds
            blk.w_bounds = dist.all_reduce(bounds, op=dist.ReduceOp.MAX, group=group, async_op=True)
    # -- stage 2: candidate pass against the seed bound, second (tight) exchange in flight
    if staged:
        from .retrieval import fm_candidates, fm_main
        for blk in blocks:
            blk.w_bounds.wait()
            ext = torch.maximum(blk.bounds[0], -blk.bounds[1]).contiguous()
            # what every shard actually kept bounds the global k-th best much more tightly: the same
            # two figures (k-th best: max over shards; ceil(k/R)-th best: min over shards, sent
            # negated) from the candidate buffers, one more MAX all-reduce
            b2 = fm_candidates(shard.spot_key, blk.q, top_k, blk.ws, ext, bank_packed=True, k_part=k_part)
            b2[0] = torch.maximum(b2[0], ext)
            b2[1].neg_()
            blk.bounds = b2
            blk.w_bounds = dist.all_reduce(b2, op=dist.ReduceOp.MAX, group=group, async_op=True)
    # -- stage 3: re-rank of what can still win (+ candidate all-gather in flight)
    for blk in blocks:
        if staged:
            blk.w_bounds.wait()
            ext2 = torch.maximum(blk.bounds[0], -blk.bounds[1]).contiguous()
            blk.val, blk.idx, blk.dst = fm_main(shard.spot_key, blk.q, top_k, blk.ws, shard.index_offset,
                                                p if need_dist else None, ext2, bank_packed=True,
                                                finish_only=True)
        else:
            blk.val, blk.idx, blk.dst = backend.local_topk(shard, blk.q, top_k, p, need_dist)
        Qb = blk.q.shape[0]
        # (similarity, index, distance) of every candidate in ONE tensor: index as two float32 words
        parts = [blk.val.view(Qb, top_k, 1), blk.idx.view(torch.float32).view(Qb, top_k, 2)]
        if need_dist:
            parts.append(blk.dst.view(Qb, top_k, 1))
        cand = torch.cat(parts, dim=2)
        if a2a and Qb % world == 0:
            # all-to-all: rank r receives every shard's candidates for ITS Qb/R queries only and merges
            # those (1/R of the merge work, (R-1)/R x 1/R of the all-gather's bytes)
            blk.g = torch.empty_like(cand)
            blk.w_g = dist.all_to_all_single(blk.g, cand, group=group, async_op=True)
            blk.a2a = True
        else:
            blk.g, blk.w_g = _all_gather_cat(cand, group, async_op=True)
            blk.a2a = False
    # -- stage 4: merge, weights, owner-only partial sums (+ reduction in flight)
    if shard.expr_ready is not None:
        torch.cuda.current_stream(shard.expression_key.device).wait_event(shard.expr_ready)
    for blk in blocks:
        blk.w_g.wait()
        Qb = blk.q.shape[0]
        Qm = Qb // world if blk.a2a else Qb                       # queries this rank merges
        g = blk.g.view(world, Qm, top_k, -1)
        vals = g[..., 0].contiguous()
        idxs = g[..., 1:3].contiguous().view(torch.int64).view(world, Qm, top_k)
        dsts = g[..., 3].contiguous() if need_dist else None
        val, idx, dst = backend.merge(vals, idxs, dsts, top_k)
        w = backend.weights(dst, val, mode)
        if blk.a2a:
            # the merged lists of every rank's slice, so that each owner can add up its winners
            m = torch.cat([val.view(Qm, top_k, 1), idx.view(torch.float32).view(Qm, top_k, 2), w.view(Qm, top_k, 1)], 2)
            mg, _ = _all_gather_cat(m, group)
            mg = mg.view(Qb, top_k, 4)
            val = mg[..., 0].contiguous()
            idx = mg[..., 1:3].contiguous().view(torch.int64).view(Qb, top_k)
            w = mg[..., 3].contiguous()
        blk.val, blk.idx = val, idx
        part = backend.partial_average(shard.expression_key, shard.index_offset, blk.idx, w)
        if want_emb:
            part = torch.cat([part, backend.partial_average(shard.spot_key, shard.index_offset, blk.idx, w)], dim=1)
        if scatter and Qb % world == 0:
            out = torch.empty((Qb // world, part.shape[1]), dtype=part.dtype, device=part.device)
            blk.w_out = dist.reduce_scatter_tensor(out, part, group=group, async_op=True)
            blk.expr = out
        else:
            blk.w_out = dist.all_reduce(part, group=group, async_op=True)
            blk.expr = part
    G = shard.expression_key.shape[1]
    outs, rows = [], []
    for b, blk in enumerate(blocks):
        blk.w_out.wait()
        Qb = blk.q.shape[0]
        if scatter_output:
            if scatter and Qb % world == 0:
                lo, hi = Qb // world * rank, Qb // world * (rank + 1)
                outs.append(blk.expr)
            else:
                lo, hi = shard_bounds(Qb, world)[rank]
                outs.append(blk.expr[lo:hi])
            rows.append(torch.arange(cuts[b] + lo, cuts[b] + hi, device=query.device))
        else:
            outs.append(blk.expr)
    full = torch.cat(outs) if len(outs) > 1 else outs[0]
    idx = torch.cat([blk.idx for blk in blocks]) if nb > 1 else blocks[0].idx
    val = torch.cat([blk.val for blk in blocks]) if nb > 1 else blocks[0].val
    expr, emb = (full[:, :G], full[:, G:]) if want_emb else (full, None)
    if scatter_output:
        return idx, val, emb, expr, (torch.cat(rows) if len(rows) > 1 else rows[0])
    return idx, val, emb, expr


@dataclass
class RetrievalGrid:
    """2-D decomposition of a retrieval job over world = query_groups x bank_shards ranks.

    Ranks [g*bank_shards, (g+1)*bank_shards) form query group g: they share one slice of the
    queries and hold one bank shard each (candidate all-gather + merge inside the group).
    Sharding the BANK multiplies the streaming top-k / re-rank work (every shard produces its
    own k + band candidates for every query); sharding the QUERIES does not and needs no
    exchange, but replicates the bank.  bank_shards is therefore a capacity knob: 1 when the
    bank fits on a GPU, larger when it does not."""
    query_groups: int
    bank_shards: int
    q_index: int
    b_index: int
    group: object          # process group of this rank's query group (None when bank_shards == 1)

    def query_slice(self, n_query: int) -> Tuple[int, int]:
        return shard_bounds(n_query, self.query_groups)[self.q_index]


def make_retrieval_grid(bank_shards: int, world: Optional[int] = None, rank: Optional[int] = None) -> RetrievalGrid:
    world = dist.get_world_size() if world is None else world
    rank = dist.get_rank() if rank is None else rank
    if world % bank_shards != 0:
        raise ValueError(f"bank_shards={bank_shards} does not divide world={world}")
    qg = world // bank_shards
    mine = None
    if bank_shards > 1:
        for g in range(qg):                     # every rank must take part in every new_group call
            h = dist.new_group(list(range(g * bank_shards, (g + 1) * bank_shards)))
            if g == rank // bank_shards:
                mine = h
    return RetrievalGrid(qg, bank_shards, rank // bank_shards, rank % bank_shards, mine)


# ----------------------------------------------------------------------------- loss
REPLICATE_LOSS_BELOW = 8192      # global batch up to which every rank evaluates the whole loss itself


class _ShardedLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s_loc, i_loc, temperature, mode, group):
        world = dist.get_world_size(group)
        rank = dist.get_rank(group)
        rows, D = s_loc.shape
        B = rows * world
        if rows % 128 != 0:
            raise _lib.MclstError("contrastive_loss_sharded: rows per rank must be a multiple of 128")
        S = torch.empty((B, D), dtype=torch.float32, device=s_loc.device)
        I = torch.empty((B, D), dtype=torch.float32, device=s_loc.device)
        dist.all_gather_into_tensor(S, s_loc.detach().contiguous(), group=group)
        dist.all_gather_into_tensor(I, i_loc.detach().contiguous(), group=group)
        if B <= REPLICATE_LOSS_BELOW and hasattr(load(), "mclst_contrastive_loss"):
            # small global batches: five blocking collectives on tiny tensors cost more than the whole
            # single-GPU loss (B = 1024 on 8 GPUs measured 3.1 ms sharded vs 0.3 ms on one GPU), so
            # every rank evaluates the full batch after the one embedding all-gather and keeps the
            # gradient rows it owns
            from .loss import contrastive_loss_fwd_bwd
            loss, dS_full, dI_full = contrastive_loss_fwd_bwd(S, I, temperature, mode, want_grad=True)
            r0 = rank * rows
            ctx.save_for_backward(dS_full[r0:r0 + rows], dI_full[r0:r0 + rows])
            return loss
        lib = load()
        nbytes = C.c_size_t()
        check(lib.mclst_contrastive_loss_workspace_bytes(B, D, mode, rows, C.byref(nbytes)), "loss workspace")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=S.device)
        stats = torch.zeros((_lib.LOSS_STAT_ROWS, B), dtype=torch.float32, device=S.device)
        loss = torch.zeros((), dtype=torch.float32, device=S.device)
        dS = torch.empty((rows, D), dtype=torch.float32, device=S.device)
        dI = torch.empty((rows, D), dtype=torch.float32, device=S.device)
        row0 = rank * rows

        def phase(ph):
            with torch.cuda.device(S.device):
                check(lib.mclst_contrastive_loss_phase(ptr(S), S.stride(0), ptr(I), I.stride(0), B, D,
                                                       float(temperature), mode, row0, rows, ph, ptr(stats),
                                                       ptr(loss), ptr(dS), dS.stride(0), ptr(dI),
                                                       dI.stride(0), ptr(ws), ws.numel(), stream_ptr()),
                      f"contrastive_loss_phase {ph}")

        def gather_rows(sel):
            loc = stats[sel, row0:row0 + rows].contiguous()
            # (output as the dim-0 concatenation of the inputs: the one shape both NCCL and gloo accept)
            full = torch.empty((world * len(sel), rows), dtype=torch.float32, device=S.device)
            dist.all_gather_into_tensor(full, loc, group=group)
            stats[sel] = full.view(world, len(sel), rows).permute(1, 0, 2).reshape(len(sel), B)

        phase(1)
        gather_rows([0, 1, 2, 5, 6, 7, 8])      # rl, cl, za, diag + the lo halves of the three LSE pairs
        if mode != _lib.T_EYE:
            phase(2)
            gather_rows([3, 4])
        phase(3)
        dist.all_reduce(loss, group=group)
        ctx.save_for_backward(dS, dI)
        return loss

    @staticmethod
    def backward(ctx, g):
        dS, dI = ctx.saved_tensors
        return g * dS, g * dI, None, None, None


def contrastive_loss_sharded(spot_emb_local: torch.Tensor, image_emb_local: torch.Tensor,
                             temperature: float = 1.0, targets: str = "eye", soft_scale: str = "div",
                             group=None) -> torch.Tensor:
    """Global-batch contrastive loss over all ranks' rows (each rank passes its [B/R, D] slice).
    Returns the full-batch loss (same value on every rank); ``backward`` yields the gradients
    of that loss w.r.t. the local slices."""
    from .loss import TARGET_MODES
    return _ShardedLoss.apply(spot_emb_local, image_emb_local, float(temperature),
                              TARGET_MODES[(targets, soft_scale)], group)
