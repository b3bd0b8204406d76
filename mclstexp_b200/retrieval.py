"""Evaluation retrieval of mclSTExp on B200: the reference's Python surface
(``find_matches`` + the per-query weighted-average loop) over libmclst_b200.so.

Reference being mirrored (paths relative to /root/reference):
  * ``find_matches``           evel_her2st.py:74-84, evel_visium.py:94-104,
                               evel_cscc.py:74-84 (returns values too)
  * the weighted-average loop  evel_her2st.py:175-187 (L1), evel_visium.py:194-205 and
                               evel_cscc.py:198-215 (L2), BLEEP_inference.ipynb cell 5

PyTorch is used only for device memory and streams; every number is produced by
the CUDA kernels in ``csrc/``.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple, Union

import numpy as np
import torch

from . import _lib
from ._lib import WEIGHT_MODES, check, load, ptr, require_cuda, stream_ptr

ArrayLike = Union[np.ndarray, torch.Tensor]

__all__ = ["find_matches", "find_matches_cscc", "find_matches_device", "fm_workspace", "fm_pack_bank", "fm_seed",
           "fm_candidates", "fm_main", "weighted_topk_average",
           "weighted_topk_average_device", "retrieve", "retrieve_device", "retrieve_workspace", "last_counters",
           "to_host", "tc_eligible", "Bank"]

_last_ws: Optional[torch.Tensor] = None
_side_streams: dict = {}
_PIN_MIN_BYTES = 1 << 20


def _side_stream(dev: torch.device) -> "torch.cuda.Stream":
    """One extra stream per device for the uploads that can run under the top-k kernels."""
    key = (dev.type, dev.index)
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=dev)
    return _side_streams[key]


def to_host(*tensors: Optional[torch.Tensor]):
    """Results to NumPy with ONE synchronisation; anything of a megabyte or more lands in a pinned
    buffer from torch's caching host allocator (PCIe rate instead of the pageable staging rate).
    The returned arrays own those buffers."""
    outs = []
    for t in tensors:
        if t is None:
            outs.append(None)
            continue
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=t.numel() * t.element_size() >= _PIN_MIN_BYTES)
        h.copy_(t, non_blocking=True)
        outs.append(h)
    torch.cuda.current_stream().synchronize()
    return [None if h is None else h.numpy() for h in outs]


def _from_numpy(x) -> torch.Tensor:
    a = np.ascontiguousarray(x)
    if not a.flags.writeable:            # read-only memory maps (io.load_fold): torch wants writable
        a = a.copy()
    return torch.from_numpy(a)


def _dev_f32(x: ArrayLike, device=None) -> torch.Tensor:
    """What ``torch.tensor(x)`` does at evel_her2st.py:76-77, but onto the GPU."""
    if isinstance(x, torch.Tensor):
        t = x
    else:
        t = _from_numpy(x)
    if t.dtype != torch.float32:
        t = t.float()
    if not t.is_cuda:
        if not torch.cuda.is_available():
            raise _lib.MclstError("no CUDA device: find_matches has no CPU fallback")
        t = t.to(device or "cuda", non_blocking=True)
    if t.dim() == 1:
        t = t[None]
    if t.stride(-1) != 1:
        t = t.contiguous()
    return t


def tc_eligible(n_bank: int, dim: int, top_k: int, flags: int = _lib.FM_DEFAULT) -> bool:
    """Whether find_matches of this shape runs the tensor-core candidate pass (and a bank of it can
    keep a packed image) or brute-forces every query: the library's own rule
    (mclst_find_matches_tc_eligible), asked rather than restated.  Needs no GPU."""
    return bool(load().mclst_find_matches_tc_eligible(int(n_bank), int(dim), int(top_k), int(flags)))


def find_matches_device(spot_embeddings: torch.Tensor, query_embeddings: torch.Tensor,
                        top_k: int = 1, index_offset: int = 0, exact_only: bool = False,
                        need_values: bool = True, dist_p: Optional[int] = None):
    """Device-resident form: float32 CUDA [N,D], [Q,D] -> (values f32 [Q,k] | None,
    indices int64 [Q,k]), rows sorted by (similarity desc, index asc).  With ``dist_p`` (1 or 2)
    a third tensor is returned: the L1 / L2 distance of every winner to the raw query."""
    global _last_ws
    require_cuda(spot_embeddings, query_embeddings)
    lib = load()
    bank, qry = spot_embeddings, query_embeddings
    assert bank.dtype == torch.float32 and qry.dtype == torch.float32
    assert bank.dim() == 2 and qry.dim() == 2 and bank.shape[1] == qry.shape[1]
    assert bank.stride(1) == 1 and qry.stride(1) == 1
    N, D = bank.shape
    Q = qry.shape[0]
    flags = _lib.FM_EXACT_ONLY if exact_only else _lib.FM_DEFAULT
    nbytes = C.c_size_t()
    check(lib.mclst_find_matches_workspace_bytes(N, Q, D, top_k, flags, C.byref(nbytes)),
          "find_matches_workspace_bytes")
    ws = torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=bank.device)
    idx = torch.empty((Q, top_k), dtype=torch.int64, device=bank.device)
    val = torch.empty((Q, top_k), dtype=torch.float32, device=bank.device) if need_values else None
    dst = torch.empty((Q, top_k), dtype=torch.float32, device=bank.device) if dist_p else None
    if Q == 0:
        return (val, idx, dst) if dist_p else (val, idx)
    with torch.cuda.device(bank.device):
        check(lib.mclst_find_matches_dist(ptr(bank), N, bank.stride(0), ptr(qry), Q, qry.stride(0), D,
                                          top_k, index_offset, ptr(idx), ptr(val), ptr(dst),
                                          dist_p or 2, ptr(ws), ws.numel(), flags, stream_ptr()),
              "find_matches")
    _last_ws = ws
    return (val, idx, dst) if dist_p else (val, idx)


def fm_workspace(n_bank: int, n_query: int, dim: int, top_k: int, device, flags: int = 0) -> torch.Tensor:
    nbytes = C.c_size_t()
    check(load().mclst_find_matches_workspace_bytes(n_bank, n_query, dim, top_k, flags, C.byref(nbytes)),
          "find_matches_workspace_bytes")
    return torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=device)


def fm_pack_bank(bank: torch.Tensor, top_k: int, ws: torch.Tensor) -> None:
    """Write the packed image of ``bank`` (normalised fp16 operand tiles, float64 norms, rounding
    residuals) into ``ws`` once; later staged calls pass ``bank_packed=True``."""
    require_cuda(bank, ws)
    with torch.cuda.device(bank.device):
        check(load().mclst_find_matches_pack_bank(ptr(bank), bank.shape[0], bank.stride(0), bank.shape[1],
                                                  top_k, ptr(ws), ws.numel(), stream_ptr()), "find_matches_pack_bank")


def fm_seed(bank: torch.Tensor, qry: torch.Tensor, top_k: int, ws: torch.Tensor, k_part: int = 1,
            want_bounds: bool = False, bank_packed: bool = False):
    """Stage 1 of find_matches (pack + seed pass).  With ``want_bounds`` returns a float32 [2, Q]
    tensor: row 0 = lower bound of this bank's own top_k-th best exact score per query, row 1 = the
    same for its k_part-th best (-inf where nothing is known)."""
    require_cuda(bank, qry, ws)
    Q = qry.shape[0]
    bounds = torch.empty((2, Q), dtype=torch.float32, device=bank.device) if want_bounds else None
    flags = _lib.FM_BANK_PACKED if bank_packed else 0
    with torch.cuda.device(bank.device):
        check(load().mclst_find_matches_seed(ptr(bank), bank.shape[0], bank.stride(0), ptr(qry), Q, qry.stride(0),
                                             bank.shape[1], top_k, k_part, ptr(bounds),
                                             ptr(bounds[1]) if want_bounds else None, ptr(ws), ws.numel(),
                                             flags, stream_ptr()), "find_matches_seed")
    if want_bounds:
        bounds = torch.nan_to_num(bounds, nan=float("-inf"), neginf=float("-inf"), posinf=float("inf"))
    return bounds


def fm_candidates(bank: torch.Tensor, qry: torch.Tensor, top_k: int, ws: torch.Tensor,
                  ext_bound: Optional[torch.Tensor] = None, bank_packed: bool = False,
                  k_part: int = 1) -> torch.Tensor:
    """Stage 2a: the tensor-core candidate pass alone.  Returns float32 [2, Q]: lower bounds of this
    bank's exact top_k-th (row 0) and k_part-th (row 1) best score per query, from the candidates it
    kept (-inf: unknown)."""
    require_cuda(bank, qry, ws)
    Q = qry.shape[0]
    out = torch.empty((2, Q), dtype=torch.float32, device=bank.device)
    flags = _lib.FM_BANK_PACKED if bank_packed else 0
    with torch.cuda.device(bank.device):
        check(load().mclst_find_matches_candidates(ptr(bank), bank.shape[0], bank.stride(0), ptr(qry), Q,
                                                   qry.stride(0), bank.shape[1], top_k, k_part, ptr(ext_bound),
                                                   ptr(out), ptr(out[1]), ptr(ws), ws.numel(), flags, stream_ptr()),
              "find_matches_candidates")
    return torch.nan_to_num(out, nan=float("-inf"), neginf=float("-inf"), posinf=float("inf"))


def fm_main(bank: torch.Tensor, qry: torch.Tensor, top_k: int, ws: torch.Tensor, index_offset: int = 0,
            dist_p: Optional[int] = None, ext_bound: Optional[torch.Tensor] = None, bank_packed: bool = False,
            finish_only: bool = False):
    """Stage 2 (main pass + re-rank + exact fallback; ``finish_only``: re-rank + fallback after
    ``fm_candidates``) -> (values, indices, distances | None).  Under an external bound a row list may
    be shorter than top_k; its tail is (-inf, 0x7fffffff, +inf)."""
    global _last_ws
    Q = qry.shape[0]
    dev = bank.device
    idx = torch.empty((Q, top_k), dtype=torch.int64, device=dev)
    val = torch.empty((Q, top_k), dtype=torch.float32, device=dev)
    dst = torch.empty((Q, top_k), dtype=torch.float32, device=dev) if dist_p else None
    if ext_bound is not None:
        assert ext_bound.dtype == torch.float32 and ext_bound.is_contiguous() and ext_bound.numel() == Q
    flags = _lib.FM_BANK_PACKED if bank_packed else 0
    fn = load().mclst_find_matches_finish if finish_only else load().mclst_find_matches_main
    with torch.cuda.device(dev):
        check(fn(ptr(bank), bank.shape[0], bank.stride(0), ptr(qry), Q, qry.stride(0),
                 bank.shape[1], top_k, index_offset, ptr(idx), ptr(val), ptr(dst),
                 dist_p or 2, ptr(ext_bound), ptr(ws), ws.numel(), flags,
                 stream_ptr()), "find_matches_finish" if finish_only else "find_matches_main")
    _last_ws = ws
    return val, idx, dst


def last_counters() -> dict:
    """{'tensor_core': n, 'exact_fallback': n} of the most recent find_matches (synchronises)."""
    if _last_ws is None:
        return {}
    out = (C.c_int64 * 4)()
    with torch.cuda.device(_last_ws.device):
        check(load().mclst_read_counters(ptr(_last_ws), out, stream_ptr()), "read_counters")
    return {"tensor_core": int(out[0]), "exact_fallback": int(out[1]), "speculation_rejected": int(out[2])}


def find_matches(spot_embeddings: ArrayLike, query_embeddings: ArrayLike, top_k: int = 1,
                 return_values: bool = False, exact_only: bool = False):
    """Drop-in for evel_her2st.py:74-84: array-likes in, ``np.ndarray`` int64 [Q,k] out
    (``(k,)`` when there is a single query: the reference's ``squeeze(0)``, :82).  With
    ``return_values`` the cSCC flavour (evel_cscc.py:74-84): ``(values, indices)``.
    Tie rule (undefined in the reference): lowest index first."""
    bank = _dev_f32(spot_embeddings)
    qry = _dev_f32(query_embeddings, bank.device)
    val, idx = find_matches_device(bank, qry, top_k, exact_only=exact_only, need_values=return_values)
    with torch.cuda.device(idx.device):
        idx_np, val_np = to_host(idx, val if return_values else None)
    if idx_np.shape[0] == 1:
        idx_np = idx_np[0]
    if return_values:
        if val_np.shape[0] == 1:
            val_np = val_np[0]
        return val_np, idx_np
    return idx_np


def find_matches_cscc(spot_embeddings, query_embeddings, top_k=1):
    """evel_cscc.py:74-84."""
    return find_matches(spot_embeddings, query_embeddings, top_k, return_values=True)


def weighted_topk_average_device(spot_key: torch.Tensor, expression_key: torch.Tensor,
                                 image_query: torch.Tensor, indices: torch.Tensor,
                                 mode: str = "inv_sq_l2", values: Optional[torch.Tensor] = None,
                                 want_emb: bool = True, out_dtype=torch.float64,
                                 distances: Optional[torch.Tensor] = None
                                 ) -> Tuple[Optional[torch.Tensor], torch.Tensor]:
    require_cuda(spot_key, expression_key, image_query, indices)
    lib = load()
    assert spot_key.dtype == torch.float32 and image_query.dtype == torch.float32
    assert expression_key.dtype in (torch.float32, torch.float64)
    assert indices.dtype == torch.int64 and indices.dim() == 2 and indices.is_contiguous()
    assert out_dtype in (torch.float32, torch.float64)
    Q, k = indices.shape
    N, D = spot_key.shape
    G = expression_key.shape[1]
    assert expression_key.shape[0] == N and image_query.shape == (Q, D)
    assert spot_key.stride(1) == 1 and expression_key.stride(1) == 1 and image_query.stride(1) == 1
    if values is not None:
        values = values.contiguous().float()
    dev = spot_key.device
    emb = torch.empty((Q, D), dtype=out_dtype, device=dev) if want_emb else None
    expr = torch.empty((Q, G), dtype=out_dtype, device=dev)
    with torch.cuda.device(dev):
        check(lib.mclst_weighted_average(
            ptr(spot_key), N, spot_key.stride(0), ptr(expression_key), expression_key.stride(0), G,
            int(expression_key.dtype == torch.float64), ptr(image_query), Q, image_query.stride(0),
            D, ptr(indices), ptr(values), ptr(distances), k, 0, WEIGHT_MODES[mode], ptr(emb), ptr(expr),
            int(out_dtype == torch.float64), stream_ptr()), "weighted_average")
    return emb, expr


def weighted_topk_average(spot_key: ArrayLike, expression_key: ArrayLike, image_query: ArrayLike,
                          indices: ArrayLike, p: int = 2, mode: Optional[str] = None,
                          values: Optional[ArrayLike] = None) -> Tuple[np.ndarray, np.ndarray]:
    """Replaces the inline loop evel_her2st.py:175-187 (``p=1``) / evel_visium.py:194-205,
    evel_cscc.py:198-215 (``p=2``); ``mode`` selects the other variants
    ('similarity', 'uniform', 'bleep_exp').  Returns float64 arrays like the reference's
    ``np.zeros`` results: (matched_spot_embeddings_pred [Q,D], matched_spot_expression_pred [Q,G])."""
    if mode is None:
        mode = {1: "inv_sq_l1", 2: "inv_sq_l2"}[p]
    sk = _dev_f32(spot_key)
    iq = _dev_f32(image_query, sk.device)
    ek = expression_key if isinstance(expression_key, torch.Tensor) else \
        torch.from_numpy(np.ascontiguousarray(expression_key))
    if ek.dtype not in (torch.float32, torch.float64):
        ek = ek.float()
    ek = ek.to(sk.device)
    idx = indices if isinstance(indices, torch.Tensor) else torch.from_numpy(np.asarray(indices))
    idx = idx.to(sk.device, torch.int64)
    if idx.dim() == 1:
        idx = idx[None]
    idx = idx.contiguous()
    val = None
    if values is not None:
        val = _dev_f32(values, sk.device)
    emb, expr = weighted_topk_average_device(sk, ek, iq, idx, mode, val)
    with torch.cuda.device(sk.device):
        emb_np, expr_np = to_host(emb, expr)
    return emb_np, expr_np


def _retrieve_call(spot_key, expression_key, image_query, top_k, mode, want_emb, out_dtype, flags, ws=None):
    """mclst_retrieve: find_matches + neighbour distances + weighted average in one C call (query
    blocks pipelined inside: the average of one block runs under the top-k pass of the next)."""
    global _last_ws
    require_cuda(spot_key, expression_key, image_query)
    lib = load()
    assert spot_key.dtype == torch.float32 and image_query.dtype == torch.float32
    assert expression_key.dtype in (torch.float32, torch.float64)
    assert out_dtype in (torch.float32, torch.float64)
    assert spot_key.dim() == 2 and image_query.dim() == 2 and spot_key.shape[1] == image_query.shape[1]
    assert spot_key.stride(1) == 1 and expression_key.stride(1) == 1 and image_query.stride(1) == 1
    N, D = spot_key.shape
    Q = image_query.shape[0]
    G = expression_key.shape[1]
    assert expression_key.shape[0] == N
    dev = spot_key.device
    idx = torch.empty((Q, top_k), dtype=torch.int64, device=dev)
    val = torch.empty((Q, top_k), dtype=torch.float32, device=dev)
    emb = torch.empty((Q, D), dtype=out_dtype, device=dev) if want_emb else None
    expr = torch.empty((Q, G), dtype=out_dtype, device=dev)
    if Q == 0:
        return idx, val, emb, expr
    if ws is None:
        ws = retrieve_workspace(N, Q, D, top_k, dev, flags)
    with torch.cuda.device(dev):
        check(lib.mclst_retrieve(ptr(spot_key), N, spot_key.stride(0), ptr(expression_key),
                                 expression_key.stride(0), G, int(expression_key.dtype == torch.float64),
                                 ptr(image_query), Q, image_query.stride(0), D, top_k, WEIGHT_MODES[mode],
                                 ptr(idx), ptr(val), ptr(emb), ptr(expr), int(out_dtype == torch.float64),
                                 ptr(ws), ws.numel(), flags, stream_ptr()), "retrieve")
    _last_ws = ws
    return idx, val, emb, expr


def retrieve_workspace(n_bank: int, n_query: int, dim: int, top_k: int, device, flags: int = 0) -> torch.Tensor:
    nbytes = C.c_size_t()
    check(load().mclst_retrieve_workspace_bytes(n_bank, n_query, dim, top_k, flags, C.byref(nbytes)),
          "retrieve_workspace_bytes")
    return torch.empty(max(nbytes.value, 256), dtype=torch.uint8, device=device)


def retrieve_device(spot_key: torch.Tensor, expression_key: torch.Tensor, image_query: torch.Tensor,
                    top_k: int = 50, mode: str = "inv_sq_l2", want_emb: bool = False,
                    out_dtype=torch.float32, exact_only: bool = False):
    """find_matches + weighted average with everything resident on the device.
    Returns (indices int64 [Q,k], values f32 [Q,k], emb_pred | None, expr_pred [Q,G])."""
    flags = _lib.FM_EXACT_ONLY if exact_only else _lib.FM_DEFAULT
    return _retrieve_call(spot_key, expression_key, image_query, top_k, mode, want_emb, out_dtype, flags)


def _to_dev(x: ArrayLike, device, dtypes=(torch.float32,)) -> torch.Tensor:
    t = x if isinstance(x, torch.Tensor) else _from_numpy(x)
    if t.dtype not in dtypes:
        t = t.float()
    return t.to(device, non_blocking=True)


def retrieve(spot_key: ArrayLike, expression_key: ArrayLike, image_query: ArrayLike, top_k: int = 50,
             p: int = 2, mode: Optional[str] = None, want_emb: bool = True, out_dtype=torch.float64):
    """The whole fold-loop body evel_her2st.py:174-187 in one call, host arrays in and out:
    (indices [Q,k] int64, matched_spot_embeddings_pred [Q,D] | None, matched_spot_expression_pred
    [Q,G]); float64 results by default, like the reference's ``np.zeros`` arrays.  Inputs may be
    NumPy arrays or (pinned) CPU tensors; the copies to and from the device happen here."""
    if mode is None:
        mode = {1: "inv_sq_l1", 2: "inv_sq_l2"}[p]
    if not torch.cuda.is_available():
        raise _lib.MclstError("no CUDA device: retrieve has no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device())
    cur = torch.cuda.current_stream(dev)
    sk = _to_dev(spot_key, dev)
    iq = _to_dev(image_query, dev)
    if iq.dim() == 1:
        iq = iq[None]
    need_dist = mode in ("inv_sq_l1", "inv_sq_l2", "bleep_exp")
    r = find_matches_device(sk, iq, top_k, dist_p=(1 if mode == "inv_sq_l1" else 2) if need_dist else None)
    val, idx, dst = (r[0], r[1], r[2]) if need_dist else (r[0], r[1], None)
    # the expression rows (the bulk of the bytes) are not needed until the average: they are
    # uploaded on a side stream, underneath the top-k kernels launched above (also when the source
    # is pageable and the copy call blocks the host)
    side = _side_stream(dev)
    with torch.cuda.stream(side):
        ek = _to_dev(expression_key, dev, (torch.float32, torch.float64))
        uploaded = side.record_event()
    ek.record_stream(cur)
    cur.wait_event(uploaded)
    emb, expr = weighted_topk_average_device(sk, ek, iq, idx, mode, val if mode == "similarity" else None,
                                             want_emb, out_dtype, distances=dst)
    idx_np, emb_np, expr_np = to_host(idx, emb, expr)
    return idx_np, emb_np, expr_np


class Bank:
    """A bank (spot_key, expression_key) kept resident on the device across many ``retrieve`` calls:
    the serving form of the fold loop, where only the queries travel per call -- and the hand-off
    from the bank build (``embed.embed_bank`` output goes straight in, no ``.npy`` round trip,
    evel_her2st.py:116-117,146-147).  Besides the raw rows the bank keeps the PACKED image the
    top-k kernels consume (normalised fp16 operand tiles, float64 norms, rounding residuals), written
    once per (top_k class, query capacity) instead of on every call."""

    def __init__(self, spot_key: ArrayLike, expression_key: ArrayLike, device=None):
        if not torch.cuda.is_available():
            raise _lib.MclstError("no CUDA device: Bank has no CPU fallback")
        dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.spot_key = _to_dev(spot_key, dev).contiguous()
        self.expression_key = _to_dev(expression_key, dev, (torch.float32, torch.float64)).contiguous()
        if self.spot_key.shape[0] != self.expression_key.shape[0]:
            raise ValueError("spot_key and expression_key must have the same number of rows")
        self._packed: dict = {}          # top_k -> (workspace, query capacity)

    def __len__(self) -> int:
        return self.spot_key.shape[0]

    def _workspace(self, n_query: int, top_k: int) -> torch.Tensor:
        """A workspace holding this bank's packed image, large enough for n_query queries."""
        ent = self._packed.get(top_k)
        if ent is None or ent[1] < n_query:
            cap = max(n_query, 1024)
            # (laid out for mclst_retrieve: the find_matches workspace first, so the staged entry
            # points can use it as well)
            ws = retrieve_workspace(len(self), cap, self.spot_key.shape[1], top_k, self.spot_key.device,
                                    _lib.FM_BANK_PACKED)
            fm_pack_bank(self.spot_key, top_k, ws)
            ent = self._packed[top_k] = (ws, cap)
        return ent[0]

    def find_matches(self, query: torch.Tensor, top_k: int = 50, dist_p: Optional[int] = None):
        """Device-resident (values, indices[, distances]) against the resident packed image."""
        N, D = self.spot_key.shape
        if not tc_eligible(N, D, top_k) or query.shape[0] == 0:
            return find_matches_device(self.spot_key, query, top_k, dist_p=dist_p)
        ws = self._workspace(query.shape[0], top_k)
        fm_seed(self.spot_key, query, top_k, ws, bank_packed=True)
        val, idx, dst = fm_main(self.spot_key, query, top_k, ws, dist_p=dist_p, bank_packed=True)
        return (val, idx, dst) if dist_p else (val, idx)

    def retrieve_device(self, image_query: torch.Tensor, top_k: int = 50, mode: str = "inv_sq_l2",
                        want_emb: bool = False, out_dtype=torch.float32):
        N, D = self.spot_key.shape
        if tc_eligible(N, D, top_k) and image_query.shape[0] > 0:
            ws = self._workspace(image_query.shape[0], top_k)
            return _retrieve_call(self.spot_key, self.expression_key, image_query, top_k, mode, want_emb,
                                  out_dtype, _lib.FM_BANK_PACKED, ws)
        return _retrieve_call(self.spot_key, self.expression_key, image_query, top_k, mode, want_emb, out_dtype,
                              _lib.FM_DEFAULT)

    def retrieve(self, image_query: ArrayLike, top_k: int = 50, p: int = 2, mode: Optional[str] = None,
                 want_emb: bool = True, out_dtype=torch.float64):
        """Host (or device) queries in, host arrays out: (indices, emb_pred | None, expr_pred)."""
        if mode is None:
            mode = {1: "inv_sq_l1", 2: "inv_sq_l2"}[p]
        dev = self.spot_key.device
        with torch.cuda.device(dev):
            iq = _to_dev(image_query, dev)
            if iq.dim() == 1:
                iq = iq[None]
            idx, _, emb, expr = self.retrieve_device(iq.contiguous(), top_k, mode, want_emb, out_dtype)
            return tuple(to_host(idx, emb, expr))


def debug_similarity(spot_embeddings: ArrayLike, query_embeddings: ArrayLike) -> torch.Tensor:
    """Testing aid: the raw similarities seen by the tensor-core candidate pass
    (fp16-rounded normalised operands, fp32 accumulate) as a CUDA tensor [Q,N]."""
    bank = _dev_f32(spot_embeddings)
    qry = _dev_f32(query_embeddings, bank.device)
    require_cuda(bank, qry)
    lib = load()
    N, D = bank.shape
    Q = qry.shape[0]
    nbytes = C.c_size_t()
    check(lib.mclst_find_matches_workspace_bytes(N, Q, D, 1, 0, C.byref(nbytes)), "workspace")
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=bank.device)
    out = torch.full((Q, N), float("nan"), dtype=torch.float32, device=bank.device)
    with torch.cuda.device(bank.device):
        check(lib.mclst_debug_similarity(ptr(bank), N, bank.stride(0), ptr(qry), Q, qry.stride(0),
                                         D, ptr(out), out.stride(0), ptr(ws), ws.numel(),
                                         stream_ptr()), "debug_similarity")
    return out
