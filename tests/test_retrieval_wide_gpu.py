"""Retrieval with embeddings 257-512 wide: the wide variant of the tensor-core candidate pass
(8 resident K slices, 3-stage bank ring, accumulation bound E_ACC_WIDE) plus the exact re-rank
must give exactly what the float64 brute force gives, and wider rows stay on the exact path."""
import numpy as np
import pytest
import torch

from mclstexp_b200 import _lib, retrieval, synth
from oracle import oracle

pytestmark = pytest.mark.gpu

E_ACC_WIDE = 4.0e-6      # the accumulation bound the kernel assumes for 256 < K <= 512 (sim_topk.cu)


def _fp16_operands(x):
    # what pack_rows builds: float32(x * float32(1 / float64 norm)), rounded to fp16
    x = np.ascontiguousarray(x, np.float32)
    inv = (1.0 / oracle.norms_spec(x)).astype(np.float32)
    xn = (x * inv[:, None]).astype(np.float32)
    xh = xn.astype(np.float16)
    resid = np.sqrt(((xn.astype(np.float64) - xh.astype(np.float64)) ** 2).sum(1))
    return xh, resid


def _pm1_half(rows, seed, dim=512):
    """+-1 in dim/2 random coordinates, 0 elsewhere: norm sqrt(dim/2) = 16 at dim 512, so the
    normalised entries are +-1/16 and every score is a multiple of 1/256 (exact in fp16 and fp32)."""
    rng = np.random.default_rng(seed)
    x = np.zeros((rows, dim), np.float32)
    on = np.argsort(rng.random((rows, dim)), axis=1)[:, :dim // 2]
    np.put_along_axis(x, on, rng.choice(np.array([-1.0, 1.0], np.float32), (rows, dim // 2)), axis=1)
    return x


def _check_spec(bank, qry, k, val, idx):
    sval, sidx = oracle.find_matches_spec(bank, qry, k)
    np.testing.assert_array_equal(np.asarray(idx).reshape(sidx.shape), sidx)
    np.testing.assert_array_equal(np.asarray(val).reshape(sval.shape), sval)


@pytest.mark.parametrize("N,Q,D,flavour", [(700, 37, 512, "iid"), (1025, 129, 512, "clustered"),
                                           (530, 140, 257, "iid"), (256, 128, 264, "clustered"),
                                           (900, 70, 320, "iid"), (600, 33, 384, "clustered"),
                                           (5000, 260, 448, "clustered"), (4100, 300, 512, "clustered")])
def test_wide_raw_tensor_core_similarities(N, Q, D, flavour):
    bank = synth.embeddings(N, D, 17 + N, flavour)
    qry = synth.embeddings(Q, D, 18 + N, flavour)
    got = retrieval.debug_similarity(bank, qry).cpu().numpy()
    assert not np.isnan(got).any(), "some similarities were never written"
    bh, rb = _fp16_operands(bank)
    qh, rq = _fp16_operands(qry)
    want16 = qh.astype(np.float64) @ bh.astype(np.float64).T       # what the MMA should compute
    acc_err = np.abs(got - want16).max()
    assert acc_err < E_ACC_WIDE / 4, f"K={D}: accumulation error {acc_err:.3e} vs bound {E_ACC_WIDE:.1e}"
    exact = oracle.similarity_spec(bank, qry).astype(np.float64)
    bound = 1.002 * (rq[:, None] + rb[None, :]) + E_ACC_WIDE + 1e-6
    assert (np.abs(got - exact) <= bound).all()
    print(f"N={N} Q={Q} D={D}: max acc err {acc_err:.2e}, max |approx-exact| "
          f"{np.abs(got - exact).max():.2e}, typical bound {bound.mean():.2e}")


def test_wide_known_answer_is_exact():
    bank = _pm1_half(600, 5)
    qry = _pm1_half(40, 6)
    got = retrieval.debug_similarity(bank, qry).cpu().numpy()
    want = (qry.astype(np.float64) / 16) @ (bank.astype(np.float64) / 16).T
    np.testing.assert_array_equal(got, want.astype(np.float32))


@pytest.mark.parametrize("D,N,Q,k", [(512, 20077, 300, 50), (512, 4099, 1, 1), (257, 9013, 129, 200),
                                     (384, 6005, 200, 600), (320, 30011, 257, 1), (448, 7777, 64, 50),
                                     (264, 5000, 100, 50), (512, 3000, 130, 600)])
def test_wide_find_matches_equals_spec(D, N, Q, k):
    """k = 600 runs the CAP 1024 candidate pass, but the re-rank holds at most 512 survivors, so its
    queries are finished by the exact path; smaller k must be resolved by the re-rank."""
    bank = synth.embeddings(N, D, 100 + D, "clustered")
    qry = synth.embeddings(Q, D, 200 + D, "clustered")
    val, idx = retrieval.find_matches(bank, qry, k, return_values=True)
    c = retrieval.last_counters()
    print(D, N, Q, k, c)
    assert c["tensor_core"] + c["exact_fallback"] == Q, c
    if k <= 200:
        assert c["tensor_core"] >= 0.99 * Q, c         # the wide candidate pass is what ran
    if Q == 1:
        assert idx.shape == (k,) and val.shape == (k,)   # the reference's squeeze(0)
    _check_spec(bank, qry, k, val, idx)
    val_e, idx_e = retrieval.find_matches(bank, qry, k, return_values=True, exact_only=True)
    assert retrieval.last_counters()["tensor_core"] == 0
    np.testing.assert_array_equal(idx, idx_e)
    np.testing.assert_array_equal(val, val_e)


@pytest.mark.parametrize("D", [512, 384])
@pytest.mark.parametrize("layout", ["ld", "unaligned"])
def test_wide_strided_and_unaligned_rows(D, layout):
    """ld > dim (scalar pack and re-rank loads) and a base that is not 16-byte aligned."""
    N, Q, k = 5003, 150, 50
    bank = synth.embeddings(N, D, 301, "clustered")
    qry = synth.embeddings(Q, D, 302, "clustered")
    pad = 5 if layout == "ld" else 4
    off = 0 if layout == "ld" else 1
    bb = torch.full((N, D + pad), float("nan"), device="cuda")
    qb = torch.full((Q, D + pad), float("nan"), device="cuda")
    bb[:, off:off + D] = torch.from_numpy(bank).cuda()
    qb[:, off:off + D] = torch.from_numpy(qry).cuda()
    bv, qv = bb[:, off:off + D], qb[:, off:off + D]
    assert bv.stride(0) == D + pad and (layout == "ld" or bv.data_ptr() % 16 != 0)
    val, idx = retrieval.find_matches_device(bv, qv, k)
    assert retrieval.last_counters()["tensor_core"] >= 0.99 * Q
    val_c, idx_c = retrieval.find_matches_device(torch.from_numpy(bank).cuda(), torch.from_numpy(qry).cuda(), k)
    assert torch.equal(idx, idx_c) and torch.equal(val, val_c)
    _check_spec(bank, qry, k, val.cpu().numpy(), idx.cpu().numpy())


def test_wide_edge_inputs_stay_exact():
    D, k = 512, 50
    bank = synth.embeddings(9000, D, 401, "clustered")
    qry = synth.embeddings(200, D, 402, "clustered")
    bank[10:20] = 0.0                        # zero rows: cosine 0 (F.normalize's eps clamp)
    qry[3] = 0.0
    bank[100:140] = bank[50]                 # duplicate rows: ties broken by the lower index
    bank[4000:4064] = qry[:64]               # exact matches of some queries
    val, idx = retrieval.find_matches(bank, qry, k, return_values=True)
    _check_spec(bank, qry, k, val, idx)
    val_e, idx_e = retrieval.find_matches(bank, qry, k, return_values=True, exact_only=True)
    np.testing.assert_array_equal(idx, idx_e)
    np.testing.assert_array_equal(val, val_e)


def test_wide_massive_ties_fall_back_and_stay_exact():
    """Scores on a 1/256 grid; on top of that 2000 exact copies of one row that eight queries equal,
    so their bands hold far more tied rows than a candidate buffer: those rows reach the exact path."""
    bank = _pm1_half(40000, 9)
    qry = _pm1_half(64, 10)
    bank[::20] = bank[0]
    qry[:8] = bank[0]
    val, idx = retrieval.find_matches(bank, qry, 50, return_values=True)
    c = retrieval.last_counters()
    print(c)
    _check_spec(bank, qry, 50, val, idx)
    assert c["exact_fallback"] >= 8 and c["tensor_core"] + c["exact_fallback"] == 64, c
    assert (idx[:8] == np.arange(0, 1000, 20)).all()      # ties: lowest indices first


def test_wide_nonfinite_inputs_take_the_exact_path():
    bank = synth.embeddings(900, 512, 3)
    qry = synth.embeddings(20, 512, 4)
    bank[5, 7] = np.inf
    val, idx = retrieval.find_matches(bank, qry, 10, return_values=True)
    c = retrieval.last_counters()
    assert c["exact_fallback"] == 20 and c["tensor_core"] == 0, c
    val_e, idx_e = retrieval.find_matches(bank, qry, 10, return_values=True, exact_only=True)
    np.testing.assert_array_equal(idx, idx_e)
    np.testing.assert_array_equal(val.view(np.uint32), val_e.view(np.uint32))


@pytest.mark.parametrize("p", [1, 2])
@pytest.mark.parametrize("aligned", [True, False])
def test_wide_distances(p, aligned):
    N, Q, D, k = 8000, 300, 512, 50
    bank = synth.embeddings(N, D, 501, "clustered")
    qry = synth.embeddings(Q, D, 502, "clustered")
    tb = torch.from_numpy(bank).cuda()
    tq = torch.from_numpy(qry).cuda()
    if not aligned:                           # the scalar re-rank loads
        tb = torch.nn.functional.pad(tb, (0, 3))[:, :D]
    val, idx, dst = retrieval.find_matches_device(tb, tq, k, dist_p=p)
    assert retrieval.last_counters()["tensor_core"] >= 0.99 * Q
    _check_spec(bank, qry, k, val.cpu().numpy(), idx.cpu().numpy())
    i = idx.cpu().numpy()
    diff = bank.astype(np.float64)[i] - qry.astype(np.float64)[:, None, :]
    want = np.abs(diff).sum(-1) if p == 1 else np.sqrt((diff ** 2).sum(-1))
    np.testing.assert_allclose(dst.cpu().numpy(), want, rtol=1e-4 if p == 1 else 1e-5, atol=1e-5)


@pytest.mark.parametrize("D", [384, 512])
def test_wide_resident_bank_keeps_packed_image(D):
    N, G, k = 20000, 200, 50
    bank = synth.embeddings(N, D, 601, "clustered")
    expr = synth.expression(N, G, 602)
    b = retrieval.Bank(bank, expr)
    for Q, p in ((100, 2), (1500, 1), (700, 2)):
        qry = synth.embeddings(Q, D, 610 + Q, "clustered")
        idx, emb, ex = b.retrieve(qry, top_k=k, p=p)
        assert retrieval.last_counters()["tensor_core"] >= 0.99 * Q
        idx1, emb1, ex1 = retrieval.retrieve(bank, expr, qry, top_k=k, p=p)
        np.testing.assert_array_equal(idx, idx1)
        np.testing.assert_array_equal(ex, ex1)
        np.testing.assert_array_equal(emb, emb1)
        mode = "inv_sq_l1" if p == 1 else "inv_sq_l2"
        e_idx, _, _, e_ex = retrieval.retrieve_device(torch.from_numpy(bank).cuda(), torch.from_numpy(expr).cuda(),
                                                      torch.from_numpy(qry).cuda(), k, mode, out_dtype=torch.float64,
                                                      exact_only=True)
        np.testing.assert_array_equal(idx, e_idx.cpu().numpy())
        np.testing.assert_allclose(ex, e_ex.cpu().numpy(), rtol=1e-6, atol=1e-9)
    assert set(b._packed) == {k}              # the packed image is kept (and reused) for this top_k
    vb, ib = b.find_matches(torch.from_numpy(qry).cuda(), k)
    val1, idx1 = retrieval.find_matches_device(torch.from_numpy(bank).cuda(), torch.from_numpy(qry).cuda(), k)
    assert torch.equal(ib, idx1) and torch.equal(vb, val1)


def test_wide_blocked_retrieve_equals_unblocked():
    """More than eight lane rounds of queries go through mclst_retrieve in blocks."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N, D, G, k, mode = 2000, 512, 24, 50, "inv_sq_l2"
    Q = 8 * 128 * sms + 777
    bank = torch.tensor(synth.embeddings(N, D, 701, "clustered")).cuda()
    expr = torch.tensor(synth.expression(N, G, 702)).cuda()
    qry = torch.tensor(synth.embeddings(Q, D, 703, "clustered")).cuda()
    idx, val, emb, ex = retrieval.retrieve_device(bank, expr, qry, k, mode, want_emb=True)
    c = retrieval.last_counters()
    assert c["tensor_core"] + c["exact_fallback"] == Q and c["tensor_core"] >= 0.99 * Q, c
    cut = Q // 2 + 5
    parts = [retrieval.retrieve_device(bank, expr, qry[a:b], k, mode, want_emb=True) for a, b in ((0, cut), (cut, Q))]
    for i, got in enumerate((idx, val, emb, ex)):
        assert torch.equal(got, torch.cat([p[i] for p in parts])), i
    rows = np.arange(0, Q, 1999)
    sval, sidx = oracle.find_matches_spec(bank.cpu().numpy(), qry.cpu().numpy()[rows], k)
    np.testing.assert_array_equal(idx.cpu().numpy()[rows], sidx)


def _merge(vals, idxs, k):
    from mclstexp_b200._lib import check, load, ptr, stream_ptr
    R, Q, _ = vals.shape
    ov = torch.empty((Q, k), dtype=torch.float32, device="cuda")
    oi = torch.empty((Q, k), dtype=torch.int64, device="cuda")
    check(load().mclst_merge_topk(ptr(vals), ptr(idxs), None, R, Q, k, ptr(ov), ptr(oi), None, stream_ptr()),
          "merge_topk")
    return ov, oi


def test_wide_bank_shards_with_bound_exchange_equal_whole_bank():
    """The bank-shard protocol (seed -> bound exchange -> candidates -> second exchange -> finish)
    replayed on one GPU at D = 384 over 3 shards: bit-identical to the whole bank."""
    N, Q, D, k, shards = 40000, 700, 384, 50, 3
    bank = torch.tensor(synth.embeddings(N, D, 61, "clustered"), device="cuda")
    qry = torch.tensor(synth.embeddings(Q, D, 62, "clustered"), device="cuda")
    wval, widx = retrieval.find_matches_device(bank, qry, k)
    assert retrieval.last_counters()["tensor_core"] >= 0.99 * Q
    cuts = [N * s // shards for s in range(shards + 1)]
    parts = [bank[cuts[s]:cuts[s + 1]].contiguous() for s in range(shards)]
    k_part = -(-k // shards)
    wss, bounds = [], []
    for pb in parts:
        ws = retrieval.fm_workspace(pb.shape[0], Q, D, k, pb.device)
        wss.append(ws)
        bounds.append(retrieval.fm_seed(pb, qry, k, ws, k_part, want_bounds=True))
    b = torch.stack(bounds)
    ext = torch.maximum(b[:, 0].max(0).values, b[:, 1].min(0).values).contiguous()
    b2 = torch.stack([retrieval.fm_candidates(pb, qry, k, wss[s], ext, bank_packed=True, k_part=k_part)
                      for s, pb in enumerate(parts)])
    ext2 = torch.maximum(torch.maximum(b2[:, 0].max(0).values, b2[:, 1].min(0).values), ext).contiguous()
    assert bool((ext2 <= wval[:, -1] + 1e-6).all())
    vals, idxs, short = [], [], 0
    for s, pb in enumerate(parts):
        v, i, _ = retrieval.fm_main(pb, qry, k, wss[s], index_offset=cuts[s], ext_bound=ext2, bank_packed=True,
                                    finish_only=True)
        short += int((i == 0x7fffffff).any(1).sum())
        vals.append(v)
        idxs.append(i)
    mv, mi = _merge(torch.stack(vals), torch.stack(idxs), k)
    assert torch.equal(mi, widx) and torch.equal(mv, wval)
    assert short > 0
    sval, sidx = oracle.find_matches_spec(bank.cpu().numpy(), qry[:64].cpu().numpy(), k)
    np.testing.assert_array_equal(mi[:64].cpu().numpy(), sidx)
    np.testing.assert_array_equal(mv[:64].cpu().numpy(), sval)


def test_513_stays_on_the_exact_path():
    N, Q, D, G, k = 3000, 40, 513, 50, 20
    bank = synth.embeddings(N, D, 801, "clustered")
    qry = synth.embeddings(Q, D, 802, "clustered")
    expr = synth.expression(N, G, 803)
    val, idx = retrieval.find_matches(bank, qry, k, return_values=True)
    c = retrieval.last_counters()
    assert c["tensor_core"] == 0, c           # the whole call is the exact path (as with exact_only)
    _check_spec(bank, qry, k, val, idx)
    val_e, idx_e = retrieval.find_matches(bank, qry, k, return_values=True, exact_only=True)
    assert retrieval.last_counters() == c
    np.testing.assert_array_equal(idx, idx_e)
    np.testing.assert_array_equal(val, val_e)
    b = retrieval.Bank(bank, expr)
    vb, ib = b.find_matches(torch.from_numpy(qry).cuda(), k)
    np.testing.assert_array_equal(ib.cpu().numpy(), idx)
    r_idx, _, _ = b.retrieve(qry, top_k=k)
    np.testing.assert_array_equal(r_idx, idx)
    assert b._packed == {}                    # nothing to pack: the exact path reads the raw rows
    with pytest.raises(_lib.MclstError):
        retrieval.debug_similarity(bank, qry)
