"""Pin the oracle against outputs of the reference's own code (tests/golden/,
made by oracle/make_golden.py inside the build container).  CPU only."""
import numpy as np
import pytest
import torch

from mclstexp_b200 import synth
from oracle import oracle
from conftest import golden_checksum, golden_cpu_threads, golden_grad, golden_sha256


def _retrieval_inputs(meta, name):
    m = meta[name]
    if name == "pm1":
        bank = synth.pm1_embeddings(m["N"], m["D"], m["seed"])
        qry = synth.pm1_embeddings(m["Q"], m["D"], m["seed"] + 1)
        assert golden_checksum(bank, qry) == m["checksum"]
        return bank, qry, None
    bank = synth.embeddings(m["N"], m["D"], m["seed"], m["flavour"])
    qry = synth.embeddings(m["Q"], m["D"], m["seed"] + 1, m["flavour"])
    expr = synth.expression(m["N"], m["G"], m["seed"] + 2)
    assert golden_checksum(bank, qry, expr) == m["checksum"], "synthetic generator drifted"
    return bank, qry, expr


@pytest.mark.parametrize("name", ["iid", "clustered"])
@pytest.mark.parametrize("k", [1, 50, 200])
def test_find_matches_ref_is_the_reference(golden_retrieval, name, k):
    z, meta = golden_retrieval
    bank, qry, _ = _retrieval_inputs(meta, name)
    val, idx = oracle.find_matches_ref(bank, qry, k, return_values=True)
    assert idx.dtype == np.int64
    np.testing.assert_array_equal(idx, z[f"{name}/find_matches/k{k}/indices"])
    np.testing.assert_array_equal(val, z[f"{name}/find_matches/k{k}/values"])


@pytest.mark.parametrize("name", ["iid", "clustered"])
def test_find_matches_q1_squeeze_quirk(golden_retrieval, name):
    z, meta = golden_retrieval
    bank, qry, _ = _retrieval_inputs(meta, name)
    idx = oracle.find_matches_ref(bank, qry[:1], 5)
    assert idx.shape == (5,)                      # evel_her2st.py:82 squeeze(0)
    np.testing.assert_array_equal(idx, z[f"{name}/find_matches/q1/indices"])


@pytest.mark.parametrize("name", ["iid", "clustered"])
@pytest.mark.parametrize("k", [1, 50, 200])
def test_spec_agrees_with_reference_on_decidable_rows(golden_retrieval, name, k):
    z, meta = golden_retrieval
    bank, qry, _ = _retrieval_inputs(meta, name)
    val, idx = oracle.find_matches_spec(bank, qry, k)
    ok = oracle.decidable_rows(bank, qry, k)
    assert ok.mean() > 0.25          # k=200 of N=700 walks deep into the dense part of the distribution
    ref_idx = z[f"{name}/find_matches/k{k}/indices"]
    np.testing.assert_array_equal(idx[ok], ref_idx[ok])
    np.testing.assert_allclose(val, z[f"{name}/find_matches/k{k}/values"], rtol=0, atol=5e-7)
    # rows that are not decidable still hold the same index SET up to the boundary element
    for r in np.where(~ok)[0]:
        assert len(set(idx[r]) ^ set(ref_idx[r])) <= 2


def test_pm1_known_answer_values_and_tie_rule(golden_retrieval):
    z, meta = golden_retrieval
    bank, qry, _ = _retrieval_inputs(meta, "pm1")
    val, idx = oracle.find_matches_spec(bank, qry, 50)
    ref_val = z["pm1/find_matches/k50/values"]
    ref_idx = z["pm1/find_matches/k50/indices"]
    # exact arithmetic: the sorted value rows are bit-identical to the reference's
    np.testing.assert_array_equal(val, ref_val)
    assert np.all(np.round(val * 256) == val * 256)
    sim = oracle.similarity_spec(bank, qry)
    for r in range(idx.shape[0]):
        # within each tie group the spec picks the lowest indices in ascending order
        for v in np.unique(val[r]):
            mine = idx[r][val[r] == v]
            allv = np.where(sim[r] == v)[0]
            np.testing.assert_array_equal(mine, allv[:len(mine)])
        # the reference picked members of the same tie groups
        np.testing.assert_array_equal(sim[r][ref_idx[r]], ref_val[r])


LOOPS = [("loop_her2st", "inv_sq_l1"), ("loop_visium", "inv_sq_l2"), ("loop_cscc", "inv_sq_l2"),
         ("bleep_simple", "uniform"), ("bleep_average", "uniform"), ("bleep_weighted_average", "bleep_exp")]


@pytest.mark.parametrize("name", ["iid", "clustered"])
@pytest.mark.parametrize("tag,mode", LOOPS)
def test_weighted_average_ref_is_the_reference(golden_retrieval, name, tag, mode):
    z, meta = golden_retrieval
    bank, qry, expr = _retrieval_inputs(meta, name)
    idx = z[f"{name}/{tag}/indices"].astype(np.int64)
    if tag == "bleep_simple":
        assert idx.shape[1] == 1
    emb, ex = oracle.weighted_average_ref(bank, expr, qry, idx, mode)
    assert emb.dtype == np.float64 and ex.dtype == np.float64
    np.testing.assert_array_equal(emb, z[f"{name}/{tag}/emb_pred"])
    np.testing.assert_array_equal(ex, z[f"{name}/{tag}/expr_pred"])
    # and the float64 spec is within float32 round-off of it
    emb64, ex64 = oracle.weighted_average_spec(bank, expr, qry, idx, mode)
    # (bleep_exp subtracts float32 squared distances ~5e2 before exp(): 1e-4-level round-off)
    tol = 1e-3 if mode == "bleep_exp" else 2e-5
    np.testing.assert_allclose(emb64, emb, rtol=tol, atol=tol)
    np.testing.assert_allclose(ex64, ex, rtol=tol, atol=tol * 0.1)


def test_similarity_weights_match_commented_variant(golden_retrieval):
    z, meta = golden_retrieval
    bank, qry, expr = _retrieval_inputs(meta, "iid")
    val, idx = oracle.find_matches_ref(bank, qry, 50, return_values=True)
    emb, ex = oracle.weighted_average_ref(bank, expr, qry, idx, "similarity", val)
    emb64, ex64 = oracle.weighted_average_spec(bank, expr, qry, idx, "similarity", val)
    np.testing.assert_allclose(ex64, ex, rtol=2e-5, atol=2e-6)


def test_zero_distance_is_defined_in_spec():
    bank = synth.embeddings(64, 32, 1)
    qry = bank[[3, 7]].copy()
    expr = synth.expression(64, 10, 2)
    idx = np.array([[3, 5, 9], [1, 7, 2]])
    _, ex = oracle.weighted_average_spec(bank, expr, qry, idx, "inv_sq_l2")
    np.testing.assert_allclose(ex[0], expr[3], rtol=1e-7)
    np.testing.assert_allclose(ex[1], expr[7], rtol=1e-7)


# ------------------------------------------------------------------ losses
@pytest.mark.parametrize("case", ["loss_b48", "loss_b65_t07", "loss_b16_t2"])
@pytest.mark.parametrize("tag", ["eye", "soft_div", "soft_mul"])
def test_losses_are_the_reference(golden_model, case, tag):
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
    with golden_cpu_threads():
        loss, dS, dI = oracle.contrastive_loss_ref(S, I, m["T"], targets, scale)
    np.testing.assert_array_equal(loss.numpy(), z[f"{case}/{tag}/loss"])
    # bit-equal to the reference's gradients (stored as digests), so dS / dI below ARE them
    dS, dI = dS.numpy(), dI.numpy()
    assert golden_sha256(dS) == str(z[f"{case}/{tag}/dS/sha256"])
    assert golden_sha256(dI) == str(z[f"{case}/{tag}/dI/sha256"])
    # closed form used by the fused kernels (float64) against the reference's autograd
    l64, dS64, dI64 = oracle.contrastive_loss_closed_form(S, I, m["T"], targets, scale)
    np.testing.assert_allclose(l64, z[f"{case}/{tag}/loss"], rtol=2e-5)
    sc = np.abs(dS).max()
    np.testing.assert_allclose(dS64, dS, rtol=0, atol=2e-5 * sc + 1e-9)
    np.testing.assert_allclose(dI64, dI, rtol=0, atol=2e-5 * sc + 1e-9)


# ------------------------------------------------------------------ modules
@pytest.mark.parametrize("case", ["small", "odd"])
def test_path_forward_backward_is_the_reference(golden_model, case):
    z, meta = golden_model
    m = meta[case]
    sd = oracle.make_state_dict(m["G"], m["E"], 256, m["heads"], m["dim_head"], m["layers"], m["seed"])
    feats = torch.tensor(synth.image_features(m["B"], m["E"], m["seed"] + 1))
    expr = torch.tensor(synth.expression(m["B"], m["G"], m["seed"] + 2))
    pos = torch.tensor(synth.positions(m["B"], m["seed"] + 3, m["kind"]))
    assert golden_checksum(feats, expr, pos, sd["x_embed.weight"][:64],
                           sd["spot_projection.fc.weight"]) == m["checksum"]
    with torch.no_grad():
        img = oracle.projection_head_ref(feats, sd, "image_projection.")
        spot = oracle.spot_embedding_ref(sd, expr, pos, m["heads"], m["layers"])
    np.testing.assert_allclose(img.numpy(), z[f"{case}/image_embeddings"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(spot.numpy(), z[f"{case}/spot_embeddings"], rtol=0, atol=2e-5)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss = oracle.path_loss_ref(params, feats, expr, pos, m["T"], m["heads"], m["layers"], "eye")
    loss.backward()
    np.testing.assert_allclose(loss.item(), z[f"{case}/loss"], rtol=1e-5)
    for k, p in params.items():
        idx, g, gmax, gnorm, shape = golden_grad(z, f"{case}/grad/{k}")
        if k in ("x_embed.weight", "y_embed.weight"):
            rows = z[f"{case}/grad_rows/{k}"].astype(np.int64)
            mine = p.grad[rows].numpy()
            mask = torch.ones(p.shape[0], dtype=torch.bool)
            mask[rows] = False
            assert float(p.grad[mask].abs().sum()) == 0.0
        else:
            mine = p.grad.numpy()
        assert mine.shape == shape, k
        atol = 1e-4 * gmax + 1e-9
        np.testing.assert_allclose(mine.ravel()[idx], g, rtol=0, atol=atol, err_msg=k)
        # every entry within atol keeps the norm of the whole array within atol * sqrt(size)
        assert abs(np.linalg.norm(mine.astype(np.float64)) - gnorm) <= atol * np.sqrt(mine.size), k


# ------------------------------------------------------------------ downstream metrics
@pytest.fixture(scope="session")
def golden_metrics():
    from conftest import _load
    return _load("metrics.npz")


@pytest.mark.parametrize("name", ["a", "b"])
def test_metrics_ref_is_the_reference(golden_metrics, name):
    z, meta = golden_metrics
    m = meta[name]
    true = synth.expression(m["Q"], m["G"], m["seed"]).astype(np.float64)
    pred = z[f"{name}/pred"].astype(np.float64)
    assert golden_checksum(true, pred) == m["checksum"]
    got = oracle.metrics_ref(true, pred)
    for key in ("heg_pcc", "hvg_pcc", "mse", "mae"):
        np.testing.assert_allclose(got[key], z[f"{name}/{key}"], rtol=1e-12, err_msg=key)
    assert np.isnan(got["pcc"][3])
