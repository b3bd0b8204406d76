"""The drop-in module surface (mclstexp_b200.model) against the reference's own forward /
backward (tests/golden/model.npz, produced by running /root/reference/model.py) and the oracle."""
import numpy as np
import pytest
import torch
from torch import nn

from mclstexp_b200 import model as mm, synth
from oracle import oracle
from conftest import golden_checksum, golden_grad

pytestmark = pytest.mark.gpu
RTOL = 1e-3


def _build(m, targets="eye"):
    net = mm.mclSTExp_Attention(encoder_name="none", temperature=m["T"], image_dim=m["E"],
                                spot_dim=m["G"], projection_dim=256, heads_num=m["heads"],
                                heads_dim=m["dim_head"], head_layers=m["layers"], dropout=0.,
                                targets=targets)
    net.image_encoder = nn.Identity()          # the CNN is outside the path: features go straight in
    sd = oracle.make_state_dict(m["G"], m["E"], 256, m["heads"], m["dim_head"], m["layers"], m["seed"])
    res = net.load_state_dict(sd, strict=True)           # identical keys and shapes as the reference
    assert not res.missing_keys and not res.unexpected_keys
    return net.cuda(), sd


def _inputs(m):
    feats = torch.tensor(synth.image_features(m["B"], m["E"], m["seed"] + 1))
    expr = torch.tensor(synth.expression(m["B"], m["G"], m["seed"] + 2))
    pos = torch.tensor(synth.positions(m["B"], m["seed"] + 3, m["kind"]))
    return feats, expr, pos


def _close(got, want, name, rtol=RTOL):
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else got
    scale = np.abs(want).max() + 1e-30
    assert np.linalg.norm(got - want) <= rtol * np.linalg.norm(want) + 1e-9, name
    np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * scale, err_msg=name)


def _close_golden_grad(got, z, key, name, rtol=RTOL):
    """_close against a reference gradient stored as a fixed sample of its entries."""
    idx, want, scale, norm, shape = golden_grad(z, key)
    got = got.detach().cpu().numpy()
    assert got.shape == shape, name
    # the norm bound of _close on the whole array implies this one
    assert abs(np.linalg.norm(got.astype(np.float64)) - norm) <= rtol * norm + 1e-9, name
    got = got.ravel()[idx]
    assert np.linalg.norm(got - want) <= rtol * np.linalg.norm(want) + 1e-9, name
    np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * (scale + 1e-30), err_msg=name)


@pytest.mark.parametrize("case", ["small", "odd"])
def test_full_path_forward_backward_vs_reference(golden_model, case):
    z, meta = golden_model
    m = meta[case]
    net, sd = _build(m)
    feats, expr, pos = _inputs(m)
    assert golden_checksum(feats, expr, pos, sd["x_embed.weight"][:64],
                           sd["spot_projection.fc.weight"]) == m["checksum"]
    loss = net({"image": feats.cuda(), "expression": expr.cuda(), "position": pos.cuda()})
    assert loss.dim() == 0
    loss.backward()
    np.testing.assert_allclose(loss.item(), z[f"{case}/loss"], rtol=RTOL)
    names = {k for k, _ in net.named_parameters()}
    ref_names = {k.split("/grad/")[1].rsplit("/", 1)[0] for k in z.files if k.startswith(f"{case}/grad/")}
    assert names == ref_names
    for k, p in net.named_parameters():
        if k in ("x_embed.weight", "y_embed.weight"):
            rows = torch.tensor(z[f"{case}/grad_rows/{k}"].astype(np.int64))
            mine = p.grad[rows.cuda()]
            mask = torch.ones(p.shape[0], dtype=torch.bool)
            mask[rows] = False
            assert float(p.grad[mask.cuda()].abs().sum()) == 0.0       # dense grad, zero elsewhere
            assert p.grad.shape == p.shape
        else:
            mine = p.grad
        _close_golden_grad(mine, z, f"{case}/grad/{k}", k)


@pytest.mark.parametrize("case", ["small", "odd"])
def test_eval_attribute_surface_vs_reference(golden_model, case):
    """What evel_her2st.py:48-69 does with the model's attributes, under no_grad."""
    z, meta = golden_model
    m = meta[case]
    net, _ = _build(m)
    net.eval()
    feats, expr, pos = (t.cuda() for t in _inputs(m))
    with torch.no_grad():
        image_embeddings = net.image_projection(net.image_encoder(feats))
        x = pos[:, 0].long()
        y = pos[:, 1].long()
        spot_feature = expr + net.x_embed(x) + net.y_embed(y)          # the caller's own torch ops
        spot_features = spot_feature.unsqueeze(dim=0)
        attn0 = net.spot_encoder[0].attn(spot_features)
        blk0 = net.spot_encoder[0](spot_features)
        enc = net.spot_encoder(spot_features)
        spot_embedding = net.spot_projection(enc).squeeze(dim=0)
        fused = net.embed_spots(expr, pos)
    _close(image_embeddings, z[f"{case}/image_embeddings"], "image_embeddings")
    _close(attn0, z[f"{case}/attn0"], "attn0")
    _close(blk0, z[f"{case}/block0"], "block0")
    _close(enc, z[f"{case}/encoder"], "encoder")
    _close(spot_embedding, z[f"{case}/spot_embeddings"], "spot_embeddings")
    _close(fused, z[f"{case}/spot_embeddings"], "embed_spots")


@pytest.mark.parametrize("targets", ["eye", "soft"])
def test_cfg2_shaped_step_vs_oracle(targets):
    """BASELINE cfg2 shape at reduced batch (B=256, G=171 cSCC genes): loss + grads vs the oracle."""
    m = dict(G=171, E=1024, heads=8, dim_head=64, layers=2, B=256, T=1.0, kind="st", seed=21)
    net, sd = _build(m, targets)
    feats, expr, pos = _inputs(m)
    loss = net({"image": feats.cuda(), "expression": expr.cuda(), "position": pos.cuda()})
    loss.backward()
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref = oracle.path_loss_ref(params, feats, expr, pos, m["T"], m["heads"], m["layers"], targets)
    ref.backward()
    np.testing.assert_allclose(loss.item(), ref.item(), rtol=RTOL)
    for k, p in net.named_parameters():
        want = params[k].grad.numpy()
        _close(p.grad, want, k, rtol=2e-3)


def test_cfg2_full_size_step_vs_oracle():
    """BASELINE cfg2 at the size it names (VERDICT r1 weak 2): B = 1024 tokens, G = 1000 genes, two
    attention blocks + heads + soft-target loss, loss and every gradient vs the oracle's autograd."""
    m = dict(G=1000, E=1024, heads=8, dim_head=64, layers=2, B=1024, T=1.0, kind="st", seed=23)
    net, sd = _build(m, "soft")
    feats, expr, pos = _inputs(m)
    loss = net({"image": feats.cuda(), "expression": expr.cuda(), "position": pos.cuda()})
    loss.backward()
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref = oracle.path_loss_ref(params, feats, expr, pos, m["T"], m["heads"], m["layers"], "soft")
    ref.backward()
    np.testing.assert_allclose(loss.item(), ref.item(), rtol=RTOL)
    for k, p in net.named_parameters():
        _close(p.grad, params[k].grad.numpy(), k, rtol=2e-3)


def test_position_out_of_range_raises():
    m = dict(G=16, E=8, heads=2, dim_head=8, layers=1, B=4, T=1.0, kind="st", seed=3)
    net, _ = _build(m)
    feats, expr, pos = _inputs(m)
    pos[1, 0] = 70000.0
    loss = net({"image": feats.cuda(), "expression": expr.cuda(), "position": pos.cuda()})
    with pytest.raises(IndexError):
        loss.backward()


def test_cpu_tensors_are_rejected():
    from mclstexp_b200._lib import MclstError
    head = mm.ProjectionHead(8, 256)
    with pytest.raises(MclstError):
        head(torch.zeros(2, 8))


def test_graphed_train_step_matches_eager():
    from mclstexp_b200.graphs import GraphedTrainStep
    m = dict(G=171, E=256, heads=8, dim_head=64, layers=2, B=128, T=1.0, kind="st", seed=31)
    net, _ = _build(m, "soft")
    feats, expr, pos = (t.cuda() for t in _inputs(m))
    batch = {"image": feats, "expression": expr, "position": pos}
    net.zero_grad(set_to_none=True)
    loss = net(batch)
    loss.backward()
    eager = {k: p.grad.clone() for k, p in net.named_parameters()}
    l_eager = loss.item()
    del loss                       # a live autograd graph from the default stream would break capture
    step = GraphedTrainStep(net, batch)
    for _ in range(2):
        l = step(batch)
    assert abs(l.item() - l_eager) <= 1e-6 * abs(l_eager)
    for k, p in net.named_parameters():
        assert torch.allclose(p.grad, eager[k], rtol=1e-5, atol=1e-6 * float(eager[k].abs().max()) + 1e-12), k
    bad = dict(batch, position=pos.clone())
    bad["position"][0, 0] = 1e6
    with pytest.raises(IndexError):
        step(bad)


@pytest.mark.parametrize("N,group", [(200, 32), (128, 32), (31, 32), (1000, 64), (333, 16)])
def test_embed_bank_equals_per_batch_loop(N, group):
    """Fused block-diagonal bank build == the reference's loop over un-shuffled batches
    (evel_her2st.py:24, 47-70), including the short last batch."""
    from mclstexp_b200.embed import embed_bank
    m = dict(G=171, E=64, heads=8, dim_head=64, layers=2, B=N, T=1.0, kind="visium", seed=41)
    net, sd = _build(m)
    net.eval()
    feats, expr, pos = _inputs(m)
    img, spot = embed_bank(net, expr.cuda(), pos.cuda(), feats.cuda(), group=group)
    want = []
    with torch.no_grad():
        for b0 in range(0, N, group):
            want.append(oracle.spot_embedding_ref(sd, expr[b0:b0 + group], pos[b0:b0 + group],
                                                  m["heads"], m["layers"]))
        want = torch.cat(want).numpy()
        want_img = oracle.projection_head_ref(feats, sd, "image_projection.").numpy()
    _close(spot, want, "spot_embeddings")
    _close(img, want_img, "image_embeddings")
    # and the module-attribute loop of the reference's get_embeddings gives the same
    with torch.no_grad():
        loop = torch.cat([net.embed_spots(expr[b0:b0 + group].cuda(), pos[b0:b0 + group].cuda())
                          for b0 in range(0, N, group)])
    _close(spot, loop.cpu().numpy(), "fused vs loop", rtol=1e-4)


def test_attention_row_block_streaming_equals_dense(monkeypatch):
    """Beyond the scratch budget the attention core streams the queries in row blocks and keeps no
    [heads, n, n] tensor (backward recomputes each block's probabilities): same output and gradients
    as the dense path, and as torch's float64 attention."""
    torch.manual_seed(3)
    n, heads, dh = 700, 8, 64
    qkv = (torch.randn(n, 3 * heads * dh, device="cuda") * 0.5).requires_grad_(True)
    w = torch.randn(n, heads * dh, device="cuda")
    out_d = mm.attention_core(qkv, heads, dh ** -0.5)
    (out_d * w).sum().backward()
    g_d = qkv.grad.clone()
    qkv.grad = None
    monkeypatch.setattr(mm, "ATTN_SCRATCH_BYTES", 1 << 20)
    assert mm._attn_block_rows(n, heads) == 128
    out_s = mm.attention_core(qkv, heads, dh ** -0.5)
    (out_s * w).sum().backward()
    g_s = qkv.grad.clone()
    _close(out_s, out_d.detach().cpu().numpy(), "streamed vs dense output", rtol=1e-5)
    _close(g_s, g_d.cpu().numpy(), "streamed vs dense grad", rtol=1e-5)
    q64 = qkv.detach().double().requires_grad_(True)
    q, k, v = (q64[:, i * heads * dh:(i + 1) * heads * dh].view(n, heads, dh).permute(1, 0, 2) for i in range(3))
    ref = (torch.softmax(q @ k.transpose(1, 2) * dh ** -0.5, -1) @ v).permute(1, 0, 2).reshape(n, heads * dh)
    (ref * w.double()).sum().backward()
    _close(out_s, ref.detach().cpu().numpy(), "streamed vs float64 output")
    _close(g_s, q64.grad.cpu().numpy(), "streamed vs float64 grad")


def test_deferred_weight_grads_equal_autograd_route():
    """model.deferred_weight_grads(): Linear weight / bias gradients computed on the side stream and
    written straight into .grad (fresh and accumulating) equal the ordinary autograd route."""
    import copy
    from mclstexp_b200 import model as mm
    torch.manual_seed(3)
    net = mm.mclSTExp_Attention("none", 1.0, 96, 171, 64, 4, 16, 2, targets="soft")
    net.image_encoder = torch.nn.Identity()
    net = net.cuda()
    ref = copy.deepcopy(net)
    g = torch.Generator(device="cuda").manual_seed(4)
    batch = {"image": torch.randn(200, 96, generator=g, device="cuda"),
             "expression": torch.rand(200, 171, generator=g, device="cuda"),
             "position": torch.randint(0, 64, (200, 2), generator=g, device="cuda").float()}
    for rounds in (1, 2):                       # second round accumulates into existing .grad
        ref(batch).backward()
        with mm.deferred_weight_grads():
            net(batch).backward()
        torch.cuda.synchronize()
        for (n, p), (_, q) in zip(net.named_parameters(), ref.named_parameters()):
            assert p.grad is not None, n
            assert torch.allclose(p.grad, q.grad, rtol=2e-4, atol=2e-5 * float(q.grad.abs().max()) + 1e-12), n


def test_graphed_step_with_deferred_weight_grads_trains():
    from mclstexp_b200 import model as mm
    from mclstexp_b200.graphs import GraphedTrainStep
    torch.manual_seed(5)
    net = mm.mclSTExp_Attention("none", 1.0, 96, 128, 64, 4, 16, 1, targets="eye")
    net.image_encoder = torch.nn.Identity()
    net = net.cuda()
    g = torch.Generator(device="cuda").manual_seed(6)
    batch = {"image": torch.randn(256, 96, generator=g, device="cuda"),
             "expression": torch.rand(256, 128, generator=g, device="cuda"),
             "position": torch.randint(0, 64, (256, 2), generator=g, device="cuda").float()}
    eager = net(batch)
    eager.backward()
    want = {n: p.grad.clone() for n, p in net.named_parameters()}
    del eager
    step = GraphedTrainStep(net, batch)
    loss = step(batch)
    torch.cuda.synchronize()
    for n, p in net.named_parameters():
        assert torch.allclose(p.grad, want[n], rtol=2e-4, atol=2e-5 * float(want[n].abs().max()) + 1e-12), n
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    l0 = float(loss)
    for _ in range(5):
        opt.zero_grad()
        loss = step(batch)
        opt.step()
    assert float(loss) < l0
