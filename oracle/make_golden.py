"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN CODE OBJECTS.

Runs only in the build container (needs /root/reference, which does not exist on
the GPU box); the fixtures it writes are committed and travel.  Test
infrastructure -- never imported by the product.

How each piece of reference code is reached without copying it:

* ``model.py`` is imported as a module with a stub ``timm`` (only used by
  ``ImageEncoder_VIT.__init__``, model.py:109).  ``ImageEncoder`` is replaced by
  an identity so ``mclSTExp_Attention.forward`` (model.py:225-247) runs verbatim
  on CNN *features* (the CNN is outside the path); ``Tensor.cuda`` is patched
  to the identity for the hard-coded ``.cuda()`` at model.py:243.
* ``find_matches`` is AST-extracted from evel_her2st.py:74-84 and
  evel_cscc.py:74-84 and exec'd (the files themselves are not importable: they
  ``os.listdir("D:\\...")`` at import, SURVEY.md section 8c).
* the weighted-average loops are module-level statements inside the fold loops
  (evel_her2st.py:174-187, evel_visium.py:193-205, evel_cscc.py:197-215); their
  AST nodes are lifted out by line range and exec'd in a namespace that provides
  ``spot_key``, ``expression_key``, ``image_query`` and ``find_matches``.
* BLEEP: ``cross_entropy`` (baselines/Bleep/models.py:228-234) is AST-extracted;
  the loss statements of ``CLIPModel.forward`` (:34-43) and ``CLIPModel_ViT.forward``
  (:70-79) are lifted by line range; the three aggregation variants are lifted
  from BLEEP_inference.ipynb cell 5.

Inputs are NOT stored: they are regenerated from seeds through
``mclstexp_b200.synth`` / ``oracle.make_state_dict`` (numpy PCG64), and a float64
checksum of every input is stored so a drifting generator is detected.
"""
from __future__ import annotations

import ast
import contextlib
import hashlib
import io
import json
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
sys.path.insert(0, ROOT)

from mclstexp_b200 import synth  # noqa: E402
from oracle import oracle  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def checksum(*arrays) -> float:
    s = 0.0
    for a in arrays:
        a = np.asarray(a, np.float64).ravel()
        s += float((a * (1.0 + (np.arange(a.size) % 7))).sum())
    return s


# ---------------------------------------------------------------- extraction
def _src(path):
    with open(os.path.join(REF, path)) as f:
        return f.read()


def extract_function(path: str, name: str, glb: dict):
    tree = ast.parse(_src(path))
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(mod, os.path.join(REF, path), "exec"), glb)
            return glb[name]
    raise KeyError(name)


def lift_statements(path_or_src: str, lo: int, hi: int, is_source=False):
    """Return a code object holding every innermost-enclosing statement whose
    line span lies inside [lo, hi]."""
    src = path_or_src if is_source else _src(path_or_src)
    tree = ast.parse(src)
    picked = []

    def visit(body):
        for st in body:
            end = getattr(st, "end_lineno", st.lineno)
            if st.lineno >= lo and end <= hi:
                picked.append(st)
            elif st.lineno <= hi and end >= lo:
                for field in ("body", "orelse", "finalbody"):
                    sub = getattr(st, field, None)
                    if isinstance(sub, list):
                        visit(sub)
    visit(tree.body)
    assert picked, (path_or_src[:40], lo, hi)
    mod = ast.Module(body=picked, type_ignores=[])
    ast.fix_missing_locations(mod)
    return compile(mod, "<reference %d-%d>" % (lo, hi), "exec")


def quiet_exec(code, ns):
    with contextlib.redirect_stdout(io.StringIO()):
        exec(code, ns)


# ---------------------------------------------------------------- retrieval
def golden_retrieval():
    import torch.nn.functional as F
    glb = {"torch": torch, "F": F, "np": np}
    fm_her = extract_function("evel_her2st.py", "find_matches", dict(glb))
    fm_cscc = extract_function("evel_cscc.py", "find_matches", dict(glb))
    loops = {
        # file, first line (find_matches call), last line of the loop, weight mode
        "her2st": ("evel_her2st.py", 174, 187, "inv_sq_l1", fm_her),
        "visium": ("evel_visium.py", 193, 205, "inv_sq_l2", extract_function(
            "evel_visium.py", "find_matches", dict(glb))),
        "cscc": ("evel_cscc.py", 197, 215, "inv_sq_l2", fm_cscc),
    }
    out = {}
    meta = {}
    cases = [
        # name, flavour, N, Q, D, G, seed
        ("iid", "iid", 700, 37, 256, 96, 101),
        ("clustered", "clustered", 900, 29, 256, 50, 202),
    ]
    for name, flavour, N, Q, D, G, seed in cases:
        bank = synth.embeddings(N, D, seed, flavour)
        qry = synth.embeddings(Q, D, seed + 1, flavour)
        expr = synth.expression(N, G, seed + 2)
        meta[name] = dict(flavour=flavour, N=N, Q=Q, D=D, G=G, seed=seed,
                          checksum=checksum(bank, qry, expr))
        for k in (1, 50, 200):
            with contextlib.redirect_stdout(io.StringIO()):
                idx = fm_her(bank, qry, top_k=k)
                val, idx2 = fm_cscc(bank, qry, top_k=k)
            assert np.array_equal(idx, idx2)
            out[f"{name}/find_matches/k{k}/indices"] = idx.astype(np.int32)
            out[f"{name}/find_matches/k{k}/values"] = val
        # Q == 1 squeeze quirk (evel_her2st.py:82 ``squeeze(0)``)
        with contextlib.redirect_stdout(io.StringIO()):
            idx1 = fm_her(bank, qry[:1], top_k=5)
        out[f"{name}/find_matches/q1/indices"] = idx1.astype(np.int32)
        # the fold-loop bodies, verbatim, with the reference's own top_k literals
        for tag, (path, lo, hi, mode, fm) in loops.items():
            code = lift_statements(path, lo, hi)
            ns = {"np": np, "find_matches": fm, "spot_key": bank, "expression_key": expr,
                  "image_query": qry}
            quiet_exec(code, ns)
            out[f"{name}/loop_{tag}/indices"] = ns["indices"].astype(np.int32)
            out[f"{name}/loop_{tag}/emb_pred"] = ns["matched_spot_embeddings_pred"]
            out[f"{name}/loop_{tag}/expr_pred"] = ns["matched_spot_expression_pred"]
            meta[name][f"loop_{tag}"] = dict(mode=mode, lines=[path, lo, hi],
                                             k=int(ns["indices"].shape[1]))
        # BLEEP aggregation variants (notebook cell 5)
        nb = json.load(open(os.path.join(REF, "baselines/Bleep/BLEEP_inference.ipynb")))
        cell5 = "".join(nb["cells"][5]["source"])
        tree = ast.parse(cell5)
        for st in tree.body:
            if isinstance(st, ast.If) and isinstance(st.test, ast.Compare) and \
                    getattr(st.test.left, "id", "") == "method":
                method = st.test.comparators[0].value
                mod = ast.Module(body=st.body, type_ignores=[])
                ns = {"np": np, "find_matches": fm_her, "spot_key": bank, "expression_key": expr,
                      "image_query": qry}
                quiet_exec(compile(mod, "<bleep cell5 %s>" % method, "exec"), ns)
                out[f"{name}/bleep_{method}/indices"] = ns["indices"].astype(np.int32)
                out[f"{name}/bleep_{method}/emb_pred"] = ns["matched_spot_embeddings_pred"]
                out[f"{name}/bleep_{method}/expr_pred"] = ns["matched_spot_expression_pred"]

    # exact-arithmetic known-answer case (+-1 entries): values are implementation independent
    N, Q, D, seed = 1500, 23, 256, 303
    bank = synth.pm1_embeddings(N, D, seed)
    qry = synth.pm1_embeddings(Q, D, seed + 1)
    with contextlib.redirect_stdout(io.StringIO()):
        val, idx = fm_cscc(bank, qry, top_k=50)
    out["pm1/find_matches/k50/indices"] = idx.astype(np.int32)
    out["pm1/find_matches/k50/values"] = val
    meta["pm1"] = dict(N=N, Q=Q, D=D, seed=seed, checksum=checksum(bank, qry))
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, "retrieval.npz"), **out)
    print("retrieval.npz:", len(out), "arrays")


# ---------------------------------------------------------------- model / loss
def import_reference_model():
    sys.modules.setdefault("timm", types.ModuleType("timm"))
    sys.path.insert(0, REF)
    import model as ref_model  # noqa
    sys.path.pop(0)

    class _Features(torch.nn.Module):          # stands in for the stock CNN (outside the path)
        def forward(self, x):
            return x
    ref_model.ImageEncoder = _Features
    return ref_model


def golden_model():
    ref_model = import_reference_model()
    torch.Tensor.cuda = lambda self, *a, **k: self          # model.py:243 hard-codes .cuda()
    torch.manual_seed(0)
    out, meta = {}, {}
    cases = [
        # name, G, E, heads, dim_head, layers, B, T, position kind, seed
        ("small", 40, 64, 8, 64, 2, 24, 1.0, "st", 7),
        ("odd", 171, 96, 4, 32, 1, 33, 0.7, "visium", 8),
    ]
    for name, G, E, H, dh, L, B, T, kind, seed in cases:
        sd = oracle.make_state_dict(G, E, 256, H, dh, L, seed)
        m = ref_model.mclSTExp_Attention(encoder_name="densenet121", temperature=T, image_dim=E,
                                         spot_dim=G, projection_dim=256, heads_num=H,
                                         heads_dim=dh, head_layers=L, dropout=0.)
        missing = m.load_state_dict(sd, strict=True)
        assert not missing.missing_keys and not missing.unexpected_keys
        feats = torch.tensor(synth.image_features(B, E, seed + 1))
        expr = torch.tensor(synth.expression(B, G, seed + 2))
        pos = torch.tensor(synth.positions(B, seed + 3, kind))
        meta[name] = dict(G=G, E=E, heads=H, dim_head=dh, layers=L, B=B, T=T, kind=kind, seed=seed,
                          checksum=checksum(feats, expr, pos, sd["x_embed.weight"][:64],
                                            sd["spot_projection.fc.weight"]))
        # verbatim forward/backward of the whole path: model.py:225-247
        loss = m({"image": feats, "expression": expr, "position": pos})
        loss.backward()
        out[f"{name}/loss"] = loss.detach().numpy()
        for k, p in m.named_parameters():
            if k in ("x_embed.weight", "y_embed.weight"):
                col = 0 if k.startswith("x") else 1
                rows = torch.unique(pos[:, col].long())
                out[f"{name}/grad_rows/{k}"] = rows.numpy().astype(np.int32)
                out[f"{name}/grad/{k}"] = p.grad[rows].numpy()
                mask = torch.ones(p.shape[0], dtype=torch.bool)
                mask[rows] = False
                assert float(p.grad[mask].abs().sum()) == 0.0
            else:
                out[f"{name}/grad/{k}"] = p.grad.numpy()
        # attribute-level eval surface used by evel_her2st.py:48-69
        with torch.no_grad():
            img_emb = m.image_projection(m.image_encoder(feats))
            h = expr + m.x_embed(pos[:, 0].long()) + m.y_embed(pos[:, 1].long())
            h = h.unsqueeze(0)
            blk0 = m.spot_encoder[0](h)
            attn0 = m.spot_encoder[0].attn(h)
            enc = m.spot_encoder(h)
            spot_emb = m.spot_projection(enc).squeeze(0)
        out[f"{name}/image_embeddings"] = img_emb.numpy()
        out[f"{name}/spot_embeddings"] = spot_emb.numpy()
        out[f"{name}/block0"] = blk0.numpy()
        out[f"{name}/attn0"] = attn0.numpy()
        out[f"{name}/encoder"] = enc.numpy()

    # losses on free-standing embeddings (LayerNorm-like rows), eye + both soft variants
    import torch.nn.functional as F
    from torch import nn
    glb = {"torch": torch, "nn": nn, "F": F}
    bleep_ce = extract_function("baselines/Bleep/models.py", "cross_entropy", glb)
    # model.py has the same six lines twice (mclSTExp_MLP :193-198 and
    # mclSTExp_Attention :242-247); the line range selects the second.
    eye_fn = lift_as_function("model.py", 242, 247)
    soft_div = lift_as_function("baselines/Bleep/models.py", 34, 43)
    soft_mul = lift_as_function("baselines/Bleep/models.py", 70, 79)
    for name, B, D, T, seed in (("b48", 48, 256, 1.0, 31), ("b65_t07", 65, 256, 0.7, 32),
                                ("b16_t2", 16, 32, 2.0, 33)):
        S0 = synth.embeddings(B, D, seed, "clustered", centres=5)
        I0 = synth.embeddings(B, D, seed + 1, "clustered", centres=5)
        if D == 256:
            S0 *= 0.25          # logits up to +-16 instead of +-256: keeps the soft targets non-degenerate
            I0 *= 0.25
        meta[f"loss_{name}"] = dict(B=B, D=D, T=T, seed=seed, scaled=(D == 256),
                                    checksum=checksum(S0, I0))
        for tag, code in (("eye", eye_fn), ("soft_div", soft_div), ("soft_mul", soft_mul)):
            S = torch.tensor(S0, requires_grad=True)
            I = torch.tensor(I0, requires_grad=True)
            ns = {"torch": torch, "F": F, "cross_entropy": bleep_ce}
            exec(code, ns)
            loss = ns["_lifted"](types.SimpleNamespace(temperature=T), S, I)
            loss.backward()
            out[f"loss_{name}/{tag}/loss"] = loss.detach().numpy()
            out[f"loss_{name}/{tag}/dS"] = S.grad.numpy()
            out[f"loss_{name}/{tag}/dI"] = I.grad.numpy()
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    out = compact_model(out)
    np.savez_compressed(os.path.join(OUT, "model.npz"), **out)
    print("model.npz:", len(out), "arrays")


GRAD_SAMPLE = 2048          # entries kept of each parameter gradient: model.npz stays well under 1 MB


def sha256(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def compact_model(out: dict) -> dict:
    """The form model.npz is committed in.  A parameter gradient ``<case>/grad/<name>`` becomes a
    fixed, seeded sample of its entries (``/idx`` flat indices, ``/val`` values) plus ``/shape`` and
    the ``/absmax`` and ``/norm`` of the whole array (the tolerances the tests use); a loss gradient
    ``loss_*/<tag>/dS|dI``, which the tests compare bit for bit, becomes its ``/sha256`` digest."""
    small = {}
    for key, a in out.items():
        if "/grad/" in key:
            flat = a.ravel()
            if flat.size > GRAD_SAMPLE:
                idx = np.sort(np.random.default_rng(0).choice(flat.size, GRAD_SAMPLE, replace=False))
            else:
                idx = np.arange(flat.size)
            small[key + "/idx"] = idx.astype(np.int32)
            small[key + "/val"] = flat[idx]
            small[key + "/shape"] = np.array(a.shape, dtype=np.int64)
            small[key + "/absmax"] = np.float64(np.abs(flat).max())
            small[key + "/norm"] = np.float64(np.linalg.norm(flat.astype(np.float64)))
        elif key.startswith("loss_") and key.endswith(("/dS", "/dI")):
            small[key + "/sha256"] = np.array(sha256(a))
        else:
            small[key] = a
    return small


def lift_as_function(path, lo, hi):
    """Lift the statements of [lo, hi] (ending in the reference's own ``return``)
    into ``def _lifted(self, spot_embeddings, image_embeddings)`` -- the names the
    reference's forward() uses for them."""
    tree = ast.parse(_src(path))
    picked = []

    def visit(body):
        for st in body:
            end = getattr(st, "end_lineno", st.lineno)
            if st.lineno >= lo and end <= hi:
                picked.append(st)
            elif st.lineno <= hi and end >= lo:
                for field in ("body", "orelse"):
                    sub = getattr(st, field, None)
                    if isinstance(sub, list):
                        visit(sub)
    visit(tree.body)
    assert picked and isinstance(picked[-1], ast.Return), (path, lo, hi)
    fn = ast.parse("def _lifted(self, spot_embeddings, image_embeddings):\n    pass").body[0]
    fn.body = picked
    mod = ast.Module(body=[fn], type_ignores=[])
    ast.fix_missing_locations(mod)
    return compile(mod, "<%s %d-%d>" % (path, lo, hi), "exec")


def golden_metrics():
    """utils.get_R (utils.py:52-65) imported from the reference and the metric lines of the fold
    loop (evel_her2st.py:201-221) lifted verbatim; AnnData is replaced by a minimal stand-in with
    the three members those lines use (.X, .shape, column selection by name)."""
    sys.path.insert(0, REF)
    import utils as ref_utils
    sys.path.pop(0)

    class Ann:                                        # what anndata.AnnData offers to those lines
        def __init__(self, X, names=None):
            self.X = np.asarray(X)
            self.shape = self.X.shape
            self.var_names = np.array(names if names is not None else [str(i) for i in range(self.X.shape[1])])

        def __getitem__(self, key):
            _, names = key
            pos = {n: i for i, n in enumerate(self.var_names)}
            cols = [pos[n] for n in names]
            return Ann(self.X[:, cols], list(names))

    out, meta = {}, {}
    for name, Q, G, seed in (("a", 300, 60, 71), ("b", 57, 130, 72)):
        true = synth.expression(Q, G, seed).astype(np.float64)
        rng = np.random.default_rng(seed)
        pred = 0.6 * true + 0.4 * rng.random((Q, G)) + 0.05 * rng.standard_normal((Q, G))
        pred[:, 3] = 0.25                                  # constant column -> pearsonr is NaN
        pred = pred.astype(np.float32).astype(np.float64)    # stored as float32 in the fixture
        meta[name] = dict(Q=Q, G=G, seed=seed, checksum=checksum(true, pred))
        code = lift_statements("evel_her2st.py", 201, 221)
        ns = {"np": np, "get_R": ref_utils.get_R, "adata_ture": Ann(true), "adata_pred": Ann(pred),
              "true": true, "pred": pred, "heg_pcc_list": [], "hvg_pcc_list": [], "mse_list": [],
              "mae_list": []}
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            quiet_exec(code, ns)
        out[f"{name}/heg_pcc"] = np.array(ns["heg_pcc_list"][0])
        out[f"{name}/hvg_pcc"] = np.array(ns["hvg_pcc_list"][0])
        out[f"{name}/mse"] = np.array(ns["mse_list"][0])
        out[f"{name}/mae"] = np.array(ns["mae_list"][0])
        out[f"{name}/pred"] = pred.astype(np.float32)        # noise is not regenerable from synth alone
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, "metrics.npz"), **out)
    print("metrics.npz:", len(out), "arrays")


IO_SIZES = [5 + (7 * i) % 13 for i in range(32)]          # spots per slide (32 her2st slides)
IO_GENES = 24


def io_inputs():
    """Seeded stand-ins for what the fold loop reads from disk: all image / spot embeddings
    (rows in slide order) and one [G, n_i] expression matrix per slide."""
    n = sum(IO_SIZES)
    img = synth.embeddings(n, 256, 301, "iid")
    spot = synth.embeddings(n, 256, 302, "iid")
    expr = synth.expression(n, IO_GENES, 303).astype(np.float64)
    mats, start = [], 0
    for s in IO_SIZES:
        mats.append(np.ascontiguousarray(expr[start:start + s].T))
        start += s
    return img, spot, mats


def golden_io():
    """The reference's own writer loop (evel_her2st.py:109-117) and fold-loop loading code
    (:145-172) executed verbatim in a scratch directory (their paths are relative); the fixture
    keeps SHA-256 digests and shapes of the four arrays they produce."""
    import tempfile
    img, spot, mats = io_inputs()
    names = [f"S{i:02d}" for i in range(32)]
    writer = lift_statements("evel_her2st.py", 109, 117)
    loader = lift_statements("evel_her2st.py", 145, 172)
    out, cwd = {}, os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for fold in (0, 17, 31):
                save_path = f"./embedding_result/her2st_result/embeddings_{fold}/"
                os.makedirs(save_path)
                quiet_exec(writer, {"np": np, "datasize": IO_SIZES, "img_embeddings_all": img,
                                    "spot_embeddings_all": spot, "save_path": save_path})
                ns = {"np": np, "os": os, "fold": fold, "names": names, "spot_expressions": list(mats)}
                quiet_exec(loader, ns)
                for key in ("spot_key", "expression_key", "image_query", "expression_gt"):
                    a = np.ascontiguousarray(ns[key])
                    out[f"{fold}/{key}"] = dict(shape=list(a.shape), dtype=str(a.dtype),
                                                sha256=hashlib.sha256(a.tobytes()).hexdigest())
        finally:
            os.chdir(cwd)
    with open(os.path.join(OUT, "io.json"), "w") as f:
        json.dump({"sizes": IO_SIZES, "genes": IO_GENES, "arrays": out}, f, indent=1)
    print("io.json:", len(out), "digests")


if __name__ == "__main__":
    torch.set_num_threads(1)        # float32 CPU products split over many threads sum in another order
    os.makedirs(OUT, exist_ok=True)
    if "--io-only" in sys.argv:
        golden_io()
        sys.exit(0)
    if "--metrics-only" not in sys.argv:
        golden_retrieval()
        golden_model()
    golden_metrics()
    golden_io()
