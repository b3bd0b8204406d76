"""find_matches and the resident-bank retrieval at several embedding widths on one GPU (cfg4 shape
by default: N = 1 000 000 bank spots, Q = 65 536 queries, k = 50, G = 1000 genes, clustered inputs
generated on the device with bench.py's recipe).  Per width it reports

  * the per-kernel times of find_matches (+ L2 distances), averaged over --reps calls after warm-ups;
  * Bank.retrieve_device ms per call (CUDA events, --reps calls after warm-ups, packed image resident);
  * last_counters() of find_matches;
  * parity of --parity sampled rows: indices and values against oracle.find_matches_spec_rows, the
    expression average against oracle.weighted_average_spec;
  * with --exact-sample S and D in --exact-dims: the exact-only path on S queries, timed and
    extrapolated linearly to Q (labelled as extrapolated).

The card name, power limit and maximum SM clock are read in the same run.  One JSON document goes to
--out (and stdout).

    python tools/width_sweep.py --dims 256,384,512 --out profiles/width_sweep.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import make_inputs_device  # noqa: E402
from mclstexp_b200 import _lib, retrieval  # noqa: E402
from oracle import oracle  # noqa: E402


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out = f"unavailable: {e}"
    return {"nvidia_smi": out, "torch_name": torch.cuda.get_device_name(0)}


def event_ms(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def one_width(D, a, dev):
    cfg = {"N": a.N, "Q": a.Q, "D": D, "G": a.G}
    bank, qry, expr = make_inputs_device(cfg, 1234 + D, dev, "clustered")
    k = a.k
    res = {"D": D}
    # ---- find_matches: per-kernel trace
    for _ in range(a.warmup):
        retrieval.find_matches_device(bank, qry, k, dist_p=2)
    torch.cuda.synchronize()
    agg = {}
    for _ in range(a.reps):
        _lib.profile_enable(True)
        retrieval.find_matches_device(bank, qry, k, dist_p=2)
        for n, t in _lib.profile_collect():
            agg[n] = agg.get(n, 0.0) + t / a.reps
        _lib.profile_enable(False)
    res["find_matches_kernels_ms"] = {n: round(t, 3) for n, t in agg.items()}
    res["find_matches_total_ms"] = round(sum(agg.values()), 3)
    res["find_matches_counters"] = retrieval.last_counters()
    res["find_matches_tc_eligible"] = retrieval.tc_eligible(a.N, D, k)
    # ---- resident bank
    b = retrieval.Bank(bank, expr)
    out = {}

    def call():
        out["r"] = b.retrieve_device(qry, k, "inv_sq_l2")
    for _ in range(a.warmup):
        call()
    res["bank_retrieve_device_ms"] = round(event_ms(call, a.reps), 3)
    res["bank_counters"] = retrieval.last_counters()
    res["bank_keeps_packed_image"] = bool(b._packed)
    idx, val, _, ex = out["r"]
    # ---- parity of sampled rows
    rows = np.random.default_rng(D).choice(a.Q, a.parity, replace=False)
    hb = bank.cpu().numpy()
    hq = qry.cpu().numpy()[rows]
    sval, sidx = oracle.find_matches_spec_rows(hb, hq, k)
    gi, gv, ge = idx.cpu().numpy()[rows], val.cpu().numpy()[rows], ex.cpu().numpy()[rows]
    _, ex64 = oracle.weighted_average_spec(hb, expr.cpu().numpy(), hq, sidx, "inv_sq_l2")
    rel = np.abs(ge - ex64) / np.maximum(np.abs(ex64), 1e-6)
    res["parity"] = {"rows": int(a.parity), "indices_equal": bool(np.array_equal(gi, sidx)),
                     "values_equal": bool(np.array_equal(gv, sval)),
                     "expr_max_rel_err_vs_float64": float(rel.max())}
    # ---- exact-only path on a sample, extrapolated
    if D in a.exact_dims and a.exact_sample > 0:
        S = min(a.exact_sample, a.Q)
        retrieval.find_matches_device(bank, qry[:128], k, exact_only=True)       # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev, ei = retrieval.find_matches_device(bank, qry[:S], k, exact_only=True)
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        res["exact_only"] = {"queries_timed": S, "ms_timed": round(ms, 3),
                             "ms_extrapolated_to_Q": round(ms * a.Q / S, 1),
                             "note": f"extrapolated linearly from {S} queries to Q = {a.Q}, not measured at Q",
                             "equals_tc_path_on_sample": bool(torch.equal(ei, retrieval.find_matches_device(
                                 bank, qry[:S], k)[1]))}
    del b, out, bank, qry, expr
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=1_000_000)
    ap.add_argument("--Q", type=int, default=65536)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--G", type=int, default=1000)
    ap.add_argument("--dims", default="256,384,512")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--parity", type=int, default=64)
    ap.add_argument("--exact-sample", type=int, default=2048)
    ap.add_argument("--exact-dims", default="512")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    a.exact_dims = [int(x) for x in a.exact_dims.split(",") if x]
    assert torch.cuda.is_available(), "width_sweep.py needs a GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    doc = {"card": card(), "shape": {"N": a.N, "Q": a.Q, "k": a.k, "G": a.G, "flavour": "clustered"},
           "widths": [one_width(int(D), a, dev) for D in a.dims.split(",")]}
    doc["card_after"] = card()
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
