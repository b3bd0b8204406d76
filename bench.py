#!/usr/bin/env python
"""Benchmark of the mclSTExp retrieval hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4|cfg3|cfg1|cfg5|cfg2] [--impl reference]

A "step" is one pass of the fold-loop body of the reference (evel_her2st.py:174-187:
find_matches + top-k weighted expression average) over one synthetic batch:
N bank spots x Q query spots, 256-d embeddings, top-50, 1000 HVGs.  The default
workload is BASELINE.json configs[3] ("cfg4": 1M-spot bank x 64k queries), the
configuration the north-star target is quoted on; it fits one B200.

One JSON line is printed by rank 0:
  value   = query spots / s with every input resident in HBM (CUDA events, max over ranks)
  e2e     = the same through the public host-array API (retrieval.retrieve): pinned-host
            inputs copied H2D and results read back D2H inside the timed region
  roofline= dominant kernel, algorithmic FLOPs or bytes / its CUDA-event time (live)
  cpu_baseline = the oracle's restatement of the reference path (torch CPU + NumPy, the
            reference's own libraries) on a bounded query sample, host cores of this box
  extra   = contrastive-loss steps/s (second half of the BASELINE metric) when available

  parity_check = after the timed region (outside it): >= 64 sampled query rows of the step's own
            result re-derived on the host with the oracle's float64 spec against the FULL bank
            (indices and float32 values bit-equal, predicted expression rtol 1e-3); done at every N,
            every rank checks rows of its own query slice; a mismatch exits non-zero

`--workload cfg5` prints the second half of the BASELINE metric as its own line: contrastive-loss
steps/s (soft targets, fwd+bwd) at B = 32768 with the whole 256..32768 sweep, a `torch_gpu` field
(the reference's own formulation, baselines/Bleep/models.py:34-43, in stock PyTorch fp32 on the same
B200) and a CPU baseline; `--workload cfg2` does the same for the B = 1024 training step (spot
self-attention + heads + soft loss).

`--impl reference` times the CPU path of the selected workload alone (all host threads) and prints
the same line with "impl": "reference".

`--dump-outputs DIR` writes what the timed path returned in its last step (retrieval: indices,
values, expr_pred; cfg5: loss, dS, dI; cfg2: loss and every parameter gradient) as DIR/<name>.npy.
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from mclstexp_b200 import synth  # noqa: E402

METRIC = "retrieval query spots/sec (cosine top-k + weighted expression average)"
UNIT = "query spots/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"],
                    source="MEASURED_PEAKS.json (measured)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="B200_PROFILING.md fallback")


# --------------------------------------------------------------------------- inputs
def make_inputs_device(cfg, seed, device, flavour="clustered"):
    """Seeded synthetic inputs generated on the device (big configs); same recipe as
    mclstexp_b200.synth (SURVEY.md section 8d)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    N, Q, D, G = cfg["N"], cfg["Q"], cfg["D"], cfg["G"]

    def emb(rows, centres):
        if flavour == "iid":
            return torch.randn(rows, D, generator=g, device=device)
        which = torch.randint(0, centres.shape[0], (rows,), generator=g, device=device)
        x = centres[which] + torch.randn(rows, D, generator=g, device=device)
        x = x - x.mean(1, keepdim=True)
        return x / (x.std(1, keepdim=True, unbiased=False) + 1e-6)

    centres = 4.0 * torch.randn(64, D, generator=g, device=device)
    bank = emb(N, centres)
    qry = emb(Q, centres)
    expr = torch.empty(N, G, device=device)
    step = 1 << 16
    for r0 in range(0, N, step):
        r1 = min(N, r0 + step)
        # Gamma(0.5, 2) == chi-square(1) * 1.0 -> (randn^2)
        lam = torch.randn(r1 - r0, G, generator=g, device=device).square_()
        cnt = torch.poisson(lam, generator=g)
        lib = cnt.sum(1, keepdim=True).clamp_(min=1.0)
        expr[r0:r1] = torch.log10(1.0 + cnt / lib * 1e4)
    return bank, qry, expr


# --------------------------------------------------------------------------- outputs
DUMP_BYTES = 60 << 20          # under 64 MB whether a megabyte is 10^6 or 2^20 bytes


def dump_outputs(dirname, arrays, seed=20261020):
    """Writes each array of `arrays` (name -> tensor the timed path returned) as DIR/<name>.npy:
    float32 stays float32, every other dtype becomes float64 (indices are exact in it).  All files
    together stay within 64 MB: smallest first, an array is kept whole while it fits its share of
    what is left; a larger one keeps a fixed, seeded sample of its rows, and the row numbers go to
    DIR/<name>.rows.npy, so two builds run with the same arguments can be compared file by file."""
    os.makedirs(dirname, exist_ok=True)
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a if a.dtype == np.float32 else a.astype(np.float64)
    left = DUMP_BYTES
    order = sorted(host, key=lambda n: host[n].nbytes)
    for i, name in enumerate(order):
        a = host[name]
        share = left // (len(order) - i) - 256                 # 128-byte .npy header per file
        if a.nbytes <= share:
            np.save(os.path.join(dirname, name + ".npy"), a)
            left -= a.nbytes + 128
            continue
        row_bytes = a.nbytes // a.shape[0] + 8                 # + its float64 row number
        n = max(1, share // row_bytes)
        rows = np.sort(np.random.default_rng(seed).choice(a.shape[0], n, replace=False))
        np.save(os.path.join(dirname, name + ".npy"), a[rows])
        np.save(os.path.join(dirname, name + ".rows.npy"), rows.astype(np.float64))
        left -= n * row_bytes + 256


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, index=0, period=0.02):
        self.samples, self.reasons, self.period, self.index = [], set(), period, index
        self._stop = threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "sw_thermal_slowdown": 0x20,
                 "applications_clocks_setting": 0x2, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------- CPU reference arm
_CPU_INPUTS: dict = {}


def cpu_reference_time(cfg, mode, budget_s=20.0, flavour="clustered", threads=None):
    """Times the oracle's literal restatement of evel_her2st.py:74-84 + :175-187 on a bounded
    query sample of the SAME workload (full bank), all host threads.  cfg4 cannot run whole on
    a CPU (the Q x N float32 similarity matrix alone is 262 GB, SURVEY.md 8d): queries go in
    chunks of <= 512 and the rate is per query."""
    from oracle import oracle
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    N, D, G, k = cfg["N"], cfg["D"], cfg["G"], cfg["k"]
    # the same recipe and seed as the GPU arm (clustered embeddings, Poisson expression), drawn
    # with the CPU generator
    key = (N, D, G, cfg["Q"], flavour)
    if key not in _CPU_INPUTS:
        # the GPU arm's own inputs (same recipe, seed and generator; drawn on the GPU when there is
        # one -- data generation is outside every timed region -- else with the CPU generator)
        _CPU_INPUTS.clear()
        gdev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))) if torch.cuda.is_available() \
            else torch.device("cpu")
        bank_t, qry_t, expr_t = make_inputs_device(cfg, 1234 + 4, gdev, flavour)
        _CPU_INPUTS[key] = (bank_t.cpu().numpy(), qry_t[:16384].cpu().numpy(), expr_t.cpu().numpy())
        del bank_t, qry_t, expr_t
        if gdev.type == "cuda":
            torch.cuda.empty_cache()
    bank, qry_all, expr = _CPU_INPUTS[key]
    done, t_total, chunk = 0, 0.0, 64
    cap = min(cfg["Q"], 16384)
    while True:
        qry = qry_all[done:done + chunk]
        chunk = qry.shape[0]
        t0 = time.perf_counter()
        oracle.retrieve_ref(bank, expr, qry, k, mode)
        dt = time.perf_counter() - t0
        done += chunk
        t_total += dt
        if t_total >= budget_s or done >= cap:
            break
        per_q = t_total / done
        chunk = int(max(1, min(512, cap - done, (budget_s - t_total) / per_q)))
    return dict(value=done / t_total, unit=UNIT, cores=threads, kind="port",
                sample=f"{done} of {cfg['Q']} queries (chunks <= 512) against the full "
                       f"{N}-spot bank, k={k}, G={G}, {t_total:.1f} s of CPU time; per-query rate, "
                       "i.e. the whole-workload figure is a linear EXTRAPOLATION from this sample",
                torch=torch.__version__, numpy=np.__version__), t_total, done


# --------------------------------------------------------------------------- second metric
def _time_cuda(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def loss_sweep(dev, peaks, world, rank, quick):
    """Contrastive-loss fwd+bwd steps/s (soft targets, D=256) over the BASELINE cfg5 batch sweep;
    at world > 1 the batch is the GLOBAL batch, sharded by rows with embedding all-gather."""
    from mclstexp_b200 import loss as mloss
    out = {}
    sizes = [256, 1024, 4096, 32768] if quick else synth.CONFIGS["cfg5"]["B_sweep"]
    g = torch.Generator(device=dev)
    g.manual_seed(99)
    for B in sizes:
        if B % (128 * world) != 0:
            continue
        x = torch.randn(B, 256, generator=g, device=dev)
        S = ((x - x.mean(1, keepdim=True)) / x.std(1, keepdim=True)).requires_grad_(True)
        y = torch.randn(B, 256, generator=g, device=dev)
        I = ((y - y.mean(1, keepdim=True)) / y.std(1, keepdim=True)).requires_grad_(True)
        if world > 1:
            from mclstexp_b200.distributed import contrastive_loss_sharded
            rows = B // world
            Sl = S.detach()[rank * rows:(rank + 1) * rows].clone().requires_grad_(True)
            Il = I.detach()[rank * rows:(rank + 1) * rows].clone().requires_grad_(True)

            def step():
                l = contrastive_loss_sharded(Sl, Il, 1.0, "soft")
                l.backward()
        else:
            def step():
                l = mloss.contrastive_loss(S, I, 1.0, "soft")
                l.backward()
        ms = _time_cuda(step)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        flops = 14.0 * B * B * 256
        out[str(B)] = {"steps_per_s": 1e3 / ms, "ms": ms,
                       "frac_of_bf16_sustained": flops / (ms * 1e-3) / (peaks["tf_sust"] * 1e12 * world)}
    return out


def train_step_cfg2(dev):
    """BASELINE cfg2: spot self-attention + projection heads + soft-target loss, fwd+bwd, B=1024."""
    from torch import nn
    from mclstexp_b200 import model as mm
    res = {}
    for G in (171, 1000):
        net = mm.mclSTExp_Attention("none", 1.0, 1024, G, 256, 8, 64, 2, targets="soft")
        net.image_encoder = nn.Identity()
        net = net.to(dev)
        g = torch.Generator(device=dev)
        g.manual_seed(7)
        batch = {"image": torch.randn(1024, 1024, generator=g, device=dev),
                 "expression": torch.rand(1024, G, generator=g, device=dev),
                 "position": torch.randint(0, 64, (1024, 2), generator=g, device=dev).float()}

        def step():
            net.zero_grad(set_to_none=True)
            net(batch).backward()
        ms = _time_cuda(step, iters=5, warm=2)
        res[f"G{G}"] = {"ms_per_step": ms, "steps_per_s": 1e3 / ms}
        try:                                   # whole step of train.py:36-38, optimiser included
            import copy
            from mclstexp_b200.optim import TrainOptimizer
            for name in ("stock_adam", "lazy_tables"):
                net2 = copy.deepcopy(net)
                opt = (torch.optim.Adam(net2.parameters(), lr=1e-4, weight_decay=1e-3) if name == "stock_adam"
                       else TrainOptimizer(net2, lr=1e-4, weight_decay=1e-3))

                def full_step():
                    opt.zero_grad()
                    net2(batch).backward()
                    opt.step()
                res[f"G{G}"][f"with_optimizer_{name}_ms"] = _time_cuda(full_step, iters=5, warm=2)
                del net2, opt
        except Exception as e:                 # report, do not hide
            res[f"G{G}"]["optimizer_error"] = f"{type(e).__name__}: {e}"[:200]
        try:                                   # same step replayed from a CUDA graph
            from mclstexp_b200.graphs import GraphedTrainStep
            gstep = GraphedTrainStep(net, batch)
            msg = _time_cuda(lambda: gstep(batch), iters=10, warm=2)
            res[f"G{G}"].update({"graph_ms_per_step": msg, "graph_steps_per_s": 1e3 / msg})
        except Exception as e:                 # report, do not hide
            res[f"G{G}"]["graph_error"] = f"{type(e).__name__}: {e}"[:200]
    return res


def bank_build(dev):
    """SURVEY 8f rank 1: fused eval embedding forward (batches of 32 un-shuffled spots, as
    evel_her2st.py:24,47-70) over 131 072 spots, G = 785 (her2st), vs the per-batch module loop."""
    from torch import nn
    from mclstexp_b200 import model as mm
    from mclstexp_b200.embed import embed_bank
    N, G = 131072, 785
    net = mm.mclSTExp_Attention("none", 1.0, 1024, G, 256, 8, 64, 2)
    net.image_encoder = nn.Identity()
    net = net.to(dev).eval()
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    expr = torch.rand(N, G, generator=g, device=dev)
    pos = torch.randint(0, 64, (N, 2), generator=g, device=dev).float()
    ms = _time_cuda(lambda: embed_bank(net, expr, pos), iters=3, warm=1)
    with torch.no_grad():
        ms_loop = _time_cuda(lambda: [net.embed_spots(expr[b:b + 32], pos[b:b + 32]) for b in range(0, 4096, 32)],
                             iters=2, warm=1) * (N / 4096)
    return {"spots": N, "genes": G, "fused_ms": ms, "fused_spots_per_s": N / (ms * 1e-3),
            "per_batch_loop_ms_extrapolated": ms_loop}



# --------------------------------------------------------------------------- loss / train-step workloads
LOSS_METRIC = "contrastive-loss steps/sec (soft targets, forward + backward, D=256)"
TRAIN_METRIC = "training steps/sec (spot self-attention + projection heads + soft-target loss, fwd+bwd)"
_FLUSH = {}


def _flush_l2(dev):
    """Writes a buffer larger than the 126 MB L2 (timing rules: flush between timed iterations)."""
    if dev not in _FLUSH:
        _FLUSH[dev] = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    _FLUSH[dev].fill_(1)


def _time_steps(fn, steps, warmup, dev, flush=True):
    """Mean device milliseconds of fn() over `steps` calls, each bracketed by its own CUDA events on
    the current stream, L2 flushed between calls (outside the events)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(steps):
        if flush:
            _flush_l2(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / steps


def _ln_rows(B, D, g, dev):
    x = torch.randn(B, D, generator=g, device=dev)
    return (x - x.mean(1, keepdim=True)) / x.std(1, keepdim=True)      # what ProjectionHead's LayerNorm leaves


def torch_soft_loss(S, I, T):
    """The reference's own formulation in stock PyTorch (baselines/Bleep/models.py:34-43, :228-234)."""
    logits = (S @ I.T) / T
    targets = torch.softmax(((I @ I.T + S @ S.T) / 2) / T, dim=-1)
    spots_loss = (-targets * torch.log_softmax(logits, dim=-1)).sum(1)
    images_loss = (-targets.T * torch.log_softmax(logits.T, dim=-1)).sum(1)
    return ((images_loss + spots_loss) / 2.0).mean()


def cpu_loss_time(B_sample, B_quote, budget_s, threads=None):
    """oracle.contrastive_loss_ref (literal restatement, fp32 autograd, torch CPU) fwd+bwd at B_sample,
    all host threads; the figure for B_quote is extrapolated with the B^2 cost model."""
    from oracle import oracle
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(99)
    S, I = _ln_rows(B_sample, 256, g, "cpu"), _ln_rows(B_sample, 256, g, "cpu")
    oracle.contrastive_loss_ref(S, I, 1.0, "soft")
    n, t_total = 0, 0.0
    while n < 3 or (t_total < budget_s and n < 50):
        t0 = time.perf_counter()
        oracle.contrastive_loss_ref(S, I, 1.0, "soft")
        t_total += time.perf_counter() - t0
        n += 1
    per = t_total / n
    scale = (B_quote / B_sample) ** 2
    return dict(value=1.0 / (per * scale), unit="steps/s", cores=threads, kind="port",
                sample=f"{n} fwd+bwd steps at B={B_sample} ({per * 1e3:.1f} ms each, {t_total:.1f} s of CPU time); "
                       f"B={B_quote} figure EXTRAPOLATED x{scale:.0f} (cost ~ B^2; B={B_quote} needs five "
                       f"{B_quote * B_quote * 4 / 2**30:.1f} GiB float32 matrices on the host)",
                measured_steps_per_s_at_sample=1.0 / per, torch=torch.__version__)


def main_loss(args, rank, world, local):
    B0 = args.loss_batch
    config = {"workload": f"cfg5: soft-target contrastive loss fwd+bwd, batch sweep 256..32768, D=256, T=1; "
                          f"value quoted at B={B0}" + (f" (global batch, rows sharded over {world} ranks, "
                                                       "embedding all-gather)" if world > 1 else ""),
              "l2": "L2 flushed (256 MB write) between timed iterations"}
    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_loss_time(min(4096, B0), B0, args.cpu_budget)
        print(json.dumps({"impl": "reference", "metric": LOSS_METRIC, "value": cb["value"], "unit": "steps/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "steps/s",
                                                      "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    from mclstexp_b200 import _lib, loss as mloss
    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        from mclstexp_b200.distributed import contrastive_loss_sharded
    peaks = load_peaks()
    g = torch.Generator(device=dev)
    g.manual_seed(99)
    sweep, value_ms, launches, prof, clocks = {}, None, None, [], None
    sizes = [b for b in synth.CONFIGS["cfg5"]["B_sweep"] if b <= B0]
    if B0 not in sizes:
        sizes.append(B0)
    for B in sizes:
        if B % (128 * world) != 0:
            continue
        S, I = _ln_rows(B, 256, g, dev), _ln_rows(B, 256, g, dev)
        if world > 1:
            rows = B // world
            Sl = S[rank * rows:(rank + 1) * rows].clone().requires_grad_(True)
            Il = I[rank * rows:(rank + 1) * rows].clone().requires_grad_(True)

            def step():
                Sl.grad = Il.grad = None
                contrastive_loss_sharded(Sl, Il, 1.0, "soft").backward()
        else:
            Sg, Ig = S.clone().requires_grad_(True), I.clone().requires_grad_(True)
            last = {}

            def step():
                Sg.grad = Ig.grad = None
                last["loss"] = mloss.contrastive_loss(Sg, Ig, 1.0, "soft")
                last["loss"].backward()
        quoted = B == B0
        if quoted:
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize()
            _lib.profile_enable(True)
            l0 = _lib.launch_count()
            with ClockSampler(local) as clk:
                ms = _time_steps(step, args.steps, 0, dev)
            launches = (_lib.launch_count() - l0) // args.steps
            prof = _lib.profile_collect()
            _lib.profile_enable(False)
            clocks = clk.summary()
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, {"loss": last["loss"], "dS": Sg.grad, "dI": Ig.grad})
        else:
            ms = _time_steps(step, max(3, min(args.steps, 10)), args.warmup, dev)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        flops = 14.0 * B * B * 256
        sweep[str(B)] = {"ms": ms, "steps_per_s": 1e3 / ms,
                         "frac_of_bf16_sustained": flops / (ms * 1e-3) / (peaks["tf_sust"] * 1e12 * world)}
        if world == 1 and not args.no_extra:
            # the reference's own formulation, stock PyTorch fp32 (TF32 off) on this GPU
            try:
                St, It = S.clone().requires_grad_(True), I.clone().requires_grad_(True)

                def tstep():
                    St.grad = It.grad = None
                    torch_soft_loss(St, It, 1.0).backward()
                tms = _time_steps(tstep, 3, 2, dev)
                sweep[str(B)]["torch_gpu_ms"] = tms
                del St, It
            except Exception as e:                       # report, do not hide (e.g. out of memory)
                sweep[str(B)]["torch_gpu_error"] = f"{type(e).__name__}: {e}"[:160]
            torch.cuda.empty_cache()
        if quoted:
            value_ms = ms
            # parity at the quoted size, outside the timed region: loss and gradients of the step's
            # own result against a float64 closed form evaluated on the GPU in row chunks
            parity = None
            if not args.no_parity and world == 1:
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                from checkers import loss_closed_form_f64
                Sg.grad = Ig.grad = None
                l = mloss.contrastive_loss(Sg, Ig, 1.0, "soft")
                l.backward()
                l64, dS64, dI64 = loss_closed_form_f64(S, I, 1.0, "soft")
                eS = float((Sg.grad.double() - dS64).norm() / dS64.norm())
                eI = float((Ig.grad.double() - dI64).norm() / dI64.norm())
                mS = float((Sg.grad.double() - dS64).abs().max() / dS64.abs().max())
                el = abs(l.item() - l64) / abs(l64)
                parity = {"B": B, "loss_rel": el, "dS_norm_rel": eS, "dI_norm_rel": eI, "dS_max_rel": mS,
                          "ok": bool(el < 1e-3 and eS < 1e-3 and eI < 1e-3 and mS < 1e-3),
                          "checker": "tests/checkers.loss_closed_form_f64 (float64, row-chunked, on the GPU)"}
                del dS64, dI64
            # end to end: pinned host embeddings in, loss + both gradients back on the host
            e2e = None
            if not args.no_e2e and world == 1:
                hS, hI = S.cpu().pin_memory(), I.cpu().pin_memory()
                gS, gI = torch.empty_like(hS).pin_memory(), torch.empty_like(hI).pin_memory()

                def e2e_step():
                    a = hS.to(dev, non_blocking=True).requires_grad_(True)
                    b = hI.to(dev, non_blocking=True).requires_grad_(True)
                    l = mloss.contrastive_loss(a, b, 1.0, "soft")
                    l.backward()
                    gS.copy_(a.grad, non_blocking=True)
                    gI.copy_(b.grad, non_blocking=True)
                    return l.item()
                e2e_step()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                n_e2e = max(1, min(args.steps, 5))
                for _ in range(n_e2e):
                    e2e_step()
                torch.cuda.synchronize()
                dt = (time.perf_counter() - t0) / n_e2e
                e2e = {"value": 1.0 / dt, "unit": "steps/s", "ms_per_step": dt * 1e3,
                       "h2d_bytes_per_step": int(2 * B * 256 * 4), "d2h_bytes_per_step": int(2 * B * 256 * 4 + 4),
                       "api": "mclstexp_b200.loss.contrastive_loss(host embeddings -> device).backward(); "
                              "loss.item() and both gradients copied to pinned host memory"}
        del S, I
        torch.cuda.empty_cache()
    per = {}
    for name, t in prof:
        per.setdefault(name, []).append(t)
    share = {n: float(np.sum(v)) / args.steps for n, v in per.items()}
    roofline = None
    if share:
        top = max(share, key=share.get)
        rows = B0 // world
        flops = 14.0 * B0 * rows * 256                       # algorithmic FLOPs of this rank's rows
        tensor_ms = sum(v for n, v in share.items() if n.startswith("gemm") or n.startswith("fused"))
        if tensor_ms > 0:
            ach = flops / (tensor_ms * 1e-3) / 1e12
            roofline = {"kernel": "tensor-core products of the step (" + ", ".join(
                            f"{n} x{len(per[n]) // args.steps}" for n in per if n.startswith(("gemm", "fused"))) + ")",
                        "bound": "tensor", "achieved": ach, "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                        "frac": ach / peaks["tf_sust"], "traffic": None, "peak_source": peaks["source"],
                        "kernel_ms": tensor_ms, "share_of_step": tensor_ms / value_ms,
                        "top_kernel": top, "kernels_ms_per_step": share,
                        "algorithmic_flops": "14 * B * rows * 256 (soft fwd 6 + bwd 8; split-precision passes "
                                             "and recomputation are not credited)"}
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_loss_time(min(4096, B0), B0, args.cpu_budget)
    if rank == 0:
        t_roof = 14.0 * B0 * B0 * 256 / (peaks["tf_sust"] * 1e12) / world
        line = {"metric": LOSS_METRIC, "value": 1e3 / value_ms, "unit": "steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": value_ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16x3",
                "dtype_note": "fp32 operands split into fp16 hi/lo, three tensor-core passes per product, "
                              "fp32 accumulate (~fp32 accuracy); statistics and gradients in fp32",
                "data": "synthetic", "config": config, "clocks": clocks, "gpu_launches": int(launches or 0),
                "e2e": e2e if world == 1 else None, "roofline": roofline,
                "step_roofline": {"t_roof_ms": t_roof * 1e3, "frac": t_roof * 1e3 / value_ms},
                "cpu_baseline": cpu_baseline, "parity_check": parity if world == 1 else None,
                "torch_gpu": ({"ms_per_step": sweep[str(B0)].get("torch_gpu_ms"),
                               "what": "baselines/Bleep/models.py:34-43 in stock PyTorch fp32 (TF32 off), same GPU, "
                                       "fwd+bwd", "error": sweep[str(B0)].get("torch_gpu_error")}
                              if world == 1 else None),
                "sweep": sweep}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if world == 1 and parity is not None and not parity["ok"]:
        sys.exit(3)


class _TorchRefStep:
    """The reference's modules restated with stock PyTorch ops (model.py:10-69 PreNorm / FeedForward /
    Attention / attn_block, :151-168 ProjectionHead, :230-240 forward; loss as baselines/Bleep/models.py:34-43),
    driven by the same state_dict: the `torch_gpu` baseline of the cfg2 step."""

    def __init__(self, sd, heads, layers, T):
        self.p = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
        self.heads, self.layers, self.T = heads, layers, T

    def _head(self, x, pre):
        F, p = torch.nn.functional, self.p
        proj = F.linear(x, p[pre + "projection.weight"], p[pre + "projection.bias"])
        y = F.linear(F.gelu(proj), p[pre + "fc.weight"], p[pre + "fc.bias"]) + proj
        return F.layer_norm(y, (y.shape[-1],), p[pre + "layer_norm.weight"], p[pre + "layer_norm.bias"])

    def __call__(self, batch):
        F, p, h = torch.nn.functional, self.p, self.heads
        pos = batch["position"].long()
        x = (batch["expression"] + F.embedding(pos[:, 0], p["x_embed.weight"]) +
             F.embedding(pos[:, 1], p["y_embed.weight"])).unsqueeze(0)
        for l in range(self.layers):
            pre = f"spot_encoder.{l}."
            y = F.layer_norm(x, (x.shape[-1],), p[pre + "attn.norm.weight"], p[pre + "attn.norm.bias"])
            q, k, v = F.linear(y, p[pre + "attn.fn.to_qkv.weight"]).chunk(3, dim=-1)
            b, n, _ = q.shape
            q, k, v = (t.view(b, n, h, -1).transpose(1, 2) for t in (q, k, v))
            att = torch.softmax(q @ k.transpose(-1, -2) * q.shape[-1] ** -0.5, dim=-1)
            o = (att @ v).transpose(1, 2).reshape(b, n, -1)
            x = F.linear(o, p[pre + "attn.fn.to_out.0.weight"], p[pre + "attn.fn.to_out.0.bias"]) + x
            y = F.layer_norm(x, (x.shape[-1],), p[pre + "ff.norm.weight"], p[pre + "ff.norm.bias"])
            y = F.linear(F.gelu(F.linear(y, p[pre + "ff.fn.net.0.weight"], p[pre + "ff.fn.net.0.bias"])),
                         p[pre + "ff.fn.net.3.weight"], p[pre + "ff.fn.net.3.bias"])
            x = y + x
        spot = self._head(x, "spot_projection.").squeeze(0)
        img = self._head(batch["image"], "image_projection.")
        return torch_soft_loss(spot, img, self.T)

    def zero_grad(self):
        for v in self.p.values():
            v.grad = None


def cpu_train_time(G, B, budget_s, threads=None):
    """oracle.path_loss_ref (the reference's modules restated, torch CPU fp32) fwd+bwd, all host threads."""
    from oracle import oracle
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = oracle.make_state_dict(G, 1024, 256, 8, 64, 2, 0)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    feats = torch.tensor(synth.image_features(B, 1024, 1))
    expr = torch.tensor(synth.expression(B, G, 2))
    pos = torch.tensor(synth.positions(B, 3, "st"))

    def one():
        for v in params.values():
            v.grad = None
        oracle.path_loss_ref(params, feats, expr, pos, 1.0, 8, 2, "soft").backward()
    one()
    n, t_total = 0, 0.0
    while n < 3 or (t_total < budget_s and n < 100):
        t0 = time.perf_counter()
        one()
        t_total += time.perf_counter() - t0
        n += 1
    return dict(value=n / t_total, unit="steps/s", cores=threads, kind="port",
                sample=f"{n} full fwd+bwd steps at B={B}, G={G} (dense [65536,G] table gradients as autograd "
                       f"builds them), {t_total:.1f} s of CPU time; the whole workload, not a sub-sample",
                torch=torch.__version__)


def main_train(args, rank, world, local):
    B, G = 1024, args.train_genes
    config = {"workload": f"cfg2: cSCC-shaped training step, B={B} spots, G={G} genes, 2 attention blocks "
                          "(8 heads x 64) + projection heads + soft-target loss, forward + backward "
                          "(no CNN, no optimiser)" + (f"; {world} data-parallel replicas" if world > 1 else ""),
              "l2": "L2 flushed (256 MB write) between timed iterations"}
    if args.impl == "reference":
        if rank != 0:
            return
        cb = cpu_train_time(G, B, args.cpu_budget)
        print(json.dumps({"impl": "reference", "metric": TRAIN_METRIC, "value": cb["value"], "unit": "steps/s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "steps/s",
                                                      "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    from torch import nn
    from mclstexp_b200 import _lib, model as mm
    from mclstexp_b200.graphs import GraphedTrainStep
    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    torch.manual_seed(0)
    net = mm.mclSTExp_Attention("none", 1.0, 1024, G, 256, 8, 64, 2, targets="soft")
    net.image_encoder = nn.Identity()
    net = net.to(dev)
    g = torch.Generator(device=dev)
    g.manual_seed(7 + rank)
    batch = {"image": torch.randn(B, 1024, generator=g, device=dev),
             "expression": torch.rand(B, G, generator=g, device=dev),
             "position": torch.randint(0, 64, (B, 2), generator=g, device=dev).float()}

    def eager():
        net.zero_grad(set_to_none=True)
        net(batch).backward()
    eager()
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    eager()
    launches = _lib.launch_count() - l0
    ms_eager = _time_steps(eager, args.steps, args.warmup, dev)
    _lib.profile_enable(True)
    for _ in range(3):
        eager()
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    per = {}
    for name, t in prof:
        per.setdefault(name, []).append(t)
    share = {n: float(np.sum(v)) / 3 for n, v in per.items()}
    # parity of this very step against the stock-PyTorch restatement (fp32) -- outside timed regions
    ref = _TorchRefStep(net.state_dict(), 8, 2, 1.0)
    ref.zero_grad()
    lref = ref(batch)
    lref.backward()
    net.zero_grad(set_to_none=True)
    lmine = net(batch)
    lmine.backward()
    worst, worst_name = 0.0, ""
    for k_, p_ in net.named_parameters():
        want = ref.p[k_].grad
        e = float((p_.grad - want).norm() / (want.norm() + 1e-30))
        if e > worst:
            worst, worst_name = e, k_
    parity = {"loss_rel": abs(lmine.item() - lref.item()) / abs(lref.item()), "worst_grad_norm_rel": worst,
              "worst_grad": worst_name, "ok": bool(abs(lmine.item() - lref.item()) <= 1e-3 * abs(lref.item()) and worst < 2e-3),
              "checker": "stock PyTorch fp32 restatement of model.py:10-69,151-168,230-240 + Bleep/models.py:34-43 "
                         "on the same GPU (every parameter gradient, norm-wise)"}
    del lmine, lref

    def tstep():
        ref.zero_grad()
        ref(batch).backward()
    ms_torch = _time_steps(tstep, args.steps, args.warmup, dev)
    torch_graph_ms = None
    try:                                      # the stock path under a CUDA graph too (fair launch-free comparison)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                tstep()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        tg = torch.cuda.CUDAGraph()
        ref.zero_grad()
        with torch.cuda.graph(tg):
            ref(batch).backward()
        torch_graph_ms = _time_steps(tg.replay, args.steps, args.warmup, dev)
    except Exception as e:
        torch_graph_ms = f"{type(e).__name__}: {e}"[:160]
    del ref
    torch.cuda.empty_cache()
    gstep = GraphedTrainStep(net, batch)
    with ClockSampler(local) as clk:
        ms_graph = _time_steps(lambda: gstep(batch), args.steps, args.warmup, dev)
    if args.dump_outputs:                     # the replay leaves the loss and every .grad in place
        dump_outputs(args.dump_outputs, {"loss": gstep.loss, **{"grad." + n: p.grad for n, p in net.named_parameters()
                                                                if p.grad is not None}})
    ms = ms_graph
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # end to end: pinned host batch in, loss value back
    hb = {k_: v.cpu().pin_memory() for k_, v in batch.items()}

    def e2e_step():
        db = {k_: v.to(dev, non_blocking=True) for k_, v in hb.items()}
        return float(gstep(db))
    e2e_step()
    torch.cuda.synchronize()
    n_e2e = max(3, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_step()
    dt = (time.perf_counter() - t0) / n_e2e
    if world > 1:
        t = torch.tensor([dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    L, H, inner, E, P = 2, 8, 512, 1024, 256
    fwd = L * (2 * B * G * 3 * inner + 4 * B * B * inner + 2 * B * inner * G + 4 * B * G * G) + \
        2 * B * (G * P + P * P) + 2 * B * (E * P + P * P)
    flops = 3.0 * fwd + 14.0 * B * B * P
    tensor_ms = sum(v for n, v in share.items() if n.startswith(("gemm", "fused")))
    roofline = {"kernel": "tensor-core products of the step (gemm_tn, all launches)", "bound": "tensor",
                "achieved": flops / (tensor_ms * 1e-3) / 1e12 if tensor_ms else None, "peak": peaks["tf_sust"],
                "unit": "TFLOP/s", "frac": (flops / (tensor_ms * 1e-3) / 1e12 / peaks["tf_sust"]) if tensor_ms else None,
                "traffic": None, "peak_source": peaks["source"], "kernel_ms": tensor_ms,
                "share_of_step": tensor_ms / ms_eager if ms_eager else None,
                "kernels_ms_per_step": share,
                "note": "launch-latency regime (BASELINE.md section 3): per-kernel times are from the eager step"}
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_train_time(G, B, args.cpu_budget)
    if rank == 0:
        t_roof = flops / (peaks["tf_sust"] * 1e12)
        line = {"metric": TRAIN_METRIC, "value": world * 1e3 / ms, "unit": "steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f16x3",
                "dtype_note": "fp32 operands split into fp16 hi/lo, three tensor-core passes per product, fp32 accumulate",
                "data": "synthetic", "config": config, "clocks": clk.summary(), "gpu_launches": int(launches),
                "value_form": "graphs.GraphedTrainStep replay (one CUDA graph per step); eager in `eager_ms_per_step`",
                "eager_ms_per_step": ms_eager,
                "e2e": {"value": world / dt, "unit": "steps/s", "ms_per_step": dt * 1e3,
                        "h2d_bytes_per_step": int(sum(v.numel() * 4 for v in hb.values())), "d2h_bytes_per_step": 4,
                        "api": "GraphedTrainStep(host batch -> device) -> float(loss)"},
                "roofline": roofline, "step_roofline": {"t_roof_ms": t_roof * 1e3, "frac": t_roof * 1e3 / ms},
                "cpu_baseline": cpu_baseline, "parity_check": parity,
                "torch_gpu": {"eager_ms_per_step": ms_torch, "graph_ms_per_step": torch_graph_ms,
                              "what": "the reference's modules in stock PyTorch fp32 (TF32 off) on the same GPU, "
                                      "same state_dict and batch, fwd+bwd"}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if not parity["ok"]:
        sys.exit(3)


# --------------------------------------------------------------------------- parity at size
def retrieval_parity_check(out, qry_local, cfg, mode, dev, flavour, world, bank=None, expr=None,
                           rows_total=64, seed=20261017):
    """OUTSIDE the timed region: re-derives sampled query rows of this rank's own result with the
    oracle's float64 spec against the FULL bank on the host (oracle.find_matches_spec_rows +
    weighted_average_spec; reference evel_her2st.py:74-84, :175-187).  Indices and float32
    similarities must be bit-equal, the predicted expression within rtol 1e-3 (atol 1e-6)."""
    from oracle import oracle
    idx, val, _, ex = out[:4]
    owned = out[4] if len(out) > 4 else torch.arange(qry_local.shape[0], device=dev)   # rows whose expr_pred is here
    k = cfg["k"]
    if bank is None:                                   # sharded run: rebuild the full inputs
        bank, _, expr = make_inputs_device(cfg, 1234 + 4, dev, flavour)
    n_rows = max(16, -(-rows_total // world))
    rng = np.random.default_rng(seed + int(os.environ.get("RANK", 0)))
    pos = np.sort(rng.choice(owned.shape[0], size=min(n_rows, owned.shape[0]), replace=False))
    pos_t = torch.as_tensor(pos, device=dev)
    pick_t = owned[pos_t]
    pick = pick_t.cpu().numpy()
    q_rows = qry_local[pick_t].cpu().numpy()
    host_bank = bank.cpu().numpy()
    t0 = time.perf_counter()
    sv, si = oracle.find_matches_spec_rows(host_bank, q_rows, k)
    got_i = idx[pick_t].cpu().numpy()
    got_v = val[pick_t].cpu().numpy()
    indices_equal = bool(np.array_equal(got_i, si))
    values_equal = bool(np.array_equal(got_v.view(np.uint32), sv.view(np.uint32)))
    uniq, inv = np.unique(si, return_inverse=True)     # only the rows the winners touch leave the GPU
    ek = expr[torch.as_tensor(uniq, device=dev)].cpu().numpy()
    _, ex64 = oracle.weighted_average_spec(host_bank[uniq], ek, q_rows, inv.reshape(si.shape), mode, values=sv)
    got_e = ex[pos_t].double().cpu().numpy()
    err = np.abs(got_e - ex64)
    expr_ok = bool((err <= 1e-3 * np.abs(ex64) + 1e-6).all())
    rel = float((err / np.maximum(np.abs(ex64), 1e-3)).max())
    return {"rows": int(pick.size), "indices_equal": indices_equal, "values_equal": values_equal,
            "expr_max_rel": rel, "expr_ok": expr_ok, "checker_s": time.perf_counter() - t0,
            "ok": indices_equal and values_equal and expr_ok}


# --------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("MCLST_BENCH_WORKLOAD", "cfg4"))
    ap.add_argument("--mode", default="inv_sq_l2")
    ap.add_argument("--flavour", default="clustered")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-bank-shards", type=int, default=0,
                    help="bank shards of the end-to-end (host array) job at N > 1; default: all ranks")
    ap.add_argument("--exact-only", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the loss / train-step metrics")
    ap.add_argument("--bank-shards", type=int, default=int(os.environ.get("MCLST_BANK_SHARDS", 0)),
                    help="ranks per query group that split the bank (default: 2 when N >= 2); "
                         "N = pure bank sharding, 1 = pure query sharding")
    ap.add_argument("--full-loss-sweep", action="store_true", help="cfg5 sweep up to B=32768")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled-row parity check against the oracle")
    ap.add_argument("--no-numa", action="store_true", help="N > 1: do not pin the rank to the CPUs next to its GPU")
    ap.add_argument("--loss-batch", type=int, default=32768, help="cfg5: batch the headline value is quoted on")
    ap.add_argument("--train-genes", type=int, default=1000, help="cfg2: spot_dim (1000 HVGs; 171 = real cSCC)")
    ap.add_argument("--no-alt-grids", action="store_true", help="N > 1: skip timing the other decompositions")
    ap.add_argument("--queries", type=int, default=0, help="tuning: override the query count of the workload")
    ap.add_argument("--query-blocks", type=int, default=0, help="tuning: query blocks of the sharded pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step to DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB: a fixed row sample of larger outputs)")
    args = ap.parse_args()
    assert args.warmup >= 3 or args.impl == "reference", "timing rules: W >= 3"
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the GPU path run by a single process")
    if args.workload == "cfg5":
        return main_loss(args, rank, world, local)
    if args.workload == "cfg2":
        return main_train(args, rank, world, local)
    cfg = dict(synth.CONFIGS[args.workload])
    if args.queries:
        cfg["Q"] = args.queries
    config = {"workload": f"{args.workload}: N={cfg['N']} bank spots x Q={cfg['Q']} queries, D={cfg['D']}, "
                          f"top_k={cfg['k']}, G={cfg['G']} genes, weights={args.mode}, {args.flavour} embeddings",
              "l2": "inputs larger than L2 (126 MB)",
              "note": "emb_pred (matched_spot_embeddings_pred, computed but never used by the reference, "
                      "evel_her2st.py:186) is not produced in the timed step (want_emb=False, SURVEY 8d)"}

    if args.impl == "reference":
        if rank != 0:
            return
        vals = []
        for _ in range(max(1, args.steps)):
            cb, t, done = cpu_reference_time(cfg, args.mode, budget_s=args.cpu_budget)
            vals.append(cb["value"])
        v = float(np.mean(vals))
        cb["value"] = v
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT,
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * cfg["Q"] / v, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": cb,
                          "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0,
                                  "d2h_bytes_per_step": 0}}))
        return

    from mclstexp_b200 import _lib, retrieval
    assert torch.cuda.is_available(), "bench.py needs a B200 (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        from mclstexp_b200 import distributed as mdist
        # host buffers of this rank on its GPU's NUMA node (the end-to-end job is upload-bound)
        config["numa_bound"] = bool(not args.no_numa and mdist.bind_to_gpu_cpus(local))
    peaks = load_peaks()
    N, Q, D, G, k = cfg["N"], cfg["Q"], cfg["D"], cfg["G"], cfg["k"]

    bank, qry, expr = make_inputs_device(cfg, 1234 + 4, dev, args.flavour)
    Q_job = Q
    if world > 1:
        bshards = args.bank_shards if args.bank_shards > 0 else min(2, world)
        grid = mdist.make_retrieval_grid(bshards, world, rank)
        config["parallelism"] = (f"{grid.query_groups} query groups x {grid.bank_shards} bank shards "
                                 "(candidate all-gather + merge inside a group)")
        shard = mdist.BankShard.from_full(bank, expr, grid.b_index, grid.bank_shards)
        e2e_host = None
        if not args.no_e2e:
            # the one-shot host-array job is upload-bound, so its decomposition shards the bank
            # over ALL ranks (every byte crosses PCIe once) and replicates the queries
            eshards = args.e2e_bank_shards if args.e2e_bank_shards > 0 else world
            egrid = grid if eshards == grid.bank_shards else mdist.make_retrieval_grid(eshards, world, rank)
            lo, hi = mdist.shard_bounds(N, egrid.bank_shards)[egrid.b_index]
            eq0, eq1 = egrid.query_slice(Q)
            e2e_host = (egrid, bank[lo:hi].cpu().pin_memory(), expr[lo:hi].cpu().pin_memory(),
                        qry[eq0:eq1].cpu().pin_memory(), lo)
        q0, q1 = grid.query_slice(Q)
        qry = qry[q0:q1].contiguous()
        del bank, expr
        torch.cuda.empty_cache()

        def step():
            # every rank ends with its share of the finished rows (reduce-scatter, SURVEY 8e)
            return mdist.retrieve_sharded(shard, qry, k, args.mode, group=grid.group, scatter_output=True,
                                          query_blocks=args.query_blocks or None)
    else:
        def step():
            return retrieval.retrieve_device(bank, expr, qry, k, args.mode, want_emb=False,
                                             out_dtype=torch.float32, exact_only=args.exact_only)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        out = step()
    barrier()
    _lib.profile_enable(True)
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        ev0.record()
        for _ in range(args.steps):
            out = step()
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = (_lib.launch_count() - l0) // args.steps
    prof = _lib.profile_collect()
    _lib.profile_enable(False)
    counters = retrieval.last_counters()
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = Q / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"indices": out[0], "values": out[1], "expr_pred": out[3]})

    # ---- roofline of the dominant kernel (live CUDA-event times from the timed region)
    per = {}
    for name, t in prof:
        per.setdefault(name, []).append(t)
    kern = {n: float(np.mean(v)) for n, v in per.items()}
    share = {n: float(np.sum(v)) / args.steps for n, v in per.items()}
    top = max(share, key=share.get) if share else None
    n_local = N // (grid.bank_shards if world > 1 else 1)
    Q = qry.shape[0]                     # per-rank query count for the per-kernel figures
    alg = {   # algorithmic work per launch (DESIGN.md): FLOPs for the similarity kernels, bytes otherwise
        "sim_topk": ("tensor", 2.0 * Q * n_local * D),
        "exact_topk": ("tensor", 2.0 * Q * n_local * D),
        "weighted_average": ("hbm", Q * k * G * 4.0 + Q * G * 4.0),   # distances come from the re-rank
        "weighted_gather": ("hbm", Q * k * G * 4.0 / (grid.bank_shards if world > 1 else 1) + Q * G * 4.0),
        "row_norms": ("hbm", (n_local + Q) * D * 4.0),
        "pack_rows": ("hbm", (n_local + Q) * D * 6.0),
    }
    roofline = None
    if top in alg:
        bound, work = alg[top]
        # per STEP: a sharded step launches the kernel once per query block, and the staged form
        # times the seed pass separately (it is part of the same algorithmic work)
        t_ms = share[top] + (share.get("sim_seed", 0.0) if top == "sim_topk" else 0.0)
        t = t_ms * 1e-3
        if bound == "tensor":
            ach, peak, unit = work / t / 1e12, peaks["tf_sust"], "TFLOP/s"
        else:
            ach, peak, unit = work / t / 1e9, peaks["hbm"], "GB/s"
        traffic = None          # DRAM bytes per launch from the committed ncu capture of this workload
        tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if not os.path.exists(tp):
            tp = os.path.join(ROOT, "profiles", "r1_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            if tj.get("workload") == args.workload and tj.get("n_gpus") == world:
                traffic = tj["bytes_per_launch"].get(top)
        roofline = {"kernel": top, "bound": bound, "achieved": ach, "peak": peak, "unit": unit,
                    "frac": ach / peak, "traffic": traffic, "peak_source": peaks["source"],
                    # the sustained figure is cuBLAS bf16 8192^3 back to back for 4 s; a kernel timed
                    # inside a step may exceed it, so the burst figure is given as well
                    **({"peak_kind": "bf16 sustained", "frac_of_burst_peak": ach / peaks["tf_burst"],
                        "burst_peak": peaks["tf_burst"]} if bound == "tensor" else {}),
                    "kernel_ms": t_ms, "launches_per_step": len(per[top]) // args.steps,
                    "share_of_step": t_ms / ms,
                    "kernels_ms_per_step": share}
    # whole-job roofline over all GPUs: max(FLOPs / tensor peak, bytes / HBM peak) (BASELINE.md section 3)
    Q = Q_job
    step_flops = 2.0 * Q * N * D
    step_bytes = Q * k * G * 4.0 + Q * G * 4.0 + (N + Q) * D * 4.0 + Q * k * D * 4.0
    t_roof = max(step_flops / (peaks["tf_sust"] * 1e12), step_bytes / (peaks["hbm"] * 1e9)) / world
    step_roof = {"t_roof_ms": t_roof * 1e3, "frac": t_roof * 1e3 / ms}

    # ---- parity at the size of record (outside every timed region, every rank, every N)
    parity = None
    if not args.no_parity:
        parity = retrieval_parity_check(out, qry, cfg, args.mode, dev, args.flavour, world,
                                        bank if world == 1 else None, expr if world == 1 else None)
        if world > 1:
            flags = torch.tensor([float(parity[f]) for f in ("indices_equal", "values_equal", "expr_ok", "ok")],
                                 device=dev)
            dist.all_reduce(flags, op=dist.ReduceOp.MIN)
            agg = torch.tensor([parity["expr_max_rel"], parity["checker_s"]], device=dev)
            dist.all_reduce(agg, op=dist.ReduceOp.MAX)
            rows = torch.tensor([float(parity["rows"])], device=dev)
            dist.all_reduce(rows)
            parity = {"rows": int(rows.item()), "indices_equal": bool(flags[0]), "values_equal": bool(flags[1]),
                      "expr_max_rel": float(agg[0]), "expr_ok": bool(flags[2]), "checker_s": float(agg[1]),
                      "ok": bool(flags[3]), "ranks_checked": world}
        parity["checker"] = ("oracle.find_matches_spec_rows + weighted_average_spec (float64, host) on rows "
                             "sampled from each rank's own query slice, against the full bank")
        torch.cuda.empty_cache()

    # ---- the other decompositions of the same job (N > 1), on record next to the default one:
    # pure bank sharding (1 x N: the north star's literal topology, every collective on the critical
    # path) and pure query sharding (N x 1: bank replicated, no exchange at all)
    other_grids = None
    if world > 1 and not args.no_alt_grids:
        other_grids = {}
        for bs in sorted({1, world} - {grid.bank_shards}):
            g2 = mdist.make_retrieval_grid(bs, world, rank)
            b2, q2, e2 = make_inputs_device(cfg, 1234 + 4, dev, args.flavour)
            sh2 = mdist.BankShard.from_full(b2, e2, g2.b_index, g2.bank_shards)
            qa, qb = g2.query_slice(cfg["Q"])
            qq = q2[qa:qb].contiguous()
            del b2, e2, q2
            torch.cuda.empty_cache()
            for _ in range(3):
                mdist.retrieve_sharded(sh2, qq, k, args.mode, group=g2.group, scatter_output=True)
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(3):
                mdist.retrieve_sharded(sh2, qq, k, args.mode, group=g2.group, scatter_output=True)
            a1.record()
            barrier()
            t2 = torch.tensor([a0.elapsed_time(a1) / 3], device=dev)
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            other_grids[f"{g2.query_groups} query groups x {g2.bank_shards} bank shards"] = {
                "ms_per_step": float(t2.item()), "value": cfg["Q"] / (float(t2.item()) * 1e-3), "unit": UNIT}
            del sh2, qq
            torch.cuda.empty_cache()

    # ---- end to end through the public host-array API: host (pinned) buffers in, host arrays
    # out, every H2D / D2H copy inside the timed region
    e2e = None
    if not args.no_e2e:
        if world == 1:
            hb, he = bank.cpu().pin_memory(), expr.cpu().pin_memory()
            del bank, expr
            hq = qry.cpu().pin_memory()
        else:
            egrid, hb, he, hq, off = e2e_host
            ntot = N
            del shard
        torch.cuda.empty_cache()

        def e2e_step():
            if world == 1:
                idx, emb, ex = retrieval.retrieve(hb, he, hq, top_k=k, mode=args.mode, want_emb=False,
                                                  out_dtype=torch.float32)
                return idx, ex
            sh = mdist.BankShard.from_host(hb, he, off, ntot, dev)
            idx, val, _, ex, rows = mdist.retrieve_sharded(sh, hq.to(dev, non_blocking=True), k, args.mode,
                                                           group=egrid.group, scatter_output=True)
            return retrieval.to_host(idx[rows], ex)      # every rank reads back its own finished rows

        r = e2e_step()
        r = e2e_step()                       # twice: both alternating pinned result buffers exist
        n_e2e = max(1, min(args.steps, 3))
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            r = e2e_step()
        barrier()
        dt = (time.perf_counter() - t0) / n_e2e
        if world > 1:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        resident = None
        if world == 1:
            # serving form: the bank stays on the device, only the queries travel per call
            bank_obj = retrieval.Bank(hb, he)
            r = bank_obj.retrieve(hq, top_k=k, mode=args.mode, want_emb=False, out_dtype=torch.float32)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                r = bank_obj.retrieve(hq, top_k=k, mode=args.mode, want_emb=False, out_dtype=torch.float32)
            dtr = (time.perf_counter() - t0) / n_e2e
            resident = {"value": Q / dtr, "unit": UNIT, "ms_per_step": dtr * 1e3,
                        "h2d_bytes_per_step": int(Q * D * 4), "d2h_bytes_per_step": int(Q * k * 8 + Q * G * 4),
                        "api": "mclstexp_b200.retrieval.Bank(...).retrieve(host queries) -> host arrays"}
            del bank_obj
        e2e = {"value": Q / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "resident_bank": resident,
               "h2d_bytes_per_step": int((N * (D + G) * (egrid.query_groups if world > 1 else 1) + Q * D *
                                          (egrid.bank_shards if world > 1 else 1)) * 4),
               "d2h_bytes_per_step": int(Q * k * 8 + Q * G * 4),
               "api": "mclstexp_b200.retrieval.retrieve(host arrays) -> host arrays" if world == 1 else
                      f"mclstexp_b200.distributed.BankShard.from_host + retrieve_sharded from pinned host "
                      f"shards, {egrid.query_groups} query groups x {egrid.bank_shards} bank shards; every rank "
                      "reads its own share of the finished rows back (reduce-scatter)"}
        del hb, he, hq

    extra = None
    if not args.no_extra:
        if args.no_e2e:                      # (the e2e block already released them otherwise)
            if world == 1:
                del bank, expr
            else:
                del shard
        torch.cuda.empty_cache()
        extra = {"contrastive_loss_soft_fwd_bwd": loss_sweep(dev, peaks, world, rank, not args.full_loss_sweep)}
        if world == 1:
            extra["train_step_cfg2_B1024"] = train_step_cfg2(dev)
            extra["bank_build_group32"] = bank_build(dev)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _, _ = cpu_reference_time(cfg, args.mode, budget_s=args.cpu_budget)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f16",
                "dtype_note": "fp16 tensor-core candidate scores; exact fp64-accumulated cosine re-rank "
                              "(bit-exact top-k); fp32 weighted average",
                "data": "synthetic", "config": config,
                "clocks": clk.summary(), "gpu_launches": int(launches), "e2e": e2e,
                "roofline": roofline, "step_roofline": step_roof, "cpu_baseline": cpu_baseline,
                "parity_check": parity, "path_counters": counters, "other_grids": other_grids, "extra": extra}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.exit(3)


if __name__ == "__main__":
    main()
