"""CPU checks of the C-ABI boundary: the library builds for sm_100a, loads, and exports
every symbol include/mclst_b200.h declares.  No compute calls (no GPU here)."""
import numpy as np
import ctypes
import json
import os
import subprocess
import sys

import pytest

from mclstexp_b200 import _lib, build


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_every_header_symbol_is_exported(lib):
    names = _lib.header_symbols()
    assert "mclst_find_matches" in names and "mclst_weighted_average" in names
    for n in names:
        assert hasattr(lib, n), n
    assert lib.mclst_version() >= 100


def test_library_is_sm100a_only():
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = {l.split(".")[-2] for l in out.splitlines() if l.strip().endswith(".cubin")}
    assert archs == {"sm_100a"}, out


def test_argument_validation_needs_no_gpu(lib):
    n = ctypes.c_size_t()
    assert lib.mclst_find_matches_workspace_bytes(1000, 10, 256, 50, 0, ctypes.byref(n)) == 0
    assert n.value > 0
    assert lib.mclst_find_matches_workspace_bytes(1000, 10, 0, 50, 0, ctypes.byref(n)) == -1
    assert b"bad shape" in lib.mclst_last_error()
    # null pointers are rejected before anything touches the device
    rc = lib.mclst_find_matches(None, 10, 256, None, 1, 256, 256, 5, 0, None, None, None, 0, 0, None)
    assert rc == -1


def test_product_has_no_cpu_fallback():
    import numpy as np
    import torch
    from mclstexp_b200 import retrieval
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.MclstError):
        retrieval.find_matches(np.zeros((4, 8), np.float32), np.zeros((2, 8), np.float32), 1)


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, "mclstexp_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def _lane_plan(lib, qt, tiles, lanes, max_slots):
    import ctypes as C
    cap = qt * max_slots + 4 * lanes + 16
    units = np.zeros((cap, 5), dtype=np.int32)
    n, slots = C.c_int64(), C.c_int()
    rc = lib.mclst_debug_lane_plan(C.c_int64(qt), C.c_int64(tiles), lanes, max_slots,
                                   units.ctypes.data_as(C.c_void_p), C.c_int64(cap), C.byref(n), C.byref(slots))
    assert rc == 0 and n.value <= cap
    return units[:n.value], slots.value


def test_lane_plan_covers_every_tile_once():
    """Host-only property of the persistent top-k kernel's work decomposition: every
    (query block, bank tile) belongs to exactly one unit, no two units share a candidate
    stream (query block, slot), slots stay below the advertised count, and the headline shapes
    are balanced to within 0.1 % of the ideal tiles-per-SM."""
    import random
    lib = _lib.load()
    rng = random.Random(7)
    cases = [(512, 7813, 148, 4), (256, 3907, 148, 4), (128, 3907, 148, 4), (64, 7813, 148, 4),
             (1, 1, 148, 4), (147, 10, 148, 4), (149, 100, 148, 4), (75, 1000, 148, 4), (5, 36, 148, 2)]
    cases += [(rng.randint(1, 500), rng.randint(1, 300), rng.choice([148, 132, 8, 3, 1]),
               rng.choice([1, 2, 4, 8])) for _ in range(120)]
    for qt, tiles, lanes, max_slots in cases:
        units, slots = _lane_plan(lib, qt, tiles, lanes, max_slots)
        assert 1 <= slots <= max_slots
        cover = np.zeros((qt, tiles), dtype=np.int32)
        load = np.zeros(lanes, dtype=np.int64)
        streams = set()
        for c, qb, t0, t1, slot in units:
            assert 0 <= c < lanes and 0 <= qb < qt and 0 <= t0 < t1 <= tiles and 0 <= slot < slots
            assert (qb, slot) not in streams
            streams.add((qb, slot))
            cover[qb, t0:t1] += 1
            load[c] += t1 - t0
        assert (cover == 1).all(), (qt, tiles, lanes, max_slots)
        if tiles > 1000 and lanes == 148:
            assert load.max() <= 1.001 * qt * tiles / lanes + 1


def test_speculative_seed_rank_is_the_binomial_tail():
    """csrc/sim_topk.cu spec_rank: the speculative start threshold is the j-th largest sample value,
    j = the smallest rank with P(Binomial(k - 1, f) >= j) < 1e-7 (never above k, never below 4)."""
    from scipy.stats import binom
    lib = _lib.load()
    for k in (8, 50, 200, 600):
        for f in (0.001, 128 / 3907, 1 / 24, 0.125, 0.3):
            j = lib.mclst_debug_spec_rank(k, f)
            assert 4 <= j <= k
            tail = lambda jj: float(binom.sf(jj - 1, k - 1, f))          # P(X >= jj)
            if j < k:
                assert tail(j) < 1e-7
            if j > 4:
                assert tail(j - 1) >= 1e-7 or j == k
    assert lib.mclst_debug_spec_rank(50, 0.6) == 50                      # sampling most of the bank: no speculation
    assert lib.mclst_debug_spec_rank(5, 0.03) == 5                       # tiny k: none either


def _sm_count(lib):
    """The SM count mclst_debug_gemm_variant decides on: the device's, 148 (B200) without one."""
    n = ctypes.c_int(0)
    lib.mclst_device_info(ctypes.byref(n), None, None)
    return n.value or 148


def test_gemm_variant_follows_the_tile_rule(lib):
    """csrc/gemm.cu gemm_variant, the tile kernel of mclst_matmul's packed route: CTA pairs (128 x 256
    tiles, B shared) once there are two row tiles and at least two 128 x 256 tiles per SM; one CTA at
    256-wide tiles while there is at least one per SM; below that 128-wide tiles, and 64-wide ones
    while two 128-wide tiles still fit per SM."""
    from checkers import gemm_variant
    if os.environ.get("MCLST_GEMM_CLUSTER"):
        pytest.skip("MCLST_GEMM_CLUSTER overrides the rule")
    sms = _sm_count(lib)
    cdiv = lambda a, b: -(-a // b)
    seen = set()
    for M in (1, 64, 128, 129, 256, 300, 1000, 2100, 5000):
        for N in (1, 100, 128, 129, 256, 257, 700, 1000, 4096, 10000):
            for batch in (1, 2, 3, 5, 8, 17, 33, 100, 1000):
                cl, width = gemm_variant(M, N, batch)
                seen.add((cl, width))
                tiles256 = cdiv(M, 128) * cdiv(N, 256) * batch
                tiles128 = cdiv(M, 128) * cdiv(N, 128) * batch
                case = (M, N, batch, sms, cl, width)
                assert (cl == 2) == (M > 128 and tiles256 >= 2 * sms), case
                assert cl == 1 or width == 256, case
                assert (width < 256) == (cl == 1 and tiles256 < sms), case
                assert width != 64 or 2 * tiles128 <= sms, case
                assert width != 128 or 2 * tiles128 > sms, case
    assert seen == {(2, 256), (1, 256), (1, 128), (1, 64)}, seen
    # a lone tile, and a product that fills every SM twice over in one row tile: SM-independent cases
    assert gemm_variant(1, 1, 1) == (1, 64)
    assert gemm_variant(128, 256 * 4 * sms, 1) == (1, 256)
    assert gemm_variant(256, 256 * sms, 1) == (2, 256)
    assert lib.mclst_debug_gemm_variant(0, 1, 1, ctypes.byref(ctypes.c_int()), ctypes.byref(ctypes.c_int())) == -1


@pytest.mark.parametrize("force,want", [("2", (2, 256)), ("1", (1, 256))])
def test_gemm_variant_honours_cluster_override(lib, force, want):
    """MCLST_GEMM_CLUSTER=2 pairs every product, even a single row tile (its partner is a ghost);
    any other value keeps the single-CTA kernels.  Read once per process, so checked in a fresh one."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import json, sys; sys.path.insert(0, 'tests'); from checkers import gemm_variant; "
            "print(json.dumps([gemm_variant(100, 700, 1), gemm_variant(5000, 10000, 8), gemm_variant(1, 1, 1)]))")
    env = dict(os.environ, MCLST_GEMM_CLUSTER=force)
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    small, big, one = (tuple(v) for v in json.loads(r.stdout.strip().splitlines()[-1]))
    assert big == want
    assert small == one == (want if force == "2" else (1, 64))
