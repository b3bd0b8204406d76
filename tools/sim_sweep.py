"""Per-kernel times of find_matches (+ distances) for one (N, Q) shape, averaged over 5 calls
after 3 warm-ups.  usage: sim_sweep.py N Q [k]"""
import sys, torch
sys.path.insert(0, ".")
from mclstexp_b200 import _lib, retrieval, synth
N, Q = int(sys.argv[1]), int(sys.argv[2]); k = int(sys.argv[3]) if len(sys.argv) > 3 else 50
dev = torch.device("cuda", 0)
bank = torch.from_numpy(synth.embeddings(N, 256, 11, "clustered")).to(dev)
qry = torch.from_numpy(synth.embeddings(Q, 256, 12, "clustered")).to(dev)
for _ in range(3):
    retrieval.find_matches_device(bank, qry, k, dist_p=2)
torch.cuda.synchronize()
agg = {}
reps = 5
for _ in range(reps):
    _lib.profile_enable(True)
    retrieval.find_matches_device(bank, qry, k, dist_p=2)
    for n, t in _lib.profile_collect():
        agg[n] = agg.get(n, 0.0) + t / reps
    _lib.profile_enable(False)
print(f"N={N} Q={Q} k={k}", {a: round(b, 3) for a, b in agg.items()}, "total", round(sum(agg.values()), 3),
      retrieval.last_counters())
