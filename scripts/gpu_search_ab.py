"""A/B of search tunables in ONE process on ONE box: the same resident batch, per-iteration device time of the
search launch (host launch loop, CUDA events), for a list of tunable settings.
    python scripts/gpu_search_ab.py <pairs> <config> "leaf_count=32" "leaf_count=24" "leaf_count=48" ..."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from concurrent.futures import ProcessPoolExecutor
import numpy as np
from mulls_b200 import synth, abi
from mulls_b200.registration import Context

def gen(a):
    p = synth.make_pair(a[0], a[1])
    return {"tgt": p["tgt"], "src": p["src"], "params": bytes(p["params"]), "init_guess": p["init_guess"]}

n_pairs, cfg = int(sys.argv[1]), sys.argv[2]
with ProcessPoolExecutor(min(16, n_pairs)) as ex:
    pairs = list(ex.map(gen, [(1000 + i, cfg) for i in range(n_pairs)]))
for p in pairs:
    p["params"] = abi.IcpParams.from_buffer_copy(p["params"])
ns = max(sum(len(s) for s in p["src"]) for p in pairs); nt = max(sum(len(t) for t in p["tgt"]) for p in pairs)
ctx = Context(0, n_pairs, ns + 16, nt + 16)
ctx.set_tunable("use_graph", 0)
ctx.upload(pairs)
ref = None
for setting in sys.argv[3:]:
    for kv in setting.split(","):
        k, v = kv.split("=")
        ctx.set_tunable(k, int(v))
    best = None
    for r in range(3):
        res, _ = ctx.run_resident()
        st = ctx.stats()
        if best is None or st["ms_search"] < best["ms_search"]:
            best = st
    T = np.array([x["T"] for x in res])
    if ref is None: ref = T
    same = bool(np.array_equal(ref, T))
    it = [round(v, 3) for v in best["ms_search_iter"][: int(best["search_launches"])]]
    print(f"{setting:40s} search {best['ms_search']:.3f} ms {it} iterate {best['ms_iterate']:.3f} total {best['ms_total']:.3f} "
          f"-> {best['algorithmic_bytes'] / 1e6 / best['ms_search']:.1f} GB/s identical={same}", flush=True)
