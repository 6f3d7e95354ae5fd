"""Latency of ONE mm_lls_icp-equivalent call (host buffers in, result out) at the reference's own operating point
(script/config/lo_gflag_list_kitti_urban.txt:39-42,64: ~2.6k down-sampled source features vs a <= 20k-point local
map) and at BASELINE config 2 (120k vs 120k), next to the oracle on the host."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from mulls_b200 import synth, abi
from mulls_b200.registration import Context
from oracle import oracle

def downsample(clouds, counts, seed):
    rng = np.random.default_rng(seed); out = []
    for c, k in zip(clouds, counts):
        idx = np.sort(rng.choice(len(c), size=min(k, len(c)), replace=False)) if len(c) else np.arange(0)
        out.append(np.ascontiguousarray(c[idx]))
    return out

ctx = Context(0, 1, 700000, 700000)
full = synth.make_pair(1000, "c2")
cases = {"c2 120k/120k": full}
small = dict(full)
small["src"] = downsample(full["src"], (800, 400, 1200, 200, 0, 0), 1)       # source budget of the urban config
small["tgt"] = downsample(full["tgt"], (9000, 2000, 7000, 2000, 0, 0), 2)    # <= 20k-point local map
p = abi.IcpParams.from_buffer_copy(full["params"]); p.used_feature_type = b"111100"; p.target_bound[:] = synth.cloud_bound(small["tgt"])
small["params"] = p
cases["slam operating point 2.6k/20k"] = small
for name, pair in [(n + m, p) for n, p in cases.items() for m in ("", " [host launch loop]", " [iteration graph]")]:
    ctx.set_tunable("use_graph", 0 if "host launch loop" in name else 1)
    ctx.set_tunable("loop_kernel", 0 if "iteration graph" in name else 1)
    for _ in range(3): res, _ = ctx.run_batch([pair])
    t0 = time.perf_counter(); n = 20
    for _ in range(n): res, _ = ctx.run_batch([pair])
    gpu_ms = (time.perf_counter() - t0) / n * 1e3
    st = ctx.stats()
    t0 = time.perf_counter(); m = 5
    for _ in range(m): o, _ = oracle.icp_run(pair["tgt"], pair["src"], pair["params"], pair["init_guess"], threads=0, want_trace=False)
    cpu_ms = (time.perf_counter() - t0) / m * 1e3
    dt, dr = synth.pose_error(res[0]["T"], o["T"])
    print(f"{name}: GPU call {gpu_ms:.3f} ms (device {st['ms_total']:.3f} ms, {st['kernel_launches']} launches, iters {res[0]['iters']}, code {res[0]['code']}); "
          f"oracle reference-shaped {cpu_ms:.1f} ms; pose diff {dt:.1e} m {dr:.1e} rad", flush=True)
