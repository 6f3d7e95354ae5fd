#!/usr/bin/env python
"""bench.py — registrations/s of the MULLS registration hot path on B200 (BASELINE.json metric).

A "step" is one pass of the whole path (ingest: intersection filter, spatial sort, grid build; all
ICP iterations; posterior) over one batch of synthetic 120k-point 64-beam scan pairs (BASELINE
config 2) per GPU. Per-GPU work is fixed as N grows (weak scaling): every rank registers its own
batch, there is no data-path collective (independent pairs, SURVEY §8e).

  value  registrations/s with the inputs already resident in HBM (CUDA-event time of the library's
         stream, max over ranks)
  e2e    the same through the C-ABI call with HOST (pinned) buffers: H2D of the clouds and D2H of the
         results inside the timed region
  --impl reference   the CPU restatement of the reference's algorithm (oracle) on the host cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "scan-pair registrations/sec (120k-pt 64-beam)"
UNIT = "registrations/s"


def rank_seeds(rank, pairs_per_gpu):
    """Independent scan pairs shard across ranks with no exchange: rank r owns seeds 1000 + r*P .. 1000 + (r+1)*P - 1."""
    return [1000 + rank * pairs_per_gpu + i for i in range(pairs_per_gpu)]


def reduce_over_ranks(dist, device, times, sums):
    """Timing = max over ranks, counters = sum over ranks (dist is torch.distributed or None)."""
    if dist is None:
        return list(times), list(sums)
    import torch

    t = torch.tensor(list(times), device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    s = torch.tensor(list(sums), device=device, dtype=torch.float64)
    dist.all_reduce(s, op=dist.ReduceOp.SUM)
    return [float(v) for v in t.tolist()], [float(v) for v in s.tolist()]


def _gen_one(args):
    seed, config = args
    from mulls_b200 import synth

    p = synth.make_pair(seed, config)
    return {"tgt": p["tgt"], "src": p["src"], "params": bytes(p["params"]), "init_guess": p["init_guess"], "T_gt": p["T_gt"]}


def make_pairs(seeds, config):
    from concurrent.futures import ProcessPoolExecutor

    from mulls_b200 import abi

    workers = max(1, min(len(seeds), (os.cpu_count() or 8) // 2, 16))
    if workers > 1:
        with ProcessPoolExecutor(workers) as ex:
            raw = list(ex.map(_gen_one, [(s, config) for s in seeds]))
    else:
        raw = [_gen_one((s, config)) for s in seeds]
    for r in raw:
        r["params"] = abi.IcpParams.from_buffer_copy(r["params"])
    return raw


def pin_pairs(pairs):
    """Move the clouds into pinned host memory (the e2e leg copies from there every step)."""
    import torch

    keep = []
    for p in pairs:
        for side in ("tgt", "src"):
            new = []
            for a in p[side]:
                t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
                keep.append(t)
                new.append(t.numpy())
            p[side] = new
    return keep


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 200"}


class NvmlClockSampler:
    """The same counters read in-process through NVML every 200 ms (no nvidia-smi process contending for the driver while
    the host-API-heavy e2e leg runs). Same output as ClockSampler.stop()."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        import pynvml

        self.nv = pynvml
        pynvml.nvmlInit()
        # CUDA_VISIBLE_DEVICES may renumber the devices: resolve through the PCI bus id torch reports
        try:
            import torch

            bus = torch.cuda.get_device_properties(gpu_index).pci_bus_id
            dom = getattr(torch.cuda.get_device_properties(gpu_index), "pci_domain_id", 0)
            dev = torch.cuda.get_device_properties(gpu_index).pci_device_id
            self.h = pynvml.nvmlDeviceGetHandleByPciBusId(f"{dom:08x}:{bus:02x}:{dev:02x}.0".encode())
        except Exception:
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        self.sm, self.mx, self.reasons, self._stop = [], 0.0, set(), threading.Event()
        self.lines = self.sm  # (len(sampler.lines) is what the bench checks)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mx = max(self.mx, float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for name, bit in self.REASONS:
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        threading.Thread(target=self._loop, daemon=True).start()

    def stop(self):
        self._stop.set()
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx or None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}


def make_clock_sampler(kind, gpu_index):
    if kind == "off":
        return None
    if kind == "nvml":
        try:
            return NvmlClockSampler(gpu_index)
        except Exception:
            pass
    return ClockSampler(gpu_index)


def host_cores():
    """Cores this process may run on (cgroup / affinity aware — os.cpu_count() is the machine's, not ours)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def gpu_numa_cpus(device_index):
    """CPUs of the NUMA node the GPU hangs off (sysfs), or None."""
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(device_index)],
                                      text=True).strip()
        bus = out[-12:].lower()  # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        return cpus & set(os.sched_getaffinity(0)) or None
    except Exception:
        return None


def cpu_reference_rate(pairs, budget_s, max_regs, all_cores=False):
    """The oracle (CPU restatement of the reference's algorithm) on the host cores.
    reference-shaped (default): kd-tree per class and 3 OpenMP sections per registration as cregistration.hpp:1268-1292,
    cores//3 registrations in flight so that every core the process may use is busy;
    all_cores (BASELINE.md section 3 ii — the best the same algorithm does on the host): `parallel for` over the queries and
    tree-parallel build, 8 threads per registration (more do not pay on one 120k-point registration: 2 s with 128 threads on
    the 128-core box against 55 ms with 8), cores // 8 registrations in flight."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle

    oracle.load()
    cores = host_cores()
    per_reg = min(8, cores)
    workers = max(1, cores // per_reg) if all_cores else max(1, cores // 3)
    n = min(max_regs, max(workers, 1) * 4)
    jobs = [pairs[i % len(pairs)] for i in range(n)]

    def one(p):
        oracle.icp_run(p["tgt"], p["src"], p["params"], p["init_guess"], threads=(per_reg if all_cores else 0), want_trace=False)
        return 1

    t0 = time.perf_counter()
    done = 0
    with ThreadPoolExecutor(workers) as ex:
        for r in ex.map(one, jobs):
            done += r
            if time.perf_counter() - t0 > budget_s and done >= workers:
                break
    dt = time.perf_counter() - t0
    return done / dt, (min(cores, workers * per_reg) if all_cores else min(cores, workers * 3)), done, dt


def dump_outputs(out_dir, results, prefix):
    """Writes the per-pair results of one batch call as out_dir/<prefix><field>.npy, one row per pair: what a caller
    of the call receives, in float64 (float32 where the ABI's field is a float), so that two builds can be compared
    output for output on the benchmark's seeded inputs."""
    os.makedirs(out_dir, exist_ok=True)
    fields = {"T": np.float64, "info": np.float64, "sigma": np.float32, "confidence": np.float32, "code": np.float64,
              "iters": np.float64, "n_corr": np.float64, "n_src": np.float64}
    for name, dtype in fields.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), np.array([r[name] for r in results], dtype=dtype))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=64,
                    help="scan pairs per GPU per step (64 = BASELINE config 4: 512 pairs over 8 GPUs)")
    ap.add_argument("--config", default="c2")
    ap.add_argument("--lanes", type=int, default=4,
                    help="concurrent contexts (CUDA streams) per GPU of the e2e leg; every one-shot call is double-buffered inside "
                         "(measured with 64 pairs: 4 lanes 5 835 reg/s, 6: 5 361, 8: 4 416-5 029, 12: 4 480)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--host-pack", default="auto", choices=["0", "1", "auto"],
                    help="e2e leg: ship the clouds as 48-byte rows (0), repacked to the 28 B wire format on the host "
                         "cores (1), or measure both and report the faster (auto)")
    ap.add_argument("--pack-threads", type=int, default=0, help="host worker threads of the repacking (0: library default)")
    ap.add_argument("--clock-sampler", default="smi", choices=["nvml", "smi", "off"],
                    help="how SM clocks / throttle reasons are sampled during the timed regions: NVML in-process, "
                         "the profiling recipe's nvidia-smi -lms 200 process (default), or not at all (A/B of the sampler's own cost: none measured)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's results of the last timed step (T, info, sigma, confidence, "
                         "code, iters, n_corr, n_src per pair; about 0.5 KB per pair) as DIR/<field>.npy for the "
                         "device-resident value leg and DIR/e2e_<field>.npy for the end-to-end leg")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    workload = {"c2": "synthetic KITTI-shape 64-beam 120k-pt scan-to-scan ICP, max 20 iters (BASELINE configs[1])",
                "c3": "120k-pt source vs 600k-pt submap (BASELINE configs[2])"}.get(args.config, args.config)
    config = {"workload": workload, "pairs_per_gpu_per_step": args.pairs, "streams_per_gpu_e2e": args.lanes, "l2_policy": "inputs larger than L2 "
              f"({args.pairs} pairs x 11.5 MB of input clouds per GPU per step)", "parallelism": f"independent pairs x{world}"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        pairs = make_pairs([1000 + i for i in range(args.pairs)], args.config)  # the GPU arm's pairs of rank 0
        per_step_budget = 8.0
        for _ in range(args.warmup):
            cpu_reference_rate(pairs, 1.0, 8)
        t0 = time.perf_counter()
        regs, cores, rates = 0, 1, []
        for k in range(args.steps):
            shift = (k * 8) % len(pairs)  # every step starts at a different pair: all of them are visited
            rate, cores, done, dt = cpu_reference_rate(pairs[shift:] + pairs[:shift], per_step_budget, 10 ** 9)
            regs += done
            rates.append(rate)
        total = time.perf_counter() - t0
        value = regs / total
        ac_rate, ac_cores, ac_done, ac_dt = cpu_reference_rate(pairs, 6.0, 10 ** 9, all_cores=True)
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(args.steps, 1),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 geometry / f64 accumulation",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"{regs} registrations over the workload's {len(pairs)} pairs, reference-shaped "
                                           f"(3 OpenMP sections each), {max(1, cores // 3)} in flight on {host_cores()} usable cores",
                                 "per_step": {"min": min(rates), "median": float(np.median(rates)), "max": max(rates)},
                                 "all_cores_variant": {"value": ac_rate, "cores": ac_cores,
                                                       "sample": f"{ac_done} registrations, parallel-for over the queries with 8 threads "
                                                                 f"each, {max(1, host_cores() // 8)} in flight, in {ac_dt:.1f} s"}},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch

    from mulls_b200 import synth
    from mulls_b200.registration import Context

    torch.cuda.set_device(local_rank)
    # several ranks share the host: keep each rank (and the library's pack workers / lane threads it spawns) on the
    # cores of its GPU's NUMA node, so that the pinned staging and the repacking stay local to the PCIe root
    affinity = "all usable cores"
    all_cpus = os.sched_getaffinity(0)
    cpus = gpu_numa_cpus(local_rank)
    if cpus:
        share = sorted(cpus)
        if world > 1:
            same = [r for r in range(world) if gpu_numa_cpus(r) == cpus]
            per_node, k = max(1, len(same)), same.index(local_rank)
            share = share[k::per_node] if len(share) >= 4 * per_node else share
        os.sched_setaffinity(0, share)
        affinity = f"{len(share)} cores of the GPU's NUMA node"
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    seeds = rank_seeds(rank, args.pairs)
    pairs = make_pairs(seeds, args.config)
    keep = pin_pairs(pairs)  # noqa: F841
    max_src = max(sum(len(s) for s in p["src"]) for p in pairs)
    max_tgt = max(sum(len(t) for t in p["tgt"]) for p in pairs)
    from mulls_b200.registration import PipelinedContext

    lanes = max(1, min(args.lanes, args.pairs))
    ctx = Context(local_rank, args.pairs, max_src, max_tgt)
    ctx.set_tunable("use_graph", 0)  # per-kernel CUDA events for the roofline: the host launch loop (the lanes run the graph)
    pipe = PipelinedContext(local_rank, lanes, (args.pairs + lanes - 1) // lanes, max_src, max_tgt)

    # ---- (A) device-resident, one stream: per-kernel attribution for the roofline ----------------
    sampler = make_clock_sampler(args.clock_sampler, local_rank)  # samples every 200 ms (the recipe's interval; a 50 ms poll measurably slowed the host-API-heavy e2e leg) through all warm-up and timed regions below
    if sampler:
        sampler.start()
    ctx.upload(pairs)
    res = None
    for _ in range(args.warmup):
        res, _ = ctx.run_resident()
    barrier()
    dev_ms = 0.0
    search_ms = 0.0
    alg_bytes = 0
    launches = 0
    iters = 0
    n_search_launches = 0
    search_iter_ms = np.zeros(64)
    for _ in range(args.steps):
        res, _ = ctx.run_resident()
        st = ctx.stats()
        dev_ms += st["ms_total"]
        search_ms += st["ms_search"]
        alg_bytes += st["algorithmic_bytes"]
        iters += st["iterations"]
        n_search_launches += st["search_launches"]
        search_iter_ms += np.array(st["ms_search_iter"])
    barrier()

    # ---- (B) device-resident throughput: K steps back to back, CUDA events around them. Measured with the whole batch
    # in ONE context (the iteration loop is a CUDA graph; its kernels keep a fixed number of resident blocks busy on the
    # batch's live chunks) and with the batch split over `lanes` concurrent contexts; the better one is the value.
    def timed_resident(p, k):
        p.upload(pairs)
        for _ in range(args.warmup):
            p.run_resident()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_w = time.perf_counter()
        e0.record()
        r, n_launch = p.run_resident_steps(k)  # every stream runs its K passes back to back
        e1.record()
        barrier()
        return r, n_launch, time.perf_counter() - t_w, e0.elapsed_time(e1) / 1e3

    one = PipelinedContext(local_rank, 1, args.pairs, max_src, max_tgt)
    two = PipelinedContext(local_rank, 2, (args.pairs + 1) // 2, max_src, max_tgt) if args.pairs >= 2 else None
    cand = [("1_context", one)] + ([("2_contexts", two)] if two else []) + ([(f"{lanes}_contexts", pipe)] if lanes > 2 else [])
    measured, resident_variants = [], {}
    for name, p in cand:
        r, n_launch, w_s, d_s = timed_resident(p, args.steps)
        measured.append((d_s, name, p, r, n_launch, w_s))
        resident_variants[name] = args.pairs * args.steps / d_s
    lanes_s, best_name, best_pipe, res_p, launches, wall_s = min(measured, key=lambda m: m[0])
    for m in measured:
        for a, b in zip(res_p, m[3]):
            assert np.array_equal(a["T"], b["T"])

    # ---- (B2) the same with convergence switched off: every pair runs all 20 iterations (BASELINE configs[1] "20 iters")
    fixed20 = None
    if args.config == "c2":
        from mulls_b200 import abi as _abi

        pairs20 = []
        for p in pairs:
            q = _abi.IcpParams.from_buffer_copy(p["params"])
            q.converge_translation, q.converge_rotation_d = 0.0, 0.0
            pairs20.append(dict(p, params=q))
        best_pipe.upload(pairs20)
        best_pipe.run_resident()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k20 = args.steps
        f0.record()
        r20, _ = best_pipe.run_resident_steps(k20)
        f1.record()
        barrier()
        assert all(r["iters"] == 20 for r in r20), [r["iters"] for r in r20]
        fixed20 = (k20, f0.elapsed_time(f1) / 1e3)

    # ---- (B3) BASELINE config 5 at N >= 2: ONE 128-beam registration with its source sharded over the ranks, the
    # per-iteration exchanges (claim table: min; counts and per-class sums: sum) as ncclAllReduce calls inside the
    # library (mulls_icp_run_sharded_nccl), next to the same registration unsharded on rank 0's GPU
    c5 = None
    if world > 1 and args.config == "c2":
        from mulls_b200.dist import nccl_init_from_torch, shard_sources

        pair5 = synth.make_pair(1000, "c5")
        shards, base5, glob5 = shard_sources(pair5["src"], rank, world)
        ctx5 = Context(local_rank, 1, max(1, sum(len(x) for x in shards)), sum(len(t) for t in pair5["tgt"]))
        nccl_init_from_torch(ctx5)
        for _ in range(3):
            r5, _ = ctx5.run_sharded_nccl(dict(pair5, src=shards), base5, glob5)
        barrier()
        ms5 = []
        for _ in range(5):
            r5, _ = ctx5.run_sharded_nccl(dict(pair5, src=shards), base5, glob5)
            ms5.append(ctx5.stats()["ms_total"])
        barrier()
        ctx5.close()
        # the exchanges alone: the three all-reduces of one iteration, timed back to back on this rank's stream
        tmin = torch.zeros(sum(len(t) for t in pair5["tgt"]), dtype=torch.int32, device="cuda")
        tcnt = torch.zeros(12, dtype=torch.int32, device="cuda")
        tsum = torch.zeros(6 * 28, dtype=torch.float64, device="cuda")
        for _ in range(3):
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN), dist.all_reduce(tcnt), dist.all_reduce(tsum)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(10):
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN), dist.all_reduce(tcnt), dist.all_reduce(tsum)
        c1.record()
        torch.cuda.synchronize()
        coll_ms = c0.elapsed_time(c1) / 10
        un_ms = None
        if rank == 0:
            one = Context(local_rank, 1, sum(len(x) for x in pair5["src"]), sum(len(t) for t in pair5["tgt"]))
            one.upload([pair5])
            for _ in range(3):
                ru, _ = one.run_resident()
            un = []
            for _ in range(5):
                ru, _ = one.run_resident()
                un.append(one.stats()["ms_total"])
            un_ms = float(np.median(un))
            dtp, drp = synth.pose_error(r5["T"], ru[0]["T"])
            same = r5["code"] == ru[0]["code"] and r5["iters"] == ru[0]["iters"] and dtp <= 1e-4 and drp <= 1e-4
            one.close()
        c5 = {"sharded_ms": float(np.median(ms5)), "collectives_ms_per_iteration": coll_ms, "unsharded_ms": un_ms,
              "iters": r5["iters"], "equal_to_unsharded": bool(same) if rank == 0 else None}

    # ---- (C) end to end through the C-ABI with host (pinned) buffers, same lanes ----------------------
    # The clouds cross PCIe either as the caller's 48-byte rows or repacked on the host cores to the 28 B/point wire
    # format (the "host_pack" tunable, csrc/host_pack.h); both are the same public call and give identical results.
    e2e_variants = {}
    if args.pack_threads > 0:
        pipe.set_tunable("pack_threads", args.pack_threads)
    for hp in ([0, 1] if args.host_pack == "auto" else [int(args.host_pack)]):
        pipe.set_tunable("host_pack", hp)
        pipe.run_batch_steps(pairs, 2)
        barrier()
        t0 = time.perf_counter()
        res_e2e = pipe.run_batch_steps(pairs, args.steps)
        torch.cuda.synchronize()
        e2e_variants[hp] = time.perf_counter() - t0
        for a, b in zip(res, res_e2e):
            assert np.array_equal(a["T"], b["T"])
        barrier()
    # the link itself: one large pinned H2D copy (what bounds the e2e leg: bytes per step / this rate)
    h2d_gbs = None
    try:
        hbuf = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
        dbuf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        dbuf.copy_(hbuf, non_blocking=True)
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(3):
            dbuf.copy_(hbuf, non_blocking=True)
        c1.record()
        torch.cuda.synchronize()
        h2d_gbs = 3 * hbuf.numel() / (c0.elapsed_time(c1) * 1e6)
        del hbuf, dbuf
    except Exception:
        pass
    best_hp = min(e2e_variants, key=e2e_variants.get)
    e2e_s = e2e_variants[best_hp]
    pipe.set_tunable("host_pack", 2)  # the library default (pack when a call ships >= 2^18 points)
    if sampler and len(sampler.lines) < 3:  # very short runs: keep the GPU under the same load until a few samples exist
        t_fill = time.perf_counter()
        while len(sampler.lines) < 3 and time.perf_counter() - t_fill < 2.0:
            pipe.run_resident()
    clocks = sampler.stop() if sampler else {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "off"}
    h2d = sum(a.nbytes for p in pairs for side in ("tgt", "src") for a in p[side])
    if best_hp == 1:  # 28 of the 48 bytes of a row cross PCIe (16 B + 12 B per point, padded per cloud)
        h2d = sum(16 * (len(a) + (3 * len(a) + 3) // 4) for p in pairs for side in ("tgt", "src") for a in p[side])
    from mulls_b200 import abi
    import ctypes

    d2h = args.pairs * ctypes.sizeof(abi.IcpResult)
    for a, b in zip(res, res_p):  # the lanes change nothing in the results
        assert np.array_equal(a["T"], b["T"])

    # quality gate: every registration must have converged onto the ground truth
    errs = [synth.pose_error(r["T"], p["T_gt"]) for r, p in zip(res, pairs)]
    ok = all(r["code"] == 1 for r in res) and max(e[0] for e in errs) < 0.05
    assert ok, ("registration failed inside the benchmark", [r["code"] for r in res], errs)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res_p, "")
        dump_outputs(args.dump_outputs, res_e2e, "e2e_")

    # ---- reduce over ranks -------------------------------------------------------------------
    dev_s = dev_ms / 1e3
    (dev_s, e2e_s, wall_s, lanes_s, f20_s, c5_ms, c5_coll), (launches_all, _, _) = reduce_over_ranks(
        dist, "cuda", [dev_s, e2e_s, wall_s, lanes_s, fixed20[1] if fixed20 else 0.0, c5["sharded_ms"] if c5 else 0.0,
                       c5["collectives_ms_per_iteration"] if c5 else 0.0], [float(launches), float(alg_bytes), float(search_ms)])
    launches = int(launches_all)
    total_regs = args.pairs * world * args.steps
    value = total_regs / lanes_s
    value_single = total_regs / dev_s
    e2e_value = total_regs / e2e_s

    line = None
    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        if os.path.exists(peaks_path):
            try:
                peak = float(json.load(open(peaks_path))["hbm_gbs"])
                peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
            except Exception:
                pass
        traffic, traffic_alg = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("k_search_dram_bytes_per_launch")
                traffic_alg = tj.get("k_search_algorithmic_bytes_per_launch_same_launches")
            except Exception:
                pass
        # rank-0 figures for the dominant kernel (k_search): algorithmic bytes per launch / mean launch time
        st_alg = alg_bytes if dist is None else alg_bytes  # rank 0's own launches
        achieved = (st_alg / 1e9) / (search_ms / 1e3) if search_ms > 0 else 0.0
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * lanes_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 geometry / f64 accumulation", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "timing": "host clock around the synchronous C-ABI calls (pinned host buffers)",
                    "host_pack": best_hp,
                    "pinned_h2d_gbs": h2d_gbs,
                    "link_note": "pinned_h2d_gbs = ONE 256 MB pinned copy at a time; link_bound_value = the e2e rate at that "
                                 "copy rate. Concurrent copies of several lanes have measured above it (38.6 vs 33.3 GB/s)",
                    "link_bound_value": (world * args.pairs * h2d_gbs * 1e9 / h2d) if h2d_gbs else None,
                    "variants": {("rows48" if k == 0 else "host_packed28"): total_regs / world / v
                                 for k, v in e2e_variants.items()} if world == 1 else None},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_search (transform + NN + claim)", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_algorithmic_same_launches": traffic_alg,
                         "traffic_note": "ncu DRAM bytes of the first six k_search launches of one 64-pair run (profiles/traffic.json) next "
                                         "to the algorithmic bytes of the SAME launches; bytes_per_launch below averages over all launches",
                         "peak_source": peak_src,
                         "bytes_per_launch": st_alg / max(n_search_launches, 1),
                         "ms_per_launch": search_ms / max(n_search_launches, 1),
                         "whole_path_frac": (alg_bytes / 1e9) / (dev_ms / 1e3) / peak,
                         "ms_search_by_iteration": [round(float(v) / args.steps, 4) for v in search_iter_ms[:10]]},
            "wall_ms_per_step": 1e3 * wall_s / args.steps,
            "value_single_stream": value_single, "ms_per_step_single_stream": 1e3 * dev_s / args.steps,
            "timing": f"value: CUDA events around {args.steps} back-to-back steps, the best of 1 / 2 / {lanes} concurrent "
                      "contexts sharing the batch (resident_variants); value_single_stream and roofline: the library's own CUDA "
                      "events on its one stream (host launch loop, per-kernel events)",
            "resident_variants": resident_variants if world == 1 else None, "resident_best": best_name,
            "mean_iterations": iters / max(args.pairs * args.steps, 1),
            "fixed_20_iterations": ({"value": args.pairs * world * fixed20[0] / f20_s, "unit": UNIT, "steps": fixed20[0],
                                     "note": "convergence test disabled: every pair runs max_iter_num = 20 iterations"}
                                    if fixed20 else None),
            "host_affinity": affinity,
            "c5_sharded": ({"workload": "one 128-beam scan pair (BASELINE configs[4]: 263k / 265k returns of 300k rays), source classes "
                                        f"sharded over {world} ranks, target replicated",
                            "ms_per_registration_sharded": c5_ms, "ms_per_registration_unsharded_1gpu": c5["unsharded_ms"],
                            "collectives_per_iteration": 3, "collectives_ms_per_iteration": c5_coll, "iterations": c5["iters"],
                            "equal_to_unsharded": c5["equal_to_unsharded"],
                            "timing": "device time of the whole call (ingest + iterations + posterior), max over ranks, median of 5"}
                           if c5 else None),
            "max_pose_err_vs_gt_m": max(e[0] for e in errs),
        }
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)  # the CPU leg uses every core the process may run on
            rate, cores, done, dt = cpu_reference_rate(pairs, 12.0, 10 ** 9)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"{done} registrations of the same pairs in {dt:.1f} s, oracle "
                                              f"reference-shaped (3 OpenMP sections each), {max(1, cores // 3)} in flight"}
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    pipe.close()
    one.close()
    if two:
        two.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
