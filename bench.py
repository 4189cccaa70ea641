#!/usr/bin/env python
"""bench.py -- the reference's headline metric on BASELINE.json configs[1]:
120 000-triangle random-cube scene (create_n_cubes(10 000), src/testbase.rs:608-615), 1 M create_ray rays
(src/testbase.rs:687-691), f32/3D.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--no-extras] [--dump-outputs DIR]

A "step" is one pass of the hot path's query side over one ray batch: batched Bvh::traverse of 1 M rays
against the device-resident tree, producing the CSR hit lists.  At N > 1 every rank traverses its own
1 M-ray shard of the seed chain (weak scaling) and the step ends with every rank holding the GLOBAL CSR:
the all-gather of the hit lists is fused into the traversal over NVLink peer memory (per-ray counts pushed
to all ranks, offsets rebuilt by a local scan, hit lists stored by the emit kernel straight into every
rank's buffer; bvh_b200/dist.py, traverse.cu) -- no NCCL call and no host synchronisation inside the step.

Timing: every step is bracketed by CUDA events on the launching stream (512 MB L2 flush before each,
outside the pair); the step time of the job is the MAX over ranks of that step; `ms_per_step` and `value`
use the MEDIAN over the K timed steps, with min / mean / max reported in `spread` (a single stalled step
used to decide a whole scaling point).  The K steps are additionally bracketed by barrier + synchronize
(`bracket_ms_per_step`, which includes the L2 flush writes).
`e2e` is the same traversal through the host-pointer C-ABI call (pinned host rays in, host CSR out).
The build side (Bvh::build + flatten, Mprims/s) is timed in the same run and reported under "build".
Extras: `sponza16M` = BASELINE configs[3] (Sponza, 16 M incoherent rays, STRONG-scaled over the N GPUs,
global CSR gathered on every rank) on every line; `hbm_bound` (N = 1) = the same walk over a 10 M-triangle
tree that does not fit L2.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CUBES = 10_000           # 120 000 triangles
N_RAYS = 1_000_000
BUILD_PRIM_VISITS = 2_144_236     # P of the 120k scene (sum over internal nodes of their shape count)
METRIC = "traversal_Mrays_per_s"
UNIT = "Mrays/s"
SPONZA_RAYS = 16_000_000


def _config(n_gpus: int) -> dict:
    """One config object for both arms (b200 and --impl reference)."""
    cfg = {"workload": "configs[1]: create_n_cubes(10000) = 120000 triangles, 1M create_ray rays per GPU from seed 0, batched Bvh::traverse -> CSR hit lists",
           "rays_per_gpu": N_RAYS, "shapes": 12 * N_CUBES, "l2": "512 MB flush write between timed iterations", "builder": "exact_sah"}
    if n_gpus > 1:
        cfg["parallelism"] = (f"ray batch sharded over {n_gpus} GPUs (1M rays each), tree replicated; all-gather of the CSR hit lists fused into the "
                              "traversal over NVLink peer memory (CUDA IPC): per-ray counts + hit lists stored into every rank's buffers, offsets rebuilt by a local scan")
    return cfg


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _stats(xs):
    s = sorted(xs)
    return {"min": s[0], "median": s[len(s) // 2], "mean": sum(s) / len(s), "max": s[-1]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        inside = [l for (t, l) in self.lines if self.t0 is not None and self.t0 - 0.15 <= t <= (self.t1 or t) + 0.15]
        window = "timed region"
        if not inside:                     # region shorter than the sampling period: fall back to the whole (loaded) run
            inside, window = [l for (_, l) in self.lines], "warm-up + timed region"
        for l in inside:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ------------------------------------------------------------------------------------------------------
def _cpu_quota():
    """CPUs this container may use on average (cgroup CFS quota), or None.  A burst over 64+ threads finishes one batch quickly and is
    then throttled for the rest of the 100 ms period: per-call times become bimodal (17 ms / 87 ms measured), the SUSTAINED rate is what
    the quota allows."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(p)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / p
    except Exception:
        return None


def _cpu_traverse_leg(steps: int, warmup: int, budget_s: float = 25.0):
    """The reference's CPU path for this workload: the C++ restatement in oracle/ (the Rust crate cannot be built in this image),
    Bvh::traverse (recursive) of the 1 M create_ray rays over the 120 k scene on a persistent pinned thread pool with dynamic
    chunking, visit counters off.  One step = the whole 1 M-ray batch.  value = SUSTAINED rate: rays of all timed steps / wall time of
    the back-to-back loop (>= 3 s), which is stable under a container CPU quota where single calls are not; per-step spread reported."""
    from oracle import oracle as O

    hw = O.hardware_threads()
    quota = _cpu_quota()
    shapes = O.create_n_cubes(N_CUBES)
    res = O.build(shapes, threads=hw)
    sample = N_RAYS
    rays, _ = O.create_rays(sample)

    def once(t):
        return O.traverse(res.nodes, shapes, rays, O.MODE_RECURSIVE, threads=t, count_stats=False).seconds

    def sustained(t, min_s, min_steps, max_steps=400):
        ts, t0 = [], time.perf_counter()
        while (len(ts) < min_steps or time.perf_counter() - t0 < min_s) and len(ts) < max_steps:
            ts.append(once(t))
        return len(ts) * sample / (time.perf_counter() - t0), ts

    cands = {t for t in (hw, hw // 2, hw // 4) if t >= 1}
    if quota:
        cands |= {max(1, min(hw, int(round(quota)))), max(1, min(hw, int(round(2 * quota))))}
    once(hw)                                          # pool creation, page faults
    sweep = {t: sustained(t, 0.6, max(2, warmup))[0] for t in sorted(cands)}
    threads = max(sweep, key=sweep.get)               # "all the host threads it can use": the count with the best sustained rate
    rate, ts = sustained(threads, min(3.0, budget_s), max(steps, 5))
    st = _stats(ts)
    tb = [O.build(shapes, threads=threads).seconds for _ in range(3)]
    b1 = O.build(shapes, threads=1).seconds
    return {"value": rate / 1e6, "seconds": st, "threads": threads, "hw": hw, "quota": quota, "sweep": {str(k): round(v / 1e6, 2) for k, v in sweep.items()},
            "steps": len(ts), "sample": sample, "build_all": len(shapes) / min(tb) / 1e6, "build_1": len(shapes) / b1 / 1e6}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    leg = _cpu_traverse_leg(args.steps, args.warmup)
    value, st = leg["value"], leg["seconds"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": leg["steps"], "warmup": max(args.warmup, 2),
        "ms_per_step": N_RAYS / (value * 1e6) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.gpus),
        "spread_ms": {k: v * 1e3 for k, v in st.items()},
        "notes": "C++ restatement of the reference (oracle/; no Rust toolchain in the image), Bvh::traverse (recursive) on the host cores; the CPU has no sharding, so the "
                 "reference value is the one-process host rate at every --gpus N",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": leg["threads"], "kind": "port", "host_threads_available": leg["hw"], "cgroup_cpu_quota": leg["quota"],
                         "thread_sweep_Mrays_per_s": leg["sweep"],
                         "sample": f"{leg['sample']} rays/step x {leg['steps']} back-to-back steps, sustained rate (total rays / wall time), persistent pinned pool of {leg['threads']} threads, dynamic 2048-ray chunks, counters off"},
        "build": {"value": leg["build_all"], "unit": "Mprims/s", "cores": leg["threads"], "what": "Bvh::build_par analogue (fork-join, grain 64), best of 3"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
def run_b200(args):
    import ctypes as C

    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench.py --gpus N ...")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    from bvh_b200 import api, capi, scenes
    from bvh_b200.dist import ShardedTraversal, shard_range
    from bvh_b200.dtypes import RAY3F

    L = capi.lib()
    ctx = api.Context(local)
    stream = torch.cuda.Stream(dev)            # everything timed runs on this one stream (torch events see it)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    steps, warmup = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def allmax(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def per_step_max(ms_list):
        """[K] per-step times of this rank -> per-step MAX over ranks, and every rank's median."""
        t = torch.tensor(ms_list, dtype=torch.float64, device=dev)
        if world == 1:
            return ms_list, [sorted(ms_list)[len(ms_list) // 2]]
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        m = torch.stack(allt)                                   # [world, K]
        return m.max(dim=0).values.tolist(), m.median(dim=1).values.tolist()

    # ---- inputs: generated on the host once, resident in HBM before anything is timed -------------------
    aabbs = scenes.create_n_cubes_aabbs(N_CUBES)
    n = len(aabbs)
    d_aabbs = torch.from_numpy(aabbs.view(np.uint8).reshape(-1)).to(dev)
    o, d = scenes.ray_endpoints(N_RAYS, first_ray=rank * N_RAYS)          # rank r owns rays [r*1M, (r+1)*1M) of the seed chain
    d_o, d_d = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    d_rays = torch.empty(N_RAYS * RAY3F.itemsize, dtype=torch.uint8, device=dev)
    capi.check(L.bvhgpu_rays_new_dev_f32x3(ctx._h, d_o.data_ptr(), d_d.data_ptr(), N_RAYS, d_rays.data_ptr()))   # Ray::new on the device
    cap = 8 * N_RAYS
    d_off = torch.empty(N_RAYS + 1, dtype=torch.int32, device=dev)
    d_hits = torch.empty(cap, dtype=torch.int32, device=dev)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)    # > 126 MB L2

    bvh = api.Bvh.build_dev(d_aabbs.data_ptr(), n, ctx=ctx)
    bvh.flatten()
    ctx.synchronize()

    sharded = ShardedTraversal(bvh, N_RAYS, 2 * N_RAYS * world) if world > 1 else None

    def step():
        if sharded is None:
            bvh.traverse_dev(d_rays.data_ptr(), N_RAYS, d_off.data_ptr(), d_hits.data_ptr(), cap)
        else:              # walk + the path's one exchange step (fused into the traversal over NVLink peer memory)
            sharded.step(d_rays.data_ptr(), N_RAYS)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(warmup):
        flush.zero_()
        step()
    barrier()
    if rank == 0:                          # nvidia-smi needs a moment for its first sample: keep the GPU loaded until it has one
        t_wait = time.time()
        while not sampler.lines and time.time() - t_wait < 5.0:
            bvh.traverse_dev(d_rays.data_ptr(), N_RAYS, d_off.data_ptr(), d_hits.data_ptr(), cap)   # local work only (no peer handshake)
            torch.cuda.synchronize(dev)
    for _ in range(2):                     # re-align the ranks after the wait loop
        flush.zero_()
        step()
    barrier()
    # ---- the timed region: K steps, nothing but enqueues on the host side (no per-step synchronisation on any rank) --------
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    launches0 = ctx.launch_count()
    sampler.mark_begin()
    t_br0 = time.perf_counter()
    for k in range(steps):
        flush.zero_()                       # L2 flush between timed iterations (outside the event pair)
        ev[k][0].record(stream)
        step()
        ev[k][1].record(stream)
    barrier()
    bracket_ms = (time.perf_counter() - t_br0) * 1e3 / steps
    sampler.mark_end()
    launches = ctx.launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:      # the CSR of the last timed step, before anything else writes the buffers
        if sharded is None:
            off = d_off.cpu().numpy().view(np.uint32)
            if int(off[-1]) > cap:
                raise SystemExit(f"--dump-outputs: {int(off[-1])} hits do not fit the hit buffer (cap {cap})")
            hits = d_hits[: int(off[-1])].cpu().numpy().view(np.uint32)
        else:
            off, hits = sharded.fetch()
        _dump_outputs(args.dump_outputs, np, off, hits)
    mine = [a.elapsed_time(b) for a, b in ev]
    job_ms, rank_medians = per_step_max(mine)
    spread = _stats(job_ms)
    step_ms = spread["median"]
    value = world * N_RAYS / (step_ms * 1e-3) / 1e6
    bracket_ms = allmax(bracket_ms)
    worst = max(range(steps), key=lambda k: job_ms[k])

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.gpus), "gpu_launches": launches, "clocks": clocks,
        "spread": {"ms_per_step": spread, "what": "per step: MAX over ranks of the CUDA-event time; value uses the median", "worst_step": worst,
                   "rank_median_ms": rank_medians, "bracket_ms_per_step": bracket_ms},
    }

    # ---- kernel time of the dominant kernel (profiled steps OUTSIDE the timed region: reading the metric synchronises) -----
    ctx.set_option("profile", 1)
    walk_ms = []
    for _ in range(10):
        flush.zero_()
        step()
        walk_ms.append(ctx.get_metric("walk_ms"))
    ctx.set_option("profile", 0)
    barrier()
    walk = sorted(walk_ms)[len(walk_ms) // 2]
    bvh.traverse_dev(d_rays.data_ptr(), N_RAYS, d_off.data_ptr(), d_hits.data_ptr(), cap, want_total=True)
    visits, hits_total = bvh.traverse_stats()
    alg_bytes = N_RAYS * 36 + visits * 32 + N_RAYS * 4 + hits_total * 4        # DESIGN.md "algorithmic bytes, traversal"
    peak, peak_src = _peaks()
    achieved = alg_bytes / (walk * 1e-3) / 1e9
    prof = _ncu_profile()
    sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    lookups = visits / (walk * 1e-3)
    roofline = {"bound": "hbm", "kernel": "pass 1 of the traversal: walk_top_kernel<false> (top of the tree in shared memory, the rest from the global records; + coherence probe; "
                                          "the one-ray-per-thread kernel is gated off for this incoherent batch)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": prof.get("walk_dram_bytes_per_launch"), "peak_source": peak_src, "bytes_per_launch": alg_bytes, "kernel_ms": walk,
                "node_visits_per_ray": visits / N_RAYS,
                "limiter": "l1tex",
                "l1tex": {"record_fetches_per_s": lookups, "peak_wavefronts_per_s": n_sm * sm_hz, "fetches_per_clk_per_sm": lookups / (n_sm * sm_hz),
                          "ncu_l1tex_throughput_pct": prof.get("walk_l1tex_throughput_pct"), "ncu_dram_throughput_pct": prof.get("walk_dram_throughput_pct"),
                          "ncu_shared_wavefronts_per_launch": prof.get("walk_shared_wavefronts_per_launch"),
                          "ncu_shared_wavefronts_ideal_per_launch": prof.get("walk_shared_wavefronts_ideal_per_launch"),
                          "ncu_global_tag_requests_per_launch": prof.get("walk_global_tag_requests_per_launch"),
                          "what": "one 32-byte record per visit: two LDS.128 in the top of the tree (92 % of the visits), one LDG.256 below it; the L1 data stage "
                                  "moves one 128-byte wavefront / clk / SM and the divergent 16-byte shared reads of a warp collide on banks (3.1 x the ideal wavefront count)"},
                "note": "the contract's bound is HBM and `achieved` counts ALGORITHMIC bytes (frac can exceed 1: 92 % of the record fetches are served by shared memory); the 7.7 MB tree is shared-memory/L1/L2-resident (DRAM traffic per launch in `traffic`), "
                        "so the binding unit is the L1 data stage (`l1tex`), not DRAM; the large-tree case is measured under `hbm_bound`"}
    line["roofline"] = roofline

    # ---- parity of the gathered result, outside the timed region ------------------------------------------------------------
    if sharded is not None:
        line["parity_ok"] = _sharded_parity(torch, dist, np, bvh, sharded, d_rays, d_off, d_hits, cap, rank, world, dev)
        tr = sharded.trace()
        seqs = sorted(tr)[-steps:]
        wt = torch.tensor([[tr[s][0] for s in seqs], [tr[s][1] for s in seqs]], dtype=torch.float64, device=dev) * 1e-6
        allw = [torch.empty_like(wt) for _ in range(world)]
        dist.all_gather(allw, wt)
        line["spread"]["exchange_wait_ms_median_per_rank"] = {"totals": [float(w[0].median()) for w in allw], "done": [float(w[1].median()) for w in allw],
                                                              "what": "time a rank spent waiting for its peers in the two hand-shakes; the rank with the smallest wait is the slowest walker"}

    # ---- e2e: host rays in (compact origin+direction layout, pinned NUMA-local staging from the library), host CSR out -------
    line["e2e"] = _e2e(torch, dist, np, C, capi, ctx, bvh, sharded, d_rays, rank, world, dev, steps, barrier, allmax)

    # ---- extras ------------------------------------------------------------------------------------------------------------
    if not args.no_extras:
        try:
            line["sponza16M"] = _sponza16m(torch, dist, np, api, capi, scenes, ctx, stream, flush, rank, world, dev, barrier, per_step_max)
        except Exception as e:                                   # an extra must never take the headline line down
            line["sponza16M"] = {"error": repr(e)[:300]}

    if world > 1:
        barrier()
        sharded.close()
        if rank == 0:
            print(json.dumps(line), flush=True)
        dist.destroy_process_group()
        return

    # ---- single GPU extras: build, HBM-bound traversal, cpu baseline ---------------------------------------------------------
    def build_median(mode):
        bt = []
        for k in range(3 + 10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            b2 = api.Bvh.build_dev(d_aabbs.data_ptr(), n, ctx=ctx, mode=mode)
            b2.flatten_dev()
            e1.record(stream)
            torch.cuda.synchronize(dev)
            b2.free()
            if k >= 3:
                bt.append(e0.elapsed_time(e1))
        bt.sort()
        return bt[len(bt) // 2]

    build_ms = build_median(capi.BUILD_EXACT_SAH)
    # algorithmic bytes of the build (SURVEY 8d / DESIGN 4.1): n*S_aabb + P*(S_aabb+8+8) + (2n-1)*S_node + n*8, P = sum over internal
    # nodes of their range size = 2 144 236 for this scene (oracle counter; asserted in tests/test_oracle_goldens.py)
    build_bytes = n * 24 + BUILD_PRIM_VISITS * (24 + 8 + 8) + (2 * n - 1) * 64 + n * 8
    line["build"] = {"value": n / (build_ms * 1e-3) / 1e6, "unit": "Mprims/s", "ms": build_ms, "what": "Bvh::build (exact SAH, bit-identical) + flatten, 120000 shapes, AABBs resident in HBM, median of 10",
                     "roofline": {"bound": "hbm", "achieved": build_bytes / (build_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": build_bytes / (build_ms * 1e-3) / 1e9 / peak,
                                  "bytes_per_build": build_bytes, "note": "latency-bound at this size: ~9 multi-warp tree levels + warp-serial subtrees on a 30 MB L2-resident working set (DESIGN.md 4.1)"}}
    lb_ms = build_median(capi.BUILD_LBVH)
    line["build_lbvh"] = {"value": n / (lb_ms * 1e-3) / 1e6, "unit": "Mprims/s", "ms": lb_ms,
                          "what": "BVHGPU_BUILD_LBVH (Morton/Karras, same node layout, identical hit sets, different topology) + flatten"}
    if not args.no_extras:
        try:
            line["hbm_bound"] = _hbm_bound(torch, np, api, capi, scenes, ctx, stream, flush, dev, peak)
        except Exception as e:
            line["hbm_bound"] = {"error": repr(e)[:300]}
    leg = _cpu_traverse_leg(12, 2, budget_s=20.0)
    line["cpu_baseline"] = {"value": leg["value"], "unit": UNIT, "cores": leg["threads"], "kind": "port", "host_threads_available": leg["hw"], "cgroup_cpu_quota": leg["quota"],
                            "thread_sweep_Mrays_per_s": leg["sweep"], "spread_s": leg["seconds"],
                            "sample": f"{leg['sample']} rays x {leg['steps']} back-to-back reps, sustained rate (total rays / wall time), Bvh::traverse (recursive), persistent pinned pool of {leg['threads']} threads, dynamic chunks",
                            "build_Mprims_per_s_1thread": leg["build_1"], "build_Mprims_per_s_all_threads": leg["build_all"]}
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def _dump_outputs(out_dir: str, np, offsets, hits):
    """Writes the CSR a caller of the traversal receives as out_dir/offsets.npy and out_dir/hits.npy, both float32: every offset
    is at most the hit-buffer capacity (<= 16 M < 2**24) and every hit is a shape index (120 000 shapes), so the values are exact."""
    arrays = {"offsets": offsets, "hits": hits}
    for name, a in arrays.items():
        if len(a) and int(a.max()) >= 1 << 24:
            raise SystemExit(f"--dump-outputs: {name} holds values float32 cannot represent exactly")
    nbytes = sum(4 * len(a) for a in arrays.values())
    if nbytes > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {nbytes} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def _sharded_parity(torch, dist, np, bvh, sharded, d_rays, d_off, d_hits, cap, rank, world, dev) -> bool:
    """This rank's slice of the GLOBAL CSR (offsets rebased) == its own single-GPU traversal of its shard, on every rank; and all
    ranks hold the same global CSR (checksum).  Outside the timed region."""
    sharded.step(d_rays.data_ptr(), N_RAYS)
    g_off, g_hits = sharded.fetch()
    bvh.traverse_dev(d_rays.data_ptr(), N_RAYS, d_off.data_ptr(), d_hits.data_ptr(), cap, want_total=True)
    torch.cuda.synchronize(dev)
    l_off = d_off.cpu().numpy().view(np.uint32)
    l_hits = d_hits[: int(l_off[-1])].cpu().numpy().view(np.uint32)
    lo = sharded.rays_before
    sl = g_off[lo: lo + N_RAYS + 1].astype(np.int64)
    ok = bool(np.array_equal(sl - sl[0], l_off.astype(np.int64)) and np.array_equal(g_hits[sl[0]: sl[-1]], l_hits))
    chk = int((g_off.astype(np.uint64).sum() * np.uint64(1000003) + g_hits.astype(np.uint64).sum()) & np.uint64(0x7FFFFFFFFFFFFFFF))
    t = torch.tensor([1 if ok else 0, chk], dtype=torch.int64, device=dev)
    allt = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(allt, t)
    return all(int(x[0]) == 1 for x in allt) and len({int(x[1]) for x in allt}) == 1


def _e2e(torch, dist, np, C, capi, ctx, bvh, sharded, d_rays, rank, world, dev, steps, barrier, allmax):
    """The same traversal through the public host-pointer path.  Inputs: this rank's 1 M rays in the compact BVHGPU_RAYS_OD layout
    (origin + normalised direction, 24 B/ray; inv_direction is recomputed on the device) in pinned host memory obtained from
    bvhgpu_host_alloc (placed on the GPU's NUMA node).  N = 1: bvhgpu_traverse_od_f32x3 (H2D streamed into the running walk kernel,
    offsets + hits back in host memory when the call returns).  N > 1: every rank copies its shard H2D and runs the fused sharded
    step; rank 0 reads the global CSR back (D2H)."""
    L = capi.lib()
    full = d_rays.cpu().numpy().view(np.float32).reshape(-1, 9)
    od_bytes = N_RAYS * 24

    def host_buf(nbytes, dtype):
        p = C.c_void_p()
        capi.check(L.bvhgpu_host_alloc(ctx._h, nbytes, C.byref(p)))
        arr = np.ctypeslib.as_array((C.c_ubyte * nbytes).from_address(p.value)).view(dtype)
        return p, arr

    p_rays, h_od = host_buf(od_bytes, np.float32)
    h_od.reshape(-1, 6)[:] = full[:, :6]
    tot = C.c_size_t(0)
    if sharded is None:
        cap = 8 * N_RAYS
        p_off, h_off = host_buf(4 * (N_RAYS + 1), np.uint32)
        p_hits, h_hits = host_buf(4 * cap, np.uint32)
        fn = L.bvhgpu_traverse_od_f32x3

        def e2e_step():
            capi.check(fn(bvh._h, capi.TRAVERSE_BVH, p_rays, N_RAYS, p_off, p_hits, cap, C.byref(tot)))

        for _ in range(3):
            e2e_step()
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            e2e_step()                       # synchronous call: returns when offsets + hits are in host memory
            ts.append(time.perf_counter() - t0)
        st = _stats(ts)
        streamed = ctx.get_metric("host_streamed")
        # the PCIe floor of this box for the same bytes: plain pinned H2D of the ray buffer, CUDA events, median of 9
        d_tmp = torch.empty(od_bytes, dtype=torch.uint8, device=dev)
        h_t = torch.from_numpy(h_od.view(np.uint8))
        cps = []
        for _ in range(9):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); capi.check(L.bvhgpu_memcpy_h2d_async(ctx._h, C.c_void_p(d_tmp.data_ptr()), p_rays, od_bytes)); b.record()
            torch.cuda.synchronize(dev)
            cps.append(a.elapsed_time(b))
        h2d_ms = sorted(cps)[len(cps) // 2]
        out = {"value": N_RAYS / st["median"] / 1e6, "unit": UNIT, "h2d_bytes_per_step": od_bytes, "d2h_bytes_per_step": (N_RAYS + 1) * 4 + int(tot.value) * 4,
               "ms_per_step": st["median"] * 1e3, "spread_ms": {k: v * 1e3 for k, v in st.items()}, "numa_node_of_gpu": ctx.get_metric("numa_node"),
               "streamed": bool(streamed == 1.0), "pcie_h2d_ms_for_the_same_bytes": h2d_ms, "pcie_h2d_GBps": od_bytes / (h2d_ms * 1e-3) / 1e9,
               "what": "bvhgpu_traverse_od_f32x3: 24 B/ray H2D streamed into the running walk kernel, u32 offsets + hit lists D2H; wall clock around the synchronous call, median"}
        for p in (p_rays, p_off, p_hits):
            L.bvhgpu_host_free(ctx._h, p)
        return out
    # N > 1
    ng = sharded.nrays_global
    d_od = torch.empty(od_bytes, dtype=torch.uint8, device=dev)
    sh = ShardedOD(sharded, capi)
    p_off, h_off = (host_buf(4 * (ng + 1), np.uint32) if rank == 0 else (None, None))
    p_hits, h_hits = (host_buf(4 * sharded.cap, np.uint32) if rank == 0 else (None, None))
    last = [0]
    phases = []

    def e2e_step():
        t0 = time.perf_counter()
        sh.step_host(p_rays.value, d_od.data_ptr(), od_bytes, N_RAYS)
        t1 = time.perf_counter()
        if rank == 0:
            ctx.synchronize()
            t2 = time.perf_counter()
            off, hits = sharded.fetch(h_off, h_hits)
            last[0] = len(hits)
            phases.append((t1 - t0, t2 - t1, time.perf_counter() - t2))

    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e_step()
    barrier()
    ms = allmax((time.perf_counter() - t0) * 1e3 / steps)
    sh.restore()
    ph = [sorted(x)[len(x) // 2] * 1e3 for x in zip(*phases[-steps:])] if phases else None
    out = {"value": world * N_RAYS / (ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": od_bytes * world, "d2h_bytes_per_step": 4 * (ng + 1) + 4 * last[0],
           "ms_per_step": ms, "rank0_phase_ms_median[enqueue H2D+step, wait for the step, D2H of the global CSR]": ph,
           "what": f"every rank: 24 B/ray H2D of its 1M-ray shard + fused sharded step; rank 0: D2H of the global CSR ({ng + 1} offsets + hits); wall clock over the K steps between barriers, MAX over ranks"}
    L.bvhgpu_host_free(ctx._h, p_rays)
    if rank == 0:
        L.bvhgpu_host_free(ctx._h, p_off)
        L.bvhgpu_host_free(ctx._h, p_hits)
    return out


class ShardedOD:
    """Temporarily switches a ShardedTraversal to the compact ray layout."""

    def __init__(self, sharded, capi):
        self.s, self.old = sharded, sharded.shard.ray_layout
        sharded.shard.ray_layout = capi.RAYS_OD

    def step_host(self, *a):
        self.s.step_host(*a)

    def restore(self):
        self.s.shard.ray_layout = self.old


def _numa(ctx):
    try:
        import glob
        import re

        import torch

        bus = torch.cuda.get_device_properties(ctx.device).pci_bus_id
        dom = torch.cuda.get_device_properties(ctx.device).pci_domain_id
        devid = torch.cuda.get_device_properties(ctx.device).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devid:02x}.0/numa_node"
        return int(open(path).read())
    except Exception:
        return None


def _sponza_aabbs(np):
    from bvh_b200.dtypes import BY_PREC

    z = np.load(os.path.join(ROOT, "tests", "golden", "sponza_tris.npz"))
    tris = z["vertices"][z["triangles"].astype(np.int64)]
    sp = np.zeros(len(tris), dtype=BY_PREC["f32"]["aabb"])
    sp["min"] = tris.min(axis=1)
    sp["max"] = tris.max(axis=1)
    return sp


def _sponza16m(torch, dist, np, api, capi, scenes, ctx, stream, flush, rank, world, dev, barrier, per_step_max):
    """BASELINE configs[3]: Sponza (66 450 triangles), 16 M incoherent rays -- create_ray with the scene AABB as bounds, seed chain
    from 0 (src/testbase.rs:619-634, 687-691) -- STRONG-scaled: rank r traverses rays [r*16M/N, (r+1)*16M/N) and every rank ends
    with the global CSR (fused gather).  `hits` and `csr_checksum` must be identical at every N."""
    from bvh_b200.dist import ShardedTraversal, shard_range
    from bvh_b200.dtypes import RAY3F

    L = capi.lib()
    sp = _sponza_aabbs(np)
    bmin, bmax = sp["min"].min(axis=0), sp["max"].max(axis=0)
    lo, hi = shard_range(SPONZA_RAYS, rank, world)
    nloc = hi - lo
    o, d = scenes.ray_endpoints(nloc, first_ray=lo, bounds=(bmin, bmax))
    d_o, d_d = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    d_rays = torch.empty(nloc * RAY3F.itemsize, dtype=torch.uint8, device=dev)
    capi.check(L.bvhgpu_rays_new_dev_f32x3(ctx._h, d_o.data_ptr(), d_d.data_ptr(), nloc, d_rays.data_ptr()))
    del d_o, d_d
    bvh = api.Bvh.build(sp, ctx=ctx)
    cap_g = 12 * SPONZA_RAYS                     # ~10 hits/ray
    if world == 1:
        d_off = torch.empty(nloc + 1, dtype=torch.int32, device=dev)
        d_hits = torch.empty(cap_g, dtype=torch.int32, device=dev)
        sh = None

        def step():
            bvh.traverse_dev(d_rays.data_ptr(), nloc, d_off.data_ptr(), d_hits.data_ptr(), cap_g)
    else:
        sh = ShardedTraversal(bvh, nloc, cap_g)

        def step():
            sh.step(d_rays.data_ptr(), nloc)
    K, W = 7, 3
    for _ in range(W):
        step()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush.zero_()
        ev[k][0].record(stream)
        step()
        ev[k][1].record(stream)
    barrier()
    job_ms, _ = per_step_max([a.elapsed_time(b) for a, b in ev])
    st = _stats(job_ms)
    # result check data (outside the timed region): total hits and a checksum of the global CSR computed on the device
    if sh is None:
        torch.cuda.synchronize(dev)
        total = int(d_off[-1].item()) & 0xFFFFFFFF
        off_t, hits_t = d_off, d_hits[:total]
    else:
        ctx.synchronize()
        g_off = _as_tensor(torch, sh._own[3].value, SPONZA_RAYS + 1, dev)
        total = int(g_off[-1].item()) & 0xFFFFFFFF
        off_t, hits_t = g_off, _as_tensor(torch, sh._own[1].value, total, dev)
    chk = (int(off_t.to(torch.int64).bitwise_and(0xFFFFFFFF).sum().item()) * 1000003 + int(hits_t.to(torch.int64).bitwise_and(0xFFFFFFFF).sum().item())) & 0x7FFFFFFFFFFFFFFF
    same = True
    if sh is not None:
        t = torch.tensor([chk], dtype=torch.int64, device=dev)
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        same = len({int(x.item()) for x in allt}) == 1
        barrier()
        sh.close()
    bvh.free()
    return {"Mrays_per_s": SPONZA_RAYS / (st["median"] * 1e-3) / 1e6, "ms": st["median"], "spread_ms": st, "hits": total, "csr_checksum": chk,
            "all_ranks_hold_the_same_csr": same, "n_gpus": world, "scaling": "strong", "rays": SPONZA_RAYS, "rays_per_gpu": nloc, "shapes": int(len(sp)),
            "what": "BASELINE configs[3]: Sponza, 16M create_ray rays in scene bounds, batched Bvh::traverse, global CSR gathered on every rank inside the step; device-resident rays, "
                    "median of 7 steps (MAX over ranks per step)"}


def _as_tensor(torch, ptr: int, count: int, dev):
    """Zero-copy int32 view of library-owned device memory (for the checksums)."""
    class _Arr:
        pass

    a = _Arr()
    a.__cuda_array_interface__ = {"shape": (count,), "typestr": "<i4", "data": (ptr, False), "version": 3}
    return torch.as_tensor(a, device=dev)


def _hbm_bound(torch, np, api, capi, scenes, ctx, stream, flush, dev, peak):
    """The same walk where the tree does NOT fit L2: 10 M triangles (create_n_cubes(833 334), f32: 20 M records x 32 B = 640 MB), 4 M
    create_ray rays.  Reports the algorithmic bytes of the walk against the measured HBM peak; the DRAM traffic of this launch is in
    profiles/ (ncu)."""
    from bvh_b200.dtypes import RAY3F

    L = capi.lib()
    n_cubes, nrays = 833_334, 4_000_000
    aabbs = scenes.create_n_cubes_aabbs(n_cubes)[:10_000_000]
    d_a = torch.from_numpy(aabbs.view(np.uint8).reshape(-1)).to(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    bvh = api.Bvh.build_dev(d_a.data_ptr(), len(aabbs), ctx=ctx)
    e1.record(stream)
    o, d = scenes.ray_endpoints(nrays)
    d_o, d_d = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    d_rays = torch.empty(nrays * RAY3F.itemsize, dtype=torch.uint8, device=dev)
    capi.check(L.bvhgpu_rays_new_dev_f32x3(ctx._h, d_o.data_ptr(), d_d.data_ptr(), nrays, d_rays.data_ptr()))
    cap = 8 * nrays
    d_off = torch.empty(nrays + 1, dtype=torch.int32, device=dev)
    d_hits = torch.empty(cap, dtype=torch.int32, device=dev)
    ctx.set_option("profile", 1)
    ws = []
    for k in range(3 + 7):
        flush.zero_()
        bvh.traverse_dev(d_rays.data_ptr(), nrays, d_off.data_ptr(), d_hits.data_ptr(), cap)
        w = ctx.get_metric("walk_ms")
        if k >= 3:
            ws.append(w)
    ctx.set_option("profile", 0)
    build_ms = e0.elapsed_time(e1)
    bvh.traverse_dev(d_rays.data_ptr(), nrays, d_off.data_ptr(), d_hits.data_ptr(), cap, want_total=True)
    visits, hits = bvh.traverse_stats()
    walk = sorted(ws)[len(ws) // 2]
    alg = nrays * 36 + visits * 32 + nrays * 4 + hits * 4
    prof = _ncu_profile()
    out = {"shapes": int(len(aabbs)), "tree_bytes": int((2 * len(aabbs) - 2) * 32), "rays": nrays, "kernel_ms": walk, "Mrays_per_s": nrays / (walk * 1e-3) / 1e6,
           "node_visits_per_ray": visits / nrays, "hits": hits, "bytes_per_launch": alg, "achieved_GBps": alg / (walk * 1e-3) / 1e9, "peak_GBps": peak,
           "frac": alg / (walk * 1e-3) / 1e9 / peak, "traffic": prof.get("hbm_bound_walk_dram_bytes_per_launch"),
           "build_ms_exact_sah_first_call": build_ms,
           "what": "walk kernel over a 640 MB tree (10 M triangles, f32), 4 M create_ray rays; algorithmic bytes / kernel time vs the measured HBM copy peak"}
    bvh.free()
    return out


def _ncu_profile():
    """Numbers taken from the committed ncu captures (profiles/traffic.json): DRAM bytes per launch etc."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return {}
    return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the sponza16M / hbm_bound extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the CSR hit lists of the last timed step (global CSR at N > 1) as DIR/offsets.npy and "
                                                          "DIR/hits.npy (float32); the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
