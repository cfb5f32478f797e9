#!/usr/bin/env python
"""bench.py — headline benchmark of the correlative scan-matching hot path.

Metric (BASELINE.json): candidate poses scored / s (+ loop-closure constraints / s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C]
                  [--dump-outputs DIR]

--config 2 (default, the headline at every N): BASELINE config[1] — 2D
  FastCorrelativeScanMatcher MatchFullSubmap, 1081-beam synthetic scans vs a 1000x1000
  @5 cm ProbabilityGrid, depth-7 PrecomputationGridStack.  A step = MATCHES_PER_STEP
  full-submap matches per GPU.  At N > 1 every rank owns its own submap + scans (weak
  scaling: the ConstraintBuilder queue sharded by submap) and ONE ncclAllGather per step,
  issued inside libcsm_b200.so (csm_cb_batch2d_run), leaves all constraints on all ranks.
--config 4: ConstraintBuilder2D batch at BASELINE size — 1000 submaps x 200 nodes local
  searches (7 m / 30 deg / depth 7 / min_score 0.55), the queue sharded submap-major over
  the N GPUs (STRONG scaling: the total queue is fixed), one allgather of the 200 k records.
--config 5: ConstraintBuilder3D batch — 500 submaps x 100 nodes (64 rings x 1024 az).
--config 3: FastCorrelativeScanMatcher3D on 32 k-point clouds (16 rings x 2048 az), a queue
  of 8 submaps x 64 nodes with 16 matches in flight.
--config 1: RealTimeCorrelativeScanMatcher2D, 1081 beams vs 200x200, 1000 scans / step.
  (`--scale f` shrinks configs 4/5 for quick runs; the line states the size it ran.)

`value`  : device-resident inputs (stacks + clouds in HBM before the timed region).
`e2e`    : the same work through the C ABI with HOST point clouds (H2D + D2H inside).
`--impl reference`: the CPU oracle (restated reference path; the real reference does
not build here, see DESIGN.md) on the host cores, same metric / workload.
`--dump-outputs DIR` (config 2): after the timed steps, rank 0 writes the result records of
  the last timed step (every rank's matches, job order) as DIR/<field>.npy, one file per
  RESULT2D field.  The inputs are seeded, so two builds run with the same arguments can be
  compared output for output.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from benchmarks import synthetic  # noqa: E402

BYTES_PER_CANDIDATE = 1081 * (8 + 1) + 16   # SURVEY.md §8d: N*(8+1)+16 @ N=1081
BYTES_PER_CANDIDATE_RT = 1081 * (8 + 2) + 16
MATCHES_PER_STEP = 64
MIN_SCORE = 0.6          # pose_graph.lua:28 global_localization_min_score
DEPTH = 7                # pose_graph.lua:27
LIN, ANG = 7.0, math.radians(30.0)
WORKLOADS = {
    1: "rt2d_Match_1081beams_200x200_5cm_0.1m_7deg",
    2: "fast2d_MatchFullSubmap_1081beams_1000x1000_5cm_depth7",
    4: "constraint_builder2d_queue_1000submaps_x_200nodes_7m_30deg_depth7",
    5: "constraint_builder3d_queue_500submaps_x_100nodes_64x1024",
    3: "fast3d_Match_queue_16x2048_32kpoints_8submaps_x_64nodes",
}


def make_world(seed, num_scans):
    """Every rank owns a submap of the same synthetic floor plan (so that weak scaling
    compares like with like) and matches its own node scans (poses and noise seeded
    by `seed` = rank) against it."""
    grid, occ = synthetic.make_grid2d(0, 1000)
    rng = np.random.RandomState(seed * 1000 + 17)
    scans = []
    for i in range(num_scans):
        pose = synthetic.random_free_pose(occ, grid, rng)
        scans.append(synthetic.cast_scan(occ, grid, pose, seed=seed * 100000 + i))
    return grid, scans


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons (separate pass, see `clocks.note`)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        super().__init__(daemon=True)
        self.device = device
        self.rows = []
        self.stop_flag = False

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                  "--format=csv,noheader,nounits", "-lms", "100"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.proc = p
        for line in p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])
            if self.stop_flag:
                break
        p.terminate()

    def summary(self):
        self.stop_flag = True
        time.sleep(0.25)
        if getattr(self, "proc", None):
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except (ValueError, IndexError):
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "reasons": sorted(reasons), "samples": len(sm)}


def sample_clocks(local_rank, workload, min_seconds=1.5, min_iters=3):
    """Clocks under load: the poller runs while `workload()` repeats the timed steps right
    after the timed region — never inside it (an nvidia-smi loop contends with kernel
    launches on the driver lock and perturbed round 1's `value`)."""
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.15)
    t_end = time.perf_counter() + min_seconds
    it = 0
    while time.perf_counter() < t_end or it < min_iters:
        workload(it)
        it += 1
    out = sampler.summary()
    out["note"] = ("nvidia-smi -lms 100 while the same steps ran again right after the timed "
                   "region; no poller inside the timed legs")
    return out


def dump_outputs(directory, records):
    """One DIR/<field>.npy per field of `records`: float32 fields stay float32, the others
    (float64 poses, int32 flags / indices / counts) are stored as float64, which holds
    int32 exactly."""
    os.makedirs(directory, exist_ok=True)
    for name in records.dtype.names:
        a = records[name]
        np.save(os.path.join(directory, name + ".npy"),
                a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured"
    except Exception:
        return 6650.0, 1965.0, "fallback"


def read_profile(lib):
    buf = C.create_string_buffer(16384)
    lib().csm_profile_read(buf, 16384)
    kernels = {}
    for ln in buf.value.decode().strip().splitlines():
        nm, n_l, ms, units = ln.split()
        kernels[nm] = {"launches": int(n_l), "ms": float(ms), "units": float(units)}
    return kernels


def roofline_block(kernels, bytes_per_unit, sm_mhz):
    """Roofline of the dominant kernel.  Three readings, all labelled:
      * `frac` / `bound`: the unit ncu shows saturated for this kernel (L1 data-pipe LSU
        wavefronts for the branch kernel: one wavefront / clk / SM), from the COMMITTED ncu
        capture's per-step count (profiles/r2_roofline.json) over the LIVE CUDA-event
        duration — a fraction that can be compared with 1;
      * `hbm`: ncu DRAM bytes over the live duration vs the measured HBM peak (the working
        set is L2-resident, so this is small — no wasted HBM traffic);
      * `algorithmic_GBps`: SURVEY §8d's byte model (one index + one cell per point per
        candidate) — NOT a bound: one loaded word serves 4 children and one staged point
        serves 32 parents, so it exceeds the HBM figure."""
    if not kernels:
        return None
    tot_ms = sum(k["ms"] for k in kernels.values())
    top = max(kernels, key=lambda k: kernels[k]["ms"])
    k = kernels[top]
    peak, sm_max, how = measured_peaks()
    sec = k["ms"] * 1e-3
    alg = k["units"] * bytes_per_unit / sec / 1e9 if sec > 0 else 0.0
    static = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r2_roofline.json")) as f:
            static = json.load(f).get(top, {})
    except Exception:
        pass
    clk_hz = (sm_mhz or sm_max) * 1e6
    out = {"kernel": top, "launches": k["launches"],
           "avg_launch_ms": k["ms"] / max(1, k["launches"]),
           "share_of_step": k["ms"] / tot_ms if tot_ms else None,
           "unit": "GB/s", "peak": peak, "peak_source": how,
           "algorithmic_GBps": alg, "algorithmic_over_hbm_peak": alg / peak,
           "bytes_per_candidate": bytes_per_unit,
           "kernels": {n: {"ms": round(v["ms"], 4), "launches": v["launches"],
                           "candidates": v["units"]} for n, v in kernels.items()}}
    # the captured per-step totals scale with the candidates the live launches scored
    cap_units = static.get("units_per_step")
    scale = (k["units"] / cap_units) if cap_units else 1.0
    if static.get("dram_bytes_per_step") is not None:
        dram = static["dram_bytes_per_step"] * scale
        out["traffic"] = dram / max(1, k["launches"])
        out["hbm"] = {"achieved": dram / sec / 1e9, "peak": peak, "frac": dram / sec / 1e9 / peak}
    else:
        out["traffic"] = None
    lsu_pct = static.get("l1_lsu_pct") or 0.0
    issue_pct = static.get("issue_active_pct") or 0.0
    if static.get("l1_lsu_wavefronts_per_step") and lsu_pct >= issue_pct:
        wf = static["l1_lsu_wavefronts_per_step"] * scale
        peak_wf = 148 * clk_hz     # one data-pipe wavefront per clock per SM
        out["bound"] = "l1tex_lsu_wavefronts"
        out["achieved"] = wf / sec
        out["peak_bound"] = peak_wf
        out["bound_unit"] = "wavefronts/s"
        out["frac"] = wf / sec / peak_wf
        out["ncu_pct_of_peak"] = lsu_pct
    elif static.get("inst_per_step"):
        inst = static["inst_per_step"] * scale
        peak_inst = 148 * 4 * clk_hz   # one warp instruction per clock per SM sub-partition
        out["bound"] = "issue_slots"
        out["achieved"] = inst / sec
        out["peak_bound"] = peak_inst
        out["bound_unit"] = "warp instructions/s"
        out["frac"] = inst / sec / peak_inst
        out["ncu_pct_of_peak"] = issue_pct
    else:
        # no capture committed for this kernel: the HBM reading is all there is
        out["bound"] = "hbm"
        out["achieved"] = out.get("hbm", {}).get("achieved")
        out["frac"] = out.get("hbm", {}).get("frac")
    if static.get("lts_bytes_per_step") is not None:
        out["l2_GBps"] = static["lts_bytes_per_step"] * scale / sec / 1e9
    out["source"] = static.get("source")
    return out


# =============================================================================
# --impl reference: the CPU oracle on the host cores
# =============================================================================
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as oracle
    oracle.build()
    threads = max(1, min(os.cpu_count() or 1, 64))
    if args.config == 1:
        return run_reference_rt(args, oracle, threads)
    full = args.config == 2
    per_step = threads if full else threads * 4  # bounded sample per step
    grid, scans = make_world(0, per_step)
    og = oracle.Grid2D(grid.cells, grid.resolution, grid.max_x, grid.max_y)
    t0 = time.perf_counter()
    om = oracle.FastCorrelativeScanMatcher2D(og, LIN, ANG, DEPTH)
    build_s = time.perf_counter() - t0
    inits = np.zeros((per_step, 3))
    min_score = MIN_SCORE if full else 0.55
    tot_s, tot_c, tot_m = 0.0, 0, 0
    for it in range(args.warmup + args.steps):
        secs, found, scores, poses, cs = oracle.fast2d_batch(
            [om], [0] * per_step, list(range(per_step)), inits, scans, full, min_score, threads)
        if it >= args.warmup:
            tot_s += secs
            tot_c += int(cs.sum())
            tot_m += per_step
    value = tot_c / tot_s
    line = {
        "impl": "reference", "metric": "candidate_poses_scored_per_sec", "value": value,
        "unit": "candidates/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_s / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak" if args.config == 2 else "strong", "vs_baseline": None,
        "dtype": "u8/int32", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.config], "matches_per_step_per_gpu": per_step,
                   "min_score": min_score, "l2": "n/a (host cores)",
                   "parallelism": "%d host threads, one search per thread" % threads,
                   "oracle_stack_build_s": build_s},
        "constraints_per_sec": tot_m / tot_s,
        "cpu_baseline": {"value": value, "unit": "candidates/s", "cores": threads,
                         "kind": "port",
                         "sample": "%d searches per step on %d host threads, oracle/ (C++ "
                                   "restatement, -O3 -DNDEBUG, no -march)" % (per_step, threads)},
        "e2e": {"value": value, "unit": "candidates/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def rt_world(n):
    big, occ = synthetic.make_grid2d(7, 1000)
    grid, occ2 = synthetic.crop_grid(big, occ, 400, 400, 200, 200)
    rng = np.random.RandomState(1)
    scans, inits = [], []
    for i in range(n):
        pose = synthetic.random_free_pose(occ2, grid, rng, margin_cells=15)
        scans.append(synthetic.cast_scan(occ2, grid, pose, seed=i, max_range=30.0))
        inits.append(pose + rng.uniform(-1, 1, 3) * [0.05, 0.05, math.radians(3)])
    return grid, scans, inits


def cpu_rt_sample(oracle, grid, scans, inits, threads):
    """All host threads, one real-time match per task (thread pool over the oracle)."""
    from concurrent.futures import ThreadPoolExecutor
    og = oracle.Grid2D(grid.cells, grid.resolution, grid.max_x, grid.max_y)

    def one(k):
        return oracle.rt2d_match(og, scans[k], inits[k], 0.1, math.radians(7.0), 0.1, 0.1)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:     # ctypes releases the GIL inside the oracle
        out = list(ex.map(one, range(len(scans))))
    return time.perf_counter() - t0, out


def run_reference_rt(args, oracle, threads):
    n = threads * 8
    grid, scans, inits = rt_world(n)
    tot_s, tot_c, tot_m = 0.0, 0, 0
    for it in range(args.warmup + args.steps):
        secs, out = cpu_rt_sample(oracle, grid, scans, inits, threads)
        if it >= args.warmup:
            tot_s += secs
            tot_c += sum(o["candidates_scored"] for o in out)
            tot_m += n
    value = tot_c / tot_s
    print(json.dumps({
        "impl": "reference", "metric": "candidate_poses_scored_per_sec", "value": value,
        "unit": "candidates/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_s / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32 ordered sum", "data": "synthetic",
        "config": {"workload": WORKLOADS[1], "matches_per_step": n},
        "matches_per_sec": tot_m / tot_s,
        "cpu_baseline": {"value": value, "unit": "candidates/s", "cores": threads, "kind": "port",
                         "sample": "%d real-time matches per step on %d host threads" % (n, threads)},
        "e2e": {"value": value, "unit": "candidates/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0}}))


# =============================================================================
# distributed plumbing: torch.distributed only carries the barrier, the scalar
# reductions of the timing and the bootstrap id; the data-path collective is the
# library's own ncclAllGather (csm_cb_batch2d_run).
# =============================================================================
class Dist:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist

    def make_context(self, sm):
        uid = None
        if self.world > 1:
            box = [sm.MultiGpuContext.unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(box, src=0)
            uid = box[0]
        return sm.MultiGpuContext(self.world, self.rank, self.local_rank, uid)

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values, op):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=getattr(self.dist.ReduceOp, op))
        return [float(v) for v in t]

    def gather_stats(self, step_seconds):
        """[[median ms, max ms] per rank] of a leg's timed steps (rank order)."""
        v = [1e3 * float(np.median(step_seconds)), 1e3 * float(np.max(step_seconds))] \
            if len(step_seconds) else [0.0, 0.0]
        t = self.torch.tensor(v, dtype=self.torch.float64, device=self.dev)
        if self.dist is None:
            return [[round(x, 3) for x in v]]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [[round(float(x), 3) for x in o] for o in out]

    def finish(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


# =============================================================================
# config 2 (headline): MatchFullSubmap, weak scaling
# =============================================================================
def bench_full_submap(args, D):
    torch = D.torch
    from cartographer_b200 import scan_matching as sm
    from cartographer_b200._lib import lib
    rank, world, dev = D.rank, D.world, D.dev
    ctx = D.make_context(sm)
    total_steps = args.warmup + args.steps
    num_scans = total_steps * MATCHES_PER_STEP
    grid, scans = make_world(rank, num_scans)
    opts = sm.FastCorrelativeScanMatcherOptions2D(LIN, ANG, DEPTH)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    matcher = sm.FastCorrelativeScanMatcher2D(grid, opts, device=D.local_rank)
    stack_build_ms = 1e3 * (time.perf_counter() - t0)
    clouds = [sm.DeviceCloud(s, device=D.local_rank) for s in scans]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    # the global queue of one step: rank r owns submap r and its MATCHES_PER_STEP searches
    matchers_g = [matcher if r == rank else None for r in range(world)]
    owner = np.arange(world, dtype=np.int32)

    # (the job list is the same every step: built once, outside the timed region)
    jobs_all = np.zeros(world * MATCHES_PER_STEP, sm.JOB2D_DTYPE)
    jobs_all["stack_index"] = np.repeat(np.arange(world), MATCHES_PER_STEP)
    jobs_all["cloud_index"] = np.arange(world * MATCHES_PER_STEP)
    jobs_all["full_submap"] = 1
    jobs_all["min_score"] = MIN_SCORE
    no_collective = bool(os.environ.get("CSM_BENCH_NO_COLLECTIVE"))
    jobs_local = np.zeros(MATCHES_PER_STEP, sm.JOB2D_DTYPE)
    jobs_local["cloud_index"] = np.arange(MATCHES_PER_STEP)
    jobs_local["full_submap"] = 1
    jobs_local["min_score"] = MIN_SCORE
    pad_lo = [None] * (rank * MATCHES_PER_STEP)
    pad_hi = [None] * ((world - 1 - rank) * MATCHES_PER_STEP)

    def run_step(step, step_clouds=None):
        """Identical job list on every rank; only this rank's clouds are materialised
        (the others are never dereferenced here)."""
        own = (step_clouds if step_clouds is not None
               else clouds[step * MATCHES_PER_STEP:(step + 1) * MATCHES_PER_STEP])
        if no_collective:   # diagnostic: the local searches alone
            res, st = sm.match_batch([matcher], list(own), jobs_local, LIN, ANG)
            full = np.zeros(world * MATCHES_PER_STEP, sm.RESULT2D_DTYPE)
            full[rank * MATCHES_PER_STEP:(rank + 1) * MATCHES_PER_STEP] = res
            return full, st
        return sm.match_batch_sharded(ctx, matchers_g, pad_lo + list(own) + pad_hi, jobs_all,
                                      LIN, ANG, owner)

    # ---- device-resident leg (value) -------------------------------------------
    launches0 = sm.kernel_launch_count()
    step_s, cand, found, dev_ms, host_syncs, coll_ms = [], 0, 0, 0.0, 0, 0.0
    mine = slice(rank * MATCHES_PER_STEP, (rank + 1) * MATCHES_PER_STEP)
    results_by_step = []
    for it in range(total_steps):
        flush.zero_()
        D.barrier()
        if it == args.warmup:
            launches0 = sm.kernel_launch_count()
        t0 = time.perf_counter()
        res, st = run_step(it)   # local searches + the allgather + the final synchronise
        dt = time.perf_counter() - t0
        results_by_step.append(res[mine].copy())
        if it >= args.warmup:
            step_s.append(dt)
            cand += st["candidates_scored"]
            found += int(res[mine]["found"].sum())
            dev_ms += st["device_ms"]
            coll_ms += st["collective_ms"]
            host_syncs = max(host_syncs, st["host_syncs"])
    launches = sm.kernel_launch_count() - launches0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res)   # the last timed step, all ranks' matches
    # per-step diagnostics: every rank's median / max step and the library-side split
    diag_v = D.gather_stats(step_s)
    elapsed = D.reduce([float(sum(step_s))], "MAX")[0]
    cand_all, found_all = D.reduce([float(cand), float(found)], "SUM")
    matches_all = world * args.steps * MATCHES_PER_STEP
    value = cand_all / elapsed

    # ---- end-to-end leg: the step's scans start in HOST memory ---------------------
    e2e_s, e2e_c = [], 0
    for it in range(total_steps):
        flush.zero_()
        D.barrier()
        t0 = time.perf_counter()
        step_clouds = [sm.DeviceCloud(scans[it * MATCHES_PER_STEP + b], device=D.local_rank)
                       for b in range(MATCHES_PER_STEP)]          # csm_cloud_create = H2D
        res_e, st_e = run_step(it, step_clouds)                    # results land in host memory
        for c in step_clouds:
            c.close()
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            e2e_s.append(dt)
            e2e_c += st_e["candidates_scored"]
    diag_e = D.gather_stats(e2e_s)
    e2e_elapsed = D.reduce([float(sum(e2e_s))], "MAX")[0]
    e2e_value = D.reduce([float(e2e_c)], "SUM")[0] / e2e_elapsed
    h2d = MATCHES_PER_STEP * 1081 * 12
    d2h = world * MATCHES_PER_STEP * sm.RESULT2D_DTYPE.itemsize

    # ---- clocks (separate pass), roofline (per-kernel CUDA events), CPU baseline ----
    def queue_local(step):
        jobs = np.zeros(MATCHES_PER_STEP, sm.JOB2D_DTYPE)
        for b in range(MATCHES_PER_STEP):
            jobs[b]["cloud_index"] = step * MATCHES_PER_STEP + b
            jobs[b]["full_submap"] = 1
            jobs[b]["min_score"] = MIN_SCORE
        return jobs

    def one(it):   # the timed steps again (clock pass)
        return sm.match_batch([matcher], clouds,
                              queue_local(args.warmup + it % max(1, args.steps)), LIN, ANG)
    clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    if rank == 0:
        clocks = sample_clocks(D.local_rank, one)
    D.barrier()
    roofline = None
    if rank == 0:
        # per-kernel CUDA events over STEP 0 of this rank — the same 16 scans the committed ncu
        # capture (profiles/r2_roofline.json: first step of the process) measured
        lib().csm_profile_enable(1)
        sm.match_batch([matcher], clouds, queue_local(0), LIN, ANG)
        kernels = read_profile(lib)
        lib().csm_profile_enable(0)
        roofline = roofline_block(kernels, BYTES_PER_CANDIDATE, clocks.get("sm_mhz"))
    cpu = None
    parity_checked = parity_failed = 0
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import pyoracle as oracle
        oracle.build()
        threads = max(1, min(os.cpu_count() or 1, 64))
        og = oracle.Grid2D(grid.cells, grid.resolution, grid.max_x, grid.max_y)
        om = oracle.FastCorrelativeScanMatcher2D(og, LIN, ANG, DEPTH)
        sample = (scans * (threads // len(scans) + 1))[:threads]
        secs, found_c, scores_c, poses_c, cs_c = oracle.fast2d_batch(
            [om], [0] * len(sample), list(range(len(sample))), np.zeros((len(sample), 3)), sample,
            True, MIN_SCORE, threads)
        # the same scans went through the engine in the timed steps: compare bit for bit
        for k in range(min(len(sample), len(scans))):
            g = results_by_step[k // MATCHES_PER_STEP][k % MATCHES_PER_STEP]
            ok = bool(g["found"]) == bool(found_c[k])
            if ok and found_c[k]:
                ok = (np.float32(g["score"]) == scores_c[k] and
                      np.array_equal(g["pose_estimate"], poses_c[k]))
            parity_checked += 1
            parity_failed += 0 if ok else 1
        cpu = {"value": float(cs_c.sum()) / secs, "unit": "candidates/s", "cores": threads,
               "kind": "port", "constraints_per_sec": len(sample) / secs,
               "sample": "%d MatchFullSubmap (one per host thread) of the same workload, "
                         "%.1f s wall" % (len(sample), secs)}

    if rank == 0:
        print(json.dumps({
            "metric": "candidate_poses_scored_per_sec", "value": value, "unit": "candidates/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / max(1, args.steps), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
            "config": {"workload": WORKLOADS[2], "matches_per_step_per_gpu": MATCHES_PER_STEP,
                       "world": "one submap of the same synthetic floor plan per rank, per-rank "
                                "node scans", "min_score": MIN_SCORE,
                       "l2": "flushed between steps (256 MB write)",
                       "collective": ("one ncclAllGather per step inside libcsm_b200.so "
                                      "(csm_cb_batch2d_run)" if world > 1 else "none (1 GPU)"),
                       "stack_build_ms": stack_build_ms, "found": found_all,
                       "parallelism": "submap-sharded x%d" % world},
            "constraints_per_sec": matches_all / elapsed,
            "device_ms_per_step": dev_ms / max(1, args.steps),
            "collective_ms_per_step": coll_ms / max(1, args.steps),
            "e2e": {"value": e2e_value, "unit": "candidates/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_elapsed / max(1, args.steps)},
            "gpu_launches": int(launches), "host_syncs_per_batch": host_syncs, "clocks": clocks,
            "parity_checked": parity_checked, "parity_failed": parity_failed,
            "step_ms_per_rank": {"value": diag_v, "e2e": diag_e,
                                 "rank0_value_steps": [round(1e3 * x, 2) for x in step_s],
                                 "note": "[median, max] of each rank's timed steps"},
            "roofline": roofline, "cpu_baseline": cpu}))
    ctx.close()


# =============================================================================
# config 4: the ConstraintBuilder2D queue at BASELINE size, strong scaling
# =============================================================================
def bench_cb2d(args, D):
    torch = D.torch
    from cartographer_b200 import scan_matching as sm
    rank, world = D.rank, D.world
    ctx = D.make_context(sm)
    n_sub = max(world, int(round(1000 * args.scale)))
    n_node = max(2, int(round(200 * args.scale)))
    min_score = 0.55
    distinct = min(n_sub, 16)
    worlds = [synthetic.make_grid2d(s, 1000) for s in range(distinct)]
    opts = sm.FastCorrelativeScanMatcherOptions2D(LIN, ANG, DEPTH)
    # node scans: every node lives in one of the floor plans; all ranks hold all scans
    rng = np.random.RandomState(3)
    scans, truths = [], []
    for nidx in range(n_node):
        g, occ = worlds[nidx % distinct]
        pose = synthetic.random_free_pose(occ, g, rng)
        scans.append(synthetic.cast_scan(occ, g, pose, seed=1000 + nidx))
        truths.append(pose)
    # the whole queue (identical on every rank): submap-major, initial pose = truth (+) U
    jobs = np.zeros(n_sub * n_node, sm.JOB2D_DTYPE)
    k = 0
    for si in range(n_sub):
        for ni in range(n_node):
            jobs[k]["stack_index"] = si
            jobs[k]["cloud_index"] = ni
            jobs[k]["initial_pose"] = truths[ni] + rng.uniform(-1, 1, 3) * [3.0, 3.0, math.radians(15)]
            jobs[k]["min_score"] = min_score
            k += 1
    owner = (np.arange(n_sub) % world).astype(np.int32)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    matchers = [sm.FastCorrelativeScanMatcher2D(worlds[s % distinct][0], opts, device=D.local_rank)
                if owner[s] == rank else None for s in range(n_sub)]
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    clouds = [sm.DeviceCloud(s, device=D.local_rank) for s in scans]
    step_s, cand = [], 0
    res = None
    for it in range(args.warmup + args.steps):
        D.barrier()
        t0 = time.perf_counter()
        res, st = sm.match_batch_sharded(ctx, matchers, clouds, jobs, LIN, ANG, owner)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            step_s.append(dt)
            cand += st["candidates_scored"]
    elapsed = D.reduce([float(sum(step_s))], "MAX")[0]
    cand_all = D.reduce([float(cand)], "SUM")[0]
    found = int(res["found"].sum())
    # e2e: node scans start in host memory (H2D of every scan on every rank), results to host
    e2e_s = []
    for it in range(max(1, min(args.steps, 2))):
        D.barrier()
        t0 = time.perf_counter()
        step_clouds = [sm.DeviceCloud(s, device=D.local_rank) for s in scans]
        sm.match_batch_sharded(ctx, matchers, step_clouds, jobs, LIN, ANG, owner)
        for c in step_clouds:
            c.close()
        e2e_s.append(time.perf_counter() - t0)
    e2e_elapsed = D.reduce([float(np.mean(e2e_s))], "MAX")[0]
    cand_step = cand_all / max(1, args.steps)
    # parity + CPU baseline on a bounded sample (rank 0, any N: results are on every rank)
    cpu, parity_checked, parity_failed = None, 0, 0
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import pyoracle as oracle
        oracle.build()
        threads = max(1, min(os.cpu_count() or 1, 64))
        sample = np.unique(np.linspace(0, len(jobs) - 1, threads * 4).astype(int))
        oms = {}
        for si in sorted({int(jobs[j]["stack_index"]) % distinct for j in sample}):
            g = worlds[si][0]
            oms[si] = oracle.FastCorrelativeScanMatcher2D(
                oracle.Grid2D(g.cells, g.resolution, g.max_x, g.max_y), LIN, ANG, DEPTH)
        keys = sorted(oms)
        secs, found_c, scores_c, poses_c, cs_c = oracle.fast2d_batch(
            [oms[kk] for kk in keys],
            [keys.index(int(jobs[j]["stack_index"]) % distinct) for j in sample],
            [int(jobs[j]["cloud_index"]) for j in sample],
            np.array([jobs[j]["initial_pose"] for j in sample]), scans, False, min_score, threads)
        for i, j in enumerate(sample):
            ok = bool(res[j]["found"]) == bool(found_c[i])
            if ok and found_c[i]:
                ok = (np.float32(res[j]["score"]) == scores_c[i] and
                      np.array_equal(res[j]["pose_estimate"], poses_c[i]))
            parity_checked += 1
            parity_failed += 0 if ok else 1
        cpu = {"value": float(cs_c.sum()) / secs, "unit": "candidates/s", "cores": threads,
               "kind": "port", "constraints_per_sec": len(sample) / secs,
               "sample": "%d of the queue's searches on %d host threads, %.1f s wall" %
                         (len(sample), threads, secs)}
    clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    if rank == 0:
        sub = jobs[owner[jobs["stack_index"]] == 0][:2000]
        dense = [m if m is not None else matchers[0] for m in matchers]
        clocks = sample_clocks(D.local_rank,
                               lambda it: sm.match_batch(dense, clouds, sub, LIN, ANG))
    D.barrier()
    if rank == 0:
        steps = max(1, args.steps)
        print(json.dumps({
            "metric": "candidate_poses_scored_per_sec", "value": cand_all / elapsed,
            "unit": "candidates/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
            "config": {"workload": WORKLOADS[4], "submaps": n_sub, "nodes": n_node,
                       "jobs": len(jobs), "found": found, "min_score": min_score,
                       "distinct_floor_plans": distinct,
                       "note": "%d device stacks built from %d distinct synthetic floor plans; "
                               "inputs (%.1f GB of stacks per rank) exceed L2" %
                               (n_sub, distinct, 0.04 * n_sub / world),
                       "collective": ("one ncclAllGather of %d x 56 B records per step inside "
                                      "libcsm_b200.so" % len(jobs) if world > 1 else "none (1 GPU)"),
                       "stack_build_s_per_rank": build_s,
                       "parallelism": "submap-major shards x%d" % world},
            "constraints_per_sec": len(jobs) * steps / elapsed,
            "e2e": {"value": cand_step / e2e_elapsed, "unit": "candidates/s",
                    "constraints_per_sec": len(jobs) / e2e_elapsed,
                    "h2d_bytes_per_step": n_node * 1081 * 12,
                    "d2h_bytes_per_step": len(jobs) * sm.RESULT2D_DTYPE.itemsize},
            "gpu_launches": int(sm.kernel_launch_count()), "clocks": clocks,
            "parity_checked": parity_checked, "parity_failed": parity_failed,
            "cpu_baseline": cpu, "roofline": None}))
    ctx.close()


# =============================================================================
# config 1: RealTimeCorrelativeScanMatcher2D, batched against a device-resident grid
# =============================================================================
def bench_rt(args, D):
    torch = D.torch
    from cartographer_b200 import scan_matching as sm
    from cartographer_b200._lib import lib
    rank, world = D.rank, D.world
    n = 1000
    grid, scans, inits = rt_world(n)
    opts = sm.RealTimeCorrelativeScanMatcherOptions(0.1, math.radians(7.0), 0.1, 0.1)
    rt = sm.RealTimeCorrelativeScanMatcher2D(opts, device=D.local_rank)
    dg = sm.RealTimeGrid2D(grid, device=D.local_rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=D.dev)
    step_s, cand, dev_ms = [], 0, 0.0
    scores = poses = None
    for it in range(args.warmup + args.steps):
        flush.zero_()
        D.barrier()
        t0 = time.perf_counter()
        scores, poses, st = rt.MatchBatch(inits, scans, dg)   # host scans in, host poses out
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            step_s.append(dt)
            cand += st["candidates_scored"]
            dev_ms += st["device_ms"]
    elapsed = D.reduce([float(sum(step_s))], "MAX")[0]
    cand_all = D.reduce([float(cand)], "SUM")[0]
    # single-call form (the reference signature: grid passed per call)
    t0 = time.perf_counter()
    for k in range(100):
        rt.Match(inits[k], scans[k], grid)
    single_s = (time.perf_counter() - t0) / 100
    roofline = None
    if rank == 0:
        lib().csm_profile_enable(1)
        rt.MatchBatch(inits, scans, dg)
        kernels = read_profile(lib)
        lib().csm_profile_enable(0)
        roofline = roofline_block(kernels, BYTES_PER_CANDIDATE_RT, None)
    cpu, parity_checked, parity_failed = None, 0, 0
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import pyoracle as oracle
        oracle.build()
        threads = max(1, min(os.cpu_count() or 1, 64))
        m = min(n, threads * 8)
        secs, out = cpu_rt_sample(oracle, grid, scans[:m], inits[:m], threads)
        for k in range(m):
            ok = (np.float32(scores[k]) == np.float32(out[k]["score"]) and
                  np.array_equal(poses[k], out[k]["pose"]))
            parity_checked += 1
            parity_failed += 0 if ok else 1
        cpu = {"value": sum(o["candidates_scored"] for o in out) / secs, "unit": "candidates/s",
               "cores": threads, "kind": "port", "matches_per_sec": m / secs,
               "sample": "%d real-time matches on %d host threads, %.2f s wall" % (m, threads, secs)}
    clocks = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    if rank == 0:
        clocks = sample_clocks(D.local_rank, lambda it: rt.MatchBatch(inits, scans, dg))
    D.barrier()
    if rank == 0:
        steps = max(1, args.steps)
        v = cand_all / elapsed
        print(json.dumps({
            "metric": "candidate_poses_scored_per_sec", "value": v, "unit": "candidates/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * elapsed / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 ordered sum / f64 weight", "data": "synthetic",
            "config": {"workload": WORKLOADS[1], "matches_per_step_per_gpu": n,
                       "l2": "flushed between steps (256 MB write)",
                       "note": "value == e2e: the batch entry takes HOST scans and returns host "
                               "poses (H2D + D2H inside every step); only the grid is resident"},
            "matches_per_sec": world * n * steps / elapsed,
            "device_ms_per_step": dev_ms / steps,
            "single_call_ms": 1e3 * single_s,
            "e2e": {"value": v, "unit": "candidates/s", "h2d_bytes_per_step": n * 1081 * 12,
                    "d2h_bytes_per_step": n * 8},
            "gpu_launches": int(sm.kernel_launch_count()), "clocks": clocks,
            "parity_checked": parity_checked, "parity_failed": parity_failed,
            "roofline": roofline, "cpu_baseline": cpu}))
    dg.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results as DIR/<field>.npy (config 2)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config != 2):
        ap.error("--dump-outputs is implemented for the device path of --config 2")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
        return
    D = Dist()
    if args.config == 2:
        bench_full_submap(args, D)
    elif args.config == 4:
        bench_cb2d(args, D)
    elif args.config == 1:
        bench_rt(args, D)
    elif args.config == 3:
        # BASELINE config 3 (FastCSM3D, 16 rings x 2048 az ~ 32 k points) as a queue of 512
        # local matches with 16 in flight (one at a time is latency-bound: ~0.7 ms each)
        from benchmarks import bench_cb3d
        bench_cb3d.run(args, D, WORKLOADS[3], sample_clocks, rings=16, az=2048, base_sub=8,
                       base_node=64)
    else:
        from benchmarks import bench_cb3d
        bench_cb3d.run(args, D, WORKLOADS[5], sample_clocks)
    D.finish()


if __name__ == "__main__":
    main()
