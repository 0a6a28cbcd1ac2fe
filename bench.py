#!/usr/bin/env python
"""bench.py — TEB trajectories/s (and LM iterations/s) of the B200-native optimizer, BASELINE.json's metric.

A "step" is one optimizeTEB pass (no_outer x no_inner LM iterations + cost) over one batch of synthetic planning
requests: `candidates` homotopy candidates x `requests` requests per GPU (weak scaling: per-GPU work is fixed).
Default workload = the north-star scene of BASELINE.json (config C3: car-like, 200 poses, 64 inflated obstacles, 32
candidates per request) x 256 requests = 8192 bands per GPU, i.e. a 629 MB H/b working set (> the 126 MB L2).

  python bench.py --gpus 1 --steps 5 --warmup 3                 # this framework
  python bench.py --impl reference --gpus 1 --steps 3 --warmup 1 # the reference's CPU path (oracle port, all host threads)
  python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR  # + the last timed step's results as DIR/*.npy

Prints ONE JSON line on rank 0 (see the contract in the task statement / DESIGN.md §6).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from teb_local_planner_b200 import abi, scenes  # noqa: E402

METRIC = "TEB trajectories/sec (complete optimizeTEB: outer x inner LM iterations + cost)"
UNIT = "trajectories/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=["C1", "C2", "C3", "C4"])
    ap.add_argument("--requests", type=int, default=256, help="planning requests per GPU per step")
    ap.add_argument("--candidates", type=int, default=None, help="candidates per request (default: config's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-reps", type=int, default=None, help="timed repetitions of the CPU sample (default: 20 for "
                    "--impl reference as BASELINE.md par. 2 asks, 5 for the cpu_baseline leg of the GPU arm)")
    ap.add_argument("--no-single-request", action="store_true")
    ap.add_argument("--total-bands", type=int, default=None, help="STRONG scaling: this many bands in total, split evenly over "
                    "the GPUs (BASELINE config 4: --workload C4 --total-bands 512 --gpus 4); overrides --requests")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last one "
                    "computed (bands, per-band cost / chi2 / status / LM iterations) as DIR/<name>.npy, float64, <= 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, poses, per_band):
    """--dump-outputs: the results a caller of the timed path receives, one DIR/<name>.npy (float64) per array, at most
    DUMP_BYTES in all. Per-band results are written whole; the bands' poses too when they fit, else those of a fixed
    seeded sample of bands. poses_bands.npy holds the indices of the bands in poses.npy. Pose rows at and past a band's
    length n are not part of the result and are written as 0."""
    os.makedirs(out_dir, exist_ok=True)
    out = {k: np.asarray(v, dtype=np.float64) for k, v in per_band.items()}
    B = poses.shape[0]
    room = DUMP_BYTES - sum(v.nbytes for v in out.values()) - 8 * B - 4096 * (len(out) + 2)     # npy headers
    keep = min(B, room // (8 * poses[0].size))
    idx = np.arange(B) if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    sel = np.array(poses[idx], dtype=np.float64)
    sel[np.arange(sel.shape[1])[None, :] >= np.asarray(per_band["n"])[idx][:, None]] = 0.0
    out["poses"], out["poses_bands"] = sel, idx.astype(np.float64)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


def make_workload(a, rank):
    n, M, cand, inflated, moving, via_pts = scenes.CONFIG_SHAPES[a.workload]
    world = max(1, int(os.environ.get("WORLD_SIZE", "1"))) if a.impl == "b200" else 1
    cand = a.candidates or (32 if a.workload in ("C1",) else cand)
    if a.workload == "C3" and a.candidates is None:
        cand = 32  # north-star scene: 200 poses / 64 obstacles / 32 candidates
    if a.workload == "C4" and a.candidates is None:
        cand = 32
    if a.total_bands:   # strong scaling: the job is fixed, every rank takes its share of the requests
        if a.total_bands % (cand * world):
            raise SystemExit(f"--total-bands {a.total_bands} is not a multiple of candidates x GPUs = {cand} x {world}")
        a.requests = a.total_bands // (cand * world)
    p = scenes.config_params(a.workload)
    p.teb_autosize = 0  # throughput runs use fixed n (SURVEY.md §8d); autosize parity is covered by tests/
    hb = scenes.make_batch(n, M, cand, a.requests, seed=1000 + rank, inflated=inflated, moving=moving,
                           via_points=via_pts)
    args = abi.make_args(p.no_inner_iterations, p.no_outer_iterations, True, p.selection_obst_cost_scale,
                         p.selection_viapoint_cost_scale, bool(p.selection_alternative_time_cost))
    desc = {"workload": f"{a.workload}: {'car-like' if p.min_turning_radius > 0 else 'diff-drive'}, {n} poses, {M} "
                        f"{'moving ' if moving else ''}{'inflated ' if inflated else 'point '}obstacles, "
                        f"{cand} candidates/request x {a.requests} requests/GPU, {p.no_outer_iterations}x"
                        f"{p.no_inner_iterations} LM iterations, teb_autosize=false",
            "n_poses": n, "n_obstacles": M, "candidates": cand, "requests_per_gpu": a.requests,
            "bands_per_gpu": hb.B, "via_points": via_pts}
    if a.total_bands:
        desc["total_bands"] = a.total_bands
    return p, hb, args, desc, cand


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark_begin(self):
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        t0 = getattr(self, "t0", 0.0)
        inside = [ln for (ts, ln) in self.lines if t0 <= ts <= self.t1]
        if not inside and self.lines:           # region shorter than one sampling period: the sample closest to it
            inside = [min(self.lines, key=lambda x: abs(x[0] - 0.5 * (t0 + self.t1)))[1]]
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def byte_models(n, M, V, B, K):
    """Bytes per launch (whole batch), N = 4n - 7 unknowns (band rows: 11 entries + rhs = 96 B).
    'algorithmic' = SURVEY.md par. 8(d), what the ALGORITHM has to move per band and LM iteration:
        kernel A  read 32n + 64M + 16V, write 8 (11N + N) + 8            (obstacle rows are 64 B in this ABI, 48 B in 8(d))
        kernel B  read 8*12*N + 32n + 64M, write 32n + 32                (one solve + update + trial chi2)
    'traffic' = what THIS implementation moves (K speculative trials; factor rows written once and read once by the
    back substitution; the solution of every trial written by the solver and read by the evaluation):
        k_solve_tpb   read 96N (band, shared by the K trials) + K 96N (factor), write K (96N + 8N)
        k_trial_eval  read K 8N + 32n + 8N + 64M, write 32n"""
    N = 4 * n - 7
    alg_a = 32 * n + 64 * M + 16 * V + 8 * (11 * N + N) + 8
    alg_b = 8 * 12 * N + 32 * n + 64 * M + 32 * n + 32
    trf_s = 96 * N + K * (2 * 96 * N + 8 * N)
    trf_e = K * 8 * N + 32 * n + 8 * N + 64 * M + 32 * n
    return {"alg_a": alg_a * B, "alg_b": alg_b * B, "traffic_solve": trf_s * B, "traffic_eval": trf_e * B}


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def cpu_quota_cores():
    """CPU bandwidth the container may use (cgroup v2 cpu.max / v1 cfs quota), in cores; None when unlimited."""
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
        if q != "max":
            return float(q) / float(per)
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
            q = float(f.read())
        with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
            per = float(f.read())
        if q > 0:
            return q / per
    except Exception:
        pass
    return None


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def sub_batch(hb, keep):
    return abi.HostBatch(hb.poses[:keep], hb.n[:keep], hb.obstacles, hb.obst_count, hb.scene_id[:keep],
                         hb.via[:keep] if hb.V_cap else None, hb.via_count[:keep] if hb.V_cap else None)


def cpu_arm(p, hb, args, cand, workload, reps, warmup):
    """The reference's CPU path on the host cores, one band at a time per pinned worker thread (the reference's own
    optimizeAllTEBs model). Two builds of it exist and BOTH are timed:
      "reference"  oracle/_ref/libteb_ref.so: the reference's own optimal_planner.cpp / timed_elastic_band.cpp /
                   obstacles.cpp + headers, compiled against stand-ins for Eigen / boost / ROS messages and a restated
                   g2o optimizer (numeric Jacobians, LM, banded Cholesky) - the primary arm whenever the library exists;
      "port"       oracle/teb_oracle.c in g2o mode, the plain-C restatement (bit-identical results, ~20 % faster).
    One repetition processes `sampled_bands` bands of the workload (throughput is per band, bands are independent); the
    thread count is chosen by a probe that runs the SAME sample; value = sampled_bands / median repetition time
    (BASELINE.md par. 2: median + p10 / p90 of >= 20 repetitions for the reference arm). `effective_cores` = process CPU
    time / wall time of the timed repetitions: what the box really served, whatever `nproc` says."""
    from tests import oracle_binding as ob
    from tests import ref_binding as rb
    have_ref = os.path.exists(rb.REF_SO)
    tmax = host_threads()
    # ~8 bands per thread and repetition, bounded to ~25 s of single-thread work per repetition
    per_band_ms = {"C1": 2.5, "C2": 6.0, "C3": 14.0, "C4": 22.0}[workload]
    keep = max(cand, ((8 * tmax + cand - 1) // cand) * cand)
    keep = min(keep, hb.B, max(cand, (int(25000.0 / per_band_ms) // cand) * cand))
    sub = sub_batch(hb, keep)

    def one(threads, kind):
        h = sub.copy()
        c0, t0 = time.process_time(), time.perf_counter()
        if kind == "reference":
            rb.optimize_batch(p, h, args, threads=threads, pin=True)
        else:
            ob.optimize_batch(p, h, args, jac_mode=ob.JAC_G2O, threads=threads, pin=True)
        t1, c1 = time.perf_counter(), time.process_time()
        return t1 - t0, c1 - c0, h

    primary = "reference" if have_ref else "port"
    # thread-count probe on the same sample: all visible CPUs, then halves (SMT siblings / quota-limited boxes)
    tried, best_t, best_sec = [], 1, float("inf")
    t = tmax
    while t >= 1:
        sec = min(one(t, primary)[0] for _ in range(2))
        tried.append((t, round(keep / sec, 1)))
        if sec < best_sec:
            best_t, best_sec = t, sec
        if t == 1 or t <= max(1, tmax // 8):
            break
        t = max(1, t // 2)

    def measure(kind, nrep):
        for _ in range(warmup):
            one(best_t, kind)
        walls, cpus, h = [], [], None
        for _ in range(nrep):
            w, c, h = one(best_t, kind)
            walls.append(w)
            cpus.append(c)
        walls = np.array(walls)
        med = float(np.median(walls))
        return {"value": keep / med, "p10": keep / float(np.percentile(walls, 90)), "p90": keep / float(np.percentile(walls, 10)),
                "ms_per_rep": med * 1e3, "effective_cores": float(np.sum(cpus) / np.sum(walls))}, h

    main, h = measure(primary, reps)
    other = None
    if have_ref:
        other, h_port = measure("port", min(reps, 5))
        assert np.array_equal(h.poses, h_port.poses) and np.array_equal(h.cost, h_port.cost), "oracle/_ref and the port disagree"
        h.lm_iters[...] = h_port.lm_iters
    cpu = {"value": main["value"], "unit": UNIT, "cores": best_t, "kind": primary,
           "p10": main["p10"], "p90": main["p90"], "reps": reps, "sampled_bands": int(keep), "ms_per_rep": main["ms_per_rep"],
           "effective_cores": main["effective_cores"],
           "host": {"visible_cpus": tmax, "cgroup_quota_cores": cpu_quota_cores(), "cpu_model": cpu_model()},
           "thread_probe": tried, "lm_iters_per_s": float(h.lm_iters.sum()) / (main["ms_per_rep"] * 1e-3),
           "port_value": other["value"] if other else None,
           "sample": f"{keep} bands of this workload per repetition, " +
                     ("oracle/_ref (the reference's own optimal_planner.cpp / timed_elastic_band.cpp / obstacles.cpp, restated g2o optimizer)"
                      if have_ref else "oracle/teb_oracle.c in g2o mode (numeric Jacobians, banded Cholesky)") +
                     f", one band at a time per pinned host thread, {best_t} threads (of {tmax} visible), median of {reps} repetitions"
                     + ("; port_value = the plain-C restatement on the same sample (identical results)" if have_ref else "")}
    return cpu, sub, h


def run_reference(a, rank, world):
    if rank != 0:
        return
    p, hb, args, desc, cand = make_workload(a, 0)
    reps = a.cpu_reps or max(20, a.steps)
    cpu, _, h = cpu_arm(p, hb, args, cand, a.workload, reps, max(1, a.warmup))
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, h.poses, {"n": h.n, "cost": h.cost, "chi2": h.chi2, "status": h.status,
                                               "lm_iters": h.lm_iters})
    value = cpu["value"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": cpu["ms_per_rep"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(desc, sampled_bands=cpu["sampled_bands"],
                           sampling="one step = sampled_bands bands of the workload (bands are independent: throughput is per band)"),
            "lm_iters_per_s": cpu["lm_iters_per_s"],
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the reference's own planner sources over a restated g2o optimizer (oracle/_ref), not the upstream g2o "
                    "binary: g2o / CSparse / Eigen / Boost / ROS are absent from the image (DESIGN.md par. 3)"}
    print(json.dumps(line), flush=True)


def run_b200(a, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import teb_local_planner_b200 as T

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    p, hb, args, desc, cand = make_workload(a, rank)
    B, n_cap = hb.B, hb.n_cap
    g = T.TebGpu(B, n_cap, hb.S, max(hb.M_cap, 1), hb.V_cap, device=local_rank)
    g.set_params(p)
    if world > 1:   # the cost all-gather lives behind the C-ABI (ncclAllGather); torch.distributed only carries the id
        from teb_local_planner_b200 import distributed as D0
        D0.init_comm(g, rank, world, device=dev)
    # a non-default torch stream: its handle is passed to the C-ABI so that torch ops (input restore, NCCL) and
    # the optimizer kernels are ordered on ONE stream, and torch.cuda.Event timing sees the kernels
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    def to_dev(arr):
        return torch.from_numpy(arr.view(np.uint8).reshape(-1)).to(dev)

    # ---------------- device-resident path ("value"): inputs already in HBM
    d_pristine = to_dev(hb.poses)
    d_poses = d_pristine.clone()
    d_n, d_sid, d_ob, d_oc = to_dev(hb.n), to_dev(hb.scene_id), to_dev(hb.obstacles), to_dev(hb.obst_count)
    d_vs, d_vg, d_rot = to_dev(hb.vel_start), to_dev(hb.vel_goal), to_dev(hb.prefer_rotdir)
    d_via = to_dev(hb.via) if hb.V_cap else None
    d_vc = to_dev(hb.via_count) if hb.V_cap else None
    d_cost = torch.zeros(B, dtype=torch.float64, device=dev)
    d_chi2 = torch.zeros_like(d_cost)
    d_status = torch.zeros(B, dtype=torch.int32, device=dev)
    d_iters = torch.zeros_like(d_status)
    d_all_cost = torch.zeros(B * world, dtype=torch.float64, device=dev)
    bs = abi.TebBatch()
    bs.B, bs.n_cap, bs.S, bs.M_cap, bs.V_cap = B, n_cap, hb.S, hb.M_cap, hb.V_cap
    bs.poses, bs.n, bs.scene_id = d_poses.data_ptr(), d_n.data_ptr(), d_sid.data_ptr()
    bs.obstacles, bs.obst_count = d_ob.data_ptr(), d_oc.data_ptr()
    bs.via = d_via.data_ptr() if hb.V_cap else None
    bs.via_count = d_vc.data_ptr() if hb.V_cap else None
    bs.vel_start, bs.vel_goal, bs.prefer_rotdir = d_vs.data_ptr(), d_vg.data_ptr(), d_rot.data_ptr()
    bs.cost, bs.chi2, bs.status, bs.lm_iters = d_cost.data_ptr(), d_chi2.data_ptr(), d_status.data_ptr(), d_iters.data_ptr()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def device_step():
        d_poses.copy_(d_pristine)                       # fresh synthetic inputs, already resident in HBM
        g.optimize_device(bs, args, stream.cuda_stream)  # all kernels of optimizeTEB for the whole batch
        if world > 1:   # the ONE collective: per-candidate costs, tebgpu_gather_costs on the same stream
            g.gather_costs_device(d_cost.data_ptr(), B, d_all_cost.data_ptr(), stream.cuda_stream)

    sampler = ClockSampler(local_rank)      # started before the warm-up so that nvidia-smi is already streaming
    sampler.start()
    for _ in range(a.warmup):
        flush.zero_()
        device_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.mark_begin()                    # only samples taken inside the timed region are reported
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    for k in range(a.steps):
        flush.zero_()                                   # L2 flush between timed iterations (outside the events)
        ev[k][0].record(stream)
        device_step()
        ev[k][1].record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    if a.dump_outputs and rank == 0:    # before the profiled pass below overwrites the results of the last timed step
        like = lambda d, arr: d.cpu().numpy().view(arr.dtype).reshape(arr.shape)     # byte tensors -> host arrays
        per_band = {"n": like(d_n, hb.n), "cost": d_cost.cpu().numpy(), "chi2": d_chi2.cpu().numpy(),
                    "status": d_status.cpu().numpy(), "lm_iters": d_iters.cpu().numpy()}
        if world > 1:
            per_band["cost_all_ranks"] = d_all_cost.cpu().numpy()
        dump_outputs(a.dump_outputs, like(d_poses, hb.poses), per_band)
    dev_ms = sum(s.elapsed_time(e) for s, e in ev)
    launches_per_step = g.launch_count()
    lm_iters_step = int(d_iters.sum().item())
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        it = torch.tensor([lm_iters_step], dtype=torch.float64, device=dev)
        dist.all_reduce(it, op=dist.ReduceOp.SUM)
        lm_iters_step = int(it.item())
    dev_ms = float(t.item())
    ms_per_step = dev_ms / a.steps
    value = B * world / (ms_per_step * 1e-3)

    # best-candidate selection on the gathered costs (host, selectBestTeb) - sanity only, outside the timing
    costs = (d_all_cost if world > 1 else d_cost).cpu().numpy()
    from teb_local_planner_b200 import distributed as D
    best = D.select_best_per_request(costs, cand, p)

    # ---------------- per-kernel times for the roofline (separate profiled pass, CUDA events around every launch)
    g.set_profiling(True)
    for _ in range(2):
        flush.zero_()
        d_poses.copy_(d_pristine)
        g.optimize_device(bs, args, stream.cuda_stream)
    kt = g.kernel_times()
    g.set_profiling(False)
    peak, peak_src = hbm_peak()
    # speculation widths the library chose (tebgpu_get_info): first LM iteration after a graph rebuild / later ones
    spec_k, spec_first = g.speculation_width(), g.info(7)
    k_avg = (spec_first + (p.no_inner_iterations - 1) * spec_k) / max(1, p.no_inner_iterations)
    bm = byte_models(desc["n_poses"], desc["n_obstacles"], desc["via_points"], B, k_avg)
    working_set_mb = B * 4 * n_cap * 96 / 1e6
    ws_note = ("H/b working set %.0f MB %s the 126 MB L2" % (working_set_mb, ">" if working_set_mb > 126 else "<=")
               + ("" if working_set_mb > 126 else ": L2-resident, latency-bound; HBM fraction is indicative only"))
    try:    # ncu-measured DRAM bytes per launch, when a capture of this workload has been summarised under profiles/
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ncu_tr = json.load(f).get(f"{a.workload}_B{B}", {})
    except Exception:
        ncu_tr = {}

    def avg_ms(*names):
        tot = 0.0
        for nme in names:
            ms, cnt = kt[nme]
            if cnt == 0:
                return None
            tot += ms / cnt
        return tot

    def roof(label, names, alg_bytes, model_traffic=None):
        """frac (= frac_algorithmic): SURVEY 8(d) bytes / CUDA-event launch time / measured peak;
        frac_traffic: the bytes this implementation really moves (model; `traffic` = ncu DRAM bytes when captured)."""
        t = avg_ms(*names)
        if t is None:
            return None
        ach = alg_bytes / (t * 1e-3) / 1e9
        r = {"kernel": label, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
             "frac_algorithmic": ach / peak, "avg_launch_ms": t, "algorithmic_bytes_per_launch": int(alg_bytes),
             "traffic": ncu_tr.get(label), "peak_source": peak_src, "note": ws_note}
        if r["traffic"] is None and all(nme in ncu_tr for nme in names):   # a launch PAIR: sum of the captured launches
            r["traffic"] = int(sum(ncu_tr[nme] for nme in names))
            r["traffic_note"] = "sum of the ncu DRAM bytes of one captured launch of each kernel (see profiles/ncu_traffic.json for which)"
        if model_traffic is not None:
            r["modelled_traffic_bytes_per_launch"] = int(model_traffic)
            r["frac_traffic"] = model_traffic / (t * 1e-3) / 1e9 / peak
        elif r["traffic"]:
            r["frac_traffic"] = r["traffic"] / (t * 1e-3) / 1e9 / peak
        return r

    total_ms = sum(v[0] for v in kt.values())
    shares = {k: (v[0] / total_ms if total_ms > 0 else 0.0) for k, v in kt.items()}
    roof_a = roof("k_linearize", ["k_linearize"], bm["alg_a"], bm["alg_a"])
    # kernel B of SURVEY 8(d) = solve + update + trial chi2 = the k_solve_tpb / k_trial_eval pair; its algorithmic bytes
    # credit ONE trial per LM iteration (what the launch pair advances), the traffic model counts all K speculative ones
    roof_b = roof("k_solve_tpb+k_trial_eval", ["k_solve_tpb", "k_trial_eval"], bm["alg_b"],
                  bm["traffic_solve"] + bm["traffic_eval"])
    roof_s = roof("k_solve_tpb", ["k_solve_tpb"], bm["alg_b"], bm["traffic_solve"])
    roof_e = roof("k_trial_eval", ["k_trial_eval"], bm["alg_b"], bm["traffic_eval"])
    cands = [(r, sum(kt[k][0] for k in names)) for r, names in ((roof_a, ["k_linearize"]),
             (roof_b, ["k_solve_tpb", "k_trial_eval"])) if r is not None]
    dominant = max(cands, key=lambda x: x[1])[0]

    # ---------------- end-to-end path: public C-ABI call with HOST (pinned) buffers, H2D + D2H inside
    pin = {}
    def pinned_like(arr):
        tt = torch.empty(arr.nbytes, dtype=torch.uint8).pin_memory()
        view = tt.numpy().view(arr.dtype).reshape(arr.shape)
        view[...] = arr
        pin[id(view)] = tt
        return view
    hp = abi.HostBatch.__new__(abi.HostBatch)
    hp.__dict__.update(hb.__dict__)
    for name in ("poses", "n", "scene_id", "obstacles", "obst_count", "via", "via_count", "vel_start", "vel_goal",
                 "prefer_rotdir", "cost", "chi2", "status", "lm_iters"):
        setattr(hp, name, pinned_like(getattr(hb, name)))
    h2d = sum(getattr(hp, k).nbytes for k in ("poses", "n", "scene_id", "obstacles", "obst_count", "vel_start",
                                               "vel_goal", "prefer_rotdir")) + (hp.via.nbytes + hp.via_count.nbytes if hb.V_cap else 0)
    d2h = sum(getattr(hp, k).nbytes for k in ("poses", "n", "cost", "chi2", "status", "lm_iters"))
    pristine_host = hb.poses.copy()
    e2e_t = []
    gather_in = torch.zeros(B, dtype=torch.float64, device=dev)
    for k in range(a.warmup + a.steps):
        hp.poses[...] = pristine_host
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        if world > 1:
            host_all = g.optimize_gather(hp, args)      # tebgpu_optimize_batch_gather: H2D, kernels, all-gather, D2H
        else:
            g.optimize(hp, args)                        # H2D, all kernels, D2H of poses/cost/status, synchronous
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        if k >= a.warmup:
            e2e_t.append(t1 - t0)
    e2e_ms = float(np.mean(e2e_t)) * 1e3
    te = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())
    e2e_value = B * world / (e2e_ms * 1e-3)
    # device-resident result == host-path result (same kernels): guard against a silently different path
    assert np.array_equal(hp.cost, d_cost.cpu().numpy()), "device-resident and host entry points disagree"

    # ---------------- one planning request alone (B = candidates): the reference's real-time call shape
    single = None
    if rank == 0 and not a.no_single_request:
        bs.B = cand                                     # the first request: bands 0 .. cand-1 of scene 0
        evs = []
        for k in range(25):
            d_poses.copy_(d_pristine)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            g.optimize_device(bs, args, stream.cuda_stream)
            e1.record(stream)
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ms = np.array([x.elapsed_time(y) for x, y in evs[5:]])
        single = {"bands": cand, "ms_per_request": float(np.median(ms)), "p10_ms": float(np.percentile(ms, 10)),
                  "p90_ms": float(np.percentile(ms, 90)), "trajectories_per_s": cand / (float(np.median(ms)) * 1e-3),
                  "gpu_launches": g.launch_count(), "speculation_width": g.speculation_width(),
                  "lm_iterations": f"{p.no_outer_iterations}x{p.no_inner_iterations}",
                  "note": "device-resident, CUDA events, median of 20 after 5 warm-ups; L2-resident, latency-bound"}
        bs.B = B

    # ---------------- CPU baseline on the host cores (rank 0, N = 1 only): oracle port, bounded sample; the same
    # sample is then optimised on the GPU and compared band by band (the oracle is the checker here, not the product)
    cpu, parity = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu, sub, ref = cpu_arm(p, hb, args, cand, a.workload, a.cpu_reps or 5, 1)
        got = sub.copy()
        g.optimize(got, args)
        dmax = np.array([np.abs(got.poses[b_, :got.n[b_]] - ref.poses[b_, :ref.n[b_]]).max() if got.n[b_] == ref.n[b_]
                         else np.inf for b_ in range(sub.B)])
        parity = {"against": "cpu_baseline run (the reference's code path: numeric Jacobians, delta 1e-9)",
                  "bands": int(sub.B), "tolerance": 1e-4,
                  "fraction_within_1e-4": float(np.mean(dmax <= 1e-4)), "fraction_within_1e-6": float(np.mean(dmax <= 1e-6)),
                  "median_abs_pose_diff": float(np.median(dmax)), "max_abs_pose_diff": float(dmax.max()),
                  "lm_iters_equal_fraction": float(np.mean(got.lm_iters == ref.lm_iters))}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if a.total_bands else "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": dict(desc, l2="flushed between timed steps (256 MB memset)", timing="CUDA events per step on the launching stream, max over ranks"),
                "lm_iters_per_s": lm_iters_step / (ms_per_step * 1e-3),
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_ms, "api": "tebgpu_optimize_batch" + ("_gather" if world > 1 else "") + " (C-ABI, pinned host buffers)"},
                "gpu_launches": int(launches_per_step * a.steps),
                "gpu_launches_per_step": int(launches_per_step),
                "roofline": dominant, "roofline_kernel_a": roof_a, "roofline_kernel_b": roof_b,
                "roofline_kernel_b_solve": roof_s, "roofline_kernel_b_eval": roof_e, "speculation_width": spec_k, "speculation_width_first_iteration": spec_first,
                "single_request": single, "parity_sample": parity,
                "kernel_time_share": shares,
                "kernel_time_share_note": "from a separate profiled pass (CUDA events around every launch); "
                                          "k_lm_step_or_retry_rounds = the solve + evaluation launches of the retry rounds "
                                          "(same stream as everything else in the throughput regime)",
                "cpu_baseline": cpu, "clocks": clocks,
                "best_candidate_of_request0": int(best[0])}
        print(json.dumps(line), flush=True)
    g.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        run_reference(a, rank, world)
    else:
        run_b200(a, rank, local_rank, world)


if __name__ == "__main__":
    main()
