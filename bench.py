#!/usr/bin/env python
"""bench.py -- turntable registration throughput on B200 (BASELINE.json metric).

A "step" is ONE registration of the whole synthetic turntable sequence (BASELINE.json configs[1]):
V views x N points, the V ring pairs (k+1 -> k, closing pair 0 -> V-1) each aligned by 30 fixed
iterations of reciprocal point-to-point ICP with a 4 mm gate (the reference's ICP settings,
mvr/src/registrator.cpp:551-560), per-pair results gathered over NCCL, then the host loop closure.
With --gpus N the V pairs are block-partitioned over N ranks (configs[2]); total work is fixed.

  value          NN queries/s of the whole job, scans already resident in HBM (device-timed)
  ms_per_step    registration time of the sequence (the second half of BASELINE's metric)
  e2e            the same job through the host-buffer C ABI: every step copies each scan H2D from pinned
                 host memory and reads poses/residuals back
  roofline       the correspondence kernel (forward + reciprocal NN): algorithmic bytes / CUDA-event time
  cpu_baseline   the CPU oracle (port of the reference's PCL path) on a bounded sample, same box

`--impl reference` times that CPU path alone (rank 0 only) and prints the same JSON shape.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = ("nn_queries_per_s (24-view x 200k turntable registration; ms_per_step = registration ms; a query = one PCL-equivalent "
          "nearest-neighbour answer: every source point per iteration + every gated match's reciprocal answer, the oracle's counter)")
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--views", type=int, default=24)
    ap.add_argument("--points", type=int, default=200_000)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--max-dist", type=float, default=4.0)
    ap.add_argument("--reciprocal", type=int, default=1)
    ap.add_argument("--cpu-sample-pairs", type=int, default=2, help="pairs the cpu_baseline leg aligns (0 = skip)")
    ap.add_argument("--cpu-reps", type=int, default=3, help="repetitions of the CPU sample (the minimum is reported)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--workload", default="registration", choices=["registration", "nn_sweep"],
                    help="registration: BASELINE configs[1]/[2] (the default, the driver's line); nn_sweep: configs[4], exact NN of 10k..16M "
                         "queries against a 1M-point target")
    ap.add_argument("--nn-target", type=int, default=1_000_000)
    ap.add_argument("--nn-queries", type=int, default=16_000_000, help="queries of the headline step of the nn_sweep workload")
    ap.add_argument("--single-process", action="store_true",
                    help="N GPUs from ONE process through mvr_register_turntable_multi (one host thread per GPU, ncclAllGather inside the "
                         "C ABI); the default for --gpus N > 1 when not launched by torchrun")
    ap.add_argument("--streams", type=int, default=1, help="GPU contexts created up front (the driver grows the pool to one per pair)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 or float64, "
                         "at most 64 MB; the NN sweep writes a fixed sample of its answers), so that two builds can be compared "
                         "output for output")
    return ap.parse_args()


DUMP_LIMIT = 64 << 20
NN_DUMP_SAMPLE = 1 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: one DIR/<name>.npy per array.  float32 arrays stay float32; everything else (float64, counts,
    indices) is written as float64, which holds each of these values exactly."""
    out = {}
    for name, x in arrays.items():
        x = np.asarray(x)
        out[name] = np.ascontiguousarray(x, dtype=np.float32 if x.dtype == np.float32 else np.float64)
    total = sum(x.nbytes for x in out.values())
    if total > DUMP_LIMIT:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (total, DUMP_LIMIT))
    os.makedirs(path, exist_ok=True)
    for name, x in out.items():
        np.save(os.path.join(path, name + ".npy"), x)


def registration_outputs(view_poses, records):
    """What a caller of the turntable registration receives: the absolute pose of every view (V x 4 x 4) and the result of
    every ring pair (the gathered pair records)."""
    import mvr_b200.ring as ring
    rec = np.asarray(records).view(ring.RECORD).reshape(-1)
    return {"view_poses": np.asarray(view_poses, dtype=np.float32).reshape(-1, 4, 4),
            "pair_poses": rec["pose"].reshape(-1, 4, 4).transpose(0, 2, 1),
            "pair_n_corr": rec["n_corr"], "pair_iterations": rec["iterations"], "pair_status": rec["status"],
            "pair_mse": rec["mse"], "pair_nn_queries": rec["nn_queries"]}


def nn_sample(n):
    """Fixed positions of the NN answers --dump-outputs keeps: at most NN_DUMP_SAMPLE of n, seeded, in ascending order."""
    if n <= NN_DUMP_SAMPLE:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, NN_DUMP_SAMPLE, replace=False))


def workload_config(a, world):
    return {
        "workload": "%d-view turntable, %d pts/view, %d ring pairs, %d fixed ICP iterations/pair, point-to-point, "
                    "reciprocal=%d, gate %.1f mm, + host loop closure" % (a.views, a.points, a.views, a.iters, a.reciprocal, a.max_dist),
        "views": a.views, "points_per_view": a.points, "pairs": a.views, "iterations": a.iters,
        "sharding": "pairs block-partitioned over %d rank(s); one NCCL all-gather of per-pair results" % world,
        "l2": "256 MiB scratch buffer rewritten between timed steps (L2 flush)",
    }


def pair_range(rank, world, n_pairs):
    import mvr_b200.ring as ring
    return ring.pair_range(rank, world, n_pairs)


def make_pairs(a, p0, p1):
    """Synthetic scans and initial guesses of pairs [p0, p1): pair p aligns view (p+1)%V onto view p (CPU arm;
    same scans and the same guesses as the native arm's view_init_poses)."""
    import mvr_b200.synth as synth
    V = a.views
    need = sorted({v % V for p in range(p0, p1) for v in (p, p + 1)})
    views, poses = {}, {}
    for v in need:
        views[v], poses[v] = synth.turntable_view(v, V, a.points)
    init = view_init_poses(a, [poses.get(v, synth.view_pose(v, V)) for v in range(V)])
    pairs = []
    for p in range(p0, p1):
        t, s = p % V, (p + 1) % V
        guess = (np.linalg.inv(init[t]) @ init[s]).astype(np.float32)   # ideal turntable step + fixed error
        pairs.append(dict(pair=p, tgt=t, src=s, guess=guess, truth=np.linalg.inv(poses[t]) @ poses[s]))
    return views, pairs


# ------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline (the oracle = port of the reference's PCL path)
# ------------------------------------------------------------------------------------------------
def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def cpu_align_pairs(a, views, pairs, threads=None, iters=None, keep=None):
    """The CPU path on `pairs`: (queries answered, seconds, threads used).  threads = None: every host thread this
    process may use (torchrun exports OMP_NUM_THREADS=1, which would cripple the CPU arm); 1 = the PCL-faithful
    single-threaded figure.  keep (list): receives the oracle's result of every pair (the parity gate reuses it)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    oracle.build()
    oracle.set_num_threads(threads or host_threads())
    prm = oracle.make_params(max_iterations=iters or a.iters, max_dist=a.max_dist, reciprocal=bool(a.reciprocal), fixed_iterations=True)
    t0 = time.perf_counter()
    q = 0
    for pr in pairs:
        o = oracle.icp_align(views[pr["src"]], views[pr["tgt"]], prm, guess=pr["guess"], max_log=max(a.iters, 1))
        q += o["nn_queries"]
        if keep is not None:
            keep.append(o)
    dt = time.perf_counter() - t0
    return q, dt, oracle.num_threads()


def cpu_baseline_block(a, n_pairs, reps, keep=None):
    """cpu_baseline of the JSON line: the oracle port on the first n_pairs ring pairs of the same sequence, all host
    threads (min of `reps`), plus the single-threaded figure (PCL 1.7's ICP is single-threaded) on pair 0 with a third of
    the iterations (min of `reps`) so that the leg stays within ~30 s."""
    V = a.views
    cviews, cpairs = make_pairs(a, 0, n_pairs)
    best = None
    for r in range(max(reps, 1)):
        got = [] if (keep is not None and r == 0) else None
        cq, cdt, cores = cpu_align_pairs(a, cviews, cpairs, keep=got)
        if got is not None:
            keep.extend(got)
        if best is None or cq / cdt > best[0] / best[1]:
            best = (cq, cdt, cores)
    it1 = max(1, a.iters // 3)
    best1 = None
    for r in range(max(reps, 1)):
        q1, dt1, _ = cpu_align_pairs(a, cviews, cpairs[:1], threads=1, iters=it1)
        if best1 is None or q1 / dt1 > best1[0] / best1[1]:
            best1 = (q1, dt1)
    cq, cdt, cores = best
    return {"value": cq / cdt, "unit": UNIT, "cores": cores, "kind": "port", "seconds": cdt, "min_of": max(reps, 1),
            "sample": "first %d pair(s) of the same sequence (%d/%d of a step), %d iterations each" % (n_pairs, n_pairs, V, a.iters),
            "single_thread": {"value": best1[0] / best1[1], "unit": UNIT, "cores": 1, "seconds": best1[1], "min_of": max(reps, 1),
                              "sample": "pair 0, first %d iterations" % it1}}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ns = max(1, min(a.cpu_sample_pairs, a.views))
    views, pairs = make_pairs(a, 0, ns)
    for _ in range(min(a.warmup, 1)):
        cpu_align_pairs(a, views, pairs[:1])
    tq, tt, cores = 0, 0.0, 1
    for _ in range(a.steps):
        last = []
        q, dt, cores = cpu_align_pairs(a, views, pairs, keep=last)
        tq += q
        tt += dt
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"pair_poses": np.stack([o["final"] for o in last]),
                                      **{"pair_" + k: [o[k] for o in last] for k in ("n_corr", "iterations", "status", "mse", "nn_queries")}})
    val = tq / tt
    q1, dt1, _ = cpu_align_pairs(a, views, pairs[:1], threads=1, iters=max(1, a.iters // 3))
    sample = "pairs 0..%d of the sequence (%d/%d of a step), %d iterations, per step" % (ns - 1, ns, a.views, a.iters)
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * tt / a.steps * a.views / ns, "ms_per_step_is": "extrapolated: measured time of %d pair(s) x %d/%d" % (ns, a.views, ns),
        "ms_per_sample": 1e3 * tt / a.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(a, a.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "single_thread": {"value": q1 / dt1, "unit": UNIT, "cores": 1, "sample": "pair 0, first %d iterations" % max(1, a.iters // 3)}},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle port of the reference's PCL ICP path (PCL itself cannot be built here); only the RATE is measured: "
                "ms_per_step extrapolates the sampled pairs to the %d pairs of a step" % a.views,
    }
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)   # a run that fails before stop() must not leave the sampler running
        except OSError:
            self.p = None

    def stop(self, t0=None, t1=None):
        """Summary of the samples taken between wall-clock times t0 and t1 (all samples when None)."""
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.05):
                    continue
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if c[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def view_init_poses(a, poses):
    """Initial pose of every view = its ideal turntable pose, with the fixed perturbation (2 deg about a seeded axis
    + 2 mm, SURVEY.md section 8d) applied to every odd view: each ring pair then starts from a guess that is off by
    that perturbation, and the ring still closes."""
    import mvr_b200.synth as synth
    E = synth.perturbation()
    return [(poses[v] @ E) if (v % 2 == 1) else poses[v].copy() for v in range(a.views)]


def run_native(a):
    import torch
    import torch.distributed as dist
    import mvr_b200
    import mvr_b200.synth as synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    V = a.views
    n = a.points
    p0, p1 = pair_range(rank, world, V)
    need = sorted({v % V for p in range(p0, p1) for v in (p, p + 1)})
    views, poses = {}, {}
    for v in range(V):
        if v in need:
            views[v], poses[v] = synth.turntable_view(v, V, n)
        else:
            poses[v] = synth.view_pose(v, V)
    init = view_init_poses(a, [poses[v] for v in range(V)])
    truth0 = np.linalg.inv(poses[p0 % V]) @ poses[(p0 + 1) % V]
    some = views[need[0]][:, :3]
    obj_radius = 0.5 * float((some.max(axis=0) - some.min(axis=0)).max())

    reg = mvr_b200.Registrator(local, a.streams)   # C++ driver: a.streams GPU contexts, one host thread each
    icp = mvr_b200.default_params(max_iterations=a.iters, max_dist=a.max_dist, reciprocal=a.reciprocal, fixed_iterations=1)
    tp = mvr_b200.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr_b200.RING_PAIRS,
                                   loop_closure=1, lum_iterations=16, pair_begin=p0, pair_end=p1, want_fitness=0)

    d_views = {v: torch.from_numpy(pts).to(dev) for v, pts in views.items()}
    h_views = {v: torch.from_numpy(pts).pin_memory() for v, pts in views.items()}
    dev_list = [(d_views[v].data_ptr(), n) if v in d_views else None for v in range(V)]
    host_list = [h_views[v].numpy() if v in h_views else None for v in range(V)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    import mvr_b200.ring as ring

    # the view descriptors (pointers, sizes, initial poses) are marshalled once; every step passes the same buffers
    bound_dev = reg.bind_views(dev_list, init)
    bound_host = reg.bind_views(host_list, init)

    def step(host_buffers):
        """One registration: this rank's ring pairs through the C++ driver, gather of the per-pair results, host
        loop closure over the whole ring.  Returns (queries of this rank, raw pair reports (numpy records), (absolute
        poses, gathered records))."""
        cposes, reps = reg.register_turntable(bound_host if host_buffers else bound_dev, tp, raw=True)
        q = int(reps["nn_queries"][p0:p1].sum())
        allrec = ring.gather_records(ring.records_from_reports(reps, p0, p1), rank, world, V, dist=dist if world > 1 else None, device=dev)
        if world == 1:   # the driver had every pair and closed the ring itself (Registrator::multiViewRegister): its poses
            abs_poses = cposes
        else:
            abs_poses = ring.close_ring(allrec, synth.PIVOT, obj_radius)
        return q, reps, (abs_poses, allrec)

    def timed(host_buffers, steps):
        tot_ms, tot_q = 0.0, 0
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        last = None
        barrier()
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            e0.record()
            q, reps, abs_poses = step(host_buffers)
            torch.cuda.synchronize()   # the driver's streams are non-blocking: make the closing event cover them
            e1.record()
            e1.synchronize()
            tot_ms += e0.elapsed_time(e1)
            tot_q += q
            last = (reps, abs_poses)
        barrier()
        return tot_ms, tot_q, last

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- device-resident leg (value) ----
    sampler = ClockSampler(local) if rank == 0 else None   # started before the warm-up: nvidia-smi takes a while to come up
    for _ in range(a.warmup):
        step(False)
    l0 = mvr_b200.kernel_launch_count()
    w0 = time.time()
    ms, q, last = timed(False, a.steps)
    w1 = time.time()
    launches = mvr_b200.kernel_launch_count() - l0
    clocks = sampler.stop(w0, w1) if sampler else None
    ms = allmax(ms)
    q = allsum(q)
    launches = allsum(launches)
    value = q / (ms * 1e-3)
    if a.dump_outputs and rank == 0:
        step_poses, allrec = last[1]
        if world == 1:   # the driver's V x 16 column-major poses
            step_poses = step_poses.reshape(-1, 4, 4).transpose(0, 2, 1)
        dump_outputs(a.dump_outputs, registration_outputs(step_poses, allrec))

    # ---- end-to-end leg (host buffers through the C ABI) ----
    e2e = None
    if not a.no_e2e:
        for _ in range(max(1, min(a.warmup, 2))):
            step(True)
        ms_e, q_e, _ = timed(True, a.steps)
        ms_e = allmax(ms_e)
        q_e = allsum(q_e)
        # what the driver copies: every DISTINCT view of the rank's pairs once (Registrator::uploadViews), the initial
        # IcpState of every pair; back: the final IcpState + per-iteration log of every pair, the bounding-box words of
        # every view, and the gathered records
        state_b, log_b = mvr_b200.icp_state_bytes(), mvr_b200.icp_log_record_bytes()
        h2d = allsum(float(len(need) * n * 16 + (p1 - p0) * state_b))
        d2h = allsum(float((p1 - p0) * state_b + (p1 - p0) * 28 + V * ring.REC))   # (the iteration logs stay on the device until asked for)
        e2e = {"value": q_e / (ms_e * 1e-3), "unit": UNIT, "ms_per_step": ms_e / a.steps,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)}

    # ---- roofline of the dominant kernels: one extra untimed step with the library's event bracket around the iterations ----
    # In profiling mode the library finishes every pair's preparation (index builds) first, then records one CUDA event before
    # the first and one after the last iteration launch of the rank's batch (all groups of pairs, which run concurrently on
    # their own streams); every pair report carries its share of that span.
    ctxs = [reg.context(k) for k in range(reg.streams())]
    for c in ctxs:
        c.set_profiling(True)
        c.kernel_stats(reset=True)
    _, preps, _ = step(False)
    iter_ms = float(preps["gpu_ms"][p0:p1].sum())
    st = {}
    for c in ctxs:
        for k, v in c.kernel_stats(reset=True).items():
            d = st.setdefault(k, dict(launches=0, ms=0.0, bytes=0.0, units=0.0))
            for f in d:
                d[f] += v[f]
        c.set_profiling(False)
    roof = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        npairs = p1 - p0
        avg_ms = iter_ms / max(a.iters, 1)                       # one iteration of every pair of the rank
        recip = bool(a.reciprocal)
        bytes_per_launch = npairs * (16.0 * n + 16.0 * n + (52.0 * n if recip else 0.0))     # SURVEY.md section 8d, N = M = n
        ach = bytes_per_launch / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        # the same without the 36 B per source point of the per-iteration source re-index, which the reference's PCL path
        # performs (SURVEY.md section 8d counts it as compulsory) and this implementation avoids with its static index
        lean_bytes = npairs * (24.0 * n + 16.0 * n + (16.0 * n if recip else 0.0))
        ach_lean = lean_bytes / (avg_ms * 1e-3) / 1e9 if avg_ms > 0 else 0.0
        # DRAM traffic of the same launches from the committed ncu --set full capture (cold cache), if it was taken with the
        # same number of pairs
        traffic, traffic_src = None, None
        try:
            import glob, re
            caps = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_icp_fused_ncu_full.txt")))
            if caps:
                m = re.search(r"one iteration of (\d+) pairs\): ([0-9.]+) MB", open(caps[-1]).read())
                if m and int(m.group(1)) == npairs:
                    traffic, traffic_src = float(m.group(2)) * 1e6, os.path.relpath(caps[-1], ROOT) + " (ncu --set full, caches flushed per replay)"
        except OSError:
            pass
        group = max(1, (npairs + 3) // 4)
        roof = {"bound": "hbm", "kernel": "k_icp_forward + k_icp_reverse (one ICP iteration of every pair of the rank: forward search, reciprocal "
                                          "search, estimator sums, solve; a launch pair serves a group of %d pairs, the %d groups run concurrently)"
                                          % (group, (npairs + group - 1) // group),
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                "bytes_per_launch": bytes_per_launch, "avg_launch_us": avg_ms * 1e3, "launches": a.iters,
                "launch_unit": "one iteration of all %d pairs = %d concurrent launch pairs; duration = (CUDA-event span of the iterations) / %d"
                               % (npairs, (npairs + group - 1) // group, a.iters),
                "algorithmic_bytes": "SURVEY.md section 8d, reciprocal fused iteration: 16 N + 16 M + 36 N (source re-index) + 16 N (reverse pass) "
                                     "= 68 N + 16 M per pair and iteration, cell tables not counted",
                "achieved_without_reindex_bytes": ach_lean, "frac_without_reindex_bytes": ach_lean / peak,
                "share_of_step": iter_ms / (ms / a.steps) if ms > 0 else None,
                "pairs_per_launch": group,
                "per_kernel_ms": {k: round(v["ms"], 4) for k, v in st.items() if v["launches"] and k != "corr"},
                "per_kernel_ms_note": "CUDA-event spans of the concurrent groups of pairs, summed (index builds: each group's four launches on its own stream)"}

    # ---- accuracy summary (parity itself lives in tests/) ----
    acc = None
    if rank == 0 and last:
        reps, (abs_poses, _) = last
        if world == 1:   # V x 16 column-major absolute poses of the driver -> relative to view 0
            base_inv = np.linalg.inv(init[0])
            abs_poses = [base_inv @ abs_poses[v].reshape(4, 4).T.astype(np.float64) for v in range(V)]
        r = dict(pose=reps["pose"][p0].reshape(4, 4).T.copy(), mse=float(reps["mse"][p0]), n_corr=int(reps["n_correspondences"][p0]))
        dT = r["pose"].astype(np.float64) @ np.linalg.inv(truth0)
        w = 0.5 * np.array([dT[2, 1] - dT[1, 2], dT[0, 2] - dT[2, 0], dT[1, 0] - dT[0, 1]])
        worst = 0.0
        for v in range(V):
            dA = abs_poses[v].astype(np.float64) @ np.linalg.inv(np.linalg.inv(poses[0]) @ poses[v])
            wv = 0.5 * np.array([dA[2, 1] - dA[1, 2], dA[0, 2] - dA[2, 0], dA[1, 0] - dA[0, 1]])
            worst = max(worst, float(np.arcsin(min(1.0, np.linalg.norm(wv)))))
        acc = {"pair0_rot_err_rad_vs_truth": float(np.arcsin(min(1.0, np.linalg.norm(w)))),
               "pair0_rmse_mm": float(np.sqrt(r["mse"])), "pair0_n_corr": int(r["n_corr"]),
               "worst_abs_rot_err_rad_vs_truth_after_loop_closure": worst}

    cpu, parity, checksum = None, None, None
    if last:
        checksum = ring.pose_checksum(last[1][1])
    if rank == 0 and a.cpu_sample_pairs > 0:
        oracle_results = []
        cpu = cpu_baseline_block(a, min(a.cpu_sample_pairs, V), a.cpu_reps, keep=oracle_results)
        # parity gate (SURVEY.md section 8d): pair 0 of the timed workload against the oracle's align of the same pair --
        # the correspondence count of EVERY iteration, the final pose and the final RMSE
        if p0 == 0 and oracle_results and last:
            o = oracle_results[0]
            c = mvr_b200.Context(local)
            c.set_target(views[0]); c.set_source(views[1 % V])
            g = c.icp_align(icp, guess=(np.linalg.inv(init[0]) @ init[1 % V]).astype(np.float32), n_source=n)
            c.close()
            rep0 = dict(pose=last[0]["pose"][0].reshape(4, 4).T.copy(), n_corr=int(last[0]["n_correspondences"][0]))
            dR = g["final"][:3, :3].astype(np.float64) @ o["final"][:3, :3].astype(np.float64).T
            w = 0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
            tb = o["final"][:3, 3].astype(np.float64)
            worst_it = 0.0
            for x, y in zip(g["log"], o["log"]):
                dd = x["delta"][:3, :3].astype(np.float64) @ y["delta"][:3, :3].astype(np.float64).T
                ww = 0.5 * np.array([dd[2, 1] - dd[1, 2], dd[0, 2] - dd[2, 0], dd[1, 0] - dd[0, 1]])
                worst_it = max(worst_it, float(np.arcsin(min(1.0, np.linalg.norm(ww)))))
            parity = {"against": "CPU oracle, pair 0 of the timed workload, %d iterations" % a.iters,
                      "n_corr_equal": bool([x["n_corr"] for x in g["log"]] == [y["n_corr"] for y in o["log"]]),
                      "nn_queries_equal": bool(g["nn_queries"] == o["nn_queries"]),
                      "rot_rad": float(np.arcsin(min(1.0, np.linalg.norm(w)))),
                      "worst_iteration_rot_rad": worst_it,
                      "trans_rel": float(np.linalg.norm(g["final"][:3, 3].astype(np.float64) - tb) / max(np.linalg.norm(tb), 1e-12)),
                      "rmse_rel": float(abs(np.sqrt(g["mse"]) - np.sqrt(o["mse"])) / np.sqrt(o["mse"])),
                      "timed_pair_bits_equal": bool(np.array_equal(g["final"], rep0["pose"]) and g["n_corr"] == rep0["n_corr"]),
                      "bars": {"rot_rad": 1e-5, "trans_rel": 1e-6, "rmse_rel": 1e-4}}

    if rank == 0:
        cfg = workload_config(a, a.gpus)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "registration_ms": ms / a.steps, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "roofline": roof, "cpu_baseline": cpu, "accuracy": acc, "parity": parity, "pose_checksum": checksum,
            "pairs_per_launch": max(1, (p1 - p0 + 3) // 4),   # mvr_ctx_set_batch_group default: a quarter of the rank's pairs per launch, the groups run concurrently
        }
        print(json.dumps(out))
    reg.close()
    if world > 1:
        dist.destroy_process_group()


def run_single_process(a):
    """--gpus N from one process: the multi-GPU entry point of the C ABI (what a C++ caller such as the reference, itself one
    process, would use).  Same workload, same JSON line; timing = host clock around the call (it returns after the exchange
    and the host loop closure), device time per GPU from CUDA events inside the library."""
    import torch
    import mvr_b200
    import mvr_b200.synth as synth
    import mvr_b200.ring as ring
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback")
    G = a.gpus
    if torch.cuda.device_count() < G:
        raise SystemExit("bench.py: %d GPUs requested, %d visible" % (G, torch.cuda.device_count()))
    V, n = a.views, a.points
    views, poses = synth.turntable_sequence(V, n)
    init = view_init_poses(a, poses)
    hv = [torch.from_numpy(p).pin_memory() for p in views]
    host_list = [t.numpy() for t in hv]
    icp = mvr_b200.default_params(max_iterations=a.iters, max_dist=a.max_dist, reciprocal=a.reciprocal, fixed_iterations=1)
    tp = mvr_b200.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr_b200.RING_PAIRS,
                                   loop_closure=1, lum_iterations=16)
    m = mvr_b200.MultiRegistrator(range(G))
    m.upload(host_list, init)
    flush = [torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % g) for g in range(G)]

    def sync_all():
        for g in range(G):
            torch.cuda.synchronize(g)

    def timed(resident, steps):
        tot, dev_ms, q, last = 0.0, 0.0, 0, None
        for _ in range(steps):
            for f in flush:
                f.fill_(1)
            sync_all()
            t0 = time.perf_counter()
            got, reps, recs, ms = m.register_turntable(host_list, tp, init_poses=init, use_resident=resident)
            tot += (time.perf_counter() - t0) * 1e3
            dev_ms += float(ms.max())
            q += sum(r["nn_queries"] for r in reps)
            last = (got, reps, recs)
        return tot, dev_ms, q, last

    sampler = ClockSampler(0)
    for _ in range(a.warmup):
        m.register_turntable(host_list, tp, init_poses=init, use_resident=True)
    l0 = mvr_b200.kernel_launch_count()
    w0 = time.time()
    ms, dms, q, last = timed(True, a.steps)
    w1 = time.time()
    launches = mvr_b200.kernel_launch_count() - l0
    clocks = sampler.stop(w0, w1)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, registration_outputs(last[0], last[2]))
    e2e = None
    if not a.no_e2e:
        for _ in range(max(1, min(a.warmup, 2))):
            m.register_turntable(host_list, tp, init_poses=init, use_resident=False)
        ms_e, _, q_e, _ = timed(False, a.steps)
        state_b, log_b = mvr_b200.icp_state_bytes(), mvr_b200.icp_log_record_bytes()
        nviews = sum(len(ring.views_needed(*ring.pair_range(r, G, V), V)) for r in range(G))
        e2e = {"value": q_e / (ms_e * 1e-3), "unit": UNIT, "ms_per_step": ms_e / a.steps,
               "h2d_bytes_per_step": int(nviews * n * 16 + V * state_b + V * ring.REC),
               "d2h_bytes_per_step": int(V * (state_b + log_b * a.iters) + nviews * 28 + G * V * ring.REC)}
    got, reps, recs = last
    out = {
        "metric": METRIC, "value": q / (ms * 1e-3), "unit": UNIT, "n_gpus": G, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, G), "registration_ms": ms / a.steps, "device_ms_max_per_step": dms / a.steps, "e2e": e2e,
        "gpu_launches": int(launches), "clocks": clocks, "roofline": None, "cpu_baseline": None,
        "pose_checksum": ring.pose_checksum(recs), "pairs_per_launch": max(1, (-(-V // G) + 3) // 4),
        "launch": "single process: mvr_register_turntable_multi (one host thread per GPU, ncclAllGather of the pair records inside the C ABI)",
    }
    print(json.dumps(out))
    m.close()


NN_METRIC = "nn_queries_per_s (exact 1-NN of N queries vs a 1M-point target grid; ms_per_step = one pass over the queries)"
NN_SIZES = [10_000, 31_600, 100_000, 316_000, 1_000_000, 3_160_000, 10_000_000, 16_000_000]


def nn_config(a):
    return {"workload": "NN-query sweep: %d-point target (full bumpy sphere), queries = target distribution + 0.5 mm noise; headline step = %d "
                        "queries in random order, un-gated exact 1-NN" % (a.nn_target, a.nn_queries),
            "target_points": a.nn_target, "queries": a.nn_queries, "order": "random",
            "l2": "queries + results of the headline step are 384 MB (> 126 MB L2): no flush needed"}


def nn_cpu(a, tgt, q, threads, keep=None):
    """keep (list): receives the answers (indices, d2) of the last repetition."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    oracle.build()
    oracle.set_num_threads(threads)
    tree = oracle.KdTree(tgt)
    best = None
    for _ in range(max(a.cpu_reps, 1)):
        t0 = time.perf_counter()
        ans = tree.query(q)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    if keep is not None:
        keep.extend(ans)
    return len(q) / best, best, oracle.num_threads()


def run_nn_reference(a):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import mvr_b200.synth as synth
    ns = min(a.nn_queries, 2_000_000)
    tgt, q = synth.nn_sweep_case(a.nn_target, ns, order="random")
    last = []
    val, sec, cores = nn_cpu(a, tgt, q, host_threads(), keep=last)
    if a.dump_outputs:
        sel = nn_sample(ns)
        dump_outputs(a.dump_outputs, {"query_index": sel, "nn_index": last[0][sel], "nn_d2": last[1][sel]})
    v1, s1, _ = nn_cpu(a, tgt, q[:200_000], 1)
    print(json.dumps({
        "impl": "reference", "metric": NN_METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * a.nn_queries / val, "ms_per_step_is": "extrapolated from the sampled rate", "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": nn_config(a),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "seconds": sec, "min_of": max(a.cpu_reps, 1),
                         "sample": "first %d queries of the headline step (kd-tree build excluded)" % ns,
                         "single_thread": {"value": v1, "unit": UNIT, "cores": 1, "seconds": s1, "sample": "first 200000 queries"}},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the oracle's exact kd-tree 1-NN (FLANN's role in the reference's PCL path), OpenMP over the queries"}))


def run_nn_sweep(a):
    """BASELINE configs[4]: exact NN-query throughput against a 1M-point target, 10k .. 16M queries in random and in cell-sorted
    order.  The headline step is the largest random-order batch; every GPU of a multi-GPU run answers its own share of the
    queries against a replicated index (no collective: "scaling": "weak" per GPU is not used -- total work is fixed)."""
    import torch
    import torch.distributed as dist
    import mvr_b200
    import mvr_b200.synth as synth
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = mvr_b200.Context(local)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)   # CUDA events of torch then bracket the library's work
    m = a.nn_target
    tgt, qall = synth.nn_sweep_case(m, a.nn_queries, order="random")
    ctx.set_target(tgt)
    lo, hi = (rank * a.nn_queries) // world, ((rank + 1) * a.nn_queries) // world
    q = qall[lo:hi]
    nq = len(q)
    dq = torch.from_numpy(q).to(dev)
    hq = torch.from_numpy(q).pin_memory()
    di = torch.empty(nq, dtype=torch.int32, device=dev); dd = torch.empty(nq, dtype=torch.float32, device=dev)
    hi_ = np.empty(nq, dtype=np.int32); hd = np.empty(nq, dtype=np.float32)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(steps, host):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        tot = 0.0
        barrier()
        for _ in range(steps):
            e0.record()
            if host:
                i2, d2 = ctx.nn_query(hq.numpy())
            else:
                ctx.nn_query_device(dq.data_ptr(), nq, di.data_ptr(), dd.data_ptr())
            e1.record(); e1.synchronize()
            tot += e0.elapsed_time(e1)
        barrier()
        return tot

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(a.warmup):
        ctx.nn_query_device(dq.data_ptr(), nq, di.data_ptr(), dd.data_ptr())
    torch.cuda.synchronize()
    l0 = mvr_b200.kernel_launch_count()
    w0 = time.time()
    ms = allmax(timed(a.steps, False))
    w1 = time.time()
    launches = mvr_b200.kernel_launch_count() - l0
    clocks = sampler.stop(w0, w1) if sampler else None
    value = a.nn_queries * a.steps / (ms * 1e-3)
    if a.dump_outputs and rank == 0:   # rank 0's share of the queries (under torchrun), sampled
        sel = nn_sample(nq)
        ts = torch.from_numpy(sel).to(dev)
        dump_outputs(a.dump_outputs, {"query_index": sel, "nn_index": di[ts].cpu().numpy(), "nn_d2": dd[ts].cpu().numpy()})
    e2e = None
    if not a.no_e2e:
        timed(1, True)
        ms_e = allmax(timed(max(1, a.steps // 2), True))
        e2e = {"value": a.nn_queries * max(1, a.steps // 2) / (ms_e * 1e-3), "unit": UNIT, "ms_per_step": ms_e / max(1, a.steps // 2),
               "h2d_bytes_per_step": int(a.nn_queries * 16), "d2h_bytes_per_step": int(a.nn_queries * 8)}
    # ---- roofline of the NN kernel (per-kernel CUDA events inside the library) + the sweep over batch sizes (rank 0)
    roof, sweep, parity, cpu = None, None, None, None
    if rank == 0:
        ctx.set_profiling(True)
        ctx.kernel_stats(reset=True)
        ctx.nn_query_device(dq.data_ptr(), nq, di.data_ptr(), dd.data_ptr()); ctx.synchronize()
        st = ctx.kernel_stats(reset=True)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        nn = st["nn"]
        ach = nn["bytes"] / (nn["ms"] * 1e-3) / 1e9 if nn["ms"] > 0 else 0.0
        tot_ms = sum(v["ms"] for v in st.values())
        roof = {"bound": "hbm", "kernel": "k_cell_nn (exact 1-NN of cell-sorted queries, warp-cooperative)" if nq >= 8 * m else "k_warp_nn (one warp per query)",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
                "bytes_per_launch": nn["bytes"] / max(nn["launches"], 1), "avg_launch_us": 1e3 * nn["ms"] / max(nn["launches"], 1),
                "algorithmic_bytes": "24 B per query + 16 B per target point", "share_of_kernel_time": nn["ms"] / tot_ms if tot_ms > 0 else None,
                "per_kernel_ms": {k: round(v["ms"], 4) for k, v in st.items() if v["launches"]}}
        ctx.set_profiling(False)
        sweep = []
        for order in ("random", "morton"):
            _, qo = synth.nn_sweep_case(m, a.nn_queries, order=order) if order == "morton" else (None, qall)
            dqo = torch.from_numpy(qo).to(dev)
            for n1 in [s_ for s_ in NN_SIZES if s_ <= a.nn_queries]:
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                best = None
                for rep in range(4):
                    e0.record()
                    ctx.nn_query_device(dqo.data_ptr(), n1, di.data_ptr(), dd.data_ptr())
                    e1.record(); e1.synchronize()
                    t = e0.elapsed_time(e1)
                    best = t if (best is None or (rep > 0 and t < best)) else best
                sweep.append({"queries": n1, "order": order, "ms": best, "gqps": n1 / best / 1e6})
            del dqo
        # parity gate: the first 200k answers of the headline step against the oracle's kd-tree, bit for bit
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle
        oracle.build()
        ctx.nn_query_device(dq.data_ptr(), nq, di.data_ptr(), dd.data_ptr()); ctx.synchronize()
        ns = min(nq, 200_000)
        oi, od = oracle.nn_kdtree(tgt, q[:ns])
        parity = {"against": "CPU oracle kd-tree, first %d queries of the headline step" % ns,
                  "indices_equal": bool(np.array_equal(di[:ns].cpu().numpy(), oi)),
                  "d2_bits_equal": bool(np.array_equal(dd[:ns].cpu().numpy().view(np.uint32), od.view(np.uint32)))}
        if a.cpu_sample_pairs > 0:
            ncs = min(nq, 2_000_000)
            val, sec, cores = nn_cpu(a, tgt, q[:ncs], host_threads())
            v1, s1, _ = nn_cpu(a, tgt, q[:200_000], 1)
            cpu = {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "seconds": sec, "min_of": max(a.cpu_reps, 1),
                   "sample": "first %d queries of the headline step (kd-tree build excluded)" % ncs,
                   "single_thread": {"value": v1, "unit": UNIT, "cores": 1, "seconds": s1, "sample": "first 200000 queries"}}
        print(json.dumps({
            "metric": NN_METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": nn_config(a),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "parity": parity, "sweep": sweep}))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse_args()
    if a.workload == "nn_sweep":
        return run_nn_reference(a) if a.impl == "reference" else run_nn_sweep(a)
    if a.impl == "reference":
        run_reference(a)
    elif a.single_process or (a.gpus > 1 and "WORLD_SIZE" not in os.environ):
        run_single_process(a)
    else:
        run_native(a)


if __name__ == "__main__":
    main()
