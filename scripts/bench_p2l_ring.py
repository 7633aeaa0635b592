#!/usr/bin/env python
"""Point-to-point vs point-to-plane vs symmetric point-to-plane turntable ring registration on one GPU (DESIGN.md section 7).

Workload: 24 views x 200k points (synth.turntable_sequence), scans resident on the device, reciprocal correspondences, max_dist 4,
loop closure on, the bench's initial guesses (ideal turntable pose, the fixed perturbation on every odd view).  In one process,
after a warm-up, the three estimators alternate; the script reports

  ring_ms        ms per register_turntable call (30 fixed iterations; host clock around the call and a device synchronise,
                 L2 overwritten before each call), median and spread over --steps calls per estimator
  normals        device time of the batched target normals (MVR_K_NORMALS and the index builds, MVR_K_SORT, of one
                 mvr_estimate_normals_batch over the 24 views) against 24 mvr_estimate_normals calls, and both as wall time
  accuracy       per estimator: max and median pair rotation error against the synthetic truth, and the absolute-pose error
                 after the loop closure (max over views)
  iterations     with the reference's criteria (transformation_epsilon 1e-6, fixed_iterations 0, at most 100 iterations): the
                 iterations each pair needs, and the registration time

It writes <out>/bench_p2l_ring.json, with the GPU's name and power limit read in the same run.

  python scripts/bench_p2l_ring.py --out /tmp/p2l_ring
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def rot_angle(A, B):
    R = np.asarray(A, dtype=np.float64)[:3, :3] @ np.asarray(B, dtype=np.float64)[:3, :3].T
    w = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(np.arcsin(min(1.0, np.linalg.norm(w))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:   # the numbers are still device-timed; the label says what could not be read
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit="not read (%s)" % e)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory the JSON result is written to")
    ap.add_argument("--views", type=int, default=24)
    ap.add_argument("--points", type=int, default=200_000)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--steps", type=int, default=10, help="timed registrations per estimator")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--normal-k", type=int, default=16)
    a = ap.parse_args()

    import torch
    import mvr_b200 as mvr
    import mvr_b200.synth as synth
    if not torch.cuda.is_available():
        raise SystemExit("bench_p2l_ring.py: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    V, n = a.views, a.points
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    d_views = [torch.from_numpy(v).to(dev) for v in views]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # 2 x the 126 MB L2
    torch.cuda.synchronize()
    res = dict(gpu=gpu_info(), workload=dict(views=V, points=n, reciprocal=1, max_dist=4.0, loop_closure=1, normal_k=a.normal_k,
                                             fixed_iterations=a.iters, steps=a.steps, warmup=a.warmup, l2="overwritten before each timed call"))

    reg = mvr.Registrator(0, 1)
    bound = reg.bind_views([(t.data_ptr(), n) for t in d_views], init)
    names = {mvr.POINT_TO_POINT: "point_to_point", mvr.POINT_TO_PLANE: "point_to_plane", mvr.SYMMETRIC: "symmetric"}

    def params(est, fixed=True, max_iterations=None, eps=0.0):
        icp = mvr.default_params(max_iterations=max_iterations or a.iters, max_dist=4.0, reciprocal=1, fixed_iterations=1 if fixed else 0,
                                 estimator=est, transformation_epsilon=eps)
        return mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1,
                                    normal_k=a.normal_k)

    def run(tp):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P, rep = reg.register_turntable(bound, tp)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, P, rep

    # ---- ring time, the estimators alternating ----
    fixed = {e: params(e) for e in names}
    for _ in range(a.warmup):
        for e in names:
            run(fixed[e])
    times = {e: [] for e in names}
    last = {}
    for _ in range(a.steps):
        for e in names:
            ms, P, rep = run(fixed[e])
            times[e].append(ms)
            last[e] = (P, rep)
    res["ring_ms"] = {names[e]: dict(median=float(np.median(t)), min=float(np.min(t)), max=float(np.max(t)), all=[round(x, 3) for x in t])
                      for e, t in times.items()}

    def accuracy(P, rep):
        pair = [rot_angle(rep[p]["pose"], np.linalg.inv(poses[p]) @ poses[(p + 1) % V]) for p in range(V)]
        absr = [rot_angle(np.linalg.inv(P[0]) @ P[v], np.linalg.inv(poses[0]) @ poses[v]) for v in range(V)]
        abst = [float(np.linalg.norm((np.linalg.inv(P[0].astype(np.float64)) @ P[v])[:3, 3] - (np.linalg.inv(poses[0]) @ poses[v])[:3, 3]))
                for v in range(V)]
        return dict(pair_rot_max=max(pair), pair_rot_median=float(np.median(pair)), abs_rot_max=max(absr), abs_trans_max_mm=max(abst),
                    statuses=sorted({int(r["status"]) for r in rep}), iterations=sorted({int(r["iterations"]) for r in rep}))
    res["accuracy_fixed"] = {names[e]: accuracy(*last[e]) for e in names}

    # ---- normals: one batch against 24 single calls ----
    ctxs = [mvr.Context(0) for _ in range(V)]
    for c, t in zip(ctxs, d_views):
        c.set_target_device(t.data_ptr(), n, keepalive=t)
    for _ in range(2):
        mvr.estimate_normals_batch(ctxs, a.normal_k)
        for c in ctxs:
            c.estimate_normals(mvr.TARGET, n, a.normal_k)
    torch.cuda.synchronize()
    reps = 10
    for c in ctxs:
        c.set_profiling(True)
        c.kernel_stats(reset=True)
    wall_b = []
    for _ in range(reps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mvr.estimate_normals_batch(ctxs, a.normal_k)
        ctxs[0].synchronize()
        wall_b.append((time.perf_counter() - t0) * 1e3)
    sb = ctxs[0].kernel_stats(reset=True)
    wall_l = []
    for _ in range(reps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for c in ctxs:
            c.estimate_normals(mvr.TARGET, n, a.normal_k)
        wall_l.append((time.perf_counter() - t0) * 1e3)
    sl = [c.kernel_stats(reset=True) for c in ctxs]
    res["normals"] = dict(
        batch=dict(normals_kernel_ms=sb["normals"]["ms"] / reps, launches_per_call=sb["normals"]["launches"] / reps,
                   build_ms=sb["sort"]["ms"] / reps, wall_ms_median=float(np.median(wall_b))),
        loop_of_single_calls=dict(normals_kernel_ms=sum(s["normals"]["ms"] for s in sl) / reps,
                                  launches_per_call=sum(s["normals"]["launches"] for s in sl) / reps,
                                  build_ms=sum(s["sort"]["ms"] for s in sl) / reps, wall_ms_median=float(np.median(wall_l))),
        note="kernel ms: CUDA events around each normals launch; build ms: the index builds (MVR_K_SORT); wall: host clock incl. synchronise")
    for c in ctxs:
        c.set_profiling(False)
        c.close()

    # ---- the reference's criteria: transformation_epsilon 1e-6, no fixed count, at most 100 iterations ----
    conv = {}
    for e in names:
        tp = params(e, fixed=False, max_iterations=100, eps=1e-6)
        run(tp)
        ms, P, rep = run(tp)
        it = [int(r["iterations"]) for r in rep]
        conv[names[e]] = dict(ring_ms=ms, iterations_median=float(np.median(it)), iterations_max=max(it), iterations_min=min(it),
                              iterations=it, accuracy=accuracy(P, rep))
    res["reference_criteria"] = conv
    reg.close()

    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, "bench_p2l_ring.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"], ring_ms={k: v["median"] for k, v in res["ring_ms"].items()}, normals=res["normals"],
                          accuracy=res["accuracy_fixed"], iterations={k: (v["iterations_median"], v["iterations_max"]) for k, v in conv.items()})))


if __name__ == "__main__":
    main()
