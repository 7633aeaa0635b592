#!/usr/bin/env python
"""Turntable ring registration from uneven table steps, with and without the angle search (DESIGN.md section 7).

Workload: 24 views x 200k points (synth.turntable_sequence), scans resident on the device, reciprocal correspondences, max_dist 4,
30 fixed iterations, loop closure on.  View v was scanned after the table turned by v * 15 degrees + e_v, e_v seeded and uniform
in +-J degrees (view 0: none) for J in --errors; the driver starts from the ideal turntable poses.  For point-to-point and
point-to-plane, with the search off and on (+-15 degrees around each guess in 1-degree steps, 4096 samples), the script reports

  pair_rot_median / max   pair rotation error against the synthetic truth (rad)
  pairs_off               pairs whose rotation error exceeds 1e-2 rad
  picked_off_by_deg       search on: the largest gap between a pair's chosen turn and its true step error (degrees)
  ring_ms                 host clock around register_turntable and a device synchronise (L2 overwritten before), median
  search_ms               the scorer alone on the 24 pairs (mvr_score_guesses_batch with its target indices built): host clock
                          around the call, which returns when the sums are on the host; and its kernel time (CUDA events)

It writes <out>/bench_angle_search.json with the GPU's name and power limit read in the same run.

  python scripts/bench_angle_search.py --out /tmp/angle_search
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
    ap.add_argument("--errors", default="0,2,4,6,8", help="step-angle error amplitudes J (degrees)")
    ap.add_argument("--steps", type=int, default=5, help="timed calls per configuration")
    ap.add_argument("--range-deg", type=float, default=15.0)
    ap.add_argument("--step-deg", type=float, default=1.0)
    ap.add_argument("--samples", type=int, default=4096)
    ap.add_argument("--scorer-only", action="store_true", help="skip the ring registrations (A/B of scorer builds)")
    a = ap.parse_args()

    import torch
    import mvr_b200 as mvr
    import mvr_b200.synth as synth
    if not torch.cuda.is_available():
        raise SystemExit("bench_angle_search.py: no CUDA device (there is no CPU fallback)")
    dev = torch.device("cuda", 0)
    V, n = a.views, a.points
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # 2 x the 126 MB L2
    res = dict(gpu=gpu_info(), workload=dict(views=V, points=n, reciprocal=1, max_dist=4.0, loop_closure=1, fixed_iterations=a.iters,
                                             search=dict(range_deg=a.range_deg, step_deg=a.step_deg, samples=a.samples), steps=a.steps,
                                             l2="overwritten before each timed ring call"), runs=[])
    names = {mvr.POINT_TO_POINT: "point_to_point", mvr.POINT_TO_PLANE: "point_to_plane"}

    def params(est):
        icp = mvr.default_params(max_iterations=a.iters, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=est)
        return mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1)

    for J in [float(x) for x in a.errors.split(",")]:
        err = synth.step_errors(V, J)
        views, poses = synth.turntable_sequence(V, n, angles=synth.uneven_angles(V, J))
        d_views = [torch.from_numpy(v).to(dev) for v in views]
        torch.cuda.synchronize()
        reg = mvr.Registrator(0, 1)
        bound = reg.bind_views([(t.data_ptr(), n) for t in d_views])
        entry = dict(error_deg=J, max_relative_step_error_deg=float(np.rad2deg(np.abs(err - np.roll(err, -1)).max())), estimators={})
        for est, name in ([] if a.scorer_only else names.items()):
            tp = params(est)
            out = {}
            for on in (False, True):
                reg.set_angle_search(np.deg2rad(a.range_deg) if on else 0.0, np.deg2rad(a.step_deg), a.samples)
                reg.register_turntable(bound, tp)   # warm-up
                times = []
                for _ in range(a.steps):
                    flush.fill_(1)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    _, rep = reg.register_turntable(bound, tp)
                    torch.cuda.synchronize()
                    times.append((time.perf_counter() - t0) * 1e3)
                e = np.array([rot_angle(rep[p]["pose"], np.linalg.inv(poses[p]) @ poses[(p + 1) % V]) for p in range(V)])
                r = dict(pair_rot_median=float(np.median(e)), pair_rot_max=float(e.max()), pairs_off=int((e > 1e-2).sum()),
                         statuses=sorted({int(x["status"]) for x in rep}), ring_ms=float(np.median(times)), ring_ms_all=[round(x, 3) for x in times])
                if on:
                    log = reg.angle_search_log()
                    r["picked_off_by_deg"] = float(max(abs(np.rad2deg(x["angle"] - (err[x["pair"]] - err[(x["pair"] + 1) % V]))) for x in log))
                    r["choices"] = [int(x["choice"]) for x in log]
                out["search_on" if on else "search_off"] = r
            entry["estimators"][name] = out
        # the scorer alone: the 24 pairs of the ring, their 2J+1 candidates, target indices already built by the first call
        cs = [mvr.Context(0) for _ in range(V)]
        for p, c in enumerate(cs):
            c.set_target_device(d_views[p].data_ptr(), n, keepalive=d_views[p])
            c.set_source_device(d_views[(p + 1) % V].data_ptr(), n, keepalive=d_views[(p + 1) % V])
        Jc = int(round(a.range_deg / a.step_deg))
        init = [np.eye(4)] + [mvr.turntable_rotation(synth.PIVOT, synth.AXIS, mvr.turntable_view_angle(v, V)) for v in range(1, V)]
        cands = np.stack([np.stack([(np.linalg.inv(init[p]) @ synth.rotation_about_axis(np.deg2rad(j * a.step_deg)) @ init[(p + 1) % V])
                                    .astype(np.float32) for j in range(-Jc, Jc + 1)]) for p in range(V)])
        mvr.score_guesses_batch(cs, cands, 4.0, a.samples)
        cs[0].set_profiling(True)
        cs[0].kernel_stats(reset=True)
        wall = []
        for _ in range(max(a.steps, 10)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mvr.score_guesses_batch(cs, cands, 4.0, a.samples)
            wall.append((time.perf_counter() - t0) * 1e3)
        st = cs[0].kernel_stats(reset=True)["nn"]
        entry["search_ms"] = dict(call_median=float(np.median(wall)), kernel_ms=st["ms"] / max(st["launches"], 1), launches=st["launches"],
                                  queries=st["units"] / max(st["launches"], 1))
        for c in cs:
            c.set_profiling(False)
            c.close()
        reg.close()
        res["runs"].append(entry)
        print(json.dumps(dict(error_deg=J, search_ms=entry["search_ms"],
                              **{k: {s: {x: v[s][x] for x in ("pair_rot_median", "pair_rot_max", "pairs_off", "ring_ms")} for s in v}
                                 for k, v in entry["estimators"].items()})), flush=True)
        del d_views

    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, "bench_angle_search.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res["gpu"], written=path)))


if __name__ == "__main__":
    main()
