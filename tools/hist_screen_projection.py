#!/usr/bin/env python
"""Host-only projection of the thread-per-sample kernel's histogram screen (qo_ts.cuh) on config 2.

The screen walks a group of points exactly only when some lane of the warp cannot rule out that a point of the group raises its
tracker.  What that costs is the fraction of 32-sample warp-groups that take the exact path over the screened runs.  This
script takes the CPU oracle's |S21| of config 2's own sample stream (FULL_S planes), the plan's seed and screened runs
(qo_plan_analyze_ts_runs / _ts_screen), and replays the kernel's decisions in the same order: the seeds set the tracker, then
per batch of QO_TS_FG2 = 3 groups (12 points) a lane needs the exact path where some v = 1 / |S21|^2 reaches m = tracker
(1 - eps), a run's last groups short of a whole batch go exactly, and the exact path moves m (at most QO_TS_SCREEN_CAP
times).  Exact values stand in for the kernel's computed ones: a relative eps of 1e-6 is far above either's error.  It also
counts the whole batches that go exactly on the sign test (not the runs' partial last batches) and the updates of m: with
QO100NET_TS_HIST_SEEDS=low (the band's lowest group as the only seed) both are non-zero.

  python tools/hist_screen_projection.py [--samples 10000] [--out FILE]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "qo-100-tools_b200", "python"))
sys.path.insert(0, ROOT)

CAP = 8          # qo_tf_launch.h: QO_TS_SCREEN_CAP
BATCH = 3        # qo_ts.cuh: QO_TS_FG2 groups screened at once


def project(samples=10000, chunk=512):
    import qo100net as Q
    from qo100net import workloads as W
    from oracle import refbind as R
    w = W.cfg2(n_samples=samples)
    scr = Q.plan_ts_screen(w.net, w.f, w.specs, w.tols, **w.hist)
    runs = Q.plan_ts_runs(w.net, w.f, w.specs, w.tols, **w.hist)
    if not scr["screened"]:
        raise SystemExit("config 2's plan does not screen: %s" % scr["reason"])
    eps = scr["eps"]
    seeds = runs[:scr["seeds"]]
    band = [r for r in runs[scr["seeds"]:] if not r["fused"] and r["any"] == r["all"] == 1 << w.hist["hist_spec"]]
    gpt = 4
    rs, rl = w.net.terminations
    el = R.make_elems(w.net.elements)
    exact = total = sign_exact = updates = 0
    lanes_exact = 0
    for a in range(0, samples, chunk):
        cfg = R.mc_cfg(w.seed, min(chunk, samples - a), w.tols, sample_offset=a)
        s21 = R.mc_run(el, rs, rl, w.f, [], cfg, full_s=True, nthreads=R.max_threads())["s"][1]
        v = 1.0 / np.abs(s21) ** 2                                         # the tracked value up to a constant factor
        for b in range(0, v.shape[0] - 31, 32):
            vw = v[b:b + 32]
            m = np.max(np.concatenate([vw[:, r["point"]:r["point"] + gpt] for r in seeds], axis=1), axis=1)
            mh = m * (1 - eps)
            nup = np.zeros(32, dtype=int)
            for r in band:
                end = r["point"] + r["points"]
                for g in range(r["point"], end, BATCH * gpt):
                    ng = min(BATCH, (end - g) // gpt)
                    vg = vw[:, g:g + ng * gpt]
                    need = (vg >= mh[:, None]).any(axis=1) | (ng < BATCH)
                    total += ng
                    if need.any():
                        exact += ng
                        sign_exact += ng == BATCH
                        lanes_exact += int(need.sum()) * ng
                        for q in range(ng):                    # group by group, as the kernel's exact path moves m
                            gm = vg[:, q * gpt:(q + 1) * gpt].max(axis=1)
                            up = (gm > m) & (nup < CAP)
                            m = np.maximum(m, gm)
                            mh = np.where(up, m * (1 - eps), mh)
                            nup += up
                            updates += int(up.sum())
    return dict(workload=w.name, samples=samples, eps=eps, seeds=[r["point"] for r in seeds],
                screened_points=sum(r["points"] for r in band), warp_groups=total,
                exact_fraction=exact / total, lane_exact_fraction=lanes_exact / (32.0 * total), sign_exact_batches=sign_exact,
                updates=updates)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=10000)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    res = project(a.samples)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
