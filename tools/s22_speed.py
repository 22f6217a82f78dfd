#!/usr/bin/env python
"""What |S22| specs cost on the GPU, in one call.

  (a) an |S22| job against the |S11| job on the reversed cascade (config 2 at 1e6 x 4096, the 100 -> 50 Ohm GPSDO filter at
      1e6 x 4096): the planner runs the first as the second, so both should take the same kernel and the same time;
  (b) the same |S22| jobs on the direct route: the opcode interpreter (QO100NET_KERNEL=interp) and the compiled chain kernel
      (QO100NET_KERNEL=interp QO100NET_CHAIN=jit);
  (c) with --parent-lib, the kernels whose code the |S22| work touched on jobs they already served -- config 2 on the
      interpreter, config 3 on the microstrip board kernel, the bench's chain-kernel jobs -- against that library (a build of
      the previous commit), each in a process of its own.
Every comparison alternates its contenders --rounds times and reports each round, so the spread is visible next to the
difference.  Times are host clocks around a launch and the read that synchronises it, after a warm-up launch of the same plan.

  python tools/s22_speed.py [--rounds 3] [--parent-lib path/libqo100net.so] [--out s22_speed.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "qo-100-tools_b200", "python"))
sys.path.insert(0, ROOT)
ENV_KEYS = ("QO100NET_KERNEL", "QO100NET_CHAIN", "QO100NET_USTRIP")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def timed(Q, ctx, net, f, specs, tols, n, env, hist, seed=3):
    """seconds of one n-sample launch of the job (plan made and warmed up first), its kernel and counters"""
    for k in ENV_KEYS:
        os.environ.pop(k, None)
    os.environ.update(env)
    try:
        p = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **hist)
        p.launch(10 ** 9, 8192)
        p.read()
        p.reset()
        t0 = time.perf_counter()
        p.launch(0, n)
        r = p.read()
        dt = time.perf_counter() - t0
        out = dict(seconds=dt, evals_per_s=n * len(f) / dt, kernel=p.kernel_name, n_pass=int(r["n_pass"]),
                   fail_per_spec=[int(x) for x in r["fail_per_spec"]], hist=[int(x) for x in r["hist"]])
        p.close()
    finally:
        for k in ENV_KEYS:
            os.environ.pop(k, None)
    return out


def s22_jobs(Q, W, ctx):
    """(name, net, grid, tols, |S22| specs, histogram) for (a) and (b); limits from a FULL_S pre-run so that the yield is not 0 or 1"""
    out = []
    w2 = W.cfg2()
    _n, g10, fc = W.gpsdo_bank()[0]
    for name, net, f, tols, band, s21 in (("cfg2", w2.net, w2.f, w2.tols, (w2.f[0], 9.5e6), w2.specs[0]),
                                          ("gpsdo10M", g10, Q.grid_log(fc / 2.5, fc * 6.25, 4096), Q.lc_tolerances(g10, 0.05, 0.05),
                                           (fc / 2.5, 0.9 * fc), (Q.SPEC_S21_MAX_DB, 2 * fc, 1e99, -30.0))):
        s = ctx.mc_run(net, f, [], 11, 256, tols, mode=Q.MODE_FULL_S)["s"][3]
        m = (f >= band[0]) & (f <= band[1])
        lim = float(np.quantile(20 * np.log10(np.abs(s[:, m])).max(axis=1), 0.45))
        specs = [s21, (Q.SPEC_S22_MAX_DB, band[0], band[1], lim)]
        out.append((name, net, f, tols, specs, dict(hist_bins=256, hist_spec=1, hist_lo=lim - 8.0, hist_hi=lim + 8.0)))
    return out


def reversed_job(Q, net, specs, tols):
    rs, rl = net.terminations
    n = len(net.elements)
    rnet = Q.Net.from_elements(list(reversed(net.elements)), rl, rs)
    return (rnet, [(Q.SPEC_S11_MAX_DB if s[0] == Q.SPEC_S22_MAX_DB else s[0],) + tuple(s[1:]) for s in specs],
            [(n - 1 - e, p, v, m, t) for (e, p, v, m, t) in tols])


def compare(rounds, contenders):
    """contenders: {label: () -> timed dict}, run alternately; per label the rounds' rates and the counters' agreement"""
    rows = {k: [] for k in contenders}
    for _ in range(rounds):
        for k, fn in contenders.items():
            rows[k].append(fn())
    out = {}
    first = None
    for k, rs in rows.items():
        rates = [r["evals_per_s"] for r in rs]
        out[k] = dict(kernel=rs[0]["kernel"], evals_per_s=rates, median=float(np.median(rates)),
                      spread=float((max(rates) - min(rates)) / np.median(rates)))
        c = (rs[0]["n_pass"], rs[0]["fail_per_spec"], rs[0]["hist"])
        first = first or c
        out[k]["counters_equal_first"] = c == first
    return out


def child(lib, samples):
    """(c), one library: the jobs of the touched kernels that existed before |S22| specs"""
    import qo100net as Q
    Q.LIB_PATH = lib
    import torch
    from qo100net import workloads as W
    from tools.chain_jit_speed import measure
    ctx = Q.Context(device=0)
    out = {}
    w2 = W.cfg2()
    r = timed(Q, ctx, w2.net, w2.f, w2.specs, w2.tols, samples, {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "interp"}, w2.hist)
    out["cfg2 interpreter"] = r
    w3 = W.cfg3()
    out["cfg3 board"] = timed(Q, ctx, w3.net, w3.f, w3.specs, w3.tols, 10 * samples, {}, w3.hist)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    for name, row in measure(Q, torch, ctx, stream, samples=100000, fs_samples=8192, modes=("jit",)).items():
        out["chain_jit: " + name] = dict(kernel=row["jit"]["kernel"], evals_per_s=row["jit"]["evals_per_s"])
    ctx.close()
    print("S22SPEED " + json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--child", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.child:
        return child(a.child, a.samples)
    import qo100net as Q
    from qo100net import workloads as W
    ctx = Q.Context(device=0)
    out = {"card": card(), "samples": a.samples, "rounds": a.rounds}
    for name, net, f, tols, specs, hist in s22_jobs(Q, W, ctx):
        rnet, rspecs, rtols = reversed_job(Q, net, specs, tols)
        n = a.samples
        out[name] = compare(a.rounds, {
            "|S22| job": lambda: timed(Q, ctx, net, f, specs, tols, n, {}, hist),
            "|S11| job on the reversed cascade": lambda: timed(Q, ctx, rnet, f, rspecs, rtols, n, {}, hist),
            "|S22| direct, interpreter": lambda: timed(Q, ctx, net, f, specs, tols, n, {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "interp"}, hist),
            "|S22| direct, compiled chain kernel": lambda: timed(Q, ctx, net, f, specs, tols, n, {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "jit"}, hist)})
    ctx.close()
    if a.parent_lib:
        libs = {"this build": os.path.join(ROOT, "qo-100-tools_b200", "lib", "libqo100net.so"), "parent build": os.path.abspath(a.parent_lib)}
        runs = {k: [] for k in libs}
        for _ in range(a.rounds):
            for k, lib in libs.items():
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", lib, "--samples", str(a.samples)],
                                   capture_output=True, text=True)
                line = [ln for ln in p.stdout.splitlines() if ln.startswith("S22SPEED ")]
                if p.returncode or not line:
                    raise RuntimeError("child on %s failed:\n%s" % (lib, p.stderr[-2000:]))
                runs[k].append(json.loads(line[0][9:]))
        cmp_ = {}
        for job in runs["this build"][0]:
            row = {}
            for k in libs:
                rates = [r[job]["evals_per_s"] for r in runs[k]]
                row[k] = dict(kernel=runs[k][0][job]["kernel"], evals_per_s=rates, median=float(np.median(rates)),
                              spread=float((max(rates) - min(rates)) / np.median(rates)))
            row["ratio_of_medians"] = row["this build"]["median"] / row["parent build"]["median"]
            cmp_[job] = row
        out["touched kernels against the parent build"] = cmp_
    print(json.dumps(out, indent=1))
    if a.out:
        open(a.out, "w").write(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
