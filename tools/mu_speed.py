#!/usr/bin/env python
"""Speed of stability (mu) specs (GPU box): the padded 20 W driver (tests/test_mu_spec.py::padded_driver, +-10 % on the four pad
resistors), 1e6 samples x 4096 points on 20 MHz - 9 GHz, on the interpreter (QO100NET_CHAIN=interp) and the compiled chain kernel
(QO100NET_CHAIN=jit), each against the same job with |S21| + |S11| specs instead.  Host clock around launch + read (read
synchronises), after one warm-up launch that also compiles the chain kernel; best and median of --reps.  The card's name and power
limit are read in the same run.

   python tools/mu_speed.py [--samples 1000000] [--reps 3] [--out mu_speed.json]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1000000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import qo100net as Q
    from test_mu_spec import PAD_TOLS, SPEC_MU_MIN, padded_driver
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    ctx = Q.Context(device=0)
    net, f = padded_driver(Q), Q.grid_lin(20e6, 9e9, 4096)
    band = (2.3e9, 2.5e9)           # the pads cost gain and match: about half the builds meet 5.4 dB gain and -5.4 dB |S11| here
    jobs = {"mu": [(SPEC_MU_MIN, 20e6, 9e9, 1.04)],
            "mu+s21+s11": [(Q.SPEC_S21_MIN_DB, band[0], band[1], 5.4), (Q.SPEC_S11_MAX_DB, band[0], band[1], -5.4), (SPEC_MU_MIN, 20e6, 9e9, 1.04)],
            "s21+s11": [(Q.SPEC_S21_MIN_DB, band[0], band[1], 5.4), (Q.SPEC_S11_MAX_DB, band[0], band[1], -5.4)]}
    rows = []
    for chain in ("interp", "jit"):
        os.environ["QO100NET_CHAIN"] = chain
        for name, specs in jobs.items():
            hs = len(specs) - 1
            hist = dict(hist_bins=64, hist_spec=hs, hist_lo=0.9 if specs[hs][0] == SPEC_MU_MIN else -20.0, hist_hi=1.2 if specs[hs][0] == SPEC_MU_MIN else 0.0)
            p = Q.Plan(ctx, net, f, specs, seed=7, tols=PAD_TOLS, **hist)
            p.launch(0, 4096)
            p.read()
            ts, out = [], None
            for _ in range(args.reps):
                p.reset()
                t0 = time.perf_counter()
                p.launch(0, args.samples)
                out = p.read()
                ts.append(time.perf_counter() - t0)
            evals = float(args.samples) * len(f)
            rows.append(dict(chain=chain, job=name, kernel=p.kernel_name, seconds_best=min(ts), seconds_median=float(np.median(ts)),
                             evals_per_s=evals / min(ts), n_pass=int(out["n_pass"]), fail_per_spec=[int(x) for x in out["fail_per_spec"]]))
            p.close()
            print(json.dumps(rows[-1]))
    os.environ.pop("QO100NET_CHAIN", None)
    ctx.close()
    res = {"card": card, "samples": args.samples, "points": 4096, "grid": "20 MHz - 9 GHz linear", "reps": args.reps, "runs": rows}
    for chain in ("interp", "jit"):
        t = {r["job"]: r["seconds_best"] for r in rows if r["chain"] == chain}
        res["mu_over_s21_s11_" + chain] = t["mu"] / t["s21+s11"]
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(json.dumps(res, indent=1) + "\n")
    return res


if __name__ == "__main__":
    main()
