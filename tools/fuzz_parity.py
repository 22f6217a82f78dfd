#!/usr/bin/env python
"""Differential fuzz of the Monte-Carlo kernels on random lumped cascades (GPU box).

For each of --nets random networks -- 3..14 branches drawn from all ten lumped branch kinds (with and without parasitics),
optionally behind a front block (coupled line, transmission line), random terminations, random tolerances, log or linear
grid of random length, 1..4 specs on |S21| / |S11| (and |S22| with --s22, a stability factor mu with --mu) placed at quantiles of a FULL_S pre-run so that the yield is never
degenerate, optional histogram -- the job runs
   (a) on the kernel the plan selects (thread-per-sample / warp-per-sample transfer-function kernel, spot kernel, chain kernel),
   (b) on the opcode interpreter (QO100NET_KERNEL=interp),
   (c) every --oracle-every-th network on the CPU oracle,
and all integer counters (n_pass, fail_per_spec, histogram) must be identical.  Prints one JSON summary.

   python tools/fuzz_parity.py [--nets 300] [--samples 3000] [--seed 1] [--out gpurun_out/fuzz.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "qo-100-tools_b200", "python"))
sys.path.insert(0, ROOT)


_BLK = {}


def _register(R, names):
    """hand the oracle the golden two-ports in the order the network holds them (block i = names[i])"""
    g = np.load(os.path.join(ROOT, "tests", "golden", "touchstone.npz"))
    R.sblock_clear()
    for i, nm in enumerate(names):
        sd = g[nm + "_s"]
        R.sblock_register(i, g[nm + "_f"], sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], float(g[nm + "_z0"]))


def _driver(Q):
    """The reference's 20 W driver (docs/pa-driver/pa_20W_vdd_32V_idq_180mA.s2p, tests/golden/touchstone.npz): active and
    non-reciprocal."""
    if "drv" not in _BLK:
        g = np.load(os.path.join(ROOT, "tests", "golden", "touchstone.npz"))
        sd = g["pa_20W_s"]
        _BLK["drv"] = Q.SBlock.from_arrays(g["pa_20W_f"], sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], float(g["pa_20W_z0"]))
    return _BLK["drv"]


def _block(Q):
    """The measured inductor of pa-bias-simulation.sch:39 (tests/golden/touchstone.npz), registered with the oracle as block 0."""
    if "blk" not in _BLK:
        from oracle import refbind as R
        g = np.load(os.path.join(ROOT, "tests", "golden", "touchstone.npz"))
        fd, sd, z0 = g["11SQ39N_f"], g["11SQ39N_s"], float(g["11SQ39N_z0"])
        _BLK["blk"] = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
        R.sblock_clear()
        R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    return _BLK["blk"]


SPEC_S21_MIN_DB, SPEC_S11_MAX_DB, SPEC_GD_MAX, SPEC_S22_MAX_DB, SPEC_MU_MIN = 1, 3, 4, 5, 6     # qo_spec_kind
_PLANE = {1: 1, 2: 1, 3: 0, 5: 3}                                                # spec kind -> FULL_S plane (S11, S21, S12, S22)


def mu_factor(s11, s21, s12, s22):
    """Edwards-Sinsky load-side stability factor: mu > 1 <=> unconditionally stable"""
    d = s11 * s22 - s12 * s21
    return (1.0 - np.abs(s11) ** 2) / (np.abs(s22 - d * np.conj(s11)) + np.abs(s12 * s21))


def oracle_counters(R, net, f, specs, cfg, nthreads=None, chunk=256):
    """The CPU oracle's counters of a cascade job.  Its own reduction (ref_mc_run) knows |S21|, |S11| and group-delay specs; a job
    with |S22| or stability (mu) specs is reduced here from the oracle's FULL_S planes of the same samples, the way ref_mc_run
    reduces the others: per spec the worst in-band 10 log10 |S|^2 (smallest for an |S21| minimum, else largest), a fail when it is
    beyond the limit, the histogram bin floor((worst - lo) / (hi - lo) * bins) clamped to the window.  A mu spec takes mu of each
    point from all four planes (S12 carries the blocks' determinant); it fails when some in-band point has !(mu >= limit), NaN
    included, and its histogram value is the smallest in-band mu that is not NaN (+inf when there is none), linear."""
    nthreads = nthreads or R.max_threads()
    rs, rl = net.terminations
    el = R.make_elems(net.elements)
    f = np.ascontiguousarray(f, dtype=np.float64)
    if not any(s[0] in (SPEC_S22_MAX_DB, SPEC_MU_MIN) for s in specs):
        return R.mc_run(el, rs, rl, f, specs, cfg, nthreads=nthreads)
    if any(s[0] not in _PLANE and s[0] != SPEC_MU_MIN for s in specs):
        raise ValueError("group-delay specs next to |S22| or mu specs are not reduced from FULL_S planes")
    n, nspec = int(cfg.n_samples), len(specs)
    bands = [(f >= s[1]) & (f <= s[2]) for s in specs]
    worst = np.zeros((nspec, n))
    fails = np.zeros((nspec, n), dtype=bool)
    for a in range(0, n, chunk):
        c = type(cfg).from_buffer_copy(cfg)              # same seed, tolerances (the pointer stays valid), distribution
        c.sample_offset, c.n_samples, c.hist_bins = cfg.sample_offset + a, min(chunk, n - a), 0
        planes = R.mc_run(el, rs, rl, f, [], c, full_s=True, nthreads=nthreads)["s"]
        for i, s in enumerate(specs):
            if not bands[i].any():
                continue
            if s[0] == SPEC_MU_MIN:
                mu = mu_factor(*(planes[q][:, bands[i]] for q in range(4)))
                worst[i, a:a + c.n_samples] = np.where(np.isnan(mu), np.inf, mu).min(axis=1)
                fails[i, a:a + c.n_samples] = ~(mu >= s[3]).all(axis=1)
                continue
            p = planes[_PLANE[s[0]]][:, bands[i]]
            v = 10.0 * np.log10(p.real * p.real + p.imag * p.imag)
            worst[i, a:a + c.n_samples] = v.min(axis=1) if s[0] == SPEC_S21_MIN_DB else v.max(axis=1)
    for i, s in enumerate(specs):
        if bands[i].any() and s[0] != SPEC_MU_MIN:
            fails[i] = ~(worst[i] >= s[3]) if s[0] == SPEC_S21_MIN_DB else ~(worst[i] <= s[3])
    hb = int(cfg.hist_bins)
    hist = np.zeros(max(hb, 0), dtype=np.uint64)
    if hb > 0 and 0 <= cfg.hist_spec < nspec and bands[cfg.hist_spec].any():
        x = (worst[cfg.hist_spec] - cfg.hist_lo) / (cfg.hist_hi - cfg.hist_lo) * hb
        np.add.at(hist, np.clip(np.floor(x), 0, hb - 1).astype(np.int64), 1)
    return dict(n_pass=int((~fails.any(axis=0)).sum()), n_total=n, fail_per_spec=fails.sum(axis=1).astype(np.uint64), hist=hist)


def random_ladder(Q, rng):
    """pcb/generic-filter family: alternating series L / shunt C of order 1..11 with the ESR / SRF parasitic model, optionally behind
    a coupled-line section -- what the straight-line chain kernel (QO100NET_KERNEL=ladder) covers."""
    fc = 10.0 ** rng.uniform(6.5, 9.3)
    order = int(rng.integers(1, 12))
    net = (Q.Net.butter_lpf(order, fc, 50.0, bool(rng.integers(0, 2))) if (rng.random() < 0.4 or order % 2 == 0) else Q.Net.cheby_lpf(order, float(rng.choice([0.05, 0.1, 0.5])), fc, 50.0, bool(rng.integers(0, 2))))
    if rng.random() < 0.8:
        net = net.add_parasitics(fc, rng.uniform(30, 150), rng.uniform(8, 40), rng.uniform(0.02, 0.5), rng.uniform(10, 60))
    tols = Q.lc_tolerances(net, float(rng.choice([0.02, 0.05, 0.1])), float(rng.choice([0.01, 0.02, 0.05])))
    if rng.random() < 0.4:
        te = rng.uniform(40, 110)
        cpl = Q.Net.from_elements([(Q.CPL_THRU, [55.2771, 45.2267, te, te * (1.0 if rng.random() < 0.5 else rng.uniform(0.93, 1.0)), fc, 50.0])], 50.0, 50.0)
        net = cpl.concat(net)
        tols = [(0, 0, 0, Q.TOL_REL, 0.02), (0, 1, 1, Q.TOL_REL, 0.02), (0, 2, 2, Q.TOL_REL, 0.01), (0, 3, 2, Q.TOL_REL, 0.01)] + [(e + 1, p, v + 3, m_, t) for (e, p, v, m_, t) in tols]
    nf = int(rng.choice([3, 33, 64, 200, 515, 1000, 4096]))
    span = rng.uniform(2.0, 6.0)
    f = Q.grid_log(fc / span, fc * span, nf) if rng.random() < 0.6 else Q.grid_lin(fc / span, fc * span, nf)
    return net, f, tols, fc


def random_net(Q, rng):
    fc = 10.0 ** rng.uniform(6.5, 9.3)
    wc = 2 * np.pi * fc
    z0 = float(rng.choice([50.0, 50.0, 75.0, 100.0]))
    n = int(rng.integers(3, 15))
    el = []
    series = bool(rng.integers(0, 2))
    for _ in range(n):
        g = rng.uniform(0.3, 2.2)
        L, C = g * z0 / wc, g / (z0 * wc)
        par = rng.random() < 0.6
        kind = rng.integers(0, 10)
        if series:
            if kind < 5:
                el.append((Q.SER_L, [L, (wc * L / rng.uniform(30, 200)) if par else 0.0, (1 / (L * (wc * rng.uniform(8, 60)) ** 2)) if par else 0.0]))
            elif kind < 7:
                el.append((Q.SER_C, [C * rng.uniform(5, 40), rng.uniform(0.02, 0.5) if par else 0.0, (1 / (C * 20 * (wc * rng.uniform(10, 60)) ** 2)) if par else 0.0]))
            elif kind == 7:
                el.append((Q.SER_R, [rng.uniform(0.2, 5.0)]))
            elif kind == 8:
                el.append((Q.SER_LC_SER, [L * 0.1, C * rng.uniform(20, 60)]))
            else:
                k = rng.uniform(1.6, 3.0)                      # trap above the pass band
                el.append((Q.SER_LC_PAR, [L * 0.15, 1 / (L * 0.15 * (k * wc) ** 2)]))
        else:
            if kind < 5:
                el.append((Q.SHUNT_C, [C, rng.uniform(0.02, 0.5) if par else 0.0, (1 / (C * (wc * rng.uniform(10, 60)) ** 2)) if par else 0.0]))
            elif kind < 7:
                el.append((Q.SHUNT_L, [L * rng.uniform(5, 40), rng.uniform(0.05, 1.0) if par else 0.0, (1 / (L * 20 * (wc * rng.uniform(8, 40)) ** 2)) if par else 0.0]))
            elif kind == 7:
                el.append((Q.SHUNT_R, [z0 * rng.uniform(10, 100)]))
            elif kind == 8:
                k = rng.uniform(1.6, 3.0)
                el.append((Q.SHUNT_LC_SER, [L * 3.0, 1 / (L * 3.0 * (k * wc) ** 2)]))
            else:
                el.append((Q.SHUNT_LC_PAR, [L * rng.uniform(8, 30), C * 0.05]))
        if rng.random() < 0.85:
            series = not series
    front = rng.integers(0, 6)
    tols = []
    if front == 1:
        te = rng.uniform(40, 110)
        el = [(Q.CPL_THRU, [z0 * 1.105, z0 / 1.105, te, te * (1.0 if rng.random() < 0.5 else rng.uniform(0.93, 1.0)), fc, z0])] + el
        tols += [(0, 0, 0, Q.TOL_REL, 0.02), (0, 1, 1, Q.TOL_REL, 0.02), (0, 2, 2, Q.TOL_REL, 0.01), (0, 3, 2, Q.TOL_REL, 0.01)]
    elif front == 5:
        # physical coupled microstrip (util/directional-couplers/dir_cpl_2.4g_20dB.trc:6-17 scaled): etch on W (and -/+ on S), H, Er
        sub = (Q.SUBST, [3.5 * rng.uniform(0.8, 1.3), 0.762e-3, 35e-6, 0.0, 0.0, 0.0])
        cpl = (Q.CPL_MS, [1.69218e-3 * rng.uniform(0.8, 1.25), 0.991476e-3 * rng.uniform(0.7, 1.5), 20e-3 * rng.uniform(0.5, 1.5) * 2.4e9 / max(fc, 3e8), 0.2, max(fc, 3e8), z0])
        el = [sub, cpl] + el
        tols += [(1, 0, 0, Q.TOL_ABS, 0.03e-3), (1, 1, 0, Q.TOL_ABS, -0.03e-3), (0, 1, 1, Q.TOL_REL, 0.05), (0, 0, 2, Q.TOL_ABS, 0.1)]
    elif front == 2:
        el = [(Q.TLINE, [z0 * rng.uniform(0.7, 1.5), rng.uniform(10, 120), fc])] + el
        tols += [(0, 0, 0, Q.TOL_REL, 0.05), (0, 1, 1, Q.TOL_REL, 0.03)]
    nv = len(tols)
    for e, (k, p) in enumerate(el):
        if k in (Q.SER_L, Q.SHUNT_L, Q.SER_C, Q.SHUNT_C, Q.SER_LC_SER, Q.SER_LC_PAR, Q.SHUNT_LC_SER, Q.SHUNT_LC_PAR) and rng.random() < 0.9:
            tols.append((e, 0, nv, Q.TOL_REL, float(rng.choice([0.01, 0.02, 0.05, 0.1]))))
            nv += 1
            if k >= Q.SER_LC_SER and rng.random() < 0.5:
                tols.append((e, 1, nv, Q.TOL_REL, 0.05))
                nv += 1
        elif k in (Q.SER_R, Q.SHUNT_R) and rng.random() < 0.5:
            tols.append((e, 0, nv, Q.TOL_REL, 0.05))
            nv += 1
    if not tols:                                     # no tolerance at all: every sample is the nominal network
        tols.append((len(el) - 1, 0, 0, Q.TOL_REL, 0.05))
    rs = z0 if rng.random() < 0.7 else z0 * rng.uniform(0.5, 2.0)
    rl = z0 if rng.random() < 0.7 else z0 * rng.uniform(0.5, 2.0)
    nf = int(rng.choice([3, 7, 33, 64, 200, 515, 1000, 2048, 4096]))
    span = rng.uniform(2.0, 6.0)
    f = Q.grid_log(fc / span, fc * span, nf) if rng.random() < 0.6 else Q.grid_lin(fc / span, fc * span, nf)
    net = Q.Net.from_elements(el, float(rs), float(rl))
    if front == 4 and fc < 2e9:                      # measured two-port in front (polar or rectangular interpolation)
        net = _block(Q).as_net(bool(rng.integers(0, 2)), float(rs), float(rl)).concat(net)
        tols = [(e + 1, p, v, m_, t) for (e, p, v, m_, t) in tols]
    return net, f, tols, fc


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--nets", type=int, default=300)
    ap.add_argument("--samples", type=int, default=3000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--oracle-every", type=int, default=5)
    ap.add_argument("--big-every", type=int, default=7, help="every k-th network runs a launch large enough for the thread-per-sample kernel")
    ap.add_argument("--ladders", action="store_true", help="pcb/generic-filter ladders only, the selected run forced onto the chain kernel (QO100NET_KERNEL=ladder)")
    ap.add_argument("--gd", action="store_true", help="add a group-delay spec (limit around the nominal network's worst in-band delay) to networks without a front block")
    ap.add_argument("--chain-jit", action="store_true", help="the selected run is the run-time compiled chain kernel (QO100NET_KERNEL=interp QO100NET_CHAIN=jit) against the "
                    "interpreter proper; 60 %% of the networks get a perturbed line BEHIND the cascade and 30 %% the measured two-port behind that -- what no polynomial kernel takes")
    ap.add_argument("--s22", action="store_true", help="|S22| specs in the random spec mix: the reversed cascade on the polynomial / ladder kernels, "
                    "or the interpreter's direct S22 (next to |S11|, behind a front block)")
    ap.add_argument("--mu", action="store_true", help="the 20 W driver (active, non-reciprocal) in front of or behind each random cascade, a "
                    "stability spec mu >= limit in every job, the selected run on the compiled chain kernel against the interpreter")
    ap.add_argument("--only", type=int, default=-1, help="run just this network (each network has its own random stream) and dump it")
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import qo100net as Q
    from oracle import refbind as R
    ctx = Q.Context(device=0)
    kernels, mism, skipped, oracle_checked, fs_checked, fused_runs, s22_jobs, mu_jobs = {}, [], 0, 0, 0, 0, 0, 0
    jit = args.chain_jit or args.mu
    big = 2 * 148 * 3 * 128 + 77          # large enough for the thread-per-sample kernel on every 7th network
    for i in range(args.nets):
        if args.only >= 0 and i != args.only:
            continue
        rng = np.random.default_rng([args.seed, i])          # one stream per network: --only reproduces it exactly
        net, f, tols, fc = random_ladder(Q, rng) if args.ladders else random_net(Q, rng)
        if args.chain_jit:
            rs_, rl_ = net.terminations
            if rng.random() < 0.6:
                ne = len(net)
                net = net.concat(Q.Net.from_elements([(Q.TLINE, [50.0 * rng.uniform(0.7, 1.5), rng.uniform(10, 120), fc])], rs_, rl_))
                nv = 1 + max(t[2] for t in tols)
                tols = list(tols) + [(ne, 0, nv, Q.TOL_REL, 0.05), (ne, 1, nv + 1, Q.TOL_REL, 0.03)]
            if rng.random() < 0.3 and fc < 2e9 and net.elements[0][0] != Q.SBLOCK:
                net = net.concat(_block(Q).as_net(True, rs_, rl_))
        if args.mu:
            # the driver's data covers 10 MHz - 10 GHz: keep the grid inside it
            f = f[(f >= 1e7) & (f <= 1e10)]
            rs_, rl_ = net.terminations
            drv = _driver(Q).as_net(bool(rng.integers(0, 2)), rs_, rl_)
            ind = ["11SQ39N"] if any(k_ == Q.SBLOCK for k_, _p in net.elements) else []
            if rng.random() < 0.5:
                net = drv.concat(net)
                tols = [(e + 1, p, v, m_, t) for (e, p, v, m_, t) in tols]
                _register(R, ["pa_20W"] + ind)
            else:
                net = net.concat(drv)
                _register(R, ind + ["pa_20W"])
        n = big if i % args.big_every == args.big_every - 1 else args.samples
        dist = Q.DIST_GAUSS3S if rng.random() < 0.3 else Q.DIST_UNIFORM
        try:
            fs = ctx.mc_run(net, f, [], 99, 200, tols, mode=Q.MODE_FULL_S, dist=dist)["s"]
        except Q.QoError:
            skipped += 1
            continue
        a21 = 20 * np.log10(np.maximum(np.abs(fs[1]), 1e-300))
        a11 = 20 * np.log10(np.maximum(np.abs(fs[0]), 1e-300))
        a22 = 20 * np.log10(np.maximum(np.abs(fs[3]), 1e-300))
        if len(f) == 0 or not (np.all(np.isfinite(a21)) and np.all(np.isfinite(a11)) and (not args.s22 or np.all(np.isfinite(a22)))):
            skipped += 1
            continue
        specs = []
        if args.mu:
            lo, hi = sorted(rng.uniform(f[0], f[-1], 2))
            band = (f >= lo) & (f <= hi)
            if band.any():
                mu = mu_factor(*(np.asarray(fs[q])[:, band] for q in range(4))).min(axis=1)
                # not a knife edge: the limit inside a real spread of the samples' smallest mu
                if np.all(np.isfinite(mu)) and np.quantile(mu, 0.9) - np.quantile(mu, 0.1) > 1e-4 * max(1.0, abs(np.median(mu))):
                    specs.append((Q.SPEC_MU_MIN, float(lo), float(hi), float(np.quantile(mu, rng.uniform(0.2, 0.8)))))
            if not specs:
                skipped += 1
                continue
        for _ in range(int(rng.choice([1, 2, 3, 4, 4, 6, 8])) - len(specs)):
            lo, hi = sorted(rng.uniform(f[0], f[-1], 2))
            if rng.random() < 0.3:
                lo = hi = float(f[int(rng.integers(0, len(f)))])
            band = (f >= lo) & (f <= hi)
            if not band.any():
                continue
            kind = int(rng.choice([Q.SPEC_S21_MIN_DB, Q.SPEC_S21_MAX_DB, Q.SPEC_S11_MAX_DB] + ([Q.SPEC_S22_MAX_DB] * 2 if args.s22 else [])))
            q = float(rng.uniform(0.2, 0.8))
            if kind == Q.SPEC_S21_MIN_DB:
                v, qq = a21[:, band].min(axis=1), 1 - q
            elif kind == Q.SPEC_S21_MAX_DB:
                v, qq = a21[:, band].max(axis=1), q
            elif kind == Q.SPEC_S22_MAX_DB:
                v, qq = a22[:, band].max(axis=1), q
            else:
                v, qq = a11[:, band].max(axis=1), q
            # no knife-edge specs: a quantity the tolerances barely move (all samples within 0.01 dB: any threshold inside that
            # cluster is decided by the last bits of whichever formulation evaluates it) or the depth of a notch sampled on the grid
            if np.quantile(v, 0.9) - np.quantile(v, 0.1) < 0.01 or v.min() < -140.0:
                continue
            specs.append((kind, float(lo), float(hi), float(np.quantile(v, qq))))
        if args.gd and net.elements[0][0] not in (Q.CPL_THRU, Q.TLINE, Q.SBLOCK) and all(k_ != Q.SBLOCK for k_, _p in net.elements) and len(specs) < 8 and not any(s_[0] in (Q.SPEC_S11_MAX_DB, Q.SPEC_S22_MAX_DB) for s_ in specs):
            gdn = ctx.sweep(net, f, gd=True)[4]
            lo, hi = sorted(rng.uniform(f[0], f[-1], 2))
            band = (f >= lo) & (f <= hi)
            # not across a transmission zero: the delay is singular there, and the kernels' analytic derivative and the
            # interpreter's / oracle's central difference over f (1 +- 1e-6) are two different approximations of it
            if band.any() and np.all(np.isfinite(gdn[band])) and gdn[band].max() > 0 and a21[:, band].min() > -60.0:
                specs.append((Q.SPEC_GD_MAX, float(lo), float(hi), float(gdn[band].max() * rng.uniform(0.97, 1.08))))
        if not specs:
            skipped += 1
            continue
        s22_jobs += any(s_[0] == Q.SPEC_S22_MAX_DB for s_ in specs)
        mu_jobs += any(s_[0] == Q.SPEC_MU_MIN for s_ in specs)
        hist = {}
        if rng.random() < 0.6:
            hs = int(rng.integers(0, len(specs)))
            hist = dict(hist_bins=int(rng.choice([16, 64, 256])), hist_spec=hs, hist_lo=specs[hs][3] - 3.0, hist_hi=specs[hs][3] + 3.0)
        os.environ.pop("QO100NET_KERNEL", None)
        if args.ladders:
            os.environ["QO100NET_KERNEL"] = "ladder"
        if jit:
            os.environ["QO100NET_KERNEL"] = "interp"
            os.environ["QO100NET_CHAIN"] = "jit"
        plan = Q.Plan(ctx, net, f, specs, seed=1000 + i, tols=tols, dist=dist, **hist)
        off = int(rng.integers(0, 2 ** 40))
        plan.launch(off, n)
        got = plan.read()
        kname = plan.kernel_name
        if kname == "qo_mc_ts_kernel" and plan.tf_info["fused_specs"]:
            fused_runs += 1                          # the thread-per-sample kernel walked a spec on its fused margin
        plan.close()
        kernels[kname] = kernels.get(kname, 0) + 1
        os.environ["QO100NET_KERNEL"] = "interp"
        os.environ.pop("QO100NET_CHAIN", None)
        plan = Q.Plan(ctx, net, f, specs, seed=1000 + i, tols=tols, dist=dist, **hist)
        plan.launch(off, n)
        ref = plan.read()
        assert plan.kernel_name == "qo_mc_lumped_kernel", plan.kernel_name
        plan.close()
        os.environ.pop("QO100NET_KERNEL", None)
        same = got["n_pass"] == ref["n_pass"] and np.array_equal(got["fail_per_spec"], ref["fail_per_spec"]) and np.array_equal(got["hist"], ref["hist"])
        if same and i % args.oracle_every == 0 and n <= args.samples:
            o = oracle_counters(R, net, f, specs, R.mc_cfg(1000 + i, n, tols, sample_offset=off, dist=dist, **hist))
            oracle_checked += 1
            same = got["n_pass"] == o["n_pass"] and np.array_equal(got["fail_per_spec"], o["fail_per_spec"]) and np.array_equal(got["hist"], o["hist"])
        if same and i % 4 == 1:
            # FULL_S: a launch large enough for qo_fs_tf_kernel against the interpreter's planes of the same samples
            if jit:
                os.environ["QO100NET_KERNEL"] = "interp"
                os.environ["QO100NET_CHAIN"] = "jit"
            a = ctx.mc_run(net, f, [], 1000 + i, 1536, tols, sample_offset=off, mode=Q.MODE_FULL_S, dist=dist)["s"]
            os.environ.pop("QO100NET_CHAIN", None)
            b = ctx.mc_run(net, f, [], 1000 + i, 64, tols, sample_offset=off, mode=Q.MODE_FULL_S, dist=dist)["s"]
            os.environ.pop("QO100NET_KERNEL", None)
            fs_checked += 1
            for pl in range(4):
                ref_ = np.asarray(b[pl]); got_ = np.asarray(a[pl])[:64]
                tol_ = 1e-9 * np.maximum(np.abs(ref_), 1e-5 if pl in (1, 2) else 0.02)      # -100 dB floor: next to an ideal trap's zero every formulation is down to ~1e-15 absolute
                if not np.all(np.abs(got_ - ref_) <= tol_):
                    same = False
                    kname = "FULL_S plane %d (1536 vs 64 samples)" % pl
        if not same:
            mism.append({"net": i, "kernel": kname, "n": n, "nf": len(f), "f0": float(f[0]), "f1": float(f[-1]), "log_grid": bool(abs(f[1] / f[0] - f[2] / f[1]) < 1e-9),
                         "terminations": [float(v) for v in net.terminations], "elements": [(int(k), [float(x) for x in p]) for k, p in net.elements],
                         "tols": [[int(a), int(b), int(c), int(d), float(e)] for a, b, c, d, e in tols], "dist": int(dist), "offset": off, "seed": 1000 + i, "hist": hist,
                         "specs": specs, "got": int(got["n_pass"]), "interp": int(ref["n_pass"]),
                         "got_fail": [int(v) for v in got["fail_per_spec"]], "interp_fail": [int(v) for v in ref["fail_per_spec"]]})
    out = {"networks": args.nets, "skipped": skipped, "compared": args.nets - skipped, "oracle_checked": oracle_checked, "full_s_checked": fs_checked,
           "fused_runs": fused_runs, "s22_jobs": s22_jobs, "mu_jobs": mu_jobs, "kernels_selected": kernels, "mismatches": len(mism), "details": mism[:10], "seed": args.seed, "samples": args.samples}
    print(json.dumps(out, indent=1))
    if args.out:
        open(args.out, "w").write(json.dumps(out, indent=1))
    ctx.close()
    return out


if __name__ == "__main__":
    sys.exit(1 if main()["mismatches"] else 0)
