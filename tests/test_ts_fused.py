"""Fused margins of the thread-per-sample kernel (qo_tf_core.h::qo_tf_fuse): where exactly one |S21| spec looks, the kernel
walks the sign of one polynomial F = +-(N2 - t E) instead of |numerator|^2 and E.  The plan accepts it per spec only where it
agrees with the unfused margin to 1e-12 of |den|^2."""
from fractions import Fraction

import numpy as np
import pytest


def test_plan_fuses_the_stop_band_of_cfg2_and_not_its_histogram_spec(Q, W, monkeypatch):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    w = W.cfg2()
    a = Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    assert a["selected"] and a["den_form"] == "E"
    assert a["fused_specs"] == 0b10                       # spec 1 (stop band); spec 0 carries the histogram
    assert 0.0 < a["fused_err"] <= 1e-12


def test_plan_refuses_the_pass_band_of_ideal11(Q, monkeypatch):
    """The -0.5 dB pass band of an ideal 11th-order Chebyshev ladder: |Num|^2 cancels inside the ripple and the fused margin
    loses more than the gate allows; with the stop band carrying the histogram nothing is fused."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    fc = 10e6
    net = Q.Net.cheby_lpf(11, 0.1, fc, 50.0, True)
    f = Q.grid_log(fc / 2.5, fc * 6.25, 1003)
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, 0.95 * fc, -0.5), (Q.SPEC_S21_MAX_DB, 1.3 * fc, 1e99, -49.0)]
    tols = Q.lc_tolerances(net, 0.05, 0.02)
    a = Q.plan_analyze(net, f, specs, tols, hist_bins=64, hist_spec=1, hist_lo=-80.0, hist_hi=-40.0)
    assert a["selected"] and a["den_form"] == "none" and a["fused_specs"] == 0 and a["fused_err"] == 0.0
    # without the histogram the stop band is fused, the pass band still is not
    assert Q.plan_analyze(net, f, specs, tols)["fused_specs"] == 0b10


# ---- numpy / exact restatement of the compensated formation ------------------------------------------------------------
def _mul(a, b):
    out = [Fraction(0)] * (len(a) + len(b) - 1)
    for i, u in enumerate(a):
        for j, v in enumerate(b):
            out[i + j] += u * v
    return out


def _add(a, b):
    n = max(len(a), len(b))
    return [(a[i] if i < len(a) else 0) + (b[i] if i < len(b) else 0) for i in range(n)]


def _fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def _dd_fma(s, c, a, b):
    p = a * b
    pe = _fma(a, b, -p)
    t = s + p
    bp = t - s
    return t, c + (((s - (t - bp)) + (p - bp)) + pe)


def _fuse(kn, ke, cn, ce, t, neg):
    """qo_tf_fuse, operation for operation"""
    out = []
    for k in range(max(2 * kn, ke)):
        s = c = 0.0
        for i in range(kn):
            j = k - i
            if i <= j < kn:
                s, c = _dd_fma(s, c, cn[2 * i] if i == j else 2.0 * cn[2 * i], cn[2 * j])
        for i in range(kn):
            j = k - 1 - i
            if i <= j < kn:
                s, c = _dd_fma(s, c, -cn[2 * i + 1] if i == j else -2.0 * cn[2 * i + 1], cn[2 * j + 1])
        if k < max(ke, 1):
            s, c = _dd_fma(s, c, -t, ce[k] if ke > 0 else 1.0)
        v = s + c
        out.append((v if neg else -v) + 0.0)
    return out


def _expand(elements, rs, rl, wr):
    """Num(sn) = P + Rs Q and prod D(sn) of the ladder (sn = s / wr), exactly, from the load end"""
    P, Qp, Dp = [Fraction(rl)], [Fraction(1)], [Fraction(1)]
    for op, prm in reversed(elements):
        if op == 3:      # series L (L, R, Cp): Z = (R + s L) / (1 + s R Cp + s^2 L Cp)
            L, R, Cp = (Fraction(v) for v in prm[:3])
            N, D = [R, L * wr], [Fraction(1), R * Cp * wr, L * Cp * wr * wr]
            P, Qp = _add(_mul(D, P), _mul(N, Qp)), _mul(D, Qp)
        else:            # shunt C (C, R, Ls): Y = s C / (1 + s R C + s^2 Ls C)
            assert op == 6
            C_, R, Ls = (Fraction(v) for v in prm[:3])
            N, D = [Fraction(0), C_ * wr], [Fraction(1), R * C_ * wr, Ls * C_ * wr * wr]
            P, Qp = _mul(D, P), _add(_mul(D, Qp), _mul(N, P))
        Dp = _mul(Dp, D)
    return _add(P, [Fraction(rs) * q for q in Qp]), Dp


def _even_odd_in_y(c):
    """c(jx) = r0(y) + j x r1(y), y = -x^2: (jx)^(2k) = y^k and (jx)^(2k+1) = j x y^k"""
    return [c[i] for i in range(0, len(c), 2)], [c[i] for i in range(1, len(c), 2)]


def _horner(c, y):
    v = Fraction(0)
    for a in reversed(c):
        v = v * y + Fraction(a)
    return v


def test_compensated_formation_holds_the_stop_band_bound(W):
    """cfg2's element values, 10 random draws (+-5 % L, +-2 % C), the plan's lengths (kn = 9, ke = 14), stop-band points
    (f >= 13 MHz): the fused F against the exact value of the same truncated polynomials, relative to |den|^2 = N2 / E."""
    w = W.cfg2()
    rs, rl = w.net.terminations
    f = np.asarray(w.f)
    wr = 2 * np.pi * np.sqrt(f.min() * f.max())
    kn, ke = 9, 14
    rng = np.random.default_rng(2)
    pts = f[f >= 13e6][::64]
    worst = 0.0
    for _ in range(10):
        els = []
        for op, prm in w.net.elements:
            prm = list(prm)
            prm[0] *= 1.0 + (0.05 if op == 3 else 0.02) * rng.uniform(-1.0, 1.0)
            els.append((op, prm))
        num, den = _expand(els, rs, rl, Fraction(float(wr)))
        a, b = _even_odd_in_y(num)
        dr, di = _even_odd_in_y(den)
        e = _add(_mul(dr, dr), [Fraction(0)] + [-v for v in _mul(di, di)])        # |D(jx)|^2 = Dr^2 - y Di^2
        cn = []
        for k in range(kn):
            cn += [float(a[k]) if k < len(a) else 0.0, float(b[k]) if k < len(b) else 0.0]
        ce = [float(v) for v in e[:ke]]
        # a threshold just below the stop band's lowest |den|^2 (at its edge), as a spec the sample nearly fails
        ys = [Fraction(-(2 * np.pi * fk / wr) ** 2) for fk in pts]
        n2 = [_horner(cn[0::2], y) ** 2 - y * _horner(cn[1::2], y) ** 2 for y in ys]
        ee = [_horner(ce, y) for y in ys]
        t = 0.99 * min(float(n / d) for n, d in zip(n2, ee))
        for neg in (False, True):
            fz = _fuse(kn, ke, cn, ce, t, neg)
            for y, n, d in zip(ys, n2, ee):
                got = fz[-1]
                for m in range(len(fz) - 2, -1, -1):
                    got = _fma(got, float(y), fz[m])
                ref = (n - Fraction(t) * d) if neg else (Fraction(t) * d - n)
                worst = max(worst, float(abs(Fraction(got) - ref) / n))
    assert worst <= 1e-13, worst


@pytest.mark.gpu
def test_fused_kernel_equals_warp_per_sample_on_cfg2(Q, W, ctx, monkeypatch):
    """cfg2 at its full 1e6 samples over three disjoint sample ranges: the default kernel (thread-per-sample, stop band on the
    fused margin) and QO100NET_KERNEL=tf (warp-per-sample, unfused) give the same counters and histogram."""
    w = W.cfg2()
    n = 1000000
    for off in (0, n, (1 << 33) + 7):
        res = {}
        for kern in ("auto", "tf"):
            if kern == "tf":
                monkeypatch.setenv("QO100NET_KERNEL", "tf")
            else:
                monkeypatch.delenv("QO100NET_KERNEL", raising=False)
            plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
            plan.launch(off, n)
            res[kern] = plan.read()
            assert plan.kernel_name == ("qo_mc_ts_kernel" if kern == "auto" else "qo_mc_tf_kernel")
            if kern == "auto":
                assert plan.tf_info["fused_specs"] == 0b10
            plan.close()
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        a, b = res["auto"], res["tf"]
        assert a["n_total"] == b["n_total"] == n and a["n_pass"] == b["n_pass"]
        assert np.array_equal(a["fail_per_spec"], b["fail_per_spec"]) and np.array_equal(a["hist"], b["hist"])
        assert 0 < a["fail_per_spec"][1] < n               # the fused spec decides some samples


# ---- an independent nominal reference: ABCD chain in mpmath at 40 digits ------------------------------------------------
_SER_L, _SHUNT_C, _SER_LC_SER, _SER_LC_PAR, _SHUNT_LC_SER, _SHUNT_LC_PAR = 3, 6, 7, 8, 9, 10     # include/qo100net.h


def _s21_chain(elements, rs, rl, w, j):
    """S21 of the cascade at angular frequency w, from the element list in include/qo100net.h order; the arithmetic is whatever
    w and j are (mpmath scalars for the reference, numpy arrays for screening a whole grid)"""
    A, B, C_, D = 1 + 0 * w, 0 * w, 0 * w, 1 + 0 * w
    for kind, p in elements:
        if kind == _SER_L:             # (L, ESR, Cp): Z = (R + jwL) || 1/(jwCp)
            z, y = (p[1] + j * w * p[0]) / (1 - w * w * p[0] * p[2] + j * w * p[1] * p[2]), None
        elif kind == _SHUNT_C:         # (C, ESR, ESL): Y = 1 / (R + jwLs + 1/(jwC))
            z, y = None, 1 / (p[1] + j * w * p[2] + 1 / (j * w * p[0]))
        elif kind == _SER_LC_SER:      # (L, C)
            z, y = j * w * p[0] + 1 / (j * w * p[1]), None
        elif kind == _SER_LC_PAR:
            z, y = 1 / (j * w * p[1] + 1 / (j * w * p[0])), None
        elif kind == _SHUNT_LC_SER:
            z, y = None, 1 / (j * w * p[0] + 1 / (j * w * p[1]))
        elif kind == _SHUNT_LC_PAR:
            z, y = None, j * w * p[1] + 1 / (j * w * p[0])
        else:
            raise ValueError("no reference for element kind %d" % kind)
        if z is not None:
            B, D = A * z + B, C_ * z + D
        else:
            A, C_ = A + B * y, C_ + D * y
    return 2 / (A * rl + B + C_ * rs * rl + D * rs) * (rs * rl) ** 0.5


def _ref_s21(net, f):
    """S21 at the given grid points, 40 significant digits (the doubles of f and of the element values taken exactly)"""
    import mpmath as mp
    rs, rl = net.terminations
    els = [(k, [mp.mpf(v) for v in p]) for k, p in net.elements]
    out = []
    with mp.workdps(40):
        for fk in f:
            w = 2 * mp.pi * mp.mpf(float(fk))
            s = _s21_chain(els, mp.mpf(rs), mp.mpf(rl), w, mp.mpc(0, 1))
            out.append(complex(s))
    return np.array(out)


def _ref_db(net, fk):
    """20 log10 |S21| at one grid point, from the 40-digit reference"""
    return float(20 * np.log10(np.abs(_ref_s21(net, [fk])[0])))


def _screen_db(net, f):
    """the same chain in numpy doubles over a whole grid: only to find a band's extreme, never for a verdict"""
    rs, rl = net.terminations
    return 20 * np.log10(np.abs(_s21_chain(net.elements, rs, rl, 2 * np.pi * np.asarray(f), 1j)))


# ---- the probe geometries ------------------------------------------------------------------------------------------------
FC = 10e6
DELTA = 1e-6                   # dB: 2.3e-7 relative on |S21|^2, far above the kernels' 1e-10 and the fused margin's ~1e-13


def _gm(f, k):
    """the geometric mean of grid points k-1 and k: a band edge with no doubt about which of the two is inside"""
    return float(np.sqrt(f[k - 1] * f[k]))


def _ladder(kind, order, par):
    import qo100net as Q
    net = Q.Net.butter_lpf(order, FC, 50.0, True) if kind == "butter" else Q.Net.cheby_lpf(order, 0.1, FC, 50.0, True)
    return net.add_parasitics(FC, 60.0, 30.0, 0.1, 50.0) if par else net


class _Geo:
    """One probe: a network and grid, and the spec list as a function of the edge position k and the bracketed spec's limit.
    edge "lo": the bracketed band starts at grid point k (its worst point), "hi": it ends there.  body: the thread-per-sample
    kernel's (KN, KE) with zero-width tolerances; fused: the spec mask the plan must accept for the fused margin."""

    def __init__(self, name, net, f, specs, hist, spec, edge, k0, body, fused, tols):
        self.name, self.net, self.f, self.specs, self.hist = name, net, np.asarray(f), specs, hist
        self.spec, self.edge, self.k0, self.body, self.fused, self.tols = spec, edge, k0, body, fused, tols

    def ztols(self):
        return [(e, p, v, m, 0.0) for (e, p, v, m, _t) in self.tols]

    def is_max(self):
        import qo100net as Q
        return self.specs(self.k0, 0.0)[self.spec][0] == Q.SPEC_S21_MAX_DB


def _in_band(f, s):
    return (f >= s[1]) & (f <= s[2])          # qo_spec: applies to grid f in [f_lo, f_hi]


def _geo_cfg2(name, f, extra=()):
    import qo100net as Q
    from qo100net import workloads as W
    w = W.cfg2()
    return _Geo(name, w.net, f, lambda k, lim: [w.specs[0], (Q.SPEC_S21_MAX_DB, _gm(f, k), 1e99, lim)] + list(extra), w.hist, 1, "lo",
                int(np.searchsorted(f, 13e6)), (9, 12), 0b10, w.tols)


def _geo_ifbpf(nf=2050):
    import qo100net as Q
    from qo100net import workloads as W
    net = W.if_bpf_net()
    f = Q.grid_log(300e6 / 3.5, 500e6 * 3.5, nf)
    return _Geo("G2 if_bpf [0, f_k]", net, f, lambda k, lim: [(Q.SPEC_S21_MIN_DB, 3.6e8, 4.4e8, -0.5), (Q.SPEC_S21_MAX_DB, 0.0, _gm(f, k + 1), lim)],
                dict(hist_bins=64, hist_spec=0, hist_lo=-6.0, hist_hi=0.0), 1, "hi", int(np.searchsorted(f, 1.5e8)), (4, 4), 0b10,
                Q.lc_tolerances(net, 0.05, 0.05))


def _geo_pass(name, kind, order, par, nf, body, extra=()):
    """a MIN-dB pass band [0.2 fc, f_k] in the middle of the grid (fused, neg = false), the histogram on a MAX-dB stop band"""
    import qo100net as Q
    net = _ladder(kind, order, par)
    f = Q.grid_log(FC / 10, 3 * FC, nf)
    return _Geo(name, net, f, lambda k, lim: [(Q.SPEC_S21_MIN_DB, 0.2 * FC, _gm(f, k + 1), lim), (Q.SPEC_S21_MAX_DB, 2 * FC, 1e99, -20.0)] + list(extra),
                dict(hist_bins=64, hist_spec=1, hist_lo=-80.0, hist_hi=0.0), 0, "hi", int(np.searchsorted(f, 0.7 * FC)), body, 0b1,
                Q.lc_tolerances(net, 0.05, 0.02))


def _geo_stop(name, kind, order, par, nf, body):
    """a MAX-dB stop band [f_k, inf) at the top of the grid (fused, neg = true), the histogram on a MIN-dB pass band"""
    import qo100net as Q
    net = _ladder(kind, order, par)
    f = Q.grid_log(FC / 10, 3 * FC, nf)
    return _Geo(name, net, f, lambda k, lim: [(Q.SPEC_S21_MIN_DB, 0.2 * FC, 0.5 * FC, -1.0), (Q.SPEC_S21_MAX_DB, _gm(f, k), 1e99, lim)],
                dict(hist_bins=64, hist_spec=0, hist_lo=-3.0, hist_hi=0.0), 1, "lo", int(np.searchsorted(f, 2 * FC)), body, 0b10,
                Q.lc_tolerances(net, 0.05, 0.02))


def _geometries():
    """name -> _Geo for every probe the GPU brackets run (G1 .. G4, G6; G5 has two bracketed specs and is built on its own)"""
    import qo100net as Q
    from qo100net import workloads as W
    g = [_geo_cfg2("G1 cfg2", W.cfg2().f)]
    g += [_geo_cfg2("G1 nf=%d" % nf, Q.grid_log(4e6, 62.5e6, nf)) for nf in (4097, 4098, 4099)]
    g.append(_geo_ifbpf())
    g += [_geo_pass("G3 butter5", "butter", 5, False, 401, (3, 0)), _geo_pass("G3 butter7 par", "butter", 7, True, 402, (7, 8)),
          _geo_pass("G3 butter11 par", "butter", 11, True, 403, (9, 10))]
    g.append(_geo_pass("G4 butter7 par, two runs", "butter", 7, True, 402, (7, 8), [(Q.SPEC_S21_MAX_DB, 0.4 * FC, 0.5 * FC, 1.0)]))
    g.append(_geo_cfg2("G4 cfg2, two runs", W.cfg2().f, [(Q.SPEC_S21_MAX_DB, 20e6, 25e6, 1.0)]))
    # G6: every other body the plain ladders reach, once with the decisive point in the fused run's first group (stop band) and
    # once in its last (pass band)
    for kind, order, par, body in (("butter", 3, False, (2, 0)), ("butter", 7, False, (4, 0)), ("butter", 9, False, (5, 0)),
                                   ("butter", 11, False, (6, 0)), ("butter", 3, True, (4, 6)), ("butter", 5, True, (5, 8)),
                                   ("butter", 6, True, (6, 8)), ("butter", 9, True, (8, 8)), ("cheby", 11, True, (8, 10))):
        nm = "G6 %s%d%s" % (kind, order, " par" if par else "")
        g.append(_geo_pass(nm + " pass", kind, order, par, 401, body))
        g.append(_geo_stop(nm + " stop", kind, order, par, 401, body))
    return {x.name: x for x in g}


def _geo_g5(f=None):
    """config 2 with two fusable stop bands: [13, 22 MHz] (spec 1, plain) and [23 MHz, inf) (spec 2, the larger: fused)"""
    import qo100net as Q
    from qo100net import workloads as W
    w = W.cfg2()
    f = w.f if f is None else f
    k1, j1, k2 = int(np.searchsorted(f, 13e6)), int(np.searchsorted(f, 22e6)), int(np.searchsorted(f, 23e6))
    specs = lambda l1, l2: [w.specs[0], (Q.SPEC_S21_MAX_DB, _gm(f, k1), _gm(f, j1), l1), (Q.SPEC_S21_MAX_DB, _gm(f, k2), 1e99, l2)]
    return w, f, specs, (k1, k2)



def _positions(geo, count):
    """The first `count` edge positions from geo.k0 on at which a bracket cannot pass vacuously: the decisive grid point k is the
    band's unique extreme by >= 10 delta, and the out-of-band neighbour on that side lies beyond v +- 2 delta in the failing
    direction (taking it in by mistake flips the passing run).  -> [(k, v)]; positions that fail the checks are reported."""
    f, mx = geo.f, geo.is_max()
    db = _screen_db(geo.net, f)
    got, refused = [], []
    for k in range(geo.k0, geo.k0 + count + 8):
        if len(got) == count:
            break
        band = _in_band(f, geo.specs(k, 0.0)[geo.spec])
        nb = k - 1 if geo.edge == "lo" else k + 1
        assert band[k] and not band[nb], (geo.name, k)
        v = _ref_db(geo.net, f[k])
        others = np.where(band)[0]
        others = others[others != k]
        vn = _ref_db(geo.net, f[nb])
        sg = 1.0 if mx else -1.0                   # the failing direction
        ok = np.all(sg * (db[others] - v) <= -10 * DELTA) and sg * (vn - v) > 2 * DELTA
        (got if ok else refused).append((k, v) if ok else k)
    assert len(got) == count, "%s: only %d of %d positions are decisive (refused: %s)" % (geo.name, len(got), count, refused)
    return got


def test_reference_matches_the_oracle(R):
    """the 40-digit chain against the oracle's double-precision sweep on every probe network, at every 8th point of its grid and
    at the first edge position: 1e-12 relative on S21 (a slip in the reference shows here, not on the GPU)"""
    geos = list(_geometries().values())
    w, f5, _s, _k = _geo_g5()
    seen = set()
    worst = 0.0
    for net, f, k0 in [(g.net, g.f, g.k0) for g in geos] + [(w.net, f5, _k[1])]:
        key = (tuple((k, tuple(p)) for k, p in net.elements), net.terminations, len(f), float(f[0]), float(f[-1]))
        if key in seen:
            continue
        seen.add(key)
        idx = np.unique(np.r_[np.arange(0, len(f), 8), len(f) - 1, k0 - 1, k0, k0 + 1])
        rs, rl = net.terminations
        o = R.sweep(R.make_elems(net.elements), rs, rl, f[idx])[1]
        ref = _ref_s21(net, f[idx])
        worst = max(worst, float(np.max(np.abs(o - ref) / np.abs(ref))))
    assert len(seen) >= 14
    assert worst <= 1e-12, worst


def test_probe_premises(Q, monkeypatch):
    """Every GPU probe below exercises the path it is meant to: with its zero-width tolerances and its thresholds, the plan selects
    the transfer-function kernel with the expected denominator form and (kn, kd), accepts the expected specs for the fused margin,
    and the fused margin agrees with the unfused one within the gate.  Together the probes reach every numerator class of the
    plain-ladder translation units."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    rows = []
    for g in _geometries().values():
        v = float(_screen_db(g.net, g.f)[g.k0])
        rows.append((g.name, g.net, g.f, g.specs(g.k0, v), g.ztols(), g.hist, g.body, g.fused))
    w, f5, specs5, (k1, k2) = _geo_g5()
    db = _screen_db(w.net, f5)
    rows.append(("G5 cfg2, two stop bands", w.net, f5, specs5(db[k1], db[k2]), [(e, p, v, m, 0.0) for (e, p, v, m, _t) in w.tols], w.hist,
                 (9, 12), 0b110))
    bodies = set()
    for name, net, f, specs, tols, hist, (kn, ke), fused in rows:
        a = Q.plan_analyze(net, f, specs, tols, **hist)
        assert a["selected"], (name, a["reason"])
        assert a["den_form"] == ("none" if ke == 0 else "E"), (name, a["den_form"])
        assert (a["kn"], a["kd"] if ke else 0) == (kn, ke), (name, a["kn"], a["kd"])
        assert a["fused_specs"] == fused, (name, bin(a["fused_specs"]))
        assert 0.0 <= a["fused_err"] <= 1e-12, (name, a["fused_err"])
        bodies.add((kn, ke))
    assert len(bodies) >= 10, sorted(bodies)
    assert any(ke == 0 for _kn, ke in bodies)
    for lo, hi in ((2, 5), (6, 8), (9, 10)):
        assert any(lo <= kn <= hi for kn, _ke in bodies), (lo, hi, sorted(bodies))


# ---- GPU: decisive-point brackets with zero-width tolerances ------------------------------------------------------------
def _launch_size():
    """enough samples for the thread-per-sample kernel, with a remainder mod 32 (warp-per-sample), at an offset above 2^33"""
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    return 2 * sm * 4 * 128 + 32 * 37 + 19, (1 << 33) + 12345


def _run(Q, ctx, monkeypatch, kern, net, f, specs, tols, hist, fused, n, off, seed=3):
    if kern == "tf":
        monkeypatch.setenv("QO100NET_KERNEL", "tf")
    else:
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    plan = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **hist)
    try:
        plan.launch(off, n)
        r = plan.read()
        assert plan.kernel_name == ("qo_mc_ts_kernel" if kern == "auto" else "qo_mc_tf_kernel"), (kern, plan.kernel_name)
        if kern == "auto":
            assert plan.tf_info["fused_specs"] == fused, bin(plan.tf_info["fused_specs"])
    finally:
        plan.close()
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    assert r["n_total"] == n
    return r


def _bracket(Q, ctx, monkeypatch, geo, k, v, n, off):
    """thresholds at v + delta and v - delta on the bracketed spec: every sample (the nominal network) passes on one side and
    fails on the other, on both kernels"""
    mx = geo.is_max()
    for side in (1.0, -1.0):
        lim = v + side * DELTA
        want = n if (side < 0) == mx else 0
        for kern in ("auto", "tf"):
            r = _run(Q, ctx, monkeypatch, kern, geo.net, geo.f, geo.specs(k, lim), geo.ztols(), geo.hist, geo.fused, n, off)
            fails = [int(x) for x in r["fail_per_spec"]]
            assert fails[geo.spec] == want, "%s, k = %d (k mod 4 = %d), limit = v %s delta, %s kernel: %d of %d samples fail spec %d, expected %d" % (
                geo.name, k, k % 4, "+" if side > 0 else "-", kern, fails[geo.spec], n, geo.spec, want)
            assert all(x in (0, n) for x in fails), (geo.name, k, kern, fails)


def _sweep_edge(Q, ctx, monkeypatch, name, count=12):
    geo = _geometries()[name]
    n, off = _launch_size()
    pos = _positions(geo, count)
    assert {k % 4 for k, _v in pos} == {0, 1, 2, 3}
    for k, v in pos:
        _bracket(Q, ctx, monkeypatch, geo, k, v, n, off)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G1 cfg2", "G1 nf=4097", "G1 nf=4098", "G1 nf=4099"])
def test_bracket_stop_band_lower_edge_at_the_top_of_the_grid(Q, ctx, monkeypatch, name):
    """G1: config 2's MAX-dB stop band, its lower edge (the worst point) swept over 12 consecutive grid points -- every position
    of the edge in a 4-point group (a straddling group runs plain on byte masks) and every length of the fused run mod 3 (the
    12-point loop's tail); on grids whose last group carries padding too"""
    _sweep_edge(Q, ctx, monkeypatch, name)


@pytest.mark.gpu
def test_bracket_lower_stop_band_upper_edge_at_the_front_of_the_grid(Q, ctx, monkeypatch):
    """G2: the IF band-pass's lower stop band [0, f_k], histogram on the pass band: the fused run is at the front, its UPPER edge
    decides (the tail loop's last group, the 12-point loop's exit), and the plain runs after it must reload their grid values"""
    _sweep_edge(Q, ctx, monkeypatch, "G2 if_bpf [0, f_k]")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G3 butter5", "G3 butter7 par", "G3 butter11 par"])
def test_bracket_min_db_pass_band_upper_edge(Q, ctx, monkeypatch, name):
    """G3: a MIN-dB pass band (fused with neg = false) in the middle of the grid, plain runs on both sides, its upper edge swept"""
    _sweep_edge(Q, ctx, monkeypatch, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G4 butter7 par, two runs", "G4 cfg2, two runs"])
def test_bracket_spec_split_into_two_fused_runs(Q, ctx, monkeypatch, name):
    """G4: a second spec inside the fused band splits it into two fused runs with a plain run between them.  On the pass band
    the decisive point lies in the second fused run; on config 2's stop band in the first, with the second one after it"""
    _sweep_edge(Q, ctx, monkeypatch, name)


@pytest.mark.gpu
def test_bracket_two_fusable_specs_count_independently(Q, ctx, monkeypatch):
    """G5: config 2 with stop bands [13, 22 MHz] and [23 MHz, inf): both pass the gate, the larger runs fused, the other plain.
    Each bracketed at its own worst point, all four above / below combinations: each fail counter follows its own threshold"""
    w, f, specs, (k1, k2) = _geo_g5()
    n, off = _launch_size()
    zt = [(e, p, v, m, 0.0) for (e, p, v, m, _t) in w.tols]
    v1, v2 = _ref_db(w.net, f[k1]), _ref_db(w.net, f[k2])
    db = _screen_db(w.net, f)
    for k, v, s, nb in ((k1, v1, 1, k1 - 1), (k2, v2, 2, k2 - 1)):
        band = np.where(_in_band(f, specs(0.0, 0.0)[s]))[0]
        assert band[0] == k and np.all(db[band[1:]] <= v - 10 * DELTA) and _ref_db(w.net, f[nb]) > v + 2 * DELTA
    for s1 in (1.0, -1.0):
        for s2 in (1.0, -1.0):
            for kern in ("auto", "tf"):
                r = _run(Q, ctx, monkeypatch, kern, w.net, f, specs(v1 + s1 * DELTA, v2 + s2 * DELTA), zt, w.hist, 0b110, n, off)
                got = [int(x) for x in r["fail_per_spec"]]
                want = [0, n if s1 < 0 else 0, n if s2 < 0 else 0]
                assert got == want, ("G5", kern, s1, s2, got, want)
                assert r["n_pass"] == (n if s1 > 0 and s2 > 0 else 0)


_G6 = ["G6 butter3", "G6 butter7", "G6 butter9", "G6 butter11", "G6 butter3 par", "G6 butter5 par", "G6 butter6 par", "G6 butter9 par",
       "G6 cheby11 par"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", _G6)
def test_bracket_every_other_body_at_the_fused_run_ends(Q, ctx, monkeypatch, name):
    """G6: the bodies the probes above do not reach, once with the decisive point in the fused run's first group (a MAX-dB stop
    band's lower edge on a group boundary) and once in its last group (a MIN-dB pass band's upper edge at a group's end)"""
    n, off = _launch_size()
    geos = _geometries()
    for suffix, residue in ((" stop", 0), (" pass", 3)):
        geo = geos[name + suffix]
        k, v = next((k, v) for k, v in _positions(geo, 12) if k % 4 == residue)
        _bracket(Q, ctx, monkeypatch, geo, k, v, n, off)


# ---- GPU: random tolerances at the same geometries, the whole launch against the oracle ----------------------------------
def _parity_case(name):
    """(net, grid <= 1 024 points, spec list, tolerances, histogram spec, expected fused mask) at one edge position"""
    import qo100net as Q
    from qo100net import workloads as W
    f2 = W.cfg2().f[::4]
    if name == "G5":
        w, f, specs, (k1, k2) = _geo_g5(f2)
        return w.net, f, specs(0.0, 0.0), w.tols, 0, 0b110
    geo = {"G1": lambda: _geo_cfg2("G1", f2), "G2": lambda: _geo_ifbpf(700), "G3": lambda: _geometries()["G3 butter7 par"],
           "G4": lambda: _geometries()["G4 butter7 par, two runs"],
           "G4 cfg2": lambda: _geo_cfg2("G4 cfg2", f2, [(Q.SPEC_S21_MAX_DB, 20e6, 25e6, 1.0)])}[name]()
    return geo.net, geo.f, geo.specs(geo.k0 + 1, 0.0), geo.tols, geo.hist["hist_spec"], geo.fused


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G1", "G2", "G3", "G4", "G4 cfg2", "G5"])
def test_random_tolerances_default_and_warp_per_sample_kernels_equal_the_oracle(Q, R, ctx, monkeypatch, name):
    """Real tolerances, every threshold at the median of the samples' in-band worst value (FULL_S pre-run of 2 000 samples), so
    that every fail counter is near n / 2: the default kernel (fused), QO100NET_KERNEL=tf and the oracle give the same n_pass,
    fail_per_spec and histogram over the whole launch"""
    net, f, specs, tols, hs, fused = _parity_case(name)
    s21 = ctx.mc_run(net, f, [], 5, 2000, tols, mode=Q.MODE_FULL_S)["s"][1]
    db = 20 * np.log10(np.abs(s21))
    lim, worst = [], []
    for sp in specs:
        band = _in_band(f, sp)
        x = db[:, band].max(axis=1) if sp[0] == Q.SPEC_S21_MAX_DB else db[:, band].min(axis=1)
        worst.append(x)
        lim.append((sp[0], sp[1], sp[2], float(np.median(x))))
    hist = dict(hist_bins=64, hist_spec=hs, hist_lo=float(np.quantile(worst[hs], 0.02)), hist_hi=float(np.quantile(worst[hs], 0.98)))
    n, off = _launch_size()
    seed = 0x5EED0F00 + len(name)
    a = _run(Q, ctx, monkeypatch, "auto", net, f, lim, tols, hist, fused, n, off, seed=seed)
    b = _run(Q, ctx, monkeypatch, "tf", net, f, lim, tols, hist, fused, n, off, seed=seed)
    rs, rl = net.terminations
    o = R.mc_run(R.make_elems(net.elements), rs, rl, f, lim, R.mc_cfg(seed, n, tols, sample_offset=off, **hist), nthreads=8)
    for r, who in ((a, "default"), (b, "tf")):
        assert r["n_pass"] == o["n_pass"], (name, who, r["n_pass"], o["n_pass"])
        assert np.array_equal(r["fail_per_spec"], o["fail_per_spec"]), (name, who, r["fail_per_spec"], o["fail_per_spec"])
        assert np.array_equal(r["hist"], o["hist"]), (name, who)
    for s in range(len(lim)):
        assert 0.4 * n < int(o["fail_per_spec"][s]) < 0.6 * n, (name, s, o["fail_per_spec"])
