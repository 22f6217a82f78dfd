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
