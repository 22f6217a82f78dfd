"""Generate tests/golden/* from a checkout of the upstream qo-100-tools tree (the tests need only the fixtures, not the tree).

  python tools/make_golden.py [<qo-100-tools checkout>]      (default: $QO100_REFERENCE)

Writes
  tests/golden/pa_lpf_dat.npz   -- util/pa-lpf-simulation/pa-lpf-simulation.dat:5-35017 (all 5000 points)
  tests/golden/networks.json    -- element lists of every rf-tools SVG / Qucs .sch in the tree,
                                   as read by the product loader (qo_net_load_*), + .trc contents
  tests/golden/touchstone.npz   -- the three Touchstone files of the tree (util/pa-bias-simulation/11SQ39N.S2P,
                                   util/preamp-bias-simulation/06HP47N.s2p, docs/pa-driver/pa_20W_vdd_32V_idq_180mA.s2p)
                                   parsed by an independent numpy parser (python tools/make_golden.py <checkout> touchstone)
  tests/golden/pa_bias_dat.npz  -- util/pa-bias-simulation/pa-bias-simulation.dat:1-85035 (5-port S entries, 5000 points)
  tests/golden/rftools_png_curves.npz -- the S21 / S11 curves of the reference's three rf-tools plots (util/if-bandpass-filter/
                                   bokeh_plot.png, util/gpsdo-ouput-filters/10M/bokeh_plot.png, docs/upconverter/
                                   upconverter-lol-filter.png) as pixel coordinates, with the axis calibration read from the
                                   tick marks (python tools/make_golden.py <checkout> png_curves)
  tests/golden/appendix_b.json  -- 40-digit mpmath evaluation of the textbook ladder / coupled-line
                                   equations (SURVEY App. B) at the frequencies the survey tabulates;
                                   an implementation independent of both the oracle and the product.
"""
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "qo-100-tools_b200", "python"))
import qo100net as Q  # noqa: E402

REF = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("QO100_REFERENCE", "")
OUT = os.path.join(ROOT, "tests", "golden")

SVGS = ["util/if-bandpass-filter/schematic.svg", "util/gpsdo-ouput-filters/10M/schematic.svg",
        "docs/gpsdo-filters/15M.svg", "docs/gpsdo-filters/40M.svg", "docs/gpsdo-filters/60M.svg",
        "docs/upconverter/upconverter-lol-filter.svg"]
SCHS = ["util/pa-lpf-simulation/pa-lpf-simulation.sch"]
TRCS = ["util/directional-couplers/dir_cpl_2.4g_20dB.trc", "util/directional-couplers/dir_cpl_2.4g_35dB.trc",
        "util/directional-couplers/dir_cpl_2.4g_35dB_pa_250W.trc", "util/directional-couplers/dir_cpl_525m_20dB.trc"]


def parse_dat(path):
    out, cur = {}, None
    for ln in open(path):
        ln = ln.strip()
        m = re.match(r"<(indep|dep) (\S+)", ln)
        if m:
            cur = m.group(2)
            out[cur] = []
            continue
        if ln.startswith("</") or ln.startswith("<Qucs"):
            cur = None
            continue
        if cur is None or not ln:
            continue
        m = re.match(r"([+-][0-9.e+-]+?)([+-])j([0-9.e+-]+)$", ln)
        out[cur].append(complex(float(m.group(1)), float(m.group(2) + m.group(3))) if m else float(ln))
    return {k: np.array(v) for k, v in out.items()}


def golden_dat():
    d = parse_dat(os.path.join(REF, "util/pa-lpf-simulation/pa-lpf-simulation.dat"))
    np.savez_compressed(os.path.join(OUT, "pa_lpf_dat.npz"), frequency=d["frequency"], zw=d["zw"],
                        S11_dB=d["S11_dB"], S21_dB=d["S21_dB"], S11=d["S[1,1]"], S12=d["S[1,2]"],
                        S21=d["S[2,1]"], S22=d["S[2,2]"])
    print("pa_lpf_dat.npz:", len(d["frequency"]), "points")


def golden_networks():
    nets = {}
    for p in SVGS:
        n = Q.Net.from_rftools_svg(os.path.join(REF, p))
        rs, rl = n.terminations
        nets[p] = dict(rs=rs, rl=rl, title=n.title, elements=[[k, pp] for k, pp in n.elements])
    for p in SCHS:
        n = Q.Net.from_qucs_sch(os.path.join(REF, p))
        rs, rl = n.terminations
        nets[p] = dict(rs=rs, rl=rl, sweep=list(Q.qucs_sch_sweep(os.path.join(REF, p))),
                       elements=[[k, pp] for k, pp in n.elements])
    for p in TRCS:
        nets[p] = Q.load_trc(os.path.join(REF, p))
    json.dump(nets, open(os.path.join(OUT, "networks.json"), "w"), indent=1)
    print("networks.json:", len(nets), "entries")


def golden_appendix_b():
    import mpmath as mp
    mp.mp.dps = 40
    J = mp.mpc(0, 1)

    def chain(elems, rs, rl, f):
        w = 2 * mp.pi * mp.mpf(f)
        A, B, Cc, D = mp.mpc(1), mp.mpc(0), mp.mpc(0), mp.mpc(1)

        def ser(z):
            nonlocal B, D
            B, D = B + A * z, D + Cc * z

        def sh(y):
            nonlocal A, Cc
            A, Cc = A + B * y, Cc + D * y

        for kind, p in elems:
            p = [mp.mpf(repr(x)) if not isinstance(x, str) else mp.mpf(x) for x in p]
            if kind in (Q.SER_L, Q.SHUNT_L):
                L, R, Cp = p[0], p[1], p[2]
                z = (R + J * w * L) / (1 - w * w * L * Cp + J * w * R * Cp)
                ser(z) if kind == Q.SER_L else sh(1 / z)
            elif kind in (Q.SER_C, Q.SHUNT_C):
                Cv, R, Ls = p[0], p[1], p[2]
                z = R + J * w * Ls + 1 / (J * w * Cv)
                ser(z) if kind == Q.SER_C else sh(1 / z)
            elif kind == Q.SER_LC_SER:
                ser(J * w * p[0] + 1 / (J * w * p[1]))
            elif kind == Q.SER_LC_PAR:
                ser(1 / (J * w * p[1] + 1 / (J * w * p[0])))
            elif kind == Q.SHUNT_LC_SER:
                sh(1 / (J * w * p[0] + 1 / (J * w * p[1])))
            elif kind == Q.SHUNT_LC_PAR:
                sh(J * w * p[1] + 1 / (J * w * p[0]))
            elif kind == Q.CPL_THRU:
                z0e, z0o, ae, ao, f0, zt = p
                te, to = ae * mp.pi / 180 * mp.mpf(f) / f0, ao * mp.pi / 180 * mp.mpf(f) / f0
                # 4-port Z matrix of the ideal coupled pair (SURVEY B.4), ports 3,4 loaded with Zt
                cot, csc = (lambda x: mp.cos(x) / mp.sin(x)), (lambda x: 1 / mp.sin(x))
                z11 = -J / 2 * (z0e * cot(te) + z0o * cot(to)); z12 = -J / 2 * (z0e * csc(te) + z0o * csc(to))
                z13 = -J / 2 * (z0e * cot(te) - z0o * cot(to)); z14 = -J / 2 * (z0e * csc(te) - z0o * csc(to))
                Zaa = mp.matrix([[z11, z12], [z12, z11]]); Zab = mp.matrix([[z13, z14], [z14, z13]])
                Zr = Zaa - Zab * mp.inverse(Zaa + zt * mp.eye(2)) * Zab
                a, b, c, d = Zr[0, 0] / Zr[1, 0], (Zr[0, 0] * Zr[1, 1] - Zr[0, 1] * Zr[1, 0]) / Zr[1, 0], 1 / Zr[1, 0], Zr[1, 1] / Zr[1, 0]
                A, B, Cc, D = A * a + B * c, A * b + B * d, Cc * a + D * c, Cc * b + D * d
            else:
                raise ValueError(kind)
        rs, rl = mp.mpf(rs), mp.mpf(rl)
        den = A * rl + B + Cc * rs * rl + D * rs
        s21 = 2 * mp.sqrt(rs * rl) / den
        s11 = (A * rl + B - Cc * rs * rl - D * rs) / den
        return s11, s21

    def dec(elems):
        # nominal values as exact decimals where the SVG prints decimals
        return [(k, [repr(x) for x in p]) for k, p in elems]

    nets = json.load(open(os.path.join(OUT, "networks.json")))
    cases = {}

    def add(name, elems, rs, rl, freqs):
        rows = []
        for f in freqs:
            s11, s21 = chain(elems, rs, rl, f)
            rows.append(dict(f=float(f), s21=[mp.nstr(s21.real, 25), mp.nstr(s21.imag, 25)],
                             s11=[mp.nstr(s11.real, 25), mp.nstr(s11.imag, 25)],
                             s21_db=mp.nstr(20 * mp.log10(abs(s21)), 20), s11_db=mp.nstr(20 * mp.log10(abs(s11)), 20)))
        cases[name] = dict(rs=rs, rl=rl, elements=[[k, [float(x) for x in p]] for k, p in elems], rows=rows)

    def svg_elems(key):
        return [(k, p) for k, p in nets[key]["elements"]], nets[key]["rs"], nets[key]["rl"]

    e, rs, rl = svg_elems(SVGS[0]); add("if_bpf", e, rs, rl, ["85714285.714", "300e6", "387298334.621", "500e6", "1e9", "1.75e9"])
    e, rs, rl = svg_elems(SVGS[1]); add("gpsdo_10m", e, rs, rl, ["4e6", "10e6", "11e6", "20e6", "30e6", "62.5e6"])
    e, rs, rl = svg_elems(SVGS[2]); add("gpsdo_15m", e, rs, rl, ["5e6", "10e6", "15e6", "17e6", "20e6", "30e6", "60e6"])
    e, rs, rl = svg_elems(SVGS[3]); add("gpsdo_40m", e, rs, rl, ["10e6", "40e6", "45e6", "60e6", "100e6"])
    e, rs, rl = svg_elems(SVGS[4]); add("gpsdo_60m", e, rs, rl, ["10e6", "60e6", "70e6", "90e6", "150e6"])
    e, rs, rl = svg_elems(SVGS[5]); add("lol_hpf", e, rs, rl, ["1e9", "1.9e9", "2.1e9", "2.4e9", "3e9", "6e9"])

    # synthesised 11th-order 0.1 dB Chebyshev (B.3) in mpmath
    def cheby_g(n, ripple):
        beta = mp.log(mp.coth(mp.mpf(ripple) * mp.log(10) / 40))
        gam = mp.sinh(beta / (2 * n))
        a = [mp.sin((2 * k - 1) * mp.pi / (2 * n)) for k in range(1, n + 1)]
        b = [gam ** 2 + mp.sin(k * mp.pi / n) ** 2 for k in range(1, n + 1)]
        g = [2 * a[0] / gam]
        for k in range(2, n + 1):
            g.append(4 * a[k - 2] * a[k - 1] / (b[k - 2] * g[-1]))
        return g

    def ladder(g, fc, z0, parasitic):
        wc = 2 * mp.pi * mp.mpf(fc)
        out = []
        for k, gk in enumerate(g):
            if k % 2 == 0:
                L = gk * z0 / wc
                R, Cp = (wc * L / 60, 1 / ((2 * mp.pi * 30 * mp.mpf(fc)) ** 2 * L)) if parasitic else (0, 0)
                out.append((Q.SER_L, [mp.nstr(L, 30), mp.nstr(R, 30), mp.nstr(Cp, 30)]))
            else:
                Cv = gk / (z0 * wc)
                R, Ls = (mp.mpf("0.1"), 1 / ((2 * mp.pi * 50 * mp.mpf(fc)) ** 2 * Cv)) if parasitic else (0, 0)
                out.append((Q.SHUNT_C, [mp.nstr(Cv, 30), mp.nstr(R, 30), mp.nstr(Ls, 30)]))
        return out

    g11 = cheby_g(11, "0.1")
    cases["cheby11_g"] = [mp.nstr(x, 25) for x in g11]
    cases["butter11_g"] = [mp.nstr(2 * mp.sin((2 * k - 1) * mp.pi / 22), 25) for k in range(1, 12)]
    fc = "10e6"
    add("cheby11_ideal", ladder(g11, fc, 50, False), 50, 50, [mp.mpf(fc) * mp.mpf(x) for x in ["0.25", "0.5", "0.9", "1.0", "1.05", "1.2", "2.0", "4.0"]])
    add("cfg2_nominal", ladder(g11, fc, 50, True), 50, 50, [mp.mpf(fc) * mp.mpf(x) for x in ["0.4", "0.5", "0.9", "0.95", "1.0", "1.05", "1.3", "2.0", "6.25"]])
    cpl = [(Q.CPL_THRU, ["55.2771", "45.2267", "95.4225", "95.4225", "2.4e9", "50"])]
    add("coupler_20db", cpl, 50, 50, ["70e6", "525e6", "1.2e9", "2.4e9", "3.2e9", "4e9"])
    add("cfg5_nominal", cpl + ladder(g11, "3e9", 50, True), 50, 50, ["70e6", "1.2e9", "2.3e9", "2.4e9", "2.5e9", "3e9", "3.9e9", "4e9"])
    json.dump(cases, open(os.path.join(OUT, "appendix_b.json"), "w"), indent=1)
    print("appendix_b.json:", len(cases), "cases")


S2PS = {"11SQ39N": "util/pa-bias-simulation/11SQ39N.S2P", "06HP47N": "util/preamp-bias-simulation/06HP47N.s2p",
        "pa_20W": "docs/pa-driver/pa_20W_vdd_32V_idq_180mA.s2p"}


def parse_s2p(path):
    """Independent (numpy) Touchstone v1 2-port parser -- NOT the product loader, so that the fixture checks it."""
    scale, fmt, z0, rows = 1e9, "MA", 50.0, []
    for ln in open(path, errors="replace"):
        ln = ln.split("!")[0].strip()
        if not ln:
            continue
        if ln.startswith("#"):
            t = ln[1:].upper().split()
            for i, tok in enumerate(t):
                if tok in ("HZ", "KHZ", "MHZ", "GHZ"):
                    scale = {"HZ": 1.0, "KHZ": 1e3, "MHZ": 1e6, "GHZ": 1e9}[tok]
                elif tok in ("MA", "DB", "RI"):
                    fmt = tok
                elif tok == "R":
                    z0 = float(t[i + 1])
            continue
        rows += [float(x) for x in ln.split()]
    a = np.array(rows).reshape(-1, 9)
    x, y = a[:, 1::2], a[:, 2::2]
    if fmt == "RI":
        s = x + 1j * y
    else:
        s = (10 ** (x / 20) if fmt == "DB" else x) * np.exp(1j * np.deg2rad(y))
    return a[:, 0] * scale, s, z0          # columns of s: S11 S21 S12 S22


def golden_pa_bias():
    """util/pa-bias-simulation/pa-bias-simulation.dat:1-85035 -- the 5-port bias network (row N4)."""
    d = parse_dat(os.path.join(REF, "util/pa-bias-simulation/pa-bias-simulation.dat"))
    keys = {k: v for k, v in d.items()}
    np.savez_compressed(os.path.join(OUT, "pa_bias_dat.npz"), **{k.replace("[", "").replace("]", "").replace(",", "_"): v for k, v in keys.items()})
    print("pa_bias_dat.npz:", len(d["frequency"]), "points,", len(keys), "variables")


def golden_touchstone():
    out = {}
    for key, p in S2PS.items():
        f, s, z0 = parse_s2p(os.path.join(REF, p))
        out[key + "_f"], out[key + "_s"], out[key + "_z0"] = f, s, np.array(z0)
        print("touchstone", key, len(f), "points", f[0], f[-1])
    np.savez_compressed(os.path.join(OUT, "touchstone.npz"), **out)


# rf-tools.com plots (Bokeh): S21 in blue against the left axis (0 .. -80 dB), S11 in red against the right axis (0 .. -40 dB),
# logarithmic frequency axis.  (labelled major tick pixel column, frequency) pairs read from each image's tick labels.
PNGS = {"if_bpf": ("util/if-bandpass-filter/bokeh_plot.png", "util/if-bandpass-filter/schematic.svg",
                   [(412, 500e6), (555, 1e9), (639, 1.5e9)]),
        "gpsdo_10m": ("util/gpsdo-ouput-filters/10M/bokeh_plot.png", "util/gpsdo-ouput-filters/10M/schematic.svg",
                      [(256, 10e6), (412, 20e6), (503, 30e6), (568, 40e6), (619, 50e6), (660, 60e6)]),
        "lol_hpf": ("docs/upconverter/upconverter-lol-filter.png", "docs/upconverter/upconverter-lol-filter.svg",
                    [(295, 1e9), (451, 2e9), (543, 3e9), (608, 4e9), (658, 5e9)])}


def golden_png_curves():
    """Pixel coordinates of the plotted curves + axis calibration.  Nothing is computed with the product or the oracle here:
    the fixture is the reference's picture, reduced to the pixels of its two curves."""
    from PIL import Image
    out = {}
    for key, (png, svg, anchors) in PNGS.items():
        im = np.array(Image.open(os.path.join(REF, png)).convert("RGB")).astype(int)
        r, g, b = im[..., 0], im[..., 1], im[..., 2]
        blue = (b > 150) & (r < 80) & (g > 90) & (g < 160)          # Bokeh's default blue #1f77b4
        red = (r > 200) & (g < 60) & (b < 60)
        dark = (r < 90) & (g < 90) & (b < 90)
        ax_l, ax_r = int(np.nonzero(blue.sum(0) > 300)[0][0]), int(np.nonzero(red.sum(0) > 300)[0][0])      # the two y axes
        ax_b = int(np.nonzero(dark.sum(1) > 300)[0][0])                                                       # the frequency axis
        yt = np.nonzero(blue[:, ax_l - 5])[0]                       # major ticks of the S21 axis: 0, -10, ... -80 dB
        assert len(yt) == 9 and yt[-1] == ax_b, (key, yt, ax_b)
        maj = [int(x) for x in np.nonzero(dark[ax_b + 4, :])[0]]   # labelled (long) ticks of the frequency axis
        assert all(a[0] in maj for a in anchors), (key, maj, anchors)

        def pts(mask):
            ys, xs = np.nonzero(mask[:, ax_l + 2:ax_r - 1])
            xs = xs + ax_l + 2
            keep = (ys >= yt[0] - 1) & (ys <= ax_b - 1)
            return np.stack([xs[keep], ys[keep]], 1).astype(np.int16)
        out[key + "_s21_px"], out[key + "_s11_px"] = pts(blue), pts(red)
        out[key + "_xticks"] = np.array(anchors, dtype=float)                   # (pixel column, Hz)
        out[key + "_frame"] = np.array([ax_l, ax_r, yt[0], ax_b], dtype=float)   # left, right, row of 0 dB, row of -80 / -40 dB
        print("png", key, png, "S21 px", len(out[key + "_s21_px"]), "S11 px", len(out[key + "_s11_px"]), "frame", out[key + "_frame"])
    np.savez_compressed(os.path.join(OUT, "rftools_png_curves.npz"), **out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if len(sys.argv) > 2 and sys.argv[2] == "png_curves":
        golden_png_curves()
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[2] == "touchstone":
        golden_touchstone()
        sys.exit(0)
    if len(sys.argv) > 2 and sys.argv[2] == "pa_bias":
        golden_pa_bias()
        sys.exit(0)
    golden_dat()
    golden_networks()
    golden_appendix_b()
    golden_touchstone()
    golden_pa_bias()
    golden_png_curves()
