"""What the reference tree itself holds for the LUMPED side of the path (SURVEY 8a rows a8-a10), turned into numbers:

  a8   rf-tools ladders: the three plots the tree ships (util/if-bandpass-filter/bokeh_plot.png, util/gpsdo-ouput-filters/
       10M/bokeh_plot.png, docs/upconverter/upconverter-lol-filter.png) reduced to the pixels of their S21 / S11 curves
       (tests/golden/rftools_png_curves.npz, tools/make_golden.py png_curves).  The model curve drawn in the same axes must pass
       through those pixels: every curve pixel within 1.5 px of the model (1 px = 0.17 dB of S21, 0.086 dB of S11, 0.49 % in
       frequency).  A 3 % change of ONE element moves the S11 curve by 10-15 px, so this pins the element models.
       Plus the edge values SURVEY 0.5 read off the plots and the spec lines of the SVGs (schematic.svg:221-222, :235-237).
  a10  coupled line: the identities the .trc files imply (util/directional-couplers/dir_cpl_*.trc:18-20):
       k = (Z0e - Z0o)/(Z0e + Z0o) = 0.100000 <-> coupling -20.000 dB at theta = 90 deg and -20.04 dB at 2.4 GHz,
       sqrt(Z0e Z0o) = 50.0000 <-> matched.
  a9   lumped L / C with ESR / SRF parasitics: pinned TRANSITIVELY -- the nodal solver reproduces the reference's
       util/pa-bias-simulation/pa-bias-simulation.dat (tests/test_nodal.py), and here the cascade evaluation must equal the nodal
       evaluation of the same parasitic ladder.

  N3/N4 the preamp bias network (util/preamp-bias-simulation): no dataset upstream, but the schematic stores its diagram markers and
       the shipped plot prints their values -- six reference-held numbers for a 5-port network with a measured inductor.

CPU tests run the oracle; the `gpu` tests run the product through the C-ABI on the same fixtures."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REFERENCE, ROOT, png_curve_distance, relerr

PNG_CASES = [("if_bpf", "util/if-bandpass-filter/schematic.svg"),
             ("gpsdo_10m", "util/gpsdo-ouput-filters/10M/schematic.svg"),
             ("lol_hpf", "docs/upconverter/upconverter-lol-filter.svg")]
# (case, f [Hz], trace, dB, tolerance dB): values read off the reference plots (SURVEY 0.5, BASELINE.md 1) and the spec lines
PLOT_VALUES = [("if_bpf", 300e6 / 3.5, "s21", -54.6, 0.15), ("if_bpf", 500e6 * 3.5, "s21", -52.2, 0.15),
               ("gpsdo_10m", 4e6, "s11", -8.8, 0.15), ("gpsdo_10m", 4e6, "s21", -0.6, 0.15),
               ("gpsdo_10m", 28.0e6, "s21", -80.0, 0.8),           # the curve leaves the plot at ~28 MHz (5.8 px per dB, steep)
               ("if_bpf", 300e6, "s21", -3.0, 2.4), ("if_bpf", 500e6, "s21", -3.0, 1.6)]    # "Cutoff 300 / 500 MHz" of a realised Butterworth


def _limits(key, trace):
    # the notch tips of the elliptic high-pass are drawn from the tool's own frequency samples: looser there
    return (5.0, 2.0) if (key, trace) == ("lol_hpf", "s21") else (1.5, 1.3)


def _check_curves(png_curves, key, sweep):
    d = png_curve_distance(png_curves, key, sweep)
    for trace in ("s21", "s11"):
        mx, p99, cov = d[trace]
        lim_max, lim_p99 = _limits(key, trace)
        assert mx <= lim_max and p99 <= lim_p99, (key, trace, d[trace])
        assert cov >= 0.75, (key, trace, cov)
    return d


def _oracle_sweep(R, golden_nets, svg):
    n = golden_nets[svg]
    e = R.make_elems([(k, p) for k, p in n["elements"]])

    def sweep(f):
        o = R.sweep(e, n["rs"], n["rl"], np.ascontiguousarray(f))
        return o[0], o[1]
    return sweep


@pytest.mark.parametrize("key,svg", PNG_CASES)
def test_rftools_plots_pin_the_oracle(R, golden_nets, png_curves, key, svg):
    _check_curves(png_curves, key, _oracle_sweep(R, golden_nets, svg))


def test_rftools_plot_is_sensitive_to_three_percent(R, golden_nets, png_curves):
    """The pin has teeth: 3 % on one element of the IF band-pass fails it."""
    n = golden_nets["util/if-bandpass-filter/schematic.svg"]
    el = [(k, list(p)) for k, p in n["elements"]]
    el[1][1][0] *= 1.03
    e = R.make_elems(el)
    d = png_curve_distance(png_curves, "if_bpf", lambda f: R.sweep(e, n["rs"], n["rl"], np.ascontiguousarray(f))[:2])
    assert d["s11"][0] > 8.0


def test_plot_values_oracle(R, golden_nets):
    svgs = dict(PNG_CASES)
    for key, f, trace, db, tol in PLOT_VALUES:
        s11, s21 = _oracle_sweep(R, golden_nets, svgs[key])(np.array([f]))
        got = 20 * np.log10(abs((s21 if trace == "s21" else s11)[0]))
        assert abs(got - db) <= tol, (key, f, trace, got, db)


def _coupler_checks(sweep, t):
    """t: one .trc record (z0e, z0o, ang at f0).  sweep(elements, f) -> (s11, s21) of the through path, far ports in 50 Ohm."""
    k = (t["z0e"] - t["z0o"]) / (t["z0e"] + t["z0o"])
    el = [(12, [t["z0e"], t["z0o"], t["ang"], t["ang"], t["f0"], 50.0])]
    f90 = t["f0"] * 90.0 / t["ang"]                       # quarter wave
    s11, s21 = sweep(el, np.array([f90, t["f0"]]))
    # what does not arrive at the through port and is not reflected went to the coupled / isolated ports
    cpl_db = 10 * np.log10(1.0 - np.abs(s21) ** 2 - np.abs(s11) ** 2)
    assert abs(cpl_db[0] - 20 * np.log10(k)) < 2e-4                        # theta = 90 deg: coupling = k exactly
    th = np.radians(t["ang"])
    c_f0 = k * np.sin(th) / np.sqrt(1 - (k * np.cos(th)) ** 2)             # textbook coupled-line coupling at theta
    assert abs(cpl_db[1] - 20 * np.log10(c_f0)) < 2e-4
    assert np.all(20 * np.log10(np.abs(s11)) < -80.0)                      # sqrt(Z0e Z0o) = 50.000
    return k, cpl_db


def test_trc_identities_oracle(R, golden_nets):
    def sweep(el, f):
        o = R.sweep(R.make_elems(el), 50.0, 50.0, f)
        return o[0], o[1]
    t = golden_nets["util/directional-couplers/dir_cpl_2.4g_20dB.trc"]
    k, cpl = _coupler_checks(sweep, t)
    assert abs(k - 0.100000) < 5e-7 and abs(cpl[0] + 20.000) < 1e-4 and abs(cpl[1] + 20.0386) < 1e-3      # SURVEY App. B.4: -20.0385520502
    assert abs(np.sqrt(t["z0e"] * t["z0o"]) - 50.0) < 1e-4
    k35, cpl35 = _coupler_checks(sweep, golden_nets["util/directional-couplers/dir_cpl_2.4g_35dB.trc"])
    assert abs(20 * np.log10(k35) + 35.000) < 2e-3 and abs(cpl35[0] + 35.000) < 2e-3
    _coupler_checks(sweep, golden_nets["util/directional-couplers/dir_cpl_525m_20dB.trc"])


def test_ref_workloads_equal_product_workloads(Q, W):
    """bench.py's reference arm builds configs 2 and 5 with the oracle alone; they must be the product's bundles bit for bit."""
    from oracle import ref_workloads as RW
    for a, b in ((RW.cfg2(), W.cfg2()), (RW.cfg5(), W.cfg5())):
        eb = b.net.elements
        assert len(a.elems) == len(eb)
        for (k1, p1), (k2, p2) in zip(a.elems, eb):
            assert k1 == k2 and list(p1) == list(p2)
        assert np.array_equal(a.f, b.f) and (a.rs, a.rl) == tuple(b.net.terminations)
        assert [tuple(x) for x in a.specs] == [tuple(x) for x in b.specs]
        assert [tuple(x) for x in a.tols] == [tuple(x) for x in b.tols]
        assert a.hist == b.hist and a.seed == b.seed and a.name == b.name


def test_reference_arm_never_loads_the_product():
    """`bench.py --impl reference` (one short step): the JSON line carries the host core count, and neither the product package
    nor libqo100net.so is mapped by that process.  OMP_NUM_THREADS=1 in the environment (torchrun's default) must not matter."""
    code = ("import sys, os, json, io, contextlib\n"
            "sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '1']\n"
            "import bench\n"
            "bench.REF_SAMPLES_PER_STEP = 400\n"
            "bench.main()\n"
            "maps = open('/proc/self/maps').read()\n"
            "sys.stderr.write('PRODUCT_LOADED=%d\\n' % int('libqo100net' in maps or 'qo100net' in sys.modules))\n"
            "sys.stderr.write('ORACLE_LOADED=%d\\n' % int('libqo100ref' in maps))\n")
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"]
    assert "PRODUCT_LOADED=0" in r.stderr and "ORACLE_LOADED=1" in r.stderr, r.stderr[-500:]


# ---- N3 / N4: the preamp bias network, pinned by the markers of the reference's own plot -------------------------------------
# util/preamp-bias-simulation: the Qucs dataset is missing upstream (.MISSING_LARGE_BLOBS), but the schematic carries the
# diagram markers (preamp-bias-simulation.sch:74,76,81,86,91: frequencies 2.38924 / 2.40324 / 2.40724 GHz, grid points of the
# 5000-point 1 MHz .. 10 GHz sweep of :23) and the tree ships the rendered plot with their values
# (preamp-bias-simulation.png): Gain_S21db -0.0645, Gain_S31db -69.5, XinA -0.0744, RinA 1.02, S[1,1] 0.00983 - j0.0365,
# Z[1,1] 50.9 - j3.72 (equations :24, :28).  Three significant digits each: that is the tolerance.
PREAMP_MARKERS = [(2.38924e9, "Gain_S21db", -0.0645, 0.5e-4), (2.40324e9, "Gain_S31db", -69.5, 0.05), (2.38924e9, "XinA", -0.0744, 0.5e-4),
                  (2.40724e9, "RinA", 1.02, 0.005), (2.40324e9, "S11re", 0.00983, 0.5e-5), (2.40324e9, "S11im", -0.0365, 0.5e-4),
                  (2.40324e9, "Z11re", 50.9, 0.05), (2.40324e9, "Z11im", -3.72, 0.005)]
NB_R, NB_C, NB_SBLOCK = 1, 3, 5


def preamp_netlist():
    """preamp-bias-simulation.sch read by hand: (kind, nodes, params) branches, node count, (node, Z0) ports in Pac-number order.
    Nodes: 1 = P1 (:30), 2 = P2 (:34), 3 = P3 (:21), 4 = P4 (:31), 5 = P5 (:40), 6 = R9-C1, 7 = inductor output, 8 = C9-R1, 9 = R10-C5."""
    br = [(NB_R, [1, 6], [0.6]), (NB_C, [6, 2], [12e-12]),                       # R9 :36, C1 :35  (DC block P1 -> P2)
          (NB_SBLOCK, [1, 7, 0], [0, 1, 50.0]),                                   # L_0603HP47N :32 (SPfile "polar" "linear", reference pin grounded :19)
          (NB_R, [7, 3], [1000.0]),                                              # R11 :27 -> P3
          (NB_C, [7, 8], [22e-6]), (NB_R, [8, 0], [10.0]),                        # C9 :41, R1 :26 to ground :22
          (NB_R, [4, 9], [0.6]), (NB_C, [9, 5], [12e-12])]                        # R10 :38, C5 :37 (the second, unconnected path P4 -> P5)
    return br, 9, [(1, 50.0), (2, 50.0), (3, 50.0), (4, 50.0), (5, 50.0)]


def _preamp_quantities(S):
    s11 = S[0, 0]
    zin = (1 + s11) / (1 - s11)
    return {"Gain_S21db": 20 * np.log10(abs(S[1, 0])), "Gain_S31db": 20 * np.log10(abs(S[2, 0])), "XinA": zin.imag, "RinA": zin.real,
            "S11re": s11.real, "S11im": s11.imag, "Z11re": 50.0 * zin.real, "Z11im": 50.0 * zin.imag}


def _check_preamp_markers(sweep):
    grid = np.linspace(1e6, 1e10, 5000)
    for fm, name, val, tol in PREAMP_MARKERS:
        k = int(np.argmin(np.abs(grid - fm)))
        assert abs(grid[k] - fm) < 1e4                                    # the markers sit on points of the reference's own grid
        got = _preamp_quantities(sweep(np.array([grid[k]]))[0])[name]
        assert abs(got - val) <= tol, (name, fm, got, val)


def test_preamp_bias_plot_markers_pin_the_oracle(R, golden_s2p):
    """Rows N3 + N4 on a second reference network: the oracle's nodal solve with the measured 0603HP-47N inductor
    (util/preamp-bias-simulation/06HP47N.s2p, polar interpolation) reproduces every marker value of the reference's plot, and the
    isolation notch the plot shows at the inductor's self-resonance (Gain_S31db ~ -94 dB between 3.4 and 3.5 GHz)."""
    br, nn, ports = preamp_netlist()
    fd, sd = golden_s2p["06HP47N_f"], golden_s2p["06HP47N_s"]
    R.sblock_clear()
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], float(golden_s2p["06HP47N_z0"]))
    _check_preamp_markers(lambda f: R.nodal_sweep(br, nn, ports, f))
    f = np.linspace(1e6, 1e10, 5000)
    g31 = 20 * np.log10(np.abs(R.nodal_sweep(br, nn, ports, f)[:, 2, 0]))
    k = int(np.argmin(g31))
    assert 3.3e9 < f[k] < 3.6e9 and -100.0 < g31[k] < -88.0, (f[k], g31[k])
    assert abs(g31[-1] - (-58.0)) < 1.5                                   # the trace ends at ~ -58 dB at 10 GHz
    R.sblock_clear()


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="the upstream qo-100-tools files are not in this repository: set QO100_REFERENCE to a checkout")
def test_preamp_bias_netlister_equals_hand_netlist(Q):
    """qo_nodal_load_qucs_sch on the reference's preamp schematic gives the hand-read netlist (up to node numbering), and the
    host-only plan analysis accepts the network (the 22 uF capacitor next to pF-sized ones: 8 orders of magnitude in admittance)."""
    nd = Q.Nodal.from_qucs_sch(os.path.join(REFERENCE, "util/preamp-bias-simulation/preamp-bias-simulation.sch"))
    br, nn, ports = preamp_netlist()
    assert nd.n_nodes == nn and [z for _, z in nd.ports] == [50.0] * 5
    got = sorted((k, round(p[0] if k != NB_SBLOCK else p[2], 15)) for k, _n, p in nd.branches)
    want = sorted((k, round(p[0] if k != NB_SBLOCK else p[2], 15)) for k, _n, p in br)
    assert got == want
    a = nd.analyze(np.linspace(1e6, 1e10, 5000))
    assert a["unknowns"] == 9 and np.isfinite(a["max_multiplier"])


# ---- the same anchors through the C-ABI on the GPU ---------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("key,svg", PNG_CASES)
def test_rftools_plots_pin_the_gpu_sweep(Q, ctx, golden_nets, png_curves, key, svg):
    n = golden_nets[svg]
    net = Q.Net.from_elements([(k, p) for k, p in n["elements"]], n["rs"], n["rl"])
    _check_curves(png_curves, key, lambda f: ctx.sweep(net, np.ascontiguousarray(f))[:2])


@pytest.mark.gpu
def test_plot_values_gpu(Q, ctx, golden_nets):
    svgs = dict(PNG_CASES)
    for key, f, trace, db, tol in PLOT_VALUES:
        n = golden_nets[svgs[key]]
        net = Q.Net.from_elements([(k, p) for k, p in n["elements"]], n["rs"], n["rl"])
        s11, s21 = ctx.sweep(net, np.array([f]))[:2]
        got = 20 * np.log10(abs((s21 if trace == "s21" else s11)[0]))
        assert abs(got - db) <= tol, (key, f, trace, got, db)


@pytest.mark.gpu
def test_trc_identities_gpu(Q, ctx, golden_nets):
    def sweep(el, f):
        return ctx.sweep(Q.Net.from_elements(el, 50.0, 50.0), f)[:2]
    # (dir_cpl_2.4g_35dB_pa_250W.trc is not a 50 Ohm design: sqrt(Z0e Z0o) = 50.69, so the matched-line identities do not apply)
    for name in ("dir_cpl_2.4g_20dB", "dir_cpl_2.4g_35dB", "dir_cpl_525m_20dB"):
        _coupler_checks(sweep, golden_nets["util/directional-couplers/%s.trc" % name])
    t = golden_nets["util/directional-couplers/dir_cpl_2.4g_20dB.trc"]
    s11, s21 = sweep([(12, [t["z0e"], t["z0o"], t["ang"], t["ang"], t["f0"], 50.0])], np.array([2.4e9]))
    assert abs(10 * np.log10(1 - abs(s21[0]) ** 2 - abs(s11[0]) ** 2) + 20.0385520502) < 1e-3           # SURVEY App. B.4 |S31| at 2.4 GHz


def _ladder_as_nodal(Q, net):
    """The same parasitic L / C ladder as a nodal netlist: series branches between consecutive nodes, shunt branches to
    ground, ports on the first and last node (branch parasitic forms are shared with QO_SER_L / QO_SHUNT_C by definition)."""
    rs, rl = net.terminations
    el = net.elements
    n_series = sum(1 for k, _ in el if k in (Q.SER_L, Q.SER_C, Q.SER_R))
    nd = Q.Nodal(n_series + 1)
    node = 1
    for k, p in el:
        if k == Q.SER_L:
            nd.add_branch(Q.NB_L, [node, node + 1], [p[0], p[1], p[2]]); node += 1
        elif k == Q.SER_C:
            nd.add_branch(Q.NB_C, [node, node + 1], [p[0], p[1], p[2]]); node += 1
        elif k == Q.SER_R:
            nd.add_branch(Q.NB_R, [node, node + 1], [p[0]]); node += 1
        elif k == Q.SHUNT_C:
            nd.add_branch(Q.NB_C, [node, 0], [p[0], p[1], p[2]])
        elif k == Q.SHUNT_L:
            nd.add_branch(Q.NB_L, [node, 0], [p[0], p[1], p[2]])
        elif k == Q.SHUNT_R:
            nd.add_branch(Q.NB_R, [node, 0], [p[0]])
        else:
            raise ValueError(k)
    nd.add_port(1, rs)
    nd.add_port(node, rl)
    return nd


@pytest.mark.gpu
@pytest.mark.parametrize("fc", [10e6, 3e9])
def test_cascade_equals_nodal_on_parasitic_ladder(Q, W, ctx, fc):
    """Row a9, transitive pin: qo_nodal_sweep reproduces the reference's pa-bias-simulation.dat (R, C + ESR, measured L;
    tests/test_nodal.py), and on the config-2 / config-5 ladder with ESR / SRF parasitics the cascade kernels give the
    nodal kernel's S-matrix."""
    net = W.cheby11(fc)
    f = Q.grid_log(fc / 2.5, fc * 2.0, 600)          # |S21| > -105 dB: above the nodal solve's absolute noise floor
    s11, s21, s12, s22 = ctx.sweep(net, f)
    nd = _ladder_as_nodal(Q, net)
    s = ctx.nodal_sweep(nd, f)
    assert relerr(s[:, 1, 0], s21) < 1e-9 and relerr(s[:, 0, 1], s12) < 1e-9
    assert np.max(np.abs(s[:, 0, 0] - s11)) < 1e-10 and np.max(np.abs(s[:, 1, 1] - s22)) < 1e-10
    nd.close()


@pytest.mark.gpu
def test_preamp_bias_plot_markers_gpu(Q, ctx, golden_s2p):
    """The marker values of the reference's preamp-bias plot from the GPU nodal sweep (qo_nodal_sweep through the C-ABI)."""
    br, nn, ports = preamp_netlist()
    fd, sd = golden_s2p["06HP47N_f"], golden_s2p["06HP47N_s"]
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], float(golden_s2p["06HP47N_z0"]))
    nd = Q.Nodal(nn)
    bi = nd.add_sblock(blk)
    for kind, nodes, p in br:
        nd.add_branch(kind, nodes, [bi, 1, 50.0] if kind == NB_SBLOCK else p)
    for node, z0 in ports:
        nd.add_port(node, z0)
    _check_preamp_markers(lambda f: ctx.nodal_sweep(nd, f))
    nd.close()
