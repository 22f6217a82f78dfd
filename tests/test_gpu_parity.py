"""Parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle on the same
seeded inputs, against the committed golden fixtures, and -- at BASELINE sizes -- through
size-independent properties.  Nothing here reads the upstream qo-100-tools tree.

Tolerances (north_star): nominal FP64 sweeps within 1e-9 relative (observed ~1e-14 for lumped
nets, ~2e-12 for the microstrip net whose pow/exp differ by an ulp between glibc and CUDA);
FP32 mode within 1e-3 dB where |S21| > -100 dB; perturbations bit-exact; integer yield counters
equal to the oracle's.
"""
import numpy as np
import pytest

import os

from conftest import ROOT, relerr, to_ref

pytestmark = pytest.mark.gpu

TOL64 = 1e-9


def _s_close(g, o, tol=TOL64):
    """S21/S12 relative; S11/S22 relative with the absolute floor of SURVEY §8c."""
    assert relerr(g[1], o[1]) <= tol, relerr(g[1], o[1])
    assert relerr(g[2], o[2]) <= tol
    for i in (0, 3):
        assert np.all(np.abs(g[i] - o[i]) <= tol * np.maximum(np.abs(o[i]), 0.02))


def test_native_library_is_loaded(Q, ctx):
    """The .so in-tree is what runs (the driver records loaded libraries)."""
    maps = open("/proc/self/maps").read()
    assert "qo-100-tools_b200/lib/libqo100net.so" in maps
    assert ctx.num_devices == 1


def test_rcp_accuracy(ctx):
    """MUFU.RCP64H + one cubic step: <= 1 ulp over 60 decades (qo_lumped.cuh::qrcp)."""
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(0.5, 2.0, 1 << 18), 10.0 ** rng.uniform(-150, 150, 1 << 18)])
    x = np.concatenate([x, -x])
    r = ctx.device_rcp(x)
    assert np.max(np.abs(r * x - 1.0)) <= 2.0 ** -52
    assert np.max(np.abs(r - 1.0 / x) / np.abs(1.0 / x)) <= 2.0 ** -52


def test_microstrip_log_accuracy(ctx):
    """qo_ustrip.cuh::ms_log (fdlibm-style reduction, degree-7 minimax, Newton reciprocal) against numpy's longdouble log:
    <= 1 ulp over 200 decades and next to 1; zero / negative / denormal / inf / nan arguments take the library path."""
    rng = np.random.default_rng(1)
    x = np.concatenate([10.0 ** rng.uniform(-100, 100, 1 << 18), 1.0 + rng.uniform(-0.3, 0.45, 1 << 18), 1.0 + rng.uniform(-1e-6, 1e-6, 1 << 16),
                        rng.uniform(0.70710, 0.70711, 1 << 12), rng.uniform(1.41421, 1.41422, 1 << 12)])
    g = ctx.device_mslog(x)
    ref = np.log(x.astype(np.longdouble))
    ulp = np.spacing(np.abs(ref.astype(np.float64)))
    assert np.max(np.abs((g.astype(np.longdouble) - ref).astype(np.float64)) / ulp) <= 1.0
    sp = np.array([0.0, -1.0, 5e-324, 1e-310, np.inf, np.nan])
    with np.errstate(all="ignore"):
        want = np.log(sp)
    got = ctx.device_mslog(sp)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(got[~np.isnan(want)], want[~np.isnan(want)])


def test_cfg1_if_bpf_nominal(Q, R, W, ctx, golden_b):
    w = W.cfg1()
    g = ctx.sweep(w.net, w.f, gd=True)
    o = R.sweep(to_ref(R, w.net), 50, 50, w.f, gd=True)
    _s_close(g, o)
    assert relerr(g[4], o[4]) < 1e-6 and np.all(g[4] > 0)
    # golden rows (40-digit mpmath), through the GPU
    c = golden_b["if_bpf"]
    f = np.array([r["f"] for r in c["rows"]])
    s21 = ctx.sweep(w.net, f)[1]
    ref = np.array([complex(float(r["s21"][0]), float(r["s21"][1])) for r in c["rows"]])
    assert relerr(s21, ref) < 1e-12


@pytest.mark.parametrize("case", ["if_bpf", "gpsdo_10m", "gpsdo_15m", "gpsdo_40m", "gpsdo_60m", "lol_hpf",
                                  "cheby11_ideal", "cfg2_nominal", "coupler_20db", "cfg5_nominal"])
def test_golden_rows_on_gpu(Q, ctx, golden_b, case):
    c = golden_b[case]
    net = Q.Net.from_elements([(k, p) for k, p in c["elements"]], c["rs"], c["rl"])
    f = np.array([r["f"] for r in c["rows"]])
    s11, s21, s12, _s22 = ctx.sweep(net, f)
    ref21 = np.array([complex(float(r["s21"][0]), float(r["s21"][1])) for r in c["rows"]])
    ref11 = np.array([complex(float(r["s11"][0]), float(r["s11"][1])) for r in c["rows"]])
    assert relerr(s21, ref21) < TOL64 and np.array_equal(s12, s21)
    assert np.max(np.abs(s11 - ref11)) < TOL64


def test_pa_lpf_dat_parity_from_gpu(Q, W, ctx, golden_dat):
    """util/pa-lpf-simulation/pa-lpf-simulation.dat:5007-35017 reproduced by the CUDA kernel."""
    g = ctx.sweep(W.pa_lpf_net(), golden_dat["frequency"])
    o = (golden_dat["S11"], golden_dat["S21"], golden_dat["S12"], golden_dat["S22"])
    _s_close(g, o)
    assert np.max(np.abs(20 * np.log10(np.abs(g[1])) - golden_dat["S21_dB"])) <= 1e-9
    assert relerr(g[1], o[1]) < 1e-10


def test_pa_lpf_vs_oracle(Q, R, W, ctx):
    net = W.pa_lpf_net()
    f = Q.grid_lin(1e7, 1e10, 1001)
    g = ctx.sweep(net, f)
    o = R.sweep(to_ref(R, net), 50, 50, f)
    _s_close(g, o, 1e-10)


@pytest.mark.parametrize("which", ["cfg2", "cfg5", "10M", "15M", "40M", "60M", "lol"])
def test_nominal_sweeps_vs_oracle(Q, R, W, ctx, golden_nets, which):
    if which == "cfg2":
        w = W.cfg2(0)
        net, f = w.net, w.f
    elif which == "cfg5":
        w = W.cfg5(0)
        net, f = w.net, w.f
    elif which == "lol":
        n = golden_nets["docs/upconverter/upconverter-lol-filter.svg"]
        net = Q.Net.from_elements([(k, p) for k, p in n["elements"]], n["rs"], n["rl"])
        f = Q.grid_log(2.1e9 / 6.25, 2.1e9 * 2.5, 4096)
    else:
        net, fc = [(n_, fc_) for nm, n_, fc_ in W.gpsdo_bank() if nm == which][0]
        f = Q.grid_log(fc / 2.5, fc * 6.25, 4096)
    rs, rl = net.terminations
    g = ctx.sweep(net, f, gd=True)
    o = R.sweep(to_ref(R, net), rs, rl, f, gd=True)
    _s_close(g, o)
    # group delay: same central-difference definition on both sides; phase noise limits it to ~1e-6
    assert np.max(np.abs(g[4] - o[4])) <= 1e-6 * np.max(np.abs(o[4]))


def test_fp32_mode_within_1e_3_db(Q, R, W, ctx):
    for w in (W.cfg1(), W.cfg2(0), W.cfg5(0)):
        rs, rl = w.net.terminations
        g = ctx.sweep(w.net, w.f, precision=32)
        o = R.sweep(to_ref(R, w.net), rs, rl, w.f)
        db_o = 20 * np.log10(np.abs(o[1]))
        db_g = 20 * np.log10(np.abs(g[1]))
        sel = db_o > -100.0
        assert np.max(np.abs(db_g[sel] - db_o[sel])) <= 1e-3


def test_sweep_edge_shapes(Q, R, ctx):
    """nf = 1, odd nf, a single element, resistors, TLINE, mismatched terminations."""
    net = Q.Net.from_elements([(Q.SER_R, [10.0]), (Q.SHUNT_R, [200.0]), (Q.TLINE, [75.0, 90.0, 1e9]),
                               (Q.SER_C, [1e-12, 0.5, 1e-9]), (Q.SHUNT_L, [10e-9, 0.2, 0.1e-12]),
                               (Q.SER_LC_PAR, [5e-9, 2e-12]), (Q.SHUNT_LC_SER, [8e-9, 1e-12])], 25.0, 100.0)
    for nf in (1, 2, 3, 31, 33, 65, 1023):
        f = Q.grid_log(1e8, 3e9, nf) if nf > 1 else np.array([1.2345e9])
        g = ctx.sweep(net, f)
        o = R.sweep(to_ref(R, net), 25.0, 100.0, f)
        _s_close(g, o)
    one = Q.Net.from_elements([(Q.SER_L, [1e-9])])
    f = np.array([1e9])
    assert relerr(ctx.sweep(one, f)[1], R.sweep(to_ref(R, one), 50, 50, f)[1]) < 1e-14


def test_sweep_errors(Q, ctx):
    net = Q.Net.from_elements([(Q.SER_L, [1e-9])])
    with pytest.raises(Q.QoError):
        ctx.sweep(net, np.array([1e9, -5.0]))
    with pytest.raises(Q.QoError):
        ctx.sweep(net, np.array([1e9]), precision=16)
    w_specs = [(Q.SPEC_GD_MAX, 0, 1e9, 1e-9)]
    with pytest.raises(Q.QoError) as ei:                      # group-delay specs: FP64 lumped networks only
        ctx.mc_run(net, np.array([1e8, 2e8]), w_specs, 1, 10, [], precision=32)
    assert ei.value.status == Q.ERR_UNSUPPORTED
    with pytest.raises(Q.QoError) as ei:
        ctx.mc_run(net, np.array([1e8, 2e8]), [(7, 0, 1e9, 1.0)], 1, 10, [])       # unknown spec kind
    assert ei.value.status == Q.ERR_ARG
    with pytest.raises(Q.QoError):
        ctx.mc_run(net, np.array([1e8, 2e8]), [(1, 0, 1e9, -1.0)] * 9, 1, 10, [])     # > 8 specs
    with pytest.raises(Q.QoError):
        ctx.mc_run(net, np.array([1e8]), [(1, 5e9, 6e9, -1.0)], 1, 10, [], hist_bins=8, hist_spec=0, hist_lo=-1.0, hist_hi=0.0)


def test_device_perturbations_bit_exact(Q, R, ctx):
    """Per-sample perturbation factors: device == the oracle's C stream, bit for bit, ALL 1e6 factors of both
    distributions (SURVEY App. C: "test = memcmp of 1e6 factors"), plus the product's host twin on a slice."""
    seed, off = 0x5EED010000000002, 123456789012
    for dist in (Q.DIST_UNIFORM, Q.DIST_GAUSS3S):
        ns, nv = 62500, 16
        got = ctx.device_perturb_factors(seed, off, ns, nv, dist, 0.05)
        ref = R.perturb_factors(seed, off, ns, nv, dist, 0.05)
        assert got.shape == ref.shape == (ns, nv) and got.size == 1000000
        assert got.tobytes() == ref.tobytes()                      # memcmp-level equality
        assert np.all(np.abs(got - 1.0) <= 0.05 + 1e-15) and np.unique(got).size > 990000
        host = np.array([[Q.perturb_factor(seed, off + s, v, dist, 0.05) for v in range(nv)] for s in range(512)])
        assert np.array_equal(got[:512], host)
    # a sample offset beyond 2^32 exercises the high counter word
    got = ctx.device_perturb_factors(seed, (1 << 40) + 5, 1000, 7, Q.DIST_UNIFORM, 0.02)
    assert got.tobytes() == R.perturb_factors(seed, (1 << 40) + 5, 1000, 7, Q.DIST_UNIFORM, 0.02).tobytes()


def _mc_both(Q, R, ctx, w, n, nthreads=8, **kw):
    rs, rl = w.net.terminations
    og = R.mc_run(to_ref(R, w.net), rs, rl, w.f, w.specs, R.mc_cfg(w.seed, n, w.tols, **w.hist, **kw), nthreads=nthreads)
    gg = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **w.hist, **kw)
    return og, gg


def _assert_counts_equal(og, gg):
    assert gg["n_total"] == og["n_total"]
    assert gg["n_pass"] == og["n_pass"]
    assert np.array_equal(gg["fail_per_spec"], og["fail_per_spec"])
    assert np.array_equal(gg["hist"], og["hist"])


def test_cfg2_yield_equals_oracle(Q, R, W, ctx):
    w = W.cfg2()
    og, gg = _mc_both(Q, R, ctx, w, 3000)
    _assert_counts_equal(og, gg)
    assert 0.55 < gg["n_pass"] / gg["n_total"] < 0.72          # SURVEY's non-degenerate yield estimate
    assert int(gg["hist"].sum()) == 3000
    og, gg = _mc_both(Q, R, ctx, w, 1500, dist=Q.DIST_GAUSS3S)
    _assert_counts_equal(og, gg)


def test_cfg5_yield_equals_oracle(Q, R, W, ctx):
    w = W.cfg5()
    og, gg = _mc_both(Q, R, ctx, w, 1500)
    _assert_counts_equal(og, gg)
    assert 0.5 < gg["n_pass"] / gg["n_total"] < 0.8


def test_cfg3_microstrip_yield_equals_oracle(Q, R, W, ctx):
    w = W.cfg3()
    og, gg = _mc_both(Q, R, ctx, w, 2000)
    _assert_counts_equal(og, gg)
    assert 0.5 < gg["n_pass"] / gg["n_total"] < 0.85


def test_microstrip_board_kernel_equals_item_kernel_and_oracle(Q, R, W, ctx, monkeypatch):
    """Microstrip yield jobs at <= 4 frequencies run one thread per board with the frequencies side by side (qo_mc_board_kernel);
    QO100NET_USTRIP=item keeps one thread per (board, frequency) item (qo_mc_generic_kernel).  Same counters from both and from
    the oracle, for 1, 2, 3 and 4 frequencies, with lumped elements mixed into the microstrip cascade and a histogram on a
    "max" spec; five frequencies stay on the item kernel."""
    w = W.cfg3()
    n = 3000
    extra = Q.Net.from_elements([(Q.SER_L, [0.4e-9, 0.05, 0.02e-12]), (Q.SHUNT_C, [0.15e-12, 0.1, 0.0])], 50.0, 50.0)
    net = w.net.concat(extra)
    tols = w.tols + [(len(w.net.elements), 0, 9, Q.TOL_REL, 0.1)]
    grids = {1: [4.8e9], 2: [2.4e9, 7.2e9], 3: [2.4e9, 4.8e9, 7.2e9], 4: [1.2e9, 2.4e9, 4.8e9, 7.2e9]}
    for nfreq, fl in grids.items():
        f = np.array(fl)
        nom = ctx.sweep(net, f)
        db = 20 * np.log10(np.abs(nom[1]))
        specs = [(Q.SPEC_S21_MAX_DB if v < -6 else Q.SPEC_S21_MIN_DB, fk * 0.99, fk * 1.01, float(v) + (0.4 if v < -6 else -0.08)) for fk, v in zip(fl, db)]
        hist = dict(hist_bins=32, hist_spec=0, hist_lo=float(db[0]) - 3.0, hist_hi=float(db[0]) + 3.0)
        monkeypatch.delenv("QO100NET_USTRIP", raising=False)
        plan = Q.Plan(ctx, net, f, specs, seed=31, tols=tols, **hist)
        assert plan.kernel_name == "qo_mc_board_kernel"
        plan.launch(2 ** 32 + 11, n)
        board = plan.read()
        plan.close()
        monkeypatch.setenv("QO100NET_USTRIP", "item")
        plan = Q.Plan(ctx, net, f, specs, seed=31, tols=tols, **hist)
        assert plan.kernel_name == "qo_mc_generic_kernel"
        plan.launch(2 ** 32 + 11, n)
        item = plan.read()
        plan.close()
        monkeypatch.delenv("QO100NET_USTRIP", raising=False)
        _assert_counts_equal(item, board)
        rs, rl = net.terminations
        ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(31, n, tols, sample_offset=2 ** 32 + 11, **hist), nthreads=8)
        _assert_counts_equal(ref, board)
        assert 0 < board["n_pass"] < n, (nfreq, board["n_pass"])
    f5 = np.array([1.2e9, 2.4e9, 3.6e9, 4.8e9, 7.2e9])
    plan = Q.Plan(ctx, net, f5, [(Q.SPEC_S21_MIN_DB, 2.3e9, 2.5e9, -1.0)], seed=31, tols=tols)
    assert plan.kernel_name == "qo_mc_generic_kernel"
    plan.close()


def test_cfg3b_lumped_twin_yield_equals_oracle(Q, R, W, ctx, monkeypatch):
    """BASELINE config 3 as worded (lumped PA LPF with ESR/SRF parasitics, 3 points per sample): counters equal the oracle's on
    the spot-frequency kernel (one thread per sample, the default for <= 8 points) and on the three warp-per-sample kernels;
    the yield sits where the oracle put it when the spec limits were chosen (0.70).  Also |S11| specs, 8 points, gaussian draws
    and an rf-tools filter with traps on the spot kernel."""
    w = W.cfg3b()
    for force, name in ((None, "qo_mc_spot_kernel"), ("tf", "qo_mc_tf_kernel"), ("ladder", "qo_mc_ladder_kernel"), ("interp", "qo_mc_lumped_kernel")):
        if force:
            monkeypatch.setenv("QO100NET_KERNEL", force)
        else:
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
        assert plan.kernel_name == name
        plan.close()
        og, gg = _mc_both(Q, R, ctx, w, 20000)
        _assert_counts_equal(og, gg)
        assert 0.65 < gg["n_pass"] / gg["n_total"] < 0.75 and np.all(gg["fail_per_spec"] > 0)
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    fc = 2.9e9
    f8 = np.array([0.5e9, 1.2e9, 2.0e9, 2.4e9, 2.7e9, 4.8e9, 6.0e9, 7.2e9])
    specs = [(Q.SPEC_S11_MAX_DB, 0.0, 2.5e9, -9.0), (Q.SPEC_S21_MIN_DB, 0.0, 2.75e9, -1.0), (Q.SPEC_S21_MAX_DB, 4.7e9, 1e99, -43.0)]
    for hs, lo, hi in ((0, -25.0, 0.0), (1, -3.0, 0.0), (2, -50.0, -38.0)):
        hist = dict(hist_bins=48, hist_spec=hs, hist_lo=lo, hist_hi=hi)
        plan = Q.Plan(ctx, w.net, f8, specs, seed=5, tols=w.tols, dist=Q.DIST_GAUSS3S, **hist)
        assert plan.kernel_name == "qo_mc_spot_kernel"
        plan.launch(9, 3000)
        got = plan.read()
        plan.close()
        ref = R.mc_run(to_ref(R, w.net), 50, 50, f8, specs, R.mc_cfg(5, 3000, w.tols, sample_offset=9, dist=Q.DIST_GAUSS3S, **hist), nthreads=8)
        _assert_counts_equal(ref, got)
        assert 0 < got["n_pass"] < 3000
    _, ell, fe = W.gpsdo_bank()[1]
    f3 = np.array([0.5 * fe, 0.8 * fe, 2.2 * fe])
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, 0.85 * fe, -0.6), (Q.SPEC_S21_MAX_DB, 2.0 * fe, 1e99, -45.0)]
    tols = Q.lc_tolerances(ell, 0.05, 0.05)
    got = ctx.mc_run(ell, f3, specs, 8, 5000, tols)
    ref = R.mc_run(to_ref(R, ell), 50, 50, f3, specs, R.mc_cfg(8, 5000, tols), nthreads=8)
    _assert_counts_equal(ref, got)
    nine = Q.Plan(ctx, w.net, np.linspace(1e9, 7e9, 9), w.specs, seed=1, tols=w.tols)       # 9 points: back to the warp-per-sample kernels
    assert nine.kernel_name == "qo_mc_tf_kernel"; nine.close()


def test_s11_spec_and_histogram(Q, R, W, ctx, monkeypatch):
    """|S11| specs against the oracle on every kernel that serves them: the transfer-function kernel (S11 =
    (P - Rs Q) / (P + Rs Q); behind the coupler block with the block's second row vector), the chain kernel's second row
    vector (forced) and the interpreter's 2x2 chain; histogram on the |S11| spec and on the |S21| specs."""
    for w in (W.cfg2(), W.cfg5()):
        fc = 10e6 if w.name.startswith("cfg2") else 3e9
        w.specs = [(Q.SPEC_S11_MAX_DB, 0.0, 0.8 * fc, -8.0), (Q.SPEC_S21_MAX_DB, 1.3 * fc, 1e99, -49.0), (Q.SPEC_S21_MIN_DB, 0, 0.5 * fc, -1.3)]
        for hs, lo, hi in ((0, -20.0, 0.0), (1, -60.0, -40.0), (2, -3.0, 0.0)):
            w.hist = dict(hist_bins=64, hist_spec=hs, hist_lo=lo, hist_hi=hi)
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
            plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
            assert plan.kernel_name == "qo_mc_tf_kernel"
            plan.close()
            og, gg = _mc_both(Q, R, ctx, w, 800)
            _assert_counts_equal(og, gg)
            assert 0 < gg["n_pass"] < 800
            for force in ("ladder", "interp"):
                monkeypatch.setenv("QO100NET_KERNEL", force)
                ig = ctx.mc_run(w.net, w.f, w.specs, w.seed, 800, w.tols, **w.hist)
                _assert_counts_equal(ig, gg)
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    # |S11| only (no denominator polynomial at all), and on the rf-tools / mixed lumped networks
    w = W.cfg2()
    only = [(Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.5)]
    plan = Q.Plan(ctx, w.net, w.f, only, seed=9, tols=w.tols, hist_bins=32, hist_spec=0, hist_lo=-20.0, hist_hi=0.0)
    assert plan.kernel_name == "qo_mc_tf_kernel" and plan.tf_info["den_form"] == "none" and plan.tf_info["numerator_chains"] == 4
    plan.launch(0, 700)
    got = plan.read()
    plan.close()
    ref = R.mc_run(to_ref(R, w.net), 50, 50, w.f, only, R.mc_cfg(9, 700, w.tols, hist_bins=32, hist_spec=0, hist_lo=-20.0, hist_hi=0.0), nthreads=8)
    _assert_counts_equal(ref, got)
    assert int(got["hist"].sum()) == 700 and np.count_nonzero(got["hist"]) > 3      # the worst in-band |S11| spreads over several bins
    for name, net, fc in _mixed_lumped_nets(Q, W):
        f = Q.grid_log(fc / 3.0, fc * 4.0, 777)
        sw = ctx.sweep(net, f)
        db21, db11 = 20 * np.log10(np.abs(sw[1])), 20 * np.log10(np.abs(sw[0]))
        pb = db21 >= db21.max() - 0.5
        f_lo, f_hi = float(f[pb].min()) * 1.03, float(f[pb].max()) * 0.97
        inb = (f >= f_lo) & (f <= f_hi)
        specs = [(Q.SPEC_S11_MAX_DB, f_lo, f_hi, float(db11[inb].max()) + 0.7), (Q.SPEC_S21_MIN_DB, f_lo, f_hi, float(db21[inb].min()) - 0.1)]
        tols = Q.lc_tolerances(net, 0.05, 0.05)
        hist = dict(hist_bins=40, hist_spec=0, hist_lo=float(db11[inb].max()) - 10.0, hist_hi=0.0)
        plan = Q.Plan(ctx, net, f, specs, seed=4, tols=tols, **hist)
        assert plan.kernel_name == "qo_mc_tf_kernel", (name, plan.tf_info)
        plan.launch(0, 500)
        got = plan.read()
        plan.close()
        rs, rl = net.terminations
        ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(4, 500, tols, **hist), nthreads=8)
        _assert_counts_equal(ref, got)
        assert int(got["fail_per_spec"].sum()) > 0, name


def test_full_s_mode_vs_oracle(Q, R, W, ctx):
    for w in W.cfg4(24, 1024) + [W.cfg2(0, 513)]:
        rs, rl = w.net.terminations
        g = ctx.mc_run(w.net, w.f, [], w.seed, 24, w.tols, mode=Q.MODE_FULL_S)["s"]
        o = R.mc_run(to_ref(R, w.net), rs, rl, w.f, [], R.mc_cfg(w.seed, 24, w.tols), full_s=True)["s"]
        _s_close(g, o)
    # microstrip network through the generic kernel
    w = W.cfg3()
    f = Q.grid_lin(1e9, 8e9, 57)
    g = ctx.mc_run(w.net, f, [], 3, 16, w.tols, mode=Q.MODE_FULL_S)["s"]
    o = R.mc_run(to_ref(R, w.net), 50, 50, f, [], R.mc_cfg(3, 16, w.tols), full_s=True)["s"]
    _s_close(g, o, 1e-10)


def test_sample_offset_and_sharding_invariance(Q, W, ctx):
    """Same seed => identical u64 counters however the global sample range is cut (1/2/4/8 shards)."""
    w = W.cfg2()
    n = 4096
    whole = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **w.hist)
    from qo100net import dist as qd
    for world in (2, 4, 8):
        tot = np.zeros(2 + 2 + 256, dtype=np.int64)
        for r in range(world):
            lo, hi = qd.shard_range(n, r, world)
            p = ctx.mc_run(w.net, w.f, w.specs, w.seed, hi - lo, w.tols, sample_offset=lo, **w.hist)
            tot += np.concatenate([[p["n_pass"], p["n_total"]], p["fail_per_spec"], p["hist"]]).astype(np.int64)
        assert tot[0] == whole["n_pass"] and tot[1] == n
        assert np.array_equal(tot[2:4], whole["fail_per_spec"].astype(np.int64))
        assert np.array_equal(tot[4:], whole["hist"].astype(np.int64))


def test_plan_resident_launches_accumulate(Q, W, ctx):
    """The HBM-resident plan: counters accumulate over launches; caller-owned device counters work."""
    import torch
    w = W.cfg2()
    plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
    assert plan.num_counters == 2 + 2 + 256 and plan.flops_per_eval == 349.0
    plan.launch(0, 1000)
    plan.launch(1000, 1000)
    a = plan.read()
    whole = ctx.mc_run(w.net, w.f, w.specs, w.seed, 2000, w.tols, **w.hist)
    assert a["n_pass"] == whole["n_pass"] and a["n_total"] == 2000 and np.array_equal(a["hist"], whole["hist"])
    cnt = torch.zeros(plan.num_counters, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    plan.launch(0, 2000, cnt.data_ptr())
    plan.read()
    c = cnt.cpu().numpy()
    assert c[0] == whole["n_pass"] and c[1] == 2000 and np.array_equal(c[4:], whole["hist"].astype(np.int64))
    assert plan.launches == 3
    plan.close()


def test_zero_tolerance_equals_nominal(Q, R, W, ctx):
    w = W.cfg2()
    zt = [(e, p, v, m, 0.0) for (e, p, v, m, _t) in w.tols]
    g = ctx.mc_run(w.net, w.f, [], 9, 3, zt, mode=Q.MODE_FULL_S)["s"]
    nom = ctx.sweep(w.net, w.f)
    for k in range(3):
        assert np.array_equal(g[1, k], nom[1]) and np.array_equal(g[0, k], nom[0])
    r = ctx.mc_run(w.net, w.f, w.specs, 9, 50, zt, **w.hist)
    assert r["n_pass"] == 50 and int(r["hist"].sum()) == 50 and np.count_nonzero(r["hist"]) == 1


def test_properties_at_baseline_size(Q, W, ctx):
    """Size-independent properties on the full cfg-2 shape (1e6 x 4096 is the bench; 2e5 here)."""
    w = W.cfg2()
    n = 200000
    r = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **w.hist)
    assert r["n_total"] == n and int(r["hist"].sum()) == n
    assert r["n_pass"] + max(r["fail_per_spec"]) <= n <= r["n_pass"] + int(r["fail_per_spec"].sum())
    y = r["n_pass"] / n
    assert 0.60 < y < 0.66
    # a second, disjoint sample range gives a statistically consistent yield (binomial 5 sigma)
    r2 = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, sample_offset=10 ** 12, **w.hist)
    assert abs(r2["n_pass"] / n - y) < 5 * np.sqrt(2 * y * (1 - y) / n)
    # passivity and reciprocity on lossless ladders, FULL_S at 4096 points
    for wl in W.cfg4(64, 4096):
        s = ctx.mc_run(wl.net, wl.f, [], wl.seed, 64, wl.tols, mode=Q.MODE_FULL_S)["s"]
        p = np.abs(s[0]) ** 2 + np.abs(s[1]) ** 2
        assert np.max(np.abs(p - 1.0)) < 1e-9                  # lossless: |S11|^2 + |S21|^2 = 1
        assert np.array_equal(s[1], s[2])
        assert np.max(np.abs(np.abs(s[0]) - np.abs(s[3]))) < 1e-9
    wl = W.cfg2(0)
    s = ctx.mc_run(wl.net, wl.f, [], 1, 64, wl.tols, mode=Q.MODE_FULL_S)["s"]
    assert np.all(np.abs(s[0]) ** 2 + np.abs(s[1]) ** 2 <= 1.0 + 1e-12)      # lossy: passive


# ---- the straight-line ladder kernel (qo_ladder.cuh) ---------------------------------------------
def _ladder_workload(Q, W, order, series_first, coupler, butter=False, fc=10e6, nf=1000):
    """An order-N pcb/generic-filter ladder with the cfg-2 parasitic model, specs placed around its own
    nominal response so that the yield is neither 0 nor 1."""
    net = (Q.Net.butter_lpf(order, fc, 50.0, series_first) if butter else Q.Net.cheby_lpf(order, 0.1, fc, 50.0, series_first))
    net = net.add_parasitics(fc, 60.0, 30.0, 0.1, 50.0)
    tols = Q.lc_tolerances(net, 0.05, 0.02)
    if coupler:
        # even orders: the coupler is referenced to 60 Ohm behind the 50 Ohm source, so the block's row vector takes its general
        # form instead of the matched one (qo_tf.cuh::tf_cpl_matched)
        zt = 60.0 if order % 2 == 0 else 50.0
        cpl = Q.Net.from_elements([(Q.CPL_THRU, [55.2771, 45.2267, 95.4225, 91.0, 4 * fc, zt])], 50.0, 50.0)
        net = cpl.concat(net)
        tols = [(0, 0, 0, Q.TOL_REL, 0.02), (0, 1, 1, Q.TOL_REL, 0.02), (0, 2, 2, Q.TOL_REL, 0.01), (0, 3, 2, Q.TOL_REL, 0.01)] + \
               [(e + 1, p, v + 3, m, t) for (e, p, v, m, t) in tols]
    f = Q.grid_log(fc / 2.5, fc * 6.25, nf)
    return net, f, tols


@pytest.mark.parametrize("order,series_first,coupler", [(1, True, False), (1, False, False), (2, True, False), (2, False, True),
                                                        (3, False, False), (4, True, True), (5, True, False), (6, False, False),
                                                        (7, False, True), (8, True, False), (9, False, False), (10, True, False),
                                                        (10, False, True), (11, True, False), (11, False, False), (11, True, True)])
def test_ladder_kernel_family_vs_oracle_and_interpreter(Q, R, W, ctx, monkeypatch, order, series_first, coupler):
    """Every instantiation family (order, series/shunt first, coupler block) gives the oracle's integer
    counters, and the same counters as the opcode interpreter forced with QO100NET_KERNEL=interp."""
    fc = 10e6
    net, f, tols = _ladder_workload(Q, W, order, series_first, coupler, butter=order % 2 == 0)   # even-order Chebyshev needs Rs != Rl
    db = 20 * np.log10(np.abs(ctx.sweep(net, f)[1]))
    pb, sb = f <= 0.8 * fc, f >= 3.0 * fc
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, 0.8 * fc, float(db[pb].min()) - 0.02),
             (Q.SPEC_S21_MAX_DB, 3.0 * fc, 1e99, float(db[sb].max()) + 0.2)]
    hist = dict(hist_bins=32, hist_spec=order % 2, hist_lo=float(db[pb].min()) - 1.0 if order % 2 == 0 else float(db[sb].max()) - 3.0,
                hist_hi=0.0 if order % 2 == 0 else float(db[sb].max()) + 3.0)
    n = 700
    rs, rl = net.terminations
    ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(77 + order, n, tols, sample_offset=5, **hist), nthreads=8)
    # default: the transfer-function kernel; QO100NET_KERNEL=ladder: the straight-line chain kernel; =interp: the interpreter
    for force, name in ((None, "qo_mc_tf_kernel"), ("ladder", "qo_mc_ladder_kernel"), ("interp", "qo_mc_lumped_kernel")):
        if force:
            monkeypatch.setenv("QO100NET_KERNEL", force)
        else:
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        plan = Q.Plan(ctx, net, f, specs, seed=77 + order, tols=tols, **hist)
        assert plan.kernel_name == name
        plan.launch(5, n)
        got = plan.read()
        plan.close()
        _assert_counts_equal(ref, got)
        if order >= 3:
            assert 0 < got["n_pass"] < n, "degenerate spec placement"
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)


def test_ladder_kernel_selection_and_edge_shapes(Q, R, W, ctx, monkeypatch):
    """Which jobs take the straight-line kernel; odd grid sizes, 3-4 specs, gaussian tolerances, Butterworth."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    w = W.cfg2()
    mk = lambda specs, **kw: Q.Plan(ctx, w.net, w.f, specs, seed=1, tols=w.tols, **kw)
    p = mk(w.specs); assert p.kernel_name == "qo_mc_tf_kernel"; p.close()                                          # |S21| specs: transfer-function kernel
    monkeypatch.setenv("QO100NET_KERNEL", "ladder")
    p = mk(w.specs); assert p.kernel_name == "qo_mc_ladder_kernel"; p.close()                                      # ... unless the chain kernel is asked for
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.setenv("QO100NET_TF_TOL", "1e-16")
    p = mk(w.specs); assert p.kernel_name == "qo_mc_ladder_kernel"; p.close()                                      # ... or the plan's self-check rejects the expansion
    monkeypatch.delenv("QO100NET_TF_TOL", raising=False)
    p = mk([(Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.0)]); assert p.kernel_name == "qo_mc_tf_kernel"; p.close()          # |S11| = |P - Rs Q| / |P + Rs Q|
    monkeypatch.setenv("QO100NET_KERNEL", "ladder")
    p = mk([(Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.0)]); assert p.kernel_name == "qo_mc_ladder_kernel"; p.close()      # chain kernel: second row vector
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    p = Q.Plan(ctx, W.cfg5().net, W.cfg5().f, [(Q.SPEC_S11_MAX_DB, 2.3e9, 2.5e9, -10.0)], seed=1, tols=W.cfg5().tols)
    assert p.kernel_name == "qo_mc_tf_kernel"; p.close()                                                          # |S11| behind the coupler block: its second row vector
    p = mk([(Q.SPEC_GD_MAX, 0.0, 8e6, 1e-6)]); assert p.kernel_name == "qo_mc_tf_kernel"; p.close()             # group delay: derivative polynomials
    p = mk([(Q.SPEC_GD_MAX, 0.0, 8e6, 1e-6), (Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.0)]); assert p.kernel_name == "qo_mc_lumped_kernel"; p.close()   # GD + |S11|: interpreter
    p = mk(w.specs * 3); assert p.kernel_name == "qo_mc_tf_kernel"; p.close()                                     # 6 specs: the 8-slot instantiation
    monkeypatch.setenv("QO100NET_KERNEL", "ladder")
    p = mk(w.specs * 3); assert p.kernel_name == "qo_mc_lumped_kernel"; p.close()                                 # the chain kernel keeps 4 trackers in registers
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    p = mk([], mode=Q.MODE_FULL_S); assert p.kernel_name == "qo_mc_lumped_kernel"; p.close()                      # HBM-bound mode
    p = mk(w.specs, precision=32); assert p.kernel_name == "qo_mc_ladder_kernel"; p.close()                       # optional FP32 mode
    p = mk([(Q.SPEC_S11_MAX_DB, 0.0, 8e6, -8.0)], precision=32); assert p.kernel_name == "qo_mc_lumped_kernel"; p.close()
    w1 = W.cfg1()
    p = Q.Plan(ctx, w1.net, w1.f, [(Q.SPEC_S21_MIN_DB, 3.5e8, 4.5e8, -1.0)], seed=1, tols=Q.lc_tolerances(w1.net, 0.05, 0.05))
    assert p.kernel_name == "qo_mc_tf_kernel"; p.close()                                                          # LC-tank branches are rational too
    w5 = W.cfg5()
    p = Q.Plan(ctx, w5.net, w5.f, w5.specs, seed=1, tols=w5.tols); assert p.kernel_name == "qo_mc_tf_kernel"; p.close()
    tl = Q.Net.from_elements([(Q.TLINE, [50.0, 90.0, 1e9])] + w.net.elements, 50.0, 50.0)
    p = Q.Plan(ctx, tl, w.f, w.specs, seed=1); assert p.kernel_name == "qo_mc_tf_kernel"; p.close()                # a line in FRONT: its row vector times the polynomials behind it
    el = w.net.elements
    tl = Q.Net.from_elements(el[:4] + [(Q.TLINE, [50.0, 90.0, 1e9])] + el[4:], 50.0, 50.0)
    p = Q.Plan(ctx, tl, w.f, w.specs, seed=1); assert p.kernel_name == "qo_mc_lumped_kernel"; p.close()            # a line inside the cascade: no polynomial form
    for nf, butter, dist in ((1, False, Q.DIST_UNIFORM), (2, False, Q.DIST_UNIFORM), (63, True, Q.DIST_GAUSS3S),
                             (130, False, Q.DIST_GAUSS3S), (257, True, Q.DIST_UNIFORM)):
        fc = 10e6
        net, f, tols = _ladder_workload(Q, W, 7, True, False, butter=butter, nf=max(nf, 2))
        f = f[:nf]
        specs = [(Q.SPEC_S21_MIN_DB, 0.0, 0.7 * fc, -1.0), (Q.SPEC_S21_MAX_DB, 2.5 * fc, 1e99, -60.0),
                 (Q.SPEC_S21_MIN_DB, 0.0, 0.5 * fc, -0.9), (Q.SPEC_S21_MAX_DB, 0.9 * fc, 1.1 * fc, -0.5)]
        hist = dict(hist_bins=16, hist_spec=3, hist_lo=-6.0, hist_hi=0.0) if nf >= 130 else {}
        if hist and not np.any((f >= 0.9 * fc) & (f <= 1.1 * fc)):
            hist = {}
        rs, rl = net.terminations
        ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(5, 300, tols, dist=dist, **hist), nthreads=8)
        for force in (None, "ladder"):
            if force:
                monkeypatch.setenv("QO100NET_KERNEL", force)
            got = ctx.mc_run(net, f, specs, 5, 300, tols, dist=dist, **hist)
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
            _assert_counts_equal(ref, got)


def test_gpu_sweep_to_qucs_dataset(Q, W, ctx, golden_dat, tmp_path):
    """Row N2 end to end: the PA-LPF sweep computed on the GPU, written as a Qucs dataset, read back, and
    compared with the reference dataset's values (tests/golden/pa_lpf_dat.npz)."""
    f = golden_dat["frequency"]
    s11, s21, s12, s22 = ctx.sweep(W.pa_lpf_net(), f)
    d = Q.Dataset.from_sweep(f, s11, s12, s21, s22)
    d.write(str(tmp_path / "gpu.dat"))
    r = Q.Dataset.read(str(tmp_path / "gpu.dat"))
    assert np.array_equal(r["S[2,1]"], s21) and np.array_equal(r["frequency"], f)
    assert relerr(r["S[2,1]"], golden_dat["S21"]) <= TOL64 and relerr(r["S[1,2]"], golden_dat["S12"]) <= TOL64
    assert np.max(np.abs(r["S21_dB"] - golden_dat["S21_dB"])) <= 1e-9
    assert np.all(np.abs(r["S[1,1]"] - golden_dat["S11"]) <= TOL64 * np.maximum(np.abs(golden_dat["S11"]), 0.02))
    # the display markers of util/pa-lpf-simulation/pa-lpf-simulation.dpl:25-28 (3 digits, on the dataset's own grid points)
    for fm, val in ((2.39009e9, -0.952), (7.20424e9, -8.85), (4.79817e9, -22.8), (3.06355e9, -2.82)):
        k = int(np.argmin(np.abs(r["frequency"] - fm)))
        assert abs(r["S21_dB"][k] - val) < 0.006 * max(1.0, abs(val) / 3)


def test_single_process_multi_gpu_ctx_matches_one_gpu(Q, W, ctx):
    """qo_ctx_create(N): one process, samples sharded over N GPUs, counters combined by ncclAllReduce --
    identical u64 counters to the one-GPU run, reduce-only and FULL_S.  Needs >= 2 visible GPUs."""
    import torch
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("needs >= 2 GPUs")
    w = W.cfg5()
    n = 20001
    one = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **w.hist)
    for g in [x for x in (2, 4, 8) if x <= ng]:
        c = Q.Context(ngpus=g)
        assert c.num_devices == g
        got = c.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **w.hist)
        assert got["n_pass"] == one["n_pass"] and got["n_total"] == n
        assert np.array_equal(got["fail_per_spec"], one["fail_per_spec"]) and np.array_equal(got["hist"], one["hist"])
        plan = Q.Plan(c, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
        plan.launch(0, 7000)
        plan.launch(7000, n - 7000)
        acc = plan.read()
        assert acc["n_pass"] == one["n_pass"] and np.array_equal(acc["hist"], one["hist"])
        plan.close()
        w4 = W.cfg4(33, 257)[1]
        a = ctx.mc_run(w4.net, w4.f, [], w4.seed, 33, w4.tols, mode=Q.MODE_FULL_S)["s"]
        b = c.mc_run(w4.net, w4.f, [], w4.seed, 33, w4.tols, mode=Q.MODE_FULL_S)["s"]
        assert np.array_equal(a, b)
        c.close()


def test_touchstone_blocks_in_cascade(Q, R, W, ctx, golden_s2p):
    """Row N3 on the GPU: measured two-ports (the reference's Coilcraft inductors, pa-bias-simulation.sch:39 /
    preamp-bias-simulation.sch:32, and the non-reciprocal driver measurement) cascaded with lumped elements:
    nominal sweep and FULL_S Monte Carlo vs the oracle and vs an independent numpy restatement."""
    from conftest import np_s_to_abcd, np_spfile
    blk = {}
    for i, key in enumerate(("11SQ39N", "06HP47N", "pa_20W")):
        fd, sd, z0 = golden_s2p[key + "_f"], golden_s2p[key + "_s"], float(golden_s2p[key + "_z0"])
        blk[key] = (Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0), fd, sd, z0)
    R.sblock_clear()
    # bias-tee like cascade: DC-block C (2.2 pF + 3 Ohm ESR, pa-bias-simulation.sch:28,32) - series inductor block -
    # shunt C - second inductor block (rectangular interpolation) - series R
    lumped1 = Q.Net.from_elements([(Q.SER_C, [12e-12, 0.6, 0.0])], 50, 50)
    lumped2 = Q.Net.from_elements([(Q.SHUNT_C, [2.2e-12, 3.0, 0.0])], 50, 50)
    lumped3 = Q.Net.from_elements([(Q.SER_R, [4.7])], 50, 75)
    net = lumped1.concat(blk["11SQ39N"][0].as_net(True)).concat(lumped2).concat(blk["06HP47N"][0].as_net(False)).concat(lumped3)
    for i, key in enumerate(("11SQ39N", "06HP47N")):
        _, fd, sd, z0 = blk[key]
        R.sblock_register(i, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    f = Q.grid_log(5e6, 5e9, 777)
    g = ctx.sweep(net, f)
    o = R.sweep(to_ref(R, net), 50, 75, f)
    _s_close(g, o)
    # third implementation: numpy 2x2 products
    w = 2 * np.pi * f
    def ser(z): return np.stack([np.ones_like(z), z, np.zeros_like(z), np.ones_like(z)], 1)
    def sh(y): return np.stack([np.ones_like(y), np.zeros_like(y), y, np.ones_like(y)], 1)
    def mul(a, b): return np.stack([a[:, 0] * b[:, 0] + a[:, 1] * b[:, 2], a[:, 0] * b[:, 1] + a[:, 1] * b[:, 3],
                                    a[:, 2] * b[:, 0] + a[:, 3] * b[:, 2], a[:, 2] * b[:, 1] + a[:, 3] * b[:, 3]], 1)
    parts = [ser(0.6 + 1 / (1j * w * 12e-12)),
             np_s_to_abcd(np_spfile(f, blk["11SQ39N"][1], blk["11SQ39N"][2], True), 50.0),
             sh(1 / (3.0 + 1 / (1j * w * 2.2e-12))),
             np_s_to_abcd(np_spfile(f, blk["06HP47N"][1], blk["06HP47N"][2], False), 50.0),
             ser(np.full_like(w, 4.7, dtype=complex))]
    M = parts[0]
    for p_ in parts[1:]:
        M = mul(M, p_)
    rs, rl = 50.0, 75.0
    den = M[:, 0] * rl + M[:, 1] + M[:, 2] * rs * rl + M[:, 3] * rs
    assert relerr(g[1], 2 * np.sqrt(rs * rl) / den) < 1e-10
    assert np.max(np.abs(g[0] - (M[:, 0] * rl + M[:, 1] - M[:, 2] * rs * rl - M[:, 3] * rs) / den)) < 1e-10
    # Monte Carlo over the lumped parts, blocks fixed: yield counters and FULL_S planes vs the oracle
    tols = [(0, 0, 0, Q.TOL_REL, 0.1), (2, 0, 1, Q.TOL_REL, 0.1), (4, 0, 2, Q.TOL_REL, 0.05)]
    b1, b2 = (f >= 3e8) & (f <= 9e8), (f >= 4e8) & (f <= 8e8)
    lim21 = float((20 * np.log10(np.abs(g[1][b1]))).min()) - 0.05
    lim11 = float((20 * np.log10(np.abs(g[0][b2]))).max()) + 0.1
    specs = [(Q.SPEC_S21_MIN_DB, 3e8, 9e8, lim21), (Q.SPEC_S11_MAX_DB, 4e8, 8e8, lim11)]
    hist = dict(hist_bins=24, hist_spec=0, hist_lo=lim21 - 3.0, hist_hi=lim21 + 3.0)
    got = ctx.mc_run(net, f, specs, 11, 600, tols, **hist)
    ref = R.mc_run(to_ref(R, net), 50, 75, f, specs, R.mc_cfg(11, 600, tols, **hist), nthreads=8)
    _assert_counts_equal(ref, got)
    assert 0 < got["n_pass"] < 600
    gs = ctx.mc_run(net, f[:301], [], 11, 9, tols, mode=Q.MODE_FULL_S)["s"]
    os_ = R.mc_run(to_ref(R, net), 50, 75, f[:301], [], R.mc_cfg(11, 9, tols), full_s=True)["s"]
    _s_close(gs, os_)
    # non-reciprocal block (the 20 W driver measurement): S12 != S21 must survive the cascade
    R.sblock_clear()
    _, fd, sd, z0 = blk["pa_20W"]
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    amp = Q.Net.from_elements([(Q.SER_L, [1e-9, 0.1, 0.0])], 50, 50).concat(blk["pa_20W"][0].as_net(True)).concat(
        Q.Net.from_elements([(Q.SHUNT_C, [0.5e-12, 0.2, 0.0])], 50, 50))
    fa = Q.grid_lin(2e7, 9e9, 500)
    g = ctx.sweep(amp, fa)
    o = R.sweep(to_ref(R, amp), 50, 50, fa)
    for i in range(4):
        assert np.max(np.abs(g[i] - o[i])) <= 1e-9 * max(1.0, float(np.max(np.abs(o[i]))))
    assert np.max(np.abs(g[1] - g[2])) > 1e-3                     # genuinely non-reciprocal
    # bare block: the sweep returns the interpolated measurement itself
    bare = ctx.sweep(blk["pa_20W"][0].as_net(True), fd[10:20])
    assert np.allclose(np.stack([bare[0], bare[1], bare[2], bare[3]], 1), sd[10:20], rtol=1e-9, atol=1e-12)
    R.sblock_clear()


def test_tf_kernel_front_block_line_and_measured_two_port(Q, R, W, ctx, golden_s2p, monkeypatch):
    """A transmission line (perturbed Z0 and length) or a measured two-port (the Coilcraft inductor of
    pa-bias-simulation.sch:39) in FRONT of a lumped ladder runs on the transfer-function kernel: the block's row vector
    [1 Rs] M is evaluated per point and contracted with the polynomials of the ladder behind it.  Counters and histogram
    equal the interpreter's (QO100NET_TF_NO_FRONT=1) and the oracle's."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    fc = 10e6
    lad, f, ltol = _ladder_workload(Q, W, 7, True, False, nf=700)
    n = 3000
    # (a) 75 Ohm line, 35 deg at fc, in a 50 Ohm system: Z0 +-5 %, length +-3 %
    line = Q.Net.from_elements([(Q.TLINE, [75.0, 35.0, fc])], 50.0, 50.0)
    net = line.concat(lad)
    tols = [(0, 0, 0, Q.TOL_REL, 0.05), (0, 1, 1, Q.TOL_REL, 0.03)] + [(e + 1, p_, v + 2, m, t) for (e, p_, v, m, t) in ltol]
    nom = ctx.sweep(net, f)
    db = 20 * np.log10(np.abs(nom[1]))
    pb, sb = f <= 0.9 * fc, f >= 2.0 * fc
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, 0.9 * fc, float(db[pb].min()) - 0.25), (Q.SPEC_S21_MAX_DB, 2.0 * fc, 1e99, float(db[sb].max()) + 1.0)]
    hist = dict(hist_bins=32, hist_spec=0, hist_lo=float(db[pb].min()) - 2.0, hist_hi=float(db[pb].min()) + 0.5)
    plan = Q.Plan(ctx, net, f, specs, seed=9, tols=tols, **hist)
    assert plan.kernel_name == "qo_mc_tf_kernel" and plan.tf_info["numerator_chains"] == 4
    plan.launch(2 ** 33 + 3, n)
    got = plan.read()
    plan.close()
    monkeypatch.setenv("QO100NET_TF_NO_FRONT", "1")
    plan = Q.Plan(ctx, net, f, specs, seed=9, tols=tols, **hist)
    assert plan.kernel_name == "qo_mc_lumped_kernel"
    plan.launch(2 ** 33 + 3, n)
    interp = plan.read()
    plan.close()
    monkeypatch.delenv("QO100NET_TF_NO_FRONT", raising=False)
    _assert_counts_equal(interp, got)
    ref = R.mc_run(to_ref(R, net), 50, 50, f, specs, R.mc_cfg(9, n, tols, sample_offset=2 ** 33 + 3, **hist), nthreads=8)
    _assert_counts_equal(ref, got)
    assert 0 < got["n_pass"] < n
    # (b) the measured inductor in front (no tolerances on the block), rectangular and polar interpolation
    fd, sd, z0 = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"], float(golden_s2p["11SQ39N_z0"])
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    R.sblock_clear()
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    lad2, f2, ltol2 = _ladder_workload(Q, W, 5, False, False, fc=400e6, nf=513)
    for polar in (True, False):
        net2 = blk.as_net(polar, 50.0, 50.0).concat(lad2)
        tols2 = [(e + 1, p_, v, m, t) for (e, p_, v, m, t) in ltol2]
        nom = ctx.sweep(net2, f2)
        db = 20 * np.log10(np.abs(nom[1]))
        pb, sb = f2 <= 0.8 * 400e6, f2 >= 2.0 * 400e6
        specs2 = [(Q.SPEC_S21_MIN_DB, 0.0, 0.8 * 400e6, float(db[pb].min()) - 0.2), (Q.SPEC_S21_MAX_DB, 2.0 * 400e6, 1e99, float(db[sb].max()) + 1.5)]
        plan = Q.Plan(ctx, net2, f2, specs2, seed=4, tols=tols2)
        assert plan.kernel_name == "qo_mc_tf_kernel"
        plan.launch(17, n)
        got2 = plan.read()
        plan.close()
        ref2 = R.mc_run(to_ref(R, net2), 50, 50, f2, specs2, R.mc_cfg(4, n, tols2, sample_offset=17), nthreads=8)
        _assert_counts_equal(ref2, got2)
        assert 0 < got2["n_pass"] < n
    R.sblock_clear()


def test_tf_kernel_s11_specs_behind_a_front_block(Q, R, W, ctx, golden_s2p, monkeypatch):
    """|S11| (and mixed |S11| + |S21|) specs behind a coupled-line section, a transmission line or a measured two-port: the
    transfer-function kernel carries the block's second row vector [1 -Rs] M as well.  Counters equal the oracle's and the chain
    kernels' (QO100NET_KERNEL=ladder -> straight-line kernel for the coupler case, interpreter otherwise)."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    n = 2500
    fc = 10e6
    fd, sd, z0 = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"], float(golden_s2p["11SQ39N_z0"])
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    R.sblock_clear()
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    cases = []
    net, f, tols = _ladder_workload(Q, W, 7, True, True, nf=600)                      # coupler (theta_e != theta_o) + ladder
    cases.append(("coupler", net, f, tols, fc))
    lad, f, ltol = _ladder_workload(Q, W, 7, True, False, nf=600)
    line = Q.Net.from_elements([(Q.TLINE, [60.0, 50.0, fc])], 50.0, 50.0)
    cases.append(("line", line.concat(lad), f, [(0, 0, 0, Q.TOL_REL, 0.05), (0, 1, 1, Q.TOL_REL, 0.03)] + [(e + 1, p_, v + 2, m, t) for (e, p_, v, m, t) in ltol], fc))
    lad2, f2, ltol2 = _ladder_workload(Q, W, 5, False, False, fc=400e6, nf=513)
    cases.append(("block", blk.as_net(True, 50.0, 50.0).concat(lad2), f2, [(e + 1, p_, v, m, t) for (e, p_, v, m, t) in ltol2], 400e6))
    cases += [(name + "-short", net, f[::12], tols, fcc) for name, net, f, tols, fcc in cases]      # <= 64 points: one pair per thread
    for name, net, f, tols, fcc in cases:
        nom = ctx.sweep(net, f)
        r11 = 20 * np.log10(np.abs(nom[0]))
        db = 20 * np.log10(np.abs(nom[1]))
        pb = (f >= 0.3 * fcc) & (f <= 0.8 * fcc)
        # thresholds at the median / upper quartile of the worst in-band |S11| over a few hundred samples: never a degenerate yield
        fs = ctx.mc_run(net, f, [], 12, 300, tols, mode=Q.MODE_FULL_S)["s"]
        worst11 = (20 * np.log10(np.abs(fs[0][:, pb]))).max(axis=1)
        worst21 = (20 * np.log10(np.abs(fs[1][:, f <= 0.8 * fcc]))).min(axis=1)
        for specs in ([(Q.SPEC_S11_MAX_DB, 0.3 * fcc, 0.8 * fcc, float(np.median(worst11)))],
                      [(Q.SPEC_S11_MAX_DB, 0.3 * fcc, 0.8 * fcc, float(np.quantile(worst11, 0.75))), (Q.SPEC_S21_MIN_DB, 0.0, 0.8 * fcc, float(np.quantile(worst21, 0.25)))]):
            hist = dict(hist_bins=24, hist_spec=0, hist_lo=float(r11[pb].max()) - 6.0, hist_hi=float(r11[pb].max()) + 6.0)
            plan = Q.Plan(ctx, net, f, specs, seed=12, tols=tols, **hist)
            assert plan.kernel_name == "qo_mc_tf_kernel", (name, plan.tf_info)
            plan.launch(40, n)
            got = plan.read()
            plan.close()
            monkeypatch.setenv("QO100NET_KERNEL", "ladder")
            plan = Q.Plan(ctx, net, f, specs, seed=12, tols=tols, **hist)
            assert plan.kernel_name in ("qo_mc_ladder_kernel", "qo_mc_lumped_kernel")
            plan.launch(40, n)
            chain = plan.read()
            plan.close()
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
            _assert_counts_equal(chain, got)
            rs, rl = net.terminations
            ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(12, n, tols, sample_offset=40, **hist), nthreads=8)
            _assert_counts_equal(ref, got)
            assert 0 < got["n_pass"] < n, (name, got["n_pass"])
    R.sblock_clear()


def test_differential_fuzz_of_the_monte_carlo_kernels(monkeypatch):
    """tools/fuzz_parity.py on a fixed seed: 80 random lumped cascades (all branch kinds, front blocks, |S21| / |S11| specs at
    quantiles of a FULL_S pre-run, short and long grids, small and thread-per-sample sized launches): the selected kernel, the
    opcode interpreter and (every 5th) the oracle return identical counters.  The long runs (thousands of networks, several
    seeds) are recorded under profiles/."""
    import importlib.util
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    spec = importlib.util.spec_from_file_location("fuzz_parity", os.path.join(ROOT, "tools", "fuzz_parity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--nets", "80", "--samples", "1500", "--seed", "7", "--big-every", "5"])
    assert out["mismatches"] == 0, out["details"]
    assert out["compared"] >= 70 and out["oracle_checked"] >= 10
    assert {"qo_mc_tf_kernel", "qo_mc_ts_kernel", "qo_mc_spot_kernel"} <= set(out["kernels_selected"])


def test_differential_fuzz_of_the_compiled_chain_kernel(Q, W, monkeypatch):
    """tools/fuzz_parity.py --chain-jit on a fixed seed: 24 random lumped cascades, most with a perturbed line and / or the measured
    two-port BEHIND them (what no polynomial kernel takes), each compiled into its own chain kernel (qo_chain_jit.h): counters equal
    the interpreter's and (every 5th) the oracle's, FULL_S planes the interpreter's.  100 networks: profiles/fuzz/fuzz_r02s_chain_jit_seed91.json."""
    import importlib.util
    w5 = W.cfg5(1000)
    a = Q.chain_jit_analyze(w5.net, w5.f[:64], w5.specs[:1], w5.tols)
    if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
        pytest.skip("libnvrtc is not loadable on this box")
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_CHAIN", raising=False)
    spec = importlib.util.spec_from_file_location("fuzz_parity", os.path.join(ROOT, "tools", "fuzz_parity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--chain-jit", "--nets", "24", "--samples", "3000", "--seed", "91"])
    assert out["mismatches"] == 0, out["details"]
    assert out["compared"] >= 20 and out["oracle_checked"] >= 3 and out["full_s_checked"] >= 4
    assert set(out["kernels_selected"]) == {"qo_mc_chain_jit_kernel"}


def test_fuzz_regressions(Q, R, ctx, monkeypatch):
    """The networks on which tools/fuzz_parity.py caught the transfer-function kernels (recorded under profiles/fuzz/):
    (a) thread-per-sample kernel: the truncated E(y) goes negative beyond the last spec band on some samples and used to fail
        spec 0 through the sink that keeps unobserved points alive;
    (b) histogram on a MIN-dB spec whose band holds a trap: on a sample that resonates exactly at a grid point E(y) rounds to
        <= 0 and the negative n2 / dd used to drop out of the running maximum.
    Both must now equal the interpreter and the oracle on the recorded sample ranges."""
    import json
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    for fn, idx, kernel in (("fuzz_r02_seed5.json", 119, "qo_mc_ts_kernel"), ("fuzz_r02d_seed12.json", 1826, "qo_mc_tf_kernel"),
                            ("fuzz_r02d_seed14.json", 242, "qo_mc_tf_kernel")):
        m = next(x for x in json.load(open(os.path.join(ROOT, "profiles", "fuzz", fn)))["details"] if x["net"] == idx)
        net = Q.Net.from_elements([(k, p) for k, p in m["elements"]], *m["terminations"])
        f = Q.grid_log(m["f0"], m["f1"], m["nf"]) if m["log_grid"] else Q.grid_lin(m["f0"], m["f1"], m["nf"])
        tols, specs = [tuple(t) for t in m["tols"]], [tuple(s_) for s_ in m["specs"]]
        res = {}
        for force in (None, "interp"):
            if force:
                monkeypatch.setenv("QO100NET_KERNEL", force)
            plan = Q.Plan(ctx, net, f, specs, seed=m["seed"], tols=tols, dist=m["dist"], **m["hist"])
            plan.launch(m["offset"], m["n"])
            res[force] = plan.read()
            if not force:
                assert plan.kernel_name == kernel
            plan.close()
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        _assert_counts_equal(res["interp"], res[None])
        assert [int(v) for v in res[None]["fail_per_spec"]] == m["interp_fail"]          # what the interpreter and the oracle said then
        rs, rl = net.terminations
        ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(m["seed"], m["n"], tols, sample_offset=m["offset"], dist=m["dist"], **m["hist"]), nthreads=8)
        _assert_counts_equal(ref, res[None])


def test_group_delay_spec_in_kernel(Q, R, W, ctx, monkeypatch):
    """north_star (c): group-delay reduction in-kernel.  QO_SPEC_GD_MAX on the Monte-Carlo path: counters and the
    histogram of the worst pass-band group delay equal the oracle's (central difference of arg S21 over f (1 +- 1e-6),
    the definition of qo_sweep's gd output) -- on the transfer-function kernel, which evaluates tau analytically from the
    derivative polynomials (GD alone, GD + |S21|), and on the interpreter, which re-runs the chain at f (1 +- 1e-6)
    (forced, and the default when |S11| specs are mixed in)."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    w = W.cfg2()
    fc = 10e6
    f = w.f[::4]
    gd = ctx.sweep(w.net, f, gd=True)[4]
    band = (f >= 0.3 * fc) & (f <= 0.9 * fc)
    lim = float(gd[band].max()) * 1.01
    ideal = Q.Net.cheby_lpf(7, 0.1, fc, 50.0, True)
    gdi = ctx.sweep(ideal, f, gd=True)[4]
    limi = float(gdi[band].max()) * 1.01
    cases = [(w.net, w.tols, [(Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, lim)], 0, lim, "qo_mc_tf_kernel"),
             (w.net, w.tols, [(Q.SPEC_S21_MIN_DB, 0.0, 0.95 * fc, -2.0), (Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, lim)], 1, lim, "qo_mc_tf_kernel"),
             (w.net, w.tols, [(Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, lim), (Q.SPEC_S21_MAX_DB, 1.3 * fc, 1e99, -49.0)], 1, None, "qo_mc_tf_kernel"),
             (ideal, Q.lc_tolerances(ideal, 0.05, 0.05), [(Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, limi)], 0, limi, "qo_mc_tf_kernel"),
             (w.net, w.tols, [(Q.SPEC_S21_MIN_DB, 0.0, 0.95 * fc, -2.0), (Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, lim),
                              (Q.SPEC_S11_MAX_DB, 0.0, 0.5 * fc, -9.0)], 1, lim, "qo_mc_lumped_kernel")]
    for net, tols, specs, hs, hl, kernel in cases:
        hist = dict(hist_bins=40, hist_spec=hs, hist_lo=0.8 * hl, hist_hi=1.3 * hl) if hl else dict(hist_bins=40, hist_spec=hs, hist_lo=-60.0, hist_hi=-40.0)
        plan = Q.Plan(ctx, net, f, specs, seed=3, tols=tols, **hist)
        assert plan.kernel_name == kernel, plan.tf_info
        if kernel == "qo_mc_tf_kernel":
            assert plan.tf_info["self_check_err"] < 1e-10
        plan.close()
        got = ctx.mc_run(net, f, specs, 3, 500, tols, **hist)
        rs, rl = net.terminations
        ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(3, 500, tols, **hist), nthreads=8)
        _assert_counts_equal(ref, got)
        gi = [i for i, s in enumerate(specs) if s[0] == Q.SPEC_GD_MAX][0]
        assert 0 < got["fail_per_spec"][gi] < 500 and int(got["hist"].sum()) == 500 and np.count_nonzero(got["hist"]) > 3
        monkeypatch.setenv("QO100NET_KERNEL", "interp")
        itp = ctx.mc_run(net, f, specs, 3, 500, tols, **hist)
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        _assert_counts_equal(itp, got)
    with pytest.raises(Q.QoError):
        ctx.mc_run(w.net, f, [(Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, lim)], 3, 10, w.tols, precision=32)


def test_fp32_ladder_mode_within_1e_3_db(Q, W, ctx, monkeypatch):
    """north_star's optional FP32 mode on the straight-line ladder kernel: the per-sample worst pass-band |S21|
    stays within 1e-3 dB of the FP64 result (earth-mover distance between 4096-bin histograms over 4 dB, i.e.
    bins of 0.001 dB) and the yield moves by less than the borderline population; the FP32 interpreter agrees."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    n = 30000
    for w in (W.cfg2(), W.cfg5()):
        lo, hi = (-4.0, 0.0) if w.name.startswith("cfg2") else (-3.0, 0.0)
        hist = dict(w.hist, hist_bins=1024, hist_lo=lo, hist_hi=hi)
        r64 = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **hist)
        r32 = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, precision=32, **hist)
        assert r32["n_total"] == n and int(r32["hist"].sum()) == n
        binw = (hi - lo) / 1024
        emd = float(np.sum(np.abs(np.cumsum(r64["hist"].astype(np.int64) - r32["hist"].astype(np.int64)))) * binw / n)
        assert emd < 1e-3, emd
        assert abs(r32["n_pass"] - r64["n_pass"]) <= 0.002 * n
        monkeypatch.setenv("QO100NET_KERNEL", "interp")
        i32 = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, precision=32, **hist)
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        emd_i = float(np.sum(np.abs(np.cumsum(i32["hist"].astype(np.int64) - r32["hist"].astype(np.int64)))) * binw / n)
        assert emd_i < 1e-3 and abs(i32["n_pass"] - r32["n_pass"]) <= 0.002 * n


def test_physical_coupled_line_element(Q, R, W, ctx, monkeypatch):
    """SURVEY 8f N1 carried into the hot path: QO_CPL_MS (physical coupled microstrip, util/directional-couplers/
    dir_cpl_2.4g_20dB.trc:6-17) = coupled-microstrip analysis per sample (device pre-pass) + the ideal coupled-line
    block.  Nominal: identical to the ideal element fed with the analysis' Z0e/Z0o/theta_e/theta_o and to the
    oracle; Monte Carlo over W/S (one etch draw), H, Er and the ladder: ladder kernel == interpreter == oracle."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    w = W.cfg5p(0, 1024)
    (k_sub, p_sub), (k_cpl, p_cpl) = w.net.elements[0], w.net.elements[1]
    assert k_sub == Q.SUBST and k_cpl == Q.CPL_MS
    ze, zo, ae, ao = Q.cpl_analyze(p_cpl[0], p_cpl[1], p_sub[1], p_sub[2], p_sub[0], p_cpl[3], p_cpl[4], p_cpl[2])
    assert abs(ze / 55.2771 - 1) < 5e-6 and abs(zo / 45.2267 - 1) < 5e-6 and abs(np.sqrt(ae * ao) / 95.4225 - 1) < 5e-6   # the .trc values
    phys = Q.Net.from_elements([(Q.SUBST, p_sub), (Q.CPL_MS, p_cpl)], 50.0, 50.0)
    ideal = Q.Net.from_elements([(Q.CPL_THRU, [ze, zo, ae, ao, p_cpl[4], p_cpl[5]])], 50.0, 50.0)
    f = Q.grid_lin(70e6, 4000e6, 400)
    gp, gi = ctx.sweep(phys, f), ctx.sweep(ideal, f)
    for a, b in zip(gp, gi):
        assert np.max(np.abs(a - b)) < 1e-12
    _s_close(gp, R.sweep(to_ref(R, phys), 50, 50, f))
    _s_close(ctx.sweep(w.net, w.f), R.sweep(to_ref(R, w.net), 50, 50, w.f))
    # Monte Carlo
    n = 1500
    plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
    assert plan.kernel_name == "qo_mc_tf_kernel"
    plan.launch(7, n)
    got = plan.read()
    assert plan.launches == 2                      # pre-pass + Monte-Carlo kernel
    plan.close()
    rs, rl = w.net.terminations
    ref = R.mc_run(to_ref(R, w.net), rs, rl, w.f, w.specs, R.mc_cfg(w.seed, n, w.tols, sample_offset=7, **w.hist), nthreads=8)
    _assert_counts_equal(ref, got)
    assert 0 < got["n_pass"] < n and np.count_nonzero(got["hist"]) > 10
    for env in (("QO100NET_KERNEL", "interp"), ("QO100NET_KERNEL", "ladder"), ("QO100NET_CPL_SINCOS", "1")):
        monkeypatch.setenv(*env)
        alt = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, sample_offset=7, **w.hist)
        monkeypatch.delenv(env[0])
        _assert_counts_equal(alt, got)
    gs = ctx.mc_run(w.net, w.f[:200], [], w.seed, 6, w.tols, mode=Q.MODE_FULL_S)["s"]
    os_ = R.mc_run(to_ref(R, w.net), rs, rl, w.f[:200], [], R.mc_cfg(w.seed, 6, w.tols), full_s=True)["s"]
    _s_close(gs, os_)
    # the draws matter: with tolerances the coupler's mid-band |S21| spreads
    assert np.std(20 * np.log10(np.abs(gs[1][:, 100]))) > 1e-4


def _mixed_lumped_nets(Q, W):
    """Lumped cascades outside the L/C ladder family: rf-tools filters with tanks and traps (util/if-bandpass-filter/
    schematic.svg:191-213, docs/gpsdo-filters/*.svg:195-241), unequal terminations (gpsdo 10M, 100/50 Ohm), and every
    remaining branch kind (series/shunt R, lossy shunt L, lossy series C, series tank, shunt tank)."""
    out = [("if-bpf", W.if_bpf_net(), 400e6)]
    for name, net, fc in W.gpsdo_bank():
        out.append(("gpsdo-" + name, net, fc))
    fc = 50e6
    wc = 2 * np.pi * fc
    mixed = Q.Net.from_elements([
        (Q.SER_R, [2.0]), (Q.SER_C, [40.0 / (50 * wc), 0.2, 1.0e-9]), (Q.SHUNT_L, [50 / (3.0 * wc), 0.5, 0.3e-12]),
        (Q.SER_LC_PAR, [50 / (6 * wc), 6 / (50 * wc * 9.0)]), (Q.SHUNT_R, [2000.0]), (Q.SHUNT_LC_PAR, [50 * 3 / wc, 1 / (50 * 3 * wc * 0.04)]),
        (Q.SER_L, [50 * 0.2 / wc, 0.3, 0.2e-12]), (Q.SHUNT_C, [0.2 / (50 * wc), 0.05, 0.5e-9]), (Q.SER_LC_SER, [50 * 0.1 / wc, 30 / (50 * wc)]),
    ], 50.0, 75.0)
    out.append(("mixed", mixed, fc))
    return out


def test_tf_kernel_general_lumped_networks(Q, R, W, ctx, monkeypatch):
    """The transfer-function kernel covers every lumped branch kind (each is a ratio of real polynomials in s):
    its integer counters equal the oracle's and the opcode interpreter's -- with a histogram on a MIN-dB spec, on a
    MAX-dB spec, without histogram (sign trackers only), uniform and gaussian draws, grids that end inside an iteration."""
    for name, net, fc in _mixed_lumped_nets(Q, W):
        for nf, hist_on, dist in ((1000, 0, Q.DIST_UNIFORM), (515, 1, Q.DIST_GAUSS3S), (4096, None, Q.DIST_UNIFORM)):
            f = Q.grid_log(fc / 3.0, fc * 4.0, nf)
            db = 20 * np.log10(np.abs(ctx.sweep(net, f)[1]))
            peak = float(db.max())
            pb = db >= peak - 1.0
            f_lo, f_hi = float(f[pb].min()), float(f[pb].max())
            f_sb = min(3.5 * fc, 2.5 * f_hi)
            sb = f >= f_sb
            inb = (f >= f_lo * 1.02) & (f <= f_hi * 0.98)
            specs = [(Q.SPEC_S21_MIN_DB, f_lo * 1.02, f_hi * 0.98, float(db[inb].min()) - 0.1), (Q.SPEC_S21_MAX_DB, f_sb, 1e99, float(db[sb].max()) + 1.5),
                     (Q.SPEC_S21_MAX_DB, f[0], f[3], peak + 3.0)]
            tols = Q.lc_tolerances(net, 0.05, 0.05)
            if hist_on is None:
                hist = {}
            elif hist_on == 0:
                hist = dict(hist_bins=48, hist_spec=0, hist_lo=peak - 4.0, hist_hi=peak)
            else:
                hist = dict(hist_bins=48, hist_spec=1, hist_lo=float(db[sb].max()) - 6.0, hist_hi=float(db[sb].max()) + 6.0)
            n = 600
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
            plan = Q.Plan(ctx, net, f, specs, seed=21, tols=tols, dist=dist, **hist)
            assert plan.kernel_name == "qo_mc_tf_kernel", name
            plan.launch(3, n)
            got = plan.read()
            plan.close()
            rs, rl = net.terminations
            ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(21, n, tols, sample_offset=3, dist=dist, **hist), nthreads=8)
            _assert_counts_equal(ref, got)
            assert got["n_pass"] < n and int(got["fail_per_spec"].sum()) > 0, (name, got["n_pass"])
            monkeypatch.setenv("QO100NET_KERNEL", "interp")
            itp = ctx.mc_run(net, f, specs, 21, n, tols, sample_offset=3, dist=dist, **hist)
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
            _assert_counts_equal(itp, got)


@pytest.mark.parametrize("which", ["cfg2", "cfg5"])
def test_tf_kernel_equals_chain_kernel_at_2e6_samples(Q, W, ctx, monkeypatch, which):
    """BASELINE configs 2 and 5 at 2e6 samples x 4096 points: the transfer-function kernel (polynomial expansion + Horner) and
    the straight-line ABCD-chain kernel (QO100NET_KERNEL=ladder) return identical integers -- n_pass, every fail_per_spec and
    all 256 histogram bins -- although they round differently (the plan's self-check bounds the difference at 1e-10 relative on
    |den|^2, see self_check_err, the max over 33 points of the tolerance box)."""
    w = W.cfg2() if which == "cfg2" else W.cfg5()
    n = 2000000
    res = {}
    for kern in ("tf", "ladder"):
        if kern == "ladder":
            monkeypatch.setenv("QO100NET_KERNEL", "ladder")
        else:
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
        assert plan.kernel_name == ("qo_mc_tf_kernel" if kern == "tf" else "qo_mc_ladder_kernel")
        if kern == "tf":
            info = plan.tf_info
            assert info["selected"] and info["self_check_err"] < 1e-10, info
        plan.launch(777, n)
        res[kern] = plan.read()
        plan.close()
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    a, b = res["tf"], res["ladder"]
    assert a["n_total"] == b["n_total"] == n and a["n_pass"] == b["n_pass"]
    assert np.array_equal(a["fail_per_spec"], b["fail_per_spec"]) and np.array_equal(a["hist"], b["hist"])
    assert int(a["hist"].sum()) == n and 0.5 < a["n_pass"] / n < 0.8


@pytest.mark.parametrize("which", ["cfg2", "cfg5", "ideal11", "if_bpf"])
def test_thread_per_sample_kernel_equals_warp_per_sample_and_oracle(Q, R, W, ctx, monkeypatch, which):
    """Large launches run thread-per-sample (qo_mc_ts_kernel: coefficients in registers, truncated in-register expansion); what
    is left of a launch after whole 32-sample batches, and every small launch, runs warp-per-sample (qo_mc_tf_kernel).  Same
    integers from both, for a sample count that is NOT a multiple of 32 and an offset beyond 2^32; a slice of the same range
    against the oracle."""
    import torch
    if which == "cfg2":
        w = W.cfg2()
    elif which == "cfg5":
        w = W.cfg5()
    elif which == "ideal11":
        fc = 10e6
        net = Q.Net.cheby_lpf(11, 0.1, fc, 50.0, True)
        w = W.Workload("ideal11", net, Q.grid_log(fc / 2.5, fc * 6.25, 1003), [(Q.SPEC_S21_MIN_DB, 0.0, 0.95 * fc, -0.5), (Q.SPEC_S21_MAX_DB, 1.3 * fc, 1e99, -49.0)],
                       Q.lc_tolerances(net, 0.05, 0.02), dict(hist_bins=64, hist_spec=1, hist_lo=-80.0, hist_hi=-40.0), 0, 13)
    else:
        net = W.if_bpf_net()
        f = Q.grid_log(300e6 / 3.5, 500e6 * 3.5, 2050)
        db = 20 * np.log10(np.abs(ctx.sweep(net, f)[1]))
        pb = (f >= 3.6e8) & (f <= 4.4e8)
        w = W.Workload("ifbpf", net, f, [(Q.SPEC_S21_MIN_DB, 3.6e8, 4.4e8, float(db[pb].min()) - 0.3), (Q.SPEC_S21_MAX_DB, 9e8, 1e99, float(db[f >= 9e8].max()) + 1.0),
                                         (Q.SPEC_S21_MAX_DB, 0.0, 1.5e8, float(db[f <= 1.5e8].max()) + 1.0)],
                       Q.lc_tolerances(net, 0.05, 0.05), dict(hist_bins=64, hist_spec=0, hist_lo=-6.0, hist_hi=0.0), 0, 11)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * sm * 4 * 128 + 37 * 32 + 19                 # enough for the thread-per-sample path, not a multiple of 32
    off = (1 << 33) + 12345
    res = {}
    for kern in ("auto", "tf"):
        if kern == "tf":
            monkeypatch.setenv("QO100NET_KERNEL", "tf")
        else:
            monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
        plan.launch(off, n)
        res[kern] = plan.read()
        assert plan.kernel_name == ("qo_mc_ts_kernel" if kern == "auto" else "qo_mc_tf_kernel"), (kern, plan.kernel_name)
        plan.close()
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    _assert_counts_equal(res["tf"], res["auto"])
    assert res["auto"]["n_total"] == n and 0 < res["auto"]["n_pass"] < n and int(res["auto"]["hist"].sum()) == n
    # the first 3000 samples of the range against the oracle (small launch: warp-per-sample) ...
    m = 3000
    rs, rl = w.net.terminations
    og = R.mc_run(to_ref(R, w.net), rs, rl, w.f, w.specs, R.mc_cfg(w.seed, m, w.tols, sample_offset=off, **w.hist), nthreads=8)
    gg = ctx.mc_run(w.net, w.f, w.specs, w.seed, m, w.tols, sample_offset=off, **w.hist)
    _assert_counts_equal(og, gg)
    # ... and additivity ties the big thread-per-sample launch to it: [off, off+n) = [off, off+m) + [off+m, off+n)
    rest = ctx.mc_run(w.net, w.f, w.specs, w.seed, n - m, w.tols, sample_offset=off + m, **w.hist)
    assert gg["n_pass"] + rest["n_pass"] == res["auto"]["n_pass"]
    assert np.array_equal(gg["hist"] + rest["hist"], res["auto"]["hist"]) and np.array_equal(gg["fail_per_spec"] + rest["fail_per_spec"], res["auto"]["fail_per_spec"])


def test_tf_kernel_values_within_1e_9(Q, W, ctx, monkeypatch):
    """north_star's FP64 tolerance on the transfer-function path, measured on VALUES rather than verdicts: the
    per-sample worst pass-band |S21| lands in the same bin of a 1024-bin histogram only 2e-3 dB wide (bins of
    2e-6 dB) as the chain kernel's for all but a handful of the samples -- a 1e-9 relative error on |S21| is
    8.7e-9 dB, i.e. 0.4 % of a bin."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    n = 20000
    for w in (W.cfg2(), W.cfg5()):
        hs = w.hist["hist_spec"]
        coarse = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **dict(w.hist, hist_bins=1024))
        width = (w.hist["hist_hi"] - w.hist["hist_lo"]) / 1024
        b = int(np.argmax(coarse["hist"][1:-1])) + 1                     # the most populated interior bin
        lo = w.hist["hist_lo"] + b * width
        fine = dict(hist_bins=1024, hist_spec=hs, hist_lo=lo + 0.4 * width, hist_hi=lo + 0.4 * width + 2e-3)
        tf = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **fine)
        monkeypatch.setenv("QO100NET_KERNEL", "ladder")
        ch = ctx.mc_run(w.net, w.f, w.specs, w.seed, n, w.tols, **fine)
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        inside = int(ch["hist"][1:-1].sum())
        assert inside >= 20, inside                                      # enough samples land in the 2e-3 dB window
        moved = int(np.abs(tf["hist"].astype(np.int64) - ch["hist"].astype(np.int64)).sum()) // 2
        assert moved <= max(2, inside // 50), (moved, inside)
        assert tf["n_pass"] == ch["n_pass"] and np.array_equal(tf["fail_per_spec"], ch["fail_per_spec"])


def test_tf_kernel_size_limits_and_degenerate_degrees(Q, R, W, ctx, monkeypatch):
    """Edges of the transfer-function kernel's coverage: a resistive pad (degree 0: one coefficient pair), a single
    reactive branch, a 24-branch ideal ladder (degree 24, the element limit), four specs at once; one branch more, or a
    total degree above 29, hands the job to the interpreter -- every case equal to the oracle's counters."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    fc = 20e6
    wc = 2 * np.pi * fc
    f = Q.grid_log(fc / 2.5, fc * 2.5, 300)

    def run(net, specs, tols, expect, f=f, **hist):
        plan = Q.Plan(ctx, net, f, specs, seed=31, tols=tols, **hist)
        assert plan.kernel_name == expect, (plan.kernel_name, plan.tf_info)
        info = plan.tf_info
        plan.launch(11, 400)
        got = plan.read()
        plan.close()
        rs, rl = net.terminations
        ref = R.mc_run(to_ref(R, net), rs, rl, f, specs, R.mc_cfg(31, 400, tols, sample_offset=11, **hist), nthreads=8)
        _assert_counts_equal(ref, got)
        return got, info

    pad = Q.Net.from_elements([(Q.SHUNT_R, [292.4]), (Q.SER_R, [17.6]), (Q.SHUNT_R, [292.4])], 50.0, 50.0)      # 3 dB pi pad
    tol_r = [(0, 0, 0, Q.TOL_REL, 0.05), (1, 0, 1, Q.TOL_REL, 0.05), (2, 0, 2, Q.TOL_REL, 0.05)]
    got, info = run(pad, [(Q.SPEC_S21_MIN_DB, 0.0, 1e99, -3.05), (Q.SPEC_S21_MAX_DB, 0.0, 1e99, -2.95)], tol_r, "qo_mc_tf_kernel",
                    hist_bins=20, hist_spec=0, hist_lo=-3.3, hist_hi=-2.7)
    assert info["degree"] == 0 and info["kn"] == 2 and 0 < got["n_pass"] < 400      # a constant is padded with a zero row (kn >= 2)
    one = Q.Net.from_elements([(Q.SER_L, [50.0 / wc])], 50.0, 50.0)
    got, info = run(one, [(Q.SPEC_S21_MIN_DB, 0.0, fc, -1.0)], [(0, 0, 0, Q.TOL_REL, 0.1)], "qo_mc_tf_kernel")
    assert info["degree"] == 1 and 0 < got["n_pass"] < 400
    g = [1.0 + 0.6 * np.sin(0.7 * k) for k in range(26)]
    long_el = [((Q.SER_L, [50.0 * g[k] / wc]) if k % 2 == 0 else (Q.SHUNT_C, [g[k] / (50.0 * wc)])) for k in range(26)]
    net24 = Q.Net.from_elements(long_el[:24], 50.0, 50.0)
    db = 20 * np.log10(np.abs(ctx.sweep(net24, f)[1]))
    pb, sb = f <= 0.5 * fc, f >= 2.0 * fc
    specs4 = [(Q.SPEC_S21_MIN_DB, 0.0, 0.5 * fc, float(db[pb].min()) - 0.05), (Q.SPEC_S21_MAX_DB, 2.0 * fc, 1e99, float(db[sb].max()) + 2.0),
              (Q.SPEC_S21_MIN_DB, 0.0, 0.45 * fc, float(db[f <= 0.45 * fc].min()) - 0.05), (Q.SPEC_S21_MAX_DB, 2.2 * fc, 1e99, float(db[f >= 2.2 * fc].max()) + 1.0)]
    got, info = run(net24, specs4, Q.lc_tolerances(net24, 0.03, 0.03), "qo_mc_tf_kernel", hist_bins=32, hist_spec=3,
                    hist_lo=float(db[f >= 2.2 * fc].max()) - 5.0, hist_hi=float(db[f >= 2.2 * fc].max()) + 5.0)
    assert info["degree"] == 24 and info["den_form"] == "none" and int(got["fail_per_spec"].sum()) > 0
    # the same network on a grid 16:1 wide: the plan's self-check rejects the 24th-degree expansion, the interpreter takes the job
    fw = Q.grid_log(fc / 4, fc * 4, 300)
    _, info = run(net24, specs4[:2], Q.lc_tolerances(net24, 0.03, 0.03), "qo_mc_lumped_kernel", f=fw)
    assert info["reason"] == "polynomial expansion is too ill-conditioned on this grid" and info["self_check_err"] > 1e-10
    net25 = Q.Net.from_elements(long_el[:25], 50.0, 50.0)
    run(net25, specs4[:2], Q.lc_tolerances(net25, 0.03, 0.03), "qo_mc_lumped_kernel")                      # one branch too many
    lossy15 = Q.Net.from_elements(long_el[:15], 50.0, 50.0).add_parasitics(fc, 60.0, 30.0, 0.1, 50.0)   # 15 lossy branches: degree 30
    run(lossy15, specs4[:2], Q.lc_tolerances(lossy15, 0.03, 0.03), "qo_mc_lumped_kernel")


def test_tf_kernel_eight_specs(Q, R, W, ctx, monkeypatch):
    """5-8 specs take the 8-slot instantiation of the transfer-function kernel: |S21| min/max bands, |S11|, with the
    histogram on a high slot, on a grid whose band edges cut through iterations -- counters equal the oracle's and the
    interpreter's."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    w = W.cfg2()
    fc = 10e6
    f = w.f[::3]
    db = 20 * np.log10(np.abs(ctx.sweep(w.net, f)[1]))

    def lo(a, b, margin):      # |S21| >= (nominal worst in [a, b]) - margin
        return (Q.SPEC_S21_MIN_DB, a, b, float(db[(f >= a) & (f <= b)].min()) - margin)

    def hi(a, b, margin):      # |S21| <= (nominal worst in [a, b]) + margin
        return (Q.SPEC_S21_MAX_DB, a, b, float(db[(f >= a) & (f <= min(b, f[-1]))].max()) + margin)

    base = [lo(0.0, 0.95 * fc, 0.15), hi(1.3 * fc, 1e99, 1.4), lo(0.0, 0.5 * fc, 0.03), hi(2.0 * fc, 3.0 * fc, 1.0), hi(3.0 * fc, 1e99, 1.0),
            lo(0.6 * fc, 0.9 * fc, 0.05), hi(1.5 * fc, 1.6 * fc, 1.5), lo(0.9 * fc, 0.97 * fc, 0.3)]
    h4 = float(db[f >= 3.0 * fc].max())
    cases = [(base[:5], 4, (h4 - 4.0, h4 + 4.0)), (base, 7, (-4.0, 0.0)), (base[:6] + [(Q.SPEC_S11_MAX_DB, 0.0, 0.8 * fc, -8.0)], 6, (-20.0, 0.0))]
    for specs, hs, (lo, hi) in cases:
        hist = dict(hist_bins=50, hist_spec=hs, hist_lo=lo, hist_hi=hi)
        plan = Q.Plan(ctx, w.net, f, specs, seed=17, tols=w.tols, **hist)
        assert plan.kernel_name == "qo_mc_tf_kernel", plan.tf_info
        plan.launch(2, 900)
        got = plan.read()
        plan.close()
        ref = R.mc_run(to_ref(R, w.net), 50, 50, f, specs, R.mc_cfg(17, 900, w.tols, sample_offset=2, **hist), nthreads=8)
        _assert_counts_equal(ref, got)
        assert np.count_nonzero(got["fail_per_spec"]) >= 3 and np.count_nonzero(got["hist"]) > 3
        monkeypatch.setenv("QO100NET_KERNEL", "interp")
        itp = ctx.mc_run(w.net, f, specs, 17, 900, w.tols, sample_offset=2, **hist)
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        _assert_counts_equal(itp, got)


def test_full_s_transfer_function_flavour(Q, R, W, ctx, monkeypatch):
    """FULL_S launches of >= 1024 samples on lumped cascades run on qo_fs_tf_kernel (S11, S21 = S12, S22 from the Num, N11, N22, D
    polynomials): planes within 1e-9 of the oracle and of the interpreter (forced), odd grid sizes and unequal terminations
    included; smaller launches and nets with a line or a coupler stay on the interpreter."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    n = 1100
    jobs = [(w.net, w.f, w.tols, w.seed) for w in W.cfg4(n, 640)] + [(W.cfg2().net, W.cfg2(0, 513).f, W.cfg2().tols, 7)]
    fc = 50e6
    jobs.append((_mixed_lumped_nets(Q, W)[-1][1], Q.grid_log(fc / 3, fc * 4, 301), Q.lc_tolerances(_mixed_lumped_nets(Q, W)[-1][1], 0.05, 0.05), 9))
    for net, f, tols, seed in jobs:
        rs, rl = net.terminations
        plan = Q.Plan(ctx, net, f, [], seed=seed, tols=tols, mode=Q.MODE_FULL_S)
        assert plan.kernel_name == "qo_mc_lumped_kernel"          # decided at the first large launch
        plan.close()
        g = ctx.mc_run(net, f, [], seed, n, tols, mode=Q.MODE_FULL_S)["s"]
        o = R.mc_run(to_ref(R, net), rs, rl, f, [], R.mc_cfg(seed, n, tols), full_s=True, nthreads=8)["s"]

        def close(a, b):
            """_s_close with an absolute floor of -120 dB on S21 / S12.  Among 1100 x nf random (sample, frequency) points one
            lands within 0.1 ppm of the transmission zero of an ideal tank / trap (|S21| ~ -170 dB); there 1 - w^2 L C cancels to
            7 digits in EVERY formulation (oracle, interpreter, transfer function differ from each other by ~1e-9 relative), so a
            purely relative bound would test rounding luck, not the kernel."""
            for pl in (1, 2):
                assert np.all(np.abs(a[pl] - b[pl]) <= TOL64 * np.maximum(np.abs(b[pl]), 1e-6))
            for pl in (0, 3):
                assert np.all(np.abs(a[pl] - b[pl]) <= TOL64 * np.maximum(np.abs(b[pl]), 0.02))

        close(g, o)
        monkeypatch.setenv("QO100NET_KERNEL", "interp")
        i = ctx.mc_run(net, f, [], seed, n, tols, mode=Q.MODE_FULL_S)["s"]
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        close(g, i)
        assert np.max(np.abs(g[1] - i[1])) > 0                     # two different kernels produced them
        assert np.array_equal(g[1], g[2])                          # reciprocal cascade: S12 == S21
    # which kernel ran is visible on a resident plan after the launch
    import torch
    w = W.cfg4(2048, 256)[1]
    plan = Q.Plan(ctx, w.net, w.f, [], seed=1, tols=w.tols, mode=Q.MODE_FULL_S)
    buf = torch.empty((4, 2048, 256, 2), dtype=torch.float64, device="cuda")
    plan.launch(0, 2048, None, buf.data_ptr())
    torch.cuda.synchronize()
    assert plan.kernel_name == "qo_fs_tf_kernel"
    plan.close()
    tl = Q.Net.from_elements([(Q.TLINE, [50.0, 90.0, 1e9])] + w.net.elements, 50.0, 50.0)
    plan = Q.Plan(ctx, tl, w.f, [], seed=1, mode=Q.MODE_FULL_S)
    plan.launch(0, 2048, None, buf.data_ptr())
    torch.cuda.synchronize()
    assert plan.kernel_name == "qo_mc_lumped_kernel"
    plan.close()


def test_compiled_chain_kernel_equals_interpreter_and_oracle(Q, R, W, ctx, golden_s2p, monkeypatch):
    """Cascades the polynomial kernels cannot take -- a line INSIDE the ladder and a measured two-port BEHIND it
    (pa-bias-simulation.sch:39 has the SPfile block in mid-network), FULL_S behind the coupled line of dir_cpl_2.4g_20dB.trc:18-20,
    group delay next to an |S11| spec -- on the run-time compiled chain kernel (QO100NET_CHAIN=jit; by default from 2e10 evals
    per launch on): the interpreter's source with the element list folded in.  Integer counters and histograms equal the
    interpreter's and the oracle's, FULL_S planes equal the interpreter's to rounding and the oracle's within 1e-9."""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_CHAIN", raising=False)
    w5 = W.cfg5(1000)
    a = Q.chain_jit_analyze(w5.net, w5.f, w5.specs, w5.tols, **w5.hist)
    if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
        pytest.skip("libnvrtc is not loadable on this box: the compiled chain kernel is not available (%s)" % a["error"])
    assert a["compiled"], a

    def both(net, f, specs, seed, n, tols, hist, off=0, force_interp_kernel=False):
        out = {}
        for mode in ("jit", "interp"):
            monkeypatch.setenv("QO100NET_CHAIN", mode)
            if force_interp_kernel:
                monkeypatch.setenv("QO100NET_KERNEL", "interp")
            plan = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **hist)
            assert plan.kernel_name == "qo_mc_lumped_kernel", plan.kernel_name        # what the plan would run without the compilation
            plan.launch(off, n)
            out[mode] = plan.read()
            assert plan.kernel_name == ("qo_mc_chain_jit_kernel" if mode == "jit" else "qo_mc_lumped_kernel")
            plan.close()
        monkeypatch.delenv("QO100NET_CHAIN", raising=False)
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        _assert_counts_equal(out["interp"], out["jit"])
        return out["jit"]

    # (a) ladder half - 75 Ohm line (perturbed) - ladder half - measured inductor - series R; |S21| x 2 + |S11| specs, histogram
    fc = 10e6
    fd, sd, z0 = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"], float(golden_s2p["11SQ39N_z0"])
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    R.sblock_clear()
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    lad, f, ltol = _ladder_workload(Q, W, 7, True, False, nf=700)
    el = lad.elements
    first = Q.Net.from_elements([(k, list(p)) for k, p in el[:3]], 50.0, 50.0)
    second = Q.Net.from_elements([(k, list(p)) for k, p in el[3:]], 50.0, 50.0)
    line = Q.Net.from_elements([(Q.TLINE, [75.0, 20.0, fc])], 50.0, 50.0)
    tail = Q.Net.from_elements([(Q.SER_R, [2.2])], 50.0, 50.0)
    net = first.concat(line).concat(second).concat(blk.as_net(True, 50.0, 50.0)).concat(tail)
    tols = [(e if e < 3 else e + 1, p_, v, m, t) for (e, p_, v, m, t) in ltol]
    nv = 1 + max(t[2] for t in tols)
    tols += [(3, 0, nv, Q.TOL_REL, 0.05), (3, 1, nv + 1, Q.TOL_REL, 0.03), (len(el) + 2, 0, nv + 2, Q.TOL_REL, 0.1)]
    nom = ctx.sweep(net, f)
    db, db11 = 20 * np.log10(np.abs(nom[1])), 20 * np.log10(np.abs(nom[0]))
    pb, sb = f <= 0.9 * fc, f >= 2.0 * fc
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, 0.9 * fc, float(db[pb].min()) - 0.3), (Q.SPEC_S21_MAX_DB, 2.0 * fc, 1e99, float(db[sb].max()) + 1.0),
             (Q.SPEC_S11_MAX_DB, 0.0, 0.5 * fc, float(db11[f <= 0.5 * fc].max()) + 1.5)]
    hist = dict(hist_bins=32, hist_spec=0, hist_lo=float(db[pb].min()) - 2.0, hist_hi=float(db[pb].min()) + 0.5)
    n = 3000
    got = both(net, f, specs, 21, n, tols, hist, off=2 ** 34 + 5)
    ref = R.mc_run(to_ref(R, net), 50, 50, f, specs, R.mc_cfg(21, n, tols, sample_offset=2 ** 34 + 5, **hist), nthreads=8)
    _assert_counts_equal(ref, got)
    assert 0 < got["n_pass"] < n and int(got["hist"].sum()) == n
    R.sblock_clear()

    # (b) group delay next to an |S11| spec (the job test_group_delay_spec_in_kernel leaves to the interpreter)
    w2 = W.cfg2()
    f2 = w2.f[::4]
    gd = ctx.sweep(w2.net, f2, gd=True)[4]
    band = (f2 >= 0.3 * fc) & (f2 <= 0.9 * fc)
    lim = float(gd[band].max()) * 1.01
    specs2 = [(Q.SPEC_S21_MIN_DB, 0.0, 0.95 * fc, -2.0), (Q.SPEC_GD_MAX, 0.3 * fc, 0.9 * fc, lim), (Q.SPEC_S11_MAX_DB, 0.0, 0.5 * fc, -9.0)]
    hist2 = dict(hist_bins=40, hist_spec=1, hist_lo=0.8 * lim, hist_hi=1.3 * lim)
    got2 = both(w2.net, f2, specs2, 3, 500, w2.tols, hist2)
    ref2 = R.mc_run(to_ref(R, w2.net), 50, 50, f2, specs2, R.mc_cfg(3, 500, w2.tols, **hist2), nthreads=8)
    _assert_counts_equal(ref2, got2)
    assert 0 < got2["fail_per_spec"][1] < 500

    # (c) the headline ladder forced onto the chain (QO100NET_KERNEL=interp keeps it off the polynomial kernels): same integers as the
    # default kernel at 20 000 samples
    got3 = both(w2.net, w2.f, w2.specs, w2.seed, 20000, w2.tols, w2.hist, force_interp_kernel=True)
    dflt = ctx.mc_run(w2.net, w2.f, w2.specs, w2.seed, 20000, w2.tols, **w2.hist)
    _assert_counts_equal(dflt, got3)

    # (d) FULL_S behind the coupler: planes of the compiled kernel vs the interpreter's and the oracle's
    import torch
    nf, ns = 1001, 300
    f5 = w5.f[:nf]
    planes = {}
    for mode in ("jit", "interp"):
        monkeypatch.setenv("QO100NET_CHAIN", mode)
        plan = Q.Plan(ctx, w5.net, f5, [], seed=w5.seed, tols=w5.tols, mode=Q.MODE_FULL_S)
        buf = torch.zeros((4, ns, nf, 2), dtype=torch.float64, device="cuda")
        plan.launch(7, ns, None, buf.data_ptr())
        torch.cuda.synchronize()
        assert plan.kernel_name == ("qo_mc_chain_jit_kernel" if mode == "jit" else "qo_mc_lumped_kernel"), plan.kernel_name
        plan.close()
        planes[mode] = torch.view_as_complex(buf).cpu().numpy()
    monkeypatch.delenv("QO100NET_CHAIN", raising=False)
    assert np.max(np.abs(planes["jit"][1])) > 0.5
    for i in range(4):
        assert np.max(np.abs(planes["jit"][i] - planes["interp"][i])) <= 1e-13
    os_ = R.mc_run(to_ref(R, w5.net), 50, 50, f5, [], R.mc_cfg(w5.seed, 12, w5.tols, sample_offset=7), full_s=True)["s"]
    _s_close([planes["jit"][i][:12] for i in range(4)], os_)
