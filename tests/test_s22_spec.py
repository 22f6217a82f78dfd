"""Output-port return loss: |S22| specs (QO_SPEC_S22_MAX_DB) on cascade Monte-Carlo jobs.

Every lumped branch and every lossless line is a symmetric, reciprocal two-port, so S22 of a cascade N between (Rs, Rl) is S11
of the reversed cascade rev(N) between (Rl, Rs).  The planner runs an |S22| job on the spot, transfer-function or ladder kernel
as the |S11| job on rev(N); everything else (a coupled line or measured block, |S11| and |S22| in one job, FP32, the interpreter
override) evaluates S22 directly on the interpreter or the compiled chain kernel.  The host-only tests pin the oracle and the
planner's decisions; the GPU tests check both routes against the oracle, against each other and against the reversed job."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

N_ORACLE = 400


# ---- networks ---------------------------------------------------------------------------------------------------------------
def reverse(Q, net, tols):
    """rev(N) between (Rl, Rs), with every tolerance on the same element"""
    rs, rl = net.terminations
    n = len(net.elements)
    return Q.Net.from_elements(list(reversed(net.elements)), rl, rs), [(n - 1 - e, p, v, m, t) for (e, p, v, m, t) in tols]


def mixed_net(Q):
    """a lossy cascade with traps and tanks: ESR / SRF inductors and capacitors, a series tank, a shunt trap, a shunt series-LC
    arm, a parallel-LC shunt, series and shunt resistors, 75 -> 50 Ohm"""
    el = [(Q.SER_L, [220e-9, 0.6, 0.4e-12]), (Q.SHUNT_C, [68e-12, 0.08, 0.6e-9]), (Q.SER_LC_PAR, [47e-9, 22e-12]),
          (Q.SHUNT_LC_SER, [120e-9, 3.3e-12]), (Q.SER_R, [1.5]), (Q.SHUNT_LC_PAR, [390e-9, 10e-12]),
          (Q.SER_C, [150e-12, 0.05, 0.8e-9]), (Q.SHUNT_R, [2200.0]), (Q.SER_LC_SER, [100e-9, 15e-12]), (Q.SHUNT_L, [680e-9, 0.9, 0.0])]
    net = Q.Net.from_elements(el, 75.0, 50.0)
    return net, Q.grid_log(8e6, 120e6, 600), 30e6


def networks(Q, W):
    """(name, net, grid, tolerances, band edges of the |S22| spec, the |S21| spec)"""
    out = []
    w2 = W.cfg2(nf=1024)
    out.append(("cfg2", w2.net, w2.f, w2.tols, (w2.f[0], 9.5e6), w2.specs[1]))
    _n, g10, fc = W.gpsdo_bank()[0]
    out.append(("gpsdo10M", g10, Q.grid_log(fc / 2.5, fc * 6.25, 800), Q.lc_tolerances(g10, 0.05, 0.05), (fc / 2.5, 0.9 * fc),
                (Q.SPEC_S21_MAX_DB, 2 * fc, 1e99, -30.0)))
    bp = W.if_bpf_net()
    out.append(("if_bpf", bp, Q.grid_log(300e6 / 3.5, 500e6 * 3.5, 700), Q.lc_tolerances(bp, 0.05, 0.05), (360e6, 440e6),
                (Q.SPEC_S21_MIN_DB, 380e6, 420e6, -3.0)))
    mx, fm, fcm = mixed_net(Q)
    out.append(("mixed", mx, fm, Q.lc_tolerances(mx, 0.05, 0.03), (fcm / 2, fcm), (Q.SPEC_S21_MIN_DB, fcm / 2, fcm, -6.0)))
    return out


def worst_db(s, f, band):
    """worst (largest) in-band |S| dB per sample of planes s[n, nf]"""
    m = (f >= band[0]) & (f <= band[1])
    return 20 * np.log10(np.abs(s[:, m])).max(axis=1)


def limit_from(v):
    """a threshold inside the spread of v: some samples pass, some fail"""
    return float(np.quantile(v, 0.45))


def oracle(R, net, f, specs, seed, n, tols, **kw):
    """the CPU oracle's counters; |S22| specs reduced from its FULL_S planes (tools/fuzz_parity.py::oracle_counters)"""
    from tools.fuzz_parity import oracle_counters
    return oracle_counters(R, net, f, specs, R.mc_cfg(seed, n, tols, **kw))


def same(a, b):
    return a["n_pass"] == b["n_pass"] and np.array_equal(a["fail_per_spec"], b["fail_per_spec"]) and np.array_equal(a["hist"], b["hist"])


def s22_limit_oracle(R, net, f, tols, band):
    rs, rl = net.terminations
    full = R.mc_run(R.make_elems(net.elements), rs, rl, f, [], R.mc_cfg(11, 64, tols), full_s=True, nthreads=R.max_threads())["s"]
    return limit_from(worst_db(full[3], f, band))


# ---- host only --------------------------------------------------------------------------------------------------------------
def test_oracle_s22_equals_reversed_s11(Q, R, W):
    """The oracle's |S22| counters on N (reduced from its FULL_S S22 plane) and its own reduction of the |S11| job on rev(N)
    (terminations swapped, tolerances remapped) are the same, integer for integer, alone and next to an |S21| spec."""
    for name, net, f, tols, band, s21 in networks(Q, W):
        lim = s22_limit_oracle(R, net, f, tols, band)
        rnet, rtols = reverse(Q, net, tols)
        for specs22 in ([(Q.SPEC_S22_MAX_DB, band[0], band[1], lim)], [s21, (Q.SPEC_S22_MAX_DB, band[0], band[1], lim)]):
            hs = len(specs22) - 1
            hist = dict(hist_bins=64, hist_spec=hs, hist_lo=lim - 8.0, hist_hi=lim + 8.0)
            a = oracle(R, net, f, specs22, 5, N_ORACLE, tols, **hist)
            specs11 = [(Q.SPEC_S11_MAX_DB if s[0] == Q.SPEC_S22_MAX_DB else s[0],) + tuple(s[1:]) for s in specs22]
            b = oracle(R, rnet, f, specs11, 5, N_ORACLE, rtols, **hist)
            assert 0 < a["fail_per_spec"][-1] < N_ORACLE, (name, a["fail_per_spec"])
            assert same(a, b), (name, a, b)


def nonrecip_block(Q, f0, f1):
    fb = np.linspace(f0, f1, 9)
    s11 = 0.2 * np.exp(1j * np.linspace(0.1, 0.9, 9))
    s21 = 0.85 * np.exp(-1j * np.linspace(0.3, 1.4, 9))
    s12 = 0.35 * np.exp(-1j * np.linspace(0.2, 1.0, 9))          # S12 != S21: no reversal can stand in for it
    s22 = 0.15j * np.exp(1j * np.linspace(0.0, 0.5, 9))
    return fb, s11, s21, s12, s22, Q.SBlock.from_arrays(fb, s11, s21, s12, s22, 50.0)


def nonrecip_net(Q, R):
    """a 5th-order Butterworth ladder behind the synthetic non-reciprocal block, registered with the oracle as block 0"""
    fc = 20e6
    fb, s11, s21, s12, s22, blk = nonrecip_block(Q, 5e6, 60e6)
    R.sblock_clear()
    R.sblock_register(0, fb, s11, s21, s12, s22, 50.0)
    lad = Q.Net.butter_lpf(5, fc, 50.0, True)
    net = blk.as_net(False, 50.0, 50.0).concat(lad)
    return net, Q.grid_lin(6e6, 50e6, 300), (fb, s11, s21, s12, s22)


def numpy_s22(net, f, blk):
    """S22 of the block (linear rectangular interpolation) + ideal ladder cascade: ABCD in numpy"""
    fb, s11, s21, s12, s22 = blk
    rs, rl = net.terminations
    out = []
    for fk in f:
        S = [np.interp(fk, fb, x.real) + 1j * np.interp(fk, fb, x.imag) for x in (s11, s21, s12, s22)]
        a11, a21, a12, a22 = S
        z0 = 50.0
        M = np.array([[((1 + a11) * (1 - a22) + a12 * a21) / (2 * a21), z0 * ((1 + a11) * (1 + a22) - a12 * a21) / (2 * a21)],
                      [((1 - a11) * (1 - a22) - a12 * a21) / (2 * a21 * z0), ((1 - a11) * (1 + a22) + a12 * a21) / (2 * a21)]])
        w = 2 * np.pi * fk
        for kind, p in net.elements[1:]:
            if kind == 3:              # SER_L
                M = M @ np.array([[1, 1j * w * p[0]], [0, 1]])
            elif kind == 6:            # SHUNT_C
                M = M @ np.array([[1, 0], [1j * w * p[0], 1]])
            else:
                raise AssertionError(kind)
        A, B, C_, D = M[0, 0], M[0, 1], M[1, 0], M[1, 1]
        den = A * rl + B + C_ * rs * rl + D * rs
        out.append((-A * rl + B - C_ * rs * rl + D * rs) / den)
    return np.array(out)


def test_oracle_s22_behind_nonreciprocal_block(Q, R):
    """On a ladder behind a non-reciprocal block (S12 != S21) with no tolerances, the oracle's worst in-band |S22| bin is the
    bin of a numpy ABCD -> S22 of the same cascade."""
    net, f, blk = nonrecip_net(Q, R)
    assert net.elements[0][0] == Q.SBLOCK
    ref = 20 * np.log10(np.abs(numpy_s22(net, f, blk)))
    band = (10e6, 30e6)
    m = (f >= band[0]) & (f <= band[1])
    worst = ref[m].max()
    lo, hi, bins = worst - 2.0005, worst + 1.9995, 4000            # 1 mdB bins, numpy's worst in the middle of one
    o = oracle(R, net, f, [(Q.SPEC_S22_MAX_DB, band[0], band[1], worst + 0.5)], 3, 2, [], hist_bins=bins, hist_spec=0, hist_lo=lo, hist_hi=hi)
    assert o["n_pass"] == 2
    want = int(np.floor((worst - lo) / (hi - lo) * bins))
    assert int(np.nonzero(o["hist"])[0][0]) == want and o["hist"][want] == 2


def analyze(Q, net, f, specs, tols, **kw):
    return Q.plan_analyze(net, f, specs, tols, **kw)


def test_plan_analyze_reversed_route(Q, W):
    """|S22|-only jobs on config 2 and the 100 -> 50 Ohm GPSDO filter take the transfer-function kernel as the |S11| job on the
    reversed cascade (4 numerator chains, no denominator: the branch denominators cancel in S11); next to an |S21| spec config 2's
    lossy branches bring a denominator back (the GPSDO filter's ideal L and C have none).  None of them runs thread-per-sample."""
    for name, net, f, tols, band, s21 in networks(Q, W)[:2]:
        s22 = (Q.SPEC_S22_MAX_DB, band[0], band[1], -15.0)
        a = analyze(Q, net, f, [s22], tols)
        assert a["selected"] and a["numerator_chains"] == 4 and a["den_form"] == "none", (name, a)
        rnet, rtols = reverse(Q, net, tols)
        b = analyze(Q, rnet, f, [(Q.SPEC_S11_MAX_DB,) + s22[1:]], rtols)
        assert (a["kn"], a["kd"], a["degree"], a["self_check_err"]) == (b["kn"], b["kd"], b["degree"], b["self_check_err"])
        c = analyze(Q, net, f, [s21, s22], tols, hist_bins=32, hist_spec=1, hist_lo=-30.0, hist_hi=0.0)
        assert c["selected"] and c["den_form"] == ("E" if name == "cfg2" else "none"), (name, c)
        assert Q.plan_ts_runs(net, f, [s22], tols) == [] and Q.plan_ts_runs(net, f, [s21, s22], tols) == []


def test_plan_analyze_refusals(Q, W, R):
    """What stays on the direct route, each with its reason."""
    w2 = W.cfg2(nf=512)
    s22 = (Q.SPEC_S22_MAX_DB, w2.f[0], 9.5e6, -15.0)
    a = analyze(Q, w2.net, w2.f, [(Q.SPEC_S11_MAX_DB,) + s22[1:], s22], w2.tols)
    assert not a["selected"] and a["reason"] == "|S11| and |S22| specs in one job"
    w5 = W.cfg5(nf=512)
    a = analyze(Q, w5.net, w5.f, [w5.specs[0], (Q.SPEC_S22_MAX_DB, 2.3e9, 2.5e9, -15.0)], w5.tols)
    assert not a["selected"] and a["reason"] == "|S22| needs a cascade of lumped branches and lines"
    net, f, _blk = nonrecip_net(Q, R)
    a = analyze(Q, net, f, [(Q.SPEC_S22_MAX_DB, 10e6, 30e6, -15.0)], [])
    assert not a["selected"] and a["reason"] == "|S22| needs a cascade of lumped branches and lines"
    a = analyze(Q, w2.net, w2.f, [s22], w2.tols, precision=32)
    assert not a["selected"] and a["reason"] == "not a reduce-only FP64 job on a lumped cascade"
    for specs, tols, nn, ff in (([(Q.SPEC_S11_MAX_DB,) + s22[1:], s22], w2.tols, w2.net, w2.f), ([s22], [], net, f)):
        assert Q.plan_ts_runs(nn, ff, specs, tols) == []


def test_chain_kernel_compiles_s22_jobs(Q, W, tmp_path, monkeypatch):
    """The compiled chain kernel takes an |S22| job in row-vector mode (den = a Rl + b, n22 = -a Rl + b) and |S11| + |S22| on the
    2x2 product: both compile for sm_100a, and the row-vector kernel is the smaller one."""
    w2 = W.cfg2(nf=256)
    s22 = (Q.SPEC_S22_MAX_DB, w2.f[0], 9.5e6, -15.0)
    dump = tmp_path / "chain.cu"
    monkeypatch.setenv("QO100NET_CHAIN_JIT_DUMP", str(dump))
    row = Q.chain_jit_analyze(w2.net, w2.f, [w2.specs[0], s22], w2.tols, hist_bins=16, hist_spec=1, hist_lo=-30.0, hist_hi=0.0)
    if not row["compiled"] and "libnvrtc" in (row["error"] or ""):
        pytest.skip("libnvrtc is not loadable here: %s" % row["error"])
    src = dump.read_text()
    assert "#define QO_JIT_ROW true" in src and "#define QO_JIT_NEED_S22 1" in src and "#define QO_JIT_HIST_KIND 5" in src
    full = Q.chain_jit_analyze(w2.net, w2.f, [(Q.SPEC_S11_MAX_DB,) + s22[1:], s22], w2.tols)
    src = dump.read_text()
    assert "#define QO_JIT_ROW false" in src and "#define QO_JIT_NEED_S22 1" in src and "#define QO_JIT_NEED_S11 1" in src
    assert row["compiled"] and full["compiled"], (row, full)
    if row["registers"] > 0 and full["registers"] > 0:
        assert row["registers"] <= full["registers"], (row, full)


def test_spec_kind_5_and_6(Q, R, W):
    """Kind 5 stays refused on the nodal path (its specs address S[row][col] themselves); kind 6 is refused everywhere."""
    w2 = W.cfg2(nf=64)
    for kind in (5, 6):
        nd = Q.Nodal(3)
        nd.add_branch(Q.NB_R, [1, 2, 0, 0], [10.0])
        nd.add_branch(Q.NB_C, [2, 0, 0, 0], [1e-9])
        nd.add_port(1, 50.0)
        nd.add_port(2, 50.0)
        with pytest.raises(Q.QoError) as e:
            nd.jit_analyze(w2.f, [(kind, 1, 0, 1e6, 1e7, -3.0)], [])
        assert e.value.status == -1                    # QO_ERR_ARG
        nd.close()
    bad = [(6, w2.f[0], w2.f[-1], -3.0)]
    a = Q.plan_analyze(w2.net, w2.f, bad, w2.tols)
    assert not a["selected"] and a["reason"] == "network does not compile"
    with pytest.raises(Q.QoError):
        Q.chain_jit_analyze(w2.net, w2.f, bad, w2.tols)
    with pytest.raises(RuntimeError):
        R.mc_run(R.make_elems(w2.net.elements), 50.0, 50.0, w2.f, bad, R.mc_cfg(1, 4, w2.tols))


# the machine code of these kernel families is what the profiles were taken on: the |S22| work must leave it alone
PARENT_SASS = {"qo_mc_ts_kernel": "435140a9b2bc0d4b", "qo_mc_tf_kernel": "e71ce5ffcc0091cd", "qo_mc_ladder_kernel": "753f7b8285c93c8d",
               "qo_fs_tf_kernel": "2e16853479cfd3f0", "qo_mc_spot_kernel": "67a9b6c129c89c83", "qo_nodal_kernel": "723d63859732b392"}


def test_fast_kernels_machine_code_unchanged():
    """tools/sass_hash.py family hashes of the polynomial, ladder, spot and nodal kernels, as build() wrote them next to the
    library, are those of the build before |S22| specs existed (nvcc of CUDA 12.9)."""
    import hashlib
    lib = os.path.join(ROOT, "qo-100-tools_b200", "lib")
    try:
        built = json.load(open(os.path.join(lib, "sass_hashes.json")))
    except OSError:
        pytest.skip("no sass_hashes.json next to the library (cuobjdump missing when build() ran)")
    if built.get("lib_sha256") != hashlib.sha256(open(os.path.join(lib, "libqo100net.so"), "rb").read()).hexdigest():
        pytest.skip("sass_hashes.json describes another build of the library")
    try:
        ver = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "--version"], capture_output=True, text=True).stdout
    except OSError:
        ver = ""
    if "release 12.9" not in ver:
        pytest.skip("the pinned hashes are of nvcc 12.9's output")
    got = {k: built["kernels"][k]["sha"] for k in PARENT_SASS}
    assert got == PARENT_SASS


# ---- GPU --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx(Q):
    c = Q.Context(device=0)
    yield c
    c.close()


def s22_limit(ctx, net, f, tols, band):
    full = ctx.mc_run(net, f, [], 11, 256, tols, mode=1)["s"]
    return limit_from(worst_db(full[3], f, band))


def run(Q, ctx, net, f, specs, tols, n, env=None, seed=21, offset=0, **hist):
    """counters of the job and the kernel that ran, under the QO100NET_* overrides in env"""
    old = {k: os.environ.get(k) for k in ("QO100NET_KERNEL", "QO100NET_CHAIN", "QO100NET_USTRIP")}
    for k in old:
        os.environ.pop(k, None)
    os.environ.update(env or {})
    try:
        p = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **hist)
        p.launch(offset, n)
        out = p.read()
        out["kernel"], out["tf"] = p.kernel_name, p.tf_info
        p.close()
    finally:
        for k, v in old.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v
    return out


def jobs(Q, W, ctx):
    """(name, net, grid, tols, [spec lists with their histogram]) of the reversed-route networks, config 3b included"""
    out = []
    nets = networks(Q, W)
    w3 = W.cfg3b(1000)
    nets.append(("cfg3b", w3.net, w3.f, w3.tols, (2.3e9, 2.5e9), w3.specs[1]))
    for name, net, f, tols, band, s21 in nets:
        lim = s22_limit(ctx, net, f, tols, band)
        s22 = (Q.SPEC_S22_MAX_DB, band[0], band[1], lim)
        h = dict(hist_bins=64, hist_lo=lim - 8.0, hist_hi=lim + 8.0)
        sets = [([s22], dict(h, hist_spec=0)), ([s21, s22], dict(h, hist_spec=1)),
                ([s21, s22], dict(hist_bins=64, hist_spec=0, hist_lo=s21[3] - 10.0, hist_hi=s21[3] + 10.0))]
        out.append((name, net, f, tols, sets))
    return out


@pytest.mark.gpu
def test_reversed_route_on_the_fast_kernels(Q, R, W, ctx):
    """|S22| alone, with an |S21| spec, histogram on either: the plan picks the kernel the |S11| job on rev(N) gets (spot,
    transfer-function, ladder under QO100NET_KERNEL=ladder), and its counters equal that job's, the oracle's and the
    interpreter's direct S22 (QO100NET_KERNEL=interp), integer for integer."""
    n = 3000
    seen = set()
    for name, net, f, tols, sets in jobs(Q, W, ctx):
        rnet, rtols = reverse(Q, net, tols)
        for specs, hist in sets:
            rspecs = [(Q.SPEC_S11_MAX_DB if s[0] == Q.SPEC_S22_MAX_DB else s[0],) + tuple(s[1:]) for s in specs]
            for env in ({"QO100NET_KERNEL": "ladder"}, {}):
                # under the ladder override an ideal or non-ladder cascade stays on the interpreter, forward and reversed alike
                a = run(Q, ctx, net, f, specs, tols, n, env, **hist)
                b = run(Q, ctx, rnet, f, rspecs, rtols, n, env, **hist)
                assert a["kernel"] == b["kernel"] and (env or a["kernel"] != "qo_mc_lumped_kernel"), (name, env, a["kernel"], b["kernel"])
                assert same(a, b), (name, env, a, b)
                seen.add(a["kernel"])
            d = run(Q, ctx, net, f, specs, tols, n, {"QO100NET_KERNEL": "interp"}, **hist)
            assert d["kernel"] == "qo_mc_lumped_kernel" and same(a, d), (name, a, d)
            assert 0 < a["fail_per_spec"][-1] < n, (name, a["fail_per_spec"])
            o = oracle(R, net, f, specs, 21, 600, tols, **hist)
            g = run(Q, ctx, net, f, specs, tols, 600, **hist)
            assert same(g, o), (name, g, o)
    assert {"qo_mc_spot_kernel", "qo_mc_tf_kernel", "qo_mc_ladder_kernel"} <= seen, seen


@pytest.mark.gpu
def test_direct_route_interpreter_and_chain_kernel(Q, R, W, ctx):
    """What no fast kernel takes -- config 5 (coupler in front), a ladder with the measured inductor behind it, the ladder behind a
    non-reciprocal block, |S11| + |S22| on config 2 -- evaluates S22 directly: interpreter and compiled chain kernel
    (QO100NET_CHAIN=jit) both equal the oracle."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "touchstone.npz"))
    cases = []
    w5 = W.cfg5(1000)
    f5 = w5.f[::16]
    cases.append(("cfg5", w5.net, f5, w5.tols, (2.3e9, 2.5e9), [w5.specs[0]]))
    R.sblock_clear()
    fd, sd, z0 = g["11SQ39N_f"], g["11SQ39N_s"], float(g["11SQ39N_z0"])
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    lad = Q.Net.butter_lpf(5, 400e6, 50.0, True)
    ind = blk.as_net(True, 50.0, 50.0).concat(lad)
    cases.append(("measured-inductor", ind, Q.grid_log(100e6, 900e6, 300), [(e + 1, p, v, m, t) for (e, p, v, m, t) in Q.lc_tolerances(lad, 0.05, 0.05)],
                  (100e6, 350e6), [(Q.SPEC_S21_MIN_DB, 100e6, 350e6, -3.0)]))
    w2 = W.cfg2(nf=512)
    both = ("cfg2-s11+s22", w2.net, w2.f, w2.tols, (w2.f[0], 9.5e6), [(Q.SPEC_S11_MAX_DB, w2.f[0], 9.5e6, -14.0)])
    for name, net, f, tols, band, extra in cases + [both]:
        if name == "measured-inductor":
            R.sblock_clear()
            R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
        lim = s22_limit(ctx, net, f, tols, band)
        specs = extra + [(Q.SPEC_S22_MAX_DB, band[0], band[1], lim)]
        hist = dict(hist_bins=64, hist_spec=len(specs) - 1, hist_lo=lim - 8.0, hist_hi=lim + 8.0)
        o = oracle(R, net, f, specs, 21, 600, tols, **hist)
        assert 0 < o["fail_per_spec"][-1] < 600, (name, o["fail_per_spec"])
        a = run(Q, ctx, net, f, specs, tols, 600, **hist)
        assert a["kernel"] in ("qo_mc_lumped_kernel", "qo_mc_chain_jit_kernel") and same(a, o), (name, a, o)
        b = run(Q, ctx, net, f, specs, tols, 600, {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "jit"}, **hist)
        if b["kernel"] == "qo_mc_chain_jit_kernel" or Q.chain_jit_analyze(net, f, specs, tols)["compiled"]:
            assert b["kernel"] == "qo_mc_chain_jit_kernel" and same(b, o), (name, b, o)
    net, f, _blk = nonrecip_net(Q, R)
    tols = [(e, 0, e, Q.TOL_REL, 0.05) for e in range(1, len(net.elements))]
    lim = s22_limit(ctx, net, f, tols, (10e6, 30e6))
    specs = [(Q.SPEC_S22_MAX_DB, 10e6, 30e6, lim)]
    hist = dict(hist_bins=64, hist_spec=0, hist_lo=lim - 8.0, hist_hi=lim + 8.0)
    o = oracle(R, net, f, specs, 21, 600, tols, **hist)
    assert 0 < o["n_pass"] < 600
    for env in ({}, {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "jit"}):
        a = run(Q, ctx, net, f, specs, tols, 600, env, **hist)
        assert same(a, o), (env, a, o)


@pytest.mark.gpu
def test_microstrip_s22(Q, R, W, ctx):
    """The PA low-pass (microstrip) with |S22| specs: board kernel at 3 points == item kernel (57 points, and at 3 points under
    QO100NET_USTRIP=item) == oracle."""
    w3 = W.cfg3(1000)
    f3 = w3.f
    full = ctx.mc_run(w3.net, f3, [], 11, 256, w3.tols, mode=1)["s"]
    p22 = 20 * np.log10(np.abs(full[3]))
    specs = [w3.specs[0], (Q.SPEC_S22_MAX_DB, 2.3e9, 2.5e9, float(np.quantile(p22[:, 0], 0.45))),
             (Q.SPEC_S22_MAX_DB, 4.7e9, 4.9e9, float(np.quantile(p22[:, 1], 0.55)))]
    hist = dict(hist_bins=64, hist_spec=1, hist_lo=specs[1][3] - 8.0, hist_hi=specs[1][3] + 8.0)
    n = 400
    o = oracle(R, w3.net, f3, specs, 21, n, w3.tols, **hist)
    assert 0 < o["fail_per_spec"][1] < n
    a = run(Q, ctx, w3.net, f3, specs, w3.tols, n, **hist)
    b = run(Q, ctx, w3.net, f3, specs, w3.tols, n, {"QO100NET_USTRIP": "item"}, **hist)
    assert a["kernel"] == "qo_mc_board_kernel" and b["kernel"] == "qo_mc_generic_kernel"
    assert same(a, o) and same(b, o), (a, b, o)
    f57 = np.concatenate([np.linspace(2.3e9, 2.5e9, 19), np.linspace(4.7e9, 4.9e9, 19), np.linspace(7.1e9, 7.3e9, 19)])
    o = oracle(R, w3.net, f57, specs, 21, 200, w3.tols, **hist)
    c = run(Q, ctx, w3.net, f57, specs, w3.tols, 200, **hist)
    assert c["kernel"] == "qo_mc_generic_kernel" and same(c, o), (c, o)


@pytest.mark.gpu
def test_reversed_route_equals_chain_kernel_at_scale(Q, W, ctx):
    """2e6 samples of config 2 with |S22| + |S21|: the reversed transfer-function run equals the compiled chain kernel's direct
    run."""
    w2 = W.cfg2()
    lim = s22_limit(ctx, w2.net, w2.f, w2.tols, (w2.f[0], 9.5e6))
    specs = [w2.specs[1], (Q.SPEC_S22_MAX_DB, w2.f[0], 9.5e6, lim)]
    hist = dict(hist_bins=256, hist_spec=1, hist_lo=lim - 8.0, hist_hi=lim + 8.0)
    n = 2000000
    a = run(Q, ctx, w2.net, w2.f, specs, w2.tols, n, **hist)
    assert a["kernel"] == "qo_mc_tf_kernel" and 0 < a["fail_per_spec"][1] < n
    if not Q.chain_jit_analyze(w2.net, w2.f[:64], specs[:1], w2.tols)["compiled"]:
        pytest.skip("libnvrtc is not loadable on this box")
    b = run(Q, ctx, w2.net, w2.f, specs, w2.tols, n, {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "jit"}, **hist)
    assert b["kernel"] == "qo_mc_chain_jit_kernel" and same(a, b), (a, b)


@pytest.mark.gpu
def test_differential_fuzz_with_s22_specs(Q, monkeypatch):
    """tools/fuzz_parity.py --s22 on a fixed seed: random lumped cascades with |S22| specs in the mix -- the selected kernel (the
    reversed route where it applies), the interpreter's direct S22 and (every 5th) the oracle agree."""
    import importlib.util
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    spec = importlib.util.spec_from_file_location("fuzz_parity", os.path.join(ROOT, "tools", "fuzz_parity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--s22", "--nets", "60", "--samples", "1500", "--seed", "23", "--big-every", "5"])
    assert out["mismatches"] == 0, out["details"]
    assert out["compared"] >= 50 and out["oracle_checked"] >= 8 and out["s22_jobs"] >= 20
