"""The histogram screen of the thread-per-sample kernel (qo_ts.cuh; its gate, qo_tf.cu::tf_hist_screen): where the histogram spec
looks alone, a group of points is walked exactly only when some lane's screen polynomial S = +-(N2 - m E) is not certainly
negative.  The counters and the histogram must stay integer for integer what the full walk (QO100NET_TS_HIST_SCREEN=0) and the
warp-per-sample kernel give."""
import numpy as np
import pytest


def _screen(Q, w, specs=None, tols=None, hist=None):
    return Q.plan_ts_screen(w.net, w.f, w.specs if specs is None else specs, w.tols if tols is None else tols,
                            **(w.hist if hist is None else hist))


def test_cfg2_screens_its_pass_band_behind_seed_runs(Q, W, monkeypatch):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SCREEN", raising=False)
    w = W.cfg2()
    s = _screen(Q, w)
    assert s["screened"] and s["reason"] == "ok", s
    assert s["screened_runs"] >= 1 and 1 <= s["seeds"] <= 10 and s["eps"] == 1e-6
    assert 0.0 < s["m_lo"] < s["m_hi"] and 0.0 < s["bound"] <= 1.0
    runs = Q.plan_ts_runs(w.net, w.f, w.specs, w.tols, **w.hist)
    seeds, rest = runs[:s["seeds"]], runs[s["seeds"]:]
    band = [r for r in rest if not r["fused"] and r["any"] == r["all"] == 1]
    for r in seeds:                                  # one group of the pass band each, at the lengths of the run that holds it
        assert r["points"] == 4 and r["any"] == r["all"] == 1
        assert any(b["point"] <= r["point"] < b["point"] + b["points"] and (b["kn"], b["ke"]) == (r["kn"], r["ke"]) for b in band)
    assert sum(r["points"] for r in rest) >= len(w.f)
    # the override: same run table without the seeds
    monkeypatch.setenv("QO100NET_TS_HIST_SCREEN", "0")
    off = _screen(Q, w)
    assert not off["screened"] and "QO100NET_TS_HIST_SCREEN" in off["reason"] and off["seeds"] == 0
    assert Q.plan_ts_runs(w.net, w.f, w.specs, w.tols, **w.hist) == rest


def test_declines_where_the_histogram_spec_shares_its_band(Q, W, monkeypatch):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SCREEN", raising=False)
    w = W.cfg2()
    specs = list(w.specs) + [(Q.SPEC_S21_MAX_DB, 0.0, 0.95e7, 1.0)]            # a second spec over the whole pass band
    s = _screen(Q, w, specs=specs)
    assert not s["screened"] and "shares every run" in s["reason"], s


def test_declines_behind_a_coupled_line_block(Q, W, monkeypatch):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SCREEN", raising=False)
    w = W.cfg5()
    s = _screen(Q, w)
    assert not s["screened"] and "coupled-line" in s["reason"], s


def test_declines_without_a_histogram(Q, W, monkeypatch):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    w = W.cfg2()
    s = _screen(Q, w, hist={})
    assert not s["screened"] and s["reason"] == "no histogram"


# ---- GPU: integer-for-integer counters ----------------------------------------------------------------------------------
def _counters(Q, ctx, monkeypatch, net, f, specs, tols, hist, seed, n, off, mode, env=None):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SCREEN", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SEEDS", raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    if mode == "off":
        monkeypatch.setenv("QO100NET_TS_HIST_SCREEN", "0")
    elif mode == "tf":
        monkeypatch.setenv("QO100NET_KERNEL", "tf")
    plan = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **hist)
    try:
        info = plan.tf_info
        plan.launch(off, n)
        r = plan.read()
        assert plan.kernel_name == ("qo_mc_tf_kernel" if mode == "tf" else "qo_mc_ts_kernel"), (mode, plan.kernel_name)
        ran = plan.tf_info["hist_screen"]["screen_kernel_ran"]
        assert ran == (mode == "auto" and info["hist_screen"]["screened"]), (mode, ran, info["hist_screen"])
    finally:
        plan.close()
        for k in ("QO100NET_KERNEL", "QO100NET_TS_HIST_SCREEN", "QO100NET_TS_HIST_SEEDS"):
            monkeypatch.delenv(k, raising=False)
    assert r["n_total"] == n
    return r, info["hist_screen"]


def _same(Q, ctx, monkeypatch, net, f, specs, tols, hist, seed, n, off, want_screen=True, env=None):
    got = {m: _counters(Q, ctx, monkeypatch, net, f, specs, tols, hist, seed, n, off, m, env) for m in ("auto", "off", "tf")}
    scr = got["auto"][1]
    assert scr["reason"] and (want_screen is None or scr["screened"] == want_screen), scr
    assert not got["off"][1]["screened"]
    a = got["auto"][0]
    for m in ("off", "tf"):
        b = got[m][0]
        assert a["n_pass"] == b["n_pass"], (m, a["n_pass"], b["n_pass"])
        assert np.array_equal(a["fail_per_spec"], b["fail_per_spec"]), (m, a["fail_per_spec"], b["fail_per_spec"])
        assert np.array_equal(a["hist"], b["hist"]), m
    return a


@pytest.mark.gpu
def test_cfg2_two_million_samples(Q, W, ctx, monkeypatch):
    w = W.cfg2()
    a = _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, w.tols, w.hist, w.seed, 2000000, 0)
    assert 0 < a["n_pass"] < 2000000


@pytest.mark.gpu
def test_narrow_histogram_window(Q, W, ctx, monkeypatch):
    """a window of 0.05 dB over 256 bins around the samples' worst pass-band |S21|: one ulp of the tracker moves samples
    between bins"""
    w = W.cfg2()
    import test_ts_fused as T
    n, off = T._launch_size()
    wide = _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, w.tols, w.hist, w.seed, n, off)
    edges = np.linspace(w.hist["hist_lo"], w.hist["hist_hi"], w.hist["hist_bins"] + 1)
    mid = edges[int(np.argmax(wide["hist"]))]
    hist = dict(hist_bins=256, hist_spec=0, hist_lo=mid - 0.025, hist_hi=mid + 0.025)
    a = _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, w.tols, hist, w.seed, n, off)
    assert np.count_nonzero(a["hist"]) > 32


@pytest.mark.gpu
def test_histogram_on_a_max_spec(Q, W, ctx, monkeypatch):
    """the histogram on config 2's MAX-dB stop band: the tracker keeps a minimum (the stop band's cancellation puts its bound
    far above eps/8 at these lengths, so the plan may decline: either way the counters stay)"""
    w = W.cfg2()
    import test_ts_fused as T
    n, off = T._launch_size()
    hist = dict(hist_bins=256, hist_spec=1, hist_lo=-120.0, hist_hi=-40.0)
    _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, w.tols, hist, w.seed, n, off, want_screen=None)


@pytest.mark.gpu
def test_wide_tolerances(Q, W, ctx, monkeypatch):
    """+-20 % on every L and C: the seeds are poor guesses of each sample's worst point (the plan may decline: either way the
    counters stay)"""
    w = W.cfg2()
    import test_ts_fused as T
    n, off = T._launch_size()
    tols = Q.lc_tolerances(w.net, 0.20, 0.20)
    _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, tols, w.hist, w.seed, n, off, want_screen=None)


def _g3():
    """'G3 butter7 par' of test_ts_fused with its own tolerances: the histogram on a MAX-dB stop band (the tracker keeps a
    minimum), screened"""
    import test_ts_fused as T
    geo = T._geometries()["G3 butter7 par"]
    k, v = T._positions(geo, 1)[0]
    return geo, geo.specs(k, v)


def test_low_seed_override_and_the_tracker_minimum_job(Q, monkeypatch):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SCREEN", raising=False)
    monkeypatch.delenv("QO100NET_TS_HIST_SEEDS", raising=False)
    geo, specs = _g3()
    s = Q.plan_ts_screen(geo.net, geo.f, specs, geo.tols, **geo.hist)
    assert s["screened"] and s["seeds"] >= 1 and not s["screen_kernel_ran"], s
    assert Q.plan_ts_runs(geo.net, geo.f, specs, geo.tols, **geo.hist)[0]["point"] > 0      # its best seed is not the band's low end
    monkeypatch.setenv("QO100NET_TS_HIST_SEEDS", "low")
    s = Q.plan_ts_screen(geo.net, geo.f, specs, geo.tols, **geo.hist)
    assert s["screened"] and s["seeds"] == 1, s
    first = Q.plan_ts_runs(geo.net, geo.f, specs, geo.tols, **geo.hist)[0]
    assert first["points"] == 4 and first["any"] == first["all"] == 1 << geo.hist["hist_spec"], first


def test_low_seed_makes_the_exact_path_move_the_screen_on_cfg2(Q, W, R, monkeypatch):
    """Replayed on config 2's own sample stream (tools/hist_screen_projection.py): with only the band's lowest group as a seed
    the tracker rises inside the band, so batches go exactly on the sign test (not only the runs' partial last batches) and the
    exact path moves the screen polynomial -- what the GPU tests with QO100NET_TS_HIST_SEEDS=low run through"""
    import sys
    import os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import hist_screen_projection as P
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.setenv("QO100NET_TS_HIST_SEEDS", "low")
    low = P.project(256)
    assert low["seeds"] == [0] and low["sign_exact_batches"] > 0 and low["updates"] > 0, low
    monkeypatch.delenv("QO100NET_TS_HIST_SEEDS")
    default = P.project(256)
    assert default["updates"] == 0 and default["sign_exact_batches"] == 0, default


@pytest.mark.gpu
def test_cfg2_eight_percent_tolerances(Q, W, ctx, monkeypatch):
    """+-8 % on every L and C: screened (the +-20 % job above is not)"""
    w = W.cfg2()
    import test_ts_fused as T
    n, off = T._launch_size()
    _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, Q.lc_tolerances(w.net, 0.08, 0.08), w.hist, w.seed, n, off)


@pytest.mark.gpu
def test_tracker_minimum_with_tolerances(Q, ctx, monkeypatch):
    geo, specs = _g3()
    import test_ts_fused as T
    n, off = T._launch_size()
    _same(Q, ctx, monkeypatch, geo.net, geo.f, specs, geo.tols, geo.hist, 3, n, off)


@pytest.mark.gpu
@pytest.mark.parametrize("job", ["cfg2", "cfg2 +-8 %", "G3 butter7 par (tracker minimum)"])
def test_low_seed_tracker_rises_inside_the_band(Q, W, ctx, monkeypatch, job):
    """QO100NET_TS_HIST_SEEDS=low: the band's lowest group is the only seed, so the tracker rises after it, batches go exactly
    on the sign test and the exact path moves the screen polynomial in place; the counters stay those of the full walk and of
    the warp-per-sample kernel"""
    import test_ts_fused as T
    n, off = T._launch_size()
    env = {"QO100NET_TS_HIST_SEEDS": "low"}
    if job.startswith("G3"):
        geo, specs = _g3()
        _same(Q, ctx, monkeypatch, geo.net, geo.f, specs, geo.tols, geo.hist, 3, n, off, env=env)
    else:
        w = W.cfg2()
        tols = w.tols if job == "cfg2" else Q.lc_tolerances(w.net, 0.08, 0.08)
        _same(Q, ctx, monkeypatch, w.net, w.f, w.specs, tols, w.hist, w.seed, n, off, env=env)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G1 cfg2", "G2 if_bpf [0, f_k]", "G3 butter7 par", "G4 cfg2, two runs"])
def test_bracket_jobs(Q, ctx, monkeypatch, name):
    """the band-edge jobs of test_ts_fused at their bracketing thresholds, with the histogram on their other spec"""
    import test_ts_fused as T
    geo = T._geometries()[name]
    n, off = T._launch_size()
    for k, v in T._positions(geo, 4):
        for side in (1.0, -1.0):
            specs = geo.specs(k, v + side * T.DELTA)
            got = {m: _counters(Q, ctx, monkeypatch, geo.net, geo.f, specs, geo.ztols(), geo.hist, 3, n, off, m)[0] for m in ("auto", "off", "tf")}
            key = {m: ([int(x) for x in r["fail_per_spec"]], int(r["n_pass"]), [int(x) for x in r["hist"]]) for m, r in got.items()}
            assert key["auto"] == key["off"] == key["tf"], (name, k, side)
