"""Per-run polynomial lengths of the thread-per-sample kernel (qo_tf.cu::tf_ts_runs, qo_ts.cuh::ts_horner): each run of the
grid walks the numerator / E (or fused-margin) lengths its own points need, never more than the plan's.  QO100NET_TS_FULL_LENGTHS
walks the plan's lengths everywhere."""
import numpy as np
import pytest


def _runs(Q, w, monkeypatch, full=False):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    if full:
        monkeypatch.setenv("QO100NET_TS_FULL_LENGTHS", "1")
    else:
        monkeypatch.delenv("QO100NET_TS_FULL_LENGTHS", raising=False)
    return Q.plan_ts_runs(w.net, w.f, w.specs, w.tols, **w.hist)


def test_cfg2_pass_band_and_transition_runs_are_shorter(Q, W, monkeypatch):
    w = W.cfg2()
    a = Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    assert (a["kn"], a["kd"]) == (9, 14)
    runs = _runs(Q, w, monkeypatch)
    f = w.f
    for r in runs:
        assert r["fused"] or (2 <= r["kn"] <= a["kn"] and 2 <= r["ke"] <= a["kd"] and r["ke"] % 2 == 0)
        assert not r["fused"] or 2 <= r["kf"] <= 2 * a["kn"]
    plain = [r for r in runs if not r["fused"] and r["any"] == r["all"]]
    band = [r for r in plain if r["all"] == 1]                      # the histogram spec's pass band
    idle = [r for r in plain if r["all"] == 0 and f[r["point"]] < 1.3e7]
    assert band and idle
    for r in band + idle:
        assert r["kn"] < a["kn"] and r["ke"] < a["kd"], r
    assert sum(r["points"] for r in runs) >= len(f)


def test_override_restores_the_plan_lengths(Q, W, monkeypatch):
    w = W.cfg2()
    a = Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    short, full = _runs(Q, w, monkeypatch), _runs(Q, w, monkeypatch, full=True)
    assert any(not r["fused"] and (r["kn"], r["ke"]) != (a["kn"], a["kd"]) for r in short)
    for r in full:
        if r["fused"]:
            assert r["kf"] == max(2 * a["kn"], a["kd"])
        else:
            assert (r["kn"], r["ke"]) == (a["kn"], a["kd"])
    # the override changes the lengths, not the runs' spec bits or the points they cover
    assert sorted({(r["any"], r["all"]) for r in short}) == sorted({(r["any"], r["all"]) for r in full})


def test_single_band_grid_keeps_the_plan_lengths(Q, monkeypatch):
    """A job whose grid is one band: its one run is the grid, and the grid's lengths are the run's"""
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_FULL_LENGTHS", raising=False)
    fc = 10e6
    net = Q.Net.cheby_lpf(11, 0.1, fc, 50.0, True)
    f = Q.grid_log(fc / 2.5, fc * 0.9, 1024)
    specs = [(Q.SPEC_S21_MIN_DB, 0.0, 1e99, -0.5)]
    tols = Q.lc_tolerances(net, 0.05, 0.02)
    a = Q.plan_analyze(net, f, specs, tols)
    runs = Q.plan_ts_runs(net, f, specs, tols)
    assert a["selected"] and len(runs) == 1
    r = runs[0]
    kd = a["kd"] if a["den_form"] == "E" else 0
    assert (r["kf"] == max(2 * a["kn"], kd)) if r["fused"] else ((r["kn"], r["ke"]) == (a["kn"], kd))


def _counters(Q, ctx, monkeypatch, w, n, off, mode):
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    monkeypatch.delenv("QO100NET_TS_FULL_LENGTHS", raising=False)
    if mode == "full":
        monkeypatch.setenv("QO100NET_TS_FULL_LENGTHS", "1")
    elif mode == "tf":
        monkeypatch.setenv("QO100NET_KERNEL", "tf")
    plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, **w.hist)
    try:
        plan.launch(off, n)
        r = plan.read()
        assert plan.kernel_name == ("qo_mc_tf_kernel" if mode == "tf" else "qo_mc_ts_kernel"), plan.kernel_name
    finally:
        plan.close()
        monkeypatch.delenv("QO100NET_KERNEL", raising=False)
        monkeypatch.delenv("QO100NET_TS_FULL_LENGTHS", raising=False)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["cfg2", "cfg5"])
def test_counters_equal_with_and_without_run_lengths(Q, W, ctx, monkeypatch, cfg):
    """per-run lengths, the plan's lengths everywhere, and the warp-per-sample kernel: the same counters and histogram"""
    w = getattr(W, cfg)()
    n = 1000000
    for off in (0, (1 << 33) + 7):
        res = {m: _counters(Q, ctx, monkeypatch, w, n, off, m) for m in ("auto", "full", "tf")}
        a = res["auto"]
        for m in ("full", "tf"):
            b = res[m]
            assert a["n_total"] == b["n_total"] == n and a["n_pass"] == b["n_pass"], (cfg, m, a["n_pass"], b["n_pass"])
            assert np.array_equal(a["fail_per_spec"], b["fail_per_spec"]), (cfg, m)
            assert np.array_equal(a["hist"], b["hist"]), (cfg, m)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["G1 cfg2", "G2 if_bpf [0, f_k]", "G3 butter7 par", "G4 cfg2, two runs"])
def test_bracket_jobs_equal_with_and_without_run_lengths(Q, ctx, monkeypatch, name):
    """the band-edge jobs of test_ts_fused at their bracketing thresholds: per-run lengths against the plan's lengths and
    against the warp-per-sample kernel"""
    import test_ts_fused as T
    geo = T._geometries()[name]
    n, off = T._launch_size()
    for k, v in T._positions(geo, 4):
        for side in (1.0, -1.0):
            specs = geo.specs(k, v + side * T.DELTA)
            got = {}
            for mode in ("auto", "full", "tf"):
                monkeypatch.delenv("QO100NET_TS_FULL_LENGTHS", raising=False)
                if mode == "full":
                    monkeypatch.setenv("QO100NET_TS_FULL_LENGTHS", "1")
                r = T._run(Q, ctx, monkeypatch, "tf" if mode == "tf" else "auto", geo.net, geo.f, specs, geo.ztols(), geo.hist, geo.fused, n, off)
                got[mode] = ([int(x) for x in r["fail_per_spec"]], int(r["n_pass"]))
            monkeypatch.delenv("QO100NET_TS_FULL_LENGTHS", raising=False)
            assert got["auto"] == got["full"] == got["tf"], (name, k, side, got)
