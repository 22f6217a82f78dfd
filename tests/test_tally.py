"""The histogram's two clamps (qo_tally.cuh::qo_hist_bin) on every Monte-Carlo kernel: with a window far narrower than the
samples' spread, worst values below it land in the first bin and values above it in the last, every sample is counted once, and
the FP64 kernels' counters equal the oracle's."""
import numpy as np
import pytest

from conftest import to_ref

pytestmark = pytest.mark.gpu

HALF = 1e-3                  # dB on either side of the nominal worst value: every tolerance draw moves it further than that


def _window(spec, value_db, bins=8):
    return dict(hist_bins=bins, hist_spec=spec, hist_lo=value_db - HALF, hist_hi=value_db + HALF)


def _assert_both_clamps(got, n):
    h = got["hist"]
    assert got["n_total"] == n and int(h.sum()) == n
    assert h[0] > 0 and h[-1] > 0, h


def _assert_counts_equal(ref, got):
    assert got["n_total"] == ref["n_total"] and got["n_pass"] == ref["n_pass"]
    assert np.array_equal(got["fail_per_spec"], ref["fail_per_spec"]) and np.array_equal(got["hist"], ref["hist"])


def _nominal_worst_db(Q, ctx, net, f, spec):
    """the histogram variable of the nominal network: the worst |S21| dB of the spec's band"""
    kind, f_lo, f_hi, _limit = spec
    db = 20 * np.log10(np.abs(ctx.sweep(net, f)[1]))[(f >= f_lo) & (f <= f_hi)]
    return float(db.min() if kind == Q.SPEC_S21_MIN_DB else db.max())


# name: (workload, QO100NET_* overrides, precision, kernel that must run, compared with the oracle)
CASCADE = {
    "spot": ("cfg3b", {}, 64, "qo_mc_spot_kernel", True),
    "tf": ("cfg3b", {"QO100NET_KERNEL": "tf"}, 64, "qo_mc_tf_kernel", True),
    "ts": ("cfg2", {}, 64, "qo_mc_ts_kernel", True),
    "ladder": ("cfg3b", {"QO100NET_KERNEL": "ladder"}, 64, "qo_mc_ladder_kernel", True),
    "ladder_fp32": ("cfg3b", {"QO100NET_KERNEL": "ladder"}, 32, "qo_mc_ladder_kernel", False),
    "interp": ("cfg3b", {"QO100NET_KERNEL": "interp"}, 64, "qo_mc_lumped_kernel", True),
    "chain_jit": ("cfg3b", {"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "jit"}, 64, "qo_mc_chain_jit_kernel", True),
    "board": ("cfg3", {}, 64, "qo_mc_board_kernel", True),
    "generic": ("cfg3", {"QO100NET_USTRIP": "item"}, 64, "qo_mc_generic_kernel", True),
}


@pytest.mark.parametrize("case", list(CASCADE))
def test_cascade_kernel_histogram_clamps(Q, R, W, ctx, monkeypatch, case):
    import torch
    wname, env, precision, kernel, vs_oracle = CASCADE[case]
    for k in ("QO100NET_KERNEL", "QO100NET_CHAIN", "QO100NET_USTRIP"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    if wname == "cfg2":
        w = W.cfg2(nf=101)
        # the thread-per-sample kernel takes launches of two waves and more; a multiple of 32 runs on it alone
        n = 2 * torch.cuda.get_device_properties(0).multi_processor_count * 4 * 128
    else:
        w = getattr(W, wname)()
        n = 4000
    if case == "chain_jit":
        a = Q.chain_jit_analyze(w.net, w.f, w.specs, w.tols)
        if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
            pytest.skip("libnvrtc is not loadable here: no compiled chain kernel (%s)" % a["error"])
    hs = w.hist["hist_spec"]
    hist = _window(hs, _nominal_worst_db(Q, ctx, w.net, w.f, w.specs[hs]))
    off = 12345
    plan = Q.Plan(ctx, w.net, w.f, w.specs, seed=w.seed, tols=w.tols, precision=precision, **hist)
    plan.launch(off, n)
    got = plan.read()
    assert plan.kernel_name == kernel, plan.kernel_name
    plan.close()
    _assert_both_clamps(got, n)
    if vs_oracle:
        rs, rl = w.net.terminations
        ref = R.mc_run(to_ref(R, w.net), rs, rl, w.f, w.specs, R.mc_cfg(w.seed, n, w.tols, sample_offset=off, **hist), nthreads=8)
        _assert_counts_equal(ref, got)


@pytest.mark.parametrize("mode", ["dense", "static", "jit"])
def test_nodal_kernel_histogram_clamps(Q, R, W, ctx, golden_s2p, monkeypatch, mode):
    fd, sd = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"]
    nd, br, tols = W.pa_bias_nodal(Q, fd, sd)
    _br, nn, ports = W.pa_bias_netlist()
    f = Q.grid_lin(1e8, 3e9, 200)
    if mode == "jit" and not nd.jit_analyze(f)["compiled"]:
        nd.close()
        pytest.skip("no NVRTC here: no compiled nodal kernel")
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    nom = ctx.nodal_sweep(nd, f)
    band = (f >= 2.3e9) & (f <= 2.5e9)
    s21 = 20 * np.log10(np.abs(nom[band, 1, 0]))
    specs = [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, -3.0), (Q.SPEC_S21_MAX_DB, 2, 0, 2.3e9, 2.5e9, -25.0)]
    hist = _window(0, float(s21.min()))
    n, off = 2000, 777
    monkeypatch.setenv("QO100NET_NODAL", mode)
    got = ctx.nodal_mc_run(nd, f, specs, 5, n, tols, sample_offset=off, **hist)
    assert ctx.nodal_last_kernel() == {"dense": "qo_nodal_kernel<dense>", "static": "qo_nodal_kernel<static,local>",
                                       "jit": "qo_nodal_jit_kernel"}[mode]
    nd.close()
    _assert_both_clamps(got, n)
    R.sblock_clear()
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], 50.0)
    ref = R.nodal_mc_run(br, nn, ports, f, specs, R.mc_cfg(5, n, tols, sample_offset=off, **hist), nthreads=8)
    R.sblock_clear()
    _assert_counts_equal(ref, got)
