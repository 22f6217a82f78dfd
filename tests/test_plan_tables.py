"""Each kernel family's device tables, uploaded once per plan and re-sent by qo_mc_run when it reuses the plan.

For one job per table set: two qo_mc_run calls on the same sample range (the second reuses the cached plan and copies its tables
to the device again) give identical counters, or FULL_S planes, and both equal a fresh Plan.launch / read over that range.  Two
plans of one job report the same Plan.h2d_bytes."""
import numpy as np
import pytest

OFF = 2 ** 33 + 7


def _ts_samples():
    """enough samples for the thread-per-sample kernel (>= two waves), plus a remainder for the warp-per-sample one"""
    import torch
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 4 * 128 + 32 * 37 + 19


def _block_job(Q, golden_s2p):
    """the 20 W driver measurement (non-reciprocal) inside a lumped cascade: not a front block, so the lumped kernel takes it"""
    fd, sd, z0 = golden_s2p["pa_20W_f"], golden_s2p["pa_20W_s"], float(golden_s2p["pa_20W_z0"])
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    net = Q.Net.from_elements([(Q.SER_L, [1e-9, 0.1, 0.0])], 50, 50).concat(blk.as_net(True)).concat(
        Q.Net.from_elements([(Q.SHUNT_C, [0.5e-12, 0.2, 0.0])], 50, 50))
    return net, [(0, 0, 0, Q.TOL_REL, 0.1), (2, 0, 1, Q.TOL_REL, 0.1)]


# name -> (environment, kernel the plan names before a launch, kernel that ran)
JOBS = {
    "spot_cfg3b": ({}, "qo_mc_spot_kernel", "qo_mc_spot_kernel"),
    "tf_ts_cfg2": ({}, "qo_mc_tf_kernel", "qo_mc_ts_kernel"),
    "tf_coupler_cfg5": ({}, "qo_mc_tf_kernel", "qo_mc_ts_kernel"),
    "ladder_cfg2": ({"QO100NET_KERNEL": "ladder"}, "qo_mc_ladder_kernel", "qo_mc_ladder_kernel"),
    "ladder_coupler_cfg5": ({"QO100NET_KERNEL": "ladder"}, "qo_mc_ladder_kernel", "qo_mc_ladder_kernel"),
    "ladder_fp32_cfg2": ({}, "qo_mc_ladder_kernel", "qo_mc_ladder_kernel"),
    "lumped_fp32_cfg2": ({"QO100NET_KERNEL": "interp"}, "qo_mc_lumped_kernel", "qo_mc_lumped_kernel"),
    "lumped_measured_block": ({}, "qo_mc_lumped_kernel", "qo_mc_lumped_kernel"),
    "chain_jit_cfg2": ({"QO100NET_KERNEL": "interp", "QO100NET_CHAIN": "jit"}, "qo_mc_lumped_kernel", "qo_mc_chain_jit_kernel"),
    "board_cfg3": ({}, "qo_mc_board_kernel", "qo_mc_board_kernel"),
    "generic_cfg3": ({"QO100NET_USTRIP": "item"}, "qo_mc_generic_kernel", "qo_mc_generic_kernel"),
    "full_s_below_tf_min": ({}, "qo_mc_lumped_kernel", "qo_mc_lumped_kernel"),
    "full_s_tf": ({}, "qo_mc_lumped_kernel", "qo_fs_tf_kernel"),
}


def _job(Q, W, ctx, golden_s2p, name):
    """-> (net, f, specs, seed, tols, keyword arguments of mc_run / Plan, n_samples)"""
    if name == "lumped_measured_block":
        net, tols = _block_job(Q, golden_s2p)
        f = Q.grid_lin(2e7, 9e9, 500)
        band = (f >= 1e9) & (f <= 4e9)
        s21 = ctx.mc_run(net, f, [], 5, 2000, tols, mode=Q.MODE_FULL_S)["s"][1]
        limit = float(np.median(20 * np.log10(np.abs(s21[:, band])).min(axis=1)))      # about half the samples fail
        return net, f, [(Q.SPEC_S21_MIN_DB, 1e9, 4e9, limit)], 5, tols, {}, 20000
    if name.startswith("full_s"):
        w = W.cfg2(0, 513)
        return w.net, w.f, [], 7, w.tols, dict(mode=Q.MODE_FULL_S), 512 if name == "full_s_below_tf_min" else 1100
    w = {"cfg2": W.cfg2, "cfg3": W.cfg3, "cfg3b": W.cfg3b, "cfg5": W.cfg5}[name.rsplit("_", 1)[1]]()
    kw = dict(w.hist, precision=32) if "fp32" in name else dict(w.hist)
    return w.net, w.f, w.specs, w.seed, w.tols, kw, _ts_samples()


def _fresh(Q, ctx, net, f, specs, seed, tols, kw, n):
    """(result, kernel that ran) of a new plan launched over the range"""
    import torch
    plan = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **kw)
    buf = None
    if kw.get("mode") == Q.MODE_FULL_S:
        buf = torch.empty((4, n, len(f), 2), dtype=torch.float64, device="cuda")
    plan.launch(OFF, n, None, buf.data_ptr() if buf is not None else None)
    res = plan.read()
    if buf is not None:
        torch.cuda.synchronize()
        res["s"] = buf.cpu().numpy().view(np.complex128)[..., 0]
    name = plan.kernel_name
    plan.close()
    return res, name


def _assert_same(a, b):
    if "s" in a:
        assert np.array_equal(a["s"], b["s"])
        return
    assert (a["n_pass"], a["n_total"]) == (b["n_pass"], b["n_total"])
    assert np.array_equal(a["fail_per_spec"], b["fail_per_spec"]) and np.array_equal(a["hist"], b["hist"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(JOBS))
def test_tables_resent_on_plan_reuse_match_a_fresh_plan(Q, W, ctx, golden_s2p, monkeypatch, name):
    env, planned, ran = JOBS[name]
    for k in ("QO100NET_KERNEL", "QO100NET_CHAIN", "QO100NET_USTRIP", "QO100NET_NO_PLAN_CACHE"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    net, f, specs, seed, tols, kw, n = _job(Q, W, ctx, golden_s2p, name)
    if name == "chain_jit_cfg2":
        a = Q.chain_jit_analyze(net, f, specs, tols, **kw)
        if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
            pytest.skip("libnvrtc is not loadable on this box: the compiled chain kernel is not available (%s)" % a["error"])
    first = ctx.mc_run(net, f, specs, seed, n, tols, sample_offset=OFF, **kw)
    again = ctx.mc_run(net, f, specs, seed, n, tols, sample_offset=OFF, **kw)     # same job: the cached plan, tables re-sent
    _assert_same(first, again)
    fresh, kernel = _fresh(Q, ctx, net, f, specs, seed, tols, kw, n)
    assert kernel == ran
    _assert_same(first, fresh)
    if "s" in first:
        assert np.all(np.isfinite(first["s"])) and np.max(np.abs(first["s"][1])) > 0
    else:
        assert first["n_total"] == n and 0 < first["n_pass"] < n
    p1 = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **kw)
    p2 = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **kw)
    assert p1.kernel_name == planned
    assert p1.h2d_bytes == p2.h2d_bytes > 0
    p1.close()
    p2.close()
