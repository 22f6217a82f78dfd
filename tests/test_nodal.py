"""Row N4: N-port nodal analysis, pinned by the reference's 5-port bias-network dataset
util/pa-bias-simulation/pa-bias-simulation.dat (schematic pa-bias-simulation.sch:19-72: R, C, GND, Pac ports,
ideal VCVS buffers :40,59 and the measured inductor 11SQ39N.S2P pulled in with SPfile "polar" "linear" :39).
CPU part: the oracle against the dataset, the product's netlister against a hand-derived netlist.
GPU part (marked): the CUDA nodal kernel against the oracle and against the dataset, through the C-ABI."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, REFERENCE, ROOT

NB_R, NB_L, NB_C, NB_VCVS, NB_SBLOCK = 1, 2, 3, 4, 5


def hand_netlist():
    """pa-bias-simulation.sch read by hand (qo100net.workloads.pa_bias_netlist holds the list, with the component line numbers)."""
    from qo100net import workloads
    return workloads.pa_bias_netlist()


DAT_ENTRIES = {"S1_1": (0, 0), "S1_2": (0, 1), "S1_3": (0, 2), "S2_1": (1, 0), "S2_2": (1, 1), "S2_3": (1, 2),
               "S3_1": (2, 0), "S3_2": (2, 1), "S3_3": (2, 2), "S5_5": (4, 4), "S5_4": (4, 3), "S4_5": (3, 4), "S4_4": (3, 3)}


@pytest.fixture(scope="module")
def pa_bias():
    return np.load(os.path.join(GOLDEN, "pa_bias_dat.npz"))


def register_inductor(R, golden_s2p, idx=0):
    fd, sd = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"]
    R.sblock_clear()
    R.sblock_register(idx, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], 50.0)


def check_vs_dat(S, d, tol_rel=1e-9, tol_abs=2e-10):
    """Every S entry the dataset holds: |dS| <= tol_rel*|S| + tol_abs (the isolation entries sit at -150 dB)."""
    worst = 0.0
    for key, (k, j) in DAT_ENTRIES.items():
        err = np.abs(S[:, k, j] - d[key])
        worst = max(worst, float(np.max(err / (tol_rel * np.abs(d[key]) + tol_abs))))
    assert worst <= 1.0, worst
    # the three Eqn traces of pa-bias-simulation.sch:72
    for key, (k, j) in (("Gain_S21db", (1, 0)), ("Gain_S31db", (2, 0)), ("Gain_S54db", (4, 3))):
        assert np.max(np.abs(20 * np.log10(np.abs(S[:, k, j])) - d[key])) < 1e-6
    # entries Qucs did not print couple the two unconnected sub-circuits: exactly zero
    assert np.all(S[:, 0:3, 3:5] == 0) and np.all(S[:, 3:5, 0:3] == 0)


def test_oracle_reproduces_pa_bias_dataset(R, pa_bias, golden_s2p):
    """The oracle (MNA + SPfile polar interpolation with linear extrapolation) against all 13 S entries x 5000
    points of the reference dataset; this also pins the SPfile restatement of row N3 (holding the end values
    instead of extrapolating fails this test by orders of magnitude above 3.3 GHz)."""
    br, nn, ports = hand_netlist()
    register_inductor(R, golden_s2p)
    f = pa_bias["frequency"]
    assert len(f) == 5000 and f[0] == 1e6 and f[-1] == 1e10
    S = R.nodal_sweep(br, nn, ports, f)
    check_vs_dat(S, pa_bias)
    # and the sensitivity claim
    fd, sd = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"]
    R.sblock_register(0, np.concatenate([[0.5e6], fd, [2e10]]), *[np.concatenate([sd[:1, c], sd[:, c], sd[-1:, c]]) for c in range(4)], 50.0)
    held = R.nodal_sweep(br, nn, ports, f)
    assert np.max(np.abs(held[:, 1, 0] - pa_bias["S2_1"]) / np.abs(pa_bias["S2_1"])) > 1e-3
    R.sblock_clear()


def test_oracle_nodal_equals_cascade_on_a_ladder(R):
    """Cross-check of the two oracle evaluators: a 2-port ladder through the nodal solver == through the ABCD chain."""
    lad = R.ladder_lpf(R.cheby_g(7, 0.1), 10e6, 50.0, True, (60, 30, 0.1, 50))
    el = R.elems_to_list(lad)
    f = R.grid_log(2e6, 80e6, 301)
    s11, s21, s12, s22 = R.sweep(lad, 50.0, 75.0, f)
    br, node = [], 1
    for kind, p in el:
        if kind == 3:       # series L: node -> node+1
            br.append((NB_L, [node, node + 1], p[:3])); node += 1
        else:               # shunt C
            br.append((NB_C, [node, 0], p[:3]))
    S = R.nodal_sweep(br, node, [(1, 50.0), (node, 75.0)], f)
    assert np.max(np.abs(S[:, 1, 0] - s21) / np.abs(s21)) < 1e-10 and np.max(np.abs(S[:, 0, 0] - s11)) < 1e-12
    assert np.max(np.abs(S[:, 1, 1] - s22)) < 1e-12 and np.max(np.abs(S[:, 0, 1] - s12) / np.abs(s12)) < 1e-10


def canon(branches, ports):
    """Node-numbering-independent signature of a netlist: relabel nodes by their sorted incident (kind, value) sets."""
    import collections
    inc = collections.defaultdict(list)
    for kind, nodes, p in branches:
        nn = {NB_VCVS: 4, NB_SBLOCK: 3}.get(kind, 2)
        for pos in range(nn):
            if nodes[pos]:
                inc[nodes[pos]].append((kind, pos if kind in (NB_VCVS, NB_SBLOCK) else 0, round(p[0], 18)))
    for i, (n, z) in enumerate(ports):
        inc[n].append((99, i, z))
    sig = {n: tuple(sorted(v)) for n, v in inc.items()}
    out = []
    for kind, nodes, p in branches:
        nn = {NB_VCVS: 4, NB_SBLOCK: 3}.get(kind, 2)
        ends = [sig.get(nodes[pos], ()) for pos in range(nn)]
        if nn == 2:
            ends = sorted(ends)
        out.append((kind, tuple(ends), tuple(round(x, 18) for x in p[:3])))
    return sorted(out)


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="the upstream qo-100-tools files are not in this repository: set QO100_REFERENCE to a checkout")
def test_netlister_reads_pa_bias_schematic(Q):
    """qo_nodal_load_qucs_sch on the reference schematic == the hand-derived netlist (up to node numbering):
    28 branches, 21 nodes, 5 ports in Pac-number order, the SPfile resolved next to the schematic."""
    nd = Q.Nodal.from_qucs_sch(os.path.join(REFERENCE, "util/pa-bias-simulation/pa-bias-simulation.sch"))
    br, nn, ports = hand_netlist()
    got = nd.branches
    assert nd.n_nodes == nn and len(got) == len(br) and [z for _, z in nd.ports] == [50.0] * 5
    hand = [(k, list(n) + [0] * (4 - len(n)), list(p) + [0.0] * (4 - len(p))) for k, n, p in br]
    assert canon(got, nd.ports) == canon(hand, ports)
    # the preamp schematic (its dataset is missing upstream, .MISSING_LARGE_BLOBS) loads too
    pre = Q.Nodal.from_qucs_sch(os.path.join(REFERENCE, "util/preamp-bias-simulation/preamp-bias-simulation.sch"))
    assert len(pre.ports) >= 2 and any(k == NB_SBLOCK for k, _, _ in pre.branches)


def test_nodal_container_errors(Q):
    nd = Q.Nodal(3)
    nd.add_branch(Q.NB_R, [1, 2], [10.0])
    assert nd.add_port(1) == 1 and nd.add_port(3, 75.0) == 2
    for bad in ((Q.NB_R, [1, 1], [10.0]), (Q.NB_R, [1, 9], [10.0]), (Q.NB_R, [1, 2], [-1.0]), (Q.NB_SBLOCK, [1, 2, 0], [0, 1, 50.0]), (77, [1, 2], [1.0])):
        with pytest.raises(Q.QoError):
            nd.add_branch(*bad)
    with pytest.raises(Q.QoError):
        nd.add_port(0)
    with pytest.raises(Q.QoError):
        Q.Nodal(0)
    with pytest.raises(Q.QoError):
        Q.Nodal.from_qucs_sch("/nonexistent.sch")


def build_nodal(Q, golden_s2p):
    """The hand netlist as a product object (the GPU box has no reference tree to load the schematic from)."""
    br, nn, ports = hand_netlist()
    nd = Q.Nodal(nn)
    fd, sd = golden_s2p["11SQ39N_f"], golden_s2p["11SQ39N_s"]
    idx = nd.add_sblock(Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], 50.0))
    for kind, nodes, p in br:
        if kind == NB_SBLOCK:
            p = [idx, p[1], p[2]]
        nd.add_branch(kind, nodes, p)
    for node, z0 in ports:
        nd.add_port(node, z0)
    return nd, br, nn, ports


def test_static_plan_analysis_host_only(Q, pa_bias, golden_s2p):
    """qo_nodal_analyze (no GPU): the reference's bias network takes the static factorisation plan on its own 5000-point grid,
    with and without tolerances, and its multipliers stay far below the device guard (1e5)."""
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    f = pa_bias["frequency"]
    a = nd.analyze(f)
    assert a["static"] and a["unknowns"] == 23 and 60 < a["nnz"] <= 160 and a["program_words"] > 100
    assert a["max_multiplier"] < 3e6            # 3.2e5 at 1 MHz: the 100 uF / 1.2 pF stiffness, harmless (dataset parity holds)
    tols = [(b, 0, v, Q.TOL_REL, 0.05) for v, b in enumerate(i for i, (k, _n, _p) in enumerate(br) if k in (NB_R, NB_C))]
    at = nd.analyze(f, tols)
    assert at["static"] and at["max_multiplier"] < 3e6


def test_static_plan_rejects_an_order_that_only_suits_part_of_the_band(Q):
    """A resonant divider whose dominant entry changes along the grid: node 2 hangs on a series-LC trap to ground that is a
    short at its resonance (5.03 MHz) and nearly open elsewhere, next to a tiny conductance.  Whatever fixed order the mid-grid
    point suggests, the analysis must either prove it at every probe (multiplier bounded) or send the job to the pivoted kernel;
    it may never accept a plan whose probes saw a multiplier above the device guard (3e6)."""
    nd = Q.Nodal(3)
    nd.add_branch(Q.NB_R, [1, 2], [1e-3])
    nd.add_branch(Q.NB_L, [2, 3], [1e-6, 0.0, 0.0])
    nd.add_branch(Q.NB_C, [3, 0], [1e-9, 1e-6, 0.0])
    nd.add_branch(Q.NB_R, [2, 0], [1e9])
    nd.add_branch(Q.NB_R, [1, 3], [1e7])
    nd.add_port(1, 50.0)
    f = Q.grid_log(1e5, 1e9, 801)
    a = nd.analyze(f, [(1, 0, 0, Q.TOL_REL, 0.2), (2, 0, 1, Q.TOL_REL, 0.2)])
    assert (not a["static"]) or a["max_multiplier"] <= 3.2e6
    nd.close()


@pytest.mark.gpu
def test_gpu_nodal_guard_falls_back_to_the_pivoted_kernel(Q, R, ctx, monkeypatch):
    """The device-side multiplier guard: a job whose static plan passes the plan-time probes but meets a huge multiplier at an
    unprobed point is re-run with per-point pivoting, and the result equals the oracle's either way."""
    nd = Q.Nodal(3)
    br = [(Q.NB_R, [1, 2], [1e-3]), (Q.NB_L, [2, 3], [1e-6, 0.0, 0.0]), (Q.NB_C, [3, 0], [1e-9, 1e-6, 0.0]),
          (Q.NB_R, [2, 0], [1e9]), (Q.NB_R, [1, 3], [1e7])]
    for b in br:
        nd.add_branch(*b)
    nd.add_port(1, 50.0)
    f = Q.grid_log(1e5, 1e9, 2001)
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    S = ctx.nodal_sweep(nd, f)
    assert ctx.nodal_last_kernel() in ("qo_nodal_kernel<static,local>", "qo_nodal_kernel<dense>")
    O = R.nodal_sweep([(k, n + [0] * (4 - len(n)), p + [0.0] * (4 - len(p))) for k, n, p in br], 3, [(1, 50.0)], f)
    assert np.max(np.abs(S - O)) < 1e-9
    assert np.all(np.isfinite(S.view(float)))
    # trip the guard on purpose (threshold |multiplier| <= 2 on the device only; the plan-time probes keep the real one): the
    # static launch flags points, the job is redone on the pivoted kernel, the result is the same
    assert ctx.nodal_last_kernel() == "qo_nodal_kernel<static,local>"
    monkeypatch.setenv("QO100NET_NODAL_GUARD2", "4.0")
    S2 = ctx.nodal_sweep(nd, f)
    assert ctx.nodal_last_kernel() == "qo_nodal_kernel<dense>"
    assert np.max(np.abs(S2 - O)) < 1e-9
    monkeypatch.setenv("QO100NET_NODAL", "static")          # ... and an explicit request for the static kernel reports the trip
    with pytest.raises(Q.QoError):
        ctx.nodal_sweep(nd, f)
    nd.close()


@pytest.mark.gpu
def test_gpu_nodal_static_and_dense_sweeps_reproduce_pa_bias_dataset(Q, R, ctx, pa_bias, golden_s2p, monkeypatch):
    """The CUDA nodal kernel through the C-ABI against the reference's 5-port dataset (all 13 entries x 5000
    points) and against the oracle."""
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    f = pa_bias["frequency"]
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    S = ctx.nodal_sweep(nd, f)
    assert ctx.nodal_last_kernel() == "qo_nodal_kernel<static,local>"    # symbolic plan accepted
    check_vs_dat(S, pa_bias)
    monkeypatch.setenv("QO100NET_NODAL", "dense")                          # per-point pivoting gives the same answer
    Sd = ctx.nodal_sweep(nd, f)
    assert ctx.nodal_last_kernel() == "qo_nodal_kernel<dense>"
    check_vs_dat(Sd, pa_bias)
    assert np.max(np.abs(S - Sd)) < 1e-9
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    register_inductor(R, golden_s2p)
    O = R.nodal_sweep(br, nn, ports, f)
    # the bias network is stiff (100 uF next to 1.2 pF): two correct LU orderings differ by ~1e-10 absolute
    assert np.max(np.abs(S - O)) < 1e-9
    R.sblock_clear()
    # a small network takes the LD=8 instantiation: a resistive pad with known S
    pad = Q.Nodal(2)
    pad.add_branch(Q.NB_R, [1, 2], [50.0])
    pad.add_port(1)
    pad.add_port(2)
    Sp = ctx.nodal_sweep(pad, np.array([1e6, 1e9]))
    assert np.allclose(Sp[:, 0, 0], 1 / 3) and np.allclose(Sp[:, 1, 0], 2 / 3) and np.allclose(Sp, Sp.transpose(0, 2, 1))


@pytest.mark.gpu
def test_gpu_nodal_monte_carlo_equals_oracle(Q, R, ctx, pa_bias, golden_s2p, monkeypatch):
    """Yield over the bias network's R/C tolerances: specs on |S21| (pass band) and |S31| (bias-port isolation);
    integer counters, histogram and FULL_S planes equal the oracle's."""
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    register_inductor(R, golden_s2p)
    f = pa_bias["frequency"][100:1400:13]                     # 0.2 - 2.8 GHz, 100 points
    nom = ctx.nodal_sweep(nd, f)
    s21 = 20 * np.log10(np.abs(nom[:, 1, 0]))
    s31 = 20 * np.log10(np.abs(nom[:, 2, 0]))
    band = (f >= 2.3e9) & (f <= 2.5e9)
    specs = [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, float(s21[band].min()) - 0.02),
             (Q.SPEC_S21_MAX_DB, 2, 0, 2.3e9, 2.5e9, float(s31[band].max()) + 0.3)]
    tols = [(i, 0, v, Q.TOL_REL, 0.05 if k == NB_C else 0.01) for v, (i, (k, _n, _p)) in
            enumerate((i, b) for i, b in enumerate(br) if b[0] in (NB_R, NB_C))]
    hist = dict(hist_bins=20, hist_spec=0, hist_lo=float(s21[band].min()) - 0.3, hist_hi=float(s21[band].min()) + 0.3)
    n = 400
    got = ctx.nodal_mc_run(nd, f, specs, 21, n, tols, **hist)
    monkeypatch.setenv("QO100NET_NODAL", "dense")
    dense = ctx.nodal_mc_run(nd, f, specs, 21, n, tols, **hist)
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    assert dense["n_pass"] == got["n_pass"] and np.array_equal(dense["hist"], got["hist"])
    from oracle import refbind
    ref = R.nodal_mc_run(br, nn, ports, f, specs, refbind.mc_cfg(21, n, tols, **hist), nthreads=8)
    assert got["n_total"] == n and got["n_pass"] == ref["n_pass"] and 0 < got["n_pass"] < n
    assert np.array_equal(got["fail_per_spec"], ref["fail_per_spec"]) and np.array_equal(got["hist"], ref["hist"])
    gs = ctx.nodal_mc_run(nd, f[:31], [], 21, 7, tols, mode=Q.MODE_FULL_S)["s"]
    os_ = R.nodal_mc_run(br, nn, ports, f[:31], [], refbind.mc_cfg(21, 7, tols), full_s=True)["s"]
    assert gs.shape == (7, 31, 5, 5) and np.max(np.abs(gs - os_)) < 1e-9
    R.sblock_clear()


def test_compiled_kernel_analysis_host_only(Q, pa_bias, golden_s2p):
    """qo_nodal_jit_analyze (no GPU: NVRTC only compiles): the reference's bias network printed as a straight-line kernel and
    compiled for sm_100a.  Minimum-degree ordering leaves 49 complex multiply-subtracts per point for a two-spec yield job
    (the netlist's own numbering: 175), nothing of the factorisation is addressed through the stack, and a yield job on two
    S entries solves fewer right-hand sides than the FULL_S job on all 25."""
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    f = pa_bias["frequency"]
    tols = [(b, 0, v, Q.TOL_REL, 0.05) for v, b in enumerate(i for i, (k, _n, _p) in enumerate(br) if k in (NB_R, NB_C))]
    specs = [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, -1.0), (Q.SPEC_S21_MAX_DB, 2, 0, 2.3e9, 2.5e9, -20.0)]
    a = nd.jit_analyze(f, specs, tols)
    if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
        pytest.skip("no NVRTC on this machine: " + a["error"][:120])
    assert a["compiled"], a
    assert 20 <= a["fms"] <= 80 and a["reciprocals"] <= 23 and a["registers"] <= 255 and a["stack_bytes"] <= 0      # -1: this NVRTC build does not echo ptxas -v into its log
    full = nd.jit_analyze(f, [], tols, mode=Q.MODE_FULL_S)
    assert full["compiled"] and full["fms"] > a["fms"]
    nd.close()


def test_compiled_kernel_generates_for_random_networks(Q):
    """The generator on six random N-port networks of tools/fuzz_nodal.py (R / L / C with parasitics, ideal buffers, 1-4 ports), host
    only: every network that takes the static plan compiles for sm_100a, FULL_S and yield flavour, with nothing on the stack."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("fuzz_nodal", os.path.join(ROOT, "tools", "fuzz_nodal.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    done = 0
    for i in range(6):
        rng = np.random.default_rng([9, i])
        br, nn, ports, tols, fc, nf, span = mod.random_network(rng)
        br = [b for b in br if b[0] != mod.NB_SBLOCK]
        f = Q.grid_log(fc / span, fc * span, nf)
        nd = Q.Nodal(nn)
        for kind, nodes, p in br:
            nd.add_branch(kind, nodes, p)
        for node, z in ports:
            nd.add_port(node, z)
        if not nd.analyze(f, tols)["static"]:
            nd.close()
            continue
        a = nd.jit_analyze(f, [(Q.SPEC_S21_MIN_DB, 0, len(ports) - 1, float(f[0]), float(f[-1]), -3.0)], tols)
        if not a["compiled"] and "libnvrtc" in (a["error"] or ""):
            pytest.skip("no NVRTC on this machine")
        b = nd.jit_analyze(f, [], tols, mode=Q.MODE_FULL_S)
        assert a["compiled"] and b["compiled"] and a["stack_bytes"] <= 0 and b["stack_bytes"] <= 0 and b["fms"] >= a["fms"], (i, a, b)
        done += 1
        nd.close()
    assert done >= 4


def test_compiled_kernel_disk_cache(Q, pa_bias, golden_s2p, tmp_path, monkeypatch):
    """QO100NET_CACHE_DIR: the cubin of a compiled network (and the compiler's log) is kept on disk under the hash of its source;
    a second process gets the kernel without running NVRTC and reports the same resource usage."""
    import subprocess
    import sys
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    f = pa_bias["frequency"][:200]
    if not nd.jit_analyze(f)["compiled"]:
        pytest.skip("no NVRTC on this machine")
    nd.close()
    code = ("import sys, json, numpy as np\n"
            "sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import qo100net as Q\n"
            "from test_nodal import build_nodal\n"
            "from conftest import GOLDEN\n"
            "import os\n"
            "g = np.load(os.path.join(GOLDEN, 'touchstone.npz')); d = np.load(os.path.join(GOLDEN, 'pa_bias_dat.npz'))\n"
            "nd, br, nn, ports = build_nodal(Q, g)\n"
            "print(json.dumps(nd.jit_analyze(d['frequency'][:200], [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, -1.0)])))\n"
            % (os.path.join(ROOT, "qo-100-tools_b200", "python"), os.path.join(ROOT, "tests"), ROOT))
    env = dict(os.environ, QO100NET_CACHE_DIR=str(tmp_path), QO100NET_NODAL_DEBUG="1")
    runs = [subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env) for _ in range(2)]
    assert all(r.returncode == 0 for r in runs), runs[0].stderr + runs[1].stderr
    a, b = [json.loads(r.stdout.strip().splitlines()[-1]) for r in runs]
    assert a["compiled"] and b == a and a["registers"] != 0
    assert "cubin from QO100NET_CACHE_DIR" not in runs[0].stderr and "cubin from QO100NET_CACHE_DIR" in runs[1].stderr
    files = sorted(os.listdir(tmp_path))
    assert len(files) == 2 and files[0].endswith("_sm100a.cubin") and files[1].endswith("_sm100a.log") and os.path.getsize(tmp_path / files[0]) > 10000


@pytest.mark.gpu
def test_gpu_nodal_compiled_kernel_equals_interpreted_dense_and_oracle(Q, R, ctx, pa_bias, golden_s2p, monkeypatch):
    """The run-time compiled kernel (QO100NET_NODAL=jit) on the reference network: the nominal sweep reproduces the reference
    dataset, Monte-Carlo counters and histogram equal the interpreted static kernel's, the pivoted kernel's and the oracle's,
    FULL_S planes agree to rounding, and the multiplier guard still hands a tripped job to the pivoted kernel."""
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    if not nd.jit_analyze(pa_bias["frequency"][:50])["compiled"]:
        pytest.skip("no NVRTC on this machine")
    register_inductor(R, golden_s2p)
    monkeypatch.setenv("QO100NET_NODAL", "jit")
    S = ctx.nodal_sweep(nd, pa_bias["frequency"])
    assert ctx.nodal_last_kernel() == "qo_nodal_jit_kernel"
    check_vs_dat(S, pa_bias)
    f = pa_bias["frequency"][100:1400:13]
    nom = ctx.nodal_sweep(nd, f)
    s21, s31 = 20 * np.log10(np.abs(nom[:, 1, 0])), 20 * np.log10(np.abs(nom[:, 2, 0]))
    band = (f >= 2.3e9) & (f <= 2.5e9)
    specs = [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, float(s21[band].min()) - 0.02),
             (Q.SPEC_S21_MAX_DB, 2, 0, 2.3e9, 2.5e9, float(s31[band].max()) + 0.3),
             (Q.SPEC_S21_MAX_DB, 4, 3, 0.0, 1e99, 3.0)]
    tols = [(i, 0, v, Q.TOL_REL, 0.05 if k == NB_C else 0.01) for v, (i, (k, _n, _p)) in
            enumerate((i, b) for i, b in enumerate(br) if b[0] in (NB_R, NB_C))]
    hist = dict(hist_bins=20, hist_spec=0, hist_lo=float(s21[band].min()) - 0.3, hist_hi=float(s21[band].min()) + 0.3)
    n = 3000
    got = ctx.nodal_mc_run(nd, f, specs, 21, n, tols, sample_offset=2 ** 33 + 5, **hist)
    assert ctx.nodal_last_kernel() == "qo_nodal_jit_kernel"
    gs = ctx.nodal_mc_run(nd, f[:31], [], 21, 7, tols, mode=Q.MODE_FULL_S)["s"]
    res = {}
    for mode in ("static", "dense"):
        monkeypatch.setenv("QO100NET_NODAL", mode)
        res[mode] = ctx.nodal_mc_run(nd, f, specs, 21, n, tols, sample_offset=2 ** 33 + 5, **hist)
        res[mode + "_s"] = ctx.nodal_mc_run(nd, f[:31], [], 21, 7, tols, mode=Q.MODE_FULL_S)["s"]
        for key in ("n_pass", "n_total"):
            assert res[mode][key] == got[key]
        assert np.array_equal(res[mode]["fail_per_spec"], got["fail_per_spec"]) and np.array_equal(res[mode]["hist"], got["hist"])
    # the compiled kernel forms ideal capacitors as j w C and its reciprocals by MUFU + Newton: last-bit differences in the stamps,
    # which this stiff network (100 uF next to 1.2 pF) amplifies to ~1e-11 absolute -- the order by which two pivot orders differ
    assert np.max(np.abs(gs - res["static_s"])) < 1e-9 and np.max(np.abs(gs - res["dense_s"])) < 1e-9
    from oracle import refbind
    ref = R.nodal_mc_run(br, nn, ports, f, specs, refbind.mc_cfg(21, n, tols, sample_offset=2 ** 33 + 5, **hist), nthreads=8)
    assert got["n_total"] == n and got["n_pass"] == ref["n_pass"] and 0 < got["n_pass"] < n
    assert np.array_equal(got["fail_per_spec"], ref["fail_per_spec"]) and np.array_equal(got["hist"], ref["hist"])
    # the guard: threshold |multiplier| <= 2 on the device only -> suspects flagged by the compiled kernel, job redone with pivoting
    monkeypatch.setenv("QO100NET_NODAL", "jit")
    monkeypatch.setenv("QO100NET_NODAL_GUARD2", "4.0")
    again = ctx.nodal_mc_run(nd, f, specs, 21, n, tols, sample_offset=2 ** 33 + 5, **hist)
    assert ctx.nodal_last_kernel() == "qo_nodal_kernel<dense>" and again["n_pass"] == got["n_pass"]
    R.sblock_clear()
    nd.close()


@pytest.mark.gpu
def test_gpu_nodal_job_sharded_over_the_gpus_of_a_ctx(Q, ctx, pa_bias, golden_s2p, monkeypatch):
    """qo_ctx_create(N): a nodal Monte-Carlo job is cut into N contiguous sample ranges, one per GPU; counters, histogram and
    FULL_S planes equal the one-GPU result (the Philox counter carries the global sample index)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    nd, br, nn, ports = build_nodal(Q, golden_s2p)
    f = pa_bias["frequency"][100:1400:13]
    specs = [(Q.SPEC_S21_MIN_DB, 1, 0, 2.3e9, 2.5e9, -3.0), (Q.SPEC_S21_MAX_DB, 2, 0, 2.3e9, 2.5e9, -25.0)]
    tols = [(i, 0, v, Q.TOL_REL, 0.05 if k == NB_C else 0.01) for v, (i, (k, _n, _p)) in
            enumerate((i, b) for i, b in enumerate(br) if b[0] in (NB_R, NB_C))]
    hist = dict(hist_bins=20, hist_spec=0, hist_lo=-6.0, hist_hi=0.0)
    ng = 4 if torch.cuda.device_count() >= 4 else 2
    cm = Q.Context(ngpus=ng)
    for mode in (("static", "jit") if nd.jit_analyze(f)["compiled"] else ("static",)):
        monkeypatch.setenv("QO100NET_NODAL", mode)
        one = ctx.nodal_mc_run(nd, f, specs, 3, 10001, tols, sample_offset=77, **hist)
        many = cm.nodal_mc_run(nd, f, specs, 3, 10001, tols, sample_offset=77, **hist)
        assert many["n_total"] == 10001 and many["n_pass"] == one["n_pass"] and 0 < one["n_pass"] < 10001
        assert np.array_equal(many["fail_per_spec"], one["fail_per_spec"]) and np.array_equal(many["hist"], one["hist"])
        s1 = ctx.nodal_mc_run(nd, f[:17], [], 3, 131, tols, mode=Q.MODE_FULL_S)["s"]
        sm = cm.nodal_mc_run(nd, f[:17], [], 3, 131, tols, mode=Q.MODE_FULL_S)["s"]
        assert np.array_equal(s1, sm)
    cm.close()
    nd.close()


@pytest.mark.gpu
def test_gpu_nodal_differential_fuzz(monkeypatch):
    """tools/fuzz_nodal.py on a fixed seed: 12 random N-port networks (3-13 nodes, R / L / C with parasitics, an ideal buffer in
    some, 1-4 ports): the run-time compiled kernel, the interpreted plan and per-point pivoting agree on FULL_S planes and on
    Monte-Carlo counters, every 4th network also with the oracle.  The long run (150 networks) is under profiles/fuzz/."""
    import importlib.util
    from conftest import ROOT
    monkeypatch.delenv("QO100NET_NODAL", raising=False)
    import qo100net
    probe = qo100net.Nodal(1)
    probe.add_branch(NB_R, [1, 0], [50.0])
    probe.add_port(1, 50.0)
    if not probe.jit_analyze(np.array([1e6, 2e6]))["compiled"]:
        pytest.skip("no NVRTC on this machine")
    spec = importlib.util.spec_from_file_location("fuzz_nodal", os.path.join(ROOT, "tools", "fuzz_nodal.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--nets", "12", "--seed", "3", "--samples", "1500"])
    assert out["mismatches"] == 0, out["details"]
    assert out["compared"] >= 10 and out["kernels"].get("qo_nodal_jit_kernel", 0) >= 10
