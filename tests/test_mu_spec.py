"""Amplifier stability yield: the Edwards-Sinsky stability factor mu as a spec (QO_SPEC_MU_MIN) on cascades with a measured block.

mu = (1 - |S11|^2) / (|S22 - Delta conj(S11)| + |S12 S21|), Delta = S11 S22 - S12 S21; mu > 1 is necessary and sufficient for
unconditional stability.  The job of interest is the reference's 20 W driver (active, non-reciprocal) between resistive pads whose
resistors carry tolerances: does it stay unconditionally stable for every build?  Such jobs run on the interpreter or the compiled
chain kernel only.  The host-only tests pin the numpy reference, the refusals, the planner's reason and that nothing else changed
(the chain kernel's source of other jobs, the interpreter's existing machine code); the GPU tests compare both kernels with the
oracle's FULL_S planes reduced in tools/fuzz_parity.py::oracle_counters."""
import hashlib
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from tools.fuzz_parity import SPEC_MU_MIN, mu_factor, oracle_counters

PAD_SHUNT = 292.0
PAD_TOLS = [(0, 0, 0, 0, 0.1), (1, 0, 1, 0, 0.1), (3, 0, 2, 0, 0.1), (4, 0, 3, 0, 0.1)]     # +-10 % uniform on the four pad resistors


def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "touchstone.npz"))


def driver(Q, R=None):
    """the 20 W driver (docs/pa-driver/pa_20W_vdd_32V_idq_180mA.s2p) as a block; registered with the oracle as block 0"""
    g = golden()
    fd, sd, z0 = g["pa_20W_f"], g["pa_20W_s"], float(g["pa_20W_z0"])
    if R is not None:
        R.sblock_clear()
        R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    return Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)


def padded_driver(Q, R=None, r=12.0):
    """shunt 292 Ohm, series r | driver | series r, shunt 292 Ohm, between 50 Ohm"""
    a = Q.Net.from_elements([(Q.SHUNT_R, [PAD_SHUNT]), (Q.SER_R, [r])], 50.0, 50.0)
    b = Q.Net.from_elements([(Q.SER_R, [r]), (Q.SHUNT_R, [PAD_SHUNT])], 50.0, 50.0)
    return a.concat(driver(Q, R).as_net(True, 50.0, 50.0)).concat(b)


def analyze(Q, net, f, specs, tols, **kw):
    return Q.plan_analyze(net, f, specs, tols, **kw)


# ---- host only --------------------------------------------------------------------------------------------------------------
def test_mu_reference_on_the_bare_driver():
    """numpy mu on the driver's 501 measured points agrees point by point with the K > 1 and |Delta| < 1 test; the closest point
    is 4.4e-4 from mu = 1, and mu reaches -2.77 at 7.22 GHz."""
    g = golden()
    s11, s21, s12, s22 = g["pa_20W_s"].T
    mu = mu_factor(s11, s21, s12, s22)
    d = s11 * s22 - s12 * s21
    k = (1 - np.abs(s11) ** 2 - np.abs(s22) ** 2 + np.abs(d) ** 2) / (2 * np.abs(s12 * s21))
    assert len(mu) == 501 and np.array_equal(mu > 1, (k > 1) & (np.abs(d) < 1))
    assert 4.3e-4 < np.min(np.abs(mu - 1)) < 4.5e-4
    assert abs(mu.min() + 2.77) < 0.01 and abs(g["pa_20W_f"][mu.argmin()] - 7.22e9) < 0.01e9
    assert 0.5 < np.mean(mu < 1) < 0.53


def test_refusals(Q, R, W):
    """A cascade without a measured block (QO_ERR_ARG), FP32 and microstrip networks (QO_ERR_UNSUPPORTED) do not compile; the nodal
    path and the oracle's own reduction still refuse kind 6; kind 7 is still unknown."""
    w2 = W.cfg2(nf=64)
    mu = (SPEC_MU_MIN, w2.f[0], w2.f[-1], 1.0)
    a = analyze(Q, w2.net, w2.f, [mu], w2.tols)
    assert not a["selected"] and a["reason"] == "network does not compile" and b"QO_SBLOCK" in Q.lib().qo_last_error()
    with pytest.raises(Q.QoError) as e:
        Q.chain_jit_analyze(w2.net, w2.f, [mu], w2.tols)
    assert e.value.status == Q.ERR_ARG
    with pytest.raises(RuntimeError):
        R.mc_run(R.make_elems(w2.net.elements), 50.0, 50.0, w2.f, [mu], R.mc_cfg(1, 4, w2.tols))
    net, f = padded_driver(Q), Q.grid_lin(20e6, 9e9, 256)
    a = analyze(Q, net, f, [(SPEC_MU_MIN, 20e6, 9e9, 1.0)], PAD_TOLS, precision=32)
    assert not a["selected"] and a["reason"] == "network does not compile" and b"FP64" in Q.lib().qo_last_error()
    w3 = W.cfg3(1000)
    a = analyze(Q, w3.net, w3.f, [(SPEC_MU_MIN, 2.3e9, 2.5e9, 1.0)], w3.tols)
    assert not a["selected"] and a["reason"] == "network does not compile" and b"microstrip" in Q.lib().qo_last_error()
    with pytest.raises(Q.QoError) as e:
        Q.chain_jit_analyze(w3.net, w3.f, [(SPEC_MU_MIN, 2.3e9, 2.5e9, 1.0)], w3.tols)
    assert e.value.status == Q.ERR_UNSUPPORTED
    nd = Q.Nodal(3)
    nd.add_branch(Q.NB_R, [1, 2, 0, 0], [10.0])
    nd.add_branch(Q.NB_C, [2, 0, 0, 0], [1e-9])
    nd.add_port(1, 50.0)
    nd.add_port(2, 50.0)
    with pytest.raises(Q.QoError) as e:
        nd.jit_analyze(w2.f, [(SPEC_MU_MIN, 1, 0, 1e6, 1e7, 1.0)], [])
    assert e.value.status == Q.ERR_ARG
    nd.close()
    a = analyze(Q, net, f, [(7, 20e6, 9e9, 1.0)], PAD_TOLS)
    assert not a["selected"] and a["reason"] == "network does not compile" and b"unknown kind 7" in Q.lib().qo_last_error()


def test_plan_analyze_reason(Q):
    """The padded-driver mu job, alone and next to |S21|, |S11| and |S22| specs, takes none of the polynomial, spot, ladder or
    thread-per-sample kernels and says why."""
    net, f = padded_driver(Q), Q.grid_lin(20e6, 9e9, 4096)
    mu = (SPEC_MU_MIN, 20e6, 9e9, 1.04)
    more = [(Q.SPEC_S21_MIN_DB, 2.3e9, 2.5e9, 10.0), (Q.SPEC_S11_MAX_DB, 2.3e9, 2.5e9, -6.0), (Q.SPEC_S22_MAX_DB, 2.3e9, 2.5e9, -6.0)]
    for specs in ([mu], [mu] + more, more[2:] + [mu]):
        a = analyze(Q, net, f, specs, PAD_TOLS, hist_bins=32, hist_spec=len(specs) - 1, hist_lo=0.9, hist_hi=1.2)
        assert not a["selected"] and a["reason"] == "stability spec needs all four S-parameters", (specs, a)
        assert Q.plan_ts_runs(net, f, specs, PAD_TOLS) == []


def chain_job(Q, W, name):
    """(net, grid, specs, tols, histogram) of the jobs whose chain-kernel source the tests look at"""
    if name == "cfg5":
        w5 = W.cfg5(nf=512)
        return w5.net, w5.f, w5.specs, w5.tols, w5.hist
    net, f = padded_driver(Q), Q.grid_lin(20e6, 9e9, 512)
    s21, mu = (Q.SPEC_S21_MIN_DB, 2.3e9, 2.5e9, 5.0), (SPEC_MU_MIN, 20e6, 9e9, 1.04)
    s11, s22 = (Q.SPEC_S11_MAX_DB, 2.3e9, 2.5e9, -6.0), (Q.SPEC_S22_MAX_DB, 2.3e9, 2.5e9, -6.0)
    if name == "padded_driver":
        return net, f, [s21, s11, s22], PAD_TOLS, dict(hist_bins=32, hist_spec=1, hist_lo=-20.0, hist_hi=0.0)
    mu_hist = dict(hist_bins=64, hist_lo=0.9, hist_hi=1.2)
    if name == "mu":
        return net, f, [mu], PAD_TOLS, dict(mu_hist, hist_spec=0)
    return net, f, [s21, mu, s22], PAD_TOLS, dict(mu_hist, hist_spec=1)


def chain_dump(tmp_path, name):
    """qo_chain_jit_analyze of chain_job(name) in a process of its own (the dump is written when a process first compiles a
    source) -> (its info, the source it compiled)"""
    dump = tmp_path / ("%s.cu" % name)
    code = ("import json, sys; sys.path[:0] = %r; import qo100net as Q; from qo100net import workloads as W; "
            "from test_mu_spec import chain_job; net, f, specs, tols, kw = chain_job(Q, W, %r); "
            "print(json.dumps(Q.chain_jit_analyze(net, f, specs, tols, **kw)))"
            % ([os.path.join(ROOT, "qo-100-tools_b200", "python"), os.path.join(ROOT, "tests"), ROOT], name))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=dict(os.environ, QO100NET_CHAIN_JIT_DUMP=str(dump)))
    assert r.returncode == 0, r.stderr
    info = json.loads(r.stdout.strip().split("\n")[-1])
    if not info["compiled"] and "libnvrtc" in (info["error"] or ""):
        pytest.skip("libnvrtc is not loadable here: %s" % info["error"])
    return info, dump.read_bytes()


def test_chain_kernel_compiles_mu_jobs(tmp_path):
    """A mu job, alone and next to |S21| and |S22| specs, compiles into the chain kernel on the 2x2 product, with no spills."""
    for name in ("mu", "mu_mix"):
        info, src = chain_dump(tmp_path, name)
        assert info["compiled"] and info["spill_bytes"] == 0, info
        assert b"#define QO_JIT_NEED_MU 1" in src and b"#define QO_JIT_ROW false" in src and b"#define QO_JIT_HIST_KIND 6" in src


# sha256 of the chain kernel's source, as QO100NET_CHAIN_JIT_DUMP writes it, before stability specs existed
PARENT_CHAIN_SOURCE = {"cfg5": "57c8bee074b92b6e0905ab1e9cd10ce257adc4022a32eb71f797d96213318acf",
                       "padded_driver": "dfd31d85a7259feb8e9f0fc13f10357ada8a6aaa45276da7c11c21977e614351"}


def test_chain_kernel_source_of_other_jobs_unchanged(tmp_path):
    """Config 5 (coupler in front, |S21|) and the padded driver with |S21|, |S11| and |S22| specs: the source handed to NVRTC --
    and so the kernel cache key under QO100NET_CACHE_DIR -- is byte for byte what it was."""
    st256 = b"#define QO_NO_ST256 1\n"           # present when the NVRTC that loaded is older than 12.9
    got = {}
    for name in PARENT_CHAIN_SOURCE:
        _info, src = chain_dump(tmp_path, name)
        assert b"QO_JIT_NEED_MU" not in src and b"//@mu" not in src
        got[name] = hashlib.sha256(src.replace(st256, b"")).hexdigest()
    assert got == PARENT_CHAIN_SOURCE


def lumped_instantiations(obj):
    """template arguments (T, then FULL_S TRIG GD S22 [MU] as 0/1) -> hash of the instruction text of that qo_mc_lumped_kernel
    instantiation, symbol names masked (cuobjdump -sass)"""
    sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    out = {}
    for blk in re.split(r"\n\s*Function : ", sass)[1:]:
        m = re.match(r"_Z19qo_mc_lumped_kernelI([df])((?:Lb[01]E)+)E", blk.split("\n", 1)[0].strip())
        if not m:
            continue
        h = hashlib.sha256()
        for ln in blk.split("\n"):
            ins = re.search(r"/\*[0-9a-f]{4,6}\*/\s+(.*?);", ln)
            if ins:
                h.update(re.sub(r"_Z\w+", "<sym>", ins.group(1).strip()).encode() + b"\n")
        out[m.group(1) + "".join(re.findall(r"Lb([01])E", m.group(2)))] = h.hexdigest()[:16]
    return out


# the interpreter's instantiations before stability specs existed, keyed T FULL_S TRIG GD S22 (nvcc of CUDA 12.9)
PARENT_INTERP_SASS = {
    "d0000": "a5623dec005d183d", "d0100": "5ea9b438829352ad", "d0010": "8df4b9ef49c62d8b", "d0110": "647048d691a98131",
    "d0001": "1ef8cf89321fad47", "d0101": "f950add3190fdb06", "d0011": "a1387547f43e087c", "d0111": "fabfb91dce069de2",
    "d1000": "e68143027d6e2fcf", "d1100": "a34dd733cfc34411", "f0000": "d35026054941958b", "f0100": "0249fb6f3a961e22",
    "f0010": "29b9f1f0f2779288", "f0110": "25f73e036c07dec8", "f0001": "16fba71c216c210e", "f0101": "175465a0eefd05ab",
    "f0011": "7a45a1b1cee02edb", "f0111": "87de02a42d551bee", "f1000": "12e0719139006b64", "f1100": "446570a17a50aed8"}


def test_interpreter_machine_code_unchanged():
    """Every existing interpreter instantiation (MU = false) compiles to the instructions it had; the one new instantiation is the
    FP64 reduce-only mu kernel (TRIG, as a mu job always holds a measured block; S22, so it serves |S22| specs too)."""
    obj = os.path.join(ROOT, "qo-100-tools_b200", "lib", "qo_cuda.o")
    if not os.path.exists(obj):
        pytest.skip("no qo_cuda.o (the library was not built in this tree)")
    try:
        ver = subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "--version"], capture_output=True, text=True).stdout
        got = lumped_instantiations(obj)
    except (OSError, subprocess.CalledProcessError):
        pytest.skip("cuobjdump / nvcc not available")
    if "release 12.9" not in ver:
        pytest.skip("the pinned hashes are of nvcc 12.9's output")
    assert {k[:-1]: v for k, v in got.items() if k[-1] == "0"} == PARENT_INTERP_SASS
    assert sorted(k for k in got if k[-1] == "1") == ["d01011"]


# ---- GPU --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ctx(Q):
    c = Q.Context(device=0)
    yield c
    c.close()


def run(Q, ctx, net, f, specs, tols, n, env=None, seed=21, **hist):
    """counters of the job and the kernel that ran, under the QO100NET_* overrides in env"""
    old = {k: os.environ.get(k) for k in ("QO100NET_KERNEL", "QO100NET_CHAIN")}
    for k in old:
        os.environ.pop(k, None)
    os.environ.update(env or {})
    try:
        p = Q.Plan(ctx, net, f, specs, seed=seed, tols=tols, **hist)
        p.launch(0, n)
        out = p.read()
        out["kernel"], out["reason"] = p.kernel_name, p.tf_info["reason"]
        p.close()
    finally:
        for k, v in old.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v
    return out


def same(a, b):
    return a["n_pass"] == b["n_pass"] and np.array_equal(a["fail_per_spec"], b["fail_per_spec"]) and np.array_equal(a["hist"], b["hist"])


def min_mu(R, net, f, band, tols, seed, n):
    """each sample's in-band minimum of mu, from the oracle's FULL_S planes"""
    rs, rl = net.terminations
    s = R.mc_run(R.make_elems(net.elements), rs, rl, f, [], R.mc_cfg(seed, n, tols), full_s=True, nthreads=R.max_threads())["s"]
    m = (f >= band[0]) & (f <= band[1])
    return mu_factor(*(np.asarray(s[q])[:, m] for q in range(4))).min(axis=1), s


def clear_limit(v, q):
    """a limit near quantile q of v, halfway between two neighbouring samples"""
    v = np.sort(v)
    i = int(q * (len(v) - 1))
    while v[i + 1] - v[i] < 1e-6 * max(1.0, abs(v[i])):
        i += 1
    return float(0.5 * (v[i] + v[i + 1]))


def clear_of(v, x):
    """no value within 1e-9 relative of x"""
    return bool(np.all(np.abs(v - x) > 1e-9 * max(1.0, abs(x))))


def hist_window(v, bins):
    lo, hi = float(np.quantile(v, 0.02)), float(np.quantile(v, 0.98))
    for k in range(100):                                  # nudge the window until no sample sits on a bin edge
        edges = lo + (hi - lo) * np.arange(bins + 1) / bins
        if all(clear_of(v, e) for e in edges):
            return dict(hist_bins=bins, hist_lo=lo, hist_hi=hi)
        lo -= 1.37e-7 * (hi - lo)
    raise AssertionError("no histogram window clear of the samples")


N_GPU = 2000
BAND = (20e6, 9e9)


@pytest.fixture(scope="module")
def mu_job(Q, R):
    net, f = padded_driver(Q, R), Q.grid_lin(BAND[0], BAND[1], 1024)
    v, planes = min_mu(R, net, f, BAND, PAD_TOLS, 21, N_GPU)
    lim = clear_limit(v, 0.5)
    return net, f, v, planes, lim


@pytest.mark.gpu
def test_mu_yield_matches_oracle(Q, R, ctx, mu_job):
    """Padded driver, +-10 % on the pads, mu >= limit over 20 MHz - 9 GHz with a histogram of the minimum mu: the interpreter and
    the compiled chain kernel both return the oracle's counters, integer for integer; the yield is strictly between 0 and 1."""
    net, f, v, _planes, lim = mu_job
    specs = [(SPEC_MU_MIN, BAND[0], BAND[1], lim)]
    hist = dict(hist_window(v, 64), hist_spec=0)
    assert clear_of(v, lim)
    o = oracle_counters(R, net, f, specs, R.mc_cfg(21, N_GPU, PAD_TOLS, **hist))
    assert 0 < o["n_pass"] < N_GPU and o["hist"].sum() == N_GPU and np.count_nonzero(o["hist"]) > 10
    a = run(Q, ctx, net, f, specs, PAD_TOLS, N_GPU, {"QO100NET_CHAIN": "interp"}, **hist)
    assert a["kernel"] == "qo_mc_lumped_kernel" and a["reason"] == "stability spec needs all four S-parameters"
    assert same(a, o), (a, o)
    b = run(Q, ctx, net, f, specs, PAD_TOLS, N_GPU, {"QO100NET_CHAIN": "jit"}, **hist)
    assert b["kernel"] == "qo_mc_chain_jit_kernel" and same(b, o), (b, o)


@pytest.mark.gpu
def test_mu_next_to_other_specs_matches_oracle(Q, R, ctx, mu_job):
    """The same job with |S21| min, |S11| and |S22| specs next to the mu spec, histogram on mu and on |S11|: both kernels equal the
    oracle."""
    net, f, v, planes, lim = mu_job
    driver(Q, R)
    m = (f >= 2.3e9) & (f <= 2.5e9)
    db = [20 * np.log10(np.abs(np.asarray(planes[q])[:, m])) for q in (1, 0, 3)]
    s21 = (Q.SPEC_S21_MIN_DB, 2.3e9, 2.5e9, clear_limit(db[0].min(axis=1), 0.4))
    w11, w22 = db[1].max(axis=1), db[2].max(axis=1)
    s11 = (Q.SPEC_S11_MAX_DB, 2.3e9, 2.5e9, clear_limit(w11, 0.6))
    s22 = (Q.SPEC_S22_MAX_DB, 2.3e9, 2.5e9, clear_limit(w22, 0.6))
    specs = [s21, s11, (SPEC_MU_MIN, BAND[0], BAND[1], lim), s22]
    for hist in (dict(hist_window(v, 64), hist_spec=2), dict(hist_window(w11, 32), hist_spec=1)):
        o = oracle_counters(R, net, f, specs, R.mc_cfg(21, N_GPU, PAD_TOLS, **hist))
        assert all(0 < x < N_GPU for x in o["fail_per_spec"]), o
        for env in ({"QO100NET_CHAIN": "interp"}, {"QO100NET_CHAIN": "jit"}):
            a = run(Q, ctx, net, f, specs, PAD_TOLS, N_GPU, env, **hist)
            assert same(a, o), (env, a, o)


@pytest.mark.gpu
def test_mu_behind_a_reciprocal_block(Q, R, W, ctx):
    """A lossy ladder (ESR / SRF parasitics) behind the measured Coilcraft inductor: every block is reciprocal, so the plan has no
    determinant table (det = 1).  The losses keep each sample's minimum mu a little above 1 (a lossless cascade sits at mu = 1 to
    rounding, a knife edge).  Both kernels equal the oracle."""
    g = golden()
    fd, sd, z0 = g["11SQ39N_f"], g["11SQ39N_s"], float(g["11SQ39N_z0"])
    R.sblock_clear()
    R.sblock_register(0, fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    blk = Q.SBlock.from_arrays(fd, sd[:, 0], sd[:, 1], sd[:, 2], sd[:, 3], z0)
    lad = Q.Net.butter_lpf(5, 400e6, 50.0, True).add_parasitics(400e6, 40.0, 20.0, 0.3, 30.0)
    net = blk.as_net(True, 50.0, 50.0).concat(lad)
    tols = [(e + 1, p, v, m, t) for (e, p, v, m, t) in Q.lc_tolerances(lad, 0.05, 0.05)]
    f, band = Q.grid_log(100e6, 900e6, 300), (100e6, 350e6)
    v, _s = min_mu(R, net, f, band, tols, 21, 600)
    assert np.all(v > 1.001)                               # passive and lossy: mu > 1
    lim = clear_limit(v, 0.5)
    specs = [(SPEC_MU_MIN, band[0], band[1], lim)]
    hist = dict(hist_window(v, 64), hist_spec=0)
    o = oracle_counters(R, net, f, specs, R.mc_cfg(21, 600, tols, **hist))
    assert 0 < o["n_pass"] < 600
    for env in ({"QO100NET_CHAIN": "interp"}, {"QO100NET_CHAIN": "jit"}):
        a = run(Q, ctx, net, f, specs, tols, 600, env, **hist)
        assert same(a, o), (env, a, o)


@pytest.mark.gpu
def test_mu_refusals_on_the_device(Q, W, ctx):
    """qo_mc_run: kind 6 on a cascade without a block is QO_ERR_ARG, in FP32 QO_ERR_UNSUPPORTED."""
    w2 = W.cfg2(nf=64)
    with pytest.raises(Q.QoError) as e:
        ctx.mc_run(w2.net, w2.f, [(SPEC_MU_MIN, w2.f[0], w2.f[-1], 1.0)], 1, 64, w2.tols)
    assert e.value.status == Q.ERR_ARG
    with pytest.raises(Q.QoError) as e:
        ctx.mc_run(padded_driver(Q), Q.grid_lin(20e6, 9e9, 64), [(SPEC_MU_MIN, 20e6, 9e9, 1.0)], 1, 64, PAD_TOLS, precision=32)
    assert e.value.status == Q.ERR_UNSUPPORTED


@pytest.mark.gpu
def test_mu_interpreter_equals_chain_kernel_at_scale(Q, ctx, mu_job):
    """2e6 samples x 4096 points of the padded-driver mu job with a histogram: interpreter and compiled chain kernel, identical
    counters."""
    _net, _f, v, _planes, lim = mu_job
    net, f = padded_driver(Q), Q.grid_lin(BAND[0], BAND[1], 4096)
    specs = [(Q.SPEC_S21_MIN_DB, 2.3e9, 2.5e9, 10.0), (SPEC_MU_MIN, BAND[0], BAND[1], lim)]
    hist = dict(hist_window(v, 128), hist_spec=1)
    n = 2000000
    a = run(Q, ctx, net, f, specs, PAD_TOLS, n, {"QO100NET_CHAIN": "interp"}, **hist)
    b = run(Q, ctx, net, f, specs, PAD_TOLS, n, {"QO100NET_CHAIN": "jit"}, **hist)
    assert a["kernel"] == "qo_mc_lumped_kernel" and b["kernel"] == "qo_mc_chain_jit_kernel"
    assert 0 < a["fail_per_spec"][1] < n and same(a, b), (a, b)


@pytest.mark.gpu
def test_differential_fuzz_with_mu_specs(Q, monkeypatch):
    """tools/fuzz_parity.py --mu on a fixed seed: random lumped cascades with the driver in front or behind and a mu spec in every
    job -- compiled chain kernel, interpreter and (every 5th) the oracle agree."""
    import importlib.util
    monkeypatch.delenv("QO100NET_KERNEL", raising=False)
    spec = importlib.util.spec_from_file_location("fuzz_parity", os.path.join(ROOT, "tools", "fuzz_parity.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--mu", "--nets", "60", "--samples", "1500", "--seed", "62", "--big-every", "5"])
    assert out["mismatches"] == 0, out["details"]
    assert out["compared"] >= 25 and out["oracle_checked"] >= 5 and out["mu_jobs"] == out["compared"]
