"""The QO100NET_* overrides of the cascade path and of the nodal path are each read in one function (csrc/qo_overrides.h:
qo_overrides_read, qo_nodal_overrides_read) and refused there when they make no sense -- CPU only."""
import os
import re

import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "qo-100-tools_b200", "csrc")
# diagnostics and I/O switches: read where they act, they choose no kernel
DIAGNOSTICS = {"CHAIN_DEBUG", "CHAIN_JIT_DUMP", "NODAL_DEBUG", "NODAL_JIT_DUMP", "CACHE_DIR", "NVRTC", "MC_TIMING", "NO_PLAN_CACHE"}


def _function_body(src, name):
    """[start, end) of the brace-delimited body of the definition of `name` in src"""
    m = re.search(r"\b%s\s*\([^;{)]*\)\s*\{" % name, src)
    assert m, name
    depth, i = 1, m.end()
    while depth:
        depth += {"{": 1, "}": -1}.get(src[i], 0)
        i += 1
    return m.end(), i


def test_cascade_and_nodal_overrides_are_read_in_one_place_each():
    """getenv("QO100NET_...") appears only inside qo_overrides_read and qo_nodal_overrides_read, apart from the diagnostics."""
    reader = os.path.join(CSRC, "qo_overrides.h")
    src = open(reader).read()
    bodies = {fn: _function_body(src, fn) for fn in ("qo_overrides_read", "qo_nodal_overrides_read")}
    stray, inside = [], {fn: set() for fn in bodies}
    for name in sorted(os.listdir(CSRC)):
        if not name.endswith((".c", ".cu", ".h", ".cuh")):
            continue
        path = os.path.join(CSRC, name)
        for m in re.finditer(r'getenv\("QO100NET_(\w+)"', open(path).read()):
            fn = next((fn for fn, (lo, hi) in bodies.items() if path == reader and lo <= m.start() < hi), None)
            if fn:
                inside[fn].add(m.group(1))
            elif m.group(1) not in DIAGNOSTICS:
                stray.append("%s: QO100NET_%s" % (name, m.group(1)))
    assert not stray, stray
    assert {"KERNEL", "CHAIN", "TF_TRUNC", "TF_TOL", "TF_NO_FRONT", "CPL_SINCOS", "USTRIP"} <= inside["qo_overrides_read"], inside
    assert {"NODAL", "NODAL_GUARD2"} <= inside["qo_nodal_overrides_read"], inside


def test_unknown_kernel_override_is_refused(Q, W, monkeypatch):
    """QO100NET_KERNEL takes auto, spot, tf, ladder or interp; anything else is an argument error, not a silent default."""
    w = W.cfg2()
    monkeypatch.setenv("QO100NET_KERNEL", "bogus")
    with pytest.raises(Q.QoError) as e:
        Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    assert e.value.status == Q.ERR_ARG and "QO100NET_KERNEL" in str(e.value)
    with pytest.raises(Q.QoError) as e:
        Q.chain_jit_analyze(w.net, w.f, w.specs, w.tols, **w.hist)
    assert e.value.status == Q.ERR_ARG
    for ok in ("auto", "spot", "tf"):
        monkeypatch.setenv("QO100NET_KERNEL", ok)
        assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)["reason"] == "ok"
    for off in ("ladder", "interp"):
        monkeypatch.setenv("QO100NET_KERNEL", off)
        assert Q.plan_analyze(w.net, w.f, w.specs, w.tols, **w.hist)["reason"] == "QO100NET_KERNEL override"


def test_unknown_nodal_override_is_refused(Q, monkeypatch):
    """QO100NET_NODAL takes auto, dense, static or jit; anything else is an argument error, not a silent default."""
    nd = Q.Nodal(2)
    nd.add_branch(Q.NB_R, [1, 2], [50.0])
    nd.add_port(1)
    nd.add_port(2)
    f = Q.grid_lin(1e6, 1e9, 16)
    monkeypatch.setenv("QO100NET_NODAL", "sttic")
    for call in (lambda: nd.analyze(f), lambda: nd.jit_analyze(f)):
        with pytest.raises(Q.QoError) as e:
            call()
        assert e.value.status == Q.ERR_ARG and "QO100NET_NODAL" in str(e.value)
    for ok in ("auto", "dense", "static", "jit"):
        monkeypatch.setenv("QO100NET_NODAL", ok)
        assert nd.analyze(f)["static"]
        nd.jit_analyze(f)
    nd.close()
