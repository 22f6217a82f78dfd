import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "qo-100-tools_b200", "python"))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
# a checkout of the upstream qo-100-tools tree, which tests/golden/ was extracted from (tools/make_golden.py): the few tests that
# read its files directly skip without it
REFERENCE = os.environ.get("QO100_REFERENCE", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def Q():
    import qo100net
    if not os.path.exists(qo100net.LIB_PATH):
        qo100net.build()
    qo100net.lib()
    return qo100net


@pytest.fixture(scope="session")
def R():
    from oracle import refbind
    refbind.lib()
    return refbind


@pytest.fixture(scope="session")
def W(Q):
    from qo100net import workloads
    return workloads


@pytest.fixture(scope="session")
def golden_dat():
    return np.load(os.path.join(GOLDEN, "pa_lpf_dat.npz"))


@pytest.fixture(scope="session")
def golden_s2p():
    return np.load(os.path.join(GOLDEN, "touchstone.npz"))


def np_spfile(f, fd, sd, polar=True):
    """Independent numpy restatement of Qucs SPfile 'linear' interpolation (third implementation next to the
    product's and the oracle's): sd is [n,4] complex (S11 S21 S12 S22) at fd; end segments extrapolated."""
    f = np.asarray(f, dtype=float)
    k = np.clip(np.searchsorted(fd, f, side="right") - 1, 0, len(fd) - 2)
    t = ((f - fd[k]) / (fd[k + 1] - fd[k]))[:, None]
    a, b = sd[k], sd[k + 1]
    if not polar:
        return a + t * (b - a)
    dp = np.angle(b) - np.angle(a)
    dp = np.where(dp > np.pi, dp - 2 * np.pi, np.where(dp < -np.pi, dp + 2 * np.pi, dp))
    return (np.abs(a) + t * (np.abs(b) - np.abs(a))) * np.exp(1j * (np.angle(a) + t * dp))


def np_s_to_abcd(s, z0):
    s11, s21, s12, s22 = s[:, 0], s[:, 1], s[:, 2], s[:, 3]
    d = 2 * s21
    return np.stack([((1 + s11) * (1 - s22) + s12 * s21) / d, z0 * ((1 + s11) * (1 + s22) - s12 * s21) / d,
                     ((1 - s11) * (1 - s22) - s12 * s21) / d / z0, ((1 - s11) * (1 + s22) + s12 * s21) / d], axis=1)


@pytest.fixture(scope="session")
def golden_nets():
    return json.load(open(os.path.join(GOLDEN, "networks.json")))


@pytest.fixture(scope="session")
def golden_b():
    return json.load(open(os.path.join(GOLDEN, "appendix_b.json")))


@pytest.fixture(scope="session")
def ctx(Q):
    """A device context; the CUDA path must be the one that runs -- no fallback."""
    c = Q.Context(device=0)
    yield c
    c.close()


def to_ref(R, net):
    return R.make_elems(net.elements)


def relerr(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b)) / np.maximum(np.abs(np.asarray(b)), 1e-300)))


@pytest.fixture(scope="session")
def png_curves():
    """Pixels of the S21 / S11 curves of the reference's rf-tools plots + axis calibration (tools/make_golden.py png_curves)."""
    return np.load(os.path.join(GOLDEN, "rftools_png_curves.npz"))


def png_curve_distance(curves, key, sweep):
    """How far the reference's plotted curves lie from a model.  sweep(f) -> (s11, s21) complex arrays.
    Returns {"s21": (max_px, p99_px, covered), "s11": ...}: distances in pixels from every curve pixel of the PNG to the model
    polyline drawn in the same axes (1 px = 0.17 dB of S21, 0.086 dB of S11, 0.49 % in frequency), and the share of the model's
    visible points that have a curve pixel (of either colour: the red curve is drawn over the blue one) within 2.5 px."""
    from scipy.spatial import cKDTree
    ticks, (ax_l, ax_r, y0, y1) = curves[key + "_xticks"], curves[key + "_frame"]
    b, a = np.polyfit(np.log10(ticks[:, 1]), ticks[:, 0], 1)              # column = a + b log10(f)
    x = np.linspace(ax_l, ax_r, 40000)
    f = 10.0 ** ((x - a) / b)
    s11, s21 = sweep(f)
    pb, pr = curves[key + "_s21_px"].astype(float), curves[key + "_s11_px"].astype(float)
    out = {}
    for name, s, pix, cover, span in (("s21", s21, pb, np.vstack([pb, pr]), 80.0), ("s11", s11, pr, pr, 40.0)):
        y = y0 - 20.0 * np.log10(np.abs(s)) * ((y1 - y0) / span)
        ok = (y >= y0) & (y <= y1 - 1) & (x >= ax_l + 3) & (x <= ax_r - 2)
        model = np.stack([x[ok], y[ok]], 1)
        d = cKDTree(model).query(pix)[0]
        dc = cKDTree(cover).query(model)[0]
        out[name] = (float(d.max()), float(np.percentile(d, 99)), float(np.mean(dc <= 2.5)))
    return out
