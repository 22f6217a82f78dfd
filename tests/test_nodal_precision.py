"""N-port nodal analysis against a 40-digit MNA solve, entry by entry, bounded by each S entry's condition number.

The reference restates oracle/qo100ref_nodal.c::nodal_point stamp for stamp in mpmath at 40 digits, from the exact doubles of the
frequency and of every branch parameter (omega = 2 pi f at 40 digits); a measured block enters with the oracle's interpolated S, the
same doubles the kernels start from.  Next to S it returns, for every entry, the componentwise condition number

    K[k][j] = 2 sqrt(Zj/Zk) sum_(r,c) |lambda_k[r]| (sum of |stamps landing on A[r][c]|) |x_j[c]|,  x_j = A^-1 b_j, lambda_k = A^-T e_k,

the first-order change of S[k][j] when every stamp moves by its own relative rounding.  A backward-stable double-precision MNA
(rounded stamps, pivoted LU) then meets |S - S_ref| <= C u K with C near 1, u = 2^-53.  A bound on the summed matrix |A| does not
hold: the bias network's 100 uF DC block stamps ~6e5 S into diagonals that also hold ~0.02 S, and rounding the sum drops the small
admittances' low digits -- that is why its isolation entries S31 / S23 cannot be computed to 1e-9 relative in double above ~1 GHz.

Entries with K = 0 are exactly zero in exact arithmetic.  Between the bias network's two unconnected sub-circuits every kernel
returns exact zeros; the reverse isolation of an ideal buffer (S12, S13, S45) cancels numerically, so it is bounded by C u times the
largest entry of its column, the scale the cancelling terms carry.

CPU part: the reference against the oracle, the exact zeros, and the premises (which kernel instantiations the networks reach).
GPU part (marked): every kernel -- pivoted dense, the static plan, the compiled plan -- against the reference on FULL_S planes and on
Monte-Carlo verdicts and histogram bins placed within a few C u K of the reference's worst value."""
import importlib.util
import os

import mpmath
import numpy as np
import pytest

from conftest import ROOT
from test_nodal import build_nodal, hand_netlist, register_inductor

NB_R, NB_L, NB_C, NB_VCVS, NB_SBLOCK = 1, 2, 3, 4, 5
U = 2.0 ** -53
# |S_kernel - S_ref| <= C_BOUND u K on every entry, every kernel: 4x the oracle's worst (8.1 u K, S44 of the bias network at 2.3 GHz).
# C lies above 16 for two reasons.  The bias ports 1 and 4 see exactly their own 50 Ohm, so S11 = S44 = 2 V - 1 = 0 with K = 1 from
# the port's own row -- but partial pivoting takes the buffer's row (|G| = 1 > 0.04 S) as that column's pivot, and V then carries the
# LU's rounding of the rows behind it (gamma_n |L||U|), which K, built from the stamps alone, does not see.  The fixed pivot orders add
# the growth of their multipliers (3.2e5 in the bias network's stiff band, ~100 on the 32-unknown mesh).  Observed on a B200: dense
# 6.2, static plan 15.2 (bias, 1.08 MHz, S32) and 28.9 (mesh, S67), compiled plan 29.0.
C_BOUND = 33.0
DPS = 40


# ---- the 40-digit reference ------------------------------------------------------------------------------------------------------
def _lu(M):
    """LU with partial pivoting, in place on a list of rows (mpc); zero multipliers skipped.  -> (M, perm)"""
    n = len(M)
    perm = list(range(n))
    for c in range(n):
        piv = max(range(c, n), key=lambda r: abs(M[r][c]))
        if M[piv][c] == 0:
            raise ZeroDivisionError("singular MNA matrix")
        if piv != c:
            M[c], M[piv] = M[piv], M[c]
            perm[c], perm[piv] = perm[piv], perm[c]
        inv = 1 / M[c][c]
        cols = [j for j in range(c + 1, n) if M[c][j] != 0]
        for r in range(c + 1, n):
            if M[r][c] == 0:
                continue
            lv = M[r][c] * inv
            M[r][c] = lv
            row, prow = M[r], M[c]
            for j in cols:
                row[j] -= lv * prow[j]
    return M, perm


def _lu_solve(M, perm, b):
    n = len(M)
    x = [b[perm[i]] for i in range(n)]
    for i in range(n):
        for q in range(i):
            if M[i][q] != 0 and x[q] != 0:
                x[i] -= M[i][q] * x[q]
    for i in range(n - 1, -1, -1):
        for q in range(i + 1, n):
            if M[i][q] != 0 and x[q] != 0:
                x[i] -= M[i][q] * x[q]
        x[i] /= M[i][i]
    return x


def _cancelled(v):
    """40-digit residues of terms that cancel exactly (an ideal buffer's reverse path) -> exact zeros"""
    top = max(abs(a) for a in v)
    return [a if abs(a) > top * mpmath.mpf(10) ** (12 - DPS) else mpmath.mpc(0) for a in v]


def ref_point(R, br, nn, ports, f):
    """S and K at one frequency (see the module docstring).  br: (kind, nodes, params) as the oracle takes them, measured blocks
    registered with the oracle.  -> (S_hi, S_lo, K): S = S_hi + S_lo to ~32 digits, K in double."""
    with mpmath.workdps(DPS):
        mpf, mpc = mpmath.mpf, mpmath.mpc
        J = mpc(0, 1)
        w = 2 * mpmath.pi * mpf(float(f))
        n = nn + sum(1 for b in br if b[0] == NB_VCVS)
        A = [[mpc(0) for _ in range(n)] for _ in range(n)]
        mag = {}

        def add(r, c, y):
            A[r][c] += y
            mag[(r, c)] = mag.get((r, c), 0.0) + float(abs(y))

        def stamp_y(a, b, y):
            if a:
                add(a - 1, a - 1, y)
            if b:
                add(b - 1, b - 1, y)
            if a and b:
                add(a - 1, b - 1, -y)
                add(b - 1, a - 1, -y)
        extra = nn
        for kind, nodes, p in br:
            p = [mpf(float(v)) for v in p] + [mpf(0)] * (4 - len(p))
            if kind == NB_R:
                stamp_y(nodes[0], nodes[1], 1 / p[0])
            elif kind == NB_L:                  # (R + jwL) || 1/(jwCp)
                stamp_y(nodes[0], nodes[1], (1 - w * w * p[0] * p[2] + J * w * p[1] * p[2]) / (p[1] + J * w * p[0]))
            elif kind == NB_C:                  # R + jwLs + 1/(jwC)
                stamp_y(nodes[0], nodes[1], 1 / (p[1] + J * (w * p[2] - 1 / (w * p[0]))))
            elif kind == NB_VCVS:               # in+, out+, out-, in-; V(o+) - V(o-) = G e^{-jwT} (V(i+) - V(i-))
                ip, op, om, im = (list(nodes) + [0, 0])[:4]
                kx = extra
                extra += 1
                g = p[0] * mpmath.expj(-w * p[1])
                if op:
                    add(op - 1, kx, mpc(1))
                    add(kx, op - 1, mpc(1))
                if om:
                    add(om - 1, kx, mpc(-1))
                    add(kx, om - 1, mpc(-1))
                if ip:
                    add(kx, ip - 1, -g)
                if im:
                    add(kx, im - 1, g)
            elif kind == NB_SBLOCK:             # Y = (I - S)(I + S)^-1 / z0, indefinite third terminal
                s11, s21, s12, s22 = [mpc(v) for v in R.sblock_s(int(p[0]), float(f), p[1] != 0)]
                a, d = 1 + s11, 1 + s22
                det = a * d - s12 * s21
                y = [[((1 - s11) * d + s12 * s21) / det, (-s12 * a - (1 - s11) * s12) / det],
                     [(-s21 * d - (1 - s22) * s21) / det, (s21 * s12 + (1 - s22) * a) / det]]
                Y3 = [[y[r][c] / p[2] for c in range(2)] for r in range(2)]
                for r in range(2):
                    Y3[r].append(-(Y3[r][0] + Y3[r][1]))
                Y3.append([-(Y3[0][c] + Y3[1][c]) for c in range(3)])
                t = list(nodes[:3])
                for r in range(3):
                    for c in range(3):
                        if t[r] and t[c]:
                            add(t[r] - 1, t[c] - 1, Y3[r][c])
            else:
                raise ValueError("branch kind %d" % kind)
        for node, z in ports:
            stamp_y(node, 0, 1 / mpf(float(z)))
        npn = len(ports)
        LU, perm = _lu([row[:] for row in A])
        LUt, permt = _lu([[A[c][r] for c in range(n)] for r in range(n)])
        X, Lam = [], []
        for j, (node, z) in enumerate(ports):
            b = [mpc(0)] * n
            b[node - 1] = 1 / mpf(float(z))
            X.append(_cancelled(_lu_solve(LU, perm, b)))
            e = [mpc(0)] * n
            e[node - 1] = mpc(1)
            Lam.append(_cancelled(_lu_solve(LUt, permt, e)))
        S_hi = np.zeros((npn, npn), complex)
        S_lo = np.zeros((npn, npn), complex)
        K = np.zeros((npn, npn))
        ax = [[float(abs(v)) for v in x] for x in X]
        al = [[float(abs(v)) for v in lam] for lam in Lam]
        for k, (nk, zk) in enumerate(ports):
            for j, (nj, zj) in enumerate(ports):
                sc = 2 * mpmath.sqrt(mpf(float(zj)) / mpf(float(zk)))
                s = sc * X[j][nk - 1] - (1 if k == j else 0)
                S_hi[k, j] = complex(s)
                S_lo[k, j] = complex(s - mpc(S_hi[k, j]))
                K[k, j] = float(sc) * sum(al[k][r] * m * ax[j][c] for (r, c), m in mag.items())
    return S_hi, S_lo, K


class Reference:
    """40-digit S and K of one network, per frequency, computed once per test session."""

    def __init__(self, R, br, nn, ports, register=None):
        self.R, self.br, self.nn, self.ports, self.register = R, br, nn, ports, register
        self.pts = {}

    def at(self, f):
        """-> (S_hi, S_lo, K) arrays [nf, np, np]"""
        f = np.asarray(f, dtype=float)
        todo = [x for x in f if float(x) not in self.pts]
        if todo:
            if self.register:
                self.register()
            for x in todo:
                self.pts[float(x)] = ref_point(self.R, self.br, self.nn, self.ports, float(x))
        out = [self.pts[float(x)] for x in f]
        return tuple(np.array([o[i] for o in out]) for i in range(3))

    def ratio(self, S, f):
        """|S - S_ref| / (u K) per entry, with the exact zeros (K = 0) bounded by u times their column's largest |S_ref|"""
        hi, lo, K = self.at(f)
        err = np.abs((np.asarray(S) - hi) - lo)
        col = np.max(np.abs(hi), axis=1, keepdims=True)
        return err / (U * np.where(K > 0, K, col))

    def oracle(self, f):
        if self.register:
            self.register()
        return self.R.nodal_sweep(self.br, self.nn, self.ports, f)


# ---- networks ------------------------------------------------------------------------------------------------------------------
def _bias_grid():
    """129 points: the stiff band 1 - 3 MHz, the decades to the preamp band, the preamp plot's three markers, the measured
    inductor's data end (3.3 GHz) and its self-resonance in the extrapolated range (4.55 GHz), up to 10 GHz"""
    f = np.concatenate([np.geomspace(1e6, 3e6, 16), np.geomspace(3.5e6, 2e9, 42), np.linspace(2.2e9, 2.6e9, 21),
                        [2.38924e9, 2.40324e9, 2.40724e9], np.linspace(3.25e9, 3.35e9, 5), np.geomspace(3.4e9, 4.5e9, 10),
                        np.linspace(4.52e9, 4.58e9, 13), np.geomspace(4.6e9, 1e10, 19)])
    assert len(f) == 129 and len(np.unique(f)) == 129
    return np.sort(f)


BIAS_GRID = _bias_grid()
STIFF = BIAS_GRID[BIAS_GRID <= 3e6]


def mesh_network(rows, cols, zports, n_buf, fc, seed):
    """A rows x cols grid of R / L / C branches (values around 50 Ohm at fc, parasitics on half of them), shunts to ground on a
    third of the nodes, and n_buf ideal buffers (the last one with a delay) from grid nodes to fresh nodes that drive the grid
    back through a resistor.  Ports on len(zports) grid nodes spread over the grid.  -> (branches, nodes, ports)"""
    rng = np.random.default_rng(seed)
    wc = 2 * np.pi * fc

    def branch(kind, a, b):
        g = rng.uniform(0.3, 3.0)
        par = rng.random() < 0.5
        if kind == NB_R:
            return (NB_R, [a, b], [50.0 * g])
        if kind == NB_L:
            L = 50.0 * g / wc
            return (NB_L, [a, b], [L, rng.uniform(0.1, 2.0), 1 / (L * (wc * rng.uniform(5, 30)) ** 2)] if par else [L, 0.0, 0.0])
        C = g / (50.0 * wc)
        return (NB_C, [a, b], [C, rng.uniform(0.05, 1.0), 1 / (C * (wc * rng.uniform(8, 40)) ** 2)] if par else [C, 0.0, 0.0])

    def node(r, c):
        return r * cols + c + 1
    kinds = [NB_R, NB_L, NB_C]
    br = []
    for r in range(rows):
        for c in range(cols):
            if c + 1 < cols:
                br.append(branch(kinds[(r + 2 * c) % 3], node(r, c), node(r, c + 1)))
            if r + 1 < rows:
                br.append(branch(kinds[(2 * r + c + 1) % 3], node(r, c), node(r + 1, c)))
            if (r + c) % 3 == 0:
                br.append(branch(kinds[(r + c) % 3], node(r, c), 0))
    nn = rows * cols
    for b in range(n_buf):
        nn += 1
        src = node((b * (rows - 1)) // max(1, n_buf - 1) if n_buf > 1 else 0, 0)
        delay = rng.uniform(0.05, 0.3) / fc if b == n_buf - 1 else 0.0
        br.append((NB_VCVS, [src, nn, 0, 0], [rng.uniform(0.5, 3.0), delay]))
        br.append((NB_R, [nn, node(rows - 1 - b % rows, cols - 1)], [50.0 * rng.uniform(0.5, 3.0)]))
    pick = [int(round(x)) + 1 for x in np.linspace(0, rows * cols - 1, len(zports))]
    assert len(set(pick)) == len(zports)
    return br, nn, [(p, float(z)) for p, z in zip(pick, zports)]


def _mesh_grid(fc):
    return np.geomspace(fc / 10, fc * 10, 129)


# name -> (branches, nodes, ports, grid); the measured block appears in the bias network only
NETS = {
    "bias": hand_netlist() + (BIAS_GRID,),
    # 28 grid nodes + 2 buffer outputs + 2 buffer currents = 32 unknowns (QO_NODAL_MAX_UNK), 8 ports (QO_NODAL_MAX_PORTS) at 50 / 75 Ohm, a delayed buffer
    "mesh32": mesh_network(4, 7, [50.0, 75.0] * 4, 2, 4e8, 32) + (_mesh_grid(4e8),),
    # 12 + 1 nodes + 1 buffer current = 14 unknowns, 2 ports at 50 / 75 Ohm, a delayed buffer
    "mesh14": mesh_network(3, 4, [75.0, 50.0], 1, 1.5e9, 14) + (_mesh_grid(1.5e9),),
    # 6 unknowns, one port
    "oneport": mesh_network(2, 3, [50.0], 0, 6e7, 6) + (_mesh_grid(6e7),),
}


_REFS = {}


def reference(R, golden_s2p, name):
    """the module's Reference of network `name` (built once per session: ~4 s on the bias grid, ~15 s on the 32-unknown mesh)"""
    if name not in _REFS:
        br, nn, ports, _f = NETS[name]
        reg = (lambda: register_inductor(R, golden_s2p)) if any(b[0] == NB_SBLOCK for b in br) else None
        _REFS[name] = Reference(R, br, nn, ports, reg)
    return _REFS[name]


def _fuzz_module():
    spec = importlib.util.spec_from_file_location("fuzz_nodal", os.path.join(ROOT, "tools", "fuzz_nodal.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def product_nodal(Q, golden_s2p, name):
    """network `name` as a product object"""
    br, nn, ports, _f = NETS[name]
    if name == "bias":
        return build_nodal(Q, golden_s2p)[0]
    nd = Q.Nodal(nn)
    for b in br:
        nd.add_branch(*b)
    for node, z in ports:
        nd.add_port(node, z)
    return nd


# ---- CPU: the reference against the oracle -------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(NETS))
def test_reference_bounds_the_oracle(R, golden_s2p, name):
    """The double-precision oracle (pivoted LU) against the 40-digit reference on every entry and grid point: within C u K.  On the
    bias grid this covers the stiff band (1 - 3 MHz), the preamp markers, the measured inductor's self-resonance in its
    extrapolated range and 10 GHz; there the oracle is off by ~1e-8 relative on S31 / S23 and still inside the bound."""
    f = NETS[name][3]
    ref = reference(R, golden_s2p, name)
    r = ref.ratio(ref.oracle(f), f)
    assert np.all(np.isfinite(r)) and r.max() <= C_BOUND, (r.max(), np.unravel_index(np.argmax(r), r.shape))
    if name == "bias":
        hi, _lo, K = ref.at(f)
        rel = np.abs(ref.oracle(f)[:, 2, 0] - hi[:, 2, 0]) / np.abs(hi[:, 2, 0])
        # the isolation entries are not computable to 1e-9 relative in double above ~1 GHz: u K / |S| reaches 2.7e-8 at 10 GHz
        assert rel.max() > 1e-9 and U * (K[:, 2, 0] / np.abs(hi[:, 2, 0]))[f >= 9.9e9].max() > 2e-8


def test_reference_bounds_the_oracle_on_random_networks(R, golden_s2p):
    """twelve networks of tools/fuzz_nodal.py (R / L / C with parasitics, ideal buffers with and without delay, the measured inductor,
    1-4 ports at 50 / 75 Ohm), nine points across each band"""
    mod = _fuzz_module()
    worst, seen = 0.0, set()
    for i in range(12):
        br, nn, ports, _tols, fc, _nf, span = mod.random_network(np.random.default_rng([17, i]))
        seen |= {b[0] for b in br}
        f = np.geomspace(fc / span, fc * span, 9)
        reg = (lambda: register_inductor(R, golden_s2p)) if any(b[0] == NB_SBLOCK for b in br) else None
        ref = Reference(R, br, nn, ports, reg)
        worst = max(worst, float(ref.ratio(ref.oracle(f), f).max()))
    assert worst <= C_BOUND, worst
    assert seen == {NB_R, NB_L, NB_C, NB_VCVS, NB_SBLOCK}


def test_reference_sees_a_one_part_per_billion_change(R, golden_s2p):
    """the bound is tight enough to notice: the reference with one branch value (the 2.2 pF capacitor C2) moved by 1e-9 relative
    no longer bounds the oracle"""
    br, nn, ports, f = NETS["bias"]
    k = next(i for i, b in enumerate(br) if b[0] == NB_C and b[2][0] == 2.2e-12)
    moved = [(kind, nodes, list(p)) for kind, nodes, p in br]
    moved[k][2][0] *= 1 + 1e-9
    ref = Reference(R, moved, nn, ports, lambda: register_inductor(R, golden_s2p))
    g = f[(f > 1e9)][::8]
    assert ref.ratio(reference(R, golden_s2p, "bias").oracle(g), g).max() > C_BOUND


REVERSE = ((0, 1), (0, 2), (3, 4))        # the bias network's reverse isolation through its ideal buffers


def test_exact_zeros(R, golden_s2p):
    """Entries between the bias network's two unconnected sub-circuits: K = 0 and the oracle returns exactly 0.  Reverse isolation
    through the ideal buffer (S12, S13): exactly 0 in the reference with K = 0; the oracle's elimination cancels numerically, within
    C u of the column's largest entry (it measures ~1 u)."""
    f = BIAS_GRID
    ref = reference(R, golden_s2p, "bias")
    hi, lo, K = ref.at(f)
    O = ref.oracle(f)
    cross = np.zeros((5, 5), bool)
    cross[0:3, 3:5] = cross[3:5, 0:3] = True
    assert np.all(K[:, cross] == 0) and np.all(hi[:, cross] == 0) and np.all(O[:, cross] == 0)
    for k, j in REVERSE:
        assert np.all(hi[:, k, j] == 0) and np.all(lo[:, k, j] == 0) and np.all(K[:, k, j] == 0)
        assert np.all(np.abs(O[:, k, j]) <= C_BOUND * U * np.max(np.abs(hi[:, :, j]), axis=1))
    assert np.sum(K == 0) == len(f) * (cross.sum() + len(REVERSE))          # and nowhere else


# ---- CPU: premises of the GPU tests --------------------------------------------------------------------------------------------
DENSE_LD = (8, 16, 24, 32)
STATIC_NNZ = (64, 128, 256, 512)


def _classes(a):
    return (min(x for x in DENSE_LD if a["unknowns"] <= x), min(x for x in STATIC_NNZ if a["nnz"] <= x) if a["static"] else None)


def test_premises(Q, golden_s2p):
    """host only: the networks of the GPU tests reach every dense instantiation (LD 8 / 16 / 24 / 32, up to 32 unknowns) and the
    static plan at three non-zero classes, NNZ 512 among them; 8 ports and a single port; unequal port impedances; a delayed buffer;
    the stiff band really meets a large multiplier under the fixed order"""
    dense, nnz = set(), set()
    for name, (br, nn, ports, f) in NETS.items():
        nd = product_nodal(Q, golden_s2p, name)
        a = nd.analyze(f)
        assert a["static"], name
        ld, cls = _classes(a)
        dense.add(ld)
        nnz.add(cls)
        nd.close()
    assert dense == set(DENSE_LD) and {64, 128, 512} <= nnz
    assert NETS["mesh32"][1] + sum(b[0] == NB_VCVS for b in NETS["mesh32"][0]) == 32
    assert [len(v[2]) for v in NETS.values()] == [5, 8, 2, 1]
    assert {z for v in NETS.values() for _n, z in v[2]} == {50.0, 75.0}
    assert any(b[0] == NB_VCVS and b[2][1] > 0 for b in NETS["mesh32"][0]) and any(b[0] == NB_VCVS and b[2][1] > 0 for b in NETS["mesh14"][0])
    nd = product_nodal(Q, golden_s2p, "bias")
    # the fixed order taken at the grid's middle meets multipliers of 3.2e5 at 1 MHz, and of < 10 without the stiff band
    assert nd.analyze(BIAS_GRID)["max_multiplier"] > 1e5 and nd.analyze(BIAS_GRID[BIAS_GRID > 1e8])["max_multiplier"] < 10
    nd.close()


# ---- GPU: every kernel against the reference -----------------------------------------------------------------------------------
KERNELS = {"dense": "qo_nodal_kernel<dense>", "static": "qo_nodal_kernel<static,local>", "jit": "qo_nodal_jit_kernel"}
CROSS = np.zeros((5, 5), bool)
CROSS[0:3, 3:5] = CROSS[3:5, 0:3] = True
ZERO_TOL = [(0, 0, 0, 0, 0.0)]          # a zero-width tolerance: every Monte-Carlo sample is the nominal network


def _subgrid(f, nf):
    """nf points of the 129-point grid, ends included (the reference is cached per point)"""
    return f[np.unique(np.round(np.linspace(0, len(f) - 1, nf)).astype(int))] if nf > 1 else f[len(f) // 2:len(f) // 2 + 1]


@pytest.mark.gpu
@pytest.mark.parametrize("kern", list(KERNELS))
@pytest.mark.parametrize("name", list(NETS))
def test_gpu_values_within_condition_bound(Q, R, ctx, golden_s2p, monkeypatch, name, kern):
    """nodal_sweep and FULL_S nodal_mc_run (zero-width tolerances, three samples at an offset above 2^33) on 1, 63, 64, 65 and 129
    points -- blocks walk 64 points, FULL_S cuts the grid into 64-point chunks -- every entry within C u K of the reference"""
    f = NETS[name][3]
    ref = reference(R, golden_s2p, name)
    nd = product_nodal(Q, golden_s2p, name)
    monkeypatch.setenv("QO100NET_NODAL", kern)
    for nf in (1, 63, 64, 65, 129):
        g = _subgrid(f, nf)
        assert len(g) == nf
        S = ctx.nodal_sweep(nd, g)
        assert ctx.nodal_last_kernel() == KERNELS[kern]
        r = ref.ratio(S, g)
        assert r.max() <= C_BOUND, (nf, r.max(), np.unravel_index(np.argmax(r), r.shape))
        M = ctx.nodal_mc_run(nd, g, [], 5, 3, ZERO_TOL, sample_offset=(1 << 33) + 5, mode=Q.MODE_FULL_S)["s"]
        assert ctx.nodal_last_kernel() == KERNELS[kern] and M.shape == (3, nf) + S.shape[1:]
        for s in range(3):
            assert ref.ratio(M[s], g).max() <= C_BOUND, (nf, s)
        if name == "bias":
            assert np.all(S[:, CROSS] == 0) and np.all(M[:, :, CROSS] == 0)
    nd.close()


# (kind, row, col, f_lo, f_hi) on the bias network: through, isolation, reflection, the second sub-circuit, the stiff band
BRACKET_SPECS = [(1, 1, 0, 2.3e9, 2.5e9),       # S21 MIN
                 (2, 1, 0, 2.3e9, 2.5e9),       # S21 MAX
                 (2, 2, 0, 2.3e9, 2.5e9),       # S31 MAX (isolation)
                 (1, 1, 2, 2.3e9, 2.5e9),       # S23 MIN (isolation)
                 (2, 1, 1, 2.3e9, 2.5e9),       # S22 MAX (reflection: 2 V - 1)
                 (1, 2, 2, 3.3e9, 1e10),        # S33 MIN, the measured block extrapolated
                 (1, 4, 3, 1e6, 3e6),           # S54 MIN, second sub-circuit, stiff band
                 (2, 2, 0, 1e6, 3e6)]           # S31 MAX, stiff band


def _worst(ref, f, spec):
    """the reference's worst in-band value of a spec (dB) and the bracket half-width delta there"""
    kind, k, j, lo, hi_f = spec
    band = (f >= lo) & (f <= hi_f)
    hi, _lo, K = ref.at(f[band])
    db = 20 * np.log10(np.abs(hi[:, k, j]))
    i = int(np.argmin(db) if kind == 1 else np.argmax(db))
    d = 4 * C_BOUND * U * K[i, k, j] / np.abs(hi[i, k, j])
    return float(db[i]), max(1e-6, float(20 * np.log10(1 + d)))


@pytest.mark.gpu
@pytest.mark.parametrize("kern", list(KERNELS))
def test_gpu_verdicts_and_histogram_bins_bracket_the_reference(Q, R, ctx, golden_s2p, monkeypatch, kern):
    """Zero-width tolerances, each spec's limit at the reference's worst in-band value -+ delta (delta = the dB equivalent of
    4 C u K there, at least 1e-6 dB): every sample passes on one side and fails on the other, on MIN and MAX specs, through,
    isolation and reflection entries, both sub-circuits.  The histogram puts the worst value delta above and delta below a bin
    boundary, on a MAX spec and on a MIN spec (the kernels track -|S|^2 there and bin its magnitude)."""
    from test_ts_fused import _launch_size
    f = NETS["bias"][3]
    ref = reference(R, golden_s2p, "bias")
    nd = product_nodal(Q, golden_s2p, "bias")
    n, off = _launch_size()
    assert n % 64 and off > 1 << 33
    worst = [_worst(ref, f, s) for s in BRACKET_SPECS]
    monkeypatch.setenv("QO100NET_NODAL", kern)

    def run(sides, **hist):
        specs = [s + (v + side * d * (1 if s[0] == 2 else -1),) for s, (v, d), side in zip(BRACKET_SPECS, worst, sides)]
        r = ctx.nodal_mc_run(nd, f, specs, 9, n, ZERO_TOL, sample_offset=off, **hist)
        assert ctx.nodal_last_kernel() == KERNELS[kern] and r["n_total"] == n
        return r
    ns = len(BRACKET_SPECS)
    r = run([-1] * ns)                                    # every limit on the failing side of the worst value
    assert r["n_pass"] == 0 and list(r["fail_per_spec"]) == [n] * ns
    alt = [(-1) ** s for s in range(ns)]
    r = run(alt)
    assert list(r["fail_per_spec"]) == [0 if a > 0 else n for a in alt]
    for hs in (2, 0):                                     # S31 MAX, S21 MIN
        v, d = worst[hs]
        for above, b in ((1, 5), (-1, 4)):
            lo = v - above * d - 5 * 0.05
            r = run([1] * ns, hist_bins=10, hist_spec=hs, hist_lo=lo, hist_hi=lo + 0.5)
            assert r["n_pass"] == n and list(r["fail_per_spec"]) == [0] * ns
            assert r["hist"][b] == n, (hs, above, list(r["hist"]))
    nd.close()
