"""ctypes binding of the CPU oracle (oracle/_build/libqo100ref.so).

TEST INFRASTRUCTURE ONLY -- imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package never
imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_build", "libqo100ref.so")

# element kinds (same numeric values as include/qo100net.h)
SER_R, SHUNT_R, SER_L, SHUNT_L, SER_C, SHUNT_C = 1, 2, 3, 4, 5, 6
SER_LC_SER, SER_LC_PAR, SHUNT_LC_SER, SHUNT_LC_PAR = 7, 8, 9, 10
TLINE, CPL_THRU, SUBST, MLIN, MCORN, MTEE, MOPEN = 11, 12, 13, 14, 15, 16, 17
SPEC_S21_MIN_DB, SPEC_S21_MAX_DB, SPEC_S11_MAX_DB, SPEC_GD_MAX = 1, 2, 3, 4
DIST_UNIFORM, DIST_GAUSS3S = 0, 1
TOL_REL, TOL_ABS = 0, 1


class Elem(C.Structure):
    _fields_ = [("kind", C.c_int32), ("flags", C.c_int32), ("p", C.c_double * 6)]


class Spec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("pad", C.c_int32), ("f_lo", C.c_double), ("f_hi", C.c_double),
                ("limit", C.c_double)]


class Tol(C.Structure):
    _fields_ = [("elem", C.c_int32), ("param", C.c_int32), ("var", C.c_int32), ("mode", C.c_int32),
                ("tol", C.c_double)]


class Branch(C.Structure):
    _fields_ = [("kind", C.c_int32), ("node", C.c_int32 * 4), ("p", C.c_double * 4)]


class NSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("row", C.c_int32), ("col", C.c_int32), ("pad", C.c_int32),
                ("f_lo", C.c_double), ("f_hi", C.c_double), ("limit", C.c_double)]


class McCfg(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("sample_offset", C.c_uint64), ("n_samples", C.c_uint64),
                ("dist", C.c_int32), ("n_tol", C.c_int32), ("tol", C.POINTER(Tol)),
                ("hist_bins", C.c_int32), ("hist_spec", C.c_int32), ("hist_lo", C.c_double),
                ("hist_hi", C.c_double)]


def build(force=False):
    """Compile the oracle with the committed Makefile (building the checker is not using it)."""
    if force or not os.path.exists(_LIB) or any(
            os.path.getmtime(os.path.join(_HERE, s)) > os.path.getmtime(_LIB)
            for s in ("qo100ref.c", "qo100ref_nodal.c", "qo100ref.h", "Makefile")):
        env = dict(os.environ)
        env.pop("CC", None)
        subprocess.run(["make", "-C", _HERE], check=True, capture_output=True, env=env)
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        dp, u64p = C.POINTER(C.c_double), C.POINTER(C.c_uint64)
        L.ref_philox4x32_10.argtypes = [C.POINTER(C.c_uint32)] * 3
        L.ref_uniform01.restype = C.c_double
        L.ref_uniform01.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32]
        L.ref_variate.restype = C.c_double
        L.ref_variate.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int]
        L.ref_perturb_factor.restype = C.c_double
        L.ref_perturb_factor.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_double]
        L.ref_perturb_factors.restype = None
        L.ref_perturb_factors.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_double, dp]
        L.ref_norminv.restype = C.c_double
        L.ref_norminv.argtypes = [C.c_double]
        L.ref_log_det.restype = C.c_double
        L.ref_log_det.argtypes = [C.c_double]
        L.ref_grid_lin.argtypes = [C.c_double, C.c_double, C.c_int, dp]
        L.ref_grid_log.argtypes = [C.c_double, C.c_double, C.c_int, dp]
        L.ref_cheby_g.argtypes = [C.c_int, C.c_double, dp]
        L.ref_butter_g.argtypes = [C.c_int, dp]
        L.ref_ladder_lpf.argtypes = [dp, C.c_int, C.c_double, C.c_double, C.c_int, C.POINTER(Elem)]
        L.ref_add_parasitics.argtypes = [C.POINTER(Elem), C.c_int] + [C.c_double] * 5
        L.ref_sweep.argtypes = [C.POINTER(Elem), C.c_int, C.c_double, C.c_double, dp, C.c_int, dp, dp, dp, dp, dp]
        L.ref_perturb.argtypes = [C.POINTER(Elem), C.c_int, C.POINTER(McCfg), C.c_uint64, C.POINTER(Elem)]
        L.ref_mc_run.argtypes = [C.POINTER(Elem), C.c_int, C.c_double, C.c_double, dp, C.c_int,
                                 C.POINTER(Spec), C.c_int, C.POINTER(McCfg), u64p, dp, C.c_int]
        L.ref_ms_quasi.argtypes = [C.c_double] * 4 + [dp] * 3
        L.ref_ms_disp.argtypes = [C.c_double] * 6 + [dp] * 2
        L.ref_cpl_analyze.argtypes = [C.c_double] * 8 + [dp] * 4
        L.ref_sblock_register.argtypes = [C.c_int, dp, dp, C.c_int, C.c_double]
        L.ref_sblock_clear.argtypes = []
        L.ref_sblock_s.argtypes = [C.c_int, C.c_double, C.c_int, dp]
        ip = C.POINTER(C.c_int)
        L.ref_nodal_sweep.argtypes = [C.POINTER(Branch), C.c_int, C.c_int, ip, dp, C.c_int, dp, C.c_int, dp]
        L.ref_nodal_mc_run.argtypes = [C.POINTER(Branch), C.c_int, C.c_int, ip, dp, C.c_int, dp, C.c_int,
                                       C.POINTER(NSpec), C.c_int, C.POINTER(McCfg), u64p, dp, C.c_int]
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def make_elems(items):
    """items: iterable of (kind, [p0..]) -> ctypes array of Elem."""
    items = list(items)
    arr = (Elem * len(items))()
    for i, (kind, p) in enumerate(items):
        arr[i].kind = int(kind)
        for k, v in enumerate(p):
            arr[i].p[k] = float(v)
    return arr


NB_R, NB_L, NB_C, NB_VCVS, NB_SBLOCK = 1, 2, 3, 4, 5


def make_branches(items):
    """items: (kind, [nodes], [params]) -> ctypes array of Branch."""
    items = list(items)
    arr = (Branch * len(items))()
    for i, (kind, nodes, p) in enumerate(items):
        arr[i].kind = int(kind)
        for k, v in enumerate(nodes):
            arr[i].node[k] = int(v)
        for k, v in enumerate(p):
            arr[i].p[k] = float(v)
    return arr


def nodal_sweep(branches, n_nodes, ports, f):
    """ports: [(node, z0)] -> S[nf, np, np] with S[:, k, j] = b_k / a_j."""
    br = branches if isinstance(branches, C.Array) else make_branches(branches)
    f = np.ascontiguousarray(f, dtype=np.float64)
    npn = len(ports)
    pn = (C.c_int * npn)(*[int(p[0]) for p in ports])
    pz = np.array([float(p[1]) for p in ports])
    out = np.empty((len(f), npn, npn), dtype=np.complex128)
    rc = lib().ref_nodal_sweep(br, len(br), int(n_nodes), pn, _dp(pz), npn, _dp(f), len(f), out.ctypes.data_as(C.POINTER(C.c_double)))
    if rc:
        raise RuntimeError("ref_nodal_sweep failed: %d" % rc)
    return out


def nodal_mc_run(branches, n_nodes, ports, f, specs, cfg, full_s=False, nthreads=1):
    """specs: [(kind, row, col, f_lo, f_hi, limit_db)] on |S[row][col]|."""
    br = branches if isinstance(branches, C.Array) else make_branches(branches)
    f = np.ascontiguousarray(f, dtype=np.float64)
    npn = len(ports)
    pn = (C.c_int * npn)(*[int(p[0]) for p in ports])
    pz = np.array([float(p[1]) for p in ports])
    sp = (NSpec * max(1, len(specs)))()
    for i, s in enumerate(specs):
        sp[i].kind, sp[i].row, sp[i].col, sp[i].f_lo, sp[i].f_hi, sp[i].limit = int(s[0]), int(s[1]), int(s[2]), float(s[3]), float(s[4]), float(s[5])
    hb = max(0, cfg.hist_bins)
    cnt = np.zeros(2 + len(specs) + hb, dtype=np.uint64)
    full = np.empty((cfg.n_samples, len(f), npn, npn), dtype=np.complex128) if full_s else None
    rc = lib().ref_nodal_mc_run(br, len(br), int(n_nodes), pn, _dp(pz), npn, _dp(f), len(f), sp, len(specs), C.byref(cfg),
                                cnt.ctypes.data_as(C.POINTER(C.c_uint64)),
                                full.ctypes.data_as(C.POINTER(C.c_double)) if full is not None else None, nthreads)
    if rc:
        raise RuntimeError("ref_nodal_mc_run failed: %d" % rc)
    out = dict(n_pass=int(cnt[0]), n_total=int(cnt[1]), fail_per_spec=cnt[2:2 + len(specs)].copy(), hist=cnt[2 + len(specs):].copy())
    if full is not None:
        out["s"] = full
    return out


def sblock_register(idx, f, s11, s21, s12, s22, z0=50.0):
    """Hand a measured two-port to the oracle under block index idx (REF_SBLOCK elements refer to it by p0)."""
    f = np.ascontiguousarray(f, dtype=np.float64)
    s = np.empty((len(f), 8))
    for j, a in enumerate((s11, s21, s12, s22)):
        a = np.asarray(a, dtype=np.complex128)
        s[:, 2 * j], s[:, 2 * j + 1] = a.real, a.imag
    rc = lib().ref_sblock_register(int(idx), _dp(f), _dp(np.ascontiguousarray(s)), len(f), float(z0))
    if rc:
        raise RuntimeError("ref_sblock_register failed: %d" % rc)


def sblock_clear():
    lib().ref_sblock_clear()


def sblock_s(idx, f, polar=True):
    """The oracle's interpolated S of measured block idx at one frequency -> (s11, s21, s12, s22), complex."""
    s = np.empty(8)
    rc = lib().ref_sblock_s(int(idx), float(f), int(bool(polar)), _dp(s))
    if rc:
        raise RuntimeError("ref_sblock_s failed: %d" % rc)
    return tuple(complex(s[2 * j], s[2 * j + 1]) for j in range(4))


def elems_to_list(arr, n=None):
    n = len(arr) if n is None else n
    return [(arr[i].kind, [arr[i].p[k] for k in range(6)]) for i in range(n)]


def philox(ctr, key):
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    o = (C.c_uint32 * 4)()
    lib().ref_philox4x32_10(c, k, o)
    return list(o)


def grid_lin(f0, f1, n):
    f = np.empty(n)
    lib().ref_grid_lin(f0, f1, n, _dp(f))
    return f


def grid_log(f0, f1, n):
    f = np.empty(n)
    lib().ref_grid_log(f0, f1, n, _dp(f))
    return f


def cheby_g(n, ripple_db):
    g = np.empty(n)
    assert lib().ref_cheby_g(n, ripple_db, _dp(g)) == 0
    return g


def butter_g(n):
    g = np.empty(n)
    assert lib().ref_butter_g(n, _dp(g)) == 0
    return g


def ladder_lpf(g, fc, z0, series_first=True, parasitics=None):
    """parasitics = (Q_L, srfL_mult, esr_C, srfC_mult) or None."""
    g = np.ascontiguousarray(g, dtype=np.float64)
    arr = (Elem * len(g))()
    lib().ref_ladder_lpf(_dp(g), len(g), fc, z0, int(series_first), arr)
    if parasitics is not None:
        lib().ref_add_parasitics(arr, len(g), fc, *[float(x) for x in parasitics])
    return arr


def sweep(elems, rs, rl, f, gd=False):
    f = np.ascontiguousarray(f, dtype=np.float64)
    nf = len(f)
    out = [np.empty(2 * nf) for _ in range(4)]
    g = np.empty(nf) if gd else None
    rc = lib().ref_sweep(elems, len(elems), rs, rl, _dp(f), nf, *[_dp(o) for o in out], _dp(g))
    if rc:
        raise RuntimeError("ref_sweep failed: %d" % rc)
    s11, s21, s12, s22 = [o.view(np.complex128) for o in out]
    return (s11, s21, s12, s22, g) if gd else (s11, s21, s12, s22)


def make_tols(tols):
    arr = (Tol * max(1, len(tols)))()
    for i, t in enumerate(tols):
        arr[i].elem, arr[i].param, arr[i].var, arr[i].mode, arr[i].tol = int(t[0]), int(t[1]), int(t[2]), int(t[3]), float(t[4])
    return arr


def make_specs(specs):
    arr = (Spec * max(1, len(specs)))()
    for i, s in enumerate(specs):
        arr[i].kind, arr[i].f_lo, arr[i].f_hi, arr[i].limit = int(s[0]), float(s[1]), float(s[2]), float(s[3])
    return arr


def mc_cfg(seed, n_samples, tols, sample_offset=0, dist=DIST_UNIFORM, hist_bins=0, hist_spec=0, hist_lo=0.0,
           hist_hi=1.0):
    cfg = McCfg()
    cfg._tols = make_tols(tols)
    cfg.seed, cfg.sample_offset, cfg.n_samples = seed, sample_offset, n_samples
    cfg.dist, cfg.n_tol, cfg.tol = dist, len(tols), cfg._tols
    cfg.hist_bins, cfg.hist_spec, cfg.hist_lo, cfg.hist_hi = hist_bins, hist_spec, hist_lo, hist_hi
    return cfg


def perturb_factors(seed, sample_offset, n_samples, n_var, dist, tol):
    """The oracle's perturbation stream, [n_samples, n_var] factors 1 + tol * x."""
    out = np.empty((n_samples, n_var))
    lib().ref_perturb_factors(seed, sample_offset, n_samples, n_var, dist, tol, _dp(out))
    return out


def perturb(elems, cfg, sample):
    out = (Elem * len(elems))()
    lib().ref_perturb(elems, len(elems), C.byref(cfg), sample, out)
    return out


def mc_run(elems, rs, rl, f, specs, cfg, full_s=False, nthreads=1):
    """-> dict(n_pass, n_total, fail_per_spec, hist[, s (4, n, nf) complex])."""
    f = np.ascontiguousarray(f, dtype=np.float64)
    nf, nspec = len(f), len(specs)
    sp = make_specs(specs)
    nb = max(0, cfg.hist_bins)
    cnt = np.zeros(2 + nspec + nb, dtype=np.uint64)
    fs = np.empty(4 * cfg.n_samples * nf * 2) if full_s else None
    rc = lib().ref_mc_run(elems, len(elems), rs, rl, _dp(f), nf, sp, nspec, C.byref(cfg),
                          cnt.ctypes.data_as(C.POINTER(C.c_uint64)), _dp(fs), nthreads)
    if rc:
        raise RuntimeError("ref_mc_run failed: %d" % rc)
    out = dict(n_pass=int(cnt[0]), n_total=int(cnt[1]), fail_per_spec=cnt[2:2 + nspec].copy(),
               hist=cnt[2 + nspec:].copy())
    if full_s:
        out["s"] = fs.view(np.complex128).reshape(4, cfg.n_samples, nf)
    return out


def max_threads():
    lib().ref_max_threads.restype = C.c_int
    return lib().ref_max_threads()


def cpl_analyze(w, s, h, t, er, ht, f, length):
    o = [C.c_double() for _ in range(4)]
    lib().ref_cpl_analyze(w, s, h, t, er, ht, f, length, *[C.byref(x) for x in o])
    return tuple(x.value for x in o)


def ms_quasi(W, h, t, er):
    o = [C.c_double() for _ in range(3)]
    lib().ref_ms_quasi(W, h, t, er, *[C.byref(x) for x in o])
    return tuple(x.value for x in o)
