"""qo100net -- thin ctypes mirror of the libqo100net C-ABI (include/qo100net.h).

The library is the product; this module only marshals arguments.  It never
evaluates a network itself and there is no CPU fallback: every compute call
goes to the CUDA kernels and raises QoError(QO_ERR_NO_DEVICE) without a GPU.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.abspath(os.path.join(_PKG, "..", ".."))        # qo-100-tools_b200/
CSRC = os.path.join(_ROOT, "csrc")
LIB_PATH = os.path.join(_ROOT, "lib", "libqo100net.so")

# enums (include/qo100net.h)
OK, ERR_ARG, ERR_IO, ERR_PARSE, ERR_UNSUPPORTED, ERR_NOMEM, ERR_NO_DEVICE, ERR_CUDA, ERR_NCCL, ERR_RANGE = \
    0, -1, -2, -3, -4, -5, -6, -7, -8, -9
SER_R, SHUNT_R, SER_L, SHUNT_L, SER_C, SHUNT_C = 1, 2, 3, 4, 5, 6
SER_LC_SER, SER_LC_PAR, SHUNT_LC_SER, SHUNT_LC_PAR = 7, 8, 9, 10
TLINE, CPL_THRU, SUBST, MLIN, MCORN, MTEE, MOPEN, SBLOCK, CPL_MS = 11, 12, 13, 14, 15, 16, 17, 18, 19
SPEC_S21_MIN_DB, SPEC_S21_MAX_DB, SPEC_S11_MAX_DB, SPEC_GD_MAX = 1, 2, 3, 4
DIST_UNIFORM, DIST_GAUSS3S = 0, 1
TOL_REL, TOL_ABS = 0, 1
MODE_REDUCE_ONLY, MODE_FULL_S = 0, 1


class QoError(RuntimeError):
    def __init__(self, status, detail=""):
        self.status = status
        super().__init__("qo100net error %d (%s)%s" % (status, strerror(status), ": " + detail if detail else ""))


class Elem(C.Structure):
    _fields_ = [("kind", C.c_int32), ("flags", C.c_int32), ("p", C.c_double * 6)]


class Spec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("pad", C.c_int32), ("f_lo", C.c_double), ("f_hi", C.c_double),
                ("limit", C.c_double)]


class Tol(C.Structure):
    _fields_ = [("elem", C.c_int32), ("param", C.c_int32), ("var", C.c_int32), ("mode", C.c_int32),
                ("tol", C.c_double)]


class McCfg(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("sample_offset", C.c_uint64), ("n_samples", C.c_uint64),
                ("dist", C.c_int32), ("n_tol", C.c_int32), ("tol", C.POINTER(Tol)),
                ("mode", C.c_int32), ("precision", C.c_int32),
                ("hist_bins", C.c_int32), ("hist_spec", C.c_int32), ("hist_lo", C.c_double), ("hist_hi", C.c_double)]


class Branch(C.Structure):
    _fields_ = [("kind", C.c_int32), ("node", C.c_int32 * 4), ("p", C.c_double * 4)]


class NSpec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("row", C.c_int32), ("col", C.c_int32), ("pad", C.c_int32),
                ("f_lo", C.c_double), ("f_hi", C.c_double), ("limit", C.c_double)]


NB_R, NB_L, NB_C, NB_VCVS, NB_SBLOCK = 1, 2, 3, 4, 5


class McResult(C.Structure):
    _fields_ = [("n_pass", C.c_uint64), ("n_total", C.c_uint64), ("fail_per_spec", C.POINTER(C.c_uint64)),
                ("hist", C.POINTER(C.c_uint64)), ("seconds", C.c_double), ("evals_per_s", C.c_double),
                ("flops_per_eval", C.c_double)]


def build(verbose=False):
    """Compile libqo100net.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    env = dict(os.environ)
    env.pop("CC", None)
    r = subprocess.run(["make", "-j", "8", "-C", CSRC], capture_output=True, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError("building libqo100net.so failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stdout)
    return LIB_PATH


_lib = None
EXPORTS = [
    "qo_net_load_rftools_svg", "qo_net_load_qucs_sch", "qo_qucs_sch_sweep", "qo_cpl_load_trc", "qo_cpl_analyze", "qo_cpl_synthesize",
    "qo_net_from_elements", "qo_net_cheby_lpf", "qo_net_butter_lpf", "qo_net_add_parasitics", "qo_net_concat",
    "qo_net_num_elements", "qo_net_get_elements", "qo_net_terminations", "qo_net_title", "qo_net_free",
    "qo_grid_lin", "qo_grid_log", "qo_ctx_create", "qo_ctx_create_on_device", "qo_ctx_set_stream",
    "qo_ctx_num_devices", "qo_ctx_destroy", "qo_sweep", "qo_mc_run", "qo_plan_create", "qo_plan_num_counters",
    "qo_plan_reset", "qo_plan_launch", "qo_plan_read", "qo_plan_flops_per_eval", "qo_plan_launches",
    "qo_plan_kernel_name", "qo_plan_tf_info", "qo_plan_h2d_bytes", "qo_plan_analyze", "qo_chain_jit_analyze",
    "qo_s2p_load", "qo_s2p_from_arrays", "qo_s2p_num_points", "qo_s2p_z0", "qo_s2p_get", "qo_s2p_interp",
    "qo_s2p_fit_inductor", "qo_s2p_free", "qo_net_from_sblock",
    "qo_nodal_create", "qo_nodal_add_branch", "qo_nodal_add_port", "qo_nodal_add_sblock", "qo_nodal_load_qucs_sch",
    "qo_nodal_num_nodes", "qo_nodal_num_ports", "qo_nodal_num_branches", "qo_nodal_get_branches", "qo_nodal_get_ports",
    "qo_nodal_free", "qo_nodal_sweep", "qo_nodal_mc_run", "qo_nodal_last_kernel", "qo_nodal_analyze", "qo_nodal_jit_analyze", "qo_nodal_last_compile_seconds",
    "qo_dat_create", "qo_dat_read", "qo_dat_write", "qo_dat_add_indep", "qo_dat_add_dep", "qo_dat_count", "qo_dat_info",
    "qo_dat_get", "qo_dat_from_sweep", "qo_dat_free",
    "qo_plan_destroy", "qo_philox4x32_10", "qo_variate", "qo_perturb_factor", "qo_device_perturb_factors",
    "qo_device_rcp", "qo_device_mslog", "qo_measure_dfma_peak", "qo_strerror", "qo_last_error", "qo_version",
]


def lib():
    """Load the in-tree shared library (fails loudly if it has not been built)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libqo100net.so is missing at %s -- run __graft_entry__.build() (there is no fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, dp, ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)
    u64p = C.POINTER(C.c_uint64)
    sig = {
        "qo_net_load_rftools_svg": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "qo_net_load_qucs_sch": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "qo_qucs_sch_sweep": (C.c_int, [C.c_char_p, ip, dp, dp, ip]),
        "qo_cpl_load_trc": (C.c_int, [C.c_char_p, dp, dp, dp, dp, dp]),
        "qo_cpl_analyze": (C.c_int, [C.c_double] * 8 + [dp] * 4),
        "qo_cpl_synthesize": (C.c_int, [C.c_double] * 8 + [dp] * 3),
        "qo_net_from_elements": (C.c_int, [C.POINTER(Elem), C.c_int, C.c_double, C.c_double, C.POINTER(vp)]),
        "qo_net_cheby_lpf": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_double, C.c_int, C.POINTER(vp)]),
        "qo_net_butter_lpf": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_int, C.POINTER(vp)]),
        "qo_net_add_parasitics": (C.c_int, [vp] + [C.c_double] * 5),
        "qo_net_concat": (C.c_int, [vp, vp, C.POINTER(vp)]),
        "qo_net_num_elements": (C.c_int, [vp]),
        "qo_net_get_elements": (C.c_int, [vp, C.POINTER(Elem), C.c_int]),
        "qo_net_terminations": (C.c_int, [vp, dp, dp]),
        "qo_net_title": (C.c_char_p, [vp]),
        "qo_net_free": (None, [vp]),
        "qo_grid_lin": (C.c_int, [C.c_double, C.c_double, C.c_int, dp]),
        "qo_grid_log": (C.c_int, [C.c_double, C.c_double, C.c_int, dp]),
        "qo_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "qo_ctx_create_on_device": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "qo_ctx_set_stream": (C.c_int, [vp, vp]),
        "qo_ctx_num_devices": (C.c_int, [vp]),
        "qo_ctx_destroy": (None, [vp]),
        "qo_sweep": (C.c_int, [vp, vp, dp, C.c_int, C.c_int, vp, vp, vp, vp, dp]),
        "qo_mc_run": (C.c_int, [vp, vp, dp, C.c_int, C.POINTER(Spec), C.c_int, C.POINTER(McCfg), C.POINTER(McResult), vp]),
        "qo_plan_create": (C.c_int, [vp, vp, dp, C.c_int, C.POINTER(Spec), C.c_int, C.POINTER(McCfg), C.POINTER(vp)]),
        "qo_plan_num_counters": (C.c_int, [vp]),
        "qo_plan_reset": (C.c_int, [vp]),
        "qo_plan_launch": (C.c_int, [vp, C.c_uint64, C.c_uint64, vp, vp]),
        "qo_plan_read": (C.c_int, [vp, C.POINTER(McResult)]),
        "qo_plan_flops_per_eval": (C.c_double, [vp]),
        "qo_plan_launches": (C.c_int, [vp]),
        "qo_plan_kernel_name": (C.c_char_p, [vp]),
        "qo_plan_tf_info": (C.c_char_p, [vp, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_uint), C.POINTER(C.c_double)]),
        "qo_plan_h2d_bytes": (C.c_uint64, [vp]),
        "qo_chain_jit_analyze": (C.c_int, [vp, C.POINTER(C.c_double), C.c_int, vp, C.c_int, vp, C.POINTER(C.c_int)]),
        "qo_plan_analyze": (C.c_char_p, [vp, C.POINTER(C.c_double), C.c_int, vp, C.c_int, vp, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_uint), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "qo_s2p_load": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "qo_s2p_from_arrays": (C.c_int, [dp, C.c_int, vp, vp, vp, vp, C.c_double, C.POINTER(vp)]),
        "qo_s2p_num_points": (C.c_int, [vp]),
        "qo_s2p_z0": (C.c_double, [vp]),
        "qo_s2p_get": (C.c_int, [vp, dp, vp, vp, vp, vp, C.c_int]),
        "qo_s2p_interp": (C.c_int, [vp, dp, C.c_int, C.c_int, vp, vp, vp, vp]),
        "qo_s2p_fit_inductor": (C.c_int, [vp, C.c_double, C.c_double, dp, dp, dp, dp, dp, dp]),
        "qo_s2p_free": (None, [vp]),
        "qo_net_from_sblock": (C.c_int, [vp, C.c_int, C.c_double, C.c_double, C.POINTER(vp)]),
        "qo_nodal_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "qo_nodal_add_branch": (C.c_int, [vp, C.POINTER(Branch)]),
        "qo_nodal_add_port": (C.c_int, [vp, C.c_int, C.c_double]),
        "qo_nodal_add_sblock": (C.c_int, [vp, vp, ip]),
        "qo_nodal_load_qucs_sch": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "qo_nodal_num_nodes": (C.c_int, [vp]),
        "qo_nodal_num_ports": (C.c_int, [vp]),
        "qo_nodal_num_branches": (C.c_int, [vp]),
        "qo_nodal_get_branches": (C.c_int, [vp, C.POINTER(Branch), C.c_int]),
        "qo_nodal_get_ports": (C.c_int, [vp, ip, dp, C.c_int]),
        "qo_nodal_free": (None, [vp]),
        "qo_nodal_sweep": (C.c_int, [vp, vp, dp, C.c_int, vp]),
        "qo_nodal_last_kernel": (C.c_char_p, []),
        "qo_nodal_analyze": (C.c_int, [vp, dp, C.c_int, C.POINTER(McCfg), ip, dp]),
        "qo_nodal_last_compile_seconds": (C.c_double, []),
        "qo_nodal_jit_analyze": (C.c_int, [vp, dp, C.c_int, C.POINTER(NSpec), C.c_int, C.POINTER(McCfg), ip]),
        "qo_nodal_mc_run": (C.c_int, [vp, vp, dp, C.c_int, C.POINTER(NSpec), C.c_int, C.POINTER(McCfg), C.POINTER(McResult), vp]),
        "qo_dat_create": (C.c_int, [C.POINTER(vp)]),
        "qo_dat_read": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "qo_dat_write": (C.c_int, [vp, C.c_char_p]),
        "qo_dat_add_indep": (C.c_int, [vp, C.c_char_p, dp, C.c_int]),
        "qo_dat_add_dep": (C.c_int, [vp, C.c_char_p, C.c_char_p, dp, dp, C.c_int]),
        "qo_dat_count": (C.c_int, [vp]),
        "qo_dat_info": (C.c_int, [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), ip, ip]),
        "qo_dat_get": (C.c_int, [vp, C.c_char_p, dp, dp, C.c_int]),
        "qo_dat_from_sweep": (C.c_int, [dp, C.c_int, vp, vp, vp, vp, C.POINTER(vp)]),
        "qo_dat_free": (None, [vp]),
        "qo_plan_destroy": (None, [vp]),
        "qo_philox4x32_10": (None, [C.POINTER(C.c_uint32)] * 3),
        "qo_variate": (C.c_double, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int]),
        "qo_perturb_factor": (C.c_double, [C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_double]),
        "qo_device_perturb_factors": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_double, dp]),
        "qo_measure_dfma_peak": (C.c_int, [vp, dp]),
        "qo_device_rcp": (C.c_int, [vp, dp, C.c_size_t, dp]),
        "qo_device_mslog": (C.c_int, [vp, dp, C.c_size_t, dp]),
        "qo_strerror": (C.c_char_p, [C.c_int]),
        "qo_last_error": (C.c_char_p, []),
        "qo_version": (C.c_char_p, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def strerror(status):
    try:
        return lib().qo_strerror(status).decode()
    except Exception:  # library not built yet
        return "?"


def _check(rc):
    if rc < 0:
        raise QoError(rc, lib().qo_last_error().decode())
    return rc


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


class Net:
    """Immutable element list + terminations (qo_net*)."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle) if not isinstance(handle, C.c_void_p) else handle

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.qo_net_free(self._h)
            self._h = None

    @staticmethod
    def _out():
        return C.c_void_p()

    @classmethod
    def from_rftools_svg(cls, path):
        h = cls._out()
        _check(lib().qo_net_load_rftools_svg(os.fsencode(path), C.byref(h)))
        return cls(h)

    @classmethod
    def from_qucs_sch(cls, path):
        h = cls._out()
        _check(lib().qo_net_load_qucs_sch(os.fsencode(path), C.byref(h)))
        return cls(h)

    @classmethod
    def from_elements(cls, items, rs=50.0, rl=50.0):
        """items: iterable of (kind, [p0..p5])."""
        items = list(items)
        arr = (Elem * max(1, len(items)))()
        for i, (kind, p) in enumerate(items):
            arr[i].kind = int(kind)
            for k, v in enumerate(p):
                arr[i].p[k] = float(v)
        h = cls._out()
        _check(lib().qo_net_from_elements(arr, len(items), rs, rl, C.byref(h)))
        return cls(h)

    @classmethod
    def cheby_lpf(cls, order, ripple_db, fc, z0=50.0, series_first=True):
        h = cls._out()
        _check(lib().qo_net_cheby_lpf(order, ripple_db, fc, z0, int(series_first), C.byref(h)))
        return cls(h)

    @classmethod
    def butter_lpf(cls, order, fc, z0=50.0, series_first=True):
        h = cls._out()
        _check(lib().qo_net_butter_lpf(order, fc, z0, int(series_first), C.byref(h)))
        return cls(h)

    def add_parasitics(self, fc, q_l=60.0, srf_l_mult=30.0, esr_c=0.1, srf_c_mult=50.0):
        _check(lib().qo_net_add_parasitics(self._h, fc, q_l, srf_l_mult, esr_c, srf_c_mult))
        return self

    def concat(self, other):
        h = self._out()
        _check(lib().qo_net_concat(self._h, other._h, C.byref(h)))
        return Net(h)

    def __len__(self):
        return _check(lib().qo_net_num_elements(self._h))

    @property
    def elements(self):
        n = len(self)
        arr = (Elem * n)()
        _check(lib().qo_net_get_elements(self._h, arr, n))
        return [(arr[i].kind, [arr[i].p[k] for k in range(6)]) for i in range(n)]

    @property
    def terminations(self):
        rs, rl = C.c_double(), C.c_double()
        _check(lib().qo_net_terminations(self._h, C.byref(rs), C.byref(rl)))
        return rs.value, rl.value

    @property
    def title(self):
        return lib().qo_net_title(self._h).decode("utf-8", "replace")


def qucs_sch_sweep(path):
    t, n, f0, f1 = C.c_int(), C.c_int(), C.c_double(), C.c_double()
    _check(lib().qo_qucs_sch_sweep(os.fsencode(path), C.byref(t), C.byref(f0), C.byref(f1), C.byref(n)))
    return ("log" if t.value else "lin"), f0.value, f1.value, n.value


def load_trc(path):
    z0e, z0o, ang, f0 = C.c_double(), C.c_double(), C.c_double(), C.c_double()
    phys = (C.c_double * 8)()
    _check(lib().qo_cpl_load_trc(os.fsencode(path), C.byref(z0e), C.byref(z0o), C.byref(ang), C.byref(f0), phys))
    keys = ["er", "h", "ht", "t", "w", "s", "l", "tand"]
    return dict(z0e=z0e.value, z0o=z0o.value, ang=ang.value, f0=f0.value, **{k: phys[i] for i, k in enumerate(keys)})


class Nodal:
    """A general N-port netlist for the nodal solver (qo_nodal*): nodes 1..n (0 = ground)."""

    def __init__(self, n_nodes=None, handle=None):
        self._h = handle or C.c_void_p()
        if handle is None:
            _check(lib().qo_nodal_create(int(n_nodes), C.byref(self._h)))

    @classmethod
    def from_qucs_sch(cls, path):
        h = C.c_void_p()
        _check(lib().qo_nodal_load_qucs_sch(os.fsencode(path), C.byref(h)))
        return cls(handle=h)

    def add_branch(self, kind, nodes, params):
        b = Branch()
        b.kind = int(kind)
        for k, v in enumerate(nodes):
            b.node[k] = int(v)
        for k, v in enumerate(params):
            b.p[k] = float(v)
        _check(lib().qo_nodal_add_branch(self._h, C.byref(b)))

    def add_port(self, node, z0=50.0):
        return _check(lib().qo_nodal_add_port(self._h, int(node), float(z0)))

    def add_sblock(self, blk):
        idx = C.c_int()
        _check(lib().qo_nodal_add_sblock(self._h, blk._h, C.byref(idx)))
        return idx.value

    @property
    def n_nodes(self):
        return _check(lib().qo_nodal_num_nodes(self._h))

    @property
    def ports(self):
        n = _check(lib().qo_nodal_num_ports(self._h))
        node, z0 = (C.c_int * max(1, n))(), np.empty(max(1, n))
        lib().qo_nodal_get_ports(self._h, node, _dp(z0), n)
        return [(node[k], float(z0[k])) for k in range(n)]

    @property
    def branches(self):
        n = _check(lib().qo_nodal_num_branches(self._h))
        arr = (Branch * max(1, n))()
        lib().qo_nodal_get_branches(self._h, arr, n)
        return [(arr[i].kind, [arr[i].node[k] for k in range(4)], [arr[i].p[k] for k in range(4)]) for i in range(n)]

    def analyze(self, f, tols=()):
        """Host-only (qo_nodal_analyze): does the static factorisation plan hold for this netlist on this grid, with these
        tolerances?  -> dict(static, unknowns, nnz, program_words, max_multiplier)."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        cfg = _cfg(0, 0, list(tols), 0, DIST_UNIFORM, MODE_FULL_S, 64, 0, 0, 0.0, 1.0)
        info = (C.c_int * 4)()
        mm = C.c_double(0.0)
        _check(lib().qo_nodal_analyze(self._h, _dp(f), len(f), C.byref(cfg), info, C.byref(mm)))
        return dict(static=bool(info[0]), unknowns=info[1], nnz=info[2], program_words=info[3], max_multiplier=mm.value)

    def jit_analyze(self, f, specs=(), tols=(), mode=MODE_REDUCE_ONLY):
        """Host-only (qo_nodal_jit_analyze): generate this job's compiled kernel and report what ptxas made of it
        -> dict(compiled, registers, stack_bytes, spill_bytes, fms, reciprocals, error)."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        cfg = _cfg(0, 0, list(tols), 0, DIST_UNIFORM, mode, 64, 0, 0, 0.0, 1.0)
        sp = (NSpec * max(1, len(specs)))()
        for i, s in enumerate(specs):
            sp[i].kind, sp[i].row, sp[i].col, sp[i].f_lo, sp[i].f_hi, sp[i].limit = int(s[0]), int(s[1]), int(s[2]), float(s[3]), float(s[4]), float(s[5])
        info = (C.c_int * 6)()
        _check(lib().qo_nodal_jit_analyze(self._h, _dp(f), len(f), sp, len(specs), C.byref(cfg), info))
        return dict(compiled=bool(info[0]), registers=info[1], stack_bytes=info[2], spill_bytes=info[3], fms=info[4],
                    reciprocals=info[5], error=None if info[0] else lib().qo_last_error().decode())

    def close(self):
        if self._h:
            lib().qo_nodal_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SBlock:
    """A measured two-port (Touchstone v1 .s2p; qo_s2p*)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def load(cls, path):
        h = C.c_void_p()
        _check(lib().qo_s2p_load(os.fsencode(path), C.byref(h)))
        return cls(h)

    @classmethod
    def from_arrays(cls, f, s11, s21, s12, s22, z0=50.0):
        f = np.ascontiguousarray(f, dtype=np.float64)
        arrs = [np.ascontiguousarray(a, dtype=np.complex128) for a in (s11, s21, s12, s22)]
        h = C.c_void_p()
        _check(lib().qo_s2p_from_arrays(_dp(f), len(f), *[a.ctypes.data_as(C.c_void_p) for a in arrs], z0, C.byref(h)))
        return cls(h)

    @property
    def z0(self):
        return lib().qo_s2p_z0(self._h)

    def __len__(self):
        return _check(lib().qo_s2p_num_points(self._h))

    def data(self):
        """(f, s11, s21, s12, s22) as stored."""
        n = len(self)
        f = np.empty(n)
        s = [np.empty(n, dtype=np.complex128) for _ in range(4)]
        _check(lib().qo_s2p_get(self._h, _dp(f), *[a.ctypes.data_as(C.c_void_p) for a in s], n))
        return (f,) + tuple(s)

    def interp(self, f, polar=True):
        """Qucs SPfile 'linear' interpolation at the frequencies f -> (s11, s21, s12, s22)."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        s = [np.empty(len(f), dtype=np.complex128) for _ in range(4)]
        _check(lib().qo_s2p_interp(self._h, _dp(f), len(f), int(bool(polar)), *[a.ctypes.data_as(C.c_void_p) for a in s]))
        return tuple(s)

    def fit_inductor(self, fmin, fmax):
        """Least-squares fit of Z = (r0 + r1 sqrt(f) + jwL) || 1/(jwCp) -> dict(L, r0, r1, cp, srf, rms_rel)."""
        v = [C.c_double() for _ in range(6)]
        _check(lib().qo_s2p_fit_inductor(self._h, fmin, fmax, *[C.byref(x) for x in v]))
        return dict(zip(("L", "r0", "r1", "cp", "srf", "rms_rel"), [x.value for x in v]))

    def as_net(self, polar=True, rs=50.0, rl=50.0):
        """A one-element network holding a copy of this block (combine with Net.concat)."""
        h = C.c_void_p()
        _check(lib().qo_net_from_sblock(self._h, int(bool(polar)), rs, rl, C.byref(h)))
        return Net(h)

    def close(self):
        if self._h:
            lib().qo_s2p_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Dataset:
    """A Qucs dataset (qo_dat*): ordered variables, each a real or complex numpy array."""

    def __init__(self, handle=None):
        self._h = handle or C.c_void_p()
        if not handle:
            _check(lib().qo_dat_create(C.byref(self._h)))

    @classmethod
    def read(cls, path):
        h = C.c_void_p()
        _check(lib().qo_dat_read(os.fsencode(path), C.byref(h)))
        return cls(h)

    @classmethod
    def from_sweep(cls, f, s11, s12, s21, s22):
        f = np.ascontiguousarray(f, dtype=np.float64)
        arrs = [np.ascontiguousarray(a, dtype=np.complex128) for a in (s11, s12, s21, s22)]
        h = C.c_void_p()
        _check(lib().qo_dat_from_sweep(_dp(f), len(f), *[a.ctypes.data_as(C.c_void_p) for a in arrs], C.byref(h)))
        return cls(h)

    def add_indep(self, name, v):
        v = np.ascontiguousarray(v, dtype=np.float64)
        _check(lib().qo_dat_add_indep(self._h, name.encode(), _dp(v), len(v)))

    def add_dep(self, name, indep, v):
        v = np.asarray(v)
        re = np.ascontiguousarray(v.real, dtype=np.float64)
        im = np.ascontiguousarray(v.imag, dtype=np.float64) if np.iscomplexobj(v) else None
        _check(lib().qo_dat_add_dep(self._h, name.encode(), indep.encode(), _dp(re), _dp(im), len(re)))

    def write(self, path):
        _check(lib().qo_dat_write(self._h, os.fsencode(path)))

    def variables(self):
        """[(name, indep or '', n, is_complex)] in file order."""
        out = []
        for i in range(_check(lib().qo_dat_count(self._h))):
            name, indep, n, cx = C.c_char_p(), C.c_char_p(), C.c_int(), C.c_int()
            _check(lib().qo_dat_info(self._h, i, C.byref(name), C.byref(indep), C.byref(n), C.byref(cx)))
            out.append((name.value.decode(), indep.value.decode(), n.value, bool(cx.value)))
        return out

    def __getitem__(self, name):
        info = {v[0]: v for v in self.variables()}
        if name not in info:
            raise KeyError(name)
        n, cx = info[name][2], info[name][3]
        re, im = np.empty(n), np.empty(n)
        _check(lib().qo_dat_get(self._h, name.encode(), _dp(re), _dp(im), n))
        return re + 1j * im if cx else re

    def close(self):
        if self._h:
            lib().qo_dat_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def cpl_analyze(w, s, h, t, er, ht, f, length):
    o = [C.c_double() for _ in range(4)]
    _check(lib().qo_cpl_analyze(w, s, h, t, er, ht, f, length, *[C.byref(x) for x in o]))
    return tuple(x.value for x in o)


def cpl_synthesize(z0e, z0o, ang_deg, h, t, er, ht, f):
    """(W, S, L) of the coupled microstrip with these mode impedances and electrical length (qo_cpl_synthesize)."""
    o = [C.c_double() for _ in range(3)]
    _check(lib().qo_cpl_synthesize(z0e, z0o, ang_deg, h, t, er, ht, f, *[C.byref(x) for x in o]))
    return tuple(x.value for x in o)


def grid_lin(f0, f1, n):
    f = np.empty(n)
    _check(lib().qo_grid_lin(f0, f1, n, _dp(f)))
    return f


def grid_log(f0, f1, n):
    f = np.empty(n)
    _check(lib().qo_grid_log(f0, f1, n, _dp(f)))
    return f


def philox(ctr, key):
    c, k, o = (C.c_uint32 * 4)(*ctr), (C.c_uint32 * 2)(*key), (C.c_uint32 * 4)()
    lib().qo_philox4x32_10(c, k, o)
    return list(o)


def variate(seed, sample, var, dist=DIST_UNIFORM):
    return lib().qo_variate(seed, sample, var, dist)


def perturb_factor(seed, sample, var, dist, tol):
    return lib().qo_perturb_factor(seed, sample, var, dist, tol)


def _specs(specs):
    arr = (Spec * max(1, len(specs)))()
    for i, s in enumerate(specs):
        arr[i].kind, arr[i].f_lo, arr[i].f_hi, arr[i].limit = int(s[0]), float(s[1]), float(s[2]), float(s[3])
    return arr


def _cfg(seed, n_samples, tols, sample_offset, dist, mode, precision, hist_bins, hist_spec, hist_lo, hist_hi):
    cfg = McCfg()
    tarr = (Tol * max(1, len(tols)))()
    for i, t in enumerate(tols):
        tarr[i].elem, tarr[i].param, tarr[i].var, tarr[i].mode, tarr[i].tol = int(t[0]), int(t[1]), int(t[2]), int(t[3]), float(t[4])
    cfg._keep = tarr
    cfg.seed, cfg.sample_offset, cfg.n_samples = seed, sample_offset, n_samples
    cfg.dist, cfg.n_tol, cfg.tol = dist, len(tols), tarr
    cfg.mode, cfg.precision = mode, precision
    cfg.hist_bins, cfg.hist_spec, cfg.hist_lo, cfg.hist_hi = hist_bins, hist_spec, hist_lo, hist_hi
    return cfg


def _result(nspec, hist_bins):
    res = McResult()
    fps = np.zeros(max(1, nspec), dtype=np.uint64)
    hist = np.zeros(max(1, hist_bins), dtype=np.uint64)
    res.fail_per_spec = fps.ctypes.data_as(C.POINTER(C.c_uint64))
    res.hist = hist.ctypes.data_as(C.POINTER(C.c_uint64))
    return res, fps, hist


def _res_dict(res, fps, hist, nspec, hist_bins):
    return dict(n_pass=int(res.n_pass), n_total=int(res.n_total), fail_per_spec=fps[:nspec].copy(),
                hist=hist[:hist_bins].copy(), seconds=res.seconds, evals_per_s=res.evals_per_s,
                flops_per_eval=res.flops_per_eval)


def plan_analyze(net, f, specs, tols=(), dist=DIST_UNIFORM, mode=MODE_REDUCE_ONLY, precision=64,
                 hist_bins=0, hist_spec=0, hist_lo=0.0, hist_hi=1.0):
    """Host-only part of plan creation (qo_plan_analyze, no GPU needed): which kernel family the job would take and the
    transfer-function kernel's polynomial lengths / self-check result."""
    f = np.ascontiguousarray(f, dtype=np.float64)
    cfg = _cfg(0, 0, list(tols), 0, dist, mode, precision, hist_bins, hist_spec, hist_lo, hist_hi)
    info = (C.c_int * 6)()
    err, sec, fused, ferr = C.c_double(0.0), C.c_double(0.0), C.c_uint(0), C.c_double(0.0)
    reason = lib().qo_plan_analyze(net._h, _dp(f), len(f), _specs(specs), len(specs), C.byref(cfg), info, C.byref(err),
                                   C.byref(fused), C.byref(ferr), C.byref(sec)).decode()
    if info[0] < 0:
        raise QoError(info[0], reason)
    return dict(selected=bool(info[0]), numerator_chains=info[1], den_form=("none", "E", "D", "DD")[info[2]] if 0 <= info[2] <= 3 else "?",
                kn=info[3], kd=info[4], degree=info[5], self_check_err=err.value, fused_specs=fused.value, fused_err=ferr.value,
                reason=reason, seconds=sec.value)


def chain_jit_analyze(net, f, specs=(), tols=(), mode=MODE_REDUCE_ONLY, hist_bins=0, hist_spec=0, hist_lo=0.0, hist_hi=1.0):
    """Host-only (qo_chain_jit_analyze): fold the job's element list into the chain kernel and compile it with NVRTC
    -> dict(compiled, registers, spill_bytes, cubin_bytes, error)."""
    f = np.ascontiguousarray(f, dtype=np.float64)
    cfg = _cfg(0, 0, list(tols), 0, DIST_UNIFORM, mode, 64, hist_bins, hist_spec, hist_lo, hist_hi)
    info = (C.c_int * 4)()
    _check(lib().qo_chain_jit_analyze(net._h, _dp(f), len(f), _specs(specs), len(specs), C.byref(cfg), info))
    return dict(compiled=bool(info[0]), registers=info[1], spill_bytes=info[2], cubin_bytes=info[3],
                error=None if info[0] else lib().qo_last_error().decode())


class Plan:
    """A Monte-Carlo job resident in HBM (qo_plan*)."""

    def __init__(self, ctx, net, f, specs, seed=0, tols=(), dist=DIST_UNIFORM, mode=MODE_REDUCE_ONLY, precision=64,
                 hist_bins=0, hist_spec=0, hist_lo=0.0, hist_hi=1.0):
        self.ctx, self.net = ctx, net
        self.f = np.ascontiguousarray(f, dtype=np.float64)
        self.nspec, self.hist_bins = len(specs), hist_bins
        self._cfg = _cfg(seed, 0, list(tols), 0, dist, mode, precision, hist_bins, hist_spec, hist_lo, hist_hi)
        self._h = C.c_void_p()
        _check(lib().qo_plan_create(ctx._h, net._h, _dp(self.f), len(self.f), _specs(specs), len(specs),
                                    C.byref(self._cfg), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().qo_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_counters(self):
        return _check(lib().qo_plan_num_counters(self._h))

    @property
    def flops_per_eval(self):
        return lib().qo_plan_flops_per_eval(self._h)

    @property
    def launches(self):
        return _check(lib().qo_plan_launches(self._h))

    @property
    def kernel_name(self):
        """Which kernel this plan launches (ladder / interpreter / microstrip)."""
        return lib().qo_plan_kernel_name(self._h).decode()

    @property
    def tf_info(self):
        """The plan's decision about the transfer-function kernel (qo_plan_tf_info)."""
        info = (C.c_int * 6)()
        err, fused, ferr = C.c_double(0.0), C.c_uint(0), C.c_double(0.0)
        reason = lib().qo_plan_tf_info(self._h, info, C.byref(err), C.byref(fused), C.byref(ferr)).decode()
        return dict(selected=bool(info[0]), numerator_chains=info[1], den_form=("none", "E", "D", "DD")[info[2]] if 0 <= info[2] <= 3 else "?",
                    kn=info[3], kd=info[4], degree=info[5], self_check_err=err.value, fused_specs=fused.value, fused_err=ferr.value,
                    reason=reason)

    @property
    def h2d_bytes(self):
        """Host->device bytes qo_plan_create copied (per GPU)."""
        return int(lib().qo_plan_h2d_bytes(self._h))

    def reset(self):
        _check(lib().qo_plan_reset(self._h))

    def launch(self, sample_offset, n_samples, counters_dev=None, full_s_dev=None):
        """Asynchronous on the ctx stream; counters_dev / full_s_dev are raw device addresses (ints) or None."""
        _check(lib().qo_plan_launch(self._h, sample_offset, n_samples, counters_dev, full_s_dev))

    def read(self):
        res, fps, hist = _result(self.nspec, self.hist_bins)
        _check(lib().qo_plan_read(self._h, C.byref(res)))
        return _res_dict(res, fps, hist, self.nspec, self.hist_bins)


class Context:
    """Owns the device(s) and stream(s) (qo_ctx*)."""

    def __init__(self, ngpus=1, device=None):
        self._h = C.c_void_p()
        if device is not None:
            _check(lib().qo_ctx_create_on_device(int(device), C.byref(self._h)))
        else:
            _check(lib().qo_ctx_create(int(ngpus), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().qo_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_devices(self):
        return _check(lib().qo_ctx_num_devices(self._h))

    def set_stream(self, cuda_stream):
        _check(lib().qo_ctx_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def sweep(self, net, f, precision=64, gd=False):
        """Nominal sweep -> (s11, s21, s12, s22[, gd]) as numpy arrays."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        nf = len(f)
        outs = [np.empty(nf, dtype=np.complex128) for _ in range(4)]
        g = np.empty(nf) if gd else None
        _check(lib().qo_sweep(self._h, net._h, _dp(f), nf, precision, *[o.ctypes.data_as(C.c_void_p) for o in outs], _dp(g)))
        return tuple(outs) + ((g,) if gd else ())

    def mc_run(self, net, f, specs, seed, n_samples, tols=(), sample_offset=0, dist=DIST_UNIFORM,
               mode=MODE_REDUCE_ONLY, precision=64, hist_bins=0, hist_spec=0, hist_lo=0.0, hist_hi=1.0):
        """Monte-Carlo yield with host buffers (qo_mc_run)."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        nf, nspec = len(f), len(specs)
        cfg = _cfg(seed, n_samples, list(tols), sample_offset, dist, mode, precision, hist_bins, hist_spec, hist_lo, hist_hi)
        res, fps, hist = _result(nspec, hist_bins)
        full = np.empty((4, n_samples, nf), dtype=np.complex128) if mode == MODE_FULL_S else None
        _check(lib().qo_mc_run(self._h, net._h, _dp(f), nf, _specs(specs), nspec, C.byref(cfg), C.byref(res),
                               full.ctypes.data_as(C.c_void_p) if full is not None else None))
        out = _res_dict(res, fps, hist, nspec, hist_bins)
        if full is not None:
            out["s"] = full
        return out

    def nodal_sweep(self, nodal, f):
        """Nominal N-port sweep -> S[nf, np, np], S[:, k, j] = b_k / a_j (Qucs S[k+1, j+1])."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        npn = len(nodal.ports)
        out = np.empty((len(f), npn, npn), dtype=np.complex128)
        _check(lib().qo_nodal_sweep(self._h, nodal._h, _dp(f), len(f), out.ctypes.data_as(C.c_void_p)))
        return out

    def nodal_mc_run(self, nodal, f, specs, seed, n_samples, tols=(), sample_offset=0, dist=DIST_UNIFORM, mode=MODE_REDUCE_ONLY,
                     hist_bins=0, hist_spec=0, hist_lo=0.0, hist_hi=1.0):
        """Monte Carlo over branch parameters; specs: [(kind, row, col, f_lo, f_hi, limit_db)] on |S[row][col]|."""
        f = np.ascontiguousarray(f, dtype=np.float64)
        nf, nspec, npn = len(f), len(specs), len(nodal.ports)
        cfg = _cfg(seed, n_samples, list(tols), sample_offset, dist, mode, 64, hist_bins, hist_spec, hist_lo, hist_hi)
        sp = (NSpec * max(1, nspec))()
        for i, s in enumerate(specs):
            sp[i].kind, sp[i].row, sp[i].col, sp[i].f_lo, sp[i].f_hi, sp[i].limit = int(s[0]), int(s[1]), int(s[2]), float(s[3]), float(s[4]), float(s[5])
        res, fps, hist = _result(nspec, hist_bins)
        full = np.empty((n_samples, nf, npn, npn), dtype=np.complex128) if mode == MODE_FULL_S else None
        _check(lib().qo_nodal_mc_run(self._h, nodal._h, _dp(f), nf, sp, nspec, C.byref(cfg), C.byref(res),
                                     full.ctypes.data_as(C.c_void_p) if full is not None else None))
        out = _res_dict(res, fps, hist, nspec, hist_bins)
        if full is not None:
            out["s"] = full
        return out

    @staticmethod
    def nodal_last_kernel():
        return lib().qo_nodal_last_kernel().decode()

    @staticmethod
    def nodal_last_compile_seconds():
        return lib().qo_nodal_last_compile_seconds()

    def device_perturb_factors(self, seed, sample_offset, n_samples, n_var, dist, tol):
        out = np.empty((n_samples, n_var))
        _check(lib().qo_device_perturb_factors(self._h, seed, sample_offset, n_samples, n_var, dist, tol, _dp(out)))
        return out

    def device_mslog(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty_like(x)
        _check(lib().qo_device_mslog(self._h, _dp(x), x.size, _dp(out)))
        return out

    def device_rcp(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty_like(x)
        _check(lib().qo_device_rcp(self._h, _dp(x), x.size, _dp(out)))
        return out

    def measure_dfma_peak(self):
        t = C.c_double()
        _check(lib().qo_measure_dfma_peak(self._h, C.byref(t)))
        return t.value


def lc_tolerances(net, tol_l, tol_c, tol_other=None):
    """One independent random variable per reactive element (var = element index): +-tol_l on every L,
    +-tol_c on every C -- the perturbation of BASELINE configs 2, 4 and 5."""
    out = []
    for i, (kind, _p) in enumerate(net.elements):
        if kind in (SER_L, SHUNT_L):
            out.append((i, 0, len(out), TOL_REL, tol_l))
        elif kind in (SER_C, SHUNT_C):
            out.append((i, 0, len(out), TOL_REL, tol_c))
        elif kind in (SER_LC_SER, SER_LC_PAR, SHUNT_LC_SER, SHUNT_LC_PAR):
            out.append((i, 0, len(out), TOL_REL, tol_l))
            out.append((i, 1, len(out), TOL_REL, tol_c))
    return out
