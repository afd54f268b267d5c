"""ORACLE python wrapper (ctypes over oracle/liboracle.so) -- test infrastructure, NOT product.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  PARITY UNPINNED (see rbd_oracle.hpp): the oracle restates the published
algorithms; the RaiSim binary is unavailable, parity with RaiSim itself is unverified.
"""
import ctypes as C
import os
import subprocess
import tempfile
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")

PARAM_ORDER = ("dt", "gx", "gy", "gz", "erp", "alpha_init", "alpha_min", "alpha_decay", "max_iter",
               "threshold", "mu", "restitution", "rest_threshold", "stall_window", "stall_ratio", "warm_start", "slip_bisect", "joint_limits", "slip_local", "accel_m", "accel_start", "stall_reg")
DEFAULT_PARAMS = dict(dt=0.0025, gx=0.0, gy=0.0, gz=-9.81, erp=0.0, alpha_init=1.0, alpha_min=1.0, alpha_decay=1.0,
                      max_iter=150, threshold=1e-7, mu=0.8, restitution=0.0, rest_threshold=0.01, stall_window=8, stall_ratio=0.5, warm_start=0, slip_bisect=0, joint_limits=1, slip_local=1, accel_m=2, accel_start=6, stall_reg=0.02)


def build(force=False):
    if force or not os.path.exists(_LIB_PATH) or any(
            os.path.getmtime(os.path.join(_HERE, f)) > os.path.getmtime(_LIB_PATH)
            for f in ("oracle_capi.cpp", "rbd_oracle.hpp")):
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s", "liboracle.so"])
    return _LIB_PATH


class _ModelDesc(C.Structure):
    _fields_ = [("nb", C.c_int), ("nq", C.c_int), ("nv", C.c_int), ("floating", C.c_int),
                ("parent", C.c_void_p), ("jtype", C.c_void_p), ("qidx", C.c_void_p), ("vidx", C.c_void_p),
                ("jpos", C.c_void_p), ("jrot", C.c_void_p), ("axis", C.c_void_p), ("mass", C.c_void_p),
                ("com", C.c_void_p), ("inertia", C.c_void_p), ("jlimit", C.c_void_p), ("jeffort", C.c_void_p),
                ("npts", C.c_int), ("pt_body", C.c_void_p), ("pt_pos", C.c_void_p), ("pt_rad", C.c_void_p),
                ("pt_type", C.c_void_p), ("pt_coll", C.c_void_p), ("pt_pos2", C.c_void_p),
                ("ncoll", C.c_int), ("coll_size", C.c_void_p), ("coll_pos", C.c_void_p), ("coll_rot", C.c_void_p)]


class _Debug(C.Structure):
    _fields_ = ([(n, C.c_void_p) for n in ("M", "h", "R", "p", "ncontacts", "c_pt", "c_body", "c_pair", "c_pos",
                                           "c_normal", "c_depth", "c_lambda", "iters", "G", "u0")]
                + [("ext_body", C.c_int), ("ext_force", C.c_void_p), ("ext_torque", C.c_void_p), ("ext_point", C.c_double * 3)]
                + [(n, C.c_void_p) for n in ("warm_pt", "warm_imp", "tau_applied", "nlimits", "lim_dof", "lim_lambda", "resid", "status")])


_libs = {}


def _declare(L):
    L.orc_create.restype = C.c_void_p
    L.orc_create.argtypes = [C.POINTER(_ModelDesc), C.c_int]
    L.orc_destroy.argtypes = [C.c_void_p]
    L.orc_set_params.argtypes = [C.c_void_p, C.c_void_p]
    L.orc_set_ground.argtypes = [C.c_void_p, C.c_double]
    L.orc_set_heightmap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p]
    L.orc_set_heightmaps.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_int]
    L.orc_clear_terrain.argtypes = [C.c_void_p]
    L.orc_step.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p]
    L.orc_solve_one.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
    L.orc_set_point_mu.argtypes = [C.c_void_p, C.c_void_p]
    L.orc_get_flops.argtypes = [C.c_void_p, C.c_int]
    L.orc_get_counts.argtypes = [C.c_void_p, C.c_int]
    return L


def lib(which="parity"):
    """parity: liboracle.so, the checker (-ffp-contract=off, portable ISA: bit-stable predicates).
    native: liboracle_native.so, the TIMING build of the same source for bench.py's CPU arm (-O3 -march=native, FMA
    contraction on), compiled on the machine it is timed on into a temporary directory (the source tree may be read-only)
    and removed once loaded; falls back to the parity build if that fails."""
    if which not in _libs:
        if which == "native":
            try:
                with tempfile.TemporaryDirectory(prefix="oracle_native_") as tmp:
                    path = os.path.join(tmp, "liboracle_native.so")
                    subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "native", "NATIVE_LIB=" + path])
                    _libs[which] = _declare(C.CDLL(path))
            except Exception:
                _libs[which] = lib("parity")
        else:
            build()
            _libs[which] = _declare(C.CDLL(_LIB_PATH))
    return _libs[which]


def native_build_available():
    return lib("native") is not lib("parity")


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Oracle:
    """CPU restatement of raisim::World::integrate() for a batch of independent environments."""

    def __init__(self, tables, precision="f64", params=None, build="parity"):
        self.L = lib(build)
        self.t = tables
        self.nb, self.nq, self.nv = tables["nb"], tables["nq"], tables["nv"]
        self._keep = {k: np.ascontiguousarray(tables[k], dtype=(np.int32 if tables[k].dtype.kind == "i" else np.float64))
                      for k in ("parent", "jtype", "qidx", "vidx", "jpos", "jrot", "axis", "mass", "com", "inertia", "jlimit", "jeffort",
                                "pt_body", "pt_pos", "pt_rad", "pt_type", "pt_coll", "pt_pos2")}
        for src, dst in (("csize", "coll_size"), ("cpos", "coll_pos"), ("crot", "coll_rot")):
            self._keep[dst] = np.ascontiguousarray(tables[src], dtype=np.float64)
        d = _ModelDesc(nb=self.nb, nq=self.nq, nv=self.nv, floating=tables["floating"], npts=tables["npts"], ncoll=tables["ncoll"])
        for k, a in self._keep.items():
            setattr(d, k, a.ctypes.data)
        self.precision = precision
        self.h = self.L.orc_create(C.byref(d), {"f64": 0, "f32": 1, "count": 2}[precision])
        self.kmax = self.L.orc_kmax()
        self.params = dict(DEFAULT_PARAMS)
        self.set_params(**(params or {}))
        self.warm_pt = self.warm_imp = None      # contact cache carried across step() calls (per environment)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.orc_destroy(self.h)
            self.h = None

    def set_params(self, **kw):
        self.params.update(kw)
        arr = np.array([float(self.params[k]) for k in PARAM_ORDER], dtype=np.float64)
        self.L.orc_set_params(self.h, _p(arr))

    def set_ground(self, z=0.0):
        self.L.orc_set_ground(self.h, float(z))

    def set_heightmap(self, xs, ys, x_size, y_size, cx, cy, heights):
        hh = np.ascontiguousarray(heights, dtype=np.float64).reshape(-1)
        assert hh.size == xs * ys
        self.L.orc_set_heightmap(self.h, xs, ys, x_size, y_size, cx, cy, _p(hh))

    def set_heightmaps(self, x_size, y_size, cx, cy, heights, env_map):
        """terrain atlas: heights [count, ys, xs], env_map [n] -> every environment collides with its own map"""
        hh = np.ascontiguousarray(heights, dtype=np.float64)
        count, ys, xs = hh.shape
        em = np.ascontiguousarray(env_map, dtype=np.int32)
        assert em.min() >= 0 and em.max() < count
        self.L.orc_set_heightmaps(self.h, count, xs, ys, x_size, y_size, cx, cy, _p(hh), em.ctypes.data, len(em))

    def clear_terrain(self):
        self.L.orc_clear_terrain(self.h)

    def set_collision_friction(self, collision_body, mu):
        """friction of every candidate point of one collision body (mu < 0: default material)"""
        if not hasattr(self, "_pt_mu"):
            self._pt_mu = np.full(self.t["npts"], -1.0)
        self._pt_mu[np.asarray(self.t["pt_coll"]) == collision_body] = mu
        self.L.orc_set_point_mu(self.h, _p(self._pt_mu))

    def step(self, gc, gv, n_steps=1, tau_ff=None, ptarget=None, vtarget=None, kp=None, kd=None, nthreads=0, debug=False, ext=None):
        """gc [n,nq], gv [n,nv] float64 C-contiguous, updated IN PLACE.  Returns debug dict or None.
        ext = (body, force [n,3] world | None, torque [n,3] world | None, point in body frame (3) | None): external wrench
        acting during this call (ArticulatedSystem::setExternalForce / setExternalTorque)."""
        assert gc.dtype == np.float64 and gv.dtype == np.float64 and gc.flags.c_contiguous and gv.flags.c_contiguous
        n = gc.shape[0]
        assert gc.shape == (n, self.nq) and gv.shape == (n, self.nv)
        f = lambda a, w: None if a is None else np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (n, w)))
        tau_ff, ptarget, vtarget = f(tau_ff, self.nv), f(ptarget, self.nq), f(vtarget, self.nv)
        g = lambda a: None if a is None else np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.nv,)))
        kp, kd = g(kp), g(kd)
        if self.warm_pt is None or self.warm_pt.shape[0] != n:
            self.reset_warm_start(n)
        out = {}
        if debug:
            K, nb, nv = self.kmax, self.nb, self.nv
            out = dict(M=np.zeros((n, nv, nv)), h=np.zeros((n, nv)), R=np.zeros((n, nb, 3, 3)), p=np.zeros((n, nb, 3)),
                       ncontacts=np.zeros(n, np.int32), c_pt=np.zeros((n, K), np.int32), c_body=np.zeros((n, K), np.int32),
                       c_pair=np.zeros((n, K), np.int32), c_pos=np.zeros((n, K, 3)), c_normal=np.zeros((n, K, 3)),
                       c_depth=np.zeros((n, K)), c_lambda=np.zeros((n, K, 3)), iters=np.zeros(n, np.int32),
                       G=np.zeros((n, 3 * K + 4, 3 * K + 4)), u0=np.zeros((n, 3 * K + 4)), tau_applied=np.zeros((n, nv)),
                       nlimits=np.zeros(n, np.int32), lim_dof=np.full((n, 4), -1, np.int32), lim_lambda=np.zeros((n, 4)), resid=np.zeros(n), status=np.zeros(n, np.int32))
        ptrs = {k: v.ctypes.data for k, v in out.items()}
        ptrs["warm_pt"], ptrs["warm_imp"] = self.warm_pt.ctypes.data, self.warm_imp.ctypes.data
        dbg = _Debug(**ptrs)
        dbg.ext_body = -1
        if ext is not None:
            eb, ef, et, ep = ext
            ef = None if ef is None else np.ascontiguousarray(np.broadcast_to(np.asarray(ef, np.float64), (n, 3)))
            et = None if et is None else np.ascontiguousarray(np.broadcast_to(np.asarray(et, np.float64), (n, 3)))
            dbg.ext_body = int(eb)
            dbg.ext_force = None if ef is None else ef.ctypes.data
            dbg.ext_torque = None if et is None else et.ctypes.data
            dbg.ext_point = (C.c_double * 3)(*(np.zeros(3) if ep is None else np.asarray(ep, np.float64)))
        self.L.orc_step(self.h, n, n_steps, _p(gc), _p(gv), _p(tau_ff), _p(ptarget), _p(vtarget), _p(kp), _p(kd),
                       int(nthreads), C.byref(dbg))
        return out if debug else None

    def reset_warm_start(self, n=None):
        """forget the contact cache (what rsb_batch_set_state does for the environments it touches)"""
        n = n if n is not None else (self.warm_pt.shape[0] if self.warm_pt is not None else 0)
        self.warm_pt = np.full((n, self.kmax), -1, np.int32)
        self.warm_imp = np.zeros((n, self.kmax, 3))

    def solve_one(self, G, c, mu):
        G = np.ascontiguousarray(G, np.float64); c = np.ascontiguousarray(c, np.float64)
        lam = np.zeros(3)
        self.L.orc_solve_one(self.h, _p(G), _p(c), float(mu), _p(lam))
        return lam


def flop_counters(reset=True):
    """counters of the FLOP-counting build (Oracle(..., precision="count")): dict add/mul/div/sqrt/trig/cmp"""
    c = (C.c_longlong * 6)()
    lib().orc_get_flops(c, 1 if reset else 0)
    return dict(zip(("add", "mul", "div", "sqrt", "trig", "cmp"), [int(x) for x in c]))


def solver_outcome_counters(reset=True):
    """per-contact rule outcomes summed over all step() calls: opening, stick, slip, slip found by the local fan"""
    c = (C.c_longlong * 4)()
    lib().orc_get_counts(c, 1 if reset else 0)
    return dict(zip(("open", "stick", "slip", "slip_local"), [int(x) for x in c]))
