"""ctypes binding of the C-ABI in include/rsb.h (raisimlib_b200/librsb.so).

Thin by design: the product is the CUDA library; Python only drives it from tests and bench.py.
There is NO CPU fallback -- if librsb.so is missing or no GPU is visible the calls fail loudly.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RSB_LIB_PATH") or os.path.join(_HERE, "librsb.so")   # RSB_LIB_PATH: another build of the same library (A/B probes in tools/)
KMAX = 8
HOST, DEVICE = 0, 1
FORCE_AND_TORQUE, PD_PLUS_FEEDFORWARD_TORQUE = 0, 1


class RsbError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [("dt", C.c_float), ("gravity", C.c_float * 3), ("erp", C.c_float), ("alpha_init", C.c_float),
                ("alpha_min", C.c_float), ("alpha_decay", C.c_float), ("max_iter", C.c_int), ("threshold", C.c_float),
                ("mu", C.c_float), ("restitution", C.c_float), ("rest_threshold", C.c_float),
                ("stall_window", C.c_int), ("stall_ratio", C.c_float), ("joint_limits", C.c_int),
                ("accel_m", C.c_int), ("accel_start", C.c_int), ("stall_reg", C.c_float)]


class Contact(C.Structure):
    _fields_ = [("local_body", C.c_int32), ("pair_index", C.c_int32), ("position", C.c_float * 3),
                ("normal", C.c_float * 3), ("impulse", C.c_float * 3), ("depth", C.c_float)]


CONTACT_DTYPE = np.dtype([("local_body", np.int32), ("pair_index", np.int32), ("position", np.float32, 3),
                          ("normal", np.float32, 3), ("impulse", np.float32, 3), ("depth", np.float32)])
assert CONTACT_DTYPE.itemsize == C.sizeof(Contact) == 48


class RayHit(C.Structure):
    _fields_ = [("distance", C.c_float), ("position", C.c_float * 3), ("normal", C.c_float * 3), ("pair_index", C.c_int32)]


RAY_HIT_DTYPE = np.dtype([("distance", np.float32), ("position", np.float32, 3), ("normal", np.float32, 3), ("pair_index", np.int32)])
assert RAY_HIT_DTYPE.itemsize == C.sizeof(RayHit) == 32


class ModelTables(C.Structure):
    _fields_ = ([(n, C.c_int) for n in ("nb", "nq", "nv", "floating", "ncoll", "npts")] +
                [(n, C.POINTER(C.c_int)) for n in ("parent", "jtype", "qidx", "vidx", "depth")] +
                [(n, C.POINTER(C.c_double)) for n in ("jpos", "jrot", "axis", "mass", "com", "inertia", "jlimit")] +
                [(n, C.POINTER(C.c_int)) for n in ("cbody", "ctype")] +
                [(n, C.POINTER(C.c_double)) for n in ("csize", "cpos", "crot")] +
                [(n, C.POINTER(C.c_int)) for n in ("pt_body", "pt_coll", "pt_feat")] +
                [(n, C.POINTER(C.c_double)) for n in ("pt_pos", "pt_rad")] +
                [("pt_type", C.POINTER(C.c_int)), ("pt_pos2", C.POINTER(C.c_double)), ("jeffort", C.POINTER(C.c_double))])


class TerrainProperties(C.Structure):
    _fields_ = [("x_samples", C.c_int), ("y_samples", C.c_int), ("x_size", C.c_double), ("y_size", C.c_double), ("frequency", C.c_double),
                ("z_scale", C.c_double), ("fractal_octaves", C.c_int), ("fractal_lacunarity", C.c_double), ("fractal_gain", C.c_double),
                ("step_size", C.c_double), ("height_offset", C.c_double), ("seed", C.c_uint32)]


def generate_terrain(x_samples=129, y_samples=129, x_size=12.8, y_size=12.8, frequency=0.2, z_scale=0.5, fractal_octaves=3,
                     fractal_lacunarity=2.0, fractal_gain=0.25, step_size=0.0, height_offset=0.0, seed=1):
    """raisim::TerrainProperties -> heights [y_samples, x_samples] float32 (host)"""
    p = TerrainProperties(x_samples, y_samples, x_size, y_size, frequency, z_scale, fractal_octaves, fractal_lacunarity, fractal_gain,
                          step_size, height_offset, seed)
    out = np.empty((y_samples, x_samples), np.float32)
    _ck(lib().rsb_terrain_generate(C.byref(p), out.ctypes.data_as(C.c_void_p)))
    return out


def read_heightmap_text(path):
    """World::addHeightMap(raisimHeightMapFileName, ...): -> (heights [ys, xs] float32, x_size, y_size)"""
    xs, ys, sx, sy = C.c_int(), C.c_int(), C.c_double(), C.c_double()
    L = lib()
    _ck(L.rsb_heightmap_read_text(path.encode(), C.byref(xs), C.byref(ys), C.byref(sx), C.byref(sy), None, 0))
    out = np.empty((ys.value, xs.value), np.float32)
    _ck(L.rsb_heightmap_read_text(path.encode(), C.byref(xs), C.byref(ys), C.byref(sx), C.byref(sy), out.ctypes.data_as(C.c_void_p), out.size))
    return out, sx.value, sy.value


def read_heightmap_png(path, height_scale=1.0, height_offset=0.0):
    """World::addHeightMap(pngFileName, cx, cy, xSize, ySize, heightScale, heightOffset): -> heights [ys, xs] float32"""
    xs, ys = C.c_int(), C.c_int()
    L = lib()
    _ck(L.rsb_heightmap_read_png(path.encode(), height_scale, height_offset, C.byref(xs), C.byref(ys), None, 0))
    out = np.empty((ys.value, xs.value), np.float32)
    _ck(L.rsb_heightmap_read_png(path.encode(), height_scale, height_offset, C.byref(xs), C.byref(ys), out.ctypes.data_as(C.c_void_p), out.size))
    return out


class DeviceView(C.Structure):
    _fields_ = ([(n, C.c_int) for n in ("num_envs", "nq", "nv", "gc_stride", "gv_stride")] +
                [(n, C.c_void_p) for n in ("gc", "gv", "tau_ff", "ptarget", "vtarget", "ncontacts", "contacts")])


EXPORTED = [
    "rsb_last_error", "rsb_version", "rsb_params_default",
    "rsb_model_create_from_urdf", "rsb_model_destroy", "rsb_model_save", "rsb_model_load", "rsb_model_dims", "rsb_model_get_tables", "rsb_model_body_index",
    "rsb_model_body_name", "rsb_model_collision_index", "rsb_model_joint_name", "rsb_model_frame_index", "rsb_model_frame",
    "rsb_batch_create", "rsb_batch_destroy", "rsb_batch_set_stream", "rsb_batch_sync", "rsb_batch_num_envs",
    "rsb_batch_set_ground", "rsb_batch_set_heightmap", "rsb_batch_set_heightmaps", "rsb_batch_clear_terrain", "rsb_batch_set_params", "rsb_batch_get_params",
    "rsb_batch_set_collision_friction",
    "rsb_batch_set_state", "rsb_batch_get_state", "rsb_batch_set_pd_gains", "rsb_batch_set_pd_target",
    "rsb_batch_set_generalized_force", "rsb_batch_set_external_wrench", "rsb_batch_set_control_mode", "rsb_batch_get_generalized_force", "rsb_batch_bind_pd_target",
    "rsb_batch_integrate1", "rsb_batch_integrate2", "rsb_batch_integrate",
    "rsb_batch_get_mass_matrix", "rsb_batch_get_nonlinearities", "rsb_batch_get_body_poses", "rsb_batch_get_contacts",
    "rsb_batch_get_contact_points", "rsb_batch_get_solver_iterations", "rsb_batch_get_diverged", "rsb_batch_get_solver_residual", "rsb_batch_get_solver_status", "rsb_batch_update_kinematics", "rsb_batch_device_ptrs", "rsb_batch_launch_count",
    "rsb_batch_ob_dim", "rsb_batch_observe", "rsb_batch_control_step", "rsb_batch_height_scan", "rsb_batch_ray_test",
    "rsb_batch_gym_configure", "rsb_batch_gym_reset", "rsb_batch_gym_step",
    "rsb_peer_buffer_create", "rsb_peer_buffer_open", "rsb_peer_buffer_close", "rsb_peer_buffer_destroy", "rsb_batch_set_observation_peers", "rsb_batch_wait_observation_peers",
    "rsb_comm_init", "rsb_comm_allgather_obs", "rsb_comm_destroy", "rsb_terrain_generate", "rsb_heightmap_read_text", "rsb_heightmap_read_png",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            # not a fallback: the same CUDA library, compiled on the spot when the prebuilt one did not travel
            import subprocess
            try:
                subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc")], stdout=subprocess.DEVNULL)
            except Exception as e:
                raise RsbError(f"{LIB_PATH} is missing and could not be built ({e}): run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
        L = C.CDLL(LIB_PATH)
        L.rsb_last_error.restype = C.c_char_p
        L.rsb_model_body_name.restype = C.c_char_p
        L.rsb_model_joint_name.restype = C.c_char_p
        L.rsb_batch_launch_count.restype = C.c_int64
        L.rsb_model_create_from_urdf.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.rsb_model_load.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.rsb_model_save.argtypes = [C.c_void_p, C.c_char_p]
        L.rsb_model_destroy.argtypes = [C.c_void_p]
        L.rsb_model_dims.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 5
        L.rsb_model_get_tables.argtypes = [C.c_void_p, C.POINTER(ModelTables)]
        L.rsb_model_body_index.argtypes = [C.c_void_p, C.c_char_p]
        L.rsb_model_collision_index.argtypes = [C.c_void_p, C.c_char_p]
        L.rsb_model_body_name.argtypes = [C.c_void_p, C.c_int]
        L.rsb_model_joint_name.argtypes = [C.c_void_p, C.c_int]
        L.rsb_model_frame_index.argtypes = [C.c_void_p, C.c_char_p]
        L.rsb_model_frame.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_void_p]
        L.rsb_batch_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.rsb_batch_destroy.argtypes = [C.c_void_p]
        L.rsb_batch_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.rsb_batch_sync.argtypes = [C.c_void_p]
        L.rsb_batch_num_envs.argtypes = [C.c_void_p]
        L.rsb_batch_set_ground.argtypes = [C.c_void_p, C.c_float]
        L.rsb_batch_set_heightmap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.rsb_batch_set_heightmaps.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        L.rsb_batch_clear_terrain.argtypes = [C.c_void_p]
        L.rsb_batch_set_collision_friction.argtypes = [C.c_void_p, C.c_int, C.c_float]
        L.rsb_batch_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
        L.rsb_batch_get_params.argtypes = [C.c_void_p, C.POINTER(Params)]
        L.rsb_params_default.argtypes = [C.POINTER(Params)]
        for n in ("rsb_batch_set_state", "rsb_batch_get_state", "rsb_batch_set_pd_target"):
            getattr(L, n).argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_set_pd_gains.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.rsb_batch_set_generalized_force.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_set_control_mode.argtypes = [C.c_void_p, C.c_int]
        L.rsb_batch_set_external_wrench.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_bind_pd_target.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.rsb_batch_get_generalized_force.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_integrate1.argtypes = [C.c_void_p]
        L.rsb_batch_integrate2.argtypes = [C.c_void_p]
        L.rsb_batch_integrate.argtypes = [C.c_void_p, C.c_int]
        for n in ("rsb_batch_get_mass_matrix", "rsb_batch_get_nonlinearities"):
            getattr(L, n).argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.rsb_batch_get_body_poses.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.rsb_batch_get_contacts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_get_contact_points.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_get_solver_iterations.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_get_diverged.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_get_solver_residual.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_get_solver_status.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_update_kinematics.argtypes = [C.c_void_p]
        L.rsb_batch_device_ptrs.argtypes = [C.c_void_p, C.POINTER(DeviceView)]
        L.rsb_batch_launch_count.argtypes = [C.c_void_p]
        L.rsb_batch_ob_dim.argtypes = [C.c_void_p]
        L.rsb_batch_observe.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_control_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.rsb_batch_height_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_ray_test.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.rsb_batch_gym_configure.argtypes = [C.c_void_p] + [C.c_void_p] * 5 + [C.c_int, C.c_float, C.c_float, C.c_float]
        L.rsb_batch_gym_reset.argtypes = [C.c_void_p]
        L.rsb_batch_gym_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.rsb_comm_init.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
        L.rsb_comm_allgather_obs.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.rsb_comm_destroy.argtypes = [C.c_void_p]
        L.rsb_terrain_generate.argtypes = [C.POINTER(TerrainProperties), C.c_void_p]
        L.rsb_heightmap_read_text.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.rsb_heightmap_read_png.argtypes = [C.c_char_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.rsb_peer_buffer_create.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_void_p), C.c_void_p]
        L.rsb_peer_buffer_open.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.rsb_peer_buffer_close.argtypes = [C.c_void_p]
        L.rsb_peer_buffer_destroy.argtypes = [C.c_void_p]
        L.rsb_batch_set_observation_peers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.rsb_batch_wait_observation_peers.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        _lib = L
    return _lib


def _ck(rc):
    if rc < 0:
        raise RsbError(lib().rsb_last_error().decode())
    return rc


def _ptr(a):
    """numpy array -> host pointer; torch CUDA tensor -> device pointer; int -> raw pointer."""
    if a is None:
        return None, HOST
    if isinstance(a, np.ndarray):
        assert a.flags.c_contiguous
        return a.ctypes.data_as(C.c_void_p), HOST
    if hasattr(a, "data_ptr"):
        assert a.is_contiguous()
        return C.c_void_p(a.data_ptr()), (DEVICE if a.is_cuda else HOST)
    raise TypeError(type(a))


class Model:
    def __init__(self, path_or_xml, cache=False):
        """URDF path / XML text, or (cache=True) a binary model cache written by Model.save()"""
        h = C.c_void_p()
        if cache:
            _ck(lib().rsb_model_load(path_or_xml.encode(), C.byref(h)))
        else:
            _ck(lib().rsb_model_create_from_urdf(path_or_xml.encode(), C.byref(h)))
        self.h = h
        d = [C.c_int() for _ in range(5)]
        _ck(lib().rsb_model_dims(h, *[C.byref(x) for x in d]))
        self.nq, self.nv, self.nb, self.ncoll, self.npts = [x.value for x in d]

    def collision_index(self, name):
        return _ck(lib().rsb_model_collision_index(self.h, name.encode()))

    def save(self, path):
        _ck(lib().rsb_model_save(self.h, path.encode()))

    def __del__(self):
        if getattr(self, "h", None) and lib is not None and _lib is not None:     # at interpreter shutdown the module globals may be gone already
            _lib.rsb_model_destroy(self.h)
            self.h = None

    def tables(self):
        t = ModelTables()
        _ck(lib().rsb_model_get_tables(self.h, C.byref(t)))
        nb, nc, npt = t.nb, t.ncoll, t.npts
        arr = lambda p, n, dt: np.ctypeslib.as_array(p, shape=(n,)).astype(dt).copy() if n > 0 else np.zeros(0, dt)
        out = dict(nb=nb, nq=t.nq, nv=t.nv, floating=t.floating, ncoll=nc, npts=npt)
        for k in ("parent", "jtype", "qidx", "vidx", "depth"):
            out[k] = arr(getattr(t, k), nb, np.int32)
        for k, w in (("jpos", 3), ("jrot", 9), ("axis", 3), ("mass", 1), ("com", 3), ("inertia", 6), ("jlimit", 2)):
            a = arr(getattr(t, k), nb * w, np.float64)
            out[k] = a.reshape(nb, w) if w > 1 else a
        for k in ("cbody", "ctype"):
            out[k] = arr(getattr(t, k), nc, np.int32)
        for k, w in (("csize", 3), ("cpos", 3), ("crot", 9)):
            out[k] = arr(getattr(t, k), nc * w, np.float64).reshape(nc, w)
        for k in ("pt_body", "pt_coll", "pt_feat"):
            out[k] = arr(getattr(t, k), npt, np.int32)
        out["pt_pos"] = arr(t.pt_pos, npt * 3, np.float64).reshape(npt, 3)
        out["pt_rad"] = arr(t.pt_rad, npt, np.float64)
        out["pt_type"] = arr(t.pt_type, npt, np.int32)
        out["pt_pos2"] = arr(t.pt_pos2, npt * 3, np.float64).reshape(npt, 3)
        out["jeffort"] = arr(t.jeffort, nb, np.float64)
        out["body_names"] = [lib().rsb_model_body_name(self.h, i).decode() for i in range(nb)]
        out["joint_names"] = [lib().rsb_model_joint_name(self.h, i).decode() for i in range(nb)]
        return out

    def body_index(self, name):
        return _ck(lib().rsb_model_body_index(self.h, name.encode()))

    def frame_index(self, name):
        return _ck(lib().rsb_model_frame_index(self.h, name.encode()))


class Batch:
    """N environments of one model on one GPU; mirrors World/ArticulatedSystem calls batch-wide."""

    def __init__(self, model, num_envs, device=0):
        self.model = model
        h = C.c_void_p()
        _ck(lib().rsb_batch_create(model.h, num_envs, device, C.byref(h)))
        self.h, self.n, self.nq, self.nv, self.nb = h, num_envs, model.nq, model.nv, model.nb

    def __del__(self):
        if getattr(self, "h", None) and lib is not None and _lib is not None:
            _lib.rsb_batch_destroy(self.h)
            self.h = None

    def _count(self, env_begin, env_count):
        """number of environments a call covers: env_count, or every environment from env_begin on when it is None"""
        return self.n - env_begin if env_count is None else env_count

    def _read(self, getter, row_shape, dtype, env_begin, env_count, range_first=False):
        """new host array [n, *row_shape] filled by the C getter `getter` for n environments from env_begin.  The getters take
        (batch, out, env_begin, env_count, where), or with range_first (batch, env_begin, env_count, out, where)."""
        n = self._count(env_begin, env_count)
        out = np.empty((n, *row_shape), dtype)
        p = out.ctypes.data_as(C.c_void_p)
        _ck(getattr(lib(), getter)(self.h, *((env_begin, n, p) if range_first else (p, env_begin, n)), HOST))
        return out

    # world set-up
    def set_stream(self, stream_ptr):
        _ck(lib().rsb_batch_set_stream(self.h, C.c_void_p(stream_ptr)))

    def sync(self):
        _ck(lib().rsb_batch_sync(self.h))

    def set_ground(self, z=0.0):
        _ck(lib().rsb_batch_set_ground(self.h, z))

    def set_heightmap(self, xs, ys, x_size, y_size, cx, cy, heights):
        hh = np.ascontiguousarray(heights, dtype=np.float32).reshape(-1)
        assert hh.size == xs * ys
        _ck(lib().rsb_batch_set_heightmap(self.h, xs, ys, x_size, y_size, cx, cy, hh.ctypes.data_as(C.c_void_p)))

    def set_heightmaps(self, x_size, y_size, cx, cy, heights, map_of_env):
        """terrain atlas: heights [count, ys, xs] float32, map_of_env [n] int32 -> one height map per environment"""
        h = np.ascontiguousarray(heights, np.float32)
        count, ys, xs = h.shape
        m = np.ascontiguousarray(map_of_env, np.int32)
        assert m.shape == (self.n,)
        _ck(lib().rsb_batch_set_heightmaps(self.h, count, xs, ys, x_size, y_size, cx, cy, h.ctypes.data_as(C.c_void_p), m.ctypes.data_as(C.c_void_p)))

    def clear_terrain(self):
        _ck(lib().rsb_batch_clear_terrain(self.h))

    def set_collision_friction(self, collision_body, mu):
        _ck(lib().rsb_batch_set_collision_friction(self.h, collision_body, mu))

    def get_params(self):
        p = Params()
        _ck(lib().rsb_batch_get_params(self.h, C.byref(p)))
        return p

    def set_params(self, **kw):
        p = self.get_params()
        for k, v in kw.items():
            if k == "gravity":
                p.gravity[0], p.gravity[1], p.gravity[2] = v
            else:
                setattr(p, k, v)
        _ck(lib().rsb_batch_set_params(self.h, C.byref(p)))

    # state / actuation
    def set_state(self, gc=None, gv=None, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        pg, w1 = _ptr(gc); pv, w2 = _ptr(gv)
        _ck(lib().rsb_batch_set_state(self.h, pg, pv, env_begin, n, w1 if gc is not None else w2))

    def get_state(self, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        gc, gv = np.empty((n, self.nq), np.float32), np.empty((n, self.nv), np.float32)
        _ck(lib().rsb_batch_get_state(self.h, gc.ctypes.data_as(C.c_void_p), gv.ctypes.data_as(C.c_void_p), env_begin, n, HOST))
        return gc, gv

    def get_state_into(self, gc, gv, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        pg, w1 = _ptr(gc); pv, w2 = _ptr(gv)
        _ck(lib().rsb_batch_get_state(self.h, pg, pv, env_begin, n, w1 if gc is not None else w2))

    def set_pd_gains(self, kp, kd):
        kp = np.ascontiguousarray(np.broadcast_to(np.asarray(kp, np.float32), (self.nv,)))
        kd = np.ascontiguousarray(np.broadcast_to(np.asarray(kd, np.float32), (self.nv,)))
        _ck(lib().rsb_batch_set_pd_gains(self.h, kp.ctypes.data_as(C.c_void_p), kd.ctypes.data_as(C.c_void_p)))

    def set_pd_target(self, ptarget=None, vtarget=None, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        pp, w1 = _ptr(ptarget); pv, w2 = _ptr(vtarget)
        _ck(lib().rsb_batch_set_pd_target(self.h, pp, pv, env_begin, n, w1 if ptarget is not None else w2))

    def bind_pd_target(self, ptarget_dev, row_stride=None):
        """zero-copy: the kernel reads PD-target rows from this device tensor (None unbinds)"""
        if ptarget_dev is None:
            _ck(lib().rsb_batch_bind_pd_target(self.h, None, 0)); return
        assert ptarget_dev.is_cuda and ptarget_dev.is_contiguous()
        self._bound = ptarget_dev        # keep alive
        _ck(lib().rsb_batch_bind_pd_target(self.h, C.c_void_p(ptarget_dev.data_ptr()), row_stride or ptarget_dev.shape[-1]))

    def set_generalized_force(self, tau, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        p, w = _ptr(tau)
        _ck(lib().rsb_batch_set_generalized_force(self.h, p, env_begin, n, w))

    def generalized_force(self, env_begin=0, env_count=None):
        return self._read("rsb_batch_get_generalized_force", (self.nv,), np.float32, env_begin, env_count)

    def set_control_mode(self, mode):
        _ck(lib().rsb_batch_set_control_mode(self.h, mode))

    # hot path
    def integrate1(self):
        _ck(lib().rsb_batch_integrate1(self.h))

    def integrate2(self):
        _ck(lib().rsb_batch_integrate2(self.h))

    def integrate(self, substeps=1):
        _ck(lib().rsb_batch_integrate(self.h, substeps))

    # read-backs
    def mass_matrix(self, env_begin=0, env_count=None):
        return self._read("rsb_batch_get_mass_matrix", (self.nv, self.nv), np.float32, env_begin, env_count, range_first=True)

    def nonlinearities(self, env_begin=0, env_count=None):
        return self._read("rsb_batch_get_nonlinearities", (self.nv,), np.float32, env_begin, env_count, range_first=True)

    def body_poses(self, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        R, p = np.empty((n, self.nb, 3, 3), np.float32), np.empty((n, self.nb, 3), np.float32)
        _ck(lib().rsb_batch_get_body_poses(self.h, env_begin, n, R.ctypes.data_as(C.c_void_p), p.ctypes.data_as(C.c_void_p), HOST))
        return R, p

    def contacts(self, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        out = np.empty((n, KMAX), CONTACT_DTYPE)
        cnt = np.empty(n, np.int32)
        _ck(lib().rsb_batch_get_contacts(self.h, out.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p), env_begin, n, HOST))
        return out, cnt

    def contact_points(self, env_begin=0, env_count=None):
        return self._read("rsb_batch_get_contact_points", (KMAX,), np.int32, env_begin, env_count)

    def solver_iterations(self, env_begin=0, env_count=None):
        return self._read("rsb_batch_get_solver_iterations", (), np.int32, env_begin, env_count)

    def solver_residual(self, env_begin=0, env_count=None):
        """largest impulse update of the last Gauss-Seidel sweep of every environment (< threshold: converged)"""
        return self._read("rsb_batch_get_solver_residual", (), np.float32, env_begin, env_count)

    def solver_status(self, env_begin=0, env_count=None):
        """0 converged, 1 converged on the compliant contact set (stall_reg), 2 stalled, 3 max_iter -- of the last solve"""
        return self._read("rsb_batch_get_solver_status", (), np.int32, env_begin, env_count)

    def update_kinematics(self):
        _ck(lib().rsb_batch_update_kinematics(self.h))

    def diverged(self, env_begin=0, env_count=None):
        return self._read("rsb_batch_get_diverged", (), np.int32, env_begin, env_count)

    def state_tensors(self):
        """zero-copy torch views of the batch state on its GPU: (gc [N, nq], gv [N, nv]) as strided views of the
        padded rows (SURVEY 8f N4).  Writes through these tensors are seen by the next integrate()."""
        import torch
        v = self.device_view()

        class _Raw:
            def __init__(self, ptr, rows, stride):
                self.__cuda_array_interface__ = {"shape": (rows, stride), "typestr": "<f4", "data": (int(ptr), False), "version": 2}

        gc = torch.as_tensor(_Raw(v.gc, v.num_envs, v.gc_stride), device="cuda")[:, :v.nq]
        gv = torch.as_tensor(_Raw(v.gv, v.num_envs, v.gv_stride), device="cuda")[:, :v.nv]
        return gc, gv

    def device_view(self):
        v = DeviceView()
        _ck(lib().rsb_batch_device_ptrs(self.h, C.byref(v)))
        return v

    def launch_count(self):
        return lib().rsb_batch_launch_count(self.h)

    def ob_dim(self):
        return lib().rsb_batch_ob_dim(self.h)

    def set_external_wrench(self, body, force=None, torque=None, point_body=None, env_begin=0, env_count=None):
        """setExternalForce / setExternalTorque: world-frame force / torque rows [n, 3] on `body`, applied at point_body (body
        frame, default = body origin) during the next integrate() / control_step() call only."""
        n = self._count(env_begin, env_count)
        conv = lambda a: a if (a is None or hasattr(a, "data_ptr")) else np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float32), (n, 3)))
        force, torque = conv(force), conv(torque)
        pf, w1 = _ptr(force); pt_, w2 = _ptr(torque)
        where = w1 if force is not None else w2
        assert force is None or torque is None or w1 == w2
        pp = None if point_body is None else np.ascontiguousarray(point_body, np.float32).ctypes.data_as(C.c_void_p)
        _ck(lib().rsb_batch_set_external_wrench(self.h, int(body), pf, pt_, pp, env_begin, n, where))

    def control_step(self, ptarget, substeps, obs_out, vtarget=None):
        """one RaisimGym control step for the whole batch: targets in, fused sub-steps, observations out"""
        pp, w1 = _ptr(ptarget); pv, _ = _ptr(vtarget); po, w2 = _ptr(obs_out)
        _ck(lib().rsb_batch_control_step(self.h, pp, pv, w1, substeps, po, w2))
        return obs_out

    # RaisimGym task (VectorizedEnvironment)
    def gym_configure(self, gc_init, gv_init, action_mean, action_std, foot_bodies, torque_coeff=-4e-5, forward_vel_coeff=0.3, terminal_reward=-10.0):
        f = lambda a: np.ascontiguousarray(a, np.float32)
        a, b_, c, d = f(gc_init), f(gv_init), f(action_mean), f(action_std)
        fb = np.ascontiguousarray(foot_bodies, np.int32)
        _ck(lib().rsb_batch_gym_configure(self.h, *[x.ctypes.data_as(C.c_void_p) for x in (a, b_, c, d, fb)], len(fb), torque_coeff, forward_vel_coeff, terminal_reward))

    def gym_reset(self):
        _ck(lib().rsb_batch_gym_reset(self.h))

    def gym_step(self, action, substeps, obs, reward, done):
        pa, w1 = _ptr(action); po, w2 = _ptr(obs); pr, _ = _ptr(reward); pd, _ = _ptr(done)
        _ck(lib().rsb_batch_gym_step(self.h, pa, w1, substeps, po, pr, pd, w2))

    def set_observation_peers(self, world, rank, obs_ptrs, flag_ptrs):
        """fused observation all-gather: obs_ptrs [2 * world] / flag_ptrs [world] raw device pointers valid in this process"""
        if world == 0:
            _ck(lib().rsb_batch_set_observation_peers(self.h, 0, 0, None, None)); return
        a = (C.c_void_p * (2 * world))(*[C.c_void_p(int(x)) for x in obs_ptrs])
        f = (C.c_void_p * world)(*[C.c_void_p(int(x)) for x in flag_ptrs])
        _ck(lib().rsb_batch_set_observation_peers(self.h, world, rank, a, f))

    def wait_observation_peers(self):
        """enqueue the wait for every rank's rows of the last control step; returns the buffer parity that holds them"""
        par = C.c_int()
        _ck(lib().rsb_batch_wait_observation_peers(self.h, C.byref(par)))
        return par.value

    def observe(self, out=None, env_begin=0, env_count=None):
        n = self._count(env_begin, env_count)
        if out is None:
            out = np.empty((n, self.ob_dim()), np.float32)
        p, w = _ptr(out)
        _ck(lib().rsb_batch_observe(self.h, p, env_begin, n, w))
        return out

    # terrain sensing
    def height_scan(self, frames, points_xy, out=None, out_stride=None, env_begin=0, env_count=None):
        """p_z - terrain height at the points [P, 2] of each frame's heading frame: out [n, out_stride], columns f * P + k
        (numpy: host; torch CUDA: device).  frames: frame indices (rsb_model_frame_index) or names."""
        n = self._count(env_begin, env_count)
        fr = np.ascontiguousarray([self.model.frame_index(f) if isinstance(f, str) else f for f in np.atleast_1d(frames)], np.int32)
        pts = np.ascontiguousarray(points_xy, np.float32).reshape(-1, 2)
        width = len(fr) * len(pts)
        out_stride = width if out_stride is None else out_stride
        if out is None:
            out = np.empty((n, out_stride), np.float32)
        p, w = _ptr(out)
        _ck(lib().rsb_batch_height_scan(self.h, fr.ctypes.data_as(C.c_void_p), len(fr), pts.ctypes.data_as(C.c_void_p), len(pts), p, out_stride,
                                        env_begin, n, w))
        return out

    def ray_test(self, origins, dirs, length, frames=None, out=None, env_begin=0, env_count=None):
        """first terrain crossing of o + t d/|d|, t in [0, length] -> RAY_HIT_DTYPE records.
        frames given: origins / dirs [R, 3] fixed in each frame, out [n, F, R].  frames None: world rays [n, R, 3] (numpy or torch CUDA,
        like out), out [n, R].  A torch CUDA `out` must be a uint8 / int32 / float32 tensor of 32 bytes per record."""
        n = self._count(env_begin, env_count)
        if frames is not None:
            fr = np.ascontiguousarray([self.model.frame_index(f) if isinstance(f, str) else f for f in np.atleast_1d(frames)], np.int32)
            o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3); d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
            assert o.shape == d.shape
            nr, shape = len(o), (n, len(fr), len(o))
            po, pd, pf = o.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p), fr.ctypes.data_as(C.c_void_p)
            w_in, nf = None, len(fr)
        else:
            if not hasattr(origins, "data_ptr"):
                origins = np.ascontiguousarray(origins, np.float32); dirs = np.ascontiguousarray(dirs, np.float32)
            assert tuple(origins.shape) == tuple(dirs.shape) and origins.shape[0] == n and origins.shape[-1] == 3
            (po, w_in), (pd, _) = _ptr(origins), _ptr(dirs)
            nr, shape, pf, nf = origins.shape[1], (n, origins.shape[1]), None, 0
        if out is None:
            out = np.empty(shape, RAY_HIT_DTYPE)
        p, w = _ptr(out)
        assert w_in is None or w_in == w, "world rays and the output must both be host or both be device memory"
        _ck(lib().rsb_batch_ray_test(self.h, pf, nf, po, pd, nr, length, p, env_begin, n, w))
        return out
