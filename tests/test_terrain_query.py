"""Terrain sensing: batched height scans and ray tests (rsb_batch_height_scan / rsb_batch_ray_test, World::rayTest).

The references live here: float64 numpy restatements of the surface of DESIGN.md section 2 written without the kernels' traversal.
  height_ref : the two-triangle surface of the cell under the (clamped) point, evaluated directly.
  ray_ref    : brute force -- every cell whose xy box overlaps the segment's xy bounding box, both triangles intersected at once, the
               smallest t kept under the tie rule (hits within 1e-6 m along the ray: the lower pair index wins).
The CPU tests pin the references against closed forms; the GPU tests hold the kernels to them.
"""
import ctypes
import os
import subprocess
import numpy as np
import pytest

from conftest import ROOT, RSC
from helpers import quat_to_rot

TIE = 1e-6
ANYMAL = os.path.join(RSC, "anymal_c_like.urdf")
FEET = ["LF_FOOT", "RF_FOOT", "LH_FOOT", "RH_FOOT"]


class Map:
    """height map geometry exactly as rsb_batch_set_heightmap takes it; H [ys, xs] float32 heights (evaluated in float64)"""

    def __init__(self, H, x_size, y_size, cx=0.0, cy=0.0):
        self.H = np.asarray(H, np.float32)
        self.ys, self.xs = self.H.shape
        self.x_size, self.y_size, self.cx, self.cy = x_size, y_size, cx, cy
        self.dx, self.dy = x_size / (self.xs - 1), y_size / (self.ys - 1)
        self.x0, self.y0 = cx - 0.5 * x_size, cy - 0.5 * y_size
        self.h = self.H.astype(np.float64)


def height_ref(m, x, y):
    """surface height at (x, y), points off the map clamped to the nearest border point"""
    gx = np.clip((np.asarray(x, np.float64) - m.x0) / m.dx, 0.0, m.xs - 1)
    gy = np.clip((np.asarray(y, np.float64) - m.y0) / m.dy, 0.0, m.ys - 1)
    ix = np.minimum(gx.astype(np.int64), m.xs - 2); iy = np.minimum(gy.astype(np.int64), m.ys - 2)
    fx, fy = gx - ix, gy - iy
    h00, h10, h01, h11 = m.h[iy, ix], m.h[iy, ix + 1], m.h[iy + 1, ix], m.h[iy + 1, ix + 1]
    return np.where(fx >= fy, h00 + (h10 - h00) * fx + (h11 - h10) * fy, h00 + (h11 - h01) * fx + (h01 - h00) * fy)


def ray_ref(m, o, d, length):
    """-> (t, pair, normal[3], edge distance of the hit [m], |d.n|) of the first crossing, or (inf, -1, 0, inf, 0) on a miss.
    d must be a unit vector.  Ground: pass m = ("ground", z0)."""
    o, d = np.asarray(o, np.float64), np.asarray(d, np.float64)
    if isinstance(m, tuple):
        if d[2] == 0.0:
            return np.inf, -1, np.zeros(3), np.inf, 0.0
        t = (m[1] - o[2]) / d[2]
        if 0.0 <= t <= length:
            return t, 0, np.array([0.0, 0.0, 1.0]), np.inf, abs(d[2])
        return np.inf, -1, np.zeros(3), np.inf, 0.0
    e = o + length * d
    lo = np.floor((np.minimum(o[:2], e[:2]) - (m.x0, m.y0)) / (m.dx, m.dy)).astype(int)
    hi = np.floor((np.maximum(o[:2], e[:2]) - (m.x0, m.y0)) / (m.dx, m.dy)).astype(int)
    ix = np.arange(max(lo[0], 0), min(hi[0], m.xs - 2) + 1); iy = np.arange(max(lo[1], 0), min(hi[1], m.ys - 2) + 1)
    if len(ix) == 0 or len(iy) == 0:
        return np.inf, -1, np.zeros(3), np.inf, 0.0
    IX, IY = np.meshgrid(ix, iy); IX, IY = IX.ravel(), IY.ravel()
    h00, h10, h01, h11 = m.h[IY, IX], m.h[IY, IX + 1], m.h[IY + 1, IX], m.h[IY + 1, IX + 1]
    ox, oy = o[0] - (m.x0 + IX * m.dx), o[1] - (m.y0 + IY * m.dy)
    oz = o[2] - h00
    best = (np.inf, -1, np.zeros(3), np.inf, 0.0)
    diag = m.dx * m.dy / np.hypot(m.dx, m.dy)
    for tri in (0, 1):
        ax = (h10 - h00 if tri == 0 else h11 - h01) / m.dx
        ay = (h11 - h10 if tri == 0 else h01 - h00) / m.dy
        den = d[2] - ax * d[0] - ay * d[1]
        with np.errstate(divide="ignore", invalid="ignore"):
            t = (ax * ox + ay * oy - oz) / den
        fx, fy = (ox + t * d[0]) / m.dx, (oy + t * d[1]) / m.dy
        E = 1e-9
        inside = (fx <= 1 + E) & (fy >= -E) & (fy <= fx + E) if tri == 0 else (fx >= -E) & (fy <= 1 + E) & (fx <= fy + E)
        ok = (den != 0) & (t >= 0) & (t <= length) & inside
        for k in np.nonzero(ok)[0]:
            pair = int(2 * (IY[k] * (m.xs - 1) + IX[k]) + tri)
            if t[k] < best[0] - TIE or (t[k] <= best[0] + TIE and pair < best[1]):
                n = np.array([-ax[k], -ay[k], 1.0]); n /= np.linalg.norm(n)
                if tri == 0:
                    edge = min(fy[k] * m.dy, (1 - fx[k]) * m.dx, (fx[k] - fy[k]) * diag)
                else:
                    edge = min(fx[k] * m.dx, (1 - fy[k]) * m.dy, (fy[k] - fx[k]) * diag)
                best = (float(t[k]), pair, n, abs(edge), abs(float(d @ n)))
    return best


def rough_map(seed, xs=513, ys=513, size=51.2, amp=0.10):
    """the benchmark's kind of terrain: value noise at three scales"""
    rng = np.random.default_rng(seed)

    def noise(c):
        n = (max(xs, ys) - 1) // c + 2
        lat = rng.uniform(-1, 1, (n, n))
        gx, gy = np.arange(xs) / c, np.arange(ys) / c
        i, j = gx.astype(int), gy.astype(int)
        fx, fy = (gx - i)[None, :], (gy - j)[:, None]
        return (lat[np.ix_(j, i)] * (1 - fy) * (1 - fx) + lat[np.ix_(j, i + 1)] * (1 - fy) * fx + lat[np.ix_(j + 1, i)] * fy * (1 - fx)
                + lat[np.ix_(j + 1, i + 1)] * fy * fx)
    H = noise(32) + 0.5 * noise(8) + 0.25 * noise(2)
    return Map((amp * H / np.abs(H).max()).astype(np.float32), size * (xs - 1) / 512, size * (ys - 1) / 512)


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


# ------------------------------------------------------------------ CPU: the references against closed forms -----------------------
def test_reference_flat_map_is_the_plane():
    m = Map(np.full((9, 11), 0.3, np.float32), 2.0, 1.6, 0.5, -0.2)
    rng = np.random.default_rng(1)
    x, y = rng.uniform(-3, 3, 200), rng.uniform(-3, 3, 200)          # on and off the map
    assert np.allclose(height_ref(m, x, y), np.float32(0.3), atol=1e-12)
    for _ in range(50):
        o = np.r_[rng.uniform(-0.4, 1.4), rng.uniform(-0.9, 0.5), rng.uniform(0.5, 2.0)]
        d = unit(np.r_[rng.uniform(-0.3, 0.3, 2), -1.0])
        t, pair, n, _, _ = ray_ref(m, o, d, 10.0)
        p = o + t * d
        inside = m.x0 <= p[0] <= m.x0 + m.x_size and m.y0 <= p[1] <= m.y0 + m.y_size
        if inside:
            assert abs(t - (o[2] - np.float32(0.3)) / -d[2]) < 1e-12 and np.allclose(n, [0, 0, 1])
        else:
            assert pair == -1                                           # nothing outside the map's rectangle is hit


def test_reference_single_pyramid():
    H = np.zeros((5, 5), np.float32); H[2, 2] = 1.0                     # apex at the centre vertex, dx = dy = 1
    m = Map(H, 4.0, 4.0)
    # on the diagonal x = y the apex is reached linearly along cells (1,1) and (2,2): z = 1 - |x|
    for s in (-0.9, -0.3, 0.2, 0.7):
        assert abs(height_ref(m, s, s) - (1 - abs(s))) < 1e-12
    # cell (2, 1), x in [0, 1], y in [-1, 0]: tri 1 = (P00, P11, P01) = ((0,-1,0), (1,0,0), (0,0,1)) is the plane z = 1 - x + y
    assert abs(height_ref(m, 0.25, -0.5) - 0.25) < 1e-12
    # a vertical ray onto the apex region and a horizontal one into the pyramid's face
    t, pair, n, _, _ = ray_ref(m, (0.1, 0.6, 3.0), (0, 0, -1.0), 5.0)
    assert abs(t - (3.0 - height_ref(m, 0.1, 0.6))) < 1e-12
    t, pair, n, _, _ = ray_ref(m, (-1.5, -0.2, 0.5), (1.0, 0, 0), 5.0)
    # cell (1, 1), tri 1 = ((-1,-1,0), (0,0,1), (-1,0,0)) is the plane z = 1 + x: the ray at z = 0.5 meets it at x = -0.5
    assert abs((-1.5 + t) - (-0.5)) < 1e-12 and np.allclose(n, unit([-1.0, 0.0, 1.0]), atol=1e-12)


def test_reference_ridge_at_known_angle():
    xs = 21
    H = np.tile(np.abs(np.linspace(-1.0, 1.0, xs)).astype(np.float32) * -0.5 + 0.5, (7, 1))   # ridge along y, slopes +-0.5
    m = Map(H, 2.0, 0.6)
    ang = np.deg2rad(30.0)
    d = np.array([np.cos(ang), 0.0, -np.sin(ang)])                     # descending at 30 deg towards +x, onto the face z = 0.5 + 0.5 x
    o = np.array([-0.9, 0.1, 1.0])
    t, pair, n, _, _ = ray_ref(m, o, d, 5.0)
    # o_z + t d_z = 0.5 + 0.5 (o_x + t d_x)
    t_exact = (0.5 + 0.5 * o[0] - o[2]) / (d[2] - 0.5 * d[0])
    assert abs(t - t_exact) < 1e-7 and np.allclose(n, unit([-0.5, 0.0, 1.0]), atol=1e-7)     # the heights are float32 roundings of the ridge


def test_reference_ray_from_below_hits_from_below():
    m = Map(np.full((6, 6), 0.2, np.float32), 1.0, 1.0)
    t, pair, n, _, _ = ray_ref(m, (0.05, -0.1, -0.3), unit((0.1, 0.05, 1.0)), 2.0)
    assert pair >= 0 and abs((-0.3 + t * unit((0.1, 0.05, 1.0))[2]) - np.float32(0.2)) < 1e-12 and n[2] > 0
    assert ray_ref(("ground", 0.0), (0, 0, -1.0), (0, 0, 1.0), 2.0)[0] == 1.0
    assert ray_ref(("ground", 0.0), (0, 0, -1.0), (0, 0, 1.0), 0.5)[1] == -1


def test_ray_hit_layout():
    from raisimlib_b200 import capi
    assert ctypes.sizeof(capi.RayHit) == 32 and capi.RAY_HIT_DTYPE.itemsize == 32


def test_argument_errors_without_gpu():
    """validation comes before any device work: errors with messages, no crash"""
    from raisimlib_b200 import capi
    L = capi.lib()
    f = (ctypes.c_int32 * 1)(0); pts = (ctypes.c_float * 2)(0, 0); out = (ctypes.c_float * 4)()
    assert L.rsb_batch_height_scan(None, f, 1, pts, 1, out, 1, 0, 1, capi.HOST) == capi_err(capi, "null batch")
    hits = (capi.RayHit * 1)()
    o = (ctypes.c_float * 3)(0, 0, 1); d = (ctypes.c_float * 3)(0, 0, -1)
    assert L.rsb_batch_ray_test(None, None, 0, o, d, 1, 1.0, hits, 0, 1, capi.HOST) == capi_err(capi, "null batch")


def capi_err(capi, text):
    assert text in capi.lib().rsb_last_error().decode()
    return -1


# ------------------------------------------------------------------ GPU -------------------------------------------------------------
@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from raisimlib_b200 import capi as c
    return c


def _frame(capi, model, f):
    body, pos, rot = ctypes.c_int(), np.zeros(3), np.zeros(9)
    capi.lib().rsb_model_frame(model.h, f, ctypes.byref(body), pos.ctypes.data_as(ctypes.c_void_p), rot.ctypes.data_as(ctypes.c_void_p))
    return body.value, pos, rot.reshape(3, 3)


def _frame_poses(capi, bt, frames, gc32):
    """world pose (p [n, F, 3], R [n, F, 3, 3]) of each frame: body 0 from the gc rows, the others from body_poses()"""
    n = len(gc32)
    Rb, pb = bt.body_poses()
    Rb, pb = Rb.astype(np.float64), pb.astype(np.float64)
    P, R = np.zeros((n, len(frames), 3)), np.zeros((n, len(frames), 3, 3))
    for j, f in enumerate(frames):
        body, fpos, frot = _frame(capi, bt.model, f)
        for e in range(n):
            if body == 0:
                Rw, pw = quat_to_rot(gc32[e, 3:7].astype(np.float64)), gc32[e, 0:3].astype(np.float64)
            else:
                Rw, pw = Rb[e, body], pb[e, body]
            P[e, j], R[e, j] = pw + Rw @ fpos, Rw @ frot
    return P, R


def _random_state(rng, n, m, z=(0.55, 0.75), tilt=0.3):
    gc = np.tile(np.array([0, 0, 0.6, 1, 0, 0, 0, 0.03, 0.4, -0.8, -0.03, 0.4, -0.8, 0.03, -0.4, 0.8, -0.03, -0.4, 0.8]), (n, 1))
    gc[:, 0] = rng.uniform(m.x0 + 1.0, m.x0 + m.x_size - 1.0, n); gc[:, 1] = rng.uniform(m.y0 + 1.0, m.y0 + m.y_size - 1.0, n)
    gc[:, 2] = rng.uniform(*z, n)
    yaw, roll, pitch = rng.uniform(-np.pi, np.pi, n), rng.uniform(-tilt, tilt, n), rng.uniform(-tilt, tilt, n)
    cy, sy, cr, sr, cp, sp = np.cos(yaw / 2), np.sin(yaw / 2), np.cos(roll / 2), np.sin(roll / 2), np.cos(pitch / 2), np.sin(pitch / 2)
    gc[:, 3:7] = np.c_[cr * cp * cy + sr * sp * sy, sr * cp * cy - cr * sp * sy, cr * sp * cy + sr * cp * sy, cr * cp * sy - sr * sp * cy]
    gc[:, 7:] += rng.uniform(-0.3, 0.3, (n, 12))
    return gc.astype(np.float32), np.zeros((n, 18), np.float32)


def _scan_ref(m_of_env, P, R, pts):
    """p_z - height at p + Rz(yaw) [x, y]; P [n, F, 3], R [n, F, 3, 3], pts [K, 2] -> [n, F * K]"""
    n, F = P.shape[:2]
    yaw = np.arctan2(R[..., 1, 0], R[..., 0, 0])
    c, s = np.cos(yaw)[..., None], np.sin(yaw)[..., None]
    x = P[..., 0:1] + c * pts[:, 0] - s * pts[:, 1]
    y = P[..., 1:2] + s * pts[:, 0] + c * pts[:, 1]
    out = np.empty((n, F, len(pts)))
    for e in range(n):
        out[e] = P[e, :, 2:3] - height_ref(m_of_env(e), x[e], y[e])
    return out.reshape(n, -1)


BASE_GRID = np.stack(np.meshgrid(0.1 * np.arange(-8, 9), 0.1 * np.arange(-5, 6)), -1).reshape(-1, 2)       # 17 x 11, 0.1 m pitch
FOOT_RING = np.stack([0.1 * np.cos(np.arange(8) * np.pi / 4), 0.1 * np.sin(np.arange(8) * np.pi / 4)], -1)


@pytest.mark.gpu
def test_height_scan_bench_map_base_and_feet(capi):
    n = 4096
    m = rough_map(11)
    rng = np.random.default_rng(12)
    gc, gv = _random_state(rng, n, m)
    gc[:8, 0] = m.x0 + 0.05; gc[8:16, 1] = m.y0 + m.y_size - 0.05     # robots at the border: part of every pattern lies off the map
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_heightmap(m.xs, m.ys, m.x_size, m.y_size, m.cx, m.cy, m.H)
    bt.set_state(gc, gv)
    pts = np.r_[BASE_GRID, [[60.0, 0.0], [0.0, -70.0]]].astype(np.float32)
    frames = [bt.model.frame_index(f) for f in ["base"] + FEET]
    got = bt.height_scan(frames, pts)
    P, R = _frame_poses(capi, bt, frames, gc)
    ref = _scan_ref(lambda e: m, P, R, pts.astype(np.float64))
    err = np.abs(got - ref).max()
    print(f"height scan, 4096 envs x 5 frames x {len(pts)} points: max |error| {err:.2e} m")
    assert err < 2e-5       # float32 world coordinates up to 26 m (ulp 2e-6) times slopes < 1, plus float32 heights on both sides


@pytest.mark.gpu
def test_height_scan_terrain_atlas(capi):
    n, maps = 512, [rough_map(20 + k, xs=129, ys=129, size=51.2) for k in range(3)]
    rng = np.random.default_rng(21)
    m0 = maps[0]
    gc, gv = _random_state(rng, n, m0)
    map_of_env = rng.integers(0, 3, n).astype(np.int32)
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_heightmaps(m0.x_size, m0.y_size, 0.0, 0.0, np.stack([mm.H for mm in maps]), map_of_env)
    bt.set_state(gc, gv)
    frames = [bt.model.frame_index(f) for f in ["base", "LF_FOOT"]]
    got = bt.height_scan(frames, FOOT_RING.astype(np.float32))
    P, R = _frame_poses(capi, bt, frames, gc)
    ref = _scan_ref(lambda e: maps[map_of_env[e]], P, R, FOOT_RING)
    assert np.abs(got - ref).max() < 2e-5


def _check_rays(hits, refs, label, dist_tol=1e-4):
    """hit / miss and pair identical, |d distance|, |d position| <= dist_tol except near-edge or grazing reference hits; returns
    (excluded, rays) for the caller's bound on the excluded fraction"""
    excluded, checked = 0, 0
    for h, (t, pair, n, edge, dn, o, d) in zip(hits, refs):
        if pair >= 0 and (edge < 1e-4 or dn < 0.05):
            excluded += 1
            continue
        checked += 1
        assert h["pair_index"] == pair, (label, h, t, pair, o, d)
        if pair >= 0:
            assert abs(h["distance"] - t) <= dist_tol, (label, h["distance"], t)
            assert np.abs(h["position"] - (o + t * d)).max() <= dist_tol
            assert np.abs(h["normal"] - n).max() < 1e-5
        else:
            assert np.isinf(h["distance"]) and not h["position"].any() and not h["normal"].any()
    frac = excluded / max(1, len(refs))
    print(f"[{label}] rays {len(refs)}: checked {checked}, near-edge / grazing excluded {excluded} ({100 * frac:.2f} %)")
    return excluded, len(refs)


# The 1e-4 m band inside the three edges of a triangle with 0.1 m legs covers 1e-4 x 0.341 m / 0.005 m^2 = 0.68 % of its area: a set
# of rays that nearly all hit loses ~0.7 % to the edge rule alone, so the 1 % bound holds for all rays of a test together, not for
# every subset of a few hundred.
def _bound_excluded(counts):
    excluded, total = map(sum, zip(*counts))
    print(f"excluded in all: {excluded} of {total} rays ({100 * excluded / total:.2f} %)")
    assert excluded < 0.01 * total


def _ray_dirs(rng, k, special=True):
    """random unit directions (|d_z| >= 0.1: a random near-horizontal ray grazes rough terrain too often to be a fair check), the first
    ones replaced by vertical, axis-parallel and cell-diagonal directions"""
    d = unit(rng.standard_normal((k, 3)))
    d[:, 2] = np.where(np.abs(d[:, 2]) < 0.1, np.copysign(0.1, d[:, 2]), d[:, 2])
    d = unit(d)
    if not special:
        return d
    special = unit(np.array([[0, 0, -1], [0, 0, 1], [1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [1, 1, 0], [1, 1, -1], [-1, 1, -0.5],
                             [0.1, 0.0, -1], [0.0, 0.1, -1], [1, 0, -0.3], [0, -1, -0.3], [1, 1, -0.2]], np.float64))
    d[:min(k, len(special))] = special[:k]
    return d


@pytest.mark.gpu
def test_ray_test_world_and_frame_rays_against_brute_force(capi):
    m = rough_map(31, xs=257, ys=193, size=25.6)
    n = 48
    rng = np.random.default_rng(32)
    gc, gv = _random_state(rng, n, m)
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_heightmap(m.xs, m.ys, m.x_size, m.y_size, m.cx, m.cy, m.H)
    bt.set_state(gc, gv)
    R_ = 64
    # world rays: origins above and below the surface and off the map, every kind of direction, lengths up to 10 m
    o = np.empty((n, R_, 3)); d = np.empty((n, R_, 3))
    for e in range(n):
        o[e, :, 0] = rng.uniform(m.x0 - 3, m.x0 + m.x_size + 3, R_); o[e, :, 1] = rng.uniform(m.y0 - 3, m.y0 + m.y_size + 3, R_)
        o[e, :, 2] = height_ref(m, o[e, :, 0], o[e, :, 1]) + rng.uniform(-0.5, 2.0, R_)
        d[e] = _ray_dirs(rng, R_, special=e % 4 == 0)
    o32, d32 = o.astype(np.float32), d.astype(np.float32)
    o64, d64 = o32.astype(np.float64), unit(d32.astype(np.float64))
    counts = []
    for length in (10.0, 1.5):
        hits = bt.ray_test(o32, d32, length)
        refs = [ray_ref(m, o64[e, k], d64[e, k], length) + (o64[e, k], d64[e, k]) for e in range(n) for k in range(R_)]
        counts.append(_check_rays(hits.reshape(-1), refs, f"world rays, length {length}"))
        assert (hits["pair_index"] >= 0).sum() > 0.1 * hits.size          # about half the directions point up, many of those miss
    # rays fixed in frames: a lidar-like fan on the base and a downward probe on a foot
    frames = [bt.model.frame_index("base"), bt.model.frame_index("LF_FOOT")]
    fo = rng.uniform(-0.3, 0.3, (16, 3)).astype(np.float32)
    fd = np.c_[rng.uniform(-0.6, 0.6, (16, 2)), rng.uniform(-1.0, -0.6, 16)].astype(np.float32)     # steep enough not to graze after the base's tilt
    fd[0] = (0, 0, -1); fd[1] = (1, 0, -0.5)
    hits = bt.ray_test(fo, fd, 10.0, frames=frames)
    assert hits.shape == (n, 2, 16)
    P, Rw = _frame_poses(capi, bt, frames, gc)
    refs = []
    for e in range(n):
        for j in range(2):
            for k in range(16):
                oo, dd = P[e, j] + Rw[e, j] @ fo[k], Rw[e, j] @ unit(fd[k].astype(np.float64))
                refs.append(ray_ref(m, oo, dd, 10.0) + (oo, dd))
    # the reference frame poses are float32 poses re-evaluated in float64: 1e-6 rad of rotation moves a 10 m ray's end by 1e-5 m
    counts.append(_check_rays(hits.reshape(-1), refs, "frame rays"))
    _bound_excluded(counts)


@pytest.mark.gpu
def test_ray_test_tile_skipping_spike_and_ridges(capi):
    xs = ys = 129
    H = np.zeros((ys, xs), np.float32)
    H[64, 64] = 1.5                                    # one tall spike in the middle of a tile
    H[:, 40] = 0.4; H[48, :] = 0.3                     # ridges on tile boundaries (8-cell tiles: vertex 40 and 48 are tile edges)
    m = Map(H, 12.8, 12.8)
    bt = capi.Batch(capi.Model(ANYMAL), 1)
    bt.set_heightmap(xs, ys, m.x_size, m.y_size, 0.0, 0.0, H)
    rng = np.random.default_rng(41)
    k = 3000
    sx, sy = m.x0 + 64 * m.dx, m.y0 + 64 * m.dy
    o = np.empty((k, 3)); d = np.empty((k, 3))
    # rays skimming past the spike at heights 0 .. 1.6, horizontal or nearly so, from all sides
    a = rng.uniform(0, 2 * np.pi, k); off = rng.uniform(-0.15, 0.15, k)
    o[:, 0] = sx - 3 * np.cos(a) - off * np.sin(a); o[:, 1] = sy - 3 * np.sin(a) + off * np.cos(a); o[:, 2] = rng.uniform(0.0, 1.6, k)
    d[:, 0], d[:, 1], d[:, 2] = np.cos(a), np.sin(a), rng.uniform(-0.3, -0.06, k)      # |d.n| >= 0.05 on the flat ground
    # every fourth ray crosses tile corners: along the diagonal through vertex (40, 48)
    c = np.arange(0, k, 4)
    o[c, 0] = m.x0 + 40 * m.dx - 2.0; o[c, 1] = m.y0 + 48 * m.dy - 2.0 + rng.uniform(-0.02, 0.02, len(c)); o[c, 2] = rng.uniform(0.05, 0.6, len(c))
    d[c] = np.c_[np.ones(len(c)), np.ones(len(c)), rng.uniform(-0.2, -0.08, len(c))]
    o32, d32 = o.astype(np.float32)[None], d.astype(np.float32)[None]
    hits = bt.ray_test(o32, d32, 8.0)
    o64, d64 = o32[0].astype(np.float64), unit(d32[0].astype(np.float64))
    refs = [ray_ref(m, o64[i], d64[i], 8.0) + (o64[i], d64[i]) for i in range(k)]
    n_spike = sum(1 for r in refs if r[1] >= 0 and abs(r[0] - 3.0) < 0.5)
    print(f"rays that hit the spike: {n_spike}")
    assert n_spike > 50
    # grazing along a ridge crest is legitimately ambiguous: those rays are excluded like the near-edge ones (< 1 %)
    _bound_excluded([_check_rays(hits.reshape(-1), refs, "spike / ridges")])


@pytest.mark.gpu
def test_ground_closed_form_and_flat_map_equal_plane(capi):
    n = 64
    rng = np.random.default_rng(51)
    o = np.c_[rng.uniform(-5, 5, (n * 32, 2)), rng.uniform(-1, 3, n * 32)].reshape(n, 32, 3).astype(np.float32)
    d = _ray_dirs(rng, n * 32).reshape(n, 32, 3).astype(np.float32)
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_ground(0.2)
    g = bt.ray_test(o, d, 10.0)
    o64, d64 = o.astype(np.float64), unit(d.astype(np.float64))
    with np.errstate(divide="ignore", invalid="ignore"):
        t = (0.2 - o64[..., 2]) / d64[..., 2]
    hit = (t >= 0) & (t <= 10.0)
    t = np.where(hit, t, 0.0)
    assert np.array_equal(g["pair_index"] == 0, hit) and (g["pair_index"][~hit] == -1).all()
    assert np.abs(g["distance"][hit] - t[hit]).max() < 1e-5
    assert np.allclose(g["normal"][hit], [0, 0, 1]) and np.abs(g["position"][hit][:, 2] - 0.2).max() < 1e-5
    # a flat height map gives the plane's distances wherever the hit lies on the map
    bt.set_heightmap(101, 101, 20.0, 20.0, 0.0, 0.0, np.full((101, 101), 0.2, np.float32))
    h = bt.ray_test(o, d, 10.0)
    on_map = hit & (np.abs(o64[..., 0] + t * d64[..., 0]) < 9.99) & (np.abs(o64[..., 1] + t * d64[..., 1]) < 9.99)
    on_map &= np.abs(d64[..., 2]) > 0.05
    assert (h["pair_index"][on_map] >= 0).all() and np.abs(h["distance"][on_map] - g["distance"][on_map]).max() < 1e-5
    # height scans on the Ground: p_z - z0
    gc, gv = _random_state(rng, n, Map(np.zeros((3, 3), np.float32), 10.0, 10.0))
    bt.set_ground(0.2); bt.set_state(gc, gv)
    s = bt.height_scan([0], BASE_GRID.astype(np.float32))
    assert np.array_equal(s, np.repeat((gc[:, 2] - np.float32(0.2))[:, None], len(BASE_GRID), 1))


@pytest.mark.gpu
def test_terrain_query_contract(capi):
    import torch
    n = 256
    m = rough_map(61, xs=257, ys=257, size=25.6)
    rng = np.random.default_rng(62)
    gc, gv = _random_state(rng, n, m, z=(0.5, 0.6))
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_heightmap(m.xs, m.ys, m.x_size, m.y_size, m.cx, m.cy, m.H)
    bt.set_state(gc, gv)
    kp = np.r_[np.zeros(6), 300.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 8.0 * np.ones(12)]
    bt.set_pd_gains(kp, kd); bt.set_pd_target(gc, np.zeros_like(gv))
    bt.integrate(4)
    c0, n0 = bt.contacts(); s0 = bt.get_state(); it0, st0 = bt.solver_iterations(), bt.solver_status()
    base, feet = [bt.model.frame_index("base")], [bt.model.frame_index(f) for f in FEET]
    pts = BASE_GRID.astype(np.float32)
    # launch counts: a base scan is one launch; a foot scan after a state change is a kinematics launch and the scan
    l0 = bt.launch_count(); a = bt.height_scan(base, pts); assert bt.launch_count() == l0 + 1
    l0 = bt.launch_count(); bt.height_scan(feet, FOOT_RING.astype(np.float32)); assert bt.launch_count() == l0 + 2
    l0 = bt.launch_count(); bt.height_scan(feet, FOOT_RING.astype(np.float32)); assert bt.launch_count() == l0 + 1
    # bit-identical repeats, sub-ranges and host / device outputs
    assert np.array_equal(a, bt.height_scan(base, pts))
    assert np.array_equal(a[37:37 + 50], bt.height_scan(base, pts, env_begin=37, env_count=50))
    dev = torch.empty((n, len(pts)), dtype=torch.float32, device="cuda")
    bt.height_scan(base, pts, out=dev); bt.sync()
    assert np.array_equal(a, dev.cpu().numpy())
    # out_stride: the scan goes into columns of a wider buffer, the other columns keep their sentinel
    width = len(pts) + 7
    wide = torch.full((n, width), -7.0, dtype=torch.float32, device="cuda")
    bt.height_scan(base, pts, out=wide, out_stride=width); bt.sync()
    w = wide.cpu().numpy()
    assert np.array_equal(w[:, :len(pts)], a) and (w[:, len(pts):] == -7.0).all()
    wh = np.full((n, width), -7.0, np.float32)
    bt.height_scan(base, pts, out=wh, out_stride=width)
    assert np.array_equal(wh, w)
    o = np.c_[gc[:, :2], gc[:, 2:3] + 1.0][:, None, :].repeat(8, 1).astype(np.float32)
    d = _ray_dirs(rng, 8)[None].repeat(n, 0).astype(np.float32)
    r1 = bt.ray_test(o, d, 5.0)
    assert r1.tobytes() == bt.ray_test(o, d, 5.0).tobytes()
    assert r1[10:30].tobytes() == bt.ray_test(o[10:30], d[10:30], 5.0, env_begin=10, env_count=20).tobytes()
    rdev = torch.empty((n, 8, 8), dtype=torch.int32, device="cuda")
    bt.ray_test(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), 5.0, out=rdev); bt.sync()
    assert rdev.cpu().numpy().tobytes() == r1.tobytes()
    # nothing of the last integrate() changed
    c1, n1 = bt.contacts(); s1 = bt.get_state()
    assert np.array_equal(n0, n1) and c0.tobytes() == c1.tobytes() and all(np.array_equal(x, y) for x, y in zip(s0, s1))
    assert np.array_equal(it0, bt.solver_iterations()) and np.array_equal(st0, bt.solver_status())
    # errors
    for call, msg in ((lambda: bt.height_scan([999], pts), "bad frame index"),
                      (lambda: bt.height_scan(base, pts, out_stride=3), "out_stride"),
                      (lambda: bt.ray_test(o, np.zeros_like(d), 5.0), "zero or non-finite ray direction"),
                      (lambda: bt.ray_test(o, d, 0.0), "length"),
                      (lambda: bt.ray_test(o[:4], d[:4], 1.0, env_begin=n - 2, env_count=4), "out of bounds")):
        with pytest.raises(capi.RsbError, match=msg):
            call()
    bt.clear_terrain()
    with pytest.raises(capi.RsbError, match="no terrain"):
        bt.height_scan(base, pts)
    assert (bt.ray_test(o, d, 5.0)["pair_index"] == -1).all()          # no terrain: all misses


@pytest.mark.gpu
def test_height_scan_after_gym_step_describes_the_new_state(capi):
    import torch
    n = 512
    m = rough_map(71, xs=257, ys=257, size=25.6)
    rng = np.random.default_rng(72)
    gc, gv = _random_state(rng, n, m, z=(0.6, 0.62), tilt=0.05)
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_heightmap(m.xs, m.ys, m.x_size, m.y_size, m.cx, m.cy, m.H)
    bt.set_state(gc, gv)
    kp = np.r_[np.zeros(6), 300.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 8.0 * np.ones(12)]
    bt.set_pd_gains(kp, kd)
    gc_init = gc[0].copy(); gc_init[2] = 3.0                             # a reset puts the robot 3 m up: easy to tell apart
    bt.gym_configure(gc_init, np.zeros(18, np.float32), gc_init[7:], np.full(12, 0.5, np.float32), [3, 6, 9, 12])
    act = torch.zeros((n, 12), dtype=torch.float32, device="cuda")
    obs = torch.empty((n, bt.ob_dim()), dtype=torch.float32, device="cuda")
    rew = torch.empty(n, dtype=torch.float32, device="cuda"); done = torch.empty(n, dtype=torch.uint8, device="cuda")
    frames = [bt.model.frame_index("base"), bt.model.frame_index("RH_FOOT")]
    for _ in range(3):
        bt.gym_step(act, 4, obs, rew, done)
        got = bt.height_scan(frames, FOOT_RING.astype(np.float32))
        g, _ = bt.get_state()
        P, R = _frame_poses(capi, bt, frames, g)
        assert np.abs(got - _scan_ref(lambda e: m, P, R, FOOT_RING)).max() < 2e-5


@pytest.mark.gpu
def test_pybind_equals_capi_and_facade_example(capi):
    import torch
    from raisimlib_b200 import _rsb_py
    n = 128
    m = rough_map(81, xs=129, ys=129, size=12.8)
    rng = np.random.default_rng(82)
    gc, gv = _random_state(rng, n, m)
    bt = capi.Batch(capi.Model(ANYMAL), n)
    bt.set_heightmap(m.xs, m.ys, m.x_size, m.y_size, 0.0, 0.0, m.H)
    bt.set_state(gc, gv)
    pb = _rsb_py.Batch(_rsb_py.Model(ANYMAL), n, 0)
    pb.set_heightmap(m.xs, m.ys, m.x_size, m.y_size, 0.0, 0.0, m.H.ravel().tolist())
    torch.from_dlpack(pb.gc()).copy_(torch.from_numpy(gc).cuda()); torch.from_dlpack(pb.gv()).copy_(torch.from_numpy(gv).cuda())
    torch.cuda.synchronize()
    pb.update_kinematics()
    frames = [bt.model.frame_index(f) for f in ["base", "LH_FOOT"]]
    pts = FOOT_RING.astype(np.float32)
    out = torch.empty((n, 2 * len(pts)), dtype=torch.float32, device="cuda")
    pb.height_scan(frames, pts.ravel().tolist(), out.data_ptr()); pb.sync()
    assert np.array_equal(out.cpu().numpy(), bt.height_scan(frames, pts))
    fo = np.array([[0.2, 0.0, 0.0], [0.0, 0.1, 0.0]], np.float32); fd = np.array([[1.0, 0.0, -1.0], [0.0, 0.0, -1.0]], np.float32)
    rh = torch.empty((n, 2, 2, 8), dtype=torch.int32, device="cuda")
    pb.ray_test(frames, fo.ravel().tolist(), fd.ravel().tolist(), 4.0, rh.data_ptr()); pb.sync()
    assert rh.cpu().numpy().tobytes() == bt.ray_test(fo, fd, 4.0, frames=frames).tobytes()
    o = torch.from_numpy(np.c_[gc[:, :3]][:, None, :].repeat(3, 1)).cuda().contiguous(); d = torch.tensor([[1.0, 0.2, -1.0]] * 3).expand(n, 3, 3).cuda().contiguous()
    rw = torch.empty((n, 3, 8), dtype=torch.int32, device="cuda")
    pb.ray_test_world(o.data_ptr(), d.data_ptr(), 3, 4.0, rw.data_ptr()); pb.sync()
    assert rw.cpu().numpy().tobytes() == bt.ray_test(o.cpu().numpy(), d.cpu().numpy(), 4.0).tobytes()
    exe = os.path.join(ROOT, "examples", "terrain_sensing")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    r = subprocess.run([exe, ANYMAL], capture_output=True, text=True, cwd=ROOT)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
