"""GPU parity tests (run on the B200 box: pytest -m gpu).  Everything goes through the C-ABI
(raisimlib_b200/librsb.so) and is compared with the CPU oracle on the same seeded inputs.

Tolerances (float32 kernel vs float64 oracle) are written next to each assertion.  Integer results
-- contact counts, candidate-point / body / terrain-pair indices -- must match BIT-EXACTLY, except
for candidates whose |depth| is below MARGIN in the oracle (a float32 rounding of the pose can move
those across zero; they are counted and excluded, see DESIGN.md "parity").

PARITY UNPINNED: the oracle restates the published algorithms; no RaiSim artefact exists to pin it
(SURVEY.md 8c).  "Matches the in-repo CPU oracle", not "matches RaiSim".
"""
import os
import numpy as np
import pytest

from conftest import RSC
from helpers import ANYMAL_GC0, PENDULUM_URDF, SPHERE_URDF, BOX_URDF, random_state
from oracle.oracle import Oracle
from oracle.urdf_tables import load_tables

pytestmark = pytest.mark.gpu

MARGIN = 2e-6          # metres; contact candidates shallower than this are excluded from index parity
THRESH = 1e-6          # solver threshold used on both sides


@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from raisimlib_b200 import capi as c
    return c


def _setup(capi, urdf, n, seed, terrain="ground", base_z=0.45, vel=0.5, tau_scale=20.0, params=None, joint_scale=0.5):
    path = os.path.join(RSC, urdf) if urdf.endswith(".urdf") else urdf
    t = load_tables(path)
    m = capi.Model(path)
    bt = capi.Batch(m, n)
    rng = np.random.default_rng(seed)
    gc, gv = random_state(t, rng, n, vel_scale=vel, base_z=base_z, pos_scale=2.0, joint_scale=joint_scale)
    tau = rng.uniform(-tau_scale, tau_scale, (n, t["nv"]))
    if t["floating"]:
        tau[:, :6] = 0
    prm = dict(threshold=THRESH)     # everything else at the library defaults = what bench.py runs (accelerated sweeps, stagnation
                                     # window 8 with the compliant fallback); tests of the plain published method pass accel_m=0, stall_window=0
    prm.update(params or {})
    o64, o32 = Oracle(t, params=prm), Oracle(t, precision="f32", params=prm)
    bt.set_params(**{k: v for k, v in prm.items() if k not in ("gx", "gy", "gz")})
    if any(k in prm for k in ("gx", "gy", "gz")):
        bt.set_params(gravity=(prm.get("gx", 0.0), prm.get("gy", 0.0), prm.get("gz", -9.81)))
    if terrain == "ground":
        for o in (o64, o32):
            o.set_ground(0.0)
        bt.set_ground(0.0)
    elif terrain == "hm":
        xs, ys = 65, 49
        H = (0.1 * rng.uniform(-1, 1, (ys, xs))).astype(np.float32)
        for o in (o64, o32):
            o.set_heightmap(xs, ys, 12.8, 9.6, 0.1, -0.2, H.astype(np.float64))
        bt.set_heightmap(xs, ys, 12.8, 9.6, 0.1, -0.2, H)
    gc32, gv32, tau32 = gc.astype(np.float32), gv.astype(np.float32), tau.astype(np.float32)
    bt.set_control_mode(capi.FORCE_AND_TORQUE)
    bt.set_state(gc32, gv32)
    bt.set_generalized_force(tau32)
    return t, bt, o64, o32, gc32.astype(np.float64), gv32.astype(np.float64), tau32.astype(np.float64)


def _index_parity(pts_gpu, cnt_gpu, d_ref, label):
    """bit-exact contact lists, excluding environments that hold a candidate inside the margin."""
    n = len(cnt_gpu)
    shallow = (np.abs(d_ref["c_depth"]) < MARGIN) & (d_ref["c_pt"] >= 0)
    ok_env = ~shallow.any(1)
    excluded = int((~ok_env).sum())
    mism = (pts_gpu != d_ref["c_pt"]).any(1) | (cnt_gpu != d_ref["ncontacts"])
    # an environment may only mismatch if it has a margin candidate in the reference ...
    hard = mism & ok_env
    # ... or a candidate that the reference rejected by less than the margin (not recorded): allow
    # those only if the contact COUNT differs by the extra near-zero candidates
    print(f"[{label}] envs={n} contacts={int(cnt_gpu.sum())} margin-excluded envs={excluded} mismatching={int(mism.sum())}")
    return hard


@pytest.mark.parametrize("urdf,base_z", [("anymal_c_like.urdf", 0.45), ("atlas_like.urdf", 0.9), (PENDULUM_URDF, 0.0)])
def test_stage_outputs_fk_crba_rnea(capi, urdf, base_z):
    """a2 FK, a3 CRBA, a4 RNEA through integrate1() + the lazy getters."""
    t, bt, o64, o32, gc, gv, tau = _setup(capi, urdf, 128, seed=11, base_z=base_z, tau_scale=1.0)
    bt.integrate1()
    M, h = bt.mass_matrix(), bt.nonlinearities()
    R, p = bt.body_poses()
    a, b = gc.copy(), gv.copy()
    d = o64.step(a, b, tau_ff=tau, debug=True)
    Ms, hs = np.abs(d["M"]).max(), np.abs(d["h"]).max()
    eM, eh = np.abs(M - d["M"]).max(), np.abs(h - d["h"]).max()
    eR, ep = np.abs(R - d["R"]).max(), np.abs(p - d["p"]).max()
    print(f"stage errors: M {eM:.2e}/{Ms:.1e}  h {eh:.2e}/{hs:.1e}  R {eR:.2e}  p {ep:.2e}")
    assert eR < 3e-6 and ep < 5e-6                     # float32 pose chain, depth <= 10
    assert eM < 2e-6 * Ms                               # relative to the largest entry (total mass)
    assert eh < 2e-6 * max(hs, 1.0) * 10
    assert np.allclose(M, np.transpose(M, (0, 2, 1)))   # symmetric by construction


@pytest.mark.parametrize("terrain", ["ground", "hm"])
def test_contact_indices_bit_exact(capi, terrain):
    """a6 narrow phase: counts, candidate-point ids, body ids and terrain pair ids must be identical."""
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", 1024, seed=21, terrain=terrain)
    bt.integrate1()
    ct, cnt = bt.contacts()
    pts = bt.contact_points()
    a, b = gc.copy(), gv.copy()
    d32 = o32.step(a, b, tau_ff=tau, debug=True)
    hard = _index_parity(pts, cnt, d32, "f32 oracle " + terrain)
    assert not hard.any(), f"contact lists differ in envs {np.where(hard)[0][:10]}"
    same = (pts == d32["c_pt"]).all(1)
    assert same.mean() > 0.99
    assert cnt.sum() > 1000
    assert (ct["local_body"][same] == d32["c_body"][same]).all()
    assert (ct["pair_index"][same] == d32["c_pair"][same]).all()
    live = same[:, None] & (d32["c_pt"] >= 0)
    assert np.abs(ct["depth"] - d32["c_depth"])[live].max() < 2e-6
    # a sphere's normal is (centre - closest terrain point) / distance: rounding of the pose (1e-7 m) over a distance of r - depth
    rad = np.where(d32["c_pt"] >= 0, t["pt_rad"][np.maximum(d32["c_pt"], 0)], 0.0)
    tol_n = 2e-6 + 4e-7 / np.maximum(rad - d32["c_depth"], 1e-4)
    assert (np.abs(ct["normal"] - d32["c_normal"]).max(2)[live] < tol_n[live]).all()
    assert (np.abs(ct["position"] - d32["c_pos"]).max(2)[live] < 5e-6 + rad[live] * tol_n[live]).all()
    if terrain == "hm":
        assert len(np.unique(ct["pair_index"][live])) > 100   # many different cells / both triangles


@pytest.mark.parametrize("urdf,terrain,base_z,tau_scale", [
    ("anymal_c_like.urdf", "ground", 0.45, 20.0),
    ("anymal_c_like.urdf", "hm", 0.45, 20.0),
    ("atlas_like.urdf", "ground", 0.9, 2.0),
])
def test_one_step_state_and_impulses(capi, urdf, terrain, base_z, tau_scale):
    """a1 whole step from the same state: gc+, gv+ and contact impulses."""
    n = 512
    t, bt, o64, o32, gc, gv, tau = _setup(capi, urdf, n, seed=31, terrain=terrain, base_z=base_z, tau_scale=tau_scale)
    bt.integrate(1)
    g1, v1 = bt.get_state()
    ct, cnt = bt.contacts()
    pts = bt.contact_points()
    it = bt.solver_iterations()
    a, b = gc.copy(), gv.copy()
    d = o64.step(a, b, tau_ff=tau, debug=True)
    assert np.isfinite(g1).all() and np.isfinite(v1).all()
    # compare where both solvers converged on the same contact set; cycling Gauss-Seidel cases
    # (both sides hit max_iter; see DESIGN.md "solver convergence") have no unique answer
    st = bt.solver_status()
    same = (pts == d["c_pt"]).all(1)
    conv = same & (st == 0) & (d["status"] == 0)
    print(f"same-contact envs {same.sum()}/{n}, of those converged on both sides {conv.sum()}; solver status gpu {np.bincount(st, minlength=4).tolist()} oracle "
          f"{np.bincount(d['status'], minlength=4).tolist()} (converged / on the compliant set / stalled / max_iter); K mean {cnt.mean():.2f}; sweeps gpu {it.mean():.1f} oracle {d['iters'].mean():.1f}")
    # Random orientations half inside the ground (a whole leg under the surface): the per-contact rule cycles on a few % of these
    # unphysical states; they finish on the compliant contact set (status 1) and are compared separately.  Round 1 excluded up
    # to 10 % here; the physical regimes (standing, fallen, humanoid on box feet) have their own tests below.
    assert (st >= 2).mean() < 0.05 and (d["status"] >= 2).mean() < 0.05        # these unphysical drops: < 5 % end without converging
    assert conv.mean() > 0.88
    ev = np.abs(v1 - b)[conv]; eq = np.abs(g1 - a)[conv]
    scale_v = 1.0 + np.abs(b[conv])
    print(f"one-step errors: gv max {ev.max():.2e} (rel {np.max(ev / scale_v):.2e}) median {np.median(ev.max(1)):.2e}; gc max {eq.max():.2e}")
    # tolerance: float32 Cholesky of Mhat (cond ~1e4-1e5) and the solver threshold dominate.  The float32
    # build of the oracle gives the scale: the kernel must be no worse than float32 arithmetic itself.
    c32, d32v = gc.copy(), gv.copy()
    o32.step(c32, d32v, tau_ff=tau)
    e32 = np.abs(d32v - b)[conv]
    print(f"float32 oracle one-step gv error: max {e32.max():.2e} median {np.median(e32.max(1)):.2e}")
    assert np.median(ev.max(1)) < max(2e-5, 3 * np.median(e32.max(1)))
    assert np.max(ev / scale_v) < max(5e-3, 3 * np.max(e32 / scale_v))
    assert eq.max() < 5e-3 * 0.0025 * (1.0 + np.abs(b[conv]).max()) + 2e-6
    # impulses (world frame) against the oracle's contact-frame impulses rotated to the world
    lam = d["c_lambda"]
    nrm = d["c_normal"]
    live = conv[:, None] & (d["c_pt"] >= 0)
    ln_gpu = np.einsum("ekj,ekj->ek", ct["impulse"], ct["normal"])
    en = np.abs(ln_gpu - lam[:, :, 2])[live]
    print(f"normal impulse error max {en.max():.2e} scale {np.abs(lam[:, :, 2][live]).max():.2e}")
    assert np.quantile(en, 0.99) < 1e-4 * max(1.0, np.abs(lam[:, :, 2][live]).max())
    # complementarity on the GPU result itself
    assert (ln_gpu[live] >= -1e-6).all()
    lt = np.linalg.norm(ct["impulse"] - ln_gpu[:, :, None] * ct["normal"], axis=2)
    assert (lt[live] <= 0.8 * ln_gpu[live] + 1e-4 * (1 + ln_gpu[live])).all()


def test_trajectory_50_steps(capi):
    """N-step drift against the float64 oracle; float32 oracle shown for scale (chaotic after contact
    changes, so the bound is on the bulk of the distribution, not the maximum)."""
    n, N = 512, 50
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=41, terrain="hm", base_z=0.6, tau_scale=10.0, joint_scale=0.3)
    bt.integrate(N)
    gN, vN = bt.get_state()
    a, b = gc.copy(), gv.copy()
    o64.step(a, b, n_steps=N, tau_ff=tau)
    c, d = gc.copy(), gv.copy()
    o32.step(c, d, n_steps=N, tau_ff=tau)
    e = np.abs(gN - a).max(1); e32 = np.abs(c - a).max(1)
    print(f"50-step gc error vs f64 oracle: median {np.median(e):.2e} p90 {np.quantile(e, .9):.2e} max {e.max():.2e} | f32 oracle: median {np.median(e32):.2e} p90 {np.quantile(e32, .9):.2e}")
    assert np.isfinite(gN).all()
    print(f"   p99 {np.quantile(e, .99):.2e} | f32 oracle p99 {np.quantile(e32, .99):.2e}")
    assert np.median(e) < 2e-5          # stated tolerance: 2e-5 (m, rad) median after 50 steps
    assert np.quantile(e, 0.9) < 1e-4
    # the tail is contact-set chaos (a foot that lands one step earlier): bounded against the float32 build of the oracle itself
    assert np.quantile(e, 0.99) < max(5e-3, 5 * np.quantile(e32, 0.99))
    assert np.median(e) < 5 * np.median(e32) + 1e-6   # no worse than float32 arithmetic itself


def test_substeps_fused_equals_repeated_launches(capi):
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", 256, seed=51, base_z=0.55)
    bt.integrate(4)
    g4, v4 = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    for _ in range(4):
        bt.integrate(1)
    g1, v1 = bt.get_state()
    assert np.array_equal(g4, g1) and np.array_equal(v4, v1)     # same arithmetic, bit-identical


def test_integrate1_plus_integrate2_equals_integrate(capi):
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", 256, seed=61, base_z=0.5)
    bt.integrate(1)
    ga, va = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.integrate1()
    gm, vm = bt.get_state()
    assert np.array_equal(gm, gc.astype(np.float32))             # integrate1 does not advance the state
    bt.integrate2()
    gb, vb = bt.get_state()
    assert np.array_equal(ga, gb) and np.array_equal(va, vb)


def test_determinism_run_to_run(capi):
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", 512, seed=71, terrain="hm")
    bt.integrate(8)
    g1, v1 = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.integrate(8)
    g2, v2 = bt.get_state()
    assert np.array_equal(g1, g2) and np.array_equal(v1, v2)


def test_pd_control_matches_oracle(capi):
    n = 256
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=81, base_z=0.62, joint_scale=0.2, vel=0.2)
    kp = np.r_[np.zeros(6), 120.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 2.0 * np.ones(12)]
    target = np.tile(ANYMAL_GC0, (n, 1)); vt = np.zeros((n, 18))
    bt.set_control_mode(capi.PD_PLUS_FEEDFORWARD_TORQUE)
    bt.set_pd_gains(kp, kd)
    bt.set_pd_target(target.astype(np.float32), vt.astype(np.float32))
    bt.integrate(20)
    g, v = bt.get_state()
    a, b = gc.copy(), gv.copy()
    o64.step(a, b, n_steps=20, tau_ff=tau, ptarget=target, vtarget=vt, kp=kp, kd=kd)
    e = np.abs(g - a).max(1)
    print(f"PD 20-step gc error: median {np.median(e):.2e} p90 {np.quantile(e, .9):.2e}")
    assert np.median(e) < 1e-5 and np.quantile(e, 0.9) < 2e-4


def test_known_answers_on_gpu(capi):
    """The oracle's analytic KATs, re-run on the kernel itself (free fall, resting sphere, slope)."""
    # free fall, closed form
    m = capi.Model(os.path.join(RSC, "anymal_c_like.urdf"))
    bt = capi.Batch(m, 4)
    gc = np.tile(ANYMAL_GC0, (4, 1)).astype(np.float32); gc[:, 2] = 10.0
    bt.set_state(gc, np.zeros((4, 18), np.float32))
    bt.integrate(200)
    g, v = bt.get_state()
    dt, G = 0.0025, 9.81
    assert np.allclose(v[:, 2], -G * 200 * dt, rtol=2e-6)
    assert np.allclose(g[:, 2], 10.0 - G * dt * dt * 200 * 201 / 2, atol=2e-5)
    assert np.allclose(g[:, 7:], ANYMAL_GC0[7:], atol=1e-5)
    # sphere at rest: lambda_n = m g dt, v+ = 0
    ms = capi.Model(SPHERE_URDF)
    bs = capi.Batch(ms, 2)
    bs.set_ground(0.0)
    bs.set_state(np.array([[0, 0, 0.0999, 1, 0, 0, 0]] * 2, np.float32), np.zeros((2, 6), np.float32))
    bs.integrate(1)
    ct, cnt = bs.contacts()
    assert (cnt == 1).all() and (ct["local_body"][:, 0] == 0).all() and (ct["pair_index"][:, 0] == 0).all()
    assert np.allclose(ct["impulse"][:, 0], [0, 0, 2.0 * G * dt], atol=1e-6)
    assert np.abs(bs.get_state()[1]).max() < 1e-5
    # box on a slope (tilted gravity): sticks below atan(mu), slides above
    mb = capi.Model(BOX_URDF)
    for deg, slides in ((35.0, False), (42.0, True)):
        th = np.deg2rad(deg)
        bb = capi.Batch(mb, 1)
        bb.set_ground(0.0)
        bb.set_params(gravity=(G * np.sin(th), 0.0, -G * np.cos(th)), mu=0.8)
        bb.set_state(np.array([[0, 0, 0.0999, 1, 0, 0, 0]], np.float32), np.zeros((1, 6), np.float32))
        bb.integrate(100)
        v = bb.get_state()[1][0]
        if slides:
            assert 0.15 < v[0] < 0.25
        else:
            assert np.abs(v).max() < 1e-4


def test_observation_rows(capi):
    n = 64
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=91)
    obs = bt.observe()
    assert obs.shape == (n, 34)
    from helpers import quat_to_rot
    for e in range(0, n, 7):
        R = quat_to_rot(gc[e, 3:7])
        ref = np.r_[gc[e, 2], R[2], gc[e, 7:], R.T @ gv[e, 0:3], R.T @ gv[e, 3:6], gv[e, 6:]]
        assert np.allclose(obs[e], ref, atol=1e-5)


def test_device_buffers_and_torch_stream(capi):
    import torch
    n = 128
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=101)
    s = torch.cuda.Stream()
    bt.set_stream(s.cuda_stream)
    with torch.cuda.stream(s):
        gct = torch.tensor(gc, dtype=torch.float32, device="cuda"); gvt = torch.tensor(gv, dtype=torch.float32, device="cuda")
        bt.set_state(gct, gvt)
        bt.integrate(2)
        og, ov = torch.empty_like(gct), torch.empty_like(gvt)
        bt.get_state_into(og, ov)
        obs = torch.empty((n, bt.ob_dim()), dtype=torch.float32, device="cuda")
        bt.observe(obs)
    s.synchronize()
    g2, v2 = bt.get_state()
    assert np.array_equal(og.cpu().numpy(), g2) and np.array_equal(ov.cpu().numpy(), v2)
    assert torch.isfinite(obs).all()
    assert bt.launch_count() >= 2
    bt.set_stream(0)


def test_full_size_properties_4096(capi):
    """BASELINE configs[2] size: 4096 ANYmal-C-like on a rough height field.  Size-independent
    properties: finite state, unit quaternions, contact complementarity, momentum in free flight."""
    n = 4096
    path = os.path.join(RSC, "anymal_c_like.urdf")
    m = capi.Model(path)
    bt = capi.Batch(m, n)
    rng = np.random.default_rng(3000)
    xs = ys = 513
    H = (0.10 * rng.uniform(-1, 1, (ys, xs))).astype(np.float32)
    bt.set_heightmap(xs, ys, 51.2, 51.2, 0.0, 0.0, H)
    gc = np.tile(ANYMAL_GC0, (n, 1)); gc[:, :2] = rng.uniform(-20, 20, (n, 2)); gc[:, 2] = 0.75
    gc[:, 7:] += rng.uniform(-0.2, 0.2, (n, 12))
    kp = np.r_[np.zeros(6), 300.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 8.0 * np.ones(12)]
    bt.set_pd_gains(kp, kd)
    bt.set_pd_target(np.tile(ANYMAL_GC0, (n, 1)).astype(np.float32), np.zeros((n, 18), np.float32))
    bt.set_state(gc.astype(np.float32), np.zeros((n, 18), np.float32))
    seen = 0
    for k in range(60):
        bt.integrate(4)
        ct, cnt = bt.contacts()
        live = np.arange(8)[None, :] < cnt[:, None]
        ln = np.einsum("ekj,ekj->ek", ct["impulse"], ct["normal"])
        assert (ln[live] >= -1e-6).all()
        lt = np.linalg.norm(ct["impulse"] - ln[:, :, None] * ct["normal"], axis=2)
        assert (lt[live] <= 0.8 * ln[live] + 1e-4 * (1 + ln[live])).all()
        assert (np.abs(np.linalg.norm(ct["normal"], axis=2)[live] - 1) < 1e-5).all()
        seen += int(cnt.sum())
    g, v = bt.get_state()
    assert np.isfinite(g).all() and np.isfinite(v).all()
    assert np.abs(np.linalg.norm(g[:, 3:7], axis=1) - 1).max() < 1e-5
    assert seen > 4096 * 60                      # contact-heavy: well over one contact per env-step
    assert (g[:, 2] > 0.2).mean() > 0.99         # robots are standing on the terrain, not through it
    it = bt.solver_iterations()
    print(f"4096-env rough terrain: mean K {cnt.mean():.2f}, mean solver iterations {it.mean():.1f}, max {it.max()}")


def test_cpp_facade_example_program(capi):
    """BASELINE configs[0]: the raisim:: facade (include/raisim/World.hpp) driving a batch of one through
    1000 World::integrate() calls; the program checks that the robot stands on four feet."""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "examples", "anymal_flat")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    out = subprocess.run([exe, os.path.join(RSC, "anymal_c_like.urdf"), "1000"], capture_output=True, text=True, timeout=120)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "contacts=4" in out.stdout


def test_cpp_kinematic_getters_example():
    """facade getters (frame pose / velocity / Jacobians, SURVEY 8b) against finite differences, from C++"""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "examples", "kinematics_check")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    out = subprocess.run([exe, os.path.join(RSC, "anymal_c_like.urdf")], capture_output=True, text=True, timeout=120)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr


def test_cpp_dynamics_getters_example():
    """facade whole-body getters (getCOM, getLinearMomentum, getKineticEnergy, getGeneralizedMomentum, getSparseJacobian, getJointLimits,
    setBasePos / setBaseOrientation, HeightMap::getHeight, jointOrder on M / h / J; SURVEY 8b) against conservation laws and the
    kernel's own M, poses and contacts, from C++"""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "examples", "dynamics_getters")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    out = subprocess.run([exe, os.path.join(RSC, "anymal_c_like.urdf")], capture_output=True, text=True, timeout=180)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr


def test_default_solver_matches_oracle_on_random_drops(capi):
    """Library defaults (Anderson-accelerated sweeps from sweep 6, stagnation window 8 with the compliant fallback, threshold 1e-6)
    on a brutal random-drop batch (knee + foot contacts on one shank, bodies on the ground): same sweep counts and the same
    endings as the oracle, < 1 % of the environments end without converging."""
    n = 1024
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=111, base_z=0.35)
    bt.integrate(1)
    it = bt.solver_iterations(); st = bt.solver_status()
    g1, v1 = bt.get_state()
    a, b = gc.copy(), gv.copy()
    d = o64.step(a, b, tau_ff=tau, debug=True)
    pts = bt.contact_points()
    same = (pts == d["c_pt"]).all(1)
    agree = (it == d["iters"])[same].mean()
    print(f"default solver: sweeps gpu mean {it.mean():.2f} max {it.max()} | oracle mean {d['iters'].mean():.2f} max {d['iters'].max()}; identical counts in "
          f"{100 * agree:.1f}% of envs; status gpu {np.bincount(st, minlength=4).tolist()} oracle {np.bincount(d['status'], minlength=4).tolist()}")
    assert (st >= 2).mean() < 0.07 and (d["status"] >= 2).mean() < 0.05     # unphysical drops (see test_one_step_state_and_impulses); oracle: 1.8 %, float32: 4.8 %
    assert it.mean() < 1.15 * d["iters"].mean() + 0.5
    print(f"   |sweeps gpu - oracle| <= 2 in {100 * (np.abs(it - d['iters'])[same] <= 2).mean():.1f}%; same fallback decision in {100 * ((st == 1) == (d['status'] == 1))[same].mean():.1f}%")
    assert agree > 0.75                                   # float32 vs float64 leave the loop one sweep apart now and then, and the cycling
    assert (np.abs(it - d["iters"])[same] <= 2).mean() > 0.85      # problems of this batch (10 %) take their exits at different checkpoints
    assert ((st == 1) == (d["status"] == 1))[same].mean() > 0.93      # (mostly) the same problems take the compliant fallback
    ok = same & (st == 0) & (d["status"] == 0)
    ev = np.abs(v1 - b)[ok].max(1)
    print(f"   one-step gv error on converged envs: median {np.median(ev):.2e} p99 {np.quantile(ev, .99):.2e} max {ev.max():.2e}")
    assert np.median(ev) < 2e-5 and np.quantile(ev, 0.99) < 2e-3
    both1 = same & (st == 1) & (d["status"] == 1)
    if both1.sum() > 5:
        e1 = np.abs(v1 - b)[both1].max(1)
        print(f"   on the compliant set ({both1.sum()} envs): gv error median {np.median(e1):.2e} max {e1.max():.2e}")
        assert np.median(e1) < 5e-3
    # plain sweeps (the published method: accel_m = 0, no stagnation check) reach the same fixed point where both converge
    bt.set_params(accel_m=0, stall_window=0)
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.integrate(1)
    it0 = bt.solver_iterations(); st0 = bt.solver_status(); v0 = bt.get_state()[1]
    both = (st == 0) & (st0 == 0)
    print(f"   plain sweeps: mean {it0.mean():.2f} max {it0.max()}, max_iter reached in {100 * (st0 == 3).mean():.2f}%; |dv| accelerated vs plain p99 {np.quantile(np.abs(v1 - v0)[both].max(1), .99):.2e}")
    assert it.mean() < 0.8 * it0.mean()
    assert np.quantile(np.abs(v1 - v0)[both].max(1), 0.99) < 1e-4


def test_atlas_standing_trajectory_and_heightmap(capi):
    """Config 4 regime, library defaults: the Atlas-like humanoid standing on box feet (8 redundant corner contacts, the case that
    needed 55 plain sweeps per step) for 50 steps, and dropped onto a height map; gc / gv against the float64 oracle."""
    n = 256
    path = os.path.join(RSC, "atlas_like.urdf")
    t = load_tables(path)
    rng = np.random.default_rng(301)
    gc0 = np.zeros(37); gc0[2] = 0.95; gc0[3] = 1.0
    gc = np.tile(gc0, (n, 1)); gc[:, 7:] += rng.uniform(-0.05, 0.05, (n, 30)); gv = np.zeros((n, 36))
    kp = np.r_[np.zeros(6), 400.0 * np.ones(30)]; kd = np.r_[np.zeros(6), 10.0 * np.ones(30)]
    tgt = gc.copy()
    prm = dict(threshold=THRESH)
    o = Oracle(t, params=prm); o.set_ground(0.0)
    o.step(gc, gv, n_steps=60, ptarget=tgt, vtarget=np.zeros((n, 36)), kp=kp, kd=kd)        # settle onto the feet (CPU)
    gc32, gv32 = gc.astype(np.float32), gv.astype(np.float32)
    bt = capi.Batch(capi.Model(path), n)
    bt.set_ground(0.0); bt.set_params(**prm)
    bt.set_pd_gains(kp, kd); bt.set_pd_target(tgt.astype(np.float32), np.zeros((n, 36), np.float32))
    bt.set_state(gc32, gv32)
    a, b = gc32.astype(np.float64), gv32.astype(np.float64)
    o32 = Oracle(t, precision="f32", params=prm); o32.set_ground(0.0)
    c, d = a.copy(), b.copy()
    sweeps, ncv = [], []
    for k in range(10):
        bt.integrate(5)
        sweeps.append(bt.solver_iterations()); ncv.append(bt.solver_status() >= 1)
        dbg = o.step(a, b, n_steps=5, ptarget=tgt.astype(np.float32).astype(np.float64), vtarget=np.zeros((n, 36)), kp=kp, kd=kd, debug=True)
    o32.step(c, d, n_steps=50, ptarget=tgt.astype(np.float32).astype(np.float64), vtarget=np.zeros((n, 36)), kp=kp, kd=kd)
    g, v = bt.get_state()
    _, cnt = bt.contacts()
    sweeps = np.array(sweeps); ncv = np.array(ncv)
    e = np.abs(g - a).max(1); e32 = np.abs(c - a).max(1); ev = np.abs(v - b).max(1)
    print(f"atlas standing 50 steps: K {cnt.mean():.2f}, sweeps mean {sweeps.mean():.1f} p99 {np.quantile(sweeps, .99):.0f} max {sweeps.max()} (oracle last {dbg['iters'].mean():.1f}), "
          f"not converged on the exact contact set {100 * ncv.mean():.2f}%; gc err median {np.median(e):.2e} p99 {np.quantile(e, .99):.2e} max {e.max():.2e} | f32 oracle median {np.median(e32):.2e} "
          f"p99 {np.quantile(e32, .99):.2e}; gv err median {np.median(ev):.2e} p99 {np.quantile(ev, .99):.2e}")
    assert cnt.mean() > 6                                   # standing on the box corners
    assert sweeps.mean() <= 15 and ncv.mean() < 0.01         # VERDICT r1 item 1: <= 15 mean sweeps, < 1 % non-converged
    assert np.median(e) < 2e-5 and np.quantile(e, 0.99) < max(1e-3, 5 * np.quantile(e32, 0.99))
    # on a height map: random drops, 20 steps
    t2, bt2, o64, o32b, gc2, gv2, tau2 = _setup(capi, "atlas_like.urdf", n, seed=302, terrain="hm", base_z=0.95, tau_scale=2.0, vel=0.3, joint_scale=0.2)
    # upright-ish: small random tilt instead of a random quaternion, so that the feet (not the head) meet the terrain
    q = np.c_[np.ones(n), 0.1 * rng.standard_normal((n, 3))]; q /= np.linalg.norm(q, axis=1, keepdims=True)
    gc2[:, 3:7] = q.astype(np.float32)
    bt2.set_state(gc2.astype(np.float32), gv2.astype(np.float32))
    a, b = gc2.astype(np.float32).astype(np.float64), gv2.copy()
    c, d = a.copy(), b.copy()
    bt2.integrate(20)
    g, v = bt2.get_state()
    dbg = o64.step(a, b, n_steps=20, tau_ff=tau2, debug=True)
    o32b.step(c, d, n_steps=20, tau_ff=tau2)
    _, cnt = bt2.contacts()
    st2 = bt2.solver_status()
    e = np.abs(g - a).max(1); e32 = np.abs(c - a).max(1)
    print(f"atlas on a height map, 20 steps: K {cnt.mean():.2f} (oracle {dbg['ncontacts'].mean():.2f}), sweeps {bt2.solver_iterations().mean():.1f}, status {np.bincount(st2, minlength=4).tolist()}; "
          f"gc err median {np.median(e):.2e} p90 {np.quantile(e, .9):.2e} p99 {np.quantile(e, .99):.2e} | f32 oracle median {np.median(e32):.2e} p99 {np.quantile(e32, .99):.2e}")
    assert cnt.sum() > n                                     # contact-rich
    assert (st2 >= 2).mean() < 0.05                          # tilted drops onto rough terrain: hands, knees and box edges at once
    # tilted 20-step drops are chaotic (hands, knees, box edges touch down one step apart): bounded by the float32 oracle itself
    assert np.median(e) < max(2e-5, 3 * np.median(e32)) and np.quantile(e, 0.99) < max(2e-3, 5 * np.quantile(e32, 0.99))


def test_bench_workload_parity(capi):
    """What bench.py measures is what is tested: the exact headline workload (4096 environments, 513 x 513 height field, PD stance
    with target jitter, library-default solver), settled on the GPU, then 1 and 20 control steps (4 fused sub-steps each) against
    the oracle from the same state: contact lists, gc, gv."""
    import bench
    n = 4096
    wl = bench.Workload("c3", 0, n)
    hm = bench.HM
    path = os.path.join(RSC, wl.urdf)
    bt = capi.Batch(capi.Model(path), n)
    bt.set_params(**bench.SOLVER)
    bt.set_heightmap(hm["xs"], hm["ys"], hm["size"], hm["size"], 0.0, 0.0, wl.H)
    bt.set_pd_gains(wl.kp, wl.kd)
    bt.set_state(wl.gc.astype(np.float32), wl.gv.astype(np.float32))
    vt = np.zeros((n, 18), np.float32)
    ring32 = wl.ring.astype(np.float32)
    for k in range(wl.settle + 5):
        bt.set_pd_target(ring32[k % bench.RING], vt)
        bt.integrate(bench.SUBSTEPS)
    g0, v0 = bt.get_state()
    t = load_tables(path)
    o64 = Oracle(t, params=bench.SOLVER); o32 = Oracle(t, precision="f32", params=bench.SOLVER)
    for o in (o64, o32):
        o.set_heightmap(hm["xs"], hm["ys"], hm["size"], hm["size"], 0.0, 0.0, wl.H.astype(np.float64))
    k0 = wl.settle + 5
    # ---- one control step ----
    tg = ring32[k0 % bench.RING]
    bt.set_pd_target(tg, vt); bt.integrate(bench.SUBSTEPS)
    g1, v1 = bt.get_state(); pts = bt.contact_points(); ct, cnt = bt.contacts(); it = bt.solver_iterations(); st = bt.solver_status()
    a, b = g0.astype(np.float64), v0.astype(np.float64)
    d = o64.step(a, b, n_steps=bench.SUBSTEPS, ptarget=tg.astype(np.float64), vtarget=vt.astype(np.float64), kp=wl.kp, kd=wl.kd, debug=True)
    c, e_ = g0.astype(np.float64), v0.astype(np.float64)
    d32 = o32.step(c, e_, n_steps=bench.SUBSTEPS, ptarget=tg.astype(np.float64), vtarget=vt.astype(np.float64), kp=wl.kp, kd=wl.kd, debug=True)
    same = (pts == d["c_pt"]).all(1) & (cnt == d["ncontacts"])
    same32 = (pts == d32["c_pt"]).all(1)
    eq = np.abs(g1 - a).max(1); ev = np.abs(v1 - b).max(1); eq32 = np.abs(c - a).max(1); ev32 = np.abs(e_ - b).max(1)
    print(f"bench workload, 1 control step: K {cnt.mean():.2f} hist {np.bincount(cnt, minlength=9).tolist()}, sweeps gpu {it.mean():.2f} max {it.max()} oracle {d['iters'].mean():.2f}; "
          f"status {np.bincount(st, minlength=4).tolist()}; identical contact lists (4th sub-step) vs f64 oracle {100 * same.mean():.2f}% vs f32 oracle {100 * same32.mean():.2f}%")
    print(f"   gc err median {np.median(eq):.2e} p99 {np.quantile(eq, .99):.2e} max {eq.max():.2e} (f32 oracle: {np.median(eq32):.2e} / {np.quantile(eq32, .99):.2e} / {eq32.max():.2e}); "
          f"gv err median {np.median(ev):.2e} p99 {np.quantile(ev, .99):.2e} max {ev.max():.2e} (f32 oracle: {np.median(ev32):.2e} / {np.quantile(ev32, .99):.2e} / {ev32.max():.2e})")
    assert (st == 0).all()                                   # every environment of the benchmarked workload converges, on the exact contact set
    assert same.mean() > 0.995                                # the few that differ have a foot within float32 rounding of touching down
    assert np.median(eq) < 2e-6 and np.quantile(eq, 0.99) < max(2e-5, 5 * np.quantile(eq32, 0.99))
    assert np.median(ev) < 5e-5 and np.quantile(ev, 0.99) < max(5e-3, 5 * np.quantile(ev32, 0.99))
    # impulses of the last sub-step where the lists agree
    live = same[:, None] & (d["c_pt"] >= 0)
    ln_gpu = np.einsum("ekj,ekj->ek", ct["impulse"], ct["normal"])
    en = np.abs(ln_gpu - d["c_lambda"][:, :, 2])[live]
    assert np.quantile(en, 0.99) < 2e-3 * max(1.0, np.abs(d["c_lambda"][:, :, 2][live]).max())
    # ---- 20 control steps ----
    for k in range(1, 20):
        tg = ring32[(k0 + k) % bench.RING]
        bt.set_pd_target(tg, vt); bt.integrate(bench.SUBSTEPS)
        o64.step(a, b, n_steps=bench.SUBSTEPS, ptarget=tg.astype(np.float64), vtarget=vt.astype(np.float64), kp=wl.kp, kd=wl.kd)
        o32.step(c, e_, n_steps=bench.SUBSTEPS, ptarget=tg.astype(np.float64), vtarget=vt.astype(np.float64), kp=wl.kp, kd=wl.kd)
    g20, v20 = bt.get_state()
    eq = np.abs(g20 - a).max(1); eq32 = np.abs(c - a).max(1)
    print(f"   20 control steps (80 sub-steps): gc err median {np.median(eq):.2e} p90 {np.quantile(eq, .9):.2e} p99 {np.quantile(eq, .99):.2e} | f32 oracle median {np.median(eq32):.2e} "
          f"p90 {np.quantile(eq32, .9):.2e} p99 {np.quantile(eq32, .99):.2e}")
    assert np.isfinite(g20).all()
    assert np.median(eq) < 2e-5                              # the stated tolerance (DESIGN.md section 5)
    assert np.quantile(eq, 0.9) < max(1e-3, 5 * np.quantile(eq32, 0.9))
    assert np.quantile(eq, 0.99) < max(2e-2, 5 * np.quantile(eq32, 0.99))   # contact-set chaos: bounded by float32 arithmetic itself


def test_fallen_quadrupeds_default_solver(capi):
    """Config 2 regime: quadrupeds lying on flat ground under random joint torques (bodies, knees and feet in contact, joints at
    their stops); state prepared by the oracle, one control step with fresh torques on both sides."""
    import bench
    n = 1024
    wl = bench.Workload("c2", 0, n)
    path = os.path.join(RSC, wl.urdf)
    t = load_tables(path)
    o = Oracle(t, params=bench.SOLVER); o.set_ground(0.0)
    a, b = wl.gc.copy(), wl.gv.copy()
    for k in range(wl.settle):
        o.step(a, b, n_steps=bench.SUBSTEPS, tau_ff=wl.ring[k % bench.RING])
    g0, v0 = a.astype(np.float32), b.astype(np.float32)
    bt = capi.Batch(capi.Model(path), n)
    bt.set_ground(0.0); bt.set_params(**bench.SOLVER)
    bt.set_control_mode(capi.FORCE_AND_TORQUE)
    bt.set_state(g0, v0)
    tau = wl.ring[wl.settle % bench.RING].astype(np.float32)
    bt.set_generalized_force(tau)
    bt.integrate(1)
    g1, v1 = bt.get_state(); pts = bt.contact_points(); _, cnt = bt.contacts(); it = bt.solver_iterations(); st = bt.solver_status()
    a, b = g0.astype(np.float64), v0.astype(np.float64)
    d = o.step(a, b, n_steps=1, tau_ff=tau.astype(np.float64), debug=True)
    same = (pts == d["c_pt"]).all(1)
    conv = same & (st == 0) & (d["status"] == 0)
    ev = np.abs(v1 - b)[conv].max(1)
    print(f"fallen quadrupeds: base z median {np.median(g0[:, 2]):.3f}, K {cnt.mean():.2f} hist {np.bincount(cnt, minlength=9).tolist()}, sweeps gpu {it.mean():.2f} (p99 {np.quantile(it, .99):.0f}, max {it.max()}) "
          f"oracle {d['iters'].mean():.2f}; status gpu {np.bincount(st, minlength=4).tolist()} oracle {np.bincount(d['status'], minlength=4).tolist()}; same lists {100 * same.mean():.2f}%; "
          f"gv err median {np.median(ev):.2e} p99 {np.quantile(ev, .99):.2e}")
    assert np.median(g0[:, 2]) < 0.2 and cnt.mean() > 3
    assert (st >= 2).mean() < 0.01 and (d["status"] >= 2).mean() < 0.01      # VERDICT r1 item 1: < 1 % non-converged
    assert same.mean() > 0.98 and conv.mean() > 0.95
    assert np.median(ev) < 5e-5 and np.quantile(ev, 0.99) < 5e-3


def test_kinematic_getters_keep_contact_records(capi):
    """ADVICE r1 (medium): kinematic getters after integrate() must not replace the last step's contacts, impulses and sweep
    count (upstream's getContacts() stays valid across getFramePosition() etc.), and the lazy getters follow the state."""
    n = 64
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=401, base_z=0.5, joint_scale=0.2)
    bt.integrate(3)
    ct0, cnt0 = bt.contacts(); it0 = bt.solver_iterations(); res0 = bt.solver_residual()
    assert cnt0.sum() > 0 and np.abs(ct0["impulse"]).max() > 0
    M = bt.mass_matrix(); h = bt.nonlinearities(); R, p = bt.body_poses()      # lazy: a kinematics-only pass at the CURRENT state
    ct1, cnt1 = bt.contacts()
    assert np.array_equal(cnt0, cnt1) and np.array_equal(ct0["impulse"], ct1["impulse"]) and np.array_equal(ct0["position"], ct1["position"])
    assert np.array_equal(it0, bt.solver_iterations()) and np.array_equal(res0, bt.solver_residual())
    g, v = bt.get_state()
    bt2 = capi.Batch(bt.model, n)
    bt2.set_ground(0.0); bt2.set_state(g, v)
    bt2.integrate1()
    assert np.array_equal(M, bt2.mass_matrix()) and np.array_equal(p, bt2.body_poses()[1]) and np.allclose(h, bt2.nonlinearities(), atol=1e-4)
    l0 = bt.launch_count()
    bt.mass_matrix(); bt.body_poses()
    assert bt.launch_count() == l0                           # nothing changed since: no relaunch
    bt.integrate(1)
    assert not np.array_equal(bt.body_poses()[1], p)         # ... and after a step the getters describe the new state


def test_control_step_equals_separate_calls(capi):
    import torch
    n = 256
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=121, base_z=0.6, joint_scale=0.2)
    kp = np.r_[np.zeros(6), 200.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 5.0 * np.ones(12)]
    bt.set_control_mode(capi.PD_PLUS_FEEDFORWARD_TORQUE)
    bt.set_pd_gains(kp, kd)
    target = np.tile(ANYMAL_GC0, (n, 1)).astype(np.float32)
    bt.set_pd_target(target, np.zeros((n, 18), np.float32))
    bt.integrate(4)
    ref_obs = bt.observe()
    g_ref, v_ref = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    pin_t = torch.from_numpy(target).pin_memory()
    pin_o = torch.empty((n, 34), dtype=torch.float32).pin_memory()
    bt.control_step(pin_t, 4, pin_o)
    g2, v2 = bt.get_state()
    assert np.array_equal(g_ref, g2) and np.array_equal(v_ref, v2)
    # zero-copy binding of device-resident targets gives the same step again
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    dev_t = torch.from_numpy(target).cuda()
    bt.bind_pd_target(dev_t)
    bt.integrate(4)
    g3, v3 = bt.get_state()
    bt.bind_pd_target(None)
    assert np.array_equal(g_ref, g3) and np.array_equal(v_ref, v3)
    assert np.array_equal(ref_obs, pin_o.numpy())          # observation rows written by the step kernel == observe kernel
    # pageable host buffers take the staged-copy path: same result
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    o_np = np.empty((n, 34), np.float32)
    bt.control_step(target.copy(), 4, o_np)
    g4, v4 = bt.get_state()
    assert np.array_equal(g_ref, g4) and np.array_equal(v_ref, v4) and np.array_equal(ref_obs, o_np)
    # row-dependent position AND velocity targets: the CTA-cooperative fetch of pinned rows (16-byte chunks of the CTA's contiguous
    # rows, staged in shared memory) must hand every environment ITS row -- pinned path == pageable (staged-copy) path, bit for bit
    rng = np.random.default_rng(5)
    tq = target.copy(); tq[:, 7:] += rng.uniform(-0.3, 0.3, (n, 12)).astype(np.float32)
    tv = rng.uniform(-0.5, 0.5, (n, 18)).astype(np.float32); tv[:, :6] = 0
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.control_step(tq.copy(), 4, o_np, vtarget=tv.copy())
    g5, v5 = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    pq, pv = torch.from_numpy(tq).pin_memory(), torch.from_numpy(tv).pin_memory()
    bt.control_step(pq, 4, pin_o, vtarget=pv)
    g6, v6 = bt.get_state()
    assert np.array_equal(g5, g6) and np.array_equal(v5, v6) and np.array_equal(o_np, pin_o.numpy())
    assert not np.array_equal(g5, g4)                      # the targets do matter
    # position targets alone from pinned memory (what bench.py's e2e arm passes), velocity targets kept from the call before
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.control_step(pq, 4, pin_o)
    g7, v7 = bt.get_state()
    assert np.array_equal(g5, g7) and np.array_equal(v5, v7)
    # the same rows at a source address that is NOT 16-byte aligned (one row = 76 bytes into a pinned allocation): head / tail words
    big = torch.empty((n + 1, 19), dtype=torch.float32).pin_memory(); big[1:] = torch.from_numpy(tq)
    bigv = torch.empty((n + 3, 18), dtype=torch.float32).pin_memory(); bigv[3:] = torch.from_numpy(tv)
    assert big[1:].data_ptr() % 16 != 0 and bigv[3:].data_ptr() % 16 != 0
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.control_step(big[1:], 4, pin_o, vtarget=bigv[3:])
    g9, v9 = bt.get_state()
    assert np.array_equal(g5, g9) and np.array_equal(v5, v9)
    bt.set_pd_target(target, np.zeros((n, 18), np.float32))
    bt.set_state(g4, v4)
    # targets read in place from pinned host memory persist like setPdTarget(): the caller may reuse its buffer
    bt.integrate(4)
    g_ref8, v_ref8 = bt.get_state()
    bt.set_pd_target(np.zeros((n, 19), np.float32), None)           # clobber the stored targets
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    scratch = pin_t.clone().pin_memory()
    bt.control_step(scratch, 4, pin_o)
    scratch.zero_()
    bt.integrate(4)
    g8, v8 = bt.get_state()
    assert np.array_equal(g_ref8, g8) and np.array_equal(v_ref8, v8)


@pytest.mark.parametrize("n", [1, 5, 4097, 9000])
def test_ragged_batch_sizes(capi, n):
    """batch sizes that do not fill a CTA / an SM wave, and more environments than resident warps
    (9000 > 148 x 28: the per-warp environment loop runs three times)."""
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=131 + n, base_z=0.5, joint_scale=0.3, params=dict(stall_window=0))
    bt.integrate(3)
    g, v = bt.get_state()
    idx = np.unique(np.r_[0, n - 1, np.random.default_rng(1).integers(0, n, 40)])
    a, b = gc[idx].copy(), gv[idx].copy()
    o64.step(a, b, n_steps=3, tau_ff=tau[idx])
    assert np.isfinite(g).all() and np.isfinite(v).all()
    e = np.abs(g[idx] - a).max(1)
    assert np.median(e) < 1e-5 and np.quantile(e, 0.9) < 1e-3


def test_contact_cap_parity_atlas(capi):
    """more penetrating candidates than RSB_KMAX: the 8 deepest are kept, in candidate order, on both sides"""
    n = 64
    path = os.path.join(RSC, "atlas_like.urdf")
    t = load_tables(path)
    m = capi.Model(path)
    bt = capi.Batch(m, n)
    bt.set_ground(0.0)
    rng = np.random.default_rng(7)
    gc = np.zeros((n, 37)); gc[:, 2] = rng.uniform(0.02, 0.12, n)
    ang = rng.uniform(0.3, 1.2, n) * np.pi / 2
    gc[:, 3] = np.cos(ang / 2); gc[:, 5] = np.sin(ang / 2)          # pitched forward towards lying face down
    gc[:, 7:] = rng.uniform(-0.3, 0.3, (n, 30))
    gc32 = gc.astype(np.float32)
    bt.set_state(gc32, np.zeros((n, 36), np.float32))
    bt.integrate1()
    ct, cnt = bt.contacts()
    pts = bt.contact_points()
    o32 = Oracle(t, precision="f32")
    o32.set_ground(0.0)
    a, b = gc32.astype(np.float64), np.zeros((n, 36))
    d = o32.step(a, b, debug=True)
    assert (cnt == 8).sum() > n // 2                       # the cap is actually exercised
    # Every list must be the 8 deepest candidates.  The only legitimate difference: candidates whose depth equals the cut-off (the
    # 8th deepest) to float32 rounding may swap -- checked candidate by candidate against depths recomputed from the oracle's poses.
    P = d["p"][:, t["pt_body"]] + np.einsum("ebij,bj->ebi", d["R"][:, t["pt_body"]], t["pt_pos"])
    depth = t["pt_rad"][None, :] - P[:, :, 2]                # plane z = 0
    n_bad = 0
    for e in range(n):
        if (pts[e] == d["c_pt"][e]).all():
            continue
        cut = np.sort(depth[e][depth[e] > 0])[::-1][7]
        diff = set(pts[e][pts[e] >= 0]) ^ set(d["c_pt"][e][d["c_pt"][e] >= 0])
        if any(abs(depth[e][k] - cut) > MARGIN for k in diff):
            n_bad += 1
    assert n_bad == 0, f"{n_bad} capped contact lists differ beyond depth ties at the cut-off"
    assert (np.diff(np.where(pts >= 0, pts, 10**6), axis=1) > 0).all()   # candidate order


def test_fixed_base_model_with_contacts(capi):
    """generic (non-specialised) kernel path: fixed base, prismatic joint, contacts on a moving link only"""
    urdf = PENDULUM_URDF.replace('<link name="l3">', '<link name="l3"><collision><origin xyz="0.1 0 0"/><geometry><sphere radius="0.08"/></geometry></collision>')
    t = load_tables(urdf)
    m = capi.Model(urdf)
    n = 128
    bt = capi.Batch(m, n)
    bt.set_ground(-0.55)
    bt.set_params(threshold=THRESH, stall_window=0)
    rng = np.random.default_rng(17)
    gc = rng.uniform(-0.6, 0.6, (n, 3)); gv = rng.standard_normal((n, 3))
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    o = Oracle(t, params=dict(threshold=THRESH, stall_window=0))
    o.set_ground(-0.55)
    a, b = gc.astype(np.float32).astype(np.float64), gv.astype(np.float32).astype(np.float64)
    tot = 0
    for k in range(30):
        bt.integrate(1)
        d = o.step(a, b, debug=True)
        tot += int(d["ncontacts"].sum())
    g, v = bt.get_state()
    e = np.abs(g - a).max(1)
    print(f"fixed-base 30-step error median {np.median(e):.2e} max {e.max():.2e}; contacts seen {tot}")
    assert tot > 50
    assert np.median(e) < 2e-5 and np.quantile(e, 0.9) < 2e-3


def test_gym_task_matches_numpy_restatement(capi):
    """row N1: VectorizedEnvironment::step/observe on the device vs the numpy restatement around the oracle."""
    from oracle.gym_ref import GymRef
    n, substeps = 256, 4
    path = os.path.join(RSC, "anymal_c_like.urdf")
    t = load_tables(path)
    m = capi.Model(path)
    bt = capi.Batch(m, n)
    bt.set_ground(0.0)
    bt.set_params(threshold=THRESH, stall_window=0)
    gc_init = ANYMAL_GC0.copy(); gc_init[2] = 0.57
    kp = np.r_[np.zeros(6), 100.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 2.0 * np.ones(12)]
    feet = [m.body_index(f"{leg}_FOOT") for leg in ("LF", "RF", "LH", "RH")]
    assert feet == [3, 6, 9, 12]
    bt.set_pd_gains(kp, kd)
    bt.gym_configure(gc_init, np.zeros(18), gc_init[7:], 0.6 * np.ones(12), feet)
    bt.gym_reset()
    o = Oracle(t, params=dict(threshold=THRESH, stall_window=0))
    o.set_ground(0.0)
    ref = GymRef(o, gc_init.astype(np.float32), np.zeros(18), gc_init[7:].astype(np.float32), (0.6 * np.ones(12)).astype(np.float32), feet, kp, kd)
    ref.reset(n)
    rng = np.random.default_rng(141)
    base = rng.normal(0, 1.5, (n, 12))                            # persistent offsets: many robots fold up and terminate
    obs = np.empty((n, 34), np.float32); rew = np.empty(n, np.float32); done = np.empty(n, np.uint8)
    n_done = 0
    agree = np.ones(n, bool)       # environments whose episode history still matches (a differing reset diverges for good)
    for k in range(40):
        act = (base + rng.normal(0, 0.3, (n, 12))).astype(np.float32)
        bt.gym_step(act, substeps, obs, rew, done)
        o_ref, r_ref, d_ref, dbg = ref.step(act.astype(np.float64), substeps)
        same_done = done.astype(bool) == d_ref
        agree &= same_done
        n_done += int(d_ref.sum())
        a = agree
        assert a.mean() > 0.9
        eo = np.abs(obs[a] - o_ref[a]).max(1)
        er = np.abs(rew[a] - r_ref[a])
        assert np.quantile(eo, 0.9) < 5e-3, (k, np.quantile(eo, 0.9))
        assert np.quantile(er, 0.9) < 5e-3 * (1 + np.abs(r_ref[a]).max())
    print(f"gym parity: {n_done} episode terminations in 40 steps x {n} envs, {100 * agree.mean():.1f}% of envs in lockstep to the end")
    assert n_done > 40
    g, v = bt.get_state()
    tau = bt.generalized_force()
    assert np.isfinite(g).all() and np.isfinite(tau).all()
    # pinned host buffers are read / written in place by the task kernels: identical to the staged-copy path
    import torch
    act = (base + rng.normal(0, 0.3, (n, 12))).astype(np.float32)
    bt.gym_step(act, substeps, obs, rew, done)
    g1, v1 = bt.get_state()
    bt.set_state(g, v)
    p_act = torch.from_numpy(act).pin_memory()
    p_obs = torch.empty((n, 34), dtype=torch.float32).pin_memory(); p_rew = torch.empty(n, dtype=torch.float32).pin_memory()
    p_done = torch.empty(n, dtype=torch.uint8).pin_memory()
    bt.gym_step(p_act, substeps, p_obs, p_rew, p_done)
    g2, v2 = bt.get_state()
    assert np.array_equal(g1, g2) and np.array_equal(v1, v2)
    assert np.array_equal(obs, p_obs.numpy()) and np.array_equal(rew, p_rew.numpy()) and np.array_equal(done, p_done.numpy())


def test_cpp_vectorized_environment_example(capi):
    """row N1 from C++: include/raisim/VectorizedEnvironment.hpp driving 512 environments for 100 control steps"""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "examples", "anymal_vecenv")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    out = subprocess.run([exe, os.path.join(RSC, "anymal_c_like.urdf"), "512"], capture_output=True, text=True, timeout=120)
    print(out.stdout)
    assert out.returncode == 0, out.stdout + out.stderr


def test_zero_copy_state_tensors_and_divergence_flag(capi):
    import torch
    n = 64
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=151, base_z=0.6)
    tg, tv = bt.state_tensors()
    assert tg.shape == (n, 19) and tv.shape == (n, 18) and tg.is_cuda
    assert np.array_equal(tg.cpu().numpy(), gc.astype(np.float32))
    tg[3, 2] = 1.25                                   # write through the view ...
    assert abs(bt.get_state()[0][3, 2] - 1.25) < 1e-7  # ... is seen by the C-ABI
    bt.integrate(1)
    assert (bt.diverged() == 0).all()
    tv[5, 7] = float("nan")                            # poison one environment
    bt.integrate(1)
    d = bt.diverged()
    assert d[5] == 1 and d.sum() == 1
    g, v = bt.get_state()
    assert np.isfinite(np.delete(g, 5, 0)).all()        # its neighbours are untouched


def test_cpp_multi_gpu_allgather_example(capi):
    """rsb_comm_* (native NCCL all-gather of the observation rows) on however many GPUs are visible"""
    import subprocess, torch
    from conftest import ROOT
    exe = os.path.join(ROOT, "examples", "multi_gpu")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    ndev = torch.cuda.device_count()
    out = subprocess.run([exe, os.path.join(RSC, "anymal_c_like.urdf"), str(ndev), "512"], capture_output=True, text=True, timeout=300)
    print(out.stdout, out.stderr[-500:])
    assert out.returncode == 0, out.stdout + out.stderr
    assert f"{ndev} GPU(s)" in out.stdout and "ok" in out.stdout


def test_joint_limits_match_oracle(capi):
    """a9 joint limits as unilateral rows of the same Gauss-Seidel solve: generic kernel (fixed-base pendulum with a
    stop) and specialised kernel (ANYmal-like HAA joints swung into their stops, on the ground with contacts)."""
    from test_oracle_kat import LIMIT_PENDULUM
    # 1. pendulum hitting its stop
    t = load_tables(LIMIT_PENDULUM)
    bt = capi.Batch(capi.Model(LIMIT_PENDULUM), 8)
    bt.set_params(gravity=(0.0, 0.0, 0.0), threshold=THRESH, stall_window=0)
    q0 = np.linspace(0.4013, 0.4679, 8)[:, None]; v0 = np.full((8, 1), 2.1)     # never lands exactly on the stop
    bt.set_state(q0.astype(np.float32), v0.astype(np.float32))
    o = Oracle(t, params=dict(gz=0.0, threshold=THRESH, stall_window=0))
    a, b = q0.astype(np.float32).astype(np.float64), v0.copy()
    for k in range(60):
        bt.integrate(1)
        o.step(a, b)
    g, v = bt.get_state()
    assert np.abs(g - a).max() < 1e-5 and np.abs(v - b).max() < 1e-5
    assert (g <= 0.5 + 2.1 * 0.0025 + 1e-6).all() and np.abs(v).max() < 1e-6
    # 2. quadruped: HAA joints driven into their stops by PD targets beyond the limits
    n = 128
    path = os.path.join(RSC, "anymal_c_like.urdf")
    t = load_tables(path)
    bt = capi.Batch(capi.Model(path), n)
    bt.set_ground(0.0)
    bt.set_params(threshold=THRESH, stall_window=0)
    rng = np.random.default_rng(161)
    gc = np.tile(ANYMAL_GC0, (n, 1)); gc[:, 2] = 0.58; gc[:, 7:] += rng.uniform(-0.1, 0.1, (n, 12))
    gv = np.zeros((n, 18))
    target = np.tile(ANYMAL_GC0, (n, 1)); target[:, [7, 10, 13, 16]] = rng.choice([-1.2, 0.9], (n, 4))   # beyond (-0.72, 0.49)
    kp = np.r_[np.zeros(6), 150.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 3.0 * np.ones(12)]
    bt.set_pd_gains(kp, kd)
    gc32, t32 = gc.astype(np.float32), target.astype(np.float32)
    bt.set_state(gc32, gv.astype(np.float32)); bt.set_pd_target(t32, np.zeros((n, 18), np.float32))
    o = Oracle(t, params=dict(threshold=THRESH, stall_window=0))
    o.set_ground(0.0)
    a, b = gc32.astype(np.float64), gv.copy()
    active = 0
    for k in range(12):
        bt.integrate(5)
        d = o.step(a, b, n_steps=5, ptarget=t32.astype(np.float64), vtarget=np.zeros((n, 18)), kp=kp, kd=kd, debug=True)
        active += int(d["nlimits"].sum())
    g, v = bt.get_state()
    haa = g[:, [7, 10, 13, 16]]
    print(f"joint-limit parity: {active} active limit rows seen; HAA range [{haa.min():.3f}, {haa.max():.3f}]")
    assert active > n                                   # the stops are really engaged
    ref_haa = a[:, [7, 10, 13, 16]]
    # the overshoot past a stop is one step of the arrival velocity (several rad/s under this PD drive)
    assert haa.max() < 0.49 + 0.1 and haa.min() > -0.72 - 0.1
    assert abs(haa.max() - ref_haa.max()) < 5e-3 and abs(haa.min() - ref_haa.min()) < 5e-3
    e = np.abs(g - a).max(1)
    assert np.median(e) < 5e-5 and np.quantile(e, 0.9) < 5e-3
    # switched off, the joints leave their range
    bt.set_params(joint_limits=0)
    bt.set_state(gc32, gv.astype(np.float32))
    bt.integrate(60)
    assert bt.get_state()[0][:, [7, 10, 13, 16]].max() > 0.6


def test_per_body_friction_matches_oracle(capi):
    """rsb_batch_set_collision_friction: feet with different friction on the quadruped, and the box-on-slope KAT"""
    n = 128
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=171, base_z=0.55, joint_scale=0.2, vel=1.0)
    feet = [i for i, nme in enumerate(t["coll_names"]) if nme.endswith("_FOOT")]
    assert len(feet) == 4
    for k, ci in enumerate(feet):
        bt.set_collision_friction(ci, 0.1 + 0.2 * k); o64.set_collision_friction(ci, 0.1 + 0.2 * k)
    bt.integrate(20)
    g, v = bt.get_state()
    a, b = gc.copy(), gv.copy()
    o64.step(a, b, n_steps=20, tau_ff=tau)
    e = np.abs(g - a).max(1)
    print(f"per-body friction 20-step error median {np.median(e):.2e} p90 {np.quantile(e, 0.9):.2e}")
    assert np.median(e) < 2e-5 and np.quantile(e, 0.9) < 2e-3
    mb = capi.Model(BOX_URDF)
    th = np.deg2rad(20.0)
    out = {}
    for mu in (-1.0, 0.2):
        bb = capi.Batch(mb, 1)
        bb.set_ground(0.0)
        bb.set_params(gravity=(9.81 * np.sin(th), 0.0, -9.81 * np.cos(th)))
        bb.set_collision_friction(0, mu)
        bb.set_state(np.array([[0, 0, 0.0999, 1, 0, 0, 0]], np.float32), np.zeros((1, 6), np.float32))
        bb.integrate(100)
        out[mu] = bb.get_state()[1][0, 0]
    assert abs(out[-1.0]) < 1e-4 and 0.3 < out[0.2] < 0.45


def test_external_wrench_matches_oracle(capi):
    """ArticulatedSystem::setExternalForce / setExternalTorque (SURVEY 8b): a per-environment world-frame wrench on a distal
    link acts during ONE integrate() call (both fused sub-steps here) and is gone afterwards."""
    n = 512
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=211, base_z=0.75, vel=0.3, tau_scale=5.0)   # airborne: no contacts
    rng = np.random.default_rng(212)
    body = 6                                            # RF_SHANK
    F = rng.uniform(-30, 30, (n, 3)).astype(np.float32); T = rng.uniform(-3, 3, (n, 3)).astype(np.float32)
    pb = np.array([0.02, -0.01, -0.2], np.float32)
    bt.integrate(2)                                     # baseline without the wrench
    g0, v0 = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.set_external_wrench(body, F, T, pb)
    bt.integrate(2)
    g1, v1 = bt.get_state()
    a, b = gc.copy(), gv.copy()
    o64.step(a, b, n_steps=2, tau_ff=tau, ext=(body, F.astype(np.float64), T.astype(np.float64), pb.astype(np.float64)))
    assert np.abs(v1 - v0).max() > 1e-2                 # the wrench did something
    ev = np.abs(v1 - b); scale = 1.0 + np.abs(b)
    c32, d32 = gc.copy(), gv.copy()
    o32.step(c32, d32, n_steps=2, tau_ff=tau, ext=(body, F.astype(np.float64), T.astype(np.float64), pb.astype(np.float64)))
    e32 = np.abs(d32 - b)
    print(f"external wrench: gv err max {ev.max():.2e} median {np.median(ev.max(1)):.2e}; float32 oracle {e32.max():.2e}")
    assert np.median(ev.max(1)) < max(2e-5, 3 * np.median(e32.max(1)))
    assert np.max(ev / scale) < max(1e-3, 3 * np.max(e32 / scale))
    # cleared after the call: the next step equals the oracle's step without a wrench
    bt.integrate(1)
    g2, v2 = bt.get_state()
    o64.step(a, b, n_steps=1, tau_ff=tau)
    assert np.median(np.abs(v2 - b).max(1)) < 5e-5
    # torque only / force only on a sub-range of environments, device-resident rows
    import torch
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.set_external_wrench(0, torch.from_numpy(F[100:200]).cuda(), None, None, env_begin=100, env_count=100)
    bt.integrate(1)
    g3, v3 = bt.get_state()
    a, b = gc.copy(), gv.copy()
    Fz = np.zeros((n, 3)); Fz[100:200] = F[100:200]
    o64.step(a, b, n_steps=1, tau_ff=tau, ext=(0, Fz, None, None))
    assert np.median(np.abs(v3 - b).max(1)) < 5e-5 and np.abs(v3 - b).max() < 5e-3


def test_terrain_atlas_matches_oracle(capi):
    """N3 per-environment terrains: three height maps in one batch, environments assigned round robin; contact indices
    bit-exact vs the float32 oracle, one step vs the float64 oracle; a single-map atlas equals rsb_batch_set_heightmap."""
    n = 384
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=231, terrain="none", base_z=0.42)
    rng = np.random.default_rng(232)
    xs, ys = 65, 49
    H = (0.1 * rng.uniform(-1, 1, (3, ys, xs))).astype(np.float32)
    H[1] += 0.05; H[2] -= 0.04
    env_map = (np.arange(n) % 3).astype(np.int32)
    bt.set_heightmaps(12.8, 9.6, 0.1, -0.2, H, env_map)
    for o in (o64, o32):
        o.set_heightmaps(12.8, 9.6, 0.1, -0.2, H.astype(np.float64), env_map)
    bt.integrate(1)
    g1, v1 = bt.get_state()
    pts = bt.contact_points(); ct, cnt = bt.contacts()
    a, b = gc.copy(), gv.copy()
    d32 = o32.step(a, b, tau_ff=tau, debug=True)
    shallow = ((np.abs(d32["c_depth"]) < MARGIN) & (d32["c_pt"] >= 0)).any(1)
    assert cnt.sum() > n                                      # contacts exist
    assert ((pts != d32["c_pt"]).any(1) & ~shallow).sum() == 0
    a, b = gc.copy(), gv.copy()
    d = o64.step(a, b, tau_ff=tau, debug=True)
    it = bt.solver_iterations()
    conv = (pts == d["c_pt"]).all(1) & (it < 150) & (d["iters"] < 150)
    assert conv.mean() > 0.9
    assert np.median(np.abs(v1 - b)[conv].max(1)) < 5e-5
    # the maps really differ: the same state on a different map gives a different contact set somewhere
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.set_heightmaps(12.8, 9.6, 0.1, -0.2, H, ((np.arange(n) + 1) % 3).astype(np.int32))
    bt.integrate1()
    assert (bt.contact_points() != pts).any()
    # atlas of one map == the plain height-map call
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.set_heightmaps(12.8, 9.6, 0.1, -0.2, H[:1], np.zeros(n, np.int32))
    bt.integrate(2)
    ga, va = bt.get_state()
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.set_heightmap(xs, ys, 12.8, 9.6, 0.1, -0.2, H[0])
    bt.integrate(2)
    gb, vb = bt.get_state()
    assert np.array_equal(ga, gb) and np.array_equal(va, vb)


def _peer_worker(rank, world, port, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__)))); sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import torch, torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)      # host channel for the 64-byte IPC handles only
    from raisimlib_b200 import capi as c
    from raisimlib_b200.sharding import ObservationGather
    n = 300                                                            # not a multiple of the CTA size
    m = c.Model(os.path.join(RSC, "anymal_c_like.urdf"))
    bt = c.Batch(m, n, device=rank)
    bt.set_ground(0.0)
    rng = np.random.default_rng(500 + rank)
    gc = np.tile(ANYMAL_GC0, (n, 1)); gc[:, 2] = rng.uniform(0.5, 0.7, n); gc[:, 7:] += rng.uniform(-0.2, 0.2, (n, 12))
    bt.set_state(gc.astype(np.float32), (0.3 * rng.standard_normal((n, 18))).astype(np.float32))
    og = ObservationGather(bt, world, rank, n, bt.ob_dim(), mode="peer", device=rank)
    obs = torch.empty((n, bt.ob_dim()), dtype=torch.float32, device=f"cuda:{rank}")
    out = []
    for k in range(3):                                                 # three steps: both buffer parities, counters accumulate
        bt.control_step(None, 2, obs)
        rows = og.gather(obs)
        bt.sync()
        out.append((obs.cpu().numpy().copy(), rows.cpu().numpy().copy()))
        dist.barrier()                                                 # nobody overwrites a buffer a peer is still copying out
    og.close()
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_fused_peer_observation_gather_two_gpus(capi):
    """SURVEY 8e without NCCL on the data path: every rank's step kernel stores its observation rows into every rank's buffer over
    NVLink peer memory (CUDA IPC), counters + a wait kernel close the exchange; rows must equal each rank's own rows, in rank order."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs with peer access")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    world = 2
    procs = [ctx.Process(target=_peer_worker, args=(r, world, 29733, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for k in range(3):
        ref = np.concatenate([got[r][k][0] for r in range(world)])     # every rank's own rows of step k, in rank order
        for r in range(world):
            assert np.array_equal(got[r][k][1], ref), (k, r)


def test_heightmap_narrow_phase_known_answers_on_gpu(capi):
    """a6 on a HeightMap, the analytic cases of tests/test_oracle_kat.py re-run on the kernel: a capsule lying across a ridge (side contact),
    a box resting on a peak (face contact), a sphere on a ridge (edge contact) and a cylinder rolling on its side on the plane."""
    from test_oracle_kat import CAPSULE_X_URDF, CYLINDER_Y_URDF, SPHERE5_URDF, ridge_map, peak_map

    def contacts(urdf, terrain, gc):
        bt = capi.Batch(capi.Model(urdf), 1)
        if terrain is None:
            bt.set_ground(0.0)
        else:
            H, size = terrain
            bt.set_heightmap(H.shape[1], H.shape[0], size, size, 0.0, 0.0, H.astype(np.float32))
        bt.set_state(np.array([gc], np.float32), np.zeros((1, 6), np.float32))
        bt.integrate1()
        ct, cnt = bt.contacts()
        return cnt[0], bt.contact_points()[0][:cnt[0]], ct[0][:cnt[0]]

    K, pt, c = contacts(CAPSULE_X_URDF, ridge_map(), [0.013, 0.27, 0.3 + 0.05 - 0.011, 1, 0, 0, 0])
    assert K == 1 and pt[0] == 2 and abs(c["depth"][0] - 0.011) < 2e-6 and np.allclose(c["normal"][0], [0, 0, 1], atol=1e-5)
    assert np.allclose(c["position"][0], [0.0, 0.27, 0.3 - 0.011], atol=2e-6)
    assert contacts(CAPSULE_X_URDF, ridge_map(), [0.0, 0.0, 0.3 + 0.05 + 1e-4, 1, 0, 0, 0])[0] == 0
    K, pt, c = contacts(BOX_URDF, peak_map(), [0.02, -0.01, 0.2 + 0.1 - 0.007, 1, 0, 0, 0])
    assert K == 1 and pt[0] == 8 and abs(c["depth"][0] - 0.007) < 2e-6 and np.allclose(c["normal"][0], [0, 0, 1], atol=1e-6)
    assert np.allclose(c["position"][0], [0, 0, 0.2], atol=1e-6) and c["pair_index"][0] == 2 * (10 * 20 + 10)
    K, pt, c = contacts(SPHERE5_URDF, ridge_map(), [0.01, 0.033, 0.3 + 0.048, 1, 0, 0, 0])
    d_edge = np.hypot(0.01, 0.048)
    assert K == 1 and abs(c["depth"][0] - (0.05 - d_edge)) < 2e-6 and np.allclose(c["normal"][0], [0.01 / d_edge, 0, 0.048 / d_edge], atol=1e-4)
    for phi in (0.0, 0.7, 1.234):
        K, pt, c = contacts(CYLINDER_Y_URDF, None, [0, 0, 0.1 - 0.002, np.cos(phi / 2), 0, np.sin(phi / 2), 0])
        rim = pt >= 9
        assert rim.sum() == 2 and np.allclose(c["depth"][rim], 0.002, atol=2e-6)
    # rolling without slipping on the plane: the axis stays one radius above the ground
    bt = capi.Batch(capi.Model(CYLINDER_Y_URDF), 1)
    bt.set_ground(0.0)
    bt.set_state(np.array([[0, 0, 0.1, 1, 0, 0, 0]], np.float32), np.array([[0.35, 0, 0, 0, 3.5, 0]], np.float32))
    z = []
    for k in range(100):
        bt.integrate(4)
        z.append(bt.get_state()[0][0, 2])
    assert max(z) - min(z) < 3e-4 and bt.get_state()[0][0, 0] > 0.33


def test_heightmap_narrow_phase_matches_oracle_on_rough_terrain(capi):
    """every candidate type at once: quadrupeds and humanoids dropped in random orientations onto a rough map (spheres on edges and
    vertices, capsule sides on ridges, boxes on peaks); contact lists bit-exact vs the float32 oracle, depths / normals to rounding"""
    for urdf, n, base_z in (("anymal_c_like.urdf", 1024, 0.3), ("atlas_like.urdf", 512, 0.5)):
        t, bt, o64, o32, gc, gv, tau = _setup(capi, urdf, n, seed=501, terrain="hm", base_z=base_z)
        bt.integrate1()
        ct, cnt = bt.contacts(); pts = bt.contact_points()
        a, b = gc.copy(), gv.copy()
        d = o32.step(a, b, tau_ff=tau, debug=True)
        hard = _index_parity(pts, cnt, d, f"narrow phase {urdf}")
        same = (pts == d["c_pt"]).all(1)
        kinds = np.bincount(t["pt_type"][pts[pts >= 0]], minlength=3)
        print(f"   contacts by candidate type (sphere/point, segment, box face): {kinds.tolist()}; identical lists {100 * same.mean():.2f}%")
        assert hard.mean() < 0.003, f"contact lists differ in envs {np.where(hard)[0][:10]}"     # near-ties between triangles (1e-6 m rule) under different rounding
        assert kinds[0] > 500 and kinds[1] + kinds[2] > 5
        live = same[:, None] & (d["c_pt"] >= 0)
        pair_same = (ct["pair_index"] == d["c_pair"])[live].mean()
        assert pair_same > 0.995                                                                   # same reason: which of two triangles sharing an edge
        ok = live & (ct["pair_index"] == d["c_pair"])
        rad = np.where(d["c_pt"] >= 0, t["pt_rad"][np.maximum(d["c_pt"], 0)], 0.0)
        # normal = (centre - closest point) / distance: both points carry float32 rounding of coordinates up to 12.8 m (ulp 9.5e-7), the
        # closest point a few operations' worth, so the normal is conditioned like 3e-6 / distance
        tol_n = 2e-6 + 3e-6 / np.maximum(rad - d["c_depth"], 1e-4)
        en = np.abs(ct["normal"] - d["c_normal"]).max(2)
        print(f"   worst normal error / tolerance {np.max(en[ok] / tol_n[ok]):.2f}, worst depth error {np.abs(ct['depth'] - d['c_depth'])[ok].max():.2e}")
        assert np.abs(ct["depth"] - d["c_depth"])[ok].max() < 5e-6 and (en[ok] < tol_n[ok]).all()


def test_cpp_generic_vectorized_environment_example(capi):
    """VERDICT r1 item 6: VectorizedEnvironment<ENVIRONMENT> runs N objects of an upstream-shaped environment class (own observation,
    reward, termination on the host; examples/rsg_custom/Environment.hpp) in lock step on one batch: ONE launch per control step although
    every environment calls world_->integrate() four times, and environment 0 reproduces the same class run standalone bit for bit."""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "examples", "custom_vecenv")
    if not os.path.exists(exe):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "examples")])
    out = subprocess.run([exe, os.path.join(RSC, "anymal_c_like.urdf"), "256"], capture_output=True, text=True, timeout=300)
    print(out.stdout, out.stderr[-500:])
    assert out.returncode == 0, out.stdout + out.stderr
    assert "1.00 per control step" in out.stdout and "max |difference| over observations and rewards 0" in out.stdout


def test_pybind_dlpack_zero_copy_views(capi):
    """N4: the pybind11 module hands out the batch rows as DLPack capsules; torch.from_dlpack() gives strided CUDA tensors that alias
    the memory the step kernel works on (writes are seen by the next integrate(), results appear in the tensors), and a control step
    driven entirely through device tensors equals the ctypes path bit for bit."""
    import torch
    from raisimlib_b200 import _rsb_py
    n = 96
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=601, base_z=0.55, joint_scale=0.2)
    pm = _rsb_py.Model(os.path.join(RSC, "anymal_c_like.urdf"))
    pb = _rsb_py.Batch(pm, n, 0)
    pb.set_ground(0.0)
    tg, tv = torch.from_dlpack(pb.gc()), torch.from_dlpack(pb.gv())
    assert tg.is_cuda and tg.shape == (n, 19) and tv.shape == (n, 18) and tg.stride(0) >= 19 and tg.dtype == torch.float32
    tg.copy_(torch.from_numpy(gc.astype(np.float32)).cuda()); tv.copy_(torch.from_numpy(gv.astype(np.float32)).cuda())     # write through the views
    kp = [0.0] * 6 + [120.0] * 12; kd = [0.0] * 6 + [3.0] * 12
    pb.set_pd_gains(kp, kd)
    target = torch.from_numpy(np.tile(ANYMAL_GC0, (n, 1)).astype(np.float32)).cuda().contiguous()
    obs = torch.empty((n, pb.ob_dim), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    pb.control_step(target.data_ptr(), 4, obs.data_ptr())
    pb.sync()
    # the ctypes path from the same state: a fresh batch at the library defaults, like the pybind one
    bt = capi.Batch(capi.Model(os.path.join(RSC, "anymal_c_like.urdf")), n)
    bt.set_ground(0.0)
    bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
    bt.set_control_mode(capi.PD_PLUS_FEEDFORWARD_TORQUE)
    bt.set_pd_gains(np.array(kp), np.array(kd))
    bt.set_pd_target(target.cpu().numpy(), np.zeros((n, 18), np.float32))
    bt.integrate(4)
    g_ref, v_ref = bt.get_state()
    assert np.array_equal(tg.cpu().numpy(), g_ref) and np.array_equal(tv.cpu().numpy(), v_ref)          # the tensors ARE the state
    assert np.array_equal(obs.cpu().numpy(), bt.observe())
    del pb                                                             # the tensors keep the batch alive
    assert torch.isfinite(tg).all()


def test_actuator_effort_limits_match_oracle(capi):
    """N2 effort limits on the GPU: (1) the pendulum KAT (alpha = tau_max / I whatever the gains; unsaturated law untouched; feed-forward
    limited too), generic kernel; (2) the quadruped instance with stiff gains and far targets, where most leg joints saturate at the
    URDF's 80 N m in the first steps: state parity with the float64 oracle over 20 steps and the same set of saturated joints."""
    from test_oracle_kat import EFFORT_PENDULUM
    I = 0.1 + 2.0 * 0.5 ** 2
    bt = capi.Batch(capi.Model(EFFORT_PENDULUM), 4)
    bt.set_params(gravity=(0.0, 0.0, 0.0))
    bt.set_control_mode(capi.PD_PLUS_FEEDFORWARD_TORQUE)
    bt.set_pd_gains(np.array([4000.0]), np.array([0.0]))
    bt.set_state(np.zeros((4, 1), np.float32), np.zeros((4, 1), np.float32))
    bt.set_pd_target(np.array([[1.0], [-1.0], [0.0002], [-0.0002]], np.float32), np.zeros((4, 1), np.float32))
    bt.integrate(1)
    _, v = bt.get_state()
    free = 0.0025 * 4000.0 * 0.0002 / (I + 0.0025 ** 2 * 4000.0)         # 0.8 N m asked, 1.5 available: implicit PD
    assert np.allclose(v[:, 0], [1.5 / I * 0.0025, -1.5 / I * 0.0025, free, -free], rtol=2e-6, atol=1e-9)
    bt.set_control_mode(capi.FORCE_AND_TORQUE)
    bt.set_state(np.zeros((4, 1), np.float32), np.zeros((4, 1), np.float32))
    bt.set_generalized_force(np.array([[7.0], [-7.0], [1.0], [0.0]], np.float32))
    bt.integrate(1)
    _, v = bt.get_state()
    assert np.allclose(v[:, 0], [1.5 / I * 0.0025, -1.5 / I * 0.0025, 1.0 / I * 0.0025, 0.0], rtol=2e-6, atol=1e-9)
    # quadruped
    n = 256
    t, bt, o64, o32, gc, gv, tau = _setup(capi, "anymal_c_like.urdf", n, seed=777, base_z=0.62, vel=0.2, tau_scale=0.0, joint_scale=0.2)
    rng = np.random.default_rng(778)
    kp = np.r_[np.zeros(6), 2000.0 * np.ones(12)]; kd = np.r_[np.zeros(6), 20.0 * np.ones(12)]
    pt = gc.copy(); pt[:, 7:] += rng.uniform(-0.6, 0.6, (n, 12))          # 2000 N m / rad * 0.3 rad >> 80 N m
    vt = np.zeros((n, 18))
    bt.set_control_mode(capi.PD_PLUS_FEEDFORWARD_TORQUE)
    bt.set_pd_gains(kp, kd)
    bt.set_pd_target(pt.astype(np.float32), vt.astype(np.float32))
    a, b = gc.copy(), gv.copy()
    sat_steps = 0
    for k in range(20):
        bt.integrate(1)
        d = o64.step(a, b, ptarget=pt.astype(np.float32).astype(np.float64), vtarget=vt, kp=kp, kd=kd, debug=True)
        ta = bt.generalized_force()           # the generalized force applied over the last step (feed-forward + PD, after the limit)
        if ta is not None and k == 0:
            sat_ref = np.abs(np.abs(d["tau_applied"][:, 6:]) - 80.0) < 1e-9
            sat_gpu = np.abs(np.abs(ta[:, 6:]) - 80.0) < 1e-4
            assert sat_ref.mean() > 0.3 and (sat_ref == sat_gpu).mean() > 0.999
            sat_steps += 1
    g, v = bt.get_state()
    conv = (bt.solver_status() <= 1) & (d["status"] <= 1)
    eg = np.abs(g - a).max(1)[conv]; ev = np.abs(v - b).max(1)[conv]
    print(f"effort limits, 20 steps: median |dgc| {np.median(eg):.2e} max {eg.max():.2e}; median |dgv| {np.median(ev):.2e}")
    assert np.median(eg) < 2e-5 and np.quantile(eg, 0.9) < 2e-4
