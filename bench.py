#!/usr/bin/env python3
"""bench.py -- env-steps/s of the batched World::integrate() hot path (BASELINE.json metric).

Headline workload (BASELINE.json configs[2], weak-scaled per GPU -> configs[4] at 8 GPUs):
  4096 ANYmal-C-like environments per GPU on a 513x513 random rough height field (51.2 m square,
  3-octave value noise, +-0.10 m), PD stance control with per-control-step target jitter.
A bench "step" is one RaisimGym control step: ONE fused launch of 4 sub-steps of World::integrate()
for every environment (= 4 x 4096 env-steps per GPU) that also writes the observation rows.  At N > 1 the
observation all-gather is FUSED into that launch: every finished row is stored straight into every rank's
gathered buffer over NVLink peer memory while the kernel runs, and one tiny wait kernel per step closes the
exchange (--nccl-gather times the torch.distributed all-gather it replaces).

  value   env-steps/s with state, targets and terrain resident in HBM (targets read in place)
  e2e     same metric through the C-ABI with HOST buffers: pinned H2D of the PD targets and D2H of
          the (all-gathered) observation rows inside the timed region
  side_results   (N = 1 only) the same measurement on BASELINE.json configs[1] (flat ground, random joint
          torques, robots fall) and configs[3] (Atlas-like humanoid standing on box feet), each with its own
          CPU baseline; the headline stays configs[2]
  --impl reference   the CPU path (oracle port of World::integrate(), OpenMP over envs, all host
          cores) on the same workload -- /root/reference holds no buildable source (SURVEY.md 8c)
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
SUBSTEPS = 4
GC0 = np.array([0, 0, 0.57, 1, 0, 0, 0, 0.03, 0.4, -0.8, -0.03, 0.4, -0.8, 0.03, -0.4, 0.8, -0.03, -0.4, 0.8], dtype=np.float64)
KP, KD = 300.0, 8.0
HM = dict(xs=513, ys=513, size=51.2, amp=0.10)
RING = 8            # distinct PD-target / torque sets cycled through (synthetic "policy output")
SETTLE = 40         # untimed control steps run while BUILDING the workload: robots are dropped from 0.75 m and must stand
                    # on the terrain before warm-up starts, whatever --warmup the caller passes
L2_FLUSH_BYTES = 256 << 20
SOLVER = dict(threshold=1e-6)   # everything else at the library defaults (rsb_params_default): accel_m=2, accel_start=6, stall_window=8, stall_reg=0.02


def value_noise(rng, n, size_cells):
    """bilinear value noise on an n x n grid with lattice spacing size_cells"""
    m = (n - 1) // size_cells + 2
    lat = rng.uniform(-1, 1, (m, m))
    x = np.arange(n) / size_cells
    i = x.astype(int); f = x - i
    a = lat[np.ix_(i, i)]; b = lat[np.ix_(i, i + 1)]; c = lat[np.ix_(i + 1, i)]; d = lat[np.ix_(i + 1, i + 1)]
    fy, fx = f[:, None], f[None, :]
    return a * (1 - fy) * (1 - fx) + b * (1 - fy) * fx + c * fy * (1 - fx) + d * fy * fx


def make_workload(rank, n_envs):
    """headline workload (configs[2]); kept as a function of its own: tools/ and tests/ build it too"""
    rng = np.random.default_rng(3000 + rank)
    n = HM["xs"]
    H = value_noise(rng, n, 32) + 0.5 * value_noise(rng, n, 8) + 0.25 * value_noise(rng, n, 2)
    H = (HM["amp"] * H / np.abs(H).max()).astype(np.float32)
    gc = np.tile(GC0, (n_envs, 1))
    gc[:, 0:2] = rng.uniform(-0.4 * HM["size"], 0.4 * HM["size"], (n_envs, 2))      # inner 80 % of the map
    gc[:, 2] = 0.75
    gc[:, 7:] += rng.uniform(-0.2, 0.2, (n_envs, 12))
    yaw = rng.uniform(-np.pi, np.pi, n_envs)
    gc[:, 3] = np.cos(yaw / 2); gc[:, 6] = np.sin(yaw / 2)
    gv = np.zeros((n_envs, 18))
    targets = np.tile(GC0, (RING, n_envs, 1))
    targets[:, :, 7:] += rng.uniform(-0.15, 0.15, (RING, n_envs, 12))
    kp = np.r_[np.zeros(6), KP * np.ones(12)]; kd = np.r_[np.zeros(6), KD * np.ones(12)]
    return H, gc, gv, targets, kp, kd


class Workload:
    """one BASELINE.json config as data: model, terrain, initial state, control ring"""

    def __init__(self, key, rank, n):
        self.key, self.n = key, n
        if key == "c3":      # configs[2]: rough height field, PD stance with target jitter (contact-heavy headline)
            H, gc, gv, targets, kp, kd = make_workload(rank, n)
            self.urdf, self.H, self.gc, self.gv, self.kp, self.kd = "anymal_c_like.urdf", H, gc, gv, kp, kd
            self.mode, self.ring, self.settle = "pd", targets, SETTLE
            self.name = workload_string(n)
        elif key == "c2":    # configs[1]: flat ground, random joint torques resampled every control step, robots fall (SURVEY 8d C2)
            rng = np.random.default_rng(2000 + rank)
            gc = np.tile(GC0, (n, 1)); gc[:, 2] = rng.uniform(0.45, 0.6, n); gc[:, 7:] += rng.uniform(-0.2, 0.2, (n, 12))
            gv = 0.5 * rng.standard_normal((n, 18))
            tau = rng.uniform(-20, 20, (RING, n, 18)); tau[:, :, :6] = 0
            self.urdf, self.H, self.gc, self.gv, self.kp, self.kd = "anymal_c_like.urdf", None, gc, gv, None, None
            self.mode, self.ring, self.settle = "torque", tau, 250      # 1000 sub-steps: every robot lies on the ground
            self.name = (f"{n} ANYmal-C-like envs per GPU on flat ground, joint torques U(-20,20) N m resampled every {SUBSTEPS} sub-steps, "
                         f"robots fallen (after 1000 sub-steps), dt=0.0025, {SUBSTEPS} sub-steps fused per step")
        elif key == "c4":    # configs[3]: Atlas-like humanoid (30 joints, depth-10 tree) standing on box feet under PD
            rng = np.random.default_rng(4000 + rank)
            gc0 = np.zeros(37); gc0[2] = 0.95; gc0[3] = 1.0
            gc = np.tile(gc0, (n, 1)); gc[:, 7:] += rng.uniform(-0.05, 0.05, (n, 30))
            gv = np.zeros((n, 36))
            targets = np.tile(gc0, (RING, n, 1)); targets[:, :, 7:] += rng.uniform(-0.03, 0.03, (RING, n, 30))
            self.urdf, self.H, self.gc, self.gv = "atlas_like.urdf", None, gc, gv
            self.kp = np.r_[np.zeros(6), 400.0 * np.ones(30)]; self.kd = np.r_[np.zeros(6), 10.0 * np.ones(30)]
            self.mode, self.ring, self.settle = "pd", targets, 20
            self.name = (f"{n} Atlas-like humanoid envs per GPU (30 joints) standing on flat ground on box feet (8 corner contacts), PD kp=400 kd=10 "
                         f"with target jitter, dt=0.0025, {SUBSTEPS} sub-steps fused per step")
        else:
            raise ValueError(key)
        self.nq, self.nv = self.gc.shape[1], self.gv.shape[1]


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML in a
    background thread every 5 ms (nvidia-smi -lms needs > 100 ms to produce its first row, longer
    than a short timed region)."""
    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz, self.stop_flag, self.t = index, [], set(), None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            uuid_order = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(uuid_order.split(",")[index]) if uuid_order and uuid_order.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _loop(self):
        while not self.stop_flag:
            try:
                self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                r = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.BAD.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        self.stop_flag = True
        self.t.join(timeout=1)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.sm)}


def usable_cores():
    """host threads this process may really use: CPU affinity, capped by the cgroup CPU quota"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p_ = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = max(1, min(n, q // p_))
        except Exception:
            pass
    return n


def algorithmic_bytes_per_env_step(nq, nv, nj, kbar):
    # SURVEY.md 8(d): reads gc, gv, tau_ff, pTarget, vTarget; writes gc+, gv+, tau_applied, count, 12 words per contact
    return 4.0 * (2 * nq + 3 * nv + 2 * nj + 1 + 12.0 * kbar)


DUMP_MAX_BYTES = 64 << 20


def write_outputs(path, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, every array one row per environment (all ranks, rank order):
      obs      observation rows of the last timed step of the device-resident arm (the headline value's path)
      gc, gv   generalized coordinates / velocities right after that step
      obs_e2e  observation rows of the last timed step of the host-buffer (e2e) arm
    The workload is seeded, so the same arguments give the same inputs on every run and two builds can be compared file by file.
    Above DUMP_MAX_BYTES in all, a fixed, seeded sample of environments is kept: the same rows of every array, their indices in
    env_index.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(a, np.float64 if a.dtype == np.float64 else np.float32) for k, a in arrays.items()}
    rows = {a.shape[0] for a in arrays.values()}
    assert len(rows) == 1, {k: a.shape for k, a in arrays.items()}
    rows = rows.pop()
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    budget = DUMP_MAX_BYTES - 4096                    # headroom for the .npy headers
    if rows * row_bytes > budget:
        keep = budget // (row_bytes + 8)
        idx = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


# ------------------------------------------------------------------ CPU arm --------------------------
class CpuSim:
    """the oracle port driving one Workload (a restatement of World::integrate(), NOT RaiSim's binary): OpenMP over
    environments on every usable host core.  build = "native": the timing build (-O3 -march=native, FMA contraction on,
    compiled on this machine); "parity": the checker's build (-march=x86-64-v3 -ffp-contract=off)."""

    def __init__(self, wl, precision="f64", build="native"):
        from oracle.oracle import Oracle, native_build_available
        from oracle.urdf_tables import load_tables
        from raisimlib_b200 import RSC_DIR
        self.wl, self.precision = wl, precision
        self.build = build if (build == "parity" or native_build_available()) else "parity (native build failed)"
        self.o = Oracle(load_tables(os.path.join(RSC_DIR, wl.urdf)), precision=precision, params=dict(slip_bisect=1, **SOLVER),   # CPU-tuned slip search
                        build="native" if self.build == "native" else "parity")
        if wl.H is not None:
            self.o.set_heightmap(HM["xs"], HM["ys"], HM["size"], HM["size"], 0.0, 0.0, wl.H.astype(np.float64))
        else:
            self.o.set_ground(0.0)
        self.gc, self.gv = wl.gc.copy(), wl.gv.copy()
        self.cores = usable_cores()          # explicit: torchrun exports OMP_NUM_THREADS=1
        self.vt = np.zeros((wl.n, wl.nv))
        self.k = 0

    def control_step(self):
        wl, r = self.wl, self.wl.ring[self.k % RING]
        if wl.mode == "pd":
            self.o.step(self.gc, self.gv, n_steps=SUBSTEPS, ptarget=r, vtarget=self.vt, kp=wl.kp, kd=wl.kd, nthreads=self.cores)
        else:
            self.o.step(self.gc, self.gv, n_steps=SUBSTEPS, tau_ff=r, nthreads=self.cores)
        self.k += 1

    def rate(self, settle, max_steps, budget_s):
        """env-steps/s over at most max_steps control steps / budget_s seconds, after `settle` untimed control steps"""
        for _ in range(settle):
            self.control_step()
        t0 = time.perf_counter(); done = 0
        while done < max_steps and (done == 0 or time.perf_counter() - t0 < budget_s):
            self.control_step(); done += 1
        dt = time.perf_counter() - t0
        return self.wl.n * SUBSTEPS * done / dt, done


def cpu_baseline(key, sample_envs, max_steps, budget_s, both_precisions=False):
    """bounded sample of the same workload on all host cores; settling is part of building the workload (untimed)"""
    wl = Workload(key, 0, sample_envs)
    sim = CpuSim(wl, "f64")
    val, done = sim.rate(wl.settle + 3, max_steps, budget_s)
    out = {"value": val, "unit": "env-steps/s", "cores": sim.cores, "kind": "port", "precision": "f64", "build": build_string(sim.build),
           "per_thread": val / sim.cores,
           "sample": f"{sample_envs} envs x {SUBSTEPS * done} sub-steps of the same workload after the same settling phase as the GPU arm "
                     f"(float64 oracle port, bisection slip search, OpenMP over envs, {sim.cores} threads)"}
    if both_precisions:
        s32 = CpuSim(wl, "f32")
        v32, d32 = s32.rate(wl.settle + 3, max_steps, budget_s)
        out["value_f32"] = v32
        out["per_thread_f32"] = v32 / s32.cores
    return out


def build_string(build):
    return {"native": "timing build: g++ -O3 -march=native -fopenmp (FMA contraction on), compiled on this host",
            "parity": "parity build: g++ -O3 -march=x86-64-v3 -ffp-contract=off -fopenmp"}.get(build, build)


def workload_string(n):
    return (f"{n} ANYmal-C-like envs per GPU on 513x513 rough height field (+-0.10 m), PD stance kp={KP} kd={KD}, dt=0.0025, "
            f"{SUBSTEPS} sub-steps fused per step")


def run_reference(args):
    """--impl reference: the CPU path on this box's host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = ENVS_PER_GPU
    wl = Workload("c3", 0, n)
    sim = CpuSim(wl, "f64")
    W = max(args.warmup, 3)
    for _ in range(wl.settle + W):
        sim.control_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sim.control_step()
    dt = time.perf_counter() - t0
    val = n * SUBSTEPS * args.steps / dt
    # float32 instance of the same port, for a same-precision comparison with the GPU arm (bounded: a quarter of the steps)
    s32 = CpuSim(wl, "f32")
    v32, _ = s32.rate(wl.settle + W, max(2, args.steps // 4), 20.0)
    line = {"impl": "reference", "metric": "env-steps/s", "value": val, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": W, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(n), "envs_per_gpu": n, "substeps_per_step": SUBSTEPS,
                       "arm": f"CPU oracle port (a restatement, not RaiSim's binary), float64, OpenMP over envs, {sim.cores} threads; each step = the full per-GPU workload"},
            "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": sim.cores, "kind": "port", "precision": "f64", "build": build_string(sim.build),
                             "per_thread": val / sim.cores, "value_f32": v32, "per_thread_f32": v32 / sim.cores,
                             "sample": f"{n} envs x {SUBSTEPS * args.steps} sub-steps (the full per-GPU workload), float64, OpenMP over envs, {sim.cores} threads"},
            "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm --------------------------
class GpuSim:
    """one Workload on one GPU through the C-ABI (raisimlib_b200.capi), state / control ring resident in HBM"""

    def __init__(self, wl, local, stream):
        import torch
        from raisimlib_b200 import capi, RSC_DIR
        self.wl, self.torch = wl, torch
        self.model = capi.Model(os.path.join(RSC_DIR, wl.urdf))
        bt = self.bt = capi.Batch(self.model, wl.n, device=local)
        bt.set_params(**SOLVER)
        if wl.H is not None:
            bt.set_heightmap(HM["xs"], HM["ys"], HM["size"], HM["size"], 0.0, 0.0, wl.H)
        else:
            bt.set_ground(0.0)
        bt.set_stream(stream.cuda_stream)
        bt.set_state(wl.gc.astype(np.float32), wl.gv.astype(np.float32))
        self.ring_dev = torch.tensor(wl.ring, dtype=torch.float32, device="cuda")           # [RING, n, nq | nv] resident in HBM
        self.ring_pin = torch.tensor(wl.ring, dtype=torch.float32).pin_memory()             # host copies for the e2e arm
        if wl.mode == "pd":
            bt.set_pd_gains(wl.kp, wl.kd)
            bt.set_pd_target(self.ring_dev[0], torch.zeros((wl.n, wl.nv), dtype=torch.float32, device="cuda"))
        else:
            bt.set_control_mode(capi.FORCE_AND_TORQUE)
        self.od = bt.ob_dim()
        self.obs = [torch.empty((wl.n, self.od), dtype=torch.float32, device="cuda") for _ in range(2)]     # double-buffered observation rows
        self.obs_host = torch.empty((wl.n, self.od), dtype=torch.float32).pin_memory()

    def step_resident(self, k, obs=None):
        """one control step, everything resident in HBM: ONE fused launch (4 x World::integrate() + observation rows)"""
        bt, r = self.bt, self.ring_dev[k % RING]
        obs = self.obs[k & 1] if obs is None else obs
        if self.wl.mode == "pd":
            bt.bind_pd_target(r)                 # resident targets read in place (zero-copy)
        else:
            bt.set_generalized_force(r)          # setGeneralizedForce: one device-to-device row copy
        bt.control_step(None, SUBSTEPS, obs)
        return obs

    def step_host(self, k, obs_host=None):
        """the call a user makes: control rows (pinned host) in, 4 fused sub-steps, observation rows (pinned host) out"""
        bt, r = self.bt, self.ring_pin[k % RING]
        obs_host = self.obs_host if obs_host is None else obs_host
        if self.wl.mode == "pd":
            bt.control_step(r, SUBSTEPS, obs_host)
        else:
            bt.set_generalized_force(r)
            bt.control_step(None, SUBSTEPS, obs_host)
        return obs_host

    def stats(self):
        _, cnt = self.bt.contacts()
        it = self.bt.solver_iterations()
        res = self.bt.solver_residual()
        g, _v = self.bt.get_state()
        zmin = 0.25 if self.wl.urdf.startswith("anymal") else 0.8
        return {"mean_contacts_per_env": float(cnt.mean()), "contacts_histogram": np.bincount(cnt, minlength=9).tolist(),
                "mean_solver_sweeps": float(it.mean()), "max_solver_sweeps": int(it.max()),
                "sweeps_histogram": {"0": int((it == 0).sum()), "1-2": int(((it >= 1) & (it <= 2)).sum()), "3-4": int(((it >= 3) & (it <= 4)).sum()),
                                     "5-8": int(((it >= 5) & (it <= 8)).sum()), "9-16": int(((it >= 9) & (it <= 16)).sum()),
                                     "17-32": int(((it >= 17) & (it <= 32)).sum()), "33+": int((it >= 33).sum())},
                "non_converged_fraction": float((res >= SOLVER["threshold"]).mean()), "standing_fraction": float((g[:, 2] > zmin).mean())}


def side_result(key, local, stream, flush, steps, warmup):
    """N = 1 side measurement of another BASELINE config: same timing rules as the headline (CUDA events per launch on the
    launching stream, L2 flushed between timed iterations), fewer steps; with its own bounded CPU baseline"""
    import torch
    wl = Workload(key, 0, ENVS_PER_GPU)
    sim = GpuSim(wl, local, stream)
    for k in range(wl.settle + warmup):
        sim.step_resident(k)
    torch.cuda.synchronize()
    k0 = wl.settle + warmup
    out = {}
    for arm in ("value", "e2e"):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for k in range(steps):
            flush.fill_(float(k))
            ev[k][0].record(stream)
            if arm == "value":
                sim.step_resident(k0 + k)
            else:
                sim.step_host(k0 + k)
            ev[k][1].record(stream)
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        out[arm] = wl.n * SUBSTEPS * steps / (ms * 1e-3)
        out[arm + "_ms_per_step"] = ms / steps
        k0 += steps
    st = sim.stats()
    nj = wl.nq - 7
    B = algorithmic_bytes_per_env_step(wl.nq, wl.nv, nj, st["mean_contacts_per_env"])
    res = {"workload": wl.name, "value": out["value"], "unit": "env-steps/s", "ms_per_step": out["value_ms_per_step"], "steps": steps, "warmup": warmup,
           "e2e": {"value": out["e2e"], "unit": "env-steps/s", "h2d_bytes_per_step": int(wl.n * (wl.nq if wl.mode == "pd" else wl.nv) * 4),
                   "d2h_bytes_per_step": int(wl.n * sim.od * 4)},
           "algorithmic_bytes_per_env_step": B, **st}
    del sim
    res["cpu_baseline"] = cpu_baseline(key, 1024 if key == "c4" else ENVS_PER_GPU, 40, 6.0)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=25)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-results", action="store_true")
    ap.add_argument("--nccl-gather", action="store_true", help="N > 1: NCCL all-gather after the step instead of the fused peer-memory gather, for comparison")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy (see write_outputs)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from raisimlib_b200.sharding import ObservationGather

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W = max(args.warmup, 3)
    n = args.envs
    stream = torch.cuda.current_stream()
    wl = Workload("c3", rank, n)
    sim = GpuSim(wl, local, stream)
    bt, od = sim.bt, sim.od
    gather = ObservationGather(bt, world, rank, n, od, mode="nccl" if args.nccl_gather else "peer", device=local) if world > 1 else None
    shared = None
    if world > 1:
        # e2e arm at N > 1: the host-side consumer reads one [world*n, obDim] array in shared, page-locked memory; every
        # rank's step kernel writes its own rows in place over its own PCIe link (no NVLink hop, no D2H funnel on rank 0)
        from raisimlib_b200.sharding import SharedHostRows
        shared = SharedHostRows(f"bench_{os.environ.get('MASTER_PORT', '0')}", world, rank, n, od)
        e2e_step = [0]
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device="cuda")

    def control_step(k):
        obs = sim.step_resident(k)
        if gather is not None:
            gather.gather(obs)                   # the only collective of the path (SURVEY 8e)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(host_io, steps, step0):
        # one event pair per step around the whole step (ms_per_step); a second pair around the launch alone only where the step
        # holds more than the launch (the NCCL arm's all-gather: with the fused peer gather the arrival wait is part of the launch and
        # nothing else is enqueued) -- two extra event records cost ~5 us of stream time per step.
        # Also returns the observation rows the caller received from the last step (all ranks' rows at N > 1).
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        inner = gather is not None and gather.mode == "nccl" and not host_io
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] if inner else ev
        rows = None
        barrier()
        for k in range(steps):
            flush.fill_(float(k))                            # evict L2 between timed iterations (256 MiB > 126 MB L2)
            ev[k][0].record(stream)
            if host_io:
                rows = sim.step_host(step0 + k, shared.local if world > 1 else None)
                if world > 1:
                    # N > 1: same call per rank (it returns when this rank's rows are in host memory); shared-memory flags are
                    # the barrier after which the trainer's rank may read every row
                    e2e_step[0] += 1
                    shared.publish_and_wait(e2e_step[0])
                    rows = shared.all
                ev[k][1].record(stream)
                continue
            if inner:
                kev[k][0].record(stream)
            rows = obs = sim.step_resident(step0 + k)        # ONE launch: 4 fused sub-steps + observation rows
            if inner:
                kev[k][1].record(stream)
            if gather is not None:
                rows = gather.gather(obs)                    # fused: nothing is enqueued (the launch ends when the rows are complete); nccl mode: the all-gather
            ev[k][1].record(stream)
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in ev)
        kms = sum(a.elapsed_time(b) for a, b in kev)
        t = torch.tensor([ms, kms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)         # max over ranks
        return float(t[0]), float(t[1]), rows

    def all_ranks(a):
        """rows of every rank in rank order (a collective at N > 1: every rank calls it)"""
        if world == 1:
            return a
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        out = torch.empty((world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device="cuda")
        dist.all_gather_into_tensor(out, t)
        return out.cpu().numpy()

    for k in range(wl.settle):       # workload construction (untimed): land and settle
        control_step(k)
    for k in range(W):
        control_step(k)
    barrier()
    l0 = bt.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, ms_kernel, rows = timed(False, args.steps, W)
    launches = bt.launch_count() - l0
    if args.dump_outputs:
        # read outside the timed region, before the e2e arm advances the state
        outputs = {"obs": rows.cpu().numpy()}
        outputs["gc"], outputs["gv"] = (all_ranks(a) for a in bt.get_state())
    ms_e2e, _, rows = timed(True, args.steps, W + args.steps)
    if args.dump_outputs:
        outputs["obs_e2e"] = np.array(rows.numpy() if isinstance(rows, torch.Tensor) else rows)
        if rank == 0:
            write_outputs(args.dump_outputs, outputs)
    clocks = sampler.stop() if rank == 0 else None
    st = sim.stats()
    keys = ["mean_contacts_per_env", "mean_solver_sweeps", "non_converged_fraction", "standing_fraction"]
    stats = torch.tensor([st[k] for k in keys] + [float(st["max_solver_sweeps"])], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = stats[-1:].clone()
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        stats /= world
        stats[-1] = mx[0]
    if rank == 0:
        total_env_steps = world * n * SUBSTEPS * args.steps
        value = total_env_steps / (ms_dev * 1e-3)
        e2e = total_env_steps / (ms_e2e * 1e-3)
        kbar = float(stats[0])
        B = algorithmic_bytes_per_env_step(19, 18, 12, kbar)
        launch_ms = ms_kernel / args.steps
        achieved = B * n * SUBSTEPS / (launch_ms * 1e-3) / 1e9
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        try:
            mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            peak, peak_src = float(mp["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["dram_bytes_per_launch"]
        except Exception:
            pass
        line = {
            "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(n),
                       "envs_per_gpu": n, "substeps_per_step": SUBSTEPS, "l2": "flushed between timed iterations (256 MiB write)",
                       "solver": "library defaults: Anderson-accelerated per-contact Gauss-Seidel (accel_m=2 from sweep 6), threshold 1e-6, maxIter 150, stagnation window 8 with compliant fallback (stall_reg 0.02)",
                       "mean_contacts_per_env": kbar, "contacts_histogram_rank0": st["contacts_histogram"],
                       "mean_solver_sweeps": float(stats[1]), "max_solver_sweeps": float(stats[4]), "sweeps_histogram_rank0": st["sweeps_histogram"],
                       "non_converged_fraction": float(stats[2]), "standing_fraction": float(stats[3]),
                       "regime": "standing under PD targets that jump +-0.15 rad every control step: a stiff-legged quadruped on rough ground rests on 3 feet most "
                                 "of the time (K = 3.3 with fixed targets, 1 % of the environments change their contact set per step) and the target jumps shake "
                                 "one more foot loose (K = 2.7-2.8, 24 % change per step): a light contact regime; configs 2 and 4 in side_results are the heavy ones",
                       "parallelism": f"env-shard x{world}" + ((", observation all-gather fused into the step kernel over NVLink peer memory" if not args.nccl_gather else ", NCCL obs all-gather after the step") if world > 1 else "")},
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": int(world * n * 19 * 4), "d2h_bytes_per_step": int(world * n * od * 4),
                    "path": "pinned host targets and observation rows read / written in place by the step kernel (zero-copy over PCIe)"
                            + ("; rows of all ranks land in one shared page-locked array, shared-memory flags as barrier" if world > 1 else "")},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "kernel": "rsb_step_kernel (fused FK+CRBA+RNEA+narrow-phase+contact solver+integrate)",
                         "algorithmic_bytes_per_env_step": B, "launch_ms": launch_ms, "peak_source": peak_src,
                         "note": "path is FP32-latency/issue bound, not HBM bound (SURVEY.md 7 hard part 2); see DESIGN.md roofline"},
            "clocks": clocks,
        }
        if gather is not None:
            line["gather"] = gather.report()
    if gather is not None:
        gather.close()
    del sim
    if rank == 0:
        if world == 1 and not args.no_side_results:
            side_steps = max(10, min(40, args.steps))
            line["side_results"] = {"config2_flat_random_torques_fallen": side_result("c2", local, stream, flush, side_steps, 5),
                                    "config4_atlas_standing": side_result("c4", local, stream, flush, side_steps, 5)}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline("c3", n, 100, 12.0, both_precisions=True)
        print(json.dumps(line), flush=True)
    if shared is not None:
        shared.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True       # the benchmark leaves the source tree as it found it
    main()
