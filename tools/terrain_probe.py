#!/usr/bin/env python3
"""What do height scans and terrain rays cost next to the gym step?  On the benchmark workload (4096 ANYmal-like environments on the
513^2 rough height field, settled on it), CUDA events time, each over many back-to-back calls on the batch's stream:
  - the base height scan (17 x 11 grid, 0.1 m pitch: 187 points),
  - the foot scans (4 foot frames x a ring of 8 points, 0.1 m radius) right after a state change (kinematics launch + scan) and on an
    unchanged state (scan alone),
  - a 10 m lidar of 16 x 32 rays fixed in the base frame,
  - rsb_batch_gym_step alone against rsb_batch_gym_step followed by the base scan.
The 1 MiB map stays in the 126 MB L2 across calls (warm L2: that is what a training loop sees).  Card name and power limit are read in
the same run.  Usage: python tools/terrain_probe.py [--out FILE]"""
import argparse
import os
import subprocess
import sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from raisimlib_b200 import capi, RSC_DIR


def timed(stream, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_us(fn, name, reps=50):
    """mean device time of the kernels whose name contains `name` over `reps` calls of fn (torch.profiler, CUDA activity)"""
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    evs = [e for e in prof.key_averages() if name in e.key]
    total = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in evs)
    count = sum(e.count for e in evs)
    return total / max(count, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    say(f"card: {q.stdout.strip() or 'nvidia-smi unavailable'}  (name, power limit, max SM clock)")
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    n = bench.ENVS_PER_GPU
    H, gc, gv, targets, kp, kd = bench.make_workload(0, n)
    with torch.cuda.stream(stream):
        bt = capi.Batch(capi.Model(os.path.join(RSC_DIR, "anymal_c_like.urdf")), n)
        bt.set_params(**bench.SOLVER)
        bt.set_heightmap(bench.HM["xs"], bench.HM["ys"], bench.HM["size"], bench.HM["size"], 0.0, 0.0, H)
        bt.set_stream(stream.cuda_stream)
        bt.set_state(gc.astype(np.float32), gv.astype(np.float32))
        bt.set_pd_gains(kp, kd)
        g0 = bench.GC0.astype(np.float32)
        bt.gym_configure(g0, np.zeros(18, np.float32), g0[7:], np.full(12, 0.5, np.float32), [bt.model.body_index(f) for f in ("LF_SHANK", "RF_SHANK", "LH_SHANK", "RH_SHANK")])
        act = torch.zeros((n, 12), dtype=torch.float32, device="cuda")
        obs = torch.empty((n, bt.ob_dim()), dtype=torch.float32, device="cuda")
        rew = torch.empty(n, dtype=torch.float32, device="cuda")
        done = torch.empty(n, dtype=torch.uint8, device="cuda")
        for _ in range(bench.SETTLE):
            bt.gym_step(act, bench.SUBSTEPS, obs, rew, done)
        torch.cuda.synchronize()
        base = [bt.model.frame_index("base")]
        feet = [bt.model.frame_index(f) for f in ("LF_FOOT", "RF_FOOT", "LH_FOOT", "RH_FOOT")]
        grid = np.stack(np.meshgrid(0.1 * np.arange(-8, 9), 0.1 * np.arange(-5, 6)), -1).reshape(-1, 2).astype(np.float32)
        ring = np.stack([0.1 * np.cos(np.arange(8) * np.pi / 4), 0.1 * np.sin(np.arange(8) * np.pi / 4)], -1).astype(np.float32)
        el, az = np.meshgrid(np.deg2rad(np.linspace(-45, 5, 16)), np.linspace(-np.pi, np.pi, 32, endpoint=False), indexing="ij")
        lidar_d = np.stack([np.cos(el) * np.cos(az), np.cos(el) * np.sin(az), np.sin(el)], -1).reshape(-1, 3).astype(np.float32)
        lidar_o = np.tile(np.array([[0.0, 0.0, 0.15]], np.float32), (len(lidar_d), 1))
        scan_base = torch.empty((n, len(grid)), dtype=torch.float32, device="cuda")
        scan_feet = torch.empty((n, 4 * len(ring)), dtype=torch.float32, device="cuda")
        hits = torch.empty((n, len(lidar_d), 8), dtype=torch.int32, device="cuda")
        # warm every shape
        for _ in range(5):
            bt.height_scan(base, grid, out=scan_base); bt.height_scan(feet, ring, out=scan_feet)
            bt.ray_test(lidar_o, lidar_d, 10.0, frames=base, out=hits)
            bt.gym_step(act, bench.SUBSTEPS, obs, rew, done)
        torch.cuda.synchronize()
        R = args.reps
        t_base = timed(stream, lambda: bt.height_scan(base, grid, out=scan_base), R)
        t_feet_warm = timed(stream, lambda: bt.height_scan(feet, ring, out=scan_feet), R)

        def feet_after_change():
            bt.gym_reset()                     # marks the state changed: the next foot scan refreshes the poses first
            bt.height_scan(feet, ring, out=scan_feet)
        t_reset = timed(stream, bt.gym_reset, R)
        t_feet_cold = timed(stream, feet_after_change, R) - t_reset
        for _ in range(bench.SETTLE):
            bt.gym_step(act, bench.SUBSTEPS, obs, rew, done)
        t_lidar = timed(stream, lambda: bt.ray_test(lidar_o, lidar_d, 10.0, frames=base, out=hits), R)
        lid = hits.cpu().numpy().view(capi.RAY_HIT_DTYPE).reshape(n, -1)
        frac_hit = float((lid["pair_index"] >= 0).mean())
        t_gym, t_gym_scan = [], []
        for _ in range(5):            # alternate the two arms: the spread of the pairs is the noise of the comparison
            t_gym.append(timed(stream, lambda: bt.gym_step(act, bench.SUBSTEPS, obs, rew, done), R // 2))
            t_gym_scan.append(timed(stream, lambda: (bt.gym_step(act, bench.SUBSTEPS, obs, rew, done), bt.height_scan(base, grid, out=scan_base)), R // 2))
        k_base = kernel_us(lambda: bt.height_scan(base, grid, out=scan_base), "rsb_height_scan_kernel")
        k_feet = kernel_us(lambda: bt.height_scan(feet, ring, out=scan_feet), "rsb_height_scan_kernel")
        k_lidar = kernel_us(lambda: bt.ray_test(lidar_o, lidar_d, 10.0, frames=base, out=hits), "rsb_ray_test_kernel")
        k_kin = kernel_us(feet_after_change, "rsb_step_kernel")
        k_gym = kernel_us(lambda: bt.gym_step(act, bench.SUBSTEPS, obs, rew, done), "rsb_step_kernel")
    samples = n * len(grid)
    say(f"workload: {n} envs, {bench.HM['xs']}^2 height map ({bench.HM['size']} m), settled {bench.SETTLE} gym steps; L2 warm (the 1 MiB map and "
        f"the {n * 32 * 4 / 1e6:.1f} MB of state rows stay in the 126 MB L2 between calls); CUDA events over {R} back-to-back calls "
        "from Python (per call: the kernel and the host submission of the next call, whichever is longer)")
    say(f"base height scan   17 x 11 points           : {1e3 * t_base:8.2f} us  ({samples / 1e6:.2f} M samples)")
    say(f"foot scans         4 frames x 8 points      : {1e3 * t_feet_warm:8.2f} us  unchanged state (scan launch only)")
    say(f"foot scans after a state change             : {1e3 * t_feet_cold:8.2f} us  (kinematics launch + scan; a gym_reset timed alone, {1e3 * t_reset:.2f} us, subtracted)")
    say(f"lidar 16 x 32 rays, 10 m, on the base       : {1e3 * t_lidar:8.2f} us  ({n * len(lidar_d) / t_lidar / 1e6:.2f} G rays/s, {100 * frac_hit:.1f} % of rays hit)")
    g, gs = np.array(t_gym), np.array(t_gym_scan)
    say(f"gym_step alone                              : {1e3 * g.mean():8.2f} us  (5 alternated windows: {', '.join(f'{1e3 * x:.1f}' for x in g)})")
    say(f"gym_step + base scan                        : {1e3 * gs.mean():8.2f} us  (5 alternated windows: {', '.join(f'{1e3 * x:.1f}' for x in gs)})")
    say(f"base scan share of the gym step             : {100 * (gs.mean() - g.mean()) / g.mean():8.2f} %")
    say("kernel times alone (torch.profiler, CUDA activity, mean of 50 launches; the event times above include host submission):")
    say(f"  rsb_height_scan_kernel, base 17 x 11      : {k_base:8.2f} us")
    say(f"  rsb_height_scan_kernel, 4 feet x 8        : {k_feet:8.2f} us")
    say(f"  rsb_ray_test_kernel, lidar 16 x 32        : {k_lidar:8.2f} us")
    say(f"  rsb_step_kernel, kinematics-only launch   : {k_kin:8.2f} us")
    say(f"  rsb_step_kernel, gym step (4 sub-steps)   : {k_gym:8.2f} us")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
