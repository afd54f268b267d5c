"""Environment sharding across GPUs (SURVEY.md 8e): contiguous blocks, one process per GPU, and the
single collective of the path -- the all-gather of the observation rows.  Backend-agnostic
(nccl on the GPU box, gloo in the CPU tests)."""
import torch
import torch.distributed as dist


def shard_range(num_envs_total, world_size, rank):
    """rank r owns [r*N/G, (r+1)*N/G); N must divide evenly (weak scaling keeps N/G fixed)."""
    if num_envs_total % world_size != 0:
        raise ValueError(f"{num_envs_total} environments do not split evenly over {world_size} ranks")
    per = num_envs_total // world_size
    return rank * per, (rank + 1) * per


def shard_seed(config_index, rank):
    """SURVEY 8d: seed = config index x 1000 + rank"""
    return config_index * 1000 + rank


def allgather_observations(obs_local, out=None):
    """obs_local [N/G, obDim] -> [N, obDim] in rank order on every rank (no-op without a process group)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        if out is not None:
            out.copy_(obs_local)
            return out
        return obs_local
    world = dist.get_world_size()
    if out is None:
        out = torch.empty((world * obs_local.shape[0], obs_local.shape[1]), dtype=obs_local.dtype, device=obs_local.device)
    dist.all_gather_into_tensor(out, obs_local.contiguous())
    return out


class ObservationGather:
    """The path's one collective (SURVEY 8e), one process per GPU.

    mode "peer" (default on NVLink boxes): the all-gather is FUSED into the step kernel.  Every rank owns two gathered-rows
    buffers [world * n, ob_dim] (double-buffered by control step) and a row of arrival counters, all plain device memory exported
    through CUDA IPC; `torch.distributed` only ships the 64-byte handles once, at set-up.  During a control step each finished
    observation row is stored straight into every rank's buffer over NVLink while the kernel is still running, and the last CTA
    of the launch stays until every rank's rows of that step have landed: the control step completes when the gathered rows do.
    No NCCL call, no extra launch on the data path.
    mode "nccl": `all_gather_into_tensor` after the step (the baseline this replaces; also what the gloo CPU test drives)."""

    def __init__(self, batch, world, rank, n, ob_dim, mode="peer", device=None):
        self.batch, self.world, self.rank, self.n, self.od, self.mode = batch, world, rank, n, ob_dim, mode
        self.steps = 0
        self._opened, self._own = [], []
        if mode == "peer":
            from . import capi
            import ctypes as C
            L = capi.lib()
            dev = torch.cuda.current_device() if device is None else device
            mine = []                                        # (pointer, handle bytes): two row buffers + the counter row
            for nbytes in (world * n * ob_dim * 4, world * n * ob_dim * 4, 256):
                ptr, h = C.c_void_p(), (C.c_ubyte * 64)()
                capi._ck(L.rsb_peer_buffer_create(dev, nbytes, C.byref(ptr), h))
                mine.append((ptr.value, bytes(h)))
                self._own.append(ptr.value)
            everyone = [None] * world
            dist.all_gather_object(everyone, [h for _, h in mine])
            obs_ptrs, flag_ptrs = [], []
            for r in range(world):
                ptrs = []
                for k in range(3):
                    if r == rank:
                        ptrs.append(mine[k][0])
                    else:
                        q = C.c_void_p()
                        hb = (C.c_ubyte * 64).from_buffer_copy(everyone[r][k])
                        capi._ck(L.rsb_peer_buffer_open(dev, hb, C.byref(q)))
                        self._opened.append(q.value)
                        ptrs.append(q.value)
                obs_ptrs += ptrs[:2]; flag_ptrs.append(ptrs[2])
            batch.set_observation_peers(world, rank, obs_ptrs, flag_ptrs)
            self.rows = [self._view(mine[0][0]), self._view(mine[1][0])]
            dist.barrier()
        else:
            self.rows = None                                 # allocated by the first gather(), where the rows live (gloo: host)

    def _view(self, ptr):
        class _Raw:
            def __init__(s, p, shape):
                s.__cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "data": (int(p), False), "version": 2}
        return torch.as_tensor(_Raw(ptr, (self.world * self.n, self.od)), device="cuda")

    def gather(self, obs_local):
        """call right after the control step that produced obs_local; returns the [world * n, ob_dim] rows of that step (valid
        in stream order on the batch's stream)"""
        self.steps += 1
        if self.mode == "peer":
            return self.rows[self.batch.wait_observation_peers()]
        if self.rows is None:
            self.rows = [torch.empty((self.world * self.n, self.od), dtype=obs_local.dtype, device=obs_local.device) for _ in range(2)]
        out = self.rows[self.steps & 1]
        allgather_observations(obs_local, out)
        return out

    def report(self):
        return {"mode": self.mode, "collective": ("observation rows stored into every rank's buffer by the step kernel over NVLink peer memory (CUDA IPC), "
                                                  "arrival counters, the wait folded into the same launch; no NCCL call and no extra launch on the data path") if self.mode == "peer"
                else "torch.distributed all_gather_into_tensor (NCCL) after the step, on the launching stream",
                "bytes_per_step_per_rank": int(self.n * self.od * 4 * self.world)}

    def close(self):
        if self.mode == "peer":
            from . import capi
            torch.cuda.synchronize()
            dist.barrier()
            self.batch.set_observation_peers(0, 0, None, None)
            self.rows = None
            L = capi.lib()
            for q in self._opened:
                L.rsb_peer_buffer_close(q)
            dist.barrier()
            for q in self._own:
                L.rsb_peer_buffer_destroy(q)
            self._opened, self._own = [], []


class SharedHostRows:
    """A [world * rows_per_rank, width] float32 array in POSIX shared memory that every rank maps and page-locks.

    Host-side consumers (a trainer process on rank 0 reading observation rows) do not need the NVLink all-gather:
    each rank's step kernel writes its own block of rows IN PLACE over its own PCIe link (the C-ABI recognises the
    page-locked buffer and binds it zero-copy), all links in parallel; one barrier later every row is visible to
    every process (`publish_and_wait`, shared-memory flags).  `local` is this rank's block (a numpy view to hand to
    Batch.control_step), `all` the whole array.
    """

    def __init__(self, tag, world, rank, rows_per_rank, width, register=True, barrier=None):
        import os
        import numpy as np
        self.path = f"/dev/shm/rsb_{tag}"
        self.rank, self.registered = rank, False
        shape = (world * rows_per_rank, width)
        row_bytes = shape[0] * shape[1] * 4
        flag_off = (row_bytes + 4095) // 4096 * 4096          # one cache line of flags per rank, behind the rows
        nbytes = flag_off + world * 64
        self.world = world
        barrier = barrier or (dist.barrier if (dist.is_available() and dist.is_initialized()) else (lambda: None))
        if rank == 0:
            with open(self.path, "wb") as f:
                f.truncate(nbytes)
        barrier()
        self.all = np.memmap(self.path, dtype=np.float32, mode="r+", shape=shape)
        self._flags = np.memmap(self.path, dtype=np.int64, mode="r+", offset=flag_off, shape=(world, 8))
        self.local = self.all[rank * rows_per_rank:(rank + 1) * rows_per_rank]
        self._ptr, self._nbytes = self.all.ctypes.data, row_bytes
        if register:
            rc = torch.cuda.cudart().cudaHostRegister(self._ptr, row_bytes, 1 | 2)   # portable | mapped
            if int(rc) != 0:
                raise RuntimeError(f"cudaHostRegister failed with {rc}")
            self.registered = True
        barrier()

    def publish_and_wait(self, step_id, timeout_s=60.0):
        """Host-side barrier for the rows of control step `step_id` (> 0, increasing): call after this rank's step call
        returned (its rows are then in host memory), returns when every rank has published the same step.  Plain
        shared-memory flags (x86 store order: rows before flag) -- no GPU work, no NCCL on the host-bound path."""
        import time
        self._flags[self.rank, 0] = step_id
        f = self._flags[:, 0]
        spins, t0 = 0, None
        while int(f.min()) < step_id:
            spins += 1
            if spins % 4096 == 0:                      # a dead peer must not hang the job
                t0 = t0 or time.monotonic()
                if time.monotonic() - t0 > timeout_s:
                    raise RuntimeError(f"SharedHostRows: rank(s) {[int(r) for r in (f < step_id).nonzero()[0]]} did not publish step {step_id} within {timeout_s} s")

    def close(self, barrier=None):
        import os
        if self.registered:
            torch.cuda.cudart().cudaHostUnregister(self._ptr)
            self.registered = False
        barrier = barrier or (dist.barrier if (dist.is_available() and dist.is_initialized()) else (lambda: None))
        barrier()
        self.local = None
        self.all = None
        self._flags = None
        if self.rank == 0:
            try:
                os.unlink(self.path)
            except OSError:
                pass
