"""Read-back entry points of the C-ABI (rsb_batch_get_*) into host and device memory, and height-map replacement.

Every getter is called through capi.lib() twice, into numpy (RSB_HOST) and into CUDA torch buffers (RSB_DEVICE), for the full
range and for an interior one, after a step on a rough height map with contacts: the bytes must be equal.  Installing a single
height map over a terrain atlas must leave the batch exactly as if it had only ever had that map.
"""
import ctypes as C
import os
import numpy as np
import pytest

from conftest import RSC
from helpers import ANYMAL_GC0

ANYMAL = os.path.join(RSC, "anymal_c_like.urdf")
N = 48
INTERIOR = (5, 17)        # env_begin, env_count


@pytest.fixture(scope="module")
def capi():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from raisimlib_b200 import capi as c
    return c


def _rough(rng, xs=65, ys=65, amp=0.08):
    """smooth random heights [ys, xs]: white noise averaged over 5 x 5 cells"""
    w = rng.uniform(-1, 1, (ys + 4, xs + 4))
    H = sum(w[j:j + ys, i:i + xs] for j in range(5) for i in range(5))
    return (amp * H / np.abs(H).max()).astype(np.float32)


def _state(rng, n):
    gc = np.tile(ANYMAL_GC0, (n, 1))
    gc[:, 0:2] = rng.uniform(-2.0, 2.0, (n, 2))
    gc[:, 2] = 0.54
    gc[:, 7:] += rng.uniform(-0.1, 0.1, (n, 12))
    return gc.astype(np.float32), (0.1 * rng.standard_normal((n, 18))).astype(np.float32)


def _stepped_batch(capi, set_terrain, gc, gv, substeps):
    bt = capi.Batch(capi.Model(ANYMAL), len(gc))
    set_terrain(bt)
    bt.set_pd_gains(np.r_[np.zeros(6), 80.0 * np.ones(12)], np.r_[np.zeros(6), 2.0 * np.ones(12)])
    bt.set_pd_target(np.tile(ANYMAL_GC0, (len(gc), 1)).astype(np.float32), np.zeros((len(gc), 18), np.float32))
    bt.set_state(gc, gv)
    bt.integrate(substeps)
    return bt


def _getters(capi, bt):
    """(C getter, [(per-environment shape, dtype) of each output], whether the range comes before the outputs)"""
    f4, i4 = np.float32, np.int32
    return [
        ("rsb_batch_get_state", [((bt.nq,), f4), ((bt.nv,), f4)], False),
        ("rsb_batch_get_generalized_force", [((bt.nv,), f4)], False),
        ("rsb_batch_get_mass_matrix", [((bt.nv, bt.nv), f4)], True),
        ("rsb_batch_get_nonlinearities", [((bt.nv,), f4)], True),
        ("rsb_batch_get_body_poses", [((bt.nb, 3, 3), f4), ((bt.nb, 3), f4)], True),
        ("rsb_batch_get_contacts", [((capi.KMAX,), capi.CONTACT_DTYPE), ((), i4)], False),
        ("rsb_batch_get_contact_points", [((capi.KMAX,), i4)], False),
        ("rsb_batch_get_solver_iterations", [((), i4)], False),
        ("rsb_batch_get_solver_status", [((), i4)], False),
        ("rsb_batch_get_solver_residual", [((), f4)], False),
        ("rsb_batch_get_diverged", [((), i4)], False),
    ]


def _read(capi, bt, name, outs, range_first, begin, count, where):
    """raw bytes of every output of one getter call; the buffers start out filled with a pattern that differs per memory kind"""
    import torch
    nbytes = [count * np.dtype(dt).itemsize * int(np.prod(shape)) for shape, dt in outs]
    if where == capi.HOST:
        bufs = [np.full(k, 0xAB, np.uint8) for k in nbytes]
        ptrs = [b.ctypes.data_as(C.c_void_p) for b in bufs]
    else:
        bufs = [torch.full((k,), 0xCD, dtype=torch.uint8, device="cuda") for k in nbytes]
        torch.cuda.synchronize()
        ptrs = [C.c_void_p(b.data_ptr()) for b in bufs]
    args = [begin, count, *ptrs] if range_first else [*ptrs, begin, count]
    assert getattr(capi.lib(), name)(bt.h, *args, where) == 0, capi.lib().rsb_last_error().decode()
    if where == capi.DEVICE:
        bt.sync()                                # the copies are ordered on the batch's stream
        bufs = [b.cpu().numpy() for b in bufs]
    return [b.tobytes() for b in bufs]


@pytest.mark.gpu
def test_every_getter_reads_the_same_bytes_into_host_and_device_memory(capi):
    rng = np.random.default_rng(3)
    gc, gv = _state(rng, N)
    H = _rough(rng)
    bt = _stepped_batch(capi, lambda b: b.set_heightmap(65, 65, 6.4, 6.4, 0.0, 0.0, H), gc, gv, substeps=2)
    _, cnt = bt.contacts()
    assert cnt[INTERIOR[0]:sum(INTERIOR)].sum() > 0, "the state must put feet into the height map"
    for name, outs, range_first in _getters(capi, bt):
        full = _read(capi, bt, name, outs, range_first, 0, N, capi.HOST)
        assert _read(capi, bt, name, outs, range_first, 0, N, capi.DEVICE) == full, name
        begin, count = INTERIOR
        part = _read(capi, bt, name, outs, range_first, begin, count, capi.HOST)
        assert _read(capi, bt, name, outs, range_first, begin, count, capi.DEVICE) == part, name
        for (shape, dt), whole, piece in zip(outs, full, part):   # the interior range is the same rows of the full read
            row = np.dtype(dt).itemsize * int(np.prod(shape))
            assert whole[begin * row:(begin + count) * row] == piece, name


@pytest.mark.gpu
def test_single_heightmap_over_an_atlas_equals_a_batch_that_only_had_it(capi):
    rng = np.random.default_rng(4)
    gc, gv = _state(rng, N)
    H = _rough(rng)
    atlas = np.stack([_rough(rng), _rough(rng)])
    map_of_env = rng.integers(0, 2, N).astype(np.int32)

    def atlas_then_single(b):
        b.set_heightmaps(6.4, 6.4, 0.0, 0.0, atlas, map_of_env)
        b.set_heightmap(65, 65, 6.4, 6.4, 0.0, 0.0, H)

    plain = _stepped_batch(capi, lambda b: b.set_heightmap(65, 65, 6.4, 6.4, 0.0, 0.0, H), gc, gv, substeps=1)
    swapped = _stepped_batch(capi, atlas_then_single, gc, gv, substeps=1)
    (ca, na), (cb, nb) = plain.contacts(), swapped.contacts()
    assert na.sum() > 0
    assert np.array_equal(na, nb) and ca.tobytes() == cb.tobytes()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(plain.get_state(), swapped.get_state()))
    frames = [plain.model.frame_index(f) for f in ("base", "LF_FOOT")]
    pts = np.stack(np.meshgrid(0.2 * np.arange(-3, 4), 0.2 * np.arange(-2, 3)), -1).reshape(-1, 2).astype(np.float32)
    assert plain.height_scan(frames, pts).tobytes() == swapped.height_scan(frames, pts).tobytes()
