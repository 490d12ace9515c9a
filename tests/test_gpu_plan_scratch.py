"""One batched spectrum plan shared by cross spectra, VDOS, projected VDOS and MSD: the entries take their per-call
tables and partials from the plan's one scratch buffer, interleaved so that it grows and is reused, and every result
is bit-identical to the same call on a fresh plan."""
import ctypes

import numpy as np
import pytest
import torch

from ramannoodle_b200 import _lib

from gpu_helpers import to_cuda

pytestmark = pytest.mark.gpu

FRAMES, BATCH, ATOMS = 600, 4, 24


def _ptr(value):
    return ctypes.c_void_p(value.data_ptr() if isinstance(value, torch.Tensor) else value.ctypes.data)


def _zeros(*shape):
    return torch.zeros(shape, dtype=torch.float64, device="cuda:0")


def _cross(lib, plan, stream, alpha):
    points = int(lib.rn_spectrum_num_points(FRAMES))
    wn, inten = _zeros(points), _zeros(alpha.shape[0], alpha.shape[0], points)
    _lib.check(lib.rn_md_cross_spectra(plan, _ptr(alpha), alpha.shape[0], 1.5, 1, 532.0, 1, 300.0, _ptr(wn),
                                       _ptr(inten), stream), "rn_md_cross_spectra")
    return wn, inten


def _groups(groups):
    offsets = np.cumsum([0] + [len(g) for g in groups]).astype(np.int64)
    return offsets, np.concatenate(groups).astype(np.int64)


def _vdos(lib, plan, stream, positions, lattice, weights, groups):
    points = int(lib.rn_spectrum_num_points(FRAMES))
    offsets, atoms = _groups(groups)
    wn, inten = _zeros(points), _zeros(len(groups), points)
    _lib.check(lib.rn_vdos(plan, _ptr(positions), ATOMS, _ptr(lattice), _ptr(weights), _ptr(offsets), _ptr(atoms),
                           len(groups), 1.5, _ptr(wn), _ptr(inten), stream), "rn_vdos")
    return wn, inten


def _projected(lib, plan, stream, positions, lattice, vectors):
    points = int(lib.rn_spectrum_num_points(FRAMES))
    wn, inten = _zeros(points), _zeros(vectors.shape[0], points)
    _lib.check(lib.rn_projected_vdos(plan, _ptr(positions), ATOMS, _ptr(lattice), _ptr(vectors), vectors.shape[0], 1.5,
                                     _ptr(wn), _ptr(inten), stream), "rn_projected_vdos")
    return wn, inten


def _msd(lib, plan, stream, positions, lattice, groups):
    offsets, atoms = _groups(groups)
    msd = _zeros(len(groups), positions.shape[0])
    _lib.check(lib.rn_msd(plan, _ptr(positions), ATOMS, _ptr(lattice), _ptr(offsets), _ptr(atoms), len(groups),
                          _ptr(msd), stream), "rn_msd")
    return (msd,)


def test_shared_plan_matches_fresh_plans():
    lib = _lib.lib()
    rng = np.random.default_rng(31)
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.array([[9.0, 0.5, 0.0], [0.0, 8.0, 1.0], [0.7, 0.0, 10.0]])
    positions = to_cuda(rng.uniform(0, 1, (FRAMES, ATOMS, 3)))
    # the MSD of S - 1 frames runs on a plan of S frames (M = S - 1, a linear autocorrelation of S - 1 values)
    msd_positions = to_cuda(rng.uniform(0, 1, (FRAMES - 1, ATOMS, 3)))
    alpha = to_cuda(6.0 * np.eye(3) + 0.05 * rng.normal(size=(BATCH, FRAMES, 3, 3)))
    weights = rng.uniform(1.0, 50.0, ATOMS)
    all_atoms, per_atom = [np.arange(ATOMS)], [np.array([i]) for i in range(ATOMS)]
    # scratch requests in bytes, growing and shrinking from call to call
    calls = [
        (_cross, (alpha[:2],)),
        (_vdos, (positions, lattice, weights, all_atoms)),
        (_msd, (msd_positions, lattice, all_atoms)),
        (_cross, (alpha,)),
        (_projected, (positions, lattice, rng.normal(size=(5, ATOMS, 3)))),
        (_vdos, (positions, lattice, weights, per_atom)),
        (_msd, (msd_positions, lattice, per_atom)),
        (_cross, (alpha[:3],)),
        (_projected, (positions, lattice, rng.normal(size=(30, ATOMS, 3)))),
        (_vdos, (positions, lattice, weights, [np.arange(0, ATOMS, 2), np.arange(5, 18)])),
    ]
    shared = ctypes.c_void_p()
    _lib.check(lib.rn_spectrum_plan_create_batched(FRAMES, BATCH, 0, ctypes.byref(shared)), "create_batched")
    try:
        for entry, args in calls:
            got = [t.cpu().numpy() for t in entry(lib, shared, stream, *args)]
            fresh = ctypes.c_void_p()
            _lib.check(lib.rn_spectrum_plan_create_batched(FRAMES, BATCH, 0, ctypes.byref(fresh)), "create_batched")
            try:
                want = [t.cpu().numpy() for t in entry(lib, fresh, stream, *args)]
            finally:
                torch.cuda.synchronize()
                lib.rn_spectrum_plan_destroy(fresh)
            for g, w in zip(got, want):
                assert np.all(np.isfinite(g))
                assert np.array_equal(g, w), entry.__name__
    finally:
        torch.cuda.synchronize()
        lib.rn_spectrum_plan_destroy(shared)
