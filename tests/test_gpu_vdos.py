"""Vibrational density of states (``Trajectory.get_vdos``) on the GPU: the oracle at ``INTENSITY_RTOL`` pointwise over
lengths around the plan shapes, structures, group layouts, weights, triclinic lattices, lattice hops and timesteps;
the wavenumbers of ``measure``; bit-identity across input forms, repeated calls, batch sizes and scaled weights; the
real LLZO OUTCAR trajectory; species partials at scale; the launch count and the C entry's errors."""
import ctypes
import gzip
import os
import shutil

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, spectrum, synthetic
from ramannoodle_b200 import io as rio

from gpu_helpers import INTENSITY_RTOL, to_cuda
from helpers import GOLDEN, pointwise_rel_err
from vdos_oracle import vdos

pytestmark = pytest.mark.gpu


def _geometry(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    """The lattice with off-diagonal entries of 1-3 Å: every entry of the lattice product is used."""
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def _groups(kind, num_atoms, numbers):
    if kind == "all":
        return None, [range(num_atoms)]
    if kind == "species":
        groups = [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
    elif kind == "odd_even_overlap":  # sizes 7, 10, 1 and an overlap of the first two
        groups = [list(range(0, 7)), list(range(3, 13)), [num_atoms - 1], list(range(num_atoms - 1, 20, -9))]
    elif kind == "per_atom":
        groups = [[i] for i in range(num_atoms)]
    else:
        raise AssertionError(kind)
    return groups, groups


def _check(positions, lattice, timestep, kind="all", weights=None, structure="TiO2"):
    _, num_atoms, numbers = _geometry(structure)
    groups, oracle_groups = _groups(kind, num_atoms, numbers)
    trajectory = rb.Trajectory(positions, timestep)
    wn, rows = trajectory.get_vdos(lattice, groups, weights)
    want_wn, want = vdos(positions, lattice, timestep, oracle_groups,
                         np.ones(num_atoms) if weights is None else weights)
    assert np.array_equal(wn, want_wn)
    assert rows.shape == want.shape
    assert pointwise_rel_err(rows, want) <= INTENSITY_RTOL
    return wn, rows


@pytest.mark.parametrize("frames", [100, 2049, 2050, 40_001])
def test_lengths_around_plan_shapes(frames):
    """No strided level (L = 4096 up to 2049 frames), the first one-level length and a mid one-level size."""
    lattice, _, _ = _geometry("TiO2")
    _check(synthetic.make_trajectory("TiO2", frames, seed=frames), lattice, 1.0, "odd_even_overlap")


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("kind", ["all", "species", "odd_even_overlap", "per_atom"])
def test_structures_and_groups(structure, kind):
    lattice, num_atoms, _ = _geometry(structure)
    weights = np.random.default_rng(num_atoms).uniform(0.5, 200.0, num_atoms)
    _check(synthetic.make_trajectory(structure, 1501, seed=21), lattice, 1.0, kind, weights, structure)


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("timestep", [0.5, 2.0])
def test_triclinic_lattice_hops_and_timesteps(structure, timestep):
    lattice, num_atoms, _ = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 1201, timestep=timestep, seed=22, lattice_hops=True)
    weights = np.random.default_rng(5).uniform(1.0, 100.0, num_atoms)
    _check(positions, lattice, timestep, "species", weights, structure)
    _check(positions, _sheared(lattice), timestep, "odd_even_overlap", weights, structure)


@pytest.mark.parametrize("frames", [4, 5, 1000, 2050])
@pytest.mark.parametrize("timestep", [0.5, 1.0, 2.0])
def test_wavenumbers_are_those_of_measure(frames, timestep):
    lattice, _, _ = _geometry("TiO2")
    wn, rows = rb.Trajectory(synthetic.make_trajectory("TiO2", frames, seed=3), timestep).get_vdos(lattice)
    want, _ = rb.MDRamanSpectrum(np.zeros((frames, 3, 3)) + np.arange(frames)[:, None, None], timestep).measure()
    assert np.array_equal(wn, want) and rows.shape == (1, len(want))


@pytest.mark.parametrize("frames", [2, 3])
def test_too_short_for_a_point_is_empty(frames):
    lattice, _, _ = _geometry("TiO2")
    trajectory = rb.Trajectory(synthetic.make_trajectory("TiO2", frames, seed=3), 1.0)
    wn, rows = trajectory.get_vdos(lattice, [[0], [1, 2]])
    assert wn.shape == (0,) and rows.shape == (2, 0)


def _equal(a, b):
    return torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_host_device_and_repeated_calls_are_bit_identical():
    lattice, num_atoms, numbers = _geometry("LLZO")
    positions = synthetic.make_trajectory("LLZO", 3001, seed=23)
    groups = [np.flatnonzero(numbers == z) for z in np.unique(numbers)] + [range(num_atoms)]
    weights = np.random.default_rng(6).uniform(1.0, 140.0, num_atoms)
    host = rb.Trajectory(positions, 1.0)
    device = rb.Trajectory(to_cuda(positions), 1.0)
    assert not host.is_device_resident and device.is_device_resident
    assert np.array_equal(host.positions_ts, device.positions_ts)
    first = host.get_vdos_device(lattice, groups, weights)
    assert _equal(first, device.get_vdos_device(lattice, groups, weights))
    assert _equal(first, host.get_vdos_device(lattice, groups, weights))
    assert _equal(first, device.get_vdos_device(lattice, groups, weights))


@pytest.mark.parametrize("slots_per_chunk", [1, 2, 3, 7])
def test_batch_size_does_not_change_a_bit(slots_per_chunk, monkeypatch):
    """Groups of 3, 9, 1, 5 and all 135 atoms (2, 5, 1, 3 and 68 slots) span chunks of every size."""
    lattice, num_atoms, _ = _geometry("STO")
    positions = to_cuda(synthetic.make_trajectory("STO", 2001, seed=24))
    groups = [range(0, 3), range(10, 19), [50], range(60, 65), range(num_atoms)]
    weights = np.random.default_rng(7).uniform(1.0, 90.0, num_atoms)
    trajectory = rb.Trajectory(positions, 1.0)
    default = trajectory.get_vdos_device(_sheared(lattice), groups, weights)
    assert spectrum._window_batch(2001, 79) == 128  # pylint: disable=protected-access  (one chunk)
    per_slot = 16 * 3 * 4096 + 8 * 3 * 2000 + 8 * ((2000 + 255) // 256 + 1) + 4  # a window of 2001 frames
    monkeypatch.setattr(spectrum, "_WINDOW_BATCH_BYTES", slots_per_chunk * per_slot)
    assert spectrum._window_batch(2001, 79) == slots_per_chunk  # pylint: disable=protected-access
    assert _equal(default, trajectory.get_vdos_device(_sheared(lattice), groups, weights))


def test_scaled_weights_scale_the_rows_exactly():
    lattice, num_atoms, numbers = _geometry("TiO2")
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("TiO2", 2500, seed=25)), 0.5)
    groups = [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
    weights = np.random.default_rng(8).uniform(1.0, 50.0, num_atoms)
    wn, rows = trajectory.get_vdos_device(lattice, groups, weights)
    wn4, rows4 = trajectory.get_vdos_device(lattice, groups, 4 * weights)
    assert torch.equal(wn, wn4) and torch.equal(rows4, 4 * rows)


def test_real_llzo_outcar_trajectory(tmp_path):
    path = tmp_path / "OUTCAR_trajectory"
    with gzip.open(os.path.join(GOLDEN, "llzo_outcar_trajectory.txt.gz"), "rb") as fin, open(path, "wb") as fout:
        shutil.copyfileobj(fin, fout)
    _, lattice, _ = rio.read_outcar_positions_ts(path)
    with np.load(os.path.join(GOLDEN, "llzo_outcar_trajectory.npz")) as data:
        positions, timestep = data["positions_ts"], float(data["timestep"])
    assert positions.shape == (15, 108, 3)
    num_atoms = positions.shape[1]
    groups = [range(0, 40), range(40, 41), range(41, num_atoms)]
    trajectory = rb.Trajectory(positions, timestep)
    wn, rows = trajectory.get_vdos(lattice, groups)
    want_wn, want = vdos(positions, lattice, timestep, groups, np.ones(num_atoms))
    assert np.array_equal(wn, want_wn) and rows.shape == (3, 6)
    assert pointwise_rel_err(rows, want) <= INTENSITY_RTOL
    _, total = trajectory.get_vdos(lattice)
    assert pointwise_rel_err(rows.sum(axis=0), total[0]) <= 1e-12


def test_species_partials_at_scale():
    lattice, num_atoms, numbers = _geometry("LLZO")
    assert sorted(set(numbers.tolist())) == [3, 8, 40, 57]
    masses = {3: 6.94, 8: 15.999, 40: 91.224, 57: 138.905}
    weights = np.array([masses[int(z)] for z in numbers])
    groups = [np.flatnonzero(numbers == z) for z in (3, 8, 40, 57)]
    positions = synthetic.make_trajectory("LLZO", 20_001, seed=26)
    trajectory = rb.Trajectory(to_cuda(positions), 1.0)
    wn, rows = trajectory.get_vdos(lattice, groups, weights)
    want_wn, want = vdos(positions, lattice, 1.0, groups, weights)
    assert np.array_equal(wn, want_wn)
    assert pointwise_rel_err(rows, want) <= INTENSITY_RTOL
    _, total = trajectory.get_vdos(lattice, None, weights)
    assert pointwise_rel_err(rows.sum(axis=0), total[0]) <= 1e-12


def _launches(fn):
    fn()  # plans are created (and cached) here
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def test_launch_count(monkeypatch):
    """One pack, the transform passes and one combine per chunk: a single measure's launches, whatever N."""
    frames = 20_001
    single = rb.MDRamanSpectrum(to_cuda(np.random.default_rng(9).normal(size=(frames, 3, 3))), 1.0)
    per_chunk = _launches(single.measure_device)
    counts = []
    for structure in ("TiO2", "LLZO"):
        lattice, _, numbers = _geometry(structure)
        trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory(structure, frames, seed=27)), 1.0)
        species = [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
        counts.append(_launches(lambda t=trajectory, l=lattice: t.get_vdos_device(l)))
        counts.append(_launches(lambda t=trajectory, l=lattice, g=species: t.get_vdos_device(l, g)))
    assert counts == [per_chunk] * 4
    lattice, num_atoms, _ = _geometry("TiO2")  # 54 slots in chunks of 8: 7 chunks
    assert num_atoms == 108
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("TiO2", frames, seed=27)), 1.0)
    per_slot = 16 * 3 * 65536 + 8 * 3 * (frames - 1) + 8 * ((frames - 1 + 255) // 256 + 1) + 4
    monkeypatch.setattr(spectrum, "_WINDOW_BATCH_BYTES", 8 * per_slot)
    assert spectrum._window_batch(frames, 54) == 8  # pylint: disable=protected-access
    assert _launches(lambda: trajectory.get_vdos_device(lattice)) == 7 * per_chunk


def test_c_entry_errors():
    frames, num_atoms = 300, 6
    lib = _lib.lib()
    rng = np.random.default_rng(10)
    positions = to_cuda(rng.uniform(0, 1, (frames, num_atoms, 3)))
    points = int(lib.rn_spectrum_num_points(frames))
    wn = torch.empty(points, dtype=torch.float64, device="cuda:0")
    inten = torch.empty((2, points), dtype=torch.float64, device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.diag([5.0, 6.0, 7.0])
    weights = np.ones(num_atoms)
    offsets = np.array([0, 2, 5], dtype=np.int64)
    atoms = np.array([0, 1, 2, 3, 5], dtype=np.int64)
    handle, dist = ctypes.c_void_p(), ctypes.c_void_p()
    _lib.check(lib.rn_spectrum_plan_create_batched(frames, 2, 0, ctypes.byref(handle)), "create_batched")
    _lib.check(lib.rn_spectrum_plan_create_dist(frames, 0, 2, 0, ctypes.byref(dist)), "create_dist")
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731

    def call(plan=handle, pos=ctypes.c_void_p(positions.data_ptr()), n=num_atoms, lat=ptr(lattice), w=ptr(weights),
             off=ptr(offsets), at=ptr(atoms), groups=2, dt=1.0, wn_ptr=ctypes.c_void_p(wn.data_ptr()),
             int_ptr=ctypes.c_void_p(inten.data_ptr())):
        return lib.rn_vdos(plan, pos, n, lat, w, off, at, groups, dt, wn_ptr, int_ptr, stream)

    try:
        assert call(plan=None) == -1
        assert call(plan=dist) == -1  # a multi-GPU plan
        assert call(pos=None) == -1
        assert call(lat=None) == -1
        assert call(off=None) == -1
        assert call(at=None) == -1
        assert call(wn_ptr=None) == -1
        assert call(int_ptr=None) == -1
        assert call(groups=0) == -1
        assert call(dt=0.0) == -1
        assert call(dt=-1.0) == -1
        bad_atoms = atoms.copy()
        bad_atoms[4] = num_atoms
        assert call(at=ptr(bad_atoms)) == -1
        bad_atoms[4] = -1
        assert call(at=ptr(bad_atoms)) == -1
        assert call(off=ptr(np.array([0, 2, 2], dtype=np.int64))) == -1  # empty group
        for value in (-1.0, np.nan, np.inf):
            bad_weights = weights.copy()
            bad_weights[3] = value
            assert call(w=ptr(bad_weights)) == -1
        assert call(w=None) == 0  # all ones
        torch.cuda.synchronize()
        trajectory = rb.Trajectory(positions, 1.0)
        want_wn, want = trajectory.get_vdos(lattice, [[0, 1], [2, 3, 5]])
        assert np.array_equal(wn.cpu().numpy(), want_wn) and np.array_equal(inten.cpu().numpy(), want)
    finally:
        torch.cuda.synchronize()
        lib.rn_spectrum_plan_destroy(handle)
        lib.rn_spectrum_plan_destroy(dist)
