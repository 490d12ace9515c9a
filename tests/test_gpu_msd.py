"""Mean squared displacement (``Trajectory.get_msd``) on the GPU: the oracle at |got - want| <= 1e-10 scale_g(m),
scale_g(m) = 2 E_g / ((S - m) |g|), over lengths around the plan shapes, structures, group layouts, sheared lattices,
lattice hops, timesteps and a diffusing species; exact lag 0 and lag times; bit-identity across input forms, repeated
calls, batch sizes and group sets; the real LLZO OUTCAR trajectory; the launch count and the C entry's errors."""
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

from gpu_helpers import to_cuda
from helpers import GOLDEN
from msd_oracle import error_ratio, msd_direct, msd_fft
from oracle import numpy_port as ora

pytestmark = pytest.mark.gpu

MSD_RTOL = 1e-10  # of scale_g(m), the size of an FFT correlation's rounding error


def _geometry(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    """The lattice with off-diagonal entries of 1-3 Å: every entry of the lattice product is used."""
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def _diffusing(structure, frames, seed, species_z, step=0.3):
    """A synthetic trajectory with a random walk (Å per frame and component) added to one species before wrapping, so
    that its paths span many cells."""
    lattice, _, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, frames, seed=seed)
    walk = np.cumsum(np.random.default_rng(seed).normal(scale=step, size=positions.shape), axis=0)
    walk[:, numbers != species_z] = 0.0
    moved = positions + walk @ np.linalg.inv(lattice)
    return moved - np.floor(moved)


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


def _check(positions, lattice, timestep, kind="all", structure="TiO2"):
    _, num_atoms, numbers = _geometry(structure)
    groups, oracle_groups = _groups(kind, num_atoms, numbers)
    lags, rows = rb.Trajectory(positions, timestep).get_msd(lattice, groups)
    oracle = msd_direct if positions.shape[0] <= 200 else msd_fft
    want_lags, want = oracle(positions, lattice, timestep, oracle_groups)
    assert np.array_equal(lags, want_lags) and np.array_equal(lags, np.arange(positions.shape[0]) * timestep)
    assert rows.shape == want.shape
    assert np.all(rows[:, 0] == 0.0)
    assert error_ratio(rows, want, positions, lattice, oracle_groups) <= MSD_RTOL
    return lags, rows


@pytest.mark.parametrize("frames", [100, 2048, 2049, 40_000])
def test_lengths_around_plan_shapes(frames):
    """A plan of S + 1 frames: L = 4096 up to 2048 frames, one strided level from 2049, a mid one-level size."""
    lattice, _, _ = _geometry("TiO2")
    _check(synthetic.make_trajectory("TiO2", frames, seed=frames), lattice, 1.0, "odd_even_overlap")


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("kind", ["all", "species", "odd_even_overlap", "per_atom"])
def test_structures_and_groups(structure, kind):
    lattice, _, _ = _geometry(structure)
    _check(synthetic.make_trajectory(structure, 1501, seed=21), lattice, 1.0, kind, structure)


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("timestep", [0.5, 2.0])
def test_sheared_lattice_hops_and_timesteps(structure, timestep):
    lattice, _, _ = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 1201, timestep=timestep, seed=22, lattice_hops=True)
    _check(positions, lattice, timestep, "species", structure)
    _check(positions, _sheared(lattice), timestep, "odd_even_overlap", structure)


@pytest.mark.parametrize("structure, species", [("LLZO", 3), ("TiO2", 8)])
def test_diffusing_species(structure, species):
    """The walkers cross many cells; MSD(1), where the two large terms cancel most, against the mean squared step."""
    lattice, _, numbers = _geometry(structure)
    positions = _diffusing(structure, 20_000, 31, species)
    _, rows = _check(positions, _sheared(lattice), 1.0, "species", structure)
    walkers = list(np.unique(numbers)).index(species)
    d = ora.apply_pbc_displacement(np.diff(ora.apply_pbc(positions), axis=0))[:, numbers == species]
    want = np.mean(np.sum((d @ _sheared(lattice)) ** 2, axis=2))
    assert abs(rows[walkers, 1] - want) <= 1e-8 * want
    assert rows[walkers, -1] > 100.0  # the walkers left their cells far behind


def test_host_device_and_repeated_calls_are_bit_identical():
    lattice, num_atoms, numbers = _geometry("LLZO")
    positions = _diffusing("LLZO", 3001, 23, 3)
    groups = [np.flatnonzero(numbers == z) for z in np.unique(numbers)] + [range(num_atoms)]
    host = rb.Trajectory(positions, 1.0)
    device = rb.Trajectory(to_cuda(positions), 1.0)
    assert not host.is_device_resident and device.is_device_resident
    first = host.get_msd_device(lattice, groups)
    for again in (device.get_msd_device(lattice, groups), host.get_msd_device(lattice, groups),
                  device.get_msd_device(lattice, groups)):
        assert torch.equal(first[0], again[0]) and torch.equal(first[1], again[1])


@pytest.mark.parametrize("slots_per_chunk", [1, 2, 3, 7])
def test_batch_size_and_group_sets_do_not_change_a_bit(slots_per_chunk, monkeypatch):
    """Groups of 3, 9, 1, 5 and all 135 atoms (2, 5, 1, 3 and 68 slots) span chunks of every size; each group computed
    alone gives its row of the set."""
    lattice, num_atoms, _ = _geometry("STO")
    trajectory = rb.Trajectory(to_cuda(_diffusing("STO", 2000, 24, 8)), 1.0)
    groups = [range(0, 3), range(10, 19), [50], range(60, 65), range(num_atoms)]
    _, default = trajectory.get_msd_device(_sheared(lattice), groups)
    assert spectrum._window_batch(2001, 79) == 128  # pylint: disable=protected-access  (one chunk)
    per_slot = 16 * 3 * 4096 + 8 * 3 * 2000 + 8 * ((2000 + 255) // 256 + 1) + 4  # a plan of 2001 frames
    monkeypatch.setattr(spectrum, "_WINDOW_BATCH_BYTES", slots_per_chunk * per_slot)
    assert spectrum._window_batch(2001, 79) == slots_per_chunk  # pylint: disable=protected-access
    assert torch.equal(default, trajectory.get_msd_device(_sheared(lattice), groups)[1])
    for g, group in enumerate(groups):
        assert torch.equal(default[g], trajectory.get_msd_device(_sheared(lattice), [group])[1][0])


def test_shortest_trajectories():
    lattice, _, _ = _geometry("TiO2")
    for frames in (2, 3, 257):
        _check(synthetic.make_trajectory("TiO2", frames, seed=3, lattice_hops=True), lattice, 2.0, "odd_even_overlap")


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
    lags, rows = rb.Trajectory(positions, timestep).get_msd(lattice, groups)
    want_lags, want = msd_direct(positions, lattice, timestep, groups)
    assert np.array_equal(lags, want_lags) and rows.shape == (3, 15)
    assert error_ratio(rows, want, positions, lattice, groups) <= MSD_RTOL


def _launches(fn):
    fn()  # plans are created (and cached) here
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def test_launch_count(monkeypatch):
    """Per chunk the launches of one measure on S + 1 frames plus the count pass, whatever N; one finish per call."""
    frames = 20_000
    single = rb.MDRamanSpectrum(to_cuda(np.random.default_rng(9).normal(size=(frames + 1, 3, 3))), 1.0)
    per_chunk = _launches(single.measure_device) + 1
    counts = []
    for structure in ("TiO2", "LLZO"):
        lattice, _, numbers = _geometry(structure)
        trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory(structure, frames, seed=27)), 1.0)
        species = [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
        counts.append(_launches(lambda t=trajectory, l=lattice: t.get_msd_device(l)))
        counts.append(_launches(lambda t=trajectory, l=lattice, g=species: t.get_msd_device(l, g)))
    assert counts == [per_chunk + 1] * 4
    lattice, num_atoms, _ = _geometry("TiO2")  # 54 slots in chunks of 8: 7 chunks
    assert num_atoms == 108
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("TiO2", frames, seed=27)), 1.0)
    per_slot = 16 * 3 * 65536 + 8 * 3 * frames + 8 * ((frames + 255) // 256 + 1) + 4
    monkeypatch.setattr(spectrum, "_WINDOW_BATCH_BYTES", 8 * per_slot)
    assert spectrum._window_batch(frames + 1, 54) == 8  # pylint: disable=protected-access
    assert _launches(lambda: trajectory.get_msd_device(lattice)) == 7 * per_chunk + 1


def test_c_entry_errors():
    frames, num_atoms = 300, 6
    lib = _lib.lib()
    rng = np.random.default_rng(10)
    positions = to_cuda(rng.uniform(0, 1, (frames, num_atoms, 3)))
    msd = torch.empty((2, frames), dtype=torch.float64, device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.diag([5.0, 6.0, 7.0])
    offsets = np.array([0, 2, 5], dtype=np.int64)
    atoms = np.array([0, 1, 2, 3, 5], dtype=np.int64)
    handle, dist = ctypes.c_void_p(), ctypes.c_void_p()
    _lib.check(lib.rn_spectrum_plan_create_batched(frames + 1, 2, 0, ctypes.byref(handle)), "create_batched")
    _lib.check(lib.rn_spectrum_plan_create_dist(frames + 1, 0, 2, 0, ctypes.byref(dist)), "create_dist")
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731

    def call(plan=handle, pos=ctypes.c_void_p(positions.data_ptr()), n=num_atoms, lat=ptr(lattice), off=ptr(offsets),
             at=ptr(atoms), groups=2, out=ctypes.c_void_p(msd.data_ptr())):
        return lib.rn_msd(plan, pos, n, lat, off, at, groups, out, stream)

    try:
        assert call(plan=None) == -1
        assert call(plan=dist) == -1  # a multi-GPU plan
        assert call(pos=None) == -1
        assert call(lat=None) == -1
        assert call(off=None) == -1
        assert call(at=None) == -1
        assert call(out=None) == -1
        assert call(groups=0) == -1
        assert call(groups=-1) == -1
        assert call(n=0) == -1
        assert call(lat=ptr(np.diag([5.0, np.nan, 7.0]))) == -1
        bad_atoms = atoms.copy()
        bad_atoms[4] = num_atoms
        assert call(at=ptr(bad_atoms)) == -1
        bad_atoms[4] = -1
        assert call(at=ptr(bad_atoms)) == -1
        assert call(off=ptr(np.array([0, 2, 2], dtype=np.int64))) == -1  # empty group
        assert call() == 0
        torch.cuda.synchronize()
        _, want = rb.Trajectory(positions, 1.0).get_msd(lattice, [[0, 1], [2, 3, 5]])
        assert np.array_equal(msd.cpu().numpy(), want)
    finally:
        torch.cuda.synchronize()
        lib.rn_spectrum_plan_destroy(handle)
        lib.rn_spectrum_plan_destroy(dist)
