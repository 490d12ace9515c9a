"""Projected VDOS (``Trajectory.get_projected_vdos``) on the GPU: the oracle at ``INTENSITY_RTOL`` pointwise over
lengths around the plan shapes, structures, vector counts, triclinic lattices, lattice hops and timesteps; the
wavenumbers of ``measure`` and ``get_vdos``; exactly zero rows of zero vectors; the sum rule and the identity basis
against ``get_vdos`` at scale and on the real LLZO OUTCAR trajectory; peaks of phonon and synthetic modes;
bit-identity across input forms, repeated calls and batch sizes; the launch count and the C entry's errors."""
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
from projected_vdos_oracle import projected_vdos
from test_projected_vdos_args import MASSES, orthonormal_mass_weighted

pytestmark = pytest.mark.gpu

CM_PER_FS = 33.35640951981521 * 1e3  # wavenumber (cm^-1) of one cycle per fs


def _geometry(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    """The lattice with off-diagonal entries of 1-3 Å: every entry of the lattice product is used."""
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def _vectors(num_vectors, num_atoms, seed):
    return np.random.default_rng(seed).normal(size=(num_vectors, num_atoms, 3))


def _check(positions, lattice, timestep, vectors):
    wn, rows = rb.Trajectory(positions, timestep).get_projected_vdos(lattice, vectors)
    want_wn, want = projected_vdos(positions, lattice, timestep, vectors)
    assert np.array_equal(wn, want_wn)
    assert rows.shape == want.shape
    assert pointwise_rel_err(rows, want) <= INTENSITY_RTOL
    return wn, rows


@pytest.mark.parametrize("frames", [100, 2049, 2050, 40_001])
def test_lengths_around_plan_shapes(frames):
    """No strided level (L = 4096 up to 2049 frames), the first one-level length and a mid one-level size."""
    lattice, num_atoms, _ = _geometry("TiO2")
    _check(synthetic.make_trajectory("TiO2", frames, seed=frames), lattice, 1.0, _vectors(7, num_atoms, frames))


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("num_vectors", [1, 2, 5, 6, 7, "3N"])
def test_structures_and_vector_counts(structure, num_vectors):
    lattice, num_atoms, _ = _geometry(structure)
    count = 3 * num_atoms if num_vectors == "3N" else num_vectors
    _check(synthetic.make_trajectory(structure, 1501, seed=31), lattice, 1.0, _vectors(count, num_atoms, count))


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("timestep", [0.5, 2.0])
def test_triclinic_lattice_hops_and_timesteps(structure, timestep):
    lattice, num_atoms, _ = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 1201, timestep=timestep, seed=32, lattice_hops=True)
    vectors = _vectors(9, num_atoms, 33)
    _check(positions, lattice, timestep, vectors)
    _check(positions, _sheared(lattice), timestep, vectors)


@pytest.mark.parametrize("frames", [4, 5, 1000, 2050])
@pytest.mark.parametrize("timestep", [0.5, 1.0, 2.0])
def test_wavenumbers_are_those_of_measure_and_vdos(frames, timestep):
    lattice, num_atoms, _ = _geometry("TiO2")
    trajectory = rb.Trajectory(synthetic.make_trajectory("TiO2", frames, seed=3), timestep)
    wn, rows = trajectory.get_projected_vdos(lattice, _vectors(3, num_atoms, 4))
    want, _ = rb.MDRamanSpectrum(np.zeros((frames, 3, 3)) + np.arange(frames)[:, None, None], timestep).measure()
    vdos_wn, _ = trajectory.get_vdos(lattice)
    assert np.array_equal(wn, want) and np.array_equal(wn, vdos_wn) and rows.shape == (3, len(want))


@pytest.mark.parametrize("frames", [2, 3])
def test_too_short_for_a_point_is_empty(frames):
    lattice, num_atoms, _ = _geometry("TiO2")
    trajectory = rb.Trajectory(synthetic.make_trajectory("TiO2", frames, seed=3), 1.0)
    wn, rows = trajectory.get_projected_vdos(lattice, _vectors(2, num_atoms, 5))
    assert wn.shape == (0,) and rows.shape == (2, 0)


def test_zero_vectors_give_exactly_zero_rows():
    """Zero vectors paired with a nonzero partner (modes 2, 5) and with each other (modes 6, 7)."""
    lattice, num_atoms, _ = _geometry("STO")
    positions = synthetic.make_trajectory("STO", 3001, seed=34)
    vectors = _vectors(9, num_atoms, 35)
    vectors[[2, 5, 6, 7]] = 0.0
    wn, rows = rb.Trajectory(positions, 1.0).get_projected_vdos(lattice, vectors)
    assert np.all(rows[[2, 5, 6, 7]] == 0.0)
    _, nonzero = rb.Trajectory(positions, 1.0).get_projected_vdos(lattice, vectors[[0, 1, 3, 4, 8]])
    want_wn, want = projected_vdos(positions, lattice, 1.0, vectors[[0, 1, 3, 4, 8]])
    assert np.array_equal(wn, want_wn)
    assert pointwise_rel_err(rows[[0, 1, 3, 4, 8]], want) <= INTENSITY_RTOL
    assert pointwise_rel_err(nonzero, want) <= INTENSITY_RTOL


def _llzo_masses(numbers):
    return np.array([MASSES[int(z)] for z in numbers])


def _identity_basis(num_atoms):
    vectors = np.zeros((3 * num_atoms, num_atoms, 3))
    vectors[np.arange(3 * num_atoms), np.arange(3 * num_atoms) // 3, np.arange(3 * num_atoms) % 3] = 1.0
    return vectors


def test_sum_rule_and_identity_basis_at_scale():
    lattice, num_atoms, numbers = _geometry("LLZO")
    masses = _llzo_masses(numbers)
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("LLZO", 100_001, seed=36)), 1.0)
    wn, rows = trajectory.get_projected_vdos(lattice, orthonormal_mass_weighted(masses, seed=37))
    vdos_wn, total = trajectory.get_vdos(lattice, None, masses)
    assert np.array_equal(wn, vdos_wn) and rows.shape == (3 * num_atoms, len(wn))
    assert pointwise_rel_err(rows.sum(axis=0), total[0]) <= 1e-8
    _, rows = trajectory.get_projected_vdos(lattice, _identity_basis(num_atoms))
    _, per_atom = trajectory.get_vdos(lattice, [[i] for i in range(num_atoms)])
    assert pointwise_rel_err(rows.reshape(num_atoms, 3, -1).sum(axis=1), per_atom) <= 1e-8


def test_real_llzo_outcar_trajectory(tmp_path):
    path = tmp_path / "OUTCAR_trajectory"
    with gzip.open(os.path.join(GOLDEN, "llzo_outcar_trajectory.txt.gz"), "rb") as fin, open(path, "wb") as fout:
        shutil.copyfileobj(fin, fout)
    _, lattice, _ = rio.read_outcar_positions_ts(path)
    with np.load(os.path.join(GOLDEN, "llzo_outcar_trajectory.npz")) as data:
        positions, timestep = data["positions_ts"], float(data["timestep"])
    assert positions.shape == (15, 108, 3)
    num_atoms = positions.shape[1]
    trajectory = rb.Trajectory(positions, timestep)
    wn, rows = trajectory.get_projected_vdos(lattice, _identity_basis(num_atoms))
    _, per_atom = trajectory.get_vdos(lattice, [[i] for i in range(num_atoms)])
    assert rows.shape == (3 * num_atoms, 6)
    assert pointwise_rel_err(rows.reshape(num_atoms, 3, -1).sum(axis=1), per_atom) <= 1e-8
    vectors = _vectors(10, num_atoms, 38)
    wn, rows = trajectory.get_projected_vdos(lattice, vectors)
    want_wn, want = projected_vdos(positions, lattice, timestep, vectors)
    assert np.array_equal(wn, want_wn)
    assert pointwise_rel_err(rows, want) <= INTENSITY_RTOL


def _peak_wavenumbers(wn, rows):
    return wn[np.argmax(rows, axis=1)]


def test_golden_phonon_modes_peak_at_their_wavenumbers():
    """A trajectory made of the 81 golden TiO2 modes, each at its own wavenumber, projected on their vectors."""
    lattice, num_atoms, numbers = _geometry("TiO2")
    masses = np.array([MASSES[int(z)] for z in numbers])
    with np.load(os.path.join(GOLDEN, "phonons_tio2.npz")) as data:
        phonons = rb.Phonons(data["ref_positions"], data["wavenumbers"], data["displacements"])
    frames, timestep = 20_001, 1.0
    steps = np.arange(frames)[:, None] * timestep
    phase = np.random.default_rng(39).uniform(0, 2 * np.pi, len(phonons.wavenumbers))
    motion = np.sin(2 * np.pi * phonons.wavenumbers[None, :] / CM_PER_FS * steps + phase)  # (S, modes)
    positions = phonons.ref_positions[None] + 0.05 * np.einsum("sk,kic->sic", motion, phonons.displacements)
    wn, rows = rb.Trajectory(positions - np.floor(positions), timestep).get_projected_vdos(
        lattice, phonons.get_mode_vectors(lattice, masses))
    bin_width = wn[1] - wn[0]
    optical = phonons.wavenumbers > 50.0
    assert optical.sum() >= 70
    peaks = _peak_wavenumbers(wn, rows)
    assert np.max(np.abs(peaks[optical] - phonons.wavenumbers[optical])) <= bin_width


def test_synthetic_modes_peak_at_their_frequencies():
    """``make_trajectory`` without noise, projected on its own eight mode vectors."""
    frames, seed = 6001, 101
    lattice, num_atoms, _ = _geometry("TiO2")
    _, frequencies, _, vectors = synthetic._mode_parameters(num_atoms, seed)  # pylint: disable=protected-access
    positions = synthetic.make_trajectory("TiO2", frames, seed=seed, noise=0.0)
    wn, rows = rb.Trajectory(positions, 1.0).get_projected_vdos(lattice, vectors.reshape(8, num_atoms, 3))
    bin_width = wn[1] - wn[0]
    peaks = _peak_wavenumbers(wn, rows)
    assert np.max(np.abs(peaks - frequencies * 33.35640951981521)) <= bin_width


def _equal(a, b):
    return torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_input_forms_and_repeated_calls_are_bit_identical():
    lattice, num_atoms, _ = _geometry("LLZO")
    positions = synthetic.make_trajectory("LLZO", 3001, seed=40)
    vectors = _vectors(45, num_atoms, 41)
    host = rb.Trajectory(positions, 1.0)
    device = rb.Trajectory(to_cuda(positions), 1.0)
    assert not host.is_device_resident and device.is_device_resident
    first = host.get_projected_vdos_device(lattice, vectors)
    assert _equal(first, device.get_projected_vdos_device(lattice, vectors))
    assert _equal(first, device.get_projected_vdos_device(lattice, to_cuda(vectors)))
    assert _equal(first, host.get_projected_vdos_device(lattice, torch.from_numpy(vectors)))
    assert _equal(first, device.get_projected_vdos_device(to_cuda(lattice), vectors))
    assert _equal(first, host.get_projected_vdos_device(lattice, vectors))


@pytest.mark.parametrize("windows_per_chunk", [1, 2, 3, 7])
def test_batch_size_does_not_change_a_bit(windows_per_chunk, monkeypatch):
    """405 vectors of STO (68 windows, 3N = 405) in chunks of every size; odd K pads the last window."""
    lattice, num_atoms, _ = _geometry("STO")
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("STO", 2001, seed=42)), 1.0)
    vectors = _vectors(3 * num_atoms, num_atoms, 43)
    default = trajectory.get_projected_vdos_device(_sheared(lattice), vectors)
    assert spectrum._window_batch(2001, 68) == 128  # pylint: disable=protected-access  (one chunk)
    per_window = 16 * 3 * 4096 + 8 * 3 * 2000 + 8 * ((2000 + 255) // 256 + 1) + 4  # a window of 2001 frames
    monkeypatch.setattr(spectrum, "_WINDOW_BATCH_BYTES", windows_per_chunk * per_window)
    assert spectrum._window_batch(2001, 68) == windows_per_chunk  # pylint: disable=protected-access
    assert _equal(default, trajectory.get_projected_vdos_device(_sheared(lattice), vectors))


def _launches(fn):
    fn()  # plans are created (and cached) here
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def test_launch_count(monkeypatch):
    """One projection, the transform passes and one combine per chunk: a single measure's launches."""
    frames = 20_001
    single = rb.MDRamanSpectrum(to_cuda(np.random.default_rng(9).normal(size=(frames, 3, 3))), 1.0)
    per_chunk = _launches(single.measure_device)
    counts = []
    for structure in ("TiO2", "LLZO"):
        lattice, num_atoms, _ = _geometry(structure)
        trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory(structure, frames, seed=44)), 1.0)
        for count in (1, 48):
            vectors = _vectors(count, num_atoms, count)
            counts.append(_launches(lambda t=trajectory, l=lattice, v=vectors: t.get_projected_vdos_device(l, v)))
    assert counts == [per_chunk] * 4
    lattice, num_atoms, _ = _geometry("TiO2")  # 324 modes: 54 windows in chunks of 8, 7 chunks
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("TiO2", frames, seed=44)), 1.0)
    per_window = 16 * 3 * 65536 + 8 * 3 * (frames - 1) + 8 * ((frames - 1 + 255) // 256 + 1) + 4
    monkeypatch.setattr(spectrum, "_WINDOW_BATCH_BYTES", 8 * per_window)
    assert spectrum._window_batch(frames, 54) == 8  # pylint: disable=protected-access
    vectors = _vectors(3 * num_atoms, num_atoms, 45)
    assert _launches(lambda: trajectory.get_projected_vdos_device(lattice, vectors)) == 7 * per_chunk


def test_c_entry_errors():
    frames, num_atoms, num_vectors = 300, 6, 3
    lib = _lib.lib()
    rng = np.random.default_rng(10)
    positions = to_cuda(rng.uniform(0, 1, (frames, num_atoms, 3)))
    points = int(lib.rn_spectrum_num_points(frames))
    wn = torch.empty(points, dtype=torch.float64, device="cuda:0")
    inten = torch.empty((num_vectors, points), dtype=torch.float64, device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.diag([5.0, 6.0, 7.0])
    vectors = rng.normal(size=(num_vectors, num_atoms, 3))
    handle, dist = ctypes.c_void_p(), ctypes.c_void_p()
    _lib.check(lib.rn_spectrum_plan_create_batched(frames, 2, 0, ctypes.byref(handle)), "create_batched")
    _lib.check(lib.rn_spectrum_plan_create_dist(frames, 0, 2, 0, ctypes.byref(dist)), "create_dist")
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731

    def call(plan=handle, pos=ctypes.c_void_p(positions.data_ptr()), n=num_atoms, lat=ptr(lattice),
             vec=ptr(vectors), k=num_vectors, dt=1.0, wn_ptr=ctypes.c_void_p(wn.data_ptr()),
             int_ptr=ctypes.c_void_p(inten.data_ptr())):
        return lib.rn_projected_vdos(plan, pos, n, lat, vec, k, dt, wn_ptr, int_ptr, stream)

    try:
        assert call(plan=None) == -1
        assert call(plan=dist) == -1  # a multi-GPU plan
        assert call(pos=None) == -1
        assert call(lat=None) == -1
        assert call(vec=None) == -1
        assert call(wn_ptr=None) == -1
        assert call(int_ptr=None) == -1
        assert call(n=0) == -1
        assert call(k=0) == -1
        assert call(dt=0.0) == -1
        assert call(dt=-1.0) == -1
        assert call(dt=float("nan")) == -1
        for value in (np.nan, np.inf):
            bad = vectors.copy()
            bad[2, 5, 1] = value
            assert call(vec=ptr(bad)) == -1
            bad_lattice = lattice.copy()
            bad_lattice[1, 2] = value
            assert call(lat=ptr(bad_lattice)) == -1
        assert call() == 0
        torch.cuda.synchronize()
        want_wn, want = rb.Trajectory(positions, 1.0).get_projected_vdos(lattice, vectors)
        assert np.array_equal(wn.cpu().numpy(), want_wn) and np.array_equal(inten.cpu().numpy(), want)
    finally:
        torch.cuda.synchronize()
        lib.rn_spectrum_plan_destroy(handle)
        lib.rn_spectrum_plan_destroy(dist)
