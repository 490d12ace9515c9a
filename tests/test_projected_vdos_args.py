"""Projected VDOS without a GPU: identities of the oracle (``projected_vdos_oracle.projected_vdos``) — unit vectors
give the velocity spectra, an atom's three rows add up to its VDOS, the sum rule for an orthonormal mass-weighted
basis, quadratic scaling — ``Phonons.get_mode_vectors`` on the golden TiO2 phonons, and the argument errors of
``get_projected_vdos`` and ``get_mode_vectors``, raised in order before any device work."""
import os

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib, synthetic

from helpers import GOLDEN
from projected_vdos_oracle import projected_vdos, velocities
from vdos_oracle import vdos

MASSES = {3: 6.94, 8: 15.999, 22: 47.867, 38: 87.62, 40: 91.224, 57: 138.905}  # amu by atomic number


def _structure(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _masses(numbers):
    return np.array([MASSES[int(z)] for z in numbers])


def _relative(a, b):
    return np.max(np.abs(a - b) / np.abs(b))


def orthonormal_mass_weighted(masses, seed):
    """vectors[k, i] = sqrt(m_i) Q[3i:3i+3, k] with Q the orthogonal factor of a random 3N x 3N matrix."""
    num_atoms = len(masses)
    q, _ = np.linalg.qr(np.random.default_rng(seed).normal(size=(3 * num_atoms, 3 * num_atoms)))
    return np.sqrt(masses)[None, :, None] * q.T.reshape(3 * num_atoms, num_atoms, 3)


def test_unit_vectors_give_the_velocity_spectra():
    lattice, num_atoms, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 301, seed=11, lattice_hops=True)
    v = velocities(positions, lattice, 0.5)
    picks = [(0, 0), (7, 1), (num_atoms - 1, 2)]
    vectors = np.zeros((len(picks), num_atoms, 3))
    for k, (i, c) in enumerate(picks):
        vectors[k, i, c] = 1.0
    wn, rows = projected_vdos(positions, lattice, 0.5, vectors)
    for k, (i, c) in enumerate(picks):
        want_wn, want = ora.calc_signal_spectrum(v[:, i, c], 0.5)
        assert np.array_equal(wn, want_wn[1:])
        assert _relative(rows[k], want[1:]) <= 1e-14


def test_three_rows_of_an_atom_add_up_to_its_vdos():
    lattice, num_atoms, _ = _structure("STO")
    positions = synthetic.make_trajectory("STO", 250, seed=12)
    for atom in (0, 77):
        vectors = np.zeros((3, num_atoms, 3))
        vectors[[0, 1, 2], atom, [0, 1, 2]] = 1.0
        wn, rows = projected_vdos(positions, lattice, 1.0, vectors)
        want_wn, want = vdos(positions, lattice, 1.0, [[atom]], np.ones(num_atoms))
        assert np.array_equal(wn, want_wn)
        assert _relative(rows.sum(axis=0), want[0]) <= 1e-12


def test_sum_rule_for_an_orthonormal_mass_weighted_basis():
    lattice, num_atoms, numbers = _structure("TiO2")
    masses = _masses(numbers)
    positions = synthetic.make_trajectory("TiO2", 201, seed=13)
    vectors = orthonormal_mass_weighted(masses, seed=14)
    assert vectors.shape == (3 * num_atoms, num_atoms, 3)
    wn, rows = projected_vdos(positions, lattice, 1.0, vectors)
    want_wn, want = vdos(positions, lattice, 1.0, [range(num_atoms)], masses)
    assert np.array_equal(wn, want_wn)
    assert _relative(rows.sum(axis=0), want[0]) <= 1e-10


def test_scaled_vectors_scale_the_rows_quadratically():
    lattice, num_atoms, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 180, seed=15)
    vectors = np.random.default_rng(16).normal(size=(5, num_atoms, 3))
    _, rows = projected_vdos(positions, lattice, 2.0, vectors)
    _, rows2 = projected_vdos(positions, lattice, 2.0, 2 * vectors)
    _, rows3 = projected_vdos(positions, lattice, 2.0, 3 * vectors)
    assert np.array_equal(rows2, 4 * rows)  # a power of two scales exactly
    assert _relative(rows3, 9 * rows) <= 1e-13


def _golden_phonons():
    lattice, _, numbers = _structure("TiO2")
    with np.load(os.path.join(GOLDEN, "phonons_tio2.npz")) as data:
        phonons = rb.Phonons(data["ref_positions"], data["wavenumbers"], data["displacements"])
    return phonons, lattice, _masses(numbers)


def test_mode_vectors_of_the_golden_tio2_phonons():
    phonons, lattice, masses = _golden_phonons()
    vectors = phonons.get_mode_vectors(lattice, masses)
    assert isinstance(vectors, np.ndarray) and vectors.shape == (81, 108, 3)
    eigenvectors = (vectors / np.sqrt(masses)[None, :, None]).reshape(81, -1)
    assert np.max(np.abs(np.linalg.norm(eigenvectors, axis=1) - 1.0)) <= 1e-12
    overlap = eigenvectors @ eigenvectors.T
    assert np.max(np.abs(overlap - np.diag(np.diag(overlap)))) <= 1e-5
    for k in (0, 40, 80):  # the formula, one mode at a time
        e = np.array([np.sqrt(masses[i]) * (phonons.displacements[k, i] @ lattice) for i in range(108)])
        want = np.sqrt(masses)[:, None] * e / np.sqrt(np.sum(e * e))
        assert np.max(np.abs(vectors[k] - want)) <= 1e-14 * np.max(np.abs(want))
    # the input forms are read on the host
    assert np.array_equal(phonons.get_mode_vectors(torch.from_numpy(lattice), torch.from_numpy(masses)), vectors)


def test_mode_vector_errors():
    phonons, lattice, masses = _golden_phonons()
    with pytest.raises(TypeError, match="lattice should have type ndarray, not list"):
        phonons.get_mode_vectors(lattice.tolist(), masses)
    with pytest.raises(ValueError, match="lattice contains non-finite values"):
        phonons.get_mode_vectors(np.diag([1.0, np.inf, 1.0]), masses)
    with pytest.raises(TypeError, match="atom_masses should have type ndarray, not list"):
        phonons.get_mode_vectors(lattice, masses.tolist())
    with pytest.raises(ValueError, match=r"atom_masses has wrong shape: \(107,\) != \(108,\)"):
        phonons.get_mode_vectors(lattice, masses[1:])
    for value in (0.0, -1.0, np.nan, np.inf):
        with pytest.raises(ValueError, match="atom_masses must be finite and > 0"):
            phonons.get_mode_vectors(lattice, np.where(np.arange(108) == 3, value, masses))
    displacements = phonons.displacements
    displacements[5] = 0.0
    zero = rb.Phonons(phonons.ref_positions, phonons.wavenumbers, displacements)
    with pytest.raises(ValueError, match="mode 5 has zero norm"):
        zero.get_mode_vectors(lattice, masses)


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("method", ["get_projected_vdos", "get_projected_vdos_device"])
def test_argument_errors_before_device_work(method, no_device):  # pylint: disable=unused-argument
    lattice, num_atoms, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 20, seed=6)
    call = getattr(rb.Trajectory._from_wrapped(positions, 1.0), method)  # pylint: disable=protected-access
    one_frame = getattr(rb.Trajectory._from_wrapped(positions[:1], 1.0), method)  # pylint: disable=protected-access
    vectors = np.ones((2, num_atoms, 3))
    with pytest.raises(TypeError, match="lattice should have type ndarray, not list"):
        call([[1, 0, 0], [0, 1, 0], [0, 0, 1]], vectors)
    with pytest.raises(ValueError, match=r"lattice has wrong shape: \(3,\) != \(3,3\)"):
        call(np.ones(3), vectors)
    with pytest.raises(ValueError, match="lattice contains non-finite values"):
        call(np.diag([1.0, np.nan, 1.0]), vectors)
    with pytest.raises(TypeError, match="vectors should have type ndarray, not list"):
        call(lattice, vectors.tolist())
    with pytest.raises(ValueError, match=r"vectors has wrong shape: \(108,3\) != \(_,_,3\)"):
        call(lattice, vectors[0])
    with pytest.raises(ValueError, match=r"vectors has wrong shape: \(2,108,2\) != \(_,_,3\)"):
        call(lattice, vectors[:, :, :2])
    with pytest.raises(ValueError, match="vectors has 107 atoms, the trajectory 108"):
        call(lattice, vectors[:, 1:])
    with pytest.raises(ValueError, match="vectors is empty"):
        call(lattice, vectors[:0])
    for value in (np.nan, np.inf, -np.inf):
        bad = vectors.copy()
        bad[1, 50, 2] = value
        with pytest.raises(ValueError, match="vectors contains non-finite values"):
            call(lattice, bad)
    with pytest.raises(ValueError, match="positions_ts must contain at least 2 frames"):
        one_frame(lattice, vectors)
    # the order: lattice, vectors (shape, atoms, finite), frames
    with pytest.raises(TypeError, match="lattice should have type"):
        one_frame([1], vectors[:0, 1:])
    with pytest.raises(ValueError, match="vectors has wrong shape"):
        one_frame(lattice, np.ones((0, 5, 2)))
    with pytest.raises(ValueError, match="vectors has 5 atoms"):
        one_frame(lattice, np.ones((0, 5, 3)))
    with pytest.raises(ValueError, match="vectors is empty"):
        one_frame(lattice, np.full((0, num_atoms, 3), np.nan))
    with pytest.raises(ValueError, match="vectors contains non-finite values"):
        one_frame(lattice, np.full((1, num_atoms, 3), np.nan))
    # numpy, CPU tensors and zero vectors are valid and reach the device
    for good in (vectors, torch.from_numpy(vectors), np.zeros((1, num_atoms, 3))):
        with pytest.raises(AssertionError, match="device work"):
            call(lattice, good)
