"""Vibrational density of states without a GPU: properties of the oracle (``vdos_oracle.vdos``) — additivity over a
partition of the atoms, linearity in the weights, invariance under lattice hops, peaks at the mode frequencies —
and the argument errors of ``Trajectory.get_vdos``, raised in order before any device work."""
import numpy as np
import pytest

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic

from vdos_oracle import vdos

THZ_TO_WAVENUMBER = 33.35640951981521  # cm^-1 per THz


def _structure(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _relative(a, b):
    return np.max(np.abs(a - b) / np.abs(b))


def test_partition_sums_to_the_total():
    lattice, num_atoms, numbers = _structure("STO")
    positions = synthetic.make_trajectory("STO", 301, seed=3)
    weights = np.random.default_rng(0).uniform(0.5, 3.0, num_atoms)
    groups = [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
    wn, parts = vdos(positions, lattice, 1.0, groups, weights)
    wn_total, total = vdos(positions, lattice, 1.0, [range(num_atoms)], weights)
    assert np.array_equal(wn, wn_total) and parts.shape == (len(groups), len(wn))
    assert _relative(parts.sum(axis=0), total[0]) <= 1e-12


def test_weights_scale_the_rows_exactly():
    lattice, num_atoms, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 200, seed=4)
    weights = np.random.default_rng(1).uniform(0.5, 3.0, num_atoms)
    groups = [range(0, 50), range(40, 108), [7]]
    _, rows = vdos(positions, lattice, 0.5, groups, weights)
    _, rows4 = vdos(positions, lattice, 0.5, groups, 4 * weights)
    assert np.array_equal(rows4, 4 * rows)


def test_lattice_hops_are_removed_by_the_minimum_image():
    lattice, num_atoms, _ = _structure("TiO2")
    plain = synthetic.make_trajectory("TiO2", 150, seed=5)
    hopped = synthetic.make_trajectory("TiO2", 150, seed=5, lattice_hops=True)
    assert np.max(np.abs(hopped - plain)) >= 1.0  # the hops are there
    groups = [range(num_atoms), range(0, num_atoms, 3)]
    wn, want = vdos(plain, lattice, 2.0, groups, np.ones(num_atoms))
    wn_hopped, got = vdos(hopped, lattice, 2.0, groups, np.ones(num_atoms))
    assert np.array_equal(wn, wn_hopped)
    assert _relative(got, want) <= 1e-12


def test_noise_free_peaks_at_the_mode_frequencies():
    """Seed 101 puts the eight modes at least ten bins apart for 6001 frames of 1 fs."""
    frames, seed = 6001, 101
    lattice, num_atoms, _ = _structure("TiO2")
    frequencies = synthetic._mode_parameters(num_atoms, seed)[1]  # pylint: disable=protected-access
    bin_width = THZ_TO_WAVENUMBER * 1e3 / (frames - 1)
    assert np.min(np.diff(np.sort(frequencies))) * THZ_TO_WAVENUMBER >= 10 * bin_width
    positions = synthetic.make_trajectory("TiO2", frames, seed=seed, noise=0.0)
    wn, rows = vdos(positions, lattice, 1.0, [range(num_atoms)], np.ones(num_atoms))
    row = rows[0]
    maxima = np.flatnonzero((row[1:-1] > row[:-2]) & (row[1:-1] > row[2:])) + 1
    largest = maxima[np.argsort(row[maxima])[::-1][:8]]
    for frequency in frequencies:
        assert np.min(np.abs(wn[largest] - frequency * THZ_TO_WAVENUMBER)) <= bin_width


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("method", ["get_vdos", "get_vdos_device"])
def test_argument_errors_before_device_work(method, no_device):  # pylint: disable=unused-argument
    lattice, num_atoms, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 20, seed=6)
    call = getattr(rb.Trajectory._from_wrapped(positions, 1.0), method)  # pylint: disable=protected-access
    one_frame = getattr(rb.Trajectory._from_wrapped(positions[:1], 1.0), method)  # pylint: disable=protected-access
    ones = np.ones(num_atoms)
    with pytest.raises(TypeError, match="lattice should have type ndarray, not list"):
        call([[1, 0, 0], [0, 1, 0], [0, 0, 1]])
    with pytest.raises(ValueError, match=r"lattice has wrong shape: \(3,\) != \(3,3\)"):
        call(np.ones(3))
    with pytest.raises(ValueError, match="lattice contains non-finite values"):
        call(np.diag([1.0, np.nan, 1.0]))
    with pytest.raises(TypeError, match="atom_groups should have type list, not int"):
        call(lattice, 3)
    with pytest.raises(TypeError, match="atom_groups should have type list, not str"):
        call(lattice, "Ti")
    with pytest.raises(ValueError, match="atom_groups is empty"):
        call(lattice, [])
    with pytest.raises(TypeError, match=r"atom_groups\[1\] should have type list, not int"):
        call(lattice, [[0, 1], 2])
    with pytest.raises(ValueError, match=r"atom_groups\[1\] is empty"):
        call(lattice, [[0], []])
    with pytest.raises(TypeError, match=r"atom_groups\[0\] entry should have type int, not float"):
        call(lattice, [[0, 1.0]])
    with pytest.raises(TypeError, match=r"atom_groups\[0\] entry should have type int, not bool"):
        call(lattice, [[True]])
    with pytest.raises(ValueError, match=r"atom_groups\[0\] has atom index 108 out of range \[0, 108\)"):
        call(lattice, [[0, 108]])
    with pytest.raises(ValueError, match=r"atom_groups\[1\] has atom index -1 out of range"):
        call(lattice, [[0], np.array([-1])])
    with pytest.raises(ValueError, match=r"atom_groups\[0\] repeats an atom"):
        call(lattice, [[3, 4, 3]])
    with pytest.raises(TypeError, match="atom_weights should have type ndarray, not list"):
        call(lattice, None, [1.0] * num_atoms)
    with pytest.raises(ValueError, match=r"atom_weights has wrong shape: \(107,\) != \(108,\)"):
        call(lattice, None, ones[1:])
    with pytest.raises(ValueError, match="atom_weights must be finite and >= 0"):
        call(lattice, None, -ones)
    with pytest.raises(ValueError, match="atom_weights must be finite and >= 0"):
        call(lattice, None, np.where(np.arange(num_atoms) == 5, np.inf, 1.0))
    with pytest.raises(ValueError, match="positions_ts must contain at least 2 frames"):
        one_frame(lattice)
    # the order: lattice, atom_groups, atom_weights, frames
    with pytest.raises(TypeError, match="lattice should have type"):
        one_frame([1], [], [1.0])
    with pytest.raises(ValueError, match="atom_groups is empty"):
        one_frame(lattice, [], [1.0])
    with pytest.raises(TypeError, match="atom_weights should have type"):
        one_frame(lattice, [[0]], [1.0])
    with pytest.raises(AssertionError, match="device work"):  # valid arguments reach the device
        call(lattice, [range(10), np.arange(5, 20)], 2 * ones)
    with pytest.raises(AssertionError, match="device work"):
        call(lattice)
