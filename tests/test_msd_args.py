"""Mean squared displacement without a GPU: properties of the oracle (``msd_oracle``) — its direct and FFT forms agree,
the integer unwrap is the running sum of the minimum-image steps, lattice hops and whole-cell shifts change nothing, a
ballistic path gives m^2 |v dt|^2, per-atom rows average to the group row, MSD(1) is the mean squared step — and the
argument errors of ``Trajectory.get_msd``, raised in the order of ``get_vdos`` before any device work."""
import numpy as np
import pytest

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic

from msd_oracle import error_ratio, msd_direct, msd_fft, unwrapped_paths
from oracle import numpy_port as ora


def _structure(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _diffusing(structure, frames, seed, species_z, step=0.3):
    """A synthetic trajectory with a random walk (Å per frame, per component) added to one species before wrapping."""
    lattice, _, numbers = _structure(structure)
    positions = synthetic.make_trajectory(structure, frames, seed=seed)
    walk = np.cumsum(np.random.default_rng(seed).normal(scale=step, size=positions.shape), axis=0)
    walk[:, numbers != species_z] = 0.0
    moved = positions + walk @ np.linalg.inv(lattice)
    return moved - np.floor(moved)


def test_direct_and_fft_forms_agree():
    lattice, num_atoms, numbers = _structure("LLZO")
    positions = _diffusing("LLZO", 400, 1, 3)
    groups = [np.flatnonzero(numbers == z) for z in np.unique(numbers)] + [range(num_atoms), [5]]
    lags, want = msd_direct(positions, lattice, 2.0, groups)
    fft_lags, got = msd_fft(positions, lattice, 2.0, groups)
    assert np.array_equal(lags, fft_lags) and np.array_equal(lags, np.arange(400) * 2.0)
    assert np.all(want[:, 0] == 0) and np.all(got[:, 0] == 0)
    assert error_ratio(got, want, positions, lattice, groups) <= 1e-13


def test_integer_unwrap_is_the_running_sum_of_the_steps():
    lattice, _, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 300, seed=2, lattice_hops=True)
    x = ora.apply_pbc(positions)
    d = ora.apply_pbc_displacement(np.diff(x, axis=0))
    want = np.concatenate([np.zeros_like(x[:1]), np.cumsum(d, axis=0)]) @ lattice
    got = unwrapped_paths(positions, lattice)
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(lattice))


def test_lattice_hops_and_whole_cell_shifts_change_nothing():
    lattice, num_atoms, _ = _structure("STO")
    plain = synthetic.make_trajectory("STO", 200, seed=3)
    hopped = synthetic.make_trajectory("STO", 200, seed=3, lattice_hops=True)
    assert np.max(np.abs(hopped - plain)) >= 1.0  # the hops are there
    shifted = plain + np.array([3.0, -2.0, 7.0])
    groups = [range(num_atoms), range(0, num_atoms, 4)]
    _, want = msd_direct(plain, lattice, 1.0, groups)
    for other in (hopped, shifted):
        _, got = msd_direct(other, lattice, 1.0, groups)
        assert error_ratio(got, want, plain, lattice, groups) <= 1e-13


def test_ballistic_path_across_the_cell():
    lattice, _, _ = _structure("TiO2")
    lattice = lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])
    frames = 120
    velocity = np.array([[0.11, -0.07, 0.23], [-0.31, 0.05, 0.0]])  # fractional per frame: crosses the cell often
    positions = np.array([[0.9, 0.2, 0.5], [0.1, 0.95, 0.3]]) + np.arange(frames)[:, None, None] * velocity
    assert np.max(np.abs(np.floor(positions))) >= 10
    _, got = msd_direct(positions, lattice, 0.5, [[0], [1], [0, 1]])
    step = np.sum((velocity @ lattice) ** 2, axis=1)
    lags = np.arange(frames)
    want = np.stack([step[0] * lags**2, step[1] * lags**2, np.mean(step) * lags**2])
    assert np.max(np.abs(got - want) / np.maximum(want, 1e-300)) <= 1e-10


def test_per_atom_rows_average_to_the_group_row():
    lattice, num_atoms, numbers = _structure("TiO2")
    positions = _diffusing("TiO2", 250, 4, 8)
    group = np.flatnonzero(numbers == 8)
    _, per_atom = msd_direct(positions, lattice, 1.0, [[i] for i in range(num_atoms)])
    _, row = msd_direct(positions, lattice, 1.0, [group])
    assert np.max(np.abs(per_atom[group].mean(axis=0) - row[0])) <= 1e-12 * np.max(row)


def test_lag_one_is_the_mean_squared_step():
    lattice, num_atoms, _ = _structure("LLZO")
    positions = synthetic.make_trajectory("LLZO", 150, seed=5, lattice_hops=True)
    _, rows = msd_direct(positions, lattice, 1.0, [range(num_atoms)])
    d = ora.apply_pbc_displacement(np.diff(ora.apply_pbc(positions), axis=0))
    want = np.mean(np.sum((d @ lattice) ** 2, axis=2))
    assert abs(rows[0, 1] - want) <= 1e-12 * want


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("method", ["get_msd", "get_msd_device"])
def test_argument_errors_before_device_work(method, no_device):  # pylint: disable=unused-argument
    lattice, _, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 20, seed=6)
    call = getattr(rb.Trajectory._from_wrapped(positions, 1.0), method)  # pylint: disable=protected-access
    one_frame = getattr(rb.Trajectory._from_wrapped(positions[:1], 1.0), method)  # pylint: disable=protected-access
    with pytest.raises(TypeError, match="lattice should have type ndarray, not list"):
        call([[1, 0, 0], [0, 1, 0], [0, 0, 1]])
    with pytest.raises(ValueError, match=r"lattice has wrong shape: \(3,\) != \(3,3\)"):
        call(np.ones(3))
    with pytest.raises(ValueError, match="lattice contains non-finite values"):
        call(np.diag([1.0, np.inf, 1.0]))
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
    with pytest.raises(ValueError, match="positions_ts must contain at least 2 frames"):
        one_frame(lattice)
    # the order: lattice, atom_groups, frames
    with pytest.raises(TypeError, match="lattice should have type"):
        one_frame([1], [])
    with pytest.raises(ValueError, match="atom_groups is empty"):
        one_frame(lattice, [])
    with pytest.raises(AssertionError, match="device work"):  # valid arguments reach the device
        call(lattice, [range(10), np.arange(5, 20)])
    with pytest.raises(AssertionError, match="device work"):
        call(lattice)
