"""Self Van Hove correlation without a GPU: properties of the oracle (``van_hove_oracle``) — lag 0, the count bound
and its equality, additivity over disjoint groups, m2 against the MSD oracle, a ballistic group in one bin with
alpha2 = -2/5, a Gaussian random walk with alpha2 near 0, invariance under lattice hops and whole-cell shifts — and
the argument errors of ``Trajectory.get_van_hove``, raised in their order before any device work."""
import numpy as np
import pytest

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic

from msd_oracle import msd_direct
from rdf_oracle import bin_edges
from van_hove_oracle import alpha2, van_hove


def _structure(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _species(numbers):
    return [np.flatnonzero(numbers == z) for z in np.unique(numbers)]


def test_lag_zero_fills_bin_zero():
    lattice, num_atoms, numbers = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 30, seed=1)
    groups = _species(numbers)
    _, g_s, moments, counts = van_hove(positions, lattice, [0, 3], 2.0, 40, groups)
    sizes = np.array([len(g) for g in groups])
    assert np.array_equal(counts[:, 0, 0], 30 * sizes)
    assert np.all(counts[:, 0, 1:] == 0)
    assert np.all(moments[:, 0] == 0.0)
    assert np.all(moments[:, 1] > 0.0)


def test_count_bound_and_equality():
    lattice, num_atoms, numbers = _structure("STO")
    positions = synthetic.make_trajectory("STO", 50, seed=2)
    groups = _species(numbers)
    lags = [1, 7, 49]
    sizes = np.array([len(g) for g in groups])
    norm = (50 - np.array(lags))[None, :] * sizes[:, None]
    _, _, _, counts = van_hove(positions, lattice, lags, 0.05, 30, groups)
    assert np.all(counts.sum(axis=2) <= norm) and np.any(counts.sum(axis=2) < norm)
    _, g_s, _, counts = van_hove(positions, lattice, lags, 50.0, 30, groups)
    assert np.array_equal(counts.sum(axis=2), norm)
    assert np.allclose(np.sum(g_s * bin_edges(50.0, 30)[2], axis=2), 1.0, rtol=1e-14, atol=0)


def test_disjoint_groups_add_up():
    lattice, num_atoms, numbers = _structure("LLZO")
    positions = synthetic.make_trajectory("LLZO", 20, seed=3)
    groups = _species(numbers)
    lags = [0, 1, 5, 19]
    _, _, moments, counts = van_hove(positions, lattice, lags, 3.0, 60, groups)
    _, _, all_moments, all_counts = van_hove(positions, lattice, lags, 3.0, 60, None)
    assert np.array_equal(counts.sum(axis=0), all_counts[0])
    sizes = np.array([len(g) for g in groups])[:, None]
    assert np.allclose((moments[..., 0] * sizes).sum(axis=0) / num_atoms, all_moments[0, :, 0], rtol=1e-13)


def test_m2_is_the_msd():
    lattice, num_atoms, numbers = _structure("LLZO")
    positions = synthetic.make_trajectory("LLZO", 60, seed=4, lattice_hops=True)
    wrapped = rb.Trajectory(positions, 1.0, pin_memory=False).positions_ts
    groups = _species(numbers)
    lags = np.array([0, 1, 2, 17, 59])
    _, msd = msd_direct(wrapped, lattice, 1.0, groups)
    _, _, moments, _ = van_hove(wrapped, lattice, lags, 4.0, 10, groups)
    assert np.all(moments[:, 0, 0] == 0.0)
    assert np.max(np.abs(moments[:, 1:, 0] - msd[:, lags[1:]]) / msd[:, lags[1:]]) <= 1e-12


def test_ballistic_group_lands_in_one_bin():
    """Atoms moving 1.3 Å per frame in different directions cross five cells of 10 Å; every displacement at lag t has
    the length 1.3 t, at least 0.15 bin widths from an edge, and alpha2 = 3 (1.3 t)^4 / (5 (1.3 t)^4) - 1 = -2/5."""
    lattice = np.diag([10.0, 10.0, 10.0])
    rng = np.random.default_rng(5)
    directions = rng.normal(size=(6, 3))
    directions /= np.linalg.norm(directions, axis=1, keepdims=True)
    frames, speed = 40, 1.3
    cart = rng.uniform(0, 10, (1, 6, 3)) + speed * np.arange(frames)[:, None, None] * directions[None]
    positions = cart @ np.linalg.inv(lattice)
    positions -= np.floor(positions)
    lags = [1, 2, 3, 5, 8]
    r_max, num_bins = 20.0, 310
    _, _, moments, counts = van_hove(positions, lattice, lags, r_max, num_bins)
    for ti, t in enumerate(lags):
        k = int(np.floor(speed * t * num_bins / r_max))
        assert counts[0, ti, k] == 6 * (frames - t)
    assert np.max(np.abs(alpha2(moments) + 0.4)) <= 1e-12


def test_gaussian_random_walk_alpha2():
    """Gaussian steps of 0.3 Å per component: every displacement is Gaussian, so alpha2 = 0 up to sampling noise.  With
    n independent samples of rr = sigma^2 chi2_3 the estimate has a standard deviation below 2/sqrt(n); origins of
    lag t overlap, so n = N (S - t) / t, and six deviations are allowed."""
    lattice = np.diag([8.0, 9.0, 10.0])
    rng = np.random.default_rng(6)
    frames, atoms = 4000, 40
    cart = np.cumsum(rng.normal(scale=0.3, size=(frames, atoms, 3)), axis=0)
    positions = cart @ np.linalg.inv(lattice)
    positions -= np.floor(positions)
    lags = np.array([1, 4, 16])
    _, _, moments, _ = van_hove(positions, lattice, lags, 10.0, 100)
    bound = 6 * 2 / np.sqrt(atoms * (frames - lags) / lags)
    assert np.all(np.abs(alpha2(moments[0])) <= bound)
    assert np.allclose(moments[0, :, 0], 3 * 0.09 * lags, rtol=0.1)


def test_invariant_under_hops_and_cell_shifts():
    """Dyadic positions (multiples of 2^-20) keep every difference exact, so integer hops of single frames and a
    shift of the whole trajectory by a lattice vector leave every count and moment unchanged bit for bit."""
    lattice, num_atoms, numbers = _structure("TiO2")
    positions = np.rint(synthetic.make_trajectory("TiO2", 40, seed=7) * 2**20) / 2**20
    rng = np.random.default_rng(7)
    hops = rng.integers(-3, 4, size=positions.shape).astype(np.float64)
    hops[np.arange(40) % 5 != 0] = 0.0
    args = (lattice, [0, 1, 6, 39], 2.5, 50, _species(numbers))
    want = van_hove(positions, *args)
    for moved in (positions + hops, positions + np.array([2.0, -1.0, 3.0])):
        got = van_hove(moved, *args)
        for a, b in zip(got, want):
            assert np.array_equal(a, b)


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("method", ["get_van_hove", "get_van_hove_device"])
def test_argument_errors_before_device_work(method, no_device):  # pylint: disable=unused-argument
    lattice, _, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 20, seed=8)
    call = getattr(rb.Trajectory._from_wrapped(positions, 1.0), method)  # pylint: disable=protected-access
    one_frame = getattr(rb.Trajectory._from_wrapped(positions[:1], 1.0), method)  # pylint: disable=protected-access
    with pytest.raises(TypeError, match="lattice should have type ndarray, not list"):
        call([[1, 0, 0], [0, 1, 0], [0, 0, 1]], [1], 1.0, 10)
    with pytest.raises(ValueError, match=r"lattice has wrong shape: \(3,\) != \(3,3\)"):
        call(np.ones(3), [1], 1.0, 10)
    with pytest.raises(ValueError, match="lattice contains non-finite values"):
        call(np.diag([1.0, np.nan, 1.0]), [1], 1.0, 10)
    with pytest.raises(ValueError, match="lattice has zero cell volume"):
        call(np.array([[1.0, 0, 0], [2.0, 0, 0], [0, 0, 1.0]]), [1], 1.0, 10)
    with pytest.raises(TypeError, match="lags should have type list, not str"):
        call(lattice, "12", 1.0, 10)
    with pytest.raises(ValueError, match=r"lags must be 1-D \(got shape \(\)\)"):
        call(lattice, 3, 1.0, 10)
    with pytest.raises(ValueError, match=r"lags must be 1-D \(got shape \(1, 2\)\)"):
        call(lattice, [[1, 2]], 1.0, 10)
    with pytest.raises(ValueError, match="lags is empty"):
        call(lattice, [], 1.0, 10)
    for bad in ([1.0, 2.0], [True, False], np.array([1.5])):
        with pytest.raises(TypeError, match="lags should have type int"):
            call(lattice, bad, 1.0, 10)
    for bad in ([2, 2], [3, 1], [0, 5, 4]):
        with pytest.raises(ValueError, match="lags must be strictly increasing"):
            call(lattice, bad, 1.0, 10)
    for bad in ([-1, 3], [0, 20]):
        with pytest.raises(ValueError, match=r"lags must be in \[0, 20\)"):
            call(lattice, bad, 1.0, 10)
    with pytest.raises(TypeError, match="r_max should have type float, not str"):
        call(lattice, [1], "3", 10)
    with pytest.raises(TypeError, match="r_max should have type float, not bool"):
        call(lattice, [1], True, 10)
    for bad in (0.0, -1.0, np.nan, np.inf):
        with pytest.raises(ValueError, match=r"r_max must be finite and > 0"):
            call(lattice, [1], bad, 10)
    with pytest.raises(TypeError, match="num_bins should have type int, not float"):
        call(lattice, [1], 2.0, 10.0)
    for bad in (0, 4097, -3):
        with pytest.raises(ValueError, match=r"num_bins must be in 1\.\.4096"):
            call(lattice, [1], 2.0, bad)
    with pytest.raises(ValueError, match="atom_groups is empty"):
        call(lattice, [1], 2.0, 10, [])
    with pytest.raises(ValueError, match=r"atom_groups\[0\] has atom index 108 out of range \[0, 108\)"):
        call(lattice, [1], 2.0, 10, [[0, 108]])
    with pytest.raises(ValueError, match=r"atom_groups\[0\] repeats an atom"):
        call(lattice, [1], 2.0, 10, [[3, 4, 3]])
    with pytest.raises(ValueError, match="positions_ts must contain at least 2 frames"):
        one_frame(lattice, [0], 2.0, 10)
    # the order: lattice, lags, r_max, num_bins, atom_groups, frames
    with pytest.raises(TypeError, match="lattice should have type"):
        one_frame([1], [5], -1.0, 0, [])
    with pytest.raises(ValueError, match="lags must be in"):
        one_frame(lattice, [5], -1.0, 0, [])
    with pytest.raises(ValueError, match="r_max must be"):
        one_frame(lattice, [0], -1.0, 0, [])
    with pytest.raises(ValueError, match="num_bins must be"):
        one_frame(lattice, [0], 2.0, 0, [])
    with pytest.raises(ValueError, match="atom_groups is empty"):
        one_frame(lattice, [0], 2.0, 10, [])
    # valid arguments reach the device: r_max beyond the cell, lags 0 and S - 1 as a list, an array and uint64, the
    # largest bin count, overlapping groups, two frames
    for args in ((lattice, [0, 19], 1e3, 4096), (lattice, np.arange(20), 2, 1, [[0], [0, 1]]),
                 (lattice, np.array([3], dtype=np.uint64), 2.0, 7)):
        with pytest.raises(AssertionError, match="device work"):
            call(*args)
    with pytest.raises(AssertionError, match="device work"):
        getattr(rb.Trajectory._from_wrapped(positions[:2], 1.0), method)(lattice, [0, 1], 2.0, 7)  # pylint: disable=protected-access
