"""Distinct Van Hove correlation without a GPU: properties of the oracle (``distinct_van_hove_oracle``) — the vectorised
form against a plain loop, lag 0 against the RDF counts, a frozen trajectory, time reversal, additivity over disjoint
groups on either side, independent uniform frames giving 1 — and the argument errors of
``Trajectory.get_distinct_van_hove``, raised in their order before any device work."""
import math

import numpy as np
import pytest

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic

from distinct_van_hove_oracle import distinct_counts, distinct_van_hove
from rdf_oracle import bin_edges, cell_widths, rdf_counts


def _structure(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def _half_width(lattice):
    return cell_widths(lattice)[1].min() / 2


def _species(numbers):
    return [np.flatnonzero(numbers == z) for z in np.unique(numbers)]


def _overlapping(num_atoms):
    """Sizes 7, 10 and 1 with an overlap of the first two; the one-atom group has n_aa = 0."""
    return [list(range(0, 7)), list(range(3, 13)), [num_atoms - 1]]


def test_oracle_against_a_plain_loop():
    """The definition written out per (t, n, i, j) with Python floats (every operation rounded on its own)."""
    lattice = _sheared(np.diag([6.0, 7.0, 8.0]))
    rng = np.random.default_rng(1)
    positions = rng.uniform(0, 1, (6, 7, 3))
    groups = [[0, 1, 2, 3], [3, 4, 5], [6]]
    lags = [0, 1, 5]
    r_max, num_bins = _half_width(lattice), 9
    want = np.zeros((3, 3, 3, num_bins), dtype=np.int64)
    L = lattice.tolist()
    for ti, t in enumerate(lags):
        for n in range(6 - t):
            for a, ga in enumerate(groups):
                for b, gb in enumerate(groups):
                    for i in ga:
                        for j in gb:
                            if i == j:
                                continue
                            d = [float(positions[n + t, j, c] - positions[n, i, c]) for c in range(3)]
                            d = [dc - math.ceil(dc - 0.5) for dc in d]
                            v = [(d[0] * L[0][c] + d[1] * L[1][c]) + d[2] * L[2][c] for c in range(3)]
                            k = math.floor(math.sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]) * (num_bins / r_max))
                            if k < num_bins:
                                want[a, b, ti, k] += 1
    got = distinct_counts(positions, lattice, lags, r_max, num_bins, groups)
    assert np.array_equal(got, want)
    assert want.sum() > 0


@pytest.mark.parametrize("kind", ["all", "species", "overlapping"])
def test_lag_zero_is_the_rdf(kind):
    lattice, num_atoms, numbers = _structure("LLZO")
    positions = synthetic.make_trajectory("LLZO", 6, seed=2)
    groups = {"all": None, "species": _species(numbers), "overlapping": _overlapping(num_atoms)}[kind]
    r_max = _half_width(lattice)
    counts = distinct_counts(positions, lattice, [0, 2], r_max, 200, groups)
    assert np.array_equal(counts[:, :, 0], rdf_counts(positions, lattice, r_max, 200, groups))


def test_frozen_trajectory():
    """Every frame the same: the counts at lag t are (S - t) / S times those at lag 0, as integers."""
    lattice, _, numbers = _structure("TiO2")
    frames = 7
    positions = np.repeat(synthetic.make_trajectory("TiO2", 1, seed=3), frames, axis=0)
    lags = np.array([0, 1, 4, 6])
    counts = distinct_counts(positions, lattice, lags, _half_width(lattice), 150, _species(numbers))
    for ti, t in enumerate(lags):
        assert np.array_equal(counts[:, :, ti] * frames, counts[:, :, 0] * (frames - t))
    assert counts[:, :, 0].sum() > 0


def test_time_reversal():
    lattice, num_atoms, numbers = _structure("STO")
    positions = synthetic.make_trajectory("STO", 9, seed=4, lattice_hops=True)
    positions -= np.floor(positions)
    groups = _species(numbers) + [_overlapping(num_atoms)[1]]
    args = (_sheared(lattice), [0, 1, 3, 8], 0.9 * _half_width(_sheared(lattice)), 120, groups)
    forward = distinct_counts(positions, *args)
    backward = distinct_counts(positions[::-1], *args)
    assert np.array_equal(backward, forward.transpose(1, 0, 2, 3))
    assert not np.array_equal(forward[0, 1, 1:], forward[1, 0, 1:])  # not mirrored for t > 0


def test_disjoint_groups_add_up_on_either_side():
    lattice, num_atoms, numbers = _structure("LLZO")
    positions = synthetic.make_trajectory("LLZO", 5, seed=5)
    species = _species(numbers)
    counts = distinct_counts(positions, lattice, [0, 1, 4], _half_width(lattice), 100, species + [range(num_atoms)])
    n = len(species)
    assert np.array_equal(counts[:n, :n].sum(axis=0), counts[n, :n])
    assert np.array_equal(counts[:n, :n].sum(axis=1), counts[:n, n])
    assert np.array_equal(counts[:n, :n].sum(axis=(0, 1)), counts[n, n])


def test_independent_uniform_frames_give_one():
    """Frames drawn independently and uniformly: at t >= 1 each bin's count has a relative spread of about
    sqrt(1 / mu), mu its expectation (pairs that share an origin or a partner add a little); every bin stays within
    six times sqrt(2 / mu)."""
    lattice = np.array([[10.0, 0.0, 0.0], [1.0, 11.0, 0.0], [0.5, 0.7, 9.0]])
    frames, atoms = 40, 150
    positions = np.random.default_rng(6).uniform(0, 1, (frames, atoms, 3))
    r_max, num_bins = _half_width(lattice), 8
    lags = np.array([1, 5, 20])
    _, g_d, _ = distinct_van_hove(positions, lattice, lags, r_max, num_bins)
    _, _, shell = bin_edges(r_max, num_bins)
    mu = (frames - lags)[:, None] * atoms * (atoms - 1) * shell[None, :] / cell_widths(lattice)[0]
    assert np.all(np.abs(g_d[0, 0] - 1) <= 6 * np.sqrt(2 / mu))


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("method", ["get_distinct_van_hove", "get_distinct_van_hove_device"])
def test_argument_errors_before_device_work(method, no_device):  # pylint: disable=unused-argument
    lattice, _, _ = _structure("TiO2")
    r_max = _half_width(lattice)
    positions = synthetic.make_trajectory("TiO2", 20, seed=7)
    call = getattr(rb.Trajectory._from_wrapped(positions, 1.0), method)  # pylint: disable=protected-access
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
    for bad in (0.0, -1.0, np.nan, np.inf, r_max * (1 + 1e-9)):
        with pytest.raises(ValueError, match=r"r_max must be finite and in \(0, .*\] Å, half the smallest"):
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
    # the order: lattice, lags, r_max, num_bins, atom_groups
    with pytest.raises(TypeError, match="lattice should have type"):
        call([1], [20], -1.0, 0, [])
    with pytest.raises(ValueError, match="lags must be in"):
        call(lattice, [20], -1.0, 0, [])
    with pytest.raises(ValueError, match="r_max must be"):
        call(lattice, [0], -1.0, 0, [])
    with pytest.raises(ValueError, match="num_bins must be"):
        call(lattice, [0], 2.0, 0, [])
    with pytest.raises(ValueError, match="atom_groups is empty"):
        call(lattice, [0], 2.0, 10, [])
    # valid arguments reach the device: r_max at w_min / 2, lags 0 and S - 1 as a list, an array and uint64, the
    # largest bin count, overlapping groups, a single frame with lag 0
    for args in ((lattice, [0, 19], r_max, 4096), (lattice, np.arange(20), 2, 1, [[0], [0, 1]]),
                 (lattice, np.array([3], dtype=np.uint64), 2.0, 7)):
        with pytest.raises(AssertionError, match="device work"):
            call(*args)
    with pytest.raises(AssertionError, match="device work"):
        getattr(rb.Trajectory._from_wrapped(positions[:1], 1.0), method)(lattice, [0], 2.0, 7)  # pylint: disable=protected-access
