"""Radial distribution functions without a GPU: properties of the oracle (``rdf_oracle``) — the shell counts of a simple
cubic crystal, g = 1 for uniform random positions, the symmetry g[a,b] = g[b,a], species partitions adding up to the
all-atom counts, additivity over frames, the per-component wrap against a search over the 27 images of a sheared cell
— and the argument errors of ``Trajectory.get_rdf``, raised in their order before any device work."""
import numpy as np
import pytest

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic

from rdf_oracle import bin_edges, cell_widths, pair_norms, rdf, rdf_counts


def _structure(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def test_simple_cubic_shell_counts():
    """4 x 4 x 4 sites of spacing 3 Å: 6, 12 and 8 neighbours at a, a sqrt 2 and a sqrt 3 (2a = 6 Å is beyond r_max)."""
    a, n = 3.0, 4
    lattice = np.eye(3) * a * n
    grid = np.array([[i, j, k] for i in range(n) for j in range(n) for k in range(n)], dtype=np.float64) / n
    positions = np.stack([grid, grid])  # two identical frames
    r_max, num_bins = 5.9, 59
    assert r_max <= cell_widths(lattice)[1].min() / 2
    r, g, counts = rdf(positions, lattice, r_max, num_bins)
    width = r_max / num_bins
    total = counts[0, 0]
    for distance, neighbours in ((a, 6), (a * np.sqrt(2), 12), (a * np.sqrt(3), 8)):
        k = int(np.floor(distance * (num_bins / r_max)))
        assert abs(r[k] - distance) <= width  # the bin holds the shell
        assert total[k] == 2 * n**3 * neighbours
    assert total.sum() == 2 * n**3 * 26
    assert np.all(g[0, 0][total == 0] == 0)


def test_uniform_random_positions_give_one():
    """Independent uniform positions: each bin's count has a relative spread of about sqrt(2 / mu), mu its expectation;
    every bin stays within six of those."""
    lattice = np.array([[10.0, 0.0, 0.0], [1.0, 11.0, 0.0], [0.5, 0.7, 9.0]])
    positions = np.random.default_rng(1).uniform(0, 1, (40, 150, 3))
    r_max = cell_widths(lattice)[1].min() / 2
    num_bins = 12
    _, g, _ = rdf(positions, lattice, r_max, num_bins)
    _, _, shell = bin_edges(r_max, num_bins)
    mu = 40 * 150 * 149 * shell / cell_widths(lattice)[0]
    assert np.all(np.abs(g[0, 0] - 1) <= 6 * np.sqrt(2 / mu))


def test_symmetry_partition_and_frame_additivity():
    lattice, num_atoms, numbers = _structure("LLZO")
    positions = synthetic.make_trajectory("LLZO", 12, seed=2)
    species = [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
    r_max, num_bins = cell_widths(lattice)[1].min() / 2, 50
    _, g, counts = rdf(positions, lattice, r_max, num_bins, species)
    assert np.array_equal(g, g.transpose(1, 0, 2)) and np.array_equal(counts, counts.transpose(1, 0, 2))
    _, g_all, all_counts = rdf(positions, lattice, r_max, num_bins)
    assert np.array_equal(counts.sum(axis=(0, 1)), all_counts[0, 0])  # the sum rule, in counts
    norms = pair_norms(species, num_atoms)
    weighted = np.einsum("ab,abk->k", norms, g)
    assert np.max(np.abs(weighted - num_atoms * (num_atoms - 1) * g_all[0, 0])) <= 1e-12 * np.max(weighted)
    _, g1, c1 = rdf(positions[:5], lattice, r_max, num_bins, species)
    _, g2, c2 = rdf(positions[5:], lattice, r_max, num_bins, species)
    assert np.array_equal(c1 + c2, counts)
    assert np.max(np.abs(12 * g - (5 * g1 + 7 * g2))) <= 1e-12 * np.max(12 * g)


def test_overlapping_groups_exclude_shared_atoms_by_index():
    lattice, num_atoms, _ = _structure("TiO2")
    positions = synthetic.make_trajectory("TiO2", 3, seed=4)
    groups = [list(range(0, 7)), list(range(3, 13)), [num_atoms - 1]]
    counts = rdf_counts(positions, lattice, 4.0, 40, groups)
    norms = pair_norms(groups, num_atoms)
    assert norms[0, 1] == 7 * 10 - 4 and norms[2, 2] == 0 and norms[0, 0] == 42
    brute = np.zeros(40, dtype=np.int64)  # the sum of the per-atom counts over i in a, j in b, i != j
    k_all = rdf_counts(positions, lattice, 4.0, 40, [[i] for i in range(13)])
    for i in range(0, 7):
        for j in range(3, 13):
            if i != j:
                brute += k_all[i, j]
    assert np.array_equal(counts[0, 1], brute)
    assert np.all(counts[2, 2] == 0)


def test_sheared_cell_wrap_agrees_with_the_27_images():
    lattice = _sheared(_structure("TiO2")[0])
    volume, widths = cell_widths(lattice)
    r_max = widths.min() / 2
    x = np.random.default_rng(3).uniform(0, 1, (300, 3))
    d = x[None, :, :] - x[:, None, :]
    wrapped = d - np.ceil(d - 0.5)
    near = np.linalg.norm(wrapped @ lattice, axis=2)
    images = np.array([[i, j, k] for i in (-1, 0, 1) for j in (-1, 0, 1) for k in (-1, 0, 1)], dtype=np.float64)
    brute = np.min(np.linalg.norm((d[:, :, None, :] + images[None, None]) @ lattice, axis=3), axis=2)
    inside = brute < r_max
    assert inside.sum() > 1000 and volume > 0
    assert np.max(np.abs(near[inside] - brute[inside])) <= 1e-12 * r_max
    assert np.array_equal(near < r_max * (1 - 1e-12), brute < r_max * (1 - 1e-12))


@pytest.fixture(name="no_device")
def fixture_no_device(monkeypatch):
    def fail():
        raise AssertionError("device work before the argument checks")

    monkeypatch.setattr(_lib, "lib", fail)


@pytest.mark.parametrize("method", ["get_rdf", "get_rdf_device"])
def test_argument_errors_before_device_work(method, no_device):  # pylint: disable=unused-argument
    lattice, _, _ = _structure("TiO2")
    half = cell_widths(lattice)[1].min() / 2
    positions = synthetic.make_trajectory("TiO2", 20, seed=6)
    call = getattr(rb.Trajectory._from_wrapped(positions, 1.0), method)  # pylint: disable=protected-access
    no_frames = getattr(rb.Trajectory._from_wrapped(positions[:0], 1.0), method)  # pylint: disable=protected-access
    with pytest.raises(TypeError, match="lattice should have type ndarray, not list"):
        call([[1, 0, 0], [0, 1, 0], [0, 0, 1]], 1.0, 10)
    with pytest.raises(ValueError, match=r"lattice has wrong shape: \(3,\) != \(3,3\)"):
        call(np.ones(3), 1.0, 10)
    with pytest.raises(ValueError, match="lattice contains non-finite values"):
        call(np.diag([1.0, np.nan, 1.0]), 1.0, 10)
    with pytest.raises(ValueError, match="lattice has zero cell volume"):
        call(np.array([[1.0, 0, 0], [2.0, 0, 0], [0, 0, 1.0]]), 1.0, 10)
    with pytest.raises(TypeError, match="r_max should have type float, not str"):
        call(lattice, "3", 10)
    with pytest.raises(TypeError, match="r_max should have type float, not bool"):
        call(lattice, True, 10)
    for bad in (0.0, -1.0, np.nan, np.inf, half * (1 + 1e-9)):
        with pytest.raises(ValueError, match=rf"r_max must be finite and in \(0, {half:.6g}\] Å"):
            call(lattice, bad, 10)
    with pytest.raises(TypeError, match="num_bins should have type int, not float"):
        call(lattice, 2.0, 10.0)
    for bad in (0, 4097, -3):
        with pytest.raises(ValueError, match=r"num_bins must be in 1\.\.4096"):
            call(lattice, 2.0, bad)
    with pytest.raises(ValueError, match="atom_groups is empty"):
        call(lattice, 2.0, 10, [])
    with pytest.raises(ValueError, match=r"atom_groups\[0\] has atom index 108 out of range \[0, 108\)"):
        call(lattice, 2.0, 10, [[0, 108]])
    with pytest.raises(ValueError, match=r"atom_groups\[0\] repeats an atom"):
        call(lattice, 2.0, 10, [[3, 4, 3]])
    with pytest.raises(ValueError, match="positions_ts must contain at least 1 frame"):
        no_frames(lattice, 2.0, 10)
    # the order: lattice, r_max, num_bins, atom_groups, frames
    with pytest.raises(TypeError, match="lattice should have type"):
        no_frames([1], -1.0, 0, [])
    with pytest.raises(ValueError, match="r_max must be"):
        no_frames(lattice, -1.0, 0, [])
    with pytest.raises(ValueError, match="num_bins must be"):
        no_frames(lattice, 2.0, 0, [])
    with pytest.raises(ValueError, match="atom_groups is empty"):
        no_frames(lattice, 2.0, 10, [])
    # valid arguments reach the device: r_max at the bound (also half the edge of an orthorhombic cell), one frame,
    # integer r_max, the largest bin count
    with pytest.raises(AssertionError, match="device work"):
        call(np.diag([5.0, 6.0, 7.0]), 2.5, 16)
    for args in ((lattice, half, 4096), (lattice, 2, 1, [[0], [0, 1]])):
        with pytest.raises(AssertionError, match="device work"):
            call(*args)
    with pytest.raises(AssertionError, match="device work"):
        getattr(rb.Trajectory._from_wrapped(positions[:1], 1.0), method)(lattice, 2.0, 7)  # pylint: disable=protected-access
