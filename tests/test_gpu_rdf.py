"""Radial distribution functions (``Trajectory.get_rdf``) on the GPU: every element within 1e-13 relative of the oracle
and exactly 0 where the oracle's count is 0 (with counts below 1e10, one count more or less would move g by more than
1e-10, so this pins the integer counts), over structures, group layouts, frame counts, bin counts, r_max at and inside
the w_min/2 limit, sheared lattices, lattice hops, the 1536-atom supercell and the real LLZO OUTCAR trajectory;
bit-identity across input forms, repeated calls, group sets and frame splits; the species sum rule; the launch count and
the C entry's errors."""
import ctypes
import gzip
import os
import shutil

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from ramannoodle_b200 import _lib, synthetic
from ramannoodle_b200 import io as rio

from gpu_helpers import to_cuda
from helpers import GOLDEN
from rdf_oracle import bin_edges, cell_widths, pair_norms, rdf

pytestmark = pytest.mark.gpu

RDF_RTOL = 1e-13


def _geometry(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    """The lattice with off-diagonal entries of 1-3 Å: every entry of the lattice product is used."""
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def _half_width(lattice):
    return cell_widths(lattice)[1].min() / 2


def _groups(kind, num_atoms, numbers):
    if kind == "all":
        return None
    if kind == "species":
        return [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
    if kind == "odd_even_overlap":  # sizes 7, 10, 1 and an overlap of the first two; the one-atom group has n_aa = 0
        return [list(range(0, 7)), list(range(3, 13)), [num_atoms - 1], list(range(num_atoms - 1, 20, -9))]
    if kind == "per_atom":
        return [[i] for i in range(num_atoms)]
    raise AssertionError(kind)


def _compare(r, g, want_r, want_g, counts):
    assert np.array_equal(r, want_r)
    assert g.shape == want_g.shape
    assert np.all(g[counts == 0] == 0.0)
    nonzero = counts > 0
    assert np.all(g[nonzero] > 0)
    if nonzero.any():
        assert np.max(np.abs(g[nonzero] - want_g[nonzero]) / want_g[nonzero]) <= RDF_RTOL


def _check(positions, lattice, r_max, num_bins, groups):
    """get_rdf against the oracle fed the positions the Trajectory stores."""
    trajectory = rb.Trajectory(positions, 1.0)
    r, g = trajectory.get_rdf(lattice, r_max, num_bins, groups)
    want_r, want_g, counts = rdf(trajectory.positions_ts, lattice, r_max, num_bins, groups)
    _compare(r, g, want_r, want_g, counts)
    return r, g, counts


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("kind", ["all", "species", "odd_even_overlap"])
def test_structures_and_groups(structure, kind):
    lattice, num_atoms, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 37, seed=11)
    _check(positions, lattice, _half_width(lattice), 400, _groups(kind, num_atoms, numbers))


@pytest.mark.parametrize("frames", [1, 2, 37, 1000])
def test_frame_counts(frames):
    lattice, num_atoms, numbers = _geometry("LLZO")
    _check(synthetic.make_trajectory("LLZO", frames, seed=frames), lattice, _half_width(lattice), 400,
           _groups("species", num_atoms, numbers))


@pytest.mark.parametrize("num_bins", [1, 7, 400, 4096])
@pytest.mark.parametrize("inside", [False, True])
def test_bin_counts_and_r_max(num_bins, inside):
    lattice, num_atoms, numbers = _geometry("TiO2")
    r_max = 0.55 * _half_width(lattice) if inside else _half_width(lattice)
    _check(synthetic.make_trajectory("TiO2", 37, seed=12), lattice, r_max, num_bins,
           _groups("odd_even_overlap", num_atoms, numbers))


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
def test_sheared_lattice_and_lattice_hops(structure):
    """Hopped frames are not wrapped: the Trajectory wraps them and the oracle reads its positions_ts."""
    lattice, num_atoms, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 40, seed=13, lattice_hops=True)
    assert np.max(np.abs(np.floor(positions))) >= 1
    sheared = _sheared(lattice)
    _check(positions, sheared, _half_width(sheared), 300, _groups("species", num_atoms, numbers))
    _check(positions, lattice, 0.7 * _half_width(lattice), 300, _groups("odd_even_overlap", num_atoms, numbers))


def test_positions_outside_the_unit_cube():
    """The C entry takes any fractional positions (the exact ceil wrap, not the [0, 1] shortcut)."""
    lattice, num_atoms, _ = _geometry("STO")
    positions = synthetic.make_trajectory("STO", 9, seed=14, lattice_hops=True)
    r_max, num_bins = _half_width(lattice), 250
    g = torch.empty((1, 1, num_bins), dtype=torch.float64, device="cuda:0")
    offsets, atoms = np.array([0, num_atoms], dtype=np.int64), np.arange(num_atoms, dtype=np.int64)
    workspace = torch.empty(int(_lib.lib().rn_rdf_workspace_size(1, num_atoms, num_bins)), dtype=torch.uint8,
                            device="cuda:0")
    device_positions = to_cuda(positions)
    status = _lib.lib().rn_rdf(ctypes.c_void_p(device_positions.data_ptr()), 9, num_atoms,
                               ctypes.c_void_p(lattice.ctypes.data), r_max, num_bins, ctypes.c_void_p(offsets.ctypes.data),
                               ctypes.c_void_p(atoms.ctypes.data), 1, ctypes.c_void_p(g.data_ptr()),
                               ctypes.c_void_p(workspace.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream))
    _lib.check(status, "rn_rdf")
    want_r, want_g, counts = rdf(positions, lattice, r_max, num_bins)
    _compare(want_r, g.cpu().numpy(), want_r, want_g, counts)


def test_per_atom_groups_short_trajectory():
    lattice, num_atoms, numbers = _geometry("TiO2")
    _check(synthetic.make_trajectory("TiO2", 3, seed=15), lattice, _half_width(lattice), 60,
           _groups("per_atom", num_atoms, numbers))


def test_llzo_supercell():
    """1536 atoms: groups of more than one tile (the all-atom group and the Li and O species)."""
    lattice, num_atoms, numbers = _geometry("LLZO_2x2x2")
    positions = synthetic.make_trajectory("LLZO_2x2x2", 20, seed=16)
    _check(positions, lattice, 12.5, 1000, _groups("species", num_atoms, numbers) + [range(num_atoms)])


def test_real_llzo_outcar_trajectory(tmp_path):
    path = tmp_path / "OUTCAR_trajectory"
    with gzip.open(os.path.join(GOLDEN, "llzo_outcar_trajectory.txt.gz"), "rb") as fin, open(path, "wb") as fout:
        shutil.copyfileobj(fin, fout)
    _, lattice, _ = rio.read_outcar_positions_ts(path)
    with np.load(os.path.join(GOLDEN, "llzo_outcar_trajectory.npz")) as data:
        positions = data["positions_ts"]
    num_atoms = positions.shape[1]
    _check(positions, lattice, _half_width(lattice), 200, [range(0, 40), range(40, 41), range(41, num_atoms)])
    _check(positions, lattice, _half_width(lattice), 200, None)


def _counts(g, frames, lattice, r_max, groups, num_atoms):
    """The integer counts behind g: exact after rounding, since g carries a relative error of a few 1e-16."""
    _, _, shell = bin_edges(r_max, g.shape[2])
    norms = pair_norms(groups, num_atoms)
    volume, _ = cell_widths(lattice)
    return np.rint(g * (frames * norms)[:, :, None].astype(np.float64) * shell / volume).astype(np.int64)


def test_bit_identity_and_frame_splits():
    lattice, num_atoms, numbers = _geometry("LLZO")
    positions = synthetic.make_trajectory("LLZO", 301, seed=17, lattice_hops=True)
    species = _groups("species", num_atoms, numbers)
    r_max, num_bins = _half_width(lattice), 400
    host = rb.Trajectory(positions, 1.0)
    device = rb.Trajectory(to_cuda(host.positions_ts), 1.0)
    assert not host.is_device_resident and device.is_device_resident
    first = host.get_rdf_device(lattice, r_max, num_bins, species)
    for again in (device.get_rdf_device(lattice, r_max, num_bins, species),
                  host.get_rdf_device(lattice, r_max, num_bins, species)):
        assert torch.equal(first[0], again[0]) and torch.equal(first[1], again[1])
    g = first[1].cpu().numpy()
    alone = device.get_rdf(lattice, r_max, num_bins, [species[1], species[3]])[1]
    assert np.array_equal(alone[0, 1], g[1, 3]) and np.array_equal(alone[1, 1], g[3, 3])
    assert np.array_equal(alone[0, 0], g[1, 1])
    counts = _counts(g, 301, lattice, r_max, species, num_atoms)
    wrapped = host.positions_ts
    parts = [rb.Trajectory(wrapped[a:b], 1.0).get_rdf(lattice, r_max, num_bins, species)[1] for a, b in
             ((0, 120), (120, 121), (121, 301))]
    split = sum(_counts(part, b - a, lattice, r_max, species, num_atoms) for part, (a, b) in
                zip(parts, ((0, 120), (120, 121), (121, 301))))
    assert np.array_equal(split, counts)


def test_species_sum_rule():
    lattice, num_atoms, numbers = _geometry("LLZO")
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("LLZO", 2000, seed=18)), 1.0)
    species = _groups("species", num_atoms, numbers)
    r_max, num_bins = _half_width(lattice), 400
    _, g = trajectory.get_rdf(lattice, r_max, num_bins, species)
    _, g_all = trajectory.get_rdf(lattice, r_max, num_bins)
    counts = _counts(g, 2000, lattice, r_max, species, num_atoms)
    all_counts = _counts(g_all, 2000, lattice, r_max, None, num_atoms)
    assert np.array_equal(counts.sum(axis=(0, 1)), all_counts[0, 0])
    assert all_counts.sum() > 10**7


def _launches(fn):
    fn()
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def test_launch_count():
    counts = []
    for structure in ("TiO2", "LLZO"):
        lattice, num_atoms, numbers = _geometry(structure)
        for frames in (100, 20_000):
            trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory(structure, frames, seed=19)), 1.0)
            r_max = _half_width(lattice)
            counts.append(_launches(lambda t=trajectory, l=lattice, r=r_max: t.get_rdf_device(l, r, 100)))
            groups = [range(0, 10), range(10, 40), range(40, num_atoms), [0, 50]]
            counts.append(_launches(lambda t=trajectory, l=lattice, r=r_max, g=groups: t.get_rdf_device(l, r, 100, g)))
    assert counts == [2] * 8


def test_c_entry_errors():
    frames, num_atoms, num_bins = 30, 6, 16
    lib = _lib.lib()
    rng = np.random.default_rng(10)
    positions = to_cuda(rng.uniform(0, 1, (frames, num_atoms, 3)))
    out = torch.empty((2, 2, num_bins), dtype=torch.float64, device="cuda:0")
    workspace = torch.empty(int(lib.rn_rdf_workspace_size(2, 5, num_bins)), dtype=torch.uint8, device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.diag([5.0, 6.0, 7.0])
    offsets = np.array([0, 2, 5], dtype=np.int64)
    atoms = np.array([0, 1, 2, 3, 5], dtype=np.int64)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731

    def call(pos=ctypes.c_void_p(positions.data_ptr()), s=frames, n=num_atoms, lat=ptr(lattice), r_max=2.5,
             bins=num_bins, off=ptr(offsets), at=ptr(atoms), groups=2, dst=ctypes.c_void_p(out.data_ptr()),
             ws=ctypes.c_void_p(workspace.data_ptr())):
        return lib.rn_rdf(pos, s, n, lat, r_max, bins, off, at, groups, dst, ws, stream)

    assert call(pos=None) == -1
    assert call(lat=None) == -1
    assert call(off=None) == -1
    assert call(at=None) == -1
    assert call(dst=None) == -1
    assert call(ws=None) == -1
    assert call(s=0) == -1
    assert call(n=0) == -1
    assert call(groups=0) == -1
    assert call(bins=0) == -1
    assert call(bins=4097) == -1
    assert call(lat=ptr(np.diag([5.0, np.inf, 7.0]))) == -1
    assert call(lat=ptr(np.array([[5.0, 0, 0], [10.0, 0, 0], [0, 0, 7.0]]))) == -1  # zero volume
    for bad in (0.0, -1.0, float("nan"), 2.5 * (1 + 1e-9)):
        assert call(r_max=bad) == -1
    bad_atoms = atoms.copy()
    bad_atoms[4] = num_atoms
    assert call(at=ptr(bad_atoms)) == -1
    bad_atoms[4] = -1
    assert call(at=ptr(bad_atoms)) == -1
    assert call(off=ptr(np.array([0, 2, 2], dtype=np.int64))) == -1  # empty group
    assert call() == 0
    torch.cuda.synchronize()
    _, want = rb.Trajectory(positions, 1.0).get_rdf(lattice, 2.5, num_bins, [[0, 1], [2, 3, 5]])
    assert np.array_equal(out.cpu().numpy(), want)
