"""Self Van Hove correlation (``Trajectory.get_van_hove``) on the GPU: G_s within 1e-13 relative of the oracle and
exactly 0 where the oracle's count is 0 (with counts below 1e10 one count more or less would move G_s by more than
1e-10, so this pins the integer counts), the moments within 1e-12 relative, over structures, group layouts, frame
counts, lags 0, 1 and S - 1, sheared lattices, lattice hops, a diffusing species, positions outside the unit cube and
the real LLZO OUTCAR trajectory; m2 against get_msd; bit-identity across input forms, repeated calls, group sets and
forced chunk sizes; the launch count and the C entry's errors."""
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
from msd_oracle import energies
from van_hove_oracle import van_hove

pytestmark = pytest.mark.gpu

G_S_RTOL = 1e-13
MOMENT_RTOL = 1e-12
MSD_RTOL = 1e-10  # the bound of get_msd: |error| <= MSD_RTOL * 2 E_g / ((S - m) |g|)


def _geometry(name):
    geom = synthetic.load_structure(name)
    return geom["lattice"], geom["positions"].shape[0], geom["atomic_numbers"]


def _sheared(lattice):
    """The lattice with off-diagonal entries of 1-3 Å: every entry of the lattice product is used."""
    return lattice + np.array([[0.0, 1.0, 2.5], [1.5, 0.0, 3.0], [2.0, 1.25, 0.0]])


def _diffusing(structure, frames, seed, species_z, step=0.3):
    """A random walk (Å per frame and component) added to one species before wrapping: its paths span many cells."""
    lattice, _, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, frames, seed=seed)
    walk = np.cumsum(np.random.default_rng(seed).normal(scale=step, size=positions.shape), axis=0)
    walk[:, numbers != species_z] = 0.0
    moved = positions + walk @ np.linalg.inv(lattice)
    return moved - np.floor(moved)


def _groups(kind, num_atoms, numbers):
    if kind == "all":
        return None
    if kind == "species":
        return [np.flatnonzero(numbers == z) for z in np.unique(numbers)]
    if kind == "odd_even_overlap":  # odd and even atoms, an overlapping range and a one-atom group
        return [list(range(1, num_atoms, 2)), list(range(0, num_atoms, 2)), list(range(3, 40)), [num_atoms - 1]]
    if kind == "per_atom":
        return [[i] for i in range(num_atoms)]
    raise AssertionError(kind)


def _compare(got, want):
    lag_times, r, g_s, moments = got
    want_r, want_g, want_m, counts = want
    assert np.array_equal(r, want_r)
    assert g_s.shape == want_g.shape and moments.shape == want_m.shape
    assert np.all(g_s[counts == 0] == 0.0)
    nonzero = counts > 0
    assert np.all(g_s[nonzero] > 0)
    if nonzero.any():
        assert np.max(np.abs(g_s[nonzero] - want_g[nonzero]) / want_g[nonzero]) <= G_S_RTOL
    assert np.all(moments[want_m == 0] == 0.0)
    pos = want_m != 0
    assert np.max(np.abs(moments[pos] - want_m[pos]) / want_m[pos], initial=0.0) <= MOMENT_RTOL


def _check(positions, lattice, lags, r_max, num_bins, groups, timestep=1.0):
    """get_van_hove against the oracle fed the positions the Trajectory stores."""
    trajectory = rb.Trajectory(positions, timestep)
    got = trajectory.get_van_hove(lattice, lags, r_max, num_bins, groups)
    assert np.array_equal(got[0], np.asarray(lags, dtype=np.float64) * timestep)
    want = van_hove(trajectory.positions_ts, lattice, lags, r_max, num_bins, groups)
    _compare(got, want)
    return got, want


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("kind", ["all", "species", "odd_even_overlap", "per_atom"])
def test_structures_and_groups(structure, kind):
    lattice, num_atoms, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 257, seed=31)
    _check(positions, lattice, [0, 1, 2, 9, 100, 256], 1.5, 300, _groups(kind, num_atoms, numbers))


@pytest.mark.parametrize("frames", [2, 255, 256, 257, 1000])
def test_frame_counts_and_lags(frames):
    lattice, num_atoms, numbers = _geometry("LLZO")
    lags = sorted({0, 1, frames // 3, frames - 1})
    _check(synthetic.make_trajectory("LLZO", frames, seed=frames), lattice, lags, 2.0, 400,
           _groups("species", num_atoms, numbers))


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
def test_sheared_lattice_and_lattice_hops(structure):
    lattice, num_atoms, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 300, seed=32, lattice_hops=True)
    _check(positions, _sheared(lattice), [0, 1, 7, 299], 1.0, 4096, _groups("species", num_atoms, numbers), 0.5)
    _check(positions, lattice, [1, 3, 50], 0.3, 1, _groups("odd_even_overlap", num_atoms, numbers))


@pytest.mark.parametrize("structure, species", [("LLZO", 3), ("TiO2", 22)])
def test_diffusing_species(structure, species):
    """The walkers cross many cells: r_max beyond the cell, and at least a quarter of the long-lag displacements
    of the walkers land beyond the cell width."""
    lattice, num_atoms, numbers = _geometry(structure)
    positions = _diffusing(structure, 3000, 33, species)
    groups = _groups("species", num_atoms, numbers)
    lags = [1, 10, 100, 1000, 2999]
    (_, _, _, moments), _ = _check(positions, _sheared(lattice), lags, 40.0, 500, groups)
    walkers = list(np.unique(numbers)).index(species)
    assert moments[walkers, 3, 0] > 100.0


def test_positions_outside_the_unit_cube():
    """The C entry takes any fractional positions: the oracle is fed the same unwrapped ones."""
    lattice, num_atoms, _ = _geometry("STO")
    positions = synthetic.make_trajectory("STO", 40, seed=34, lattice_hops=True) + np.array([3.0, -2.0, 7.0])
    assert np.max(np.abs(np.floor(positions))) >= 1
    lags = np.array([0, 1, 5, 39], dtype=np.int64)
    num_bins, r_max = 250, 2.0
    g_s = torch.empty((1, 4, num_bins), dtype=torch.float64, device="cuda:0")
    moments = torch.empty((1, 4, 2), dtype=torch.float64, device="cuda:0")
    offsets, atoms = np.array([0, num_atoms], dtype=np.int64), np.arange(num_atoms, dtype=np.int64)
    lib = _lib.lib()
    workspace = torch.empty(int(lib.rn_van_hove_workspace_size(40, num_atoms, 1, 4, num_bins)), dtype=torch.uint8,
                            device="cuda:0")
    device_positions = to_cuda(positions)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    status = lib.rn_van_hove(ctypes.c_void_p(device_positions.data_ptr()), 40, num_atoms, ptr(lattice), ptr(lags), 4,
                             r_max, num_bins, ptr(offsets), ptr(atoms), 1, ctypes.c_void_p(g_s.data_ptr()),
                             ctypes.c_void_p(moments.data_ptr()), ctypes.c_void_p(workspace.data_ptr()),
                             ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream))
    _lib.check(status, "rn_van_hove")
    want = van_hove(positions, lattice, lags, r_max, num_bins)
    _compare((None, want[0], g_s.cpu().numpy(), moments.cpu().numpy()), want)


def test_real_llzo_outcar_trajectory(tmp_path):
    path = tmp_path / "OUTCAR_trajectory"
    with gzip.open(os.path.join(GOLDEN, "llzo_outcar_trajectory.txt.gz"), "rb") as fin, open(path, "wb") as fout:
        shutil.copyfileobj(fin, fout)
    _, lattice, _ = rio.read_outcar_positions_ts(path)
    with np.load(os.path.join(GOLDEN, "llzo_outcar_trajectory.npz")) as data:
        positions = data["positions_ts"]
    frames, num_atoms = positions.shape[:2]
    lags = [0, 1, frames // 2, frames - 1]
    _check(positions, lattice, lags, 3.0, 200, [range(0, 40), range(40, 41), range(41, num_atoms)])
    _check(positions, lattice, lags, 3.0, 200, None)


def test_m2_against_get_msd():
    lattice, num_atoms, numbers = _geometry("LLZO")
    trajectory = rb.Trajectory(_diffusing("LLZO", 2000, 35, 3), 1.0)
    groups = _groups("species", num_atoms, numbers)
    lags = np.array([0, 1, 2, 30, 999, 1999])
    _, _, _, moments = trajectory.get_van_hove(_sheared(lattice), lags, 5.0, 100, groups)
    _, msd = trajectory.get_msd(_sheared(lattice), groups)
    sizes = np.array([len(g) for g in groups], dtype=np.float64)
    scale = 2 * energies(trajectory.positions_ts, _sheared(lattice), groups)[:, None] / ((2000 - lags) * sizes[:, None])
    assert np.all(np.abs(moments[..., 0] - msd[:, lags]) <= MSD_RTOL * scale)


@pytest.fixture(name="chunk")
def fixture_chunk():
    lib = _lib.lib()
    yield lib.rn_debug_set_van_hove_chunk
    lib.rn_debug_set_van_hove_chunk(0)


def test_bit_identity_across_inputs_calls_group_sets_and_chunks(chunk):
    """Groups of 56, 24, 16 and 96 atoms (2, 1, 1 and 3 member tiles of 32) and all 192 (6 tiles); chunks of one tile
    up to all of them."""
    lattice, num_atoms, numbers = _geometry("LLZO")
    positions = _diffusing("LLZO", 3001, 36, 3)
    groups = _groups("species", num_atoms, numbers) + [range(num_atoms)]
    args = (_sheared(lattice), [0, 1, 2, 100, 2048, 3000], 6.0, 600)
    host = rb.Trajectory(positions, 1.0)
    device = rb.Trajectory(to_cuda(host.positions_ts), 1.0)
    assert not host.is_device_resident and device.is_device_resident
    first = host.get_van_hove_device(*args, groups)
    runs = [device.get_van_hove_device(*args, groups), host.get_van_hove_device(*args, groups)]
    for memberships in (1, 33, 64, 100):
        chunk(memberships)
        runs.append(device.get_van_hove_device(*args, groups))
    chunk(0)
    for again in runs:
        for a, b in zip(first, again):
            assert torch.equal(a, b)
    alone = device.get_van_hove_device(*args, [groups[2], groups[0]])
    assert torch.equal(alone[2][0], first[2][2]) and torch.equal(alone[2][1], first[2][0])
    assert torch.equal(alone[3][0], first[3][2]) and torch.equal(alone[3][1], first[3][0])


def _launches(fn):
    fn()
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def test_launch_count(chunk):
    """4 launches per membership chunk + 1: one chunk by default; with chunks of one tile, one per member tile."""
    lattice, num_atoms, numbers = _geometry("LLZO")
    trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory("LLZO", 5000, seed=37)), 1.0)
    species = _groups("species", num_atoms, numbers)  # 2 + 1 + 1 + 3 member tiles
    for lags, num_bins in (([1], 10), (np.arange(0, 5000, 50), 4096)):
        assert _launches(lambda l=lags, b=num_bins: trajectory.get_van_hove_device(lattice, l, 3.0, b, species)) == 5
        assert _launches(lambda l=lags, b=num_bins: trajectory.get_van_hove_device(lattice, l, 3.0, b)) == 5
        chunk(1)
        assert _launches(lambda l=lags, b=num_bins: trajectory.get_van_hove_device(lattice, l, 3.0, b, species)) == 29
        assert _launches(lambda l=lags, b=num_bins: trajectory.get_van_hove_device(lattice, l, 3.0, b)) == 25
        chunk(0)


def test_c_entry_errors():
    frames, num_atoms, num_bins = 30, 6, 16
    lib = _lib.lib()
    rng = np.random.default_rng(38)
    positions = to_cuda(rng.uniform(0, 1, (frames, num_atoms, 3)))
    g_s = torch.empty((2, 3, num_bins), dtype=torch.float64, device="cuda:0")
    moments = torch.empty((2, 3, 2), dtype=torch.float64, device="cuda:0")
    workspace = torch.empty(int(lib.rn_van_hove_workspace_size(frames, 5, 2, 3, num_bins)), dtype=torch.uint8,
                            device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.diag([5.0, 6.0, 7.0])
    lags = np.array([0, 4, 29], dtype=np.int64)
    offsets = np.array([0, 2, 5], dtype=np.int64)
    atoms = np.array([0, 1, 2, 3, 5], dtype=np.int64)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731

    def call(pos=ctypes.c_void_p(positions.data_ptr()), s=frames, n=num_atoms, lat=ptr(lattice), lg=ptr(lags), t=3,
             r_max=2.5, bins=num_bins, off=ptr(offsets), at=ptr(atoms), groups=2, dst=ctypes.c_void_p(g_s.data_ptr()),
             mom=ctypes.c_void_p(moments.data_ptr()), ws=ctypes.c_void_p(workspace.data_ptr())):
        return lib.rn_van_hove(pos, s, n, lat, lg, t, r_max, bins, off, at, groups, dst, mom, ws, stream)

    for name in ("pos", "lat", "lg", "off", "at", "dst", "mom", "ws"):
        assert call(**{name: None}) == -1
    assert call(s=1) == -1
    assert call(n=0) == -1
    assert call(t=0) == -1
    assert call(groups=0) == -1
    assert call(bins=0) == -1
    assert call(bins=4097) == -1
    for bad in ([0, 4, 30], [-1, 4, 29], [0, 4, 4], [4, 0, 29]):
        assert call(lg=ptr(np.array(bad, dtype=np.int64))) == -1
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        assert call(r_max=bad) == -1
    assert call(lat=ptr(np.diag([5.0, np.inf, 7.0]))) == -1
    assert call(lat=ptr(np.array([[5.0, 0, 0], [10.0, 0, 0], [0, 0, 7.0]]))) == -1  # zero volume
    bad_atoms = atoms.copy()
    bad_atoms[4] = num_atoms
    assert call(at=ptr(bad_atoms)) == -1
    bad_atoms[4] = -1
    assert call(at=ptr(bad_atoms)) == -1
    bad_atoms[4] = 2
    assert call(at=ptr(bad_atoms)) == -1  # group 1 repeats atom 2
    assert call(off=ptr(np.array([0, 2, 2], dtype=np.int64))) == -1  # empty group
    assert call() == 0
    torch.cuda.synchronize()
    _, _, want_g, want_m = rb.Trajectory(positions, 1.0).get_van_hove(lattice, lags, 2.5, num_bins, [[0, 1], [2, 3, 5]])
    assert np.array_equal(g_s.cpu().numpy(), want_g) and np.array_equal(moments.cpu().numpy(), want_m)
