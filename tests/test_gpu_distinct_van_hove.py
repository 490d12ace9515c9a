"""Distinct Van Hove correlation (``Trajectory.get_distinct_van_hove``) on the GPU: every element within 1e-13 relative
of the oracle and exactly 0 where the oracle's count is 0 (with counts below 1e10 one count more or less would move
g_d by more than 1e-10, so this pins the integer counts), over structures, group layouts, frame counts with lags 0, 1
and S - 1, sheared lattices at r_max = w_min/2, positions outside the unit cube and the real LLZO OUTCAR trajectory;
lag-0 rows bit-identical to get_rdf; time reversal bit for bit; a frozen trajectory against get_rdf at every lag;
bit-identity across input forms, repeated calls and group sets; the launch count and the C entry's errors."""
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

from distinct_van_hove_oracle import distinct_van_hove
from gpu_helpers import to_cuda
from helpers import GOLDEN
from rdf_oracle import cell_widths

pytestmark = pytest.mark.gpu

G_D_RTOL = 1e-13
FROZEN_RTOL = 2e-15  # (S - t) n_ab rounds differently from S n_ab only in the last bits


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
    if kind == "overlapping":  # sizes 7, 10, 1 and an overlap of the first two; the one-atom group has n_aa = 0
        return [list(range(0, 7)), list(range(3, 13)), [num_atoms - 1], list(range(num_atoms - 1, 20, -9))]
    raise AssertionError(kind)


def _compare(g_d, want_g, counts):
    assert g_d.shape == want_g.shape
    assert np.all(g_d[counts == 0] == 0.0)
    nonzero = counts > 0
    assert np.all(g_d[nonzero] > 0)
    if nonzero.any():
        assert np.max(np.abs(g_d[nonzero] - want_g[nonzero]) / want_g[nonzero]) <= G_D_RTOL


def _check(positions, lattice, lags, r_max, num_bins, groups, timestep=1.0):
    """get_distinct_van_hove against the oracle fed the positions the Trajectory stores; lag-0 rows against get_rdf
    bit for bit."""
    trajectory = rb.Trajectory(positions, timestep)
    lag_times, r, g_d = trajectory.get_distinct_van_hove(lattice, lags, r_max, num_bins, groups)
    assert np.array_equal(lag_times, np.asarray(lags, dtype=np.float64) * timestep)
    want_r, want_g, counts = distinct_van_hove(trajectory.positions_ts, lattice, lags, r_max, num_bins, groups)
    assert np.array_equal(r, want_r)
    _compare(g_d, want_g, counts)
    if lags[0] == 0:
        rdf_r, rdf = trajectory.get_rdf(lattice, r_max, num_bins, groups)
        assert np.array_equal(rdf_r, r)
        assert np.array_equal(g_d[:, :, 0], rdf)
    return g_d, counts


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
@pytest.mark.parametrize("kind", ["all", "species", "overlapping"])
def test_structures_and_groups(structure, kind):
    lattice, num_atoms, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 37, seed=41)
    _check(positions, lattice, [0, 1, 5, 36], _half_width(lattice), 400, _groups(kind, num_atoms, numbers))


def test_per_atom_groups_on_a_subset():
    lattice, _, _ = _geometry("TiO2")
    positions = synthetic.make_trajectory("TiO2", 6, seed=42)
    _check(positions, lattice, [0, 1, 5], _half_width(lattice), 60, [[i] for i in range(0, 36, 3)])


@pytest.mark.parametrize("frames", [1, 2, 255, 256, 257, 1000])
def test_frame_counts_and_lags(frames):
    lattice, num_atoms, numbers = _geometry("LLZO")
    lags = sorted({0, 1, frames - 1} & set(range(frames)))
    _check(synthetic.make_trajectory("LLZO", frames, seed=frames), lattice, lags, _half_width(lattice), 400,
           _groups("species", num_atoms, numbers))


@pytest.mark.parametrize("structure", ["TiO2", "STO", "LLZO"])
def test_sheared_lattice_at_half_width(structure):
    """Hopped frames are not wrapped: the Trajectory wraps them and the oracle reads its positions_ts."""
    lattice, num_atoms, numbers = _geometry(structure)
    positions = synthetic.make_trajectory(structure, 40, seed=43, lattice_hops=True)
    sheared = _sheared(lattice)
    _check(positions, sheared, [0, 1, 7, 39], _half_width(sheared), 300, _groups("species", num_atoms, numbers), 0.5)


def test_positions_outside_the_unit_cube():
    """The C entry takes any fractional positions (the exact ceil wrap, not the [0, 1] shortcut)."""
    lattice, num_atoms, _ = _geometry("STO")
    positions = synthetic.make_trajectory("STO", 12, seed=44, lattice_hops=True) + np.array([3.0, -2.0, 7.0])
    assert np.max(np.abs(np.floor(positions))) >= 1
    lags = np.array([0, 1, 5, 11], dtype=np.int64)
    r_max, num_bins = _half_width(lattice), 250
    groups = [list(range(0, 20)), list(range(10, num_atoms))]
    offsets = np.array([0, 20, 20 + num_atoms - 10], dtype=np.int64)
    atoms = np.concatenate([np.arange(0, 20), np.arange(10, num_atoms)]).astype(np.int64)
    g_d = torch.empty((2, 2, 4, num_bins), dtype=torch.float64, device="cuda:0")
    lib = _lib.lib()
    workspace = torch.empty(int(lib.rn_distinct_van_hove_workspace_size(len(atoms), 2, 4, num_bins)),
                            dtype=torch.uint8, device="cuda:0")
    device_positions = to_cuda(positions)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    status = lib.rn_distinct_van_hove(ctypes.c_void_p(device_positions.data_ptr()), 12, num_atoms, ptr(lattice),
                                      ptr(lags), 4, r_max, num_bins, ptr(offsets), ptr(atoms), 2,
                                      ctypes.c_void_p(g_d.data_ptr()), ctypes.c_void_p(workspace.data_ptr()),
                                      ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream))
    _lib.check(status, "rn_distinct_van_hove")
    _, want_g, counts = distinct_van_hove(positions, lattice, lags, r_max, num_bins, groups)
    _compare(g_d.cpu().numpy(), want_g, counts)


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


def test_time_reversal_bit_for_bit():
    lattice, num_atoms, numbers = _geometry("LLZO")
    positions = synthetic.make_trajectory("LLZO", 301, seed=45)
    groups = _groups("species", num_atoms, numbers) + [range(num_atoms)]
    args = (lattice, [0, 1, 2, 50, 300], _half_width(lattice), 400, groups)
    forward = rb.Trajectory(positions, 1.0)
    backward = rb.Trajectory(np.ascontiguousarray(forward.positions_ts[::-1]), 1.0)
    _, _, g_f = forward.get_distinct_van_hove(*args)
    _, _, g_b = backward.get_distinct_van_hove(*args)
    assert np.array_equal(g_b, g_f.transpose(1, 0, 2, 3))
    assert not np.array_equal(g_f[0, 1, 1:], g_f[1, 0, 1:])


def test_frozen_trajectory_is_the_rdf_at_every_lag():
    lattice, num_atoms, numbers = _geometry("LLZO")
    positions = np.repeat(synthetic.make_trajectory("LLZO", 1, seed=46), 200, axis=0)
    trajectory = rb.Trajectory(to_cuda(positions), 1.0)
    groups = _groups("overlapping", num_atoms, numbers)
    r_max = _half_width(lattice)
    _, _, g_d = trajectory.get_distinct_van_hove(lattice, [0, 1, 7, 150, 199], r_max, 500, groups)
    _, rdf = trajectory.get_rdf(lattice, r_max, 500, groups)
    assert np.any(rdf > 0)
    for ti in range(5):
        assert np.all(g_d[:, :, ti][rdf == 0] == 0)
        assert np.all(np.abs(g_d[:, :, ti] - rdf) <= FROZEN_RTOL * rdf)


def test_bit_identity_across_inputs_calls_and_group_sets():
    """LLZO_2x2x2 (1536 atoms): the all-atom group and the Li and O species span several tiles of 256."""
    lattice, num_atoms, numbers = _geometry("LLZO_2x2x2")
    positions = synthetic.make_trajectory("LLZO_2x2x2", 12, seed=47, lattice_hops=True)
    species = _groups("species", num_atoms, numbers)
    groups = species + [range(num_atoms)]
    args = (lattice, [0, 1, 11], 12.5, 1000)
    host = rb.Trajectory(positions, 1.0)
    device = rb.Trajectory(to_cuda(host.positions_ts), 1.0)
    assert not host.is_device_resident and device.is_device_resident
    first = host.get_distinct_van_hove_device(*args, groups)
    for again in (device.get_distinct_van_hove_device(*args, groups), host.get_distinct_van_hove_device(*args, groups)):
        for a, b in zip(first, again):
            assert torch.equal(a, b)
    g = first[2]
    alone = device.get_distinct_van_hove_device(*args, [groups[3], groups[1]])[2]
    assert torch.equal(alone[0, 1], g[3, 1]) and torch.equal(alone[1, 0], g[1, 3])
    assert torch.equal(alone[0, 0], g[3, 3]) and torch.equal(alone[1, 1], g[1, 1])
    assert torch.count_nonzero(g[3, 1]) > 0


def _launches(fn):
    fn()
    torch.cuda.synchronize()
    before = _lib.launch_count()
    fn()
    return _lib.launch_count() - before


def test_launch_count():
    counts = []
    for structure in ("TiO2", "LLZO"):
        lattice, num_atoms, _ = _geometry(structure)
        r_max = _half_width(lattice)
        for frames in (100, 20_000):
            trajectory = rb.Trajectory(to_cuda(synthetic.make_trajectory(structure, frames, seed=48)), 1.0)
            for lags in ([0], np.arange(0, frames, frames // 10)):
                counts.append(_launches(lambda t=trajectory, l=lattice, r=r_max, g=lags:
                                        t.get_distinct_van_hove_device(l, g, r, 100)))
            groups = [range(0, 10), range(10, 40), range(40, num_atoms), [0, 50]]
            counts.append(_launches(lambda t=trajectory, l=lattice, r=r_max, g=groups:
                                    t.get_distinct_van_hove_device(l, [1, 5], r, 100, g)))
    assert counts == [2] * 12


def test_c_entry_errors():
    frames, num_atoms, num_bins = 30, 6, 16
    lib = _lib.lib()
    rng = np.random.default_rng(49)
    positions = to_cuda(rng.uniform(0, 1, (frames, num_atoms, 3)))
    out = torch.empty((2, 2, 3, num_bins), dtype=torch.float64, device="cuda:0")
    workspace = torch.empty(int(lib.rn_distinct_van_hove_workspace_size(5, 2, 3, num_bins)), dtype=torch.uint8,
                            device="cuda:0")
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    lattice = np.diag([5.0, 6.0, 7.0])
    lags = np.array([0, 4, 29], dtype=np.int64)
    offsets = np.array([0, 2, 5], dtype=np.int64)
    atoms = np.array([0, 1, 2, 3, 5], dtype=np.int64)
    ptr = lambda a: ctypes.c_void_p(a.ctypes.data)  # noqa: E731

    def call(pos=ctypes.c_void_p(positions.data_ptr()), s=frames, n=num_atoms, lat=ptr(lattice), lg=ptr(lags), t=3,
             r_max=2.5, bins=num_bins, off=ptr(offsets), at=ptr(atoms), groups=2, dst=ctypes.c_void_p(out.data_ptr()),
             ws=ctypes.c_void_p(workspace.data_ptr())):
        return lib.rn_distinct_van_hove(pos, s, n, lat, lg, t, r_max, bins, off, at, groups, dst, ws, stream)

    for name in ("pos", "lat", "lg", "off", "at", "dst", "ws"):
        assert call(**{name: None}) == -1
    assert call(s=0) == -1
    assert call(n=0) == -1
    assert call(t=0) == -1
    assert call(groups=0) == -1
    assert call(bins=0) == -1
    assert call(bins=4097) == -1
    for bad in ([0, 4, 30], [-1, 4, 29], [0, 4, 4], [4, 0, 29]):
        assert call(lg=ptr(np.array(bad, dtype=np.int64))) == -1
    for bad in (0.0, -1.0, float("nan"), 2.5 * (1 + 1e-9)):
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
    _, _, want = rb.Trajectory(positions, 1.0).get_distinct_van_hove(lattice, lags, 2.5, num_bins, [[0, 1], [2, 3, 5]])
    assert np.array_equal(out.cpu().numpy(), want)
