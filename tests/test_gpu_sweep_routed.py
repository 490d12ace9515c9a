"""Routed mask sweeps (``rn_calc_polarizabilities_sweep_routed``): G masked copies of a model evaluated on
one rank's block of a frame-sharded trajectory, every row stored locally and to the ranks whose spectrum
stage consumes it.  The ranks are emulated on one GPU: each (rank, mask) pair has its own NaN-filled full
series buffer and the blocks of all ranks are evaluated one after the other, so that afterwards every buffer
can be compared with what the routing rule (owner(n) and owner(n - 1)) puts there."""
import ctypes

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib, synthetic
from ramannoodle_b200.distributed import shard_bounds
from ramannoodle_b200.pmodel import calc_polarizabilities_sweep_routed

from gpu_helpers import ALPHA_RTOL, to_cuda
from helpers import oracle_model, rel_err

pytestmark = pytest.mark.gpu


def _masked_copies(model, count, seed):
    rng = np.random.default_rng(seed)
    num_dofs = model.state.num_dofs
    return [model.get_masked_model(np.flatnonzero(rng.random(num_dofs) < 0.3)) for _ in range(count)]


def _dense_split(frames):
    """Whether the single-GPU dense sweep balances (frame tile, DOF tile) units over the SMs for a block of
    ``frames`` (it then finishes shared tiles with atomic adds in no fixed order; the routed sweep never
    does, its peers need finished rows), rn_dense_sweep.cu."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = -(-frames // 128)
    return -(-tiles // sms) * sms > 1.04 * tiles


def _emulate(models, positions, world, period, width, host=False, chunk_frames=0,
             route=calc_polarizabilities_sweep_routed):
    """Evaluates every rank's block of ``positions`` with the routed sweep (or ``route``, called with its
    arguments); returns the series buffers ``[rank][mask]`` as (S,9) arrays."""
    frames = positions.shape[0]
    count = len(models)
    buffers = [[torch.full((frames * 9,), float("nan"), dtype=torch.float64, device="cuda:0") for _ in range(count)]
               for _ in range(world)]
    for rank in range(world):
        start, stop = shard_bounds(frames, world, rank)
        block = positions[start:stop]
        block = np.ascontiguousarray(block) if host else to_cuda(block)
        local = [buffers[rank][g].data_ptr() + start * 72 for g in range(count)]
        peers = [[0 if r == rank else buffers[r][g].data_ptr() for r in range(world)] for g in range(count)]
        route(models, block, local, peers, start, period, width, chunk_frames=chunk_frames)
    torch.cuda.synchronize()
    return [[b.cpu().numpy().reshape(frames, 9) for b in row] for row in buffers]


def _check_routing(buffers, world, period, width, exact):
    """Rank r's buffer of mask g holds its own block and the rows routed to it, bit-identical to the rows the
    evaluating rank wrote locally; ``exact[g]``: NaN everywhere else (fused kernels store row by row; a model
    evaluated on its own keeps the single-model routing, whose bulk tile stores and block copies may also
    deliver rows no stage reads)."""
    frames = buffers[0][0].shape[0]
    n = np.arange(frames)
    owner = (n % period) // width
    owner_prev = np.where(n >= 1, ((n - 1) % period) // width, -1)
    for g in range(len(buffers[0])):
        full = np.concatenate([buffers[r][g][slice(*shard_bounds(frames, world, r))] for r in range(world)])
        assert not np.isnan(full).any()
        for rank in range(world):
            start, stop = shard_bounds(frames, world, rank)
            want = (owner == rank) | (owner_prev == rank) | ((n >= start) & (n < stop))
            got = buffers[rank][g]
            present = ~np.isnan(got).any(axis=1)
            assert present[want].all(), (g, rank)
            assert np.array_equal(got[present], full[present]), (g, rank)
            if exact[g]:
                assert np.array_equal(present, want), (g, rank)
                assert np.isnan(got[~want]).all()
    return [np.concatenate([buffers[r][g][slice(*shard_bounds(frames, world, r))] for r in range(world)])
            for g in range(len(buffers[0]))]


def _check_against_sweep_and_oracle(models, positions, world, series, dense=False):
    frames = positions.shape[0]
    for rank in range(world):
        start, stop = shard_bounds(frames, world, rank)
        want = rb.calc_polarizabilities_sweep(models, to_cuda(positions[start:stop])).cpu().numpy().reshape(
            len(models), -1, 9)
        for g, model in enumerate(models):
            if dense and _dense_split(stop - start):
                assert rel_err(series[g][start:stop], want[g]) <= 1e-13
            else:
                assert np.array_equal(series[g][start:stop], want[g]), (rank, g)
    sel = np.unique(np.r_[0:64, frames // 2 - 32:frames // 2 + 32, frames - 64:frames])
    for g, model in enumerate(models):
        oracle = ora.calc_polarizabilities(oracle_model(model.state), positions[sel])
        assert rel_err(series[g][sel].reshape(-1, 3, 3), oracle) <= ALPHA_RTOL


# 2 ranks: period 128, width 64; 4 ranks: period 256, width 64; 3 ranks of which only 2 share the transform.
# Frame counts leave blocks that start off the 8-frame tile and end in ragged tails.
ROUTES = [(2, 128, 64), (4, 256, 64), (3, 128, 64)]


@pytest.mark.parametrize("world,period,width", ROUTES)
@pytest.mark.parametrize("count", [1, 3, 4, 5])
def test_art_sweep_routed(world, period, width, count):
    """ARTModel masks: runs of three or four share affine_sweep_kernel (routed epilogue); five masks split
    into four + one, and a single mask takes the single-model routed path."""
    state = synthetic.make_model("LLZO", "art")
    models = _masked_copies(rb.ARTModel(state), count, seed=count)
    positions = synthetic.make_trajectory("LLZO", 2051, seed=7, lattice_hops=True)
    buffers = _emulate(models, positions, world, period, width)
    exact = [count >= 3 and g < 4 for g in range(count)]
    series = _check_routing(buffers, world, period, width, exact)
    _check_against_sweep_and_oracle(models, positions, world, series)


def _linear_and_cubic(structure, cubic_dofs, linear_dofs):
    """A model with cubic spline DOFs and single-piece linear DOFs (the latter collapse into the affine term)."""
    state = synthetic.make_model(structure, "cubic", num_dofs=cubic_dofs, seed=5)
    art = synthetic.make_model(structure, "art", num_dofs=cubic_dofs + linear_dofs, seed=6)
    for j in range(cubic_dofs, cubic_dofs + linear_dofs):
        state.add_dof(art.basis_vectors[j], *art.splines[j])
    return state


@pytest.mark.parametrize("structure,kind,count,world,period,width,frames", [
    ("STO", "cubic", 2, 2, 128, 64, 2 * 18944 - 5),   # whole-tile schedule on 148 SMs
    ("STO", "cubic", 4, 4, 256, 64, 75703),
    ("TiO2", "linear+cubic", 4, 2, 64, 32, 3001),     # affine part first, then the spline sums on top
    ("TiO2", "cubic", 2, 3, 256, 128, 999),
])
def test_spline_sweep_routed(structure, kind, count, world, period, width, frames):
    """Spline masks share one dense_kernel_tp<..., NG> projection; the epilogue of mask g stores to mask g's
    peers.  Models with linear and spline DOFs route only the finished sums."""
    if kind == "linear+cubic":
        state = _linear_and_cubic(structure, 40, 40)
    else:
        state = synthetic.make_model(structure, kind, num_dofs=None if structure == "STO" else 60, seed=5)
    model = rb.InterpolationModel(state)
    if kind == "linear+cubic":
        assert model.path_info()["affine_dofs"] == 40 and model.path_info()["dense_dofs"] == 40
    models = _masked_copies(model, count, seed=count + 10)
    positions = synthetic.make_trajectory(structure, frames, seed=11)
    buffers = _emulate(models, positions, world, period, width)
    series = _check_routing(buffers, world, period, width, [True] * count)
    _check_against_sweep_and_oracle(models, positions, world, series, dense=True)


def test_models_that_do_not_fuse():
    """Models of one structure that share no kernel (different tables, an ART pair below the fused run length)
    are evaluated one by one with their own routed destinations."""
    art = synthetic.make_model("TiO2", "art")
    models = [rb.ARTModel(art), rb.InterpolationModel(synthetic.make_model("TiO2", "cubic", num_dofs=40)),
              rb.ARTModel(synthetic.make_model("TiO2", "art", seed=77)), rb.ARTModel(art).get_masked_model([0, 1, 5])]
    positions = synthetic.make_trajectory("TiO2", 1501, seed=21)
    buffers = _emulate(models, positions, 2, 128, 64)
    series = _check_routing(buffers, 2, 128, 64, [False] * 4)
    _check_against_sweep_and_oracle(models, positions, 2, series, dense=True)


@pytest.mark.parametrize("kind,count", [("art", 4), ("cubic", 4)])
def test_host_sweep_routed_in_chunks(kind, count):
    """The host form sends each chunk across PCIe once for all masks and shifts first_frame per chunk: with
    small chunks it stores exactly what the device form stores."""
    state = synthetic.make_model("TiO2", kind, num_dofs=None if kind == "art" else 48, seed=3)
    cls = rb.ARTModel if kind == "art" else rb.InterpolationModel
    models = _masked_copies(cls(state), count, seed=4)
    positions = synthetic.make_trajectory("TiO2", 2999, seed=5)
    device = _emulate(models, positions, 4, 256, 64)
    host = _emulate(models, positions, 4, 256, 64, host=True, chunk_frames=100)
    for rank in range(4):
        for g in range(count):
            assert np.array_equal(host[rank][g], device[rank][g], equal_nan=True), (rank, g)
    series = _check_routing(host, 4, 256, 64, [True] * count)
    sel = np.r_[0:50, 2949:2999]
    for g, model in enumerate(models):
        oracle = ora.calc_polarizabilities(oracle_model(model.state), positions[sel])
        assert rel_err(series[g][sel].reshape(-1, 3, 3), oracle) <= ALPHA_RTOL


def test_sweep_routed_argument_errors():
    state = synthetic.make_model("TiO2", "art", num_dofs=6)
    model = rb.ARTModel(state)
    positions = to_cuda(synthetic.make_trajectory("TiO2", 64))
    series = torch.zeros((2, 64 * 9), dtype=torch.float64, device="cuda:0")
    local = [series[0].data_ptr()]
    peers = [[0, series[1].data_ptr()]]
    with pytest.raises(ValueError, match="at least one model"):
        calc_polarizabilities_sweep_routed([], positions, [], [], 0, 64, 32)
    with pytest.raises(ValueError, match="at most 64"):
        calc_polarizabilities_sweep_routed([model] * 65, positions, local * 65, peers * 65, 0, 64, 32)
    with pytest.raises(ValueError, match="one local pointer"):
        calc_polarizabilities_sweep_routed([model, model], positions, local, peers, 0, 64, 32)
    with pytest.raises(ValueError, match="between 1 and 8 ranks"):
        calc_polarizabilities_sweep_routed([model], positions, local, [[0] * 9], 0, 64, 32)
    with pytest.raises(ValueError, match="between 1 and 8 ranks"):
        calc_polarizabilities_sweep_routed([model, model], positions, local * 2, [peers[0], peers[0][:1]], 0, 64, 32)
    with pytest.raises(ValueError, match="powers of two"):
        calc_polarizabilities_sweep_routed([model], positions, local, peers, 0, 96, 32)
    with pytest.raises(ValueError, match="powers of two"):
        calc_polarizabilities_sweep_routed([model], positions, local, peers, 0, 64, 16)
    with pytest.raises(ValueError, match="powers of two"):
        calc_polarizabilities_sweep_routed([model], positions, local, peers, 0, 256, 32)  # 8 owners for 2 ranks
    with pytest.raises(ValueError, match="first_frame"):
        calc_polarizabilities_sweep_routed([model], positions, local, peers, -1, 64, 32)
    with pytest.raises(ValueError, match="positions has wrong shape"):
        calc_polarizabilities_sweep_routed([model], to_cuda(synthetic.make_trajectory("STO", 4)), local, peers,
                                           0, 64, 32)
    with pytest.raises(ValueError, match="same structure"):
        other = rb.ARTModel(synthetic.make_model("STO", "art", num_dofs=6))
        calc_polarizabilities_sweep_routed([model, other], positions, local * 2, peers * 2, 0, 64, 32)
    # the C-ABI checks its pointers itself
    lib = _lib.lib()
    handles = (ctypes.c_void_p * 1)(model._native_model().handle)  # pylint: disable=protected-access
    outs = (ctypes.c_void_p * 1)(ctypes.c_void_p(local[0]))
    status = lib.rn_calc_polarizabilities_sweep_routed(handles, 1, ctypes.c_void_p(positions.data_ptr()), 64, outs,
                                                       None, 2, 0, 64, 32, None)
    assert status == -1 and "peer series" in _lib.last_error()
    status = lib.rn_calc_polarizabilities_host_sweep_routed(handles, 0, None, 64, outs, None, 2, 0, 64, 32, 0, None)
    assert status == -1
