"""Single-model evaluation routes that write rows to more than one destination, on one GPU: the routed form
(``calc_polarizabilities_routed``, device and host blocks), the broadcast form (``calc_polarizabilities_multi``)
and the chunked host pipeline behind ``rn_calc_polarizabilities_host``, ``_host_multi`` and ``_host_routed``.
Ranks are emulated as in ``test_gpu_sweep_routed.py``: every rank has its own NaN-filled full series buffer.

"Matches" means within 1e-13 relative of the reference rows (different chunkings and frame counts may pick
different kernel schedules) and a sample of rows within ALPHA_RTOL of the oracle; copies of one row are
compared bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

import ramannoodle_b200 as rb
from oracle import numpy_port as ora
from ramannoodle_b200 import _lib, synthetic
from ramannoodle_b200.distributed import shard_bounds

from gpu_helpers import ALPHA_RTOL, to_cuda
from helpers import oracle_model, rel_err
from test_gpu_sweep_routed import _check_routing, _emulate

pytestmark = pytest.mark.gpu

# 2 ranks that share the transform; 3 ranks of which only 2 share it (rank 2 receives no routed rows)
ROUTES = [(2, 128, 64), (3, 128, 64)]
MODELS = {"art": ("LLZO", "art", rb.ARTModel), "spline": ("STO", "cubic", rb.InterpolationModel)}


def _model_and_positions(kind, frames):
    structure, model_kind, cls = MODELS[kind]
    model = cls(synthetic.make_model(structure, model_kind, seed=5))
    return model, synthetic.make_trajectory(structure, frames, seed=7, lattice_hops=True)


def _assert_matches(got, want, model, positions):
    got = np.asarray(got).reshape(-1, 9)
    assert not np.isnan(got).any()
    assert rel_err(got, np.asarray(want).reshape(-1, 9)) <= 1e-13
    frames = positions.shape[0]
    sel = np.unique(np.r_[0:16, frames // 2 - 8:frames // 2 + 8, frames - 16:frames])
    oracle = ora.calc_polarizabilities(oracle_model(model.state), positions[sel])
    assert rel_err(got[sel].reshape(-1, 3, 3), oracle) <= ALPHA_RTOL


def _route_single(models, block, local, peers, start, period, width, chunk_frames=0):
    assert chunk_frames == 0
    models[0].calc_polarizabilities_routed(block, local[0], peers[0], start, period, width)


def _route_host_routed(models, block, local, peers, start, period, width, chunk_frames=0):
    """``rn_calc_polarizabilities_host_routed`` called directly, with an explicit chunk size."""
    world = len(peers[0])
    table = (ctypes.c_void_p * world)(*[ctypes.c_void_p(int(ptr)) if ptr else None for ptr in peers[0]])
    handle = models[0]._native_model().handle  # pylint: disable=protected-access
    stream = ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream)
    status = _lib.lib().rn_calc_polarizabilities_host_routed(
        handle, ctypes.c_void_p(block.ctypes.data), block.shape[0], ctypes.c_void_p(local[0]), table, world, start,
        period, width, chunk_frames, stream)
    _lib.check(status, "rn_calc_polarizabilities_host_routed")


@pytest.mark.parametrize("world,period,width", ROUTES)
@pytest.mark.parametrize("host", [False, True], ids=["cuda", "numpy"])
@pytest.mark.parametrize("kind", sorted(MODELS))
def test_single_model_routed(kind, host, world, period, width):
    """Every row the routing rule requires is present in every rank's buffer, equal bit for bit to the row the
    evaluating rank stored locally, and the local rows are ``calc_polarizabilities`` of the block."""
    model, positions = _model_and_positions(kind, 2051)
    buffers = _emulate([model], positions, world, period, width, host=host, route=_route_single)
    series = _check_routing(buffers, world, period, width, [False])[0]
    for rank in range(world):
        start, stop = shard_bounds(positions.shape[0], world, rank)
        block = positions[start:stop]
        _assert_matches(series[start:stop], model.calc_polarizabilities(block), model, block)


@pytest.mark.parametrize("host", [False, True], ids=["cuda", "numpy"])
@pytest.mark.parametrize("kind", sorted(MODELS))
def test_multi_broadcast(kind, host):
    """``calc_polarizabilities_multi`` stores the same rows to all three outputs."""
    model, positions = _model_and_positions(kind, 2051)
    frames = positions.shape[0]
    outputs = torch.full((3, frames * 9), float("nan"), dtype=torch.float64, device="cuda:0")
    block = np.ascontiguousarray(positions) if host else to_cuda(positions)
    model.calc_polarizabilities_multi(block, [outputs[i].data_ptr() for i in range(3)])
    torch.cuda.synchronize()
    got = outputs.cpu().numpy().reshape(3, frames, 9)
    assert np.array_equal(got[1], got[0]) and np.array_equal(got[2], got[0])
    _assert_matches(got[0], model.calc_polarizabilities(positions), model, positions)


@pytest.mark.parametrize("kind", sorted(MODELS))
def test_chunked_host_entries(kind):
    """Chunks of 100 frames over an odd frame count give what one chunk gives, for every host entry."""
    model, positions = _model_and_positions(kind, 1001)
    frames = positions.shape[0]
    positions = np.ascontiguousarray(positions, dtype=np.float64)
    lib = _lib.lib()
    handle = model._native_model().handle  # pylint: disable=protected-access
    pos_ptr = ctypes.c_void_p(positions.ctypes.data)

    def host(chunk, to_host=True, to_device=True):
        h_alpha = np.full((frames, 9), np.nan) if to_host else None
        d_alpha = torch.full((frames * 9,), float("nan"), dtype=torch.float64, device="cuda:0") if to_device else None
        torch.cuda.synchronize()
        status = lib.rn_calc_polarizabilities_host(
            handle, pos_ptr, frames, ctypes.c_void_p(h_alpha.ctypes.data) if to_host else None,
            ctypes.c_void_p(d_alpha.data_ptr()) if to_device else None, chunk)
        _lib.check(status, "rn_calc_polarizabilities_host")
        return h_alpha, (d_alpha.cpu().numpy().reshape(frames, 9) if to_device else None)

    whole, whole_device = host(0)
    assert np.array_equal(whole, whole_device)
    _assert_matches(whole, model.calc_polarizabilities(positions), model, positions)
    h_alpha, d_alpha = host(100)
    assert np.array_equal(h_alpha, d_alpha)
    _assert_matches(h_alpha, whole, model, positions)
    h_alpha, _ = host(100, to_device=False)
    _assert_matches(h_alpha, whole, model, positions)

    outputs = torch.full((3, frames * 9), float("nan"), dtype=torch.float64, device="cuda:0")
    table = (ctypes.c_void_p * 3)(*[ctypes.c_void_p(outputs[i].data_ptr()) for i in range(3)])
    torch.cuda.synchronize()
    status = lib.rn_calc_polarizabilities_host_multi(handle, pos_ptr, frames, table, 3, 100,
                                                     ctypes.c_void_p(torch.cuda.current_stream(0).cuda_stream))
    _lib.check(status, "rn_calc_polarizabilities_host_multi")
    got = outputs.cpu().numpy().reshape(3, frames, 9)
    assert np.array_equal(got[1], got[0]) and np.array_equal(got[2], got[0])
    _assert_matches(got[0], whole, model, positions)

    world, period, width = 3, 128, 64
    one = _emulate([model], positions, world, period, width, host=True, route=_route_host_routed)
    chunked = _emulate([model], positions, world, period, width, host=True, chunk_frames=100, route=_route_host_routed)
    one_series = _check_routing(one, world, period, width, [False])[0]
    chunked_series = _check_routing(chunked, world, period, width, [False])[0]
    _assert_matches(one_series, whole, model, positions)
    _assert_matches(chunked_series, one_series, model, positions)
