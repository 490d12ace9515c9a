"""Cross spectra of frame-sharded mask sweeps: one process per GPU under torchrun runs
tools/check_sharded_cross.py — ShardedTrajectory.get_raman_spectra(models) followed by measure_cross_spectra,
with the shared transform context and with the all-gather fallback, on host and HBM-resident blocks, against
the single-GPU result of the gathered series (bit for bit) and the oracle.  World 1 runs the single-GPU path;
world 3 has a rank outside the transform group."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from helpers import REPO

pytestmark = pytest.mark.gpu

CASE_LINES = 2 * 3  # two cases x (host shared, resident shared, resident all-gather)


def _free_port():
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _run_check(world):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(REPO, "tools", "check_sharded_cross.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=REPO)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-6000:]
    assert res.stdout.count("ok=True") == world * CASE_LINES and "ok=False" not in res.stdout, res.stdout[-6000:]
    if world > 1:  # the shared transform context really held the series
        assert res.stdout.count("shared=True (used=True)") == world * 2 * 2, res.stdout[-6000:]


@pytest.mark.skipif(torch.cuda.device_count() < 1, reason="needs a GPU")
def test_sharded_cross_one_rank():
    _run_check(1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_cross_two_ranks():
    _run_check(2)


@pytest.mark.skipif(torch.cuda.device_count() < 3, reason="needs at least 3 GPUs")
def test_sharded_cross_spectator_rank():
    _run_check(3)


@pytest.mark.skipif(torch.cuda.device_count() < 4, reason="needs more than 3 GPUs")
def test_sharded_cross_all_ranks():
    _run_check(min(torch.cuda.device_count(), 8))
