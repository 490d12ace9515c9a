"""Multi-GPU mask sweeps (skipped below 2 GPUs): one process per GPU under torchrun runs
tools/check_sharded_sweep.py — ShardedTrajectory.get_raman_spectra on host and HBM-resident blocks, with the
routed sweep and one shared chirp-z transform per mask, and with the all-gather fallback, against the oracle,
per-mask get_raman_spectrum and the single-GPU Trajectory.get_raman_spectra.  World 3 has a rank outside
the transform group.  Tolerances: 1e-10 on polarizabilities, 1e-8 on intensities."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from helpers import REPO

pytestmark = pytest.mark.gpu

MASK_LINES = 4 + 3 + 2 + 4  # species of LLZO, STO, TiO2 and the large LLZO case


def _free_port():
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _run_check(world):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(REPO, "tools", "check_sharded_sweep.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, cwd=REPO)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-6000:]
    # every mask of every case x (host | HBM-resident) x (shared transform | all-gather), per rank
    assert res.stdout.count("ok=True") == world * 4 * MASK_LINES and "ok=False" not in res.stdout, res.stdout[-6000:]
    # the routed sweep and the shared transform really ran (not the all-gather fallback)
    assert res.stdout.count("shared=True (used=True)") == world * 2 * MASK_LINES, res.stdout[-6000:]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least 2 GPUs")
def test_sharded_sweep_two_ranks():
    _run_check(2)


@pytest.mark.skipif(torch.cuda.device_count() < 3, reason="needs at least 3 GPUs")
def test_sharded_sweep_spectator_rank():
    _run_check(3)


@pytest.mark.skipif(torch.cuda.device_count() < 4, reason="needs more than 3 GPUs")
def test_sharded_sweep_all_ranks():
    _run_check(min(torch.cuda.device_count(), 8))
