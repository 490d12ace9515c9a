"""Mask sweeps on frame-sharded trajectories, timed (launch with torchrun, one rank per GPU):
  A = per-mask ShardedTrajectory.get_raman_spectrum(m) + measure_device(), one mask after the other;
  B = ShardedTrajectory.get_raman_spectra(models) + measure_device() of every mask.
Both run on HBM-resident blocks with the routed evaluation and the shared transform, alternated in the same
process after warm-ups; each repetition is timed with CUDA events on every rank and the maximum over the ranks
is kept.  Workloads: the LLZO ARTModel with one mask per species, 1M frames per GPU (c3 shape), and the c5
InterpolationModel (1536-atom supercell, 4600 cubic DOFs) with one mask per species, 1M frames in total.
torchrun --nproc-per-node N tools/run_sharded_sweep.py OUT.json [REPEATS]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402
from ramannoodle_b200.distributed import ShardedTrajectory, shard_bounds  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
device = torch.device(f"cuda:{local}")
dist.init_process_group("nccl", device_id=device)
out_path = sys.argv[1]
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5


def species_masks(model, structure):
    numbers = synthetic.load_structure(structure)["atomic_numbers"]
    finder = rb.ARTModel(model.state)  # get_dof_indexes only reads the basis vectors
    return [model.get_masked_model(finder.get_dof_indexes([int(a) for a in np.flatnonzero(numbers == z)]))
            for z in np.unique(numbers)]


def timed(fn):
    """ms of fn() on this rank (CUDA events), max over the ranks."""
    dist.barrier()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    ms = torch.tensor([start.elapsed_time(stop)], device=device)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def per_mask(sharded, models):
    for model in models:
        sharded.get_raman_spectrum(model).measure_device()


def sweep(sharded, models):
    for spectrum in sharded.get_raman_spectra(models):
        spectrum.measure_device()


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(local), "unknown"


results = []
workloads = [("c3_llzo_art", "LLZO", "art", None, world * 1_000_000),
             ("c5_supercell_cubic", "LLZO_2x2x2", "cubic", 4600, 1_000_000)]
for name, structure, kind, dofs, frames in workloads:
    state = synthetic.make_model(structure, kind, num_dofs=dofs)
    model = (rb.ARTModel if kind == "art" else rb.InterpolationModel)(state, device=local)
    models = species_masks(model, structure)
    start, stop = shard_bounds(frames, world, rank)
    block = synthetic.make_trajectory_cuda(structure, stop - start, device, seed=1000, first_frame=start)
    sharded = ShardedTrajectory(block, 1.0, frames)
    for _ in range(2):  # warm-up: contexts, native models, kernel modules
        per_mask(sharded, models)
        sweep(sharded, models)
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(lambda: per_mask(sharded, models)))
        b_ms.append(timed(lambda: sweep(sharded, models)))
    used = sharded.get_raman_spectra(models)[0]._context is not None  # pylint: disable=protected-access
    results.append({"workload": name, "structure": structure, "kind": kind, "dofs": state.num_dofs,
                    "atoms": state.num_atoms, "masks": len(models), "total_frames": frames,
                    "frames_per_gpu": -(-frames // world), "shared_transform": used,
                    "per_mask_ms": {"median": float(np.median(a_ms)), "min": min(a_ms), "max": max(a_ms)},
                    "sweep_ms": {"median": float(np.median(b_ms)), "min": min(b_ms), "max": max(b_ms)},
                    "speedup_median": float(np.median(a_ms) / np.median(b_ms)),
                    "per_mask_runs_ms": a_ms, "sweep_runs_ms": b_ms})
    del sharded, block
    torch.cuda.empty_cache()

if rank == 0:
    card, power = gpu_info()
    record = {"what": "ShardedTrajectory mask sweep: A = per-mask get_raman_spectrum + measure_device, "
                      "B = get_raman_spectra + measure_device per mask (HBM-resident blocks, routed evaluation, "
                      "shared transform); CUDA events, max over ranks, A and B alternated",
              "n_gpus": world, "gpu": card, "power_limit": power, "repeats": repeats, "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w", encoding="utf-8") as handle:
        json.dump(record, handle, indent=1)
    print(json.dumps(record), flush=True)
dist.destroy_process_group()
