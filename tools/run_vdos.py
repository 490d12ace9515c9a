"""Vibrational density of states, timed on one GPU with device-resident synthetic trajectories:
  A = Trajectory.get_vdos_device(lattice, groups, weights): every group in one batched transform;
  B = the loop a user writes without A: torch.diff and the minimum image on the device, then one
      rb.calc_signal_spectrum per velocity signal (3 per atom membership), weighted and summed per group.
A and B run alternately in one process after warm-ups and are timed with CUDA events around the whole call
(median of REPEATS).  Kernel times come from separate torch.profiler passes over one call of each.  Workloads:
(a) LLZO, 192 atoms, S = 1e6, one group; (b) the same with one group per species and mass weights; (c) TiO2,
108 atoms, S = 1e5, one group.  The transform rate is 3 * slots * L points over A's kernel time.  The numpy
oracle (tests/vdos_oracle.py) is timed on what it is run on here, one atom, and A is checked against it there.
python tools/run_vdos.py [OUT.json] [REPEATS]"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402
from ramannoodle_b200.spectrum import clear_plan_cache  # noqa: E402
from vdos_oracle import vdos  # noqa: E402  pylint: disable=wrong-import-position

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r07_vdos.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)
MASSES = {3: 6.94, 8: 15.999, 22: 47.867, 38: 87.62, 40: 91.224, 57: 138.905}


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def loop(positions, lattice, timestep, groups, weights):
    """What a user writes today: velocities on the device, then calc_signal_spectrum per signal on the host path."""
    d = torch.diff(positions, dim=0)
    d = d - torch.ceil(d - 0.5)
    v = (d @ torch.as_tensor(lattice, device=positions.device)) / timestep
    rows, wn = [], None
    for group in groups:
        row = None
        for i in group:
            for c in range(3):
                wn, inten = rb.calc_signal_spectrum(v[:, i, c].cpu().numpy(), timestep)
                term = weights[i] * inten[1:]
                row = term if row is None else row + term
        rows.append(row)
    return wn[1:], np.stack(rows)


def timed(fn):
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return float(start.elapsed_time(stop))


def kernel_ms(fn):
    """Device time per kernel name of one fn() call (torch.profiler, a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile  # pylint: disable=import-outside-toplevel

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    times = {}
    for event in prof.key_averages():
        value = float(getattr(event, "self_device_time_total", getattr(event, "self_cuda_time_total", 0.0)))
        if value > 0:
            times[event.key] = times.get(event.key, 0.0) + value / 1000.0
    return times


def kernel_total(times):
    return sum(v for k, v in times.items() if not k.startswith(("Memcpy", "Memset")))


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def transform_length(frames):
    log2l = 12
    while (1 << log2l) < max(2 * (frames - 1) - 1, 4096):
        log2l += 1
    return 1 << log2l


def run(name, structure, frames, grouping):
    geom = synthetic.load_structure(structure)
    lattice, numbers = geom["lattice"], geom["atomic_numbers"]
    num_atoms = len(numbers)
    if grouping == "species":
        groups = [np.flatnonzero(numbers == z).tolist() for z in np.unique(numbers)]
        weights = np.array([MASSES[int(z)] for z in numbers])
    else:
        groups, weights = [list(range(num_atoms))], np.ones(num_atoms)
    positions = synthetic.make_trajectory_cuda(structure, frames, device, seed=31)
    trajectory = rb.Trajectory(positions, 1.0)
    new = lambda: trajectory.get_vdos_device(lattice, groups, weights)  # noqa: E731
    old = lambda: loop(trajectory._positions_ts, lattice, 1.0, groups, weights)  # noqa: E731  pylint: disable=protected-access
    new()
    old()  # warm-up: plans, kernel modules
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(new))
        b_ms.append(timed(old))
    slots = sum((len(g) + 1) // 2 for g in groups)
    a_kernels = kernel_ms(new)
    b_kernels = kernel_ms(old)
    a_kernel_total = kernel_total(a_kernels)
    points = 3 * slots * transform_length(frames)
    wn, rows = (t.cpu().numpy() for t in new())
    loop_wn, loop_rows = old()
    # the numpy oracle, run on one atom only (the full trajectory does not fit its host temporaries in reasonable time)
    one_atom = trajectory._positions_ts[:, :1].cpu().numpy()  # pylint: disable=protected-access
    start = time.perf_counter()
    oracle_wn, oracle_row = vdos(one_atom, lattice, 1.0, [[0]], [weights[0]])
    oracle_s = time.perf_counter() - start
    _, gpu_row = (t.cpu().numpy() for t in trajectory.get_vdos_device(lattice, [[0]], weights))
    result = {
        "workload": name, "structure": structure, "atoms": num_atoms, "frames": frames, "groups": len(groups),
        "slots": slots, "transform_length": transform_length(frames),
        "vdos_ms": stats(a_ms), "loop_ms": stats(b_ms), "speedup_median": float(np.median(b_ms) / np.median(a_ms)),
        "vdos_kernel_ms_total": a_kernel_total, "vdos_kernel_ms": a_kernels,
        "loop_kernel_ms_total": kernel_total(b_kernels),
        "loop_memcpy_ms_total": sum(v for k, v in b_kernels.items() if k.startswith("Memcpy")),
        "transform_points": points, "transform_rate_points_per_s": points / (a_kernel_total * 1e-3),
        "loop_max_rel_dev": float(np.max(np.abs(loop_rows - rows) / np.abs(rows))),
        "loop_wavenumbers_equal": bool(np.array_equal(loop_wn, wn)),
        "numpy_oracle_one_atom_s": oracle_s,
        "one_atom_max_rel_err_vs_oracle": float(np.max(np.abs(gpu_row - oracle_row) / np.abs(oracle_row))),
        "one_atom_wavenumbers_equal": bool(np.array_equal(oracle_wn, wn)),
        "vdos_runs_ms": a_ms, "loop_runs_ms": b_ms,
    }
    print(json.dumps({k: v for k, v in result.items() if not k.endswith("runs_ms") and k != "vdos_kernel_ms"}),
          flush=True)
    del trajectory, positions
    clear_plan_cache()
    torch.cuda.empty_cache()
    return result


card, power = gpu_info()
results = [
    run("(a) LLZO, one group", "LLZO", 1_000_000, "all"),
    run("(b) LLZO, four species groups, mass weights", "LLZO", 1_000_000, "species"),
    run("(c) TiO2, one group", "TiO2", 100_000, "all"),
]
record = {"what": "Trajectory.get_vdos_device (A) against the per-signal loop (B: device torch.diff + minimum image, "
                  "then rb.calc_signal_spectrum per velocity signal); CUDA events around each call, A and B "
                  "alternated, medians of the repeats; kernel times from separate torch.profiler passes over one "
                  "call of each; trajectories HBM-resident float64, timestep 1 fs; the numpy oracle timed on one "
                  "atom only",
          "gpu": card, "power_limit": power, "repeats": repeats, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)
