"""Projected VDOS, timed on one GPU with device-resident synthetic trajectories:
  A = Trajectory.get_projected_vdos_device(lattice, vectors): the projection on the FP64 tensor pipe fused with the
      batched transforms;
  B = the loop a user writes without A: torch.diff and the minimum image on the device, torch.matmul with the
      vectors, then one rb.calc_signal_spectrum per mode.
A and B run alternately in one process after warm-ups and are timed with CUDA events around the whole call
(median of REPEATS).  Kernel times come from separate torch.profiler passes over one call of each.  Workloads:
(a) LLZO, 192 atoms, S = 1e6, K = 576 vectors of a random orthonormal mass-weighted basis (LLZO has no phonon
fixture); (b) TiO2, 108 atoms, S = 1e5, the 81 golden phonon modes via Phonons.get_mode_vectors; (c) LLZO, S = 1e6,
K = 48 (one chunk: isolates the projection).  The projection rate is 2 M 3N K flop over the time of
project_velocity_kernel, set against the measured DMMA peak (profiles/fp64_peaks.json) and against B's
torch.matmul on the same shapes (CUDA events, median of REPEATS); the transform rate is 3 ceil(K/6) L points over
the time of the transform passes.
python tools/run_projected_vdos.py [OUT.json] [REPEATS]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200 import synthetic  # noqa: E402
from ramannoodle_b200.spectrum import clear_plan_cache  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r08_projected_vdos.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)
MASSES = {3: 6.94, 8: 15.999, 22: 47.867, 38: 87.62, 40: 91.224, 57: 138.905}
DMMA_PEAK_TFLOPS = 37.16  # profiles/fp64_peaks.json, measured on a B200


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def velocities(positions, lattice, timestep):
    d = torch.diff(positions, dim=0)
    d = d - torch.ceil(d - 0.5)
    return (d @ torch.as_tensor(lattice, device=positions.device)) / timestep


def loop(positions, lattice, timestep, vectors):
    """What a user writes today: velocities and their projection on the device, calc_signal_spectrum per mode."""
    v = velocities(positions, lattice, timestep)
    q = torch.matmul(v.reshape(v.shape[0], -1), vectors.reshape(vectors.shape[0], -1).T)  # (M, K)
    rows, wn = [], None
    for k in range(q.shape[1]):
        wn, inten = rb.calc_signal_spectrum(q[:, k].cpu().numpy(), timestep)
        rows.append(inten[1:])
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


def kernel_total(times, *names):
    return sum(v for k, v in times.items() if not k.startswith(("Memcpy", "Memset")) and
               (not names or any(n in k for n in names)))


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def transform_length(frames):
    log2l = 12
    while (1 << log2l) < max(2 * (frames - 1) - 1, 4096):
        log2l += 1
    return 1 << log2l


def orthonormal_mass_weighted(masses, seed):
    num_atoms = len(masses)
    q, _ = np.linalg.qr(np.random.default_rng(seed).normal(size=(3 * num_atoms, 3 * num_atoms)))
    return np.sqrt(masses)[None, :, None] * q.T.reshape(3 * num_atoms, num_atoms, 3)


def run(name, structure, frames, kind):
    geom = synthetic.load_structure(structure)
    lattice, numbers = geom["lattice"], geom["atomic_numbers"]
    num_atoms = len(numbers)
    masses = np.array([MASSES[int(z)] for z in numbers])
    if kind == "phonons":
        with np.load(os.path.join(REPO, "tests", "golden", "phonons_tio2.npz")) as data:
            phonons = rb.Phonons(data["ref_positions"], data["wavenumbers"], data["displacements"])
        vectors = phonons.get_mode_vectors(lattice, masses)
    else:
        vectors = orthonormal_mass_weighted(masses, seed=7)[:kind]
    num_vectors = vectors.shape[0]
    positions = synthetic.make_trajectory_cuda(structure, frames, device, seed=31)
    trajectory = rb.Trajectory(positions, 1.0)
    d_vectors = torch.from_numpy(vectors).to(device)
    new = lambda: trajectory.get_projected_vdos_device(lattice, vectors)  # noqa: E731
    old = lambda: loop(trajectory._positions_ts, lattice, 1.0, d_vectors)  # noqa: E731  pylint: disable=protected-access
    new()
    old()  # warm-up: plans, kernel modules, cuBLAS
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(new))
        b_ms.append(timed(old))
    # torch.matmul of the loop on its own, same shapes
    v = velocities(trajectory._positions_ts, lattice, 1.0).reshape(frames - 1, -1)  # pylint: disable=protected-access
    w = d_vectors.reshape(num_vectors, -1).T
    torch.matmul(v, w)
    matmul_ms = [timed(lambda: torch.matmul(v, w)) for _ in range(repeats)]
    del v
    a_kernels = kernel_ms(new)
    b_kernels = kernel_ms(old)
    a_total = kernel_total(a_kernels)
    projection = kernel_total(a_kernels, "project_velocity_kernel")
    transform = kernel_total(a_kernels, "level_kernel", "tile_kernel")
    flop = 2.0 * (frames - 1) * 3 * num_vectors * num_atoms
    windows = -(-num_vectors // 6)
    points = 3 * windows * transform_length(frames)
    wn, rows = (t.cpu().numpy() for t in new())
    loop_wn, loop_rows = old()
    nonzero = loop_rows != 0
    result = {
        "workload": name, "structure": structure, "atoms": num_atoms, "frames": frames, "vectors": num_vectors,
        "windows": windows, "transform_length": transform_length(frames),
        "projected_vdos_ms": stats(a_ms), "loop_ms": stats(b_ms),
        "speedup_median": float(np.median(b_ms) / np.median(a_ms)),
        "projected_vdos_kernel_ms_total": a_total, "projected_vdos_kernel_ms": a_kernels,
        "projection_kernel_ms": projection, "projection_flop": flop,
        "projection_tflops": flop / (projection * 1e-3) / 1e12,
        "projection_share_of_dmma_peak": flop / (projection * 1e-3) / 1e12 / DMMA_PEAK_TFLOPS,
        "loop_matmul_ms": stats(matmul_ms),
        "loop_matmul_tflops": flop / (float(np.median(matmul_ms)) * 1e-3) / 1e12,
        "transform_kernel_ms": transform, "transform_points": points,
        "transform_rate_points_per_s": points / (transform * 1e-3),
        "loop_kernel_ms_total": kernel_total(b_kernels),
        "loop_memcpy_ms_total": sum(v for k, v in b_kernels.items() if k.startswith("Memcpy")),
        "loop_max_rel_dev": float(np.max(np.abs(loop_rows - rows)[nonzero] / np.abs(loop_rows)[nonzero])),
        "loop_wavenumbers_equal": bool(np.array_equal(loop_wn, wn)),
        "projected_vdos_runs_ms": a_ms, "loop_runs_ms": b_ms,
    }
    print(json.dumps({k: v for k, v in result.items() if not k.endswith("runs_ms") and k != "projected_vdos_kernel_ms"}),
          flush=True)
    del trajectory, positions
    clear_plan_cache()
    torch.cuda.empty_cache()
    return result


card, power = gpu_info()
results = [
    run("(a) LLZO, S = 1e6, K = 576 (orthonormal mass-weighted basis)", "LLZO", 1_000_000, 576),
    run("(b) TiO2, S = 1e5, the 81 golden phonon modes", "TiO2", 100_000, "phonons"),
    run("(c) LLZO, S = 1e6, K = 48 (one chunk)", "LLZO", 1_000_000, 48),
]
record = {"what": "Trajectory.get_projected_vdos_device (A) against the per-mode loop (B: device torch.diff + minimum "
                  "image, torch.matmul with the vectors, then rb.calc_signal_spectrum per mode); CUDA events around "
                  "each call, A and B alternated, medians of the repeats; kernel times from separate torch.profiler "
                  "passes over one call of each; trajectories HBM-resident float64, timestep 1 fs",
          "gpu": card, "power_limit": power, "repeats": repeats, "dmma_peak_tflops": DMMA_PEAK_TFLOPS,
          "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)
