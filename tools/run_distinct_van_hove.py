"""Distinct Van Hove correlation, timed on one GPU with device-resident synthetic trajectories:
  A = Trajectory.get_distinct_van_hove_device(lattice, lags, r_max, num_bins, groups): one histogram launch and one
      finishing launch;
  B = the chunked torch composition a user writes without A: per lag, ordered group pair and chunk of origins the
      (origins, |a|, |b|, 3) difference tensor, the wrap, the lattice product, norms, the i != j mask and
      torch.bincount.
A and B run alternately in one process after warm-ups and are timed with CUDA events around the whole call (median of
REPEATS); the peak device memory of each is torch.cuda.max_memory_allocated over one call, above what was allocated
before it.  Kernel times come from a separate torch.profiler pass over one call of A.  Workloads:
  (a) LLZO, 192 atoms, S = 1e4, the four species groups (16 ordered pairs), Li random walk, lag 0 and 31 log-spaced
      lags in [1, S/2], r_max = w_min/2, B = 400;
  (b) LLZO, S = 1e5, the Li group (56 atoms), Li random walk, lag 0 and 63 log-spaced lags up to S/10, r_max = w_min/2,
      B = 400;
  (c) TiO2, 108 atoms, S = 1e4, one group, lags 0..31, r_max 4.8 Å, B = 200.
Then, on (a)'s trajectory, a lag-0-only call of A against Trajectory.get_rdf_device, alternated in the same way: the
distinct call evaluates every ordered pair, the RDF kernel every unordered pair once, so A should take about twice
as long at the same per-pair rate.
Rates: pairs evaluated per second over the histogram kernel's time, sum_t (S - t) sum_ab n_ab for A; the FP64 issue
bound is the DFMA rate of profiles/fp64_peaks.json over FP64_PER_PAIR instructions per pair and FP64_PER_BINNED more
per pair within r_max (the SASS counts of the [0, 1] path of rdf_bin, DESIGN.md 4.5).
python tools/run_distinct_van_hove.py [OUT.json] [REPEATS]"""
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

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r12_distinct_van_hove.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)
FP64_PER_PAIR = 36
FP64_PER_BINNED = 11
LI_STEP = 0.01  # Å per frame and Cartesian component of the Li random walk (tools/run_msd.py)
CHUNK_ELEMENTS = 1 << 24  # origins x |a| x |b| pairs per step of the torch composition


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def fp64_peak():
    with open(os.path.join(REPO, "profiles", "fp64_peaks.json"), encoding="utf-8") as handle:
        return float(json.load(handle)["dfma_tflops"]) * 1e12 / 2


def cell(lattice):
    cross = np.cross(lattice[[1, 2, 0]], lattice[[2, 0, 1]])
    volume = abs(float(np.dot(lattice[0], cross[0])))
    return volume, 0.5 * float(np.min(volume / np.sqrt(np.sum(cross * cross, axis=1))))


def make_positions(structure, frames, diffusing_z):
    positions = synthetic.make_trajectory_cuda(structure, frames, device, seed=61)
    if diffusing_z is None:
        return positions
    geom = synthetic.load_structure(structure)
    walkers = torch.as_tensor(np.flatnonzero(geom["atomic_numbers"] == diffusing_z), device=device)
    gen = torch.Generator(device=device)
    gen.manual_seed(62)
    walk = torch.randn((frames, len(walkers), 3), generator=gen, device=device, dtype=torch.float64) * LI_STEP
    walk = torch.cumsum(walk, dim=0) @ torch.as_tensor(np.linalg.inv(geom["lattice"]), device=device)
    moved = positions[:, walkers] + walk
    positions[:, walkers] = moved - torch.floor(moved)
    return positions


def pair_norms(groups):
    return np.array([[len(a) * len(b) - len(set(a) & set(b)) for b in groups] for a in groups], dtype=np.int64)


def composition(x, lattice, lags, r_max, num_bins, groups):
    """What a user writes today, on the device: g_d (G, G, T, B)."""
    frames = x.shape[0]
    lat = torch.as_tensor(lattice, device=device)
    volume, _ = cell(lattice)
    index = [torch.as_tensor(g, device=device) for g in groups]
    inv = num_bins / r_max
    edges = torch.arange(num_bins + 1, dtype=torch.float64, device=device) * (r_max / num_bins)
    shell = 4 * np.pi / 3 * (edges[1:] ** 3 - edges[:-1] ** 3)
    counts = torch.zeros((len(groups), len(groups), len(lags), num_bins), dtype=torch.int64, device=device)
    for ti, t in enumerate(lags):
        for a, ia in enumerate(index):
            for b, ib in enumerate(index):
                keep = ia[:, None] != ib[None, :]
                chunk = max(1, CHUNK_ELEMENTS // (len(ia) * len(ib)))
                for n0 in range(0, frames - t, chunk):
                    n1 = min(frames - t, n0 + chunk)
                    d = x[n0 + t:n1 + t][:, None, ib] - x[n0:n1][:, ia, None]
                    d = d - torch.ceil(d - 0.5)
                    k = torch.floor(torch.linalg.vector_norm(d @ lat, dim=-1) * inv)[:, keep]
                    counts[a, b, ti] += torch.bincount(k[k < num_bins].to(torch.int64), minlength=num_bins)
    norms = torch.as_tensor(pair_norms(groups), device=device, dtype=torch.float64)
    origins = frames - torch.as_tensor(lags, device=device, dtype=torch.float64)
    denom = (norms[:, :, None] * origins[None, None, :])[..., None] * shell
    return torch.where(denom > 0, counts * volume / torch.where(denom > 0, denom, 1.0), 0.0)


def timed(fn):
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return float(start.elapsed_time(stop))


def peak_bytes(fn):
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    result = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - before
    del result
    return int(peak)


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


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def log_lags(low, high, count):
    """count distinct integers from low to high, log-spaced: the rounded geometric sequence, made longer until its
    distinct values number count."""
    num = count
    while True:
        lags = np.unique(np.rint(np.geomspace(low, high, num)).astype(np.int64))
        if len(lags) >= count:
            return lags
        num += 1


def alternate(new, old):
    a_ms, b_ms = [], []
    for _ in range(repeats):
        a_ms.append(timed(new))
        b_ms.append(timed(old))
    return a_ms, b_ms


def run(name, structure, frames, grouping, lags, r_max, num_bins, diffusing_z, fp64_rate):
    geom = synthetic.load_structure(structure)
    lattice, numbers = geom["lattice"], geom["atomic_numbers"]
    if grouping == "species":
        groups = [np.flatnonzero(numbers == z).tolist() for z in np.unique(numbers)]
    elif grouping == "li":
        groups = [np.flatnonzero(numbers == 3).tolist()]
    else:
        groups = [list(range(len(numbers)))]
    lags = [int(t) for t in lags]
    volume, half_width = cell(lattice)
    r_max = half_width if r_max is None else r_max
    trajectory = rb.Trajectory(make_positions(structure, frames, diffusing_z), 1.0)
    stored = trajectory._positions_ts  # pylint: disable=protected-access
    new = lambda: trajectory.get_distinct_van_hove_device(lattice, lags, r_max, num_bins, groups)  # noqa: E731
    old = lambda: composition(stored, lattice, lags, r_max, num_bins, groups)  # noqa: E731
    new()
    old()  # warm-up: kernel modules, torch kernels
    before = rb._lib.launch_count()  # pylint: disable=protected-access
    new()
    torch.cuda.synchronize()
    launches = rb._lib.launch_count() - before  # pylint: disable=protected-access
    a_ms, b_ms = alternate(new, old)
    a_peak, b_peak = peak_bytes(new), peak_bytes(old)
    a_kernels = kernel_ms(new)
    hist_ms = sum(v for k, v in a_kernels.items() if "dvh_histogram_kernel" in k)
    got = new()[2].cpu().numpy()
    ref = old().cpu().numpy()
    norms = pair_norms(groups)
    origins = frames - np.array(lags)
    pairs = float(norms.sum() * origins.sum())
    edges = np.arange(num_bins + 1) * (r_max / num_bins)
    shell = 4 * np.pi / 3 * (edges[1:] ** 3 - edges[:-1] ** 3)
    binned = float(np.rint(got * (norms[:, :, None] * origins[None, None, :])[..., None] * shell / volume).sum())
    fp64 = FP64_PER_PAIR * pairs + FP64_PER_BINNED * binned
    nonzero = np.abs(got) > 0
    result = {
        "workload": name, "structure": structure, "atoms": len(numbers), "frames": frames, "groups": len(groups),
        "lags": len(lags), "max_lag": max(lags), "r_max": r_max, "num_bins": num_bins, "launches": launches,
        "distinct_ms": stats(a_ms), "torch_ms": stats(b_ms), "speedup_median": float(np.median(b_ms) / np.median(a_ms)),
        "distinct_peak_bytes": a_peak, "torch_peak_bytes": b_peak,
        "distinct_kernel_ms": a_kernels, "histogram_kernel_ms": hist_ms,
        "pairs": pairs, "pairs_within_r_max": binned,
        "pairs_per_s_call": pairs / (np.median(a_ms) * 1e-3), "pairs_per_s_kernel": pairs / (hist_ms * 1e-3),
        "fp64_issue_bound_pairs_per_s": fp64_rate * pairs / fp64,
        "fp64_share_of_dfma_rate": fp64 / (hist_ms * 1e-3) / fp64_rate,
        "torch_g_d_max_rel_dev": float(np.max(np.abs(got - ref)[nonzero] / np.abs(got)[nonzero], initial=0.0)),
        "torch_bins_differing": int(np.sum(got != ref)),
        "distinct_runs_ms": a_ms, "torch_runs_ms": b_ms,
    }
    print(json.dumps({k: v for k, v in result.items() if not k.endswith(("runs_ms", "kernel_ms"))}), flush=True)
    return result, trajectory, lattice, groups, r_max, num_bins


def lag_zero_against_rdf(trajectory, lattice, groups, r_max, num_bins, frames):
    """A lag-0-only distinct call against get_rdf on the same trajectory: both alternated, kernel times from one
    profiler pass over each."""
    new = lambda: trajectory.get_distinct_van_hove_device(lattice, [0], r_max, num_bins, groups)  # noqa: E731
    rdf = lambda: trajectory.get_rdf_device(lattice, r_max, num_bins, groups)  # noqa: E731
    new()
    rdf()
    a_ms, b_ms = alternate(new, rdf)
    a_kernel = sum(v for k, v in kernel_ms(new).items() if "dvh_histogram_kernel" in k)
    b_kernel = sum(v for k, v in kernel_ms(rdf).items() if "rdf_histogram_kernel" in k)
    norms = pair_norms(groups)
    sizes = np.array([len(g) for g in groups], dtype=np.int64)
    ordered = float(frames * norms.sum())
    # the RDF kernel evaluates p < q once for a == b and every pair of a < b
    unordered = float(frames * (np.triu(norms, 1).sum() + np.sum(sizes * (sizes - 1) // 2)))
    identical = bool(torch.equal(new()[2][:, :, 0], rdf()[1]))
    result = {
        "workload": "lag 0 only on (a)'s trajectory against get_rdf", "distinct_ms": stats(a_ms), "rdf_ms": stats(b_ms),
        "time_ratio_median": float(np.median(a_ms) / np.median(b_ms)),
        "distinct_histogram_kernel_ms": a_kernel, "rdf_histogram_kernel_ms": b_kernel,
        "distinct_pairs": ordered, "rdf_pairs": unordered,
        "distinct_pairs_per_s_kernel": ordered / (a_kernel * 1e-3), "rdf_pairs_per_s_kernel": unordered / (b_kernel * 1e-3),
        "lag0_bit_identical_to_rdf": identical, "distinct_runs_ms": a_ms, "rdf_runs_ms": b_ms,
    }
    print(json.dumps({k: v for k, v in result.items() if not k.endswith("runs_ms")}), flush=True)
    return result


card, power = gpu_info()
fp64_rate = fp64_peak()
results = []
res, traj_a, lattice_a, groups_a, r_max_a, bins_a = run(
    "(a) LLZO, species groups, Li diffusing", "LLZO", 10_000, "species", [0] + list(log_lags(1, 5_000, 31)), None, 400,
    3, fp64_rate)
results.append(res)
lag_zero = lag_zero_against_rdf(traj_a, lattice_a, groups_a, r_max_a, bins_a, 10_000)
del traj_a
torch.cuda.empty_cache()
for args in (("(b) LLZO, Li group, Li diffusing", "LLZO", 100_000, "li", [0] + list(log_lags(1, 10_000, 63)), None,
              400, 3),
             ("(c) TiO2, one group", "TiO2", 10_000, "all", np.arange(0, 32), 4.8, 200, None)):
    res, traj, *_ = run(*args, fp64_rate)
    results.append(res)
    del traj
    torch.cuda.empty_cache()
record = {"what": "Trajectory.get_distinct_van_hove_device (A) against the chunked torch composition (B: per lag, "
                  "ordered group pair and chunk of origins the difference tensor, wrap, lattice product, norms, i != j "
                  "mask and torch.bincount); CUDA events around each call, A and B alternated, medians of the repeats; "
                  "peak memory from torch.cuda.max_memory_allocated over one call; kernel times from a separate "
                  "torch.profiler pass over one call; trajectories HBM-resident float64",
          "gpu": card, "power_limit": power, "repeats": repeats, "fp64_instructions_per_s": fp64_rate,
          "fp64_per_pair": FP64_PER_PAIR, "fp64_per_binned_pair": FP64_PER_BINNED,
          "rdf_kernel_pairs_per_s_r10": [1.15e11, 1.91e11], "results": results, "lag_zero_against_rdf": lag_zero}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k not in ("results", "lag_zero_against_rdf")}), flush=True)
