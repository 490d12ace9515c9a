"""Batched smearing against a per-row loop, timed on one GPU (gaussian and lorentzian, width 5, default grid):
  batched = convolve_spectra (numpy output) and convolve_spectra_device (CUDA output), timed separately;
  loop    = convolve_spectrum on every row (numpy output), the loop a user writes without convolve_spectra.
Every form starts from device inputs.  Cases: (a) measure_windows rows, S = 1e6, window 2000, hop 500 (W = 1997);
(b) window 20000, hop 5000 (W = 197); (c) measure_cross_spectra, G = 4, S = 1e6 (16 rows); (d) one c3-sized
spectrum (S = 1e6, one row).  The forms alternate in one process after a warm-up of every shape, CUDA events around
each whole call, median of REPEATS; batched and loop outputs are compared bit for bit.  Kernel times come from a
torch.profiler run of its own per case (a child process: one profiler session per process, one batched call and
one loop per function, kernels attributed in launch order).  Factor evaluations are counted from the shapes and the
skip rule (gaussian: an (input chunk, output tile) pair is skipped when every distance exceeds 39 w; lorentzian:
nothing is skipped): the batched kernel evaluates a factor once per group of 8 rows (one row runs the single-row
kernels), the loop once per row.
python tools/run_convolve_spectra.py [OUT.json] [REPEATS]        (python tools/run_convolve_spectra.py --profile CASE)"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200.spectrum import clear_plan_cache  # noqa: E402

PROFILE = len(sys.argv) > 2 and sys.argv[1] == "--profile"
out_path = sys.argv[1] if len(sys.argv) > 1 and not PROFILE else os.path.join("profiles", "r06_convolve_spectra.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 and not PROFILE else 5
FRAMES = 1_000_000
WIDTH = 5.0
IN_CHUNK, OUT_TILE, ROWS = 2048, 256, 8  # kInChunk, kOutTile, kRows of csrc/rn_smear.cu
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


def synthetic_series(frames, seed, count=None):
    gen = torch.Generator(device).manual_seed(seed)
    lead = () if count is None else (count,)
    steps = torch.arange(frames, dtype=torch.float64, device=device)[:, None, None]
    phase = torch.rand(lead + (1, 3, 3), dtype=torch.float64, device=device, generator=gen) * 6
    noise = torch.randn(lead + (frames, 3, 3), dtype=torch.float64, device=device, generator=gen)
    return 6.0 * torch.eye(3, dtype=torch.float64, device=device) + 0.05 * torch.sin(0.013 * steps + phase) \
        + 0.01 * noise


def default_grid(wn):
    low, high = (float(v) for v in torch.aminmax(wn))
    return np.linspace(low - 100, high + 100, int(np.rint((high + 100) - (low - 100))))


def evaluated_pairs(wn, grid, function):
    """(input, output) pairs whose factor the kernels evaluate for one row: every pair of an (input chunk,
    output tile) block that the skip rule keeps (outputs past the grid are not counted)."""
    wn = wn.cpu().numpy()
    chunks = [wn[c:c + IN_CHUNK] for c in range(0, len(wn), IN_CHUNK)]
    tiles = [grid[t:t + OUT_TILE] for t in range(0, len(grid), OUT_TILE)]
    n_in = np.array([len(c) for c in chunks])[:, None]
    n_out = np.array([len(t) for t in tiles])[None, :]
    if function == "lorentzian":
        return int((n_in * n_out).sum())
    c_lo, c_hi = (np.array([f(c) for c in chunks])[:, None] for f in (np.min, np.max))
    t_lo, t_hi = (np.array([f(t) for t in tiles])[None, :] for f in (np.min, np.max))
    cut = 39.0 * WIDTH
    far = (c_lo - t_hi > cut) | (t_lo - c_hi > cut)
    return int((n_in * n_out * ~far).sum())


def timed(fn):
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return float(start.elapsed_time(stop))


def profile_case(wn, rows):
    """Kernel times of one batched call and one loop per function, from one torch.profiler session: smear kernels
    in launch order, a reduce belonging to the partial kernel launched before it."""
    from torch.profiler import ProfilerActivity, profile  # pylint: disable=import-outside-toplevel

    flat = rows.reshape(-1, rows.shape[-1])
    for function in ("gaussian", "lorentzian"):  # warm-up
        rb.convolve_spectra_device(wn, rows, function, WIDTH)
        rb.convolve_spectrum(wn, flat[0], function, WIDTH)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for function in ("gaussian", "lorentzian"):
            rb.convolve_spectra_device(wn, rows, function, WIDTH)
            torch.cuda.synchronize()
            for b in range(flat.shape[0]):
                rb.convolve_spectrum(wn, flat[b], function, WIDTH)
            torch.cuda.synchronize()
    kernels = sorted((e for e in prof.events() if "smear_" in e.name and "cuda" in str(e.device_type).lower()),
                     key=lambda e: e.time_range.start)
    segments = []  # (batched or loop, function) in launch order
    times = {}
    for event in kernels:
        if "smear_reduce_kernel" not in event.name:
            batched = "smear_rows_partial_kernel" in event.name or (flat.shape[0] == 1 and len(segments) % 2 == 0)
            key = ("batched" if batched else "loop", "gaussian" if "<0>" in event.name else "lorentzian")
            if not segments or segments[-1] != key:
                segments.append(key)
        kind = "reduce" if "smear_reduce_kernel" in event.name else "partial"
        slot = times.setdefault(f"{segments[-1][0]}_{segments[-1][1]}", {"partial_ms": 0.0, "reduce_ms": 0.0,
                                                                          "launches": 0})
        slot[f"{kind}_ms"] += event.time_range.elapsed_us() / 1000.0
        slot["launches"] += 1
    return times


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def run(name, wn, rows):
    """rows: a (..., P) CUDA tensor of spectra on the CUDA wavenumbers wn."""
    flat = rows.reshape(-1, rows.shape[-1])
    count = flat.shape[0]
    results = []
    for function in ("gaussian", "lorentzian"):
        def batched():
            return rb.convolve_spectra(wn, rows, function, WIDTH)[1]

        def batched_device():
            return rb.convolve_spectra_device(wn, rows, function, WIDTH)[1]

        def loop():
            return [rb.convolve_spectrum(wn, flat[b], function, WIDTH)[1] for b in range(count)]

        for _ in range(2):  # warm-up of every shape
            batched()
            batched_device()
            loop()
        a_ms, d_ms, l_ms = [], [], []
        for _ in range(repeats):
            a_ms.append(timed(batched))
            d_ms.append(timed(batched_device))
            l_ms.append(timed(loop))
        got = batched().reshape(count, -1)
        got_device = batched_device().reshape(count, -1).cpu().numpy()
        want = np.stack(loop())
        pairs = evaluated_pairs(wn, default_grid(wn), function)
        result = {
            "case": name, "function": function, "width": WIDTH, "rows": count, "in_points": int(rows.shape[-1]),
            "out_points": int(got.shape[1]), "batched_ms": stats(a_ms), "batched_device_ms": stats(d_ms),
            "loop_ms": stats(l_ms), "speedup_numpy_output": float(np.median(l_ms) / np.median(a_ms)),
            "evaluated_pairs_per_row": pairs,
            "bit_identical": bool(np.array_equal(got, want) and np.array_equal(got_device, want)),
            "batched_runs_ms": a_ms, "batched_device_runs_ms": d_ms, "loop_runs_ms": l_ms,
        }
        print(json.dumps({k: v for k, v in result.items() if not k.endswith("runs_ms")}), flush=True)
        results.append(result)
    return results


CASES = ["(a) measure_windows, S = 1e6, window 2000, hop 500", "(b) measure_windows, S = 1e6, window 20000, hop 5000",
         "(c) measure_cross_spectra, G = 4, S = 1e6", "(d) one c3-sized spectrum, S = 1e6"]


def case_inputs(index):
    """(wavenumbers, rows) of case ``index``, both CUDA tensors."""
    if index == 2:
        series = synthetic_series(FRAMES, 2, count=4)
        return rb.measure_cross_spectra_device([rb.MDRamanSpectrum(series[g], 1.0) for g in range(4)])
    spectrum = rb.MDRamanSpectrum(synthetic_series(FRAMES, 1), 1.0)
    if index == 3:
        return spectrum.measure_device()
    return spectrum.measure_windows_device(*((2000, 500), (20000, 5000))[index])


def add_kernel_times(result, times):
    count = result["rows"]
    pairs = result["evaluated_pairs_per_row"]
    groups = 1 if count == 1 else -(-count // ROWS)
    batched, loop = times[f"batched_{result['function']}"], times[f"loop_{result['function']}"]
    result["batched_kernel"], result["loop_kernel"] = batched, loop
    result["batched_factor_evaluations_per_s"] = pairs * groups / (batched["partial_ms"] * 1e-3)
    result["batched_row_pairs_per_s"] = pairs * count / (batched["partial_ms"] * 1e-3)
    result["loop_factor_evaluations_per_s"] = pairs * count / (loop["partial_ms"] * 1e-3)


if PROFILE:
    print(json.dumps(profile_case(*case_inputs(int(sys.argv[2])))), flush=True)
    sys.exit(0)

results = []
for index, name in enumerate(CASES):
    results += run(name, *case_inputs(index))
    clear_plan_cache()
    torch.cuda.empty_cache()
for index, name in enumerate(CASES):  # kernel times: a profiler run of its own per case
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--profile", str(index)], capture_output=True,
                           text=True, check=False)
    for result in results:
        if result["case"] != name:
            continue
        if child.returncode == 0:
            add_kernel_times(result, json.loads(child.stdout.strip().splitlines()[-1]))
        else:
            result["kernel_error"] = child.stderr[-2000:]
            print(json.dumps({k: v for k, v in result.items() if not k.endswith("runs_ms")}), flush=True)

card, power = gpu_info()
record = {"what": "convolve_spectra (numpy output) and convolve_spectra_device against a loop of convolve_spectrum "
                  "over the rows, all from device inputs; default grid, width 5; CUDA events around each whole call, "
                  "the three forms alternated after warm-ups, medians of the repeats; kernel times from a torch.profiler "
                  "run of its own per case (one batched call and one loop per function); factor evaluations counted "
                  "from the shapes and the skip rule",
          "gpu": card, "power_limit": power, "repeats": repeats, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)
