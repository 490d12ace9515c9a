"""Windowed MD Raman spectra, timed on one GPU:
  A = a Python loop of MDRamanSpectrum(series[w*hop : w*hop+Lw], dt).measure_device() over the windows;
  B = MDRamanSpectrum(series, dt).measure_windows_device(Lw, hop): all windows in one batched transform.
A and B run alternately in the same process after warm-ups and are timed with CUDA events around the whole
call (launch gaps included).  Kernel time comes from a separate torch.profiler pass (sum of the device time
of every kernel of one call), and the transform rate is 3 W L points over it; the single-series
measure_device of the whole series is the yardstick (3 L points).  Rows of A and B are compared bit for bit.
python tools/run_windows.py [OUT.json] [REPEATS]"""
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ramannoodle_b200 as rb  # noqa: E402
from ramannoodle_b200.spectrum import _window_batch, clear_plan_cache, num_windows  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join("profiles", "r04_windows.json")
repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
device = torch.device("cuda:0")
rb._lib.require_device(0)  # pylint: disable=protected-access  (fails loudly without an sm_100 GPU)

SHAPES = [("spectrogram", 1_000_000, 2000, 500), ("spectrogram_wide", 1_000_000, 20_000, 5000),
          ("block_average", 10_000_000, 1_000_000, None)]


def chirp_length(frames):
    m, log2l = frames - 1, 12
    while (1 << log2l) < max(2 * m - 1, 4096):
        log2l += 1
    return 1 << log2l


def series_of(frames, seed):
    gen = torch.Generator(device).manual_seed(seed)
    steps = torch.arange(frames, dtype=torch.float64, device=device)[:, None, None]
    phase = torch.rand((1, 3, 3), dtype=torch.float64, device=device, generator=gen) * 6
    noise = torch.randn((frames, 3, 3), dtype=torch.float64, device=device, generator=gen)
    return 6.0 * torch.eye(3, dtype=torch.float64, device=device) + 0.05 * torch.sin(0.013 * steps + phase) + 0.01 * noise


def loop(series, window, hop):
    rows = []
    for w in range(num_windows(len(series), window, hop)):
        rows.append(rb.MDRamanSpectrum(series[w * hop: w * hop + window], 1.0).measure_device()[1])
    return rows


def batched(series, window, hop):
    return rb.MDRamanSpectrum(series, 1.0).measure_windows_device(window, hop)[1]


def whole(series):
    return rb.MDRamanSpectrum(series, 1.0).measure_device()[1]


def timed(fn):
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn()
    stop.record()
    torch.cuda.synchronize()
    return float(start.elapsed_time(stop))


def kernel_ms(fn):
    """Device time of every kernel fn() launches (torch.profiler, a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile  # pylint: disable=import-outside-toplevel

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total = 0.0
    for event in prof.key_averages():
        total += float(getattr(event, "self_device_time_total", getattr(event, "self_cuda_time_total", 0.0)))
    return total / 1000.0


def stats(values):
    return {"median": float(np.median(values)), "min": min(values), "max": max(values)}


def gpu_info():
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30, check=True).stdout.strip()
        name, power = (part.strip() for part in line.split(","))
        return name, power
    except (OSError, subprocess.SubprocessError, ValueError):
        return torch.cuda.get_device_name(0), "unknown"


results = []
for name, frames, window, hop_arg in SHAPES:
    hop = window if hop_arg is None else hop_arg
    series = series_of(frames, 7)
    windows = num_windows(frames, window, hop)
    for _ in range(2):  # warm-up: plans, kernel modules
        loop(series, window, hop)
        batched(series, window, hop)
        whole(series)
    a_ms, b_ms, y_ms = [], [], []
    for _ in range(repeats):
        a_ms.append(timed(lambda: loop(series, window, hop)))
        b_ms.append(timed(lambda: batched(series, window, hop)))
        y_ms.append(timed(lambda: whole(series)))
    same = bool(torch.equal(torch.stack(loop(series, window, hop)), batched(series, window, hop)))
    k_a, k_b, k_y = kernel_ms(lambda: loop(series, window, hop)), kernel_ms(lambda: batched(series, window, hop)), \
        kernel_ms(lambda: whole(series))
    length, whole_length = chirp_length(window), chirp_length(frames)
    points = 3 * windows * length
    results.append({
        "shape": name, "frames": frames, "window_frames": window, "hop_frames": hop, "windows": windows,
        "chirp_length": length, "batch": _window_batch(window, windows), "rows_bit_identical": same,
        "loop_ms": stats(a_ms), "batched_ms": stats(b_ms), "whole_series_measure_ms": stats(y_ms),
        "speedup_median": float(np.median(a_ms) / np.median(b_ms)),
        "kernel_ms": {"loop": k_a, "batched": k_b, "whole_series_measure": k_y},
        "transform_points_per_s": {"batched": points / (k_b * 1e-3), "loop": points / (k_a * 1e-3),
                                   "whole_series_measure": 3 * whole_length / (k_y * 1e-3)},
        "loop_runs_ms": a_ms, "batched_runs_ms": b_ms, "whole_series_runs_ms": y_ms})
    print(json.dumps(results[-1]), flush=True)
    del series
    clear_plan_cache()
    torch.cuda.empty_cache()

card, power = gpu_info()
record = {"what": "MDRamanSpectrum windows: A = per-window measure_device loop over slices, B = measure_windows_device "
                  "(one batched transform per chunk); CUDA events around each call, A and B alternated; kernel time "
                  "from a separate torch.profiler pass; series HBM-resident float64",
          "gpu": card, "power_limit": power, "repeats": repeats, "results": results}
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
with open(out_path, "w", encoding="utf-8") as handle:
    json.dump(record, handle, indent=1)
print(json.dumps({k: v for k, v in record.items() if k != "results"}), flush=True)
