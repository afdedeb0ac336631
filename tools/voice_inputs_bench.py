"""Input-track bank: 16 384 graph inputs, each through its own effect chain -- input_i -> SvfFilter(Low, per-voice cutoff) ->
* EnvAsr.wr_mul(1/N) (8 notes per voice per 10 s) -> Pan2 -> bus (knaster_b200.banks.input_bank).  Every input is a port of
the one voice template: render_jit reads it in place from the caller's input blocks [block][input][frame].
Arms, 10-second steps (seeded noise plus a sine per track as the input):
  device   inputs already in device memory (kgpu_render_inputs_device): 31.5 GB read per step
  host     inputs in host memory (kgpu_render_inputs): staged through page-locked memory launch by launch
  saw      the same bank with a PolyBlep saw per voice in place of the input: what the chain costs without input reads
Prints per arm: voice-kernel ms (CUDA events) and end-to-end ms per step (wall clock around the call and a device
synchronise), voice-samples/s, input bytes/s against the 7.7 TB/s of HBM3e, host-to-device bytes/s for the host arm, and the
card's name and power limit, read in the same run.

usage: python tools/voice_inputs_bench.py [--voices 16384] [--seconds 10] [--host-seconds 10] [--steps 3] [--warmup 1]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from knaster_b200 import banks  # noqa: E402
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions  # noqa: E402

SR, BS = 48000, 64
HBM_BYTES_PER_S = 7.7e12


def device_tracks(n, n_blocks, seed=99):
    """[n_blocks][n][BS] f32 on the device: 0.3 sin(2 pi f t) + 0.1 noise, f per track"""
    import torch

    gen = torch.Generator(device="cuda").manual_seed(seed)
    f = 55.0 * 2.0 ** (torch.rand(n, generator=gen, device="cuda", dtype=torch.float64) * 6.0)
    x = torch.empty((n_blocks, n, BS), dtype=torch.float32, device="cuda")
    for b0 in range(0, n_blocks, 250):
        b1 = min(n_blocks, b0 + 250)
        t = torch.arange(b0 * BS, b1 * BS, device="cuda", dtype=torch.float64).reshape(b1 - b0, 1, BS) / SR
        x[b0:b1] = (0.3 * torch.sin(2.0 * np.pi * f.reshape(1, -1, 1) * t)
                    + 0.1 * torch.randn((b1 - b0, n, BS), generator=gen, device="cuda", dtype=torch.float64)).float()
    return x


def notes(graph, env_ids, n, step, n_frames, seed=11):
    """8 notes per voice in the step's window"""
    r = np.random.Generator(np.random.PCG64(seed + step))
    t0 = step * n_frames
    on = np.sort(r.integers(0, n_frames - SR // 2, (n, 8)), axis=1) + t0
    off = on + SR // 4
    banks._notes(graph, env_ids, on, off, t0 + n_frames)


def measure(arm, n, seconds, steps, warmup, x_dev=None, x_host=None):
    import torch

    n_blocks = int(seconds * SR) // BS
    n_frames = n_blocks * BS
    graph, proc = AudioProcessor.new(0 if arm == "saw" else n, 2, AudioProcessorOptions(sample_rate=SR, block_size=BS))
    ids = banks.input_bank(graph, n, seconds, n_notes=0, source="saw" if arm == "saw" else "input")
    out = torch.zeros((n_blocks, 2, BS), dtype=torch.float32, device="cuda")
    wall, kern = [], []
    for s in range(warmup + steps):
        notes(graph, ids["env"], n, s, n_frames)
        torch.cuda.synchronize()
        t = time.perf_counter()
        if arm == "device":
            proc.render_device(n_blocks, out.data_ptr(), inputs_device_ptr=x_dev.data_ptr())
            proc.synchronize()
        elif arm == "saw":
            proc.render_device(n_blocks, out.data_ptr())
            proc.synchronize()
        else:
            host_out = proc.render(n_blocks, inputs=x_host)
        dt = (time.perf_counter() - t) * 1e3
        if s >= warmup:
            wall.append(dt)
            kern.append(proc.last_kernel_ms(0)[0])
    bus = host_out if arm == "host" else out.cpu().numpy()
    assert np.isfinite(bus).all() and np.abs(bus).max() > 1e-4
    ms, kms = float(np.median(wall)), float(np.median(kern))
    in_bytes = 0 if arm == "saw" else n * n_frames * 4
    row = {"arm": arm, "voices": n, "seconds": seconds, "kernels": sorted(set(proc.info()["kernels"])),
           "ms_per_step": round(ms, 2), "ms_per_step_all": [round(v, 2) for v in wall], "voice_kernel_ms": round(kms, 2),
           "voice_samples_per_s": n * n_frames / (ms * 1e-3), "voice_samples_per_s_kernel": n * n_frames / (kms * 1e-3)}
    if in_bytes:
        row["input_bytes_per_step"] = in_bytes
        row["input_bytes_per_s_kernel"] = in_bytes / (kms * 1e-3)
        row["input_share_of_hbm_peak"] = round(in_bytes / (kms * 1e-3) / HBM_BYTES_PER_S, 4)
    if arm == "host":
        row["h2d_bytes_per_s"] = in_bytes / (ms * 1e-3)
    return row


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        return "nvidia-smi unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--voices", type=int, default=16384)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--host-seconds", type=float, default=10.0)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this benchmark measures the GPU")
    n = a.voices
    rows = []
    x = device_tracks(n, int(a.seconds * SR) // BS)
    rows.append(measure("device", n, a.seconds, a.steps, a.warmup, x_dev=x))
    print(json.dumps(rows[-1]), flush=True)
    x_host = x[: int(a.host_seconds * SR) // BS].cpu().numpy()
    del x
    torch.cuda.empty_cache()
    rows.append(measure("host", n, a.host_seconds, a.steps, a.warmup, x_host=x_host))
    print(json.dumps(rows[-1]), flush=True)
    del x_host
    rows.append(measure("saw", n, a.seconds, a.steps, a.warmup))
    print(json.dumps(rows[-1]), flush=True)
    print(f"gpu: {gpu_info()}")
    dev, host, saw = rows
    print(f"{n} tracks x {a.seconds:g} s: device-fed kernel {dev['voice_kernel_ms']} ms ({dev['input_share_of_hbm_peak'] * 100:.1f} % of "
          f"7.7 TB/s in input reads), end to end {dev['ms_per_step']} ms; saw in place of the input: kernel {saw['voice_kernel_ms']} ms; "
          f"host-fed {a.host_seconds:g} s: {host['ms_per_step']} ms end to end, {host['h2d_bytes_per_s'] / 1e9:.1f} GB/s host to device")


if __name__ == "__main__":
    main()
