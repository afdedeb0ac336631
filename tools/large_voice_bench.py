"""Banks of voices larger than 24 nodes on render_interp and render_jit.

Two voice shapes (knaster_b200/banks.py), four notes per voice per 10 s step (EnvAsr t_restart / t_release at any frame):
  partials   32 x SinWt.wr_mul -> Add chain -> SvfFilter -> * EnvAsr.wr_mul(1/N)       66 nodes per voice
  operators  saw -> 12 x (x * a + b) -> SvfFilter -> * EnvAsr.wr_mul(1/N)             52 nodes per voice
at 1024 and 16 384 voices.  Each bank runs on the interpreter and on the generated kernel; --grp 4,8,16 adds one generated
kernel per frames-per-group value (KGPU_JIT_GRP) to choose the default of templates over 24 nodes.  Prints, per row: ms per
step (wall clock around render(), which ends in a device synchronise), the voice kernels' ms (CUDA events), voice-samples/s
and node-samples/s from the kernel time, and the kernel name; then the GPU name and power limit read in the same run.
Generated kernels are cached in a temporary directory unless KGPU_JIT_CACHE is set.

usage: python tools/large_voice_bench.py [--steps 2] [--warmup 1] [--seconds 10] [--voices 1024,16384] [--grp 4,8,16]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from knaster_b200 import banks  # noqa: E402
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions  # noqa: E402

SR, BS = 48000, 64
NOTES_PER_STEP = 4
BANKS = {"partials": (banks.partials_bank, 2 * 32 + 2), "operators": (banks.operator_bank, 4 * 12 + 4)}


def measure(bank, n, arm, grp, seconds, steps, warmup):
    build, nodes = BANKS[bank]
    n_blocks = int(seconds * SR) // BS
    if grp:
        os.environ["KGPU_JIT_GRP"] = str(grp)
    else:
        os.environ.pop("KGPU_JIT_GRP", None)
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, block_size=BS, force_interpreter=arm == "interp",
                                                                 force_jit=arm == "jit"))
    total = warmup + steps
    build(graph, n, seconds * total, n_notes=NOTES_PER_STEP * total)   # the notes of every step, scheduled up front
    wall, kern = [], []
    for s in range(total):
        t = time.perf_counter()
        out = proc.render(n_blocks)
        dt = (time.perf_counter() - t) * 1e3
        if s >= warmup:
            wall.append(dt)
            kern.append(proc.last_kernel_ms(0)[0])
    os.environ.pop("KGPU_JIT_GRP", None)
    assert np.isfinite(out).all() and np.abs(out).max() > 1e-4
    kernels = sorted(set(proc.info()["kernels"]))
    ms, kms = float(np.median(wall)), float(np.median(kern))
    vs = n * n_blocks * BS / (kms * 1e-3)
    return {"bank": bank, "voices": n, "nodes_per_voice": nodes, "kernels": kernels, "grp": grp or "default",
            "ms_per_step": round(ms, 2), "voice_kernel_ms": round(kms, 2), "voice_kernel_ms_all": [round(x, 2) for x in kern],
            "voice_samples_per_s": float(f"{vs:.4g}"), "node_samples_per_s": float(f"{vs * nodes:.4g}")}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--voices", default="1024,16384")
    ap.add_argument("--grp", default="", help="comma-separated frames per group to measure the generated kernel at besides its default")
    a = ap.parse_args()
    os.environ.setdefault("KGPU_JIT_CACHE", tempfile.mkdtemp(prefix="knaster_jit_"))
    grps = [int(x) for x in a.grp.split(",") if x]
    rows = []
    for bank in BANKS:
        for n in (int(x) for x in a.voices.split(",")):
            for arm, grp in [("interp", 0), ("jit", 0)] + [("jit", g) for g in grps]:
                row = measure(bank, n, arm, grp, a.seconds, a.steps, a.warmup)
                rows.append(row)
                print(json.dumps(row), flush=True)
    print(f"gpu: {gpu_info()}")
    for r in rows:
        print(f"{r['bank']:9s} {r['voices']:6d} voices  {r['kernels'][0]:13s} grp {str(r['grp']):7s}  kernel {r['voice_kernel_ms']:9.2f} ms/step  "
              f"{r['voice_samples_per_s']:.3g} voice-samples/s  {r['node_samples_per_s']:.3g} node-samples/s")


if __name__ == "__main__":
    main()
