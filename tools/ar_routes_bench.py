"""Auto-pan bank: the cost of driving Pan2's `pan` at audio rate.

N voices of PolyBlep saw -> SvfFilter(Low) -> * EnvAsr.wr_mul(1/N) -> Pan2 -> stereo out, with four notes per voice and
10-second steps.  Two arms of the same bank:
  routed   Pan2.ar_params() with a per-voice SinWt LFO linked into `pan`: fastapprox sin + cos every frame on the device
  events   Pan2 with `pan` set by eight events per voice and step (the host evaluates the gains)
Sizes: 16 384 voices on render_jit (the generated kernel of banks >= 256 voices) and 256 voices on render_interp.
Prints, per arm: ms per 10 s step (wall clock around render(), which ends in a device synchronise), the voice kernels' ms
(CUDA events), voice-samples/s and the kernel name, plus the GPU name and power limit read in the same run.

usage: python tools/ar_routes_bench.py [--steps 3] [--warmup 1] [--seconds 10]
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
import knaster_b200 as kn  # noqa: E402
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions  # noqa: E402

SR, BS = 48000, 64
FLOAT, TRIG = 1, 2


def build(graph, n, routed, seed=7):
    r = np.random.Generator(np.random.PCG64(seed))
    f0 = 55.0 * 2.0 ** r.uniform(0.0, 5.0, n)
    fc = r.uniform(300.0, 6000.0, n)
    q = r.uniform(0.5, 4.0, n)
    rate = r.uniform(0.1, 2.0, n)
    ids = {"env": [], "pan": []}
    with graph.edit() as g:
        for i in range(n):
            saw = g.push(kn.PolyBlep(kn.Waveform.Sawtooth, float(f0[i])))
            svf = g.push(kn.SvfFilter(kn.SvfFilterType.Low, float(fc[i]), float(q[i]), 0.0))
            env = g.push(kn.EnvAsr(0.01, 0.3).wr_mul(1.0 / n))
            pan = g.push(kn.Pan2(0.0).ar_params() if routed else kn.Pan2(0.0))
            if routed:
                pan.link("pan", g.push(kn.SinWt(float(rate[i]))))
            ((saw >> svf) * env >> pan).to_graph_out()
            ids["env"].append(env.id())
            ids["pan"].append(pan.id())
    return {k: np.asarray(v, dtype=np.uint32) for k, v in ids.items()}


def schedule(graph, ids, n, step, n_frames, routed, seed):
    """four notes per voice in the step's window; the events arm also moves `pan` eight times"""
    r = np.random.Generator(np.random.PCG64(seed + step))
    t0 = step * n_frames
    on = np.sort(r.integers(0, n_frames - SR // 2, (n, 4)), axis=1) + t0
    off = on + SR // 4
    voice = [np.repeat(np.arange(n), 4)] * 2
    nodes = [np.repeat(ids["env"], 4), np.repeat(ids["env"], 4)]
    params = [np.full(n * 4, 3), np.full(n * 4, 2)]              # EnvAsr t_restart / t_release
    kinds = [np.full(n * 4, TRIG), np.full(n * 4, TRIG)]
    vals = [np.zeros(n * 4), np.zeros(n * 4)]
    frames = [on.reshape(-1), off.reshape(-1)]
    if not routed:
        pf = np.sort(r.integers(0, n_frames, (n, 8)), axis=1) + t0
        voice.append(np.repeat(np.arange(n), 8))
        nodes.append(np.repeat(ids["pan"], 8)); params.append(np.zeros(n * 8)); kinds.append(np.full(n * 8, FLOAT))
        vals.append(r.uniform(-1.0, 1.0, n * 8)); frames.append(pf.reshape(-1))
    voice, nodes, params, kinds, vals, frames = (np.concatenate(x) for x in (voice, nodes, params, kinds, vals, frames))
    order = np.lexsort((frames, voice))                          # voice by voice, each in time order
    graph.schedule_bulk(nodes[order], params[order], kinds[order], vals[order], frames[order].astype(np.uint64))


def measure(n, routed, interp, seconds, steps, warmup):
    n_blocks = int(seconds * SR) // BS
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, block_size=BS, force_interpreter=interp,
                                                                 force_jit=not interp))
    ids = build(graph, n, routed)
    wall, kern = [], []
    for s in range(warmup + steps):
        schedule(graph, ids, n, s, n_blocks * BS, routed, seed=11)
        t = time.perf_counter()
        out = proc.render(n_blocks)
        dt = (time.perf_counter() - t) * 1e3
        if s >= warmup:
            wall.append(dt)
            kern.append(proc.last_kernel_ms(0)[0])
    assert np.isfinite(out).all() and np.abs(out).max() > 1e-4
    k = proc.info()["kernels"]
    ms = float(np.median(wall))
    kms = float(np.median(kern))
    return {"voices": n, "arm": "routed" if routed else "events", "kernels": sorted(set(k)), "ms_per_step": round(ms, 2),
            "ms_per_step_all": [round(x, 2) for x in wall], "voice_kernel_ms": round(kms, 2),
            "voice_samples_per_s": n * n_blocks * BS / (ms * 1e-3), "voice_samples_per_s_kernel": n * n_blocks * BS / (kms * 1e-3)}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--jit-voices", type=int, default=16384)
    ap.add_argument("--interp-voices", type=int, default=256)
    a = ap.parse_args()
    rows = []
    for n, interp in ((a.jit_voices, False), (a.interp_voices, True)):
        for routed in (False, True):
            row = measure(n, routed, interp, a.seconds, a.steps, a.warmup)
            rows.append(row)
            print(json.dumps(row), flush=True)
    info = gpu_info()
    print(f"gpu: {info}")
    for n, interp in ((a.jit_voices, False), (a.interp_voices, True)):
        ev, ro = [r for r in rows if r["voices"] == n]
        print(f"{n} voices ({ro['kernels'][0]}): pan by events {ev['ms_per_step']} ms/step (kernel {ev['voice_kernel_ms']} ms), "
              f"pan routed {ro['ms_per_step']} ms/step (kernel {ro['voice_kernel_ms']} ms); routed kernel / events kernel "
              f"{ro['voice_kernel_ms'] / ev['voice_kernel_ms']:.3f}")


if __name__ == "__main__":
    main()
