"""Parity at BASELINE.json's own sizes: every bench configuration rendered for its full 10 s by the engine
(through the C ABI) and by the threaded oracle (oracle/sharded.py: the -O3 build, voices sharded over the host
cores), bus and >= 64 sampled pre-mix voice taps compared sample by sample.

    configs[1]  additive, 4096 SinWt partials x 10 s      taps bit-identical (integer phase), bus <= 1e-5
    configs[2]  subtractive, 16 384 voices x 10 s         taps <= 1e-4 (IIR budget), bus <= 1e-5
    configs[2B] the same with Envelope segments           taps <= 1e-4, bus <= 1e-5
    subtractive, 1024 voices x 10 s (render_sub_scan)    taps <= 1e-4, bus <= 1e-5
    configs[3]  FM, 8192 voices x 10 s                    carrier taps <= 1e-5 (oscillator budget), bus <= 1e-5

Tolerances are the north star's (BASELINE.json); what is measured is printed and is far tighter.  Ten seconds
matter: the f32 phase / envelope recurrences drift 4.4e-3 over 10 s if re-associated (SURVEY F5, App. C)."""
import numpy as np
import pytest

from knaster_b200.processor import AudioProcessor, AudioProcessorOptions
from oracle.sharded import ShardedOracle, bank_builder, sample_voices

pytestmark = pytest.mark.gpu
SR, BLOCK = 48000, 64
SECONDS = 10.0
N_BLOCKS = int(SECONDS * SR) // BLOCK
N_TAPS = 64


def full_size(workload, n_voices, kernel):
    build = bank_builder(workload, SECONDS)
    voices = sample_voices(n_voices, N_TAPS)
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions())
    ids = build(graph, n_voices, 0, n_voices)
    for v in voices:
        proc.add_tap(ids[v], 0)
    assert proc.info()["kernels"] == [kernel]
    gpu = proc.render(N_BLOCKS)
    gpu_taps = proc.read_taps()
    del proc
    ref, ref_taps = ShardedOracle(build, n_voices, tap_voices=voices).render(N_BLOCKS)
    assert np.abs(ref).max() > 1e-3 and np.abs(ref_taps).max(axis=1).min() > 0.0, "silent reference"
    bus_err = float(np.abs(gpu - ref).max())
    # every voice carries a gain of 1/n_voices (normalised bus, SURVEY H4): tap errors are judged at UNIT voice gain,
    # i.e. scaled by n_voices, so that the tolerance is not vacuous against a 6e-5 signal
    scale = float(n_voices)
    tap_err = np.abs(gpu_taps - ref_taps).max(axis=1) * scale
    # drift check: the last second must be as good as the first
    last = slice(-SR, None)
    tail_err = float(np.abs(gpu_taps[:, last] - ref_taps[:, last]).max()) * scale
    print(f"{workload}: {n_voices} voices x {SECONDS:g} s: max|bus| {np.abs(ref).max():.3f}, bus err {bus_err:.3e}, "
          f"tap err at unit voice gain max {tap_err.max():.3e} (last second {tail_err:.3e}), taps bit-identical: {int((tap_err == 0).sum())}/{len(voices)}")
    return bus_err, tap_err, tail_err


def test_config1_additive_4096_partials_10s():
    bus_err, tap_err, _ = full_size("additive", 4096, "render_add_wt")
    assert tap_err.max() == 0.0          # integer phase, per-partial gain ramp in f64 on the host: bit-identical
    assert bus_err <= 1e-5


def test_config2_subtractive_16384_voices_10s():
    bus_err, tap_err, tail = full_size("subtractive", 16384, "render_sub_asr")
    assert tap_err.max() <= 1e-4 and tail <= 1e-4
    assert bus_err <= 1e-5


def test_subtractive_1024_voices_10s_on_the_scan_kernel():
    # the largest bank the time-parallel kernel takes: the scan re-associates the filter's sums, so the IIR budget, over 10 s
    bus_err, tap_err, tail = full_size("subtractive", 1024, "render_sub_scan")
    assert tap_err.max() <= 1e-4 and tail <= 1e-4
    assert bus_err <= 1e-5


def test_config2b_subtractive_envelope_segments_16384_voices_10s():
    bus_err, tap_err, tail = full_size("subtractive_seg", 16384, "render_sub_seg")
    assert tap_err.max() <= 1e-4 and tail <= 1e-4
    assert bus_err <= 1e-5


def test_config3_fm_8192_voices_10s():
    bus_err, tap_err, tail = full_size("fm", 8192, "render_fm2")
    assert tap_err.max() <= 1e-5 and tail <= 1e-5
    assert bus_err <= 1e-5
