"""Audio-rate routes into the float parameters that were added last (WrArParams, audio_rate.rs:42-57): Pan2 pan (pan.rs:26-36),
Phasor freq (osc.rs:191-197), RandomLin freq (noise.rs:206-213) and Envelope time_scale (envelopes.rs:477-479), and nodes with
every float parameter routed at once (an SvfFilter Bell: cutoff, q, gain and three wr_mul values; a SinNumeric: freq,
phase_offset and its wr_mul).  knaster calls param_apply with the routed sample before every frame; the kernels do the same
arithmetic (f32 / f64 restatements of the host setters, fastapprox.h for the pan law), so the taps of every shape but the
filter's are bit-identical to the oracle.  The filter recomputes tanf / powf per frame and is held to the 1e-4 budget of
tests/test_gpu_ar_filters.py."""
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200.graph import Graph
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions, Snapshot

pytestmark = pytest.mark.gpu
SR = 48000
N_VOICES = 12
N_BLOCKS = 7500                                       # 10 s at 64 frames


def at(f):
    return kn.Seconds.from_samples(int(f), SR)


# ---- voice shapes: each returns (signal, [(node, channel) to tap]) ----------------------------------------------------------
def pan_lfo(g, i):
    src = g.push(kn.SinWt(220.0 + 31.0 * i).wr_mul(0.5))
    lfo = g.push(kn.SinWt(0.5 + 0.37 * i))
    pan = g.push(kn.Pan2(0.25).ar_params())
    pan.link("pan", lfo * (0.6 + 0.07 * i))               # voices 6.. swing past +-1: the pan law outside its range
    pan.param("pan").set_at(-0.5, at(20000 + 7 * i))     # ignored while routed (audio_rate.rs:70-74)
    sig = src >> pan
    return sig, [(pan.id(), 0), (pan.id(), 1)]


def phasor_lfo(g, i):
    lfo = g.push(kn.SinWt(0.7 + 0.3 * i))
    ph = g.push(kn.Phasor(100.0).ar_params())
    depth, centre = (300.0, 100.0) if i % 4 == 3 else (50.0 + 10.0 * i, 200.0 + 40.0 * i)   # i % 4 == 3: negative rates too
    ph.link("freq", lfo * depth + centre)
    ph.param("freq").set_at(5.0, at(30000 + i))
    return ph * (1.0 / N_VOICES), [(ph.id(), 0)]


def randlin_lfo(g, i):
    lfo = g.push(kn.SinWt(0.4 + 0.2 * i))
    rl = g.push(kn.RandomLin(10.0).ar_params())
    rl.link("freq", lfo * (20.0 + 5.0 * i) + (40.0 + 30.0 * i))
    rl.param("freq").set_at(1.0, at(25000 + i))
    return rl * (1.0 / N_VOICES), [(rl.id(), 0)]


def envelope_time_scale(g, i):
    lfo = g.push(kn.SinWt(1.1 + 0.3 * i))
    env = g.push(kn.Envelope(0.0, [kn.EnvelopeSegment(0.05 + 0.01 * i, 1.0), kn.EnvelopeSegment(0.2, 0.3),
                                   kn.EnvelopeSegment(0.4, 0.0)]).looping(i % 2 == 0).ar_params())
    env.link("time_scale", lfo * 0.5 + (1.0 + 0.1 * i))
    for k in range(6):
        env.param("t_restart").trig_at(at(1000 + 70000 * k + 13 * i))
    env.param("time_scale").set_at(3.0, at(50000 + i))
    env.param("t_stop").trig_at(at(400000 + 11 * i))
    return env * (1.0 / N_VOICES), [(env.id(), 0)]


def svf_bell_all_routes(g, i):
    """all six float parameters of an SvfFilter: cutoff, q, gain and the values of its three WrMul wrappers"""
    saw = g.push(kn.PolyBlep(kn.Waveform.Sawtooth, 90.0 + 23.0 * i))
    lfo = g.push(kn.SinWt(0.9 + 0.4 * i))
    ph = g.push(kn.Phasor(0.3 + 0.1 * i))
    lfo2 = g.push(kn.SinWt(2.0 + 0.5 * i))
    svf = g.push(kn.SvfFilter(kn.SvfFilterType.Bell, 1000.0, 1.0, 0.0).wr_mul(1.0).wr_mul(1.0).wr_mul(1.0).ar_params())
    svf.link("cutoff_freq", lfo * (300.0 + 50.0 * i) + (1200.0 + 100.0 * i))
    svf.link("q", ph + 0.7)
    svf.link("gain", lfo * (6.0 + 0.5 * i))
    svf.link(5, ph)
    svf.link(6, lfo2)
    svf.link(7, lfo)
    sig = saw >> svf
    return sig * (1.0 / N_VOICES), [(svf.id(), 0)]


def sinnum_all_routes(g, i):
    """SinNumeric freq, phase_offset and wr_mul together"""
    lfo = g.push(kn.SinWt(3.0 + 0.5 * i))
    lfo2 = g.push(kn.SinWt(0.25 + 0.1 * i))
    ph = g.push(kn.Phasor(0.2 + 0.05 * i))
    sn = g.push(kn.SinNumeric(300.0).wr_mul(1.0).ar_params())
    sn.link("freq", lfo * (30.0 + 4.0 * i) + (200.0 + 50.0 * i))
    sn.link("phase_offset", lfo2)
    sn.link("wr_mul", ph)
    sn.param("freq").set_at(1000.0, at(10000 + i))
    return sn * (1.0 / N_VOICES), [(sn.id(), 0)]


SHAPES = [pan_lfo, phasor_lfo, randlin_lfo, envelope_time_scale, svf_bell_all_routes, sinnum_all_routes]
EXACT = {pan_lfo, phasor_lfo, randlin_lfo, envelope_time_scale, sinnum_all_routes}


def to_out(shape, sig):
    if shape is pan_lfo:
        sig.to_graph_out()                              # stereo already
    else:
        sig.out([0, 0]).to_graph_out()


def build_voices(graph, shape, n=N_VOICES):
    kn.reset_randomness_seed(0)                         # RandomLin seeds: the engine and the oracle draw the same streams
    taps = []
    with graph.edit() as g:
        for i in range(n):
            sig, t = shape(g, i)
            to_out(shape, sig)
            taps += t
    return taps


def engine_render(shape, n_blocks, jit):
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_jit=jit, force_interpreter=not jit))
    taps = build_voices(graph, shape)
    for node, ch in taps:
        proc.add_tap(node, ch)
    out = proc.render(n_blocks)
    return out, proc.read_taps(), proc


@pytest.fixture(scope="module")
def oracle_renders():
    from oracle.oracle import OracleProcessor

    cache = {}

    def get(shape):
        if shape not in cache:
            g = Graph(0, 2, 64, SR)
            taps = build_voices(g, shape)
            orc = OracleProcessor(g, ring_buffer_size=1 << 22)
            for node, ch in taps:
                orc.add_tap(node, ch)
            cache[shape] = orc.render(N_BLOCKS)
        return cache[shape]

    return get


@pytest.fixture(scope="module")
def engine_renders():
    cache = {}

    def get(shape, jit):
        if (shape, jit) not in cache:
            out, taps, proc = engine_render(shape, N_BLOCKS, jit)
            cache[(shape, jit)] = (out, taps, proc.info()["kernels"])
        return cache[(shape, jit)]

    return get


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: s.__name__)
@pytest.mark.parametrize("jit", [False, True])
def test_routes_against_the_oracle(shape, jit, oracle_renders, engine_renders):
    out, taps, kernels = engine_renders(shape, jit)
    assert all(k == ("render_jit" if jit else "render_interp") for k in kernels), kernels
    ref, ref_taps = oracle_renders(shape)
    assert np.isfinite(ref_taps).all() and np.abs(ref_taps).max() > 1e-2
    assert taps.shape == ref_taps.shape
    if shape in EXACT:
        bad = np.count_nonzero(taps.view(np.uint32) != ref_taps.view(np.uint32))
        assert bad == 0, f"{shape.__name__} jit={jit}: {bad} of {taps.size} tap samples differ from the oracle"
    else:
        err = np.abs(taps - ref_taps) / np.maximum(1.0, np.abs(ref_taps).max(axis=1, keepdims=True))   # the filter's tap: unit gain
        print(f"{shape.__name__} jit={jit}: max err at unit voice gain {err.max():.3e} (last second {err[:, -SR:].max():.3e})")
        assert err.max() <= 1e-4
    assert np.abs(out - ref).max() <= 1e-5 * max(1.0, float(np.abs(ref).max()))


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: s.__name__)
def test_generated_kernel_equals_the_interpreter(shape, engine_renders):
    out_i, taps_i, _ = engine_renders(shape, False)
    out_j, taps_j, _ = engine_renders(shape, True)
    assert np.array_equal(taps_i.view(np.uint32), taps_j.view(np.uint32))
    assert np.abs(out_i - out_j).max() <= 1e-6 * max(1.0, float(np.abs(out_i).max()))   # the bus sums differ in order only


def all_shapes(graph, n_per_shape=2):
    kn.reset_randomness_seed(0)
    taps = []
    with graph.edit() as g:
        for shape in SHAPES:
            for i in range(n_per_shape):
                sig, t = shape(g, 5 * i + 1)
                to_out(shape, sig)
                taps += t
    return taps


def new_all_shapes(jit):
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_jit=jit, force_interpreter=not jit))
    taps = all_shapes(graph)
    for node, ch in taps:
        proc.add_tap(node, ch)
    return graph, proc


@pytest.mark.parametrize("jit", [False, True])
def test_split_invariance_with_routes(jit):
    n_blocks = 1500
    _, p1 = new_all_shapes(jit)
    one = p1.render(n_blocks)
    one_taps = p1.read_taps()
    assert set(p1.info()["kernels"]) == {"render_jit" if jit else "render_interp"}
    _, p7 = new_all_shapes(jit)
    p7.set_blocks_per_launch(7)
    assert np.array_equal(p7.render(n_blocks), one)
    assert np.array_equal(p7.read_taps(), one_taps)
    # render_block (run_without_inputs) block by block equals the batched render, taps included
    n_bb = 300
    _, pb = new_all_shapes(jit)
    outs, taps = [], []
    for _ in range(n_bb):
        pb.run_without_inputs()
        outs.append(pb.output_block())
        taps.append(pb.read_taps())
    assert np.array_equal(np.stack(outs), one[:n_bb])
    assert np.array_equal(np.concatenate(taps, axis=1), one_taps[:, : n_bb * 64])


@pytest.mark.parametrize("jit", [False, True])
def test_snapshot_restored_into_a_fresh_processor_continues_bit_identically(jit):
    _, p1 = new_all_shapes(jit)
    first = p1.render(777)                              # mid-note, mid-segment, mid-ramp
    image = p1.snapshot().to_bytes()
    cont = p1.render(700)
    cont_taps = p1.read_taps()
    g2, p2 = new_all_shapes(jit)
    g2.take_events()                                    # its events are inside the image
    p2.restore(Snapshot.from_bytes(image))
    assert p2.frame_clock() == 777 * 64
    assert np.array_equal(p2.render(700), cont)
    assert np.array_equal(p2.read_taps(), cont_taps)
    assert np.abs(first).max() > 1e-3


# ---- the pan law on the device: every float, against the host instantiation of the same header --------------------------------
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NVCC = os.environ.get("NVCC", shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc")
# the library's numeric flags (knaster_b200/csrc/Makefile), host side as plan.cpp is built
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-prec-div=true", "-prec-sqrt=true",
         "-ftz=false", "-Xcompiler", "-ffp-contract=off,-fno-fast-math"]


def test_device_pan_law_equals_the_host_for_every_float(tmp_path):
    exe = tmp_path / "pan2_exhaustive"
    subprocess.run([NVCC, *FLAGS, "-I" + os.path.join(ROOT, "knaster_b200", "csrc"), os.path.join(ROOT, "tools", "pan2_exhaustive.cu"),
                    "-o", str(exe), "-lpthread"], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True, timeout=900).stdout
    print(out.strip())
    r = json.loads(out.strip().splitlines()[-1])
    assert r["arguments"] == 1 << 32
    assert r["mismatches"] == 0, r
    assert r["nan"] > 0 and r["finite"] > 0
