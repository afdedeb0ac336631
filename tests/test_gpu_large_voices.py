"""Voices beyond 24 nodes, 192 registers and 24 value slots, up to the limits of dev.h (128 nodes, 1024 registers, 32 slots):
an additive voice of 32 partials with its own partial sum, a voice of builder arithmetic (12 x `x * a + b`), a voice of
exactly 128 nodes, a voice with 32 live value slots, and the segment-envelope voice of render_sub_seg with a 167-segment
Envelope, which brings the voice to exactly 1024 registers (the interpreter keeps them in more than 48 KB of shared memory).
Every shape plays notes (t_restart / t_release, or t_restart / t_stop) at frames that are not block-aligned.  Both kernels
evaluate each voice sequentially in the reference's order, so the taps are bit-identical to the oracle; the generated kernel
equals the interpreter bit for bit."""
import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200 import banks
from knaster_b200.graph import Graph
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions, Snapshot

pytestmark = pytest.mark.gpu
SR = 48000
SECONDS = 2.0
N_BLOCKS = int(SECONDS * SR) // 64


def at(f):
    return kn.Seconds.from_samples(int(f), SR)


# ---- voice shapes: build(graph, n) -> one tap (node id) per voice ---------------------------------------------------------
def partials(graph, n):
    """32 x SinWt.wr_mul -> Add chain -> SvfFilter -> * EnvAsr: 66 nodes, 142 registers"""
    return banks.partials_bank(graph, n, SECONDS)


def operators(graph, n):
    """saw -> 12 x (x * a + b) -> SvfFilter -> * EnvAsr: 52 nodes"""
    return banks.operator_bank(graph, n, SECONDS)


def nodes_128(graph, n):
    """saw -> 31 x (x * a + b) -> SvfFilter -> * EnvAsr: 128 nodes, the limit"""
    return banks.operator_bank(graph, n, SECONDS, n_ops=31)


def slots_32(graph, n):
    """32 SinWt partials combined by a right-nested chain p0 - (p1 - (... - p31)): the voice's post-order evaluates all 32
    partials before the first subtraction, so 32 values are live at once (the limit); then * EnvAsr.  65 nodes."""
    taps = []
    with graph.edit() as g:
        for i in range(n):
            ps = [g.push(kn.SinWt(60.0 * (1 + i % 5) * (k + 1) + 0.37 * k).wr_mul(0.5 / (k + 1))) for k in range(32)]
            acc = ps[-1]
            for p in reversed(ps[:-1]):
                acc = p - acc
            env = g.push(kn.EnvAsr(0.005 + 0.001 * i, 0.1).wr_mul(1.0 / n))
            sig = acc * env
            sig.out([0, 0]).to_graph_out()
            for k in range(3):
                env.param("t_restart").trig_at(at(1001 + 29000 * k + 13 * i))
                env.param("t_release").trig_at(at(15003 + 29000 * k + 7 * i))
            taps.append(sig._outputs[0][0])
    return taps


N_SEG = 167


def envelope_167(graph, n):
    """render_sub_seg's voice -- saw -> SvfFilter -> * Envelope.wr_mul -- with a 167-segment Envelope: 5 + 8 + 8 + 6 * 167 + 1
    = 1024 registers, the limit; notes by t_restart / t_stop"""
    taps = []
    with graph.edit() as g:
        for i in range(n):
            saw = g.push(kn.PolyBlep(kn.Waveform.Sawtooth, 80.0 + 17.0 * i))
            svf = g.push(kn.SvfFilter(kn.SvfFilterType.Low, 1500.0 + 100.0 * i, 1.0, 0.0))
            segs = [kn.EnvelopeSegment(0.002 + 0.0003 * ((k * 7 + i) % 11), ((k * 37 + i) % 19) / 19.0) for k in range(N_SEG)]
            env = g.push(kn.Envelope(0.0, segs).looping(i % 3 == 0).wr_mul(1.0 / n))
            sig = (saw >> svf) * env
            sig.out([0, 0]).to_graph_out()
            for k in range(3):
                env.param("t_restart").trig_at(at(999 + 30000 * k + 11 * i))
                env.param("t_stop").trig_at(at(21001 + 30000 * k + 5 * i))
            taps.append(sig._outputs[0][0])
    return taps


SHAPES = {partials: 64, operators: 32, nodes_128: 16, slots_32: 16, envelope_167: 32}
# per shape: the kernel of each arm ("interp": KGPU_PLAN_FORCE_INTERPRETER; "other": KGPU_PLAN_FORCE_JIT, where the hand-written
# render_sub_seg takes its own shape)
KERNELS = {"interp": lambda s: "render_interp", "other": lambda s: "render_sub_seg" if s is envelope_167 else "render_jit"}


def new_processor(arm):
    return AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_jit=arm == "other", force_interpreter=arm == "interp"))


def engine_render(shape, arm):
    graph, proc = new_processor(arm)
    taps = shape(graph, SHAPES[shape])
    for node in taps:
        proc.add_tap(node, 0)
    out = proc.render(N_BLOCKS)
    return out, proc.read_taps(), proc.info()["kernels"]


@pytest.fixture(scope="module")
def oracle_renders():
    from oracle.oracle import OracleProcessor

    cache = {}

    def get(shape):
        if shape not in cache:
            g = Graph(0, 2, 64, SR)
            taps = shape(g, SHAPES[shape])
            orc = OracleProcessor(g, ring_buffer_size=1 << 22)
            for node in taps:
                orc.add_tap(node, 0)
            cache[shape] = orc.render(N_BLOCKS)
        return cache[shape]

    return get


@pytest.fixture(scope="module")
def engine_renders():
    cache = {}

    def get(shape, arm):
        if (shape, arm) not in cache:
            cache[(shape, arm)] = engine_render(shape, arm)
        return cache[(shape, arm)]

    return get


@pytest.mark.parametrize("shape", list(SHAPES), ids=lambda s: s.__name__)
@pytest.mark.parametrize("arm", ["interp", "other"])
def test_large_voices_against_the_oracle(shape, arm, oracle_renders, engine_renders):
    out, taps, kernels = engine_renders(shape, arm)
    assert set(kernels) == {KERNELS[arm](shape)}, kernels
    ref, ref_taps = oracle_renders(shape)
    assert np.isfinite(ref_taps).all() and np.abs(ref_taps).max(axis=1).min() > 1e-4
    assert taps.shape == ref_taps.shape
    bad = np.count_nonzero(taps.view(np.uint32) != ref_taps.view(np.uint32))
    assert bad == 0, f"{shape.__name__} {arm}: {bad} of {taps.size} tap samples differ from the oracle"
    assert np.abs(out - ref).max() <= 1e-5 * max(1.0, float(np.abs(ref).max()))


@pytest.mark.parametrize("shape", list(SHAPES), ids=lambda s: s.__name__)
def test_both_kernels_agree_bit_for_bit(shape, engine_renders):
    out_i, taps_i, _ = engine_renders(shape, "interp")
    out_o, taps_o, _ = engine_renders(shape, "other")
    assert np.array_equal(taps_i.view(np.uint32), taps_o.view(np.uint32))
    assert np.abs(out_i - out_o).max() <= 1e-6 * max(1.0, float(np.abs(out_i).max()))   # the bus sums differ in order only


def all_shapes(arm, n_per_shape=2):
    graph, proc = new_processor(arm)
    for shape in SHAPES:
        for node in shape(graph, n_per_shape):
            proc.add_tap(node, 0)
    return graph, proc


@pytest.mark.parametrize("arm", ["interp", "other"])
def test_split_invariance(arm):
    n_blocks = 1500
    _, p1 = all_shapes(arm)
    one = p1.render(n_blocks)
    one_taps = p1.read_taps()
    assert set(p1.info()["kernels"]) == {KERNELS[arm](s) for s in SHAPES}
    _, p7 = all_shapes(arm)
    p7.set_blocks_per_launch(7)
    assert np.array_equal(p7.render(n_blocks), one)
    assert np.array_equal(p7.read_taps(), one_taps)
    # render_block (run_without_inputs) block by block equals the batched render, taps included
    n_bb = 300
    _, pb = all_shapes(arm)
    outs, taps = [], []
    for _ in range(n_bb):
        pb.run_without_inputs()
        outs.append(pb.output_block())
        taps.append(pb.read_taps())
    assert np.array_equal(np.stack(outs), one[:n_bb])
    assert np.array_equal(np.concatenate(taps, axis=1), one_taps[:, : n_bb * 64])
    assert np.abs(one_taps).max() > 1e-4


@pytest.mark.parametrize("arm", ["interp", "other"])
def test_snapshot_restored_into_a_fresh_processor_continues_bit_identically(arm):
    _, p1 = all_shapes(arm)
    first = p1.render(777)                              # mid-note, mid-segment
    image = p1.snapshot().to_bytes()
    cont = p1.render(700)
    cont_taps = p1.read_taps()
    g2, p2 = all_shapes(arm)
    g2.take_events()                                    # its events are inside the image
    p2.restore(Snapshot.from_bytes(image))
    assert p2.frame_clock() == 777 * 64
    assert np.array_equal(p2.render(700), cont)
    assert np.array_equal(p2.read_taps(), cont_taps)
    assert np.abs(first).max() > 1e-4


def test_partials_bank_1024_voices_10s_against_the_sharded_oracle():
    from oracle.sharded import ShardedOracle, bank_builder, sample_voices

    n_voices, seconds = 1024, 10.0
    n_blocks = int(seconds * SR) // 64
    build = bank_builder("partials", seconds)
    voices = sample_voices(n_voices, 64)
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions())
    ids = build(graph, n_voices, 0, n_voices)
    for v in voices:
        proc.add_tap(ids[v], 0)
    assert proc.info()["kernels"] == ["render_jit"]
    gpu = proc.render(n_blocks)
    gpu_taps = proc.read_taps()
    del proc
    ref, ref_taps = ShardedOracle(build, n_voices, tap_voices=voices).render(n_blocks)
    assert np.abs(ref).max() > 1e-3 and np.abs(ref_taps).max(axis=1).min() > 0.0, "silent reference"
    same = int(np.all(gpu_taps.view(np.uint32) == ref_taps.view(np.uint32), axis=1).sum())
    bus_err = float(np.abs(gpu - ref).max())
    print(f"partials: {n_voices} voices x {seconds:g} s: taps bit-identical {same}/{len(voices)}, bus err {bus_err:.3e}")
    assert same == len(voices)
    assert bus_err <= 1e-5 * max(1.0, float(np.abs(ref).max()))
