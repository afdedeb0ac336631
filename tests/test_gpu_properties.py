"""GPU property and edge-case tests for the fused voice-bank path (through the C ABI).

The parity tests in test_gpu_parity.py compare against the CPU oracle at small sizes, and
test_gpu_full_size.py at BASELINE.json's full sizes (16 384 voices x 10 s against the threaded oracle).
The full-size cases here add the properties that do not depend on an oracle: invariance under the
way a render is split into launches, exact scaling by a power of two, silence without notes,
determinism, and bus == sum of the voices.  The edge cases (ragged voice counts, odd block sizes and frame counts,
event collisions, dense event streams, events on the first and last frame, parameters outside the
straight-line domain) are small and are checked against the oracle."""
import os
import subprocess
import sys

import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200 import banks
from knaster_b200.graph import Graph
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions
from oracle.oracle import OracleProcessor

pytestmark = pytest.mark.gpu
SR = 48000
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def render_bank(n_voices, seconds, n_blocks, blocks_per_launch=0, gain_scale=1.0, n_notes=8, seed=2002):
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(no_scan=True))
    banks.subtractive_bank(graph, n_voices, seconds, seed=seed, n_notes=n_notes)
    if gain_scale != 1.0:  # WrMul's parameter ("wr_mul", index 4 of EnvAsr.wr_mul) on every envelope node
        from knaster_b200 import ugens as U

        with graph.edit() as g:
            for node, n in enumerate(graph.nodes):
                if n.ugen.kind == U.KIND_ENV_ASR:
                    g.set(node, "wr_mul", gain_scale / n_voices, kn.Time.asap())
    if blocks_per_launch:
        proc.set_blocks_per_launch(blocks_per_launch)
    out = proc.render(n_blocks)
    return out, proc


def oracle_render(build, n_blocks, outputs=1, block_size=64, taps=()):
    g = Graph(0, outputs, block_size, SR)
    ids = build(g)
    orc = OracleProcessor(g, ring_buffer_size=1 << 22)
    for i in taps or ids:
        orc.add_tap(i, 0)
    return orc.render(n_blocks)


def gpu_render(build, n_blocks, outputs=1, block_size=64, blocks_per_launch=0, taps=True):
    # no_scan: the small banks of this file are edge cases of the one-lane-per-voice kernels (bit-exact); the scan kernel
    # that small subtractive banks take by default has its own file, test_gpu_scan.py
    graph, proc = AudioProcessor.new(0, outputs, AudioProcessorOptions(block_size=block_size, sample_rate=SR, no_scan=True))
    ids = build(graph)
    if taps:
        for i in ids:
            proc.add_tap(i, 0)
    if blocks_per_launch:
        proc.set_blocks_per_launch(blocks_per_launch)
    out = proc.render(n_blocks)
    return out, (proc.read_taps() if taps and ids else None), proc


# ---- full size: BASELINE.json configs[2], 16 384 voices ----------------------------------------
FULL_V, FULL_SECONDS, FULL_BLOCKS = 16384, 2.0, 1500


@pytest.fixture(scope="module")
def full_render():
    out, proc = render_bank(FULL_V, FULL_SECONDS, FULL_BLOCKS)
    assert proc.info()["kernels"] == ["render_sub_asr"]
    return out


def test_full_size_launch_split_invariance(full_render):
    # 1024-block launches vs 96-block launches vs 7-block launches (frame counts that are not
    # multiples of the 16-frame group either way): bit-identical audio
    for bpl in (96, 7):
        out, _ = render_bank(FULL_V, FULL_SECONDS, FULL_BLOCKS, blocks_per_launch=bpl)
        assert np.array_equal(out, full_render), f"render differs with {bpl} blocks per launch"


def test_full_size_determinism_and_stereo(full_render):
    out, _ = render_bank(FULL_V, FULL_SECONDS, FULL_BLOCKS)
    assert np.array_equal(out, full_render)
    assert np.array_equal(full_render[:, 0, :], full_render[:, 1, :])  # .out([0, 0]): both channels carry the same bus
    assert np.isfinite(full_render).all()
    assert 1e-4 < np.abs(full_render).max() < 1.0


def test_full_size_gain_scaling_is_exact(full_render):
    # every voice's WrMul gain doubled: each voice sample, each partial sum and the bus double exactly
    out, _ = render_bank(FULL_V, FULL_SECONDS, FULL_BLOCKS, gain_scale=2.0)
    assert np.array_equal(out, 2.0 * full_render)


def test_full_size_silence_without_notes():
    out, _ = render_bank(FULL_V, 1.0, 750, n_notes=0)
    assert not out.any()


def test_bus_is_the_sum_of_the_voices():
    # 200 voices (6 full warps + a ragged one): the bus against the f64 sum of every tapped voice
    def build(graph):
        return banks.subtractive_bank(graph, 200, 1.0, n_notes=4, stereo=False)

    out, taps, proc = gpu_render(build, 750)
    assert proc.info()["kernels"] == ["render_sub_asr"]
    ref = taps.astype(np.float64).sum(axis=0).reshape(750, 64)
    assert np.abs(out[:, 0, :] - ref).max() <= 2e-7
    assert np.abs(ref).max() > 1e-3


# ---- edge cases against the oracle ---------------------------------------------------------------
@pytest.mark.parametrize("n_voices", [1, 31, 33, 65])
def test_ragged_voice_counts(n_voices):
    def build(graph):
        return banks.subtractive_bank(graph, n_voices, 0.5, n_notes=3, stereo=False)

    out, taps, proc = gpu_render(build, 375)
    ref, ref_taps = oracle_render(build, 375)
    assert proc.info()["kernels"] == ["render_sub_asr"]
    assert np.abs(taps - ref_taps).max() <= 1e-6
    assert np.abs(out - ref).max() <= 1e-6


@pytest.mark.parametrize("block_size,n_blocks", [(16, 333), (8, 1001), (1, 700), (256, 41)])
def test_block_sizes_and_frame_counts(block_size, n_blocks):
    # frame counts that are not multiples of the 16-frame group, one-frame blocks, long blocks
    def build(graph):
        return banks.subtractive_bank(graph, 40, n_blocks * block_size / SR, n_notes=3, stereo=False)

    out, taps, _ = gpu_render(build, n_blocks, block_size=block_size)
    ref, ref_taps = oracle_render(build, n_blocks, block_size=block_size)
    assert np.abs(taps - ref_taps).max() <= 1e-6
    assert np.abs(out - ref).max() <= 1e-6
    assert np.abs(ref).max() > 1e-4


def _voice(g, f=220.0, fc=1200.0, q=2.0, att=0.003, rel=0.05, gain=0.25):
    saw = g.push(kn.PolyBlep(kn.Waveform.Sawtooth, f).precise_timing(8))
    svf = g.push(kn.SvfFilter(kn.SvfFilterType.Low, fc, q, 0.0).precise_timing(8))
    env = g.push(kn.EnvAsr(att, rel).wr_mul(gain).precise_timing(8))
    sig = (saw >> svf) * env
    sig.to_graph_out()
    return saw, svf, env, sig


def at(frame):
    return kn.Seconds.from_samples(frame, SR)


def test_event_collisions_and_boundaries():
    # every voice gets its note-on at the SAME frame; events on frame 0, on a launch boundary
    # (64 blocks per launch = frame 4096) and on the very last frame; a release during the attack
    n_blocks = 200
    last = n_blocks * 64 - 1

    def build(graph):
        ids = []
        with graph.edit() as g:
            for i in range(40):
                saw, svf, env, sig = _voice(g, f=110.0 + 7.0 * i, fc=500.0 + 100.0 * i, att=0.002 + 0.001 * (i % 5))
                env.param("t_restart").trig_at(at(0))
                saw.param("freq").set_at(150.0 + i, at(0))
                env.param("t_release").trig_at(at(50 + i))            # still attacking: release_scale = t
                env.param("t_restart").trig_at(at(4096))              # all voices, launch boundary
                svf.param("cutoff_freq").set_at(2000.0 + 10.0 * i, at(4096))
                svf.param("q").set_at(0.7 + 0.1 * (i % 7), at(4097))
                env.param("t_release").trig_at(at(9000))
                env.param("t_restart").trig_at(at(last))
                saw.param("freq").set_at(300.0 + i, at(last))
                ids.append(sig._outputs[0][0])
        return ids

    out, taps, proc = gpu_render(build, n_blocks, blocks_per_launch=64)
    ref, ref_taps = oracle_render(build, n_blocks)
    assert proc.info()["kernels"] == ["render_sub_asr"]
    assert np.abs(taps - ref_taps).max() <= 1e-6
    assert np.abs(out - ref).max() <= 1e-6
    assert np.abs(ref_taps[:, 4200:5000]).max() > 1e-3


def test_dense_event_stream():
    # one voice receives a cutoff change on every frame of a block and 8 frequency changes inside
    # one block (the precise_timing::<8> queue is full), its neighbours none
    def build(graph):
        ids = []
        with graph.edit() as g:
            voices = [_voice(g, f=200.0 + 50 * i) for i in range(5)]
            for saw, svf, env, sig in voices:
                env.param("t_restart").trig_at(at(10))
                ids.append(sig._outputs[0][0])
            saw, svf, env, _ = voices[2]
            for k in range(8):
                saw.param("freq").set_at(300.0 + 40.0 * k, at(640 + 3 + 7 * k))
            for k in range(64):
                svf.param("cutoff_freq").set_at(600.0 + 25.0 * k, at(1280 + k))
        return ids

    out, taps, proc = gpu_render(build, 60)
    ref, ref_taps = oracle_render(build, 60)
    assert np.abs(taps - ref_taps).max() <= 1e-6
    assert np.abs(out - ref).max() <= 1e-6
    assert proc.info()["dropped_changes"] > 0  # queue overflow is counted, like knaster's rt_log warning


def test_parameters_outside_the_straight_line_domain():
    # freq >= sr/4 (PolyBlep's sine guard), freq 0 (dt = 0), negative freq (t leaves [0,1)), a
    # non-lowpass filter in the same warp, very slow envelopes: lanes fall back to the generic tick
    def build(graph):
        ids = []
        with graph.edit() as g:
            specs = [(13000.0, 900.0), (0.0, 900.0), (-220.0, 900.0), (220.0, 900.0), (30.0, 50.0)]
            for i, (f, fc) in enumerate(specs):
                saw, svf, env, sig = _voice(g, f=f, fc=fc, att=0.2 if i == 4 else 0.003, rel=2.0 if i == 4 else 0.05)
                env.param("t_restart").trig_at(at(5 + i))
                env.param("t_release").trig_at(at(6000 + i))
                ids.append(sig._outputs[0][0])
            saw, svf, env, sig = _voice(g, f=330.0)
            svf.param("filter").set_at(int(kn.SvfFilterType.Band), at(2000))   # warp leaves the lowpass specialisation
            saw.param("freq").set_at(14000.0, at(3000))
            saw.param("freq").set_at(-5.0, at(4000))
            saw.param("freq").set_at(440.0, at(5000))
            env.param("t_restart").trig_at(at(1))
            ids.append(sig._outputs[0][0])
        return ids

    out, taps, proc = gpu_render(build, 150)
    ref, ref_taps = oracle_render(build, 150)
    assert proc.info()["kernels"] == ["render_sub_asr"]
    assert np.isfinite(ref_taps).all()
    # the negative-frequency voice runs the blep far outside its window (|t/dt| is large): per-voice
    # errors are compared relative to that voice's peak, the bus relative to the largest voice
    # (the mix bus is a tree sum here and a left fold in knaster, SURVEY H4)
    peak = np.maximum(1.0, np.abs(ref_taps).max(axis=1, keepdims=True))
    assert (np.abs(taps - ref_taps) / peak).max() <= 1e-5
    assert np.abs(out - ref).max() <= 1e-6 * peak.max()
    assert np.abs(ref_taps).max() > 1e-2


def test_late_events_keep_arrival_order():
    # events pushed after their due time become ready in the next block, in ARRIVAL order
    # (graph_gen.rs:276 saturating_sub): the last one pushed wins
    def run(proc, graph, handles):
        saw, svf, env, sig = handles
        proc.render(10)
        with graph.edit():
            saw.param("freq").set_at(500.0, at(300))   # due in the past (frame clock is 640)
            saw.param("freq").set_at(250.0, at(100))   # due even earlier, pushed later: applied last
            env.param("t_restart").trig_at(at(0))
        return proc.render(20)

    graph, proc = AudioProcessor.new(0, 1, AudioProcessorOptions(no_scan=True))
    with graph.edit() as g:
        handles = _voice(g)
    gpu = run(proc, graph, handles)
    g2 = Graph(0, 1, 64, SR)
    with g2.edit() as g:
        handles2 = _voice(g)
    orc = OracleProcessor(g2, ring_buffer_size=1 << 16)
    ref = run(orc, g2, handles2)[0]
    assert np.abs(gpu - ref).max() <= 1e-6
    assert np.abs(ref).max() > 1e-3


def test_two_warp_kernel_variant_matches(tmp_path):
    # the warp-specialised experiment (KGPU_SUB_TWO_WARPS=1) must stay bit-identical to the default
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r)\n"
        "from knaster_b200 import banks\n"
        "from knaster_b200.processor import AudioProcessor, AudioProcessorOptions\n"
        "g, p = AudioProcessor.new(0, 2, AudioProcessorOptions())\n"
        "banks.subtractive_bank(g, 100, 1.0, n_notes=4)\n"
        "np.save(sys.argv[1], p.render(750))\n" % ROOT
    )
    outs = []
    for flag in ("0", "1"):
        path = str(tmp_path / f"two_warp_{flag}.npy")
        env = dict(os.environ, KGPU_SUB_TWO_WARPS=flag, KGPU_SUB_SCAN="0")
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=300)
        outs.append(np.load(path))
    assert np.array_equal(outs[0], outs[1])
    assert np.abs(outs[0]).max() > 1e-3


# ---- additive wavetable bank (configs[1]): the time-parallel recipe -------------------------------
def test_additive_bank_fused_kernel_without_taps():
    # no taps: the unrolled accumulation path of render_add_wt; bus against the oracle's left fold
    def build(graph):
        banks.additive_bank(graph, 300, 1.0)
        return []

    out, _, proc = gpu_render(build, 750, outputs=2, taps=False)
    ref, _ = oracle_render(build, 750, outputs=2)
    assert proc.info()["kernels"] == ["render_add_wt"]
    assert np.abs(out - ref).max() <= 1e-6
    assert np.abs(ref).max() > 1e-3
    # launch-split invariance and the interpreter agree bit for bit / within the summation order
    out7, _, _ = gpu_render(build, 750, outputs=2, taps=False, blocks_per_launch=7)
    assert np.array_equal(out7, out)
    graph, p = AudioProcessor.new(0, 2, AudioProcessorOptions(force_interpreter=True))
    build(graph)
    assert np.abs(p.render(750) - out).max() <= 1e-6


def test_additive_bank_full_size_properties():
    # BASELINE.json configs[1]: 4096 partials, 10 s.  Launch-split invariance + determinism.
    def render(bpl=0):
        graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions())
        banks.additive_bank(graph, 4096, 10.0)
        if bpl:
            proc.set_blocks_per_launch(bpl)
        return proc.render(7500), proc

    a, proc = render()
    assert proc.info()["kernels"] == ["render_add_wt"]
    b, _ = render(bpl=333)
    assert np.array_equal(a, b)
    assert np.isfinite(a).all() and 1e-3 < np.abs(a).max() < 1.0
    assert np.array_equal(a[:, 0], a[:, 1])


def test_sinwt_with_precise_timing_stays_on_the_interpreter():
    # sample-accurate changes inside a block cannot be expressed per block: no fused recipe
    def build(graph):
        with graph.edit() as g:
            v = g.push(kn.SinWt(330.0).wr_mul(0.5).precise_timing(4))
            v.to_graph_out()
            v.param("freq").set_at(500.0, at(1000))
            v.param("wr_mul").set_at(0.25, at(1501))
        return [v.id()]

    out, taps, proc = gpu_render(build, 40)
    ref, ref_taps = oracle_render(build, 40)
    assert proc.info()["kernels"] == ["render_interp"]
    assert np.array_equal(taps, ref_taps)



def test_fm_bank_one_lane_form_above_the_two_lane_threshold():
    # recipe "render_fm2" has two forms (fused.cu fm_two_lanes): two lanes per voice up to 9472 voices,
    # one lane per voice above.  The parity tests run the first; this one runs the second against the
    # interpreter (same arithmetic, same order => per-voice bit-identical).
    n_voices, n_blocks = 9600, 24

    def run(force_interp):
        graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_interpreter=force_interp))
        ids = banks.fm_bank(graph, n_voices)
        for i in (ids[0], ids[1], ids[4735], ids[-2], ids[-1]):
            proc.add_tap(i, 0)
        out = proc.render(n_blocks)
        return out, proc.read_taps(), proc.info()["kernels"]

    fo, ft, fk = run(False)
    io, it, ik = run(True)
    assert fk == ["render_fm2"] and ik == ["render_interp"]
    assert np.abs(ft).max() > 1e-5
    assert np.array_equal(ft, it)
    assert np.abs(fo - io).max() <= 1e-6


@pytest.mark.parametrize("block_size,n_blocks,per_block", [(24, 60, True), (1, 90, True), (100, 13, False), (7, 301, False), (64, 5, True)])
@pytest.mark.parametrize("bank", ["fm", "segments"])
def test_fused_fm_and_segment_kernels_with_odd_launch_lengths(bank, block_size, n_blocks, per_block):
    # render_fm2 pipelines its carriers two 16-frame groups behind its modulators and drains that
    # pipeline at every launch end; render_sub_seg carries f64 envelope state across launches.  Launch
    # lengths that are not multiples of 16 (or shorter than one group), and one launch per block
    # (run_without_inputs), must give what one long render gives and what the oracle gives.
    def build(graph):
        if bank == "fm":
            ids = banks.fm_bank(graph, 37)
            with graph.edit() as g:      # parameter events through the slow path of the two-lane kernel
                for k, frame in enumerate((3, block_size * n_blocks // 3, block_size * n_blocks // 2 + 5)):
                    # node 0 / 1: modulator / carrier of voice 0 (fm_bank pushes them first)
                    g.set(k % 2, "phase_offset", 0.1 * (k + 1), kn.Time.at(kn.Seconds.from_samples(frame, SR)))
            return ids
        return banks.subtractive_bank(graph, 37, n_blocks * block_size / SR, n_notes=3, envelope="segments")

    out, taps, proc = gpu_render(build, n_blocks, block_size=block_size, outputs=2)
    assert proc.info()["kernels"] == ["render_fm2" if bank == "fm" else "render_sub_seg"]
    ref, ref_taps = oracle_render(build, n_blocks, block_size=block_size, outputs=2)
    assert np.abs(taps - ref_taps).max() <= 1e-5
    assert np.abs(out - ref).max() <= 1e-5
    assert np.abs(ref).max() > 1e-4
    if per_block:
        graph, p1 = AudioProcessor.new(0, 2, AudioProcessorOptions(block_size=block_size, sample_rate=SR))
        build(graph)
        blocks = []
        for _ in range(n_blocks):
            p1.run_without_inputs()
            blocks.append(p1.output_block())
        assert np.array_equal(np.stack(blocks), out)


def test_readme_shape_bank_runs_the_time_parallel_wavetable_kernel():
    # `sine * 0.2` (README.md:35-47) = SinWt -> MathUGen<Mul> with a Constant: rendered by render_add_wt
    # (time is the parallel axis), with `value` events on the Constant acting as gain changes and
    # `freq` / `phase_offset` / `reset_phase` events on the oscillator; both operand orders of the Mul
    def build(graph):
        ids = []
        with graph.edit() as g:
            for i in range(9):
                sine = g.push(kn.SinWt(110.0 * (i + 1)))
                c = g.push(kn.Constant(0.05 + 0.01 * i))
                sig = sine * c
                sig.out([0, 0]).to_graph_out()
                c.param("value").set_at(0.02 * (i + 1), at(64 * (3 + i)))
                c.param("value").set_at(0.01, at(64 * 40 + 17))           # inside a block: applies at its start
                sine.param("freq").set_at(333.0 + i, at(64 * 20))
                sine.param("phase_offset").set_at(0.25, at(64 * 30))
                sine.param("reset_phase").trig_at(at(64 * 50))
                ids.append(sig._outputs[0][0])
        return ids

    out, taps, proc = gpu_render(build, 120, outputs=2)
    assert proc.info()["kernels"] == ["render_add_wt"]
    ref, ref_taps = oracle_render(build, 120, outputs=2)
    assert np.array_equal(taps, ref_taps)          # integer phase, one f32 product
    assert np.abs(out - ref).max() <= 1e-6
    assert np.abs(ref).max() > 0.05


def test_block_by_block_under_a_large_event_backlog_equals_batched():
    # run_without_inputs() once per block with seconds of schedule queued: the host keeps a calendar (only the
    # events that can become ready soon are scanned per call, plan.cpp calendar_update).  Same result as batched
    # renders, including events pushed while the calendar is active: near ones, ones beyond its horizon, a late
    # one, and two for the same frame whose arrival order matters.
    n_voices, n_blocks = 600, 750

    def extra(graph, ids_saw, clock):
        with graph.edit() as g:
            g.set(ids_saw[5], "freq", 333.0, kn.Time.at(at(clock + 10)))
            g.set(ids_saw[6], "freq", 444.0, kn.Time.at(at(clock + 64 * 200)))       # beyond the horizon
            g.set(ids_saw[6], "freq", 555.0, kn.Time.at(at(clock + 64 * 200)))       # same frame: the later push wins
            g.set(ids_saw[7], "freq", 222.0, kn.Time.at(at(max(0, clock - 500))))    # late: next block
            g.set(ids_saw[8], "freq", 111.0, kn.Time.at(at(clock + 64 * 70 + 3)))    # just beyond the look-ahead

    def saws(graph):
        from knaster_b200 import ugens as U
        return [i for i, n in enumerate(graph.nodes) if n.ugen.kind == U.KIND_POLYBLEP]

    g1, p1 = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR))
    banks.subtractive_bank(g1, n_voices, 1.0, n_notes=16)
    assert sum(len(a) for a in g1.pending_event_arrays) + len(g1.pending_events) > 16384
    s1 = saws(g1)
    blocks = []
    for b in range(n_blocks):
        if b in (100, 300):
            extra(g1, s1, b * 64)
        p1.run_without_inputs()
        blocks.append(p1.output_block())
    per_block = np.stack(blocks)

    g2, p2 = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR))
    banks.subtractive_bank(g2, n_voices, 1.0, n_notes=16)
    s2 = saws(g2)
    parts = [p2.render(100)]
    extra(g2, s2, 100 * 64)
    parts.append(p2.render(200))
    extra(g2, s2, 300 * 64)
    parts.append(p2.render(450))
    batched = np.concatenate(parts)
    assert np.abs(batched).max() > 1e-3
    assert np.array_equal(per_block, batched)


@pytest.mark.parametrize("bank", ["asr", "segments", "additive", "fm", "interp"])
def test_snapshot_restore_rewinds_the_render(bank):
    # kgpu_plan_snapshot / kgpu_plan_restore: voice registers, control-side state (smoothing ramps, precise-timing
    # queues), queued events and the frame clock all come back; what was pushed after the snapshot does not
    def build(graph):
        if bank == "additive":
            return banks.additive_bank(graph, 70, 1.0)
        if bank == "fm":
            return banks.fm_bank(graph, 40)
        return banks.subtractive_bank(graph, 70, 1.0, n_notes=6, envelope="segments" if bank == "segments" else "asr")

    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_interpreter=bank == "interp"))
    build(graph)
    first = proc.render(130)                      # stops in the middle of notes / smoothing ramps
    snap = proc.snapshot()
    a = proc.render(400)
    assert proc.frame_clock() == 530 * 64
    proc.restore(snap)
    assert proc.frame_clock() == 130 * 64
    b = proc.render(400)
    assert np.array_equal(a, b)
    assert np.abs(a).max() > 1e-3
    # an event pushed after the snapshot changes the render, and is gone after the next restore
    with graph.edit() as g:
        g.set(0, 0, 987.0, kn.Time.asap())        # node 0 / parameter 0 is a frequency in every bank
    c = proc.render(60)
    assert not np.array_equal(c, a[:60])
    proc.restore(snap)
    d = proc.render(400)
    assert np.array_equal(d, a)
    # the whole run equals an uninterrupted one
    g2, p2 = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_interpreter=bank == "interp"))
    build(g2)
    assert np.array_equal(p2.render(530), np.concatenate([first, a]))
    # the snapshot as bytes, restored into ANOTHER processor built from the same graph (checkpoint / resume)
    from knaster_b200.processor import Snapshot

    image = snap.to_bytes()
    g3, p3 = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_interpreter=bank == "interp"))
    build(g3)
    g3.take_events()                                  # its events are inside the image
    p3.restore(Snapshot.from_bytes(image))
    assert p3.frame_clock() == 130 * 64
    assert np.array_equal(p3.render(400), a)
    with pytest.raises(Exception):
        Snapshot.from_bytes(image[:-3])
    with pytest.raises(Exception):
        Snapshot.from_bytes(b"x" * 64)


@pytest.mark.parametrize("bank,voices", [("segments", 16384), ("fm", 8192), ("fm", 9600)])
def test_full_size_launch_split_invariance_of_the_other_recipes(bank, voices):
    # BASELINE.json sizes for configs[2] variant B and configs[3] (and the one-lane FM form above 9472 voices):
    # one launch against 97-block and 5-block launches -- the f64 envelope state, the FM kernel's drained carrier
    # pipeline and the partial-row layout must make the split invisible, bit for bit
    def run(bpl):
        graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR))
        if bank == "fm":
            banks.fm_bank(graph, voices)
        else:
            banks.subtractive_bank(graph, voices, 0.5, envelope="segments")
        if bpl:
            proc.set_blocks_per_launch(bpl)
        return proc.render(375), proc.info()["kernels"]

    whole, kernels = run(0)
    assert kernels == ["render_fm2" if bank == "fm" else "render_sub_seg"]
    assert np.isfinite(whole).all() and np.abs(whole).max() > 1e-4
    for bpl in (97, 5):
        out, _ = run(bpl)
        assert np.array_equal(out, whole), f"{bank}: render differs with {bpl} blocks per launch"


def test_prepare_must_be_followed_by_the_render_it_prepared():
    # kgpu_plan_prepare(N) consumes the queued events and advances every ramp / queue by N blocks: any other call
    # in between is KGPU_ERR_STATE instead of a silently wrong render (ADVICE r1)
    from knaster_b200 import _ffi

    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions())
    banks.subtractive_bank(graph, 40, 0.5, n_notes=3)
    ev = graph.take_events()
    graph.pending_event_arrays = [ev.copy()]
    proc.prepare(100)
    for call in (lambda: proc.render(50), lambda: proc.set_blocks_per_launch(7), lambda: proc.prepare(100),
                 lambda: proc.add_tap(0, 0)):
        with pytest.raises(_ffi.KgpuError) as e:
            call()
        assert e.value.code == _ffi.KGPU_ERR_STATE
    graph.pending_event_arrays = [ev[:1].copy()]
    with pytest.raises(_ffi.KgpuError) as e:
        proc.render(100)            # pushes the pending event first: refused, nothing rendered
    assert e.value.code == _ffi.KGPU_ERR_STATE
    graph.take_events()
    a = proc.render(100)            # the prepared render itself is still valid ...
    g2, p2 = AudioProcessor.new(0, 2, AudioProcessorOptions())
    banks.subtractive_bank(g2, 40, 0.5, n_notes=3)
    assert np.array_equal(a, p2.render(100))   # ... and equals the unprepared one


def test_restore_rejects_foreign_and_corrupt_snapshots():
    # ADVICE r1: a deserialized image is checked against the plan before any of it is used as an index --
    # another graph of the same shape, flipped bytes and hostile lengths all come back as KGPU_ERR_INVALID
    from knaster_b200 import _ffi
    from knaster_b200.processor import Snapshot

    def make(seed):
        graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR))
        banks.additive_bank(graph, 40, 1.0, seed=seed)          # smoothing ramps + queued events: every table is non-trivial
        proc.render(20)
        return graph, proc

    g1, p1 = make(1001)
    image = p1.snapshot().to_bytes()
    g2, p2 = make(1002)                                          # same shape, other frequencies / gains
    with pytest.raises(_ffi.KgpuError) as e:
        p2.restore(Snapshot.from_bytes(image))
    assert e.value.code == _ffi.KGPU_ERR_INVALID
    ref = p1.render(50)
    r = np.random.Generator(np.random.PCG64(5))
    rejected = 0
    for trial in range(300):
        bad = bytearray(image)
        for _ in range(int(r.integers(1, 4))):
            pos = int(r.integers(12, len(bad)))                  # keep magic + version intact: the interesting paths lie behind them
            bad[pos] = int(r.integers(0, 256)) if r.random() < 0.5 else 0xFF
        try:
            snap = Snapshot.from_bytes(bytes(bad))
            p1.restore(snap)
        except _ffi.KgpuError as err:
            assert err.code == _ffi.KGPU_ERR_INVALID
            rejected += 1
            continue
        out = p1.render(5)                                       # accepted images differ in values only: rendering must not fault
        assert out.shape == (5, 2, 64)
    assert rejected > 30
    p1.restore(Snapshot.from_bytes(image))                       # and the pristine image still restores exactly
    assert np.array_equal(p1.render(50), ref)
