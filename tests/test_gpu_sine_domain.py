"""SinNumeric, FM and the PolyBlep sine family against the oracle, bit for bit, where their sine arguments leave [-120, 120].

knaster's SinNumeric wraps its phase from above only (osc.rs:266-268: `if phase > 1 { phase -= 1 }`), so at a negative
frequency the phase descends without bound (-440 Hz passes -19 after 43 ms) and the argument (phase + phase_offset) * TAU
passes glibc's |y| = 120, where sinf switches to its large-argument reduction; a phase_offset above ~19 gets there at once.
An FM carrier integrates its modulator's samples, so a 1-ulp difference in the modulator's sine random-walks the carrier.
The PolyBlep Cosine is `f32::cos` (glibc cosf).  Every tap here must be bit-identical to the oracle's (libm's) values.
"""
import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200.graph import Graph
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions
from oracle.oracle import OracleProcessor

pytestmark = pytest.mark.gpu
SR = 48000


def at(frame):
    return kn.Seconds.from_samples(frame, SR)


def render_both(build, n_blocks, **opts):
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, **opts))
    ids = build(graph)
    for i in ids:
        proc.add_tap(i, 0)
    out = proc.render(n_blocks)
    taps = proc.read_taps()
    g2 = Graph(0, 2, 64, SR)
    ids2 = build(g2)
    orc = OracleProcessor(g2, ring_buffer_size=1 << 22)
    for i in ids2:
        orc.add_tap(i, 0)
    ref, ref_taps = orc.render(n_blocks)
    return out, taps, ref, ref_taps, proc.info()["kernels"]


def mismatches(a, b):
    return int((a.view(np.uint32) != b.view(np.uint32)).sum())


def sinnum_voices(graph):
    with graph.edit() as g:
        down = g.push(kn.SinNumeric(-440.0))                 # phase descends: -4400 after 10 s
        off = g.push(kn.SinNumeric(220.0))
        off.param("phase_offset").set(25.3)                  # arguments from 159 up
        jump = g.push(kn.SinNumeric(330.0).precise_timing(4))
        jump.param("phase_offset").set_at(40.0, at(5 * SR + 17))   # mid-render
        for n in (down, off, jump):
            (n * 0.25).to_graph_out()
    return [down.id(), off.id(), jump.id()]


@pytest.mark.parametrize("path", ["interpreter", "jit"])
def test_sin_numeric_beyond_120_bit_identical(path):
    n_blocks = 10 * SR // 64
    opts = {"force_interpreter": True} if path == "interpreter" else {"force_jit": True}
    out, taps, ref, ref_taps, kernels = render_both(sinnum_voices, n_blocks, **opts)
    assert set(kernels) == ({"render_interp"} if path == "interpreter" else {"render_jit"}), kernels
    assert np.isfinite(ref_taps).all() and np.abs(ref_taps).max() > 0.99
    bad = [mismatches(taps[k], ref_taps[k]) for k in range(3)]
    assert bad == [0, 0, 0], f"taps differing from libm's sinf: {bad} of {taps.shape[1]} frames each"


def fm_voice(g, fm, fc, idx, amp):
    mod = g.push(kn.SinNumeric(fm))
    car = g.push(kn.SinNumeric(fc).ar_params())
    car.link("freq", mod * idx + fc)
    sig = car * amp
    sig.out([0, 0]).to_graph_out()
    return mod, sig


def test_fm_voice_with_descending_modulator_phase_bit_identical():
    # banks.fm_bank's shape (render_fm2, two lanes per voice), modulators at negative frequencies.  The fused kernel taps a voice's
    # output (carrier * amp); the carrier integrates every modulator sample, so a modulator that differs shows there.
    n_blocks = 10 * SR // 64

    def build(graph):
        ids = []
        with graph.edit() as g:
            for k, (fm, fc, ratio) in enumerate([(-440.0, 220.0, 1.5), (-97.5, 650.0, 3.0), (330.0, 440.0, 0.8), (-2.0, 300.0, 2.0)]):
                mod, sig = fm_voice(g, fm, fc, ratio * abs(fm), 0.25)
                ids.append(sig._outputs[0][0])
        return ids

    out, taps, ref, ref_taps, kernels = render_both(build, n_blocks)
    assert kernels == ["render_fm2"], kernels
    assert np.abs(ref_taps).max() > 0.2 and np.isfinite(ref_taps).all()
    bad = [mismatches(taps[k], ref_taps[k]) for k in range(len(taps))]
    assert bad == [0] * len(taps), f"voice taps differing from the oracle: {bad}"


def test_fm_one_lane_form_with_descending_modulator_phase():
    # render_fm2's one-lane form (above 9472 voices) against the interpreter, bit for bit, with a few descending modulators
    n_voices, n_blocks = 9600, 2 * SR // 64
    rng = np.random.Generator(np.random.PCG64(41))
    fc = rng.uniform(110.0, 880.0, n_voices)
    fm = fc * rng.choice(np.array([0.5, 1.0, 2.0, 3.0]), n_voices)
    idx = rng.uniform(0.0, 4.0, n_voices) * fm
    neg = [0, 1, 4735, n_voices - 1]
    fm[neg] = -fm[neg]

    def run(force_interp):
        graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(sample_rate=SR, force_interpreter=force_interp))
        taps = []
        with graph.edit() as g:
            for i in range(n_voices):
                mod, sig = fm_voice(g, float(fm[i]), float(fc[i]), float(idx[i]), 1.0 / n_voices)
                if i in neg:
                    taps.append(sig._outputs[0][0])
        for t in taps:
            proc.add_tap(t, 0)
        out = proc.render(n_blocks)
        return proc.read_taps(), proc.info()["kernels"]

    ft, fk = run(False)
    it, ik = run(True)
    assert fk == ["render_fm2"] and ik == ["render_interp"]
    assert np.abs(it).max() > 0.2 / n_voices
    bad = [mismatches(ft[k], it[k]) for k in range(len(ft))]
    assert bad == [0] * len(ft), f"one-lane form against the interpreter: {bad}"


def test_polyblep_sine_family_bit_identical():
    # polyblep.rs:243-276: Sine, Cosine, HalfWaveRectifiedSine, FullWaveRectifiedSine at test_all_polyblep_waveforms' pitches
    # (the last one above the sr/4 sine guard)
    waves = [kn.Waveform.Sine, kn.Waveform.Cosine, kn.Waveform.HalfWaveRectifiedSine, kn.Waveform.FullWaveRectifiedSine]

    def build(graph):
        ids = []
        with graph.edit() as g:
            for wf in waves:
                for f in (55.0, 1234.5, 12500.0):
                    osc = g.push(kn.PolyBlep(wf, f))
                    (osc * 0.1).to_graph_out()
                    ids.append(osc.id())
        return ids

    out, taps, ref, ref_taps, kernels = render_both(build, 1500)
    assert np.abs(ref_taps).max() > 0.9
    bad = [mismatches(taps[k], ref_taps[k]) for k in range(len(taps))]
    assert bad == [0] * len(taps), f"PolyBlep taps differing from the oracle (Sine x3, Cosine x3, HalfWave x3, FullWave x3): {bad}"
