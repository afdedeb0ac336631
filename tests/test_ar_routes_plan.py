"""CPU: the plan side of audio-rate routes into Pan2 pan, Phasor freq, RandomLin freq and Envelope time_scale, and of nodes with
every float parameter routed (up to six routes per node).  The plans build, their generated kernels compile with NVRTC for
sm_100a, and an event into a routed parameter produces no device event (audio_rate.rs:70-74).  What the kernels compute is
checked on the GPU (tests/test_gpu_ar_routes.py)."""
import pytest

import knaster_b200 as kn
from knaster_b200 import _ffi
from knaster_b200.graph import Graph

import test_gpu_ar_routes as ar
from test_jit_compile import nvrtc_available

SR = 48000


def voice_graph(shape, n=1):
    g = Graph(0, 2, 64, SR)
    ar.build_voices(g, shape, n)
    return g


@pytest.mark.parametrize("shape", ar.SHAPES, ids=lambda s: s.__name__)
def test_each_route_builds_a_plan(shape):
    g = voice_graph(shape)
    _evs, _nodes, info = _ffi.debug_simulate(g, g.take_events(), 4)
    assert info["n_voices"] == 1


def routed_svf_graph(routes):
    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        saw = e.push(kn.PolyBlep(kn.Waveform.Sawtooth, 110.0))
        lfo = e.push(kn.SinWt(0.5))
        svf = e.push(kn.SvfFilter(kn.SvfFilterType.Bell, 1000.0, 1.0, 0.0).wr_mul(1.0).wr_mul(1.0).wr_mul(1.0).ar_params())
        for p in routes:
            svf.link(p, lfo + 1.5)
        (saw >> svf).to_graph_out()
    return g


def test_all_six_float_parameters_of_an_svf_route_at_once():
    g = routed_svf_graph(["cutoff_freq", "q", "gain", 5, 6, 7])   # cutoff, q, gain and the three wr_mul values
    _evs, _nodes, info = _ffi.debug_simulate(g, g.take_events(), 4)
    assert info["n_voices"] == 1


@pytest.mark.parametrize("param", ["filter", "t_calculate_coefficients"])
def test_routes_into_integer_and_trigger_parameters_stay_rejected(param):
    g = routed_svf_graph(["cutoff_freq", param])
    with pytest.raises(_ffi.KgpuError) as ei:
        _ffi.debug_simulate(g, g.take_events(), 1)
    assert ei.value.code == _ffi.KGPU_ERR_UNSUPPORTED


@pytest.mark.parametrize("param", ["jump_to_segment", "t_restart", "t_stop"])
def test_envelope_routes_other_than_time_scale_stay_rejected(param):
    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        lfo = e.push(kn.SinWt(2.0))
        env = e.push(kn.Envelope(0.0, [kn.EnvelopeSegment(0.1, 1.0)]).ar_params())
        env.link(param, lfo * 0.5 + 1.0)
        env.to_graph_out()
    with pytest.raises(_ffi.KgpuError) as ei:
        _ffi.debug_simulate(g, g.take_events(), 1)
    assert ei.value.code == _ffi.KGPU_ERR_UNSUPPORTED


def pan_graph(routed):
    g = Graph(0, 2, 64, SR)
    with g.edit() as e:
        src = e.push(kn.SinWt(300.0))
        lfo = e.push(kn.SinWt(1.0))
        pan = e.push(kn.Pan2(0.0).ar_params() if routed else kn.Pan2(0.0))
        if routed:
            pan.link("pan", lfo * 0.5)
        else:
            (lfo * 0.5).to_graph_out()              # the same nodes, the LFO heard instead of routed
        (src >> pan).to_graph_out()
        pan.param("pan").set_at(0.7, kn.Seconds.from_samples(200, SR))
    return g, pan.id()


@pytest.mark.parametrize("routed", [False, True])
def test_event_into_a_routed_pan_is_ignored(routed):
    g, pan_id = pan_graph(routed)
    evs, nodes, _info = _ffi.debug_simulate(g, g.take_events(), 8)
    grp, voice, local, _reg = nodes[pan_id]
    mine = [e for e in evs if (e[0], e[1], e[2]) == (grp, voice, local)]
    if routed:
        assert mine == []
    else:
        assert [(e[3], e[6]) for e in mine] == [(0, 192), (0, 192)]   # OP_SET of both gains, at the start of frame 200's block


@pytest.mark.parametrize("shape", [ar.phasor_lfo, ar.randlin_lfo, ar.envelope_time_scale, ar.sinnum_all_routes],
                         ids=lambda s: s.__name__)
def test_events_into_routed_frequencies_and_time_scale_are_ignored(shape):
    # each shape sets its routed parameter with an event: freq, or the envelope's time_scale
    g = voice_graph(shape)
    evs, _nodes, _info = _ffi.debug_simulate(g, g.take_events(), 7500)
    ops = sorted({e[3] for e in evs})
    if shape is ar.envelope_time_scale:
        assert ops == [2, 3]                        # OP_ENV_STOP, OP_ENV_RESTART; no OP_ENV_STEP (5)
    else:
        assert ops == []


@pytest.mark.skipif(not nvrtc_available(), reason="libnvrtc is not installed")
@pytest.mark.parametrize("shape", ar.SHAPES, ids=lambda s: s.__name__)
def test_each_route_generates_and_compiles(shape):
    g = voice_graph(shape, 2)
    n, _cached = _ffi.jit_compile(g, tap_outputs=True)
    assert n == (2 if shape is ar.envelope_time_scale else 1)   # a looping and a one-shot envelope are two templates


@pytest.mark.skipif(not nvrtc_available(), reason="libnvrtc is not installed")
def test_six_routes_into_one_node_generate_and_compile():
    g = routed_svf_graph(["cutoff_freq", "q", "gain", 5, 6, 7])
    n, _cached = _ffi.jit_compile(g, tap_outputs=True)
    assert n == 1
