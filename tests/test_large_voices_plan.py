"""CPU: voices beyond 24 nodes, 192 registers and 24 value slots plan, up to the limits of dev.h (128 nodes, 1024 registers,
32 live value slots, an Envelope of 169 segments); one more is rejected with a message that names the limit.  Graphs that
planned before keep their plan: voice discovery only falls back to whole large voices where the small-voice discoveries
fail.  What the kernels compute is checked on the GPU (tests/test_gpu_large_voices.py)."""
import pytest

import knaster_b200 as kn
from knaster_b200 import _ffi
from knaster_b200.graph import Graph

import test_gpu_large_voices as lv
from test_jit_compile import nvrtc_available

SR = 48000


def plan_info(g):
    _evs, _nodes, info = _ffi.debug_simulate(g, g.take_events(), 4)
    return info["n_groups"], info["n_voices"]


def rejected(g):
    with pytest.raises(_ffi.KgpuError) as ei:
        _ffi.debug_simulate(g, g.take_events(), 1)
    assert ei.value.code == _ffi.KGPU_ERR_UNSUPPORTED
    return str(ei.value)


def operator_graph(n_voices, n_ops, tail=()):
    """saw -> n_ops x (x * 0.99 + 0.001) -> SvfFilter [-> OnePoleLpf] [* 0.5]: 2 + 4 n_ops nodes (+ 1, + 2)"""
    g = Graph(0, 2, 64, SR)
    with g.edit() as e:
        for i in range(n_voices):
            x = e.push(kn.PolyBlep(kn.Waveform.Sawtooth, 100.0 + i))
            for _ in range(n_ops):
                x = x * 0.99 + 0.001
            x = x >> e.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0, 1.0, 0.0))
            if "onepole" in tail:
                x = x >> e.push(kn.OnePoleLpf(3000.0))
            if "gain" in tail:
                x = x * 0.5
            x.out([0, 0]).to_graph_out()
    return g


def additive_graph(n_voices, n_partials):
    """n_partials x SinWt.wr_mul summed -> SvfFilter: 2 n_partials nodes"""
    g = Graph(0, 2, 64, SR)
    with g.edit() as e:
        for i in range(n_voices):
            mix = None
            for k in range(n_partials):
                p = e.push(kn.SinWt(100.0 * (k + 1) + i).wr_mul(0.01))
                mix = p if mix is None else mix + p
            (mix >> e.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0, 1.0, 0.0))).out([0, 0]).to_graph_out()
    return g


def test_operator_voices_of_50_nodes_plan_as_one_group():
    assert plan_info(operator_graph(4, 12)) == (1, 4)


def test_additive_voices_keep_their_partial_sums():
    # 64 voices x 20 partials: one internal signal per voice would exceed the 32 outputs + signals of a plan
    assert plan_info(additive_graph(64, 20)) == (1, 64)


def test_graphs_that_planned_before_keep_their_plan():
    assert plan_info(operator_graph(4, 6)) == (52, 52)        # 26 nodes: every fan-in / fan-out point is cut, as before
    assert plan_info(additive_graph(4, 20)) == (8, 84)        # each voice's partial sum stays an internal signal


def test_a_voice_of_128_nodes_plans_and_129_is_rejected():
    assert plan_info(operator_graph(4, 31, ("gain",))) == (1, 4)                 # 2 + 124 + 2 = 128 nodes
    msg = rejected(operator_graph(4, 31, ("onepole", "gain")))                   # 129
    assert "129 nodes" in msg and "limit of 128" in msg, msg


def envelope_graph(n_segments, n_gains):
    """Envelope(n_segments).wr_mul(1) * 0.5 * 0.5 ...: 8 + 6 n_segments + 1 + n_gains registers"""
    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        env = e.push(kn.Envelope(0.0, [kn.EnvelopeSegment(0.01, (k % 3) / 2.0) for k in range(n_segments)]).wr_mul(1.0))
        x = env
        for _ in range(n_gains):
            x = x * 0.5
        x.to_graph_out()
    return g


def test_a_voice_at_the_register_limit_plans_and_one_more_register_is_rejected():
    assert plan_info(envelope_graph(169, 1)) == (1, 1)        # 8 + 1014 + 1 + 1 = 1024 registers
    msg = rejected(envelope_graph(169, 2))
    assert "1025 registers" in msg and "limit 1024" in msg, msg


def test_an_envelope_with_the_most_segments_plans_and_one_more_is_rejected():
    assert plan_info(envelope_graph(169, 0)) == (1, 1)
    msg = rejected(envelope_graph(170, 0))
    assert "170 segments" in msg and "at most 169" in msg, msg


def subtraction_graph(n_partials):
    """p0 - (p1 - (... - p_{n-1})) over SinWt partials, 2 voices: n_partials values live at once"""
    g = Graph(0, 2, 64, SR)
    with g.edit() as e:
        for i in range(2):
            ps = [e.push(kn.SinWt(50.0 * (k + 1) + i)) for k in range(n_partials)]
            acc = ps[-1]
            for p in reversed(ps[:-1]):
                acc = p - acc
            acc.out([0, 0]).to_graph_out()
    return g


def test_a_voice_at_the_slot_limit_plans_and_one_more_slot_is_rejected():
    assert plan_info(subtraction_graph(32)) == (1, 2)
    msg = rejected(subtraction_graph(33))
    assert "33 live value slots" in msg and "limit 32" in msg, msg


@pytest.mark.parametrize("shape", list(lv.SHAPES), ids=lambda s: s.__name__)
def test_the_gpu_test_shapes_plan_as_whole_voices(shape):
    # at the GPU test's sizes: 4 voices of partials would still plan as before, each voice's partial sum an internal signal
    g = Graph(0, 2, 64, SR)
    n = lv.SHAPES[shape]
    shape(g, n)
    assert plan_info(g) == (2 if shape is lv.envelope_167 else 1, n)   # looping and one-shot Envelopes are two templates


@pytest.mark.skipif(not nvrtc_available(), reason="libnvrtc is not installed")
@pytest.mark.parametrize("shape", [lv.partials, lv.operators, lv.nodes_128, lv.slots_32], ids=lambda s: s.__name__)
def test_large_templates_generate_and_compile(shape):
    g = Graph(0, 2, 64, SR)
    shape(g, lv.SHAPES[shape])
    n, _cached = _ffi.jit_compile(g, tap_outputs=True)
    assert n == 1


def test_a_master_bus_over_large_voices_is_still_cut():
    # 20 voices of 30 nodes summed into a master SvfFilter: a sum of 20 leaves would glue the bank into one component, so the
    # first discovery's cut at 16 leaves stands -- 20 voices of 30 nodes, then the master filter reading their sum
    g = Graph(0, 2, 64, SR)
    with g.edit() as e:
        mix = None
        for i in range(20):
            x = e.push(kn.PolyBlep(kn.Waveform.Sawtooth, 100.0 + i))
            for _ in range(7):
                x = x * 0.99 + 0.001
            x = x >> e.push(kn.SvfFilter(kn.SvfFilterType.Low, 2000.0, 1.0, 0.0))
            mix = x if mix is None else mix + x
        (mix >> e.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0, 1.0, 0.0))).out([0, 0]).to_graph_out()
    assert plan_info(g) == (2, 21)


def node_event_graph(with_saw_events):
    """4 voices of saw -> 12 x (x * 0.99 + 0.001) -> SvfFilter -> * EnvAsr (52 nodes): notes on the EnvAsr, whose template index
    is past 31, and optionally frequency changes of the saw (template index 0) in the same blocks"""
    g = Graph(0, 2, 64, SR)
    ids = []
    with g.edit() as e:
        for i in range(4):
            saw = e.push(kn.PolyBlep(kn.Waveform.Sawtooth, 100.0 + i))
            x = saw
            for _ in range(12):
                x = x * 0.99 + 0.001
            env = e.push(kn.EnvAsr(0.01, 0.1))
            ((x >> e.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0, 1.0, 0.0))) * env).out([0, 0]).to_graph_out()
            for k in range(3):
                f = 1000 + 5000 * k + 7 * i
                env.param("t_restart").trig_at(kn.Seconds.from_samples(f, SR))
                env.param("t_release").trig_at(kn.Seconds.from_samples(f + 2000, SR))
                if with_saw_events:
                    saw.param("freq").set_at(200.0 + 10 * k, kn.Seconds.from_samples(f, SR))
            ids.append((saw.id(), env.id()))
    return g, ids


def test_events_reach_nodes_past_index_31_of_a_voice():
    # the control simulation marks, per block, which template nodes have an event: node indices past 31 need more than one
    # 32-bit word.  Events of the EnvAsr (index >= 32) come out alone and unchanged beside events of the saw (index 0).
    runs = {}
    for with_saw in (False, True):
        g, ids = node_event_graph(with_saw)
        evs, nodes, info = _ffi.debug_simulate(g, g.take_events(), 375)
        assert info["n_groups"] == 1
        saw_local, env_local = nodes[ids[0][0]][2], nodes[ids[0][1]][2]
        runs[with_saw] = [e for e in evs if e[2] == env_local], {e[2] for e in evs}
        assert saw_local < 32 <= env_local
        assert runs[with_saw][1] == ({saw_local, env_local} if with_saw else {env_local})
        for v in range(4):
            assert len([e for e in runs[with_saw][0] if e[1] == v]) >= 6     # 3 notes: restart + release each
    assert runs[False][0] == runs[True][0]
