"""CPU: graph inputs that one voice reads are ports of its template (include/knaster_gpu.h, kgpu_render_inputs).  Banks of
thousands of input tracks, each through its own effect chain, plan as one voice group; every other input stays a shared
signal row, at most 16 of them.  What the kernels compute is checked on the GPU (tests/test_gpu_voice_inputs.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200 import _ffi, banks
from knaster_b200.graph import Graph

from test_jit_compile import nvrtc_available

SR = 48000
HERE = os.path.dirname(os.path.abspath(__file__))


def plan(g):
    _evs, nodes, info = _ffi.debug_simulate(g, g.take_events(), 1)
    return nodes, info


def n_regs(info):
    assert info["n_groups"] == 1
    return info["state_bytes"] // (4 * info["n_voices"])


def rejected(g):
    with pytest.raises(_ffi.KgpuError) as ei:
        _ffi.debug_simulate(g, g.take_events(), 1)
    assert ei.value.code == _ffi.KGPU_ERR_UNSUPPORTED
    return str(ei.value)


def port_channels(g, node_ids, info, n_ports):
    """the channel register of every port of the voices that hold node_ids[k] (the last n_ports registers of the template)"""
    nodes, _ = plan(g)
    gd, _keep = _ffi.graph_desc(g)
    L = _ffi.lib()
    R = n_regs(info)
    out = []
    for nid in node_ids:
        base = nodes[nid][3]
        row = []
        for k in range(n_ports):
            v = _ffi.C.c_uint32(0)
            _ffi.check(L.kgpu_debug_init_reg(_ffi.C.byref(gd), nid, R - n_ports + k - base, _ffi.C.byref(v)))
            row.append(v.value)
        out.append(row)
    return out


def test_16384_input_tracks_plan_as_one_group_and_each_voice_holds_its_channel():
    g = Graph(16384, 2, 64, SR)
    ids = banks.input_bank(g, 16384, 1.0)
    g2 = Graph(16384, 2, 64, SR)
    banks.input_bank(g2, 16384, 1.0, source="saw")
    _nodes, info = plan(g)
    assert (info["n_groups"], info["n_voices"]) == (1, 16384)
    _nodes, info_saw = plan(g2)
    # the saw voice has a PolyBlep (5 registers) where the input voice has one port register
    assert n_regs(info) == n_regs(info_saw) - 5 + 1
    pick = [0, 1, 2, 777, 8191, 16383]
    assert port_channels(g, [ids["svf"][i] for i in pick], info, 1) == [[i] for i in pick]


def test_8192_stereo_tracks_plan_as_one_group_of_two_ports():
    g = Graph(16384, 2, 64, SR)
    ids = banks.input_bank(g, 8192, 1.0, stereo=True)
    _nodes, info = plan(g)
    assert (info["n_groups"], info["n_voices"]) == (1, 8192)
    pick = [0, 5, 4095, 8191]
    assert port_channels(g, [ids["env"][i] for i in pick], info, 2) == [[2 * i, 2 * i + 1] for i in pick]


def filter_voice(g, src, cutoff):
    return src.to(g.push(kn.SvfFilter(kn.SvfFilterType.Low, cutoff, 1.0, 0.0)))


def test_an_input_read_by_two_voices_stays_a_shared_signal():
    shared, own = Graph(1, 2, 64, SR), Graph(2, 2, 64, SR)
    with shared.edit() as e:
        for i in range(2):
            filter_voice(e, e.from_inputs(0), 500.0 * (i + 1)).out([0, 0]).to_graph_out()
    with own.edit() as e:
        for i in range(2):
            filter_voice(e, e.from_inputs(i), 500.0 * (i + 1)).out([0, 0]).to_graph_out()
    _n, info_shared = plan(shared)
    _n, info_own = plan(own)
    assert n_regs(info_shared) + 1 == n_regs(info_own)   # no port register: the input is read from its signal row


def test_17_shared_inputs_are_rejected_with_the_limit_in_the_message():
    def graph(n_in):
        g = Graph(n_in, 2, 64, SR)
        with g.edit() as e:
            for i in range(n_in):                          # every input read by two voices
                for k in range(2):
                    filter_voice(e, e.from_inputs(i), 300.0 * (k + 1) + i).out([0, 0]).to_graph_out()
        return g

    _n, info = plan(graph(16))
    assert info["n_voices"] == 32
    msg = rejected(graph(17))
    assert "17 graph inputs are shared" in msg and "at most 16" in msg, msg


def test_a_voice_reading_five_inputs_of_its_own_is_rejected():
    def graph(n_ports):
        g = Graph(n_ports, 1, 64, SR)
        with g.edit() as e:
            mix = e.from_inputs(0)
            for i in range(1, n_ports):
                mix = mix + e.from_inputs(i)
            filter_voice(e, mix, 800.0).to_graph_out()
        return g

    _n, info = plan(graph(4))
    assert info["n_voices"] == 1
    msg = rejected(graph(5))
    assert "5 graph inputs" in msg and "limit 4" in msg, msg


def test_65537_inputs_are_rejected():
    g = Graph(65536, 1, 64, SR)
    with g.edit() as e:
        filter_voice(e, e.from_inputs(65535), 800.0).to_graph_out()
    _n, info = plan(g)
    assert info["n_voices"] == 1
    g = Graph(65537, 1, 64, SR)
    with g.edit() as e:
        filter_voice(e, e.from_inputs(0), 800.0).to_graph_out()
    msg = rejected(g)
    assert "65537 graph inputs" in msg and "at most 65536" in msg, msg


def test_a_subtractive_bank_beside_an_input_bank_keeps_its_recipe():
    g = Graph(64, 2, 64, SR)
    banks.subtractive_bank(g, 64, 1.0)
    banks.input_bank(g, 64, 1.0)
    _n, info = plan(g)
    assert info["n_groups"] == 2
    g.take_events()
    srcs = _ffi.jit_source(g)                     # the templates no hand-written recipe takes
    assert len(srcs) == 1 and "ldin(" in srcs[0]  # ... is the input voice's alone


def port_route_graph(n):
    """input i -> SvfFilter whose cutoff is routed from input i * 2000 + 2500 -> out: one port read twice"""
    g = Graph(n, 2, 64, SR)
    with g.edit() as e:
        for i in range(n):
            svf = e.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0, 1.0, 0.0).ar_params())
            svf.link("cutoff_freq", e.from_inputs(i) * 2000.0 + 2500.0)
            e.from_inputs(i).to(svf).out([0, 0]).to_graph_out()
    return g


@pytest.mark.skipif(not nvrtc_available(), reason="libnvrtc not installed")
def test_port_templates_compile_with_nvrtc():
    shapes = [port_route_graph(4)]
    for kw in ({}, {"stereo": True}):
        g = Graph(8, 2, 64, SR)
        banks.input_bank(g, 4, 0.1, **kw)
        shapes.append(g)
    for g in shapes:
        g.take_events()
        srcs = _ffi.jit_source(g, tap_outputs=True)
        assert len(srcs) == 1 and "render_jit(FusedArgs a, const float *__restrict__ gin, uint32_t n_in)" in srcs[0]
        generated, _cached = _ffi.jit_compile(g, tap_outputs=True)
        assert generated == 1
    assert "pin[0]" in _ffi.jit_source(shapes[0])[0]


def digest_graphs():
    """the templates of the banks, fuzz seeds 11-26 and the route shapes, by name"""
    import test_gpu_ar_filters as arf
    import test_gpu_ar_routes as arr
    import test_gpu_fuzz as fz
    import test_gpu_large_voices as lv

    for bname in ("chain_bank", "partials_bank", "operator_bank", "subtractive_bank", "additive_bank"):
        g = Graph(0, 2, 64, SR)
        getattr(banks, bname)(g, 8, 0.1)
        yield bname, g
    g = Graph(0, 2, 64, SR)
    banks.fm_bank(g, 8)
    yield "fm", g
    for seed in range(11, 27):
        g = Graph(0, 2, 64, SR)
        kn.reset_randomness_seed(0)
        r = np.random.Generator(np.random.PCG64(seed))
        with g.edit() as ge:
            for vi in range(20):
                fz.random_voice(ge, r, vi).out([0, 0]).to_graph_out()
        yield f"fuzz{seed}", g
    for voice in (arf.lfo_cutoff, arf.env_cutoff, arf.lfo_q_and_onepole, arf.lfo_envelope_times):
        g = Graph(0, 2, 64, SR)
        with g.edit() as ge:
            for i in range(12):
                voice(ge, i).out([0, 0]).to_graph_out()
        yield voice.__name__, g
    for shape in arr.SHAPES:
        g = Graph(0, 2, 64, SR)
        arr.build_voices(g, shape)
        yield shape.__name__, g
    for shape in (lv.partials, lv.operators, lv.nodes_128, lv.slots_32):
        g = Graph(0, 2, 64, SR)
        shape(g, lv.SHAPES[shape])
        yield shape.__name__, g


def test_templates_without_ports_generate_the_same_source_as_before():
    # tests/golden/jit_source_digests.json: sha-256 (first 16 hex digits) of every generated source, written before ports existed
    with open(os.path.join(HERE, "golden", "jit_source_digests.json")) as f:
        golden = json.load(f)
    got = {}
    for name, g in digest_graphs():
        for tap in (False, True):
            if tap:
                g.take_events()
            got[f"{name}/{tap}"] = [hashlib.sha256(s.encode()).hexdigest()[:16] for s in _ffi.jit_source(g, tap)]
    assert got == golden
