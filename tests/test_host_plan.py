"""CPU tests of the product's host side: the C ABI surface, the plan compiler (voice discovery,
template grouping) and the control-rate event simulation.  No GPU needed: the device's part for
the fixtures used here is trivial ("hold the last value written to a register"), so the device
event stream can be replayed in numpy and compared with the oracle's render of the same graph."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200 import _ffi
from knaster_b200.graph import Graph
from oracle.oracle import OracleProcessor

SR = 48000


def f32(bits):
    return np.array([bits], dtype=np.uint32).view(np.float32)[0]


def test_library_exports_every_declared_symbol():
    lib = _ffi.lib()
    src = open(_ffi.HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = set(re.findall(r"\b(kgpu_[a-z_0-9]+)\s*\(", src))
    assert len(names) >= 18
    for n in sorted(names):
        assert hasattr(lib, n), f"libknaster_gpu.so does not export {n}"
    assert lib.kgpu_abi_version() == _ffi.KGPU_ABI_VERSION
    assert lib.kgpu_device_count() >= 0


def test_rust_binding_declares_every_entry_point():
    # rust/knaster_gpu/src/ffi.rs (the text of INTEGRATION.md as a crate; not compiled here: no cargo/rustc in
    # this image) must at least name every function the header exports, and nothing else
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = re.sub(r"/\*.*?\*/", "", open(_ffi.HEADER).read(), flags=re.S)
    names = set(re.findall(r"\b(kgpu_[a-z_0-9]+)\s*\(", src))
    for path in ("rust/knaster_gpu/src/ffi.rs", "INTEGRATION.md"):
        decl = set(re.findall(r"pub fn (kgpu_[a-z_0-9]+)\(", open(os.path.join(root, path)).read()))
        assert decl == names, (path, sorted(names ^ decl))


def test_event_struct_layout_matches_header():
    from knaster_b200.graph import EVENT_DTYPE

    assert EVENT_DTYPE.itemsize == 48
    assert EVENT_DTYPE.fields["value"][1] == 16 and EVENT_DTYPE.fields["seconds"][1] == 36


def held_value_render(graph, node, n_blocks, reg_offset=0, blocks_per_call=0, init=0.0):
    """Replay the device events of `node`'s register reg_base+reg_offset: out[f] = last write."""
    ev = graph.take_events()
    evs, nodes, info = _ffi.debug_simulate(graph, ev, n_blocks, blocks_per_call)
    grp, voice, local, reg_base = nodes[node]
    out = np.full(n_blocks * graph.block_size, init, dtype=np.float32)
    writes = [(fr, f32(val)) for (g, v, n, op, reg, val, fr) in evs if (g, v, n) == (grp, voice, local) and op == 0 and reg == reg_base + reg_offset]
    last = -1
    for fr, val in writes:  # device order per voice
        assert fr >= last, "device events must be time-ordered for a frame-major kernel"
        last = fr
        out[fr:] = val
    return out, info, ev


def oracle_render(graph, events, n_blocks):
    p = OracleProcessor(graph, ring_buffer_size=1 << 20)
    graph.pending_event_arrays = [events] if len(events) else []
    out, _ = p.render(n_blocks)
    return out[:, 0, :].reshape(-1), p


def two_ways(build, n_blocks, block_size=16, reg_offset=0, blocks_per_call=0):
    g1 = Graph(0, 1, block_size, SR)
    n1 = build(g1)
    dev, info, ev = held_value_render(g1, n1, n_blocks, reg_offset, blocks_per_call)
    g2 = Graph(0, 1, block_size, SR)
    build(g2)
    g2.take_events()
    ref, orc = oracle_render(g2, ev, n_blocks)
    return dev, ref, info, orc


def at(fr):
    return kn.Seconds.from_samples(fr, SR)


def test_precise_timing_events_match_oracle():
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestInPlusParamUGen().precise_timing(4))
            n.to_graph_out()
            p = n.param("number")
            p.set(0.5)                       # no time: block 0 start
            p.set_at(1.0, at(5))
            p.set_at(2.0, at(6))
            p.set_at(3.0, at(32))            # aligned after non-aligned: sticky delay 6 (App. B1)
            p.set_at(4.0, at(70))
            p.set_at(5.0, at(71))
            p.set_at(6.0, at(71))
            p.set_at(7.0, at(100))
        return n.id()

    dev, ref, info, _ = two_ways(build, 8)
    assert np.array_equal(dev, ref)
    assert info["dropped_changes"] == 0


def test_precise_timing_queue_overflow_and_blocking_order():
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestInPlusParamUGen().precise_timing(2))
            n.to_graph_out()
            p = n.param(0)
            p.set_at(1.0, at(10))   # queued (delay 10)
            p.set_at(2.0, at(4))    # queued behind the first: waits until frame 10 (precise_timing.rs:82-94)
            p.set_at(3.0, at(12))   # queue full (N=2): dropped + logged (precise_timing.rs:129-134)
            p.set_at(4.0, at(40))
        return n.id()

    dev, ref, info, orc = two_ways(build, 4)
    assert np.array_equal(dev, ref)
    assert info["dropped_changes"] == 1 and orc.log_count() == 1
    assert ref[9] == 0.0 and ref[10] == 2.0  # both applied at frame 10, in queue order


def test_events_without_precise_timing_apply_at_block_start():
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestInPlusParamUGen())
            n.to_graph_out()
            n.param(0).set_at(1.0, at(21))
            n.param(0).set_at(2.0, at(47))
        return n.id()

    dev, ref, info, orc = two_ways(build, 4)
    assert np.array_equal(dev, ref)
    assert info["ignored_delays"] == 2 == orc.log_count()


@pytest.mark.parametrize("blocks_per_call", [0, 1, 3])
def test_smoothing_ramp_matches_oracle(blocks_per_call):
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestInPlusParamUGen().smooth_params())
            n.to_graph_out()
            p = n.param("number")
            p.smooth(kn.ParameterSmoothing.Linear(0.01))       # 480 frames = 30 blocks of 16
            p.set(1.0)                                         # ramp starts from 0.0 (App. B2)
            p.set_at(-0.5, at(16 * 12))                        # retarget mid-ramp
            p.smooth_at(kn.ParameterSmoothing.Linear(0.002), at(16 * 50))
            p.set_at(0.25, at(16 * 50))
            p.smooth_at(kn.ParameterSmoothing.NoSmoothing(), at(16 * 70))
            p.set_at(2.0, at(16 * 71))
        return n.id()

    dev, ref, _, _ = two_ways(build, 80, blocks_per_call=blocks_per_call)
    assert np.array_equal(dev, ref)
    assert 0.0 < ref[16 * 5] < 1.0


def test_smoothing_advances_once_per_partial_block():
    # App. B3: under an outer WrPreciseTiming split the ramp advances per process_block call
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestInPlusParamUGen().smooth_params().precise_timing(4))
            n.to_graph_out()
            p = n.param(0)
            p.smooth(kn.ParameterSmoothing.Linear(0.01))
            p.set(1.0)
            p.set_at(0.0, at(16 * 3 + 5))
            p.set_at(0.5, at(16 * 3 + 9))
        return n.id()

    dev, ref, _, _ = two_ways(build, 40)
    assert np.array_equal(dev, ref)


def test_wr_mul_param_and_smoothing():
    # SinWt.wr_mul(a).smooth_params(): "wr_mul" is parameter index 3 (T::Parameters, math.rs:78)
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestNumUGen(1.0).wr_mul(0.25).smooth_params())
            n.to_graph_out()
            assert n.param("wr_mul").param_index == 0
            n.param("wr_mul").smooth(kn.ParameterSmoothing.Linear(0.004))
            n.param("wr_mul").set_at(0.75, at(64))
        return n.id()

    g1 = Graph(0, 1, 16, SR)
    n1 = build(g1)
    # register 0 = TestNum value, register 1 = WrMul value
    dev, info, ev = held_value_render(g1, n1, 20, reg_offset=1, init=0.25)
    g2 = Graph(0, 1, 16, SR)
    build(g2)
    g2.take_events()
    ref, _ = oracle_render(g2, ev, 20)
    assert np.array_equal(dev, ref)  # 1.0 * value


def test_relative_and_late_events():
    def build(graph):
        with graph.edit() as g:
            n = g.push(kn.TestInPlusParamUGen().precise_timing(4))
            n.to_graph_out()
            n.param(0).set_after(1.0, at(37))   # Time::after
            n.param(0).set_time(2.0, kn.Time.asap())
        return n.id()

    dev, ref, _, _ = two_ways(build, 5)
    assert np.array_equal(dev, ref)
    assert ref[0] == 2.0 and ref[36] == 2.0 and ref[37] == 1.0


# ---------------------------------------------------------------- plan compiler
def build_bank(n_voices, stereo=True, vary=False):
    graph = Graph(0, 2 if stereo else 1, 64, SR)
    with graph.edit() as g:
        for i in range(n_voices):
            saw = g.push(kn.PolyBlep(kn.Waveform.Sawtooth, 110.0 + i).precise_timing(8))
            svf = g.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0 + i, 0.7, 0.0).precise_timing(8))
            env = g.push(kn.EnvAsr(0.01, 0.1).wr_mul(1.0 / n_voices).precise_timing(8))
            sig = (saw >> svf) * env
            if vary and i % 2:
                sig = sig * 0.5
            (sig.out([0, 0]) if stereo else sig).to_graph_out()
    return graph


def test_voice_discovery_groups_isomorphic_voices():
    graph = build_bank(40)
    _, nodes, info = _ffi.debug_simulate(graph, graph.take_events(), 1)
    assert info["n_groups"] == 1 and info["n_voices"] == 40
    assert info["n_mix_nodes"] == 2 * 39            # one left-fold Add chain per output channel
    assert sum(1 for n in nodes if n[0] < 0) == 2 * 39
    # voice order follows the left fold = call order; 4 nodes per voice (saw, svf, env, mul)
    voices = [n[1] for n in nodes if n[0] == 0]
    assert voices[:8] == [0, 0, 0, 0, 1, 1, 1, 1]


def test_voice_discovery_two_shapes_two_groups():
    graph = build_bank(10, vary=True)
    _, _, info = _ffi.debug_simulate(graph, graph.take_events(), 1)
    assert info["n_groups"] == 2 and info["n_voices"] == 10


def test_readme_graph_is_one_voice():
    graph = Graph(0, 2, 64, SR)
    with graph.edit() as g:
        sine = g.push(kn.SinWt(440.0))
        (sine * 0.2).out([0, 0]).to_graph_out()
    _, nodes, info = _ffi.debug_simulate(graph, graph.take_events(), 1)
    assert (info["n_groups"], info["n_voices"], info["n_mix_nodes"]) == (1, 1, 0)
    gd, _keep = _ffi.graph_desc(graph)
    val = C.c_uint32()
    _ffi.check(_ffi.lib().kgpu_debug_init_reg(C.byref(gd), 0, 2, C.byref(val)))
    k = 16384.0 * 65536.0 * (1.0 / 48000.0)
    assert val.value == int(float(np.float32(440.0)) * k)   # SinWt phase_increment after init(), osc.rs:142-147


def expect_error(graph, code, events=None):
    with pytest.raises(_ffi.KgpuError) as ei:
        _ffi.debug_simulate(graph, graph.take_events() if events is None else events, 1)
    assert ei.value.code == code, ei.value


def test_unsupported_shapes_are_rejected_not_faked():
    g = Graph(1, 1, 64, SR)                              # graph inputs compile since round 2 (rendered with kgpu_render_inputs)
    with g.edit() as e:
        e.from_inputs(0).to_graph_out()
    _evs, _nodes, info = _ffi.debug_simulate(g, g.take_events(), 2)
    assert info["n_voices"] == 0

    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        lfo = e.push(kn.SinWt(3.0))
        env = e.push(kn.EnvAsr(0.01, 0.1).ar_params())
        env.link("t_restart", lfo * 0.001 + 0.01)
        (e.push(kn.SinWt(100.0)) * env).to_graph_out()
    expect_error(g, _ffi.KGPU_ERR_UNSUPPORTED)          # audio-rate route into a trigger (a type error in knaster too): rejected

    g = Graph(0, 1, 64, SR)                             # ... into an envelope TIME it compiles (round 2)
    with g.edit() as e:
        lfo = e.push(kn.SinWt(3.0))
        env = e.push(kn.EnvAsr(0.01, 0.1).ar_params())
        env.link("attack_time", lfo * 0.001 + 0.01)
        (e.push(kn.SinWt(100.0)) * env).to_graph_out()
    _evs, _nodes, info = _ffi.debug_simulate(g, g.take_events(), 2)
    assert info["n_voices"] == 1

    g = Graph(0, 1, 64, SR)                             # ... into filter parameters it is (round 2): the plan compiles
    with g.edit() as e:
        lfo = e.push(kn.SinWt(3.0))
        f = e.push(kn.SvfFilter(kn.SvfFilterType.Low, 500.0, 1.0, 0.0).ar_params())
        f.link("cutoff_freq", lfo * 100.0 + 500.0)
        e.push(kn.SinWt(100.0)).to(f).to_graph_out()
    _evs, _nodes, info = _ffi.debug_simulate(g, g.take_events(), 4)
    assert info["n_voices"] == 1

    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        n = e.push(kn.PolyBlep(kn.Waveform.Square, 100.0))
        n.to_graph_out()
        n.param("waveform").set(14)
    expect_error(g, _ffi.KGPU_ERR_PARAMETER)            # no such Waveform


    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        a = e.push(kn.SinWt(100.0))
        b = e.push(kn.SinWt(200.0))
        f = e.push(kn.OnePoleLpf(500.0))
        a.to_graph_out()
        b.to_graph_out()
    g.connect2(2 + 1, 0, 0, f.id())                     # the mix Add feeds a filter: post-mix processing
    g.connect2(f.id(), 0, 0, -2)
    g.commit_changes()
    # the Add now has fan-out 2 => it is an ordinary voice node and everything merges into one voice
    _, _, info = _ffi.debug_simulate(g, g.take_events(), 1)
    assert info["n_voices"] == 1


def test_bad_events_are_reported_with_knaster_error_names():
    g = Graph(0, 1, 64, SR)
    with g.edit() as e:
        n = e.push(kn.SinWt(100.0))
        n.to_graph_out()
    from knaster_b200.graph import EVENT_DTYPE

    ev = np.zeros(1, EVENT_DTYPE)
    ev["node"], ev["param"], ev["value_kind"] = 0, 7, 1
    expect_error(g, _ffi.KGPU_ERR_PARAMETER, ev)        # ParameterIndexOutOfBounds
    ev["param"], ev["value_kind"] = 0, 3
    expect_error(g, _ffi.KGPU_ERR_PARAMETER, ev)        # integer sent to a float parameter
    ev["value_kind"], ev["smoothing_kind"] = 1, 2
    expect_error(g, _ffi.KGPU_ERR_PARAMETER, ev)        # smoothing without WrSmoothParams
    ev["smoothing_kind"], ev["node"] = 0, 5
    expect_error(g, _ffi.KGPU_ERR_INVALID, ev)          # NodeNotFound


def test_sinf_restatement_matches_libm():
    """csrc/sinf_glibc.h (the device sine, host instantiation) against the libm the oracle links:
    bit-for-bit over random + structured arguments in the domain SinNumeric / PolyBlep use, and over large ones
    (a SinNumeric at a negative frequency or with a large phase offset reaches |x| >= 120)."""
    import ctypes.util

    lib = _ffi.lib()
    lib.kgpu_debug_sinf.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.sinf.restype = C.c_float
    libm.sinf.argtypes = [C.c_float]
    rng = np.random.Generator(np.random.PCG64(7))
    xs = np.concatenate([
        rng.uniform(0.0, 2.0 * np.pi * 1.5, 400_000),            # (phase + offset) * TAU, phase in [0, 1]
        rng.uniform(-16.0, 16.0, 200_000),
        rng.uniform(-119.9, 119.9, 100_000),                     # whole reduce_fast domain
        np.float32(np.pi / 4) + np.arange(-2000, 2000) * np.float32(1e-7),
        np.logspace(-14, 0, 5000), [0.0, -0.0, 1e-30, 130.0, -500.0],
        rng.uniform(-2.0 ** 20, -120.0, 100_000),                # glibc's reduce_large domain
        rng.uniform(120.0, 2.0 ** 20, 100_000),
        np.float32(120.0) + np.arange(-500, 500) * np.float32(2.0 ** -17),   # both sides of the path switch
        -np.logspace(2.08, 38.5, 20_000), np.logspace(2.08, 38.5, 20_000),
        [np.finfo(np.float32).max, -np.finfo(np.float32).max],
    ]).astype(np.float32)
    ys = np.empty_like(xs)
    _ffi.check(lib.kgpu_debug_sinf(xs.ctypes.data, ys.ctypes.data, len(xs)))
    ref = np.array([libm.sinf(float(x)) for x in xs], dtype=np.float32)
    assert (np.abs(xs) >= 120.0).sum() > 200_000
    assert np.array_equal(ys.view(np.uint32), ref.view(np.uint32))
    special = np.array([np.inf, -np.inf, np.nan], dtype=np.float32)
    ys = np.empty_like(special)
    _ffi.check(lib.kgpu_debug_sinf(special.ctypes.data, ys.ctypes.data, len(special)))
    assert np.isnan(ys).all()


def test_event_calendar_does_not_change_what_the_device_sees():
    # Block-by-block calls under a long queue of scheduled events switch the host's calendar on (plan.cpp
    # calendar_update: near / far queues).  The device event stream must be the one a single call produces --
    # including same-frame events whose arrival order decides the final value, and events due far ahead.
    n_nodes, n_blocks = 48, 400
    rng = np.random.Generator(np.random.PCG64(9))
    g = Graph(0, 1, 16, SR)
    ids = []
    with g.edit() as e:
        for i in range(n_nodes):
            n = e.push(kn.Constant(float(i)).precise_timing(8))
            n.to_graph_out()
            ids.append(n.id())
    frames = rng.integers(0, n_blocks * 16, (n_nodes, 420))
    frames[:, :40] = frames[:, 40:80]                     # same-frame pairs: the later arrival must win
    order = rng.permutation(n_nodes * 420)                # arrival order unrelated to due time
    nodes = np.repeat(np.asarray(ids, dtype=np.uint32), 420)[order]
    fr = frames.reshape(-1)[order].astype(np.uint64)
    vals = rng.uniform(-1.0, 1.0, len(fr))
    g.schedule_bulk(nodes, np.zeros(len(fr)), np.ones(len(fr)), vals, fr)
    ev = g.take_events()
    assert len(ev) > 16384
    one, _, info1 = _ffi.debug_simulate(g, ev, n_blocks, 0)
    per_block, _, info2 = _ffi.debug_simulate(g, ev, n_blocks, 1)
    assert info1["device_events"] == info2["device_events"] and info1["dropped_changes"] == info2["dropped_changes"]

    def per_voice(evs):
        d = {}
        for (grp, voice, node, op, reg, val, frame) in evs:
            d.setdefault((grp, voice), []).append((frame, node, op, reg, val))
        return d

    a, b = per_voice(one), per_voice(per_block)
    assert a.keys() == b.keys()
    for k in a:
        assert a[k] == b[k], f"voice {k}: device events differ between one call and block-by-block calls"


def test_driver_slice_leaves_the_event_stream_unchanged(monkeypatch):
    """With few worker threads the calling thread simulates a slice of the voices itself (HostPlan::driver_slice_through).
    The device event stream -- per voice and in order -- must not depend on how the voices are split over threads:
    1 thread (inline), 3 workers + the caller's half slice, 9 workers (no slice of its own), for two launch splits,
    on a bank with smoothing ramps (additive) and one with sample-accurate events (subtractive)."""
    from knaster_b200 import banks

    for wl, nv, secs in (("subtractive", 1536, 2.0), ("additive", 4608, 2.0)):
        n_blocks = int(secs * 48000) // 64
        ref = None
        for threads in ("1", "3", "9"):
            monkeypatch.setenv("KGPU_THREADS", threads)
            for bpc in (0, 400):
                g = Graph(0, 2, 64, 48000)
                banks.bank_builder(wl, secs)(g, nv, 0, nv)
                ev = g.take_events()
                assert len(ev) > 20000  # large enough for the pooled path
                evs, _, info = _ffi.debug_simulate(g, ev, n_blocks, bpc, cap=1 << 21)
                key = (sorted(evs, key=lambda e: (e[0], e[1])), info["device_events"], info["dropped_changes"], info["ignored_delays"])
                if ref is None:
                    ref = key
                assert key[1:] == ref[1:], (wl, threads, bpc)
                assert key[0] == ref[0], (wl, threads, bpc)


def test_traffic_records_are_well_formed():
    """profiles/traffic.json feeds `roofline.traffic` of every bench line (bench.py roofline_of): numbers where numbers are read."""
    import json
    import os

    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "traffic.json")) as f:
        tj = json.load(f)
    assert {"render_sub_asr", "render_sub_seg", "render_fm2", "render_add_wt", "render_jit"} <= set(tj)
    for name, rec in tj.items():
        assert isinstance(rec["source"], str), name
        for key in ("frames_per_launch", "voices"):
            assert isinstance(rec[key], int) and rec[key] > 0, (name, key)
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum", "traffic_bytes_per_launch"):
            assert isinstance(rec[key], (int, float)) and rec[key] >= 0, (name, key)
        assert abs(rec["traffic_bytes_per_launch"] - rec["dram__bytes_read.sum"] - rec["dram__bytes_write.sum"]) < 1.0, name
