"""GPU: graph inputs that one voice reads are ports of its template, read by the kernels from the caller's input blocks in
place -- host memory staged launch by launch (kgpu_render_inputs) or device memory (kgpu_render_inputs_device).  The chain:
input_i -> SvfFilter(Low) -> * EnvAsr.wr_mul(1/N) -> Pan2 -> bus (knaster_b200.banks.input_bank), against the oracle fed block by
block like knaster's AudioProcessor::run, on render_interp and render_jit."""
import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200 import banks
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions, Snapshot
from oracle.oracle import OracleProcessor

pytestmark = pytest.mark.gpu

SR = 48000
TOL = 1e-5


def tracks(n_tracks, n_blocks, bs, seed=21):
    """seeded noise plus a sine per track, [n_blocks][n_tracks][bs]"""
    r = np.random.Generator(np.random.PCG64(seed))
    t = np.arange(n_blocks * bs) / SR
    f = 55.0 * 2.0 ** r.uniform(0.0, 6.0, n_tracks)
    x = 0.3 * np.sin(2.0 * np.pi * f[:, None] * t[None, :]) + 0.1 * r.standard_normal((n_tracks, n_blocks * bs))
    return np.ascontiguousarray(x.astype(np.float32).reshape(n_tracks, n_blocks, bs).transpose(1, 0, 2))


def processor(n_in, n_out, build, bs=64, kernel="jit"):
    graph, proc = AudioProcessor.new(n_in, n_out, AudioProcessorOptions(block_size=bs, force_interpreter=kernel == "interp",
                                                                        force_jit=kernel == "jit"))
    return graph, proc, build(graph)


def oracle_render(n_in, n_out, build, x, bs=64):
    from knaster_b200.graph import Graph

    g = Graph(n_in, n_out, bs, SR)
    build(g)
    # events reach the oracle a block before they are due: like knaster, it drops an event that waits in its scheduler for longer
    # than it keeps them (the engine keeps every event, include/knaster_gpu.h kgpu_plan_push_events)
    ev = g.take_events()
    assert (ev["time_kind"] == 1).all()
    due = (ev["seconds"].astype(np.int64) * 282240000 + ev["subsec"]) * SR // 282240000
    orc = OracleProcessor(g, ring_buffer_size=1 << 22)
    out = np.zeros((x.shape[0], n_out, bs), np.float32)
    sent = 0
    order = np.argsort(due, kind="stable")
    for b in range(x.shape[0]):
        upto = int(np.searchsorted(due[order], (b + 2) * bs, side="left"))
        if upto > sent:
            g.pending_event_arrays.append(ev[np.sort(order[sent:upto])])
            sent = upto
        orc.run(list(x[b]))
        out[b] = orc.output_block()
    return out


def device_render(proc, x, n_out, bs):
    import torch

    xd = torch.from_numpy(x).cuda()
    out = torch.zeros((x.shape[0], n_out, bs), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    proc.render_device(x.shape[0], out.data_ptr(), inputs_device_ptr=xd.data_ptr())
    proc.synchronize()
    return out.cpu().numpy()


# ---- the chain bank against the oracle ------------------------------------------------------------------------------------
N_BANK, BANK_S = 512, 2.0
SAMPLED = [0, 1, 255, 511]


@pytest.fixture(scope="module")
def bank_renders():
    nb = int(BANK_S * SR) // 64
    x = tracks(N_BANK, nb, 64)
    res = {}
    for kernel in ("interp", "jit"):
        _g, proc, ids = processor(N_BANK, 2, lambda g: banks.input_bank(g, N_BANK, BANK_S), kernel=kernel)
        for v in SAMPLED:
            proc.add_tap(ids["pan"][v], 0)
            proc.add_tap(ids["pan"][v], 1)
        for v in range(2, N_BANK, 8):                  # voices not in SAMPLED: one tap per voice and channel
            proc.add_tap(ids["pan"][v], 0)
        out = proc.render(nb, inputs=x)
        res[kernel] = (out, proc.read_taps(), proc.info()["kernels"])
    ref = oracle_render(N_BANK, 2, lambda g: banks.input_bank(g, N_BANK, BANK_S), x)
    # the sampled voices alone, each on its own two outputs: their taps
    ref_own = oracle_render(len(SAMPLED), 2 * len(SAMPLED),
                            lambda g: banks.input_bank(g, N_BANK, BANK_S, only=SAMPLED, own_outputs=True), x[:, SAMPLED])
    return res, ref, ref_own


@pytest.mark.parametrize("kernel", ["interp", "jit"])
def test_input_bank_matches_the_oracle(kernel, bank_renders):
    res, ref, ref_own = bank_renders
    out, taps, kernels = res[kernel]
    assert kernels == ["render_interp" if kernel == "interp" else "render_jit"]
    assert np.abs(ref).max() > 1e-3 and np.isfinite(out).all()
    assert np.abs(out - ref).max() <= TOL
    own = ref_own.transpose(1, 0, 2).reshape(2 * len(SAMPLED), -1)     # [voice * 2 + channel][frame]
    assert np.abs(taps[: 2 * len(SAMPLED)] - own).max() <= TOL


def test_interpreter_and_generated_kernel_taps_are_bit_identical(bank_renders):
    res, _ref, _own = bank_renders
    assert np.array_equal(res["interp"][1], res["jit"][1])
    assert np.abs(res["jit"][1]).max() > 1e-3


# ---- other shapes -----------------------------------------------------------------------------------------------------------
def stereo(g):
    return banks.input_bank(g, 16, 0.5, stereo=True)


def port_routes(g):
    """input i -> SvfFilter(Low) with cutoff routed from input i * 2000 + 2500, times an EnvAsr"""
    with g.edit() as e:
        for i in range(16):
            svf = e.push(kn.SvfFilter(kn.SvfFilterType.Low, 1000.0, 2.0, 0.0).ar_params())
            svf.link("cutoff_freq", e.from_inputs(i) * 2000.0 + 2500.0)
            env = e.push(kn.EnvAsr(0.01, 0.05).wr_mul(1.0 / 16))
            env.param("t_restart").trig_at(kn.Seconds.from_samples(100 + 300 * i, SR))
            env.param("t_release").trig_at(kn.Seconds.from_samples(12000 + 50 * i, SR))
            (e.from_inputs(i).to(svf) * env).out([0, 0]).to_graph_out()


def mixed(g):
    """ports 0..11 through their own filters, each multiplied by the shared side chain (input 12); input 13 wired to output 1"""
    with g.edit() as e:
        for i in range(12):
            svf = e.push(kn.SvfFilter(kn.SvfFilterType.Band, 300.0 * (i + 1), 3.0, 0.0))
            (e.from_inputs(i).to(svf) * e.from_inputs(12) * (1.0 / 12)).out([0, 0]).to_graph_out()
        e.from_inputs(13).to_graph_out_channels(1)


SHAPES = {"stereo": (16 * 2, stereo), "port_routes": (16, port_routes), "mixed": (14, mixed)}


@pytest.mark.parametrize("kernel", ["interp", "jit"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_shapes_match_the_oracle(shape, kernel):
    n_in, build = SHAPES[shape]
    nb = SR // 2 // 64
    x = tracks(n_in, nb, 64, seed=5)
    _g, proc, _ids = processor(n_in, 2, build, kernel=kernel)
    out = proc.render(nb, inputs=x)
    ref = oracle_render(n_in, 2, build, x)
    assert np.abs(ref).max() > 1e-3
    assert np.abs(out - ref).max() <= TOL, (shape, kernel, float(np.abs(out - ref).max()))
    assert np.array_equal(device_render(processor(n_in, 2, build, kernel=kernel)[1], x, 2, 64), out)


# ---- host, device, block by block, launch splits, block sizes ------------------------------------------------------------
def small_bank(n, seconds):
    return lambda g: banks.input_bank(g, n, seconds)


@pytest.mark.parametrize("kernel", ["interp", "jit"])
def test_host_device_and_launch_splits_are_bit_identical(kernel):
    n, nb = 64, 300
    x = tracks(n, nb, 64, seed=8)

    def fresh():
        _g, proc, ids = processor(n, 2, small_bank(n, nb * 64 / SR), kernel=kernel)
        for v in range(0, n, 4):
            proc.add_tap(ids["pan"][v], 0)
        return proc

    p = fresh()
    one = p.render(nb, inputs=x)
    one_taps = p.read_taps()
    assert np.abs(one).max() > 1e-4
    p = fresh()
    assert np.array_equal(device_render(p, x, 2, 64), one)
    assert np.array_equal(p.read_taps(), one_taps)
    for bpl in (1, 7):
        p = fresh()
        p.set_blocks_per_launch(bpl)
        assert np.array_equal(p.render(nb, inputs=x), one), bpl
        assert np.array_equal(p.read_taps(), one_taps), bpl
    p = fresh()
    outs, taps = [], []
    for b in range(nb):
        p.run(list(x[b]))
        outs.append(p.output_block())
        taps.append(p.read_taps())
    assert np.array_equal(np.stack(outs), one)
    assert np.array_equal(np.concatenate(taps, axis=1), one_taps)


@pytest.mark.parametrize("bs", [16, 40, 64, 96])
def test_block_sizes(bs):
    n, nb = 32, (SR // 4) // bs
    x = tracks(n, nb, bs, seed=bs)
    build = small_bank(n, nb * bs / SR)
    ref = oracle_render(n, 2, build, x, bs=bs)
    taps = {}
    for kernel in ("interp", "jit"):
        _g, proc, ids = processor(n, 2, build, bs=bs, kernel=kernel)
        for v in range(n):
            proc.add_tap(ids["pan"][v], 1)
        out = proc.render(nb, inputs=x)
        taps[kernel] = proc.read_taps()
        assert np.abs(out - ref).max() <= TOL, (bs, kernel)
        assert np.array_equal(device_render(processor(n, 2, build, bs=bs, kernel=kernel)[1], x, 2, bs), out)
    assert np.array_equal(taps["interp"], taps["jit"])


@pytest.mark.parametrize("kernel", ["interp", "jit"])
def test_snapshot_restored_into_a_fresh_processor_continues_bit_identically(kernel):
    n, nb = 64, 600
    x = tracks(n, nb, 64, seed=13)
    build = small_bank(n, nb * 64 / SR)
    _g, p1, ids = processor(n, 2, build, kernel=kernel)
    p1.add_tap(ids["pan"][3], 0)
    p1.render(277, inputs=x[:277])                          # mid-note, mid-block of a launch
    image = p1.snapshot().to_bytes()
    cont = p1.render(nb - 277, inputs=x[277:])
    cont_taps = p1.read_taps()
    g2, p2, ids2 = processor(n, 2, build, kernel=kernel)
    p2.add_tap(ids2["pan"][3], 0)
    g2.take_events()                                        # its events are inside the image
    p2.restore(Snapshot.from_bytes(image))
    assert p2.frame_clock() == 277 * 64
    assert np.array_equal(p2.render(nb - 277, inputs=x[277:]), cont)
    assert np.array_equal(p2.read_taps(), cont_taps)
    assert np.abs(cont).max() > 1e-4


# ---- full size ---------------------------------------------------------------------------------------------------------------
def device_tracks(n_tracks, n_blocks, bs, seed=99):
    """tracks() on the device, [n_blocks][n_tracks][bs]: 31.5 GB for 16 384 tracks x 10 s"""
    import torch

    gen = torch.Generator(device="cuda").manual_seed(seed)
    f = 55.0 * 2.0 ** (torch.rand(n_tracks, generator=gen, device="cuda", dtype=torch.float64) * 6.0)
    x = torch.empty((n_blocks, n_tracks, bs), dtype=torch.float32, device="cuda")
    step = 250
    for b0 in range(0, n_blocks, step):
        b1 = min(n_blocks, b0 + step)
        t = torch.arange(b0 * bs, b1 * bs, device="cuda", dtype=torch.float64).reshape(b1 - b0, 1, bs) / SR
        s = 0.3 * torch.sin(2.0 * np.pi * f.reshape(1, -1, 1) * t)
        x[b0:b1] = (s + 0.1 * torch.randn((b1 - b0, n_tracks, bs), generator=gen, device="cuda", dtype=torch.float64)).float()
    return x


def test_16384_tracks_10s_from_device_memory_equal_each_voice_alone():
    import torch

    n, seconds = 16384, 10.0
    nb = int(seconds * SR) // 64
    x = device_tracks(n, nb, 64)
    graph, proc = AudioProcessor.new(n, 2, AudioProcessorOptions())
    ids = banks.input_bank(graph, n, seconds)
    r = np.random.Generator(np.random.PCG64(3))
    sampled = sorted(r.choice(n, 64, replace=False).tolist())
    for v in sampled:
        proc.add_tap(ids["pan"][v], 0)
    out = torch.zeros((nb, 2, 64), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    proc.render_device(nb, out.data_ptr(), inputs_device_ptr=x.data_ptr())
    proc.synchronize()
    assert proc.info()["kernels"] == ["render_jit"]
    taps = proc.read_taps()
    bus = out.cpu().numpy()
    assert np.isfinite(bus).all() and np.abs(bus).max() > 1e-3
    for k, v in enumerate(sampled):
        # the same voice alone, its input also read by a second voice: a shared input, rendered through its signal row
        g1, p1 = AudioProcessor.new(1, 2, AudioProcessorOptions())
        own = banks.input_bank(g1, n, seconds, only=[v])
        with g1.edit() as e:
            e.from_inputs(0).to(e.push(kn.SvfFilter(kn.SvfFilterType.High, 500.0, 1.0, 0.0))).out([0, 0]).to_graph_out()
        p1.add_tap(own["pan"][0], 0)
        p1.render(nb, inputs=np.ascontiguousarray(x[:, v : v + 1].cpu().numpy()))
        assert np.array_equal(p1.read_taps()[0], taps[k]), v
    assert np.abs(taps).max() > 1e-5                        # a voice's share of the bus: wr_mul(1 / 16384)
    # host-fed, 1 s: the same as device-fed
    nb1 = SR // 64
    x1 = x[:nb1].contiguous()
    g_h, p_h = AudioProcessor.new(n, 2, AudioProcessorOptions())
    banks.input_bank(g_h, n, 1.0)
    host = p_h.render(nb1, inputs=x1.cpu().numpy())
    g_d, p_d = AudioProcessor.new(n, 2, AudioProcessorOptions())
    banks.input_bank(g_d, n, 1.0)
    out1 = torch.zeros((nb1, 2, 64), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    p_d.render_device(nb1, out1.data_ptr(), inputs_device_ptr=x1.data_ptr())
    p_d.synchronize()
    assert np.array_equal(out1.cpu().numpy(), host)
    assert np.abs(host).max() > 1e-3
