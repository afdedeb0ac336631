"""Synthetic voice banks: the workloads of BASELINE.json / SURVEY.md section 8d, built through
the knaster-style builder API.  Used by bench.py and by the parity tests (at reduced sizes)."""
from __future__ import annotations

from typing import List, Tuple

import numpy as np

from . import ugens as U
from .graph import Graph


def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64(seed))


def readme_sine(graph: Graph) -> List[int]:
    """configs[0]: README.md:35-47 -- SinWt 440 Hz * 0.2 to stereo out."""
    with graph.edit() as g:
        sine = g.push(U.SinWt(440.0))
        sig = sine * 0.2
        sig.out([0, 0]).to_graph_out()
    return [sig._outputs[0][0]]


def additive_bank(graph: Graph, n_voices: int, seconds: float, seed: int = 1001, n_changes: int = 4,
                  voice_offset: int = 0, total_voices: int = 0) -> List[int]:
    """configs[1]: n_voices x SinWt(f).wr_mul(a).smooth_params() -> stereo, amplitude smoothing
    Linear(0.05) and `n_changes` block-aligned amplitude changes per voice.
    voice_offset/total_voices select a shard of a larger bank (same random stream)."""
    total = total_voices or n_voices
    r = _rng(seed)
    f = 55.0 * 2.0 ** r.uniform(0.0, 7.0, total)
    a = r.uniform(0.2, 1.0, total) / total
    n_blocks = int(round(seconds * graph.sample_rate)) // graph.block_size
    ch_block = r.integers(0, max(1, n_blocks), (total, n_changes))
    ch_val = r.uniform(0.0, 1.0, (total, n_changes)) / total
    sl = slice(voice_offset, voice_offset + n_voices)
    f, a, ch_block, ch_val = f[sl], a[sl], ch_block[sl], ch_val[sl]
    ids = []
    with graph.edit() as g:
        for i in range(n_voices):
            v = g.push(U.SinWt(float(f[i])).wr_mul(float(a[i])).smooth_params())
            v.out([0, 0]).to_graph_out()
            ids.append(v.id())
    ids_a = np.asarray(ids, dtype=np.uint32)
    wr_mul = 3  # SinWt has 3 parameters; "wr_mul" is index T::Parameters
    # smoothing setting at t = 0, then the changes (sorted per voice by time)
    n = n_voices
    graph.schedule_bulk(ids_a, np.full(n, wr_mul), np.zeros(n), np.zeros(n), np.zeros(n, dtype=np.uint64),
                        smooth_seconds=np.full(n, 0.05, dtype=np.float32))
    order = np.argsort(ch_block, axis=1, kind="stable")
    cb = np.take_along_axis(ch_block, order, 1)
    cv = np.take_along_axis(ch_val, order, 1)
    graph.schedule_bulk(np.repeat(ids_a, n_changes), np.full(n * n_changes, wr_mul), np.ones(n * n_changes),
                        cv.reshape(-1), (cb.reshape(-1) * graph.block_size).astype(np.uint64))
    return ids


def subtractive_bank(graph: Graph, n_voices: int, seconds: float, seed: int = 2002, n_notes: int = 8,
                     envelope: str = "asr", voice_offset: int = 0, total_voices: int = 0,
                     stereo: bool = True) -> List[int]:
    """configs[2] / configs[4]: n_voices x PolyBlep(Sawtooth) -> SvfFilter(Low) -> * EnvAsr.wr_mul(1/N)
    (VCA = MathUGen<Mul>), every UGen under precise_timing::<8>(), with sample-accurate note events:
    note-on = t_restart + freq + cutoff_freq at a random frame, note-off = t_release 0.1-0.4 s later.
    envelope="segments": the Envelope variant (A, D, R segments; t_restart / t_stop / jump_to_segment)."""
    total = total_voices or n_voices
    sr = graph.sample_rate
    n_frames = int(round(seconds * sr))
    r = _rng(seed)
    midi = r.integers(36, 85, total)
    fc = r.uniform(200.0, 8000.0, total)
    q = r.uniform(0.5, 8.0, total)
    att = r.uniform(0.002, 0.05, total)
    rel = r.uniform(0.05, 0.5, total)
    on = np.sort(r.integers(0, max(1, n_frames), (total, n_notes)), axis=1)
    note_midi = r.integers(36, 85, (total, n_notes))
    note_fc = r.uniform(200.0, 8000.0, (total, n_notes))
    off = on + (r.uniform(0.1, 0.4, (total, n_notes)) * sr).astype(np.int64)
    sl = slice(voice_offset, voice_offset + n_voices)
    midi, fc, q, att, rel, on, note_midi, note_fc, off = (x[sl] for x in (midi, fc, q, att, rel, on, note_midi, note_fc, off))
    f0 = 440.0 * 2.0 ** ((midi - 69) / 12.0)
    note_f = 440.0 * 2.0 ** ((note_midi - 69) / 12.0)
    saw_ids, svf_ids, env_ids, out_ids = [], [], [], []
    with graph.edit() as g:
        for i in range(n_voices):
            saw = g.push(U.PolyBlep(U.Waveform.Sawtooth, float(f0[i])).precise_timing(8))
            svf = g.push(U.SvfFilter(U.SvfFilterType.Low, float(fc[i]), float(q[i]), 0.0).precise_timing(8))
            if envelope == "asr":
                env = g.push(U.EnvAsr(float(att[i]), float(rel[i])).wr_mul(1.0 / total).precise_timing(8))
            else:
                env = g.push(U.Envelope(0.0, [U.EnvelopeSegment(float(att[i]), 1.0), U.EnvelopeSegment(0.05, 0.6),
                                              U.EnvelopeSegment(float(rel[i]), 0.0)]).wr_mul(1.0 / total).precise_timing(8))
            sig = (saw >> svf) * env
            (sig.out([0, 0]) if stereo else sig).to_graph_out()
            saw_ids.append(saw.id()); svf_ids.append(svf.id()); env_ids.append(env.id()); out_ids.append(sig._outputs[0][0])
    saw_a, svf_a, env_a = (np.asarray(x, dtype=np.uint32) for x in (saw_ids, svf_ids, env_ids))
    V, K = n_voices, n_notes
    rep = lambda a: np.repeat(a, K)
    FLOAT, TRIG, INT = 1, 2, 3
    if envelope == "asr":
        # per note: t_restart(3), freq(0), cutoff(0) at `on`; t_release(2) at `off`
        nodes = np.stack([rep(env_a), rep(saw_a), rep(svf_a), rep(env_a)], 1).reshape(V, K, 4)
        params = np.tile(np.array([3, 0, 0, 2]), (V, K, 1))
        kinds = np.tile(np.array([TRIG, FLOAT, FLOAT, TRIG]), (V, K, 1))
        vals = np.stack([np.zeros(V * K), note_f.reshape(-1), note_fc.reshape(-1), np.zeros(V * K)], 1).reshape(V, K, 4)
        frames = np.stack([on.reshape(-1), on.reshape(-1), on.reshape(-1), off.reshape(-1)], 1).reshape(V, K, 4)
    else:
        # t_restart(2) + freq + cutoff at `on`; t_stop(3) at end of decay; jump_to_segment(1)=2 at `off`
        hold = on + ((att[:, None] + 0.05) * sr).astype(np.int64) + 1
        nodes = np.stack([rep(env_a), rep(saw_a), rep(svf_a), rep(env_a), rep(env_a)], 1).reshape(V, K, 5)
        params = np.tile(np.array([2, 0, 0, 3, 1]), (V, K, 1))
        kinds = np.tile(np.array([TRIG, FLOAT, FLOAT, TRIG, INT]), (V, K, 1))
        vals = np.stack([np.zeros(V * K), note_f.reshape(-1), note_fc.reshape(-1), np.zeros(V * K), np.full(V * K, 2.0)], 1).reshape(V, K, 5)
        frames = np.stack([on.reshape(-1), on.reshape(-1), on.reshape(-1), hold.reshape(-1), np.maximum(off, hold + 1).reshape(-1)], 1).reshape(V, K, 5)
    E = nodes.shape[2]
    nodes, params, kinds, vals, frames = (x.reshape(V, K * E) for x in (nodes, params, kinds, vals, frames))
    order = np.argsort(frames, axis=1, kind="stable")  # events pre-sorted per voice by frame
    tk = lambda x: np.take_along_axis(x, order, 1).reshape(-1)
    keep = tk(frames) < n_frames
    graph.schedule_bulk(tk(nodes)[keep], tk(params)[keep], tk(kinds)[keep], tk(vals)[keep], tk(frames)[keep].astype(np.uint64))
    return out_ids


def fm_bank(graph: Graph, n_voices: int, seed: int = 3003, voice_offset: int = 0, total_voices: int = 0) -> List[int]:
    """configs[3]: n_voices x (SinNumeric mod -> *idx + fc -> SinNumeric.ar_params() "freq") * amp."""
    total = total_voices or n_voices
    r = _rng(seed)
    fc = r.uniform(110.0, 880.0, total)
    ratio = r.choice(np.array([0.5, 1.0, 2.0, 3.0, 3.5]), total)
    fm = fc * ratio
    idx = r.uniform(0.0, 4.0, total) * fm
    sl = slice(voice_offset, voice_offset + n_voices)
    fc, fm, idx = fc[sl], fm[sl], idx[sl]
    amp = 1.0 / total
    out_ids = []
    with graph.edit() as g:
        for i in range(n_voices):
            mod = g.push(U.SinNumeric(float(fm[i])))
            car = g.push(U.SinNumeric(float(fc[i])).ar_params())
            car.link("freq", mod * float(idx[i]) + float(fc[i]))
            sig = car * amp
            sig.out([0, 0]).to_graph_out()
            out_ids.append(sig._outputs[0][0])
    return out_ids


def chain_bank(graph: Graph, n_voices: int, seconds: float, seed: int = 5005, n_notes: int = 8, voice_offset: int = 0,
               total_voices: int = 0) -> List[int]:
    """A voice shape NO hand-written recipe matches: PolyBlep(Sawtooth) -> SvfFilter(Low) -> OnePoleLpf -> * EnvAsr.wr_mul(1/N),
    note events like subtractive_bank.  What renders it is the kernel generated for its template (csrc/jit.cpp)."""
    total = total_voices or n_voices
    sr = graph.sample_rate
    n_frames = int(round(seconds * sr))
    r = _rng(seed)
    midi = r.integers(36, 85, total)
    fc = r.uniform(200.0, 8000.0, total)
    q = r.uniform(0.5, 8.0, total)
    lp = r.uniform(1000.0, 12000.0, total)
    att = r.uniform(0.002, 0.05, total)
    rel = r.uniform(0.05, 0.5, total)
    on = np.sort(r.integers(0, max(1, n_frames), (total, n_notes)), axis=1)
    note_midi = r.integers(36, 85, (total, n_notes))
    note_fc = r.uniform(200.0, 8000.0, (total, n_notes))
    off = on + (r.uniform(0.1, 0.4, (total, n_notes)) * sr).astype(np.int64)
    sl = slice(voice_offset, voice_offset + n_voices)
    midi, fc, q, lp, att, rel, on, note_midi, note_fc, off = (x[sl] for x in (midi, fc, q, lp, att, rel, on, note_midi, note_fc, off))
    f0 = 440.0 * 2.0 ** ((midi - 69) / 12.0)
    note_f = 440.0 * 2.0 ** ((note_midi - 69) / 12.0)
    saw_ids, svf_ids, env_ids, out_ids = [], [], [], []
    with graph.edit() as g:
        for i in range(n_voices):
            saw = g.push(U.PolyBlep(U.Waveform.Sawtooth, float(f0[i])).precise_timing(8))
            svf = g.push(U.SvfFilter(U.SvfFilterType.Low, float(fc[i]), float(q[i]), 0.0).precise_timing(8))
            opl = g.push(U.OnePoleLpf(float(lp[i])))
            env = g.push(U.EnvAsr(float(att[i]), float(rel[i])).wr_mul(1.0 / total).precise_timing(8))
            sig = (saw >> svf >> opl) * env
            sig.out([0, 0]).to_graph_out()
            saw_ids.append(saw.id()); svf_ids.append(svf.id()); env_ids.append(env.id()); out_ids.append(sig._outputs[0][0])
    saw_a, svf_a, env_a = (np.asarray(x, dtype=np.uint32) for x in (saw_ids, svf_ids, env_ids))
    V, K = n_voices, n_notes
    rep = lambda a: np.repeat(a, K)
    FLOAT, TRIG = 1, 2
    nodes = np.stack([rep(env_a), rep(saw_a), rep(svf_a), rep(env_a)], 1).reshape(V, K * 4)
    params = np.tile(np.array([3, 0, 0, 2]), (V, K, 1)).reshape(V, K * 4)
    kinds = np.tile(np.array([TRIG, FLOAT, FLOAT, TRIG]), (V, K, 1)).reshape(V, K * 4)
    vals = np.stack([np.zeros(V * K), note_f.reshape(-1), note_fc.reshape(-1), np.zeros(V * K)], 1).reshape(V, K * 4)
    frames = np.stack([on.reshape(-1), on.reshape(-1), on.reshape(-1), off.reshape(-1)], 1).reshape(V, K * 4)
    order = np.argsort(frames, axis=1, kind="stable")
    tk = lambda x: np.take_along_axis(x, order, 1).reshape(-1)
    keep = tk(frames) < n_frames
    graph.schedule_bulk(tk(nodes)[keep], tk(params)[keep], tk(kinds)[keep], tk(vals)[keep], tk(frames)[keep].astype(np.uint64))
    return out_ids


def _notes(graph: Graph, env_ids: List[int], on: np.ndarray, off: np.ndarray, n_frames: int) -> None:
    """EnvAsr notes: t_restart (3) at `on`, t_release (2) at `off`, any frame of a block."""
    V, K = on.shape
    env_a = np.repeat(np.asarray(env_ids, dtype=np.uint32), 2 * K).reshape(V, 2 * K)
    frames = np.concatenate([on, off], axis=1)
    params = np.concatenate([np.full((V, K), 3), np.full((V, K), 2)], axis=1)
    order = np.argsort(frames, axis=1, kind="stable")
    tk = lambda x: np.take_along_axis(x, order, 1).reshape(-1)
    keep = tk(frames) < n_frames
    n = int(keep.sum())
    graph.schedule_bulk(tk(env_a)[keep], tk(params)[keep], np.full(n, 2), np.zeros(n), tk(frames)[keep].astype(np.uint64))


def partials_bank(graph: Graph, n_voices: int, seconds: float, seed: int = 6006, n_partials: int = 32, n_notes: int = 4,
                  voice_offset: int = 0, total_voices: int = 0) -> List[int]:
    """A voice larger than 24 nodes: n_partials x SinWt(k f0).wr_mul(a_k) summed by an Add chain -> SvfFilter(Low) ->
    * EnvAsr.wr_mul(1/N), note events (t_restart / t_release) at any frame.  32 partials = 66 nodes, 142 registers."""
    total = total_voices or n_voices
    sr = graph.sample_rate
    n_frames = int(round(seconds * sr))
    r = _rng(seed)
    f0 = 55.0 * 2.0 ** r.uniform(0.0, 2.0, total)
    amp = r.uniform(0.5, 1.0, (total, n_partials)) / np.arange(1, n_partials + 1) * 0.25
    fc = r.uniform(500.0, 8000.0, total)
    q = r.uniform(0.5, 4.0, total)
    att = r.uniform(0.002, 0.05, total)
    rel = r.uniform(0.05, 0.5, total)
    on = np.sort(r.integers(0, max(1, n_frames), (total, n_notes)), axis=1)
    off = on + (r.uniform(0.1, 0.4, (total, n_notes)) * sr).astype(np.int64)
    sl = slice(voice_offset, voice_offset + n_voices)
    f0, amp, fc, q, att, rel, on, off = (x[sl] for x in (f0, amp, fc, q, att, rel, on, off))
    env_ids, out_ids = [], []
    with graph.edit() as g:
        for i in range(n_voices):
            mix = None
            for k in range(n_partials):
                p = g.push(U.SinWt(float(f0[i] * (k + 1))).wr_mul(float(amp[i, k])))
                mix = p if mix is None else mix + p
            svf = g.push(U.SvfFilter(U.SvfFilterType.Low, float(fc[i]), float(q[i]), 0.0))
            env = g.push(U.EnvAsr(float(att[i]), float(rel[i])).wr_mul(1.0 / total))
            sig = (mix >> svf) * env
            sig.out([0, 0]).to_graph_out()
            env_ids.append(env.id()); out_ids.append(sig._outputs[0][0])
    _notes(graph, env_ids, on, off, n_frames)
    return out_ids


def operator_bank(graph: Graph, n_voices: int, seconds: float, seed: int = 7007, n_ops: int = 12, n_notes: int = 4,
                  voice_offset: int = 0, total_voices: int = 0) -> List[int]:
    """A voice larger than 24 nodes made of builder arithmetic: PolyBlep(Sawtooth) -> n_ops x (x * a + b) -> SvfFilter(Low)
    -> * EnvAsr.wr_mul(1/N), note events (t_restart / t_release) at any frame.  Each `x * a + b` pushes two Constants and two
    MathUGens (graph_edit.rs:936-1225): 12 operators = 52 nodes."""
    total = total_voices or n_voices
    sr = graph.sample_rate
    n_frames = int(round(seconds * sr))
    r = _rng(seed)
    f0 = 55.0 * 2.0 ** r.uniform(0.0, 4.0, total)
    mul = r.uniform(0.9, 1.0, (total, n_ops))
    add = r.uniform(-0.01, 0.01, (total, n_ops))
    fc = r.uniform(500.0, 8000.0, total)
    q = r.uniform(0.5, 4.0, total)
    att = r.uniform(0.002, 0.05, total)
    rel = r.uniform(0.05, 0.5, total)
    on = np.sort(r.integers(0, max(1, n_frames), (total, n_notes)), axis=1)
    off = on + (r.uniform(0.1, 0.4, (total, n_notes)) * sr).astype(np.int64)
    sl = slice(voice_offset, voice_offset + n_voices)
    f0, mul, add, fc, q, att, rel, on, off = (x[sl] for x in (f0, mul, add, fc, q, att, rel, on, off))
    env_ids, out_ids = [], []
    with graph.edit() as g:
        for i in range(n_voices):
            x = g.push(U.PolyBlep(U.Waveform.Sawtooth, float(f0[i])))
            for k in range(n_ops):
                x = x * float(mul[i, k]) + float(add[i, k])
            svf = g.push(U.SvfFilter(U.SvfFilterType.Low, float(fc[i]), float(q[i]), 0.0))
            env = g.push(U.EnvAsr(float(att[i]), float(rel[i])).wr_mul(1.0 / total))
            sig = (x >> svf) * env
            sig.out([0, 0]).to_graph_out()
            env_ids.append(env.id()); out_ids.append(sig._outputs[0][0])
    _notes(graph, env_ids, on, off, n_frames)
    return out_ids


def bank_builder(workload: str, seconds: float, seed=None):
    """The bench / parity workloads of BASELINE.json by name: returns build(graph, n_voices, voice_offset,
    total_voices) -> one tap node id per voice (the voice's pre-mix signal).  voice_offset / total_voices select a
    slice of a larger bank (a GPU rank's share of configs[4], or a checker thread's shard) from the same random stream."""

    def build(graph, nv, offset, total):
        kw = {} if seed is None else {"seed": seed}
        if workload in ("subtractive", "subtractive_seg"):
            return subtractive_bank(graph, nv, seconds, voice_offset=offset, total_voices=total,
                                    envelope="asr" if workload == "subtractive" else "segments", **kw)
        if workload == "additive":
            return additive_bank(graph, nv, seconds, voice_offset=offset, total_voices=total, **kw)
        if workload == "fm":
            return fm_bank(graph, nv, voice_offset=offset, total_voices=total, **kw)
        if workload == "chain":
            return chain_bank(graph, nv, seconds, voice_offset=offset, total_voices=total, **kw)
        if workload == "partials":
            return partials_bank(graph, nv, seconds, voice_offset=offset, total_voices=total, **kw)
        if workload == "operators":
            return operator_bank(graph, nv, seconds, voice_offset=offset, total_voices=total, **kw)
        raise ValueError(f"unknown workload {workload}")

    return build
