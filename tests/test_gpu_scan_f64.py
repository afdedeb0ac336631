"""render_sub_scan against an f64 evaluation of the same filter.

The scan kernel is the one recipe that re-associates arithmetic: its SvfFilter runs as a chunked linear-recurrence scan, so it
can only be held to a tolerance.  "<= 1e-4 against the oracle" compares one f32 rounding order with another, and the oracle's
own f32 error is largest exactly where the scan is worst conditioned (low cutoff with high q: poles near 1, so A^64 and the
carried state accumulate; cutoff near Nyquist: g = tan(pi fc / sr) ~ 30).  Here the truth is the filter evaluated in f64 on the
same f32 input:

    saw, env      the oracle's PolyBlep and EnvAsr (.wr_mul) taps: the filter's input and the VCA's gain, f32 exactly as the
                  engine computes them (phases, envelopes and events are sample-exact in the scan kernel);
    coefficients  plan.cpp::svf_coeffs restated in f32 numpy, with glibc's tanf / powf through ctypes;
    svf32         svf.rs's tick in f32, in the kernel's operation order: must equal the oracle's SvfFilter tap bit for bit
                  (which proves the restatement);
    truth         svf64(saw) * env.

Per voice the kernel's error against the truth must stay within twice the sequential f32 filter's (the oracle's) plus 2^-20 of
the voice's peak: a kernel whose scan is a few times worse than plain f32 fails, where the blanket 1e-4 would not notice."""
import ctypes
import ctypes.util
import functools

import numpy as np
import pytest

import knaster_b200 as kn
from knaster_b200.graph import Graph
from knaster_b200.processor import AudioProcessor, AudioProcessorOptions
from oracle.oracle import OracleProcessor

SR = 48000
N_BLOCKS = 1500                     # 2 s at block size 64
F32 = np.float32

LOW_FC = (15.0, 40.0, 60.0, 200.0, 1000.0, 8000.0, 20000.0, 23500.0)
LOW_Q = (0.5, 2.0, 8.0, 50.0)
# the other eight types at the four corners of that grid; shelves and bells at +-12 dB
CORNERS = ((15.0, 0.5, 12.0), (15.0, 50.0, -12.0), (23500.0, 0.5, -12.0), (23500.0, 50.0, 12.0))


def voices():
    """(type, cutoff, q, gain_db) of every voice: 32 lowpasses, then 4 corners of each other type."""
    vs = [(0, fc, q, 0.0) for fc in LOW_FC for q in LOW_Q]
    for ty in range(1, 9):
        vs += [(ty, fc, q, gain if ty >= 6 else 0.0) for fc, q, gain in CORNERS]
    return vs


def build(graph, seed=4242):
    """saw -> SvfFilter (fixed coefficients) -> * EnvAsr.wr_mul(1/V) voices, 4 notes each: t_restart + a new saw frequency at the
    note-on, t_release 0.1-0.4 s later.  Returns the node ids: saw, svf, env, voice output."""
    vs = voices()
    n = len(vs)
    n_frames = N_BLOCKS * graph.block_size
    r = np.random.Generator(np.random.PCG64(seed))
    ids = {"saw": [], "svf": [], "env": [], "out": []}
    with graph.edit() as g:
        for i, (ty, fc, q, gain) in enumerate(vs):
            f0 = 55.0 * 2.0 ** (r.integers(0, 48) / 12.0)
            saw = g.push(kn.PolyBlep(kn.Waveform.Sawtooth, f0).precise_timing(8))
            svf = g.push(kn.SvfFilter(kn.SvfFilterType(ty), fc, q, gain).precise_timing(8))
            env = g.push(kn.EnvAsr(float(r.uniform(0.002, 0.05)), float(r.uniform(0.05, 0.5))).wr_mul(1.0 / n).precise_timing(8))
            sig = (saw >> svf) * env
            sig.out([0, 0]).to_graph_out()
            on = np.sort(r.integers(0, n_frames - SR // 10, 4))
            on[0] = min(on[0], int(r.integers(0, 64)))     # every voice sounds from its first chunk on
            for f in on:
                env.param("t_restart").trig_at(kn.Seconds.from_samples(int(f), SR))
                saw.param("freq").set_at(55.0 * 2.0 ** (r.integers(0, 48) / 12.0), kn.Seconds.from_samples(int(f), SR))
                off = int(f + r.uniform(0.1, 0.4) * SR)
                if off < n_frames:
                    env.param("t_release").trig_at(kn.Seconds.from_samples(off, SR))
            for k, h in (("saw", saw), ("svf", svf), ("env", env)):
                ids[k].append(h.id())
            ids["out"].append(sig._outputs[0][0])
    return ids


_libm = ctypes.CDLL(ctypes.util.find_library("m"))
for _fn in ("tanf", "sqrtf"):
    getattr(_libm, _fn).restype = ctypes.c_float
    getattr(_libm, _fn).argtypes = [ctypes.c_float]
_libm.powf.restype = ctypes.c_float
_libm.powf.argtypes = [ctypes.c_float, ctypes.c_float]


def svf_coeffs(ty, cutoff, q, gain_db, sr=SR):
    """plan.cpp::svf_coeffs (SvfFilter::set_coeffs, svf.rs:146-242) in f32: a1 a2 a3 m0 m1 m2."""
    pi, one, cutoff, q, gain_db, sr = F32(np.pi), F32(1.0), F32(cutoff), F32(q), F32(gain_db), F32(sr)
    tan = lambda x: F32(_libm.tanf(float(x)))
    amp = one                                                       # Bell, LowShelf, HighShelf only
    if ty >= 6:
        amp = F32(_libm.powf(10.0, float(gain_db / F32(40.0))))
        sq = F32(_libm.sqrtf(float(amp)))
        g = tan((pi * cutoff) / sr) / sq if ty in (6, 7) else tan((pi * cutoff) / sr) * sq
        k = one / (q * amp) if ty == 6 else one / q
    else:
        g = tan((pi * cutoff) / sr)
        k = one / q
    a1 = one / (one + g * (g + k))
    a2 = g * a1
    a3 = g * a2
    m = {0: (0.0, 0.0, 1.0), 1: (1.0, -k, -1.0), 2: (0.0, 1.0, 0.0), 3: (1.0, -k, 0.0), 4: (1.0, -k, -2.0),
         5: (1.0, F32(-2.0) * k, 0.0), 6: (1.0, k * (amp * amp - one), 0.0), 7: (1.0, k * (amp - one), amp * amp - one),
         8: (amp * amp, k * (one - amp) * amp, one - amp * amp)}[ty]
    return np.array([a1, a2, a3, *m], dtype=F32)


def svf_run(x, c, dtype):
    """svf.rs:245-280 over x [voices, frames] with coefficients c [voices, 6], every operation rounded to `dtype` in the
    kernel's (and the oracle's) order: no contraction, sums left to right."""
    x = np.ascontiguousarray(x.T, dtype=dtype)
    a1, a2, a3, m0, m1, m2 = (np.ascontiguousarray(c[:, i], dtype=dtype) for i in range(6))
    two = dtype(2.0)
    ic1 = np.zeros(x.shape[1], dtype)
    ic2 = np.zeros(x.shape[1], dtype)
    y = np.empty_like(x)
    for n in range(x.shape[0]):
        v0 = x[n]
        v3 = v0 - ic2
        v1 = a1 * ic1 + a2 * v3
        v2 = (ic2 + a2 * ic1) + a3 * v3
        ic1 = two * v1 - ic1
        ic2 = two * v2 - ic2
        y[n] = (m0 * v0 + m1 * v1) + m2 * v2
    return y.T


@functools.lru_cache(maxsize=1)
def oracle_and_truth():
    """The oracle's taps (saw, svf, env, voice) and the f64 truth of every voice."""
    g = Graph(0, 2, 64, SR)
    ids = build(g)
    orc = OracleProcessor(g, ring_buffer_size=1 << 22)
    for k in ("saw", "svf", "env", "out"):
        for i in ids[k]:
            orc.add_tap(i, 0)
    bus, taps = orc.render(N_BLOCKS)
    saw, svf, env, out = np.split(taps, 4)
    c = np.stack([svf_coeffs(*v) for v in voices()])
    svf32 = svf_run(saw, c, np.float32)
    truth = svf_run(saw, c.astype(np.float64), np.float64) * env.astype(np.float64)
    return bus, saw, svf, env, out, svf32, truth


def test_f32_restatement_is_the_oracle_filter():
    # on the CPU alone: the restated coefficients and tick must be the oracle's bit for bit, or the f64 truth below is the truth
    # of some other filter
    _, saw, svf, env, out, svf32, truth = oracle_and_truth()
    assert np.array_equal(svf32, svf)
    assert np.array_equal((svf32 * env).astype(F32), out)
    assert np.isfinite(truth).all()


@pytest.mark.gpu
def test_scan_kernel_against_f64_filter():
    ref_bus, saw, svf, env, orc, svf32, truth = oracle_and_truth()
    assert np.array_equal(svf32, svf), "the f32 restatement is not the oracle's filter"
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions())
    ids = build(graph)
    for i in ids["out"]:
        proc.add_tap(i, 0)
    assert set(proc.info()["kernels"]) == {"render_sub_scan"}      # one voice template (group) per filter type
    bus = proc.render(N_BLOCKS)
    gpu = proc.read_taps()

    peak = np.abs(truth).max(axis=1)
    gpu_err = np.abs(gpu - truth).max(axis=1)
    orc_err = np.abs(orc - truth).max(axis=1)
    par = np.abs(gpu - orc).max(axis=1) / np.abs(orc).max(axis=1)
    bound = 2.0 * orc_err + 2.0 ** -20 * peak
    names = [t.name for t in kn.SvfFilterType]
    vs = voices()
    print(f"\n{'type':>9} {'fc':>7} {'q':>5} {'gain':>5} {'peak':>9} {'oracle err':>10} {'scan err':>10} {'scan/orc':>8} "
          f"{'/ bound':>7} {'vs oracle':>9}")
    for i, (ty, fc, q, gain) in enumerate(vs):
        print(f"{names[ty]:>9} {fc:7.0f} {q:5.1f} {gain:5.0f} {peak[i]:9.3e} {orc_err[i] / peak[i]:10.3e} "
              f"{gpu_err[i] / peak[i]:10.3e} {gpu_err[i] / max(orc_err[i], 1e-30):8.3f} {gpu_err[i] / bound[i]:7.3f} {par[i]:9.3e}")
    print(f"(errors relative to the voice's peak; the peak at the voice's gain of 1/{len(vs)})")
    assert (peak > 1e-3 / len(peak)).all(), "a silent voice"
    bad = [i for i in range(len(peak)) if not gpu_err[i] <= bound[i]]
    assert not bad, "scan error above 2 x the f32 filter's + 2^-20 peak: " + ", ".join(
        f"{names[vs[i][0]]} fc {vs[i][1]:g} q {vs[i][2]:g} ({gpu_err[i] / bound[i]:.2f}x)" for i in bad)
    assert par.max() <= 1e-4, f"voice {int(np.argmax(par))}: {par.max():.3e} against the oracle"
    assert np.abs(bus - ref_bus).max() <= 1e-5
