// plan.cpp -- graph -> kernel plan compiler and control-rate simulation (host, C++).
//
// What knaster does on its control thread at Graph::commit_changes (graph.rs:1707-1726:
// node order, buffer plan, TaskData) and on its audio thread at the top of every block
// (graph_gen.rs:111-166,269-305: drain the event ring, apply parameter changes through the
// wrapper stack) is done here, ahead of time, for a static graph:
//
//  * build():    find the mix-bus Add chains (graph.rs:850-864), split the rest into
//                independent voices, batch isomorphic voices into groups (SoA registers),
//                lay out registers and value slots (the analogue of buffer_allocator.rs),
//                run every node's init() (graph.rs:462-475) to get the initial registers.
//  * simulate(): replay the parameter-change queue through an exact model of the wrapper
//                stack (WrPreciseTiming / WrSmoothParams / WrArParams / WrMul..) and of every
//                UGen's setters; all f64 / libm work (tanf, expf, f64 ramps) happens here with
//                the same libm knaster uses, and the device only sees
//                "write register r at frame f" events plus three state-dependent triggers.
//
// Compiled with -ffp-contract=off: f32 expressions below must round exactly like rustc's.
#include "plan.hpp"
#include "fastapprox.h"

#include <algorithm>
#include <atomic>
#include <memory>
#include <cmath>
#include <cstdarg>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <new>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#if defined(__linux__)
#include <sys/mman.h>
#endif
#include <thread>
#include <tuple>
#include <unordered_map>

namespace kgpu {

std::string format(const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    return buf;
}

namespace {

constexpr float F_PI = 3.14159265358979323846264338327950288f;

inline uint32_t sat_u32(double v) { // Rust `as u32`
    if (!(v == v) || v <= 0.0) return 0;
    if (v >= 4294967295.0) return 4294967295u;
    return (uint32_t)v;
}
inline uint64_t sat_usize(double v) {
    if (!(v == v) || v <= 0.0) return 0;
    if (v >= 18446744073709551615.0) return UINT64_MAX;
    return (uint64_t)v;
}
inline uint32_t fbits(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
}
inline void dbits(double d, uint32_t &lo, uint32_t &hi) {
    uint64_t u;
    std::memcpy(&u, &d, 8);
    lo = (uint32_t)u;
    hi = (uint32_t)(u >> 32);
}

// fastrand 2.3.0 (wyrand), restated for RandomLin's constructor draws (noise.rs:173-185): see csrc/nodes.cuh wy_next
inline float wy_f32(uint64_t &state) {
    state += 0x2d358dccaa6c78a5ull;
    const unsigned __int128 t = (unsigned __int128)state * (unsigned __int128)(state ^ 0x8bb84b93962eacc9ull);
    const uint32_t u = (uint32_t)((uint64_t)t ^ (uint64_t)(t >> 64));
    uint32_t bits = 0x3F800000u + (u >> 9);
    float f;
    std::memcpy(&f, &bits, 4);
    return f - 1.0f;
}

// ---- static facts about node kinds ------------------------------------------------------
struct KindInfo {
    int n_in, n_out, n_params, dev_kind, n_regs;
};
KindInfo kind_info(const kgpu_node_desc &d) {
    switch (d.kind) {
    case KGPU_SIN_WT: return {0, 1, 3, DK_SINWT, REGS_SINWT};
    case KGPU_SIN_NUMERIC: return {0, 1, 3, DK_SINNUM, REGS_SINNUM};
    case KGPU_POLYBLEP: return {0, 1, 3, DK_POLYBLEP, REGS_POLYBLEP};
    case KGPU_SVF: return {1, 1, 5, DK_SVF, REGS_SVF};
    case KGPU_ONEPOLE_LPF: return {1, 1, 1, DK_ONEPOLE_LP, REGS_ONEPOLE};
    case KGPU_ONEPOLE_HPF: return {1, 1, 1, DK_ONEPOLE_HP, REGS_ONEPOLE};
    case KGPU_ENV_ASR: return {0, 1, 4, DK_ENVASR, REGS_ENV};
    case KGPU_ENV_AR: return {0, 1, 3, DK_ENVAR, REGS_ENV};
    case KGPU_ENVELOPE: return {0, 1, 4, DK_ENVELOPE, (int)(REGS_ENVELOPE_BASE + REGS_ENVELOPE_PER_SEG * d.n_segments)};
    case KGPU_MATH: return {(int)(2 * d.channels), (int)d.channels, 0, DK_MATH, 0};
    case KGPU_CONSTANT: return {0, 1, 1, DK_CONST, REGS_CONST};
    case KGPU_TEST_NUM: return {0, 1, 0, DK_CONST, REGS_CONST};
    case KGPU_TEST_IN_PLUS_PARAM: return {1, 1, 1, DK_INPLUS, REGS_CONST};
    case KGPU_MATH1: return {1, 1, 0, DK_MATH1, 0};
    case KGPU_PHASOR: return {0, 1, 1, DK_PHASOR, REGS_PHASOR};
    case KGPU_WHITE_NOISE: return {0, 1, 0, DK_WHITE, REGS_WHITE};
    case KGPU_PINK_NOISE: return {0, 1, 0, DK_PINK, REGS_PINK};
    case KGPU_BROWN_NOISE: return {0, 1, 0, DK_BROWN, REGS_BROWN};
    case KGPU_RANDOM_LIN: return {0, 1, 1, DK_RANDLIN, REGS_RANDLIN};
    case KGPU_PAN2: return {1, 2, 1, DK_PAN2, REGS_PAN2};
    default: KGPU_THROW(KGPU_ERR_UNSUPPORTED, "unknown ugen kind %u", d.kind);
    }
}
// expected ParameterValue kind per base parameter ('t' = trigger: any value fires)
const char *param_types(uint32_t kind) {
    switch (kind) {
    case KGPU_SIN_WT: case KGPU_SIN_NUMERIC: return "fft";
    case KGPU_POLYBLEP: return "ffi";
    case KGPU_SVF: return "fffit";
    case KGPU_ONEPOLE_LPF: case KGPU_ONEPOLE_HPF: return "f";
    case KGPU_ENV_ASR: return "fftt";
    case KGPU_ENV_AR: return "fft";
    case KGPU_ENVELOPE: return "fitt";
    case KGPU_CONSTANT: case KGPU_TEST_IN_PLUS_PARAM: case KGPU_PHASOR: case KGPU_RANDOM_LIN: case KGPU_PAN2: return "f";
    default: return "";
    }
}
bool is_math_wrapper(uint32_t k) { return k >= KGPU_WR_MUL && k <= KGPU_WR_POWI; }

void validate_node(const kgpu_node_desc &d, uint32_t idx) {
    kind_info(d); // rejects an unknown kind
    if (d.kind == KGPU_MATH) {
        if (d.channels < 1 || d.channels > (uint32_t)MAX_OUT)
            KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %u: MathUGen with %u channels (1..%d supported)", idx, d.channels, MAX_OUT);
        if (d.mode > KGPU_OP_POW) KGPU_THROW(KGPU_ERR_INVALID, "node %u: bad MathUGen operation %u", idx, d.mode);
    }
    if (d.kind == KGPU_MATH1 && d.mode > KGPU_OP1_EXP) KGPU_THROW(KGPU_ERR_INVALID, "node %u: bad Math1UGen operation %u", idx, d.mode);
    if (d.kind == KGPU_POLYBLEP && d.mode > 13) KGPU_THROW(KGPU_ERR_INVALID, "node %u: bad PolyBlep Waveform %u", idx, d.mode);
    if (d.kind == KGPU_SVF && d.mode > 8) KGPU_THROW(KGPU_ERR_INVALID, "node %u: bad SvfFilterType %u", idx, d.mode);
    if (d.kind == KGPU_ENVELOPE) {
        if (d.n_segments < 1 || !d.segments) KGPU_THROW(KGPU_ERR_INVALID, "node %u: Envelope needs >= 1 segment", idx);
        if (d.n_segments > (uint32_t)(MAX_REGS - REGS_ENVELOPE_BASE) / REGS_ENVELOPE_PER_SEG)
            KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %u: Envelope with %u segments is too large (at most %d: %d registers per voice)", idx,
                       d.n_segments, (MAX_REGS - REGS_ENVELOPE_BASE) / REGS_ENVELOPE_PER_SEG, MAX_REGS);
    }
    if (d.n_wrappers && !d.wrappers) KGPU_THROW(KGPU_ERR_INVALID, "node %u: wrappers pointer is NULL", idx);
    int n_post = 0, n_ar = 0, n_smooth = 0, n_precise = 0;
    for (uint32_t i = 0; i < d.n_wrappers; i++) {
        uint32_t k = d.wrappers[i].kind;
        if (is_math_wrapper(k)) n_post++;
        else if (k == KGPU_WR_AR_PARAMS) {
            n_ar++;
            if (n_smooth || n_precise)
                KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %u: WrArParams outside WrSmoothParams/WrPreciseTiming is not supported "
                           "(knaster's WrPreciseTiming must be outermost, precise_timing.rs:13)", idx);
        } else if (k == KGPU_WR_SMOOTH_PARAMS) n_smooth++;
        else if (k == KGPU_WR_PRECISE_TIMING) {
            n_precise++;
            if (d.wrappers[i].capacity == 0 || d.wrappers[i].capacity > 4096) KGPU_THROW(KGPU_ERR_INVALID, "node %u: bad WrPreciseTiming capacity", idx);
        } else KGPU_THROW(KGPU_ERR_INVALID, "node %u: unknown wrapper kind %u", idx, k);
    }
    if (n_post > MAX_POST) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %u: more than %d arithmetic wrappers", idx, MAX_POST);
    if (n_ar > 1 || n_smooth > 1 || n_precise > 1) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %u: duplicate wrapper of one kind", idx);
}

uint32_t total_params(const kgpu_node_desc &d) {
    uint32_t n = (uint32_t)kind_info(d).n_params;
    for (uint32_t i = 0; i < d.n_wrappers; i++)
        if (d.wrappers[i].kind == KGPU_WR_MUL) n++;
    return n;
}

// SvfFilter::set_coeffs, svf.rs:146-242.  out: a1 a2 a3 m0 m1 m2
void svf_coeffs(uint32_t ty, float cutoff, float q, float gain_db, float sr, float *c) {
    float g, k, amp;
    switch (ty) {
    case 6: // Bell
        amp = powf(10.0f, gain_db / 40.0f);
        g = tanf((F_PI * cutoff) / sr) / sqrtf(amp);
        k = 1.0f / (q * amp);
        c[0] = 1.0f / (1.0f + g * (g + k)); c[1] = g * c[0]; c[2] = g * c[1];
        c[3] = 1.0f; c[4] = k * (amp * amp - 1.0f); c[5] = 0.0f;
        return;
    case 7: // LowShelf
        amp = powf(10.0f, gain_db / 40.0f);
        g = tanf((F_PI * cutoff) / sr) / sqrtf(amp);
        k = 1.0f / q;
        c[0] = 1.0f / (1.0f + g * (g + k)); c[1] = g * c[0]; c[2] = g * c[1];
        c[3] = 1.0f; c[4] = k * (amp - 1.0f); c[5] = amp * amp - 1.0f;
        return;
    case 8: // HighShelf
        amp = powf(10.0f, gain_db / 40.0f);
        g = tanf((F_PI * cutoff) / sr) * sqrtf(amp);
        k = 1.0f / q;
        c[0] = 1.0f / (1.0f + g * (g + k)); c[1] = g * c[0]; c[2] = g * c[1];
        c[3] = amp * amp; c[4] = k * (1.0f - amp) * amp; c[5] = 1.0f - amp * amp;
        return;
    default: break;
    }
    g = tanf((F_PI * cutoff) / sr);
    k = 1.0f / q;
    c[0] = 1.0f / (1.0f + g * (g + k));
    c[1] = g * c[0];
    c[2] = g * c[1];
    switch (ty) {
    case 0: c[3] = 0.f; c[4] = 0.f; c[5] = 1.f; break;        // Low
    case 1: c[3] = 1.f; c[4] = -k; c[5] = -1.f; break;        // High
    case 2: c[3] = 0.f; c[4] = 1.f; c[5] = 0.f; break;        // Band
    case 3: c[3] = 1.f; c[4] = -k; c[5] = 0.f; break;         // Notch
    case 4: c[3] = 1.f; c[4] = -k; c[5] = -2.0f; break;       // Peak
    default: c[3] = 1.f; c[4] = -2.0f * k; c[5] = 0.f; break; // All
    }
}

// ---- control simulation ------------------------------------------------------------------
// per-thread sink of the control simulation: the device events of the block being simulated, in emission order
// (node-major; inside a node by frame, then arrival), frames relative to the launch window's first frame
struct Sink {
    std::vector<DevEvent> *dst = nullptr; // the launch's event list of the worker's slice: events are written in place, field by field
    uint64_t t0 = 0;
    uint64_t dropped = 0, ignored = 0, devev = 0;
};
struct Sim {
    HostPlan &P;
    Sink &out;
    uint32_t local;
    HostNode &hn;
    void emit(uint64_t frame, uint16_t op, uint32_t reg, uint32_t value) {
        // (built in place: a DevEvent assembled in a local and copied as 16 bytes reads narrow stores back with one wide load,
        // which the store buffer cannot forward -- that copy was the hottest line of the whole simulation)
        DevEvent &d = out.dst->emplace_back();
        d.frame = (uint32_t)(frame - out.t0);
        d.node = (uint16_t)local;
        d.op = op;
        d.reg = reg;
        d.value = value;
    }
    void set_f(uint64_t frame, uint32_t reg, float v) { emit(frame, OP_SET, reg, fbits(v)); }
    void set_u(uint64_t frame, uint32_t reg, uint32_t v) { emit(frame, OP_SET, reg, v); }
    void set_d(uint64_t frame, uint32_t reg, double v) {
        uint32_t lo, hi;
        dbits(v, lo, hi);
        emit(frame, OP_SET, reg, lo);
        emit(frame, OP_SET, reg + 1, hi);
    }
};

// the UGen's own param_apply: every #[param] setter of the supported UGens
void ugen_param_apply(Sim &s, uint32_t param, const PV &v, uint64_t frame) {
    HostNode &h = s.hn;
    const float sr = (float)s.P.sample_rate;
    const uint32_t r = h.reg;
    switch (h.kind) {
    case KGPU_SIN_WT: // osc.rs:126-140
        if (param == 0) {
            h.f0 = (float)v.f;
            double k = 16384.0 * 65536.0 * (1.0 / (double)s.P.sample_rate);
            s.set_u(frame, r + 2, sat_u32((double)h.f0 * k));
        } else if (param == 1) s.set_u(frame, r + 1, sat_u32(v.f * 65536.0));
        else if (param == 2) s.set_u(frame, r + 0, 0);
        break;
    case KGPU_SIN_NUMERIC: // osc.rs:239-252
        if (param == 0) s.set_f(frame, r + 2, (float)v.f / sr);
        else if (param == 1) s.set_f(frame, r + 1, (float)v.f);
        else if (param == 2) s.set_f(frame, r + 0, 0.0f);
        break;
    case KGPU_PHASOR: // osc.rs:191-197
        if (param == 0) s.set_d(frame, r + 2, v.f * h.d0);
        break;
    case KGPU_PAN2: // pan.rs:26-29: self.pan = pan * 0.5 + 0.5 (f32), gains re-evaluated per sample from it
        if (param == 0) {
            float gl, gr;
            pan2_gains((float)v.f * 0.5f + 0.5f, gl, gr);
            s.set_f(frame, r + 0, gl);
            s.set_f(frame, r + 1, gr);
        }
        break;
    case KGPU_RANDOM_LIN: // noise.rs:206-213 (after init(): phase_step = F::new(value) * freq_to_phase_inc)
        if (param == 0) s.set_f(frame, r + 5, (float)v.f * h.f0);
        break;
    case KGPU_POLYBLEP: // polyblep.rs:162-184
        if (param == 0) {
            h.f0 = (float)v.f;
            float dt = h.f0 / sr;
            s.set_f(frame, r + 1, dt);
            s.set_u(frame, r + 2, (dt * sr >= sr / 4.0f) ? 1u : 0u); // guard of next_sample, polyblep.rs:210
        } else if (param == 1) s.set_f(frame, r + 3, (float)v.f);
        else if (param == 2) s.set_u(frame, r + 4, (uint32_t)(int64_t)v.f); // polyblep.rs:172-175
        break;
    case KGPU_SVF: { // svf.rs:81-133
        if (param == 0) h.f0 = (float)v.f;
        else if (param == 1) h.f1 = (float)v.f;
        else if (param == 2) h.f2 = (float)v.f;
        else if (param == 3) h.mode = (uint32_t)(int64_t)v.f;
        else if (param != 4) break;
        if (h.ar_regs && param < 4) { // the device recomputes the coefficients from these every frame (audio-rate route)
            if (param == 3) s.set_u(frame, r + 11, h.mode);
            else s.set_f(frame, r + 8 + param, param == 0 ? h.f0 : (param == 1 ? h.f1 : h.f2));
        }
        float c[6];
        svf_coeffs(h.mode, h.f0, h.f1, h.f2, sr, c);
        for (int i = 0; i < 6; i++)
            if (fbits(c[i]) != fbits(h.svf_coef[i])) {
                h.svf_coef[i] = c[i];
                s.set_f(frame, r + 2 + i, c[i]);
            }
        break;
    }
    case KGPU_ONEPOLE_LPF: case KGPU_ONEPOLE_HPF: // onepole.rs:135-139,172-176,35-46
        if (param == 0) {
            float f = (float)v.f / sr;
            float b1 = expf(-2.0f * F_PI * f);
            s.set_f(frame, r + 2, b1);
            s.set_f(frame, r + 1, 1.0f - b1);
        }
        break;
    case KGPU_ENV_ASR: case KGPU_ENV_AR: // envelopes.rs:84-133,234-266
        if (param == 0) {
            float atk = (float)v.f;
            if (h.f0 != atk) {
                h.f0 = atk;
                s.set_f(frame, r + 2, atk == 0.f ? 1.0f : 1.0f / (atk * sr));
            }
        } else if (param == 1) {
            float rel = (float)v.f;
            if (h.f1 != rel) {
                h.f1 = rel;
                s.set_f(frame, r + 3, rel == 0.f ? 1.0f : 1.0f / (rel * sr));
            }
        } else if (h.kind == KGPU_ENV_ASR && param == 2) s.emit(frame, OP_ASR_RELEASE, r, 0);
        else if ((h.kind == KGPU_ENV_ASR && param == 3) || (h.kind == KGPU_ENV_AR && param == 2))
            s.set_u(frame, r + 0, ASR_ATTACKING);
        break;
    case KGPU_ENVELOPE: // envelopes.rs:476-526; one compound device event per trigger (dev.h OP_ENV_*)
        if (param == 0) {
            double ts = (double)(float)v.f;
            uint32_t lo, hi;
            dbits(ts * (1.0 / (double)s.P.sample_rate), lo, hi);
            s.emit(frame, OP_ENV_STEP, lo, hi);
        } else if (param == 1) {
            uint64_t j = sat_usize(v.f);
            if (j >= h.n_seg) j = h.n_seg - 1;
            s.emit(frame, OP_ENV_JUMP, r, (uint32_t)j);
        } else if (param == 2) {
            uint32_t lo, hi;
            dbits(h.d0, lo, hi);
            s.emit(frame, OP_ENV_RESTART, lo, hi);
        } else if (param == 3) s.emit(frame, OP_ENV_STOP, r, 0);
        break;
    case KGPU_CONSTANT: case KGPU_TEST_IN_PLUS_PARAM: // util.rs:45-48
        if (param == 0) s.set_f(frame, r + 0, (float)v.f);
        break;
    default: break;
    }
}

void wr_param_apply(Sim &s, int level, uint32_t param, const PV &v, uint64_t frame);

// ParameterSmoothingState::next_value, BlockRate branch (smooth_params.rs:263-300)
bool smooth_next_value(SmoothState &st, uint64_t block_size, double *out) {
    if (!st.linear || st.done) return false;
    double mix = (double)st.frames_elapsed / (double)st.duration_frames;
    double cur = (st.end_value - st.start_value) * mix + st.start_value;
    if (st.frames_elapsed == st.duration_frames) st.done = true;
    else st.frames_elapsed = std::min<uint64_t>(st.frames_elapsed + block_size, st.duration_frames);
    *out = cur;
    return true;
}

void wr_param_apply(Sim &s, int level, uint32_t param, const PV &v, uint64_t frame) {
    if (level < 0) {
        if (v.kind == PV::Smoothing) return; // rejected at push time (would panic in knaster)
        ugen_param_apply(s, param, v, frame);
        return;
    }
    WrapSim &w = s.hn.wr[level];
    switch (w.kind) {
    case KGPU_WR_MUL:
        if (param == w.inner_params) { // wrappers_core/math.rs:92-98
            if (v.kind == PV::Float) s.set_f(frame, w.reg, (float)v.f);
            return;
        }
        wr_param_apply(s, level - 1, param, v, frame);
        return;
    case KGPU_WR_ADD: case KGPU_WR_SUB: case KGPU_WR_VSUB: case KGPU_WR_DIV: case KGPU_WR_VDIV:
    case KGPU_WR_POWF: case KGPU_WR_POWI:
        wr_param_apply(s, level - 1, param, v, frame);
        return;
    case KGPU_WR_AR_PARAMS: // audio_rate.rs:70-74
        if (param < w.ar_bound.size() && w.ar_bound[param]) return;
        wr_param_apply(s, level - 1, param, v, frame);
        return;
    case KGPU_WR_SMOOTH_PARAMS: { // smooth_params.rs:200-244
        if (param >= w.smooth.size()) return;
        SmoothState &st = w.smooth[param];
        if (v.kind == PV::Integer || v.kind == PV::Trigger || v.kind == PV::Bool) {
            wr_param_apply(s, level - 1, param, v, frame);
        } else if (v.kind == PV::Float) {
            if (!st.linear) wr_param_apply(s, level - 1, param, v, frame);
            else {
                if (st.done) st.start_value = st.end_value;
                else {
                    double mix = (double)st.frames_elapsed / (double)st.duration_frames;
                    st.start_value = (st.end_value - st.start_value) * mix + st.start_value;
                }
                st.end_value = v.f;
                st.done = false;
                st.frames_elapsed = 0;
            }
        } else if (v.kind == PV::Smoothing) { // set_smoothing, smooth_params.rs:31-102
            if (v.smoothing == 0) {
                if (st.linear) {
                    double mix = (double)st.frames_elapsed / (double)st.duration_frames;
                    double cur = (st.end_value - st.start_value) * mix + st.start_value;
                    st = SmoothState{};
                    st.current_value = cur;
                }
            } else {
                uint64_t dur = sat_usize((double)v.smooth_seconds * (double)s.P.sample_rate);
                if (!st.linear) {
                    double cur = st.current_value;
                    st.linear = true;
                    st.start_value = cur; st.end_value = cur;
                    st.duration_frames = dur; st.frames_elapsed = 0; st.done = true;
                } else if (st.done) {
                    st.start_value = st.end_value;
                    st.duration_frames = dur; st.frames_elapsed = 0; st.done = true;
                } else {
                    double mix = (double)st.frames_elapsed / (double)st.duration_frames;
                    st.start_value = (st.end_value - st.start_value) * mix + st.start_value;
                    st.duration_frames = dur; st.done = true;
                }
            }
        }
        return;
    }
    case KGPU_WR_PRECISE_TIMING: // precise_timing.rs:126-135
        if (param >= w.next_delay.size()) return; // would index out of bounds in knaster
        if (w.next_delay[param] == 0) wr_param_apply(s, level - 1, param, v, frame);
        else if (w.queue.size() < w.capacity) w.queue.push_back(QueuedChange{w.next_delay[param], param, v});
        else s.out.dropped++;
        return;
    default: return;
    }
}

// set_delay_within_block_for_param through the wrapper stack
void wr_set_delay(Sim &s, int level, uint32_t param, uint16_t delay) {
    for (; level >= 0; level--) {
        WrapSim &w = s.hn.wr[level];
        if (w.kind == KGPU_WR_PRECISE_TIMING) { // precise_timing.rs:146-148
            if (param < w.next_delay.size()) w.next_delay[param] = delay;
            return;
        }
        if (!is_math_wrapper(w.kind)) break; // WrSmoothParams / WrArParams do not forward (trait default)
    }
    s.out.ignored++; // ugen.rs:339-341: warning, no effect
}

// control-side effects of process_block through the wrapper stack for one (partial) block
void wr_process_block(Sim &s, int level, uint64_t block_start, uint32_t offset, uint32_t frames) {
    for (; level >= 0; level--) {
        WrapSim &w = s.hn.wr[level];
        if (w.kind == KGPU_WR_SMOOTH_PARAMS) { // smooth_params.rs:179-188
            for (uint32_t j = 0; j < w.smooth.size(); j++) {
                double v;
                if (smooth_next_value(w.smooth[j], s.P.block_size, &v)) {
                    PV pv;
                    pv.kind = PV::Float;
                    pv.f = v;
                    wr_param_apply(s, level - 1, j, pv, block_start + offset);
                }
            }
        } else if (w.kind == KGPU_WR_PRECISE_TIMING) { // precise_timing.rs:65-114
            uint32_t block_i = 0;
            size_t change_i = 0;
            const size_t num = w.queue.size();
            // next_delay_i = 0 at the end; next_delay[] stays.  Small fixed scratch: the queue holds
            // at most `capacity` entries and nested WrPreciseTiming is rejected at plan time.
            QueuedChange qbuf[16];
            std::vector<QueuedChange> qheap;
            QueuedChange *q = qbuf;
            if (num > 16) {
                qheap = w.queue;
                q = qheap.data();
            } else std::copy(w.queue.begin(), w.queue.end(), qbuf);
            w.queue.clear();
            uint8_t some_buf[16];
            std::vector<uint8_t> some_heap;
            uint8_t *some = some_buf;
            if (num > 16) {
                some_heap.assign(num, 1);
                some = some_heap.data();
            } else std::fill(some_buf, some_buf + 16, (uint8_t)1);
            while (true) {
                uint32_t local_frames = frames - block_i;
                while (change_i < num) {
                    if (some[change_i]) {
                        if ((uint32_t)q[change_i].delay <= block_i + offset) {
                            wr_param_apply(s, level - 1, q[change_i].param, q[change_i].value, block_start + offset + block_i);
                            some[change_i] = 0;
                        } else {
                            local_frames = std::min(local_frames, (uint32_t)q[change_i].delay - offset - block_i);
                            break;
                        }
                    }
                    change_i++;
                }
                if (block_i >= frames) break;
                wr_process_block(s, level - 1, block_start, offset + block_i, local_frames);
                block_i += local_frames;
            }
            return;
        } else if (w.kind == KGPU_WR_AR_PARAMS) {
            return; // per-frame inner.process(); nothing control-rate inside (validated)
        }
    }
}

bool needs_processing(const HostNode &h) {
    if (h.precise_level >= 0 && !h.wr[h.precise_level].queue.empty()) return true;
    if (h.smooth_level >= 0)
        for (const SmoothState &st : h.wr[h.smooth_level].smooth)
            if (st.linear && !st.done) return true;
    return false;
}

uint64_t hash_mix(uint64_t h, uint64_t v) {
    h ^= v + 0x9e3779b97f4a7c15ULL + (h << 6) + (h >> 2);
    return h;
}

} // namespace

bool TemplateNode::same_shape(const TemplateNode &o) const {
    if (kind != o.kind || mode != o.mode || channels != o.channels || flags != o.flags || n_segments != o.n_segments) return false;
    if (wrappers.size() != o.wrappers.size() || in != o.in || par != o.par) return false;
    for (size_t i = 0; i < wrappers.size(); i++)
        if (wrappers[i].kind != o.wrappers[i].kind || wrappers[i].capacity != o.wrappers[i].capacity) return false;
    return true;
}
bool Template::same_shape(const Template &o) const {
    if (nodes.size() != o.nodes.size() || outs != o.outs || level != o.level) return false;
    for (size_t i = 0; i < nodes.size(); i++)
        if (!nodes[i].same_shape(o.nodes[i])) return false;
    return true;
}

namespace {

uint64_t template_hash(const Template &t) {
    uint64_t h = 1469598103934665603ULL;
    for (const TemplateNode &n : t.nodes) {
        h = hash_mix(h, n.kind | ((uint64_t)n.mode << 8) | ((uint64_t)n.channels << 16) | ((uint64_t)n.flags << 24) | ((uint64_t)n.n_segments << 32));
        for (auto &w : n.wrappers) h = hash_mix(h, w.kind | ((uint64_t)w.capacity << 8));
        for (auto &e : n.in) h = hash_mix(h, (uint64_t)(uint32_t)e.first | ((uint64_t)e.second << 32));
        for (auto &p : n.par) h = hash_mix(h, std::get<0>(p) | ((uint64_t)(uint32_t)std::get<1>(p) << 16) | ((uint64_t)std::get<2>(p) << 40));
    }
    for (auto &o : t.outs) h = hash_mix(h, (uint64_t)(uint32_t)std::get<0>(o) | ((uint64_t)std::get<1>(o) << 20) | ((uint64_t)std::get<2>(o) << 40));
    return hash_mix(h, (uint64_t)t.level);
}

// resolve an audio-rate parameter route of a node to a device action
uint8_t ar_code_for(const TemplateNode &tn, uint32_t param, int ar_level) {
    // walk inward from the WrArParams wrapper
    int post_index = 0;
    for (int l = 0; l < ar_level; l++)
        if (is_math_wrapper(tn.wrappers[l].kind)) post_index++;
    uint32_t inner = 0; // parameters of the stack below the AR wrapper
    {
        kgpu_node_desc tmp{};
        tmp.kind = tn.kind;
        tmp.channels = tn.channels;
        tmp.n_segments = tn.n_segments;
        inner = (uint32_t)kind_info(tmp).n_params;
    }
    // parameters contributed by WrMul wrappers below the AR level, innermost first
    uint32_t pcount = inner;
    int pi = 0;
    for (int l = 0; l < ar_level; l++) {
        uint32_t k = tn.wrappers[l].kind;
        if (is_math_wrapper(k)) {
            if (k == KGPU_WR_MUL) {
                if (param == pcount) return (uint8_t)(AR_POST + pi);
                pcount++;
            }
            pi++;
        }
    }
    (void)post_index;
    if (param >= inner) KGPU_THROW(KGPU_ERR_PARAMETER, "audio-rate route to parameter %u: index out of bounds", param);
    switch (tn.kind) {
    case KGPU_SIN_NUMERIC: if (param == 0) return AR_SINNUM_FREQ; if (param == 1) return AR_SINNUM_OFFSET; break;
    case KGPU_SIN_WT: if (param == 0) return AR_SINWT_FREQ; if (param == 1) return AR_SINWT_OFFSET; break;
    case KGPU_POLYBLEP:
        if (param == 0) return AR_POLYBLEP_FREQ;
        if (param == 1) return AR_POLYBLEP_PW;
        break;
    case KGPU_CONSTANT: case KGPU_TEST_IN_PLUS_PARAM: if (param == 0) return AR_REG0; break;
    case KGPU_SVF:
        if (param == 0) return AR_SVF_CUTOFF;
        if (param == 1) return AR_SVF_Q;
        if (param == 2) return AR_SVF_GAIN;
        break;
    case KGPU_ONEPOLE_LPF: case KGPU_ONEPOLE_HPF: if (param == 0) return AR_ONEPOLE_CUTOFF; break;
    case KGPU_ENV_ASR: case KGPU_ENV_AR:
        if (param == 0) return AR_ENV_ATTACK;
        if (param == 1) return AR_ENV_RELEASE;
        break; // the triggers are not floats: WrArParams would hand them a Float (a type error in knaster too)
    case KGPU_PAN2: if (param == 0) return AR_PAN2_PAN; break;
    case KGPU_PHASOR: if (param == 0) return AR_PHASOR_FREQ; break;
    case KGPU_RANDOM_LIN: if (param == 0) return AR_RANDLIN_FREQ; break;
    case KGPU_ENVELOPE: if (param == 0) return AR_ENVELOPE_TIME_SCALE; break; // jump_to_segment is an integer, the rest triggers
    default: break;
    }
    KGPU_THROW(KGPU_ERR_UNSUPPORTED, "audio-rate route to parameter %u of ugen kind %u is not supported yet", param, tn.kind);
}

// lay out registers + value slots of a template and fill its DevProgram
void compile_template(Group &g, uint32_t sample_rate, const std::vector<std::pair<uint32_t, uint32_t>> &pinned) {
    const Template &t = g.tpl;
    DevProgram &p = g.prog;
    std::memset(&p, 0, sizeof p);
    const size_t n = t.nodes.size();
    if (n > (size_t)MAX_NODES)
        KGPU_THROW(KGPU_ERR_UNSUPPORTED, "a voice with %zu nodes exceeds the per-voice limit of %d (sources shared between voices "
                   "merge them into one voice; not supported yet)", n, MAX_NODES);
    p.n_nodes = (uint32_t)n;
    p.sample_rate = (float)sample_rate;
    p.sinwt_k = 16384.0 * 65536.0 * (1.0 / (double)sample_rate);
    // registers
    uint32_t reg = 0;
    std::vector<std::vector<uint16_t>> post_regs(n);
    for (size_t i = 0; i < n; i++) {
        const TemplateNode &tn = t.nodes[i];
        kgpu_node_desc tmp{};
        tmp.kind = tn.kind; tmp.channels = tn.channels; tmp.n_segments = tn.n_segments;
        KindInfo ki = kind_info(tmp);
        DevNode &dn = p.nodes[i];
        dn.kind = (uint8_t)ki.dev_kind;
        dn.mode = (uint8_t)tn.mode;
        dn.n_in = (uint8_t)ki.n_in;
        dn.n_out = (uint8_t)ki.n_out;
        dn.reg = (uint16_t)reg;
        dn.n_seg = (uint16_t)tn.n_segments;
        dn.looping = (uint8_t)(tn.flags & 1);
        reg += (uint32_t)ki.n_regs;
        // an SvfFilter whose cutoff / q / gain is driven at audio rate keeps those parameters (and its type) in registers
        // too: the device recomputes the coefficients every frame
        {
            bool has_ar = false;
            for (auto &w : tn.wrappers) has_ar |= w.kind == KGPU_WR_AR_PARAMS;
            bool svf_route = false;
            for (auto &pe : tn.par) svf_route |= std::get<0>(pe) <= 2;
            if (tn.kind == KGPU_SVF && has_ar && svf_route) reg += REGS_SVF_AR - REGS_SVF;
        }
        int ar_level = -1;
        for (size_t l = 0; l < tn.wrappers.size(); l++) {
            uint32_t k = tn.wrappers[l].kind;
            if (is_math_wrapper(k)) {
                dn.post_op[dn.n_post] = (uint8_t)k; // PO_* == KGPU_WR_* for 1..8
                dn.post_reg[dn.n_post] = (uint16_t)reg;
                post_regs[i].push_back((uint16_t)reg);
                dn.n_post++;
                reg++;
            } else if (k == KGPU_WR_AR_PARAMS) ar_level = (int)l;
        }
        for (auto &pe : tn.par) {
            if (ar_level < 0) continue; // no WrArParams: set_ar_param_buffer has no effect (ugen.rs:322-329)
            if (dn.n_ar >= MAX_AR) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "more than %d audio-rate routes into one node", MAX_AR);
            dn.ar_code[dn.n_ar] = ar_code_for(tn, std::get<0>(pe), ar_level);
            dn.ar_slot[dn.n_ar] = -1; // filled below
            dn.n_ar++;
        }
    }
    // ports: one register each after every node's, holding the voice's input channel
    uint32_t n_ports = 0;
    for (const TemplateNode &tn : t.nodes) {
        for (auto &e : tn.in)
            if (is_port_src(e.first)) n_ports = std::max(n_ports, (uint32_t)(e.first - PORT_SRC0) + 1);
        for (auto &pe : tn.par)
            if (is_port_src(std::get<1>(pe))) n_ports = std::max(n_ports, (uint32_t)(std::get<1>(pe) - PORT_SRC0) + 1);
    }
    if (n_ports > (uint32_t)MAX_PORTS)
        KGPU_THROW(KGPU_ERR_UNSUPPORTED, "a voice reads %u graph inputs that no other voice reads (limit %d per voice)", n_ports, MAX_PORTS);
    p.n_ports = (uint16_t)n_ports;
    p.port_reg = (uint16_t)(n_ports ? std::min<uint32_t>(reg, 0xFFFF) : 0u);
    reg += n_ports;
    if (reg > (uint32_t)MAX_REGS) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "voice needs %u registers (limit %d)", reg, MAX_REGS);
    p.n_regs = reg;
    // value slots: liveness-based reuse, the analogue of allocate_node_buffers (graph.rs:1588-1704)
    std::vector<std::vector<int>> last_use(n);
    for (size_t i = 0; i < n; i++) last_use[i].assign(p.nodes[i].n_out, -1);
    const int INF = 1 << 30;
    for (size_t i = 0; i < n; i++) {
        for (auto &e : t.nodes[i].in)
            if (e.first >= 0) last_use[e.first][e.second] = std::max(last_use[e.first][e.second], (int)i);
        for (auto &pe : t.nodes[i].par)
            if (std::get<1>(pe) >= 0) last_use[std::get<1>(pe)][std::get<2>(pe)] = std::max(last_use[std::get<1>(pe)][std::get<2>(pe)], (int)i);
    }
    for (auto &o : t.outs) last_use[std::get<0>(o)][std::get<1>(o)] = INF;
    for (auto &pin : pinned) last_use[pin.first][pin.second] = INF;
    std::vector<uint16_t> free_slots;
    uint32_t n_slots = 0;
    g.slot_of.assign(n, {});
    for (size_t i = 0; i < n; i++) {
        DevNode &dn = p.nodes[i];
        const TemplateNode &tn = t.nodes[i];
        // inputs (+ release the ones that die here: in-place reuse is safe, every node reads a frame before writing it)
        std::vector<std::pair<int, uint32_t>> dying;
        for (int c = 0; c < MAX_IN; c++) dn.in_slot[c] = -1;
        for (size_t c = 0; c < tn.in.size(); c++) {
            auto &e = tn.in[c];
            if (e.first <= EXT_BASE) // an internal signal, read from its buffer, or a port
                dn.in_slot[c] = (int16_t)(is_port_src(e.first) ? SLOT_PORT0 + (e.first - PORT_SRC0) : e.first);
            if (e.first < 0) continue;
            dn.in_slot[c] = (int16_t)g.slot_of[e.first][e.second];
            if (last_use[e.first][e.second] == (int)i) dying.push_back(e);
        }
        int ai = 0;
        bool has_ar = false;
        for (auto &w : tn.wrappers) has_ar |= (w.kind == KGPU_WR_AR_PARAMS);
        for (auto &pe : tn.par) {
            int src = std::get<1>(pe);
            uint32_t ch = std::get<2>(pe);
            if (src <= EXT_BASE) { // routed from an internal signal or a port
                if (has_ar) dn.ar_slot[ai++] = (int16_t)(is_port_src(src) ? SLOT_PORT0 + (src - PORT_SRC0) : src);
                continue;
            }
            if (has_ar) dn.ar_slot[ai++] = (int16_t)g.slot_of[src][ch];
            if (last_use[src][ch] == (int)i) dying.push_back({src, ch});
        }
        std::sort(dying.begin(), dying.end());
        dying.erase(std::unique(dying.begin(), dying.end()), dying.end());
        for (auto &d : dying) free_slots.push_back(g.slot_of[d.first][d.second]);
        g.slot_of[i].resize(dn.n_out);
        for (int c = 0; c < dn.n_out; c++) {
            uint16_t s;
            if (!free_slots.empty()) {
                s = free_slots.back();
                free_slots.pop_back();
            } else s = (uint16_t)n_slots++;
            g.slot_of[i][c] = s;
            dn.out_slot[c] = s;
        }
        for (int c = 0; c < dn.n_out; c++)
            if (last_use[i][c] < 0) free_slots.push_back(g.slot_of[i][c]); // dead output
    }
    if (n_slots > (uint32_t)MAX_SLOTS) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "voice needs %u live value slots (limit %d)", n_slots, MAX_SLOTS);
    p.n_slots = std::max(1u, n_slots);
    // mix-bus outputs: one partial-sum row per distinct (node, channel), with the set of graph outputs it feeds
    p.n_ubus = 0;
    for (auto &o : t.outs) {
        uint16_t slot = g.slot_of[std::get<0>(o)][std::get<1>(o)];
        uint32_t u = 0;
        for (; u < p.n_ubus; u++)
            if (p.ubus_slot[u] == slot) break;
        if (u == p.n_ubus) {
            if (p.n_ubus >= (uint32_t)MAX_BUS) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "voice feeds more than %d distinct bus signals", MAX_BUS);
            p.ubus_slot[u] = slot;
            p.ubus_mask[u] = 0;
            p.n_ubus++;
        }
        p.ubus_mask[u] |= 1u << std::get<2>(o);
    }
}

} // namespace

void recompile_group_slots(Group &g, uint32_t sample_rate, const std::vector<std::pair<uint32_t, uint32_t>> &pinned) {
    compile_template(g, sample_rate, pinned);
}

void HostPlan::build(const kgpu_graph_desc &d) {
    if (d.abi_version != KGPU_ABI_VERSION) KGPU_THROW(KGPU_ERR_INVALID, "abi_version %u != %u", d.abi_version, KGPU_ABI_VERSION);
    if (d.sample_rate == 0 || d.block_size == 0) KGPU_THROW(KGPU_ERR_INVALID, "sample_rate and block_size must be non-zero"); // processor.rs:75
    if (d.block_size > 65535) KGPU_THROW(KGPU_ERR_INVALID, "block_size must fit the u16 in-block delay (graph_gen.rs:292)");
    if (d.n_outputs < 1 || d.n_outputs > (uint32_t)MAX_BUS) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "n_outputs must be 1..%d", MAX_BUS);
    if (d.n_inputs > MAX_GRAPH_INPUTS) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "%u graph inputs: at most %u", d.n_inputs, MAX_GRAPH_INPUTS);
    n_inputs = d.n_inputs;
    input_to_output.clear();
    shared_inputs.clear();
    has_ports = false;
    if ((d.n_nodes && !d.nodes) || (d.n_edges && !d.edges) || (d.n_param_edges && !d.param_edges))
        KGPU_THROW(KGPU_ERR_INVALID, "NULL array in graph description");
    sample_rate = d.sample_rate;
    block_size = d.block_size;
    bs_pow2 = (block_size & (block_size - 1)) == 0;
    bs_shift = bs_pow2 ? (uint32_t)__builtin_ctz(block_size) : 0;
    n_outputs = d.n_outputs;
    const uint32_t N = d.n_nodes;
    for (uint32_t i = 0; i < N; i++) validate_node(d.nodes[i], i);
    {
        auto hd = [](double x) { uint64_t u; std::memcpy(&u, &x, 8); return u; };
        uint64_t h = hash_mix(0x6b67707573ull, ((uint64_t)d.sample_rate << 32) | d.block_size);
        h = hash_mix(h, ((uint64_t)d.n_outputs << 32) | d.n_nodes);
        for (uint32_t i = 0; i < N; i++) {
            const kgpu_node_desc &n = d.nodes[i];
            h = hash_mix(h, n.kind | ((uint64_t)n.mode << 8) | ((uint64_t)n.channels << 24) | ((uint64_t)n.flags << 32) | ((uint64_t)n.n_wrappers << 40) | ((uint64_t)n.n_segments << 48));
            for (double a : n.args) h = hash_mix(h, hd(a));
            for (uint32_t w = 0; w < n.n_wrappers; w++) h = hash_mix(hash_mix(h, n.wrappers[w].kind | ((uint64_t)n.wrappers[w].capacity << 8)), hd(n.wrappers[w].value));
            if (n.kind == KGPU_ENVELOPE)
                for (uint32_t k = 0; k < 2 * n.n_segments; k++) h = hash_mix(h, hd(n.segments[k]));
        }
        for (uint32_t e = 0; e < d.n_edges; e++)
            h = hash_mix(h, (uint64_t)(uint32_t)d.edges[e].source_node | ((uint64_t)d.edges[e].source_channel << 32)), h = hash_mix(h, (uint64_t)(uint32_t)d.edges[e].sink_node | ((uint64_t)d.edges[e].sink_channel << 32));
        for (uint32_t e = 0; e < d.n_param_edges; e++)
            h = hash_mix(h, (uint64_t)(uint32_t)d.param_edges[e].source_node | ((uint64_t)d.param_edges[e].source_channel << 32)), h = hash_mix(h, (uint64_t)(uint32_t)d.param_edges[e].sink_node | ((uint64_t)d.param_edges[e].param_index << 32));
        graph_hash = h;
    }

    // adjacency
    std::vector<uint32_t> in_off(N + 1, 0);
    for (uint32_t i = 0; i < N; i++) in_off[i + 1] = in_off[i] + (uint32_t)kind_info(d.nodes[i]).n_in;
    std::vector<std::pair<int, uint32_t>> in_edges(in_off[N], {-1, 0u});
    std::vector<std::pair<int, uint32_t>> out_edges(n_outputs, {-1, 0u});
    std::vector<uint32_t> fanout(N, 0);
    auto check_src = [&](int32_t src, uint32_t ch, const char *what) {
        if (src == KGPU_GRAPH) { // NodeOrGraph::Graph as a source: a graph input
            if (ch >= d.n_inputs) KGPU_THROW(KGPU_ERR_INVALID, "%s: GraphInputOutOfBounds(%u)", what, ch);
            return;
        }
        if (src < 0 || (uint32_t)src >= N) KGPU_THROW(KGPU_ERR_INVALID, "%s: source node %d not found", what, src);
        if (ch >= (uint32_t)kind_info(d.nodes[src]).n_out) KGPU_THROW(KGPU_ERR_INVALID, "%s: OutputOutOfBounds(%u)", what, ch);
    };
    for (uint32_t e = 0; e < d.n_edges; e++) {
        const kgpu_edge &ed = d.edges[e];
        check_src(ed.source_node, ed.source_channel, "edge");
        if (ed.sink_node == KGPU_GRAPH) {
            if (ed.sink_channel >= n_outputs) KGPU_THROW(KGPU_ERR_INVALID, "edge: GraphOutputOutOfBounds(%u)", ed.sink_channel);
            out_edges[ed.sink_channel] = {ed.source_node, ed.source_channel};
        } else {
            if (ed.sink_node < 0 || (uint32_t)ed.sink_node >= N) KGPU_THROW(KGPU_ERR_INVALID, "edge: sink node %d not found", ed.sink_node);
            if (ed.sink_channel >= in_off[ed.sink_node + 1] - in_off[ed.sink_node]) KGPU_THROW(KGPU_ERR_INVALID, "edge: InputOutOfBounds(%u)", ed.sink_channel);
            in_edges[in_off[ed.sink_node] + ed.sink_channel] = {ed.source_node, ed.source_channel};
        }
    }
    std::vector<std::vector<std::tuple<uint32_t, int, uint32_t>>> par_edges(N);
    for (uint32_t e = 0; e < d.n_param_edges; e++) {
        const kgpu_param_edge &pe = d.param_edges[e];
        check_src(pe.source_node, pe.source_channel, "param edge");
        if (pe.sink_node < 0 || (uint32_t)pe.sink_node >= N) KGPU_THROW(KGPU_ERR_INVALID, "param edge: sink node %d not found", pe.sink_node);
        if (pe.param_index >= total_params(d.nodes[pe.sink_node])) KGPU_THROW(KGPU_ERR_PARAMETER, "param edge: ParameterIndexOutOfBounds");
        par_edges[pe.sink_node].push_back({pe.param_index, pe.source_node, pe.source_channel});
    }
    for (auto &e : in_edges)
        if (e.first >= 0) fanout[e.first]++;
    for (auto &e : out_edges)
        if (e.first >= 0) fanout[e.first]++;
    for (auto &pl : par_edges)
        for (auto &pe : pl)
            if (std::get<1>(pe) >= 0) fanout[std::get<1>(pe)]++;

    // ---- mix buses, internal signals, voices ---------------------------------------------------------------------------
    // A graph output is the left fold ((v0+v1)+v2)+... of an Add chain (graph.rs:850-864): its leaves are voice outputs and
    // the chain becomes the mix-bus reduction.  The same happens INSIDE the graph when a node reads the sum of many voices
    // (post-mix processing) or when one source feeds many voices: such a source is an internal signal, reduced into its own
    // buffer one level before the voices that read it, and what reads it is cut loose from what produces it -- otherwise
    // the whole bank would be one connected "voice".  Thresholds: a sum of >= mix_min leaves, a node with >= shared_min
    // consumers.  16 keeps every graph that fitted a small voice (SMALL_VOICE_NODES) exactly as it was; if a component still
    // outgrows one the discovery is repeated with 2 (every fan-in / fan-out point is a cut).  Only where neither gives small
    // voices within the signal budget is a third one tried that cuts a sum only when it has more leaves than one voice can
    // hold (a master bus over a bank): a voice of up to MAX_NODES nodes then keeps its own partial sums (additive partials).
    // If that fails too, the first discovery stands, with voices of up to MAX_NODES nodes (a master bus over large voices).
    auto sum_like = [&](int node) {
        if (node < 0) return false;
        const kgpu_node_desc &nd = d.nodes[node];
        if (nd.kind != KGPU_MATH || nd.mode != KGPU_OP_ADD || nd.channels != 1 || nd.n_wrappers != 0) return false;
        return in_edges[in_off[node]].first >= 0 && in_edges[in_off[node] + 1].first >= 0;
    };
    auto is_mix = [&](int node) { return sum_like(node) && fanout[node] == 1; };
    struct Leaf { int node; uint32_t ch; uint32_t target; };
    struct Discovery {
        std::vector<Leaf> leaves;
        std::vector<char> mix_node;
        std::vector<int> in_ext;                               // per input edge: internal signal or -1
        std::vector<std::vector<int>> par_ext;                 // per parameter edge likewise
        std::vector<int> comp;
        std::vector<int> uf;
        uint32_t n_signals = 0, n_mix = 0;
    };
    auto discover = [&](uint32_t mix_min, uint32_t shared_min, Discovery &D) {
        D = Discovery{};
        D.mix_node.assign(N, 0);
        D.in_ext.assign(in_off[N], -1);
        D.par_ext.resize(N);
        for (uint32_t i = 0; i < N; i++) D.par_ext[i].assign(par_edges[i].size(), -1);
        D.comp.assign(N, -1);
        D.n_signals = n_inputs; // the graph's inputs come first
        // expands the Add chain rooted at `root` (the root itself may have any fan-out, inner Adds exactly one consumer)
        auto expand = [&](std::pair<int, uint32_t> root, uint32_t target, bool root_any_fanout, bool commit, std::vector<Leaf> &out) {
            std::vector<std::pair<int, uint32_t>> stack{root};
            bool first = true;
            while (!stack.empty()) {
                auto cur = stack.back();
                stack.pop_back();
                const bool through = first && root_any_fanout ? sum_like(cur.first) : is_mix(cur.first);
                first = false;
                if (through) {
                    if (commit && !D.mix_node[cur.first]) {
                        D.mix_node[cur.first] = 1;
                        D.n_mix++;
                    }
                    stack.push_back(in_edges[in_off[cur.first] + 1]); // right operand after ...
                    stack.push_back(in_edges[in_off[cur.first]]);     // ... the left one (in-order)
                } else out.push_back({cur.first, cur.second, target});
            }
        };
        for (uint32_t oc = 0; oc < n_outputs; oc++) {
            if (out_edges[oc].first == KGPU_SOURCE_NONE) continue;
            // a large sum that feeds this output AND something else (the dry mix beside a master effect): its leaves go to the
            // output directly, whatever else reads the sum gets it as an internal signal made of the same leaves
            std::vector<Leaf> probe;
            const bool shared_root = sum_like(out_edges[oc].first) && fanout[out_edges[oc].first] > 1;
            if (shared_root) expand(out_edges[oc], oc, true, false, probe);
            expand(out_edges[oc], oc, shared_root && probe.size() >= mix_min, true, D.leaves);
        }
        std::unordered_map<uint64_t, int> sig_of; // (node, channel) -> signal
        // what (src, ch) is to a consumer: the node itself (-1) or an internal signal
        auto resolve = [&](int src, uint32_t ch) -> int {
            const uint64_t key = ((uint64_t)(uint32_t)src << 8) | ch;
            auto it = sig_of.find(key);
            if (it != sig_of.end()) return it->second;
            std::vector<Leaf> lv;
            bool cut = false;
            if (sum_like(src)) {
                expand({src, ch}, 0, true, false, lv);
                cut = lv.size() >= mix_min;
            }
            if (!cut && fanout[src] >= shared_min) {
                lv.assign(1, Leaf{src, ch, 0});
                cut = true;
            }
            if (!cut) return sig_of[key] = -1;
            if (sum_like(src) && lv.size() > 1) {
                lv.clear();
                expand({src, ch}, 0, true, true, lv); // now for real: the chain's Adds disappear into the reduction
            }
            const int sidx = (int)D.n_signals++;
            for (Leaf &l : lv) {
                l.target = n_outputs + (uint32_t)sidx;
                D.leaves.push_back(l);
            }
            return sig_of[key] = sidx;
        };
        auto find = [&](int x) {
            while (D.uf[x] != x) x = D.uf[x] = D.uf[D.uf[x]];
            return x;
        };
        std::vector<int> stack;
        for (size_t li = 0; li < D.leaves.size(); li++) { // grows while signals are found
            const Leaf lf = D.leaves[li];
            if (lf.node == KGPU_GRAPH) continue; // a graph input summed straight into an output: no voice behind it
            if (D.mix_node[lf.node]) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %d is both summed into a mix and read on its own", lf.node);
            if (D.comp[lf.node] >= 0) continue;
            const int c = (int)D.uf.size();
            D.uf.push_back(c);
            D.comp[lf.node] = c;
            stack.assign(1, lf.node);
            while (!stack.empty()) {
                const int nk = stack.back();
                stack.pop_back();
                auto visit = [&](int src, uint32_t ch, int &ext) {
                    if (src == KGPU_GRAPH) {
                        ext = (int)ch; // graph input ch = signal ch
                        return;
                    }
                    if (src < 0) return;
                    ext = resolve(src, ch);
                    if (ext >= 0) return; // read through the signal's buffer: no edge between the two voices
                    if (D.mix_node[src]) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "node %d reads a node that is summed into a mix", nk);
                    if (D.comp[src] < 0) {
                        D.comp[src] = c;
                        stack.push_back(src);
                    } else {
                        const int a = find(D.comp[src]), b = find(c);
                        if (a != b) D.uf[std::max(a, b)] = std::min(a, b);
                    }
                };
                for (uint32_t k = in_off[nk]; k < in_off[nk + 1]; k++) visit(in_edges[k].first, in_edges[k].second, D.in_ext[k]);
                for (size_t k = 0; k < par_edges[nk].size(); k++) visit(std::get<1>(par_edges[nk][k]), std::get<2>(par_edges[nk][k]), D.par_ext[nk][k]);
            }
        }
        // the largest component, in nodes
        std::unordered_map<int, uint32_t> size;
        uint32_t largest = 0;
        for (uint32_t i = 0; i < N; i++)
            if (D.comp[i] >= 0) largest = std::max(largest, ++size[find(D.comp[i])]);
        return largest;
    };
    // Graph inputs after a discovery: owner[i] = the component of the one voice that reads input i (a port of its template), -1
    // for a shared input (read by several voices, summed into a mix, wired to an output), -2 for one nothing reads.  Returns the
    // number of shared inputs: only they take signal rows.
    auto classify_inputs = [&](const Discovery &D, std::vector<int> &owner) -> uint32_t {
        owner.assign(n_inputs, -2);
        auto root = [&](int x) {
            while (D.uf[x] != x) x = D.uf[x];
            return x;
        };
        auto read = [&](uint32_t in, uint32_t nk) {
            const int c = root(D.comp[nk]);
            owner[in] = owner[in] == -2 || owner[in] == c ? c : -1;
        };
        for (uint32_t nk = 0; nk < N; nk++) {
            if (D.comp[nk] < 0) continue;
            for (uint32_t k = in_off[nk]; k < in_off[nk + 1]; k++)
                if (in_edges[k].first == KGPU_GRAPH) read(in_edges[k].second, nk);
            for (auto &pe : par_edges[nk])
                if (std::get<1>(pe) == KGPU_GRAPH) read(std::get<2>(pe), nk);
        }
        for (const Leaf &lf : D.leaves)
            if (lf.node == KGPU_GRAPH) owner[lf.ch] = -1;
        uint32_t n_shared = 0;
        for (int o : owner) n_shared += o == -1;
        return n_shared;
    };
    // outputs + shared inputs + internal signals within the 32 rows of the partial-sum masks
    auto signals_fit = [&](const Discovery &D) {
        std::vector<int> owner;
        return n_outputs + classify_inputs(D, owner) + (D.n_signals - n_inputs) <= 32;
    };
    Discovery D;
    const bool small = discover(16, 16, D) <= (uint32_t)SMALL_VOICE_NODES;
    bool ok = small && signals_fit(D);
    if (!small) {
        Discovery D2;
        try {
            ok = discover(2, 2, D2) <= (uint32_t)SMALL_VOICE_NODES && signals_fit(D2);
        } catch (const Error &) {
        }
        if (ok) D = std::move(D2);
    }
    if (!ok) {
        Discovery D3;
        bool ok3 = false;
        try {
            ok3 = discover(MAX_NODES + 1, 16, D3) <= (uint32_t)MAX_NODES && signals_fit(D3);
        } catch (const Error &) {
        }
        if (ok3) D = std::move(D3);
        // otherwise D stays the first discovery: its voices may now have up to MAX_NODES nodes (compile_template checks).  That is
        // how a master bus over fewer than MAX_NODES + 1 large voices plans -- the third discovery keeps such a sum whole and
        // glues the bank into one component, the first cuts it at 16 leaves
    }
    // shared inputs become signal rows 0 .. n_shared - 1, the internal signals follow; a port edge is marked -2 - input
    std::vector<int> owner;
    const uint32_t n_shared = classify_inputs(D, owner);
    if (n_shared > (uint32_t)MAX_SHARED_INPUTS)
        KGPU_THROW(KGPU_ERR_UNSUPPORTED, "%u graph inputs are shared (read by more than one voice, summed into a mix or wired to an output): at most %d",
                   n_shared, MAX_SHARED_INPUTS);
    {
        std::vector<int> remap(D.n_signals);
        for (uint32_t i = 0; i < n_inputs; i++) {
            if (owner[i] >= 0) {
                remap[i] = -2 - (int)i;
                has_ports = true;
            } else if (owner[i] == -1) {
                remap[i] = (int)shared_inputs.size();
                shared_inputs.push_back(i);
            }
        }
        for (uint32_t sg = n_inputs; sg < D.n_signals; sg++) remap[sg] = (int)(n_shared + sg - n_inputs);
        for (int &e : D.in_ext)
            if (e >= 0) e = remap[e];
        for (auto &pl : D.par_ext)
            for (int &e : pl)
                if (e >= 0) e = remap[e];
        for (Leaf &lf : D.leaves)
            if (lf.target >= n_outputs) lf.target = n_outputs + (uint32_t)remap[lf.target - n_outputs];
        D.n_signals = n_shared + (D.n_signals - n_inputs);
    }
    if (n_outputs + D.n_signals > 32)
        KGPU_THROW(KGPU_ERR_UNSUPPORTED, "%u internal signals (sums of voices read by nodes, sources shared between voices, shared graph inputs): at most %u",
                   D.n_signals, 32 - n_outputs);
    n_mix_nodes = D.n_mix;
    std::vector<Leaf> &leaves = D.leaves;
    std::vector<int> &comp = D.comp;
    auto find = [&](int x) {
        while (D.uf[x] != x) x = D.uf[x] = D.uf[D.uf[x]];
        return x;
    };
    // per component: leaves in order
    std::unordered_map<int, std::vector<Leaf>> comp_leaves;
    std::vector<int> comp_order;
    for (auto &lf : leaves) {
        if (lf.node == KGPU_GRAPH) {
            if (lf.target >= n_outputs) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "a graph input summed into an internal mix is not supported");
            const uint32_t row = (uint32_t)(std::lower_bound(shared_inputs.begin(), shared_inputs.end(), lf.ch) - shared_inputs.begin());
            input_to_output.push_back({row, lf.target});
            continue;
        }
        int c = find(comp[lf.node]);
        auto it = comp_leaves.find(c);
        if (it == comp_leaves.end()) {
            comp_order.push_back(c);
            comp_leaves[c] = {lf};
        } else it->second.push_back(lf);
    }
    // levels: a voice renders after every signal it reads, a signal is complete after its last contributor
    std::unordered_map<int, int> comp_level;
    signal_level.assign(D.n_signals, -1);
    {
        std::unordered_map<int, std::vector<int>> reads;    // component -> signals read
        for (uint32_t nk = 0; nk < N; nk++) {
            if (comp[nk] < 0) continue;
            const int c = find(comp[nk]);
            for (uint32_t k = in_off[nk]; k < in_off[nk + 1]; k++)
                if (D.in_ext[k] >= 0) reads[c].push_back(D.in_ext[k]);
            for (int e : D.par_ext[nk])
                if (e >= 0) reads[c].push_back(e);
        }
        std::vector<std::vector<int>> feeders(D.n_signals);  // signal -> contributing components
        for (auto &lf : leaves)
            if (lf.target >= n_outputs && lf.node >= 0) feeders[lf.target - n_outputs].push_back(find(comp[lf.node]));
        std::unordered_map<int, int> state; // 1 visiting, 2 done
        std::function<int(int)> level_of = [&](int c) -> int {
            if (state[c] == 2) return comp_level[c];
            if (state[c] == 1) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "a voice reads a signal it contributes to: feedback is not supported");
            state[c] = 1;
            int lv = 0;
            for (int sg : reads[c]) {
                if ((uint32_t)sg < n_shared) continue; // a graph input: there before the first launch
                int sl = 0;
                for (int f : feeders[sg]) sl = std::max(sl, level_of(f));
                signal_level[sg] = std::max(signal_level[sg], sl);
                lv = std::max(lv, sl + 1);
            }
            state[c] = 2;
            return comp_level[c] = lv;
        };
        max_level = 0;
        for (int c : comp_order) max_level = std::max(max_level, level_of(c));
        for (uint32_t sg = n_shared; sg < D.n_signals; sg++)
            if (signal_level[sg] < 0) { // a signal nobody reads cannot exist; keep it well-defined anyway
                int sl = 0;
                for (int f : feeders[sg]) sl = std::max(sl, comp_level[f]);
                signal_level[sg] = sl;
            }
    }
    node_ref.assign(N, NodeRef{});
    for (uint32_t i = 0; i < N; i++) node_ref[i].n_params = (uint16_t)total_params(d.nodes[i]);
    std::unordered_map<uint64_t, std::vector<uint32_t>> by_hash;
    std::vector<int> local_of(N, -1);
    groups.clear();
    std::vector<std::pair<int, size_t>> dstack;
    for (int c : comp_order) {
        // local topological order: post-order DFS from the leaves, inputs in channel order then parameter edges
        std::vector<uint32_t> order;
        for (auto &lf : comp_leaves[c]) {
            if (local_of[lf.node] >= 0) continue;
            local_of[lf.node] = -2; // on stack / visited marker
            dstack.assign(1, {lf.node, 0});
            while (!dstack.empty()) {
                int nk = dstack.back().first;
                size_t &cur = dstack.back().second;
                const size_t ne = in_off[nk + 1] - in_off[nk], np = par_edges[nk].size();
                bool pushed = false;
                while (cur < ne + np) {
                    int src = cur < ne ? in_edges[in_off[nk] + cur].first : std::get<1>(par_edges[nk][cur - ne]);
                    const int ext = cur < ne ? D.in_ext[in_off[nk] + cur] : D.par_ext[nk][cur - ne];
                    cur++;
                    if (ext >= 0) continue; // an internal signal: not a node of this voice
                    if (src >= 0 && local_of[src] == -1) {
                        local_of[src] = -2;
                        dstack.push_back({src, 0});
                        pushed = true;
                        break;
                    } else if (src >= 0 && local_of[src] == -2) {
                        // visited-but-unfinished on the current DFS path means a cycle
                        for (auto &st : dstack)
                            if (st.first == src) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "cycle through node %d: feedback edges are not supported", src);
                    }
                }
                if (!pushed) {
                    local_of[nk] = (int)order.size();
                    order.push_back((uint32_t)nk);
                    dstack.pop_back();
                }
            }
        }
        Template t;
        t.level = comp_level[c];
        t.nodes.resize(order.size());
        std::vector<uint32_t> ports; // the graph input of each port, in the order the template first reads them
        auto port_src = [&](int ext) {
            const uint32_t in = (uint32_t)(-2 - ext);
            size_t k = std::find(ports.begin(), ports.end(), in) - ports.begin();
            if (k == ports.size()) ports.push_back(in);
            return PORT_SRC0 + (int)k;
        };
        for (size_t li = 0; li < order.size(); li++) {
            uint32_t nk = order[li];
            const kgpu_node_desc &nd = d.nodes[nk];
            TemplateNode &tn = t.nodes[li];
            tn.kind = nd.kind; tn.mode = nd.mode; tn.channels = nd.kind == KGPU_MATH ? nd.channels : 1; tn.flags = nd.flags;
            tn.n_segments = nd.kind == KGPU_ENVELOPE ? nd.n_segments : 0;
            tn.wrappers.assign(nd.wrappers, nd.wrappers + nd.n_wrappers);
            for (uint32_t k = in_off[nk]; k < in_off[nk + 1]; k++) {
                if (D.in_ext[k] >= 0) tn.in.push_back({EXT_BASE - D.in_ext[k], 0u});
                else if (D.in_ext[k] <= -2) tn.in.push_back({port_src(D.in_ext[k]), 0u});
                else tn.in.push_back({in_edges[k].first >= 0 ? local_of[in_edges[k].first] : -1, in_edges[k].second});
            }
            for (size_t k = 0; k < par_edges[nk].size(); k++) {
                auto &pe = par_edges[nk][k];
                if (D.par_ext[nk][k] >= 0) tn.par.push_back({std::get<0>(pe), EXT_BASE - D.par_ext[nk][k], 0u});
                else if (D.par_ext[nk][k] <= -2) tn.par.push_back({std::get<0>(pe), port_src(D.par_ext[nk][k]), 0u});
                else tn.par.push_back({std::get<0>(pe), local_of[std::get<1>(pe)], std::get<2>(pe)});
            }
        }
        for (auto &lf : comp_leaves[c]) t.outs.push_back({local_of[lf.node], lf.ch, lf.target});
        uint64_t h = template_hash(t);
        int gi = -1;
        for (uint32_t cand : by_hash[h])
            if (groups[cand].tpl.same_shape(t)) { gi = (int)cand; break; }
        if (gi < 0) {
            gi = (int)groups.size();
            groups.emplace_back();
            groups.back().tpl = std::move(t);
            compile_template(groups.back(), sample_rate, {});
            by_hash[h].push_back((uint32_t)gi);
        }
        Group &g = groups[gi];
        uint32_t voice = g.n_voices++;
        g.voice_nodes.push_back(order);
        g.port_input.insert(g.port_input.end(), ports.begin(), ports.end());
        for (size_t li = 0; li < order.size(); li++) {
            node_ref[order[li]].group = gi;
            node_ref[order[li]].voice = voice;
            node_ref[order[li]].local = (uint16_t)li;
        }
    }
    // groups in level order (a level's groups launch together, then its signals are reduced): stable, with node_ref remapped
    if (max_level > 0) {
        std::vector<uint32_t> perm(groups.size());
        for (uint32_t i = 0; i < perm.size(); i++) perm[i] = i;
        std::stable_sort(perm.begin(), perm.end(), [&](uint32_t a, uint32_t b) { return groups[a].tpl.level < groups[b].tpl.level; });
        std::vector<int> new_of(groups.size());
        std::vector<Group> sorted;
        sorted.reserve(groups.size());
        for (uint32_t i = 0; i < perm.size(); i++) {
            new_of[perm[i]] = (int)i;
            sorted.push_back(std::move(groups[perm[i]]));
        }
        groups = std::move(sorted);
        for (NodeRef &nr : node_ref)
            if (nr.group >= 0) nr.group = new_of[nr.group];
    }
    // initial registers + control state: Node::init (graph.rs:462-475) of every node of every voice
    const float sr = (float)sample_rate;
    for (Group &g : groups) {
        const uint32_t V = g.n_voices, nn = (uint32_t)g.tpl.nodes.size();
        g.init_regs.assign((size_t)g.prog.n_regs * V, 0u);
        g.host.assign((size_t)V * nn, HostNode{});
        // the template's wrapper stacks, once per group
        g.nstat.assign(nn, NodeStatic{});
        for (uint32_t li = 0; li < nn; li++) {
            const TemplateNode &tn = g.tpl.nodes[li];
            const DevNode &dn = g.prog.nodes[li];
            NodeStatic &ns = g.nstat[li];
            kgpu_node_desc tmp{};
            tmp.kind = tn.kind; tmp.channels = tn.channels; tmp.n_segments = tn.n_segments;
            ns.kind = (uint8_t)tn.kind;
            ns.base_params = (uint32_t)kind_info(tmp).n_params;
            uint32_t inner = ns.base_params;
            int post_i = 0;
            bool only_math_above = true; // walking inwards from the top is done below; here: innermost first
            ns.n_levels = (uint8_t)std::min<size_t>(tn.wrappers.size(), MAX_WRAP_LEVELS);
            for (size_t l = 0; l < tn.wrappers.size(); l++) {
                const uint32_t k = tn.wrappers[l].kind;
                if (l < (size_t)MAX_WRAP_LEVELS) {
                    ns.lv_kind[l] = (uint8_t)k;
                    ns.lv_inner[l] = inner;
                }
                if (is_math_wrapper(k)) {
                    if (l < (size_t)MAX_WRAP_LEVELS) ns.lv_reg[l] = dn.post_reg[post_i];
                    post_i++;
                    if (k == KGPU_WR_MUL) inner++;
                } else if (k == KGPU_WR_SMOOTH_PARAMS) ns.smooth_level = (int8_t)l;
                else if (k == KGPU_WR_PRECISE_TIMING) {
                    ns.precise_level = (int8_t)l;
                    ns.capacity = tn.wrappers[l].capacity;
                    ns.nd_size = inner;
                } else if (k == KGPU_WR_AR_PARAMS && l < (size_t)MAX_WRAP_LEVELS) {
                    for (auto &pe : tn.par)
                        if (std::get<0>(pe) < inner && std::get<0>(pe) < 32) ns.lv_ar_mask[l] |= 1u << std::get<0>(pe);
                }
            }
            ns.total_params = inner;
            (void)only_math_above;
            // set_delay walks inwards from the outermost wrapper: math wrappers forward, the first WrPreciseTiming takes it,
            // WrSmoothParams / WrArParams swallow it (trait default, ugen.rs:339-341)
            ns.delay_reaches = false;
            for (int l = (int)tn.wrappers.size() - 1; l >= 0; l--) {
                const uint32_t k = tn.wrappers[l].kind;
                if (k == KGPU_WR_PRECISE_TIMING) { ns.delay_reaches = true; break; }
                if (!is_math_wrapper(k)) break;
            }
            ns.fast = ns.smooth_level < 0 && tn.wrappers.size() <= (size_t)MAX_WRAP_LEVELS && ns.total_params <= 8 && ns.capacity <= 32;
            if (getenv("KGPU_HOST_GENERIC")) ns.fast = false; // tests: the block-by-block model for every node
        }
        auto R = [&](uint32_t reg, uint32_t v) -> uint32_t & { return g.init_regs[(size_t)reg * V + v]; };
        for (uint32_t v = 0; v < V; v++)
            for (uint32_t k = 0; k < g.prog.n_ports; k++) R(g.prog.port_reg + k, v) = g.port_input[(size_t)v * g.prog.n_ports + k];
        for (uint32_t v = 0; v < V; v++)
            for (uint32_t li = 0; li < nn; li++) {
                const kgpu_node_desc &nd = d.nodes[g.voice_nodes[v][li]];
                const DevNode &dn = g.prog.nodes[li];
                HostNode &h = g.host[(size_t)v * nn + li];
                h.kind = (uint8_t)nd.kind;
                h.dev_kind = dn.kind;
                h.mode = nd.mode;
                h.reg = dn.reg;
                h.n_seg = dn.n_seg;
                h.base_params = (uint32_t)kind_info(nd).n_params;
                const uint32_t r = dn.reg;
                switch (nd.kind) {
                case KGPU_SIN_WT: { // osc.rs:110-123,142-147
                    h.f0 = (float)nd.args[0];
                    R(r + 2, v) = sat_u32((double)h.f0 * g.prog.sinwt_k);
                    break;
                }
                case KGPU_SIN_NUMERIC: { // osc.rs:231-237,253-261
                    float f = (float)nd.args[0];
                    R(r + 2, v) = fbits(f / sr);
                    break;
                }
                case KGPU_PHASOR: { // osc.rs:179-202: phase 0; init(): step = freq * (1 / sr), all f64
                    h.d0 = 1.0 / (double)sample_rate;
                    uint32_t lo, hi;
                    dbits(0.0, lo, hi);
                    R(r + 0, v) = lo; R(r + 1, v) = hi;
                    dbits(nd.args[0] * h.d0, lo, hi);
                    R(r + 2, v) = lo; R(r + 3, v) = hi;
                    break;
                }
                case KGPU_WHITE_NOISE: case KGPU_PINK_NOISE: case KGPU_BROWN_NOISE: { // noise.rs:33-38,69-78,134-139
                    const uint64_t seed = (uint64_t)nd.args[0];    // fastrand::Rng::with_seed(seed): the state IS the seed
                    R(r + 0, v) = (uint32_t)seed; R(r + 1, v) = (uint32_t)(seed >> 32);
                    if (nd.kind == KGPU_PINK_NOISE) R(r + 12, v) = 1u; // counter: 1 (noise.rs:74)
                    break;
                }
                case KGPU_PAN2: { // pan.rs:19-24
                    float gl, gr;
                    pan2_gains((float)nd.args[0] * 0.5f + 0.5f, gl, gr);
                    R(r + 0, v) = fbits(gl);
                    R(r + 1, v) = fbits(gr);
                    break;
                }
                case KGPU_RANDOM_LIN: { // noise.rs:170-185: new() draws current_value, init() scales the step and calls new_value()
                    uint64_t st = (uint64_t)nd.args[1];
                    const float current = wy_f32(st);
                    h.f0 = 1.0f / (float)sample_rate;                  // freq_to_phase_inc = F::ONE / F::from(sample_rate)
                    const float step = (float)nd.args[0] * h.f0;       // phase_step *= freq_to_phase_inc
                    const float old_target = current + 0.0f, nv = wy_f32(st);
                    R(r + 0, v) = (uint32_t)st; R(r + 1, v) = (uint32_t)(st >> 32);
                    R(r + 2, v) = fbits(old_target);
                    R(r + 3, v) = fbits(nv - old_target);
                    R(r + 4, v) = fbits(0.0f);
                    R(r + 5, v) = fbits(step);
                    break;
                }
                case KGPU_POLYBLEP: { // polyblep.rs:139-155
                    h.f0 = (float)nd.args[0];
                    float dt = 0.f;
                    if (h.f0 != 0.f) dt = h.f0 / sr;
                    R(r + 1, v) = fbits(dt);
                    R(r + 2, v) = (dt * sr >= sr / 4.0f) ? 1u : 0u;
                    R(r + 3, v) = fbits(0.5f);
                    R(r + 4, v) = nd.mode;
                    break;
                }
                case KGPU_SVF: { // svf.rs:64-79,134-141
                    h.f0 = (float)nd.args[0]; h.f1 = (float)nd.args[1]; h.f2 = (float)nd.args[2];
                    svf_coeffs(h.mode, h.f0, h.f1, h.f2, sr, h.svf_coef);
                    for (int i = 0; i < 6; i++) R(r + 2 + i, v) = fbits(h.svf_coef[i]);
                    for (int k = 0; k < dn.n_ar; k++)
                        if (dn.ar_code[k] >= AR_SVF_CUTOFF && dn.ar_code[k] <= AR_SVF_GAIN) h.ar_regs = true;
                    if (h.ar_regs) {
                        R(r + 8, v) = fbits(h.f0); R(r + 9, v) = fbits(h.f1); R(r + 10, v) = fbits(h.f2); R(r + 11, v) = h.mode;
                    }
                    break;
                }
                case KGPU_ONEPOLE_LPF: case KGPU_ONEPOLE_HPF: { // onepole.rs:118-129,157-167,35-46
                    float freq = nd.kind == KGPU_ONEPOLE_LPF ? (float)nd.args[0] : 0.0f;
                    float f = freq / sr;
                    float b1 = expf(-2.0f * F_PI * f);
                    R(r + 2, v) = fbits(b1);
                    R(r + 1, v) = fbits(1.0f - b1);
                    break;
                }
                case KGPU_ENV_ASR: case KGPU_ENV_AR: { // envelopes.rs:33-43,135-151
                    h.f0 = (float)nd.args[0]; h.f1 = (float)nd.args[1];
                    R(r + 2, v) = fbits(h.f0 == 0.f ? 1.0f : 1.0f / (h.f0 * sr));
                    R(r + 3, v) = fbits(h.f1 == 0.f ? 1.0f : 1.0f / (h.f1 * sr));
                    R(r + 4, v) = fbits(1.0f);
                    break;
                }
                case KGPU_ENVELOPE: { // envelopes.rs:372-384,403-405,329-335
                    h.d0 = nd.args[0];
                    uint32_t lo, hi;
                    dbits(nd.args[0], lo, hi);
                    R(r + 4, v) = lo; R(r + 5, v) = hi;
                    dbits(nd.args[1] * (1.0 / (double)sample_rate), lo, hi);
                    R(r + 6, v) = lo; R(r + 7, v) = hi;
                    for (uint32_t sgi = 0; sgi < nd.n_segments; sgi++) {
                        double dur = nd.segments[2 * sgi], val = nd.segments[2 * sgi + 1];
                        uint32_t b = r + REGS_ENVELOPE_BASE + REGS_ENVELOPE_PER_SEG * sgi;
                        dbits(1.0 / dur, lo, hi); R(b + 0, v) = lo; R(b + 1, v) = hi;
                        dbits(dur, lo, hi); R(b + 2, v) = lo; R(b + 3, v) = hi;
                        dbits(val, lo, hi); R(b + 4, v) = lo; R(b + 5, v) = hi;
                    }
                    break;
                }
                case KGPU_CONSTANT: case KGPU_TEST_NUM: R(r, v) = fbits((float)nd.args[0]); break;
                default: break;
                }
                // wrappers
                uint32_t inner = h.base_params;
                int post_i = 0;
                if (g.nstat[li].fast) { // everything but the wrapper VALUES is static (NodeStatic); next_delay lives in h.nd
                    for (uint32_t l = 0; l < nd.n_wrappers; l++)
                        if (is_math_wrapper(nd.wrappers[l].kind)) R(dn.post_reg[post_i++], v) = fbits((float)nd.wrappers[l].value);
                    continue;
                }
                h.wr.resize(nd.n_wrappers);
                for (uint32_t l = 0; l < nd.n_wrappers; l++) {
                    WrapSim &w = h.wr[l];
                    w.kind = (uint8_t)nd.wrappers[l].kind;
                    w.capacity = nd.wrappers[l].capacity;
                    w.inner_params = inner;
                    if (is_math_wrapper(w.kind)) {
                        w.reg = dn.post_reg[post_i++];
                        R(w.reg, v) = fbits((float)nd.wrappers[l].value);
                        if (w.kind == KGPU_WR_MUL) inner++;
                    } else if (w.kind == KGPU_WR_SMOOTH_PARAMS) {
                        w.smooth.assign(inner, SmoothState{});
                        h.has_smooth = true;
                        h.smooth_level = (int8_t)l;
                    } else if (w.kind == KGPU_WR_PRECISE_TIMING) {
                        w.next_delay.assign(inner, 0);
                        w.queue.reserve(std::min<uint32_t>(w.capacity, 8));
                        h.has_precise = true;
                        h.precise_level = (int8_t)l;
                    } else if (w.kind == KGPU_WR_AR_PARAMS) {
                        w.ar_bound.assign(inner, 0);
                        for (auto &pe : g.tpl.nodes[li].par)
                            if (std::get<0>(pe) < inner) w.ar_bound[std::get<0>(pe)] = 1;
                    }
                }
            }
    }
    finish_build();
}

// Validation of an event only depends on (group, node-in-template, parameter): cache it.
struct ParamRule {
    char want = 'f';      // expected ParameterValue kind ('t' trigger: anything fires)
    bool smooth_ok = false;
    bool polyblep_wave = false, svf_type = false;
};
static ParamRule param_rule(const TemplateNode &tn, uint32_t base_params, uint32_t p) {
    ParamRule r;
    bool wr_mul_target = false;
    std::vector<uint32_t> inner(tn.wrappers.size() + 1, base_params); // parameters visible below wrapper l
    for (size_t l = 0; l < tn.wrappers.size(); l++) inner[l + 1] = inner[l] + (tn.wrappers[l].kind == KGPU_WR_MUL ? 1u : 0u);
    for (int l = (int)tn.wrappers.size() - 1; l >= 0; l--) { // outermost -> innermost, like param_apply
        const uint32_t k = tn.wrappers[l].kind;
        if (k == KGPU_WR_MUL && p == inner[l]) { wr_mul_target = true; break; }
        if (k == KGPU_WR_SMOOTH_PARAMS && p < inner[l]) r.smooth_ok = true;
    }
    if (!wr_mul_target) {
        const char *types = param_types(tn.kind);
        r.want = p < std::strlen(types) ? types[p] : 'f';
        r.polyblep_wave = tn.kind == KGPU_POLYBLEP && p == 2;
        r.svf_type = tn.kind == KGPU_SVF && p == 3;
    }
    return r;
}

void HostPlan::finish_build() {
    const size_t n_groups = groups.size();
    voice_base.assign(n_groups + 1, 0);
    for (size_t gi = 0; gi < n_groups; gi++) voice_base[gi + 1] = voice_base[gi] + groups[gi].n_voices;
    voice_ramps.assign(voice_base.back(), 0);
    later.assign(n_groups, {});
    // validation rules, flat: [group][local][param] -> rule_base of the (group, local) + param
    rules.clear();
    std::vector<std::vector<uint32_t>> base(n_groups);
    for (size_t gi = 0; gi < n_groups; gi++) {
        const Group &g = groups[gi];
        base[gi].resize(g.tpl.nodes.size());
        for (size_t li = 0; li < g.tpl.nodes.size(); li++) {
            base[gi][li] = (uint32_t)rules.size();
            for (uint32_t p = 0; p < g.nstat[li].total_params; p++) {
                ParamRule pr = param_rule(g.tpl.nodes[li], g.nstat[li].base_params, p);
                const uint8_t ok_kinds = pr.want == 't' ? 0x1Eu : (pr.want == 'f' ? 1u << 1 : (pr.want == 'i' ? 1u << 3 : (pr.want == 'b' ? 1u << 4 : 0u)));
                rules.push_back({pr.want, (uint8_t)pr.smooth_ok, (uint8_t)pr.polyblep_wave, (uint8_t)pr.svf_type, ok_kinds});
            }
        }
    }
    for (NodeRef &nr : node_ref)
        if (nr.group >= 0) nr.rule_base = base[nr.group][nr.local];
}

void *kgpu_big_alloc(size_t bytes, size_t align) {
    constexpr size_t HUGE = size_t(2) << 20;
    if (bytes == 0) bytes = 1;
    const bool big = bytes >= HUGE;
    const size_t a = big ? HUGE : std::max<size_t>(align, 16);
    const size_t rounded = (bytes + a - 1) / a * a;
    void *p = aligned_alloc(a, rounded);
    if (!p) throw std::bad_alloc();
#if defined(__linux__) && defined(MADV_HUGEPAGE)
    if (big) madvise(p, rounded, MADV_HUGEPAGE); // a hint; failure changes nothing
#endif
    return p;
}

// ---- WorkPool -----------------------------------------------------------------------------------
struct WorkPool::Impl {
    std::mutex m;
    std::condition_variable cv_work, cv_done;
    std::vector<std::thread> threads;
    std::function<void(unsigned)> fn;
    unsigned n_tasks = 0, next = 0, running = 0;
    uint64_t generation = 0;
    bool stop = false;
    // claims and runs tasks of the current generation; called with the lock held
    void drain(std::unique_lock<std::mutex> &lk) {
        while (next < n_tasks) {
            const unsigned i = next++;
            running++;
            lk.unlock();
            fn(i);
            lk.lock();
            running--;
        }
        if (running == 0) cv_done.notify_all();
    }
    void loop() {
        std::unique_lock<std::mutex> lk(m);
        uint64_t seen = 0;
        for (;;) {
            cv_work.wait(lk, [&] { return stop || generation != seen; });
            if (stop) return;
            seen = generation;
            drain(lk);
        }
    }
};
WorkPool::WorkPool(unsigned n) : impl_(new Impl()), n_threads_(std::max(1u, n)) {
    for (unsigned i = 0; i < n_threads_; i++) impl_->threads.emplace_back([this] { impl_->loop(); });
}
WorkPool::~WorkPool() {
    {
        std::lock_guard<std::mutex> lk(impl_->m);
        impl_->stop = true;
    }
    impl_->cv_work.notify_all();
    for (auto &t : impl_->threads) t.join();
    delete impl_;
}
void WorkPool::start(unsigned n_tasks, std::function<void(unsigned)> fn) {
    std::unique_lock<std::mutex> lk(impl_->m);
    impl_->cv_done.wait(lk, [&] { return impl_->next >= impl_->n_tasks && impl_->running == 0; });
    impl_->fn = std::move(fn);
    impl_->n_tasks = n_tasks;
    impl_->next = 0;
    impl_->generation++;
    lk.unlock();
    impl_->cv_work.notify_all();
}
void WorkPool::wait() {
    std::unique_lock<std::mutex> lk(impl_->m);
    impl_->cv_done.wait(lk, [&] { return impl_->next >= impl_->n_tasks && impl_->running == 0; });
}
void WorkPool::run(unsigned n_tasks, std::function<void(unsigned)> fn) {
    start(n_tasks, std::move(fn));
    std::unique_lock<std::mutex> lk(impl_->m);
    impl_->drain(lk); // the caller helps
    impl_->cv_done.wait(lk, [&] { return impl_->next >= impl_->n_tasks && impl_->running == 0; });
}
WorkPool &HostPlan::workers() {
    if (!pool) {
        // one core is left to the thread that drives the device: it must not be starved while the
        // workers are busy, or the first launch waits for ALL of the simulation
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        unsigned n = std::min<unsigned>(hw > 2 ? hw - 1 : hw, 16u);
        if (pool_threads) n = pool_threads;
        if (const char *e = getenv("KGPU_THREADS")) n = (unsigned)std::max(1, atoi(e));
        pool = new WorkPool(n);
    }
    return *pool;
}

void HostPlan::push(const kgpu_event *evs, size_t n, uint64_t frame_clock) {
    struct PushTimer {
        std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
        size_t n;
        ~PushTimer() {
            static const bool on = getenv("KGPU_TIMING") != nullptr;
            if (on && n > 1000) fprintf(stderr, "[kgpu timing]   push %zu events %.1f ms\n", n, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count());
        }
    } push_timer;
    push_timer.n = n;
    // One pass: every event is validated and converted into its own position of `pending` (grown uninitialised).
    // A failing call queues nothing: `pending` is cut back and the first failing event, in event order, is reported.
    // Events of unreachable nodes are rare and are squeezed out afterwards.
    const NodeRef *nref = node_ref.data();
    const size_t n_nodes = node_ref.size();
    const Rule *rl = rules.data();
    const uint64_t *vbase = voice_base.data();
    const uint64_t sr = sample_rate;
    auto one = [&](size_t i, RawEvent &r) -> bool { // false: dropped (the node reaches no output)
        const kgpu_event &e = evs[i];
        if (e.node >= n_nodes) KGPU_THROW(KGPU_ERR_INVALID, "event %zu: NodeNotFound (%u)", i, e.node);
        const NodeRef nr = nref[e.node];
        if (e.param >= nr.n_params) KGPU_THROW(KGPU_ERR_PARAMETER, "event %zu: ParameterIndexOutOfBounds (node %u param %u)", i, e.node, e.param);
        if (e.value_kind > 4 || e.smoothing_kind > 2 || e.time_kind > 2) KGPU_THROW(KGPU_ERR_INVALID, "event %zu: bad enum field", i);
        if (e.smoothing_kind != 0 && e.smooth_rate != 0)
            KGPU_THROW(KGPU_ERR_UNSUPPORTED, "event %zu: Rate::AudioRate smoothing is not supported (its branch is unreachable in knaster, "
                       "smooth_params.rs:140-146)", i);
        if (nr.group < 0) return false; // unreachable node: knaster would run it, but nothing can hear it
        const Rule &ru = rl[nr.rule_base + e.param];
        if (e.smoothing_kind != 0 && !ru.smooth_ok)
            KGPU_THROW(KGPU_ERR_PARAMETER, "event %zu: smoothing sent to node %u param %u which has no WrSmoothParams around it "
                       "(knaster would panic: parameter value is expected to be a float)", i, e.node, e.param);
        if (e.value_kind != 0) {
            const bool ok = (ru.ok_kinds >> e.value_kind) & 1u; // value_kind <= 4 (checked above)
            if (!ok) KGPU_THROW(KGPU_ERR_PARAMETER, "event %zu: wrong value type for node %u param %u", i, e.node, e.param);
            if (ru.polyblep_wave && ((int64_t)e.value < 0 || (int64_t)e.value > 13))
                KGPU_THROW(KGPU_ERR_PARAMETER, "event %zu: bad PolyBlep Waveform %lld", i, (long long)e.value);
            if (ru.svf_type && ((int64_t)e.value < 0 || (int64_t)e.value > 8))
                KGPU_THROW(KGPU_ERR_PARAMETER, "event %zu: bad SvfFilterType", i);
        }
        r.node = e.node;
        r.gvoice = (uint32_t)(vbase[nr.group] + nr.voice);
        r.param = (uint16_t)e.param;
        r.local = (uint8_t)nr.local;
        r.kinds = (uint8_t)(e.value_kind | (e.smoothing_kind << 3) | ((e.time_kind != 0 ? 1u : 0u) << 5));
        r.smooth_seconds = e.smooth_seconds;
        r.value = e.value_kind == 3 ? (double)(int64_t)e.value : e.value;
        const uint64_t samples = (uint64_t)e.seconds * sr + ((uint64_t)e.subsec * sr) / 282240000ull; // time.rs:86-90
        uint64_t due;
        if (e.time_kind == 1) due = samples;                    // scheduling.rs:102-108
        else if (e.time_kind == 2) due = frame_clock + samples; // scheduling.rs:110-119
        else due = frame_clock;
        r.due_frame = due < frame_clock ? frame_clock : due;    // late: saturating_sub -> delay 0
        return true;
    };
    // (one chunk more than the pool has threads: WorkPool::run lets the calling thread take one as well)
    const unsigned T = n >= 32768 ? std::min<unsigned>(workers().size() + 1, (unsigned)(n / 8192)) : 1u;
    std::vector<size_t> dropped(T, 0);
    std::vector<Error> errs(T, Error{0, ""});
    const size_t base = pending.size();
    pending.resize(base + n);
    // A large batch pushed into an empty queue is bucketed by voice while it is converted (the per-chunk histograms
    // stream_begin needs, and whether the events already arrive grouped by voice and in time order): the render call
    // that follows then has no pass of its own over the events before its first launch.
    BucketPrep &bp = bucket_prep;
    const bool track = base == 0 && n >= 32768 && far_horizon == UINT64_MAX;
    bp.valid = false;
    if (track) bp.reset(T, voice_base.back());
    auto chunk = [&](unsigned c) {
        const size_t i0 = n * c / T, i1 = n * (c + 1) / T;
        size_t d = 0;
        RawEvent *dst = pending.data() + base;
        uint32_t *hc = track ? bp.hist[c].data() : nullptr;
        uint32_t prev = 0;
        uint64_t prev_due = 0, max_due = 0;
        bool mono = true;
        try {
            for (size_t i = i0; i < i1; i++) {
                if (!one(i, dst[i])) {
                    dst[i].node = 0xFFFFFFFFu; // dropped
                    d++;
                    continue;
                }
                if (track) {
                    const RawEvent &r = dst[i];
                    if (i == i0) {
                        bp.first_v[c] = r.gvoice;
                        bp.first_due[c] = r.due_frame;
                    }
                    // voices ascending, and inside a voice in time order (then also in ready-block order)
                    mono &= r.gvoice > prev || (r.gvoice == prev && r.due_frame >= prev_due) || i == i0;
                    prev = r.gvoice;
                    prev_due = r.due_frame;
                    max_due = std::max(max_due, r.due_frame);
                    hc[r.gvoice]++;
                }
            }
        } catch (const Error &e) {
            errs[c] = e;
        }
        dropped[c] = d;
        if (track) {
            bp.last_v[c] = prev;
            bp.last_due[c] = prev_due;
            bp.mono[c] = mono;
            bp.max_due[c] = max_due;
        }
    };
    if (T == 1) chunk(0);
    else workers().run(T, chunk);
    for (unsigned c = 0; c < T; c++)
        if (errs[c].code) {
            pending.resize(base);
            throw errs[c]; // chunks are in event order: this is the first failing event
        }
    size_t n_dropped = 0;
    for (unsigned c = 0; c < T; c++) n_dropped += dropped[c];
    if (n_dropped) {
        size_t w = base;
        for (size_t i = base; i < base + n; i++)
            if (pending[i].node != 0xFFFFFFFFu) pending[w++] = pending[i];
        pending.resize(w);
    } else if (track) {
        bp.valid = true;
        bp.n = n;
    }
}

namespace {
struct PhaseTimer {
    const char *name;
    std::chrono::steady_clock::time_point t;
    explicit PhaseTimer(const char *n) : name(n), t(std::chrono::steady_clock::now()) {}
    void lap(const char *what) {
        static const bool on = getenv("KGPU_TIMING") != nullptr;
        auto n = std::chrono::steady_clock::now();
        if (on) fprintf(stderr, "[kgpu timing]   %s/%s %.1f ms\n", name, what, std::chrono::duration<double, std::milli>(n - t).count());
        t = n;
    }
};

inline PV pv_of(const RawEvent &r) {
    PV pv;
    pv.kind = (PV::Kind)r.value_kind();
    pv.f = r.value;
    return pv;
}

// ---- one node, one block, block-by-block model (any wrapper stack): what GraphGen does with the node's ready events at
// the top of the block (graph_gen.rs:269-305) and what the wrapper stack's process_block then does at control rate.
// ev[0..n): the voice's ready events of this block in arrival order; only those of node `local` are this node's.
void generic_node_block(Sim &s, const RawEvent *const *ev, size_t n, uint32_t local, uint64_t block_start, uint64_t bs) {
    HostNode &hn = s.hn;
    const int top = (int)hn.wr.size() - 1;
    for (size_t i = 0; i < n; i++) { // apply_parameter_change, graph_gen.rs:269-305
        const RawEvent &r = *ev[i];
        if (r.local != local) continue;
        const uint64_t delay = r.timed() && r.due_frame > block_start ? r.due_frame - block_start : 0;
        if (delay > 0) wr_set_delay(s, top, r.param, (uint16_t)delay);
        if (r.smoothing_kind()) {
            PV pv;
            pv.kind = PV::Smoothing;
            pv.smoothing = r.smoothing_kind() == 2 ? 1 : 0;
            pv.smooth_seconds = r.smooth_seconds;
            wr_param_apply(s, top, r.param, pv, block_start);
        }
        if (r.value_kind()) wr_param_apply(s, top, r.param, pv_of(r), block_start);
    }
    if (needs_processing(hn)) wr_process_block(s, top, block_start, 0, (uint32_t)bs);
}

// ---- the same for a node WITHOUT WrSmoothParams (NodeStatic::fast), in closed form.  Such a node's wrapper stack has no
// control-rate state besides WrPreciseTiming's sticky next_delay[]: its queue is filled by the block's events and drained
// by the same block's process_block, which applies queued change k at the frame of the largest delay among changes
// 0..k (the scan stops at the first change that is not due yet and resumes there, precise_timing.rs:82-101).  Changes
// that are not delayed apply at the block start, before every queued one.  Device events come out in the order the
// block-by-block model emits them.
inline bool route_levels(Sim &s, const NodeStatic &ns, int from, int stop, const RawEvent &r, uint64_t frame) {
    for (int l = from; l > stop; l--) {
        const uint8_t k = ns.lv_kind[l];
        if (k == KGPU_WR_MUL) {
            if (r.param == ns.lv_inner[l]) { // the wrapper's own parameter, wrappers_core/math.rs:92-98
                if (r.value_kind() == PV::Float) s.set_f(frame, ns.lv_reg[l], (float)r.value);
                return false;
            }
        } else if (k == KGPU_WR_AR_PARAMS) { // audio_rate.rs:70-74: ignored while a buffer is set
            if (r.param < 32 && ((ns.lv_ar_mask[l] >> r.param) & 1u)) return false;
        }
    }
    return true;
}
void fast_node_block(Sim &s, const NodeStatic &ns, const RawEvent *const *ev, size_t n, uint32_t local, uint64_t block_start) {
    HostNode &hn = s.hn;
    const int top = (int)ns.n_levels - 1, pl = ns.precise_level;
    const RawEvent *queue[32];
    uint16_t qdelay[32];
    uint32_t nq = 0;
    for (size_t i = 0; i < n; i++) {
        const RawEvent &r = *ev[i];
        if (r.local != local) continue;
        const uint64_t delay = r.timed() && r.due_frame > block_start ? r.due_frame - block_start : 0;
        if (delay > 0) { // set_delay_within_block_for_param through the stack
            if (ns.delay_reaches) {
                if (r.param < ns.nd_size) hn.nd[r.param] = (uint16_t)delay; // precise_timing.rs:146-148
            } else s.out.ignored++;                                         // ugen.rs:339-341: warning, no effect
        }
        if (!r.value_kind()) continue; // (smoothing settings never reach a node without WrSmoothParams: rejected at push time)
        if (pl < 0) {
            if (route_levels(s, ns, top, -1, r, block_start)) ugen_param_apply(s, r.param, pv_of(r), block_start);
            continue;
        }
        if (!route_levels(s, ns, top, pl, r, block_start)) continue;
        if (r.param >= ns.nd_size) continue;                     // would index out of bounds in knaster
        const uint16_t nd = hn.nd[r.param];
        if (nd == 0) {                                           // precise_timing.rs:127-128: apply now
            if (route_levels(s, ns, pl - 1, -1, r, block_start)) ugen_param_apply(s, r.param, pv_of(r), block_start);
        } else if (nq < ns.capacity) {                           // :129-131
            queue[nq] = &r;
            qdelay[nq++] = nd;
        } else s.out.dropped++;                                  // :132-134
    }
    uint32_t run_max = 0;
    for (uint32_t k = 0; k < nq; k++) {
        run_max = std::max<uint32_t>(run_max, qdelay[k]);
        const uint64_t frame = block_start + run_max;
        if (route_levels(s, ns, pl - 1, -1, *queue[k], frame)) ugen_param_apply(s, queue[k]->param, pv_of(*queue[k]), frame);
    }
}
} // namespace

// ------------------------------------------------------------------------------------------------
// The host half of a render call for frames [bounds.front(), bounds.back()), launch L covering
// [bounds[L], bounds[L+1]).  The control simulation runs per voice (voices are independent) on
// worker threads that each own a slice of every group's voices and walk the launches IN ORDER,
// publishing how many launches they have finished: the caller can upload launch L and start its
// kernels while the workers are already simulating launch L+1 (stream_begin / stream_launch /
// stream_end).  A voice is walked block by block over the blocks in which something happens (a ready
// event, an active smoothing ramp); the device events of a block are ordered the way the kernels
// consume them -- (frame / chunk, node, frame, arrival) -- and appended to the launch's list.
struct StreamState {
    struct PerGroup {
        uint32_t v_begin = 0, v_end = 0;
        std::vector<std::vector<DevEvent>> ev;   // per launch (capacity kept from call to call)
        std::vector<std::vector<uint32_t>> cnt;  // per launch, per voice of the slice
        std::vector<uint32_t> cursor;            // per voice of the slice: next unconsumed ready event
        std::vector<uint64_t> next_due;          // ... and its due frame (UINT64_MAX: none left): the per-window skip test
    };
    struct alignas(128) ThreadCtx {
        std::vector<PerGroup> g;
        Sink sink;
        std::vector<const RawEvent *> evp;
        int64_t ramp_delta = 0;
        uint64_t prof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        std::atomic<uint32_t> done{0};           // launches finished
        std::string error;
        int error_code = 0;
    };
    std::vector<uint64_t> bounds;
    std::vector<uint32_t> chunks;
    size_t n_launch = 0, n_ready = 0;
    uint64_t b0 = 0;
    bool any_work = false;
    bool identity = false;                       // the ready events are `pending` itself, already grouped by voice: vorder unused
    bool all_ready = false;                      // every queued event is consumed by this call (known from push's bucketing): the queue is simply cleared
    unsigned n_threads = 0;                      // contexts of this call: th[0..n_threads)
    int driver_ctx = -1;                         // >= 0: th[driver_ctx] (the last slice) is simulated by the calling thread, launch by launch
    size_t driver_done = 0;                      // launches of that slice already simulated
    std::vector<std::unique_ptr<ThreadCtx>> th;
    std::vector<std::vector<uint32_t>> hist;     // bucketing scratch
    bool pooled = false; // workers run on HostPlan::pool
    std::chrono::steady_clock::time_point t_begin = std::chrono::steady_clock::now();
};

#ifdef KGPU_PROFILE_HOST
// cycle counters of the control simulation, summed over the worker threads and printed by stream_end
#include <x86intrin.h>
#define PROF_T(var) const uint64_t var = __rdtsc()
#define PROF_ADD(i, a, b) tc.prof[i] += (b) - (a)
#else
#define PROF_T(var)
#define PROF_ADD(i, a, b)
#endif

namespace {
constexpr int NODE_MASK_WORDS = (MAX_NODES + 63) / 64;
static_assert(MAX_NODES <= 256, "RawEvent::local holds a template node index in a byte");
// one voice, one launch window: what a separate render call over that window would do
void simulate_voice_window(HostPlan &P, StreamState &S, StreamState::ThreadCtx &tc, uint32_t gi, uint32_t v, size_t L) {
    Group &g = P.groups[gi];
    StreamState::PerGroup &pg = tc.g[gi];
    const uint64_t bs = P.block_size;
    const uint32_t nn = (uint32_t)g.tpl.nodes.size();
    const uint64_t t0 = S.bounds[L], t1 = S.bounds[L + 1];
    const uint64_t wb0 = t0 / bs, wb1 = t1 / bs;
    const size_t gv = P.voice_base[gi] + v;
    const RawEvent *pend = P.pending.data();
    PROF_T(p0);
    // ready events of this voice inside the window (sorted by ready block inside a voice)
    uint32_t &cur = pg.cursor[v - pg.v_begin];
    const uint32_t e0 = cur, vend = P.vcount[gv + 1];
    const uint32_t *vo = S.identity ? nullptr : P.vorder.data();
    auto ev_at = [&](uint32_t k) -> const RawEvent & { return pend[vo ? vo[k] : k]; };
    if (L == 0 && vend - e0 > 1 && !S.identity) { // first visit: (ready block, arrival) order; identity bucketing has checked it
        // events that arrive in frame order (the usual case) are in block order: checked without a division
        bool sorted = true;
        for (uint32_t k = e0 + 1; k < vend && sorted; k++) sorted = ev_at(k - 1).due_frame <= ev_at(k).due_frame;
        if (!sorted) {
            auto rb = [&](const RawEvent &r) { return std::max(r.due_frame / bs, S.b0); };
            sorted = true;
            for (uint32_t k = e0 + 1; k < vend && sorted; k++) sorted = rb(ev_at(k - 1)) <= rb(ev_at(k));
            if (!sorted) {
                std::stable_sort(P.vorder.begin() + e0, P.vorder.begin() + vend, [&](uint32_t x, uint32_t y) { return rb(pend[x]) < rb(pend[y]); });
            }
        }
    }
    uint32_t e1 = e0;
    while (e1 < vend && ev_at(e1).due_frame < t1) e1++; // t1 is a block boundary: same as due block < wb1
    cur = e1;
    pg.next_due[v - pg.v_begin] = e1 < vend ? ev_at(e1).due_frame : UINT64_MAX;
    PROF_T(p1);
    PROF_ADD(0, p0, p1);
    if (e0 == e1 && !P.voice_ramps[gv]) return;

    const uint32_t chunk_shift = (uint32_t)__builtin_ctz(S.chunks[gi]); // chunk is a power of two (capi.cpp pick_chunk; recipes: 1)
    Sink &sk = tc.sink;
    sk.t0 = t0;
    std::vector<DevEvent> &out = pg.ev[L];
    sk.dst = &out;
    const size_t out0 = out.size();
    auto ready_block = [&](uint32_t k) { return std::max(P.block_of(ev_at(k).due_frame), wb0); };
    uint32_t ei = e0;
    uint64_t b = P.voice_ramps[gv] ? wb0 : ready_block(ei);
    std::vector<const RawEvent *> &evp = tc.evp;
    while (b < wb1) {
        const uint64_t block_start = b * bs;
        // this block's ready events, arrival order
        PROF_T(q0);
        evp.clear();
        // nodes of the voice with a ready event: one bit per template node (MAX_NODES of them)
        uint64_t mask[NODE_MASK_WORDS] = {};
        while (ei < e1 && ready_block(ei) == b) {
            const RawEvent &r = ev_at(ei++);
            evp.push_back(&r);
            mask[r.local >> 6] |= 1ull << (r.local & 63u);
        }
        const size_t blk0 = out.size(); // this block's device events: out[blk0 ..)
        PROF_T(q1);
        PROF_ADD(1, q0, q1);
        for (uint32_t li = 0; li < nn; li++) {
            const NodeStatic &ns = g.nstat[li];
            HostNode &hn = g.host[(size_t)v * nn + li];
            if (!((mask[li >> 6] >> (li & 63u)) & 1u) && (ns.fast || !hn.ramp_active)) continue; // (a fast node never ramps: its state is not even touched)
            Sim s{P, sk, li, hn};
            if (ns.fast) {
                fast_node_block(s, ns, evp.data(), evp.size(), li, block_start);
            } else {
                const bool was = hn.ramp_active;
                generic_node_block(s, evp.data(), evp.size(), li, block_start, bs);
                hn.ramp_active = needs_processing(hn);
                if (hn.ramp_active != was) {
                    tc.ramp_delta += hn.ramp_active ? 1 : -1;
                    P.voice_ramps[gv] += hn.ramp_active ? 1 : -1;
                }
            }
        }
        // device order inside the block: (frame / chunk, node, frame, arrival).  Emission order is (node, frame, arrival),
        // so a stable sort by chunk is all that is left (insertion sort: a block holds a handful of events)
        const size_t nb = out.size() - blk0;
        PROF_T(q2);
        PROF_ADD(2, q1, q2);
        if (nb) {
            sk.devev += nb;
            DevEvent *be = out.data() + blk0;
            bool sorted = true; // the usual block: a handful of events that share a frame, or come in frame order
            for (size_t i = 1; i < nb && sorted; i++) sorted = (be[i - 1].frame >> chunk_shift) <= (be[i].frame >> chunk_shift);
            if (!sorted)
                for (size_t i = 1; i < nb; i++) {
                    const DevEvent x = be[i];
                    const uint32_t kx = x.frame >> chunk_shift;
                    size_t j = i;
                    while (j > 0 && (be[j - 1].frame >> chunk_shift) > kx) {
                        be[j] = be[j - 1];
                        j--;
                    }
                    be[j] = x;
                }
        }
        PROF_T(q3);
        PROF_ADD(3, q2, q3);
        if (P.voice_ramps[gv]) b++;
        else if (ei < e1) b = ready_block(ei);
        else break;
    }
    pg.cnt[L][v - pg.v_begin] = (uint32_t)(out.size() - out0);
}

#ifndef KGPU_HOST_PREFETCH
#define KGPU_HOST_PREFETCH 8 // voices of look-ahead in the control simulation's walk (0: none)
#endif
// one slice of the voices, one launch window
void stream_worker_step(HostPlan &P, StreamState &S, StreamState::ThreadCtx &tc, size_t L) {
    for (uint32_t gi = 0; gi < P.groups.size(); gi++) {
        StreamState::PerGroup &pg = tc.g[gi];
        // calls without active ramps (block-by-block rendering, banks without smoothing): a voice without a
        // ready event has nothing to do -- skip it on two loads instead of entering the simulation
        const bool quick = P.n_active_ramps == 0 && tc.ramp_delta == 0;
        const uint64_t t1 = S.bounds[L + 1];
        const uint64_t *nd = pg.next_due.data();
        // The walk is latency-bound: a voice's control-side nodes and its next events were last touched a launch ago (megabytes
        // of other voices in between).  They are fetched KGPU_PF voices ahead of their use.
        Group &g = P.groups[gi];
        const size_t nn = g.tpl.nodes.size(), node_bytes = nn * sizeof(HostNode);
        const char *hosts = reinterpret_cast<const char *>(g.host.data());
        const uint32_t *cur = pg.cursor.data();
        const uint32_t *vo = S.identity ? nullptr : P.vorder.data();
        const RawEvent *pend = P.pending.data();
        constexpr uint32_t KGPU_PF = KGPU_HOST_PREFETCH;
        for (uint32_t v = pg.v_begin; v < pg.v_end; v++) {
            const uint32_t vp = v + KGPU_PF;
            if (KGPU_PF && vp < pg.v_end && !(quick && nd[vp - pg.v_begin] >= t1)) {
                const char *h = hosts + (size_t)vp * node_bytes;
                for (size_t o = 0; o < node_bytes; o += sizeof(HostNode)) __builtin_prefetch(h + o, 0, 3); // the hot line of every node (plan.hpp)
                const uint32_t c = cur[vp - pg.v_begin];
                if (c < P.vcount[P.voice_base[gi] + vp + 1]) {
                    const char *e = reinterpret_cast<const char *>(pend + (vo ? vo[c] : c));
                    __builtin_prefetch(e, 0, 3);
                    __builtin_prefetch(e + 64, 0, 3); // a window holds two to four of the voice's events on average
                }
            }
            if (quick && nd[v - pg.v_begin] >= t1) continue; // nothing of this voice becomes ready in this window
            simulate_voice_window(P, S, tc, gi, v, L);
        }
    }
}

void stream_worker(HostPlan &P, StreamState &S, unsigned ti) {
    StreamState::ThreadCtx &tc = *S.th[ti];
    static const bool timing = getenv("KGPU_TIMING") != nullptr;
    try {
        for (size_t L = 0; L < S.n_launch; L++) {
            stream_worker_step(P, S, tc, L);
            tc.done.store((uint32_t)L + 1, std::memory_order_release);
            if (timing && L < 2 && ti < 3 && S.n_launch > 2)
                fprintf(stderr, "[kgpu timing]     worker %u finished launch %zu at +%.2f ms\n", ti, L,
                        std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - S.t_begin).count());
        }
    } catch (const Error &e) {
        tc.error = e.msg;
        tc.error_code = e.code;
        tc.done.store((uint32_t)S.n_launch, std::memory_order_release);
    }
}
} // namespace

HostPlan::~HostPlan() {
    if (stream) {
        if (stream_active && stream->pooled && pool) pool->wait();
        delete stream;
    }
    delete pool;
}

// Keeps `pending` short for small render windows.  Invariant while active: every event of `pending` is due
// before block far_horizon, every event of `pending_far` at or after it; both in arrival order.  Moving
// events between the two never reorders events that become ready in the same block: the two sets are
// separated by due block, moves are stable, and an event is due no earlier than the frame clock at which
// it was pushed (HostPlan::push clamps), so "due block" IS the block in which it becomes ready.
void HostPlan::calendar_update(uint64_t b0, uint64_t b1) {
    constexpr uint64_t H = 64; // blocks of look-ahead kept in `pending`
    const uint64_t bs = block_size;
    if (far_horizon == UINT64_MAX) {
        // switch on when a short window faces a long queue (one block at a time under seconds of schedule)
        if (pending.size() < 16384 || b1 - b0 > H / 4) return;
        far_horizon = b1 + H;
        pending_clean = 0;
    }
    // first: newly pushed events that lie beyond the horizon go to the END of the far queue
    size_t w = pending_clean;
    for (size_t i = pending_clean; i < pending.size(); i++) {
        if (pending[i].due_frame / bs >= far_horizon) pending_far.push_back(pending[i]);
        else {
            if (w != i) pending[w] = pending[i];
            w++;
        }
    }
    pending.resize(w);
    pending_clean = w;
    if (b1 > far_horizon || (b1 + H / 4 > far_horizon && !pending_far.empty())) {
        // the window comes close to the horizon: pull the next stretch in (one scan of the far queue per ~H blocks)
        const uint64_t nh = b1 + H;
        size_t w = 0;
        for (size_t i = 0; i < pending_far.size(); i++) {
            if (pending_far[i].due_frame / bs < nh) pending.push_back(pending_far[i]);
            else {
                if (w != i) pending_far[w] = pending_far[i];
                w++;
            }
        }
        pending_far.resize(w);
        // (events pushed since the last call that lie beyond the OLD horizon were appended to the far queue just
        // above, behind everything that arrived before them, and come back in that order)
        far_horizon = nh;
        pending_clean = pending.size();
    }
    if (pending_far.empty()) { // nothing left to hold back
        far_horizon = UINT64_MAX;
        pending_clean = 0;
    }
}

void HostPlan::stream_begin(const std::vector<uint64_t> &bounds, const std::vector<uint32_t> &chunk_of_group) {
    PhaseTimer pt("stream_begin");
    if (stream_active) KGPU_THROW(KGPU_ERR_STATE, "stream_begin: a render call is already in progress");
    const uint64_t bs = block_size;
    const uint64_t t0 = bounds.front(), t1 = bounds.back();
    const uint64_t b0 = t0 / bs, b1 = t1 / bs;
    const size_t n_launch = bounds.size() - 1, n_groups = groups.size();
    calendar_update(b0, b1);
    // ---- ready events: due block < b1 (graph_gen.rs:283: ready iff delay < block_size).
    // `pending` stays in arrival order.  Inside a voice the workers need (block in which the event
    // becomes ready, arrival) order -- late events become ready in block b0 whatever their due time
    // (saturating_sub, graph_gen.rs:276) and keep their arrival order among the events of that
    // block, which is the order knaster's waiting queue applies them in.  Bucketing by voice keeps
    // arrival order; each worker then stable-sorts the (rare) voices whose events did not arrive
    // in time order.
    const size_t NV = voice_base.back();
    const size_t NP = pending.size();
    const uint64_t t_ready = b1 * bs; // ready iff due_frame < t_ready
    if (!stream) stream = new StreamState();
    StreamState *S = stream;
    S->t_begin = std::chrono::steady_clock::now();
    // per-chunk histograms over the voices (chunks in arrival order => a stable bucket sort).  The same pass notices
    // when there is nothing to sort: every queued event is ready and the events already arrive grouped by voice, voices
    // ascending (a schedule written voice by voice) -- then `pending` itself is the bucketed list.
    BucketPrep &bp = bucket_prep;
    bool prepped = bp.valid && bp.n == NP && far_horizon == UINT64_MAX && bp.hist.size() >= bp.T && NP > 0;
    if (prepped)
        for (unsigned c = 0; c < bp.T; c++) prepped &= bp.max_due[c] < t_ready; // every queued event is ready
    bp.valid = false; // one use: the queue changes below / at the end of the call
    S->all_ready = prepped;
    const unsigned TB = prepped ? bp.T : (NP >= 65536 ? workers().size() : 1u);
    std::vector<std::vector<uint32_t>> &hist = prepped ? bp.hist : S->hist;
    hist.resize(std::max<size_t>(hist.size(), TB));
    std::vector<uint8_t> mono(TB, 1);
    std::vector<uint32_t> first_v(TB, 0xFFFFFFFFu), last_v(TB, 0);
    std::vector<uint64_t> first_due(TB, 0), last_due(TB, 0);
    if (prepped) {
        mono = bp.mono;
        first_v = bp.first_v; last_v = bp.last_v;
        first_due = bp.first_due; last_due = bp.last_due;
    }
    auto count_chunk = [&](unsigned c) {
        std::vector<uint32_t> &hc = hist[c];
        hc.assign(NV, 0);
        const size_t i0 = NP * c / TB, i1 = NP * (c + 1) / TB;
        uint32_t prev = 0;
        uint64_t prev_due = 0;
        bool m = true;
        for (size_t i = i0; i < i1; i++) {
            const RawEvent &r = pending[i];
            if (r.due_frame >= t_ready) {
                m = false;
                continue;
            }
            if (i == i0) {
                first_v[c] = r.gvoice;
                first_due[c] = r.due_frame;
            }
            // voices ascending, and inside a voice in time order (then also in ready-block order)
            m &= r.gvoice > prev || (r.gvoice == prev && r.due_frame >= prev_due) || i == i0;
            prev = r.gvoice;
            prev_due = r.due_frame;
            hc[r.gvoice]++;
        }
        last_v[c] = prev;
        last_due[c] = prev_due;
        mono[c] = m;
    };
    if (prepped) {}
    else if (TB == 1) count_chunk(0);
    else workers().run(TB, count_chunk);
    bool identity = NP > 0;
    for (unsigned c = 0; c < TB && identity; c++) {
        identity = mono[c] != 0;
        if (c > 0 && NP * c / TB < NP * (c + 1) / TB && first_v[c] != 0xFFFFFFFFu)
            identity &= first_v[c] > last_v[c - 1] || (first_v[c] == last_v[c - 1] && first_due[c] >= last_due[c - 1]);
    }
    // hist[c][v] becomes chunk c's first slot for voice v, relative to the voice's first slot vcount[v]; the TB x NV walk is
    // shared between the workers (it was 0.2 ms of the 0.7 ms a render call spends before its first launch)
    vcount.assign(NV + 1, 0);
    auto voice_totals = [&](size_t v0, size_t v1) {
        for (size_t v = v0; v < v1; v++) {
            uint32_t run = 0;
            for (unsigned c = 0; c < TB; c++) {
                const uint32_t k = hist[c][v];
                hist[c][v] = run;
                run += k;
            }
            vcount[v + 1] = run;
        }
    };
    if (TB > 1 && NV >= 4096) {
        const unsigned TV = workers().size();
        workers().run(TV, [&](unsigned c) { voice_totals(NV * c / TV, NV * (c + 1) / TV); });
    } else voice_totals(0, NV);
    for (size_t v = 0; v < NV; v++) vcount[v + 1] += vcount[v];
    const size_t n_ready = vcount[NV];
    bool any_work = n_ready > 0 || n_active_ramps > 0;
    S->bounds = bounds;
    S->chunks = chunk_of_group;
    S->n_launch = n_launch;
    S->n_ready = n_ready;
    S->b0 = b0;
    S->any_work = any_work;
    S->identity = identity;
    S->pooled = false;
    S->n_threads = 0;
    S->driver_ctx = -1;
    S->driver_done = 0;
    stream_active = true;
    if (!any_work) return;
    // bucket by global voice (arrival order inside a voice)
    if (!identity) {
        vorder.resize(n_ready);
        auto scatter_chunk = [&](unsigned c) {
            std::vector<uint32_t> &hc = hist[c];
            const size_t i0 = NP * c / TB, i1 = NP * (c + 1) / TB;
            for (size_t i = i0; i < i1; i++) {
                const RawEvent &r = pending[i];
                if (r.due_frame >= t_ready) continue;
                vorder[vcount[r.gvoice] + hc[r.gvoice]++] = (uint32_t)i;
            }
        };
        if (TB == 1) scatter_chunk(0);
        else workers().run(TB, scatter_chunk);
    }
    pt.lap("bucket");
    const size_t work = n_ready + n_active_ramps;
    unsigned T = work > 20000 ? workers().size() : 1u;
    T = std::min<unsigned>(T, std::max<unsigned>(1u, (unsigned)(NV / 64)));
    // With few workers (several GPUs sharing one box's cores) the control simulation, not the device, paces the call, and the
    // calling thread would only wait for them: it takes a slice of the voices of its own -- half a worker's, it also merges,
    // uploads and launches -- and simulates it launch by launch inside stream_launch.
    // Measured on the bench configuration (one B200, 16 host cores): 3 workers 15.35 -> 15.07 ms per step end to end; 7 workers
    // 14.48 -> 14.53 ms (the device paces that call, nothing to gain), so the slice is taken with up to 4 workers only.
    static const char *drv_env = getenv("KGPU_DRIVER_SLICE"); // 0 = never, 1 = whenever workers run (default: up to 4 workers)
    const bool driver_slice = T > 1 && (drv_env ? atoi(drv_env) != 0 : T <= 4) && NV >= 64u * (T + 1);
    // slice weights: a worker 100, the calling thread KGPU_DRIVER_WEIGHT (default 50: it also merges, uploads and launches)
    static const unsigned drv_weight = [] {
        const char *e = getenv("KGPU_DRIVER_WEIGHT");
        const int w = e ? atoi(e) : 50;
        return (unsigned)std::min(100, std::max(5, w));
    }();
    const unsigned NT = T + (driver_slice ? 1u : 0u), WT = driver_slice ? 100 * T + drv_weight : T;
    S->n_threads = NT;
    S->driver_ctx = driver_slice ? (int)T : -1;
    while (S->th.size() < NT) S->th.emplace_back(new StreamState::ThreadCtx());
    // every worker lays out its own context (per-launch event lists and counts, per-voice cursors) before it starts on
    // launch 0: in parallel, 0.3 ms of the call's start-up when the driver thread did it for all of them
    for (unsigned ti = 0; ti < NT; ti++) { // what the driver thread polls (stream_launch) is reset before any worker runs
        StreamState::ThreadCtx &tc = *S->th[ti];
        tc.done.store(0, std::memory_order_relaxed);
        tc.error.clear();
        tc.error_code = 0;
    }
    const uint32_t *vo_all = identity ? nullptr : vorder.data();
    auto init_ctx = [this, S, n_groups, n_launch, T, WT, driver_slice, identity, vo_all](unsigned ti) {
        const uint32_t *vo = vo_all;
        StreamState::ThreadCtx &tc = *S->th[ti];
        tc.g.resize(n_groups);
        tc.ramp_delta = 0;
        tc.sink.dropped = tc.sink.ignored = tc.sink.devev = 0;
        const unsigned w0 = driver_slice ? 100 * ti : ti, w1 = driver_slice ? std::min(100 * ti + 100, WT) : ti + 1;
        (void)T;
        for (size_t gi = 0; gi < n_groups; gi++) {
            StreamState::PerGroup &pg = tc.g[gi];
            const uint32_t V = groups[gi].n_voices;
            pg.v_begin = (uint32_t)((uint64_t)V * w0 / WT);
            pg.v_end = (uint32_t)((uint64_t)V * w1 / WT);
            const uint32_t nv = pg.v_end - pg.v_begin;
            if (pg.ev.size() < n_launch) pg.ev.resize(n_launch);
            if (pg.cnt.size() < n_launch) pg.cnt.resize(n_launch);
            for (size_t L = 0; L < n_launch; L++) {
                pg.ev[L].clear();
                pg.cnt[L].assign(nv, 0);
            }
            pg.cursor.resize(nv);
            pg.next_due.resize(nv);
            for (uint32_t v = pg.v_begin; v < pg.v_end; v++) {
                const uint32_t c0 = vcount[voice_base[gi] + v], c1 = vcount[voice_base[gi] + v + 1];
                pg.cursor[v - pg.v_begin] = c0;
                // events of a voice are in ready-block order only after the first visit's sort: until then the skip test
                // must let every voice with events through (0), afterwards it is exact
                pg.next_due[v - pg.v_begin] = c0 == c1 ? UINT64_MAX : (identity ? pending[vo ? vo[c0] : c0].due_frame : 0);
            }
        }
    };
    pt.lap("contexts");
    if (T == 1) { // small jobs (block-by-block rendering): inline
        init_ctx(0);
        stream_worker(*this, *S, 0);
    } else {
        S->pooled = true;
        workers().start(T, [this, S, init_ctx](unsigned ti) {
            init_ctx(ti);
            stream_worker(*this, *S, ti);
        });
        if (driver_slice) init_ctx(T);
    }
}

// The calling thread's own slice (StreamState::driver_ctx), up to and including launch L
void HostPlan::driver_slice_through(size_t L) {
    StreamState *S = stream;
    if (S->driver_ctx < 0) return;
    StreamState::ThreadCtx &tc = *S->th[S->driver_ctx];
    while (S->driver_done <= L && S->driver_done < S->n_launch) {
        if (!tc.error_code) {
            try {
                stream_worker_step(*this, *S, tc, S->driver_done);
            } catch (const Error &e) {
                tc.error = e.msg;
                tc.error_code = e.code;
            }
        }
        S->driver_done++;
        tc.done.store((uint32_t)S->driver_done, std::memory_order_release);
    }
}

// Waits until every worker has finished launch L, then lays its events out per group: events in
// voice order + CSR offsets (n_voices + 1), pieces indexed by group.
void HostPlan::stream_launch(size_t L, CompiledEvents &out) {
    StreamState *S = stream;
    if (!S || !stream_active) KGPU_THROW(KGPU_ERR_STATE, "stream_launch without stream_begin");
    const size_t n_groups = groups.size();
    out.events.clear();
    out.offsets.clear();
    out.ext_used = false;
    out.ext_n_ev = out.ext_n_off = 0;
    out.piece_ev.assign(n_groups, 0);
    out.piece_off.assign(n_groups, 0);
    out.piece_any.assign(n_groups, 0);
    if (!S->any_work) return;
    PhaseTimer pt("stream_launch");
    driver_slice_through(L);
    pt.lap("own slice");
    for (unsigned ti = 0; ti < S->n_threads; ti++) {
        StreamState::ThreadCtx *tc = S->th[ti].get();
        // The driver thread has a core of its own (the pool leaves one free), and what it waits for is short: spin on the
        // counter for up to ~0.5 ms before sleeping.  A sleep_for(20 us) returns after 70-80 us (timer slack), which with
        // few workers per GPU -- where the driver does wait at every launch of the ramp -- left the device idle between launches.
        unsigned spins = 0;
        const auto t_wait = std::chrono::steady_clock::now();
        while (tc->done.load(std::memory_order_acquire) <= L) {
            if (++spins < 4096 || std::chrono::steady_clock::now() - t_wait < std::chrono::microseconds(500)) {
#if defined(__x86_64__) || defined(__i386__)
                __builtin_ia32_pause();
#else
                std::this_thread::yield();
#endif
            } else std::this_thread::sleep_for(std::chrono::microseconds(20));
        }
        if (tc->error_code) throw Error{tc->error_code, tc->error};
    }
    pt.lap("wait");
    // sizes first: the caller's buffers are used when the whole launch fits
    size_t all_ev = 0, all_off = 0;
    for (size_t gi = 0; gi < n_groups; gi++) {
        size_t total = 0;
        for (unsigned ti = 0; ti < S->n_threads; ti++) total += S->th[ti]->g[gi].ev[L].size();
        if (!total) continue;
        all_ev += total;
        all_off += groups[gi].n_voices + 1;
    }
    const bool ext = out.ext_ev && out.ext_off && all_ev <= out.ext_ev_cap && all_off <= out.ext_off_cap;
    if (ext) {
        out.ext_used = true;
        out.ext_n_ev = all_ev;
        out.ext_n_off = all_off;
    } else {
        out.events.resize(all_ev);
        out.offsets.resize(all_off);
    }
    DevEvent *ev_dst = ext ? out.ext_ev : out.events.data();
    uint32_t *off_dst = ext ? out.ext_off : out.offsets.data();
    size_t ev0 = 0, off0 = 0;
    for (size_t gi = 0; gi < n_groups; gi++) {
        size_t total = 0;
        for (unsigned ti = 0; ti < S->n_threads; ti++) total += S->th[ti]->g[gi].ev[L].size();
        out.piece_ev[gi] = ev0;
        if (!total) continue;
        out.piece_any[gi] = 1;
        out.piece_off[gi] = off0;
        uint32_t run_off = 0;
        uint32_t *off = off_dst + off0;
        for (unsigned ti = 0; ti < S->n_threads; ti++) {
            StreamState::PerGroup &pg = S->th[ti]->g[gi];
            if (!pg.ev[L].empty()) std::memcpy(ev_dst + ev0 + run_off, pg.ev[L].data(), pg.ev[L].size() * sizeof(DevEvent));
            for (uint32_t c : pg.cnt[L]) {
                *off++ = run_off;
                run_off += c;
            }
        }
        *off = run_off;
        ev0 += total;
        off0 += groups[gi].n_voices + 1;
    }
}

// drops the events the finished call consumed (due block < b1), keeping arrival order
void HostPlan::consume_ready(uint64_t b1) {
    const uint64_t bs = block_size;
    size_t w = 0;
    const uint64_t t_keep = b1 * bs; // due block >= b1, without a division per event
    for (size_t i = 0; i < pending.size(); i++)
        if (pending[i].due_frame >= t_keep) {
            if (w != i) pending[w] = pending[i];
            w++;
        }
    pending.resize(w);
    if (far_horizon != UINT64_MAX) pending_clean = w; // what is left was checked against the horizon by calendar_update
}

void HostPlan::stream_end() {
    StreamState *S = stream;
    if (!S || !stream_active) return;
    if (S->any_work) driver_slice_through(S->n_launch); // a call that ended early: the slice's state still advances over the whole range, like the workers'
    if (S->pooled) workers().wait();
#ifdef KGPU_PROFILE_HOST
    {
        uint64_t t[8] = {0};
        for (unsigned ti = 0; ti < S->n_threads; ti++)
            for (int i = 0; i < 8; i++) { t[i] += S->th[ti]->prof[i]; S->th[ti]->prof[i] = 0; }
        fprintf(stderr, "[prof] select %.1f gather %.1f nodes %.1f sort+append %.1f Mcycles (thread-summed)\n", t[0] / 1e6, t[1] / 1e6, t[2] / 1e6, t[3] / 1e6);
    }
#endif
    stream_active = false;
    if (!S->any_work) return;
    Error err{0, ""};
    for (unsigned ti = 0; ti < S->n_threads; ti++) {
        StreamState::ThreadCtx *tc = S->th[ti].get();
        dropped_changes += tc->sink.dropped;
        ignored_delays += tc->sink.ignored;
        device_events += tc->sink.devev;
        n_active_ramps = (uint64_t)((int64_t)n_active_ramps + tc->ramp_delta);
        if (tc->error_code && !err.code) err = Error{tc->error_code, tc->error};
    }
    if (S->all_ready && far_horizon == UINT64_MAX) pending.clear(); // nothing to keep: no pass over the queue
    else consume_ready(S->bounds.back() / block_size);
    if (err.code) throw err;
}

// whole range at once (kgpu_plan_prepare, debug entry points): pieces indexed [launch * n_groups + group]
void HostPlan::compile_events(const std::vector<uint64_t> &bounds, const std::vector<uint32_t> &chunk_of_group, CompiledEvents &out) {
    PhaseTimer pt("compile_events");
    const size_t n_launch = bounds.size() - 1, n_groups = groups.size();
    out.events.clear();
    out.offsets.clear();
    out.ext_used = false;
    out.ext_ev = nullptr;
    out.ext_off = nullptr;
    out.piece_ev.assign(n_launch * n_groups, 0);
    out.piece_off.assign(n_launch * n_groups, 0);
    out.piece_any.assign(n_launch * n_groups, 0);
    stream_begin(bounds, chunk_of_group);
    try {
        CompiledEvents one;
        for (size_t L = 0; L < n_launch; L++) {
            stream_launch(L, one);
            for (size_t gi = 0; gi < n_groups; gi++) {
                const size_t pi = L * n_groups + gi;
                out.piece_ev[pi] = out.events.size();
                if (!one.piece_any[gi]) continue;
                out.piece_any[pi] = 1;
                out.piece_off[pi] = out.offsets.size();
                const size_t ev_end = gi + 1 < n_groups ? one.piece_ev[gi + 1] : one.events.size();
                out.events.insert(out.events.end(), one.events.begin() + one.piece_ev[gi], one.events.begin() + ev_end);
                const size_t V1 = groups[gi].n_voices + 1;
                out.offsets.insert(out.offsets.end(), one.offsets.begin() + one.piece_off[gi], one.offsets.begin() + one.piece_off[gi] + V1);
            }
        }
    } catch (...) {
        stream_end();
        throw;
    }
    stream_end();
}

} // namespace kgpu
