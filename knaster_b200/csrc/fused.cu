// fused.cu -- register-resident bank kernels for known voice shapes.
//
// A voice template that matches one of the recipes below is rendered by a kernel in which the
// whole voice (every node of the template) lives in registers for the entire launch: no node
// buffer is ever materialised, per-voice state is read from HBM once at launch start and
// written once at launch end, and the only per-frame memory traffic is the mix-bus staging in
// shared memory.  One lane = one voice, evaluated strictly sequentially in the reference's
// rounding order (SURVEY F5: the f32 phase / envelope recurrences cannot be re-associated).
//
//   recipe 0  "render_sub_asr"   PolyBlep(saw) -> SvfFilter -> (* EnvAsr.wr_mul) [MathUGen<Mul>]   (configs[2], [4])
//   recipe 1  "render_fm2"       (SinNumeric * idx + fc) -> SinNumeric.ar_params() freq, * amp       (configs[3])
//   recipe 2  "render_add_wt"    SinWt[.wr_mul][.smooth_params] -> bus (fused_wt.cu)                     (configs[1])
//   recipe 3  "render_sub_seg"   recipe 0 with Envelope (f64 segments) in place of EnvAsr                (configs[2] variant B)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "dev.h"
#include "kernels.h"
#include "nodes.cuh"
#include "evcursor.cuh"
#include "plan.hpp"

namespace kgpu {

namespace {

constexpr int SUB_TILE = 32;          // frames between mix-bus reductions (render_fm2)
constexpr int SUB_PAD = 33;           // smem row stride (bank-conflict-free transpose)
constexpr int SUBW_PAD = 36;          // render_sub_asr: row stride that also keeps 16-byte row reads conflict-free

// register file of the subtractive voice (absolute register indices inside the voice, fixed by
// compile_template's allocation order: node 0 PolyBlep, node 1 Svf, node 2 EnvAsr + WrMul)
enum : uint32_t {
    R_T = 0, R_DT = 1, R_USESIN = 2, R_PW = 3, R_WF = 4,
    R_IC1 = 5, R_IC2 = 6, R_A1 = 7, R_A2 = 8, R_A3 = 9, R_M0 = 10, R_M1 = 11, R_M2 = 12,
    R_EST = 13, R_ET = 14, R_AR = 15, R_RR = 16, R_SC = 17, R_GAIN = 18, SUB_NREGS = 19,
};

// The voice minus its envelope: PolyBlep + SvfFilter registers; the envelope (and the WrMul gain that
// wraps it) is a policy, AsrEnv or SegEnv below.
template <class ENV> struct SubVoice {
    float t, dt;
    uint32_t use_sin;
    float pw;      // pulse_width and waveform: only the generic tick reads them (straight-line code = Sawtooth)
    uint32_t wf;
    float ic1, ic2, a1, a2, a3, m0, m1, m2;
    ENV e;
    KN_DEV void set_core(uint32_t reg, uint32_t bits) { // registers below R_EST
        const float f = __uint_as_float(bits);
        switch (reg) {
        case R_T: t = f; break;
        case R_DT: dt = f; break;
        case R_USESIN: use_sin = bits; break;
        case R_PW: pw = f; break;
        case R_WF: wf = bits; break;
        case R_IC1: ic1 = f; break;
        case R_IC2: ic2 = f; break;
        case R_A1: a1 = f; break;
        case R_A2: a2 = f; break;
        case R_A3: a3 = f; break;
        case R_M0: m0 = f; break;
        case R_M1: m1 = f; break;
        case R_M2: m2 = f; break;
        default: break;
        }
    }
    KN_DEV void set(uint32_t reg, uint32_t bits) {
        set_core(reg, bits);
        e.set(reg, bits); // two flat switches of plain assignments: ptxas turns both into selects
    }
    // reference-order evaluation, any parameter values (used on tiles with events / odd dt)
    KN_DEV float tick() {
        const float saw = polyblep_tick(t, dt, use_sin, pw, wf);
        const float y = svf_tick(saw, ic1, ic2, a1, a2, a3, m0, m1, m2);
        const float env = e.tick_ref(); // envelope * WrMul gain, wrappers_core/math.rs:63-67
        return y * env;                 // MathUGen<Mul>, math.rs:45-47
    }
    KN_DEV void idle() { // idle lane: a silent voice whose arithmetic stays finite (its output is +-0)
        t = 0.f; dt = 0.125f; use_sin = 0; pw = 0.5f; wf = 0;
        ic1 = ic2 = a1 = a2 = a3 = m0 = m1 = 0.f; m2 = 1.f;
        e.idle();
    }
};

// wrap01, div_prep, div_rc, saw_eval: csrc/nodes.cuh (shared with the interpreter's fast path)

#ifndef SUB_SUB
#define SUB_SUB 8 // frames per straight-line group (8, 16 or 32).  Measured, 16 384 voices x 10 s: 8 -> 13.65 ms, 16 -> 14.47 ms,
                  // 32 -> 14.85 ms: the 8-frame group (~300 instructions, 4.8 KB) stays in the instruction cache
#endif
#ifndef SUB_ROT
#define SUB_ROT 1     // rotated main loop: filter(group g) beside oscillator + envelope(group g + 1), see sub_produce / sub_consume
#endif
#ifndef SUB_F32X2
#define SUB_F32X2 0   // (measured: no gain) the frame-parallel half of a group (saw + blep, the envelope's products, the VCA) on packed f32x2
                      // instructions, two frames per instruction (nodes.cuh::saw_eval2): bit-identical, the 8-frame loop shrinks from 317 to 254
                      // instructions -- and takes 13.60 ms per step against 13.40 (16-frame groups: 13.43): a packed instruction holds the FMA pipe
                      // for two cycles, so the pipe sees the same 248 cycles per group either way; issue slots were not what the loop waits for
#endif
#ifndef SUB_SAT_RELEASE
#define SUB_SAT_RELEASE 1 // EnvAsr's Releasing -> Stopped transition inside the straight-line groups (saturating ramp steps, FADD.SAT: no extra
                          // instruction): one limit frame fewer per note, 13.60 -> 13.40 ms per step
#endif
#ifndef SUB_SAT_ATTACK
#define SUB_SAT_ATTACK 1  // EnvAsr's Attacking -> Sustaining transition inside the straight-line groups as well: the saturating ramp step leaves
                          // 1.0 where Sustaining outputs 1, and the first t >= 1 (which Sustaining keeps and t_restart resumes from) is replayed
                          // from a per-group checkpoint of the last ramp value below 1 when the next limit frame / the launch's end needs it
#endif
#ifndef SUB_PTRS
#define SUB_PTRS 0   // (measured: much slower, 15.86 ms per step against 13.33) rotated loop: staging / partial-row addresses carried as running values
                     // instead of rebuilt from `half` and `f` -- 314-316 instead of 319 instructions per group, still one basic block, but ptxas
                     // schedules the group differently (the previous group's staged rows are loaded and summed at the loop's head, the
                     // filter chain starts behind them): the instruction count is not what this loop is short of
#endif
#ifndef SUB_COMPACT
#define SUB_COMPACT 0 // (measured: slower, 14.7 ms against 14.1 -- an exact frame costs more than a 4- / 1-frame group) the frames between the last whole group and the limit frame run through ONE rolled exact-frame loop
                      // instead of 4- and 1-frame straight-line groups: a limit costs ~1900 cycles of mostly instruction
                      // fetch (r2a profile: 2.7 % of the instructions, 9.8 % of the time), so the path is kept small
#endif
#ifndef SUB_MINB
#define SUB_MINB 8 // __launch_bounds__ minimum CTAs per SM of the one-warp kernels (caps the registers per thread)
#endif
constexpr int SUBW_TILE = 2 * SUB_SUB; // render_sub_asr staging tile: two halves of SUB_SUB frames

// ---- envelope policies of the subtractive recipe ------------------------------------------------
// What a policy provides: the envelope's registers (loaded from / stored to the voice's register
// columns from R_EST on), `D` = what a straight-line group needs and is constant while the state
// machine does not move, group<N>() = N frames of `envelope * gain` with the state fixed,
// safe_frames() = how many coming frames provably stay in that state, exact1() = one frame with
// the whole state machine, and the event operations.

// EnvAsr.wr_mul: regs R_EST state, R_ET t, R_AR attack_rate, R_RR release_rate, R_SC release_scale, R_GAIN
struct AsrEnv {
    uint32_t est;
    float et, ar, rr, sc, gain;
    float tck; // SUB_SAT_ATTACK: the attack ramp's last group-end value below 1 (see group_ck / settle)
    // What a straight-line group needs, fixed while the state machine does not move.  The group is
    // select-free: every lane evaluates ((tl * u) * u) * sc2 with
    //   Releasing  tl = u = t (both step by -release_rate, so they stay equal), sc2 = release_scale:
    //              ((t * t) * t) * release_scale, the reference's t.powi(3) * release_scale;
    //   Attacking  u = 1 (step 0), sc2 = 1: ((t * 1) * 1) * 1 == t;
    //   Sustaining / Stopped  tl = 1 / 0 (step 0), u = 1, sc2 = 1: the constant itself.
    struct D {
        float delta;   // per-frame increment of t: +attack_rate, -release_rate or 0
        float du;      // per-frame increment of u: -release_rate or 0
        float sc2;     // release_scale while Releasing, else 1
        float cval;    // output of the constant states: Sustaining 1, Stopped 0
        bool att, rel;
    };
    KN_DEV void load(const FusedArgs &a, uint32_t v) {
        const uint32_t V = a.n_voices;
        uint32_t r[6];
#pragma unroll
        for (int i = 0; i < 6; i++) r[i] = a.regs[(size_t)(R_EST + i) * V + v];
#pragma unroll
        for (int i = 0; i < 6; i++) set(R_EST + i, r[i]);
        tck = et;
    }
    KN_DEV void idle() { est = ASR_STOPPED; et = 0.f; ar = rr = 1.f; sc = 0.f; gain = 0.f; tck = 0.f; }
    KN_DEV void set(uint32_t reg, uint32_t bits) {
        const float f = __uint_as_float(bits);
        switch (reg) {
        case R_EST: est = bits; break;
        case R_ET: et = f; break;
        case R_AR: ar = f; break;
        case R_RR: rr = f; break;
        case R_SC: sc = f; break;
        case R_GAIN: gain = f; break;
        default: break;
        }
    }
    KN_DEV void op(const DevEvent &e) {
        if (e.op == OP_ASR_RELEASE) envasr_release(est, et, sc);
    }
    KN_DEV void derive(D &d) {
        d.att = est == ASR_ATTACKING;
        d.rel = est == ASR_RELEASING;
        d.delta = d.att ? ar : (d.rel ? -rr : 0.0f);
        d.du = d.rel ? -rr : 0.0f;
        d.sc2 = d.rel ? sc : 1.0f;
        d.cval = est == ASR_SUSTAINING ? 1.0f : 0.0f;
#if SUB_SAT_ATTACK
        tck = et;
#endif
    }
    // Number of coming frames in which the envelope state machine provably cannot change state.
    // Attacking: t_n = t + n*ar + err with |err| <= n*2^-25 (one rounding of a value below 2 per add),
    // so the first tick whose sum can reach 1 is no earlier than (1-t)/(ar + 2^-25); the same bound
    // holds for the release ramp reaching 0.  The margin used here is twice that, minus one frame
    // (ticks 0 .. m-2 are safe when tick m-1 is the first that can cross).
    KN_DEV uint32_t safe_frames() const {
        const bool att = est == ASR_ATTACKING, rel = est == ASR_RELEASING;
        if (!att && !rel) return 0x40000000u;
        const float dist = att ? 1.0f - et : et;
        const float rate = (att ? ar : rr) + 5.9604644775390625e-8f;
        const float n = __fdividef(dist, rate) - 1.0f;
        return n >= 1.0f ? (uint32_t)fminf(n, 1073741824.0f) : 0u; // NaN -> 0: always the exact path
    }
    // The same bound for callers that render with group_ck(): the end of a release needs no limit there -- the groups step both
    // ramps with a saturating add, so a ramp that reaches <= 0 stays at +0, exactly what Stopped produces (t = 0, output 0;
    // envelopes.rs:71-76), and settle() names the state before it is read or stored.  Attack -> Sustaining (SUB_SAT_ATTACK): the
    // saturated ramp stays at 1.0, which is what Sustaining outputs; Sustaining keeps t at its first value >= 1 (t_restart
    // resumes from it, envelopes.rs:131-133), which settle() recomputes from the checkpoint group_ck() keeps.
    KN_DEV uint32_t safe_frames_group() const {
#if SUB_SAT_RELEASE
        if (est == ASR_RELEASING) return 0x40000000u;
#endif
#if SUB_SAT_ATTACK && SUB_SAT_RELEASE
        // an attack that has not reached 1 yet and does move towards it: group_ck() carries it through its end (ar > 0 is false for NaN)
        if (est == ASR_ATTACKING && et < 1.0f && ar > 0.0f) return 0x40000000u;
#endif
        return safe_frames();
    }
    // group() for the kernels that let an attack run through its end (render_sub_body): the ramp's value at the end of the group is
    // remembered while it is below 1, so that settle() finds the first value >= 1 within N additions
    template <int N> KN_DEV void group_ck(const D &d, float (&env)[N]) {
        group<N>(d, env);
#if SUB_SAT_ATTACK && SUB_SAT_RELEASE
        tck = et < 1.0f ? et : tck;
#endif
    }
    // EnvAsr::next_sample (envelopes.rs:52-81) with the state fixed over the group
    template <int N, bool SAT = true> KN_DEV void group(const D &d, float (&env)[N]) {
        const bool ramp = d.att || d.rel;
        float tl = ramp ? et : d.cval;
        float u = d.rel ? et : 1.0f;
#if SUB_F32X2
        if constexpr (N % 2 == 0) { // the two ramps stay scalar chains; the four products of a frame pair are packed
#pragma unroll
            for (int k = 0; k < N; k += 2) {
                const float tl1 = asr_step<SAT>(tl, d.delta), u1 = asr_step<SAT>(u, d.du);
                const float2 t2 = make_float2(tl, tl1), u2 = make_float2(u, u1);
                const float2 e2 = mul2(mul2(mul2(mul2(t2, u2), u2), dup2(d.sc2)), dup2(gain));
                env[k] = e2.x;
                env[k + 1] = e2.y;
                tl = asr_step<SAT>(tl1, d.delta);
                u = asr_step<SAT>(u1, d.du);
            }
            et = ramp ? tl : et;
            return;
        }
#endif
#pragma unroll
        for (int k = 0; k < N; k++) {
            const float o = ((tl * u) * u) * d.sc2;
            tl = asr_step<SAT>(tl, d.delta);
            u = asr_step<SAT>(u, d.du);
            env[k] = o * gain;      // WrMul, wrappers_core/math.rs:63-67
        }
        et = ramp ? tl : et;
    }
    // A ramp step of a straight-line group.  Inside a group every ramp value lies in [0, 1] (an attack's limit frame comes
    // before its sum can reach 1), so FADD.SAT only ever acts on a release that crosses 0: it leaves +0 where the
    // reference's Stopped state sets t = 0, and 0 - rate stays there.
    template <bool SAT> static KN_DEV float asr_step(float x, float dx) {
#if SUB_SAT_RELEASE
        if (SAT) return __saturatef(x + dx);
#endif
        return x + dx;
    }
    // Releasing with t at 0 is Stopped (a group may have carried the ramp through its end, see safe_frames)
    // ... and Attacking with t at 1 (the saturated ramp; a real attack leaves Attacking with its first t >= 1) is Sustaining with the
    // value the unsaturated ramp reaches first: at most SUB_SUB additions from the checkpoint.  Called where no event has been applied
    // since the last group, so Attacking with t >= 1 can only be the saturated ramp (t_restart on a sustaining envelope makes the same
    // pair, but the exact frame that follows the event resolves it at once).
    KN_DEV bool settle() { // true: the state's name changed, what derive() made of it is stale
        bool changed = false;
#if SUB_SAT_RELEASE
        if (est == ASR_RELEASING && et <= 0.0f) {
            est = ASR_STOPPED;
            et = 0.0f;
            changed = true;
        }
#if SUB_SAT_ATTACK
        if (est == ASR_ATTACKING && et >= 1.0f) {
            float t = tck;
#pragma unroll 1
            for (int i = 0; i < 32 && t < 1.0f; i++) t = t + ar;
            et = t;
            est = ASR_SUSTAINING;
            changed = true;
        }
#endif
#endif
        return changed;
    }
    // one frame, then EnvAsr's transitions (envelopes.rs:60-77): they only change what FOLLOWING frames do
    KN_DEV float exact1(const D &d) {
        float env[1];
        group<1, false>(d, env); // not saturating: an attack keeps its first t >= 1 (see safe_frames_group)
        if (d.att && et >= 1.0f) est = ASR_SUSTAINING;
        if (d.rel && et <= 0.0f) {
            est = ASR_STOPPED;
            et = 0.0f;
        }
        return env[0];
    }
    // EnvAsr::next_sample as straight-line selects: same values, no divergence
    KN_DEV float tick_sel() {
        const bool att = est == ASR_ATTACKING, rel = est == ASR_RELEASING;
        const float cube = ((et * et) * et) * sc;
        const float out = att ? et : (est == ASR_SUSTAINING ? 1.0f : (rel ? cube : 0.0f));
        float tn = att ? et + ar : (rel ? et - rr : et);
        const bool to_sus = att && tn >= 1.0f;
        const bool to_stop = rel && tn <= 0.0f;
        est = to_sus ? (uint32_t)ASR_SUSTAINING : (to_stop ? (uint32_t)ASR_STOPPED : est);
        et = to_stop ? 0.0f : tn;
        return out * gain;
    }
    KN_DEV float tick_ref() { return envasr_tick(est, et, ar, rr, sc) * gain; }
    KN_DEV void store(const FusedArgs &a, uint32_t v) const {
        const uint32_t V = a.n_voices;
        a.regs[(size_t)R_EST * V + v] = est;
        a.regs[(size_t)R_ET * V + v] = __float_as_uint(et);
        a.regs[(size_t)R_SC * V + v] = __float_as_uint(sc);
        a.regs[(size_t)R_AR * V + v] = __float_as_uint(ar);
        a.regs[(size_t)R_RR * V + v] = __float_as_uint(rr);
        a.regs[(size_t)R_GAIN * V + v] = __float_as_uint(gain);
    }
};

// Envelope.wr_mul (envelopes.rs:359-527): f64 segment envelope.  Registers from R_EST: +0 running,
// +1 segment, +2,3 time, +4,5 from_value, +6,7 step = time_scale * (1/sr), then per segment
// {reciprocal_duration, duration, value} (f64 each, never written by events), then the WrMul gain.
// The current segment's three numbers are cached in registers and re-read from the voice's register
// columns whenever the segment index changes (a few times per note).
struct SegEnv {
    uint32_t running, seg;
    double time, from, step;
    double recip, dur, val;       // segments[seg]
    float gain;
    uint32_t n_seg, looping, gain_reg;
    const uint32_t *segs;         // &regs[(R_EST + 8) * V + v]
    uint32_t V;
    struct D {
        double recip, diff, step; // 0, -0, 0 while stopped: from + (0*0)*(-0) == from, for every from
        bool run;
    };
    KN_DEV static double mk(uint32_t lo, uint32_t hi) { return __hiloint2double((int)hi, (int)lo); }
    KN_DEV void reload() {
        uint32_t r[6];
        const uint32_t sg = seg < n_seg ? seg : 0u;
#pragma unroll
        for (int i = 0; i < 6; i++) r[i] = __ldg(segs + (size_t)(REGS_ENVELOPE_PER_SEG * sg + i) * V);
        recip = mk(r[0], r[1]);
        dur = mk(r[2], r[3]);
        val = mk(r[4], r[5]);
    }
    KN_DEV void load(const FusedArgs &a, uint32_t v) {
        V = a.n_voices;
        n_seg = a.prog->nodes[2].n_seg;
        looping = a.prog->nodes[2].looping;
        gain_reg = R_EST + REGS_ENVELOPE_BASE + REGS_ENVELOPE_PER_SEG * n_seg;
        segs = a.regs + (size_t)(R_EST + REGS_ENVELOPE_BASE) * V + v;
        uint32_t r[8];
#pragma unroll
        for (int i = 0; i < 8; i++) r[i] = a.regs[(size_t)(R_EST + i) * V + v];
        running = r[0];
        seg = r[1];
        time = mk(r[2], r[3]);
        from = mk(r[4], r[5]);
        step = mk(r[6], r[7]);
        gain = __uint_as_float(a.regs[(size_t)gain_reg * V + v]);
        reload();
    }
    KN_DEV void idle() {
        running = seg = 0;
        time = from = step = recip = dur = val = 0.0;
        gain = 0.f;
        n_seg = 1; looping = 0; gain_reg = 0xFFFFFFFFu; segs = nullptr; V = 0;
    }
    KN_DEV void set(uint32_t reg, uint32_t bits) {
        if (reg == gain_reg) {
            gain = __uint_as_float(bits);
            return;
        }
        switch (reg - R_EST) {
        case 0: running = bits; break;
        case 1: seg = bits; reload(); break; // a t_stop later in the same frame reads the new segment
        case 2: time = mk(bits, (uint32_t)__double2hiint(time)); break;
        case 3: time = mk((uint32_t)__double2loint(time), bits); break;
        case 4: from = mk(bits, (uint32_t)__double2hiint(from)); break;
        case 5: from = mk((uint32_t)__double2loint(from), bits); break;
        case 6: step = mk(bits, (uint32_t)__double2hiint(step)); break;
        case 7: step = mk((uint32_t)__double2loint(step), bits); break;
        default: break;
        }
    }
    KN_DEV double level() const { // from_value + (t * reciprocal_duration) * (value - from_value), envelopes.rs:425-429
        return __dadd_rn(from, __dmul_rn(__dmul_rn(time, recip), __dsub_rn(val, from)));
    }
    KN_DEV void op(const DevEvent &e) {
        if (e.op == OP_ENV_STOP) {           // t_stop, envelopes.rs:511-523
            if (running) from = level();
            running = 0;
        } else if (e.op == OP_ENV_RESTART) { // t_restart, envelopes.rs:504-510; (reg, value) = from_value
            running = 1;
            time = 0.0;
            from = mk(e.reg, e.value);
            if (seg != 0) {
                seg = 0;
                reload();
            }
        } else if (e.op == OP_ENV_JUMP) {    // jump_to_segment, envelopes.rs:480-503
            running = 1;
            time = 0.0;
            if (seg != e.value) {
                seg = e.value;
                reload();
            }
        } else if (e.op == OP_ENV_STEP) {    // time_scale, envelopes.rs:477-479; (reg, value) = step
            step = mk(e.reg, e.value);
        }
    }
    KN_DEV void derive(D &d) const {
        d.run = running != 0;
        d.recip = d.run ? recip : 0.0;
        d.diff = d.run ? __dsub_rn(val, from) : -0.0;
        d.step = d.run ? step : 0.0;
    }
    // Leading frames that take the `t < duration` branch (envelopes.rs:423-433) for certain: the k-th
    // coming frame sees t_k = time + k*step up to k roundings of 2^-53 relative each, so the first
    // frame with t_k >= duration is no earlier than (duration - time)/step * (1 - 1e-6) - 1 for any
    // frame count below 2^30 (the f32 quotient itself is within 3e-7 of the exact one).
    KN_DEV uint32_t safe_frames() const {
        if (!running) return 0x40000000u;
        if (!(time < dur)) return 0u;
        if (!(step > 0.0)) return step <= 0.0 ? 0x40000000u : 0u; // time only falls / NaN: exact path
        const float n = __fdividef((float)__dsub_rn(dur, time), (float)step) * 0.999999f - 1.0f;
        return n >= 1.0f ? (uint32_t)fminf(n, 1073741824.0f) : 0u;
    }
    KN_DEV uint32_t safe_frames_group() const { return safe_frames(); }
    KN_DEV bool settle() { return false; }
    template <int N> KN_DEV void group_ck(const D &d, float (&env)[N]) { group<N>(d, env); }
    template <int N> KN_DEV void group(const D &d, float (&env)[N]) {
        double tl = d.run ? time : 0.0;
#pragma unroll
        for (int k = 0; k < N; k++) {
            const double y = __dadd_rn(from, __dmul_rn(__dmul_rn(tl, d.recip), d.diff));
            tl = __dadd_rn(tl, d.step);
            env[k] = (float)y * gain; // F::new(f64) rounds to nearest; WrMul, wrappers_core/math.rs:63-67
        }
        time = d.run ? tl : time;
    }
    // Envelope::process (envelopes.rs:407-463), the whole state machine
    KN_DEV float tick_ref() {
        float y;
        if (!running) {
            y = (float)from;
        } else if (time < dur) {
            y = (float)level();
            time = __dadd_rn(time, step);
        } else if (seg + 1 < n_seg) {
            from = val;
            y = (float)level();
            time = __dadd_rn(__dsub_rn(time, dur), step);
            seg = seg + 1;
            reload();
        } else {
            from = val;
            y = (float)from;
            if (looping) {
                seg = 0;
                time = 0.0;
                reload();
            } else {
                running = 0;
            }
        }
        return y * gain;
    }
    KN_DEV float tick_sel() { return tick_ref(); }
    KN_DEV float exact1(const D &) { return tick_ref(); }
    KN_DEV void store(const FusedArgs &a, uint32_t v) const {
        const uint32_t Vn = a.n_voices;
        const uint32_t r[8] = {running, seg, (uint32_t)__double2loint(time), (uint32_t)__double2hiint(time),
                               (uint32_t)__double2loint(from), (uint32_t)__double2hiint(from),
                               (uint32_t)__double2loint(step), (uint32_t)__double2hiint(step)};
#pragma unroll
        for (int i = 0; i < 8; i++) a.regs[(size_t)(R_EST + i) * Vn + v] = r[i];
        a.regs[(size_t)gain_reg * Vn + v] = __float_as_uint(gain);
    }
};

// Canonical mix-bus order for one frame: T(voices 0..15) + T(voices 16..31), T a fixed tree over
// four float4 reads.  Every path that sums a staged frame uses it, so a render is bit-identical
// however it is split into launches.
KN_DEV float sum16(const float *p) {
    const float4 *q = reinterpret_cast<const float4 *>(p);
    const float4 a = q[0], b = q[1], c = q[2], e = q[3];
    const float s0 = (a.x + a.y) + (a.z + a.w), s1 = (b.x + b.y) + (b.z + b.w);
    const float s2 = (c.x + c.y) + (c.z + c.w), s3 = (e.x + e.y) + (e.z + e.w);
    return (s0 + s1) + (s2 + s3);
}

// the first level of sum16's tree over 8 voices: (s0 + s1) of the canonical order
KN_DEV float sum8(const float *p) {
    const float4 *q = reinterpret_cast<const float4 *>(p);
    const float4 a = q[0], b = q[1];
    return ((a.x + a.y) + (a.z + a.w)) + ((b.x + b.y) + (b.z + b.w));
}

// N frames, no events, no envelope transition, fast conditions hold for every lane: the three
// recurrences (phase, envelope, filter) are independent dependency chains that ptxas interleaves
// in one basic block.  LP: m0 == 0, m1 == 0, m2 == 1 (lowpass) for every lane, where
// m0*v0 + m1*v1 + m2*v2 == v2 for finite signals.  Frame k goes to strow[k * SUBW_PAD] (the
// lane's column of the staging tile) and, when the voice is tapped, to tap[k].
// SUM: the same basic block also reduces the 16 frames staged by the PREVIOUS group (lane = (frame
// r = lane & 15, voice half c = lane >> 4)), so the mix-bus reduction costs issue slots only.
template <class ENV, bool LP, int N, bool TAPS, bool SUM, bool EXACT = false>
KN_DEV void sub_group_fast(SubVoice<ENV> &s, const typename ENV::D &d, float omd, float rc, float *strow, float *tap,
                           const float *sum_src = nullptr, float *sum_dst = nullptr, bool sum_store = false) {
    float ph[N], env[N];
    if (SUM) {
        float tot;
        if (N == 32) {        // lane = frame: all 32 voices
            tot = sum16(sum_src) + sum16(sum_src + 16);
        } else if (N == 16) { // lane = (frame, voice half)
            const float h = sum16(sum_src);
            tot = h + __shfl_xor_sync(0xFFFFFFFFu, h, 16);
        } else {              // N == 8: lane = (frame, voice quarter); same tree: ((q0 + q1) + (q2 + q3))
            const float q = sum8(sum_src);
            const float h = q + __shfl_xor_sync(0xFFFFFFFFu, q, 8);
            tot = h + __shfl_xor_sync(0xFFFFFFFFu, h, 16);
        }
        if (sum_store) *sum_dst = tot;
    }
#pragma unroll
    for (int k = 0; k < N; k++) {
        ph[k] = s.t;
        s.t = wrap01(s.t + s.dt); // inc(), polyblep.rs:232-235
    }
    if constexpr (EXACT) env[0] = s.e.exact1(d); // N == 1: the envelope's whole state machine
    else s.e.template group_ck<N>(d, env);        // envelope * WrMul gain with the state fixed over the group
#pragma unroll
    for (int k = 0; k < N; k++) {
        const float v0 = saw_eval(ph[k], s.dt, omd, rc);
        float y;
        if (LP) {                 // svf.rs:272-278; 2*v is exact, so fma(2,v,-ic) == 2*v - ic
            const float v3 = v0 - s.ic2;
            const float v1 = s.a1 * s.ic1 + s.a2 * v3;
            const float v2 = (s.ic2 + s.a2 * s.ic1) + s.a3 * v3;
            s.ic1 = __fmaf_rn(2.0f, v1, -s.ic1);
            s.ic2 = __fmaf_rn(2.0f, v2, -s.ic2);
            y = v2;
        } else {
            y = svf_tick(v0, s.ic1, s.ic2, s.a1, s.a2, s.a3, s.m0, s.m1, s.m2);
        }
        const float o = y * env[k]; // MathUGen<Mul>, math.rs:45-47
        strow[k * SUBW_PAD] = o;
        if (TAPS && tap) tap[k] = o;
    }
}

// The same group cut where no state crosses, for the rotated main loop (SUB_ROT): sub_produce advances the phase and the
// envelope by N frames and leaves the N saw samples and envelope gains in registers; sub_consume runs the filter, the VCA
// and the staging stores on them (and the previous group's mix-bus sum).  The loop body is consume(group g) followed by
// produce(group g + 1): the filter's dependency chain starts at the top of the basic block on operands that are already
// there, and the independent work of the next group fills its latency gaps up to the last instruction -- the one-piece
// group spent 8 % of its cycles waiting at its head (first saw sample) and tail (last filter steps, r2a profile).
template <class ENV, int N>
KN_DEV void sub_produce(SubVoice<ENV> &s, const typename ENV::D &d, float omd, float rc, float (&x)[N], float (&env)[N]) {
    float ph[N];
#pragma unroll
    for (int k = 0; k < N; k++) {
        ph[k] = s.t;
        s.t = wrap01(s.t + s.dt); // inc(), polyblep.rs:232-235
    }
    s.e.template group_ck<N>(d, env);
#if SUB_F32X2
    if constexpr (N % 2 == 0) {
#pragma unroll
        for (int k = 0; k < N; k += 2) {
            const float2 y = saw_eval2(make_float2(ph[k], ph[k + 1]), s.dt, omd, rc);
            x[k] = y.x;
            x[k + 1] = y.y;
        }
        return;
    }
#endif
#pragma unroll
    for (int k = 0; k < N; k++) x[k] = saw_eval(ph[k], s.dt, omd, rc);
}
template <class ENV, bool LP, int N, bool TAPS>
KN_DEV void sub_consume(SubVoice<ENV> &s, const float (&x)[N], const float (&env)[N], float *strow, float *tap,
                        const float *sum_src, float *sum_dst, bool sum_store) {
    float tot;
    if (N == 32) {
        tot = sum16(sum_src) + sum16(sum_src + 16);
    } else if (N == 16) {
        const float h = sum16(sum_src);
        tot = h + __shfl_xor_sync(0xFFFFFFFFu, h, 16);
    } else {
        const float q = sum8(sum_src);
        const float h = q + __shfl_xor_sync(0xFFFFFFFFu, q, 8);
        tot = h + __shfl_xor_sync(0xFFFFFFFFu, h, 16);
    }
#if SUB_PTRS
    // a predicated store, spelled out (no branch whatever ptxas makes of the running destination pointer)
    asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p st.global.f32 [%0], %1; }" ::"l"(sum_dst), "f"(tot), "r"((uint32_t)sum_store));
#else
    if (sum_store) *sum_dst = tot;
#endif
    float yy[N];
#pragma unroll
    for (int k = 0; k < N; k++) {
        const float v0 = x[k];
        float y;
        if (LP) {
            const float v3 = v0 - s.ic2;
            const float v1 = s.a1 * s.ic1 + s.a2 * v3;
            const float v2 = (s.ic2 + s.a2 * s.ic1) + s.a3 * v3;
            s.ic1 = __fmaf_rn(2.0f, v1, -s.ic1);
            s.ic2 = __fmaf_rn(2.0f, v2, -s.ic2);
            y = v2;
        } else {
            y = svf_tick(v0, s.ic1, s.ic2, s.a1, s.a2, s.a3, s.m0, s.m1, s.m2);
        }
        yy[k] = y;
#if SUB_F32X2
        if (N % 2 == 0 && (k & 1)) { // the VCA of a frame pair as one packed multiplication
            const float2 o2 = mul2(make_float2(yy[k - 1], y), make_float2(env[k - 1], env[k]));
            strow[(k - 1) * SUBW_PAD] = o2.x;
            strow[k * SUBW_PAD] = o2.y;
            if (TAPS && tap) { tap[k - 1] = o2.x; tap[k] = o2.y; }
        }
        if (N % 2 == 0) continue;
#endif
        const float o = y * env[k];
        strow[k * SUBW_PAD] = o;
        if (TAPS && tap) tap[k] = o;
    }
}

// per-lane validity of the straight-line formulation
template <class ENV> KN_DEV bool sub_lane_fast(const SubVoice<ENV> &s) {
    return s.dt >= 9.5367431640625e-7f && s.dt < 0.25f && s.t >= 0.0f && s.t < 1.0f && !s.use_sin && s.wf == 0u;
}
template <class ENV> KN_DEV bool sub_lane_lp(const SubVoice<ENV> &s) { return s.m0 == 0.0f && s.m1 == 0.0f && s.m2 == 1.0f; }

#include "fused_scan.cuh" // recipe 4 "render_sub_scan": the same voice, one warp per voice, for small banks

// The body of render_sub_asr / render_sub_seg: ENV = AsrEnv or SegEnv.
template <class ENV, bool TAPS>
KN_DEV void render_sub_body(const FusedArgs &a, float *st) {
    const uint32_t lane = threadIdx.x;
    const uint32_t gwarp = blockIdx.x;
    const uint32_t v = gwarp * 32 + lane;
    const uint32_t V = a.n_voices;
    const bool active = v < V;

    SubVoice<ENV> s;
    if (active) {
        uint32_t r[R_EST];
#pragma unroll
        for (int i = 0; i < R_EST; i++) r[i] = a.regs[(size_t)i * V + v];
#pragma unroll
        for (int i = 0; i < R_EST; i++) s.set_core(i, r[i]); // not set(): the envelope is not loaded yet (SegEnv::set reads gain_reg)
        s.e.load(a, v);
    } else {
        s.idle();
    }
    EvCursor ec;
    ec.init(a.events, a.ev_off, v, active);
    int tap_row = -1;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (active && a.taps[i].voice == v) tap_row = (int)a.taps[i].tap;
    float *tap = TAPS && tap_row >= 0 ? a.tap_out + (size_t)tap_row * a.tap_stride + a.tap_frame0 : nullptr;

    float *prow = a.partials + (size_t)(a.row0 + gwarp) * a.n_frames;
    // the straight-line group needs t in [0,1), 2^-20 <= dt < 1/4 and the sawtooth branch of next_sample
    bool lane_fast = sub_lane_fast(s);
    bool all_lp = __all_sync(0xFFFFFFFFu, sub_lane_lp(s));
    float omd = 1.0f - s.dt, rc = div_prep(s.dt);
    typename ENV::D d;
    s.e.derive(d);
    // `limit`: first frame at which SOME lane needs the exact per-frame path (an event is due, its
    // envelope may change state, or its parameters are outside the fast domain).  Warp-uniform.
    auto lane_limit = [&](uint32_t f) -> uint32_t {
        if (!lane_fast) return 0u;
        const uint32_t safe = f + s.e.safe_frames_group();
        return min(ec.next_frame, safe);
    };
    uint32_t limit = __reduce_min_sync(0xFFFFFFFFu, lane_limit(0));
    bool all_fast = __all_sync(0xFFFFFFFFu, lane_fast);

    uint32_t NF = a.n_frames;
    asm volatile("" : "+r"(NF)); // keep it in a register (ptxas would re-read the constant bank in every loop test)
    uint32_t next_ev = __reduce_min_sync(0xFFFFFFFFu, ec.next_frame);
    uint32_t f = 0;      // next frame to render
    // frames staged in st[] since the last flush: rows [rbase, rbase + rows), frame f - rows first
    uint32_t rows = 0, rbase = 0;
    // lane l sums staged frame l over the warp's 32 voices
    auto flush = [&]() {
        __syncwarp();
        const float *row = st + (rbase + (lane < rows ? lane : 0u)) * SUBW_PAD;
        const float tot = sum16(row) + sum16(row + 16);
        if (lane < rows) prow[f - rows + lane] = tot;
        rows = 0;
        rbase = 0;
        __syncwarp();
    };
    auto stage_room = [&](uint32_t n) {
        if (rows + n > 32 || rbase + rows + n > SUBW_TILE) flush(); // flush() sums one staged frame per lane
    };
    // straight-line groups of N frames while N frames are safe
    auto run_groups = [&](auto lp_tag, auto n_tag, uint32_t lim) {
        constexpr bool LP = decltype(lp_tag)::value;
        constexpr int N = decltype(n_tag)::value;
#pragma unroll 1
        while (f + N <= lim) {
            stage_room(N);
            sub_group_fast<ENV, LP, N, TAPS, false>(s, d, omd, rc, st + (rbase + rows) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr);
            rows += N;
            f += N;
        }
    };
    auto run_fast = [&](auto lp_tag, uint32_t lim) {
        constexpr bool LP = decltype(lp_tag)::value;
        if (f + SUB_SUB <= lim) {
            // 16-frame groups ping-pong between the two halves of the tile; each group also sums the
            // half the previous one staged (the first finds nothing pending and stores nothing)
            if (rows) flush();
            uint32_t half = 0;
            bool pending = false;
            // lane = (staged frame r, voice group c of 32 / (32 / SUB_SUB) voices)
            const uint32_t r = lane & (SUB_SUB - 1u), c = lane / SUB_SUB, cw = SUB_SUB == 32 ? 32u : (SUB_SUB == 16 ? 16u : 8u);
#if SUB_ROT && SUB_PTRS
            // the staging addresses as running values: the write column and the read row swap halves by "sum minus itself" (one
            // integer addition each), the destination of the sums advances by a group -- the loop spent 14 instructions per
            // iteration rebuilding the three from `half` and `f`
            constexpr uint32_t TOG = SUB_SUB * SUBW_PAD;
            const uint32_t ro0 = r * SUBW_PAD + c * cw;
            uint32_t wo = lane, ro = TOG + ro0;
            const uint32_t wsum = 2u * lane + TOG, rsum = 2u * ro0 + TOG;
            float *pd = prow + ((ptrdiff_t)f - (ptrdiff_t)SUB_SUB + (ptrdiff_t)r); // never stored to before a group is pending
            float gx[SUB_SUB], ge[SUB_SUB];
            sub_produce<ENV, SUB_SUB>(s, d, omd, rc, gx, ge);      // the group at f; the oscillator / envelope state is now at f + SUB_SUB
#pragma unroll 1
            while (f + 2 * SUB_SUB <= lim) {
                __syncwarp();
                sub_consume<ENV, LP, SUB_SUB, TAPS>(s, gx, ge, st + wo, TAPS && tap ? tap + f : nullptr, st + ro, pd, pending && c == 0);
                sub_produce<ENV, SUB_SUB>(s, d, omd, rc, gx, ge);
                pending = true;
                wo = wsum - wo;
                ro = rsum - ro;
                pd += SUB_SUB;
                f += SUB_SUB;
            }
            __syncwarp();
            sub_consume<ENV, LP, SUB_SUB, TAPS>(s, gx, ge, st + wo, TAPS && tap ? tap + f : nullptr, st + ro, pd, pending && c == 0);
            half = wo >= TOG ? 0u : 1u; // as if toggled after the last group: the group just staged sits in half ^ 1
            f += SUB_SUB;
#elif SUB_ROT
            float gx[SUB_SUB], ge[SUB_SUB];
            sub_produce<ENV, SUB_SUB>(s, d, omd, rc, gx, ge);      // the group at f; the oscillator / envelope state is now at f + SUB_SUB
#pragma unroll 1
            while (f + 2 * SUB_SUB <= lim) {
                __syncwarp();
                sub_consume<ENV, LP, SUB_SUB, TAPS>(s, gx, ge, st + (half * SUB_SUB) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr,
                                                    st + ((half ^ 1u) * SUB_SUB + r) * SUBW_PAD + c * cw, prow + (f - SUB_SUB + r), pending && c == 0);
                sub_produce<ENV, SUB_SUB>(s, d, omd, rc, gx, ge);
                pending = true;
                half ^= 1u;
                f += SUB_SUB;
            }
            __syncwarp();
            sub_consume<ENV, LP, SUB_SUB, TAPS>(s, gx, ge, st + (half * SUB_SUB) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr,
                                                st + ((half ^ 1u) * SUB_SUB + r) * SUBW_PAD + c * cw, prow + (f - SUB_SUB + r), pending && c == 0);
            half ^= 1u;
            f += SUB_SUB;
#else
#pragma unroll 1
            do {
                __syncwarp();
                sub_group_fast<ENV, LP, SUB_SUB, TAPS, true>(s, d, omd, rc, st + (half * SUB_SUB) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr,
                                                             st + ((half ^ 1u) * SUB_SUB + r) * SUBW_PAD + c * cw, prow + (f - SUB_SUB + r),
                                                             pending && c == 0);
                pending = true;
                half ^= 1u;
                f += SUB_SUB;
            } while (f + SUB_SUB <= lim);
#endif
            rbase = (half ^ 1u) * SUB_SUB;
            rows = SUB_SUB;
        }
#if !SUB_COMPACT
        run_groups(lp_tag, std::integral_constant<int, 4>{}, lim);
        run_groups(lp_tag, std::integral_constant<int, 1>{}, lim);
#endif
    };
    for (;;) {
        const uint32_t lim = min(limit, NF);
        if (all_lp) run_fast(std::true_type{}, lim);
        else run_fast(std::false_type{}, lim);
        if (f >= NF) break;
        // frame `limit`: events are applied, then the frame runs with the envelope state machine checked.  (SUB_COMPACT: the
        // frames between the last whole group and `limit` come through here as well -- nothing is due in them and the
        // envelope cannot move, the exact frame is simply the general one -- and keep `limit` as it is.)
        const bool at_limit = f >= limit;
        if (s.e.settle()) s.e.derive(d); // a ramp the groups carried through its end gets its state's name (and an attack its exact t) before anything reads it
        if (f >= next_ev) {
            bool touched = false;
            while (ec.next_frame <= f) { // events are sorted by (frame, node, arrival)
                if (ec.e0.op == OP_SET) s.set(ec.e0.reg, ec.e0.value);
                else s.e.op(ec.e0);
                ec.pop();
                touched = true;
            }
            if (touched) {
                omd = 1.0f - s.dt;
                rc = div_prep(s.dt);
                lane_fast = sub_lane_fast(s);
                s.e.derive(d);
            }
            all_lp = __all_sync(0xFFFFFFFFu, sub_lane_lp(s));
            all_fast = __all_sync(0xFFFFFFFFu, lane_fast);
            next_ev = __reduce_min_sync(0xFFFFFFFFu, ec.next_frame);
        }
        stage_room(1);
        float *strow = st + (rbase + rows) * SUBW_PAD + lane;
        if (all_fast) {
            // the straight-line frame with the envelope's state machine checked (ENV::exact1)
            if (all_lp) sub_group_fast<ENV, true, 1, TAPS, false, true>(s, d, omd, rc, strow, TAPS && tap ? tap + f : nullptr);
            else sub_group_fast<ENV, false, 1, TAPS, false, true>(s, d, omd, rc, strow, TAPS && tap ? tap + f : nullptr);
        } else {
            float o;
            if (lane_fast) {
                const float ph = s.t;
                s.t = wrap01(s.t + s.dt);
                const float e = s.e.tick_sel();
                o = svf_tick(saw_eval(ph, s.dt, omd, rc), s.ic1, s.ic2, s.a1, s.a2, s.a3, s.m0, s.m1, s.m2) * e;
            } else {
                o = s.tick();
                lane_fast = sub_lane_fast(s); // t is back in [0,1) after one generic tick
            }
            all_fast = __all_sync(0xFFFFFFFFu, lane_fast);
            *strow = o;
            if (TAPS && tap) tap[f] = o;
        }
        rows += 1;
        f += 1;
        if (at_limit) {
            s.e.derive(d);
            limit = __reduce_min_sync(0xFFFFFFFFu, lane_limit(f));
        }
    }
    if (rows) flush();
    if (active) {
        a.regs[(size_t)R_T * V + v] = __float_as_uint(s.t);
        a.regs[(size_t)R_IC1 * V + v] = __float_as_uint(s.ic1);
        a.regs[(size_t)R_IC2 * V + v] = __float_as_uint(s.ic2);
        // parameter registers change only through events: write them back as well
        a.regs[(size_t)R_DT * V + v] = __float_as_uint(s.dt);
        a.regs[(size_t)R_USESIN * V + v] = s.use_sin;
        a.regs[(size_t)R_PW * V + v] = __float_as_uint(s.pw);
        a.regs[(size_t)R_WF * V + v] = s.wf;
        a.regs[(size_t)R_A1 * V + v] = __float_as_uint(s.a1);
        a.regs[(size_t)R_A2 * V + v] = __float_as_uint(s.a2);
        a.regs[(size_t)R_A3 * V + v] = __float_as_uint(s.a3);
        a.regs[(size_t)R_M0 * V + v] = __float_as_uint(s.m0);
        a.regs[(size_t)R_M1 * V + v] = __float_as_uint(s.m1);
        a.regs[(size_t)R_M2 * V + v] = __float_as_uint(s.m2);
        s.e.settle();
        s.e.store(a, v);
    }
}

template <bool TAPS>
__global__ void __launch_bounds__(32, SUB_MINB) render_sub_asr(FusedArgs a) {
    __shared__ __align__(16) float st[SUBW_TILE * SUBW_PAD];
    render_sub_body<AsrEnv, TAPS>(a, st);
}

// recipe 3: the same voice with Envelope (f64 linear segments) in place of EnvAsr -- configs[2]
// variant B (SURVEY section 8d).  The envelope's 4 f64 operations per frame run on the FP64 pipe
// beside the FP32 work; its state machine only moves at segment boundaries (SegEnv::safe_frames).
template <bool TAPS>
__global__ void __launch_bounds__(32, 8) render_sub_seg(FusedArgs a) {
    __shared__ __align__(16) float st[SUBW_TILE * SUBW_PAD];
    render_sub_body<SegEnv, TAPS>(a, st);
}

// ------------------------------------------------------------------------------------------------
// "render_sub_asr2": the same recipe as TWO cooperating warps per 32 voices.  EXPERIMENT, not the
// default (see launch_fused): parity-identical, but measured slower than the one-warp kernel -- the
// filter warp is left with little more than the serial filter recurrence (17 cycles per frame of
// dependent latency for 21 instructions) plus the per-group hand-over, and the osc warp idles at
// the EMPTY barrier; the one-warp kernel hides that recurrence behind the saw arithmetic instead.
//
// One warp per 32 voices leaves every SM sub-partition with a single warp: nothing hides the idle
// cycles at the head and tail of each straight-line group (profiles/README.md).  Here the voice is
// cut where no state crosses: the OSC warp owns the phase recurrence and evaluates saw + blep
// (19 instructions per frame), the FILTER warp owns envelope, filter, VCA and the mix-bus
// reduction (21 per frame).  The saw signal travels through a shared-memory ring of 4 chunks x
// 16 frames, handed over with named barriers (FULL[c]: osc arrives / filter syncs; EMPTY[c]:
// filter arrives / osc syncs), so the osc warp runs up to 64 frames ahead and neither warp ever
// waits in the steady state.  CTAs are placed on consecutive warp slots (measured,
// tools/microbench/warp_slots.cu), so swapping the roles with bit 2 of the hardware warp slot gives
// every sub-partition one osc and one filter warp: two independent instruction streams per
// scheduler and the same 40 instructions per frame on each.
// Each warp walks the voice's event list with its own cursor and skips the other role's events.
#ifndef W2_GROUP
#define W2_GROUP 32 // frames per straight-line group of both warps = frames per ring chunk (16 or 32)
#endif
constexpr int RING_CHUNK = W2_GROUP, RING_CHUNKS = 4, RING_FRAMES = RING_CHUNK * RING_CHUNKS;
constexpr int W2_TILE = 2 * W2_GROUP; // the filter warp's staging tile: two halves of W2_GROUP frames
constexpr uint32_t BAR_FULL = 1, BAR_EMPTY = 1 + RING_CHUNKS;
KN_DEV void bar_sync(uint32_t id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
KN_DEV void bar_arrive(uint32_t id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }

KN_DEV bool ev_is_osc(const DevEvent &e) { return e.op == OP_SET && e.reg <= R_WF; }
template <bool OSC> KN_DEV void cursor_skip(EvCursor &ec) {
    while (ec.next_frame != 0xFFFFFFFFu && ev_is_osc(ec.e0) != OSC) ec.pop();
}
KN_DEV bool osc_lane_fast(float t, float dt, uint32_t use_sin, uint32_t wf) {
    return dt >= 9.5367431640625e-7f && dt < 0.25f && t >= 0.0f && t < 1.0f && !use_sin && wf == 0u;
}

template <int N> KN_DEV void osc_group(float &t, float dt, float omd, float rc, float *dst) {
    float ph[N];
#pragma unroll
    for (int k = 0; k < N; k++) {
        ph[k] = t;
        t = wrap01(t + dt); // inc(), polyblep.rs:232-235
    }
#pragma unroll
    for (int k = 0; k < N; k++) dst[k * 32] = saw_eval(ph[k], dt, omd, rc);
}

KN_DEV void sub2_osc_role(const FusedArgs &a, float *ring, uint32_t lane, uint32_t v, bool active) {
    const uint32_t V = a.n_voices;
    float t = 0.f, dt = 0.125f, pw = 0.5f;
    uint32_t use_sin = 0, wf = 0;
    if (active) {
        t = __uint_as_float(a.regs[(size_t)R_T * V + v]);
        dt = __uint_as_float(a.regs[(size_t)R_DT * V + v]);
        use_sin = a.regs[(size_t)R_USESIN * V + v];
        pw = __uint_as_float(a.regs[(size_t)R_PW * V + v]);
        wf = a.regs[(size_t)R_WF * V + v];
    }
    EvCursor ec;
    ec.init(a.events, a.ev_off, v, active);
    cursor_skip<true>(ec);
    bool lane_fast = osc_lane_fast(t, dt, use_sin, wf);
    bool all_fast = __all_sync(0xFFFFFFFFu, lane_fast);
    float omd = 1.0f - dt, rc = div_prep(dt);
    uint32_t next_ev = __reduce_min_sync(0xFFFFFFFFu, ec.next_frame);
    uint32_t NF = a.n_frames;
    asm volatile("" : "+r"(NF));
    const uint32_t n_chunks = (NF + RING_CHUNK - 1) / RING_CHUNK;
#pragma unroll 1
    for (uint32_t c = 0; c < n_chunks; c++) {
        const uint32_t slot = c & (RING_CHUNKS - 1);
        if (c >= RING_CHUNKS) bar_sync(BAR_EMPTY + slot); // the filter warp is done with this slot
        const uint32_t f0 = c * RING_CHUNK, f1 = min(f0 + RING_CHUNK, NF);
        float *row0 = ring + slot * RING_CHUNK * 32 + lane;
        if (all_fast && next_ev >= f1 && f1 - f0 == RING_CHUNK) {
            osc_group<RING_CHUNK>(t, dt, omd, rc, row0);
        } else {
#pragma unroll 1
            for (uint32_t f = f0; f < f1; f++) {
                if (f >= next_ev) {
                    bool touched = false;
                    while (ec.next_frame <= f) { // this role's events only (cursor_skip)
                        const float val = __uint_as_float(ec.e0.value);
                        if (ec.e0.reg == R_T) t = val;
                        else if (ec.e0.reg == R_DT) dt = val;
                        else if (ec.e0.reg == R_USESIN) use_sin = ec.e0.value;
                        else if (ec.e0.reg == R_PW) pw = val;
                        else if (ec.e0.reg == R_WF) wf = ec.e0.value;
                        ec.pop();
                        cursor_skip<true>(ec);
                        touched = true;
                    }
                    if (touched) {
                        omd = 1.0f - dt;
                        rc = div_prep(dt);
                        lane_fast = osc_lane_fast(t, dt, use_sin, wf);
                    }
                    all_fast = __all_sync(0xFFFFFFFFu, lane_fast);
                    next_ev = __reduce_min_sync(0xFFFFFFFFu, ec.next_frame);
                }
                float *dst = row0 + (f - f0) * 32;
                if (all_fast) {
                    osc_group<1>(t, dt, omd, rc, dst);
                } else {
                    float y;
                    if (lane_fast) {
                        const float ph = t;
                        t = wrap01(t + dt);
                        y = saw_eval(ph, dt, omd, rc);
                    } else {
                        y = polyblep_tick(t, dt, use_sin, pw, wf);
                        lane_fast = osc_lane_fast(t, dt, use_sin, wf); // t is back in [0,1) after one generic tick
                    }
                    *dst = y;
                    all_fast = __all_sync(0xFFFFFFFFu, lane_fast);
                }
            }
        }
        bar_arrive(BAR_FULL + slot);
    }
    if (active) {
        a.regs[(size_t)R_T * V + v] = __float_as_uint(t);
        a.regs[(size_t)R_DT * V + v] = __float_as_uint(dt);
        a.regs[(size_t)R_USESIN * V + v] = use_sin;
        a.regs[(size_t)R_PW * V + v] = __float_as_uint(pw);
        a.regs[(size_t)R_WF * V + v] = wf;
    }
}

// the filter warp's straight-line group: envelope + filter + VCA on saw frames read from the ring
template <bool LP, int N, bool TAPS, bool SUM>
KN_DEV void filt_group_fast(SubVoice<AsrEnv> &s, const AsrEnv::D &d, const float *v0src, float *strow, float *tap,
                            const float *sum_src = nullptr, float *sum_dst = nullptr, bool sum_store = false) {
    float env[N], saw[N];
    // all shared-memory reads first: the compiler cannot move a ring load above a staging store
#pragma unroll
    for (int k = 0; k < N; k++) saw[k] = v0src[k * 32];
    if (SUM) {
        float tot;
        if (N == 32) { // lane = frame: all 32 voices
            tot = sum16(sum_src) + sum16(sum_src + 16);
        } else {       // N == 16: lane = (frame, voice half)
            const float h = sum16(sum_src);
            tot = h + __shfl_xor_sync(0xFFFFFFFFu, h, 16);
        }
        if (sum_store) *sum_dst = tot;
    }
#pragma unroll
    for (int k = 0; k < N; k++) {
        // EnvAsr::next_sample (envelopes.rs:52-81) with the state fixed over the group
        const float cube = ((s.e.et * s.e.et) * s.e.et) * s.e.sc;
        const float o = d.att ? s.e.et : (d.rel ? cube : d.cval);
        s.e.et = s.e.et + d.delta;
        env[k] = o * s.e.gain;      // WrMul, wrappers_core/math.rs:63-67
    }
#pragma unroll
    for (int k = 0; k < N; k++) {
        const float v0 = saw[k];
        float y;
        if (LP) {                 // svf.rs:272-278; 2*v is exact, so fma(2,v,-ic) == 2*v - ic
            const float v3 = v0 - s.ic2;
            const float v1 = s.a1 * s.ic1 + s.a2 * v3;
            const float v2 = (s.ic2 + s.a2 * s.ic1) + s.a3 * v3;
            s.ic1 = __fmaf_rn(2.0f, v1, -s.ic1);
            s.ic2 = __fmaf_rn(2.0f, v2, -s.ic2);
            y = v2;
        } else {
            y = svf_tick(v0, s.ic1, s.ic2, s.a1, s.a2, s.a3, s.m0, s.m1, s.m2);
        }
        const float o = y * env[k]; // MathUGen<Mul>, math.rs:45-47
        strow[k * SUBW_PAD] = o;
        if (TAPS && tap) tap[k] = o;
    }
}

template <bool TAPS>
KN_DEV void sub2_filter_role(const FusedArgs &a, const float *ring, float *st, uint32_t lane, uint32_t v, bool active) {
    const uint32_t V = a.n_voices;
    const uint32_t gwarp = blockIdx.x;
    SubVoice<AsrEnv> s;
    s.t = 0.f; s.dt = 0.125f; s.use_sin = 0; // the osc warp's registers: unused here
    if (active) {
#pragma unroll
        for (int i = R_IC1; i < SUB_NREGS; i++) s.set(i, a.regs[(size_t)i * V + v]);
    } else { // idle lane: a silent voice whose arithmetic stays finite (its output is +-0)
        s.ic1 = s.ic2 = s.a1 = s.a2 = s.a3 = s.m0 = s.m1 = 0.f; s.m2 = 1.f;
        s.e.est = ASR_STOPPED; s.e.et = 0.f; s.e.ar = s.e.rr = 1.f; s.e.sc = 0.f; s.e.gain = 0.f;
    }
    EvCursor ec;
    ec.init(a.events, a.ev_off, v, active);
    cursor_skip<false>(ec);
    int tap_row = -1;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (active && a.taps[i].voice == v) tap_row = (int)a.taps[i].tap;
    float *tap = TAPS && tap_row >= 0 ? a.tap_out + (size_t)tap_row * a.tap_stride + a.tap_frame0 : nullptr;
    float *prow = a.partials + (size_t)(a.row0 + gwarp) * a.n_frames;

    bool all_lp = __all_sync(0xFFFFFFFFu, sub_lane_lp(s));
    AsrEnv::D d;
    s.e.derive(d);
    // `limit`: first frame at which SOME lane has an event due or may change envelope state
    auto lane_limit = [&](uint32_t f) -> uint32_t {
        const uint32_t safe = f + s.e.safe_frames();
        return min(ec.next_frame, safe);
    };
    uint32_t limit = __reduce_min_sync(0xFFFFFFFFu, lane_limit(0));
    uint32_t next_ev = __reduce_min_sync(0xFFFFFFFFu, ec.next_frame);
    uint32_t NF = a.n_frames;
    asm volatile("" : "+r"(NF));
    const uint32_t n_chunks = (NF + RING_CHUNK - 1) / RING_CHUNK;
    uint32_t f = 0;                 // next frame to render
    uint32_t have = 0, freed = 0;   // ring chunks acquired from / handed back to the osc warp
    auto need = [&](uint32_t fend) {
        while (have * RING_CHUNK < fend) {
            bar_sync(BAR_FULL + (have & (RING_CHUNKS - 1)));
            have++;
        }
    };
    auto release = [&]() {
        while ((freed + 1) * RING_CHUNK <= f) {
            if (freed + RING_CHUNKS < n_chunks) bar_arrive(BAR_EMPTY + (freed & (RING_CHUNKS - 1)));
            freed++;
        }
    };
    // frames staged in st[] since the last flush: rows [rbase, rbase + rows), frame f - rows first
    uint32_t rows = 0, rbase = 0;
    auto flush = [&]() { // lane l sums staged frame l over the warp's 32 voices
        __syncwarp();
        const float *row = st + (rbase + (lane < rows ? lane : 0u)) * SUBW_PAD;
        const float tot = sum16(row) + sum16(row + 16);
        if (lane < rows) prow[f - rows + lane] = tot;
        rows = 0;
        rbase = 0;
        __syncwarp();
    };
    auto stage_room = [&](uint32_t n) {
        if (rows + n > 32 || rbase + rows + n > W2_TILE) flush();
    };
    auto ring_at = [&](uint32_t frame) { return ring + (frame & (RING_FRAMES - 1)) * 32 + lane; };
    auto run_fast = [&](auto lp_tag, uint32_t lim) {
        constexpr bool LP = decltype(lp_tag)::value;
        for (;;) {
            const uint32_t pos = f & (RING_FRAMES - 1);
            if (f + W2_GROUP <= lim && pos + W2_GROUP <= RING_FRAMES) {
                // 16-frame groups ping-pong between the two halves of the tile; each group also sums
                // the half the previous one staged (the first finds nothing pending and stores nothing)
                if (rows) flush();
                uint32_t half = 0;
                bool pending = false;
                const uint32_t r = W2_GROUP == 32 ? lane : (lane & 15u), c = W2_GROUP == 32 ? 0u : (lane >> 4);
#pragma unroll 1
                do {
                    need(f + W2_GROUP);
                    __syncwarp();
                    filt_group_fast<LP, W2_GROUP, TAPS, true>(s, d, ring_at(f), st + (half * W2_GROUP) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr,
                                                             st + ((half ^ 1u) * W2_GROUP + r) * SUBW_PAD + c * 16, prow + (f - W2_GROUP + r),
                                                             pending && c == 0);
                    pending = true;
                    half ^= 1u;
                    f += W2_GROUP;
                    release();
                } while (f + W2_GROUP <= lim && (f & (RING_FRAMES - 1)) + W2_GROUP <= RING_FRAMES);
                rbase = (half ^ 1u) * W2_GROUP;
                rows = W2_GROUP;
            } else if (f + 4 <= lim && pos + 4 <= RING_FRAMES) {
                stage_room(4);
                need(f + 4);
                filt_group_fast<LP, 4, TAPS, false>(s, d, ring_at(f), st + (rbase + rows) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr);
                rows += 4;
                f += 4;
                release();
            } else if (f < lim) {
                stage_room(1);
                need(f + 1);
                filt_group_fast<LP, 1, TAPS, false>(s, d, ring_at(f), st + (rbase + rows) * SUBW_PAD + lane, TAPS && tap ? tap + f : nullptr);
                rows += 1;
                f += 1;
                release();
            } else {
                break;
            }
        }
    };
    for (;;) {
        const uint32_t lim = min(limit, NF);
        if (all_lp) run_fast(std::true_type{}, lim);
        else run_fast(std::false_type{}, lim);
        if (f >= NF) break;
        // frame `limit`: events are applied, then the frame runs with the envelope state machine checked
        if (f >= next_ev) {
            bool touched = false;
            while (ec.next_frame <= f) { // this role's events only, sorted by (frame, node, arrival)
                if (ec.e0.op == OP_SET) s.set(ec.e0.reg, ec.e0.value);
                else if (ec.e0.op == OP_ASR_RELEASE) envasr_release(s.e.est, s.e.et, s.e.sc);
                ec.pop();
                cursor_skip<false>(ec);
                touched = true;
            }
            if (touched) s.e.derive(d);
            all_lp = __all_sync(0xFFFFFFFFu, sub_lane_lp(s));
            next_ev = __reduce_min_sync(0xFFFFFFFFu, ec.next_frame);
        }
        stage_room(1);
        need(f + 1);
        float *strow = st + (rbase + rows) * SUBW_PAD + lane;
        // the straight-line frame, then EnvAsr's transitions (envelopes.rs:60-77): they only change
        // what FOLLOWING frames do
        if (all_lp) filt_group_fast<true, 1, TAPS, false>(s, d, ring_at(f), strow, TAPS && tap ? tap + f : nullptr);
        else filt_group_fast<false, 1, TAPS, false>(s, d, ring_at(f), strow, TAPS && tap ? tap + f : nullptr);
        if (d.att && s.e.et >= 1.0f) s.e.est = ASR_SUSTAINING;
        if (d.rel && s.e.et <= 0.0f) {
            s.e.est = ASR_STOPPED;
            s.e.et = 0.0f;
        }
        rows += 1;
        f += 1;
        release();
        s.e.derive(d);
        limit = __reduce_min_sync(0xFFFFFFFFu, lane_limit(f));
    }
    if (rows) flush();
    if (active) {
        const uint32_t out_regs[] = {R_IC1, R_IC2, R_A1, R_A2, R_A3, R_M0, R_M1, R_M2, R_ET, R_AR, R_RR, R_SC, R_GAIN};
        const float out_vals[] = {s.ic1, s.ic2, s.a1, s.a2, s.a3, s.m0, s.m1, s.m2, s.e.et, s.e.ar, s.e.rr, s.e.sc, s.e.gain};
#pragma unroll
        for (int i = 0; i < 13; i++) a.regs[(size_t)out_regs[i] * V + v] = __float_as_uint(out_vals[i]);
        a.regs[(size_t)R_EST * V + v] = s.e.est;
    }
}

template <bool TAPS>
__global__ void __launch_bounds__(64, 8) render_sub_asr2(FusedArgs a) {
    __shared__ __align__(16) float ring[RING_FRAMES * 32];
    __shared__ __align__(16) float st[W2_TILE * SUBW_PAD];
    __shared__ uint32_t role_swap;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        uint32_t slot;
        asm volatile("mov.u32 %0, %%warpid;" : "=r"(slot));
        role_swap = (slot >> 2) & 1u; // alternate the roles between the CTAs that share a sub-partition pair
    }
    __syncthreads();
    const uint32_t v = blockIdx.x * 32 + lane;
    const bool active = v < a.n_voices;
    if ((warp ^ role_swap) == 0) sub2_osc_role(a, ring, lane, v, active);
    else sub2_filter_role<TAPS>(a, ring, st, lane, v, active);
}

bool match_sub_asr(const DevProgram &p) {
    if (p.n_nodes != 4 || p.n_regs != SUB_NREGS || p.n_ubus != 1) return false;
    const DevNode &saw = p.nodes[0], &svf = p.nodes[1], &env = p.nodes[2], &mul = p.nodes[3];
    if (saw.kind != DK_POLYBLEP || saw.mode != 0 || saw.n_post || saw.n_ar || saw.reg != R_T) return false;
    if (svf.kind != DK_SVF || svf.n_post || svf.n_ar || svf.reg != R_IC1 || svf.in_slot[0] != (int)saw.out_slot[0]) return false;
    if (env.kind != DK_ENVASR || env.n_post != 1 || env.post_op[0] != PO_MUL || env.post_reg[0] != R_GAIN || env.n_ar || env.reg != R_EST) return false;
    if (mul.kind != DK_MATH || mul.mode != 2 || mul.n_out != 1 || mul.n_post || mul.n_ar) return false;
    if (mul.in_slot[0] != (int)svf.out_slot[0] || mul.in_slot[1] != (int)env.out_slot[0]) return false;
    return p.ubus_slot[0] == mul.out_slot[0];
}


// recipe 3: node 2 is Envelope.wr_mul instead of EnvAsr.wr_mul
bool match_sub_seg(const DevProgram &p) {
    if (p.n_nodes != 4 || p.n_ubus != 1) return false;
    const DevNode &saw = p.nodes[0], &svf = p.nodes[1], &env = p.nodes[2], &mul = p.nodes[3];
    if (env.kind != DK_ENVELOPE || env.n_seg < 1) return false;
    const uint32_t gain_reg = R_EST + REGS_ENVELOPE_BASE + REGS_ENVELOPE_PER_SEG * env.n_seg;
    if (p.n_regs != gain_reg + 1) return false;
    if (saw.kind != DK_POLYBLEP || saw.mode != 0 || saw.n_post || saw.n_ar || saw.reg != R_T) return false;
    if (svf.kind != DK_SVF || svf.n_post || svf.n_ar || svf.reg != R_IC1 || svf.in_slot[0] != (int)saw.out_slot[0]) return false;
    if (env.n_post != 1 || env.post_op[0] != PO_MUL || env.post_reg[0] != gain_reg || env.n_ar || env.reg != R_EST) return false;
    if (mul.kind != DK_MATH || mul.mode != 2 || mul.n_out != 1 || mul.n_post || mul.n_ar) return false;
    if (mul.in_slot[0] != (int)svf.out_slot[0] || mul.in_slot[1] != (int)env.out_slot[0]) return false;
    return p.ubus_slot[0] == mul.out_slot[0];
}

// ------------------------------------------------------------------------------------------------
// recipe 1 "render_fm2": (SinNumeric mod * idx + fc) -> SinNumeric.ar_params() "freq", * amp  (configs[3])
// template order: 0 mod, 1 Constant idx, 2 Mul, 3 Constant fc, 4 Add, 5 car, 6 Constant amp, 7 Mul
enum : uint32_t { F_MPH = 0, F_MOFF = 1, F_MINC = 2, F_IDX = 3, F_FC = 4, F_CPH = 5, F_COFF = 6, F_CINC = 7, F_AMP = 8, FM_NREGS = 9 };
#ifndef FM_SUB_N
#define FM_SUB_N 32 // frames per straight-line group of render_fm2: 8 -> 23.9 ms, 16 -> 18.7 ms, 32 -> 17.7 ms per 10 s step of configs[3] (236 registers, no spills)
#endif
constexpr int FM_SUB = FM_SUB_N; // independent f64 sine chains in flight per lane

// ---- one lane per voice ("render_fm2_wide"): the form for banks with more warps than SM sub-partitions.
// Both oscillators of a voice run in sequence on one lane: 94 instructions per 32 voice-frames against
// 2 x 62 for the two-lane form below, which in exchange halves the time of ONE warp -- so the two-lane
// form wins while its warps (n_voices / 16) still find a sub-partition each (fm_two_lanes()).
constexpr int FM1_SUB = 8; // frames per straight-line group: 16 independent f64 sine chains in flight
struct FmVoice {
    float mph, moff, minc, idx, fc, cph, coff, cinc, amp;
    KN_DEV void set(uint32_t reg, uint32_t bits) {
        const float f = __uint_as_float(bits);
        switch (reg) {
        case F_MPH: mph = f; break;
        case F_MOFF: moff = f; break;
        case F_MINC: minc = f; break;
        case F_IDX: idx = f; break;
        case F_FC: fc = f; break;
        case F_CPH: cph = f; break;
        case F_COFF: coff = f; break;
        case F_CINC: cinc = f; break;
        case F_AMP: amp = f; break;
        default: break;
        }
    }
    // one frame in graph order: mod.process, Mul, Add, WrArParams(car): freq(v) then process, Mul
    // INRANGE: |phase_offset| < 16 on both oscillators, so every sine argument is below 120 and the
    // branch-free restatement applies: the frames of a group then form one basic block and their
    // (long, f64) sine chains overlap
    template <bool INRANGE> KN_DEV float tick(float sr, float rc_sr) {
        const float am = (mph + moff) * KN_TAU;
        const float m = INRANGE ? kn_sinf_glibc_inrange(am) : kn_sinf(am);  // osc.rs:264
        const float mn = mph + minc;
        mph = mn > 1.0f ? mn - 1.0f : mn;                        // osc.rs:266-268
        const float v = m * idx + fc;                            // MathUGen<Mul>, MathUGen<Add>
        // audio_rate.rs:42-57 + osc.rs:240-242: phase_increment = F::new(v as f64) / F::new(sr as f32)
        if (INRANGE) {
            // div_rc needs a quotient well inside the normal range: tiny numerators are scaled by 2^64
            // (exact) and the quotient scaled back (exact unless it is subnormal, |v| < 6e-34, where
            // the last bit of a 1e-45 increment cannot move a phase)
            const bool tiny = fabsf(v) <= 1e-20f;
            const float q = div_rc(tiny ? v * 0x1p64f : v, sr, rc_sr);
            cinc = tiny ? q * 0x1p-64f : q;
        } else {
            cinc = fabsf(v) > 1e-20f ? div_rc(v, sr, rc_sr) : v / sr;
        }
        const float ac = (cph + coff) * KN_TAU;
        const float c = INRANGE ? kn_sinf_glibc_inrange(ac) : kn_sinf(ac);
        const float cn = cph + cinc;
        cph = cn > 1.0f ? cn - 1.0f : cn;
        return c * amp;
    }
    // Every sine argument of the next FM1_SUB frames stays below 120 (the branch-free restatement's domain): a phase moves by
    // at most |increment| per frame (the wrap only brings a phase above 1 closer to 0), the modulator's increment is minc and
    // the carrier's |v| / sr <= (|idx| + |fc|) / sr (|m| <= 1), and 18.5 * TAU = 116.2 leaves room for the roundings (and for
    // rc_sr = div_prep(sr), which is within an ulp of 1 / sr: no division in the loop).
    // Evaluated before every group: SinNumeric wraps its phase from above only, so at a negative frequency it descends
    // without bound (osc.rs:266-268).
    KN_DEV bool inrange(float rc_sr) const {
        const float mspan = fabsf(mph) + fabsf(moff) + FM1_SUB * fabsf(minc);
        const float cspan = fabsf(cph) + fabsf(coff) + FM1_SUB * ((fabsf(idx) + fabsf(fc)) * rc_sr);
        return mspan < 18.5f && cspan < 18.5f;
    }
};

template <bool TAPS>
__global__ void __launch_bounds__(32, 8) render_fm2_wide(FusedArgs a) {
    __shared__ float st[SUB_TILE * SUB_PAD];
    const uint32_t lane = threadIdx.x;
    const uint32_t gwarp = blockIdx.x;
    const uint32_t v = gwarp * 32 + lane;
    const uint32_t V = a.n_voices;
    const bool active = v < V;
    const float sr = a.prog->sample_rate;
    const float rc_sr = div_prep(sr);

    FmVoice s;
#pragma unroll
    for (int i = 0; i < FM_NREGS; i++) s.set(i, active ? a.regs[(size_t)i * V + v] : 0u);
    uint32_t cur = 0, end = 0, next_frame = 0xFFFFFFFFu;
    if (a.events && active) {
        cur = a.ev_off[v];
        end = a.ev_off[v + 1];
        if (cur < end) next_frame = a.events[cur].frame;
    }
    int tap_row = -1;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (active && a.taps[i].voice == v) tap_row = (int)a.taps[i].tap;

    float *prow = a.partials + (size_t)(a.row0 + gwarp) * a.n_frames;
    bool all_inrange = __all_sync(0xFFFFFFFFu, !active || s.inrange(rc_sr));
    for (uint32_t f0 = 0; f0 < a.n_frames; f0 += SUB_TILE) {
        const uint32_t nf = min((uint32_t)SUB_TILE, a.n_frames - f0);
#pragma unroll 1
        for (uint32_t g0 = 0; g0 < SUB_TILE; g0 += FM1_SUB) {
            const uint32_t gf = f0 + g0;
            all_inrange = __all_sync(0xFFFFFFFFu, !active || s.inrange(rc_sr));   // the phases have moved since the last group
            const bool ev_group = __any_sync(0xFFFFFFFFu, next_frame < gf + FM1_SUB);
            if (!ev_group && all_inrange && g0 + FM1_SUB <= nf) {
#pragma unroll
                for (int k = 0; k < FM1_SUB; k++) {
                    const float o = s.tick<true>(sr, rc_sr);
                    st[(g0 + k) * SUB_PAD + lane] = active ? o : 0.f;
                    if (TAPS && tap_row >= 0) a.tap_out[(size_t)tap_row * a.tap_stride + a.tap_frame0 + gf + k] = o;
                }
            } else {
#pragma unroll 1
                for (uint32_t k = 0; k < FM1_SUB; k++) {
                    float o = 0.f;
                    if (g0 + k < nf) {
                        bool touched = false;
                        while (next_frame <= gf + k) {
                            const DevEvent e = a.events[cur];
                            if (e.op == OP_SET) s.set(e.reg, e.value);
                            cur++;
                            next_frame = cur < end ? a.events[cur].frame : 0xFFFFFFFFu;
                            touched = true;
                        }
                        if (__any_sync(0xFFFFFFFFu, touched)) all_inrange = __all_sync(0xFFFFFFFFu, !active || s.inrange(rc_sr));
                        o = s.tick<false>(sr, rc_sr);
                        if (TAPS && tap_row >= 0) a.tap_out[(size_t)tap_row * a.tap_stride + a.tap_frame0 + gf + k] = o;
                    }
                    st[(g0 + k) * SUB_PAD + lane] = active ? o : 0.f;
                }
            }
        }
        __syncwarp();
        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            acc0 = acc0 + st[lane * SUB_PAD + j];
            acc1 = acc1 + st[lane * SUB_PAD + j + 1];
            acc2 = acc2 + st[lane * SUB_PAD + j + 2];
            acc3 = acc3 + st[lane * SUB_PAD + j + 3];
        }
        if (lane < nf) prow[f0 + lane] = (acc0 + acc1) + (acc2 + acc3);
        __syncwarp();
    }
    if (active) {
        const float regs_out[FM_NREGS] = {s.mph, s.moff, s.minc, s.idx, s.fc, s.cph, s.coff, s.cinc, s.amp};
#pragma unroll
        for (int i = 0; i < FM_NREGS; i++) a.regs[(size_t)i * V + v] = __float_as_uint(regs_out[i]);
    }
}

// ---- two lanes per voice ("render_fm2") ---------------------------------------------------------------
// A voice is two SinNumeric oscillators, so it occupies TWO lanes that run one instruction stream
// (arg = (phase + offset) * TAU, sinf(arg), phase update): lane j is the modulator, lane j + 16 the
// carrier of voice (warp * 16 + j).  The carrier's phase increment at frame k is made from the
// modulator's sample of frame k (osc.rs:240-242 through WrArParams), which in one SIMT stream would
// chain every sine behind the previous one.  So the carrier lanes run TWO GROUPS BEHIND the modulator
// lanes: a group's sines are independent on every lane (the carriers read modulator samples that
// were exchanged an iteration earlier), their f64 chains overlap, and a warp executes one sine per
// frame instead of two.  Twice the warps for the same bank (8192 voices = 512 warps, one per SM
// sub-partition), half the instructions per warp.  A launch runs three extra iterations: the
// carriers sit out the first two, the modulators the last ones, so the state saved at the end of a
// launch has both oscillators at the same frame.
constexpr int FM_VPW = 16; // voices per warp

// element k of a register array with k a loop variable of a partially unrolled loop (the exact path): a select chain, no local memory
template <int N> KN_DEV float fm_pick(const float (&a)[N], int k) {
    float r = a[0];
#pragma unroll
    for (int i = 1; i < N; i++) r = k == i ? a[i] : r;
    return r;
}
template <int N> KN_DEV void fm_put(float (&a)[N], int k, float v) {
#pragma unroll
    for (int i = 0; i < N; i++) a[i] = k == i ? v : a[i];
}

struct FmLane {
    float ph, off, inc;   // this lane's oscillator: modulator (F_MPH..) or carrier (F_CPH..)
    float idx, fc, amp;   // carrier lanes: the Mul / Add constants of the route and the output gain
    uint32_t base;        // F_MPH or F_CPH
    bool car;
    KN_DEV void set(uint32_t reg, uint32_t bits) {
        const float f = __uint_as_float(bits);
        if (reg == base) ph = f;
        else if (reg == base + 1) off = f;
        else if (reg == base + 2) inc = f;
        else if (reg == F_IDX) idx = f;
        else if (reg == F_FC) fc = f;
        else if (reg == F_AMP) amp = f;
    }
    // The phase half of one frame, in graph order: mod.process / Mul, Add, WrArParams(car): freq(v),
    // then process: returns the sine argument of this frame and advances the phase.  m = the
    // modulator's sample of this frame (carrier lanes).  commit = false leaves the state untouched.
    template <bool INRANGE> KN_DEV float advance(float m, float sr, float rc_sr, bool commit) {
        const float arg = (ph + off) * KN_TAU;                                // osc.rs:264
        // carrier lanes only, but evaluated branch-free on every lane (modulator lanes discard it): a
        // branch here would cut the group into basic blocks and keep its sine chains from overlapping
        const float v = m * idx + fc;                                         // MathUGen<Mul>, MathUGen<Add>
        // audio_rate.rs:42-57 + osc.rs:240-242: phase_increment = F::new(v as f64) / F::new(sr as f32)
        float q;
        if (INRANGE) {
            // div_rc needs a quotient well inside the normal range: tiny numerators are scaled by 2^64
            // (exact) and the quotient scaled back (exact unless it is subnormal, |v| < 6e-34, where
            // the last bit of a 1e-45 increment cannot move a phase)
            const bool tiny = fabsf(v) <= 1e-20f;
            const float q0 = div_rc(tiny ? v * 0x1p64f : v, sr, rc_sr);
            q = tiny ? q0 * 0x1p-64f : q0;
        } else {
            q = fabsf(v) > 1e-20f ? div_rc(v, sr, rc_sr) : v / sr;
        }
        const float ninc = car ? q : inc;
        const float pn = ph + ninc;
        const float nph = pn > 1.0f ? pn - 1.0f : pn;                         // osc.rs:266-268
        if (commit) {
            inc = ninc;
            ph = nph;
        }
        return arg;
    }
    // Every sine argument of this lane's next FM_SUB frames stays below 120, so the branch-free restatement of sinf applies
    // (the bound of FmVoice::inrange: a carrier's increment is at most (|idx| + |fc|) / sr, a modulator's is inc; rc_sr ~ 1 / sr).
    // Evaluated before every group: at a negative frequency the phase descends without bound.
    KN_DEV bool inrange(float rc_sr) const {
        const float step = car ? (fabsf(idx) + fabsf(fc)) * rc_sr : fabsf(inc);
        return fabsf(ph) + fabsf(off) + FM_SUB * step < 18.5f;
    }
};

template <bool TAPS>
__global__ void __launch_bounds__(32, 8) render_fm2(FusedArgs a) {
    __shared__ float st[SUB_TILE * SUB_PAD];
    const uint32_t lane = threadIdx.x;
    const uint32_t gwarp = blockIdx.x;
    const uint32_t mod_lane = lane & (FM_VPW - 1);
    const uint32_t v = gwarp * FM_VPW + mod_lane;
    const uint32_t V = a.n_voices;
    const bool active = v < V;
    const float sr = a.prog->sample_rate;
    const float rc_sr = div_prep(sr);

    FmLane s;
    s.car = lane >= FM_VPW;
    s.base = s.car ? (uint32_t)F_CPH : (uint32_t)F_MPH;
    s.ph = s.off = s.inc = s.idx = s.fc = s.amp = 0.f;
    if (active) {
        s.ph = __uint_as_float(a.regs[(size_t)s.base * V + v]);
        s.off = __uint_as_float(a.regs[(size_t)(s.base + 1) * V + v]);
        s.inc = __uint_as_float(a.regs[(size_t)(s.base + 2) * V + v]);
        s.idx = __uint_as_float(a.regs[(size_t)F_IDX * V + v]);
        s.fc = __uint_as_float(a.regs[(size_t)F_FC * V + v]);
        s.amp = __uint_as_float(a.regs[(size_t)F_AMP * V + v]);
    }
    const bool emit = active && s.car;
    uint32_t cur = 0, end = 0, next_frame = 0xFFFFFFFFu; // both lanes of a voice walk its event list, each at its own frame
    if (a.events && active) {
        cur = a.ev_off[v];
        end = a.ev_off[v + 1];
        if (cur < end) next_frame = a.events[cur].frame;
    }
    int tap_row = -1;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (emit && a.taps[i].voice == v) tap_row = (int)a.taps[i].tap;
    float *tap = TAPS && tap_row >= 0 ? a.tap_out + (size_t)tap_row * a.tap_stride + a.tap_frame0 : nullptr;

    float *prow = a.partials + (size_t)(a.row0 + gwarp) * a.n_frames;
    const uint32_t NF = a.n_frames, NG = (NF + FM_SUB - 1) / FM_SUB;
    const uint32_t lag = s.car ? 2u * FM_SUB : 0u;       // the carriers run two groups behind the modulators
    // Software pipeline, per iteration G:  (1) phases of this lane's group, from the carrier increments the previous iteration made out
    // of the modulator samples it exchanged;  (2) this group's sines are ISSUED (sn_new);  (3) the previous iteration's sines (sn_old,
    // complete by now) are staged as output on the carrier lanes and shuffled from the modulator lanes to the carrier lanes, which turn
    // them into the increments of their next group.  Nothing in an iteration waits for a sine issued in the same iteration, and an
    // event-free iteration is ONE basic block: the f64 pipe takes a warp instruction every other cycle (8 cycles latency; measured,
    // tools/microbench/fp64_bench.cu), so the sixteen f64 operations of a sine leave sixteen issue slots that only the f32 / integer /
    // shared-memory work of steps (1) and (3) can fill -- if it sits in the same block.
    // The output gain of a group: event-free groups have ONE gain per lane (0 on lanes that emit nothing: a sine of an in-range argument
    // is finite, so sine * 0 is a zero); groups that took the exact path multiply per frame as they go, zero what is not to be heard and
    // hand over the products with gain 1 (x * 1 is exact).  The modulator lanes' staging columns are never read.
    float mcur[FM_SUB], q[FM_SUB], sn_old[FM_SUB];
    float amp_old = 0.f;
    bool q_ok = false;                                   // q[] holds the carrier increments of the next group (no numerator was tiny)
#pragma unroll
    for (int k = 0; k < FM_SUB; k++) mcur[k] = q[k] = sn_old[k] = 0.f;
    bool all_inrange = __all_sync(0xFFFFFFFFu, !active || s.inrange(rc_sr));
    uint32_t tile0 = 0;                                  // first frame of the staging tile the carriers are filling
    // steps (3): staging, exchange, increments of the next group.  Part of both branches below, so that the event-free one stays whole.
    auto hand_over = [&](uint32_t G, uint32_t gf) {
        if (G >= 3) { // the carriers' sines of the previous iteration: frames (G - 3) * FM_SUB + k
            float *row = st + (gf - 3u * FM_SUB - tile0) * SUB_PAD + lane;
#pragma unroll
            for (int k = 0; k < FM_SUB; k++) {
                const float o = sn_old[k] * amp_old;     // MathUGen<Mul> with the gain as it was at that frame
                row[k * SUB_PAD] = o;
                if (TAPS) {
                    const uint32_t fr = gf - 3u * FM_SUB + k;
                    if (tap && emit && fr < NF) tap[fr] = o;
                }
            }
        }
        // the modulators' sines of the previous iteration (frames (G - 1) * FM_SUB + k) reach the carrier lanes, which get to those
        // frames in the next iteration: audio_rate.rs:42-57 + osc.rs:240-242, phase_increment = F::new(v as f64) / F::new(sr as f32).
        // The increments depend on the exchanged samples and the route's constants only, not on the phase; if a numerator is too small
        // for div_rc's exactness argument (|v| <= 1e-20: the quotient's last bit would need the scaled form) the next group takes the
        // exact path, as it does when an event changes the constants
        float vmin = 1.0f;
#pragma unroll
        for (int k = 0; k < FM_SUB; k++) {
            mcur[k] = __shfl_sync(0xFFFFFFFFu, sn_old[k], mod_lane);
            const float vv = mcur[k] * s.idx + s.fc;     // MathUGen<Mul>, MathUGen<Add>
            vmin = fminf(vmin, fabsf(vv));
            q[k] = div_rc(vv, sr, rc_sr);
        }
        q_ok = !__any_sync(0xFFFFFFFFu, s.car && vmin <= 1e-20f);
    };
#pragma unroll 1
    for (uint32_t G = 0; G <= NG + 2; G++) {
        const uint32_t gf = G * FM_SUB;                  // the modulators' first frame in this iteration
        const uint32_t lf = gf - lag;                    // this lane's first frame (meaningful while role_on)
        const bool role_on = s.car ? (G >= 2 && G < NG + 2) : G < NG;
        all_inrange = __all_sync(0xFFFFFFFFu, !active || s.inrange(rc_sr));       // the phases have moved since the last group
        const bool ev_group = __any_sync(0xFFFFFFFFu, role_on && next_frame < lf + FM_SUB);
        if (!ev_group && all_inrange && q_ok && G >= 3 && gf + FM_SUB <= NF) { // both roles have a whole group
            float arg[FM_SUB], sn_new[FM_SUB];
            float ph = s.ph;
#pragma unroll
            for (int k = 0; k < FM_SUB; k++) {
                arg[k] = (ph + s.off) * KN_TAU;          // osc.rs:264
                const float pn = ph + (s.car ? q[k] : s.inc);
                ph = pn > 1.0f ? pn - 1.0f : pn;         // osc.rs:266-268
            }
            s.ph = ph;
            s.inc = s.car ? q[FM_SUB - 1] : s.inc;
#ifdef FM_STAGED
            kn_sinf_glibc_lean_n(arg, sn_new);
#else
#pragma unroll
            for (int k = 0; k < FM_SUB; k++) sn_new[k] = kn_sinf_glibc_lean(arg[k]);
#endif
            hand_over(G, gf);
#pragma unroll
            for (int k = 0; k < FM_SUB; k++) sn_old[k] = sn_new[k];
            amp_old = emit ? s.amp : 0.f;
        } else {
            float sn_new[FM_SUB];
#pragma unroll 1
            for (int k0 = 0; k0 < FM_SUB; k0 += 4) {
#pragma unroll
                for (int kk = 0; kk < 4; kk++) {
                    const int k = k0 + kk;
                    const uint32_t fr = lf + k;
                    const bool valid = role_on && fr < NF;
                    bool touched = false;
                    while (valid && next_frame <= fr) {
                        const DevEvent e = a.events[cur];
                        if (e.op == OP_SET) s.set(e.reg, e.value);
                        cur++;
                        next_frame = cur < end ? a.events[cur].frame : 0xFFFFFFFFu;
                        touched = true;
                    }
                    if (__any_sync(0xFFFFFFFFu, touched)) all_inrange = __all_sync(0xFFFFFFFFu, !active || s.inrange(rc_sr));
                    const float sn = kn_sinf(s.advance<false>(fm_pick(mcur, k), sr, rc_sr, valid));
                    // carriers: MathUGen<Mul> with the gain of this frame; modulators hand over the bare sample
                    fm_put(sn_new, k, s.car ? (valid && emit ? sn * s.amp : 0.f) : sn);
                }
            }
            hand_over(G, gf);
#pragma unroll
            for (int k = 0; k < FM_SUB; k++) sn_old[k] = sn_new[k];
            amp_old = 1.0f;
        }
        if (G >= 3) {
            const uint32_t cend = min(gf - 2u * FM_SUB, NF); // every frame below cend is staged
            if (cend - tile0 == SUB_TILE || G == NG + 2) {
                __syncwarp();
                // lane = frame: sum the 16 carrier columns
                float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll
                for (int j = FM_VPW; j < 32; j += 4) {
                    acc0 = acc0 + st[lane * SUB_PAD + j];
                    acc1 = acc1 + st[lane * SUB_PAD + j + 1];
                    acc2 = acc2 + st[lane * SUB_PAD + j + 2];
                    acc3 = acc3 + st[lane * SUB_PAD + j + 3];
                }
                if (lane < cend - tile0) prow[tile0 + lane] = (acc0 + acc1) + (acc2 + acc3);
                tile0 = cend;
                __syncwarp();
            }
        }
    }
    if (active) {
        a.regs[(size_t)s.base * V + v] = __float_as_uint(s.ph);
        a.regs[(size_t)(s.base + 1) * V + v] = __float_as_uint(s.off);
        a.regs[(size_t)(s.base + 2) * V + v] = __float_as_uint(s.inc);
        if (s.car) {
            a.regs[(size_t)F_IDX * V + v] = __float_as_uint(s.idx);
            a.regs[(size_t)F_FC * V + v] = __float_as_uint(s.fc);
            a.regs[(size_t)F_AMP * V + v] = __float_as_uint(s.amp);
        }
    }
}

bool match_fm2(const DevProgram &p) {
    if (p.n_nodes != 8 || p.n_regs != FM_NREGS || p.n_ubus != 1) return false;
    const DevNode *n = p.nodes;
    auto plain = [](const DevNode &d) { return d.n_post == 0 && d.n_ar == 0; };
    if (n[0].kind != DK_SINNUM || !plain(n[0]) || n[0].reg != F_MPH) return false;
    if (n[1].kind != DK_CONST || !plain(n[1]) || n[1].reg != F_IDX) return false;
    if (n[2].kind != DK_MATH || n[2].mode != 2 || n[2].n_out != 1 || !plain(n[2])) return false;
    if (n[2].in_slot[0] != (int)n[0].out_slot[0] || n[2].in_slot[1] != (int)n[1].out_slot[0]) return false;
    if (n[3].kind != DK_CONST || !plain(n[3]) || n[3].reg != F_FC) return false;
    if (n[4].kind != DK_MATH || n[4].mode != 0 || n[4].n_out != 1 || !plain(n[4])) return false;
    if (n[4].in_slot[0] != (int)n[2].out_slot[0] || n[4].in_slot[1] != (int)n[3].out_slot[0]) return false;
    if (n[5].kind != DK_SINNUM || n[5].n_post || n[5].n_ar != 1 || n[5].ar_code[0] != AR_SINNUM_FREQ || n[5].reg != F_CPH) return false;
    if (n[5].ar_slot[0] != (int)n[4].out_slot[0]) return false;
    if (n[6].kind != DK_CONST || !plain(n[6]) || n[6].reg != F_AMP) return false;
    if (n[7].kind != DK_MATH || n[7].mode != 2 || n[7].n_out != 1 || !plain(n[7])) return false;
    if (n[7].in_slot[0] != (int)n[5].out_slot[0] || n[7].in_slot[1] != (int)n[6].out_slot[0]) return false;
    return p.ubus_slot[0] == n[7].out_slot[0];
}

} // namespace

int match_fused_recipe(const DevProgram &p, uint32_t block_size) {
    if (match_sub_asr(p)) return 0;
    if (match_fm2(p)) return 1;
    if (match_add_wt(p, block_size)) return 2;
    if (match_sub_seg(p)) return 3;
    return -1;
}
const char *fused_recipe_name(int recipe) {
    switch (recipe) {
    case 0: return "render_sub_asr";
    case 1: return "render_fm2";
    case 2: return "render_add_wt";
    case 3: return "render_sub_seg";
    case 4: return "render_sub_scan";
    default: return "render_interp";
    }
}
// recipe 1: two lanes per voice while that still leaves at most one warp per SM sub-partition (148 x 4)
bool fm_two_lanes(uint32_t n_voices) { return (n_voices + FM_VPW - 1) / FM_VPW <= 148u * 4u; }
// recipe 4's form, read once from the environment: launch_fused runs it and sub_scan_applies accepts the block sizes its chunks tile
struct ScanForm {
    // Default: two warps per voice (render_sub_scan2, 64-frame chunks): 4.3 ms per 10 s step of 256 voices.  KGPU_SCAN_WARPS=1
    // selects the one-warp kernels, kept for measurements: render_sub_scan_n (KGPU_SCAN_FPL=2, 5.0 ms) and render_sub_scan
    // (KGPU_SCAN_FPL=1, 5.8 ms)
    bool two_warps;
    // KGPU_SCAN_FPL: frames per lane of render_sub_scan_n (2 or 4; anything else = render_sub_scan)
    int fpl;
    // KGPU_SCAN_PIPE=0: render_sub_scan's unpipelined form (pre-pass, then the frame-parallel half), kept for measurements
    bool pipe;
    uint32_t chunk_frames() const {
        if (two_warps) return 2 * SCAN_CHUNK;                         // render_sub_scan2<.., 2>
        return fpl == 2 || fpl == 4 ? fpl * SCAN_CHUNK : SCAN_CHUNK;  // render_sub_scan_n<.., fpl>, render_sub_scan
    }
};
static const ScanForm &scan_form() {
    static const ScanForm f = [] {
        const char *w = getenv("KGPU_SCAN_WARPS"), *n = getenv("KGPU_SCAN_FPL"), *p = getenv("KGPU_SCAN_PIPE");
        return ScanForm{!(w && *w == '1'), n && *n ? atoi(n) : 2, !(p && *p == '0')};
    }();
    return f;
}
// recipe 0 -> 4: a bank this small leaves most schedulers without a warp under one-lane-per-voice; one warp per voice
// with the frames of a chunk across the lanes is faster up to ~1500 voices (measured, 10 s steps: 256 voices 6.7 ms against
// 13.0, 1024 9.3 against 13.1, 2048 15.2 against 13.2; DESIGN.md section 3).  The kernels number their chunks from the start
// of each launch, and which frames a chunk scans decides their last bits: the chunks of the form launch_fused runs must tile
// the block grid, so that a render is identical however it is split into launches.  Other block sizes take render_sub_asr.
bool sub_scan_applies(uint32_t n_voices, uint32_t block_size) {
    static const int force = [] { const char *e = getenv("KGPU_SUB_SCAN"); return e ? atoi(e) : -1; }(); // 0 never, 1 always (tests / measurements)
    if (block_size % scan_form().chunk_frames()) return false;
    if (force >= 0) return force != 0;
    return n_voices <= 1024;
}
uint32_t fused_rows(int recipe, uint32_t n_voices, uint32_t n_ubus) {
    if (recipe == 4) return n_voices * n_ubus;                // one partial row per voice
    if (recipe == 2) return add_wt_slices(n_voices) * n_ubus; // one partial row per voice slice
    if (recipe == 1 && fm_two_lanes(n_voices)) return ((n_voices + FM_VPW - 1) / FM_VPW) * n_ubus;
    return ((n_voices + 31) / 32) * n_ubus;                   // one partial row per warp
}
size_t fused_scratch_bytes(int recipe, uint32_t n_voices, uint32_t n_frames, uint32_t block_size) {
    return recipe == 2 ? add_wt_scratch_bytes(n_voices, n_frames, block_size) : 0;
}
cudaError_t launch_fused(int recipe, const FusedArgs &a, cudaStream_t stream) {
    if (recipe == 1) {
        if (fm_two_lanes(a.n_voices)) {
            const uint32_t nw = (a.n_voices + FM_VPW - 1) / FM_VPW;
            if (a.n_taps) render_fm2<true><<<nw, 32, 0, stream>>>(a);
            else render_fm2<false><<<nw, 32, 0, stream>>>(a);
        } else {
            const uint32_t nw = (a.n_voices + 31) / 32;
            if (a.n_taps) render_fm2_wide<true><<<nw, 32, 0, stream>>>(a);
            else render_fm2_wide<false><<<nw, 32, 0, stream>>>(a);
        }
        return cudaGetLastError();
    }
    if (recipe == 2) return launch_add_wt(a, stream);
    if (recipe == 4) {
        const ScanForm &form = scan_form();
        const bool pipe = form.pipe, two_warps = form.two_warps;
        const int fpl = form.fpl;
        if (!two_warps && fpl == 2) {
            if (a.n_taps) render_sub_scan_n<true, 2><<<a.n_voices, 32, 0, stream>>>(a);
            else render_sub_scan_n<false, 2><<<a.n_voices, 32, 0, stream>>>(a);
            return cudaGetLastError();
        }
        if (!two_warps && fpl == 4) {
            if (a.n_taps) render_sub_scan_n<true, 4><<<a.n_voices, 32, 0, stream>>>(a);
            else render_sub_scan_n<false, 4><<<a.n_voices, 32, 0, stream>>>(a);
            return cudaGetLastError();
        }
        if (two_warps) {
            if (a.n_taps) render_sub_scan2<true, 2><<<a.n_voices, 64, 0, stream>>>(a);
            else render_sub_scan2<false, 2><<<a.n_voices, 64, 0, stream>>>(a);
            return cudaGetLastError();
        }
        if (pipe) {
            if (a.n_taps) render_sub_scan<true, true><<<a.n_voices, 32, 0, stream>>>(a);
            else render_sub_scan<false, true><<<a.n_voices, 32, 0, stream>>>(a);
        } else {
            if (a.n_taps) render_sub_scan<true, false><<<a.n_voices, 32, 0, stream>>>(a);
            else render_sub_scan<false, false><<<a.n_voices, 32, 0, stream>>>(a);
        }
        return cudaGetLastError();
    }
    if (recipe == 3) {
        const uint32_t nw = (a.n_voices + 31) / 32;
        if (a.n_taps) render_sub_seg<true><<<nw, 32, 0, stream>>>(a);
        else render_sub_seg<false><<<nw, 32, 0, stream>>>(a);
        return cudaGetLastError();
    }
    if (recipe != 0) return cudaErrorNotSupported;
    // one CTA = one warp per 32 voices: 16384 voices = 512 CTAs spread over all 148 SMs (3-4 per SM)
    const uint32_t n_warps = (a.n_voices + 31) / 32;
    // Default: one warp per 32 voices (render_sub_asr).  KGPU_SUB_TWO_WARPS=1 selects the
    // warp-specialised pair (render_sub_asr2), kept as a measured negative result: 18.1 ms per 10 s
    // step against 15.7 ms (DESIGN.md section 3).
    static const bool two = [] { const char *e = getenv("KGPU_SUB_TWO_WARPS"); return e && *e == '1'; }();
    if (!two) {
        if (a.n_taps) render_sub_asr<true><<<n_warps, 32, 0, stream>>>(a);
        else render_sub_asr<false><<<n_warps, 32, 0, stream>>>(a);
    } else {
        if (a.n_taps) render_sub_asr2<true><<<n_warps, 64, 0, stream>>>(a);
        else render_sub_asr2<false><<<n_warps, 64, 0, stream>>>(a);
    }
    return cudaGetLastError();
}

} // namespace kgpu
