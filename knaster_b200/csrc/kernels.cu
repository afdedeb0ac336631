// kernels.cu -- sm_100a kernels of the batched render engine.
//
//   render_interp   generic plan interpreter: one warp = 32 voices of one template, nodes run
//                   in topological order over 16-frame chunks, node buffers live in shared
//                   memory (never in HBM), per-voice registers are loaded from / stored to HBM
//                   once per launch.  This is GraphGen::process_block's task loop
//                   (graph_gen.rs:196-200) turned inside out: the loop over nodes is
//                   warp-uniform, the 32 lanes are 32 independent voices.
//   reduce_bus      deterministic mix-bus reduction of the per-warp partial sums into the
//                   [block][channel][frame] output layout (graph.rs:850-864 + graph_gen.rs:205-224).
//   fused kernels   see fused.cuh (register-resident specialisations for known voice shapes).
#include <cuda_runtime.h>

#include <algorithm>
#include <stdint.h>

#include "dev.h"
#include "kernels.h"
#include "nodes.cuh"

namespace kgpu {

namespace {

struct LaneEv {
    const DevEvent *ev;
    uint32_t cur, end;
    uint32_t next_frame, next_node;
    KN_DEV void fetch() {
        if (cur < end) {
            next_frame = ev[cur].frame;
            next_node = ev[cur].node;
        } else {
            next_frame = 0xFFFFFFFFu;
            next_node = 0xFFFFFFFFu;
        }
    }
};

KN_DEV double ld_d(const uint32_t *sreg, uint32_t r) {
    return __hiloint2double((int)sreg[(r + 1) * 32], (int)sreg[r * 32]);
}
KN_DEV void st_d(uint32_t *sreg, uint32_t r, double v) {
    sreg[r * 32] = (uint32_t)__double2loint(v);
    sreg[(r + 1) * 32] = (uint32_t)__double2hiint(v);
}

// apply every event of `node` due at or before `frame` to the lane's registers (in shared memory)
KN_DEV void apply_events(LaneEv &L, uint32_t node, uint32_t node_reg, uint32_t frame, uint32_t *sreg) {
    while (L.next_node == node && L.next_frame <= frame) {
        const DevEvent e = L.ev[L.cur];
        if (e.op == OP_SET) {
            sreg[e.reg * 32] = e.value;
        } else if (e.op == OP_ASR_RELEASE) {
            uint32_t st = sreg[e.reg * 32];
            float t = __uint_as_float(sreg[(e.reg + 1) * 32]);
            float sc = __uint_as_float(sreg[(e.reg + 4) * 32]);
            envasr_release(st, t, sc);
            sreg[e.reg * 32] = st;
            sreg[(e.reg + 1) * 32] = __float_as_uint(t);
            sreg[(e.reg + 4) * 32] = __float_as_uint(sc);
        } else if (e.op == OP_ENV_STOP) { // envelopes.rs:511-523
            if (sreg[e.reg * 32]) {
                uint32_t seg = sreg[(e.reg + 1) * 32];
                double t = ld_d(sreg, e.reg + 2), from = ld_d(sreg, e.reg + 4);
                uint32_t sb = e.reg + REGS_ENVELOPE_BASE + REGS_ENVELOPE_PER_SEG * seg;
                double recip = ld_d(sreg, sb), val = ld_d(sreg, sb + 4);
                from = __dadd_rn(from, __dmul_rn(__dmul_rn(t, recip), __dsub_rn(val, from)));
                st_d(sreg, e.reg + 4, from);
            }
            sreg[e.reg * 32] = 0;
        } else if (e.op == OP_ENV_RESTART) { // envelopes.rs:504-510; (reg, value) = from_value
            sreg[node_reg * 32] = 1;
            sreg[(node_reg + 1) * 32] = 0;
            sreg[(node_reg + 2) * 32] = 0;
            sreg[(node_reg + 3) * 32] = 0;
            sreg[(node_reg + 4) * 32] = e.reg;
            sreg[(node_reg + 5) * 32] = e.value;
        } else if (e.op == OP_ENV_JUMP) {    // envelopes.rs:480-503
            sreg[e.reg * 32] = 1;
            sreg[(e.reg + 1) * 32] = e.value;
            sreg[(e.reg + 2) * 32] = 0;
            sreg[(e.reg + 3) * 32] = 0;
        } else if (e.op == OP_ENV_STEP) {    // envelopes.rs:477-479; (reg, value) = step
            sreg[(node_reg + 6) * 32] = e.reg;
            sreg[(node_reg + 7) * 32] = e.value;
        }
        L.cur++;
        L.fetch();
    }
}

} // namespace

// One CTA = one warp = 32 voices.  Shared memory: registers [n_regs][32] u32, then value slots
// [n_slots][chunk][32] f32 -- lane-contiguous, so every access is bank-conflict free.
__global__ void __launch_bounds__(32) render_interp(InterpArgs a) {
    extern __shared__ uint32_t smem[];
    const DevProgram *__restrict__ prog = a.prog;
    const uint32_t lane = threadIdx.x;
    const uint32_t warp = blockIdx.x;
    const uint32_t v = warp * 32 + lane;
    const bool active = v < a.n_voices;
    const uint32_t n_regs = prog->n_regs, n_nodes = prog->n_nodes;
    const uint32_t CH = a.chunk;
    uint32_t *sreg = smem + lane;                              // sreg[r*32]
    float *sval = reinterpret_cast<float *>(smem + n_regs * 32) + lane; // sval[(slot*CH + f)*32]
    const float sr = prog->sample_rate;
    const double sinwt_k = prog->sinwt_k;

    for (uint32_t r = 0; r < n_regs; r++) sreg[r * 32] = active ? a.regs[(size_t)r * a.n_voices + v] : 0u;
    LaneEv L;
    L.ev = a.events;
    L.cur = L.end = 0;
    if (a.events && active) {
        L.cur = a.ev_off[v];
        L.end = a.ev_off[v + 1];
    }
    L.fetch();

    for (uint32_t c0 = 0; c0 < a.n_frames; c0 += CH) {
        const uint32_t nf = min(CH, a.n_frames - c0);
        for (uint32_t n = 0; n < n_nodes; n++) {
            const DevNode &dn = prog->nodes[n];
            const bool evc = __any_sync(0xFFFFFFFFu, L.next_node == n && L.next_frame < c0 + nf);
            const uint32_t rb = dn.reg;
            // arithmetic wrapper values
            float pv[MAX_POST];
#pragma unroll
            for (int k = 0; k < MAX_POST; k++) pv[k] = k < dn.n_post ? __uint_as_float(sreg[dn.post_reg[k] * 32]) : 0.f;
            // Fast path of a node over a whole chunk (16, 32 or 64 frames, in groups of 16 at offset g0_): no event
            // of this node falls into the chunk, no audio-rate route, at most one arithmetic wrapper and that one
            // a WrMul.  The 16 frames of a group are unrolled into one basic block (the per-frame event / route / wrapper checks of the generic loops
            // below cost more than the arithmetic and serialise it), and the wrapper is "times g_" with
            // g_ = 1 when there is none (x * 1 == x exactly).
            const uint32_t n_post_ = dn.n_post, o0_ = dn.out_slot[0];
            const bool plain_ok = dn.n_ar == 0 && (CH & 15u) == 0 && (n_post_ == 0 || (n_post_ == 1 && dn.post_op[0] == PO_MUL));
            // a chunk is walked in groups of 16 frames; a group takes the fast path unless an event of this node
            // falls into it (warp-uniform test on the lanes' event cursors) or it is a partial group
            // the same with audio-rate routes into the node's own parameters (not into a wrapper value): SinWt,
            // SinNumeric and PolyBlep read the routed samples 16 at a time and update the parameter per frame
            bool plain_ar_ok = dn.n_ar > 0 && (CH & 15u) == 0 && (n_post_ == 0 || (n_post_ == 1 && dn.post_op[0] == PO_MUL));
            int ar_s0 = -1, ar_s1 = -1; // value slots of the routes into parameter 0 (freq) / parameter 1 (phase_offset, pulse_width)
            for (int ai = 0; ai < dn.n_ar; ai++) {
                const uint32_t code = dn.ar_code[ai];
                if (code == AR_SINWT_FREQ || code == AR_SINNUM_FREQ || code == AR_POLYBLEP_FREQ) ar_s0 = dn.ar_slot[ai];
                else if (code == AR_SINWT_OFFSET || code == AR_SINNUM_OFFSET || code == AR_POLYBLEP_PW) ar_s1 = dn.ar_slot[ai];
                else plain_ar_ok = false;
            }
#define GROUP_PLAIN_AR (plain_ar_ok && fe_ - g0_ == 16 && !(evc && __any_sync(0xFFFFFFFFu, L.next_node == n && L.next_frame < c0 + fe_)))
#define FOR_GROUPS for (uint32_t g0_ = 0, fe_ = min(nf, 16u); g0_ < nf; g0_ += 16, fe_ = min(nf, g0_ + 16u))
#define GROUP_PLAIN (plain_ok && fe_ - g0_ == 16 && !(evc && __any_sync(0xFFFFFFFFu, L.next_node == n && L.next_frame < c0 + fe_)))
#define PLAIN16(EXPR_)                                                                 \
    {                                                                                  \
        float y_[16];                                                                  \
        const float g_ = n_post_ ? pv[0] : 1.0f; /* an event in an earlier group of the chunk may have changed it */ \
        _Pragma("unroll") for (int k = 0; k < 16; k++) y_[k] = (EXPR_);                \
        _Pragma("unroll") for (int k = 0; k < 16; k++) sval[(o0_ * CH + g0_ + k) * 32] = y_[k] * g_; \
    }
// the value a node reads: a value slot of the voice (>= 0), the permanent zero channel (-1), or an internal signal of the plan
// (<= -2: sums of voices read by nodes, sources shared between voices -- a.ext[signal][frame of the launch], the same for every voice)
#define RDV(slot_, f_) ((slot_) >= 0 ? sval[((slot_) * CH + (f_)) * 32] : ((slot_) == -1 ? 0.f : a.ext[(size_t)(-2 - (slot_)) * a.ext_stride + c0 + (f_)]))
#define LOAD16(x_, slot_)                                                              \
    float x_[16];                                                                      \
    _Pragma("unroll") for (int k = 0; k < 16; k++) x_[k] = RDV(slot_, g0_ + k);
#define EVENTS_AT(f_, STORE_, LOAD_)                                                   \
    if (evc && L.next_node == n && L.next_frame <= c0 + (f_)) {                        \
        STORE_;                                                                        \
        apply_events(L, n, rb, c0 + (f_), sreg);                                       \
        LOAD_;                                                                         \
        _Pragma("unroll") for (int k = 0; k < MAX_POST; k++) if (k < dn.n_post)        \
            pv[k] = __uint_as_float(sreg[dn.post_reg[k] * 32]);                        \
    }
#define AR_POST_ROUTES(f_)                                                             \
    for (int ai = 0; ai < dn.n_ar; ai++)                                               \
        if (dn.ar_code[ai] >= AR_POST) pv[dn.ar_code[ai] - AR_POST] = RDV(dn.ar_slot[ai], f_);
#define EMIT(f_, ch_, y_)                                                              \
    {                                                                                  \
        float _y = (y_);                                                               \
        _Pragma("unroll") for (int k = 0; k < MAX_POST; k++) if (k < dn.n_post)        \
            _y = post_apply(dn.post_op[k], _y, pv[k]);                                 \
        sval[(dn.out_slot[ch_] * CH + (f_)) * 32] = _y;                                \
    }
            switch (dn.kind) {
            case DK_SINWT: {
                uint32_t phase = sreg[rb * 32], off = sreg[(rb + 1) * 32], inc = sreg[(rb + 2) * 32];
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        PLAIN16(sinwt_tick(phase, off, inc, a.sine_table))
                        continue;
                    }
                    if (GROUP_PLAIN_AR) {
                        LOAD16(xf_, ar_s0)
                        LOAD16(xo_, ar_s1)
                        auto tk = [&](int k) {
                            if (ar_s0 >= 0) inc = kn_sat_u32(__dmul_rn((double)xf_[k], sinwt_k));
                            if (ar_s1 >= 0) off = kn_sat_u32(__dmul_rn((double)xo_[k], 65536.0));
                            return sinwt_tick(phase, off, inc, a.sine_table);
                        };
                        PLAIN16(tk(k))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, sreg[rb * 32] = phase, (phase = sreg[rb * 32], off = sreg[(rb + 1) * 32], inc = sreg[(rb + 2) * 32]))
                    for (int ai = 0; ai < dn.n_ar; ai++) {
                        float x = RDV(dn.ar_slot[ai], f);
                        if (dn.ar_code[ai] == AR_SINWT_FREQ) inc = kn_sat_u32(__dmul_rn((double)x, sinwt_k));
                        else if (dn.ar_code[ai] == AR_SINWT_OFFSET) off = kn_sat_u32(__dmul_rn((double)x, 65536.0));
                        else pv[dn.ar_code[ai] - AR_POST] = x;
                    }
                    float y = sinwt_tick(phase, off, inc, a.sine_table);
                    EMIT(f, 0, y)
                }
                }
                sreg[rb * 32] = phase;
                // audio-rate routes leave their last value in the ugen, like param_apply does
                if (dn.n_ar) { sreg[(rb + 1) * 32] = off; sreg[(rb + 2) * 32] = inc; }
                break;
            }
            case DK_SINNUM: {
                float phase = __uint_as_float(sreg[rb * 32]), off = __uint_as_float(sreg[(rb + 1) * 32]),
                      inc = __uint_as_float(sreg[(rb + 2) * 32]);
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        PLAIN16(sinnum_tick(phase, off, inc))
                        continue;
                    }
                    if (GROUP_PLAIN_AR) {
                        LOAD16(xf_, ar_s0)
                        LOAD16(xo_, ar_s1)
                        auto tk = [&](int k) {
                            if (ar_s0 >= 0) inc = xf_[k] / sr; // osc.rs:240-242
                            if (ar_s1 >= 0) off = xo_[k];
                            return sinnum_tick(phase, off, inc);
                        };
                        PLAIN16(tk(k))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, sreg[rb * 32] = __float_as_uint(phase),
                              (phase = __uint_as_float(sreg[rb * 32]), off = __uint_as_float(sreg[(rb + 1) * 32]),
                               inc = __uint_as_float(sreg[(rb + 2) * 32])))
                    for (int ai = 0; ai < dn.n_ar; ai++) {
                        float x = RDV(dn.ar_slot[ai], f);
                        if (dn.ar_code[ai] == AR_SINNUM_FREQ) inc = x / sr; // osc.rs:240-242
                        else if (dn.ar_code[ai] == AR_SINNUM_OFFSET) off = x;
                        else pv[dn.ar_code[ai] - AR_POST] = x;
                    }
                    float y = sinnum_tick(phase, off, inc);
                    EMIT(f, 0, y)
                }
                }
                sreg[rb * 32] = __float_as_uint(phase);
                if (dn.n_ar) { sreg[(rb + 1) * 32] = __float_as_uint(off); sreg[(rb + 2) * 32] = __float_as_uint(inc); }
                break;
            }
            case DK_POLYBLEP: {
                float t = __uint_as_float(sreg[rb * 32]), dt = __uint_as_float(sreg[(rb + 1) * 32]);
                uint32_t use_sin = sreg[(rb + 2) * 32];
                float pw = __uint_as_float(sreg[(rb + 3) * 32]);
                uint32_t wf = sreg[(rb + 4) * 32];
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        if (__all_sync(0xFFFFFFFFu, wf == 0u && !use_sin)) { // every lane a sawtooth below sr/4
                            if (__all_sync(0xFFFFFFFFu, saw_domain(t, dt))) { // the fused recipe's 15-instruction form (hoisted reciprocal)
                                const float omd = 1.0f - dt, rc = div_prep(dt);
                                PLAIN16(saw_fast_tick(t, dt, omd, rc))
                            } else PLAIN16(polyblep_saw_tick_sel(t, dt))
                        }
                        else PLAIN16(polyblep_tick(t, dt, use_sin, pw, wf))
                        continue;
                    }
                    if (GROUP_PLAIN_AR) {
                        LOAD16(xf_, ar_s0)
                        LOAD16(xo_, ar_s1)
                        auto tk = [&](int k) {
                            if (ar_s0 >= 0) {
                                dt = xf_[k] / sr;
                                use_sin = (dt * sr >= sr / 4.0f) ? 1u : 0u;
                            }
                            if (ar_s1 >= 0) pw = xo_[k];
                            return polyblep_tick(t, dt, use_sin, pw, wf);
                        };
                        PLAIN16(tk(k))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, sreg[rb * 32] = __float_as_uint(t),
                              (t = __uint_as_float(sreg[rb * 32]), dt = __uint_as_float(sreg[(rb + 1) * 32]), use_sin = sreg[(rb + 2) * 32],
                               pw = __uint_as_float(sreg[(rb + 3) * 32]), wf = sreg[(rb + 4) * 32]))
                    for (int ai = 0; ai < dn.n_ar; ai++) {
                        float x = RDV(dn.ar_slot[ai], f);
                        if (dn.ar_code[ai] == AR_POLYBLEP_FREQ) {
                            dt = x / sr;
                            use_sin = (dt * sr >= sr / 4.0f) ? 1u : 0u;
                        } else if (dn.ar_code[ai] == AR_POLYBLEP_PW) {
                            pw = x;
                        } else pv[dn.ar_code[ai] - AR_POST] = x;
                    }
                    float y = polyblep_tick(t, dt, use_sin, pw, wf);
                    EMIT(f, 0, y)
                }
                }
                sreg[rb * 32] = __float_as_uint(t);
                if (dn.n_ar) {
                    sreg[(rb + 1) * 32] = __float_as_uint(dt);
                    sreg[(rb + 2) * 32] = use_sin;
                    sreg[(rb + 3) * 32] = __float_as_uint(pw);
                }
                break;
            }
            case DK_SVF: {
                float ic1, ic2, a1, a2, a3, m0, m1, m2;
#define SVF_LOAD (ic1 = __uint_as_float(sreg[rb * 32]), ic2 = __uint_as_float(sreg[(rb + 1) * 32]),       \
                  a1 = __uint_as_float(sreg[(rb + 2) * 32]), a2 = __uint_as_float(sreg[(rb + 3) * 32]),    \
                  a3 = __uint_as_float(sreg[(rb + 4) * 32]), m0 = __uint_as_float(sreg[(rb + 5) * 32]),    \
                  m1 = __uint_as_float(sreg[(rb + 6) * 32]), m2 = __uint_as_float(sreg[(rb + 7) * 32]))
#define SVF_STORE (sreg[rb * 32] = __float_as_uint(ic1), sreg[(rb + 1) * 32] = __float_as_uint(ic2))
                SVF_LOAD;
                const int is = dn.in_slot[0];
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        LOAD16(x_, is)
                        PLAIN16(svf_tick(x_[k], ic1, ic2, a1, a2, a3, m0, m1, m2))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, SVF_STORE, SVF_LOAD)
                    AR_POST_ROUTES(f)
                    // audio-rate routes into cutoff / q / gain (regs 8..10, type in 11): set_coeffs every frame, svf.rs:81-109
                    bool recalc = false;
                    for (int ai = 0; ai < dn.n_ar; ai++) {
                        const uint32_t code = dn.ar_code[ai];
                        if (code >= AR_SVF_CUTOFF && code <= AR_SVF_GAIN) {
                            sreg[(rb + 8 + (code - AR_SVF_CUTOFF)) * 32] = __float_as_uint(RDV(dn.ar_slot[ai], f));
                            recalc = true;
                        }
                    }
                    if (recalc)
                        svf_coeffs_dev(sreg[(rb + 11) * 32], __uint_as_float(sreg[(rb + 8) * 32]), __uint_as_float(sreg[(rb + 9) * 32]),
                                       __uint_as_float(sreg[(rb + 10) * 32]), sr, a1, a2, a3, m0, m1, m2);
                    float x = RDV(is, f);
                    float y = svf_tick(x, ic1, ic2, a1, a2, a3, m0, m1, m2);
                    EMIT(f, 0, y)
                }
                }
                SVF_STORE;
                if (dn.n_ar) { // routed coefficients persist like a param_apply would
                    sreg[(rb + 2) * 32] = __float_as_uint(a1); sreg[(rb + 3) * 32] = __float_as_uint(a2); sreg[(rb + 4) * 32] = __float_as_uint(a3);
                    sreg[(rb + 5) * 32] = __float_as_uint(m0); sreg[(rb + 6) * 32] = __float_as_uint(m1); sreg[(rb + 7) * 32] = __float_as_uint(m2);
                }
                break;
            }
            case DK_ONEPOLE_LP:
            case DK_ONEPOLE_HP: {
                float y1 = __uint_as_float(sreg[rb * 32]), a0 = __uint_as_float(sreg[(rb + 1) * 32]), b1 = __uint_as_float(sreg[(rb + 2) * 32]);
                const int is = dn.in_slot[0];
                const bool hp = dn.kind == DK_ONEPOLE_HP;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        LOAD16(x_, is)
                        if (hp) PLAIN16(onepole_hp_tick(x_[k], y1, a0, b1))
                        else PLAIN16(onepole_lp_tick(x_[k], y1, a0, b1))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, sreg[rb * 32] = __float_as_uint(y1),
                              (y1 = __uint_as_float(sreg[rb * 32]), a0 = __uint_as_float(sreg[(rb + 1) * 32]), b1 = __uint_as_float(sreg[(rb + 2) * 32])))
                    AR_POST_ROUTES(f)
                    for (int ai = 0; ai < dn.n_ar; ai++)
                        if (dn.ar_code[ai] == AR_ONEPOLE_CUTOFF) onepole_coeffs_dev(RDV(dn.ar_slot[ai], f), sr, a0, b1); // onepole.rs:135-139
                    float x = RDV(is, f);
                    float y = hp ? onepole_hp_tick(x, y1, a0, b1) : onepole_lp_tick(x, y1, a0, b1);
                    EMIT(f, 0, y)
                }
                }
                sreg[rb * 32] = __float_as_uint(y1);
                if (dn.n_ar) { sreg[(rb + 1) * 32] = __float_as_uint(a0); sreg[(rb + 2) * 32] = __float_as_uint(b1); }
                break;
            }
            case DK_ENVASR:
            case DK_ENVAR: {
                uint32_t st;
                float t, ar, rr, sc;
#define ENV_LOAD (st = sreg[rb * 32], t = __uint_as_float(sreg[(rb + 1) * 32]), ar = __uint_as_float(sreg[(rb + 2) * 32]), \
                  rr = __uint_as_float(sreg[(rb + 3) * 32]), sc = __uint_as_float(sreg[(rb + 4) * 32]))
#define ENV_STORE (sreg[rb * 32] = st, sreg[(rb + 1) * 32] = __float_as_uint(t), sreg[(rb + 2) * 32] = __float_as_uint(ar), \
                   sreg[(rb + 3) * 32] = __float_as_uint(rr), sreg[(rb + 4) * 32] = __float_as_uint(sc))
                ENV_LOAD;
                const bool asr = dn.kind == DK_ENVASR;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        if (asr) PLAIN16(envasr_tick_sel(st, t, ar, rr, sc))
                        else PLAIN16(envar_tick(st, t, ar, rr, sc))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, ENV_STORE, ENV_LOAD)
                    AR_POST_ROUTES(f)
                    for (int ai = 0; ai < dn.n_ar; ai++) { // envelopes.rs:84-111: F::ONE / (seconds * sample_rate), 1 for 0 s
                        if (dn.ar_code[ai] == AR_ENV_ATTACK) ar = env_rate_dev(RDV(dn.ar_slot[ai], f), sr);
                        else if (dn.ar_code[ai] == AR_ENV_RELEASE) rr = env_rate_dev(RDV(dn.ar_slot[ai], f), sr);
                    }
                    float y = asr ? envasr_tick(st, t, ar, rr, sc) : envar_tick(st, t, ar, rr, sc);
                    EMIT(f, 0, y)
                }
                }
                ENV_STORE;
                break;
            }
            case DK_ENVELOPE: { // envelopes.rs:407-463
                uint32_t running, seg;
                double time, from, step;
#define ENVL_LOAD (running = sreg[rb * 32], seg = sreg[(rb + 1) * 32], time = ld_d(sreg, rb + 2), from = ld_d(sreg, rb + 4), step = ld_d(sreg, rb + 6))
#define ENVL_STORE (sreg[rb * 32] = running, sreg[(rb + 1) * 32] = seg, st_d(sreg, rb + 2, time), st_d(sreg, rb + 4, from))
                ENVL_LOAD;
                const uint32_t n_seg = dn.n_seg;
                const bool looping = dn.looping;
                auto env_tick = [&]() -> float {
                    float y;
                    if (!running) {
                        y = (float)from;
                    } else {
                        const uint32_t sb = rb + REGS_ENVELOPE_BASE + REGS_ENVELOPE_PER_SEG * seg;
                        const double recip = ld_d(sreg, sb), dur = ld_d(sreg, sb + 2), val = ld_d(sreg, sb + 4);
                        if (time < dur) {
                            y = (float)__dadd_rn(from, __dmul_rn(__dmul_rn(time, recip), __dsub_rn(val, from)));
                            time = __dadd_rn(time, step);
                        } else if (seg + 1 < n_seg) {
                            from = val;
                            y = (float)__dadd_rn(from, __dmul_rn(__dmul_rn(time, recip), __dsub_rn(val, from)));
                            seg = seg + 1;
                            time = __dadd_rn(__dsub_rn(time, dur), step);
                        } else {
                            from = val;
                            y = (float)from;
                            if (looping) {
                                seg = 0;
                                time = 0.0;
                            } else running = 0;
                        }
                    }
                    return y;
                };
                const double isr = dn.n_ar ? 1.0 / (double)sr : 0.0; // (f64)(f32)sr is the integer rate: the host's 1 / sr exactly
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        PLAIN16(env_tick())
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                        EVENTS_AT(f, ENVL_STORE, ENVL_LOAD)
                        AR_POST_ROUTES(f)
                        for (int ai = 0; ai < dn.n_ar; ai++) // envelopes.rs:477-479
                            if (dn.ar_code[ai] == AR_ENVELOPE_TIME_SCALE) step = __dmul_rn((double)RDV(dn.ar_slot[ai], f), isr);
                        float y = env_tick();
                        EMIT(f, 0, y)
                    }
                }
                ENVL_STORE;
                if (dn.n_ar) st_d(sreg, rb + 6, step);
                break;
            }
            case DK_MATH: {
                const uint32_t nch = dn.n_out;
                FOR_GROUPS {
                    if (GROUP_PLAIN && nch == 1) {
                        const int sa = dn.in_slot[0], sb = dn.in_slot[1];
                        LOAD16(a_, sa)
                        LOAD16(b_, sb)
                        switch (dn.mode) { // the operation is chosen once per group, not once per frame
                        case 0: PLAIN16(a_[k] + b_[k]) break;
                        case 1: PLAIN16(a_[k] - b_[k]) break;
                        case 2: PLAIN16(a_[k] * b_[k]) break;
                        case 3: PLAIN16(a_[k] / b_[k]) break;
                        default: PLAIN16(math_apply(4, a_[k], b_[k])) break;
                        }
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, (void)0, (void)0)
                    AR_POST_ROUTES(f)
                    float ain[MAX_IN];
#pragma unroll
                    for (int c = 0; c < MAX_IN; c++) ain[c] = c < 2 * (int)nch ? RDV(dn.in_slot[c], f) : 0.f;
#pragma unroll
                    for (int c = 0; c < MAX_OUT; c++)
                        if (c < (int)nch) {
                            float y = math_apply(dn.mode, ain[c], ain[c + nch]);
                            EMIT(f, c, y)
                        }
                }
                }
                break;
            }
            case DK_MATH1: {
                const int is = dn.in_slot[0];
                const uint32_t op1 = dn.mode;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        LOAD16(x_, is)
                        PLAIN16(math1_apply(op1, x_[k]))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                        EVENTS_AT(f, (void)0, (void)0)
                        AR_POST_ROUTES(f)
                        float y = math1_apply(op1, RDV(is, f));
                        EMIT(f, 0, y)
                    }
                }
                break;
            }
            case DK_PHASOR: {
                double phase = ld_d(sreg, rb), step = ld_d(sreg, rb + 2);
                const double isr = dn.n_ar ? 1.0 / (double)sr : 0.0;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        PLAIN16(phasor_tick(phase, step))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                        EVENTS_AT(f, st_d(sreg, rb, phase), (phase = ld_d(sreg, rb), step = ld_d(sreg, rb + 2)))
                        AR_POST_ROUTES(f)
                        for (int ai = 0; ai < dn.n_ar; ai++) // osc.rs:191-197
                            if (dn.ar_code[ai] == AR_PHASOR_FREQ) step = __dmul_rn((double)RDV(dn.ar_slot[ai], f), isr);
                        float y = phasor_tick(phase, step);
                        EMIT(f, 0, y)
                    }
                }
                st_d(sreg, rb, phase);
                if (dn.n_ar) st_d(sreg, rb + 2, step);
                break;
            }
            case DK_WHITE:
            case DK_BROWN: { // noise.rs:26-46,122-153 (no parameters: only wrapper events can be due)
                uint64_t rng = ((uint64_t)sreg[(rb + 1) * 32] << 32) | sreg[rb * 32];
                float last = dn.kind == DK_BROWN ? __uint_as_float(sreg[(rb + 2) * 32]) : 0.f;
                const bool brown = dn.kind == DK_BROWN;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        if (brown) PLAIN16(brown_tick(rng, last))
                        else PLAIN16(white_sample(rng))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                        EVENTS_AT(f, (void)0, (void)0)
                        AR_POST_ROUTES(f)
                        float y = brown ? brown_tick(rng, last) : white_sample(rng);
                        EMIT(f, 0, y)
                    }
                }
                sreg[rb * 32] = (uint32_t)rng;
                sreg[(rb + 1) * 32] = (uint32_t)(rng >> 32);
                if (dn.kind == DK_BROWN) sreg[(rb + 2) * 32] = __float_as_uint(last);
                break;
            }
            case DK_PINK: { // noise.rs:94-114; white_noises[] stays in the lane's shared-memory registers
                uint64_t rng = ((uint64_t)sreg[(rb + 1) * 32] << 32) | sreg[rb * 32];
                uint32_t counter = sreg[(rb + 12) * 32];
                float pink = __uint_as_float(sreg[(rb + 13) * 32]), always = __uint_as_float(sreg[(rb + 11) * 32]);
                auto pink_tick = [&]() -> float {
                    const uint32_t idx = (uint32_t)(__ffs((int)counter) - 1); // counter.trailing_zeros(), 0..8
                    pink = pink - __uint_as_float(sreg[(rb + 2 + idx) * 32]);
                    const float w = white_sample(rng);
                    sreg[(rb + 2 + idx) * 32] = __float_as_uint(w);
                    pink = pink + w;
                    pink = pink - always;
                    always = white_sample(rng);
                    pink = pink + always;
                    counter = (counter & 255u) + 1u;                           // mask = 2^(9-1) = 256
                    return pink / 10.0f;                                       // PINK_NOISE_OCTAVES + 1
                };
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        PLAIN16(pink_tick())
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                        EVENTS_AT(f, (void)0, (void)0)
                        AR_POST_ROUTES(f)
                        float y = pink_tick();
                        EMIT(f, 0, y)
                    }
                }
                sreg[rb * 32] = (uint32_t)rng;
                sreg[(rb + 1) * 32] = (uint32_t)(rng >> 32);
                sreg[(rb + 11) * 32] = __float_as_uint(always);
                sreg[(rb + 12) * 32] = counter;
                sreg[(rb + 13) * 32] = __float_as_uint(pink);
                break;
            }
            case DK_RANDLIN: { // noise.rs:186-203
                uint64_t rng = ((uint64_t)sreg[(rb + 1) * 32] << 32) | sreg[rb * 32];
                float cur = __uint_as_float(sreg[(rb + 2) * 32]), width = __uint_as_float(sreg[(rb + 3) * 32]),
                      phase = __uint_as_float(sreg[(rb + 4) * 32]), step = __uint_as_float(sreg[(rb + 5) * 32]);
                const float isr = dn.n_ar ? 1.0f / sr : 0.0f;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        PLAIN16(randlin_tick(rng, cur, width, phase, step))
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                        EVENTS_AT(f, (void)0, step = __uint_as_float(sreg[(rb + 5) * 32]))
                        AR_POST_ROUTES(f)
                        for (int ai = 0; ai < dn.n_ar; ai++) // noise.rs:206-213
                            if (dn.ar_code[ai] == AR_RANDLIN_FREQ) step = RDV(dn.ar_slot[ai], f) * isr;
                        float y = randlin_tick(rng, cur, width, phase, step);
                        EMIT(f, 0, y)
                    }
                }
                sreg[rb * 32] = (uint32_t)rng;
                sreg[(rb + 1) * 32] = (uint32_t)(rng >> 32);
                sreg[(rb + 2) * 32] = __float_as_uint(cur);
                sreg[(rb + 3) * 32] = __float_as_uint(width);
                sreg[(rb + 4) * 32] = __float_as_uint(phase);
                if (dn.n_ar) sreg[(rb + 5) * 32] = __float_as_uint(step);
                break;
            }
            case DK_PAN2: { // pan.rs:31-36: [signal * left_gain, signal * right_gain]
                float gl = __uint_as_float(sreg[rb * 32]), gr = __uint_as_float(sreg[(rb + 1) * 32]);
                const int is = dn.in_slot[0];
                for (uint32_t f = 0; f < nf; f++) {
                    EVENTS_AT(f, (void)0, (gl = __uint_as_float(sreg[rb * 32]), gr = __uint_as_float(sreg[(rb + 1) * 32])))
                    AR_POST_ROUTES(f)
                    for (int ai = 0; ai < dn.n_ar; ai++) // pan.rs:26-36: the gains of the routed pan position, every frame
                        if (dn.ar_code[ai] == AR_PAN2_PAN) pan2_gains(RDV(dn.ar_slot[ai], f) * 0.5f + 0.5f, gl, gr);
                    const float x = RDV(is, f);
                    EMIT(f, 0, x * gl)
                    EMIT(f, 1, x * gr)
                }
                if (dn.n_ar) { sreg[rb * 32] = __float_as_uint(gl); sreg[(rb + 1) * 32] = __float_as_uint(gr); }
                break;
            }
            case DK_CONST:
            case DK_INPLUS: {
                float val = __uint_as_float(sreg[rb * 32]);
                const int is = dn.kind == DK_INPLUS ? dn.in_slot[0] : -1;
                FOR_GROUPS {
                    if (GROUP_PLAIN) {
                        if (dn.kind == DK_INPLUS) {
                            LOAD16(x_, is)
                            PLAIN16(val + x_[k])
                        } else {
                            PLAIN16(val)
                        }
                        continue;
                    }
                    for (uint32_t f = g0_; f < fe_; f++) {
                    EVENTS_AT(f, (void)0, val = __uint_as_float(sreg[rb * 32]))
                    for (int ai = 0; ai < dn.n_ar; ai++) {
                        float x = RDV(dn.ar_slot[ai], f);
                        if (dn.ar_code[ai] == AR_REG0) val = x;
                        else pv[dn.ar_code[ai] - AR_POST] = x;
                    }
                    float y = val;
                    if (dn.kind == DK_INPLUS) y = val + RDV(is, f);
                    EMIT(f, 0, y)
                }
                }
                if (dn.n_ar) sreg[rb * 32] = __float_as_uint(val);
                break;
            }
            default: break;
            }
            // an audio-rate route into a wrapper value persists like a param_apply would
            for (int ai = 0; ai < dn.n_ar; ai++)
                if (dn.ar_code[ai] >= AR_POST) sreg[dn.post_reg[dn.ar_code[ai] - AR_POST] * 32] = __float_as_uint(pv[dn.ar_code[ai] - AR_POST]);
            // events due in this chunk but after its last processed frame cannot exist (sorted by chunk)
        }
        // mix bus: per-warp partial sums in a fixed order => deterministic
        if ((CH & 15u) == 0 && nf == CH) {
            // lane f < 16 sums frame g0 + f of the chunk over the warp's active voices straight from the value
            // slots ([slot][frame][lane] in shared memory), four accumulators, columns visited from lane f
            // onwards so that the readers hit different banks.  The order is a function of the frame's position
            // in its chunk only, and chunks start on block boundaries: independent of how a render is split.
            __syncwarp();
            const float *vbase = reinterpret_cast<const float *>(smem + n_regs * 32);
            const uint32_t na = min(32u, a.n_voices - warp * 32);
            for (uint32_t u = 0; u < prog->n_ubus; u++)
                for (uint32_t g0 = 0; g0 < CH; g0 += 16) {
                    const float *row = vbase + ((size_t)prog->ubus_slot[u] * CH + g0 + (lane & 15u)) * 32;
                    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        const uint32_t col = (j + lane) & 31u;
                        const float x = row[col];
                        acc[j & 3] = acc[j & 3] + (col < na ? x : 0.f);
                    }
                    if (lane < 16) a.partials[(size_t)(a.row0 + warp * prog->n_ubus + u) * a.n_frames + c0 + g0 + lane] = (acc[0] + acc[1]) + (acc[2] + acc[3]);
                }
        } else
        for (uint32_t u = 0; u < prog->n_ubus; u++) {
            const uint32_t slot = prog->ubus_slot[u];
            float mine = 0.f;
            for (uint32_t f = 0; f < nf; f++) {
                float x = active ? sval[(slot * CH + f) * 32] : 0.f;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x = x + __shfl_xor_sync(0xFFFFFFFFu, x, o);
                if (lane == (f & 31)) mine = x;
                if ((f & 31) == 31 || f + 1 == nf) {
                    const uint32_t fbase = f & ~31u;
                    if (lane <= (f & 31)) a.partials[(size_t)(a.row0 + warp * prog->n_ubus + u) * a.n_frames + c0 + fbase + lane] = mine;
                }
            }
        }
        for (uint32_t ti = 0; ti < a.n_taps; ti++) {
            const DevTap tp = a.taps[ti];
            if (tp.voice == v)
                for (uint32_t f = 0; f < nf; f++) a.tap_out[(size_t)tp.tap * a.tap_stride + a.tap_frame0 + c0 + f] = sval[(tp.slot * CH + f) * 32];
        }
        __syncwarp();
    }
    if (active)
        for (uint32_t r = 0; r < n_regs; r++) a.regs[(size_t)r * a.n_voices + v] = sreg[r * 32];
}

// out[block][ch][i] = sum over the partial rows feeding ch (graph.rs:850-864 as a fixed tree):
// the rows are cut into RB_GROUPS contiguous groups, each summed in row order by one thread per
// frame (a warp reads 32 consecutive frames of a row: one 128-byte line), and the group sums are
// folded left to right.  The order depends on n_rows only, so a render is bit-identical however it
// is split into launches.  `out` may be peer memory (the multi-GPU bus slot on rank 0).
constexpr int RB_GROUPS = 8, RB_FRAMES = 32;
__global__ void __launch_bounds__(RB_GROUPS *RB_FRAMES) reduce_bus(const float *__restrict__ partials, const uint32_t *__restrict__ row_mask,
                                                                    uint32_t n_rows, uint32_t n_frames, float *__restrict__ out,
                                                                    uint32_t n_out, uint32_t block_size) {
    __shared__ float part[RB_GROUPS][MAX_BUS][RB_FRAMES];
    const uint32_t fi = threadIdx.x & (RB_FRAMES - 1), g = threadIdx.x / RB_FRAMES;
    const uint32_t t = blockIdx.x * RB_FRAMES + fi;
    const uint32_t per = (n_rows + RB_GROUPS - 1) / RB_GROUPS;
    const uint32_t r0 = min(n_rows, g * per), r1 = min(n_rows, r0 + per);
    float acc[MAX_BUS];
#pragma unroll
    for (int c = 0; c < MAX_BUS; c++) acc[c] = 0.f;
    if (t < n_frames) {
        const float *src = partials + t;
        uint32_t r = r0;
        for (; r + 4 <= r1; r += 4) { // four loads in flight per thread
            const float x0 = src[(size_t)r * n_frames], x1 = src[(size_t)(r + 1) * n_frames];
            const float x2 = src[(size_t)(r + 2) * n_frames], x3 = src[(size_t)(r + 3) * n_frames];
            const uint32_t m0 = row_mask[r], m1 = row_mask[r + 1], m2 = row_mask[r + 2], m3 = row_mask[r + 3];
#pragma unroll
            for (int c = 0; c < MAX_BUS; c++) {
                if ((m0 >> c) & 1u) acc[c] = acc[c] + x0;
                if ((m1 >> c) & 1u) acc[c] = acc[c] + x1;
                if ((m2 >> c) & 1u) acc[c] = acc[c] + x2;
                if ((m3 >> c) & 1u) acc[c] = acc[c] + x3;
            }
        }
        for (; r < r1; r++) {
            const float x = src[(size_t)r * n_frames];
            const uint32_t m = row_mask[r];
#pragma unroll
            for (int c = 0; c < MAX_BUS; c++)
                if ((m >> c) & 1u) acc[c] = acc[c] + x;
        }
    }
#pragma unroll
    for (int c = 0; c < MAX_BUS; c++)
        if (c < (int)n_out) part[g][c][fi] = acc[c];
    __syncthreads();
    // thread (g = channel slot, fi): folds the groups of one channel of one frame
    for (uint32_t c = g; c < n_out; c += RB_GROUPS) {
        float sum = part[0][c][fi];
#pragma unroll
        for (int k = 1; k < RB_GROUPS; k++) sum = sum + part[k][c][fi];
        if (t < n_frames) {
            const uint32_t blk = t / block_size, i = t % block_size;
            out[((size_t)blk * n_out + c) * block_size + i] = sum;
        }
    }
}

// Internal signals (plan.hpp): sig[w][t] = sum, in row order, of the partial rows whose mask carries bit first_bit + which[w].
// One thread per frame; a handful of signals, each summed by its own pass over the rows (deterministic).
__global__ void reduce_signals(const float *__restrict__ partials, const uint32_t *__restrict__ row_mask, uint32_t n_rows, uint32_t n_frames,
                               float *__restrict__ sig, uint32_t first_bit, const uint32_t *__restrict__ which, uint32_t n_which) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_frames) return;
    for (uint32_t w = 0; w < n_which; w++) {
        const uint32_t sgn = which[w], bit = 1u << (first_bit + sgn);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        uint32_t k = 0;
        for (uint32_t r = 0; r < n_rows; r++) {
            if (!(row_mask[r] & bit)) continue;
            const float x = partials[(size_t)r * n_frames + t];
            switch (k & 3u) {
            case 0: a0 = a0 + x; break;
            case 1: a1 = a1 + x; break;
            case 2: a2 = a2 + x; break;
            default: a3 = a3 + x; break;
            }
            k++;
        }
        sig[(size_t)sgn * n_frames + t] = (a0 + a1) + (a2 + a3);
    }
}

// graph inputs that reach a graph output without a node in between (graph_tests.rs:49-79): added to the reduced bus
__global__ void add_inputs(const float *__restrict__ sig, uint32_t n_frames, float *__restrict__ out, uint32_t n_out, uint32_t block_size,
                           const uint32_t *__restrict__ pairs, uint32_t n_pairs) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_frames) return;
    const uint32_t blk = t / block_size, i = t % block_size;
    for (uint32_t k = 0; k < n_pairs; k++) {
        float *o = out + ((size_t)blk * n_out + pairs[2 * k + 1]) * block_size + i;
        *o = *o + sig[(size_t)pairs[2 * k] * n_frames + t];
    }
}

// ---- multi-GPU mix bus over peer memory (NVLink) ------------------------------------------------
// Every rank's reduce_bus writes its bus straight into its slot of a buffer in rank 0's memory;
// signal_flag then publishes "launch L of epoch E is there" with a system-scope release store, and
// rank 0's sum_slots waits for all ranks' flags before it folds the slots (rank order: fixed).
// Spins give up after ~2 s and raise *timeout_flag instead of hanging the device.
KN_DEV uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
KN_DEV void st_release_sys(uint32_t *p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
// epochs are compared as signed distances so that the counter may wrap
KN_DEV bool spin_until_at_least(const uint32_t *flag, uint32_t epoch, uint32_t *timeout_flag) {
    const long long t0 = clock64();
    while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
        if (clock64() - t0 > 4000000000ll) {
            if (timeout_flag) *timeout_flag = 1u;
            return false;
        }
        __nanosleep(200);
    }
    return true;
}

__global__ void signal_flag(uint32_t *flag, uint32_t value) {
    __threadfence_system();
    st_release_sys(flag, value);
}
__global__ void wait_flag(const uint32_t *flag, uint32_t value, uint32_t *timeout_flag) { spin_until_at_least(flag, value, timeout_flag); }

__global__ void sum_slots(const float *__restrict__ slots, size_t slot_stride, uint32_t world, const uint32_t *flags, uint32_t flag_stride,
                          uint32_t epoch, float *__restrict__ out, size_t n, uint32_t *timeout_flag) {
    if (threadIdx.x == 0)
        for (uint32_t r = 0; r < world; r++) spin_until_at_least(flags + (size_t)r * flag_stride, epoch, timeout_flag);
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float acc = slots[i];
        for (uint32_t r = 1; r < world; r++) acc = acc + slots[(size_t)r * slot_stride + i];
        out[i] = acc;
    }
}

// host-callable launchers ---------------------------------------------------------------------
cudaError_t launch_interp(const InterpArgs &a, uint32_t n_regs, uint32_t n_slots, cudaStream_t stream) {
    const uint32_t n_warps = (a.n_voices + 31) / 32;
    const size_t smem = ((size_t)n_regs + (size_t)n_slots * a.chunk) * 32 * sizeof(uint32_t);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(render_interp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    render_interp<<<n_warps, 32, smem, stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_reduce_bus(const float *partials, const uint32_t *row_mask, uint32_t n_rows, uint32_t n_frames, float *out,
                              uint32_t n_out, uint32_t block_size, cudaStream_t stream) {
    reduce_bus<<<(n_frames + RB_FRAMES - 1) / RB_FRAMES, RB_GROUPS * RB_FRAMES, 0, stream>>>(partials, row_mask, n_rows, n_frames, out, n_out, block_size);
    return cudaGetLastError();
}
cudaError_t launch_reduce_signals(const float *partials, const uint32_t *row_mask, uint32_t n_rows, uint32_t n_frames, float *sig,
                                  uint32_t first_bit, const uint32_t *which, uint32_t n_which, cudaStream_t stream) {
    reduce_signals<<<(n_frames + 127) / 128, 128, 0, stream>>>(partials, row_mask, n_rows, n_frames, sig, first_bit, which, n_which);
    return cudaGetLastError();
}
cudaError_t launch_add_inputs(const float *sig, uint32_t n_frames, float *out, uint32_t n_out, uint32_t block_size, const uint32_t *pairs,
                              uint32_t n_pairs, cudaStream_t stream) {
    add_inputs<<<(n_frames + 127) / 128, 128, 0, stream>>>(sig, n_frames, out, n_out, block_size, pairs, n_pairs);
    return cudaGetLastError();
}
cudaError_t launch_signal_flag(uint32_t *flag, uint32_t value, cudaStream_t stream) {
    signal_flag<<<1, 1, 0, stream>>>(flag, value);
    return cudaGetLastError();
}
cudaError_t launch_wait_flag(const uint32_t *flag, uint32_t value, uint32_t *timeout_flag, cudaStream_t stream) {
    wait_flag<<<1, 1, 0, stream>>>(flag, value, timeout_flag);
    return cudaGetLastError();
}
cudaError_t launch_sum_slots(const float *slots, size_t slot_stride, uint32_t world, const uint32_t *flags, uint32_t flag_stride, uint32_t epoch,
                             float *out, size_t n, uint32_t *timeout_flag, cudaStream_t stream) {
    const uint32_t threads = 256;
    const uint32_t blocks = (uint32_t)std::min<size_t>((n + threads - 1) / threads, 148 * 4);
    sum_slots<<<std::max(1u, blocks), threads, 0, stream>>>(slots, slot_stride, world, flags, flag_stride, epoch, out, n, timeout_flag);
    return cudaGetLastError();
}

#ifndef KGPU_HAVE_FUSED
int match_fused_recipe(const DevProgram &, uint32_t) { return -1; }
size_t fused_scratch_bytes(int, uint32_t, uint32_t, uint32_t) { return 0; }
const char *fused_recipe_name(int) { return "render_interp"; }
uint32_t fused_rows(int, uint32_t, uint32_t) { return 0; }
bool sub_scan_applies(uint32_t, uint32_t) { return false; }
cudaError_t launch_fused(int, const FusedArgs &, cudaStream_t) { return cudaErrorNotSupported; }
#endif

} // namespace kgpu
