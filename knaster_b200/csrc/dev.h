// dev.h -- POD structures shared by the host plan/event compilers and the CUDA kernels.
#pragma once
#include <stdint.h>

namespace kgpu {

// ---- per-voice register layout (32-bit registers, SoA [reg][voice] in HBM) -------------
// Node kinds as the device sees them.
enum DevKind : uint8_t {
    DK_SINWT = 1,    // regs: 0 phase(u32) 1 phase_offset(u32) 2 phase_increment(u32)      osc.rs:97-105
    DK_SINNUM = 2,   // regs: 0 phase 1 phase_offset 2 phase_increment (f32)               osc.rs:222-226
    DK_POLYBLEP = 3, // regs: 0 t 1 dt 2 use_sin(u32) 3 pulse_width 4 waveform(u32)        polyblep.rs:128-135
    DK_SVF = 4,      // regs: 0 ic1eq 1 ic2eq 2 a1 3 a2 4 a3 5 m0 6 m1 7 m2                svf.rs:44-59
                     //       with an audio-rate route into cutoff / q / gain also: 8 cutoff 9 q 10 gain_db 11 type(u32)
    DK_ONEPOLE_LP = 5, // regs: 0 last_output 1 a0 2 b1                                    onepole.rs:13-17
    DK_ONEPOLE_HP = 6,
    DK_ENVASR = 7,   // regs: 0 state(u32) 1 t 2 attack_rate 3 release_rate 4 release_scale envelopes.rs:19-28
    DK_ENVAR = 8,    // same layout (state: 0 Stopped 1 Attacking 3 Releasing)             envelopes.rs:174-183
    DK_ENVELOPE = 9, // regs: 0 running(u32) 1 segment(u32) 2,3 time(f64) 4,5 from(f64) 6,7 step(f64)
                     //       then per segment 6 regs: recip(f64) duration(f64) value(f64)  envelopes.rs:322-369
    DK_MATH = 10,    // no regs                                                            math.rs:94-100
    DK_CONST = 11,   // regs: 0 value   (Constant and the TestNumUGen fixture)             util.rs:37-40
    DK_INPLUS = 12,  // regs: 0 number  (TestInPlusParamUGen fixture)
    DK_MATH1 = 13,   // no regs; mode = kgpu_math1_op                                      math.rs:167-305
    DK_PHASOR = 14,  // regs: 0,1 phase(f64) 2,3 step(f64)                                 osc.rs:170-213
    // noise.rs; regs 0,1 = the wyrand state (u64, fastrand 2.3.0)
    DK_WHITE = 15,   // regs: 0,1 rng                                                      noise.rs:26-46
    DK_PINK = 16,    // regs: 0,1 rng 2..10 white_noises[9] 11 always_on 12 counter(u32) 13 pink  noise.rs:53-115
    DK_BROWN = 17,   // regs: 0,1 rng 2 last_output                                        noise.rs:122-153
    DK_RANDLIN = 18, // regs: 0,1 rng 2 current_value 3 current_change_width 4 phase 5 phase_step  noise.rs:156-217
    DK_PAN2 = 19,    // regs: 0 left_gain 1 right_gain (fast::cos / fast::sin of the pan position: evaluated by the host when a
                     //       pan event arrives, by the kernel every frame while pan is routed at audio rate)  pan.rs:12-38
};
enum { REGS_SINWT = 3, REGS_SINNUM = 3, REGS_POLYBLEP = 5, REGS_SVF = 8, REGS_SVF_AR = 12, REGS_ONEPOLE = 3, REGS_ENV = 5,
       REGS_ENVELOPE_BASE = 8, REGS_ENVELOPE_PER_SEG = 6, REGS_CONST = 1, REGS_PHASOR = 4,
       REGS_WHITE = 2, REGS_PINK = 14, REGS_BROWN = 3, REGS_RANDLIN = 6, REGS_PAN2 = 2 };
enum { ASR_STOPPED = 0, ASR_ATTACKING = 1, ASR_SUSTAINING = 2, ASR_RELEASING = 3 };

// arithmetic wrappers applied to a node's outputs, innermost first (wrappers_core/math.rs)
enum PostOp : uint8_t { PO_MUL = 1, PO_ADD = 2, PO_SUB = 3, PO_VSUB = 4, PO_DIV = 5, PO_VDIV = 6, PO_POWF = 7, PO_POWI = 8 };

// audio-rate parameter routes (WrArParams, audio_rate.rs:42-57): what to do with the sample
enum ArCode : uint8_t {
    AR_NONE = 0,
    AR_SINNUM_FREQ = 1,   // inc = v / sr                      osc.rs:240-242
    AR_SINNUM_OFFSET = 2, // phase_offset = v                  osc.rs:245-247
    AR_SINWT_FREQ = 3,    // inc = ((f64)v * k) as u32         osc.rs:127-130
    AR_SINWT_OFFSET = 4,  // offset = ((f64)v * 65536) as u32  osc.rs:133-135
    AR_POLYBLEP_FREQ = 5, // dt = v / sr                       polyblep.rs:163-165,181-184
    AR_REG0 = 6,          // regs[0] = v (Constant.value, TestInPlusParam.number)
    AR_POLYBLEP_PW = 7,   // pulse_width = v                   polyblep.rs:167-170
    // routes into filter parameters: the coefficients are recomputed every frame, as knaster's per-frame param_apply does
    AR_SVF_CUTOFF = 8,    // cutoff = v; set_coeffs            svf.rs:81-89,146-242
    AR_SVF_Q = 9,         // q = v; set_coeffs                 svf.rs:91-99
    AR_SVF_GAIN = 10,     // gain_db = v; set_coeffs           svf.rs:101-109
    AR_ONEPOLE_CUTOFF = 11, // b1 = exp(-2 pi v / sr), a0 = 1 - b1   onepole.rs:35-46,135-139
    // routes into an EnvAsr / EnvAr time: the rate is remade from the sample (idempotent, so the reference's "if changed" guard drops out)
    AR_ENV_ATTACK = 12,   // attack_rate = v == 0 ? 1 : 1 / (v * sr)    envelopes.rs:84-97,246-259
    AR_ENV_RELEASE = 13,  // release_rate likewise                       envelopes.rs:98-111,260-273
    AR_PAN2_PAN = 14,     // pan2_gains(v * 0.5 + 0.5) -> left_gain, right_gain (fastapprox.h)   pan.rs:26-36
    AR_PHASOR_FREQ = 15,  // step = (f64)v * (1 / (f64)sr)              osc.rs:191-197
    AR_RANDLIN_FREQ = 16, // phase_step = v * (1 / sr) (f32)            noise.rs:206-213
    AR_ENVELOPE_TIME_SCALE = 17, // step = (f64)v * (1 / (f64)sr)       envelopes.rs:477-479
    AR_POST = 32,         // AR_POST + k: value of arithmetic wrapper k = v (wr_mul)   math.rs:92-98
};

// Per-voice limits.  A node index inside a template travels as a u8 on the host (RawEvent::local), so 128 nodes leave room;
// the interpreter keeps registers and MAX_SLOTS x 16 frames of value slots of 32 lanes in shared memory:
// (1024 + 32 * 16) * 128 B = 192 KB, under the 227 KB a block may opt into (capi.cpp pick_chunk).
constexpr int MAX_NODES = 128;  // nodes per voice template
constexpr int MAX_IN = 8;       // MathUGen<N<=4>
constexpr int MAX_OUT = 4;
constexpr int MAX_POST = 3;
constexpr int MAX_AR = 6;       // every float parameter of a node: SvfFilter's three + one per WrMul (MAX_POST)
constexpr int MAX_BUS = 8;      // graph outputs
constexpr int MAX_REGS = 1024;  // registers per voice
constexpr int MAX_SLOTS = 32;   // live value slots per voice
// The limits before voices of up to MAX_NODES nodes: a template inside all three is "small".  Voice discovery keeps cutting
// the graph where it did for such voices, and the interpreter keeps their chunk, so graphs that fitted them plan as before.
constexpr int SMALL_VOICE_NODES = 24, SMALL_VOICE_REGS = 192, SMALL_VOICE_SLOTS = 24;

struct DevNode {
    uint8_t kind, mode, n_in, n_out;
    uint16_t reg;                 // first register of this node
    uint16_t n_seg;               // DK_ENVELOPE
    uint16_t out_slot[MAX_OUT];
    int16_t in_slot[MAX_IN];      // -1: unconnected (the permanent zero channel, buffer_allocator.rs:41-48)
    uint8_t n_post, n_ar;
    uint8_t post_op[MAX_POST];
    uint8_t ar_code[MAX_AR];
    uint8_t looping, _pad;
    uint16_t post_reg[MAX_POST];
    int16_t ar_slot[MAX_AR];
};

struct DevProgram {
    uint32_t n_nodes, n_regs, n_slots;
    uint32_t n_ubus;               // distinct voice outputs that reach the mix bus
    uint16_t ubus_slot[MAX_BUS];   // value slot of each
    uint32_t ubus_mask[MAX_BUS];   // graph output channels each one feeds (stereo .out([0,0]) => 0b11)
    float sample_rate;             // F::new(sr as f32)
    float _pad;
    double sinwt_k;                // TABLE_SIZE * FRACTIONAL_PART * (1 / sr)   osc.rs:144-145
    DevNode nodes[MAX_NODES];
};

// ---- device events: the parameter-change queue after the host's control simulation -------
enum DevOp : uint16_t {
    OP_SET = 0,          // regs[reg] = value
    OP_ASR_RELEASE = 1,  // EnvAsr::t_release (envelopes.rs:112-128); reg = node base
    OP_ENV_STOP = 2,     // Envelope t_stop   (envelopes.rs:511-523); reg = node base
    // Envelope triggers as ONE event each instead of a register write per (half) field; the node's register
    // base comes from `node` (interpreter) or is fixed by the recipe (render_sub_seg):
    OP_ENV_RESTART = 3,  // t_restart (envelopes.rs:504-510): running, segment 0, time 0, from_value = the f64 in (reg = lo, value = hi)
    OP_ENV_JUMP = 4,     // jump_to_segment (envelopes.rs:480-503): running, segment = value (already clamped), time 0; reg = node base
    OP_ENV_STEP = 5,     // time_scale (envelopes.rs:477-479): step = time_scale * (1 / sr) = the f64 in (reg = lo, value = hi)
};
struct DevEvent {
    uint32_t frame;  // relative to the first frame of the render call
    uint16_t node;   // node index inside the voice template
    uint16_t op;
    uint32_t reg;
    uint32_t value;
};

struct DevTap {
    uint32_t voice;  // voice index inside the group
    uint32_t slot;   // value slot holding the tapped channel
    uint32_t tap;    // row in the tap output buffer
    uint32_t _pad;
};

constexpr int SINE_TABLE_SIZE = 16384; // wavetable.rs:8-10

} // namespace kgpu
