// fused_scan.cuh -- "render_sub_scan": the subtractive recipe for SMALL banks, time-parallel.
// Included by fused.cu (inside its anonymous namespace, after SubVoice / AsrEnv / EvCursor).
//
// render_sub_asr gives a voice one lane for the whole render: a launch takes as long as ONE voice
// whatever the bank size (14.5 ms per 10 s), so a bank of a few hundred voices leaves > 95 % of the
// machine idle.  Here a voice owns a whole WARP and the lanes are the 32 frames of a chunk:
//
//   pre-pass (sequential, reference rounding order -- SURVEY F5: the f32 phase and envelope ramps
//       drift 4.4e-3 over 10 s if re-associated): t_{k+1} = wrap01(t_k + dt), et_{k+1} = et_k + delta
//       for the chunk's 32 frames, all lanes in step, lane 0 leaves (t_k, et_k) in shared memory;
//   frame-parallel: lane k evaluates saw + blep at t_k (polyblep.rs:490-498) and the envelope at et_k
//       (envelopes.rs:52-81) exactly as the reference does;
//   SvfFilter (svf.rs:245-280) as a chunked linear-recurrence scan: the two states obey
//       s_{k+1} = A s_k + b x_k,  A = [[2 a1 - 1, -2 a2], [2 a2, 1 - 2 a3]],  b = [2 a2, 2 a3]  (SURVEY App. A.4),
//       so the states before every frame of the chunk are s_k = A^k s_0 + sum_{j<k} A^(k-1-j) b x_j: a
//       Hillis-Steele scan of 2-vectors over the warp with shuffle carries (5 rounds; the powers A^(2^r)
//       and A^lane only change when a coefficient does and are kept in registers), then every lane forms its
//       frame's v1, v2 and output from its own pre-update state.  This re-associates the filter's sums:
//       <= 1e-4 against the reference (BASELINE.json's budget for scan-reordered IIR filters; measured
//       ~1e-6), where render_sub_asr is bit-identical.
//
// Measured (256 voices x 10 s, one warp per scheduler): 6.7 ms against 13.0 ms for render_sub_asr.  The chunk is latency-bound:
// the frame-parallel half is a ~320-cycle dependent path (saw, 5 shuffle rounds, state fix-up) and the pre-pass a ~530-cycle
// one (32 x add / compare / subtract); software-pipelining them against each other (PIPE) took 8.1 -> 6.7 ms.  Tried and
// reverted, both parity-clean: running the phase chain without its wrap and redoing only the chunks (later: only the
// frames) behind a wrap -- 7.1 ms, the redo's extra branches and barriers cost what the shorter chain saved; two chunks
// per iteration with independent scans -- 10.0 ms.
//
// Chunks that hold a parameter event, may move the envelope's state machine, or lie outside the
// straight-line domain (other waveforms, dt >= 1/4, ...) run the reference-order per-frame code on
// all lanes instead (a few per note), so events and envelope transitions stay sample-exact.
// One warp per CTA: a bank of V voices is V CTAs spread over all SMs.

constexpr int SCAN_CHUNK = 32;

// wrap_threshold, wrap_flag_const, wrap_flag (the phase recurrence's wrap as a compare on the old phase): csrc/nodes.cuh

struct ScanK {
    float a[4];        // A, row-major
    float b[2];
    float pw[5][4];    // A^(2^r), r = 0..4
    float p32[4];      // A^32
    float pk[4];       // A^lane
    KN_DEV static void mul(const double *x, const double *y, double *z) { // z = x y (2x2, row-major)
        const double z0 = x[0] * y[0] + x[1] * y[2], z1 = x[0] * y[1] + x[1] * y[3];
        const double z2 = x[2] * y[0] + x[3] * y[2], z3 = x[2] * y[1] + x[3] * y[3];
        z[0] = z0; z[1] = z1; z[2] = z2; z[3] = z3;
    }
    // powers in f64 (a handful of operations per coefficient change), rounded once
    KN_DEV void build(float a1, float a2, float a3, uint32_t lane) {
        double A[4] = {2.0 * (double)a1 - 1.0, -2.0 * (double)a2, 2.0 * (double)a2, 1.0 - 2.0 * (double)a3};
        b[0] = 2.0f * a2;
        b[1] = 2.0f * a3;
        double P[4] = {A[0], A[1], A[2], A[3]};
        double K[4] = {1.0, 0.0, 0.0, 1.0};
#pragma unroll
        for (int r = 0; r < 5; r++) {
#pragma unroll
            for (int i = 0; i < 4; i++) pw[r][i] = (float)P[i];
            if ((lane >> r) & 1u) mul(P, K, K);
            mul(P, P, P);
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            a[i] = (float)A[i];
            p32[i] = (float)P[i];
            pk[i] = (float)K[i];
        }
    }
};

template <bool TAPS, bool PIPE>
__global__ void __launch_bounds__(32, 16) render_sub_scan(FusedArgs a) {
    __shared__ float2 pre[2][SCAN_CHUNK];
    const uint32_t lane = threadIdx.x;
    const uint32_t v = blockIdx.x;
    const uint32_t V = a.n_voices;
    constexpr uint32_t FULL = 0xFFFFFFFFu;

    // the voice's registers, identical on every lane
    SubVoice<AsrEnv> s;
    {
        uint32_t r[R_EST];
#pragma unroll
        for (int i = 0; i < R_EST; i++) r[i] = a.regs[(size_t)i * V + v];
#pragma unroll
        for (int i = 0; i < R_EST; i++) s.set_core(i, r[i]);
        s.e.load(a, v);
    }
    uint32_t cur = 0, end = 0, next_frame = 0xFFFFFFFFu;
    if (a.events) {
        cur = a.ev_off[v];
        end = a.ev_off[v + 1];
        if (cur < end) next_frame = __ldg(&a.events[cur].frame);
    }
    float *tap = nullptr;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (a.taps[i].voice == v) tap = a.tap_out + (size_t)a.taps[i].tap * a.tap_stride + a.tap_frame0;
    float *prow = a.partials + (size_t)(a.row0 + v) * a.n_frames;

    ScanK K;
    K.build(s.a1, s.a2, s.a3, lane);
    float omd = 1.0f - s.dt, rc = div_prep(s.dt), tstar = wrap_flag_const(wrap_threshold(s.dt));
    AsrEnv::D d;
    s.e.derive(d);
    const uint32_t NF = a.n_frames;
    const bool writer = lane == 0;

    // the pre-pass of one chunk: the two f32 recurrences, sequentially, in the reference's rounding order.  Every lane
    // runs the same chain (the stores are predicated); lane 0 leaves (t_k, et_k) in `dst`.
    auto prepass = [&](float2 *dst) {
        float t = s.t, et = s.e.et;
#pragma unroll
        for (int k = 0; k < SCAN_CHUNK; k++) {
            if (writer) dst[k] = make_float2(t, et);
            t = (t + s.dt) - wrap_flag(t, tstar);        // inc(), polyblep.rs:232-235: wrap01(t + dt), see wrap_threshold
            et = et + d.delta;         // envelopes.rs:58-66 with the state fixed over the chunk
        }
        s.t = t;
        s.e.et = (d.att || d.rel) ? et : s.e.et;
    };
    // whether the chunk starting at f0 can take the scan path, given the state at its first frame
    auto chunk_fast = [&](uint32_t f0) {
        return f0 + SCAN_CHUNK <= NF && next_frame >= f0 + SCAN_CHUNK && sub_lane_fast(s) && s.e.safe_frames() >= (uint32_t)SCAN_CHUNK;
    };
    // the frame-parallel half of a chunk: lane k renders frame f0 + k from (t_k, et_k)
    auto parallel = [&](const float2 pk, uint32_t f0) {
        const bool ramp = d.att || d.rel;
        const float x = saw_eval(pk.x, s.dt, omd, rc);             // saw + blep, polyblep.rs:490-498
        const float tl = ramp ? pk.y : d.cval;
        const float u = d.rel ? pk.y : 1.0f;
        const float env = (((tl * u) * u) * d.sc2) * s.e.gain;     // EnvAsr::next_sample, then WrMul (wrappers_core/math.rs:63-67)
        // SvfFilter: inclusive scan of c_k = sum_{j<=k} A^(k-j) b x_j
        float c1 = K.b[0] * x, c2 = K.b[1] * x;
#pragma unroll
        for (int r = 0; r < 5; r++) {
            const float u1 = __shfl_up_sync(FULL, c1, 1u << r), u2 = __shfl_up_sync(FULL, c2, 1u << r);
            if (lane >= (1u << r)) {
                c1 = __fmaf_rn(K.pw[r][0], u1, __fmaf_rn(K.pw[r][1], u2, c1));
                c2 = __fmaf_rn(K.pw[r][2], u1, __fmaf_rn(K.pw[r][3], u2, c2));
            }
        }
        // the state before this lane's frame: s_k = A^k s_0 + c_(k-1)
        float e1 = __shfl_up_sync(FULL, c1, 1), e2 = __shfl_up_sync(FULL, c2, 1);
        if (lane == 0) e1 = e2 = 0.0f;
        const float ic1 = __fmaf_rn(K.pk[0], s.ic1, __fmaf_rn(K.pk[1], s.ic2, e1));
        const float ic2 = __fmaf_rn(K.pk[2], s.ic1, __fmaf_rn(K.pk[3], s.ic2, e2));
        // svf.rs:272-278 from the pre-update state
        const float v3 = x - ic2;
        const float v1 = s.a1 * ic1 + s.a2 * v3;
        const float v2 = (ic2 + s.a2 * ic1) + s.a3 * v3;
        const float y = (s.m0 * x + s.m1 * v1) + s.m2 * v2;
        const float out = y * env;                                  // MathUGen<Mul>, math.rs:45-47
        // the state after the chunk: s_32 = A^32 s_0 + c_31
        const float l1 = __shfl_sync(FULL, c1, 31), l2 = __shfl_sync(FULL, c2, 31);
        const float n1 = __fmaf_rn(K.p32[0], s.ic1, __fmaf_rn(K.p32[1], s.ic2, l1));
        const float n2 = __fmaf_rn(K.p32[2], s.ic1, __fmaf_rn(K.p32[3], s.ic2, l2));
        s.ic1 = n1;
        s.ic2 = n2;
        prow[f0 + lane] = out;
        if (TAPS && tap) tap[f0 + lane] = out;
    };

    bool have = false;   // the pre-pass of the chunk at f0 is already in pre[buf] (PIPE)
    uint32_t buf = 0;
#pragma unroll 1
    for (uint32_t f0 = 0; f0 < NF; f0 += SCAN_CHUNK) {
        if (have || chunk_fast(f0)) {
            if (!have) {
                prepass(pre[buf]);
                __syncwarp();
            }
            const float2 pk = pre[buf][lane];
            // PIPE: the NEXT chunk's pre-pass (a latency-bound chain of 32 x 3 dependent operations) is issued in the same
            // basic block as this chunk's frame-parallel half (shuffle latencies): each fills the other's stalls.  Its
            // inputs are all known here -- the state at the next chunk's first frame is where this chunk's pre-pass ended.
            if (PIPE && chunk_fast(f0 + SCAN_CHUNK)) {
                prepass(pre[buf ^ 1]);
                parallel(pk, f0);
                have = true;
            } else {
                parallel(pk, f0);
                have = false;
            }
            __syncwarp();
            buf ^= 1;
        } else {
            // ---- exact chunk: events applied at their frames, every frame in reference order, all lanes in step
            float out = 0.0f;
            bool touched = false;
            const uint32_t nf = min((uint32_t)SCAN_CHUNK, NF - f0);
#pragma unroll 1
            for (uint32_t k = 0; k < nf; k++) {
                while (next_frame <= f0 + k) { // sorted by (frame, node, arrival)
                    const DevEvent e = ldg_event(a.events + cur);
                    if (e.op == OP_SET) s.set(e.reg, e.value);
                    else s.e.op(e);
                    cur++;
                    next_frame = cur < end ? __ldg(&a.events[cur].frame) : 0xFFFFFFFFu;
                    touched = true;
                }
                const float o = s.tick();
                if (lane == k) out = o;
            }
            if (touched) {
                K.build(s.a1, s.a2, s.a3, lane);
                omd = 1.0f - s.dt;
                rc = div_prep(s.dt);
                tstar = wrap_flag_const(wrap_threshold(s.dt));
            }
            s.e.derive(d);
            if (f0 + lane < NF) {
                prow[f0 + lane] = out;
                if (TAPS && tap) tap[f0 + lane] = out;
            }
        }
    }
    if (lane == 0) {
        const uint32_t regs_out[R_EST] = {__float_as_uint(s.t), __float_as_uint(s.dt), s.use_sin, __float_as_uint(s.pw), s.wf,
                                           __float_as_uint(s.ic1), __float_as_uint(s.ic2), __float_as_uint(s.a1), __float_as_uint(s.a2),
                                           __float_as_uint(s.a3), __float_as_uint(s.m0), __float_as_uint(s.m1), __float_as_uint(s.m2)};
#pragma unroll
        for (int i = 0; i < R_EST; i++) a.regs[(size_t)i * V + v] = regs_out[i];
        s.e.store(a, v);
    }
}

// ------------------------------------------------------------------------------------------------------------------------------
// "render_sub_scan_n": FPL frames per lane.  In render_sub_scan a chunk is 32 frames and its critical path is the scan itself:
// five rounds of shuffle + two dependent FFMAs (~30 cycles each) behind the oscillator, ~350 cycles, against 256 for the phase
// chain.  Here a lane owns FPL CONSECUTIVE frames: it folds them locally (the filter's own recurrence, one step per frame), the
// warp scans the 32 lane totals with the powers A^(FPL 2^r), and every lane replays its FPL frames from the state before its
// first one -- in the reference's arithmetic (svf.rs:272-278), so only the state at every FPL-th frame carries re-associated
// sums.  The five rounds now serve 32 * FPL frames; the phase chain (8 cycles per frame, nothing to amortise) becomes the bound.
template <int FPL> struct ScanKN {
    float a[4];        // A, row-major
    float b[2];
    float pw[5][4];    // A^(FPL 2^r), r = 0..4
    float pn[4];       // A^(32 FPL)
    float pk[4];       // A^(FPL lane)
    KN_DEV void build(float a1, float a2, float a3, uint32_t lane) {
        double A[4] = {2.0 * (double)a1 - 1.0, -2.0 * (double)a2, 2.0 * (double)a2, 1.0 - 2.0 * (double)a3};
        b[0] = 2.0f * a2;
        b[1] = 2.0f * a3;
        double P[4] = {A[0], A[1], A[2], A[3]};
#pragma unroll
        for (int i = 1; i < FPL; i <<= 1) ScanK::mul(P, P, P);   // A^FPL (FPL a power of two)
        double K[4] = {1.0, 0.0, 0.0, 1.0};
#pragma unroll
        for (int r = 0; r < 5; r++) {
#pragma unroll
            for (int i = 0; i < 4; i++) pw[r][i] = (float)P[i];
            if ((lane >> r) & 1u) ScanK::mul(P, K, K);
            ScanK::mul(P, P, P);
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            a[i] = (float)A[i];
            pn[i] = (float)P[i];
            pk[i] = (float)K[i];
        }
    }
};

template <bool TAPS, int FPL>
__global__ void __launch_bounds__(32, 16) render_sub_scan_n(FusedArgs a) {
    static_assert(FPL == 1 || FPL == 2 || FPL == 4, "frames per lane");
    constexpr int CH = SCAN_CHUNK * FPL;                  // frames per chunk
    __shared__ __align__(16) float pre_t[2][CH];
    __shared__ __align__(16) float pre_e[2][CH];
    const uint32_t lane = threadIdx.x;
    const uint32_t v = blockIdx.x;
    const uint32_t V = a.n_voices;
    constexpr uint32_t FULL = 0xFFFFFFFFu;

    SubVoice<AsrEnv> s; // the voice's registers, identical on every lane
    {
        uint32_t r[R_EST];
#pragma unroll
        for (int i = 0; i < R_EST; i++) r[i] = a.regs[(size_t)i * V + v];
#pragma unroll
        for (int i = 0; i < R_EST; i++) s.set_core(i, r[i]);
        s.e.load(a, v);
    }
    uint32_t cur = 0, end = 0, next_frame = 0xFFFFFFFFu;
    if (a.events) {
        cur = a.ev_off[v];
        end = a.ev_off[v + 1];
        if (cur < end) next_frame = __ldg(&a.events[cur].frame);
    }
    float *tap = nullptr;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (a.taps[i].voice == v) tap = a.tap_out + (size_t)a.taps[i].tap * a.tap_stride + a.tap_frame0;
    float *prow = a.partials + (size_t)(a.row0 + v) * a.n_frames;

    ScanKN<FPL> K;
    K.build(s.a1, s.a2, s.a3, lane);
    float omd = 1.0f - s.dt, rc = div_prep(s.dt), tflag = wrap_flag_const(wrap_threshold(s.dt));
    AsrEnv::D d;
    s.e.derive(d);
    const uint32_t NF = a.n_frames;

    // the pre-pass of one chunk: the two f32 recurrences, sequentially, in the reference's rounding order.  Every lane runs the
    // same chain; lane 0 leaves (t_k, et_k) in shared memory, four frames per store.
    auto prepass = [&](uint32_t buf) {
        float t = s.t, et = s.e.et;
        float4 *dt4 = reinterpret_cast<float4 *>(pre_t[buf]), *de4 = reinterpret_cast<float4 *>(pre_e[buf]);
#pragma unroll
        for (int k = 0; k < CH; k += 4) {
            float tt[4], ee[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                tt[j] = t;
                ee[j] = et;
                t = (t + s.dt) - wrap_flag(t, tflag);     // inc(), polyblep.rs:232-235: wrap01(t + dt), see wrap_threshold
                et = et + d.delta;                        // envelopes.rs:58-66 with the state fixed over the chunk
            }
            if (lane == 0) {
                dt4[k / 4] = make_float4(tt[0], tt[1], tt[2], tt[3]);
                de4[k / 4] = make_float4(ee[0], ee[1], ee[2], ee[3]);
            }
        }
        s.t = t;
        s.e.et = (d.att || d.rel) ? et : s.e.et;
    };
    // whether the chunk starting at f0 can take the scan path, given the state at its first frame
    auto chunk_fast = [&](uint32_t f0) {
        return f0 + CH <= NF && next_frame >= f0 + CH && sub_lane_fast(s) && s.e.safe_frames() >= (uint32_t)CH;
    };
    // the frame-parallel half of a chunk: lane k renders frames f0 + FPL k .. + FPL - 1
    auto parallel = [&](uint32_t buf, uint32_t f0) {
        const bool ramp = d.att || d.rel;
        float x[FPL], env[FPL];
#pragma unroll
        for (int j = 0; j < FPL; j++) {
            const float t = pre_t[buf][FPL * lane + j], et = pre_e[buf][FPL * lane + j];
            x[j] = saw_eval(t, s.dt, omd, rc);                      // saw + blep, polyblep.rs:490-498
            const float tl = ramp ? et : d.cval;
            const float u = d.rel ? et : 1.0f;
            env[j] = (((tl * u) * u) * d.sc2) * s.e.gain;           // EnvAsr::next_sample, then WrMul
        }
        // the lane's own frames folded from a zero state: c = sum_j A^(FPL-1-j) b x_j
        float c1 = K.b[0] * x[0], c2 = K.b[1] * x[0];
#pragma unroll
        for (int j = 1; j < FPL; j++) {
            const float n1 = __fmaf_rn(K.a[0], c1, __fmaf_rn(K.a[1], c2, K.b[0] * x[j]));
            const float n2 = __fmaf_rn(K.a[2], c1, __fmaf_rn(K.a[3], c2, K.b[1] * x[j]));
            c1 = n1;
            c2 = n2;
        }
        // inclusive scan of the lane totals: c_L = sum_{j<=L} (A^FPL)^(L-j) c_j
#pragma unroll
        for (int r = 0; r < 5; r++) {
            const float u1 = __shfl_up_sync(FULL, c1, 1u << r), u2 = __shfl_up_sync(FULL, c2, 1u << r);
            if (lane >= (1u << r)) {
                c1 = __fmaf_rn(K.pw[r][0], u1, __fmaf_rn(K.pw[r][1], u2, c1));
                c2 = __fmaf_rn(K.pw[r][2], u1, __fmaf_rn(K.pw[r][3], u2, c2));
            }
        }
        float e1 = __shfl_up_sync(FULL, c1, 1), e2 = __shfl_up_sync(FULL, c2, 1);
        if (lane == 0) e1 = e2 = 0.0f;
        const float l1 = __shfl_sync(FULL, c1, 31), l2 = __shfl_sync(FULL, c2, 31);
        // the state before this lane's first frame: s = A^(FPL lane) s_0 + c_(lane-1); then its frames as the filter runs them
        float ic1 = __fmaf_rn(K.pk[0], s.ic1, __fmaf_rn(K.pk[1], s.ic2, e1));
        float ic2 = __fmaf_rn(K.pk[2], s.ic1, __fmaf_rn(K.pk[3], s.ic2, e2));
        const float n1 = __fmaf_rn(K.pn[0], s.ic1, __fmaf_rn(K.pn[1], s.ic2, l1));
        const float n2 = __fmaf_rn(K.pn[2], s.ic1, __fmaf_rn(K.pn[3], s.ic2, l2));
        s.ic1 = n1;
        s.ic2 = n2;
        float out[FPL];
#pragma unroll
        for (int j = 0; j < FPL; j++) {
            const float v3 = x[j] - ic2;                            // svf.rs:272-278
            const float v1 = s.a1 * ic1 + s.a2 * v3;
            const float v2 = (ic2 + s.a2 * ic1) + s.a3 * v3;
            ic1 = 2.0f * v1 - ic1;
            ic2 = 2.0f * v2 - ic2;
            const float y = (s.m0 * x[j] + s.m1 * v1) + s.m2 * v2;
            out[j] = y * env[j];                                    // MathUGen<Mul>, math.rs:45-47
        }
        float *dst = prow + f0 + FPL * lane;
        if (FPL == 1) dst[0] = out[0];
        else if (FPL == 2) *reinterpret_cast<float2 *>(dst) = make_float2(out[0], out[FPL > 1 ? 1 : 0]);
        else *reinterpret_cast<float4 *>(dst) = make_float4(out[0], out[FPL > 1 ? 1 : 0], out[FPL > 2 ? 2 : 0], out[FPL > 3 ? 3 : 0]);
        if (TAPS && tap) {
#pragma unroll
            for (int j = 0; j < FPL; j++) tap[f0 + FPL * lane + j] = out[j];
        }
    };

    // Both halves of the steady state in ONE hand-interleaved instruction stream: the pre-pass of the NEXT chunk (a latency-bound
    // chain, ~9 cycles per frame) cut into eight segments, and between them the stages of THIS chunk's frame-parallel half
    // (oscillator, local fold, the five scan rounds, the replay): each stage's shuffle latencies sit inside a chain segment.
    // ptxas keeps the order it is given (measured: written one after the other, the two halves ran one after the other,
    // 820 + 470 cycles per chunk).
    auto fused_chunk = [&](uint32_t buf, uint32_t f0) {
        float t = s.t, et = s.e.et;
        float4 *dt4 = reinterpret_cast<float4 *>(pre_t[buf ^ 1]), *de4 = reinterpret_cast<float4 *>(pre_e[buf ^ 1]);
        auto seg = [&](auto seg_c) {
            constexpr int S = decltype(seg_c)::value;
            constexpr int N = CH / 8;                      // frames per segment
#pragma unroll
            for (int k = S * N; k < (S + 1) * N; k += 4) {
                float tt[4], ee[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    tt[j] = t;
                    ee[j] = et;
                    t = (t + s.dt) - wrap_flag(t, tflag);
                    et = et + d.delta;
                }
                if (lane == 0) {
                    dt4[k / 4] = make_float4(tt[0], tt[1], tt[2], tt[3]);
                    de4[k / 4] = make_float4(ee[0], ee[1], ee[2], ee[3]);
                }
            }
        };
        const bool ramp = d.att || d.rel;
        float x[FPL], env[FPL], c1, c2;
        seg(std::integral_constant<int, 0>{});
#pragma unroll
        for (int j = 0; j < FPL; j++) {
            const float tj = pre_t[buf][FPL * lane + j], ej = pre_e[buf][FPL * lane + j];
            x[j] = saw_eval(tj, s.dt, omd, rc);
            const float tl = ramp ? ej : d.cval;
            const float u = d.rel ? ej : 1.0f;
            env[j] = (((tl * u) * u) * d.sc2) * s.e.gain;
        }
        seg(std::integral_constant<int, 1>{});
        c1 = K.b[0] * x[0], c2 = K.b[1] * x[0];
#pragma unroll
        for (int j = 1; j < FPL; j++) {
            const float n1 = __fmaf_rn(K.a[0], c1, __fmaf_rn(K.a[1], c2, K.b[0] * x[j]));
            const float n2 = __fmaf_rn(K.a[2], c1, __fmaf_rn(K.a[3], c2, K.b[1] * x[j]));
            c1 = n1;
            c2 = n2;
        }
        auto round = [&](auto r_c) {
            constexpr int r = decltype(r_c)::value;
            const float u1 = __shfl_up_sync(FULL, c1, 1u << r), u2 = __shfl_up_sync(FULL, c2, 1u << r);
            if (lane >= (1u << r)) {
                c1 = __fmaf_rn(K.pw[r][0], u1, __fmaf_rn(K.pw[r][1], u2, c1));
                c2 = __fmaf_rn(K.pw[r][2], u1, __fmaf_rn(K.pw[r][3], u2, c2));
            }
        };
        round(std::integral_constant<int, 0>{});
        seg(std::integral_constant<int, 2>{});
        round(std::integral_constant<int, 1>{});
        seg(std::integral_constant<int, 3>{});
        round(std::integral_constant<int, 2>{});
        seg(std::integral_constant<int, 4>{});
        round(std::integral_constant<int, 3>{});
        seg(std::integral_constant<int, 5>{});
        round(std::integral_constant<int, 4>{});
        seg(std::integral_constant<int, 6>{});
        float e1 = __shfl_up_sync(FULL, c1, 1), e2 = __shfl_up_sync(FULL, c2, 1);
        if (lane == 0) e1 = e2 = 0.0f;
        const float l1 = __shfl_sync(FULL, c1, 31), l2 = __shfl_sync(FULL, c2, 31);
        seg(std::integral_constant<int, 7>{});
        s.t = t;
        s.e.et = ramp ? et : s.e.et;
        float ic1 = __fmaf_rn(K.pk[0], s.ic1, __fmaf_rn(K.pk[1], s.ic2, e1));
        float ic2 = __fmaf_rn(K.pk[2], s.ic1, __fmaf_rn(K.pk[3], s.ic2, e2));
        const float n1 = __fmaf_rn(K.pn[0], s.ic1, __fmaf_rn(K.pn[1], s.ic2, l1));
        const float n2 = __fmaf_rn(K.pn[2], s.ic1, __fmaf_rn(K.pn[3], s.ic2, l2));
        s.ic1 = n1;
        s.ic2 = n2;
        float out[FPL];
#pragma unroll
        for (int j = 0; j < FPL; j++) {
            const float v3 = x[j] - ic2;                            // svf.rs:272-278
            const float v1 = s.a1 * ic1 + s.a2 * v3;
            const float v2 = (ic2 + s.a2 * ic1) + s.a3 * v3;
            ic1 = 2.0f * v1 - ic1;
            ic2 = 2.0f * v2 - ic2;
            const float y = (s.m0 * x[j] + s.m1 * v1) + s.m2 * v2;
            out[j] = y * env[j];
        }
        float *dst = prow + f0 + FPL * lane;
        if (FPL == 1) dst[0] = out[0];
        else if (FPL == 2) *reinterpret_cast<float2 *>(dst) = make_float2(out[0], out[FPL > 1 ? 1 : 0]);
        else *reinterpret_cast<float4 *>(dst) = make_float4(out[0], out[FPL > 1 ? 1 : 0], out[FPL > 2 ? 2 : 0], out[FPL > 3 ? 3 : 0]);
        if (TAPS && tap) {
#pragma unroll
            for (int j = 0; j < FPL; j++) tap[f0 + FPL * lane + j] = out[j];
        }
    };

    bool have = false;   // the pre-pass of the chunk at f0 is already in pre[buf]
    uint32_t buf = 0;
    uint32_t f0 = 0;
#pragma unroll 1
    while (f0 < NF) {
        if (have || chunk_fast(f0)) {
            if (!have) {
                prepass(buf);
                __syncwarp();
            }
            // the NEXT chunk's pre-pass (a latency-bound chain) is issued in the same basic block as this chunk's frame-parallel
            // half (shuffle latencies): each fills the other's stalls
            if (chunk_fast(f0 + CH)) {
                fused_chunk(buf, f0);
                have = true;
            } else {
                parallel(buf, f0);
                have = false;
            }
            __syncwarp();
            buf ^= 1;
            f0 += CH;
        } else {
            // ---- exact chunk: events applied at their frames, every frame in reference order, all lanes in step (32 frames at a
            // time: lane k keeps frame k).  The WHOLE chunk, so that the chunk grid stays where it is: which frames are scanned must
            // not depend on how the render is cut into launches (multiples of 64 frames).
            bool touched = false;
            const uint32_t fe = min(f0 + (uint32_t)CH, NF);
#pragma unroll 1
            for (; f0 < fe; f0 += SCAN_CHUNK) {
                float out = 0.0f;
                const uint32_t nf = min((uint32_t)SCAN_CHUNK, fe - f0);
#pragma unroll 1
                for (uint32_t k = 0; k < nf; k++) {
                    while (next_frame <= f0 + k) { // sorted by (frame, node, arrival)
                        const DevEvent e = ldg_event(a.events + cur);
                        if (e.op == OP_SET) s.set(e.reg, e.value);
                        else s.e.op(e);
                        cur++;
                        next_frame = cur < end ? __ldg(&a.events[cur].frame) : 0xFFFFFFFFu;
                        touched = true;
                    }
                    const float o = s.tick();
                    if (lane == k) out = o;
                }
                if (lane < nf) {
                    prow[f0 + lane] = out;
                    if (TAPS && tap) tap[f0 + lane] = out;
                }
            }
            if (touched) {
                K.build(s.a1, s.a2, s.a3, lane);
                omd = 1.0f - s.dt;
                rc = div_prep(s.dt);
                tflag = wrap_flag_const(wrap_threshold(s.dt));
            }
            s.e.derive(d);
        }
    }
    if (lane == 0) {
        const uint32_t regs_out[R_EST] = {__float_as_uint(s.t), __float_as_uint(s.dt), s.use_sin, __float_as_uint(s.pw), s.wf,
                                           __float_as_uint(s.ic1), __float_as_uint(s.ic2), __float_as_uint(s.a1), __float_as_uint(s.a2),
                                           __float_as_uint(s.a3), __float_as_uint(s.m0), __float_as_uint(s.m1), __float_as_uint(s.m2)};
#pragma unroll
        for (int i = 0; i < R_EST; i++) a.regs[(size_t)i * V + v] = regs_out[i];
        s.e.store(a, v);
    }
}

// ------------------------------------------------------------------------------------------------------------------------------
// "render_sub_scan2": the same chunks on TWO warps per voice.  One warp issues in order: when the chain and the scan share a warp,
// every stall of one (a shuffle not back yet) also holds the other (measured on render_sub_scan_n: 1070 cycles per 64-frame chunk
// where the chain alone needs 592).  Here the halves are roles, on two SM sub-partitions (warps of a CTA are spread over them):
//   warp 0 (phase warp)  runs the sequential f32 recurrences and nothing else and leaves (t_k, et_k) of every frame in a ring of
//       chunks in shared memory; it also owns the decision "scan or exact";
//   warp 1 (filter warp) takes the chunks from the ring: saw + blep, envelope, the SvfFilter scan (FPL frames per lane), output.
// Hand-over: named barriers, the producer / consumer pattern of the PTX manual (st.shared; bar.arrive -- bar.sync; ld.shared): per
// ring slot one barrier "full" (phase warp arrives, filter warp waits) and one "empty" (the reverse), plus one for the return of
// an exact chunk.  Barrier ids are immediates and the loop is unrolled over the ring's slots: a barrier named by a register costs a
// warp-synchronising prologue of ~100 cycles per use, and a first version with sequence counters behind __threadfence_block()
// also waited for the filter warp's global stores.  An EXACT chunk (parameter event, envelope transition, outside the
// straight-line domain) is rendered by the filter warp in reference order, as in render_sub_scan; the phase warp hands it
// (t, et), waits, and takes the voice's registers back.
constexpr int SCAN2_RING = 2;     // chunks between the two warps
constexpr int SCAN2_WORDS = 19;   // the voice's registers: 13 core + 6 envelope

KN_DEV void scan2_pack(const SubVoice<AsrEnv> &s, uint32_t *w) {
    w[0] = __float_as_uint(s.t); w[1] = __float_as_uint(s.dt); w[2] = s.use_sin; w[3] = __float_as_uint(s.pw); w[4] = s.wf;
    w[5] = __float_as_uint(s.ic1); w[6] = __float_as_uint(s.ic2); w[7] = __float_as_uint(s.a1); w[8] = __float_as_uint(s.a2);
    w[9] = __float_as_uint(s.a3); w[10] = __float_as_uint(s.m0); w[11] = __float_as_uint(s.m1); w[12] = __float_as_uint(s.m2);
    w[13] = s.e.est; w[14] = __float_as_uint(s.e.et); w[15] = __float_as_uint(s.e.ar); w[16] = __float_as_uint(s.e.rr);
    w[17] = __float_as_uint(s.e.sc); w[18] = __float_as_uint(s.e.gain);
}
KN_DEV void scan2_unpack(SubVoice<AsrEnv> &s, const uint32_t *w) {
#pragma unroll
    for (int i = 0; i < R_EST; i++) s.set_core(i, w[i]);
#pragma unroll
    for (int i = 0; i < 6; i++) s.e.set(R_EST + i, w[R_EST + i]);
}
// four floats to a shared-memory address given as such (a generic pointer makes the compiler rebuild the shared window's base --
// S2R + LEA -- in front of every store)
KN_DEV void scan2_sts4(uint32_t addr, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
// barrier ids (0 is __syncthreads'): full[slot] = 1 + slot, empty[slot] = 1 + RING + slot, returned = 1 + 2 * RING; 64 threads each
template <int ID> KN_DEV void scan2_sync() { asm volatile("bar.sync %0, 64;" ::"n"(ID) : "memory"); }
template <int ID> KN_DEV void scan2_arrive() { asm volatile("bar.arrive %0, 64;" ::"n"(ID) : "memory"); }
constexpr int SCAN2_FULL = 1, SCAN2_EMPTY = 1 + SCAN2_RING, SCAN2_RETURNED = 1 + 2 * SCAN2_RING;

template <bool TAPS, int FPL>
__global__ void __launch_bounds__(64, 8) render_sub_scan2(FusedArgs a) {
    static_assert(SCAN2_RING == 2, "the loops below are unrolled over two slots");
    constexpr int CH = SCAN_CHUNK * FPL;                                 // frames per chunk
    __shared__ __align__(16) float ring_t[SCAN2_RING][CH];               // the phase before every frame ([0]: at an exact chunk's start)
    __shared__ __align__(16) float ring_et[SCAN2_RING][CH];              // the envelope ramp likewise
    __shared__ uint32_t ring_exact[SCAN2_RING];
    __shared__ uint32_t hand[SCAN2_WORDS];
    const uint32_t lane = threadIdx.x & 31u;
    const bool phase_warp = threadIdx.x < 32u;
    const uint32_t v = blockIdx.x;
    const uint32_t V = a.n_voices;
    constexpr uint32_t FULL = 0xFFFFFFFFu;

    SubVoice<AsrEnv> s;
    {
        uint32_t r[R_EST];
#pragma unroll
        for (int i = 0; i < R_EST; i++) r[i] = a.regs[(size_t)i * V + v];
#pragma unroll
        for (int i = 0; i < R_EST; i++) s.set_core(i, r[i]);
        s.e.load(a, v);
    }
    uint32_t cur = 0, end = 0, next_frame = 0xFFFFFFFFu;
    if (a.events) {
        cur = a.ev_off[v];
        end = a.ev_off[v + 1];
        if (cur < end) next_frame = __ldg(&a.events[cur].frame);
    }
    const uint32_t NF = a.n_frames, NC = (NF + CH - 1) / CH;
    AsrEnv::D d;
    s.e.derive(d);

    if (phase_warp) {
        float tthr = wrap_threshold(s.dt), tflag = wrap_flag_const(tthr);
        // Whether a chunk takes the scan path is a function of the state at ITS first frame only (so that a render does not depend on
        // how it is cut into launches): no event inside, the straight-line domain, no envelope transition possible inside.
        bool lane_fast = sub_lane_fast(s);                 // the voice's parameters: they only change in exact chunks
        uint32_t ring_t_sa = (uint32_t)__cvta_generic_to_shared(&ring_t[0][0]);
        uint32_t ring_et_sa = (uint32_t)__cvta_generic_to_shared(&ring_et[0][0]);
        asm volatile("" : "+r"(ring_t_sa), "+r"(ring_et_sa)); // opaque: kept in registers instead of being rebuilt before every store
        auto chunk = [&](auto slot_c, uint32_t c) {
            constexpr int SLOT = decltype(slot_c)::value;
            const uint32_t f0 = c * CH;
            if (c >= SCAN2_RING) scan2_sync<SCAN2_EMPTY + SLOT>();                // the slot is free again
            const bool fast = lane_fast && f0 + CH <= min(next_frame, NF) && (!(d.att || d.rel) || s.e.safe_frames() >= (uint32_t)CH);
            if (fast) {
                // the f32 recurrences of the chunk, sequentially, in the reference's rounding order (every lane the same chain;
                // lane 0 leaves the values before each frame in the ring)
                float t = s.t, et = s.e.et;
                // A chunk that provably does not wrap skips the flag: t_k <= t_0 + k (dt + 2^-24) (every sum below 1 rounds by at
                // most 2^-25), so if that stays below the threshold T for the whole chunk the chain is one FADD per frame (4 cycles
                // instead of 9).  One decision per chunk: a branch per group of frames cost more than it saved (6.8 ms against 4.4).
                const bool calm = __fmaf_rn((float)CH, s.dt + 5.9604644775390625e-8f, t) < tthr;
                if (calm) {
#pragma unroll
                    for (int k = 0; k < CH; k += 4) {
                        float tt[4], ee[4];
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            tt[j] = t;
                            ee[j] = et;
                            t = t + s.dt;                                         // no wrap here: (t + dt) - 0
                            et = et + d.delta;
                        }
                        if (lane == 0) {
                            scan2_sts4(ring_t_sa + (SLOT * CH + k) * 4, tt[0], tt[1], tt[2], tt[3]);
                            scan2_sts4(ring_et_sa + (SLOT * CH + k) * 4, ee[0], ee[1], ee[2], ee[3]);
                        }
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < CH; k += 4) {
                        float tt[4], ee[4];
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            tt[j] = t;
                            ee[j] = et;
                            t = (t + s.dt) - wrap_flag(t, tflag);                 // inc(), polyblep.rs:232-235 (wrap_threshold)
                            et = et + d.delta;                                    // envelopes.rs:58-66, state fixed over the chunk
                        }
                        if (lane == 0) {
                            scan2_sts4(ring_t_sa + (SLOT * CH + k) * 4, tt[0], tt[1], tt[2], tt[3]);
                            scan2_sts4(ring_et_sa + (SLOT * CH + k) * 4, ee[0], ee[1], ee[2], ee[3]);
                        }
                    }
                }
                s.t = t;
                s.e.et = (d.att || d.rel) ? et : s.e.et;
                if (lane == 0) ring_exact[SLOT] = 0u;
                scan2_arrive<SCAN2_FULL + SLOT>();
            } else {
                if (lane == 0) {
                    ring_t[SLOT][0] = s.t;
                    ring_et[SLOT][0] = s.e.et;
                    ring_exact[SLOT] = 1u;
                }
                scan2_arrive<SCAN2_FULL + SLOT>();
                // the filter warp renders this chunk in reference order and returns the voice
                scan2_sync<SCAN2_RETURNED>();
                uint32_t w[SCAN2_WORDS];
#pragma unroll
                for (int i = 0; i < SCAN2_WORDS; i++) w[i] = hand[i];
                scan2_unpack(s, w);
                const uint32_t fe = min(f0 + (uint32_t)CH, NF);
                while (next_frame < fe) { // the events of the chunk are applied (by the filter warp): step over them
                    cur++;
                    next_frame = cur < end ? __ldg(&a.events[cur].frame) : 0xFFFFFFFFu;
                }
                s.e.derive(d);
                tthr = wrap_threshold(s.dt);
                tflag = wrap_flag_const(tthr);
                lane_fast = sub_lane_fast(s);
            }
        };
#pragma unroll 1
        for (uint32_t c = 0; c < NC; c += SCAN2_RING) {
            chunk(std::integral_constant<int, 0>{}, c);
            if (c + 1 < NC) chunk(std::integral_constant<int, 1>{}, c + 1);
        }
        // the phase warp's share of the state: the phase and the envelope
        if (lane == 0) {
            a.regs[(size_t)0 * V + v] = __float_as_uint(s.t);
            s.e.store(a, v);
        }
        return;
    }

    // ---- filter warp
    float *tap = nullptr;
    if (TAPS)
        for (uint32_t i = 0; i < a.n_taps; i++)
            if (a.taps[i].voice == v) tap = a.tap_out + (size_t)a.taps[i].tap * a.tap_stride + a.tap_frame0;
    float *prow = a.partials + (size_t)(a.row0 + v) * a.n_frames;
    ScanKN<FPL> K;
    K.build(s.a1, s.a2, s.a3, lane);
    float omd = 1.0f - s.dt, rc = div_prep(s.dt);

    auto chunk = [&](auto slot_c, uint32_t c) {
        constexpr int SLOT = decltype(slot_c)::value;
        uint32_t f0 = c * CH;
        scan2_sync<SCAN2_FULL + SLOT>();
        const bool exact = __shfl_sync(FULL, ring_exact[SLOT], 0) != 0u; // (one lane's reading: the branches hold barriers)
        if (!exact) {
            float tq[FPL], eq[FPL];
#pragma unroll
            for (int j = 0; j < FPL; j++) {
                tq[j] = ring_t[SLOT][FPL * lane + j];
                eq[j] = ring_et[SLOT][FPL * lane + j];
            }
            // the slot is handed back as soon as it has been read -- except the last RING chunks, whose "empty" nobody waits for
            if (c + SCAN2_RING < NC) scan2_arrive<SCAN2_EMPTY + SLOT>();
            const bool ramp = d.att || d.rel;
            float x[FPL], env[FPL];
#pragma unroll
            for (int j = 0; j < FPL; j++) {
                x[j] = saw_eval(tq[j], s.dt, omd, rc);                  // saw + blep, polyblep.rs:490-498
                const float tl = ramp ? eq[j] : d.cval;
                const float u = d.rel ? eq[j] : 1.0f;
                env[j] = (((tl * u) * u) * d.sc2) * s.e.gain;           // EnvAsr::next_sample, then WrMul
            }
            // the lane's own frames folded from a zero state, then the inclusive scan of the lane totals (render_sub_scan_n)
            float c1 = K.b[0] * x[0], c2 = K.b[1] * x[0];
#pragma unroll
            for (int j = 1; j < FPL; j++) {
                const float n1 = __fmaf_rn(K.a[0], c1, __fmaf_rn(K.a[1], c2, K.b[0] * x[j]));
                const float n2 = __fmaf_rn(K.a[2], c1, __fmaf_rn(K.a[3], c2, K.b[1] * x[j]));
                c1 = n1;
                c2 = n2;
            }
#pragma unroll
            for (int r = 0; r < 5; r++) {
                const float u1 = __shfl_up_sync(FULL, c1, 1u << r), u2 = __shfl_up_sync(FULL, c2, 1u << r);
                if (lane >= (1u << r)) {
                    c1 = __fmaf_rn(K.pw[r][0], u1, __fmaf_rn(K.pw[r][1], u2, c1));
                    c2 = __fmaf_rn(K.pw[r][2], u1, __fmaf_rn(K.pw[r][3], u2, c2));
                }
            }
            float e1 = __shfl_up_sync(FULL, c1, 1), e2 = __shfl_up_sync(FULL, c2, 1);
            if (lane == 0) e1 = e2 = 0.0f;
            const float l1 = __shfl_sync(FULL, c1, 31), l2 = __shfl_sync(FULL, c2, 31);
            float ic1 = __fmaf_rn(K.pk[0], s.ic1, __fmaf_rn(K.pk[1], s.ic2, e1));
            float ic2 = __fmaf_rn(K.pk[2], s.ic1, __fmaf_rn(K.pk[3], s.ic2, e2));
            const float n1 = __fmaf_rn(K.pn[0], s.ic1, __fmaf_rn(K.pn[1], s.ic2, l1));
            const float n2 = __fmaf_rn(K.pn[2], s.ic1, __fmaf_rn(K.pn[3], s.ic2, l2));
            s.ic1 = n1;
            s.ic2 = n2;
            float out[FPL];
#pragma unroll
            for (int j = 0; j < FPL; j++) {
                const float v3 = x[j] - ic2;                            // svf.rs:272-278
                const float v1 = s.a1 * ic1 + s.a2 * v3;
                const float v2 = (ic2 + s.a2 * ic1) + s.a3 * v3;
                ic1 = 2.0f * v1 - ic1;
                ic2 = 2.0f * v2 - ic2;
                const float y = (s.m0 * x[j] + s.m1 * v1) + s.m2 * v2;
                out[j] = y * env[j];                                    // MathUGen<Mul>, math.rs:45-47
            }
            float *dst = prow + f0 + FPL * lane;
            if (FPL == 1) dst[0] = out[0];
            else if (FPL == 2) *reinterpret_cast<float2 *>(dst) = make_float2(out[0], out[FPL > 1 ? 1 : 0]);
            else *reinterpret_cast<float4 *>(dst) = make_float4(out[0], out[FPL > 1 ? 1 : 0], out[FPL > 2 ? 2 : 0], out[FPL > 3 ? 3 : 0]);
            if (TAPS && tap) {
#pragma unroll
                for (int j = 0; j < FPL; j++) tap[f0 + FPL * lane + j] = out[j];
            }
            return;
        }
        // ---- exact chunk: events applied at their frames, every frame in reference order, all lanes in step (32 frames at a time)
        s.t = ring_t[SLOT][0];
        s.e.et = ring_et[SLOT][0];
        bool touched = false;
        const uint32_t fe = min(f0 + (uint32_t)CH, NF);
#pragma unroll 1
        for (; f0 < fe; f0 += SCAN_CHUNK) {
            float out = 0.0f;
            const uint32_t nf = min((uint32_t)SCAN_CHUNK, fe - f0);
#pragma unroll 1
            for (uint32_t k = 0; k < nf; k++) {
                while (next_frame <= f0 + k) { // sorted by (frame, node, arrival)
                    const DevEvent e = ldg_event(a.events + cur);
                    if (e.op == OP_SET) s.set(e.reg, e.value);
                    else s.e.op(e);
                    cur++;
                    next_frame = cur < end ? __ldg(&a.events[cur].frame) : 0xFFFFFFFFu;
                    touched = true;
                }
                const float o = s.tick();
                if (lane == k) out = o;
            }
            if (lane < nf) {
                prow[f0 + lane] = out;
                if (TAPS && tap) tap[f0 + lane] = out;
            }
        }
        if (touched) {
            K.build(s.a1, s.a2, s.a3, lane);
            omd = 1.0f - s.dt;
            rc = div_prep(s.dt);
        }
        s.e.derive(d);
        if (lane == 0) {
            uint32_t w[SCAN2_WORDS];
            scan2_pack(s, w);
#pragma unroll
            for (int i = 0; i < SCAN2_WORDS; i++) hand[i] = w[i];
        }
        if (c + SCAN2_RING < NC) scan2_arrive<SCAN2_EMPTY + SLOT>();
        scan2_arrive<SCAN2_RETURNED>();
    };
#pragma unroll 1
    for (uint32_t c = 0; c < NC; c += SCAN2_RING) {
        chunk(std::integral_constant<int, 0>{}, c);
        if (c + 1 < NC) chunk(std::integral_constant<int, 1>{}, c + 1);
    }
    // the filter warp's share of the state: everything but the phase and the envelope
    if (lane == 0) {
        uint32_t w[SCAN2_WORDS];
        scan2_pack(s, w);
#pragma unroll
        for (int i = 1; i < R_EST; i++) a.regs[(size_t)i * V + v] = w[i];
    }
}
