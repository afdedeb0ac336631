// devmath_exhaustive.cu -- the device arithmetic under the engine's "bit-identical to the oracle" results, checked on the GPU
// over whole domains.  It includes the headers the kernels include (knaster_b200/csrc/nodes.cuh, sinf_glibc.h) and is
// compiled with the library's numeric flags, so every function below is the device code the kernels run:
//
//   a. sine    kn_sinf on all 2^32 floats against host sinf (bit-identical; NaN where libm gives NaN);
//              kn_sinf_glibc_inrange, kn_sinf_glibc_lean and kn_sinf_glibc_lean_n<32> (render_fm2's FM_SUB_N = 32 frames)
//              against kn_sinf for every |y| < 120 (lean: sin(-0) = +0 is the documented exception)
//   b. cosine  kn_cosf on all 2^32 floats against host cosf
//   c. division div_rc(n, d, div_prep(d)) against IEEE n / d for every pair of significands n, d in [1, 2) (2^46 pairs): while
//              q0 = n * rc, the FMA remainder and the corrected quotient stay normal, their rounding depends on the significands
//              only, so this covers every normal quotient the saw and FM paths form.  Also render_fm2's increment
//              (v / sr via div_rc, |v| <= 1e-20 scaled by 2^64) for every finite v at seven sample rates against IEEE v / sr
//   d. saw     saw_fast_tick against polyblep_saw_tick (output and next phase) and saw_eval2 against two saw_evals, for
//              every t in [0, 1) at 64 increments dt
//   e. wrap    wrap_threshold(dt) for every dt in [2^-20, 1/4): RN(T + dt) >= 1 > RN(prev(T) + dt); wrap_flag at six phases
//   f. tan / exp / pow  kn_tanf on every float in (-pi/2, pi/2), kn_expf on every float whose result is finite,
//              kn_powf(10, g / 40) for every f32 g in [-120, 120] and kn_powf on a seeded 2-D sample: ulp distance from
//              glibc, and agreement with the correctly rounded value (host f64, and long double near f32 midpoints;
//              arguments within 2^-40 relative of a midpoint are "undecided" and not counted)
//
// Device results come back with cudaMemcpyAsync into pinned memory, 2^28 floats (1 GiB) at a time, and host threads compare
// them with libm; the pair sweeps count on the device (an atomic mismatch count and the first 64 failing operands).
// Prints one JSON line.  tests/test_gpu_devmath.py builds and runs it:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -fmad=false -prec-div=true -prec-sqrt=true -ftz=false
//        -Iknaster_b200/csrc tools/devmath_exhaustive.cu -o devmath_exhaustive -lpthread
// usage: devmath_exhaustive [stride]   (stride k: every k-th argument / divisor, for a quick run; 1 = everything)
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <thread>
#include <vector>

#include "nodes.cuh"

using namespace kgpu;

#define CK(x)                                                                                                              \
    do {                                                                                                                   \
        cudaError_t e_ = (x);                                                                                              \
        if (e_ != cudaSuccess) {                                                                                           \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));                              \
            exit(2);                                                                                                       \
        }                                                                                                                  \
    } while (0)

constexpr int MAX_REC = 64;
struct Fails {                          // one per device-side check
    unsigned long long count;
    unsigned long long aux;             // a second, check-specific count
    uint32_t rec[MAX_REC][4];           // operands, result, expected
};
__device__ void record(Fails *f, uint32_t a, uint32_t b, uint32_t got, uint32_t want) {
    const unsigned long long i = atomicAdd(&f->count, 1ull);
    if (i < MAX_REC) {
        f->rec[i][0] = a, f->rec[i][1] = b, f->rec[i][2] = got, f->rec[i][3] = want;
    }
}
__device__ __forceinline__ uint32_t fb(float x) { return __float_as_uint(x); }
__device__ __forceinline__ float bf(uint32_t x) { return __uint_as_float(x); }

// ---- a/b/f: one function over a range of arguments, results to memory ---------------------------------------------------
enum Fn { F_SIN, F_COS, F_TAN, F_EXP, F_POW_DB, F_POW2 };
template <int FN> __global__ void k_map(uint32_t first_bits, uint32_t step, uint32_t n, const float *__restrict__ x2,
                                        const float *__restrict__ y2, float *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = bf(first_bits + i * step);
    float r;
    if (FN == F_SIN) r = kn_sinf(x);
    else if (FN == F_COS) r = kn_cosf(x);
    else if (FN == F_TAN) r = kn_tanf(x);
    else if (FN == F_EXP) r = kn_expf(x);
    else if (FN == F_POW_DB) r = kn_powf(10.0f, x / 40.0f);    // svf_coeffs_dev: amp = powf(10, gain_db / 40)
    else r = kn_powf(x2[i], y2[i]);
    out[i] = r;
}

// ---- a: the |y| < 120 restatements against kn_sinf, 32 consecutive arguments per thread ---------------------------------
constexpr int LEAN_N = 32; // render_fm2's group (FM_SUB_N in fused.cu)
__global__ void k_sine_forms(uint32_t n_groups, uint32_t step, Fails *inrange, Fails *lean, Fails *lean_n) {
    const uint32_t g = (blockIdx.x * blockDim.x + threadIdx.x) * step;
    if (g >= n_groups) return;
    const uint32_t LIM = 0x42f00000u; // 120.0f
    for (uint32_t sgn = 0; sgn < 2; sgn++) {
        float y[LEAN_N], o[LEAN_N];
#pragma unroll
        for (int k = 0; k < LEAN_N; k++) {
            const uint32_t b = g * LEAN_N + k;
            y[k] = bf((b < LIM ? b : 0u) | (sgn << 31));
        }
        kn_sinf_glibc_lean_n(y, o);
#pragma unroll 4
        for (int k = 0; k < LEAN_N; k++) {
            if (g * LEAN_N + k >= LIM) continue;
            const float ref = kn_sinf(y[k]), a = kn_sinf_glibc_inrange(y[k]), b = kn_sinf_glibc_lean(y[k]);
            if (fb(a) != fb(ref)) record(inrange, fb(y[k]), 0, fb(a), fb(ref));
            if (fb(b) != fb(ref)) {
                if (b == ref) atomicAdd(&lean->aux, 1ull); // -0 against +0
                else record(lean, fb(y[k]), 0, fb(b), fb(ref));
            }
            if (fb(o[k]) != fb(ref)) {
                if (o[k] == ref) atomicAdd(&lean_n->aux, 1ull);
                else record(lean_n, fb(y[k]), 0, fb(o[k]), fb(ref));
            }
        }
    }
}

// ---- c: division ----------------------------------------------------------------------------------------------------------
// one divisor significand per block, every numerator significand over its threads; aux counts divisors whose refined
// reciprocal div_prep(d) is not the correctly rounded 1/d
__global__ void k_div_pairs(uint32_t first_d, uint32_t d_stride, Fails *f) {
    const uint32_t dsig = first_d + blockIdx.x * d_stride;
    if (dsig >= (1u << 23)) return;
    const float d = bf(0x3f800000u | dsig), rc = div_prep(d);
    if (threadIdx.x == 0 && fb(rc) != fb(__frcp_rn(d))) atomicAdd(&f->aux, 1ull);
    for (uint32_t k = threadIdx.x; k < (1u << 23); k += blockDim.x) {
        const float n = bf(0x3f800000u | k);
        const float q = div_rc(n, d, rc), want = __fdiv_rn(n, d);
        if (fb(q) != fb(want)) record(f, fb(n), fb(d), fb(q), fb(want));
    }
}
// render_fm2's carrier increment (fused.cu, FmVoice::tick / the group's q[k]): aux counts differences where the IEEE quotient
// is subnormal or zero (|v| < 6e-34: the scaled form rounds twice there; a 1e-45 increment cannot move a phase)
__global__ void k_div_fm(uint32_t first_bits, uint32_t n, float sr, Fails *f) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float rc_sr = div_prep(sr);
    for (uint32_t sgn = 0; sgn < 2; sgn++) {
        const float v = bf((first_bits + i) | (sgn << 31));
        const bool tiny = fabsf(v) <= 1e-20f;
        const float q0 = div_rc(tiny ? v * 0x1p64f : v, sr, rc_sr);
        const float q = tiny ? q0 * 0x1p-64f : q0;
        const float want = __fdiv_rn(v, sr);
        if (fb(q) != fb(want)) {
            if (fabsf(want) < FLT_MIN) atomicAdd(&f->aux, 1ull);
            else record(f, fb(v), fb(sr), fb(q), fb(want));
        }
    }
}

// ---- d: the straight-line saw against the reference-order one ------------------------------------------------------------
__global__ void k_saw(uint32_t first_t, uint32_t n, const float *__restrict__ dts, int n_dt, Fails *tick, Fails *pair) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float t = bf(first_t + i);
    for (int j = 0; j < n_dt; j++) {
        const float dt = dts[j], omd = 1.0f - dt, rc = div_prep(dt);
        float t1 = t, t2 = t;
        const float a = saw_fast_tick(t1, dt, omd, rc), b = polyblep_saw_tick(t2, dt, 0u);
        if (fb(a) != fb(b) || fb(t1) != fb(t2)) record(tick, fb(t), fb(dt), fb(a) != fb(b) ? fb(a) : fb(t1), fb(a) != fb(b) ? fb(b) : fb(t2));
        // two frames of one voice: this phase and the next
        const float2 p = saw_eval2(make_float2(t, t1), dt, omd, rc);
        const float e0 = saw_eval(t, dt, omd, rc), e1 = saw_eval(t1, dt, omd, rc);
        if (fb(p.x) != fb(e0) || fb(p.y) != fb(e1)) record(pair, fb(t), fb(dt), fb(p.x) != fb(e0) ? fb(p.x) : fb(p.y), fb(p.x) != fb(e0) ? fb(e0) : fb(e1));
    }
}

// ---- e: the wrap threshold ------------------------------------------------------------------------------------------------
__global__ void k_wrap(uint32_t first_dt, uint32_t n, Fails *thr, Fails *flag) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float dt = bf(first_dt + i);
    const float T = wrap_threshold(dt), Tp = bf(fb(T) - 1u);
    if (!(__fadd_rn(T, dt) >= 1.0f) || !(__fadd_rn(Tp, dt) < 1.0f)) record(thr, fb(dt), 0, fb(T), 0);
    const float c = wrap_flag_const(T);
    const float ts[6] = {Tp, T, bf(fb(T) + 1u), 0.0f, 0.5f, bf(0x3f7fffffu)};
#pragma unroll
    for (int k = 0; k < 6; k++) {
        if (!(ts[k] < 1.0f)) continue; // phases live in [0, 1)
        const float got = wrap_flag(ts[k], c), want = __fadd_rn(ts[k], dt) >= 1.0f ? 1.0f : 0.0f;
        if (fb(got) != fb(want)) record(flag, fb(ts[k]), fb(dt), fb(got), fb(want));
    }
}

// ---- host side -------------------------------------------------------------------------------------------------------------
static uint32_t hb(float x) {
    uint32_t b;
    memcpy(&b, &x, 4);
    return b;
}
static float hf(uint32_t b) {
    float x;
    memcpy(&x, &b, 4);
    return x;
}
static int64_t ord(float x) { // a float's position on the number line, in ulps
    const uint32_t b = hb(x);
    return (b & 0x80000000u) ? -(int64_t)(b & 0x7fffffffu) : (int64_t)b;
}
static unsigned n_threads() { return std::max(1u, std::thread::hardware_concurrency()); }
template <class F> static void parallel(uint64_t n, F f) { // f(begin, end, worker)
    const unsigned T = n_threads();
    std::vector<std::thread> th;
    for (unsigned w = 0; w < T; w++) th.emplace_back([&, w] { f(n * w / T, n * (w + 1) / T, w); });
    for (auto &t : th) t.join();
}

struct Dev {
    float *out = nullptr, *host = nullptr, *x2 = nullptr, *y2 = nullptr;
    cudaStream_t st = nullptr;
    static constexpr uint32_t CHUNK = 1u << 28; // floats per round trip: 1 GiB
};

// The correctly rounded f32 of a function value, and whether the argument is "undecided": its value lies within 2^-40
// (relative) of an f32 rounding midpoint, where the reference's own error could decide the rounding.  Two stages: glibc's
// f64 function (error below 1 ulp of f64, 2^-52 relative) decides every argument more than 2^-30 from a midpoint; the rest
// are evaluated again in long double (64-bit significand) and held to the 2^-40 rule.  (Long double for every argument
// would cost ~0.4 us per powl: minutes of host time per sweep.)
static long double midpoint_distance(long double v, float f) { // relative distance from v to the midpoint on v's side of f
    const float g = nextafterf(f, v > (long double)f ? INFINITY : -INFINITY);
    if (std::isinf(g)) return 1.0L;
    const long double mid = ((long double)f + (long double)g) * 0.5L;
    return fabsl(v - mid) / fabsl(v);
}
template <class FD, class FL> static float correctly_rounded(FD fd, FL fl, bool *undecided) {
    *undecided = false;
    const double v = fd();
    float f = (float)v;
    if (std::isinf(f) || std::isnan(f) || v == 0.0) return f;
    if (midpoint_distance(v, f) > 0x1p-30L) return f;
    const long double w = fl();
    f = (float)w;
    if (std::isinf(f) || w == 0.0L || (long double)f == w) return f;
    *undecided = midpoint_distance(w, f) <= 0x1p-40L;
    return f;
}

struct Cmp { // libm comparison of one function
    std::string name;
    std::atomic<uint64_t> n{0}, bad{0};                               // a, b: bit identity with libm
    std::atomic<uint64_t> dev_vs_glibc{0}, over_1ulp{0}, dev_not_cr{0}, glibc_not_cr{0}, undecided{0}; // f
    std::atomic<uint64_t> first_bad{~0ull};
};

// Runs one function over the bit patterns lo, lo + step, ... below hi (or over the sample xs, ys) on the device and compares
// the results with libm on the host
template <int FN>
static void sweep(Dev &D, Cmp &c, uint64_t lo, uint64_t hi, uint32_t step, const std::vector<float> *xs = nullptr,
                  const std::vector<float> *ys = nullptr) {
    const bool sample = FN == F_POW2;
    const uint64_t total = sample ? xs->size() : (hi - lo + step - 1) / step;
    for (uint64_t base = 0; base < total; base += Dev::CHUNK) {
        const uint32_t n = (uint32_t)std::min<uint64_t>(Dev::CHUNK, total - base);
        const uint32_t first = sample ? 0u : (uint32_t)(lo + base * step);
        if (sample) {
            CK(cudaMemcpyAsync(D.x2, xs->data() + base, n * 4ull, cudaMemcpyHostToDevice, D.st));
            CK(cudaMemcpyAsync(D.y2, ys->data() + base, n * 4ull, cudaMemcpyHostToDevice, D.st));
        }
        k_map<FN><<<(n + 255) / 256, 256, 0, D.st>>>(first, step, n, D.x2, D.y2, D.out);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(D.host, D.out, n * 4ull, cudaMemcpyDeviceToHost, D.st));
        CK(cudaStreamSynchronize(D.st));
        parallel(n, [&](uint64_t b, uint64_t e, unsigned) {
            uint64_t nn = 0, bad = 0, dg = 0, o1 = 0, dcr = 0, gcr = 0, und = 0, fbad = ~0ull;
            for (uint64_t i = b; i < e; i++) {
                const float got = D.host[i];
                const uint32_t xb = first + (uint32_t)i * step;
                if (FN == F_SIN || FN == F_COS) {
                    const float x = hf(xb);
                    const float ref = FN == F_SIN ? sinf(x) : cosf(x);
                    nn++;
                    const bool ok = std::isnan(ref) ? std::isnan(got) : hb(ref) == hb(got);
                    if (!ok) {
                        bad++;
                        fbad = std::min<uint64_t>(fbad, xb);
                    }
                    continue;
                }
                float glibc, cr;
                bool u;
                if (FN == F_TAN) {
                    const float x = hf(xb);
                    glibc = tanf(x);
                    cr = correctly_rounded([&] { return tan((double)x); }, [&] { return tanl((long double)x); }, &u);
                } else if (FN == F_EXP) {
                    const float x = hf(xb);
                    glibc = expf(x);
                    cr = correctly_rounded([&] { return exp((double)x); }, [&] { return expl((long double)x); }, &u);
                    if (std::isinf(cr)) continue; // result not finite: outside the domain
                } else if (FN == F_POW_DB) {
                    const float y = hf(xb) / 40.0f;
                    glibc = powf(10.0f, y);
                    cr = correctly_rounded([&] { return pow(10.0, (double)y); }, [&] { return powl(10.0L, (long double)y); }, &u);
                } else {
                    const float x = (*xs)[base + i], y = (*ys)[base + i];
                    glibc = powf(x, y);
                    cr = correctly_rounded([&] { return pow((double)x, (double)y); }, [&] { return powl((long double)x, (long double)y); },
                                           &u);
                }
                nn++;
                if (hb(got) != hb(glibc)) dg++;
                if (std::llabs(ord(got) - ord(glibc)) > 1) {
                    o1++;
                    fbad = std::min<uint64_t>(fbad, sample ? base + i : xb);
                }
                if (u) und++;
                else {
                    if (hb(got) != hb(cr)) dcr++;
                    if (hb(glibc) != hb(cr)) gcr++;
                }
            }
            c.n += nn, c.bad += bad, c.dev_vs_glibc += dg, c.over_1ulp += o1, c.dev_not_cr += dcr, c.glibc_not_cr += gcr,
                c.undecided += und;
            uint64_t cur = c.first_bad.load();
            while (fbad < cur && !c.first_bad.compare_exchange_weak(cur, fbad)) {
            }
        });
    }
}

static std::string fails_json(const Fails &f) {
    char buf[256];
    snprintf(buf, sizeof buf, "{\"mismatches\": %llu, \"aux\": %llu, \"first\": [", f.count, f.aux);
    std::string s = buf;
    for (unsigned long long i = 0; i < std::min<unsigned long long>(f.count, 4); i++) {
        snprintf(buf, sizeof buf, "%s[\"0x%08x\", \"0x%08x\", \"0x%08x\", \"0x%08x\"]", i ? ", " : "", f.rec[i][0], f.rec[i][1],
                 f.rec[i][2], f.rec[i][3]);
        s += buf;
    }
    return s + "]}";
}
static std::string libm_json(const Cmp &c, bool bounds) {
    char buf[512];
    if (!bounds)
        snprintf(buf, sizeof buf, "{\"arguments\": %llu, \"mismatches\": %llu, \"first_mismatch\": \"0x%08llx\"}",
                 (unsigned long long)c.n.load(), (unsigned long long)c.bad.load(),
                 (unsigned long long)(c.first_bad.load() == ~0ull ? 0 : c.first_bad.load()));
    else
        snprintf(buf, sizeof buf,
                 "{\"arguments\": %llu, \"differs_from_glibc\": %llu, \"over_1ulp_from_glibc\": %llu, \"not_correctly_rounded\": %llu, "
                 "\"glibc_not_correctly_rounded\": %llu, \"undecided\": %llu, \"fraction_differs_from_glibc\": %.3e, "
                 "\"fraction_glibc_not_correctly_rounded\": %.3e}",
                 (unsigned long long)c.n.load(), (unsigned long long)c.dev_vs_glibc.load(), (unsigned long long)c.over_1ulp.load(),
                 (unsigned long long)c.dev_not_cr.load(), (unsigned long long)c.glibc_not_cr.load(),
                 (unsigned long long)c.undecided.load(), (double)c.dev_vs_glibc.load() / std::max<uint64_t>(1, c.n.load()),
                 (double)c.glibc_not_cr.load() / std::max<uint64_t>(1, c.n.load()));
    return buf;
}

int main(int argc, char **argv) {
    const uint32_t stride = argc > 1 ? std::max(1, atoi(argv[1])) : 1u;
    Dev D;
    CK(cudaStreamCreateWithFlags(&D.st, cudaStreamNonBlocking));
    CK(cudaMalloc(&D.out, Dev::CHUNK * 4ull));
    CK(cudaMallocHost(&D.host, Dev::CHUNK * 4ull));
    const size_t N2 = 1u << 24;
    CK(cudaMalloc(&D.x2, N2 * 4));
    CK(cudaMalloc(&D.y2, N2 * 4));
    enum { FA_INRANGE, FA_LEAN, FA_LEAN_N, FC_PAIRS, FC_FM, FD_TICK, FD_PAIR, FE_THR, FE_FLAG, N_FAILS };
    Fails *dfails = nullptr;
    CK(cudaMalloc(&dfails, sizeof(Fails) * N_FAILS));
    CK(cudaMemsetAsync(dfails, 0, sizeof(Fails) * N_FAILS, D.st));
    float *ddts = nullptr;

    // a, b: sine and cosine over all 2^32 floats (positive and negative halves)
    Cmp sin_c, cos_c;
    sweep<F_SIN>(D, sin_c, 0, 1ull << 32, stride);
    sweep<F_COS>(D, cos_c, 0, 1ull << 32, stride);
    {
        const uint32_t groups = (0x42f00000u + LEAN_N - 1) / LEAN_N, threads = (groups + stride - 1) / stride;
        k_sine_forms<<<(threads + 255) / 256, 256, 0, D.st>>>(groups, stride, dfails + FA_INRANGE, dfails + FA_LEAN, dfails + FA_LEAN_N);
        CK(cudaGetLastError());
    }
    // c: every significand pair (2^23 divisors x 2^23 numerators), 2^16 divisors per launch
    {
        const uint32_t per = 1u << 16;
        for (uint32_t d = 0; d < (1u << 23); d += per * stride) {
            k_div_pairs<<<per, 256, 0, D.st>>>(d, stride, dfails + FC_PAIRS);
            CK(cudaGetLastError());
        }
        const float srs[7] = {8000.f, 22050.f, 44100.f, 48000.f, 88200.f, 96000.f, 192000.f};
        for (float sr : srs)
            for (uint64_t b = 0; b < 0x7f800000ull; b += (uint64_t)Dev::CHUNK * stride) {
                const uint32_t n = (uint32_t)std::min<uint64_t>(Dev::CHUNK, 0x7f800000ull - b);
                k_div_fm<<<(n + 255) / 256, 256, 0, D.st>>>((uint32_t)b, n, sr, dfails + FC_FM);
                CK(cudaGetLastError());
            }
    }
    // d: 64 increments: the domain's ends, all-ones significands (and all ones but one bit) at every exponent of the
    // domain, and note pitches at 44.1, 48 and 96 kHz
    std::vector<float> dts = {hf(0x35800000u) /* 2^-20 */, hf(0x3e7fffffu) /* largest below 1/4 */};
    for (uint32_t e = 0x35800000u; e < 0x3e800000u; e += 0x00800000u) dts.push_back(hf(e | 0x7fffffu));
    for (uint32_t e : {0x36000000u, 0x38800000u, 0x3b000000u, 0x3d800000u, 0x3e000000u})
        dts.push_back(hf(e | 0x7ffffeu)), dts.push_back(hf(e | 0x3fffffu)), dts.push_back(hf(e | 0x7fbfffu));
    for (float sr : {44100.f, 48000.f, 96000.f})
        for (float f : {20.f, 27.5f, 55.f, 110.f, 220.f, 261.6256f, 440.f, 880.f, 1760.f, 3520.f, 5000.f, 7040.f, 9000.f})
            if (dts.size() < 64) dts.push_back(f / sr);
    while (dts.size() < 64) dts.push_back(hf(0x3c23d70au + (uint32_t)dts.size() * 7919u)); // around 0.01
    CK(cudaMalloc(&ddts, dts.size() * 4));
    CK(cudaMemcpyAsync(ddts, dts.data(), dts.size() * 4, cudaMemcpyHostToDevice, D.st));
    for (uint64_t b = 0; b < 0x3f800000ull; b += (uint64_t)Dev::CHUNK * stride) {
        const uint32_t n = (uint32_t)std::min<uint64_t>(Dev::CHUNK, 0x3f800000ull - b);
        k_saw<<<(n + 255) / 256, 256, 0, D.st>>>((uint32_t)b, n, ddts, (int)dts.size(), dfails + FD_TICK, dfails + FD_PAIR);
        CK(cudaGetLastError());
    }
    // e: every dt in [2^-20, 1/4)
    k_wrap<<<(0x3e800000u - 0x35800000u + 255) / 256, 256, 0, D.st>>>(0x35800000u, 0x3e800000u - 0x35800000u, dfails + FE_THR,
                                                                        dfails + FE_FLAG);
    CK(cudaGetLastError());
    Fails hfails[N_FAILS];
    CK(cudaMemcpyAsync(hfails, dfails, sizeof hfails, cudaMemcpyDeviceToHost, D.st));
    CK(cudaStreamSynchronize(D.st));

    // f: tan, exp, pow
    Cmp tan_c, exp_c, powdb_c, pow2_c;
    const uint32_t HALF_PI_UP = 0x3fc90fdbu; // the first float above pi/2
    const uint32_t EXP_HI = 0x42b20000u;     // above log(FLT_MAX): results that overflow are skipped
    const uint32_t DB_120 = 0x42f00000u;     // 120.0f
    for (uint64_t s : {0ull, 0x80000000ull}) {
        sweep<F_TAN>(D, tan_c, s, s + HALF_PI_UP, stride);
        sweep<F_POW_DB>(D, powdb_c, s, s + DB_120 + 1, stride);
    }
    sweep<F_EXP>(D, exp_c, 0, EXP_HI, stride);
    sweep<F_EXP>(D, exp_c, 0x80000000ull, 0xff800001ull, stride); // every negative float, -inf included
    {
        // Pow / WrPowf operands: positive bases 2^-16 .. 2^16 (log-uniform) with exponents in [-8, 8], and negative bases with
        // integer exponents
        std::mt19937_64 rng(20261021);
        std::uniform_real_distribution<double> lb(-16.0, 16.0), ye(-8.0, 8.0);
        std::uniform_int_distribution<int> yi(-12, 12);
        std::vector<float> xs(N2 / stride), ys(N2 / stride); // at most N2: the device buffers' size
        for (size_t i = 0; i < xs.size(); i++) {
            xs[i] = (float)exp2(lb(rng));
            ys[i] = (float)ye(rng);
            if (i % 8 == 7) xs[i] = -xs[i], ys[i] = (float)yi(rng);
        }
        sweep<F_POW2>(D, pow2_c, 0, 0, 1, &xs, &ys);
    }

    const char *names[N_FAILS] = {"sin_inrange", "sin_lean", "sin_lean_n", "div_pairs", "div_fm", "saw_tick", "saw_pair",
                                  "wrap_threshold", "wrap_flag"};
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, 0));
    std::string js = "{\"device\": \"" + std::string(prop.name) + "\", \"stride\": " + std::to_string(stride) +
                     ", \"host_threads\": " + std::to_string(n_threads()) + ", \"saw_dts\": " + std::to_string(dts.size()) +
                     ", \"sin\": " + libm_json(sin_c, false) + ", \"cos\": " + libm_json(cos_c, false);
    for (int i = 0; i < N_FAILS; i++) js += ", \"" + std::string(names[i]) + "\": " + fails_json(hfails[i]);
    js += ", \"tan\": " + libm_json(tan_c, true) + ", \"exp\": " + libm_json(exp_c, true) + ", \"pow_db\": " + libm_json(powdb_c, true) +
          ", \"pow_sample\": " + libm_json(pow2_c, true) + "}";
    printf("%s\n", js.c_str());

    CK(cudaFree(ddts));
    CK(cudaFree(dfails));
    CK(cudaFree(D.x2));
    CK(cudaFree(D.y2));
    CK(cudaFreeHost(D.host));
    CK(cudaFree(D.out));
    CK(cudaStreamDestroy(D.st));
    return 0;
}
