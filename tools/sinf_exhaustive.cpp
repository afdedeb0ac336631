// sinf_exhaustive.cpp -- compares the restatements of glibc's sinf and cosf in knaster_b200/csrc/sinf_glibc.h (host
// instantiation: the same f64 and integer operations the device executes) with the libm this machine runs, for EVERY float:
//   kn_sinf_glibc, kn_cosf_glibc           all 2^32 bit patterns (NaN wherever libm gives NaN, else the same bits)
//   kn_sinf_glibc_inrange, kn_sinf_glibc_lean   every |y| < 120 (2 x 0x42f00000 arguments), their domain
// Test infrastructure (tests/test_sinf_exhaustive.py builds and runs it); prints one JSON line.
//   g++ -O2 -mfma -ffp-contract=off -pthread -Iknaster_b200/csrc tools/sinf_exhaustive.cpp -o sinf_exhaustive
// usage: sinf_exhaustive [stride]   (stride 1 = all arguments; k = every k-th bit pattern)
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "sinf_glibc.h"

static uint32_t bits(float f) {
    uint32_t b;
    memcpy(&b, &f, 4);
    return b;
}
// the same result: identical bits, or both NaN (a NaN's payload and sign are not part of sinf's contract)
static bool same(float ref, float got) { return std::isnan(ref) ? std::isnan(got) : bits(ref) == bits(got); }

int main(int argc, char **argv) {
    const uint32_t stride = argc > 1 ? (uint32_t)atoi(argv[1]) : 1u;
    const uint32_t LIM = 0x42f00000u; // 120.0f
    const unsigned T = std::max(1u, std::thread::hardware_concurrency());
    std::atomic<uint64_t> n_args{0}, n_inrange{0}, bad_sin{0}, bad_cos{0}, bad_inrange{0}, bad_lean{0}, lean_zero_sign{0};
    std::vector<std::thread> th;
    for (unsigned w = 0; w < T; w++)
        th.emplace_back([&, w] {
            uint64_t n = 0, m = 0, s = 0, c = 0, a = 0, b = 0, z = 0;
            for (uint64_t i = (uint64_t)w * stride; i < 0x80000000u; i += (uint64_t)T * stride)
                for (uint32_t sgn = 0; sgn < 2; sgn++) {
                    const uint32_t yb = (uint32_t)i | (sgn << 31);
                    float y;
                    memcpy(&y, &yb, 4);
                    const float rs = sinf(y);
                    n++;
                    if (!same(rs, kgpu::kn_sinf_glibc(y))) s++;
                    if (!same(cosf(y), kgpu::kn_cosf_glibc(y))) c++;
                    if (i >= LIM) continue;
                    const float f1 = kgpu::kn_sinf_glibc_inrange(y), f2 = kgpu::kn_sinf_glibc_lean(y);
                    m++;
                    if (bits(rs) != bits(f1)) a++;
                    if (bits(rs) != bits(f2)) {
                        if (rs == f2) z++; // -0.0 against +0.0
                        else b++;
                    }
                }
            n_args += n, n_inrange += m, bad_sin += s, bad_cos += c, bad_inrange += a, bad_lean += b, lean_zero_sign += z;
        });
    for (auto &t : th) t.join();
    printf("{\"arguments\": %llu, \"inrange_arguments\": %llu, \"stride\": %u, \"threads\": %u, \"sin_mismatches\": %llu, "
           "\"cos_mismatches\": %llu, \"inrange_mismatches\": %llu, \"lean_mismatches\": %llu, \"lean_zero_sign_only\": %llu, "
           "\"fma_cpu\": %s}\n",
           (unsigned long long)n_args.load(), (unsigned long long)n_inrange.load(), stride, T, (unsigned long long)bad_sin.load(),
           (unsigned long long)bad_cos.load(), (unsigned long long)bad_inrange.load(), (unsigned long long)bad_lean.load(),
           (unsigned long long)lean_zero_sign.load(), __builtin_cpu_supports("fma") ? "true" : "false");
    return 0;
}
