// fastapprox.h -- Pan2's gains (pan.rs:31-36), usable on host and device.
//
// knaster's Pan2 evaluates fastapprox 0.3.1's fast::cos / fast::sin (Paul Mineiro's fastcos / fastsin) of its stored pan
// position every sample.  The crate is not under the reference tree: parity of these two functions is unpinned
// (DESIGN.md section 7).  This is the engine's one restatement of them: the host plan evaluates it when a `pan` event
// arrives, the kernels every frame while `pan` is driven at audio rate.  The oracle keeps its own, independent restatement.
// Every f32 operation rounds once (the library's -fmad=false / -ffp-contract=off); tests/test_gpu_ar_routes.py checks the
// device instantiation against the host one for all 2^32 pan values (tools/pan2_exhaustive.cu).
#pragma once
#include <stdint.h>
#include <string.h>
#if defined(__CUDACC__)
#define KN_FA_HD __host__ __device__ __forceinline__
#else
#define KN_FA_HD inline
#endif

namespace kgpu {

KN_FA_HD uint32_t fa_bits(float f) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(f);
#else
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
#endif
}
KN_FA_HD float fa_from_bits(uint32_t u) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
}
KN_FA_HD float fa_sin(float x) {
    const float FOUROVERPI = 1.2732395447351627f, FOUROVERPISQ = 0.40528473456935109f, Q = 0.78444488374548933f;
    uint32_t p = fa_bits(0.20363937680730309f), r = fa_bits(0.015124940802184233f), s = fa_bits(-0.0032225901625579573f);
    uint32_t v = fa_bits(x);
    const uint32_t sign = v & 0x80000000u;
    v &= 0x7FFFFFFFu;
    const float qpprox = FOUROVERPI * x - FOUROVERPISQ * x * fa_from_bits(v);
    const float qpproxsq = qpprox * qpprox;
    p |= sign;
    r |= sign;
    s ^= sign;
    return Q * qpprox + qpproxsq * (fa_from_bits(p) + qpproxsq * (fa_from_bits(r) + qpproxsq * fa_from_bits(s)));
}
KN_FA_HD float fa_cos(float x) {
    const float HALFPI = 1.5707963267948966f, HALFPIMINUSTWOPI = -4.7123889803846899f;
    return fa_sin(x + (x > HALFPI ? HALFPIMINUSTWOPI : HALFPI));
}
// Pan2::process's two gains for a stored pan position (pan.rs:31-35)
KN_FA_HD void pan2_gains(float pan01, float &gl, float &gr) {
    const float rad = pan01 * 1.57079632679489661923f; // core::f32::consts::FRAC_PI_2
    gl = fa_cos(rad);
    gr = fa_sin(rad);
}

} // namespace kgpu
