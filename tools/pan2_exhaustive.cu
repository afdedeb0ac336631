// pan2_exhaustive.cu -- Pan2's gains on the device against the host, for every float.  A Pan2 whose `pan` is routed at audio
// rate evaluates pan2_gains(x * 0.5 + 0.5) (knaster_b200/csrc/fastapprox.h) in the kernels every frame; without a route the
// host plan evaluates the same header when a pan event arrives.  Both must give the same two gains for every sample x, so this
// runs the device instantiation over all 2^32 floats x and compares both gains bitwise with the host instantiation (NaN
// matches NaN).  Built with the library's numeric flags, host side as plan.cpp (-ffp-contract=off).  Prints one JSON line;
// tests/test_gpu_ar_routes.py builds and runs it:
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -fmad=false -prec-div=true -prec-sqrt=true -ftz=false
//        -Xcompiler -ffp-contract=off,-fno-fast-math -Iknaster_b200/csrc tools/pan2_exhaustive.cu -o pan2_exhaustive -lpthread
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "fastapprox.h"

using namespace kgpu;

#define CK(x)                                                                                                              \
    do {                                                                                                                   \
        cudaError_t e_ = (x);                                                                                              \
        if (e_ != cudaSuccess) {                                                                                           \
            fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));                              \
            exit(2);                                                                                                       \
        }                                                                                                                  \
    } while (0)

__global__ void k_gains(uint32_t first, uint32_t n, float *__restrict__ gl, float *__restrict__ gr) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = __uint_as_float(first + i);
    float l, r;
    pan2_gains(x * 0.5f + 0.5f, l, r); // the routed form: pan.rs:26-29 then :31-35
    gl[i] = l;
    gr[i] = r;
}

static bool same(float a, float b) {
    if (std::isnan(a) || std::isnan(b)) return std::isnan(a) && std::isnan(b);
    uint32_t ua, ub;
    memcpy(&ua, &a, 4);
    memcpy(&ub, &b, 4);
    return ua == ub;
}

int main() {
    const uint32_t CHUNK = 1u << 28;
    float *d_l, *d_r, *h_l, *h_r;
    CK(cudaMalloc(&d_l, (size_t)CHUNK * 4));
    CK(cudaMalloc(&d_r, (size_t)CHUNK * 4));
    CK(cudaMallocHost(&h_l, (size_t)CHUNK * 4));
    CK(cudaMallocHost(&h_r, (size_t)CHUNK * 4));
    cudaStream_t st;
    CK(cudaStreamCreate(&st));
    const unsigned n_thr = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    std::atomic<unsigned long long> mismatches{0}, nan{0}, finite{0};
    std::atomic<uint32_t> first_bad{0};
    std::atomic<bool> any_bad{false};
    for (uint64_t c0 = 0; c0 < (1ull << 32); c0 += CHUNK) {
        k_gains<<<CHUNK / 256, 256, 0, st>>>((uint32_t)c0, CHUNK, d_l, d_r);
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(h_l, d_l, (size_t)CHUNK * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h_r, d_r, (size_t)CHUNK * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        std::vector<std::thread> th;
        for (unsigned t = 0; t < n_thr; t++)
            th.emplace_back([&, t] {
                unsigned long long bad = 0, nn = 0, fin = 0;
                for (uint64_t i = t; i < CHUNK; i += n_thr) {
                    const uint32_t bits = (uint32_t)(c0 + i);
                    float x;
                    memcpy(&x, &bits, 4);
                    float l, r;
                    pan2_gains(x * 0.5f + 0.5f, l, r);
                    if (std::isnan(l) || std::isnan(r)) nn++;
                    else fin++;
                    if (!same(l, h_l[i]) || !same(r, h_r[i])) {
                        if (!any_bad.exchange(true)) first_bad = bits;
                        bad++;
                    }
                }
                mismatches += bad;
                nan += nn;
                finite += fin;
            });
        for (auto &t : th) t.join();
    }
    CK(cudaStreamDestroy(st));
    CK(cudaFree(d_l));
    CK(cudaFree(d_r));
    CK(cudaFreeHost(h_l));
    CK(cudaFreeHost(h_r));
    printf("{\"arguments\": %llu, \"mismatches\": %llu, \"first_mismatch_bits\": %u, \"nan\": %llu, \"finite\": %llu}\n", 1ull << 32,
           (unsigned long long)mismatches, (unsigned)first_bad, (unsigned long long)nan, (unsigned long long)finite);
    return 0;
}
