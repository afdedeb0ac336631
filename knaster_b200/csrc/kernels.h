// kernels.h -- launch interface between the plan runtime (capi.cpp) and the CUDA kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dev.h"
#include "launch_args.h" // struct FusedArgs (also compiled by NVRTC for the generated kernels, jit.cpp)

namespace kgpu {

struct InterpArgs {
    const DevProgram *prog; // device
    uint32_t *regs;         // [n_regs][n_voices]
    uint32_t n_voices;
    const DevEvent *events; // device, sorted per voice in processing order; NULL if none this launch
    const uint32_t *ev_off; // [n_voices+1]
    uint32_t n_frames;
    uint32_t chunk;         // frames per interpreter chunk (power of two <= 64 that divides block_size, capi.cpp pick_chunk)
    float *partials;        // [rows][n_frames]
    uint32_t row0;          // first partial row of this group
    const DevTap *taps;
    uint32_t n_taps;
    float *tap_out;         // [n_taps][tap_stride]
    uint64_t tap_stride;
    uint64_t tap_frame0;
    const float *sine_table; // device, 16384 f32 (wavetable.rs:130-139)
    const float *ext;        // internal signals [signal][ext_stride] of this launch; NULL if none
    uint32_t ext_stride;
    const float *in;         // ports (dev.h): the caller's input blocks [block][n_in][block_size] from the launch's first block
    uint32_t n_in, block_size;
};

cudaError_t launch_interp(const InterpArgs &a, uint32_t n_regs, uint32_t n_slots, cudaStream_t stream);
cudaError_t launch_reduce_bus(const float *partials, const uint32_t *row_mask, uint32_t n_rows, uint32_t n_frames, float *out,
                              uint32_t n_out, uint32_t block_size, cudaStream_t stream);

// internal signals (plan.hpp): signal s = sum of the partial rows [0, n_rows) whose mask has bit (first_bit + s), for the
// signals listed in `which` (n_which of them), written to sig[s * n_frames + frame]
cudaError_t launch_reduce_signals(const float *partials, const uint32_t *row_mask, uint32_t n_rows, uint32_t n_frames, float *sig,
                                  uint32_t first_bit, const uint32_t *which, uint32_t n_which, cudaStream_t stream);

// graph inputs wired straight into graph outputs: out[block][pairs[2k+1]][i] += sig[pairs[2k]][frame]
cudaError_t launch_add_inputs(const float *sig, uint32_t n_frames, float *out, uint32_t n_out, uint32_t block_size, const uint32_t *pairs,
                              uint32_t n_pairs, cudaStream_t stream);

// multi-GPU mix bus over peer memory (kernels.cu)
cudaError_t launch_signal_flag(uint32_t *flag, uint32_t value, cudaStream_t stream);
cudaError_t launch_wait_flag(const uint32_t *flag, uint32_t value, uint32_t *timeout_flag, cudaStream_t stream);
cudaError_t launch_sum_slots(const float *slots, size_t slot_stride, uint32_t world, const uint32_t *flags, uint32_t flag_stride, uint32_t epoch,
                             float *out, size_t n, uint32_t *timeout_flag, cudaStream_t stream);

// fused bank kernels (fused.cu): struct FusedArgs is in launch_args.h
// recipe 0 (render_sub_asr) is replaced by recipe 4 (render_sub_scan) for banks this small (fused.cu)
bool sub_scan_applies(uint32_t n_voices, uint32_t block_size);
// number of partial rows a fused recipe produces for n_voices voices
uint32_t fused_rows(int recipe, uint32_t n_voices, uint32_t n_ubus);
cudaError_t launch_fused(int recipe, const FusedArgs &a, cudaStream_t stream);
// device scratch a recipe needs for one launch of n_frames frames (0 for most)
size_t fused_scratch_bytes(int recipe, uint32_t n_voices, uint32_t n_frames, uint32_t block_size);

// recipe 2 (fused_wt.cu)
bool match_add_wt(const DevProgram &p, uint32_t block_size);
uint32_t add_wt_slices(uint32_t n_voices);
size_t add_wt_scratch_bytes(uint32_t n_voices, uint32_t n_frames, uint32_t block_size);
cudaError_t launch_add_wt(const FusedArgs &a, cudaStream_t stream);

} // namespace kgpu
