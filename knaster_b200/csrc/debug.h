/* debug.h -- host-only introspection of the plan / event compilers.  NOT part of the drop-in
 * ABI (include/knaster_gpu.h); used by the CPU test-suite to check the control-rate simulation
 * without a GPU.  None of these functions touch CUDA. */
#ifndef KNASTER_GPU_DEBUG_H
#define KNASTER_GPU_DEBUG_H
#include "../../include/knaster_gpu.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    uint32_t group, voice, node; /* node: index inside the voice template */
    uint32_t op, reg, value;
    uint64_t frame;              /* absolute frame at which the device applies it */
} kgpu_debug_event;

typedef struct {
    int32_t group;   /* -1: mix-bus Add / unreachable */
    uint32_t voice, local, reg_base;
} kgpu_debug_node;

/* Compile `desc`, push `events`, simulate n_blocks from frame 0 in sub-ranges of
 * `blocks_per_call` blocks (as a sequence of render calls would), and return every device
 * event in device order per voice.  nodes_out: one record per graph node (may be NULL). */
int kgpu_debug_simulate(const kgpu_graph_desc *desc, const kgpu_event *events, size_t n_events,
                        uint64_t n_blocks, uint64_t blocks_per_call, kgpu_debug_event *out, size_t cap,
                        size_t *n_out, kgpu_debug_node *nodes_out, kgpu_plan_info *info);
/* Times the host half of n_steps render calls (no device): see capi.cpp.  out_ms: [n_steps][4]. */
int kgpu_debug_host_bench(const kgpu_graph_desc *desc, const kgpu_event *events, size_t n_events, uint64_t n_blocks, uint64_t bpl,
                          uint32_t n_steps, uint32_t n_threads, double *out_ms);
/* Generate + compile (NVRTC, cubin cache) the kernels of the voice templates of `desc` that have no hand-written recipe. */
int kgpu_debug_jit_compile(const kgpu_graph_desc *desc, uint32_t tap_outputs, uint32_t *n_generated, uint32_t *n_cached);
/* The generated CUDA source of the same templates, concatenated, each followed by "\n// ---- end of template\n" (no NVRTC).
 * Call with buf == NULL for *len; copies at most cap bytes. */
int kgpu_debug_jit_source(const kgpu_graph_desc *desc, uint32_t tap_outputs, char *buf, uint64_t cap, uint64_t *len);
/* initial register value of a node register after init() */
int kgpu_debug_init_reg(const kgpu_graph_desc *desc, uint32_t node, uint32_t reg_offset, uint32_t *value);

/* host instantiation of the device sine (csrc/sinf_glibc.h), for the libm bit-exactness test */
int kgpu_debug_sinf(const float *x, float *y, size_t n);

#ifdef __cplusplus
}
#endif
#endif
