/*
 * knaster_gpu.h -- C ABI of the B200 batched render engine for knaster's audio graph.
 *
 * knaster has no plugin/FFI ABI of its own; the seam this library plugs into is the
 * set of Rust types on the audio side of knaster_graph (SURVEY.md 8b).  The entry
 * points below are what a `knaster_gpu` host crate binds with `extern "C"` (see
 * INTEGRATION.md for the Rust-side stub).  All citations are file:line under the
 * reference tree (/root/reference).
 *
 * Conventions: every function returns 0 on success or a negative kgpu_status; the
 * message for the last failure on the calling thread is kgpu_last_error().  Nothing
 * aborts, nothing calls back into the host.  All pointers are caller-owned and only
 * read during the call unless stated.  One host thread drives a plan.  There is no
 * CPU fallback: unsupported UGens / wrappers / wrapper nestings are rejected by
 * kgpu_plan_create, and every entry point fails if no CUDA device is usable.
 */
#ifndef KNASTER_GPU_H
#define KNASTER_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KGPU_ABI_VERSION 1

typedef enum {
    KGPU_OK = 0,
    KGPU_ERR_INVALID = -1,     /* malformed description / out-of-range index (GraphError, graph.rs:2222-2274) */
    KGPU_ERR_UNSUPPORTED = -2, /* UGen / wrapper / graph shape the engine does not implement */
    KGPU_ERR_CUDA = -3,        /* CUDA runtime failure or no device */
    KGPU_ERR_PARAMETER = -4,   /* ParameterError (knaster_core/src/parameters.rs:65-85): bad index / value type */
    KGPU_ERR_STATE = -5,       /* call not valid in the plan's current state */
} kgpu_status;

/* Node kinds: the UGens of knaster_core_dsp/src/ugens that the engine renders. */
typedef enum {
    KGPU_SIN_WT = 1,             /* osc.rs:97-168        params: 0 freq, 1 phase_offset, 2 reset_phase      */
    KGPU_SIN_NUMERIC = 2,        /* osc.rs:222-271       params: 0 freq, 1 phase_offset, 2 reset_phase      */
    KGPU_POLYBLEP = 3,           /* polyblep.rs:128-241  params: 0 freq, 1 pulse_width, 2 waveform          */
    KGPU_SVF = 4,                /* svf.rs:44-280        params: 0 cutoff_freq, 1 q, 2 gain, 3 filter, 4 t_calculate_coefficients */
    KGPU_ONEPOLE_LPF = 5,        /* onepole.rs:111-140   params: 0 cutoff_freq                              */
    KGPU_ONEPOLE_HPF = 6,        /* onepole.rs:144-177   params: 0 cutoff_freq                              */
    KGPU_ENV_ASR = 7,            /* envelopes.rs:19-163  params: 0 attack_time, 1 release_time, 2 t_release, 3 t_restart */
    KGPU_ENV_AR = 8,             /* envelopes.rs:174-303 params: 0 attack_time, 1 release_time, 2 t_restart  */
    KGPU_ENVELOPE = 9,           /* envelopes.rs:359-527 params: 0 time_scale, 1 jump_to_segment, 2 t_restart, 3 t_stop */
    KGPU_MATH = 10,              /* math.rs:94-165       no params; inputs a0..aN-1,b0..bN-1                */
    KGPU_CONSTANT = 11,          /* util.rs:37-64        params: 0 value                                    */
    KGPU_TEST_NUM = 12,          /* knaster_graph/src/tests/utils.rs:4-17  (reference test fixture)          */
    KGPU_TEST_IN_PLUS_PARAM = 13,/* knaster_graph/src/tests/utils.rs:20-67 (reference test fixture)          */
    KGPU_MATH1 = 14,             /* math.rs:167-305      Math1UGen: 1 in, 1 out, no params; mode = kgpu_math1_op */
    KGPU_PHASOR = 15,            /* osc.rs:170-213       params: 0 freq (f64 phase, 0..1 ramp)               */
    /* noise.rs: the RNG is the fastrand 2.3.0 crate (wyrand), which is NOT under the reference tree;
       its published algorithm is restated (csrc/nodes.cuh wy_next).  args[last] = the seed the
       reference would have drawn from its global construction-order counter (noise.rs:11-22).     */
    KGPU_WHITE_NOISE = 16,       /* noise.rs:26-46       no params; args[0] = seed                          */
    KGPU_PINK_NOISE = 17,        /* noise.rs:53-115      no params; args[0] = seed                          */
    KGPU_BROWN_NOISE = 18,       /* noise.rs:122-153     no params; args[0] = seed                          */
    KGPU_RANDOM_LIN = 19,        /* noise.rs:156-217     params: 0 freq; args[0] = freq, args[1] = seed (already *94+53) */
    /* pan.rs: the gains are fastapprox 0.3.1's fast::cos / fast::sin (a crate that is NOT under the reference
       tree; restated from its published source, parity unpinned); 1 input, 2 outputs                     */
    KGPU_PAN2 = 20               /* pan.rs:12-38         params: 0 pan; args[0] = pan (-1..1)                */
} kgpu_ugen_kind;

/* kgpu_node_desc.mode for KGPU_MATH (math.rs:22-85) */
typedef enum { KGPU_OP_ADD = 0, KGPU_OP_SUB = 1, KGPU_OP_MUL = 2, KGPU_OP_DIV = 3, KGPU_OP_POW = 4 } kgpu_math_op;
/* kgpu_node_desc.mode for KGPU_MATH1 (math.rs:172-243) */
typedef enum { KGPU_OP1_CEIL = 0, KGPU_OP1_SQRT = 1, KGPU_OP1_FLOOR = 2, KGPU_OP1_TRUNC = 3, KGPU_OP1_FRACT = 4, KGPU_OP1_EXP = 5 } kgpu_math1_op;

/* Wrappers (knaster_core_dsp/src/wrappers_core.rs:26-56), listed innermost first. */
typedef enum {
    KGPU_WR_MUL = 1,             /* wrappers_core/math.rs:15-113; adds param "wr_mul" at index T::Parameters */
    KGPU_WR_ADD = 2,             /* math.rs:116-192 */
    KGPU_WR_SUB = 3,             /* math.rs:194-270 */
    KGPU_WR_VSUB = 4,            /* math.rs:272-349  value - x */
    KGPU_WR_DIV = 5,             /* math.rs:351-427 */
    KGPU_WR_VDIV = 6,            /* math.rs:429-505  value / x */
    KGPU_WR_POWF = 7,            /* math.rs:507-583  x.powf(value) */
    KGPU_WR_POWI = 8,            /* math.rs:586-661  x.powi(value), value = the i32 exponent */
    KGPU_WR_SMOOTH_PARAMS = 9,   /* smooth_params.rs */
    KGPU_WR_PRECISE_TIMING = 10, /* precise_timing.rs; capacity = DELAYED_CHANGES_PER_BLOCK */
    KGPU_WR_AR_PARAMS = 11       /* audio_rate.rs:11-85 */
} kgpu_wrapper_kind;

typedef struct {
    uint32_t kind;     /* kgpu_wrapper_kind */
    uint32_t capacity; /* KGPU_WR_PRECISE_TIMING: N */
    double value;      /* arithmetic wrappers: the f32 value, passed as f64 */
} kgpu_wrapper_desc;

/* One node as knaster's Graph holds it after push (graph.rs:373-389, node.rs:86).
 * args: SinWt/SinNumeric {freq}; PolyBlep {freq} (mode = Waveform); SvfFilter {cutoff, q, gain_db}
 * (mode = SvfFilterType); OnePoleLpf {cutoff}; EnvAsr/EnvAr {attack_time, release_time};
 * Envelope {start_value, time_scale} + segments; Constant/TestNum {value}; Math: mode = op,
 * channels = N. */
typedef struct {
    uint32_t kind;     /* kgpu_ugen_kind */
    uint32_t mode;
    uint32_t channels;
    uint32_t flags;    /* bit0: Envelope looping (envelopes.rs:392-395) */
    double args[4];
    uint32_t n_wrappers;
    uint32_t n_segments;
    const kgpu_wrapper_desc *wrappers;
    const double *segments; /* Envelope: (duration, value) pairs, envelopes.rs:322-336 */
} kgpu_node_desc;

#define KGPU_SOURCE_NONE (-1)
#define KGPU_GRAPH (-2) /* NodeOrGraph::Graph: graph input as a source, graph output as a sink */

/* An input edge exactly as Graph::node_input_edges / output_edges store it after
 * additive connects were resolved into MathUGen<Add> nodes (graph.rs:768-881). */
typedef struct {
    int32_t source_node;     /* >= 0 node index, KGPU_GRAPH = graph input */
    uint32_t source_channel;
    int32_t sink_node;       /* >= 0 node index, KGPU_GRAPH = graph output */
    uint32_t sink_channel;
} kgpu_edge;

/* Graph::node_parameter_edges (graph.rs:620-760): audio-rate parameter route. */
typedef struct {
    int32_t source_node;
    uint32_t source_channel;
    int32_t sink_node;
    uint32_t param_index;
} kgpu_param_edge;

/* What Graph::commit_changes hands to the audio side (TaskData, graph.rs:1565-1582,
 * task.rs:70-100) plus AudioProcessorOptions (processor.rs:23-45). */
typedef struct {
    uint32_t abi_version;  /* KGPU_ABI_VERSION */
    uint32_t sample_rate;
    uint32_t block_size;
    uint32_t n_inputs;     /* graph inputs (<= 65536; at most 16 of them shared, see kgpu_render_inputs): rendered with
                              kgpu_render_inputs[_device]; 0: run_without_inputs() */
    uint32_t n_outputs;    /* 1..8 */
    int32_t device;        /* CUDA device ordinal, -1 = current */
    uint32_t n_nodes;
    uint32_t n_edges;
    uint32_t n_param_edges;
    uint32_t flags;        /* KGPU_PLAN_* */
    const kgpu_node_desc *nodes;
    const kgpu_edge *edges;
    const kgpu_param_edge *param_edges;
} kgpu_graph_desc;

#define KGPU_PLAN_FORCE_INTERPRETER 1u /* use the generic plan interpreter even if a fused kernel matches */
#define KGPU_PLAN_FORCE_JIT 4u         /* generate a kernel per voice template (csrc/jit.cpp) even for banks below the size at which the
                                          compilation pays for itself (default: >= 256 voices; KGPU_JIT=0 turns generation off) */
#define KGPU_PLAN_NO_SCAN 2u           /* small saw -> SVF -> EnvAsr banks: keep the bit-exact one-lane-per-voice kernel instead of
                                          the time-parallel scan kernel (render_sub_scan, <= 1e-4 on the filter) */

/* SchedulingEvent (scheduling.rs:29-36) + Time (scheduling.rs:73-92) + ParameterValue
 * (parameters/types.rs:25-37).  Tokens are not supported (SchedulingToken::activate is
 * todo!() in the reference, scheduling.rs:175-178). */
typedef struct {
    uint32_t node;
    uint32_t param;
    uint32_t value_kind;     /* 0 none, 1 Float, 2 Trigger, 3 Integer, 4 Bool */
    uint32_t smoothing_kind; /* 0 no smoothing field, 1 ParameterSmoothing::None, 2 Linear(smooth_seconds) */
    double value;
    float smooth_seconds;
    uint32_t smooth_rate;    /* 0 Rate::BlockRate; Rate::AudioRate is rejected (SURVEY App. B4) */
    uint32_t time_kind;      /* 0 None (next block), 1 Time::at (absolute), 2 Time::after (relative) */
    uint32_t seconds;        /* Seconds.seconds            (knaster_primitives/src/time.rs:25-28) */
    uint32_t subsec;         /* Seconds.subsecond_tesimals (1/282 240 000 s) */
    uint32_t _pad;
} kgpu_event;

typedef struct kgpu_plan kgpu_plan; /* opaque, owned by the library */

/* Compile the graph into a fixed kernel plan and upload it (replaces TaskData generation +
 * hand-over, graph.rs:1707-1726 / graph_gen.rs:93-109; node init = graph.rs:462-475). */
int kgpu_plan_create(const kgpu_graph_desc *desc, kgpu_plan **out);
void kgpu_plan_destroy(kgpu_plan *plan);

/* Queue parameter changes (replaces the rtrb scheduling ring, handle.rs:38-73 and
 * graph_gen.rs:111-166,269-305).  Events take effect as if each had reached knaster's
 * audio thread in the block that contains its due frame, in push order; late events
 * apply at the next rendered block.  Unlike knaster nothing is ever dropped for waiting
 * too long or for a full ring (documented divergence, SURVEY App. B6).  Per-node
 * WrPreciseTiming capacity overflow IS reproduced (the change is dropped and counted). */
int kgpu_plan_push_events(kgpu_plan *plan, const kgpu_event *events, size_t n_events);

/* AudioProcessor::run_without_inputs (processor.rs:142-148): render one block. */
int kgpu_render_block(kgpu_plan *plan);
/* AudioProcessor::output_block (processor.rs:182-184): host copy of the last block,
 * [n_outputs][block_size], valid until the next render call. */
const float *kgpu_output_block(kgpu_plan *plan);
/* Render n_blocks back to back.  host_out: [n_blocks][n_outputs][block_size] or NULL. */
int kgpu_render(kgpu_plan *plan, uint64_t n_blocks, float *host_out);
/* AudioProcessor::run(&[&[F]]) (processor.rs:119-141), batched: the graph's inputs for n_blocks blocks,
 * host_in: [n_blocks][n_inputs][block_size].  A graph with inputs is rendered with this call or kgpu_render_inputs_device only
 * (kgpu_render* fail with KGPU_ERR_STATE, like run_without_inputs() asserts inputs() == 0, processor.rs:143); host_out as in
 * kgpu_render.
 * An input that only one voice reads (a track through its own effect chain) is a port of that voice: the kernels read it
 * from the input blocks in place, so a graph may have up to 65536 such inputs.  Any other input -- read by several voices,
 * summed into a mix or wired straight to an output -- is shared: at most 16 per graph.  host_in is staged launch by launch
 * through two page-locked buffers of one launch each (a launch's input slice is at most 256 MiB), each copy beside the
 * previous launch's rendering; host_in is read during the call only. */
int kgpu_render_inputs(kgpu_plan *plan, uint64_t n_blocks, const float *host_in, float *host_out);
/* The same with the input blocks already in DEVICE memory on the plan's device (device_in, same layout; read in place, no
 * copy, and it does not limit the launch length) and the result left in device memory as kgpu_render_device does: enqueued on
 * `cuda_stream` (NULL = the plan's own stream) without synchronising.  device_in must stay valid until the work has run.
 * A plan whose voices have ports cannot be sharded over a peer bus (KGPU_ERR_UNSUPPORTED). */
int kgpu_render_inputs_device(kgpu_plan *plan, uint64_t n_blocks, const float *device_in, float *device_out, void *cuda_stream);
/* Same, leaving the result in DEVICE memory (device_out: n_blocks*n_outputs*block_size floats
 * on the plan's device) and enqueued on `cuda_stream` (a cudaStream_t, NULL = the plan's own
 * stream) without synchronising: the multi-GPU path reduces the bus from here. */
int kgpu_render_device(kgpu_plan *plan, uint64_t n_blocks, float *device_out, void *cuda_stream);
/* Block until everything enqueued by the plan has finished. */
int kgpu_plan_synchronize(kgpu_plan *plan);

/* AudioProcessor accessors (processor.rs:186-197) and the frame clock (processor.rs:57). */
uint32_t kgpu_plan_block_size(const kgpu_plan *plan);
uint32_t kgpu_plan_outputs(const kgpu_plan *plan);
uint64_t kgpu_plan_frame_clock(const kgpu_plan *plan);

/* Pre-mix tap: record output `channel` of `node` for every rendered frame (parity/debug).
 * Must be called before the first render.  Returns the tap index (>= 0). */
int kgpu_plan_add_tap(kgpu_plan *plan, uint32_t node, uint32_t channel);
/* Copy the frames recorded by the last kgpu_render* call: out[n_taps][n_frames]. */
int kgpu_plan_read_taps(kgpu_plan *plan, float *out, uint64_t n_frames);

/* Introspection of the compiled plan. */
typedef struct {
    uint32_t n_groups;          /* voice templates found (isomorphic voice sub-graphs batched SoA) */
    uint32_t n_voices;          /* total voices over all groups */
    uint32_t n_mix_nodes;       /* Add nodes folded into the mix-bus reduction (graph.rs:850-864) */
    uint32_t n_fused_groups;    /* groups rendered by a fused kernel (rest: plan interpreter) */
    uint64_t state_bytes;       /* per-voice register bytes summed over voices */
    uint64_t dropped_changes;   /* WrPreciseTiming queue overflows so far (precise_timing.rs:129-134) */
    uint64_t ignored_delays;    /* set_delay calls that reached no WrPreciseTiming (ugen.rs:339-341) */
    uint64_t device_events;     /* device register-write events generated so far */
    uint64_t kernel_launches;   /* engine kernels launched so far */
} kgpu_plan_info;
int kgpu_plan_get_info(kgpu_plan *plan, kgpu_plan_info *info);
/* Name of the kernel that renders group `group` ("render_interp", "render_fused<...>", ...). */
const char *kgpu_plan_group_kernel(kgpu_plan *plan, uint32_t group);
/* Device time (ms, CUDA events on the plan's stream) spent in render kernels by the last
 * kgpu_render* call that has completed; <0 if unavailable. */
float kgpu_plan_last_render_ms(kgpu_plan *plan);

/* Optional split of a render call: do the host work of the next n_blocks (control-rate
 * simulation of the queued parameter changes + upload of the resulting device events) now, so
 * that the following kgpu_render*(plan, n_blocks, ..) only launches kernels. */
int kgpu_plan_prepare(kgpu_plan *plan, uint64_t n_blocks);
/* Device time (ms, CUDA events around each launch) of the last render call, summed per kernel
 * class: 0 = voice-bank render kernels, 1 = reduce_bus.  *n_launches receives the launch count. */
float kgpu_plan_last_kernel_ms(kgpu_plan *plan, uint32_t kernel_class, uint32_t *n_launches);
/* Host-to-device bytes (compiled parameter events) uploaded by the last kgpu_render* call. */
uint64_t kgpu_plan_last_upload_bytes(kgpu_plan *plan);
/* K = blocks rendered per kernel launch (default: as many as fit a 256 MiB partial-sum buffer,
 * at most 2048).  K = 1 reproduces "one launch per 64-frame block". */
int kgpu_plan_set_blocks_per_launch(kgpu_plan *plan, uint64_t blocks);
/* ---- snapshot / restore (no counterpart in the reference: knaster cannot rewind a running graph) ------------
 * kgpu_plan_snapshot copies the whole render state of the plan -- the voices' registers (device -> host), the
 * control-side state of every node of every voice, the queued events, the frame clock and the counters -- into
 * an object owned by the caller; kgpu_plan_restore puts it back (events pushed after the snapshot are gone,
 * the next render continues from the snapshot's frame clock).  Not valid between kgpu_plan_prepare and its
 * render.  With a peer bus every rank snapshots / restores at the same point. */
typedef struct kgpu_snapshot kgpu_snapshot;
int kgpu_plan_snapshot(kgpu_plan *plan, kgpu_snapshot **out);
int kgpu_plan_restore(kgpu_plan *plan, const kgpu_snapshot *snapshot);
void kgpu_snapshot_destroy(kgpu_snapshot *snapshot);
/* A snapshot as bytes (checkpoint on disk; restore into a plan created from the same graph description, in
 * this or another process).  Serialize: call with buf == NULL to get the size, then with a buffer of at least
 * that many bytes.  Deserialize rejects truncated, foreign or other-version images with KGPU_ERR_INVALID. */
int kgpu_snapshot_serialize(const kgpu_snapshot *snapshot, void *buf, uint64_t cap, uint64_t *size);
int kgpu_snapshot_deserialize(const void *buf, uint64_t size, kgpu_snapshot **out);

/* ---- multi-GPU mix bus over peer memory -------------------------------------------------------
 * One process per GPU, voices sharded across ranks (SURVEY 8e).  Instead of reducing the rank-local
 * buses with a collective afterwards, every rank's bus-reduction kernel stores straight into its slot
 * of ONE buffer that lives in rank 0's memory (peer stores over NVLink) and publishes each launch
 * with a system-scope flag; rank 0 folds the slots in rank order as the launches arrive, beside the
 * rendering of the next launch.  knaster has no counterpart (one process, one audio thread): this is
 * the distributed form of the graph-out Add chain (graph.rs:850-864).
 *
 * root_buffer: device pointer, valid ON THIS RANK, to the same allocation in rank 0's memory (rank 0:
 * its own allocation; other ranks: a peer mapping of it, e.g. from CUDA IPC or torch symmetric
 * memory), kgpu_peer_bus_bytes(world, floats_per_rank) bytes, zero-filled before the first render,
 * 16-byte aligned.  floats_per_rank >= n_blocks * block_size * outputs of the largest render call.
 * Every rank must make the same sequence of kgpu_render* calls.  Only rank 0's output buffer
 * receives audio (the sum over all ranks); the other ranks' output buffers are left untouched.
 * world <= 1 or root_buffer == NULL detaches. */
#define KGPU_PEER_MAX_LAUNCHES 16384 /* 10 s at one launch per 64-frame block (configs[4] read literally) is 7500 */
uint64_t kgpu_peer_bus_header_bytes(uint32_t world);
uint64_t kgpu_peer_bus_bytes(uint32_t world, uint64_t floats_per_rank);
int kgpu_plan_set_peer_bus(kgpu_plan *plan, uint32_t rank, uint32_t world, void *root_buffer, uint64_t buffer_bytes);
/* 1 if a rank gave up waiting (~2 s) for another rank's data since the buffer was zero-filled. */
int kgpu_plan_peer_bus_timed_out(kgpu_plan *plan);

/* Host worker threads a plan uses for the control-rate simulation (validation, bucketing and the
 * per-voice event replay that runs one launch ahead of the device).  0 = default: hardware threads
 * - 1, at most 16.  Call before the first render; with several plans/processes per box (one per
 * GPU) give each its share of the cores.  No counterpart in knaster, which renders on one thread. */
int kgpu_plan_set_host_threads(kgpu_plan *plan, uint32_t n_threads);

const char *kgpu_last_error(void); /* thread-local */
uint32_t kgpu_abi_version(void);
/* Number of usable CUDA devices (0 if none / driver missing). */
int kgpu_device_count(void);

#ifdef __cplusplus
}
#endif
#endif
