// plan.hpp -- host side of the engine: graph -> voice templates -> kernel plan, and the
// control-rate simulation that turns knaster's parameter-change queue into device events.
#pragma once
#include <cstdint>
#include <functional>
#include <memory>
#include <string>
#include <cstddef>
#include <cstdlib>
#include <vector>

#include "../../include/knaster_gpu.h"
#include "dev.h"

namespace kgpu {

struct Error {
    int code;
    std::string msg;
};
#define KGPU_THROW(code_, ...) throw ::kgpu::Error{(code_), ::kgpu::format(__VA_ARGS__)}
std::string format(const char *fmt, ...);

// ParameterValue (knaster_core/src/parameters/types.rs:25-37)
struct PV {
    enum Kind : uint8_t { None = 0, Float = 1, Trigger = 2, Integer = 3, Bool = 4, Smoothing = 5 } kind = None;
    double f = 0.0;      // Float / Integer / Bool payload
    uint8_t smoothing = 0; // Smoothing: 0 ParameterSmoothing::None, 1 Linear
    float smooth_seconds = 0.f;
};

// smooth_params.rs:249-261
struct SmoothState {
    bool linear = false;
    double current_value = 0.0;
    double start_value = 0.0, end_value = 0.0;
    uint64_t duration_frames = 0, frames_elapsed = 0;
    bool done = true;
};

struct QueuedChange { // precise_timing.rs:17
    uint16_t delay;
    uint32_t param;
    PV value;
};

// control-side state of one wrapper instance
struct WrapSim {
    uint8_t kind = 0;        // kgpu_wrapper_kind
    uint32_t capacity = 0;   // WrPreciseTiming<N>
    uint16_t reg = 0;        // arithmetic wrappers: register holding the value
    uint32_t inner_params = 0; // T::Parameters of what it wraps
    std::vector<SmoothState> smooth;   // WrSmoothParams, one per parameter
    std::vector<uint16_t> next_delay;  // WrPreciseTiming, sticky (App. B1)
    std::vector<QueuedChange> queue;   // WrPreciseTiming waiting_changes[0..next_delay_i)
    std::vector<uint8_t> ar_bound;     // WrArParams: parameter has a buffer (audio_rate.rs:70-74)
};

// control-side state of one node of one voice: the fields knaster's setters read/write
// Allocator of the host path's big arrays (the event queue, the control-side nodes): allocations of 2 MiB and more are aligned
// to 2 MiB and advised as huge pages -- the control simulation walks them with a stride of a voice, and with 4 KiB pages the
// tens of megabytes one plan touches are far beyond the TLB's reach (every first touch of a voice's events was a page walk on top
// of the cache miss).  The advice is a hint: where transparent huge pages are off nothing changes.
void *kgpu_big_alloc(size_t bytes, size_t align);
template <class T> struct HugeAllocator {
    using value_type = T;
    HugeAllocator() = default;
    template <class U> HugeAllocator(const HugeAllocator<U> &) noexcept {}
    template <class U> struct rebind { using other = HugeAllocator<U>; };
    T *allocate(size_t n) { return static_cast<T *>(kgpu_big_alloc(n * sizeof(T), alignof(T))); }
    void deallocate(T *p, size_t) noexcept { free(p); }
    template <class U> bool operator==(const HugeAllocator<U> &) const noexcept { return true; }
    template <class U> bool operator!=(const HugeAllocator<U> &) const noexcept { return false; }
};
// ... whose value-less construct() default-initialises: vector::resize() of a POD then leaves
// the new elements uninitialised instead of zero-filling them (HostPlan::push fills them in parallel)
template <class T> struct DefaultInitAllocator : HugeAllocator<T> {
    DefaultInitAllocator() = default;
    template <class U> DefaultInitAllocator(const DefaultInitAllocator<U> &) noexcept {}
    template <class U> struct rebind { using other = DefaultInitAllocator<U>; };
    template <class U> void construct(U *p) noexcept { ::new (static_cast<void *>(p)) U; }
    template <class U, class... A> void construct(U *p, A &&...a) { ::new (static_cast<void *>(p)) U(std::forward<A>(a)...); }
};

// One cache line of what the control simulation reads and writes per parameter change, then the rest: the walk over the voices
// is latency-bound (megabytes of other voices between two visits of a voice), so a node costs one line, fetched ahead of its use.
struct alignas(64) HostNode {
    // ---- hot: the fast path of a parameter change (ugen_param_apply, fast_node_block)
    uint8_t kind = 0;        // kgpu_ugen_kind
    uint8_t dev_kind = 0;
    bool ramp_active = false;
    bool ar_regs = false;    // SvfFilter with an audio-rate route into cutoff / q / gain: the parameters live on the device too
    uint16_t reg = 0;        // register base inside the voice
    uint16_t n_seg = 0;
    uint32_t mode = 0;       // waveform / filter type
    // SinWt.freq, PolyBlep.freq_in_hz; Svf cutoff,q,gain; EnvAsr attack_seconds,release_seconds
    float f0 = 0.f, f1 = 0.f, f2 = 0.f;
    float svf_coef[6] = {0, 0, 0, 0, 0, 0};
    // WrPreciseTiming::next_delay of a node on the fast path (NodeStatic::fast): sticky, App. B1.  Such a node keeps
    // no WrapSim at all -- everything else about its wrapper stack is static and lives in the template's NodeStatic.
    uint16_t nd[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // ---- the second line: nodes with WrSmoothParams / Envelope / Phasor, plan-time data
    double d0 = 0.0;         // Envelope start_value
    uint32_t base_params = 0;
    uint32_t ramp_list_pos = 0;
    bool has_smooth = false, has_precise = false;
    int8_t smooth_level = -1, precise_level = -1;
    std::vector<WrapSim> wr; // innermost first
};
static_assert(sizeof(HostNode) == 128 && offsetof(HostNode, d0) == 64, "HostNode: the hot fields fill exactly the first cache line");

// What the control simulation needs to know about one node of a voice TEMPLATE (the same for every voice of the
// group): its wrapper stack, innermost first.  A node without WrSmoothParams takes the fast path: parameter changes
// have no effect outside the block they become ready in, so the block-by-block model of the wrapper stack
// collapses to "apply now, or at block_start + running maximum of the queued delays" (precise_timing.rs:65-114).
constexpr int MAX_WRAP_LEVELS = 8;
struct NodeStatic {
    uint8_t kind = 0;            // kgpu_ugen_kind
    uint8_t n_levels = 0;
    bool fast = false;
    bool delay_reaches = false;  // set_delay_within_block_for_param reaches a WrPreciseTiming (only math wrappers above it)
    int8_t precise_level = -1, smooth_level = -1;
    uint32_t base_params = 0, total_params = 0;
    uint32_t capacity = 0;       // of the WrPreciseTiming
    uint32_t nd_size = 0;        // parameters visible at the WrPreciseTiming (its next_delay array)
    uint8_t lv_kind[MAX_WRAP_LEVELS] = {0};
    uint16_t lv_reg[MAX_WRAP_LEVELS] = {0};
    uint32_t lv_inner[MAX_WRAP_LEVELS] = {0};
    uint32_t lv_ar_mask[MAX_WRAP_LEVELS] = {0}; // WrArParams: parameters that have a buffer (audio_rate.rs:70-74)
};

struct TemplateNode {
    uint32_t kind, mode, channels, flags, n_segments;
    std::vector<kgpu_wrapper_desc> wrappers; // value ignored for the signature
    std::vector<std::pair<int, uint32_t>> in;           // per input channel: (local node | -1, channel)
    std::vector<std::tuple<uint32_t, int, uint32_t>> par; // (param, local source node, channel)
    bool same_shape(const TemplateNode &o) const;
};

struct Template {
    std::vector<TemplateNode> nodes;                         // local topological order
    std::vector<std::tuple<int, uint32_t, uint32_t>> outs;   // (local node, channel, target): target < n_outputs = graph output
                                                             // channel, else n_outputs + internal signal (HostPlan::signal_level)
    int level = 0;                                           // 0: reads no internal signal; else 1 + the highest level it reads
    bool same_shape(const Template &o) const;
};
// an input / parameter-route source that is not a node of the same voice: internal signal s is encoded as EXT_BASE - s,
// port k of the template (a graph input only this voice reads, dev.h) as PORT_SRC0 + k
constexpr int EXT_BASE = -2;
constexpr int PORT_SRC0 = -(1 << 30);
constexpr uint32_t MAX_GRAPH_INPUTS = 65536;
constexpr int MAX_SHARED_INPUTS = 16; // graph inputs that are not ports: each takes a signal row
inline bool is_port_src(int src) { return src < PORT_SRC0 / 2; }

struct Group {
    Template tpl;
    DevProgram prog;
    std::vector<std::vector<uint32_t>> voice_nodes; // [voice][local] -> graph node index
    uint32_t n_voices = 0;
    std::vector<uint32_t> init_regs;                // [reg][voice]
    std::vector<HostNode, HugeAllocator<HostNode>> host; // [voice * n_nodes + local]
    std::vector<NodeStatic> nstat;                  // [local]
    std::vector<std::vector<uint16_t>> slot_of;     // [local][channel] -> value slot
    std::vector<uint32_t> port_input;               // [voice * prog.n_ports + port] -> graph input (init_regs holds it too)
    int fused_recipe = -1;                          // index into the fused-kernel table, -1 = interpreter
    std::string kernel_name;
};

struct NodeRef { // 16 bytes
    int32_t group = -1; // -1: mix-bus Add node or unreachable node
    uint32_t voice = 0;
    uint16_t local = 0;
    uint16_t n_params = 0;
    uint32_t rule_base = 0; // first validation rule of this node's parameters in HostPlan::rules
};

struct RawEvent { // 32 bytes
    uint32_t node;
    uint32_t gvoice;        // global voice index (voice_base[group] + voice), resolved once at push time
    uint16_t param;
    uint8_t local;          // node index inside the voice template
    uint8_t kinds;          // value_kind (0 none, 1 float, 2 trigger, 3 integer, 4 bool) | smoothing_kind << 3 (0 none,
                            // 1 ParameterSmoothing::None, 2 Linear) | timed << 5 (0: `time: None`, delay 0 by construction)
    float smooth_seconds;
    double value;
    uint64_t due_frame;     // absolute; events without time: frame clock at push
    uint8_t value_kind() const { return kinds & 7u; }
    uint8_t smoothing_kind() const { return (kinds >> 3) & 3u; }
    bool timed() const { return (kinds >> 5) & 1u; }
};

struct VoiceEvent { // a device event tagged with its destination
    uint32_t voice;
    uint32_t seq;   // arrival order inside the voice
    uint64_t frame; // absolute
    DevEvent ev;
};

struct StreamState;

// A small persistent pool for the host half of a render call (thread creation per call costs more
// than the work of a short call).  start() hands out task indices to the pool threads and returns
// at once; wait() blocks until they are done; run() = start + help + wait.
class WorkPool {
  public:
    explicit WorkPool(unsigned n_threads);
    ~WorkPool();
    unsigned size() const { return n_threads_; }
    void start(unsigned n_tasks, std::function<void(unsigned)> fn);
    void wait();
    void run(unsigned n_tasks, std::function<void(unsigned)> fn);
  private:
    struct Impl;
    Impl *impl_;
    unsigned n_threads_;
};

struct HostPlan {
    uint32_t sample_rate = 48000, block_size = 64, n_outputs = 2;
    uint32_t bs_shift = 6;
    bool bs_pow2 = true;
    uint64_t block_of(uint64_t frame) const { return bs_pow2 ? frame >> bs_shift : frame / block_size; }
    std::vector<Group> groups;
    std::vector<NodeRef> node_ref; // per graph node
    uint32_t n_mix_nodes = 0;
    // Internal signals: what a node reads from OUTSIDE its own voice -- the sum of many voices' outputs (post-mix
    // processing: `mix * 0.5`, a master filter; graph_edit.rs:1145-1225 over graph.rs:850-864) or a source shared by many voices
    // (one LFO into every voice's cutoff).  Each is rendered like a graph output -- its contributors' partial rows are
    // reduced into a buffer [signal][frame] -- one level before the voices that read it.  signal_level[s] = the level of
    // its highest contributor; groups are sorted by level.
    // The graph's own inputs (AudioProcessor::run(&[&[F]]), processor.rs:119-141) are of two sorts.  One that a single voice
    // reads is a port of that voice's template (dev.h): the kernels read it from the caller's input blocks in place.  Every other
    // one -- read by several voices, summed into a mix, wired to an output -- is shared: the first shared_inputs.size() signals,
    // level -1, whose rows are copied from the caller's input blocks before a launch.
    std::vector<int> signal_level;
    int max_level = 0;
    uint32_t n_inputs = 0;
    std::vector<uint32_t> shared_inputs;                        // [signal row] -> graph input
    bool has_ports = false;
    std::vector<std::pair<uint32_t, uint32_t>> input_to_output; // (signal row of a graph input, graph output) wired or summed straight
    uint64_t graph_hash = 0;       // of the whole graph description (snapshots only restore into the same graph)
    uint64_t dropped_changes = 0, ignored_delays = 0, device_events = 0;
    std::vector<RawEvent, DefaultInitAllocator<RawEvent>> pending; // not yet simulated, arrival order
    // Calendar for block-by-block rendering under a large backlog of scheduled events: while it is active
    // `pending` only holds events due before block `far_horizon`, the rest waits in `pending_far` (arrival
    // order too), so that a render call scans what can become ready soon instead of everything queued.
    std::vector<RawEvent, DefaultInitAllocator<RawEvent>> pending_far;
    uint64_t far_horizon = UINT64_MAX; // UINT64_MAX: calendar inactive (everything is in `pending`)
    size_t pending_clean = 0;          // leading events of `pending` already known to be due before far_horizon
    void calendar_update(uint64_t b0, uint64_t b1);

    // caches / scratch of the hot host path (push / compile_events)
    struct Rule { // ok_kinds: bit k set = an event of value_kind k is accepted ('t' any, 'f' float, 'i' integer, 'b' bool): one shift instead of a branch chain per event
        char want; uint8_t smooth_ok, polyblep_wave, svf_type, ok_kinds; };
    std::vector<Rule> rules;                             // flat: NodeRef::rule_base + param
    uint64_t n_active_ramps = 0;
    std::vector<uint64_t> voice_base;                    // prefix sum of voices per group
    std::vector<int32_t> voice_ramps;                    // per global voice: nodes with active ramps / queues
    std::vector<std::vector<VoiceEvent>> later;          // per group: simulated events at/after the last render's end
    std::vector<uint32_t> vcount, vfill, vorder;

    struct CompiledEvents {
        std::vector<DevEvent, DefaultInitAllocator<DevEvent>> events;   // concatenated pieces
        std::vector<uint32_t, DefaultInitAllocator<uint32_t>> offsets;  // concatenated CSR offset arrays (n_voices+1 each)
        std::vector<uint64_t> piece_ev, piece_off; // [launch * n_groups + group]
        std::vector<uint8_t> piece_any;
        // stream_launch only: where the caller wants the launch's events and offsets laid out (page-locked staging memory,
        // so that the merge of the workers' lists is the only copy before the upload).  Used when both fit; `ext_used` says so,
        // `events` / `offsets` stay empty then.
        DevEvent *ext_ev = nullptr;
        uint32_t *ext_off = nullptr;
        size_t ext_ev_cap = 0, ext_off_cap = 0, ext_n_ev = 0, ext_n_off = 0;
        bool ext_used = false;
        size_t n_events() const { return ext_used ? ext_n_ev : events.size(); }
        size_t n_offsets() const { return ext_used ? ext_n_off : offsets.size(); }
        const DevEvent *events_data() const { return ext_used ? ext_ev : events.data(); }
        const uint32_t *offsets_data() const { return ext_used ? ext_off : offsets.data(); }
    };

    void build(const kgpu_graph_desc &d);
    void finish_build();
    // push_events: validate + timestamp (frame_clock = next block to render)
    void push(const kgpu_event *ev, size_t n, uint64_t frame_clock);
    // host half of a render call, see plan.cpp
    void compile_events(const std::vector<uint64_t> &bounds, const std::vector<uint32_t> &chunk_of_group, CompiledEvents &out);
    // the same work as a stream: launch L can be fetched (and rendered) while later launches are
    // still being simulated on the worker threads.  stream_launch fills `out` with ONE launch
    // (pieces indexed by group).  Always pair stream_begin with stream_end.
    void stream_begin(const std::vector<uint64_t> &bounds, const std::vector<uint32_t> &chunk_of_group);
    void stream_launch(size_t launch, CompiledEvents &out);
    void driver_slice_through(size_t launch);
    void stream_end();
    void consume_ready(uint64_t b1);
    // what HostPlan::push learns about a large batch while converting it (see push / stream_begin)
    struct BucketPrep {
        bool valid = false;
        size_t n = 0;
        unsigned T = 0;
        std::vector<std::vector<uint32_t>> hist; // [chunk][global voice]
        std::vector<uint8_t> mono;
        std::vector<uint32_t> first_v, last_v;
        std::vector<uint64_t> first_due, last_due, max_due;
        void reset(unsigned t, size_t n_voices) {
            T = t;
            if (hist.size() < t) hist.resize(t);
            for (unsigned c = 0; c < t; c++) hist[c].assign(n_voices, 0);
            mono.assign(t, 1);
            first_v.assign(t, 0xFFFFFFFFu); last_v.assign(t, 0);
            first_due.assign(t, 0); last_due.assign(t, 0); max_due.assign(t, 0);
        }
    } bucket_prep;
    StreamState *stream = nullptr;       // kept between calls (its buffers are reused); valid while stream_active
    bool stream_active = false;
    WorkPool *pool = nullptr;            // created on first use
    uint32_t pool_threads = 0;           // 0: hardware threads - 1, at most 16
    WorkPool &workers();
    HostPlan() = default;
    HostPlan(const HostPlan &) = delete;
    HostPlan &operator=(const HostPlan &) = delete;
    ~HostPlan();
};

// fused-kernel recipes (kernels.cu): returns recipe index or -1
int match_fused_recipe(const DevProgram &p, uint32_t block_size);
const char *fused_recipe_name(int recipe);

} // namespace kgpu
