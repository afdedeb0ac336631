// capi.cpp -- the C ABI (include/knaster_gpu.h) and the plan runtime: device memory, uploads,
// kernel sequencing.  No torch, no CPU render path: if CUDA is unusable every call fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/knaster_gpu.h"
#include "jit.hpp"
#include "kernels.h"
#include "plan.hpp"

namespace kgpu {
void recompile_group_slots(Group &g, uint32_t sample_rate, const std::vector<std::pair<uint32_t, uint32_t>> &pinned);
}

using namespace kgpu;

namespace {
thread_local std::string g_err;

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) KGPU_THROW(KGPU_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

template <class T> struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) cudaFree(p);
        p = nullptr;
        size_t want = std::max(n, cap + cap / 2);
        cudaError_t e = cudaMalloc((void **)&p, want * sizeof(T));
        if (e != cudaSuccess) {
            p = nullptr;
            cap = 0;
            KGPU_THROW(KGPU_ERR_CUDA, "cudaMalloc(%zu bytes) failed: %s", want * sizeof(T), cudaGetErrorString(e));
        }
        cap = want;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// page-locked host memory (async copies that really are asynchronous to the host)
template <class T> struct PinBuf {
    T *p = nullptr;
    size_t cap = 0;
    void ensure(size_t n) {
        if (n <= cap) return;
        if (p) cudaFreeHost(p);
        p = nullptr;
        size_t want = std::max(n, cap + cap / 2);
        cudaError_t e = cudaHostAlloc((void **)&p, want * sizeof(T), cudaHostAllocDefault);
        if (e != cudaSuccess) {
            p = nullptr;
            cap = 0;
            KGPU_THROW(KGPU_ERR_CUDA, "cudaHostAlloc(%zu bytes) failed: %s", want * sizeof(T), cudaGetErrorString(e));
        }
        cap = want;
    }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
    }
};

// one in-flight upload of a launch's device events (host side of the render pipeline)
struct Staging {
    PinBuf<DevEvent> ev;
    PinBuf<uint32_t> off;
    cudaEvent_t copied = nullptr; // recorded after the H2D copies that read this buffer
    bool in_flight = false;
};

struct GroupDev {
    DevBuf<DevProgram> prog;
    DevBuf<uint32_t> regs;
    DevBuf<DevEvent> events;
    DevBuf<uint32_t> ev_off;
    DevBuf<DevTap> taps;
    std::vector<DevTap> host_taps;
    std::vector<std::pair<uint32_t, uint32_t>> pinned; // (local node, channel) kept live for taps
    uint32_t rows = 0, row0 = 0;
    uint32_t chunk = 1;
    int recipe = -1;   // fused.cu recipes 0..4, RECIPE_JIT, or -1 = the plan interpreter
    JitKernel jit;     // RECIPE_JIT: the kernel generated for this group's voice template (jit.cpp)
};
constexpr int RECIPE_JIT = 5;
} // namespace

struct kgpu_plan {
    HostPlan host;
    int device = 0;
    cudaStream_t stream = nullptr;
    std::vector<GroupDev> gd;
    DevBuf<float> partials;
    DevBuf<uint32_t> row_mask;
    DevBuf<float> out;
    DevBuf<float> sine;
    DevBuf<float> tap_out;
    // internal signals (plan.hpp HostPlan::signal_level): [signal][frames of the launch], reduced level by level
    DevBuf<float> signals;
    DevBuf<uint32_t> in_pairs;              // device: (graph input, graph output) pairs wired without a node in between
    PinBuf<float> in_pinned;                // the caller's input blocks of the current render call
    DevBuf<uint32_t> sig_which;             // device: the signals of level 0, then level 1, ... (sig_level_off indexes it)
    std::vector<uint32_t> sig_level_off;    // [max_level + 2]
    std::vector<uint32_t> level_rows_end;   // [max_level + 1]: partial rows of the groups up to and including that level
    DevBuf<uint8_t> scratch;               // fused_scratch_bytes() of the largest group, reused launch after launch
    uint32_t n_rows = 0, n_taps = 0;
    uint64_t tap_frames = 0;
    uint64_t frame_clock = 0;
    bool rendered = false;
    bool force_interp = false;
    bool force_jit = false;                 // KGPU_PLAN_FORCE_JIT
    std::string jit_note;                   // why the last template that could have been generated was not (diagnostics)
    bool no_scan = false;                   // KGPU_PLAN_NO_SCAN: keep small banks on the bit-exact one-lane-per-voice kernel
    std::vector<float> last_block;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    uint64_t kernel_launches = 0;
    HostPlan::CompiledEvents ce;
    DevBuf<DevEvent> d_events_all;
    DevBuf<uint32_t> d_off_all;
    uint64_t max_blocks_per_launch = 2048;  // measured: 256 -> 15.24 ms, 1024 -> 14.67 ms, 2048 -> 14.49 ms per 10 s step (fixed cost per launch ~ 25 us)
    std::vector<cudaEvent_t> kev;          // per-launch event pairs (profile of the last render call)
    std::vector<uint8_t> kev_class;        // 0 render kernel, 1 reduce_bus
    size_t kev_used = 0;
    bool prepared = false;                 // phase 1 already done for `prepared_blocks`
    uint64_t prepared_blocks = 0;
    uint64_t prepared_bpl = 0;             // launch split the prepared events were compiled for

    uint64_t last_h2d_bytes = 0;
    // pipelined render (kgpu_render without a prior kgpu_plan_prepare): launch L's events are
    // compiled and staged while the device renders launch L-1
    Staging staging[3];
    uint32_t staging_next = 0;
    PinBuf<float> out_pinned;
    // pieces of out_pinned in the order their downloads were enqueued, each with the event recorded behind its copy:
    // kgpu_render hands a piece to the caller's buffer as soon as it has landed, while later launches still render
    struct OutPiece { size_t off, n; };
    std::vector<OutPiece> out_pieces;
    std::vector<cudaEvent_t> out_ev;
    // copies of the streaming path run beside the kernels: events of launch L+1 go up (h2d_stream,
    // device buffers ping-pong) and the bus of launch L-1 comes down (d2h_stream) while launch L renders
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    DevBuf<DevEvent> d_events_pp[2];
    DevBuf<uint32_t> d_off_pp[2];
    cudaEvent_t h2d_done[2] = {nullptr, nullptr}, kern_done[2] = {nullptr, nullptr}, red_done[2] = {nullptr, nullptr};
    bool kern_recorded[2] = {false, false};
    // multi-GPU mix bus over peer memory (kgpu_plan_set_peer_bus): every rank's reduce_bus writes into
    // its slot of a buffer that lives in rank 0's memory, rank 0 folds the slots
    uint32_t peer_rank = 0, peer_world = 0, peer_epoch = 0;
    uint32_t *peer_flags = nullptr, *peer_consumed = nullptr, *peer_timeout = nullptr;
    float *peer_slots = nullptr;
    uint64_t peer_slot_floats = 0;
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t peer_ev[2] = {nullptr, nullptr};
    // the mix-bus reduction of launch L runs on its own stream beside the rendering of launch L+1 (the partial rows
    // ping-pong between two buffers): part_ready[b] = the render kernels have filled buffer b, part_free[b] = its
    // reduction has read it
    cudaStream_t red_stream = nullptr;
    cudaEvent_t part_ready[2] = {nullptr, nullptr}, part_free[2] = {nullptr, nullptr};
};

namespace {

// Frames a node of the interpreter processes per visit: the largest power of two <= 64 that divides the
// block size and whose value slots ([slot][chunk][32 lanes] f32) + registers fit 48 KB of shared memory.
// A long chunk amortises what a node visit costs beside its arithmetic (dispatch, register load / store,
// and above all instruction fetch: every node kind is its own block of code and a scheduler holds ONE warp).
// A template beyond the small-voice limits (dev.h) that gets fewer than 16 frames so goes up to 16 -- the length of the fast
// paths' groups -- wherever the block size allows, in up to the 227 KB a block can opt into: (MAX_REGS + MAX_SLOTS * 16) * 128 B
// fit.  Not more than 16: every kilobyte above 48 costs CTAs per SM, and a CTA is one warp.
uint32_t pick_chunk(uint32_t block_size, const DevProgram &prog) {
    auto fit = [&](uint32_t c, size_t budget) {
        while (c > 1 && (block_size % c || ((size_t)prog.n_regs + (size_t)prog.n_slots * c) * 128 > budget)) c >>= 1;
        return c;
    };
    const bool small = prog.n_nodes <= (uint32_t)SMALL_VOICE_NODES && prog.n_regs <= (uint32_t)SMALL_VOICE_REGS &&
                       prog.n_slots <= (uint32_t)SMALL_VOICE_SLOTS;
    const uint32_t c = fit(64, 48 * 1024);
    return small || c >= 16 ? c : fit(16, 227 * 1024);
}
static_assert(((size_t)MAX_REGS + (size_t)MAX_SLOTS * 16) * 128 <= 227 * 1024, "a template inside the limits gets 16-frame chunks");

void upload_program(kgpu_plan *p, uint32_t gi) {
    Group &g = p->host.groups[gi];
    GroupDev &d = p->gd[gi];
    d.prog.ensure(1);
    CUDA_TRY(cudaMemcpyAsync(d.prog.p, &g.prog, sizeof(DevProgram), cudaMemcpyHostToDevice, p->stream));
}

void layout_rows(kgpu_plan *p) {
    uint32_t row = 0;
    std::vector<uint32_t> mask;
    for (uint32_t gi = 0; gi < p->gd.size(); gi++) {
        Group &g = p->host.groups[gi];
        GroupDev &d = p->gd[gi];
        d.row0 = row;
        uint32_t units = d.recipe >= 0 ? fused_rows(d.recipe, g.n_voices, g.prog.n_ubus) / std::max(1u, g.prog.n_ubus) : (g.n_voices + 31) / 32;
        d.rows = units * g.prog.n_ubus;
        for (uint32_t w = 0; w < units; w++)
            for (uint32_t u = 0; u < g.prog.n_ubus; u++) mask.push_back(g.prog.ubus_mask[u]);
        row += d.rows;
    }
    p->n_rows = row;
    // groups are sorted by level: the rows of the levels <= L are a prefix
    const int max_level = p->host.max_level;
    p->level_rows_end.assign((size_t)max_level + 1, 0);
    for (uint32_t gi = 0; gi < p->gd.size(); gi++) {
        const int lv = p->host.groups[gi].tpl.level;
        for (int l = lv; l <= max_level; l++) p->level_rows_end[l] = std::max(p->level_rows_end[l], p->gd[gi].row0 + p->gd[gi].rows);
    }
    std::vector<uint32_t> which;
    p->sig_level_off.assign((size_t)max_level + 2, 0);
    for (int l = 0; l <= max_level; l++) {
        for (uint32_t sg = 0; sg < p->host.signal_level.size(); sg++)
            if (p->host.signal_level[sg] == l) which.push_back(sg);
        p->sig_level_off[l + 1] = (uint32_t)which.size();
    }
    {
        std::vector<uint32_t> pairs;
        for (auto &io : p->host.input_to_output) { pairs.push_back(io.first); pairs.push_back(io.second); }
        p->in_pairs.ensure(std::max<size_t>(1, pairs.size()));
        if (!pairs.empty()) CUDA_TRY(cudaMemcpyAsync(p->in_pairs.p, pairs.data(), pairs.size() * 4, cudaMemcpyHostToDevice, p->stream));
    }
    p->sig_which.ensure(std::max<size_t>(1, which.size()));
    if (!which.empty()) CUDA_TRY(cudaMemcpyAsync(p->sig_which.p, which.data(), which.size() * 4, cudaMemcpyHostToDevice, p->stream));
    p->row_mask.ensure(std::max<size_t>(1, mask.size()));
    if (!mask.empty()) CUDA_TRY(cudaMemcpyAsync(p->row_mask.p, mask.data(), mask.size() * 4, cudaMemcpyHostToDevice, p->stream));
    CUDA_TRY(cudaStreamSynchronize(p->stream));
}

void choose_kernels(kgpu_plan *p) {
    for (uint32_t gi = 0; gi < p->gd.size(); gi++) {
        Group &g = p->host.groups[gi];
        GroupDev &d = p->gd[gi];
        int recipe = p->force_interp ? -1 : match_fused_recipe(g.prog, p->host.block_size);
        if (recipe == 0 && !p->no_scan && sub_scan_applies(g.n_voices, p->host.block_size)) recipe = 4;
        if (recipe == 2) // the block-table recipe needs every parameter change on a block boundary
            for (const TemplateNode &tn : g.tpl.nodes)
                for (const kgpu_wrapper_desc &w : tn.wrappers)
                    if (w.kind == KGPU_WR_PRECISE_TIMING) recipe = -1;
        // a fused kernel can only tap signals that reach the bus (everything else lives in registers)
        if (recipe >= 0)
            for (auto &pin : d.pinned) {
                bool on_bus = false;
                for (auto &o : g.tpl.outs)
                    if ((uint32_t)std::get<0>(o) == pin.first && std::get<1>(o) == pin.second) on_bus = true;
                if (!on_bus) recipe = -1;
            }
        // no hand-written recipe: a kernel generated for this voice template (register-resident, bit-identical to the
        // interpreter); banks too small to pay for a compilation stay on the interpreter
        jit_unload(d.jit);
        static const bool jit_on = [] { const char *e = getenv("KGPU_JIT"); return !(e && *e == '0'); }();
        static const uint32_t jit_min = [] { const char *e = getenv("KGPU_JIT_MIN_VOICES"); return e ? (uint32_t)atoi(e) : 256u; }();
        if (recipe < 0 && !p->force_interp && jit_on && (g.n_voices >= jit_min || p->force_jit)) {
            std::vector<uint16_t> tapped;
            for (auto &pin : d.pinned) {
                const uint16_t slot = g.slot_of[pin.first][pin.second];
                if (std::find(tapped.begin(), tapped.end(), slot) == tapped.end()) tapped.push_back(slot);
            }
            const std::string src = jit_source(g.prog, tapped);
            std::vector<char> cubin;
            std::string err;
            if (!src.empty() && jit_cubin(src, cubin, err) && jit_load(cubin, d.jit, err)) recipe = RECIPE_JIT;
            else if (!err.empty()) p->jit_note = err;
        }
        d.recipe = recipe;
        d.chunk = recipe >= 0 ? 1 : pick_chunk(p->host.block_size, g.prog);
        g.fused_recipe = recipe;
        g.kernel_name = recipe == RECIPE_JIT ? "render_jit" : recipe >= 0 ? fused_recipe_name(recipe) : "render_interp";
    }
    layout_rows(p);
}

// phase 1 (host): control simulation of the whole range + per-launch device event lists + upload
void prepare_range(kgpu_plan *p, uint64_t n_blocks, uint64_t bpl, cudaStream_t stream) {
    const uint32_t bs = p->host.block_size;
    const uint64_t t_begin = p->frame_clock, t_end = t_begin + n_blocks * bs;
    std::vector<uint64_t> bounds;
    for (uint64_t done = 0; done < n_blocks; done += bpl) bounds.push_back(t_begin + done * bs);
    bounds.push_back(t_end);
    std::vector<uint32_t> chunks;
    for (GroupDev &d : p->gd) chunks.push_back(d.chunk);
    p->host.compile_events(bounds, chunks, p->ce);
    p->last_h2d_bytes = 0;
    if (!p->ce.events.empty()) {
        p->d_events_all.ensure(p->ce.events.size());
        p->d_off_all.ensure(p->ce.offsets.size());
        // pageable source: the runtime stages the copy before returning, the vectors may be reused
        CUDA_TRY(cudaMemcpyAsync(p->d_events_all.p, p->ce.events.data(), p->ce.events.size() * sizeof(DevEvent), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(p->d_off_all.p, p->ce.offsets.data(), p->ce.offsets.size() * 4, cudaMemcpyHostToDevice, stream));
        p->last_h2d_bytes = p->ce.events.size() * sizeof(DevEvent) + p->ce.offsets.size() * 4;
    }
}

uint64_t blocks_per_launch(kgpu_plan *p) {
    // bound the partial-sum buffer (rows x frames x 4 B) to ~256 MiB
    uint64_t max_frames = (256ull << 20) / (4ull * std::max(1u, p->n_rows));
    uint64_t bpl = std::max<uint64_t>(1, max_frames / p->host.block_size);
    return std::min<uint64_t>(bpl, p->max_blocks_per_launch);
}

void ensure_stream_objects(kgpu_plan *p) {
    if (p->h2d_stream) return;
    CUDA_TRY(cudaStreamCreateWithFlags(&p->h2d_stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&p->d2h_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        CUDA_TRY(cudaEventCreateWithFlags(&p->h2d_done[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&p->kern_done[i], cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&p->red_done[i], cudaEventDisableTiming));
    }
}

// Uploads the events of ONE launch (the only launch in p->ce): pinned staging buffer -> device
// buffer (launch & 1) on h2d_stream, which first waits until the kernels of launch - 2 (the last
// readers of that buffer) are done.  `stream` then waits for the copy.
// The staging buffer the next launch's events go through: stream_launch lays them out in it directly when they fit
// (HostPlan::CompiledEvents::ext_*), so the merge of the workers' lists is the only host copy before the upload.
void offer_staging(kgpu_plan *p) {
    Staging &sg = p->staging[p->staging_next];
    if (sg.in_flight && sg.copied) {
        CUDA_TRY(cudaEventSynchronize(sg.copied));
        sg.in_flight = false;
    }
    p->ce.ext_ev = sg.ev.p;
    p->ce.ext_ev_cap = sg.ev.cap;
    p->ce.ext_off = sg.off.p;
    p->ce.ext_off_cap = sg.off.cap;
}
void upload_launch_events(kgpu_plan *p, size_t launch, cudaStream_t stream) {
    const size_t n_ev = p->ce.n_events(), n_off = p->ce.n_offsets();
    if (!n_ev) return;
    const int pp = (int)(launch & 1);
    Staging &sg = p->staging[p->staging_next];
    p->staging_next = (p->staging_next + 1) % 3;
    if (!sg.copied) CUDA_TRY(cudaEventCreateWithFlags(&sg.copied, cudaEventDisableTiming));
    if (!p->ce.ext_used) {
        if (sg.in_flight) CUDA_TRY(cudaEventSynchronize(sg.copied));
        if (n_ev > sg.ev.cap || n_off > sg.off.cap) {
            // grow all three staging buffers together (with headroom): page-locked allocation is slow
            // and synchronises, so it should happen in the first render call only
            for (Staging &o : p->staging) {
                if (o.in_flight && o.copied) CUDA_TRY(cudaEventSynchronize(o.copied));
                o.in_flight = false;
                o.ev.ensure(n_ev + n_ev / 2);
                o.off.ensure(n_off + n_off / 2);
            }
        }
        std::memcpy(sg.ev.p, p->ce.events.data(), n_ev * sizeof(DevEvent));
        std::memcpy(sg.off.p, p->ce.offsets.data(), n_off * 4);
    }
    if (n_ev > p->d_events_pp[pp].cap || n_off > p->d_off_pp[pp].cap) {
        CUDA_TRY(cudaStreamSynchronize(stream)); // cudaFree of a buffer a queued kernel still reads: first render call only
        for (int i = 0; i < 2; i++) {
            p->d_events_pp[i].ensure(n_ev + n_ev / 2);
            p->d_off_pp[i].ensure(n_off + n_off / 2);
        }
    }
    if (p->kern_recorded[pp]) CUDA_TRY(cudaStreamWaitEvent(p->h2d_stream, p->kern_done[pp], 0));
    CUDA_TRY(cudaMemcpyAsync(p->d_events_pp[pp].p, sg.ev.p, n_ev * sizeof(DevEvent), cudaMemcpyHostToDevice, p->h2d_stream));
    CUDA_TRY(cudaMemcpyAsync(p->d_off_pp[pp].p, sg.off.p, n_off * 4, cudaMemcpyHostToDevice, p->h2d_stream));
    CUDA_TRY(cudaEventRecord(sg.copied, p->h2d_stream));
    CUDA_TRY(cudaEventRecord(p->h2d_done[pp], p->h2d_stream));
    CUDA_TRY(cudaStreamWaitEvent(stream, p->h2d_done[pp], 0));
    sg.in_flight = true;
    p->last_h2d_bytes += n_ev * sizeof(DevEvent) + n_off * 4;
}

// Renders n_blocks blocks into device_out.  If the range was prepared (kgpu_plan_prepare) the
// device events are already resident and the launches go back to back; otherwise the host half
// runs launch by launch, one launch ahead of the device: while launch L renders, the control
// simulation of launch L+1 runs on the host threads and its events are staged in pinned memory.
// pinned_out: optional page-locked mirror of device_out, filled launch by launch.
void render_range(kgpu_plan *p, uint64_t n_blocks, float *device_out, cudaStream_t stream, float *pinned_out = nullptr,
                  const float *host_in = nullptr) {
    const uint32_t bs = p->host.block_size, n_out = p->host.n_outputs;
    p->rendered = true;
    const uint64_t total_frames = n_blocks * bs;
    if (p->n_taps) {
        p->tap_out.ensure((size_t)p->n_taps * total_frames);
        p->tap_frames = total_frames;
    }
    // kgpu_plan_prepare(N) has already consumed the queued events and advanced every ramp / queue by N blocks: the
    // only valid continuation is the render of exactly those N blocks, with the launch split they were compiled for
    if (p->prepared && p->prepared_blocks != n_blocks)
        KGPU_THROW(KGPU_ERR_STATE, "kgpu_plan_prepare(%llu) must be followed by a render of %llu blocks, not %llu",
                   (unsigned long long)p->prepared_blocks, (unsigned long long)p->prepared_blocks, (unsigned long long)n_blocks);
    const bool was_prepared = p->prepared;
    const uint64_t bpl = was_prepared ? p->prepared_bpl : blocks_per_launch(p);
    p->prepared = false;
    if (!was_prepared) p->last_h2d_bytes = 0;
    // Streaming path with more than one launch: launch L's mix-bus reduction runs beside launch L+1's rendering, on two
    // partial-row buffers (device span of a 10 s step 14.48 -> 14.20 ms).  Prepared renders keep the kernels back to back on
    // one stream -- their launches are few and large, and the concurrent reduction costs the render kernel 1.2 % for 0.8 % of
    // the step (measured; KGPU_REDUCE_OVERLAP=1 / 0 forces either).
    static const char *ov_env = getenv("KGPU_REDUCE_OVERLAP");
    const bool overlap = n_blocks > bpl && (ov_env ? *ov_env == '1' : !was_prepared);
    const size_t part_stride = (size_t)std::max(1u, p->n_rows) * std::min<uint64_t>(bpl, n_blocks) * bs;
    p->partials.ensure(part_stride * (overlap ? 2 : 1));
    if (overlap && !p->red_stream) {
        CUDA_TRY(cudaStreamCreateWithFlags(&p->red_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CUDA_TRY(cudaEventCreateWithFlags(&p->part_ready[i], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&p->part_free[i], cudaEventDisableTiming));
        }
    }
    cudaStream_t rs = overlap ? p->red_stream : stream; // the stream the reduction (and what follows it) runs on
    const uint64_t t_begin = p->frame_clock, t_end = t_begin + total_frames;
    std::vector<uint32_t> chunks;
    for (GroupDev &d : p->gd) chunks.push_back(d.chunk);

    const bool peer = p->peer_world > 1;
    const uint32_t n_signals = (uint32_t)p->host.signal_level.size();
    const uint32_t n_in = p->host.n_inputs;
    if (n_in && !host_in) KGPU_THROW(KGPU_ERR_STATE, "this graph has %u inputs: render it with kgpu_render_inputs (AudioProcessor::run), not run_without_inputs", n_in);
    if (n_in) { // the input blocks, page-locked for the strided copies below
        p->in_pinned.ensure((size_t)n_blocks * n_in * bs);
        std::memcpy(p->in_pinned.p, host_in, (size_t)n_blocks * n_in * bs * 4);
    }
    if (n_signals) {
        if (peer) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "a plan with internal signals (post-mix nodes, sources shared between voices) cannot be sharded over a peer bus");
        p->signals.ensure((size_t)n_signals * std::min<uint64_t>(bpl, n_blocks) * bs);
    }
    if (peer) {
        if ((uint64_t)total_frames * n_out > p->peer_slot_floats)
            KGPU_THROW(KGPU_ERR_INVALID, "peer bus holds %llu floats per rank, this render needs %llu", (unsigned long long)p->peer_slot_floats,
                       (unsigned long long)(total_frames * n_out));
        if (!p->aux_stream) {
            CUDA_TRY(cudaStreamCreateWithFlags(&p->aux_stream, cudaStreamNonBlocking));
            for (auto &e : p->peer_ev) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        p->peer_epoch++;
        // a slot may be overwritten only after rank 0 has folded the previous call's data
        if (p->peer_epoch > 1) CUDA_TRY(launch_wait_flag(p->peer_consumed, p->peer_epoch - 1, p->peer_timeout, stream));
    }
    if (p->timed) CUDA_TRY(cudaEventRecord(p->ev0, stream));
    size_t piece = 0;
    p->out_pieces.clear();
    auto piece_landed = [&](size_t off, size_t n, cudaStream_t s) { // call right after the D2H copy of out_pinned[off, off + n) was enqueued on s
        if (p->out_pieces.size() == p->out_ev.size()) {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            p->out_ev.push_back(e);
        }
        CUDA_TRY(cudaEventRecord(p->out_ev[p->out_pieces.size()], s));
        p->out_pieces.push_back({off, n});
    };
    p->kev_used = 0;
    p->kev_class.clear();
    auto mark = [&](int cls, bool begin, cudaStream_t on = nullptr) {
        if (p->kev_used == p->kev.size()) {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreate(&e));
            p->kev.push_back(e);
        }
        CUDA_TRY(cudaEventRecord(p->kev[p->kev_used++], on ? on : stream));
        if (begin) p->kev_class.push_back((uint8_t)cls);
    };
    struct StreamGuard { // stream_begin is always paired with stream_end, also when a launch throws
        HostPlan *h = nullptr;
        ~StreamGuard() {
            if (h) try { h->stream_end(); } catch (...) {}
        }
    } guard;
    // launch sizes in blocks.  Prepared: bpl each.  Streaming: a short geometric ramp first, so the
    // device starts as soon as the host has simulated 1/8 of a full launch and is not starved afterwards.
    // Measured on the bench configuration (16384 voices, 15 workers): the host needs ~0.45 ms per launch
    // plus ~0.6 us per block, the device 2 us per block -- from 256 blocks on a launch is simulated faster
    // than its predecessor renders, below that the device waits for the host (ramp from 128: 1.7 ms idle).
    std::vector<uint64_t> sizes;
    {
        // (the ramp starts at bpl / 64: the device is busy ~0.1 ms after the host has its first 32 blocks, and a launch costs ~25 us)
        uint64_t left = n_blocks, next = was_prepared || bpl < 64 || n_blocks < 2 * bpl ? bpl : std::max<uint64_t>(32, bpl / 64);
        while (left) {
            const uint64_t nb = std::min(next, left);
            sizes.push_back(nb);
            left -= nb;
            next = std::min(bpl, next + next / 2); // x1.5: the host stays ahead of the device with a 1.6x margin (3 workers per GPU)
        }
    }
    if (peer && sizes.size() > KGPU_PEER_MAX_LAUNCHES)
        KGPU_THROW(KGPU_ERR_INVALID, "a render call with a peer bus is limited to %d launches", KGPU_PEER_MAX_LAUNCHES);
    if (!was_prepared) {
        ensure_stream_objects(p);
        std::vector<uint64_t> bounds{t_begin};
        for (uint64_t nb : sizes) bounds.push_back(bounds.back() + nb * bs);
        p->host.stream_begin(bounds, chunks);
        guard.h = &p->host;
    }
    uint64_t done = 0;
    for (size_t launch = 0; launch < sizes.size(); done += sizes[launch], launch++) {
        const uint64_t nb = sizes[launch];
        const uint32_t nf = (uint32_t)(nb * bs);
        const int pb = overlap ? (int)(launch & 1) : 0;
        float *part = p->partials.p + (size_t)pb * part_stride;
        if (overlap && launch >= 2) CUDA_TRY(cudaStreamWaitEvent(stream, p->part_free[pb], 0)); // launch - 2's reduction has read this buffer
        if (!was_prepared) {
            static const bool timing = getenv("KGPU_TIMING") != nullptr;
            const auto ta = std::chrono::steady_clock::now();
            offer_staging(p);
            p->host.stream_launch(launch, p->ce);
            const auto tb = std::chrono::steady_clock::now();
            upload_launch_events(p, launch, stream);
            if (timing && n_blocks > 100)
                fprintf(stderr, "[kgpu timing]   launch %zu: wait+merge %.2f ms, stage+enqueue %.2f ms\n", launch,
                        std::chrono::duration<double, std::milli>(tb - ta).count(),
                        std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb).count());
            piece = 0;
        }
        // graph inputs: [block][input][frame] from the caller -> rows [0, n_inputs) of the signal buffer, [input][frame of the launch]
        for (uint32_t c = 0; c < n_in; c++)
            CUDA_TRY(cudaMemcpy2DAsync(p->signals.p + (size_t)c * nf, (size_t)bs * 4, p->in_pinned.p + ((size_t)done * n_in + c) * bs, (size_t)n_in * bs * 4,
                                       (size_t)bs * 4, (size_t)nb, cudaMemcpyHostToDevice, stream));
        for (uint32_t gi = 0; gi < p->gd.size(); gi++, piece++) {
            Group &g = p->host.groups[gi];
            GroupDev &d = p->gd[gi];
            // a level's groups are done: the signals they complete are reduced before the next level's voices read them
            if (n_signals && gi > 0 && g.tpl.level != p->host.groups[gi - 1].tpl.level) {
                const int lv = p->host.groups[gi - 1].tpl.level;
                const uint32_t w0 = p->sig_level_off[lv], w1 = p->sig_level_off[lv + 1];
                if (w1 > w0) {
                    mark(1, true);
                    CUDA_TRY(launch_reduce_signals(part, p->row_mask.p, p->level_rows_end[lv], nf, p->signals.p, n_out, p->sig_which.p + w0, w1 - w0, stream));
                    mark(1, false);
                    p->kernel_launches++;
                }
            }
            const bool any = !p->ce.piece_any.empty() && p->ce.piece_any[piece];
            const DevEvent *ev_base = was_prepared ? p->d_events_all.p : p->d_events_pp[launch & 1].p;
            const uint32_t *off_base = was_prepared ? p->d_off_all.p : p->d_off_pp[launch & 1].p;
            const DevEvent *d_ev = any ? ev_base + p->ce.piece_ev[piece] : nullptr;
            const uint32_t *d_off = any ? off_base + p->ce.piece_off[piece] : nullptr;
            mark(0, true);
            if (d.recipe >= 0) {
                FusedArgs a{};
                a.prog = d.prog.p; a.regs = d.regs.p; a.n_voices = g.n_voices; a.events = d_ev; a.ev_off = d_off;
                a.n_frames = nf; a.partials = part; a.row0 = d.row0;
                a.taps = d.taps.p; a.n_taps = (uint32_t)d.host_taps.size(); a.tap_out = p->tap_out.p;
                a.tap_stride = total_frames; a.tap_frame0 = done * bs; a.sine_table = p->sine.p;
                a.host_prog = &g.prog; a.block_size = bs;
                a.ext = n_signals ? p->signals.p : nullptr; a.ext_stride = nf;
                const size_t sb = fused_scratch_bytes(d.recipe, g.n_voices, nf, bs);
                if (sb > p->scratch.cap) {
                    CUDA_TRY(cudaStreamSynchronize(stream)); // a queued launch may still use the old buffer
                    p->scratch.ensure(sb);
                }
                a.scratch = p->scratch.p;
                if (d.recipe == RECIPE_JIT) {
                    void *args[] = {&a};
                    CUDA_TRY(cudaLaunchKernel((const void *)d.jit.kernel, dim3((g.n_voices + 31) / 32), dim3(32), args, 0, stream));
                } else CUDA_TRY(launch_fused(d.recipe, a, stream));
            } else {
                InterpArgs a{};
                a.prog = d.prog.p; a.regs = d.regs.p; a.n_voices = g.n_voices; a.events = d_ev; a.ev_off = d_off;
                a.n_frames = nf; a.chunk = d.chunk; a.partials = part; a.row0 = d.row0;
                a.taps = d.taps.p; a.n_taps = (uint32_t)d.host_taps.size(); a.tap_out = p->tap_out.p;
                a.tap_stride = total_frames; a.tap_frame0 = done * bs; a.sine_table = p->sine.p;
                a.ext = n_signals ? p->signals.p : nullptr; a.ext_stride = nf;
                CUDA_TRY(launch_interp(a, g.prog.n_regs, g.prog.n_slots, stream));
            }
            mark(0, false);
            p->kernel_launches++;
        }
        if (!was_prepared) {
            CUDA_TRY(cudaEventRecord(p->kern_done[launch & 1], stream));
            p->kern_recorded[launch & 1] = true;
        }
        if (overlap) {
            CUDA_TRY(cudaEventRecord(p->part_ready[pb], stream));
            CUDA_TRY(cudaStreamWaitEvent(rs, p->part_ready[pb], 0));
        }
        mark(1, true, rs);
        float *dst = device_out + (size_t)done * n_out * bs;
        if (peer) { // reduce straight into this rank's slot in rank 0's memory (NVLink stores), then publish the launch
            float *slot = p->peer_slots + (size_t)p->peer_rank * p->peer_slot_floats + (size_t)done * n_out * bs;
            CUDA_TRY(launch_reduce_bus(part, p->row_mask.p, p->n_rows, nf, slot, n_out, bs, rs));
            CUDA_TRY(launch_signal_flag(p->peer_flags + (size_t)p->peer_rank * KGPU_PEER_MAX_LAUNCHES + launch, p->peer_epoch, rs));
            p->kernel_launches++;
        } else {
            CUDA_TRY(launch_reduce_bus(part, p->row_mask.p, p->n_rows, nf, dst, n_out, bs, rs));
            if (!p->host.input_to_output.empty()) {
                CUDA_TRY(launch_add_inputs(p->signals.p, nf, dst, n_out, bs, p->in_pairs.p, (uint32_t)p->host.input_to_output.size(), rs));
                p->kernel_launches++;
            }
        }
        mark(1, false, rs);
        if (overlap) CUDA_TRY(cudaEventRecord(p->part_free[pb], rs));
        p->kernel_launches++;
        if (peer) {
            if (p->peer_rank == 0) { // fold the slots beside the next launch's rendering
                CUDA_TRY(cudaEventRecord(p->peer_ev[launch & 1], rs));
                CUDA_TRY(cudaStreamWaitEvent(p->aux_stream, p->peer_ev[launch & 1], 0));
                CUDA_TRY(launch_sum_slots(p->peer_slots + (size_t)done * n_out * bs, p->peer_slot_floats, p->peer_world, p->peer_flags + launch,
                                          KGPU_PEER_MAX_LAUNCHES, p->peer_epoch, dst, (size_t)nf * n_out, p->peer_timeout, p->aux_stream));
                p->kernel_launches++;
                if (pinned_out) {
                    CUDA_TRY(cudaMemcpyAsync(pinned_out + (size_t)done * n_out * bs, dst, (size_t)nf * n_out * 4, cudaMemcpyDeviceToHost, p->aux_stream));
                    piece_landed((size_t)done * n_out * bs, (size_t)nf * n_out, p->aux_stream);
                }
            }
        } else if (pinned_out) {
            // the bus of a launch comes down behind its reduction: on the reduction's own stream when that runs beside the
            // rendering, else (one launch per call) on the copy stream of the streaming path
            cudaStream_t cs = overlap || was_prepared ? rs : p->d2h_stream;
            if (cs != rs) {
                CUDA_TRY(cudaEventRecord(p->red_done[launch & 1], rs));
                CUDA_TRY(cudaStreamWaitEvent(cs, p->red_done[launch & 1], 0));
            }
            CUDA_TRY(cudaMemcpyAsync(pinned_out + (size_t)done * n_out * bs, dst, (size_t)nf * n_out * 4, cudaMemcpyDeviceToHost, cs));
            piece_landed((size_t)done * n_out * bs, (size_t)nf * n_out, cs);
            if (cs != rs && launch + 1 == sizes.size()) { // `stream` ends after the last download
                CUDA_TRY(cudaEventRecord(p->red_done[0], cs));
                CUDA_TRY(cudaStreamWaitEvent(stream, p->red_done[0], 0));
            }
        }
    }
    if (peer) {
        if (p->peer_rank == 0) { // tell the ranks their slots are free again; `stream` ends after the last fold
            CUDA_TRY(launch_signal_flag(p->peer_consumed, p->peer_epoch, p->aux_stream));
            CUDA_TRY(cudaEventRecord(p->peer_ev[0], p->aux_stream));
            CUDA_TRY(cudaStreamWaitEvent(stream, p->peer_ev[0], 0));
        }
    }
    if (overlap) { // `stream` ends after the last reduction (and its download)
        CUDA_TRY(cudaEventRecord(p->part_ready[0], rs));
        CUDA_TRY(cudaStreamWaitEvent(stream, p->part_ready[0], 0));
    }
    if (guard.h) {
        guard.h = nullptr;
        p->host.stream_end();
    }
    p->frame_clock = t_end;
    if (p->timed) CUDA_TRY(cudaEventRecord(p->ev1, stream));
}

} // namespace

extern "C" {

const char *kgpu_last_error(void) { return g_err.c_str(); }
uint32_t kgpu_abi_version(void) { return KGPU_ABI_VERSION; }
int kgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int kgpu_plan_create(const kgpu_graph_desc *desc, kgpu_plan **out) {
    if (!desc || !out) return fail(KGPU_ERR_INVALID, "kgpu_plan_create: NULL argument");
    *out = nullptr;
    kgpu_plan *p = nullptr;
    try {
        p = new kgpu_plan();
        p->host.build(*desc);
        p->force_interp = (desc->flags & KGPU_PLAN_FORCE_INTERPRETER) != 0;
        p->no_scan = (desc->flags & KGPU_PLAN_NO_SCAN) != 0;
        p->force_jit = (desc->flags & KGPU_PLAN_FORCE_JIT) != 0;
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
            cudaGetLastError();
            KGPU_THROW(KGPU_ERR_CUDA, "no usable CUDA device: the engine has no CPU fallback");
        }
        if (desc->device >= 0) {
            if (desc->device >= ndev) KGPU_THROW(KGPU_ERR_CUDA, "device %d out of range (%d devices)", desc->device, ndev);
            CUDA_TRY(cudaSetDevice(desc->device));
            p->device = desc->device;
        } else CUDA_TRY(cudaGetDevice(&p->device));
        CUDA_TRY(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreate(&p->ev0));
        CUDA_TRY(cudaEventCreate(&p->ev1));
        // shared sine table: NonAaWavetable::sine(), wavetable.rs:130-139 (f64 sin, rounded to f32)
        {
            std::vector<float> tab(SINE_TABLE_SIZE);
            for (int i = 0; i < SINE_TABLE_SIZE; i++) tab[i] = (float)std::sin(((double)i / (double)SINE_TABLE_SIZE) * M_PI * 2.0);
            p->sine.ensure(SINE_TABLE_SIZE);
            CUDA_TRY(cudaMemcpy(p->sine.p, tab.data(), SINE_TABLE_SIZE * 4, cudaMemcpyHostToDevice));
        }
        p->gd.resize(p->host.groups.size());
        for (uint32_t gi = 0; gi < p->gd.size(); gi++) {
            Group &g = p->host.groups[gi];
            GroupDev &d = p->gd[gi];
            upload_program(p, gi);
            d.regs.ensure(std::max<size_t>(1, g.init_regs.size()));
            if (!g.init_regs.empty())
                CUDA_TRY(cudaMemcpyAsync(d.regs.p, g.init_regs.data(), g.init_regs.size() * 4, cudaMemcpyHostToDevice, p->stream));
        }
        choose_kernels(p);
        p->last_block.assign((size_t)p->host.block_size * p->host.n_outputs, 0.f);
        CUDA_TRY(cudaStreamSynchronize(p->stream));
        *out = p;
        return KGPU_OK;
    } catch (const Error &e) {
        if (p) kgpu_plan_destroy(p);
        return fail(e.code, e.msg);
    } catch (const std::exception &e) {
        if (p) kgpu_plan_destroy(p);
        return fail(KGPU_ERR_INVALID, std::string("kgpu_plan_create: ") + e.what());
    }
}

void kgpu_plan_destroy(kgpu_plan *p) {
    if (!p) return;
    if (p->stream) cudaStreamSynchronize(p->stream);
    for (GroupDev &d : p->gd) {
        d.prog.release(); d.regs.release(); d.events.release(); d.ev_off.release(); d.taps.release();
        jit_unload(d.jit);
    }
    p->d_events_all.release(); p->d_off_all.release();
    for (Staging &sg : p->staging) {
        sg.ev.release(); sg.off.release();
        if (sg.copied) cudaEventDestroy(sg.copied);
    }
    p->out_pinned.release();
    for (int i = 0; i < 2; i++) {
        p->d_events_pp[i].release(); p->d_off_pp[i].release();
        if (p->h2d_done[i]) cudaEventDestroy(p->h2d_done[i]);
        if (p->kern_done[i]) cudaEventDestroy(p->kern_done[i]);
        if (p->red_done[i]) cudaEventDestroy(p->red_done[i]);
    }
    if (p->aux_stream) cudaStreamDestroy(p->aux_stream);
    if (p->red_stream) cudaStreamDestroy(p->red_stream);
    for (int i = 0; i < 2; i++) {
        if (p->part_ready[i]) cudaEventDestroy(p->part_ready[i]);
        if (p->part_free[i]) cudaEventDestroy(p->part_free[i]);
    }
    for (cudaEvent_t e : p->peer_ev)
        if (e) cudaEventDestroy(e);
    if (p->h2d_stream) cudaStreamDestroy(p->h2d_stream);
    if (p->d2h_stream) cudaStreamDestroy(p->d2h_stream);
    p->scratch.release(); p->signals.release(); p->sig_which.release(); p->in_pairs.release(); p->in_pinned.release();
    p->partials.release(); p->row_mask.release(); p->out.release(); p->sine.release(); p->tap_out.release();
    for (cudaEvent_t e : p->kev) cudaEventDestroy(e);
    for (cudaEvent_t e : p->out_ev) cudaEventDestroy(e);
    if (p->ev0) cudaEventDestroy(p->ev0);
    if (p->ev1) cudaEventDestroy(p->ev1);
    if (p->stream) cudaStreamDestroy(p->stream);
    delete p;
}

int kgpu_plan_push_events(kgpu_plan *p, const kgpu_event *events, size_t n) {
    if (!p || (n && !events)) return fail(KGPU_ERR_INVALID, "kgpu_plan_push_events: NULL argument");
    if (p->prepared) return fail(KGPU_ERR_STATE, "kgpu_plan_push_events: a prepared render is pending (its range is already simulated)");
    try {
        p->host.push(events, n, p->frame_clock);
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

int kgpu_render_device(kgpu_plan *p, uint64_t n_blocks, float *device_out, void *cuda_stream) {
    if (!p || !device_out) return fail(KGPU_ERR_INVALID, "kgpu_render_device: NULL argument");
    if (n_blocks == 0) return KGPU_OK;
    try {
        CUDA_TRY(cudaSetDevice(p->device));
        p->timed = true;
        render_range(p, n_blocks, device_out, cuda_stream ? (cudaStream_t)cuda_stream : p->stream);
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

static int render_host(kgpu_plan *p, uint64_t n_blocks, const float *host_in, float *host_out);
int kgpu_render(kgpu_plan *p, uint64_t n_blocks, float *host_out) { return render_host(p, n_blocks, nullptr, host_out); }
int kgpu_render_inputs(kgpu_plan *p, uint64_t n_blocks, const float *host_in, float *host_out) {
    if (p && p->host.n_inputs && !host_in) return fail(KGPU_ERR_INVALID, "kgpu_render_inputs: NULL input buffer");
    return render_host(p, n_blocks, host_in, host_out);
}
static int render_host(kgpu_plan *p, uint64_t n_blocks, const float *host_in, float *host_out) {
    if (!p) return fail(KGPU_ERR_INVALID, "kgpu_render: NULL plan");
    if (n_blocks == 0) return KGPU_OK;
    try {
        CUDA_TRY(cudaSetDevice(p->device));
        const size_t per_block = (size_t)p->host.block_size * p->host.n_outputs;
        p->out.ensure(per_block * n_blocks);
        p->timed = true;
        if (host_out) {
            static const bool timing = getenv("KGPU_TIMING") != nullptr;
            auto now = [] { return std::chrono::steady_clock::now(); };
            auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            const auto t0 = now();
            p->out_pinned.ensure(per_block * n_blocks);
            render_range(p, n_blocks, p->out.p, p->stream, p->out_pinned.p, host_in);
            const auto t1 = now();
            // hand the audio over piece by piece, each as soon as its download has landed (the rest still renders)
            for (size_t i = 0; i < p->out_pieces.size(); i++) {
                CUDA_TRY(cudaEventSynchronize(p->out_ev[i]));
                std::memcpy(host_out + p->out_pieces[i].off, p->out_pinned.p + p->out_pieces[i].off, p->out_pieces[i].n * 4);
            }
            CUDA_TRY(cudaStreamSynchronize(p->stream));
            const auto t2 = now();
            // with a peer bus only rank 0 receives audio (the sum over all ranks): the other ranks' host buffers and
            // kgpu_output_block stay untouched, as the header says
            if (!(p->peer_world > 1 && p->peer_rank != 0)) {
                std::memcpy(p->last_block.data(), host_out + per_block * (n_blocks - 1), per_block * 4);
            }
            if (timing && n_blocks > 100) {
                float span = 0.f, kern = 0.f, red = 0.f;
                cudaEventElapsedTime(&span, p->ev0, p->ev1);
                for (size_t i = 0; i < p->kev_class.size(); i++) {
                    float m = 0.f;
                    cudaEventElapsedTime(&m, p->kev[2 * i], p->kev[2 * i + 1]);
                    (p->kev_class[i] == 0 ? kern : red) += m;
                }
                fprintf(stderr, "[kgpu timing] kgpu_render: device span %.2f ms (render kernels %.2f, reduce_bus %.2f, rest = copies + gaps)\n", span, kern, red);
            }
            if (timing && n_blocks > 100)
                fprintf(stderr, "[kgpu timing] kgpu_render: host loop %.1f ms, device tail %.1f ms, copy out %.1f ms\n", ms(t0, t1), ms(t1, t2), ms(t2, now()));
        } else {
            render_range(p, n_blocks, p->out.p, p->stream, nullptr, host_in);
            if (!(p->peer_world > 1 && p->peer_rank != 0))
                CUDA_TRY(cudaMemcpyAsync(p->last_block.data(), p->out.p + per_block * (n_blocks - 1), per_block * 4, cudaMemcpyDeviceToHost, p->stream));
            CUDA_TRY(cudaStreamSynchronize(p->stream));
        }
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

int kgpu_render_block(kgpu_plan *p) { return kgpu_render(p, 1, nullptr); }
const float *kgpu_output_block(kgpu_plan *p) { return p ? p->last_block.data() : nullptr; }

int kgpu_plan_synchronize(kgpu_plan *p) {
    if (!p) return fail(KGPU_ERR_INVALID, "NULL plan");
    cudaError_t e = cudaStreamSynchronize(p->stream);
    if (e != cudaSuccess) return fail(KGPU_ERR_CUDA, cudaGetErrorString(e));
    return KGPU_OK;
}

uint32_t kgpu_plan_block_size(const kgpu_plan *p) { return p ? p->host.block_size : 0; }
uint32_t kgpu_plan_outputs(const kgpu_plan *p) { return p ? p->host.n_outputs : 0; }
uint64_t kgpu_plan_frame_clock(const kgpu_plan *p) { return p ? p->frame_clock : 0; }

int kgpu_plan_add_tap(kgpu_plan *p, uint32_t node, uint32_t channel) {
    if (!p) return fail(KGPU_ERR_INVALID, "NULL plan");
    if (p->rendered || p->prepared) return fail(KGPU_ERR_STATE, "kgpu_plan_add_tap must be called before the first render / prepare");
    try {
        if (node >= p->host.node_ref.size()) KGPU_THROW(KGPU_ERR_INVALID, "tap: NodeNotFound (%u)", node);
        const NodeRef &nr = p->host.node_ref[node];
        if (nr.group < 0) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "tap: node %u is a mix-bus Add or is not connected to an output", node);
        Group &g = p->host.groups[nr.group];
        GroupDev &d = p->gd[nr.group];
        if (channel >= g.prog.nodes[nr.local].n_out) KGPU_THROW(KGPU_ERR_INVALID, "tap: OutputOutOfBounds(%u)", channel);
        CUDA_TRY(cudaSetDevice(p->device));
        d.pinned.push_back({nr.local, channel});
        recompile_group_slots(g, p->host.sample_rate, d.pinned); // keep tapped values live
        upload_program(p, (uint32_t)nr.group);
        const uint32_t tap = p->n_taps++;
        d.host_taps.push_back(DevTap{nr.voice, 0, tap, 0});
        // slots may have moved: refresh every tap of the group
        for (size_t i = 0; i < d.host_taps.size(); i++) d.host_taps[i].slot = g.slot_of[d.pinned[i].first][d.pinned[i].second];
        d.taps.ensure(d.host_taps.size());
        CUDA_TRY(cudaMemcpyAsync(d.taps.p, d.host_taps.data(), d.host_taps.size() * sizeof(DevTap), cudaMemcpyHostToDevice, p->stream));
        choose_kernels(p);
        return (int)tap;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

int kgpu_plan_read_taps(kgpu_plan *p, float *out, uint64_t n_frames) {
    if (!p || !out) return fail(KGPU_ERR_INVALID, "NULL argument");
    if (n_frames != p->tap_frames || !p->n_taps) return fail(KGPU_ERR_STATE, "kgpu_plan_read_taps: n_frames must equal the frames of the last render");
    cudaError_t e = cudaStreamSynchronize(p->stream);
    if (e == cudaSuccess) e = cudaMemcpy(out, p->tap_out.p, (size_t)p->n_taps * n_frames * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(KGPU_ERR_CUDA, cudaGetErrorString(e));
    return KGPU_OK;
}

int kgpu_plan_get_info(kgpu_plan *p, kgpu_plan_info *info) {
    if (!p || !info) return fail(KGPU_ERR_INVALID, "NULL argument");
    std::memset(info, 0, sizeof *info);
    info->n_groups = (uint32_t)p->host.groups.size();
    for (size_t gi = 0; gi < p->host.groups.size(); gi++) {
        const Group &g = p->host.groups[gi];
        info->n_voices += g.n_voices;
        info->state_bytes += (uint64_t)g.n_voices * g.prog.n_regs * 4;
        if (p->gd[gi].recipe >= 0) info->n_fused_groups++;
    }
    info->n_mix_nodes = p->host.n_mix_nodes;
    info->dropped_changes = p->host.dropped_changes;
    info->ignored_delays = p->host.ignored_delays;
    info->device_events = p->host.device_events;
    info->kernel_launches = p->kernel_launches;
    return KGPU_OK;
}

const char *kgpu_plan_group_kernel(kgpu_plan *p, uint32_t group) {
    if (!p || group >= p->host.groups.size()) return "";
    return p->host.groups[group].kernel_name.c_str();
}

int kgpu_plan_prepare(kgpu_plan *p, uint64_t n_blocks) {
    if (!p || n_blocks == 0) return fail(KGPU_ERR_INVALID, "kgpu_plan_prepare: bad argument");
    try {
        CUDA_TRY(cudaSetDevice(p->device));
        if (p->prepared) KGPU_THROW(KGPU_ERR_STATE, "kgpu_plan_prepare: a prepared render is already pending");
        const uint64_t bpl = blocks_per_launch(p);
        prepare_range(p, n_blocks, bpl, p->stream);
        CUDA_TRY(cudaStreamSynchronize(p->stream));
        p->prepared = true;
        p->prepared_blocks = n_blocks;
        p->prepared_bpl = bpl;
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

float kgpu_plan_last_kernel_ms(kgpu_plan *p, uint32_t kernel_class, uint32_t *n_launches) {
    if (!p) return -1.f;
    float total = 0.f;
    uint32_t n = 0;
    for (size_t i = 0; i < p->kev_class.size(); i++) {
        if (p->kev_class[i] != kernel_class) continue;
        if (cudaEventSynchronize(p->kev[2 * i + 1]) != cudaSuccess) return -1.f;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p->kev[2 * i], p->kev[2 * i + 1]) != cudaSuccess) return -1.f;
        total += ms;
        n++;
    }
    if (n_launches) *n_launches = n;
    return total;
}

uint64_t kgpu_plan_last_upload_bytes(kgpu_plan *p) { return p ? p->last_h2d_bytes : 0; }

int kgpu_plan_set_peer_bus(kgpu_plan *p, uint32_t rank, uint32_t world, void *root_buffer, uint64_t buffer_bytes) {
    if (!p) return fail(KGPU_ERR_INVALID, "kgpu_plan_set_peer_bus: NULL plan");
    if (world <= 1 || !root_buffer) { // detach
        p->peer_world = 0;
        return KGPU_OK;
    }
    const uint64_t header = kgpu_peer_bus_header_bytes(world);
    if (rank >= world || buffer_bytes <= header || ((uintptr_t)root_buffer & 15u))
        return fail(KGPU_ERR_INVALID, "kgpu_plan_set_peer_bus: bad rank / buffer");
    uint8_t *base = (uint8_t *)root_buffer;
    p->peer_rank = rank;
    p->peer_world = world;
    p->peer_flags = (uint32_t *)base;
    p->peer_consumed = p->peer_flags + (size_t)world * KGPU_PEER_MAX_LAUNCHES;
    p->peer_timeout = p->peer_consumed + 1;
    p->peer_slots = (float *)(base + header);
    p->peer_slot_floats = ((buffer_bytes - header) / 4 / world) & ~(uint64_t)63;
    p->peer_epoch = 0;
    return KGPU_OK;
}

uint64_t kgpu_peer_bus_header_bytes(uint32_t world) { return (((uint64_t)world * KGPU_PEER_MAX_LAUNCHES + 2) * 4 + 255) & ~(uint64_t)255; }
uint64_t kgpu_peer_bus_bytes(uint32_t world, uint64_t floats_per_rank) {
    return kgpu_peer_bus_header_bytes(world) + (uint64_t)world * ((floats_per_rank + 63) & ~(uint64_t)63) * 4;
}

int kgpu_plan_peer_bus_timed_out(kgpu_plan *p) {
    if (!p || !p->peer_world) return 0;
    uint32_t v = 0;
    if (cudaMemcpy(&v, p->peer_timeout, 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (int)v;
}

int kgpu_plan_set_host_threads(kgpu_plan *p, uint32_t n_threads) {
    if (!p) return fail(KGPU_ERR_INVALID, "kgpu_plan_set_host_threads: NULL plan");
    if (p->host.pool) return fail(KGPU_ERR_STATE, "kgpu_plan_set_host_threads must be called before the first render / large push");
    p->host.pool_threads = n_threads;
    return KGPU_OK;
}

int kgpu_plan_set_blocks_per_launch(kgpu_plan *p, uint64_t blocks) {
    if (!p || blocks == 0) return fail(KGPU_ERR_INVALID, "kgpu_plan_set_blocks_per_launch: bad argument");
    if (p->prepared) return fail(KGPU_ERR_STATE, "kgpu_plan_set_blocks_per_launch: a prepared render is pending");
    p->max_blocks_per_launch = blocks;
    return KGPU_OK;
}

// ---- snapshot / restore of the whole render state (SURVEY 8f rank 4) ---------------------------
// Everything a later render depends on: the voices' registers on the device, the control-side state of every
// node of every voice (wrapper queues, smoothing ramps, setters' cached fields), the queued events (near and
// far), the simulated events that lie beyond the last render's end, the frame clock and the counters.
struct kgpu_snapshot {
    std::vector<std::vector<uint32_t>> regs;       // per group: [n_regs][n_voices]
    std::vector<std::vector<HostNode, HugeAllocator<HostNode>>> host; // per group
    decltype(HostPlan::pending) pending, pending_far;
    uint64_t far_horizon = UINT64_MAX;
    size_t pending_clean = 0;
    std::vector<std::vector<VoiceEvent>> later;
    std::vector<int32_t> voice_ramps;
    std::vector<uint64_t> voice_base;
    uint64_t n_active_ramps = 0, dropped_changes = 0, ignored_delays = 0, device_events = 0, frame_clock = 0;
    uint64_t graph_hash = 0; // HostPlan::graph_hash of the plan the snapshot was taken from
    bool rendered = false;
};

namespace {
// A snapshot may come from a byte image (kgpu_snapshot_deserialize): before any of it is used as an index, everything
// that is immutable in a plan must equal the plan's own, and every index it carries must be in range.
void validate_snapshot(const kgpu_plan *p, const kgpu_snapshot *s) {
    const HostPlan &H = p->host;
    auto bad = [](const char *what) { KGPU_THROW(KGPU_ERR_INVALID, "kgpu_plan_restore: the snapshot does not fit this plan (%s)", what); };
    if (s->graph_hash != H.graph_hash) bad("it was taken from another graph");
    if (s->regs.size() != p->gd.size() || s->host.size() != p->gd.size()) bad("group count");
    if (s->voice_base != H.voice_base) bad("voices per group");
    if (s->voice_ramps.size() != H.voice_ramps.size()) bad("voice count");
    if (s->pending_clean > s->pending.size()) bad("pending_clean");
    for (const auto &l : s->later)
        if (!l.empty()) bad("leftover device events");
    for (size_t gi = 0; gi < p->gd.size(); gi++) {
        const Group &g = H.groups[gi];
        if (s->regs[gi].size() != (size_t)g.prog.n_regs * g.n_voices || s->host[gi].size() != g.host.size()) bad("group size");
        for (size_t i = 0; i < g.host.size(); i++) {
            const HostNode &a = s->host[gi][i], &b = g.host[i];
            if (a.kind != b.kind || a.dev_kind != b.dev_kind || a.reg != b.reg || a.n_seg != b.n_seg || a.base_params != b.base_params ||
                a.has_smooth != b.has_smooth || a.has_precise != b.has_precise || a.smooth_level != b.smooth_level ||
                a.precise_level != b.precise_level || a.wr.size() != b.wr.size() || a.ar_regs != b.ar_regs)
                bad("node layout");
            if (a.kind == KGPU_SVF ? a.mode > 8 : a.mode != b.mode) bad("node mode");
            for (size_t l = 0; l < a.wr.size(); l++) {
                const WrapSim &x = a.wr[l], &y = b.wr[l];
                if (x.kind != y.kind || x.capacity != y.capacity || x.reg != y.reg || x.inner_params != y.inner_params ||
                    x.smooth.size() != y.smooth.size() || x.next_delay.size() != y.next_delay.size() || x.ar_bound.size() != y.ar_bound.size())
                    bad("wrapper layout");
                if (x.queue.size() > x.capacity) bad("WrPreciseTiming queue longer than its capacity");
                for (const QueuedChange &q : x.queue)
                    if (q.param >= x.next_delay.size() || q.value.kind > PV::Smoothing) bad("queued change");
            }
        }
    }
    auto check_events = [&](const decltype(HostPlan::pending) &v) {
        for (const RawEvent &e : v) {
            if (e.node >= H.node_ref.size()) bad("event node");
            const NodeRef &nr = H.node_ref[e.node];
            if (nr.group < 0 || e.param >= nr.n_params || e.local != nr.local || e.gvoice != H.voice_base[nr.group] + nr.voice ||
                e.value_kind() > 4 || e.smoothing_kind() > 2)
                bad("queued event");
        }
    };
    check_events(s->pending);
    check_events(s->pending_far);
}
} // namespace

int kgpu_plan_snapshot(kgpu_plan *p, kgpu_snapshot **out) {
    if (!p || !out) return fail(KGPU_ERR_INVALID, "kgpu_plan_snapshot: NULL argument");
    *out = nullptr;
    try {
        if (p->prepared) KGPU_THROW(KGPU_ERR_STATE, "kgpu_plan_snapshot: a prepared render is pending");
        if (p->host.stream_active) KGPU_THROW(KGPU_ERR_STATE, "kgpu_plan_snapshot: a render call is in progress");
        CUDA_TRY(cudaSetDevice(p->device));
        CUDA_TRY(cudaStreamSynchronize(p->stream));
        std::unique_ptr<kgpu_snapshot> s(new kgpu_snapshot());
        for (size_t gi = 0; gi < p->gd.size(); gi++) {
            const Group &g = p->host.groups[gi];
            s->regs.emplace_back((size_t)g.prog.n_regs * g.n_voices);
            if (!s->regs.back().empty())
                CUDA_TRY(cudaMemcpy(s->regs.back().data(), p->gd[gi].regs.p, s->regs.back().size() * 4, cudaMemcpyDeviceToHost));
            s->host.push_back(g.host);
        }
        s->pending = p->host.pending;
        s->pending_far = p->host.pending_far;
        s->far_horizon = p->host.far_horizon;
        s->pending_clean = p->host.pending_clean;
        s->later = p->host.later;
        s->voice_ramps = p->host.voice_ramps;
        s->voice_base = p->host.voice_base;
        s->n_active_ramps = p->host.n_active_ramps;
        s->dropped_changes = p->host.dropped_changes;
        s->ignored_delays = p->host.ignored_delays;
        s->device_events = p->host.device_events;
        s->frame_clock = p->frame_clock;
        s->rendered = p->rendered;
        s->graph_hash = p->host.graph_hash;
        *out = s.release();
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

int kgpu_plan_restore(kgpu_plan *p, const kgpu_snapshot *s) {
    if (!p || !s) return fail(KGPU_ERR_INVALID, "kgpu_plan_restore: NULL argument");
    try {
        if (p->host.stream_active) KGPU_THROW(KGPU_ERR_STATE, "kgpu_plan_restore: a render call is in progress");
        if (p->prepared) KGPU_THROW(KGPU_ERR_STATE, "kgpu_plan_restore: a prepared render is pending");
        validate_snapshot(p, s);
        CUDA_TRY(cudaSetDevice(p->device));
        CUDA_TRY(cudaStreamSynchronize(p->stream));
        for (size_t gi = 0; gi < p->gd.size(); gi++) {
            if (!s->regs[gi].empty())
                CUDA_TRY(cudaMemcpy(p->gd[gi].regs.p, s->regs[gi].data(), s->regs[gi].size() * 4, cudaMemcpyHostToDevice));
            p->host.groups[gi].host = s->host[gi];
        }
        p->host.pending = s->pending;
        p->host.pending_far = s->pending_far;
        p->host.far_horizon = s->far_horizon;
        p->host.pending_clean = s->pending_clean;
        p->host.later = s->later;
        // the ramp bookkeeping is derived state: rebuilt from the nodes' flags rather than trusted
        p->host.voice_ramps.assign(p->host.voice_base.back(), 0);
        p->host.n_active_ramps = 0;
        for (size_t gi = 0; gi < p->gd.size(); gi++) {
            const Group &g = p->host.groups[gi];
            const size_t nn = g.tpl.nodes.size();
            for (size_t i = 0; i < g.host.size(); i++)
                if (g.host[i].ramp_active) {
                    p->host.voice_ramps[p->host.voice_base[gi] + i / nn]++;
                    p->host.n_active_ramps++;
                }
        }
        p->host.dropped_changes = s->dropped_changes;
        p->host.ignored_delays = s->ignored_delays;
        p->host.device_events = s->device_events;
        p->frame_clock = s->frame_clock;
        p->rendered = s->rendered;
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    } catch (const std::exception &e) {
        return fail(KGPU_ERR_INVALID, std::string("kgpu_plan_restore: ") + e.what());
    }
}

void kgpu_snapshot_destroy(kgpu_snapshot *s) { delete s; }

// ---- a snapshot as bytes (checkpoint on disk, resume in another process on the same graph) ------------
// Flat little-endian image: magic, version, then every field length-prefixed.  The leaf structs are plain data
// and are written field by field (no padding bytes, no pointers), so the image depends on this file's version
// number only.
extern "C++" {
namespace {
constexpr uint64_t SNAP_MAGIC = 0x50414E5355504B47ull; // "GKPUSNAP"
constexpr uint32_t SNAP_VERSION = 3;
struct Writer {
    uint8_t *buf;
    uint64_t cap, pos = 0;
    void raw(const void *p, size_t n) {
        if (buf && pos + n <= cap) std::memcpy(buf + pos, p, n);
        pos += n;
    }
    template <class T> void pod(const T &v) { static_assert(std::is_trivially_copyable<T>::value, "pod"); raw(&v, sizeof v); }
    template <class V> void pods(const V &v) { // vector of padding-free scalars
        pod<uint64_t>(v.size());
        if (!v.empty()) raw(v.data(), v.size() * sizeof(v[0]));
    }
};
struct Reader {
    const uint8_t *buf;
    uint64_t size, pos = 0;
    void raw(void *p, size_t n) {
        if (pos + n > size) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: truncated image");
        std::memcpy(p, buf + pos, n);
        pos += n;
    }
    template <class T> T pod() { T v; raw(&v, sizeof v); return v; }
    template <class V> void pods(V &v) {
        const uint64_t n = pod<uint64_t>();
        if (n > (size - pos) / sizeof(v[0])) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
        v.resize(n);
        if (n) raw(v.data(), n * sizeof(v[0]));
    }
};
void put_pv(Writer &w, const PV &v) { w.pod<uint8_t>(v.kind); w.pod(v.f); w.pod(v.smoothing); w.pod(v.smooth_seconds); }
void get_pv(Reader &r, PV &v) { v.kind = (PV::Kind)r.pod<uint8_t>(); v.f = r.pod<double>(); v.smoothing = r.pod<uint8_t>(); v.smooth_seconds = r.pod<float>(); }
void put_raw_events(Writer &w, const decltype(HostPlan::pending) &v) {
    w.pod<uint64_t>(v.size());
    for (const RawEvent &e : v) { w.pod(e.node); w.pod(e.gvoice); w.pod(e.param); w.pod(e.local); w.pod(e.kinds); w.pod(e.smooth_seconds); w.pod(e.value); w.pod(e.due_frame); }
}
void get_raw_events(Reader &r, decltype(HostPlan::pending) &v) {
    const uint64_t n = r.pod<uint64_t>();
    if (n > (r.size - r.pos) / 32) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
    v.resize(n);
    for (RawEvent &e : v) {
        std::memset(&e, 0, sizeof e);
        e.node = r.pod<uint32_t>(); e.gvoice = r.pod<uint32_t>(); e.param = r.pod<uint16_t>(); e.local = r.pod<uint8_t>(); e.kinds = r.pod<uint8_t>();
        e.smooth_seconds = r.pod<float>(); e.value = r.pod<double>(); e.due_frame = r.pod<uint64_t>();
    }
}
void put_node(Writer &w, const HostNode &h) {
    w.pod(h.kind); w.pod(h.dev_kind); w.pod(h.mode); w.pod(h.reg); w.pod(h.n_seg); w.pod(h.base_params);
    w.pod(h.f0); w.pod(h.f1); w.pod(h.f2); w.pod(h.d0);
    for (float c : h.svf_coef) w.pod(c);
    w.pod<uint8_t>(h.has_smooth); w.pod<uint8_t>(h.has_precise); w.pod(h.smooth_level); w.pod(h.precise_level);
    w.pod<uint8_t>(h.ramp_active); w.pod<uint8_t>(h.ar_regs); w.pod(h.ramp_list_pos);
    for (uint16_t d : h.nd) w.pod(d);
    w.pod<uint64_t>(h.wr.size());
    for (const WrapSim &x : h.wr) {
        w.pod(x.kind); w.pod(x.capacity); w.pod(x.reg); w.pod(x.inner_params);
        w.pod<uint64_t>(x.smooth.size());
        for (const SmoothState &m : x.smooth) {
            w.pod<uint8_t>(m.linear); w.pod(m.current_value); w.pod(m.start_value); w.pod(m.end_value);
            w.pod(m.duration_frames); w.pod(m.frames_elapsed); w.pod<uint8_t>(m.done);
        }
        w.pods(x.next_delay);
        w.pod<uint64_t>(x.queue.size());
        for (const QueuedChange &q : x.queue) { w.pod(q.delay); w.pod(q.param); put_pv(w, q.value); }
        w.pods(x.ar_bound);
    }
}
void get_node(Reader &r, HostNode &h) {
    h.kind = r.pod<uint8_t>(); h.dev_kind = r.pod<uint8_t>(); h.mode = r.pod<uint32_t>(); h.reg = r.pod<uint16_t>(); h.n_seg = r.pod<uint16_t>();
    h.base_params = r.pod<uint32_t>();
    h.f0 = r.pod<float>(); h.f1 = r.pod<float>(); h.f2 = r.pod<float>(); h.d0 = r.pod<double>();
    for (float &c : h.svf_coef) c = r.pod<float>();
    h.has_smooth = r.pod<uint8_t>() != 0; h.has_precise = r.pod<uint8_t>() != 0; h.smooth_level = r.pod<int8_t>(); h.precise_level = r.pod<int8_t>();
    h.ramp_active = r.pod<uint8_t>() != 0; h.ar_regs = r.pod<uint8_t>() != 0; h.ramp_list_pos = r.pod<uint32_t>();
    for (uint16_t &d : h.nd) d = r.pod<uint16_t>();
    const uint64_t nw = r.pod<uint64_t>();
    if (nw > 64) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad wrapper count");
    h.wr.resize(nw);
    for (WrapSim &x : h.wr) {
        x.kind = r.pod<uint8_t>(); x.capacity = r.pod<uint32_t>(); x.reg = r.pod<uint16_t>(); x.inner_params = r.pod<uint32_t>();
        const uint64_t ns = r.pod<uint64_t>();
        if (ns > 4096) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
        x.smooth.resize(ns);
        for (SmoothState &m : x.smooth) {
            m.linear = r.pod<uint8_t>() != 0; m.current_value = r.pod<double>(); m.start_value = r.pod<double>(); m.end_value = r.pod<double>();
            m.duration_frames = r.pod<uint64_t>(); m.frames_elapsed = r.pod<uint64_t>(); m.done = r.pod<uint8_t>() != 0;
        }
        r.pods(x.next_delay);
        const uint64_t nq = r.pod<uint64_t>();
        if (nq > (1u << 20)) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
        x.queue.resize(nq);
        for (QueuedChange &q : x.queue) { q.delay = r.pod<uint16_t>(); q.param = r.pod<uint32_t>(); get_pv(r, q.value); }
        r.pods(x.ar_bound);
    }
}
void put_voice_events(Writer &w, const std::vector<VoiceEvent> &v) {
    w.pod<uint64_t>(v.size());
    for (const VoiceEvent &e : v) { w.pod(e.voice); w.pod(e.seq); w.pod(e.frame); w.pod(e.ev.frame); w.pod(e.ev.node); w.pod(e.ev.op); w.pod(e.ev.reg); w.pod(e.ev.value); }
}
void get_voice_events(Reader &r, std::vector<VoiceEvent> &v) {
    const uint64_t n = r.pod<uint64_t>();
    if (n > (r.size - r.pos) / 32) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
    v.resize(n);
    for (VoiceEvent &e : v) {
        e.voice = r.pod<uint32_t>(); e.seq = r.pod<uint32_t>(); e.frame = r.pod<uint64_t>();
        e.ev.frame = r.pod<uint32_t>(); e.ev.node = r.pod<uint16_t>(); e.ev.op = r.pod<uint16_t>(); e.ev.reg = r.pod<uint32_t>(); e.ev.value = r.pod<uint32_t>();
    }
}
void write_snapshot(Writer &w, const kgpu_snapshot &s) {
    w.pod(SNAP_MAGIC); w.pod(SNAP_VERSION); w.pod(s.graph_hash);
    w.pod<uint64_t>(s.regs.size());
    for (size_t gi = 0; gi < s.regs.size(); gi++) {
        w.pods(s.regs[gi]);
        w.pod<uint64_t>(s.host[gi].size());
        for (const HostNode &h : s.host[gi]) put_node(w, h);
    }
    put_raw_events(w, s.pending); put_raw_events(w, s.pending_far);
    w.pod(s.far_horizon); w.pod<uint64_t>(s.pending_clean);
    w.pod<uint64_t>(s.later.size());
    for (const auto &l : s.later) put_voice_events(w, l);
    w.pods(s.voice_ramps); w.pods(s.voice_base);
    w.pod(s.n_active_ramps); w.pod(s.dropped_changes); w.pod(s.ignored_delays); w.pod(s.device_events); w.pod(s.frame_clock);
    w.pod<uint8_t>(s.rendered);
}
} // namespace
} // extern "C++"

/* Size query: buf == NULL.  Returns KGPU_ERR_INVALID if cap is too small (*size still receives the need). */
int kgpu_snapshot_serialize(const kgpu_snapshot *s, void *buf, uint64_t cap, uint64_t *size) {
    if (!s || !size) return fail(KGPU_ERR_INVALID, "kgpu_snapshot_serialize: NULL argument");
    Writer w{static_cast<uint8_t *>(buf), buf ? cap : 0};
    write_snapshot(w, *s);
    *size = w.pos;
    if (buf && w.pos > cap) return fail(KGPU_ERR_INVALID, "kgpu_snapshot_serialize: buffer too small");
    return KGPU_OK;
}

int kgpu_snapshot_deserialize(const void *buf, uint64_t size, kgpu_snapshot **out) {
    if (!buf || !out) return fail(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: NULL argument");
    *out = nullptr;
    try {
        Reader r{static_cast<const uint8_t *>(buf), size};
        if (r.pod<uint64_t>() != SNAP_MAGIC) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: not a snapshot image");
        if (r.pod<uint32_t>() != SNAP_VERSION) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: unsupported image version");
        std::unique_ptr<kgpu_snapshot> s(new kgpu_snapshot());
        s->graph_hash = r.pod<uint64_t>();
        const uint64_t ng = r.pod<uint64_t>();
        if (ng > (1u << 20)) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad group count");
        s->regs.resize(ng);
        s->host.resize(ng);
        for (uint64_t gi = 0; gi < ng; gi++) {
            r.pods(s->regs[gi]);
            const uint64_t nh = r.pod<uint64_t>();
            if (nh > (size - r.pos)) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
            s->host[gi].resize(nh);
            for (HostNode &h : s->host[gi]) get_node(r, h);
        }
        get_raw_events(r, s->pending);
        get_raw_events(r, s->pending_far);
        s->far_horizon = r.pod<uint64_t>();
        s->pending_clean = (size_t)r.pod<uint64_t>();
        const uint64_t nl = r.pod<uint64_t>();
        if (nl > (1u << 20)) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: bad length");
        s->later.resize(nl);
        for (auto &l : s->later) get_voice_events(r, l);
        r.pods(s->voice_ramps);
        r.pods(s->voice_base);
        s->n_active_ramps = r.pod<uint64_t>(); s->dropped_changes = r.pod<uint64_t>(); s->ignored_delays = r.pod<uint64_t>();
        s->device_events = r.pod<uint64_t>(); s->frame_clock = r.pod<uint64_t>();
        s->rendered = r.pod<uint8_t>() != 0;
        if (r.pos != size) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_snapshot_deserialize: trailing bytes");
        *out = s.release();
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    } catch (const std::exception &e) { // bad_alloc / length_error from a hostile length field
        return fail(KGPU_ERR_INVALID, std::string("kgpu_snapshot_deserialize: ") + e.what());
    }
}

float kgpu_plan_last_render_ms(kgpu_plan *p) {
    if (!p || !p->timed) return -1.f;
    if (cudaEventSynchronize(p->ev1) != cudaSuccess) return -1.f;
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, p->ev0, p->ev1) != cudaSuccess) return -1.f;
    return ms;
}

} // extern "C"

// ---- host-only debug entry points (csrc/debug.h) ------------------------------------------------
#include "debug.h"
#include "sinf_glibc.h"
extern "C" {

int kgpu_debug_sinf(const float *x, float *y, size_t n) {
    for (size_t i = 0; i < n; i++) y[i] = kgpu::kn_sinf_glibc(x[i]);
    return KGPU_OK;
}


int kgpu_debug_simulate(const kgpu_graph_desc *desc, const kgpu_event *events, size_t n_events, uint64_t n_blocks,
                        uint64_t blocks_per_call, kgpu_debug_event *out, size_t cap, size_t *n_out, kgpu_debug_node *nodes_out,
                        kgpu_plan_info *info) {
    try {
        HostPlan hp;
        const bool timing = getenv("KGPU_TIMING") != nullptr;
        auto now = [] { return std::chrono::steady_clock::now(); };
        auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        auto t0_ = now();
        hp.build(*desc);
        auto t1_ = now();
        hp.push(events, n_events, 0);
        auto t2_ = now();
        double sim_ms = 0;
        size_t n = 0;
        const uint64_t bs = hp.block_size;
        if (blocks_per_call == 0) blocks_per_call = n_blocks;
        HostPlan::CompiledEvents ce;
        std::vector<uint32_t> chunks(hp.groups.size(), 1);
        for (uint64_t b = 0; b < n_blocks; b += blocks_per_call) {
            const uint64_t t0 = b * bs, t1 = std::min(n_blocks, b + blocks_per_call) * bs;
            auto a_ = now();
            hp.compile_events({t0, t1}, chunks, ce);
            sim_ms += ms(a_, now());
            for (uint32_t gi = 0; gi < hp.groups.size(); gi++) {
                if (!ce.piece_any[gi]) continue;
                const DevEvent *ev = ce.events.data() + ce.piece_ev[gi];
                const uint32_t *off = ce.offsets.data() + ce.piece_off[gi];
                for (uint32_t v = 0; v < hp.groups[gi].n_voices; v++)
                    for (uint32_t k = off[v]; k < off[v + 1]; k++) {
                        if (n < cap) out[n] = kgpu_debug_event{gi, v, ev[k].node, ev[k].op, ev[k].reg, ev[k].value, t0 + ev[k].frame};
                        n++;
                    }
            }
        }
        if (timing) fprintf(stderr, "[kgpu timing] build %.1f ms, push %.1f ms, compile_events %.1f ms\n", ms(t0_, t1_), ms(t1_, t2_), sim_ms);
        if (n_out) *n_out = n;
        if (nodes_out)
            for (uint32_t i = 0; i < desc->n_nodes; i++) {
                const NodeRef &nr = hp.node_ref[i];
                nodes_out[i] = kgpu_debug_node{nr.group, nr.voice, nr.local,
                                               nr.group >= 0 ? (uint32_t)hp.groups[nr.group].prog.nodes[nr.local].reg : 0u};
            }
        if (info) {
            std::memset(info, 0, sizeof *info);
            info->n_groups = (uint32_t)hp.groups.size();
            for (auto &g : hp.groups) {
                info->n_voices += g.n_voices;
                info->state_bytes += (uint64_t)g.n_voices * g.prog.n_regs * 4;
            }
            info->n_mix_nodes = hp.n_mix_nodes;
            info->dropped_changes = hp.dropped_changes;
            info->ignored_delays = hp.ignored_delays;
            info->device_events = hp.device_events;
        }
        return n > cap ? KGPU_ERR_INVALID : KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

/* Times the host half of `n_steps` render calls of n_blocks blocks each the way kgpu_render drives it (launch sizes
 * ramping 1/8, 1/4, 1/2, 1, 1, ... of `bpl` blocks; stream_begin, then stream_launch per launch), without a device.
 * The event schedule repeats every step (whole seconds per step).  out_ms: [n_steps][4] = push, stream_begin,
 * first launch ready (since the start of the call), all launches fetched. */
int kgpu_debug_host_bench(const kgpu_graph_desc *desc, const kgpu_event *events, size_t n_events, uint64_t n_blocks, uint64_t bpl,
                          uint32_t n_steps, uint32_t n_threads, double *out_ms) {
    try {
        HostPlan hp;
        hp.build(*desc);
        hp.pool_threads = n_threads;
        const uint64_t bs = hp.block_size;
        const uint64_t step_frames = n_blocks * bs;
        if (step_frames % hp.sample_rate) KGPU_THROW(KGPU_ERR_INVALID, "kgpu_debug_host_bench: a step must be a whole number of seconds");
        const uint32_t step_seconds = (uint32_t)(step_frames / hp.sample_rate);
        std::vector<kgpu_event> ev(events, events + n_events);
        std::vector<uint32_t> chunks(hp.groups.size(), 1);
        HostPlan::CompiledEvents ce;
        auto now = [] { return std::chrono::steady_clock::now(); };
        auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
        uint64_t clock = 0;
        size_t total_ev = 0;
        for (uint32_t s = 0; s < n_steps; s++) {
            std::vector<uint64_t> bounds{clock};
            uint64_t left = n_blocks, next = bpl < 64 || n_blocks < 2 * bpl ? bpl : std::max<uint64_t>(32, bpl / 64);
            while (left) {
                const uint64_t nb = std::min(next, left);
                bounds.push_back(bounds.back() + nb * bs);
                left -= nb;
                next = std::min(bpl, next + next / 2);
            }
            const auto t0 = now();
            hp.push(ev.data(), ev.size(), clock);
            const auto t1 = now();
            hp.stream_begin(bounds, chunks);
            const auto t2 = now();
            auto t3 = t2;
            for (size_t L = 0; L + 1 < bounds.size(); L++) {
                hp.stream_launch(L, ce);
                total_ev += ce.events.size();
                if (L == 0) t3 = now();
            }
            const auto t4 = now();
            hp.stream_end();
            out_ms[4 * s + 0] = ms(t0, t1);
            out_ms[4 * s + 1] = ms(t1, t2);
            out_ms[4 * s + 2] = ms(t0, t3);
            out_ms[4 * s + 3] = ms(t0, t4);
            clock += step_frames;
            for (kgpu_event &e : ev)
                if (e.time_kind == 1) e.seconds += step_seconds;
        }
        return total_ev ? KGPU_OK : KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

/* Host-only: generate and compile (NVRTC -> cubin cache, no device needed) the kernel of every voice template of `desc`
 * that has no hand-written recipe.  *n_generated / *n_cached count them; fails with the compiler's log otherwise. */
int kgpu_debug_jit_compile(const kgpu_graph_desc *desc, uint32_t tap_outputs, uint32_t *n_generated, uint32_t *n_cached) {
    try {
        HostPlan hp;
        hp.build(*desc);
        uint32_t ng = 0, nc = 0;
        for (Group &g : hp.groups) {
            if (match_fused_recipe(g.prog, hp.block_size) >= 0) continue;
            std::vector<uint16_t> tapped;
            if (tap_outputs) { // what kgpu_plan_add_tap on a voice's bus output does: keep that value slot live to the end of the frame
                std::vector<std::pair<uint32_t, uint32_t>> pinned;
                for (auto &o : g.tpl.outs) {
                    std::pair<uint32_t, uint32_t> pin{(uint32_t)std::get<0>(o), std::get<1>(o)};
                    if (std::find(pinned.begin(), pinned.end(), pin) == pinned.end()) pinned.push_back(pin);
                }
                recompile_group_slots(g, hp.sample_rate, pinned);
                for (auto &pin : pinned) {
                    const uint16_t slot = g.slot_of[pin.first][pin.second];
                    if (std::find(tapped.begin(), tapped.end(), slot) == tapped.end()) tapped.push_back(slot);
                }
            }
            const std::string src = jit_source(g.prog, tapped);
            if (src.empty()) KGPU_THROW(KGPU_ERR_UNSUPPORTED, "jit: the generator does not cover a node of this template");
            std::vector<char> cubin;
            std::string err;
            bool cached = false;
            if (!jit_cubin(src, cubin, err, &cached)) KGPU_THROW(KGPU_ERR_INVALID, "%s", err.c_str());
            ng++;
            nc += cached;
        }
        if (n_generated) *n_generated = ng;
        if (n_cached) *n_cached = nc;
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}

int kgpu_debug_init_reg(const kgpu_graph_desc *desc, uint32_t node, uint32_t reg_offset, uint32_t *value) {
    try {
        HostPlan hp;
        hp.build(*desc);
        if (node >= hp.node_ref.size() || hp.node_ref[node].group < 0) return fail(KGPU_ERR_INVALID, "node not in a voice");
        const NodeRef &nr = hp.node_ref[node];
        const Group &g = hp.groups[nr.group];
        uint32_t reg = g.prog.nodes[nr.local].reg + reg_offset;
        if (reg >= g.prog.n_regs) return fail(KGPU_ERR_INVALID, "register out of range");
        *value = g.init_regs[(size_t)reg * g.n_voices + nr.voice];
        return KGPU_OK;
    } catch (const Error &e) {
        return fail(e.code, e.msg);
    }
}
}
