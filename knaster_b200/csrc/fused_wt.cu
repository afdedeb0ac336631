// fused_wt.cu -- recipe 2 "render_add_wt": the additive wavetable bank (BASELINE.json configs[1]).
//
//   voice = SinWt (osc.rs:97-168) [.wr_mul(a)] [.smooth_params()]  ->  mix bus
//
// SinWt's phase is a wrapping u32 (wavetable.rs:21-53), so -- unlike the f32 recurrences of the
// other recipes -- it has an exact closed form: the phase at frame k of a block is
// phase_block + k * inc (mod 2^32), and the phase at a block start is the wrapping prefix sum of
// inc * block_size over the blocks before it.  Without a WrPreciseTiming wrapper every parameter
// change lands on a block boundary (graph_gen.rs:269-305; WrSmoothParams advances once per
// process_block call, smooth_params.rs:143-188), so a voice is fully described by one 16-byte
// record per block.  That makes TIME the parallel axis:
//
//   add_wt_params   one thread per voice walks the launch's blocks in order (the phase prefix
//                   scan: one IMAD per block), applies the parameter events at block boundaries
//                   and writes {phase, inc, offset, gain} per (block, voice);
//   add_wt_render   one thread per frame and voice slice, the 64 KiB sine table staged in shared
//                   memory: out[f] = sum_v gain_v * table[((phase_v + k*inc_v + off_v) >> 16) & 0x3FFF]
//                   accumulated in registers in voice order (deterministic), one partial row per
//                   slice.  A warp covers 32 consecutive frames of ONE block, so the per-voice
//                   record is a single broadcast load.
//
// Per voice-sample: 1 IMAD + 1 IADD + 1 shift/mask + 1 LDS + 1 FMUL + 1 FADD (+ 1/32 LDG.128).
#include <cuda_runtime.h>

#include <atomic>
#include <stdint.h>

#include "dev.h"
#include "kernels.h"
#include "nodes.cuh"
#include "plan.hpp"

namespace kgpu {

namespace {

struct __align__(16) WtParam {
    uint32_t phase, inc, off;
    float gain;
};

constexpr uint32_t WT_REG_PHASE = 0, WT_REG_OFF = 1, WT_REG_INC = 2;
constexpr int WT_THREADS = 256;
constexpr int WT_TILES_PER_CTA = 8;

constexpr uint32_t WT_CHUNK = 32; // blocks per add_wt_params thread

// one thread per (voice, chunk of WT_CHUNK blocks).  The state at the chunk start comes from a
// scan over the voice's EVENTS before it (a handful per launch), not over its blocks: between two
// events the phase advances by inc * block_size * (blocks in between), exactly, mod 2^32.
__global__ void add_wt_params(FusedArgs a, uint32_t gain_reg, WtParam *__restrict__ table) {
    const uint32_t V = a.n_voices;
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t chunk = blockIdx.y;
    if (v >= V) return;
    const uint32_t bs = a.block_size, n_blocks = a.n_frames / bs;
    const uint32_t b_begin = chunk * WT_CHUNK, b_end = min(n_blocks, b_begin + WT_CHUNK);
    uint32_t phase = a.regs[(size_t)WT_REG_PHASE * V + v];
    uint32_t off = a.regs[(size_t)WT_REG_OFF * V + v];
    uint32_t inc = a.regs[(size_t)WT_REG_INC * V + v];
    float gain = gain_reg != 0xFFFFFFFFu ? __uint_as_float(a.regs[(size_t)gain_reg * V + v]) : 1.0f;
    uint32_t cur = 0, end = 0;
    if (a.events) {
        cur = a.ev_off[v];
        end = a.ev_off[v + 1];
    }
    auto apply = [&](const DevEvent &e) {
        if (e.op != OP_SET) return;
        if (e.reg == WT_REG_PHASE) phase = e.value;
        else if (e.reg == WT_REG_OFF) off = e.value;
        else if (e.reg == WT_REG_INC) inc = e.value;
        else if (e.reg == gain_reg) gain = __uint_as_float(e.value);
    };
    // block in which an event takes effect: the first block starting at or after its frame
    auto ev_block = [&](const DevEvent &e) { return (e.frame + bs - 1) / bs; };
    // ---- events before the chunk: jump from event to event
    uint32_t b = 0; // `phase` is the phase at the start of block b
    while (cur < end) {
        const DevEvent e = a.events[cur];
        const uint32_t eb = ev_block(e);
        if (eb >= b_begin) break;
        phase += inc * bs * (eb - b);
        b = eb;
        apply(e);
        cur++;
    }
    phase += inc * bs * (b_begin - b);
    // ---- the chunk's own blocks
    uint32_t next_block = cur < end ? ev_block(a.events[cur]) : 0xFFFFFFFFu;
    for (b = b_begin; b < b_end; b++) {
        while (next_block <= b) { // parameter changes take effect at the block start
            apply(a.events[cur]);
            cur++;
            next_block = cur < end ? ev_block(a.events[cur]) : 0xFFFFFFFFu;
        }
        WtParam p;
        p.phase = phase;
        p.inc = inc;
        p.off = off;
        p.gain = gain;
        table[(size_t)b * V + v] = p;
        phase += inc * bs; // bs samples of `phase += inc` (wavetable.rs:50-52), wrapping
    }
    if (b_end == n_blocks) { // the thread of the last chunk leaves the voice's state for the next launch
        while (cur < end) apply(a.events[cur++]); // (none: every event of the launch lies before its end)
        a.regs_out[(size_t)WT_REG_PHASE * V + v] = phase;
        a.regs_out[(size_t)WT_REG_OFF * V + v] = off;
        a.regs_out[(size_t)WT_REG_INC * V + v] = inc;
        if (gain_reg != 0xFFFFFFFFu) a.regs_out[(size_t)gain_reg * V + v] = __float_as_uint(gain);
    }
}

constexpr uint32_t WT_VCHUNK = 128;     // voices staged in shared memory at a time
constexpr uint32_t WT_MAX_TILE_BLOCKS = WT_THREADS / 32; // a 256-frame tile touches at most 8 blocks (block_size >= 32)

// FPT = frames per thread.  FPT = 2 (block sizes that are multiples of 64): a thread renders frames k and k + 32 of ONE block, so the
// voice's record (a broadcast LDS.128) is loaded once per two samples.  Measured: 1.73 -> 1.70 ms per 10 s step of the 4096-partial
// bank -- the record load was not what keeps the shared-memory path 89 % busy (r2j capture); the table lookups are (1.34 wavefronts
// each: consecutive frames of a high partial stride through the 64 KiB table).
template <bool TAPS, int FPT>
__global__ void __launch_bounds__(WT_THREADS) add_wt_render(FusedArgs a, const WtParam *__restrict__ table, uint32_t n_slices, uint32_t n_tiles) {
    extern __shared__ __align__(16) float tab[]; // the sine table (wavetable.rs:130-139), then the staged voice records
    uint4 *stage = reinterpret_cast<uint4 *>(tab + SINE_TABLE_SIZE); // [tile block][WT_VCHUNK]
    {
        const float4 *src = reinterpret_cast<const float4 *>(a.sine_table);
        float4 *dst = reinterpret_cast<float4 *>(tab);
        for (uint32_t i = threadIdx.x; i < SINE_TABLE_SIZE / 4; i += WT_THREADS) dst[i] = src[i];
    }
    constexpr uint32_t TILE = WT_THREADS * FPT;
    const uint32_t V = a.n_voices, bs = a.block_size;
    const uint32_t slice = blockIdx.y;
    const uint32_t v0 = (uint32_t)((uint64_t)V * slice / n_slices), v1 = (uint32_t)((uint64_t)V * (slice + 1) / n_slices);
    float *prow = a.partials + (size_t)(a.row0 + slice) * a.n_frames;
    for (uint32_t tile = blockIdx.x * WT_TILES_PER_CTA; tile < min(n_tiles, (blockIdx.x + 1) * WT_TILES_PER_CTA); tile++) {
        const uint32_t f_tile = tile * TILE;
        // FPT = 2: warp w renders frames [64 w, 64 w + 64) of the tile, lane l the frames 64 w + l and 64 w + 32 + l (one block: bs % 64 == 0)
        const uint32_t f = FPT == 1 ? f_tile + threadIdx.x : f_tile + (threadIdx.x >> 5) * 64u + (threadIdx.x & 31u);
        const bool on = f < a.n_frames;
        const bool on2 = FPT == 2 && f + 32u < a.n_frames;
        const uint32_t b_first = f_tile / bs;
        const uint32_t b_last = (min(a.n_frames, f_tile + TILE) - 1) / bs;
        const uint32_t nb = b_last - b_first + 1;
        const uint32_t b = on ? f / bs : b_first, k = f - b * bs, k2 = k + 32u;
        float acc = 0.f, acc2 = 0.f;
        for (uint32_t vc = v0; vc < v1; vc += WT_VCHUNK) {
            const uint32_t nv = min(WT_VCHUNK, v1 - vc);
            __syncthreads(); // the previous chunk's readers are done (and the sine table is in place)
            for (uint32_t i = threadIdx.x; i < nb * nv; i += WT_THREADS) {
                const uint32_t bi = i / nv, vi = i - bi * nv;
                stage[bi * WT_VCHUNK + vi] = __ldg(reinterpret_cast<const uint4 *>(table + (size_t)(b_first + bi) * V + vc + vi));
            }
            __syncthreads();
            const uint4 *row = stage + (b - b_first) * WT_VCHUNK; // one broadcast LDS.128 per voice and warp
            uint32_t vi = 0;
            if (!TAPS) {
                for (; vi + 4 <= nv; vi += 4) {
                    const uint4 p0 = row[vi], p1 = row[vi + 1], p2 = row[vi + 2], p3 = row[vi + 3];
                    const uint32_t q0 = p0.x + p0.z, q1 = p1.x + p1.z, q2 = p2.x + p2.z, q3 = p3.x + p3.z; // (phase + k inc) + off, mod 2^32: any order
                    const float s0 = tab[((q0 + k * p0.y) >> 16) & 0x3FFFu] * __uint_as_float(p0.w); // WrMul, wrappers_core/math.rs:63-67
                    const float s1 = tab[((q1 + k * p1.y) >> 16) & 0x3FFFu] * __uint_as_float(p1.w);
                    const float s2 = tab[((q2 + k * p2.y) >> 16) & 0x3FFFu] * __uint_as_float(p2.w);
                    const float s3 = tab[((q3 + k * p3.y) >> 16) & 0x3FFFu] * __uint_as_float(p3.w);
                    acc = (((acc + s0) + s1) + s2) + s3;
                    if (FPT == 2) {
                        const float t0 = tab[((q0 + k2 * p0.y) >> 16) & 0x3FFFu] * __uint_as_float(p0.w);
                        const float t1 = tab[((q1 + k2 * p1.y) >> 16) & 0x3FFFu] * __uint_as_float(p1.w);
                        const float t2 = tab[((q2 + k2 * p2.y) >> 16) & 0x3FFFu] * __uint_as_float(p2.w);
                        const float t3 = tab[((q3 + k2 * p3.y) >> 16) & 0x3FFFu] * __uint_as_float(p3.w);
                        acc2 = (((acc2 + t0) + t1) + t2) + t3;
                    }
                }
            }
            for (; vi < nv; vi++) {
                const uint4 p = row[vi];
                const float s = tab[((p.x + k * p.y + p.z) >> 16) & 0x3FFFu] * __uint_as_float(p.w);
                if (TAPS && on)
                    for (uint32_t i = 0; i < a.n_taps; i++)
                        if (a.taps[i].voice == vc + vi) a.tap_out[(size_t)a.taps[i].tap * a.tap_stride + a.tap_frame0 + f] = s;
                acc = acc + s;
                if (FPT == 2) acc2 = acc2 + tab[((p.x + k2 * p.y + p.z) >> 16) & 0x3FFFu] * __uint_as_float(p.w);
            }
        }
        if (on) prow[f] = acc;
        if (on2) prow[f + 32u] = acc2;
    }
}

} // namespace

// Two voice shapes: SinWt[.wr_mul][.smooth_params] alone, and SinWt -> MathUGen<Mul> with a Constant (the
// README example `sine * 0.2`, README.md:35-47: table[..] * 0.2 is the same single f32 product as
// wr_mul(0.2), and a `value` event on the Constant is a write to the gain register like a `wr_mul` event).
static bool add_wt_shape(const DevProgram &p, uint32_t &gain_reg) {
    if (p.n_ubus != 1) return false;
    const DevNode &n = p.nodes[0];
    if (n.kind != DK_SINWT || n.reg != 0 || n.n_ar) return false;
    if (p.n_nodes == 1) {
        if (n.n_post > 1 || (n.n_post == 1 && n.post_op[0] != PO_MUL)) return false;
        gain_reg = n.n_post == 1 ? n.post_reg[0] : 0xFFFFFFFFu;
        return p.ubus_slot[0] == n.out_slot[0];
    }
    if (p.n_nodes != 3 || n.n_post) return false;
    const DevNode &c = p.nodes[1], &m = p.nodes[2];
    if (c.kind != DK_CONST || c.n_post || c.n_ar) return false;
    if (m.kind != DK_MATH || m.mode != 2 || m.n_out != 1 || m.n_post || m.n_ar) return false;
    const bool ab = m.in_slot[0] == (int)n.out_slot[0] && m.in_slot[1] == (int)c.out_slot[0];
    const bool ba = m.in_slot[1] == (int)n.out_slot[0] && m.in_slot[0] == (int)c.out_slot[0];
    if (!ab && !ba) return false;
    gain_reg = c.reg;
    return p.ubus_slot[0] == m.out_slot[0];
}
bool match_add_wt(const DevProgram &p, uint32_t block_size) {
    uint32_t gain_reg;
    return block_size % 32 == 0 && add_wt_shape(p, gain_reg);
}
uint32_t add_wt_slices(uint32_t n_voices) { return std::max(1u, std::min(32u, (n_voices + 127) / 128)); }
size_t add_wt_scratch_bytes(uint32_t n_voices, uint32_t n_frames, uint32_t block_size) {
    // the per-(block, voice) records, then a second copy of the voice registers (see launch_add_wt); the shape holds a few
    // registers, far below the small-voice limit the copy is sized for
    return (size_t)n_voices * (n_frames / block_size) * sizeof(WtParam) + (size_t)n_voices * SMALL_VOICE_REGS * 4;
}
cudaError_t launch_add_wt(const FusedArgs &a, cudaStream_t stream) {
    uint32_t gain_reg = 0xFFFFFFFFu;
    if (!add_wt_shape(*a.host_prog, gain_reg)) return cudaErrorNotSupported;
    WtParam *table = reinterpret_cast<WtParam *>(a.scratch);
    FusedArgs ap = a;
    ap.regs_out = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(a.scratch) + (size_t)a.n_voices * (a.n_frames / a.block_size) * sizeof(WtParam));
    // the params threads of different chunks read the launch-start registers while the last chunk's
    // thread writes the launch-end ones: they go to a second register file that is swapped in afterwards
    const uint32_t n_blocks = a.n_frames / a.block_size;
    const dim3 pgrid((a.n_voices + 127) / 128, (n_blocks + WT_CHUNK - 1) / WT_CHUNK);
    cudaError_t ce = cudaMemcpyAsync(ap.regs_out, a.regs, (size_t)a.host_prog->n_regs * a.n_voices * 4, cudaMemcpyDeviceToDevice, stream);
    if (ce != cudaSuccess) return ce;
    add_wt_params<<<pgrid, 128, 0, stream>>>(ap, gain_reg, table);
    ce = cudaMemcpyAsync(a.regs, ap.regs_out, (size_t)a.host_prog->n_regs * a.n_voices * 4, cudaMemcpyDeviceToDevice, stream);
    if (ce != cudaSuccess) return ce;
    const uint32_t n_slices = add_wt_slices(a.n_voices);
    // two frames per thread where a block holds both of a lane's frames (and no taps: the tapped form is test-only)
    const bool two = !a.n_taps && a.block_size % 64 == 0;
    const uint32_t tile_frames = WT_THREADS * (two ? 2u : 1u);
    const uint32_t n_tiles = (a.n_frames + tile_frames - 1) / tile_frames;
    const dim3 grid((n_tiles + WT_TILES_PER_CTA - 1) / WT_TILES_PER_CTA, n_slices);
    const size_t smem = SINE_TABLE_SIZE * sizeof(float) + (size_t)WT_MAX_TILE_BLOCKS * WT_VCHUNK * sizeof(uint4);
    // the opt-in above 48 KB of dynamic shared memory is a PER-DEVICE function attribute: one flag per device, so
    // that a second plan on another GPU of the same process (INTEGRATION.md "Several GPUs") gets it too
    static std::atomic<bool> attr_set[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64 || !attr_set[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(add_wt_render<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(add_wt_render<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(add_wt_render<true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64) attr_set[dev].store(true, std::memory_order_release);
    }
    if (a.n_taps) add_wt_render<true, 1><<<grid, WT_THREADS, smem, stream>>>(a, table, n_slices, n_tiles);
    else if (two) add_wt_render<false, 2><<<grid, WT_THREADS, smem, stream>>>(a, table, n_slices, n_tiles);
    else add_wt_render<false, 1><<<grid, WT_THREADS, smem, stream>>>(a, table, n_slices, n_tiles);
    return cudaGetLastError();
}

} // namespace kgpu
