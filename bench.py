#!/usr/bin/env python
"""bench.py -- voice-samples/sec of the batched render path on N B200s (BASELINE.json metric).

A "step" renders `--seconds` (default 10 s = 7500 blocks of 64 frames @ 48 kHz) of the
subtractive polysynth bank -- 16384 voices per GPU of PolyBlep saw -> SvfFilter lowpass ->
EnvAsr -> VCA with sample-accurate note events (BASELINE.json configs[2]; with N GPUs the
voices are sharded 16384/GPU and the stereo mix bus is summed onto rank 0: configs[4]).

  value            device-resident: events already compiled + uploaded; times kernels (+ bus sum)
  e2e              through the C ABI with HOST buffers: kgpu_plan_push_events(host events) +
                   kgpu_render(host_out): control simulation, H2D of events, kernels, D2H of audio
  parity           one UNTIMED step of the same workload rendered by the engine and by the CPU oracle
                   (threaded -O3 build, oracle/sharded.py): max |bus| and max |voice tap| differences
  bus_check        N > 1: the same step summed over peer memory and by an NCCL reduce of the rank-local
                   buses; the run fails above 1e-6
  other_workloads  N = 1: short device-resident runs of the other BASELINE configs, each against its own bound
  --impl reference the CPU oracle (C++ restatement of knaster's render path; knaster is Rust
                   and cannot be built in this image) on all host cores, bounded sample
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, BLOCK = 48000, 64
# SURVEY 8d: algorithmic ops per voice-sample (Envelope: 7 f64 + cvt in place of EnvAsr's 5 + scale)
W_FLOPS = {"subtractive": 40.0, "subtractive_seg": 42.0, "additive": 6.0, "fm": 15.0, "chain": 43.0}  # chain: + OnePoleLpf 3
N_SM, FP32_LANES, FP64_LANES, LDS_BANKS = 148, 128, 64, 32
F64_OPS_PER_SINF = 16
DEFAULT_VOICES = {"subtractive": 16384, "subtractive_seg": 16384, "additive": 4096, "fm": 8192, "chain": 16384}
WORKLOAD_NAMES = {
    "subtractive": "subtractive polysynth: saw -> SvfFilter lowpass -> EnvAsr -> VCA, sample-accurate note events",
    "subtractive_seg": "subtractive polysynth, Envelope variant: saw -> SvfFilter lowpass -> Envelope (A/D/R segments) -> VCA, sample-accurate note events",
    "additive": "additive bank: SinWt partials with per-partial amp smoothing",
    "fm": "FM bank: SinNumeric -> SinNumeric audio-rate freq",
    "chain": "a voice shape without a hand-written recipe: saw -> SvfFilter lowpass -> OnePoleLpf -> EnvAsr -> VCA, on the kernel generated for its template",
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    except OSError:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device=0):
        self.rows, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower() == "active":
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def shift_events(ev, frames):
    """Copy of an EVENT_DTYPE array with every absolute time moved `frames` later."""
    T = 282_240_000
    out = ev.copy()
    fr = out["seconds"].astype(np.uint64) * SR + (out["subsec"].astype(np.uint64) * SR) // T + np.uint64(frames)
    out["seconds"] = (fr // SR).astype(np.uint32)
    out["subsec"] = ((fr % SR) * T // SR).astype(np.uint32)
    return out


def bank_seed(workload, world):
    if workload in ("subtractive", "subtractive_seg"):
        return 2002 if world == 1 else 4004  # SURVEY 8d: configs[2] / configs[4]
    return None


def build_bank(graph, workload, voices, seconds, rank, world):
    """This rank's slice of the bank; returns (tap node id per voice, events)."""
    from knaster_b200.banks import bank_builder

    ids = bank_builder(workload, seconds, bank_seed(workload, world))(graph, voices, rank * voices, voices * world)
    return ids, graph.take_events()


def workload_config(args, world):
    """The workload, identically in both arms (the reference arm renders a bounded sample of it: see its
    `cpu_baseline.sample` / `sample_seconds_per_step`)."""
    return {"workload": WORKLOAD_NAMES[args.workload], "voices_per_gpu": args.voices, "total_voices": args.voices * world,
            "seconds_per_step": args.seconds, "blocks_per_step": int(round(args.seconds * SR)) // BLOCK, "block_size": BLOCK,
            "sample_rate": SR, "notes_per_voice_per_step": 8 if args.workload.startswith("subtractive") or args.workload == "chain" else 0,
            "l2": "per-voice state + events stream once per launch; working set changes every launch (no L2 reuse to flush)"}


# ------------------------------------------------------------------------------------------------
# --impl reference
def run_reference(args, rank, world):
    """--impl reference: the oracle (kind "port") on all host cores, bounded sample per step."""
    if rank != 0:
        return
    from oracle.sharded import ShardedOracle, bank_builder

    cores = os.cpu_count() or 1
    sample_seconds = min(args.seconds, args.ref_seconds)
    voices = args.voices  # one GPU's share of the bank
    n_blocks = int(round(sample_seconds * SR)) // BLOCK
    orc = ShardedOracle(bank_builder(args.workload, args.seconds, bank_seed(args.workload, 1)), voices, threads=cores)
    period = int(round(args.seconds * SR))
    window = n_blocks * BLOCK
    T = 282_240_000
    step = [0]

    def window_events(ev):
        # each step renders the NEXT `sample_seconds` of the bank (the oracle's clock runs on);
        # the 10 s event schedule repeats with period `--seconds`, exactly like the GPU arm's steps
        pos = step[0] * window
        e = shift_events(ev, (pos // period) * period)
        fr = e["seconds"].astype(np.uint64) * SR + (e["subsec"].astype(np.uint64) * SR) // T
        return e[(fr >= pos) & (fr < pos + window)]

    times = []
    for s in range(args.warmup + args.steps):
        step[0] = s
        t0 = time.perf_counter()
        bus, _ = orc.render(n_blocks, events_filter=window_events)  # voice-shard replicas summed at the end
        dt = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bus)
    ms = 1e3 * float(np.mean(times))
    value = voices * n_blocks * BLOCK / (ms / 1e3)
    sample = (f"{voices} voices x {sample_seconds:g} s of audio per step ({voices * n_blocks * BLOCK:.3g} voice-samples; the workload's "
              f"step is {args.seconds:g} s), voice-sharded over {len(orc.shards)} threads")
    line = {
        "impl": "reference", "metric": "voice-samples/sec (f32, 48 kHz)", "value": value, "unit": "voice-samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world),
        "sample_seconds_per_step": sample_seconds, "sample_voices": voices,
        "cpu_baseline": {"value": value, "unit": "voice-samples/s", "cores": len(orc.shards), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "voice-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "C++ restatement of knaster's CPU render path (oracle/); knaster itself is Rust and cannot be built here. "
                "knaster renders on ONE audio thread; the all-core figure is an upper bound it does not offer. ms_per_step is the "
                "time of the bounded sample (sample_seconds_per_step of audio for one GPU's share of the voices), not of a whole step.",
    }
    emit_json(line)


def cpu_baseline(args):
    """Oracle, single thread (the faithful figure: knaster renders on one audio thread), bounded sample."""
    from oracle.sharded import ShardedOracle, bank_builder

    voices = min(args.voices, args.cpu_voices)
    secs = min(args.seconds, args.cpu_seconds)
    orc = ShardedOracle(bank_builder(args.workload, secs, bank_seed(args.workload, 1)), voices, threads=1, total_voices=args.voices)
    n_blocks = int(round(secs * SR)) // BLOCK
    t0 = time.perf_counter()
    orc.render(n_blocks)
    dt = time.perf_counter() - t0
    return {"value": voices * n_blocks * BLOCK / dt, "unit": "voice-samples/s", "cores": 1, "kind": "port",
            "sample": f"first {voices} voices x first {secs:g} s of the same bank ({dt:.1f} s of CPU); C++ restatement of knaster's "
                      f"one-audio-thread render path (oracle/), host has {os.cpu_count()} cores"}


_JSON_FD = None


def emit_json(line) -> None:
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line
    to stdout when NCCL_DEBUG asks for it), so main() points fd 1 at stderr for the duration of the run
    and the result goes to the saved original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(dirname, bus) -> None:
    """--dump-outputs: the mix bus [n_blocks, outputs, block] of the last timed step as DIR/bus.npy (f32), so that two
    builds can be compared output for output.  A bus larger than DUMP_LIMIT_BYTES is cut to a fixed, seeded sample of
    whole blocks; their indices go to DIR/bus_blocks.npy (f64, exact for any block count)."""
    os.makedirs(dirname, exist_ok=True)
    bus = np.ascontiguousarray(bus, dtype=np.float32)
    n_blocks = bus.shape[0]
    keep = min(n_blocks, (DUMP_LIMIT_BYTES - 4096) // (bus[:1].nbytes + 8))  # + one f64 index per block, + .npy headers
    if keep < n_blocks:
        blocks = np.sort(np.random.Generator(np.random.PCG64(0)).choice(n_blocks, keep, replace=False))
        bus = bus[blocks]
        np.save(os.path.join(dirname, "bus_blocks.npy"), blocks.astype(np.float64))
    np.save(os.path.join(dirname, "bus.npy"), bus)


# ------------------------------------------------------------------------------------------------
# the GPU arm
class Env:
    """torch / torch.distributed plumbing shared by every measurement of a run."""

    def __init__(self, rank, world, local_rank):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank, self.world, self.local_rank = rank, world, local_rank
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        # one process per GPU shares the box's host cores: each plan's event-pipeline workers get their share
        self.host_threads = max(1, min(16, (os.cpu_count() or 1) // max(1, local_world) - 1))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


def make_processor(env, args, workload, voices, seconds, taps=()):
    from knaster_b200.processor import AudioProcessor, AudioProcessorOptions

    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(device=env.local_rank, force_interpreter=args.force_interpreter))
    t0 = time.perf_counter()
    ids, ev0 = build_bank(graph, workload, voices, seconds, env.rank, env.world)
    build_s = time.perf_counter() - t0
    for v in taps:
        proc.add_tap(ids[v], 0)
    info = proc.info()
    if args.blocks_per_launch:
        proc.set_blocks_per_launch(args.blocks_per_launch)
    proc.set_host_threads(args.host_threads or env.host_threads)
    return graph, proc, ev0, info, build_s


def attach_peer_bus(env, proc, n_blocks, want):
    """(PeerBus | None, mode): all ranks or none."""
    torch, dist = env.torch, env.dist
    if env.world == 1:
        return None, "none (1 GPU)"
    if not want:
        return None, "nccl"
    peer_bus = None
    try:
        from knaster_b200.multi_gpu import PeerBus

        peer_bus = PeerBus(proc, n_blocks)
        ok = torch.ones(1, device="cuda")
    except Exception as e:  # no symmetric memory / no peer access on this box
        sys.stderr.write(f"[bench] peer bus unavailable ({type(e).__name__}: {e}); using the NCCL reduce\n")
        ok = torch.zeros(1, device="cuda")
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if ok.item() < 1:
        if peer_bus is not None:
            peer_bus.close()
        return None, "nccl"
    return peer_bus, "peer"


def measure(env, args, workload, voices, seconds, steps, warmup, want_peer=True, with_e2e=True, sample_clocks=False, keep_output=False):
    """Device-resident `value` (+ optionally e2e) of one workload on this run's GPUs.  keep_output: res["bus"] is the
    mix bus of the last timed step, on the host."""
    from knaster_b200.multi_gpu import reduce_bus

    torch = env.torch
    world = env.world
    n_blocks = int(round(seconds * SR)) // BLOCK
    step_frames = n_blocks * BLOCK
    graph, proc, ev0, info, build_s = make_processor(env, args, workload, voices, seconds)
    step_no = [0]

    def push_step_events():
        graph.pending_event_arrays = [shift_events(ev0, step_no[0] * step_frames)] if len(ev0) else []
        step_no[0] += 1

    bus = torch.empty((n_blocks, 2, BLOCK), dtype=torch.float32, device="cuda")
    chunks = max(1, min(args.chunks, n_blocks)) if world > 1 else 1
    peer_bus, bus_mode = attach_peer_bus(env, proc, n_blocks, want_peer)

    def device_step():
        """kernels + mix-bus sum onto rank 0 (peer-memory stores inside the engine, or an NCCL reduce of
        the rank-local buses) with inputs already in HBM"""
        cur = torch.cuda.current_stream()
        proc.render_device(n_blocks, bus.data_ptr(), cur.cuda_stream)
        if peer_bus is None:
            reduce_bus(bus, dst=0, chunks=chunks)

    # ---- value: device-resident inputs.  Each step's events are compiled + uploaded (prepare)
    # outside the timed region, then K steps of kernels are timed back to back.
    for _ in range(warmup):
        push_step_events()
        proc.prepare(n_blocks)
        device_step()
    env.barrier()
    sampler = ClockSampler(env.local_rank) if sample_clocks else None
    if sampler:
        sampler.start()
    step_ms, kern_ms, red_ms, kern_launches, launches = [], 0.0, 0.0, 0, 0
    for _ in range(steps):
        push_step_events()
        proc.prepare(n_blocks)               # host work + H2D, outside the timed region
        env.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        device_step()
        e1.record()
        env.barrier()
        step_ms.append(e0.elapsed_time(e1))
        k, n = proc.last_kernel_ms(0)
        r, n2 = proc.last_kernel_ms(1)
        kern_ms += k; red_ms += r; kern_launches += n; launches += n + n2
    clocks = sampler.stop() if sampler else None
    total_ms = env.max_over_ranks(sum(step_ms))
    ms_per_step = total_ms / steps
    vs_per_step = voices * world * step_frames
    res = {"workload": workload, "voices": voices, "seconds": seconds, "steps": steps, "value": vs_per_step / (ms_per_step / 1e3),
           "ms_per_step": ms_per_step, "kern_ms": kern_ms, "red_ms": red_ms, "kern_launches": kern_launches, "launches": launches,
           "step_ms_sum": sum(step_ms), "clocks": clocks, "info": info, "build_s": build_s, "bus_mode": bus_mode, "chunks": chunks,
           "n_blocks": n_blocks, "step_frames": step_frames, "h2d": proc.last_upload_bytes()}
    if keep_output:
        res["bus"] = bus.cpu().numpy()  # before the e2e leg below: at N > 1 it renders into the same buffer

    # ---- e2e: through the C ABI with host buffers (rank-local; N>1: plus the bus sum)
    if with_e2e:
        host_out = np.empty((n_blocks, 2, BLOCK), dtype=np.float32)
        host_pin = None
        if world > 1 and env.rank == 0:
            # the summed bus comes down into page-locked host memory (bus.cpu() went through a fresh pageable tensor: ~1 ms per step)
            try:
                host_pin = torch.empty((n_blocks, 2, BLOCK), dtype=torch.float32, pin_memory=True)
                host_out = host_pin.numpy()
            except Exception:
                host_pin = None
        e2e_times, h2d = [], 0
        for i in range(1 + min(steps, 3)):
            push_step_events()
            env.barrier()
            t0 = time.perf_counter()
            if world == 1:
                proc.render(n_blocks, host_out)
            else:
                device_step()
                if env.rank == 0 and host_pin is not None:
                    host_pin.copy_(bus, non_blocking=True)  # on the stream the step ran on; complete after the synchronize
                    torch.cuda.synchronize()
                else:
                    torch.cuda.synchronize()
                    if env.rank == 0:
                        host_out[:] = bus.cpu().numpy()
            dt = time.perf_counter() - t0
            h2d = proc.last_upload_bytes()
            if i > 0:
                e2e_times.append(dt)
        t_e2e = env.max_over_ranks(float(np.mean(e2e_times)))
        res["e2e"] = {"value": vs_per_step / t_e2e, "unit": "voice-samples/s", "h2d_bytes_per_step": int(h2d),
                      "d2h_bytes_per_step": int(host_out.nbytes), "ms_per_step": 1e3 * t_e2e}
        res["h2d"] = h2d
    if peer_bus is not None and peer_bus.timed_out():
        sys.stderr.write("[bench] WARNING: a rank timed out waiting for peer-bus data\n")
        res["peer_timeout"] = True
    if peer_bus is not None:
        peer_bus.close()
    del proc
    return res


def roofline_of(res, peaks, peak_src):
    """Roofline of the dominant kernel of one measurement, against the bound that limits that workload."""
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    wl, voices = res["workload"], res["voices"]
    avg_launch_ms = res["kern_ms"] / max(1, res["kern_launches"])
    vs_per_launch = voices * res["step_frames"] * res["steps"] / max(1, res["kern_launches"])
    rate = vs_per_launch / (avg_launch_ms / 1e3)  # voice-samples/s of the render kernel(s) alone
    kernel = res["info"]["kernels"][0]
    if wl == "fm":
        # knaster's SinNumeric is libm's sinf (osc.rs:264): glibc evaluates it in f64 (reduction + degree-7 / degree-8 polynomial) and
        # so must the device, bit for bit -- 16 f64 operations per sine (csrc/sinf_glibc.h::kn_sinf_glibc_lean), 2 sines per voice-sample,
        # on a pipe that takes 16 lanes per SM sub-partition per cycle (measured: tools/microbench/fp64_bench.cu, 2.07 cycles per warp DFMA)
        peak = N_SM * FP64_LANES * sm_max * 1e6 / 1e9
        out = {"bound": "fp64", "achieved": rate * 2.0 * F64_OPS_PER_SINF / 1e9, "peak": peak,
               "unit": "G f64 instr/s (FP64 pipe; 16 per sinf, 2 sinf per voice-sample)",
               "peak_source": f"{N_SM} SMs x {FP64_LANES} FP64 lanes x sm_max_mhz {sm_max:g} ({peak_src})",
               "sinf_per_s": rate * 2.0,
               "fp32_frac": rate * W_FLOPS[wl] / 1e9 / (N_SM * FP32_LANES * sm_max * 1e6 / 1e9)}
    elif wl == "additive":
        # one 4-byte shared-memory table lookup per voice-sample: peak_lds = n_SM x 32 banks x f_SM (conflict-free)
        peak = N_SM * LDS_BANKS * sm_max * 1e6 / 1e9
        out = {"bound": "lds", "achieved": rate / 1e9, "peak": peak, "unit": "G 4-byte shared-memory lookups/s (conflict-free)",
               "peak_source": f"{N_SM} SMs x {LDS_BANKS} banks x sm_max_mhz {sm_max:g} ({peak_src}); random reads of a 64 KiB table "
                              "conflict 1.5-way (ncu r1c), which alone caps the fraction near 0.67"}
    else:
        peak = N_SM * FP32_LANES * sm_max * 1e6 / 1e9  # G un-fused FP32 instr/s
        out = {"bound": "fp32", "achieved": rate * W_FLOPS[wl] / 1e9, "peak": peak, "unit": "GFLOP/s (un-fused FP32 instr)",
               "flops_per_voice_sample": W_FLOPS[wl],
               "peak_source": f"{N_SM} SMs x {FP32_LANES} FP32 lanes x sm_max_mhz {sm_max:g} ({peak_src}); no tensor/HBM bound: "
                              "nothing here is a dense contraction and intermediates never touch HBM"}
    out["frac"] = out["achieved"] / out["peak"]
    if kernel == "render_sub_asr" and voices == 16384:
        # measured, not derived: profiles/r2_microbench_issue_mix.txt (tools/microbench/issue_mix.cu)
        out["formulation_ceiling"] = {"frac": 0.865 * 0.914, "why": "one lane per voice: 512 warps on 592 schedulers (0.865) x the issue rate of ONE warp "
                                      "on this kernel's FADD / FMUL / FFMA / FSET mix as independent chains (1.094 cycles per instruction, 0.914)",
                                      "frac_of_ceiling": out["frac"] / (0.865 * 0.914)}
    out.update({"kernel": kernel, "avg_launch_ms": avg_launch_ms, "launches": res["kern_launches"],
                "kernel_share_of_step": res["kern_ms"] / max(1e-9, res["step_ms_sum"]), "reduce_bus_ms_per_step": res["red_ms"] / res["steps"]})
    # HBM side: algorithmic bytes per launch (state in + out, events, per-warp partial rows) against the measured copy peak
    frames_per_launch = res["step_frames"] * res["steps"] / max(1, res["kern_launches"])
    rows = (voices + 31) // 32
    alg_bytes = 2 * res["info"]["state_bytes"] + (res["h2d"] / max(1, res["kern_launches"] / res["steps"])) + rows * frames_per_launch * 4
    hbm_gbs = alg_bytes / (avg_launch_ms / 1e3) / 1e9
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    out["hbm"] = {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak, "algorithmic_bytes_per_launch": alg_bytes}
    out["traffic"], out["traffic_source"] = None, None
    try:  # DRAM bytes of the dominant kernel from the committed ncu capture, scaled to this run's launch size
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)[kernel]
        if tj["voices"] == voices:
            out["traffic"] = tj["traffic_bytes_per_launch"] * frames_per_launch / tj["frames_per_launch"]
            out["traffic_source"] = f"{tj['source']} (ncu --set full capture of one launch, scaled by frames per launch; NOT measured in this run)"
    except (OSError, KeyError, ValueError, TypeError, ZeroDivisionError):  # a malformed record must not take the bench line down
        pass
    return out


def parity_and_bus_check(env, args, n_taps=64):
    """One UNTIMED step of the bench workload, from t = 0, on fresh processors:
       parity     rank 0's slice rendered by the engine (with >= 64 pre-mix voice taps) against the threaded oracle;
       bus_check  (N > 1) the whole bank's bus summed over peer memory against an NCCL reduce of the rank-local buses."""
    from knaster_b200.multi_gpu import reduce_bus
    from oracle.sharded import ShardedOracle, bank_builder, sample_voices

    torch, world, rank = env.torch, env.world, env.rank
    seconds = min(args.seconds, args.parity_seconds)
    n_blocks = int(round(seconds * SR)) // BLOCK
    voices = sample_voices(args.voices, n_taps)
    out = {}
    # (1) rank-local render with taps, host buffers
    graph, proc, ev0, info, _ = make_processor(env, args, args.workload, args.voices, args.seconds, taps=voices)
    graph.pending_event_arrays = [ev0.copy()] if len(ev0) else []
    local = proc.render(n_blocks)
    taps = proc.read_taps()
    del proc
    if rank == 0:
        t0 = time.perf_counter()
        orc = ShardedOracle(bank_builder(args.workload, args.seconds, bank_seed(args.workload, world)), args.voices, tap_voices=voices,
                            voice_offset=0, total_voices=args.voices * world)
        ref, ref_taps = orc.render(n_blocks)
        total = float(args.voices * world)  # every voice carries a gain of 1/total: tap errors are quoted at UNIT voice gain
        out["parity"] = {
            "max_abs_bus": float(np.abs(local - ref).max()), "max_abs_tap": float(np.abs(taps - ref_taps).max() * total),
            "max_abs_tap_last_second": float(np.abs(taps[:, -SR:] - ref_taps[:, -SR:]).max() * total),
            "taps_bit_identical": int((np.abs(taps - ref_taps).max(axis=1) == 0).sum()), "voices_checked": len(voices),
            "bus_voices": args.voices, "seconds": seconds, "peak_abs_bus": float(np.abs(ref).max()),
            "tap_scale": "differences of the pre-mix voice signal at unit voice gain (raw difference x total_voices)",
            "oracle": f"oracle/ -O3 build, {len(orc.shards)} threads, {time.perf_counter() - t0:.1f} s" + ("" if world == 1 else "; rank 0's slice of the bank, before the bus sum"),
            "tolerance": {"bus": 1e-5, "tap": 1e-4 if args.workload.startswith("subtractive") else 1e-5},
        }
    if world > 1:
        # (2) NCCL reduce of the rank-local buses, (3) the same step over the peer bus
        nccl = torch.from_numpy(local).cuda()
        reduce_bus(nccl, dst=0, chunks=1)
        graph, proc, ev0, _, _ = make_processor(env, args, args.workload, args.voices, args.seconds)
        peer_bus, mode = attach_peer_bus(env, proc, n_blocks, args.bus == "peer")
        if peer_bus is not None:
            graph.pending_event_arrays = [ev0.copy()] if len(ev0) else []
            bus = torch.zeros((n_blocks, 2, BLOCK), dtype=torch.float32, device="cuda")
            proc.render_device(n_blocks, bus.data_ptr(), torch.cuda.current_stream().cuda_stream)
            env.barrier()
            if rank == 0:
                out["bus_check"] = {"max_abs_peer_minus_nccl": float((bus - nccl).abs().max().item()), "peak_abs_bus": float(nccl.abs().max().item()),
                                    "seconds": seconds, "ranks": world, "timed_out": bool(peer_bus.timed_out()), "tolerance": 1e-6}
            peer_bus.close()
        elif rank == 0:
            out["bus_check"] = {"max_abs_peer_minus_nccl": None, "note": "peer bus unavailable on this box: the NCCL reduce is the only path"}
        del proc
        env.barrier()
    return out


def other_workloads(env, args, peaks, peak_src):
    """N = 1: the other BASELINE configs, 3 device-resident steps each, every one against its own bound."""
    out = {}
    for wl in ("additive", "fm", "subtractive_seg", "subtractive", "chain"):
        if wl == args.workload:
            continue
        r = measure(env, args, wl, DEFAULT_VOICES[wl], args.seconds, steps=3, warmup=3, with_e2e=True)
        rf = roofline_of(r, peaks, peak_src)
        out[wl] = {"config": WORKLOAD_NAMES[wl], "voices": r["voices"], "seconds_per_step": args.seconds, "value": r["value"], "unit": "voice-samples/s",
                   "ms_per_step": r["ms_per_step"], "e2e_value": r["e2e"]["value"], "e2e_ms_per_step": r["e2e"]["ms_per_step"],
                   "kernel": rf["kernel"], "bound": rf["bound"], "frac": rf["frac"], "achieved": rf["achieved"], "peak": rf["peak"], "roofline_unit": rf["unit"]}
    # configs[0], the README example: one SinWt voice * 0.2, 10 s, through the C ABI with the host copy included
    from knaster_b200 import banks
    from knaster_b200.processor import AudioProcessor, AudioProcessorOptions

    n_blocks = int(round(args.seconds * SR)) // BLOCK
    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions(device=env.local_rank))
    banks.readme_sine(graph)
    host = np.empty((n_blocks, 2, BLOCK), dtype=np.float32)
    times = []
    for i in range(6):
        t0 = time.perf_counter()
        proc.render(n_blocks, host)
        if i >= 3:
            times.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(times))
    out["readme"] = {"config": "README example: SinWt 440 Hz * 0.2 -> stereo, one voice", "voices": 1, "seconds_per_step": args.seconds,
                     "value": n_blocks * BLOCK / (ms / 1e3), "unit": "voice-samples/s", "ms_per_step": ms, "kernel": proc.info()["kernels"][0],
                     "bound": "launch latency (one voice; e2e through kgpu_render with the host copy)", "frac": None}
    return out


def main():
    global _JSON_FD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="subtractive", choices=["subtractive", "subtractive_seg", "additive", "fm", "chain"])
    ap.add_argument("--voices", type=int, default=0, help="voices per GPU (default: the BASELINE config's)")
    ap.add_argument("--seconds", type=float, default=10.0, help="audio seconds per step")
    ap.add_argument("--chunks", type=int, default=10, help="NCCL reduce chunks per step (N>1, --bus nccl)")
    ap.add_argument("--bus", default="peer", choices=["peer", "nccl"],
                    help="N>1: sum the mix bus over peer memory inside the engine's own kernels (falls back to nccl if torch "
                         "symmetric memory is unavailable) or with an NCCL reduce of the rank-local buses")
    ap.add_argument("--blocks-per-launch", type=int, default=0)
    ap.add_argument("--host-threads", type=int, default=0, help="event-pipeline worker threads per GPU (default: cores / GPUs - 1, at most 16)")
    ap.add_argument("--force-interpreter", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed parity step (and the N>1 bus check)")
    ap.add_argument("--no-other-workloads", action="store_true")
    ap.add_argument("--parity-seconds", type=float, default=10.0)
    ap.add_argument("--cpu-voices", type=int, default=4096)
    ap.add_argument("--cpu-seconds", type=float, default=4.0)
    ap.add_argument("--ref-seconds", type=float, default=1.0, help="--impl reference: audio seconds per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the mix bus of the last timed step to DIR/bus.npy (f32; over 64 MB a seeded sample of whole blocks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if not args.voices:
        args.voices = DEFAULT_VOICES[args.workload]
    sys.stdout.flush()
    _JSON_FD = os.dup(1)   # see emit_json
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    env = Env(rank, world, local_rank)
    # a non-default torch stream: its cudaStream_t is handed to the C ABI, so the engine's kernels,
    # the NCCL reduce and the torch.cuda.Event timers all live on the same stream
    torch.cuda.set_stream(torch.cuda.Stream())

    res = measure(env, args, args.workload, args.voices, args.seconds, args.steps, args.warmup, want_peer=args.bus == "peer", sample_clocks=True,
                  keep_output=bool(args.dump_outputs) and rank == 0)
    if args.dump_outputs and rank == 0:  # rank 0 holds the summed bus
        dump_outputs(args.dump_outputs, res.pop("bus"))
    checks = {} if args.no_parity else parity_and_bus_check(env, args)
    peaks, peak_src = measured_peaks()
    others = None
    if world == 1 and not args.no_other_workloads and args.workload == "subtractive":
        others = other_workloads(env, args, peaks, peak_src)

    failed = None
    if rank == 0:
        bus_mode, chunks = res["bus_mode"], res["chunks"]
        line = {
            "metric": "voice-samples/sec (f32, 48 kHz)", "value": res["value"], "unit": "voice-samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),
            "bus": ("peer memory: every rank's reduce_bus kernel stores its bus into rank 0 over NVLink, rank 0 folds the slots per launch"
                    if bus_mode == "peer" else f"NCCL reduce(sum) of the rank-local stereo bus to rank 0, {chunks} chunks per step"
                    if bus_mode == "nccl" else bus_mode),
            "kernels": res["info"]["kernels"],
            "roofline": roofline_of(res, peaks, peak_src),
            "e2e": res["e2e"],
            "gpu_launches": int(res["launches"]),
            "clocks": res["clocks"],
            "plan": {k: res["info"][k] for k in ("n_groups", "n_voices", "n_mix_nodes", "n_fused_groups", "state_bytes")},
            "build_graph_s": res["build_s"],
            "host": {"cores": os.cpu_count(), "event_pipeline_threads_per_gpu": args.host_threads or env.host_threads},
        }
        line.update(checks)
        if others is not None:
            line["other_workloads"] = others
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args)
        emit_json(line)
        par, bc = checks.get("parity"), checks.get("bus_check")
        if par and (par["max_abs_bus"] > par["tolerance"]["bus"] or par["max_abs_tap"] > par["tolerance"]["tap"]):
            failed = f"parity out of tolerance: {par}"
        if bc and bc.get("max_abs_peer_minus_nccl") is not None and (bc["max_abs_peer_minus_nccl"] > bc["tolerance"] or bc["timed_out"]):
            failed = f"bus_check failed: {bc}"
    if world > 1:
        dist.destroy_process_group()
    if failed:
        sys.stderr.write(f"[bench] FAILED: {failed}\n")
        sys.exit(3)


if __name__ == "__main__":
    main()
