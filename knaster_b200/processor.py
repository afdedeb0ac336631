"""``AudioProcessor``: the render surface of the drop-in boundary
(knaster_graph/src/processor.rs:23-197), backed by the CUDA engine.

    graph, proc = AudioProcessor.new(0, 2, AudioProcessorOptions())   # new::<U0, U2>(options)
    with graph.edit() as g: ...
    proc.run_without_inputs(); block = proc.output_block()            # [outputs][block_size]

plus the batched calls a non-realtime render actually wants: ``render(n_blocks)`` and
``render_device(n_blocks, out_ptr, stream)``.  The graph must be static once rendering
has started (SURVEY section 2: dynamic editing while running is out of scope).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import _ffi
from .graph import Graph, GraphError


@dataclass
class AudioProcessorOptions:
    """processor.rs:23-45 (+ the CUDA device to render on)."""

    block_size: int = 64
    sample_rate: int = 48000
    ring_buffer_size: int = 1000      # kept for source compatibility; the engine never drops events
    log_channel_capacity: int = 100   # kept for source compatibility
    device: int = -1                  # CUDA device ordinal, -1 = current
    force_interpreter: bool = False   # render with the generic plan interpreter only
    force_jit: bool = False           # generate a kernel per voice template even for small banks (default: >= 256 voices)
    no_scan: bool = False             # small saw -> SVF -> EnvAsr banks: bit-exact one-lane-per-voice kernel instead of the scan kernel


class AudioProcessor:
    def __init__(self, graph: Graph, options: AudioProcessorOptions):
        self._lib = _ffi.lib()  # fails loudly if the CUDA library is missing
        self.graph = graph
        self.options = options
        self._plan = C.c_void_p(None)
        self._plan_version = -1
        self._started = False
        self._taps: List[Tuple[int, int]] = []
        self._last_render_frames = 0

    @staticmethod
    def new(inputs: int, outputs: int, options: Optional[AudioProcessorOptions] = None):
        """``AudioProcessor::<f32>::new::<Inputs, Outputs>(options)`` (processor.rs:69-116).
        Returns (graph, audio_processor); knaster's third element, the RT log receiver, has no
        counterpart: errors are returned, not logged (SURVEY section 5)."""
        options = options or AudioProcessorOptions()
        if options.block_size == 0:
            raise GraphError("The block size must not be 0")  # processor.rs:75
        if outputs == 0:
            raise GraphError("Outputs must be non-zero")       # Outputs: Size + NonZero
        graph = Graph(inputs, outputs, options.block_size, options.sample_rate)
        return graph, AudioProcessor(graph, options)

    def __del__(self):
        try:
            if self._plan:
                self._lib.kgpu_plan_destroy(self._plan)
                self._plan = C.c_void_p(None)
        except Exception:
            pass

    # -- plan management: Graph::commit_changes -> kgpu_plan_create
    def _ensure_plan(self) -> None:
        g = self.graph
        g.commit_changes()
        if self._plan and self._plan_version == g.version:
            return
        if self._started:
            raise GraphError("the graph was edited after rendering started: the GPU engine renders static graphs only")
        if self._plan:
            self._lib.kgpu_plan_destroy(self._plan)
            self._plan = C.c_void_p(None)
        flags = _ffi.KGPU_PLAN_FORCE_INTERPRETER if self.options.force_interpreter else 0
        if self.options.no_scan:
            flags |= _ffi.KGPU_PLAN_NO_SCAN
        if self.options.force_jit:
            flags |= _ffi.KGPU_PLAN_FORCE_JIT
        gd, _keep = _ffi.graph_desc(g, self.options.device, flags)
        plan = C.c_void_p(None)
        _ffi.check(self._lib.kgpu_plan_create(C.byref(gd), C.byref(plan)))
        self._plan = plan
        self._plan_version = g.version
        for (node, ch) in self._taps:
            rc = self._lib.kgpu_plan_add_tap(self._plan, node, ch)
            if rc < 0:
                _ffi.check(rc)

    def _push_events(self) -> None:
        ev = self.graph.take_events()
        if len(ev):
            _ffi.check(self._lib.kgpu_plan_push_events(self._plan, ev.ctypes.data, len(ev)))

    # -- processor.rs:119-197
    def run_without_inputs(self) -> None:
        if self.inputs() != 0:
            raise GraphError("run_without_inputs on a graph with inputs")  # processor.rs:143
        self._ensure_plan()
        self._push_events()
        self._started = True
        _ffi.check(self._lib.kgpu_render_block(self._plan))
        self._last_render_frames = self.block_size()   # read_taps() returns this block's frames

    def run(self, inputs) -> None:
        """``AudioProcessor::run(&[&[F]])`` (processor.rs:119-141): one block, one slice of block_size samples per graph input."""
        if len(inputs) != self.inputs():
            raise GraphError("wrong number of input channels")  # processor.rs:120
        if self.inputs() == 0:
            self.run_without_inputs()
            return
        blk = np.stack([np.ascontiguousarray(x, dtype=np.float32).reshape(self.block_size()) for x in inputs])[None]
        self.render(1, inputs=blk)

    def output_block(self) -> np.ndarray:
        """[outputs][block_size] copy of the last rendered block (processor.rs:182-184)."""
        if not self._plan:
            return np.zeros((self.outputs(), self.block_size()), dtype=np.float32)
        p = self._lib.kgpu_output_block(self._plan)
        return np.ctypeslib.as_array(p, shape=(self.outputs(), self.block_size())).copy()

    def block_size(self) -> int:
        return self.options.block_size

    def inputs(self) -> int:
        return self.graph.num_inputs

    def outputs(self) -> int:
        return self.graph.num_outputs

    def frame_clock(self) -> int:
        return int(self._lib.kgpu_plan_frame_clock(self._plan)) if self._plan else 0

    # -- batched rendering
    def render(self, n_blocks: int, out: Optional[np.ndarray] = None, inputs: Optional[np.ndarray] = None) -> np.ndarray:
        """Render n_blocks; returns host audio [n_blocks][outputs][block_size].  inputs: [n_blocks][graph inputs][block_size]
        for a graph with inputs (the batched form of ``run``)."""
        self._ensure_plan()
        self._push_events()
        self._started = True
        if out is None:
            out = np.empty((n_blocks, self.outputs(), self.block_size()), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags["C_CONTIGUOUS"] and out.size == n_blocks * self.outputs() * self.block_size()
        if inputs is not None:
            inp = np.ascontiguousarray(inputs, dtype=np.float32)
            if inp.shape != (n_blocks, self.inputs(), self.block_size()):
                raise GraphError("inputs must be [n_blocks][graph inputs][block_size]")
            _ffi.check(self._lib.kgpu_render_inputs(self._plan, n_blocks, inp.ctypes.data, out.ctypes.data))
            self._last_render_frames = n_blocks * self.block_size()
            return out
        _ffi.check(self._lib.kgpu_render(self._plan, n_blocks, out.ctypes.data))
        self._last_render_frames = n_blocks * self.block_size()
        return out

    def render_device(self, n_blocks: int, device_ptr: int, stream: int = 0) -> None:
        """Render into device memory (n_blocks*outputs*block_size floats at device_ptr), enqueued
        on `stream` (cudaStream_t as int, 0 = the plan's own stream), without synchronising."""
        self._ensure_plan()
        self._push_events()
        self._started = True
        _ffi.check(self._lib.kgpu_render_device(self._plan, n_blocks, C.c_void_p(device_ptr), C.c_void_p(stream)))
        self._last_render_frames = n_blocks * self.block_size()

    def synchronize(self) -> None:
        if self._plan:
            _ffi.check(self._lib.kgpu_plan_synchronize(self._plan))

    # -- parity / debug
    def add_tap(self, node, channel: int = 0) -> int:
        """Record `channel` of `node` (pre-mix) on every render; call before the first render."""
        node = int(node)
        self._taps.append((node, channel))
        if self._plan and self._plan_version == self.graph.version:
            rc = self._lib.kgpu_plan_add_tap(self._plan, node, channel)
            if rc < 0:
                _ffi.check(rc)
        return len(self._taps) - 1

    def read_taps(self) -> np.ndarray:
        """[n_taps][frames of the last render]"""
        out = np.empty((len(self._taps), self._last_render_frames), dtype=np.float32)
        _ffi.check(self._lib.kgpu_plan_read_taps(self._plan, out.ctypes.data, self._last_render_frames))
        return out

    def info(self) -> dict:
        self._ensure_plan()
        info = _ffi.PlanInfo()
        _ffi.check(self._lib.kgpu_plan_get_info(self._plan, C.byref(info)))
        d = info.as_dict()
        d["kernels"] = [self._lib.kgpu_plan_group_kernel(self._plan, i).decode() for i in range(d["n_groups"])]
        return d

    def prepare(self, n_blocks: int) -> None:
        """Do the host half of the next render(n_blocks) now (event simulation + upload)."""
        self._ensure_plan()
        self._push_events()
        _ffi.check(self._lib.kgpu_plan_prepare(self._plan, n_blocks))

    def last_kernel_ms(self, kernel_class: int = 0):
        """(total ms, launches) of the last render call for kernel class 0 (voice banks) / 1 (reduce_bus)."""
        n = C.c_uint32(0)
        ms = float(self._lib.kgpu_plan_last_kernel_ms(self._plan, kernel_class, C.byref(n)))
        return ms, int(n.value)

    def last_upload_bytes(self) -> int:
        return int(self._lib.kgpu_plan_last_upload_bytes(self._plan))

    def set_blocks_per_launch(self, blocks: int) -> None:
        self._ensure_plan()
        _ffi.check(self._lib.kgpu_plan_set_blocks_per_launch(self._plan, blocks))

    def set_peer_bus(self, rank: int, world: int, root_buffer_ptr: int, nbytes: int) -> None:
        """Attach (or, with world <= 1, detach) the multi-GPU mix bus over peer memory."""
        self._ensure_plan()
        _ffi.check(self._lib.kgpu_plan_set_peer_bus(self._plan, rank, world, C.c_void_p(root_buffer_ptr or None), nbytes))

    def peer_bus_timed_out(self) -> bool:
        return bool(self._plan) and int(self._lib.kgpu_plan_peer_bus_timed_out(self._plan)) != 0

    def snapshot(self) -> "Snapshot":
        """Copy of the whole render state (voice registers, control-side state, queued events, frame clock):
        ``restore()`` rewinds the processor to it.  Events must be pushed first, so the graph's pending ones are."""
        self._ensure_plan()
        self._push_events()
        h = C.c_void_p()
        _ffi.check(self._lib.kgpu_plan_snapshot(self._plan, C.byref(h)))
        return Snapshot(self._lib, h)

    def restore(self, snap: "Snapshot") -> None:
        self._ensure_plan()
        self._push_events()          # what the graph still holds belongs to "before the restore": queued, then discarded
        _ffi.check(self._lib.kgpu_plan_restore(self._plan, snap._h))

    def set_host_threads(self, n_threads: int) -> None:
        """Worker threads of the host event pipeline (0 = hardware threads - 1, at most 16)."""
        self._ensure_plan()
        _ffi.check(self._lib.kgpu_plan_set_host_threads(self._plan, n_threads))

    def last_render_ms(self) -> float:
        return float(self._lib.kgpu_plan_last_render_ms(self._plan))


class Snapshot:
    """Owner of a ``kgpu_snapshot`` (include/knaster_gpu.h)."""

    def __init__(self, lib, handle):
        self._lib, self._h = lib, handle

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.kgpu_snapshot_destroy(self._h)
            self._h = None

    def to_bytes(self) -> bytes:
        """The snapshot as a flat byte image (kgpu_snapshot_serialize): a checkpoint that can be written to disk."""
        n = C.c_uint64(0)
        _ffi.check(self._lib.kgpu_snapshot_serialize(self._h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        _ffi.check(self._lib.kgpu_snapshot_serialize(self._h, buf, n.value, C.byref(n)))
        return buf.raw[: n.value]

    @staticmethod
    def from_bytes(data: bytes) -> "Snapshot":
        lib = _ffi.lib()
        h = C.c_void_p()
        _ffi.check(lib.kgpu_snapshot_deserialize(data, len(data), C.byref(h)))
        return Snapshot(lib, h)
