"""ctypes binding of the C ABI in include/knaster_gpu.h (libknaster_gpu.so, built in-tree
from knaster_b200/csrc).  Loading fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import List, Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("KNASTER_GPU_LIB") or os.path.join(CSRC, "_build", "libknaster_gpu.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "knaster_gpu.h")

KGPU_ABI_VERSION = 1
KGPU_OK = 0
KGPU_ERR_INVALID, KGPU_ERR_UNSUPPORTED, KGPU_ERR_CUDA, KGPU_ERR_PARAMETER, KGPU_ERR_STATE = -1, -2, -3, -4, -5
KGPU_GRAPH = -2
KGPU_PLAN_FORCE_INTERPRETER = 1
KGPU_PLAN_NO_SCAN = 2
KGPU_PLAN_FORCE_JIT = 4


class KgpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"kgpu error {code}: {msg}")
        self.code = code
        self.msg = msg


class WrapperDesc(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("capacity", C.c_uint32), ("value", C.c_double)]


class NodeDesc(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("mode", C.c_uint32), ("channels", C.c_uint32), ("flags", C.c_uint32),
                ("args", C.c_double * 4), ("n_wrappers", C.c_uint32), ("n_segments", C.c_uint32),
                ("wrappers", C.POINTER(WrapperDesc)), ("segments", C.POINTER(C.c_double))]


class Edge(C.Structure):
    _fields_ = [("source_node", C.c_int32), ("source_channel", C.c_uint32), ("sink_node", C.c_int32),
                ("sink_channel", C.c_uint32)]


class ParamEdge(C.Structure):
    _fields_ = [("source_node", C.c_int32), ("source_channel", C.c_uint32), ("sink_node", C.c_int32),
                ("param_index", C.c_uint32)]


class GraphDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("sample_rate", C.c_uint32), ("block_size", C.c_uint32),
                ("n_inputs", C.c_uint32), ("n_outputs", C.c_uint32), ("device", C.c_int32),
                ("n_nodes", C.c_uint32), ("n_edges", C.c_uint32), ("n_param_edges", C.c_uint32),
                ("flags", C.c_uint32), ("nodes", C.POINTER(NodeDesc)), ("edges", C.POINTER(Edge)),
                ("param_edges", C.POINTER(ParamEdge))]


class PlanInfo(C.Structure):
    _fields_ = [("n_groups", C.c_uint32), ("n_voices", C.c_uint32), ("n_mix_nodes", C.c_uint32),
                ("n_fused_groups", C.c_uint32), ("state_bytes", C.c_uint64), ("dropped_changes", C.c_uint64),
                ("ignored_delays", C.c_uint64), ("device_events", C.c_uint64), ("kernel_launches", C.c_uint64)]

    def as_dict(self):
        return {f: int(getattr(self, f)) for f, _ in self._fields_}


class DebugEvent(C.Structure):
    _fields_ = [("group", C.c_uint32), ("voice", C.c_uint32), ("node", C.c_uint32), ("op", C.c_uint32),
                ("reg", C.c_uint32), ("value", C.c_uint32), ("frame", C.c_uint64)]


class DebugNode(C.Structure):
    _fields_ = [("group", C.c_int32), ("voice", C.c_uint32), ("local", C.c_uint32), ("reg_base", C.c_uint32)]


def build(verbose: bool = False) -> None:
    """Compile libknaster_gpu.so for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-j", str(min(8, os.cpu_count() or 1)), "-C", CSRC], capture_output=True, text=True)
    if verbose:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("building libknaster_gpu.so failed:\n" + r.stdout + r.stderr)


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(or `make -C knaster_b200/csrc`).  knaster_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
    L.kgpu_last_error.restype = C.c_char_p
    L.kgpu_abi_version.restype = u32
    L.kgpu_device_count.restype = C.c_int
    L.kgpu_plan_create.argtypes = [C.POINTER(GraphDesc), C.POINTER(vp)]
    L.kgpu_plan_destroy.argtypes = [vp]
    L.kgpu_plan_destroy.restype = None
    L.kgpu_plan_push_events.argtypes = [vp, vp, C.c_size_t]
    L.kgpu_render_block.argtypes = [vp]
    L.kgpu_output_block.argtypes = [vp]
    L.kgpu_output_block.restype = C.POINTER(C.c_float)
    L.kgpu_render.argtypes = [vp, u64, vp]
    L.kgpu_render_inputs.argtypes = [vp, u64, vp, vp]
    L.kgpu_render_device.argtypes = [vp, u64, vp, vp]
    L.kgpu_render_inputs_device.argtypes = [vp, u64, vp, vp, vp]
    L.kgpu_plan_synchronize.argtypes = [vp]
    L.kgpu_plan_block_size.argtypes = [vp]
    L.kgpu_plan_block_size.restype = u32
    L.kgpu_plan_outputs.argtypes = [vp]
    L.kgpu_plan_outputs.restype = u32
    L.kgpu_plan_frame_clock.argtypes = [vp]
    L.kgpu_plan_frame_clock.restype = u64
    L.kgpu_plan_add_tap.argtypes = [vp, u32, u32]
    L.kgpu_plan_read_taps.argtypes = [vp, vp, u64]
    L.kgpu_plan_get_info.argtypes = [vp, C.POINTER(PlanInfo)]
    L.kgpu_plan_group_kernel.argtypes = [vp, u32]
    L.kgpu_plan_group_kernel.restype = C.c_char_p
    L.kgpu_plan_last_render_ms.argtypes = [vp]
    L.kgpu_plan_last_render_ms.restype = C.c_float
    L.kgpu_plan_prepare.argtypes = [vp, u64]
    L.kgpu_plan_last_kernel_ms.argtypes = [vp, u32, C.POINTER(u32)]
    L.kgpu_plan_last_kernel_ms.restype = C.c_float
    L.kgpu_plan_last_upload_bytes.argtypes = [vp]
    L.kgpu_plan_last_upload_bytes.restype = u64
    L.kgpu_plan_set_blocks_per_launch.argtypes = [vp, u64]
    L.kgpu_plan_set_host_threads.argtypes = [vp, u32]
    L.kgpu_plan_snapshot.argtypes = [vp, C.POINTER(vp)]
    L.kgpu_plan_restore.argtypes = [vp, vp]
    L.kgpu_snapshot_destroy.argtypes = [vp]
    L.kgpu_snapshot_destroy.restype = None
    L.kgpu_snapshot_serialize.argtypes = [vp, vp, u64, C.POINTER(u64)]
    L.kgpu_snapshot_deserialize.argtypes = [vp, u64, C.POINTER(vp)]
    L.kgpu_plan_set_peer_bus.argtypes = [vp, u32, u32, vp, u64]
    L.kgpu_plan_peer_bus_timed_out.argtypes = [vp]
    L.kgpu_peer_bus_header_bytes.argtypes = [u32]
    L.kgpu_peer_bus_header_bytes.restype = u64
    L.kgpu_peer_bus_bytes.argtypes = [u32, u64]
    L.kgpu_peer_bus_bytes.restype = u64
    L.kgpu_debug_simulate.argtypes = [C.POINTER(GraphDesc), vp, C.c_size_t, u64, u64, vp, C.c_size_t,
                                      C.POINTER(C.c_size_t), vp, C.POINTER(PlanInfo)]
    L.kgpu_debug_init_reg.argtypes = [C.POINTER(GraphDesc), u32, u32, C.POINTER(u32)]
    L.kgpu_debug_jit_compile.argtypes = [C.POINTER(GraphDesc), u32, C.POINTER(u32), C.POINTER(u32)]
    L.kgpu_debug_jit_source.argtypes = [C.POINTER(GraphDesc), u32, C.c_char_p, u64, C.POINTER(u64)]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != KGPU_OK:
        raise KgpuError(rc, lib().kgpu_last_error().decode())


def graph_desc(graph, device: int = -1, flags: int = 0) -> Tuple[GraphDesc, list]:
    """Lower a knaster_b200.graph.Graph into a kgpu_graph_desc (+ keep-alive objects)."""
    keep: list = []
    ugens, in_edges, p_edges, o_edges = graph.lowered()
    nodes = (NodeDesc * max(1, len(ugens)))()
    for i, ug in enumerate(ugens):
        d = nodes[i]
        d.kind, d.mode, d.channels, d.flags = ug.kind, ug.mode, ug.channels, ug.flags
        for k, a in enumerate(ug.args[:4]):
            d.args[k] = a
        d.n_wrappers = len(ug.wrappers)
        if ug.wrappers:
            arr = (WrapperDesc * len(ug.wrappers))()
            for k, w in enumerate(ug.wrappers):
                arr[k].kind, arr[k].capacity, arr[k].value = w.kind, w.capacity, w.value
            keep.append(arr)
            d.wrappers = C.cast(arr, C.POINTER(WrapperDesc))
        d.n_segments = len(ug.segments)
        if ug.segments:
            flat = (C.c_double * (2 * len(ug.segments)))()
            for k, (du, va) in enumerate(ug.segments):
                flat[2 * k], flat[2 * k + 1] = du, va
            keep.append(flat)
            d.segments = C.cast(flat, C.POINTER(C.c_double))
    n_e = len(in_edges) + len(o_edges)
    edges = (Edge * max(1, n_e))()
    k = 0
    for (s, sc, sink, kc) in in_edges:
        edges[k].source_node, edges[k].source_channel, edges[k].sink_node, edges[k].sink_channel = s, sc, sink, kc
        k += 1
    for (s, sc, oc) in o_edges:
        edges[k].source_node, edges[k].source_channel, edges[k].sink_node, edges[k].sink_channel = s, sc, KGPU_GRAPH, oc
        k += 1
    pes = (ParamEdge * max(1, len(p_edges)))()
    for k, (s, sc, sink, p) in enumerate(p_edges):
        pes[k].source_node, pes[k].source_channel, pes[k].sink_node, pes[k].param_index = s, sc, sink, p
    gd = GraphDesc()
    gd.abi_version = KGPU_ABI_VERSION
    gd.sample_rate, gd.block_size = graph.sample_rate, graph.block_size
    gd.n_inputs, gd.n_outputs = graph.num_inputs, graph.num_outputs
    gd.device = device
    gd.n_nodes, gd.n_edges, gd.n_param_edges = len(ugens), n_e, len(p_edges)
    gd.flags = flags
    gd.nodes = C.cast(nodes, C.POINTER(NodeDesc))
    gd.edges = C.cast(edges, C.POINTER(Edge))
    gd.param_edges = C.cast(pes, C.POINTER(ParamEdge))
    keep += [nodes, edges, pes]
    return gd, keep


def debug_simulate(graph, events: np.ndarray, n_blocks: int, blocks_per_call: int = 0, cap: int = 1 << 20):
    """Host-only: run the plan + event compilers (no CUDA).  Returns (events, nodes, info)."""
    L = lib()
    gd, _keep = graph_desc(graph)
    out = (DebugEvent * cap)()
    nodes = (DebugNode * max(1, gd.n_nodes))()
    n = C.c_size_t(0)
    info = PlanInfo()
    ev = np.ascontiguousarray(events)
    check(L.kgpu_debug_simulate(C.byref(gd), ev.ctypes.data if len(ev) else None, len(ev), n_blocks, blocks_per_call,
                                C.cast(out, C.c_void_p), cap, C.byref(n), C.cast(nodes, C.c_void_p), C.byref(info)))
    evs = [(e.group, e.voice, e.node, e.op, e.reg, e.value, e.frame) for e in out[: n.value]]
    nds = [(d.group, d.voice, d.local, d.reg_base) for d in nodes[: gd.n_nodes]]
    return evs, nds, info.as_dict()


def jit_compile(graph, tap_outputs: bool = False):
    """Host-only: generate + compile (NVRTC -> the cubin cache next to the library; no GPU needed) the kernels of every voice
    template of `graph` that has no hand-written recipe.  Returns (generated, already cached)."""
    L = lib()
    gd, _keep = graph_desc(graph)
    a, b = C.c_uint32(0), C.c_uint32(0)
    check(L.kgpu_debug_jit_compile(C.byref(gd), 1 if tap_outputs else 0, C.byref(a), C.byref(b)))
    return a.value, b.value


def jit_source(graph, tap_outputs: bool = False) -> List[str]:
    """Host-only: the CUDA source generated for every voice template of `graph` that has no hand-written recipe (no NVRTC)."""
    L = lib()
    gd, _keep = graph_desc(graph)
    n = C.c_uint64(0)
    check(L.kgpu_debug_jit_source(C.byref(gd), 1 if tap_outputs else 0, None, 0, C.byref(n)))
    buf = C.create_string_buffer(n.value)
    check(L.kgpu_debug_jit_source(C.byref(gd), 1 if tap_outputs else 0, buf, n.value, C.byref(n)))
    return buf.raw[: n.value].decode().split("\n// ---- end of template\n")[:-1]
