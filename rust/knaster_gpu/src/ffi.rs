// NOT COMPILED IN THIS REPOSITORY'S IMAGE (no cargo/rustc, SURVEY F2).  The text of INTEGRATION.md as files:
// the binding a knaster maintainer would add next to knaster_graph.  tests/test_host_plan.py checks that
// src/ffi.rs declares every entry point of include/knaster_gpu.h.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct kgpu_wrapper_desc { pub kind: u32, pub capacity: u32, pub value: f64 }
#[repr(C)] pub struct kgpu_node_desc {
    pub kind: u32, pub mode: u32, pub channels: u32, pub flags: u32, pub args: [f64; 4],
    pub n_wrappers: u32, pub n_segments: u32,
    pub wrappers: *const kgpu_wrapper_desc, pub segments: *const f64,
}
#[repr(C)] pub struct kgpu_edge { pub source_node: i32, pub source_channel: u32, pub sink_node: i32, pub sink_channel: u32 }
#[repr(C)] pub struct kgpu_param_edge { pub source_node: i32, pub source_channel: u32, pub sink_node: i32, pub param_index: u32 }
#[repr(C)] pub struct kgpu_graph_desc {
    pub abi_version: u32, pub sample_rate: u32, pub block_size: u32, pub n_inputs: u32, pub n_outputs: u32,
    pub device: i32, pub n_nodes: u32, pub n_edges: u32, pub n_param_edges: u32, pub flags: u32,
    pub nodes: *const kgpu_node_desc, pub edges: *const kgpu_edge, pub param_edges: *const kgpu_param_edge,
}
#[repr(C)] pub struct kgpu_event {
    pub node: u32, pub param: u32, pub value_kind: u32, pub smoothing_kind: u32, pub value: f64,
    pub smooth_seconds: f32, pub smooth_rate: u32, pub time_kind: u32, pub seconds: u32, pub subsec: u32, pub _pad: u32,
}
#[repr(C)] #[derive(Default)] pub struct kgpu_plan_info {
    pub n_groups: u32, pub n_voices: u32, pub n_mix_nodes: u32, pub n_fused_groups: u32, pub state_bytes: u64,
    pub dropped_changes: u64, pub ignored_delays: u64, pub device_events: u64, pub kernel_launches: u64,
}
#[repr(C)] pub struct kgpu_plan { _private: [u8; 0] }
#[repr(C)] pub struct kgpu_snapshot { _private: [u8; 0] }

extern "C" {
    pub fn kgpu_plan_create(desc: *const kgpu_graph_desc, out: *mut *mut kgpu_plan) -> c_int;
    pub fn kgpu_plan_destroy(plan: *mut kgpu_plan);
    pub fn kgpu_plan_push_events(plan: *mut kgpu_plan, events: *const kgpu_event, n: usize) -> c_int;
    pub fn kgpu_render_block(plan: *mut kgpu_plan) -> c_int;
    pub fn kgpu_output_block(plan: *mut kgpu_plan) -> *const f32;
    pub fn kgpu_render(plan: *mut kgpu_plan, n_blocks: u64, host_out: *mut f32) -> c_int;
    pub fn kgpu_render_inputs(plan: *mut kgpu_plan, n_blocks: u64, host_in: *const f32, host_out: *mut f32) -> c_int;
    pub fn kgpu_render_device(plan: *mut kgpu_plan, n_blocks: u64, device_out: *mut f32, cuda_stream: *mut c_void) -> c_int;
    pub fn kgpu_render_inputs_device(plan: *mut kgpu_plan, n_blocks: u64, device_in: *const f32, device_out: *mut f32,
                                     cuda_stream: *mut c_void) -> c_int;
    pub fn kgpu_plan_prepare(plan: *mut kgpu_plan, n_blocks: u64) -> c_int;
    pub fn kgpu_plan_synchronize(plan: *mut kgpu_plan) -> c_int;
    pub fn kgpu_plan_block_size(plan: *const kgpu_plan) -> u32;
    pub fn kgpu_plan_outputs(plan: *const kgpu_plan) -> u32;
    pub fn kgpu_plan_frame_clock(plan: *const kgpu_plan) -> u64;
    pub fn kgpu_plan_add_tap(plan: *mut kgpu_plan, node: u32, channel: u32) -> c_int;
    pub fn kgpu_plan_read_taps(plan: *mut kgpu_plan, out: *mut f32, n_frames: u64) -> c_int;
    pub fn kgpu_plan_set_host_threads(plan: *mut kgpu_plan, n_threads: u32) -> c_int;
    pub fn kgpu_plan_set_blocks_per_launch(plan: *mut kgpu_plan, blocks: u64) -> c_int;
    // multi-GPU (one GpuProcessor per device): the mix bus over peer memory
    pub fn kgpu_peer_bus_bytes(world: u32, floats_per_rank: u64) -> u64;
    pub fn kgpu_plan_set_peer_bus(plan: *mut kgpu_plan, rank: u32, world: u32, root_buffer: *mut c_void, buffer_bytes: u64) -> c_int;
    pub fn kgpu_plan_peer_bus_timed_out(plan: *mut kgpu_plan) -> c_int;
    // snapshot / restore of the whole render state
    pub fn kgpu_plan_snapshot(plan: *mut kgpu_plan, out: *mut *mut kgpu_snapshot) -> c_int;
    pub fn kgpu_plan_restore(plan: *mut kgpu_plan, snapshot: *const kgpu_snapshot) -> c_int;
    pub fn kgpu_snapshot_destroy(snapshot: *mut kgpu_snapshot);
    pub fn kgpu_snapshot_serialize(snapshot: *const kgpu_snapshot, buf: *mut c_void, cap: u64, size: *mut u64) -> c_int;
    pub fn kgpu_snapshot_deserialize(buf: *const c_void, size: u64, out: *mut *mut kgpu_snapshot) -> c_int;
    // introspection / measurement
    pub fn kgpu_plan_get_info(plan: *mut kgpu_plan, info: *mut kgpu_plan_info) -> c_int;
    pub fn kgpu_plan_group_kernel(plan: *mut kgpu_plan, group: u32) -> *const c_char;
    pub fn kgpu_plan_last_render_ms(plan: *mut kgpu_plan) -> f32;
    pub fn kgpu_plan_last_kernel_ms(plan: *mut kgpu_plan, kernel_class: u32, n_launches: *mut u32) -> f32;
    pub fn kgpu_plan_last_upload_bytes(plan: *mut kgpu_plan) -> u64;
    pub fn kgpu_peer_bus_header_bytes(world: u32) -> u64;
    pub fn kgpu_last_error() -> *const c_char;
    pub fn kgpu_abi_version() -> u32;
    pub fn kgpu_device_count() -> c_int;
}
