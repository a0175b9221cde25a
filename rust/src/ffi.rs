//! `extern "C"` binding of include/mdim.h (ABI version 1).  UNVERIFIED — see rust/README.md.
//! Field-for-field with `mdim_node` / `mdim_expr` / `mdim_error_info`; the Python binding
//! (multidimension_b200/_ffi.py) is the same table and IS checked against the C compiler's sizeof.
#![allow(non_camel_case_types, dead_code)]
use core::ffi::{c_char, c_void};

#[repr(C)] pub struct MdimCtx { _private: [u8; 0] }

pub const MDIM_ABI_VERSION: i32 = 1;
pub const MDIM_MAX_RANK: usize = 8;
pub const MDIM_MAX_NODES: usize = 48;
pub const MDIM_MAX_PEERS: usize = 8;
pub const MDIM_COMM_ID_BYTES: usize = 128;

// mdim_status: every reference panic site maps to one of these
pub const MDIM_OK: i32 = 0;
pub const MDIM_ERR_OOB: i32 = 1;          // src/int.rs:17
pub const MDIM_ERR_SIZE: i32 = 2;         // src/array.rs:12, src/broadcast.rs:38
pub const MDIM_ERR_UNSUPPORTED: i32 = 3;
pub const MDIM_ERR_CUDA: i32 = 4;
pub const MDIM_ERR_ARITH: i32 = 5;
pub const MDIM_ERR_INVALID: i32 = 6;
pub const MDIM_ERR_NOMEM: i32 = 7;
pub const MDIM_ERR_NCCL: i32 = 8;

// mdim_dtype (usize = U64, bool = U8)
pub const U8: i32 = 0; pub const I32: i32 = 1; pub const U32: i32 = 2; pub const I64: i32 = 3;
pub const U64: i32 = 4; pub const F32: i32 = 5; pub const F64: i32 = 6;
pub const I8: i32 = 7; pub const I16: i32 = 8; pub const U16: i32 = 9;
// mdim_binary_op = the enums of src/ops.rs:23-129
pub const ADD: i32 = 0; pub const SUB: i32 = 1; pub const MUL: i32 = 2; pub const DIV: i32 = 3; pub const REM: i32 = 4;
pub const AND: i32 = 5; pub const OR: i32 = 6; pub const XOR: i32 = 7; pub const SHL: i32 = 8; pub const SHR: i32 = 9;
pub const REDUCE_MIN: i32 = 100; pub const REDUCE_MAX: i32 = 101;
// mdim_unary_op
pub const NEG: i32 = 0; pub const NOT: i32 = 1; pub const ABS: i32 = 2; pub const SQRT: i32 = 3; pub const CAST: i32 = 4;
// mdim_node_kind
pub const LEAF: i32 = 0; pub const IOTA: i32 = 1; pub const CONST: i32 = 2; pub const UNARY: i32 = 3; pub const BINARY: i32 = 4;
pub const DIAG: i32 = 5; pub const GATHER: i32 = 6; pub const FOLD: i32 = 7; pub const CONCAT: i32 = 8;

pub const COLLECT_ASYNC: u32 = 1; pub const COLLECT_NO_FASTPATH: u32 = 2; pub const COLLECT_NO_STATIC: u32 = 4; pub const COLLECT_NO_JIT: u32 = 8;

#[repr(C)] #[derive(Copy, Clone)]
pub union MdimScalar { pub u64_: u64, pub i64_: i64, pub f64_: f64, pub f32_: f32, pub u32_: u32, pub i32_: i32, pub u8_: u8, pub i8_: i8, pub i16_: i16, pub u16_: u16 }

#[repr(C)] #[derive(Copy, Clone)]
pub struct MdimNode {
    pub kind: i32, pub dtype: i32, pub op: i32, pub n_comp: i32, pub src_dtype: i32, pub n_peers: i32,
    pub data: *const c_void, pub offset: i64,
    pub stride: [i64; MDIM_MAX_RANK], pub gstride: [i64; MDIM_MAX_RANK], pub bound: [u64; MDIM_MAX_RANK],
    pub axis_a: [i32; MDIM_MAX_RANK], pub axis_b: [i32; MDIM_MAX_RANK], pub axis_c: [u64; MDIM_MAX_RANK],
    pub imm: MdimScalar, pub peer: [*const c_void; MDIM_MAX_PEERS], pub peer_block: u64,
}

impl MdimNode {
    pub fn zeroed() -> Self { unsafe { core::mem::zeroed() } }
}

#[repr(C)]
pub struct MdimExpr {
    pub abi_version: i32, pub rank: i32, pub red_rank: i32, pub n_nodes: i32,
    pub length: [u64; MDIM_MAX_RANK], pub nodes: *const MdimNode,
}

#[repr(C)]
pub struct MdimErrorInfo {
    pub status: i32, pub node: i32, pub position: u64, pub value: u64, pub bound: u64,
    pub component: i32, pub reserved: i32, pub message: [c_char; 160],
}

#[link(name = "mdim_b200")]
extern "C" {
    pub fn mdim_abi_version() -> i32;
    pub fn mdim_init(device: i32, ctx: *mut *mut MdimCtx) -> i32;
    pub fn mdim_shutdown(ctx: *mut MdimCtx) -> i32;
    pub fn mdim_set_stream(ctx: *mut MdimCtx, cuda_stream: *mut c_void) -> i32;
    pub fn mdim_get_stream(ctx: *mut MdimCtx, cuda_stream: *mut *mut c_void) -> i32;
    pub fn mdim_sync(ctx: *mut MdimCtx) -> i32;
    pub fn mdim_last_error(ctx: *mut MdimCtx, info: *mut MdimErrorInfo) -> i32;
    pub fn mdim_status_string(status: i32) -> *const c_char;
    pub fn mdim_launch_count(ctx: *mut MdimCtx) -> u64;
    pub fn mdim_last_kernel(ctx: *mut MdimCtx, buf: *mut c_char, buf_len: usize) -> i32;
    pub fn mdim_device_info(ctx: *mut MdimCtx, sm_count: *mut i32, cc_major: *mut i32, cc_minor: *mut i32, hbm_bytes: *mut usize) -> i32;
    // the device-resident Box<[T]> of Array (src/array.rs:5-8)
    pub fn mdim_buf_alloc(ctx: *mut MdimCtx, bytes: usize, dptr: *mut *mut c_void) -> i32;
    pub fn mdim_buf_free(ctx: *mut MdimCtx, dptr: *mut c_void) -> i32;
    pub fn mdim_upload(ctx: *mut MdimCtx, dst_device: *mut c_void, src_host: *const c_void, bytes: usize) -> i32;
    pub fn mdim_download(ctx: *mut MdimCtx, dst_host: *mut c_void, src_device: *const c_void, bytes: usize) -> i32;
    pub fn mdim_host_alloc(ctx: *mut MdimCtx, bytes: usize, hptr: *mut *mut c_void) -> i32;
    pub fn mdim_host_free(ctx: *mut MdimCtx, hptr: *mut c_void) -> i32;
    // View::collect (src/view.rs:146-150)
    pub fn mdim_collect(ctx: *mut MdimCtx, e: *const MdimExpr, out_device: *mut c_void, flags: u32) -> i32;
    pub fn mdim_collect_host(ctx: *mut MdimCtx, e: *const MdimExpr, out_host: *mut c_void, flags: u32) -> i32;
    pub fn mdim_plan_describe_nodevice(e: *const MdimExpr, flags: u32, buf: *mut c_char, buf_len: usize) -> i32;
    // several GPUs, one process each (SURVEY.md §8e)
    pub fn mdim_comm_unique_id(id: *mut u8) -> i32;
    pub fn mdim_comm_init(ctx: *mut MdimCtx, rank: i32, world: i32, id: *const u8) -> i32;
    pub fn mdim_comm_destroy(ctx: *mut MdimCtx) -> i32;
    pub fn mdim_comm_info(ctx: *mut MdimCtx, rank: *mut i32, world: *mut i32, nccl_version: *mut i32) -> i32;
    pub fn mdim_allgather(ctx: *mut MdimCtx, send_device: *const c_void, recv_device: *mut c_void, block_bytes: usize) -> i32;
    pub fn mdim_allreduce(ctx: *mut MdimCtx, data_device: *mut c_void, n: usize, dtype: i32, op: i32) -> i32;
    pub fn mdim_barrier(ctx: *mut MdimCtx) -> i32;
    pub fn mdim_peer_table(ctx: *mut MdimCtx, local_device: *mut c_void, block_bytes: usize, peers: *mut *mut c_void) -> i32;
    pub fn mdim_peer_table_close(ctx: *mut MdimCtx) -> i32;
    // fold over the sharded (outermost) axis as one fused compute + exchange kernel per GPU: the reference's sequential chain through the
    // ranks (bit-exact), and per-rank partial folds combined in rank order inside the kernel (the all-reduce route, no NCCL call)
    pub fn mdim_fold_sharded_axis(ctx: *mut MdimCtx, local_rows: *const c_void, n_rows_local: u64, n_cols: u64, dtype: i32, op: i32, init: MdimScalar, out_device: *mut c_void) -> i32;
    pub fn mdim_fold_sharded_axis_blocked(ctx: *mut MdimCtx, local_rows: *const c_void, n_rows_local: u64, n_cols: u64, dtype: i32, op: i32, init: MdimScalar, out_device: *mut c_void) -> i32;
    pub fn mdim_fold_sharded_axis_status(ctx: *mut MdimCtx) -> i32;
    pub fn mdim_ipc_export(ctx: *mut MdimCtx, dptr: *mut c_void, handle: *mut u8) -> i32;
    pub fn mdim_ipc_open(ctx: *mut MdimCtx, handle: *const u8, dptr: *mut *mut c_void) -> i32;
    pub fn mdim_ipc_close(ctx: *mut MdimCtx, dptr: *mut c_void) -> i32;
}
