//! Raw bindings to libgarage_ec.so -- mirror of include/garage_ec.h (see INTEGRATION.md section 1).
//! NOT compiled in this repository's environment (no rustc); kept in sync by tests/test_abi.py,
//! which checks that every symbol of the header appears here.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct garage_ec_ctx { _private: [u8; 0] }

pub const GARAGE_EC_OK: c_int = 0;
pub const GARAGE_EC_E_INVALID: c_int = -1;
pub const GARAGE_EC_E_CUDA: c_int = -2;
pub const GARAGE_EC_E_NOMEM: c_int = -3;
pub const GARAGE_EC_E_UNRECOVERABLE: c_int = -4;
pub const GARAGE_EC_E_NODEVICE: c_int = -5;
pub const GARAGE_EC_E_ALIGN: c_int = -6;
pub const GARAGE_EC_E_UNCORRECTABLE: c_int = -7;
pub const GARAGE_EC_VANDERMONDE: c_int = 0;
pub const GARAGE_EC_CAUCHY: c_int = 1;
pub const GARAGE_EC_MEM_HOST: c_int = 0;
pub const GARAGE_EC_MEM_DEVICE: c_int = 1;

#[link(name = "garage_ec")]
extern "C" {
    pub fn garage_ec_create(out: *mut *mut garage_ec_ctx, cuda_device: c_int, k: c_int, m: c_int,
                            matrix_kind: c_int) -> c_int;
    pub fn garage_ec_create_with_matrix(out: *mut *mut garage_ec_ctx, cuda_device: c_int, k: c_int,
                            m: c_int, parity_rows: *const u8) -> c_int;
    pub fn garage_ec_destroy(ctx: *mut garage_ec_ctx);
    pub fn garage_ec_matrix(ctx: *const garage_ec_ctx, out_m_by_k: *mut u8) -> c_int;
    pub fn garage_ec_params(ctx: *const garage_ec_ctx, k: *mut c_int, m: *mut c_int, dev: *mut c_int) -> c_int;
    pub fn garage_ec_strerror(code: c_int) -> *const c_char;
    pub fn garage_ec_last_error(ctx: *const garage_ec_ctx) -> *const c_char;
    pub fn garage_ec_abi_version() -> c_int;
    pub fn garage_ec_shard_len(block_len: u32, k: c_int) -> u32;
    pub fn garage_ec_stride_for(shard_len: u32) -> usize;
    pub fn garage_ec_encode(ctx: *mut garage_ec_ctx, data: *const u8, parity: *mut u8,
                            shard_len: *const u32, stride: usize, n_stripes: usize,
                            mem_kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_reconstruct(ctx: *mut garage_ec_ctx, shards: *mut u8, present: *const u8,
                            want: *const u8, status: *mut i32, shard_len: *const u32, stride: usize,
                            n_stripes: usize, mem_kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_verify(ctx: *mut garage_ec_ctx, shards: *const u8, mismatch: *mut u32,
                            shard_len: *const u32, stride: usize, n_stripes: usize,
                            mem_kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_correct(ctx: *mut garage_ec_ctx, shards: *mut u8, present: *const u8, status: *mut i32,
                            fixed: *mut u8, shard_len: *const u32, stride: usize, n_stripes: usize,
                            mem_kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_encode_blocks(ctx: *mut garage_ec_ctx, blocks: *const *const u8,
                            block_len: *const u32, n_blocks: usize, parity_out: *mut u8,
                            stride: usize) -> c_int;
    pub fn garage_ec_decode_blocks(ctx: *mut garage_ec_ctx, shards: *const u8, present: *const u8,
                            block_len: *const u32, n_blocks: usize, stride: usize,
                            blocks_out: *const *mut u8, status: *mut i32) -> c_int;
    pub fn garage_ec_encode_blocks_with_sums(ctx: *mut garage_ec_ctx, blocks: *const *const u8,
                            block_len: *const u32, n_blocks: usize, parity_out: *mut u8,
                            sums_out: *mut u8, stride: usize) -> c_int;
    pub fn garage_ec_shard_sums(ctx: *mut garage_ec_ctx, shards: *const u8, shard_len: *const u32,
                            stride: usize, n_stripes: usize, shards_per_stripe: c_int,
                            sums_out: *mut u8, mem_kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_check_sums(ctx: *mut garage_ec_ctx, shards: *const u8, expect: *const u8,
                            shard_len: *const u32, stride: usize, n_stripes: usize,
                            shards_per_stripe: c_int, bad_out: *mut u8, mem_kind: c_int,
                            cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_scrub_repair(ctx: *mut garage_ec_ctx, shards: *mut u8, expect_sums: *const u8,
                            bad_out: *mut u8, status: *mut i32, shard_len: *const u32, stride: usize,
                            n_stripes: usize, mem_kind: c_int, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_blake2sum(data: *const u8, len: usize, out32: *mut u8);
    pub fn garage_ec_host_alloc(ctx: *mut garage_ec_ctx, out: *mut *mut c_void, bytes: usize) -> c_int;
    pub fn garage_ec_host_alloc_wc(ctx: *mut garage_ec_ctx, out: *mut *mut c_void, bytes: usize) -> c_int;
    pub fn garage_ec_host_free(ctx: *mut garage_ec_ctx, ptr: *mut c_void);
    pub fn garage_ec_fill_random(ctx: *mut garage_ec_ctx, dst: *mut u8, len: usize, seed: u64,
                            offset: u64, cuda_stream: *mut c_void) -> c_int;
    pub fn garage_ec_launch_count(ctx: *const garage_ec_ctx) -> u64;
    pub fn garage_ec_set_timing(ctx: *mut garage_ec_ctx, enabled: c_int) -> c_int;
    pub fn garage_ec_timing_read(ctx: *mut garage_ec_ctx, total_ms: *mut f64, launches: *mut u64) -> c_int;
    pub fn garage_ec_numa_info(ctx: *const garage_ec_ctx, gpu_node: *mut c_int, last_alloc_node: *mut c_int) -> c_int;
    pub fn garage_ec_bind_thread(ctx: *const garage_ec_ctx) -> c_int;
    pub fn garage_ec_reconstruct_stripes(ctx: *mut garage_ec_ctx, stripes: *const *mut u8, present: *const u8,
                            want: *const u8, status: *mut i32, shard_len: *const u32, stride: usize,
                            n_stripes: usize) -> c_int;
    pub fn garage_ec_set_sum_kind(ctx: *mut garage_ec_ctx, kind: c_int) -> c_int;
    pub fn garage_ec_set_wait_mode(ctx: *mut garage_ec_ctx, blocking: c_int) -> c_int;
    pub fn garage_ec_copy_for_dma(dst_pinned: *mut c_void, src: *const c_void, n: usize);
    pub fn garage_ec_shard_sum_host(kind: c_int, data: *const u8, len: usize, out32: *mut u8) -> c_int;
    pub fn garage_ec_debug_fail_after(ctx: *mut garage_ec_ctx, n_calls: std::os::raw::c_long) -> c_int;
}
