//! Raw bindings of include/bz2b200.h (C ABI of libbz2b200.so).  UNBUILT in this repository's image.
//! Every function returns 0 or a negative BZ2B200_E_* code; nothing unwinds across the boundary.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct bz2b200_ctx { _private: [u8; 0] }
#[repr(C)] pub struct bz2b200_mctx { _private: [u8; 0] }
#[repr(C)] pub struct bz2b200_zstream { _private: [u8; 0] }
#[repr(C)] pub struct bz2b200_dstream { _private: [u8; 0] }
pub type bz2b200_sink = Option<unsafe extern "C" fn(user: *mut c_void, data: *const u8, n: usize) -> c_int>;

pub const BZ2B200_OK: c_int = 0;
pub const BZ2B200_E_ARG: c_int = -1;
pub const BZ2B200_E_CAP: c_int = -2;
pub const BZ2B200_E_CUDA: c_int = -3;
pub const BZ2B200_E_NOMEM: c_int = -4;
pub const BZ2B200_E_FORMAT: c_int = -5;
pub const BZ2B200_E_CRC: c_int = -6;
pub const BZ2B200_MAX_BLOCK: u32 = 900_000;
pub const BZ2B200_REC_FOOTER: u32 = 1;
pub const BZ2B200_REC_NO_MAGIC: u32 = 2;

/// One block candidate or footer found by `bz2b200_recover`.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct bz2b200_rec_entry {
    pub bit: u64,
    pub end_bit: u64,
    pub out_off: u64,
    pub out_len: u32,
    pub crc: u32,
    pub status: i32,
    pub flags: u32,
}

extern "C" {
    // ---- context ----
    pub fn bz2b200_create(device: c_int, out: *mut *mut bz2b200_ctx) -> c_int;
    pub fn bz2b200_destroy(ctx: *mut bz2b200_ctx);
    pub fn bz2b200_trim(ctx: *mut bz2b200_ctx) -> c_int;
    pub fn bz2b200_last_error(ctx: *const bz2b200_ctx) -> *const c_char;
    pub fn bz2b200_version() -> *const c_char;
    pub fn bz2b200_launch_count(ctx: *const bz2b200_ctx) -> u64;
    // ---- seam: compress_block (src/compression/compress_block.rs:24), batched ----
    pub fn bz2b200_compress_blocks(ctx: *mut bz2b200_ctx, nblk: c_int, blk: *const *const u8, len: *const u32,
        crc: *const u32, out: *const *mut u8, out_cap: *const usize, out_bits: *mut u64) -> c_int;
    // ---- seam: compress (src/compression/compress.rs:40) + BitWriter (bitwriter.rs:42-132) ----
    pub fn bz2b200_compress_stream(ctx: *mut bz2b200_ctx, input: *const u8, n: usize, level: c_int,
        out: *mut u8, out_cap: usize, out_len: *mut usize) -> c_int;
    pub fn bz2b200_compress_stream_dev(ctx: *mut bz2b200_ctx, d_in: *const u8, n: usize, level: c_int,
        d_out: *mut u8, out_cap: usize, out_len: *mut usize) -> c_int;
    pub fn bz2b200_compress_bound(n: usize) -> usize;
    // ---- sharding helpers (one process per GPU) ----
    pub fn bz2b200_stream_plan(ctx: *mut bz2b200_ctx, input: *const u8, n: usize, level: c_int,
        block_start: *mut u64, cap: u32, nblocks: *mut u32) -> c_int;
    pub fn bz2b200_compress_range(ctx: *mut bz2b200_ctx, input: *const u8, n: usize, level: c_int,
        block_start: *const u64, nblocks_total: u32, first: u32, count: u32,
        out: *mut u8, out_cap: usize, out_bits: *mut u64, block_crcs: *mut u32) -> c_int;
    pub fn bz2b200_stream_plan_dev(ctx: *mut bz2b200_ctx, d_in: *const u8, n: usize, level: c_int,
        block_start: *mut u64, cap: u32, nblocks: *mut u32) -> c_int;
    pub fn bz2b200_compress_range_dev(ctx: *mut bz2b200_ctx, d_in: *const u8, n: usize, level: c_int,
        block_start: *const u64, nblocks_total: u32, first: u32, count: u32,
        d_out: *mut u8, out_cap: usize, out_bits: *mut u64, block_crcs: *mut u32) -> c_int;
    pub fn bz2b200_shard_plan_dev(ctx: *mut bz2b200_ctx, d_win: *const u8, win_lo: usize, win_len: usize, n_total: usize,
        level: c_int, start: usize, stop_at: usize, next_start: *mut usize, nblocks: *mut u32) -> c_int;
    pub fn bz2b200_shard_scan_dev(ctx: *mut bz2b200_ctx, d_win: *const u8, win_lo: usize, win_len: usize, n_total: usize,
        level: c_int) -> c_int;
    pub fn bz2b200_shard_compress_dev(ctx: *mut bz2b200_ctx, d_out: *mut u8, out_cap: usize, out_bits: *mut u64,
        block_crcs: *mut u32) -> c_int;
    pub fn bz2b200_shift_bits_dev(ctx: *mut bz2b200_ctx, d_src: *const u8, nbits: u64, phase: c_int, d_dst: *mut u8) -> c_int;
    pub fn bz2b200_merge_streams(level: c_int, nparts: c_int, part: *const *const u8, part_bits: *const u64,
        part_crcs: *const *const u32, part_ncrc: *const u32, out: *mut u8, out_cap: usize, out_len: *mut usize) -> c_int;
    // ---- seam: compress as a pipeline (compress.rs:69-132): pieces in, finished bytes to a sink ----
    pub fn bz2b200_zstream_open(ctx: *mut bz2b200_ctx, level: c_int, sink: bz2b200_sink, user: *mut c_void,
        out: *mut *mut bz2b200_zstream) -> c_int;
    pub fn bz2b200_zstream_write(z: *mut bz2b200_zstream, data: *const u8, n: usize) -> c_int;
    pub fn bz2b200_zstream_close(z: *mut bz2b200_zstream, total_in: *mut u64, total_out: *mut u64) -> c_int;
    // ---- seam: decompress as a pipeline: pieces in, checked bytes to a sink (None: test mode) ----
    pub fn bz2b200_dstream_open(ctx: *mut bz2b200_ctx, sink: bz2b200_sink, user: *mut c_void,
        out: *mut *mut bz2b200_dstream) -> c_int;
    pub fn bz2b200_dstream_write(d: *mut bz2b200_dstream, data: *const u8, n: usize) -> c_int;
    pub fn bz2b200_dstream_close(d: *mut bz2b200_dstream, total_in: *mut u64, total_out: *mut u64) -> c_int;
    // ---- seam: compress on several GPUs of one process ----
    pub fn bz2b200_create_multi(n_devices: c_int, device_ids: *const c_int, out: *mut *mut bz2b200_mctx) -> c_int;
    pub fn bz2b200_destroy_multi(m: *mut bz2b200_mctx);
    pub fn bz2b200_last_error_multi(m: *const bz2b200_mctx) -> *const c_char;
    pub fn bz2b200_multi_devices(m: *const bz2b200_mctx) -> c_int;
    pub fn bz2b200_multi_context(m: *mut bz2b200_mctx, rank: c_int) -> *mut bz2b200_ctx;
    pub fn bz2b200_compress_stream_multi(m: *mut bz2b200_mctx, input: *const u8, n: usize, level: c_int,
        out: *mut u8, out_cap: usize, out_len: *mut usize) -> c_int;
    pub fn bz2b200_decompress_stream_multi(m: *mut bz2b200_mctx, input: *const u8, n: usize, out: *mut u8,
        out_cap: usize, out_len: *mut usize) -> c_int;
    pub fn bz2b200_multi_stats(m: *const bz2b200_mctx, st: *mut u64) -> c_int;
    // ---- stage seams (one per reference function) ----
    pub fn bz2b200_crc32(ctx: *mut bz2b200_ctx, data: *const u8, n: usize, crc: *mut u32) -> c_int;
    pub fn bz2b200_rle1_split(ctx: *mut bz2b200_ctx, input: *const u8, n: usize, level: c_int,
        rle1_out: *mut u8, rle1_cap: usize, rle1_off: *mut u64, in_off: *mut u64,
        crc: *mut u32, cap_blocks: u32, nblocks: *mut u32) -> c_int;
    pub fn bz2b200_bwt_encode(ctx: *mut bz2b200_ctx, input: *const u8, n: u32, bwt: *mut u8, key: *mut u32) -> c_int;
    pub fn bz2b200_bwt_encode_batch(ctx: *mut bz2b200_ctx, nblk: c_int, input: *const *const u8, n: *const u32,
        bwt: *const *mut u8, key: *mut u32) -> c_int;
    pub fn bz2b200_mtf_rle2(ctx: *mut bz2b200_ctx, bwt: *const u8, n: u32, sym: *mut u16, m: *mut u32,
        freq: *mut u32, symmap: *mut u16, nmap: *mut c_int) -> c_int;
    pub fn bz2b200_huffman(ctx: *mut bz2b200_ctx, sym: *const u16, m: u32, freq: *const u32,
        symmap: *const u16, nmap: c_int, out: *mut u8, out_cap: usize, out_bits: *mut u64,
        lengths: *mut u8, selectors: *mut u8, table_count: *mut c_int) -> c_int;
    pub fn bz2b200_bwt_decode(ctx: *mut bz2b200_ctx, key: u32, bwt: *const u8, n: u32, out: *mut u8) -> c_int;
    pub fn bz2b200_decompress_stream(ctx: *mut bz2b200_ctx, input: *const u8, n: usize, out: *mut u8, out_cap: usize,
        out_len: *mut usize) -> c_int;
    // ---- block recovery: every intact block of a damaged input to a sink (None: report only) ----
    pub fn bz2b200_recover(ctx: *mut bz2b200_ctx, input: *const u8, n: usize, sink: bz2b200_sink, user: *mut c_void,
        ent: *mut bz2b200_rec_entry, ent_cap: u32, nent: *mut u32, total_out: *mut u64) -> c_int;
    // ---- measurement hooks ----
    pub fn bz2b200_set_timing(ctx: *mut bz2b200_ctx, on: c_int);
    pub fn bz2b200_get_timing(ctx: *const bz2b200_ctx, ms: *mut f32) -> c_int;
    pub fn bz2b200_kernel_stats(ctx: *mut bz2b200_ctx, idx: c_int, name: *mut c_char, ms: *mut f64,
        launches: *mut u64, bytes: *mut u64) -> c_int;
    pub fn bz2b200_reset_kernel_stats(ctx: *mut bz2b200_ctx);
    pub fn bz2b200_get_bwt_stats(ctx: *const bz2b200_ctx, st: *mut u64) -> c_int;
}
