/*
 * bz2b200.h -- C ABI of the B200-native bzip2 compression engine (libbz2b200.so).
 *
 * This is the drop-in boundary for the per-block compression hot path of
 * ohsnyt/bzip2-rust.  The reference has no FFI layer; each entry point below names the
 * Rust function (reference file:line) whose body a thin `extern "C"` crate would replace
 * (INTEGRATION.md shows the binding).  Plain pointers and sizes only.
 *
 * Conventions
 *   - return 0 on success, negative BZ2B200_E_* otherwise; nothing ever unwinds or aborts
 *     across this boundary (the reference panics freely; a library must not).
 *   - functions WITHOUT the _dev suffix take HOST pointers and copy results back.
 *     bz2b200_compress_stream uploads in chunks on its own stream while the first kernels
 *     run and downloads finished output on another; pass page-locked buffers for full
 *     overlap (pageable memory works, the copies then block).  _dev functions take DEVICE
 *     pointers on the context's GPU (used for HBM-resident measurement); device OUTPUT buffers
 *     (d_out, d_dst) and the d_src of bz2b200_shift_bits_dev must be 4-byte aligned (the bit
 *     merge works on 32-bit words): BZ2B200_E_ARG otherwise.  A context works on its own
 *     non-blocking CUDA streams and returns when its work is complete: whatever the caller
 *     still has in flight on a device buffer it passes (a copy into d_in, a memset of d_out)
 *     must have finished before the call.
 *   - a context owns one GPU (streams, workspaces).  Calls on one context are serialised
 *     by an internal mutex; use one context per GPU for multi-GPU sharding.
 *   - there is no CPU fallback: if no CUDA device is usable, bz2b200_create fails.
 */
#ifndef BZ2B200_H
#define BZ2B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bz2b200_ctx bz2b200_ctx;

enum {
    BZ2B200_OK = 0,
    BZ2B200_E_ARG = -1,      /* bad argument (null pointer, level outside 1..9, block too large) */
    BZ2B200_E_CAP = -2,      /* caller's output buffer too small */
    BZ2B200_E_CUDA = -3,     /* CUDA runtime error; see bz2b200_last_error */
    BZ2B200_E_NOMEM = -4,
    BZ2B200_E_FORMAT = -5,   /* decoder: malformed / unsupported stream */
    BZ2B200_E_CRC = -6       /* decoder: CRC mismatch */
};

#define BZ2B200_MAX_BLOCK 900000u   /* largest RLE1 block accepted (level 9: 899 986, rle1.rs:110) */

/* ---- context ---------------------------------------------------------------------------- */
/* device < 0 selects the current CUDA device. */
int  bz2b200_create(int device, bz2b200_ctx **out);
void bz2b200_destroy(bz2b200_ctx *ctx);
/* Frees the context's device workspaces (they are grow-only and sized by the largest call so far: about 45 bytes per
 * input byte of one 256 MiB window plus the resident input / output of the host-buffer entry points).  The next call
 * allocates what it needs again. */
int  bz2b200_trim(bz2b200_ctx *ctx);
const char *bz2b200_last_error(const bz2b200_ctx *ctx);
const char *bz2b200_version(void);
/* number of kernel launches issued by this context since creation (bench.py's gpu_launches) */
uint64_t bz2b200_launch_count(const bz2b200_ctx *ctx);

/* ---- seam: compress_block (src/compression/compress_block.rs:24), batched ---------------- */
/* Replaces `compress_block(block:&[u8], block_crc:u32) -> (Vec<u8>, u8)` for nblk blocks at
 * once (the reference calls it once per block from rayon workers, compress.rs:129-131).
 * blk[i]/len[i]/crc[i]: RLE1 blocks as produced by RLE1Block::next (rle1.rs:250).
 * out[i] receives the packed block (block magic .. last Huffman code), zero padded to a byte;
 * out_bits[i] = exact bit length, so the reference's padding value is (8 - out_bits%8)%8. */
int bz2b200_compress_blocks(bz2b200_ctx *ctx, int nblk, const uint8_t *const *blk, const uint32_t *len,
                            const uint32_t *crc, uint8_t *const *out, const size_t *out_cap,
                            uint64_t *out_bits);

/* ---- seam: compress (src/compression/compress.rs:40) + BitWriter (bitwriter.rs:42-132) --- */
/* Whole stream in memory: RLE1 + block split + CRC, all blocks, header/footer/combined CRC.
 * Byte-identical to the reference's output file for `level` (1..9). */
int bz2b200_compress_stream(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level,
                            uint8_t *out, size_t out_cap, size_t *out_len);
/* Same, input already resident in device memory, output left in device memory. */
int bz2b200_compress_stream_dev(bz2b200_ctx *ctx, const uint8_t *d_in, size_t n, int level,
                                uint8_t *d_out, size_t out_cap, size_t *out_len);
/* Upper bound of the compressed size for n input bytes (for sizing `out`). */
size_t bz2b200_compress_bound(size_t n);

/* Multi-GPU sharding helpers (SURVEY 8e): compress only blocks [first, first+count) of the
 * stream's block sequence and return them as one bit string WITHOUT stream header/footer.
 * block_crcs receives the per-block CRCs so the caller can fold the combined CRC in order.
 * The host merges the pieces with bz2b200_merge_streams. */
int bz2b200_stream_plan(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level,
                        uint64_t *block_start /* cap entries */, uint32_t cap, uint32_t *nblocks);
int bz2b200_compress_range(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level,
                           const uint64_t *block_start, uint32_t nblocks_total,
                           uint32_t first, uint32_t count,
                           uint8_t *out, size_t out_cap, uint64_t *out_bits, uint32_t *block_crcs);
/* Device-resident variants: d_in = the WHOLE stream on this context's GPU, output stays on the device. */
int bz2b200_stream_plan_dev(bz2b200_ctx *ctx, const uint8_t *d_in, size_t n, int level,
                            uint64_t *block_start, uint32_t cap, uint32_t *nblocks);
int bz2b200_compress_range_dev(bz2b200_ctx *ctx, const uint8_t *d_in, size_t n, int level,
                               const uint64_t *block_start, uint32_t nblocks_total,
                               uint32_t first, uint32_t count,
                               uint8_t *d_out, size_t out_cap, uint64_t *out_bits, uint32_t *block_crcs);
/* Sharded planning without replicating the plan: the chain of block starts (rle1.rs:245-264 is a serial
 * iterator) is handed from rank to rank as one number.  d_win = bytes [win_lo, win_lo+win_len) of the stream on
 * this GPU.  Plans the blocks starting in [start, stop_at); *next_start is what the next rank starts from.
 * BZ2B200_E_CAP = the window ends before the last such block does (make the window longer and call again).
 * bz2b200_shard_compress_dev then compresses exactly those blocks (window must still be resident). */
int bz2b200_shard_plan_dev(bz2b200_ctx *ctx, const uint8_t *d_win, size_t win_lo, size_t win_len, size_t n_total,
                           int level, size_t start, size_t stop_at, size_t *next_start, uint32_t *nblocks);
/* Optional first phase of bz2b200_shard_plan_dev that needs no hand-off (run it while the chain arrives): the
 * per-position scans of the window.  A following shard_plan on the same window skips them. */
int bz2b200_shard_scan_dev(bz2b200_ctx *ctx, const uint8_t *d_win, size_t win_lo, size_t win_len, size_t n_total,
                           int level);
int bz2b200_shard_compress_dev(bz2b200_ctx *ctx, uint8_t *d_out, size_t out_cap, uint64_t *out_bits,
                               uint32_t *block_crcs);
/* d_dst = d_src shifted right by phase (0..7) bits, so a rank can pre-align its bit string to its final offset
 * and the ordered merge becomes a byte copy with an OR on the seam byte. */
int bz2b200_shift_bits_dev(bz2b200_ctx *ctx, const uint8_t *d_src, uint64_t nbits, int phase, uint8_t *d_dst);
/* Ordered concatenation at bit granularity + "BZh<level>" header + footer with combined CRC
 * (bitwriter.rs:67-72, :89-114; crc.rs:25-27).  Pure host code. */
int bz2b200_merge_streams(int level, int nparts, const uint8_t *const *part, const uint64_t *part_bits,
                          const uint32_t *const *part_crcs, const uint32_t *part_ncrc,
                          uint8_t *out, size_t out_cap, size_t *out_len);

/* ---- seam: compress (compress.rs:40-136) as a pipeline: the input arrives in pieces ------------------------- */
/* The reference never holds the file: RLE1Block refills block_size bytes at a time (src/tools/rle1.rs:63-85) while
 * rayon workers compress and a writer thread appends finished blocks (compress.rs:74-122).  A zstream does the same
 * with the GPU: bz2b200_zstream_write copies the caller's bytes into page-locked staging (two windows of 64 MiB); a
 * worker thread uploads a full window behind the unconsumed tail of the previous one, runs all block kernels and hands
 * the finished .bz2 bytes to `sink` (called on the worker thread, in stream order; a non-zero return aborts), so the
 * caller's reading overlaps upload, kernels, download and the sink's writing.  bz2b200_zstream_close compresses what is
 * left, writes the footer and frees the stream (also after an error).  The sink receives exactly the bytes
 * bz2b200_compress_stream produces for the concatenated input.  The context must not be used by other threads while a
 * zstream is open on it (calls are serialised, so they would only wait). */
typedef struct bz2b200_zstream bz2b200_zstream;
typedef int (*bz2b200_sink)(void *user, const uint8_t *data, size_t n);
int bz2b200_zstream_open(bz2b200_ctx *ctx, int level, bz2b200_sink sink, void *user, bz2b200_zstream **out);
int bz2b200_zstream_write(bz2b200_zstream *z, const uint8_t *data, size_t n);
int bz2b200_zstream_close(bz2b200_zstream *z, uint64_t *total_in, uint64_t *total_out);

/* ---- seam: compress (src/compression/compress.rs:40-136) on SEVERAL GPUs of one process -------------------- */
/* The reference fans blocks out to rayon workers (compress.rs:125-132) and a writer thread puts them back in
 * order (compress.rs:74-122).  A multi context owns n_devices single-GPU contexts and one host thread per GPU
 * (device_ids == NULL: devices 0 .. n_devices-1; an id may repeat).  bz2b200_compress_stream_multi cuts the input
 * into windows dealt round robin to the GPUs (two per GPU, the first one a quarter of its share; at most 256 MiB
 * each); a GPU uploads and scans a window while it compresses the one before, the uploads of all GPUs are ordered like
 * the windows, the block chain (rle1.rs:245-264) is handed from window to window as one number through host memory,
 * every GPU compresses the blocks that start in its windows and copies each bit string, pre-shifted to its final bit
 * phase, over its own PCIe link straight into `out`; the calling thread ORs the seam bytes, folds the combined CRC
 * (crc.rs:25-27) and writes header and footer (bitwriter.rs:67-72, :103-114).  No collective, no NCCL.  `out` holds
 * exactly the bytes bz2b200_compress_stream produces for the same input, for every n_devices.  Pass page-locked
 * `in` / `out`
 * for full copy overlap.  One call at a time per multi context. */
typedef struct bz2b200_mctx bz2b200_mctx;
int  bz2b200_create_multi(int n_devices, const int *device_ids, bz2b200_mctx **out);
void bz2b200_destroy_multi(bz2b200_mctx *m);
const char *bz2b200_last_error_multi(const bz2b200_mctx *m);
int  bz2b200_multi_devices(const bz2b200_mctx *m);
/* the single-GPU context of one rank (timing / statistics hooks); owned by the multi context */
bz2b200_ctx *bz2b200_multi_context(bz2b200_mctx *m, int rank);
int  bz2b200_compress_stream_multi(bz2b200_mctx *m, const uint8_t *in, size_t n, int level,
                                   uint8_t *out, size_t out_cap, size_t *out_len);
/* decompress (src/compression/decompress.rs:38) on the same GPUs: the input bz2b200_decompress_stream accepts (several
 * streams one after the other, any levels, legacy randomised blocks) is cut into byte windows dealt round robin (about
 * 24 MiB each; each is uploaded with 4 MiB of look-ahead, enough for the longest block that can start in it).  A GPU
 * finds the block magics of its window and entropy-decodes them while the block chain arrives from the window before as
 * one number through host memory; it hands the chain on before its inverse BWT, and copies every decoded batch over
 * its own PCIe link straight to its place in `out` once the lengths of the windows before it are known.  The calling
 * thread checks every stream's combined CRC and the block size its headers allow; block CRCs are checked on the GPUs.
 * `out` receives exactly the bytes bz2b200_decompress_stream produces.  Return codes: those of
 * bz2b200_decompress_stream for an input with a single defect; with several defects E_FORMAT and E_CRC may be
 * swapped.  On BZ2B200_E_CAP, *out_len holds the exact decompressed size.  Inputs smaller than two windows are
 * decoded by bz2b200_decompress_stream on the first GPU.  One call at a time per multi context. */
int  bz2b200_decompress_stream_multi(bz2b200_mctx *m, const uint8_t *in, size_t n,
                                     uint8_t *out, size_t out_cap, size_t *out_len);
/* last call: [0] = bytes copied host -> device (all GPUs), [1] = device -> host */
int  bz2b200_multi_stats(const bz2b200_mctx *m, uint64_t st[8]);

/* ---- stage seams (used by the parity tests, one per reference function) ------------------ */
/* do_crc (src/tools/crc.rs:15) */
int bz2b200_crc32(bz2b200_ctx *ctx, const uint8_t *data, size_t n, uint32_t *crc);
/* RLE1Block::next (src/tools/rle1.rs:250): all blocks of a stream at once.
 * blocks are written back to back into rle1_out; block i spans
 * [rle1_off[i], rle1_off[i+1]) and covers input [in_off[i], in_off[i+1]). */
int bz2b200_rle1_split(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level,
                       uint8_t *rle1_out, size_t rle1_cap, uint64_t *rle1_off, uint64_t *in_off,
                       uint32_t *crc, uint32_t cap_blocks, uint32_t *nblocks);
/* bwt_encode (src/bwt_algorithms/bwt_sort.rs:27): true cyclic-rotation BWT, key = first row of
 * the class of rotation 0 (the reference's native path; see DESIGN.md for the SA-IS divergence) */
int bz2b200_bwt_encode(bz2b200_ctx *ctx, const uint8_t *in, uint32_t n, uint8_t *bwt, uint32_t *key);
int bz2b200_bwt_encode_batch(bz2b200_ctx *ctx, int nblk, const uint8_t *const *in, const uint32_t *n,
                             uint8_t *const *bwt, uint32_t *key);
/* rle2_mtf_encode (src/tools/rle2_mtf.rs:23): sym needs n+1 entries; symmap 17 entries */
int bz2b200_mtf_rle2(bz2b200_ctx *ctx, const uint8_t *bwt, uint32_t n, uint16_t *sym, uint32_t *m,
                     uint32_t freq[256], uint16_t symmap[17], int *nmap);
/* huf_encode (src/huffman_coding/huffman.rs:79) on an empty BitPacker: bits of
 * symbol map .. last code.  lengths (6*258 bytes) and selectors (ceil(m/50) bytes) are optional
 * debug outputs. */
int bz2b200_huffman(bz2b200_ctx *ctx, const uint16_t *sym, uint32_t m, const uint32_t freq[256],
                    const uint16_t *symmap, int nmap, uint8_t *out, size_t out_cap, uint64_t *out_bits,
                    uint8_t *lengths, uint8_t *selectors, int *table_count);
/* bwt_decode (src/bwt_algorithms/bwt_sort.rs:91) */
int bz2b200_bwt_decode(bz2b200_ctx *ctx, uint32_t key, const uint8_t *bwt, uint32_t n, uint8_t *out);
/* decompress (src/compression/decompress.rs:38): what libbz2 accepts -- one or several bzip2 streams one after the
 * other, legacy randomised blocks; block and combined CRCs are enforced (the reference only logs a mismatch) */
int bz2b200_decompress_stream(bz2b200_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap,
                              size_t *out_len);

/* ---- measurement hooks ------------------------------------------------------------------- */
/* Per-stage device time (ms, CUDA events on the context's stream) of the last compress call:
 * [0]=rle1+crc+split [1]=bwt [2]=mtf/rle2 [3]=huffman select+lengths [4]=bit pack [5]=total.
 * Only filled when enabled with bz2b200_set_timing(ctx, 1) (2 = also per-kernel events). */
void bz2b200_set_timing(bz2b200_ctx *ctx, int on);
int  bz2b200_get_timing(const bz2b200_ctx *ctx, float ms[8]);
/* Per-kernel device time, enabled with bz2b200_set_timing(ctx, 2): CUDA events on the context's stream
 * around every launch.  idx = 0..; returns BZ2B200_E_ARG past the last kernel.  `bytes` is the
 * ALGORITHMIC byte count of those launches (per-element figures in DESIGN.md), not DRAM traffic. */
int  bz2b200_kernel_stats(bz2b200_ctx *ctx, int idx, char name[64], double *ms, uint64_t *launches,
                          uint64_t *bytes);
void bz2b200_reset_kernel_stats(bz2b200_ctx *ctx);
/* statistics of the last BWT batch: [0]=blocks [1]=sum n [2]=max doubling rounds
 * [3]=sum over rounds of unresolved list lengths [4]=blocks the reference's path selector (bwt_sort.rs:29) would have
 * sent to its SA-IS fallback; since the context was created: [5]=such blocks [6]=all blocks */
int  bz2b200_get_bwt_stats(const bz2b200_ctx *ctx, uint64_t st[8]);

#ifdef __cplusplus
}
#endif
#endif
