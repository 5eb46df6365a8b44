// shard.cu -- multi-GPU sharding of ONE stream without replicating the block plan (SURVEY 8e).
//
// The block chain s_{k+1} = e(s_k) is sequential over the whole input (rle1.rs:245-264 is an iterator),
// but each link only needs the per-position arrays around it.  So every rank scans its own slice in
// parallel, and the chain is handed from rank to rank as ONE number:
//     rank r:  scan own window (run starts, RLE1 output prefix)          bz2b200_shard_scan_dev   -- parallel
//              start_r = (r == 0) ? 0 : recv(r-1)
//              chain the blocks whose start lies in [start_r, stop_r)    bz2b200_shard_plan_dev   -- ~5 us / block
//              send(next_start) to r+1                                    -- before the heavy work
//              compress the planned blocks                                bz2b200_shard_compress_dev
// The scan may start anywhere (it treats the window origin as a run boundary): a block that starts inside a
// run re-chunks that run from its own start anyway, and everything behind the first run boundary is global.
// The ranks' bit strings are then shifted to their final bit phase on the device (bz2b200_shift_bits_dev) so
// that the ordered merge is a byte copy with an OR on the seam byte.
#include "common.cuh"
#include <algorithm>
#include <string.h>

u32 off_from_for(size_t n, int level, size_t window_pos);
int bz_concat_blocks(bz2b200_ctx *ctx, const HufOut &H, u32 nb, const u64 *hoff, u64 maxbits, u8 *d_out);
int bz_shift_bits(bz2b200_ctx *ctx, const u8 *d_src, u64 nbits, int phase, u8 *d_dst);

namespace {
constexpr u32 MAX_SHARD_BLOCKS = 4096;

int do_scan(bz2b200_ctx *ctx, ShardPlan &P, const u8 *d_win, size_t win_lo, size_t win_len, size_t n_total, int level) {
    P.scanned = false; P.planned = false;
    Batch B; u32 nb = 0, consumed = 0;
    bool eof = win_lo + win_len == n_total;
    int rc = bz_rle1_window(ctx, d_win, (u32)win_len, level, eof, 0, MAX_SHARD_BLOCKS, B, &nb, &consumed, nullptr, true,
                            0xFFFFFFFFu, /*skip chain*/ 2, 0);
    if (rc) return rc;
    P.scanned = true; P.d_win = d_win; P.win_lo = win_lo; P.win_len = win_len; P.n_total = n_total; P.level = level;
    return BZ2B200_OK;
}
}  // namespace

// Phase 1 for a window that still sits in HOST memory (multi.cu), in two steps so that the upload of a rank's NEXT window
// can run under the compression of the current one:
//   bz_shard_post_upload   the window is copied in chunks on the context's upload stream, one event per chunk
//   bz_shard_scan_arriving the scan kernels follow the chunks as they land (bz_rle1_window, "arrival")
int bz_shard_post_upload(bz2b200_ctx *ctx, const u8 *h_src, u8 *d_win, size_t win_len, size_t chunk,
                         std::vector<cudaEvent_t> &evs) {
    if (!ctx || !h_src || !d_win || win_len == 0 || chunk == 0) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    if (!ctx->s_up) {
        BZ_CHECK(cudaStreamCreateWithFlags(&ctx->s_up, cudaStreamNonBlocking));
        BZ_CHECK(cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking));
    }
    size_t nchunks = (win_len + chunk - 1) / chunk;
    while (evs.size() < nchunks) {
        cudaEvent_t e;
        BZ_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        evs.push_back(e);
    }
    for (size_t i = 0; i < nchunks; i++) {
        size_t off = i * chunk, len = std::min(chunk, win_len - off);
        BZ_CHECK(cudaMemcpyAsync(d_win + off, h_src + off, len, cudaMemcpyHostToDevice, ctx->s_up));
        BZ_CHECK(cudaEventRecord(evs[i], ctx->s_up));
    }
    return BZ2B200_OK;
}

int bz_shard_scan_arriving(bz2b200_ctx *ctx, u8 *d_win, size_t win_lo, size_t win_len, size_t n_total, int level,
                           size_t chunk, std::vector<cudaEvent_t> &evs) {
    int mode = BZ_MODE_REF;
    if (!ctx || !d_win || !bz_parse_level(&level, &mode) || win_lo + win_len > n_total || win_len > 0xFFFFFF00ull || win_len == 0)
        return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    size_t nchunks = (win_len + chunk - 1) / chunk;
    if (evs.size() < nchunks) return BZ2B200_E_ARG;
    std::vector<cudaEvent_t> mine(evs.begin(), evs.begin() + nchunks);
    Arrival arr;
    arr.ev = &mine; arr.chunk = chunk; arr.win_off = 0; arr.waited = 0;
    ctx->arrival = &arr;
    int rc = do_scan(ctx, ctx->shard, d_win, win_lo, win_len, n_total, level);
    ctx->arrival = nullptr;
    if (rc) { cudaStreamSynchronize(ctx->s_up); return rc; }
    // everything the later phases read must be resident: the compute stream waits for the last chunk
    while (arr.waited < nchunks) { BZ_CHECK(cudaStreamWaitEvent(ctx->stream, mine[arr.waited], 0)); arr.waited++; }
    return BZ2B200_OK;
}

extern "C" {

// Phase 1 (needs no hand-off): scans d_win[0 .. win_len) = bytes [win_lo, win_lo + win_len) of the stream.
int bz2b200_shard_scan_dev(bz2b200_ctx *ctx, const uint8_t *d_win, size_t win_lo, size_t win_len, size_t n_total,
                           int level) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || !d_win || !bz_parse_level(&level, &mode) || win_lo + win_len > n_total || win_len > 0xFFFFFF00ull || win_len == 0)
        return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    return do_scan(ctx, ctx->shard, d_win, win_lo, win_len, n_total, level);
    BZ_API_CATCH
}

// Phase 2: chains every block whose first byte lies in [start, stop_at) (absolute offsets; `start` must be a true
// block start).  *next_start = first block start >= stop_at (or n_total).  Scans first unless the same window was
// just scanned.  BZ2B200_E_CAP: the window ends before the last such block does (lengthen it and call again).
int bz2b200_shard_plan_dev(bz2b200_ctx *ctx, const uint8_t *d_win, size_t win_lo, size_t win_len, size_t n_total,
                           int level, size_t start, size_t stop_at, size_t *next_start, uint32_t *nblocks) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || !d_win || !next_start || !nblocks || !bz_parse_level(&level, &mode) || win_lo + win_len > n_total ||
        win_len > 0xFFFFFF00ull)
        return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    ShardPlan &P = ctx->shard;
    P.planned = false;
    *nblocks = 0;
    // the previous rank's last block may already cover this whole shard: nothing to do, pass the chain on
    if (start >= stop_at || start >= n_total) { *next_start = start; P.nb = 0; P.planned = true; return BZ2B200_OK; }
    if (start < win_lo) return BZ2B200_E_ARG;
    if (start >= win_lo + win_len) return BZ2B200_E_CAP;          // window does not reach the first block yet
    bool same = P.scanned && P.d_win == d_win && P.win_lo == win_lo && P.win_len == win_len && P.n_total == n_total &&
                P.level == level;          // the scans do not depend on the mode
    if (!same) {
        int rc = do_scan(ctx, P, d_win, win_lo, win_len, n_total, level);
        if (rc) return rc;
    }
    bool eof = win_lo + win_len == n_total;
    u32 W = (u32)win_len;
    u32 s0 = (u32)(start - win_lo);
    u32 stop_rel = (u32)std::min<size_t>(stop_at - win_lo, 0xFFFFFFF0u);
    u32 off_from = off_from_for(n_total, level, win_lo);
    Batch B; u32 nb = 0, consumed = 0;
    int rc = bz_rle1_window(ctx, d_win, W, level, eof, off_from, MAX_SHARD_BLOCKS, B, &nb, &consumed, nullptr, true, stop_rel,
                            /*skip scans*/ 1, s0);
    if (rc) return rc;
    if (consumed < stop_rel && !(eof && consumed == W)) return BZ2B200_E_CAP;   // ran out of window (or 4096 blocks)
    *next_start = win_lo + consumed;
    *nblocks = nb;
    P.planned = true; P.eof = eof; P.off_from = off_from; P.stop_rel = stop_rel; P.s0 = s0; P.nb = nb; P.mode = mode;
    return BZ2B200_OK;
    BZ_API_CATCH
}

// Phase 3: compresses the blocks of the preceding bz2b200_shard_plan_dev call (same context, window still
// resident).  d_out receives one bit string (no stream header/footer); block_crcs[nblocks].
int bz2b200_shard_compress_dev(bz2b200_ctx *ctx, uint8_t *d_out, size_t out_cap, uint64_t *out_bits,
                               uint32_t *block_crcs) {
    BZ_API_TRY
    if (!ctx || !d_out || !out_bits || ((uintptr_t)d_out & 3u)) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    ShardPlan &P = ctx->shard;
    if (!P.planned) { ctx->err = "shard_compress: no pending plan"; return BZ2B200_E_ARG; }
    P.planned = false;
    ctx->mode = P.mode;
    *out_bits = 0;
    cudaStream_t st = ctx->stream;
    if (ctx->timing) cudaEventRecord(ctx->ev_total[0], st);
    BZ_CHECK(cudaMemsetAsync(d_out, 0, out_cap & ~(size_t)3, st));
    if (P.nb == 0) return BZ2B200_OK;
    if (!block_crcs) return BZ2B200_E_ARG;
    Batch B; u32 nb = 0, consumed = 0;
    int rc = bz_rle1_window(ctx, P.d_win, (u32)P.win_len, P.level, P.eof, P.off_from, MAX_SHARD_BLOCKS, B, &nb, &consumed,
                            nullptr, false, P.stop_rel, /*skip scans + chain*/ 3, P.s0);
    P.scanned = false;
    if (rc) return rc;
    if (nb != P.nb) { ctx->err = "shard_compress: plan changed"; return BZ2B200_E_ARG; }
    // the BWT workspace is sized per batch; a shard is compressed in sub-batches of whole blocks
    u32 stride = B.stride;
    u32 batch_blocks = (u32)std::max<size_t>(1, ((size_t)272 << 20) / stride);
    u64 bitpos = 0;
    std::vector<u64> hoff;
    for (u32 first = 0; first < nb; first += batch_blocks) {
        u32 cnt = std::min(batch_blocks, nb - first);
        Batch S = B;
        S.nblk = (int)cnt;
        S.T = B.T + (size_t)first * stride;
        S.len = B.len + first;
        S.total_n = B.total_n * cnt / nb;
        HufOut H;
        rc = bz_compress_batch(ctx, S, ctx->d_crc.as<u32>() + first, H);
        if (rc) return rc;
        BZ_CHECK(ctx->h_small.ensure((size_t)cnt * 12 + 64));
        u64 *hbits = ctx->h_small.as<u64>();
        u32 *hcrc = (u32 *)(hbits + cnt);
        BZ_CHECK(cudaMemcpyAsync(hbits, H.d_bits, (size_t)cnt * 8, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaMemcpyAsync(hcrc, ctx->d_crc.as<u32>() + first, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaStreamSynchronize(st));
        hoff.resize(cnt);
        u64 maxbits = 0;
        for (u32 k = 0; k < cnt; k++) {
            if (hbits[k] == ~0ull) { ctx->err = "huffman: packed block exceeds its slot"; return BZ2B200_E_CAP; }
            hoff[k] = bitpos; bitpos += hbits[k]; maxbits = std::max(maxbits, hbits[k]);
            block_crcs[first + k] = hcrc[k];
        }
        if ((bitpos + 7) / 8 + 16 > out_cap) return BZ2B200_E_CAP;
        rc = bz_concat_blocks(ctx, H, cnt, hoff.data(), maxbits, d_out);
        if (rc) return rc;
    }
    if (ctx->timing) {
        cudaEventRecord(ctx->ev_total[1], st);
        cudaEventSynchronize(ctx->ev_total[1]);
        cudaEventElapsedTime(&ctx->stage_ms[5], ctx->ev_total[0], ctx->ev_total[1]);
    }
    *out_bits = bitpos;
    return BZ2B200_OK;
    BZ_API_CATCH
}

// d_dst = d_src shifted right by `phase` bits (0..7): byte k of d_dst then lines up with byte (offset/8 + k)
// of the final stream when phase = offset % 8.  d_dst needs (nbits + phase + 7)/8 + 8 bytes.
int bz2b200_shift_bits_dev(bz2b200_ctx *ctx, const uint8_t *d_src, uint64_t nbits, int phase, uint8_t *d_dst) {
    BZ_API_TRY
    if (!ctx || !d_src || !d_dst || phase < 0 || phase > 7 || (((uintptr_t)d_src | (uintptr_t)d_dst) & 3u)) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    return bz_shift_bits(ctx, d_src, nbits, phase, d_dst);
    BZ_API_CATCH
}

}  // extern "C"
