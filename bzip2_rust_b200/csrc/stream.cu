// stream.cu -- whole-stream entry points: compress (reference src/compression/compress.rs:40-136)
// and the BitWriter (src/bitstream/bitwriter.rs:42-173): "BZh<level>" header, ordered bit-granular
// concatenation of the packed blocks, combined CRC (crc.rs:25-27), footer magic + CRC, byte padding.
//
// The reference strips each block's byte padding by shifting a 64-bit queue (bitwriter.rs:97-100);
// here every block carries its exact bit length, an exclusive prefix sum gives its absolute bit
// offset, and one kernel ORs the blocks of a batch into the final buffer at those offsets.
#include "common.cuh"
#include <stdlib.h>
#include <string.h>
#include <algorithm>

namespace {

__device__ __forceinline__ u32 bswap32s(u32 v) { return __byte_perm(v, 0, 0x0123); }

// grid (words tiles, nblk): OR block k's big-endian bit string into dst at bit offset off[k]
__global__ void __launch_bounds__(256) k_concat_bits(const u8 *src, size_t src_stride, const u64 *nbits,
                                                     const u64 *off, u32 *dst) {
    u32 k = blockIdx.y;
    u64 nb = nbits[k];
    u32 nwords = (u32)((nb + 31) >> 5);
    u32 w = blockIdx.x * 256 + threadIdx.x;
    if (w >= nwords) return;
    const u32 *s = (const u32 *)(src + (size_t)k * src_stride);
    u32 v = bswap32s(s[w]);
    if (v == 0) return;
    u64 pos = off[k] + ((u64)w << 5);
    u64 dw = pos >> 5;
    int sh = (int)(pos & 31);
    u32 hi = v >> sh;
    u32 lo = sh ? (v << (32 - sh)) : 0u;
    if (hi) atomicOr(&dst[dw], bswap32s(hi));
    if (lo) atomicOr(&dst[dw + 1], bswap32s(lo));
}

// header "BZh<level>" at byte 0 and footer (48-bit magic, 32-bit combined CRC) at bit `pos`
__global__ void k_header_footer(u32 *dst, int level, u64 pos, u32 combined, int write_header) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (write_header) {
        u32 h = ((u32)'B' << 24) | ((u32)'Z' << 16) | ((u32)'h' << 8) | (u32)('0' + level);   // bitwriter.rs:67-72
        atomicOr(&dst[0], bswap32s(h));
    }
    u32 parts[3] = {0x177245u, 0x385090u, 0};                   // bitwriter.rs:105
    int lens[3] = {24, 24, 32};
    parts[2] = combined;
    for (int i = 0; i < 3; i++) {
        u64 w = pos >> 5;
        int off = (int)(pos & 31);
        u64 v = ((u64)parts[i] << (64 - lens[i])) >> off;
        u32 hi = (u32)(v >> 32), lo = (u32)v;
        if (hi) atomicOr(&dst[w], bswap32s(hi));
        if (lo) atomicOr(&dst[w + 1], bswap32s(lo));
        pos += lens[i];
    }
}

constexpr size_t WINDOW = 256u << 20;       // input bytes planned per pass
constexpr u32 MAX_BATCH_BLOCKS = 4096;
constexpr size_t MAX_BATCH_BYTES = 272u << 20;   // RLE1 bytes per BWT batch (workspace ~40 B per byte)

}  // namespace

#define LAUNCH_OK()                                                  \
    do {                                                             \
        ctx->prof_end();                                             \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) { ctx->fail("kernel launch", e_, __FILE__, __LINE__); return BZ2B200_E_CUDA; } \
    } while (0)

// OR nb packed blocks (H) into d_out at the absolute bit offsets hoff[] (host array); synchronises the stream.
int bz_concat_blocks(bz2b200_ctx *ctx, const HufOut &H, u32 nb, const u64 *hoff, u64 maxbits, u8 *d_out) {
    cudaStream_t st = ctx->stream;
    BZ_CHECK(ctx->d_bitoff.ensure((size_t)nb * 8));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_bitoff.p, hoff, (size_t)nb * 8, cudaMemcpyHostToDevice, st));
    dim3 gc((u32)(((maxbits + 31) / 32 + 255) / 256), nb);
    ctx->prof_begin(K_CONCAT, maxbits / 4 * nb);
    k_concat_bits<<<gc, 256, 0, st>>>(H.d_out, H.out_stride, H.d_bits, ctx->d_bitoff.as<u64>(), (u32 *)d_out);
    LAUNCH_OK();
    BZ_CHECK(cudaStreamSynchronize(st));
    return BZ2B200_OK;
}
// dst = src shifted right by `phase` bits (0..7); dst must hold (nbits + phase + 7) / 8 + 8 zeroed-able bytes
int bz_shift_bits(bz2b200_ctx *ctx, const u8 *d_src, u64 nbits, int phase, u8 *d_dst) {
    cudaStream_t st = ctx->stream;
    size_t dst_bytes = (size_t)((nbits + phase + 7) / 8);
    BZ_CHECK(cudaMemsetAsync(d_dst, 0, (dst_bytes + 7) & ~(size_t)3, st));
    BZ_CHECK(ctx->d_bitoff.ensure(16));
    u64 h[2] = {nbits, (u64)phase};
    BZ_CHECK(cudaMemcpyAsync(ctx->d_bitoff.p, h, 16, cudaMemcpyHostToDevice, st));
    dim3 gc((u32)(((nbits + 31) / 32 + 255) / 256), 1);
    if (nbits) {
        ctx->prof_begin(K_CONCAT, nbits / 4);
        k_concat_bits<<<gc, 256, 0, st>>>(d_src, 0, ctx->d_bitoff.as<u64>(), ctx->d_bitoff.as<u64>() + 1, (u32 *)d_dst);
        LAUNCH_OK();
    }
    BZ_CHECK(cudaStreamSynchronize(st));
    return BZ2B200_OK;
}

u32 off_from_for(size_t n, int level, size_t window_pos) {
    // Position (window relative) after which a group leaves the reference's `remaining` counter one high at EOF:
    // the last short read happens when fewer than 260 bytes are left of the last full read (rle1.rs:63-85,:143).
    size_t Bsz = (size_t)level * 100000 - 19;
    size_t t_r = (n % Bsz != 0) ? (n / Bsz) * Bsz : n;
    size_t abs_from = t_r > 260 ? t_r - 260 : 0;
    return abs_from > window_pos ? (u32)std::min<size_t>(abs_from - window_pos, 0xFFFFFFF0u) : 0u;
}

// Host-buffer pipelining of one bz2b200_compress_stream call: the input arrives in chunks on an upload stream while
// earlier windows are being compressed, and finished output bytes leave on a download stream.
struct Pipe {
    cudaStream_t down;
    std::vector<cudaEvent_t> *up_ev;   // up_ev[i] fires when input bytes [0, (i+1)*chunk) are on the device
    size_t chunk;
    size_t waited;                     // upload events the compute stream already waits for
    u8 *h_out; size_t out_cap;
    size_t down_done;                  // output bytes already handed to the download stream
};

// Core: d_in[0..n) on the device -> d_out (device), both owned by the caller.
// If block_crcs != nullptr the stream header/footer are omitted and only blocks
// [first, first+count) of the sequence starting at d_in are emitted (multi-GPU range mode: d_in then
// points at the first block's first byte and n_is_eof says whether d_in+n is the end of the stream).
static int compress_core(bz2b200_ctx *ctx, const u8 *d_in, size_t n, int level, u8 *d_out, size_t out_cap,
                         u64 *out_bits, bool whole_stream, bool n_is_eof, size_t stream_n, size_t stream_pos,
                         u32 max_count, std::vector<u32> *crcs_out, size_t window = WINDOW, Pipe *pipe = nullptr) {
    cudaStream_t st = ctx->stream;
    if (out_cap < 16) return BZ2B200_E_CAP;
    if (ctx->timing) cudaEventRecord(ctx->ev_total[0], st);
    // the merge ORs bits into d_out: clear what this input can produce, not the caller's whole buffer
    BZ_CHECK(cudaMemsetAsync(d_out, 0, std::min(out_cap, (bz2b200_compress_bound(n) + 64) & ~(size_t)3), st));
    u64 bitpos = whole_stream ? 32 : 0;
    u32 combined = 0;
    size_t pos = 0;
    u32 done_blocks = 0;
    float t_rle = 0, t_bwt = 0, t_mtf = 0, t_huf = 0;
    u32 Bsz = (u32)level * 100000u - 19u;
    u32 stride = (((Bsz + 8) + 64 + BZ_TILE - 1) / BZ_TILE) * BZ_TILE;
    u32 batch_blocks = (u32)std::min<size_t>(MAX_BATCH_BLOCKS, std::max<size_t>(1, MAX_BATCH_BYTES / stride));
    std::vector<u64> hoff;
    while (pos < n && done_blocks < max_count) {
        size_t W = std::min(n - pos, window);
        if (n - pos - W < window / 2) W = std::min(n - pos, WINDOW);   // no small tail window
        bool eof = n_is_eof && (pos + W == n);
        Batch B;
        u32 nb = 0, consumed = 0;
        u32 want = std::min(batch_blocks, max_count - done_blocks);
        Arrival arr;
        if (pipe) {                                              // the RLE1 scan follows the upload chunk by chunk
            arr.ev = pipe->up_ev; arr.chunk = pipe->chunk; arr.win_off = pos; arr.waited = pipe->waited;
            ctx->arrival = &arr;
        }
        if (ctx->timing) cudaEventRecord(ctx->ev[4], st);
        int rc = bz_rle1_window(ctx, d_in + pos, (u32)W, level, eof, off_from_for(stream_n, level, stream_pos + pos),
                                want, B, &nb, &consumed, nullptr, false);
        if (pipe) { pipe->waited = arr.waited; ctx->arrival = nullptr; }
        if (rc) return rc;
        if (ctx->timing) { cudaEventRecord(ctx->ev[5], st); }
        if (nb == 0) { ctx->err = "rle1: window too small for one block"; return BZ2B200_E_ARG; }
        HufOut H;
        rc = bz_compress_batch(ctx, B, ctx->d_crc.as<u32>(), H);
        if (rc) return rc;
        if (ctx->timing) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[5]);
            t_rle += ms; t_bwt += ctx->stage_ms[1]; t_mtf += ctx->stage_ms[2]; t_huf += ctx->stage_ms[3];
        }
        // per-block bit lengths and CRCs -> offsets and combined CRC on the host (a few KB)
        BZ_CHECK(ctx->h_small.ensure((size_t)nb * 12 + 64));
        u64 *hbits = ctx->h_small.as<u64>();
        u32 *hcrc = (u32 *)(hbits + nb);
        BZ_CHECK(cudaMemcpyAsync(hbits, H.d_bits, (size_t)nb * 8, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaMemcpyAsync(hcrc, ctx->d_crc.p, (size_t)nb * 4, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaStreamSynchronize(st));
        hoff.resize(nb);
        u64 maxbits = 0;
        for (u32 k = 0; k < nb; k++) {
            if (hbits[k] == ~0ull) { ctx->err = "huffman: packed block exceeds its slot"; return BZ2B200_E_CAP; }
            hoff[k] = bitpos;
            bitpos += hbits[k];
            maxbits = std::max(maxbits, hbits[k]);
            combined = bz_crc_step(combined, hcrc[k]);   // bitwriter.rs:89-91
            if (crcs_out) crcs_out->push_back(hcrc[k]);
        }
        if ((bitpos + 80 + 7) / 8 + 8 > out_cap) return BZ2B200_E_CAP;
        BZ_CHECK(ctx->d_bitoff.ensure((size_t)nb * 8));
        BZ_CHECK(cudaMemcpyAsync(ctx->d_bitoff.p, hoff.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, st));
        dim3 gc((u32)(((maxbits + 31) / 32 + 255) / 256), nb);
        ctx->prof_begin(K_CONCAT, maxbits / 4 * nb); k_concat_bits<<<gc, 256, 0, st>>>(H.d_out, H.out_stride, H.d_bits, ctx->d_bitoff.as<u64>(), (u32 *)d_out);
        LAUNCH_OK();
        BZ_CHECK(cudaStreamSynchronize(st));                    // hoff is reused by the next batch
        if (pipe) {                                              // whole words below the bit position are final
            size_t fin = (size_t)(bitpos / 32) * 4;
            if (fin > pipe->out_cap) return BZ2B200_E_CAP;
            if (fin > pipe->down_done) {
                BZ_CHECK(cudaMemcpyAsync(pipe->h_out + pipe->down_done, d_out + pipe->down_done, fin - pipe->down_done,
                                         cudaMemcpyDeviceToHost, pipe->down));
                pipe->down_done = fin;
            }
        }
        pos += consumed;
        done_blocks += nb;
    }
    if (whole_stream) {
        ctx->prof_begin(K_FOOTER, 16); k_header_footer<<<1, 32, 0, st>>>((u32 *)d_out, level, bitpos, combined, 1); LAUNCH_OK();   // bitwriter.rs:103-114
        bitpos += 80;
    }
    if (ctx->timing) cudaEventRecord(ctx->ev_total[1], st);
    BZ_CHECK(cudaStreamSynchronize(st));
    *out_bits = bitpos;
    if (ctx->timing) cudaEventElapsedTime(&ctx->stage_ms[5], ctx->ev_total[0], ctx->ev_total[1]);
    if (ctx->timing) { ctx->stage_ms[0] = t_rle; ctx->stage_ms[1] = t_bwt; ctx->stage_ms[2] = t_mtf; ctx->stage_ms[3] = t_huf; }
    return BZ2B200_OK;
}

static int upload(bz2b200_ctx *ctx, const u8 *in, size_t n, DevBuf &buf) {
    BZ_CHECK(buf.ensure(n + 64));
    if (n) BZ_CHECK(cudaMemcpyAsync(buf.p, in, n, cudaMemcpyHostToDevice, ctx->stream));
    return BZ2B200_OK;
}

extern "C" {

size_t bz2b200_compress_bound(size_t n) {
    // worst case: incompressible data costs ~1.13 bytes per RLE1 byte plus ~1.4 KB of tables per block
    return n + n / 4 + (n / 99000 + 2) * 2048 + 4096;
}

int bz2b200_compress_stream_dev(bz2b200_ctx *ctx, const uint8_t *d_in, size_t n, int level, uint8_t *d_out,
                                size_t out_cap, size_t *out_len) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || (!d_in && n) || !d_out || !out_len || !bz_parse_level(&level, &mode)) return BZ2B200_E_ARG;
    if ((uintptr_t)d_out & 3u) return BZ2B200_E_ARG;            // the bit merge works on 32-bit words of d_out
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    u64 bits = 0;
    int rc = compress_core(ctx, d_in, n, level, d_out, out_cap & ~(size_t)3, &bits, true, true, n, 0, 0xFFFFFFFFu, nullptr);
    if (rc) return rc;
    *out_len = (size_t)((bits + 7) / 8);
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_compress_stream(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, uint8_t *out, size_t out_cap,
                            size_t *out_len) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || (!in && n) || !out || !out_len || !bz_parse_level(&level, &mode)) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    // knobs: windows per call (1 = upload everything, compress, download) and upload chunk size
    static const int n_windows = [] { const char *e = getenv("BZ2B200_E2E_WINDOWS"); int v = e ? atoi(e) : 1; return v < 1 ? 1 : v; }();
    static const size_t CHUNK = [] { const char *e = getenv("BZ2B200_E2E_CHUNK_MB"); int v = e ? atoi(e) : 8; return (size_t)(v < 1 ? 1 : v) << 20; }();
    size_t cap = bz2b200_compress_bound(n);
    BZ_CHECK(ctx->d_in.ensure(n + 64));
    BZ_CHECK(ctx->d_stream.ensure(cap + 64));
    if (!ctx->s_up) {
        BZ_CHECK(cudaStreamCreateWithFlags(&ctx->s_up, cudaStreamNonBlocking));
        BZ_CHECK(cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking));
    }
    size_t nchunks = (n + CHUNK - 1) / CHUNK;
    while (ctx->up_ev.size() < nchunks) {
        cudaEvent_t e;
        BZ_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->up_ev.push_back(e);
    }
    std::vector<cudaEvent_t> evs(ctx->up_ev.begin(), ctx->up_ev.begin() + nchunks);
    for (size_t i = 0; i < nchunks; i++) {
        size_t off = i * CHUNK, len = std::min(CHUNK, n - off);
        BZ_CHECK(cudaMemcpyAsync(ctx->d_in.as<u8>() + off, in + off, len, cudaMemcpyHostToDevice, ctx->s_up));
        BZ_CHECK(cudaEventRecord(evs[i], ctx->s_up));
    }
    Pipe pipe;
    pipe.down = ctx->s_down; pipe.up_ev = &evs; pipe.chunk = CHUNK; pipe.waited = 0;
    pipe.h_out = out; pipe.out_cap = out_cap; pipe.down_done = 0;
    // windows of whole MiB, at least 16 MiB each: small windows leave the GPU under-filled
    size_t window = WINDOW;
    if (n_windows > 1 && n > (32u << 20)) {
        window = std::max<size_t>(n / n_windows + (1u << 20), 16u << 20) & ~(size_t)0xFFFFF;
        if (window > WINDOW) window = WINDOW;
    }
    u64 bits = 0;
    int rc = compress_core(ctx, ctx->d_in.as<u8>(), n, level, ctx->d_stream.as<u8>(), cap & ~(size_t)3, &bits, true, true, n, 0,
                           0xFFFFFFFFu, nullptr, window, &pipe);
    if (rc) { cudaStreamSynchronize(ctx->s_up); cudaStreamSynchronize(ctx->s_down); return rc; }
    size_t len = (size_t)((bits + 7) / 8);
    if (len > out_cap) { cudaStreamSynchronize(ctx->s_down); return BZ2B200_E_CAP; }
    if (len > pipe.down_done)
        BZ_CHECK(cudaMemcpyAsync(out + pipe.down_done, ctx->d_stream.as<u8>() + pipe.down_done, len - pipe.down_done,
                                 cudaMemcpyDeviceToHost, ctx->s_down));
    // the stream header is written together with the footer, after the first words may already have left
    if (pipe.down_done) BZ_CHECK(cudaMemcpyAsync(out, ctx->d_stream.p, std::min<size_t>(4, len), cudaMemcpyDeviceToHost, ctx->s_down));
    BZ_CHECK(cudaStreamSynchronize(ctx->s_down));
    *out_len = len;
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_crc32(bz2b200_ctx *ctx, const uint8_t *data, size_t n, uint32_t *crc) {
    BZ_API_TRY
    if (!ctx || (!data && n) || !crc || n > 0xFFFFFF00u) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    int rc = upload(ctx, data, n, ctx->d_in);
    if (rc) return rc;
    BZ_CHECK(ctx->d_crc.ensure(64));
    rc = bz_crc_dev(ctx, ctx->d_in.as<u8>(), (u32)n, ctx->d_crc.as<u32>());
    if (rc) return rc;
    BZ_CHECK(cudaMemcpyAsync(crc, ctx->d_crc.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_rle1_split(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, uint8_t *rle1_out, size_t rle1_cap,
                       uint64_t *rle1_off, uint64_t *in_off, uint32_t *crc, uint32_t cap_blocks, uint32_t *nblocks) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || (!in && n) || !rle1_out || !rle1_off || !in_off || !crc || !nblocks || !bz_parse_level(&level, &mode))
        return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    int rc = upload(ctx, in, n, ctx->d_in);
    if (rc) return rc;
    size_t pos = 0, opos = 0;
    u32 total = 0;
    rle1_off[0] = 0; in_off[0] = 0;
    std::vector<u32> spans;
    while (pos < n) {
        size_t W = std::min(n - pos, WINDOW);
        bool eof = pos + W == n;
        Batch B; u32 nb = 0, consumed = 0;
        rc = bz_rle1_window(ctx, ctx->d_in.as<u8>() + pos, (u32)W, level, eof, off_from_for(n, level, pos), 256, B, &nb,
                            &consumed, &spans, false);
        if (rc) return rc;
        if (nb == 0) { ctx->err = "rle1: window too small for one block"; return BZ2B200_E_ARG; }
        if (total + nb > cap_blocks) return BZ2B200_E_CAP;
        BZ_CHECK(cudaMemcpyAsync(crc + total, ctx->d_crc.p, (size_t)nb * 4, cudaMemcpyDeviceToHost, ctx->stream));
        for (u32 k = 0; k < nb; k++) {
            u32 s = spans[4 * k], e = spans[4 * k + 1], ol = spans[4 * k + 2];
            (void)s;
            if (opos + ol > rle1_cap) return BZ2B200_E_CAP;
            BZ_CHECK(cudaMemcpyAsync(rle1_out + opos, B.T + (size_t)k * B.stride, ol, cudaMemcpyDeviceToHost, ctx->stream));
            opos += ol;
            rle1_off[total + k + 1] = opos;
            in_off[total + k + 1] = pos + e;
        }
        BZ_CHECK(cudaStreamSynchronize(ctx->stream));
        total += nb;
        pos += consumed;
    }
    *nblocks = total;
    return BZ2B200_OK;
    BZ_API_CATCH
}

// ---- multi-GPU sharding helpers (SURVEY 8e) -------------------------------------------------------------
int bz2b200_stream_plan(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, uint64_t *block_start, uint32_t cap,
                        uint32_t *nblocks) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || (!in && n) || !block_start || !nblocks || !bz_parse_level(&level, &mode)) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    // plan window by window; only the window being planned has to be resident
    size_t pos = 0;
    u32 total = 0;
    std::vector<u32> spans;
    while (pos < n) {
        size_t W = std::min(n - pos, WINDOW);
        bool eof = pos + W == n;
        BZ_CHECK(ctx->d_in.ensure(W + 64));
        BZ_CHECK(cudaMemcpyAsync(ctx->d_in.p, in + pos, W, cudaMemcpyHostToDevice, ctx->stream));
        Batch B; u32 nb = 0, consumed = 0;
        int rc = bz_rle1_window(ctx, ctx->d_in.as<u8>(), (u32)W, level, eof, off_from_for(n, level, pos), MAX_BATCH_BLOCKS,
                                B, &nb, &consumed, &spans, true);
        if (rc) return rc;
        if (nb == 0) { ctx->err = "rle1: window too small for one block"; return BZ2B200_E_ARG; }
        if (total + nb + 1 > cap) return BZ2B200_E_CAP;
        for (u32 k = 0; k < nb; k++) block_start[total + k] = pos + spans[4 * k];
        total += nb;
        pos += consumed;
    }
    block_start[total] = n;
    *nblocks = total;
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_compress_range(bz2b200_ctx *ctx, const uint8_t *in, size_t n, int level, const uint64_t *block_start,
                           uint32_t nblocks_total, uint32_t first, uint32_t count, uint8_t *out, size_t out_cap,
                           uint64_t *out_bits, uint32_t *block_crcs) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || !in || !block_start || !out || !out_bits || !block_crcs || !bz_parse_level(&level, &mode) ||
        first + count > nblocks_total)
        return BZ2B200_E_ARG;
    *out_bits = 0;
    if (count == 0) return BZ2B200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    size_t a = (size_t)block_start[first], b = (size_t)block_start[first + count];
    bool to_eof = (first + count == nblocks_total);
    // the chain needs look-ahead past the last block's end to reproduce its boundary
    size_t hi = to_eof ? n : std::min(n, b + 4096);
    bool eof = hi == n;
    int rc = upload(ctx, in + a, hi - a, ctx->d_in);
    if (rc) return rc;
    size_t cap = bz2b200_compress_bound(b - a);
    BZ_CHECK(ctx->d_stream.ensure(cap + 64));
    std::vector<u32> crcs;
    u64 bits = 0;
    rc = compress_core(ctx, ctx->d_in.as<u8>(), hi - a, level, ctx->d_stream.as<u8>(), cap & ~(size_t)3, &bits, false, eof, n, a,
                       count, &crcs);
    if (rc) return rc;
    if (crcs.size() != count) { ctx->err = "compress_range: block plan mismatch"; return BZ2B200_E_ARG; }
    size_t len = (size_t)((bits + 7) / 8);
    if (len > out_cap) return BZ2B200_E_CAP;
    BZ_CHECK(cudaMemcpyAsync(out, ctx->d_stream.p, len, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    memcpy(block_crcs, crcs.data(), (size_t)count * 4);
    *out_bits = bits;
    return BZ2B200_OK;
    BZ_API_CATCH
}

// Host-side ordered merge of bit strings (the writer thread of compress.rs:74-122 + bitwriter.rs:77-132).
int bz2b200_merge_streams(int level, int nparts, const uint8_t *const *part, const uint64_t *part_bits,
                          const uint32_t *const *part_crcs, const uint32_t *part_ncrc, uint8_t *out, size_t out_cap,
                          size_t *out_len) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!bz_parse_level(&level, &mode) || nparts < 0 || !out || !out_len) return BZ2B200_E_ARG;
    u64 total = 32 + 80;
    for (int i = 0; i < nparts; i++) total += part_bits[i];
    size_t len = (size_t)((total + 7) / 8);
    if (len > out_cap) return BZ2B200_E_CAP;
    memset(out, 0, len);
    out[0] = 'B'; out[1] = 'Z'; out[2] = 'h'; out[3] = (uint8_t)('0' + level);
    u64 pos = 32;
    u32 combined = 0;
    for (int i = 0; i < nparts; i++) {
        for (u32 k = 0; k < part_ncrc[i]; k++) combined = bz_crc_step(combined, part_crcs[i][k]);
        u64 nb = part_bits[i];
        size_t nbytes = (size_t)((nb + 7) / 8);
        int sh = (int)(pos & 7);
        uint8_t *d = out + (pos >> 3);
        const uint8_t *s = part[i];
        if (nbytes == 0) continue;
        if (sh == 0) {
            // last source byte may carry padding zeros only, so OR-ing the seam byte and copying the rest is exact
            d[0] |= s[0];
            if (nbytes > 1) memcpy(d + 1, s + 1, nbytes - 1);
        } else {
            // 8 source bytes per step: big-endian 64-bit word shifted right by sh, the spill goes to the next byte
            size_t j = 0;
            uint8_t carry = 0;                             // low `sh` bits of the previous source byte, left aligned
            d[0] |= (uint8_t)(s[0] >> sh);
            carry = (uint8_t)(s[0] << (8 - sh));
            j = 1;
            for (; j + 8 <= nbytes; j += 8) {
                u64 w;
                memcpy(&w, s + j, 8);
                w = __builtin_bswap64(w);
                u64 o = ((u64)carry << 56) | (w >> sh);
                carry = (uint8_t)(w << (8 - sh));
                o = __builtin_bswap64(o);
                memcpy(d + j, &o, 8);                      // bytes d[1..] of this part are still zero: plain stores
            }
            for (; j < nbytes; j++) {
                d[j] = (uint8_t)(carry | (s[j] >> sh));
                carry = (uint8_t)(s[j] << (8 - sh));
            }
            d[nbytes] |= carry;                            // bits past `nb` are zero in the source
        }
        pos += nb;
    }
    const uint8_t foot[10] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90, (uint8_t)(combined >> 24), (uint8_t)(combined >> 16),
                              (uint8_t)(combined >> 8), (uint8_t)combined};
    int sh = (int)(pos & 7);
    uint8_t *d = out + (pos >> 3);
    for (int j = 0; j < 10; j++) {
        d[j] |= (uint8_t)(foot[j] >> sh);
        if (sh) d[j + 1] |= (uint8_t)(foot[j] << (8 - sh));
    }
    *out_len = len;
    return BZ2B200_OK;
    BZ_API_CATCH
}

}  // extern "C"

// ---- device-resident variants of the sharding helpers (HBM-resident measurement at N > 1) --------------
extern "C" int bz2b200_stream_plan_dev(bz2b200_ctx *ctx, const uint8_t *d_in, size_t n, int level,
                                       uint64_t *block_start, uint32_t cap, uint32_t *nblocks) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || (!d_in && n) || !block_start || !nblocks || !bz_parse_level(&level, &mode)) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    size_t pos = 0;
    u32 total = 0;
    std::vector<u32> spans;
    while (pos < n) {
        size_t W = std::min(n - pos, WINDOW);
        bool eof = pos + W == n;
        Batch B; u32 nb = 0, consumed = 0;
        int rc = bz_rle1_window(ctx, d_in + pos, (u32)W, level, eof, off_from_for(n, level, pos), MAX_BATCH_BLOCKS, B, &nb,
                                &consumed, &spans, true);
        if (rc) return rc;
        if (nb == 0) { ctx->err = "rle1: window too small for one block"; return BZ2B200_E_ARG; }
        if (total + nb + 1 > cap) return BZ2B200_E_CAP;
        for (u32 k = 0; k < nb; k++) block_start[total + k] = pos + spans[4 * k];
        total += nb;
        pos += consumed;
    }
    block_start[total] = n;
    *nblocks = total;
    return BZ2B200_OK;
    BZ_API_CATCH
}

extern "C" int bz2b200_compress_range_dev(bz2b200_ctx *ctx, const uint8_t *d_in, size_t n, int level,
                                          const uint64_t *block_start, uint32_t nblocks_total, uint32_t first,
                                          uint32_t count, uint8_t *d_out, size_t out_cap, uint64_t *out_bits,
                                          uint32_t *block_crcs) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || !d_in || !block_start || !d_out || !out_bits || !block_crcs || !bz_parse_level(&level, &mode) ||
        first + count > nblocks_total || ((uintptr_t)d_out & 3u))
        return BZ2B200_E_ARG;
    *out_bits = 0;
    if (count == 0) return BZ2B200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    size_t a = (size_t)block_start[first], b = (size_t)block_start[first + count];
    bool to_eof = (first + count == nblocks_total);
    size_t hi = to_eof ? n : std::min(n, b + 4096);
    std::vector<u32> crcs;
    u64 bits = 0;
    int rc = compress_core(ctx, d_in + a, hi - a, level, d_out, out_cap & ~(size_t)3, &bits, false, hi == n, n, a, count,
                           &crcs);
    if (rc) return rc;
    if (crcs.size() != count) { ctx->err = "compress_range: block plan mismatch"; return BZ2B200_E_ARG; }
    memcpy(block_crcs, crcs.data(), (size_t)count * 4);
    *out_bits = bits;
    return BZ2B200_OK;
    BZ_API_CATCH
}
