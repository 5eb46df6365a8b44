// zstream.cu -- streaming compression: input arrives in pieces, finished .bz2 bytes leave through a callback.
//
// The reference's `compress` (src/compression/compress.rs:40-136) never holds the file: RLE1Block reads block_size
// bytes per refill (src/tools/rle1.rs:63-85), rayon workers compress blocks while the iterator reads on, and a writer
// thread appends finished blocks in order (compress.rs:74-122).  bz2b200_compress_stream needs the whole input in one
// buffer; this is the pipelined form of the same function:
//   caller thread   bz2b200_zstream_write copies the caller's bytes into one of two page-locked staging buffers
//   worker thread   when a staging buffer is full (a "window" of 64 MiB): H2D behind the unconsumed tail of the
//                   previous window, RLE1 scan + block chain + all block kernels (bz_rle1_window, bz_compress_batch),
//                   bit-granular concatenation behind the carried partial byte, D2H, sink() with the finished bytes
// so reading / producing the next window overlaps upload, kernels, download and the sink's write of the previous one.
// Blocks never straddle a call: the bytes after the last complete block (the chain needs look-ahead, rle1.rs:29) stay
// on the device as the head of the next window.  The bytes are exactly those of bz2b200_compress_stream for the
// concatenated input, whatever the piece sizes (the EOF corner of the splitter needs the total length, which is known
// when the last window is planned).
#include "common.cuh"
#include <algorithm>
#include <condition_variable>
#include <memory>
#include <stdlib.h>
#include <string.h>
#include <thread>

u32 off_from_for(size_t n, int level, size_t window_pos);
int bz_concat_blocks(bz2b200_ctx *ctx, const HufOut &H, u32 nb, const u64 *hoff, u64 maxbits, u8 *d_out);

struct bz2b200_zstream {
    bz2b200_ctx *ctx = nullptr;
    int level = 9;
    int mode = BZ_MODE_REF;
    bz2b200_sink sink = nullptr;
    void *user = nullptr;
    size_t WF = 64u << 20;                   // fresh bytes per window
    PinBuf stage[2];
    int cur = 0;                             // staging buffer the caller fills
    size_t fill = 0;
    // worker
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    bool busy = false, quit = false;
    int job_slot = 0; size_t job_len = 0; bool job_eof = false;
    int rc = BZ2B200_OK;                     // sticky
    std::string err;
    // device / stream state (worker only)
    DevBuf d_in[2];
    int dcur = 0;
    size_t tail_off = 0, tail_len = 0;       // unconsumed bytes of the previous window: d_in[dcur] + tail_off
    u64 abs_pos = 0;                         // stream offset of the first unconsumed byte
    DevBuf d_out;
    PinBuf h_out;
    u64 bitpos = 32;                         // bits written so far (header included)
    u32 combined = 0;
    u8 carry = 0;                            // the partial last byte (bitpos % 8 bits are valid)
    u64 total_in = 0, total_out = 0;
};

namespace {

int emit(bz2b200_zstream *z, const u8 *p, size_t n) {
    if (n == 0) return BZ2B200_OK;
    z->total_out += n;
    if (z->sink(z->user, p, n) != 0) { z->err = "the sink reported an error"; return BZ2B200_E_ARG; }
    return BZ2B200_OK;
}

// one window: the previous tail + `len` fresh bytes from staging buffer `slot`
int process(bz2b200_zstream *z, int slot, size_t len, bool eof) {
    bz2b200_ctx *ctx = z->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = z->mode;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    cudaStream_t st = ctx->stream;
    const size_t W = z->tail_len + len;
    if (W > 0xFFFFFF00ull) { z->err = "zstream: a block spans more than 4 GiB of input"; return BZ2B200_E_ARG; }
    z->total_in += len;
    if (W) {
        // the new window = [tail of the previous one | fresh bytes] in the other device buffer
        DevBuf &nw = z->d_in[z->dcur ^ 1];
        BZ_CHECK(nw.ensure(W + 64));
        if (z->tail_len) BZ_CHECK(cudaMemcpyAsync(nw.p, z->d_in[z->dcur].as<u8>() + z->tail_off, z->tail_len, cudaMemcpyDeviceToDevice, st));
        if (len) BZ_CHECK(cudaMemcpyAsync(nw.as<u8>() + z->tail_len, z->stage[slot].p, len, cudaMemcpyHostToDevice, st));
        z->dcur ^= 1;
        z->tail_off = 0; z->tail_len = W;
        Batch B;
        u32 nb = 0, consumed = 0;
        u32 off_from = eof ? off_from_for((size_t)z->total_in, z->level, (size_t)z->abs_pos) : 0xFFFFFFF0u;
        int rc = bz_rle1_window(ctx, nw.as<u8>(), (u32)W, z->level, eof, off_from, 4096, B, &nb, &consumed, nullptr, false);
        if (rc) { z->err = ctx->err; return rc; }
        if (nb == 0) {
            if (eof) { z->err = "zstream: the final window produced no block"; return BZ2B200_E_ARG; }
            return BZ2B200_OK;                                  // one block needs more input than this window holds: wait for more
        }
        HufOut H;
        rc = bz_compress_batch(ctx, B, ctx->d_crc.as<u32>(), H);
        if (rc) { z->err = ctx->err; return rc; }
        BZ_CHECK(ctx->h_small.ensure((size_t)nb * 12 + 64));
        u64 *hbits = ctx->h_small.as<u64>();
        u32 *hcrc = (u32 *)(hbits + nb);
        BZ_CHECK(cudaMemcpyAsync(hbits, H.d_bits, (size_t)nb * 8, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaMemcpyAsync(hcrc, ctx->d_crc.p, (size_t)nb * 4, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaStreamSynchronize(st));
        const u32 phase = (u32)(z->bitpos & 7);
        std::vector<u64> hoff(nb);
        u64 pos = phase, maxbits = 0;
        for (u32 k = 0; k < nb; k++) {
            if (hbits[k] == ~0ull) { z->err = "huffman: packed block exceeds its slot"; return BZ2B200_E_CAP; }
            hoff[k] = pos; pos += hbits[k]; maxbits = std::max(maxbits, hbits[k]);
            z->combined = bz_crc_step(z->combined, hcrc[k]);    // bitwriter.rs:89-91
        }
        const size_t nbytes = (size_t)((pos + 7) / 8);
        BZ_CHECK(z->d_out.ensure(nbytes + 64));
        BZ_CHECK(z->h_out.ensure(nbytes + 64));
        BZ_CHECK(cudaMemsetAsync(z->d_out.p, 0, (nbytes + 8) & ~(size_t)3, st));
        rc = bz_concat_blocks(ctx, H, nb, hoff.data(), maxbits, z->d_out.as<u8>());
        if (rc) { z->err = ctx->err; return rc; }
        BZ_CHECK(cudaMemcpyAsync(z->h_out.p, z->d_out.p, nbytes, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaStreamSynchronize(st));
        u8 *ho = z->h_out.as<u8>();
        ho[0] |= z->carry;                                      // the bits the previous window left in its last byte
        const size_t full = (size_t)(pos / 8);
        z->carry = (pos & 7) ? ho[full] : 0;
        z->bitpos += pos - phase;
        rc = emit(z, ho, full);
        if (rc) return rc;
        z->tail_off = consumed; z->tail_len = W - consumed;
        z->abs_pos += consumed;
    }
    if (eof) {
        if (z->tail_len) { z->err = "zstream: input left over after the last block"; return BZ2B200_E_ARG; }
        // footer (bitwriter.rs:103-114) behind the carried bits
        const u32 c = z->combined;
        const u8 foot[10] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90, (u8)(c >> 24), (u8)(c >> 16), (u8)(c >> 8), (u8)c};
        const int sh = (int)(z->bitpos & 7);
        u8 tailb[11] = {z->carry, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int j = 0; j < 10; j++) {
            tailb[j] |= (u8)(foot[j] >> sh);
            if (sh) tailb[j + 1] |= (u8)(foot[j] << (8 - sh));
        }
        z->bitpos += 80;
        int rc = emit(z, tailb, sh ? 11 : 10);
        if (rc) return rc;
    }
    return BZ2B200_OK;
}

void worker(bz2b200_zstream *z) {
    for (;;) {
        int slot; size_t len; bool eof;
        {
            std::unique_lock<std::mutex> lk(z->mu);
            z->cv.wait(lk, [&] { return z->busy || z->quit; });
            if (!z->busy) return;
            slot = z->job_slot; len = z->job_len; eof = z->job_eof;
        }
        int rc;
        try { rc = process(z, slot, len, eof); } catch (...) { rc = BZ2B200_E_NOMEM; z->err = "out of memory"; }
        {
            std::lock_guard<std::mutex> lk(z->mu);
            if (rc && z->rc == BZ2B200_OK) z->rc = rc;
            z->busy = false;
        }
        z->cv.notify_all();
    }
}

// hands the staging buffer to the worker once the previous window is done
int submit(bz2b200_zstream *z, bool eof) {
    std::unique_lock<std::mutex> lk(z->mu);
    z->cv.wait(lk, [&] { return !z->busy; });
    if (z->rc) return z->rc;
    z->job_slot = z->cur; z->job_len = z->fill; z->job_eof = eof;
    z->busy = true;
    z->cur ^= 1; z->fill = 0;
    lk.unlock();
    z->cv.notify_all();
    return BZ2B200_OK;
}

}  // namespace

extern "C" {

int bz2b200_zstream_open(bz2b200_ctx *ctx, int level, bz2b200_sink sink, void *user, bz2b200_zstream **out) {
    BZ_API_TRY
    int mode = BZ_MODE_REF;
    if (!ctx || !sink || !out || !bz_parse_level(&level, &mode)) return BZ2B200_E_ARG;
    *out = nullptr;
    std::unique_ptr<bz2b200_zstream> z(new bz2b200_zstream());
    z->ctx = ctx; z->level = level; z->mode = mode; z->sink = sink; z->user = user;
    if (const char *e = getenv("BZ2B200_ZSTREAM_WINDOW_MB")) { int v = atoi(e); if (v >= 1 && v <= 1024) z->WF = (size_t)v << 20; }
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    for (int i = 0; i < 2; i++) if (z->stage[i].ensure(z->WF) != cudaSuccess) return BZ2B200_E_NOMEM;
    const u8 head[4] = {'B', 'Z', 'h', (u8)('0' + level)};      // bitwriter.rs:67-72
    int rc = emit(z.get(), head, 4);
    if (rc) return rc;
    z->th = std::thread(worker, z.get());
    *out = z.release();
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_zstream_write(bz2b200_zstream *z, const uint8_t *data, size_t n) {
    BZ_API_TRY
    if (!z || (!data && n)) return BZ2B200_E_ARG;
    while (n) {
        size_t take = std::min(n, z->WF - z->fill);
        memcpy(z->stage[z->cur].as<u8>() + z->fill, data, take);
        z->fill += take; data += take; n -= take;
        if (z->fill == z->WF) {
            int rc = submit(z, false);
            if (rc) return rc;
        }
    }
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_zstream_close(bz2b200_zstream *z, uint64_t *total_in, uint64_t *total_out) {
    if (!z) return BZ2B200_E_ARG;
    int rc;
    try { rc = submit(z, true); } catch (...) { rc = BZ2B200_E_NOMEM; }
    {
        std::unique_lock<std::mutex> lk(z->mu);
        z->cv.wait(lk, [&] { return !z->busy; });
        if (rc == BZ2B200_OK) rc = z->rc;
        z->quit = true;
    }
    z->cv.notify_all();
    if (z->th.joinable()) z->th.join();
    if (total_in) *total_in = z->total_in;
    if (total_out) *total_out = z->total_out;
    if (rc) z->ctx->err = "zstream: " + z->err;
    cudaSetDevice(z->ctx->device);
    for (int i = 0; i < 2; i++) { z->stage[i].release(); z->d_in[i].release(); }
    z->d_out.release(); z->h_out.release();
    delete z;
    return rc;
}

}  // extern "C"
