// dstream.cu -- streaming decompression: a .bz2 input arrives in pieces, decoded bytes leave through a callback.
//
// bz2b200_decompress_stream needs the whole input in one buffer and an output buffer for everything it decodes to.
// A dstream is the same decode core (bz_decode_core, decode.cu) driven window by window from one context:
//   caller thread    bz2b200_dstream_write copies the caller's bytes into one of two page-locked staging buffers
//   worker thread    when a staging buffer holds WF fresh bytes (a "window", 64 MiB): uploads [carried tail | fresh
//                    bytes], finds the magic candidates and decodes the chain elements that start before the window's
//                    decode edge, end - LOOK; each decoded batch passes its block CRCs on the device
//   delivery thread  copies every checked batch down (ctx->s_down) in page-locked pieces of 32 MiB and calls the sink
//                    on one piece while the next one downloads and the next batch decodes
// so reading the input overlaps upload and kernels, and the sink's writing overlaps download and kernels.
// Window edges depend only on absolute input positions: window k ends at byte (k + 1) * WF (or at the input's end).
// LOOK (4 MiB) exceeds the bound on a block's span, 20 x (900000 + 64) + 2^19 bits ~ 2.3 MB, so an element that starts
// before the edge ends inside the window, and a footer before the edge is never taken for the end of the input.
// The bytes from where the chain leaves the window onward (at most LOOK + 1) are carried in front of the next window;
// a window whose edge is not past the chain's start is carried whole and waits for more input.
// The chain's start and the stream's running combined CRC are always known here, so every footer's combined CRC is
// checked when it is reached.  Blocks are decoded with level-9 geometry; the rule that a block is at most 100000 x the
// level of its own stream's header is applied to each window's blocks once the window is decoded.  Host memory is the
// staging buffers and the output pieces whatever the input or output size; device memory is the decode workspaces, one
// window and two batch outputs.  In test mode (no sink) nothing is downloaded.
#include "common.cuh"
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <memory>
#include <stdlib.h>
#include <string.h>
#include <thread>

namespace {
const size_t LOOK = 4u << 20;            // look-ahead behind a window's decode edge (the multi decoder's)
const size_t PREFIX = LOOK + 64;         // room in front of each staging buffer for the carried tail
const size_t PIECE = 32u << 20;          // page-locked output piece
inline u32 crc_step(u32 s, u32 b) { return ((s << 1) | (s >> 31)) ^ b; }   // crc.rs:25-27
}  // namespace

struct bz2b200_dstream {
    bz2b200_ctx *ctx = nullptr;
    bz2b200_sink sink = nullptr;             // nullptr: test mode
    void *user = nullptr;
    size_t WF = 64u << 20;                   // fresh bytes per window
    bool chance = false;                     // BZ2B200_MULTI_DEC_CHANCE test knob
    PinBuf *stage = nullptr;                 // [2] (the context's): [PREFIX: carried tail, right-aligned | WF fresh bytes]
    int cur = 0;                             // staging buffer the caller fills
    size_t fill = 0;
    std::thread th, th_out;
    std::mutex mu;                           // guards everything below up to the worker state, and the delivery queue
    std::condition_variable cv;
    bool busy = false, quit = false;
    int job_slot = 0; size_t job_len = 0; bool job_eof = false;
    int rc = BZ2B200_OK;                     // sticky
    std::string err;
    // delivery
    struct Job { const u8 *d; u64 n; };
    std::deque<Job> jobs;
    u64 queued = 0, delivered = 0;           // batches handed to / finished by the delivery thread
    bool out_quit = false;
    bool out_failed = false;                 // the sink or a download failed: the sink receives nothing more
    PinBuf *piece = nullptr;                 // [2] (the context's)
    cudaEvent_t ev_piece[2] = {nullptr, nullptr};
    // worker state
    DevBuf *d_win = nullptr, *d_dec = nullptr;   // the context's: one window, two batch outputs ([2])
    u64 nbatch = 0;                          // batches counted so far (d_dec[nbatch & 1] is the next one's)
    size_t tail_len = 0; u64 tail_lo = 0;    // carried bytes in front of the next staging buffer, and their input offset
    long long expect = 32;                   // absolute bit where the next chain element starts
    u32 combined = 0;                        // running combined CRC of the current stream
    bool ended = false;                      // the chain ended after the input's last footer
    int level = 0;                           // level of the current stream's header (0: none seen yet)
    std::vector<u64> cand;
    std::vector<DecEvent> ev;
    u64 total_in = 0, total_out = 0;
};

namespace {

// where the worker's decoded batches go
struct DSink : DecSink {
    bz2b200_dstream *d;
    bz2b200_ctx *ctx;
    long long end = -1;
    void chain_end(long long bit) override { end = bit; }
    int counted(u64 nbytes, bool, u8 **d_out, u8 **h_out) override {
        if (d->sink) {                       // back-pressure: the batch that last used this buffer has been delivered
            std::unique_lock<std::mutex> lk(d->mu);
            d->cv.wait(lk, [&] { return d->rc != BZ2B200_OK || d->nbatch <= d->delivered + 1; });
            if (d->rc) return d->rc;
        }
        DevBuf &b = d->d_dec[d->nbatch & 1];
        BZ_CHECK(b.ensure((size_t)nbytes + 64));
        d->nbatch++;
        *d_out = b.as<u8>();
        *h_out = nullptr;
        return BZ2B200_OK;
    }
    int ready(const u8 *d_out, u64 nbytes) override {           // the batch passed its block CRCs
        d->total_out += nbytes;
        if (!d->sink) return BZ2B200_OK;
        {
            std::lock_guard<std::mutex> lk(d->mu);
            d->jobs.push_back({d_out, nbytes});
            d->queued++;
        }
        d->cv.notify_all();
        return BZ2B200_OK;
    }
};

// the bytes from input offset `from` to the window's end go in front of the next staging buffer
int carry(bz2b200_dstream *d, int slot, const u8 *h, u64 lo, size_t W, u64 from) {
    if (from < lo || from > lo + W || lo + W - from > PREFIX) { d->ctx->err = "decode: lost the block chain"; return BZ2B200_E_FORMAT; }
    const size_t t = (size_t)(lo + W - from);
    memcpy(d->stage[slot ^ 1].as<u8>() + PREFIX - t, h + (from - lo), t);   // the caller fills that buffer from PREFIX on
    d->tail_lo = from; d->tail_len = t;
    return BZ2B200_OK;
}

// one window: the carried tail + `len` fresh bytes of staging buffer `slot`
int process(bz2b200_dstream *d, int slot, size_t len, bool eof) {
    bz2b200_ctx *ctx = d->ctx;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    cudaStream_t st = ctx->stream;
    d->total_in += len;
    const u8 *h = d->stage[slot].as<u8>() + PREFIX - d->tail_len;
    const size_t W = d->tail_len + len;
    const u64 lo = d->tail_lo, end = lo + W;
    if (d->level == 0) {                                        // the first window (>= 1024 bytes unless it is the last)
        if (eof && d->total_in < 14) { ctx->err = "the input is shorter than 14 bytes"; return BZ2B200_E_FORMAT; }
        if (h[0] != 'B' || h[1] != 'Z' || h[2] != 'h' || h[3] < '1' || h[3] > '9') { ctx->err = "the input does not start with BZh<level>"; return BZ2B200_E_FORMAT; }
        d->level = h[3] - '0';
    }
    const u64 hi = eof ? ~0ull : (end > LOOK ? (u64)(end - LOOK) * 8 : 0);
    if (!eof && hi <= (u64)d->expect) return carry(d, slot, h, lo, W, (u64)d->expect / 8);   // wait for more input
    BZ_CHECK(d->d_win->ensure(W + 64));
    u8 *dw = d->d_win->as<u8>();
    BZ_CHECK(cudaMemcpyAsync(dw, h, W, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemsetAsync(dw + W, 0, 64, st));              // word loads of the entropy stage read past the last byte
    // at most one magic per 32 bits whatever the data: a window is never refused where the whole input is accepted
    int rc = bz_dec_candidates(ctx, dw, W, (u32)std::min<size_t>(W / 4 + 64, 0x7fffff00u), d->cand);
    if (rc) return rc;
    if (d->chance) bz_add_chance_candidates(d->cand);
    DecWindow w{h, (size_t)lo, (size_t)end, dw, (size_t)lo, W, hi, d->expect, d->combined, BZ2B200_MAX_BLOCK, &d->cand};
    DSink sink;
    sink.d = d; sink.ctx = ctx;
    d->ev.clear();
    rc = bz_decode_core(ctx, w, sink, d->ev);
    if (rc) return rc;
    rc = bz_check_block_sizes(ctx->err, d->level, d->ev);
    if (rc) return rc;
    for (const DecEvent &e : d->ev) {
        if (e.kind == DEC_BLOCK) {
            d->combined = crc_step(d->combined, e.val);
        } else if (e.kind == DEC_STREAM) {
            d->combined = 0;
            d->level = (int)e.val;
        }
    }
    if (eof) {
        if (sink.end != DEC_ENDED) { ctx->err = "decode: the input does not end with a stream footer"; return BZ2B200_E_FORMAT; }
        d->ended = true;
        return BZ2B200_OK;
    }
    // a footer before the edge ends at least LOOK - 11 bytes before the window's end: never the end of the input
    if (sink.end < 0 || sink.end == DEC_ENDED) { ctx->err = "decode: trailing bytes after the stream footer"; return BZ2B200_E_FORMAT; }
    d->expect = sink.end;
    return carry(d, slot, h, lo, W, (u64)sink.end / 8);
}

void worker(bz2b200_dstream *d) {
    for (;;) {
        int slot; size_t len; bool eof;
        {
            std::unique_lock<std::mutex> lk(d->mu);
            d->cv.wait(lk, [&] { return d->busy || d->quit; });
            if (!d->busy) return;
            slot = d->job_slot; len = d->job_len; eof = d->job_eof;
        }
        int rc;
        try { rc = process(d, slot, len, eof); } catch (...) { rc = BZ2B200_E_NOMEM; d->ctx->err = "out of memory"; }
        if (rc) cudaStreamSynchronize(d->ctx->stream);         // no copy may still read the staging buffer the caller refills
        {
            std::lock_guard<std::mutex> lk(d->mu);
            if (rc && d->rc == BZ2B200_OK) { d->rc = rc; d->err = d->ctx->err; }
            d->busy = false;
        }
        d->cv.notify_all();
    }
}

// one batch to the sink: piece i downloads while the sink takes piece i - 1
int deliver(bz2b200_dstream *d, const u8 *src, u64 n) {
    cudaStream_t s = d->ctx->s_down;
    int rc = BZ2B200_OK;
    u64 prev = 0;
    for (u64 off = 0, i = 0; off < n || prev; i++) {
        u64 sz = std::min<u64>(PIECE, n - off);
        if (sz) {
            if (cudaMemcpyAsync(d->piece[i & 1].p, src + off, (size_t)sz, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                cudaEventRecord(d->ev_piece[i & 1], s) != cudaSuccess) { rc = BZ2B200_E_CUDA; break; }
            off += sz;
        }
        if (prev) {
            if (cudaEventSynchronize(d->ev_piece[(i - 1) & 1]) != cudaSuccess) { rc = BZ2B200_E_CUDA; break; }
            if (d->sink(d->user, d->piece[(i - 1) & 1].as<u8>(), (size_t)prev) != 0) { rc = BZ2B200_E_ARG; break; }
        }
        prev = sz;
    }
    cudaStreamSynchronize(s);                                   // also after an error: the pieces stay untouched
    return rc;
}

void delivery(bz2b200_dstream *d) {
    cudaSetDevice(d->ctx->device);
    for (;;) {
        bz2b200_dstream::Job j;
        bool skip;
        {
            std::unique_lock<std::mutex> lk(d->mu);
            d->cv.wait(lk, [&] { return !d->jobs.empty() || d->out_quit; });
            if (d->jobs.empty()) return;
            j = d->jobs.front(); d->jobs.pop_front();
            skip = d->out_failed;       // a decode error leaves the batches checked before it to be delivered
        }
        int rc = skip ? BZ2B200_OK : deliver(d, j.d, j.n);
        {
            std::lock_guard<std::mutex> lk(d->mu);
            if (rc) d->out_failed = true;
            if (rc && d->rc == BZ2B200_OK) {
                d->rc = rc;
                d->err = rc == BZ2B200_E_ARG ? "the sink reported an error" : "download of a decoded batch failed";
            }
            d->delivered++;
        }
        d->cv.notify_all();
    }
}

// hands the staging buffer to the worker once the previous window is done
int submit(bz2b200_dstream *d, bool eof) {
    std::unique_lock<std::mutex> lk(d->mu);
    d->cv.wait(lk, [&] { return !d->busy; });
    if (d->rc) return d->rc;
    d->job_slot = d->cur; d->job_len = d->fill; d->job_eof = eof;
    d->busy = true;
    d->cur ^= 1; d->fill = 0;
    lk.unlock();
    d->cv.notify_all();
    return BZ2B200_OK;
}

// stops both threads (after the worker's window and every queued batch); the buffers stay with the context
void finish(bz2b200_dstream *d) {
    {
        std::unique_lock<std::mutex> lk(d->mu);
        d->cv.wait(lk, [&] { return !d->busy && d->delivered == d->queued; });
        d->quit = d->out_quit = true;
    }
    d->cv.notify_all();
    if (d->th.joinable()) d->th.join();
    if (d->th_out.joinable()) d->th_out.join();
    bz2b200_ctx *ctx = d->ctx;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->s_hi) cudaStreamSynchronize(ctx->s_hi);
    for (int i = 0; i < 2; i++) if (d->ev_piece[i]) cudaEventDestroy(d->ev_piece[i]);
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->dstream_open = false;
}

}  // namespace

extern "C" {

int bz2b200_dstream_open(bz2b200_ctx *ctx, bz2b200_sink sink, void *user, bz2b200_dstream **out) {
    BZ_API_TRY
    if (!ctx || !out) return BZ2B200_E_ARG;
    *out = nullptr;
    std::unique_ptr<bz2b200_dstream> d(new bz2b200_dstream());
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->dstream_open) return BZ2B200_E_ARG;
        ctx->dstream_open = true;
    }
    d->ctx = ctx; d->sink = sink; d->user = user;
    d->stage = ctx->h_dstage; d->piece = ctx->h_dpiece; d->d_win = &ctx->d_dwin; d->d_dec = ctx->d_ddec;
    if (const char *e = getenv("BZ2B200_DSTREAM_WINDOW")) { long long v = atoll(e); if (v >= 1024 && v <= (1ll << 30)) d->WF = (size_t)v; }
    d->chance = getenv("BZ2B200_MULTI_DEC_CHANCE") != nullptr;
    int rc = cudaSetDevice(ctx->device) != cudaSuccess ? BZ2B200_E_CUDA : BZ2B200_OK;
    for (int i = 0; i < 2 && !rc; i++) if (d->stage[i].ensure(PREFIX + d->WF) != cudaSuccess) rc = BZ2B200_E_NOMEM;
    if (sink && !rc) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (int i = 0; i < 2 && !rc; i++) {
            if (d->piece[i].ensure(PIECE) != cudaSuccess) rc = BZ2B200_E_NOMEM;
            else if (cudaEventCreateWithFlags(&d->ev_piece[i], cudaEventDisableTiming) != cudaSuccess) rc = BZ2B200_E_CUDA;
        }
        if (!rc && !ctx->s_up &&
            (cudaStreamCreateWithFlags(&ctx->s_up, cudaStreamNonBlocking) != cudaSuccess ||
             cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking) != cudaSuccess)) rc = BZ2B200_E_CUDA;
    }
    if (rc) { finish(d.get()); return rc; }
    d->th = std::thread(worker, d.get());
    if (sink) d->th_out = std::thread(delivery, d.get());
    *out = d.release();
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_dstream_write(bz2b200_dstream *d, const uint8_t *data, size_t n) {
    BZ_API_TRY
    if (!d || (!data && n)) return BZ2B200_E_ARG;
    {
        std::lock_guard<std::mutex> lk(d->mu);
        if (d->rc) return d->rc;
    }
    while (n) {
        size_t take = std::min(n, d->WF - d->fill);
        memcpy(d->stage[d->cur].as<u8>() + PREFIX + d->fill, data, take);
        d->fill += take; data += take; n -= take;
        if (d->fill == d->WF) {
            int rc = submit(d, false);
            if (rc) return rc;
        }
    }
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_dstream_close(bz2b200_dstream *d, uint64_t *total_in, uint64_t *total_out) {
    if (!d) return BZ2B200_E_ARG;
    int rc;
    try { rc = submit(d, true); } catch (...) { rc = BZ2B200_E_NOMEM; }
    finish(d);
    if (rc == BZ2B200_OK) rc = d->rc;
    if (rc == BZ2B200_OK && !d->ended) { rc = BZ2B200_E_FORMAT; d->err = "the input does not end with a stream footer"; }
    if (total_in) *total_in = d->total_in;
    if (total_out) *total_out = d->total_out;
    if (rc) d->ctx->err = "dstream: " + d->err;
    delete d;
    return rc;
}

}  // extern "C"
