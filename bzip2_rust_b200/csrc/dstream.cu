// dstream.cu -- streaming decompression: a .bz2 input arrives in pieces, decoded bytes leave through a callback.
//
// bz2b200_decompress_stream needs the whole input in one buffer and an output buffer for everything it decodes to.
// A dstream is the same decode core (bz_decode_core, decode.cu) driven window by window from one context by the window
// pump (pump.cuh): the caller's thread fills page-locked staging, a worker thread runs step() on every window of WF
// fresh bytes (64 MiB), a delivery thread downloads every checked batch in pieces of 32 MiB and calls the sink.  step()
// uploads [carried tail | fresh bytes], finds the magic candidates and decodes the chain elements that start before the
// window's decode edge, end - DEC_LOOK; each decoded batch passes its block CRCs on the device.
// Window edges depend only on absolute input positions: window k ends at byte (k + 1) * WF (or at the input's end).
// DEC_LOOK (4 MiB) exceeds the bound on a block's span (bz_dec_span_bits, ~2.3 MB), so an element that starts before the edge
// ends inside the window, and a footer before the edge is never taken for the end of the input.
// The bytes from where the chain leaves the window onward (at most DEC_LOOK + 1) are carried in front of the next window;
// a window whose edge is not past the chain's start is carried whole and waits for more input.
// The chain's start and the stream's running combined CRC are always known here, so every footer's combined CRC is
// checked when it is reached.  Blocks are decoded with level-9 geometry; the rules over the chain (bz_dec_fold) are
// applied to each window's events once the window is decoded.  Host memory is the staging buffers and the output pieces
// whatever the input or output size; device memory is the decode workspaces, one window and two batch outputs.  In test
// mode (no sink) nothing is downloaded.
#include "pump.cuh"
#include <memory>

struct bz2b200_dstream : DecPump {
    long long expect = 32;                   // absolute bit where the next chain element starts
    DecFold fold{0, 0, true};                // the chain's rules so far (level 0: no window decoded yet)
    bool ended = false;                      // the chain ended after the input's last footer
    std::vector<DecEvent> ev;
    u64 total_out = 0;
    int step(int slot, size_t len, bool eof) override;
};

namespace {

// where the worker's decoded batches go
struct DSink : DecSink {
    bz2b200_dstream *d;
    long long end = -1;
    void chain_end(long long bit) override { end = bit; }
    int counted(u64 nbytes, bool, u8 **d_out, u8 **h_out) override {
        *h_out = nullptr;
        return d->out_buffer(nbytes, d_out);
    }
    int ready(const u8 *d_out, u64 nbytes) override {           // the batch passed its block CRCs
        d->total_out += nbytes;
        if (d->sink) d->queue(DecPump::Job{{{d_out, nbytes}}, {}}, true);
        return BZ2B200_OK;
    }
};

}  // namespace

// one window: the carried tail + `len` fresh bytes of staging buffer `slot`
int bz2b200_dstream::step(int slot, size_t len, bool eof) {
    const u8 *h = window(slot);
    const size_t W = tail_len + len;
    const u64 lo = tail_lo, end = lo + W;
    if (fold.level == 0) {                                      // the first window (>= 1024 bytes unless it is the last)
        if (eof && total_in < 14) { ctx->err = "the input is shorter than 14 bytes"; return BZ2B200_E_FORMAT; }
        fold.level = bz_header_level(h, W);
        if (!fold.level) { ctx->err = "the input does not start with BZh<level>"; return BZ2B200_E_FORMAT; }
    }
    const u64 hi = eof ? ~0ull : (end > DEC_LOOK ? (u64)(end - DEC_LOOK) * 8 : 0);
    if (!eof && hi <= (u64)expect) return carry(slot, h, lo, W, (u64)expect / 8);   // wait for more input
    u8 *dw;
    int rc = upload(h, W, &dw);
    if (rc) return rc;
    DecWindow w{h, (size_t)lo, (size_t)end, dw, (size_t)lo, W, hi, expect, fold.combined, BZ2B200_MAX_BLOCK, &cand};
    DSink sink;
    sink.d = this;
    ev.clear();
    rc = bz_decode_core(ctx, w, sink, ev);
    if (rc) return rc;
    rc = bz_dec_fold(fold, ev, ctx->err);
    if (rc) return rc;
    if (eof) {
        if (sink.end != DEC_ENDED) { ctx->err = "decode: the input does not end with a stream footer"; return BZ2B200_E_FORMAT; }
        ended = true;
        return BZ2B200_OK;
    }
    // a footer before the edge ends at least DEC_LOOK - 11 bytes before the window's end: never the end of the input
    if (sink.end < 0 || sink.end == DEC_ENDED) { ctx->err = "decode: trailing bytes after the stream footer"; return BZ2B200_E_FORMAT; }
    expect = sink.end;
    return carry(slot, h, lo, W, (u64)sink.end / 8);
}

extern "C" {

int bz2b200_dstream_open(bz2b200_ctx *ctx, bz2b200_sink sink, void *user, bz2b200_dstream **out) {
    BZ_API_TRY
    if (!ctx || !out) return BZ2B200_E_ARG;
    *out = nullptr;
    std::unique_ptr<bz2b200_dstream> d(new bz2b200_dstream());
    int rc = d->open(ctx, sink, nullptr, user, "BZ2B200_DSTREAM_WINDOW");
    if (rc) return rc;
    *out = d.release();
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_dstream_write(bz2b200_dstream *d, const uint8_t *data, size_t n) {
    BZ_API_TRY
    if (!d || (!data && n)) return BZ2B200_E_ARG;
    return d->write(data, n);
    BZ_API_CATCH
}

int bz2b200_dstream_close(bz2b200_dstream *d, uint64_t *total_in, uint64_t *total_out) {
    if (!d) return BZ2B200_E_ARG;
    int rc = d->close();
    if (rc == BZ2B200_OK && !d->ended) { rc = BZ2B200_E_FORMAT; d->err = "the input does not end with a stream footer"; }
    if (total_in) *total_in = d->total_in;
    if (total_out) *total_out = d->total_out;
    if (rc) d->ctx->err = "dstream: " + d->err;
    delete d;
    return rc;
}

}  // extern "C"
