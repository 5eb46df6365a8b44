// recover.cu -- block recovery: every intact block of a damaged .bz2 input, and a report of what was lost.
//
// bzip2recover cuts a file at every block magic and leaves the caller to test and decode the pieces one by one; a
// damaged magic there merges two blocks into one piece that fails, so one bit loses two blocks.  Here the GPU does it:
// the magic candidates come from k_dec_find_magic (bz_dec_candidates), and the candidates are decoded in batches of
// DEC_BATCH in bit order with the decoder's two batch steps (decode.cu): the entropy decode, then for EVERY member that
// parsed (not only the members of a chain) the inverse BWT, RLE1 and block CRC.  Each member is judged on its own
// (include/bz2b200.h lists the rules); candidates inside the span of an intact block found before are chance magics in
// its data and are skipped, also when a later batch is built.
// An intact block knows where the next one starts: its end bit.  When no magic starts there (the magic is the damaged
// part), that bit is decoded as a block anyway, before the candidates after it: the batch is cut after the intact block,
// and the next batch is [that bit, the candidates after it].  The cut re-decodes the members behind it, which costs time
// on damaged inputs only.
// That judgement is one function over a window (bz_recover_window) with a carried state, and two drivers call it:
//   bz2b200_recover     one window that covers the whole input; intact bytes leave each batch in input order through
//                       bz_deliver_pieces, in the context's two page-locked pieces of recovery, on the calling thread
//   the rstream         the window pump of the dstream (pump.cuh).  A window that ends at input byte `end` judges the
//                       candidates in [its start, (end - DEC_LOOK) * 8), the last window everything to the end.  The
//                       whole-input result depends only on what lies inside each block's span, and a block that starts
//                       before the edge ends in the window (DEC_LOOK * 8 > bz_dec_span_bits), with its `rends` bound
//                       and the candidate at its end bit; a footer's stored CRC lies in the window's host bytes.  The
//                       last DEC_LOOK bytes are carried: the next window skips the candidates below the carried `cover`
//                       (chance magics inside a block that crossed the edge) and decodes a carried rescue bit first.
#include "pump.cuh"
#include <algorithm>
#include <memory>
#include <stdlib.h>

namespace {

// What carries from window to window
struct RecState {
    u64 cover = 0;                   // end bit of the last intact block: candidates below are chance magics
    long long rescue = -1;           // bit to decode as a block before the candidates (a lost magic)
    u32 comb = 0; bool stream_ok = true;   // fold of the block CRCs since the last footer; all those blocks intact
    u64 out_total = 0;
    u64 count = 0;                   // entries so far
};
struct RecWindow {
    const u8 *in; u64 lo; size_t len;      // host bytes [lo, lo + len) of the input, in[0] = byte lo
    const u8 *d_bits;                      // the same bytes on the device, followed by 64 zero bytes
    u64 hi_bit;                            // candidates from here on belong to the next window (~0: the last window)
    const std::vector<u64> *cand;          // absolute candidate bits, sorted, bit 63 = footer magic
};
// Where a window's batches go
struct RecOut {
    virtual int buffer(u64 nbytes, u8 **d_out) = 0;        // the device buffer (>= nbytes + 64) of a batch's intact bytes
    virtual int batch(DecRanges &runs, std::vector<bz2b200_rec_entry> &ent, bool used_buffer) = 0;   // in input order
    virtual ~RecOut() {}
};

// Judges the candidates of window `w` that lie below w.hi_bit (and a pending rescue bit below it), in batches
int bz_recover_window(bz2b200_ctx *ctx, const RecWindow &w, RecState &s, RecOut &out) {
    cudaStream_t st = ctx->stream;
    const std::vector<u64> &cand = *w.cand;
    const size_t ncand = cand.size();
    const u64 lo8 = w.lo * 8, nbits = lo8 + (u64)w.len * 8;
    const DecGeom g(BZ2B200_MAX_BLOCK);
    const u32 NB = DEC_BATCH;
    auto at = [&](size_t k) { return cand[k] & ~DEC_FOOT; };
    auto first_at_or_after = [&](u64 bit) {
        return (size_t)(std::lower_bound(cand.begin(), cand.end(), bit, [](u64 c, u64 b) { return (c & ~DEC_FOOT) < b; }) - cand.begin());
    };
    const size_t nown = w.hi_bit == ~0ull ? ncand : first_at_or_after(w.hi_bit);   // the candidates this window judges

    std::vector<bz2b200_rec_entry> ents;
    auto emit = [&](const bz2b200_rec_entry &e) { ents.push_back(e); s.count++; };
    size_t pos = 0;                                             // next candidate to look at
    std::vector<u64> starts, rends, rel_starts, rel_rends;
    std::vector<size_t> mk;                                     // candidate index of each member (ncand: the rescued start)
    std::vector<DecTail> db;
    std::vector<u32> hlen(NB), hkey(NB), hrand(NB), crcs(NB);
    std::vector<u64> olen(NB), ooff(NB);
    std::vector<int> status(NB);
    for (;;) {
        const bool resc = s.rescue >= 0 && (u64)s.rescue < w.hi_bit;   // a rescue bit past the edge is the next window's
        if (pos >= nown && !resc) break;
        starts.clear(); rends.clear(); mk.clear(); ents.clear();
        if (resc) { starts.push_back((u64)s.rescue); mk.push_back(ncand); }
        size_t kend = pos;
        for (; kend < nown && starts.size() < NB; kend++) {
            if ((cand[kend] & DEC_FOOT) || at(kend) < s.cover) continue;
            starts.push_back(at(kend)); mk.push_back(kend);
        }
        const u32 nb = (u32)starts.size();
        for (u32 m = 0; m < nb; m++) {                          // as in bz_decode_core: up to the next candidate, bounded
            size_t k = first_at_or_after(starts[m] + 1);
            u64 re = k < ncand ? at(k) : nbits;
            rends.push_back(std::min<u64>(re, starts[m] + bz_dec_span_bits(g.max_block)));
        }
        // ---- the two decode steps on every member; verdicts ----
        u32 nblk = 0;
        int rc;
        if (nb) {
            const std::vector<u64> *ps = &starts, *pr = &rends;
            if (lo8) {                                          // the decoder takes bits relative to d_bits
                rel_starts.clear(); rel_rends.clear();
                for (u32 m = 0; m < nb; m++) { rel_starts.push_back(starts[m] - lo8); rel_rends.push_back(rends[m] - lo8); }
                ps = &rel_starts; pr = &rel_rends;
            }
            rc = bz_dec_entropy(ctx, g, w.d_bits, w.len, *ps, *pr, db);
            if (rc) return rc;
            for (u32 m = 0; m < nb; m++) {
                DecTail &t = db[m];
                t.end_bit += lo8;
                const bool parsed = t.status == 0 && t.key < t.nblock && t.nblock <= g.max_block;
                hlen[m] = parsed ? t.nblock : 0; hkey[m] = parsed ? t.key : 0; hrand[m] = parsed ? t.pad : 0;
                status[m] = parsed ? BZ2B200_OK : BZ2B200_E_FORMAT;
                if (parsed) nblk = m + 1;
            }
        }
        u8 *d_out = nullptr;
        if (nblk) {
            rc = bz_dec_unbwt(ctx, g, nblk, hlen.data(), hkey.data(), hrand.data(), olen.data());
            if (rc) return rc;
            u64 btotal = 0;
            for (u32 m = 0; m < nblk; m++) {
                if (olen[m] == RLE1_OPEN) { olen[m] = 0; status[m] = BZ2B200_E_FORMAT; }
                ooff[m] = btotal; btotal += olen[m];
            }
            rc = out.buffer(btotal, &d_out);
            if (rc) return rc;
            rc = bz_dec_write(ctx, g, nblk, olen.data(), ooff.data(), d_out, crcs.data());
            if (rc) return rc;
            BZ_CHECK(cudaStreamSynchronize(st));
            for (u32 m = 0; m < nblk; m++)
                if (status[m] == BZ2B200_OK && crcs[m] != db[m].crc) status[m] = BZ2B200_E_CRC;
        }
        // ---- entries in input order; an intact block without a magic at its end cuts the batch there ----
        DecRanges runs;
        size_t next_pos = kend;
        long long next_rescue = resc ? -1 : s.rescue;
        auto block = [&](u32 m, u32 flags) {                   // true: the batch is cut after this member
            const u64 b = starts[m];
            if (b < s.cover) return false;                      // inside an intact block found in this batch
            if (status[m] != BZ2B200_OK && (flags & BZ2B200_REC_NO_MAGIC)) return false;   // a lost block: the gap shows it
            const bool ok = status[m] == BZ2B200_OK;
            emit(bz2b200_rec_entry{b, db[m].status == 0 ? db[m].end_bit : 0, s.out_total, ok ? (u32)olen[m] : 0u, db[m].crc,
                                   status[m], flags});
            s.comb = bz_crc_step(s.comb, db[m].crc);
            s.stream_ok &= ok;
            if (!ok) return false;
            const u64 e = db[m].end_bit;
            if (olen[m]) runs.push_back({d_out + ooff[m], olen[m]});
            s.out_total += olen[m];
            s.cover = e;
            const size_t k = first_at_or_after(e);
            if ((k < ncand && at(k) == e) || e + 128 > nbits) return false;    // the next magic is there, or the input ends
            next_rescue = (long long)e; next_pos = k;
            return true;
        };
        bool cut = false;
        u32 m = 0;
        if (resc) cut = block(m++, BZ2B200_REC_NO_MAGIC);
        for (size_t k = pos; k < kend && !cut; k++) {
            if (cand[k] & DEC_FOOT) {
                const u64 b = at(k);
                if (b < s.cover) continue;                      // a chance magic inside an intact block
                const u32 stored = bz_read32(w.in, w.len, b + 48 - lo8);
                const int fs = !s.stream_ok ? BZ2B200_E_FORMAT : s.comb != stored ? BZ2B200_E_CRC : BZ2B200_OK;
                emit(bz2b200_rec_entry{b, b + 80, s.out_total, 0u, stored, fs, BZ2B200_REC_FOOTER});
                s.comb = 0; s.stream_ok = true;
            } else if (m < nb && mk[m] == k) {
                cut = block(m++, 0);
            }
        }
        rc = out.batch(runs, ents, d_out != nullptr);
        if (rc) return rc;
        pos = next_pos; s.rescue = next_rescue;
    }
    return BZ2B200_OK;
}

// bz2b200_recover: entries into the caller's array, bytes to the sink on the calling thread
struct WholeOut : RecOut {
    bz2b200_ctx *ctx; bz2b200_sink sink; void *user; bz2b200_rec_entry *ent; u32 ent_cap; u64 written = 0;
    int buffer(u64 nbytes, u8 **d_out) override {
        BZ_CHECK(ctx->d_stream.ensure((size_t)nbytes + 64));
        *d_out = ctx->d_stream.as<u8>();
        return BZ2B200_OK;
    }
    int batch(DecRanges &runs, std::vector<bz2b200_rec_entry> &e, bool) override {
        for (const bz2b200_rec_entry &x : e) { if (written < ent_cap) ent[written] = x; written++; }
        if (!sink) return BZ2B200_OK;
        int rc = bz_deliver_pieces(runs, ctx->stream, ctx->h_rec, ctx->ev_rec, sink, user);
        if (rc) ctx->err = rc == BZ2B200_E_ARG ? "recover: the sink reported an error" : "recover: download of intact bytes failed";
        return rc;
    }
};

}  // namespace

struct bz2b200_rstream : DecPump, RecOut {
    RecState s;
    int step(int slot, size_t len, bool eof) override;
    int buffer(u64 nbytes, u8 **d_out) override { return out_buffer(nbytes, d_out); }
    int batch(DecRanges &runs, std::vector<bz2b200_rec_entry> &e, bool used_buffer) override {
        if (!delivers || (runs.empty() && e.empty())) return BZ2B200_OK;
        if (!sink) runs.clear();
        queue(Job{std::move(runs), std::move(e)}, used_buffer);
        return BZ2B200_OK;
    }
};

// one window: the carried tail + `len` fresh bytes of staging buffer `slot`
int bz2b200_rstream::step(int slot, size_t len, bool eof) {
    const u8 *h = window(slot);
    const size_t W = tail_len + len;
    const u64 lo = tail_lo, end = lo + W;
    if (end == 0) { ctx->err = "no input"; return BZ2B200_E_ARG; }
    const u64 hi = eof ? ~0ull : (end > DEC_LOOK ? (u64)(end - DEC_LOOK) * 8 : 0);
    if (!eof && hi <= lo * 8) return carry(slot, h, lo, W, lo);            // no own range yet: wait for more input
    u8 *dw;
    int rc = upload(h, W, &dw);
    if (rc) return rc;
    for (u64 &c : cand) c += lo * 8;                                        // absolute bits; the footer flag stays
    rc = bz_recover_window(ctx, RecWindow{h, lo, W, dw, hi, &cand}, s, *this);
    if (rc || eof) return rc;
    return carry(slot, h, lo, W, hi / 8);
}

extern "C" {

int bz2b200_recover(bz2b200_ctx *ctx, const uint8_t *in, size_t n, bz2b200_sink sink, void *user,
                    bz2b200_rec_entry *ent, uint32_t ent_cap, uint32_t *nent, uint64_t *total_out) {
    BZ_API_TRY
    if (!ctx || !in || n == 0 || !nent || !total_out || (!ent && ent_cap) || n > DEC_MAX_INPUT) return BZ2B200_E_ARG;
    *nent = 0; *total_out = 0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    std::vector<u64> cand;
    int rc = bz_dec_upload(ctx, in, n, getenv("BZ2B200_MULTI_DEC_CHANCE") != nullptr, cand);
    if (rc) return rc;
    RecState s;
    WholeOut out;
    out.ctx = ctx; out.sink = sink; out.user = user; out.ent = ent; out.ent_cap = ent_cap;
    rc = bz_recover_window(ctx, RecWindow{in, 0, n, ctx->d_in.as<u8>(), ~0ull, &cand}, s, out);
    if (rc) return rc;
    *nent = (u32)s.count;
    *total_out = s.out_total;
    if (s.count > ent_cap) { ctx->err = "recover: more entries than ent_cap (*nent = the count needed)"; return BZ2B200_E_CAP; }
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_rstream_open(bz2b200_ctx *ctx, bz2b200_sink sink, bz2b200_rec_report report, void *user,
                         bz2b200_rstream **out) {
    BZ_API_TRY
    if (!ctx || !out) return BZ2B200_E_ARG;
    *out = nullptr;
    std::unique_ptr<bz2b200_rstream> r(new bz2b200_rstream());
    int rc = r->open(ctx, sink, report, user, "BZ2B200_RSTREAM_WINDOW");
    if (rc) return rc;
    *out = r.release();
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_rstream_write(bz2b200_rstream *r, const uint8_t *data, size_t n) {
    BZ_API_TRY
    if (!r || (!data && n)) return BZ2B200_E_ARG;
    return r->write(data, n);
    BZ_API_CATCH
}

int bz2b200_rstream_close(bz2b200_rstream *r, uint64_t *total_in, uint64_t *total_out, uint64_t *nent) {
    if (!r) return BZ2B200_E_ARG;
    const int rc = r->close();
    if (total_in) *total_in = r->total_in;
    if (total_out) *total_out = r->s.out_total;
    if (nent) *nent = r->s.count;
    if (rc) r->ctx->err = "rstream: " + r->err;
    delete r;
    return rc;
}

}  // extern "C"
