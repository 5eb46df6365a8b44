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
// Intact bytes leave a batch in input order, copied down in page-locked pieces of 32 MiB (two, kept by the context):
// piece i downloads while the sink takes piece i - 1 on the calling thread.
#include "common.cuh"
#include <algorithm>
#include <stdlib.h>
#include <utility>

namespace {
const size_t PIECE = 32u << 20;
inline u32 crc_step(u32 s, u32 b) { return ((s << 1) | (s >> 31)) ^ b; }   // crc.rs:25-27

typedef std::vector<std::pair<const u8 *, u64>> Runs;   // device ranges of intact bytes, in input order

int deliver(bz2b200_ctx *ctx, const Runs &runs, bz2b200_sink sink, void *user) {
    cudaStream_t st = ctx->stream;
    Runs pieces;
    for (const auto &r : runs)
        for (u64 o = 0; o < r.second; o += PIECE) pieces.push_back({r.first + o, std::min<u64>(PIECE, r.second - o)});
    if (pieces.empty()) return BZ2B200_OK;
    for (int i = 0; i < 2; i++) {
        BZ_CHECK(ctx->h_rec[i].ensure(PIECE));
        if (!ctx->ev_rec[i]) BZ_CHECK(cudaEventCreateWithFlags(&ctx->ev_rec[i], cudaEventDisableTiming));
    }
    int rc = BZ2B200_OK;
    for (size_t i = 0; i <= pieces.size(); i++) {
        if (i < pieces.size()) {            // the buffer's previous piece (i - 2) went to the sink in the last round
            BZ_CHECK(cudaMemcpyAsync(ctx->h_rec[i & 1].p, pieces[i].first, (size_t)pieces[i].second, cudaMemcpyDeviceToHost, st));
            BZ_CHECK(cudaEventRecord(ctx->ev_rec[i & 1], st));
        }
        if (i > 0) {
            BZ_CHECK(cudaEventSynchronize(ctx->ev_rec[(i - 1) & 1]));
            if (sink(user, ctx->h_rec[(i - 1) & 1].as<u8>(), (size_t)pieces[i - 1].second) != 0) {
                ctx->err = "recover: the sink reported an error"; rc = BZ2B200_E_ARG; break;
            }
        }
    }
    BZ_CHECK(cudaStreamSynchronize(st));    // also after an error: no copy may still write a piece
    return rc;
}

}  // namespace

extern "C" int bz2b200_recover(bz2b200_ctx *ctx, const uint8_t *in, size_t n, bz2b200_sink sink, void *user,
                               bz2b200_rec_entry *ent, uint32_t ent_cap, uint32_t *nent, uint64_t *total_out) {
    BZ_API_TRY
    if (!ctx || !in || n == 0 || !nent || !total_out || (!ent && ent_cap) || n > 0xFFFFFF00ull * 4ull) return BZ2B200_E_ARG;
    *nent = 0; *total_out = 0;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    cudaStream_t st = ctx->stream;
    BZ_CHECK(ctx->d_in.ensure(n + 64));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_in.p, in, n, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemsetAsync(ctx->d_in.as<u8>() + n, 0, 64, st));       // word loads of the entropy stage read past the last byte
    const u8 *d_bits = ctx->d_in.as<u8>();
    std::vector<u64> cand;
    int rc = bz_dec_candidates(ctx, d_bits, n, (u32)std::min<size_t>(n / 32 + 64, 0x7fffff00u), cand);
    if (rc) return rc;
    if (getenv("BZ2B200_MULTI_DEC_CHANCE")) bz_add_chance_candidates(cand);
    const size_t ncand = cand.size();
    const u64 nbits = (u64)n * 8;
    const DecGeom g(BZ2B200_MAX_BLOCK);
    const u32 NB = DEC_BATCH;
    auto at = [&](size_t k) { return cand[k] & ~DEC_FOOT; };
    auto first_at_or_after = [&](u64 bit) {
        return (size_t)(std::lower_bound(cand.begin(), cand.end(), bit, [](u64 c, u64 b) { return (c & ~DEC_FOOT) < b; }) - cand.begin());
    };
    auto read32 = [&](u64 bit) {                                // 32 bits at a bit offset of the input
        size_t byte = (size_t)(bit >> 3); int sh = (int)(bit & 7);
        u64 v = 0;
        for (int k = 0; k < 5; k++) v = (v << 8) | (byte + k < n ? in[byte + k] : 0);
        return (u32)((v >> (8 - sh)) & 0xffffffffull);
    };

    u32 count = 0;                                              // entries found (written while below ent_cap)
    auto emit = [&](const bz2b200_rec_entry &e) { if (count < ent_cap) ent[count] = e; count++; };
    u64 out_total = 0;
    u64 cover = 0;                                              // end bit of the last intact block: candidates below are chance magics
    u32 comb = 0; bool stream_ok = true;                        // fold of the block CRCs since the last footer; all those blocks intact
    size_t pos = 0;                                             // next candidate to look at
    long long rescue = -1;                                      // bit to decode as a block before the candidates (a lost magic)
    std::vector<u64> starts, rends;
    std::vector<size_t> mk;                                     // candidate index of each member (ncand: the rescued start)
    std::vector<DecTail> db;
    std::vector<u32> hlen(NB), hkey(NB), hrand(NB), crcs(NB);
    std::vector<u64> olen(NB), ooff(NB);
    std::vector<int> status(NB);
    while (pos < ncand || rescue >= 0) {
        starts.clear(); rends.clear(); mk.clear();
        if (rescue >= 0) { starts.push_back((u64)rescue); mk.push_back(ncand); }
        size_t kend = pos;
        for (; kend < ncand && starts.size() < NB; kend++) {
            if ((cand[kend] & DEC_FOOT) || at(kend) < cover) continue;
            starts.push_back(at(kend)); mk.push_back(kend);
        }
        const u32 nb = (u32)starts.size();
        for (u32 m = 0; m < nb; m++) {                          // as in bz_decode_core: up to the next candidate, bounded
            size_t k = first_at_or_after(starts[m] + 1);
            u64 re = k < ncand ? at(k) : nbits;
            rends.push_back(std::min<u64>(re, starts[m] + (u64)20 * (g.max_block + 64) + ((u64)1 << 19)));
        }
        // ---- the two decode steps on every member; verdicts ----
        u32 nblk = 0;
        if (nb) {
            rc = bz_dec_entropy(ctx, g, d_bits, n, starts, rends, db);
            if (rc) return rc;
            for (u32 m = 0; m < nb; m++) {
                const DecTail &t = db[m];
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
            BZ_CHECK(ctx->d_stream.ensure((size_t)btotal + 64));
            d_out = ctx->d_stream.as<u8>();
            rc = bz_dec_write(ctx, g, nblk, olen.data(), ooff.data(), d_out, crcs.data());
            if (rc) return rc;
            BZ_CHECK(cudaStreamSynchronize(st));
            for (u32 m = 0; m < nblk; m++)
                if (status[m] == BZ2B200_OK && crcs[m] != db[m].crc) status[m] = BZ2B200_E_CRC;
        }
        // ---- entries in input order; an intact block without a magic at its end cuts the batch there ----
        Runs runs;
        size_t next_pos = kend;
        long long next_rescue = -1;
        auto block = [&](u32 m, u32 flags) {                   // true: the batch is cut after this member
            const u64 b = starts[m];
            if (b < cover) return false;                        // inside an intact block found in this batch
            if (status[m] != BZ2B200_OK && (flags & BZ2B200_REC_NO_MAGIC)) return false;   // a lost block: the gap shows it
            const bool ok = status[m] == BZ2B200_OK;
            emit(bz2b200_rec_entry{b, db[m].status == 0 ? db[m].end_bit : 0, out_total, ok ? (u32)olen[m] : 0u, db[m].crc,
                                   status[m], flags});
            comb = crc_step(comb, db[m].crc);
            stream_ok &= ok;
            if (!ok) return false;
            const u64 e = db[m].end_bit;
            if (olen[m]) runs.push_back({d_out + ooff[m], olen[m]});
            out_total += olen[m];
            cover = e;
            const size_t k = first_at_or_after(e);
            if ((k < ncand && at(k) == e) || e + 128 > nbits) return false;    // the next magic is there, or the input ends
            next_rescue = (long long)e; next_pos = k;
            return true;
        };
        bool cut = false;
        u32 m = 0;
        if (rescue >= 0) cut = block(m++, BZ2B200_REC_NO_MAGIC);
        for (size_t k = pos; k < kend && !cut; k++) {
            if (cand[k] & DEC_FOOT) {
                const u64 b = at(k);
                if (b < cover) continue;                        // a chance magic inside an intact block
                const u32 stored = read32(b + 48);
                const int s = !stream_ok ? BZ2B200_E_FORMAT : comb != stored ? BZ2B200_E_CRC : BZ2B200_OK;
                emit(bz2b200_rec_entry{b, b + 80, out_total, 0u, stored, s, BZ2B200_REC_FOOTER});
                comb = 0; stream_ok = true;
            } else if (m < nb && mk[m] == k) {
                cut = block(m++, 0);
            }
        }
        if (sink) {
            rc = deliver(ctx, runs, sink, user);
            if (rc) return rc;
        }
        pos = next_pos; rescue = next_rescue;
    }
    *nent = count;
    *total_out = out_total;
    if (count > ent_cap) { ctx->err = "recover: more entries than ent_cap (*nent = the count needed)"; return BZ2B200_E_CAP; }
    return BZ2B200_OK;
    BZ_API_CATCH
}
