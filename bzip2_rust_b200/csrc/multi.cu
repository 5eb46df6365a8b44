// multi.cu -- ONE bzip2 stream compressed on N GPUs of one process: the fan-out / ordered fan-in of the reference's
// `compress` (src/compression/compress.rs:40-136: par_bridge over blocks :125-132, writer thread :74-122) as a
// library entry point.  No torch, no NCCL, no collective: blocks never exchange data (SURVEY 8e).
//
//   The input is cut into windows of at most 256 MiB (a multiple of N of them, dealt round robin: window k belongs to
//   rank k mod N; one window per rank when the input is small).  Rank r (one host thread + one context per GPU),
//   for each of its windows:
//     1. uploads the window (+ look-ahead for its last block) in chunks; the RLE1 scan follows the chunks.  The upload of
//        the rank's NEXT window is posted first (second buffer, upload stream), so it runs under this window's kernels
//     2. receives the first block start of the window from the window before it (a host atomic: the block chain
//        s_{k+1} = e(s_k) of rle1.rs:245-264 is sequential, but a link only needs the scans around it),
//        chains its own blocks and hands the next start to the next window BEFORE the heavy work
//     3. compresses its blocks into one bit string (no stream header / footer)
//     4. publishes its bit count; once the counts of the windows before it are known it shifts the string to its
//        final bit phase on the device and copies it over its own PCIe link straight into the caller's buffer (download
//        stream: the copy runs under the next window's kernels)
//   the calling thread then ORs the seam bytes, folds the combined CRC in block order (crc.rs:25-27) and writes
//   "BZh<level>" and the footer (bitwriter.rs:67-72, :103-114).
// The output is the byte string a single bz2b200_compress_stream call produces, for any N.
#include "common.cuh"
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <memory>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <thread>

int bz_shard_post_upload(bz2b200_ctx *ctx, const u8 *h_src, u8 *d_win, size_t win_len, size_t chunk,
                         std::vector<cudaEvent_t> &evs);
int bz_shard_scan_arriving(bz2b200_ctx *ctx, u8 *d_win, size_t win_lo, size_t win_len, size_t n_total, int level,
                           size_t chunk, std::vector<cudaEvent_t> &evs);

namespace {

struct MWin {                                // one input window
    size_t lo = 0, hi = 0;
    std::vector<u32> crcs;
    u64 bits = 0;
    u8 first_byte = 0;                       // of the shifted string when it shares a byte with the window before
    size_t byte_lo = 0;
    bool seam = false;
    std::atomic<long long> chain_in{-1};     // first block start of this window (absolute input offset), written by window - 1
    std::atomic<long long> bits_pub{-1};     // bit count, published when the window's blocks are compressed
    cudaEvent_t ev_up = nullptr;             // fires when the window's upload has landed (recorded on its rank's upload stream)
    std::atomic<int> up_rec{0};              // ev_up has been recorded (an event that was never recorded cannot be waited for)
    // decompression
    std::vector<DecEvent> events;            // the window's chain, in order
    std::atomic<long long> len_pub{-1};      // decoded length, published after the count pass of the window's last batch
    u64 out_len = 0, copied = 0;             // bytes decoded / already handed to the download stream
    long long chain_out = -1;                // where the chain leaves the window (DEC_ENDED after the input's last footer)
    int rc = 0;                              // BZ2B200_E_*, DEC_ABORTED when it stopped because another window failed
    std::string err;
};
struct MRank {
    bz2b200_ctx *ctx = nullptr;
    std::thread th;
    DevBuf d_win[2], d_out, d_shift[2];      // two windows in flight: one being compressed, the next one arriving
    DevBuf d_dec[2];                         // decompression: decoded batches, one being written while the other downloads
    u64 ndec = 0;                            // batches decoded in the current call
    std::vector<cudaEvent_t> up_ev[2];       // upload progress of each window buffer
    cudaEvent_t ev_shift = nullptr;
    std::vector<cudaEvent_t> win_ev;         // one per window of this rank in the current call (MWin::ev_up)
    size_t posted_len[2] = {0, 0};
    int rc = 0;
    std::string err;
    size_t h2d = 0, d2h = 0;
    u32 nblk = 0;
    double t_scan = 0, t_chain = 0, t_comp = 0, t_wait = 0, t_d2h = 0;
};

}  // namespace

struct bz2b200_mctx {
    int n = 0;
    std::vector<std::unique_ptr<MRank>> rk;
    std::vector<std::unique_ptr<MWin>> win;  // windows of the current call
    std::mutex call_mu;                      // one call at a time
    bool decode = false;                     // the job: decompression (else compression)
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    u64 seq = 0;
    int done = 0;
    bool quit = false;
    // the job
    const u8 *in = nullptr; size_t nbytes = 0; int level = 9; u8 *out = nullptr; size_t out_cap = 0;
    std::atomic<int> abort{0};
    std::string err;
    u64 stat[8] = {0};
};

namespace {

using clk = std::chrono::steady_clock;
inline double ms_since(clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); }


// waits for a value >= 0 (or the abort flag); the hand-offs arrive within microseconds to a few milliseconds
inline long long wait_value(bz2b200_mctx *m, std::atomic<long long> &a) {
    for (int spin = 0;; spin++) {
        if (m->abort.load(std::memory_order_relaxed)) return -1;
        long long v = a.load(std::memory_order_acquire);
        if (v >= 0) return v;
        if (spin > 2000) std::this_thread::yield();
    }
}

int rank_fail(bz2b200_mctx *m, MRank &R, int rc, const char *what) {
    R.rc = rc;
    R.err = std::string(what) + ": " + bz2b200_last_error(R.ctx);
    m->abort.store(1);
    return rc;
}

#define MCHECK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { R.rc = BZ2B200_E_CUDA; R.err = std::string(#call) + ": " + cudaGetErrorString(e_); m->abort.store(1); return R.rc; } } while (0)

const size_t LOOK0 = 4u << 20;               // look-ahead for the last block of a window, grown on demand
constexpr u64 FOOT_BIT = 1ull << 63;          // a decoder candidate that is a footer magic
inline size_t chunk_bytes() {
    static const size_t c = [] { const char *e = getenv("BZ2B200_E2E_CHUNK_MB"); int v = e ? atoi(e) : 8; return (size_t)(v < 1 ? 1 : v) << 20; }();
    return c;
}

// Uploads in the order the data is needed.  All ranks read the caller's buffer at once and share the host's memory
// bandwidth (measured on 8 GPUs: 20 MB per GPU take 2.3 ms when all eight copy together, 0.4 ms alone), but the block
// chain visits the windows in order: window k's upload waits for window k - depth's (an event of another rank's upload
// stream), so the first windows land one after the other at full speed, the chain follows them while the later ones are
// still arriving, and no more than `depth` copies compete.  0 = unordered.
inline size_t upload_depth(int n) {
    static const int e = [] { const char *v = getenv("BZ2B200_MULTI_UPLOAD_DEPTH"); return v ? atoi(v) : -1; }();
    if (e >= 0) return (size_t)e;
    return n >= 4 ? 3 : 0;
}

// posts the upload of window k (the rank's i-th) into buffer `slot` of rank r (upload stream; returns at once)
int post_window(bz2b200_mctx *m, int r, size_t k, int slot, size_t i) {
    MRank &R = *m->rk[r];
    MWin &W = *m->win[k];
    bz2b200_ctx *ctx = R.ctx;
    const size_t n = m->nbytes;
    size_t win_len = std::min(n - W.lo, (W.hi - W.lo) + LOOK0);
    MCHECK(R.d_win[slot].ensure(std::min(n - W.lo, (W.hi - W.lo) + (64u << 20)) + 64));
    if (!ctx->s_up) {
        MCHECK(cudaStreamCreateWithFlags(&ctx->s_up, cudaStreamNonBlocking));
        MCHECK(cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking));
    }
    const size_t depth = upload_depth(m->n);
    if (depth && k >= depth) {
        MWin &P = *m->win[k - depth];
        bool rec = P.up_rec.load(std::memory_order_acquire) != 0;
        if (!rec && k < 2 * (size_t)m->n) {                      // the first rounds are posted by all ranks at the same moment
            auto t0 = clk::now();
            while (!(rec = P.up_rec.load(std::memory_order_acquire) != 0) && ms_since(t0) < 0.5 && !m->abort.load(std::memory_order_relaxed)) {}
        }
        if (rec) MCHECK(cudaStreamWaitEvent(ctx->s_up, P.ev_up, 0));
    }
    int rc = bz_shard_post_upload(ctx, m->in + W.lo, R.d_win[slot].as<u8>(), win_len, chunk_bytes(), R.up_ev[slot]);
    if (rc) return rank_fail(m, R, rc, "upload");
    while (R.win_ev.size() <= i) {
        cudaEvent_t e;
        MCHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        R.win_ev.push_back(e);
    }
    MCHECK(cudaEventRecord(R.win_ev[i], ctx->s_up));
    W.ev_up = R.win_ev[i];
    W.up_rec.store(1, std::memory_order_release);
    R.posted_len[slot] = win_len;
    R.h2d += win_len;
    return BZ2B200_OK;
}

// one window on rank r; its upload has been posted into buffer `slot`; `i` = how many windows this rank did before
int run_window(bz2b200_mctx *m, int r, size_t k, int slot, size_t i) {
    MRank &R = *m->rk[r];
    MWin &W = *m->win[k];
    bz2b200_ctx *ctx = R.ctx;
    const int level = m->level;
    const size_t n = m->nbytes, nwin = m->win.size();
    const size_t lo = W.lo, hi = W.hi;
    auto t0 = clk::now();
    // ---- 1. scan behind the upload ----
    size_t look = LOOK0;
    size_t win_len = R.posted_len[slot];
    DevBuf &dwin = R.d_win[slot];
    size_t cap_out = bz2b200_compress_bound(hi - lo + (64u << 20));
    MCHECK(R.d_out.ensure(cap_out + 64));
    {
        int rc = bz_shard_scan_arriving(ctx, dwin.as<u8>(), lo, win_len, n, level, chunk_bytes(), R.up_ev[slot]);
        if (rc) return rank_fail(m, R, rc, "scan");
    }
    R.t_scan += ms_since(t0);
    // ---- 2. the chain ----
    auto t1 = clk::now();
    long long start = k == 0 ? 0 : wait_value(m, W.chain_in);
    if (start < 0) return BZ2B200_E_CUDA;                      // another rank failed
    R.t_wait += ms_since(t1);
    auto t2 = clk::now();
    size_t nxt = (size_t)start;
    u32 nb = 0;
    for (;;) {
        int rc = bz2b200_shard_plan_dev(ctx, dwin.as<u8>(), lo, win_len, n, level, (size_t)start, hi, &nxt, &nb);
        if (rc == BZ2B200_OK) break;
        if (rc != BZ2B200_E_CAP || lo + win_len >= n) return rank_fail(m, R, rc, "plan");
        // a block of this window spans more input than the look-ahead (long runs): lengthen the window and plan again
        size_t new_len = std::min(n - lo, win_len + 8 * look);
        look *= 8;
        if (dwin.cap < new_len + 64) {                          // keep what is already resident
            DevBuf bigger;
            MCHECK(bigger.ensure(std::min(n - lo, 2 * new_len) + 64));
            MCHECK(cudaMemcpyAsync(bigger.p, dwin.p, win_len, cudaMemcpyDeviceToDevice, ctx->stream));
            MCHECK(cudaStreamSynchronize(ctx->stream));
            dwin.release();
            dwin = bigger;
        }
        MCHECK(cudaMemcpyAsync(dwin.as<u8>() + win_len, m->in + lo + win_len, new_len - win_len, cudaMemcpyHostToDevice, ctx->stream));
        MCHECK(cudaStreamSynchronize(ctx->stream));
        R.h2d += new_len - win_len;
        win_len = new_len;
    }
    if (k + 1 < nwin) m->win[k + 1]->chain_in.store((long long)nxt, std::memory_order_release);
    R.t_chain += ms_since(t2);
    // ---- 3. compress ----
    auto t3 = clk::now();
    W.bits = 0;
    if (nb) {
        W.crcs.resize(nb);
        int rc = bz2b200_shard_compress_dev(ctx, R.d_out.as<u8>(), cap_out & ~(size_t)3, &W.bits, W.crcs.data());
        if (rc) return rank_fail(m, R, rc, "compress");
        R.nblk += nb;
    }
    W.bits_pub.store((long long)W.bits, std::memory_order_release);
    R.t_comp += ms_since(t3);
    // ---- 4. final position, shift, download (asynchronous: the copy runs under the next window) ----
    auto t4 = clk::now();
    u64 off = 32;
    for (size_t q = 0; q < k; q++) {
        long long b = wait_value(m, m->win[q]->bits_pub);
        if (b < 0) return BZ2B200_E_CUDA;
        off += (u64)b;
    }
    if (W.bits) {
        int phase = (int)(off & 7);
        size_t nby = (size_t)((W.bits + phase + 7) / 8);
        W.byte_lo = (size_t)(off >> 3);
        if (W.byte_lo + nby + 16 > m->out_cap) { R.rc = BZ2B200_E_CAP; R.err = "output buffer too small"; m->abort.store(1); return R.rc; }
        DevBuf &dsh = R.d_shift[i & 1];
        if (i >= 2) MCHECK(cudaStreamSynchronize(ctx->s_down));  // the copy that last used this buffer (two windows ago)
        MCHECK(dsh.ensure(cap_out + 128));
        int rc = bz2b200_shift_bits_dev(ctx, R.d_out.as<u8>(), W.bits, phase, dsh.as<u8>());
        if (rc) return rank_fail(m, R, rc, "shift");
        W.seam = phase != 0;                                    // the first byte is shared with whatever precedes (window 0: phase 0)
        size_t skip = W.seam ? 1 : 0;
        MCHECK(cudaEventRecord(R.ev_shift, ctx->stream));
        MCHECK(cudaStreamWaitEvent(ctx->s_down, R.ev_shift, 0));
        if (W.seam) MCHECK(cudaMemcpyAsync(&W.first_byte, dsh.p, 1, cudaMemcpyDeviceToHost, ctx->s_down));
        if (nby > skip) MCHECK(cudaMemcpyAsync(m->out + W.byte_lo + skip, dsh.as<u8>() + skip, nby - skip, cudaMemcpyDeviceToHost, ctx->s_down));
        R.d2h += nby;
    }
    R.t_d2h += ms_since(t4);
    return BZ2B200_OK;
}

int run_rank(bz2b200_mctx *m, int r) {
    MRank &R = *m->rk[r];
    R.rc = 0; R.err.clear(); R.h2d = R.d2h = 0; R.nblk = 0;
    R.t_scan = R.t_chain = R.t_comp = R.t_wait = R.t_d2h = 0;
    MCHECK(cudaSetDevice(R.ctx->device));
    if (!R.ev_shift) MCHECK(cudaEventCreateWithFlags(&R.ev_shift, cudaEventDisableTiming));
    const size_t N = (size_t)m->n, nwin = m->win.size();
    if ((size_t)r < nwin) { int rc = post_window(m, r, (size_t)r, 0, 0); if (rc) return rc; }
    size_t i = 0;
    for (size_t k = (size_t)r; k < nwin; k += N, i++) {
        if (k + N < nwin) { int rc = post_window(m, r, k + N, (int)((i + 1) & 1), i + 1); if (rc) return rc; }   // arrives under this window's kernels
        int rc = run_window(m, r, k, (int)(i & 1), i);
        if (rc) return rc;
    }
    if (R.ctx->s_down) MCHECK(cudaStreamSynchronize(R.ctx->s_down));
    return BZ2B200_OK;
}

// ---- decompression ---------------------------------------------------------------------------------------------
// The compressed input is cut into byte windows dealt round robin like the compressor's.  Rank r, for each window:
//   1. waits for its upload (window + 4 MiB look-ahead: the longest block that can start in it), finds the magic
//      candidates and entropy-decodes the first batch of those in its range -- work needed wherever the chain enters
//   2. waits for the chain from window - 1, walks it (decode.cu) and hands where it leaves to window + 1 before the
//      inverse BWT; a footer belongs to the window it starts in, which also checks the next "BZh<level>" header
//   3. publishes its decoded length after the count pass of its last batch; once the lengths of the windows before it
//      are known, every batch is copied from the device straight to its final place in `out` (download stream)
// the calling thread then walks the windows' events in order: combined CRCs, the block size the headers allow.
// 24 MiB of -9 text (3.8-4.0:1 on the decode benchmark's text) hold some 105 blocks: one decoder batch of 128.  Less
// compressible data gives fewer blocks per window; -1 streams and very compressible data give several batches per
// window, which then copies batch by batch (a rank still holds at most two decoded batches while it waits for its offset).
const size_t DEC_WIN_MAX = 24u << 20, DEC_WIN_MIN = 4u << 20;

struct WinSink : DecSink {
    bz2b200_mctx *m; MRank *R; MWin *W; size_t k;
    bz2b200_ctx *ctx;
    double t_wait = 0, t_out = 0;
    long long chain_start() override {
        auto t0 = clk::now();
        long long v = wait_value(m, W->chain_in);
        t_wait += ms_since(t0);
        return v;
    }
    void chain_end(long long bit) override {
        W->chain_out = bit;
        if (k + 1 < m->win.size()) m->win[k + 1]->chain_in.store(bit, std::memory_order_release);
    }
    int counted(u64 nbytes, bool last, u8 **d_out, u8 **h_out) override {
        W->out_len += nbytes;                                   // counted even when `out` cannot take it (E_CAP reports the size)
        if (last) W->len_pub.store((long long)W->out_len, std::memory_order_release);
        DevBuf &b = R->d_dec[R->ndec & 1];
        if (R->ndec >= 2) BZ_CHECK(cudaStreamSynchronize(ctx->s_down));   // the download that last read this buffer
        R->ndec++;
        BZ_CHECK(b.ensure((size_t)nbytes + 64));
        *d_out = b.as<u8>();
        *h_out = nullptr;
        return BZ2B200_OK;
    }
    int ready(const u8 *d_out, u64 nbytes) override {
        auto t0 = clk::now();
        u64 off = W->copied;
        for (size_t q = 0; q < k; q++) {
            long long v = wait_value(m, m->win[q]->len_pub);
            if (v < 0) return DEC_ABORTED;
            off += (u64)v;
        }
        W->copied += nbytes;
        if (nbytes && off + nbytes <= m->out_cap) {
            BZ_CHECK(cudaEventRecord(R->ev_shift, ctx->stream));
            BZ_CHECK(cudaStreamWaitEvent(ctx->s_down, R->ev_shift, 0));
            BZ_CHECK(cudaMemcpyAsync(m->out + off, d_out, (size_t)nbytes, cudaMemcpyDeviceToHost, ctx->s_down));
            R->d2h += nbytes;
        }
        t_out += ms_since(t0);
        return BZ2B200_OK;
    }
};

// test knob: a spurious block candidate at the first bit of the window and between any two candidates, as chance magics
// inside compressed data would be
void add_chance_candidates(std::vector<u64> &cand) {
    std::vector<u64> add;
    if (cand.empty() || (cand[0] & ~FOOT_BIT) != 0) add.push_back(0);
    for (size_t i = 0; i + 1 < cand.size(); i++) {
        u64 a = cand[i] & ~FOOT_BIT, b = cand[i + 1] & ~FOOT_BIT;
        if (b - a >= 2) add.push_back((a + b) / 2);
    }
    cand.insert(cand.end(), add.begin(), add.end());
    std::sort(cand.begin(), cand.end(), [](u64 x, u64 y) { return (x & ~FOOT_BIT) < (y & ~FOOT_BIT); });
}

int run_dec_window(bz2b200_mctx *m, int r, size_t k, int slot) {
    MRank &R = *m->rk[r];
    MWin &W = *m->win[k];
    bz2b200_ctx *ctx = R.ctx;
    const size_t nwin = m->win.size();
    const size_t len = R.posted_len[slot];
    u8 *d = R.d_win[slot].as<u8>();
    const bool chance = getenv("BZ2B200_MULTI_DEC_CHANCE") != nullptr;
    auto t0 = clk::now();
    WinSink sink;
    sink.m = m; sink.R = &R; sink.W = &W; sink.k = k; sink.ctx = ctx;
    int rc;
    double t_scan;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->err.clear();
        MCHECK(cudaStreamWaitEvent(ctx->stream, W.ev_up, 0));
        MCHECK(cudaMemsetAsync(d + len, 0, 64, ctx->stream));  // word loads of the entropy stage read past the last byte
        std::vector<u64> cand;
        // at most one magic per 32 bits whatever the data: a window is never refused where the whole input is accepted
        rc = bz_dec_candidates(ctx, d, len, (u32)std::min<size_t>(len / 4 + 64, 0x7fffff00u), cand);
        t_scan = ms_since(t0);
        if (!rc) {
            if (chance) add_chance_candidates(cand);
            // level-9 geometry: the headers of later windows are not known yet; the calling thread applies the block
            // size they allow
            DecWindow w{m->in, m->nbytes, d, W.lo, len, k + 1 == nwin ? ~0ull : (u64)W.hi * 8, k == 0 ? 32ll : -1ll,
                        BZ2B200_MAX_BLOCK, &cand};
            rc = bz_decode_core(ctx, w, sink, W.events);
        }
    }
    R.t_scan += t_scan; R.t_wait += sink.t_wait; R.t_d2h += sink.t_out;
    R.t_comp += ms_since(t0) - t_scan - sink.t_wait - sink.t_out;
    if (rc) {
        W.rc = rc;
        if (rc != DEC_ABORTED) W.err = ctx->err;
        m->abort.store(1);
        return rc;
    }
    W.len_pub.store((long long)W.out_len, std::memory_order_release);
    return BZ2B200_OK;
}

int run_dec_windows(bz2b200_mctx *m, int r) {
    MRank &R = *m->rk[r];
    MCHECK(cudaSetDevice(R.ctx->device));
    if (!R.ev_shift) MCHECK(cudaEventCreateWithFlags(&R.ev_shift, cudaEventDisableTiming));
    const size_t N = (size_t)m->n, nwin = m->win.size();
    if ((size_t)r < nwin) { int rc = post_window(m, r, (size_t)r, 0, 0); if (rc) return rc; }
    size_t i = 0;
    for (size_t k = (size_t)r; k < nwin; k += N, i++) {
        if (k + N < nwin) { int rc = post_window(m, r, k + N, (int)((i + 1) & 1), i + 1); if (rc) return rc; }   // arrives under this window's kernels
        int rc = run_dec_window(m, r, k, (int)(i & 1));
        if (rc) return rc;
    }
    return BZ2B200_OK;
}

int run_dec_rank(bz2b200_mctx *m, int r) {
    MRank &R = *m->rk[r];
    R.rc = 0; R.err.clear(); R.h2d = R.d2h = 0; R.nblk = 0; R.ndec = 0;
    R.t_scan = R.t_chain = R.t_comp = R.t_wait = R.t_d2h = 0;
    int rc;
    try { rc = run_dec_windows(m, r); } catch (...) { rc = BZ2B200_E_NOMEM; R.rc = rc; R.err = "out of memory"; m->abort.store(1); }
    // whatever failed: no copy from `in` or into `out` may still run when the call returns
    bz2b200_ctx *ctx = R.ctx;
    cudaSetDevice(ctx->device);
    if (ctx->s_up) cudaStreamSynchronize(ctx->s_up);
    if (ctx->s_hi) cudaStreamSynchronize(ctx->s_hi);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->s_down) cudaStreamSynchronize(ctx->s_down);
    return rc;
}

void worker(bz2b200_mctx *m, int r) {
    u64 seen = 0;
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_job.wait(lk, [&] { return m->quit || m->seq != seen; });
            if (m->quit) return;
            seen = m->seq;
        }
        int rc;
        try { rc = m->decode ? run_dec_rank(m, r) : run_rank(m, r); } catch (...) { rc = BZ2B200_E_NOMEM; m->rk[r]->rc = rc; m->rk[r]->err = "out of memory"; m->abort.store(1); }
        (void)rc;                                               // a failed rank has raised the abort flag: nobody waits for it
        {
            std::lock_guard<std::mutex> lk(m->mu);
            m->done++;
        }
        m->cv_done.notify_all();
    }
}

inline u32 crc_step(u32 s, u32 b) { return ((s << 1) | (s >> 31)) ^ b; }   // crc.rs:25-27

}  // namespace

extern "C" {

int bz2b200_create_multi(int n_devices, const int *device_ids, bz2b200_mctx **out) {
    BZ_API_TRY
    if (!out || n_devices < 1 || n_devices > 64) return BZ2B200_E_ARG;
    *out = nullptr;
    std::unique_ptr<bz2b200_mctx> m(new bz2b200_mctx());
    m->n = n_devices;
    for (int r = 0; r < n_devices; r++) {
        m->rk.emplace_back(new MRank());
        int rc = bz2b200_create(device_ids ? device_ids[r] : r, &m->rk[r]->ctx);
        if (rc) {
            for (auto &R : m->rk) if (R->ctx) bz2b200_destroy(R->ctx);
            return rc;
        }
    }
    for (int r = 0; r < n_devices; r++) m->rk[r]->th = std::thread(worker, m.get(), r);
    *out = m.release();
    return BZ2B200_OK;
    BZ_API_CATCH
}

void bz2b200_destroy_multi(bz2b200_mctx *m) {
    if (!m) return;
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->quit = true;
    }
    m->cv_job.notify_all();
    for (auto &R : m->rk) if (R->th.joinable()) R->th.join();
    for (auto &R : m->rk) {
        if (R->ctx) {
            cudaSetDevice(R->ctx->device);
            for (int q = 0; q < 2; q++) {
                R->d_win[q].release(); R->d_shift[q].release();
                for (cudaEvent_t e : R->up_ev[q]) cudaEventDestroy(e);
            }
            R->d_out.release();
            if (R->ev_shift) cudaEventDestroy(R->ev_shift);
            for (cudaEvent_t e : R->win_ev) cudaEventDestroy(e);
            bz2b200_destroy(R->ctx);
        }
    }
    delete m;
}

const char *bz2b200_last_error_multi(const bz2b200_mctx *m) { return m ? m->err.c_str() : "null context"; }
int bz2b200_multi_devices(const bz2b200_mctx *m) { return m ? m->n : 0; }
bz2b200_ctx *bz2b200_multi_context(bz2b200_mctx *m, int rank) { return (m && rank >= 0 && rank < m->n) ? m->rk[rank]->ctx : nullptr; }

int bz2b200_compress_stream_multi(bz2b200_mctx *m, const uint8_t *in, size_t n, int level, uint8_t *out,
                                  size_t out_cap, size_t *out_len) {
    BZ_API_TRY
    if (!m || (!in && n) || !out || !out_len || level < 1 || level > 9) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> call(m->call_mu);
    // small inputs (or one device): the single-GPU path, same bytes
    if (m->n == 1 || n < (size_t)m->n * (8u << 20)) {
        int rc = bz2b200_compress_stream(m->rk[0]->ctx, in, n, level, out, out_cap, out_len);
        if (rc) m->err = bz2b200_last_error(m->rk[0]->ctx);
        m->stat[0] = n; m->stat[1] = rc ? 0 : *out_len;
        return rc;
    }
    if (out_cap < 64) return BZ2B200_E_CAP;
    auto t0 = clk::now();
    m->in = in; m->nbytes = n; m->level = level; m->out = out; m->out_cap = out_cap;
    m->decode = false;
    m->abort.store(0);
    {   // windows: a multiple of n_devices, at most 256 MiB each, whole 4 KiB pages
        // Two windows per rank when a window still holds 32 MiB: nothing can be compressed before a rank's first window is on
        // its device and the chain has passed the windows before it, and the second window's upload hides under the first
        // one's kernels; a window costs about 0.8 ms of fixed work (measured, 2 GPUs x 100 MB: 17.2 ms with one window per
        // rank, 15.8 ms with a quarter + three quarters; 8 GPUs: see profiles/r02_experiments.md section 6).
        const size_t WMAX = 256u << 20, WMIN = 32u << 20;
        size_t per_rank = (n + (size_t)m->n - 1) / (size_t)m->n;
        size_t per = std::max<size_t>((per_rank + WMAX - 1) / WMAX, (per_rank >= 2 * WMIN && m->n >= 2) ? 2 : 1);
        if (const char *e = getenv("BZ2B200_MULTI_WINDOWS")) { int v = atoi(e); if (v >= 1) per = std::max<size_t>((per_rank + WMAX - 1) / WMAX, (size_t)v); }
        // The first window of every rank is the smaller one (25% of its share): all ranks upload at once and share the
        // host's memory bandwidth, and nothing can be compressed before the first windows are on the devices (measured on
        // 8 GPUs: 8 x 50 MB arrive after 3.3 ms); the larger second windows arrive under the first ones' kernels.
        size_t first_pct = 25;
        if (const char *e = getenv("BZ2B200_MULTI_FIRST_PCT")) { int v = atoi(e); if (v >= 5 && v <= 100) first_pct = (size_t)v; }
        std::vector<size_t> round_sz(per);
        for (size_t q = 0; q < per; q++) round_sz[q] = (per_rank + per - 1) / per;
        if (per == 2 && per_rank - per_rank * first_pct / 100 <= WMAX) { round_sz[0] = per_rank * first_pct / 100; round_sz[1] = per_rank - round_sz[0]; }
        m->win.clear();
        size_t lo = 0;
        for (size_t q = 0; q < per && lo < n; q++) {
            const size_t wsz = std::max<size_t>(4096, (round_sz[q] + 4095) & ~(size_t)4095);
            for (int r = 0; r < m->n && lo < n; r++) {
                m->win.emplace_back(new MWin());
                m->win.back()->lo = lo;
                m->win.back()->hi = (q + 1 == per && r + 1 == m->n) ? n : std::min(n, lo + wsz);
                lo = m->win.back()->hi;
            }
        }
        if (lo < n) m->win.back()->hi = n;
    }
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->done = 0;
        m->seq++;
    }
    m->cv_job.notify_all();
    {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv_done.wait(lk, [&] { return m->done == m->n; });
    }
    for (auto &R : m->rk) {
        if (R->rc) { m->err = "rank failed: " + R->err; return R->rc; }
    }
    // ---- ordered fan-in on the host: seam bytes, combined CRC, header, footer ----
    u64 pos = 32;
    u32 combined = 0;
    for (auto &W : m->win) {
        if (W->bits) {
            if (W->seam) out[W->byte_lo] |= W->first_byte;
            pos += W->bits;
        }
        for (u32 c : W->crcs) combined = crc_step(combined, c);            // bitwriter.rs:89-91
    }
    out[0] = 'B'; out[1] = 'Z'; out[2] = 'h'; out[3] = (u8)('0' + level);  // bitwriter.rs:67-72
    size_t len = (size_t)((pos + 80 + 7) / 8);
    if (len > out_cap) return BZ2B200_E_CAP;
    const u8 foot[10] = {0x17, 0x72, 0x45, 0x38, 0x50, 0x90, (u8)(combined >> 24), (u8)(combined >> 16), (u8)(combined >> 8), (u8)combined};
    const int sh = (int)(pos & 7);
    u8 *d = out + (pos >> 3);
    if (sh == 0) d[0] = 0;                                      // otherwise the byte holds the last bits of the last block
    for (size_t j = 1; j <= 10 && (size_t)(pos >> 3) + j < len; j++) d[j] = 0;
    for (int j = 0; j < 10; j++) {                              // bitwriter.rs:103-114
        d[j] |= (u8)(foot[j] >> sh);
        if (sh) d[j + 1] |= (u8)(foot[j] << (8 - sh));
    }
    *out_len = len;
    u64 h2d = 0, d2h = 0;
    for (auto &R : m->rk) { h2d += R->h2d; d2h += R->d2h; }
    m->stat[0] = h2d; m->stat[1] = d2h;
    if (getenv("BZ2B200_MULTI_TRACE")) {
        fprintf(stderr, "[multi] total %.2f ms\n", ms_since(t0));
        for (int r = 0; r < m->n; r++) {
            MRank &R = *m->rk[r];
            fprintf(stderr, "[multi rank %d] upload+scan %.2f wait %.2f chain %.2f compress %.2f offsets+shift+d2h %.2f ms, %u blocks\n", r,
                    R.t_scan, R.t_wait, R.t_chain, R.t_comp, R.t_d2h, (unsigned)R.nblk);
        }
    }
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_decompress_stream_multi(bz2b200_mctx *m, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap,
                                    size_t *out_len) {
    BZ_API_TRY
    if (!m || !in || !out_len || (!out && out_cap) || n < 14 || n > 0xFFFFFF00ull * 4ull) return BZ2B200_E_ARG;
    if (in[0] != 'B' || in[1] != 'Z' || in[2] != 'h' || in[3] < '1' || in[3] > '9') return BZ2B200_E_FORMAT;
    std::lock_guard<std::mutex> call(m->call_mu);
    *out_len = 0;
    size_t win = std::min(DEC_WIN_MAX, std::max(DEC_WIN_MIN, ((n + 2 * (size_t)m->n - 1) / (2 * (size_t)m->n) + 4095) & ~(size_t)4095));
    if (const char *e = getenv("BZ2B200_MULTI_DEC_WINDOW")) { long long v = atoll(e); if (v >= 1024) win = (size_t)v; }
    // small inputs (or one device): the single-GPU path
    if (m->n == 1 || n < 2 * win) {
        int rc = bz2b200_decompress_stream(m->rk[0]->ctx, in, n, out, out_cap, out_len);
        // That call stops at the first batch that does not fit; the caller is owed the exact size, so the input is decoded
        // again into scratch memory (growing twofold while it does not fit) to learn it.  A defect behind the point where
        // the first call stopped does not change the code: it stays E_CAP, with the size the first call reported.
        const size_t first_len = *out_len;
        for (std::vector<u8> tmp; rc == BZ2B200_E_CAP;) {
            tmp.resize(std::max<size_t>(2 * *out_len, 1 << 20));
            rc = bz2b200_decompress_stream(m->rk[0]->ctx, in, n, tmp.data(), tmp.size(), out_len);
            if (rc == BZ2B200_OK) { rc = BZ2B200_E_CAP; break; }
            if (rc != BZ2B200_E_CAP) { rc = BZ2B200_E_CAP; *out_len = first_len; break; }
        }
        if (rc) m->err = bz2b200_last_error(m->rk[0]->ctx);
        m->stat[0] = n; m->stat[1] = rc ? 0 : *out_len;
        return rc;
    }
    auto t0 = clk::now();
    m->in = in; m->nbytes = n; m->out = out; m->out_cap = out_cap;
    m->decode = true;
    m->abort.store(0);
    m->win.clear();
    for (size_t lo = 0; lo < n; lo += win) {
        m->win.emplace_back(new MWin());
        m->win.back()->lo = lo;
        m->win.back()->hi = std::min(n, lo + win);
    }
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->done = 0;
        m->seq++;
    }
    m->cv_job.notify_all();
    {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv_done.wait(lk, [&] { return m->done == m->n; });
    }
    u64 h2d = 0, d2h = 0;
    for (auto &R : m->rk) { h2d += R->h2d; d2h += R->d2h; }
    m->stat[0] = h2d; m->stat[1] = d2h;
    if (getenv("BZ2B200_MULTI_TRACE")) {
        fprintf(stderr, "[multi decode] total %.2f ms, %zu windows of %zu bytes\n", ms_since(t0), m->win.size(), win);
        for (int r = 0; r < m->n; r++) {
            MRank &R = *m->rk[r];
            fprintf(stderr, "[multi decode rank %d] upload+magics %.2f chain wait %.2f decode %.2f offsets+d2h %.2f ms\n", r,
                    R.t_scan, R.t_wait, R.t_comp, R.t_d2h);
        }
    }
    // ---- ordered fan-in: the first error in chain order wins; combined CRCs; block size the headers allow ----
    // Every block is bounded by 100000 x the largest level among the first header and every header after a footer on
    // the chain (windows decode with level-9 buffers).  bz2b200_decompress_stream takes the maximum over every footer
    // magic followed by "BZh<level>", chance ones inside compressed data included; the two differ only where such a
    // chance footer is followed by a larger level digit.  With several defects in one input the
    // code returned may be E_FORMAT where the single-GPU call returns E_CRC or the reverse.
    int level = in[3] - '0';
    for (auto &W : m->win)
        for (const DecEvent &e : W->events) if (e.kind == DEC_STREAM) level = std::max(level, (int)e.val);
    const u32 max_block = (u32)level * 100000u;
    u32 combined = 0;
    bool fold = true;                                           // `combined` covers the whole stream so far
    u64 total = 0;
    for (auto &W : m->win) {
        for (const DecEvent &e : W->events) {
            if (e.kind == DEC_BLOCK) {
                if (e.nblock > max_block) { m->err = "decode: block at bit " + std::to_string(e.bit) + " longer than its stream's level allows"; return BZ2B200_E_FORMAT; }
                combined = crc_step(combined, e.val);
            } else if (e.kind == DEC_FOOTER) {
                if (fold && e.val != combined) { m->err = "decode: combined CRC mismatch at bit " + std::to_string(e.bit); return BZ2B200_E_CRC; }
            } else {
                combined = 0; fold = true;
            }
        }
        if (W->rc < 0) { m->err = W->err; return W->rc; }
        if (W->rc) fold = false;                                // stopped early: its events are incomplete
        total += W->out_len;
    }
    for (auto &R : m->rk) if (R->rc) { m->err = "rank failed: " + R->err; return R->rc; }
    for (auto &W : m->win) if (W->rc) { m->err = "decode: a window stopped without an error"; return BZ2B200_E_CUDA; }
    if (m->win.back()->chain_out != DEC_ENDED) { m->err = "decode: the input does not end with a stream footer"; return BZ2B200_E_FORMAT; }
    *out_len = (size_t)total;
    if (total > out_cap) { m->err = "output buffer too small"; return BZ2B200_E_CAP; }
    return BZ2B200_OK;
    BZ_API_CATCH
}

int bz2b200_multi_stats(const bz2b200_mctx *m, uint64_t st[8]) {
    if (!m || !st) return BZ2B200_E_ARG;
    memcpy(st, m->stat, sizeof(u64) * 8);
    return BZ2B200_OK;
}

}  // extern "C"
