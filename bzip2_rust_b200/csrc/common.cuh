// common.cuh -- shared internals of libbz2b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <mutex>
#include <string>
#include <vector>
#include <new>
#include "../../include/bz2b200.h"

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;

#define BZ_CHECK(call)                                                                     \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            ctx->fail(#call, e_, __FILE__, __LINE__);                                      \
            return BZ2B200_E_CUDA;                                                         \
        }                                                                                  \
    } while (0)

// No exception may cross the C ABI (include/bz2b200.h): std::vector / std::string growth inside the entry points can throw.
#define BZ_API_TRY try {
#define BZ_API_CATCH } catch (const std::bad_alloc &) { return BZ2B200_E_NOMEM; } catch (...) { return BZ2B200_E_CUDA; }

// Grow-only device / pinned buffers.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

// Geometry shared by all per-block kernels: grid = (tiles, nblk); one bzip2 block per blockIdx.y.
constexpr int BZ_THREADS = 256;
constexpr int BZ_IPT = 16;
constexpr int BZ_TILE = BZ_THREADS * BZ_IPT;   // 4096 elements per CTA tile
constexpr int BZ_GROUP = 50;                   // Huffman group size (huffman.rs:137)
constexpr int BZ_MAXSYM = 258;

// Device-side description of a batch of RLE1 blocks (all arrays indexed by block, fixed stride).
struct Batch {
    int nblk;
    u32 stride;        // elements reserved per block (multiple of BZ_TILE, >= max n + 64)
    u32 tiles;         // stride / BZ_TILE
    u32 max_n;
    int nbits;         // bit length of (max_n - 1), >= 1
    const u8 *T;       // [nblk * stride] RLE1 block bytes
    const u32 *len;    // [nblk] block lengths (device)
    u64 total_n;       // sum of block lengths (host copy, for profiling byte counts)
};

enum KernelId { K_RADIX_HIST0, K_RADIX_SCAN, K_RADIX_SCATTER0, K_REF_PATH, K_BYTE_HIST, K_DIGIT_SCAN, K_SWEEP_GATHER, K_SWEEP_CARRY, K_SWEEP_LIST, K_INIT_RANKS, K_LIST_KEY, K_LIST_REFINE, K_REFINE_LOCAL, K_BWT_OUT, K_USED, K_MTF_SUMMARY, K_MTF_SCAN, K_MTF_EMIT, K_HUF_INIT, K_HUF_SELECT, K_HUF_LENGTHS, K_HUF_GBITS, K_HUF_LAYOUT, K_HUF_EMIT, K_RLE_SCAN, K_RLE_CHAIN, K_RLE_EMIT, K_CRC_PIECES, K_CRC_FINAL, K_CONCAT, K_FOOTER, K_DEC_MISC, K_DEC_MAGIC, K_DEC_HEADER, K_DEC_JUMPS, K_DEC_BOUNDS, K_DEC_SYMS, K_DEC_CHUNKS, K_DEC_EXPAND, K_DEC_CHUNK_SCAN, K_IBWT_CHASE, K_IBWT_RANK, K_IBWT_WRITE, K_DEC_RLE1_COUNT, K_DEC_RLE1_WRITE, K_COUNT };
static const char *const kKernelNames[] = { "k_radix_hist0", "k_radix_scan", "k_radix_scatter0", "k_ref_path", "k_byte_hist", "k_digit_scan", "k_sweep_gather", "k_sweep_carry", "k_sweep_list", "k_init_ranks", "k_list_key", "k_list_refine", "k_refine_local", "k_bwt_out", "k_used", "k_mtf_summary", "k_mtf_scan", "k_mtf_emit", "k_huf_init", "k_huf_select", "k_huf_lengths", "k_huf_gbits", "k_huf_layout", "k_huf_emit", "k_rle_scan", "k_rle_chain", "k_rle_emit", "k_crc_pieces", "k_crc_final", "k_concat", "k_footer", "k_dec_misc", "k_dec_find_magic", "k_dec_header", "k_dec_jumps", "k_dec_bounds", "k_dec_syms", "k_dec_chunks", "k_dec_expand", "k_dec_chunk_scan", "k_ibwt_chase", "k_ibwt_rank", "k_ibwt_write", "k_dec_rle1_count", "k_dec_rle1_write" };

struct KStat { double ms = 0; u64 launches = 0; u64 bytes = 0; };
struct PendingEv { int id; u64 bytes; cudaEvent_t a, b; };

// Input that is still arriving on an upload stream (host-buffer entry points): event i fires when stream bytes
// [0, (i+1)*chunk) are on the device.  bz_rle1_window launches its scan chunk by chunk behind the upload.
struct Arrival {
    std::vector<cudaEvent_t> *ev;
    size_t chunk;
    size_t win_off;      // stream offset of the window being scanned
    size_t waited;       // events the compute stream already waits for
};

// Pending state of the three-phase sharding entry points (shard.cu): scan -> plan -> compress on one window.
struct ShardPlan {
    bool scanned = false;
    const u8 *d_win = nullptr; size_t win_lo = 0, win_len = 0, n_total = 0; int level = 0;
    bool planned = false;
    bool eof = false; u32 off_from = 0, stop_rel = 0, s0 = 0, nb = 0;
};

struct bz2b200_ctx {
    int device = 0;
    ShardPlan shard;                 // guarded by `mu` like everything else in the context
    cudaStream_t stream = nullptr;
    cudaStream_t s_up = nullptr, s_down = nullptr;      // host-buffer pipelining (stream.cu)
    std::vector<cudaEvent_t> up_ev;
    Arrival *arrival = nullptr;
    std::mutex mu;
    std::string err;
    u64 launches = 0;
    bool timing = false;
    bool dec_attr_done = false;      // k_dec_bounds opted in to > 48 KB of dynamic shared memory on this device
    bool loc_attr_done = false;      // k_refine_local likewise
    float stage_ms[8] = {0};
    u64 bwt_stats[8] = {0};
    cudaEvent_t ev[8] = {nullptr};
    cudaEvent_t ev_total[2] = {nullptr, nullptr};
    cudaStream_t s_hi = nullptr;                            // decoder: the walkers of k_dec_bounds run beside the jump-table producer (high priority)
    cudaEvent_t ev_dec[2] = {nullptr, nullptr};

    // ---- batch staging ----
    DevBuf d_T, d_len, d_crc;
    PinBuf h_stage, h_small, h_out;
    // ---- BWT workspace ----
    DevBuf d_SA, d_SA2, d_RANK, d_F, d_KEYA, d_KEYB, d_VALA, d_VALB, d_thist, d_tagg, d_cnt, d_bwt, d_key;
    // ---- MTF / RLE2 workspace ----
    DevBuf d_mtfstate, d_chunkrec, d_R, d_sym, d_m, d_freq, d_used, d_agg2;
    // ---- Huffman workspace ----
    DevBuf d_len6, d_rfreq, d_sel, d_gbits, d_hdr, d_bitoff, d_out, d_outbits, d_hmisc;
    // ---- stream / rle1 / decode ----
    DevBuf d_in, d_runflag, d_misc, d_stream, d_dec1, d_dec2, d_dec3;
    // ---- dstream (dstream.cu): window, batch outputs, staging and output pieces, kept for the next stream ----
    DevBuf d_dwin, d_ddec[2];
    PinBuf h_dstage[2], h_dpiece[2];
    bool dstream_open = false;       // one dstream at a time uses them
    // ---- recovery (recover.cu): page-locked pieces of intact bytes on their way to the sink ----
    PinBuf h_rec[2];
    cudaEvent_t ev_rec[2] = {nullptr, nullptr};

    // ---- per-kernel profiling (timing level 2): CUDA events around every launch ----
    KStat kstat[K_COUNT];
    std::vector<cudaEvent_t> ev_pool;
    std::vector<PendingEv> pending;
    size_t ev_used = 0;
    int cur_id = -1;
    int prof_level = 0;
    cudaEvent_t next_event() {
        if (ev_used == ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); ev_pool.push_back(e); }
        return ev_pool[ev_used++];
    }
    void prof_begin(int id, u64 bytes) {
        cur_id = id;
        if (prof_level < 2) return;
        PendingEv p; p.id = id; p.bytes = bytes; p.a = next_event(); p.b = next_event();
        cudaEventRecord(p.a, stream);
        pending.push_back(p);
    }
    void prof_end() {
        launches++;
        if (prof_level < 2 || pending.empty()) return;
        cudaEventRecord(pending.back().b, stream);
    }
    void prof_collect() {          // call after a stream synchronize
        for (auto &p : pending) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) { kstat[p.id].ms += ms; kstat[p.id].launches++; kstat[p.id].bytes += p.bytes; }
        }
        pending.clear();
        ev_used = 0;
    }

    void fail(const char *what, cudaError_t e, const char *file, int line) {
        err = std::string(what) + ": " + cudaGetErrorString(e) + " at " + file + ":" + std::to_string(line);
    }
    ~bz2b200_ctx();
};

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ u32 warp_incl_sum(u32 v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= o) v += t;
    }
    return v;
}
__device__ __forceinline__ int warp_incl_max(int v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) >= o) v = max(v, t);
    }
    return v;
}
// Exclusive sum over the 256 threads of a CTA. `ws` = 8+ u32 of shared scratch. All threads call.
__device__ __forceinline__ u32 block_excl_sum(u32 v, u32 *ws, u32 &total) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    u32 inc = warp_incl_sum(v);
    __syncthreads();
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    u32 wsum = (lane < (int)(blockDim.x >> 5)) ? ws[lane] : 0;
    u32 winc = warp_incl_sum(wsum);
    u32 wbase = __shfl_sync(0xffffffffu, winc, w) - __shfl_sync(0xffffffffu, wsum, w);
    total = __shfl_sync(0xffffffffu, winc, (blockDim.x >> 5) - 1);
    return wbase + inc - v;
}
// Exclusive running max over the threads of a CTA (identity = -1). `ws` = 8+ ints of scratch.
__device__ __forceinline__ int block_excl_max(int v, int *ws, int &total) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = warp_incl_max(v);
    __syncthreads();
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    int wv = (lane < (int)(blockDim.x >> 5)) ? ws[lane] : -1;
    int winc = warp_incl_max(wv);
    int wprev = __shfl_up_sync(0xffffffffu, winc, 1);
    if (lane == 0) wprev = -1;
    int wbase = __shfl_sync(0xffffffffu, wprev, w);
    total = __shfl_sync(0xffffffffu, winc, (blockDim.x >> 5) - 1);
    int prev = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) prev = -1;
    return max(wbase, prev);
}
// Exclusive running min FROM THE RIGHT over the threads of a CTA: min of v over all higher threads
// (identity = 0x7fffffff). `ws` = 8+ ints of scratch. All threads call.
__device__ __forceinline__ int block_excl_min_rev(int v, int *ws, int &total) {
    const int INF = 0x7fffffff;
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_down_sync(0xffffffffu, inc, o);
        if (lane + o < 32) inc = min(inc, t);
    }
    __syncthreads();
    if (lane == 0) ws[w] = inc;
    __syncthreads();
    int wv = (lane < (int)(blockDim.x >> 5)) ? ws[lane] : INF;
    int winc = wv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_down_sync(0xffffffffu, winc, o);
        if (lane + o < 32) winc = min(winc, t);
    }
    int wnext = __shfl_down_sync(0xffffffffu, winc, 1);
    if (lane == 31) wnext = INF;
    int wbase = __shfl_sync(0xffffffffu, wnext, w);
    total = __shfl_sync(0xffffffffu, winc, 0);
    int nxt = __shfl_down_sync(0xffffffffu, inc, 1);
    if (lane == 31) nxt = INF;
    return min(wbase, nxt);
}
#endif

// stage entry points (host side, implemented in the .cu files)
int bz_stage_blocks(bz2b200_ctx *ctx, int nblk, const u8 *const *blk, const u32 *len, Batch &B);
int bz_make_batch_dev(bz2b200_ctx *ctx, int nblk, u32 stride, u32 max_n, const u8 *dT, const u32 *dlen, Batch &B);
// d_usedbits (optional, [nblk*8] u32): the 256-bit used-byte bitmap of every block, a by-product of the byte histogram
int bz_bwt_batch(bz2b200_ctx *ctx, const Batch &B, u8 *d_bwt /*[nblk*stride]*/, u32 *d_key /*[nblk]*/,
                 u32 *d_usedbits = nullptr);
int bz_mtf_batch(bz2b200_ctx *ctx, const Batch &B, const u8 *d_bwt, u16 *d_sym /*[nblk*(stride)]*/, u32 *d_m,
                 u32 *d_freq /*[nblk*256]*/, u8 *d_used /*[nblk*32]*/, bool used_ready = false);
struct HufOut {
    u8 *d_out;          // [nblk * out_stride] packed bits, zero padded
    u64 *d_bits;        // [nblk]
    size_t out_stride;  // bytes per block, multiple of 16
    u8 *d_len6;         // [nblk*6*258] final code lengths
    u8 *d_sel;          // [nblk*sel_stride] selectors
    u32 sel_stride;
    u32 *d_ntab;        // [nblk]
};
// emit_header: 1 = full compress_block output (block magic, crc, rand bit, key first), 0 = huf_encode only
int bz_huf_batch(bz2b200_ctx *ctx, const Batch &B, const u16 *d_sym, const u32 *d_m, const u32 *d_freq,
                 const u8 *d_used, int emit_header, const u32 *d_crc, const u32 *d_key, HufOut &out);

// rle1.cu
int bz_rle1_window(bz2b200_ctx *ctx, const u8 *d_x, u32 W, int level, bool is_eof, u32 off_from, u32 max_blocks,
                   Batch &B, u32 *nblocks, u32 *consumed, std::vector<u32> *h_spans, bool plan_only,
                   u32 stop_at = 0xFFFFFFFFu, int skip = 0, u32 s0 = 0);
int bz_crc_dev(bz2b200_ctx *ctx, const u8 *d_x, u32 n, u32 *d_crc_out);
// api.cu
int bz_compress_batch(bz2b200_ctx *ctx, const Batch &B, const u32 *d_crc, HufOut &H);
// Contexts of this process on one device, and a lock per device.  The decoder's walkers spin on flags their producer
// kernel sets (decode_bounds.cuh); with several contexts on one device it runs that phase under the lock.
int bz_contexts_on_device(int device);
std::mutex &bz_device_lock(int device);

// ---- decode.cu: the decode core shared by bz2b200_decompress_stream, bz2b200_decompress_stream_multi and the dstream ----
// It decodes the chain of blocks and footers that starts in bits [8*lo, hi_bit) of the input; the device holds bytes
// [lo, lo + len) of it, followed by 64 zero bytes.  Bit positions it reports are absolute (from the input's start).
enum { DEC_BLOCK = 0, DEC_FOOTER = 1, DEC_STREAM = 2 };
struct DecEvent {                  // in chain order
    u64 bit;                       // where the element starts
    u32 val;                       // block: stored CRC; footer: stored combined CRC; stream: level of its header
    u32 nblock;                    // block: RLE1 length
    int kind;
};
constexpr long long DEC_ENDED = 1ll << 62;   // chain end after the footer of the input's last stream
constexpr int DEC_ABORTED = 1;               // DecSink::chain_start gave up (another window failed)
struct DecSink {
    // absolute bit where the window's chain begins (DEC_ENDED: before the window), < 0 = abort; called once, after
    // the first batch's entropy decode, when the window did not know its start
    virtual long long chain_start() { return -1; }
    // the chain leaves the window at this absolute bit (or DEC_ENDED); may be called more than once with one value
    virtual void chain_end(long long) {}
    // a batch decodes to `nbytes`; `last` = no element of the window follows.  Sets the device buffer the bytes are
    // written to (>= nbytes + 64) and optionally a host destination the core copies them to before its CRC check.
    virtual int counted(u64 nbytes, bool last, u8 **d_out, u8 **h_out) = 0;
    // the batch's bytes in d_out passed their block CRCs
    virtual int ready(const u8 *, u64) { return BZ2B200_OK; }
    virtual ~DecSink() {}
};
struct DecWindow {
    const u8 *in; size_t in_lo, n; // host bytes [in_lo, n) of the input, in[0] = byte in_lo; n = the input's end when
                                   // the window is the last one (a footer whose header byte would be n ends the input)
    const u8 *d_win; size_t lo, len;
    u64 hi_bit;                    // elements from here on belong to the next window (~0: none)
    long long expect;              // absolute bit of the first element, -1 = ask DecSink::chain_start
    u32 combined;                  // running combined CRC of the stream at `expect` (when expect >= 0)
    u32 max_block;                 // buffers and bounds of every block
    const std::vector<u64> *cand;  // candidate bits relative to d_win, sorted by position, bit 63 = footer magic
};
constexpr u64 DEC_FOOT = 1ull << 63;         // candidate flag: a footer magic
constexpr u32 DEC_BATCH = 128;               // candidate blocks decoded per pass (one pass for 100 MB at level 9)
constexpr u64 RLE1_OPEN = ~0ull;             // RLE1 length of a block that ends with four equal bytes and no count byte
// per candidate block, after the entropy decode: the tail of its decode tables (decode4.cuh DecTables)
struct DecTail { u32 T, alpha, G, status, crc, key; u64 data_bit, end_bit; u32 nsym, ngroups, nblock, pad; };
// The two steps of a batch of at most DEC_BATCH candidate blocks, in the context's decode workspaces.  `max_block`
// bounds every block (the buffer strides).  bz_decode_core runs them on chain members, the recovery driver
// (recover.cu) on every candidate.
struct DecGeom {
    u32 max_block, stride, sel_stride, max_sym, sym_stride, ch_stride;
    explicit DecGeom(u32 max_block);
};
// (a) entropy decode of the candidates starting at bits `starts` of d_bits[0, n) (the data of candidate k does not
// reach past rends[k] unless a chance magic cut it): header, group boundaries, symbols, inverse MTF -> the BWT
// strings in ctx->d_T; db[k] = the candidate's DecTail (status 0 = parsed)
int bz_dec_entropy(bz2b200_ctx *ctx, const DecGeom &g, const u8 *d_bits, size_t n, const std::vector<u64> &starts,
                   const std::vector<u64> &rends, std::vector<DecTail> &db);
// (b) of members k < nblk with hlen[k] > 0 (BWT length; 0 = skip): inverse BWT with origin pointers hkey, de-randomisation
// where hrand[k], RLE1 count -> olen[k] (RLE1_OPEN: no count byte at the end).  Synchronises.
int bz_dec_unbwt(bz2b200_ctx *ctx, const DecGeom &g, u32 nblk, const u32 *hlen, const u32 *hkey, const u32 *hrand,
                 u64 *olen);
// ... then the RLE1 write of those members at d_out + ooff[k] (d_out >= sum olen + 64 bytes) and their block CRCs
// -> crcs[k], valid after the next synchronisation of ctx->stream.  olen = the counted lengths with RLE1_OPEN replaced
// by 0: such a member is not written.
int bz_dec_write(bz2b200_ctx *ctx, const DecGeom &g, u32 nblk, const u64 *olen, const u64 *ooff, u8 *d_out, u32 *crcs);
int bz_dec_candidates(bz2b200_ctx *ctx, const u8 *d_win, size_t len, u32 cap, std::vector<u64> &cand);
// test knob BZ2B200_MULTI_DEC_CHANCE: spurious block candidates, as chance magics inside compressed data would be
void bz_add_chance_candidates(std::vector<u64> &cand);
int bz_decode_core(bz2b200_ctx *ctx, const DecWindow &w, DecSink &sink, std::vector<DecEvent> &ev);
// BZ2B200_E_FORMAT (and `err`) when a block of `ev` is longer than 100000 x its own stream's level; `level` = the first
// stream's, for blocks before any stream event
int bz_check_block_sizes(std::string &err, int level, const std::vector<DecEvent> &ev);
