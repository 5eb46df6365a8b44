// rle1.cu -- RLE1 run collapsing, block splitting and block CRC32 on the device.
//
// Replaces the RLE1Block iterator (reference src/tools/rle1.rs:33-264: refill_buffer :63,
// get_block :89, count_dups :226, next :250) and do_crc (src/tools/crc.rs:15-22).
//
// The reference scans the file serially, two bytes per step, and cuts a block when
// out_len + (cursor - start) >= block_size (rle1.rs:110).  Here the same block ends are derived
// in closed form (SURVEY App. C) from three per-position arrays built by parallel scans over an
// input window:
//   RS[i]    start of the maximal run containing i
//   OUT[i]   bytes the greedy RLE1 emits for [0,i) (literal 1, group start 5, rest of group 0);
//            groups are the 255-byte chunks of a run that are >= 4 long (count_dups takes <= 251)
//   LASTQ[i] last group start <= i
// A single warp then walks the chain s_{k+1} = e(s_k): binary search of OUT for the first position
// whose output offset reaches block_size-1, the cursor-parity rule of the reference's stride-2 scan
// ("a group at q is seen at cursor q if q-start is odd, else at q+1"), and the exit cursor
// c = start+1 | start+R | start+R+1.  A block that begins inside a run restarts the run count, so
// its first run is parsed from the block start in closed form.  With BZ2B200_LIBBZ2 the chain is libbz2's instead
// (plan_block_libbz2): a block ends at the first chunk end where OUT reaches OUT[s] + B, and runs are chunked from
// their own start across block starts; both chain variants (BZ2B200_CHAIN_TABLES) evaluate links with it.
// Finally one thread per input byte writes the RLE1 bytes straight into the fixed-stride batch
// text array consumed by the BWT stage, and the block CRCs are computed as a polynomial in
// X = x^(8*PIECE) over end-aligned pieces (leading zero bytes do not change a zero-init CRC).
#include "common.cuh"
#include <algorithm>
#include <stdlib.h>

namespace {

constexpr u32 CRC_POLY = 0x04C11DB7u;
constexpr int PIECE = 1024;          // bytes per CRC piece (one thread)
constexpr u32 NOQ = 0xFFFFFFFFu;

struct BlockRec {        // one per planned block, all positions window relative
    u32 s, e;            // input span [s, e)
    u32 re;              // end of the first run (parsed from s)
    u32 g_last;          // end of the last group taken in this block (s if none)
    u32 out_re;          // output bytes for [s, re)
    u32 out_g;           // output bytes for [s, g_last)
    u32 out_len;         // RLE1 block length
    u32 last;            // 1 = final block of the stream
};

// ---------------------------------------------------------------------------------------
// GF(2) helpers for CRC combination (MSB-first polynomials, bit k <-> x^k)
// ---------------------------------------------------------------------------------------
__host__ __device__ inline u32 gf_mul(u32 a, u32 b) {
    u32 r = 0;
    for (int i = 31; i >= 0; i--) {
        r = (r << 1) ^ ((r & 0x80000000u) ? CRC_POLY : 0u);
        if ((b >> i) & 1u) r ^= a;
    }
    return r;
}
__host__ __device__ inline u32 gf_pow_x8(u64 nbytes) {      // x^(8 nbytes) mod P
    u32 result = 1, base = 0x100;                            // base = x^8
    while (nbytes) {
        if (nbytes & 1) result = gf_mul(result, base);
        base = gf_mul(base, base);
        nbytes >>= 1;
    }
    return result;
}

__device__ __forceinline__ void make_crc_table(u32 *tab) {
    u32 c = threadIdx.x << 24;
#pragma unroll
    for (int k = 0; k < 8; k++) c = (c & 0x80000000u) ? (c << 1) ^ CRC_POLY : (c << 1);
    tab[threadIdx.x] = c;
}

// ---------------------------------------------------------------------------------------
// window scan: RS, OUT and LASTQ in ONE pass over the input window
// ---------------------------------------------------------------------------------------
// Flat tiles of 4096 input bytes (thread = 16 consecutive bytes, loaded as aligned words).  The two running
// quantities that cross tile borders -- the start of the current run (a max) and (last group start, emitted
// bytes) (a max and a sum) -- come from two decoupled look-backs on 64-bit state words:
//   [63:62] 1 = tile aggregate, 2 = inclusive prefix; [59:30] max + 1 (0 = none); [29:0] sum.
// The first version used five kernels (aggregate / scan / apply twice) with byte loads at a 16-byte thread
// stride; it ran at a fifth of the copy bandwidth.
struct Pair { int a; u32 c; };
__device__ __forceinline__ u64 pair_pack(u32 flag, Pair v) { return ((u64)flag << 62) | ((u64)(u32)(v.a + 1) << 30) | (u64)v.c; }
__device__ __forceinline__ Pair pair_unpack(u64 w) {
    Pair v;
    v.a = (int)((w >> 30) & 0x3fffffffu) - 1; v.c = (u32)(w & 0x3fffffffu);
    return v;
}
__device__ __forceinline__ u64 ld_vol64(const u64 *p) {
    u64 v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_vol64(u64 *p, u64 v) { asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }

// All lanes of warp 0 call.  Lane l inspects tile hi - l: a window of 32 predecessors per L2 round trip.
__device__ __forceinline__ Pair pair_lookback(u64 *st, u32 t, Pair agg) {
    const int lane = threadIdx.x & 31;
    Pair ex; ex.a = -1; ex.c = 0;
    if (t == 0) { if (lane == 0) st_vol64(st, pair_pack(2, agg)); return ex; }
    if (lane == 0) st_vol64(st + t, pair_pack(1, agg));
    for (int hi = (int)t - 1;;) {
        int tt = hi - lane;
        u64 w = tt >= 0 ? ld_vol64(st + tt) : (2ull << 62);
        u32 f = (u32)(w >> 62);
        u32 incm = __ballot_sync(0xffffffffu, f == 2);
        u32 nrm = __ballot_sync(0xffffffffu, f == 0);
        u32 need = incm ? ((2u << (__ffs(incm) - 1)) - 1u) : 0xffffffffu;
        if (nrm & need) continue;
        Pair v = pair_unpack(w);
        if (!((need >> lane) & 1u)) { v.a = -1; v.c = 0; }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            v.a = max(v.a, __shfl_xor_sync(0xffffffffu, v.a, o));
            v.c += __shfl_xor_sync(0xffffffffu, v.c, o);
        }
        ex.a = max(ex.a, v.a); ex.c += v.c;
        if (incm) break;
        hi -= 32;
    }
    Pair inc; inc.a = max(ex.a, agg.a); inc.c = ex.c + agg.c;
    if (lane == 0) st_vol64(st + t, pair_pack(2, inc));
    return ex;
}

struct ScanArgs {
    const u8 *x; u32 W;
    u32 *RS, *OUT, *LASTQ;      // 16-byte aligned, W + 1 entries each
    u64 *st1, *st2;             // look-back state, one word per tile, zeroed
    u32 *ticket;                // zeroed
};

constexpr int SC_IPT = 16;
constexpr int SC_TILE = BZ_THREADS * SC_IPT;

#ifndef BZ_SCAN_MINB
#define BZ_SCAN_MINB 5      /* 48 registers: five CTAs per SM hide the two look-back waits better than four (0.76 -> 0.67 ms) */
#endif
__global__ void __launch_bounds__(BZ_THREADS, BZ_SCAN_MINB) k_rle_scan(ScanArgs a) {
    __shared__ u32 s_tile;
    __shared__ int wsi[8];
    __shared__ u32 wsu[8];
    __shared__ Pair s_ex1, s_ex2;
    const int tid = threadIdx.x;
    if (tid == 0) s_tile = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const u32 t = s_tile, W = a.W;
    const u32 i0 = t * SC_TILE + tid * SC_IPT;
    // bytes i0-4 .. i0+19 as six words v[0..5] (v[k] = bytes i0-4+4k ..), from aligned loads
    u32 v[6];
    {
        uintptr_t addr = (uintptr_t)(a.x + i0) - 4;
        const u32 *gw = (const u32 *)(addr & ~(uintptr_t)3);
        const u32 mis = (u32)(addr & 3);
        long long j = (long long)i0 - 4 - (long long)mis;       // index (relative to x) of the first byte of gw[0]
        u32 w[7];
#pragma unroll
        for (int k = 0; k < 7; k++) {
            long long jk = j + 4 * k;
            w[k] = (jk + 3 >= 0 && jk < (long long)W) ? __ldg(gw + k) : 0u;
        }
#pragma unroll
        for (int k = 0; k < 6; k++) v[k] = __funnelshift_r(w[k], w[k + 1], mis * 8);
    }
#define XB(r) ((v[((r) + 4) >> 2] >> ((((r) + 4) & 3) * 8)) & 255u)      /* byte i0 + r, r in [-4, 19] */
    // ---- run starts ----
    int last = -1; u32 bdmask = 0;
#pragma unroll
    for (int r = 0; r < SC_IPT; r++) {
        u32 i = i0 + r;
        if (i < W && (i == 0 || XB(r) != XB(r - 1))) { last = (int)i; bdmask |= 1u << r; }
    }
    int tot1;
    int rs = block_excl_max(last, wsi, tot1);
    if (tid < 32) {
        Pair agg; agg.a = tot1; agg.c = 0;
        Pair ex = pair_lookback(a.st1, t, agg);
        if (tid == 0) s_ex1 = ex;
    }
    __syncthreads();
    rs = max(rs, s_ex1.a);
    // ---- greedy parse: bytes emitted "at" each position (literal 1, group start 5, rest of a group 0) ----
    u32 qmask = 0, litmask = 0, sum = 0;
    int lq = -1;
    const bool full = i0 + SC_IPT <= W;
    u32 rsv[SC_IPT];
#pragma unroll
    for (int r = 0; r < SC_IPT; r++) {
        u32 i = i0 + r;
        rsv[r] = 0;
        if (i < W) {
            if ((bdmask >> r) & 1u) rs = (int)i;
            rsv[r] = (u32)rs;
            u32 d = i - (u32)rs;
            u32 co = d - (d / 255u) * 255u;                     // offset inside the 255-byte chunk of the run
            bool grp;
            if (co >= 3) grp = true;                            // chunk start .. i are equal and i >= chunk start + 3
            else {
                u32 c = XB(r);
                grp = (i - co) + 3 < W;
                if (co < 3) grp = grp && XB(r + 1) == c;
                if (co < 2) grp = grp && XB(r + 2) == c;
                if (co < 1) grp = grp && XB(r + 3) == c;
            }
            if (!grp) { litmask |= 1u << r; sum += 1; }
            else if (co == 0) { qmask |= 1u << r; sum += 5; lq = (int)i; }
        }
    }
    if (full) {
        uint4 *o = (uint4 *)(a.RS + i0);
#pragma unroll
        for (int k = 0; k < 4; k++) o[k] = make_uint4(rsv[4 * k], rsv[4 * k + 1], rsv[4 * k + 2], rsv[4 * k + 3]);
    } else {
#pragma unroll
        for (int r = 0; r < SC_IPT; r++) if (i0 + r < W) a.RS[i0 + r] = rsv[r];
    }
    int tq; u32 ts;
    int q = block_excl_max(lq, wsi, tq);
    u32 o = block_excl_sum(sum, wsu, ts);
    if (tid < 32) {
        Pair agg; agg.a = tq; agg.c = ts;
        Pair ex = pair_lookback(a.st2, t, agg);
        if (tid == 0) s_ex2 = ex;
    }
    __syncthreads();
    q = max(q, s_ex2.a);
    o += s_ex2.c;
    u32 ov[SC_IPT], qv[SC_IPT];
#pragma unroll
    for (int r = 0; r < SC_IPT; r++) {
        if ((qmask >> r) & 1u) q = (int)(i0 + r);
        ov[r] = o; qv[r] = q < 0 ? NOQ : (u32)q;
        o += ((litmask >> r) & 1u) + 5u * ((qmask >> r) & 1u);
        if (i0 + r == W - 1) a.OUT[W] = o;
    }
    if (full) {
        uint4 *po = (uint4 *)(a.OUT + i0), *pq = (uint4 *)(a.LASTQ + i0);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            po[k] = make_uint4(ov[4 * k], ov[4 * k + 1], ov[4 * k + 2], ov[4 * k + 3]);
            pq[k] = make_uint4(qv[4 * k], qv[4 * k + 1], qv[4 * k + 2], qv[4 * k + 3]);
        }
    } else {
#pragma unroll
        for (int r = 0; r < SC_IPT; r++) if (i0 + r < W) { a.OUT[i0 + r] = ov[r]; a.LASTQ[i0 + r] = qv[r]; }
    }
#undef XB
}

// ---------------------------------------------------------------------------------------
// the block chain (one warp; lane 0 carries the logic)
// ---------------------------------------------------------------------------------------
struct ChainArgs {
    const u8 *x; const u32 *RS; const u32 *OUT; const u32 *LASTQ;
    u32 W;            // window length
    u32 B;            // block_size = level*100000 - 19 (compress.rs:55)
    u32 is_eof;       // window ends at the end of the stream
    u32 max_blocks;
    u32 max_out;      // largest RLE1 block the batch stride can hold
    u32 s0;           // first block start (window relative)
    u32 stop_at;      // stop the chain at the first block start >= stop_at (shard end), window relative
    u32 out_w;        // OUT[W]: RLE1 bytes of the whole window (read once by the kernel)
    u32 off_from;     // EOF bookkeeping: a group starting at/after this position since the last refill puts the
                      // reference's `remaining` counter one high (rle1.rs:207) -- see DESIGN.md "EOF corner"
    u32 mode;         // BzMode: BZ_MODE_LIBBZ2 plans libbz2's blocks (plan_block_libbz2)
    BlockRec *rec; u32 *nrec; u32 *consumed;
};

// Warp-cooperative lower bound on the monotone array OUT: first x in [lo, hi] with OUT[x] >= target
// (the caller guarantees OUT[hi] >= target).  32 probes per step instead of one: ~6 dependent loads for 1e8.
__device__ u32 warp_lower_bound(const u32 *OUT, u32 lo, u32 hi, long long target) {
    int lane = threadIdx.x & 31;
    while (hi - lo > 32) {
        u32 step = (hi - lo + 31) / 32;
        u64 pp = (u64)lo + (u64)step * (u32)(lane + 1);
        u32 p = pp > hi ? hi : (u32)pp;
        bool ge = (long long)OUT[p] >= target;
        unsigned bal = __ballot_sync(0xffffffffu, ge);
        int f = __ffs(bal) - 1;                                 // last probe is hi, so f >= 0
        u64 nh = (u64)lo + (u64)step * (u32)(f + 1);
        u32 new_hi = nh > hi ? hi : (u32)nh;
        u32 new_lo = f == 0 ? lo : lo + step * (u32)f + 1;
        lo = new_lo; hi = new_hi;
    }
    u32 p = lo + (u32)lane;
    bool ge = p <= hi && (long long)OUT[p] >= target;
    unsigned bal = __ballot_sync(0xffffffffu, ge);
    return lo + (u32)(__ffs(bal) - 1);
}

__device__ u32 run_end_from(const u32 *RS, u32 W, u32 s) {      // first p > s with RS[p] != RS[s] (or W)
    u32 key = RS[s];
    // gallop first: runs are short in most data
    u32 d = 1;
    while (s + d < W && RS[s + d] == key && d < (1u << 30)) d <<= 1;
    u32 lo = s + (d >> 1) + 1, hi = (s + d < W) ? s + d : W;    // answer in [lo, hi]
    if (d == 1) lo = s + 1;
    while (lo < hi) {
        u32 mid = lo + (hi - lo) / 2;
        if (RS[mid] > key) hi = mid; else lo = mid + 1;
    }
    return lo;
}
__device__ u32 group_end(const u8 *x, u32 W, u32 q) {           // q + 4 + dups, dups <= 251 (rle1.rs:226-241)
    u8 c = x[q];
    u32 p = q + 4, lim = min(W, q + 255);
    while (p < lim && x[p] == c) p++;
    return p;
}
__device__ __forceinline__ u32 exit_cursor(u32 g, long long R) {   // SURVEY App. C
    if (R <= 1) return g + 1;
    return (R & 1) ? g + (u32)R : g + (u32)R + 1;
}

enum { PLAN_OK = 0, PLAN_STOP = 1, PLAN_SEARCH = 2 };

// libbz2's block (DESIGN.md §10): every maximal run is cut greedily from its own start into
// chunks of at most 255 bytes (RLE1 size: the length below 4, else 5), and a block ends right after the first chunk at
// which its RLE1 length reaches B.  A block start is therefore a chunk boundary, chunking from it is the global one,
// and OUT (which counts exactly those chunks, 5 bytes at a group start) gives the whole link: the first run is cut
// from s (the window may have begun inside it), then a lower bound on OUT and a round-up to the end of the chunk that
// crossed B.  No cursor parity and no end-of-file arm.  The record uses BlockRec's fields the way k_rle_emit reads them:
// [s, re) is the first run chunked from s, [re, e) the global parse, g_last = e (no trailing literals).
template <bool COOP>
__device__ __forceinline__ int plan_block_libbz2(const ChainArgs &a, u32 s, BlockRec &r) {
    const u32 W = a.W, B = a.B;
    const u32 margin = a.is_eof ? 0u : 1024u;
    r.s = s; r.last = 0;
    u32 re = run_end_from(a.RS, W, s);
    if (!a.is_eof && re + margin > W) return PLAN_STOP;         // run may continue past the window
    const u32 Lc = re - s, nfull = Lc / 255u, rem = Lc % 255u;
    const u32 jb = (B + 4) / 5;                                 // full chunks that reach B on their own
    u32 e, out_len;
    if (jb <= nfull) {                                          // B is reached inside the first run
        e = s + 255u * jb; out_len = 5u * jb;
        r.re = e; r.out_re = out_len;
    } else {
        const u32 out_re = 5u * nfull + (rem >= 4 ? 5u : rem);
        r.re = re; r.out_re = out_re;
        if (out_re >= B) { e = re; out_len = out_re; }          // ... by the run's last, shorter chunk
        else {
            const long long off = (long long)out_re - (long long)a.OUT[re];
            const long long target = (long long)B - off;        // first x > re with OUT[x] >= target
            if ((long long)a.out_w < target) {
                if (!a.is_eof) return PLAN_STOP;
                e = W; out_len = (u32)((long long)a.out_w + off);
            } else {
                u32 x1;
                if (COOP) x1 = warp_lower_bound(a.OUT, re, W, target);
                else {
                    u32 lo = re, hi = W;
                    while (lo < hi) {
                        u32 mid = lo + (hi - lo) / 2;
                        if ((long long)a.OUT[mid] >= target) hi = mid; else lo = mid + 1;
                    }
                    x1 = lo;
                }
                // byte x1 - 1 emitted the bytes that crossed B: a group start (its chunk ends where group_end says) or a
                // literal of a chunk of 1 to 3 equal bytes (the chunk ends with the run)
                const u32 p = x1 - 1;
                if (a.OUT[x1] - a.OUT[p] == 5u) e = group_end(a.x, W, p);
                else { e = x1; const u8 c = a.x[p]; while (e < W && a.x[e] == c) e++; }
                out_len = (u32)((long long)a.OUT[e] + off);
            }
        }
    }
    if (a.is_eof) { if (e == W) r.last = 1; }
    else if (e + margin > W) return PLAN_STOP;                  // needs bytes beyond this window
    r.e = e; r.g_last = e; r.out_g = out_len; r.out_len = out_len;
    if (r.out_len > a.max_out) return PLAN_STOP;
    return PLAN_OK;
}

// One block of the chain: the block that starts at input position s.  COOP = true: called by all lanes with the
// same s (the binary search over OUT is warp cooperative); COOP = false would let a lane plan on its own.
template <bool COOP>
__device__ __forceinline__ int plan_block(const ChainArgs &a, u32 s, BlockRec &r) {
    if (a.mode == BZ_MODE_LIBBZ2) return plan_block_libbz2<COOP>(a, s, r);
    const u32 W = a.W, B = a.B;
    const u32 margin = a.is_eof ? 0u : 1024u;
    r.s = s; r.last = 0;
    // ---- first run, parsed from s ----
    u32 re = run_end_from(a.RS, W, s);
    if (!a.is_eof && re + margin > W) return PLAN_STOP;         // run may continue past the window
    u32 Lc = re - s;
    u32 nfull = Lc / 255u, rem = Lc % 255u;
    u32 ng_avail = nfull + (rem >= 4 ? 1u : 0u);
    u32 jmax = (B - 1 + 4) / 5;                                 // groups j with 5j + 1 < B
    u32 g, out_g;
    bool done = false;
    u32 e = 0;
    if (ng_avail > jmax) {                                      // the size limit falls inside the first run
        g = s + 255u * jmax; out_g = 5u * jmax;
        e = g + 1;
        r.re = re; r.out_re = 0;                                // unused: block ends before re
        done = true;
    } else {
        g = s + 255u * nfull + (rem >= 4 ? rem : 0u);
        out_g = 5u * ng_avail;
        r.re = re; r.out_re = out_g + (re - g);
    }
    bool has_group_after_off = ng_avail > 0 && g > a.off_from;
    if (!done) {
        // OUTs(x) = OUT[x] + off for x >= re
        long long off = (long long)r.out_re - (long long)a.OUT[re];
        long long target = (long long)B - 1 - off;              // first x >= re with OUT[x] >= target
        u32 x1;
        u32 lq_m1 = NOQ, lq_p3 = NOQ;                           // LASTQ[x1 - 1], LASTQ[min(x1 + 3, W - 1)] when the probe below saw them
        bool have_m1 = false, have_p3 = false;
        if ((long long)a.out_w < target) x1 = W + 1;            // never reached inside the window
        else {
            // run-free data emits one byte per input byte, so the answer is usually re + (bytes still to emit):
            // verify that guess with two independent loads before falling back to the search
            long long need = target - (long long)a.OUT[re];
            u64 guess = (u64)re + (u64)(need > 0 ? need : 0);
            bool solved = false;
            if (need <= 0) { x1 = re; solved = true; }
            else if (COOP) {
                // One probe by the whole warp: lane l looks at position guess - 15 + l of OUT and LASTQ.  A few runs per block
                // move the answer a few bytes off the guess, so this usually finds it -- the first position at or above the
                // target whose predecessor is below it -- together with the two LASTQ entries the group test below needs,
                // in ONE round trip instead of four (the chain is a sequence of dependent L2 / DRAM accesses).
                const int lane = threadIdx.x & 31;
                const long long wlo = (long long)guess - 15;
                const long long p = wlo + lane;
                const bool inb = p >= (long long)re && p <= (long long)W;
                const u32 o = inb ? a.OUT[p] : 0u;
                const u32 lqv = (p >= 0 && p < (long long)W) ? a.LASTQ[p] : NOQ;
                const unsigned bal = __ballot_sync(0xffffffffu, inb && (long long)o >= target);
                const unsigned inm = __ballot_sync(0xffffffffu, inb);
                if (bal) {
                    const int f = __ffs(bal) - 1;
                    const long long xp = wlo + f;
                    if (xp == (long long)re || (f > 0 && ((inm >> (f - 1)) & 1u))) {      // its predecessor was probed and is below
                        x1 = (u32)xp; solved = true;
                        if (f >= 1) { lq_m1 = __shfl_sync(0xffffffffu, lqv, f - 1); have_m1 = true; }
                        const long long hl = (long long)min(x1 + 3, W - 1) - wlo;
                        if (hl >= 0 && hl < 32) { lq_p3 = __shfl_sync(0xffffffffu, lqv, (int)hl); have_p3 = true; }
                    }
                }
            }
            if (!solved) {
                if (guess <= W && (long long)a.OUT[guess] >= target && (long long)a.OUT[guess - 1] < target) x1 = (u32)guess;
                else if (COOP) {
                    // search +-512 positions first (two probe rounds, and that neighbourhood was prefetched) before the whole
                    // window (five rounds)
                    u64 g64 = guess > W ? W : guess;
                    u32 lo_w = g64 > (u64)re + 512 ? (u32)g64 - 512u : re;
                    u32 hi_w = g64 + 512 < (u64)W ? (u32)g64 + 512u : W;
                    if ((long long)a.OUT[lo_w] < target && (long long)a.OUT[hi_w] >= target) x1 = warp_lower_bound(a.OUT, lo_w, hi_w, target);
                    else x1 = warp_lower_bound(a.OUT, re, W, target);
                } else {                                        // one thread on its own (k_rle_tab_fill): plain binary search
                    u32 lo = re, hi = W;                        // OUT[W] >= target was checked above
                    while (lo < hi) {
                        u32 mid = lo + (hi - lo) / 2;
                        if ((long long)a.OUT[mid] >= target) hi = mid; else lo = mid + 1;
                    }
                    x1 = lo;
                }
            }
        }
        u32 gl = NOQ;                                           // start of the last taken global group
        if (x1 <= W) {
            // the only group that can sit exactly at the limit starts in [x1, x1+3]
            u32 hiq = min(x1 + 3, W - 1);
            // both look-ups depend only on x1: issue them together (each is a DRAM/L2 round trip on the serial chain)
            u32 q1_pre = x1 < W ? (have_p3 ? lq_p3 : a.LASTQ[hiq]) : NOQ;
            u32 qp_pre = x1 > re ? (have_m1 ? lq_m1 : a.LASTQ[x1 - 1]) : NOQ;
            if (x1 < W) {
                u32 q1 = q1_pre;
                if (q1 != NOQ && q1 >= x1 && q1 >= re && (long long)a.OUT[q1] + off == (long long)B - 1) {
                    // taken iff it is seen at cursor q1 itself: (q1 - previous group end) odd
                    u32 gp = g;
                    if (q1 > 0) {
                        u32 qp = a.LASTQ[q1 - 1];
                        if (qp != NOQ && qp >= re) gp = group_end(a.x, W, qp);
                    }
                    if (((q1 - gp) & 1u) == 1u) gl = q1;
                }
            }
            if (gl == NOQ && x1 > re) {
                u32 qp = qp_pre;
                if (qp != NOQ && qp >= re) gl = qp;
            }
        } else if (W > re) {
            u32 qp = a.LASTQ[W - 1];
            if (qp != NOQ && qp >= re) gl = qp;
        }
        if (gl != NOQ) {
            u32 out_gl = a.OUT[gl];                             // independent of the group_end walk below
            g = group_end(a.x, W, gl);
            out_g = (u32)((long long)out_gl + off + 5);
            if (gl >= a.off_from) has_group_after_off = true;
        }
        // else: no global group taken, the literal stretch continues from the first run's last group
        long long R = (long long)B - (long long)out_g;
        e = exit_cursor(g, R);
    }
    // ---- window / EOF handling ----
    if (a.is_eof) {
        u32 lim = has_group_after_off ? W - 1 : W - 2;          // size exit only at a cursor visited before the EOF arms
        if (W < 2 || e > lim || e > W) {                         // final block takes everything (rle1.rs:115-139)
            e = W; r.last = 1;
            if (!done) {
                // every group up to the end is taken
                if (W > re) {
                    u32 qp = a.LASTQ[W - 1];
                    if (qp != NOQ && qp >= re) {
                        long long off = (long long)r.out_re - (long long)a.OUT[re];
                        g = group_end(a.x, W, qp);
                        out_g = (u32)((long long)a.OUT[qp] + off + 5);
                    }
                }
            } else {
                // limit fell inside the first run but the file ends here: recompute as "all groups taken"
                g = s + 255u * nfull + (rem >= 4 ? rem : 0u);
                out_g = 5u * ng_avail;
                r.out_re = out_g + (re - g);
            }
        }
    } else if (e + margin > W) {
        return PLAN_STOP;                                       // needs bytes beyond this window
    }
    r.e = e; r.g_last = g; r.out_g = out_g;
    r.out_len = out_g + (e - g);
    if (r.out_len > a.max_out) return PLAN_STOP;                // cannot happen for level <= 9; guards the batch stride
    return PLAN_OK;
}

// The chain s_{k+1} = e(s_k) is sequential, and one warp needs ~3 us per link (a few dependent L2 / DRAM accesses plus
// ~600 dependent instructions with nobody to hide their latency behind): 0.36 ms for the 112 blocks of 100 MB, paid once
// per GPU and in SERIES across the GPUs of a multi-GPU call.  So the links are evaluated SPECULATIVELY in parallel:
// a block emits B .. B+5 bytes, hence the k-th block after a known start s begins where the global output offset OUT is
// within [OUT[s] + k (B - 10), OUT[s] + k (B + 15)] (the slack covers runs that are re-chunked at a block start).
//   k_rle_tab_bounds  the candidate window of every block of a segment of 128 blocks (three binary searches per block)
//   k_rle_tab_fill    one THREAD per candidate start evaluates the full link e(s) (plan_block, ~10^5 of them per segment)
//   k_rle_chain       walks the segment: a link is one table look-up; a start outside its window (long runs) falls back
//                     to the cooperative evaluation, so the tables only ever make the walk faster, never different
// The running state (blocks planned, next start, finished) lives in device memory, so segment after segment is launched
// without any host round trip.
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

constexpr u32 CH_SEG = 128;                                      // blocks per speculative segment
__host__ __device__ inline u32 tab_cap(u32 k) { return 32u * k + 256u; }                        // candidates kept for link k (k >= 1)
__host__ __device__ inline u32 tab_off(u32 k) { return 16u * k * (k - 1u) + 256u * (k - 1u); }  // sum of tab_cap(1 .. k-1)
constexpr u32 TAB_ENTRIES = 16u * (CH_SEG + 1) * CH_SEG + 256u * CH_SEG;                        // tab_off(CH_SEG + 1)
constexpr u32 REC_BAD = 0xFFFFFFFFu;

struct ChainState { u32 nb, s, done, hits; };                    // blocks planned so far, start of the next block, chain finished, table hits

struct TabArgs {
    ChainArgs a;
    ChainState *state;
    u32 *tlo, *tcnt;          // [CH_SEG + 1] candidate window of link k of the current segment
    BlockRec *tab;            // [TAB_ENTRIES]
};

__device__ u32 lower_bound_out(const u32 *OUT, u32 lo, u32 hi, u64 target) {     // first x in [lo, hi] with OUT[x] >= target, hi + 1 if none
    if ((u64)OUT[hi] < target) return hi + 1;
    while (lo < hi) {
        u32 mid = lo + (hi - lo) / 2;
        if ((u64)OUT[mid] >= target) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__global__ void __launch_bounds__(128) k_rle_tab_bounds(TabArgs t) {
    const u32 k = blockIdx.x * 128 + threadIdx.x + 1;            // link k: the k-th block after the segment's first one
    if (k > CH_SEG) return;
    const ChainState st = *t.state;
    t.tcnt[k] = 0;
    if (st.done || st.s >= t.a.W) return;
    const u32 W = t.a.W, B = t.a.B;
    const u64 base = t.a.OUT[st.s];
    u32 lo = lower_bound_out(t.a.OUT, st.s, W, base + (u64)k * (B - 10));
    if (lo > W) return;
    u32 hi = lower_bound_out(t.a.OUT, lo, W, base + (u64)k * (B + 15) + 1);
    if (hi > W) hi = W;
    u32 cap = tab_cap(k);
    if (hi - lo + 1 > cap) {                                     // keep the part around the expected offset (blocks average B + 2.5 bytes)
        u32 c = lower_bound_out(t.a.OUT, lo, hi, base + (u64)k * B + (5ull * k) / 2);
        u32 from = c > lo + cap / 2 ? c - cap / 2 : lo;
        if (from + cap - 1 > hi) from = hi + 1 - cap;
        lo = from; hi = from + cap - 1;
    }
    t.tlo[k] = lo; t.tcnt[k] = hi - lo + 1;
}

__global__ void __launch_bounds__(128) k_rle_tab_fill(TabArgs t) {
    const u32 k = blockIdx.y + 1;
    const u32 j = blockIdx.x * 128 + threadIdx.x;
    if (j >= t.tcnt[k]) return;
    const u32 s = t.tlo[k] + j;
    BlockRec r;
    r.out_len = REC_BAD;
    if (s < t.a.W) {
        ChainArgs a = t.a;
        a.out_w = a.OUT[a.W];
        if (plan_block<false>(a, s, r) != PLAN_OK) r.out_len = REC_BAD;
    }
    t.tab[tab_off(k) + j] = r;
}

__global__ void __launch_bounds__(32) k_rle_chain(TabArgs t) {
    // all 32 lanes run the same control flow (every value is warp-uniform); lane 0 writes the results
    ChainArgs a = t.a;
    const int lane = threadIdx.x;
    const u32 W = a.W;
    ChainState st = *t.state;
    if (st.done) return;
    a.out_w = a.OUT[W];
    u32 s = st.s, nb = st.nb, hits = st.hits;
    u32 span = a.B;
    bool finished = true;                                        // left the loop for good (not because the segment is over)
    for (u32 k = 0;; k++) {
        if (!(s < W && s < a.stop_at && nb < a.max_blocks)) break;
        if (k > CH_SEG) { finished = false; break; }             // the next segment continues from here
        BlockRec r;
        bool have = false;
        if (t.tab && k >= 1) {
            u32 lo = t.tlo[k], cnt = t.tcnt[k];
            if (s >= lo && s - lo < cnt) {
                const uint4 *src = (const uint4 *)(t.tab + tab_off(k) + (s - lo));
                uint4 q0 = src[0], q1 = src[1];
                r.s = q0.x; r.e = q0.y; r.re = q0.z; r.g_last = q0.w; r.out_re = q1.x; r.out_g = q1.y; r.out_len = q1.z; r.last = q1.w;
                have = r.out_len != REC_BAD && r.s == s;
                hits += have ? 1u : 0u;
            }
        }
        if (!have) {
            {   // lanes 0..15: around the next block's start; lanes 16..31: around its end.  128-byte lines of u32 = 32 entries.
                u64 c = (u64)s + (u64)span * (lane < 16 ? 1u : 2u);
                long long p = (long long)c - 1024 + (long long)(lane & 15) * 128;       // 2 KB window of positions
                if (p >= 0 && (u64)p + 32 < (u64)W) {
                    prefetch_l2(a.OUT + p); prefetch_l2(a.OUT + p + 32); prefetch_l2(a.OUT + p + 64); prefetch_l2(a.OUT + p + 96);
                    prefetch_l2(a.LASTQ + p); prefetch_l2(a.LASTQ + p + 32); prefetch_l2(a.LASTQ + p + 64); prefetch_l2(a.LASTQ + p + 96);
                    prefetch_l2(a.RS + p); prefetch_l2(a.RS + p + 32); prefetch_l2(a.RS + p + 64); prefetch_l2(a.RS + p + 96);
                    prefetch_l2(a.x + p);
                }
            }
            if (plan_block<true>(a, s, r) != PLAN_OK) break;
        }
        if (lane == 0) a.rec[nb] = r;
        nb++;
        span = r.e - s;
        s = r.e;
    }
    if (lane == 0) {
        ChainState o; o.nb = nb; o.s = s; o.done = finished ? 1u : 0u; o.hits = hits;
        *t.state = o;
        *a.nrec = nb; *a.consumed = s;
    }
}

// ---------------------------------------------------------------------------------------
// RLE1 byte emission: thread per input byte of each planned block
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BZ_THREADS) k_rle_emit(const u8 *x, u32 W, const u32 *RS, const u32 *OUT,
                                                         const BlockRec *rec, u8 *T, u32 *len, u32 stride) {
    u32 k = blockIdx.y;
    BlockRec r = rec[k];
    u32 span = r.e - r.s;
    u32 base = blockIdx.x * BZ_TILE;
    if (base >= span) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) len[k] = r.out_len;
    u8 *out = T + (size_t)k * stride;
    long long off = (long long)r.out_re - (long long)OUT[min(r.re, W)];
#pragma unroll 4
    for (int q = 0; q < BZ_IPT; q++) {
        u32 rel = base + q * BZ_THREADS + threadIdx.x;
        if (rel >= span) continue;
        u32 i = r.s + rel;
        u8 c = x[i];
        if (i >= r.g_last) {                                    // trailing literals of the block
            out[r.out_g + (i - r.g_last)] = c;
        } else if (i < r.re) {                                  // first run, chunked from s
            u32 j = (i - r.s) / 255u, cs = r.s + j * 255u;
            u32 cl = min(255u, r.re - cs);
            if (cl >= 4) {
                if (i == cs) {
                    u8 *o = out + 5u * j;
                    o[0] = c; o[1] = c; o[2] = c; o[3] = c; o[4] = (u8)(cl - 4);
                }
            } else out[5u * j + (i - cs)] = c;
        } else {                                                // global parse: OUT[i+1] - OUT[i] = bytes emitted at i
            u32 o0 = OUT[i], o1 = OUT[i + 1];
            u32 o = (u32)((long long)o0 + off);
            if (o1 - o0 == 1u) out[o] = c;                      // literal
            else if (o1 != o0) {                                // group start (5 bytes); the rest of a group emits nothing
                u32 ge = group_end(x, W, i);
                out[o] = c; out[o + 1] = c; out[o + 2] = c; out[o + 3] = c; out[o + 4] = (u8)(ge - i - 4);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// CRC32 (crc.rs:15-22): pieces aligned to the END of each span
// ---------------------------------------------------------------------------------------
// spans[k*span_stride + 0/1] = s/e (BlockRec has them in its first two words), or one explicit span.
__global__ void __launch_bounds__(256) k_crc_pieces(const u8 *x, const u32 *spans, u32 span_stride, u32 s0, u32 e0,
                                                    u32 *part, u32 parts_stride, u32 xp /* x^(8*PIECE) */) {
    __shared__ u32 tab[256];
    __shared__ u32 red[256];
    make_crc_table(tab);
    u32 k = blockIdx.y;
    u32 s = spans ? spans[(size_t)k * span_stride] : s0, e = spans ? spans[(size_t)k * span_stride + 1] : e0;
    u32 span = e - s;
    u32 npieces = (span + PIECE - 1) / PIECE;
    u32 p = blockIdx.x * 256 + threadIdx.x;                     // piece 0 ends at e
    __syncthreads();
    u32 crc = 0;
    if (p < npieces) {
        u32 hi = e - p * PIECE;
        u32 lo = (hi - s >= (u32)PIECE) ? hi - PIECE : s;
        const u8 *d = x + lo;
        u32 n = hi - lo;
        // Pieces of neighbouring threads are 1 KB apart, so every load instruction touches 32 cache lines: byte
        // loads made the L1 tag stage the limiter.  Load 16 bytes at a time from 16-byte aligned addresses.
        u32 i = 0;
        for (; i < n && (((uintptr_t)(d + i)) & 15u); i++) crc = (crc << 8) ^ tab[(crc >> 24) ^ d[i]];
        for (; i + 16 <= n; i += 16) {
            uint4 q = *(const uint4 *)(d + i);
            u32 w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
#pragma unroll
                for (int j = 0; j < 4; j++) crc = (crc << 8) ^ tab[(crc >> 24) ^ ((w[k] >> (8 * j)) & 255u)];
            }
        }
        for (; i < n; i++) crc = (crc << 8) ^ tab[(crc >> 24) ^ d[i]];
    }
    // CTA partial = sum_j crc_j * X^j  (j = threadIdx.x): pairwise tree with powers X^(2^l)
    red[threadIdx.x] = crc;
    __syncthreads();
    u32 pw = xp;
    for (int st = 1; st < 256; st <<= 1) {
        u32 v = 0;
        bool act = (threadIdx.x % (2 * st)) == 0;
        if (act) v = red[threadIdx.x] ^ gf_mul(red[threadIdx.x + st], pw);
        __syncthreads();
        if (act) red[threadIdx.x] = v;
        __syncthreads();
        pw = gf_mul(pw, pw);
    }
    if (threadIdx.x == 0 && blockIdx.x * 256 < npieces) part[(size_t)k * parts_stride + blockIdx.x] = red[0];
}

__global__ void __launch_bounds__(32) k_crc_final(const u32 *spans, u32 span_stride, u32 s0, u32 e0, const u32 *part,
                                                  u32 parts_stride, u32 xp256 /* x^(8*PIECE*256) */, u32 *crc_out) {
    u32 k = blockIdx.x;
    if (threadIdx.x != 0) return;
    u32 s = spans ? spans[(size_t)k * span_stride] : s0, e = spans ? spans[(size_t)k * span_stride + 1] : e0;
    u32 span = e - s;
    u32 npieces = (span + PIECE - 1) / PIECE;
    u32 nparts = (npieces + 255) / 256;
    u32 acc = 0;
    for (int c = (int)nparts - 1; c >= 0; c--) acc = gf_mul(acc, xp256) ^ part[(size_t)k * parts_stride + c];
    // init ~0 contributes 0xFFFFFFFF * x^(8 len); final complement (crc.rs:17,:21)
    u32 init = gf_mul(0xFFFFFFFFu, gf_pow_x8(span));
    crc_out[k] = ~(acc ^ init);
}

}  // namespace

#define LAUNCH_OK()                                                  \
    do {                                                             \
        ctx->prof_end();                                             \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) { ctx->fail("kernel launch", e_, __FILE__, __LINE__); return BZ2B200_E_CUDA; } \
    } while (0)

// Plans and emits the RLE1 blocks of one input window that is already on the device.
// On return: *nblocks blocks were written into the context's batch text array (ctx->d_T, ctx->d_len,
// ctx->d_crc), `B` describes them, *consumed = input bytes covered.  h_rec (optional) receives the records.
int bz_rle1_window(bz2b200_ctx *ctx, const u8 *d_x, u32 W, int level, bool is_eof, u32 off_from, u32 max_blocks,
                   Batch &B, u32 *nblocks, u32 *consumed, std::vector<u32> *h_spans, bool plan_only, u32 stop_at,
                   int skip, u32 s0) {
    // skip bit0: the scans of the immediately preceding call on the same window are still in d_runflag;
    // skip bit1: so is the chain result in d_misc (bz2b200_shard_scan_dev -> _plan_dev -> _compress_dev)
    const bool skip_scan = skip & 1, skip_chain = skip & 2;
    cudaStream_t st = ctx->stream;
    u32 Bsz = (u32)level * 100000u - 19u;
    u32 max_n = Bsz + 8;                                        // RLE1 block length <= B + 5 (SURVEY App. C)
    u32 stride = ((max_n + 64 + BZ_TILE - 1) / BZ_TILE) * BZ_TILE;
    u32 tiles = (W + BZ_TILE - 1) / BZ_TILE;
    const size_t W4 = ((size_t)W + 1 + 3) & ~(size_t)3;          // entries per array, keeps all three 16-byte aligned
    BZ_CHECK(ctx->d_runflag.ensure(W4 * 4 * 3 + 64));
    u32 *RS = ctx->d_runflag.as<u32>();
    u32 *OUT = RS + W4;
    u32 *LASTQ = OUT + W4;
    const size_t state_bytes = ((size_t)tiles * 8 * 2 + 64 + 15) & ~(size_t)15;     // st1 | st2 | ticket
    BZ_CHECK(ctx->d_misc.ensure(state_bytes + (size_t)max_blocks * sizeof(BlockRec) + 256));
    u64 *st1 = ctx->d_misc.as<u64>();
    u64 *st2 = st1 + tiles;
    u32 *ticket = (u32 *)(st2 + tiles);
    BlockRec *rec = (BlockRec *)(ctx->d_misc.as<u8>() + state_bytes);
    u32 *d_small = (u32 *)(rec + max_blocks);                   // [0]=nrec [1]=consumed
    BZ_CHECK(ctx->h_small.ensure(64 + (size_t)max_blocks * sizeof(BlockRec)));

    // skip_scan: the scan of the immediately preceding call on the same window is still in d_runflag
    if (!skip_scan && W > 0) {
        BZ_CHECK(cudaMemsetAsync(st1, 0, state_bytes, st));
        ScanArgs sa;
        sa.x = d_x; sa.W = W; sa.RS = RS; sa.OUT = OUT; sa.LASTQ = LASTQ; sa.st1 = st1; sa.st2 = st2; sa.ticket = ticket;
        if (!ctx->arrival) {
            ctx->prof_begin(K_RLE_SCAN, (u64)W * 13); k_rle_scan<<<tiles, BZ_THREADS, 0, st>>>(sa); LAUNCH_OK();
        } else {
            // the window is still being uploaded: scan the tiles of every chunk as it lands (tiles take their index
            // from the ticket counter, so consecutive launches simply continue; a tile looks 19 bytes ahead)
            Arrival &A = *ctx->arrival;
            const size_t nev = A.ev->size();
            u32 launched = 0;
            while (launched < tiles) {
                if (A.waited < nev) { BZ_CHECK(cudaStreamWaitEvent(st, (*A.ev)[A.waited], 0)); A.waited++; }
                size_t have = A.waited >= nev ? (size_t)-1 : A.waited * A.chunk;     // stream bytes present
                size_t have_win = have > A.win_off ? have - A.win_off : 0;
                u32 upto = have_win >= W ? tiles : (have_win > 64 ? (u32)((have_win - 64) / SC_TILE) : 0u);
                if (upto > launched) {
                    ctx->prof_begin(K_RLE_SCAN, (u64)(upto - launched) * SC_TILE * 13);
                    k_rle_scan<<<upto - launched, BZ_THREADS, 0, st>>>(sa); LAUNCH_OK();
                    launched = upto;
                }
            }
        }
    }
    ChainArgs a;
    a.x = d_x; a.RS = RS; a.OUT = OUT; a.LASTQ = LASTQ; a.W = W; a.B = Bsz; a.is_eof = is_eof ? 1u : 0u;
    a.max_blocks = max_blocks; a.max_out = max_n; a.off_from = off_from; a.stop_at = stop_at; a.s0 = s0;
    a.mode = (u32)ctx->mode;
    a.rec = rec; a.nrec = d_small; a.consumed = d_small + 1;
    if (plan_only && skip_chain) { *nblocks = 0; *consumed = 0; return BZ2B200_OK; }   // scan-only call
    if (!skip_chain) {
        // segment after segment of 1 + CH_SEG blocks: candidate windows, speculative links, walk -- no host round trip in between
        static const bool use_tab = [] { const char *e = getenv("BZ2B200_CHAIN_TABLES"); return !e || atoi(e) != 0; }();
        BZ_CHECK(ctx->d_F.ensure(sizeof(ChainState) + 2 * (size_t)(CH_SEG + 1) * 4 + (size_t)TAB_ENTRIES * sizeof(BlockRec) + 256));
        TabArgs t;
        t.a = a;
        t.state = ctx->d_F.as<ChainState>();
        t.tlo = (u32 *)(t.state + 1);
        t.tcnt = t.tlo + (CH_SEG + 1);
        t.tab = use_tab ? (BlockRec *)(((uintptr_t)(t.tcnt + (CH_SEG + 1)) + 15) & ~(uintptr_t)15) : nullptr;
        ChainState st0; st0.nb = 0; st0.s = s0; st0.done = 0; st0.hits = 0;
        BZ_CHECK(cudaMemcpyAsync(t.state, &st0, sizeof st0, cudaMemcpyHostToDevice, st));
        // upper bound of the blocks this call can plan: B output bytes need at least 4/5 B input bytes (runs of exactly four
        // grow to five bytes)
        u64 span_in = (u64)W - (u64)(s0 < W ? s0 : W);
        u32 kmax = (u32)std::min<u64>(max_blocks, span_in / ((u64)Bsz * 4 / 5 - 8) + 2);
        u32 nseg = (kmax + CH_SEG) / (CH_SEG + 1);
        for (u32 g = 0; g < nseg; g++) {
            if (use_tab) {
                ctx->prof_begin(K_RLE_CHAIN, 0); k_rle_tab_bounds<<<(CH_SEG + 127) / 128, 128, 0, st>>>(t); LAUNCH_OK();
                dim3 gf((tab_cap(CH_SEG) + 127) / 128, CH_SEG);
                ctx->prof_begin(K_RLE_CHAIN, 0); k_rle_tab_fill<<<gf, 128, 0, st>>>(t); LAUNCH_OK();
            }
            ctx->prof_begin(K_RLE_CHAIN, (u64)max_blocks * 32); k_rle_chain<<<1, 32, 0, st>>>(t); LAUNCH_OK();
        }
    }
    u32 *hs = ctx->h_small.as<u32>();
    BZ_CHECK(cudaMemcpyAsync(hs, d_small, 8, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    u32 nb = hs[0];
    *nblocks = nb; *consumed = hs[1];
    B.nblk = (int)nb; B.max_n = max_n; B.stride = stride; B.tiles = stride / BZ_TILE;
    { int bits = 0; u32 v = max_n - 1; while (v) { bits++; v >>= 1; } B.nbits = bits; }
    if (nb == 0) return BZ2B200_OK;
    BZ_CHECK(ctx->d_T.ensure((size_t)nb * stride + 64));
    BZ_CHECK(ctx->d_len.ensure((size_t)nb * 4));
    BZ_CHECK(ctx->d_crc.ensure((size_t)nb * 4));
    BlockRec *hrec = (BlockRec *)(hs + 16);
    BZ_CHECK(cudaMemcpyAsync(hrec, rec, (size_t)nb * sizeof(BlockRec), cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    u32 max_span = 0;
    B.total_n = 0;
    for (u32 k = 0; k < nb; k++) B.total_n += hrec[k].out_len;
    for (u32 k = 0; k < nb; k++) max_span = hrec[k].e - hrec[k].s > max_span ? hrec[k].e - hrec[k].s : max_span;
    if (h_spans) { h_spans->clear(); for (u32 k = 0; k < nb; k++) { h_spans->push_back(hrec[k].s); h_spans->push_back(hrec[k].e); h_spans->push_back(hrec[k].out_len); h_spans->push_back(hrec[k].last); } }
    if (plan_only) return BZ2B200_OK;
    dim3 ge((max_span + BZ_TILE - 1) / BZ_TILE, nb);
    ctx->prof_begin(K_RLE_EMIT, (u64)max_span * nb * 2); k_rle_emit<<<ge, BZ_THREADS, 0, st>>>(d_x, W, RS, OUT, rec, ctx->d_T.as<u8>(), ctx->d_len.as<u32>(), stride);
    LAUNCH_OK();
    // block CRCs
    u32 max_pieces = (max_span + PIECE - 1) / PIECE;
    u32 parts_stride = (max_pieces + 255) / 256;
    BZ_CHECK(ctx->d_agg2.ensure((size_t)nb * parts_stride * 4 + 64));
    u32 xp = gf_pow_x8(PIECE), xp256 = gf_pow_x8((u64)PIECE * 256);
    dim3 gc(parts_stride, nb);
    ctx->prof_begin(K_CRC_PIECES, (u64)*consumed); k_crc_pieces<<<gc, 256, 0, st>>>(d_x, (const u32 *)rec, sizeof(BlockRec) / 4, 0, 0, ctx->d_agg2.as<u32>(), parts_stride, xp); LAUNCH_OK();
    ctx->prof_begin(K_CRC_FINAL, 0); k_crc_final<<<nb, 32, 0, st>>>((const u32 *)rec, sizeof(BlockRec) / 4, 0, 0, ctx->d_agg2.as<u32>(), parts_stride, xp256, ctx->d_crc.as<u32>()); LAUNCH_OK();
    B.T = ctx->d_T.as<u8>();
    B.len = ctx->d_len.as<u32>();
    return BZ2B200_OK;
}

// CRC of one device span (do_crc seam)
int bz_crc_dev(bz2b200_ctx *ctx, const u8 *d_x, u32 n, u32 *d_crc_out) {
    cudaStream_t st = ctx->stream;
    u32 pieces = (n + PIECE - 1) / PIECE;
    u32 parts = (pieces + 255) / 256;
    if (parts == 0) parts = 1;
    BZ_CHECK(ctx->d_agg2.ensure((size_t)parts * 4 + 64));
    BZ_CHECK(cudaMemsetAsync(ctx->d_agg2.p, 0, (size_t)parts * 4, st));
    u32 xp = gf_pow_x8(PIECE), xp256 = gf_pow_x8((u64)PIECE * 256);
    if (n) { ctx->prof_begin(K_CRC_PIECES, n); k_crc_pieces<<<dim3(parts, 1), 256, 0, st>>>(d_x, nullptr, 0, 0, n, ctx->d_agg2.as<u32>(), parts, xp); LAUNCH_OK(); }
    ctx->prof_begin(K_CRC_FINAL, 0); k_crc_final<<<1, 32, 0, st>>>(nullptr, 0, 0, n, ctx->d_agg2.as<u32>(), parts, xp256, d_crc_out); LAUNCH_OK();
    return BZ2B200_OK;
}

// CRCs of nb spans [se[2k], se[2k+1]) of one device buffer (decoder side)
int bz_crc_spans_dev(bz2b200_ctx *ctx, const u8 *d_x, const u32 *d_se, u32 nb, u32 max_span, u32 *d_crc_out) {
    cudaStream_t st = ctx->stream;
    u32 max_pieces = (max_span + PIECE - 1) / PIECE;
    u32 parts_stride = (max_pieces + 255) / 256;
    if (parts_stride == 0) parts_stride = 1;
    BZ_CHECK(ctx->d_agg2.ensure((size_t)nb * parts_stride * 4 + 64));
    BZ_CHECK(cudaMemsetAsync(ctx->d_agg2.p, 0, (size_t)nb * parts_stride * 4, st));
    u32 xp = gf_pow_x8(PIECE), xp256 = gf_pow_x8((u64)PIECE * 256);
    dim3 gc(parts_stride, nb);
    ctx->prof_begin(K_CRC_PIECES, 0); k_crc_pieces<<<gc, 256, 0, st>>>(d_x, d_se, 2, 0, 0, ctx->d_agg2.as<u32>(), parts_stride, xp); LAUNCH_OK();
    ctx->prof_begin(K_CRC_FINAL, 0); k_crc_final<<<nb, 32, 0, st>>>(d_se, 2, 0, 0, ctx->d_agg2.as<u32>(), parts_stride, xp256, d_crc_out); LAUNCH_OK();
    return BZ2B200_OK;
}
