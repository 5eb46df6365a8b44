// decode.cu -- block-parallel bzip2 decoder (the round-trip side of the path).
//
// Replaces decompress (reference src/compression/decompress.rs:38-404), huf_decode_map (:426-486),
// rle2_mtf_decode_fast (src/tools/rle2_mtf.rs:191-287), decode_sym_map (symbol_map.rs:20-42),
// bwt_decode (src/bwt_algorithms/bwt_sort.rs:91-130) and rle1_decode (src/tools/rle1.rs:267-316).
// The reference decodes one block after another on one thread; blocks are independent once their
// start bits are known, so:
//   k_dec_find_magic  every bit offset is tested for the 48-bit block / footer magic
//   decode4.cuh       entropy decode, parallel inside a block: header -> tables, the bit offset of every 50-symbol
//                     group (decode_bounds.cuh: jump tables over all bit offsets, then 7 look-ups per group), one
//                     thread per group for the symbols, inverse MTF + RUNA/RUNB by chunks whose start lists come
//                     from composing per-chunk permutations
//   inverse BWT       stable counting sort of rows by byte = one pass of the BWT stage's radix kernels
//                     (P[j] = row of the j-th smallest byte), then the n-step pointer chase of
//                     bwt_decode is cut into ~n/32 segments at splitter rows: k_ibwt_chase measures
//                     every segment in parallel, a two-level walk orders them from the origin pointer
//                     (k_ibwt_coarse / _crank / _fill), k_ibwt_write replays each segment at its output offset
//   k_dec_rle1_*      inverse RLE1 (count pass, then write pass at the block's output offset)
//   CRC               block CRCs with the encoder's CRC kernels; combined CRC on the host.
// The standard run semantics are used (a count byte follows every 4 equal bytes, also at a block's end: without it
// libbz2 reports the block corrupt, and so does this decoder); the reference's rle1_decode drops run expansion in a
// block's last 5 bytes (SURVEY D.6) -- libbz2 is the authority.
#include "common.cuh"
#include "radix.cuh"
#include <algorithm>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

int bz_crc_spans_dev(bz2b200_ctx *ctx, const u8 *d_x, const u32 *d_se /* [nb][2] */, u32 nb, u32 max_span,
                     u32 *d_crc_out);

namespace {

constexpr u64 MAGIC_BLOCK = 0x314159265359ull;
constexpr u64 MAGIC_END = 0x177245385090ull;
#ifndef BZ_IBWT_SPLIT
#define BZ_IBWT_SPLIT 32
#endif
constexpr int SPLIT = BZ_IBWT_SPLIT;     // inverse BWT: one splitter row every SPLIT rows

__device__ __forceinline__ u64 load_be64(const u8 *p, size_t n, size_t byte) {
    u64 v = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) v = (v << 8) | (byte + k < n ? p[byte + k] : 0);
    return v;
}

// candidates[*ncand] = bit positions where a block or footer magic starts (bit 63 set = footer)
__global__ void __launch_bounds__(256) k_dec_find_magic(const u8 *in, size_t n, u64 *cand, u32 *ncand, u32 cap) {
    size_t byte = (size_t)blockIdx.x * 256 + threadIdx.x;
    if (byte >= n) return;
    u64 hi = load_be64(in, n, byte);
    u64 lo = load_be64(in, n, byte + 8);
#pragma unroll
    for (int sh = 0; sh < 8; sh++) {
        u64 w = sh ? ((hi << sh) | (lo >> (64 - sh))) : hi;
        u64 m = w >> 16;
        if (m == MAGIC_BLOCK || m == MAGIC_END) {
            u32 k = atomicAdd(ncand, 1u);
            if (k < cap) cand[k] = ((u64)byte * 8 + sh) | (m == MAGIC_END ? (1ull << 63) : 0);
        }
    }
}

// ---- inverse BWT ------------------------------------------------------------------------------
__device__ __forceinline__ bool is_split(u32 row, u32 key) { return (row % SPLIT) == 0 || row == key; }
__device__ __forceinline__ u32 split_index(u32 row, u32 key, u32 nreg) { return (row % SPLIT) == 0 ? row / SPLIT : nreg; }

// thread per splitter: length of its segment and the splitter that ends it
__global__ void __launch_bounds__(256) k_ibwt_chase(const u32 *P, const u32 *len, const u32 *keys, u32 stride,
                                                    u32 *seglen, u32 *segnext, u32 sstride) {
    u32 b = blockIdx.y, n = len[b], key = keys[b];
    if (n == 0) return;                                     // off-chain candidate of the batch: nothing to rank
    u32 nreg = (n + SPLIT - 1) / SPLIT;
    u32 j = blockIdx.x * 256 + threadIdx.x;
    if (j > nreg) return;
    u32 row = j < nreg ? j * SPLIT : key;
    if (j == nreg && (key % SPLIT) == 0) { seglen[(size_t)b * sstride + j] = 0; return; }   // origin is a regular splitter
    const u32 *p = P + (size_t)b * stride;
    u32 steps = 0;
    do { row = p[row]; steps++; } while (!is_split(row, key));
    seglen[(size_t)b * sstride + j] = steps;
    segnext[(size_t)b * sstride + j] = split_index(row, key, nreg);
}

// Ranking the splitters (which one is visited when, at which text offset) is a walk along segnext from the origin
// pointer: serial, one dependent load per splitter.  Two levels keep it short: every CSPLIT-th splitter (and the origin's)
// is a COARSE splitter; a thread per coarse splitter measures its stretch of the list (k_ibwt_coarse), one thread per
// block walks the coarse list (k_ibwt_crank, ~n / (SPLIT * CSPLIT) steps), a thread per coarse visit then numbers the
// splitters of its stretch (k_ibwt_fill).  A block whose permutation has several cycles (a periodic block walks its short
// cycle many times; corrupt data) can visit more coarse splitters than exist: it is flagged and ranked by the plain walk.
constexpr int CSPLIT = 64;
struct CoarseGeom {                      // jk = the origin's splitter: regular (key on a splitter row) or the extra slot nreg
    u32 nreg, ncr, jk; bool origin_regular_coarse;
    __device__ CoarseGeom(u32 n, u32 key) {
        nreg = (n + SPLIT - 1) / SPLIT;
        ncr = (nreg + CSPLIT - 1) / CSPLIT;                       // regular coarse splitters; coarse index ncr = the origin's
        jk = (key % SPLIT) == 0 ? key / SPLIT : nreg;
        origin_regular_coarse = jk != nreg && (jk % CSPLIT) == 0;
    }
    __device__ bool is_coarse(u32 j) const { return ((j % CSPLIT) == 0 && j != nreg) || j == jk; }
    __device__ u32 coarse_index(u32 j) const { return (j == jk && !origin_regular_coarse) ? ncr : j / CSPLIT; }
    __device__ u32 splitter_of(u32 c) const { return c < ncr ? c * CSPLIT : jk; }
    __device__ u32 origin_coarse() const { return origin_regular_coarse ? jk / CSPLIT : ncr; }
};

__global__ void __launch_bounds__(128) k_ibwt_coarse(const u32 *len, const u32 *keys, const u32 *seglen, const u32 *segnext,
                                                     u32 sstride, u32 *clen, u32 *chops, u32 *cnext, u32 cstride) {
    u32 b = blockIdx.y;
    if (len[b] == 0) return;                                // k_ibwt_chase wrote no segnext for it
    const CoarseGeom g(len[b], keys[b]);
    u32 c = blockIdx.x * 128 + threadIdx.x;
    if (c > g.ncr) return;
    if (c == g.ncr && g.origin_regular_coarse) { clen[(size_t)b * cstride + c] = 0; chops[(size_t)b * cstride + c] = 0; cnext[(size_t)b * cstride + c] = 0; return; }
    u32 j = g.splitter_of(c);
    const u32 *sl = seglen + (size_t)b * sstride, *sn = segnext + (size_t)b * sstride;
    u32 rows = 0, hops = 0;
    do { rows += sl[j]; j = sn[j]; hops++; } while (!g.is_coarse(j) && hops <= g.nreg + 1);
    clen[(size_t)b * cstride + c] = rows;
    chops[(size_t)b * cstride + c] = hops;
    cnext[(size_t)b * cstride + c] = g.coarse_index(j);
}

// one thread per block: coarse visits in text order; flag[b] = 1 when the bound is exceeded (several cycles)
__global__ void __launch_bounds__(32) k_ibwt_crank(const u32 *len, const u32 *keys, const u32 *clen, const u32 *chops,
                                                   const u32 *cnext, u32 cstride, u32 *cv_split, u32 *cv_off, u32 *cv_vbase,
                                                   u32 *ncvisit, u32 *nvisit, u32 *flag, u32 vstride) {
    u32 b = blockIdx.x;
    if (threadIdx.x != 0) return;
    u32 n = len[b];
    const CoarseGeom g(n, keys[b]);
    u32 c = g.origin_coarse();
    u32 off = 0, v = 0, u = 0;
    bool over = false;
    while (off < n) {
        if (u >= cstride) { over = true; break; }
        cv_split[(size_t)b * cstride + u] = c;
        cv_off[(size_t)b * cstride + u] = off;
        cv_vbase[(size_t)b * cstride + u] = v;
        off += clen[(size_t)b * cstride + c];
        v += chops[(size_t)b * cstride + c];
        c = cnext[(size_t)b * cstride + c];
        u++;
    }
    if (v > vstride) over = true;
    flag[b] = over ? 1u : 0u;
    ncvisit[b] = over ? 0u : u;
    if (!over) nvisit[b] = v;       // an upper bound: the last stretch may reach n before its last splitter (k_ibwt_write checks off < n)
}

// thread per coarse visit: the splitters of its stretch, in order
__global__ void __launch_bounds__(128) k_ibwt_fill(const u32 *len, const u32 *keys, const u32 *seglen, const u32 *segnext,
                                                   u32 sstride, const u32 *chops, const u32 *cv_split, const u32 *cv_off,
                                                   const u32 *cv_vbase, const u32 *ncvisit, u32 cstride, u32 *visit_split,
                                                   u32 *visit_off, u32 vstride) {
    u32 b = blockIdx.y;
    u32 u = blockIdx.x * 128 + threadIdx.x;
    if (len[b] == 0 || u >= ncvisit[b]) return;
    const CoarseGeom g(len[b], keys[b]);
    u32 c = cv_split[(size_t)b * cstride + u];
    u32 j = g.splitter_of(c);
    u32 off = cv_off[(size_t)b * cstride + u], v = cv_vbase[(size_t)b * cstride + u];
    u32 hops = chops[(size_t)b * cstride + c];
    const u32 *sl = seglen + (size_t)b * sstride, *sn = segnext + (size_t)b * sstride;
    for (u32 i = 0; i < hops && v < vstride; i++) {
        visit_split[(size_t)b * vstride + v] = j;
        visit_off[(size_t)b * vstride + v] = off;
        off += sl[j]; j = sn[j]; v++;
    }
}

// one thread per FLAGGED block: visit splitters in text order starting at the origin pointer until n rows are covered
__global__ void __launch_bounds__(32) k_ibwt_rank(const u32 *len, const u32 *keys, const u32 *seglen, const u32 *segnext,
                                                  u32 sstride, u32 *visit_split, u32 *visit_off, u32 vstride, u32 *nvisit,
                                                  const u32 *flag) {
    u32 b = blockIdx.x;
    if (threadIdx.x != 0 || !flag[b]) return;
    u32 n = len[b], key = keys[b];
    u32 nreg = (n + SPLIT - 1) / SPLIT;
    u32 j = (key % SPLIT) == 0 ? key / SPLIT : nreg;
    u32 off = 0, v = 0;
    while (off < n && v < vstride) {
        visit_split[(size_t)b * vstride + v] = j;
        visit_off[(size_t)b * vstride + v] = off;
        off += seglen[(size_t)b * sstride + j];
        j = segnext[(size_t)b * sstride + j];
        v++;
    }
    nvisit[b] = v;
}

// thread per visit: replay the segment; text position i (0-based) receives L[P^(i+1)(key)]  (bwt_sort.rs:118-128), i < n.
// That is n steps from the origin, as libbz2 walks them: position n - 1 holds L[P^n(key)], which is L[key] only when the
// origin's cycle length divides n -- always so for a true BWT, not for every L a stream can carry.
__global__ void __launch_bounds__(256) k_ibwt_write(const u32 *P, const u8 *L, const u32 *len, const u32 *keys, u32 stride,
                                                    const u32 *visit_split, const u32 *visit_off, u32 vstride,
                                                    const u32 *nvisit, u8 *out) {
    u32 b = blockIdx.y, n = len[b], key = keys[b];
    u32 v = blockIdx.x * 256 + threadIdx.x;
    if (v >= nvisit[b]) return;
    u32 nreg = (n + SPLIT - 1) / SPLIT;
    u32 j = visit_split[(size_t)b * vstride + v];
    u32 off = visit_off[(size_t)b * vstride + v];
    if (off > n) return;                                    // past the walk (k_ibwt_crank's visit count is an upper bound)
    u32 row = j < nreg ? j * SPLIT : key;
    const u32 *p = P + (size_t)b * stride;
    const u8 *l = L + (size_t)b * stride;
    u8 *o = out + (size_t)b * stride;
    // row = P^off(key): position off-1 holds L[row] for 1 <= off <= n.  No visit starts at off = n, so the visit that
    // reaches it writes it even on a splitter row (a visit listed at n writes the same byte).
    for (;;) {
        if (off) o[off - 1] = l[row];
        if (off == n) break;
        row = p[row];
        off++;
        if (off < n && is_split(row, key)) break;
    }
}

#include "decode4.cuh"        // entropy decode: header, symbols, chunked inverse MTF
#include "decode_bounds.cuh"  // ... and the group boundaries (jump tables + walk)
#include "decode_rle1.cuh"   // k_rle1_inv

}  // namespace

#define LAUNCH_OK()                                                \
    do {                                                             \
        ctx->prof_end();                                             \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) { ctx->fail("kernel launch", e_, __FILE__, __LINE__); return BZ2B200_E_CUDA; } \
    } while (0)

// Inverse BWT of a batch already on the device: L = last column, keys = origin pointers.
static int ibwt_batch(bz2b200_ctx *ctx, const Batch &B, const u32 *d_keys, u8 *d_out) {
    cudaStream_t st = ctx->stream;
    size_t ne = (size_t)B.nblk * B.stride;
    const u32 rtiles = B.stride / radix::R_TILE;
    BZ_CHECK(ctx->d_SA.ensure(ne * 4));
    BZ_CHECK(ctx->d_thist.ensure((size_t)B.nblk * rtiles * 256 * 4));
    u32 sstride = B.stride / SPLIT + 2;
    u32 vstride = B.stride + sstride;   // a periodic block walks its (short) cycle many times: up to n visits
    BZ_CHECK(ctx->d_dec2.ensure((size_t)B.nblk * sstride * 8 + (size_t)B.nblk * vstride * 8 + (size_t)B.nblk * 4 + 64));
    u32 *seglen = ctx->d_dec2.as<u32>();
    u32 *segnext = seglen + (size_t)B.nblk * sstride;
    u32 *vsplit = segnext + (size_t)B.nblk * sstride;
    u32 *voff = vsplit + (size_t)B.nblk * vstride;
    u32 *nvisit = voff + (size_t)B.nblk * vstride;
    u32 *P = ctx->d_SA.as<u32>();
    // P = rows sorted stably by their byte: one radix pass with digit = L[row]
    radix::RadixArgs a{};
    a.T = B.T; a.len = B.len; a.sa_out = P; a.thist = ctx->d_thist.as<u32>(); a.stride = B.stride; a.rtiles = rtiles;
    dim3 gr((B.max_n + radix::R_TILE - 1) / radix::R_TILE, B.nblk);
    ctx->prof_begin(K_RADIX_HIST0, B.total_n * 5); radix::k_radix_hist<<<gr, BZ_THREADS, 0, st>>>(a); LAUNCH_OK();
    ctx->prof_begin(K_RADIX_SCAN, 0); radix::k_radix_scan<<<B.nblk, 256, 0, st>>>(a.thist, B.len, rtiles); LAUNCH_OK();
    ctx->prof_begin(K_RADIX_SCATTER0, B.total_n * 9); radix::k_radix_scatter<<<gr, BZ_THREADS, 0, st>>>(a); LAUNCH_OK();
    dim3 gs((B.max_n / SPLIT + 2 + 255) / 256, B.nblk);
    ctx->prof_begin(K_IBWT_CHASE, B.total_n * 4); k_ibwt_chase<<<gs, 256, 0, st>>>(P, B.len, d_keys, B.stride, seglen, segnext, sstride); LAUNCH_OK();
    {
        u32 cstride = sstride / CSPLIT + 8;
        BZ_CHECK(ctx->d_KEYA.ensure((size_t)B.nblk * cstride * 4 * 6 + (size_t)B.nblk * 8 + 64));
        u32 *clen = ctx->d_KEYA.as<u32>();
        u32 *chops = clen + (size_t)B.nblk * cstride, *cnext = chops + (size_t)B.nblk * cstride;
        u32 *cv_split = cnext + (size_t)B.nblk * cstride, *cv_off = cv_split + (size_t)B.nblk * cstride;
        u32 *cv_vbase = cv_off + (size_t)B.nblk * cstride;
        u32 *ncvisit = cv_vbase + (size_t)B.nblk * cstride, *flag = ncvisit + B.nblk;
        dim3 gc((cstride + 127) / 128, B.nblk);
        ctx->prof_begin(K_IBWT_RANK, 0);
        k_ibwt_coarse<<<gc, 128, 0, st>>>(B.len, d_keys, seglen, segnext, sstride, clen, chops, cnext, cstride); LAUNCH_OK();
        ctx->prof_begin(K_IBWT_RANK, 0);
        k_ibwt_crank<<<B.nblk, 32, 0, st>>>(B.len, d_keys, clen, chops, cnext, cstride, cv_split, cv_off, cv_vbase, ncvisit, nvisit, flag, vstride); LAUNCH_OK();
        ctx->prof_begin(K_IBWT_RANK, 0);
        k_ibwt_fill<<<gc, 128, 0, st>>>(B.len, d_keys, seglen, segnext, sstride, chops, cv_split, cv_off, cv_vbase, ncvisit, cstride, vsplit, voff, vstride); LAUNCH_OK();
        ctx->prof_begin(K_IBWT_RANK, 0);
        k_ibwt_rank<<<B.nblk, 32, 0, st>>>(B.len, d_keys, seglen, segnext, sstride, vsplit, voff, vstride, nvisit, flag); LAUNCH_OK();
    }
    dim3 gv((vstride + 255) / 256, B.nblk);
    ctx->prof_begin(K_IBWT_WRITE, B.total_n * 6); k_ibwt_write<<<gv, 256, 0, st>>>(P, B.T, B.len, d_keys, B.stride, vsplit, voff, vstride, nvisit, d_out); LAUNCH_OK();
    return BZ2B200_OK;
}

extern "C" int bz2b200_bwt_decode(bz2b200_ctx *ctx, uint32_t key, const uint8_t *bwt, uint32_t n, uint8_t *out) {
    BZ_API_TRY
    if (!ctx || !bwt || !out || n == 0 || key >= n) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    Batch B;
    const u8 *ins[1] = {bwt};
    int rc = bz_stage_blocks(ctx, 1, ins, &n, B);
    if (rc) return rc;
    BZ_CHECK(ctx->d_key.ensure(4));
    BZ_CHECK(ctx->d_bwt.ensure(B.stride));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_key.p, &key, 4, cudaMemcpyHostToDevice, ctx->stream));
    rc = ibwt_batch(ctx, B, ctx->d_key.as<u32>(), ctx->d_bwt.as<u8>());
    if (rc) return rc;
    BZ_CHECK(cudaMemcpyAsync(out, ctx->d_bwt.p, n, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    return BZ2B200_OK;
    BZ_API_CATCH
}

// ---- legacy randomised blocks (bzip2 <= 0.9.0): the un-BWT'd bytes are XORed with 1 at pseudo-random distances ----
// The 512 distances are a constant of the .bz2 format (BZ2_rNums of libbz2; the reference keeps the same numbers in
// src/unused/randomizing_table.rs:1-32 without using them, its decoder ignores the flag).  Byte i of the block is
// flipped when the countdown started from the current table entry stands at 1, i.e. at cum(t) + rNums[t] - 2.
__constant__ u16 c_rnums[512] = {
    619, 720, 127, 481, 931, 816, 813, 233, 566, 247, 985, 724, 205, 454, 863, 491, 741, 242, 949, 214, 733, 859, 335, 708,
    621, 574, 73, 654, 730, 472, 419, 436, 278, 496, 867, 210, 399, 680, 480, 51, 878, 465, 811, 169, 869, 675, 611, 697,
    867, 561, 862, 687, 507, 283, 482, 129, 807, 591, 733, 623, 150, 238, 59, 379, 684, 877, 625, 169, 643, 105, 170, 607,
    520, 932, 727, 476, 693, 425, 174, 647, 73, 122, 335, 530, 442, 853, 695, 249, 445, 515, 909, 545, 703, 919, 874, 474,
    882, 500, 594, 612, 641, 801, 220, 162, 819, 984, 589, 513, 495, 799, 161, 604, 958, 533, 221, 400, 386, 867, 600, 782,
    382, 596, 414, 171, 516, 375, 682, 485, 911, 276, 98, 553, 163, 354, 666, 933, 424, 341, 533, 870, 227, 730, 475, 186,
    263, 647, 537, 686, 600, 224, 469, 68, 770, 919, 190, 373, 294, 822, 808, 206, 184, 943, 795, 384, 383, 461, 404, 758,
    839, 887, 715, 67, 618, 276, 204, 918, 873, 777, 604, 560, 951, 160, 578, 722, 79, 804, 96, 409, 713, 940, 652, 934,
    970, 447, 318, 353, 859, 672, 112, 785, 645, 863, 803, 350, 139, 93, 354, 99, 820, 908, 609, 772, 154, 274, 580, 184,
    79, 626, 630, 742, 653, 282, 762, 623, 680, 81, 927, 626, 789, 125, 411, 521, 938, 300, 821, 78, 343, 175, 128, 250,
    170, 774, 972, 275, 999, 639, 495, 78, 352, 126, 857, 956, 358, 619, 580, 124, 737, 594, 701, 612, 669, 112, 134, 694,
    363, 992, 809, 743, 168, 974, 944, 375, 748, 52, 600, 747, 642, 182, 862, 81, 344, 805, 988, 739, 511, 655, 814, 334,
    249, 515, 897, 955, 664, 981, 649, 113, 974, 459, 893, 228, 433, 837, 553, 268, 926, 240, 102, 654, 459, 51, 686, 754,
    806, 760, 493, 403, 415, 394, 687, 700, 946, 670, 656, 610, 738, 392, 760, 799, 887, 653, 978, 321, 576, 617, 626, 502,
    894, 679, 243, 440, 680, 879, 194, 572, 640, 724, 926, 56, 204, 700, 707, 151, 457, 449, 797, 195, 791, 558, 945, 679,
    297, 59, 87, 824, 713, 663, 412, 693, 342, 606, 134, 108, 571, 364, 631, 212, 174, 643, 304, 329, 343, 97, 430, 751,
    497, 314, 983, 374, 822, 928, 140, 206, 73, 263, 980, 736, 876, 478, 430, 305, 170, 514, 364, 692, 829, 82, 855, 953,
    676, 246, 369, 970, 294, 750, 807, 827, 150, 790, 288, 923, 804, 378, 215, 828, 592, 281, 565, 555, 710, 82, 896, 831,
    547, 261, 524, 462, 293, 465, 502, 56, 661, 821, 976, 991, 658, 869, 905, 758, 745, 193, 768, 550, 608, 933, 378, 286,
    215, 979, 792, 961, 61, 688, 793, 644, 986, 403, 106, 366, 905, 644, 372, 567, 466, 434, 645, 210, 389, 550, 919, 135,
    780, 773, 635, 389, 707, 100, 626, 958, 165, 504, 920, 176, 193, 713, 857, 265, 203, 50, 668, 108, 645, 990, 626, 197,
    510, 357, 358, 850, 858, 364, 936, 638};

// one CTA per block, thread per table entry (cycled): flips of a randomised block
__global__ void __launch_bounds__(512) k_derandomize(u8 *blk, const u32 *len, const u32 *randflag, u32 stride) {
    u32 b = blockIdx.x;
    if (!randflag[b]) return;
    u32 n = len[b];
    __shared__ u32 cum[513];
    if (threadIdx.x == 0) { u32 a = 0; for (int t = 0; t < 512; t++) { cum[t] = a; a += c_rnums[t]; } cum[512] = a; }
    __syncthreads();
    u8 *x = blk + (size_t)b * stride;
    const u32 period = cum[512];
    for (u32 base = 0; base < n; base += period) {
        u32 pos = base + cum[threadIdx.x] + c_rnums[threadIdx.x] - 2u;
        if (pos < n) x[pos] ^= 1;
    }
}

static_assert(sizeof(DecTail) == sizeof(DecTables) - offsetof(DecTables, T), "DecTail mirrors the tail of DecTables");

DecGeom::DecGeom(u32 mb) {
    max_block = mb;
    stride = ((max_block + 64 + BZ_TILE - 1) / BZ_TILE) * BZ_TILE;
    sel_stride = max_block / 50 + 8;
    max_sym = max_block + 2;                                    // every symbol but EOB yields at least one byte
    sym_stride = ((max_sym + 64 + DCH - 1) / DCH) * DCH;
    ch_stride = sym_stride / DCH + 2;
}

namespace {
// the batch's device workspaces (grow-only context buffers) and where each array lives in them
struct DecWork {
    DecTables *tabs; u32 *gbit; u16 *sym; u8 *vid, *lists; u32 *ccount, *coff;
    u64 *starts, *olen, *ooff; u32 *len, *keys, *rand, *se; u64 *rend;
};
int dec_work(bz2b200_ctx *ctx, const DecGeom &g, DecWork &W) {
    const u32 NB = DEC_BATCH;
    BZ_CHECK(ctx->d_T.ensure((size_t)NB * g.stride + 64));
    BZ_CHECK(ctx->d_bwt.ensure((size_t)NB * g.stride + 64));
    BZ_CHECK(ctx->d_sel.ensure((size_t)NB * g.sel_stride));
    BZ_CHECK(ctx->d_gbits.ensure((size_t)NB * g.sel_stride * 4));
    BZ_CHECK(ctx->d_sym.ensure((size_t)NB * g.sym_stride * 2));
    BZ_CHECK(ctx->d_mtfstate.ensure((size_t)NB * g.ch_stride * 256));
    BZ_CHECK(ctx->d_chunkrec.ensure((size_t)NB * g.ch_stride * 8));
    BZ_CHECK(ctx->d_hdr.ensure((size_t)NB * sizeof(DecTables)));
    BZ_CHECK(ctx->d_dec3.ensure((size_t)NB * (8 + 4 + 4 + 4 + 8 + 8 + 8 + 8) + 256));
    BZ_CHECK(ctx->d_crc.ensure((size_t)NB * 4));
    BZ_CHECK(ctx->d_KEYB.ensure((size_t)NB * g.sym_stride));
    W.tabs = ctx->d_hdr.as<DecTables>();
    W.gbit = ctx->d_gbits.as<u32>();
    W.sym = ctx->d_sym.as<u16>();
    W.vid = ctx->d_KEYB.as<u8>();                               // start-list position selected by every MTF symbol (k_dec_chunks -> k_dec_expand)
    W.lists = ctx->d_mtfstate.as<u8>();
    W.ccount = ctx->d_chunkrec.as<u32>();
    W.coff = W.ccount + (size_t)NB * g.ch_stride;
    W.starts = ctx->d_dec3.as<u64>();
    W.olen = W.starts + NB;
    W.ooff = W.olen + NB;
    W.len = (u32 *)(W.ooff + NB);
    W.keys = W.len + NB;
    W.rand = W.keys + NB;
    W.se = W.rand + NB;
    W.rend = (u64 *)(W.se + 2 * (size_t)NB);                    // after the spans; 8-byte aligned (all counts are multiples of NB * 4, NB even)
    if (!ctx->dec_attr_done) { BZ_CHECK(cudaFuncSetAttribute(k_dec_bounds, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)JRING_BYTES)); ctx->dec_attr_done = true; }
    return BZ2B200_OK;
}
}  // namespace

int bz_dec_entropy(bz2b200_ctx *ctx, const DecGeom &g, const u8 *d_bits, size_t n, const std::vector<u64> &starts,
                   const std::vector<u64> &rends, std::vector<DecTail> &db) {
    cudaStream_t st = ctx->stream;
    DecWork W;
    int rc = dec_work(ctx, g, W);
    if (rc) return rc;
    const u32 nb = (u32)starts.size();
    const u32 sel_stride = g.sel_stride, sym_stride = g.sym_stride, ch_stride = g.ch_stride;
    u64 max_range = 0;
    for (u32 k = 0; k < nb; k++) max_range = std::max(max_range, rends[k] - starts[k]);
    BZ_CHECK(cudaMemcpyAsync(W.starts, starts.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemcpyAsync(W.rend, rends.data(), (size_t)nb * 8, cudaMemcpyHostToDevice, st));
    ctx->prof_begin(K_DEC_HEADER, 0); k_dec_header<<<nb, 32, 0, st>>>(d_bits, n, W.starts, ctx->d_sel.as<u8>(), sel_stride, W.tabs); LAUNCH_OK();
    {   // group boundaries: jump tables (2 bytes per bit offset and table), and the walkers of the same blocks following
        // them window by window from a second, high-priority stream (their few CTAs are placed as soon as the producer's
        // first ones retire); in slices of the batch when the tables of all its blocks would not fit the budget
        // (incompressible data: 88 MB per block).  The producer is launched first: a tool that serialises kernels in
        // launch order (ncu, compute-sanitizer) then still terminates.
        // The walkers spin until their producer's CTAs have run.  One context's walkers (at most DEC_BATCH CTAs, two per
        // SM by shared memory) leave most SMs to its producer; the walkers of several contexts on one device could take
        // every SM while their producers wait for one.  So when this process holds more than one context on the device,
        // the phase runs under a per-device lock until its walkers are done: then the walkers on the device are those of
        // one batch, and every other kernel of the process on it finishes without waiting for anything.  (The count is
        // read without the lock: a context created while the device's only other context runs this phase unlocked
        // overlaps it once -- two batches, at most 128 of the 148 SMs, still leave SMs to both producers.)
        std::unique_lock<std::mutex> dev_lk;
        if (bz_contexts_on_device(ctx->device) > 1) dev_lk = std::unique_lock<std::mutex>(bz_device_lock(ctx->device));
        const u32 nwin_max = jump_windows(max_range);
        const size_t jstride = (size_t)nwin_max * 6 * 2 * JW;
        const size_t budget = (size_t)6 << 30;
        const u32 slice = (u32)std::max<size_t>(1, std::min<size_t>(nb, budget / jstride));
        BZ_CHECK(ctx->d_VALA.ensure((size_t)slice * jstride));
        BZ_CHECK(ctx->d_VALB.ensure((size_t)slice * nwin_max * 4));
        u32 *d_flags = ctx->d_VALB.as<u32>();
        if (!ctx->s_hi) {
            int lo = 0, hi_p = 0;
            BZ_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi_p));
            BZ_CHECK(cudaStreamCreateWithPriority(&ctx->s_hi, cudaStreamNonBlocking, hi_p));
            for (int q = 0; q < 2; q++) BZ_CHECK(cudaEventCreateWithFlags(&ctx->ev_dec[q], cudaEventDisableTiming));
        }
        for (u32 b0 = 0; b0 < nb; b0 += slice) {
            const u32 cnt = std::min(slice, nb - b0);
            BZ_CHECK(cudaMemsetAsync(d_flags, 0, (size_t)cnt * nwin_max * 4, st));
            BZ_CHECK(cudaEventRecord(ctx->ev_dec[0], st));                   // headers parsed, flags clear, the previous slice done
            ctx->prof_begin(K_DEC_JUMPS, (u64)cnt * jstride);
            k_dec_jumps<<<dim3(cnt, nwin_max), 256, 0, st>>>(d_bits, n, W.tabs, W.rend, ctx->d_VALA.as<u8>(), jstride, d_flags, nwin_max, b0); LAUNCH_OK();
            BZ_CHECK(cudaStreamWaitEvent(ctx->s_hi, ctx->ev_dec[0], 0));
            k_dec_bounds<<<cnt, 32, JRING_BYTES, ctx->s_hi>>>(d_bits, n, ctx->d_sel.as<u8>(), sel_stride, W.tabs, W.rend, ctx->d_VALA.as<u8>(), jstride, d_flags, nwin_max, W.gbit, g.max_sym, b0);
            ctx->launches++;
            if (cudaGetLastError() != cudaSuccess) { ctx->err = "decode: k_dec_bounds launch"; cudaStreamSynchronize(st); return BZ2B200_E_CUDA; }
            BZ_CHECK(cudaEventRecord(ctx->ev_dec[1], ctx->s_hi));
            ctx->prof_begin(K_DEC_BOUNDS, n);                                // as timed on the main stream: what the walk adds after the producer
            BZ_CHECK(cudaStreamWaitEvent(st, ctx->ev_dec[1], 0));
            ctx->prof_end(); ctx->launches--;
        }
        if (dev_lk.owns_lock()) BZ_CHECK(cudaStreamSynchronize(ctx->s_hi));
    }
    dim3 gs((sel_stride + 127) / 128, nb);
    ctx->prof_begin(K_DEC_SYMS, n); k_dec_syms<<<gs, 128, 0, st>>>(d_bits, n, ctx->d_sel.as<u8>(), sel_stride, W.tabs, W.gbit, W.sym, sym_stride); LAUNCH_OK();
    dim3 gch((ch_stride + 7) / 8, nb);
    ctx->prof_begin(K_DEC_CHUNKS, 0); k_dec_chunks<<<gch, 256, 0, st>>>(W.tabs, W.sym, sym_stride, W.lists, W.ccount, ch_stride, W.vid, g.max_block); LAUNCH_OK();
    ctx->prof_begin(K_DEC_CHUNK_SCAN, 0); k_dec_chunk_scan<<<nb, 256, 0, st>>>(W.tabs, W.lists, W.ccount, W.coff, ch_stride, g.max_block); LAUNCH_OK();
    ctx->prof_begin(K_DEC_EXPAND, 0); k_dec_expand<<<gch, 256, 0, st>>>(W.tabs, W.sym, sym_stride, W.lists, W.coff, ch_stride, W.vid, ctx->d_T.as<u8>(), g.stride); LAUNCH_OK();
    db.resize(nb);
    BZ_CHECK(cudaMemcpy2DAsync(db.data(), sizeof(DecTail), (const u8 *)W.tabs + offsetof(DecTables, T), sizeof(DecTables),
                               sizeof(DecTail), nb, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    return BZ2B200_OK;
}

int bz_dec_unbwt(bz2b200_ctx *ctx, const DecGeom &g, u32 nblk, const u32 *hlen, const u32 *hkey, const u32 *hrand, u64 *olen) {
    cudaStream_t st = ctx->stream;
    DecWork W;
    int rc = dec_work(ctx, g, W);
    if (rc) return rc;
    u32 max_n = 0; u64 total_n = 0;
    bool any_rand = false;
    for (u32 k = 0; k < nblk; k++) { max_n = std::max(max_n, hlen[k]); total_n += hlen[k]; any_rand |= hlen[k] && hrand[k]; }
    BZ_CHECK(cudaMemcpyAsync(W.len, hlen, (size_t)nblk * 4, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemcpyAsync(W.keys, hkey, (size_t)nblk * 4, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemcpyAsync(W.rand, hrand, (size_t)nblk * 4, cudaMemcpyHostToDevice, st));
    // ---- inverse BWT (+ de-randomisation of legacy blocks) ----
    Batch B;
    B.nblk = (int)nblk; B.stride = g.stride; B.tiles = g.stride / BZ_TILE; B.max_n = max_n; B.nbits = 20; B.T = ctx->d_T.as<u8>();
    B.len = W.len; B.total_n = total_n;
    rc = ibwt_batch(ctx, B, W.keys, ctx->d_bwt.as<u8>());
    if (rc) return rc;
    if (any_rand) { ctx->prof_begin(K_DEC_MISC, total_n); k_derandomize<<<nblk, 512, 0, st>>>(ctx->d_bwt.as<u8>(), W.len, W.rand, g.stride); LAUNCH_OK(); }
    // ---- inverse RLE1, count pass ----
    ctx->prof_begin(K_DEC_RLE1_COUNT, total_n); k_rle1_inv<0><<<nblk, 256, 0, st>>>(ctx->d_bwt.as<u8>(), W.len, g.stride, W.olen, nullptr, nullptr); LAUNCH_OK();
    BZ_CHECK(cudaMemcpyAsync(olen, W.olen, (size_t)nblk * 8, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    return BZ2B200_OK;
}

int bz_dec_write(bz2b200_ctx *ctx, const DecGeom &g, u32 nblk, const u64 *olen, const u64 *ooff, u8 *d_out, u32 *crcs) {
    cudaStream_t st = ctx->stream;
    DecWork W;
    int rc = dec_work(ctx, g, W);
    if (rc) return rc;
    u64 btotal = 0;
    for (u32 k = 0; k < nblk; k++) btotal += olen[k];
    BZ_CHECK(cudaMemcpyAsync(W.ooff, ooff, (size_t)nblk * 8, cudaMemcpyHostToDevice, st));
    ctx->prof_begin(K_DEC_RLE1_WRITE, btotal); k_rle1_inv<1><<<nblk, 256, 0, st>>>(ctx->d_bwt.as<u8>(), W.len, g.stride, W.olen, W.ooff, d_out); LAUNCH_OK();
    // block CRCs in sub-ranges of at most 2 GiB of output (a block decodes to at most ~46 MB; spans are 32-bit)
    std::vector<u32> se(2 * (size_t)nblk);
    for (u32 k0 = 0; k0 < nblk;) {
        u32 k1 = k0; u64 sub = 0, max_span = 0;
        while (k1 < nblk && (k1 == k0 || sub + olen[k1] <= (1ull << 31))) {
            se[2 * k1] = (u32)sub; se[2 * k1 + 1] = (u32)(sub + olen[k1]);
            sub += olen[k1]; max_span = std::max(max_span, olen[k1]); k1++;
        }
        BZ_CHECK(cudaMemcpyAsync(W.se + 2 * k0, se.data() + 2 * k0, (size_t)(k1 - k0) * 8, cudaMemcpyHostToDevice, st));
        rc = bz_crc_spans_dev(ctx, d_out + ooff[k0], W.se + 2 * k0, k1 - k0, (u32)max_span, ctx->d_crc.as<u32>() + k0);
        if (rc) return rc;
        BZ_CHECK(cudaStreamSynchronize(st));                    // se is reused by the next sub-range
        k0 = k1;
    }
    BZ_CHECK(cudaMemcpyAsync(crcs, ctx->d_crc.p, (size_t)nblk * 4, cudaMemcpyDeviceToHost, st));
    return BZ2B200_OK;
}

// every bit offset of d_win[0, len) that looks like a block or footer magic, sorted; BZ2B200_E_FORMAT past `cap`
int bz_dec_candidates(bz2b200_ctx *ctx, const u8 *d_win, size_t len, u32 cap, std::vector<u64> &cand) {
    cudaStream_t st = ctx->stream;
    BZ_CHECK(ctx->d_dec1.ensure((size_t)cap * 8 + 64));
    u64 *d_cand = ctx->d_dec1.as<u64>();
    u32 *d_ncand = (u32 *)(d_cand + cap);
    BZ_CHECK(cudaMemsetAsync(d_ncand, 0, 4, st));
    ctx->prof_begin(K_DEC_MAGIC, len); k_dec_find_magic<<<(u32)((len + 255) / 256), 256, 0, st>>>(d_win, len, d_cand, d_ncand, cap); LAUNCH_OK();
    u32 ncand = 0;
    BZ_CHECK(cudaMemcpyAsync(&ncand, d_ncand, 4, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    cand.clear();
    if (ncand > cap) { ctx->err = "decode: more magic candidates than the candidate buffer holds"; return BZ2B200_E_FORMAT; }
    cand.resize(ncand);
    if (ncand) BZ_CHECK(cudaMemcpy(cand.data(), d_cand, (size_t)ncand * 8, cudaMemcpyDeviceToHost));
    std::sort(cand.begin(), cand.end(), [](u64 a, u64 b) { return (a & ~DEC_FOOT) < (b & ~DEC_FOOT); });
    return BZ2B200_OK;
}

// test knob: a spurious block candidate at the first bit of the window and between any two candidates, as chance magics
// inside compressed data would be
void bz_add_chance_candidates(std::vector<u64> &cand) {
    std::vector<u64> add;
    if (cand.empty() || (cand[0] & ~DEC_FOOT) != 0) add.push_back(0);
    for (size_t i = 0; i + 1 < cand.size(); i++) {
        u64 a = cand[i] & ~DEC_FOOT, b = cand[i + 1] & ~DEC_FOOT;
        if (b - a >= 2) add.push_back((a + b) / 2);
    }
    cand.insert(cand.end(), add.begin(), add.end());
    std::sort(cand.begin(), cand.end(), [](u64 x, u64 y) { return (x & ~DEC_FOOT) < (y & ~DEC_FOOT); });
}

// A magic can also occur by chance inside entropy-coded data, and a file may hold several streams one after the other
// (decompress.rs handles neither; libbz2 walks the blocks serially and accepts both).  So the candidates are only where
// blocks MAY start: the chain is walked from every decoded block's end, candidates off the chain are dropped, and a
// footer that is not the end of the input must be followed by the next stream's "BZh<level>".
// A window that does not know where its chain enters entropy-decodes the first batch of its candidates first: the true
// start is the first element at or after the window's first bit, so it is among them.
int bz_decode_core(bz2b200_ctx *ctx, const DecWindow &w, DecSink &sink, std::vector<DecEvent> &ev) {
    const std::vector<u64> &cand = *w.cand;
    const size_t ncand = cand.size();
    const size_t n = w.len;                                     // bytes on the device
    const u64 lo8 = (u64)w.lo * 8;
    const u64 hi = w.hi_bit == ~0ull ? ~0ull : w.hi_bit - lo8;  // window-relative, like every bit below
    const u32 max_block = w.max_block;
    const DecGeom g(max_block);
    const u32 NB = DEC_BATCH;
    const u8 *d_bits = w.d_win;

    auto read32 = [&](u64 bit) {                                // 32 bits at an absolute bit offset of the host input
        size_t byte = (size_t)(bit >> 3); int sh = (int)(bit & 7);
        u64 v = 0;
        for (int k = 0; k < 5; k++) v = (v << 8) | (byte + k < w.n ? w.in[byte + k - w.in_lo] : 0);
        return (u32)((v >> (8 - sh)) & 0xffffffffull);
    };
    size_t ci = 0;                                              // next candidate to look at
    bool known = w.expect >= 0;                                 // the chain start is known
    u64 expect = known ? (u64)w.expect - lo8 : 0;               // bit offset where the next block / footer must start
    bool comb_known = known;                                    // the window has seen the start of the current stream
    u32 combined = known ? w.combined : 0;                      // running combined CRC of the current stream
    bool have_batch = false;                                    // `starts` were decoded before the chain start was known
    std::vector<u64> starts, rends;
    const u64 range_limit = [] { const char *e = getenv("BZ2B200_DEC_RANGE_LIMIT"); return e ? (u64)strtoull(e, nullptr, 10) : 0ull; }();
    std::vector<DecTail> db;
    std::vector<u32> hlen(NB), hkey(NB), hrand(NB), crcs(NB);
    std::vector<u64> olen(NB), ooff(NB);
    for (;;) {
        if (known) {
            if (expect >= hi) { sink.chain_end((long long)(expect + lo8)); return BZ2B200_OK; }
            while (ci < ncand && (cand[ci] & ~DEC_FOOT) < expect) ci++;
            if (ci == ncand || (cand[ci] & ~DEC_FOOT) != expect) { ctx->err = "decode: no block or footer magic at bit " + std::to_string(expect + lo8); return BZ2B200_E_FORMAT; }
            if (cand[ci] & DEC_FOOT) {                              // end of a stream: combined CRC, then end of input or another stream
                const u32 stored = read32(expect + lo8 + 48);
                ev.push_back(DecEvent{expect + lo8, stored, 0, DEC_FOOTER});
                if (comb_known && stored != combined) return BZ2B200_E_CRC;                    // enforced, unlike decompress.rs:394-402
                size_t hb = (size_t)((expect + lo8 + 80 + 7) / 8);
                if (hb == w.n) { sink.chain_end(DEC_ENDED); return BZ2B200_OK; }
                const u8 *in = hb + 4 <= w.n ? w.in + (hb - w.in_lo) : nullptr;   // hb > the footer's first byte >= in_lo
                if (!in || in[0] != 'B' || in[1] != 'Z' || in[2] != 'h' || in[3] < '1' || in[3] > '9') {
                    ctx->err = "decode: trailing bytes after the stream footer"; return BZ2B200_E_FORMAT;
                }
                ev.push_back(DecEvent{(u64)hb * 8, (u32)(in[3] - '0'), 0, DEC_STREAM});
                combined = 0; comb_known = true;
                expect = (u64)hb * 8 + 32 - lo8;
                continue;
            }
        }
        bool reuse = false;
        if (have_batch) for (u64 s : starts) reuse |= s == expect;
        have_batch = false;
        u32 nb = (u32)starts.size();
        if (!reuse) {
            // ---- 2. entropy decode of the next candidate blocks (decode4.cuh) ----
            // A block's data cannot reach past the next candidate -- unless that one is a chance magic inside it: the walk
            // then leaves the range its jump tables cover and finishes code by code.
            starts.clear(); rends.clear();
            for (size_t k = ci; k < ncand && starts.size() < NB; k++) {
                if (cand[k] & DEC_FOOT) continue;
                if ((cand[k] & ~DEC_FOOT) >= hi) break;             // the next window's
                u64 re = k + 1 < ncand ? (cand[k + 1] & ~DEC_FOOT) : (u64)n * 8;
                // no valid block is longer than 20 bits per symbol plus its header (symbol map, selectors, six tables): a
                // damaged stream whose next magic is far away must not size the jump tables
                re = std::min<u64>(re, cand[k] + (u64)20 * (max_block + 64) + ((u64)1 << 19));
                if (range_limit) re = std::min(re, cand[k] + range_limit);     // test knob: as if a chance magic cut the range
                starts.push_back(cand[k]); rends.push_back(re);
            }
            nb = (u32)starts.size();
            if (nb) {
                int rc = bz_dec_entropy(ctx, g, d_bits, n, starts, rends, db);
                if (rc) return rc;
            }
        }
        if (!known) {                                           // the hand-off from the window before
            long long s = sink.chain_start();
            if (s < 0) return DEC_ABORTED;
            if (s == DEC_ENDED) { sink.chain_end(DEC_ENDED); return BZ2B200_OK; }
            if ((u64)s < lo8) { ctx->err = "decode: chain enters the window before its first bit"; return BZ2B200_E_FORMAT; }
            known = true;
            expect = (u64)s - lo8;
            have_batch = nb != 0;
            continue;
        }
        // ---- the chain inside this batch: candidate k is a block iff the block before it ends exactly there ----
        u32 used = 0;
        for (u32 k = 0; k < nb; k++) {
            hlen[k] = 0; hkey[k] = 0; hrand[k] = 0;
            if (starts[k] != expect) continue;                  // inside another block's data: not a block
            if (db[k].status != 0) { ctx->err = "decode: block at bit " + std::to_string(starts[k] + lo8) + " status " + std::to_string(db[k].status); return BZ2B200_E_FORMAT; }
            if (db[k].key >= db[k].nblock) { ctx->err = "decode: origin pointer outside the block"; return BZ2B200_E_FORMAT; }
            hlen[k] = db[k].nblock; hkey[k] = db[k].key; hrand[k] = db[k].pad;
            combined = ((combined << 1) | (combined >> 31)) ^ db[k].crc;                       // crc.rs:25-27
            ev.push_back(DecEvent{starts[k] + lo8, db[k].crc, db[k].nblock, DEC_BLOCK});
            expect = db[k].end_bit;
            used = k + 1;
        }
        if (used == 0) { ctx->err = "decode: lost the block chain"; return BZ2B200_E_FORMAT; }
        const bool last = expect >= hi;                         // the chain left the window: the next one may go on
        if (last) sink.chain_end((long long)(expect + lo8));
        // candidates up to the last block of the chain are consumed (the next loop skips what lies below `expect`)
        while (ci < ncand && (cand[ci] & ~DEC_FOOT) <= starts[used - 1]) ci++;
        // ---- 3. inverse BWT (+ de-randomisation of legacy blocks), inverse RLE1 + CRC; the batch's bytes go where the
        // sink says ----
        int rc = bz_dec_unbwt(ctx, g, used, hlen.data(), hkey.data(), hrand.data(), olen.data());
        if (rc) return rc;
        u64 btotal = 0;
        for (u32 k = 0; k < used; k++) {
            if (olen[k] == RLE1_OPEN) { ctx->err = "decode: the block at bit " + std::to_string(starts[k] + lo8) + " ends with four equal bytes and no count byte"; return BZ2B200_E_FORMAT; }
            ooff[k] = btotal; btotal += olen[k];
        }
        u8 *d_out = nullptr, *h_out = nullptr;
        rc = sink.counted(btotal, last, &d_out, &h_out);
        if (rc) return rc;
        rc = bz_dec_write(ctx, g, used, olen.data(), ooff.data(), d_out, crcs.data());
        if (rc) return rc;
        if (btotal && h_out) BZ_CHECK(cudaMemcpyAsync(h_out, d_out, (size_t)btotal, cudaMemcpyDeviceToHost, ctx->stream));
        BZ_CHECK(cudaStreamSynchronize(ctx->stream));
        for (u32 k = 0; k < used; k++)
            if (hlen[k] && crcs[k] != db[k].crc) { ctx->err = "decode: CRC mismatch in the block at bit " + std::to_string(starts[k] + lo8); return BZ2B200_E_CRC; }   // enforced, unlike decompress.rs:379-386
        rc = sink.ready(d_out, btotal);
        if (rc) return rc;
    }
}

// Every block is at most 100000 x the level of ITS stream's "BZh<level>", as libbz2 checks it; the events are in chain
// order and a stream's header event precedes its blocks.  `level` is the first stream's.
int bz_check_block_sizes(std::string &err, int level, const std::vector<DecEvent> &ev) {
    for (const DecEvent &e : ev) {
        if (e.kind == DEC_STREAM) level = (int)e.val;
        else if (e.kind == DEC_BLOCK && e.nblock > (u32)level * 100000u) {
            err = "decode: block at bit " + std::to_string(e.bit) + " longer than its stream's level allows";
            return BZ2B200_E_FORMAT;
        }
    }
    return BZ2B200_OK;
}

namespace {
// the whole input is one window; bytes go straight to the caller's buffer
struct WholeSink : DecSink {
    bz2b200_ctx *ctx; u8 *out; size_t out_cap; size_t *out_len; size_t total = 0;
    int counted(u64 nbytes, bool, u8 **d_out, u8 **h_out) override {
        *out_len = total + (size_t)nbytes;
        if (total + nbytes > out_cap) return BZ2B200_E_CAP;
        BZ_CHECK(ctx->d_stream.ensure((size_t)nbytes + 64));
        *d_out = ctx->d_stream.as<u8>();
        *h_out = out + total;
        total += (size_t)nbytes;
        return BZ2B200_OK;
    }
};
}  // namespace

extern "C" int bz2b200_decompress_stream(bz2b200_ctx *ctx, const uint8_t *in, size_t n, uint8_t *out, size_t out_cap,
                                         size_t *out_len) {
    BZ_API_TRY
    if (!ctx || !in || !out_len || (!out && out_cap) || n < 14 || n > 0xFFFFFF00ull * 4ull) return BZ2B200_E_ARG;
    if (in[0] != 'B' || in[1] != 'Z' || in[2] != 'h' || in[3] < '1' || in[3] > '9') return BZ2B200_E_FORMAT;   // decompress.rs:46-62
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    cudaStream_t st = ctx->stream;
    *out_len = 0;
    BZ_CHECK(ctx->d_in.ensure(n + 64));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_in.p, in, n, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemsetAsync(ctx->d_in.as<u8>() + n, 0, 64, st));       // word loads of the entropy stage read past the last byte
    // ---- 1. every bit offset that looks like a block or footer magic ----
    std::vector<u64> cand;
    int rc = bz_dec_candidates(ctx, ctx->d_in.as<u8>(), n, (u32)std::min<size_t>(n / 32 + 64, 0x7fffff00u), cand);
    if (rc) return rc;
    if (cand.empty()) return BZ2B200_E_FORMAT;
    int level = in[3] - '0';
    for (u64 c : cand) {                                        // buffer geometry: the largest block size any header may announce
        if (!(c & DEC_FOOT)) continue;
        size_t hb = (size_t)(((c & ~DEC_FOOT) + 80 + 7) / 8);
        if (hb + 4 <= n && in[hb] == 'B' && in[hb + 1] == 'Z' && in[hb + 2] == 'h' && in[hb + 3] >= '1' && in[hb + 3] <= '9')
            level = std::max(level, in[hb + 3] - '0');
    }
    DecWindow w{in, 0, n, ctx->d_in.as<u8>(), 0, n, ~0ull, 32, 0, (u32)level * 100000u, &cand};
    WholeSink sink;
    sink.ctx = ctx; sink.out = out; sink.out_cap = out_cap; sink.out_len = out_len;
    std::vector<DecEvent> ev;
    rc = bz_decode_core(ctx, w, sink, ev);
    if (rc) return rc;
    rc = bz_check_block_sizes(ctx->err, in[3] - '0', ev);
    if (rc) return rc;
    *out_len = sink.total;
    return BZ2B200_OK;
    BZ_API_CATCH
}
