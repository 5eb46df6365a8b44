// bwt.cu -- cyclic-rotation BWT of a batch of RLE1 blocks as a GPU suffix sort.
//
// Replaces bwt_encode (reference src/bwt_algorithms/bwt_sort.rs:27-58): sort all n cyclic
// rotations of the block, key = row of rotation 0, bwt[i] = x[(idx[i]-1) mod n].  The reference
// does this with a comparison sort of full rotations (block_compare, bwt_sort.rs:61-86); here it
// is prefix doubling over packed rank keys:
//   1. LSD radix sort of all rotations by their first 8 bytes (sweep.cuh).  Keys are implicit: the
//      digit of a pass is gathered from the (L2 resident) block text, so a pass moves only the
//      4-byte rotation index; every other pass takes its digit from a byte carried in the index word.
//   2. k_init_ranks: head flags of the 8-byte groups -> rank[s] = first row of s's group; rotations in
//      groups of size > 1 are compacted into the "unresolved" list (one packed u64 per rotation).
//   3. doubling rounds h = 8,16,..: k_list_key sets key2 = rank[(s+h) mod n].  Unresolved groups live in one
//      of two lists per block:
//        LOC  groups of at most LCAP rotations (all but a few percent of real data).  k_refine_local sorts
//             every group inside shared memory -- all-pairs counting for groups up to SCAP, a segmented
//             LSD radix sort of (group | key2) for the rest -- and never touches global memory in between:
//             one read of the list, one write of SA / RANK / the next list per round.
//        BIG  larger groups (long runs, short periods).  The packed list is radix sorted globally by
//             (group head, key2) with five sweep passes and k_list_refine splits the groups.
//      Both rewrite SA and the ranks of the refined groups and re-compact what is still tied.  Stops when
//      every list is empty or h >= n (rotations still tied are equal: periodic block).
//   4. key = rank[0] (first row of the class of rotation 0), bwt[j] = T[(SA[j]-1) mod n].  With BZ2B200_LIBBZ2 the
//      other members of that class are counted too: a periodic block gets libbz2's row from the host (libbz2_order.cu).
// Steps 2 and 3 are single-pass kernels: the running (last head, list length) prefix over the tiles of a
// block comes from a decoupled look-back on one 64-bit state word per tile.
#include "common.cuh"
#include "sweep.cuh"

namespace {

// packed list element: [59:40] first row of the group, [39:20] key2, [19:0] rotation index
constexpr int FB = 20;
constexpr u64 FMASK = (1ull << FB) - 1;
static_assert(BZ2B200_MAX_BLOCK < (1u << FB) - 1, "packed list fields are 20 bits");

constexpr int RT_IPT = 8;
constexpr int RT = BZ_THREADS * RT_IPT;        // rows per refine tile
__device__ __forceinline__ u32 padi(u32 i) { return i + (i >> 5); }   // conflict-free blocked and striped access
constexpr int RT_PAD = RT + RT / 32 + 1;

// ---- local (shared memory) refinement: geometry ----
#ifndef BZ_LW
#define BZ_LW 3072
#endif
constexpr int LW = BZ_LW;               // window capacity of k_refine_local (elements)
constexpr int LIPT = LW / BZ_THREADS;    // 16 per thread, blocked
#ifndef BZ_LCAP
#define BZ_LCAP 1024
#endif
constexpr int LCAP = BZ_LCAP;            // largest group that is refined locally
constexpr int LTILE = LW - LCAP;         // nominal tile: a tile owns the groups that START inside it
#ifndef BZ_SCAP
#define BZ_SCAP 128
#endif
constexpr int SCAP = BZ_SCAP;            // groups up to this size are ranked by all-pairs counting
static_assert(LW % BZ_THREADS == 0 && LW <= 4096 && LCAP <= RT && LCAP * 2 <= LW && LCAP <= (1 << 11) && SCAP < LCAP && LW / (SCAP + 1) < 256, "local refinement geometry");
constexpr int LWP = LW + LW / 32 + 1;    // padded u32 arrays (padi)
__device__ __forceinline__ u32 padh(u32 i) { return i + 2u * (i >> 6); }   // u16 arrays, blocked access of 16
constexpr int LWH = LW + 2 * (LW / 64) + 2;

// 8 bytes of rotation s (memory order; only compared for equality).  T is 8-byte aligned and padded so
// that aligned loads up to offset n+15 stay inside the block's stride.
__device__ __forceinline__ u64 rot_key8(const u8 *T, u32 n, u32 s) {
    if (s + 8 <= n) {
        const u64 *w = (const u64 *)(T + (s & ~7u));
        u64 w0 = __ldg(w);
        u32 sh = (s & 7u) * 8u;
        if (sh == 0) return w0;
        u64 w1 = __ldg(w + 1);
        return (w0 >> sh) | (w1 << (64 - sh));
    }
    u64 k = 0;
    u32 p = s;
    for (int q = 0; q < 8; q++) { k |= (u64)T[p] << (8 * q); p++; if (p >= n) p = 0; }
    return k;
}

// ---- decoupled look-back over the tiles of one block: (max, max, sum) of three 20-bit quantities ----
// state word: [63:62] 1 = tile aggregate, 2 = inclusive prefix; [59:40] a+1, [39:20] b+1 (maxima, 0 = none), [19:0] sum
struct Tri { int a, b; u32 c; };
__device__ __forceinline__ u64 tri_pack(u32 flag, Tri v) {
    return ((u64)flag << 62) | ((u64)(u32)(v.a + 1) << 40) | ((u64)(u32)(v.b + 1) << 20) | (u64)v.c;
}
__device__ __forceinline__ Tri tri_unpack(u64 w) {
    Tri v;
    v.a = (int)((w >> 40) & FMASK) - 1; v.b = (int)((w >> 20) & FMASK) - 1; v.c = (u32)(w & FMASK);
    return v;
}
__device__ __forceinline__ u64 ld_vol64(const u64 *p) {
    u64 v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_vol64(u64 *p, u64 v) { asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory"); }

// Called by all lanes of warp 0.  `st` = state words of this block, `t` = tile, `agg` = this tile's aggregate.
// Returns the exclusive prefix over tiles [0, t).  Lane l inspects tile hi - l, so a window of 32 predecessors
// costs one L2 round trip (the tiles of one block that are in flight at the same time form a long chain).
// BSUM: field b is a sum (of at most 2^20 - 2) instead of a maximum; its identity is then 0 (packed as b + 1 = 1).
template <bool BSUM = false>
__device__ __forceinline__ Tri tile_lookback(u64 *st, u32 t, Tri agg) {
    const int lane = threadIdx.x & 31;
    const int bid = BSUM ? 0 : -1;
    Tri ex; ex.a = -1; ex.b = bid; ex.c = 0;
    if (t == 0) { if (lane == 0) st_vol64(st, tri_pack(2, agg)); return ex; }
    if (lane == 0) st_vol64(st + t, tri_pack(1, agg));
    for (int hi = (int)t - 1;;) {
        int tt = hi - lane;
        u64 w = tt >= 0 ? ld_vol64(st + tt) : ((2ull << 62) | ((u64)(u32)(bid + 1) << 20));   // before tile 0: an inclusive prefix of nothing
        u32 f = (u32)(w >> 62);
        u32 incm = __ballot_sync(0xffffffffu, f == 2);
        u32 nrm = __ballot_sync(0xffffffffu, f == 0);
        u32 need = incm ? ((2u << (__ffs(incm) - 1)) - 1u) : 0xffffffffu;   // lanes up to the nearest inclusive prefix
        if (nrm & need) continue;                                 // one of them is not published yet
        Tri v = tri_unpack(w);
        if (!((need >> lane) & 1u)) { v.a = -1; v.b = bid; v.c = 0; }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            v.a = max(v.a, __shfl_xor_sync(0xffffffffu, v.a, o));
            int ob = __shfl_xor_sync(0xffffffffu, v.b, o);
            v.b = BSUM ? v.b + ob : max(v.b, ob);
            v.c += __shfl_xor_sync(0xffffffffu, v.c, o);
        }
        ex.a = max(ex.a, v.a); ex.b = BSUM ? ex.b + v.b : max(ex.b, v.b); ex.c += v.c;
        if (incm) break;
        hi -= 32;
    }
    Tri inc; inc.a = max(ex.a, agg.a); inc.b = BSUM ? ex.b + agg.b : max(ex.b, agg.b); inc.c = ex.c + agg.c;
    if (lane == 0) st_vol64(st + t, tri_pack(2, inc));
    return ex;
}

struct RefineArgs {
    const u8 *T; const u32 *len;
    const u32 *cnt;        // rows per block (init: len; refine: current list length)
    u32 *SA; u32 *RANK;
    const u64 *LIN; u64 *LOUT;
    u32 *cnt_out;          // next list length per block
    u64 *LOUT2;            // k_init_ranks: the BIG list (groups of more than LCAP rotations)
    u32 *cnt_out2;
    u64 *tstate;           // [nblk][rtiles]
    u32 *ticket;
    u32 stride, rtiles, tiles_x, nblk, group;
    u32 depth_after;       // sorted depth once this kernel has run: lists of blocks it covers are dropped
};

// ticket -> (block, tile), the same interleaving as the sweep passes
__device__ __forceinline__ bool ticket_tile(const RefineArgs &a, u32 *s_ticket, u32 &b, u32 &t) {
    if (threadIdx.x == 0) *s_ticket = atomicAdd(a.ticket, 1u);
    __syncthreads();
    u32 ticket = *s_ticket;
    u32 per_group = a.group * a.tiles_x;
    u32 g = ticket / per_group, r = ticket - g * per_group;
    t = r / a.group;
    b = g * a.group + (r - t * a.group);
    return b < a.nblk;
}

// --------------------------------------------------------------------------------------
// step 2: groups of the 8-byte sort -> ranks and the first unresolved lists
// --------------------------------------------------------------------------------------
// Rotations in groups of size > 1 go to the LOC list (group of at most LCAP rows: refined in shared memory) or to the
// BIG list.  A group's size is exact even when it crosses tiles: rows are sorted, so "row start + LCAP has the same
// key" (tile where the group begins) and "row end - 1 - LCAP has the same key" (tile where it ends) are both the test
// size > LCAP; a tile without any head lies inside a group of more than RT >= LCAP rows.
#ifndef BZ_REFINE_MINB
#define BZ_REFINE_MINB 5
#endif
__global__ void __launch_bounds__(BZ_THREADS, BZ_REFINE_MINB) k_init_ranks(RefineArgs a) {
    __shared__ u64 sk[RT + 2];          // sk[i] = key of row base - 1 + i
    __shared__ __align__(8) u8 fl[RT + 8];
    __shared__ u32 hd[RT_PAD];
    __shared__ u16 ls[RT];
    __shared__ int wsi[8];
    __shared__ u32 wsu[8];
    __shared__ u32 s_ticket;
    __shared__ Tri s_ex;
    __shared__ int s_big[2];            // [0] the group that began before this tile, [1] the group that runs past it
    u32 b, t;
    if (!ticket_tile(a, &s_ticket, b, t)) return;
    const u32 n = a.len[b];
    const u32 base = t * RT;
    if (base >= n) return;
    const int tid = threadIdx.x;
    const size_t ob = (size_t)b * a.stride;
    const u8 *Tb = a.T + ob;
    const u32 *sa = a.SA + ob;
    u32 s[RT_IPT];
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 e = r * BZ_THREADS + tid, j = base + e;
        s[r] = 0;
        if (j < n) { s[r] = __ldg(sa + j); sk[e + 1] = rot_key8(Tb, n, s[r]); }
    }
    if (tid == 0 && base > 0) sk[0] = rot_key8(Tb, n, sa[base - 1]);
    if (tid == 32 && base + RT < n) sk[RT + 1] = rot_key8(Tb, n, sa[base + RT]);
    __syncthreads();
    for (u32 e = tid; e <= RT; e += BZ_THREADS) {
        u32 j = base + e;
        fl[e] = (j == 0 || j >= n || sk[e + 1] != sk[e]) ? 1 : 0;     // rows past the end count as heads
    }
    __syncthreads();
    // blocked: thread owns rows [tid*8, tid*8+8)
    const u32 eb = tid * RT_IPT;
    const u64 f8 = *(const u64 *)(fl + eb);
    const u32 f9 = fl[eb + 8];
    u32 fm = 0;                                                  // bit r: row eb + r is a head (rows past n included)
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) fm |= (u32)((f8 >> (8 * r)) & 1) << r;
    int last = -1;
    u32 hmask = 0, umask = 0;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 j = base + eb + r;
        bool h = (fm >> r) & 1;
        bool hn = (r == RT_IPT - 1) ? (f9 != 0) : ((fm >> (r + 1)) & 1);
        if (j < n) {
            if (h) { last = (int)j; hmask |= 1u << r; }
            if (!(h && hn)) umask |= 1u << r;
        }
    }
    int tl, fe;
    int head = block_excl_max(last, wsi, tl);                    // tl: last head row of the tile (absolute) or -1
    int nxa = block_excl_min_rev(fm ? (int)(eb + __ffs(fm) - 1) : 0x7fffffff, wsi, fe);   // fe: first head of the tile (relative)
    const bool cont = fl[RT] == 0;                               // the last group continues in the next tile
    if (tid == 64) {                                             // the group that began before this tile
        int big = 0;
        if (fl[0] == 0) {
            if (fe == 0x7fffffff && cont) big = 1;
            else {
                long long E = (long long)base + (fe == 0x7fffffff ? (int)RT : fe);      // its end row
                long long q = E - 1 - LCAP;
                if (q >= (long long)base) big = 1;
                else if (q >= 0) big = rot_key8(Tb, n, sa[q]) == sk[1];
            }
        }
        s_big[0] = big;
    }
    if (tid == 96) {                                             // the group that runs past this tile
        int big = 0;
        if (cont) {
            if (tl < 0) big = 1;
            else {
                u32 P = (u32)tl + LCAP;
                if (P < base + RT) big = 1;
                else if (P < n) big = rot_key8(Tb, n, sa[P]) == sk[RT];
            }
        }
        s_big[1] = big;
    }
    __syncthreads();
    // class of every unresolved row: next head after it -> size of its group
    const int nx_out = f9 ? (int)(eb + 8) : (nxa != 0x7fffffff ? nxa : (cont ? 0x7fffffff : (int)RT));
    u32 bmask = 0, nloc = 0, nbig = 0;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        if ((umask >> r) & 1) {
            u32 below = fm & ((2u << r) - 1u);
            int hh = below ? (int)(base + eb + 31 - __clz(below)) : head;           // in-tile head of this row or -1
            u32 above = fm >> (r + 1);
            int nx = above ? (int)(eb + r + __ffs(above)) : nx_out;                 // next head (relative) or "none"
            bool big;
            if (hh < 0) big = s_big[0] != 0;
            else if (nx == 0x7fffffff) big = s_big[1] != 0;
            else big = (int)base + nx - hh > LCAP;
            if (big) { bmask |= 1u << r; nbig++; } else nloc++;
        }
    }
    u32 tot;
    u32 kk = block_excl_sum(nloc | (nbig << 16), wsu, tot);     // both fit: a tile has 2048 rows
    const u32 tloc = tot & 0xffffu, tbig = tot >> 16;
    if (tid < 32) {
        Tri agg; agg.a = tl; agg.b = (int)tbig; agg.c = tloc;
        Tri ex = tile_lookback<true>(a.tstate + (size_t)b * a.rtiles, t, agg);
        if (tid == 0) {
            s_ex = ex;
            if (base + RT >= n) {
                bool done = a.depth_after >= n;
                a.cnt_out[b] = done ? 0u : ex.c + tloc;
                a.cnt_out2[b] = done ? 0u : (u32)ex.b + tbig;
            }
        }
    }
    __syncthreads();
    head = max(head, s_ex.a);
    u32 kl = kk & 0xffffu, kb = kk >> 16;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 e = eb + r;
        if ((hmask >> r) & 1) head = (int)(base + e);
        hd[padi(e)] = (u32)head;
        u16 v = 0xffff;
        if ((umask >> r) & 1) v = ((bmask >> r) & 1) ? (u16)(0x8000u | kb++) : (u16)(kl++);
        ls[e] = v;
    }
    __syncthreads();
    u32 *rank = a.RANK + ob;
    u64 *lout = a.LOUT + ob + s_ex.c;
    u64 *lout2 = a.LOUT2 + ob + (u32)s_ex.b;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 e = r * BZ_THREADS + tid, j = base + e;
        if (j < n) {
            u32 h = hd[padi(e)];
            rank[s[r]] = h;
            u32 slot = ls[e];
            if (slot != 0xffffu) {
                u64 v = ((u64)h << (2 * FB)) | s[r];
                if (slot & 0x8000u) lout2[slot & 0x7fffu] = v; else lout[slot] = v;
            }
        }
    }
}

// --------------------------------------------------------------------------------------
// step 3: doubling round
// --------------------------------------------------------------------------------------
// key2 = rank[(s+h) mod n] into every list element; HIST: also the digit totals of all 5 sort passes (BIG list only)
template <bool HIST>
__global__ void __launch_bounds__(BZ_THREADS) k_list_key(const u32 *cntp, const u32 *len, const u32 *RANK, u64 *LIST,
                                                         u32 *counts, u32 stride, u32 h) {
    u32 b = blockIdx.y, cnt = cntp[b], n = len[b];
    u32 base = blockIdx.x * BZ_TILE;
    if (base >= cnt) return;
    __shared__ u32 hist[HIST ? 5 : 1][256];
    if (HIST) {
        for (int i = threadIdx.x; i < 5 * 256; i += BZ_THREADS) (&hist[0][0])[i] = 0;
        __syncthreads();
    }
    size_t ob = (size_t)b * stride;
    u64 *list = LIST + ob;
    const u32 *rank = RANK + ob;
    u32 hh = h >= n ? h % n : h;
#pragma unroll 4
    for (int r = 0; r < BZ_IPT; r++) {
        u32 k = base + r * BZ_THREADS + threadIdx.x;
        if (k < cnt) {
            u64 x = list[k];
            u32 p = (u32)(x & FMASK) + hh;
            if (p >= n) p -= n;
            x = (x & ~(FMASK << FB)) | ((u64)__ldg(rank + p) << FB);
            list[k] = x;
            if (HIST) {
#pragma unroll
                for (int q = 0; q < 5; q++) atomicAdd(&hist[q][(u32)(x >> (FB + 8 * q)) & 255u], 1u);
            }
        }
    }
    if (HIST) {
        __syncthreads();
        for (int i = threadIdx.x; i < 5 * 256; i += BZ_THREADS) {
            u32 v = (&hist[0][0])[i];
            if (v) atomicAdd(&counts[(size_t)b * 8 * 256 + i], v);
        }
    }
}

// Sorted list -> refined groups: SA rows and ranks rewritten, still-tied entries compacted into the next list.
__global__ void __launch_bounds__(BZ_THREADS, BZ_REFINE_MINB > 5 ? 5 : BZ_REFINE_MINB) k_list_refine(RefineArgs a) {
    __shared__ u64 sk[RT + 2];          // sk[i] = (head, key2) of list entry base - 1 + i
    __shared__ __align__(8) u8 fl[RT + 8];
    __shared__ u32 kgs[RT_PAD], kss[RT_PAD];
    __shared__ u16 ls[RT];
    __shared__ int wsi[8];
    __shared__ u32 wsu[8];
    __shared__ u32 s_ticket;
    __shared__ Tri s_ex;
    u32 b, t;
    if (!ticket_tile(a, &s_ticket, b, t)) return;
    const u32 cnt = a.cnt[b];
    const u32 base = t * RT;
    const int tid = threadIdx.x;
    if (cnt == 0 && t == 0 && tid == 0) a.cnt_out[b] = 0;     // a finished block stays finished
    if (base >= cnt) return;
    const size_t ob = (size_t)b * a.stride;
    const u64 *lin = a.LIN + ob;
    u64 x[RT_IPT];
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 e = r * BZ_THREADS + tid, k = base + e;
        x[r] = 0;
        if (k < cnt) { x[r] = __ldg(lin + k); sk[e + 1] = x[r] >> FB; }
    }
    if (tid == 0 && base > 0) sk[0] = lin[base - 1] >> FB;
    if (tid == 32 && base + RT < cnt) sk[RT + 1] = lin[base + RT] >> FB;
    __syncthreads();
    for (u32 e = tid; e <= RT; e += BZ_THREADS) {
        u32 k = base + e;
        u8 f = 3;                                   // bit 0: subgroup start, bit 1: group start; past the end = both
        if (k != 0 && k < cnt) {
            u64 c = sk[e + 1], p = sk[e];
            f = (u8)((c != p ? 1 : 0) | ((c >> FB) != (p >> FB) ? 2 : 0));
        }
        fl[e] = f;
    }
    __syncthreads();
    const u32 eb = tid * RT_IPT;
    u64 f8 = *(const u64 *)(fl + eb);
    u32 f9 = fl[eb + 8];
    int la = -1, lb = -1; u32 unres = 0;
    u32 smask = 0, gmask = 0, umask = 0;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 k = base + eb + r;
        u32 f = (u32)(f8 >> (8 * r)) & 3u;
        u32 fn = (r == RT_IPT - 1) ? f9 : ((u32)(f8 >> (8 * r + 8)) & 3u);
        if (k < cnt) {
            if (f & 2) { la = (int)k; gmask |= 1u << r; }
            if (f & 1) { lb = (int)k; smask |= 1u << r; }
            if (!((f & 1) && (fn & 1))) { unres++; umask |= 1u << r; }
        }
    }
    int ta, tb; u32 tu;
    int kg = block_excl_max(la, wsi, ta);       // list index of the current group's first entry
    int ks = block_excl_max(lb, wsi, tb);       // list index of the current subgroup's first entry
    u32 ko = block_excl_sum(unres, wsu, tu);    // slot in the next list
    if (tid < 32) {
        Tri agg; agg.a = ta; agg.b = tb; agg.c = tu;
        Tri ex = tile_lookback(a.tstate + (size_t)b * a.rtiles, t, agg);
        if (tid == 0) {
            s_ex = ex;
            if (base + RT >= cnt) a.cnt_out[b] = (a.depth_after >= a.len[b]) ? 0u : ex.c + tu;
        }
    }
    __syncthreads();
    kg = max(kg, s_ex.a); ks = max(ks, s_ex.b);
    const u32 kbase = s_ex.c;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 e = eb + r;
        if ((gmask >> r) & 1) kg = (int)(base + e);
        if ((smask >> r) & 1) ks = (int)(base + e);
        kgs[padi(e)] = (u32)kg; kss[padi(e)] = (u32)ks;
        ls[e] = ((umask >> r) & 1) ? (u16)(ko++) : (u16)0xffff;
    }
    __syncthreads();
    u32 *sa = a.SA + ob, *rank = a.RANK + ob;
    u64 *lout = a.LOUT + ob + kbase;
#pragma unroll
    for (int r = 0; r < RT_IPT; r++) {
        u32 e = r * BZ_THREADS + tid, k = base + e;
        if (k < cnt) {
            u32 g = (u32)(x[r] >> (2 * FB));            // row of the group's first member
            u32 s = (u32)(x[r] & FMASK);
            u32 kgv = kgs[padi(e)], ksv = kss[padi(e)];
            u32 nh = g + (ksv - kgv);                   // row of the subgroup's first member = new rank
            sa[g + (k - kgv)] = s;
            rank[s] = nh;
            u32 slot = ls[e];
            if (slot != 0xffffu) lout[slot] = ((u64)nh << (2 * FB)) | s;
        }
    }
}

// --------------------------------------------------------------------------------------
// step 3, LOC list: groups of at most LCAP rotations are refined inside shared memory
// --------------------------------------------------------------------------------------
// A tile owns the groups that START in its LTILE list entries; its window reaches LCAP entries further, so every
// owned group is completely inside (the entries of a group are contiguous in the list).  Work is blocked: thread t
// owns window entries [16 t, 16 t + 16).
//   1. group extents from the head field (forward max / backward min scan of the group-start flags)
//   2. groups of at most SCAP entries: every entry counts the members with a smaller / equal key2 (all-pairs):
//      no sort, ~|group| shared-memory reads per entry
//   3. larger groups: their entries are numbered (group number | key2) and the window indices are sorted by that
//      32-bit key with 3-4 stable LSD passes in shared memory (warp match ranking, as the global sweeps do)
//   4. "still tied" flags by sorted position -> slots of the next list (exclusive scan + look-back over tiles),
//      then SA rows, ranks and the next list are written once.
// shared memory of k_refine_local (dynamic, > 48 KB): K | IDXA | IDXB | GSE | UP | wh; the next-list staging reuses K..IDXB
constexpr size_t LOC_K_BYTES = (size_t)LW * 4;
constexpr size_t LOC_I_BYTES = ((size_t)LWH * 2 + 15) & ~(size_t)15;
constexpr size_t LOC_G_BYTES = ((size_t)LWP * 4 + 15) & ~(size_t)15;
constexpr size_t LOC_U_BYTES = ((size_t)LWH * 2 + 15) & ~(size_t)15;
constexpr size_t LOC_W_BYTES = (size_t)(LW * 4 > 8 * 256 * 4 ? LW * 4 : 8 * 256 * 4);
constexpr size_t LOC_SMEM = LOC_K_BYTES + 2 * LOC_I_BYTES + LOC_G_BYTES + LOC_U_BYTES + LOC_W_BYTES;
static_assert(LOC_K_BYTES + 2 * LOC_I_BYTES >= (size_t)LW * 8, "staging area");
#ifndef BZ_LOCAL_MINB
#define BZ_LOCAL_MINB 3
#endif
__global__ void __launch_bounds__(BZ_THREADS, BZ_LOCAL_MINB) k_refine_local(RefineArgs a, u32 *err) {
    extern __shared__ __align__(16) u8 loc_smem[];
    u32 *K = (u32 *)loc_smem;                                   // by window index: key2 << 12 | index (unique); medium entries: group number << 20 | key2
    u16 *IDXA = (u16 *)(loc_smem + LOC_K_BYTES);                // window indices of the medium entries (ping)
    u16 *IDXB = (u16 *)(loc_smem + LOC_K_BYTES + LOC_I_BYTES);  // (pong)
    u32 *GSE = (u32 *)(loc_smem + LOC_K_BYTES + 2 * LOC_I_BYTES);   // by window index (padded): group head row; then group start | end << 16 (~0: not owned)
    u16 *UP = (u16 *)((u8 *)GSE + LOC_G_BYTES);                 // by SORTED window position (padded): window index of the entry (0xffff: none)
    u32 *wh = (u32 *)((u8 *)UP + LOC_U_BYTES);                  // LSD counters; later, by sorted position: slot | distance to the subgroup start << 12 | tied << 31
    __shared__ u16 MG_GS[LW / (SCAP + 1) + 4], MG_MB[LW / (SCAP + 1) + 4];
    __shared__ int wsi[8];
    __shared__ u32 wsu[8];
    __shared__ u32 s_ticket, s_prevhead;
    __shared__ Tri s_ex;
    u32 b, t;
    if (!ticket_tile(a, &s_ticket, b, t)) return;
    const u32 cnt = a.cnt[b];
    const u32 base = t * LTILE;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (cnt == 0 && t == 0 && tid == 0) a.cnt_out[b] = 0;      // a finished block stays finished
    if (base >= cnt) return;
    const size_t ob = (size_t)b * a.stride;
    const u64 *lin = a.LIN + ob + base;
    const u32 wlen = min((u32)LW, cnt - base);                  // entries in the window
    const u32 nom = min((u32)LTILE, cnt - base);                // ... of which the tile proper
    const int INF = 0x7fffffff;
    // ---- load (coalesced) ----
#pragma unroll 4
    for (int r = 0; r < LIPT; r++) {
        u32 i = r * BZ_THREADS + tid;
        if (i < wlen) {
            u64 x = __ldg(lin + i);
            K[i] = (((u32)(x >> FB) & (u32)FMASK) << 12) | i;
            GSE[padi(i)] = (u32)(x >> (2 * FB));
        }
        UP[padh(i)] = 0xffffu;
    }
    if (tid == 0) s_prevhead = base > 0 ? (u32)(__ldg(lin - 1) >> (2 * FB)) : 0xffffffffu;
    __syncthreads();
    // ---- 1. group extents (blocked: thread owns entries [IPT tid, IPT tid + IPT)) ----
    const u32 eb = tid * LIPT;
    u32 gfm = 0;                                                // bit r: entry eb + r starts a group
    {
        u32 prev = tid == 0 ? s_prevhead : GSE[padi(eb - 1)];
#pragma unroll 4
        for (int r = 0; r < LIPT; r++) {
            u32 i = eb + r;
            if (i < wlen) {
                u32 hc = GSE[padi(i)];
                if (hc != prev) gfm |= 1u << r;
                prev = hc;
            }
        }
    }
    int dummy;
    const int gin = block_excl_max(gfm ? (int)(eb + 31 - __clz(gfm)) : -1, wsi, dummy);      // last group start before my entries
    int nout = block_excl_min_rev(gfm ? (int)(eb + __ffs(gfm) - 1) : INF, wsi, dummy);       // first group start after them
    if (nout == INF) nout = (int)wlen;
    // an entry is OWNED when its group starts inside the tile proper; medium = owned, more than SCAP members
    u32 mcount = 0, mstarts = 0, medmask = 0;
    {
        int ge = nout;                                          // backwards: the end of the group of entry eb + r
        u32 gem[LIPT];
#pragma unroll
        for (int r = LIPT - 1; r >= 0; r--) {
            gem[r] = (u32)ge;
            if ((gfm >> r) & 1u) ge = (int)(eb + r);
        }
        int gs = gin;
#pragma unroll
        for (int r = 0; r < LIPT; r++) {
            u32 i = eb + r;
            if ((gfm >> r) & 1u) gs = (int)i;
            if (i < wlen) {
                u32 v = 0xffffffffu;
                if (gs >= 0 && gs < (int)nom) {
                    v = (u32)gs | (gem[r] << 16);
                    u32 size = gem[r] - (u32)gs;
                    if (size > (u32)LCAP) atomicOr(err, 1u);     // cannot happen: LOC groups are at most LCAP long
                    if (size > (u32)SCAP) { medmask |= 1u << r; mcount++; if ((u32)gs == i) mstarts++; }
                }
                GSE[padi(i)] = v;                               // the head rows are not needed any more (all flags are computed)
            }
        }
    }
    u32 mtot;
    const u32 mex = block_excl_sum(mcount | (mstarts << 16), wsu, mtot);
    const u32 M = mtot & 0xffffu, nmg = mtot >> 16;
    if (medmask) {
        u32 midx = mex & 0xffffu;
        u32 mgnext = mex >> 16;                                 // number of the next medium group to start
#pragma unroll 1
        for (int r = 0; r < LIPT; r++) {
            if ((medmask >> r) & 1u) {
                u32 i = eb + r;
                if ((gfm >> r) & 1u) { MG_GS[mgnext] = (u16)i; MG_MB[mgnext] = (u16)midx; mgnext++; }
                K[i] = ((mgnext - 1u) << FB) | (K[i] >> 12);    // the group of this entry is the last one that started
                IDXA[padh(midx)] = (u16)i;
                midx++;
            }
        }
    }
    __syncthreads();
    // ---- 2. small groups: all-pairs, entry i = r * 256 + tid (neighbouring lanes sit in the same or adjacent groups, so a
    //         warp's loop count is the largest group among 32 consecutive entries and the key reads are broadcasts).
    //         Keys are unique (index in the low bits): the members with a smaller key give the sorted position. ----
#pragma unroll 1
    for (int r = 0; r < LIPT; r++) {
        u32 i = r * BZ_THREADS + tid;
        if (i < wlen) {
            u32 g = GSE[padi(i)];
            u32 gs = g & 0xffffu, ge = g >> 16;
            if (g != 0xffffffffu && ge - gs <= (u32)SCAP) {
                const u32 mine = K[i];
                u32 off = 0;
#pragma unroll 4
                for (u32 q = gs; q < ge; q++) off += K[q] < mine;
                UP[padh(gs + off)] = (u16)i;
            }
        }
    }
    // ---- 3. medium groups: stable LSD sort of the window indices by (group number | key2), 8 bits per pass ----
    if (M) {
        u16 *src = IDXA, *dst = IDXB;
        const int gb = nmg > 1 ? 32 - __clz((int)nmg - 1) : 0;
        const int passes = (FB + gb + 7) / 8;
        const u32 C = ((M + BZ_THREADS - 1) / BZ_THREADS) * 32;  // entries per warp, a multiple of 32
        const u32 lt = (1u << lane) - 1u;
        u32 *whw = wh + w * 256;
        const u32 j0 = (u32)w * C + lane;
#pragma unroll 1
        for (int p = 0; p < passes; p++) {
            const int shift = 8 * p;
#pragma unroll
            for (int k = 0; k < 8; k++) wh[k * 256 + tid] = 0;
            __syncthreads();
#pragma unroll 1
            for (u32 o = 0; o < C; o += 32) {                   // digit counts of this warp's entries
                u32 j = j0 + o;
                bool valid = j < M;
                u32 d = valid ? (K[src[padh(j)]] >> shift) & 255u : 256u + (u32)lane;
                u32 peers = __match_any_sync(0xffffffffu, d);
                if (valid && (peers & lt) == 0) whw[d] += __popc(peers);
                __syncwarp();
            }
            __syncthreads();
            {   // digit = tid: exclusive bases, digit major, then warp
                u32 c[8], total = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) { c[k] = wh[k * 256 + tid]; total += c[k]; }
                u32 all;
                u32 run = block_excl_sum(total, wsu, all);
#pragma unroll
                for (int k = 0; k < 8; k++) { wh[k * 256 + tid] = run; run += c[k]; }
            }
            __syncthreads();
#pragma unroll 1
            for (u32 o = 0; o < C; o += 32) {                   // stable ranks, scatter
                u32 j = j0 + o;
                bool valid = j < M;
                u32 idx = valid ? (u32)src[padh(j)] : 0u;
                u32 d = valid ? (K[idx] >> shift) & 255u : 256u + (u32)lane;
                u32 peers = __match_any_sync(0xffffffffu, d);
                u32 before = __popc(peers & lt);
                u32 old = 0;
                if (before == 0 && valid) { old = whw[d]; whw[d] = old + __popc(peers); }
                old = __shfl_sync(0xffffffffu, old, __ffs(peers) - 1);
                if (valid) dst[padh(old + before)] = (u16)idx;
                __syncwarp();
            }
            __syncthreads();
            u16 *sw = src; src = dst; dst = sw;
        }
        for (u32 j = tid; j < M; j += BZ_THREADS) {             // sorted medium entry j -> its window position
            u32 i = src[padh(j)];
            u32 g = K[i] >> FB;
            UP[padh((u32)MG_GS[g] + (j - (u32)MG_MB[g]))] = (u16)i;
        }
    }
    __syncthreads();
    // ---- 4. subgroups and slots, by sorted position (blocked): position p starts a subgroup when it starts a group or
    //         its key2 differs from the one before; entries of subgroups with more than one member stay tied ----
    u32 tu;
    {
        u32 sfm = 0;                                            // bit r: position eb + r starts a subgroup (or holds nothing); bit IPT: position eb + IPT
        u32 occ = 0;                                            // bit r: position eb + r holds an entry
        u32 pk = 0xffffffffu;                                   // key2 of position eb - 1 (only compared inside a group)
        if (eb > 0) {
            u32 e = UP[padh(eb - 1)];
            if (e != 0xffffu) { u32 g = GSE[padi(e)]; pk = (g >> 16) - (g & 0xffffu) > (u32)SCAP ? K[e] & (u32)FMASK : K[e] >> 12; }
        }
#pragma unroll 2
        for (int r = 0; r <= LIPT; r++) {
            u32 p = eb + r;
            u32 e = p < (u32)LW ? (u32)UP[padh(p)] : 0xffffu;
            if (e == 0xffffu) { sfm |= 1u << r; pk = 0xffffffffu; continue; }
            u32 g = GSE[padi(e)];
            u32 k2 = (g >> 16) - (g & 0xffffu) > (u32)SCAP ? K[e] & (u32)FMASK : K[e] >> 12;
            if (p == (g & 0xffffu) || k2 != pk) sfm |= 1u << r;
            pk = k2;
            occ |= 1u << r;
        }
        occ &= (1u << LIPT) - 1u;
        const u32 own = sfm & ((1u << LIPT) - 1u);
        const u32 tm = occ & ~(own & (sfm >> 1));               // tied: not (subgroup start and the next position starts one)
        const int pin = block_excl_max(own ? (int)(eb + 31 - __clz(own)) : -1, wsi, dummy);   // last subgroup start before my positions
        u32 run = block_excl_sum((u32)__popc(tm), wsu, tu);
        int ps = pin;
#pragma unroll 4
        for (int r = 0; r < LIPT; r++) {
            u32 p = eb + r;
            if ((own >> r) & 1u) ps = (int)p;
            wh[p] = run | ((p - (u32)ps) << 12) | (((tm >> r) & 1u) << 31);
            run += (tm >> r) & 1u;
        }
    }
    __syncthreads();
    // ---- write SA rows and ranks, by sorted position (the rows of a group are consecutive); entries that stay tied
    //      are staged in slot order.  Warp 0 first obtains this tile's offset in the next list: it waits for the tiles
    //      before it while the other warps are busy with their stores. ----
    if (tid < 32) {
        Tri agg; agg.a = -1; agg.b = -1; agg.c = tu;
        Tri ex = tile_lookback(a.tstate + (size_t)b * a.rtiles, t, agg);
        if (tid == 0) {
            s_ex = ex;
            if (base + LTILE >= cnt) a.cnt_out[b] = (a.depth_after >= a.len[b]) ? 0u : ex.c + tu;
        }
    }
    u64 *stg = (u64 *)loc_smem;                                  // [tu] next-list entries in slot order (K, IDXA, IDXB are free)
    u32 *sa = a.SA + ob, *rank = a.RANK + ob;
#pragma unroll 2
    for (int r = 0; r < LIPT; r++) {
        u32 p = r * BZ_THREADS + tid;
        u32 e = UP[padh(p)];
        if (e != 0xffffu) {
            u32 gs = GSE[padi(e)] & 0xffffu;
            u32 v = wh[p];
            u64 x = __ldg(lin + e);
            u32 head = (u32)(x >> (2 * FB)), s = (u32)(x & FMASK);
            u32 off = p - gs;                                   // position inside the group
            u32 nh = head + off - ((v >> 12) & 0x7ffffu);       // row of the first member of the subgroup = new rank
            sa[head + off] = s;
            rank[s] = nh;
            if (v >> 31) stg[v & 0xfffu] = ((u64)nh << (2 * FB)) | s;
        }
    }
    __syncthreads();
    u64 *lout = a.LOUT + ob + s_ex.c;
    for (u32 q = tid; q < tu; q += BZ_THREADS) lout[q] = stg[q];
}

// Path selector of the reference (bwt_sort.rs:29, lms_complexity sais_fallback.rs:821-829, LMS typing :59-131): a block
// longer than 5000 bytes goes to the SA-IS fallback when its first 5000 bytes hold at most 1499 LMS positions (the
// sentinel counts as one).  The engine always computes the true rotation BWT (DESIGN.md section 3); this only COUNTS the
// blocks the reference would have routed to its fallback, so that a run can report them.  One CTA per block: a thread
// replays the reference's right-to-left scan over 40 positions, starting from the type of the position after them
// (S iff the first different byte to its right, inside the 5000-byte window, is larger).
__global__ void __launch_bounds__(128) k_ref_path(const u8 *T, const u32 *len, u32 stride, u32 *sais_blocks) {
    const u32 b = blockIdx.x;
    const u32 n = len[b];
    if (n <= 5000) return;
    const u8 *x = T + (size_t)b * stride;
    __shared__ u32 s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const int lo = threadIdx.x * 40;
    u32 lms = 0;
    if (lo < 4999) {
        const int top = min(lo + 40, 4999);                     // scan k = top - 1 .. lo; position `top` is the right neighbour
        bool cur_s = false;                                     // is position `top` of type S
        if (top < 4999) {
            u32 c = x[top];
            int j = top + 1;
            while (j <= 4999 && x[j] == c) j++;
            cur_s = j <= 4999 && x[j] > c;
        }
        u32 prev = x[top];
        for (int k = top - 1; k >= lo; k--) {
            u32 el = x[k];
            if (el < prev) cur_s = true;
            else if (el > prev) { if (cur_s) { lms++; cur_s = false; } }
            prev = el;
        }
    }
    lms = __reduce_add_sync(0xffffffffu, lms);
    if ((threadIdx.x & 31) == 0 && lms) atomicAdd(&s_cnt, lms);
    __syncthreads();
    if (threadIdx.x == 0 && s_cnt + 1u <= 1499u) atomicAdd(sais_blocks, 1u);     // + 1: the sentinel
}

// used-byte bitmap of every block from its byte histogram (rle2_mtf.rs:26-39 builds the same set by scanning)
__global__ void __launch_bounds__(256) k_used_from_hist(const u32 *counts, u32 cstride, u32 *usedbits) {
    u32 b = blockIdx.x;
    bool used = counts[(size_t)b * cstride + threadIdx.x] != 0;
    u32 m = __ballot_sync(0xffffffffu, used);
    if ((threadIdx.x & 31) == 0) usedbits[b * 8 + (threadIdx.x >> 5)] = m;
}

// --------------------------------------------------------------------------------------
// step 4
// --------------------------------------------------------------------------------------
// others (BZ2B200_LIBBZ2, zeroed before the launch): others[b] = the rotations other than 0 whose final rank is rank[0],
// i.e. k - 1 for a periodic block u^k.  libbz2 stores the row where its own sort leaves rotation 0 among those k equal
// rotations; the host finds it for the blocks with others[b] > 0 (bz_libbz2_fallback_origin).
__global__ void __launch_bounds__(BZ_THREADS) k_bwt_out(const u8 *T, const u32 *len, const u32 *SA, const u32 *RANK,
                                                        u8 *bwt, u32 *keyout, u32 stride, u32 *others) {
    u32 b = blockIdx.y, n = len[b];
    size_t ob = (size_t)b * stride;
    u32 base = blockIdx.x * BZ_TILE;
    if (blockIdx.x == 0 && threadIdx.x == 0) keyout[b] = n ? RANK[ob] : 0;
    if (others && base < n) {
        const u32 r0 = RANK[ob];
        u32 c = 0;
        for (int r = 0; r < BZ_IPT; r++) {
            u32 s = base + r * BZ_THREADS + threadIdx.x;
            if (s < n && s != 0 && RANK[ob + s] == r0) c++;
        }
        c = __reduce_add_sync(0xffffffffu, c);
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(&others[b], c);
    }
#pragma unroll 4
    for (int r = 0; r < BZ_IPT; r++) {
        u32 j = base + r * BZ_THREADS + threadIdx.x;
        if (j < n) {
            u32 s = SA[ob + j];
            bwt[ob + j] = T[ob + (s == 0 ? n - 1 : s - 1)];
        }
    }
}

}  // namespace

#define LAUNCH_OK()                                                  \
    do {                                                             \
        ctx->prof_end();                                             \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) { ctx->fail("kernel launch", e_, __FILE__, __LINE__); return BZ2B200_E_CUDA; } \
    } while (0)

int bz_bwt_batch(bz2b200_ctx *ctx, const Batch &B, u8 *d_bwt, u32 *d_key, u32 *d_usedbits) {
    if (B.nblk == 0) return BZ2B200_OK;
    if (B.max_n > BZ2B200_MAX_BLOCK || ((uintptr_t)B.T & 7u) || (B.stride & 7u)) { ctx->err = "bwt: bad batch geometry"; return BZ2B200_E_ARG; }
    cudaStream_t st = ctx->stream;
    const u64 ne_act = B.total_n;
    const size_t ne = (size_t)B.nblk * B.stride;
    const u32 min_tile = BZ_THREADS * 8;                                   // smallest sweep / refine tile
    const u32 tiles_min = B.stride / min_tile;
    const u32 DSTRIDE = 8 * 256;                                            // per block: up to 8 passes x 256 digit offsets
    const u32 NTICKET = 512;
    BZ_CHECK(ctx->d_SA.ensure(ne * 4));
    BZ_CHECK(ctx->d_SA2.ensure(ne * 4));
    BZ_CHECK(ctx->d_RANK.ensure(ne * 4));
    BZ_CHECK(ctx->d_KEYA.ensure(ne * 8));
    BZ_CHECK(ctx->d_KEYB.ensure(ne * 8));
    BZ_CHECK(ctx->d_thist.ensure((size_t)B.nblk * tiles_min * 256 * 4));
    BZ_CHECK(ctx->d_tagg.ensure((size_t)B.nblk * tiles_min * 8));
    BZ_CHECK(ctx->d_VALA.ensure(ne * 8));
    BZ_CHECK(ctx->d_VALB.ensure(ne * 8));
    BZ_CHECK(ctx->d_cnt.ensure((size_t)B.nblk * 4 * 4 + 16));
    BZ_CHECK(ctx->d_R.ensure(((size_t)B.nblk * DSTRIDE + NTICKET) * 4));
    BZ_CHECK(ctx->h_small.ensure((size_t)B.nblk * 8 + 64));
    u32 *d_sais = ctx->d_cnt.as<u32>() + (size_t)B.nblk * 4;      // [0] SA-IS block count, [1] error flag of k_refine_local
    BZ_CHECK(cudaMemsetAsync(d_sais, 0, 8, ctx->stream));
    if (!ctx->loc_attr_done) {
        BZ_CHECK(cudaFuncSetAttribute(k_refine_local, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LOC_SMEM));
        ctx->loc_attr_done = true;
    }
    u32 *SAa = ctx->d_SA.as<u32>(), *SAb = ctx->d_SA2.as<u32>(), *RANK = ctx->d_RANK.as<u32>();
    u64 *L0 = ctx->d_KEYA.as<u64>(), *L1 = ctx->d_KEYB.as<u64>();      // LOC lists (ping-pong)
    u64 *G0 = ctx->d_VALA.as<u64>(), *G1 = ctx->d_VALB.as<u64>();      // BIG lists
    u32 *tstate = ctx->d_thist.as<u32>();
    u64 *rstate = ctx->d_tagg.as<u64>();
    u32 *dcounts = ctx->d_R.as<u32>();
    u32 *tickets = dcounts + (size_t)B.nblk * DSTRIDE;
    const size_t rstate_bytes = (size_t)B.nblk * tiles_min * 8;

    BZ_CHECK(cudaMemsetAsync(dcounts, 0, ((size_t)B.nblk * DSTRIDE + NTICKET) * 4, st));
    BZ_CHECK(cudaMemsetAsync(tstate, 0, (size_t)B.nblk * tiles_min * 256 * 4, st));
    u32 epoch = 0, tk = 0;
    dim3 gfull((B.max_n + BZ_TILE - 1) / BZ_TILE, B.nblk);
    // The refine kernels scatter into RANK (and SA): few blocks in flight keep that working set inside the L2.
    static const u32 group_knob = [] { const char *e = getenv("BZ2B200_REFINE_GROUP"); u32 g = e ? (u32)atoi(e) : 4u; return g < 1 ? 1u : g; }();
    const u32 group = group_knob < (u32)B.nblk ? group_knob : (u32)B.nblk;

    // ---- 1. initial 8-byte LSD sort (implicit keys) ----
    // every pass has the same digit totals: the block's byte histogram (each byte is digit p of exactly one rotation)
    ctx->prof_begin(K_BYTE_HIST, ne_act); sweep::k_byte_hist<<<gfull, BZ_THREADS, 0, st>>>(B.T, B.len, dcounts, B.stride, DSTRIDE); LAUNCH_OK();
    ctx->prof_begin(K_REF_PATH, (u64)B.nblk * 5000); k_ref_path<<<B.nblk, 128, 0, st>>>(B.T, B.len, B.stride, d_sais); LAUNCH_OK();
    if (d_usedbits) { ctx->prof_begin(K_USED, (u64)B.nblk * 1024); k_used_from_hist<<<B.nblk, 256, 0, st>>>(dcounts, DSTRIDE, d_usedbits); LAUNCH_OK(); }
    ctx->prof_begin(K_DIGIT_SCAN, (u64)B.nblk * DSTRIDE * 4); sweep::k_digit_scan<<<B.nblk * 8, 256, 0, st>>>(dcounts); LAUNCH_OK();
    u32 *bufs[2] = {SAa, SAb};
    const u32 *src = nullptr;
    for (int p = 0; p < 8; p++) {
        sweep::Args a{};
        a.T = B.T; a.len = B.len; a.cnt = B.len; a.in = src; a.out = bufs[p & 1];
        a.stride = B.stride; a.off = 7 - p; a.nblk = (u32)B.nblk;
        epoch++;
        a.dbase = dcounts; a.dbase_stride = DSTRIDE; a.tstate = tstate; a.ticket = tickets + tk++; a.epoch = epoch;
        if ((p & 1) == 0) { ctx->prof_begin(K_SWEEP_GATHER, ne_act * 9); sweep::launch<sweep::M_GATHER>(a, B.max_n, st); }
        else { ctx->prof_begin(K_SWEEP_CARRY, ne_act * 8); sweep::launch<sweep::M_CARRY>(a, B.max_n, st); }
        LAUNCH_OK();
        src = bufs[p & 1];
    }
    u32 *SA = bufs[1];   // 8 passes end in the second buffer

    // ---- 2. heads, ranks, first unresolved lists ----
    u32 *cntL_cur = ctx->d_cnt.as<u32>(), *cntL_nxt = cntL_cur + B.nblk;
    u32 *cntB_cur = cntL_nxt + B.nblk, *cntB_nxt = cntB_cur + B.nblk;
    RefineArgs ra{};
    ra.T = B.T; ra.len = B.len; ra.SA = SA; ra.RANK = RANK; ra.stride = B.stride; ra.rtiles = tiles_min;
    ra.nblk = (u32)B.nblk; ra.group = group; ra.tstate = rstate;
    {
        BZ_CHECK(cudaMemsetAsync(rstate, 0, rstate_bytes, st));
        ra.cnt = B.len; ra.LIN = nullptr; ra.LOUT = L0; ra.cnt_out = cntL_cur; ra.LOUT2 = G0; ra.cnt_out2 = cntB_cur;
        ra.ticket = tickets + tk++;
        ra.tiles_x = (B.max_n + RT - 1) / RT; ra.depth_after = 8;
        u32 grid = ((ra.nblk + group - 1) / group) * group * ra.tiles_x;
        ctx->prof_begin(K_INIT_RANKS, ne_act * 16); k_init_ranks<<<grid, BZ_THREADS, 0, st>>>(ra); LAUNCH_OK();
    }

    // ---- 3. doubling rounds ----
    u32 *h_cnt = ctx->h_small.as<u32>();
    const int passes = 5;                      // bits [20, 60) of the packed element
    u64 rounds = 0, listsum = 0, bigsum = 0;
    for (u32 h = 8;; h *= 2) {
        BZ_CHECK(cudaMemcpyAsync(h_cnt + 2 * B.nblk, d_sais, 8, cudaMemcpyDeviceToHost, st));    // the last read-back has the final flag
        BZ_CHECK(cudaMemcpyAsync(h_cnt, cntL_cur, (size_t)B.nblk * 4, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaMemcpyAsync(h_cnt + B.nblk, cntB_cur, (size_t)B.nblk * 4, cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaStreamSynchronize(st));
        u32 maxl = 0, maxb = 0;
        u64 lsum = 0, bsum = 0;
        for (int b = 0; b < B.nblk; b++) {
            if (h_cnt[b] > maxl) maxl = h_cnt[b];
            if (h_cnt[B.nblk + b] > maxb) maxb = h_cnt[B.nblk + b];
            lsum += h_cnt[b]; bsum += h_cnt[B.nblk + b];
        }
        listsum += lsum + bsum; bigsum += bsum;
        if (maxl == 0 && maxb == 0) break;
        if (h >= (1u << 30)) { ctx->err = "bwt: doubling did not terminate"; return BZ2B200_E_CUDA; }
        rounds++;
        if (tk + (u32)passes + 3 > NTICKET) { BZ_CHECK(cudaMemsetAsync(tickets, 0, NTICKET * 4, st)); tk = 0; }
        // -- LOC list: shared-memory refinement --
        if (maxl) {
            dim3 gl((maxl + BZ_TILE - 1) / BZ_TILE, B.nblk);
            ctx->prof_begin(K_LIST_KEY, lsum * 20); k_list_key<false><<<gl, BZ_THREADS, 0, st>>>(cntL_cur, B.len, RANK, L0, nullptr, B.stride, h); LAUNCH_OK();
            BZ_CHECK(cudaMemsetAsync(rstate, 0, rstate_bytes, st));
            ra.cnt = cntL_cur; ra.LIN = L0; ra.LOUT = L1; ra.cnt_out = cntL_nxt; ra.LOUT2 = nullptr; ra.cnt_out2 = nullptr;
            ra.ticket = tickets + tk++;
            ra.tiles_x = (maxl + LTILE - 1) / LTILE; ra.depth_after = 2 * h;
            u32 grid = ((ra.nblk + group - 1) / group) * group * ra.tiles_x;
            ctx->prof_begin(K_REFINE_LOCAL, lsum * 24); k_refine_local<<<grid, BZ_THREADS, LOC_SMEM, st>>>(ra, d_sais + 1); LAUNCH_OK();
            { u64 *tl = L0; L0 = L1; L1 = tl; }
        } else BZ_CHECK(cudaMemsetAsync(cntL_nxt, 0, (size_t)B.nblk * 4, st));
        // -- BIG list: global radix sort by (group head, key2) --
        if (maxb) {
            dim3 gl((maxb + BZ_TILE - 1) / BZ_TILE, B.nblk);
            BZ_CHECK(cudaMemsetAsync(dcounts, 0, (size_t)B.nblk * DSTRIDE * 4, st));
            ctx->prof_begin(K_LIST_KEY, bsum * 20); k_list_key<true><<<gl, BZ_THREADS, 0, st>>>(cntB_cur, B.len, RANK, G0, dcounts, B.stride, h); LAUNCH_OK();
            ctx->prof_begin(K_DIGIT_SCAN, (u64)B.nblk * DSTRIDE * 4); sweep::k_digit_scan<<<B.nblk * 8, 256, 0, st>>>(dcounts); LAUNCH_OK();
            if (epoch + (u32)passes > 254) {                        // epochs are 8 bits: start over with a clean state array
                BZ_CHECK(cudaMemsetAsync(tstate, 0, (size_t)B.nblk * tiles_min * 256 * 4, st));
                epoch = 0;
            }
            for (int p = 0; p < passes; p++) {
                sweep::Args a{};
                a.T = B.T; a.len = B.len; a.cnt = cntB_cur; a.in = G0; a.out = G1;
                a.stride = B.stride; a.shift = FB + 8 * p; a.nblk = (u32)B.nblk;
                epoch++;
                a.dbase = dcounts + p * 256; a.dbase_stride = DSTRIDE; a.tstate = tstate; a.ticket = tickets + tk++; a.epoch = epoch;
                ctx->prof_begin(K_SWEEP_LIST, bsum * 16); sweep::launch<sweep::M_LIST>(a, maxb, st); LAUNCH_OK();
                u64 *tl = G0; G0 = G1; G1 = tl;
            }
            // sorted list now in G0; the next list is written to G1
            BZ_CHECK(cudaMemsetAsync(rstate, 0, rstate_bytes, st));
            ra.cnt = cntB_cur; ra.LIN = G0; ra.LOUT = G1; ra.cnt_out = cntB_nxt; ra.LOUT2 = nullptr; ra.cnt_out2 = nullptr;
            ra.ticket = tickets + tk++;
            ra.tiles_x = (maxb + RT - 1) / RT; ra.depth_after = 2 * h;
            u32 grid = ((ra.nblk + group - 1) / group) * group * ra.tiles_x;
            ctx->prof_begin(K_LIST_REFINE, bsum * 24); k_list_refine<<<grid, BZ_THREADS, 0, st>>>(ra); LAUNCH_OK();
            { u64 *tl = G0; G0 = G1; G1 = tl; }
        } else BZ_CHECK(cudaMemsetAsync(cntB_nxt, 0, (size_t)B.nblk * 4, st));
        { u32 *tc = cntL_cur; cntL_cur = cntL_nxt; cntL_nxt = tc; }
        { u32 *tc = cntB_cur; cntB_cur = cntB_nxt; cntB_nxt = tc; }
    }
    if (h_cnt[2 * B.nblk + 1]) { ctx->err = "bwt: a local group exceeded its capacity"; return BZ2B200_E_CUDA; }
    // ---- 4. output ----
    // BZ2B200_LIBBZ2: d_key has 2 * nblk entries, the second half receives the class counts of rotation 0
    u32 *others = ctx->mode == BZ_MODE_LIBBZ2 ? d_key + B.nblk : nullptr;
    if (others) BZ_CHECK(cudaMemsetAsync(others, 0, (size_t)B.nblk * 4, st));
    ctx->prof_begin(K_BWT_OUT, ne_act * (others ? 10 : 6));
    k_bwt_out<<<gfull, BZ_THREADS, 0, st>>>(B.T, B.len, SA, RANK, d_bwt, d_key, B.stride, others); LAUNCH_OK();
    ctx->bwt_stats[0] = (u64)B.nblk; ctx->bwt_stats[1] = ne_act; ctx->bwt_stats[2] = rounds; ctx->bwt_stats[3] = listsum;
    ctx->bwt_stats[4] = h_cnt[2 * B.nblk];                       // blocks of this batch the reference would send to SA-IS
    ctx->bwt_stats[5] += h_cnt[2 * B.nblk];                      // ... and since the context was created
    ctx->bwt_stats[6] += (u64)B.nblk;
    ctx->bwt_stats[7] = bigsum;                                  // part of [3] that went through the global (BIG) path
    return BZ2B200_OK;
}
