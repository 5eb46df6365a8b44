// huff.cu -- multi-table Huffman stage + bit packing, batched over blocks.
//
// Replaces huf_encode (reference src/huffman_coding/huffman.rs:79-468), init_tables (:472-532),
// improve_code_len_from_weights (huffman_code_from_weights.rs:17-84) and the BitPacker
// (src/bitstream/bitpacker.rs:17-112); with emit_header it also writes the block header of
// compress_block (src/compression/compress_block.rs:34-48).
//
//   k_huf_init     table count by m (:87-93), initial 0/15 cost tables (:472-532)
//   4 x { k_huf_select   one thread per 50-symbol group: 6 packed 10-bit costs per symbol, first
//                        minimum wins (:137-153), rfreq[winner][sym]++ (:165-167)
//         k_huf_lengths  one warp per (block, table): exact (weight, syms) ordered tree build with
//                        the depth-17 halving retry (huffman_code_from_weights.rs:17-84) }
//   k_huf_gbits    final bit cost per group, selector MTF position by look-back (:237-275)
//   k_huf_layout   section sizes, exclusive scans -> bit offsets, canonical codes (:322-374),
//                  header / symbol map / table deltas (:209-224, :391-438)
//   k_huf_emit     one thread per group: selector unary code (:282-292) and the 50 symbol codes
//                  (:452-466) written MSB first at absolute bit offsets (atomicOr only at seams).
#include "common.cuh"

namespace {

constexpr int NSYM = BZ_MAXSYM;       // 258

struct HufWs {
    u8 *len6;       // [nblk][6][258]
    u64 *tab64;     // [nblk][258]  6 x 10-bit costs per symbol
    u32 *rfreq;     // [nblk][6][258]
    u8 *sel;        // [nblk][sel_stride]
    u32 *gbits;     // [nblk][sel_stride] data bits per group -> exclusive offsets
    u32 *sbits;     // [nblk][sel_stride] selector code bits per group -> exclusive offsets
    u32 *codes;     // [nblk][6][258] len<<24 | code
    u32 *misc;      // [nblk][8]: 0=T 1=G 2=nsym(eob+1) 3=sel_start 4=data_start 5=selector bits
    u32 sel_stride;
};

__device__ __forceinline__ u32 bswap32(u32 v) { return __byte_perm(v, 0, 0x0123); }

// MSB-first bit write of `nbits` (<= 32) low bits of `value` at absolute bit position `pos`.
__device__ __forceinline__ void put_bits(u32 *out, u64 pos, u32 value, int nbits) {
    if (nbits == 0) return;
    u32 w = (u32)(pos >> 5);
    int off = (int)(pos & 31);
    u64 v = ((u64)value << (64 - nbits)) >> off;
    u32 hi = (u32)(v >> 32), lo = (u32)v;
    if (hi) atomicOr(&out[w], bswap32(hi));
    if (lo) atomicOr(&out[w + 1], bswap32(lo));
}

__device__ __forceinline__ u32 used_count(const u32 *ub) {
    u32 c = 0;
    for (int k = 0; k < 8; k++) c += __popc(ub[k]);
    return c;
}

// ---- k_huf_init: one CTA per block ---------------------------------------------------------
__global__ void __launch_bounds__(256) k_huf_init(const u32 *m_in, const u32 *freq, const u32 *usedbits, HufWs W) {
    u32 b = blockIdx.x;
    u32 m = m_in[b];
    u32 eob = used_count(usedbits + b * 8) + 1;
    int T = m < 200 ? 2 : m < 600 ? 3 : m < 1200 ? 4 : m < 2400 ? 5 : 6;     // huffman.rs:87-93
    u8 *len = W.len6 + (size_t)b * 6 * NSYM;
    for (int i = threadIdx.x; i < 6 * NSYM; i += 256) len[i] = 15;
    __shared__ u32 sfreq[256];
    __shared__ u32 ws[8];
    u32 f = freq[b * 256 + threadIdx.x];
    sfreq[threadIdx.x] = f;
    u32 total;
    block_excl_sum(f, ws, total);
    __syncthreads();
    if (threadIdx.x == 0) {
        // init_tables, huffman.rs:472-532
        u32 limit = total / (u32)T;
        int ti = T - 1;
        u32 portion = 0;
        int lim = (int)eob + 1; if (lim > 256) lim = 256;
        for (int i = 0; i < lim; i++) {
            u32 fi = sfreq[i];
            if (portion + fi > limit && (ti == 2 || ti == 4)) {
                ti = ti > 0 ? ti - 1 : 0;
                len[ti * NSYM + i] = 0;
                portion = fi;
                if (portion > limit) { ti = ti > 0 ? ti - 1 : 0; portion = 0; }
            } else {
                portion += fi;
                len[ti * NSYM + i] = 0;
                if (portion > limit) { ti = ti > 0 ? ti - 1 : 0; portion = 0; }
            }
        }
        u32 *mi = W.misc + b * 8;
        mi[0] = (u32)T; mi[1] = (m + BZ_GROUP - 1) / BZ_GROUP; mi[2] = eob + 1;
    }
    __syncthreads();
    for (int s = threadIdx.x; s < NSYM; s += 256) {
        u64 v = 0;
        for (int t = 0; t < 6; t++) v |= (u64)len[t * NSYM + s] << (10 * t);
        W.tab64[(size_t)b * NSYM + s] = v;
    }
}

// ---- k_huf_select: thread per group ---------------------------------------------------------
__global__ void __launch_bounds__(256) k_huf_select(const u16 *sym, const u32 *m_in, HufWs W, u32 stride) {
    u32 b = blockIdx.y;
    u32 m = m_in[b];
    u32 g0 = blockIdx.x * 256;
    u32 G = (m + BZ_GROUP - 1) / BZ_GROUP;
    if (g0 >= G) return;
    __shared__ __align__(16) u16 ssym[256 * BZ_GROUP];
    __shared__ u64 stab[NSYM];
    __shared__ u32 srf[6 * NSYM];
    const u16 *s = sym + (size_t)b * stride;
    u32 first = g0 * BZ_GROUP;
    u32 cnt = min((u32)(256 * BZ_GROUP), m - first);
    for (u32 i = threadIdx.x; i < cnt; i += 256) ssym[i] = s[first + i];
    for (int i = threadIdx.x; i < NSYM; i += 256) stab[i] = W.tab64[(size_t)b * NSYM + i];
    for (int i = threadIdx.x; i < 6 * NSYM; i += 256) srf[i] = 0;
    __syncthreads();
    int T = (int)W.misc[b * 8 + 0];
    u32 g = g0 + threadIdx.x;
    if (g < G) {
        u32 a = threadIdx.x * BZ_GROUP;
        u32 e = min(a + BZ_GROUP, cnt);
        u64 acc = 0;
        for (u32 i = a; i < e; i++) acc += stab[ssym[i]];
        int bt = 0; u32 best = (u32)(acc & 1023);
        for (int t = 1; t < T; t++) {
            u32 c = (u32)((acc >> (10 * t)) & 1023);
            if (c < best) { best = c; bt = t; }          // first minimum, huffman.rs:150-153
        }
        for (u32 i = a; i < e; i++) atomicAdd(&srf[bt * NSYM + ssym[i]], 1u);
        W.sel[(size_t)b * W.sel_stride + g] = (u8)bt;
    }
    __syncthreads();
    u32 *rf = W.rfreq + (size_t)b * 6 * NSYM;
    for (int i = threadIdx.x; i < 6 * NSYM; i += 256) if (srf[i]) atomicAdd(&rf[i], srf[i]);
}

// ---- k_huf_lengths: one warp per (block, table) ---------------------------------------------
// Node order = descending (weight, syms), the two smallest are popped from the end, the parent is
// re-inserted after existing equal keys (the rule the oracle pins, SURVEY D.3).
__global__ void __launch_bounds__(192) k_huf_lengths(HufWs W) {
    u32 b = blockIdx.x;
    int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int T = (int)W.misc[b * 8 + 0];
    int nsym = (int)W.misc[b * 8 + 2];
    __shared__ u64 okey[6][264];
    __shared__ u16 oid[6][264];
    __shared__ u16 parent[6][528];
    __shared__ u32 wt[6][264];
    u32 *rf = W.rfreq + ((size_t)b * 6 + t) * NSYM;
    u8 *len = W.len6 + ((size_t)b * 6 + t) * NSYM;
    if (t < T) {
        for (int s = lane; s < nsym; s += 32) {
            u32 f = rf[s];
            wt[t][s] = (f == 0 ? 1u : f) << 8;                 // huffman_code_from_weights.rs:31
        }
        for (int s = lane; s < NSYM; s += 32) rf[s] = 0;       // ready for the next pass
        __syncwarp();
        for (;;) {
            // sort leaves by key descending (keys are distinct: syms = symbol id)
            for (int s = lane; s < nsym; s += 32) {
                u64 k = ((u64)wt[t][s] << 32) | (u32)s;
                int r = 0;
                for (int q = 0; q < nsym; q++) {
                    u64 kq = ((u64)wt[t][q] << 32) | (u32)q;
                    r += (kq > k);
                }
                okey[t][r] = k; oid[t][r] = (u16)s;
            }
            __syncwarp();
            int cnt = nsym, nn = nsym;
            while (cnt > 1) {
                u64 kr = okey[t][cnt - 1], kl = okey[t][cnt - 2];      // right = smallest, left = next
                u16 ir = oid[t][cnt - 1], il = oid[t][cnt - 2];
                cnt -= 2;
                u32 wr = (u32)(kr >> 32), wl = (u32)(kl >> 32);
                u32 dr = wr & 0xff, dl = wl & 0xff;
                u32 pw = ((wl & 0xffffff00u) + (wr & 0xffffff00u)) | (1 + max(dl, dr));   // add_weights :105-109
                u32 ps = (u32)kl + (u32)kr;                                               // syms sum :56
                u64 pk = ((u64)pw << 32) | ps;
                if (lane == 0) { parent[t][il] = (u16)nn; parent[t][ir] = (u16)nn; }
                // number of list entries with key < pk (they form the tail of the descending list)
                int smaller = 0;
                for (int base = cnt - 1; base >= 0; base -= 32) {
                    int idx = base - lane;
                    bool lt = idx >= 0 && okey[t][idx] < pk;
                    unsigned bal = __ballot_sync(0xffffffffu, lt);
                    if (bal == 0xffffffffu) { smaller += 32; continue; }
                    smaller += __ffs(~bal) - 1;
                    break;
                }
                int pos = cnt - smaller;
                // shift [pos, cnt) right by one, highest first
                for (int base = cnt - 1; base >= pos; base -= 32) {
                    int idx = base - lane;
                    u64 kk = 0; u16 ii = 0;
                    bool mv = idx >= pos;
                    if (mv) { kk = okey[t][idx]; ii = oid[t][idx]; }
                    __syncwarp();
                    if (mv) { okey[t][idx + 1] = kk; oid[t][idx + 1] = ii; }
                    __syncwarp();
                }
                if (lane == 0) { okey[t][pos] = pk; oid[t][pos] = (u16)nn; }
                __syncwarp();
                cnt++; nn++;
            }
            int root = nn - 1;
            // leaf depths (return_leaves, :88-101)
            int maxd = 0;
            int dep[9];
#pragma unroll
            for (int k = 0; k < 9; k++) {
                int s = lane + 32 * k;
                int d = 0;
                if (s < nsym) { int x = s; while (x != root) { x = parent[t][x]; d++; } }
                dep[k] = d;
                maxd = max(maxd, d);
            }
            maxd = __reduce_max_sync(0xffffffffu, maxd);
            if (maxd <= 17) {                                    // :65
#pragma unroll
                for (int k = 0; k < 9; k++) { int s = lane + 32 * k; if (s < nsym) len[s] = (u8)dep[k]; }
                break;
            }
            for (int s = lane; s < nsym; s += 32) { u32 j = wt[t][s] >> 8; j = 1 + j / 2; wt[t][s] = j << 8; }   // :76-80
            __syncwarp();
        }
    }
    __syncthreads();
    // repack the 6 x 10-bit cost words
    u8 *l6 = W.len6 + (size_t)b * 6 * NSYM;
    for (int s = threadIdx.x; s < NSYM; s += 192) {
        u64 v = 0;
        for (int q = 0; q < 6; q++) v |= (u64)l6[q * NSYM + s] << (10 * q);
        W.tab64[(size_t)b * NSYM + s] = v;
    }
}

// ---- BZ2B200_LIBBZ2: libbz2's initial partition and code lengths (DESIGN.md §10) ----------
// k_huf_init_libbz2: one CTA per block.  Exact counts of every MTF symbol 0..EOB (EOB once), then libbz2's partition
// of the alphabet into nGroups ranges of about remF / nPart symbols each (the odd-numbered inner ranges give their
// last symbol back).  Same outputs as k_huf_init.
__global__ void __launch_bounds__(256) k_huf_init_libbz2(const u16 *sym, const u32 *m_in, const u32 *usedbits, HufWs W,
                                                         u32 stride) {
    u32 b = blockIdx.x;
    u32 m = m_in[b];
    int alpha = (int)used_count(usedbits + b * 8) + 2;          // nInUse + 2 = EOB + 1
    int T = m < 200 ? 2 : m < 600 ? 3 : m < 1200 ? 4 : m < 2400 ? 5 : 6;
    u8 *len = W.len6 + (size_t)b * 6 * NSYM;
    __shared__ u32 mf[NSYM];
    for (int i = threadIdx.x; i < 6 * NSYM; i += 256) len[i] = 15;
    for (int i = threadIdx.x; i < NSYM; i += 256) mf[i] = 0;
    __syncthreads();
    const u16 *s = sym + (size_t)b * stride;
    for (u32 i = threadIdx.x; i < m; i += 256) atomicAdd(&mf[s[i]], 1u);
    __syncthreads();
    if (threadIdx.x == 0) {
        int nPart = T, gs = 0;
        u32 remF = m;
        while (nPart > 0) {
            u32 tFreq = remF / (u32)nPart, aFreq = 0;
            int ge = gs - 1;
            while (aFreq < tFreq && ge < alpha - 1) { ge++; aFreq += mf[ge]; }
            if (ge > gs && nPart != T && nPart != 1 && ((T - nPart) % 2 == 1)) { aFreq -= mf[ge]; ge--; }
            for (int v = gs; v <= ge; v++) len[(nPart - 1) * NSYM + v] = 0;
            nPart--; gs = ge + 1; remF -= aFreq;
        }
        u32 *mi = W.misc + b * 8;
        mi[0] = (u32)T; mi[1] = (m + BZ_GROUP - 1) / BZ_GROUP; mi[2] = (u32)alpha;
    }
    __syncthreads();
    for (int v = threadIdx.x; v < NSYM; v += 256) {
        u64 w = 0;
        for (int t = 0; t < 6; t++) w |= (u64)len[t * NSYM + v] << (10 * t);
        W.tab64[(size_t)b * NSYM + v] = w;
    }
}

// k_huf_lengths_libbz2: one warp per (block, table), BZ2_hbMakeCodeLengths(maxLen = 17) restated exactly: a binary
// heap of leaves keyed by weight = (freq or 1) << 8 | depth, ties broken by the heap's own sift order (part of the
// output), parents weighted (sum of counts) | (1 + max depth); while a code is longer than 17 bits every count is
// halved (1 + c / 2) and the tree is built again.  Lane 0 runs the heap (it is serial); the lanes walk the leaf depths.
__global__ void __launch_bounds__(192) k_huf_lengths_libbz2(HufWs W) {
    u32 b = blockIdx.x;
    int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int T = (int)W.misc[b * 8 + 0];
    int alpha = (int)W.misc[b * 8 + 2];
    __shared__ u32 weight[6][2 * NSYM + 2];
    __shared__ int parent[6][2 * NSYM + 2];
    __shared__ int heap[6][NSYM + 2];
    u32 *rf = W.rfreq + ((size_t)b * 6 + t) * NSYM;
    u8 *len = W.len6 + ((size_t)b * 6 + t) * NSYM;
    if (t < T) {
        u32 *wt = weight[t];
        int *par = parent[t], *hp = heap[t];
        for (int i = lane; i < alpha; i += 32) { u32 f = rf[i]; wt[i + 1] = (f == 0 ? 1u : f) << 8; }
        for (int s = lane; s < NSYM; s += 32) rf[s] = 0;         // ready for the next pass
        __syncwarp();
        for (;;) {
            if (lane == 0) {
                int nNodes = alpha, nHeap = 0;
                hp[0] = 0; wt[0] = 0; par[0] = -2;
                for (int i = 1; i <= alpha; i++) {
                    par[i] = -1;
                    int z = ++nHeap; hp[z] = i;                              // UPHEAP(nHeap)
                    int tmp = hp[z]; u32 wtmp = wt[tmp];
                    while (wtmp < wt[hp[z >> 1]]) { hp[z] = hp[z >> 1]; z >>= 1; }
                    hp[z] = tmp;
                }
                while (nHeap > 1) {
                    int nn[2];
                    for (int k = 0; k < 2; k++) {
                        nn[k] = hp[1]; hp[1] = hp[nHeap--];                 // DOWNHEAP(1)
                        int z = 1, tmp = hp[z]; u32 wtmp = wt[tmp];
                        for (;;) {
                            int y = z << 1;
                            if (y > nHeap) break;
                            if (y < nHeap && wt[hp[y + 1]] < wt[hp[y]]) y++;
                            if (wtmp < wt[hp[y]]) break;
                            hp[z] = hp[y]; z = y;
                        }
                        hp[z] = tmp;
                    }
                    int n1 = nn[0], n2 = nn[1];
                    nNodes++;
                    par[n1] = par[n2] = nNodes;
                    u32 w1 = wt[n1], w2 = wt[n2];
                    wt[nNodes] = ((w1 & 0xffffff00u) + (w2 & 0xffffff00u)) | (1u + max(w1 & 0xffu, w2 & 0xffu));
                    par[nNodes] = -1;
                    int z = ++nHeap; hp[z] = nNodes;                         // UPHEAP(nHeap)
                    int tmp = hp[z]; u32 wtmp = wt[tmp];
                    while (wtmp < wt[hp[z >> 1]]) { hp[z] = hp[z >> 1]; z >>= 1; }
                    hp[z] = tmp;
                }
            }
            __syncwarp();
            int maxd = 0;
            int dep[9];
#pragma unroll
            for (int k = 0; k < 9; k++) {
                int i = lane + 32 * k + 1;
                int d = 0;
                if (i <= alpha) { int x = i; while (par[x] >= 0) { x = par[x]; d++; } }
                dep[k] = d;
                maxd = max(maxd, d);
            }
            maxd = __reduce_max_sync(0xffffffffu, maxd);
            if (maxd <= 17) {
#pragma unroll
                for (int k = 0; k < 9; k++) { int i = lane + 32 * k; if (i < alpha) len[i] = (u8)dep[k]; }
                break;
            }
            for (int i = lane + 1; i <= alpha; i += 32) wt[i] = (1u + (wt[i] >> 8) / 2) << 8;
            __syncwarp();
        }
    }
    __syncthreads();
    u8 *l6 = W.len6 + (size_t)b * 6 * NSYM;
    for (int s = threadIdx.x; s < NSYM; s += 192) {
        u64 v = 0;
        for (int q = 0; q < 6; q++) v |= (u64)l6[q * NSYM + s] << (10 * q);
        W.tab64[(size_t)b * NSYM + s] = v;
    }
}

// ---- k_huf_gbits: thread per group -----------------------------------------------------------
__global__ void __launch_bounds__(256) k_huf_gbits(const u16 *sym, const u32 *m_in, HufWs W, u32 stride) {
    u32 b = blockIdx.y;
    u32 m = m_in[b];
    u32 g0 = blockIdx.x * 256;
    u32 G = (m + BZ_GROUP - 1) / BZ_GROUP;
    if (g0 >= G) return;
    __shared__ __align__(16) u16 ssym[256 * BZ_GROUP];
    __shared__ u64 stab[NSYM];
    const u16 *s = sym + (size_t)b * stride;
    u32 first = g0 * BZ_GROUP;
    u32 cnt = min((u32)(256 * BZ_GROUP), m - first);
    for (u32 i = threadIdx.x; i < cnt; i += 256) ssym[i] = s[first + i];
    for (int i = threadIdx.x; i < NSYM; i += 256) stab[i] = W.tab64[(size_t)b * NSYM + i];
    const u8 *sel = W.sel + (size_t)b * W.sel_stride;
    __shared__ u8 ssel[256];
    __shared__ int s_last[6];
    const int T = (int)W.misc[b * 8 + 0];
    ssel[threadIdx.x] = g0 + threadIdx.x < G ? sel[g0 + threadIdx.x] : (u8)0;
    if (threadIdx.x < 6) s_last[threadIdx.x] = -1;
    __syncthreads();
    for (int hi = (int)g0; hi > 0; hi -= 256) {                  // last use of every table before g0 (all threads take part)
        int j = hi - 1 - (int)threadIdx.x;
        if (j >= 0) { int u = sel[j]; if (u < 6) atomicMax(&s_last[u], j); }
        __syncthreads();
        bool all = true;
        for (int t = 0; t < T; t++) all = all && s_last[t] >= 0;
        __syncthreads();
        if (all) break;
    }
    u32 g = g0 + threadIdx.x;
    if (g >= G) return;
    int v = ssel[threadIdx.x];
    u32 a = threadIdx.x * BZ_GROUP, e = min(a + BZ_GROUP, cnt);
    u64 acc = 0;
    for (u32 i = a; i < e; i++) acc += stab[ssym[i]];
    W.gbits[(size_t)b * W.sel_stride + g] = (u32)((acc >> (10 * v)) & 1023);
    // selector MTF position (huffman.rs:237-275) = number of distinct tables used since the last use of v.  Looking back
    // selector by selector is one dependent load per step, and a table that was last used thousands of groups ago (with
    // fewer than T - 1 others in between) made one thread do that alone: 0.2-0.3 ms whatever the batch size.  So: the CTA
    // first finds, together, the last use of every table before its 256 groups; a thread then looks back inside the CTA's
    // groups (shared memory) and, if that does not decide, through those at most six positions.
    int pos = -1;
    {
        u32 mask = 0;
        for (int k = (int)threadIdx.x - 1; k >= 0; k--) {
            int u = ssel[k];
            if (u == v) { pos = __popc(mask); break; }
            mask |= 1u << u;
            if (__popc(mask) == T - 1) { pos = T - 1; break; }
        }
        if (pos < 0) {
            u32 visited = 0;
            for (int it = 0; it < T && pos < 0; it++) {
                int best = -1, bt = -1;
                for (int t = 0; t < T; t++) if (!((visited >> t) & 1u) && s_last[t] > best) { best = s_last[t]; bt = t; }
                if (bt < 0) break;
                visited |= 1u << bt;
                if (bt == v) pos = __popc(mask);
                else if (!((mask >> bt) & 1u)) { mask |= 1u << bt; if (__popc(mask) == T - 1) pos = T - 1; }
            }
            if (pos < 0) pos = __popc(mask) + __popc(~mask & ((1u << v) - 1));   // never used before: initial order 0..5
        }
    }
    W.sbits[(size_t)b * W.sel_stride + g] = (u32)pos + 1;
}

// ---- k_huf_layout: one CTA per block ---------------------------------------------------------
__global__ void __launch_bounds__(256) k_huf_layout(HufWs W, const u32 *usedbits, int emit_header, const u32 *crc,
                                                    const u32 *key, u8 *outb, size_t out_stride, u64 *bits_out) {
    u32 b = blockIdx.x;
    u32 *mi = W.misc + b * 8;
    int T = (int)mi[0]; u32 G = mi[1]; int nsym = (int)mi[2];
    u32 *out = (u32 *)(outb + (size_t)b * out_stride);
    const u32 *ub = usedbits + b * 8;
    const u8 *l6 = W.len6 + (size_t)b * 6 * NSYM;
    __shared__ u32 ws[8];
    __shared__ u32 s_pos, s_tabbits[6];
    // canonical codes, huffman.rs:322-374: sort by (len, sym); code increments, shifts when len grows
    for (int idx = threadIdx.x; idx < T * NSYM; idx += 256) {
        int t = idx / NSYM, s = idx % NSYM;
        u32 code = 0;
        if (s < nsym) {
            const u8 *l = l6 + t * NSYM;
            int mylen = l[s];
            // code(s) = sum over symbols q ordered before s of 2^(mylen - len[q])  (Kraft prefix sum)
            u64 c = 0;
            for (int q = 0; q < nsym; q++) {
                int lq = l[q];
                if (lq < mylen || (lq == mylen && q < s)) c += 1ull << (mylen - lq);
            }
            code = ((u32)mylen << 24) | (u32)c;
        }
        W.codes[((size_t)b * 6 + t) * NSYM + s] = code;
    }
    if (threadIdx.x == 0) {
        u64 p = 0;
        if (emit_header) {                                   // compress_block.rs:34-48
            put_bits(out, p, 0x314159, 24); p += 24;
            put_bits(out, p, 0x265359, 24); p += 24;
            put_bits(out, p, crc[b], 32); p += 32;
            put_bits(out, p, 0, 1); p += 1;
            put_bits(out, p, key[b] & 0xffffff, 24); p += 24;
        }
        // symbol map, rle2_mtf.rs:293-322 / huffman.rs:209-212
        u32 l1 = 0; u32 l2[16];
        for (int i = 0; i < 16; i++) {
            u32 w = (ub[i >> 1] >> ((i & 1) * 16)) & 0xffff;     // bit k of w = byte value 16 i + k present
            l2[i] = __brev(w) >> 16;                             // MSB first: 0x8000 >> k
            if (w) l1 |= 0x8000u >> i;
        }
        put_bits(out, p, l1, 16); p += 16;
        for (int i = 0; i < 16; i++) if (l2[i]) { put_bits(out, p, l2[i], 16); p += 16; }
        put_bits(out, p, (u32)T, 3); p += 3;                     // huffman.rs:216
        put_bits(out, p, G, 15); p += 15;                        // huffman.rs:224
        s_pos = (u32)p;
    }
    // table section sizes (5-bit origin + deltas, huffman.rs:391-438)
    if (threadIdx.x < 6) {
        u32 tb = 0;
        if ((int)threadIdx.x < T) {
            const u8 *l = l6 + threadIdx.x * NSYM;
            tb = 5; int cur = l[0];
            for (int s = 0; s < nsym; s++) { int d = (int)l[s] - cur; cur = l[s]; tb += 2 * (u32)abs(d) + 1; }
        }
        s_tabbits[threadIdx.x] = tb;
    }
    __syncthreads();
    // exclusive scan of selector code lengths
    u32 *sb = W.sbits + (size_t)b * W.sel_stride;
    u32 carry = 0;
    for (u32 g0 = 0; g0 < G; g0 += 256) {
        u32 g = g0 + threadIdx.x;
        u32 v = g < G ? sb[g] : 0, tot;
        u32 ex = block_excl_sum(v, ws, tot);
        if (g < G) sb[g] = carry + ex;
        carry += tot;
        __syncthreads();
    }
    u32 sel_start = s_pos;
    u32 sel_total = carry;
    u32 tab_start = sel_start + carry;
    u32 data_start = tab_start;
    for (int t = 0; t < 6; t++) data_start += s_tabbits[t];
    // table deltas: one thread per table
    if ((int)threadIdx.x < T) {
        u64 p = tab_start;
        for (int t = 0; t < (int)threadIdx.x; t++) p += s_tabbits[t];
        const u8 *l = l6 + threadIdx.x * NSYM;
        int cur = l[0];
        put_bits(out, p, (u32)cur, 5); p += 5;
        for (int s = 0; s < nsym; s++) {
            int d = (int)l[s] - cur; cur = l[s];
            while (d > 0) { put_bits(out, p, 2, 2); p += 2; d--; }
            while (d < 0) { put_bits(out, p, 3, 2); p += 2; d++; }
            p += 1;                                              // terminating 0 bit
        }
    }
    // exclusive scan of group data bits
    u32 *gb = W.gbits + (size_t)b * W.sel_stride;
    carry = 0;
    for (u32 g0 = 0; g0 < G; g0 += 256) {
        u32 g = g0 + threadIdx.x;
        u32 v = g < G ? gb[g] : 0, tot;
        u32 ex = block_excl_sum(v, ws, tot);
        if (g < G) gb[g] = carry + ex;
        carry += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        mi[3] = sel_start; mi[4] = data_start; mi[5] = sel_total;
        u64 total_bits = (u64)data_start + carry;
        // codes can be 17 bits long: a block that does not fit its slot is reported, never written past it
        // (~0 = "does not fit"; the host turns it into BZ2B200_E_CAP, k_huf_emit skips the block)
        bits_out[b] = (total_bits + 7) / 8 + 16 > (u64)out_stride ? ~0ull : total_bits;
    }
}

// ---- k_huf_emit: thread per group -------------------------------------------------------------
__global__ void __launch_bounds__(256) k_huf_emit(const u16 *sym, const u32 *m_in, HufWs W, u32 stride, u8 *outb,
                                                  size_t out_stride, const u64 *bits_out) {
    u32 b = blockIdx.y;
    if (bits_out[b] == ~0ull) return;                           // k_huf_layout: the block does not fit its slot
    u32 m = m_in[b];
    u32 g0 = blockIdx.x * 256;
    u32 G = (m + BZ_GROUP - 1) / BZ_GROUP;
    if (g0 >= G) return;
    __shared__ __align__(16) u16 ssym[256 * BZ_GROUP];
    __shared__ u32 scode[6 * NSYM];
    const u16 *s = sym + (size_t)b * stride;
    u32 first = g0 * BZ_GROUP;
    u32 cnt = min((u32)(256 * BZ_GROUP), m - first);
    for (u32 i = threadIdx.x; i < cnt; i += 256) ssym[i] = s[first + i];
    for (int i = threadIdx.x; i < 6 * NSYM; i += 256) scode[i] = W.codes[(size_t)b * 6 * NSYM + i];
    __syncthreads();
    u32 g = g0 + threadIdx.x;
    if (g >= G) return;
    u32 *out = (u32 *)(outb + (size_t)b * out_stride);
    const u32 *mi = W.misc + b * 8;
    int t = W.sel[(size_t)b * W.sel_stride + g];
    // selector: `pos` ones then a zero (huffman.rs:282-292); sbits holds exclusive offsets
    {
        u32 so = W.sbits[(size_t)b * W.sel_stride + g];
        u32 sn = (g + 1 < G) ? W.sbits[(size_t)b * W.sel_stride + g + 1] : mi[5];
        u32 slen = sn - so;
        put_bits(out, (u64)mi[3] + so, (1u << slen) - 2u, (int)slen);
    }
    u64 p = (u64)mi[4] + W.gbits[(size_t)b * W.sel_stride + g];
    u32 w = (u32)(p >> 5);
    int nacc = (int)(p & 31);
    u64 acc = 0;
    bool firstw = true;
    const u32 *ct = scode + t * NSYM;
    u32 a = threadIdx.x * BZ_GROUP, e = min(a + BZ_GROUP, cnt);
    for (u32 i = a; i < e; i++) {
        u32 c = ct[ssym[i]];
        int l = (int)(c >> 24);
        acc = (acc << l) | (c & 0xffffff);
        nacc += l;
        if (nacc >= 32) {
            u32 word = (u32)(acc >> (nacc - 32));
            nacc -= 32;
            if (firstw) { atomicOr(&out[w], bswap32(word)); firstw = false; }
            else out[w] = bswap32(word);
            w++;
        }
    }
    if (nacc > 0) {
        u32 word = (u32)(acc << (32 - nacc));
        atomicOr(&out[w], bswap32(word));
    }
}

}  // namespace

#define LAUNCH_OK()                                                  \
    do {                                                             \
        ctx->prof_end();                                             \
        cudaError_t e_ = cudaGetLastError();                         \
        if (e_ != cudaSuccess) { ctx->fail("kernel launch", e_, __FILE__, __LINE__); return BZ2B200_E_CUDA; } \
    } while (0)

int bz_huf_batch(bz2b200_ctx *ctx, const Batch &B, const u16 *d_sym, const u32 *d_m, const u32 *d_freq,
                 const u8 *d_used, int emit_header, const u32 *d_crc, const u32 *d_key, HufOut &out) {
    if (B.nblk == 0) return BZ2B200_OK;
    cudaStream_t st = ctx->stream;
    const u64 ne_act = B.total_n;
    u32 maxG = (B.max_n + 1 + BZ_GROUP - 1) / BZ_GROUP;
    u32 sel_stride = ((maxG + 255) / 256) * 256;
    size_t nb = (size_t)B.nblk;
    BZ_CHECK(ctx->d_len6.ensure(nb * 6 * NSYM + nb * NSYM * 8 + 64));
    BZ_CHECK(ctx->d_rfreq.ensure(nb * 6 * NSYM * 4));
    BZ_CHECK(ctx->d_sel.ensure(nb * sel_stride));
    BZ_CHECK(ctx->d_gbits.ensure(nb * sel_stride * 4 * 2));
    BZ_CHECK(ctx->d_hdr.ensure(nb * 6 * NSYM * 4));
    BZ_CHECK(ctx->d_hmisc.ensure(nb * 8 * 4));
    size_t out_stride = (((size_t)B.max_n + B.max_n / 2 + 4096) + 15) / 16 * 16;
    BZ_CHECK(ctx->d_out.ensure(nb * out_stride));
    BZ_CHECK(ctx->d_outbits.ensure(nb * 8));
    HufWs W;
    W.len6 = ctx->d_len6.as<u8>();
    W.tab64 = (u64 *)(W.len6 + ((nb * 6 * NSYM + 15) / 16) * 16);
    W.rfreq = ctx->d_rfreq.as<u32>();
    W.sel = ctx->d_sel.as<u8>();
    W.gbits = ctx->d_gbits.as<u32>();
    W.sbits = W.gbits + nb * sel_stride;
    W.codes = ctx->d_hdr.as<u32>();
    W.misc = ctx->d_hmisc.as<u32>();
    W.sel_stride = sel_stride;
    const u32 *usedbits = (const u32 *)d_used;
    BZ_CHECK(cudaMemsetAsync(W.rfreq, 0, nb * 6 * NSYM * 4, st));
    BZ_CHECK(cudaMemsetAsync(ctx->d_out.p, 0, nb * out_stride, st));
    dim3 gg((maxG + 255) / 256, B.nblk);
    const bool lib = ctx->mode == BZ_MODE_LIBBZ2;
    if (lib) { ctx->prof_begin(K_HUF_INIT_LIBBZ2, ne_act * 2); k_huf_init_libbz2<<<B.nblk, 256, 0, st>>>(d_sym, d_m, usedbits, W, B.stride); LAUNCH_OK(); }
    else { ctx->prof_begin(K_HUF_INIT, (u64)B.nblk * 4096); k_huf_init<<<B.nblk, 256, 0, st>>>(d_m, d_freq, usedbits, W); LAUNCH_OK(); }
    for (int iter = 0; iter < 4; iter++) {                       // huffman.rs:114
        ctx->prof_begin(K_HUF_SELECT, ne_act * 2); k_huf_select<<<gg, 256, 0, st>>>(d_sym, d_m, W, B.stride); LAUNCH_OK();
        if (lib) { ctx->prof_begin(K_HUF_LENGTHS_LIBBZ2, (u64)B.nblk * 6 * 258 * 5); k_huf_lengths_libbz2<<<B.nblk, 192, 0, st>>>(W); LAUNCH_OK(); }
        else { ctx->prof_begin(K_HUF_LENGTHS, (u64)B.nblk * 6 * 258 * 5); k_huf_lengths<<<B.nblk, 192, 0, st>>>(W); LAUNCH_OK(); }
    }
    ctx->prof_begin(K_HUF_GBITS, ne_act * 2); k_huf_gbits<<<gg, 256, 0, st>>>(d_sym, d_m, W, B.stride); LAUNCH_OK();
    ctx->prof_begin(K_HUF_LAYOUT, (u64)B.nblk * 4096); k_huf_layout<<<B.nblk, 256, 0, st>>>(W, usedbits, emit_header, d_crc, d_key, ctx->d_out.as<u8>(), out_stride,
                                         ctx->d_outbits.as<u64>());
    LAUNCH_OK();
    ctx->prof_begin(K_HUF_EMIT, ne_act * 3); k_huf_emit<<<gg, 256, 0, st>>>(d_sym, d_m, W, B.stride, ctx->d_out.as<u8>(), out_stride, ctx->d_outbits.as<u64>()); LAUNCH_OK();
    out.d_out = ctx->d_out.as<u8>();
    out.d_bits = ctx->d_outbits.as<u64>();
    out.out_stride = out_stride;
    out.d_len6 = W.len6;
    out.d_sel = W.sel;
    out.sel_stride = sel_stride;
    out.d_ntab = W.misc;
    return BZ2B200_OK;
}
