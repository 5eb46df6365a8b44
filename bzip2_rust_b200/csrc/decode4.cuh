// decode4.cuh -- entropy decoding of all blocks of a stream, parallel INSIDE a block (included by decode.cu).
//
// Replaces the per-block loop of decompress (reference src/compression/decompress.rs:98-358) and
// rle2_mtf_decode_fast (src/tools/rle2_mtf.rs:191-287).  The earlier versions walked a block with one warp
// (Huffman decode and MTF replay symbol by symbol): 160 ms for 112 blocks, the GPU empty.  A bzip2 block has two
// serial dependences -- where each Huffman code starts, and the MTF list -- and both are cut here:
//   k_dec_header   one warp per block: symbol map, selectors, code lengths -> canonical tables + 10-bit LUTs
//   k_dec_jumps / k_dec_bounds (decode_bounds.cuh)  the bit offset of every 50-symbol group: jump tables over all bit
//                  offsets built in parallel, then one lane per block walks 7 look-ups per group
//   k_dec_syms     one thread per group decodes its 50 symbols from that offset with the group's table
//   k_dec_chunks   one warp per ~1024-symbol chunk (cut where no RUNA/RUNB run is open): bytes the chunk
//                  produces, the PERMUTATION its MTF ranks apply to the list (replayed on the identity), and
//                  for every MTF symbol the start-list position of the value it selects
//   k_dec_chunk_scan one CTA per block: composes the permutations in order -> the MTF list at every chunk
//                  start, and the output offset of every chunk
//   k_dec_expand   position parallel: start list [selected position] per MTF symbol, RUNA/RUNB expansion by a warp
//                  scan -> the BWT string

constexpr int LUTBITS = 10;
constexpr int DCH = 1024;              // nominal symbols per MTF chunk

struct DecTables {                     // per block, global memory
    u16 lut[6][1 << LUTBITS];          // (code length << 9) | symbol; 0 = longer than LUTBITS
    u16 perm[6][258];
    int limit[6][22], base[6][22];
    u8 seq[256];                       // used byte values ascending = initial MTF list
    u32 T, alpha, G, status;           // G = selectors kept (at most sel_stride)
    u32 crc, key;
    u64 data_bit;                      // first bit of the symbol data
    u64 end_bit;                       // bit after the EOB code            (k_dec_bounds)
    u32 nsym, ngroups;                 // symbols incl. EOB, groups in use  (k_dec_bounds)
    u32 nblock, pad;                   // decoded BWT string length (k_dec_chunk_scan); pad = the block's "randomised" bit
};

struct BitBuf {
    const u8 *p; size_t n; size_t byte;      // next byte to load
    u64 buf; int nb;                         // `nb` valid bits, MSB aligned
    __device__ void init(const u8 *in, size_t len, u64 bitpos) {
        p = in; n = len; byte = (size_t)(bitpos >> 3); buf = 0; nb = 0;
        refill();
        int sk = (int)(bitpos & 7);
        buf <<= sk; nb -= sk;
    }
    __device__ __forceinline__ void refill() {
        while (nb <= 32) {
            u32 w;
            if (byte + 4 <= n) {
                w = ((u32)p[byte] << 24) | ((u32)p[byte + 1] << 16) | ((u32)p[byte + 2] << 8) | (u32)p[byte + 3];
            } else {
                w = 0;
                for (int k = 0; k < 4; k++) w = (w << 8) | (byte + k < n ? p[byte + k] : 0);
            }
            byte += 4;
            buf |= (u64)w << (32 - nb);
            nb += 32;
        }
    }
    __device__ __forceinline__ u32 peek(int k) const { return (u32)(buf >> (64 - k)); }     // 1 <= k <= 32
    __device__ __forceinline__ void skip(int k) { buf <<= k; nb -= k; }
    __device__ __forceinline__ u32 get(int k) { if (k == 0) return 0; refill(); u32 v = peek(k); skip(k); return v; }
    __device__ u64 bitpos() const { return (u64)byte * 8 - (u64)nb; }
};

// ---------------------------------------------------------------------------------------------------------
// header: decompress.rs:98-260 + huf_decode_map (:426-486)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_dec_header(const u8 *in, size_t n, const u64 *start_bits, u8 *sel_all,
                                                   u32 sel_stride, DecTables *tabs) {
    u32 b = blockIdx.x;
    __shared__ u8 len[6][258];
    __shared__ u16 perm[6][258];
    __shared__ int limit[6][22], base[6][22];
    __shared__ u16 lut[6][1 << LUTBITS];
    __shared__ u8 seq[256];
    __shared__ int s_T, s_alpha, s_status;
    __shared__ u32 s_G, s_crc, s_key, s_rand;
    __shared__ u64 s_data, s_selbit, s_lenbit;
    __shared__ u32 s_perm[32];
    const int lane = threadIdx.x;
    u8 *sel = sel_all + (size_t)b * sel_stride;
    for (int i = lane; i < 256; i += 32) seq[i] = 0;
    __syncwarp();
    if (lane == 0) {
        BitBuf br;
        s_status = 0;
        br.init(in, n, start_bits[b] + 48);
        { u32 hi16 = br.get(16); u32 lo16 = br.get(16); s_crc = (hi16 << 16) | lo16; }
        s_rand = br.get(1);                                     // legacy randomised block (decode.cu k_derandomize); encoders write 0 (compress_block.rs:41)
        s_key = br.get(24);
        u32 l1 = br.get(16);
        int nused = 0;
        for (int i = 0; i < 16; i++) if (l1 & (0x8000u >> i)) {
            u32 l2 = br.get(16);
            for (int j = 0; j < 16; j++) if (l2 & (0x8000u >> j)) seq[nused++] = (u8)(i * 16 + j);
        }
        if (nused == 0 && !s_status) s_status = 2;
        int alpha = nused + 2;
        int T = (int)br.get(3);
        u32 G = br.get(15);                                     // any 1..32767 (libbz2 1.0.8 ignores those past its 18002)
        if (!s_status && (T < 2 || T > 6 || G < 1)) s_status = 3;
        s_T = T; s_alpha = alpha; s_G = G; s_selbit = br.bitpos();
    }
    __syncwarp();
    // ---- selectors (decompress.rs:140-203): G unary numbers (j ones, then a zero), each an index into a move-to-front
    // list of the table numbers.  Selector g ends at the g-th zero bit, so the warp finds them 1024 bits at a time
    // (zeros per word, one scan); the MTF list has 6 entries, so a lane replays its share of the numbers on the
    // identity list, the 32 results are composed in order, and the lane replays its share again from its true list.
    // All G are scanned and checked (j < T), the code lengths start after the last; only the first Gs = min(G,
    // sel_stride) are kept.  A block has at most max_block + 1 symbols, so it never needs more groups than that: one that
    // runs past the kept selectors fails in k_dec_bounds, where libbz2 fails it too (18002 kept, more than 900 000 bytes).
    if (s_status == 0) {
        const int T = s_T;
        const u32 G = s_G, Gs = min(G, sel_stride);
        const u32 *wsrc = (const u32 *)in;
        const u64 lastw = (u64)((n + 3) / 4) - 1;
        u32 found = 0, carry = 0;
        bool bad = false;
        for (u64 c0 = s_selbit; found < G; c0 += 1024) {
            const u64 bp = c0 + 32u * (u32)lane;
            const u64 wi = bp >> 5;
            const u32 hi = __byte_perm(__ldg(wsrc + min(wi, lastw)), 0, 0x0123), lo = __byte_perm(__ldg(wsrc + min(wi + 1, lastw)), 0, 0x0123);
            const u32 w = __funnelshift_l(lo, hi, (u32)(bp & 31));
            u32 m = ~w;                                         // set bits: the zeros, MSB first
            const u32 nz = __popc(m);
            const u32 inc = warp_incl_sum(nz);
            const u32 tr = m ? (u32)(__ffs(m) - 1) : 32u;       // ones at the end of this word
            u32 ptr = __shfl_up_sync(0xffffffffu, tr, 1);
            if (lane == 0) ptr = carry;
            u32 gidx = found + inc - nz;
            int lastpos = -1;
            while (m && gidx < G) {
                const int pos = __clz(m);
                const u32 j = lastpos < 0 ? ptr + (u32)pos : (u32)(pos - lastpos - 1);
                if (j >= (u32)T) bad = true;
                if (gidx < Gs) sel[gidx] = (u8)j;
                if (gidx == G - 1) s_lenbit = bp + (u64)pos + 1;
                gidx++; lastpos = pos;
                m &= ~(0x80000000u >> pos);
            }
            if (nz == 0 && gidx < G) bad = true;                // 32 ones in a row inside the selectors
            carry = __shfl_sync(0xffffffffu, tr, 31);
            found += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (__any_sync(0xffffffffu, bad)) { if (lane == 0) s_status = 4; }
        __syncwarp();
        if (s_status == 0) {
            const u32 per = (Gs + 31) / 32;
            const u32 g0 = min(Gs, (u32)lane * per), g1 = min(Gs, g0 + per);
            u32 Lp = 0x543210u;                                 // nibble k = table number at list position k
            for (u32 g = g0; g < g1; g++) {
                const u32 j4 = 4u * sel[g];
                const u32 v = (Lp >> j4) & 15u, low = Lp & ((1u << j4) - 1u);
                Lp = (Lp & ~((16u << j4) - 1u)) | (low << 4) | v;
            }
            s_perm[lane] = Lp;
            __syncwarp();
            if (lane == 0) {                                    // start list of every lane: compose in order
                u32 S = 0x543210u;
                for (int k = 0; k < 32; k++) {
                    const u32 F = s_perm[k];
                    s_perm[k] = S;
                    u32 N = 0;
                    for (int q = 0; q < 6; q++) N |= ((S >> (4u * ((F >> (4 * q)) & 15u))) & 15u) << (4 * q);
                    S = N;
                }
            }
            __syncwarp();
            Lp = s_perm[lane];
            for (u32 g = g0; g < g1; g++) {
                const u32 j4 = 4u * sel[g];
                const u32 v = (Lp >> j4) & 15u, low = Lp & ((1u << j4) - 1u);
                Lp = (Lp & ~((16u << j4) - 1u)) | (low << 4) | v;
                sel[g] = (u8)v;
            }
        }
    }
    __syncwarp();
    if (lane == 0 && s_status == 0) {
        const int T = s_T, alpha = s_alpha;
        BitBuf br;
        br.init(in, n, s_lenbit);
        for (int t = 0; t < T && !s_status; t++) {             // code lengths (decompress.rs:216-260)
            int c = (int)br.get(5);
            for (int s = 0; s < alpha && !s_status; s++) {
                for (;;) {
                    if (c < 1 || c > 20) { s_status = 5; break; }
                    if (!br.get(1)) break;
                    c += br.get(1) ? -1 : 1;
                }
                len[t][s] = (u8)c;
            }
        }
        s_data = br.bitpos();
    }
    __syncwarp();
    const int T = s_T, alpha = s_alpha;
    if (s_status == 0) {
        if (lane < T) {
            int t = lane;
            int mn = 32, mx = 0;
            for (int s = 0; s < alpha; s++) { int l = len[t][s]; mn = min(mn, l); mx = max(mx, l); }
            int pp = 0;
            for (int l = mn; l <= mx; l++) for (int s = 0; s < alpha; s++) if (len[t][s] == l) perm[t][pp++] = (u16)s;
            int cnt[22];
            for (int l = 0; l < 22; l++) cnt[l] = 0;
            for (int s = 0; s < alpha; s++) cnt[len[t][s]]++;
            int code = 0, idx = 0;
            for (int l = 1; l <= 20; l++) {
                base[t][l] = idx - code; code += cnt[l]; idx += cnt[l]; limit[t][l] = code - 1; code <<= 1;
            }
            for (int l = 1; l <= 20; l++) if (l > mx) limit[t][l] = 0x7fffffff;
            limit[t][0] = -1; limit[t][21] = 0x7fffffff; base[t][0] = 0; base[t][21] = 0;
        }
        for (int i = lane; i < 6 * (1 << LUTBITS); i += 32) (&lut[0][0])[i] = 0;
        __syncwarp();
        for (int t = 0; t < T; t++) {
            for (int pi = lane; pi < alpha; pi += 32) {
                int s = perm[t][pi];
                int l = len[t][s];
                if (l <= LUTBITS) {
                    int code = pi - base[t][l];
                    int lo = code << (LUTBITS - l), hi = lo + (1 << (LUTBITS - l));
                    u16 e = (u16)((l << 9) | s);
                    for (int k = lo; k < hi && k < (1 << LUTBITS); k++) lut[t][k] = e;
                }
            }
        }
    }
    __syncwarp();
    DecTables *o = tabs + b;
    for (int i = lane; i < 6 * (1 << LUTBITS); i += 32) (&o->lut[0][0])[i] = (&lut[0][0])[i];
    for (int i = lane; i < 6 * 258; i += 32) (&o->perm[0][0])[i] = (&perm[0][0])[i];
    for (int i = lane; i < 6 * 22; i += 32) { (&o->limit[0][0])[i] = (&limit[0][0])[i]; (&o->base[0][0])[i] = (&base[0][0])[i]; }
    for (int i = lane; i < 256; i += 32) o->seq[i] = seq[i];
    if (lane == 0) {
        o->T = (u32)T; o->alpha = (u32)alpha; o->G = min(s_G, sel_stride); o->status = (u32)s_status; o->crc = s_crc; o->key = s_key;
        o->data_bit = s_data; o->end_bit = 0; o->nsym = 0; o->ngroups = 0; o->nblock = 0; o->pad = s_rand;
    }
}

// shared copy of the decode tables of one block (all threads of the CTA call)
struct SmemTables {
    u16 lut[6][1 << LUTBITS];
    u16 perm[6][258];
    int limit[6][22], base[6][22];
};
__device__ __forceinline__ void load_tables(SmemTables &s, const DecTables *g) {
    for (int i = threadIdx.x; i < 6 * (1 << LUTBITS) / 2; i += blockDim.x) ((u32 *)&s.lut[0][0])[i] = ((const u32 *)&g->lut[0][0])[i];
    for (int i = threadIdx.x; i < 6 * 258 / 2; i += blockDim.x) ((u32 *)&s.perm[0][0])[i] = ((const u32 *)&g->perm[0][0])[i];
    for (int i = threadIdx.x; i < 6 * 22; i += blockDim.x) { (&s.limit[0][0])[i] = (&g->limit[0][0])[i]; (&s.base[0][0])[i] = (&g->base[0][0])[i]; }
}

// one Huffman symbol with table t; returns the symbol, or -1 on a malformed code.  R = BitBuf.
template <class R>
__device__ __forceinline__ int decode_one(R &br, const SmemTables &s, int t, int alpha) {
    br.refill();
    u16 e = s.lut[t][br.peek(LUTBITS)];
    if (e) { br.skip(e >> 9); return (int)(e & 511u); }
    int l = LUTBITS + 1;
    int code = (int)br.peek(l);
    while (l <= 20 && code > s.limit[t][l]) { l++; code = (int)br.peek(l); }
    if (l > 20) return -1;
    int pi = code + s.base[t][l];
    if (pi < 0 || pi >= alpha) return -1;
    br.skip(l);
    return (int)s.perm[t][pi];
}

// ---------------------------------------------------------------------------------------------------------
// symbols: one thread per 50-symbol group
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_dec_syms(const u8 *in, size_t n, const u8 *sel_all, u32 sel_stride,
                                                  const DecTables *tabs, const u32 *gbit_all, u16 *sym_all, u32 sym_stride) {
    u32 b = blockIdx.y;
    const DecTables *tb = tabs + b;
    if (tb->status) return;
    const u32 ng = tb->ngroups;
    if (blockIdx.x * 128 >= ng) return;
    __shared__ SmemTables st;
    load_tables(st, tb);
    __syncthreads();
    u32 g = blockIdx.x * 128 + threadIdx.x;
    if (g >= ng) return;
    const int alpha = (int)tb->alpha;
    const int t = sel_all[(size_t)b * sel_stride + g];
    BitBuf br;
    br.init(in, n, tb->data_bit + gbit_all[(size_t)b * sel_stride + g]);
    u16 *so = sym_all + (size_t)b * sym_stride + (size_t)g * 50;
    u32 left = tb->nsym - g * 50;
    int cnt = (int)min(50u, left);
    for (int k = 0; k < cnt; k++) {
        int s = decode_one(br, st, t, alpha);
        so[k] = (u16)(s < 0 ? alpha - 1 : s);                  // k_dec_bounds already validated every code
    }
}

// ---------------------------------------------------------------------------------------------------------
// inverse MTF + RUNA/RUNB (rle2_mtf.rs:191-287) by chunks
// ---------------------------------------------------------------------------------------------------------
// chunk c covers symbols [cut(c), cut(c+1)): cut(0) = 0, cut(c) = first index >= c*DCH holding a non-run symbol
// (a run is at most 20 symbols long), cut(nch) = nsym.
__device__ __forceinline__ u32 chunk_cut(const u16 *sym, u32 nsym, u32 c, u32 nch) {
    if (c == 0) return 0;
    if (c >= nch) return nsym;
    u32 i = c * DCH;
    while (i < nsym && sym[i] <= 1) i++;
    return i;
}

// Pass 1, one warp per chunk: the chunk's ranks replayed on the IDENTITY list.  Results: the permutation the chunk
// applies (perm_out[i] = start-list position of the value that ends at position i), the number of bytes it produces,
// and for every MTF symbol the start-list position of the value it selects (vid).  Once the start list of the chunk
// is known (k_dec_chunk_scan) its bytes are slist[vid]: pass 2 (k_dec_expand) is position parallel.
__global__ void __launch_bounds__(256) k_dec_chunks(const DecTables *tabs, const u16 *sym_all, u32 sym_stride,
                                                    u8 *lists, u32 *ccount, u32 ch_stride, u8 *vid_all, u32 max_block) {
    const u32 b = blockIdx.y;
    const DecTables *tb = tabs + b;
    if (tb->status) return;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const u32 nsym = tb->nsym;
    const u32 nch = (nsym + DCH - 1) / DCH;
    const u32 c = blockIdx.x * 8 + w;
    if (c >= nch) return;
    const u16 *sym = sym_all + (size_t)b * sym_stride;
    u8 *vid = vid_all + (size_t)b * sym_stride;
    const u32 eob = tb->alpha - 1;
    u32 i = chunk_cut(sym, nsym, c, nch);
    const u32 e = chunk_cut(sym, nsym, c + 1, nch);
    u8 *lst = lists + ((size_t)b * ch_stride + c) * 256;
    // MTF list across the warp: positions 0..31 one per lane, 32..255 as 7 bytes per lane (low 56 bits)
    u32 fw = (u32)lane; u64 tl = 0;
#pragma unroll
    for (int k = 0; k < 7; k++) tl |= (u64)(32 + 7 * lane + k) << (8 * k);
    const u64 LOW7 = 0x00FFFFFFFFFFFFFFull;
    u32 nblk = 0;                             // produced bytes
    u32 runlen = 0, runbit = 1;
    bool bad = false;
    for (u32 i0 = i; i0 < e && !bad; i0 += 32) {
        const int cnt = (int)min(32u, e - i0);
        const u32 mine = lane < cnt ? (u32)sym[i0 + lane] : 0u;
        u32 myvid = 0;
        for (int q = 0; q < cnt; q++) {
            const u32 s = __shfl_sync(0xffffffffu, mine, q);
            if (s <= 1) { runlen += runbit << s; runbit <<= 1; if (runlen > max_block) { bad = true; break; } continue; }
            if (runlen) {
                if (nblk + runlen > max_block) { bad = true; break; }
                nblk += runlen; runlen = 0;
            }
            runbit = 1;
            if (s == eob) break;
            const u32 pos = s - 1;
            u32 v;
            const u32 up = __shfl_up_sync(0xffffffffu, fw, 1);
            if (pos < 32) {
                v = __shfl_sync(0xffffffffu, fw, (int)pos);
                if ((u32)lane <= pos) fw = lane ? up : v;
            } else {
                int Lh = (int)((pos - 32) / 7), kb = (int)((pos - 32) % 7);
                u32 mb = (u32)(tl >> (8 * kb)) & 0xffu;
                v = __shfl_sync(0xffffffffu, mb, Lh);
                u32 carry = __shfl_sync(0xffffffffu, fw, 31);
                u32 top = (u32)(tl >> 48) & 0xffu;
                u32 incoming = __shfl_up_sync(0xffffffffu, top, 1);
                if (lane == 0) incoming = carry;
                if (lane < Lh) tl = ((tl << 8) | incoming) & LOW7;
                else if (lane == Lh) {
                    u64 lowmask = kb ? ((1ull << (8 * kb)) - 1) : 0ull;
                    u64 keepmask = (~((1ull << (8 * (kb + 1))) - 1)) & LOW7;
                    tl = (tl & keepmask) | (((tl & lowmask) << 8) | incoming);
                }
                fw = lane ? up : v;
            }
            if (lane == q) myvid = v;
            nblk++;
            if (nblk > max_block) { bad = true; break; }
        }
        if (lane < cnt) vid[i0 + lane] = (u8)myvid;
    }
    if (runlen && !bad) {                     // the run that ends exactly at the cut
        if (nblk + runlen > max_block) bad = true;
        else nblk += runlen;
    }
    lst[lane] = (u8)fw;
#pragma unroll
    for (int k = 0; k < 7; k++) lst[32 + 7 * lane + k] = (u8)(tl >> (8 * k));
    if (lane == 0) ccount[(size_t)b * ch_stride + c] = bad ? 0xFFFFFFFFu : nblk;
}

// Pass 2, one warp per chunk, 32 symbols per step: an MTF symbol yields the byte slist[vid]; a RUNA/RUNB symbol that is
// the k-th of its run yields (s + 1) << k copies of the list front, i.e. of the byte of the last MTF symbol before the
// run (rle2_mtf.rs:223-262) -- counts and sources are lane-local, the output offsets one warp scan.
__global__ void __launch_bounds__(256) k_dec_expand(const DecTables *tabs, const u16 *sym_all, u32 sym_stride,
                                                    const u8 *lists, const u32 *coff, u32 ch_stride, const u8 *vid_all,
                                                    u8 *tt_all, u32 stride) {
    const u32 b = blockIdx.y;
    const DecTables *tb = tabs + b;
    if (tb->status) return;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const u32 nsym = tb->nsym;
    const u32 nch = (nsym + DCH - 1) / DCH;
    const u32 c = blockIdx.x * 8 + w;
    __shared__ u8 slist[8][256];
    if (c >= nch) return;
    const u16 *sym = sym_all + (size_t)b * sym_stride;
    const u8 *vid = vid_all + (size_t)b * sym_stride;
    const u32 eob = tb->alpha - 1;
    const u32 i = chunk_cut(sym, nsym, c, nch);
    const u32 e = chunk_cut(sym, nsym, c + 1, nch);
    const u8 *lst = lists + ((size_t)b * ch_stride + c) * 256;
    for (int k = lane; k < 256; k += 32) slist[w][k] = lst[k];
    __syncwarp();
    u8 *tt = tt_all + (size_t)b * stride;
    u32 out = coff[(size_t)b * ch_stride + c];
    u32 carry_k = 0;                          // run symbols at the end of the previous step (the run goes on)
    u32 carry_front = 0;                      // start-list position of the list front at the start of the step
    const u32 lt = (1u << lane) - 1u;
    for (u32 i0 = i; i0 < e; i0 += 32) {
        const bool valid = i0 + lane < e;
        const u32 s = valid ? (u32)sym[i0 + lane] : 0xffffu;
        const bool isrun = valid && s <= 1;
        const bool ismtf = valid && s > 1 && s != eob;
        const u32 myvid = ismtf ? (u32)vid[i0 + lane] : 0u;
        const u32 mtfmask = __ballot_sync(0xffffffffu, ismtf);
        const u32 below = mtfmask & lt;
        const int src = below ? 31 - __clz(below) : -1;
        u32 fv = __shfl_sync(0xffffffffu, myvid, src < 0 ? 0 : src);
        if (src < 0) fv = carry_front;
        u32 cntb = ismtf ? 1u : 0u;
        if (isrun) {
            const u32 k = src < 0 ? carry_k + (u32)lane : (u32)(lane - src - 1);
            cntb = (s + 1u) << min(k, 24u);               // pass 1 bounded every run by the block size
        }
        u32 inc = cntb;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { u32 t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
        const u32 off = out + inc - cntb;
        const u32 byte = slist[w][ismtf ? myvid : fv];
        if (ismtf) tt[off] = (u8)byte;
        else if (isrun && cntb <= 8) { for (u32 q = 0; q < cntb; q++) tt[off + q] = (u8)byte; }
        u32 longmask = __ballot_sync(0xffffffffu, isrun && cntb > 8);
        while (longmask) {                                 // long runs: the whole warp fills
            const int L = __ffs(longmask) - 1;
            longmask &= longmask - 1;
            const u32 lo = __shfl_sync(0xffffffffu, off, L), ln = __shfl_sync(0xffffffffu, cntb, L);
            const u32 bv = __shfl_sync(0xffffffffu, byte, L);
            for (u32 q = lane; q < ln; q += 32) tt[lo + q] = (u8)bv;
        }
        out += __shfl_sync(0xffffffffu, inc, 31);
        // state for the next step
        if (mtfmask) {
            const int last = 31 - __clz(mtfmask);
            carry_front = __shfl_sync(0xffffffffu, myvid, last);
            const u32 runmask = __ballot_sync(0xffffffffu, isrun);
            carry_k = (u32)__popc(runmask & ~((2u << last) - 1u));      // run symbols after the last MTF symbol
        } else {
            carry_k += (u32)__popc(__ballot_sync(0xffffffffu, isrun));
        }
    }
}

// one CTA per block: lists[c] := MTF list at the start of chunk c (it holds chunk c's permutation on entry),
// coff[c] = output offset of chunk c, nblock = total
__global__ void __launch_bounds__(256) k_dec_chunk_scan(DecTables *tabs, u8 *lists, const u32 *ccount, u32 *coff,
                                                        u32 ch_stride, u32 max_block) {
    const u32 b = blockIdx.x;
    DecTables *tb = tabs + b;
    if (tb->status) return;
    const u32 nch = (tb->nsym + DCH - 1) / DCH;
    __shared__ u8 cur[2][256];
    const int i = threadIdx.x;
    cur[0][i] = tb->seq[i];
    __syncthreads();
    u8 *L = lists + (size_t)b * ch_stride * 256;
    int ph = 0;
    u32 pnext = nch ? L[i] : 0;
    for (u32 c = 0; c < nch; c++) {
        u32 p = pnext;                                           // position (in the start list) of what ends at i
        if (c + 1 < nch) pnext = L[(size_t)(c + 1) * 256 + i];   // next permutation is independent of the state
        u8 mine = cur[ph][i];
        L[(size_t)c * 256 + i] = mine;                           // start list of chunk c
        cur[ph ^ 1][i] = cur[ph][p];
        __syncthreads();
        ph ^= 1;
    }
    if (i == 0) {
        u64 sum = 0; u32 status = 0;
        for (u32 c = 0; c < nch; c++) {
            u32 v = ccount[(size_t)b * ch_stride + c];
            coff[(size_t)b * ch_stride + c] = (u32)sum;
            if (v == 0xFFFFFFFFu) { status = 9; break; }
            sum += v;
            if (sum > max_block) { status = 9; break; }
        }
        tb->nblock = (u32)sum;
        if (!status && (sum == 0 || tb->key >= sum)) status = 10;
        if (status) tb->status = status;
    }
}
