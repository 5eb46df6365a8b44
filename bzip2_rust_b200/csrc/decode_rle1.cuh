// decode_rle1.cuh -- inverse RLE1 in parallel (included by decode.cu inside its namespace).
//
// k_rle1_inv: rle1_decode (reference src/tools/rle1.rs:267-316) with the standard run semantics, exact at block
//   tails.  The sequential rule "the byte after four equal bytes is a repeat count" is a 5-state automaton driven
//   only by eq[i] = (r[i]==r[i-1]): state = run length so far (0 = just consumed a count).  Transition functions
//   compose associatively, so a scan over 15-bit packed functions gives every byte's state; a second scan of the
//   output sizes gives offsets.  One CTA walks one block tile by tile (carry in registers), blocks run concurrently.

// ---- parallel inverse RLE1 ------------------------------------------------------------------------------
// packed transition function: 5 states x 3 bits; F(s) = (f >> (3 s)) & 7
__device__ __forceinline__ u32 fn_compose(u32 f, u32 g) {       // apply f, then g
    u32 r = 0;
#pragma unroll
    for (int s = 0; s < 5; s++) { u32 m = (f >> (3 * s)) & 7u; r |= ((g >> (3 * m)) & 7u) << (3 * s); }
    return r;
}
constexpr u32 FN_ID = (0u) | (1u << 3) | (2u << 6) | (3u << 9) | (4u << 12);
constexpr u32 FN_EQ = (1u) | (2u << 3) | (3u << 6) | (4u << 9) | (0u << 12);    // 0->1 1->2 2->3 3->4 4->0(count)
constexpr u32 FN_NE = (1u) | (1u << 3) | (1u << 6) | (1u << 9) | (0u << 12);    // 0..3->1 4->0(count)

// WRITE = 0: outlen[b] = decoded length, or RLE1_OPEN (common.cuh) for a block that ends with four equal bytes and no
// count byte (libbz2 then takes a count from past the block's end and reports the block corrupt).  WRITE = 1: bytes
// written at out + outoff[b], except for a block the count pass found open (no room is reserved for it).
template <int WRITE>
__global__ void __launch_bounds__(256) k_rle1_inv(const u8 *blk, const u32 *len, u32 stride, u64 *outlen, const u64 *outoff,
                                                  u8 *out) {
    u32 b = blockIdx.x;
    if (WRITE && outlen[b] == RLE1_OPEN) return;
    const u8 *r = blk + (size_t)b * stride;
    u32 n = len[b];
    u8 *o = WRITE ? out + outoff[b] : nullptr;
    __shared__ u32 wfn[8];
    __shared__ u32 wsum[8];
    __shared__ u32 s_state;      // automaton state after the previous tile
    __shared__ u64 s_off;        // output bytes before this tile
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_state = 0; s_off = 0; }
    __syncthreads();
    constexpr int PT = 32;                                 // bytes per thread: the tile loop is a chain of CTA-wide scans,
                                                           // 8 KB tiles keep it at ~110 steps per block (8: 440 steps, 2.4 -> 1.x ms)
    for (u32 base = 0; base < n; base += 256 * PT) {
        u32 i0 = base + threadIdx.x * PT;
        u8 c[PT + 1];
        c[0] = (i0 > 0 && i0 - 1 < n) ? r[i0 - 1] : 0;
        if (i0 + PT <= n) {                                // blocks start 16-byte aligned (stride is a multiple of 4096)
            const uint4 *q4 = (const uint4 *)(r + i0);
#pragma unroll
            for (int v = 0; v < PT / 16; v++) {
                const uint4 q = q4[v];
                const u32 wv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int k = 0; k < 16; k++) c[16 * v + k + 1] = (u8)(wv[k >> 2] >> (8 * (k & 3)));
            }
        } else {
#pragma unroll
            for (int k = 0; k < PT; k++) c[k + 1] = (i0 + k < n) ? r[i0 + k] : 0;
        }
        // thread function over its bytes
        u32 f = FN_ID;
#pragma unroll
        for (int k = 0; k < PT; k++) {
            if (i0 + k < n) {
                bool eq = (i0 + k > 0) && c[k + 1] == c[k];
                f = fn_compose(f, eq ? FN_EQ : FN_NE);
            }
        }
        // exclusive scan of functions across the CTA
        u32 inc = f;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            u32 tpre = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc = fn_compose(tpre, inc);
        }
        if (lane == 31) wfn[w] = inc;
        __syncthreads();
        u32 pre = FN_ID;
        for (int k = 0; k < w; k++) pre = fn_compose(pre, wfn[k]);
        u32 excl = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) excl = FN_ID;
        u32 before = fn_compose(pre, excl);                // function from tile start to just before this thread
        u32 st = (before >> (3 * s_state)) & 7u;           // state before this thread's first byte
        // walk own bytes: classify, size
        u32 sz = 0;
        u32 st0 = st;
#pragma unroll
        for (int k = 0; k < PT; k++) {
            if (i0 + k < n) {
                bool eq = (i0 + k > 0) && c[k + 1] == c[k];
                if (st == 4) { sz += c[k + 1]; st = 0; }   // repeat count
                else { sz += 1; st = (st >= 1 && eq) ? st + 1 : 1; }
            }
        }
        // exclusive sum of sizes
        u32 sinc = sz;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { u32 tv = __shfl_up_sync(0xffffffffu, sinc, d); if (lane >= d) sinc += tv; }
        if (lane == 31) wsum[w] = sinc;
        __syncthreads();
        u32 wpre = 0, tot = 0;
        for (int k = 0; k < 8; k++) { if (k < w) wpre += wsum[k]; tot += wsum[k]; }
        u64 off = s_off + wpre + (sinc - sz);
        if (WRITE) {
            st = st0;
#pragma unroll
            for (int k = 0; k < PT; k++) {
                if (i0 + k < n) {
                    bool eq = (i0 + k > 0) && c[k + 1] == c[k];
                    if (st == 4) {
                        u32 cntv = c[k + 1]; u8 v = c[k];
                        // v is the run byte only if the previous byte was a run byte, which it is when st == 4
                        for (u32 q = 0; q < cntv; q++) o[off + q] = v;
                        off += cntv; st = 0;
                    } else { o[off++] = c[k + 1]; st = (st >= 1 && eq) ? st + 1 : 1; }
                }
            }
        }
        // carry to the next tile: state after the tile's last byte, total size
        u32 tile_fn = FN_ID;
        for (int k = 0; k < 8; k++) tile_fn = fn_compose(tile_fn, wfn[k]);
        __syncthreads();
        if (threadIdx.x == 0) { s_state = (tile_fn >> (3 * s_state)) & 7u; s_off += tot; }
        __syncthreads();
    }
    if (!WRITE && threadIdx.x == 0) outlen[b] = s_state == 4 ? RLE1_OPEN : s_off;
}
