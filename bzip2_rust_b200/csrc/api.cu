// api.cu -- C ABI of libbz2b200 (include/bz2b200.h): context, staging, stage seams.
#include "common.cuh"
#include <atomic>
#include <string.h>
#include <new>

// every grow-only device buffer of a context
static void release_device_buffers(bz2b200_ctx *c) {
    DevBuf *all[] = {&c->d_T, &c->d_len, &c->d_crc, &c->d_SA, &c->d_SA2, &c->d_RANK, &c->d_F, &c->d_KEYA, &c->d_KEYB, &c->d_VALA,
                     &c->d_VALB, &c->d_thist, &c->d_tagg, &c->d_cnt, &c->d_bwt, &c->d_key, &c->d_mtfstate, &c->d_chunkrec, &c->d_R,
                     &c->d_sym, &c->d_m, &c->d_freq, &c->d_used, &c->d_agg2, &c->d_len6, &c->d_rfreq, &c->d_sel, &c->d_gbits,
                     &c->d_hdr, &c->d_bitoff, &c->d_out, &c->d_outbits, &c->d_hmisc, &c->d_in, &c->d_runflag, &c->d_misc,
                     &c->d_stream, &c->d_dec1, &c->d_dec2, &c->d_dec3, &c->d_dwin, &c->d_ddec[0], &c->d_ddec[1]};
    for (DevBuf *b : all) b->release();
}

namespace {
constexpr int DEV_SLOTS = 64;                // devices beyond share a slot: the lock is then merely taken more often
std::atomic<int> g_ctx_on_dev[DEV_SLOTS];
std::mutex g_dev_lock[DEV_SLOTS];
}  // namespace
int bz_contexts_on_device(int device) { return g_ctx_on_dev[device % DEV_SLOTS].load(); }
std::mutex &bz_device_lock(int device) { return g_dev_lock[device % DEV_SLOTS]; }

bz2b200_ctx::~bz2b200_ctx() {
    g_ctx_on_dev[device % DEV_SLOTS]--;
    cudaSetDevice(device);
    release_device_buffers(this);
    h_stage.release(); h_small.release(); h_out.release();
    for (int i = 0; i < 2; i++) { h_dstage[i].release(); h_dpiece[i].release(); h_rec[i].release(); }
    for (int i = 0; i < 8; i++) if (ev[i]) cudaEventDestroy(ev[i]);
    for (int i = 0; i < 2; i++) if (ev_dec[i]) cudaEventDestroy(ev_dec[i]);
    for (int i = 0; i < 2; i++) { if (ev_rec[i]) cudaEventDestroy(ev_rec[i]); if (ev_dpiece[i]) cudaEventDestroy(ev_dpiece[i]); }
    if (s_hi) cudaStreamDestroy(s_hi);
    for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : up_ev) cudaEventDestroy(e);
    if (s_up) cudaStreamDestroy(s_up);
    if (s_down) cudaStreamDestroy(s_down);
    if (stream) cudaStreamDestroy(stream);
}

extern "C" {

const char *bz2b200_version(void) { return "bz2b200 0.2 (sm_100a)"; }

int bz2b200_create(int device, bz2b200_ctx **out) {
    BZ_API_TRY
    if (!out) return BZ2B200_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return BZ2B200_E_CUDA;   // no CPU fallback
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) return BZ2B200_E_CUDA; }
    if (device >= ndev) return BZ2B200_E_ARG;
    bz2b200_ctx *ctx = new (std::nothrow) bz2b200_ctx();
    if (!ctx) return BZ2B200_E_NOMEM;
    ctx->device = device;
    g_ctx_on_dev[device % DEV_SLOTS]++;      // the destructor counts it down
    if (cudaSetDevice(device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return BZ2B200_E_CUDA;
    }
    for (int i = 0; i < 8; i++) cudaEventCreate(&ctx->ev[i]);
    cudaEventCreate(&ctx->ev_total[0]);
    cudaEventCreate(&ctx->ev_total[1]);
    *out = ctx;
    return BZ2B200_OK;
    BZ_API_CATCH
}
void bz2b200_destroy(bz2b200_ctx *ctx) { delete ctx; }
int bz2b200_trim(bz2b200_ctx *ctx) {
    if (!ctx) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    cudaStreamSynchronize(ctx->stream);
    release_device_buffers(ctx);
    for (int i = 0; i < 2; i++) ctx->h_rec[i].release();
    ctx->shard = ShardPlan();                                    // a pending shard plan pointed into the freed scans
    return BZ2B200_OK;
}
const char *bz2b200_last_error(const bz2b200_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
uint64_t bz2b200_launch_count(const bz2b200_ctx *ctx) { return ctx ? ctx->launches : 0; }
void bz2b200_set_timing(bz2b200_ctx *ctx, int on) { if (ctx) { ctx->timing = on != 0; ctx->prof_level = on; } }
int bz2b200_kernel_stats(bz2b200_ctx *ctx, int idx, char name[64], double *ms, uint64_t *launches, uint64_t *bytes) {
    BZ_API_TRY
    if (!ctx || idx < 0 || idx >= K_COUNT || !name || !ms || !launches || !bytes) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->prof_collect();
    strncpy(name, kKernelNames[idx], 63); name[63] = 0;
    *ms = ctx->kstat[idx].ms; *launches = ctx->kstat[idx].launches; *bytes = ctx->kstat[idx].bytes;
    return BZ2B200_OK;
    BZ_API_CATCH
}
void bz2b200_reset_kernel_stats(bz2b200_ctx *ctx) {
    if (!ctx) return;
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->prof_collect();
    for (int i = 0; i < K_COUNT; i++) ctx->kstat[i] = KStat();
}
int bz2b200_get_timing(const bz2b200_ctx *ctx, float ms[8]) {
    BZ_API_TRY
    if (!ctx || !ms) return BZ2B200_E_ARG;
    memcpy(ms, ctx->stage_ms, sizeof(float) * 8);
    return BZ2B200_OK;
    BZ_API_CATCH
}
int bz2b200_get_bwt_stats(const bz2b200_ctx *ctx, uint64_t st[8]) {
    BZ_API_TRY
    if (!ctx || !st) return BZ2B200_E_ARG;
    memcpy(st, ctx->bwt_stats, sizeof(u64) * 8);
    return BZ2B200_OK;
    BZ_API_CATCH
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// staging: host blocks -> fixed-stride device batch
// ------------------------------------------------------------------------------------------
static int bitlen32(u32 v) { int b = 0; while (v) { b++; v >>= 1; } return b; }

static void batch_geometry(Batch &B, int nblk, u32 max_n) {
    B.nblk = nblk;
    B.max_n = max_n;
    B.stride = ((max_n + 64 + BZ_TILE - 1) / BZ_TILE) * BZ_TILE;
    B.tiles = B.stride / BZ_TILE;
    B.nbits = bitlen32(max_n ? max_n - 1 : 0);
    if (B.nbits < 1) B.nbits = 1;
}

int bz_stage_blocks(bz2b200_ctx *ctx, int nblk, const u8 *const *blk, const u32 *len, Batch &B) {
    u32 max_n = 0;
    for (int i = 0; i < nblk; i++) {
        if (!blk[i] || len[i] == 0 || len[i] > BZ2B200_MAX_BLOCK) return BZ2B200_E_ARG;
        if (len[i] > max_n) max_n = len[i];
    }
    batch_geometry(B, nblk, max_n);
    B.total_n = 0;
    for (int i = 0; i < nblk; i++) B.total_n += len[i];
    size_t bytes = (size_t)nblk * B.stride;
    BZ_CHECK(ctx->d_T.ensure(bytes + 64));
    BZ_CHECK(ctx->d_len.ensure((size_t)nblk * 4));
    // stage through pinned memory in slabs so that copies overlap the host memcpy of the next slab
    const size_t SLAB = 64u << 20;
    BZ_CHECK(ctx->h_stage.ensure(2 * SLAB + (size_t)nblk * 4));
    u8 *hs = ctx->h_stage.as<u8>();
    u32 *hlen = (u32 *)(hs + 2 * SLAB);
    memcpy(hlen, len, (size_t)nblk * 4);
    BZ_CHECK(cudaMemcpyAsync(ctx->d_len.p, hlen, (size_t)nblk * 4, cudaMemcpyHostToDevice, ctx->stream));
    int slot = 0;
    for (int i = 0; i < nblk; i++) {
        size_t off = 0;
        while (off < len[i]) {
            size_t chunk = len[i] - off < SLAB ? len[i] - off : SLAB;
            // a slot is reused only after its previous copy has been issued two slots ago -> wait on the stream
            if (ctx->ev[6 + slot]) cudaEventSynchronize(ctx->ev[6 + slot]);
            memcpy(hs + (size_t)slot * SLAB, blk[i] + off, chunk);
            BZ_CHECK(cudaMemcpyAsync(ctx->d_T.as<u8>() + (size_t)i * B.stride + off, hs + (size_t)slot * SLAB, chunk,
                                     cudaMemcpyHostToDevice, ctx->stream));
            BZ_CHECK(cudaEventRecord(ctx->ev[6 + slot], ctx->stream));
            slot ^= 1;
            off += chunk;
        }
    }
    B.T = ctx->d_T.as<u8>();
    B.len = ctx->d_len.as<u32>();
    return BZ2B200_OK;
}

int bz_make_batch_dev(bz2b200_ctx *ctx, int nblk, u32 stride, u32 max_n, const u8 *dT, const u32 *dlen, Batch &B) {
    (void)ctx;
    batch_geometry(B, nblk, max_n);
    B.total_n = (u64)nblk * max_n;
    if (stride % BZ_TILE != 0 || stride < max_n + 64) return BZ2B200_E_ARG;
    B.stride = stride;
    B.tiles = stride / BZ_TILE;
    B.T = dT;
    B.len = dlen;
    return BZ2B200_OK;
}

// copy per-block device regions [i*stride, i*stride + bytes_i) back to caller buffers
template <class T>
static int fetch_blocks(bz2b200_ctx *ctx, int nblk, const T *d_src, size_t stride_elems, const u32 *count,
                        T *const *dst) {
    for (int i = 0; i < nblk; i++) {
        BZ_CHECK(cudaMemcpyAsync(dst[i], d_src + (size_t)i * stride_elems, (size_t)count[i] * sizeof(T),
                                 cudaMemcpyDeviceToHost, ctx->stream));
    }
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    return BZ2B200_OK;
}

extern "C" {

int bz2b200_bwt_encode_batch(bz2b200_ctx *ctx, int nblk, const uint8_t *const *in, const uint32_t *n,
                             uint8_t *const *bwt, uint32_t *key) {
    BZ_API_TRY
    if (!ctx || nblk < 0 || (nblk && (!in || !n || !bwt || !key))) return BZ2B200_E_ARG;
    if (nblk == 0) return BZ2B200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = BZ_MODE_REF;                                    // per-block seams: reference semantics
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    Batch B;
    int rc = bz_stage_blocks(ctx, nblk, in, n, B);
    if (rc) return rc;
    BZ_CHECK(ctx->d_bwt.ensure((size_t)nblk * B.stride));
    BZ_CHECK(ctx->d_key.ensure((size_t)nblk * 4));
    rc = bz_bwt_batch(ctx, B, ctx->d_bwt.as<u8>(), ctx->d_key.as<u32>());
    if (rc) return rc;
    BZ_CHECK(cudaMemcpyAsync(key, ctx->d_key.p, (size_t)nblk * 4, cudaMemcpyDeviceToHost, ctx->stream));
    return fetch_blocks<u8>(ctx, nblk, ctx->d_bwt.as<u8>(), B.stride, n, bwt);
    BZ_API_CATCH
}

int bz2b200_bwt_encode(bz2b200_ctx *ctx, const uint8_t *in, uint32_t n, uint8_t *bwt, uint32_t *key) {
    BZ_API_TRY
    const uint8_t *ins[1] = {in};
    uint8_t *outs[1] = {bwt};
    return bz2b200_bwt_encode_batch(ctx, 1, ins, &n, outs, key);
    BZ_API_CATCH
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// rle2_mtf_encode seam
// ------------------------------------------------------------------------------------------
static void symmap_from_used(const u32 ub[8], uint16_t symmap[17], int *nmap) {
    // encode_sym_map_from_bool_map, rle2_mtf.rs:293-322: L1 word + the non-empty 16-bit L2 words
    uint16_t maps[17];
    memset(maps, 0, sizeof maps);
    for (int idx = 0; idx < 256; idx++) {
        if ((ub[idx >> 5] >> (idx & 31)) & 1) {
            maps[0] |= (uint16_t)(0x8000 >> (idx >> 4));
            maps[1 + (idx >> 4)] |= (uint16_t)(0x8000 >> (idx & 15));
        }
    }
    int k = 0;
    for (int i = 0; i < 17; i++) if (maps[i]) symmap[k++] = maps[i];
    *nmap = k;
}

extern "C" int bz2b200_mtf_rle2(bz2b200_ctx *ctx, const uint8_t *bwt, uint32_t n, uint16_t *sym, uint32_t *m,
                                uint32_t freq[256], uint16_t symmap[17], int *nmap) {
    BZ_API_TRY
    if (!ctx || !bwt || !sym || !m || !freq || !symmap || !nmap || n == 0) return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    Batch B;
    const u8 *ins[1] = {bwt};
    int rc = bz_stage_blocks(ctx, 1, ins, &n, B);      // the "block text" slot holds the BWT string here
    if (rc) return rc;
    BZ_CHECK(ctx->d_sym.ensure((size_t)B.stride * 2));
    BZ_CHECK(ctx->d_m.ensure(4));
    BZ_CHECK(ctx->d_freq.ensure(256 * 4));
    BZ_CHECK(ctx->d_used.ensure(32));
    rc = bz_mtf_batch(ctx, B, B.T, ctx->d_sym.as<u16>(), ctx->d_m.as<u32>(), ctx->d_freq.as<u32>(), ctx->d_used.as<u8>());
    if (rc) return rc;
    u32 ub[8];
    BZ_CHECK(cudaMemcpyAsync(m, ctx->d_m.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaMemcpyAsync(freq, ctx->d_freq.p, 256 * 4, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaMemcpyAsync(ub, ctx->d_used.p, 32, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    BZ_CHECK(cudaMemcpyAsync(sym, ctx->d_sym.p, (size_t)(*m) * 2, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    symmap_from_used(ub, symmap, nmap);
    return BZ2B200_OK;
    BZ_API_CATCH
}

// ------------------------------------------------------------------------------------------
// huf_encode seam and the batched compress_block seam
// ------------------------------------------------------------------------------------------
// BZ2B200_LIBBZ2: the origin pointer of every periodic block of the batch (k_bwt_out counted the other members of
// rotation 0's class into d_key[nblk ..]) becomes the row libbz2's sort leaves rotation 0 in.  Only such blocks are
// downloaded; consecutive equal blocks (the inside of a long run of one byte) reuse the last answer.
static int libbz2_periodic_origins(bz2b200_ctx *ctx, const Batch &B) {
    cudaStream_t st = ctx->stream;
    const size_t nb = (size_t)B.nblk;
    std::vector<u32> h(2 * nb), len(nb);
    BZ_CHECK(cudaMemcpyAsync(h.data(), ctx->d_key.p, 2 * nb * 4, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaMemcpyAsync(len.data(), B.len, nb * 4, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    bool any = false;
    for (size_t b = 0; b < nb; b++) {
        if (h[nb + b] == 0) continue;
        std::vector<u8> blk(len[b]);
        BZ_CHECK(cudaMemcpyAsync(blk.data(), B.T + b * B.stride, len[b], cudaMemcpyDeviceToHost, st));
        BZ_CHECK(cudaStreamSynchronize(st));
        if (blk != ctx->lib_last_block) {
            long long o = bz_libbz2_fallback_origin(blk.data(), len[b]);
            if (o < 0) { ctx->err = "libbz2 mode: origin pointer of a periodic block"; return BZ2B200_E_CUDA; }
            ctx->lib_last_block.swap(blk);
            ctx->lib_last_origin = (u32)o;
        }
        h[b] = ctx->lib_last_origin;
        any = true;
    }
    if (any) {
        BZ_CHECK(cudaMemcpyAsync(ctx->d_key.p, h.data(), nb * 4, cudaMemcpyHostToDevice, st));
        BZ_CHECK(cudaStreamSynchronize(st));                    // h is freed on return
    }
    return BZ2B200_OK;
}

int bz_compress_batch(bz2b200_ctx *ctx, const Batch &B, const u32 *d_crc, HufOut &H) {
    size_t ne = (size_t)B.nblk * B.stride;
    BZ_CHECK(ctx->d_bwt.ensure(ne));
    BZ_CHECK(ctx->d_key.ensure((size_t)B.nblk * 8));
    BZ_CHECK(ctx->d_sym.ensure(ne * 2));
    BZ_CHECK(ctx->d_m.ensure((size_t)B.nblk * 4));
    BZ_CHECK(ctx->d_freq.ensure((size_t)B.nblk * 256 * 4));
    BZ_CHECK(ctx->d_used.ensure((size_t)B.nblk * 32));
    cudaStream_t st = ctx->stream;
    if (ctx->timing) cudaEventRecord(ctx->ev[0], st);
    int rc = bz_bwt_batch(ctx, B, ctx->d_bwt.as<u8>(), ctx->d_key.as<u32>(), ctx->d_used.as<u32>());
    if (rc) return rc;
    if (ctx->mode == BZ_MODE_LIBBZ2 && (rc = libbz2_periodic_origins(ctx, B))) return rc;
    if (ctx->timing) cudaEventRecord(ctx->ev[1], st);
    rc = bz_mtf_batch(ctx, B, ctx->d_bwt.as<u8>(), ctx->d_sym.as<u16>(), ctx->d_m.as<u32>(), ctx->d_freq.as<u32>(),
                      ctx->d_used.as<u8>(), true);
    if (rc) return rc;
    if (ctx->timing) cudaEventRecord(ctx->ev[2], st);
    rc = bz_huf_batch(ctx, B, ctx->d_sym.as<u16>(), ctx->d_m.as<u32>(), ctx->d_freq.as<u32>(), ctx->d_used.as<u8>(), 1,
                      d_crc, ctx->d_key.as<u32>(), H);
    if (rc) return rc;
    if (ctx->timing) {
        cudaEventRecord(ctx->ev[3], st);
        BZ_CHECK(cudaEventSynchronize(ctx->ev[3]));
        cudaEventElapsedTime(&ctx->stage_ms[1], ctx->ev[0], ctx->ev[1]);
        cudaEventElapsedTime(&ctx->stage_ms[2], ctx->ev[1], ctx->ev[2]);
        cudaEventElapsedTime(&ctx->stage_ms[3], ctx->ev[2], ctx->ev[3]);
    }
    return BZ2B200_OK;
}

extern "C" int bz2b200_compress_blocks(bz2b200_ctx *ctx, int nblk, const uint8_t *const *blk, const uint32_t *len,
                                       const uint32_t *crc, uint8_t *const *out, const size_t *out_cap,
                                       uint64_t *out_bits) {
    BZ_API_TRY
    if (!ctx || nblk < 0 || (nblk && (!blk || !len || !crc || !out || !out_cap || !out_bits))) return BZ2B200_E_ARG;
    if (nblk == 0) return BZ2B200_OK;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = BZ_MODE_REF;                                    // per-block seams: reference semantics
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    Batch B;
    int rc = bz_stage_blocks(ctx, nblk, blk, len, B);
    if (rc) return rc;
    BZ_CHECK(ctx->d_crc.ensure((size_t)nblk * 4));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_crc.p, crc, (size_t)nblk * 4, cudaMemcpyHostToDevice, ctx->stream));
    HufOut H;
    rc = bz_compress_batch(ctx, B, ctx->d_crc.as<u32>(), H);
    if (rc) return rc;
    BZ_CHECK(cudaMemcpyAsync(out_bits, H.d_bits, (size_t)nblk * 8, cudaMemcpyDeviceToHost, ctx->stream));
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < nblk; i++) {
        if (out_bits[i] == ~0ull) { ctx->err = "huffman: packed block exceeds its slot"; return BZ2B200_E_CAP; }
        size_t nb = (size_t)((out_bits[i] + 7) / 8);
        if (nb > out_cap[i]) return BZ2B200_E_CAP;
        BZ_CHECK(cudaMemcpyAsync(out[i], H.d_out + (size_t)i * H.out_stride, nb, cudaMemcpyDeviceToHost, ctx->stream));
    }
    BZ_CHECK(cudaStreamSynchronize(ctx->stream));
    return BZ2B200_OK;
    BZ_API_CATCH
}

extern "C" int bz2b200_huffman(bz2b200_ctx *ctx, const uint16_t *sym, uint32_t m, const uint32_t freq[256],
                               const uint16_t *symmap, int nmap, uint8_t *out, size_t out_cap, uint64_t *out_bits,
                               uint8_t *lengths, uint8_t *selectors, int *table_count) {
    BZ_API_TRY
    if (!ctx || !sym || !freq || !symmap || !out || !out_bits || m < 2 || m > BZ2B200_MAX_BLOCK + 1 || nmap < 2 || nmap > 17)
        return BZ2B200_E_ARG;
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->mode = BZ_MODE_REF;                                    // per-block seams: reference semantics
    if (cudaSetDevice(ctx->device) != cudaSuccess) return BZ2B200_E_CUDA;
    // used bitmap from the symbol map (decode_sym_map, symbol_map.rs:20-42)
    u32 ub[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int k = 1;
    for (int i = 0; i < 16; i++) {
        if (symmap[0] & (0x8000 >> i)) {
            if (k >= nmap) return BZ2B200_E_ARG;
            for (int j = 0; j < 16; j++)
                if (symmap[k] & (0x8000 >> j)) { int v = i * 16 + j; ub[v >> 5] |= 1u << (v & 31); }
            k++;
        }
    }
    Batch B;
    B.nblk = 1; B.max_n = m; B.stride = ((m + 64 + BZ_TILE - 1) / BZ_TILE) * BZ_TILE; B.tiles = B.stride / BZ_TILE;
    B.nbits = 1; B.T = nullptr; B.len = nullptr; B.total_n = m;
    BZ_CHECK(ctx->d_sym.ensure((size_t)B.stride * 2));
    BZ_CHECK(ctx->d_m.ensure(4));
    BZ_CHECK(ctx->d_freq.ensure(256 * 4));
    BZ_CHECK(ctx->d_used.ensure(32));
    cudaStream_t st = ctx->stream;
    BZ_CHECK(cudaMemcpyAsync(ctx->d_sym.p, sym, (size_t)m * 2, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_m.p, &m, 4, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_freq.p, freq, 256 * 4, cudaMemcpyHostToDevice, st));
    BZ_CHECK(cudaMemcpyAsync(ctx->d_used.p, ub, 32, cudaMemcpyHostToDevice, st));
    HufOut H;
    int rc = bz_huf_batch(ctx, B, ctx->d_sym.as<u16>(), ctx->d_m.as<u32>(), ctx->d_freq.as<u32>(), ctx->d_used.as<u8>(), 0,
                          nullptr, nullptr, H);
    if (rc) return rc;
    u32 misc[8];
    BZ_CHECK(cudaMemcpyAsync(out_bits, H.d_bits, 8, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaMemcpyAsync(misc, H.d_ntab, 32, cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    if (*out_bits == ~0ull) { ctx->err = "huffman: packed block exceeds its slot"; return BZ2B200_E_CAP; }
    size_t nb = (size_t)((*out_bits + 7) / 8);
    if (nb > out_cap) return BZ2B200_E_CAP;
    BZ_CHECK(cudaMemcpyAsync(out, H.d_out, nb, cudaMemcpyDeviceToHost, st));
    if (lengths) BZ_CHECK(cudaMemcpyAsync(lengths, H.d_len6, 6 * 258, cudaMemcpyDeviceToHost, st));
    if (selectors) BZ_CHECK(cudaMemcpyAsync(selectors, H.d_sel, misc[1], cudaMemcpyDeviceToHost, st));
    BZ_CHECK(cudaStreamSynchronize(st));
    if (table_count) *table_count = (int)misc[0];
    return BZ2B200_OK;
    BZ_API_CATCH
}
