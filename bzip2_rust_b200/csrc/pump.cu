// pump.cu -- the window pump of the streaming decode drivers (pump.cuh).
#include "pump.cuh"
#include <algorithm>
#include <stdlib.h>
#include <string.h>

int DecPump::open(bz2b200_ctx *c, bz2b200_sink s, bz2b200_rec_report r, void *u, const char *window_env) {
    {
        std::lock_guard<std::mutex> lk(c->mu);
        if (c->pump_open) return BZ2B200_E_ARG;
        c->pump_open = true;
    }
    ctx = c; sink = s; report = r; user = u;
    delivers = s || r;
    stage = ctx->h_dstage; d_win = &ctx->d_dwin; d_dec = ctx->d_ddec;
    if (const char *e = getenv(window_env)) { long long v = atoll(e); if (v >= 1024 && v <= (1ll << 30)) WF = (size_t)v; }
    chance = getenv("BZ2B200_MULTI_DEC_CHANCE") != nullptr;
    int rc = cudaSetDevice(ctx->device) != cudaSuccess ? BZ2B200_E_CUDA : BZ2B200_OK;
    for (int i = 0; i < 2 && !rc; i++) if (stage[i].ensure(DEC_PREFIX + WF) != cudaSuccess) rc = BZ2B200_E_NOMEM;
    if (sink && !rc) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        for (int i = 0; i < 2 && !rc; i++) if (ctx->h_dpiece[i].ensure(DEC_PIECE) != cudaSuccess) rc = BZ2B200_E_NOMEM;
        if (!rc && !ctx->s_up &&
            (cudaStreamCreateWithFlags(&ctx->s_up, cudaStreamNonBlocking) != cudaSuccess ||
             cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking) != cudaSuccess)) rc = BZ2B200_E_CUDA;
    }
    if (rc) { finish(); return rc; }
    th = std::thread(&DecPump::worker, this);
    if (delivers) th_out = std::thread(&DecPump::delivery, this);
    return BZ2B200_OK;
}

int DecPump::write(const u8 *data, size_t n) {
    {
        std::lock_guard<std::mutex> lk(mu);
        if (rc) return rc;
    }
    while (n) {
        size_t take = std::min(n, WF - fill);
        memcpy(stage[cur].as<u8>() + DEC_PREFIX + fill, data, take);
        fill += take; data += take; n -= take;
        if (fill == WF) {
            int r = submit(false);
            if (r) return r;
        }
    }
    return BZ2B200_OK;
}

int DecPump::close() {
    int r;
    try { r = submit(true); } catch (...) { r = BZ2B200_E_NOMEM; }
    finish();
    return r ? r : rc;
}

int DecPump::upload(const u8 *h, size_t W, u8 **dw) {
    BZ_CHECK(d_win->ensure(W + 64));
    *dw = d_win->as<u8>();
    BZ_CHECK(cudaMemcpyAsync(*dw, h, W, cudaMemcpyHostToDevice, ctx->stream));
    // at most one magic per 32 bits whatever the data: a window is never refused where the whole input is accepted
    return bz_dec_prepare(ctx, *dw, W, 4, chance, cand);
}

int DecPump::carry(int slot, const u8 *h, u64 lo, size_t W, u64 from) {
    if (from < lo || from > lo + W || lo + W - from > DEC_PREFIX) { ctx->err = "decode: lost the block chain"; return BZ2B200_E_FORMAT; }
    const size_t t = (size_t)(lo + W - from);
    memcpy(stage[slot ^ 1].as<u8>() + DEC_PREFIX - t, h + (from - lo), t);   // the caller fills that buffer from DEC_PREFIX on
    tail_lo = from; tail_len = t;
    return BZ2B200_OK;
}

int DecPump::out_buffer(u64 nbytes, u8 **d_out) {
    if (delivers) {                          // back-pressure: the last job that reads this buffer has been delivered
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return rc != BZ2B200_OK || delivered >= buf_job[nbatch & 1]; });
        if (rc) return rc;
    }
    DevBuf &b = d_dec[nbatch & 1];
    BZ_CHECK(b.ensure((size_t)nbytes + 64));
    nbatch++;
    *d_out = b.as<u8>();
    return BZ2B200_OK;
}

void DecPump::queue(Job &&j, bool uses_buf) {
    {
        std::lock_guard<std::mutex> lk(mu);
        jobs.push_back(std::move(j));
        queued++;
        if (uses_buf) buf_job[(nbatch - 1) & 1] = queued;
    }
    cv.notify_all();
}

void DecPump::worker() {
    for (;;) {
        int slot; size_t len; bool eof;
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return busy || quit; });
            if (!busy) return;
            slot = job_slot; len = job_len; eof = job_eof;
        }
        int r;
        try {
            std::lock_guard<std::mutex> lk(ctx->mu);
            total_in += len;
            r = cudaSetDevice(ctx->device) != cudaSuccess ? BZ2B200_E_CUDA : step(slot, len, eof);
        } catch (...) { r = BZ2B200_E_NOMEM; ctx->err = "out of memory"; }
        if (r) cudaStreamSynchronize(ctx->stream);             // no copy may still read the staging buffer the caller refills
        {
            std::lock_guard<std::mutex> lk(mu);
            if (r && rc == BZ2B200_OK) { rc = r; err = ctx->err; }
            busy = false;
        }
        cv.notify_all();
    }
}

void DecPump::delivery() {
    cudaSetDevice(ctx->device);
    for (;;) {
        Job j;
        bool skip;
        {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return !jobs.empty() || out_quit; });
            if (jobs.empty()) return;
            j = std::move(jobs.front()); jobs.pop_front();
            skip = out_failed;          // a decode error leaves the jobs queued before it to be delivered
        }
        int r = BZ2B200_OK;
        const char *why = "";
        if (!skip && sink) {
            r = bz_deliver_pieces(j.runs, ctx->s_down, ctx->h_dpiece, ctx->ev_dpiece, sink, user);
            why = r == BZ2B200_E_ARG ? "the sink reported an error" : "download of a decoded batch failed";
        }
        if (!skip && !r && report && !j.ent.empty() && report(user, j.ent.data(), (uint32_t)j.ent.size()) != 0) {
            r = BZ2B200_E_ARG;
            why = "the report callback reported an error";
        }
        {
            std::lock_guard<std::mutex> lk(mu);
            if (r) out_failed = true;
            if (r && rc == BZ2B200_OK) { rc = r; err = why; }
            delivered++;
        }
        cv.notify_all();
    }
}

// hands the staging buffer to the worker once the previous window is done
int DecPump::submit(bool eof) {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return !busy; });
    if (rc) return rc;
    job_slot = cur; job_len = fill; job_eof = eof;
    busy = true;
    cur ^= 1; fill = 0;
    lk.unlock();
    cv.notify_all();
    return BZ2B200_OK;
}

// stops both threads (after the worker's window and every queued job); the buffers stay with the context
void DecPump::finish() {
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return !busy && delivered == queued; });
        quit = out_quit = true;
    }
    cv.notify_all();
    if (th.joinable()) th.join();
    if (th_out.joinable()) th_out.join();
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->s_hi) cudaStreamSynchronize(ctx->s_hi);
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->pump_open = false;
}
