// pump.cuh -- the window pump of the streaming decode drivers: the dstream (dstream.cu) and the rstream (recover.cu).
//
//   caller thread    write() copies the caller's bytes into one of two page-locked staging buffers (the context's)
//   worker thread    when a staging buffer holds WF fresh bytes (a "window"), the driver's step() decodes
//                    [carried tail | fresh bytes] and carries what the next window needs in front of the other buffer
//   delivery thread  takes the queued jobs in order: downloads a job's device ranges (ctx->s_down) in page-locked pieces
//                    of 32 MiB and calls the sink on one piece while the next one downloads, then reports its entries
// so reading the input overlaps upload and kernels, and the sink's writing overlaps download and kernels.  A batch's
// bytes are written to one of two device buffers (out_buffer); with a delivery thread the buffer is reused only when
// the job that last used it has been delivered.  Errors are sticky.  One pump at a time per context (ctx->pump_open):
// the staging buffers, window, batch outputs and output pieces stay with the context for the next one.
#pragma once
#include "common.cuh"
#include <condition_variable>
#include <deque>
#include <thread>

// Look-ahead behind a window's own range (the multi decoder's): a block that starts in the own range ends in the window
constexpr size_t DEC_LOOK = 4u << 20;
static_assert((u64)DEC_LOOK * 8 > bz_dec_span_bits(BZ2B200_MAX_BLOCK), "a block that starts before the edge ends in the window");
constexpr size_t DEC_PREFIX = DEC_LOOK + 64;   // room in front of each staging buffer for the carried tail

struct DecPump {
    bz2b200_ctx *ctx = nullptr;
    bz2b200_sink sink = nullptr;             // nullptr: nothing is downloaded
    bz2b200_rec_report report = nullptr;
    void *user = nullptr;
    bool delivers = false;                   // a delivery thread runs
    size_t WF = 64u << 20;                   // fresh bytes per window
    bool chance = false;                     // BZ2B200_MULTI_DEC_CHANCE test knob
    u64 total_in = 0;
    std::string err;                         // the first error's text (the driver prefixes it on close)

    // a batch for the delivery thread: device ranges for the sink, then entries for the report
    struct Job { DecRanges runs; std::vector<bz2b200_rec_entry> ent; };

    // claims the context's buffers, reads the window size from the environment variable `window_env` and starts the
    // threads; on an error nothing stays claimed
    int open(bz2b200_ctx *c, bz2b200_sink s, bz2b200_rec_report r, void *u, const char *window_env);
    int write(const u8 *data, size_t n);
    // decodes what is left, waits for the worker and every queued job, stops the threads: the sticky code
    int close();

    // for step(): one window, the carried tail + `len` fresh bytes of staging buffer `slot`, with ctx->mu held
    virtual int step(int slot, size_t len, bool eof) = 0;
    const u8 *window(int slot) const { return stage[slot].as<u8>() + DEC_PREFIX - tail_len; }
    size_t tail_len = 0; u64 tail_lo = 0;    // carried bytes in front of the window, and their input offset
    // the window h[0, W) to the device (*dw), prepared, with its magic candidates in `cand` (window-relative bits)
    int upload(const u8 *h, size_t W, u8 **dw);
    std::vector<u64> cand;
    // the bytes from input offset `from` to the window's end go in front of the next staging buffer
    int carry(int slot, const u8 *h, u64 lo, size_t W, u64 from);
    // the device buffer (>= nbytes + 64) of the next batch's bytes, after back-pressure
    int out_buffer(u64 nbytes, u8 **d_out);
    // hands a batch to the delivery thread; uses_buf: its ranges lie in the buffer out_buffer gave last
    void queue(Job &&j, bool uses_buf);
    virtual ~DecPump() {}

  private:
    PinBuf *stage = nullptr;                 // [2]: [DEC_PREFIX: carried tail, right-aligned | WF fresh bytes]
    DevBuf *d_win = nullptr, *d_dec = nullptr;   // one window, two batch outputs ([2])
    int cur = 0;                             // staging buffer the caller fills
    size_t fill = 0;
    std::thread th, th_out;
    std::mutex mu;                           // guards the worker hand-off, `rc`, `err` and the delivery queue
    std::condition_variable cv;
    bool busy = false, quit = false;
    int job_slot = 0; size_t job_len = 0; bool job_eof = false;
    int rc = BZ2B200_OK;                     // sticky
    std::deque<Job> jobs;
    u64 queued = 0, delivered = 0;           // jobs handed to / finished by the delivery thread
    u64 buf_job[2] = {0, 0};                 // per batch output: the number of the last job that reads it
    bool out_quit = false;
    bool out_failed = false;                 // the sink or a download failed: nothing more is delivered
    u64 nbatch = 0;                          // batch outputs handed out so far (d_dec[nbatch & 1] is the next one)
    void worker();
    void delivery();
    int submit(bool eof);
    void finish();
};
