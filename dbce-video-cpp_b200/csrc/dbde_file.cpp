// Streaming .dbde file writer and reader around the batched GPU codec (SURVEY.md 8 f-1).
//
// The container is what the reference's walker reads (dbde_util.cpp:362-426) and what its test
// writes by hand (dbde_util_test.cpp:204-211): a 28-byte video header (dbde_util.cpp:198-209) followed
// by frame records back to back.  The reference has no writer and a one-frame-at-a-time reader; here
//   * the writer encodes a batch on the GPU while a background thread writes the previous batch, and
//   * the reader decodes a batch on the GPU while a background thread reads the next bytes ahead,
// so disk I/O overlaps the PCIe copies.  Host code only: no codec arithmetic lives here.
#include "../../include/dbde_b200.h"
#include "dbde_record.h"

#include <stdio.h>
#include <string.h>

#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace {

thread_local std::string g_ferr;
int ffail(int code, const std::string &what) {
    g_ferr = what;
    return code;
}

void put32(uint8_t *p, uint32_t v) { memcpy(p, &v, 4); }
void put64(uint8_t *p, uint64_t v) { memcpy(p, &v, 8); }
uint32_t get32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
uint64_t get64(const uint8_t *p) { uint64_t v; memcpy(&v, p, 8); return v; }

// one background job at a time: submit() hands a closure to the helper thread, wait() joins it
struct Helper {
    std::thread th;
    std::mutex mx;
    std::condition_variable cv;
    std::function<void()> job;
    bool busy = false, quit = false;
    Helper() {
        th = std::thread([this] {
            std::unique_lock<std::mutex> lk(mx);
            for (;;) {
                cv.wait(lk, [this] { return quit || (busy && job); });
                if (quit && !(busy && job)) return;
                auto j = std::move(job);
                job = nullptr;
                lk.unlock();
                j();
                lk.lock();
                busy = false;
                cv.notify_all();
            }
        });
    }
    void submit(std::function<void()> j) {
        std::unique_lock<std::mutex> lk(mx);
        cv.wait(lk, [this] { return !busy; });
        job = std::move(j);
        busy = true;
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(mx);
        cv.wait(lk, [this] { return !busy; });
    }
    ~Helper() {
        {
            std::unique_lock<std::mutex> lk(mx);
            cv.wait(lk, [this] { return !busy; });
            quit = true;
            cv.notify_all();
        }
        th.join();
    }
};

}  // namespace

// ---------------------------------------------------------------------------------------------- writer
struct dbde_b200_writer {
    dbde_b200_ctx *ctx = nullptr;
    FILE *f = nullptr;
    int W = 0, H = 0;
    uint64_t next_index = 0, frames = 0, bytes = 0;
    uint8_t *buf[2] = {nullptr, nullptr};      // pinned record buffers: one being encoded into, one being written
    size_t cap[2] = {0, 0};
    int cur = 0;
    std::vector<uint64_t> offs;
    bool io_error = false;
    Helper io;
};

extern "C" const char *dbde_b200_file_last_error(void) { return g_ferr.c_str(); }

extern "C" int dbde_b200_writer_open(dbde_b200_ctx *ctx, const char *path, int W, int H, double frame_hz,
                                     uint64_t first_index, dbde_b200_writer **out) {
    if (!ctx || !path || !out || W <= 0 || H <= 0) return ffail(DBDE_B200_E_INVALID, "writer_open: bad argument");
    *out = nullptr;
    FILE *f = fopen(path, "wb");
    if (!f) return ffail(DBDE_B200_E_INVALID, std::string("writer_open: cannot create ") + path);
    uint8_t hdr[28];                           // dbde_util.cpp:198-209: I32 3 | U64 height | U64 width | F64 frame_hz
    put32(hdr, 3);
    put64(hdr + 4, (uint64_t)H);
    put64(hdr + 12, (uint64_t)W);
    // the container follows the process-wide DBDE_HZ_AS_INTEGER variant exactly as the drop-in
    // dbde_pack_video_header does (dbde_util.cpp:203-204): one library, one file format
    int hz_int = 0;
    dbde_b200_get_format_variants(nullptr, &hz_int);
    if (hz_int) {
        const uint64_t hz = (uint64_t)(long long)(frame_hz + 0.5);
        memcpy(hdr + 20, &hz, 8);
    } else {
        memcpy(hdr + 20, &frame_hz, 8);
    }
    if (fwrite(hdr, 1, 28, f) != 28) {
        fclose(f);
        return ffail(DBDE_B200_E_INVALID, "writer_open: cannot write the video header");
    }
    dbde_b200_writer *w = new dbde_b200_writer();
    w->ctx = ctx; w->f = f; w->W = W; w->H = H; w->next_index = first_index; w->bytes = 28;
    *out = w;
    return 0;
}

extern "C" int dbde_b200_writer_append(dbde_b200_writer *w, const uint8_t *frames_host, int nframes) {
    if (!w || !w->f || nframes < 0 || (nframes > 0 && !frames_host)) return ffail(DBDE_B200_E_INVALID, "writer_append: bad argument");
    if (nframes == 0) return 0;
    const int b = w->cur;
    // buf[b] was handed to the I/O thread two appends ago at the latest; only one job is ever in
    // flight and it uses buf[1-b], so buf[b] is free
    const size_t need = dbde_b200_stream_bound(w->W, w->H, nframes);
    if (w->cap[b] < need) {
        if (w->buf[b]) dbde_b200_host_free(w->buf[b]);
        w->buf[b] = nullptr;
        w->cap[b] = 0;
        void *p = nullptr;
        int rc = dbde_b200_host_alloc(need, &p);
        if (rc) return ffail(rc, std::string("writer_append: ") + dbde_b200_last_error());
        w->buf[b] = (uint8_t *)p;
        w->cap[b] = need;
    }
    w->offs.resize((size_t)nframes + 1);
    int rc = dbde_b200_encode_host(w->ctx, frames_host, w->W, w->H, w->next_index, nframes, w->buf[b], w->cap[b], w->offs.data());
    if (rc) return ffail(rc, std::string("writer_append: ") + dbde_b200_last_error());
    const size_t bytes = (size_t)w->offs[nframes];
    w->io.wait();                              // the previous batch is on disk (or failed)
    if (w->io_error) return ffail(DBDE_B200_E_INVALID, "writer_append: short write");
    uint8_t *src = w->buf[b];
    w->io.submit([w, src, bytes] {
        if (fwrite(src, 1, bytes, w->f) != bytes) w->io_error = true;
    });
    w->cur = 1 - b;
    w->next_index += (uint64_t)nframes;
    w->frames += (uint64_t)nframes;
    w->bytes += bytes;
    return 0;
}

extern "C" int dbde_b200_writer_close(dbde_b200_writer *w, uint64_t *frames_written, uint64_t *bytes_written) {
    if (!w) return ffail(DBDE_B200_E_INVALID, "writer_close: bad argument");
    w->io.wait();
    int rc = 0;
    if (w->f && fclose(w->f) != 0) w->io_error = true;
    if (w->io_error) rc = ffail(DBDE_B200_E_INVALID, "writer_close: write error");
    if (frames_written) *frames_written = w->frames;
    if (bytes_written) *bytes_written = w->bytes;
    for (int i = 0; i < 2; i++)
        if (w->buf[i]) dbde_b200_host_free(w->buf[i]);
    delete w;
    return rc;
}

// ---------------------------------------------------------------------------------------------- reader
struct dbde_b200_reader {
    dbde_b200_ctx *ctx = nullptr;
    FILE *f = nullptr;
    int W = 0, H = 0, batch = 1;
    size_t rec_bound = 0, fixed = 0;
    // two pinned byte buffers: `cur` holds [pos, have) unconsumed bytes; the I/O thread fills `nxt`
    uint8_t *buf[2] = {nullptr, nullptr};
    size_t cap = 0;
    int cur = 0;
    size_t pos = 0, have = 0;
    size_t ahead = 0;                          // bytes the I/O thread read into buf[1-cur]
    bool ahead_pending = false, eof = false, io_error = false, stopped = false;
    bool roi = false;                          // hand out the region rx0, ry0, rw x rh of every frame
    int rx0 = 0, ry0 = 0, rw = 0, rh = 0;
    std::vector<uint64_t> offs;
    Helper io;
};

static void reader_start_readahead(dbde_b200_reader *r) {
    if (r->eof || r->ahead_pending) return;
    uint8_t *dst = r->buf[1 - r->cur];
    const size_t room = r->cap / 2;            // leave the other half for the bytes carried over at the swap
    r->ahead_pending = true;
    r->io.submit([r, dst, room] {
        r->ahead = fread(dst + r->cap / 2, 1, room, r->f);
        if (ferror(r->f)) r->io_error = true;
    });
}

extern "C" int dbde_b200_reader_open(dbde_b200_ctx *ctx, const char *path, int batch_frames, int *W, int *H,
                                     double *frame_hz, dbde_b200_reader **out) {
    if (!ctx || !path || !out) return ffail(DBDE_B200_E_INVALID, "reader_open: bad argument");
    *out = nullptr;
    FILE *f = fopen(path, "rb");
    if (!f) return ffail(DBDE_B200_E_INVALID, std::string("reader_open: cannot open ") + path);
    uint8_t hdr[28];
    if (fread(hdr, 1, 28, f) != 28 || get32(hdr) != 3) {      // dbde_util.cpp:347-359: u64s must be 3
        fclose(f);
        return ffail(DBDE_B200_E_INVALID, "reader_open: not a DBDE video header");
    }
    const uint64_t h = get64(hdr + 4), w = get64(hdr + 12);
    // same sanity limits as the reference's walker (dbde_util.cpp:374-378)
    if (h == 0 || w == 0 || h > 0x37FFFFFF || w > 0x37FFFFFF || h * w > 0x37FFFFFF) {
        fclose(f);
        return ffail(DBDE_B200_E_INVALID, "reader_open: implausible frame size");
    }
    dbde_b200_reader *r = new dbde_b200_reader();
    r->ctx = ctx; r->f = f; r->W = (int)w; r->H = (int)h;
    r->batch = batch_frames > 0 ? batch_frames : 16;
    r->rec_bound = dbde_b200_frame_record_bound(r->W, r->H);
    const size_t wh = (size_t)((r->W + 7) / 8) * ((r->H + 7) / 8);
    r->fixed = dbde::rec_fixed(wh, 1);
    // each buffer: [carry-over half | read-ahead half], each half holds a full batch of worst-case records
    r->cap = 2 * (r->rec_bound * (size_t)r->batch + 64);
    for (int i = 0; i < 2; i++) {
        void *p = nullptr;
        int rc = dbde_b200_host_alloc(r->cap, &p);
        if (rc) {
            if (r->buf[0]) dbde_b200_host_free(r->buf[0]);
            fclose(f);
            delete r;
            return ffail(rc, std::string("reader_open: ") + dbde_b200_last_error());
        }
        r->buf[i] = (uint8_t *)p;
    }
    if (W) *W = r->W;
    if (H) *H = r->H;
    if (frame_hz) {
        int hz_int = 0;
        dbde_b200_get_format_variants(nullptr, &hz_int);       // dbde_util.cpp:352-353
        if (hz_int) {
            uint64_t hz;
            memcpy(&hz, hdr + 20, 8);
            *frame_hz = (double)hz;
        } else {
            memcpy(frame_hz, hdr + 20, 8);
        }
    }
    r->offs.resize((size_t)r->batch + 1);
    // prime: first half-buffer of bytes, synchronously, into the read-ahead half of buf[cur]
    r->pos = r->cap / 2;
    r->have = r->pos + fread(r->buf[r->cur] + r->pos, 1, r->cap / 2, f);
    if (r->have - r->pos < r->cap / 2) r->eof = true;
    reader_start_readahead(r);
    *out = r;
    return 0;
}

// Decodes up to max_frames (<= the reader's batch size) frames -- or their regions, dbde_b200_reader_set_roi --
// into frames_host.  Returns the number of frames handed out (0 at the end of the file) or a negative
// error.  status[i] != 0 marks a record
// the decoder rejected (its pixels are untouched); reading stops after the first rejected record,
// like the reference's walker (dbde_util.cpp:416).
extern "C" long dbde_b200_reader_next(dbde_b200_reader *r, uint8_t *frames_host, int max_frames, uint64_t *indices,
                                      uint32_t *status) {
    if (!r || !r->f || !frames_host || !status || max_frames <= 0)
        return ffail(DBDE_B200_E_INVALID, "reader_next: bad argument");
    if (max_frames > r->batch) max_frames = r->batch;
    if (r->stopped) return 0;
    // top up: if fewer than a worst-case batch of bytes is left, append the read-ahead
    if (r->have - r->pos < r->rec_bound * (size_t)max_frames && (r->ahead_pending || !r->eof)) {
        r->io.wait();
        if (r->io_error) return ffail(DBDE_B200_E_INVALID, "reader_next: read error");
        if (r->ahead_pending) {
            // the new bytes sit in the upper half of the other buffer; carry the unconsumed tail over in front of them
            const int n = 1 - r->cur;
            const size_t left = r->have - r->pos;
            memcpy(r->buf[n] + r->cap / 2 - left, r->buf[r->cur] + r->pos, left);
            r->cur = n;
            r->pos = r->cap / 2 - left;
            r->have = r->cap / 2 + r->ahead;
            if (r->ahead < r->cap / 2) r->eof = true;
            r->ahead_pending = false;
            reader_start_readahead(r);
        }
    }
    uint8_t *p = r->buf[r->cur] + r->pos;
    const long n = dbde_b200_index_stream(p, r->have - r->pos, r->W, r->H, r->offs.data(), max_frames);
    if (n <= 0) return 0;                      // end of file (or a torn last record)
    int rc = r->roi ? dbde_b200_decode_roi_host(r->ctx, p, (size_t)r->offs[n], r->offs.data(), r->W, r->H, (int)n, r->rx0, r->ry0,
                                                r->rw, r->rh, frames_host, status, indices)
                    : dbde_b200_decode_host(r->ctx, p, (size_t)r->offs[n], r->offs.data(), r->W, r->H, (int)n, frames_host, status, indices);
    if (rc) return ffail(rc, std::string("reader_next: ") + dbde_b200_last_error());
    long ok = n;
    for (long i = 0; i < n; i++)
        if (status[i] != 0) { ok = i + 1; break; }
    r->pos += (size_t)r->offs[ok];
    if (ok < n || status[ok - 1] != 0) r->stopped = true;                    // stop at the first bad record
    return ok;
}

extern "C" int dbde_b200_reader_set_roi(dbde_b200_reader *r, int x0, int y0, int roi_w, int roi_h) {
    if (!r || x0 < 0 || y0 < 0 || roi_w < 1 || roi_h < 1 || (long long)x0 + roi_w > r->W || (long long)y0 + roi_h > r->H)
        return ffail(DBDE_B200_E_INVALID, "reader_set_roi: the region must lie inside the frame");
    r->roi = true;                             // dbde_b200_decode_roi_host runs a full-frame region as the full decode
    r->rx0 = x0; r->ry0 = y0; r->rw = roi_w; r->rh = roi_h;
    return 0;
}

extern "C" int dbde_b200_reader_close(dbde_b200_reader *r) {
    if (!r) return ffail(DBDE_B200_E_INVALID, "reader_close: bad argument");
    r->io.wait();
    if (r->f) fclose(r->f);
    for (int i = 0; i < 2; i++)
        if (r->buf[i]) dbde_b200_host_free(r->buf[i]);
    delete r;
    return 0;
}
