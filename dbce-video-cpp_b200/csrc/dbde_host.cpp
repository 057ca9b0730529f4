// Host-side mirror of the reference's C++ interface (include/dbde_util.h).
//
// The frame entry points forward to the extern "C" layer (GPU); headers are marshalled here
// (no arithmetic to accelerate, SURVEY.md C9); the tile-level functions are expressed as
// one-tile frames so they run the very same device code; the file walker decodes whole
// buffers of frames per GPU batch and hands them out one per call.
#pragma GCC visibility push(default)      // the sixteen reference entry points are the library's C++ surface
#include "../../include/dbde_util.h"
bool dbde_advance_file_buffer(dbde_file_walker &w);      // exported by the reference object, not in its header
#pragma GCC visibility pop
#include "../../include/dbde_b200.h"
#include "dbde_record.h"

#include <stdlib.h>
#include <string.h>

#include <condition_variable>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <vector>

namespace {

// One context per calling thread, lazily taken: keeps the reference's "re-entrant, callable from several
// threads on disjoint buffers" property (SURVEY.md 8b) without a global lock.  A thread that ends does NOT
// destroy its context -- freeing device and page-locked memory takes the driver's global lock for hundreds of
// milliseconds, and every other thread's next CUDA call waits behind it (measured: callers that finished early
// stalled the remaining dbde_unpack_frame callers for 0.3-1.3 s per call, 6 k -> 100 frames/s) -- it parks the
// context in a process-wide pool, where the next new thread finds it warm.  The pool is emptied at process exit.
struct ContextPool {
    std::mutex m;
    std::vector<dbde_b200_ctx *> idle;
    ~ContextPool() {
        for (dbde_b200_ctx *c : idle) dbde_b200_destroy(c);
    }
    static ContextPool &get() {
        static ContextPool p;
        return p;
    }
};
struct ThreadCtx {
    dbde_b200_ctx *ctx = nullptr;
    ~ThreadCtx() {
        if (!ctx) return;
        ContextPool &p = ContextPool::get();
        std::lock_guard<std::mutex> lk(p.m);
        p.idle.push_back(ctx);
    }
};

dbde_b200_ctx *ctx() {
    static thread_local ThreadCtx t;
    if (!t.ctx) {
        {
            ContextPool &p = ContextPool::get();
            std::lock_guard<std::mutex> lk(p.m);
            if (!p.idle.empty()) {
                t.ctx = p.idle.back();
                p.idle.pop_back();
            }
        }
        if (!t.ctx) {
            const char *dev = getenv("DBDE_B200_DEVICE");
            int rc = dbde_b200_create(dev ? atoi(dev) : 0, &t.ctx);
            if (rc != 0 || !t.ctx) {
                // there is no CPU fallback: the drop-in signatures cannot report this, so stop loudly
                fprintf(stderr, "dbde_b200: cannot create a GPU context (%d): %s\n", rc, dbde_b200_last_error());
                abort();
            }
        }
    }
    int inv = 0;
    dbde_b200_get_format_variants(&inv, nullptr);       // follow the process-wide DBDE_INVERT_ENDIAN setting
    dbde_b200_set_invert_endian(t.ctx, inv);
    return t.ctx;
}

bool hz_as_integer() {
    int hz = 0;
    dbde_b200_get_format_variants(nullptr, &hz);
    return hz != 0;
}

void die(const char *what, int rc) {
    fprintf(stderr, "dbde_b200: %s failed (%d): %s\n", what, rc, dbde_b200_last_error());
    abort();
}

// A per-thread page-locked scratch record for the image-block entry points (dbde_pack_image /
// dbde_unpack_image add or strip the 20-byte frame header around the GPU's frame records): grown on
// demand, never zero-filled, and DMA-able, so it costs one memcpy of the record and nothing else.
struct ScratchRecord {
    uint8_t *p = nullptr;
    size_t cap = 0;
};
struct ScratchPool {                 // like ContextPool: a thread that ends parks its page-locked scratch, it does not free it
    std::mutex m;
    std::vector<ScratchRecord> idle;
    ~ScratchPool() {
        for (ScratchRecord &r : idle)
            if (r.p) dbde_b200_host_free(r.p);
    }
    static ScratchPool &get() {
        static ScratchPool p;
        return p;
    }
};
struct ThreadScratch {
    ScratchRecord r;
    ~ThreadScratch() {
        if (!r.p) return;
        ScratchPool &p = ScratchPool::get();
        std::lock_guard<std::mutex> lk(p.m);
        p.idle.push_back(r);
    }
};
uint8_t *scratch_record(size_t bytes) {
    static thread_local ThreadScratch t;
    ScratchRecord &r = t.r;
    if (r.cap < bytes) {
        ScratchPool &pool = ScratchPool::get();
        {
            std::lock_guard<std::mutex> lk(pool.m);
            if (r.p) pool.idle.push_back(r);           // too small for this geometry: somebody else may still use it
            r = ScratchRecord();
            for (size_t i = 0; i < pool.idle.size(); i++)
                if (pool.idle[i].cap >= bytes) {
                    r = pool.idle[i];
                    pool.idle[i] = pool.idle.back();
                    pool.idle.pop_back();
                    break;
                }
        }
        if (!r.p) {
            void *q = nullptr;
            if (dbde_b200_host_alloc(bytes + bytes / 4, &q) != 0 || !q) {
                fprintf(stderr, "dbde_b200: cannot allocate %zu bytes of page-locked scratch: %s\n", bytes, dbde_b200_last_error());
                abort();
            }
            r.p = (uint8_t *)q;
            r.cap = bytes + bytes / 4;
        }
    }
    return r.p;
}

inline void put32(uint8_t *p, uint32_t v) { memcpy(p, &v, 4); }
inline void put64(uint8_t *p, uint64_t v) { memcpy(p, &v, 8); }
inline uint32_t get32(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline uint64_t get64(const uint8_t *p) { uint64_t v; memcpy(&v, p, 8); return v; }

}  // namespace

// ---------------------------------------------------------------- headers (host only)
// reference dbde_util.cpp:182-188
size_t dbde_pack_frame_header(frame_header fh, uint8_t *target) {
    const double e = (double)fh.elapsed_ns;
    put32(target, fh.u64s);
    put64(target + 4, fh.index);
    memcpy(target + 12, &e, 8);
    return 20;
}
// reference dbde_util.cpp:198-209 (frame_hz is a double; a rounded U64 under DBDE_HZ_AS_INTEGER, :203-204)
size_t dbde_pack_video_header(video_header vh, uint8_t *target) {
    put32(target, vh.u64s);
    put64(target + 4, vh.height);
    put64(target + 12, vh.width);
    if (hz_as_integer()) put64(target + 20, (uint64_t)(long long)(vh.frame_hz + 0.5));
    else memcpy(target + 20, &vh.frame_hz, 8);
    return 28;
}
// reference dbde_util.cpp:330-337
frame_header dbde_unpack_frame_header(uint8_t **packed) {
    const uint8_t *p = *packed;
    frame_header fh;
    double e;
    fh.u64s = get32(p);
    fh.index = get64(p + 4);
    memcpy(&e, p + 12, 8);
    fh.elapsed_ns = (uint64_t)e;
    *packed += 20;
    if (fh.u64s != 2) fh.u64s = (uint32_t)-1;
    return fh;
}
// reference dbde_util.cpp:347-359
video_header dbde_unpack_video_header(uint8_t **packed) {
    const uint8_t *p = *packed;
    video_header vh;
    vh.u64s = get32(p);
    vh.height = get64(p + 4);
    vh.width = get64(p + 12);
    if (hz_as_integer()) vh.frame_hz = (double)get64(p + 20);      // :352-353
    else memcpy(&vh.frame_hz, p + 20, 8);
    *packed += 28;
    if (vh.u64s != 3) vh.u64s = (uint32_t)-1;
    return vh;
}

// The checks dbde_unpack_image makes before it touches the image (dbde_util.cpp:295-303), made on the
// host in the reference's order and reading no more than the reference reads: nb (4 bytes), then nm,
// then n64 against the depth sum.  `blk` points at the image block (after the 20-byte frame header).
// Returns false for a block the reference rejects -- and for a depth byte > 8, which this library
// rejects (documented deviation) -- so a malformed or foreign buffer never reaches the GPU path.
namespace {
bool image_block_ok(const uint8_t *blk, size_t wh, size_t *n64_out) {
    using namespace dbde;
    if (get32(blk) != (uint32_t)wh) return false;                   // nb != w*h  (:296)
    const uint8_t *depth = blk + (kRecDepth - kRecDepthCount);
    if (get32(blk + (rec_min_count(wh) - kRecDepthCount)) != (uint32_t)wh) return false;   // nm != w*h  (:299)
    const uint32_t n64 = get32(blk + (rec_n64(wh, 1) - kRecDepthCount));
    uint64_t sum = 0;
    uint32_t big = 0;
    for (size_t i = 0; i < wh; i++) {
        sum += depth[i];
        big |= depth[i] > 8u;
    }
    if (sum != n64 || big) return false;                            // sum(depth) != n64  (:302-303)
    *n64_out = n64;
    return true;
}
}  // namespace

// ---------------------------------------------------------------- frames (GPU)
// reference dbde_util.cpp:190-196
size_t dbde_pack_frame(uint64_t index, uint8_t *image, int W, int H, uint8_t *target) {
    uint64_t offs[2];
    int rc = dbde_b200_encode_host(ctx(), image, W, H, index, 1, target, dbde_b200_frame_record_bound(W, H), offs);
    if (rc) die("dbde_pack_frame", rc);
    return (size_t)offs[1];
}
// reference dbde_util.cpp:137-180: the frame record minus its 20-byte header
size_t dbde_pack_image(uint8_t *image, int W, int H, uint8_t *target) {
    uint8_t *rec = scratch_record(dbde_b200_frame_record_bound(W, H));
    const size_t n = dbde_pack_frame(0, image, W, H, rec);
    memcpy(target, rec + 20, n - 20);
    return n - 20;
}
// reference dbde_util.cpp:339-345
frame_header dbde_unpack_frame(uint8_t **packed, int W, int H, uint8_t *image) {
    uint8_t *rec = *packed;
    frame_header fh = dbde_unpack_frame_header(packed);        // always advances 20 bytes
    // the reference has no length argument: validate in its order (:295-303), then bound the record by
    // its own fields; a rejected block leaves the pointer after the header and the image untouched
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    size_t n64 = 0;
    if (!image_block_ok(rec + 20, wh, &n64)) {
        fh.u64s = (uint32_t)-1;
        return fh;
    }
    const size_t fixed = dbde::rec_fixed(wh, 1), bytes = fixed + 8 * n64;
    uint8_t hdr_ok[4];
    put32(hdr_ok, 2);                                          // image validity is independent of the tag (:341)
    std::vector<uint8_t> tmp;
    const uint8_t *src = rec;
    if (get32(rec) != 2) {
        tmp.assign(rec, rec + (bytes < fixed ? fixed : bytes));
        memcpy(tmp.data(), hdr_ok, 4);
        src = tmp.data();
    }
    const uint64_t off0 = 0;
    uint32_t status = 0;
    int rc = dbde_b200_decode_host(ctx(), src, bytes, &off0, W, H, 1, image, &status, nullptr);
    if (rc) die("dbde_unpack_frame", rc);
    if (status != 0) fh.u64s = (uint32_t)-1;                   // pointer stays just after the header (:342)
    else *packed = rec + bytes;
    return fh;
}
// reference dbde_util.cpp:291-328: returns bytes consumed, 0 on a malformed block
size_t dbde_unpack_image(uint8_t *packed, int W, int H, uint8_t *image) {
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    size_t n64 = 0;
    if (!image_block_ok(packed, wh, &n64)) return 0;           // :296,299,303 before anything else is read
    const size_t body = dbde::rec_fixed(wh, 1) - dbde::kRecDepthCount + 8 * n64;
    uint8_t *rec = scratch_record(20 + body);
    frame_header fh = {2, 0, 0};
    dbde_pack_frame_header(fh, rec);
    memcpy(rec + 20, packed, body);
    uint8_t *p = rec;
    frame_header out = dbde_unpack_frame(&p, W, H, image);
    return out.u64s == 2 ? body : 0;
}

// ---------------------------------------------------------------- single tiles (GPU, as 1-tile frames)
// reference dbde_util.cpp:105-135: an (downmargin x rightmargin) corner IS a W=rightmargin,
// H=downmargin frame; the device clamp-pads it exactly as dbde_pack_8x8_partial does
uint32_t dbde_pack_8x8_partial(uint8_t *image, int stride, int rightmargin, int downmargin, uint8_t *target) {
    using namespace dbde;
    uint8_t px[64], rec[rec_bound(1, 1)];
    for (int y = 0; y < downmargin; y++) memcpy(px + y * rightmargin, image + (size_t)y * stride, rightmargin);
    const size_t n = dbde_pack_frame(0, px, rightmargin, downmargin, rec);
    const uint32_t depth = rec[kRecDepth], mn = rec[rec_min(1)];
    memcpy(target, rec + rec_fixed(1, 1), n - rec_fixed(1, 1));          // exactly 8*depth bytes
    return (depth << 8) | mn;
}
// reference dbde_util.cpp:22-103
uint32_t dbde_pack_8x8(uint8_t *image, int stride, uint8_t *target) {
    return dbde_pack_8x8_partial(image, stride, 8, 8, target);
}
// reference dbde_util.cpp:216-279 (depth >= 8 reads 64 raw bytes, :229)
void dbde_unpack_8x8(uint8_t depth, uint8_t minval, uint8_t *packed, size_t stride, uint8_t *image) {
    const uint32_t k = depth > 8 ? 8 : depth;
    using namespace dbde;
    uint8_t rec[rec_bound(1, 1)], px[64];
    frame_header fh = {2, 0, 0};
    dbde_pack_frame_header(fh, rec);
    put32(rec + kRecDepthCount, 1);
    rec[kRecDepth] = (uint8_t)k;
    put32(rec + rec_min_count(1), 1);
    rec[rec_min(1)] = minval;
    put32(rec + rec_n64(1, 1), k);
    memcpy(rec + rec_fixed(1, 1), packed, 8 * k);
    uint8_t *p = rec;
    dbde_unpack_frame(&p, 8, 8, px);
    for (int y = 0; y < 8; y++) memcpy(image + y * stride, px + 8 * y, 8);
}
// reference dbde_util.cpp:281-289
void dbde_unpack_8x8_partial(uint8_t depth, uint8_t minval, uint8_t *packed, size_t stride, int rightmargin,
                             int downmargin, uint8_t *image) {
    uint8_t img[64];
    dbde_unpack_8x8(depth, minval, packed, 8, img);
    for (int y = 0; y < downmargin; y++) memcpy(image + stride * y, img + 8 * y, rightmargin);
}

// ---------------------------------------------------------------- file walker
// Same interface and field meanings as the reference (dbde_util.cpp:362-426) but: the buffer is
// sized for the true worst-case record (rec_bound(wh, 1), not npix + npix/8 + 32, which under-sizes
// small odd frames), it is freed in dbde_end_file_walk, and frames are decoded on the GPU in
// batches of `frames_buffered`.  A helper thread reads, indexes and decodes batch k+1 (fread -> page-locked
// file buffer -> H2D -> kernels -> D2H into a pinned batch buffer) while the caller is still being handed
// the frames of batch k, one per call: disk I/O and PCIe overlap the caller's own work (SURVEY 8 f-1).
namespace {
struct WalkerSide {
    // file state: owned by the helper thread after start (the caller's struct only mirrors it)
    FILE *f = nullptr;
    uint8_t *buffer = nullptr;
    size_t i = 0, n = 0, N = 0;
    int W = 1, H = 1, batch = 1;
    bool registered = false;            // `buffer` is page-locked (dbde_b200_host_register)
    // two decoded batches (pinned: the D2H copy of a batch runs at PCIe speed)
    uint8_t *frames[2] = {nullptr, nullptr};
    std::vector<frame_header> hdrs[2];
    size_t have[2] = {0, 0};
    // the reference's bookkeeping for the caller's struct (dbde_util.h:42-43): where each record of the
    // batch ended in the buffer (`i` after that frame) and how much of the buffer was good data (`n`)
    std::vector<size_t> iafter[2];
    size_t nat[2] = {0, 0};
    bool io_error = false;              // fread failed (dbde_advance_file_buffer's `false`)
    // hand-off: batch k lives in slot k & 1; the helper may run at most two batches ahead of `consumed`
    std::mutex m;
    std::condition_variable cv;
    size_t produced = 0, consumed = 0;
    bool finished = false, stop = false;
    std::thread worker;
    // caller side
    size_t next = 0;                    // next frame of the current batch
    bool holding = false;               // the caller is inside batch `consumed`
};
std::mutex g_wmx;
std::unordered_map<uint8_t *, WalkerSide *> g_wside;      // keyed by walker->buffer

WalkerSide *side_of(const dbde_file_walker *w) {
    std::lock_guard<std::mutex> lk(g_wmx);
    auto it = g_wside.find(w->buffer);
    return it == g_wside.end() ? nullptr : it->second;
}

// keep [i, n) topped up from the file (reference dbde_advance_file_buffer, :394-406)
bool refill(WalkerSide *s) {
    if (s->i > 0) {
        if (s->i < s->n) memmove(s->buffer, s->buffer + s->i, s->n - s->i);
        s->n -= s->i;
        s->i = 0;
    }
    if (!feof(s->f)) {
        s->n += fread(s->buffer + s->n, 1, s->N - s->n, s->f);
        if (ferror(s->f)) {
            s->io_error = true;
            return false;
        }
    }
    return true;
}

// decode the next batch of whole records into slot `b`; false = nothing more to hand out after this
bool produce(WalkerSide *s, int b) {
    s->have[b] = 0;
    if (!refill(s)) return false;
    std::vector<uint64_t> offs(s->batch + 1);
    const long n = dbde_b200_index_stream(s->buffer + s->i, s->n - s->i, s->W, s->H, offs.data(), s->batch);
    if (n <= 0) return false;                              // end of file (or a torn last record)
    s->nat[b] = s->n;
    std::vector<uint32_t> status(n);
    std::vector<uint64_t> index(n);
    int rc = dbde_b200_decode_host(ctx(), s->buffer + s->i, (size_t)offs[n], offs.data(), s->W, s->H, (int)n, s->frames[b],
                                   status.data(), index.data());
    if (rc) die("dbde_walk_a_file", rc);
    bool more = true;
    for (long k = 0; k < n; k++) {
        uint8_t *p = s->buffer + s->i + offs[k];
        s->hdrs[b][k] = dbde_unpack_frame_header(&p);
        if (status[k] != 0) s->hdrs[b][k].u64s = (uint32_t)-1;
        s->iafter[b][k] = s->i + (size_t)offs[k + 1];
        s->have[b]++;
        if (s->hdrs[b][k].u64s != 2) { more = false; break; }      // the reference stops at the first bad frame (:416)
    }
    s->i += (size_t)offs[n];
    return more;
}

void worker_main(WalkerSide *s) {
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(s->m);
            s->cv.wait(lk, [&] { return s->stop || s->produced - s->consumed < 2; });
            if (s->stop) return;
        }
        const bool more = produce(s, (int)(s->produced & 1));
        {
            std::lock_guard<std::mutex> lk(s->m);
            if (s->have[s->produced & 1] > 0) s->produced++;
            if (!more) s->finished = true;
        }
        s->cv.notify_all();
        if (!more) return;
    }
}

void destroy_side(WalkerSide *s) {
    {
        std::lock_guard<std::mutex> lk(s->m);
        s->stop = true;
    }
    s->cv.notify_all();
    if (s->worker.joinable()) s->worker.join();
    if (s->registered) dbde_b200_host_unregister(s->buffer);
    for (int b = 0; b < 2; b++)
        if (s->frames[b]) dbde_b200_host_free(s->frames[b]);
    if (s->f) fclose(s->f);
    free(s->buffer);
    delete s;
}
}  // namespace

dbde_file_walker dbde_start_file_walk(const char *name, int frames_buffered, video_header *vh) {
    if (frames_buffered < 1) frames_buffered = 2;
    dbde_file_walker w = {NULL, 0, 0, 0, 0, 1, 1, NULL};
    FILE *f = fopen(name, "rb");
    if (!f) return w;
    uint8_t head[28];
    if (fread(head, 1, 28, f) != 28) { fclose(f); return w; }
    uint8_t *hp = head;
    *vh = dbde_unpack_video_header(&hp);
    // same sanity limits as the reference (:374-378)
    if (vh->u64s != 3 || vh->height == 0 || vh->width == 0 || vh->height > 0x37FFFFFF || vh->width > 0x37FFFFFF ||
        vh->height * vh->width > 0x37FFFFFF) {
        fclose(f);
        return w;
    }
    const size_t bound = dbde_b200_frame_record_bound((int)vh->width, (int)vh->height);
    const size_t N = bound * (size_t)frames_buffered + 64;
    if (N >= 0x7FFFFFFF) { fclose(f); return w; }
    WalkerSide *s = new WalkerSide();
    s->buffer = (uint8_t *)malloc(N);
    if (!s->buffer) { fclose(f); delete s; return w; }
    s->f = f;
    s->N = N;
    s->W = (int)vh->width;
    s->H = (int)vh->height;
    s->batch = frames_buffered;
    const size_t px = (size_t)s->W * s->H;
    for (int b = 0; b < 2; b++) {
        if (dbde_b200_host_alloc((size_t)frames_buffered * px, (void **)&s->frames[b]) != 0) {
            destroy_side(s);
            return w;
        }
        s->hdrs[b].resize(frames_buffered);
        s->iafter[b].resize(frames_buffered);
    }
    // the file buffer is ours from malloc to free: page-lock it so the records go to the GPU by DMA
    s->registered = dbde_b200_host_register(s->buffer, N) == 0;
    // the caller's struct mirrors the reference's fields; the file itself now belongs to the helper thread
    w.fptr = f;
    w.buffer = s->buffer;
    w.N = N;
    w.width = (int32_t)vh->width;
    w.height = (int32_t)vh->height;
    {
        std::lock_guard<std::mutex> lk(g_wmx);
        g_wside[w.buffer] = s;
    }
    s->worker = std::thread(worker_main, s);
    return w;
}

bool dbde_walk_a_file(dbde_file_walker *w, frame_header *fh, uint8_t *image) {
    if (!w || !w->fptr) return false;
    WalkerSide *s = side_of(w);
    if (!s) return false;
    const size_t px = (size_t)s->W * s->H;
    if (!s->holding || s->next == s->have[s->consumed & 1]) {
        // hand the finished batch back to the helper and wait for the next one
        std::unique_lock<std::mutex> lk(s->m);
        if (s->holding) {
            s->consumed++;
            s->holding = false;
            s->cv.notify_all();
        }
        s->cv.wait(lk, [&] { return s->produced > s->consumed || s->finished; });
        if (s->produced == s->consumed) return false;      // end of file (or a torn last record)
        s->holding = true;
        s->next = 0;
    }
    const int b = (int)(s->consumed & 1);
    *fh = s->hdrs[b][s->next];
    if (fh->u64s != 2) { dbde_end_file_walk(w); return false; }   // reference :416
    memcpy(image, s->frames[b] + px * s->next, px);
    // mirror the reference's bookkeeping (:421): `i` just after the record handed out, `n` the good data
    // of the buffer it was read from; `frames` stays untouched, as in the reference
    w->i = s->iafter[b][s->next];
    w->n = s->nat[b];
    s->next++;
    return true;
}

// reference dbde_util.cpp:394-406 (exported by the reference object although dbde_util.h does not
// declare it): "make sure there is always plenty of buffer past the current index"; false only when
// reading the file failed.  Here the helper thread tops the buffer up on its own, so the call waits
// until the next batch is ready (or the file has ended) and reports the helper's read status.
bool dbde_advance_file_buffer(dbde_file_walker &w) {
    if (!w.fptr) return false;
    WalkerSide *s = side_of(&w);
    if (!s) return false;
    std::unique_lock<std::mutex> lk(s->m);
    s->cv.wait(lk, [&] { return s->produced > s->consumed || s->finished; });
    return !s->io_error;
}

void dbde_end_file_walk(dbde_file_walker *w) {
    if (!w) return;
    WalkerSide *s = nullptr;
    if (w->buffer) {
        std::lock_guard<std::mutex> lk(g_wmx);
        auto it = g_wside.find(w->buffer);
        if (it != g_wside.end()) {
            s = it->second;
            g_wside.erase(it);
        }
    }
    if (s) destroy_side(s);                                // joins the helper, closes the file, frees the buffers
    else if (w->fptr) fclose(w->fptr);
    w->fptr = NULL;
    w->buffer = NULL;
}
