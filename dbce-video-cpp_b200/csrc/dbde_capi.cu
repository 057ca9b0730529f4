// extern "C" layer of the B200 DBDE codec (see include/dbde_b200.h for the contracts).
// Host-side plumbing only: geometry, scratch, launches, and the chunked pinned-staging pipeline
// for host buffers.  No codec arithmetic lives here and there is no CPU fallback.
#include "../../include/dbde_b200.h"
#include "dbde_kernels.h"
#include "dbde_copy_pool.h"

#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <deque>
#include <mutex>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace dbde;

static thread_local std::string g_err;
static int fail(int code, const char *what) {
    g_err = what;
    return code;
}
static int cuda_fail(cudaError_t e, const char *where) {
    g_err = std::string(where) + ": " + cudaGetErrorString(e);
    return (int)e;
}
#define CK(call)                                              \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// DBDE_B200_PROFILE=1: per-thread wall-clock sums of the host path's phases, printed when the thread ends
// (where the time of a one-frame call goes: staging copies, launches, waiting for the GPU, copy-out)
namespace {
struct PhaseProfile {
    static bool on() {
        static const bool v = getenv("DBDE_B200_PROFILE") != nullptr;
        return v;
    }
    const char *name[8] = {};
    double sum[8] = {};
    double gpu[3] = {};                 // GPU timeline of the encode path: H2D DMAs, kernels, size copy + flag (ms)
    cudaEvent_t ge[4] = {};
    long calls = 0;
    std::chrono::steady_clock::time_point t;
    void start() { if (on()) t = std::chrono::steady_clock::now(); }
    void gpu_mark(int i, cudaStream_t st) {
        if (!on()) return;
        if (!ge[0]) for (auto &e : ge) cudaEventCreate(&e);
        cudaEventRecord(ge[i], st);
    }
    void gpu_collect() {
        if (!on() || !ge[0]) return;
        for (int i = 0; i < 3; i++) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, ge[i], ge[i + 1]) == cudaSuccess) gpu[i] += ms;
        }
    }
    void mark(int i, const char *what) {
        if (!on()) return;
        const auto n = std::chrono::steady_clock::now();
        name[i] = what;
        sum[i] += std::chrono::duration<double, std::micro>(n - t).count();
        t = n;
    }
    ~PhaseProfile() {
        if (!on() || !calls) return;
        std::string line = "dbde_b200 profile (" + std::to_string(calls) + " calls, us per call):";
        for (int i = 0; i < 8; i++)
            if (name[i]) line += std::string(" ") + name[i] + "=" + std::to_string((long)(sum[i] / calls));
        if (ge[0]) line += " | gpu: h2d=" + std::to_string((long)(1e3 * gpu[0] / calls)) + " kernels=" + std::to_string((long)(1e3 * gpu[1] / calls)) +
                           " sizes+flag=" + std::to_string((long)(1e3 * gpu[2] / calls));
        fprintf(stderr, "%s\n", line.c_str());
    }
};
thread_local PhaseProfile g_enc_prof, g_dec_prof;
}  // namespace

constexpr int kMaxHostSlots = 8;
constexpr int kDefaultHostSlots = 3;

struct HostSlot {
    cudaStream_t st = nullptr;
    cudaEvent_t ev = nullptr;
    uint8_t *d_a = nullptr;      // encode: frames   | decode: stream bytes
    uint8_t *d_b = nullptr;      // encode: records in their slots | decode: frames
    uint8_t *d_c = nullptr;      // encode: records back to back (compacted on the device) | decode crops: the chunk's corners
    uint64_t *d_off = nullptr;
    uint64_t *d_size = nullptr;
    uint32_t *d_status = nullptr;
    uint64_t *d_index = nullptr;
    uint64_t *h_off = nullptr;   // pinned
    uint64_t *h_size = nullptr;  // pinned
    uint32_t *h_status = nullptr;   // pinned mirrors of d_status / d_index (decode)
    uint64_t *h_index = nullptr;
    // pageable caller buffers (the reference's callers pass malloc'd memory, dbde_util.h:24-35): pinned
    // bounce buffers the bytes are relayed through in pieces, by parallel memcpy overlapped with the DMA
    uint8_t *h_in = nullptr, *h_out = nullptr;
    size_t cap_hin = 0, cap_hout = 0;
    int32_t *h_corners = nullptr;   // pinned staging of the chunk's crop corners (decode crops)
    size_t cap_hcorners = 0;
    // completion flags in pinned memory: a 4-byte D2H copy of the context's device word `1`, queued behind the
    // work it reports, sets one; host threads wait on them by reading memory, not by calling the driver
    volatile uint32_t *h_flag = nullptr;    // kMaxDmaPieces for relayed D2H pieces + 1 for the chunk's kernels
    size_t cap_a = 0, cap_b = 0, cap_c = 0;
    int cap_n = 0;
    int n = 0, first = 0;
    size_t piece = 0;            // DMA piece size of the chunk's relayed pixel copy (decode, pageable output)
};

// Scan scratch (encode: ticket + look-back descriptors; decode: word prefixes) belongs to the STREAM a
// launch goes to: launches on one stream are ordered, launches on different streams are not, so two
// chunks in flight on two staging streams must never share a ticket counter or a prefix table.
constexpr int kMaxStreamScratch = 16;
struct StreamScratch {
    bool used = false;
    cudaStream_t st = nullptr;
    void *enc = nullptr, *dec = nullptr;
    size_t enc_bytes = 0, dec_bytes = 0;
    uint64_t last_use = 0;
};

struct dbde_b200_ctx {
    int device = 0;
    int num_sms = 0;
    StreamScratch scratch[kMaxStreamScratch];
    uint64_t scratch_clock = 0;
    HostSlot slots[kMaxHostSlots];
    int nslots = kDefaultHostSlots;   // staging slots in flight (DBDE_B200_SLOTS)
    int chunk_frames = 0;             // frames per chunk, 0 = auto (DBDE_B200_CHUNK_FRAMES)
    int invert_endian = 0;            // DBDE_INVERT_ENDIAN variant; initialised from the process-wide setting
    uint64_t launches = 0;
    uint32_t *d_one = nullptr;        // a device word holding 1: the source of the completion-flag copies
};

// ------------------------------------------------------------------ geometry
static PartGeom make_geom(int W, int H, bool fast) {
    PartGeom g;
    g.W = W; g.H = H;
    g.w = (W + 7) / 8; g.h = (H + 7) / 8; g.wh = g.w * g.h;
    g.linear = 0;
    int ntx_max;
    if (g.w > kTilesPerPart) {
        g.nseg = (g.w + kTilesPerPart - 1) / kTilesPerPart;
        g.G = 1;
        g.ppf = g.h * g.nseg;
        ntx_max = kTilesPerPart;
    } else {
        g.nseg = 1;
        g.G = kTilesPerPart / g.w;
        if (g.G > kMaxBandsPerPart) g.G = kMaxBandsPerPart;
        if (g.G > g.h) g.G = g.h;
        ntx_max = g.w;
    }
    // odd sizes: a row's 16-byte hull is up to 30 bytes longer than the row, and for band segments (w > 256) the
    // pitch is W modulo 16, which lets every row sit at its global alignment at a constant stride (dbde_encode.cu)
    auto pitch_of = [&](int ntx) { return fast ? 8 * ntx : ((8 * ntx + 15) / 16) * 16 + 48 + (g.w > kTilesPerPart ? (W & 15) : 0); };
    g.pitch = pitch_of(ntx_max);
    while (g.G > 1 && 8 * g.G * g.pitch > 20480) g.G--;
    if (g.nseg == 1) g.ppf = (g.h + g.G - 1) / g.G;
    // Band-aligned partitions leave lanes idle when the width does not fill them: 2304 pixels = 288 tiles is a
    // 256-tile and a 32-tile segment per band (56 % of the lanes work), 1280 pixels = 160 tiles is one band per
    // partition (63 %).  Aligned frames at least 32 tiles wide then use LINEAR partitions: 256 consecutive tiles
    // of the row-major tile order, staged as the <= 256/w + 2 band pieces they consist of, side by side at the
    // constant row pitch 2048 -- every lane has a tile (measured: 2304x2304 3.55 -> see DESIGN.md section 6).
    if (fast && g.w >= 32 && g.w % kTilesPerPart != 0) {
        const double used = g.nseg > 1 ? (double)g.w / (g.nseg * kTilesPerPart) : (double)(g.G * g.w) / kTilesPerPart;
        if (used < 0.9 && getenv("DBDE_B200_NO_LINEAR") == nullptr) g = linear_geom(W, H);
    }
    int need = 8 * g.G * g.pitch;
    if (need < 64 * kTilesPerPart) need = 64 * kTilesPerPart;
    g.stage_bytes = ((need + 64 + 127) / 128) * 128;
    return g;
}

static bool dims_ok(int W, int H, int nframes) {
    if (W <= 0 || H <= 0 || nframes < 0) return false;
    const long long wh = (((long long)W + 7) / 8) * (((long long)H + 7) / 8);   // W + 7 overflows int near INT32_MAX
    return wh <= 0x0FFFFFFF && (long long)W * H <= 0x7FFFFFFFLL;
}

// ------------------------------------------------------------------ format variants
// The reference's two compile-time variants (SURVEY 8 f-3).  Building this library with the same
// macros makes them the defaults; dbde_b200_set_format_variants() switches them at run time.
#ifdef DBDE_INVERT_ENDIAN
static std::atomic<int> g_invert_endian{1};
#else
static std::atomic<int> g_invert_endian{0};
#endif
#ifdef DBDE_HZ_AS_INTEGER
static std::atomic<int> g_hz_as_integer{1};
#else
static std::atomic<int> g_hz_as_integer{0};
#endif
extern "C" void dbde_b200_set_format_variants(int invert_endian, int hz_as_integer) {
    g_invert_endian.store(invert_endian ? 1 : 0, std::memory_order_relaxed);
    g_hz_as_integer.store(hz_as_integer ? 1 : 0, std::memory_order_relaxed);
}
extern "C" void dbde_b200_get_format_variants(int *invert_endian, int *hz_as_integer) {
    if (invert_endian) *invert_endian = g_invert_endian.load(std::memory_order_relaxed);
    if (hz_as_integer) *hz_as_integer = g_hz_as_integer.load(std::memory_order_relaxed);
}

// ------------------------------------------------------------------ lifetime
extern "C" int dbde_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

extern "C" int dbde_b200_create(int device, dbde_b200_ctx **out) {
    if (!out) return fail(DBDE_B200_E_INVALID, "dbde_b200_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(DBDE_B200_E_NO_DEVICE, "dbde_b200: no CUDA device; this library has no CPU fallback");
    if (device < 0 || device >= n) return fail(DBDE_B200_E_INVALID, "dbde_b200_create: device out of range");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(DBDE_B200_E_NO_DEVICE, "dbde_b200: kernels are built for sm_100a (B200) only; no fallback");
    CK(cudaSetDevice(device));
    dbde_b200_ctx *c = new dbde_b200_ctx();
    c->device = device;
    c->num_sms = prop.multiProcessorCount;
    c->invert_endian = g_invert_endian.load(std::memory_order_relaxed);
    if (const char *e = getenv("DBDE_B200_SLOTS")) {
        const int n = atoi(e);
        if (n >= 2 && n <= kMaxHostSlots) c->nslots = n;
    }
    if (const char *e = getenv("DBDE_B200_CHUNK_FRAMES")) {
        const int n = atoi(e);
        if (n > 0) c->chunk_frames = n;
    }
    *out = c;
    return 0;
}

static void free_slot(HostSlot &s) {
    if (s.d_a) cudaFree(s.d_a);
    if (s.d_b) cudaFree(s.d_b);
    if (s.d_c) cudaFree(s.d_c);
    if (s.d_off) cudaFree(s.d_off);
    if (s.d_size) cudaFree(s.d_size);
    if (s.h_size) cudaFreeHost(s.h_size);
    if (s.d_status) cudaFree(s.d_status);
    if (s.d_index) cudaFree(s.d_index);
    if (s.h_off) cudaFreeHost(s.h_off);
    if (s.h_status) cudaFreeHost(s.h_status);
    if (s.h_index) cudaFreeHost(s.h_index);
    if (s.h_in) cudaFreeHost(s.h_in);
    if (s.h_out) cudaFreeHost(s.h_out);
    if (s.h_corners) cudaFreeHost(s.h_corners);
    if (s.h_flag) cudaFreeHost((void *)s.h_flag);
    if (s.ev) cudaEventDestroy(s.ev);
    if (s.st) cudaStreamDestroy(s.st);
    s = HostSlot();
}

extern "C" void dbde_b200_destroy(dbde_b200_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto &s : c->slots) free_slot(s);
    for (auto &x : c->scratch) {
        if (x.enc) cudaFree(x.enc);
        if (x.dec) cudaFree(x.dec);
    }
    if (c->d_one) cudaFree(c->d_one);
    delete c;
}

extern "C" const char *dbde_b200_last_error(void) { return g_err.c_str(); }
extern "C" uint64_t dbde_b200_kernel_launches(const dbde_b200_ctx *c) { return c ? c->launches : 0; }

extern "C" int dbde_b200_set_invert_endian(dbde_b200_ctx *c, int on) {
    if (!c) return fail(DBDE_B200_E_INVALID, "set_invert_endian: bad argument");
    c->invert_endian = on ? 1 : 0;
    return 0;
}

extern "C" int dbde_b200_set_chunk_frames(dbde_b200_ctx *c, int frames) {
    if (!c || frames < 0) return fail(DBDE_B200_E_INVALID, "set_chunk_frames: bad argument");
    c->chunk_frames = frames;
    return 0;
}

// ------------------------------------------------------------------ sizes
extern "C" size_t dbde_b200_frame_record_bound(int W, int H) {
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    return rec_bound(wh, 1);
}
extern "C" size_t dbde_b200_slot_stride(int W, int H) { return (dbde_b200_frame_record_bound(W, H) + 15) / 16 * 16; }
extern "C" size_t dbde_b200_stream_bound(int W, int H, int nframes) {
    return dbde_b200_slot_stride(W, H) * (size_t)(nframes < 0 ? 0 : nframes) + 16;
}

// ------------------------------------------------------------------ memory helpers
extern "C" int dbde_b200_device_alloc(dbde_b200_ctx *c, size_t bytes, void **out) {
    if (!c || !out) return fail(DBDE_B200_E_INVALID, "device_alloc: bad argument");
    CK(cudaSetDevice(c->device));
    CK(cudaMalloc(out, bytes + 32));
    return 0;
}
extern "C" int dbde_b200_device_free(dbde_b200_ctx *c, void *p) {
    if (!c) return fail(DBDE_B200_E_INVALID, "device_free: bad argument");
    CK(cudaSetDevice(c->device));
    CK(cudaFree(p));
    return 0;
}
extern "C" int dbde_b200_host_alloc(size_t bytes, void **out) {
    if (!out) return fail(DBDE_B200_E_INVALID, "host_alloc: bad argument");
    CK(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return 0;
}
extern "C" int dbde_b200_host_free(void *p) {
    CK(cudaFreeHost(p));
    return 0;
}
// Page-locks memory the CALLER owns (malloc, new, a mapped file ...) so the host entry points copy
// it by DMA instead of through the driver's pageable staging.  The caller must unregister before
// freeing it; the library never registers anything behind the caller's back (a cached registration
// of memory that was freed and re-mapped would DMA into the wrong pages).
extern "C" int dbde_b200_host_register(void *p, size_t bytes) {
    if (!p || !bytes) return fail(DBDE_B200_E_INVALID, "host_register: bad argument");
    CK(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return 0;
}
extern "C" int dbde_b200_host_unregister(void *p) {
    if (!p) return fail(DBDE_B200_E_INVALID, "host_unregister: bad argument");
    CK(cudaHostUnregister(p));
    return 0;
}
extern "C" int dbde_b200_memcpy_h2d(dbde_b200_ctx *c, void *dst, const void *src, size_t bytes) {
    if (!c) return fail(DBDE_B200_E_INVALID, "memcpy_h2d: bad argument");
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return 0;
}
extern "C" int dbde_b200_memcpy_d2h(dbde_b200_ctx *c, void *dst, const void *src, size_t bytes) {
    if (!c) return fail(DBDE_B200_E_INVALID, "memcpy_d2h: bad argument");
    CK(cudaSetDevice(c->device));
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return 0;
}

static int grow(void **p, size_t *have, size_t need) {
    if (*have >= need) return 0;
    if (*p) CK(cudaFree(*p));
    *p = nullptr;
    *have = 0;
    need += need / 4;
    CK(cudaMalloc(p, need));
    *have = need;
    return 0;
}

// the scratch entry of `st`; when all entries are taken the least recently used one is recycled
// (cudaFree waits for the device, so nothing in flight still reads it)
static StreamScratch &scratch_for(dbde_b200_ctx *c, cudaStream_t st) {
    StreamScratch *lru = nullptr;
    for (auto &x : c->scratch)
        if (x.used && x.st == st) {
            x.last_use = ++c->scratch_clock;
            return x;
        }
    for (auto &x : c->scratch) {
        if (!x.used) { lru = &x; break; }
        if (!lru || x.last_use < lru->last_use) lru = &x;
    }
    if (lru->used) {
        cudaDeviceSynchronize();
        if (lru->enc) cudaFree(lru->enc);
        if (lru->dec) cudaFree(lru->dec);
        *lru = StreamScratch();
    }
    lru->used = true;
    lru->st = st;
    lru->last_use = ++c->scratch_clock;
    return *lru;
}

// ------------------------------------------------------------------ requests
// Every codec entry point describes its call as one Request: the pixel format, the output form and its fields, and
// its public name.  check_decode / check_encode hold every argument rule; enqueue_decode / enqueue_encode pick and
// queue the kernels and check nothing.  A device entry point is request, check, enqueue; a host entry point is
// request, check, then the chunk pipeline, which enqueues once per chunk.
enum class Form { Full, Validate, Region, Crops, Binned };

// What the pixel format fixes for frames of w x h pixels
struct Fmt {
    size_t px, bound, stride;   // bytes per frame, the record bound, the slot stride
    size_t delta;               // where a slot's record starts so that its U64 words are 16-byte aligned
    size_t stream_bound(int n) const { return stride * (size_t)(n < 0 ? 0 : n) + 16; }
};

struct Request {
    const char *name;           // the entry point, for dbde_b200_last_error()
    bool u16;                   // DBDE16 records of U16 frames, else the reference's 8-bit records
    Form form;                  // encoders: Full or Crops
    int W, H, nframes;
    int factor = 0;             // Binned: 1, 2, 4 or 8
    int x0 = 0, y0 = 0;         // Region: the rectangle's corner
    int w = 0, h = 0;           // Region: its size; Crops: the crop size
    const int32_t *corners = nullptr;    // Crops, in the caller's memory: nframes * ncrops {x0, y0} pairs if per_frame, else ncrops
    int ncrops = 1, per_frame = 0, pad = 0;

    int pad_max() const { return u16 ? 65535 : 255; }
    Fmt fmt(int fw, int fh) const {
        const size_t wh = (size_t)((fw + 7) / 8) * ((fh + 7) / 8);
        Fmt f;
        f.px = (size_t)fw * fh * (u16 ? 2 : 1);
        f.bound = u16 ? dbde_b200_frame_record_bound16(fw, fh) : dbde_b200_frame_record_bound(fw, fh);
        f.stride = (f.bound + 15) & ~(size_t)15;
        f.delta = (16 - rec_fixed(wh, u16 ? 2 : 1) % 16) % 16;
        return f;
    }
    int records() const { return form == Form::Crops ? ncrops : 1; }      // per frame
    Fmt record_fmt() const { return form == Form::Crops ? fmt(w, h) : fmt(W, H); }
    // bytes per frame a decode writes: the frame, the region, the crops or the bins
    size_t out_bytes() const {
        switch (form) {
        case Form::Region: return fmt(w, h).px;
        case Form::Crops: return fmt(w, h).px * (size_t)ncrops;
        case Form::Binned: return fmt((W - 1) / factor + 1, (H - 1) / factor + 1).px;
        default: return fmt(W, H).px;
        }
    }
    size_t corner_bytes(int n) const { return form == Form::Crops ? 8 * (size_t)ncrops * (size_t)(per_frame ? n : 1) : 0; }
};

static int reject(const Request &r, int code, const char *why) {
    g_err = std::string(r.name) + ": " + why;
    return code;
}

static bool roi_ok(int W, int H, int x0, int y0, int roi_w, int roi_h) {
    return x0 >= 0 && y0 >= 0 && roi_w >= 1 && roi_h >= 1 && (long long)x0 + roi_w <= W && (long long)y0 + roi_h <= H;
}
// the size limit counts pixels whatever their width
static bool crops_ok(int ncrops, int corners_per_frame, int crop_w, int crop_h, int pad, int pad_max) {
    return ncrops >= 1 && crop_w >= 1 && crop_h >= 1 && dims_ok(crop_w, crop_h, 0) &&
           (long long)ncrops * crop_w * crop_h <= 0x7FFFFFFFLL && (corners_per_frame == 0 || corners_per_frame == 1) && pad >= 0 &&
           pad <= pad_max;
}
static bool factor_ok(int factor) { return factor == 1 || factor == 2 || factor == 4 || factor == 8; }

// the rules every form shares: the frame, and the output form's own fields
static bool request_ok(const dbde_b200_ctx *c, const Request &r) {
    if (!c || !dims_ok(r.W, r.H, r.nframes)) return false;
    switch (r.form) {
    case Form::Region: return roi_ok(r.W, r.H, r.x0, r.y0, r.w, r.h);
    case Form::Crops: return crops_ok(r.ncrops, r.per_frame, r.w, r.h, r.pad, r.pad_max());
    case Form::Binned: return factor_ok(r.factor);
    default: return true;
    }
}

// Every argument rule of the decoders.  `out` is the frames, region, crops or bins (unused by Validate).  host: the
// buffers are in host memory; the offsets must then ascend within the stream.  0: run the request (nothing to run for
// an empty batch).
static int check_decode(const dbde_b200_ctx *c, const Request &r, const uint8_t *stream, size_t stream_bytes, const uint64_t *offs,
                        const void *out, const uint32_t *status, bool host) {
    // DBDE16 output is 2-byte aligned, but for decode16_host, which has always copied out of staging to any address
    const bool odd_ok = !r.u16 || (host && r.form == Form::Full);
    if (!request_ok(c, r) || (!odd_ok && ((uintptr_t)out & 1)) ||
        (r.nframes > 0 && (!stream || !offs || (!out && r.form != Form::Validate) || !status || (r.form == Form::Crops && !r.corners))))
        return reject(r, DBDE_B200_E_INVALID, "bad argument");
    if (host)
        for (int i = 0; i < r.nframes; i++) {
            const uint64_t end = i + 1 < r.nframes ? offs[i + 1] : stream_bytes;
            if (offs[i] > end || end > stream_bytes) return reject(r, DBDE_B200_E_INVALID, "frame offsets must ascend within the stream");
        }
    return 0;
}

// Every argument rule of the encoders.  slot_stride: the device forms' (0 picks the default and is replaced by it);
// null for the host forms, whose capacity can only be checked against the records' sizes once they are known.
static int check_encode(const dbde_b200_ctx *c, const Request &r, const void *frames, const uint8_t *out, size_t out_capacity,
                        size_t *slot_stride, const uint64_t *offs, const uint64_t *sizes) {
    const bool device = slot_stride != nullptr;
    // the device forms read DBDE16 frames in place, 2-byte aligned; the host forms copy them into staging first
    if (!request_ok(c, r) || (r.u16 && device && ((uintptr_t)frames & 1)) ||
        (r.nframes > 0 && (!frames || !out || !offs || (device && !sizes) || (r.form == Form::Crops && !r.corners))))
        return reject(r, DBDE_B200_E_INVALID, "bad argument");
    if (r.nframes == 0) return 0;
    const Fmt f = r.record_fmt();
    if (device) {
        if (*slot_stride == 0) *slot_stride = f.stride;
        if (*slot_stride < f.bound) return reject(r, DBDE_B200_E_INVALID, "slot_stride < the record bound");
    }
    const long long nrec = (long long)r.nframes * r.records();
    if (nrec > 0x7FFFFFFFLL) return reject(r, DBDE_B200_E_INVALID, "nframes * ncrops > 2^31 - 1");
    if (device && *slot_stride > out_capacity / (size_t)nrec)
        return reject(r, DBDE_B200_E_CAPACITY, "out_capacity < records * slot_stride");
    return 0;
}

// ------------------------------------------------------------------ the kernels of a request
// The frame encoders' look-back scratch on stream st, zeroed: [ticket | pad to 128][desc: nparts u64]
static int encode_scratch(dbde_b200_ctx *c, cudaStream_t st, const Request &r, unsigned long long nparts, unsigned int **ticket,
                          uint64_t **desc) {
    if (nparts >= 0xFFFFFFF0ull) return reject(r, DBDE_B200_E_INVALID, "batch too large");
    const size_t sbytes = 128 + 8 * (size_t)nparts;
    StreamScratch &sc = scratch_for(c, st);
    int rc = grow(&sc.enc, &sc.enc_bytes, sbytes);
    if (rc) return rc;
    CK(cudaMemsetAsync(sc.enc, 0, sbytes, st));
    *ticket = (unsigned int *)sc.enc;
    *desc = (uint64_t *)((uint8_t *)sc.enc + 128);
    return 0;
}

// the fields the 8-bit and DBDE16 crop encoders share
template <class P>
static P crop_params(const Request &r, const uint8_t *frames, uint64_t first_index, int n, const int32_t *corners, uint8_t *out,
                     size_t slot_stride, uint64_t *offs, uint64_t *sizes) {
    P p;
    p.frames = (decltype(p.frames))frames;
    p.W = r.W;
    p.H = r.H;
    p.corners = corners;
    p.ncrops = r.ncrops;
    p.corner_stride = r.per_frame ? r.ncrops : 0;
    p.crop_w = r.w;
    p.crop_h = r.h;
    p.w = (r.w + 7) / 8;
    p.wh = p.w * ((r.h + 7) / 8);
    p.out = out;
    p.slot_stride = slot_stride;
    p.frame_offsets = offs;
    p.frame_sizes = sizes;
    p.first_index = first_index;
    p.nrec = n * r.ncrops;
    return p;
}

// The encoder of a checked request for n frames at `frames` (device; Crops: the corners at `corners`, device), queued on st.
// A crop equal to the frame still runs the crop kernel: its records are the frame encoder's records, byte for byte.
static int enqueue_encode(dbde_b200_ctx *c, const Request &r, const uint8_t *frames, uint64_t first_index, int n, const int32_t *corners,
                          uint8_t *out, size_t slot_stride, uint64_t *offs, uint64_t *sizes, cudaStream_t st) {
    CK(cudaSetDevice(c->device));
    int rc = 0;
    if (r.form == Form::Crops && r.u16) {
        Enc16CropParams P = crop_params<Enc16CropParams>(r, frames, first_index, n, corners, out, slot_stride, offs, sizes);
        P.pad = (uint32_t)r.pad;
        CK(launch_encode16_crops(P, c->num_sms, st));
    } else if (r.form == Form::Crops) {
        EncCropParams P = crop_params<EncCropParams>(r, frames, first_index, n, corners, out, slot_stride, offs, sizes);
        P.pad8 = (uint64_t)r.pad * 0x0101010101010101ull;
        P.flags = c->invert_endian ? kFlagInvertRows : 0u;
        CK(launch_encode_crops(P, c->num_sms, st));
    } else if (r.u16) {
        Enc16Params P;
        P.W = r.W; P.H = r.H; P.w = (r.W + 7) / 8; P.h = (r.H + 7) / 8; P.wh = P.w * P.h;
        P.ppf = (P.wh + 255) / 256;
        const unsigned long long nparts = (unsigned long long)n * P.ppf;
        if ((rc = encode_scratch(c, st, r, nparts, &P.ticket, &P.desc))) return rc;
        P.frames = (const uint16_t *)frames; P.out = out; P.slot_stride = slot_stride;
        P.frame_offsets = offs; P.frame_sizes = sizes;
        P.first_index = first_index; P.nframes = n; P.nparts = (unsigned)nparts;
        P.aligned = (r.W % 8 == 0) && (((uintptr_t)frames & 15) == 0);
        CK(launch_encode16(P, c->num_sms, st));
    } else {
        const bool fast = (r.W % 16 == 0) && (r.H % 8 == 0) && (((uintptr_t)frames & 15) == 0);
        EncParams P;
        P.g = make_geom(r.W, r.H, fast);
        const unsigned long long nparts = (unsigned long long)n * P.g.ppf;
        if ((rc = encode_scratch(c, st, r, nparts, &P.ticket, &P.desc))) return rc;
        P.frames = frames;
        P.out = out;
        P.slot_stride = slot_stride;
        P.frame_offsets = offs;
        P.frame_sizes = sizes;
        P.first_index = first_index;
        P.nframes = n;
        P.nparts = (unsigned)nparts;
        P.flags = c->invert_endian ? kFlagInvertRows : 0u;
        CK(launch_encode(P, fast, c->num_sms, st));
    }
    c->launches += 1;
    return 0;
}

// The 8-bit validation pre-pass over geometry g, queued on st.  Its word-prefix table lives in the scratch of st.
// P->frames is what a full decode writes (null for the other forms).
static int decode_scan(dbde_b200_ctx *c, cudaStream_t st, const Request &r, const PartGeom &g, const uint8_t *stream_dev,
                       size_t stream_bytes, const uint64_t *frame_offsets_dev, int nframes, uint8_t *frames_dev, uint32_t *status_dev,
                       uint64_t *indices_dev, DecParams *P) {
    if ((unsigned long long)nframes * g.ppf >= 0xFFFFFFF0ull) return reject(r, DBDE_B200_E_INVALID, "batch too large");
    const size_t sbytes = 4 * (size_t)nframes * ((size_t)g.ppf * kConsumerWarps + 1);
    StreamScratch &sc = scratch_for(c, st);
    int rc = grow(&sc.dec, &sc.dec_bytes, sbytes);
    if (rc) return rc;
    P->g = g;
    P->stream = stream_dev;
    P->stream_bytes = stream_bytes;
    P->frame_offsets = frame_offsets_dev;
    P->frames = frames_dev;
    P->status = status_dev;
    P->indices = indices_dev;
    P->wprefix = (uint32_t *)sc.dec;
    P->nframes = nframes;
    P->nparts = (unsigned)((unsigned long long)nframes * g.ppf);
    P->flags = c->invert_endian ? kFlagInvertRows : 0u;
    CK(launch_decode_scan(*P, st));
    c->launches += 1;
    return 0;
}

// The DBDE16 validation pass (dbde16_scan_kernel: every check, over the whole record, and the word prefix of every
// 32 raster-order tiles), queued on st: the first launch of every DBDE16 decode.  P is what the second kernel reads;
// its output fields are left to the caller.
static int decode16_scan(dbde_b200_ctx *c, cudaStream_t st, const Request &r, const uint8_t *stream_dev, size_t stream_bytes,
                         const uint64_t *frame_offsets_dev, int nframes, uint32_t *status_dev, uint64_t *indices_dev, Dec16Params *P) {
    *P = Dec16Params();
    P->W = r.W; P->H = r.H; P->w = (r.W + 7) / 8; P->h = (r.H + 7) / 8; P->wh = P->w * P->h;
    P->ppf = (P->wh + 255) / 256;
    const unsigned long long nparts = (unsigned long long)nframes * P->ppf;
    if (nparts >= 0xFFFFFFF0ull) return reject(r, DBDE_B200_E_INVALID, "batch too large");
    const size_t sbytes = 4 * (size_t)nframes * ((size_t)(P->wh + 31) / 32 + 1);
    StreamScratch &sc = scratch_for(c, st);
    int rc = grow(&sc.dec, &sc.dec_bytes, sbytes);
    if (rc) return rc;
    P->stream = stream_dev; P->stream_bytes = stream_bytes; P->frame_offsets = frame_offsets_dev;
    P->status = status_dev; P->indices = indices_dev;
    P->wprefix = (uint32_t *)sc.dec;
    P->nframes = nframes; P->nparts = (unsigned)nparts;
    CK(launch_decode16_scan(*P, st));
    c->launches += 1;
    return 0;
}

// The kernels of a checked decode request for n records (Crops: the corners at `corners`, device), queued on st: the
// validation scan, then the pixels of the output form into `out`.  Validate stops after the scan.  The full decode's
// 8-bit scan runs on the geometry the full decoder picks from the output's alignment; the region, crop and binned
// decoders read a scan on linear partitions (dbde_roi.cu).  A region equal to the frame and factor 1 are the full
// decode; a crop equal to the frame still runs the crop kernel, whose output layout is the crop layout.
static int enqueue_decode(dbde_b200_ctx *c, const Request &r, const uint8_t *stream, size_t stream_bytes, const uint64_t *offs, int n,
                          const int32_t *corners, void *out, uint32_t *status, uint64_t *indices, cudaStream_t st) {
    CK(cudaSetDevice(c->device));
    Form form = r.form;
    if ((form == Form::Region && r.x0 == 0 && r.y0 == 0 && r.w == r.W && r.h == r.H) || (form == Form::Binned && r.factor == 1))
        form = Form::Full;
    const bool whole = form == Form::Full || form == Form::Validate;
    const bool fast = whole && (r.W % 16 == 0) && (r.H % 8 == 0) && (((uintptr_t)out & 15) == 0);
    uint8_t *out8 = (uint8_t *)out;
    uint16_t *out16 = (uint16_t *)out;
    DecParams D;
    Dec16Params P;
    int rc = r.u16 ? decode16_scan(c, st, r, stream, stream_bytes, offs, n, status, indices, &P)
                   : decode_scan(c, st, r, whole ? make_geom(r.W, r.H, fast) : linear_geom(r.W, r.H), stream, stream_bytes, offs, n,
                                 whole ? out8 : nullptr, status, indices, &D);
    if (rc) return rc;
    switch (form) {
    case Form::Validate:
        return 0;
    case Form::Full:
        if (r.u16) {
            P.frames = out16;
            P.aligned = (r.W % 8 == 0) && (((uintptr_t)out & 15) == 0);
            CK(launch_decode16(P, c->num_sms, st));
        } else {
            CK(launch_decode(D, fast, c->num_sms, st));
        }
        break;
    case Form::Region:          // 8-bit only
        CK(launch_decode_roi(D, r.x0, r.y0, r.w, r.h, out8, st));
        break;
    case Form::Crops:
        CK(r.u16 ? launch_decode16_crops(P, corners, r.ncrops, r.per_frame != 0, r.w, r.h, r.pad, out16, st)
                 : launch_decode_crops(D, corners, r.ncrops, r.per_frame != 0, r.w, r.h, r.pad, out8, st));
        break;
    case Form::Binned:
        CK(r.u16 ? launch_decode16_binned(P, r.factor, out16, c->num_sms, st) : launch_decode_binned(D, r.factor, out8, c->num_sms, st));
        break;
    }
    c->launches += 1;
    return 0;
}

// ------------------------------------------------------------------ device-resident hot path
static int encode_device(dbde_b200_ctx *c, const Request &r, const void *frames_dev, uint64_t first_index, uint8_t *out_dev,
                         size_t out_capacity, size_t slot_stride, uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    int rc = check_encode(c, r, frames_dev, out_dev, out_capacity, &slot_stride, frame_offsets_dev, frame_sizes_dev);
    if (rc || r.nframes == 0) return rc;
    return enqueue_encode(c, r, (const uint8_t *)frames_dev, first_index, r.nframes, r.corners, out_dev, slot_stride, frame_offsets_dev,
                          frame_sizes_dev, (cudaStream_t)stream);
}

static int decode_device(dbde_b200_ctx *c, const Request &r, const uint8_t *stream_dev, size_t stream_bytes,
                         const uint64_t *frame_offsets_dev, void *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    int rc = check_decode(c, r, stream_dev, stream_bytes, frame_offsets_dev, out_dev, status_dev, false);
    if (rc || r.nframes == 0) return rc;
    return enqueue_decode(c, r, stream_dev, stream_bytes, frame_offsets_dev, r.nframes, r.corners, out_dev, status_dev, indices_dev,
                          (cudaStream_t)stream);
}

extern "C" int dbde_b200_encode_device(dbde_b200_ctx *c, const uint8_t *frames_dev, int W, int H,
                                       uint64_t first_index, int nframes, uint8_t *out_dev, size_t out_capacity,
                                       size_t slot_stride, uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev,
                                       void *stream) {
    return encode_device(c, {"encode_device", false, Form::Full, W, H, nframes}, frames_dev, first_index, out_dev, out_capacity,
                         slot_stride, frame_offsets_dev, frame_sizes_dev, stream);
}

extern "C" int dbde_b200_decode_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                       const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                       uint8_t *frames_dev, uint32_t *status_dev, uint64_t *indices_dev,
                                       void *stream) {
    return decode_device(c, {"decode_device", false, Form::Full, W, H, nframes}, stream_dev, stream_bytes, frame_offsets_dev,
                         frames_dev, status_dev, indices_dev, stream);
}

// The indexer's optional GPU validation (SURVEY 8 f-2): the checks dbde_unpack_image makes before it
// touches the image (dbde_util.cpp:295-303: nb == wh, nm == wh, sum(depth) == n64; plus tag, depth <= 8,
// bounds), for every record of a device-resident stream, without decoding a pixel.
extern "C" int dbde_b200_validate_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                         const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                         uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"validate_device", false, Form::Validate, W, H, nframes}, stream_dev, stream_bytes, frame_offsets_dev,
                         nullptr, status_dev, indices_dev, stream);
}

// The scan, then one warp per 32 tile columns of each tile row of the region (dbde_roi.cu).
extern "C" int dbde_b200_decode_roi_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                           const uint64_t *frame_offsets_dev, int W, int H, int nframes, int x0, int y0,
                                           int roi_w, int roi_h, uint8_t *roi_dev, uint32_t *status_dev,
                                           uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"decode_roi_device", false, Form::Region, W, H, nframes, 0, x0, y0, roi_w, roi_h}, stream_dev,
                         stream_bytes, frame_offsets_dev, roi_dev, status_dev, indices_dev, stream);
}

// The region decode's scan and kernel body with one rectangle per task taken from `corners` (dbde_roi.cu).
extern "C" int dbde_b200_decode_crops_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                             const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                             const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint8_t *crops_dev, uint32_t *status_dev,
                                             uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"decode_crops_device", false, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_dev, ncrops,
                             corners_per_frame, pad},
                         stream_dev, stream_bytes, frame_offsets_dev, crops_dev, status_dev, indices_dev, stream);
}

// One CTA per record of a persistent grid, one lane per crop tile (dbde_encode.cu).
extern "C" int dbde_b200_encode_crops_device(dbde_b200_ctx *c, const uint8_t *frames_dev, int W, int H, uint64_t first_index,
                                             int nframes, const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint8_t *out_dev, size_t out_capacity, size_t slot_stride,
                                             uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    return encode_device(c, {"encode_crops_device", false, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_dev, ncrops,
                             corners_per_frame, pad},
                         frames_dev, first_index, out_dev, out_capacity, slot_stride, frame_offsets_dev, frame_sizes_dev, stream);
}

// The scan on linear partitions, then the full decoder's pipeline with each tile reduced to its block means in
// registers (dbde_decode.cu).
extern "C" int dbde_b200_decode_binned_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                              const uint64_t *frame_offsets_dev, int W, int H, int nframes, int factor,
                                              uint8_t *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"decode_binned_device", false, Form::Binned, W, H, nframes, factor}, stream_dev, stream_bytes,
                         frame_offsets_dev, out_dev, status_dev, indices_dev, stream);
}

// ------------------------------------------------------------------ DBDE16 (SURVEY 8 f-4)
extern "C" size_t dbde_b200_frame_record_bound16(int W, int H) {
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    return rec_bound(wh, 2);
}
extern "C" size_t dbde_b200_slot_stride16(int W, int H) { return (dbde_b200_frame_record_bound16(W, H) + 15) & ~(size_t)15; }

extern "C" int dbde_b200_encode16_device(dbde_b200_ctx *c, const uint16_t *frames_dev, int W, int H, uint64_t first_index,
                                         int nframes, uint8_t *out_dev, size_t out_capacity, size_t slot_stride,
                                         uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    return encode_device(c, {"encode16_device", true, Form::Full, W, H, nframes}, frames_dev, first_index, out_dev, out_capacity,
                         slot_stride, frame_offsets_dev, frame_sizes_dev, stream);
}

// One CTA per record of a persistent grid, one lane per crop tile (dbde16.cu): dbde_b200_encode_crops_device with U16
// pixels.
extern "C" int dbde_b200_encode16_crops_device(dbde_b200_ctx *c, const uint16_t *frames_dev, int W, int H, uint64_t first_index,
                                               int nframes, const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                               int crop_h, int pad, uint8_t *out_dev, size_t out_capacity, size_t slot_stride,
                                               uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    return encode_device(c, {"encode16_crops_device", true, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_dev, ncrops,
                             corners_per_frame, pad},
                         frames_dev, first_index, out_dev, out_capacity, slot_stride, frame_offsets_dev, frame_sizes_dev, stream);
}

extern "C" int dbde_b200_decode16_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                         const uint64_t *frame_offsets_dev, int W, int H, int nframes, uint16_t *frames_dev,
                                         uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"decode16_device", true, Form::Full, W, H, nframes}, stream_dev, stream_bytes, frame_offsets_dev,
                         frames_dev, status_dev, indices_dev, stream);
}

// The scan, then one warp per 32 tile columns of each tile row of each crop (dbde16.cu).
extern "C" int dbde_b200_decode16_crops_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                               const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                               const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                               int crop_h, int pad, uint16_t *crops_dev, uint32_t *status_dev,
                                               uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"decode16_crops_device", true, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_dev, ncrops,
                             corners_per_frame, pad},
                         stream_dev, stream_bytes, frame_offsets_dev, crops_dev, status_dev, indices_dev, stream);
}

// The scan, then the full decoder's partitions with each tile reduced to its bin means in registers (dbde16.cu).
extern "C" int dbde_b200_decode16_binned_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                                const uint64_t *frame_offsets_dev, int W, int H, int nframes, int factor,
                                                uint16_t *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    return decode_device(c, {"decode16_binned_device", true, Form::Binned, W, H, nframes, factor}, stream_dev, stream_bytes,
                         frame_offsets_dev, out_dev, status_dev, indices_dev, stream);
}

// ------------------------------------------------------------------ pageable host memory
// The reference's callers pass malloc'd buffers (dbde_util.h:24-35).  cudaMemcpyAsync on pageable memory
// goes through the driver's own staging at ~15 GB/s and blocks the caller, and one host thread's memcpy is
// no faster (~14 GB/s).  The library therefore relays pageable buffers itself through pinned bounce
// buffers: the bytes are cut into 256 KiB copy jobs that a small process-wide pool of copy threads AND
// every calling thread that is waiting for something execute, each stretch of finished pieces is sent with
// one DMA (H2D) / each DMA piece is copied out as soon as it has landed (D2H).  Every wait on this path --
// for one's own pieces, for a kernel, for a DMA -- is a helping wait: the waiting thread runs queued jobs
// (anyone's), so sixteen callers share the copying among themselves instead of spinning in the driver while
// the threads that hold their data are descheduled.  Nothing is page-locked behind the caller's back.
namespace {
bool is_pageable(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

constexpr size_t kCopyJobBytes = 256u << 10;      // one memcpy job
constexpr int kMaxCopyJobs = 64;                  // per relayed buffer (larger buffers use larger jobs)
constexpr int kMaxDmaPieces = 16;                 // D2H pieces per relayed buffer (one event each)
size_t copy_job_bytes(size_t n) {
    size_t job = kCopyJobBytes;
    while ((n + job - 1) / job > (size_t)kMaxCopyJobs) job *= 2;
    return job;
}
constexpr int kFlagKernels = kMaxDmaPieces;       // index of the "this chunk's kernels are done" flag
// wait for a completion flag, copying queued pieces meanwhile
void wait_flag_helping(volatile uint32_t *flag) {
    CopyPool::get().help_until([flag] { return *flag != 0u; });
    std::atomic_thread_fence(std::memory_order_acquire);       // the bytes the flag reports are read after it
}
}  // namespace

static bool h2d_streaming() {
    static const bool v = [] {
        const char *e = getenv("DBDE_B200_H2D_STREAMING");
        return !(e && e[0] == '0');
    }();
    return v;
}

static int ensure_bounce(dbde_b200_ctx *c, HostSlot &s, size_t need_in, size_t need_out) {
    if (need_in && s.cap_hin < need_in) {
        if (s.h_in) CK(cudaFreeHost(s.h_in));
        s.h_in = nullptr;
        CK(cudaHostAlloc(&s.h_in, need_in, cudaHostAllocDefault));
        s.cap_hin = need_in;
    }
    if (need_out && s.cap_hout < need_out) {
        if (s.h_out) CK(cudaFreeHost(s.h_out));
        s.h_out = nullptr;
        CK(cudaHostAlloc(&s.h_out, need_out, cudaHostAllocDefault));
        s.cap_hout = need_out;
    }
    if (!s.h_flag) {
        void *p = nullptr;
        CK(cudaHostAlloc(&p, 4 * (kMaxDmaPieces + 1), cudaHostAllocDefault));
        memset(p, 0, 4 * (kMaxDmaPieces + 1));
        s.h_flag = (volatile uint32_t *)p;
    }
    if (!c->d_one) {
        const uint32_t one = 1;
        CK(cudaMalloc(&c->d_one, 4));
        CK(cudaMemcpy(c->d_one, &one, 4, cudaMemcpyHostToDevice));
    }
    return 0;
}

// queue "set flag i" behind everything already on the slot's stream
static int signal_flag(dbde_b200_ctx *c, HostSlot &s, int i) {
    s.h_flag[i] = 0u;
    CK(cudaMemcpyAsync((void *)&s.h_flag[i], c->d_one, 4, cudaMemcpyDeviceToHost, s.st));
    return 0;
}

// pageable src -> device, through the slot's pinned h_in (at offset hoff), queued on the slot's stream.
// Returns when every piece's DMA is queued; the bounce bytes stay valid until the stream has passed them.
// Copy jobs are 256 KiB (many hands), DMAs at least 1 MiB (a DMA costs microseconds to start).
static int relay_h2d(HostSlot &s, uint8_t *d_dst, const uint8_t *src, size_t n, size_t hoff) {
    if (!n) return 0;
    CopyPool &pool = CopyPool::get();
    const size_t job = copy_job_bytes(n);
    const int nj = (int)((n + job - 1) / job);
    std::atomic<int> pend[kMaxCopyJobs];
    CopyPool::Job jobs[kMaxCopyJobs];
    for (int i = 0; i < nj; i++) {
        const size_t o = (size_t)i * job;
        pend[i].store(1, std::memory_order_relaxed);
        jobs[i] = CopyPool::Job{s.h_in + hoff + o, src + o, n - o < job ? n - o : job, &pend[i], (uint8_t)(h2d_streaming() ? CopyPool::kStreamingStores : CopyPool::kPlain)};
    }
    pool.submit(jobs, nj);
    static const size_t dma_min = [] {
        const char *e = getenv("DBDE_B200_H2D_DMA_KB");
        return (size_t)(e && atoi(e) > 0 ? atoi(e) : 1024) << 10;
    }();
    const int group = (int)((dma_min + job - 1) / job);      // jobs per DMA
    for (int i = 0; i < nj;) {
        int j = i + group < nj ? i + group : nj;
        for (int q = i; q < j; q++) pool.help_until([&] { return pend[q].load(std::memory_order_acquire) == 0; });
        while (j < nj && pend[j].load(std::memory_order_acquire) == 0) j++;      // whatever else is already there
        const size_t o0 = (size_t)i * job, o1 = j < nj ? (size_t)j * job : n;
        CK(cudaMemcpyAsync(d_dst + o0, s.h_in + hoff + o0, o1 - o0, cudaMemcpyHostToDevice, s.st));
        i = j;
    }
    return 0;
}

// device -> the slot's pinned h_out (at offset hoff), in DMA pieces with one completion flag each, queued on
// the slot's stream.  Returns the piece size; pieces k = 0 .. ceil(n / piece) - 1 report on h_flag[k].
// the DMA piece size for relaying up to n bytes (at most kMaxDmaPieces pieces, one completion flag each)
static size_t d2h_piece_bytes(size_t n) {
    static const size_t piece_min = [] {
        const char *e = getenv("DBDE_B200_D2H_DMA_KB");
        return (size_t)(e && atoi(e) > 0 ? atoi(e) : 1024) << 10;
    }();
    size_t piece = piece_min;
    while ((n + piece - 1) / piece > (size_t)kMaxDmaPieces) piece *= 2;
    return piece;
}
// pieces k_first, k_first + 1, ... of the first n bytes at d_src, each to its place in h_out and each followed by its flag
static int relay_d2h_enqueue_from(dbde_b200_ctx *c, HostSlot &s, const uint8_t *d_src, size_t n, size_t hoff, size_t piece,
                                  int k_first) {
    for (int k = k_first; (size_t)k * piece < n; k++) {
        const size_t o = (size_t)k * piece;
        CK(cudaMemcpyAsync(s.h_out + hoff + o, d_src + o, n - o < piece ? n - o : piece, cudaMemcpyDeviceToHost, s.st));
        int rc = signal_flag(c, s, k);
        if (rc) return rc;
    }
    return 0;
}
static int relay_d2h_enqueue(dbde_b200_ctx *c, HostSlot &s, const uint8_t *d_src, size_t n, size_t hoff, size_t *piece_out) {
    *piece_out = d2h_piece_bytes(n);
    return relay_d2h_enqueue_from(c, s, d_src, n, hoff, *piece_out, 0);
}
// ... and out of h_out into pageable memory as the pieces land: bytes [lo, hi) of the n relayed bytes go to
// dst + (their offset - lo).  Pieces are copied out by the pool and the waiting callers while later pieces
// are still crossing PCIe; `pend` counts the jobs (the caller waits for it once, after its last range).
static void relay_d2h_collect(HostSlot &s, uint8_t *dst, size_t lo, size_t hi, size_t n, size_t piece, size_t hoff,
                              std::atomic<int> &pend) {
    CopyPool &pool = CopyPool::get();
    const size_t job = copy_job_bytes(piece);
    for (size_t k = lo / piece; k * piece < hi && k * piece < n; k++) {
        wait_flag_helping(&s.h_flag[k]);
        const size_t p0 = k * piece > lo ? k * piece : lo, p1 = (k + 1) * piece < hi ? (k + 1) * piece : hi;
        CopyPool::Job jobs[kMaxCopyJobs + 1];
        int nj = 0;
        for (size_t q = p0; q < p1; q += job) jobs[nj++] = CopyPool::Job{dst + (q - lo), s.h_out + hoff + q, p1 - q < job ? p1 - q : job, &pend, (uint8_t)CopyPool::kPlain};
        pend.fetch_add(nj, std::memory_order_relaxed);
        pool.submit(jobs, nj);
    }
}
// device -> pageable dst.  Synchronous: the bytes are in dst on return.
static int relay_d2h(dbde_b200_ctx *c, HostSlot &s, uint8_t *dst, const uint8_t *d_src, size_t n, size_t hoff) {
    if (!n) return 0;
    size_t piece = 0;
    int rc = relay_d2h_enqueue(c, s, d_src, n, hoff, &piece);
    if (rc) return rc;
    std::atomic<int> pend{0};
    relay_d2h_collect(s, dst, 0, n, n, piece, hoff, pend);
    CopyPool::get().help_until([&] { return pend.load(std::memory_order_acquire) == 0; });
    return 0;
}

// ------------------------------------------------------------------ host-buffer hot path
// The 8-bit and DBDE16 host forms share one encode and one decode chunk pipeline (staging slots in flight, records
// compacted on the device, pageable buffers relayed through the copy pool); the request picks the kernels.
static int default_chunk(const dbde_b200_ctx *c, const Request &r) {
    int n = c->chunk_frames;
    if (n <= 0) {
        const size_t px = r.fmt(r.W, r.H).px;
        n = (int)((64u << 20) / (px ? px : 1));
        if (n < 1) n = 1;
    }
    if (n > r.nframes) n = r.nframes;
    return n;
}

static int ensure_slot(dbde_b200_ctx *c, HostSlot &s, size_t need_a, size_t need_b, size_t need_c, int n) {
    if (!s.st) CK(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
    if (!s.ev) CK(cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming));
    if (s.cap_a < need_a) {
        if (s.d_a) CK(cudaFree(s.d_a));
        s.d_a = nullptr;
        CK(cudaMalloc(&s.d_a, need_a));
        s.cap_a = need_a;
    }
    if (s.cap_b < need_b) {
        if (s.d_b) CK(cudaFree(s.d_b));
        s.d_b = nullptr;
        CK(cudaMalloc(&s.d_b, need_b));
        s.cap_b = need_b;
    }
    if (s.cap_c < need_c) {
        if (s.d_c) CK(cudaFree(s.d_c));
        s.d_c = nullptr;
        CK(cudaMalloc(&s.d_c, need_c));
        s.cap_c = need_c;
    }
    if (s.cap_n < n) {
        if (s.d_off) CK(cudaFree(s.d_off));
        if (s.d_size) CK(cudaFree(s.d_size));
        if (s.h_size) CK(cudaFreeHost(s.h_size));
        if (s.d_status) CK(cudaFree(s.d_status));
        if (s.d_index) CK(cudaFree(s.d_index));
        if (s.h_off) CK(cudaFreeHost(s.h_off));
        if (s.h_status) CK(cudaFreeHost(s.h_status));
        if (s.h_index) CK(cudaFreeHost(s.h_index));
        s.d_off = nullptr; s.d_size = nullptr; s.h_size = nullptr; s.d_status = nullptr; s.d_index = nullptr; s.h_off = nullptr;
        s.h_status = nullptr; s.h_index = nullptr;
        CK(cudaMalloc(&s.d_off, 8 * (size_t)(n + 1)));
        CK(cudaMalloc(&s.d_size, 8 * (size_t)(n + 1)));
        CK(cudaHostAlloc(&s.h_size, 8 * (size_t)(n + 1), cudaHostAllocDefault));
        CK(cudaMalloc(&s.d_status, 4 * (size_t)n));
        CK(cudaMalloc(&s.d_index, 8 * (size_t)n));
        CK(cudaHostAlloc(&s.h_off, 8 * (size_t)(n + 1), cudaHostAllocDefault));
        CK(cudaHostAlloc(&s.h_status, 4 * (size_t)(n + 1), cudaHostAllocDefault));
        CK(cudaHostAlloc(&s.h_index, 8 * (size_t)(n + 1), cudaHostAllocDefault));
        s.cap_n = n;
    }
    return 0;
}
// pinned staging of a chunk's crop corners
static int ensure_corner_staging(HostSlot &s, size_t need) {
    if (s.cap_hcorners >= need) return 0;
    if (s.h_corners) CK(cudaFreeHost(s.h_corners));
    s.h_corners = nullptr;
    s.cap_hcorners = 0;
    CK(cudaHostAlloc(&s.h_corners, need, cudaHostAllocDefault));
    s.cap_hcorners = need;
    return 0;
}

// Where the next chunk's records go in the output stream.  Chunks are claimed strictly in chunk
// order -- by one worker (plain encode_host) or by several (encode_host_sharded: chunk ci belongs to
// worker ci mod G) -- so the records land back to back without any pass over the bytes afterwards.
struct EncSequencer {
    std::atomic<int> next{0};      // the chunk whose position is claimed next
    std::atomic<int> err{0};       // first failure; waiting workers bail out on it
    size_t out_pos = 0;            // guarded by `next`
};


// Worker `my` of `nworkers`: encodes chunks my, my + nworkers, ... of the checked request r on context c.  Crops: every
// frame gives r.ncrops records of r.w x r.h instead of its own record; the chunk's corners travel behind its frames in
// the slot's frame buffer.
static int encode_host_worker(dbde_b200_ctx *c, const Request &r, const uint8_t *frames_host, uint64_t first_index,
                              uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host, int chunk, int my, int nworkers,
                              EncSequencer *seq) {
    CK(cudaSetDevice(c->device));
    const bool crops = r.form == Form::Crops;
    const int nframes = r.nframes;
    const Fmt F = r.record_fmt();                                      // the records' format
    const size_t px = r.fmt(r.W, r.H).px;                              // input bytes per frame
    const int per = r.records();                                       // records per frame
    const int nrec = chunk * per;                                      // records per chunk
    const size_t delta = F.delta;
    const size_t corner_at = (px * chunk + 15) & ~(size_t)15, need_corners = r.corner_bytes(chunk);
    const size_t need_a = crops ? corner_at + need_corners : px * chunk + 32, need_b = F.stream_bound(nrec) + 32;
    const int nchunks = (nframes + chunk - 1) / chunk;
    const int mine = nchunks > my ? (nchunks - my + nworkers - 1) / nworkers : 0;
    const int ns = mine < c->nslots ? mine : c->nslots;            // a one-frame call sets up one slot
    // pageable caller memory is relayed through pinned bounce buffers (see CopyPool)
    const bool in_pageable = is_pageable(frames_host), out_pageable = is_pageable(out_host);
    for (int i = 0; i < ns; i++) {
        int rc = ensure_slot(c, c->slots[i], need_a, need_b, nrec > 1 ? need_b : 0, nrec);
        if (!rc) rc = ensure_bounce(c, c->slots[i], in_pageable ? px * chunk : 0, out_pageable ? need_b : 0);
        if (!rc) rc = ensure_corner_staging(c->slots[i], need_corners);
        if (rc) return rc;
    }
    const size_t stride = F.stride;
    // One frame per call into pageable memory (the drop-in functions): the record's size is not known until the
    // kernel has run, but its first DMA piece can follow the kernel at once -- most records are longer than a piece.
    const size_t spec_piece = (nrec == 1 && out_pageable) ? d2h_piece_bytes(stride) : 0;
    // finish(): wait for a chunk's kernels, learn the record sizes, claim the chunk's place in the
    // stream, and queue ONE D2H copy of its records -- already laid back to back on the device
    // (a one-frame chunk's record is contiguous in its slot as it is: no compaction pass).
    auto finish = [&](int li) -> int {
        HostSlot &s = c->slots[li % ns];
        const int ci = my + li * nworkers;
        if (in_pageable || out_pageable) wait_flag_helping(&s.h_flag[kFlagKernels]);    // copy (anyone's pieces) while waiting
        else CK(cudaEventSynchronize(s.ev));
        g_enc_prof.mark(3, "gpu");
        g_enc_prof.gpu_collect();
        const int nr = s.n * per;
        uint64_t total = 0;
        for (int i = 0; i < nr; i++) total += s.h_size[i];
        while (seq->next.load(std::memory_order_acquire) != ci) {
            if (seq->err.load(std::memory_order_relaxed)) return DBDE_B200_E_INVALID;   // another worker failed
            std::this_thread::yield();
        }
        const size_t pos = seq->out_pos;
        if (pos + total > out_capacity) return fail(DBDE_B200_E_CAPACITY, "encode_host: out_capacity too small");
        seq->out_pos = pos + total;
        seq->next.store(ci + 1, std::memory_order_release);
        uint64_t run = pos;
        for (int i = 0; i < nr; i++) {
            frame_offsets_host[(size_t)s.first * per + i] = run;
            run += s.h_size[i];
        }
        const uint8_t *d_rec = nrec > 1 ? s.d_c : s.d_b + delta;
        if (out_pageable && spec_piece) {
            // the record's first piece has been on its way since the kernel was queued; now that the size is known
            // the remaining pieces follow, and everything up to `total` leaves the bounce buffer
            int rc = relay_d2h_enqueue_from(c, s, d_rec, total, 0, spec_piece, 1);
            if (rc) return rc;
            std::atomic<int> pend{0};
            relay_d2h_collect(s, out_host + pos, 0, total, total, spec_piece, 0, pend);
            CopyPool::get().help_until([&] { return pend.load(std::memory_order_acquire) == 0; });
            g_enc_prof.mark(4, "d2h");
            return 0;
        }
        if (out_pageable) {
            const int rc = relay_d2h(c, s, out_host + pos, d_rec, total, 0);
            g_enc_prof.mark(4, "d2h");
            return rc;
        }
        CK(cudaMemcpyAsync(out_host + pos, d_rec, total, cudaMemcpyDeviceToHost, s.st));
        return 0;
    };
    int pending = -1, rc_all = 0;
    PhaseProfile &prof = g_enc_prof;
    prof.calls++;
    prof.start();
    for (int li = 0; li < mine && !rc_all; li++) {
        HostSlot &s = c->slots[li % ns];
        const int ci = my + li * nworkers;
        CK(cudaStreamSynchronize(s.st));            // the slot's previous chunk has fully drained
        prof.mark(0, "setup");
        s.first = ci * chunk;
        s.n = nframes - s.first < chunk ? nframes - s.first : chunk;
        prof.gpu_mark(0, s.st);
        if (in_pageable) {
            rc_all = relay_h2d(s, s.d_a, frames_host + px * s.first, px * s.n, 0);
            if (rc_all) break;
        } else {
            CK(cudaMemcpyAsync(s.d_a, frames_host + px * s.first, px * s.n, cudaMemcpyHostToDevice, s.st));
        }
        if (crops) {
            // this chunk's corners (the staging is free: the slot's stream has drained)
            const size_t nb = r.corner_bytes(s.n);
            memcpy(s.h_corners, r.corners + (r.per_frame ? 2 * (size_t)r.ncrops * (size_t)s.first : 0), nb);
            CK(cudaMemcpyAsync(s.d_a + corner_at, s.h_corners, nb, cudaMemcpyHostToDevice, s.st));
        }
        prof.mark(1, "h2d");
        prof.gpu_mark(1, s.st);
        rc_all = enqueue_encode(c, r, s.d_a, first_index + s.first, s.n, (const int32_t *)(s.d_a + corner_at), s.d_b + delta, stride,
                                s.d_off, s.d_size, s.st);
        if (rc_all) break;
        prof.gpu_mark(2, s.st);
        CK(cudaMemcpyAsync(s.h_size, s.d_size, 8 * (size_t)s.n * per, cudaMemcpyDeviceToHost, s.st));
        if (crops && nrec > 1) {
            // thousands of records per chunk: the prefix once (into d_off, which the host does not read back)
            CK(launch_compact_prefixed(s.d_b + delta, stride, s.d_size, s.d_off, s.n * per, s.d_c, s.st));
            c->launches += 2;
        } else if (chunk > 1) {
            CK(launch_compact(s.d_b + delta, stride, s.d_size, s.n, s.d_c, s.st));
            c->launches += 1;
        }
        if (in_pageable || out_pageable) {
            rc_all = signal_flag(c, s, kFlagKernels);
            if (!rc_all && spec_piece)
                rc_all = relay_d2h_enqueue_from(c, s, s.d_b + delta, spec_piece < stride ? spec_piece : stride, 0, spec_piece, 0);
            if (rc_all) break;
        } else {
            CK(cudaEventRecord(s.ev, s.st));
        }
        prof.gpu_mark(3, s.st);
        prof.mark(2, "launch");
        if (pending >= 0) rc_all = finish(pending);
        pending = li;
    }
    if (!rc_all && pending >= 0) rc_all = finish(pending);
    for (auto &s : c->slots)
        if (s.st) cudaStreamSynchronize(s.st);
    prof.mark(5, "drain");
    return rc_all;
}

// The host form of an encode request: the chunk pipeline, for crops with ncrops records per frame.
static int encode_host(dbde_b200_ctx *c, const Request &r, const uint8_t *frames_host, uint64_t first_index, uint8_t *out_host,
                       size_t out_capacity, uint64_t *frame_offsets_host) {
    int rc = check_encode(c, r, frames_host, out_host, out_capacity, nullptr, frame_offsets_host, nullptr);
    if (rc) return rc;
    if (r.nframes == 0) {
        if (frame_offsets_host) frame_offsets_host[0] = 0;
        return 0;
    }
    int chunk = default_chunk(c, r);
    const size_t rec = (size_t)r.records() * r.record_fmt().stride;      // one frame's record slots
    if (rec > r.fmt(r.W, r.H).stride) {            // crops larger than the frame: a chunk's records stay within 64 MiB
        const size_t most = (64u << 20) / rec;
        if ((size_t)chunk > most) chunk = most > 0 ? (int)most : 1;
    }
    EncSequencer seq;
    rc = encode_host_worker(c, r, frames_host, first_index, out_host, out_capacity, frame_offsets_host, chunk, 0, 1, &seq);
    if (rc) return rc;
    frame_offsets_host[(size_t)r.nframes * r.records()] = seq.out_pos;
    return 0;
}

extern "C" int dbde_b200_encode_host(dbde_b200_ctx *c, const uint8_t *frames_host, int W, int H,
                                     uint64_t first_index, int nframes, uint8_t *out_host, size_t out_capacity,
                                     uint64_t *frame_offsets_host) {
    return encode_host(c, {"encode_host", false, Form::Full, W, H, nframes}, frames_host, first_index, out_host, out_capacity,
                       frame_offsets_host);
}

// The host forms of dbde_b200_encode_crops_device and dbde_b200_encode16_crops_device: each chunk's corners go up behind
// its frames.
extern "C" int dbde_b200_encode_crops_host(dbde_b200_ctx *c, const uint8_t *frames_host, int W, int H, uint64_t first_index,
                                           int nframes, const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                           int crop_h, int pad, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host) {
    return encode_host(c, {"encode_crops_host", false, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_host, ncrops,
                           corners_per_frame, pad},
                       frames_host, first_index, out_host, out_capacity, frame_offsets_host);
}

extern "C" int dbde_b200_encode16_host(dbde_b200_ctx *c, const uint16_t *frames_host, int W, int H, uint64_t first_index,
                                       int nframes, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host) {
    return encode_host(c, {"encode16_host", true, Form::Full, W, H, nframes}, (const uint8_t *)frames_host, first_index, out_host,
                       out_capacity, frame_offsets_host);
}

extern "C" int dbde_b200_encode16_crops_host(dbde_b200_ctx *c, const uint16_t *frames_host, int W, int H, uint64_t first_index,
                                             int nframes, const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host) {
    return encode_host(c, {"encode16_crops_host", true, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_host, ncrops,
                           corners_per_frame, pad},
                       (const uint8_t *)frames_host, first_index, out_host, out_capacity, frame_offsets_host);
}

// The host form of a decode request: the records cross PCIe whole, and what the request asks for comes back -- the
// frames, the region, the crops (each chunk's corners go up on its slot's stream) or the bins; nothing for Validate
// but 4 (+8) bytes per frame.
static int decode_host(dbde_b200_ctx *c, const Request &r, const uint8_t *stream_host, size_t stream_bytes,
                       const uint64_t *frame_offsets_host, void *out_host, uint32_t *status_host, uint64_t *indices_host) {
    int rc = check_decode(c, r, stream_host, stream_bytes, frame_offsets_host, out_host, status_host, true);
    if (rc || r.nframes == 0) return rc;
    CK(cudaSetDevice(c->device));
    const int nframes = r.nframes;
    const bool scan_only = r.form == Form::Validate;
    uint8_t *frames_host = (uint8_t *)out_host;
    const Fmt F = r.fmt(r.W, r.H);
    const size_t px = r.out_bytes();                 // output bytes per frame
    int chunk = default_chunk(c, r);
    if (px > F.px) {                                 // crops larger than the frame: a chunk's output stays within 64 MiB
        const size_t most = (64u << 20) / px;
        if ((size_t)chunk > most) chunk = most > 0 ? (int)most : 1;
    }
    const size_t delta = F.delta;
    const int nchunks = (nframes + chunk - 1) / chunk;
    size_t need_a = 0;
    for (int ci = 0; ci < nchunks; ci++) {
        const int first = ci * chunk, n = nframes - first < chunk ? nframes - first : chunk;
        const uint64_t b0 = frame_offsets_host[first];
        const uint64_t b1 = first + n < nframes ? frame_offsets_host[first + n] : stream_bytes;
        if (b1 - b0 > need_a) need_a = b1 - b0;
    }
    need_a += 64;
    // Size the stream staging for the worst case of this geometry, not for this call's records: a caller
    // that decodes frame after frame (the drop-in dbde_unpack_frame, the file walker) would otherwise
    // pay a cudaFree + cudaMalloc every time a record is larger than any before it.
    const size_t bound_a = F.stream_bound(chunk) + 64;
    if (need_a < bound_a) need_a = bound_a;
    const size_t need_b = scan_only ? 0 : px * chunk + 32;
    const int ns = nchunks < c->nslots ? nchunks : c->nslots;
    // pageable caller memory is relayed through pinned bounce buffers (see CopyPool)
    const bool in_pageable = is_pageable(stream_host), out_pageable = !scan_only && is_pageable(frames_host);
    const size_t need_corners = r.corner_bytes(chunk);
    for (int i = 0; i < ns; i++) {
        HostSlot &s = c->slots[i];
        int rc = ensure_slot(c, s, need_a, need_b, need_corners, chunk);
        if (!rc) rc = ensure_bounce(c, s, in_pageable ? need_a : 0, out_pageable ? px * chunk : 0);
        if (!rc) rc = ensure_corner_staging(s, need_corners);
        if (rc) return rc;
    }
    // finish(): wait for a chunk's status words, then queue the D2H of its accepted frames.  A
    // rejected frame must leave the caller's image untouched (dbde_util.cpp:296-303), so pixels
    // come back as maximal runs of accepted frames.
    auto finish = [&](int ci) -> int {
        HostSlot &s = c->slots[ci % ns];
        if (in_pageable || out_pageable) wait_flag_helping(&s.h_flag[kFlagKernels]);
        else CK(cudaEventSynchronize(s.ev));
        g_dec_prof.mark(3, "gpu");
        memcpy(status_host + s.first, s.h_status, 4 * (size_t)s.n);
        if (indices_host) memcpy(indices_host + s.first, s.h_index, 8 * (size_t)s.n);
        if (scan_only) return 0;
        // pageable output: the chunk's pixels are already on their way to the bounce buffer (queued right
        // behind the kernels, before the status words were known); only accepted frames leave it
        std::atomic<int> pend{0};
        int run0 = 0;
        for (int i = 0; i <= s.n; i++) {
            const bool ok = i < s.n && s.h_status[i] == 0;
            if (!ok) {
                if (i > run0) {
                    const size_t bytes = px * (size_t)(i - run0);
                    if (out_pageable) {
                        relay_d2h_collect(s, frames_host + px * (s.first + run0), px * run0, px * run0 + bytes, px * s.n, s.piece, 0, pend);
                    } else {
                        CK(cudaMemcpyAsync(frames_host + px * (s.first + run0), s.d_b + px * run0, bytes, cudaMemcpyDeviceToHost, s.st));
                    }
                }
                run0 = i + 1;
            }
        }
        if (out_pageable) CopyPool::get().help_until([&] { return pend.load(std::memory_order_acquire) == 0; });
        g_dec_prof.mark(4, "d2h");
        return 0;
    };
    int pending = -1, rc_all = 0;
    PhaseProfile &prof = g_dec_prof;
    prof.calls++;
    prof.start();
    for (int ci = 0; ci < nchunks && !rc_all; ci++) {
        HostSlot &s = c->slots[ci % ns];
        CK(cudaStreamSynchronize(s.st));
        prof.mark(0, "setup");
        s.first = ci * chunk;
        s.n = nframes - s.first < chunk ? nframes - s.first : chunk;
        const uint64_t b0 = frame_offsets_host[s.first];
        const uint64_t b1 = s.first + s.n < nframes ? frame_offsets_host[s.first + s.n] : stream_bytes;
        for (int i = 0; i < s.n; i++) s.h_off[i] = frame_offsets_host[s.first + i] - b0;
        CK(cudaMemcpyAsync(s.d_off, s.h_off, 8 * (size_t)s.n, cudaMemcpyHostToDevice, s.st));
        if (in_pageable) {
            rc_all = relay_h2d(s, s.d_a + delta, stream_host + b0, b1 - b0, 0);
            if (rc_all) break;
        } else {
            CK(cudaMemcpyAsync(s.d_a + delta, stream_host + b0, b1 - b0, cudaMemcpyHostToDevice, s.st));
        }
        if (r.form == Form::Crops) {
            // this chunk's corners (the staging is free: the slot's stream has drained)
            const size_t nb = r.corner_bytes(s.n);
            memcpy(s.h_corners, r.corners + (r.per_frame ? 2 * (size_t)r.ncrops * (size_t)s.first : 0), nb);
            CK(cudaMemcpyAsync(s.d_c, s.h_corners, nb, cudaMemcpyHostToDevice, s.st));
        }
        prof.mark(1, "h2d");
        rc_all = enqueue_decode(c, r, s.d_a + delta, b1 - b0, s.d_off, s.n, (const int32_t *)s.d_c, s.d_b, s.d_status, s.d_index, s.st);
        if (rc_all) break;
        CK(cudaMemcpyAsync(s.h_status, s.d_status, 4 * (size_t)s.n, cudaMemcpyDeviceToHost, s.st));
        if (indices_host) CK(cudaMemcpyAsync(s.h_index, s.d_index, 8 * (size_t)s.n, cudaMemcpyDeviceToHost, s.st));
        if (in_pageable || out_pageable) {
            rc_all = signal_flag(c, s, kFlagKernels);
            if (!rc_all && out_pageable && !scan_only) rc_all = relay_d2h_enqueue(c, s, s.d_b, px * (size_t)s.n, 0, &s.piece);
            if (rc_all) break;
        } else {
            CK(cudaEventRecord(s.ev, s.st));
        }
        prof.mark(2, "launch");
        if (pending >= 0) rc_all = finish(pending);
        pending = ci;
    }
    if (!rc_all && pending >= 0) rc_all = finish(pending);
    for (auto &s : c->slots)
        if (s.st) cudaStreamSynchronize(s.st);
    prof.mark(5, "drain");
    return rc_all;
}

extern "C" int dbde_b200_decode_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                     const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                     uint8_t *frames_host, uint32_t *status_host, uint64_t *indices_host) {
    return decode_host(c, {"decode_host", false, Form::Full, W, H, nframes}, stream_host, stream_bytes, frame_offsets_host, frames_host,
                       status_host, indices_host);
}

extern "C" int dbde_b200_decode_roi_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                         const uint64_t *frame_offsets_host, int W, int H, int nframes, int x0, int y0,
                                         int roi_w, int roi_h, uint8_t *roi_host, uint32_t *status_host,
                                         uint64_t *indices_host) {
    return decode_host(c, {"decode_roi_host", false, Form::Region, W, H, nframes, 0, x0, y0, roi_w, roi_h}, stream_host, stream_bytes,
                       frame_offsets_host, roi_host, status_host, indices_host);
}

extern "C" int dbde_b200_decode_crops_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                           const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                           const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                           int crop_h, int pad, uint8_t *crops_host, uint32_t *status_host,
                                           uint64_t *indices_host) {
    return decode_host(c, {"decode_crops_host", false, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_host, ncrops,
                           corners_per_frame, pad},
                       stream_host, stream_bytes, frame_offsets_host, crops_host, status_host, indices_host);
}

extern "C" int dbde_b200_decode_binned_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                            const uint64_t *frame_offsets_host, int W, int H, int nframes, int factor,
                                            uint8_t *out_host, uint32_t *status_host, uint64_t *indices_host) {
    return decode_host(c, {"decode_binned_host", false, Form::Binned, W, H, nframes, factor}, stream_host, stream_bytes,
                       frame_offsets_host, out_host, status_host, indices_host);
}

extern "C" int dbde_b200_validate_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                       const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                       uint32_t *status_host, uint64_t *indices_host) {
    return decode_host(c, {"validate_host", false, Form::Validate, W, H, nframes}, stream_host, stream_bytes, frame_offsets_host,
                       nullptr, status_host, indices_host);
}

extern "C" int dbde_b200_decode16_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                       const uint64_t *frame_offsets_host, int W, int H, int nframes, uint16_t *frames_host,
                                       uint32_t *status_host, uint64_t *indices_host) {
    return decode_host(c, {"decode16_host", true, Form::Full, W, H, nframes}, stream_host, stream_bytes, frame_offsets_host,
                       frames_host, status_host, indices_host);
}

extern "C" int dbde_b200_decode16_crops_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                             const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                             const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint16_t *crops_host, uint32_t *status_host,
                                             uint64_t *indices_host) {
    return decode_host(c, {"decode16_crops_host", true, Form::Crops, W, H, nframes, 0, 0, 0, crop_w, crop_h, corners_host, ncrops,
                           corners_per_frame, pad},
                       stream_host, stream_bytes, frame_offsets_host, crops_host, status_host, indices_host);
}

extern "C" int dbde_b200_decode16_binned_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                              const uint64_t *frame_offsets_host, int W, int H, int nframes, int factor,
                                              uint16_t *out_host, uint32_t *status_host, uint64_t *indices_host) {
    return decode_host(c, {"decode16_binned_host", true, Form::Binned, W, H, nframes, factor}, stream_host, stream_bytes,
                       frame_offsets_host, out_host, status_host, indices_host);
}

// ------------------------------------------------------------------ multi-GPU sharding
// contiguous frame ranges, one host thread per context; there is no cross-GPU exchange on the
// data path, the host only prefix-sums the shard sizes (SURVEY.md section 8e)
extern "C" int dbde_b200_encode_host_sharded(dbde_b200_ctx **ctxs, int nctx, const uint8_t *frames_host, int W,
                                             int H, uint64_t first_index, int nframes, uint8_t *out_host,
                                             size_t out_capacity, uint64_t *frame_offsets_host) {
    const Request r = {"encode_host_sharded", false, Form::Full, W, H, nframes};
    if (!ctxs || nctx < 1) return reject(r, DBDE_B200_E_INVALID, "bad argument");
    for (int g = 0; g < nctx; g++)
        if (!ctxs[g]) return reject(r, DBDE_B200_E_INVALID, "null context");
    if (int bad = check_encode(ctxs[0], r, frames_host, out_host, out_capacity, nullptr, frame_offsets_host, nullptr)) return bad;
    if (nframes == 0) {
        if (frame_offsets_host) frame_offsets_host[0] = 0;
        return 0;
    }
    // The batch is cut into contiguous frame ranges of one chunk each; range ci goes to context
    // ci mod G.  Every context streams its ranges over its own PCIe link, and the ranges' records are
    // placed in stream order as their sizes become known (EncSequencer): the stream is complete when
    // the last copy lands -- no shard is moved afterwards.
    const int chunk = default_chunk(ctxs[0], r);
    EncSequencer seq;
    std::vector<int> rc(nctx, 0);
    std::vector<std::string> err(nctx);
    std::vector<std::thread> th;
    for (int g = 0; g < nctx; g++) {
        th.emplace_back([&, g]() {
            rc[g] = encode_host_worker(ctxs[g], r, frames_host, first_index, out_host, out_capacity, frame_offsets_host, chunk, g,
                                       nctx, &seq);
            if (rc[g]) {
                err[g] = dbde_b200_last_error();
                seq.err.store(rc[g], std::memory_order_relaxed);
            }
        });
    }
    for (auto &t : th) t.join();
    for (int g = 0; g < nctx; g++)
        if (rc[g] && !err[g].empty()) return fail(rc[g], err[g].c_str());
    for (int g = 0; g < nctx; g++)
        if (rc[g]) return fail(rc[g], "encode_host_sharded: a worker failed");
    frame_offsets_host[nframes] = seq.out_pos;
    return 0;
}

extern "C" int dbde_b200_decode_host_sharded(dbde_b200_ctx **ctxs, int nctx, const uint8_t *stream_host,
                                             size_t stream_bytes, const uint64_t *frame_offsets_host, int W, int H,
                                             int nframes, uint8_t *frames_host, uint32_t *status_host,
                                             uint64_t *indices_host) {
    if (!ctxs || nctx < 1 || !dims_ok(W, H, nframes)) return fail(DBDE_B200_E_INVALID, "decode_host_sharded: bad argument");
    if (nctx == 1 || nframes < nctx)
        return dbde_b200_decode_host(ctxs[0], stream_host, stream_bytes, frame_offsets_host, W, H, nframes, frames_host,
                                     status_host, indices_host);
    const size_t px = (size_t)W * H;
    std::vector<int> rc(nctx, 0);
    std::vector<std::string> err(nctx);
    std::vector<std::thread> th;
    for (int g = 0; g < nctx; g++) {
        th.emplace_back([&, g]() {
            const int a = (int)((long long)nframes * g / nctx), b = (int)((long long)nframes * (g + 1) / nctx);
            // a shard's records end where the next shard's begin
            const uint64_t base = frame_offsets_host[a];
            const uint64_t end = b < nframes ? frame_offsets_host[b] : stream_bytes;
            std::vector<uint64_t> rel(b - a);
            for (int i = a; i < b; i++) rel[i - a] = frame_offsets_host[i] - base;
            rc[g] = dbde_b200_decode_host(ctxs[g], stream_host + base, end - base, rel.data(), W, H, b - a,
                                          frames_host + px * a, status_host + a, indices_host ? indices_host + a : nullptr);
            if (rc[g]) err[g] = dbde_b200_last_error();
        });
    }
    for (auto &t : th) t.join();
    for (int g = 0; g < nctx; g++)
        if (rc[g]) return fail(rc[g], err[g].c_str());
    return 0;
}

// ------------------------------------------------------------------ host indexer
// minbytes: bytes per tile in the minimum plane (1: the reference's records, 2: DBDE16)
static long index_stream_impl(const uint8_t *p, size_t bytes, int W, int H, uint64_t *offs, long max_frames, size_t minbytes) {
    if (!p || !offs || !dims_ok(W, H, 0)) return fail(DBDE_B200_E_INVALID, "index_stream: bad argument");
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    const size_t fixed = rec_fixed(wh, minbytes);
    size_t cur = 0;
    long n = 0;
    while (cur + fixed <= bytes && n < max_frames) {
        uint32_t n64;
        memcpy(&n64, p + cur + rec_n64(wh, minbytes), 4);
        const size_t next = cur + fixed + 8 * (size_t)n64;
        if (next > bytes) break;
        offs[n++] = cur;
        cur = next;
    }
    offs[n] = cur;
    return n;
}
extern "C" long dbde_b200_index_stream(const uint8_t *p, size_t bytes, int W, int H, uint64_t *offs, long max_frames) {
    return index_stream_impl(p, bytes, W, H, offs, max_frames, 1);
}
extern "C" long dbde_b200_index_stream16(const uint8_t *p, size_t bytes, int W, int H, uint64_t *offs, long max_frames) {
    return index_stream_impl(p, bytes, W, H, offs, max_frames, 2);
}
