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
    const long long wh = (long long)((W + 7) / 8) * ((H + 7) / 8);
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
    return 32 + 66 * wh;
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

// ------------------------------------------------------------------ device-resident hot path
extern "C" int dbde_b200_encode_device(dbde_b200_ctx *c, const uint8_t *frames_dev, int W, int H,
                                       uint64_t first_index, int nframes, uint8_t *out_dev, size_t out_capacity,
                                       size_t slot_stride, uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev,
                                       void *stream) {
    if (!c || !dims_ok(W, H, nframes) ||
        (nframes > 0 && (!frames_dev || !out_dev || !frame_offsets_dev || !frame_sizes_dev)))
        return fail(DBDE_B200_E_INVALID, "encode_device: bad argument");
    if (nframes == 0) return 0;
    if (slot_stride == 0) slot_stride = dbde_b200_slot_stride(W, H);
    if (slot_stride < dbde_b200_frame_record_bound(W, H))
        return fail(DBDE_B200_E_INVALID, "encode_device: slot_stride < dbde_b200_frame_record_bound()");
    if (out_capacity < slot_stride * (size_t)nframes)
        return fail(DBDE_B200_E_CAPACITY, "encode_device: out_capacity < nframes * slot_stride");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool fast = (W % 16 == 0) && (H % 8 == 0) && (((uintptr_t)frames_dev & 15) == 0);
    EncParams P;
    P.g = make_geom(W, H, fast);
    const unsigned long long nparts = (unsigned long long)nframes * P.g.ppf;
    if (nparts >= 0xFFFFFFF0ull) return fail(DBDE_B200_E_INVALID, "encode_device: batch too large");
    // scratch: [ticket | pad to 128][desc: nparts u64], zeroed per launch
    const size_t sbytes = 128 + 8 * (size_t)nparts;
    StreamScratch &sc = scratch_for(c, st);
    int rc = grow(&sc.enc, &sc.enc_bytes, sbytes);
    if (rc) return rc;
    CK(cudaMemsetAsync(sc.enc, 0, sbytes, st));
    P.frames = frames_dev;
    P.out = out_dev;
    P.slot_stride = slot_stride;
    P.frame_offsets = frame_offsets_dev;
    P.frame_sizes = frame_sizes_dev;
    P.ticket = (unsigned int *)sc.enc;
    P.desc = (uint64_t *)((uint8_t *)sc.enc + 128);
    P.first_index = first_index;
    P.nframes = nframes;
    P.nparts = (unsigned)nparts;
    P.flags = c->invert_endian ? kFlagInvertRows : 0u;
    CK(launch_encode(P, fast, c->num_sms, st));
    c->launches += 1;
    return 0;
}

// The validation pre-pass over geometry g.  Its word-prefix table lives in the scratch of stream st.  P->frames
// is left null.
static int scan_params(dbde_b200_ctx *c, cudaStream_t st, const PartGeom &g, const uint8_t *stream_dev, size_t stream_bytes,
                       const uint64_t *frame_offsets_dev, int nframes, uint32_t *status_dev, uint64_t *indices_dev,
                       DecParams *P) {
    const size_t sbytes = 4 * (size_t)nframes * ((size_t)g.ppf * kConsumerWarps + 1);
    StreamScratch &sc = scratch_for(c, st);
    int rc = grow(&sc.dec, &sc.dec_bytes, sbytes);
    if (rc) return rc;
    P->g = g;
    P->stream = stream_dev;
    P->stream_bytes = stream_bytes;
    P->frame_offsets = frame_offsets_dev;
    P->frames = nullptr;
    P->status = status_dev;
    P->indices = indices_dev;
    P->wprefix = (uint32_t *)sc.dec;
    P->nframes = nframes;
    P->nparts = (unsigned)((unsigned long long)nframes * g.ppf);
    P->flags = c->invert_endian ? kFlagInvertRows : 0u;
    return 0;
}

// scan_only: run the validation pre-pass alone (status + indices, no pixels): dbde_b200_validate_*
static int decode_device_impl(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                              const uint64_t *frame_offsets_dev, int W, int H, int nframes, uint8_t *frames_dev,
                              uint32_t *status_dev, uint64_t *indices_dev, void *stream, bool scan_only) {
    if (!c || !dims_ok(W, H, nframes) ||
        (nframes > 0 && (!stream_dev || !frame_offsets_dev || (!frames_dev && !scan_only) || !status_dev)))
        return fail(DBDE_B200_E_INVALID, "decode_device: bad argument");
    if (nframes == 0) return 0;
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool fast = (W % 16 == 0) && (H % 8 == 0) && (((uintptr_t)frames_dev & 15) == 0);
    const PartGeom g = make_geom(W, H, fast);
    if ((unsigned long long)nframes * g.ppf >= 0xFFFFFFF0ull) return fail(DBDE_B200_E_INVALID, "decode_device: batch too large");
    DecParams P;
    int rc = scan_params(c, st, g, stream_dev, stream_bytes, frame_offsets_dev, nframes, status_dev, indices_dev, &P);
    if (rc) return rc;
    P.frames = frames_dev;
    CK(launch_decode_scan(P, st));
    c->launches += 1;
    if (scan_only) return 0;
    CK(launch_decode(P, fast, c->num_sms, st));
    c->launches += 1;
    return 0;
}

extern "C" int dbde_b200_decode_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                       const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                       uint8_t *frames_dev, uint32_t *status_dev, uint64_t *indices_dev,
                                       void *stream) {
    return decode_device_impl(c, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, frames_dev, status_dev,
                              indices_dev, stream, false);
}

// The indexer's optional GPU validation (SURVEY 8 f-2): the checks dbde_unpack_image makes before it
// touches the image (dbde_util.cpp:295-303: nb == wh, nm == wh, sum(depth) == n64; plus tag, depth <= 8,
// bounds), for every record of a device-resident stream, without decoding a pixel.
extern "C" int dbde_b200_validate_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                         const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                         uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    return decode_device_impl(c, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, nullptr, status_dev,
                              indices_dev, stream, true);
}

// ------------------------------------------------------------------ region of interest
static bool roi_ok(int W, int H, int x0, int y0, int roi_w, int roi_h) {
    return x0 >= 0 && y0 >= 0 && roi_w >= 1 && roi_h >= 1 && (long long)x0 + roi_w <= W && (long long)y0 + roi_h <= H;
}

// The validation pre-pass on linear partitions (every check of the full decode, over the whole record), queued on
// st: the first launch of the region and crop decodes.  D is what their kernels read.
static int linear_scan(dbde_b200_ctx *c, cudaStream_t st, int W, int H, const uint8_t *stream_dev, size_t stream_bytes,
                       const uint64_t *frame_offsets_dev, int nframes, uint32_t *status_dev, uint64_t *indices_dev, DecParams *D) {
    CK(cudaSetDevice(c->device));
    int rc = scan_params(c, st, linear_geom(W, H), stream_dev, stream_bytes, frame_offsets_dev, nframes, status_dev, indices_dev, D);
    if (rc) return rc;
    CK(launch_decode_scan(*D, st));
    c->launches += 1;
    return 0;
}

// The scan, then one warp per 32 tile columns of each tile row of the region (dbde_roi.cu).  A region equal to the
// frame is the full decode.
extern "C" int dbde_b200_decode_roi_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                           const uint64_t *frame_offsets_dev, int W, int H, int nframes, int x0, int y0,
                                           int roi_w, int roi_h, uint8_t *roi_dev, uint32_t *status_dev,
                                           uint64_t *indices_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !roi_ok(W, H, x0, y0, roi_w, roi_h) ||
        (nframes > 0 && (!stream_dev || !frame_offsets_dev || !roi_dev || !status_dev)))
        return fail(DBDE_B200_E_INVALID, "decode_roi_device: bad argument");
    if (nframes == 0) return 0;
    if (x0 == 0 && y0 == 0 && roi_w == W && roi_h == H)
        return decode_device_impl(c, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, roi_dev, status_dev,
                                  indices_dev, stream, false);
    DecParams D;
    int rc = linear_scan(c, (cudaStream_t)stream, W, H, stream_dev, stream_bytes, frame_offsets_dev, nframes, status_dev,
                         indices_dev, &D);
    if (rc) return rc;
    CK(launch_decode_roi(D, x0, y0, roi_w, roi_h, roi_dev, (cudaStream_t)stream));
    c->launches += 1;
    return 0;
}

// ------------------------------------------------------------------ crops
// pad_max: 255 for 8-bit frames, 65535 for DBDE16; the size limit counts pixels whatever their width
static bool crops_ok(int ncrops, int corners_per_frame, int crop_w, int crop_h, int pad, int pad_max = 255) {
    return ncrops >= 1 && crop_w >= 1 && crop_h >= 1 && dims_ok(crop_w, crop_h, 0) &&
           (long long)ncrops * crop_w * crop_h <= 0x7FFFFFFFLL && (corners_per_frame == 0 || corners_per_frame == 1) && pad >= 0 &&
           pad <= pad_max;
}

// The region decode's scan and kernel body with one rectangle per task taken from `corners` (dbde_roi.cu).  A crop
// equal to the frame still runs the crop kernel: its output layout is the crop layout whatever the corners.
extern "C" int dbde_b200_decode_crops_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                             const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                             const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint8_t *crops_dev, uint32_t *status_dev,
                                             uint64_t *indices_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad) ||
        (nframes > 0 && (!stream_dev || !frame_offsets_dev || !corners_dev || !crops_dev || !status_dev)))
        return fail(DBDE_B200_E_INVALID, "decode_crops_device: bad argument");
    if (nframes == 0) return 0;
    DecParams D;
    int rc = linear_scan(c, (cudaStream_t)stream, W, H, stream_dev, stream_bytes, frame_offsets_dev, nframes, status_dev,
                         indices_dev, &D);
    if (rc) return rc;
    CK(launch_decode_crops(D, corners_dev, ncrops, corners_per_frame != 0, crop_w, crop_h, pad, crops_dev, (cudaStream_t)stream));
    c->launches += 1;
    return 0;
}

// One CTA per record of a persistent grid, one lane per crop tile (dbde_encode.cu).  A crop equal to the frame still
// runs the crop kernel: its records are the frame encoder's records, byte for byte.
extern "C" int dbde_b200_encode_crops_device(dbde_b200_ctx *c, const uint8_t *frames_dev, int W, int H, uint64_t first_index,
                                             int nframes, const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint8_t *out_dev, size_t out_capacity, size_t slot_stride,
                                             uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad) ||
        (nframes > 0 && (!frames_dev || !corners_dev || !out_dev || !frame_offsets_dev || !frame_sizes_dev)))
        return fail(DBDE_B200_E_INVALID, "encode_crops_device: bad argument");
    if (nframes == 0) return 0;
    if (slot_stride == 0) slot_stride = dbde_b200_slot_stride(crop_w, crop_h);
    if (slot_stride < dbde_b200_frame_record_bound(crop_w, crop_h))
        return fail(DBDE_B200_E_INVALID, "encode_crops_device: slot_stride < dbde_b200_frame_record_bound(crop_w, crop_h)");
    const long long nrec = (long long)nframes * ncrops;
    if (nrec > 0x7FFFFFFFLL) return fail(DBDE_B200_E_INVALID, "encode_crops_device: nframes * ncrops > 2^31 - 1");
    if (slot_stride > out_capacity / (size_t)nrec)
        return fail(DBDE_B200_E_CAPACITY, "encode_crops_device: out_capacity < nframes * ncrops * slot_stride");
    CK(cudaSetDevice(c->device));
    EncCropParams P;
    P.frames = frames_dev;
    P.W = W;
    P.H = H;
    P.corners = corners_dev;
    P.ncrops = ncrops;
    P.corner_stride = corners_per_frame ? ncrops : 0;
    P.crop_w = crop_w;
    P.crop_h = crop_h;
    P.w = (crop_w + 7) / 8;
    P.wh = P.w * ((crop_h + 7) / 8);
    P.pad8 = (uint64_t)pad * 0x0101010101010101ull;
    P.out = out_dev;
    P.slot_stride = slot_stride;
    P.frame_offsets = frame_offsets_dev;
    P.frame_sizes = frame_sizes_dev;
    P.first_index = first_index;
    P.nrec = (int)nrec;
    P.flags = c->invert_endian ? kFlagInvertRows : 0u;
    CK(launch_encode_crops(P, c->num_sms, (cudaStream_t)stream));
    c->launches += 1;
    return 0;
}

// ------------------------------------------------------------------ binned
static bool factor_ok(int factor) { return factor == 1 || factor == 2 || factor == 4 || factor == 8; }

// The scan on linear partitions, then the full decoder's pipeline with each tile reduced to its block means in
// registers (dbde_decode.cu).  Factor 1 is the full decode.
extern "C" int dbde_b200_decode_binned_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                              const uint64_t *frame_offsets_dev, int W, int H, int nframes, int factor,
                                              uint8_t *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !factor_ok(factor) ||
        (nframes > 0 && (!stream_dev || !frame_offsets_dev || !out_dev || !status_dev)))
        return fail(DBDE_B200_E_INVALID, "decode_binned_device: bad argument");
    if (nframes == 0) return 0;
    if (factor == 1)
        return decode_device_impl(c, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, out_dev, status_dev,
                                  indices_dev, stream, false);
    if ((unsigned long long)nframes * linear_geom(W, H).ppf >= 0xFFFFFFF0ull)
        return fail(DBDE_B200_E_INVALID, "decode_binned_device: batch too large");
    DecParams D;
    int rc = linear_scan(c, (cudaStream_t)stream, W, H, stream_dev, stream_bytes, frame_offsets_dev, nframes, status_dev,
                         indices_dev, &D);
    if (rc) return rc;
    CK(launch_decode_binned(D, factor, out_dev, c->num_sms, (cudaStream_t)stream));
    c->launches += 1;
    return 0;
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
// What differs on the host path between the reference's 8-bit records and the DBDE16 extension: bytes per
// frame, slot stride, where a slot's record starts so that its U64 words are 16-byte aligned.
struct HostFmt {
    bool u16;
    size_t px, stride, delta;
    size_t stream_bound(int n) const { return stride * (size_t)(n < 0 ? 0 : n) + 16; }
};
static HostFmt host_fmt(int W, int H, bool u16) {
    HostFmt f;
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    f.u16 = u16;
    f.px = (size_t)W * H * (u16 ? 2 : 1);
    f.stride = u16 ? dbde_b200_slot_stride16(W, H) : dbde_b200_slot_stride(W, H);
    f.delta = (16 - (32 + (u16 ? 3 : 2) * wh) % 16) % 16;
    return f;
}

static int default_chunk(const dbde_b200_ctx *c, int W, int H, int nframes, bool u16 = false) {
    int n = c->chunk_frames;
    if (n <= 0) {
        const size_t px = (size_t)W * H * (u16 ? 2 : 1);
        n = (int)((64u << 20) / (px ? px : 1));
        if (n < 1) n = 1;
    }
    if (n > nframes) n = nframes;
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

// What the host pipeline hands back per frame instead of the whole image: the region (x0, y0, w, h), ncrops crops
// of w x h with host corners (per_frame: nframes * ncrops {x0, y0} pairs, else ncrops pairs for every frame), or the
// frame binned by `factor` (w x h = ceil(W / factor) x ceil(H / factor)).  Sizes count pixels: DBDE16 frames (u16)
// have two bytes each, and no region form.  The encoder takes the crops form: ncrops records of w x h per frame.
struct SubFrame {
    int x0, y0, w, h;
    const int32_t *corners;     // null: the region or the binned frame
    int ncrops, per_frame, pad;
    int factor;                 // > 0: the binned frame
    size_t bytes() const { return (size_t)w * (size_t)h * (size_t)(corners ? ncrops : 1); }
    size_t corner_bytes(int n) const { return corners ? 8 * (size_t)ncrops * (size_t)(per_frame ? n : 1) : 0; }
};

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

// Worker `my` of `nworkers`: encodes chunks my, my + nworkers, ... of the batch on context c.  crops: every frame
// gives crops->ncrops records of crops->w x crops->h (dbde_b200_encode_crops_device, or dbde_b200_encode16_crops_device
// when u16) instead of its own record; the chunk's corners travel behind its frames in the slot's frame buffer.
static int encode_host_worker(dbde_b200_ctx *c, const uint8_t *frames_host, int W, int H, uint64_t first_index,
                              int nframes, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host,
                              int chunk, int my, int nworkers, EncSequencer *seq, bool u16 = false, const SubFrame *crops = nullptr) {
    CK(cudaSetDevice(c->device));
    const HostFmt F = crops ? host_fmt(crops->w, crops->h, u16) : host_fmt(W, H, u16);     // the records' format
    const size_t px = crops ? (size_t)W * (size_t)H * (u16 ? 2 : 1) : F.px;                 // input bytes per frame
    const int per = crops ? crops->ncrops : 1;                                                // records per frame
    const int nrec = chunk * per;                                                             // records per chunk
    const size_t delta = F.delta;
    const size_t corner_at = (px * chunk + 15) & ~(size_t)15, need_corners = crops ? crops->corner_bytes(chunk) : 0;
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
            const size_t nb = crops->corner_bytes(s.n);
            memcpy(s.h_corners, crops->corners + (crops->per_frame ? 2 * (size_t)crops->ncrops * (size_t)s.first : 0), nb);
            CK(cudaMemcpyAsync(s.d_a + corner_at, s.h_corners, nb, cudaMemcpyHostToDevice, s.st));
        }
        prof.mark(1, "h2d");
        prof.gpu_mark(1, s.st);
        rc_all = crops && u16 ? dbde_b200_encode16_crops_device(c, (const uint16_t *)s.d_a, W, H, first_index + s.first, s.n,
                                                                (const int32_t *)(s.d_a + corner_at), crops->ncrops, crops->per_frame,
                                                                crops->w, crops->h, crops->pad, s.d_b + delta, need_b - 32, stride,
                                                                s.d_off, s.d_size, s.st)
                 : crops ? dbde_b200_encode_crops_device(c, s.d_a, W, H, first_index + s.first, s.n, (const int32_t *)(s.d_a + corner_at),
                                                         crops->ncrops, crops->per_frame, crops->w, crops->h, crops->pad, s.d_b + delta,
                                                         need_b - 32, stride, s.d_off, s.d_size, s.st)
                 : u16 ? dbde_b200_encode16_device(c, (const uint16_t *)s.d_a, W, H, first_index + s.first, s.n, s.d_b + delta,
                                                   need_b - 32, stride, s.d_off, s.d_size, s.st)
                       : dbde_b200_encode_device(c, s.d_a, W, H, first_index + s.first, s.n, s.d_b + delta, need_b - 32, stride,
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

extern "C" int dbde_b200_encode_host(dbde_b200_ctx *c, const uint8_t *frames_host, int W, int H,
                                     uint64_t first_index, int nframes, uint8_t *out_host, size_t out_capacity,
                                     uint64_t *frame_offsets_host) {
    if (!c || !dims_ok(W, H, nframes) || (nframes > 0 && (!frames_host || !out_host || !frame_offsets_host)))
        return fail(DBDE_B200_E_INVALID, "encode_host: bad argument");
    if (nframes == 0) {
        if (frame_offsets_host) frame_offsets_host[0] = 0;
        return 0;
    }
    EncSequencer seq;
    int rc = encode_host_worker(c, frames_host, W, H, first_index, nframes, out_host, out_capacity, frame_offsets_host,
                                default_chunk(c, W, H, nframes), 0, 1, &seq);
    if (rc) return rc;
    frame_offsets_host[nframes] = seq.out_pos;
    return 0;
}

// The host forms of dbde_b200_encode_crops_device and dbde_b200_encode16_crops_device (u16): the encode_host chunk
// pipeline with ncrops records per frame; each chunk's corners go up behind its frames.
static int encode_crops_host_impl(dbde_b200_ctx *c, const uint8_t *frames_host, int W, int H, uint64_t first_index, int nframes,
                                  const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w, int crop_h, int pad,
                                  uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host, bool u16) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad, u16 ? 65535 : 255) ||
        (nframes > 0 && (!frames_host || !corners_host || !out_host || !frame_offsets_host)))
        return fail(DBDE_B200_E_INVALID, u16 ? "encode16_crops_host: bad argument" : "encode_crops_host: bad argument");
    if (nframes == 0) {
        if (frame_offsets_host) frame_offsets_host[0] = 0;
        return 0;
    }
    if ((long long)nframes * ncrops > 0x7FFFFFFFLL)
        return fail(DBDE_B200_E_INVALID, u16 ? "encode16_crops_host: nframes * ncrops > 2^31 - 1" : "encode_crops_host: nframes * ncrops > 2^31 - 1");
    int chunk = default_chunk(c, W, H, nframes, u16);
    const HostFmt crop = host_fmt(crop_w, crop_h, u16), frame = host_fmt(W, H, u16);
    const size_t rec = (size_t)ncrops * crop.stride;                   // one frame's record slots
    if (rec > frame.stride) {                      // crops larger than the frame: a chunk's records stay within 64 MiB
        const size_t most = (64u << 20) / rec;
        if ((size_t)chunk > most) chunk = most > 0 ? (int)most : 1;
    }
    const SubFrame crops = {0, 0, crop_w, crop_h, corners_host, ncrops, corners_per_frame, pad, 0};
    EncSequencer seq;
    int rc = encode_host_worker(c, frames_host, W, H, first_index, nframes, out_host, out_capacity, frame_offsets_host, chunk, 0, 1,
                                &seq, u16, &crops);
    if (rc) return rc;
    frame_offsets_host[(size_t)nframes * ncrops] = seq.out_pos;
    return 0;
}

extern "C" int dbde_b200_encode_crops_host(dbde_b200_ctx *c, const uint8_t *frames_host, int W, int H, uint64_t first_index,
                                           int nframes, const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                           int crop_h, int pad, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host) {
    return encode_crops_host_impl(c, frames_host, W, H, first_index, nframes, corners_host, ncrops, corners_per_frame, crop_w, crop_h,
                                  pad, out_host, out_capacity, frame_offsets_host, false);
}

extern "C" int dbde_b200_encode16_crops_host(dbde_b200_ctx *c, const uint16_t *frames_host, int W, int H, uint64_t first_index,
                                             int nframes, const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host) {
    return encode_crops_host_impl(c, (const uint8_t *)frames_host, W, H, first_index, nframes, corners_host, ncrops, corners_per_frame,
                                  crop_w, crop_h, pad, out_host, out_capacity, frame_offsets_host, true);
}

static int decode_host_impl(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                            const uint64_t *frame_offsets_host, int W, int H, int nframes, uint8_t *frames_host,
                            uint32_t *status_host, uint64_t *indices_host, bool scan_only, bool u16 = false,
                            const SubFrame *sub = nullptr) {
    if (!c || !dims_ok(W, H, nframes) ||
        (nframes > 0 && (!stream_host || !frame_offsets_host || (!frames_host && !scan_only) || !status_host)))
        return fail(DBDE_B200_E_INVALID, "decode_host: bad argument");
    if (nframes == 0) return 0;
    CK(cudaSetDevice(c->device));
    for (int i = 0; i < nframes; i++) {
        const uint64_t end = i + 1 < nframes ? frame_offsets_host[i + 1] : stream_bytes;
        if (frame_offsets_host[i] > end || end > stream_bytes)
            return fail(DBDE_B200_E_INVALID, "decode_host: frame offsets must ascend within the stream");
    }
    const HostFmt F = host_fmt(W, H, u16);
    const size_t px = sub ? sub->bytes() * (u16 ? 2 : 1) : F.px;    // output bytes per frame
    int chunk = default_chunk(c, W, H, nframes, u16);
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
    const size_t need_corners = sub ? sub->corner_bytes(chunk) : 0;
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
        if (sub && sub->corners) {
            // this chunk's corners (the staging is free: the slot's stream has drained)
            const size_t nb = sub->corner_bytes(s.n);
            memcpy(s.h_corners, sub->corners + (sub->per_frame ? 2 * (size_t)sub->ncrops * (size_t)s.first : 0), nb);
            CK(cudaMemcpyAsync(s.d_c, s.h_corners, nb, cudaMemcpyHostToDevice, s.st));
        }
        prof.mark(1, "h2d");
        rc_all = u16 && sub && sub->corners
                       ? dbde_b200_decode16_crops_device(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, (const int32_t *)s.d_c,
                                                         sub->ncrops, sub->per_frame, sub->w, sub->h, sub->pad, (uint16_t *)s.d_b,
                                                         s.d_status, s.d_index, s.st)
                 : u16 && sub ? dbde_b200_decode16_binned_device(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, sub->factor,
                                                                 (uint16_t *)s.d_b, s.d_status, s.d_index, s.st)
                 : u16 ? dbde_b200_decode16_device(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, (uint16_t *)s.d_b, s.d_status,
                                                   s.d_index, s.st)
                 : sub && sub->corners
                       ? dbde_b200_decode_crops_device(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, (const int32_t *)s.d_c,
                                                       sub->ncrops, sub->per_frame, sub->w, sub->h, sub->pad, s.d_b, s.d_status,
                                                       s.d_index, s.st)
                 : sub && sub->factor
                       ? dbde_b200_decode_binned_device(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, sub->factor, s.d_b, s.d_status,
                                                        s.d_index, s.st)
                 : sub ? dbde_b200_decode_roi_device(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, sub->x0, sub->y0, sub->w, sub->h,
                                                     s.d_b, s.d_status, s.d_index, s.st)
                       : decode_device_impl(c, s.d_a + delta, b1 - b0, s.d_off, W, H, s.n, s.d_b, s.d_status, s.d_index, s.st,
                                            scan_only);
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
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, frames_host, status_host,
                            indices_host, false);
}

// The host form of dbde_b200_decode_roi_device: the same chunk pipeline with roi_w * roi_h bytes per frame
// coming back.  Records still cross PCIe whole.
extern "C" int dbde_b200_decode_roi_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                         const uint64_t *frame_offsets_host, int W, int H, int nframes, int x0, int y0,
                                         int roi_w, int roi_h, uint8_t *roi_host, uint32_t *status_host,
                                         uint64_t *indices_host) {
    if (!c || !dims_ok(W, H, nframes) || !roi_ok(W, H, x0, y0, roi_w, roi_h) ||
        (nframes > 0 && (!stream_host || !frame_offsets_host || !roi_host || !status_host)))
        return fail(DBDE_B200_E_INVALID, "decode_roi_host: bad argument");
    const SubFrame roi = {x0, y0, roi_w, roi_h, nullptr, 1, 0, 0, 0};
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, roi_host, status_host,
                            indices_host, false, false, &roi);
}

// The host form of dbde_b200_decode_crops_device: the same chunk pipeline with ncrops * crop_w * crop_h bytes per
// frame coming back; each chunk's corners go up on its slot's stream.
extern "C" int dbde_b200_decode_crops_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                           const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                           const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                           int crop_h, int pad, uint8_t *crops_host, uint32_t *status_host,
                                           uint64_t *indices_host) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad) ||
        (nframes > 0 && (!stream_host || !frame_offsets_host || !corners_host || !crops_host || !status_host)))
        return fail(DBDE_B200_E_INVALID, "decode_crops_host: bad argument");
    const SubFrame crops = {0, 0, crop_w, crop_h, corners_host, ncrops, corners_per_frame, pad, 0};
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, crops_host, status_host,
                            indices_host, false, false, &crops);
}

// The host form of dbde_b200_decode_binned_device: the same chunk pipeline with ceil(W / factor) * ceil(H / factor)
// bytes per frame coming back.  Records still cross PCIe whole.
extern "C" int dbde_b200_decode_binned_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                            const uint64_t *frame_offsets_host, int W, int H, int nframes, int factor,
                                            uint8_t *out_host, uint32_t *status_host, uint64_t *indices_host) {
    if (!c || !dims_ok(W, H, nframes) || !factor_ok(factor) ||
        (nframes > 0 && (!stream_host || !frame_offsets_host || !out_host || !status_host)))
        return fail(DBDE_B200_E_INVALID, "decode_binned_host: bad argument");
    const SubFrame binned = {0, 0, (W - 1) / factor + 1, (H - 1) / factor + 1, nullptr, 1, 0, 0, factor};
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, out_host, status_host,
                            indices_host, false, false, &binned);
}

// dbde_b200_validate_device for a stream in host memory: the records cross PCIe once, nothing comes
// back but 4 (+8) bytes per frame.
extern "C" int dbde_b200_validate_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                       const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                       uint32_t *status_host, uint64_t *indices_host) {
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, nullptr, status_host,
                            indices_host, true);
}

// ------------------------------------------------------------------ DBDE16 (SURVEY 8 f-4)
extern "C" size_t dbde_b200_frame_record_bound16(int W, int H) {
    const size_t wh = (size_t)((W + 7) / 8) * ((H + 7) / 8);
    return 32 + 3 * wh + 128 * wh;
}
extern "C" size_t dbde_b200_slot_stride16(int W, int H) { return (dbde_b200_frame_record_bound16(W, H) + 15) & ~(size_t)15; }

extern "C" int dbde_b200_encode16_device(dbde_b200_ctx *c, const uint16_t *frames_dev, int W, int H, uint64_t first_index,
                                         int nframes, uint8_t *out_dev, size_t out_capacity, size_t slot_stride,
                                         uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || (nframes > 0 && (!frames_dev || !out_dev || !frame_offsets_dev || !frame_sizes_dev)) ||
        ((uintptr_t)frames_dev & 1))
        return fail(DBDE_B200_E_INVALID, "encode16_device: bad argument");
    if (nframes == 0) return 0;
    if (slot_stride == 0) slot_stride = dbde_b200_slot_stride16(W, H);
    if (slot_stride < dbde_b200_frame_record_bound16(W, H))
        return fail(DBDE_B200_E_INVALID, "encode16_device: slot_stride < dbde_b200_frame_record_bound16()");
    if (out_capacity < slot_stride * (size_t)nframes)
        return fail(DBDE_B200_E_CAPACITY, "encode16_device: out_capacity < nframes * slot_stride");
    CK(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    Enc16Params P;
    P.W = W; P.H = H; P.w = (W + 7) / 8; P.h = (H + 7) / 8; P.wh = P.w * P.h;
    P.ppf = (P.wh + 255) / 256;
    const unsigned long long nparts = (unsigned long long)nframes * P.ppf;
    if (nparts >= 0xFFFFFFF0ull) return fail(DBDE_B200_E_INVALID, "encode16_device: batch too large");
    const size_t sbytes = 128 + 8 * (size_t)nparts;
    StreamScratch &sc = scratch_for(c, st);
    int rc = grow(&sc.enc, &sc.enc_bytes, sbytes);
    if (rc) return rc;
    CK(cudaMemsetAsync(sc.enc, 0, sbytes, st));
    P.frames = frames_dev; P.out = out_dev; P.slot_stride = slot_stride;
    P.frame_offsets = frame_offsets_dev; P.frame_sizes = frame_sizes_dev;
    P.ticket = (unsigned int *)sc.enc;
    P.desc = (uint64_t *)((uint8_t *)sc.enc + 128);
    P.first_index = first_index; P.nframes = nframes; P.nparts = (unsigned)nparts;
    P.aligned = (W % 8 == 0) && (((uintptr_t)frames_dev & 15) == 0);
    CK(launch_encode16(P, c->num_sms, st));
    c->launches += 1;
    return 0;
}

// One CTA per record of a persistent grid, one lane per crop tile (dbde16.cu): dbde_b200_encode_crops_device with U16
// pixels.  A crop equal to the frame still runs the crop kernel: its records are the frame encoder's records.
extern "C" int dbde_b200_encode16_crops_device(dbde_b200_ctx *c, const uint16_t *frames_dev, int W, int H, uint64_t first_index,
                                               int nframes, const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                               int crop_h, int pad, uint8_t *out_dev, size_t out_capacity, size_t slot_stride,
                                               uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad, 65535) ||
        (nframes > 0 && (!frames_dev || !corners_dev || !out_dev || !frame_offsets_dev || !frame_sizes_dev)) ||
        ((uintptr_t)frames_dev & 1))
        return fail(DBDE_B200_E_INVALID, "encode16_crops_device: bad argument");
    if (nframes == 0) return 0;
    if (slot_stride == 0) slot_stride = dbde_b200_slot_stride16(crop_w, crop_h);
    if (slot_stride < dbde_b200_frame_record_bound16(crop_w, crop_h))
        return fail(DBDE_B200_E_INVALID, "encode16_crops_device: slot_stride < dbde_b200_frame_record_bound16(crop_w, crop_h)");
    const long long nrec = (long long)nframes * ncrops;
    if (nrec > 0x7FFFFFFFLL) return fail(DBDE_B200_E_INVALID, "encode16_crops_device: nframes * ncrops > 2^31 - 1");
    if (slot_stride > out_capacity / (size_t)nrec)
        return fail(DBDE_B200_E_CAPACITY, "encode16_crops_device: out_capacity < nframes * ncrops * slot_stride");
    CK(cudaSetDevice(c->device));
    Enc16CropParams P;
    P.frames = frames_dev;
    P.W = W;
    P.H = H;
    P.corners = corners_dev;
    P.ncrops = ncrops;
    P.corner_stride = corners_per_frame ? ncrops : 0;
    P.crop_w = crop_w;
    P.crop_h = crop_h;
    P.w = (crop_w + 7) / 8;
    P.wh = P.w * ((crop_h + 7) / 8);
    P.pad = (uint32_t)pad;
    P.out = out_dev;
    P.slot_stride = slot_stride;
    P.frame_offsets = frame_offsets_dev;
    P.frame_sizes = frame_sizes_dev;
    P.first_index = first_index;
    P.nrec = (int)nrec;
    CK(launch_encode16_crops(P, c->num_sms, (cudaStream_t)stream));
    c->launches += 1;
    return 0;
}

// The DBDE16 validation pass (dbde16_scan_kernel: every check, over the whole record, and the word prefix of every
// 32 raster-order tiles), queued on st: the first launch of every DBDE16 decode.  P is what the second kernel reads;
// its output fields are left to the caller.
static int decode16_scan(dbde_b200_ctx *c, cudaStream_t st, const uint8_t *stream_dev, size_t stream_bytes,
                         const uint64_t *frame_offsets_dev, int W, int H, int nframes, uint32_t *status_dev, uint64_t *indices_dev,
                         Dec16Params *P, const char *what) {
    CK(cudaSetDevice(c->device));
    *P = Dec16Params();
    P->W = W; P->H = H; P->w = (W + 7) / 8; P->h = (H + 7) / 8; P->wh = P->w * P->h;
    P->ppf = (P->wh + 255) / 256;
    const unsigned long long nparts = (unsigned long long)nframes * P->ppf;
    if (nparts >= 0xFFFFFFF0ull) return fail(DBDE_B200_E_INVALID, what);
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

extern "C" int dbde_b200_decode16_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                         const uint64_t *frame_offsets_dev, int W, int H, int nframes, uint16_t *frames_dev,
                                         uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || (nframes > 0 && (!stream_dev || !frame_offsets_dev || !frames_dev || !status_dev)) ||
        ((uintptr_t)frames_dev & 1))
        return fail(DBDE_B200_E_INVALID, "decode16_device: bad argument");
    if (nframes == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    Dec16Params P;
    int rc = decode16_scan(c, st, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, status_dev, indices_dev, &P,
                           "decode16_device: batch too large");
    if (rc) return rc;
    P.frames = frames_dev;
    P.aligned = (W % 8 == 0) && (((uintptr_t)frames_dev & 15) == 0);
    CK(launch_decode16(P, c->num_sms, st));
    c->launches += 1;
    return 0;
}

// The scan, then one warp per 32 tile columns of each tile row of each crop (dbde16.cu).  A crop equal to the frame
// still runs the crop kernel: its output layout is the crop layout whatever the corners.
extern "C" int dbde_b200_decode16_crops_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                               const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                               const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                               int crop_h, int pad, uint16_t *crops_dev, uint32_t *status_dev,
                                               uint64_t *indices_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad, 65535) ||
        (nframes > 0 && (!stream_dev || !frame_offsets_dev || !corners_dev || !crops_dev || !status_dev)) ||
        ((uintptr_t)crops_dev & 1))
        return fail(DBDE_B200_E_INVALID, "decode16_crops_device: bad argument");
    if (nframes == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    Dec16Params P;
    int rc = decode16_scan(c, st, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, status_dev, indices_dev, &P,
                           "decode16_crops_device: batch too large");
    if (rc) return rc;
    CK(launch_decode16_crops(P, corners_dev, ncrops, corners_per_frame != 0, crop_w, crop_h, pad, crops_dev, st));
    c->launches += 1;
    return 0;
}

// The scan, then the full decoder's partitions with each tile reduced to its bin means in registers (dbde16.cu).
// Factor 1 is the full decode.
extern "C" int dbde_b200_decode16_binned_device(dbde_b200_ctx *c, const uint8_t *stream_dev, size_t stream_bytes,
                                                const uint64_t *frame_offsets_dev, int W, int H, int nframes, int factor,
                                                uint16_t *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream) {
    if (!c || !dims_ok(W, H, nframes) || !factor_ok(factor) ||
        (nframes > 0 && (!stream_dev || !frame_offsets_dev || !out_dev || !status_dev)) || ((uintptr_t)out_dev & 1))
        return fail(DBDE_B200_E_INVALID, "decode16_binned_device: bad argument");
    if (nframes == 0) return 0;
    if (factor == 1)
        return dbde_b200_decode16_device(c, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, out_dev, status_dev,
                                         indices_dev, stream);
    cudaStream_t st = (cudaStream_t)stream;
    Dec16Params P;
    int rc = decode16_scan(c, st, stream_dev, stream_bytes, frame_offsets_dev, W, H, nframes, status_dev, indices_dev, &P,
                           "decode16_binned_device: batch too large");
    if (rc) return rc;
    CK(launch_decode16_binned(P, factor, out_dev, c->num_sms, st));
    c->launches += 1;
    return 0;
}

// Host-buffer forms: the 8-bit path's chunk pipeline (staging slots in flight, records compacted on the
// device, pageable buffers relayed through the copy pool), with the DBDE16 kernels underneath.
extern "C" int dbde_b200_encode16_host(dbde_b200_ctx *c, const uint16_t *frames_host, int W, int H, uint64_t first_index,
                                       int nframes, uint8_t *out_host, size_t out_capacity, uint64_t *frame_offsets_host) {
    if (!c || !dims_ok(W, H, nframes) || (nframes > 0 && (!frames_host || !out_host || !frame_offsets_host)))
        return fail(DBDE_B200_E_INVALID, "encode16_host: bad argument");
    if (nframes == 0) {
        if (frame_offsets_host) frame_offsets_host[0] = 0;
        return 0;
    }
    EncSequencer seq;
    int rc = encode_host_worker(c, (const uint8_t *)frames_host, W, H, first_index, nframes, out_host, out_capacity,
                                frame_offsets_host, default_chunk(c, W, H, nframes, true), 0, 1, &seq, true);
    if (rc) return rc;
    frame_offsets_host[nframes] = seq.out_pos;
    return 0;
}

extern "C" int dbde_b200_decode16_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                       const uint64_t *frame_offsets_host, int W, int H, int nframes, uint16_t *frames_host,
                                       uint32_t *status_host, uint64_t *indices_host) {
    if (!c || !dims_ok(W, H, nframes) || (nframes > 0 && (!stream_host || !frame_offsets_host || !frames_host || !status_host)))
        return fail(DBDE_B200_E_INVALID, "decode16_host: bad argument");
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, (uint8_t *)frames_host, status_host,
                            indices_host, false, true);
}

// The host forms of the DBDE16 crop and binned decodes: the same chunk pipeline with the crops' or the bins' pixels
// coming back.  Records still cross PCIe whole.
extern "C" int dbde_b200_decode16_crops_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                             const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                             const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                             int crop_h, int pad, uint16_t *crops_host, uint32_t *status_host,
                                             uint64_t *indices_host) {
    if (!c || !dims_ok(W, H, nframes) || !crops_ok(ncrops, corners_per_frame, crop_w, crop_h, pad, 65535) ||
        (nframes > 0 && (!stream_host || !frame_offsets_host || !corners_host || !crops_host || !status_host)) ||
        ((uintptr_t)crops_host & 1))
        return fail(DBDE_B200_E_INVALID, "decode16_crops_host: bad argument");
    const SubFrame crops = {0, 0, crop_w, crop_h, corners_host, ncrops, corners_per_frame, pad, 0};
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, (uint8_t *)crops_host, status_host,
                            indices_host, false, true, &crops);
}

extern "C" int dbde_b200_decode16_binned_host(dbde_b200_ctx *c, const uint8_t *stream_host, size_t stream_bytes,
                                              const uint64_t *frame_offsets_host, int W, int H, int nframes, int factor,
                                              uint16_t *out_host, uint32_t *status_host, uint64_t *indices_host) {
    if (!c || !dims_ok(W, H, nframes) || !factor_ok(factor) ||
        (nframes > 0 && (!stream_host || !frame_offsets_host || !out_host || !status_host)) || ((uintptr_t)out_host & 1))
        return fail(DBDE_B200_E_INVALID, "decode16_binned_host: bad argument");
    if (factor == 1)
        return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, (uint8_t *)out_host, status_host,
                                indices_host, false, true);
    const SubFrame binned = {0, 0, (W - 1) / factor + 1, (H - 1) / factor + 1, nullptr, 1, 0, 0, factor};
    return decode_host_impl(c, stream_host, stream_bytes, frame_offsets_host, W, H, nframes, (uint8_t *)out_host, status_host,
                            indices_host, false, true, &binned);
}

// ------------------------------------------------------------------ multi-GPU sharding
// contiguous frame ranges, one host thread per context; there is no cross-GPU exchange on the
// data path, the host only prefix-sums the shard sizes (SURVEY.md section 8e)
extern "C" int dbde_b200_encode_host_sharded(dbde_b200_ctx **ctxs, int nctx, const uint8_t *frames_host, int W,
                                             int H, uint64_t first_index, int nframes, uint8_t *out_host,
                                             size_t out_capacity, uint64_t *frame_offsets_host) {
    if (!ctxs || nctx < 1 || !dims_ok(W, H, nframes) || (nframes > 0 && (!frames_host || !out_host || !frame_offsets_host)))
        return fail(DBDE_B200_E_INVALID, "encode_host_sharded: bad argument");
    for (int g = 0; g < nctx; g++)
        if (!ctxs[g]) return fail(DBDE_B200_E_INVALID, "encode_host_sharded: null context");
    if (nframes == 0) {
        frame_offsets_host[0] = 0;
        return 0;
    }
    // The batch is cut into contiguous frame ranges of one chunk each; range ci goes to context
    // ci mod G.  Every context streams its ranges over its own PCIe link, and the ranges' records are
    // placed in stream order as their sizes become known (EncSequencer): the stream is complete when
    // the last copy lands -- no shard is moved afterwards.
    const int chunk = default_chunk(ctxs[0], W, H, nframes);
    EncSequencer seq;
    std::vector<int> rc(nctx, 0);
    std::vector<std::string> err(nctx);
    std::vector<std::thread> th;
    for (int g = 0; g < nctx; g++) {
        th.emplace_back([&, g]() {
            rc[g] = encode_host_worker(ctxs[g], frames_host, W, H, first_index, nframes, out_host, out_capacity,
                                       frame_offsets_host, chunk, g, nctx, &seq);
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
    const size_t fixed = 32 + (1 + minbytes) * wh;
    size_t cur = 0;
    long n = 0;
    while (cur + fixed <= bytes && n < max_frames) {
        uint32_t n64;
        memcpy(&n64, p + cur + fixed - 4, 4);
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
