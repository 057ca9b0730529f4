// DBDE B200 codec -- device-side building blocks (sm_100a only).
//
// Everything here is written for Blackwell: bulk-TMA (cp.async.bulk -> SASS UBLKCP) staged
// through mbarrier pipelines, VIMNMX3.U16x2 byte-min reduction, REDUX warp sums, a predicate-
// returning SHFL scan, and a single-word decoupled look-back.  No tensor cores: the path has no
// contraction.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "dbde_record.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "dbde_b200 kernels are written for sm_100a (B200) only"
#endif

namespace dbde {

// ------------------------------------------------------------------ geometry
constexpr int kTilesPerPart = 256;              // tiles per partition == consumer threads per CTA
constexpr int kConsumerWarps = kTilesPerPart / 32;
constexpr int kMaxBandsPerPart = 8;             // a partition is <= 8 bands of a narrow frame ...
constexpr int kMaxRowsPerPart = 8 * kMaxBandsPerPart;   // ... i.e. <= 64 pixel rows in one stage

// How a frame is cut into partitions (the unit of the scan and of one pipeline stage).
//   w <= 256 tiles : a partition is G consecutive 8-row bands (G*w <= 256 tiles)
//   w  > 256 tiles : a band is cut into nseg segments of <= 256 tiles
//   linear         : tiles [256 q, 256 q + 256) of the row-major tile order, across band boundaries
// Either way a partition's tiles are CONTIGUOUS in the frame's row-major tile order, so the
// partition order is the order of the reference's running output pointer (dbde_util.cpp:155).
struct PartGeom {
    int W, H, w, h, wh;
    int nseg;     // segments per band (1 when w <= 256)
    int G;        // bands per partition when nseg == 1
    int ppf;      // partitions per frame
    int pitch;    // smem row pitch in bytes (multiple of 16)
    int stage_bytes;
    int linear;   // 1: a partition is 256 CONSECUTIVE tiles of the frame's row-major tile order, whatever bands
                  //    they fall in (aligned frames whose width would leave lanes idle otherwise, see make_geom)
};

// Linear partitions (make_geom for aligned frames, the region-of-interest scan): word-prefix item i of the scan
// is exactly tiles [32 i, 32 i + 32).  stage_bytes is left to the caller that stages partitions.
inline PartGeom linear_geom(int W, int H) {
    PartGeom g;
    g.W = W; g.H = H;
    g.w = (W + 7) / 8; g.h = (H + 7) / 8; g.wh = g.w * g.h;
    g.linear = 1;
    g.nseg = 1;
    g.G = 1;
    g.ppf = (g.wh + kTilesPerPart - 1) / kTilesPerPart;
    g.pitch = 8 * kTilesPerPart;
    g.stage_bytes = 0;
    return g;
}

struct PartInfo {
    int f;        // frame within the batch
    int q;        // partition within the frame
    int y0;       // first band
    int nbands;   // bands in this partition
    int tx0;      // first tile column
    int ntx;      // tile columns
    int nt;       // tiles = nbands * ntx
    int tfirst;   // first tile's row-major index in the frame
};

__host__ __device__ inline PartInfo part_info(const PartGeom &g, unsigned p) {
    PartInfo o;
    o.f = (int)(p / (unsigned)g.ppf);
    o.q = (int)(p - (unsigned)o.f * (unsigned)g.ppf);
    if (g.linear) {
        o.tfirst = o.q * kTilesPerPart;
        o.nt = g.wh - o.tfirst < kTilesPerPart ? g.wh - o.tfirst : kTilesPerPart;
        o.y0 = o.tfirst / g.w;
        o.tx0 = o.tfirst - o.y0 * g.w;
        o.nbands = (o.tx0 + o.nt + g.w - 1) / g.w;        // bands the partition touches
        o.ntx = g.w;
        return o;
    }
    if (g.nseg > 1) {
        o.y0 = o.q / g.nseg;
        int seg = o.q - o.y0 * g.nseg;
        o.nbands = 1;
        o.tx0 = seg * kTilesPerPart;
        o.ntx = g.w - o.tx0 < kTilesPerPart ? g.w - o.tx0 : kTilesPerPart;
    } else {
        o.y0 = o.q * g.G;
        o.nbands = g.h - o.y0 < g.G ? g.h - o.y0 : g.G;
        o.tx0 = 0;
        o.ntx = g.w;
    }
    o.nt = o.nbands * o.ntx;
    o.tfirst = o.y0 * g.w + o.tx0;
    return o;
}

#ifdef __CUDACC__
// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// For the service warps (producer, scan), which spend most of their life waiting: a failed try_wait
// comes back after well under 100 ns (ncu: ~45 polls per partition per service warp, 10 % of all issued
// instructions), so they sleep between polls and leave the issue slots to the tile warps.  The
// added wake-up latency is hidden by the stages the producer runs ahead / the deferred copy-out.
#ifndef DBDE_SERVICE_SLEEP_NS
#define DBDE_SERVICE_SLEEP_NS 256
#endif
__device__ __forceinline__ void mbar_wait_sleepy(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE_S;\n"
        "LAB_WAIT_S:\n"
        "nanosleep.u32 %2;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE_S;\n"
        "bra LAB_WAIT_S;\n"
        "DONE_S:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity), "r"((uint32_t)DBDE_SERVICE_SLEEP_NS) : "memory");
}
// bulk TMA, global -> shared, completion on an mbarrier (SASS: UBLKCP).  16-byte aligned both sides.
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// order this thread's generic-proxy smem accesses against later async-proxy (TMA) accesses
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 1, %0;" ::"n"(kTilesPerPart) : "memory"); }

__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t *p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// streaming global stores (written once, never re-read by this kernel)
__device__ __forceinline__ void st_stream_u64(void *p, uint64_t v) {
    asm volatile("st.global.cs.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_stream_v4u32(void *p, uint4 v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_stream_u32(void *p, uint32_t v) {
    asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// ------------------------------------------------------------------ decoupled look-back
// One 64-bit word per partition: [63:62] status, [61:0] value (U64 words).  Status and value
// travel in ONE relaxed 64-bit access, so no fence is needed between them.
constexpr uint64_t kDescInvalid = 0, kDescAggregate = 1, kDescPrefix = 2;
constexpr uint64_t kDescValueMask = (1ull << 62) - 1;
__device__ __forceinline__ uint64_t desc_make(uint64_t status, uint64_t value) { return (status << 62) | value; }

// Called by all 32 lanes of one warp.  Chains restart at every frame (the reference zeroes n64
// per frame, dbde_util.cpp:146): `first` is the frame's first partition, `p` > `first`.  Returns
// the sum of the aggregates of partitions [first, p).  The first round reads the 32 nearest
// predecessors (with frame-interleaved tickets the nearest one is normally already resolved);
// later rounds read 128 at a time with four independent loads per lane.
constexpr int kLookbackSub = 4;
constexpr uint64_t kLookbackNotReady = ~0ull;
// WAIT = true : spins until every needed predecessor has published something (the classic look-back).
// WAIT = false: one opportunistic pass -- returns kLookbackNotReady as soon as it meets an unpublished
//               descriptor.  The exclusive prefix does not depend on the caller's own aggregate, so
//               the scan warp can take it BEFORE its partition's depth sums exist; with
//               frame-interleaved tickets the predecessors are long finished and this succeeds.
template <bool WAIT>
__device__ __forceinline__ uint64_t lookback_exclusive(const uint64_t *desc, unsigned p, unsigned first, int lane) {
    uint64_t sum = 0;
    long long look = (long long)p - 1;
    int nsub = 1;
    while (true) {
        uint64_t d[kLookbackSub];
#pragma unroll
        for (int j = 0; j < kLookbackSub; j++) {
            const long long idx = look - 32 * j - lane;
            d[j] = (j < nsub && idx >= (long long)first) ? ld_relaxed_u64(desc + idx) : desc_make(kDescPrefix, 0);
        }
        bool done = false, stall = false;
        int consumed = 0;
#pragma unroll
        for (int j = 0; j < kLookbackSub; j++) {
            if (done || stall || j >= nsub) continue;
            const unsigned st = (unsigned)(d[j] >> 62);
            const unsigned inval = __ballot_sync(0xffffffffu, st == kDescInvalid);
            const unsigned pre = __ballot_sync(0xffffffffu, st == kDescPrefix);
            if (pre) {
                const int jn = __ffs((int)pre) - 1;      // nearest predecessor that knows its prefix
                if (inval & ((1u << jn) - 1u)) { stall = true; continue; }   // a nearer one is unpublished
                const uint32_t part = lane < jn ? (uint32_t)(d[j] & kDescValueMask) : 0u;   // aggregates <= 2048
                sum += __reduce_add_sync(0xffffffffu, part);                               // REDUX.SUM
                sum += __shfl_sync(0xffffffffu, d[j], jn) & kDescValueMask;
                done = true;
            } else if (inval) {
                stall = true;
            } else {
                sum += __reduce_add_sync(0xffffffffu, (uint32_t)(d[j] & kDescValueMask));
                consumed++;
            }
        }
        if (done) return sum;
        if (!WAIT && stall) return kLookbackNotReady;
        look -= 32 * consumed;                           // fully aggregated sub-windows are never re-read
        nsub = kLookbackSub;
    }
}

// ------------------------------------------------------------------ warp scan
// shfl.up hands back "was my source lane in range" as a predicate, so a scan step is SHFL + one
// predicated add (no lane compares).
__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v, int lane) {
    (void)lane;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        asm volatile(
            "{\n"
            ".reg .u32 t;\n"
            ".reg .pred p;\n"
            "shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n"
            "@p add.u32 %0, %0, t;\n"
            "}"
            : "+r"(v)
            : "r"(d));
    }
    return v;
}

// ------------------------------------------------------------------ per-tile arithmetic (one lane == one 8x8 tile)
// px[2r], px[2r+1] = the 8 pixels of tile row r, little-endian.

// DBDE_INVERT_ENDIAN variant: reverse the 8 bytes of every tile row (dbde_util.cpp:15-19)
__device__ __forceinline__ void reverse_rows(uint32_t (&px)[16]) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint32_t lo = __byte_perm(px[2 * r + 1], 0u, 0x0123), hi = __byte_perm(px[2 * r], 0u, 0x0123);
        px[2 * r] = lo;
        px[2 * r + 1] = hi;
    }
}

// exact minimum of the 64 bytes: u16x2 min over {w, w<<8} puts every byte in a high-byte slot
// (VIMNMX3.U16x2; the byte-wise __vminu4 is a 7-instruction emulation on sm_100a).
__device__ __forceinline__ uint32_t tile_min(const uint32_t (&px)[16]) {
    uint32_t a = 0xffffffffu;
#pragma unroll
    for (int i = 0; i < 16; i++) a = __vimin3_u16x2(a, px[i], px[i] << 8);
    uint32_t hi = a >> 24, lo = (a >> 8) & 0xffu;
    return hi < lo ? hi : lo;
}

// px -= min (no byte borrows: every byte >= min); returns depth = bits(max - min) via the OR of
// the differences (the top set bit of an OR is the top set bit of the maximum).  dbde_util.cpp:48-68.
__device__ __forceinline__ int tile_subtract_depth(uint32_t (&px)[16], uint32_t mn) {
    const uint32_t m4 = mn * 0x01010101u;
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        px[i] -= m4;
        o |= px[i];
    }
    o |= o >> 16;
    o |= o >> 8;
    return 32 - __clz((int)(o & 0xffu));
}

// 4 bytes of <= k bits each  ->  one 4k-bit field.  Two multiply-adds per word, valid for k = 1..8:
//   pairs : w = e + 256*o        ->  p = e + 2^k*o      = w + o*(2^k - 256)
//   quads : p = l + 65536*h      ->  q = l + 2^(2k)*h   = p + h*(2^2k - 65536)
// (the role pmaddubsw/pmaddwd play at dbde_util.cpp:70-80).  Measured alternative: two IDP.4A with weights
// {1, 2^k, 0, 0} / {0, 0, 1, 2^k} + one multiply-add is 3 instructions instead of 4 but 11 % SLOWER
// (micro-2048 5.97 -> 5.32 TB/s): IDP.4A does not issue at the IMAD rate.  It pays only where one
// IDP.4A replaces all four (pack_low_depths).
__device__ __forceinline__ uint32_t squeeze4(uint32_t d, uint32_t c1, uint32_t c2) {
    uint32_t odd = __byte_perm(d, 0u, 0x4341);       // {b1, 0, b3, 0}
    uint32_t p = d + odd * c1;
    return p + (p >> 16) * c2;
}
// inverse: one 4k-bit field -> 4 bytes
//   q = l + 2^2k*h -> p = q + h*(65536 - 2^2k);   p = e + 2^k*o (per u16) -> w = p + o*(256 - 2^k)
// (SHF, IMAD, SHF, LOP3, IMAD: three ALU-pipe and two FMA-pipe instructions, which the scheduler pairs.  Measured
// alternatives, both rejected: a shift-free form p = q + (q & hmask)*(2^(16-2k) - 1), w = p + (p & omask)*(2^(8-k) - 1) --
// the compiler turns x*(2^n - 1) into shift-and-subtract, all on the ALU pipe: low-4096 decode 5.05 -> 4.20 TB/s; with the
// multiplies forced (mad.lo) it is neutral, 4.79 vs 4.82 on mix-1001x1003 -- and the two shifts as multiply-high by a
// power of two, which moves them to the FMA pipe but IMAD.HI issues slowly: 4.82 -> 4.35 TB/s.)
struct SpreadK {
    uint32_t k, c2n, kmask2, c1n;
};
__device__ __forceinline__ SpreadK spread_consts(int k) {           // k = 1..8
    SpreadK s;
    s.k = (uint32_t)k;
    s.c2n = 65536u - (1u << (2 * k));
    s.kmask2 = ((1u << k) - 1u) * 0x00010001u;
    s.c1n = 256u - (1u << k);
    return s;
}
__device__ __forceinline__ uint32_t spread4(uint32_t q, const SpreadK &s) {
    const uint32_t p = q + (q >> (2 * s.k)) * s.c2n;
    const uint32_t odd = (p >> s.k) & s.kmask2;
    return p + odd * s.c1n;
}

// Concatenate sixteen 4K-bit fields LSB-first into K little-endian U64 words (2K u32 halves).
// Everything is compile-time after unrolling.  Fields never overlap, so "or" is "add" and a
// field lands with ONE shift-add (IMAD/LEA) plus, when it straddles a 32-bit boundary, one
// shift for the spill-over; the spill is always the first contributor of the next half-word.
template <int K, typename Store>
__device__ __forceinline__ void concat_fields(const uint32_t (&q)[16], Store &&store) {
    uint32_t w[2 * K + 1];
#pragma unroll
    for (int n = 0; n < 2 * K + 1; n++) w[n] = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const int bit = 4 * K * i, n = bit >> 5, sh = bit & 31;
        if (sh == 0) w[n] = q[i];
        else w[n] += q[i] << sh;
        if (sh + 4 * K > 32) w[n + 1] = q[i] >> (32 - sh);
    }
#pragma unroll
    for (int n = 0; n < K; n++) store(n, w[2 * n], w[2 * n + 1]);
}
// inverse of concat_fields: K U64 words (as 2K u32) -> sixteen 4K-bit fields
template <int K>
__device__ __forceinline__ void split_fields(const uint32_t (&x)[16], uint32_t (&q)[16]) {
    constexpr uint32_t fmask = (K == 8) ? 0xffffffffu : ((1u << (4 * K)) - 1u);
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const int bit = 4 * K * i;
        const int j = bit >> 5, sh = bit & 31;
        uint32_t v = x[j] >> sh;
        if (sh + 4 * K > 32) v |= x[j + 1] << (32 - sh);
        q[i] = v & fmask;
    }
}

// ------------------------------------------------------------------ depth-agnostic pack / unpack
// concat_fields<K> / split_fields<K> are the shortest code for ONE depth, but a warp whose 32 tiles
// hold many different depths runs one specialisation after the other.  Tile row r is exactly k bytes
// at byte k*r of the tile's payload (8 pixels x k bits), so a row can also be moved with
// byte-granular VARIABLE shifts: the same instruction stream for every depth 1..8, no divergence.
// The tile warps vote per partition and take this path when the warp holds three or more depths.

// unpack: rows of k bytes at pay + k*r -> px[2r], px[2r+1] (before +min).  `pay` may have any byte
// alignment; reads at most 11 bytes past a row's first byte (the stage has that slack).
__device__ __forceinline__ void unpack_rows_var(const uint8_t *pay, int k, uint32_t (&px)[16], uint32_t m4) {
    const uint32_t a0 = smem_u32(pay);
    const uint32_t fmask = 0xffffffffu >> (32 - 4 * k);
    const SpreadK sk = spread_consts(k);
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint32_t a = a0 + (uint32_t)(k * r);
        const uint32_t *wv = reinterpret_cast<const uint32_t *>(pay + k * r - (a & 3u));
        const uint32_t w0 = wv[0], w1 = wv[1], w2 = wv[2];
        const uint32_t sh = a << 3;                                   // funnel shifts use the low 5 bits: 8 * (a & 3)
        const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
        const uint32_t f0 = lo & fmask;
        const uint32_t f1 = __funnelshift_rc(lo, hi, 4 * k) & fmask;  // clamped: 4k == 32 selects hi
        px[2 * r] = spread4(f0, sk) + m4;
        px[2 * r + 1] = spread4(f1, sk) + m4;
    }
}

// The same unpacker for payloads on 8-byte boundaries (the usual case: records are 8-byte aligned and a
// tile's words are U64s), with the shared-memory traffic cut to what the tile really holds.  The
// three-word version above issues 24 four-byte loads per tile whatever k is, each with the lanes'
// addresses scattered over the banks (ncu on the odd-size decoder: 75 % of the shared-memory wavefront
// budget, about half of it these loads).  Here a lane keeps a 16-byte window {cur, nxt} of two aligned
// U64s; row r sits at byte (k*r) & 7 of `cur` and ends inside the window (k <= 8); the window moves on by
// ONE predicated 8-byte load when a row crosses into `nxt` -- k + 1 loads per tile, each word read once.
// Reads at most 8 bytes past the tile's last word (the stage has that slack).
#ifndef DBDE_DEC_VAR64
#define DBDE_DEC_VAR64 1
#endif
__device__ __forceinline__ void unpack_rows_var64(const uint8_t *pay, int k, uint32_t (&px)[16], uint32_t m4) {
    uint32_t addr = smem_u32(pay);
    const uint32_t fmask = 0xffffffffu >> (32 - 4 * k);
    const SpreadK sk = spread_consts(k);
    uint32_t c_lo, c_hi, n_lo, n_hi;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(c_lo), "=r"(c_hi) : "r"(addr));
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+8];" : "=r"(n_lo), "=r"(n_hi) : "r"(addr));
    addr += 16u;
    uint32_t pos = 0;                                               // k * r
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const bool up = (pos & 4u) != 0u;                           // the row starts in the upper half of `cur`
        const uint32_t t0 = up ? c_hi : c_lo, t1 = up ? n_lo : c_hi, t2 = up ? n_hi : n_lo;
        const uint32_t sh = pos << 3;                               // funnel shifts use the low 5 bits: 8 * (pos & 3)
        const uint32_t lo = __funnelshift_r(t0, t1, sh), hi = __funnelshift_r(t1, t2, sh);
        const uint32_t f0 = lo & fmask;
        const uint32_t f1 = __funnelshift_rc(lo, hi, 4 * k) & fmask;
        px[2 * r] = spread4(f0, sk) + m4;
        px[2 * r + 1] = spread4(f1, sk) + m4;
        if (r < 7) {
            const uint32_t nx = pos + (uint32_t)k;
            if ((pos ^ nx) & 8u) {                                  // the next row starts in `nxt`: slide (predicated)
                c_lo = n_lo;
                c_hi = n_hi;
                asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(n_lo), "=r"(n_hi) : "r"(addr));
                addr += 8u;
            }
            pos = nx;
        }
    }
}

// unaligned-safe shared load for payloads that are not 8-byte aligned (records at odd offsets)
__device__ __forceinline__ uint32_t lds_u32_unaligned(const uint8_t *p) {
    uint32_t a = smem_u32(p);
    const uint32_t *q = (const uint32_t *)(p - (a & 3u));
    uint32_t sh = (a & 3u) * 8u;
    uint32_t x0 = q[0];
    if (sh == 0) return x0;
    return __funnelshift_r(x0, q[1], sh);
}

// The per-depth specialisations: K payload words -> the sixteen 4K-bit fields.  ALIGN = 8: the words are 8-byte
// aligned in shared memory (LDS.64); 1: any byte offset (funnel-shifted pairs).  Uniform per warp.
template <int K, int ALIGN>
__device__ __forceinline__ void load_split(const uint8_t *pay, uint32_t (&q)[16]) {
    uint32_t x[16];
#pragma unroll
    for (int j = 0; j < 16; j++) x[j] = 0;
    if (ALIGN == 8) {
#pragma unroll
        for (int j = 0; j < K; j++) {
            const uint2 v = reinterpret_cast<const uint2 *>(pay)[j];
            x[2 * j] = v.x;
            x[2 * j + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int j = 0; j < 2 * K; j++) x[j] = lds_u32_unaligned(pay + 4 * j);
    }
    split_fields<K>(x, q);
}

template <int ALIGN>
__device__ __forceinline__ void load_split_any(int k, const uint8_t *pay, uint32_t (&q)[16]) {
    switch (k) {
        case 1: load_split<1, ALIGN>(pay, q); break;
        case 2: load_split<2, ALIGN>(pay, q); break;
        case 3: load_split<3, ALIGN>(pay, q); break;
        case 4: load_split<4, ALIGN>(pay, q); break;
        case 5: load_split<5, ALIGN>(pay, q); break;
        case 6: load_split<6, ALIGN>(pay, q); break;
        case 7: load_split<7, ALIGN>(pay, q); break;
        default: load_split<8, ALIGN>(pay, q); break;
    }
}

// ------------------------------------------------------------------ one lane == one tile: payload -> pixels
// The unpacker of both decoders (dbde_decode.cu, dbde_roi.cu).  The warp votes on how many different non-zero
// depths it holds: each one is a pass through its own specialisation, so from kDecVarMinDepths on the
// depth-agnostic row unpacker is shorter.
// Measured (mix-2048, all nine depths per warp): threshold 99 (never) 4.41 TB/s, 3 -> 5.71, 2 -> 5.70; micro-2048
// is indifferent (5.80-5.92 in all three), low-4096 loses 7 % at 2.  Re-measured with the sliding-window unpacker:
// threshold 2 costs low-4096 10 % and low-1001x1003 8 %, threshold 1 (always) the same and gains 2 % on noise only.
constexpr int kDecVarMinDepths = 3;
// pay: the tile's k payload words in shared memory, 8-byte aligned when al8 (the stage has the unpackers' slack
// past them); m4: its minimum in every byte.  Returns the 64 pixels (+min applied, rows byte-reversed when
// invert) in px.  Warp-wide call (the vote); lanes without a tile pass k = 0.
__device__ __forceinline__ void unpack_tile(const uint8_t *pay, int k, uint32_t m4, bool al8, bool invert, uint32_t (&px)[16]) {
    const uint32_t kinds = __reduce_or_sync(0xffffffffu, (1u << k) >> 1);
    // (a warp of nothing but depth-8 tiles also goes this way: the K = 8 specialisation reads its 64-byte payloads with
    // 8-way bank conflicts, the sliding window does not -- noise-2048 5.71 -> 5.83 TB/s)
    if (__popc(kinds) >= kDecVarMinDepths || kinds == 0x80u) {
        if (k > 0) {
            if (DBDE_DEC_VAR64 && al8) unpack_rows_var64(pay, k, px, m4);
            else unpack_rows_var(pay, k, px, m4);
        } else {
#pragma unroll
            for (int i = 0; i < 16; i++) px[i] = m4;
        }
    } else if (k > 0) {
        uint32_t q[16];
        if (al8) load_split_any<8>(k, pay, q);                     // the usual case: records on 8-byte boundaries
        else load_split_any<1>(k, pay, q);
        const SpreadK sk = spread_consts(k);
#pragma unroll
        for (int i = 0; i < 16; i++) px[i] = spread4(q[i], sk) + m4;   // +min (dbde_util.cpp:246)
    } else {
#pragma unroll
        for (int i = 0; i < 16; i++) px[i] = m4;                                        // depth 0 (dbde_util.cpp:218-226)
    }
    if (invert) reverse_rows(px);                                                       // ENDIAN() at dbde_util.cpp:246-270
}

// ------------------------------------------------------------------ cropped row stores (global memory)
// Bytes [s, e) of the little-endian 64-bit `w` go to q + s .. q + e; q is 8-byte aligned, 0 <= s <= e <= 8.
// At most six naturally aligned stores (1-2-4 up to alignment, then 4-2-1 down).
__device__ __forceinline__ void store_partial(uint8_t *q, uint64_t w, uint32_t s, uint32_t e) {
    if ((s & 1u) && e - s >= 1u) { q[s] = (uint8_t)(w >> (8 * s)); s += 1; }
    if ((s & 2u) && e - s >= 2u) { *reinterpret_cast<uint16_t *>(q + s) = (uint16_t)(w >> (8 * s)); s += 2; }
    if ((s & 4u) && e - s >= 4u) { *reinterpret_cast<uint32_t *>(q + s) = (uint32_t)(w >> (8 * s)); s += 4; }
    if (e - s >= 4u) { *reinterpret_cast<uint32_t *>(q + s) = (uint32_t)(w >> (8 * s)); s += 4; }
    if (e - s >= 2u) { *reinterpret_cast<uint16_t *>(q + s) = (uint16_t)(w >> (8 * s)); s += 2; }
    if (e - s >= 1u) q[s] = (uint8_t)(w >> (8 * s));
}

// pack: q[16] = the sixteen 4k-bit fields (squeeze4) -> k U64 words at wp (8-byte aligned shared
// memory).  A 64-bit accumulator takes one k-byte row per step at byte position (k*r) & 7 and is
// flushed with a predicated store whenever a word completes.
__device__ __forceinline__ void pack_rows_var(const uint32_t (&q)[16], int k, uint8_t *wp) {
    uint64_t acc = 0;
    uint32_t addr = smem_u32(wp);
    const uint32_t k4 = 4u * (uint32_t)k, k8 = 8u * (uint32_t)k;
    uint32_t s = 0;                                                   // bit position inside the open word: 0, 8, .., 56
#pragma unroll
    for (int r = 0; r < 8; r++) {
        // the row as a 64-bit value: q[2r] | q[2r+1] << 4k   (clamped funnel shifts: 4k == 32 is legal)
        const uint32_t rlo = q[2 * r] | __funnelshift_lc(0u, q[2 * r + 1], k4);
        const uint32_t rhi = __funnelshift_lc(q[2 * r + 1], 0u, k4);
        const uint64_t row = ((uint64_t)rhi << 32) | rlo;
        acc |= row << s;
        const uint32_t t = s + k8;
        if (t >= 64u) {                                               // the open word is complete (predicated, not a branch)
            asm volatile("st.shared.b64 [%0], %1;" ::"r"(addr), "l"(acc) : "memory");
            addr += 8u;
            // spill-over = row >> (64 - s); PTX shifts clamp at the register width, so s == 0 (depth 8) gives 0
            asm("shr.b64 %0, %1, %2;" : "=l"(acc) : "l"(row), "r"(64u - s));
        }
        s = t & 63u;
    }
}

// pack for a warp whose tiles all have depth <= 2 (low-entropy video: flat background, 1-2 bits of
// noise).  A byte-weighted dot product squeezes 4 pixels in ONE instruction when the weights
// 1, 2^k, 2^2k, 2^3k fit in bytes (IDP.4A; k <= 2), and the fields of both depths are then joined by
// the same three multiply-adds with lane-varying multipliers: no per-depth specialisation runs, no
// divergence.  px = (pixel - min); wp = the tile's 8-byte aligned staging address.  Lanes with k == 0
// compute zeros and store nothing.
__device__ __forceinline__ void pack_low_depths(const uint32_t (&px)[16], int k, uint8_t *wp) {
    const uint32_t wts = k == 2 ? 0x40100401u : 0x08040201u;
    const uint32_t m1 = 1u << (4 * k), m2 = 1u << (8 * k);
    uint32_t r[4];                                   // r[m] = tile rows 2m, 2m+1 = 16 pixels = 16k bits
#pragma unroll
    for (int m = 0; m < 4; m++) {
        const uint32_t q0 = __dp4a(px[4 * m], wts, 0u), q1 = __dp4a(px[4 * m + 1], wts, 0u);
        const uint32_t q2 = __dp4a(px[4 * m + 2], wts, 0u), q3 = __dp4a(px[4 * m + 3], wts, 0u);
        r[m] = (q0 + q1 * m1) + (q2 + q3 * m1) * m2;
    }
    const uint32_t addr = smem_u32(wp);
    if (k == 2) {
        asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(r[0]), "r"(r[1]) : "memory");
        asm volatile("st.shared.v2.u32 [%0+8], {%1, %2};" ::"r"(addr), "r"(r[2]), "r"(r[3]) : "memory");
    } else if (k == 1) {
        asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(r[0] + (r[1] << 16)), "r"(r[2] + (r[3] << 16)) : "memory");
    }
}

// ------------------------------------------------------------------ record fixed fields
// Warp-wide, after the record's last word count is known: lane i writes byte i of {I32 2 | U64 index | F64 0.0 | I32 wh}
// and the lanes above write the two counts behind the planes, {I32 mb*wh} and {I32 n64} (dbde_util.cpp:141-146,
// 182-188,191); lane 0 stores record j's offset (j slots of slot_stride bytes) and size.
__device__ __forceinline__ void write_fixed_fields(uint8_t *rec, int lane, uint64_t index, size_t wh, uint32_t mb, uint32_t n64,
                                                   uint64_t *offsets, uint64_t *sizes, uint64_t j, uint64_t slot_stride) {
    uint32_t b;
    size_t at = lane;
    if (lane < 4) b = 2u >> (8 * lane);
    else if (lane < 12) b = (uint32_t)(index >> (8 * (lane - 4)));
    else if (lane < 20) b = 0;
    else if (lane < 24) b = (uint32_t)wh >> (8 * (lane - 20));
    else if (lane < 28) { b = (uint32_t)(mb * wh) >> (8 * (lane - 24)); at = rec_min_count(wh) + (lane - 24); }
    else { b = n64 >> (8 * (lane - 28)); at = rec_n64(wh, mb) + (lane - 28); }
    rec[at] = (uint8_t)b;
    if (lane == 0) {
        offsets[j] = j * slot_stride;
        sizes[j] = rec_fixed(wh, mb) + 8ull * n64;
    }
}

// a little-endian U32 at any byte address
__device__ __forceinline__ uint32_t ld_le32(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
#endif  // __CUDACC__

}  // namespace dbde
