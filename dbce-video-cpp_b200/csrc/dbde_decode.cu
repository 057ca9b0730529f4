// DBDE B200 decoder: DBDE frame records in HBM -> raw U8 frames in HBM, pixel-identical to
// dbde_unpack_frame (dbde_util.cpp:339-345) and with its accept/reject behaviour
// (dbde_util.cpp:295-303: a rejected frame leaves the image untouched).
//
// Three kernels:
//   dbde_decode_scan_kernel   : one CTA per frame. Validates the record (header tag, plane lengths,
//                               sum(depth) == n64, depth <= 8, bounds) and turns the depth plane into
//                               exclusive U64-word prefixes at partition-warp granularity (32 tiles),
//                               i.e. the reference's running input pointer (dbde_util.cpp:312) made
//                               explicit.  Reads 1 byte per tile (~1 % of the traffic).
//   dbde_decode_kernel<MODE>  : persistent, warp-specialised.  A producer warp bulk-TMAs each
//                               partition's payload words + depth/min bytes into a ring of stages;
//                               tile warps (one lane == one 8x8 tile) unpack with shifts and masks,
//                               add the minimum and store their rows straight from registers: a
//                               warp's 32 tiles make each row store one coalesced 256-byte segment,
//                               so the warps never synchronise with each other.  MODE -1: aligned
//                               frames; -2: aligned frames with linear partitions; 0..7 = W & 7: odd
//                               geometries, rows re-aligned across lanes with compile-time shapes
//                               (what odd frames wider than 2048 run).
//   dbde_decode_staged_kernel<WM> : odd frames whose partitions span the full width (W <= 2048): the
//                               partition's pixels are built in shared memory as they lie in the frame
//                               (compile-time row shapes) and leave with one bulk-TMA store.
//   dbde_decode_binned_kernel<B> : any frame on linear partitions, each tile reduced in registers to the
//                               rounded means of its B x B blocks (B = 2, 4, 8) before it is stored.
#include "dbde_device.cuh"
#include "dbde_kernels.h"
#include <stdlib.h>

namespace dbde {

constexpr int kDecStages = 3;
// The producer keeps at most kDecStages partitions in flight, and fewer when they are large: it
// does not let the payload bytes of the issued-but-unconsumed partitions exceed this many per CTA.
// Measured (micro-2048, 4 CTAs/SM): an unconditional depth of 3 runs at 5.32 TB/s, depth 2 at 5.85 --
// the 25/75 read/write stream is fastest with ~50 KB of reads in flight per SM -- while
// low-entropy records (1.3 KB per partition) want all three (5.04 vs 4.83 TB/s).
#ifndef DBDE_DEC_INFLIGHT_BYTES
#define DBDE_DEC_INFLIGHT_BYTES 6144
#endif
constexpr uint32_t kDecInflightBytes = DBDE_DEC_INFLIGHT_BYTES;
constexpr int kDecThreads = kTilesPerPart + 32;
constexpr int kDecPayloadBytes = 64 * kTilesPerPart + 32;        // worst-case words + 16-byte hull slack
constexpr int kDecPlaneBytes = kTilesPerPart + 32;
constexpr int kDecStageBytes = ((kDecPayloadBytes + 2 * kDecPlaneBytes + 127) / 128) * 128;

// ------------------------------------------------------------------ scan / validate pre-pass
__global__ void __launch_bounds__(256) dbde_decode_scan_kernel(const DecParams P) {
    __shared__ uint32_t s_warp[8];
    __shared__ uint32_t s_flag;
    const PartGeom &g = P.g;
    const int f = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nitems = g.ppf * kConsumerWarps;
    uint32_t *wp = P.wprefix + (size_t)f * (nitems + 1);
    ScanHead h;
    if (!scan_head(P.stream, P.stream_bytes, P.frame_offsets[f], g.wh, 1, f, P.status, P.indices, h)) return;
    if (tid == 0) s_flag = 0;
    __syncthreads();

    // phase 1: depth sum of every partition-warp (32 consecutive tiles of a partition).  One warp
    // takes a whole partition per step: lane l owns tiles 8l..8l+7 (8 depth bytes, summed with
    // two IDP.4A), four lanes make one 32-tile item.  Four partitions are loaded before any is
    // reduced so four global loads are in flight per lane.
    const uint8_t *dp = h.rec + kRecDepth;
    bool big = false;
    if (g.wh == kTilesPerPart * g.ppf && (((uintptr_t)dp) & 7) == 0) {
        // Every partition is a full run of 256 tiles starting at tile 256*q and the plane is 8-byte
        // aligned (the usual case): no geometry, no edge handling -- one 8-byte load per lane per
        // partition, eight independent partitions in flight per warp.
        constexpr int kFastBatch = 8;
        for (int q0 = warp * kFastBatch; q0 < g.ppf; q0 += 8 * kFastBatch) {
            uint2 v[kFastBatch];
#pragma unroll
            for (int b = 0; b < kFastBatch; b++)
                v[b] = q0 + b < g.ppf ? *reinterpret_cast<const uint2 *>(dp + (size_t)kTilesPerPart * (q0 + b) + 8 * lane)
                                      : make_uint2(0u, 0u);
#pragma unroll
            for (int b = 0; b < kFastBatch; b++) {
                const uint32_t over = ((((v[b].x & 0x7f7f7f7fu) + 0x77777777u) | v[b].x) |
                                       (((v[b].y & 0x7f7f7f7fu) + 0x77777777u) | v[b].y)) & 0x80808080u;
                uint32_t sum;
                if (over) {                                          // rare: clamp byte-wise like the general path
                    big = true;
                    sum = 0;
                    for (int i = 0; i < 4; i++) sum += min((v[b].x >> (8 * i)) & 0xffu, 8u) + min((v[b].y >> (8 * i)) & 0xffu, 8u);
                } else {
                    sum = __dp4a(v[b].x, 0x01010101u, __dp4a(v[b].y, 0x01010101u, 0u));
                }
                sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                if (q0 + b < g.ppf && (lane & 3) == 0) wp[(q0 + b) * kConsumerWarps + (lane >> 2)] = sum;
            }
        }
    } else {
    constexpr int kBatch = 4;
    for (int q0 = warp * kBatch; q0 < g.ppf; q0 += 8 * kBatch) {
        uint32_t lo[kBatch], hi[kBatch];
#pragma unroll
        for (int b = 0; b < kBatch; b++) {
            lo[b] = hi[b] = 0;
            const int q = q0 + b;
            if (q < g.ppf) {
                const PartInfo pi = part_info(g, (unsigned)q);
                const uint8_t *src = dp + pi.tfirst + 8 * lane;
                const int left = pi.nt - 8 * lane;               // tiles this lane really owns
                if (left >= 8 && (((uintptr_t)src) & 3) == 0) {
                    lo[b] = *reinterpret_cast<const uint32_t *>(src);
                    hi[b] = *reinterpret_cast<const uint32_t *>(src + 4);
                } else {
                    for (int i = 0; i < 8; i++) {
                        const uint32_t d = i < left ? src[i] : 0u;
                        if (i < 4) lo[b] |= d << (8 * i);
                        else hi[b] |= d << (8 * (i - 4));
                    }
                }
            }
        }
#pragma unroll
        for (int b = 0; b < kBatch; b++) {
            const int q = q0 + b;
            // any byte > 8 ?  (low 7 bits + 0x77 carries into bit 7 when >= 9; bit 7 itself means >= 128)
            const uint32_t over = ((((lo[b] & 0x7f7f7f7fu) + 0x77777777u) | lo[b]) |
                                   (((hi[b] & 0x7f7f7f7fu) + 0x77777777u) | hi[b])) & 0x80808080u;
            uint32_t sum;
            if (over) {                                          // rare: clamp byte-wise like the slow path
                big = true;
                sum = 0;
                for (int i = 0; i < 4; i++) {
                    sum += min((lo[b] >> (8 * i)) & 0xffu, 8u) + min((hi[b] >> (8 * i)) & 0xffu, 8u);
                }
            } else {
                sum = __dp4a(lo[b], 0x01010101u, __dp4a(hi[b], 0x01010101u, 0u));
            }
            sum += __shfl_xor_sync(0xffffffffu, sum, 1);
            sum += __shfl_xor_sync(0xffffffffu, sum, 2);
            if (q < g.ppf && (lane & 3) == 0) wp[q * kConsumerWarps + (lane >> 2)] = sum;
        }
    }
    }
    if (big) atomicOr(&s_flag, 1u);
    __syncthreads();

    // phase 2: exclusive scan of the nitems sums
    const uint32_t total = scan_items(wp, nitems, s_warp, tid, warp, lane);
    if (tid == 0) scan_finish(h, wp, nitems, total, s_flag != 0, f, P.status, P.indices);
}

// ------------------------------------------------------------------ main kernel
struct alignas(16) DecCtl {
    int part;                  // -1 = no more work
    int skip;                  // bit 0: frame was rejected by the scan, leave the image untouched; bit 1: every band of
                               // the partition has its 8 pixel rows inside the frame (no cropped rows)
    int f;                     // frame within the batch
    int nt;                    // tiles in this partition
    uint32_t pres, kres, mres; // residual byte offsets of payload / depth / min inside their hulls
    uint32_t pixoff;           // byte offset of the partition's first pixel inside its frame
    int y0, tx0, ntx, pad1;    // first band / first tile column / tile columns (generic path)
    uint32_t wbase[kConsumerWarps];   // word offset of each tile warp inside the partition's payload
};
constexpr int kCtlSkip = 1, kCtlAllRows = 2;
template <int NSTAGES>
struct DecSmemT {
    uint64_t full[NSTAGES], empty[NSTAGES];
    uint64_t outfull[2], outempty[2];      // staged-store kernel only
    DecCtl ctl[NSTAGES];
};
using DecSmem = DecSmemT<kDecStages>;

// ------------------------------------------------------------------ generic (unaligned / cropped) row stores
// One pixel row of a warp's tiles, any alignment, cropped to `ncol` columns (dbde_util.cpp:281-289).
// Consecutive lanes of a band hold consecutive 8-byte pieces of the row, so every lane assembles the
// ALIGNED 8-byte word its piece starts in -- the tail of its left neighbour (one shuffle) plus its own
// head -- and stores it whole: a warp's row is one run of aligned 8-byte stores.  Only the ends of a
// run (first/last lane of the warp, first/last tile of the row) are written with narrower stores.
// `a` = row address & 7 is the same for every lane (bands are a multiple of 8 bytes apart).
// All 32 lanes call this (the shuffle is warp-wide); `live` says whether this lane has a row to write.
__device__ __forceinline__ void store_row_generic(uint8_t *rp, uint64_t x, int ncol, bool live, bool first_in_run,
                                                  bool last_in_run) {
    const uint64_t prev = __shfl_up_sync(0xffffffffu, x, 1);
    if (!live) return;
    const uint32_t a = (uint32_t)(uintptr_t)rp & 7u;
    if (a == 0) {
        if (ncol == 8) *reinterpret_cast<uint2 *>(rp) = make_uint2((uint32_t)x, (uint32_t)(x >> 32));
        else store_partial(rp, x, 0u, (uint32_t)ncol);
        return;
    }
    uint8_t *q = rp - a;
    const uint32_t sh = 8u * a;
    uint64_t w = x << sh;
    if (!first_in_run) w |= prev >> (64u - sh);
    const uint32_t s = first_in_run ? a : 0u;
    const uint32_t e = min(8u, a + (uint32_t)ncol);
    if (s == 0u && e == 8u) *reinterpret_cast<uint2 *>(q) = make_uint2((uint32_t)w, (uint32_t)(w >> 32));
    else store_partial(q, w, s, e);
    // my bytes past the word boundary: the next lane's word carries them unless I end the run
    if (last_in_run && a + (uint32_t)ncol > 8u) store_partial(q + 8, x >> (64u - sh), 0u, a + (uint32_t)ncol - 8u);
}

// ------------------------------------------------------------------ direct re-aligned row stores (odd sizes)
// An odd-size frame's rows start at any byte address, so a lane's 8-byte row piece straddles two
// aligned words.  Consecutive lanes of a band hold consecutive pieces of the same image row, so every
// lane builds ONE aligned 8-byte word out of its own piece and a neighbour's (a single shuffle plus two
// funnel shifts) and stores it: a warp's row is one coalesced run of aligned 8-byte stores straight from
// registers -- no shared-memory image, no store warp, no barrier between tile warps.
//   alignment a = (row address) & 7 is the same for every lane (bands are multiples of 8 bytes apart);
//   a == 0      : the piece is the word
//   a in 1..4   : word at T - a     = [left neighbour's last a bytes | my first 8 - a]   (needs the neighbour's high half)
//   a in 5..7   : word at T + 8 - a = [my last a bytes | right neighbour's first 8 - a] (needs the neighbour's low half)
// With W & 7 a template parameter and the partition's first alignment a switch case, every row's
// shape and shift amount is a compile-time constant.  What the words cannot cover -- the first 8 - a
// bytes of a run's first lane and the last a bytes of its last lane -- those two lanes store as at most
// three naturally aligned narrow pieces per row, also of compile-time shape (store_row_ends).
// (Measured alternative: the end lanes leave their pixels in a per-warp scratch and a per-partition
// boundary pass -- lane = (run, row, end) -- writes the pieces: 12 % slower, mix-1001x1003 3.57 vs 4.05 TB/s.)
__device__ __forceinline__ void stg_u64(uint8_t *p, uint32_t lo, uint32_t hi) {
    asm volatile("st.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(lo), "r"(hi) : "memory");
}
__device__ __forceinline__ void stg_u32(uint8_t *p, uint32_t v) { asm volatile("st.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ void stg_u16(uint8_t *p, uint32_t v) {
    asm volatile("{ .reg .b16 t; cvt.u16.u32 t, %1; st.global.u16 [%0], t; }" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void stg_u8(uint8_t *p, uint32_t v) { asm volatile("st.global.u8 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

constexpr uint32_t kDirFull = 1, kDirFirst = 2, kDirLast = 4, kDirPartial = 8;
// Where this lane's tile sits in its image row: kDirFull (all 8 columns inside the frame), kDirFirst / kDirLast
// (no full tile of the same band in the lane to the left / right: a run of re-aligned words starts / ends
// here), kDirPartial (the frame's last column when W % 8 != 0) | its column count << 8.
// tx0/ntx: the partition's first tile column and tile columns; tiles_max: tiles a partition can hold.
__device__ __forceinline__ uint32_t direct_lane_flags(const PartGeom &g, int tid, int lane, int stx, int tx0, int ntx, int tiles_max) {
    const bool ingeo = tid < tiles_max;
    const int ncol = ingeo ? min(8, g.W - 8 * (tx0 + stx)) : 0;       // lanes past the partition's tiles: nothing
    const bool full = ingeo && ncol == 8;
    const bool left_full = lane > 0 && stx > 0;                                           // only a last column can be partial
    const bool right_full = lane < 31 && stx + 1 < ntx && g.W - 8 * (tx0 + stx + 1) >= 8;
    return (full ? kDirFull : 0u) | (full && !left_full ? kDirFirst : 0u) | (full && !right_full ? kDirLast : 0u) |
           (ingeo && ncol < 8 ? kDirPartial : 0u) | ((uint32_t)ncol << 8);
}

// bytes [O, O + 4) of the 8-byte row {lo, hi}, O a compile-time constant (zero-filled past byte 7)
template <int O>
__device__ __forceinline__ uint32_t row_bytes_from(uint32_t lo, uint32_t hi) {
    if constexpr (O == 0) return lo;
    else if constexpr (O < 4) return __funnelshift_r(lo, hi, 8 * O);
    else if constexpr (O == 4) return hi;
    else return hi >> (8 * (O - 4));
}
// The pieces of a row that the aligned words cannot cover, shapes known at compile time: the first
// N = 8 - A bytes of a run's first lane (ascending sizes from the row address) and the last A bytes of
// its last lane (descending sizes from the 8-byte boundary), every store naturally aligned.
template <int A>
__device__ __forceinline__ void store_row_ends(uint8_t *rp, uint32_t lo, uint32_t hi, bool first, bool last) {
    constexpr int N = 8 - A;
    if (first) {
        if constexpr ((N & 1) != 0) stg_u8(rp, lo);
        if constexpr ((N & 2) != 0) stg_u16(rp + (N & 1), row_bytes_from<(N & 1)>(lo, hi));
        if constexpr ((N & 4) != 0) stg_u32(rp + (N & 3), row_bytes_from<(N & 3)>(lo, hi));
    }
    if (last) {
        constexpr int S = 8 - A;
        if constexpr ((A & 4) != 0) stg_u32(rp + S, row_bytes_from<S>(lo, hi));
        if constexpr ((A & 2) != 0) stg_u16(rp + S + (A & 4), row_bytes_from<S + (A & 4)>(lo, hi));
        if constexpr ((A & 1) != 0) stg_u8(rp + S + (A & 6), row_bytes_from<S + (A & 6)>(lo, hi));
    }
}

// the eight rows of every lane's tile, alignment of row 0 = A0, frame width & 7 = WM.  Warp-wide call.
template <int WM, int A0, int R>
__device__ __forceinline__ void store_rows_direct_from(uint8_t *rp, size_t W, const uint32_t (&px)[16], bool full, bool has_left,
                                                       bool has_right, bool efirst, bool elast) {
    if constexpr (R < 8) {
        constexpr int a = (A0 + R * WM) & 7;
        const uint32_t lo = px[2 * R], hi = px[2 * R + 1];
        if constexpr (a == 0) {
            if (full) stg_u64(rp, lo, hi);
        } else if constexpr (a <= 4) {
            const uint32_t ph = __shfl_up_sync(0xffffffffu, hi, 1);
            const uint32_t w0 = a == 4 ? ph : __funnelshift_l(ph, lo, 8 * a);
            const uint32_t w1 = a == 4 ? lo : __funnelshift_l(lo, hi, 8 * a);
            if (has_left) stg_u64(rp - a, w0, w1);
        } else {
            const uint32_t nl = __shfl_down_sync(0xffffffffu, lo, 1);
            const uint32_t w0 = __funnelshift_r(lo, hi, 8 * (8 - a)), w1 = __funnelshift_r(hi, nl, 8 * (8 - a));
            if (has_right) stg_u64(rp + (8 - a), w0, w1);
        }
        if constexpr (a != 0) store_row_ends<a>(rp, lo, hi, efirst, elast);
        store_rows_direct_from<WM, A0, R + 1>(rp + W, W, px, full, has_left, has_right, efirst, elast);
    }
}
template <int WM, int A0>
__device__ __forceinline__ void store_rows_direct(uint8_t *rp, size_t W, const uint32_t (&px)[16], bool full, bool first,
                                                  bool last) {
    store_rows_direct_from<WM, A0, 0>(rp, W, px, full, full && !first, full && !last, full && first, full && last);
}
template <int WM>
__device__ __forceinline__ void store_rows_direct_any(uint32_t a0, uint8_t *rp, size_t W, const uint32_t (&px)[16], bool full,
                                                      bool first, bool last) {
    switch (a0 & 7u) {
        case 0: store_rows_direct<WM, 0>(rp, W, px, full, first, last); break;
        case 1: store_rows_direct<WM, 1>(rp, W, px, full, first, last); break;
        case 2: store_rows_direct<WM, 2>(rp, W, px, full, first, last); break;
        case 3: store_rows_direct<WM, 3>(rp, W, px, full, first, last); break;
        case 4: store_rows_direct<WM, 4>(rp, W, px, full, first, last); break;
        case 5: store_rows_direct<WM, 5>(rp, W, px, full, first, last); break;
        case 6: store_rows_direct<WM, 6>(rp, W, px, full, first, last); break;
        default: store_rows_direct<WM, 7>(rp, W, px, full, first, last); break;
    }
}

// ------------------------------------------------------------------ one lane == one tile: stage -> pixels
// Reads the tile's depth and minimum from the staged planes and finds its k words in the staged payload,
// returns the 64 pixels (+min applied) in px.  Warp-wide call (scan + vote).
__device__ __forceinline__ void dec_unpack_tile(const uint8_t *stage, const uint4 &c1, uint32_t wbase, int tid, int lane,
                                                bool valid, bool invert, uint32_t (&px)[16]) {
    const uint32_t pres = c1.x;
    int k = 0;
    uint32_t mn = 0;
    if (valid) {
        k = stage[kDecPayloadBytes + c1.y + tid];
        mn = stage[kDecPayloadBytes + kDecPlaneBytes + c1.z + tid];
    }
    const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
    const uint32_t woff = wbase + incl - (uint32_t)k;
    unpack_tile(stage + pres + 8 * (size_t)woff, k, mn * 0x01010101u, (pres & 7u) == 0, invert, px);
}

// ------------------------------------------------------------------ producer warp (both unpack kernels)
// INFLIGHT: payload bytes the producer lets a CTA have in flight (adaptive depth), see kDecInflightBytes.
template <int NSTAGES, uint32_t INFLIGHT>
__device__ __forceinline__ void dec_producer(const DecParams &P, DecSmemT<NSTAGES> &S, uint8_t *stages, int lane) {
    const PartGeom &g = P.g;
    const int nitems = g.ppf * kConsumerWarps;
    // ============================ producer warp ============================
    // static round-robin: nothing waits on another CTA here, so no ticket is needed and the
    // next partition's bookkeeping loads can be issued one iteration early
    unsigned p = blockIdx.x;
    uint32_t nx_status = 0, nx_v = 0;
    uint64_t nx_off = 0;
    auto prefetch = [&](unsigned pp) {
        if (pp < P.nparts) {
            const PartInfo pi = part_info(g, pp);
            nx_status = P.status[pi.f];
            nx_off = P.frame_offsets[pi.f];
            nx_v = lane <= kConsumerWarps ? P.wprefix[(size_t)pi.f * (nitems + 1) + pi.q * kConsumerWarps + lane] : 0u;
        }
    };
    prefetch(p);
    uint32_t b1 = 0, b2 = 0;                   // payload bytes of the two previous iterations
    for (unsigned it = 0;; it++, p += gridDim.x) {
        const int s = it % NSTAGES;
        const uint32_t ph = (it / NSTAGES) & 1;
        const uint32_t status = nx_status, v = nx_v;
        const uint64_t off = nx_off;
        prefetch(p + gridDim.x);
        mbar_wait_sleepy(&S.empty[s], ph ^ 1);
        if (p >= P.nparts) {
            if (lane == 0) {
                S.ctl[s].part = -1;
                mbar_arrive(&S.full[s]);
            }
            break;
        }
        if (status != 0) {
            if (lane == 0) {
                *reinterpret_cast<int2 *>(&S.ctl[s].part) = make_int2((int)p, kCtlSkip);
                mbar_arrive(&S.full[s]);
            }
            b2 = b1;
            b1 = 0;
            continue;
        }
        const PartInfo pi = part_info(g, p);
        const uint8_t *rec = P.stream + off;
        const uint32_t v0 = __shfl_sync(0xffffffffu, v, 0), v8 = __shfl_sync(0xffffffffu, v, kConsumerWarps);
        const uint32_t agg = v8 - v0;
        // adaptive depth: with large payloads, wait until the partition issued two iterations ago
        // has been consumed (at most two in flight) before adding this one
        if (NSTAGES > 2 && it >= 2 && 8u * agg + b1 + b2 > INFLIGHT)
            mbar_wait_sleepy(&S.empty[(it - 2) % NSTAGES], ((it - 2) / NSTAGES) & 1);
        b2 = b1;
        b1 = 8u * agg;
        uint8_t *stage = stages + (size_t)s * kDecStageBytes;
        // lane 0: payload words, lane 1: depth bytes, lane 2: minimum bytes (16-byte hulls)
        const uint8_t *src = nullptr;
        uint32_t nbytes = 0;
        uint8_t *dst = stage;
        if (lane == 0) { src = rec + rec_fixed(g.wh, 1) + 8ull * v0; nbytes = 8 * agg; }
        if (lane == 1) { src = rec + kRecDepth + pi.tfirst; nbytes = (uint32_t)pi.nt; dst = stage + kDecPayloadBytes; }
        if (lane == 2) { src = rec + rec_min(g.wh) + pi.tfirst; nbytes = (uint32_t)pi.nt; dst = stage + kDecPayloadBytes + kDecPlaneBytes; }
        const uintptr_t a0 = (uintptr_t)src & ~(uintptr_t)15;
        const uintptr_t a1 = ((uintptr_t)src + nbytes + 15) & ~(uintptr_t)15;
        const uint32_t len = nbytes ? (uint32_t)(a1 - a0) : 0u;
        const uint32_t res = (uint32_t)((uintptr_t)src - a0);
        if (lane < kConsumerWarps) S.ctl[s].wbase[lane] = v - v0;
        // lanes 0..2 hold the three residuals: gather them so lane 0 writes the block with two 16-byte stores
        const uint32_t kres = __shfl_sync(0xffffffffu, res, 1), mres = __shfl_sync(0xffffffffu, res, 2);
        if (lane == 0) {
            *reinterpret_cast<int4 *>(&S.ctl[s].part) =
                make_int4((int)p, 8 * (pi.y0 + pi.nbands) <= g.H ? kCtlAllRows : 0, pi.f, pi.nt);
            *reinterpret_cast<uint4 *>(&S.ctl[s].pres) =
                make_uint4(res, kres, mres, (uint32_t)(8 * pi.y0) * (uint32_t)g.W + 8u * (uint32_t)pi.tx0);
            // pad1: low 32 bits of the global address of the partition's first pixel (its alignment decides the
            // staged kernel's shared-memory image shift and row-store shapes)
            const uint32_t pixoff = (uint32_t)(8 * pi.y0) * (uint32_t)g.W + 8u * (uint32_t)pi.tx0;
            *reinterpret_cast<int4 *>(&S.ctl[s].y0) =
                make_int4(pi.y0, pi.tx0, pi.ntx, (int)(uint32_t)((uintptr_t)P.frames + (size_t)pi.f * ((size_t)g.W * g.H) + pixoff));
        }
        const uint32_t total = __reduce_add_sync(0xffffffffu, lane < 3 ? len : 0u);
        __syncwarp();
        if (lane == 0) mbar_arrive_expect_tx(&S.full[s], total);
        __syncwarp();
        if (lane < 3 && len) tma_load_1d(dst, (const void *)a0, len, &S.full[s]);
    }
}

// MODE -1: aligned frames (W % 16 == 0, H % 8 == 0, 16-byte aligned base): rows are stored as they are.
// MODE -2: the same with linear partitions (make_geom): a lane finds its tile's band and column per partition.
// MODE 0..7 = W & 7: every other geometry; rows are re-aligned across lanes (store_rows_direct) unless the
//           partition has cropped rows (the frame's last band when H % 8 != 0), which are stored piecewise.
template <int MODE>
__global__ void __launch_bounds__(kDecThreads, MODE == -1 ? 3 : 4) dbde_decode_kernel(const DecParams P) {
    constexpr bool FAST = MODE < 0;
    constexpr bool LIN = MODE == -2;          // aligned frame, linear partitions (a separate instantiation: its
                                              // per-lane tile arithmetic must not cost the plain aligned kernel registers)
    extern __shared__ __align__(128) uint8_t smem_raw[];
    DecSmem &S = *reinterpret_cast<DecSmem *>(smem_raw);
    uint8_t *stages = smem_raw + ((sizeof(DecSmem) + 127) & ~127);
    const PartGeom &g = P.g;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t fbytes = (size_t)g.W * g.H;

    if (tid == 0) {
        for (int s = 0; s < kDecStages; s++) {
            mbar_init(&S.full[s], 1);
            mbar_init(&S.empty[s], kConsumerWarps);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        dec_producer<kDecStages, kDecInflightBytes>(P, S, stages, lane);
    } else {
        // ============================ tile warps: one lane == one 8x8 tile ============================
        int sb = 0, stx = tid;
        if (g.nseg == 1 && g.G > 1) {
            sb = tid / g.w;
            stx = tid - sb * g.w;
        }
        const uint32_t toff = (uint32_t)(8 * sb) * (uint32_t)g.W + 8u * (uint32_t)stx;   // my tile inside a partition's pixels
        const size_t rowstride = (size_t)g.W;
        // linear partitions (aligned frames only): my tile is tile tid after the partition's first one, i.e.
        // lin_dy bands down and lin_dx columns right of it, wrapping once more if that passes the last column
        const int lin_dy = LIN ? tid / g.w : 0, lin_dx = LIN ? tid - lin_dy * g.w : 0;
        // direct re-aligned stores: a lane's place in its image row is fixed for full-width partitions and is
        // worked out per partition for band segments of wider frames (the last segment is shorter)
        uint32_t dflags = 0;
        if (!FAST && g.nseg == 1) dflags = direct_lane_flags(g, tid, lane, stx, 0, g.w, g.G * g.w);
        for (unsigned it = 0;; it++) {
            const int s = it % kDecStages;
            const uint32_t ph = (it / kDecStages) & 1;
            mbar_wait(&S.full[s], ph);
            const int4 c0 = *reinterpret_cast<const int4 *>(&S.ctl[s].part);      // part, flags, f, nt
            if (c0.x < 0) break;
            if (c0.y & kCtlSkip) {
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.empty[s]);
                continue;
            }
            const uint4 c1 = *reinterpret_cast<const uint4 *>(&S.ctl[s].pres);    // pres, kres, mres, pixoff
            int4 c2 = make_int4(0, 0, 0, 0);
            if (!FAST) c2 = *reinterpret_cast<const int4 *>(&S.ctl[s].y0);        // y0, tx0, ntx, image address (low 32 bits)
            const uint8_t *stage = stages + (size_t)s * kDecStageBytes;
            const bool valid = tid < c0.w;
            uint32_t px[16];
            dec_unpack_tile(stage, c1, S.ctl[s].wbase[warp], tid, lane, valid, (P.flags & kFlagInvertRows) != 0, px);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.empty[s]);       // payload is in registers: free the stage early

            uint8_t *const part0 = P.frames + (size_t)c0.z * fbytes + c1.w;       // the partition's first pixel
            uint8_t *rp = part0 + toff;
            if (LIN) {
                const int2 c2l = *reinterpret_cast<const int2 *>(&S.ctl[s].y0);   // first tile's band and column
                int ty = c2l.x + lin_dy, tx = c2l.y + lin_dx;
                if (tx >= g.w) {
                    tx -= g.w;
                    ty++;
                }
                rp = P.frames + (size_t)c0.z * fbytes + ((size_t)(8 * ty) * g.W + 8 * (size_t)tx);
            }
            if (FAST) {
                // no edges, 8-byte aligned rows: lane t stores 8 bytes of each row, a warp 256 contiguous bytes
                if (valid) {
#pragma unroll
                    for (int r = 0; r < 8; r++) {
                        st_stream_u64(rp, ((uint64_t)px[2 * r + 1] << 32) | px[2 * r]);
                        rp += rowstride;
                    }
                }
            } else if (c0.y & kCtlAllRows) {
                if (g.nseg > 1) dflags = direct_lane_flags(g, tid, lane, stx, c2.y, c2.z, c2.z);
                store_rows_direct_any<(MODE < 0 ? 0 : MODE)>((uint32_t)c2.w, rp, rowstride, px, valid && (dflags & kDirFull),
                                                             (dflags & kDirFirst) != 0, (dflags & kDirLast) != 0);
                if (valid && (dflags & kDirPartial)) {
                    // the frame's last tile column when W % 8 != 0 (dbde_util.cpp:281-289): its columns byte by byte
                    const int ncol = (int)((dflags >> 8) & 15u);
                    for (int c = 0; c < ncol; c++) {
                        const uint32_t sh = 8u * (uint32_t)(c & 3);
                        uint8_t *q = rp + c;
#pragma unroll
                        for (int r = 0; r < 8; r++) {
                            stg_u8(q, ((c & 4) ? px[2 * r + 1] : px[2 * r]) >> sh);
                            q += rowstride;
                        }
                    }
                }
            } else {
                // crop the padding (dbde_util.cpp:281-289): only rows < H and columns < W are written
                const int rows_valid = valid ? min(8, g.H - 8 * (c2.x + sb)) : 0;
                const int ncol = min(8, g.W - 8 * (c2.y + stx));
                const bool first_in_run = lane == 0 || stx == 0;
                const bool last_in_run = lane == 31 || stx == c2.z - 1 || tid + 1 >= c0.w;
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    store_row_generic(rp, ((uint64_t)px[2 * r + 1] << 32) | px[2 * r], ncol, r < rows_valid, first_in_run,
                                      last_in_run);
                    rp += rowstride;
                }
            }
        }
    }
}

// ------------------------------------------------------------------ binned decode (B x B block means)
// Bin sums of a tile whose px[i] hold the 16-bit sums of their two byte pairs (px[2r] = [c0+c1, c2+c3] of row r,
// px[2r+1] = [c4+c5, c6+c7]).  Bin row j of the tile's 8 / B; the sums come back as 16-bit halves:
//   B = 2: s0 = [bin 0, bin 1], s1 = [bin 2, bin 3];  B = 4: s0 = [bin 0, bin 1];  B = 8: s0 = bin 0.
// The largest, an 8x8 sum, is 64 * 255 = 16320: no half ever carries into the next.
template <int B>
__device__ __forceinline__ void bin_row_sums(const uint32_t (&px)[16], int j, uint32_t &s0, uint32_t &s1) {
    s1 = 0;
    if constexpr (B == 2) {
        s0 = px[4 * j] + px[4 * j + 2];
        s1 = px[4 * j + 1] + px[4 * j + 3];
    } else if constexpr (B == 4) {
        const uint32_t a0 = px[8 * j] + px[8 * j + 2] + px[8 * j + 4] + px[8 * j + 6];
        const uint32_t a1 = px[8 * j + 1] + px[8 * j + 3] + px[8 * j + 5] + px[8 * j + 7];
        s0 = __byte_perm(a0, a1, 0x5410) + __byte_perm(a0, a1, 0x7632);
    } else {
        uint32_t a = 0;
#pragma unroll
        for (int i = 0; i < 16; i++) a += px[i];
        s0 = (a & 0xffffu) + (a >> 16);
    }
}

// n <= 4 bytes of v to p, any alignment, as naturally aligned pieces
__device__ __forceinline__ void store_bytes(uint8_t *p, uint32_t v, uint32_t n) {
    const uint32_t a = (uint32_t)(uintptr_t)p & 7u;
    uint8_t *q = p - a;
    if (a + n <= 8u) {
        store_partial(q, (uint64_t)v << (8 * a), a, a + n);
    } else {
        store_partial(q, (uint64_t)v << (8 * a), a, 8u);
        store_partial(q + 8, v >> (8 * (8 - a)), 0u, a + n - 8u);
    }
}

// The full decoder's pipeline (dec_producer, dec_unpack_tile) on linear partitions, with each lane's 64 pixels
// reduced in registers to the (8 / B)^2 rounded means of its B x B bins before anything is stored: a lane writes
// 8 / B pieces of 8 / B bytes, one per bin row, and the 4 MiB full-size frame never exists.  Interior tiles divide by
// shifting; the frame's last tile column / row (W % 8 or H % 8 != 0) first zeroes the encoder's clamp padding past
// W and H -- it must not enter the mean -- and divides each bin by its count of in-frame pixels.
template <int B>
__global__ void __launch_bounds__(kDecThreads, 4) dbde_decode_binned_kernel(const DecParams P) {
    constexpr int NB = 8 / B;                 // bins per tile side
    extern __shared__ __align__(128) uint8_t smem_raw[];
    DecSmem &S = *reinterpret_cast<DecSmem *>(smem_raw);
    uint8_t *stages = smem_raw + ((sizeof(DecSmem) + 127) & ~127);
    const PartGeom &g = P.g;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int Wb = (g.W + B - 1) / B, Hb = (g.H + B - 1) / B;
    const size_t fbytes = (size_t)Wb * (size_t)Hb;

    if (tid == 0) {
        for (int s = 0; s < kDecStages; s++) {
            mbar_init(&S.full[s], 1);
            mbar_init(&S.empty[s], kConsumerWarps);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        dec_producer<kDecStages, kDecInflightBytes>(P, S, stages, lane);
        return;
    }
    // my tile is tile tid after the partition's first one: lin_dy bands down, lin_dx columns right, wrapping once
    // more if that passes the last column
    const int lin_dy = tid / g.w, lin_dx = tid - lin_dy * g.w;
    for (unsigned it = 0;; it++) {
        const int s = it % kDecStages;
        const uint32_t ph = (it / kDecStages) & 1;
        mbar_wait(&S.full[s], ph);
        const int4 c0 = *reinterpret_cast<const int4 *>(&S.ctl[s].part);      // part, flags, f, nt
        if (c0.x < 0) break;
        if (c0.y & kCtlSkip) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.empty[s]);
            continue;
        }
        const uint4 c1 = *reinterpret_cast<const uint4 *>(&S.ctl[s].pres);    // pres, kres, mres, pixoff
        const int2 c2 = *reinterpret_cast<const int2 *>(&S.ctl[s].y0);        // first tile's band and column
        const uint8_t *stage = stages + (size_t)s * kDecStageBytes;
        const bool valid = tid < c0.w;
        uint32_t px[16];
        dec_unpack_tile(stage, c1, S.ctl[s].wbase[warp], tid, lane, valid, (P.flags & kFlagInvertRows) != 0, px);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.empty[s]);       // payload is in registers: free the stage early
        if (!valid) continue;

        int ty = c2.x + lin_dy, tx = c2.y + lin_dx;
        if (tx >= g.w) {
            tx -= g.w;
            ty++;
        }
        const int wc = g.W - 8 * tx, hr = g.H - 8 * ty;                    // in-frame columns / rows of the tile, if < 8
        const bool edge = wc < 8 || hr < 8;
        if (edge) {
            // the clamp padding past W and H (after the invert-endian row reversal) leaves the sums
            const uint32_t mlo = wc >= 4 ? ~0u : (1u << (8 * wc)) - 1u;
            const uint32_t mhi = wc >= 8 ? ~0u : wc > 4 ? (1u << (8 * (wc - 4))) - 1u : 0u;
#pragma unroll
            for (int r = 0; r < 8; r++) {
                px[2 * r] = r < hr ? px[2 * r] & mlo : 0u;
                px[2 * r + 1] = r < hr ? px[2 * r + 1] & mhi : 0u;
            }
        }
#pragma unroll
        for (int i = 0; i < 16; i++) px[i] = (px[i] & 0x00ff00ffu) + ((px[i] >> 8) & 0x00ff00ffu);

        uint8_t *op = P.frames + (size_t)c0.z * fbytes + (size_t)(NB * ty) * (size_t)Wb + (size_t)(NB * tx);
        if (!edge) {
#pragma unroll
            for (int j = 0; j < NB; j++) {
                uint32_t s0, s1;
                bin_row_sums<B>(px, j, s0, s1);
                if constexpr (B == 2) {
                    const uint32_t m0 = ((s0 + 0x00020002u) >> 2) & 0x00ff00ffu, m1 = ((s1 + 0x00020002u) >> 2) & 0x00ff00ffu;
                    const uint32_t v = __byte_perm(m0, m1, 0x6420);
                    if (((uintptr_t)op & 3u) == 0) st_stream_u32(op, v);
                    else store_bytes(op, v, 4u);
                } else if constexpr (B == 4) {
                    const uint32_t m = ((s0 + 0x00080008u) >> 4) & 0x00ff00ffu;
                    const uint32_t v = __byte_perm(m, 0u, 0x4420);
                    if (((uintptr_t)op & 1u) == 0) *reinterpret_cast<uint16_t *>(op) = (uint16_t)v;
                    else store_bytes(op, v, 2u);
                } else {
                    *op = (uint8_t)((s0 + 32u) >> 6);
                }
                op += Wb;
            }
        } else {
            // the frame's last tile column / row: bins past W / H are not in the output, the others divide their sum
            // by their in-frame pixel count, rounded half up
            const int ncb = min(NB, Wb - NB * tx), nrb = min(NB, Hb - NB * ty);
#pragma unroll
            for (int j = 0; j < NB; j++) {                 // unrolled: px is indexed with constants only
                if (j < nrb) {
                    uint32_t s0, s1;
                    bin_row_sums<B>(px, j, s0, s1);
                    const uint32_t rows = (uint32_t)min(B, hr - B * j);
                    uint32_t v = 0;
                    for (int i = 0; i < ncb; i++) {
                        const uint32_t sum = B == 8 ? s0 : ((i < 2 ? s0 : s1) >> (16 * (i & 1))) & 0xffffu;
                        const uint32_t n = rows * (uint32_t)min(B, wc - B * i);
                        v |= ((sum + n / 2) / n) << (8 * i);
                    }
                    store_bytes(op, v, (uint32_t)ncb);
                }
                op += Wb;
            }
        }
    }
}

// ------------------------------------------------------------------ staged-store kernel (odd sizes, W <= 2048)
// Frames whose rows are not 8-byte aligned (W % 8 != 0), or that end in partial tiles, cannot use the
// direct row stores: a warp's row would be cut into unaligned pieces.  But a full-width partition's
// pixels are ONE contiguous byte range of the frame -- rows 8*y0 .. of W bytes each, back to back --
// so the tile warps build that range in shared memory exactly as it lies in global memory (row pitch
// W, shifted by the range's global address mod 16 so both sides agree on 16-byte boundaries), and a
// store warp sends the 16-byte-aligned interior out with ONE bulk-TMA store (cp.async.bulk
// shared -> global, SASS UBLKCP) and the < 16 head and tail bytes with byte stores.  The crop of
// dbde_unpack_8x8_partial (dbde_util.cpp:281-289) happens on the way into shared memory: lanes of the
// last tile column write only their valid columns, rows past H are not written at all.
//   warps 0-7 tile warps, warp 8 producer (loads), warp 9 store warp.
// Measured on mix/micro/noise/low 1001x1003: 3 input stages (2 CTAs/SM) -11 %; spinning instead of sleeping in
// the store warp: no change; without the bulk store: -3 % time; without the shared-memory row stores:
// -30 % -- the unaligned row stores (narrow pieces, 2-way bank conflicts), not the TMA traffic, are the cost.
// Tried instead: tile warps store aligned 8-byte rows at a 16-byte-multiple pitch and the store warp
// re-aligns row by row (2 x LDS.128 + 4 funnel shifts + one 16-byte global store per chunk): correct, but
// 2x SLOWER (0.85 vs 0.43 ms per 1000 frames) -- ~90 instructions per image row on ONE warp that gets a
// seventh of its scheduler; spread over the tile warps it would cost what the narrow stores cost now.
constexpr int kStgStages = 2;                                    // input stages
// One output image per CTA: 2 x 17 KiB in + 16.5 KiB out = 4 CTAs/SM.  Measured against two images (3 CTAs/SM):
// +7-10 % on every 1001x1003 workload (mix 3.54 -> 3.81 TB/s) -- a fourth CTA hides more than a second image does.
constexpr int kStgOut = 1;                                       // output images
constexpr int kStgThreads = kTilesPerPart + 64;
constexpr int kStgOutBytes = 64 * kTilesPerPart + 128;           // image of <= 16 KiB + the 16-byte shift, 128-byte multiple
using StgSmem = DecSmemT<kStgStages>;

__device__ __forceinline__ void tma_store_1d(void *gdst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void sts_u8(uint32_t addr, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u16(uint32_t addr, uint32_t v) {
    asm volatile("{ .reg .b16 t; cvt.u16.u32 t, %1; st.shared.u16 [%0], t; }" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_v2u32(uint32_t addr, uint32_t lo, uint32_t hi) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(lo), "r"(hi) : "memory");
}
// The eight rows of a tile with every alignment known at compile time (WM = W & 7, A0 = alignment of row 0,
// a switch case per partition): each row is its naturally aligned pieces at immediate offsets with constant
// shifts -- 8 | 4+4 | 2+4+2 | 1+2+4+1 | 1+4+2+1 -- and no alignment test is executed per row.
template <int WM, int A0>
__device__ __forceinline__ void sts_rows_static(uint32_t rp, uint32_t W, const uint32_t (&px)[16]) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int a = (A0 + r * WM) & 7;                       // compile-time after unrolling
        const uint32_t lo = px[2 * r], hi = px[2 * r + 1];
        if (a == 0) {
            sts_v2u32(rp, lo, hi);
        } else if (a == 4) {
            sts_u32(rp, lo);
            sts_u32(rp + 4, hi);
        } else if ((a & 1) == 0) {                             // 2, 6
            sts_u16(rp, lo);
            sts_u32(rp + 2, __funnelshift_r(lo, hi, 16));
            sts_u16(rp + 6, hi >> 16);
        } else if ((a & 3) == 1) {                             // 1, 5: rp + 3 is the 4-byte boundary
            sts_u8(rp, lo);
            sts_u16(rp + 1, lo >> 8);
            sts_u32(rp + 3, __funnelshift_r(lo, hi, 24));
            sts_u8(rp + 7, hi >> 24);
        } else {                                               // 3, 7: rp + 1 is the 4-byte boundary
            sts_u8(rp, lo);
            sts_u32(rp + 1, __funnelshift_r(lo, hi, 8));
            sts_u16(rp + 5, hi >> 8);
            sts_u8(rp + 7, hi >> 24);
        }
        rp += W;
    }
}
template <int WM>
__device__ __forceinline__ void sts_rows_static_any(uint32_t a0, uint32_t rp, uint32_t W, const uint32_t (&px)[16]) {
    switch (a0 & 7u) {
        case 0: sts_rows_static<WM, 0>(rp, W, px); break;
        case 1: sts_rows_static<WM, 1>(rp, W, px); break;
        case 2: sts_rows_static<WM, 2>(rp, W, px); break;
        case 3: sts_rows_static<WM, 3>(rp, W, px); break;
        case 4: sts_rows_static<WM, 4>(rp, W, px); break;
        case 5: sts_rows_static<WM, 5>(rp, W, px); break;
        case 6: sts_rows_static<WM, 6>(rp, W, px); break;
        default: sts_rows_static<WM, 7>(rp, W, px); break;
    }
}

template <int WM>
__global__ void __launch_bounds__(kStgThreads, kStgOut == 1 ? 4 : 3) dbde_decode_staged_kernel(const DecParams P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    StgSmem &S = *reinterpret_cast<StgSmem *>(smem_raw);
    uint8_t *stages = smem_raw + ((sizeof(StgSmem) + 127) & ~127);
    uint8_t *outst = stages + (size_t)kStgStages * kDecStageBytes;
    const PartGeom &g = P.g;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t fbytes = (size_t)g.W * g.H;

    if (tid == 0) {
        for (int s = 0; s < kStgStages; s++) {
            mbar_init(&S.full[s], 1);
            mbar_init(&S.empty[s], kConsumerWarps + 1);        // tile warps + the store warp (reads the control block)
        }
        for (int s = 0; s < 2; s++) {
            mbar_init(&S.outfull[s], kConsumerWarps);
            mbar_init(&S.outempty[s], 1);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        dec_producer<kStgStages, 0xffffffffu>(P, S, stages, lane);
    } else if (warp == kConsumerWarps + 1) {
        // ============================ store warp ============================
        unsigned oi = 0;                                   // partitions actually stored (skipped frames do not count)
        for (unsigned it = 0;; it++) {
            const int s = it % kStgStages;
            mbar_wait_sleepy(&S.full[s], (it / kStgStages) & 1);
            const int4 c0 = *reinterpret_cast<const int4 *>(&S.ctl[s].part);      // part, skip, f, nt
            const uint32_t pixoff = S.ctl[s].pixoff;
            const int y0 = S.ctl[s].y0;
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.empty[s]);
            if (c0.x < 0) break;
            if (c0.y & kCtlSkip) continue;
            const int os = oi % kStgOut;
            const int nbands = c0.w / g.w;
            const int rows = min(8 * nbands, g.H - 8 * y0);
            const uint32_t n = (uint32_t)rows * (uint32_t)g.W;
            uint8_t *g0 = P.frames + (size_t)c0.z * fbytes + pixoff;
            const uint32_t a16 = (uint32_t)(uintptr_t)g0 & 15u;
            const uint8_t *img = outst + (size_t)os * kStgOutBytes + a16;          // img[i] <-> g0[i]
            const uint32_t head = min((16u - a16) & 15u, n);                       // bytes before the first 16-byte boundary
            const uint32_t mid = (n - head) & ~15u;                                // the aligned interior
            const uint32_t tail = n - head - mid;
            mbar_wait_sleepy(&S.outfull[os], (oi / kStgOut) & 1);
            if (lane == 0 && mid) tma_store_1d(g0 + head, img + head, mid);
            if (lane == 0) tma_store_commit();
            if (lane < 16) {
                if ((uint32_t)lane < head) g0[lane] = img[lane];
            } else {
                const uint32_t i = head + mid + (uint32_t)(lane - 16);
                if ((uint32_t)(lane - 16) < tail) g0[i] = img[i];
            }
            __syncwarp();
            // hand the buffer back as soon as the bulk store has READ it (the global writes may still be in
            // flight); this also keeps shared memory alive until the last store's reads are done
            if (lane == 0) {
                tma_store_wait_read<0>();
                mbar_arrive(&S.outempty[os]);
            }
            oi++;
        }
    } else {
        // ============================ tile warps: one lane == one 8x8 tile ============================
        const int sb = tid / g.w, stx = tid - sb * g.w;
        const uint32_t toff = (uint32_t)(8 * sb) * (uint32_t)g.W + 8u * (uint32_t)stx;   // my tile inside the image
        const int ncol = min(8, g.W - 8 * stx);
        unsigned oi = 0;
        for (unsigned it = 0;; it++) {
            const int s = it % kStgStages;
            mbar_wait(&S.full[s], (it / kStgStages) & 1);
            const int4 c0 = *reinterpret_cast<const int4 *>(&S.ctl[s].part);      // part, skip, f, nt
            if (c0.x < 0) break;
            if (c0.y & kCtlSkip) {
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.empty[s]);
                continue;
            }
            const uint4 c1 = *reinterpret_cast<const uint4 *>(&S.ctl[s].pres);    // pres, kres, mres, pixoff
            const int4 c2 = *reinterpret_cast<const int4 *>(&S.ctl[s].y0);        // y0, tx0, ntx, image address (low 32 bits)
            const int y0 = c2.x;
            const uint8_t *stage = stages + (size_t)s * kDecStageBytes;
            const bool valid = tid < c0.w;
            uint32_t px[16];
            dec_unpack_tile(stage, c1, S.ctl[s].wbase[warp], tid, lane, valid, (P.flags & kFlagInvertRows) != 0, px);
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.empty[s]);       // payload is in registers: free the stage early

            const int os = oi % kStgOut;
            if (oi >= kStgOut) mbar_wait(&S.outempty[os], ((oi / kStgOut) - 1) & 1);
            // the image's global address (its low bits), from the control block: the same value in every lane,
            // so the shape branches of the row stores below never diverge
            const uint32_t ag = (uint32_t)c2.w;
            const uint32_t img = smem_u32(outst) + (uint32_t)os * kStgOutBytes + (ag & 15u);
            const int rows_valid = valid ? min(8, g.H - 8 * (y0 + sb)) : 0;
            uint32_t rp = img + toff;
            if (rows_valid == 8 && ncol == 8) {
                sts_rows_static_any<WM>(ag, rp, (uint32_t)g.W, px);      // `ag & 7` is the same in every lane: a uniform switch
            } else {
                // last tile column of an odd-width frame / last band of an odd-height one: only the
                // valid columns and rows (dbde_util.cpp:281-289); a few lanes per partition.  Column by
                // column, so the common one-or-two-column edge costs one or two passes over the rows.
                // (lanes past the partition's tiles come here too, with rows_valid == 0: they must not loop)
                const int nc = rows_valid > 0 ? ncol : 0;
                for (int c = 0; c < nc; c++) {
                    const uint32_t sh = 8u * (uint32_t)(c & 3);
                    uint32_t q = rp + (uint32_t)c;
#pragma unroll
                    for (int r = 0; r < 8; r++) {
                        if (r < rows_valid) sts_u8(q, ((c & 4) ? px[2 * r + 1] : px[2 * r]) >> sh);
                        q += g.W;
                    }
                }
            }
            fence_proxy_async();                           // my generic-proxy writes, then the store warp's bulk read
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.outfull[os]);
            oi++;
        }
    }
}

size_t dec_smem_bytes(const PartGeom &g) {
    (void)g;
    return ((sizeof(DecSmem) + 127) & ~(size_t)127) + (size_t)kDecStages * kDecStageBytes;
}

cudaError_t launch_decode_scan(const DecParams &P, cudaStream_t stream) {
    if (P.nframes <= 0) return cudaSuccess;
    dbde_decode_scan_kernel<<<P.nframes, 256, 0, stream>>>(P);
    return cudaGetLastError();
}

static size_t stg_smem_bytes() {
    return ((sizeof(StgSmem) + 127) & ~(size_t)127) + (size_t)kStgStages * kDecStageBytes + kStgOut * (size_t)kStgOutBytes;
}

static bool odd_decode_staged() {
    const char *e = getenv("DBDE_B200_ODD_DECODE");       // read per launch: tests switch it inside one process
    return !(e && e[0] == 'd');
}

cudaError_t launch_decode(const DecParams &P, bool fast, int num_sms, cudaStream_t stream) {
    const size_t smem = dec_smem_bytes(P.g);
    if (fast && P.g.linear) return launch_persistent(dbde_decode_kernel<-2>, P, P.nparts, kDecThreads, smem, num_sms, stream);
    if (fast) return launch_persistent(dbde_decode_kernel<-1>, P, P.nparts, kDecThreads, smem, num_sms, stream);
    if (P.g.nseg == 1 && odd_decode_staged()) {
        const size_t ss = stg_smem_bytes();
        switch (P.g.W & 7) {
            case 0: return launch_persistent(dbde_decode_staged_kernel<0>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            case 1: return launch_persistent(dbde_decode_staged_kernel<1>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            case 2: return launch_persistent(dbde_decode_staged_kernel<2>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            case 3: return launch_persistent(dbde_decode_staged_kernel<3>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            case 4: return launch_persistent(dbde_decode_staged_kernel<4>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            case 5: return launch_persistent(dbde_decode_staged_kernel<5>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            case 6: return launch_persistent(dbde_decode_staged_kernel<6>, P, P.nparts, kStgThreads, ss, num_sms, stream);
            default: return launch_persistent(dbde_decode_staged_kernel<7>, P, P.nparts, kStgThreads, ss, num_sms, stream);
        }
    }
    switch (P.g.W & 7) {
        case 0: return launch_persistent(dbde_decode_kernel<0>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 1: return launch_persistent(dbde_decode_kernel<1>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 2: return launch_persistent(dbde_decode_kernel<2>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 3: return launch_persistent(dbde_decode_kernel<3>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 4: return launch_persistent(dbde_decode_kernel<4>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 5: return launch_persistent(dbde_decode_kernel<5>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 6: return launch_persistent(dbde_decode_kernel<6>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        default: return launch_persistent(dbde_decode_kernel<7>, P, P.nparts, kDecThreads, smem, num_sms, stream);
    }
}

cudaError_t launch_decode_binned(const DecParams &scan, int factor, uint8_t *out, int num_sms, cudaStream_t stream) {
    DecParams P = scan;
    P.frames = out;
    const size_t smem = dec_smem_bytes(P.g);
    switch (factor) {
        case 2: return launch_persistent(dbde_decode_binned_kernel<2>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 4: return launch_persistent(dbde_decode_binned_kernel<4>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        case 8: return launch_persistent(dbde_decode_binned_kernel<8>, P, P.nparts, kDecThreads, smem, num_sms, stream);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace dbde
