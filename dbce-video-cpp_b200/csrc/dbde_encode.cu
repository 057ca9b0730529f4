// DBDE B200 encoder: raw U8 frames in HBM -> DBDE frame records in HBM, byte-identical to what
// dbde_pack_frame (dbde_util.cpp:190-196) writes frame after frame.
//
// One persistent kernel, one pass over the pixels:
//   warp 8  (producer) : claims partitions from an atomic ticket and bulk-TMAs their pixel rows
//                        into a ring of shared-memory stages (mbarrier full/empty pipeline)
//   warps 0-7 (tiles)  : one lane per 8x8 tile -- min, depth = bits(max-min), bit packing.  A tile
//                        warp never meets the other tile warps: it hands the pixel stage back as
//                        soon as its pixels are in registers and stages its payload words in its
//                        OWN 2 KiB region of a double-buffered output ring (immediate-offset 8-byte
//                        stores), then copies its run out with coalesced stores one partition later
//   warp 9  (scan)     : sums the warps' depth totals, publishes the partition aggregate, resolves
//                        its exclusive prefix with a single-pass decoupled look-back, and hands the
//                        tile warps {frame, exclusive prefix, each warp's offset inside the
//                        partition}; writes the frame's fixed fields (header, lengths, n64)
// Word offsets are per-frame quantities (the reference zeroes n64 per frame, dbde_util.cpp:146),
// so there is one look-back chain per frame, and tickets are INTERLEAVED across the frames of the
// batch (ticket t -> frame t mod N, partition t div N): the partitions in flight at any moment
// belong to different frames, a partition's predecessor was finished a whole generation earlier,
// and the look-back is one descriptor read instead of a convoy of L2 round trips.  Frame f's
// record is written to its own slot (out + f * slot_stride); sizes go to frame_sizes[].
//
// The kernel is issue/latency-bound before it is HBM-bound (ncu: ~72 % issue-slot utilisation with
// 7.5 warps per scheduler), so the tile warps' loop is written for instruction count and for
// independence: no staging swizzle, one 16-byte control read per partition, no CTA-wide barrier
// (the in-place staging of the first versions needed one per partition: 12 % of the stall samples).
#include "dbde_device.cuh"
#include "dbde_kernels.h"

#include <mutex>
#include <vector>

namespace dbde {

// A warp with this many different non-zero depths packs with the depth-agnostic row packer.  Measured
// (mix-2048): never 4.11 TB/s, 4 -> 5.06, 3 -> 5.05; micro-2048 unchanged within noise.
constexpr int kEncVarMinDepths = 4;

// Copy-out with 16-byte stores (the north star's "128-bit vectorised stores") is implemented and measured, and
// loses to 8-byte stores on everything but all-depth-8 noise (algorithmic TB/s, 8-byte vs 16-byte: micro-2048
// 6.10 vs 6.06, low-4096 5.29 vs 5.18, mix-1001x1003 4.67 vs 4.65, noise-2048 6.24 vs 6.29): a warp's run starts
// on an odd word half the time, so the vector path needs a leading and a trailing single-word store and two
// 8-byte shared loads per vector, and the run is only ~100 words long.  -DDBDE_ENC_COPY16=1 builds it.
#ifndef DBDE_ENC_COPY16
#define DBDE_ENC_COPY16 0
#endif
constexpr int kEncRing = 4;        // bookkeeping slots (aggregates, bases): a tile warp is <= 2 partitions ahead of the scan warp
constexpr int kEncThreads = kTilesPerPart + 64;

struct alignas(16) EncCtl {     // per-stage control block, written by the producer warp
    int part;                   // partition id, -1 = no more work
    int f;                      // frame within the batch
    int tfirst;                 // first tile's row-major index in the frame
    int nt;                     // tiles in this partition
    int q;                      // partition within the frame
    int y0, tx0, pad;           // first band / first tile column (generic path only)
};
struct alignas(16) EncBase {    // per-stage, written by the scan warp
    uint8_t *frame;             // where this frame's record starts
    uint32_t excl;              // U64 words of this frame before this partition
    uint32_t nwords;            // U64 words of this partition
};

struct EncSmem {
    uint64_t full[kEncRing], empty[kEncRing], aggbar[kEncRing], basebar[kEncRing];
    EncCtl ctl[kEncRing];
    EncBase base[kEncRing];
    uint32_t warptot[kEncRing][kConsumerWarps];   // depth sum of each tile warp
    uint32_t wbase[kEncRing][kConsumerWarps];       // its word offset inside the partition (scan warp)
};

// depth 8: the words are the (p - min) rows themselves (dbde_util.cpp:57-64).  Equal-depth
// neighbours sit 64 bytes apart -- an 8-way bank conflict for 8-byte stores -- so the 64 bytes go
// out as 16-byte stores around the 16-byte boundary nearest to the tile's first word (4-way).
__device__ __forceinline__ void enc_store_depth8(const uint32_t (&w)[16], uint8_t *wb, uint32_t off) {
    if (off & 1u) {
        *reinterpret_cast<uint2 *>(wb) = make_uint2(w[0], w[1]);
#pragma unroll
        for (int j = 0; j < 3; j++)
            *reinterpret_cast<uint4 *>(wb + 8 + 16 * j) = make_uint4(w[4 * j + 2], w[4 * j + 3], w[4 * j + 4], w[4 * j + 5]);
        *reinterpret_cast<uint2 *>(wb + 56) = make_uint2(w[14], w[15]);
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++)
            *reinterpret_cast<uint4 *>(wb + 16 * j) = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
    }
}

// Shared memory per CTA: 2 pixel stages x 16 KiB + 2 x 8 x 2 KiB of output ring = 66 KiB -> 3 CTAs/SM.
// (The in-place design held 4 x 16 KiB; there 3 stages cost 7 % and 5-6 stages at 2 CTAs/SM 19 %.)
constexpr int kEncStages = 2;                                  // pixel stages (handed back as soon as the pixels are in registers)
constexpr int kEncWarpBytes = 64 * 32 + 16;                     // a warp's private staging region: worst case 32 tiles x 64 bytes
constexpr int kWidePitch = 8 * kTilesPerPart;
// FAST : 16-byte aligned rows, no partial tiles (W % 16 == 0, H % 8 == 0).
// WIDE : FAST and w % 256 == 0 (2048-, 4096-pixel-wide frames): every partition is one full 256-tile
//        band segment, so the smem pitch is the constant 2048 (immediate-offset row loads) and no
//        lane is ever idle.
// CONTIG: every odd size.  Full-width partitions (W <= 2048): the partition's pixels are one contiguous byte
//        range of the frame, staged with ONE bulk copy of its 16-byte hull at row pitch W.  Band segments of
//        wider frames: eight per-row hull copies at a pitch that is W modulo 16.  Either way a lane's row r is
//        `first row + r * pitch` at the alignment it has in global memory, read as aligned words + funnel shift.
// CONTIG row loads with every shape known at compile time: WM = W & 7, A0 = alignment of the tile's row 0
// (the same for every lane: tiles and bands are multiples of 8 bytes apart).  A row at byte alignment a is
// one 8-byte load (a == 0), two 4-byte loads (a == 4), or an 8-byte and a 4-byte load of the three aligned
// words it touches plus two funnel shifts by a constant.
template <int WM, int A0>
__device__ __forceinline__ void load_rows_contig(uint32_t addr, uint32_t W, uint32_t (&px)[16]) {
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int a = (A0 + r * WM) & 7;                       // compile-time after unrolling
        const uint32_t b = addr - (uint32_t)a;                 // 8-byte aligned
        uint32_t w0, w1, w2;
        if (a == 0) {
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(px[2 * r]), "=r"(px[2 * r + 1]) : "r"(b));
        } else if (a == 4) {
            asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(px[2 * r]) : "r"(b));
            asm volatile("ld.shared.u32 %0, [%1+8];" : "=r"(px[2 * r + 1]) : "r"(b));
        } else if (a < 4) {
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(w0), "=r"(w1) : "r"(b));
            asm volatile("ld.shared.u32 %0, [%1+8];" : "=r"(w2) : "r"(b));
            px[2 * r] = __funnelshift_r(w0, w1, 8 * a);
            px[2 * r + 1] = __funnelshift_r(w1, w2, 8 * a);
        } else {
            asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(w0) : "r"(b));
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+8];" : "=r"(w1), "=r"(w2) : "r"(b));
            px[2 * r] = __funnelshift_r(w0, w1, 8 * (a - 4));
            px[2 * r + 1] = __funnelshift_r(w1, w2, 8 * (a - 4));
        }
        addr += W;
    }
}
template <int WM>
__device__ __forceinline__ void load_rows_contig_any(uint32_t addr, uint32_t W, uint32_t (&px)[16]) {
    switch (addr & 7u) {
        case 0: load_rows_contig<WM, 0>(addr, W, px); break;
        case 1: load_rows_contig<WM, 1>(addr, W, px); break;
        case 2: load_rows_contig<WM, 2>(addr, W, px); break;
        case 3: load_rows_contig<WM, 3>(addr, W, px); break;
        case 4: load_rows_contig<WM, 4>(addr, W, px); break;
        case 5: load_rows_contig<WM, 5>(addr, W, px); break;
        case 6: load_rows_contig<WM, 6>(addr, W, px); break;
        default: load_rows_contig<WM, 7>(addr, W, px); break;
    }
}

// WM: W & 7 for the CONTIG kernel (compile-time row shapes), 0 otherwise.
// LIN: FAST with linear partitions (make_geom): staged like WIDE -- tile t at byte 8t of every row, pitch 2048 --
//      but the frame's last partition may be short.
template <bool FAST, bool WIDE, bool CONTIG, int WM = 0, bool LIN = false>
__global__ void __launch_bounds__(kEncThreads, 3) dbde_encode_kernel(const EncParams P) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    EncSmem &S = *reinterpret_cast<EncSmem *>(smem_raw);
    uint8_t *stages = smem_raw + ((sizeof(EncSmem) + 127) & ~127);
    const PartGeom &g = P.g;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // warp-private output ring: out[2][8 warps][kEncWarpBytes], after the kEncStages input stages
    uint8_t *outring = stages + (size_t)kEncStages * g.stage_bytes;

    if (tid == 0) {
        for (int s = 0; s < kEncRing; s++) {
            mbar_init(&S.full[s], 1);
            mbar_init(&S.empty[s], kConsumerWarps + 1);       // the eight tile warps and the scan warp
            mbar_init(&S.aggbar[s], kConsumerWarps);
            mbar_init(&S.basebar[s], 1);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        // ============================ producer warp ============================
        const size_t fbytes = (size_t)g.W * g.H;
        // The ticket for the NEXT partition is claimed one iteration early, so the atomic's L2 round
        // trip overlaps the wait for a free stage instead of delaying the refill (with two stages the
        // refill latency is the budget).  A claimed ticket is always processed next: progress holds.
        unsigned t_next = 0;
        if (lane == 0) t_next = atomicAdd(P.ticket, 1u);
        for (unsigned it = 0;; it++) {
            const int s = it % kEncStages;
            const uint32_t ph = (it / kEncStages) & 1;
            unsigned t = __shfl_sync(0xffffffffu, t_next, 0);
            if (lane == 0 && t < P.nparts) t_next = atomicAdd(P.ticket, 1u);
            mbar_wait_sleepy(&S.empty[s], ph ^ 1);
            // frame-interleaved order: all frames' partition 0, then all frames' partition 1, ...
            const unsigned tq = t / (unsigned)P.nframes;
            const unsigned p = (t - tq * (unsigned)P.nframes) * (unsigned)g.ppf + tq;
            if (t >= P.nparts) {
                if (lane == 0) {
                    S.ctl[s].part = -1;
                    mbar_arrive(&S.full[s]);
                }
                break;
            }
            const PartInfo pi = part_info(g, p);
            const uint8_t *fptr = P.frames + (size_t)pi.f * fbytes;
            uint8_t *stage = stages + (size_t)s * g.stage_bytes;
            const int nrows = pi.nbands * 8;
            if (FAST && g.pitch == g.W) {
                // full-width partitions of tightly packed rows: the bands are ONE contiguous run in
                // memory and in the stage -> a single bulk copy (2048-pixel-wide frames: 16 KiB)
                if (lane == 0) {
                    const uint32_t bytes = (uint32_t)nrows * (uint32_t)g.W;
                    *reinterpret_cast<int4 *>(&S.ctl[s].part) = make_int4((int)p, pi.f, pi.tfirst, pi.nt);
                    *reinterpret_cast<int4 *>(&S.ctl[s].q) = make_int4(pi.q, pi.y0, pi.tx0, 0);
                    mbar_arrive_expect_tx(&S.full[s], bytes);
                    tma_load_1d(stage, fptr + (size_t)(8 * pi.y0) * g.W, bytes, &S.full[s]);
                }
                continue;
            }
            if (CONTIG && g.nseg == 1) {
                if (lane == 0) {
                    const uint8_t *g0 = fptr + (size_t)(8 * pi.y0) * g.W;
                    const uint32_t n = (uint32_t)min(nrows, g.H - 8 * pi.y0) * (uint32_t)g.W;
                    const uintptr_t a0 = (uintptr_t)g0 & ~(uintptr_t)15;
                    const uintptr_t a1 = ((uintptr_t)g0 + n + 15) & ~(uintptr_t)15;
                    *reinterpret_cast<int4 *>(&S.ctl[s].part) = make_int4((int)p, pi.f, pi.tfirst, pi.nt);
                    *reinterpret_cast<int4 *>(&S.ctl[s].q) = make_int4(pi.q, pi.y0, pi.tx0, (int)((uintptr_t)g0 - a0));
                    mbar_arrive_expect_tx(&S.full[s], (uint32_t)(a1 - a0));
                    tma_load_1d(stage, (const void *)a0, (uint32_t)(a1 - a0), &S.full[s]);
                }
                continue;
            }
            if (CONTIG) {
                // a band segment of an odd frame wider than 2048: its rows are not contiguous in the frame, so each
                // row's 16-byte hull is copied on its own -- to a row pitch that is W modulo 16 (launch_encode), so that
                // every row lands at its global alignment AND at a constant stride: the tile warps read it exactly
                // like a contiguous partition (compile-time row shapes), only the stride differs.
                const int rowbytes = min(8 * pi.ntx, g.W - 8 * pi.tx0);
                const uint8_t *g0 = fptr + (size_t)(8 * pi.y0) * g.W + 8 * pi.tx0;
                const uint32_t off0 = (uint32_t)((uintptr_t)g0 & 15);
                const uint8_t *src = nullptr;
                uint32_t len = 0, dst = 0;
                if (lane < 8 && 8 * pi.y0 + lane < g.H) {
                    const uint8_t *gr = g0 + (size_t)lane * g.W;
                    const uintptr_t a0 = (uintptr_t)gr & ~(uintptr_t)15;
                    const uintptr_t a1 = ((uintptr_t)gr + rowbytes + 15) & ~(uintptr_t)15;
                    src = (const uint8_t *)a0;
                    len = (uint32_t)(a1 - a0);
                    dst = off0 + (uint32_t)lane * (uint32_t)g.pitch - (uint32_t)((uintptr_t)gr - a0);     // a multiple of 16
                }
                const uint32_t total = __reduce_add_sync(0xffffffffu, len);
                if (lane == 0) {
                    *reinterpret_cast<int4 *>(&S.ctl[s].part) = make_int4((int)p, pi.f, pi.tfirst, pi.nt);
                    *reinterpret_cast<int4 *>(&S.ctl[s].q) = make_int4(pi.q, pi.y0, pi.tx0, (int)off0);
                    mbar_arrive_expect_tx(&S.full[s], total);
                }
                __syncwarp();
                if (len) tma_load_1d(stage + dst, src, len, &S.full[s]);
                continue;
            }
            if (LIN) {
                // linear partition: tiles [tfirst, tfirst + nt) of the row-major tile order = the tail of one band,
                // whole bands, the head of another.  Each piece is 8 row copies of 8*ntx bytes, and the pieces sit
                // side by side in the stage's 8 rows (pitch 2048), so tile t of the partition is at byte 8t of every
                // row whatever band it came from.  Lane group i & 3 issues piece i (lane & 7 = the row).
                if (lane == 0) {
                    *reinterpret_cast<int4 *>(&S.ctl[s].part) = make_int4((int)p, pi.f, pi.tfirst, pi.nt);
                    *reinterpret_cast<int4 *>(&S.ctl[s].q) = make_int4(pi.q, pi.y0, pi.tx0, 0);
                    mbar_arrive_expect_tx(&S.full[s], 64u * (uint32_t)pi.nt);
                }
                __syncwarp();
                int band = pi.y0, tx = pi.tx0, done = 0;
                for (int i = 0; done < pi.nt; i++) {
                    const int ntx = min(g.w - tx, pi.nt - done);
                    if ((lane >> 3) == (i & 3)) {
                        const int r = lane & 7;
                        tma_load_1d(stage + (size_t)r * g.pitch + 8 * done, fptr + (size_t)(8 * band + r) * g.W + 8 * tx,
                                    8u * (uint32_t)ntx, &S.full[s]);
                    }
                    done += ntx;
                    tx = 0;
                    band++;
                }
                continue;
            }
            const int rowbytes = min(8 * pi.ntx, g.W - 8 * pi.tx0);
            // each lane owns rows lane, lane+32
            uint32_t mybytes = 0;
            const uint8_t *src[2];
            uint32_t len[2];
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int row = lane + 32 * j;
                len[j] = 0;
                src[j] = nullptr;
                if (row < nrows) {
                    const int y = 8 * pi.y0 + row;
                    if (y < g.H) {
                        const uint8_t *a = fptr + (size_t)y * g.W + 8 * pi.tx0;
                        const uintptr_t a0 = (uintptr_t)a & ~(uintptr_t)15;
                        const uintptr_t a1 = ((uintptr_t)a + rowbytes + 15) & ~(uintptr_t)15;
                        src[j] = (const uint8_t *)a0;
                        len[j] = (uint32_t)(a1 - a0);
                    }
                }
                mybytes += len[j];
            }
            const uint32_t total = __reduce_add_sync(0xffffffffu, mybytes);
            if (lane == 0) {
                *reinterpret_cast<int4 *>(&S.ctl[s].part) = make_int4((int)p, pi.f, pi.tfirst, pi.nt);
                *reinterpret_cast<int4 *>(&S.ctl[s].q) = make_int4(pi.q, pi.y0, pi.tx0, 0);
                mbar_arrive_expect_tx(&S.full[s], total);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 2; j++)
                if (len[j]) tma_load_1d(stage + (size_t)(lane + 32 * j) * g.pitch, src[j], len[j], &S.full[s]);
        }
    } else if (warp == kConsumerWarps + 1) {
        // ============================ scan warp ============================
        for (unsigned it = 0;; it++) {
            const int s = it % kEncStages, ss = it % kEncRing;
            mbar_wait_sleepy(&S.full[s], (it / kEncStages) & 1);
            const int4 c0 = *reinterpret_cast<const int4 *>(&S.ctl[s].part);
            const int q = S.ctl[s].q;
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.empty[s]);          // the control block has been read
            if (c0.x < 0) break;
            const unsigned p = (unsigned)c0.x;
            const int f = c0.y;
            // The exclusive prefix only needs the PREDECESSORS' descriptors: take it while the tile warps
            // are still computing this partition's depths, so that nothing but a shared-memory hand-off
            // stands between their last arrival and the base they wait for at copy-out time.
            uint64_t excl = q == 0 ? 0ull : lookback_exclusive<false>(P.desc, p, p - (unsigned)q, lane);
            mbar_wait_sleepy(&S.aggbar[ss], (it / kEncRing) & 1);
            const uint32_t wt = lane < kConsumerWarps ? S.warptot[ss][lane] : 0u;
            const uint32_t winc = warp_inclusive_scan(wt, lane);
            const uint64_t agg = __shfl_sync(0xffffffffu, winc, kConsumerWarps - 1);
            if (lane < kConsumerWarps) S.wbase[ss][lane] = winc - wt;      // each tile warp's offset inside the partition
            if (excl == kLookbackNotReady) {
                // a predecessor is still in flight (few frames in the batch): the classic protocol
                if (lane == 0) st_relaxed_u64(P.desc + p, desc_make(kDescAggregate, agg));
                excl = lookback_exclusive<true>(P.desc, p, p - (unsigned)q, lane);
            }
            if (lane == 0) st_relaxed_u64(P.desc + p, desc_make(kDescPrefix, excl + agg));
            const size_t fixed = rec_fixed(g.wh, 1);        // frame header + lengths + planes
            uint8_t *frame = P.out + (size_t)f * P.slot_stride;
            __syncwarp();
            if (lane == 0) {
                S.base[ss].frame = frame;
                *reinterpret_cast<uint2 *>(&S.base[ss].excl) = make_uint2((uint32_t)excl, (uint32_t)agg);
                mbar_arrive(&S.basebar[ss]);
            }
            if (q == g.ppf - 1) {
                // last partition of the frame: the fixed fields, byte for byte write_fixed_fields(frame, lane, index,
                // g.wh, 1, n64, ...).  Kept as its own copy: with the shared writer ptxas schedules this kernel
                // differently, and the micro-2048 encode measured 0.5 % slower (B200, 1000 W power limit)
                const uint32_t n64 = (uint32_t)(excl + agg);
                const uint64_t index = P.first_index + (uint64_t)f;
                uint32_t b;      // lane i writes one byte of {I32 2 | U64 index | F64 0.0 | I32 wh} {I32 wh} {I32 n64}
                uint8_t *dst;
                if (lane < 4) { b = (2u >> (8 * lane)) & 0xff; dst = frame + lane; }
                else if (lane < 12) { b = (uint32_t)(index >> (8 * (lane - 4))) & 0xff; dst = frame + lane; }
                else if (lane < 20) { b = 0; dst = frame + lane; }
                else if (lane < 24) { b = ((uint32_t)g.wh >> (8 * (lane - 20))) & 0xff; dst = frame + lane; }
                else if (lane < 28) { b = ((uint32_t)g.wh >> (8 * (lane - 24))) & 0xff; dst = frame + rec_min_count(g.wh) + (lane - 24); }
                else { b = (n64 >> (8 * (lane - 28))) & 0xff; dst = frame + rec_n64(g.wh, 1) + (lane - 28); }
                *dst = (uint8_t)b;
                if (lane == 0) {
                    P.frame_offsets[f] = (uint64_t)f * P.slot_stride;
                    P.frame_sizes[f] = fixed + 8ull * n64;
                }
            }
        }
    } else {
        // ============================ tile warps: one lane == one 8x8 tile ============================
        // The copy-out of partition i is deferred until partition i+1 has been packed, so the
        // scan warp's look-back for i overlaps the arithmetic of i+1.
        int sb = 0, stx = tid;                  // slot -> (band within partition, tile column)
        if (g.nseg == 1 && g.G > 1) {
            sb = tid / g.w;
            stx = tid - sb * g.w;
        }
        const uint32_t toff = (uint32_t)(sb * 8) * (uint32_t)g.pitch + (uint32_t)stx * 8u;   // my tile inside a stage
        const size_t fixed = rec_fixed(g.wh, 1);
        // deferred partition (iteration it-1): its depth/min/word count stay in registers until its
        // addresses are known.  d_km = depth | min << 8 | valid << 16.
        uint32_t d_km = 0, d_wtot = 0;
        int d_tfirst = 0;

        auto flush_deferred = [&](unsigned dit) {
            const int ds = dit % kEncRing;
            const uint8_t *src = outring + ((size_t)(dit & 1) * kConsumerWarps + warp) * kEncWarpBytes;
            mbar_wait(&S.basebar[ds], (dit / kEncRing) & 1);
            const uint4 b = *reinterpret_cast<const uint4 *>(&S.base[ds]);
            uint8_t *frame = reinterpret_cast<uint8_t *>(((uint64_t)b.y << 32) | b.x);
            // ---- depth and minimum planes (dbde_util.cpp:156-157)
            if (WIDE || (d_km >> 16)) {
                uint8_t *pl = frame + d_tfirst + tid;
                pl[kRecDepth] = (uint8_t)d_km;
                pl[rec_min(g.wh)] = (uint8_t)(d_km >> 8);
            }
            // ---- this warp's words, by this warp: one coalesced run per warp
            uint8_t *dst = frame + fixed + 8 * ((size_t)b.z + S.wbase[ds][warp]);
            const uint32_t n = d_wtot;
#if DBDE_ENC_COPY16
            if (((uintptr_t)dst & 7) == 0) {
                // 16-byte stores: one leading word when the run starts on an odd word, then pairs of words
                // (the warp's staging region is 16-byte aligned, so an even start also loads 16 bytes at a time)
                const uint32_t head = n ? ((uint32_t)(uintptr_t)dst >> 3) & 1u : 0u;
                const uint32_t npair = (n - head) >> 1;
                if (head) {
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        if (32u * j >= npair) break;
                        const uint32_t i = lane + 32u * j;
                        if (i < npair) {
                            const uint2 lo = *reinterpret_cast<const uint2 *>(src + 8 + 16 * i);
                            const uint2 hi = *reinterpret_cast<const uint2 *>(src + 16 + 16 * i);
                            st_stream_v4u32(dst + 8 + 16 * i, make_uint4(lo.x, lo.y, hi.x, hi.y));
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        if (32u * j >= npair) break;
                        const uint32_t i = lane + 32u * j;
                        if (i < npair) st_stream_v4u32(dst + 16 * i, *reinterpret_cast<const uint4 *>(src + 16 * i));
                    }
                }
                // the single words at the ends -- the leading one of a run that starts on an odd word (lane 0) and
                // the last one of a run with an odd number of words after it (lane 31) -- in ONE predicated store
                const bool tail = ((n - head) & 1u) != 0u;
                if ((lane == 0 && head) || (lane == 31 && tail)) {
                    const uint32_t w = lane == 0 ? 0u : n - 1u;
                    st_stream_u64(dst + 8 * w, *reinterpret_cast<const uint64_t *>(src + 8 * w));
                }
#else
            if (((uintptr_t)dst & 7) == 0) {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if (32u * j >= n) break;
                    if (lane + 32u * j < n)
                        st_stream_u64(dst + 8 * (lane + 32 * j), *reinterpret_cast<const uint64_t *>(src + 8 * (lane + 32 * j)));
                }
#endif
            } else {
                for (uint32_t i = lane; i < 8 * n; i += 32) dst[i] = src[i];
            }
        };

        unsigned it = 0;
        for (;; it++) {
            const int s = it % kEncStages, ss = it % kEncRing;
            mbar_wait(&S.full[s], (it / kEncStages) & 1);
            const int4 c0 = *reinterpret_cast<const int4 *>(&S.ctl[s].part);   // part, f, tfirst, nt
            if (c0.x < 0) break;
            uint8_t *stage = stages + (size_t)s * g.stage_bytes;
            const bool valid = WIDE || tid < c0.w;

            // ---- stage (1)->registers: 8 rows x 8 bytes
            uint32_t px[16];
            if (WIDE || LIN) {
                const uint8_t *base = stage + 8 * tid;
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    const uint2 v = *reinterpret_cast<const uint2 *>(base + r * kWidePitch);
                    px[2 * r] = v.x;
                    px[2 * r + 1] = v.y;
                }
            } else if (FAST) {
                const uint8_t *base = stage + (valid ? toff : 0u);     // idle lanes read (and discard) tile 0
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    const uint2 v = *reinterpret_cast<const uint2 *>(base);
                    base += g.pitch;
                    px[2 * r] = v.x;
                    px[2 * r + 1] = v.y;
                }
            } else if (CONTIG) {
                const int4 c1 = *reinterpret_cast<const int4 *>(&S.ctl[s].q);      // q, y0, tx0, first pixel's offset in the hull
                const int rows_valid = min(8, g.H - 8 * (c1.y + sb));
                const int ncol = min(8, g.W - 8 * (c1.z + stx));
                uint32_t addr = smem_u32(stage) + (uint32_t)c1.w + (valid ? toff : 0u);      // idle lanes read (and discard) tile 0
                auto load8 = [&](uint32_t a) {
                    uint32_t w0, w1, w2;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(a & ~3u));
                    asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(w1) : "r"(a & ~3u));
                    asm volatile("ld.shared.u32 %0, [%1+8];" : "=r"(w2) : "r"(a & ~3u));
                    return make_uint2(__funnelshift_r(w0, w1, a << 3), __funnelshift_r(w1, w2, a << 3));
                };
                // `addr & 7` is the same in every lane (tiles and bands are multiples of 8 bytes apart), so the
                // switch inside is a uniform branch.  A tile of the last column (ncol < 8) loads its rows the same
                // way -- the bytes past the row end are the next row's, or stage slack -- and then repeats its
                // last valid pixel over them (dbde_util.cpp:119-127): one byte-broadcast and two selects per row.
                if (!valid || rows_valid == 8) {
                    load_rows_contig_any<WM>(addr, (uint32_t)g.pitch, px);
                    if (ncol < 8) {
                        const uint32_t bsel = 0x1111u * (uint32_t)(ncol - 1);                       // PRMT selector: byte ncol-1 of {lo, hi} four times
                        const uint32_t klo = ncol >= 4 ? 0xffffffffu : (1u << (8 * ncol)) - 1u;     // bytes of the low / high word that are real pixels
                        const uint32_t khi = ncol <= 4 ? 0u : (1u << (8 * (ncol - 4))) - 1u;
#pragma unroll
                        for (int r = 0; r < 8; r++) {
                            const uint32_t fill = __byte_perm(px[2 * r], px[2 * r + 1], bsel);
                            px[2 * r] = (px[2 * r] & klo) | (fill & ~klo);
                            px[2 * r + 1] = (px[2 * r + 1] & khi) | (fill & ~khi);
                        }
                    }
                } else {
                    // the frame's last band when H % 8 != 0: rows past H repeat the last valid row (dbde_util.cpp:111-117)
#pragma unroll
                    for (int r = 0; r < 8; r++) {
                        uint2 v = load8(addr + (uint32_t)(min(r, rows_valid - 1) * g.pitch));
                        if (ncol < 8) {
                            uint64_t x = ((uint64_t)v.y << 32) | v.x;
                            const uint64_t last = (x >> (8 * (ncol - 1))) & 0xffull;
                            const uint64_t keep = (1ull << (8 * ncol)) - 1ull;
                            x = (x & keep) | ((last * 0x0101010101010101ull) & ~keep);
                            v = make_uint2((uint32_t)x, (uint32_t)(x >> 32));
                        }
                        px[2 * r] = v.x;
                        px[2 * r + 1] = v.y;
                    }
                }
            }
            if (P.flags & kFlagInvertRows) reverse_rows(px);      // after the clamp padding, as ENDIAN() at dbde_util.cpp:24-27
            // the pixels are in registers: hand the stage back to the producer right away
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.empty[s]);
            // ---- stage (2): min, depth
            uint32_t mn = tile_min(px);
            int k = tile_subtract_depth(px, mn);
            if (!valid) { k = 0; mn = 0; }
            // ---- stage (3a): depth sums -> scan warp
            const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
            if (lane == 31) {
                S.warptot[ss][warp] = incl;
                mbar_arrive(&S.aggbar[ss]);
            }
            // my tile's word offset inside this WARP's private staging region: no other warp is involved
            const uint32_t off = incl - (uint32_t)k;
            uint8_t *stage_out = outring + ((size_t)(it & 1) * kConsumerWarps + warp) * kEncWarpBytes;
            // ---- stage (4): pack (p - min) into k U64 words, staged linearly in the dead pixel bytes
            // a warp holding many different depths would run concat_fields<K> once per depth: from
            // kEncVarMinDepths distinct non-zero depths on, the depth-agnostic row packer is shorter
            const uint32_t kinds = __reduce_or_sync(0xffffffffu, (1u << k) >> 1);      // bit d-1 set: some tile has depth d
            const bool many_depths = __popc(kinds) >= kEncVarMinDepths;
            if ((kinds & ~3u) == 0u) {
                // low-entropy warp (every depth <= 2): one dot-product squeeze for all lanes, no specialisation
                if (kinds) pack_low_depths(px, k, stage_out + 8 * off);
            } else if (k > 0) {
                const uint32_t c1 = (1u << k) - 256u, c2 = (1u << (2 * k)) - 65536u;
                uint32_t q[16];
#pragma unroll
                for (int i = 0; i < 16; i++) q[i] = squeeze4(px[i], c1, c2);
                uint2 *wp = reinterpret_cast<uint2 *>(stage_out + 8 * off);
                auto store = [&](int n, uint32_t lo, uint32_t hi) { wp[n] = make_uint2(lo, hi); };
                if (many_depths) pack_rows_var(q, k, stage_out + 8 * off);
                else switch (k) {
                    case 1: concat_fields<1>(q, store); break;
                    case 2: concat_fields<2>(q, store); break;
                    case 3: concat_fields<3>(q, store); break;
                    case 4: concat_fields<4>(q, store); break;
                    case 5: concat_fields<5>(q, store); break;
                    case 6: concat_fields<6>(q, store); break;
                    case 7: concat_fields<7>(q, store); break;
                    default: enc_store_depth8(q, stage_out + 8 * off, off); break;   // squeeze4 is the identity at depth 8
                }
            }
            __syncwarp();               // the warp's words are staged before any lane copies them out
            if (it > 0) flush_deferred(it - 1);
            d_km = (uint32_t)k | (mn << 8) | ((uint32_t)valid << 16);
            d_wtot = __shfl_sync(0xffffffffu, incl, 31);
            d_tfirst = c0.z;
        }
        if (it > 0) flush_deferred(it - 1);
    }
}

// ------------------------------------------------------------------ crop encoder
// One CTA per record (frame f, crop r) of a persistent grid, one lane per tile of the crop.  The CTA walks the crop's
// tiles in raster order, 256 at a time; a record's word offsets depend on its own tiles only, so a CTA-wide scan per
// chunk plus a running carry replaces the frame encoder's look-back and tickets, and no scratch is zeroed.

// The 8 rows of crop tile (tx, ty): pixel (x, y) of the crop image is frame[y0 + y][x0 + x] inside the frame and the
// pad byte outside it; the reference's clamp padding at the crop's own partial last column / row repeats the crop
// image's last valid pixel (dbde_util.cpp:105-135), which may be pad.  A tile inside the frame and the crop loads each
// row as the one or two aligned 8-byte words it touches (32 lanes of a tile row read 256 consecutive bytes); a tile
// at an edge reads each in-frame pixel it needs as a byte and nothing else.
__device__ __forceinline__ void load_crop_tile(const EncCropParams &P, const uint8_t *fr, long long x0, long long y0, int tx, int ty,
                                               uint32_t (&px)[16]) {
    const long long xs = x0 + 8 * tx, ys = y0 + 8 * ty;
    const bool inner = 8 * tx + 8 <= P.crop_w && 8 * ty + 8 <= P.crop_h && xs >= 0 && xs + 8 <= P.W && ys >= 0 && ys + 8 <= P.H;
    if (inner) {
        const uint8_t *p = fr + (size_t)ys * (size_t)P.W + (size_t)xs;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint64_t *a = reinterpret_cast<const uint64_t *>((uintptr_t)p & ~(uintptr_t)7);
            const uint32_t sh = ((uint32_t)(uintptr_t)p & 7u) * 8u;
            uint64_t v = __ldg(a);
            if (sh) v = (v >> sh) | (__ldg(a + 1) << (64u - sh));
            px[2 * r] = (uint32_t)v;
            px[2 * r + 1] = (uint32_t)(v >> 32);
            p += P.W;
        }
        return;
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const long long y = y0 + min(8 * ty + r, P.crop_h - 1);
        uint64_t v = P.pad8;
        if (y >= 0 && y < P.H) {
            const uint8_t *row = fr + (size_t)y * (size_t)P.W;
            v = 0;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const long long x = x0 + min(8 * tx + i, P.crop_w - 1);
                const uint64_t b = x >= 0 && x < P.W ? (uint64_t)__ldg(row + x) : (P.pad8 & 0xffu);
                v |= b << (8 * i);
            }
        }
        px[2 * r] = (uint32_t)v;
        px[2 * r + 1] = (uint32_t)(v >> 32);
    }
}

__global__ void __launch_bounds__(kTilesPerPart) dbde_encode_crops_kernel(const EncCropParams P) {
    __shared__ __align__(16) uint8_t s_words[kConsumerWarps][kEncWarpBytes];   // each warp's packed words of one chunk
    __shared__ uint32_t s_wtot[2][kConsumerWarps];                            // each warp's word count, by chunk parity
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint8_t *stage_out = s_words[warp];
    const size_t fbytes = (size_t)P.W * (size_t)P.H;
    const size_t fixed = rec_fixed(P.wh, 1);
    unsigned cc = 0;                                   // chunks done by this CTA: selects the s_wtot half
    for (int j = blockIdx.x; j < P.nrec; j += gridDim.x) {
        const int f = j / P.ncrops, r = j - f * P.ncrops;
        const int32_t *cp = P.corners + 2 * ((size_t)f * (size_t)P.corner_stride + (size_t)r);
        const long long x0 = __ldg(cp), y0 = __ldg(cp + 1);
        const uint8_t *fr = P.frames + (size_t)f * fbytes;
        uint8_t *rec = P.out + (size_t)j * P.slot_stride;
        uint32_t carry = 0;                            // U64 words of the record's earlier chunks
        for (int t0 = 0; t0 < P.wh; t0 += kTilesPerPart, cc++) {
            const int t = t0 + tid;
            const bool valid = t < P.wh;
            uint32_t px[16];
            if (valid) {
                const int ty = t / P.w;
                load_crop_tile(P, fr, x0, y0, t - ty * P.w, ty, px);
            } else {
#pragma unroll
                for (int i = 0; i < 16; i++) px[i] = 0;
            }
            if (P.flags & kFlagInvertRows) reverse_rows(px);      // after the clamp padding, as ENDIAN() at dbde_util.cpp:24-27
            uint32_t mn = tile_min(px);
            int k = tile_subtract_depth(px, mn);
            if (!valid) { k = 0; mn = 0; }
            const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
            if (lane == 31) s_wtot[cc & 1][warp] = incl;
            const uint32_t off = incl - (uint32_t)k;
            // the frame encoder's depth vote and packers (dbde_encode_kernel, stage (4))
            const uint32_t kinds = __reduce_or_sync(0xffffffffu, (1u << k) >> 1);
            const bool many_depths = __popc(kinds) >= kEncVarMinDepths;
            if ((kinds & ~3u) == 0u) {
                if (kinds) pack_low_depths(px, k, stage_out + 8 * off);
            } else if (k > 0) {
                const uint32_t c1 = (1u << k) - 256u, c2 = (1u << (2 * k)) - 65536u;
                uint32_t q[16];
#pragma unroll
                for (int i = 0; i < 16; i++) q[i] = squeeze4(px[i], c1, c2);
                uint2 *wp = reinterpret_cast<uint2 *>(stage_out + 8 * off);
                auto store = [&](int n, uint32_t lo, uint32_t hi) { wp[n] = make_uint2(lo, hi); };
                if (many_depths) pack_rows_var(q, k, stage_out + 8 * off);
                else switch (k) {
                    case 1: concat_fields<1>(q, store); break;
                    case 2: concat_fields<2>(q, store); break;
                    case 3: concat_fields<3>(q, store); break;
                    case 4: concat_fields<4>(q, store); break;
                    case 5: concat_fields<5>(q, store); break;
                    case 6: concat_fields<6>(q, store); break;
                    case 7: concat_fields<7>(q, store); break;
                    default: enc_store_depth8(q, stage_out + 8 * off, off); break;
                }
            }
            __syncthreads();                           // every warp's count and words are in shared memory
            uint32_t wbase = 0, tot = 0;
#pragma unroll
            for (int w = 0; w < kConsumerWarps; w++) {
                const uint32_t v = s_wtot[cc & 1][w];
                wbase += w < warp ? v : 0u;
                tot += v;
            }
            // depth and minimum planes (dbde_util.cpp:156-157)
            if (valid) {
                rec[kRecDepth + t] = (uint8_t)k;
                rec[rec_min(P.wh) + t] = (uint8_t)mn;
            }
            // this warp's words: one coalesced run
            const uint32_t n = s_wtot[cc & 1][warp];
            uint8_t *dst = rec + fixed + 8 * ((size_t)carry + wbase);
            if (((uintptr_t)dst & 7) == 0) {
                for (uint32_t i = lane; i < n; i += 32)
                    st_stream_u64(dst + 8 * i, *reinterpret_cast<const uint64_t *>(stage_out + 8 * i));
            } else {
                for (uint32_t i = lane; i < 8 * n; i += 32) dst[i] = stage_out[i];
            }
            carry += tot;
            __syncwarp();                              // the copy has read the staging before the next chunk packs into it
        }
        if (warp == 0)
            write_fixed_fields(rec, lane, P.first_index + (uint64_t)f, P.wh, 1, carry, P.frame_offsets, P.frame_sizes,
                               j, P.slot_stride);
    }
}

cudaError_t launch_encode_crops(const EncCropParams &P, int num_sms, cudaStream_t stream) {
    if (P.nrec <= 0) return cudaSuccess;
    return launch_persistent(dbde_encode_crops_kernel, P, (unsigned)P.nrec, kTilesPerPart, 0, num_sms, stream);
}

// ------------------------------------------------------------------ record compaction
// Lays the records of a batch back to back on the device (slot f -> dst + sum of the sizes before f),
// so the host path brings a chunk home with ONE large D2H copy instead of one per record: small
// copies cost PCIe duplex throughput (measured 70 vs 97 GB/s with 1.6 MB vs 64 MiB pieces).
// grid = (blocks per record, records).  HBM traffic: 2 x record bytes, ~1 % of the PCIe time.
__global__ void __launch_bounds__(256) dbde_compact_kernel(const uint8_t *slots, uint64_t slot_stride,
                                                           const uint64_t *sizes, int n, uint8_t *dst) {
    const int f = blockIdx.y;
    uint64_t before = 0;
    for (int i = 0; i < f; i++) before += sizes[i];           // n is a chunk (tens of records)
    const uint64_t bytes = sizes[f];
    const uint8_t *src = slots + (uint64_t)f * slot_stride;
    uint8_t *d = dst + before;
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (uint64_t)gridDim.x * blockDim.x;
    if ((((uintptr_t)src | (uintptr_t)d) & 7) == 0) {
        const uint64_t *s8 = reinterpret_cast<const uint64_t *>(src);
        const uint64_t n8 = bytes >> 3;
        for (uint64_t i = t; i < n8; i += nt) st_stream_u64(d + 8 * i, __ldcs(s8 + i));
        for (uint64_t i = (n8 << 3) + t; i < bytes; i += nt) d[i] = src[i];
    } else {
        for (uint64_t i = t; i < bytes; i += nt) d[i] = src[i];
    }
}

cudaError_t launch_compact(const uint8_t *slots, uint64_t slot_stride, const uint64_t *sizes, int n, uint8_t *dst,
                           cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    unsigned bx = (unsigned)((slot_stride / 8 + 256 * 8 - 1) / (256 * 8));     // ~8 words per thread at worst-case size
    if (bx < 1) bx = 1;
    if (bx > 64) bx = 64;
    dbde_compact_kernel<<<dim3(bx, (unsigned)n), 256, 0, stream>>>(slots, slot_stride, sizes, n, dst);
    return cudaGetLastError();
}

// The exclusive prefix of n record sizes, once, by one CTA: prefix[0..n], prefix[n] = the total.
__global__ void __launch_bounds__(1024) dbde_prefix_kernel(const uint64_t *sizes, int n, uint64_t *prefix) {
    __shared__ uint64_t s_warp[32];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t carry = 0;
    for (int b = 0; b < n; b += 1024) {
        const int i = b + tid;
        const uint64_t v = i < n ? sizes[i] : 0ull;
        uint64_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint64_t u = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += u;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint64_t before = carry, tot = 0;
        for (int w = 0; w < 32; w++) {
            before += w < warp ? s_warp[w] : 0ull;
            tot += s_warp[w];
        }
        if (i < n) prefix[i] = before + incl - v;
        carry += tot;
        __syncthreads();
    }
    if (tid == 0) prefix[n] = carry;
}

// dbde_compact_kernel with the prefix given, one record row per gridDim.y rows
__global__ void __launch_bounds__(256) dbde_compact_prefixed_kernel(const uint8_t *slots, uint64_t slot_stride, const uint64_t *sizes,
                                                                    const uint64_t *prefix, int n, uint8_t *dst) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (uint64_t)gridDim.x * blockDim.x;
    for (int f = blockIdx.y; f < n; f += gridDim.y) {
        const uint64_t bytes = sizes[f];
        const uint8_t *src = slots + (uint64_t)f * slot_stride;
        uint8_t *d = dst + prefix[f];
        if ((((uintptr_t)src | (uintptr_t)d) & 7) == 0) {
            const uint64_t *s8 = reinterpret_cast<const uint64_t *>(src);
            const uint64_t n8 = bytes >> 3;
            for (uint64_t i = t; i < n8; i += nt) st_stream_u64(d + 8 * i, __ldcs(s8 + i));
            for (uint64_t i = (n8 << 3) + t; i < bytes; i += nt) d[i] = src[i];
        } else {
            for (uint64_t i = t; i < bytes; i += nt) d[i] = src[i];
        }
    }
}

cudaError_t launch_compact_prefixed(const uint8_t *slots, uint64_t slot_stride, const uint64_t *sizes, uint64_t *prefix, int n,
                                    uint8_t *dst, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    dbde_prefix_kernel<<<1, 1024, 0, stream>>>(sizes, n, prefix);
    unsigned bx = (unsigned)((slot_stride / 8 + 256 * 8 - 1) / (256 * 8));
    if (bx < 1) bx = 1;
    if (bx > 64) bx = 64;
    const unsigned by = n < 65535 ? (unsigned)n : 65535u;
    dbde_compact_prefixed_kernel<<<dim3(bx, by), 256, 0, stream>>>(slots, slot_stride, sizes, prefix, n, dst);
    return cudaGetLastError();
}

cudaError_t cached_occupancy(const void *kernel, int threads, size_t smem, int *occ) {
    struct Entry {
        const void *kernel;
        int dev, threads, occ;
        size_t smem;
    };
    struct Limit {                   // the kernel's dynamic shared-memory opt-in on a device: only ever raised
        const void *kernel;
        int dev;
        size_t smem;
    };
    static std::mutex mu;
    static std::vector<Entry> table;
    static std::vector<Limit> limits;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(mu);
    for (const Entry &x : table)
        if (x.kernel == kernel && x.dev == dev && x.threads == threads && x.smem == smem) {
            *occ = x.occ;
            return cudaSuccess;
        }
    Limit *lim = nullptr;
    for (Limit &l : limits)
        if (l.kernel == kernel && l.dev == dev) lim = &l;
    if (!lim || lim->smem < smem) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        if (lim) lim->smem = smem;
        else limits.push_back(Limit{kernel, dev, smem});
    }
    int n = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem);
    if (e != cudaSuccess) return e;
    if (n < 1) return cudaErrorLaunchOutOfResources;
    table.push_back(Entry{kernel, dev, threads, n, smem});
    *occ = n;
    return cudaSuccess;
}

size_t enc_smem_bytes(const PartGeom &g) {
    return ((sizeof(EncSmem) + 127) & ~(size_t)127) + (size_t)kEncStages * g.stage_bytes + 2 * (size_t)kConsumerWarps * kEncWarpBytes;
}

cudaError_t launch_encode(const EncParams &Pin, bool fast, int num_sms, cudaStream_t stream) {
    EncParams P = Pin;
    const size_t smem = enc_smem_bytes(P.g);
    const bool wide = fast && (P.g.w % kTilesPerPart == 0) && P.g.pitch == kWidePitch;
    const bool contig = !fast;
    // the stage holds the partition's pixels exactly as they lie in the frame (full-width partitions, pitch W), or
    // a band segment's eight rows at a pitch that is W modulo 16 (wider frames; make_geom sized the stage for it)
    if (contig && P.g.nseg == 1) P.g.pitch = P.g.W;
    void (*kern)(const EncParams) = nullptr;
    if (wide) kern = dbde_encode_kernel<true, true, false>;
    else if (fast && P.g.linear) kern = dbde_encode_kernel<true, false, false, 0, true>;
    else if (fast) kern = dbde_encode_kernel<true, false, false>;
    else switch (P.g.W & 7) {
        case 0: kern = dbde_encode_kernel<false, false, true, 0>; break;
        case 1: kern = dbde_encode_kernel<false, false, true, 1>; break;
        case 2: kern = dbde_encode_kernel<false, false, true, 2>; break;
        case 3: kern = dbde_encode_kernel<false, false, true, 3>; break;
        case 4: kern = dbde_encode_kernel<false, false, true, 4>; break;
        case 5: kern = dbde_encode_kernel<false, false, true, 5>; break;
        case 6: kern = dbde_encode_kernel<false, false, true, 6>; break;
        default: kern = dbde_encode_kernel<false, false, true, 7>; break;
    }
    return launch_persistent(kern, P, P.nparts, kEncThreads, smem, num_sms, stream);
}

}  // namespace dbde
