// DBDE16 on B200: the 16-bit extension of the DBDE frame codec that the format note hints at
// (reference README.md:65 "could expand size to handle higher bit depth images"; SURVEY.md 8 f-4).
// The reference has no such code, so nothing here replaces a reference function; the layout is the
// reference's with a two-byte minimum plane (restated for the tests in the checker's "DBDE16" section):
//   I32 2 | U64 index | F64 0.0 | I32 wh | U8 depth[wh] (0..16) | I32 2*wh | U16 min[wh] | I32 n64 | U64 words[n64]
// and a frame whose pixels fit in 8 bits gets the 8-bit codec's depth plane and words.
//
// Simpler than the 8-bit kernels (this is the "next" row, not the headline path), same ideas:
// one lane == one 8x8 tile, min/max with VIMNMX.U16x2, depth = 32 - clz(max - min), a partition of 256
// consecutive tiles per CTA iteration, frame-interleaved tickets + the single-word decoupled look-back for
// the word offsets, words staged in shared memory and copied out coalesced.  Pixels are read and written
// with 16-byte accesses when rows allow it (W % 8 == 0, aligned base), element-wise with clamp/crop otherwise.
// Sub-frame decodes run after the same scan and share the decoder's pair extraction (unpack_tile16):
// dbde16_decode_crops_kernel unpacks only the tiles under each crop, dbde16_decode_binned_kernel<B> stores each tile's
// B x B block means instead of its pixels.
#include "dbde_device.cuh"
#include "dbde_kernels.h"

namespace dbde {

constexpr int kT16 = 256;                      // tiles per partition == threads per CTA
constexpr int kWordBytes16 = 128 * kT16;       // worst case: 16 words per tile
// The staged words are addressed as 32-bit units with one unit of padding after every 32: a tile's words
// start 2k units after its neighbour's, and without the padding equal-depth neighbours at k = 8 / 16 land
// on 2 / 1 of the 32 banks (measured: all-depth-16 noise 2.0 / 1.1 TB/s before, see DESIGN.md).
__device__ __forceinline__ uint32_t pad16(uint32_t unit) { return unit + (unit >> 5); }
constexpr int kWordBytesPadded16 = kWordBytes16 + kWordBytes16 / 32 + 64;

// ------------------------------------------------------------------ tile <-> registers
// px[4r + j] = pixels (2j, 2j+1) of tile row r, low half first.  Clamp-to-edge padding as
// dbde_pack_8x8_partial (dbde_util.cpp:105-135).
__device__ __forceinline__ void load_tile16(const uint16_t *frame, int W, int H, int ty, int tx, bool aligned, uint32_t (&px)[32]) {
    const int rows_valid = min(8, H - 8 * ty), cols_valid = min(8, W - 8 * tx);
    if (aligned && rows_valid == 8 && cols_valid == 8) {          // the common case: one pointer, eight 16-byte loads
        const uint4 *row = reinterpret_cast<const uint4 *>(frame + (size_t)(8 * ty) * W + 8 * tx);
        const size_t pitch = (size_t)W / 8;                       // in 16-byte units
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint4 v = __ldcs(row + r * pitch);
            px[4 * r] = v.x; px[4 * r + 1] = v.y; px[4 * r + 2] = v.z; px[4 * r + 3] = v.w;
        }
        return;
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint16_t *row = frame + (size_t)(8 * ty + min(r, rows_valid - 1)) * W + 8 * tx;
        if (aligned && cols_valid == 8) {
            const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(row));
            px[4 * r] = v.x; px[4 * r + 1] = v.y; px[4 * r + 2] = v.z; px[4 * r + 3] = v.w;
        } else if (cols_valid == 8) {
            // a full row of an odd-width frame: 4-byte accesses (the row starts on an even or an odd pixel)
            if (((uintptr_t)row & 3) == 0) {
                const uint32_t *r32 = reinterpret_cast<const uint32_t *>(row);
#pragma unroll
                for (int j = 0; j < 4; j++) px[4 * r + j] = r32[j];
            } else {
                const uint32_t *r32 = reinterpret_cast<const uint32_t *>(row + 1);
                const uint32_t a0 = row[0], w0 = r32[0], w1 = r32[1], w2 = r32[2], a7 = row[7];
                px[4 * r] = a0 | (w0 << 16);
                px[4 * r + 1] = __funnelshift_r(w0, w1, 16);
                px[4 * r + 2] = __funnelshift_r(w1, w2, 16);
                px[4 * r + 3] = (w2 >> 16) | (a7 << 16);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t a = row[min(2 * j, cols_valid - 1)], b = row[min(2 * j + 1, cols_valid - 1)];
                px[4 * r + j] = a | (b << 16);
            }
        }
    }
}

// crop as dbde_unpack_8x8_partial (dbde_util.cpp:281-289): only rows < H and columns < W are written
__device__ __forceinline__ void store_tile16(uint16_t *frame, int W, int H, int ty, int tx, bool aligned, const uint32_t (&px)[32]) {
    const int rows_valid = min(8, H - 8 * ty), cols_valid = min(8, W - 8 * tx);
    if (aligned && rows_valid == 8 && cols_valid == 8) {
        uint4 *row = reinterpret_cast<uint4 *>(frame + (size_t)(8 * ty) * W + 8 * tx);
        const size_t pitch = (size_t)W / 8;
#pragma unroll
        for (int r = 0; r < 8; r++) st_stream_v4u32(row + r * pitch, make_uint4(px[4 * r], px[4 * r + 1], px[4 * r + 2], px[4 * r + 3]));
        return;
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        if (r >= rows_valid) break;
        uint16_t *row = frame + (size_t)(8 * ty + r) * W + 8 * tx;
        if (aligned && cols_valid == 8) {
            st_stream_v4u32(row, make_uint4(px[4 * r], px[4 * r + 1], px[4 * r + 2], px[4 * r + 3]));
        } else if (cols_valid == 8) {
            if (((uintptr_t)row & 3) == 0) {
                uint32_t *r32 = reinterpret_cast<uint32_t *>(row);
#pragma unroll
                for (int j = 0; j < 4; j++) r32[j] = px[4 * r + j];
            } else {
                uint32_t *r32 = reinterpret_cast<uint32_t *>(row + 1);
                row[0] = (uint16_t)px[4 * r];
                r32[0] = __funnelshift_r(px[4 * r], px[4 * r + 1], 16);
                r32[1] = __funnelshift_r(px[4 * r + 1], px[4 * r + 2], 16);
                r32[2] = __funnelshift_r(px[4 * r + 2], px[4 * r + 3], 16);
                row[7] = (uint16_t)(px[4 * r + 3] >> 16);
            }
        } else {
#pragma unroll
            for (int c = 0; c < 8; c++)
                if (c < cols_valid) row[c] = (uint16_t)(px[4 * r + (c >> 1)] >> (16 * (c & 1)));
        }
    }
}

// The 8 pixels of the combined row [prev (pixels 0-7), x (pixels 8-15)] starting at pixel 8 - s, s = 0..7: a shifter
// of selects that is branch-free for any s, so segments of one warp may differ in s
__device__ __forceinline__ uint4 shift_in16(uint4 prev, uint4 x, uint32_t s) {
    const uint32_t v[8] = {prev.x, prev.y, prev.z, prev.w, x.x, x.y, x.z, x.w};
    const uint32_t q = s >> 1;
    uint32_t a[6], u[5];
#pragma unroll
    for (int i = 0; i < 6; i++) a[i] = (q & 2u) ? v[i] : v[i + 2];            // a[i] = v[2 + i - 2 (q >> 1)]
#pragma unroll
    for (int i = 0; i < 5; i++) u[i] = (q & 1u) ? a[i] : a[i + 1];            // u[i] = v[3 + i - q]
    uint32_t r[4];
#pragma unroll
    for (int j = 0; j < 4; j++) r[j] = (s & 1u) ? __funnelshift_r(u[j], u[j + 1], 16) : u[j + 1];
    return make_uint4(r[0], r[1], r[2], r[3]);
}

// ------------------------------------------------------------------ encoder
// The pair packer every DBDE16 encoder shares: (p - min), k bits each, LSB first, two pixels (2k bits) per step into a
// 64-bit accumulator, flushed 32 bits at a time to the staging at shared address sbase in the padded layout (pad16);
// the tile's k U64 words start at 32-bit unit `unit` of the staging.  k = 1..16: a tile of depth 0 has no words.
__device__ __forceinline__ void pack_tile16(uint32_t sbase, uint32_t unit, int k, uint32_t mn, const uint32_t (&px)[32]) {
    const uint32_t m2 = mn * 0x00010001u, kk = 2u * (uint32_t)k;
    uint32_t acc = 0, fill = 0;                                          // `fill` (< 32) valid low bits in acc
    const uint32_t kmul = 1u << k;
#pragma unroll
    for (int i = 0; i < 32; i++) {
        const uint32_t d = px[i] - m2;                                   // no borrow: every pixel >= min
        const uint32_t pair = (d >> 16) * kmul + (d & 0xffffu);          // 2k bits
        const uint32_t lo = acc | (pair << fill);
        const uint32_t hi = __funnelshift_l(pair, 0u, fill);             // what does not fit in 32 bits (0 when fill == 0)
        fill += kk;
        // a unit is complete: predicated store (no branch), carry the overflow
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ge.u32 p, %2, 32;\n\t@p st.shared.u32 [%0], %1;\n\t}"
                     ::"r"(sbase + 4u * pad16(unit)), "r"(lo), "r"(fill) : "memory");
        const bool full = fill >= 32u;
        acc = full ? hi : lo;
        unit += full ? 1u : 0u;
        fill &= 31u;
    }
}

// min of the 64 pixels (two per word, VIMNMX.U16x2) into mn; returns the depth bits(max - min), 0..16
__device__ __forceinline__ int tile_stats16(const uint32_t (&px)[32], uint32_t &mn) {
    uint32_t lo2 = px[0], hi2 = px[0];
#pragma unroll
    for (int i = 1; i < 32; i++) {
        lo2 = __vminu2(lo2, px[i]);
        hi2 = __vmaxu2(hi2, px[i]);
    }
    mn = min(lo2 & 0xffffu, lo2 >> 16);
    const uint32_t mx = max(hi2 & 0xffffu, hi2 >> 16);
    return 32 - __clz((int)(mx - mn));
}

__global__ void __launch_bounds__(kT16, 4) dbde16_encode_kernel(const Enc16Params P) {
    extern __shared__ __align__(16) uint8_t s_words[];
    __shared__ uint32_t s_ticket, s_wtot[kT16 / 32];
    __shared__ uint64_t s_excl;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t fpix = (size_t)P.W * P.H;
    const size_t fixed = rec_fixed(P.wh, 2);
    for (;;) {
        if (tid == 0) s_ticket = atomicAdd(P.ticket, 1u);
        __syncthreads();
        const unsigned t = s_ticket;
        if (t >= P.nparts) break;
        // frame-interleaved order (ticket t -> frame t mod N, partition t div N): a partition's predecessors
        // in its frame hold smaller tickets, so they have started and the look-back below terminates
        const unsigned q = t / (unsigned)P.nframes, f = t - q * (unsigned)P.nframes;
        const unsigned p = f * (unsigned)P.ppf + q;
        const int tile = (int)q * kT16 + tid;
        const bool valid = tile < P.wh;
        const int ty = valid ? tile / P.w : 0, tx = valid ? tile - ty * P.w : 0;
        uint32_t px[32];
        load_tile16(P.frames + (size_t)f * fpix, P.W, P.H, ty, tx, P.aligned != 0, px);
        uint32_t mn;
        int k = tile_stats16(px, mn);
        if (!valid) { k = 0; mn = 0; }
        const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
        if (lane == 31) s_wtot[warp] = incl;
        __syncthreads();
        uint32_t wbase = 0, agg = 0;
#pragma unroll
        for (int v = 0; v < kT16 / 32; v++) {
            const uint32_t x = s_wtot[v];
            if (v < warp) wbase += x;
            agg += x;
        }
        if (warp == 0) {
            // decoupled look-back over this frame's partitions (one chain per frame: the word count restarts
            // at every frame, as n64 does at dbde_util.cpp:146)
            uint64_t excl = 0;
            if (q > 0) {
                if (lane == 0) st_relaxed_u64(P.desc + p, desc_make(kDescAggregate, agg));
                excl = lookback_exclusive<true>(P.desc, p, p - q, lane);
            }
            if (lane == 0) {
                st_relaxed_u64(P.desc + p, desc_make(kDescPrefix, excl + agg));
                s_excl = excl;
            }
        }
        // the tile's words start at word wbase + incl - k of the partition
        if (k > 0) pack_tile16(smem_u32(s_words), 2u * (wbase + incl - (uint32_t)k), k, mn, px);
        __syncthreads();                                      // words staged, s_excl published
        const uint64_t excl = s_excl;
        uint8_t *rec = P.out + (size_t)f * P.slot_stride;
        if (valid) {
            rec[kRecDepth + tile] = (uint8_t)k;                                           // depth plane
            rec[rec_min(P.wh) + 2 * (size_t)tile] = (uint8_t)mn;                          // minimum plane, little-endian U16
            rec[rec_min(P.wh) + 2 * (size_t)tile + 1] = (uint8_t)(mn >> 8);
        }
        uint8_t *dst = rec + fixed + 8 * excl;
        const uint32_t *su = reinterpret_cast<const uint32_t *>(s_words);
        if (((uintptr_t)dst & 7) == 0) {
            for (uint32_t i = (uint32_t)tid; i < agg; i += kT16)
                st_stream_u64(dst + 8 * (size_t)i, (uint64_t)su[pad16(2u * i)] | ((uint64_t)su[pad16(2u * i + 1u)] << 32));
        } else {
            for (uint32_t i = (uint32_t)tid; i < 8u * agg; i += kT16) dst[i] = s_words[4u * pad16(i >> 2) + (i & 3u)];
        }
        if (q == (unsigned)P.ppf - 1 && warp == 0)
            write_fixed_fields(rec, lane, P.first_index + f, P.wh, 2, (uint32_t)(excl + agg), P.frame_offsets, P.frame_sizes, f,
                               P.slot_stride);
        __syncthreads();                                      // s_words / s_ticket are reused by the next partition
    }
}

// ------------------------------------------------------------------ crop encoder
// dbde_encode_crops_kernel's scheme with DBDE16 tiles: one CTA per record (frame f, crop r) of a persistent grid, one
// lane per tile of the crop.  The CTA walks the crop's tiles in raster order, 256 at a time; a record's word offsets
// depend on its own tiles only, so a CTA-wide scan per chunk plus a running carry replaces the frame encoder's look-back
// and tickets, and no scratch is zeroed.  Each warp packs its 32 tiles into a region of its own of the staging (1024
// units, at most 32 tiles of 16 words), so the scan's one barrier per chunk is the only CTA-wide wait.

// The 8 rows of crop tile (tx, ty): pixel (x, y) of the crop image is frame[y0 + y][x0 + x] inside the frame and pad
// outside it; the clamp padding at the crop's own partial last column / row repeats the crop image's last valid pixel
// (dbde_util.cpp:105-135), which may be pad.  A tile inside the frame and the crop loads each row as the one or two
// aligned 16-byte words it touches and shifts the 8 pixels out of them (any x0, any W, any 2-byte aligned frame base);
// a tile at an edge reads each in-frame pixel it needs as a U16 and nothing else.
__device__ __forceinline__ void load_crop_tile16(const Enc16CropParams &P, const uint16_t *fr, long long x0, long long y0, int tx, int ty,
                                                 uint32_t (&px)[32]) {
    const long long xs = x0 + 8 * tx, ys = y0 + 8 * ty;
    const bool inner = 8 * tx + 8 <= P.crop_w && 8 * ty + 8 <= P.crop_h && xs >= 0 && xs + 8 <= P.W && ys >= 0 && ys + 8 <= P.H;
    if (inner) {
        const uint16_t *p = fr + (size_t)ys * (size_t)P.W + (size_t)xs;
#pragma unroll
        for (int r = 0; r < 8; r++) {
            const uint4 *a = reinterpret_cast<const uint4 *>((uintptr_t)p & ~(uintptr_t)15);
            const uint32_t s = ((uint32_t)(uintptr_t)p & 15u) >> 1;              // the row starts at pixel s of word a
            uint4 v = __ldg(a);
            if (s) v = shift_in16(v, __ldg(a + 1), 8u - s);
            px[4 * r] = v.x; px[4 * r + 1] = v.y; px[4 * r + 2] = v.z; px[4 * r + 3] = v.w;
            p += P.W;
        }
        return;
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const long long y = y0 + min(8 * ty + r, P.crop_h - 1);
        if (y >= 0 && y < P.H) {
            const uint16_t *row = fr + (size_t)y * (size_t)P.W;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const long long xa = x0 + min(8 * tx + 2 * j, P.crop_w - 1), xb = x0 + min(8 * tx + 2 * j + 1, P.crop_w - 1);
                const uint32_t a = xa >= 0 && xa < P.W ? (uint32_t)__ldg(row + xa) : P.pad;
                const uint32_t b = xb >= 0 && xb < P.W ? (uint32_t)__ldg(row + xb) : P.pad;
                px[4 * r + j] = a | (b << 16);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) px[4 * r + j] = P.pad * 0x00010001u;
        }
    }
}

constexpr uint32_t kCropWarpUnits16 = 32 * 16 * 2;   // one warp's staging region: 32 tiles of at most 16 U64 words

__global__ void __launch_bounds__(kT16, 4) dbde16_encode_crops_kernel(const Enc16CropParams P) {
    extern __shared__ __align__(16) uint8_t s_words[];
    __shared__ uint32_t s_wtot[2][kT16 / 32];                // each warp's word count, by chunk parity
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t fpix = (size_t)P.W * (size_t)P.H;
    const size_t fixed = rec_fixed(P.wh, 2);
    const uint32_t wunit = (uint32_t)warp * kCropWarpUnits16;   // a multiple of 32: pad16(wunit + u) = pad16(wunit) + pad16(u)
    const uint32_t *su = reinterpret_cast<const uint32_t *>(s_words);
    unsigned cc = 0;                                         // chunks done by this CTA: selects the s_wtot half
    for (int j = blockIdx.x; j < P.nrec; j += gridDim.x) {
        const int f = j / P.ncrops, r = j - f * P.ncrops;
        const int32_t *cp = P.corners + 2 * ((size_t)f * (size_t)P.corner_stride + (size_t)r);
        const long long x0 = __ldg(cp), y0 = __ldg(cp + 1);
        const uint16_t *fr = P.frames + (size_t)f * fpix;
        uint8_t *rec = P.out + (size_t)j * P.slot_stride;
        uint32_t carry = 0;                                  // U64 words of the record's earlier chunks
        for (int t0 = 0; t0 < P.wh; t0 += kT16, cc++) {
            const int t = t0 + tid;
            const bool valid = t < P.wh;
            uint32_t px[32];
            if (valid) {
                const int ty = t / P.w;
                load_crop_tile16(P, fr, x0, y0, t - ty * P.w, ty, px);
            } else {
#pragma unroll
                for (int i = 0; i < 32; i++) px[i] = 0;
            }
            // dbde16_encode_kernel's tile: min, depth (0 for the zeros past the crop's last tile), the pair packer
            uint32_t mn;
            const int k = tile_stats16(px, mn);
            const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
            if (lane == 31) s_wtot[cc & 1][warp] = incl;
            if (k > 0) pack_tile16(smem_u32(s_words), wunit + 2u * (incl - (uint32_t)k), k, mn, px);
            // depth and minimum planes (dbde_util.cpp:156-157), the minimum little-endian U16
            if (valid) {
                rec[kRecDepth + (size_t)t] = (uint8_t)k;
                rec[rec_min(P.wh) + 2 * (size_t)t] = (uint8_t)mn;
                rec[rec_min(P.wh) + 1 + 2 * (size_t)t] = (uint8_t)(mn >> 8);
            }
            __syncthreads();                                 // every warp's count is in shared memory
            uint32_t wbase = 0, tot = 0;
#pragma unroll
            for (int w = 0; w < kT16 / 32; w++) {
                const uint32_t v = s_wtot[cc & 1][w];
                wbase += w < warp ? v : 0u;
                tot += v;
            }
            // this warp's words: one coalesced run
            const uint32_t n = s_wtot[cc & 1][warp];
            uint8_t *dst = rec + fixed + 8 * ((size_t)carry + wbase);
            if (((uintptr_t)dst & 7) == 0) {
                for (uint32_t i = lane; i < n; i += 32)
                    st_stream_u64(dst + 8 * (size_t)i, (uint64_t)su[pad16(wunit + 2u * i)] | ((uint64_t)su[pad16(wunit + 2u * i + 1u)] << 32));
            } else {
                for (uint32_t i = lane; i < 8u * n; i += 32) dst[i] = s_words[4u * pad16(wunit + (i >> 2)) + (i & 3u)];
            }
            carry += tot;
            __syncwarp();                                    // the copy has read the staging before the next chunk packs into it
        }
        if (warp == 0)   // wh widened from unsigned: from int, ptxas reschedules the chunk loop and the crops encode 2.5 % slower
            write_fixed_fields(rec, lane, P.first_index + (uint64_t)f, (uint32_t)P.wh, 2, carry, P.frame_offsets, P.frame_sizes, j,
                               P.slot_stride);
    }
}

// ------------------------------------------------------------------ decoder: validate + scan
// One CTA per frame: the checks of dbde_unpack_image carried over (dbde_util.cpp:295-303: nb == wh,
// nm == 2*wh, sum(depth) == n64; plus the tag, depth <= 16, bounds) and the exclusive word prefix of every
// 32-tile group (the running input pointer of :312 made explicit).
__global__ void __launch_bounds__(256) dbde16_scan_kernel(const Dec16Params P) {
    __shared__ uint32_t s_warp[8], s_flag;
    const int f = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ng = (P.wh + 31) / 32;
    uint32_t *wp = P.wprefix + (size_t)f * (ng + 1);
    ScanHead h;
    if (!scan_head(P.stream, P.stream_bytes, P.frame_offsets[f], P.wh, 2, f, P.status, P.indices, h)) return;
    if (tid == 0) s_flag = 0;
    __syncthreads();
    const uint8_t *dp = h.rec + kRecDepth;
    bool big = false;
    for (int g0 = warp * 4; g0 < ng; g0 += 32) {              // four groups in flight per warp
        uint32_t d[4];
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int t = 32 * (g0 + b) + lane;
            d[b] = (g0 + b < ng && t < P.wh) ? dp[t] : 0u;
        }
#pragma unroll
        for (int b = 0; b < 4; b++) {
            if (d[b] > 16u) { big = true; d[b] = 16u; }
            const uint32_t sum = __reduce_add_sync(0xffffffffu, d[b]);
            if (lane == 0 && g0 + b < ng) wp[g0 + b] = sum;
        }
    }
    if (big) atomicOr(&s_flag, 1u);
    __syncthreads();
    const uint32_t total = scan_items(wp, ng, s_warp, tid, warp, lane);
    if (tid == 0) scan_finish(h, wp, ng, total, s_flag != 0, f, P.status, P.indices);
}

// ------------------------------------------------------------------ decoder: unpack
// The pair extraction every DBDE16 decoder shares.  `su` is staged payload in the padded layout (pad16): after every
// 32 units comes one padding unit holding a COPY of the unit that follows it, so "this unit and the next" is always
// two adjacent loads.  The tile's k words start at word `woff` of the staging; px[4r + j] = pixels (2j, 2j+1) of tile
// row r.  Depth 0 is the minimum everywhere.
__device__ __forceinline__ void unpack_tile16(const uint32_t *su, uint32_t woff, int k, uint32_t mn, uint32_t (&px)[32]) {
    const uint32_t m2 = mn * 0x00010001u;
    if (k > 0) {
        const uint32_t kk = 2u * (uint32_t)k, mk = (1u << k) - 1u;
#pragma unroll
        for (int i = 0; i < 32; i++) {
            const uint32_t bit = kk * (uint32_t)i;                               // pair i: bits [2k i, 2k i + 2k)
            const uint32_t at = pad16(2u * woff + (bit >> 5));
            const uint32_t a = su[at], b = su[at + 1u];                          // the next unit, or its copy in the padding slot
            const uint32_t v = __funnelshift_r(a, b, bit);                       // low 2k bits = the pair
            px[i] = ((v & mk) | (((v >> k) & mk) << 16)) + m2;                    // + min, wrapping per pixel is impossible: <= 65535
        }
    } else {
#pragma unroll
        for (int i = 0; i < 32; i++) px[i] = m2;
    }
}

// bytes [s, e) of the 64-bit word w at the 8-byte-aligned q: store_partial, which leaves the whole word to its
// callers, or one 8-byte store
__device__ __forceinline__ void store_word_part(uint8_t *q, uint64_t w, uint32_t s, uint32_t e) {
    if (s == 0u && e == 8u) *reinterpret_cast<uint64_t *>(q) = w;
    else store_partial(q, w, s, e);
}

// n <= 4 U16 values (v, lowest first) to p, any even address, as naturally aligned pieces
__device__ __forceinline__ void store_u16s(uint16_t *p, uint64_t v, uint32_t n) {
    const uint32_t a = (uint32_t)(uintptr_t)p & 7u, e = a + 2u * n;
    uint8_t *q = reinterpret_cast<uint8_t *>(p) - a;
    if (e <= 8u) {
        store_word_part(q, v << (8 * a), a, e);
    } else {                                                  // a > 0 here
        store_partial(q, v << (8 * a), a, 8u);
        store_partial(q + 8, v >> (64 - 8 * a), 0u, e - 8u);
    }
}

// Binned epilogue: one tile's pixels -> the rounded means of its (8 / B)^2 bins of B x B, one piece of 8 / B values
// per bin row at `op` (frame row pitch Wb).  wc / hr: the tile's in-frame columns / rows.  A tile in the frame's last
// tile column / row (W % 8 or H % 8 != 0) first zeroes the encoder's clamp padding past W and H -- it must not enter
// the mean -- divides each bin by its count of in-frame pixels and skips the bins past ceil(W / B) and ceil(H / B).
// Sums are 32-bit: an 8 x 8 bin sums to at most 64 * 65535.
template <int B>
__device__ __forceinline__ void store_bins16(uint16_t *op, int Wb, int ncb, int nrb, int wc, int hr, uint32_t (&px)[32]) {
    constexpr int NB = 8 / B;                                 // bins per tile side
    const bool edge = wc < 8 || hr < 8;
    if (edge) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t m = 2 * j + 2 <= wc ? ~0u : 2 * j + 1 == wc ? 0xffffu : 0u;
#pragma unroll
            for (int r = 0; r < 8; r++) px[4 * r + j] = r < hr ? px[4 * r + j] & m : 0u;
        }
    }
#pragma unroll
    for (int by = 0; by < NB; by++) {
        uint64_t v = 0;
#pragma unroll
        for (int bx = 0; bx < NB; bx++) {
            uint32_t s = 0;
#pragma unroll
            for (int r = B * by; r < B * by + B; r++)
#pragma unroll
                for (int j = B * bx / 2; j < (B * bx + B) / 2; j++) s += (px[4 * r + j] & 0xffffu) + (px[4 * r + j] >> 16);
            uint32_t m;
            if (!edge) {
                m = (s + B * B / 2) >> (B == 2 ? 2 : B == 4 ? 4 : 6);
            } else {
                const uint32_t n = (uint32_t)max(1, min(B, hr - B * by)) * (uint32_t)max(1, min(B, wc - B * bx));
                m = (s + n / 2) / n;
            }
            v |= (uint64_t)m << (16 * bx);
        }
        if (!edge) {
            if constexpr (B == 2) {
                if (((uintptr_t)op & 7u) == 0) st_stream_u64(op, v);
                else store_u16s(op, v, 4u);
            } else if constexpr (B == 4) {
                if (((uintptr_t)op & 3u) == 0) st_stream_u32(op, (uint32_t)v);
                else store_u16s(op, v, 2u);
            } else {
                *op = (uint16_t)v;
            }
        } else if (by < nrb) {
            store_u16s(op, v, (uint32_t)ncb);
        }
        op += Wb;
    }
}

// agg words at src (any alignment), spread over nlanes threads (this one is `lane`), into the padded layout of
// unpack_tile16 at su.  Padded layout (pad16): after every 32 units comes one padding unit, and that padding unit holds a
// COPY of the unit that follows it, so the reader's "this unit and the next" is always two adjacent loads.
// CROP = false, the full decoders: each partition is read once, streaming (__ldcs), and a run that is not 8-byte aligned
// is copied a byte at a time, the code these decoders have always had.  CROP = true, the crop decoder: loads take the
// read-only path, and an unaligned run is read four bytes per 32-bit unit -- with byte copies its 1001x1003 crops ran
// 21 % slower.
template <bool CROP>
__device__ __forceinline__ void stage_words16(uint32_t *su, const uint8_t *src, uint32_t agg, uint32_t lane, uint32_t nlanes) {
    if (((uintptr_t)src & 7) == 0) {
        for (uint32_t i = lane; i < agg; i += nlanes) {
            const uint64_t *p = reinterpret_cast<const uint64_t *>(src) + i;
            const uint64_t v = CROP ? __ldg(p) : __ldcs(p);
            const uint32_t at = pad16(2u * i);                                  // units 2i and 2i+1 share a block of 32
            su[at] = (uint32_t)v;
            su[at + 1u] = (uint32_t)(v >> 32);
            if (((2u * i) & 31u) == 0u && i > 0u) su[at - 1u] = (uint32_t)v;    // the copy in the padding slot before it
        }
    } else if (CROP) {
        for (uint32_t u = lane; u < 2u * agg; u += nlanes) {
            const uint32_t v = ld_le32(src + 4u * u);
            const uint32_t at = pad16(u);
            su[at] = v;
            if ((u & 31u) == 0u && u > 0u) su[at - 1u] = v;
        }
    } else {
        uint8_t *s8 = reinterpret_cast<uint8_t *>(su);
        for (uint32_t i = lane; i < 8u * agg; i += nlanes) {
            const uint32_t u = i >> 2;
            s8[4u * pad16(u) + (i & 3u)] = src[i];
            if ((u & 31u) == 0u && u > 0u) s8[4u * (pad16(u) - 1u) + (i & 3u)] = src[i];
        }
    }
    if (lane < 2) {                                                           // the reader looks one unit past the end
        const uint32_t u = 2u * agg + lane;
        su[pad16(u)] = 0u;
        if ((u & 31u) == 0u && u > 0u) su[pad16(u) - 1u] = 0u;
    }
}

__global__ void __launch_bounds__(kT16) dbde16_decode_kernel(const Dec16Params P) {
    extern __shared__ __align__(16) uint8_t s_words[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const size_t fpix = (size_t)P.W * P.H;
    const int ng = (P.wh + 31) / 32;
    for (unsigned p = blockIdx.x; p < P.nparts; p += gridDim.x) {
        const unsigned f = p / (unsigned)P.ppf, q = p - f * (unsigned)P.ppf;
        if (P.status[f] != 0) continue;                       // rejected by the scan: the image stays untouched
        const uint8_t *rec = P.stream + P.frame_offsets[f];
        const uint32_t *wp = P.wprefix + (size_t)f * (ng + 1);
        const int g0 = (int)q * (kT16 / 32), g1 = min(g0 + kT16 / 32, ng);
        const uint32_t w0 = wp[g0], agg = wp[g1] - w0;
        // the partition's words, coalesced, into shared memory
        const uint8_t *src = rec + rec_fixed(P.wh, 2) + 8ull * w0;
        stage_words16<false>(reinterpret_cast<uint32_t *>(s_words), src, agg, (uint32_t)tid, kT16);
        const int tile = (int)q * kT16 + tid;
        const bool valid = tile < P.wh;
        int k = 0;
        uint32_t mn = 0;
        if (valid) {
            k = rec[kRecDepth + tile];
            const uint8_t *mp = rec + rec_min(P.wh) + 2 * (size_t)tile;
            mn = (uint32_t)mp[0] | ((uint32_t)mp[1] << 8);
        }
        const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
        const uint32_t woff = (g0 + warp < ng ? wp[g0 + warp] - w0 : 0u) + incl - (uint32_t)k;
        __syncthreads();
        uint32_t px[32];
        unpack_tile16(reinterpret_cast<const uint32_t *>(s_words), woff, k, mn, px);
        if (valid) {
            const int ty = tile / P.w, tx = tile - ty * P.w;
            store_tile16(P.frames + (size_t)f * fpix, P.W, P.H, ty, tx, P.aligned != 0, px);
        }
        __syncthreads();                                      // s_words is reused by the next partition
    }
}

// Binned decode: dbde16_decode_kernel's partition loop with the bin epilogue (store_bins16) in place of the tile
// store; P.frames is the binned output, frames of ceil(W / B) x ceil(H / B) U16.  B divides 8, so no bin crosses a
// tile.  A kernel of its own, not a template of the full decoder: folding the two into one loop changes the full
// decoder's code.
template <int B>
__global__ void __launch_bounds__(kT16) dbde16_decode_binned_kernel(const Dec16Params P) {
    extern __shared__ __align__(16) uint8_t s_words[];
    constexpr int NB = 8 / B;                                 // bins per tile side
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ng = (P.wh + 31) / 32;
    const int Wb = (P.W + B - 1) / B, Hb = (P.H + B - 1) / B;
    const size_t fbins = (size_t)Wb * (size_t)Hb;
    for (unsigned p = blockIdx.x; p < P.nparts; p += gridDim.x) {
        const unsigned f = p / (unsigned)P.ppf, q = p - f * (unsigned)P.ppf;
        if (P.status[f] != 0) continue;                       // rejected by the scan: the output stays untouched
        const uint8_t *rec = P.stream + P.frame_offsets[f];
        const uint32_t *wp = P.wprefix + (size_t)f * (ng + 1);
        const int g0 = (int)q * (kT16 / 32), g1 = min(g0 + kT16 / 32, ng);
        const uint32_t w0 = wp[g0], agg = wp[g1] - w0;
        stage_words16<false>(reinterpret_cast<uint32_t *>(s_words), rec + rec_fixed(P.wh, 2) + 8ull * w0, agg, (uint32_t)tid, kT16);
        const int tile = (int)q * kT16 + tid;
        const bool valid = tile < P.wh;
        int k = 0;
        uint32_t mn = 0;
        if (valid) {
            k = rec[kRecDepth + tile];
            const uint8_t *mp = rec + rec_min(P.wh) + 2 * (size_t)tile;
            mn = (uint32_t)mp[0] | ((uint32_t)mp[1] << 8);
        }
        const uint32_t incl = warp_inclusive_scan((uint32_t)k, lane);
        const uint32_t woff = (g0 + warp < ng ? wp[g0 + warp] - w0 : 0u) + incl - (uint32_t)k;
        __syncthreads();
        uint32_t px[32];
        unpack_tile16(reinterpret_cast<const uint32_t *>(s_words), woff, k, mn, px);
        if (valid) {
            const int ty = tile / P.w, tx = tile - ty * P.w;
            uint16_t *op = P.frames + (size_t)f * fbins + (size_t)(NB * ty) * (size_t)Wb + (size_t)(NB * tx);
            store_bins16<B>(op, Wb, min(NB, Wb - NB * tx), min(NB, Hb - NB * ty), P.W - 8 * tx, P.H - 8 * ty, px);
        }
        __syncthreads();                                      // s_words is reused by the next partition
    }
}

// ------------------------------------------------------------------ decoder: crops
// ncrops rectangles of crop_w x crop_h per frame at int32 corners, after dbde16_scan_kernel, on the task grid of the
// 8-bit crop decoder (crop_task): one warp == up to 32 consecutive tile columns of one tile row of a crop of one frame,
// one lane == one tile, in segments of S lanes for crops narrower than 32 tiles.  A segment stages its payload run in
// the padded layout and unpacks with unpack_tile16.  Lanes whose tile lies outside the frame unpack depth 0 with the
// pad value as minimum.  Rows are cropped on all four sides and leave as aligned 16-byte words assembled across lanes.
struct Crop16Params {
    CropGrid g;                 // the scan's outputs, the frame, the crops and their tasks
    uint16_t *out;              // nframes * ncrops * crop_w * crop_h, tightly packed, 2-byte aligned
    uint32_t pad2;              // the pad value in both halves
};

constexpr int kCrop16Warps = 8;
// per segment of S lanes: 32 S units of payload (S tiles of <= 16 words), the unit past the end, the padding: 33 S + 2
// units; 32 / S segments per warp
constexpr int kCrop16BufUnits = 1120;

// pixels [st, en) of the 16-byte-aligned 8-pixel word w at q, as naturally aligned pieces
__device__ __forceinline__ void store_pixels16(uint16_t *q, uint4 w, int st, int en) {
    uint8_t *q8 = reinterpret_cast<uint8_t *>(q);
    if (st < 4) store_word_part(q8, ((uint64_t)w.y << 32) | w.x, 2u * st, 2u * min(en, 4));
    if (en > 4) store_word_part(q8 + 8, ((uint64_t)w.w << 32) | w.z, 2u * max(st - 4, 0), 2u * (en - 4));
}

// One pixel row of a segment's tiles into a crop row of cw pixels.  Lane l's 8 pixels belong at row + pos.
// Consecutive lanes hold consecutive 16-byte pieces, so every lane assembles the ALIGNED 16-byte word its piece
// starts in -- its left neighbour's tail and its own head -- and stores the part inside [row, row + cw).  A segment's
// first lane leaves the pixels before its piece to the last lane of the previous chunk, which stores its tail past its
// word.  Warp-wide call; `live`: this lane has a tile of the crop in a row of the crop.
__device__ __forceinline__ void crop16_store_row(uint16_t *row, int pos, uint4 x, int cw, bool live, bool first, bool last) {
    uint4 prev;
    prev.x = __shfl_up_sync(0xffffffffu, x.x, 1);
    prev.y = __shfl_up_sync(0xffffffffu, x.y, 1);
    prev.z = __shfl_up_sync(0xffffffffu, x.z, 1);
    prev.w = __shfl_up_sync(0xffffffffu, x.w, 1);
    if (!live) return;
    const uint32_t s = (((uint32_t)(uintptr_t)row + 2u * (uint32_t)pos) & 15u) >> 1;   // the same in every lane of a segment
    const int qo = pos - (int)s;                                                         // my aligned word: row + qo
    const uint4 w = shift_in16(prev, x, s);
    const int st = max(-qo, first ? (int)s : 0), en = min(cw - qo, 8);
    uint16_t *q = row + qo;
    if (st == 0 && en == 8) st_stream_v4u32(q, w);
    else if (st < en) store_pixels16(q, w, st, en);
    if (last && s) {                                                                      // my pixels past that word
        const int st2 = max(-qo - 8, 0), en2 = min(cw - qo - 8, (int)s);
        if (st2 < en2) store_pixels16(q + 8, shift_in16(x, make_uint4(0u, 0u, 0u, 0u), s), st2, en2);
    }
}

__global__ void __launch_bounds__(kCrop16Warps * 32) dbde16_decode_crops_kernel(const Crop16Params P) {
    __shared__ __align__(16) uint32_t s_buf[kCrop16Warps][kCrop16BufUnits];
    const CropGrid &G = P.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    CropTask T;
    if (!crop_task<true>(G, (unsigned long long)blockIdx.x * kCrop16Warps + warp, lane, T)) return;
    const int S = T.S, sl = T.sl, tx = T.tx;
    uint32_t mn = P.pad2 & 0xffffu;                          // outside the frame: depth 0 with the pad value as minimum
    if (T.inframe) {
        const uint8_t *mp = T.rec + rec_min(G.wh) + 2 * (size_t)T.tl;
        mn = (uint32_t)mp[0] | ((uint32_t)mp[1] << 8);
    }
    // stage the segment's run (nothing outside it is read)
    uint32_t *su = s_buf[warp] + T.seg * (33 * S + 2);
    stage_words16<true>(su, T.rec + rec_fixed(G.wh, 2) + 8 * (size_t)T.wbase, T.nwords, (uint32_t)sl, (uint32_t)S);
    __syncwarp();

    uint32_t px[32];
    unpack_tile16(su, T.incl - T.k, (int)T.k, mn, px);

    // the frame's partial last tile column / row: pixels past column W and rows past H are pad
    const int wc = T.inframe && tx == G.w - 1 ? (G.W & 7) : 0;          // kept pixels of each row, 0 = all
    const int hr = T.inframe && T.ty == G.h - 1 ? G.H - 8 * T.ty : 8;     // kept rows
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t m = wc == 0 || 2 * j + 2 <= wc ? ~0u : 2 * j + 1 == wc ? 0xffffu : 0u;
#pragma unroll
        for (int rr = 0; rr < 8; rr++) px[4 * rr + j] = rr < hr ? (px[4 * rr + j] & m) | (P.pad2 & ~m) : P.pad2;
    }
    // crop and store: rows of the tile inside [y0, y0 + crop_h), columns inside [x0, x0 + crop_w).  Offsets are taken
    // from the crop's first tile, so corners near INT32_MAX do not overflow
    uint16_t *rout = P.out + (size_t)T.rect * ((size_t)G.crop_w * (size_t)G.crop_h);
    const int pos = 8 * (tx - T.tx0) - (T.x0 & 7);
    const bool last = sl == S - 1 || tx + 1 >= T.tx_end;
#pragma unroll
    for (int rr = 0; rr < 8; rr++) {
        const int yr = 8 * T.rowi + rr - (T.y0 & 7);                           // the same in every lane of a segment
        const bool in = T.live && yr >= 0 && yr < G.crop_h;
        crop16_store_row(rout + (in ? (size_t)yr * (size_t)G.crop_w : 0), pos,
                         make_uint4(px[4 * rr], px[4 * rr + 1], px[4 * rr + 2], px[4 * rr + 3]), G.crop_w, in, sl == 0, last);
    }
}

// ------------------------------------------------------------------ launches
cudaError_t launch_encode16(const Enc16Params &P, int num_sms, cudaStream_t stream) {
    return launch_persistent(dbde16_encode_kernel, P, P.nparts, kT16, kWordBytesPadded16, num_sms, stream);
}
cudaError_t launch_encode16_crops(const Enc16CropParams &P, int num_sms, cudaStream_t stream) {
    if (P.nrec <= 0) return cudaSuccess;
    return launch_persistent(dbde16_encode_crops_kernel, P, (unsigned)P.nrec, kT16, kWordBytesPadded16, num_sms, stream);
}
cudaError_t launch_decode16_scan(const Dec16Params &P, cudaStream_t stream) {
    if (P.nframes <= 0) return cudaSuccess;
    dbde16_scan_kernel<<<P.nframes, 256, 0, stream>>>(P);
    return cudaGetLastError();
}
cudaError_t launch_decode16(const Dec16Params &P, int num_sms, cudaStream_t stream) {
    return launch_persistent(dbde16_decode_kernel, P, P.nparts, kT16, kWordBytesPadded16, num_sms, stream);
}

cudaError_t launch_decode16_binned(const Dec16Params &scan, int factor, uint16_t *out, int num_sms, cudaStream_t stream) {
    Dec16Params P = scan;
    P.frames = out;
    switch (factor) {
        case 2: return launch_persistent(dbde16_decode_binned_kernel<2>, P, P.nparts, kT16, kWordBytesPadded16, num_sms, stream);
        case 4: return launch_persistent(dbde16_decode_binned_kernel<4>, P, P.nparts, kT16, kWordBytesPadded16, num_sms, stream);
        case 8: return launch_persistent(dbde16_decode_binned_kernel<8>, P, P.nparts, kT16, kWordBytesPadded16, num_sms, stream);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_decode16_crops(const Dec16Params &scan, const int32_t *corners, int ncrops, bool per_frame, int crop_w,
                                  int crop_h, int pad, uint16_t *out, cudaStream_t stream) {
    Crop16Params P = Crop16Params();
    unsigned blocks = 0;
    // a crop starting 7 columns / rows into a tile spans one tile more than one starting on a tile boundary
    const cudaError_t e = crop_grid(P.g, scan, scan.W, scan.H, (scan.wh + 31) / 32, crop_w, crop_h, ncrops,
                                    (int)(((long long)crop_w + 14) / 8), (int)(((long long)crop_h + 14) / 8), kCrop16Warps, &blocks);
    if (e != cudaSuccess) return e;
    if (blocks == 0) return cudaSuccess;
    P.g.corners = corners;
    P.g.corner_stride = per_frame ? ncrops : 0;
    P.out = out;
    P.pad2 = (uint32_t)(pad & 0xFFFF) * 0x00010001u;
    dbde16_decode_crops_kernel<<<blocks, kCrop16Warps * 32, 0, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace dbde
