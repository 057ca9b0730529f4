// DBDE B200 region-of-interest and crop decoder: frame records in HBM -> the pixels of rectangles of every
// frame, tightly packed, equal to the crop of dbde_unpack_frame's image (dbde_util.cpp:291-328, 339-345) and
// with its accept/reject behaviour.
//
// Two launches:
//   dbde_decode_scan_kernel (dbde_decode.cu, unchanged) on a LINEAR geometry (linear_geom): partitions of
//     256 consecutive tiles, so word-prefix item i is exactly tiles [32 i, 32 i + 32) of the frame's
//     row-major tile order.  It validates the WHOLE record (a record damaged outside the region is still
//     rejected, with the same status bits as dbde_b200_decode_device) and reads 1 byte per tile.
//   dbde_decode_roi_kernel (one rectangle inside the frame, the same for every frame) or
//   dbde_decode_crops_kernel (ncrops fixed-size rectangles per frame at corners read from device memory, any
//     position, pixels outside the frame set to a pad byte) -- one kernel body, roi_body<CROPS>: one warp ==
//     32 consecutive tile columns of one tile row of a rectangle in one frame, one lane == one tile.  Payloads
//     lie in row-major tile order, so the warp's in-frame payloads are ONE contiguous byte run of the record:
//     the warp stages it into shared memory with coalesced 16-byte loads and unpacks with the decoder's
//     unpack_tile.  Its first tile's word offset is the item prefix plus at most 31 depth bytes; the rest is a
//     warp scan of the 32 depths.  Rows are cropped on all four sides and stored at the rectangle's pitch, any
//     alignment, as runs of aligned 8-byte words assembled across lanes.
//     A rectangle narrower than 32 tiles gives a tile row a SEGMENT of S lanes (the next power of two >= its
//     width) and a warp 32 / S tile rows, each segment doing all of the above on its own: a one-pixel
//     column keeps 32 lanes busy instead of one.
#include "dbde_device.cuh"
#include "dbde_kernels.h"

namespace dbde {

// one launch of dbde_decode_roi_kernel / dbde_decode_crops_kernel
struct RoiParams {
    CropGrid g;                 // the scan's outputs, the frame, the rectangles and their tasks
    uint8_t *out;               // nframes * ncrops * crop_w * crop_h, tightly packed, any alignment
    uint32_t flags;             // kFlagInvertRows
    uint32_t pad4;              // crops: the pad byte in every byte
};

namespace {

constexpr int kRoiWarps = 8;
// per segment of S lanes: its payload run (<= S tiles x 64 bytes) + its offset inside the first 16-byte granule
// (< 16) + the unpackers' over-read past a tile's last byte (< 16); 32 / S segments per warp
constexpr int kRoiBufBytes = 32 * (64 + 32);

// One pixel row of a segment's tiles into an output row of roi_w bytes at any alignment.  Lane l's 8 pixels
// belong at row + pos (pos = 8 l + 256 chunk - (x0 & 7), l the lane within its segment: the region's first
// tile starts up to 7 columns left of the region, the left crop).  Consecutive lanes hold consecutive 8-byte
// pieces, so every lane assembles the ALIGNED word its piece starts in -- its left neighbour's tail (one
// shuffle) and its own head -- and stores the part of it inside [row, row + roi_w): a row is a run of aligned
// 8-byte stores, with narrow stores only at the region's edges and at the ends of a 32-tile chunk (the model
// is store_rows_direct, DESIGN.md section 4).  A segment's first lane leaves the bytes before its piece to the
// last lane of the previous chunk, which stores its tail past its word.  Warp-wide call; `live`: this lane
// has a tile of the region in a row of the region.
__device__ __forceinline__ void roi_store_row(uint8_t *row, int pos, uint64_t x, int roi_w, bool live, bool first, bool last) {
    const uint64_t prev = __shfl_up_sync(0xffffffffu, x, 1);
    if (!live) return;
    const uint32_t a = (uint32_t)((uintptr_t)row + (intptr_t)pos) & 7u;     // the same in every lane of a segment
    const int qo = pos - (int)a;                                             // my aligned word starts at row + qo
    uint64_t w = x;
    if (a) {
        w = x << (8 * a);
        if (!first) w |= prev >> (64 - 8 * a);
    }
    const int s = max(-qo, first ? (int)a : 0), e = min(roi_w - qo, 8);
    uint8_t *q = row + qo;
    if (s == 0 && e == 8) st_stream_u64(q, w);
    else if (s < e) store_partial(q, w, (uint32_t)s, (uint32_t)e);
    if (last && a) {                                                         // my bytes past that word
        // (a one-tile-wide region can start inside them: the left crop applies here too)
        const int s2 = max(-qo - 8, 0), e2 = min(roi_w - qo - 8, (int)a);
        if (s2 < e2) store_partial(q + 8, x >> (64 - 8 * a), (uint32_t)s2, (uint32_t)e2);
    }
}

// The one kernel body.  CROPS = false: the rectangle is the launch's region, inside the frame.  CROPS = true: the
// task's rectangle comes from `corners`; lanes whose tile lies outside the frame load nothing and give pad
// pixels, and the frame's partial last tile column / row is padded past W / H.  Everything after the prologue
// is shared.
template <bool CROPS>
__device__ __forceinline__ void roi_body(const RoiParams &P, uint8_t *s_wbuf, int warp, int lane) {
    const CropGrid &G = P.g;
    CropTask T;
    if (!crop_task<CROPS>(G, (unsigned long long)blockIdx.x * kRoiWarps + warp, lane, T)) return;
    const int S = T.S, sl = T.sl, tx = T.tx;
    // a lane outside the frame unpacks depth 0 with the pad byte as its minimum: pad pixels
    const uint32_t k = T.k;
    const uint32_t mn = T.inframe ? (uint32_t)T.rec[rec_min(G.wh) + T.tl] : (CROPS ? P.pad4 & 0xFFu : 0u);

    // stage the segment's payload run [gs, ge): sbuf[i] <-> byte a0 + i.  16-byte loads for the aligned interior,
    // byte loads for the < 16 head and tail bytes -- nothing outside the run is read
    uint8_t *sbuf = s_wbuf + T.seg * (64 * S + 32);
    const uintptr_t gs = (uintptr_t)(T.rec + rec_fixed(G.wh, 1)) + 8 * (uintptr_t)T.wbase;
    const uintptr_t ge = gs + 8 * (uintptr_t)T.nwords;
    const uintptr_t a0 = gs & ~(uintptr_t)15;
    const uintptr_t h = min((gs + 15) & ~(uintptr_t)15, ge);
    const uintptr_t e16 = max(ge & ~(uintptr_t)15, h);
    for (uintptr_t a = h + 16 * (uintptr_t)sl; a < e16; a += 16 * (uintptr_t)S)
        *reinterpret_cast<uint4 *>(sbuf + (a - a0)) = __ldg(reinterpret_cast<const uint4 *>(a));
    for (int j = sl; j < 32; j += S) {
        const uintptr_t a = j < 16 ? gs + (uintptr_t)j : e16 + (uintptr_t)(j - 16);
        if (j < 16 ? a < h : a < ge) sbuf[a - a0] = *reinterpret_cast<const uint8_t *>(a);
    }
    __syncwarp();

    uint32_t px[16];
    unpack_tile(sbuf + (gs - a0) + 8 * (size_t)(T.incl - k), (int)k, mn * 0x01010101u, (gs & 7u) == 0, (P.flags & kFlagInvertRows) != 0,
                px);

    if constexpr (CROPS) {
        // the frame's partial last tile column / row: bytes past column W and rows past H are pad (after the
        // invert-endian row reversal)
        const int wc = T.inframe && tx == G.w - 1 ? (G.W & 7) : 0;            // kept bytes of each row, 0 = all
        const uint32_t mlo = wc == 0 || wc >= 4 ? ~0u : (1u << (8 * wc)) - 1u;
        const uint32_t mhi = wc == 0 ? ~0u : wc > 4 ? (1u << (8 * (wc - 4))) - 1u : 0u;
        const int hr = T.ty == G.h - 1 ? G.H - 8 * T.ty : 8;                    // kept rows
#pragma unroll
        for (int r = 0; r < 8; r++) {
            px[2 * r] = r < hr ? (px[2 * r] & mlo) | (P.pad4 & ~mlo) : P.pad4;
            px[2 * r + 1] = r < hr ? (px[2 * r + 1] & mhi) | (P.pad4 & ~mhi) : P.pad4;
        }
    }
    // crop and store: rows of the tile inside [y0, y0 + roi_h), columns inside [x0, x0 + roi_w).  Offsets are taken
    // from the rectangle's first tile, so corners near INT32_MAX do not overflow
    uint8_t *rout = P.out + (size_t)T.rect * ((size_t)G.crop_w * (size_t)G.crop_h);
    const int pos = 8 * (tx - T.tx0) - (T.x0 & 7);
    const bool last = sl == S - 1 || tx + 1 >= T.tx_end;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int yr = 8 * T.rowi + r - (T.y0 & 7);                            // the same in every lane of a segment
        const bool in = T.live && yr >= 0 && yr < G.crop_h;
        roi_store_row(rout + (in ? (size_t)yr * (size_t)G.crop_w : 0), pos, ((uint64_t)px[2 * r + 1] << 32) | px[2 * r], G.crop_w,
                      in, sl == 0, last);
    }
}

}  // namespace

__global__ void __launch_bounds__(kRoiWarps * 32) dbde_decode_roi_kernel(const RoiParams P) {
    __shared__ __align__(16) uint8_t s_buf[kRoiWarps][kRoiBufBytes];
    roi_body<false>(P, s_buf[threadIdx.x >> 5], threadIdx.x >> 5, threadIdx.x & 31);
}

// The region kernel's occupancy (40 registers, 6 CTAs per SM): left alone, ptxas takes 43 registers here, which
// allows 5, and with the bound it still needs no spills
__global__ void __launch_bounds__(kRoiWarps * 32, 6) dbde_decode_crops_kernel(const RoiParams P) {
    __shared__ __align__(16) uint8_t s_buf[kRoiWarps][kRoiBufBytes];
    roi_body<true>(P, s_buf[threadIdx.x >> 5], threadIdx.x >> 5, threadIdx.x & 31);
}

namespace {

template <bool CROPS>
cudaError_t launch_roi_body(const RoiParams &P, unsigned blocks, cudaStream_t stream) {
    if (blocks == 0) return cudaSuccess;
    if (CROPS) dbde_decode_crops_kernel<<<blocks, kRoiWarps * 32, 0, stream>>>(P);
    else dbde_decode_roi_kernel<<<blocks, kRoiWarps * 32, 0, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace

// Both take the scan of scan.g = linear_geom(W, H): its word-prefix items are ppf * 8 per frame
cudaError_t launch_decode_roi(const DecParams &scan, int x0, int y0, int roi_w, int roi_h, uint8_t *out, cudaStream_t stream) {
    RoiParams P = RoiParams();
    unsigned blocks = 0;
    const cudaError_t e = crop_grid(P.g, scan, scan.g.W, scan.g.H, scan.g.ppf * kConsumerWarps, roi_w, roi_h, 1,
                                    (x0 + roi_w + 7) / 8 - x0 / 8, (y0 + roi_h + 7) / 8 - y0 / 8, kRoiWarps, &blocks);
    if (e != cudaSuccess) return e;
    P.g.x0 = x0;
    P.g.y0 = y0;
    P.out = out;
    P.flags = scan.flags;
    return launch_roi_body<false>(P, blocks, stream);
}

cudaError_t launch_decode_crops(const DecParams &scan, const int32_t *corners, int ncrops, bool per_frame, int crop_w, int crop_h,
                                int pad, uint8_t *out, cudaStream_t stream) {
    RoiParams P = RoiParams();
    unsigned blocks = 0;
    // a crop starting 7 columns / rows into a tile spans one tile more than one starting on a tile boundary
    const cudaError_t e = crop_grid(P.g, scan, scan.g.W, scan.g.H, scan.g.ppf * kConsumerWarps, crop_w, crop_h, ncrops,
                                    (int)(((long long)crop_w + 14) / 8), (int)(((long long)crop_h + 14) / 8), kRoiWarps, &blocks);
    if (e != cudaSuccess) return e;
    P.g.corners = corners;
    P.g.corner_stride = per_frame ? ncrops : 0;
    P.out = out;
    P.flags = scan.flags;
    P.pad4 = (uint32_t)(pad & 0xFF) * 0x01010101u;
    return launch_roi_body<true>(P, blocks, stream);
}

}  // namespace dbde
