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

// one launch of dbde_decode_roi_kernel / dbde_decode_crops_kernel: the scan's outputs and the rectangles' tiling
struct RoiParams {
    const uint8_t *stream;
    const uint64_t *frame_offsets;
    const uint32_t *status;     // from the scan: frames with status != 0 are skipped
    const uint32_t *wprefix;    // nframes * (nitems + 1)
    uint8_t *out;               // nframes * ncrops * roi_w * roi_h, tightly packed, any alignment
    int w, wh, nitems;          // tile columns, tiles, word-prefix items per frame (ppf * 8)
    int x0, y0, roi_w, roi_h;   // crops: x0, y0 unused (per task from `corners`)
    int tx0, ty0, tx_end;       // the region's first tile column / row, one past its last tile column (region only)
    int nty, nchunks;           // tile rows of the region (crops: at most), 32-tile warps per tile row
    int seg_shift;              // log2 of the lanes per tile row: 5, or fewer for rectangles narrower than 32 tiles
    int nrg;                    // warps (groups of 32 >> seg_shift tile rows) per 32-tile column chunk and rectangle
    unsigned long long ntasks;  // nframes * ncrops * nrg * nchunks warps
    uint32_t flags;             // kFlagInvertRows
    // crops only
    const int32_t *corners;     // {x0, y0} of crop r of frame f at corners + 2 * (f * corner_stride + r)
    int ncrops, corner_stride;  // corner_stride: ncrops (per-frame corners) or 0 (shared)
    int W, H, h;                // the frame in pixels and tile rows: what lies outside it is `pad`
    uint32_t pad4;              // the pad byte in every byte
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
    const unsigned long long task = (unsigned long long)blockIdx.x * kRoiWarps + warp;
    if (task >= P.ntasks) return;
    // task = ((f * ncrops + r) * nrg + row group) * nchunks + chunk: neighbouring warps read neighbouring payloads
    const int chunk = (int)(task % (unsigned)P.nchunks);
    const unsigned long long fr = task / (unsigned)P.nchunks;
    const unsigned long long fc = fr / (unsigned)P.nrg;
    const int rg = (int)(fr - fc * (unsigned)P.nrg);
    int f, x0, y0, tx0, ty0, tx_end, nty;
    uint8_t *rout;
    if constexpr (CROPS) {
        f = (int)(fc / (unsigned)P.ncrops);
        const int r = (int)(fc - (unsigned long long)f * (unsigned)P.ncrops);
        const int32_t *cp = P.corners + 2 * ((size_t)f * (size_t)P.corner_stride + (size_t)r);
        x0 = __ldg(cp);
        y0 = __ldg(cp + 1);
        // floor division (negative corners), the far edge in 64 bits (corners up to INT32_MAX)
        tx0 = x0 >> 3;
        ty0 = y0 >> 3;
        tx_end = (int)(((long long)x0 + P.roi_w + 7) >> 3);
        nty = (int)(((long long)y0 + P.roi_h + 7) >> 3) - ty0;
        rout = P.out + (size_t)fc * ((size_t)P.roi_w * (size_t)P.roi_h);
    } else {
        f = (int)fc;
        x0 = P.x0; y0 = P.y0; tx0 = P.tx0; ty0 = P.ty0; tx_end = P.tx_end; nty = P.nty;
        rout = P.out + (size_t)f * ((size_t)P.roi_w * (size_t)P.roi_h);
    }
    if (P.status[f] != 0) return;                            // rejected by the scan: its rectangles stay untouched
    // S = 1 << seg_shift lanes per tile row: a rectangle narrower than 32 tiles puts 32 / S tile rows in one warp
    const int S = 1 << P.seg_shift;
    const int seg = lane >> P.seg_shift, sl = lane & (S - 1);
    const int rowi = (rg << (5 - P.seg_shift)) + seg;        // tile row of the rectangle
    const bool rowok = rowi < nty;
    const int ty = ty0 + rowi;
    const int txc = tx0 + 32 * chunk;                        // my segment's first tile column
    const int tx = txc + sl;
    const bool live = rowok && tx < tx_end;
    // the segment's tiles inside the frame: columns [txa, txb) of tile row ty, one contiguous payload run
    int txa = txc;
    bool segin = rowok, inframe = live;
    if constexpr (CROPS) {
        txa = max(txc, 0);
        const int txb = min(min(txc + S, tx_end), P.w);
        segin = rowok && ty >= 0 && ty < P.h && txa < txb;
        inframe = live && segin && tx >= 0 && tx < P.w;
    }
    const uint8_t *rec = P.stream + P.frame_offsets[f];
    const int t0 = ty * P.w + txa;                           // its first row-major tile index (used when segin)
    const int item = t0 >> 5, rem = t0 & 31;
    const int tl = ty * P.w + tx;                            // my tile (when inframe)

    // word offset of tile t0: the item's exclusive prefix plus the depths of the item's tiles before t0
    // (dbde_util.cpp:312, the reference's running input pointer, made explicit)
    uint32_t before = 0;
    if (segin)
        for (int j = sl; j < rem; j += S) before += rec[24 + 32 * item + j];
    for (int o = 1; o < S; o <<= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    const uint32_t k = inframe ? (uint32_t)rec[24 + tl] : 0u;
    // a lane outside the frame unpacks depth 0 with the pad byte as its minimum: pad pixels
    const uint32_t mn = inframe ? (uint32_t)rec[28 + P.wh + tl] : (CROPS ? P.pad4 & 0xFFu : 0u);
    const uint32_t wbase = segin ? P.wprefix[(size_t)f * (P.nitems + 1) + item] + before : 0u;
    uint32_t incl = k;                                       // inclusive scan of the depths inside the segment
    for (int d = 1; d < S; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d, S);
        if (sl >= d) incl += t;
    }
    const uint32_t nwords = __shfl_sync(0xffffffffu, incl, S - 1, S);

    // stage the segment's payload run [gs, ge): sbuf[i] <-> byte a0 + i.  16-byte loads for the aligned interior,
    // byte loads for the < 16 head and tail bytes -- nothing outside the run is read
    uint8_t *sbuf = s_wbuf + seg * (64 * S + 32);
    const uintptr_t gs = (uintptr_t)(rec + 32 + 2 * (size_t)P.wh) + 8 * (uintptr_t)wbase;
    const uintptr_t ge = gs + 8 * (uintptr_t)nwords;
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
    unpack_tile(sbuf + (gs - a0) + 8 * (size_t)(incl - k), (int)k, mn * 0x01010101u, (gs & 7u) == 0, (P.flags & kFlagInvertRows) != 0,
                px);

    if constexpr (CROPS) {
        // the frame's partial last tile column / row: bytes past column W and rows past H are pad (after the
        // invert-endian row reversal)
        const int wc = inframe && tx == P.w - 1 ? (P.W & 7) : 0;              // kept bytes of each row, 0 = all
        const uint32_t mlo = wc == 0 || wc >= 4 ? ~0u : (1u << (8 * wc)) - 1u;
        const uint32_t mhi = wc == 0 ? ~0u : wc > 4 ? (1u << (8 * (wc - 4))) - 1u : 0u;
        const int hr = ty == P.h - 1 ? P.H - 8 * ty : 8;                        // kept rows
#pragma unroll
        for (int r = 0; r < 8; r++) {
            px[2 * r] = r < hr ? (px[2 * r] & mlo) | (P.pad4 & ~mlo) : P.pad4;
            px[2 * r + 1] = r < hr ? (px[2 * r + 1] & mhi) | (P.pad4 & ~mhi) : P.pad4;
        }
    }
    // crop and store: rows of the tile inside [y0, y0 + roi_h), columns inside [x0, x0 + roi_w).  Offsets are taken
    // from the rectangle's first tile, so corners near INT32_MAX do not overflow
    const int pos = 8 * (tx - tx0) - (x0 & 7);
    const bool last = sl == S - 1 || tx + 1 >= tx_end;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int yr = 8 * rowi + r - (y0 & 7);                                // the same in every lane of a segment
        const bool in = live && yr >= 0 && yr < P.roi_h;
        roi_store_row(rout + (in ? (size_t)yr * (size_t)P.roi_w : 0), pos, ((uint64_t)px[2 * r + 1] << 32) | px[2 * r], P.roi_w,
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

// The fields both launches share: the scan's outputs, and the task grid for rectangles of roi_w x roi_h that
// span at most `span` tile columns and `nty` tile rows
void roi_grid(RoiParams &P, const DecParams &scan, int roi_w, int roi_h, int span, int nty, int ncrops, uint8_t *out) {
    P = RoiParams();
    P.stream = scan.stream;
    P.frame_offsets = scan.frame_offsets;
    P.status = scan.status;
    P.wprefix = scan.wprefix;
    P.out = out;
    P.w = scan.g.w;
    P.wh = scan.g.wh;
    P.nitems = scan.g.ppf * kConsumerWarps;
    P.roi_w = roi_w; P.roi_h = roi_h;
    P.nty = nty;
    P.nchunks = (span + 31) / 32;
    // segments: the next power of two >= the rectangle's width in tiles, at most 32 lanes
    P.seg_shift = 0;
    while ((1 << P.seg_shift) < span && P.seg_shift < 5) P.seg_shift++;
    P.nrg = (nty + (32 >> P.seg_shift) - 1) / (32 >> P.seg_shift);
    P.ncrops = ncrops;
    P.ntasks = (unsigned long long)scan.nframes * (unsigned long long)ncrops * (unsigned long long)P.nrg *
               (unsigned long long)P.nchunks;
    P.flags = scan.flags;
}

template <bool CROPS>
cudaError_t launch_roi_body(const RoiParams &P, cudaStream_t stream) {
    if (P.ntasks == 0) return cudaSuccess;
    const unsigned long long blocks = (P.ntasks + kRoiWarps - 1) / kRoiWarps;
    if (blocks > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
    if (CROPS) dbde_decode_crops_kernel<<<(unsigned)blocks, kRoiWarps * 32, 0, stream>>>(P);
    else dbde_decode_roi_kernel<<<(unsigned)blocks, kRoiWarps * 32, 0, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_decode_roi(const DecParams &scan, int x0, int y0, int roi_w, int roi_h, uint8_t *out, cudaStream_t stream) {
    RoiParams P;
    const int tx0 = x0 / 8, ty0 = y0 / 8, tx_end = (x0 + roi_w + 7) / 8;
    roi_grid(P, scan, roi_w, roi_h, tx_end - tx0, (y0 + roi_h + 7) / 8 - ty0, 1, out);
    P.x0 = x0; P.y0 = y0;
    P.tx0 = tx0; P.ty0 = ty0; P.tx_end = tx_end;
    return launch_roi_body<false>(P, stream);
}

cudaError_t launch_decode_crops(const DecParams &scan, const int32_t *corners, int ncrops, bool per_frame, int crop_w, int crop_h,
                                int pad, uint8_t *out, cudaStream_t stream) {
    RoiParams P;
    // a crop starting 7 columns / rows into a tile spans one tile more than one starting on a tile boundary
    roi_grid(P, scan, crop_w, crop_h, (int)(((long long)crop_w + 14) / 8), (int)(((long long)crop_h + 14) / 8), ncrops, out);
    P.corners = corners;
    P.corner_stride = per_frame ? ncrops : 0;
    P.W = scan.g.W;
    P.H = scan.g.H;
    P.h = scan.g.h;
    P.pad4 = (uint32_t)(pad & 0xFF) * 0x01010101u;
    return launch_roi_body<true>(P, stream);
}

}  // namespace dbde
