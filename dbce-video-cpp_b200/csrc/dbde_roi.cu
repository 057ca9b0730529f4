// DBDE B200 region-of-interest decoder: frame records in HBM -> the pixels of one rectangle of every
// frame, tightly packed (roi_w x roi_h per frame), equal to the crop of dbde_unpack_frame's image
// (dbde_util.cpp:291-328, 339-345) and with its accept/reject behaviour.
//
// Two launches:
//   dbde_decode_scan_kernel (dbde_decode.cu, unchanged) on a LINEAR geometry (linear_geom): partitions of
//     256 consecutive tiles, so word-prefix item i is exactly tiles [32 i, 32 i + 32) of the frame's
//     row-major tile order.  It validates the WHOLE record (a record damaged outside the region is still
//     rejected, with the same status bits as dbde_b200_decode_device) and reads 1 byte per tile.
//   dbde_decode_roi_kernel : one warp == 32 consecutive tile columns of one tile row of the region in one
//     frame, one lane == one tile.  Payloads lie in row-major tile order, so the warp's 32 payloads are ONE
//     contiguous byte run of the record: the warp stages it into shared memory with coalesced 16-byte loads
//     and unpacks with the decoder's unpack_tile.  Its first tile's word offset is the item prefix plus at most
//     31 depth bytes; the rest is a warp scan of the 32 depths.  Rows are cropped on all four sides and
//     stored at pitch roi_w, any alignment, as runs of aligned 8-byte words assembled across lanes.
//     A region narrower than 32 tiles gives a tile row a SEGMENT of S lanes (the next power of two >= its
//     width) and a warp 32 / S tile rows, each segment doing all of the above on its own: a one-pixel
//     column keeps 32 lanes busy instead of one.
#include "dbde_device.cuh"
#include "dbde_kernels.h"

namespace dbde {

// one launch of dbde_decode_roi_kernel: the scan's outputs and the region's tiling (launch_decode_roi)
struct RoiParams {
    const uint8_t *stream;
    const uint64_t *frame_offsets;
    const uint32_t *status;     // from the scan: frames with status != 0 are skipped
    const uint32_t *wprefix;    // nframes * (nitems + 1)
    uint8_t *out;               // nframes * roi_w * roi_h, tightly packed, any alignment
    int w, wh, nitems;          // tile columns, tiles, word-prefix items per frame (ppf * 8)
    int x0, y0, roi_w, roi_h;
    int tx0, ty0, tx_end;       // the region's first tile column / row, one past its last tile column
    int nty, nchunks;           // tile rows of the region, 32-tile warps per tile row
    int seg_shift;              // log2 of the lanes per tile row: 5, or fewer for regions narrower than 32 tiles
    int nrg;                    // warps (groups of 32 >> seg_shift tile rows) per 32-tile column chunk and frame
    unsigned long long ntasks;  // nframes * nrg * nchunks warps
    uint32_t flags;             // kFlagInvertRows
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

}  // namespace

__global__ void __launch_bounds__(kRoiWarps * 32) dbde_decode_roi_kernel(const RoiParams P) {
    __shared__ __align__(16) uint8_t s_buf[kRoiWarps][kRoiBufBytes];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned long long task = (unsigned long long)blockIdx.x * kRoiWarps + warp;
    if (task >= P.ntasks) return;
    // task = (f * nrg + row group) * nchunks + chunk: neighbouring warps read neighbouring payloads
    const int chunk = (int)(task % (unsigned)P.nchunks);
    const unsigned long long fr = task / (unsigned)P.nchunks;
    const int f = (int)(fr / (unsigned)P.nrg);
    const int rg = (int)(fr - (unsigned long long)f * (unsigned)P.nrg);
    if (P.status[f] != 0) return;                            // rejected by the scan: the region stays untouched
    // S = 1 << seg_shift lanes per tile row: a region narrower than 32 tiles puts 32 / S tile rows in one warp
    const int S = 1 << P.seg_shift;
    const int seg = lane >> P.seg_shift, sl = lane & (S - 1);
    const int rowi = (rg << (5 - P.seg_shift)) + seg;        // tile row of the region
    const bool rowok = rowi < P.nty;
    const int ty = P.ty0 + rowi;
    const int txc = P.tx0 + 32 * chunk;                      // my segment's first tile column
    const bool live = rowok && txc + sl < P.tx_end;
    const uint8_t *rec = P.stream + P.frame_offsets[f];
    const int t0 = ty * P.w + txc;                           // its row-major tile index
    const int item = t0 >> 5, rem = t0 & 31;

    // word offset of tile t0: the item's exclusive prefix plus the depths of the item's tiles before t0
    // (dbde_util.cpp:312, the reference's running input pointer, made explicit)
    uint32_t before = 0;
    if (rowok)
        for (int j = sl; j < rem; j += S) before += rec[24 + 32 * item + j];
    for (int o = 1; o < S; o <<= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    const uint32_t k = live ? (uint32_t)rec[24 + t0 + sl] : 0u;
    const uint32_t mn = live ? (uint32_t)rec[28 + P.wh + t0 + sl] : 0u;
    const uint32_t wbase = rowok ? P.wprefix[(size_t)f * (P.nitems + 1) + item] + before : 0u;
    uint32_t incl = k;                                       // inclusive scan of the depths inside the segment
    for (int d = 1; d < S; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d, S);
        if (sl >= d) incl += t;
    }
    const uint32_t nwords = __shfl_sync(0xffffffffu, incl, S - 1, S);

    // stage the segment's payload run [gs, ge): sbuf[i] <-> byte a0 + i.  16-byte loads for the aligned interior,
    // byte loads for the < 16 head and tail bytes -- nothing outside the run is read
    uint8_t *sbuf = s_buf[warp] + seg * (64 * S + 32);
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

    // crop and store: rows of the tile inside [y0, y0 + roi_h), columns inside [x0, x0 + roi_w)
    uint8_t *fout = P.out + (size_t)f * ((size_t)P.roi_w * (size_t)P.roi_h);
    const int pos = 8 * (txc - P.tx0 + sl) - (P.x0 & 7);
    const bool last = sl == S - 1 || txc + sl + 1 >= P.tx_end;
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int yr = 8 * ty + r - P.y0;                                      // the same in every lane of a segment
        const bool in = live && yr >= 0 && yr < P.roi_h;
        roi_store_row(fout + (in ? (size_t)yr * (size_t)P.roi_w : 0), pos, ((uint64_t)px[2 * r + 1] << 32) | px[2 * r], P.roi_w,
                      in, sl == 0, last);
    }
}

cudaError_t launch_decode_roi(const DecParams &scan, int x0, int y0, int roi_w, int roi_h, uint8_t *out, cudaStream_t stream) {
    RoiParams P;
    P.stream = scan.stream;
    P.frame_offsets = scan.frame_offsets;
    P.status = scan.status;
    P.wprefix = scan.wprefix;
    P.out = out;
    P.w = scan.g.w;
    P.wh = scan.g.wh;
    P.nitems = scan.g.ppf * kConsumerWarps;
    P.x0 = x0; P.y0 = y0; P.roi_w = roi_w; P.roi_h = roi_h;
    P.tx0 = x0 / 8;
    P.ty0 = y0 / 8;
    P.tx_end = (x0 + roi_w + 7) / 8;
    P.nty = (y0 + roi_h + 7) / 8 - P.ty0;
    P.nchunks = (P.tx_end - P.tx0 + 31) / 32;
    // segments: the next power of two >= the region's width in tiles, at most 32 lanes
    P.seg_shift = 0;
    while ((1 << P.seg_shift) < P.tx_end - P.tx0 && P.seg_shift < 5) P.seg_shift++;
    P.nrg = (P.nty + (32 >> P.seg_shift) - 1) / (32 >> P.seg_shift);
    P.ntasks = (unsigned long long)scan.nframes * (unsigned long long)P.nrg * (unsigned long long)P.nchunks;
    P.flags = scan.flags;
    if (P.ntasks == 0) return cudaSuccess;
    const unsigned long long blocks = (P.ntasks + kRoiWarps - 1) / kRoiWarps;
    if (blocks > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
    dbde_decode_roi_kernel<<<(unsigned)blocks, kRoiWarps * 32, 0, stream>>>(P);
    return cudaGetLastError();
}

}  // namespace dbde
