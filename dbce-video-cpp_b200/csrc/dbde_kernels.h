// Internal interface between the C ABI (dbde_capi.cu) and the kernels, and the pieces the 8-bit and DBDE16 kernels
// share beyond the tile arithmetic of dbde_device.cuh: the decode pre-pass, the crop-decode task grid, the persistent launch.
#pragma once
#include "dbde_device.cuh"

namespace dbde {

struct EncParams {
    PartGeom g;
    const uint8_t *frames;      // nframes * W * H, tightly packed, device
    uint8_t *out;               // slot of frame record 0, device; record f lives at out + f * slot_stride
    uint64_t slot_stride;       // bytes between consecutive frame slots (>= rec_bound(wh, 1))
    uint64_t *frame_offsets;    // nframes entries (= f * slot_stride), device
    uint64_t *frame_sizes;      // nframes entries (record bytes), device
    uint64_t *desc;             // nparts look-back descriptors (index f*ppf + q), zeroed
    unsigned int *ticket;       // zeroed
    uint64_t first_index;
    int nframes;
    unsigned nparts;
    uint32_t flags;             // kFlagInvertRows
};

// Crop encode (dbde_encode.cu): record j = f * ncrops + r is the reference's record of the crop_w x crop_h image at
// corner r of frame f (pixels outside the frame are the pad byte), at out + j * slot_stride.
struct EncCropParams {
    const uint8_t *frames;      // nframes * W * H, tightly packed, device, any alignment
    int W, H;
    const int32_t *corners;     // {x0, y0} of crop r of frame f at corners + 2 * (f * corner_stride + r), any int32 values
    int ncrops, corner_stride;  // corner_stride: ncrops (per-frame corners) or 0 (shared)
    int crop_w, crop_h, w, wh;  // the crop in pixels, its tile columns and tiles
    uint64_t pad8;              // the pad byte in every byte
    uint8_t *out;
    uint64_t slot_stride;       // >= rec_bound(wh, 1)
    uint64_t *frame_offsets;    // nrec entries (= j * slot_stride), device
    uint64_t *frame_sizes;      // nrec entries (record bytes), device
    uint64_t first_index;
    int nrec;                   // nframes * ncrops
    uint32_t flags;             // kFlagInvertRows
};

struct DecParams {
    PartGeom g;
    const uint8_t *stream;      // frame records, device
    uint64_t stream_bytes;
    const uint64_t *frame_offsets;   // nframes entries (record starts), device
    uint8_t *frames;            // nframes * W * H out, device
    uint32_t *status;           // nframes
    uint64_t *indices;          // nframes or null
    uint32_t *wprefix;          // nframes * (ppf*8 + 1) exclusive word prefixes per partition-warp
    int nframes;
    unsigned nparts;
    uint32_t flags;             // kFlagInvertRows
};

// The reference's DBDE_INVERT_ENDIAN build variant (dbde_util.cpp:15-19,24-27,246-270): every 8-pixel tile
// row is byte-reversed before packing and after unpacking.  A launch-uniform flag here.
enum : uint32_t { kFlagInvertRows = 1 };

// status bits reported by the decoder (0 = frame decoded)
enum : uint32_t {
    kStBadFrameHeader = 1,   // u64s != 2                 (dbde_util.cpp:335)
    kStBadDepthCount = 2,    // nb != w*h                 (dbde_util.cpp:296)
    kStBadMinCount = 4,      // nm != w*h                 (dbde_util.cpp:299)
    kStBadWordCount = 8,     // sum(depth) != n64         (dbde_util.cpp:302-303)
    kStDepthTooBig = 16,     // a depth byte > 8 (the reference does not reject this; we do)
    kStTruncated = 32,       // record runs past the end of the stream buffer
};

// ---- the decode pre-pass (dbde_decode_scan_kernel, dbde16_scan_kernel): one CTA of 256 threads per frame validates the
// record as dbde_unpack_image does (dbde_util.cpp:295-303) and turns its depth plane into exclusive U64-word prefixes of
// 32-tile items, the reference's running input pointer (:312) made explicit.  The kernels differ only in how they sum
// the items' depths.
struct ScanHead {
    const uint8_t *rec;
    uint64_t room;              // payload bytes the stream holds after the fixed fields
    uint32_t status, n64;       // the status bits of the fixed fields, the record's word count
};
// The fixed fields of record f at `off`, of wh tiles and mb minimum bytes per tile.  A stream that cannot even hold them
// (no wrap for any off): thread 0 reports the frame truncated and false comes back, the CTA has nothing else to do.
__device__ __forceinline__ bool scan_head(const uint8_t *stream, uint64_t stream_bytes, uint64_t off, int wh, int mb, int f,
                                          uint32_t *status, uint64_t *indices, ScanHead &h) {
    const uint64_t fixed = rec_fixed(wh, mb);
    if (off > stream_bytes || stream_bytes - off < fixed) {
        if (threadIdx.x == 0) {
            status[f] = kStTruncated;
            if (indices) indices[f] = 0;
        }
        return false;
    }
    h.room = stream_bytes - off - fixed;
    h.rec = stream + off;
    h.status = 0;
    if (ld_le32(h.rec) != 2u) h.status |= kStBadFrameHeader;
    if (ld_le32(h.rec + kRecDepthCount) != (uint32_t)wh) h.status |= kStBadDepthCount;
    if (ld_le32(h.rec + rec_min_count(wh)) != (uint32_t)(mb * wh)) h.status |= kStBadMinCount;
    h.n64 = ld_le32(h.rec + rec_n64(wh, mb));
    return true;
}
// Exclusive scan in place of the n item sums at wp, 2048 per round; returns their total.  s_warp: 8 words of shared
// memory.  CTA-wide call.
__device__ __forceinline__ uint32_t scan_items(uint32_t *wp, int n, uint32_t *s_warp, int tid, int warp, int lane) {
    uint32_t carry = 0;
    for (int base = 0; base < n; base += 2048) {
        uint32_t v[8], local = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int idx = base + tid * 8 + i;
            v[i] = idx < n ? wp[idx] : 0u;
            local += v[i];
        }
        const uint32_t incl = warp_inclusive_scan(local, lane);
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t pre = carry + incl - local, tot = 0;
#pragma unroll
        for (int wv = 0; wv < 8; wv++) {
            const uint32_t t = s_warp[wv];
            if (wv < warp) pre += t;
            tot += t;
        }
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int idx = base + tid * 8 + i;
            if (idx < n) wp[idx] = pre;
            pre += v[i];
        }
        carry += tot;
        __syncthreads();
    }
    return carry;
}
// Thread 0, after the scan: the total behind the n prefixes, the remaining status bits, the frame's status and index.
__device__ __forceinline__ void scan_finish(const ScanHead &h, uint32_t *wp, int n, uint32_t total, bool big, int f,
                                           uint32_t *status, uint64_t *indices) {
    wp[n] = total;
    uint32_t st = h.status;
    if (total != h.n64) st |= kStBadWordCount;
    if (big) st |= kStDepthTooBig;
    if (h.room < 8ull * total) st |= kStTruncated;
    status[f] = st;
    if (indices) indices[f] = (uint64_t)ld_le32(h.rec + kRecIndex) | ((uint64_t)ld_le32(h.rec + kRecIndex + 4) << 32);
}

// ---- the task grid of the region and crop decoders (dbde_roi.cu, dbde16.cu), after the pre-pass: one warp == up to 32
// consecutive tile columns of one tile row of a rectangle in one frame, one lane == one tile.  The pre-pass's item i
// covers tiles [32 i, 32 i + 32) in raster order, so a run of consecutive tiles of one tile row has ONE contiguous
// payload run, starting at the item's prefix plus the depths of the item's tiles before the run.  A rectangle narrower
// than 32 tiles gives each tile row a SEGMENT of S lanes (the next power of two >= its width in tiles) and a warp 32 / S
// tile rows, each segment a run of its own.
struct CropGrid {
    const uint8_t *stream;
    const uint64_t *frame_offsets;
    const uint32_t *status;     // from the scan: frames with status != 0 are skipped
    const uint32_t *wprefix;    // nframes * (nitems + 1)
    const int32_t *corners;     // crops: {x0, y0} of crop r of frame f at corners + 2 * (f * corner_stride + r)
    int corner_stride;          // crops: ncrops (per-frame corners) or 0 (shared)
    int x0, y0;                 // region: its corner, the same in every frame
    int W, H, w, h, wh, nitems; // the frame in pixels and tiles, word-prefix items per frame
    int crop_w, crop_h, ncrops; // the rectangles, ncrops per frame
    int nchunks;                // 32-tile column chunks per rectangle
    int seg_shift;              // log2 of the lanes per tile row: 5, or fewer for rectangles narrower than 32 tiles
    int nrg;                    // warps (groups of 32 >> seg_shift tile rows) per chunk and rectangle
    unsigned long long ntasks;  // nframes * ncrops * nrg * nchunks warps
};

// The grid for the scan's frames and ncrops rectangles of crop_w x crop_h per frame that span at most `span` tile columns
// and `nty` tile rows, run by CTAs of `warps` warps: *blocks of them (0: nothing to do), or cudaErrorInvalidConfiguration
// when a launch cannot hold that many.  The caller adds the corners (G.corners, G.corner_stride, or G.x0, G.y0).
template <typename Scan>
cudaError_t crop_grid(CropGrid &G, const Scan &scan, int W, int H, int nitems, int crop_w, int crop_h, int ncrops, int span,
                      int nty, int warps, unsigned *blocks) {
    G = CropGrid();
    G.stream = scan.stream;
    G.frame_offsets = scan.frame_offsets;
    G.status = scan.status;
    G.wprefix = scan.wprefix;
    G.W = W; G.H = H;
    G.w = (W + 7) / 8; G.h = (H + 7) / 8; G.wh = G.w * G.h;
    G.nitems = nitems;
    G.crop_w = crop_w; G.crop_h = crop_h; G.ncrops = ncrops;
    G.nchunks = (span + 31) / 32;
    G.seg_shift = 0;                                          // segments: the next power of two >= the span, <= 32 lanes
    while ((1 << G.seg_shift) < span && G.seg_shift < 5) G.seg_shift++;
    G.nrg = (nty + (32 >> G.seg_shift) - 1) / (32 >> G.seg_shift);
    G.ntasks = (unsigned long long)scan.nframes * (unsigned long long)ncrops * (unsigned long long)G.nrg *
               (unsigned long long)G.nchunks;
    const unsigned long long n = (G.ntasks + warps - 1) / warps;
    if (n > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
    *blocks = (unsigned)n;
    return cudaSuccess;
}

// One lane's part of a task: its segment's rectangle, frame and payload run, and its own tile.
struct CropTask {
    const uint8_t *rec;         // the frame's record
    unsigned long long rect;    // f * ncrops + r: the rectangle's place in the output
    int f, x0, y0, tx0, tx_end; // the frame, the corner, the rectangle's first tile column and one past its last
    int S, seg, sl, rowi;       // lanes per segment, the segment in the warp, this lane in it, its tile row of the rectangle
    int ty, tx, tl;             // this lane's tile: row, column, raster index (0 unless inframe)
    bool live, inframe;         // the tile is in the rectangle / in the rectangle and the frame
    uint32_t k, incl, nwords;   // its depth, the inclusive scan of the segment's depths, the segment's words
    uint32_t wbase;             // the segment's first word in the record's payload
};

// Decodes warp task `task` for this lane; false: no such task, or its frame was rejected by the scan (its rectangles
// stay untouched).  CROPS = false: the rectangle is the region at G.x0, G.y0, inside the frame.  CROPS = true: the
// corner comes from G.corners, and a lane whose tile lies outside the frame is live but not inframe -- depth 0, and a
// segment entirely outside the frame reads nothing of the record.  Warp-wide call.
template <bool CROPS>
__device__ __forceinline__ bool crop_task(const CropGrid &G, unsigned long long task, int lane, CropTask &T) {
    if (task >= G.ntasks) return false;
    // task = ((f * ncrops + r) * nrg + row group) * nchunks + chunk: neighbouring warps read neighbouring payloads
    const int chunk = (int)(task % (unsigned)G.nchunks);
    const unsigned long long fr = task / (unsigned)G.nchunks;
    T.rect = fr / (unsigned)G.nrg;
    const int rg = (int)(fr - T.rect * (unsigned)G.nrg);
    if constexpr (CROPS) {
        T.f = (int)(T.rect / (unsigned)G.ncrops);
        const int r = (int)(T.rect - (unsigned long long)T.f * (unsigned)G.ncrops);
        const int32_t *cp = G.corners + 2 * ((size_t)T.f * (size_t)G.corner_stride + (size_t)r);
        T.x0 = __ldg(cp);
        T.y0 = __ldg(cp + 1);
    } else {
        T.f = (int)T.rect;
        T.x0 = G.x0;
        T.y0 = G.y0;
    }
    if (G.status[T.f] != 0) return false;
    // floor division (negative corners), the far edge in 64 bits (corners up to INT32_MAX)
    T.tx0 = T.x0 >> 3;
    const int ty0 = T.y0 >> 3;
    T.tx_end = (int)(((long long)T.x0 + G.crop_w + 7) >> 3);
    const int nty = (int)(((long long)T.y0 + G.crop_h + 7) >> 3) - ty0;
    T.S = 1 << G.seg_shift;
    T.seg = lane >> G.seg_shift;
    T.sl = lane & (T.S - 1);
    T.rowi = (rg << (5 - G.seg_shift)) + T.seg;
    const bool rowok = T.rowi < nty;
    T.ty = ty0 + T.rowi;
    const int txc = T.tx0 + 32 * chunk;                       // the segment's first tile column
    T.tx = txc + T.sl;
    T.live = rowok && T.tx < T.tx_end;
    // the segment's tiles inside the frame: columns [txa, txb) of tile row ty, one contiguous payload run
    int txa = txc;
    bool segin = rowok;
    T.inframe = T.live;
    if constexpr (CROPS) {
        txa = max(txc, 0);
        const int txb = min(min(txc + T.S, T.tx_end), G.w);
        segin = rowok && T.ty >= 0 && T.ty < G.h && txa < txb;
        T.inframe = T.live && segin && T.tx >= 0 && T.tx < G.w;
    }
    T.rec = G.stream + G.frame_offsets[T.f];
    const int t0 = segin ? T.ty * G.w + txa : 0;              // the run's first raster tile
    const int item = t0 >> 5, rem = t0 & 31;
    T.tl = T.inframe ? T.ty * G.w + T.tx : 0;
    // word offset of tile t0: the item's exclusive prefix plus the depths of the item's tiles before t0
    uint32_t before = 0;
    if (segin)
        for (int j = T.sl; j < rem; j += T.S) before += T.rec[kRecDepth + 32 * item + j];
    for (int o = 1; o < T.S; o <<= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    T.k = T.inframe ? (uint32_t)T.rec[kRecDepth + T.tl] : 0u;
    T.wbase = segin ? G.wprefix[(size_t)T.f * (G.nitems + 1) + item] + before : 0u;
    uint32_t incl = T.k;                                      // inclusive scan of the depths inside the segment
    for (int d = 1; d < T.S; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d, T.S);
        if (T.sl >= d) incl += t;
    }
    T.incl = incl;
    T.nwords = __shfl_sync(0xffffffffu, incl, T.S - 1, T.S);
    return true;
}

// ---- DBDE16, the 16-bit extension (dbde16.cu; SURVEY 8 f-4): partitions of 256 consecutive tiles
struct Enc16Params {
    const uint16_t *frames;     // nframes * W * H u16, tightly packed, device
    uint8_t *out;               // record f at out + f * slot_stride
    uint64_t slot_stride;       // >= rec_bound(wh, 2)
    uint64_t *frame_offsets, *frame_sizes;
    uint64_t *desc;             // nparts look-back descriptors (index f*ppf + q), zeroed
    unsigned int *ticket;       // zeroed
    uint64_t first_index;
    int W, H, w, h, wh, ppf, nframes, aligned;   // aligned: rows can be moved 16 bytes at a time
    unsigned nparts;
};
struct Dec16Params {
    const uint8_t *stream;
    uint64_t stream_bytes;
    const uint64_t *frame_offsets;
    uint16_t *frames;
    uint32_t *status;
    uint64_t *indices;          // or null
    uint32_t *wprefix;          // nframes * (ceil(wh/32) + 1) exclusive word prefixes per 32-tile group
    int W, H, w, h, wh, ppf, nframes, aligned;
    unsigned nparts;
};
// DBDE16 crop encode (dbde16.cu): record j = f * ncrops + r is the DBDE16 record of the crop_w x crop_h image at corner
// r of frame f (pixels outside the frame are pad), at out + j * slot_stride.
struct Enc16CropParams {
    const uint16_t *frames;     // nframes * W * H u16, tightly packed, device, 2-byte aligned
    int W, H;
    const int32_t *corners;     // {x0, y0} of crop r of frame f at corners + 2 * (f * corner_stride + r), any int32 values
    int ncrops, corner_stride;  // corner_stride: ncrops (per-frame corners) or 0 (shared)
    int crop_w, crop_h, w, wh;  // the crop in pixels, its tile columns and tiles
    uint32_t pad;               // 0..65535
    uint8_t *out;
    uint64_t slot_stride;       // >= rec_bound(wh, 2)
    uint64_t *frame_offsets;    // nrec entries (= j * slot_stride), device
    uint64_t *frame_sizes;      // nrec entries (record bytes), device
    uint64_t first_index;
    int nrec;                   // nframes * ncrops
};
cudaError_t launch_encode16(const Enc16Params &P, int num_sms, cudaStream_t stream);
cudaError_t launch_encode16_crops(const Enc16CropParams &P, int num_sms, cudaStream_t stream);
cudaError_t launch_decode16_scan(const Dec16Params &P, cudaStream_t stream);
cudaError_t launch_decode16(const Dec16Params &P, int num_sms, cudaStream_t stream);
// DBDE16 crop decode (dbde16.cu), after launch_decode16_scan(scan): ncrops rectangles of crop_w x crop_h per frame with
// top-left corners {x0, y0} at corners (device; per_frame: nframes * ncrops pairs, else ncrops pairs for every frame),
// any int32 values; pixels outside the frame are `pad`.  Crop r of frame f goes to out + (f * ncrops + r) * crop_w *
// crop_h U16.  Frames the scan rejected stay untouched.
cudaError_t launch_decode16_crops(const Dec16Params &scan, const int32_t *corners, int ncrops, bool per_frame, int crop_w,
                                  int crop_h, int pad, uint16_t *out, cudaStream_t stream);
// DBDE16 binned decode (dbde16.cu), after launch_decode16_scan(scan): every frame reduced to the rounded means of its
// factor x factor blocks (factor 2, 4 or 8), ceil(H / factor) rows of ceil(W / factor) U16 per frame, tightly packed
// from `out`.  Frames the scan rejected stay untouched.
cudaError_t launch_decode16_binned(const Dec16Params &scan, int factor, uint16_t *out, int num_sms, cudaStream_t stream);

// The persistent kernels' launch configuration (dynamic shared memory opt-in + resident CTAs per SM) is a
// property of (device, kernel, shared-memory size): looked up once and remembered, because the two runtime
// calls cost as much as the launch itself when a caller encodes one frame per call.
cudaError_t cached_occupancy(const void *kernel, int threads, size_t smem, int *occ);

// A persistent grid: as many CTAs as are resident at once, at most one per work item.
template <typename Kern, typename Params>
cudaError_t launch_persistent(Kern kern, const Params &P, unsigned work, int threads, size_t smem, int num_sms, cudaStream_t stream) {
    int occ = 0;
    cudaError_t e = cached_occupancy((const void *)kern, threads, smem, &occ);
    if (e != cudaSuccess) return e;
    unsigned grid = (unsigned)(num_sms * occ);
    if (grid > work) grid = work;
    if (grid == 0) return cudaSuccess;
    kern<<<grid, threads, smem, stream>>>(P);
    return cudaGetLastError();
}

size_t enc_smem_bytes(const PartGeom &g);
size_t dec_smem_bytes(const PartGeom &g);
cudaError_t launch_encode(const EncParams &P, bool fast, int num_sms, cudaStream_t stream);
cudaError_t launch_compact(const uint8_t *slots, uint64_t slot_stride, const uint64_t *sizes, int n, uint8_t *dst,
                           cudaStream_t stream);
cudaError_t launch_encode_crops(const EncCropParams &P, int num_sms, cudaStream_t stream);
// launch_compact for batches of thousands of records (crop encodes): the exclusive prefix of the sizes is computed
// once into prefix (n + 1 entries, device; prefix[n] = the total), then the records are copied by a grid of at most
// 65535 record rows.
cudaError_t launch_compact_prefixed(const uint8_t *slots, uint64_t slot_stride, const uint64_t *sizes, uint64_t *prefix, int n,
                                    uint8_t *dst, cudaStream_t stream);
cudaError_t launch_decode_scan(const DecParams &P, cudaStream_t stream);
cudaError_t launch_decode(const DecParams &P, bool fast, int num_sms, cudaStream_t stream);
// Region-of-interest decode (dbde_roi.cu): the rectangle [x0, x0 + roi_w) x [y0, y0 + roi_h) of every frame into
// `out` (nframes * roi_w * roi_h bytes, tightly packed, any alignment), after launch_decode_scan(scan) with
// scan.g = linear_geom(W, H) (word prefixes per 32 consecutive tiles).  Frames the scan rejected stay untouched.
cudaError_t launch_decode_roi(const DecParams &scan, int x0, int y0, int roi_w, int roi_h, uint8_t *out, cudaStream_t stream);
// Crop decode (dbde_roi.cu, the same kernel body): ncrops rectangles of crop_w x crop_h per frame with top-left
// corners {x0, y0} at corners (device; per_frame: nframes * ncrops pairs, else ncrops pairs for every frame), any
// int32 values; pixels outside the frame are `pad`.  Crop r of frame f goes to out + (f * ncrops + r) * crop_w * crop_h.
// Same scan as launch_decode_roi; frames the scan rejected stay untouched.
cudaError_t launch_decode_crops(const DecParams &scan, const int32_t *corners, int ncrops, bool per_frame, int crop_w, int crop_h,
                                int pad, uint8_t *out, cudaStream_t stream);
// Binned decode (dbde_decode.cu): every frame reduced to the rounded means of its factor x factor blocks (factor 2, 4
// or 8), ceil(H / factor) rows of ceil(W / factor) bytes per frame, tightly packed from `out`, any alignment.  Same
// scan as launch_decode_roi; frames the scan rejected stay untouched.
cudaError_t launch_decode_binned(const DecParams &scan, int factor, uint8_t *out, int num_sms, cudaStream_t stream);

}  // namespace dbde
