// Internal interface between the C ABI (dbde_capi.cu) and the kernels.
#pragma once
#include "dbde_device.cuh"

namespace dbde {

struct EncParams {
    PartGeom g;
    const uint8_t *frames;      // nframes * W * H, tightly packed, device
    uint8_t *out;               // slot of frame record 0, device; record f lives at out + f * slot_stride
    uint64_t slot_stride;       // bytes between consecutive frame slots (>= 32 + 66*wh)
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
    uint64_t slot_stride;       // >= 32 + 66 * wh
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

// ---- DBDE16, the 16-bit extension (dbde16.cu; SURVEY 8 f-4): partitions of 256 consecutive tiles
struct Enc16Params {
    const uint16_t *frames;     // nframes * W * H u16, tightly packed, device
    uint8_t *out;               // record f at out + f * slot_stride
    uint64_t slot_stride;       // >= 32 + 131 * wh
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
    uint64_t slot_stride;       // >= 32 + 131 * wh
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
