/* dbde_b200.h -- the C ABI of the B200-native DBDE frame codec.
 *
 * This is the thin extern "C" layer beneath the reference's C++ entry points
 * (include/dbde_util.h mirrors /root/reference/dbde_util.h:21-52 and forwards here).
 * Plain pointers and sizes only.  Every entry point names the reference interface it replaces.
 *
 * On-disk layout (unchanged; README.md:27-67 of the reference, dbde_util.cpp:137-209):
 *   file         := video_header(28) frame_record*
 *   frame_record := I32 2 | U64 index | F64 0.0 | I32 wh | U8 depth[wh] | I32 wh | U8 min[wh]
 *                   | I32 n64 | U64 words[n64]                      (w=ceil(W/8), h=ceil(H/8), wh=w*h)
 * A "stream" below is a byte buffer holding frame records plus a table of their offsets; records
 * laid back to back are the file minus its 28-byte header.  The device encoder writes each record
 * into its own fixed-stride SLOT (frames are independent, dbde_util.cpp:146 zeroes n64 per frame);
 * the host entry points concatenate the slots back to back while copying them off the GPU.
 *
 * All functions return 0 on success or a negative dbde_b200_error / positive cudaError_t value;
 * dbde_b200_last_error() describes the last failure on the calling thread.  There is NO CPU
 * fallback: without a CUDA device of compute capability 10.x every call fails loudly.
 *
 * Environment (all optional; read once unless noted):
 *   DBDE_B200_DEVICE          device the C++ drop-in functions use (default 0)
 *   DBDE_B200_SLOTS           staging slots in flight on the host path, 2..8 (default 3)
 *   DBDE_B200_CHUNK_FRAMES    frames per staged chunk (default: 64 MiB of pixels)
 *   DBDE_B200_COPY_THREADS    size of the pool that relays pageable buffers (default min(6, cores/2 - 1))
 *   DBDE_B200_COPY_CROWD      calling threads helping at once from which the pool stands back (default cores/2)
 *   DBDE_B200_H2D_DMA_KB / DBDE_B200_D2H_DMA_KB   smallest DMA on the pageable path (default 1024)
 *   DBDE_B200_H2D_STREAMING=0 ordinary instead of streaming stores into the bounce buffers
 *   DBDE_B200_PROFILE=1       per-thread phase times of the host path on stderr when a thread ends
 *   measurement switches, read per call: DBDE_B200_ODD_DECODE=staged|direct (odd-size unpack kernel),
 *   DBDE_B200_NO_LINEAR=1 (band-aligned partitions for every aligned frame)
 */
#ifndef DBDE_B200_H
#define DBDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBDE_B200_API __attribute__((visibility("default")))

typedef struct dbde_b200_ctx dbde_b200_ctx;

enum dbde_b200_error {
    DBDE_B200_OK = 0,
    DBDE_B200_E_INVALID = -1,      /* bad argument */
    DBDE_B200_E_NO_DEVICE = -2,    /* no sm_100 device / CUDA runtime unusable */
    DBDE_B200_E_CAPACITY = -3,     /* output buffer too small */
    DBDE_B200_E_NOMEM = -4
};

/* per-frame decode status bits (0 = decoded); mirrors the reject paths of dbde_unpack_image /
 * dbde_unpack_frame(_header), dbde_util.cpp:296,299,303,335 */
#define DBDE_B200_ST_BAD_FRAME_HEADER 1u
#define DBDE_B200_ST_BAD_DEPTH_COUNT 2u
#define DBDE_B200_ST_BAD_MIN_COUNT 4u
#define DBDE_B200_ST_BAD_WORD_COUNT 8u
#define DBDE_B200_ST_DEPTH_TOO_BIG 16u   /* depth byte > 8: unpinned in the reference, rejected here */
#define DBDE_B200_ST_TRUNCATED 32u

/* ---- lifetime ------------------------------------------------------------------------------ */
/* One context per GPU and per host thread (contexts are not thread-safe; distinct contexts are). */
DBDE_B200_API int dbde_b200_create(int device, dbde_b200_ctx **out);
DBDE_B200_API void dbde_b200_destroy(dbde_b200_ctx *ctx);
DBDE_B200_API const char *dbde_b200_last_error(void);
DBDE_B200_API int dbde_b200_device_count(void);

/* ---- sizes (pure host arithmetic) ------------------------------------------------------------ */
/* worst-case bytes of one frame record, 32 + 66*wh  (the `target` contract of dbde_pack_frame,
 * dbde_util.h:26, which has no capacity argument) */
DBDE_B200_API size_t dbde_b200_frame_record_bound(int W, int H);
/* default distance between the per-frame slots the device encoder writes: the record bound
 * rounded up to 16 bytes */
DBDE_B200_API size_t dbde_b200_slot_stride(int W, int H);
/* bytes a stream buffer for n frames must hold: n * slot_stride + 16 bytes of tail slack */
DBDE_B200_API size_t dbde_b200_stream_bound(int W, int H, int nframes);

/* ---- device memory / pinned host memory helpers ---------------------------------------------- */
/* cudaMalloc on the context's device; the block is 256-byte aligned and 16-byte tail-padded so
 * the kernels' 16-byte-aligned bulk copies may touch the aligned hull of any sub-range. */
DBDE_B200_API int dbde_b200_device_alloc(dbde_b200_ctx *ctx, size_t bytes, void **out);
DBDE_B200_API int dbde_b200_device_free(dbde_b200_ctx *ctx, void *p);
DBDE_B200_API int dbde_b200_host_alloc(size_t bytes, void **out);        /* pinned */
DBDE_B200_API int dbde_b200_host_free(void *p);
/* Page-lock / release memory the caller already owns (a malloc'd frame buffer, a `target` array): the
 * host entry points -- and the C++ drop-in functions of dbde_util.h -- then move it by DMA (~55 GB/s)
 * instead of through pageable staging (~15 GB/s).  Unregister before freeing the memory. */
DBDE_B200_API int dbde_b200_host_register(void *p, size_t bytes);
DBDE_B200_API int dbde_b200_host_unregister(void *p);
DBDE_B200_API int dbde_b200_memcpy_h2d(dbde_b200_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
DBDE_B200_API int dbde_b200_memcpy_d2h(dbde_b200_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);

/* ---- the hot path, device-resident ---------------------------------------------------------- */
/* Batched dbde_pack_frame (dbde_util.cpp:190-196, which calls dbde_pack_image :137-180):
 * encodes frames first_index .. first_index+nframes-1.  Record i is written at
 * out_dev + i * slot_stride (slot_stride 0 = dbde_b200_slot_stride(W, H)) and is byte-identical
 * to what dbde_pack_frame writes; frame_offsets_dev[i] receives i * slot_stride and
 * frame_sizes_dev[i] the record's size (nframes entries each).  frames_dev: nframes*W*H bytes,
 * tightly packed rows (stride = W), as the reference's `image` argument.  Asynchronous on
 * `stream` (a cudaStream_t, NULL = default).  out_capacity must be >= nframes * slot_stride.
 * Fastest when (out_dev + 32 + 2*wh) is 16-byte aligned (U64 words land on 16-byte boundaries).
 * Streams: the scan scratch a launch needs (ticket + look-back descriptors here, word prefixes in
 * decode_device) is kept PER STREAM inside the context, so calls queued on different streams of one
 * context may overlap on the device; calls on one stream are ordered by the stream.  The context
 * itself is still driven by one host thread at a time. */
DBDE_B200_API int dbde_b200_encode_device(dbde_b200_ctx *ctx, const uint8_t *frames_dev, int W, int H,
                                          uint64_t first_index, int nframes, uint8_t *out_dev,
                                          size_t out_capacity, size_t slot_stride, uint64_t *frame_offsets_dev,
                                          uint64_t *frame_sizes_dev, void *stream);

/* Batched dbde_unpack_frame (dbde_util.cpp:339-345 -> dbde_unpack_image :291-328): decodes the
 * nframes records found at stream_dev + frame_offsets_dev[i] into frames_dev (nframes*W*H).
 * status_dev[i] = 0 or DBDE_B200_ST_* bits; a rejected frame's image is left untouched, as in the
 * reference.  indices_dev (may be NULL) receives each record's frame index. */
DBDE_B200_API int dbde_b200_decode_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                          const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                          uint8_t *frames_dev, uint32_t *status_dev, uint64_t *indices_dev,
                                          void *stream);

/* ---- the hot path, host buffers (H2D + kernels + D2H inside the call) ------------------------ */
/* Same codec with HOST pointers (pinned memory from dbde_b200_host_alloc streams fastest;
 * pageable memory works).  Frames are processed in chunks through triple-buffered device staging
 * so copies and kernels overlap.  encode_host lays the records BACK TO BACK in out_host (what a
 * writer appends to the file after the video header) and fills frame_offsets_host[0..nframes]
 * (record starts; the last entry is the total size).  Synchronous: results are in host memory
 * on return, like the reference's calls. */
DBDE_B200_API int dbde_b200_encode_host(dbde_b200_ctx *ctx, const uint8_t *frames_host, int W, int H,
                                        uint64_t first_index, int nframes, uint8_t *out_host,
                                        size_t out_capacity, uint64_t *frame_offsets_host);
DBDE_B200_API int dbde_b200_decode_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                        const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                        uint8_t *frames_host, uint32_t *status_host, uint64_t *indices_host);

/* ---- multi-GPU: contiguous frame ranges, one host thread per context, host-side concatenation -- */
/* Frames carry no inter-frame state (dbde_util.cpp:146), so a long video shards by frame range with
 * no device-to-device traffic and no collective.  encode: the batch is cut into contiguous ranges of
 * one staging chunk each, range i goes to context i mod G, every context streams its ranges over
 * its own PCIe link, and the ranges' records are placed in stream order as their sizes become
 * known (an exclusive prefix sum over range byte counts, taken on the host as the ranges finish).
 * decode: context g takes frames [g*n/G, (g+1)*n/G).  Output is byte-identical to the one-GPU calls.
 * Each ctxs[g] must be a distinct context (they may share a device); out_capacity must be
 * >= dbde_b200_stream_bound(W, H, nframes). */
DBDE_B200_API int dbde_b200_encode_host_sharded(dbde_b200_ctx **ctxs, int nctx, const uint8_t *frames_host, int W,
                                                int H, uint64_t first_index, int nframes, uint8_t *out_host,
                                                size_t out_capacity, uint64_t *frame_offsets_host);
DBDE_B200_API int dbde_b200_decode_host_sharded(dbde_b200_ctx **ctxs, int nctx, const uint8_t *stream_host,
                                                size_t stream_bytes, const uint64_t *frame_offsets_host, int W,
                                                int H, int nframes, uint8_t *frames_host, uint32_t *status_host,
                                                uint64_t *indices_host);

/* Host-side frame indexer (the pointer chase dbde_walk_a_file does implicitly, dbde_util.cpp:408-421;
 * next = cur + 32 + 2wh + 8*n64).  Fills up to max_frames+1 offsets; returns the frame count or < 0. */
DBDE_B200_API long dbde_b200_index_stream(const uint8_t *stream_host, size_t stream_bytes, int W, int H,
                                          uint64_t *frame_offsets, long max_frames);

/* Optional GPU validation for the indexer (SURVEY.md 8 f-2): every check dbde_unpack_image makes before
 * it touches the image (dbde_util.cpp:295-303: nb == wh, nm == wh, sum(depth) == n64), plus the frame
 * tag (:335), depth <= 8 and bounds, for each record -- status[i] = 0 or DBDE_B200_ST_* bits exactly as
 * the decoders report them -- without decoding a pixel.  indices (may be NULL) receives the frame
 * indices.  _device: stream and outputs in device memory, asynchronous on `stream`; _host: host memory,
 * synchronous (the records cross PCIe once, 4 (+8) bytes per frame come back). */
DBDE_B200_API int dbde_b200_validate_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                            const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                            uint32_t *status_dev, uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_validate_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                          const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                          uint32_t *status_host, uint64_t *indices_host);

/* ---- region of interest: one rectangle of every frame ------------------------------------------------
 * dbde_unpack_frame (dbde_util.cpp:339-345 -> dbde_unpack_image :291-328) followed by a crop, without
 * decoding the rest of the frame: roi_out receives nframes * roi_h * roi_w bytes, tightly packed, frame i
 * at roi_out + i * roi_w * roi_h, byte for byte image_i[y0 .. y0+roi_h-1][x0 .. x0+roi_w-1] of the full
 * decode.  The region must satisfy 0 <= x0, 0 <= y0, roi_w >= 1, roi_h >= 1, x0 + roi_w <= W and
 * y0 + roi_h <= H, else DBDE_B200_E_INVALID before any work is queued.  Validation covers the WHOLE record
 * (dbde_util.cpp:295-303, 335 plus depth <= 8 and bounds): status and indices are exactly what
 * dbde_b200_decode_device reports for the same records, a record damaged outside the region is rejected
 * too, and a rejected frame's region of the output is left untouched.  roi_out may have any alignment and
 * nothing outside [roi_out, roi_out + nframes * roi_w * roi_h) is written.  Follows the context's
 * DBDE_INVERT_ENDIAN setting.  A region equal to the frame is dbde_b200_decode_device.
 * _device: asynchronous on `stream`, with decode_device's per-stream scratch.  _host: the chunk pipeline of
 * dbde_b200_decode_host (staging slots in flight, pageable buffers relayed, only accepted frames copied
 * out); records still cross PCIe whole, only the region's pixels come back. */
DBDE_B200_API int dbde_b200_decode_roi_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                              const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                              int x0, int y0, int roi_w, int roi_h, uint8_t *roi_dev,
                                              uint32_t *status_dev, uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_decode_roi_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                            const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                            int x0, int y0, int roi_w, int roi_h, uint8_t *roi_host,
                                            uint32_t *status_host, uint64_t *indices_host);

/* ---- crops: N fixed-size windows of every frame, anywhere, padded outside the frame ---------------------------
 * Many rectangles of crop_w x crop_h per frame in one call -- the wells of a plate, a window that follows an animal
 * from frame to frame, animal-centred windows that run past the frame's edge -- without decoding the rest of the
 * frame.  corners: {x0, y0} int32 pairs, the top-left corner of each crop; any values, including negative ones and
 * ones past the frame.  corners_per_frame = 0: ncrops pairs used for every frame; 1: nframes * ncrops pairs, frame
 * f's crops at corners + 2 * f * ncrops.  Crop r of frame f goes to crops + ((size_t)f * ncrops + r) * crop_w *
 * crop_h: crop_h rows of crop_w bytes, tightly packed, any alignment.  Pixel (x, y) of a crop is
 * image[y0 + y][x0 + x] of the full decode where that lies inside the frame, and `pad` elsewhere; a crop entirely
 * outside the frame is all `pad` and reads nothing of the record.  Validation covers the WHOLE record: status and
 * indices are exactly what dbde_b200_decode_device reports for the same records, a record damaged outside every
 * crop is rejected too, and all crops of a rejected frame are left untouched.  Nothing outside
 * [crops, crops + nframes * ncrops * crop_w * crop_h) is written.  Follows the context's DBDE_INVERT_ENDIAN setting
 * (a tile row is byte-reversed before the columns past W are set to `pad`; pad bytes are never reversed).
 * DBDE_B200_E_INVALID before any work is queued for: NULL pointers (when nframes > 0), ncrops < 1, crop_w or
 * crop_h < 1, a crop size the frame limits reject, ncrops * crop_w * crop_h > 2^31 - 1, corners_per_frame not 0 or
 * 1, pad outside 0..255.  nframes == 0 returns 0.
 * _device: corners in device memory (a tracker on the GPU can feed its positions straight in), asynchronous on
 * `stream`.  _host: host memory, the chunk pipeline of dbde_b200_decode_host (records still cross PCIe whole, only
 * the accepted frames' crops come back; a chunk's corners go up with it). */
DBDE_B200_API int dbde_b200_decode_crops_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                                const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                                const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                                int crop_h, int pad, uint8_t *crops_dev, uint32_t *status_dev,
                                                uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_decode_crops_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                              const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                              const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                              int crop_h, int pad, uint8_t *crops_host, uint32_t *status_host,
                                              uint64_t *indices_host);

/* ---- crop encoding: N fixed-size windows of every frame, each recorded as a frame of its own ---------------------
 * Records only the wells of a plate or a window that follows an animal instead of the whole sensor, without first
 * gathering the windows into frames of their own.  The crop image is exactly what dbde_b200_decode_crops_* returns
 * for the same arguments: corners are {x0, y0} int32 pairs, any values; corners_per_frame = 0: ncrops pairs for
 * every frame, 1: nframes * ncrops pairs, frame f's at corners + 2 * f * ncrops; pixel (x, y) is frame[y0 + y][x0 + x]
 * inside the frame and `pad` (0..255) outside it.  Record j = f * ncrops + r is byte for byte dbde_pack_frame(
 * first_index + f, crop image (f, r), crop_w, crop_h): the reference's record of a crop_w x crop_h frame, so the
 * records of one crop, in frame order behind a video header of crop_h x crop_w, are a .dbde video the reference's
 * walker reads, and every crop keeps the source frame's index.  The clamp padding of the crop's partial last tile
 * column and row repeats the crop image's last valid pixel, which may be `pad`.  Follows the context's
 * DBDE_INVERT_ENDIAN setting (tile rows are reversed after the crop image is assembled).  frames: nframes * W * H
 * bytes, tightly packed, any alignment; the only frame bytes read are in aligned 8-byte words that hold in-frame
 * pixels of some crop, and a crop entirely outside the frame reads none.
 * DBDE_B200_E_INVALID before any work is queued for: NULL pointers (when nframes > 0), the crop arguments
 * dbde_b200_decode_crops_* rejects, frame dimensions the frame limits reject, a slot_stride below
 * dbde_b200_frame_record_bound(crop_w, crop_h) (device form), and nframes * ncrops > 2^31 - 1.
 * DBDE_B200_E_CAPACITY for out_capacity < nframes * ncrops * slot_stride (device form) or less than the records'
 * total (host form).  nframes == 0 returns 0 (the host form writes frame_offsets_host[0] = 0).
 * _device: record j at out_dev + j * slot_stride (slot_stride 0 = dbde_b200_slot_stride(crop_w, crop_h));
 * frame_offsets_dev[j] = j * slot_stride and frame_sizes_dev[j] = the record's size, nframes * ncrops entries each;
 * nothing outside [out_dev, out_dev + nframes * ncrops * slot_stride) is written.  Corners in device memory (a
 * tracker on the GPU can feed its positions straight in); asynchronous on `stream`.  One CTA encodes one record, so
 * a batch of fewer records than the GPU holds CTAs (a few large crops) does not fill the GPU.
 * _host: the chunk pipeline of dbde_b200_encode_host, pinned or pageable buffers, synchronous; the records back to
 * back in the same order, frame_offsets_host[0 .. nframes * ncrops] (the last entry is the total size). */
DBDE_B200_API int dbde_b200_encode_crops_device(dbde_b200_ctx *ctx, const uint8_t *frames_dev, int W, int H,
                                                uint64_t first_index, int nframes, const int32_t *corners_dev, int ncrops,
                                                int corners_per_frame, int crop_w, int crop_h, int pad, uint8_t *out_dev,
                                                size_t out_capacity, size_t slot_stride, uint64_t *frame_offsets_dev,
                                                uint64_t *frame_sizes_dev, void *stream);
DBDE_B200_API int dbde_b200_encode_crops_host(dbde_b200_ctx *ctx, const uint8_t *frames_host, int W, int H,
                                              uint64_t first_index, int nframes, const int32_t *corners_host, int ncrops,
                                              int corners_per_frame, int crop_w, int crop_h, int pad, uint8_t *out_host,
                                              size_t out_capacity, uint64_t *frame_offsets_host);

/* ---- binned: every frame at 1/2, 1/4 or 1/8 of its size, as block means ---------------------------------------
 * The whole field of view at lower resolution -- a tracker on a quarter-size image, previews, motion energy over a
 * plate, a network that takes downsampled frames -- without writing the full-size frame anywhere.  factor must be
 * 1, 2, 4 or 8; factor 1 is dbde_b200_decode_device.  Frame i's output is Hb = ceil(H / factor) rows of
 * Wb = ceil(W / factor) bytes, tightly packed, at out + i * Wb * Hb; any alignment, and nothing outside
 * [out, out + nframes * Wb * Hb) is written.  Output pixel (X, Y) is the mean of the IN-FRAME pixels of the full
 * decode in [factor X, factor X + factor) x [factor Y, factor Y + factor), rounded half up: (sum + n / 2) / n in
 * integers, n the number of in-frame pixels (factor^2 except in the last column when W % factor != 0 and the last row
 * when H % factor != 0).  "The full decode" follows the context's DBDE_INVERT_ENDIAN setting.  Validation covers the
 * WHOLE record: status and indices are exactly what dbde_b200_decode_device reports for the same records, and a
 * rejected frame's output is left untouched.  DBDE_B200_E_INVALID before any work is queued for: NULL pointers (when
 * nframes > 0), a factor other than 1, 2, 4 or 8, frame dimensions the frame limits reject.  nframes == 0 returns 0.
 * _device: asynchronous on `stream`.  _host: the chunk pipeline of dbde_b200_decode_host (records still cross PCIe
 * whole, only the accepted frames' binned pixels come back). */
DBDE_B200_API int dbde_b200_decode_binned_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                                 const uint64_t *frame_offsets_dev, int W, int H, int nframes, int factor,
                                                 uint8_t *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_decode_binned_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                               const uint64_t *frame_offsets_host, int W, int H, int nframes, int factor,
                                               uint8_t *out_host, uint32_t *status_host, uint64_t *indices_host);

/* ---- DBDE16: 16-bit frames (SURVEY.md 8 f-4) -------------------------------------------------------
 * The extension the format note hints at (reference README.md:65, "could expand size to handle higher
 * bit depth images").  NOT in the reference code: the layout is defined here and restated by the test oracle
 * ("DBDE16"): the reference's frame record with depths 0..16 and a two-byte little-endian minimum per tile,
 *   I32 2 | U64 index | F64 0.0 | I32 wh | U8 depth[wh] | I32 2*wh | U16 min[wh] | I32 n64 | U64 words[n64]
 * (a reader tells the layouts apart by the minimum plane's length).  A frame whose pixels fit in 8 bits
 * gets exactly the 8-bit codec's depth plane and words.  Same conventions as the 8-bit entry points;
 * frames are W*H U16 per frame, tightly packed; fastest when W % 8 == 0 and the frame buffer is 16-byte
 * aligned.  The host forms share the 8-bit entry points' chunk pipeline (staging slots in flight, pageable
 * buffers relayed through pinned bounce buffers). */
DBDE_B200_API size_t dbde_b200_frame_record_bound16(int W, int H);    /* 32 + 131*wh */
DBDE_B200_API size_t dbde_b200_slot_stride16(int W, int H);
DBDE_B200_API int dbde_b200_encode16_device(dbde_b200_ctx *ctx, const uint16_t *frames_dev, int W, int H,
                                            uint64_t first_index, int nframes, uint8_t *out_dev, size_t out_capacity,
                                            size_t slot_stride, uint64_t *frame_offsets_dev, uint64_t *frame_sizes_dev,
                                            void *stream);
DBDE_B200_API int dbde_b200_decode16_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                            const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                            uint16_t *frames_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_encode16_host(dbde_b200_ctx *ctx, const uint16_t *frames_host, int W, int H,
                                          uint64_t first_index, int nframes, uint8_t *out_host, size_t out_capacity,
                                          uint64_t *frame_offsets_host);
/* the indexer for DBDE16 streams: next = cur + 32 + 3wh + 8*n64 */
DBDE_B200_API long dbde_b200_index_stream16(const uint8_t *stream_host, size_t stream_bytes, int W, int H,
                                            uint64_t *frame_offsets, long max_frames);
DBDE_B200_API int dbde_b200_decode16_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                          const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                          uint16_t *frames_host, uint32_t *status_host, uint64_t *indices_host);

/* ---- DBDE16 crops: N fixed-size windows of every 16-bit frame, anywhere, padded outside the frame ---------------
 * dbde_b200_decode_crops_* for DBDE16 records: the wells of a plate, a tracked window or animal-centred windows from
 * a scientific camera's frames without decoding the rest of each frame.  corners, corners_per_frame and the output
 * layout are those of dbde_b200_decode_crops_*, counted in U16 pixels: crop r of frame f goes to crops +
 * ((size_t)f * ncrops + r) * crop_w * crop_h, crop_h rows of crop_w U16, tightly packed.  Pixel (x, y) of a crop is
 * image[y0 + y][x0 + x] of dbde_b200_decode16_device's image where that lies inside the frame, and `pad` elsewhere; a
 * crop entirely outside the frame is all `pad` and reads nothing of the record.  A region of interest is one crop
 * with a shared corner inside the frame.  Validation covers the WHOLE record: status and indices are exactly what
 * dbde_b200_decode16_device reports for the same records, a record damaged outside every crop is rejected too, and
 * all crops of a rejected frame are left untouched.  Nothing outside [crops, crops + nframes * ncrops * crop_w *
 * crop_h * 2 bytes) is written.  Like dbde_b200_decode16_device, these ignore the context's DBDE_INVERT_ENDIAN
 * setting: DBDE16 has no such variant.  DBDE_B200_E_INVALID before any work is queued for: NULL pointers (when
 * nframes > 0), an output pointer that is not 2-byte aligned (any even address works), ncrops < 1, crop_w or crop_h
 * < 1, a crop size the frame limits reject, ncrops * crop_w * crop_h > 2^31 - 1 pixels, corners_per_frame not 0 or 1,
 * pad outside 0..65535.  nframes == 0 returns 0.
 * _device: corners in device memory, asynchronous on `stream`.  _host: host memory, the chunk pipeline of
 * dbde_b200_decode16_host (records still cross PCIe whole, only the accepted frames' crops come back). */
DBDE_B200_API int dbde_b200_decode16_crops_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                                  const uint64_t *frame_offsets_dev, int W, int H, int nframes,
                                                  const int32_t *corners_dev, int ncrops, int corners_per_frame, int crop_w,
                                                  int crop_h, int pad, uint16_t *crops_dev, uint32_t *status_dev,
                                                  uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_decode16_crops_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                                const uint64_t *frame_offsets_host, int W, int H, int nframes,
                                                const int32_t *corners_host, int ncrops, int corners_per_frame, int crop_w,
                                                int crop_h, int pad, uint16_t *crops_host, uint32_t *status_host,
                                                uint64_t *indices_host);

/* ---- DBDE16 crop encoding: N fixed-size windows of every 16-bit frame, each recorded as a frame of its own ----------
 * dbde_b200_encode_crops_* for 16-bit frames: records only the wells of a plate or a window that follows an animal
 * instead of the whole sensor, without first gathering the windows into frames of their own.  Arguments and semantics
 * are those of dbde_b200_encode_crops_*, with pixels counted as U16.  The crop image is exactly what
 * dbde_b200_decode16_crops_* returns for the same arguments: corners are {x0, y0} int32 pairs, any values;
 * corners_per_frame = 0: ncrops pairs for every frame, 1: nframes * ncrops pairs, frame f's at corners + 2 * f * ncrops;
 * pixel (x, y) is frame[y0 + y][x0 + x] inside the frame and `pad` (0..65535) outside it.  Record j = f * ncrops + r is
 * byte for byte the DBDE16 record of the crop_w x crop_h crop image (f, r) with frame index first_index + f:
 *   I32 2 | U64 index | F64 0.0 | I32 wh | U8 depth[wh] | I32 2*wh | U16 min[wh] | I32 n64 | U64 words[n64]
 * The clamp padding of the crop's partial last tile column and row repeats the crop image's last valid pixel, which may
 * be `pad`.  Like every DBDE16 call, these ignore the context's DBDE_INVERT_ENDIAN setting: DBDE16 has no such
 * variant.  frames: nframes * W * H U16, tightly packed, 2-byte aligned; the only frame bytes read are in aligned
 * 16-byte words that hold in-frame pixels of some crop, and a crop entirely outside the frame reads none.
 * DBDE_B200_E_INVALID before any work is queued for: NULL pointers (when nframes > 0), a frame pointer that is not
 * 2-byte aligned (device form), the crop arguments dbde_b200_decode16_crops_* rejects, frame dimensions the frame limits
 * reject, a slot_stride below dbde_b200_frame_record_bound16(crop_w, crop_h) (device form), and nframes * ncrops >
 * 2^31 - 1.  DBDE_B200_E_CAPACITY for out_capacity < nframes * ncrops * slot_stride (device form) or less than the
 * records' total (host form).  nframes == 0 returns 0 (the host form writes frame_offsets_host[0] = 0).
 * _device: record j at out_dev + j * slot_stride (slot_stride 0 = dbde_b200_slot_stride16(crop_w, crop_h));
 * frame_offsets_dev[j] = j * slot_stride and frame_sizes_dev[j] = the record's size, nframes * ncrops entries each;
 * nothing outside [out_dev, out_dev + nframes * ncrops * slot_stride) is written, nor anything between a record's end
 * and its slot's end.  Corners in device memory; asynchronous on `stream`; one kernel launch and nothing else (no
 * scratch, no memset).  One CTA encodes one record, so a batch of fewer records than the GPU holds CTAs does not
 * fill the GPU.
 * _host: the chunk pipeline of dbde_b200_encode16_host, pinned or pageable buffers, synchronous; the records back to
 * back in the same order, frame_offsets_host[0 .. nframes * ncrops] (the last entry is the total size). */
DBDE_B200_API int dbde_b200_encode16_crops_device(dbde_b200_ctx *ctx, const uint16_t *frames_dev, int W, int H,
                                                  uint64_t first_index, int nframes, const int32_t *corners_dev, int ncrops,
                                                  int corners_per_frame, int crop_w, int crop_h, int pad, uint8_t *out_dev,
                                                  size_t out_capacity, size_t slot_stride, uint64_t *frame_offsets_dev,
                                                  uint64_t *frame_sizes_dev, void *stream);
DBDE_B200_API int dbde_b200_encode16_crops_host(dbde_b200_ctx *ctx, const uint16_t *frames_host, int W, int H,
                                                uint64_t first_index, int nframes, const int32_t *corners_host, int ncrops,
                                                int corners_per_frame, int crop_w, int crop_h, int pad, uint8_t *out_host,
                                                size_t out_capacity, uint64_t *frame_offsets_host);

/* ---- DBDE16 binned: every 16-bit frame at 1/2, 1/4 or 1/8 of its size, as block means -----------------------------
 * dbde_b200_decode_binned_* for DBDE16 records.  factor must be 1, 2, 4 or 8; factor 1 is dbde_b200_decode16_device.
 * Frame i's output is Hb = ceil(H / factor) rows of Wb = ceil(W / factor) U16, tightly packed, at out + i * Wb * Hb
 * U16; nothing outside [out, out + nframes * Wb * Hb * 2 bytes) is written.  Output pixel (X, Y) is the mean of the
 * IN-FRAME pixels of dbde_b200_decode16_device's image in [factor X, factor X + factor) x [factor Y, factor Y +
 * factor), rounded half up: (sum + n / 2) / n in integers with 32-bit sums, n the number of in-frame pixels (factor^2
 * except in the last column when W % factor != 0 and the last row when H % factor != 0).  Validation, status, indices
 * and rejected frames as for the DBDE16 crops above; DBDE_INVERT_ENDIAN is ignored.  DBDE_B200_E_INVALID before any
 * work is queued for: NULL pointers (when nframes > 0), an output pointer that is not 2-byte aligned, a factor other
 * than 1, 2, 4 or 8, frame dimensions the frame limits reject.  nframes == 0 returns 0.
 * _device: asynchronous on `stream`.  _host: the chunk pipeline of dbde_b200_decode16_host (records still cross PCIe
 * whole, only the accepted frames' binned pixels come back). */
DBDE_B200_API int dbde_b200_decode16_binned_device(dbde_b200_ctx *ctx, const uint8_t *stream_dev, size_t stream_bytes,
                                                   const uint64_t *frame_offsets_dev, int W, int H, int nframes, int factor,
                                                   uint16_t *out_dev, uint32_t *status_dev, uint64_t *indices_dev, void *stream);
DBDE_B200_API int dbde_b200_decode16_binned_host(dbde_b200_ctx *ctx, const uint8_t *stream_host, size_t stream_bytes,
                                                 const uint64_t *frame_offsets_host, int W, int H, int nframes, int factor,
                                                 uint16_t *out_host, uint32_t *status_host, uint64_t *indices_host);

/* ---- .dbde files (SURVEY.md 8 f-1): 28-byte video header + frame records back to back ------------- */
/* The container the reference's walker reads (dbde_util.cpp:362-426; dbde_start_file_walk /
 * dbde_walk_a_file / dbde_end_file_walk in include/dbde_util.h remain available as the drop-in).
 * The reference has no writer (only dbde_util_test.cpp:204-211); these stream whole batches through
 * the GPU codec with disk I/O overlapped on a helper thread.  A writer/reader belongs to the thread
 * that owns its context. */
typedef struct dbde_b200_writer dbde_b200_writer;
typedef struct dbde_b200_reader dbde_b200_reader;
/* creates/truncates `path` and writes the video header {3, H, W, frame_hz} (dbde_util.cpp:198-209);
 * frame indices start at first_index */
DBDE_B200_API int dbde_b200_writer_open(dbde_b200_ctx *ctx, const char *path, int W, int H, double frame_hz,
                                        uint64_t first_index, dbde_b200_writer **out);
/* encodes nframes frames (host memory, tightly packed) and appends their records; the bytes reach
 * the file while the next batch is being encoded */
DBDE_B200_API int dbde_b200_writer_append(dbde_b200_writer *w, const uint8_t *frames_host, int nframes);
DBDE_B200_API int dbde_b200_writer_close(dbde_b200_writer *w, uint64_t *frames_written, uint64_t *bytes_written);
/* opens `path`, parses the video header (rejects u64s != 3 and the reference's size limits,
 * dbde_util.cpp:374-378); batch_frames = frames decoded per GPU batch (<= 0: 16) */
DBDE_B200_API int dbde_b200_reader_open(dbde_b200_ctx *ctx, const char *path, int batch_frames, int *W, int *H,
                                        double *frame_hz, dbde_b200_reader **out);
/* decodes the next <= min(max_frames, batch_frames) frames into frames_host; returns how many were
 * handed out, 0 at the end of the file, < 0 on error.  status[i] != 0 marks a rejected record (pixels
 * untouched); reading stops after the first one, like the reference's walker (dbde_util.cpp:416). */
DBDE_B200_API long dbde_b200_reader_next(dbde_b200_reader *r, uint8_t *frames_host, int max_frames,
                                         uint64_t *indices, uint32_t *status);
/* from the next dbde_b200_reader_next on, hand out the region (x0, y0, roi_w, roi_h) of every frame,
 * roi_w * roi_h bytes per frame (dbde_b200_decode_roi_host); (0, 0, W, H) restores whole frames.  May be
 * called between reader_next calls.  A region outside the frame is DBDE_B200_E_INVALID. */
DBDE_B200_API int dbde_b200_reader_set_roi(dbde_b200_reader *r, int x0, int y0, int roi_w, int roi_h);
DBDE_B200_API int dbde_b200_reader_close(dbde_b200_reader *r);
DBDE_B200_API const char *dbde_b200_file_last_error(void);

/* ---- the reference's compile-time format variants (SURVEY.md 8 f-3) --------------------------- */
/* DBDE_INVERT_ENDIAN (dbde_util.cpp:15-19,24-27,246-270): every 8-pixel tile row is byte-reversed
 * before packing and after unpacking.  DBDE_HZ_AS_INTEGER (dbde_util.cpp:203-204,352-353): the video
 * header carries frame_hz as a rounded U64 instead of a double.  Compiling this library with the
 * same macros makes them its defaults (as in the reference); these calls switch them at run time.
 * set_format_variants is process-wide: it sets the default of contexts created afterwards, and the
 * C++ drop-in functions (dbde_util.h) follow it on every call.  set_invert_endian changes one context. */
DBDE_B200_API void dbde_b200_set_format_variants(int invert_endian, int hz_as_integer);
DBDE_B200_API void dbde_b200_get_format_variants(int *invert_endian, int *hz_as_integer);
DBDE_B200_API int dbde_b200_set_invert_endian(dbde_b200_ctx *ctx, int on);

/* Tuning knob for the host path: frames per staged chunk (default: ~64 MiB of pixels). */
DBDE_B200_API int dbde_b200_set_chunk_frames(dbde_b200_ctx *ctx, int frames);

/* Launch accounting for benchmarks: kernels launched by this context since creation. */
DBDE_B200_API uint64_t dbde_b200_kernel_launches(const dbde_b200_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
