"""ctypes face of libdbde_b200.so (the B200-native DBDE codec) for tests and bench.py.

The product is the shared library: sm_100a kernels behind the extern "C" layer declared in
include/dbde_b200.h plus the C++ mirror of the reference interface (include/dbde_util.h).
This module only loads it and marshals numpy / raw device pointers.  It never touches oracle/
and there is no fallback: a missing library raises, a missing GPU makes `Codec()` raise.

Import with  importlib.import_module("dbce-video-cpp_b200")  (the directory name carries a hyphen).
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# DBDE_B200_LIB selects an alternative build of the SAME library (A/B profiling variants)
LIB_PATH = os.environ.get("DBDE_B200_LIB") or os.path.join(HERE, "libdbde_b200.so")

_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)

ST_BAD_FRAME_HEADER, ST_BAD_DEPTH_COUNT, ST_BAD_MIN_COUNT = 1, 2, 4
ST_BAD_WORD_COUNT, ST_DEPTH_TOO_BIG, ST_TRUNCATED = 8, 16, 32

# every extern "C" symbol include/dbde_b200.h declares
C_SYMBOLS = [
    "dbde_b200_create", "dbde_b200_destroy", "dbde_b200_last_error", "dbde_b200_device_count",
    "dbde_b200_frame_record_bound", "dbde_b200_slot_stride", "dbde_b200_stream_bound", "dbde_b200_device_alloc", "dbde_b200_device_free",
    "dbde_b200_host_alloc", "dbde_b200_host_free", "dbde_b200_host_register", "dbde_b200_host_unregister", "dbde_b200_memcpy_h2d", "dbde_b200_memcpy_d2h",
    "dbde_b200_encode_device", "dbde_b200_decode_device", "dbde_b200_encode_host", "dbde_b200_decode_host",
    "dbde_b200_encode_host_sharded", "dbde_b200_decode_host_sharded",
    "dbde_b200_frame_record_bound16", "dbde_b200_slot_stride16", "dbde_b200_encode16_device", "dbde_b200_decode16_device",
    "dbde_b200_encode16_host", "dbde_b200_decode16_host", "dbde_b200_index_stream16",
    "dbde_b200_index_stream", "dbde_b200_validate_device", "dbde_b200_validate_host", "dbde_b200_set_chunk_frames", "dbde_b200_kernel_launches",
    "dbde_b200_set_format_variants", "dbde_b200_get_format_variants", "dbde_b200_set_invert_endian",
    "dbde_b200_writer_open", "dbde_b200_writer_append", "dbde_b200_writer_close",
    "dbde_b200_reader_open", "dbde_b200_reader_next", "dbde_b200_reader_close", "dbde_b200_file_last_error",
    "dbde_b200_decode_roi_device", "dbde_b200_decode_roi_host", "dbde_b200_reader_set_roi",
    "dbde_b200_decode_crops_device", "dbde_b200_decode_crops_host",
    "dbde_b200_decode_binned_device", "dbde_b200_decode_binned_host",
    "dbde_b200_decode16_crops_device", "dbde_b200_decode16_crops_host",
    "dbde_b200_decode16_binned_device", "dbde_b200_decode16_binned_host",
    "dbde_b200_encode_crops_device", "dbde_b200_encode_crops_host",
    "dbde_b200_encode16_crops_device", "dbde_b200_encode16_crops_host",
]
# the reference's C++ entry points (include/dbde_util.h), by mangled name (SURVEY.md 8b)
CXX_SYMBOLS = {
    "dbde_pack_8x8": "_Z13dbde_pack_8x8PhiS_",
    "dbde_pack_8x8_partial": "_Z21dbde_pack_8x8_partialPhiiiS_",
    "dbde_pack_image": "_Z15dbde_pack_imagePhiiS_",
    "dbde_pack_frame_header": "_Z22dbde_pack_frame_header12frame_headerPh",
    "dbde_pack_frame": "_Z15dbde_pack_framemPhiiS_",
    "dbde_pack_video_header": "_Z22dbde_pack_video_header12video_headerPh",
    "dbde_unpack_8x8": "_Z15dbde_unpack_8x8hhPhmS_",
    "dbde_unpack_8x8_partial": "_Z23dbde_unpack_8x8_partialhhPhmiiS_",
    "dbde_unpack_image": "_Z17dbde_unpack_imagePhiiS_",
    "dbde_unpack_frame_header": "_Z24dbde_unpack_frame_headerPPh",
    "dbde_unpack_frame": "_Z17dbde_unpack_framePPhiiS_",
    "dbde_unpack_video_header": "_Z24dbde_unpack_video_headerPPh",
    "dbde_start_file_walk": "_Z20dbde_start_file_walkPKciP12video_header",
    "dbde_walk_a_file": "_Z16dbde_walk_a_fileP16dbde_file_walkerP12frame_headerPh",
    "dbde_end_file_walk": "_Z18dbde_end_file_walkP16dbde_file_walker",
}


def build(verbose=False):
    """Compile the library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", os.path.join(HERE, "csrc")], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout + r.stderr)
    if r.returncode or not os.path.exists(LIB_PATH):
        raise RuntimeError("building libdbde_b200.so failed:\n" + r.stdout + r.stderr)


def load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(LIB_PATH + " is missing: run __graft_entry__.build() (there is no fallback path)")
    lib = C.CDLL(LIB_PATH)
    lib.dbde_b200_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.dbde_b200_destroy.argtypes = [C.c_void_p]
    lib.dbde_b200_destroy.restype = None
    lib.dbde_b200_last_error.restype = C.c_char_p
    lib.dbde_b200_frame_record_bound.restype = C.c_size_t
    lib.dbde_b200_frame_record_bound.argtypes = [C.c_int, C.c_int]
    lib.dbde_b200_slot_stride.restype = C.c_size_t
    lib.dbde_b200_slot_stride.argtypes = [C.c_int, C.c_int]
    lib.dbde_b200_stream_bound.restype = C.c_size_t
    lib.dbde_b200_stream_bound.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.dbde_b200_device_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    lib.dbde_b200_device_free.argtypes = [C.c_void_p, C.c_void_p]
    lib.dbde_b200_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    lib.dbde_b200_host_free.argtypes = [C.c_void_p]
    lib.dbde_b200_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.dbde_b200_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    lib.dbde_b200_encode_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                            C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int,
                                            C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_encode_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                          C.c_void_p, C.c_size_t, C.c_void_p]
    lib.dbde_b200_decode_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int,
                                          C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_encode_host_sharded.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                                  C.c_void_p, C.c_size_t, C.c_void_p]
    lib.dbde_b200_decode_host_sharded.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int,
                                                  C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_index_stream16.restype = C.c_long
    lib.dbde_b200_index_stream16.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_long]
    lib.dbde_b200_index_stream.restype = C.c_long
    lib.dbde_b200_index_stream.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_long]
    lib.dbde_b200_set_chunk_frames.argtypes = [C.c_void_p, C.c_int]
    for fn in (lib.dbde_b200_frame_record_bound16, lib.dbde_b200_slot_stride16):
        fn.restype = C.c_size_t
        fn.argtypes = [C.c_int, C.c_int]
    lib.dbde_b200_encode16_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_size_t,
                                            C.c_void_p]
    lib.dbde_b200_decode16_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_void_p]
    lib.dbde_b200_encode16_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_size_t,
                                              C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode16_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.dbde_b200_host_unregister.argtypes = [C.c_void_p]
    lib.dbde_b200_set_format_variants.restype = None
    lib.dbde_b200_set_format_variants.argtypes = [C.c_int, C.c_int]
    lib.dbde_b200_get_format_variants.restype = None
    lib.dbde_b200_get_format_variants.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.dbde_b200_set_invert_endian.argtypes = [C.c_void_p, C.c_int]
    lib.dbde_b200_kernel_launches.restype = C.c_uint64
    lib.dbde_b200_kernel_launches.argtypes = [C.c_void_p]
    lib.dbde_b200_writer_open.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_double, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.dbde_b200_writer_append.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    lib.dbde_b200_writer_close.argtypes = [C.c_void_p, _u64p, _u64p]
    lib.dbde_b200_reader_open.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                          C.POINTER(C.c_double), C.POINTER(C.c_void_p)]
    lib.dbde_b200_reader_next.restype = C.c_long
    lib.dbde_b200_reader_next.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.dbde_b200_reader_close.argtypes = [C.c_void_p]
    lib.dbde_b200_reader_set_roi.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.dbde_b200_decode_roi_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode_roi_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode_crops_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                  C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode_crops_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                                C.c_void_p]
    lib.dbde_b200_decode_binned_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                   C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode_binned_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                 C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.dbde_b200_decode16_crops_device.argtypes = lib.dbde_b200_decode_crops_device.argtypes
    lib.dbde_b200_decode16_crops_host.argtypes = lib.dbde_b200_decode_crops_host.argtypes
    lib.dbde_b200_decode16_binned_device.argtypes = lib.dbde_b200_decode_binned_device.argtypes
    lib.dbde_b200_decode16_binned_host.argtypes = lib.dbde_b200_decode_binned_host.argtypes
    lib.dbde_b200_encode_crops_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_int,
                                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                                  C.c_void_p, C.c_void_p]
    lib.dbde_b200_encode_crops_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_void_p, C.c_int,
                                                C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.dbde_b200_encode16_crops_device.argtypes = lib.dbde_b200_encode_crops_device.argtypes
    lib.dbde_b200_encode16_crops_host.argtypes = lib.dbde_b200_encode_crops_host.argtypes
    lib.dbde_b200_validate_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p]
    lib.dbde_b200_file_last_error.restype = C.c_char_p
    return lib


def _corners(corners, N):
    """int32 crop corners (R, 2), the same for every frame, or (N, R, 2), per frame -> (contiguous corners, per_frame, R)"""
    corners = np.ascontiguousarray(corners, dtype=np.int32)
    if corners.ndim == 3 and corners.shape[0] == N and corners.shape[2] == 2:
        per_frame = 1
    elif corners.ndim == 2 and corners.shape[1] == 2:
        per_frame = 0
    else:
        raise ValueError("corners must have shape (R, 2) or (N, R, 2), got %r" % (corners.shape,))
    return corners, per_frame, corners.shape[-2]


def _binned_shape(W, H, factor):
    return (-(-H // factor), -(-W // factor)) if factor > 0 else (0, 0)


class DbdeError(RuntimeError):
    pass


class PinnedArray:
    """numpy view over pinned host memory from dbde_b200_host_alloc."""

    def __init__(self, lib, nbytes):
        self.lib, self.nbytes = lib, int(nbytes)
        p = C.c_void_p()
        rc = lib.dbde_b200_host_alloc(self.nbytes, C.byref(p))
        if rc:
            raise DbdeError("host_alloc: %s" % lib.dbde_b200_last_error().decode())
        self.ptr = p.value
        self.array = np.ctypeslib.as_array((C.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr))[:self.nbytes]

    def free(self):
        if self.ptr:
            self.array = None
            self.lib.dbde_b200_host_free(self.ptr)
            self.ptr = None


class Codec:
    """One GPU context.  Raises if there is no B200: there is no CPU path."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.dbde_b200_create(device, C.byref(h))
        if rc or not h.value:
            raise DbdeError("dbde_b200_create(%d) failed (%d): %s" % (device, rc, self.lib.dbde_b200_last_error().decode()))
        self.h = h

    def close(self):
        if self.h:
            self.lib.dbde_b200_destroy(self.h)
            self.h = None

    def _ck(self, rc, what):
        if rc:
            raise DbdeError("%s failed (%d): %s" % (what, rc, self.lib.dbde_b200_last_error().decode()))

    # ---- sizes / memory
    def frame_record_bound(self, W, H):
        return self.lib.dbde_b200_frame_record_bound(W, H)

    def stream_bound(self, W, H, n):
        return self.lib.dbde_b200_stream_bound(W, H, n)

    def slot_stride(self, W, H):
        return self.lib.dbde_b200_slot_stride(W, H)

    def pinned(self, nbytes):
        return PinnedArray(self.lib, nbytes)

    def device_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.lib.dbde_b200_device_alloc(self.h, nbytes, C.byref(p)), "device_alloc")
        return p.value

    def device_free(self, ptr):
        self._ck(self.lib.dbde_b200_device_free(self.h, ptr), "device_free")

    def h2d(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self._ck(self.lib.dbde_b200_memcpy_h2d(self.h, dptr, arr.ctypes.data, arr.nbytes), "memcpy_h2d")

    def d2h(self, dptr, nbytes, dtype=np.uint8):
        out = np.empty(nbytes // np.dtype(dtype).itemsize, dtype=dtype)
        self._ck(self.lib.dbde_b200_memcpy_d2h(self.h, out.ctypes.data, dptr, out.nbytes), "memcpy_d2h")
        return out

    def launches(self):
        return int(self.lib.dbde_b200_kernel_launches(self.h))

    def set_chunk_frames(self, n):
        self._ck(self.lib.dbde_b200_set_chunk_frames(self.h, n), "set_chunk_frames")

    def set_invert_endian(self, on):
        """the reference's DBDE_INVERT_ENDIAN build variant for this context (dbde_util.cpp:15-19)"""
        self._ck(self.lib.dbde_b200_set_invert_endian(self.h, int(bool(on))), "set_invert_endian")

    # ---- device-resident hot path (raw device pointers, asynchronous on `stream`)
    def encode_device(self, frames_ptr, W, H, first_index, n, out_ptr, out_cap, offs_ptr, sizes_ptr, stream=0,
                      slot_stride=0):
        """record i -> out_ptr + i*slot_stride; offs[i] = i*slot_stride, sizes[i] = record bytes"""
        self._ck(self.lib.dbde_b200_encode_device(self.h, frames_ptr, W, H, first_index, n, out_ptr, out_cap,
                                                  slot_stride, offs_ptr, sizes_ptr, stream), "encode_device")

    def encode_crops_device(self, frames_ptr, W, H, first_index, n, corners_ptr, ncrops, per_frame, size, out_ptr, out_cap,
                            offs_ptr, sizes_ptr, pad=0, stream=0, slot_stride=0):
        """ncrops crops of size = (crop_w, crop_h) per frame at the int32 {x0, y0} corners at corners_ptr (device; per_frame:
        n * ncrops pairs, else ncrops pairs for every frame), pixels outside the frame `pad`: record f * ncrops + r is the
        record of crop r of frame f as a crop_w x crop_h frame with index first_index + f, at out_ptr + (f * ncrops + r) *
        slot_stride; offs[j] = j * slot_stride, sizes[j] = record bytes"""
        cw, ch = (int(v) for v in size)
        self._ck(self.lib.dbde_b200_encode_crops_device(self.h, frames_ptr, W, H, first_index, n, corners_ptr, ncrops, int(per_frame),
                                                        cw, ch, pad, out_ptr, out_cap, slot_stride, offs_ptr, sizes_ptr, stream),
                 "encode_crops_device")

    def decode_device(self, stream_ptr, stream_bytes, offs_ptr, W, H, n, frames_ptr, status_ptr, index_ptr=None,
                      stream=0):
        self._ck(self.lib.dbde_b200_decode_device(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, n, frames_ptr,
                                                  status_ptr, index_ptr, stream), "decode_device")

    def decode_roi_device(self, stream_ptr, stream_bytes, offs_ptr, W, H, n, roi, out_ptr, status_ptr, index_ptr=None,
                          stream=0):
        """region roi = (x0, y0, roi_w, roi_h) of every frame -> out_ptr, n * roi_w * roi_h bytes tightly packed"""
        x0, y0, rw, rh = (int(v) for v in roi)
        self._ck(self.lib.dbde_b200_decode_roi_device(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, n, x0, y0, rw, rh,
                                                      out_ptr, status_ptr, index_ptr, stream), "decode_roi_device")

    def decode_crops_device(self, stream_ptr, stream_bytes, offs_ptr, W, H, n, corners_ptr, ncrops, per_frame, size, out_ptr,
                            status_ptr, index_ptr=None, pad=0, stream=0):
        """ncrops crops of size = (crop_w, crop_h) per frame at the int32 {x0, y0} corners at corners_ptr (device; per_frame:
        n * ncrops pairs, else ncrops pairs for every frame) -> out_ptr, n * ncrops * crop_w * crop_h bytes tightly packed;
        pixels outside the frame are `pad`"""
        cw, ch = (int(v) for v in size)
        self._ck(self.lib.dbde_b200_decode_crops_device(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, n, corners_ptr, ncrops,
                                                        int(per_frame), cw, ch, pad, out_ptr, status_ptr, index_ptr, stream),
                 "decode_crops_device")

    def decode_binned_device(self, stream_ptr, stream_bytes, offs_ptr, W, H, n, factor, out_ptr, status_ptr, index_ptr=None,
                             stream=0):
        """every frame binned by factor (1, 2, 4 or 8): the rounded means of its in-frame factor x factor blocks -> out_ptr,
        n * ceil(H / factor) * ceil(W / factor) bytes tightly packed"""
        self._ck(self.lib.dbde_b200_decode_binned_device(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, n, int(factor), out_ptr,
                                                         status_ptr, index_ptr, stream), "decode_binned_device")

    # ---- host-buffer hot path (numpy or raw host pointers)
    def encode_host(self, frames, first_index=0):
        """frames (N,H,W) u8 -> (stream bytes, offsets[N+1])"""
        return self._encode_host(self.lib.dbde_b200_encode_host, "encode_host", frames, np.uint8, first_index)

    def encode_crops_host(self, frames, corners, size, pad=0, first_index=0):
        """frames (N,H,W) u8, crops of size = (crop_w, crop_h) at int32 corners (R, 2) (the same for every frame) or
        (N, R, 2) (per frame), pixels outside the frame `pad` -> (stream bytes, offsets[N*R+1]); record f * R + r is crop r
        of frame f, with frame index first_index + f"""
        return self._encode_host(self.lib.dbde_b200_encode_crops_host, "encode_crops_host", frames, np.uint8, first_index, corners,
                                 size, pad)

    def _encode_host(self, fn, name, frames, dtype, first_index, corners=None, size=None, pad=0):
        """the numpy host encodes: frames (N,H,W) of dtype -> (stream bytes, offsets[N*R+1]), R = 1 or, with corners, the
        crops per frame"""
        frames = np.ascontiguousarray(frames, dtype=dtype)
        N, H, W = frames.shape
        rw, rh, R, crops = W, H, 1, ()
        if corners is not None:
            rw, rh = (int(v) for v in size)
            corners, per_frame, R = _corners(corners, N)
            crops = (corners.ctypes.data, R, per_frame, rw, rh, pad)
        stride = self.lib.dbde_b200_slot_stride16 if dtype == np.uint16 else self.lib.dbde_b200_slot_stride
        cap = int(stride(rw, rh)) * max(N * R, 1) + 16 if rw > 0 and rh > 0 else 16
        out = np.empty(cap, dtype=np.uint8)
        offs = np.zeros(N * R + 1, dtype=np.uint64)
        self._ck(fn(self.h, frames.ctypes.data, W, H, first_index, N, *crops, out.ctypes.data, cap, offs.ctypes.data), name)
        return out[:int(offs[N * R])].copy(), offs

    def encode_host_raw(self, frames_ptr, W, H, first_index, N, out_ptr, out_cap, offs_ptr):
        self._ck(self.lib.dbde_b200_encode_host(self.h, frames_ptr, W, H, first_index, N, out_ptr, out_cap, offs_ptr),
                 "encode_host")

    def decode_host(self, stream, offsets, W, H, fill=None):
        """-> (frames (N,H,W), status[N], indices[N]); rejected frames keep `fill`"""
        return self._decode_host(self.lib.dbde_b200_decode_host, "decode_host", stream, offsets, W, H, (H, W), np.uint8, fill)

    def decode_roi_host(self, stream, offsets, W, H, roi, fill=None):
        """region roi = (x0, y0, roi_w, roi_h) of every frame -> (frames (N, roi_h, roi_w), status[N], indices[N]);
        rejected frames keep `fill`"""
        x0, y0, rw, rh = (int(v) for v in roi)
        return self._decode_host(self.lib.dbde_b200_decode_roi_host, "decode_roi_host", stream, offsets, W, H, (max(rh, 0), max(rw, 0)),
                                 np.uint8, fill, x0, y0, rw, rh)

    def decode_crops_host(self, stream, offsets, W, H, corners, size, pad=0, fill=None):
        """crops of size = (crop_w, crop_h) at int32 corners (R, 2) (the same for every frame) or (N, R, 2) (per frame) ->
        (crops (N, R, crop_h, crop_w), status[N], indices[N]); pixels outside the frame are `pad`, rejected frames keep
        `fill`"""
        cw, ch = (int(v) for v in size)
        corners, per_frame, R = _corners(corners, len(offsets))
        return self._decode_host(self.lib.dbde_b200_decode_crops_host, "decode_crops_host", stream, offsets, W, H, (R, max(ch, 0), max(cw, 0)),
                                 np.uint8, fill, corners.ctypes.data, R, per_frame, cw, ch, pad)

    def decode_binned_host(self, stream, offsets, W, H, factor, fill=None):
        """every frame binned by factor (1, 2, 4 or 8) -> (frames (N, ceil(H / factor), ceil(W / factor)), status[N],
        indices[N]); rejected frames keep `fill`"""
        factor = int(factor)
        return self._decode_host(self.lib.dbde_b200_decode_binned_host, "decode_binned_host", stream, offsets, W, H,
                                 _binned_shape(W, H, factor), np.uint8, fill, factor)

    def _decode_host(self, fn, name, stream, offsets, W, H, shape, dtype, fill, *args):
        """the numpy host decodes: N = len(offsets) records -> (output (N,) + shape of dtype, status[N], indices[N]) with
        rejected frames keeping `fill`; shape None (validation): -> (status[N], indices[N])"""
        stream = np.ascontiguousarray(stream, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        N = len(offsets)
        out = None if shape is None else np.zeros((N,) + shape, dtype=dtype) if fill is None else np.full((N,) + shape, fill, dtype=dtype)
        status = np.zeros(N, dtype=np.uint32)
        index = np.zeros(N, dtype=np.uint64)
        out_ptr = () if out is None else (out.ctypes.data,)
        self._ck(fn(self.h, stream.ctypes.data, stream.nbytes, offsets.ctypes.data, W, H, N, *args, *out_ptr, status.ctypes.data,
                    index.ctypes.data), name)
        return (status, index) if out is None else (out, status, index)

    def decode_host_raw(self, stream_ptr, stream_bytes, offs_ptr, W, H, N, frames_ptr, status_ptr, index_ptr=None):
        self._ck(self.lib.dbde_b200_decode_host(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, N, frames_ptr,
                                                status_ptr, index_ptr), "decode_host")

    # ---- DBDE16, the 16-bit extension (SURVEY 8 f-4)
    def encode16_host(self, frames, first_index=0):
        """frames (N,H,W) u16 -> (stream bytes, offsets[N+1])"""
        return self._encode_host(self.lib.dbde_b200_encode16_host, "encode16_host", frames, np.uint16, first_index)

    def encode16_crops_device(self, frames_ptr, W, H, first_index, n, corners_ptr, ncrops, per_frame, size, out_ptr, out_cap,
                              offs_ptr, sizes_ptr, pad=0, stream=0, slot_stride=0):
        """U16 frames (2-byte aligned): ncrops crops of size = (crop_w, crop_h) per frame at the int32 {x0, y0} corners at
        corners_ptr (device; per_frame: n * ncrops pairs, else ncrops pairs for every frame), pixels outside the frame
        `pad` (0..65535): record f * ncrops + r is the DBDE16 record of crop r of frame f as a crop_w x crop_h frame with
        index first_index + f, at out_ptr + (f * ncrops + r) * slot_stride; offs[j] = j * slot_stride, sizes[j] = record
        bytes"""
        cw, ch = (int(v) for v in size)
        self._ck(self.lib.dbde_b200_encode16_crops_device(self.h, frames_ptr, W, H, first_index, n, corners_ptr, ncrops,
                                                          int(per_frame), cw, ch, pad, out_ptr, out_cap, slot_stride, offs_ptr,
                                                          sizes_ptr, stream), "encode16_crops_device")

    def encode16_crops_host(self, frames, corners, size, pad=0, first_index=0):
        """frames (N,H,W) u16, crops of size = (crop_w, crop_h) at int32 corners (R, 2) (the same for every frame) or
        (N, R, 2) (per frame), pixels outside the frame `pad` -> (stream bytes, offsets[N*R+1]); record f * R + r is the
        DBDE16 record of crop r of frame f, with frame index first_index + f"""
        return self._encode_host(self.lib.dbde_b200_encode16_crops_host, "encode16_crops_host", frames, np.uint16, first_index, corners,
                                 size, pad)

    def decode16_host(self, stream, offsets, W, H, fill=None):
        """-> (frames (N,H,W) u16, status[N], indices[N]); rejected frames keep `fill`"""
        return self._decode_host(self.lib.dbde_b200_decode16_host, "decode16_host", stream, offsets, W, H, (H, W), np.uint16, fill)

    def decode16_crops_device(self, stream_ptr, stream_bytes, offs_ptr, W, H, n, corners_ptr, ncrops, per_frame, size, out_ptr,
                              status_ptr, index_ptr=None, pad=0, stream=0):
        """DBDE16 records: ncrops crops of size = (crop_w, crop_h) per frame at the int32 {x0, y0} corners at corners_ptr
        (device; per_frame: n * ncrops pairs, else ncrops pairs for every frame) -> out_ptr (2-byte aligned), n * ncrops *
        crop_w * crop_h U16 tightly packed; pixels outside the frame are `pad` (0..65535)"""
        cw, ch = (int(v) for v in size)
        self._ck(self.lib.dbde_b200_decode16_crops_device(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, n, corners_ptr, ncrops,
                                                          int(per_frame), cw, ch, pad, out_ptr, status_ptr, index_ptr, stream),
                 "decode16_crops_device")

    def decode16_binned_device(self, stream_ptr, stream_bytes, offs_ptr, W, H, n, factor, out_ptr, status_ptr, index_ptr=None,
                               stream=0):
        """DBDE16 records, every frame binned by factor (1, 2, 4 or 8): the rounded means of its in-frame factor x factor
        blocks -> out_ptr (2-byte aligned), n * ceil(H / factor) * ceil(W / factor) U16 tightly packed"""
        self._ck(self.lib.dbde_b200_decode16_binned_device(self.h, stream_ptr, stream_bytes, offs_ptr, W, H, n, int(factor),
                                                           out_ptr, status_ptr, index_ptr, stream), "decode16_binned_device")

    def decode16_crops_host(self, stream, offsets, W, H, corners, size, pad=0, fill=None):
        """DBDE16 records: crops of size = (crop_w, crop_h) at int32 corners (R, 2) (the same for every frame) or (N, R, 2)
        (per frame) -> (crops (N, R, crop_h, crop_w) u16, status[N], indices[N]); pixels outside the frame are `pad`,
        rejected frames keep `fill`"""
        cw, ch = (int(v) for v in size)
        corners, per_frame, R = _corners(corners, len(offsets))
        return self._decode_host(self.lib.dbde_b200_decode16_crops_host, "decode16_crops_host", stream, offsets, W, H, (R, max(ch, 0), max(cw, 0)),
                                 np.uint16, fill, corners.ctypes.data, R, per_frame, cw, ch, pad)

    def decode16_binned_host(self, stream, offsets, W, H, factor, fill=None):
        """DBDE16 records, every frame binned by factor (1, 2, 4 or 8) -> (frames (N, ceil(H / factor), ceil(W / factor))
        u16, status[N], indices[N]); rejected frames keep `fill`"""
        factor = int(factor)
        return self._decode_host(self.lib.dbde_b200_decode16_binned_host, "decode16_binned_host", stream, offsets, W, H,
                                 _binned_shape(W, H, factor), np.uint16, fill, factor)

    def validate_host(self, stream, offsets, W, H):
        """GPU validation without decoding (SURVEY 8 f-2) -> (status[N], indices[N])"""
        return self._decode_host(self.lib.dbde_b200_validate_host, "validate_host", stream, offsets, W, H, None, None, None)

    def index_stream(self, stream, W, H, max_frames=1 << 20):
        stream = np.ascontiguousarray(stream, dtype=np.uint8)
        offs = np.zeros(max_frames + 1, dtype=np.uint64)
        n = self.lib.dbde_b200_index_stream(stream.ctypes.data, stream.nbytes, W, H, offs.ctypes.data, max_frames)
        if n < 0:
            raise DbdeError("index_stream failed")
        return offs[:n + 1].copy()


def encode_host_sharded(codecs, frames, first_index=0):
    """dbde_b200_encode_host_sharded over several Codec contexts -> (stream, offsets[N+1])."""
    lib = codecs[0].lib
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    N, H, W = frames.shape
    cap = codecs[0].stream_bound(W, H, N)
    out = np.empty(cap, dtype=np.uint8)
    offs = np.zeros(N + 1, dtype=np.uint64)
    arr = (C.c_void_p * len(codecs))(*[c.h.value for c in codecs])
    rc = lib.dbde_b200_encode_host_sharded(arr, len(codecs), frames.ctypes.data, W, H, first_index, N, out.ctypes.data,
                                           cap, offs.ctypes.data)
    if rc:
        raise DbdeError("encode_host_sharded failed (%d): %s" % (rc, lib.dbde_b200_last_error().decode()))
    return out[:int(offs[N])].copy(), offs


def decode_host_sharded(codecs, stream, offsets, W, H):
    lib = codecs[0].lib
    stream = np.ascontiguousarray(stream, dtype=np.uint8)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    N = len(offsets)
    frames = np.zeros((N, H, W), dtype=np.uint8)
    status = np.zeros(N, dtype=np.uint32)
    index = np.zeros(N, dtype=np.uint64)
    arr = (C.c_void_p * len(codecs))(*[c.h.value for c in codecs])
    rc = lib.dbde_b200_decode_host_sharded(arr, len(codecs), stream.ctypes.data, stream.nbytes, offsets.ctypes.data, W, H,
                                           N, frames.ctypes.data, status.ctypes.data, index.ctypes.data)
    if rc:
        raise DbdeError("decode_host_sharded failed (%d): %s" % (rc, lib.dbde_b200_last_error().decode()))
    return frames, status, index


def write_file(codec, path, frames, hz=30.0, first_index=0, batch=16):
    """dbde_b200_writer_*: stream `frames` (N,H,W) into a .dbde file in batches -> (frames, bytes) written"""
    lib = codec.lib
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    N, H, W = frames.shape
    w = C.c_void_p()
    if lib.dbde_b200_writer_open(codec.h, path.encode(), W, H, hz, first_index, C.byref(w)):
        raise DbdeError("writer_open: " + lib.dbde_b200_file_last_error().decode())
    try:
        for a in range(0, N, batch):
            part = frames[a:a + batch]
            if lib.dbde_b200_writer_append(w, part.ctypes.data, len(part)):
                raise DbdeError("writer_append: " + lib.dbde_b200_file_last_error().decode())
    finally:
        nf, nb = C.c_uint64(), C.c_uint64()
        rc = lib.dbde_b200_writer_close(w, C.byref(nf), C.byref(nb))
    if rc:
        raise DbdeError("writer_close: " + lib.dbde_b200_file_last_error().decode())
    return nf.value, nb.value


def read_file(codec, path, batch=16, fill=0xCD, roi=None):
    """dbde_b200_reader_*: -> ((W, H, hz), frames (N,H,W), indices[N], status[N]).  roi = (x0, y0, roi_w, roi_h):
    only that region of every frame, frames (N, roi_h, roi_w)"""
    lib = codec.lib
    r, W, H, hz = C.c_void_p(), C.c_int(), C.c_int(), C.c_double()
    if lib.dbde_b200_reader_open(codec.h, path.encode(), batch, C.byref(W), C.byref(H), C.byref(hz), C.byref(r)):
        raise DbdeError("reader_open: " + lib.dbde_b200_file_last_error().decode())
    out, idx, st = [], [], []
    ow, oh = W.value, H.value
    try:
        if roi is not None:
            x0, y0, ow, oh = (int(v) for v in roi)
            if lib.dbde_b200_reader_set_roi(r, x0, y0, ow, oh):
                raise DbdeError("reader_set_roi: " + lib.dbde_b200_file_last_error().decode())
        while True:
            fr = np.full((batch, oh, ow), fill, dtype=np.uint8)
            ii = np.zeros(batch, dtype=np.uint64)
            ss = np.zeros(batch, dtype=np.uint32)
            n = lib.dbde_b200_reader_next(r, fr.ctypes.data, batch, ii.ctypes.data, ss.ctypes.data)
            if n < 0:
                raise DbdeError("reader_next: " + lib.dbde_b200_file_last_error().decode())
            if n == 0:
                break
            out.append(fr[:n]); idx.append(ii[:n]); st.append(ss[:n])
    finally:
        lib.dbde_b200_reader_close(r)
    if not out:
        return (W.value, H.value, hz.value), np.zeros((0, oh, ow), np.uint8), np.zeros(0, np.uint64), np.zeros(0, np.uint32)
    return (W.value, H.value, hz.value), np.concatenate(out), np.concatenate(idx), np.concatenate(st)


# ---------------------------------------------------------------------------------------------
# The reference's own C++ entry points, called by mangled name exactly as a program linked
# against the reference would call them (include/dbde_util.h).  Used by the parity tests so they
# read like the reference's tests (dbde_util_test.cpp).
class _FrameHeader(C.Structure):
    _fields_ = [("u64s", C.c_uint32), ("index", C.c_uint64), ("elapsed_ns", C.c_uint64)]


class _VideoHeader(C.Structure):
    _fields_ = [("u64s", C.c_uint32), ("height", C.c_uint64), ("width", C.c_uint64), ("frame_hz", C.c_double)]


class _Walker(C.Structure):
    _fields_ = [("fptr", C.c_void_p), ("frames", C.c_int32), ("i", C.c_size_t), ("n", C.c_size_t), ("N", C.c_size_t),
                ("width", C.c_int32), ("height", C.c_int32), ("buffer", C.c_void_p)]


def set_format_variants(invert_endian, hz_as_integer):
    """process-wide: the reference's DBDE_INVERT_ENDIAN / DBDE_HZ_AS_INTEGER build variants (the C++
    drop-in functions follow it on every call; contexts created afterwards start with it)"""
    load().dbde_b200_set_format_variants(int(bool(invert_endian)), int(bool(hz_as_integer)))


def get_format_variants():
    a, b = C.c_int(0), C.c_int(0)
    load().dbde_b200_get_format_variants(C.byref(a), C.byref(b))
    return bool(a.value), bool(b.value)


class DropIn:
    """dbde_util.h through the C++ symbols of libdbde_b200.so."""

    def __init__(self):
        lib = self.lib = load()
        g = lambda n: getattr(lib, CXX_SYMBOLS[n])
        self._pack_frame = g("dbde_pack_frame"); self._pack_frame.restype = C.c_size_t
        self._pack_frame.argtypes = [C.c_uint64, _u8p, C.c_int, C.c_int, _u8p]
        self._pack_image = g("dbde_pack_image"); self._pack_image.restype = C.c_size_t
        self._pack_image.argtypes = [_u8p, C.c_int, C.c_int, _u8p]
        self._unpack_image = g("dbde_unpack_image"); self._unpack_image.restype = C.c_size_t
        self._unpack_image.argtypes = [_u8p, C.c_int, C.c_int, _u8p]
        self._unpack_frame = g("dbde_unpack_frame"); self._unpack_frame.restype = _FrameHeader
        self._unpack_frame.argtypes = [C.POINTER(_u8p), C.c_int, C.c_int, _u8p]
        self._pack_fh = g("dbde_pack_frame_header"); self._pack_fh.restype = C.c_size_t
        self._pack_fh.argtypes = [_FrameHeader, _u8p]
        self._pack_vh = g("dbde_pack_video_header"); self._pack_vh.restype = C.c_size_t
        self._pack_vh.argtypes = [_VideoHeader, _u8p]
        self._unpack_fh = g("dbde_unpack_frame_header"); self._unpack_fh.restype = _FrameHeader
        self._unpack_fh.argtypes = [C.POINTER(_u8p)]
        self._unpack_vh = g("dbde_unpack_video_header"); self._unpack_vh.restype = _VideoHeader
        self._unpack_vh.argtypes = [C.POINTER(_u8p)]
        self._pack_8x8 = g("dbde_pack_8x8"); self._pack_8x8.restype = C.c_uint32
        self._pack_8x8.argtypes = [_u8p, C.c_int, _u8p]
        self._pack_8x8_partial = g("dbde_pack_8x8_partial"); self._pack_8x8_partial.restype = C.c_uint32
        self._pack_8x8_partial.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, _u8p]
        self._unpack_8x8 = g("dbde_unpack_8x8"); self._unpack_8x8.restype = None
        self._unpack_8x8.argtypes = [C.c_uint8, C.c_uint8, _u8p, C.c_size_t, _u8p]
        self._unpack_8x8_partial = g("dbde_unpack_8x8_partial"); self._unpack_8x8_partial.restype = None
        self._unpack_8x8_partial.argtypes = [C.c_uint8, C.c_uint8, _u8p, C.c_size_t, C.c_int, C.c_int, _u8p]
        self._start = g("dbde_start_file_walk"); self._start.restype = _Walker
        self._start.argtypes = [C.c_char_p, C.c_int, C.POINTER(_VideoHeader)]
        self._walk = g("dbde_walk_a_file"); self._walk.restype = C.c_bool
        self._walk.argtypes = [C.POINTER(_Walker), C.POINTER(_FrameHeader), _u8p]
        self._end = g("dbde_end_file_walk"); self._end.restype = None
        self._end.argtypes = [C.POINTER(_Walker)]

    @staticmethod
    def _p(a):
        return a.ctypes.data_as(_u8p)

    def bound(self, W, H):
        return 32 + 66 * ((W + 7) // 8) * ((H + 7) // 8)

    def pack_frame(self, index, img):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        H, W = img.shape
        out = np.zeros(self.bound(W, H) + 64, dtype=np.uint8)
        n = self._pack_frame(index, self._p(img), W, H, self._p(out))
        return out[:n].copy()

    def pack_image(self, img):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        H, W = img.shape
        out = np.zeros(self.bound(W, H) + 64, dtype=np.uint8)
        n = self._pack_image(self._p(img), W, H, self._p(out))
        return out[:n].copy()

    def unpack_image(self, packed, W, H, fill=0xCD):
        pad = np.concatenate([np.ascontiguousarray(packed, dtype=np.uint8), np.zeros(80, dtype=np.uint8)])
        img = np.full((H, W), fill, dtype=np.uint8)
        n = self._unpack_image(self._p(pad), W, H, self._p(img))
        return n, img

    def unpack_frame(self, packed, W, H, fill=0xCD):
        pad = np.concatenate([np.ascontiguousarray(packed, dtype=np.uint8), np.zeros(80, dtype=np.uint8)])
        img = np.full((H, W), fill, dtype=np.uint8)
        pp = self._p(pad)
        start = C.addressof(pp.contents)
        fh = self._unpack_frame(C.byref(pp), W, H, self._p(img))
        used = C.addressof(pp.contents) - start
        return used, (fh.u64s, fh.index, fh.elapsed_ns), img

    def pack_frame_header(self, u64s, index, elapsed_ns):
        out = np.zeros(20, dtype=np.uint8)
        assert self._pack_fh(_FrameHeader(u64s, index, elapsed_ns), self._p(out)) == 20
        return out

    def pack_video_header(self, u64s, height, width, hz):
        out = np.zeros(28, dtype=np.uint8)
        assert self._pack_vh(_VideoHeader(u64s, height, width, hz), self._p(out)) == 28
        return out

    def unpack_video_header(self, packed):
        buf = np.ascontiguousarray(packed, dtype=np.uint8).copy()
        pp = self._p(buf)
        start = C.addressof(pp.contents)
        vh = self._unpack_vh(C.byref(pp))
        return C.addressof(pp.contents) - start, (vh.u64s, vh.height, vh.width, vh.frame_hz)

    def pack_8x8(self, tile):
        t = np.ascontiguousarray(tile, dtype=np.uint8).reshape(8, 8)
        out = np.full(64 + 16, 0xA5, dtype=np.uint8)
        r = self._pack_8x8(self._p(t), 8, self._p(out))
        k = r >> 8
        assert (out[8 * k:] == 0xA5).all(), "wrote past 8*depth bytes"
        return r, out[:8 * k].copy()

    def pack_8x8_partial(self, tile, rm, dm):
        t = np.ascontiguousarray(tile, dtype=np.uint8).reshape(8, 8)
        out = np.zeros(64, dtype=np.uint8)
        r = self._pack_8x8_partial(self._p(t), 8, rm, dm, self._p(out))
        return r, out[:8 * (r >> 8)].copy()

    def unpack_8x8(self, depth, minval, payload, stride=8):
        pay = np.concatenate([np.ascontiguousarray(payload, dtype=np.uint8), np.zeros(64, dtype=np.uint8)])
        img = np.zeros((8, stride), dtype=np.uint8)
        self._unpack_8x8(depth, minval, self._p(pay), stride, self._p(img))
        return img[:, :8].copy()

    def unpack_8x8_partial(self, depth, minval, payload, rm, dm, fill=0xCD):
        pay = np.concatenate([np.ascontiguousarray(payload, dtype=np.uint8), np.zeros(64, dtype=np.uint8)])
        img = np.full((8, 8), fill, dtype=np.uint8)
        self._unpack_8x8_partial(depth, minval, self._p(pay), 8, rm, dm, self._p(img))
        return img

    def walk_open(self, path, frames_buffered=4):
        """dbde_start_file_walk -> (walker struct, video header tuple) for stepwise use with walk_next / walk_close"""
        vh = _VideoHeader()
        w = self._start(path.encode(), frames_buffered, C.byref(vh))
        return w, (vh.u64s, vh.height, vh.width, vh.frame_hz)

    def walk_next(self, w):
        """dbde_walk_a_file -> (frame header tuple, image) or None at the end"""
        img = np.zeros((w.height, w.width), dtype=np.uint8)
        fh = _FrameHeader()
        if not self._walk(C.byref(w), C.byref(fh), self._p(img)):
            return None
        return (fh.u64s, fh.index, fh.elapsed_ns), img

    def walk_close(self, w):
        self._end(C.byref(w))

    def walk_file(self, path, frames_buffered=4):
        """-> (video header tuple, [(frame header tuple, image)])"""
        vh = _VideoHeader()
        w = self._start(path.encode(), frames_buffered, C.byref(vh))
        out = []
        if not w.fptr:
            return None, out
        img = np.zeros((w.height, w.width), dtype=np.uint8)
        fh = _FrameHeader()
        while self._walk(C.byref(w), C.byref(fh), self._p(img)):
            out.append(((fh.u64s, fh.index, fh.elapsed_ns), img.copy()))
        self._end(C.byref(w))
        return (vh.u64s, vh.height, vh.width, vh.frame_hz), out
