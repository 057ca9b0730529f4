"""ctypes bindings for the DBDE checkers -- TEST / BENCH INFRASTRUCTURE ONLY.

`oracle.port`  : liboracle.so, the plain-C restatement (oracle/dbde_oracle.c).
`oracle.ref`   : oracle/_ref/libdbde_ref.so, the UNMODIFIED reference (dbde_util.cpp) behind
                 ref_shim.cpp, or None when it has not been built.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this package; the product (dbce-video-cpp_b200/) never does.
"""
import ctypes as C
import os
import subprocess
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

_u8p = C.POINTER(C.c_uint8)
_u64p = C.POINTER(C.c_uint64)


def build(verbose=False):
    """Compile the checkers (make -C oracle).  Building the checker is not using it."""
    r = subprocess.run(["make", "-C", HERE], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("oracle build failed")


def _ptr(a):
    return a.ctypes.data_as(_u8p)


def frame_record_bound(W, H):
    wh = ((W + 7) // 8) * ((H + 7) // 8)
    return 32 + 66 * wh


class _Codec:
    """Common python face over either shared library (prefix 'oracle_' or 'ref_')."""

    def __init__(self, lib, prefix):
        self.lib, self.prefix = lib, prefix
        f = lambda n: getattr(lib, prefix + n)
        self._pack_image = f("pack_image"); self._pack_image.restype = C.c_size_t
        self._pack_image.argtypes = [_u8p, C.c_int, C.c_int, _u8p]
        self._pack_frame = f("pack_frame"); self._pack_frame.restype = C.c_size_t
        self._pack_frame.argtypes = [C.c_uint64, _u8p, C.c_int, C.c_int, _u8p]
        self._pack_frames = f("pack_frames"); self._pack_frames.restype = C.c_size_t
        self._pack_frames.argtypes = [_u8p, C.c_int, C.c_int, C.c_uint64, C.c_int, _u8p, _u64p]
        self._unpack_image = f("unpack_image"); self._unpack_image.restype = C.c_size_t
        self._unpack_image.argtypes = [_u8p, C.c_int, C.c_int, _u8p]
        self._unpack_frame = f("unpack_frame"); self._unpack_frame.restype = C.c_size_t
        self._unpack_frame.argtypes = [_u8p, C.c_int, C.c_int, _u8p, _u64p]
        self._pack_fh = f("pack_frame_header"); self._pack_fh.restype = C.c_size_t
        self._pack_fh.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64, _u8p]
        self._pack_vh = f("pack_video_header"); self._pack_vh.restype = C.c_size_t
        self._pack_vh.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64, C.c_double, _u8p]
        self._unpack_vh = f("unpack_video_header"); self._unpack_vh.restype = C.c_size_t
        self._unpack_vh.argtypes = [_u8p, _u64p, C.POINTER(C.c_double)]
        self._pack_8x8 = f("pack_8x8"); self._pack_8x8.restype = C.c_uint32
        self._pack_8x8.argtypes = [_u8p, C.c_int, _u8p]
        self._pack_8x8_partial = f("pack_8x8_partial"); self._pack_8x8_partial.restype = C.c_uint32
        self._pack_8x8_partial.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, _u8p]

    def pack_8x8(self, tile):
        t = np.ascontiguousarray(tile, dtype=np.uint8).reshape(8, 8)
        out = np.full(64 + 16, 0xA5, dtype=np.uint8)       # sentinel tail
        r = self._pack_8x8(_ptr(t), 8, _ptr(out))
        k = r >> 8
        assert (out[8 * k:] == 0xA5).all(), "wrote past 8*depth bytes"
        return r, out[:8 * k].copy()

    def pack_8x8_partial(self, tile, rm, dm):
        t = np.ascontiguousarray(tile, dtype=np.uint8).reshape(8, 8)
        out = np.zeros(64, dtype=np.uint8)
        r = self._pack_8x8_partial(_ptr(t), 8, rm, dm, _ptr(out))
        return r, out[:8 * (r >> 8)].copy()

    def pack_image(self, img):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        H, W = img.shape
        out = np.zeros(frame_record_bound(W, H) + 64, dtype=np.uint8)
        n = self._pack_image(_ptr(img), W, H, _ptr(out))
        return out[:n].copy()

    def pack_frame(self, index, img):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        H, W = img.shape
        out = np.zeros(frame_record_bound(W, H) + 64, dtype=np.uint8)
        n = self._pack_frame(index, _ptr(img), W, H, _ptr(out))
        return out[:n].copy()

    def pack_frames(self, frames, first_index=0):
        """frames: (N,H,W) u8 -> (stream bytes, sizes[N])"""
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        N, H, W = frames.shape
        out = np.zeros(N * frame_record_bound(W, H) + 64, dtype=np.uint8)
        sizes = np.zeros(N, dtype=np.uint64)
        n = self._pack_frames(_ptr(frames), W, H, first_index, N, _ptr(out), sizes.ctypes.data_as(_u64p))
        return out[:n].copy(), sizes

    def unpack_image(self, packed, W, H, fill=0xCD):
        """-> (bytes consumed (0 = rejected), image)"""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        pad = np.concatenate([packed, np.zeros(80, dtype=np.uint8)])
        img = np.full((H, W), fill, dtype=np.uint8)
        n = self._unpack_image(_ptr(pad), W, H, _ptr(img))
        return n, img

    def unpack_frame(self, packed, W, H, fill=0xCD):
        """-> (bytes consumed, (u64s, index, elapsed_ns), image)"""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        pad = np.concatenate([packed, np.zeros(80, dtype=np.uint8)])
        img = np.full((H, W), fill, dtype=np.uint8)
        hdr = np.zeros(3, dtype=np.uint64)
        n = self._unpack_frame(_ptr(pad), W, H, _ptr(img), hdr.ctypes.data_as(_u64p))
        return n, tuple(int(x) for x in hdr), img

    def unpack_frames(self, stream, W, H, N):
        """Decode N back-to-back frame records -> (frames (N,H,W), indices, consumed)."""
        frames = np.zeros((N, H, W), dtype=np.uint8)
        idx = []
        off = 0
        for i in range(N):
            n, hdr, img = self.unpack_frame(stream[off:], W, H)
            if hdr[0] != 2:
                return None, idx, off
            frames[i] = img
            idx.append(hdr[1])
            off += n
        return frames, idx, off

    def pack_frame_header(self, u64s, index, elapsed_ns):
        out = np.zeros(20, dtype=np.uint8)
        assert self._pack_fh(u64s, index, elapsed_ns, _ptr(out)) == 20
        return out

    def pack_video_header(self, u64s, height, width, hz):
        out = np.zeros(28, dtype=np.uint8)
        assert self._pack_vh(u64s, height, width, float(hz), _ptr(out)) == 28
        return out

    def unpack_video_header(self, packed):
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        u = np.zeros(3, dtype=np.uint64)
        hz = C.c_double(0)
        n = self._unpack_vh(_ptr(packed), u.ctypes.data_as(_u64p), C.byref(hz))
        return n, (int(u[0]), int(u[1]), int(u[2]), hz.value)


def _load(path):
    return C.CDLL(path) if os.path.exists(path) else None


_port_lib = _load(os.path.join(HERE, "liboracle.so"))
if _port_lib is None:
    build()
    _port_lib = _load(os.path.join(HERE, "liboracle.so"))
port = _Codec(_port_lib, "oracle_")

_ref_lib = _load(os.path.join(HERE, "_ref", "libdbde_ref.so"))
ref = _Codec(_ref_lib, "ref_") if _ref_lib is not None else None

# The reference built with -DDBDE_INVERT_ENDIAN -DDBDE_HZ_AS_INTEGER (its two compile-time format
# variants, SURVEY 8 f-3), and a second instance of the port switched to the same variants.
_refv_lib = _load(os.path.join(HERE, "_ref", "libdbde_ref_variants.so"))
ref_variants = _Codec(_refv_lib, "ref_") if _refv_lib is not None else None


def port_variants():
    """A private copy of the port with both variants on (the flag is a global of the library, so the
    copy is loaded from its own file to leave `port` untouched)."""
    import shutil
    import tempfile
    d = tempfile.mkdtemp(prefix="dbde_oracle_")
    path = os.path.join(d, "liboracle_variants.so")
    shutil.copy(os.path.join(HERE, "liboracle.so"), path)
    lib = C.CDLL(path)
    lib.oracle_set_variants.argtypes = [C.c_int, C.c_int]
    lib.oracle_set_variants(1, 1)
    return _Codec(lib, "oracle_")


class _Codec16:
    """DBDE16 (SURVEY 8 f-4), the 16-bit extension: defined by the port only -- the reference has no
    such code, so there is no compiled-reference counterpart ("parity unpinned")."""

    def __init__(self, lib):
        self.lib = lib
        lib.oracle_frame_record_bound16.restype = C.c_size_t
        lib.oracle_frame_record_bound16.argtypes = [C.c_int, C.c_int]
        lib.oracle_pack_frames16.restype = C.c_size_t
        lib.oracle_pack_frames16.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_int, _u8p, _u64p]
        lib.oracle_unpack_frame16.restype = C.c_size_t
        lib.oracle_unpack_frame16.argtypes = [_u8p, C.c_int, C.c_int, C.c_void_p, _u64p]

    def bound(self, W, H):
        return int(self.lib.oracle_frame_record_bound16(W, H))

    def pack_frames(self, frames, first_index=0):
        """frames: (N,H,W) u16 -> (stream bytes, sizes[N])"""
        frames = np.ascontiguousarray(frames, dtype=np.uint16)
        N, H, W = frames.shape
        out = np.zeros(N * self.bound(W, H) + 64, dtype=np.uint8)
        sizes = np.zeros(N, dtype=np.uint64)
        n = self.lib.oracle_pack_frames16(frames.ctypes.data, W, H, first_index, N, _ptr(out), sizes.ctypes.data_as(_u64p))
        return out[:n].copy(), sizes

    def unpack_frame(self, packed, W, H, fill=0xCDCD):
        """-> (bytes consumed, (u64s, index, elapsed_ns), image u16)"""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        pad = np.concatenate([packed, np.zeros(160, dtype=np.uint8)])
        img = np.full((H, W), fill, dtype=np.uint16)
        hdr = np.zeros(3, dtype=np.uint64)
        n = self.lib.oracle_unpack_frame16(_ptr(pad), W, H, img.ctypes.data, hdr.ctypes.data_as(_u64p))
        return n, tuple(int(x) for x in hdr), img


port16 = _Codec16(_port_lib)


def best():
    """The strongest checker available: the compiled reference, else the port."""
    return ref if ref is not None else port


def best_variants():
    return ref_variants if ref_variants is not None else port_variants()


if _ref_lib is not None:
    _ref_lib.ref_encode_mt.restype = C.c_double
    _ref_lib.ref_encode_mt.argtypes = [_u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p, C.c_size_t, _u64p]
    _ref_lib.ref_decode_mt.restype = C.c_double
    _ref_lib.ref_decode_mt.argtypes = [_u8p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p,
                                       C.POINTER(C.c_int)]


def ref_encode_mt(frames, threads, reps=1):
    """Time the unmodified reference's dbde_pack_frame over `threads` std::threads.
    -> (seconds, slots (N,slot) u8, sizes)"""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    N, H, W = frames.shape
    slot = (frame_record_bound(W, H) + 63) // 64 * 64
    slots = np.zeros((N, slot), dtype=np.uint8)
    sizes = np.zeros(N, dtype=np.uint64)
    s = _ref_lib.ref_encode_mt(_ptr(frames), W, H, N, threads, reps, _ptr(slots), slot, sizes.ctypes.data_as(_u64p))
    return s, slots, sizes


def ref_decode_mt(slots, W, H, threads, reps=1):
    slots = np.ascontiguousarray(slots, dtype=np.uint8)
    N, slot = slots.shape
    frames = np.zeros((N, H, W), dtype=np.uint8)
    bad = C.c_int(0)
    s = _ref_lib.ref_decode_mt(_ptr(slots), slot, W, H, N, threads, reps, _ptr(frames), C.byref(bad))
    return s, frames, bad.value


def _fan_out(n, threads, work):
    """work(a, b) over `threads` contiguous ranges of range(n) on host threads (ctypes releases the GIL
    during each call into the library) -> the sum of what the calls return"""
    from concurrent.futures import ThreadPoolExecutor
    threads = max(1, min(threads, n))
    with ThreadPoolExecutor(threads) as ex:
        return sum(ex.map(lambda t: work(n * t // threads, n * (t + 1) // threads), range(threads)))


def port_encode_mt(frames, threads, reps=1):
    """ref_encode_mt with the port's pack_frame: the CPU baseline where oracle/_ref is not built.
    -> (seconds, slots (N,slot) u8, sizes)"""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    N, H, W = frames.shape
    slot = (frame_record_bound(W, H) + 63) // 64 * 64
    slots = np.zeros((N, slot), dtype=np.uint8)
    sizes = np.zeros(N, dtype=np.uint64)

    def work(a, b):
        for i in range(a, b):
            sizes[i] = port._pack_frame(i, _ptr(frames[i]), W, H, _ptr(slots[i]))
        return 0

    t0 = time.perf_counter()
    for _ in range(reps):
        _fan_out(N, threads, work)
    return time.perf_counter() - t0, slots, sizes


def port_decode_mt(slots, W, H, threads, reps=1):
    """ref_decode_mt with the port's unpack_frame -> (seconds, frames, records rejected over all reps)"""
    slots = np.ascontiguousarray(slots, dtype=np.uint8)
    N, slot = slots.shape
    frames = np.zeros((N, H, W), dtype=np.uint8)

    def work(a, b):
        hdr = np.zeros(3, dtype=np.uint64)
        bad = 0
        for i in range(a, b):
            port._unpack_frame(_ptr(slots[i]), W, H, _ptr(frames[i]), hdr.ctypes.data_as(_u64p))
            bad += int(hdr[0]) != 2
        return bad

    t0 = time.perf_counter()
    bad = sum(_fan_out(N, threads, work) for _ in range(reps))
    return time.perf_counter() - t0, frames, bad
