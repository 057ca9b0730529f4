"""Region-of-interest decode (dbde_b200_decode_roi_*, dbde_b200_reader_set_roi) on a B200: the output is the
crop of the full decode (the oracle's, which equals the source frames) byte for byte, validation covers the
whole record with the full decoder's status bits, and nothing outside the output range is written."""
import hashlib
import importlib
import os
import tempfile

import numpy as np
import pytest

import oracle
import synth
from conftest import rand_frame

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()
E_INVALID = -1

GEOMETRIES = [(2048, 2048), (2304, 48), (1280, 64), (4096, 8), (4104, 16), (2049, 9), (4100, 1003), (1001, 1003),
              (17, 23), (3, 5), (1, 1)]


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


def content(W, H):
    """rand_frame styles (every depth 0-8 inside one warp with 'classes') and synthetic mix / low / noise video"""
    rng = np.random.default_rng(W * 7919 + H)
    fr = [rand_frame(rng, W, H, s) for s in ("classes", "noise", "flat")]
    for i, kind in enumerate(("mix", "low", "noise")):
        fr.append(synth.gen_frames(kind, 1, W, H, f0=i)[0])
    return np.stack(fr)


def regions(W, H):
    w, h = (W + 7) // 8, (H + 7) // 8
    R = {(0, 0, W, H), (0, 0, 1, 1), (W - 1, H - 1, 1, 1), (W // 2, H // 2, 1, 1)}
    if W > 2 and H > 2:
        R.add((1, 1, W - 2, H - 2))
    if W > 1:
        R |= {(1, 0, W - 1, H), (0, 0, W - 1, H)}
    if H > 1:
        R |= {(0, 1, W, H - 1), (0, 0, W, H - 1)}
    tx, ty = (w - 1) // 2, (h - 1) // 2                         # one exact tile
    R.add((8 * tx, 8 * ty, min(8, W - 8 * tx), min(8, H - 8 * ty)))
    R.add((8 * (w - 1), 0, W - 8 * (w - 1), H))                 # the partial last tile column / row
    R.add((0, 8 * (h - 1), W, H - 8 * (h - 1)))
    R.add((max(0, W - 13), max(0, H - 11), min(W, 13), min(H, 11)))
    for x in sorted({0, W // 3, W - 1}):                         # 1-pixel columns and rows
        R.add((x, 0, 1, H))
    for y in sorted({0, H // 2, H - 1}):
        R.add((0, y, W, 1))
    # around 32-tile item and 256-tile partition boundaries of the row-major tile order, and tile column 32 / 256
    for t in (31, 32, 255, 256, 257, 511, 512, 4095, 4096):
        if t < w * h:
            ty, tx = divmod(t, w)
            x0, y0 = max(0, 8 * tx - 19), max(0, 8 * ty - 5)
            R.add((x0, y0, min(W - x0, 45), min(H - y0, 13)))
    for tc in (32, 256):
        if w > tc + 1:
            R.add((8 * tc - 3, 0, 20, H))
            x0 = 8 * (tc - 33) + 5 if tc >= 33 else 5
            R.add((x0, H // 3, min(W - x0, 8 * 40 + 3), min(H - H // 3, 9)))
    # every x0 mod 8 crossed with every roi_w mod 8, within a tile, across a few tiles, across more than 32 tiles
    for a in range(8):
        for b in range(8):
            for m in (0, 2, 35):
                rw = b + 8 * m if b + 8 * m > 0 else 8
                if a + rw > W:
                    continue
                q = (a + b + m) % ((W - rw - a) // 8 + 1)
                y0 = (5 * a + 3 * b + m) % H
                R.add((a + 8 * q, y0, rw, min(H - y0, 1 + (a + 2 * b + m) % 19)))
    for r in R:
        x0, y0, rw, rh = r
        assert x0 >= 0 and y0 >= 0 and rw >= 1 and rh >= 1 and x0 + rw <= W and y0 + rh <= H, (W, H, r)
    return sorted(R)


def crop(frames, r):
    x0, y0, rw, rh = r
    return frames[:, y0:y0 + rh, x0:x0 + rw]


class DevStream:
    """records (and their offsets) uploaded once, plus a guarded output buffer"""
    G = 32

    def __init__(self, codec, stream, offs, N, out_bytes):
        self.codec, self.N = codec, N
        self.d_s = codec.device_alloc(len(stream) + 64)
        self.d_o = codec.device_alloc(8 * N)
        self.d_st = codec.device_alloc(4 * N)
        self.d_ix = codec.device_alloc(8 * N)
        self.cap = out_bytes + 2 * self.G + 16
        self.d_out = codec.device_alloc(self.cap)
        self.nbytes = len(stream)
        codec.h2d(self.d_s, stream)
        codec.h2d(self.d_o, np.ascontiguousarray(offs[:N], dtype=np.uint64))

    def roi(self, r, shift=0, fill=0xA7):
        """decode_roi_device at output base offset `shift`; checks the guards -> (frames, status, indices)"""
        c, N, G = self.codec, self.N, self.G
        x0, y0, rw, rh = r
        n = N * rw * rh
        c.h2d(self.d_out, np.full(n + 2 * G + 16, fill, dtype=np.uint8))
        c.decode_roi_device(self.d_s, self.nbytes, self.d_o, self.W, self.H, N, r, self.d_out + G + shift, self.d_st, self.d_ix)
        buf = c.d2h(self.d_out, n + 2 * G + 16)
        assert (buf[:G + shift] == fill).all() and (buf[G + shift + n:] == fill).all(), ("wrote outside the output", r, shift)
        return (buf[G + shift:G + shift + n].reshape(N, rh, rw), c.d2h(self.d_st, 4 * N, np.uint32),
                c.d2h(self.d_ix, 8 * N, np.uint64))

    def free(self):
        for p in (self.d_s, self.d_o, self.d_st, self.d_ix, self.d_out):
            self.codec.device_free(p)


def dev_stream(codec, stream, offs, N, W, H):
    d = DevStream(codec, stream, offs, N, N * W * H)
    d.W, d.H = W, H
    return d


@pytest.mark.parametrize("W,H", GEOMETRIES)
def test_regions_equal_the_crop_of_the_full_decode(codec, W, H):
    """every kind of region on every geometry class (aligned, linear partitions, band segments, odd and wide odd,
    tiny), at output base offsets 0-15 with guard bytes on both sides"""
    fr = content(W, H)
    N = len(fr)
    stream, sizes = ORA.pack_frames(fr, 11)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    full, idx, _ = ORA.unpack_frames(stream, W, H, N)
    assert (full == fr).all() and idx == list(range(11, 11 + N))
    d = dev_stream(codec, stream, offs, N, W, H)
    try:
        for i, r in enumerate(regions(W, H)):
            got, status, index = d.roi(r, shift=i % 16)
            assert (status == 0).all() and index.tolist() == list(range(11, 11 + N)), r
            want = crop(full, r)
            if not np.array_equal(got, want):
                bad = np.argwhere(got != want)[0]
                pytest.fail("region %r of %dx%d differs first at (frame, row, col) %r" % (r, W, H, tuple(bad)))
    finally:
        d.free()


def test_damage_outside_the_region_is_rejected_like_the_full_decode(codec):
    """the damage of the full decoder's invalid-stream test, all of it outside the region: the same status bits as
    decode_host, the region of a rejected frame keeps its fill, good frames of the batch still decode"""
    W, H, N = 48, 40, 7
    wh = 6 * 5
    r = (17, 9, 13, 11)                          # tiles (2..3, 1..2)
    outside = 4 * 6 + 5                          # tile (5, 4): not in the region
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    bad = stream.copy()
    bad[int(offs[1]) + 20] += 1                 # nb != wh
    bad[int(offs[2]) + 24 + wh] += 1            # nm != wh
    bad[int(offs[3]) + 28 + 2 * wh] += 1        # n64 != sum(depth)
    bad[int(offs[4])] = 9                       # frame tag != 2
    bad[int(offs[5]) + 24 + outside] = 9        # a depth byte > 8
    cases = [(bad, offs[:N]), (stream[:int(offs[N]) - 8], offs[:N])]                 # + a truncated last record
    for s, o in cases:
        _, want_status, want_idx = codec.decode_host(s, o, W, H, fill=0xCD)
        assert want_status.any()
        got, status, index = codec.decode_roi_host(s, o, W, H, r, fill=0xCD)
        assert status.tolist() == want_status.tolist() and index.tolist() == want_idx.tolist()
        d = dev_stream(codec, s, o, N, W, H)
        try:
            dgot, dstatus, _ = d.roi(r, shift=5, fill=0xCD)
        finally:
            d.free()
        assert dstatus.tolist() == want_status.tolist()
        for i in range(N):
            if status[i]:
                assert (got[i] == 0xCD).all() and (dgot[i] == 0xCD).all(), i
            else:
                assert (got[i] == crop(fr, r)[i]).all() and (dgot[i] == crop(fr, r)[i]).all(), i
    assert codec.decode_roi_host(bad, offs[:N], W, H, r)[1][5] & pkg.ST_DEPTH_TOO_BIG


@pytest.mark.parametrize("W,H", [(64, 40), (1001, 43), (2048, 16), (4104, 16), (2049, 9), (10, 10)])
def test_invert_endian_variant(codec, W, H):
    """DBDE_INVERT_ENDIAN (dbde_util.cpp:15-19,246-270) records, against the reference built with the macro where it
    is built and the port's variant otherwise"""
    V = oracle.best_variants()
    rng = np.random.default_rng(W + 31 * H)
    fr = np.stack([rand_frame(rng, W, H, ["classes", "noise", "classes"][i % 3]) for i in range(3)])
    want, sizes = V.pack_frames(fr, 9)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    c = pkg.Codec(0)
    try:
        c.set_invert_endian(True)
        for r in [(0, 0, W, H), (3, 1, W - 5, H - 2), (W // 2, H // 3, W - W // 2, 1), (1, 0, 1, H)]:
            got, status, _ = c.decode_roi_host(want, offs[:3], W, H, r)
            assert (status == 0).all() and (got == crop(fr, r)).all(), r
        plain, _, _ = codec.decode_roi_host(want, offs[:3], W, H, (3, 1, W - 5, H - 2))
        assert not np.array_equal(plain, crop(fr, (3, 1, W - 5, H - 2)))
    finally:
        c.close()


def test_host_form_pinned_pageable_and_chunked(codec):
    """decode_roi_host on pageable numpy and pinned buffers, several chunks in flight: equal to the device form"""
    W, H, N = 1001, 203, 10
    fr = synth.gen_frames("mix", N, W, H, f0=4)
    stream, offs = codec.encode_host(fr, 3)
    r = (333, 17, 401, 150)
    x0, y0, rw, rh = r
    d = dev_stream(codec, stream, offs, N, W, H)
    try:
        dev, dstatus, _ = d.roi(r, shift=3)
    finally:
        d.free()
    assert (dstatus == 0).all() and (dev == crop(fr, r)).all()
    c = pkg.Codec(0)
    try:
        c.set_chunk_frames(3)
        got, status, index = c.decode_roi_host(stream, offs[:N], W, H, r)
        assert (status == 0).all() and index.tolist() == list(range(3, 3 + N)) and (got == dev).all()
        ps, po, pf = c.pinned(len(stream)), c.pinned(8 * N), c.pinned(N * rw * rh + 1)
        pst, pix = c.pinned(4 * N), c.pinned(8 * N)
        try:
            ps.array[:] = stream
            po.array[:] = offs[:N].view(np.uint8)
            pf.array[:] = 0
            assert c.lib.dbde_b200_decode_roi_host(c.h, ps.ptr, len(stream), po.ptr, W, H, N, x0, y0, rw, rh, pf.ptr + 1,
                                                   pst.ptr, pix.ptr) == 0
            assert (pst.array.view(np.uint32) == 0).all() and pf.array[0] == 0
            assert (pf.array[1:].reshape(N, rh, rw) == dev).all()
        finally:
            for p in (ps, po, pf, pst, pix):
                p.free()
    finally:
        c.close()


def test_file_reader_region(codec):
    """read_file(roi=...) equals the crop of read_file; the region can change between reader_next calls; a bad
    record still stops the read"""
    W, H, N = 264, 40, 23
    fr = synth.gen_frames("mix", N, W, H, f0=2)
    r = (13, 5, 100, 30)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "v.dbde")
        pkg.write_file(codec, path, fr, batch=7)
        _, full, idx, st = pkg.read_file(codec, path, batch=5)
        assert (st == 0).all() and (full == fr).all()
        _, part, pidx, pst = pkg.read_file(codec, path, batch=5, roi=r)
        assert (pst == 0).all() and pidx.tolist() == idx.tolist() and (part == crop(full, r)).all()
        # switch the region between batches: (r, whole frame, another region, r)
        lib = codec.lib
        import ctypes as C
        rd, w_, h_, hz = C.c_void_p(), C.c_int(), C.c_int(), C.c_double()
        assert lib.dbde_b200_reader_open(codec.h, path.encode(), 6, C.byref(w_), C.byref(h_), C.byref(hz), C.byref(rd)) == 0
        try:
            pos = 0
            for rr in [r, (0, 0, W, H), (200, 33, 64, 7), r, (7, 0, 1, H)]:
                assert lib.dbde_b200_reader_set_roi(rd, *rr) == 0
                out = np.full((6, rr[3], rr[2]), 0xCD, dtype=np.uint8)
                ii, ss = np.zeros(6, np.uint64), np.zeros(6, np.uint32)
                n = lib.dbde_b200_reader_next(rd, out.ctypes.data, 6, ii.ctypes.data, ss.ctypes.data)
                assert n == min(6, N - pos) and (ss[:n] == 0).all()
                assert (out[:n] == crop(fr[pos:pos + n], rr)).all(), rr
                pos += n
            assert pos == N
            assert lib.dbde_b200_reader_set_roi(rd, 0, 0, W + 1, H) == E_INVALID
        finally:
            lib.dbde_b200_reader_close(rd)
        # a damaged record stops the read after it, as without a region
        raw = bytearray(open(path, "rb").read())
        offs = codec.index_stream(np.frombuffer(bytes(raw[28:]), dtype=np.uint8), W, H)
        raw[28 + int(offs[9])] = 9                                             # frame tag != 2
        with open(path, "wb") as f:
            f.write(raw)
        _, part, pidx, pst = pkg.read_file(codec, path, batch=4, roi=r)
        assert len(part) == 10 and (pst[:9] == 0).all() and pst[9] & pkg.ST_BAD_FRAME_HEADER
        assert (part[:9] == crop(fr[:9], r)).all() and (part[9] == 0xCD).all()


def test_scale_1000_frames_micro_2048(codec):
    """1000 frames of 2048^2 'micro' in HBM: a 512x384 region at (517, 301) equals the crop of the full GPU decode
    (SHA-256 over all frames)"""
    N, W, H = 1000, 2048, 2048
    px = W * H
    r = (517, 301, 512, 384)
    x0, y0, rw, rh = r
    wh = (W // 8) * (H // 8)
    cap = codec.stream_bound(W, H, N)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    d_fr, d_out = codec.device_alloc(N * px), codec.device_alloc(cap + 64)
    d_off, d_sz, d_st, d_st2 = (codec.device_alloc(8 * N), codec.device_alloc(8 * N), codec.device_alloc(4 * N),
                                codec.device_alloc(4 * N))
    d_roi = codec.device_alloc(N * rw * rh)
    try:
        synth.gen_frames_device("micro", N, W, H, d_fr, seed=42, f0=0)
        codec.encode_device(d_fr, W, H, 0, N, d_out + delta, cap, d_off, d_sz)
        codec.decode_roi_device(d_out + delta, cap, d_off, W, H, N, r, d_roi, d_st2)
        codec.decode_device(d_out + delta, cap, d_off, W, H, N, d_fr, d_st)      # the full decode over the source frames
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all() and (codec.d2h(d_st2, 4 * N, np.uint32) == 0).all()
        h_full, h_roi = hashlib.sha256(), hashlib.sha256()
        step = 50
        for a in range(0, N, step):
            full = codec.d2h(d_fr + a * px, step * px).reshape(step, H, W)
            h_full.update(np.ascontiguousarray(crop(full, r)).tobytes())
        h_roi.update(codec.d2h(d_roi, N * rw * rh).tobytes())
        assert h_roi.hexdigest() == h_full.hexdigest()
    finally:
        for p in (d_fr, d_out, d_off, d_sz, d_st, d_st2, d_roi):
            codec.device_free(p)


def test_bad_arguments(codec):
    """negative, empty and out-of-frame regions and NULL pointers: DBDE_B200_E_INVALID, nothing queued"""
    lib, h = codec.lib, codec.h
    W, H, N = 40, 24, 2
    fr = synth.gen_frames("mix", N, W, H)
    stream, offs = codec.encode_host(fr, 0)
    d = dev_stream(codec, stream, offs, N, W, H)
    st = np.zeros(N, np.uint32)
    out = np.zeros(N * W * H, np.uint8)
    try:
        bad = [(-1, 0, 4, 4), (0, -1, 4, 4), (0, 0, 0, 4), (0, 0, 4, 0), (0, 0, -3, 4), (37, 0, 4, 4), (0, 21, 4, 4),
               (0, 0, W + 1, H), (0, 0, W, H + 1), (W, 0, 1, 1), (0, H, 1, 1), (2**31 - 1, 0, 2**31 - 1, 1)]
        for r in bad:
            assert lib.dbde_b200_decode_roi_device(h, d.d_s, d.nbytes, d.d_o, W, H, N, *r, d.d_out, d.d_st, None, None) == E_INVALID, r
            assert lib.dbde_b200_decode_roi_host(h, stream.ctypes.data, stream.nbytes, offs.ctypes.data, W, H, N, *r,
                                                 out.ctypes.data, st.ctypes.data, None) == E_INVALID, r
            assert lib.dbde_b200_decode_roi_device(h, d.d_s, d.nbytes, d.d_o, W, H, 0, *r, d.d_out, d.d_st, None, None) == E_INVALID, r
        r = (1, 2, 3, 4)
        args = [h, d.d_s, d.nbytes, d.d_o, W, H, N, *r, d.d_out, d.d_st, None, None]
        for i in (0, 1, 3, 11, 12):                                  # ctx, stream, offsets, output, status
            a = list(args)
            a[i] = None
            assert lib.dbde_b200_decode_roi_device(*a) == E_INVALID, i
        hargs = [h, stream.ctypes.data, stream.nbytes, offs.ctypes.data, W, H, N, *r, out.ctypes.data, st.ctypes.data, None]
        for i in (0, 1, 3, 11, 12):
            a = list(hargs)
            a[i] = None
            assert lib.dbde_b200_decode_roi_host(*a) == E_INVALID, i
        assert lib.dbde_b200_decode_roi_device(h, d.d_s, d.nbytes, d.d_o, 0, H, N, 0, 0, 1, 1, d.d_out, d.d_st, None, None) == E_INVALID
        assert lib.dbde_b200_reader_set_roi(None, 0, 0, 1, 1) == E_INVALID
        # the context is still usable, and the last good call decodes
        got, status, _ = codec.decode_roi_host(stream, offs[:N], W, H, r)
        assert (status == 0).all() and (got == crop(fr, r)).all()
    finally:
        d.free()
