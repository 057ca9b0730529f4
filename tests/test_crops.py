"""Crop decode (dbde_b200_decode_crops_*) on a B200: N fixed-size crops per frame at shared or per-frame corners,
anywhere, pixels outside the frame set to a pad byte.  The expected output is a numpy pad-crop of the source frames
(the codec is lossless, so they are the full decode); validation covers the whole record with the full decoder's
status bits, and nothing outside the output range is written."""
import hashlib
import importlib

import numpy as np
import pytest

import oracle
import synth
from conftest import rand_frame

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()
E_INVALID = -1
I32_MIN, I32_MAX = -2**31, 2**31 - 1

GEOMETRIES = [(2048, 2048), (2304, 48), (1280, 64), (4096, 8), (4104, 16), (2049, 9), (4100, 1003), (1001, 1003),
              (17, 23), (3, 5), (1, 1)]


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


def content(W, H):
    """rand_frame styles (every depth 0-8 inside one warp with 'classes') and synthetic mix / low / noise video"""
    rng = np.random.default_rng(W * 7919 + H + 5)
    fr = [rand_frame(rng, W, H, s) for s in ("classes", "noise", "flat")]
    for i, kind in enumerate(("mix", "low", "noise")):
        fr.append(synth.gen_frames(kind, 1, W, H, f0=i)[0])
    return np.stack(fr)


def pad_crop(frames, corners, cw, ch, pad):
    """the reference: frames (N, H, W), corners (R, 2) or (N, R, 2) -> (N, R, ch, cw)"""
    N, H, W = frames.shape
    c = np.broadcast_to(corners, (N,) + corners.shape) if corners.ndim == 2 else corners
    out = np.full((N, c.shape[1], ch, cw), pad, dtype=np.uint8)
    for f in range(N):
        for r in range(c.shape[1]):
            x0, y0 = int(c[f, r, 0]), int(c[f, r, 1])
            xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
            if xa < xb and ya < yb:
                out[f, r, ya - y0:yb - y0, xa - x0:xb - x0] = frames[f, ya:yb, xa:xb]
    return out


class DevStream:
    """records and their offsets uploaded once; crops() decodes into a guarded output buffer"""
    G = 32

    def __init__(self, codec, stream, offs, N, W, H):
        self.codec, self.N, self.W, self.H = codec, N, W, H
        self.d_s = codec.device_alloc(len(stream) + 64)
        self.d_o = codec.device_alloc(8 * N)
        self.d_st = codec.device_alloc(4 * N)
        self.d_ix = codec.device_alloc(8 * N)
        self.nbytes = len(stream)
        codec.h2d(self.d_s, stream)
        codec.h2d(self.d_o, np.ascontiguousarray(offs[:N], dtype=np.uint64))

    def crops(self, corners, size, pad=0, shift=0, fill=0xA7, codec=None):
        """decode_crops_device at output base offset `shift`; checks the guards -> (crops (N, R, ch, cw), status, indices)"""
        c, N, G = codec or self.codec, self.N, self.G
        corners = np.ascontiguousarray(corners, dtype=np.int32)
        per_frame = corners.ndim == 3
        R = corners.shape[-2]
        cw, ch = size
        n = N * R * cw * ch
        d_c = c.device_alloc(corners.nbytes)
        d_out = c.device_alloc(n + 2 * G + 16)
        try:
            c.h2d(d_c, corners)
            c.h2d(d_out, np.full(n + 2 * G + 16, fill, dtype=np.uint8))
            c.decode_crops_device(self.d_s, self.nbytes, self.d_o, self.W, self.H, N, d_c, R, per_frame, size, d_out + G + shift,
                                  self.d_st, self.d_ix, pad=pad)
            buf = c.d2h(d_out, n + 2 * G + 16)
        finally:
            c.device_free(d_c)
            c.device_free(d_out)
        assert (buf[:G + shift] == fill).all() and (buf[G + shift + n:] == fill).all(), ("wrote outside the output", size, shift)
        return (buf[G + shift:G + shift + n].reshape(N, R, ch, cw), c.d2h(self.d_st, 4 * N, np.uint32),
                c.d2h(self.d_ix, 8 * N, np.uint64))

    def roi(self, r):
        c, N = self.codec, self.N
        x0, y0, rw, rh = r
        d_out = c.device_alloc(N * rw * rh)
        try:
            c.decode_roi_device(self.d_s, self.nbytes, self.d_o, self.W, self.H, N, r, d_out, self.d_st)
            return c.d2h(d_out, N * rw * rh).reshape(N, rh, rw)
        finally:
            c.device_free(d_out)

    def free(self):
        for p in (self.d_s, self.d_o, self.d_st, self.d_ix):
            self.codec.device_free(p)


def encoded(W, H, frames=None, first=11):
    fr = content(W, H) if frames is None else frames
    stream, sizes = ORA.pack_frames(fr, first)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    return fr, stream, offs


def crop_sizes(W, H):
    S = {(1, 1), (1, H), (W, 1), (W, H), (W + 9, H + 5), (13, 11), (8, 8), (256, 3), (8 * 33 + 3, 5), (7, 8 * 33 + 1)}
    for b in range(8):                                     # every crop_w mod 8, within a few tiles and across 32-tile chunks
        S |= {(b + 8, 1 + b), (b + 8 * 33, 2)}
    return sorted(S)


def corner_set(W, H, cw, ch):
    """every x0 mod 8 (inside the frame and negative), corners straddling each edge and each corner of the frame, crops
    entirely outside it, and the int32 extremes"""
    C = set()
    for a in range(8):
        C |= {(a + 8 * ((a * 5) % max(1, (W - a) // 8 + 1)), (3 * a) % H), (a - 24, a), (a - 8, -a)}
    C |= {(-(cw // 2), H // 2), (W - cw // 2 - 1, H // 2), (W // 2, -(ch // 2)), (W // 2, H - ch // 2 - 1),
          (-3, -3), (W - 3, -3), (-3, H - 3), (W - 3, H - 3), (-cw + 1, -ch + 1), (W - 1, H - 1)}
    C |= {(W, 0), (W + 5, 7), (-cw, 0), (-cw - 9, 3), (0, H), (2, H + 17), (0, -ch), (1, -ch - 30)}
    C |= {(I32_MIN, I32_MIN), (I32_MAX, I32_MAX), (I32_MIN, 0), (0, I32_MAX), (I32_MAX, 0), (0, I32_MIN), (I32_MAX - cw, 0)}
    return np.array(sorted(C), dtype=np.int64).clip(I32_MIN, I32_MAX).astype(np.int32)


@pytest.mark.parametrize("W,H", GEOMETRIES)
def test_crops_equal_the_pad_crop(codec, W, H):
    """every kind of crop size and corner on every geometry class, shared corners, pad 0 and 255, output base offsets
    0-15 with guard bytes on both sides"""
    fr, stream, offs = encoded(W, H)
    full, idx, _ = ORA.unpack_frames(stream, W, H, len(fr))
    assert (full == fr).all() and idx == list(range(11, 11 + len(fr)))
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        for i, (cw, ch) in enumerate(crop_sizes(W, H)):
            corners = corner_set(W, H, cw, ch)
            nf = len(fr) if cw * ch <= 1 << 16 else 2
            d.N = nf                                        # the first nf records only: large crops stay small in memory
            per_call = max(1, (16 << 20) // (nf * cw * ch))
            for j in range(0, len(corners), per_call):
                cs = corners[j:j + per_call]
                pad = 255 if (i + j) % 2 else 0
                got, status, index = d.crops(cs, (cw, ch), pad=pad, shift=(i + j) % 16)
                assert (status == 0).all() and index.tolist() == list(range(11, 11 + nf)), (cw, ch)
                want = pad_crop(fr[:nf], cs, cw, ch, pad)
                if not np.array_equal(got, want):
                    bad = tuple(np.argwhere(got != want)[0])
                    pytest.fail("crop %dx%d at %r of %dx%d differs first at (frame, crop, row, col) %r"
                                % (cw, ch, tuple(cs[bad[1]]), W, H, bad))
    finally:
        d.free()


@pytest.mark.parametrize("W,H", [(2048, 2048), (1001, 1003), (2049, 9), (17, 23)])
def test_in_frame_crops_equal_the_region_decode(codec, W, H):
    """per-frame corners of crops inside the frame: each crop equals decode_roi_device of the same rectangle"""
    fr, stream, offs = encoded(W, H)
    N = len(fr)
    rng = np.random.default_rng(W + H)
    d = DevStream(codec, stream, offs, N, W, H)
    try:
        for cw, ch in [(1, 1), (min(W, 45), min(H, 13)), (min(W, 300), min(H, 7)), (W, H)]:
            corners = np.stack([rng.integers(0, W - cw + 1, (N, 5)), rng.integers(0, H - ch + 1, (N, 5))], axis=-1)
            got, status, _ = d.crops(corners, (cw, ch), pad=0x5A, shift=3)
            assert (status == 0).all()
            for f in range(N):
                for r in range(5):
                    x0, y0 = (int(v) for v in corners[f, r])
                    want = d.roi((x0, y0, cw, ch))[f]
                    assert np.array_equal(got[f, r], want), (cw, ch, f, r)
    finally:
        d.free()


def test_wells_overlap_and_per_frame_corners(codec):
    """96 wells of a 12 x 8 plate as shared corners, overlapping crops, and 96 per-frame crops scattered in and around
    the frame, some the same for several frames"""
    W, H = 1001, 1003
    fr, stream, offs = encoded(W, H)
    N = len(fr)
    d = DevStream(codec, stream, offs, N, W, H)
    try:
        wells = np.array([(30 + 80 * i, 40 + 120 * j) for j in range(8) for i in range(12)], dtype=np.int32)
        got, status, _ = d.crops(wells, (120, 120), pad=0, shift=7)
        assert (status == 0).all() and len(wells) == 96 and np.array_equal(got, pad_crop(fr, wells, 120, 120, 0))
        overlap = np.array([(100, 100), (101, 100), (100, 103), (100, 100), (96, 97), (40, 990)], dtype=np.int32)
        got, status, _ = d.crops(overlap, (64, 33), pad=255, shift=1)
        assert np.array_equal(got, pad_crop(fr, overlap, 64, 33, 255))
        rng = np.random.default_rng(96)
        per = np.stack([rng.integers(-80, W + 20, (N, 96)), rng.integers(-80, H + 20, (N, 96))], axis=-1).astype(np.int32)
        per[1] = per[0]
        got, status, _ = d.crops(per, (61, 77), pad=255, shift=14)
        assert (status == 0).all() and np.array_equal(got, pad_crop(fr, per, 61, 77, 255))
    finally:
        d.free()


@pytest.mark.parametrize("pad", [0, 255, 0x3C])
def test_crops_outside_the_frame_are_all_pad(codec, pad):
    W, H = 40, 24
    fr, stream, offs = encoded(W, H)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        far = np.array([(I32_MIN, I32_MIN), (I32_MAX, I32_MAX), (I32_MAX, I32_MIN), (I32_MIN, I32_MAX), (W, H), (-9, 0),
                        (0, -5)], dtype=np.int32)
        got, status, _ = d.crops(far, (9, 5), pad=pad)
        assert (status == 0).all() and (got == pad).all()
    finally:
        d.free()


def test_damage_outside_every_crop_is_rejected_like_the_full_decode(codec):
    """the damage of the full decoder's invalid-stream test, all of it outside every crop: the same status bits as
    decode_host, the crops of a rejected frame keep their fill, good frames of the batch still decode"""
    W, H, N = 48, 40, 7
    wh = 6 * 5
    corners = np.array([(17, 9), (-5, -5), (60, 3)], dtype=np.int32)   # tiles (2..3, 1..2), (0, 0), none
    cw, ch = 13, 11
    outside = 4 * 6 + 5                          # tile (5, 4): under no crop
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    bad = stream.copy()
    bad[int(offs[1]) + 20] += 1                 # nb != wh
    bad[int(offs[2]) + 24 + wh] += 1            # nm != wh
    bad[int(offs[3]) + 28 + 2 * wh] += 1        # n64 != sum(depth)
    bad[int(offs[4])] = 9                       # frame tag != 2
    bad[int(offs[5]) + 24 + outside] = 9        # a depth byte > 8
    want_ok = pad_crop(fr, corners, cw, ch, 0x11)
    for s, o in [(bad, offs[:N]), (stream[:int(offs[N]) - 8], offs[:N])]:                 # + a truncated last record
        _, want_status, want_idx = codec.decode_host(s, o, W, H, fill=0xCD)
        assert want_status.any()
        got, status, index = codec.decode_crops_host(s, o, W, H, corners, (cw, ch), pad=0x11, fill=0xCD)
        assert status.tolist() == want_status.tolist() and index.tolist() == want_idx.tolist()
        d = DevStream(codec, s, o, N, W, H)
        try:
            dgot, dstatus, dindex = d.crops(corners, (cw, ch), pad=0x11, shift=5, fill=0xCD)
        finally:
            d.free()
        assert dstatus.tolist() == want_status.tolist() and dindex.tolist() == want_idx.tolist()
        for i in range(N):
            if status[i]:
                assert (got[i] == 0xCD).all() and (dgot[i] == 0xCD).all(), i      # the all-outside crop too
            else:
                assert (got[i] == want_ok[i]).all() and (dgot[i] == want_ok[i]).all(), i
    assert codec.decode_crops_host(bad, offs[:N], W, H, corners, (cw, ch))[1][5] & pkg.ST_DEPTH_TOO_BIG


@pytest.mark.parametrize("W,H", [(1001, 43), (2049, 9), (61, 20), (10, 10)])
def test_invert_endian_variant(codec, W, H):
    """DBDE_INVERT_ENDIAN records (dbde_util.cpp:15-19,246-270), crops straddling the right edge of a W % 8 != 0 frame:
    rows are reversed before the columns past W are padded, pad bytes are never reversed"""
    V = oracle.best_variants()
    rng = np.random.default_rng(W + 31 * H)
    fr = np.stack([rand_frame(rng, W, H, ["classes", "noise", "classes"][i % 3]) for i in range(3)])
    want, sizes = V.pack_frames(fr, 9)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    corners = np.array([(W - 5, 0), (W - 3, H - 4), (W - 12, -2), (-3, 1), (W - 1, H // 2), (0, 0)], dtype=np.int32)
    c = pkg.Codec(0)
    d = DevStream(c, want, offs, 3, W, H)
    try:
        c.set_invert_endian(True)
        for size in [(9, 7), (20, 3), (W + 4, H + 2)]:
            got, status, _ = c.decode_crops_host(want, offs[:3], W, H, corners, size, pad=0xE1)
            assert (status == 0).all() and np.array_equal(got, pad_crop(fr, corners, *size, 0xE1)), size
            dgot, dstatus, _ = d.crops(corners, size, pad=0xE1, shift=9)
            assert (dstatus == 0).all() and np.array_equal(dgot, got), size
        plain, _, _ = codec.decode_crops_host(want, offs[:3], W, H, corners, (9, 7), pad=0xE1)
        assert not np.array_equal(plain, pad_crop(fr, corners, 9, 7, 0xE1))
    finally:
        d.free()
        c.close()


def test_host_form_pinned_pageable_and_chunked(codec):
    """decode_crops_host on pageable numpy and pinned buffers; chunks of 3 frames in flight with per-frame corners
    that differ across chunk boundaries; a rejected frame in the middle of a chunk"""
    W, H, N = 1001, 203, 10
    cw, ch = 97, 45
    fr = synth.gen_frames("mix", N, W, H, f0=4)
    stream, offs = codec.encode_host(fr, 3)
    rng = np.random.default_rng(7)
    per = np.stack([rng.integers(-60, W, (N, 4)), rng.integers(-30, H, (N, 4))], axis=-1).astype(np.int32)
    shared = per[0]
    want_per, want_shared = pad_crop(fr, per, cw, ch, 0x42), pad_crop(fr, shared, cw, ch, 0x42)
    c = pkg.Codec(0)
    try:
        c.set_chunk_frames(3)
        for corners, want in [(per, want_per), (shared, want_shared)]:
            got, status, index = c.decode_crops_host(stream, offs[:N], W, H, corners, (cw, ch), pad=0x42)
            assert (status == 0).all() and index.tolist() == list(range(3, 3 + N)) and np.array_equal(got, want)
        # pinned everything, output at an odd address
        n = N * 4 * cw * ch
        ps, po, pc, pf = c.pinned(len(stream)), c.pinned(8 * N), c.pinned(per.nbytes), c.pinned(n + 1)
        pst, pix = c.pinned(4 * N), c.pinned(8 * N)
        try:
            ps.array[:] = stream
            po.array[:] = offs[:N].view(np.uint8)
            pc.array[:] = per.view(np.uint8).ravel()
            pf.array[:] = 0
            assert c.lib.dbde_b200_decode_crops_host(c.h, ps.ptr, len(stream), po.ptr, W, H, N, pc.ptr, 4, 1, cw, ch, 0x42,
                                                     pf.ptr + 1, pst.ptr, pix.ptr) == 0
            assert (pst.array.view(np.uint32) == 0).all() and pf.array[0] == 0
            assert np.array_equal(pf.array[1:].reshape(N, 4, ch, cw), want_per)
        finally:
            for p in (ps, po, pc, pf, pst, pix):
                p.free()
        # frame 4 (the middle of the second chunk) rejected: its crops keep the fill, its neighbours decode
        bad = stream.copy()
        bad[int(offs[4])] = 9
        got, status, _ = c.decode_crops_host(bad, offs[:N], W, H, per, (cw, ch), pad=0x42, fill=0xCD)
        assert status[4] & pkg.ST_BAD_FRAME_HEADER and (np.delete(status, 4) == 0).all()
        assert (got[4] == 0xCD).all() and np.array_equal(np.delete(got, 4, axis=0), np.delete(want_per, 4, axis=0))
    finally:
        c.close()


def test_host_form_crops_larger_than_the_frame(codec):
    """many crops larger than the frame: more output per frame than W * H, still one call"""
    W, H, N = 64, 40, 5
    fr = synth.gen_frames("mix", N, W, H)
    stream, offs = codec.encode_host(fr, 0)
    corners = np.array([(-10, -20), (5, 3), (-200, 0)] * 30, dtype=np.int32)
    got, status, _ = codec.decode_crops_host(stream, offs[:N], W, H, corners, (100, 70), pad=9)
    assert (status == 0).all() and np.array_equal(got, pad_crop(fr, corners, 100, 70, 9))


def test_scale_1000_frames_micro_2048_random_walk(codec):
    """1000 frames of 2048^2 'micro' in HBM, one 256^2 crop per frame on a random walk that reaches past the edges:
    equal to the pad-crop of the full GPU decode (SHA-256 over all crops)"""
    N, W, H = 1000, 2048, 2048
    cw = ch = 256
    px = W * H
    wh = (W // 8) * (H // 8)
    rng = np.random.default_rng(1000)
    walk = np.cumsum(rng.integers(-40, 41, (N, 2)), axis=0) + (1000, 1000)
    corners = np.clip(walk, -300, W + 40).astype(np.int32).reshape(N, 1, 2)
    cap = codec.stream_bound(W, H, N)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    d_fr, d_out = codec.device_alloc(N * px), codec.device_alloc(cap + 64)
    d_off, d_sz, d_st, d_st2 = (codec.device_alloc(8 * N), codec.device_alloc(8 * N), codec.device_alloc(4 * N),
                                codec.device_alloc(4 * N))
    d_c, d_crops = codec.device_alloc(corners.nbytes), codec.device_alloc(N * cw * ch)
    try:
        synth.gen_frames_device("micro", N, W, H, d_fr, seed=42, f0=0)
        codec.encode_device(d_fr, W, H, 0, N, d_out + delta, cap, d_off, d_sz)
        codec.h2d(d_c, corners)
        codec.decode_crops_device(d_out + delta, cap, d_off, W, H, N, d_c, 1, True, (cw, ch), d_crops, d_st2, pad=0x80)
        codec.decode_device(d_out + delta, cap, d_off, W, H, N, d_fr, d_st)      # the full decode over the source frames
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all() and (codec.d2h(d_st2, 4 * N, np.uint32) == 0).all()
        h_want, h_got = hashlib.sha256(), hashlib.sha256()
        step = 50
        for a in range(0, N, step):
            full = codec.d2h(d_fr + a * px, step * px).reshape(step, H, W)
            h_want.update(pad_crop(full, corners[a:a + step], cw, ch, 0x80).tobytes())
        h_got.update(codec.d2h(d_crops, N * cw * ch).tobytes())
        assert h_got.hexdigest() == h_want.hexdigest()
    finally:
        for p in (d_fr, d_out, d_off, d_sz, d_st, d_st2, d_c, d_crops):
            codec.device_free(p)


def test_bad_arguments(codec):
    """each bad argument returns DBDE_B200_E_INVALID with nothing queued (the launch count does not move); an empty
    batch returns 0"""
    lib, h = codec.lib, codec.h
    W, H, N = 40, 24, 2
    fr = synth.gen_frames("mix", N, W, H)
    stream, offs = codec.encode_host(fr, 0)
    d = DevStream(codec, stream, offs, N, W, H)
    corners = np.array([[1, 2], [3, 4]], dtype=np.int32)
    d_c, d_out = codec.device_alloc(corners.nbytes), codec.device_alloc(1 << 16)
    codec.h2d(d_c, corners)
    st = np.zeros(N, np.uint32)
    out = np.zeros(1 << 16, np.uint8)

    def dev(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0)
        a.update(kw)
        args = [h, d.d_s, d.nbytes, d.d_o, W, H, n, d_c, a["ncrops"], a["per_frame"], a["cw"], a["ch"], a["pad"], d_out, d.d_st,
                None, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode_crops_device(*args)

    def host(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0)
        a.update(kw)
        args = [h, stream.ctypes.data, stream.nbytes, offs.ctypes.data, W, H, n, corners.ctypes.data, a["ncrops"], a["per_frame"],
                a["cw"], a["ch"], a["pad"], out.ctypes.data, st.ctypes.data, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode_crops_host(*args)

    try:
        l0 = codec.launches()
        bad = [dict(ncrops=0), dict(ncrops=-1), dict(cw=0), dict(ch=0), dict(cw=-4), dict(ch=-3),
               dict(cw=2**31 - 1, ch=2), dict(cw=1 << 16, ch=1 << 16), dict(ncrops=1 << 20, cw=64, ch=64), dict(ncrops=2**31 - 1, cw=1, ch=2),
               dict(per_frame=2), dict(per_frame=-1), dict(pad=-1), dict(pad=256)]
        for kw in bad:
            assert dev(**kw) == E_INVALID, kw
            assert host(**kw) == E_INVALID, kw
            assert dev(n=0, **kw) == E_INVALID, kw
        for i in (0, 1, 3, 7, 13, 14):                               # ctx, stream, offsets, corners, output, status
            assert dev((i, None)) == E_INVALID, i
            assert host((i, None)) == E_INVALID, i
        assert dev((4, 0)) == E_INVALID and dev((5, -1)) == E_INVALID and dev(n=-1) == E_INVALID
        assert codec.launches() == l0
        assert dev(n=0) == 0 and host(n=0) == 0
        assert dev((1, None), (3, None), (7, None), (13, None), (14, None), n=0) == 0      # nothing to do, nothing read
        assert codec.launches() == l0
        # the context is still usable, and the last good call decodes
        assert dev() == 0 and codec.launches() == l0 + 2
        got = codec.d2h(d_out, N * 2 * 4 * 3).reshape(N, 2, 3, 4)
        assert (codec.d2h(d.d_st, 4 * N, np.uint32) == 0).all() and np.array_equal(got, pad_crop(fr, corners, 4, 3, 0))
        got, status, _ = codec.decode_crops_host(stream, offs[:N], W, H, corners, (4, 3))
        assert (status == 0).all() and np.array_equal(got, pad_crop(fr, corners, 4, 3, 0))
    finally:
        codec.device_free(d_c)
        codec.device_free(d_out)
        d.free()
