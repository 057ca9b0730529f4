"""DBDE16 crop and binned decoding (dbde_b200_decode16_crops_* / dbde_b200_decode16_binned_*) on a B200: fixed-size
U16 windows at shared or per-frame corners, padded outside the frame, and 2x2 / 4x4 / 8x8 block means of 16-bit frames.
The expected output is numpy applied to the source frames (the codec is lossless, so they are the full decode);
validation covers the whole record with dbde_b200_decode16_device's status bits, and nothing outside the output range
is written."""
import importlib

import numpy as np
import pytest

import oracle
import synth

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()
P16 = oracle.port16
E_INVALID = -1
I32_MIN, I32_MAX = -2**31, 2**31 - 1
FACTORS = [1, 2, 4, 8]

# the crop and binned tests' eleven geometries plus the sCMOS sizes
GEOMETRIES = [(2048, 2048), (2304, 48), (1280, 64), (4096, 8), (4104, 16), (2049, 9), (4100, 1003), (1001, 1003),
              (17, 23), (3, 5), (1, 1), (2304, 2304), (2560, 2160)]


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


def rand_frame16(rng, W, H, style):
    """'classes': every depth 0..16 among the tiles of one warp; 'sensor12': a 12-bit camera-like smooth field plus 5
    bits of noise"""
    if style == "noise":
        return rng.integers(0, 65536, (H, W), dtype=np.uint16)
    if style == "flat":
        return np.full((H, W), rng.integers(0, 65536), dtype=np.uint16)
    if style == "byte":
        return rng.integers(0, 256, (H, W)).astype(np.uint16)
    if style == "sensor12":
        y, x = np.mgrid[0:H, 0:W]
        return (600 + x // 16 + y // 8 + rng.integers(0, 32, (H, W))).astype(np.uint16)
    th, tw = (H + 7) // 8, (W + 7) // 8
    k = rng.integers(0, 17, (th, tw))
    rg = (1 << k) - 1
    mn = (rng.random((th, tw)) * (65536 - rg)).astype(np.int64)
    big = (mn[:, :, None, None] + (rng.integers(0, 65536, (th, tw, 8, 8)) & rg[:, :, None, None]))
    return big.transpose(0, 2, 1, 3).reshape(th * 8, tw * 8)[:H, :W].astype(np.uint16)


def content(W, H):
    rng = np.random.default_rng(W * 7919 + H + 16)
    return np.stack([rand_frame16(rng, W, H, s) for s in ("classes", "noise", "flat", "byte", "sensor12")])


def pad_crop(frames, corners, cw, ch, pad):
    """the reference: frames (N, H, W), corners (R, 2) or (N, R, 2) -> (N, R, ch, cw)"""
    N, H, W = frames.shape
    c = np.broadcast_to(corners, (N,) + corners.shape) if corners.ndim == 2 else corners
    out = np.full((N, c.shape[1], ch, cw), pad, dtype=frames.dtype)
    for f in range(N):
        for r in range(c.shape[1]):
            x0, y0 = int(c[f, r, 0]), int(c[f, r, 1])
            xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
            if xa < xb and ya < yb:
                out[f, r, ya - y0:yb - y0, xa - x0:xb - x0] = frames[f, ya:yb, xa:xb]
    return out


def block_mean(frames, b):
    """the reference: frames (N, H, W) -> (N, ceil(H / b), ceil(W / b)), the mean of each block's in-frame pixels,
    rounded half up"""
    N, H, W = frames.shape
    Hb, Wb = -(-H // b), -(-W // b)
    p = np.zeros((N, Hb * b, Wb * b), np.uint64)
    p[:, :H, :W] = frames
    m = np.zeros((Hb * b, Wb * b), np.uint64)
    m[:H, :W] = 1
    s = p.reshape(N, Hb, b, Wb, b).sum(axis=(2, 4))
    n = m.reshape(Hb, b, Wb, b).sum(axis=(1, 3))
    return ((s + n // 2) // n).astype(np.uint16)


def encoded(W, H, frames=None, first=11):
    fr = content(W, H) if frames is None else frames
    stream, sizes = P16.pack_frames(fr, first)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    return fr, stream, offs


class DevStream:
    """records and their offsets uploaded once; the calls decode into a guarded output buffer at a base offset of
    `shift` bytes (even) and check the guards"""
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

    def _guarded(self, n, shift, fill, call, shape):
        c, G = self.codec, self.G
        nb = 2 * n
        d_out = c.device_alloc(nb + 2 * G + 16)
        try:
            c.h2d(d_out, np.full(nb + 2 * G + 16, fill, dtype=np.uint8))
            call(d_out + G + shift)
            buf = c.d2h(d_out, nb + 2 * G + 16)
        finally:
            c.device_free(d_out)
        assert (buf[:G + shift] == fill).all() and (buf[G + shift + nb:] == fill).all(), ("wrote outside the output", shift)
        return (buf[G + shift:G + shift + nb].view(np.uint16).reshape(shape), c.d2h(self.d_st, 4 * self.N, np.uint32),
                c.d2h(self.d_ix, 8 * self.N, np.uint64))

    def crops(self, corners, size, pad=0, shift=0, fill=0xA7):
        """decode16_crops_device -> (crops (N, R, ch, cw), status, indices)"""
        c, N = self.codec, self.N
        corners = np.ascontiguousarray(corners, dtype=np.int32)
        R = corners.shape[-2]
        cw, ch = size
        d_c = c.device_alloc(corners.nbytes)
        try:
            c.h2d(d_c, corners)
            return self._guarded(N * R * cw * ch, shift, fill,
                                 lambda out: c.decode16_crops_device(self.d_s, self.nbytes, self.d_o, self.W, self.H, N, d_c, R,
                                                                     corners.ndim == 3, size, out, self.d_st, self.d_ix, pad=pad),
                                 (N, R, ch, cw))
        finally:
            c.device_free(d_c)

    def binned(self, factor, shift=0, fill=0xA7):
        """decode16_binned_device -> (frames (N, Hb, Wb), status, indices)"""
        c, N = self.codec, self.N
        Hb, Wb = -(-self.H // factor), -(-self.W // factor)
        return self._guarded(N * Hb * Wb, shift, fill,
                             lambda out: c.decode16_binned_device(self.d_s, self.nbytes, self.d_o, self.W, self.H, N, factor, out,
                                                                  self.d_st, self.d_ix),
                             (N, Hb, Wb))

    def full(self, fill=0xA7):
        """decode16_device -> (frames (N, H, W), status, indices)"""
        c, N = self.codec, self.N
        return self._guarded(N * self.W * self.H, 0, fill,
                             lambda out: c._ck(c.lib.dbde_b200_decode16_device(c.h, self.d_s, self.nbytes, self.d_o, self.W, self.H,
                                                                               N, out, self.d_st, self.d_ix, None),
                                               "decode16_device"),
                             (N, self.H, self.W))

    def free(self):
        for p in (self.d_s, self.d_o, self.d_st, self.d_ix):
            self.codec.device_free(p)


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
def test_crops16_equal_the_pad_crop(codec, W, H):
    """every kind of crop size and corner on every geometry, shared corners, pad 0 and 65535, output base offsets
    0, 2, ..., 14 bytes with guard bytes on both sides; a crop equal to the frame at (0, 0) is decode16_device"""
    fr, stream, offs = encoded(W, H)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        full, status, index = d.full()
        assert (status == 0).all() and index.tolist() == list(range(11, 11 + len(fr))) and np.array_equal(full, fr)
        got, status, _ = d.crops(np.array([[0, 0]]), (W, H), pad=7, shift=6)
        assert (status == 0).all() and np.array_equal(got[:, 0], full)
        for i, (cw, ch) in enumerate(crop_sizes(W, H)):
            corners = corner_set(W, H, cw, ch)
            nf = len(fr) if cw * ch <= 1 << 16 else 2
            d.N = nf                                        # the first nf records only: large crops stay small in memory
            per_call = max(1, (16 << 20) // (2 * nf * cw * ch))
            for j in range(0, len(corners), per_call):
                cs = corners[j:j + per_call]
                pad = 65535 if (i + j) % 2 else 0
                got, status, index = d.crops(cs, (cw, ch), pad=pad, shift=2 * ((i + j) % 8))
                assert (status == 0).all() and index.tolist() == list(range(11, 11 + nf)), (cw, ch)
                want = pad_crop(fr[:nf], cs, cw, ch, pad)
                if not np.array_equal(got, want):
                    bad = tuple(np.argwhere(got != want)[0])
                    pytest.fail("crop %dx%d at %r of %dx%d differs first at (frame, crop, row, col) %r"
                                % (cw, ch, tuple(cs[bad[1]]), W, H, bad))
            d.N = len(fr)
    finally:
        d.free()


@pytest.mark.parametrize("W,H", GEOMETRIES)
def test_binned16_equal_the_block_mean(codec, W, H):
    """every factor on every geometry at output base offsets 0, 2, ..., 14 bytes; factor 1 is decode16_device"""
    fr, stream, offs = encoded(W, H)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        full = d.full()[0]
        for i, b in enumerate(FACTORS):
            for shift in ((0, 2, 4, 6, 8, 10, 12, 14) if W * H <= 1 << 16 else (2 * i, 2 * i + 6)):
                got, status, index = d.binned(b, shift=shift)
                assert (status == 0).all() and index.tolist() == list(range(11, 11 + len(fr)))
                want = full if b == 1 else block_mean(fr, b)
                if not np.array_equal(got, want):
                    bad = tuple(np.argwhere(got != want)[0])
                    pytest.fail("b=%d of %dx%d differs first at (frame, row, col) %r: %d != %d"
                                % (b, W, H, bad, got[bad], want[bad]))
    finally:
        d.free()


@pytest.mark.parametrize("W,H", [(16, 16), (10, 16), (16, 10), (13, 11), (2050, 6), (6, 2050), (1003, 1001)])
def test_binned16_partial_last_bins(codec, W, H):
    """partial last bins in x, in y and in both, inside a full tile and in a partial last tile, host and device"""
    rng = np.random.default_rng(W * 3 + H)
    fr = np.stack([rand_frame16(rng, W, H, s) for s in ("noise", "classes", "noise")])
    fr[2] = 65535                                          # the largest sums
    _, stream, offs = encoded(W, H, fr)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        for b in (2, 4, 8):
            want = block_mean(fr, b)
            got, status, _ = d.binned(b, shift=2)
            assert (status == 0).all() and np.array_equal(got, want), b
            hgot, hstatus, _ = codec.decode16_binned_host(stream, offs[:3], W, H, b)
            assert (hstatus == 0).all() and np.array_equal(hgot, want), b
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
        got, status, _ = d.crops(wells, (120, 120), pad=0, shift=6)
        assert (status == 0).all() and len(wells) == 96 and np.array_equal(got, pad_crop(fr, wells, 120, 120, 0))
        overlap = np.array([(100, 100), (101, 100), (100, 103), (100, 100), (96, 97), (40, 990)], dtype=np.int32)
        got, status, _ = d.crops(overlap, (64, 33), pad=65535, shift=2)
        assert np.array_equal(got, pad_crop(fr, overlap, 64, 33, 65535))
        rng = np.random.default_rng(96)
        per = np.stack([rng.integers(-80, W + 20, (N, 96)), rng.integers(-80, H + 20, (N, 96))], axis=-1).astype(np.int32)
        per[1] = per[0]
        got, status, _ = d.crops(per, (61, 77), pad=65535, shift=14)
        assert (status == 0).all() and np.array_equal(got, pad_crop(fr, per, 61, 77, 65535))
    finally:
        d.free()


@pytest.mark.parametrize("pad", [0, 65535, 0x1234])
def test_crops_outside_the_frame_are_all_pad(codec, pad):
    W, H = 40, 24
    fr, stream, offs = encoded(W, H)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        far = np.array([(I32_MIN, I32_MIN), (I32_MAX, I32_MAX), (I32_MAX, I32_MIN), (I32_MIN, I32_MAX), (W, H), (-9, 0),
                        (0, -5)], dtype=np.int32)
        got, status, _ = d.crops(far, (9, 5), pad=pad, shift=4)
        assert (status == 0).all() and (got == pad).all()
    finally:
        d.free()


def test_damage_is_rejected_like_decode16_device(codec):
    """damaged records, part of the damage outside every crop, and a truncated last record: the status bits and indices
    of decode16_device, a rejected frame's crops and bins keep their fill, good frames of the batch still decode"""
    W, H, N = 48, 40, 7
    wh = 6 * 5
    corners = np.array([(17, 9), (-5, -5), (60, 3)], dtype=np.int32)   # tiles (2..3, 1..2), (0, 0), none
    cw, ch = 13, 11
    outside = 4 * 6 + 5                          # tile (5, 4): under no crop
    rng = np.random.default_rng(77)
    fr = np.stack([rand_frame16(rng, W, H, "classes") for _ in range(N)])
    _, stream, offs = encoded(W, H, fr, first=0)
    bad = stream.copy()
    bad[int(offs[1]) + 20] += 1                 # nb != wh
    bad[int(offs[2]) + 24 + wh] += 1            # nm != 2 wh
    bad[int(offs[3]) + 28 + 3 * wh] += 1        # n64 != sum(depth)
    bad[int(offs[4])] = 9                       # frame tag != 2
    bad[int(offs[5]) + 24 + outside] = 17       # a depth byte > 16, outside every crop
    want_crops = pad_crop(fr, corners, cw, ch, 0x1111)
    for s in (bad, stream[:int(offs[N]) - 8]):
        d = DevStream(codec, s, offs, N, W, H)
        try:
            _, want_status, want_idx = d.full(fill=0xCD)
            assert want_status.any()
            results = [d.crops(corners, (cw, ch), pad=0x1111, shift=10, fill=0xCD) + (want_crops,)]
            results += [d.binned(b, shift=4, fill=0xCD) + (block_mean(fr, b),) for b in (2, 4, 8)]
        finally:
            d.free()
        results.append(codec.decode16_crops_host(s, offs[:N], W, H, corners, (cw, ch), pad=0x1111, fill=0xCDCD) + (want_crops,))
        results += [codec.decode16_binned_host(s, offs[:N], W, H, b, fill=0xCDCD) + (block_mean(fr, b),) for b in (2, 4, 8)]
        for got, status, index, want in results:
            assert status.tolist() == want_status.tolist() and index.tolist() == want_idx.tolist()
            for i in range(N):
                if status[i]:
                    assert (got[i] == 0xCDCD).all(), i                          # the all-outside crop too
                else:
                    assert np.array_equal(got[i], want[i]), i
    assert codec.decode16_crops_host(bad, offs[:N], W, H, corners, (cw, ch))[1][5] & pkg.ST_DEPTH_TOO_BIG


def test_invert_endian_setting_changes_nothing(codec):
    """DBDE16 has no DBDE_INVERT_ENDIAN variant: with the context's setting on, crops and bins are unchanged"""
    W, H = 1001, 43
    fr, stream, offs = encoded(W, H)
    N = len(fr)
    corners = np.array([(W - 5, 0), (W - 3, H - 4), (-3, 1), (0, 0)], dtype=np.int32)
    want = pad_crop(fr, corners, 20, 9, 0xE1E1)
    c = pkg.Codec(0)
    d = DevStream(c, stream, offs, N, W, H)
    try:
        c.set_invert_endian(True)
        got, status, _ = c.decode16_crops_host(stream, offs[:N], W, H, corners, (20, 9), pad=0xE1E1)
        assert (status == 0).all() and np.array_equal(got, want)
        got, status, _ = d.crops(corners, (20, 9), pad=0xE1E1, shift=2)
        assert (status == 0).all() and np.array_equal(got, want)
        for b in (2, 8):
            got, status, _ = d.binned(b)
            assert (status == 0).all() and np.array_equal(got, block_mean(fr, b))
            got, status, _ = c.decode16_binned_host(stream, offs[:N], W, H, b)
            assert (status == 0).all() and np.array_equal(got, block_mean(fr, b))
    finally:
        d.free()
        c.close()


def test_8_bit_content_matches_the_8_bit_crops(codec):
    """frames whose pixels fit in 8 bits: the DBDE16 crops are the 8-bit decode_crops of the same pixels widened"""
    W, H, N = 1001, 203, 4
    fr8 = synth.gen_frames("mix", N, W, H)
    s8, sizes8 = ORA.pack_frames(fr8, 0)
    o8 = np.concatenate([[0], np.cumsum(sizes8)]).astype(np.uint64)
    _, s16, o16 = encoded(W, H, fr8.astype(np.uint16), first=0)
    rng = np.random.default_rng(8)
    per = np.stack([rng.integers(-60, W, (N, 5)), rng.integers(-30, H, (N, 5))], axis=-1).astype(np.int32)
    for size in [(97, 45), (8, 8), (300, 2)]:
        g8, st8, _ = codec.decode_crops_host(s8, o8[:N], W, H, per, size, pad=200)
        g16, st16, _ = codec.decode16_crops_host(s16, o16[:N], W, H, per, size, pad=200)
        assert (st8 == 0).all() and (st16 == 0).all() and np.array_equal(g16, g8.astype(np.uint16)), size


def test_host_forms_pinned_pageable_and_chunked(codec):
    """the host forms on pageable numpy and pinned buffers; chunks of 3 frames in flight with per-frame corners that
    differ across chunk boundaries; a rejected frame in the middle of a chunk"""
    W, H, N = 1001, 203, 10
    cw, ch = 97, 45
    rng = np.random.default_rng(10)
    fr = np.stack([rand_frame16(rng, W, H, ["sensor12", "classes"][i % 2]) for i in range(N)])
    c = pkg.Codec(0)
    try:
        c.set_chunk_frames(3)
        stream, offs = c.encode16_host(fr, 3)
        per = np.stack([rng.integers(-60, W, (N, 4)), rng.integers(-30, H, (N, 4))], axis=-1).astype(np.int32)
        want_per, want_shared = pad_crop(fr, per, cw, ch, 0x4242), pad_crop(fr, per[0], cw, ch, 0x4242)
        for corners, want in [(per, want_per), (per[0], want_shared)]:
            got, status, index = c.decode16_crops_host(stream, offs[:N], W, H, corners, (cw, ch), pad=0x4242)
            assert (status == 0).all() and index.tolist() == list(range(3, 3 + N)) and np.array_equal(got, want)
        for b in (2, 4, 8):
            got, status, _ = c.decode16_binned_host(stream, offs[:N], W, H, b)
            assert (status == 0).all() and np.array_equal(got, block_mean(fr, b)), b
        # pinned everything, output at an even address that is not 4-byte aligned
        n = N * 4 * cw * ch
        Hb, Wb = -(-H // 2), -(-W // 2)
        ps, po, pc, pf = c.pinned(len(stream)), c.pinned(8 * N), c.pinned(per.nbytes), c.pinned(2 * max(n, N * Hb * Wb) + 2)
        pst, pix = c.pinned(4 * N), c.pinned(8 * N)
        try:
            ps.array[:] = stream
            po.array[:] = offs[:N].view(np.uint8)
            pc.array[:] = per.view(np.uint8).ravel()
            pf.array[:] = 0
            assert c.lib.dbde_b200_decode16_crops_host(c.h, ps.ptr, len(stream), po.ptr, W, H, N, pc.ptr, 4, 1, cw, ch, 0x4242,
                                                       pf.ptr + 2, pst.ptr, pix.ptr) == 0
            assert (pst.array.view(np.uint32) == 0).all() and (pf.array[:2] == 0).all()
            assert np.array_equal(pf.array[2:2 + 2 * n].view(np.uint16).reshape(N, 4, ch, cw), want_per)
            pf.array[:] = 0
            assert c.lib.dbde_b200_decode16_binned_host(c.h, ps.ptr, len(stream), po.ptr, W, H, N, 2, pf.ptr + 2, pst.ptr,
                                                        pix.ptr) == 0
            assert (pst.array.view(np.uint32) == 0).all() and (pf.array[:2] == 0).all()
            assert np.array_equal(pf.array[2:2 + 2 * N * Hb * Wb].view(np.uint16).reshape(N, Hb, Wb), block_mean(fr, 2))
        finally:
            for p in (ps, po, pc, pf, pst, pix):
                p.free()
        # frame 4 (the middle of the second chunk) rejected: its output keeps the fill, its neighbours decode
        bad = stream.copy()
        bad[int(offs[4])] = 9
        got, status, _ = c.decode16_crops_host(bad, offs[:N], W, H, per, (cw, ch), pad=0x4242, fill=0xCDCD)
        assert status[4] & pkg.ST_BAD_FRAME_HEADER and (np.delete(status, 4) == 0).all()
        assert (got[4] == 0xCDCD).all() and np.array_equal(np.delete(got, 4, axis=0), np.delete(want_per, 4, axis=0))
        got, status, _ = c.decode16_binned_host(bad, offs[:N], W, H, 4, fill=0xCDCD)
        assert status[4] & pkg.ST_BAD_FRAME_HEADER and (np.delete(status, 4) == 0).all()
        assert (got[4] == 0xCDCD).all() and np.array_equal(np.delete(got, 4, axis=0), np.delete(block_mean(fr, 4), 4, axis=0))
        # crops larger than the frame: more output per frame than W * H
        corners = np.array([(-10, -20), (5, 3), (-200, 0)] * 30, dtype=np.int32)
        got, status, _ = c.decode16_crops_host(stream[:int(offs[2])], offs[:2], W, H, corners, (W + 40, 70), pad=9)
        assert (status == 0).all() and np.array_equal(got, pad_crop(fr[:2], corners, W + 40, 70, 9))
    finally:
        c.close()


def test_bad_arguments(codec):
    """each bad argument returns DBDE_B200_E_INVALID with nothing queued (the launch count does not move); an empty
    batch returns 0"""
    lib, h = codec.lib, codec.h
    W, H, N = 40, 24, 2
    fr, stream, offs = encoded(W, H, content(W, H)[:N], first=0)
    d = DevStream(codec, stream, offs, N, W, H)
    corners = np.array([[1, 2], [3, 4]], dtype=np.int32)
    d_c, d_out = codec.device_alloc(corners.nbytes), codec.device_alloc(1 << 16)
    codec.h2d(d_c, corners)
    st = np.zeros(N, np.uint32)
    out = np.zeros(1 << 16, np.uint16)

    def cdev(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0)
        a.update(kw)
        args = [h, d.d_s, d.nbytes, d.d_o, W, H, n, d_c, a["ncrops"], a["per_frame"], a["cw"], a["ch"], a["pad"], d_out, d.d_st,
                None, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode16_crops_device(*args)

    def chost(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0)
        a.update(kw)
        args = [h, stream.ctypes.data, stream.nbytes, offs.ctypes.data, W, H, n, corners.ctypes.data, a["ncrops"], a["per_frame"],
                a["cw"], a["ch"], a["pad"], out.ctypes.data, st.ctypes.data, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode16_crops_host(*args)

    def bdev(*over, n=N, factor=2):
        args = [h, d.d_s, d.nbytes, d.d_o, W, H, n, factor, d_out, d.d_st, None, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode16_binned_device(*args)

    def bhost(*over, n=N, factor=2):
        args = [h, stream.ctypes.data, stream.nbytes, offs.ctypes.data, W, H, n, factor, out.ctypes.data, st.ctypes.data, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode16_binned_host(*args)

    try:
        l0 = codec.launches()
        bad = [dict(ncrops=0), dict(ncrops=-1), dict(cw=0), dict(ch=0), dict(cw=-4), dict(ch=-3),
               dict(cw=2**31 - 1, ch=2), dict(cw=1 << 16, ch=1 << 16), dict(ncrops=1 << 20, cw=64, ch=64), dict(ncrops=2**31 - 1, cw=1, ch=2),
               dict(per_frame=2), dict(per_frame=-1), dict(pad=-1), dict(pad=65536)]
        for kw in bad:
            assert cdev(**kw) == E_INVALID, kw
            assert chost(**kw) == E_INVALID, kw
            assert cdev(n=0, **kw) == E_INVALID, kw
        for factor in (0, 3, 5, 16, -2):
            assert bdev(factor=factor) == E_INVALID and bhost(factor=factor) == E_INVALID and bdev(n=0, factor=factor) == E_INVALID
        for i in (0, 1, 3, 7, 13, 14):                               # ctx, stream, offsets, corners, output, status
            assert cdev((i, None)) == E_INVALID, i
            assert chost((i, None)) == E_INVALID, i
        for i in (0, 1, 3, 8, 9):                                    # ctx, stream, offsets, output, status
            assert bdev((i, None)) == E_INVALID, i
            assert bhost((i, None)) == E_INVALID, i
        for factor in (1, 2, 4, 8):                                  # an odd output pointer
            assert bdev((8, d_out + 1), factor=factor) == E_INVALID and bhost((8, out.ctypes.data + 1), factor=factor) == E_INVALID
        assert cdev((13, d_out + 1)) == E_INVALID and chost((13, out.ctypes.data + 3)) == E_INVALID
        assert cdev((4, 0)) == E_INVALID and cdev((5, -1)) == E_INVALID and cdev(n=-1) == E_INVALID
        assert bdev((4, 0)) == E_INVALID and bdev(n=-1) == E_INVALID
        assert codec.launches() == l0
        assert cdev(n=0) == 0 and chost(n=0) == 0 and bdev(n=0) == 0 and bhost(n=0) == 0
        assert cdev((1, None), (3, None), (7, None), (13, None), (14, None), n=0) == 0      # nothing to do, nothing read
        assert codec.launches() == l0
        # the context is still usable, and the last good calls decode
        assert cdev() == 0 and codec.launches() == l0 + 2
        got = codec.d2h(d_out, 2 * N * 2 * 4 * 3, np.uint16).reshape(N, 2, 3, 4)
        assert (codec.d2h(d.d_st, 4 * N, np.uint32) == 0).all() and np.array_equal(got, pad_crop(fr, corners, 4, 3, 0))
        assert bdev(factor=4) == 0 and codec.launches() == l0 + 4
        got = codec.d2h(d_out, 2 * N * 6 * 10, np.uint16).reshape(N, 6, 10)
        assert np.array_equal(got, block_mean(fr, 4))
    finally:
        codec.device_free(d_c)
        codec.device_free(d_out)
        d.free()


def test_scale_300_frames_sensor12_2048(codec):
    """300 frames of sensor12 2048^2 encoded on the device and kept in HBM: a 256^2 crop per frame on a random walk that
    reaches past the edges, 96 wells, and every factor, against numpy on the source frames"""
    N, W, H, K = 300, 2048, 2048, 6                          # K distinct frames, frame i is src[i % K]
    px = W * H
    rng = np.random.default_rng(300)
    src = np.stack([rand_frame16(rng, W, H, "sensor12") for _ in range(K)])
    stride = int(codec.lib.dbde_b200_slot_stride16(W, H))
    cap = stride * N
    d_fr, d_rec = codec.device_alloc(2 * N * px), codec.device_alloc(cap + 64)
    d_off, d_sz, d_st = codec.device_alloc(8 * N), codec.device_alloc(8 * N), codec.device_alloc(4 * N)
    walk = np.cumsum(rng.integers(-40, 41, (N, 2)), axis=0) + (1000, 1000)
    corners = np.clip(walk, -300, W + 40).astype(np.int32).reshape(N, 1, 2)
    wells = np.array([(60 + 160 * i, 100 + 240 * j) for j in range(8) for i in range(12)], dtype=np.int32)
    d_c = codec.device_alloc(corners.nbytes)
    d_w = codec.device_alloc(wells.nbytes)
    d_out = codec.device_alloc(2 * N * 96 * 120 * 120)
    try:
        for i in range(N):
            codec.h2d(d_fr + 2 * px * i, src[i % K])
        codec._ck(codec.lib.dbde_b200_encode16_device(codec.h, d_fr, W, H, 0, N, d_rec, cap, 0, d_off, d_sz, None), "encode16_device")
        codec.h2d(d_c, corners)
        codec.h2d(d_w, wells)
        codec.decode16_crops_device(d_rec, cap, d_off, W, H, N, d_c, 1, True, (256, 256), d_out, d_st, pad=0x8000)
        got = codec.d2h(d_out, 2 * N * 256 * 256, np.uint16).reshape(N, 256, 256)
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
        for i in range(N):
            assert np.array_equal(got[i], pad_crop(src[i % K][None], corners[i], 256, 256, 0x8000)[0, 0]), i
        codec.decode16_crops_device(d_rec, cap, d_off, W, H, N, d_w, 96, False, (120, 120), d_out, d_st)
        got = codec.d2h(d_out, 2 * N * 96 * 120 * 120, np.uint16).reshape(N, 96, 120, 120)
        want = pad_crop(src, wells, 120, 120, 0)
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
        for i in range(N):
            assert np.array_equal(got[i], want[i % K]), i
        for b in (2, 4, 8):
            codec.decode16_binned_device(d_rec, cap, d_off, W, H, N, b, d_out, d_st)
            got = codec.d2h(d_out, 2 * N * (px // (b * b)), np.uint16).reshape(N, H // b, W // b)
            want = block_mean(src, b)
            assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
            for i in range(N):
                assert np.array_equal(got[i], want[i % K]), (b, i)
    finally:
        for p in (d_fr, d_rec, d_off, d_sz, d_st, d_c, d_w, d_out):
            codec.device_free(p)
