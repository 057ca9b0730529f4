"""DBDE16 crop encode (dbde_b200_encode16_crops_*) on a B200: N fixed-size windows of every 16-bit frame at shared or
per-frame corners, anywhere, pixels outside the frame set to a U16 pad value, each recorded as a DBDE16 frame of its own.
Record f * R + r must be byte for byte oracle.port16's record of the crop image (f, r) with frame index first + f, where
the crop image is exactly what decode16_crops returns; nothing outside the output range is written."""
import importlib

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("dbce-video-cpp_b200")
P16 = oracle.port16
E_INVALID, E_CAPACITY = -1, -3
I32_MIN, I32_MAX = -2**31, 2**31 - 1

# the DBDE16 sub-frame decode tests' geometries, sCMOS sizes included
GEOMETRIES = [(2048, 2048), (2304, 48), (1280, 64), (4096, 8), (4104, 16), (2049, 9), (4100, 1003), (1001, 1003),
              (17, 23), (3, 5), (1, 1), (2304, 2304), (2560, 2160)]
PADS = (0, 65535, 0x1234)


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


def rand_frame16(rng, W, H, style):
    """'classes': every depth 0..16 among the tiles of one warp; 'sensor12': a 12-bit camera-like smooth field plus 5
    bits of noise; 'byte': pixels that fit in 8 bits"""
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


def content(W, H, styles=("classes", "noise", "flat", "byte", "sensor12")):
    rng = np.random.default_rng(W * 7919 + H + 1616)
    return np.stack([rand_frame16(rng, W, H, s) for s in styles])


def pad_crop(frames, corners, cw, ch, pad):
    """the crop image (decode16_crops' output): frames (N, H, W), corners (R, 2) or (N, R, 2) -> (N, R, ch, cw)"""
    N, H, W = frames.shape
    corners = np.asarray(corners)
    c = np.broadcast_to(corners, (N,) + corners.shape) if corners.ndim == 2 else corners
    out = np.full((N, c.shape[1], ch, cw), pad, dtype=frames.dtype)
    for f in range(N):
        for r in range(c.shape[1]):
            x0, y0 = int(c[f, r, 0]), int(c[f, r, 1])
            xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
            if xa < xb and ya < yb:
                out[f, r, ya - y0:yb - y0, xa - x0:xb - x0] = frames[f, ya:yb, xa:xb]
    return out


def want_records(frames, corners, cw, ch, pad, first):
    """the oracle's DBDE16 records, in the order f * R + r: crop r of every frame packed with frame indices first + f"""
    crops = pad_crop(frames, corners, cw, ch, pad)
    N, R = crops.shape[:2]
    recs = [None] * (N * R)
    for r in range(R):
        stream, sizes = P16.pack_frames(crops[:, r], first)
        offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        for f in range(N):
            recs[f * R + r] = stream[offs[f]:offs[f + 1]]
    return recs


def stride16(codec, W, H):
    return int(codec.lib.dbde_b200_slot_stride16(W, H))


def bound16(codec, W, H):
    return int(codec.lib.dbde_b200_frame_record_bound16(W, H))


def dev_encode(codec, frames, corners, size, pad=0, first=0, fshift=0, oshift=0, slot_stride=0, fill=0xA7):
    """encode16_crops_device with the frames at base offset fshift (even) and the slots at oshift, guard bytes before,
    between and after the records; checks the guards, frame_offsets and the one launch -> (records, sizes)"""
    frames = np.ascontiguousarray(frames, dtype=np.uint16)
    corners = np.ascontiguousarray(corners, dtype=np.int32)
    N, H, W = frames.shape
    cw, ch = size
    per_frame = corners.ndim == 3
    R = corners.shape[-2]
    n = N * R
    stride = slot_stride or stride16(codec, cw, ch)
    total, G = n * stride, 64
    d_fr, d_c = codec.device_alloc(frames.nbytes + 32), codec.device_alloc(corners.nbytes)
    d_out, d_off, d_sz = codec.device_alloc(total + 2 * G + 16), codec.device_alloc(8 * n), codec.device_alloc(8 * n)
    try:
        codec.h2d(d_fr + fshift, frames)
        codec.h2d(d_c, corners)
        codec.h2d(d_out, np.full(total + 2 * G + 16, fill, dtype=np.uint8))
        l0 = codec.launches()
        codec.encode16_crops_device(d_fr + fshift, W, H, first, N, d_c, R, per_frame, size, d_out + G + oshift, total, d_off, d_sz,
                                    pad=pad, slot_stride=slot_stride)
        assert codec.launches() == l0 + 1
        buf = codec.d2h(d_out, total + 2 * G + 16)
        offs, sizes = codec.d2h(d_off, 8 * n, np.uint64), codec.d2h(d_sz, 8 * n, np.uint64)
    finally:
        for p in (d_fr, d_c, d_out, d_off, d_sz):
            codec.device_free(p)
    assert (buf[:G + oshift] == fill).all() and (buf[G + oshift + total:] == fill).all(), ("wrote outside the slots", size)
    assert offs.tolist() == [j * stride for j in range(n)]
    recs = []
    for j in range(n):
        a = G + oshift + j * stride
        recs.append(buf[a:a + int(sizes[j])])
        assert (buf[a + int(sizes[j]):a + stride] == fill).all(), ("wrote past record", j)
    return recs, sizes


def assert_records(got, want, what):
    assert len(got) == len(want), what
    for j, (g, w) in enumerate(zip(got, want)):
        if len(g) != len(w) or not np.array_equal(g, w):
            n = min(len(g), len(w))
            bad = np.argwhere(g[:n] != w[:n])
            pytest.fail("%s: record %d differs (sizes %d, %d; first differing byte %s)"
                        % (what, j, len(g), len(w), bad[0][0] if len(bad) else n))


def crop_sizes(W, H):
    """every crop_w and crop_h mod 8, widths across the 32- and 256-tile boundaries, chunks of 256 tiles ending
    mid-row, crops larger than the frame, 1 x 1 and the whole frame"""
    S = {(1, 1), (W, H), (W + 9, H + 5), (13, 11), (8, 8), (8 * 33 + 3, 5), (8 * 257 + 5, 2), (8 * 17 + 1, 8 * 16 + 3)}
    for b in range(8):
        S |= {(b + 8, 1 + b)}
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
def test_records_equal_the_oracle(codec, W, H):
    """every kind of crop size and corner on every geometry class, the five content classes, shared corners, pads 0,
    65535 and 0x1234, frame bases at every even offset mod 16 and record slots at every offset mod 8"""
    fr = content(W, H)
    for i, (cw, ch) in enumerate(crop_sizes(W, H)):
        corners = corner_set(W, H, cw, ch)
        big = cw * ch > 1 << 16
        nf = 2 if big else len(fr)
        if big:
            corners = corners[i % 3::6]                     # a spread subset: large records stay small in memory
        pad = PADS[i % 3]
        got, _ = dev_encode(codec, fr[:nf], corners, (cw, ch), pad=pad, first=11 + i, fshift=(2 * i) % 16, oshift=i % 8)
        assert_records(got, want_records(fr[:nf], corners, cw, ch, pad, 11 + i), "%dx%d crops of %dx%d" % (cw, ch, W, H))


@pytest.mark.parametrize("W,H", [(1001, 1003), (2048, 2048), (61, 20)])
def test_per_frame_corners_random_walk(codec, W, H):
    """per-frame corners on a random walk that wanders in and out of the frame, frame indices above 2^32 (all eight
    index bytes differ from zero)"""
    fr = content(W, H)
    N = len(fr)
    rng = np.random.default_rng(W + H)
    first = 0x0102030405060708
    for cw, ch in [(61, 77), (256, 256), (9, 3)]:
        start = np.array([rng.integers(-cw // 2, W), rng.integers(-ch // 2, H)])
        walk = (start + np.cumsum(rng.integers(-max(W, H) // 4 - 1, max(W, H) // 4 + 2, (N, 3, 2)), axis=0)).astype(np.int32)
        walk[1] = walk[0]
        got, _ = dev_encode(codec, fr, walk, (cw, ch), pad=0x1234, first=first, oshift=3)
        assert_records(got, want_records(fr, walk, cw, ch, 0x1234, first), "per-frame %dx%d" % (cw, ch))


@pytest.mark.parametrize("wmod", [0, 1, 3, 4, 7])
def test_load_paths(codec, wmod):
    """frame bases 0, 2, ..., 14 bytes past a 16-byte boundary crossed with W % 8 and every x0 residue: inner tile rows
    from one aligned word, from two shifted words, and edge tiles"""
    W, H = 64 + wmod, 40
    fr = content(W, H, ("classes", "noise", "sensor12"))
    corners = np.array([(8 + a, 3 + a) for a in range(8)] + [(a - 8, 5) for a in range(8)] + [(W - 20 + a, H - 18) for a in range(8)],
                       dtype=np.int32)
    for fshift in range(0, 16, 2):
        for size in [(40, 24), (17, 9)]:
            got, _ = dev_encode(codec, fr, corners, size, pad=0x1234, first=2, fshift=fshift, oshift=fshift % 8)
            assert_records(got, want_records(fr, corners, *size, 0x1234, 2), "W %d base %d size %r" % (W, fshift, size))
    # an odd frame pointer
    d_fr, d_out, d_off, d_sz = codec.device_alloc(fr.nbytes + 32), codec.device_alloc(1 << 20), codec.device_alloc(512), codec.device_alloc(512)
    d_c = codec.device_alloc(corners.nbytes)
    try:
        codec.h2d(d_c, corners)
        l0 = codec.launches()
        assert codec.lib.dbde_b200_encode16_crops_device(codec.h, d_fr + 1, W, H, 0, 1, d_c, len(corners), 0, 17, 9, 0, d_out, 1 << 20, 0,
                                                         d_off, d_sz, None) == E_INVALID
        assert codec.launches() == l0
    finally:
        for p in (d_fr, d_out, d_off, d_sz, d_c):
            codec.device_free(p)


@pytest.mark.parametrize("oshift", range(8))
def test_slot_stride_and_output_alignment(codec, oshift):
    """the default slot stride and the bound plus 1, 3 and 7 (the byte copy-out), record bases at every offset mod 8;
    guard bytes before, between and after the records, and past each record in its slot, stay untouched"""
    W, H = 1001, 203
    fr = content(W, H, ("classes", "noise", "sensor12"))
    corners = np.array([(0, 0), (-5, 7), (990, 100), (333, 190), (500, -40)], dtype=np.int32)
    for cw, ch in [(64, 40), (37, 29), (300, 9)]:
        want = want_records(fr, corners, cw, ch, 0x3333, 5)
        bound = bound16(codec, cw, ch)
        for stride in (0, bound + 1, bound + 3, bound + 7):
            got, sizes = dev_encode(codec, fr, corners, (cw, ch), pad=0x3333, first=5, oshift=oshift, slot_stride=stride)
            assert_records(got, want, "%dx%d stride %d shift %d" % (cw, ch, stride, oshift))
            assert sizes.tolist() == [len(x) for x in want]


@pytest.mark.parametrize("W,H", [(2048, 64), (1001, 43), (2560, 40), (13, 7)])
def test_whole_frame_crop_equals_encode16_device(codec, W, H):
    """one shared corner (0, 0) and a crop of W x H: the same records, sizes and offsets as encode16_device"""
    fr = content(W, H)
    N = len(fr)
    stride = stride16(codec, W, H)
    d_fr, d_out = codec.device_alloc(fr.nbytes), codec.device_alloc(N * stride)
    d_off, d_sz = codec.device_alloc(8 * N), codec.device_alloc(8 * N)
    try:
        codec.h2d(d_fr, fr)
        codec.h2d(d_out, np.full(N * stride, 0xA7, np.uint8))
        codec._ck(codec.lib.dbde_b200_encode16_device(codec.h, d_fr, W, H, 21, N, d_out, N * stride, 0, d_off, d_sz, None),
                  "encode16_device")
        buf, offs, sizes = codec.d2h(d_out, N * stride), codec.d2h(d_off, 8 * N, np.uint64), codec.d2h(d_sz, 8 * N, np.uint64)
    finally:
        for p in (d_fr, d_out, d_off, d_sz):
            codec.device_free(p)
    got, gsizes = dev_encode(codec, fr, np.array([[0, 0]], np.int32), (W, H), first=21)
    assert gsizes.tolist() == sizes.tolist() and offs.tolist() == [j * stride for j in range(N)]
    for j in range(N):
        assert np.array_equal(got[j], buf[j * stride:j * stride + int(sizes[j])]), j


@pytest.mark.parametrize("W,H", [(1001, 203), (64, 48)])
def test_8bit_embedding(codec, W, H):
    """pixels and pad that fit in 8 bits: each DBDE16 record has the 8-bit crop encoder's index, depth plane and words,
    and its minimum plane is the 8-bit one widened"""
    rng = np.random.default_rng(W)
    fr8 = np.stack([rng.integers(0, 256, (H, W)).astype(np.uint8), (np.arange(W)[None, :] // 7 + np.arange(H)[:, None] // 5).astype(np.uint8),
                    (rng.integers(0, 4, (H, W)) + 100).astype(np.uint8)])
    corners = np.array([(0, 0), (-5, 7), (W - 30, H // 2), (W // 3, -9), (W + 3, 0)], dtype=np.int32)
    N, R = len(fr8), len(corners)
    for (cw, ch), pad in [((61, 37), 0x5A), ((8, 8), 0), ((130, 11), 255)]:
        got16, _ = dev_encode(codec, fr8.astype(np.uint16), corners, (cw, ch), pad=pad, first=77)
        n = N * R
        stride = codec.slot_stride(cw, ch)
        d_fr, d_c = codec.device_alloc(fr8.nbytes), codec.device_alloc(corners.nbytes)
        d_out, d_off, d_sz = codec.device_alloc(n * stride), codec.device_alloc(8 * n), codec.device_alloc(8 * n)
        try:
            codec.h2d(d_fr, fr8)
            codec.h2d(d_c, corners)
            codec.encode_crops_device(d_fr, W, H, 77, N, d_c, R, False, (cw, ch), d_out, n * stride, d_off, d_sz, pad=pad)
            buf, sizes = codec.d2h(d_out, n * stride), codec.d2h(d_sz, 8 * n, np.uint64)
        finally:
            for p in (d_fr, d_c, d_out, d_off, d_sz):
                codec.device_free(p)
        wh = ((cw + 7) // 8) * ((ch + 7) // 8)
        for j in range(n):
            r8, r16 = buf[j * stride:j * stride + int(sizes[j])], got16[j]
            assert np.array_equal(r8[:24 + wh], r16[:24 + wh]), j                       # tag, index, 0.0, wh, depths
            assert np.array_equal(r8[28 + wh:28 + 2 * wh], r16[28 + wh:28 + 3 * wh:2]), j   # minimum: low bytes
            assert not r16[29 + wh:28 + 3 * wh:2].any(), j                              # minimum: high bytes zero
            assert np.array_equal(r8[28 + 2 * wh:], r16[28 + 3 * wh:]), j               # n64 and words


def test_round_trips(codec):
    """decode16_device at crop_w x crop_h returns the crop images; index_stream16 of the host form's stream returns its
    offsets; decode16_crops_host of a full-frame encode16_host stream at the same corners returns the same images"""
    W, H = 1001, 203
    fr = content(W, H)
    N = len(fr)
    corners = np.array([(10, 10), (-20, 150), (960, -3), (400, 100), (-500, 0)], dtype=np.int32)
    R, (cw, ch), first = len(corners), (61, 57), 40
    crops = pad_crop(fr, corners, cw, ch, 0xBEEF)
    stream, offs = codec.encode16_crops_host(fr, corners, (cw, ch), pad=0xBEEF, first_index=first)
    n = N * R
    assert len(offs) == n + 1 and int(offs[-1]) == len(stream)
    d_s, d_o = codec.device_alloc(len(stream)), codec.device_alloc(8 * n)
    d_fr, d_st, d_ix = codec.device_alloc(2 * n * cw * ch), codec.device_alloc(4 * n), codec.device_alloc(8 * n)
    try:
        codec.h2d(d_s, stream)
        codec.h2d(d_o, offs[:n])
        codec._ck(codec.lib.dbde_b200_decode16_device(codec.h, d_s, len(stream), d_o, cw, ch, n, d_fr, d_st, d_ix, None),
                  "decode16_device")
        dec = codec.d2h(d_fr, 2 * n * cw * ch, np.uint16)
        status, index = codec.d2h(d_st, 4 * n, np.uint32), codec.d2h(d_ix, 8 * n, np.uint64)
    finally:
        for p in (d_s, d_o, d_fr, d_st, d_ix):
            codec.device_free(p)
    assert (status == 0).all() and index.tolist() == [first + j // R for j in range(n)]
    assert np.array_equal(dec.reshape(N, R, ch, cw), crops)
    ix = np.zeros(n + 2, np.uint64)
    assert codec.lib.dbde_b200_index_stream16(stream.ctypes.data, len(stream), cw, ch, ix.ctypes.data, n + 1) == n
    assert ix[:n + 1].tolist() == offs.tolist()
    full, foffs = codec.encode16_host(fr, first)
    dcrops, status, _ = codec.decode16_crops_host(full, foffs[:N], W, H, corners, (cw, ch), pad=0xBEEF)
    assert (status == 0).all() and np.array_equal(dcrops, crops)


def test_invert_endian_changes_nothing(codec):
    """DBDE16 has no invert-endian variant: with set_invert_endian(1) the device and host forms write the same bytes"""
    W, H = 1001, 43
    fr = content(W, H, ("classes", "noise", "sensor12"))
    corners = np.array([(W - 5, 0), (W - 3, H - 4), (W - 12, -2), (-3, 1), (W - 1, H // 2), (0, 0)], dtype=np.int32)
    c = pkg.Codec(0)
    try:
        c.set_invert_endian(True)
        for size in [(9, 7), (20, 3), (W + 4, H + 2)]:
            want = want_records(fr, corners, *size, 0xE1E1, 9)
            got, _ = dev_encode(c, fr, corners, size, pad=0xE1E1, first=9, oshift=1)
            assert_records(got, want, "invert %r" % (size,))
            stream, _ = c.encode16_crops_host(fr, corners, size, pad=0xE1E1, first_index=9)
            assert np.array_equal(stream, np.concatenate(want))
    finally:
        c.close()


def test_host_form_equals_device_pinned_pageable_and_chunked(codec):
    """encode16_crops_host: pageable numpy and pinned buffers, chunks of 3 frames in flight (a partial last chunk) with
    per-frame corners that differ across chunk boundaries; its bytes are the device form's records back to back"""
    W, H, N = 1001, 203, 10
    cw, ch = 97, 45
    rng = np.random.default_rng(7)
    fr = np.stack([rand_frame16(rng, W, H, ("sensor12", "classes")[i % 2]) for i in range(N)])
    per = np.stack([rng.integers(-60, W, (N, 4)), rng.integers(-30, H, (N, 4))], axis=-1).astype(np.int32)
    want_per = want_records(fr, per, cw, ch, 0x4242, 3)
    dev, _ = dev_encode(codec, fr, per, (cw, ch), pad=0x4242, first=3, oshift=5)
    assert_records(dev, want_per, "device")
    want = np.concatenate(want_per)
    c = pkg.Codec(0)
    try:
        for chunk in (0, 3, 1):
            c.set_chunk_frames(chunk)
            stream, offs = c.encode16_crops_host(fr, per, (cw, ch), pad=0x4242, first_index=3)
            assert np.array_equal(stream, want), chunk
            assert offs.tolist() == np.concatenate([[0], np.cumsum([len(x) for x in want_per])]).tolist()
        shared = per[0]
        stream, _ = c.encode16_crops_host(fr, shared, (cw, ch), pad=0x4242, first_index=3)
        assert np.array_equal(stream, np.concatenate(want_records(fr, shared, cw, ch, 0x4242, 3)))
        # pinned everything, output at an odd address; then pinned frames into pageable output and the reverse
        n = N * 4
        cap = stride16(c, cw, ch) * n + 16
        pfr, pc, pout, poff = c.pinned(fr.nbytes), c.pinned(per.nbytes), c.pinned(cap + 1), c.pinned(8 * (n + 1))
        try:
            pfr.array[:] = fr.view(np.uint8).ravel()
            pc.array[:] = per.view(np.uint8).ravel()
            lib = c.lib.dbde_b200_encode16_crops_host
            for chunk in (3, 0):
                c.set_chunk_frames(chunk)
                assert lib(c.h, pfr.ptr, W, H, 3, N, pc.ptr, 4, 1, cw, ch, 0x4242, pout.ptr + 1, cap, poff.ptr) == 0
                o = poff.array.view(np.uint64)
                assert int(o[n]) == len(want) and np.array_equal(pout.array[1:1 + len(want)], want)
                out = np.zeros(cap, np.uint8)
                offs = np.zeros(n + 1, np.uint64)
                assert lib(c.h, pfr.ptr, W, H, 3, N, per.ctypes.data, 4, 1, cw, ch, 0x4242, out.ctypes.data, cap, offs.ctypes.data) == 0
                assert np.array_equal(out[:len(want)], want)
                pout.array[:] = 0
                assert lib(c.h, fr.ctypes.data, W, H, 3, N, pc.ptr, 4, 1, cw, ch, 0x4242, pout.ptr, cap, poff.ptr) == 0
                assert np.array_equal(pout.array[:len(want)], want)
        finally:
            for p in (pfr, pc, pout, poff):
                p.free()
        # one byte short of the records' total
        out = np.zeros(len(want), np.uint8)
        offs = np.zeros(n + 1, np.uint64)
        lib = c.lib.dbde_b200_encode16_crops_host
        assert lib(c.h, fr.ctypes.data, W, H, 3, N, per.ctypes.data, 4, 1, cw, ch, 0x4242, out.ctypes.data, len(want) - 1,
                   offs.ctypes.data) == E_CAPACITY
        assert lib(c.h, fr.ctypes.data, W, H, 3, N, per.ctypes.data, 4, 1, cw, ch, 0x4242, out.ctypes.data, len(want), offs.ctypes.data) == 0
        assert np.array_equal(out, want)
    finally:
        c.close()


def test_host_form_thousands_of_records_per_chunk(codec):
    """64 frames x 1100 crops of 8 x 8: more records in one chunk than a grid dimension holds, compacted with one
    prefix; then 100 crops of 256 x 256 of 16 x 16 frames: crops larger than the frame, 13 MB of record slots per frame,
    so the 64 MiB cap splits 12 frames into chunks of 5, 5 and 2"""
    W, H, N = 512, 256, 64
    rng = np.random.default_rng(1100)
    fr = np.stack([rand_frame16(rng, W, H, "sensor12") for _ in range(N)])
    corners = np.stack([rng.integers(-4, W - 4, 1100), rng.integers(-4, H - 4, 1100)], axis=-1).astype(np.int32)
    stream, offs = codec.encode16_crops_host(fr, corners, (8, 8), pad=7, first_index=100)
    assert len(offs) == N * 1100 + 1
    want = want_records(fr, corners, 8, 8, 7, 100)
    assert int(offs[-1]) == len(stream) == sum(len(x) for x in want)
    assert np.array_equal(stream, np.concatenate(want))
    small = np.stack([rand_frame16(rng, 16, 16, "noise") for _ in range(12)])
    big = np.array([(-10, -20), (5, 3), (-200, 0), (-120, -120)] * 25, dtype=np.int32)
    assert 100 * stride16(codec, 256, 256) * 5 <= 64 << 20 < 100 * stride16(codec, 256, 256) * 6
    stream, offs = codec.encode16_crops_host(small, big, (256, 256), pad=9, first_index=1)
    assert np.array_equal(stream, np.concatenate(want_records(small, big, 256, 256, 9, 1)))


def test_bad_arguments(codec):
    """each bad argument returns DBDE_B200_E_INVALID with nothing queued (the launch count does not move); too little
    capacity returns DBDE_B200_E_CAPACITY; an empty batch returns 0 and the host form writes offsets[0] = 0"""
    lib, h = codec.lib, codec.h
    W, H, N = 40, 24, 2
    fr = content(W, H, ("sensor12", "noise"))
    corners = np.array([[1, 2], [3, 4]], dtype=np.int32)
    d_fr, d_c = codec.device_alloc(fr.nbytes), codec.device_alloc(corners.nbytes)
    cap = 1 << 16
    d_out, d_off, d_sz = codec.device_alloc(cap), codec.device_alloc(64), codec.device_alloc(64)
    codec.h2d(d_fr, fr)
    codec.h2d(d_c, corners)
    out = np.zeros(cap, np.uint8)
    offs = np.zeros(8, np.uint64)

    def dev(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0, cap=cap, stride=0)
        a.update(kw)
        args = [h, d_fr, W, H, 5, n, d_c, a["ncrops"], a["per_frame"], a["cw"], a["ch"], a["pad"], d_out, a["cap"], a["stride"], d_off,
                d_sz, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_encode16_crops_device(*args)

    def host(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0, cap=cap)
        a.update(kw)
        args = [h, fr.ctypes.data, W, H, 5, n, corners.ctypes.data, a["ncrops"], a["per_frame"], a["cw"], a["ch"], a["pad"],
                out.ctypes.data, a["cap"], offs.ctypes.data]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_encode16_crops_host(*args)

    try:
        l0 = codec.launches()
        bad = [dict(ncrops=0), dict(ncrops=-1), dict(cw=0), dict(ch=0), dict(cw=-4), dict(ch=-3),
               dict(cw=2**31 - 1, ch=2), dict(cw=1 << 16, ch=1 << 16), dict(ncrops=1 << 20, cw=64, ch=64), dict(ncrops=2**31 - 1, cw=1, ch=2),
               dict(per_frame=2), dict(per_frame=-1), dict(pad=-1), dict(pad=65536)]
        for kw in bad:
            assert dev(**kw) == E_INVALID, kw
            assert host(**kw) == E_INVALID, kw
            assert dev(n=0, **kw) == E_INVALID, kw
            assert host(n=0, **kw) == E_INVALID, kw
        for i in (0, 1, 6, 12, 15, 16):                              # ctx, frames, corners, output, offsets, sizes
            assert dev((i, None)) == E_INVALID, i
        for i in (0, 1, 6, 12, 14):                                  # ctx, frames, corners, output, offsets
            assert host((i, None)) == E_INVALID, i
        assert dev((1, d_fr + 1)) == E_INVALID and dev((1, d_fr + 3), n=0) == E_INVALID    # frames not 2-byte aligned
        for i, v in ((2, 0), (3, -1), (2, 1 << 30), (5, -1)):       # frame dims the limits reject, nframes < 0
            assert dev((i, v)) == E_INVALID and host((i, v)) == E_INVALID, (i, v)
        bound = bound16(codec, 4, 3)
        assert dev(stride=bound - 1) == E_INVALID
        # nframes * ncrops past the int range (a 1 x 1 frame keeps the batch itself legal)
        assert lib.dbde_b200_encode16_crops_device(h, d_fr, 1, 1, 0, 1 << 16, d_c, 1 << 16, 0, 1, 1, 0, d_out, cap, 0, d_off, d_sz,
                                                   None) == E_INVALID
        assert lib.dbde_b200_encode16_crops_host(h, fr.ctypes.data, 1, 1, 0, 1 << 16, corners.ctypes.data, 1 << 16, 0, 1, 1, 0,
                                                 out.ctypes.data, cap, offs.ctypes.data) == E_INVALID
        stride = stride16(codec, 4, 3)
        assert dev(cap=2 * N * stride - 1) == E_CAPACITY and dev(cap=2 * N * (bound + 1) - 1, stride=bound + 1) == E_CAPACITY
        assert codec.launches() == l0
        offs[0] = 99
        assert dev(n=0) == 0 and host(n=0) == 0 and offs[0] == 0
        assert dev((1, None), (6, None), (12, None), (15, None), (16, None), n=0) == 0      # nothing to do, nothing read
        assert codec.launches() == l0
        # the context is still usable, pad 65535 is accepted, and the last good calls encode
        assert dev(cap=2 * N * stride, pad=65535) == 0 and codec.launches() == l0 + 1
        want = want_records(fr, corners, 4, 3, 65535, 5)
        sizes = codec.d2h(d_sz, 8 * 2 * N, np.uint64)
        buf = codec.d2h(d_out, 2 * N * stride)
        for j in range(2 * N):
            assert np.array_equal(buf[j * stride:j * stride + int(sizes[j])], want[j]), j
        assert host(pad=65535) == 0 and np.array_equal(out[:int(offs[2 * N])], np.concatenate(want))
    finally:
        for p in (d_fr, d_c, d_out, d_off, d_sz):
            codec.device_free(p)
