"""Crop encode (dbde_b200_encode_crops_*) on a B200: N fixed-size windows per frame at shared or per-frame corners,
anywhere, pixels outside the frame set to a pad byte, each recorded as a frame of its own.  Record f * R + r must be
byte for byte the reference's dbde_pack_frame(first + f, crop image (f, r), crop_w, crop_h), where the crop image is
exactly what decode_crops returns; nothing outside the output range is written."""
import importlib
import os

import numpy as np
import pytest

import oracle
import synth
from conftest import rand_frame

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()
E_INVALID, E_CAPACITY = -1, -3
I32_MIN, I32_MAX = -2**31, 2**31 - 1

GEOMETRIES = [(2048, 2048), (2304, 48), (4104, 16), (2049, 9), (4100, 1003), (1001, 1003), (17, 23), (3, 5), (1, 1)]


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


def content(W, H, n=6):
    """rand_frame styles (every depth 0-8 inside one warp with 'classes') and synthetic mix / low / noise video"""
    rng = np.random.default_rng(W * 7919 + H + 5)
    fr = [rand_frame(rng, W, H, s) for s in ("classes", "noise", "flat")]
    for i, kind in enumerate(("mix", "low", "noise")):
        fr.append(synth.gen_frames(kind, 1, W, H, f0=i)[0])
    return np.stack(fr)[:n]


def pad_crop(frames, corners, cw, ch, pad):
    """the crop image (decode_crops' output): frames (N, H, W), corners (R, 2) or (N, R, 2) -> (N, R, ch, cw)"""
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


def want_records(frames, corners, cw, ch, pad, first, ora=ORA):
    """the reference's records, in the order f * R + r: crop r of every frame packed with frame indices first + f"""
    crops = pad_crop(frames, np.asarray(corners), cw, ch, pad)
    N, R = crops.shape[:2]
    recs = [None] * (N * R)
    for r in range(R):
        stream, sizes = ora.pack_frames(crops[:, r], first)
        offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        for f in range(N):
            recs[f * R + r] = stream[offs[f]:offs[f + 1]]
    return recs


def dev_encode(codec, frames, corners, size, pad=0, first=0, fshift=0, oshift=0, slot_stride=0, fill=0xA7):
    """encode_crops_device with the frames at base offset fshift and the slots at oshift, guard bytes before, between
    and after the records -> (records, sizes)"""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    corners = np.ascontiguousarray(corners, dtype=np.int32)
    N, H, W = frames.shape
    cw, ch = size
    per_frame = corners.ndim == 3
    R = corners.shape[-2]
    n = N * R
    stride = slot_stride or codec.slot_stride(cw, ch)
    total, G = n * stride, 64
    d_fr, d_c = codec.device_alloc(frames.nbytes + 32), codec.device_alloc(corners.nbytes)
    d_out, d_off, d_sz = codec.device_alloc(total + 2 * G + 16), codec.device_alloc(8 * n), codec.device_alloc(8 * n)
    try:
        codec.h2d(d_fr + fshift, frames)
        codec.h2d(d_c, corners)
        codec.h2d(d_out, np.full(total + 2 * G + 16, fill, dtype=np.uint8))
        codec.encode_crops_device(d_fr + fshift, W, H, first, N, d_c, R, per_frame, size, d_out + G + oshift, total, d_off, d_sz,
                                  pad=pad, slot_stride=slot_stride)
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
    mid-row, crops larger than the frame"""
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
    """every kind of crop size and corner on every geometry class, shared corners, pad 0, 255 and 0x5A, frame bases
    0-15 bytes off alignment and record slots at every offset mod 8"""
    fr = content(W, H)
    for i, (cw, ch) in enumerate(crop_sizes(W, H)):
        corners = corner_set(W, H, cw, ch)
        big = cw * ch > 1 << 16
        nf = 2 if big else len(fr)
        if big:
            corners = corners[i % 3::6]                     # a spread subset: large records stay small in memory
        pad = (0, 255, 0x5A)[i % 3]
        got, sizes = dev_encode(codec, fr[:nf], corners, (cw, ch), pad=pad, first=11 + i, fshift=(5 * i) % 16, oshift=i % 8)
        assert_records(got, want_records(fr[:nf], corners, cw, ch, pad, 11 + i), "%dx%d crops of %dx%d" % (cw, ch, W, H))


@pytest.mark.parametrize("W,H", [(1001, 1003), (2048, 2048), (61, 20)])
def test_per_frame_corners(codec, W, H):
    """per-frame corners scattered in and around the frame, some frames sharing theirs"""
    fr = content(W, H)
    N = len(fr)
    rng = np.random.default_rng(W + H)
    for cw, ch in [(61, 77), (120, 120), (9, 3)]:
        per = np.stack([rng.integers(-cw - 10, W + 10, (N, 7)), rng.integers(-ch - 10, H + 10, (N, 7))], axis=-1).astype(np.int32)
        per[1] = per[0]
        got, _ = dev_encode(codec, fr, per, (cw, ch), pad=0x5A, first=3, oshift=3)
        assert_records(got, want_records(fr, per, cw, ch, 0x5A, 3), "per-frame %dx%d" % (cw, ch))


@pytest.mark.parametrize("W,H", [(1001, 43), (2049, 9), (61, 20), (10, 10)])
def test_invert_endian_variant(codec, W, H):
    """DBDE_INVERT_ENDIAN: the crop image is assembled (pad and clamp padding) first, its tile rows reversed after"""
    V = oracle.best_variants()
    rng = np.random.default_rng(W + 31 * H)
    fr = np.stack([rand_frame(rng, W, H, ["classes", "noise", "classes"][i % 3]) for i in range(3)])
    corners = np.array([(W - 5, 0), (W - 3, H - 4), (W - 12, -2), (-3, 1), (W - 1, H // 2), (0, 0)], dtype=np.int32)
    c = pkg.Codec(0)
    try:
        c.set_invert_endian(True)
        for size in [(9, 7), (20, 3), (W + 4, H + 2)]:
            got, _ = dev_encode(c, fr, corners, size, pad=0xE1, first=9, oshift=1)
            want = want_records(fr, corners, *size, 0xE1, 9, ora=V)
            assert_records(got, want, "invert %r" % (size,))
            stream, offs = c.encode_crops_host(fr, corners, size, pad=0xE1, first_index=9)
            assert np.array_equal(stream, np.concatenate(want))
        plain, _ = dev_encode(codec, fr, corners, (9, 7), pad=0xE1, first=9)
        assert any(not np.array_equal(a, b) for a, b in zip(plain, want_records(fr, corners, 9, 7, 0xE1, 9, ora=V)))
    finally:
        c.close()


@pytest.mark.parametrize("oshift", [0, 2, 4, 6, 3])
def test_slot_stride_and_output_alignment(codec, oshift):
    """the default and larger slot strides (an odd one too), record bases at every alignment class: the aligned and
    the byte copy-out; guard bytes before, between and after the records stay untouched"""
    W, H = 1001, 203
    fr = content(W, H, 3)
    corners = np.array([(0, 0), (-5, 7), (990, 100), (333, 190), (500, -40)], dtype=np.int32)
    for cw, ch in [(64, 40), (37, 29), (300, 9)]:
        want = want_records(fr, corners, cw, ch, 0x33, 5)
        bound = codec.frame_record_bound(cw, ch)
        for stride in (0, bound + 16, bound + 3):
            got, _ = dev_encode(codec, fr, corners, (cw, ch), pad=0x33, first=5, oshift=oshift, slot_stride=stride)
            assert_records(got, want, "%dx%d stride %d shift %d" % (cw, ch, stride, oshift))


@pytest.mark.parametrize("W,H", [(2048, 64), (1001, 43)])
def test_whole_frame_crop_equals_encode_device(codec, W, H):
    """one shared corner (0, 0) and a crop of W x H: the same records, sizes and offsets as encode_device"""
    fr = content(W, H)
    N = len(fr)
    stride = codec.slot_stride(W, H)
    d_fr, d_out = codec.device_alloc(fr.nbytes), codec.device_alloc(N * stride)
    d_off, d_sz = codec.device_alloc(8 * N), codec.device_alloc(8 * N)
    try:
        codec.h2d(d_fr, fr)
        codec.h2d(d_out, np.full(N * stride, 0xA7, np.uint8))
        codec.encode_device(d_fr, W, H, 21, N, d_out, N * stride, d_off, d_sz)
        buf, offs, sizes = codec.d2h(d_out, N * stride), codec.d2h(d_off, 8 * N, np.uint64), codec.d2h(d_sz, 8 * N, np.uint64)
    finally:
        for p in (d_fr, d_out, d_off, d_sz):
            codec.device_free(p)
    got, gsizes = dev_encode(codec, fr, np.array([[0, 0]], np.int32), (W, H), first=21)
    assert gsizes.tolist() == sizes.tolist() and offs.tolist() == [j * stride for j in range(N)]
    for j in range(N):
        assert np.array_equal(got[j], buf[j * stride:j * stride + int(sizes[j])]), j


def test_round_trips(codec, tmp_path):
    """decode_device of the crop records is the crop image; decode_crops_device of the full records at the same
    corners gives the same pixels; a per-crop .dbde file (video header {3, crop_h, crop_w, hz}, then records
    f * R + r) reads back through read_file and the drop-in walker as that crop's frames with indices first + f"""
    W, H = 1001, 203
    fr = content(W, H)
    N = len(fr)
    corners = np.array([(10, 10), (-20, 150), (960, -3), (400, 100)], dtype=np.int32)
    R, (cw, ch), first = len(corners), (61, 57), 40
    crops = pad_crop(fr, corners, cw, ch, 0x5A)
    stream, offs = codec.encode_crops_host(fr, corners, (cw, ch), pad=0x5A, first_index=first)
    assert len(offs) == N * R + 1 and int(offs[-1]) == len(stream)
    dec, status, index = codec.decode_host(stream, offs[:N * R], cw, ch)
    assert (status == 0).all() and index.tolist() == [first + j // R for j in range(N * R)]
    assert np.array_equal(dec.reshape(N, R, ch, cw), crops)
    # decode_crops of the full frames' records at the same corners
    full, foffs = codec.encode_host(fr, first)
    dcrops, status, _ = codec.decode_crops_host(full, foffs[:N], W, H, corners, (cw, ch), pad=0x5A)
    assert (status == 0).all() and np.array_equal(dcrops, crops)
    # one .dbde file per crop
    drop = pkg.DropIn()
    for r in (0, 2):
        path = str(tmp_path / ("crop%d.dbde" % r))
        with open(path, "wb") as f:
            f.write(drop.pack_video_header(3, ch, cw, 25.0).tobytes())
            for fi in range(N):
                j = fi * R + r
                f.write(stream[int(offs[j]):int(offs[j + 1])].tobytes())
        (rw, rh, hz), frames, idx, st = pkg.read_file(codec, path)
        assert (rw, rh, hz) == (cw, ch, 25.0) and (st == 0).all() and idx.tolist() == [first + fi for fi in range(N)]
        assert np.array_equal(frames, crops[:, r])
        vh, walked = drop.walk_file(path)
        assert vh[1:3] == (ch, cw) and len(walked) == N
        for fi, (fh, img) in enumerate(walked):
            assert fh[1] == first + fi and np.array_equal(img, crops[fi, r])
        os.remove(path)


def test_host_form_equals_device_pinned_pageable_and_chunked(codec):
    """encode_crops_host: pageable numpy and pinned buffers, chunks of 3 frames in flight with per-frame corners that
    differ across chunk boundaries; its bytes are the device form's records back to back"""
    W, H, N = 1001, 203, 10
    cw, ch = 97, 45
    fr = synth.gen_frames("mix", N, W, H, f0=4)
    rng = np.random.default_rng(7)
    per = np.stack([rng.integers(-60, W, (N, 4)), rng.integers(-30, H, (N, 4))], axis=-1).astype(np.int32)
    want_per = want_records(fr, per, cw, ch, 0x42, 3)
    dev, _ = dev_encode(codec, fr, per, (cw, ch), pad=0x42, first=3, oshift=5)
    assert_records(dev, want_per, "device")
    want = np.concatenate(want_per)
    c = pkg.Codec(0)
    try:
        for chunk in (0, 3, 1):
            c.set_chunk_frames(chunk)
            stream, offs = c.encode_crops_host(fr, per, (cw, ch), pad=0x42, first_index=3)
            assert np.array_equal(stream, want), chunk
            assert offs.tolist() == np.concatenate([[0], np.cumsum([len(x) for x in want_per])]).tolist()
        shared = per[0]
        stream, _ = c.encode_crops_host(fr, shared, (cw, ch), pad=0x42, first_index=3)
        assert np.array_equal(stream, np.concatenate(want_records(fr, shared, cw, ch, 0x42, 3)))
        # pinned everything, output at an odd address; then pinned frames into pageable output and the reverse
        n = N * 4
        cap = codec.stream_bound(cw, ch, n)
        pfr, pc, pout, poff = c.pinned(fr.nbytes), c.pinned(per.nbytes), c.pinned(cap + 1), c.pinned(8 * (n + 1))
        try:
            pfr.array[:] = fr.ravel()
            pc.array[:] = per.view(np.uint8).ravel()
            for chunk in (3, 0):
                c.set_chunk_frames(chunk)
                assert c.lib.dbde_b200_encode_crops_host(c.h, pfr.ptr, W, H, 3, N, pc.ptr, 4, 1, cw, ch, 0x42, pout.ptr + 1, cap,
                                                         poff.ptr) == 0
                o = poff.array.view(np.uint64)
                assert int(o[n]) == len(want) and np.array_equal(pout.array[1:1 + len(want)], want)
                out = np.zeros(cap, np.uint8)
                offs = np.zeros(n + 1, np.uint64)
                assert c.lib.dbde_b200_encode_crops_host(c.h, pfr.ptr, W, H, 3, N, per.ctypes.data, 4, 1, cw, ch, 0x42,
                                                         out.ctypes.data, cap, offs.ctypes.data) == 0
                assert np.array_equal(out[:len(want)], want)
                pout.array[:] = 0
                assert c.lib.dbde_b200_encode_crops_host(c.h, fr.ctypes.data, W, H, 3, N, pc.ptr, 4, 1, cw, ch, 0x42, pout.ptr,
                                                         cap, poff.ptr) == 0
                assert np.array_equal(pout.array[:len(want)], want)
        finally:
            for p in (pfr, pc, pout, poff):
                p.free()
        # one byte short of the records' total
        out = np.zeros(len(want), np.uint8)
        offs = np.zeros(n + 1, np.uint64)
        assert c.lib.dbde_b200_encode_crops_host(c.h, fr.ctypes.data, W, H, 3, N, per.ctypes.data, 4, 1, cw, ch, 0x42,
                                                 out.ctypes.data, len(want) - 1, offs.ctypes.data) == E_CAPACITY
        assert c.lib.dbde_b200_encode_crops_host(c.h, fr.ctypes.data, W, H, 3, N, per.ctypes.data, 4, 1, cw, ch, 0x42,
                                                 out.ctypes.data, len(want), offs.ctypes.data) == 0
        assert np.array_equal(out, want)
    finally:
        c.close()


def test_host_form_thousands_of_records_per_chunk(codec):
    """64 frames x 1100 crops of 8 x 8: more records in one chunk than a grid dimension holds, compacted with one
    prefix; crops larger than the frame cap a chunk's records"""
    W, H, N = 512, 256, 64
    fr = synth.gen_frames("mix", N, W, H, f0=2)
    rng = np.random.default_rng(1100)
    corners = np.stack([rng.integers(-4, W - 4, 1100), rng.integers(-4, H - 4, 1100)], axis=-1).astype(np.int32)
    stream, offs = codec.encode_crops_host(fr, corners, (8, 8), pad=7, first_index=100)
    assert len(offs) == N * 1100 + 1
    want = want_records(fr, corners, 8, 8, 7, 100)
    assert int(offs[-1]) == len(stream) == sum(len(x) for x in want)
    assert np.array_equal(stream, np.concatenate(want))
    # many crops larger than the frame
    Ws, Hs, Ns = 64, 40, 5
    small = synth.gen_frames("mix", Ns, Ws, Hs)
    big = np.array([(-10, -20), (5, 3), (-200, 0)] * 30, dtype=np.int32)
    stream, _ = codec.encode_crops_host(small, big, (100, 70), pad=9, first_index=1)
    assert np.array_equal(stream, np.concatenate(want_records(small, big, 100, 70, 9, 1)))


def test_bad_arguments(codec):
    """each bad argument returns DBDE_B200_E_INVALID with nothing queued (the launch count does not move); too little
    capacity returns DBDE_B200_E_CAPACITY; an empty batch returns 0 and the host form writes offsets[0] = 0"""
    lib, h = codec.lib, codec.h
    W, H, N = 40, 24, 2
    fr = synth.gen_frames("mix", N, W, H)
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
        return lib.dbde_b200_encode_crops_device(*args)

    def host(*over, n=N, **kw):
        a = dict(ncrops=2, per_frame=0, cw=4, ch=3, pad=0, cap=cap)
        a.update(kw)
        args = [h, fr.ctypes.data, W, H, 5, n, corners.ctypes.data, a["ncrops"], a["per_frame"], a["cw"], a["ch"], a["pad"],
                out.ctypes.data, a["cap"], offs.ctypes.data]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_encode_crops_host(*args)

    try:
        l0 = codec.launches()
        bad = [dict(ncrops=0), dict(ncrops=-1), dict(cw=0), dict(ch=0), dict(cw=-4), dict(ch=-3),
               dict(cw=2**31 - 1, ch=2), dict(cw=1 << 16, ch=1 << 16), dict(ncrops=1 << 20, cw=64, ch=64), dict(ncrops=2**31 - 1, cw=1, ch=2),
               dict(per_frame=2), dict(per_frame=-1), dict(pad=-1), dict(pad=256)]
        for kw in bad:
            assert dev(**kw) == E_INVALID, kw
            assert host(**kw) == E_INVALID, kw
            assert dev(n=0, **kw) == E_INVALID, kw
            assert host(n=0, **kw) == E_INVALID, kw
        for i in (0, 1, 6, 12, 15, 16):                              # ctx, frames, corners, output, offsets, sizes
            assert dev((i, None)) == E_INVALID, i
        for i in (0, 1, 6, 12, 14):                                  # ctx, frames, corners, output, offsets
            assert host((i, None)) == E_INVALID, i
        for i, v in ((2, 0), (3, -1), (2, 1 << 30), (5, -1)):       # frame dims the limits reject, nframes < 0
            assert dev((i, v)) == E_INVALID and host((i, v)) == E_INVALID, (i, v)
        bound = codec.frame_record_bound(4, 3)
        assert dev(stride=bound - 1) == E_INVALID
        # nframes * ncrops past the int range (a 1 x 1 frame keeps the batch itself legal)
        assert lib.dbde_b200_encode_crops_device(h, d_fr, 1, 1, 0, 1 << 16, d_c, 1 << 16, 0, 1, 1, 0, d_out, cap, 0, d_off, d_sz,
                                                 None) == E_INVALID
        assert lib.dbde_b200_encode_crops_host(h, fr.ctypes.data, 1, 1, 0, 1 << 16, corners.ctypes.data, 1 << 16, 0, 1, 1, 0,
                                               out.ctypes.data, cap, offs.ctypes.data) == E_INVALID
        stride = codec.slot_stride(4, 3)
        assert dev(cap=2 * N * stride - 1) == E_CAPACITY and dev(cap=2 * N * (bound + 1) - 1, stride=bound + 1) == E_CAPACITY
        assert codec.launches() == l0
        offs[0] = 99
        assert dev(n=0) == 0 and host(n=0) == 0 and offs[0] == 0
        assert dev((1, None), (6, None), (12, None), (15, None), (16, None), n=0) == 0      # nothing to do, nothing read
        assert codec.launches() == l0
        # the context is still usable, and the last good calls encode
        assert dev(cap=2 * N * stride) == 0 and codec.launches() == l0 + 1
        want = want_records(fr, corners, 4, 3, 0, 5)
        sizes = codec.d2h(d_sz, 8 * 2 * N, np.uint64)
        buf = codec.d2h(d_out, 2 * N * stride)
        for j in range(2 * N):
            assert np.array_equal(buf[j * stride:j * stride + int(sizes[j])], want[j]), j
        assert host() == 0 and np.array_equal(out[:int(offs[2 * N])], np.concatenate(want))
    finally:
        for p in (d_fr, d_c, d_out, d_off, d_sz):
            codec.device_free(p)
