"""Binned decode (dbde_b200_decode_binned_*) on a B200: every frame reduced to the rounded means of its factor x factor
blocks.  The expected output is a numpy block mean of the source frames (the codec is lossless, so they are the full
decode) over the in-frame pixels only, (sum + n // 2) // n; validation covers the whole record with the full decoder's
status bits, and nothing outside the output range is written."""
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
FACTORS = [1, 2, 4, 8]

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


def block_mean(frames, b):
    """the reference: frames (N, H, W) -> (N, ceil(H / b), ceil(W / b)), the mean of each block's in-frame pixels,
    rounded half up"""
    N, H, W = frames.shape
    Hb, Wb = -(-H // b), -(-W // b)
    p = np.zeros((N, Hb * b, Wb * b), np.uint32)
    p[:, :H, :W] = frames
    m = np.zeros((Hb * b, Wb * b), np.uint32)
    m[:H, :W] = 1
    s = p.reshape(N, Hb, b, Wb, b).sum(axis=(2, 4))
    n = m.reshape(Hb, b, Wb, b).sum(axis=(1, 3))
    return ((s + n // 2) // n).astype(np.uint8)


def encoded(W, H, frames=None, first=11, ora=ORA):
    fr = content(W, H) if frames is None else frames
    stream, sizes = ora.pack_frames(fr, first)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    return fr, stream, offs


class DevStream:
    """records and their offsets uploaded once; binned() decodes into a guarded output buffer"""
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

    def binned(self, b, shift=0, fill=0xA7, codec=None):
        """decode_binned_device at output base offset `shift`; checks the guards -> (frames (N, Hb, Wb), status, indices)"""
        c, N, G = codec or self.codec, self.N, self.G
        Hb, Wb = -(-self.H // b), -(-self.W // b)
        n = N * Hb * Wb
        d_out = c.device_alloc(n + 2 * G + 16)
        try:
            c.h2d(d_out, np.full(n + 2 * G + 16, fill, dtype=np.uint8))
            c.decode_binned_device(self.d_s, self.nbytes, self.d_o, self.W, self.H, N, b, d_out + G + shift, self.d_st, self.d_ix)
            buf = c.d2h(d_out, n + 2 * G + 16)
        finally:
            c.device_free(d_out)
        assert (buf[:G + shift] == fill).all() and (buf[G + shift + n:] == fill).all(), ("wrote outside the output", b, shift)
        return (buf[G + shift:G + shift + n].reshape(N, Hb, Wb), c.d2h(self.d_st, 4 * N, np.uint32),
                c.d2h(self.d_ix, 8 * N, np.uint64))

    def free(self):
        for p in (self.d_s, self.d_o, self.d_st, self.d_ix):
            self.codec.device_free(p)


def check(got, want, what):
    if not np.array_equal(got, want):
        bad = tuple(np.argwhere(got != want)[0])
        pytest.fail("%s differs first at (frame, row, col) %r: %d != %d" % (what, bad, got[bad], want[bad]))


@pytest.mark.parametrize("W,H", GEOMETRIES)
def test_binned_equals_the_block_mean(codec, W, H):
    """every factor on every geometry class of the region tests, at a few output offsets"""
    fr, stream, offs = encoded(W, H)
    full, idx, _ = ORA.unpack_frames(stream, W, H, len(fr))
    assert (full == fr).all() and idx == list(range(11, 11 + len(fr)))
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        for i, b in enumerate(FACTORS):
            got, status, index = d.binned(b, shift=(3 * i + W) % 16)
            assert (status == 0).all() and index.tolist() == list(range(11, 11 + len(fr))), b
            check(got, block_mean(fr, b), "%dx%d binned by %d" % (W, H, b))
    finally:
        d.free()


def partial_geometries():
    """per factor: the last bin partial in x only, in y only, in both; a partial last tile whose bins are all full; one
    row and one column"""
    out = []
    for b in (2, 4, 8):
        r = b - 1
        out += [(b, 72 + r, 40), (b, 40, 72 + r), (b, 64 + 1, 40 + r), (b, 2048 + 8 + r, 19), (b, 1, 77), (b, 77, 1)]
        if b < 8:
            out += [(b, 72 + b, 40 + b)]
    return out


@pytest.mark.parametrize("b,W,H", partial_geometries())
def test_partial_last_bins_average_only_in_frame_pixels(codec, b, W, H):
    """the encoder pads a partial tile by repeating the last valid pixel: that padding must not enter the edge bins.
    Noise and 'classes' content make any such bias visible."""
    fr, stream, offs = encoded(W, H)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        got, status, _ = d.binned(b, shift=b + 1)
        assert (status == 0).all()
        want = block_mean(fr, b)
        check(got, want, "%dx%d binned by %d" % (W, H, b))
        if W % b >= 2 or H % b >= 2:
            # a partial bin with two or more in-frame columns or rows: counting the last pixel's repeats would differ
            Hb, Wb = want.shape[1:]
            pw = np.pad(fr, ((0, 0), (0, Hb * b - H), (0, Wb * b - W)), mode="edge").astype(np.uint32)
            biased = ((pw.reshape(len(fr), Hb, b, Wb, b).sum(axis=(2, 4)) + b * b // 2) // (b * b)).astype(np.uint8)
            assert not np.array_equal(biased, want)
    finally:
        d.free()


@pytest.mark.parametrize("W,H", [(2048, 16), (61, 21), (1003, 9)])
def test_output_offsets_and_guards(codec, W, H):
    """output base offsets 0-15 with guard bytes on both sides: aligned and unaligned row pieces"""
    fr, stream, offs = encoded(W, H)
    d = DevStream(codec, stream, offs, len(fr), W, H)
    try:
        for b in (2, 4, 8):
            want = block_mean(fr, b)
            for shift in range(16):
                got, status, _ = d.binned(b, shift=shift, fill=0x5C if shift % 2 else 0xA7)
                assert (status == 0).all()
                check(got, want, "%dx%d binned by %d at offset %d" % (W, H, b, shift))
    finally:
        d.free()


def test_damaged_records_are_rejected_like_the_full_decode(codec):
    """the damage of the full decoder's invalid-stream test: the same status bits and indices as decode_device, the output
    of a rejected frame keeps its fill, good frames of the batch still decode"""
    W, H, N = 45, 37, 7
    wh = 6 * 5
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    bad = stream.copy()
    bad[int(offs[1]) + 20] += 1                 # nb != wh
    bad[int(offs[2]) + 24 + wh] += 1            # nm != wh
    bad[int(offs[3]) + 28 + 2 * wh] += 1        # n64 != sum(depth)
    bad[int(offs[4])] = 9                       # frame tag != 2
    bad[int(offs[5]) + 24 + 17] = 9             # a depth byte > 8
    for s, o in [(bad, offs[:N]), (stream[:int(offs[N]) - 8], offs[:N])]:                 # + a truncated last record
        dfull = DevStream(codec, s, o, N, W, H)
        try:
            _, want_status, want_idx = dfull.binned(1, fill=0xCD)
            assert want_status.any()
            for b in (2, 4, 8):
                want_ok = block_mean(fr, b)
                got, status, index = codec.decode_binned_host(s, o, W, H, b, fill=0xCD)
                dgot, dstatus, dindex = dfull.binned(b, shift=5, fill=0xCD)
                for st, ix in ((status, index), (dstatus, dindex)):
                    assert st.tolist() == want_status.tolist() and ix.tolist() == want_idx.tolist(), b
                for i in range(N):
                    if status[i]:
                        assert (got[i] == 0xCD).all() and (dgot[i] == 0xCD).all(), (b, i)
                    else:
                        assert (got[i] == want_ok[i]).all() and (dgot[i] == want_ok[i]).all(), (b, i)
        finally:
            dfull.free()
    assert codec.decode_binned_host(bad, offs[:N], W, H, 4)[1][5] & pkg.ST_DEPTH_TOO_BIG


@pytest.mark.parametrize("W,H", [(1001, 43), (2049, 9), (61, 20), (10, 10)])
def test_invert_endian_variant(codec, W, H):
    """DBDE_INVERT_ENDIAN records (dbde_util.cpp:15-19,246-270) with the context switch: bins are taken after the row
    reversal, edge bins of W % 8 != 0 frames included"""
    V = oracle.best_variants()
    rng = np.random.default_rng(W + 31 * H)
    fr = np.stack([rand_frame(rng, W, H, ["classes", "noise", "classes"][i % 3]) for i in range(3)])
    fr, stream, offs = encoded(W, H, frames=fr, first=9, ora=V)
    c = pkg.Codec(0)
    d = DevStream(c, stream, offs, 3, W, H)
    try:
        c.set_invert_endian(True)
        for b in FACTORS:
            want = block_mean(fr, b)
            got, status, _ = c.decode_binned_host(stream, offs[:3], W, H, b)
            assert (status == 0).all()
            check(got, want, "invert-endian host %dx%d by %d" % (W, H, b))
            dgot, dstatus, _ = d.binned(b, shift=9)
            assert (dstatus == 0).all()
            check(dgot, want, "invert-endian device %dx%d by %d" % (W, H, b))
        plain, _, _ = codec.decode_binned_host(stream, offs[:3], W, H, 2)
        assert not np.array_equal(plain, block_mean(fr, 2))
    finally:
        d.free()
        c.close()


def test_host_form_pinned_pageable_and_chunked(codec):
    """decode_binned_host on pageable numpy and pinned buffers, in chunks of 3 frames; a rejected frame in the middle of
    a chunk"""
    W, H, N = 1001, 203, 10
    fr = synth.gen_frames("mix", N, W, H, f0=4)
    stream, offs = codec.encode_host(fr, 3)
    c = pkg.Codec(0)
    try:
        c.set_chunk_frames(3)
        for b in FACTORS:
            got, status, index = c.decode_binned_host(stream, offs[:N], W, H, b)
            assert (status == 0).all() and index.tolist() == list(range(3, 3 + N))
            check(got, block_mean(fr, b), "pageable chunked by %d" % b)
        # pinned everything, output at an odd address
        for b in (2, 8):
            Hb, Wb = -(-H // b), -(-W // b)
            n = N * Hb * Wb
            ps, po, pf, pst, pix = c.pinned(len(stream)), c.pinned(8 * N), c.pinned(n + 2), c.pinned(4 * N), c.pinned(8 * N)
            try:
                ps.array[:] = stream
                po.array[:] = offs[:N].view(np.uint8)
                pf.array[:] = 0xEE
                assert c.lib.dbde_b200_decode_binned_host(c.h, ps.ptr, len(stream), po.ptr, W, H, N, b, pf.ptr + 1, pst.ptr,
                                                          pix.ptr) == 0
                assert (pst.array.view(np.uint32) == 0).all() and pf.array[0] == 0xEE and pf.array[-1] == 0xEE
                assert pix.array.view(np.uint64).tolist() == list(range(3, 3 + N))
                check(pf.array[1:1 + n].reshape(N, Hb, Wb), block_mean(fr, b), "pinned by %d" % b)
            finally:
                for p in (ps, po, pf, pst, pix):
                    p.free()
        # frame 4 (the middle of the second chunk) rejected: its output keeps the fill, its neighbours decode
        bad = stream.copy()
        bad[int(offs[4])] = 9
        want = block_mean(fr, 4)
        got, status, _ = c.decode_binned_host(bad, offs[:N], W, H, 4, fill=0xCD)
        assert status[4] & pkg.ST_BAD_FRAME_HEADER and (np.delete(status, 4) == 0).all()
        assert (got[4] == 0xCD).all() and np.array_equal(np.delete(got, 4, axis=0), np.delete(want, 4, axis=0))
    finally:
        c.close()


def test_scale_1000_frames_micro_2048(codec):
    """1000 frames of 2048^2 'micro' in HBM, binned by every factor in one call each: equal to the block mean of the
    full GPU decode, compared in full"""
    N, W, H = 1000, 2048, 2048
    px = W * H
    wh = (W // 8) * (H // 8)
    cap = codec.stream_bound(W, H, N)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    d_fr, d_out = codec.device_alloc(N * px), codec.device_alloc(cap + 64)
    d_off, d_sz, d_st = codec.device_alloc(8 * N), codec.device_alloc(8 * N), codec.device_alloc(4 * N)
    d_bin = {b: codec.device_alloc(N * px // (b * b)) for b in (2, 4, 8)}
    d_bst = {b: codec.device_alloc(4 * N) for b in (2, 4, 8)}
    try:
        synth.gen_frames_device("micro", N, W, H, d_fr, seed=42, f0=0)
        codec.encode_device(d_fr, W, H, 0, N, d_out + delta, cap, d_off, d_sz)
        for b in (2, 4, 8):
            codec.decode_binned_device(d_out + delta, cap, d_off, W, H, N, b, d_bin[b], d_bst[b])
        codec.decode_device(d_out + delta, cap, d_off, W, H, N, d_fr, d_st)      # the full decode over the source frames
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
        for b in (2, 4, 8):
            assert (codec.d2h(d_bst[b], 4 * N, np.uint32) == 0).all(), b
        step = 25
        for a in range(0, N, step):
            full = codec.d2h(d_fr + a * px, step * px).reshape(step, H, W)
            for b in (2, 4, 8):
                nb = px // (b * b)
                got = codec.d2h(d_bin[b] + a * nb, step * nb).reshape(step, H // b, W // b)
                check(got, block_mean(full, b), "frames %d.. binned by %d" % (a, b))
    finally:
        for p in [d_fr, d_out, d_off, d_sz, d_st] + list(d_bin.values()) + list(d_bst.values()):
            codec.device_free(p)


def test_bad_arguments(codec):
    """each bad argument returns DBDE_B200_E_INVALID with nothing queued (the launch count does not move); an empty
    batch returns 0; factor 1 is the full decode"""
    lib, h = codec.lib, codec.h
    W, H, N = 40, 24, 2
    fr = synth.gen_frames("mix", N, W, H)
    stream, offs = codec.encode_host(fr, 0)
    d = DevStream(codec, stream, offs, N, W, H)
    d_out = codec.device_alloc(1 << 16)
    st = np.zeros(N, np.uint32)
    out = np.zeros(1 << 16, np.uint8)

    def dev(*over, n=N, factor=2):
        args = [h, d.d_s, d.nbytes, d.d_o, W, H, n, factor, d_out, d.d_st, None, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode_binned_device(*args)

    def host(*over, n=N, factor=2):
        args = [h, stream.ctypes.data, stream.nbytes, offs.ctypes.data, W, H, n, factor, out.ctypes.data, st.ctypes.data, None]
        for i, v in over:
            args[i] = v
        return lib.dbde_b200_decode_binned_host(*args)

    try:
        l0 = codec.launches()
        for f in (0, 3, 16, -1, 5, 6, 7, 9, 2**31 - 1, -2**31):
            assert dev(factor=f) == E_INVALID, f
            assert host(factor=f) == E_INVALID, f
            assert dev(n=0, factor=f) == E_INVALID, f
        for i in (0, 1, 3, 8, 9):                                    # ctx, stream, offsets, output, status
            assert dev((i, None)) == E_INVALID, i
            assert host((i, None)) == E_INVALID, i
        assert dev((4, 0)) == E_INVALID and dev((5, -1)) == E_INVALID and dev(n=-1) == E_INVALID
        assert host((4, 0)) == E_INVALID and host(n=-1) == E_INVALID
        assert codec.launches() == l0
        assert dev(n=0) == 0 and host(n=0) == 0
        assert dev((1, None), (3, None), (8, None), (9, None), n=0) == 0      # nothing to do, nothing read
        assert codec.launches() == l0
        # the context is still usable, and the last good call decodes
        assert dev() == 0 and codec.launches() == l0 + 2
        got = codec.d2h(d_out, N * 12 * 20).reshape(N, 12, 20)
        assert (codec.d2h(d.d_st, 4 * N, np.uint32) == 0).all() and np.array_equal(got, block_mean(fr, 2))
        # factor 1 is decode_device: two launches, the full frames
        assert dev(factor=1) == 0 and codec.launches() == l0 + 4
        assert np.array_equal(codec.d2h(d_out, N * W * H).reshape(N, H, W), fr)
        with pytest.raises(pkg.DbdeError):
            codec.decode_binned_host(stream, offs[:N], W, H, 3)
    finally:
        codec.device_free(d_out)
        d.free()
