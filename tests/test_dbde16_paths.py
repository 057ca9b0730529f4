"""Every DBDE16 load, store, copy-out and staging path of the device encoder and decoder, against the oracle.

encode16_device and decode16_device (csrc/dbde16.cu) pick their memory paths from addresses the caller controls: the
frame base (16-byte tile rows, 4-byte rows, or rows that start on an odd pixel), the record base and slot stride (the
encoder copies a partition's words out as U64 stores or as bytes) and the payload address of each record (the decoder
stages words with U64 loads or bytes, and keeps a copy of every 33rd unit in a padding slot).  The host forms always
hand the kernels 16-byte aligned frames and 16-byte aligned payloads, so a caller passing slices of larger tensors takes
paths the host forms never do.  This file restates that path choice in Python, keeps a table of geometries with the
frame bases, record bases, slot strides and payload residues the GPU tests run them at, and checks on the CPU that the
table reaches every path.  The GPU tests then compare the device forms with the oracle on every run of the table: the
encoder's records byte for byte, with guard bytes before, between and after the slots; the decoder's frames, crops and
bins exactly, with guard bytes on both sides of the output."""
import functools
import importlib
import itertools
from collections import namedtuple

import numpy as np
import pytest

import oracle

pkg = importlib.import_module("dbce-video-cpp_b200")
P16 = oracle.port16
FIRST = 5
TILES_PER_PART = 256        # kT16 (dbde16.cu:21): one partition is 256 consecutive raster-order tiles
GUARD = 64                  # guard bytes on each side of every device output


def tiles(W, H):
    return -(-W // 8), -(-H // 8)


def record_bound16(W, H):
    """dbde_b200_frame_record_bound16 (dbde_capi.cu:1201)"""
    w, h = tiles(W, H)
    return 32 + 131 * w * h


def slot_stride16(W, H):
    """dbde_b200_slot_stride16, the slot stride encode16_device takes for slot_stride 0"""
    return (record_bound16(W, H) + 15) // 16 * 16


# ------------------------------------------------------------------ path mirror
def tile_row_classes(W, H, base):
    """load_tile16 / store_tile16 (dbde16.cu:32-109) on a frame at byte address `base` (mod 16) -> the branches its tile
    rows take: L1 aligned full tile, L2 aligned tile with partial rows, L3 full row by 4-byte accesses, L4 full row that
    starts on an odd pixel, L5 partial columns element by element"""
    aligned = W % 8 == 0 and base % 16 == 0             # dbde_capi.cu:1236 and :1280
    out = set()
    if W % 8:
        out.add("L5")                                   # the last tile column
    if W < 8:
        return out
    if aligned:
        out |= ({"L1"} if H >= 8 else set()) | ({"L2"} if H % 8 else set())
        return out
    # a full-column tile row y starts at base + 2 (y W + 8 tx): 4-byte aligned iff base / 2 + y W is even
    y = np.arange(H if W % 2 else 1)
    odd = (base // 2 + y * W) % 2
    return out | ({"L3"} if (odd == 0).any() else set()) | ({"L4"} if (odd == 1).any() else set())


def partition_words(depth):
    """a frame's depth plane -> the word count (agg) of each of its partitions"""
    return np.add.reduceat(depth.astype(np.int64), np.arange(0, len(depth), TILES_PER_PART))


def encode_classes(W, H, frame_base, out_base, stride, depths):
    """encode16_device on frames at frame_base + 2 W H f and records at out_base + stride f: load_tile16's branches and,
    for every partition with words, the copy-out (dbde16.cu:198-205): U64 stores when its words start 8-byte aligned
    (rec + 32 + 3 wh + 8 excl), else bytes"""
    wh = np.prod(tiles(W, H))
    cls = set()
    for f, depth in enumerate(depths):
        cls |= {"load-" + c for c in tile_row_classes(W, H, frame_base + 2 * W * H * f)}
        if partition_words(depth).any():
            cls.add("copy-u64" if (out_base + stride * f + 32 + 3 * wh) % 8 == 0 else "copy-bytes")
    return cls


def stage_class(residue, agg):
    """stage_words16 (dbde16.cu:410-432) for a partition of agg > 0 words whose payload is at `residue` mod 8: U64 loads
    or bytes; "-pad" when its 2 agg units run past unit 32, so copies go into padding slots; "-end" when 2 agg is a
    multiple of 32, so the zeroed unit past the end goes into a padding slot as well"""
    return "stage-%s%s%s" % ("u64" if residue % 8 == 0 else "bytes", "-pad" if 2 * agg > 32 else "",
                             "-end" if (2 * agg) % 32 == 0 else "")


def decode_classes(W, H, frame_base, residues, depths):
    """decode16_device into frames at frame_base + 2 W H f, frame f's payload at residues[f] mod 8: store_tile16's
    branches and stage_words16's"""
    cls = set()
    for f, depth in enumerate(depths):
        cls |= {"store-" + c for c in tile_row_classes(W, H, frame_base + 2 * W * H * f)}
        cls |= {stage_class(residues[f], int(a)) for a in partition_words(depth) if a > 0}
    return cls


ROW_CLASSES = {"L%d" % i for i in range(1, 6)}
ENC_CLASSES = {"load-" + c for c in ROW_CLASSES} | {"copy-u64", "copy-bytes"}
DEC_CLASSES = ({"store-" + c for c in ROW_CLASSES} |
               {"stage-%s%s%s" % (m, p, e) for m in ("u64", "bytes") for p in ("", "-pad") for e in ("", "-end")})


# ------------------------------------------------------------------ the table
Path = namedtuple("Path", "W H")
PATHS = [
    # one partition (wh <= 256)
    Path(8, 8),           # one tile: the partition's word count is the tile's depth
    Path(16, 8),          # two tiles
    Path(40, 13),         # W % 8 == 0 with a partial last tile row
    Path(64, 32),
    Path(136, 72),        # wh = 153
    Path(17, 23),         # W % 8 = 1, wh = 9
    Path(26, 64),         # W % 8 = 2, wh = 32
    Path(100, 7),         # W % 8 = 4, a single partial tile row
    Path(118, 32),        # W % 8 = 6, wh = 60
    Path(127, 127),       # W % 8 = 7, one full partition
    Path(3, 5),           # narrower than a tile
    # several partitions, the last one partial
    Path(3840, 2160),     # wh = 129600 = 506 * 256 + 64
    Path(2592, 1944),     # wh = 78732 = 307 * 256 + 140
    Path(1440, 1080),     # wh = 24300 = 94 * 256 + 236
    Path(1001, 1000),     # W % 8 = 1, wh = 15750
    Path(1002, 19),       # W % 8 = 2, wh = 378
    Path(1020, 40),       # W % 8 = 4, wh = 640
    Path(1006, 33),       # W % 8 = 6, wh = 630
    Path(1015, 24),       # W % 8 = 7, wh = 381
]


def path_id(p):
    return "%dx%d" % (p.W, p.H)


def is_large(p):
    return p.W * p.H > 1_000_000


FRAME_BASES = (0, 2, 4, 6, 8, 10, 14)      # frame buffers: bytes past a 16-byte boundary
STRIDE_EXTRAS = (None, 1, 3, 7)            # None: slot_stride 0 (the default); s: record_bound16 + s


def stride_of(p, s):
    return slot_stride16(p.W, p.H) if s is None else record_bound16(p.W, p.H) + s


def encode_runs(p):
    """(frame base, record base mod 8, slot stride extra) of each encode16_device call: every frame base with every
    stride and the record bases in turn; frames of more than a megapixel take eight runs that still use each base"""
    if is_large(p):
        pairs = [(FRAME_BASES[i % len(FRAME_BASES)], STRIDE_EXTRAS[i % len(STRIDE_EXTRAS)]) for i in range(8)]
    else:
        pairs = list(itertools.product(FRAME_BASES, STRIDE_EXTRAS))
    return [(fb, i % 8, s) for i, (fb, s) in enumerate(pairs)]


# decode16_device call j reads the laid-out records from a stream j bytes past a 16-byte boundary and writes frames
# 2 j bytes past one
DECODE_SHIFTS = tuple(range(8))


# ------------------------------------------------------------------ depth-set content
def depth_set_frame16(rng, W, H, S, rot):
    """A frame whose tile (tx, ty) has depth S[(tx + ty + rot) % |S|].  A tile's minimum is 0, 65535 - (2^k - 1) or
    anything between, and it holds both its minimum and minimum + 2^k - 1 (at (0, 0) and at (0, 1) and (1, 0), so that
    partial tiles of two or more pixels keep depth k)."""
    S = sorted(S)
    w, h = tiles(W, H)
    ty, tx = np.mgrid[0:h, 0:w]
    k = np.array(S)[(tx + ty + rot) % len(S)]
    rg = (1 << k) - 1
    mn = np.choose(rng.integers(0, 3, (h, w)), [np.zeros_like(rg), 65535 - rg, rng.integers(0, 65536 - rg)])
    px = mn[:, :, None, None] + (rng.integers(0, 65536, (h, w, 8, 8)) & rg[:, :, None, None])
    px[:, :, 0, 0] = mn
    px[:, :, 0, 1] = px[:, :, 1, 0] = mn + rg
    return px.transpose(0, 2, 1, 3).reshape(8 * h, 8 * w)[:H, :W].astype(np.uint16)


# one-partition frames: every depth alone (on one tile, word counts 1..16), pairs and triples that give word counts
# past 16 and not a multiple of 16, depth 0 mixed in, and {0}
_SMALL_SETS = ([(k,) for k in range(1, 17)] + [(1, 16), (7, 9), (15, 16), (3, 8, 13), (0, 16), (0, 1), (0, 5, 11),
                                                (2, 4, 6, 8, 10, 12, 14, 16), (0,)])
# frames of more than a megapixel
_LARGE_SETS = [(16,), (1, 2, 3), (0, 7, 12)]


@functools.lru_cache(maxsize=None)
def content(W, H):
    """frames (each small set twice with the same layout, so that lay_out puts it at an aligned and at an unaligned
    payload), the oracle's records and record sizes"""
    rng = np.random.default_rng(W * 7919 + H + 16)
    if W * H > 1_000_000:
        fr = [depth_set_frame16(rng, W, H, S, int(rng.integers(0, len(S)))) for S in _LARGE_SETS]
    else:
        fr = []
        for S in _SMALL_SETS:
            rot = int(rng.integers(0, len(S)))
            fr += [depth_set_frame16(rng, W, H, S, rot) for _ in range(2)]
    fr = np.stack(fr)
    want, sizes = P16.pack_frames(fr, FIRST)
    return fr, want, sizes


def depth_planes(W, H):
    _, want, sizes = content(W, H)
    wh = np.prod(tiles(W, H))
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    return [want[s + 24:s + 24 + wh] for s in starts]


def lay_out16(stream, sizes, W, H):
    """The records of `stream` with 0-7 junk bytes in front of each: record i's payload (at offset + 32 + 3 wh) is
    8-byte aligned for even i and at residue 1 + (i // 2) % 7 mod 8 for odd i -> (records, offsets)"""
    wh = np.prod(tiles(W, H))
    rng = np.random.default_rng(len(stream))
    parts, offs, pos, start = [], [], 0, 0
    for i, n in enumerate(int(s) for s in sizes):
        junk = ((0 if i % 2 == 0 else 1 + (i // 2) % 7) - (pos + 32 + 3 * wh)) % 8
        parts += [rng.integers(0, 256, junk, dtype=np.uint8), stream[start:start + n]]
        offs.append(pos + junk)
        pos += junk + n
        start += n
    return np.concatenate(parts), np.array(offs, dtype=np.uint64)


@functools.lru_cache(maxsize=None)
def laid_out(W, H):
    _, want, sizes = content(W, H)
    return lay_out16(want, sizes, W, H)


def reached(p):
    """the classes the entry's encode and decode runs reach -> (encoder classes, decoder classes)"""
    W, H = p.W, p.H
    depths = depth_planes(W, H)
    enc = set()
    for fb, ob, s in encode_runs(p):
        enc |= encode_classes(W, H, fb, ob, stride_of(p, s), depths)
    wh = np.prod(tiles(W, H))
    _, offs = laid_out(W, H)
    dec = set()
    for j in DECODE_SHIFTS:
        dec |= decode_classes(W, H, 2 * j, [j + int(o) + 32 + 3 * wh for o in offs], depths)
    return enc, dec


# ------------------------------------------------------------------ CPU checks
def test_the_mirror_on_known_cases():
    """spot checks of the restatement"""
    assert tile_row_classes(64, 32, 0) == {"L1"} and tile_row_classes(40, 13, 0) == {"L1", "L2"}
    assert tile_row_classes(64, 32, 8) == {"L3"} and tile_row_classes(64, 32, 2) == {"L4"}
    assert tile_row_classes(17, 23, 0) == {"L3", "L4", "L5"} and tile_row_classes(26, 64, 2) == {"L4", "L5"}
    assert tile_row_classes(3, 5, 0) == {"L5"} and tile_row_classes(17, 1, 2) == {"L4", "L5"}
    # the default slot stride puts every record's words at 3 wh mod 8 past a 16-byte record base: bytes at 1440 x 1080
    # (wh = 24300) and 2592 x 1944 (wh = 78732), U64 stores at 3840 x 2160 (wh = 129600)
    d = [np.full(24300, 3, np.uint8)] * 3
    assert encode_classes(1440, 1080, 0, 0, slot_stride16(1440, 1080), d) == {"load-L1", "copy-bytes"}
    d = [np.full(129600, 3, np.uint8)] * 3
    assert encode_classes(3840, 2160, 0, 0, slot_stride16(3840, 2160), d) == {"load-L1", "copy-u64"}
    assert [stage_class(0, a) for a in (1, 15, 16, 17, 32, 33)] == [
        "stage-u64", "stage-u64", "stage-u64-end", "stage-u64-pad", "stage-u64-pad-end", "stage-u64-pad"]
    assert stage_class(5, 48) == "stage-bytes-pad-end"
    assert partition_words(np.array([1] * 300 + [2] * 10)).tolist() == [256, 44 + 20]


def test_the_table_spans_the_geometry_classes():
    """W % 8 in {0, 1, 2, 4, 6, 7} with H % 8 zero and not, one-partition frames and frames whose last partition is
    partial at wh % 8 == 0 and != 0, wh odd, 4 and 0 mod 8, and three or more frames per batch"""
    whs = [np.prod(tiles(p.W, p.H)) for p in PATHS]
    assert {(p.W % 8, p.H % 8 == 0) for p in PATHS} >= set(itertools.product((0, 1, 2, 4, 6, 7), (True, False)))
    assert any(wh <= TILES_PER_PART for wh in whs)
    partial = [wh for wh in whs if wh > TILES_PER_PART and wh % TILES_PER_PART]
    assert any(wh % 8 == 0 for wh in partial) and any(wh % 8 for wh in partial)
    assert {wh % 8 for wh in whs} >= {0, 4} and any(wh % 2 for wh in whs)
    assert all(len(content(p.W, p.H)[0]) >= 3 for p in PATHS)


@pytest.mark.parametrize("W,H", [(136, 72), (17, 23), (3840, 64), (1015, 24)])
def test_depth_set_frames_have_the_intended_depth_plane(W, H):
    """the generator's depth plane is the oracle's, except for tiles of a single pixel (depth 0)"""
    w, h = tiles(W, H)
    ty, tx = np.mgrid[0:h, 0:w]
    one = (np.minimum(8, W - 8 * tx) == 1) & (np.minimum(8, H - 8 * ty) == 1)
    for S in [(16,), (1, 16), (0, 5, 11), (3, 8, 13), (2, 4, 6, 8, 10, 12, 14, 16), (0,)]:
        img = depth_set_frame16(np.random.default_rng(7), W, H, S, 1)
        want = np.array(sorted(S))[(tx + ty + 1) % len(S)]
        want[one] = 0
        rec, _ = P16.pack_frames(img[None], 0)
        assert (rec[24:24 + w * h].reshape(h, w) == want).all(), S


def test_the_table_reaches_every_path():
    """the encode runs of the table reach every load and copy-out class, the decode runs every store and staging class"""
    enc, dec = set(), set()
    for p in PATHS:
        e, d = reached(p)
        enc |= e
        dec |= d
    assert enc == ENC_CLASSES, sorted(ENC_CLASSES - enc)
    assert dec == DEC_CLASSES, sorted(DEC_CLASSES - dec)


# ------------------------------------------------------------------ GPU parity over the table
@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


def first_diff(got, want, what):
    if not np.array_equal(got, want):
        assert got.shape == want.shape, (what, got.shape, want.shape)
        bad = tuple(int(x) for x in np.argwhere(got != want)[0])
        pytest.fail("%s differs first at %r: %d != %d" % (what, bad, got[bad], want[bad]))


class Buffers:
    """device allocations freed together"""

    def __init__(self, codec):
        self.codec, self.ptrs = codec, []

    def alloc(self, nbytes):
        self.ptrs.append(self.codec.device_alloc(nbytes))
        return self.ptrs[-1]

    def free(self):
        for d in self.ptrs:
            self.codec.device_free(d)


def encode_device(codec, frames_ptr, W, H, N, out_ptr, cap, stride, d_o, d_sz):
    codec._ck(codec.lib.dbde_b200_encode16_device(codec.h, frames_ptr, W, H, FIRST, N, out_ptr, cap, stride, d_o, d_sz,
                                                  None), "encode16_device")


def decode_device(codec, stream_ptr, nbytes, d_o, W, H, N, out_ptr, d_st, d_ix):
    codec._ck(codec.lib.dbde_b200_decode16_device(codec.h, stream_ptr, nbytes, d_o, W, H, N, out_ptr, d_st, d_ix, None),
              "decode16_device")


def check_encode_runs(codec, p, runs):
    """encode16_device on every run: slot f of the records holds the oracle's record f, frame_offsets[f] = f * stride,
    frame_sizes are the record sizes, and every byte before the first slot, between a record's end and the next slot
    and after the last slot keeps its fill"""
    W, H = p.W, p.H
    fr, want, sizes = content(W, H)
    N = len(fr)
    assert codec.lib.dbde_b200_frame_record_bound16(W, H) == record_bound16(W, H)
    assert codec.lib.dbde_b200_slot_stride16(W, H) == slot_stride16(W, H)
    starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    nbuf = N * max(stride_of(p, s) for s in STRIDE_EXTRAS) + 2 * GUARD + 8
    fill = np.random.default_rng(N).integers(0, 256, nbuf, dtype=np.uint8)
    b = Buffers(codec)
    try:
        d_fr, d_out = b.alloc(fr.nbytes + 16), b.alloc(nbuf)
        d_o, d_sz = b.alloc(8 * N), b.alloc(8 * N)
        for fb in sorted({r[0] for r in runs}):
            codec.h2d(d_fr + fb, fr)
            for _, ob, s in (r for r in runs if r[0] == fb):
                stride = stride_of(p, s)
                base = GUARD + ob
                codec.h2d(d_out, fill)
                encode_device(codec, d_fr + fb, W, H, N, d_out + base, N * stride, 0 if s is None else stride, d_o, d_sz)
                run = "frames +%d, records +%d, stride %d" % (fb, ob, stride)
                assert codec.d2h(d_o, 8 * N, np.uint64).tolist() == [stride * f for f in range(N)], run
                assert codec.d2h(d_sz, 8 * N, np.uint64).tolist() == sizes.tolist(), run
                exp = fill.copy()
                for f in range(N):
                    exp[base + f * stride:base + f * stride + int(sizes[f])] = want[starts[f]:starts[f + 1]]
                got = codec.d2h(d_out, nbuf)
                if not np.array_equal(got, exp):
                    at = int(np.argmax(got != exp)) - base
                    f = max(0, min(N - 1, at // stride))
                    pytest.fail("%s: byte %d of slot %d differs (record size %d): %d != %d"
                                % (run, at - f * stride, f, int(sizes[f]), got[at + base], exp[at + base]))
    finally:
        b.free()


def check_decode_runs(codec, p, shifts):
    """decode16_device of the laid-out records from a stream j bytes past a 16-byte boundary into frames 2 j bytes past
    one: status 0, the right indices, the source frames exactly, and every guard byte keeps its fill"""
    W, H = p.W, p.H
    fr = content(W, H)[0]
    N = len(fr)
    stream, offs = laid_out(W, H)
    nbuf = fr.nbytes + 2 * GUARD + 16
    fill = np.random.default_rng(N + 1).integers(0, 256, nbuf, dtype=np.uint8)
    b = Buffers(codec)
    try:
        d_s, d_out, d_o = b.alloc(len(stream) + 8), b.alloc(nbuf), b.alloc(8 * N)
        d_st, d_ix = b.alloc(4 * N), b.alloc(8 * N)
        codec.h2d(d_o, offs)
        for j in shifts:
            codec.h2d(d_s + j, stream)
            codec.h2d(d_out, fill)
            codec.h2d(d_st, np.full(N, 0xFFFFFFFF, dtype=np.uint32))
            decode_device(codec, d_s + j, len(stream), d_o, W, H, N, d_out + GUARD + 2 * j, d_st, d_ix)
            run = "stream +%d, frames +%d" % (j, 2 * j)
            assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all(), run
            assert codec.d2h(d_ix, 8 * N, np.uint64).tolist() == list(range(FIRST, FIRST + N)), run
            got = codec.d2h(d_out, nbuf)
            lo, hi = GUARD + 2 * j, GUARD + 2 * j + fr.nbytes
            assert np.array_equal(got[:lo], fill[:lo]) and np.array_equal(got[hi:], fill[hi:]), ("wrote outside", run)
            first_diff(got[lo:hi].view(np.uint16).reshape(fr.shape), fr, run)
    finally:
        b.free()


@pytest.mark.gpu
@pytest.mark.parametrize("p", PATHS, ids=path_id)
def test_encode16_device_matches_the_oracle(codec, p):
    check_encode_runs(codec, p, encode_runs(p))


@pytest.mark.gpu
@pytest.mark.parametrize("p", PATHS, ids=path_id)
def test_decode16_device_matches_the_source_frames(codec, p):
    check_decode_runs(codec, p, DECODE_SHIFTS)


def pad_crop(frames, corners, cw, ch, pad):
    """the reference: frames (N, H, W), corners (R, 2) -> (N, R, ch, cw)"""
    N, H, W = frames.shape
    out = np.full((N, len(corners), ch, cw), pad, dtype=frames.dtype)
    for r, (x0, y0) in enumerate(corners.tolist()):
        xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
        if xa < xb and ya < yb:
            out[:, r, ya - y0:yb - y0, xa - x0:xb - x0] = frames[:, ya:yb, xa:xb]
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


@pytest.mark.gpu
@pytest.mark.parametrize("p", PATHS, ids=path_id)
def test_crops16_and_binned16_on_the_same_layout(codec, p):
    """decode16_crops_device and decode16_binned_device (factors 2, 4, 8) of the laid-out records, from streams at two
    alignments into outputs at several even offsets with guard bytes: exactly numpy's pad-crop and block mean"""
    W, H = p.W, p.H
    fr = content(W, H)[0]
    N = len(fr)
    stream, offs = laid_out(W, H)
    cw, ch = min(W, 37), min(H, 19)
    corners = np.array([[W // 3, H // 4], [W - cw // 2, H - ch // 2], [-5, 3]], dtype=np.int32)
    pad = 0xBEEF
    refs = {0: pad_crop(fr, corners, cw, ch, pad)} | {b: block_mean(fr, b) for b in (2, 4, 8)}
    nbuf = 2 * max(r.size for r in refs.values()) + 2 * GUARD + 16
    fill = np.random.default_rng(N + 2).integers(0, 256, nbuf, dtype=np.uint8)
    b = Buffers(codec)
    try:
        d_s, d_out, d_o, d_c = b.alloc(len(stream) + 8), b.alloc(nbuf), b.alloc(8 * N), b.alloc(corners.nbytes)
        d_st, d_ix = b.alloc(4 * N), b.alloc(8 * N)
        codec.h2d(d_o, offs)
        codec.h2d(d_c, corners)
        for j in (0, 5):
            codec.h2d(d_s + j, stream)
            for factor, ref in refs.items():
                shift = (2 * factor + 2 * j + 2) % 16
                codec.h2d(d_out, fill)
                codec.h2d(d_st, np.full(N, 0xFFFFFFFF, dtype=np.uint32))
                out = d_out + GUARD + shift
                if factor == 0:
                    codec.decode16_crops_device(d_s + j, len(stream), d_o, W, H, N, d_c, len(corners), False, (cw, ch), out,
                                                d_st, d_ix, pad=pad)
                    run = "crops %dx%d, stream +%d, output +%d" % (cw, ch, j, shift)
                else:
                    codec.decode16_binned_device(d_s + j, len(stream), d_o, W, H, N, factor, out, d_st, d_ix)
                    run = "binned by %d, stream +%d, output +%d" % (factor, j, shift)
                assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all(), run
                assert codec.d2h(d_ix, 8 * N, np.uint64).tolist() == list(range(FIRST, FIRST + N)), run
                got = codec.d2h(d_out, nbuf)
                lo, hi = GUARD + shift, GUARD + shift + ref.nbytes
                assert np.array_equal(got[:lo], fill[:lo]) and np.array_equal(got[hi:], fill[hi:]), ("wrote outside", run)
                first_diff(got[lo:hi].view(np.uint16).reshape(ref.shape), ref, run)
    finally:
        b.free()


@pytest.mark.gpu
@pytest.mark.parametrize("p", PATHS, ids=path_id)
def test_invert_endian_setting_leaves_encode16_and_decode16_device_alone(codec, p):
    """DBDE16 has no DBDE_INVERT_ENDIAN variant: with the context's setting on, the device encode still writes the
    oracle's records and the device decode still returns the source frames, on a run that takes the unaligned paths"""
    codec.set_invert_endian(True)
    try:
        check_encode_runs(codec, p, [(2, 3, 1), (14, 0, None)])
        check_decode_runs(codec, p, [3])
    finally:
        codec.set_invert_endian(False)
