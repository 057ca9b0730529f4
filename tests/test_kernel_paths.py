"""Every encoder and decoder instantiation, and every branch of the per-warp depth votes inside them, against the oracle.

The codec picks one of about forty kernels per call from the frame geometry, the alignment of the caller's frame base and
two per-call switches (DBDE_B200_NO_LINEAR, DBDE_B200_ODD_DECODE), and inside each kernel every warp votes on the depths
its 32 tiles hold to pick a packer or unpacker.  This file restates that dispatch in Python, keeps a table of cases
tagged with the instantiation each one reaches, builds frames from chosen depth sets so that every vote branch runs on
every path, and checks on the CPU that the table and the content really do reach all of them.  The GPU tests then
compare the encoders, the decoders and the region, crop and binned forms with the oracle on every table entry, plain
and DBDE_INVERT_ENDIAN, and check that the device forms reject frame offsets at or past the end of the stream."""
import functools
import importlib
import itertools
from collections import namedtuple

import numpy as np
import pytest

import oracle
from test_binned import block_mean
from test_crops import pad_crop

pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()
FIRST = 21

# ------------------------------------------------------------------ dispatch mirror
TILES_PER_PART = 256        # kTilesPerPart (dbde_device.cuh:18)
MAX_BANDS_PER_PART = 8      # kMaxBandsPerPart (dbde_device.cuh:20)

Geom = namedtuple("Geom", "W H w h nseg G ppf pitch linear")


def linear_geom(W, H):
    """dbde_device.cuh:42-53: partition q is tiles [256 q, 256 q + 256) of the row-major tile order"""
    w, h = -(-W // 8), -(-H // 8)
    return Geom(W, H, w, h, 1, 1, -(-(w * h) // TILES_PER_PART), 8 * TILES_PER_PART, True)


def make_geom(W, H, fast, no_linear=False):
    """dbde_capi.cu:142-179 (no_linear: DBDE_B200_NO_LINEAR is set)"""
    w, h = -(-W // 8), -(-H // 8)
    if w > TILES_PER_PART:                                               # :148-152 band segments
        nseg, G, ntx_max = -(-w // TILES_PER_PART), 1, TILES_PER_PART
        ppf = h * nseg
    else:                                                                # :153-159 G bands per partition
        nseg, G, ntx_max = 1, min(TILES_PER_PART // w, MAX_BANDS_PER_PART, h), w
    if fast:                                                             # :162 pitch_of
        pitch = 8 * ntx_max
    else:
        pitch = (8 * ntx_max + 15) // 16 * 16 + 48 + ((W & 15) if w > TILES_PER_PART else 0)
    while G > 1 and 8 * G * pitch > 20480:                               # :164
        G -= 1
    if nseg == 1:                                                        # :165
        ppf = -(-h // G)
    if fast and w >= 32 and w % TILES_PER_PART != 0:                     # :171-174
        used = w / (nseg * TILES_PER_PART) if nseg > 1 else G * w / TILES_PER_PART
        if used < 0.9 and not no_linear:
            return linear_geom(W, H)
    return Geom(W, H, w, h, nseg, G, ppf, pitch, False)


def part_span(g, q):
    """part_info (dbde_device.cuh:66-94) -> (first tile's row-major index, tiles) of partition q of a frame"""
    if g.linear:
        t0 = q * TILES_PER_PART
        return t0, min(TILES_PER_PART, g.w * g.h - t0)
    if g.nseg > 1:
        y0, seg = divmod(q, g.nseg)
        tx0 = seg * TILES_PER_PART
        return y0 * g.w + tx0, min(TILES_PER_PART, g.w - tx0)
    y0 = q * g.G
    return y0 * g.w, min(g.G, g.h - y0) * g.w


def is_fast(W, H, misalign):
    """dbde_capi.cu:405 and :465: the caller's frame base decides as well as the geometry (host forms stage frames at
    aligned device addresses: misalign 0)"""
    return W % 16 == 0 and H % 8 == 0 and misalign % 16 == 0


def encoder_of(g, fast):
    """launch_encode (dbde_encode.cu:651-669) -> the instantiation's tag"""
    if fast and g.w % TILES_PER_PART == 0 and g.pitch == 8 * TILES_PER_PART:
        return "wide"                                  # dbde_encode_kernel<true, true, false>
    if fast and g.linear:
        return "linear"                                # <true, false, false, 0, true>
    if fast:
        return "band-seg" if g.nseg > 1 else "band"    # <true, false, false>
    return "contig%d%s" % (g.W & 7, "-seg" if g.nseg > 1 else "")   # <false, false, true, W & 7>


def decoder_of(g, fast, odd_direct):
    """launch_decode (dbde_decode.cu:991-1018) -> the instantiation's tag (odd_direct: DBDE_B200_ODD_DECODE=direct)"""
    if fast and g.linear:
        return "<-2>"
    if fast:
        return "<-1>-seg" if g.nseg > 1 else "<-1>"
    if g.nseg == 1 and not odd_direct:
        return "staged%d" % (g.W & 7)                  # dbde_decode_staged_kernel<W & 7>
    return "direct%d%s" % (g.W & 7, "-seg" if g.nseg > 1 else "")   # dbde_decode_kernel<W & 7>


ENCODERS = {"wide", "band", "band-seg", "linear"} | {"contig%d%s" % (m, s) for m in range(8) for s in ("", "-seg")}
DECODERS = ({"<-1>", "<-1>-seg", "<-2>"} | {"staged%d" % m for m in range(8)} |
            {"direct%d%s" % (m, s) for m in range(8) for s in ("", "-seg")})


# ------------------------------------------------------------------ the path table
# env: "" (defaults), "no-linear" (DBDE_B200_NO_LINEAR=1) or "direct" (DBDE_B200_ODD_DECODE=direct).  dev: None for the
# host forms only, else the device forms run too with the frame buffers dev bytes past a 16-byte boundary.  enc / dec:
# the instantiations the entry is there to reach (the device forms' when dev is set).
Path = namedtuple("Path", "W H env dev enc dec")
PATHS = [
    Path(2048, 16, "", 0, "wide", "<-1>"),
    Path(4096, 8, "", None, "wide", "<-1>-seg"),
    Path(512, 64, "", None, "band", "<-1>"),                 # four bands per partition
    Path(1920, 1080, "", None, "band", "<-1>"),              # one band per partition, 16 lanes idle
    # band segments with a short last segment: 3840 = 256 + 224 tiles, 3712 = 256 + 208, 4080 = 256 + 254
    Path(3840, 2160, "", None, "band-seg", "<-1>-seg"),
    Path(3712, 16, "", None, "band-seg", "<-1>-seg"),
    Path(4080, 8, "", None, "band-seg", "<-1>-seg"),
    # widths that take linear partitions, and the band layouts they would have without them
    Path(1280, 64, "", None, "linear", "<-2>"),
    Path(1280, 64, "no-linear", None, "band", "<-1>"),
    Path(2304, 48, "", None, "linear", "<-2>"),
    Path(2304, 48, "no-linear", None, "band-seg", "<-1>-seg"),
    Path(4112, 16, "", None, "linear", "<-2>"),
    Path(4112, 16, "no-linear", None, "band-seg", "<-1>-seg"),
    # aligned geometries through the device forms with frame bases off a 16-byte boundary
    Path(512, 64, "", 1, "contig0", "staged0"),
    Path(512, 64, "direct", 9, "contig0", "direct0"),
    Path(4096, 16, "", 3, "contig0-seg", "direct0-seg"),
    # W % 16 == 8
    Path(264, 24, "", None, "contig0", "staged0"),
    Path(264, 24, "direct", None, "contig0", "direct0"),
]
# the odd-size classes W & 7 = 0..7 of tests/test_gpu_parity.py with full-width partitions, both odd decoders ...
for _W, _H in [(1016, 30), (2041, 33), (1002, 19), (1003, 8), (1004, 21), (5, 1000), (1006, 17), (2047, 17)]:
    PATHS += [Path(_W, _H, "", None, "contig%d" % (_W & 7), "staged%d" % (_W & 7)),
              Path(_W, _H, "direct", None, "contig%d" % (_W & 7), "direct%d" % (_W & 7))]
# ... and with band segments (W > 2048)
for _W, _H in [(4104, 16), (2049, 9), (2050, 8), (2051, 16), (4100, 12), (2053, 8), (2054, 24), (2055, 9)]:
    PATHS.append(Path(_W, _H, "", None, "contig%d-seg" % (_W & 7), "direct%d-seg" % (_W & 7)))


def path_id(p):
    return "%dx%d%s%s" % (p.W, p.H, "-" + p.env if p.env else "", "" if p.dev is None else "-dev%d" % p.dev)


def path_geom(p):
    fast = is_fast(p.W, p.H, p.dev or 0)
    return make_geom(p.W, p.H, fast, p.env == "no-linear"), fast


def path_kernels(p):
    g, fast = path_geom(p)
    return encoder_of(g, fast), decoder_of(g, fast, p.env == "direct")


# ------------------------------------------------------------------ depth-set content
def depth_set_frame(rng, W, H, S):
    """A frame whose tile (tx, ty) has depth S[(tx + ty + rot) % |S|] (rot random), so every run of |S| tiles of a row
    holds every member of S.  A tile's minimum is 0 or 255 - (2^k - 1) at random, and it holds both its minimum and
    minimum + 2^k - 1 (at (0, 0) and at (0, 1) and (1, 0), so that partial tiles of two or more pixels keep depth k)."""
    S = sorted(S)
    h, w = -(-H // 8), -(-W // 8)
    ty, tx = np.mgrid[0:h, 0:w]
    k = np.array(S)[(tx + ty + int(rng.integers(0, len(S)))) % len(S)]
    rg = (1 << k) - 1
    mn = np.where(rng.random((h, w)) < 0.5, 0, 255 - rg)
    px = mn[:, :, None, None] + (rng.integers(0, 256, (h, w, 8, 8)) & rg[:, :, None, None])
    px[:, :, 0, 0] = mn
    px[:, :, 0, 1] = px[:, :, 1, 0] = mn + rg
    return px.transpose(0, 2, 1, 3).reshape(8 * h, 8 * w)[:H, :W].astype(np.uint8)


# every subset of 1..8 of size 1 and 2, and sets of 3 and 4 on the decoder's (3 depths) and the encoder's (4 depths)
# threshold of the depth-agnostic path
_BASE_SETS = ([(a,) for a in range(1, 9)] + list(itertools.combinations(range(1, 9), 2)) +
              [(1, 2, 3), (2, 5, 8), (1, 2, 3, 4), (3, 5, 7, 8)])
# frames of more than a megapixel: a dozen sets that reach every class
_LARGE_SETS = [(1, 8), (2, 7), (3, 6), (4, 5), (1, 2), (8,), (1, 2, 3), (1, 2, 3, 4)]


def depth_sets(W, H):
    """each base set, then the same set with depth 0 mixed in (which leaves both votes as they are and lands at the
    other payload alignment, see lay_out), then {0}"""
    base = _LARGE_SETS if W * H > 1_000_000 else _BASE_SETS
    return [s for b in base for s in (b, (0,) + b)] + [(0,)]


@functools.lru_cache(maxsize=4)
def content(W, H):
    rng = np.random.default_rng(W * 7919 + H)
    return np.stack([depth_set_frame(rng, W, H, S) for S in depth_sets(W, H)])


def lay_out(stream, sizes, W, H):
    """The records of `stream` with 0-7 junk bytes in front of each: record i's payload (at offset + 32 + 2 wh) is
    8-byte aligned for even i and at residue 1 + (i // 2) % 7 mod 8 for odd i, so every depth set is decoded from an
    aligned and from an unaligned payload -> (records, offsets)"""
    wh = -(-W // 8) * -(-H // 8)
    rng = np.random.default_rng(len(stream))
    parts, offs, pos, start = [], [], 0, 0
    for i, n in enumerate(int(s) for s in sizes):
        junk = ((0 if i % 2 == 0 else 1 + (i // 2) % 7) - (pos + 32 + 2 * wh)) % 8
        parts += [rng.integers(0, 256, junk, dtype=np.uint8), stream[start:start + n]]
        offs.append(pos + junk)
        pos += junk + n
        start += n
    return np.concatenate(parts), np.array(offs, dtype=np.uint64)


# ------------------------------------------------------------------ vote classes
ENC_CLASSES = {"low", "var", "depth8-even", "depth8-odd"} | {"spec%d" % k for k in range(1, 8)}
DEC_CLASSES = {(c, al) for c in ["var", "depth8-only"] + ["spec%d" % k for k in range(1, 9)] for al in ("al8", "unaligned")}


def warp_tiles(g):
    """the tiles of every warp: 32 consecutive tiles of each partition (lane = tile index in the partition in both
    the encoder and the decoders), -1 for lanes past the partition's end"""
    rows = []
    for q in range(g.ppf):
        t0, nt = part_span(g, q)
        idx = np.full(-(-nt // 32) * 32, -1, dtype=np.int64)
        idx[:nt] = t0 + np.arange(nt)
        rows.append(idx.reshape(-1, 32))
    return np.concatenate(rows)


def vote_classes(depth, tiles, al8):
    """the branches the warps of one frame take -> (encoder classes, decoder classes)"""
    k = np.where(tiles >= 0, depth[np.maximum(tiles, 0)], 0).astype(np.int64)
    kinds = np.bitwise_or.reduce((1 << k) >> 1, axis=1)
    ndist = np.array([bin(int(x)).count("1") for x in kinds])
    enc, dec = set(), set()
    # encoder, dbde_encode.cu:535-557: all depths <= 2 -> pack_low_depths; >= 4 distinct -> pack_rows_var; else
    # concat_fields<K>, and enc_store_depth8 with its own branch for a tile at an odd word offset in the warp
    low, var = (kinds & ~3) == 0, ndist >= 4
    spec = ~low & ~var
    if (low & (kinds != 0)).any():
        enc.add("low")
    if var.any():
        enc.add("var")
    ks = k[spec]
    before = np.cumsum(ks, axis=1) - ks
    enc |= {"spec%d" % K for K in range(1, 8) if (ks == K).any()}
    if ((ks == 8) & (before % 2 == 0)).any():
        enc.add("depth8-even")
    if ((ks == 8) & (before % 2 == 1)).any():
        enc.add("depth8-odd")
    # decoder, unpack_tile (dbde_device.cuh:486-508): >= 3 distinct or depth 8 alone -> unpack_rows_var64 (aligned) or
    # unpack_rows_var; else load_split<K, 8> (aligned) or load_split<K, 1>
    al = "al8" if al8 else "unaligned"
    var = (ndist >= 3) | (kinds == 0x80)
    if (ndist >= 3).any():
        dec.add(("var", al))
    if (kinds == 0x80).any():
        dec.add(("depth8-only", al))
    dec |= {("spec%d" % K, al) for K in range(1, 9) if (k[~var] == K).any()}
    return enc, dec


@functools.lru_cache(maxsize=None)
def reached(W, H, env, dev):
    """the vote classes the table entry's content reaches on its encoder and its decoder, from the oracle's depth
    planes and the payload alignments of lay_out"""
    p = Path(W, H, env, dev, None, None)
    g, _ = path_geom(p)
    tiles = warp_tiles(g)
    fr = content(W, H)
    stream, sizes = oracle.port.pack_frames(fr, FIRST)
    _, offs = lay_out(stream, sizes, W, H)
    wh = g.w * g.h
    enc, dec = set(), set()
    start = 0
    for i, n in enumerate(int(s) for s in sizes):
        depth = stream[start + 24:start + 24 + wh]
        e, d = vote_classes(depth, tiles, (int(offs[i]) + 32 + 2 * wh) % 8 == 0)
        enc |= e
        dec |= d
        start += n
    return enc, dec


# ------------------------------------------------------------------ CPU checks
def test_the_table_reaches_every_instantiation():
    """each entry's tags are what the mirrored dispatch picks, and the entries together reach every encoder and decoder
    instantiation"""
    for p in PATHS:
        assert path_kernels(p) == (p.enc, p.dec), path_id(p)
    assert {p.enc for p in PATHS} == ENCODERS, sorted(ENCODERS - {p.enc for p in PATHS})
    assert {p.dec for p in PATHS} == DECODERS, sorted(DECODERS - {p.dec for p in PATHS})
    for W, H in [(3840, 2160), (3712, 16), (4080, 8)]:
        g = make_geom(W, H, True)
        assert g.nseg > 1 and part_span(g, g.nseg - 1)[1] < TILES_PER_PART


def test_the_mirror_against_known_geometries():
    """spot checks of the mirror against the layouts the C++ comments state (dbde_capi.cu:166-170)"""
    assert make_geom(2304, 48, True).linear and make_geom(1280, 64, True).linear
    g = make_geom(2304, 48, True, no_linear=True)
    assert (g.nseg, g.ppf, part_span(g, 1)) == (2, 12, (256, 32))
    g = make_geom(1920, 1080, True)
    assert (g.linear, g.nseg, g.G, g.ppf) == (False, 1, 1, 135)
    g = make_geom(512, 64, True)
    assert (g.G, g.ppf, part_span(g, 1)) == (4, 2, (256, 256))
    g = make_geom(1003, 8, False)
    assert (g.G, g.ppf, part_span(g, 0)) == (1, 1, (0, 126))


@pytest.mark.parametrize("W,H", [(3840, 64), (264, 24), (2049, 9), (5, 1000)])
def test_depth_set_frames_have_the_intended_depth_plane(W, H):
    """the generator's depth plane is the oracle's, except for tiles of a single pixel (depth 0)"""
    h, w = -(-H // 8), -(-W // 8)
    for S in [(3, 8), (1, 8), (1, 2), (1, 2, 3), (1, 2, 3, 4), (0, 5), (8,)]:
        img = depth_set_frame(np.random.default_rng(7), W, H, S)
        rot = int(np.random.default_rng(7).integers(0, len(S)))     # the generator's first draw
        ty, tx = np.mgrid[0:h, 0:w]
        want = np.array(sorted(S))[(tx + ty + rot) % len(S)]
        one = (np.minimum(8, W - 8 * tx) == 1) & (np.minimum(8, H - 8 * ty) == 1)
        want[one] = 0
        rec = oracle.port.pack_frame(0, img)
        assert (rec[24:24 + w * h].reshape(h, w) == want).all(), S
        t = img[:8 * (H // 8), :8 * (W // 8)].reshape(H // 8, 8, W // 8, 8)
        mins = t.min(axis=(1, 3))
        assert set(np.unique(mins).tolist()) <= {0} | {255 - (1 << k) + 1 for k in S}


@pytest.mark.parametrize("p", PATHS, ids=path_id)
def test_every_vote_branch_runs_on_every_path(p):
    """the entry's depth-set records reach every branch class of the encoder's vote and, at both payload alignments,
    of the decoder's vote"""
    enc, dec = reached(p.W, p.H, p.env, p.dev)
    assert enc == ENC_CLASSES, sorted(ENC_CLASSES - enc)
    assert dec == DEC_CLASSES, sorted(DEC_CLASSES - dec)


# ------------------------------------------------------------------ GPU parity over the table
@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


@pytest.fixture(scope="module")
def variants():
    return oracle.best_variants()


@pytest.fixture
def path_env(monkeypatch):
    def apply(p):
        monkeypatch.delenv("DBDE_B200_NO_LINEAR", raising=False)
        monkeypatch.delenv("DBDE_B200_ODD_DECODE", raising=False)
        if p.env == "no-linear":
            monkeypatch.setenv("DBDE_B200_NO_LINEAR", "1")
        elif p.env == "direct":
            monkeypatch.setenv("DBDE_B200_ODD_DECODE", "direct")
    return apply


def first_diff(got, want, what):
    if not np.array_equal(got, want):
        assert got.shape == want.shape, (what, got.shape, want.shape)
        bad = tuple(int(x) for x in np.argwhere(got != want)[0])
        pytest.fail("%s differs first at %r: %d != %d" % (what, bad, got[bad], want[bad]))


def region(W, H):
    """not tile-aligned; on frames of more than one partition it crosses partition boundaries"""
    x0, y0 = min(3, W - 1), min(5, H - 1)
    return x0, y0, max(1, W - x0 - 2), max(1, H - y0 - 3)


def crop_set(W, H):
    cw, ch = min(W, 37), min(H, 19)
    return np.array([[W // 3, H // 4], [W - cw // 2, H - ch // 2], [-5, 3]], dtype=np.int32), (cw, ch)


def check_device_forms(codec, p, fr, want, sizes, stream, offs):
    """encode_device from frames at a base dev bytes off 16, decode_device of the laid-out records into frames at the
    same offset"""
    N, H, W = fr.shape
    m = p.dev
    stride = codec.slot_stride(W, H)
    d_fr, d_out = codec.device_alloc(fr.nbytes + 16), codec.device_alloc(stride * N)
    d_s, d_o, d_sz = codec.device_alloc(len(stream)), codec.device_alloc(8 * N), codec.device_alloc(8 * N)
    d_st, d_ix = codec.device_alloc(4 * N), codec.device_alloc(8 * N)
    try:
        codec.h2d(d_fr + m, fr)
        codec.encode_device(d_fr + m, W, H, FIRST, N, d_out, stride * N, d_o, d_sz)
        assert codec.d2h(d_sz, 8 * N, np.uint64).tolist() == sizes.tolist()
        buf = codec.d2h(d_out, stride * N)
        starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        for i in range(N):
            first_diff(buf[i * stride:i * stride + int(sizes[i])], want[starts[i]:starts[i + 1]], "encode_device record %d" % i)
        codec.h2d(d_s, stream)
        codec.h2d(d_o, offs)
        codec.h2d(d_fr, np.full(fr.nbytes + 16, 0xA7, dtype=np.uint8))
        codec.decode_device(d_s, len(stream), d_o, W, H, N, d_fr + m, d_st, d_ix)
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
        assert codec.d2h(d_ix, 8 * N, np.uint64).tolist() == list(range(FIRST, FIRST + N))
        out = codec.d2h(d_fr, fr.nbytes + 16)
        assert (out[:m] == 0xA7).all() and (out[m + fr.nbytes:] == 0xA7).all()
        first_diff(out[m:m + fr.nbytes].reshape(fr.shape), fr, "decode_device")
    finally:
        for d in (d_fr, d_out, d_s, d_o, d_sz, d_st, d_ix):
            codec.device_free(d)


@pytest.mark.gpu
@pytest.mark.parametrize("invert", [False, True], ids=["plain", "invert"])
@pytest.mark.parametrize("p", PATHS, ids=path_id)
def test_path_matches_the_oracle(codec, variants, path_env, p, invert):
    """records byte-equal to the oracle's; the oracle's records, laid out at every payload alignment, decode to the
    source frames in full, in a region, in crops and binned, and validate with status 0"""
    path_env(p)
    W, H = p.W, p.H
    fr = content(W, H)
    N = len(fr)
    want, sizes = (variants if invert else ORA).pack_frames(fr, FIRST)
    stream, offs = lay_out(want, sizes, W, H)
    ok = list(range(FIRST, FIRST + N))
    codec.set_invert_endian(invert)
    codec.set_chunk_frames(N)          # one chunk: payload alignments on the device are those lay_out chose
    try:
        got, goffs = codec.encode_host(fr, FIRST)
        assert np.diff(goffs).tolist() == sizes.tolist()
        first_diff(got, want, "encode_host")
        dec, status, index = codec.decode_host(stream, offs, W, H)
        assert (status == 0).all() and index.tolist() == ok
        first_diff(dec, fr, "decode_host")
        status, index = codec.validate_host(stream, offs, W, H)
        assert (status == 0).all() and index.tolist() == ok
        r = region(W, H)
        got, status, index = codec.decode_roi_host(stream, offs, W, H, r)
        assert (status == 0).all() and index.tolist() == ok
        first_diff(got, fr[:, r[1]:r[1] + r[3], r[0]:r[0] + r[2]], "region %r" % (r,))
        corners, size = crop_set(W, H)
        got, status, index = codec.decode_crops_host(stream, offs, W, H, corners, size, pad=0x5A)
        assert (status == 0).all() and index.tolist() == ok
        first_diff(got, pad_crop(fr, corners, size[0], size[1], 0x5A), "crops")
        for b in (2, 4, 8):
            got, status, index = codec.decode_binned_host(stream, offs, W, H, b)
            assert (status == 0).all() and index.tolist() == ok
            first_diff(got, block_mean(fr, b), "binned by %d" % b)
        if p.dev is not None:
            check_device_forms(codec, p, fr, want, sizes, stream, offs)
    finally:
        codec.set_invert_endian(False)
        codec.set_chunk_frames(0)


# ------------------------------------------------------------------ device frame offsets
def offset_batch(good, stream_bytes, fixed):
    """good records, one twice, good records in reverse order, and offsets at and past the end of the stream up to
    2^64 - 1, where off + fixed wraps -> (offsets, source record per entry or None)"""
    g0, g1, g2 = good
    past = [stream_bytes, stream_bytes - 1, stream_bytes + 12345, 1 << 63, (1 << 64) - 1, (1 << 64) - fixed + 1]
    offs = [g0, g1, g2, g2, g1, g0] + past + [g1]
    src = [0, 1, 2, 2, 1, 0] + [None] * len(past) + [1]
    return np.array(offs, dtype=np.uint64), src


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(2048, 16), (1001, 43)])
def test_device_forms_reject_offsets_past_the_stream(codec, W, H):
    """decode, region, crops and binned device forms: offsets whose fixed fields do not fit in the stream report
    ST_TRUNCATED with index 0 and leave their output untouched, whatever the offset; the good frames of the batch,
    repeated and reordered, decode to their source frames"""
    rng = np.random.default_rng(W + H)
    fr = np.stack([depth_set_frame(rng, W, H, S) for S in [(1, 8), (0, 2, 3), (1, 2, 3, 4)]])
    want, sizes = ORA.pack_frames(fr, FIRST)
    wh = -(-W // 8) * -(-H // 8)
    good = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64).tolist()
    offs, src = offset_batch(good, len(want), 32 + 2 * wh)
    N = len(offs)
    r = region(W, H)
    corners, (cw, ch) = crop_set(W, H)
    cases = {
        "decode": (fr, W * H, lambda d_s, d_o, out, st, ix: codec.decode_device(d_s, len(want), d_o, W, H, N, out, st, ix)),
        "region": (fr[:, r[1]:r[1] + r[3], r[0]:r[0] + r[2]], r[2] * r[3],
                   lambda d_s, d_o, out, st, ix: codec.decode_roi_device(d_s, len(want), d_o, W, H, N, r, out, st, ix)),
        "crops": (pad_crop(fr, corners, cw, ch, 0), len(corners) * cw * ch,
                  lambda d_s, d_o, out, st, ix: codec.decode_crops_device(d_s, len(want), d_o, W, H, N, d_c, len(corners), 0,
                                                                          (cw, ch), out, st, ix)),
        "binned": (block_mean(fr, 2), -(-W // 2) * -(-H // 2),
                   lambda d_s, d_o, out, st, ix: codec.decode_binned_device(d_s, len(want), d_o, W, H, N, 2, out, st, ix)),
    }
    d_s, d_o, d_c = codec.device_alloc(len(want)), codec.device_alloc(8 * N), codec.device_alloc(corners.nbytes)
    d_st, d_ix = codec.device_alloc(4 * N), codec.device_alloc(8 * N)
    try:
        codec.h2d(d_s, want)
        codec.h2d(d_o, offs)
        codec.h2d(d_c, corners)
        for name, (ref, per, run) in cases.items():
            d_out = codec.device_alloc(N * per)
            try:
                codec.h2d(d_out, np.full(N * per, 0xA7, dtype=np.uint8))
                codec.h2d(d_st, np.full(N, 0xFFFFFFFF, dtype=np.uint32))
                run(d_s, d_o, d_out, d_st, d_ix)
                out = codec.d2h(d_out, N * per).reshape((N,) + ref.shape[1:])
                status, index = codec.d2h(d_st, 4 * N, np.uint32), codec.d2h(d_ix, 8 * N, np.uint64)
            finally:
                codec.device_free(d_out)
            for i, s in enumerate(src):
                if s is None:
                    assert status[i] == pkg.ST_TRUNCATED and index[i] == 0, (name, int(offs[i]))
                    assert (out[i] == 0xA7).all(), (name, int(offs[i]))
                else:
                    assert status[i] == 0 and index[i] == FIRST + s, (name, i)
                    first_diff(out[i], ref[s], "%s entry %d" % (name, i))
    finally:
        for d in (d_s, d_o, d_c, d_st, d_ix):
            codec.device_free(d)


@pytest.mark.gpu
def test_dbde16_device_decode_rejects_offsets_past_the_stream(codec):
    """the same batch through the DBDE16 device decode (dbde16_scan_kernel), called through the C ABI"""
    W, H = 136, 72
    rng = np.random.default_rng(16)
    fr = (rng.integers(0, 1 << 12, (3, H, W)) + np.array([0, 40000, 7])[:, None, None]).astype(np.uint16)
    want, sizes = oracle.port16.pack_frames(fr, FIRST)
    wh = -(-W // 8) * -(-H // 8)
    good = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64).tolist()
    offs, src = offset_batch(good, len(want), 32 + 3 * wh)
    offs = np.append(offs, np.uint64((1 << 64) - (32 + 2 * wh) + 1))
    src.append(None)
    N = len(offs)
    d_s, d_o, d_out = codec.device_alloc(len(want)), codec.device_alloc(8 * N), codec.device_alloc(2 * N * W * H)
    d_st, d_ix = codec.device_alloc(4 * N), codec.device_alloc(8 * N)
    try:
        codec.h2d(d_s, want)
        codec.h2d(d_o, offs)
        codec.h2d(d_out, np.full(2 * N * W * H, 0xA7, dtype=np.uint8))
        codec._ck(codec.lib.dbde_b200_decode16_device(codec.h, d_s, len(want), d_o, W, H, N, d_out, d_st, d_ix, None),
                  "decode16_device")
        out = codec.d2h(d_out, 2 * N * W * H, np.uint16).reshape(N, H, W)
        status, index = codec.d2h(d_st, 4 * N, np.uint32), codec.d2h(d_ix, 8 * N, np.uint64)
    finally:
        for d in (d_s, d_o, d_out, d_st, d_ix):
            codec.device_free(d)
    for i, s in enumerate(src):
        if s is None:
            assert status[i] == pkg.ST_TRUNCATED and index[i] == 0 and (out[i] == 0xA7A7).all(), int(offs[i])
        else:
            assert status[i] == 0 and index[i] == FIRST + s and (out[i] == fr[s]).all(), i
