"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI and the
reference's C++ entry points, against the oracle (the compiled reference when oracle/_ref is
there, else the pinned port) and the committed golden vectors.  Bit-exact: this is integer /
byte work, so every comparison is equality."""
import hashlib
import importlib
import os
import tempfile

import numpy as np
import pytest

import oracle
import synth
from conftest import golden_random_frames, rand_frame

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint8).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


@pytest.fixture(scope="module")
def dropin():
    return pkg.DropIn()


def roundtrip_check(codec, frames, first_index=0):
    """encode on GPU == oracle bytes; decode on GPU == oracle pixels == source."""
    N, H, W = frames.shape
    want, sizes = ORA.pack_frames(frames, first_index)
    got, offs = codec.encode_host(frames, first_index)
    assert int(offs[N]) == len(want), (W, H, N)
    assert offs[:N].tolist() == [0] + np.cumsum(sizes).tolist()[:-1]
    assert (got == want).all(), (W, H, N, int(np.argmax(got != want)))
    dec, status, index = codec.decode_host(want, offs[:N], W, H)
    assert (status == 0).all()
    assert index.tolist() == [first_index + i for i in range(N)]
    assert (dec == frames).all(), (W, H, N)


# ------------------------------------------------------------------ golden vectors
def test_readme_10x10(codec, dropin, golden):
    """BASELINE config 1."""
    img = np.array(golden["readme"]["image"], dtype=np.uint8)
    enc = dropin.pack_image(img)
    assert enc.tobytes().hex() == golden["readme"]["pack_image"]
    assert dropin.pack_frame(7, img).tobytes().hex() == golden["readme"]["pack_frame_index7"]
    n, dec = dropin.unpack_image(enc, 10, 10)
    assert n == 92 and (dec == img).all()
    roundtrip_check(codec, img[None], 7)


def test_kat_8x16_like_the_reference_test(dropin, golden):
    """dbde_util_test.cpp:134-213 step for step, through the same C++ symbols."""
    img = np.array(golden["kat_8x16"]["image"], dtype=np.uint8).reshape(8, 16)
    stream = np.array(golden["kat_8x16"]["stream"], dtype=np.uint8)
    n, vh = dropin.unpack_video_header(stream)
    assert n == 28 and vh == (3, 8, 16, 1.0)
    used, hdr, dec = dropin.unpack_frame(stream[28:], 16, 8)
    assert used == 100 and hdr == (2, 1, 0) and (dec == img).all()
    enc = np.concatenate([dropin.pack_video_header(3, 8, 16, 1.0), dropin.pack_frame(1, img)])
    assert len(enc) == 128 and (enc == stream).all()


def test_headers(dropin, golden):
    assert dropin.pack_video_header(3, 10, 10, 30.0).tobytes().hex() == golden["headers"]["video_3_10_10_30hz"]
    assert dropin.pack_frame_header(2, 5, 123456789012345).tobytes().hex() == golden["headers"]["frame_2_5_123456789012345"]


def test_small_flat_and_single_tiles(dropin, golden):
    s = golden["small_3x5"]
    img = np.array(s["image"], dtype=np.uint8)
    assert dropin.pack_image(img).tobytes().hex() == s["pack_image"]
    flat = np.full((8, 8), golden["flat_8x8"]["value"], dtype=np.uint8)
    assert dropin.pack_image(flat).tobytes().hex() == golden["flat_8x8"]["pack_image"]
    for t in golden["single_tiles"]:
        tile = np.full((8, 8), t["min"], dtype=np.uint8)
        tile[3, 5] = t["min"] + t["range"]
        tile[7, 7] = t["min"] + t["range"] // 2
        r, pay = dropin.pack_8x8(tile)
        assert r == t["ret"] and pay.tobytes().hex() == t["payload"], t
        back = dropin.unpack_8x8(r >> 8, r & 0xFF, pay, stride=11)
        assert (back == tile).all()


def test_partial_tiles(dropin):
    rng = np.random.default_rng(5)
    for rm, dm in [(1, 1), (2, 8), (8, 2), (2, 2), (7, 3), (3, 7), (8, 7), (7, 8), (5, 5)]:
        tile = rng.integers(0, 256, (8, 8), dtype=np.uint8) >> int(rng.integers(0, 6))
        r0, p0 = ORA.pack_8x8_partial(tile, rm, dm)
        r1, p1 = dropin.pack_8x8_partial(tile, rm, dm)
        assert r0 == r1 and (p0 == p1).all(), (rm, dm)
        crop = dropin.unpack_8x8_partial(r1 >> 8, r1 & 0xFF, p1, rm, dm, fill=0xCD)
        assert (crop[:dm, :rm] == tile[:dm, :rm]).all()
        assert (crop[dm:, :] == 0xCD).all() and (crop[:, rm:] == 0xCD).all()   # never writes outside the crop


def test_golden_random_frames(dropin, golden):
    for c, img in golden_random_frames(golden):
        rec = dropin.pack_frame(c["index"], img)
        assert len(rec) == c["record_len"] and sha(rec) == c["record_sha256"], (c["W"], c["H"])
        used, hdr, dec = dropin.unpack_frame(rec, c["W"], c["H"])
        assert used == len(rec) and hdr == (2, c["index"], 0) and (dec == img).all()


def test_golden_synthetic_streams(codec, golden):
    for s in golden["synthetic"]:
        fr = synth.gen_frames(s["kind"], s["n"], s["W"], s["H"], seed=s["seed"])
        stream, offs = codec.encode_host(fr, 0)
        assert np.diff(offs).astype(np.int64).tolist() == s["sizes"]
        assert sha(stream) == s["stream_sha256"], s


# ------------------------------------------------------------------ differential vs the oracle
@pytest.mark.parametrize("W,H", [(8, 8), (16, 8), (1, 1), (3, 5), (7, 9), (9, 7), (17, 23), (64, 64), (100, 37),
                                 (257, 129), (255, 8), (256, 16), (264, 24), (1001, 83), (2048, 16), (2056, 24),
                                 (2049, 9), (4096, 8), (4104, 16), (520, 520),
                                 # aligned widths that do not fill 256-tile partitions band by band: linear partitions
                                 # (256 consecutive tiles across band boundaries), full and partial last partitions
                                 (1280, 64), (2304, 48), (2560, 40), (1392, 104), (1104, 24), (4112, 16), (1280, 8),
                                 (2304, 2304), (1280, 1024)])
def test_sizes_and_edges(codec, W, H):
    rng = np.random.default_rng(W * 10007 + H)
    frames = np.stack([rand_frame(rng, W, H, ["classes", "noise", "flat"][i % 3]) for i in range(3)])
    roundtrip_check(codec, frames, first_index=1000)


@pytest.fixture(params=["direct", "staged"])
def odd_decode(request, monkeypatch):
    """both unpack kernels for odd-size frames with full-width partitions: re-aligned row stores straight from
    registers (the default) and the image staged in shared memory + one bulk store (DBDE_B200_ODD_DECODE=staged)"""
    monkeypatch.setenv("DBDE_B200_ODD_DECODE", request.param)
    return request.param


@pytest.mark.parametrize("W,H", [(1002, 19), (1004, 21), (1006, 17), (1003, 8), (2047, 17), (2041, 33), (2044, 9),
                                 (5, 1000), (33, 515), (15, 64), (250, 250), (1999, 41), (1000, 1003), (257, 64),
                                 (263, 70), (1016, 30), (2040, 12)])
def test_odd_sizes_full_width_partitions(codec, odd_decode, W, H):
    """W <= 2048 with W % 16 != 0 or H % 8 != 0: the contiguous-hull encoder staging and both odd-size
    decoders (every row alignment class: W % 8 = 0..7; one to eight bands per partition; partial last
    columns of 1..7 pixels; frames of exactly 32 tiles per band and narrower ones that keep the piecewise stores)"""
    rng = np.random.default_rng(W * 7919 + H)
    frames = np.stack([rand_frame(rng, W, H, ["classes", "noise", "flat", "classes"][i % 4]) for i in range(4)])
    roundtrip_check(codec, frames, first_index=7)
    roundtrip_check(codec, synth.gen_frames("mix", 3, W, H, f0=5))


def test_rejected_frames_between_good_ones_odd_size(codec, odd_decode):
    """the odd-size decoders skip rejected frames (the staged one without losing step with its store warp;
    dbde_util.cpp:296-303: image untouched), odd size, several partitions per frame"""
    W, H, N = 1001, 43, 9
    wh = ((W + 7) // 8) * ((H + 7) // 8)
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    bad = stream.copy()
    for i in (0, 3, 4, 8):
        bad[int(offs[i]) + 28 + 2 * wh] ^= 1       # n64 != sum(depth)
    dec, status, _ = codec.decode_host(bad, offs[:N], W, H, fill=0xCD)
    for i in range(N):
        if i in (0, 3, 4, 8):
            assert status[i] == pkg.ST_BAD_WORD_COUNT and (dec[i] == 0xCD).all(), i
        else:
            assert status[i] == 0 and (dec[i] == fr[i]).all(), i


@pytest.mark.parametrize("W,H", [(512, 64), (2048, 24), (4096, 16), (264, 40)])
def test_many_depths_per_warp_aligned(codec, W, H):
    """all nine depths inside every warp on the aligned kernels: the depth-agnostic row packer /
    unpacker (taken when a warp holds several depths) against the per-depth specialisations' oracle"""
    roundtrip_check(codec, synth.gen_frames("mix", 5, W, H, f0=3))
    rng = np.random.default_rng(W + H)
    roundtrip_check(codec, np.stack([rand_frame(rng, W, H, "classes") for _ in range(3)]))


@pytest.mark.parametrize("W,H", [(64, 40), (1001, 43), (2048, 16), (4096, 8), (2049, 9), (10, 10)])
def test_invert_endian_variant_matches_the_reference_built_with_the_macro(dropin, W, H):
    """DBDE_INVERT_ENDIAN (dbde_util.cpp:15-19,24-27,246-270): tile rows byte-reversed on the way in and
    out; every kernel family (wide, aligned, contiguous odd, segmented odd) against the unmodified
    reference compiled with the macro.  Also through the C++ drop-in, which follows the process setting."""
    V = oracle.best_variants()
    rng = np.random.default_rng(W + 31 * H)
    fr = np.stack([rand_frame(rng, W, H, ["classes", "noise", "classes"][i % 3]) for i in range(3)])
    want, sizes = V.pack_frames(fr, 9)
    c = pkg.Codec(0)
    try:
        c.set_invert_endian(True)
        got, offs = c.encode_host(fr, 9)
        assert (got == want).all()
        dec, status, _ = c.decode_host(want, offs[:3], W, H)
        assert (status == 0).all() and (dec == fr).all()
        plain, _ = ORA.pack_frames(fr, 9)
        assert not np.array_equal(plain, want)
    finally:
        c.close()
    try:
        pkg.set_format_variants(True, True)
        rec = dropin.pack_frame(9, fr[0])
        assert (rec == want[:int(sizes[0])]).all()
        used, hdr, img = dropin.unpack_frame(rec, W, H)
        assert used == int(sizes[0]) and hdr == (2, 9, 0) and (img == fr[0]).all()
        assert (dropin.pack_video_header(3, H, W, 59.94) == V.pack_video_header(3, H, W, 59.94)).all()
    finally:
        pkg.set_format_variants(False, False)
    assert (dropin.pack_frame(9, fr[0]) == ORA.pack_frame(9, fr[0])).all()


def test_stored_differential_and_variant_records(codec, dropin):
    """tests/golden/golden_differential.json through the CUDA path: the 60 small random frames through the C++
    drop-in, and the DBDE_INVERT_ENDIAN + DBDE_HZ_AS_INTEGER streams and video header with both variants on"""
    import importlib.util
    import json
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    spec = importlib.util.spec_from_file_location("make_golden_differential", os.path.join(gdir, "make_golden_differential.py"))
    mg = importlib.util.module_from_spec(spec); spec.loader.exec_module(mg)
    gold = json.load(open(os.path.join(gdir, "golden_differential.json")))
    for (i, W, H, img), c in zip(mg.differential_frames(), gold["differential"], strict=True):
        rec = dropin.pack_frame(i, img)
        assert len(rec) == c["record_len"] and sha(rec) == c["record_sha256"], (W, H)
        used, hdr, dec = dropin.unpack_frame(rec, W, H)
        assert used == len(rec) and hdr == (2, i, 0) and (dec == img).all()
    c = pkg.Codec(0)
    try:
        c.set_invert_endian(True)
        for (W, H, style, fr), g in zip(mg.variant_frames(), gold["variants"]["cases"], strict=True):
            got, offs = c.encode_host(fr, 5)
            assert np.diff(offs).astype(np.int64).tolist() == g["sizes"] and sha(got) == g["stream_sha256"], (W, H, style)
            dec, status, _ = c.decode_host(got, offs[:2], W, H)
            assert (status == 0).all() and (dec == fr).all()
    finally:
        c.close()
    try:
        pkg.set_format_variants(True, True)
        assert dropin.pack_video_header(3, 480, 640, 29.97).tobytes().hex() == gold["variants"]["video_header"]["hex"]
    finally:
        pkg.set_format_variants(False, False)


def test_empty_batch_and_bad_arguments(codec):
    """nframes == 0 is a no-op that succeeds; nonsense dimensions and short output buffers are refused
    with an error code instead of a launch (the reference has no such checks: SURVEY 8b 'no bounds
    checking anywhere' -- the C ABI adds capacity arguments, the drop-in layer keeps the contract)"""
    got, offs = codec.encode_host(np.zeros((0, 16, 16), dtype=np.uint8), 0)
    assert len(got) == 0 and offs.tolist() == [0]
    dec, status, _ = codec.decode_host(np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.uint64), 16, 16)
    assert dec.shape == (0, 16, 16) and len(status) == 0
    lib, h = codec.lib, codec.h
    buf = np.zeros(4096, dtype=np.uint8)
    offs = np.zeros(4, dtype=np.uint64)
    assert lib.dbde_b200_encode_host(h, buf.ctypes.data, 0, 8, 0, 1, buf.ctypes.data, 4096, offs.ctypes.data) != 0
    assert lib.dbde_b200_encode_host(h, buf.ctypes.data, 8, -1, 0, 1, buf.ctypes.data, 4096, offs.ctypes.data) != 0
    assert lib.dbde_b200_encode_host(h, buf.ctypes.data, 8, 8, 0, -1, buf.ctypes.data, 4096, offs.ctypes.data) != 0
    fr = np.arange(64, dtype=np.uint8).reshape(1, 8, 8)           # depth 6: a 32 + 2 + 48 = 82-byte record
    assert lib.dbde_b200_encode_host(h, fr.ctypes.data, 8, 8, 0, 1, buf.ctypes.data, 40, offs.ctypes.data) != 0
    assert b"" != lib.dbde_b200_last_error()
    roundtrip_check(codec, fr)                                    # the context is still usable after refusals


@pytest.mark.parametrize("W,H,N", [(8200, 9, 2), (16384, 24, 1), (32768, 8, 1), (16400, 17, 1), (1, 3000, 2), (3000, 1, 2),
                                   (8192, 4096, 1)])
def test_very_wide_tall_and_big_frames(codec, W, H, N):
    """many band segments per band (w up to 4096 tiles = 16 segments), degenerate 1-pixel-wide/high
    frames, and one 32 MiB frame (131 072 partitions-worth of look-back in one chain)"""
    if W * H > 1 << 22:
        fr = synth.gen_frames("mix", N, W, H, f0=2)
    else:
        rng = np.random.default_rng(W ^ H)
        fr = np.stack([rand_frame(rng, W, H, "classes") for _ in range(N)])
    roundtrip_check(codec, fr, first_index=2 ** 63 + 5)


def test_caller_owned_buffers_can_be_page_locked(codec, dropin):
    """dbde_b200_host_register / _unregister on memory the caller owns (what a maintainer adds around a
    long-lived frame buffer so the drop-in calls copy by DMA): same bytes, and the buffers work again after
    unregistering"""
    W, H = 520, 264
    fr = synth.gen_frames("mix", 1, W, H, f0=9)[0].copy()
    rec_buf = np.zeros(codec.lib.dbde_b200_frame_record_bound(W, H), dtype=np.uint8)
    assert codec.lib.dbde_b200_host_register(fr.ctypes.data, fr.nbytes) == 0
    assert codec.lib.dbde_b200_host_register(rec_buf.ctypes.data, rec_buf.nbytes) == 0
    try:
        want = ORA.pack_frame(3, fr)
        for _ in range(3):
            got = dropin.pack_frame(3, fr)
            assert (got == want).all()
        offs = np.zeros(2, dtype=np.uint64)
        codec.encode_host_raw(fr.ctypes.data, W, H, 3, 1, rec_buf.ctypes.data, rec_buf.nbytes, offs.ctypes.data)
        assert int(offs[1]) == len(want) and (rec_buf[:len(want)] == want).all()
    finally:
        assert codec.lib.dbde_b200_host_unregister(fr.ctypes.data) == 0
        assert codec.lib.dbde_b200_host_unregister(rec_buf.ctypes.data) == 0
    assert (dropin.pack_frame(3, fr) == want).all()
    assert codec.lib.dbde_b200_host_register(None, 16) != 0 and codec.lib.dbde_b200_host_unregister(None) != 0


def test_integration_example_writes_the_references_bytes():
    """examples/batched_roundtrip.cpp (the C++ binding of INTEGRATION.md section 2): built with g++ on the
    box, run, and its .dbde file compared with what the reference's dbde_pack_video_header +
    dbde_pack_frame write for the same frames"""
    import subprocess
    from conftest import build_example
    exe = build_example()
    W, H, N = 333, 251, 7
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "example.dbde")
        r = subprocess.run([exe, path, str(W), str(H), str(N)], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "round trip exact" in r.stdout
        got = np.fromfile(path, dtype=np.uint8)
    # the example's frame generator, restated
    z = np.uint64(42)
    a, c = np.uint64(6364136223846793005), np.uint64(1442695040888963407)
    n = N * H * W
    zs = np.empty(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        for i in range(n):
            z = z * a + c
            zs[i] = z
    f, y, x = np.meshgrid(np.arange(N), np.arange(H), np.arange(W), indexing="ij")
    fr = ((((x + 3 * f) >> 3) + ((y >> 4) & 15) + ((zs.reshape(N, H, W) >> np.uint64(60)) & np.uint64(3)).astype(np.int64)) & 255).astype(np.uint8)
    want, _ = ORA.pack_frames(fr, 0)
    hdr = ORA.pack_video_header(3, H, W, 25.0)
    assert len(got) == 28 + len(want) and (got[:28] == hdr).all() and (got[28:] == want).all()


def test_random_geometries(codec):
    """120 seeded random cases: any width/height from 1 to 300 (and a few wide ones), 1-5 frames, every
    content style, random first index -- sweeps W % 8, H % 8, bands per partition and tiles per warp
    through both the aligned and the odd-size kernels"""
    rng = np.random.default_rng(20261018)
    for case in range(120):
        if case % 10 == 9:
            W, H = int(rng.integers(2040, 2300)), int(rng.integers(1, 40))
        else:
            W, H = int(rng.integers(1, 301)), int(rng.integers(1, 301))
        N = int(rng.integers(1, 6))
        styles = ["classes", "noise", "flat", "low"]
        frames = []
        for i in range(N):
            st = styles[int(rng.integers(0, 4))]
            if st == "low":
                img = (int(rng.integers(0, 250)) + (rng.integers(0, 256, (H, W)) & int(rng.integers(0, 4)))).astype(np.uint8)
            else:
                img = rand_frame(rng, W, H, st)
            frames.append(img)
        roundtrip_check(codec, np.stack(frames), first_index=int(rng.integers(0, 2 ** 62)))


def test_gpu_validation_without_decoding(codec):
    """dbde_b200_validate_host (SURVEY 8 f-2): the reference's accept/reject decision for every record
    (dbde_util.cpp:295-303,335), taken on the GPU without decoding; must agree with what the decoder and
    the oracle say, for good and for damaged records"""
    W, H, N = 1001, 43, 12
    wh = ((W + 7) // 8) * ((H + 7) // 8)
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 40)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    status, index = codec.validate_host(stream, offs[:N], W, H)
    assert (status == 0).all() and index.tolist() == list(range(40, 40 + N))
    bad = stream.copy()
    bad[int(offs[1]) + 20] += 1                 # nb != wh
    bad[int(offs[2]) + 24 + wh] += 1            # nm != wh
    bad[int(offs[5]) + 28 + 2 * wh] ^= 1        # n64 != sum(depth)
    bad[int(offs[7])] = 9                       # frame tag != 2
    bad[int(offs[9]) + 24 + 3] = 9              # a depth byte > 8
    status, _ = codec.validate_host(bad, offs[:N], W, H)
    _, dstatus, _ = codec.decode_host(bad, offs[:N], W, H)
    assert status.tolist() == dstatus.tolist()
    assert status[1] == pkg.ST_BAD_DEPTH_COUNT and status[2] == pkg.ST_BAD_MIN_COUNT and status[5] == pkg.ST_BAD_WORD_COUNT
    assert status[7] == pkg.ST_BAD_FRAME_HEADER and status[9] & pkg.ST_DEPTH_TOO_BIG
    for i in range(N):
        o_used, o_hdr, _ = ORA.unpack_frame(bad[int(offs[i]):int(offs[i + 1])], W, H)
        if i != 9:                               # depth > 8 is the documented deviation (reference: unpinned)
            assert (status[i] == 0) == (o_hdr[0] == 2), i
    launches = codec.launches()
    codec.validate_host(stream, offs[:N], W, H)
    assert codec.launches() - launches == 1      # the scan pre-pass alone


# ------------------------------------------------------------------ DBDE16 (SURVEY 8 f-4)
def rand_frame16(rng, W, H, style):
    if style == "noise":
        return rng.integers(0, 65536, (H, W), dtype=np.uint16)
    if style == "flat":
        return np.full((H, W), rng.integers(0, 65536), dtype=np.uint16)
    if style == "byte":
        return rng.integers(0, 256, (H, W)).astype(np.uint16)
    th, tw = (H + 7) // 8, (W + 7) // 8
    k = rng.integers(0, 17, (th, tw))
    rg = (1 << k) - 1
    mn = (rng.random((th, tw)) * (65536 - rg)).astype(np.int64)
    big = (mn[:, :, None, None] + (rng.integers(0, 65536, (th, tw, 8, 8)) & rg[:, :, None, None]))
    return big.transpose(0, 2, 1, 3).reshape(th * 8, tw * 8)[:H, :W].astype(np.uint16)


@pytest.mark.parametrize("W,H", [(8, 8), (10, 10), (64, 64), (1, 1), (7, 9), (17, 23), (264, 24), (1001, 83), (2048, 16), (2056, 24),
                                 (520, 520), (3000, 1), (1, 300)])
def test_dbde16_matches_its_oracle(codec, W, H):
    """16-bit frames: records byte-identical to oracle.port16 (the definition of the extension), decode
    identical to the source, aligned (W % 8 == 0) and element-wise paths, every depth 0..16"""
    rng = np.random.default_rng(W * 31 + H)
    fr = np.stack([rand_frame16(rng, W, H, ["classes", "noise", "flat", "byte", "classes"][i % 5]) for i in range(5)])
    want, sizes = oracle.port16.pack_frames(fr, 77)
    got, offs = codec.encode16_host(fr, 77)
    assert int(offs[5]) == len(want) and offs[:5].tolist() == [0] + np.cumsum(sizes).tolist()[:-1]
    assert (got == want).all(), int(np.argmax(got != want))
    dec, status, index = codec.decode16_host(want, offs[:5], W, H)
    assert (status == 0).all() and index.tolist() == list(range(77, 82)) and (dec == fr).all()


def test_dbde16_frozen_fixtures_on_the_gpu(codec):
    """the committed DBDE16 fixtures (tests/golden/golden16.json) through the CUDA path"""
    import importlib.util
    import json
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    spec = importlib.util.spec_from_file_location("make_golden16", os.path.join(gdir, "make_golden16.py"))
    mg = importlib.util.module_from_spec(spec); spec.loader.exec_module(mg)
    for c in json.load(open(os.path.join(gdir, "golden16.json")))["cases"]:
        fr = mg.frames16(c)
        got, offs = codec.encode16_host(fr, 11)
        assert np.diff(offs).astype(np.int64).tolist() == c["sizes"] and sha(got) == c["stream_sha256"], c
        dec, status, _ = codec.decode16_host(got, offs[:c["N"]], c["W"], c["H"])
        assert (status == 0).all() and (dec == fr).all()


def test_dbde16_of_8_bit_content_is_the_8_bit_codec(codec):
    """the embedding that ties the extension to the reference: pixels < 256 -> the reference's depth plane
    and U64 words, minima widened to two bytes"""
    W, H, N = 1001, 43, 3
    wh = ((W + 7) // 8) * ((H + 7) // 8)
    fr8 = synth.gen_frames("mix", N, W, H)
    a, sa = ORA.pack_frames(fr8, 0)
    b, offs = codec.encode16_host(fr8.astype(np.uint16), 0)
    pa = 0
    for i in range(N):
        ra, rb = a[pa:pa + int(sa[i])], b[int(offs[i]):int(offs[i + 1])]
        assert len(rb) == len(ra) + wh and (ra[:24 + wh] == rb[:24 + wh]).all() and (ra[28 + 2 * wh:] == rb[28 + 3 * wh:]).all()
        assert (rb[28 + wh:28 + 3 * wh].view(np.uint16) == ra[28 + wh:28 + 2 * wh]).all()
        pa += int(sa[i])


def test_dbde16_full_size_frames_across_staging_batches(codec):
    """2048x2048 U16 (8 MiB per frame): 20 frames cross the host path's 128 MiB staging batch, 256 partitions per
    frame exercise the per-frame look-back chains; 12-bit camera-like content + two full-range frames"""
    W = H = 2048
    rng = np.random.default_rng(12)
    y, x = np.mgrid[0:H, 0:W]
    base = (600 + x // 16 + y // 8).astype(np.uint16)
    fr = np.stack([base + rng.integers(0, 32, (H, W), dtype=np.uint16) for _ in range(18)]
                  + [rng.integers(0, 65536, (H, W), dtype=np.uint16) for _ in range(2)])
    want, sizes = oracle.port16.pack_frames(fr, 1000)
    got, offs = codec.encode16_host(fr, 1000)
    assert int(offs[20]) == len(want) and (got == want).all()
    dec, status, index = codec.decode16_host(got, offs[:20], W, H)
    assert (status == 0).all() and index.tolist() == list(range(1000, 1020)) and (dec == fr).all()


def test_dbde16_rejects_damaged_records_and_many_frames(codec):
    W, H, N = 136, 72, 40
    wh = 17 * 9
    rng = np.random.default_rng(8)
    fr = np.stack([rand_frame16(rng, W, H, "classes") for _ in range(N)])
    stream, sizes = oracle.port16.pack_frames(fr, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    bad = stream.copy()
    bad[int(offs[3]) + 24 + wh] ^= 1            # nm != 2*wh
    bad[int(offs[9]) + 28 + 3 * wh] ^= 1        # n64 != sum(depth)
    bad[int(offs[20]) + 24 + 5] = 17            # depth > 16
    dec, status, _ = codec.decode16_host(bad, offs[:N], W, H, fill=0xCDCD)
    assert status[3] == pkg.ST_BAD_MIN_COUNT and status[9] == pkg.ST_BAD_WORD_COUNT and status[20] & pkg.ST_DEPTH_TOO_BIG
    for i in range(N):
        if i in (3, 9, 20):
            assert (dec[i] == 0xCDCD).all()
        else:
            assert status[i] == 0 and (dec[i] == fr[i]).all()


def test_many_tiny_frames(codec):
    """20 000 README-sized frames in one batch: one partition per frame, chunking and slot compaction
    at a record size (<= 296 bytes) far below any staging granularity"""
    N = 20000
    rng = np.random.default_rng(5)
    fr = rng.integers(0, 256, (N, 10, 10), dtype=np.uint8)
    fr[::3] &= 0x0F
    fr[::7] = 200
    roundtrip_check(codec, fr, first_index=123456789)


def test_every_depth_class_uniform(codec):
    """a whole frame at each depth 0..8 (uniform-depth warps hit the worst staging strides)"""
    rng = np.random.default_rng(11)
    for k in range(9):
        rg = (1 << k) - 1
        mn = 0 if k == 8 else 10
        fr = (mn + (rng.integers(0, 256, (2, 64, 512)) & rg)).astype(np.uint8)
        fr[:, ::8, ::8] = mn
        fr[:, ::8, 1::8] = mn + rg
        roundtrip_check(codec, fr)


def test_batches_and_chunking(codec):
    """many frames, forced small chunks: chunk seams must not show in the stream"""
    fr = synth.gen_frames("mix", 37, 136, 72)
    codec.set_chunk_frames(5)
    try:
        roundtrip_check(codec, fr, first_index=2 ** 40)
    finally:
        codec.set_chunk_frames(0)
    roundtrip_check(codec, fr, first_index=2 ** 40)


def test_synthetic_configs_small(codec):
    """BASELINE configs 3 and 4 (odd 1001x1003 depth mix; low-entropy) + noise, against the oracle"""
    roundtrip_check(codec, synth.gen_frames("mix", 2, 1001, 1003))
    roundtrip_check(codec, synth.gen_frames("low", 1, 4096, 512))
    roundtrip_check(codec, synth.gen_frames("noise", 2, 2048, 256))
    roundtrip_check(codec, synth.gen_frames("micro", 2, 2048, 2048))


def test_device_resident_api(codec):
    """the batched device entry points on HBM-resident buffers: one slot per record, every slot
    byte-identical to the oracle's record; unaligned slot bases and a custom stride included"""
    W, H, N = 256, 128, 9
    fr = synth.gen_frames("mix", N, W, H)
    want, sizes = ORA.pack_frames(fr, 3)
    starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    d_fr = codec.device_alloc(fr.nbytes)
    d_dec = codec.device_alloc(fr.nbytes)
    d_off = codec.device_alloc(8 * N)
    d_sz = codec.device_alloc(8 * N)
    d_st = codec.device_alloc(4 * N)
    d_ix = codec.device_alloc(8 * N)
    stride0 = codec.slot_stride(W, H)
    cap = (stride0 + 48) * N + 64
    d_out = codec.device_alloc(cap + 64)
    try:
        codec.h2d(d_fr, fr)
        for shift, stride in ((0, 0), (4, 0), (12, stride0 + 48), (1, stride0 + 3), (2, 0)):
            st = stride or stride0
            codec.h2d(d_out, np.full(cap + 64, 0xEE, dtype=np.uint8))
            codec.encode_device(d_fr, W, H, 3, N, d_out + shift, cap, d_off, d_sz, slot_stride=stride)
            offs = codec.d2h(d_off, 8 * N, np.uint64)
            szs = codec.d2h(d_sz, 8 * N, np.uint64)
            assert offs.tolist() == [i * st for i in range(N)] and szs.tolist() == sizes.tolist()
            buf = codec.d2h(d_out + shift, st * N)
            for i in range(N):
                rec = buf[i * st:i * st + int(szs[i])]
                assert (rec == want[starts[i]:starts[i + 1]]).all(), (shift, i)
                assert (buf[i * st + int(szs[i]):(i + 1) * st] == 0xEE).all()      # nothing written past the record
            codec.h2d(d_dec, np.zeros_like(fr))
            codec.decode_device(d_out + shift, st * N, d_off, W, H, N, d_dec, d_st, d_ix)
            assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
            assert codec.d2h(d_ix, 8 * N, np.uint64).tolist() == list(range(3, 3 + N))
            assert (codec.d2h(d_dec, fr.nbytes).reshape(fr.shape) == fr).all(), shift
    finally:
        for p in (d_fr, d_out, d_off, d_sz, d_dec, d_st, d_ix):
            codec.device_free(p)


def test_single_frame_many_partitions(codec):
    """one big frame alone: every partition of the frame is in flight at once, so the per-frame
    look-back chain has to resolve across concurrently running CTAs"""
    for W, H in [(2048, 2048), (4096, 1024), (1001, 1003)]:
        roundtrip_check(codec, synth.gen_frames("mix", 1, W, H))
    roundtrip_check(codec, synth.gen_frames("micro", 3, 2048, 1024))


def test_invalid_streams_are_rejected_and_leave_the_image_untouched(codec, dropin):
    """dbde_util.cpp:296,299,303 (+ header tag :335): status bits, image untouched, good frames
    in the same batch still decode"""
    W, H, N = 48, 40, 6
    wh = 6 * 5
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    bad = stream.copy()
    bad[int(offs[1]) + 20] += 1                 # nb != wh
    bad[int(offs[2]) + 24 + wh] += 1            # nm != wh
    bad[int(offs[3]) + 28 + 2 * wh] += 1        # n64 != sum(depth)
    bad[int(offs[4])] = 9                       # frame tag != 2
    dec, status, _ = codec.decode_host(bad, offs[:N], W, H, fill=0xCD)
    assert status.tolist() == [0, pkg.ST_BAD_DEPTH_COUNT, pkg.ST_BAD_MIN_COUNT, pkg.ST_BAD_WORD_COUNT,
                               pkg.ST_BAD_FRAME_HEADER, 0]
    for i in range(N):
        if status[i]:
            assert (dec[i] == 0xCD).all()
        else:
            assert (dec[i] == fr[i]).all()
    # a depth byte > 8 is rejected (documented deviation: the reference does not pin this case)
    bad = stream.copy()
    bad[int(offs[0]) + 24] = 9
    _, status, _ = codec.decode_host(bad, offs[:N], W, H)
    assert status[0] & pkg.ST_DEPTH_TOO_BIG
    # truncated stream
    _, status, _ = codec.decode_host(stream[:int(offs[N]) - 8], offs[:N], W, H)
    assert status[N - 1] & pkg.ST_TRUNCATED and (status[:N - 1] == 0).all()
    # the drop-in signatures: 0 / u64s == -1, pointer left just after the header (:342-343)
    rec = ORA.pack_frame(3, fr[0])
    b = rec.copy(); b[20] += 1
    used, hdr, img = dropin.unpack_frame(b, W, H, fill=0xCD)
    o_used, o_hdr, o_img = ORA.unpack_frame(b, W, H, fill=0xCD)
    assert (used, hdr) == (o_used, o_hdr) == (20, (0xFFFFFFFF, 3, 0)) and (img == o_img).all()
    n, img = dropin.unpack_image(b[20:], W, H, fill=0xCD)
    assert n == 0 and (img == 0xCD).all()


def test_full_size_properties(codec):
    """BASELINE config 2 at full frame size: 2048x2048 micro, 24 frames: byte-equal to the
    reference, decode(encode(x)) == x, and the stream indexes back to the same offsets."""
    N, W, H = 24, 2048, 2048
    fr = synth.gen_frames("micro", N, W, H)
    stream, offs = codec.encode_host(fr, 0)
    if oracle.ref is not None:
        want, sizes = oracle.ref.pack_frames(fr, 0)
        assert len(want) == len(stream) and (want == stream).all()
    assert codec.index_stream(stream, W, H).tolist() == offs.tolist()
    dec, status, index = codec.decode_host(stream, offs[:N], W, H)
    assert (status == 0).all() and index.tolist() == list(range(N)) and (dec == fr).all()
    depth = stream[24:24 + 65536]
    assert abs((depth == 3).mean() - 0.80) < 0.02           # SURVEY.md 8d histogram


def test_gpu_synth_matches_cpu_generator(codec):
    for kind, W, H in [("noise", 70, 33), ("micro", 512, 256), ("mix", 1001, 64), ("low", 256, 256)]:
        n = 2
        d = codec.device_alloc(n * W * H)
        synth.gen_frames_device(kind, n, W, H, d, seed=42, f0=5)
        got = codec.d2h(d, n * W * H).reshape(n, H, W)
        codec.device_free(d)
        assert (got == synth.gen_frames(kind, n, W, H, seed=42, f0=5)).all(), kind


def test_sharded_host_api_matches_single_context(codec):
    """dbde_b200_{en,de}code_host_sharded: contiguous frame ranges over several contexts (here two
    contexts on one GPU; on a multi-GPU box one per device) == the single-context stream"""
    fr = synth.gen_frames("mix", 11, 264, 136)
    want, sizes = ORA.pack_frames(fr, 50)
    others = [pkg.Codec(0), pkg.Codec(0)]
    try:
        for group in ([codec] + others, others):
            stream, offs = pkg.encode_host_sharded(group, fr, 50)
            assert len(stream) == len(want) and (stream == want).all()
            assert offs.tolist() == [0] + np.cumsum(sizes).tolist()
            dec, status, index = pkg.decode_host_sharded(group, stream, offs[:-1], 264, 136)
            assert (status == 0).all() and index.tolist() == list(range(50, 61)) and (dec == fr).all()
    finally:
        for c in others:
            c.close()


def test_file_walker(dropin):
    """dbde_start_file_walk / dbde_walk_a_file / dbde_end_file_walk on a written .dbde file,
    including the tiny odd frames that overflow the reference's buffer estimate (SURVEY C10)."""
    for W, H, N, buffered in [(10, 10, 7, 2), (136, 72, 11, 4), (64, 64, 3, 8)]:
        fr = synth.gen_frames("noise" if W == 10 else "mix", N, W, H)
        stream, _ = ORA.pack_frames(fr, 100)
        with tempfile.NamedTemporaryFile(suffix=".dbde", delete=False) as f:
            f.write(ORA.pack_video_header(3, H, W, 30.0).tobytes())
            f.write(stream.tobytes())
            path = f.name
        try:
            vh, frames = dropin.walk_file(path, buffered)
            assert vh == (3, H, W, 30.0) and len(frames) == N
            for i, (hdr, img) in enumerate(frames):
                assert hdr == (2, 100 + i, 0) and (img == fr[i]).all()
        finally:
            os.unlink(path)


def test_file_walkers_side_by_side_early_close_and_damaged_frame(dropin):
    """the walker's helper thread: two files walked alternately, one closed long before its end (the helper is
    mid-batch or waiting), a file whose 6th record is damaged (frames 0-4 come out, then the walk ends as at
    dbde_util.cpp:416), and a file cut in the middle of a record"""
    W, H, N = 200, 120, 23
    wh = 25 * 15
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    hdr = ORA.pack_video_header(3, H, W, 30.0).tobytes()
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    with tempfile.TemporaryDirectory() as d:
        good, bad, cut = (os.path.join(d, n) for n in ("good.dbde", "bad.dbde", "cut.dbde"))
        open(good, "wb").write(hdr + stream.tobytes())
        dmg = stream.copy(); dmg[int(offs[5]) + 28 + 2 * wh] ^= 1
        open(bad, "wb").write(hdr + dmg.tobytes())
        open(cut, "wb").write(hdr + stream[:int(offs[9]) + 100].tobytes())
        a, vha = dropin.walk_open(good, 3)
        b, vhb = dropin.walk_open(good, 5)
        assert vha == vhb == (3, H, W, 30.0)
        for i in range(N):
            ra = dropin.walk_next(a)
            assert ra[0] == (2, i, 0) and (ra[1] == fr[i]).all()
            if i < 4:
                rb = dropin.walk_next(b)
                assert rb[0] == (2, i, 0) and (rb[1] == fr[i]).all()
            if i == 4:
                dropin.walk_close(b)                      # 19 frames early
        assert dropin.walk_next(a) is None
        dropin.walk_close(a)
        vh, frames = dropin.walk_file(bad, 4)
        assert len(frames) == 5 and all((img == fr[i]).all() for i, (_, img) in enumerate(frames))
        vh, frames = dropin.walk_file(cut, 4)
        assert len(frames) == 9 and all((img == fr[i]).all() for i, (_, img) in enumerate(frames))


def test_the_references_own_test_program_passes_against_this_library():
    """SURVEY 8(f-3): dbde_util_test.cpp -- the reference's whole test main (example tiles incl. the
    three partial-tile cases, the 8x16 known-answer test in both directions, the 2536x2048 noise
    round trip, 1024 random single-tile round trips) -- linked against libdbde_b200.so instead of
    dbde_util.o (oracle/Makefile `reftest`).  It must exit 0 and print exactly what the same program
    linked against the unmodified reference prints, apart from its three rdtsc timing lines."""
    import subprocess
    d = os.path.join(os.path.dirname(os.path.abspath(oracle.__file__)), "_ref")
    ours, ref = os.path.join(d, "dbde_test_b200"), os.path.join(d, "dbde_test_ref")
    if not (os.path.exists(ours) and os.path.exists(ref)):
        pytest.skip("oracle/_ref test programs not built (needs /root/reference at build time)")
    a = subprocess.run([ours], capture_output=True, text=True, timeout=300)
    b = subprocess.run([ref], capture_output=True, text=True, timeout=300)
    assert b.returncode == 0, b.stdout[-2000:]
    assert a.returncode == 0, a.stdout[-2000:] + a.stderr[-2000:]
    la, lb = a.stdout.splitlines(), b.stdout.splitlines()
    assert len(la) == len(lb) and len(la) > 10
    assert la[:-3] == lb[:-3]
    assert "!! 0 of 5193728" in a.stdout and "Failed iteration" not in a.stdout


def test_sharded_encode_interleaves_chunk_ranges_in_stream_order(codec):
    """encode_host_sharded deals chunk-sized frame ranges round-robin to the contexts and places them
    in stream order as their sizes become known: many small chunks over three contexts (on a multi-GPU
    box: spread over the devices), uneven last chunk, and fewer chunks than contexts."""
    ndev = pkg.load().dbde_b200_device_count()
    group = [codec] + [pkg.Codec(i % ndev) for i in range(1, 3)]
    try:
        for n, chunk in [(29, 2), (29, 3), (2, 5), (1, 1), (16, 1)]:
            fr = synth.gen_frames("mix", n, 200, 104, f0=n)
            want, sizes = ORA.pack_frames(fr, 1000)
            group[0].set_chunk_frames(chunk)           # the sharded call takes its chunk size from context 0
            try:
                stream, offs = pkg.encode_host_sharded(group, fr, 1000)
            finally:
                group[0].set_chunk_frames(0)
            assert len(stream) == len(want) and (stream == want).all(), (n, chunk)
            assert offs.tolist() == [0] + np.cumsum(sizes).tolist()
            dec, status, index = pkg.decode_host_sharded(group, stream, offs[:-1], 200, 104)
            assert (status == 0).all() and index.tolist() == list(range(1000, 1000 + n)) and (dec == fr).all()
    finally:
        for c in group[1:]:
            c.close()


def test_sharded_encode_reports_a_short_output_buffer_instead_of_hanging(codec):
    """a worker that cannot place its range must fail the whole call (and release the workers waiting
    for their turn), not deadlock or write past the buffer"""
    import ctypes as C
    lib = codec.lib
    fr = synth.gen_frames("noise", 12, 64, 64)
    others = [pkg.Codec(0)]
    try:
        codec.set_chunk_frames(2)
        cap = 3 * (32 + 66 * 64) + 100                 # room for about three of the twelve records
        out = np.full(cap + 4096, 0xEE, dtype=np.uint8)
        offs = np.zeros(13, dtype=np.uint64)
        arr = (C.c_void_p * 2)(codec.h.value, others[0].h.value)
        rc = lib.dbde_b200_encode_host_sharded(arr, 2, fr.ctypes.data, 64, 64, 0, 12, out.ctypes.data, cap, offs.ctypes.data)
        assert rc != 0
        assert (out[cap:] == 0xEE).all()               # nothing beyond the stated capacity was touched
        rc = lib.dbde_b200_encode_host(codec.h, fr.ctypes.data, 64, 64, 0, 12, out.ctypes.data, cap, offs.ctypes.data)
        assert rc == pkg.load().dbde_b200_encode_host(codec.h, fr.ctypes.data, 64, 64, 0, 12, out.ctypes.data, cap,
                                                      offs.ctypes.data) != 0
        assert (out[cap:] == 0xEE).all()
        # and the contexts still work afterwards
        codec.set_chunk_frames(0)
        want, _ = ORA.pack_frames(fr, 0)
        stream, _ = pkg.encode_host_sharded([codec] + others, fr, 0)
        assert (stream == want).all()
    finally:
        codec.set_chunk_frames(0)
        for c in others:
            c.close()


def test_file_writer_and_reader_roundtrip_against_the_oracle_file(codec, dropin):
    """SURVEY 8(f-1): dbde_b200_writer_* must produce byte for byte the file the reference's functions
    would (dbde_pack_video_header + dbde_pack_frame per frame, dbde_util_test.cpp:204-211), for batch
    sizes that do and do not divide the frame count; dbde_b200_reader_* and the reference-compatible
    walker must both read it back; a corrupted record stops the reader like the walker (:416)."""
    for W, H, N, batch in [(10, 10, 9, 4), (136, 72, 23, 5), (264, 136, 12, 16), (1001, 1003, 3, 2)]:
        fr = synth.gen_frames("mix", N, W, H, f0=3)
        stream, sizes = ORA.pack_frames(fr, 500)
        want = np.concatenate([ORA.pack_video_header(3, H, W, 12.5), stream])
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "a.dbde")
            nf, nb = pkg.write_file(codec, path, fr, hz=12.5, first_index=500, batch=batch)
            got = np.fromfile(path, dtype=np.uint8)
            assert nf == N and nb == len(want) and len(got) == len(want) and (got == want).all(), (W, H, N, batch)
            for rb in (1, batch, N + 3):
                (w, h, hz), frames, idx, st = pkg.read_file(codec, path, batch=rb)
                assert (w, h, hz) == (W, H, 12.5) and (st == 0).all()
                assert idx.tolist() == list(range(500, 500 + N)) and (frames == fr).all()
            vh, frames = dropin.walk_file(path, 4)
            assert vh == (3, H, W, 12.5) and len(frames) == N and all((img == fr[i]).all() for i, (_, img) in enumerate(frames))
            # break the depth plane of frame 5 (if there is one): frames 0..4 come back, frame 5 is flagged, then EOF
            if N > 5:
                bad = got.copy()
                off5 = 28 + int(np.sum(sizes[:5]))
                bad[off5 + 24] = 9                                    # a depth byte > 8
                bad.tofile(path)
                _, frames, idx, st = pkg.read_file(codec, path, batch=4, fill=0xCD)
                assert len(frames) == 6 and (st[:5] == 0).all() and st[5] != 0
                assert (frames[:5] == fr[:5]).all() and (frames[5] == 0xCD).all()
            # a file cut in the middle of its last record: the torn record is not handed out
            got[:len(got) - 7].tofile(path)
            _, frames, idx, st = pkg.read_file(codec, path, batch=batch)
            assert len(frames) == N - 1 and (frames == fr[:N - 1]).all()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "junk.dbde")
        np.arange(100, dtype=np.uint8).tofile(path)
        with pytest.raises(pkg.DbdeError):
            pkg.read_file(codec, path)


@pytest.mark.parametrize("kind,N,W,H", [("micro", 256, 2048, 2048), ("mix", 160, 1001, 1003), ("low", 40, 4096, 4096),
                                        ("noise", 12, 2536, 2048), ("micro", 24, 4096, 4096), ("micro", 48, 2560, 2160),
                                        ("mix", 96, 1280, 1024)])
def test_baseline_configs_device_resident_at_scale(codec, kind, N, W, H):
    """BASELINE configs 2-4 (+ the reference's own 2536x2048 noise frame, + micro at 4096^2) as the bench
    runs them -- generated, encoded and decoded in HBM, hundreds of frames per launch so the persistent
    kernels, the frame-interleaved tickets and the look-back chains run at depth.  Size-independent
    properties on the whole batch (decode(encode(x)) == x on the device, every status 0, record sizes
    consistent with the depth planes) and byte equality of EVERY record with the unmodified reference."""
    px = W * H
    wh = ((W + 7) // 8) * ((H + 7) // 8)
    stride = codec.slot_stride(W, H)
    cap = codec.stream_bound(W, H, N)
    d_fr, d_dec, d_out = codec.device_alloc(N * px), codec.device_alloc(N * px), codec.device_alloc(cap + 64)
    d_off, d_sz, d_st, d_ix = codec.device_alloc(8 * N), codec.device_alloc(8 * N), codec.device_alloc(4 * N), codec.device_alloc(8 * N)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    try:
        synth.gen_frames_device(kind, N, W, H, d_fr, seed=42, f0=0)
        codec.encode_device(d_fr, W, H, 7, N, d_out + delta, cap, d_off, d_sz)
        codec.decode_device(d_out + delta, cap, d_off, W, H, N, d_dec, d_st, d_ix)
        sizes = codec.d2h(d_sz, 8 * N, np.uint64)
        assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
        assert codec.d2h(d_ix, 8 * N, np.uint64).tolist() == list(range(7, 7 + N))
        assert codec.d2h(d_off, 8 * N, np.uint64).tolist() == [i * stride for i in range(N)]
        # whole-batch round trip, compared frame by frame to bound host memory
        for i in range(N):
            a, b = codec.d2h(d_fr + i * px, px), codec.d2h(d_dec + i * px, px)
            assert (a == b).all(), i
        # EVERY record against the unmodified reference (its threaded batch encoder where oracle/_ref is built, else
        # sampled records against the port), and size == 32 + 2wh + 8 * sum(depth plane)
        import oracle
        if oracle.ref is not None:
            step = max(1, (128 << 20) // px)
            for a in range(0, N, step):
                b = min(N, a + step)
                fr = codec.d2h(d_fr + a * px, (b - a) * px).reshape(b - a, H, W)
                _, want, wsz = oracle.ref_encode_mt(fr, os.cpu_count() or 4, 1)      # writes frame index i - a
                assert (wsz.astype(np.int64) == sizes[a:b].astype(np.int64)).all(), (a, b)
                for i in range(a, b):
                    n = int(sizes[i])
                    rec = codec.d2h(d_out + delta + i * stride, n)
                    assert rec[:4].tobytes() == want[i - a, :4].tobytes() and rec[12:].tobytes() == want[i - a, 12:n].tobytes(), i
                    assert int(rec[4:12].view(np.uint64)[0]) == 7 + i, i
                    assert n == 32 + 2 * wh + 8 * int(rec[24:24 + wh].astype(np.int64).sum())
        else:
            for i in sorted({0, 1, N // 2, N - 1}):
                rec = codec.d2h(d_out + delta + i * stride, int(sizes[i]))
                fr = codec.d2h(d_fr + i * px, px).reshape(1, H, W)
                want, wsz = ORA.pack_frames(fr, 7 + i)
                assert int(sizes[i]) == int(wsz[0]) and (rec == want).all(), i
                assert int(sizes[i]) == 32 + 2 * wh + 8 * int(rec[24:24 + wh].astype(np.int64).sum())
    finally:
        for p in (d_fr, d_dec, d_out, d_off, d_sz, d_st, d_ix):
            codec.device_free(p)


@pytest.mark.parametrize("W,H,N", [(1001, 1003, 3), (13, 9, 5), (7, 5, 4), (2048, 16, 2), (264, 24, 3), (4100, 12, 2), (1004, 40, 3),
                                   (1006, 24, 2), (259, 16, 3), (2304, 24, 2), (1280, 40, 3)])
def test_decoder_and_encoder_never_write_outside_their_buffers(codec, odd_decode, W, H, N):
    """guard bytes around the decoder's pixel output and the encoder's slots, at every misalignment of
    the output base: the generic store path assembles aligned 8-byte words across lanes, so a frame's
    first/last bytes share words with the neighbouring memory and must be written with narrow stores"""
    px = W * H
    fr = synth.gen_frames("mix", N, W, H, f0=11)
    want, sizes = ORA.pack_frames(fr, 0)
    stride = codec.slot_stride(W, H)
    G = 64
    d_fr = codec.device_alloc(N * px + 2 * G + 16)
    d_out = codec.device_alloc(N * stride + 2 * G + 16)
    d_dec = codec.device_alloc(N * px + 2 * G + 16)
    d_off, d_sz, d_st = codec.device_alloc(8 * N), codec.device_alloc(8 * N), codec.device_alloc(4 * N)
    try:
        for shift in (0, 1, 3, 4, 7, 8, 13):
            codec.h2d(d_fr, np.full(N * px + 2 * G + 16, 0x5A, dtype=np.uint8))
            codec.h2d(d_fr + G + shift, fr)
            codec.h2d(d_out, np.full(N * stride + 2 * G + 16, 0xEE, dtype=np.uint8))
            codec.encode_device(d_fr + G + shift, W, H, 0, N, d_out + G + shift, N * stride, d_off, d_sz)
            out = codec.d2h(d_out, N * stride + 2 * G + 16)
            assert (out[:G + shift] == 0xEE).all() and (out[G + shift + N * stride:] == 0xEE).all(), shift
            szs = codec.d2h(d_sz, 8 * N, np.uint64)
            pos = 0
            for i in range(N):
                rec = out[G + shift + i * stride: G + shift + i * stride + int(szs[i])]
                assert (rec == want[pos:pos + int(szs[i])]).all(), (shift, i)
                assert (out[G + shift + i * stride + int(szs[i]): G + shift + (i + 1) * stride] == 0xEE).all(), (shift, i)
                pos += int(szs[i])
            for dshift in (shift, (shift * 5 + 2) % 16):
                codec.h2d(d_dec, np.full(N * px + 2 * G + 16, 0xA7, dtype=np.uint8))
                codec.decode_device(d_out + G + shift, N * stride, d_off, W, H, N, d_dec + G + dshift, d_st, None)
                dec = codec.d2h(d_dec, N * px + 2 * G + 16)
                assert (codec.d2h(d_st, 4 * N, np.uint32) == 0).all()
                assert (dec[G + dshift:G + dshift + N * px].reshape(fr.shape) == fr).all(), (shift, dshift)
                assert (dec[:G + dshift] == 0xA7).all() and (dec[G + dshift + N * px:] == 0xA7).all(), (shift, dshift)
    finally:
        for p in (d_fr, d_out, d_dec, d_off, d_sz, d_st):
            codec.device_free(p)


def test_sharded_host_api_across_all_visible_devices():
    """SURVEY 8e on real hardware: one context per visible GPU, a batch cut into many chunk ranges dealt
    round-robin over the DEVICES; the whole stream must hash like the reference's, decode must return the
    source frames.  Skipped on a one-GPU box (test_sharded_* then put all contexts on device 0)."""
    ndev = pkg.load().dbde_b200_device_count()
    if ndev < 2:
        pytest.skip("one visible GPU")
    group = [pkg.Codec(i) for i in range(ndev)]
    try:
        for kind, W, H, n, chunk in [("micro", 1024, 512, 16 * ndev + 5, 4), ("mix", 1001, 1003, 6 * ndev + 1, 2),
                                     ("low", 4096, 256, 3 * ndev, 1)]:
            fr = synth.gen_frames(kind, n, W, H)
            want, sizes = ORA.pack_frames(fr, 9000)
            group[0].set_chunk_frames(chunk)
            try:
                stream, offs = pkg.encode_host_sharded(group, fr, 9000)
            finally:
                group[0].set_chunk_frames(0)
            assert len(stream) == len(want) and sha(stream) == sha(want), (kind, ndev)
            assert offs.tolist() == [0] + np.cumsum(sizes).tolist()
            dec, status, index = pkg.decode_host_sharded(group, stream, offs[:-1], W, H)
            assert (status == 0).all() and index.tolist() == list(range(9000, 9000 + n)) and sha(dec) == sha(fr)
    finally:
        for c in group:
            c.close()


def test_walker_struct_bookkeeping_mirrors_the_reference(dropin):
    """dbde_util.h:40-47: after each dbde_walk_a_file the reference leaves `i` just past the record it
    handed out and `n` at the end of the buffer's good data, never touches `frames`, and exports
    dbde_advance_file_buffer (dbde_util.cpp:394-406: false only when reading the file failed)."""
    import ctypes as C
    W, H, N = 136, 72, 9
    fr = synth.gen_frames("mix", N, W, H)
    stream, sizes = ORA.pack_frames(fr, 0)
    ends = np.cumsum(sizes).tolist()
    adv = getattr(dropin.lib, "_Z24dbde_advance_file_bufferR16dbde_file_walker")
    adv.restype = C.c_bool
    with tempfile.NamedTemporaryFile(suffix=".dbde", delete=False) as f:
        f.write(ORA.pack_video_header(3, H, W, 30.0).tobytes())
        f.write(stream.tobytes())
        path = f.name
    try:
        w, vh = dropin.walk_open(path, N + 3)            # the whole file fits in one buffer: i == record ends
        assert adv(C.byref(w)) is True
        for k in range(N):
            hdr, img = dropin.walk_next(w)
            assert hdr == (2, k, 0) and (img == fr[k]).all()
            assert w.i == ends[k] and w.n == len(stream) and w.i <= w.n <= w.N and w.frames == 0
        assert dropin.walk_next(w) is None
        dropin.walk_close(w)
        w, vh = dropin.walk_open(path, 2)                # small buffer: the invariants still hold
        seen = 0
        while True:
            r = dropin.walk_next(w)
            if r is None:
                break
            assert (r[1] == fr[seen]).all() and 0 < w.i <= w.n <= w.N and w.frames == 0
            seen += 1
        assert seen == N
        dropin.walk_close(w)
        assert adv(C.byref(w)) is False                  # a closed walker
    finally:
        os.unlink(path)


def test_file_api_follows_the_hz_as_integer_variant(codec, dropin):
    """one library, one container: a file written by dbde_b200_writer_* is read by the drop-in walker and
    by dbde_b200_reader_* under both settings of DBDE_HZ_AS_INTEGER (dbde_util.cpp:203-204,352-353), and
    its header bytes are the reference's (the variant build of the reference for the integer form)."""
    fr = synth.gen_frames("micro", 5, 200, 96)
    for hz_int, ora in ((False, ORA), (True, oracle.best_variants())):
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "v.dbde")
            try:
                pkg.set_format_variants(False, hz_int)
                pkg.write_file(codec, path, fr, hz=29.97, first_index=3, batch=2)
                head = np.frombuffer(open(path, "rb").read(28), dtype=np.uint8)
                assert (head == ora.pack_video_header(3, 96, 200, 29.97)).all(), hz_int
                vh, frames = dropin.walk_file(path, 3)
                assert vh == (3, 96, 200, 30.0 if hz_int else 29.97) and len(frames) == 5
                assert all((img == fr[i]).all() and hdr == (2, 3 + i, 0) for i, (hdr, img) in enumerate(frames))
                (W, H, hz), got, idx, st = pkg.read_file(codec, path, batch=2)
                assert (W, H, hz) == (200, 96, 30.0 if hz_int else 29.97) and (got == fr).all() and (st == 0).all()
            finally:
                pkg.set_format_variants(False, False)


def test_drop_in_functions_from_many_short_lived_threads(dropin):
    """the reference's functions are re-entrant (SURVEY 8b), so callers use them from threads that come and go:
    three waves of eight threads, each packing and unpacking its own frames through the C++ symbols on numpy
    (pageable) buffers -- the copy pool's helping waits, the completion flags and the context pool (a thread that
    ends parks its GPU context, the next wave picks the warm ones up) under real CUDA traffic; every record must be
    the reference's and every image must come back"""
    import threading
    W, H = 520, 264
    errors = []

    def worker(seed):
        try:
            rng = np.random.default_rng(seed)
            for i in range(4):
                img = rand_frame(rng, W, H, ["classes", "noise", "flat"][(seed + i) % 3])
                rec = dropin.pack_frame(1000 * seed + i, img)
                want, _ = ORA.pack_frames(img[None], 1000 * seed + i)
                assert (rec == want).all(), (seed, i)
                used, (u64s, index, _), back = dropin.unpack_frame(rec, W, H)
                assert used == len(rec) and u64s == 2 and index == 1000 * seed + i and (back == img).all(), (seed, i)
        except Exception as e:           # noqa: BLE001 -- reported by the main thread
            errors.append(repr(e))

    for wave in range(3):
        ts = [threading.Thread(target=worker, args=(8 * wave + t,)) for t in range(8)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
    assert not errors, errors[:3]
