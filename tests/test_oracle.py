"""CPU tests: pin the oracle port (oracle/dbde_oracle.c) against the reference's golden vectors
(tests/golden/golden.json, produced by the unmodified reference), against the stored records of the
differential and format-variant comparisons (tests/golden/golden_differential.json) and, when
oracle/_ref is built, differentially against the reference itself."""
import hashlib
import os

import numpy as np
import pytest

import oracle
import synth
from conftest import golden_random_frames, rand_frame

CODECS = [("port", oracle.port)] + ([("ref", oracle.ref)] if oracle.ref is not None else [])
ids = [c[0] for c in CODECS]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint8).tobytes()).hexdigest()


def unhex(s):
    return np.frombuffer(bytes.fromhex(s), dtype=np.uint8)


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_readme_example(golden, name, cd):
    """BASELINE config 1: README 10x10 image (README.md:75-84)."""
    img = np.array(golden["readme"]["image"], dtype=np.uint8)
    enc = cd.pack_image(img)
    assert enc.tobytes().hex() == golden["readme"]["pack_image"]
    assert len(enc) == 92
    # planes and words 1-6 exactly as printed in README.md:173-187
    assert enc[:4].tolist() == [4, 0, 0, 0] and enc[4:8].tolist() == [4, 2, 3, 0]
    assert enc[12:16].tolist() == [0x13, 0x18, 0x1C, 0x1A] and enc[16:20].tolist() == [9, 0, 0, 0]
    words = enc[20:].view("<u8")
    assert ["%016X" % int(w) for w in words[:6]] == golden["readme"]["words_1_6_readme"]
    n, dec = cd.unpack_image(enc, 10, 10)
    assert n == 92 and (dec == img).all()
    assert cd.pack_frame(7, img).tobytes().hex() == golden["readme"]["pack_frame_index7"]


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_kat_8x16_both_directions(golden, name, cd):
    """The reference's own known-answer test, dbde_util_test.cpp:134-213."""
    img = np.array(golden["kat_8x16"]["image"], dtype=np.uint8).reshape(8, 16)
    stream = np.array(golden["kat_8x16"]["stream"], dtype=np.uint8)
    n, vh = cd.unpack_video_header(stream)
    assert n == 28 and vh == (3, 8, 16, 1.0)
    n, hdr, dec = cd.unpack_frame(stream[28:], 16, 8)
    assert n == 100 and hdr == (2, 1, 0) and (dec == img).all()
    enc = np.concatenate([cd.pack_video_header(3, 8, 16, 1.0), cd.pack_frame(1, img)])
    assert len(enc) == 128 and (enc == stream).all()


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_headers(golden, name, cd):
    assert cd.pack_video_header(3, 10, 10, 30.0).tobytes().hex() == golden["headers"]["video_3_10_10_30hz"]
    # elapsed_ns travels as a double (dbde_util.cpp:186)
    assert cd.pack_frame_header(2, 5, 123456789012345).tobytes().hex() == golden["headers"]["frame_2_5_123456789012345"]
    bad = cd.pack_video_header(4, 1, 1, 1.0)
    assert cd.unpack_video_header(bad)[1][0] == 0xFFFFFFFF


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_small_and_flat(golden, name, cd):
    s = golden["small_3x5"]
    img = np.array(s["image"], dtype=np.uint8)
    enc = cd.pack_image(img)
    assert enc.tobytes().hex() == s["pack_image"] and len(enc) == 46
    n, dec = cd.unpack_image(enc, 3, 5)
    assert n == 46 and (dec == img).all()
    flat = np.full((8, 8), golden["flat_8x8"]["value"], dtype=np.uint8)
    assert cd.pack_image(flat).tobytes().hex() == golden["flat_8x8"]["pack_image"]


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_single_tile_returns(golden, name, cd):
    for t in golden["single_tiles"]:
        tile = np.full((8, 8), t["min"], dtype=np.uint8)
        tile[3, 5] = t["min"] + t["range"]
        tile[7, 7] = t["min"] + t["range"] // 2
        r, pay = cd.pack_8x8(tile)          # also checks nothing is written past 8*depth bytes
        assert r == t["ret"], t
        assert pay.tobytes().hex() == t["payload"]
        assert (r >> 8) == int(t["range"]).bit_length()


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_golden_random_frames(golden, name, cd):
    for c, img in golden_random_frames(golden):
        assert sha(img) == c["image_sha256"], "rng drifted; regenerate golden"
        rec = cd.pack_frame(c["index"], img)
        assert len(rec) == c["record_len"] and sha(rec) == c["record_sha256"], (c["W"], c["H"])
        if "record" in c:
            assert rec.tobytes().hex() == c["record"]
        n, hdr, dec = cd.unpack_frame(rec, c["W"], c["H"])
        assert n == len(rec) and hdr == (2, c["index"], 0) and (dec == img).all()


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_golden_synthetic(golden, name, cd):
    for s in golden["synthetic"]:
        if s["W"] * s["H"] * s["n"] > 1100000 and name == "port":
            continue  # the bit-loop port is slow; the big case is covered by the reference codec
        fr = synth.gen_frames(s["kind"], s["n"], s["W"], s["H"], seed=s["seed"])
        assert sha(fr) == s["frames_sha256"]
        stream, sizes = cd.pack_frames(fr, 0)
        assert [int(x) for x in sizes] == s["sizes"] and sha(stream) == s["stream_sha256"]


def test_micro_histogram_matches_survey(golden):
    """SURVEY.md 8d-2: depth 0 12.1 %, depth 3 80.3 %, depth 4 4.3 % on micro-2048^2."""
    s = [x for x in golden["synthetic"] if x["kind"] == "micro" and x["W"] == 2048][0]
    h = np.array(s["depth_hist_frame0"]) / 65536.0
    assert abs(h[0] - 0.121) < 0.005 and abs(h[3] - 0.803) < 0.005 and abs(h[4] - 0.043) < 0.005


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_partial_tiles_clamp(name, cd):
    """Padding is clamp-to-edge and the padded values ARE packed (README.md:131-146)."""
    rng = np.random.default_rng(1)
    for rm in range(1, 9):
        for dm in range(1, 9):
            if rm == 8 and dm == 8:
                continue
            tile = rng.integers(0, 256, (8, 8), dtype=np.uint8)
            full = tile.copy()
            full[:, rm:] = full[:, rm - 1:rm]
            full[dm:, :] = full[dm - 1:dm, :]
            r1, p1 = cd.pack_8x8_partial(tile, rm, dm)
            r2, p2 = cd.pack_8x8(full)
            assert r1 == r2 and (p1 == p2).all()


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_invalid_streams_rejected(name, cd):
    """dbde_util.cpp:296,299,303: nb != wh, nm != wh, sum(depth) != n64 -> 0, image untouched."""
    rng = np.random.default_rng(2)
    img = rng.integers(0, 64, (16, 24), dtype=np.uint8)
    enc = cd.pack_image(img)
    wh = 6
    for pos, delta in [(0, 1), (4 + wh, 1), (8 + 2 * wh, 1), (4, 1)]:
        bad = enc.copy()
        bad[pos] = bad[pos] + delta
        n, dec = cd.unpack_image(bad, 24, 16, fill=0xCD)
        assert n == 0 and (dec == 0xCD).all()
    rec = cd.pack_frame(3, img)
    bad = rec.copy(); bad[20] += 1
    n, hdr, dec = cd.unpack_frame(bad, 24, 16)
    assert n == 20 and hdr[0] == 0xFFFFFFFF and hdr[1] == 3   # pointer left just after the header (:342-343)
    bad = rec.copy(); bad[0] = 7
    n, hdr, dec = cd.unpack_frame(bad, 24, 16)
    assert hdr[0] == 0xFFFFFFFF and n == len(rec)             # header parse always advances (:330-337)


def differential_golden():
    """tests/golden/make_golden_differential.py (the inputs) and golden_differential.json (the stored records)"""
    import importlib.util
    import json
    gdir = os.path.join(os.path.dirname(__file__), "golden")
    spec = importlib.util.spec_from_file_location("make_golden_differential", os.path.join(gdir, "make_golden_differential.py"))
    mg = importlib.util.module_from_spec(spec); spec.loader.exec_module(mg)
    return mg, json.load(open(os.path.join(gdir, "golden_differential.json")))


def test_port_vs_reference_differential():
    """Random sizes incl. W<8, H<8, odd; all depth classes; both directions: every record against the stored
    vectors, and against the reference itself where oracle/_ref is built."""
    mg, gold = differential_golden()
    frames = mg.differential_frames()
    assert len(frames) == len(gold["differential"]) == 60
    for (i, W, H, img), c in zip(frames, gold["differential"]):
        assert (W, H, sha(img)) == (c["W"], c["H"], c["image_sha256"]), "rng drifted; regenerate golden"
        a = oracle.port.pack_frame(i, img)
        assert len(a) == c["record_len"] and sha(a) == c["record_sha256"], (W, H)
        n1, h1, d1 = oracle.port.unpack_frame(a, W, H)
        assert n1 == len(a) and h1 == (2, i, 0) and (d1 == img).all()
        if oracle.ref is not None:
            b = oracle.ref.pack_frame(i, img)
            assert len(a) == len(b) and (a == b).all(), (W, H)
            n2, h2, d2 = oracle.ref.unpack_frame(b, W, H)
            assert n1 == n2 and h1 == h2 and (d1 == d2).all()


@pytest.mark.parametrize("name,cd", CODECS, ids=ids)
def test_depth8_stores_pixel_minus_min(name, cd):
    """SURVEY 0.4: depth 8 stores (p - min) mod 256, not the raw pixel."""
    tile = (np.arange(64).reshape(8, 8) * 3 + 50).astype(np.uint8)      # range 189 -> depth 8, min 50
    r, pay = cd.pack_8x8(tile)
    assert r == 0x832 and pay[:3].tolist() == [0, 3, 6] and len(pay) == 64


# ------------------------------------------------------------------ the reference's compile-time variants
def test_port_variants_match_the_reference_built_with_both_macros():
    """DBDE_INVERT_ENDIAN + DBDE_HZ_AS_INTEGER (dbde_util.cpp:15-19,203-204,352-353): the port's run-time
    switches against the stored vectors (tests/golden/golden_differential.json) and against the unmodified
    reference compiled with the two macros where oracle/_ref is built."""
    mg, gold = differential_golden()
    pv, rv = oracle.port_variants(), oracle.ref_variants
    cases = mg.variant_frames()
    assert len(cases) == len(gold["variants"]["cases"]) == 15
    differs = False
    for (W, H, style, fr), c in zip(cases, gold["variants"]["cases"]):
        assert (W, H, style, sha(fr)) == (c["W"], c["H"], c["style"], c["frames_sha256"]), "rng drifted; regenerate golden"
        a, sa = pv.pack_frames(fr, 5)
        assert [int(s) for s in sa] == c["sizes"] and sha(a) == c["stream_sha256"], (W, H, style)
        if rv is not None:
            b, sb = rv.pack_frames(fr, 5)
            assert list(sa) == list(sb) and (a == b).all(), (W, H, style)
            assert (rv.unpack_frames(a, W, H, 2)[0] == fr).all()
        differs |= not np.array_equal(a, oracle.port.pack_frames(fr, 5)[0])
        assert (pv.unpack_frames(a, W, H, 2)[0] == fr).all()
    assert differs, "the variant must change the payload bytes"
    hv = pv.pack_video_header(3, 480, 640, 29.97)
    assert hv.tobytes().hex() == gold["variants"]["video_header"]["hex"] and hv[20:].tolist() == [30, 0, 0, 0, 0, 0, 0, 0]
    assert pv.unpack_video_header(hv) == (28, (3, 480, 640, 30.0))
    if rv is not None:
        assert (rv.pack_video_header(3, 480, 640, 29.97) == hv).all() and rv.unpack_video_header(hv) == (28, (3, 480, 640, 30.0))


# ------------------------------------------------------------------ DBDE16 (SURVEY 8 f-4; not in the reference)
def test_dbde16_embeds_the_8_bit_codec_and_round_trips():
    """The 16-bit extension has no reference implementation ("parity unpinned"); what pins its definition:
    a frame whose pixels fit in 8 bits must get the reference-pinned 8-bit codec's depth plane, minima and
    U64 words (only the minimum plane is two bytes wide), true 16-bit frames must round-trip, and a
    hand-computed tile must give the expected words."""
    o16, o8 = oracle.port16, oracle.best()
    rng = np.random.default_rng(3)
    for W, H in [(8, 8), (10, 10), (17, 23), (64, 40), (1001, 24)]:
        wh = ((W + 7) // 8) * ((H + 7) // 8)
        for style in ("classes", "noise", "flat"):
            fr8 = np.stack([rand_frame(rng, W, H, style) for _ in range(2)])
            a, sa = o8.pack_frames(fr8, 5)
            b, sb = o16.pack_frames(fr8.astype(np.uint16), 5)
            pa = pb = 0
            for i in range(2):
                ra, rb = a[pa:pa + int(sa[i])], b[pb:pb + int(sb[i])]
                assert int(sb[i]) == int(sa[i]) + wh
                assert (ra[:24 + wh] == rb[:24 + wh]).all()                      # frame header, nb, depth plane
                assert int.from_bytes(rb[24 + wh:28 + wh].tobytes(), "little") == 2 * wh
                assert (rb[28 + wh:28 + 3 * wh].view(np.uint16) == ra[28 + wh:28 + 2 * wh]).all()
                assert (ra[28 + 2 * wh:] == rb[28 + 3 * wh:]).all()              # n64 and every word
                n, hdr, img = o16.unpack_frame(rb, W, H)
                assert n == len(rb) and hdr == (2, 5 + i, 0) and (img == fr8[i]).all()
                pa += int(sa[i]); pb += int(sb[i])
    fr = rng.integers(0, 65536, (3, 37, 53), dtype=np.uint16)
    s, sz = o16.pack_frames(fr, 0)
    off = 0
    for i in range(3):
        n, hdr, img = o16.unpack_frame(s[off:off + int(sz[i])], 53, 37)
        assert hdr[0] == 2 and (img == fr[i]).all()
        off += n
    # one tile by hand: min 1000, values 1000 + (i % 4) * 300 -> range 900 -> depth 10; pixel i at bits [10 i, 10 i + 10)
    tile = (1000 + (np.arange(64) % 4) * 300).astype(np.uint16).reshape(1, 8, 8)
    s, sz = o16.pack_frames(tile, 0)
    assert s[24] == 10 and int.from_bytes(s[29:31].tobytes(), "little") == 1000 and int(sz[0]) == 32 + 3 + 80
    bits = 0
    for i in range(64):
        bits |= int((i % 4) * 300) << (10 * i)
    assert s[35:115].tobytes() == bits.to_bytes(80, "little")
    # rejects: a damaged minimum-plane length, a depth above 16
    bad = s.copy(); bad[25] ^= 1
    assert o16.unpack_frame(bad, 8, 8)[1][0] == 0xFFFFFFFF
    bad = s.copy(); bad[24] = 17
    assert o16.unpack_frame(bad, 8, 8)[1][0] == 0xFFFFFFFF


def test_dbde16_frozen_fixtures():
    """tests/golden/golden16.json freezes the extension's bytes (made by tests/golden/make_golden16.py from the
    oracle's definition when DBDE16 was introduced): the format cannot drift silently"""
    import json
    sys_path = os.path.join(os.path.dirname(__file__), "golden")
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden16", os.path.join(sys_path, "make_golden16.py"))
    mg = importlib.util.module_from_spec(spec); spec.loader.exec_module(mg)
    gold = json.load(open(os.path.join(sys_path, "golden16.json")))
    for c in gold["cases"]:
        fr = mg.frames16(c)
        assert hashlib.sha256(fr.tobytes()).hexdigest() == c["frames_sha256"]
        stream, sizes = oracle.port16.pack_frames(fr, 11)
        assert [int(x) for x in sizes] == c["sizes"]
        assert hashlib.sha256(stream.tobytes()).hexdigest() == c["stream_sha256"]
        if "stream_hex" in c:
            assert stream.tobytes().hex() == c["stream_hex"]
