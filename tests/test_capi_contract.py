"""The argument contract of every codec entry point, as one table: each of the 24 extern "C" encode, decode, validate,
region, crop and binned functions (8-bit and DBDE16, device and host form) crossed with every class of bad argument
that applies to it.  Every rejection returns the exact code with nothing queued (the launch count does not move), an
empty batch returns 0 without reading a buffer, and the inputs accepted that a stricter reading might reject (odd
pointers to the DBDE16 host forms that copy through staging) are pinned as accepted, with their results checked."""
import ctypes as C
import importlib

import numpy as np
import pytest

pkg = importlib.import_module("dbce-video-cpp_b200")
E_INVALID, E_CAPACITY = -1, -3
W, H, N = 40, 24, 2
CORNERS = np.array([[1, 2], [3, 4]], dtype=np.int32)
CROP = dict(corners=None, ncrops=2, per_frame=0, cw=4, ch=3, pad=0)
CAP = 1 << 20

# name -> (encode?, DBDE16?, device form?, output form)
ENTRIES = {}
for _u16 in (False, True):
    for _dev in (True, False):
        _e, _d, _side = ("encode16" if _u16 else "encode"), ("decode16" if _u16 else "decode"), ("device" if _dev else "host")
        ENTRIES["%s_%s" % (_e, _side)] = (True, _u16, _dev, "full")
        ENTRIES["%s_crops_%s" % (_e, _side)] = (True, _u16, _dev, "crops")
        ENTRIES["%s_%s" % (_d, _side)] = (False, _u16, _dev, "full")
        ENTRIES["%s_crops_%s" % (_d, _side)] = (False, _u16, _dev, "crops")
        ENTRIES["%s_binned_%s" % (_d, _side)] = (False, _u16, _dev, "binned")
        if not _u16:
            ENTRIES["validate_" + _side] = (False, False, _dev, "validate")
            ENTRIES["decode_roi_" + _side] = (False, False, _dev, "roi")

POINTERS = ("ctx", "frames", "stream", "offs", "corners", "out", "eoffs", "sizes", "dout", "status", "index", "st")
TYPES = dict({p: C.c_void_p for p in POINTERS}, nbytes=C.c_size_t, cap=C.c_size_t, stride=C.c_size_t, first=C.c_uint64)


def params(name):
    """the entry point's parameters, in order"""
    enc, _, dev, form = ENTRIES[name]
    sub = {"full": [], "validate": [], "roi": ["x0", "y0", "rw", "rh"], "crops": list(CROP), "binned": ["factor"]}[form]
    if enc:
        return ["ctx", "frames", "W", "H", "first", "n"] + sub + ["out", "cap"] + (["stride", "eoffs", "sizes", "st"] if dev else ["eoffs"])
    return (["ctx", "stream", "nbytes", "offs", "W", "H", "n"] + sub + ([] if form == "validate" else ["dout"]) + ["status", "index"] +
            (["st"] if dev else []))


def test_table_covers_every_codec_entry_point():
    """every extern "C" encode / decode / validate function but the sharded ones has its row"""
    codec_fns = {s[len("dbde_b200_"):] for s in pkg.C_SYMBOLS
                 if s.split("_")[2].startswith(("encode", "decode", "validate")) and not s.endswith("sharded")}
    assert codec_fns == set(ENTRIES) and len(ENTRIES) == 24


@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    yield c
    c.close()


@pytest.fixture(scope="module")
def env(codec):
    """valid arguments for every (DBDE16?, device?) pair, plus the expected encoder output"""
    rng = np.random.default_rng(2026)
    d_ptrs, keep, out = [], [], {}

    def dev(arr=None, nbytes=None):
        p = codec.device_alloc(arr.nbytes if arr is not None else nbytes)
        d_ptrs.append(p)
        if arr is not None:
            codec.h2d(p, arr)
        return p

    def host(arr):
        keep.append(arr)
        return arr.ctypes.data

    for u16 in (False, True):
        frames = rng.integers(0, 4096 if u16 else 256, (N, H, W)).astype(np.uint16 if u16 else np.uint8)
        stream, offs = (codec.encode16_host if u16 else codec.encode_host)(frames, 5)
        crops_stream, _ = (codec.encode16_crops_host if u16 else codec.encode_crops_host)(frames, CORNERS, (4, 3), first_index=5)
        odd = np.zeros(frames.nbytes + 2, np.uint8)
        odd[1:1 + frames.nbytes] = frames.view(np.uint8).ravel()
        common = dict(W=W, H=H, n=N, first=5, x0=8, y0=4, rw=16, rh=8, factor=2, index=None, st=None, stride=0, cap=CAP, **CROP)
        out[u16, True] = dict(common, ctx=codec.h.value, frames=dev(frames), stream=dev(stream), nbytes=stream.nbytes,
                              offs=dev(offs[:N]), corners=dev(CORNERS), out=dev(nbytes=CAP), eoffs=dev(nbytes=512), sizes=dev(nbytes=512),
                              dout=dev(nbytes=CAP), status=dev(nbytes=256))
        h_out, h_eoffs, h_dout = np.zeros(CAP, np.uint8), np.zeros(64, np.uint64), np.zeros(CAP, np.uint8)
        out[u16, False] = dict(common, ctx=codec.h.value, frames=host(frames), stream=host(stream), nbytes=stream.nbytes,
                               offs=host(offs[:N].copy()), corners=host(CORNERS), out=host(h_out), eoffs=host(h_eoffs),
                               dout=host(h_dout), status=host(np.zeros(64, np.uint32)), sizes=None,
                               # what the checks of accepted cases compare with
                               x_frames=frames, x_stream=stream, x_crops_stream=crops_stream, x_odd=host(odd) + 1, x_offs=offs[:N],
                               x_out=h_out, x_eoffs=h_eoffs, x_dout=h_dout)
    yield out
    for p in d_ptrs:
        codec.device_free(p)


def call(codec, name, args):
    fn = getattr(codec.lib, "dbde_b200_" + name)
    return fn(*[TYPES.get(p, C.c_int)(args[p]) for p in params(name)])


def stride(codec, u16, w, h, bound=False):
    fn = "dbde_b200_%s%s" % ("frame_record_bound" if bound else "slot_stride", "16" if u16 else "")
    return int(getattr(codec.lib, fn)(w, h))


def cases(codec, name, a):
    """(what, overrides, expected return code, launch count unchanged?, check or None) for every rejection class that
    applies to the entry point, the empty batch, and the accepted inputs worth pinning"""
    enc, u16, dev, form = ENTRIES[name]
    ps = params(name)
    out = []

    def add(what, want, over, same=True, check=None, also_empty=False):
        out.append((what, over, want, same, check))
        if also_empty:
            out.append((what + ", nframes 0", dict(over, n=0), want, same, check))

    add("valid", 0, {}, same=False)
    add("nframes 0, no buffers", 0, dict({p: None for p in ps if p in POINTERS and p != "ctx"}, n=0))
    add("null context", E_INVALID, dict(ctx=None), also_empty=True)
    required = [p for p in ("frames", "stream", "offs", "corners", "out", "eoffs", "sizes", "dout", "status") if p in ps]
    for p in required:
        add("null " + p, E_INVALID, {p: None})
    for over in (dict(W=0), dict(H=-1), dict(W=1 << 30), dict(W=1 << 16, H=1 << 16), dict(n=-1)):
        add("dims %r" % over, E_INVALID, over)
    if form == "roi":
        for over in (dict(x0=-1), dict(y0=-1), dict(rw=0), dict(rh=-1), dict(x0=W - 15), dict(y0=H - 7), dict(x0=2**31 - 1)):
            add("region %r" % over, E_INVALID, over, also_empty=True)
    if form == "crops":
        for over in (dict(ncrops=0), dict(ncrops=-1), dict(cw=0), dict(ch=-1), dict(per_frame=2), dict(per_frame=-1), dict(pad=-1),
                     dict(pad=65536 if u16 else 256), dict(ncrops=1 << 20, cw=64, ch=64), dict(cw=1 << 16, ch=1 << 16)):
            add("crops %r" % over, E_INVALID, over, also_empty=True)
        add("pad maximum", 0, dict(pad=65535 if u16 else 255), same=False)
    if form == "binned":
        for f in (0, 3, 16, -2):
            add("factor %d" % f, E_INVALID, dict(factor=f), also_empty=True)
        add("factor 1", 0, dict(factor=1), same=False)
    if u16:
        p = "frames" if enc else "dout"
        if dev or (not enc and form != "full"):
            add("odd " + p, E_INVALID, {p: a[p] + 1}, also_empty=True)
        elif enc:
            # the frames are copied into staging first: any address works
            want = a["x_crops_stream"] if form == "crops" else a["x_stream"]
            add("odd frames accepted", 0, dict(frames=a["x_odd"]), same=False,
                check=lambda: np.array_equal(a["x_out"][:want.nbytes], want) and int(a["x_eoffs"][N * (2 if form == "crops" else 1)]) == want.nbytes)
        else:
            # decode16_host copies the frames out of staging: any address works
            nb = a["x_frames"].nbytes
            add("odd output accepted", 0, dict(dout=a["dout"] + 1), same=False,
                check=lambda: np.array_equal(a["x_dout"][1:1 + nb], a["x_frames"].view(np.uint8).ravel()))
    if enc:
        nrec = N * (2 if form == "crops" else 1)
        rw, rh = (4, 3) if form == "crops" else (W, H)
        if dev:
            bound = stride(codec, u16, rw, rh, bound=True)
            add("slot_stride < bound", E_INVALID, dict(stride=bound - 1))
            add("slot_stride < bound and no capacity", E_INVALID, dict(stride=bound - 1, cap=0))
            add("capacity one byte short", E_CAPACITY, dict(cap=nrec * stride(codec, u16, rw, rh) - 1))
            add("capacity one byte short, own slot_stride", E_CAPACITY, dict(stride=bound + 1, cap=nrec * (bound + 1) - 1))
        else:
            # the records' sizes are known only after the kernels ran
            total = (a["x_crops_stream"] if form == "crops" else a["x_stream"]).nbytes
            add("capacity one byte short", E_CAPACITY, dict(cap=total - 1), same=False)
            z = np.full(1, 99, np.uint64)
            add("nframes 0 writes offsets[0]", 0, dict(n=0, eoffs=z.ctypes.data, keep=z), check=lambda: int(z[0]) == 0)
        if form == "crops":
            # a 1 x 1 frame keeps the batch itself legal
            add("nframes * ncrops > 2^31 - 1", E_INVALID, dict(W=1, H=1, n=1 << 16, ncrops=1 << 16, cw=1, ch=1))
    elif not dev:
        o = a["x_offs"]
        desc = np.array([o[1], o[0]], np.uint64)
        add("descending offsets", E_INVALID, dict(offs=desc.ctypes.data, keep=desc))
        add("offsets past the stream", E_INVALID, dict(nbytes=int(o[1]) - 1))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ENTRIES))
def test_argument_contract(codec, env, name):
    enc, u16, dev, form = ENTRIES[name]
    a = env[u16, dev]
    for what, over, want, same, check in cases(codec, name, a):       # `keep`: an array an override points into
        l0 = codec.launches()
        rc = call(codec, name, dict(a, **over))
        assert rc == want, (name, what, rc, codec.lib.dbde_b200_last_error())
        if same:
            assert codec.launches() == l0, (name, what)
        if check is not None:
            assert check(), (name, what)
