"""Every codec kernel past 32-bit extents: frames at the size limit, batches and outputs over 4 GiB, more than 2^32 crop
tasks, host buffers over 4 GiB, and calls queued on streams of their own.

The kernels mix 32-bit and 64-bit index arithmetic: in-frame pixel and tile offsets fit 32 bits because a frame has at
most 2^31 - 1 pixels and 0x0FFFFFFF tiles (dims_ok, dbde_capi.cu), while frame bases, record offsets, slot offsets,
crop outputs and task numbers do not.  A narrowing of one of the latter passes every test that stays below 2^32, so
the cases here are chosen to cross those boundaries, and a CPU test checks from the shapes that each case really
crosses the boundary it is there for.

The references are the oracle for records and plain integer gathers and sums for everything else.  A record of a
frame at the size limit is assembled from the oracle's records of the frame's bands (tiles are independent and stored
in raster order), which bounds host memory and lets the bands run on threads; a CPU test pins the assembler against
whole-frame oracle records.  The GPU tests generate their frames on the device on a non-blocking stream, queue the
codec calls on that stream without a synchronise in between, and read results after synchronising only that stream."""
import ctypes as C
import importlib
import os
import resource
import struct
from collections import namedtuple
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import oracle
import synth

pkg = importlib.import_module("dbce-video-cpp_b200")
ORA = oracle.best()
FIRST = 1000
THREADS = os.cpu_count() or 1
INT32_MAX = 0x7FFFFFFF
E_INVALID = -1
TILE_CAP = 0x0FFFFFFF          # dims_ok: tiles per frame
PIXEL_CAP = 0x7FFFFFFF         # dims_ok: pixels per frame


# ------------------------------------------------------------------ sizes, mirrored from dbde_record.h and dbde_capi.cu
def tiles(W, H):
    return -(-W // 8), -(-H // 8)


def record_bound(W, H, mb):
    """rec_bound: every tile at the full depth of 8 * mb bits"""
    w, h = tiles(W, H)
    return 32 + (1 + mb) * w * h + 64 * mb * w * h


def slot_stride(W, H, mb):
    return (record_bound(W, H, mb) + 15) // 16 * 16


def straddler(fbytes, row_bytes, base, boundary):
    """the frame of a batch at `base` whose bytes cross `boundary`, with the boundary inside a row (None: it falls on a
    frame start, or between two rows)"""
    f, rem = divmod(boundary - base, fbytes)
    return f if rem and rem % row_bytes else None


# ------------------------------------------------------------------ the case table
# A: frames at the size limit (mb: bytes per pixel, 1 = 8-bit, 2 = DBDE16; kind: the content)
Limit = namedtuple("Limit", "name mb W H kind bins")
LIMITS = [
    Limit("A1", 1, 46336, 46336, "mix", (2, 8)),
    Limit("A2", 1, 46337, 46341, "mix", (8,)),
    Limit("A3", 1, 1, 2147483640, "low", (8,)),
    Limit("A4", 1, 2147483640, 1, "low", (8,)),
    Limit("A5", 2, 46336, 46336, "noise", (2, 8)),
    Limit("A6", 2, 46337, 46341, "depths", (8,)),
]
# B: batches past 2^32 bytes, of noise, so that the host forms' packed streams pass 2^32 as well.  fbase / obase: the
# frame and output buffers' offsets from a 16-byte boundary; crop: the crop encoders' crop size, with per-frame corners,
# and the slot stride that puts their slot area past 4 GiB
Batch = namedtuple("Batch", "name mb W H N fbase obase crop crop_stride")
BATCHES = [
    Batch("B1", 1, 1001, 1003, 4300, 3, 5, (256, 200), 1 << 20),
    Batch("B2", 1, 2560, 2160, 800, 0, 0, None, 0),
    Batch("B3", 2, 2048, 2048, 520, 0, 0, None, 0),
    Batch("B4", 2, 1001, 1003, 2150, 0, 0, (256, 200), 2 << 20),
]
# C: crop task counts past 2^32 -- nframes frames of 64 x 64, 2^27 shared 1 x 1 crops (one warp task each)
Tasks = namedtuple("Tasks", "name mb N W H ncrops")
TASKS = [Tasks("C1", 1, 40, 64, 64, 1 << 27), Tasks("C2", 2, 34, 64, 64, 1 << 27)]


def limit_extents(c):
    w, h = tiles(c.W, c.H)
    return {"pixels": c.W * c.H, "tiles": w * h, "frame bytes": c.mb * c.W * c.H,
            "record bound": record_bound(c.W, c.H, c.mb), "far pixel offset": c.W * c.H - 1}


def batch_extents(b):
    fb = b.mb * b.W * b.H
    ext = {"frame bytes": b.fbase + b.N * fb, "stream bytes": b.N * slot_stride(b.W, b.H, b.mb),
           "output bytes": b.obase + b.N * fb, "first damaged record": (b.N - 3) * slot_stride(b.W, b.H, b.mb),
           "straddles 2^31": straddler(fb, b.mb * b.W, b.fbase, 1 << 31),
           "straddles 2^32": straddler(fb, b.mb * b.W, b.fbase, 1 << 32),
           "starts at 2^32": (1 << 32) // fb if (1 << 32) % fb == 0 and (1 << 32) // fb < b.N else None}
    if b.crop:
        ext["crop slot area"] = b.N * b.crop_stride
    return ext


def task_extents(t):
    # a 1 x 1 crop spans at most two tile columns and rows: one row group and one chunk, one warp task per crop
    return {"warp tasks": t.N * t.ncrops, "output bytes": t.mb * t.N * t.ncrops, "corner bytes": 8 * t.ncrops}


# ------------------------------------------------------------------ the band-assembled reference record
def band_ranges(W, H, max_px):
    """pieces of a frame that are frames of their own and whose tiles are consecutive in the raster order: runs of
    whole tile rows or, for a frame one tile high, runs of tile columns -> [(x0, x1, y0, y1, t0, t1)]"""
    w, h = tiles(W, H)
    if h == 1:
        c = max(1, max_px // (8 * H))
        return [(8 * a, min(8 * (a + c), W), 0, H, a, min(a + c, w)) for a in range(0, w, c)]
    r = max(1, max_px // (8 * W))
    return [(0, W, 8 * a, min(8 * (a + r), H), a * w, min(a + r, h) * w) for a in range(0, h, r)]


def pack_one(img, mb, index):
    """the oracle's record of one frame"""
    if mb == 1:
        return ORA.pack_frame(index, img)
    return oracle.port16.pack_frames(img[None], index)[0]


def record_pieces(W, H, mb, index, fetch, max_px=1 << 24, threads=min(THREADS, 32)):
    """The record of a W x H frame as (byte offset, bytes) pieces that cover it exactly: the fixed header, then for each
    band its depth plane, its minimum plane and its words at their places, then the two counts.  fetch(x0, x1, y0, y1)
    -> the band's pixels.  The bands are encoded by the oracle on `threads` threads, a group at a time."""
    w, h = tiles(W, H)
    wh = w * h
    words = 32 + (1 + mb) * wh
    n64 = 0
    head = None
    bands = band_ranges(W, H, max_px)

    def one(b):
        x0, x1, y0, y1, _, _ = b
        return pack_one(fetch(x0, x1, y0, y1), mb, index)

    with ThreadPoolExecutor(max(1, threads)) as ex:
        for g in range(0, len(bands), threads):
            group = bands[g:g + threads]
            for (_, _, _, _, t0, t1), rec in zip(group, ex.map(one, group)):
                bw = t1 - t0
                k = int(np.frombuffer(rec[28 + (1 + mb) * bw:32 + (1 + mb) * bw].tobytes(), "<i4")[0])
                assert len(rec) == 32 + (1 + mb) * bw + 8 * k
                if head is None:
                    head = rec[:20]
                yield 24 + t0, rec[24:24 + bw]
                yield 28 + wh + mb * t0, rec[28 + bw:28 + bw + mb * bw]
                yield words + 8 * n64, rec[32 + (1 + mb) * bw:]
                n64 += k
    yield 0, np.concatenate([head, np.frombuffer(struct.pack("<i", wh), np.uint8)])
    yield 24 + wh, np.frombuffer(struct.pack("<i", mb * wh), np.uint8)
    yield 28 + (1 + mb) * wh, np.frombuffer(struct.pack("<i", n64), np.uint8)


def assemble(W, H, mb, index, img, max_px, threads=2):
    """the whole record from record_pieces, for frames that fit in host memory"""
    pieces = list(record_pieces(W, H, mb, index, lambda x0, x1, y0, y1: img[y0:y1, x0:x1], max_px, threads))
    out = np.full(max(o + len(p) for o, p in pieces), 0xEE, dtype=np.uint8)
    covered = 0
    for o, p in pieces:
        out[o:o + len(p)] = p
        covered += len(p)
    assert covered == len(out)
    return out


def depth_class_frame(rng, W, H, mb):
    """each tile's pixels span 2^k - 1 above a random minimum, k random per tile in 0 .. 8 * mb"""
    w, h = tiles(W, H)
    k = rng.integers(0, 8 * mb + 1, (h, w))
    top = (1 << (8 * mb)) - 1
    rg = (1 << k) - 1
    mn = rng.integers(0, top - rg + 1)
    px = mn[:, :, None, None] + (rng.integers(0, top + 1, (h, w, 8, 8)) & rg[:, :, None, None])
    return px.transpose(0, 2, 1, 3).reshape(8 * h, 8 * w)[:H, :W].astype(np.uint8 if mb == 1 else np.uint16)


# ------------------------------------------------------------------ CPU checks
def test_every_case_crosses_the_boundary_it_is_there_for():
    """the extents each case claims, computed from its shapes; an edit of the table that loses a crossing fails here"""
    a = {c.name: limit_extents(c) for c in LIMITS}
    for n in ("A1", "A2", "A5", "A6"):
        assert a[n]["pixels"] > (1 << 31) - (1 << 24) and a[n]["pixels"] <= PIXEL_CAP, n
    assert a["A2"]["pixels"] == 46337 * 46341 and 46337 % 8 == 1 and 46341 % 8 == 5
    for n in ("A3", "A4"):
        assert a[n]["tiles"] == TILE_CAP, n                             # exactly the tile cap
    assert tiles(1, 2147483640)[1] == TILE_CAP and tiles(2147483640, 1)[0] == TILE_CAP
    assert a["A3"]["record bound"] > 17.7e9                             # the 17.7 GB slot
    assert a["A5"]["record bound"] == 4394691616 > 1 << 32              # the DBDE16 record of the limit frame ends past 2^32
    assert a["A5"]["frame bytes"] < 1 << 32 < a["A5"]["frame bytes"] + (1 << 28)
    # the boundary shapes of the refusal test
    assert tiles(1, 2147483641)[1] > TILE_CAP and tiles(2147483641, 1)[0] > TILE_CAP
    assert 46341 * 46341 > PIXEL_CAP >= 46340 * 46341

    b = {c.name: batch_extents(c) for c in BATCHES}
    for n, e in b.items():
        assert e["frame bytes"] > 1 << 32 and e["stream bytes"] > 1 << 32 and e["output bytes"] > 1 << 32, n
        assert e["first damaged record"] > 1 << 32, n                   # the damaged records lie past 2^32
    assert b["B1"]["straddles 2^31"] == 2138 and b["B1"]["straddles 2^32"] == 4277   # both mid-row
    assert BATCHES[0].fbase % 16 == 3 and BATCHES[0].obase % 16 == 5
    assert b["B3"]["starts at 2^32"] == 512
    assert b["B4"]["straddles 2^32"] == 2138
    for c in BATCHES:
        if c.crop:
            assert b[c.name]["crop slot area"] > 1 << 32, c.name
            assert c.crop_stride >= slot_stride(c.crop[0], c.crop[1], c.mb) and c.crop_stride % 16 == 0
    # B2 runs the linear-partition kernels: 320 tiles a row fill 320 / 512 < 0.9 of two band segments
    w = tiles(2560, 2160)[0]
    assert w > 256 and w % 256 and w / (256 * -(-w // 256)) < 0.9

    for t in TASKS:
        e = task_extents(t)
        assert e["warp tasks"] > 1 << 32 and e["output bytes"] > 1 << 32 and e["corner bytes"] == 1 << 30, t.name


SMALL = [(64, 45), (65, 43), (71, 37), (72, 8), (1, 333), (333, 1), (1, 1), (9, 9)]


@pytest.mark.parametrize("mb", [1, 2], ids=["8bit", "dbde16"])
@pytest.mark.parametrize("W,H", SMALL)
def test_band_assembled_record_equals_the_whole_frame_record(W, H, mb):
    """the assembler against the oracle's record of the whole frame, with bands of one tile row (column), of a few and
    of the whole frame"""
    img = depth_class_frame(np.random.default_rng(W * 131 + H + mb), W, H, mb)
    want = pack_one(img, mb, FIRST + 7)
    for max_px in (1, 8 * max(W, H) * 3, 1 << 30):
        got = assemble(W, H, mb, FIRST + 7, img, max_px)
        assert len(got) == len(want) and (got == want).all(), max_px


def test_band_ranges_tile_the_frame():
    for W, H, max_px in [(46337, 46341, 1 << 26), (1, 2147483640, 1 << 26), (2147483640, 1, 1 << 26), (17, 3, 8)]:
        w, h = tiles(W, H)
        r = band_ranges(W, H, max_px)
        assert r[0][4] == 0 and r[-1][5] == w * h
        assert all(a[5] == b[4] for a, b in zip(r, r[1:]))
        assert all((x1 - x0) * (y1 - y0) <= max(max_px, 64) for x0, x1, y0, y1, _, _ in r)


# ------------------------------------------------------------------ GPU harness
@pytest.fixture(scope="module")
def codec():
    c = pkg.Codec(0)        # raises without a B200: no fallback
    lib = c.lib
    lib.dbde_b200_validate_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                              C.c_void_p, C.c_void_p, C.c_void_p]
    yield c
    c.close()


@pytest.fixture
def S():
    """a non-blocking stream of its own; the device peak of the test is printed, and its memory freed after it"""
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    s = torch.cuda.Stream()
    assert s.cuda_stream != 0
    with torch.cuda.stream(s):
        yield s
    s.synchronize()
    print("\n[extents] device peak %.2f GB (torch allocations), host peak so far %.2f GB" %
          (torch.cuda.max_memory_allocated() / 1e9, resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6))
    torch.cuda.empty_cache()


def need(gb):
    free = torch.cuda.mem_get_info()[0]
    if free < gb * 1e9:
        pytest.skip("needs %.0f GB of free device memory, %.1f GB free" % (gb, free / 1e9))


def dev(nbytes):
    return torch.empty(int(nbytes), dtype=torch.uint8, device="cuda")


def u64(n):
    return torch.zeros(int(n), dtype=torch.int64, device="cuda")


def u32(n):
    return torch.zeros(int(n), dtype=torch.int32, device="cuda")


def ptr(t):
    return t.data_ptr()


def fill_frames(buf, mb, kind, N, W, H, seed, s):
    """N frames into the byte tensor buf on stream s: the synth generator's 8-bit kinds, or for DBDE16 uniform 16-bit
    noise ("noise") or tile rows of depth (ty + f) % 17 ("depths")"""
    if mb == 1:
        synth.gen_frames_device(kind, N, W, H, ptr(buf), seed=seed, stream=s.cuda_stream)
        return
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    buf.random_(0, 256, generator=g)
    if kind == "noise":
        return
    ty = torch.arange(H, device="cuda") // 8
    step = max(1, (1 << 28) // (2 * W * H))
    for f0 in range(0, N, step):
        f1 = min(N, f0 + step)
        k = (ty[None, :] + torch.arange(f0, f1, device="cuda")[:, None]) % 17
        m = (1 << k) - 1
        v = buf[2 * f0 * W * H:2 * f1 * W * H].view(f1 - f0, H, W, 2)
        v[..., 0].bitwise_and_((m & 255).to(torch.uint8)[:, :, None])
        v[..., 1].bitwise_and_((m >> 8).to(torch.uint8)[:, :, None])


def as_np(t, mb):
    a = t.cpu().numpy()
    return a.view(np.uint16) if mb == 2 else a


def first_diff(got, want, what):
    if not torch.equal(got, want):
        assert got.shape == want.shape, (what, got.shape, want.shape)
        bad = tuple(int(x) for x in (got != want).nonzero()[0])
        pytest.fail("%s differs first at %r: %d != %d" % (what, bad, int(got[bad]), int(want[bad])))


def oracle_pack(frames, mb, first):
    """the oracle's records of frames (n, H, W) on host threads -> (stream, sizes)"""
    n = len(frames)
    parts = {}

    def work(a, b):
        parts[a] = (ORA.pack_frames(frames[a:b], first + a) if mb == 1 else oracle.port16.pack_frames(frames[a:b], first + a))
        return 0

    oracle._fan_out(n, THREADS, work)
    keys = sorted(parts)
    return np.concatenate([parts[k][0] for k in keys]), np.concatenate([parts[k][1] for k in keys])


def check_slots(rec, stride, sizes, offs, frames_of, mb, first, N, what, chunk_bytes=1 << 28):
    """records j at rec[j * stride] against the oracle's records of frames_of(a, b) (numpy), a chunk at a time"""
    assert offs.tolist() == [j * stride for j in range(N)], what
    step = max(1, min(N, chunk_bytes // stride))
    for a in range(0, N, step):
        b = min(N, a + step)
        want, wsz = oracle_pack(frames_of(a, b), mb, first + a)
        assert sizes[a:b].tolist() == wsz.tolist(), (what, a)
        top = int(wsz.max())
        got = rec[a * stride:b * stride].view(b - a, stride)[:, :top].cpu().numpy()
        at = 0
        for j in range(b - a):
            n = int(wsz[j])
            if not np.array_equal(got[j, :n], want[at:at + n]):
                i = int(np.argwhere(got[j, :n] != want[at:at + n])[0][0])
                pytest.fail("%s record %d differs first at byte %d" % (what, a + j, i))
            at += n


def block_mean_t(x, b):
    """x (n, H, W) int32 -> the rounded means of its in-frame b x b blocks, (sum + count / 2) / count"""
    n, H, W = x.shape
    Hb, Wb = -(-H // b), -(-W // b)
    p = torch.zeros((n, Hb * b, Wb * b), dtype=torch.int32, device=x.device)
    p[:, :H, :W] = x
    m = torch.zeros((Hb * b, Wb * b), dtype=torch.int32, device=x.device)
    m[:H, :W] = 1
    s = p.view(n, Hb, b, Wb, b).sum(dim=(2, 4))
    c = m.view(Hb, b, Wb, b).sum(dim=(1, 3))
    return (s + c // 2) // c


def values(t, mb):
    """pixels (bytes, or int16 views of U16) -> int32 pixel values"""
    if mb == 1:
        return t.to(torch.int32)
    return (t.view(torch.int16) if t.dtype == torch.uint8 else t).to(torch.int32) & 0xFFFF


def pad_crop_t(frame, x0, y0, cw, ch, pad):
    """frame (H, W) on the device -> the cw x ch window at (x0, y0), `pad` outside the frame"""
    H, W = frame.shape
    out = torch.full((ch, cw), pad, dtype=frame.dtype, device=frame.device)
    xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
    if xa < xb and ya < yb:
        out[ya - y0:yb - y0, xa - x0:xb - x0] = frame[ya:yb, xa:xb]
    return out


class Calls:
    """the device entry points of one format on stream s"""

    def __init__(self, codec, mb, s):
        self.c, self.lib, self.mb, self.st = codec, codec.lib, mb, s.cuda_stream

    def encode(self, fr, W, H, n, out, stride, offs, sizes):
        f = self.lib.dbde_b200_encode_device if self.mb == 1 else self.lib.dbde_b200_encode16_device
        self.c._ck(f(self.c.h, fr, W, H, FIRST, n, out, n * stride, stride, offs, sizes, self.st), "encode")

    def decode(self, rec, nbytes, offs, W, H, n, out, st, ix):
        f = self.lib.dbde_b200_decode_device if self.mb == 1 else self.lib.dbde_b200_decode16_device
        self.c._ck(f(self.c.h, rec, nbytes, offs, W, H, n, out, st, ix, self.st), "decode")

    def validate(self, rec, nbytes, offs, W, H, n, st, ix):
        assert self.mb == 1
        self.c._ck(self.lib.dbde_b200_validate_device(self.c.h, rec, nbytes, offs, W, H, n, st, ix, self.st), "validate")

    def crops(self, rec, nbytes, offs, W, H, n, corners, ncrops, per_frame, size, out, st, ix, pad):
        f = self.c.decode_crops_device if self.mb == 1 else self.c.decode16_crops_device
        f(rec, nbytes, offs, W, H, n, corners, ncrops, per_frame, size, out, st, ix, pad=pad, stream=self.st)

    def binned(self, rec, nbytes, offs, W, H, n, factor, out, st, ix):
        f = self.c.decode_binned_device if self.mb == 1 else self.c.decode16_binned_device
        f(rec, nbytes, offs, W, H, n, factor, out, st, ix, stream=self.st)

    def encode_crops(self, fr, W, H, n, corners, ncrops, per_frame, size, out, cap, stride, offs, sizes, pad):
        f = self.c.encode_crops_device if self.mb == 1 else self.c.encode16_crops_device
        f(fr, W, H, FIRST, n, corners, ncrops, per_frame, size, out, cap, offs, sizes, pad=pad, stream=self.st,
          slot_stride=stride)


def check_status(s, st, ix, n, bad=()):
    s.synchronize()
    status, index = st.cpu().numpy().view(np.uint32), ix.cpu().numpy().view(np.uint64)
    for j in range(n):
        if j not in bad:
            assert status[j] == 0 and index[j] == FIRST + j, (j, int(status[j]), int(index[j]))
    return status, index


# ------------------------------------------------------------------ A: frames at the size limit
@pytest.mark.gpu
def test_boundary_shapes_are_refused(codec):
    """one tile or one pixel over the caps is E_INVALID in every device entry point; the largest legal shape is taken
    (nframes = 0: nothing is allocated or launched)"""
    lib, h = codec.lib, codec.h
    over = [(1, 2147483641), (2147483641, 1), (46341, 46341)]
    for W, H in over + [(46340, 46341)]:
        want = E_INVALID if (W, H) in over else 0
        for f in (lib.dbde_b200_encode_device, lib.dbde_b200_encode16_device):
            assert f(h, None, W, H, 0, 0, None, 0, 0, None, None, None) == want, (f, W, H)
        for f in (lib.dbde_b200_decode_device, lib.dbde_b200_decode16_device):
            assert f(h, None, 0, None, W, H, 0, None, None, None, None) == want, (f, W, H)
        assert lib.dbde_b200_validate_device.argtypes is not None
        assert lib.dbde_b200_validate_device(h, None, 0, None, W, H, 0, None, None, None) == want, (W, H)
        for f in (lib.dbde_b200_decode_binned_device, lib.dbde_b200_decode16_binned_device):
            assert f(h, None, 0, None, W, H, 0, 8, None, None, None, None) == want, (f, W, H)
        for f in (lib.dbde_b200_decode_crops_device, lib.dbde_b200_decode16_crops_device):
            assert f(h, None, 0, None, W, H, 0, None, 1, 0, 8, 8, 0, None, None, None, None) == want, (f, W, H)


@pytest.mark.gpu
@pytest.mark.parametrize("c", LIMITS, ids=lambda c: c.name)
def test_frame_at_the_size_limit(codec, S, c):
    """encode against the band-assembled oracle record, decode, validate, the far-corner region, crops at the corners,
    past the far edges and near INT32_MAX, binned, and a crop-encoder crop over the far corner"""
    mb, W, H = c.mb, c.W, c.H
    need(24)
    calls = Calls(codec, mb, S)
    fb = mb * W * H
    stride = slot_stride(W, H, mb)
    src = dev(fb)
    fill_frames(src, mb, c.kind, 1, W, H, 77, S)
    rec = dev(stride)
    offs, sizes = u64(1), u64(1)
    calls.encode(ptr(src), W, H, 1, ptr(rec), stride, ptr(offs), ptr(sizes))
    S.synchronize()
    size = int(sizes[0])
    assert int(offs[0]) == 0
    img = src.view(H, W * mb)
    end = 0
    for o, want in record_pieces(W, H, mb, FIRST,
                                 lambda x0, x1, y0, y1: as_np(img[y0:y1, mb * x0:mb * x1], mb)):
        got = rec[o:o + len(want)].cpu().numpy()
        if not np.array_equal(got, want):
            i = int(np.argwhere(got != want)[0][0])
            pytest.fail("record byte %d differs: %d != %d" % (o + i, got[i], want[i]))
        end = max(end, o + len(want))
    assert size == end
    w, h = tiles(W, H)
    if c.name == "A5":
        n64 = size - (32 + 3 * w * h)
        assert size > 1 << 32 and n64 >= 0.98 * 16 * w * h, (size, n64)
    tight = rec[:size].clone()           # the record in a buffer of its own size: an overrun reads past it
    del rec
    one = torch.zeros(1, dtype=torch.int64, device="cuda")
    st, ix = u32(1), u64(1)

    out = dev(fb)
    out.fill_(0xA7)
    calls.decode(ptr(tight), size, ptr(one), W, H, 1, ptr(out), ptr(st), ptr(ix))
    check_status(S, st, ix, 1)
    for a in range(0, fb, 1 << 30):
        first_diff(out[a:a + (1 << 30)], src[a:a + (1 << 30)], "decode at byte %d" % a)
    del out
    frame = src.view(H, W) if mb == 1 else src.view(torch.int16).view(H, W)
    if mb == 1:
        st.fill_(-1)
        calls.validate(ptr(tight), size, ptr(one), W, H, 1, ptr(st), ptr(ix))
        check_status(S, st, ix, 1)
        rw, rh = min(W, 37), min(H, 19)
        out = dev(rw * rh)
        codec.decode_roi_device(ptr(tight), size, ptr(one), W, H, 1, (W - rw, H - rh, rw, rh), ptr(out), ptr(st), ptr(ix),
                                stream=S.cuda_stream)
        check_status(S, st, ix, 1)
        first_diff(out.view(rh, rw), frame[H - rh:, W - rw:], "far-corner region")

    cw, ch = min(W, 37), min(H, 19)
    corners = [(0, 0), (W - cw, 0), (0, H - ch), (W - cw, H - ch), (W - cw // 2, H - ch // 2), (-3, H - 5),
               (W - 4, -7), (INT32_MAX - cw // 2, H - ch), (W - cw, INT32_MAX - 2), (INT32_MAX, INT32_MAX)]
    pad = 0x5A if mb == 1 else 0x5A5A
    d_c = torch.tensor(corners, dtype=torch.int32, device="cuda")
    out = dev(mb * len(corners) * cw * ch)
    calls.crops(ptr(tight), size, ptr(one), W, H, 1, ptr(d_c), len(corners), 0, (cw, ch), ptr(out), ptr(st), ptr(ix), pad)
    check_status(S, st, ix, 1)
    got = out.view(len(corners), ch, cw) if mb == 1 else out.view(torch.int16).view(len(corners), ch, cw)
    for r, (x0, y0) in enumerate(corners):
        first_diff(got[r], pad_crop_t(frame, x0, y0, cw, ch, pad), "crop at %r" % ((x0, y0),))

    for b in c.bins:
        bw, bh = -(-W // b), -(-H // b)
        out = dev(mb * bw * bh)
        calls.binned(ptr(tight), size, ptr(one), W, H, 1, b, ptr(out), ptr(st), ptr(ix))
        check_status(S, st, ix, 1)
        got = values(out, mb).view(bh, bw)
        rows = b * max(1, (1 << 26) // (b * W))
        cols = min(W, b * max(1, (1 << 26) // (b * rows)))
        for y0 in range(0, H, rows):
            for x0 in range(0, W, cols):
                want = block_mean_t(values(frame[y0:y0 + rows, x0:x0 + cols], mb)[None], b)[0]
                first_diff(got[y0 // b:y0 // b + want.shape[0], x0 // b:x0 // b + want.shape[1]], want,
                           "binned by %d at (%d, %d)" % (b, x0, y0))
        del out

    # the crop encoder over the far corner: its last bytes are the frame's last bytes
    cw, ch = min(W, 40), min(H, 24)
    x0, y0 = W - cw // 2, H - ch // 2
    d_c = torch.tensor([[x0, y0]], dtype=torch.int32, device="cuda")
    cs = slot_stride(cw, ch, mb)
    out = dev(cs)
    calls.encode_crops(ptr(src), W, H, 1, ptr(d_c), 1, 0, (cw, ch), ptr(out), cs, cs, ptr(offs), ptr(sizes), 0x33)
    S.synchronize()
    crop = pad_crop_t(frame, x0, y0, cw, ch, 0x33).cpu().numpy()
    want = pack_one(crop.view(np.uint16) if mb == 2 else crop, mb, FIRST)
    assert int(sizes[0]) == len(want)
    assert np.array_equal(out[:len(want)].cpu().numpy(), want)


# ------------------------------------------------------------------ B and D: batches past 2^32 bytes, device and host forms
def damage(rec, offs, sizes, W, H, mb, N):
    """three records past 2^32: a bad tag, a first tile over the depth limit (with n64 raised to match), and the last
    record cut short by 8 bytes -> ({frame: status bit}, stream bytes)"""
    wh = tiles(W, H)[0] * tiles(W, H)[1]
    tag, deep, last = N - 3, N - 2, N - 1
    assert all(int(offs[j]) > 1 << 32 for j in (tag, deep, last))
    rec[int(offs[tag])] = 9
    o = int(offs[deep])
    k = int(rec[o + 24])
    rec[o + 24] = 8 * mb + 1
    n = o + 28 + (1 + mb) * wh
    n64 = int(np.frombuffer(rec[n:n + 4].cpu().numpy().tobytes(), "<i4")[0]) + 8 * mb + 1 - k
    rec[n:n + 4] = torch.tensor(np.frombuffer(struct.pack("<i", n64), np.uint8).copy(), device="cuda")
    return {tag: pkg.ST_BAD_FRAME_HEADER, deep: pkg.ST_DEPTH_TOO_BIG, last: pkg.ST_TRUNCATED}, int(offs[last]) + int(sizes[last]) - 8


def check_batch_output(s, out, ref_of, shape, N, bad, st, ix, what, chunk=1 << 28):
    """outputs (N,) + shape of bytes: frame j equal to ref_of(a, b)[j - a], and the damaged frames still 0xA7"""
    status, index = check_status(s, st, ix, N, bad)
    for j, bit in bad.items():
        assert status[j] & bit, (what, j, int(status[j]))
    per = int(np.prod(shape))
    got = out[:N * per].view((N,) + tuple(shape))
    step = max(1, chunk // per)
    for a in range(0, N, step):
        b = min(N, a + step)
        diff = (got[a:b] != ref_of(a, b)).flatten(1).any(1).nonzero().flatten().tolist()
        assert sorted(a + d for d in diff) == sorted(j for j in bad if a <= j < b), (what, [a + d for d in diff][:5])
    for j in bad:
        assert bool((got[j] == 0xA7).all()), (what, j)


def host_forms(codec, b, rec, stride, sizes, src):
    """encode_host / encode16_host on a pageable buffer past 4 GiB, index_stream(16), decode_host / decode16_host:
    byte-equal to the device records and the source frames"""
    mb, W, H, N = b.mb, b.W, b.H, b.N
    lib = codec.lib
    cap = stride * N + 16
    src_np = src.cpu().numpy().view(np.uint8 if mb == 1 else np.uint16)
    out = np.empty(cap, dtype=np.uint8)
    offs = np.zeros(N + 1, dtype=np.uint64)
    enc = lib.dbde_b200_encode_host if mb == 1 else lib.dbde_b200_encode16_host
    codec._ck(enc(codec.h, src_np.ctypes.data, W, H, FIRST, N, out.ctypes.data, cap, offs.ctypes.data), "encode_host")
    del src_np
    assert np.diff(offs).tolist() == sizes.tolist() and int(offs[N]) > 1 << 32
    step = max(1, (1 << 28) // stride)
    for a in range(0, N, step):
        e = min(N, a + step)
        got = rec[a * stride:e * stride].view(e - a, stride).cpu().numpy()
        for j in range(a, e):
            assert np.array_equal(out[int(offs[j]):int(offs[j + 1])], got[j - a, :int(sizes[j])]), ("encode_host", j)
    idx = np.zeros(N + 1, dtype=np.uint64)
    index_fn = lib.dbde_b200_index_stream if mb == 1 else lib.dbde_b200_index_stream16
    assert index_fn(out.ctypes.data, int(offs[N]), W, H, idx.ctypes.data, N) == N
    assert np.array_equal(idx, offs)
    dec = np.empty(N * H * W, dtype=np.uint8 if mb == 1 else np.uint16)
    status, index = np.zeros(N, np.uint32), np.zeros(N, np.uint64)
    decf = lib.dbde_b200_decode_host if mb == 1 else lib.dbde_b200_decode16_host
    codec._ck(decf(codec.h, out.ctypes.data, int(offs[N]), offs.ctypes.data, W, H, N, dec.ctypes.data, status.ctypes.data,
                   index.ctypes.data), "decode_host")
    assert (status == 0).all() and index.tolist() == list(range(FIRST, FIRST + N))
    fb = mb * W * H
    del out
    for a in range(0, N, max(1, (1 << 28) // fb)):
        e = min(N, a + max(1, (1 << 28) // fb))
        assert np.array_equal(dec.view(np.uint8)[a * fb:e * fb], src[a * fb:e * fb].cpu().numpy()), ("decode_host", a)


@pytest.mark.gpu
@pytest.mark.parametrize("b", BATCHES, ids=lambda b: b.name)
def test_batch_past_4gib(codec, S, b):
    """encode against the oracle; decode, validate, region, crops and binned over outputs past 4 GiB, with three damaged
    records past stream offset 2^32; both crop encoders over a slot area past 4 GiB; the host forms on the same batch"""
    mb, W, H, N = b.mb, b.W, b.H, b.N
    need(24)
    calls = Calls(codec, mb, S)
    fb = mb * W * H
    stride = slot_stride(W, H, mb)
    sbuf = dev(N * fb + 16)
    src = sbuf[b.fbase:b.fbase + N * fb]
    fill_frames(src, mb, "noise", N, W, H, 1234, S)
    rec = dev(N * stride)
    d_o, d_sz = u64(N), u64(N)
    calls.encode(ptr(src), W, H, N, ptr(rec), stride, ptr(d_o), ptr(d_sz))
    S.synchronize()
    offs, sizes = d_o.cpu().numpy().view(np.uint64), d_sz.cpu().numpy().view(np.uint64)
    dt = np.uint8 if mb == 1 else np.uint16
    frames_of = lambda a, e: as_np(src[a * fb:e * fb], mb).reshape(e - a, H, W)
    check_slots(rec, stride, sizes, offs, frames_of, mb, FIRST, N, "encode")

    # D: the host forms on pageable buffers of the same batch
    host_forms(codec, b, rec, stride, sizes, src)

    bad, nbytes = damage(rec, offs, sizes, W, H, mb, N)
    st, ix = u32(N), u64(N)
    obuf = dev(N * fb + 16)
    out = obuf[b.obase:b.obase + N * fb]
    frames = src.view(N, H, W * mb)

    out.fill_(0xA7)
    st.fill_(-1)
    calls.decode(ptr(rec), nbytes, ptr(d_o), W, H, N, ptr(out), ptr(st), ptr(ix))
    check_batch_output(S, out, lambda a, e: frames[a:e], (H, W * mb), N, bad, st, ix, "decode")
    if mb == 1:
        st.fill_(-1)
        calls.validate(ptr(rec), nbytes, ptr(d_o), W, H, N, ptr(st), ptr(ix))
        status, _ = check_status(S, st, ix, N, bad)
        assert all(status[j] & bit for j, bit in bad.items()), status[-3:]
        out.fill_(0xA7)
        codec.decode_roi_device(ptr(rec), nbytes, ptr(d_o), W, H, N, (1, 0, W - 1, H), ptr(out), ptr(st), ptr(ix),
                                stream=S.cuda_stream)
        check_batch_output(S, out, lambda a, e: frames[a:e, :, 1:], (H, W - 1), N, bad, st, ix, "region")
    out.fill_(0xA7)
    pad = 0x5A if mb == 1 else 0x5A5A
    d_c = torch.tensor([[-3, -5]], dtype=torch.int32, device="cuda")
    calls.crops(ptr(rec), nbytes, ptr(d_o), W, H, N, ptr(d_c), 1, 0, (W, H), ptr(out), ptr(st), ptr(ix), pad)

    def shifted(a, e):
        r = torch.full((e - a, H, W * mb), 0x5A, dtype=torch.uint8, device="cuda")
        r[:, 5:, 3 * mb:] = frames[a:e, :H - 5, :(W - 3) * mb]
        return r

    check_batch_output(S, out, shifted, (H, W * mb), N, bad, st, ix, "crops at (-3, -5)")
    del obuf, out

    bw, bh = -(-W // 2), -(-H // 2)
    out = dev(N * mb * bw * bh)
    out.fill_(0xA7)
    calls.binned(ptr(rec), nbytes, ptr(d_o), W, H, N, 2, ptr(out), ptr(st), ptr(ix))

    def binned(a, e):
        m = block_mean_t(values(src[a * fb:e * fb], mb).view(e - a, H, W), 2)
        return m.to(torch.uint8) if mb == 1 else m.to(torch.int16).view(torch.uint8).view(e - a, bh, 2 * bw)

    check_batch_output(S, out, binned, (bh, mb * bw), N, bad, st, ix, "binned by 2", chunk=1 << 26)
    del out, rec

    if b.crop:
        cw, ch = b.crop
        j = torch.arange(N, device="cuda")
        d_c = torch.stack([(j * 37) % (W + 60) - 50, (j * 53) % (H + 40) - 30], 1).to(torch.int32).contiguous()
        cap = N * b.crop_stride
        out = dev(cap)
        calls.encode_crops(ptr(src), W, H, N, ptr(d_c), 1, 1, (cw, ch), ptr(out), cap, b.crop_stride, ptr(d_o), ptr(d_sz),
                           0x77)
        S.synchronize()
        corners = d_c.cpu().numpy()
        padv = 0x77

        def crops_of(a, e):
            r = np.full((e - a, ch, cw), padv, dtype=dt)
            fr = frames_of(a, e)
            for f in range(a, e):
                x0, y0 = (int(v) for v in corners[f])
                xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
                if xa < xb and ya < yb:
                    r[f - a, ya - y0:yb - y0, xa - x0:xb - x0] = fr[f - a, ya:yb, xa:xb]
            return r

        check_slots(out, b.crop_stride, d_sz.cpu().numpy().view(np.uint64), d_o.cpu().numpy().view(np.uint64), crops_of, mb,
                    FIRST, N, "crop encoder")


# ------------------------------------------------------------------ C: crop task counts past 2^32
@pytest.mark.gpu
@pytest.mark.parametrize("t", TASKS, ids=lambda t: t.name)
def test_crop_tasks_past_2_32(codec, S, t):
    """2^27 shared 1 x 1 crops inside and outside 64 x 64 frames: more than 2^32 warp tasks, rectangle indices and
    output offsets past 2^32, against a gather on the device"""
    mb, W, H, N, R = t.mb, t.W, t.H, t.N, t.ncrops
    need(20)
    calls = Calls(codec, mb, S)
    fb = mb * W * H
    src = dev(N * fb)
    fill_frames(src, mb, "mix" if mb == 1 else "depths", N, W, H, 99, S)
    stride = slot_stride(W, H, mb)
    rec, d_o, d_sz = dev(N * stride), u64(N), u64(N)
    calls.encode(ptr(src), W, H, N, ptr(rec), stride, ptr(d_o), ptr(d_sz))
    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    xy = torch.randint(-9, 74, (R, 2), generator=g, device="cuda", dtype=torch.int32)
    pad = 0x66 if mb == 1 else 0x6666
    out = dev(mb * N * R)
    out.fill_(0xA7)
    st, ix = u32(N), u64(N)
    calls.crops(ptr(rec), N * stride, ptr(d_o), W, H, N, ptr(xy), R, 0, (1, 1), ptr(out), ptr(st), ptr(ix), pad)
    check_status(S, st, ix, N)
    x, y = xy[:, 0].long(), xy[:, 1].long()
    inside = (x >= 0) & (x < W) & (y >= 0) & (y < H)
    lin = y.clamp(0, H - 1) * W + x.clamp(0, W - 1)
    got = out.view(N, R) if mb == 1 else out.view(torch.int16).view(N, R)
    frames = src.view(N, W * H) if mb == 1 else src.view(torch.int16).view(N, W * H)
    for f in range(N):
        want = torch.where(inside, frames[f][lin], torch.tensor(pad, dtype=frames.dtype, device="cuda"))
        first_diff(got[f], want, "frame %d crops" % f)


# ------------------------------------------------------------------ E: streams
@pytest.mark.gpu
def test_scratch_grows_behind_queued_work_and_streams_overlap(codec, S):
    """on stream S: decode of the 4300-frame batch, then, without a synchronise, validation of the tile-cap frame's
    record, whose word-prefix scratch is far larger than the batch's; meanwhile a DBDE16 encode on a second stream"""
    need(24)
    # the tile-cap record (A3), encoded on a stream of its own, kept in a tight buffer
    W3, H3 = 1, 2147483640
    S0 = torch.cuda.Stream()
    with torch.cuda.stream(S0):
        a3 = dev(W3 * H3)
        fill_frames(a3, 1, "low", 1, W3, H3, 3, S0)
        rec3, o3, sz3 = dev(slot_stride(W3, H3, 1)), u64(1), u64(1)
        Calls(codec, 1, S0).encode(ptr(a3), W3, H3, 1, ptr(rec3), slot_stride(W3, H3, 1), ptr(o3), ptr(sz3))
        S0.synchronize()
        size3 = int(sz3[0])
        tight3 = rec3[:size3].clone()
        S0.synchronize()
        del rec3, a3
    torch.cuda.empty_cache()

    b = BATCHES[0]
    W, H, N = b.W, b.H, b.N
    stride = slot_stride(W, H, 1)
    src, rec, d_o, d_sz = dev(N * W * H), dev(N * stride), u64(N), u64(N)
    calls = Calls(codec, 1, S)
    fill_frames(src, 1, "mix", N, W, H, 4321, S)
    calls.encode(ptr(src), W, H, N, ptr(rec), stride, ptr(d_o), ptr(d_sz))
    S.synchronize()                          # the batch stands; what follows is queued without a synchronise
    out, st, ix = dev(N * W * H), u32(N), u64(N)
    out.fill_(0xA7)
    one, st3, ix3 = torch.zeros(1, dtype=torch.int64, device="cuda"), u32(1), u64(1)
    st3.fill_(-1)
    calls.decode(ptr(rec), N * stride, ptr(d_o), W, H, N, ptr(out), ptr(st), ptr(ix))
    calls.validate(ptr(tight3), size3, ptr(one), W3, H3, 1, ptr(st3), ptr(ix3))

    S2 = torch.cuda.Stream()
    W2, H2, N2 = 2048, 2048, 64
    with torch.cuda.stream(S2):
        src2 = dev(2 * N2 * W2 * H2)
        fill_frames(src2, 2, "depths", N2, W2, H2, 8, S2)
        st2 = slot_stride(W2, H2, 2)
        rec2, o2, sz2 = dev(N2 * st2), u64(N2), u64(N2)
        Calls(codec, 2, S2).encode(ptr(src2), W2, H2, N2, ptr(rec2), st2, ptr(o2), ptr(sz2))
    S2.synchronize()
    check_slots(rec2, st2, sz2.cpu().numpy().view(np.uint64), o2.cpu().numpy().view(np.uint64),
                lambda a, e: as_np(src2[2 * a * W2 * H2:2 * e * W2 * H2], 2).reshape(e - a, H2, W2), 2, FIRST, N2,
                "DBDE16 encode on a second stream")
    check_batch_output(S, out, lambda a, e: src.view(N, H, W)[a:e], (H, W), N, {}, st, ix, "decode on S")
    check_status(S, st3, ix3, 1)


@pytest.mark.gpu
def test_seventeen_streams_of_one_context(codec, S):
    """encode and decode cycled through 17 streams (the scratch table holds 16), queued without a synchronise"""
    W, H, N = 1001, 67, 9
    streams = [torch.cuda.Stream() for _ in range(17)]
    runs = []
    for rnd in range(2):
        for i, s in enumerate(streams):
            with torch.cuda.stream(s):
                calls = Calls(codec, 1, s)
                stride = slot_stride(W, H, 1)
                src, rec, o, sz = dev(N * W * H), dev(N * stride), u64(N), u64(N)
                fill_frames(src, 1, "mix", N, W, H, 100 * rnd + i, s)
                calls.encode(ptr(src), W, H, N, ptr(rec), stride, ptr(o), ptr(sz))
                out, st, ix = dev(N * W * H), u32(N), u64(N)
                out.fill_(0xA7)
                calls.decode(ptr(rec), N * stride, ptr(o), W, H, N, ptr(out), ptr(st), ptr(ix))
                runs.append((s, src, rec, o, sz, out, st, ix, stride))
    for s, src, rec, o, sz, out, st, ix, stride in runs:
        s.synchronize()
        check_slots(rec, stride, sz.cpu().numpy().view(np.uint64), o.cpu().numpy().view(np.uint64),
                    lambda a, e: src[a * W * H:e * W * H].cpu().numpy().reshape(e - a, H, W), 1, FIRST, N, "encode")
        check_batch_output(s, out, lambda a, e: src.view(N, H, W)[a:e], (H, W), N, {}, st, ix, "decode")
