"""Byte-for-byte parity of this tree's library with another build of it (normally the parent commit's), in one process.

    python scratch/kernel_parity.py --parent-lib LIB [--frames 48] [--out FILE]

Runs every entry point whose kernels share the record layout helpers, the fixed-field writer, the decode pre-pass and
the crop-task decoder -- the 8-bit and DBDE16 frame and crop encoders, the pre-pass (validation), the region, crop and
binned decoders and the full decoders -- through the host forms of both libraries on the same inputs, and asserts that
records, offsets, pixels, statuses and indices are identical.  The workloads are those of scratch/roi_bench.py,
crops_bench.py, encode_crops_bench.py (2048x2048 'micro' frames, seed 42), dbde16_subframe_bench.py and
encode16_crops_bench.py (the 12-bit 'sensor12' field plus noise), at fewer frames, plus odd sizes (1001x1003, 2304x48),
corners outside the frame and near INT32_MIN / INT32_MAX, and damaged records (bad tag, counts, depths, word count,
truncation) for every status bit.  LIB: make -C dbce-video-cpp_b200/csrc OUT=LIB in a checkout of the other commit.
One JSON line per case on stdout (and in --out).  Needs a GPU.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scratch"))

I32_MAX, I32_MIN = 2**31 - 1, -2**31


def parse():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--parent-lib", required=True)
    p.add_argument("--frames", type=int, default=48)
    p.add_argument("--out", default=None)
    return p.parse_args()


def other_codec(pkg, codec, path):
    """a Codec on the other library, every entry point bound with this build's signatures (the C ABI is unchanged)"""
    lib = C.CDLL(os.path.abspath(path))
    for name in dir(codec.lib):
        if name.startswith("dbde_b200_"):
            fn, own = getattr(lib, name), getattr(codec.lib, name)
            fn.argtypes, fn.restype = own.argtypes, own.restype
    c = pkg.Codec.__new__(pkg.Codec)
    c.lib, c.h = lib, C.c_void_p()
    if lib.dbde_b200_create(0, C.byref(c.h)) or not c.h.value:
        raise RuntimeError("dbde_b200_create failed in " + path)
    return c


def walk(N, W, H, crop, margin, rng):
    """the benches' random walk of crop corners, rescaled into [-margin, W - crop + margin] x [-margin, H - crop + margin]"""
    w = np.cumsum(rng.integers(-24, 25, (N, 2)), axis=0).astype(np.float64)
    u = (w - w.min(axis=0)) / np.maximum(w.max(axis=0) - w.min(axis=0), 1)
    span = np.array([W - crop, H - crop]) + 2 * margin
    return np.round(u * span - margin).astype(np.int32).reshape(N, 1, 2)


def wells(W, H, size):
    """the benches' 12 x 8 grid of wells, shared by every frame"""
    xs = np.linspace(0, W - size, 12).astype(np.int32)
    ys = np.linspace(0, H - size, 8).astype(np.int32)
    return np.array([(x, y) for y in ys for x in xs], dtype=np.int32)


def extreme(W, H, size):
    """corners outside the frame on every side, straddling its edges, and near INT32_MIN / INT32_MAX"""
    cw, ch = size
    return np.array([(-cw + 1, -ch + 1), (W - 1, H - 1), (-7, 3), (W - cw + 5, -9), (-cw, 0), (W, H), (3, H - 2),
                     (I32_MAX, I32_MAX), (I32_MAX - cw, I32_MAX - ch - 3), (I32_MIN, I32_MIN), (I32_MIN + 5, 17),
                     (11, I32_MAX - 1)], dtype=np.int32)


def sensor12(N, W, H, rng):
    """dbde16_subframe_bench.py's content: a smooth 12-bit field plus 5 bits of noise"""
    y, x = np.mgrid[0:H, 0:W].astype(np.float32)
    out = np.empty((N, H, W), dtype=np.uint16)
    for i in range(N):
        f = 2048 + 1500 * np.sin((x + 37 * i) / 211.0) * np.cos((y - 11 * i) / 157.0)
        out[i] = (f + rng.integers(0, 32, (H, W))).clip(0, 65535).astype(np.uint16)
    return out


def damaged(stream, offs, W, H, mb):
    """copies of a stream with one defect per record: every status bit of the pre-pass, the stream cut in a record's
    payload and in its fixed fields"""
    wh = ((W + 7) // 8) * ((H + 7) // 8)
    s = stream.copy()
    o = [int(v) for v in offs]
    n = len(o) - 1

    def put32(at, v):
        s[at:at + 4] = np.frombuffer(np.uint32(v & 0xFFFFFFFF).tobytes(), dtype=np.uint8)

    for j in range(n):
        r = o[j]
        kind = j % 6
        if kind == 0:
            put32(r, 3)                                   # tag
        elif kind == 1:
            put32(r + 20, wh + 1)                         # depth count
        elif kind == 2:
            put32(r + 24 + wh, mb * wh - 1)               # min count
        elif kind == 3:
            s[r + 24 + j % wh] = 8 * mb + 1 + j % 7       # a depth too big (and then the word count)
        elif kind == 4:
            n64 = int(np.frombuffer(s[r + 28 + (1 + mb) * wh:r + 32 + (1 + mb) * wh].tobytes(), dtype=np.uint32)[0])
            put32(r + 28 + (1 + mb) * wh, n64 + 1)        # word count
    cut_payload = s[:o[n - 1] + 32 + (1 + mb) * wh + 3]   # the last record's payload cut short
    cut_fixed = s[:o[n - 1] + 10]                          # ... and its fixed fields
    return [("damaged", s), ("cut_payload", cut_payload), ("cut_fixed", cut_fixed)]


def main():
    a = parse()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("kernel_parity.py: no CUDA device -- this check runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    import synth
    from roi_bench import card
    new = pkg.Codec(0)
    old = other_codec(pkg, new, a.parent_lib)
    info = card()
    lines = []
    fails = []
    N = a.frames
    rng = np.random.default_rng(42)

    def same(case, fn, *args, **kw):
        x, y = fn(new, *args, **kw), fn(old, *args, **kw)
        ok = len(x) == len(y) and all(np.array_equal(np.asarray(p), np.asarray(q)) for p, q in zip(x, y))
        rows = int(np.asarray(x[-1]).size)
        lines.append(dict(case=case, identical=bool(ok), items=rows, **info))
        print(json.dumps(lines[-1]), flush=True)
        if not ok:
            fails.append(case)
        return x

    # ---- 8-bit: the benches' 2048^2 micro frames, an odd size, a linear-partition size
    for kind, W, H, n in [("micro", 2048, 2048, N), ("mix", 1001, 1003, N), ("micro", 2304, 48, 8), ("low", 4096, 64, 8)]:
        fr = synth.gen_frames(kind, n, W, H)
        tag = "%s-%dx%d" % (kind, W, H)
        stream, offs = same(tag + " encode_host", lambda c: c.encode_host(fr, 7))
        offs = offs[:n]
        same(tag + " decode_host", lambda c: c.decode_host(stream, offs, W, H, fill=0xCD))
        same(tag + " validate_host", lambda c: c.validate_host(stream, offs, W, H))
        for b in (2, 4, 8):
            same(tag + " decode_binned_host %d" % b, lambda c: c.decode_binned_host(stream, offs, W, H, b, fill=0xCD))
        for roi in [(0, 0, W, H), (W // 4 + 3, H // 4 + 5, W // 2 - 1, H // 3), (W - 1, H - 1, 1, 1), (5, 0, 7, H)]:
            same(tag + " decode_roi_host %s" % (roi,), lambda c: c.decode_roi_host(stream, offs, W, H, roi, fill=0xCD))
        crop = min(256, W, H)
        for name, corners, size in [("walk-inside", walk(n, W, H, crop, 0, rng), (crop, crop)),
                                    ("walk-edges", walk(n, W, H, crop, 110, rng), (crop, crop)),
                                    ("wells", wells(W, H, min(120, W, H)), (min(120, W, H),) * 2),
                                    ("extreme", extreme(W, H, (37, 29)), (37, 29)),
                                    ("narrow", extreme(W, H, (1, 300)), (1, 300))]:
            same(tag + " decode_crops_host " + name, lambda c: c.decode_crops_host(stream, offs, W, H, corners, size, pad=0x5A, fill=0xCD))
            same(tag + " encode_crops_host " + name, lambda c: c.encode_crops_host(fr, corners, size, pad=0xA5, first_index=3))
        for dname, ds in damaged(stream, np.append(offs, len(stream)), W, H, 1):
            same(tag + " validate_host " + dname, lambda c: c.validate_host(ds, offs, W, H))
            same(tag + " decode_crops_host " + dname,
                 lambda c: c.decode_crops_host(ds, offs, W, H, extreme(W, H, (37, 29)), (37, 29), pad=1, fill=0xCD))
            same(tag + " decode_roi_host " + dname, lambda c: c.decode_roi_host(ds, offs, W, H, (1, 2, W - 3, H - 2), fill=0xCD))

    # ---- DBDE16: the benches' sensor12 content at 2048^2, 2304^2 and 1001x1003, and a small noisy odd size
    for W, H, n in [(2048, 2048, N // 2), (2304, 2304, 8), (1001, 1003, 16), (136, 72, 8)]:
        fr = sensor12(n, W, H, rng)
        if W == 136:
            fr = rng.integers(0, 65536, (n, H, W)).astype(np.uint16)    # every depth up to 16
        tag = "u16-%dx%d" % (W, H)
        stream, offs = same(tag + " encode16_host", lambda c: c.encode16_host(fr, 9))
        offs = offs[:n]
        same(tag + " decode16_host", lambda c: c.decode16_host(stream, offs, W, H, fill=0xABCD))
        for b in (2, 4, 8):
            same(tag + " decode16_binned_host %d" % b, lambda c: c.decode16_binned_host(stream, offs, W, H, b, fill=0xABCD))
        crop = min(256, W, H)
        for name, corners, size in [("walk-inside", walk(n, W, H, crop, 0, rng), (crop, crop)),
                                    ("walk-edges", walk(n, W, H, crop, int(0.14 * (W - crop)), rng), (crop, crop)),
                                    ("wells", wells(W, H, min(120, W, H)), (min(120, W, H),) * 2),
                                    ("extreme", extreme(W, H, (37, 29)), (37, 29)),
                                    ("narrow", extreme(W, H, (1, 300)), (1, 300))]:
            same(tag + " decode16_crops_host " + name,
                 lambda c: c.decode16_crops_host(stream, offs, W, H, corners, size, pad=0x1234, fill=0xABCD))
            same(tag + " encode16_crops_host " + name, lambda c: c.encode16_crops_host(fr, corners, size, pad=0x4321, first_index=5))
        for dname, ds in damaged(stream, np.append(offs, len(stream)), W, H, 2):
            same(tag + " decode16_host " + dname, lambda c: c.decode16_host(ds, offs, W, H, fill=0xABCD))
            same(tag + " decode16_crops_host " + dname,
                 lambda c: c.decode16_crops_host(ds, offs, W, H, extreme(W, H, (37, 29)), (37, 29), pad=7, fill=0xABCD))

    new.close()
    old.close()
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))
    print(json.dumps(dict(cases=len(lines), identical=len(lines) - len(fails), differ=fails, **info)))
    if fails:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
