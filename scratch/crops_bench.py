"""Crop decode against the region decode it generalises, the full decode, and the parent commit's region decode.

    python scratch/crops_bench.py [--frames 1000] [--reps 20] [--warmup 3] [--rounds 3] [--parent-lib LIB] [--out FILE]

The workload is bench.py's and scratch/roi_bench.py's: 2048x2048 'micro' frames from the GPU generator with seed 42,
encoded on the device into fixed-stride slots (~1.6 GB of records, larger than L2, so every launch reads them from
HBM).  Before anything is timed, every crop case's output is compared with the pad-crop of the full GPU decode of the
same batch, and every region with the crop of it.  Device variants are timed with CUDA events over --reps launches
after --warmup launches, in --rounds rounds that interleave the variants (the median is reported, the rounds beside
it).  Host variants: frames/s over --host-reps calls on pinned buffers.

--parent-lib: a build of the parent commit's library (make -C dbce-video-cpp_b200/csrc OUT=... in a checkout of it).
Its region decode is timed in the same process, alternating with this tree's, for the seven device regions and the
two host regions of roi_bench.py.  One JSON line per variant on stdout (and in --out).  Needs a GPU.
"""
import argparse
import importlib
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scratch"))

from roi_bench import REGIONS, card  # noqa: E402

W = H = 2048
CROP = 256


def parse():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--frames", type=int, default=1000)
    p.add_argument("--kind", default="micro")
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--host-frames", type=int, default=200, help="frames of the host-buffer leg")
    p.add_argument("--host-reps", type=int, default=5)
    p.add_argument("--parent-lib", default=None, help="the parent commit's libdbde_b200.so, for the region regression")
    p.add_argument("--out", default=None, help="also write the JSON lines here")
    a = p.parse_args()
    if a.reps < 20:
        p.error("--reps must be at least 20")
    return a


def walks(N, rng):
    """one random walk of N steps, rescaled twice: into [0, W - CROP] (every crop inside the frame), and into a range
    wider by 110 pixels on each side (about a quarter of the crops partly outside)"""
    w = np.cumsum(rng.integers(-24, 25, (N, 2)), axis=0).astype(np.float64)
    u = (w - w.min(axis=0)) / np.maximum(w.max(axis=0) - w.min(axis=0), 1)
    inside = np.round(u * (W - CROP)).astype(np.int32)
    edges = np.round(u * (W - CROP + 220) - 110).astype(np.int32)
    return inside.reshape(N, 1, 2), edges.reshape(N, 1, 2)


def parent_codec(pkg, codec, path):
    """a Codec on the parent commit's library.  pkg.load() would look up the crop entry points, which that library
    does not have, so only what the region regression calls is bound, with this build's signatures."""
    import ctypes as C
    lib = C.CDLL(os.path.abspath(path))
    for name in ("dbde_b200_create", "dbde_b200_destroy", "dbde_b200_last_error", "dbde_b200_decode_device",
                 "dbde_b200_decode_roi_device", "dbde_b200_decode_roi_host"):
        fn, own = getattr(lib, name), getattr(codec.lib, name)
        fn.argtypes, fn.restype = own.argtypes, own.restype
    c = pkg.Codec.__new__(pkg.Codec)
    c.lib, c.h = lib, C.c_void_p()
    if lib.dbde_b200_create(0, C.byref(c.h)) or not c.h.value:
        raise RuntimeError("dbde_b200_create failed in " + path)
    return c


def main():
    a = parse()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("crops_bench.py: no CUDA device -- this measurement runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    import synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    codec = pkg.Codec(0)
    parent = parent_codec(pkg, codec, a.parent_lib) if a.parent_lib else None
    N = a.frames
    wh, px = (W // 8) * (H // 8), W * H
    cap, stride = codec.stream_bound(W, H, N), codec.slot_stride(W, H)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    frames = torch.empty(N * px, dtype=torch.uint8, device=dev)
    slots = torch.empty(cap + 64, dtype=torch.uint8, device=dev)
    full = torch.empty(N * px, dtype=torch.uint8, device=dev)
    out = torch.empty(N * px, dtype=torch.uint8, device=dev)
    offs = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    sizes = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    status = torch.zeros(N, dtype=torch.int32, device=dev)
    cs = torch.cuda.current_stream().cuda_stream
    sp = slots.data_ptr() + delta
    synth.gen_frames_device(a.kind, N, W, H, frames.data_ptr(), seed=42, f0=0, stream=cs)
    codec.encode_device(frames.data_ptr(), W, H, 0, N, sp, cap, offs.data_ptr(), sizes.data_ptr(), cs)
    torch.cuda.synchronize()
    rec_sizes = sizes[:N].cpu().numpy().astype(np.int64)

    # ---- the cases
    rng = np.random.default_rng(2026)
    walk_in, walk_edge = walks(N, rng)
    partly_out = float(np.mean((walk_edge[:, 0] < 0).any(axis=1) | (walk_edge[:, 0] > W - CROP).any(axis=1)))
    wells = np.array([(25 + 170 * i, 68 + 256 * j) for j in range(8) for i in range(12)], dtype=np.int32)
    cases = [("crop 256x256 shared @1001,999", np.array([[1001, 999]], dtype=np.int32), (CROP, CROP)),
             ("crop 256x256 per-frame walk inside", walk_in, (CROP, CROP)),
             ("crop 256x256 per-frame walk to the edges", walk_edge, (CROP, CROP)),
             ("crop 96 wells 12x8 120x120 shared", wells, (120, 120))]
    d_corners = {name: torch.from_numpy(c.reshape(-1, 2).copy()).to(dev) for name, c, _ in cases}

    def full_decode(c=codec):
        return lambda: c.decode_device(sp, cap, offs.data_ptr(), W, H, N, full.data_ptr(), status.data_ptr(), None, cs)

    def roi_decode(r, c=codec):
        r = r or (0, 0, W, H)
        return lambda: c.decode_roi_device(sp, cap, offs.data_ptr(), W, H, N, r, out.data_ptr(), status.data_ptr(), None, cs)

    def crops_decode(name, corners, size):
        return lambda: codec.decode_crops_device(sp, cap, offs.data_ptr(), W, H, N, d_corners[name].data_ptr(), corners.shape[-2],
                                                 corners.ndim == 3, size, out.data_ptr(), status.data_ptr(), None, 0, cs)

    def wells_by_roi():
        for x0, y0 in wells:
            roi_decode((int(x0), int(y0), 120, 120))()

    gidx = torch.from_numpy(np.concatenate([((y0 + np.arange(120))[:, None] * W + x0 + np.arange(120)[None, :]).ravel()
                                            for x0, y0 in wells])).to(dev)
    gout = out[:N * gidx.numel()].view(N, gidx.numel())

    def full_and_gather():
        full_decode()()
        torch.index_select(full.view(N, px), 1, gidx, out=gout)

    def pad_crop(fv, corners, size, pad=0):
        cw, ch = size
        res = torch.full((N, corners.shape[-2], ch, cw), pad, dtype=torch.uint8, device=dev)
        c = np.broadcast_to(corners, (N,) + corners.shape) if corners.ndim == 2 else corners
        shared = corners.ndim == 2
        for f in range(1 if shared else N):
            for r in range(c.shape[1]):
                x0, y0 = int(c[f, r, 0]), int(c[f, r, 1])
                xa, xb, ya, yb = max(x0, 0), min(x0 + cw, W), max(y0, 0), min(y0 + ch, H)
                if xa < xb and ya < yb:
                    fs = slice(None) if shared else f
                    res[fs, r, ya - y0:yb - y0, xa - x0:xb - x0] = fv[fs, ya:yb, xa:xb]
        return res

    # ---- correctness before timing
    full_decode()()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0 and torch.equal(full, frames), "full decode != source frames"
    fv = full.view(N, H, W)
    for name, corners, size in cases:
        n = N * corners.shape[-2] * size[0] * size[1]
        out.fill_(0xA5)
        crops_decode(name, corners, size)()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0, name
        assert torch.equal(out[:n].view(N, corners.shape[-2], size[1], size[0]), pad_crop(fv, corners, size)), name
        assert bool((out[n:] == 0xA5).all()), name
    full_and_gather()
    torch.cuda.synchronize()
    assert torch.equal(gout.view(N, 96, 120, 120), pad_crop(fv, wells, (120, 120))), "gather"
    roi_codecs = [("", codec)] + ([("parent ", parent)] if parent else [])
    for tag, c in roi_codecs:
        for name, r in REGIONS:
            x0, y0, rw, rh = r or (0, 0, W, H)
            out.fill_(0xA5)
            roi_decode(r, c)()
            torch.cuda.synchronize()
            assert int(status.abs().sum()) == 0, tag + name
            assert torch.equal(out[:N * rw * rh].view(N, rh, rw), fv[:, y0:y0 + rh, x0:x0 + rw]), tag + name
    checked = ("every crop case's output == pad-crop of the full GPU decode (guard bytes past it untouched); decode_device + "
               "gather == the wells' pad-crop; every region of this build%s == crop of the full decode; full decode == source "
               "frames" % (" and of the parent build" if parent else ""))

    def timeit(fn):
        for _ in range(a.warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.reps):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / a.reps

    variants = [("decode_device", full_decode()), ("decode_roi_device 256x256@1001,999", roi_decode((1001, 999, CROP, CROP)))]
    variants += [("decode_crops_device " + name, crops_decode(name, c, s)) for name, c, s in cases]
    variants += [("96 x decode_roi_device 120x120 (the wells)", wells_by_roi),
                 ("decode_device + torch.index_select gather of the wells", full_and_gather)]
    for tag, c in roi_codecs:                            # the region regression: this build and the parent, alternating
        variants += [("%sdecode_roi_device %s" % (tag, name), roi_decode(r, c)) for name, r in REGIONS]
    times = {v[0]: [] for v in variants}
    for _ in range(a.rounds):
        for name, fn in variants:
            times[name].append(timeit(fn))
    meta = dict(card(), frames=N, W=W, H=H, kind=a.kind, seed=42, reps=a.reps, warmup=a.warmup, rounds=a.rounds,
                record_bytes=int(rec_sizes.sum()), checked=checked)
    med = {k: statistics.median(v) for k, v in times.items()}
    ref = {"decode_crops_device crop 256x256 shared @1001,999": "decode_roi_device 256x256@1001,999",
           "decode_crops_device crop 256x256 per-frame walk inside": "decode_roi_device 256x256@1001,999",
           "decode_crops_device crop 256x256 per-frame walk to the edges": "decode_roi_device 256x256@1001,999",
           "decode_crops_device crop 96 wells 12x8 120x120 shared": "96 x decode_roi_device 120x120 (the wells)"}
    lines = []
    for name, _ in variants:
        line = dict(variant=name, ms=round(med[name], 4), ms_rounds=[round(x, 4) for x in times[name]],
                    x_full_decode=round(med[name] / med["decode_device"], 4))
        if name in ref:
            line["vs"] = ref[name]
            line["x_vs"] = round(med[name] / med[ref[name]], 4)
        if "wells" in name and name.startswith("decode_crops"):
            line["x_decode_device_plus_gather"] = round(med[name] / med["decode_device + torch.index_select gather of the wells"], 4)
        if "to the edges" in name:
            line["crops_partly_outside"] = round(partly_out, 3)
        if parent and name.startswith("decode_roi_device ") and "parent " + name in med:
            line["x_parent"] = round(med[name] / med["parent " + name], 4)
        lines.append(dict(line, **meta))

    # ---- host leg: pinned buffers, frames/s
    Nh = min(a.host_frames, N)
    slot_bytes = slots[delta:delta + N * stride].view(N, stride)
    hoffs = np.zeros(Nh + 1, dtype=np.uint64)
    hoffs[1:] = np.cumsum(rec_sizes[:Nh])
    ps = codec.pinned(int(hoffs[Nh]))
    for i in range(Nh):
        ps.array[int(hoffs[i]):int(hoffs[i + 1])] = slot_bytes[i, :int(rec_sizes[i])].cpu().numpy()
    po, pst, pout = codec.pinned(8 * Nh), codec.pinned(4 * Nh), codec.pinned(Nh * px)
    po.array[:] = hoffs[:Nh].view(np.uint8)
    hc = np.ascontiguousarray(walk_in[:Nh])

    def host_full():
        codec.decode_host_raw(ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, pout.ptr, pst.ptr, None)

    def host_crops():
        assert codec.lib.dbde_b200_decode_crops_host(codec.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, hc.ctypes.data, 1, 1, CROP,
                                                     CROP, 0, pout.ptr, pst.ptr, None) == 0

    def host_roi(r, c):
        def fn():
            assert c.lib.dbde_b200_decode_roi_host(c.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, *r, pout.ptr, pst.ptr, None) == 0
        return fn

    host = [("decode_host", host_full), ("decode_crops_host 256x256 per-frame walk inside", host_crops)]
    for tag, c in roi_codecs:
        host += [("%sdecode_roi_host %s" % (tag, n), host_roi(r, c)) for n, r in REGIONS if r and r[2] in (1024, 256)]
    host_crops()                                         # the host form's crops (all inside the frame) before timing
    got = pout.array[:Nh * CROP * CROP].reshape(Nh, CROP, CROP)
    for i in range(Nh):
        x0, y0 = (int(v) for v in hc[i, 0])
        assert np.array_equal(got[i], fv[i, y0:y0 + CROP, x0:x0 + CROP].cpu().numpy()), ("host crops", i)
    ht = {n: [] for n, _ in host}
    for n, fn in host:
        fn()
    for _ in range(a.rounds):
        for n, fn in host:
            t0 = time.perf_counter()
            for _ in range(a.host_reps):
                fn()
            ht[n].append(Nh * a.host_reps / (time.perf_counter() - t0))
    assert (pst.array.view(np.uint32) == 0).all()
    f_full = statistics.median(ht["decode_host"])
    for n, _ in host:
        f = statistics.median(ht[n])
        line = dict(variant=n, frames_per_s=round(f, 1), fps_rounds=[round(x, 1) for x in ht[n]], x_decode_host=round(f / f_full, 3),
                    host_frames=Nh, host_reps=a.host_reps, buffers="pinned")
        if parent and n.startswith("decode_roi_host "):
            line["x_parent_fps"] = round(f / statistics.median(ht["parent " + n]), 4)
        lines.append(dict(line, **meta))
    for p in (ps, po, pst, pout):
        p.free()
    if parent:
        parent.close()
    codec.close()
    text = [json.dumps(x) for x in lines]
    print("\n".join(text))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(text) + "\n")


if __name__ == "__main__":
    main()
