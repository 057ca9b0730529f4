"""Crop encode against the gather-then-encode it replaces, the full-frame encoder, and the parent commit's codec.

    python scratch/encode_crops_bench.py [--frames 1000] [--reps 20] [--warmup 3] [--rounds 3] [--parent-lib LIB] [--out FILE]

The workload is bench.py's: 2048x2048 'micro' frames from the GPU generator with seed 42, in HBM (4.2 GB, larger than
L2).  Cases: 96 wells (a 12 x 8 grid of 120x120, shared corners) and one 256x256 crop per frame on a random walk of
which about a quarter of the crops lie partly outside the frame.  Before anything is timed, every crop record is
compared byte for byte with the oracle's record of the pad-crop of the source frame, the baselines' records with the
crop records (all bytes but the frame index, which the baselines number per crop), and the full-frame encoder's first
50 records with the oracle's.  Device variants are timed with CUDA events over --reps launches after --warmup
launches, in --rounds rounds that interleave the variants (the median is reported, the rounds beside it).  Host
variants: frames/s over --host-reps calls on pinned buffers.

--parent-lib: a build of the parent commit's library (make -C dbce-video-cpp_b200/csrc OUT=... in a checkout of it).
Its encode_device, encode_host and decode_device are timed in the same process, alternating with this tree's.  One
JSON line per variant on stdout (and in --out).  Needs a GPU.
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

from crops_bench import walks  # noqa: E402
from roi_bench import card  # noqa: E402

W = H = 2048
CROP = 256
WELL = 120


def parse():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--frames", type=int, default=1000)
    p.add_argument("--kind", default="micro")
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--host-frames", type=int, default=200, help="frames of the host-buffer leg")
    p.add_argument("--host-reps", type=int, default=5)
    p.add_argument("--parent-lib", default=None, help="the parent commit's libdbde_b200.so, for the regression rows")
    p.add_argument("--out", default=None, help="also write the JSON lines here")
    a = p.parse_args()
    if a.reps < 20:
        p.error("--reps must be at least 20")
    return a


def parent_codec(pkg, codec, path):
    """a Codec on the parent commit's library, with only what the regression rows call bound (this build's
    signatures; pkg.load() would look up entry points that library does not have)"""
    import ctypes as C
    lib = C.CDLL(os.path.abspath(path))
    for name in ("dbde_b200_create", "dbde_b200_destroy", "dbde_b200_last_error", "dbde_b200_encode_device",
                 "dbde_b200_encode_host", "dbde_b200_decode_device"):
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
        raise SystemExit("encode_crops_bench.py: no CUDA device -- this measurement runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    import oracle
    import synth
    ora = oracle.best()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    codec = pkg.Codec(0)
    parent = parent_codec(pkg, codec, a.parent_lib) if a.parent_lib else None
    N = a.frames
    px = W * H
    wh = (W // 8) * (H // 8)
    cs = torch.cuda.current_stream().cuda_stream
    frames = torch.empty(N * px, dtype=torch.uint8, device=dev)
    synth.gen_frames_device(a.kind, N, W, H, frames.data_ptr(), seed=42, f0=0, stream=cs)
    fv = frames.view(N, H, W)

    # ---- outputs: full-frame slots (records 16-byte aligned as encode_host lays them), crop slots, contiguous crops
    cap, stride = codec.stream_bound(W, H, N), codec.slot_stride(W, H)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    slots = torch.empty(cap + 64, dtype=torch.uint8, device=dev)
    sp = slots.data_ptr() + delta
    full = torch.empty(N * px, dtype=torch.uint8, device=dev)
    status = torch.zeros(N, dtype=torch.int32, device=dev)
    wells = np.array([(64 + 160 * i, 64 + 240 * j) for j in range(8) for i in range(12)], dtype=np.int32)
    rng = np.random.default_rng(2026)
    _, walk = walks(N, rng)
    partly_out = float(np.mean((walk[:, 0] < 0).any(axis=1) | (walk[:, 0] > W - CROP).any(axis=1)))
    cases = {"wells": (wells, (WELL, WELL)), "walk": (walk, (CROP, CROP))}
    d_corners = {k: torch.from_numpy(c.reshape(-1, 2).copy()).to(dev) for k, (c, _) in cases.items()}
    nmax = max(N * c.shape[-2] for c, _ in cases.values())
    offs = torch.zeros(nmax + 1, dtype=torch.int64, device=dev)          # the crop variants'
    sizes = torch.zeros(nmax + 1, dtype=torch.int64, device=dev)
    foffs = torch.zeros(N + 1, dtype=torch.int64, device=dev)            # the full-frame encode's, which the decode reads
    fsizes = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    cbuf, gbuf, crop_img = {}, {}, {}
    for k, (c, (cw, ch)) in cases.items():
        n = N * c.shape[-2]
        st = codec.slot_stride(cw, ch)
        cbuf[k] = (torch.empty(n * st + 64, dtype=torch.uint8, device=dev), st, n)
        gbuf[k] = torch.empty(n * st + 64, dtype=torch.uint8, device=dev)
        crop_img[k] = torch.empty(n * cw * ch, dtype=torch.uint8, device=dev)
    # torch gather indices: the wells (all inside the frame) and the walk's pad-gather (clamped index + in-frame mask)
    widx = torch.from_numpy(np.concatenate([((y0 + np.arange(WELL))[:, None] * W + x0 + np.arange(WELL)[None, :]).ravel()
                                            for x0, y0 in wells])).to(dev)
    xs = torch.from_numpy(walk[:, 0, 0].astype(np.int64)).to(dev)[:, None, None] + torch.arange(CROP, device=dev)[None, None, :]
    ys = torch.from_numpy(walk[:, 0, 1].astype(np.int64)).to(dev)[:, None, None] + torch.arange(CROP, device=dev)[None, :, None]
    inside = ((xs >= 0) & (xs < W) & (ys >= 0) & (ys < H)).reshape(-1)
    pidx = (torch.arange(N, device=dev)[:, None, None] * px + ys.clamp(0, H - 1) * W + xs.clamp(0, W - 1)).reshape(-1)
    pad0 = torch.zeros((), dtype=torch.uint8, device=dev)

    def enc_full(c=codec):
        return lambda: c.encode_device(frames.data_ptr(), W, H, 0, N, sp, cap, foffs.data_ptr(), fsizes.data_ptr(), cs)

    def dec_full(c=codec):
        return lambda: c.decode_device(sp, cap, foffs.data_ptr(), W, H, N, full.data_ptr(), status.data_ptr(), None, cs)

    def enc_crops(k, nf=N):
        c, size = cases[k]
        buf, st, n = cbuf[k]
        return lambda: codec.encode_crops_device(frames.data_ptr(), W, H, 0, nf, d_corners[k].data_ptr(), c.shape[-2], c.ndim == 3, size,
                                                 buf.data_ptr(), n * st, offs.data_ptr(), sizes.data_ptr(), 0, cs)

    def enc_contig(k):
        _, (cw, ch) = cases[k]
        buf, st, n = cbuf[k]
        g = gbuf[k]
        return lambda: codec.encode_device(crop_img[k].data_ptr(), cw, ch, 0, n, g.data_ptr(), n * st, offs.data_ptr(),
                                           sizes.data_ptr(), cs)

    def gather_wells():
        torch.index_select(fv.view(N, px), 1, widx, out=crop_img["wells"].view(N, -1))

    def gather_walk():
        torch.where(inside, torch.take(frames, pidx), pad0, out=crop_img["walk"])

    def gather_and(gather, k):
        e = enc_contig(k)

        def fn():
            gather()
            e()
        return fn

    # ---- correctness before timing
    def records(buf, st, n, sizes=sizes):
        torch.cuda.synchronize()
        sz = sizes[:n].cpu().numpy().astype(np.int64)
        host = buf[:n * st].cpu().numpy().reshape(n, st)
        return [host[j, :sz[j]] for j in range(n)]

    def drop_index(rec):
        return np.concatenate([rec[:4], rec[12:]])

    checked = []
    gather_wells()
    gather_walk()
    for k, (c, (cw, ch)) in cases.items():
        buf, st, n = cbuf[k]
        R = c.shape[-2]
        buf.fill_(0xA5)
        enc_crops(k)()
        got = records(buf, st, n)
        assert bool((buf[n * st:] == 0xA5).all()), k
        imgs = crop_img[k].view(N, R, ch, cw).cpu().numpy()
        for r in range(R):
            s, sz = ora.pack_frames(imgs[:, r], 0)
            o = np.concatenate([[0], np.cumsum(sz)]).astype(np.int64)
            for f in range(N):
                assert np.array_equal(got[f * R + r], s[o[f]:o[f + 1]]), (k, f, r)
        enc_contig(k)()
        base = records(gbuf[k], st, n)
        assert all(np.array_equal(drop_index(x), drop_index(y)) for x, y in zip(base, got)), k
        checked.append("%s: %d crop records == oracle; gather + encode_device records == them but for the index" % (k, n))
    # the torch pad-gather is the crop image: check the walk's one against numpy on a few frames
    wi = crop_img["walk"].view(N, CROP, CROP)
    for f in (0, N // 2, N - 1):
        x0, y0 = (int(v) for v in walk[f, 0])
        ref = np.zeros((CROP, CROP), np.uint8)
        xa, xb, ya, yb = max(x0, 0), min(x0 + CROP, W), max(y0, 0), min(y0 + CROP, H)
        ref[ya - y0:yb - y0, xa - x0:xb - x0] = fv[f, ya:yb, xa:xb].cpu().numpy()
        assert np.array_equal(wi[f].cpu().numpy(), ref), f
    for tag, c in [("", codec)] + ([("parent ", parent)] if parent else []):
        slots.fill_(0)
        enc_full(c)()
        got = records(slots[delta:], stride, N, fsizes)
        s, sz = ora.pack_frames(fv[:50].cpu().numpy(), 0)
        o = np.concatenate([[0], np.cumsum(sz)]).astype(np.int64)
        assert all(np.array_equal(got[f], s[o[f]:o[f + 1]]) for f in range(50)), tag
        dec_full(c)()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0 and torch.equal(full, frames), tag
        checked.append("%sencode_device: first 50 records == oracle; %sdecode_device == source frames" % (tag, tag))

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

    # the regression rows first, each beside its parent row
    variants = [("encode_device", enc_full())] + ([("parent encode_device", enc_full(parent))] if parent else [])
    variants += [("decode_device", dec_full())] + ([("parent decode_device", dec_full(parent))] if parent else [])
    variants += [("encode_crops_device 96 wells 120x120 shared", enc_crops("wells")),
                ("torch gather of the wells + encode_device", gather_and(gather_wells, "wells")),
                ("encode_crops_device 256x256 walk", enc_crops("walk")),
                ("torch pad-gather of the walk + encode_device", gather_and(gather_walk, "walk")),
                ("encode_device of the walk's crops, contiguous", enc_contig("walk")),
                ("encode_crops_device 256x256 walk, first %d frames" % (N // 2), enc_crops("walk", N // 2))]
    times = {v[0]: [] for v in variants}
    for _ in range(a.rounds):
        for name, fn in variants:
            times[name].append(timeit(fn))
    med = {k: statistics.median(v) for k, v in times.items()}
    meta = dict(card(), frames=N, W=W, H=H, kind=a.kind, seed=42, reps=a.reps, warmup=a.warmup, rounds=a.rounds,
                checked="; ".join(checked))
    vs = {"encode_crops_device 96 wells 120x120 shared": ["torch gather of the wells + encode_device", "encode_device"],
          "encode_crops_device 256x256 walk": ["torch pad-gather of the walk + encode_device", "encode_device of the walk's crops, contiguous"],
          "encode_device": ["parent encode_device"], "decode_device": ["parent decode_device"]}
    lines = []
    for name, _ in variants:
        line = dict(variant=name, ms=round(med[name], 4), ms_rounds=[round(x, 4) for x in times[name]])
        for i, ref in enumerate(vs.get(name, [])):
            if ref in med:
                line["vs%d" % (i + 1)] = ref
                line["x_vs%d" % (i + 1)] = round(med[name] / med[ref], 4)
        if "walk" in name:
            line["crops_partly_outside"] = round(partly_out, 3)
        lines.append(dict(line, **meta))

    # ---- host leg: pinned buffers, frames/s
    Nh = min(a.host_frames, N)
    pfr = codec.pinned(Nh * px)
    pfr.array[:] = frames[:Nh * px].cpu().numpy()
    hcap = codec.stream_bound(W, H, Nh)
    wcap = codec.stream_bound(WELL, WELL, Nh * len(wells))
    pout, pwout = codec.pinned(hcap), codec.pinned(wcap)
    poff, pwoff = codec.pinned(8 * (Nh + 1)), codec.pinned(8 * (Nh * len(wells) + 1))

    def host_full(c):
        def fn():
            assert c.lib.dbde_b200_encode_host(c.h, pfr.ptr, W, H, 0, Nh, pout.ptr, hcap, poff.ptr) == 0
        return fn

    def host_wells():
        assert codec.lib.dbde_b200_encode_crops_host(codec.h, pfr.ptr, W, H, 0, Nh, wells.ctypes.data, len(wells), 0, WELL, WELL, 0,
                                                     pwout.ptr, wcap, pwoff.ptr) == 0

    host = [("encode_host", host_full(codec)), ("encode_crops_host 96 wells 120x120 shared", host_wells)]
    if parent:
        host.append(("parent encode_host", host_full(parent)))
    host_wells()                                     # the host form's bytes == the device form's records back to back
    enc_crops("wells")()
    got = records(*cbuf["wells"])[:Nh * len(wells)]
    tot = int(pwoff.array.view(np.uint64)[Nh * len(wells)])
    assert np.array_equal(pwout.array[:tot], np.concatenate(got)), "encode_crops_host != encode_crops_device"
    checked.append("encode_crops_host (%d frames) == encode_crops_device's records back to back" % Nh)
    meta["checked"] = "; ".join(checked)
    for line in lines:
        line["checked"] = meta["checked"]
    ht = {n: [] for n, _ in host}
    for n, fn in host:
        fn()
    for _ in range(a.rounds):
        for n, fn in host:
            t0 = time.perf_counter()
            for _ in range(a.host_reps):
                fn()
            ht[n].append(Nh * a.host_reps / (time.perf_counter() - t0))
    f_full = statistics.median(ht["encode_host"])
    for n, _ in host:
        f = statistics.median(ht[n])
        line = dict(variant=n, frames_per_s=round(f, 1), fps_rounds=[round(x, 1) for x in ht[n]], x_encode_host=round(f / f_full, 4),
                    host_frames=Nh, host_reps=a.host_reps, buffers="pinned")
        if n == "encode_host" and parent:
            line["x_parent_fps"] = round(f / statistics.median(ht["parent encode_host"]), 4)
        lines.append(dict(line, **meta))
    for p in (pfr, pout, pwout, poff, pwoff):
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
