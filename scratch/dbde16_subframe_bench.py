"""DBDE16 crop and binned decoding against the full DBDE16 decode, and the full decode against the parent commit's.

    python scratch/dbde16_subframe_bench.py [--frames 300] [--reps 20] [--warmup 3] [--rounds 3] [--parent-lib LIB] [--out FILE]

The workload is scratch/enc16_only.py's sensor12 content (a 12-bit camera-like smooth field plus 5 bits of noise, seed
42) at 2048x2048, generated on the GPU and encoded on the device into fixed-stride slots; the 2.8 MB records per frame
(0.85 GB for 300 frames, larger than L2) are read from HBM by every launch.  2304x2304 and 1001x1003 batches of the
same content are measured beside it.  Before anything is timed, every output is compared with torch applied to the
source frames: crops with slices, the wells with a gather, bins with a block mean over the in-frame pixels; the full
decode with the source frames.  Device variants are timed with CUDA events over --reps launches after --warmup
launches, in --rounds rounds that interleave the variants (the median is reported, the rounds beside it).  Host
variants: frames/s over --host-reps calls on pinned buffers.

--parent-lib: a build of the parent commit's library (make -C dbce-video-cpp_b200/csrc OUT=... in a checkout of it).
Its decode16_device is timed in the same process, alternating with this tree's.  One JSON line per variant on stdout
(and in --out), each with the card's name and power limit.  Needs a GPU.
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

from roi_bench import card  # noqa: E402

CROP = 256
WELL = 120


def parse():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--frames", type=int, default=300)
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--host-frames", type=int, default=200, help="frames of the host-buffer leg")
    p.add_argument("--host-reps", type=int, default=5)
    p.add_argument("--parent-lib", default=None, help="the parent commit's libdbde_b200.so, for the decode16_device regression")
    p.add_argument("--out", default=None, help="also write the JSON lines here")
    a = p.parse_args()
    if a.reps < 20:
        p.error("--reps must be at least 20")
    if a.frames < 300:
        p.error("--frames must be at least 300")
    return a


def parent_codec(pkg, codec, path):
    """a Codec on the parent commit's library, with only what the regression calls bound (this build's signatures)"""
    import ctypes as C
    lib = C.CDLL(os.path.abspath(path))
    for name in ("dbde_b200_create", "dbde_b200_destroy", "dbde_b200_last_error", "dbde_b200_decode16_device"):
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
        raise SystemExit("dbde16_subframe_bench.py: no CUDA device -- this measurement runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    codec = pkg.Codec(0)
    parent = parent_codec(pkg, codec, a.parent_lib) if a.parent_lib else None
    lib = codec.lib
    N = a.frames
    cs = torch.cuda.current_stream().cuda_stream
    status = torch.zeros(N, dtype=torch.int32, device=dev)

    def dataset(W, H):
        """sensor12 frames, their records in fixed-stride slots and the offsets, on the device"""
        g = torch.Generator(device=dev)
        g.manual_seed(42)
        y = torch.arange(H, device=dev).view(1, H, 1)
        x = torch.arange(W, device=dev).view(1, 1, W)
        fr = (600 + x // 16 + y // 8 + torch.randint(0, 32, (N, H, W), device=dev, generator=g, dtype=torch.int32)).to(torch.int32)
        d = dict(W=W, H=H, frames=fr.to(torch.uint16).contiguous())
        del fr
        stride = int(lib.dbde_b200_slot_stride16(W, H))
        d["cap"] = stride * N
        d["slots"] = torch.empty(d["cap"] + 64, dtype=torch.uint8, device=dev)
        d["offs"] = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        d["sizes"] = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        codec._ck(lib.dbde_b200_encode16_device(codec.h, d["frames"].data_ptr(), W, H, 0, N, d["slots"].data_ptr(), d["cap"], 0,
                                                d["offs"].data_ptr(), d["sizes"].data_ptr(), cs), "encode16_device")
        torch.cuda.synchronize()
        d["rec_bytes"] = int(d["sizes"][:N].sum())
        # one CROP^2 crop per frame on a random walk inside the frame
        rng = np.random.default_rng(W + H)
        walk = np.cumsum(rng.integers(-40, 41, (N, 2)), axis=0) + ((W - CROP) // 2, (H - CROP) // 2)
        d["walk"] = np.stack([np.clip(walk[:, 0], 0, W - CROP), np.clip(walk[:, 1], 0, H - CROP)], axis=-1).astype(np.int32)
        d["d_walk"] = torch.from_numpy(d["walk"].reshape(-1)).to(dev)
        return d

    def full16(d, dst, c=codec):
        return lambda: c._ck(c.lib.dbde_b200_decode16_device(c.h, d["slots"].data_ptr(), d["cap"], d["offs"].data_ptr(), d["W"],
                                                             d["H"], N, dst.data_ptr(), status.data_ptr(), None, cs),
                             "decode16_device")

    def crops16(d, dst, corners, ncrops, per_frame, size):
        return lambda: codec.decode16_crops_device(d["slots"].data_ptr(), d["cap"], d["offs"].data_ptr(), d["W"], d["H"], N,
                                                   corners.data_ptr(), ncrops, per_frame, size, dst.data_ptr(), status.data_ptr(),
                                                   None, 0, cs)

    def binned16(d, dst, b):
        return lambda: codec.decode16_binned_device(d["slots"].data_ptr(), d["cap"], d["offs"].data_ptr(), d["W"], d["H"], N, b,
                                                    dst.data_ptr(), status.data_ptr(), None, cs)

    def block_mean(fr, b):
        """torch reference on the device: the rounded mean of each block's in-frame pixels"""
        n_, h, w = fr.shape
        hb, wb = -(-h // b), -(-w // b)
        p = torch.zeros((n_, hb * b, wb * b), dtype=torch.int32, device=dev)
        p[:, :h, :w] = fr.to(torch.int32)
        m = torch.zeros((hb * b, wb * b), dtype=torch.int32, device=dev)
        m[:h, :w] = 1
        s = p.view(n_, hb, b, wb, b).sum(dim=(2, 4))
        cnt = m.view(hb, b, wb, b).sum(dim=(1, 3))
        return ((s + cnt // 2) // cnt).to(torch.uint16)

    def check_full(d, full):
        full16(d, full)()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0 and torch.equal(full[:N * d["W"] * d["H"]].view(N, d["H"], d["W"]).view(torch.int16),
                                                             d["frames"].view(torch.int16)), "decode16_device != source frames"

    def check_walk(d, out):
        crops16(d, out, d["d_walk"], 1, True, (CROP, CROP))()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0
        got = out[:N * CROP * CROP].view(N, CROP, CROP).view(torch.int16)
        src = d["frames"].view(torch.int16)
        for i, (x0, y0) in enumerate(d["walk"].tolist()):
            assert torch.equal(got[i], src[i, y0:y0 + CROP, x0:x0 + CROP]), ("crop", d["W"], i)

    def check_binned(d, out, b):
        binned16(d, out, b)()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0
        hb, wb = -(-d["H"] // b), -(-d["W"] // b)
        for f0 in range(0, N, 50):
            want = block_mean(d["frames"][f0:f0 + 50], b)
            assert torch.equal(out[f0 * hb * wb:(f0 + len(want)) * hb * wb].view(-1, hb, wb).view(torch.int16), want.view(torch.int16)), \
                ("binned", d["W"], b, f0)

    # ---- the 2048^2 batch: correctness before timing
    W = H = 2048
    big = dataset(W, H)
    full = torch.empty(N * W * H, dtype=torch.uint16, device=dev)
    out = torch.empty(N * W * H // 4 + 64, dtype=torch.uint16, device=dev)
    check_full(big, full)
    check_walk(big, out)
    for b in (2, 4, 8):
        check_binned(big, out, b)
    wells = torch.tensor([(50 + 165 * i, 60 + 245 * j) for j in range(8) for i in range(12)], dtype=torch.int32, device=dev)
    wl = wells.cpu().numpy()
    idx = torch.cat([(torch.arange(WELL, device=dev).view(WELL, 1) + int(y0)) * W + torch.arange(WELL, device=dev).view(1, WELL) + int(x0)
                     for x0, y0 in wl]).view(-1)
    gathered = torch.empty((N, idx.numel()), dtype=torch.int16, device=dev)
    wells_out = torch.empty(N * idx.numel(), dtype=torch.uint16, device=dev)

    def full_and_gather():
        """what a user writes today: the full decode, then one gather of the 96 wells"""
        full16(big, full)()
        torch.index_select(full.view(torch.int16).view(N, W * H), 1, idx, out=gathered)

    crops16(big, wells_out, wells, 96, False, (WELL, WELL))()
    full_and_gather()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0 and torch.equal(wells_out.view(torch.int16).view(N, -1), gathered), "wells != gather"
    assert torch.equal(gathered, big["frames"].view(torch.int16).view(N, W * H)[:, idx]), "gather != source frames"

    # ---- 2304^2 and 1001x1003
    others = []
    for ow, oh in ((2304, 2304), (1001, 1003)):
        d = dataset(ow, oh)
        ofull = torch.empty(N * ow * oh, dtype=torch.uint16, device=dev)
        oout = torch.empty(N * ow * oh // 4 + N * oh + N * ow + 64, dtype=torch.uint16, device=dev)
        check_full(d, ofull)
        check_walk(d, oout)
        check_binned(d, oout, 2)
        check_binned(d, oout, 8)
        others.append((d, ofull, oout))
    checked = ("every output == torch on the source frames: decode16_device == the frames, each 256^2 crop == its slice, the "
               "96 wells == the torch gather == the frames' pixels, every binned output == the block mean of the in-frame "
               "pixels (2048^2 b = 2, 4, 8; 2304^2 and 1001x1003 b = 2, 8)")

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

    variants = [("decode16_device", full16(big, full))]
    if parent:
        variants.append(("parent decode16_device", full16(big, full, parent)))
    variants += [("decode16_crops_device 256^2 walk", crops16(big, out, big["d_walk"], 1, True, (CROP, CROP))),
                 ("decode16_crops_device 96 wells 120^2", crops16(big, wells_out, wells, 96, False, (WELL, WELL))),
                 ("decode16_device + torch gather of the wells", full_and_gather),
                 ("decode16_binned_device b=2", binned16(big, out, 2)), ("decode16_binned_device b=4", binned16(big, out, 4)),
                 ("decode16_binned_device b=8", binned16(big, out, 8))]
    for d, ofull, oout in others:
        tag = "%dx%d " % (d["W"], d["H"])
        variants += [(tag + "decode16_device", full16(d, ofull)),
                     (tag + "decode16_crops_device 256^2 walk", crops16(d, oout, d["d_walk"], 1, True, (CROP, CROP))),
                     (tag + "decode16_binned_device b=2", binned16(d, oout, 2)), (tag + "decode16_binned_device b=8", binned16(d, oout, 8))]
    times = {v[0]: [] for v in variants}
    for _ in range(a.rounds):
        for name, fn in variants:
            times[name].append(timeit(fn))
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0
    meta = dict(card(), frames=N, kind="sensor12", reps=a.reps, warmup=a.warmup, rounds=a.rounds, seed=42, checked=checked)
    med = {k: statistics.median(v) for k, v in times.items()}
    geo = {"decode16_device": (W, H, big["rec_bytes"])}
    for d, _, _ in others:
        geo["%dx%d " % (d["W"], d["H"])] = (d["W"], d["H"], d["rec_bytes"])
    lines = []
    for name, _ in variants:
        tag = name.split(" ")[0] + " " if name[0].isdigit() else ""
        w_, h_, rb = geo[tag] if tag else geo["decode16_device"]
        ref = tag + "decode16_device"
        line = dict(variant=name, ms=round(med[name], 4), ms_rounds=[round(x, 4) for x in times[name]], W=w_, H=h_,
                    record_bytes_per_frame=round(rb / N))
        if name != ref and not name.startswith("parent"):
            line["vs"] = ref
            line["x_vs"] = round(med[name] / med[ref], 4)
        if name == "decode16_device" and parent:
            line["x_parent"] = round(med[name] / med["parent decode16_device"], 4)
        if name == "decode16_crops_device 96 wells 120^2":
            line["x_decode16_device_plus_gather"] = round(med[name] / med["decode16_device + torch gather of the wells"], 4)
        lines.append(dict(line, **meta))

    # ---- host leg: pinned buffers, frames/s
    Nh = min(a.host_frames, N)
    stride = int(lib.dbde_b200_slot_stride16(W, H))
    slot_bytes = big["slots"][:N * stride].view(N, stride)
    rec_sizes = big["sizes"][:N].cpu().numpy().astype(np.int64)
    hoffs = np.zeros(Nh + 1, dtype=np.uint64)
    hoffs[1:] = np.cumsum(rec_sizes[:Nh])
    ps = codec.pinned(int(hoffs[Nh]))
    for i in range(Nh):
        ps.array[int(hoffs[i]):int(hoffs[i + 1])] = slot_bytes[i, :int(rec_sizes[i])].cpu().numpy()
    po, pst, pout, pc = codec.pinned(8 * Nh), codec.pinned(4 * Nh), codec.pinned(2 * Nh * W * H), codec.pinned(8 * Nh)
    po.array[:] = hoffs[:Nh].view(np.uint8)
    pc.array[:] = big["walk"][:Nh].view(np.uint8).ravel()

    def host_full():
        assert lib.dbde_b200_decode16_host(codec.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, pout.ptr, pst.ptr, None) == 0

    def host_crops():
        assert lib.dbde_b200_decode16_crops_host(codec.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, pc.ptr, 1, 1, CROP, CROP, 0,
                                                 pout.ptr, pst.ptr, None) == 0

    def host_binned():
        assert lib.dbde_b200_decode16_binned_host(codec.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, 2, pout.ptr, pst.ptr, None) == 0

    src = big["frames"][:Nh].cpu().numpy()
    host_crops()
    assert (pst.array.view(np.uint32) == 0).all()
    hc = pout.array[:2 * Nh * CROP * CROP].view(np.uint16).reshape(Nh, CROP, CROP)
    for i, (x0, y0) in enumerate(big["walk"][:Nh].tolist()):
        assert np.array_equal(hc[i], src[i, y0:y0 + CROP, x0:x0 + CROP]), ("host crop", i)
    host_binned()
    assert (pst.array.view(np.uint32) == 0).all()
    want = block_mean(big["frames"][:Nh], 2).cpu().numpy()
    assert np.array_equal(pout.array[:2 * want.size].view(np.uint16).reshape(want.shape), want), "host binned"
    host_full()
    assert (pst.array.view(np.uint32) == 0).all() and np.array_equal(pout.array.view(np.uint16).reshape(Nh, H, W), src), "host full"
    host = [("decode16_host", host_full), ("decode16_crops_host 256^2 walk", host_crops), ("decode16_binned_host b=2", host_binned)]
    ht = {n: [] for n, _ in host}
    for _ in range(a.rounds):
        for n, fn in host:
            t0 = time.perf_counter()
            for _ in range(a.host_reps):
                fn()
            ht[n].append(Nh * a.host_reps / (time.perf_counter() - t0))
    f_full = statistics.median(ht["decode16_host"])
    for n, _ in host:
        f = statistics.median(ht[n])
        lines.append(dict(dict(variant=n, frames_per_s=round(f, 1), fps_rounds=[round(x, 1) for x in ht[n]],
                               x_decode16_host=round(f / f_full, 3), host_frames=Nh, host_reps=a.host_reps, buffers="pinned",
                               W=W, H=H), **meta))
    for p in (ps, po, pst, pout, pc):
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
