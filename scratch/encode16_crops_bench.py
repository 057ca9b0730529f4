"""DBDE16 crop encode against the gather-then-encode it replaces, the full-frame DBDE16 encoder, and the parent commit's
codec.

    python scratch/encode16_crops_bench.py [--frames 300] [--reps 20] [--warmup 3] [--rounds 3] [--parent-lib LIB] [--out FILE]

The workload is scratch/dbde16_subframe_bench.py's sensor12 content (a 12-bit camera-like smooth field plus 5 bits of
noise, seed 42) at 2048x2048, generated on the GPU: 300 frames are 2.5 GB in HBM, larger than L2.  Cases: 96 wells (a
12 x 8 grid of 120x120, shared corners) and one 256x256 crop per frame on a random walk of which about a quarter of the
crops lie partly outside the frame; the same walk kept inside the frame, and the walk on the first half of the frames,
show what bounds the walk (edge tiles, and records fewer than the resident CTAs).  The baselines are what a user
writes today: an index_select gather of the wells (through an int16 view: torch's uint16 support is limited) or a
clamped pad-gather of the walk, then encode16_device on the gathered crops.  2304x2304 and 1001x1003 batches of the same content give report rows for the full-frame encode and
the walk.  Before anything is timed, every crop record is compared byte for byte with oracle.port16's record of the
crop image, the baselines' records with the crop records (all bytes but the frame index, which the baselines number per
crop), and the full-frame encoder's first 20 records with the oracle's.  Device variants are timed with CUDA events
over --reps launches after --warmup launches, in --rounds rounds that interleave the variants (the median is reported,
the rounds beside it).  Host variants: frames/s over --host-reps calls on pinned buffers.

--parent-lib: a build of the parent commit's library (make -C dbce-video-cpp_b200/csrc OUT=... in a checkout of it).
Its encode16_device, encode16_host and the 8-bit encode_crops_device (96 wells of 2048x2048 'micro' frames) are timed in
the same process, alternating with this tree's.  One JSON line per variant on stdout (and in --out), each with the
card's name and power limit.  Needs a GPU.
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
    p.add_argument("--parent-lib", default=None, help="the parent commit's libdbde_b200.so, for the regression rows")
    p.add_argument("--out", default=None, help="also write the JSON lines here")
    a = p.parse_args()
    if a.reps < 20:
        p.error("--reps must be at least 20")
    return a


def walk(N, W, H, rng):
    """one random walk of N steps, rescaled twice: into [0, W - CROP] x [0, H - CROP] (every crop inside the frame),
    and into a range wider by 14 % of W - CROP on each side (at 2048^2, 250 pixels: a quarter of the crops partly
    outside the frame) -> two (N, 1, 2) int32 arrays"""
    w = np.cumsum(rng.integers(-24, 25, (N, 2)), axis=0).astype(np.float64)
    u = (w - w.min(axis=0)) / np.maximum(w.max(axis=0) - w.min(axis=0), 1)
    span = np.array([W, H]) - CROP
    m = np.round(0.14 * span)
    inside = np.round(u * span).astype(np.int32)
    edges = np.round(u * (span + 2 * m) - m).astype(np.int32)
    return inside.reshape(N, 1, 2), edges.reshape(N, 1, 2)


def parent_codec(pkg, codec, path):
    """a Codec on the parent commit's library, with only what the regression rows call bound (this build's
    signatures; pkg.load() would look up entry points that library does not have)"""
    import ctypes as C
    lib = C.CDLL(os.path.abspath(path))
    for name in ("dbde_b200_create", "dbde_b200_destroy", "dbde_b200_last_error", "dbde_b200_encode16_device",
                 "dbde_b200_encode16_host", "dbde_b200_encode_crops_device"):
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
        raise SystemExit("encode16_crops_bench.py: no CUDA device -- this measurement runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    import oracle
    import synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    codec = pkg.Codec(0)
    parent = parent_codec(pkg, codec, a.parent_lib) if a.parent_lib else None
    lib = codec.lib
    N = a.frames
    cs = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(2026)
    wells = np.array([(64 + 160 * i, 64 + 240 * j) for j in range(8) for i in range(12)], dtype=np.int32)
    checked = []

    def stride16(w, h):
        return int(lib.dbde_b200_slot_stride16(w, h))

    def dataset(W, H):
        """sensor12 frames on the device (an int16 view beside them), slots for the full-frame encode, the walk"""
        g = torch.Generator(device=dev)
        g.manual_seed(42)
        y = torch.arange(H, device=dev).view(1, H, 1)
        x = torch.arange(W, device=dev).view(1, 1, W)
        fr = (600 + x // 16 + y // 8 + torch.randint(0, 32, (N, H, W), device=dev, generator=g, dtype=torch.int32)).to(torch.int32)
        d = dict(W=W, H=H, frames=fr.to(torch.uint16).contiguous())
        del fr
        d["i16"] = d["frames"].view(torch.int16)
        d["cap"] = stride16(W, H) * N
        d["slots"] = torch.empty(d["cap"] + 64, dtype=torch.uint8, device=dev)
        d["inside"], d["walk"] = walk(N, W, H, rng)
        d["partly_out"] = float(np.mean(((d["walk"][:, 0] < 0) | (d["walk"][:, 0] > np.array([W, H]) - CROP)).any(axis=1)))
        return d

    offs = torch.zeros(N * len(wells) + 1, dtype=torch.int64, device=dev)
    sizes = torch.zeros(N * len(wells) + 1, dtype=torch.int64, device=dev)

    def enc_full(d, c=codec):
        return lambda: c._ck(c.lib.dbde_b200_encode16_device(c.h, d["frames"].data_ptr(), d["W"], d["H"], 0, N, d["slots"].data_ptr(),
                                                             d["cap"], 0, offs.data_ptr(), sizes.data_ptr(), cs), "encode16_device")

    class Case:
        """crops of one dataset: corners (R, 2) shared or (N, R, 2) per frame, the crop slots, the gathered crop images,
        the baseline's slots"""
        def __init__(self, d, corners, size):
            self.d, self.corners, (self.cw, self.ch) = d, corners, size
            self.R = corners.shape[-2]
            self.n = N * self.R
            self.st = stride16(*size)
            self.dc = torch.from_numpy(corners.reshape(-1, 2).copy()).to(dev)
            self.buf = torch.empty(self.n * self.st + 64, dtype=torch.uint8, device=dev)
            self.gbuf = torch.empty(self.n * self.st + 64, dtype=torch.uint8, device=dev)
            self.img = torch.empty(self.n * self.cw * self.ch, dtype=torch.int16, device=dev)
            cw, ch, W, H = self.cw, self.ch, d["W"], d["H"]
            if corners.ndim == 2:            # shared corners inside the frame: one index_select over every frame
                self.idx = torch.from_numpy(np.concatenate([((y0 + np.arange(ch))[:, None] * W + x0 + np.arange(cw)[None, :]).ravel()
                                                            for x0, y0 in corners])).to(dev)
            else:                            # per-frame corners anywhere: clamped index + in-frame mask
                xs = torch.from_numpy(corners[:, 0, 0].astype(np.int64)).to(dev)[:, None, None] + torch.arange(cw, device=dev)[None, None, :]
                ys = torch.from_numpy(corners[:, 0, 1].astype(np.int64)).to(dev)[:, None, None] + torch.arange(ch, device=dev)[None, :, None]
                self.inside = ((xs >= 0) & (xs < W) & (ys >= 0) & (ys < H)).reshape(-1)
                self.pidx = (torch.arange(N, device=dev)[:, None, None] * W * H + ys.clamp(0, H - 1) * W + xs.clamp(0, W - 1)).reshape(-1)
                self.pad0 = torch.zeros((), dtype=torch.int16, device=dev)

        def crops(self, nf=N):
            d = self.d
            return lambda: codec.encode16_crops_device(d["frames"].data_ptr(), d["W"], d["H"], 0, nf, self.dc.data_ptr(), self.R,
                                                       self.corners.ndim == 3, (self.cw, self.ch), self.buf.data_ptr(), self.n * self.st,
                                                       offs.data_ptr(), sizes.data_ptr(), 0, cs)

        def gather(self):
            if self.corners.ndim == 2:
                torch.index_select(self.d["i16"].view(N, -1), 1, self.idx, out=self.img.view(N, -1))
            else:
                torch.where(self.inside, torch.take(self.d["i16"], self.pidx), self.pad0, out=self.img)

        def contig(self):
            return lambda: codec._ck(lib.dbde_b200_encode16_device(codec.h, self.img.data_ptr(), self.cw, self.ch, 0, self.n,
                                                                   self.gbuf.data_ptr(), self.n * self.st, 0, offs.data_ptr(),
                                                                   sizes.data_ptr(), cs), "encode16_device")

        def gather_and_encode(self):
            e = self.contig()

            def fn():
                self.gather()
                e()
            return fn

        def records(self, buf):
            torch.cuda.synchronize()
            sz = sizes[:self.n].cpu().numpy().astype(np.int64)
            host = buf[:self.n * self.st].cpu().numpy().reshape(self.n, self.st)
            return [host[j, :sz[j]] for j in range(self.n)]

        def check(self, tag):
            """every crop record == the oracle's record of the gathered crop image; the baseline's records == them
            but for the index"""
            self.gather()
            self.buf.fill_(0xA5)
            self.crops()()
            got = self.records(self.buf)
            assert bool((self.buf[self.n * self.st:] == 0xA5).all()), tag
            imgs = self.img.view(N, self.R, self.ch, self.cw).cpu().numpy().view(np.uint16)
            for r in range(self.R):
                s, sz = oracle.port16.pack_frames(imgs[:, r], 0)
                o = np.concatenate([[0], np.cumsum(sz)]).astype(np.int64)
                for f in range(N):
                    assert np.array_equal(got[f * self.R + r], s[o[f]:o[f + 1]]), (tag, f, r)
            self.contig()()
            base = self.records(self.gbuf)
            drop = lambda rec: np.concatenate([rec[:4], rec[12:]])        # noqa: E731
            assert all(np.array_equal(drop(x), drop(y)) for x, y in zip(base, got)), tag
            checked.append("%s: %d crop records == oracle.port16; gather + encode16_device records == them but for the index"
                           % (tag, self.n))

    def check_full(d, c=codec, tag=""):
        d["slots"].fill_(0)
        enc_full(d, c)()
        torch.cuda.synchronize()
        st = stride16(d["W"], d["H"])
        sz = sizes[:20].cpu().numpy().astype(np.int64)
        s, wsz = oracle.port16.pack_frames(d["frames"][:20].cpu().numpy(), 0)
        o = np.concatenate([[0], np.cumsum(wsz)]).astype(np.int64)
        host = d["slots"][:20 * st].cpu().numpy().reshape(20, st)
        assert all(np.array_equal(host[f, :sz[f]], s[o[f]:o[f + 1]]) for f in range(20)), (tag, d["W"])
        checked.append("%s%dx%d encode16_device: first 20 records == oracle.port16" % (tag, d["W"], d["H"]))

    # ---- 2048^2: correctness before timing
    big = dataset(2048, 2048)
    cw_ = Case(big, wells, (WELL, WELL))
    cwalk = Case(big, big["walk"], (CROP, CROP))
    cw_.check("2048x2048 wells")
    cwalk.check("2048x2048 walk")
    cin = Case(big, big["inside"], (CROP, CROP))
    cin.check("2048x2048 walk inside the frame")
    check_full(big)
    if parent:
        check_full(big, parent, "parent ")
    # the clamped pad-gather is the crop image: a few frames against numpy
    wi = cwalk.img.view(N, CROP, CROP)
    for f in (0, N // 2, N - 1):
        x0, y0 = (int(v) for v in big["walk"][f, 0])
        ref = np.zeros((CROP, CROP), np.int16)
        xa, xb, ya, yb = max(x0, 0), min(x0 + CROP, 2048), max(y0, 0), min(y0 + CROP, 2048)
        ref[ya - y0:yb - y0, xa - x0:xb - x0] = big["i16"][f, ya:yb, xa:xb].cpu().numpy()
        assert np.array_equal(wi[f].cpu().numpy(), ref), f
    # the 8-bit crop encode on 8-bit frames, for its regression row
    f8 = torch.empty(N * 2048 * 2048, dtype=torch.uint8, device=dev)
    synth.gen_frames_device("micro", N, 2048, 2048, f8.data_ptr(), seed=42, f0=0, stream=cs)
    st8 = codec.slot_stride(WELL, WELL)
    buf8 = torch.empty(N * len(wells) * st8 + 64, dtype=torch.uint8, device=dev)
    dw8 = torch.from_numpy(wells.reshape(-1).copy()).to(dev)

    def enc_crops8(c=codec):
        return lambda: c._ck(c.lib.dbde_b200_encode_crops_device(c.h, f8.data_ptr(), 2048, 2048, 0, N, dw8.data_ptr(), len(wells), 0,
                                                                 WELL, WELL, 0, buf8.data_ptr(), N * len(wells) * st8, 0, offs.data_ptr(),
                                                                 sizes.data_ptr(), cs), "encode_crops_device")
    if parent:
        enc_crops8()()
        torch.cuda.synchronize()
        mine = buf8.clone()
        enc_crops8(parent)()
        torch.cuda.synchronize()
        assert torch.equal(mine, buf8), "encode_crops_device differs from the parent's"
        checked.append("encode_crops_device (8-bit, 96 wells) == the parent build's, byte for byte")
        del mine

    # ---- 2304^2 and 1001x1003: the full-frame encode and the walk
    others = []
    for ow, oh in ((2304, 2304), (1001, 1003)):
        d = dataset(ow, oh)
        c = Case(d, d["walk"], (CROP, CROP))
        c.check("%dx%d walk" % (ow, oh))
        check_full(d)
        others.append((d, c))

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
    variants = [("encode16_device", enc_full(big))] + ([("parent encode16_device", enc_full(big, parent))] if parent else [])
    variants += [("encode_crops_device 8-bit 96 wells", enc_crops8())] + \
        ([("parent encode_crops_device 8-bit 96 wells", enc_crops8(parent))] if parent else [])
    variants += [("encode16_crops_device 96 wells 120x120 shared", cw_.crops()),
                 ("int16 index_select gather of the wells + encode16_device", cw_.gather_and_encode()),
                 ("encode16_crops_device 256x256 walk", cwalk.crops()),
                 ("clamped pad-gather of the walk + encode16_device", cwalk.gather_and_encode()),
                 ("encode16_device of the walk's crops, contiguous", cwalk.contig()),
                 ("encode16_crops_device 256x256 walk inside the frame", cin.crops()),
                 ("encode16_crops_device 256x256 walk, first %d frames" % (N // 2), cwalk.crops(N // 2))]
    for d, c in others:
        tag = "%dx%d " % (d["W"], d["H"])
        variants += [(tag + "encode16_device", enc_full(d)), (tag + "encode16_crops_device 256x256 walk", c.crops()),
                     (tag + "clamped pad-gather of the walk + encode16_device", c.gather_and_encode()),
                     (tag + "encode16_device of the walk's crops, contiguous", c.contig())]
    times = {v[0]: [] for v in variants}
    for _ in range(a.rounds):
        for name, fn in variants:
            times[name].append(timeit(fn))
    med = {k: statistics.median(v) for k, v in times.items()}
    meta = dict(card(), frames=N, kind="sensor12", seed=42, reps=a.reps, warmup=a.warmup, rounds=a.rounds)
    vs = {"encode16_crops_device 96 wells 120x120 shared": ["int16 index_select gather of the wells + encode16_device", "encode16_device"],
          "encode16_crops_device 256x256 walk": ["clamped pad-gather of the walk + encode16_device",
                                                 "encode16_device of the walk's crops, contiguous"],
          "encode16_crops_device 256x256 walk inside the frame": ["encode16_device of the walk's crops, contiguous"],
          "encode16_device": ["parent encode16_device"],
          "encode_crops_device 8-bit 96 wells": ["parent encode_crops_device 8-bit 96 wells"]}
    for d, _ in others:
        tag = "%dx%d " % (d["W"], d["H"])
        vs[tag + "encode16_crops_device 256x256 walk"] = [tag + "clamped pad-gather of the walk + encode16_device",
                                                           tag + "encode16_device of the walk's crops, contiguous", tag + "encode16_device"]
    lines = []
    for name, _ in variants:
        W_, H_ = (2304, 2304) if name.startswith("2304") else (1001, 1003) if name.startswith("1001") else (2048, 2048)
        line = dict(variant=name, ms=round(med[name], 4), ms_rounds=[round(x, 4) for x in times[name]], W=W_, H=H_)
        for i, ref in enumerate(vs.get(name, [])):
            if ref in med:
                line["vs%d" % (i + 1)] = ref
                line["x_vs%d" % (i + 1)] = round(med[name] / med[ref], 4)
        if "walk" in name and "inside" not in name:
            line["crops_partly_outside"] = round(dict([(2048, big)] + [(d["W"], d) for d, _ in others])[W_]["partly_out"], 3)
        lines.append(dict(line, **meta))

    # ---- host leg: pinned buffers, frames/s
    Nh = min(a.host_frames, N)
    W = H = 2048
    pfr = codec.pinned(Nh * W * H * 2)
    pfr.array[:] = big["frames"][:Nh].cpu().numpy().view(np.uint8).ravel()
    hcap = stride16(W, H) * Nh + 16
    wcap = stride16(WELL, WELL) * Nh * len(wells) + 16
    pout, pwout = codec.pinned(hcap), codec.pinned(wcap)
    poff, pwoff = codec.pinned(8 * (Nh + 1)), codec.pinned(8 * (Nh * len(wells) + 1))

    def host_full(c):
        def fn():
            assert c.lib.dbde_b200_encode16_host(c.h, pfr.ptr, W, H, 0, Nh, pout.ptr, hcap, poff.ptr) == 0
        return fn

    def host_wells():
        assert lib.dbde_b200_encode16_crops_host(codec.h, pfr.ptr, W, H, 0, Nh, wells.ctypes.data, len(wells), 0, WELL, WELL, 0,
                                                 pwout.ptr, wcap, pwoff.ptr) == 0

    host = [("encode16_host", host_full(codec)), ("encode16_crops_host 96 wells 120x120 shared", host_wells)]
    if parent:
        host.append(("parent encode16_host", host_full(parent)))
    host_wells()                                     # the host form's bytes == the device form's records back to back
    cw_.crops()()
    got = cw_.records(cw_.buf)[:Nh * len(wells)]
    tot = int(pwoff.array.view(np.uint64)[Nh * len(wells)])
    assert np.array_equal(pwout.array[:tot], np.concatenate(got)), "encode16_crops_host != encode16_crops_device"
    checked.append("encode16_crops_host (%d frames) == encode16_crops_device's records back to back" % Nh)
    if parent:
        host_full(codec)()
        mine = pout.array[:int(poff.array.view(np.uint64)[Nh])].copy()
        host_full(parent)()
        assert np.array_equal(mine, pout.array[:int(poff.array.view(np.uint64)[Nh])]), "encode16_host differs from the parent's"
        checked.append("encode16_host == the parent build's, byte for byte")
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
    f_full = statistics.median(ht["encode16_host"])
    for n, _ in host:
        f = statistics.median(ht[n])
        line = dict(variant=n, frames_per_s=round(f, 1), fps_rounds=[round(x, 1) for x in ht[n]], x_encode16_host=round(f / f_full, 4),
                    host_frames=Nh, host_reps=a.host_reps, buffers="pinned", W=W, H=H)
        if n == "encode16_host" and parent:
            line["x_parent_fps"] = round(f / statistics.median(ht["parent encode16_host"]), 4)
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
