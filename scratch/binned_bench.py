"""Binned decode against the full decode, and against the full decode followed by the pooling a user would write in torch.

    python scratch/binned_bench.py [--frames 1000] [--reps 20] [--warmup 3] [--rounds 3] [--out FILE]

The workload is bench.py's and scratch/crops_bench.py's: 2048x2048 'micro' frames from the GPU generator with seed 42,
encoded on the device into fixed-stride slots (~1.6 GB of records, larger than L2, so every launch reads them from
HBM), plus the same number of 1001x1003 'mix' frames (odd size: partial last bins in x and y).  Before anything is
timed, every binned output is compared with a numpy block mean of the full GPU decode of the same batch (which is
checked against the source frames), and the torch pooling with it too.  Device variants are timed with CUDA events
over --reps launches after --warmup launches, in --rounds rounds that interleave the variants (the median is reported,
the rounds beside it).  Host variants: frames/s over --host-reps calls on pinned buffers.  One JSON line per variant on
stdout (and in --out), each with the card's name and power limit.  Needs a GPU.
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

W = H = 2048
OW, OH = 1001, 1003


def parse():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--frames", type=int, default=1000)
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--host-frames", type=int, default=200, help="frames of the host-buffer leg")
    p.add_argument("--host-reps", type=int, default=5)
    p.add_argument("--out", default=None, help="also write the JSON lines here")
    a = p.parse_args()
    if a.reps < 20:
        p.error("--reps must be at least 20")
    return a


def block_mean(frames, b):
    """numpy reference: (N, H, W) -> (N, ceil(H / b), ceil(W / b)), the rounded mean of each block's in-frame pixels"""
    N, h, w = frames.shape
    hb, wb = -(-h // b), -(-w // b)
    p = np.zeros((N, hb * b, wb * b), np.uint32)
    p[:, :h, :w] = frames
    m = np.zeros((hb * b, wb * b), np.uint32)
    m[:h, :w] = 1
    s = p.reshape(N, hb, b, wb, b).sum(axis=(2, 4))
    n = m.reshape(hb, b, wb, b).sum(axis=(1, 3))
    return ((s + n // 2) // n).astype(np.uint8)


def block_means_248(frames):
    """the same for b = 2, 4, 8 of frames whose sides are multiples of 8, each level summing the one before"""
    s = frames.astype(np.uint16)
    out = {}
    for b in (2, 4, 8):
        s = s[:, 0::2, 0::2] + s[:, 0::2, 1::2] + s[:, 1::2, 0::2] + s[:, 1::2, 1::2]
        out[b] = ((s + b * b // 2) // (b * b)).astype(np.uint8)
    return out


def main():
    a = parse()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("binned_bench.py: no CUDA device -- this measurement runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    import synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    codec = pkg.Codec(0)
    N = a.frames
    cs = torch.cuda.current_stream().cuda_stream

    def dataset(kind, w, h):
        """frames, records in fixed-stride slots, offsets and sizes on the device"""
        px, wh = w * h, ((w + 7) // 8) * ((h + 7) // 8)
        cap = codec.stream_bound(w, h, N)
        delta = (16 - (32 + 2 * wh) % 16) % 16
        d = dict(w=w, h=h, px=px, cap=cap, delta=delta, stride=codec.slot_stride(w, h))
        d["frames"] = torch.empty(N * px, dtype=torch.uint8, device=dev)
        d["slots"] = torch.empty(cap + 64, dtype=torch.uint8, device=dev)
        d["offs"] = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        d["sizes"] = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        d["sp"] = d["slots"].data_ptr() + delta
        synth.gen_frames_device(kind, N, w, h, d["frames"].data_ptr(), seed=42, f0=0, stream=cs)
        codec.encode_device(d["frames"].data_ptr(), w, h, 0, N, d["sp"], cap, d["offs"].data_ptr(), d["sizes"].data_ptr(), cs)
        torch.cuda.synchronize()
        d["rec_sizes"] = d["sizes"][:N].cpu().numpy().astype(np.int64)
        return d

    micro = dataset("micro", W, H)
    full = torch.empty(N * W * H, dtype=torch.uint8, device=dev)
    out = torch.empty(N * W * H // 4 + 64, dtype=torch.uint8, device=dev)
    status = torch.zeros(N, dtype=torch.int32, device=dev)

    def full_decode(d=micro, dst=full):
        return lambda: codec.decode_device(d["sp"], d["cap"], d["offs"].data_ptr(), d["w"], d["h"], N, dst.data_ptr(),
                                           status.data_ptr(), None, cs)

    def binned(b, d=micro):
        return lambda: codec.decode_binned_device(d["sp"], d["cap"], d["offs"].data_ptr(), d["w"], d["h"], N, b, out.data_ptr(),
                                                  status.data_ptr(), None, cs)

    pooled = out[:N * (W // 2) * (H // 2)].view(N, H // 2, W // 2)

    def full_and_pool():
        """what a user writes today: the full decode, then 2x2 block sums, rounded half up, back to uint8"""
        full_decode()()
        s = full.view(N, H // 2, 2, W // 2, 2).sum(dim=(2, 4), dtype=torch.int32)
        pooled.copy_(((s + 2) // 4).to(torch.uint8))

    # ---- correctness before timing
    full_decode()()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0 and torch.equal(full, micro["frames"]), "full decode != source frames"
    got = {}
    for b in (2, 4, 8):
        nb = N * (W // b) * (H // b)
        out.fill_(0xA5)
        binned(b)()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0, b
        assert bool((out[nb:] == 0xA5).all()), ("wrote past the output", b)
        got[b] = out[:nb].cpu().numpy().reshape(N, H // b, W // b)
    full_and_pool()
    torch.cuda.synchronize()
    got["pool"] = pooled.cpu().numpy()
    step = 25
    for f0 in range(0, N, step):
        want = block_means_248(full[f0 * W * H:(f0 + step) * W * H].view(step, H, W).cpu().numpy())
        for b in (2, 4, 8):
            assert np.array_equal(got[b][f0:f0 + step], want[b]), ("micro binned", b, f0)
        assert np.array_equal(got["pool"][f0:f0 + step], want[2]), ("torch pooling", f0)
    del got

    odd = dataset("mix", OW, OH)
    ofull = torch.empty(N * OW * OH, dtype=torch.uint8, device=dev)
    full_decode(odd, ofull)()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0 and torch.equal(ofull, odd["frames"]), "odd full decode != source frames"
    ohb, owb = -(-OH // 2), -(-OW // 2)
    out.fill_(0xA5)
    binned(2, odd)()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0 and bool((out[N * ohb * owb:] == 0xA5).all())
    og = out[:N * ohb * owb].cpu().numpy().reshape(N, ohb, owb)
    for f0 in range(0, N, 100):
        assert np.array_equal(og[f0:f0 + 100], block_mean(ofull[f0 * OW * OH:(f0 + 100) * OW * OH].view(-1, OH, OW).cpu().numpy(), 2)), \
            ("odd binned", f0)
    del og, ofull
    checked = ("every binned output (micro-2048 b = 2, 4, 8; mix-1001x1003 b = 2) == numpy block mean of the full GPU decode, "
               "guard bytes past it untouched; torch pooling == the same; full decodes == source frames")

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

    odd_full = torch.empty(N * OW * OH, dtype=torch.uint8, device=dev)
    variants = [("decode_device", full_decode()),
                ("decode_binned_device b=2", binned(2)), ("decode_binned_device b=4", binned(4)), ("decode_binned_device b=8", binned(8)),
                ("decode_device + torch 2x2 pooling", full_and_pool),
                ("mix-1001x1003 decode_device", full_decode(odd, odd_full)),
                ("mix-1001x1003 decode_binned_device b=2", binned(2, odd))]
    times = {v[0]: [] for v in variants}
    for _ in range(a.rounds):
        for name, fn in variants:
            times[name].append(timeit(fn))
    del odd_full
    meta = dict(card(), frames=N, reps=a.reps, warmup=a.warmup, rounds=a.rounds, seed=42, checked=checked)
    med = {k: statistics.median(v) for k, v in times.items()}
    ref = {"decode_binned_device b=2": "decode_device", "decode_binned_device b=4": "decode_device",
           "decode_binned_device b=8": "decode_device", "decode_device + torch 2x2 pooling": "decode_device",
           "mix-1001x1003 decode_binned_device b=2": "mix-1001x1003 decode_device"}
    lines = []
    for name, _ in variants:
        geo = dict(W=OW, H=OH, kind="mix") if name.startswith("mix") else dict(W=W, H=H, kind="micro")
        line = dict(variant=name, ms=round(med[name], 4), ms_rounds=[round(x, 4) for x in times[name]], **geo)
        if name in ref:
            line["vs"] = ref[name]
            line["x_vs"] = round(med[name] / med[ref[name]], 4)
        if name == "decode_binned_device b=2":
            line["x_decode_device_plus_torch_pooling"] = round(med[name] / med["decode_device + torch 2x2 pooling"], 4)
        lines.append(dict(line, **meta))

    # ---- host leg: pinned buffers, frames/s
    Nh = min(a.host_frames, N)
    slot_bytes = micro["slots"][micro["delta"]:micro["delta"] + N * micro["stride"]].view(N, micro["stride"])
    rec_sizes = micro["rec_sizes"]
    hoffs = np.zeros(Nh + 1, dtype=np.uint64)
    hoffs[1:] = np.cumsum(rec_sizes[:Nh])
    ps = codec.pinned(int(hoffs[Nh]))
    for i in range(Nh):
        ps.array[int(hoffs[i]):int(hoffs[i + 1])] = slot_bytes[i, :int(rec_sizes[i])].cpu().numpy()
    po, pst, pout = codec.pinned(8 * Nh), codec.pinned(4 * Nh), codec.pinned(Nh * W * H)
    po.array[:] = hoffs[:Nh].view(np.uint8)

    def host_full():
        codec.decode_host_raw(ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, pout.ptr, pst.ptr, None)

    def host_binned(b):
        def fn():
            assert codec.lib.dbde_b200_decode_binned_host(codec.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, b, pout.ptr, pst.ptr,
                                                          None) == 0
        return fn

    host = [("decode_host", host_full), ("decode_binned_host b=2", host_binned(2)), ("decode_binned_host b=8", host_binned(8))]
    fv = full[:Nh * W * H].view(Nh, H, W).cpu().numpy()
    want = block_means_248(fv)
    for b in (2, 8):                                     # the host form's output before timing
        host_binned(b)()
        nb = Nh * (W // b) * (H // b)
        assert (pst.array.view(np.uint32) == 0).all()
        assert np.array_equal(pout.array[:nb].reshape(Nh, H // b, W // b), want[b]), ("host binned", b)
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
        lines.append(dict(dict(variant=n, frames_per_s=round(f, 1), fps_rounds=[round(x, 1) for x in ht[n]],
                               x_decode_host=round(f / f_full, 3), host_frames=Nh, host_reps=a.host_reps, buffers="pinned",
                               W=W, H=H, kind="micro"), **meta))
    for p in (ps, po, pst, pout):
        p.free()
    codec.close()
    text = [json.dumps(x) for x in lines]
    print("\n".join(text))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(text) + "\n")


if __name__ == "__main__":
    main()
