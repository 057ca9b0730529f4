"""Region-of-interest decode against the full decode and the validation pre-pass, device-resident and through
host buffers.

    python scratch/roi_bench.py [--frames 1000] [--reps 20] [--warmup 3] [--rounds 3] [--out FILE]

The workload is bench.py's: 2048x2048 'micro' frames from the GPU generator with seed 42, encoded on the device
into fixed-stride slots.  Before anything is timed, every region's output is compared with the crop of the full
GPU decode of the same batch, and the full decode with the oracle's decode of sampled records.  Each variant is
timed with CUDA events over --reps launches after --warmup launches, in --rounds rounds (the median is reported,
the spread beside it).  One JSON line per variant on stdout (and in --out); the records (~1.6 GB) are larger
than L2, so every launch reads them from HBM.  Needs a GPU: without one it stops after parsing its arguments.
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

REGIONS = [("whole", None), ("1024x1024@517,301", (517, 301, 1024, 1024)), ("512x512@13,7", (13, 7, 512, 512)),
           ("256x256@1001,999", (1001, 999, 256, 256)), ("64x64@3,5", (3, 5, 64, 64)), ("column1x2048@777", (777, 0, 1, 2048)),
           ("row2048x1@1029", (0, 1029, 2048, 1))]


def parse():
    p = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    p.add_argument("--frames", type=int, default=1000)
    p.add_argument("--kind", default="micro")
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


def card():
    import torch
    name, limit = torch.cuda.get_device_name(0), None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        limit = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        pynvml.nvmlShutdown()
    except Exception as e:                      # noqa: BLE001 -- reported, not hidden
        limit = "unknown (%s)" % type(e).__name__
    return {"gpu": name, "power_limit_w": limit}


def main():
    a = parse()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("roi_bench.py: no CUDA device -- this measurement runs on the GPU only")
    pkg = importlib.import_module("dbce-video-cpp_b200")
    import oracle
    import synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    codec = pkg.Codec(0)
    N, W, H = a.frames, 2048, 2048
    w, h = W // 8, H // 8
    wh, px = w * h, W * H
    cap, stride = codec.stream_bound(W, H, N), codec.slot_stride(W, H)
    delta = (16 - (32 + 2 * wh) % 16) % 16
    frames = torch.empty(N * px, dtype=torch.uint8, device=dev)
    slots = torch.empty(cap + 64, dtype=torch.uint8, device=dev)
    full = torch.empty(N * px, dtype=torch.uint8, device=dev)
    roi_out = torch.empty(N * px, dtype=torch.uint8, device=dev)
    offs = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    sizes = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    status = torch.zeros(N, dtype=torch.int32, device=dev)
    cs = torch.cuda.current_stream().cuda_stream
    sp = slots.data_ptr() + delta
    synth.gen_frames_device(a.kind, N, W, H, frames.data_ptr(), seed=42, f0=0, stream=cs)
    codec.encode_device(frames.data_ptr(), W, H, 0, N, sp, cap, offs.data_ptr(), sizes.data_ptr(), cs)
    torch.cuda.synchronize()
    rec_sizes = sizes[:N].cpu().numpy().astype(np.int64)

    def full_decode():
        codec.decode_device(sp, cap, offs.data_ptr(), W, H, N, full.data_ptr(), status.data_ptr(), None, cs)

    import ctypes as C
    codec.lib.dbde_b200_validate_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                    C.c_void_p, C.c_void_p, C.c_void_p]

    def validate():
        codec.lib.dbde_b200_validate_device(codec.h, sp, cap, offs.data_ptr(), W, H, N, status.data_ptr(), None, cs)

    def roi_decode(r):
        r = r or (0, 0, W, H)
        return lambda: codec.decode_roi_device(sp, cap, offs.data_ptr(), W, H, N, r, roi_out.data_ptr(), status.data_ptr(),
                                               None, cs)

    # ---- correctness before timing
    full_decode()
    torch.cuda.synchronize()
    assert int(status.abs().sum()) == 0 and torch.equal(full, frames), "full decode != source frames"
    ora = oracle.best()
    slot_bytes = slots[delta:delta + N * stride].view(N, stride)
    for i in sorted({0, 1, N // 2, N - 1}):
        rec = slot_bytes[i, :int(rec_sizes[i])].cpu().numpy()
        n, hdr, img = ora.unpack_frame(rec, W, H)
        assert n == len(rec) and hdr[1] == i and np.array_equal(img, full[i * px:(i + 1) * px].view(H, W).cpu().numpy()), i
    fv = full.view(N, H, W)
    for name, r in REGIONS:
        x0, y0, rw, rh = r or (0, 0, W, H)
        roi_out.fill_(0xA5)
        roi_decode(r)()
        torch.cuda.synchronize()
        assert int(status.abs().sum()) == 0, name
        assert torch.equal(roi_out[:N * rw * rh].view(N, rh, rw), fv[:, y0:y0 + rh, x0:x0 + rw]), name
        assert bool((roi_out[N * rw * rh:] == 0xA5).all()), name
    checked = ("every region's output == crop of the full GPU decode of the batch; full decode == source frames and == "
               "%s decode of records %s" % ("reference" if oracle.ref is not None else "port", sorted({0, 1, N // 2, N - 1})))

    # ---- algorithmic bytes
    depth = slot_bytes[:, 24:24 + wh].view(N, h, w).to(torch.int64)
    total_rec = int(rec_sizes.sum())

    def roi_bytes(r):
        x0, y0, rw, rh = r or (0, 0, W, H)
        tx0, ty0, tx1, ty1 = x0 // 8, y0 // 8, (x0 + rw + 7) // 8, (y0 + rh + 7) // 8
        ntiles = (tx1 - tx0) * (ty1 - ty0)
        words = int(depth[:, ty0:ty1, tx0:tx1].sum())
        return N * wh + N * ntiles * 2 + 8 * words + N * rw * rh

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

    variants = [("decode_device", full_decode, total_rec + N * px), ("validate_device", validate, N * wh)]
    variants += [("decode_roi_device " + name, roi_decode(r), roi_bytes(r)) for name, r in REGIONS]
    times = {v[0]: [] for v in variants}
    for _ in range(a.rounds):                    # rounds interleave the variants
        for name, fn, _ in variants:
            times[name].append(timeit(fn))
    meta = dict(card(), frames=N, W=W, H=H, kind=a.kind, seed=42, reps=a.reps, warmup=a.warmup, rounds=a.rounds,
                record_bytes=total_rec, checked=checked)
    lines = []
    t_full = statistics.median(times["decode_device"])
    t_val = statistics.median(times["validate_device"])
    for name, _, nbytes in variants:
        t = statistics.median(times[name])
        lines.append(dict(variant=name, ms=round(t, 4), ms_rounds=[round(x, 4) for x in times[name]], algorithmic_bytes=nbytes,
                          gbs=round(nbytes / t / 1e6, 1), x_full_decode=round(t / t_full, 4), x_validate=round(t / t_val, 3),
                          **meta))

    # ---- host leg: pinned buffers, frames/s
    Nh = min(a.host_frames, N)
    hoffs = np.zeros(Nh + 1, dtype=np.uint64)
    hoffs[1:] = np.cumsum(rec_sizes[:Nh])
    ps = codec.pinned(int(hoffs[Nh]))
    for i in range(Nh):
        ps.array[int(hoffs[i]):int(hoffs[i + 1])] = slot_bytes[i, :int(rec_sizes[i])].cpu().numpy()
    po, pst = codec.pinned(8 * Nh), codec.pinned(4 * Nh)
    po.array[:] = hoffs[:Nh].view(np.uint8)
    pout = codec.pinned(Nh * px)

    def host_full():
        codec.decode_host_raw(ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, pout.ptr, pst.ptr, None)

    def host_roi(r):
        def fn():
            rc = codec.lib.dbde_b200_decode_roi_host(codec.h, ps.ptr, int(hoffs[Nh]), po.ptr, W, H, Nh, *r, pout.ptr, pst.ptr, None)
            assert rc == 0
        return fn

    host = [("decode_host", host_full)] + [("decode_roi_host " + n, host_roi(r)) for n, r in REGIONS if r and r[2] in (1024, 256)]
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
        lines.append(dict(variant=n, frames_per_s=round(f, 1), fps_rounds=[round(x, 1) for x in ht[n]],
                          x_decode_host=round(f / f_full, 3), host_frames=Nh, host_reps=a.host_reps, buffers="pinned", **meta))
    for p in (ps, po, pst, pout):
        p.free()
    codec.close()
    out = [json.dumps(x) for x in lines]
    print("\n".join(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
