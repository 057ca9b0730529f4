#!/usr/bin/env python
"""DBDE encode+decode benchmark on B200 (the contract in the task statement, tier framing (4)).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA, sm_100a)
  python bench.py --impl reference [...]                          the reference's CPU path
  python bench.py [...] --dump-outputs DIR                        also save the last timed step's results

Workload (BASELINE.json configs[1]): 2048x2048 U8 synthetic microscopy-like video, 1000 frames per
GPU; one STEP = encode the whole batch, then decode it again (device-resident).  Metric: raw-pixel
GB/s = pixels encoded + pixels decoded per second (2 * frames * W * H / step time), summed over
GPUs; frames/s for each direction are reported next to it.  Frames are independent, so N GPUs
take N disjoint frame ranges (weak scaling: 1000 frames each) with no data-path collective;
torch.distributed (NCCL) is used only for the timing barrier and the max over ranks.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # no __pycache__ either: the benchmark writes nothing into the source tree

METRIC = "dbde_encode_decode_raw_pixel_throughput"
UNIT = "GB/s"
W = H = 2048
KIND = "micro"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=1000, help="frames per GPU per step")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames per GPU in the end-to-end leg (0 = all that can be pinned)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip BASELINE configs 3 and 4 (run device-resident after the headline)")
    ap.add_argument("--extra-steps", type=int, default=10)
    ap.add_argument("--kind", default=KIND, choices=["micro", "mix", "low", "noise"])
    ap.add_argument("--width", type=int, default=W)
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed on rank 0 as DIR/*.npy: record "
                         "sizes, offsets, decode status, and a fixed seeded sample of record bytes and decoded pixels")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def workload_config(a, extra=None):
    cfg = {"workload": "%dx%d U8 synthetic '%s' video (SURVEY 8d, seed 42), %d frames per GPU, encode+decode per step"
                       % (a.width, a.height, a.kind, a.frames),
           "frames_per_gpu": a.frames, "width": a.width, "height": a.height, "generator": a.kind,
           "sharding": "contiguous frame ranges per GPU, no collective",
           "l2": "inputs (%.1f GB per direction) exceed the 126 MB L2; no explicit flush"
                 % (a.frames * a.width * a.height / 1e9)}
    if extra:
        cfg.update(extra)
    return cfg


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML as fast as the calls return (~1 ms; power
    every 8th sample) on a thread -- the timed region is tens to hundreds of milliseconds, which
    nvidia-smi -lms cannot resolve.  stop(t0, t1) keeps only the samples taken inside the timed
    region [t0, t1] (time.perf_counter)."""

    def __init__(self, index):
        import threading
        self.samples = []
        self.ok = False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        power, k = 0.0, 0
        while not self._stop.is_set():
            try:
                if k % 8 == 0:
                    power = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                k += 1
                self.samples.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM), power,
                                     nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:
                pass
            time.sleep(0.0005)

    def stop(self, t0, t1):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.ok:
            return out
        self._stop.set()
        self.t.join(timeout=2)
        nv = self.nv
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples[-3:]
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        reasons = sorted(n for n, b in bits.items() if any(s[3] & b for s in inside))
        if inside:
            out.update(sm_mhz=float(np.median([s[1] for s in inside])), sm_max_mhz=float(self.max_mhz), reasons=reasons,
                       samples=len(inside), power_w_max=max(s[2] for s in inside))
        return out


# ------------------------------------------------------------------------------------------ CPU arm
# what cpu_baseline.kind stands for; only "reference" is the reference's own speed
CPU_CODECS = {
    "reference": "dbde_pack_frame/dbde_unpack_frame of the unmodified dbde_util.cpp (g++ -O3 -march=corei7, SSE4.1) "
                 "via oracle/_ref",
    "port": "oracle_pack_frame/oracle_unpack_frame of the plain-C port oracle/dbde_oracle.c (oracle/_ref is not built): "
            "a bit-at-a-time restatement far slower than the reference, not a baseline to quote speed-ups against",
}


def cpu_reference_rates(frames, threads, target_s=1.0):
    """Time the reference's own CPU implementation (oracle/_ref: dbde_util.cpp compiled unmodified;
    where that is not built, the plain-C port oracle/dbde_oracle.c, reported as kind "port") on
    `threads` host threads over contiguous frame ranges.  -> dict of rates."""
    import oracle
    if oracle.ref is not None:
        encode_mt, decode_mt, kind = oracle.ref_encode_mt, oracle.ref_decode_mt, "reference"
    else:
        encode_mt, decode_mt, kind = oracle.port_encode_mt, oracle.port_decode_mt, "port"
    n, Hh, Ww = frames.shape
    # calibrate repetitions so each direction runs for about target_s
    s, slots, sizes = encode_mt(frames, threads, 1)
    reps_e = max(1, int(target_s / max(s, 1e-4)))
    s_e, slots, sizes = encode_mt(frames, threads, reps_e)
    s, dec, bad = decode_mt(slots, Ww, Hh, threads, 1)
    reps_d = max(1, int(target_s / max(s, 1e-4)))
    s_d, dec, bad = decode_mt(slots, Ww, Hh, threads, reps_d)
    assert bad == 0 and (dec == frames).all(), "%s round trip failed" % kind
    enc_fps, dec_fps = n * reps_e / s_e, n * reps_d / s_d
    px = Ww * Hh
    t_pair = 1.0 / enc_fps + 1.0 / dec_fps            # seconds to encode AND decode one frame
    return {"encode_fps": enc_fps, "decode_fps": dec_fps, "value": 2 * px / t_pair / 1e9, "kind": kind,
            "cpu_seconds": threads * (s_e + s_d), "reps": [reps_e, reps_d], "sizes": sizes}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import synth
    threads = os.cpu_count() or 1
    nsample = min(a.frames, 64)
    frames = synth.gen_frames(a.kind, nsample, a.width, a.height)
    per = []
    for _ in range(a.warmup):
        cpu_reference_rates(frames, threads, target_s=0.2)
    t0 = time.time()
    target = max(0.1, min(0.5, 15.0 / max(a.steps, 1)))       # ~30 s of timed CPU work in total, whatever K is
    for _ in range(a.steps):
        per.append(cpu_reference_rates(frames, threads, target_s=target))
    wall = time.time() - t0
    val = float(np.mean([p["value"] for p in per]))
    enc = float(np.mean([p["encode_fps"] for p in per]))
    dec = float(np.mean([p["decode_fps"] for p in per]))
    kind = per[0]["kind"]
    sample = "%d frames of the same workload, ~%.2f s per direction per step" % (nsample, target)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1000.0 * wall / max(a.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(a), "encode_fps": enc, "decode_fps": dec,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "%s; %d host threads over contiguous frame ranges; host only, no GPU" % (CPU_CODECS[kind], threads)}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ our arm
class DeviceLeg:
    """One workload resident in HBM: frames, record slots, decoded frames.  encode()/decode() are the two
    launches of a step; gate() is the parity check that precedes any timing."""

    def __init__(self, torch, synth, codec, dev, kind, Ww, Hh, N, f0):
        self.torch, self.codec, self.dev = torch, codec, dev
        self.kind, self.W, self.H, self.N, self.f0 = kind, Ww, Hh, N, f0
        self.px = Ww * Hh
        self.wh = ((Ww + 7) // 8) * ((Hh + 7) // 8)
        self.cap = codec.stream_bound(Ww, Hh, N)
        self.stride = codec.slot_stride(Ww, Hh)
        self.frames = torch.empty(N * self.px + 64, dtype=torch.uint8, device=dev)
        self.stream_buf = torch.empty(self.cap + 64, dtype=torch.uint8, device=dev)
        self.decoded = torch.empty(N * self.px + 64, dtype=torch.uint8, device=dev)
        self.offs = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        self.sizes = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        self.status = torch.zeros(N, dtype=torch.int32, device=dev)
        self.delta = (16 - (32 + 2 * self.wh) % 16) % 16       # puts every frame's U64 words on 8/16-byte boundaries
        self.out_ptr = self.stream_buf.data_ptr() + self.delta
        self.cs = torch.cuda.current_stream().cuda_stream
        synth.gen_frames_device(kind, N, Ww, Hh, self.frames.data_ptr(), seed=42, f0=f0, stream=self.cs)
        torch.cuda.synchronize()

    def encode(self):
        self.codec.encode_device(self.frames.data_ptr(), self.W, self.H, self.f0, self.N, self.out_ptr, self.cap,
                                 self.offs.data_ptr(), self.sizes.data_ptr(), self.cs)

    def decode(self):
        # the decoder reads each record from its slot (offs[i] = i * slot_stride)
        self.codec.decode_device(self.out_ptr, self.cap, self.offs.data_ptr(), self.W, self.H, self.N,
                                 self.decoded.data_ptr(), self.status.data_ptr(), None, self.cs)

    def gate(self, threads):
        """Parity before timing: decode(encode(x)) == x, and EVERY record byte-identical to what the
        reference's dbde_pack_frame writes for the same frame (oracle/_ref when it is there, else the port
        on a sample).  -> (total record bytes, algorithmic bytes per launch, description of the check)"""
        torch, N, px, wh = self.torch, self.N, self.px, self.wh
        self.encode()
        torch.cuda.synchronize()
        sizes = self.sizes[:N].cpu().numpy().astype(np.int64)
        total = int(sizes.sum())
        self.decode()
        torch.cuda.synchronize()
        assert int(self.status.abs().sum().item()) == 0, "decode rejected frames"
        assert torch.equal(self.frames[:N * px], self.decoded[:N * px]), "decode(encode(x)) != x"
        import oracle
        slots = self.stream_buf[self.delta:self.delta + N * self.stride].view(N, self.stride)
        frames = self.frames[:N * px].view(N, self.H, self.W)
        step = max(1, min(N, (256 << 20) // max(px, 1)))
        checked = 0
        if oracle.ref is not None:
            for a in range(0, N, step):
                b = min(N, a + step)
                fr = frames[a:b].cpu().numpy()
                _, want, wsz = oracle.ref_encode_mt(fr, threads, 1)        # the reference writes index i - a
                got = slots[a:b].cpu().numpy()
                assert (wsz.astype(np.int64) == sizes[a:b]).all(), "record sizes differ from the reference"
                for i in range(b - a):
                    n = int(sizes[a + i])
                    assert got[i, :4].tobytes() == want[i, :4].tobytes() and got[i, 12:n].tobytes() == want[i, 12:n].tobytes(), \
                        "record %d differs from the reference" % (a + i)
                    assert int(got[i, 4:12].view(np.uint64)[0]) == self.f0 + a + i, "frame index field"
                checked += b - a
            how = "all %d records byte-identical to the unmodified reference (oracle/_ref), round trip exact" % checked
        else:
            ns = min(N, 4)
            want, wsz = oracle.port.pack_frames(frames[:ns].cpu().numpy(), self.f0)
            got = np.concatenate([slots[i, :int(sizes[i])].cpu().numpy() for i in range(ns)])
            assert np.array_equal(got, want), "records differ from the oracle port"
            how = "first %d records byte-identical to the oracle port (oracle/_ref absent), round trip exact" % ns
        n64_total = (total - N * (32 + 2 * wh)) // 8
        alg = N * px + 2 * N * wh + 8 * n64_total            # per launch, same both directions (SURVEY 8d)
        return total, alg, how

    def timed(self, steps, warmup, barrier):
        """`warmup` untimed steps, then EXACTLY `steps` timed ones (CUDA events on the launching stream)."""
        torch = self.torch
        for _ in range(warmup):
            self.encode(); self.decode()
        barrier()
        l0 = self.codec.launches()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        start.record()
        for k in range(steps):
            ev[k][0].record()
            self.encode()
            ev[k][1].record()
            self.decode()
            ev[k][2].record()
        end.record()
        barrier()
        t1 = time.perf_counter()
        return {"elapsed_ms": start.elapsed_time(end), "launches": self.codec.launches() - l0, "t_host": (t0, t1),
                "enc_ms": float(np.mean([e[0].elapsed_time(e[1]) for e in ev])),
                "dec_ms": float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))}

    def dump(self, out_dir):
        """Save what the last encode()/decode() handed back as out_dir/<name>.npy.  Per frame (frames
        per_frame_index, all of them up to 2^19): record_sizes, record_offsets, decode_status (float64).  For
        8 frames (sample_frame_index): record_bytes_sample at 2^19 byte positions of the slot
        (sample_byte_position; -1 past the record's end) and decoded_pixels_sample at 2^19 pixel positions
        (sample_pixel_position), float32.  The indices are drawn with a fixed seed from the shape alone, so
        two runs with the same arguments compare entry by entry; at most 56 MB in all."""
        torch, N, px, stride = self.torch, self.N, self.px, self.stride
        rng = np.random.default_rng(20261020)

        def pick(n, k):
            return np.arange(n) if n <= k else np.sort(rng.choice(n, k, replace=False))

        every, frames, bpos, ppos = pick(N, 1 << 19), pick(N, 8), pick(stride, 1 << 19), pick(px, 1 << 19)
        sizes = self.sizes[:N].cpu().numpy()
        fi = torch.from_numpy(frames).to(self.dev)
        slots = self.stream_buf[self.delta:self.delta + N * stride].view(N, stride)
        rec = slots.index_select(0, fi).index_select(1, torch.from_numpy(bpos).to(self.dev)).cpu().numpy().astype(np.float32)
        rec[bpos[None, :] >= sizes[frames][:, None]] = -1
        dec = self.decoded[:N * px].view(N, px).index_select(0, fi).index_select(1, torch.from_numpy(ppos).to(self.dev))
        os.makedirs(out_dir, exist_ok=True)
        for name, arr in (("per_frame_index", every), ("record_sizes", sizes[every]),
                          ("record_offsets", self.offs[:N].cpu().numpy()[every]),
                          ("decode_status", self.status[:N].cpu().numpy()[every]),
                          ("sample_frame_index", frames), ("sample_byte_position", bpos), ("sample_pixel_position", ppos),
                          ("record_bytes_sample", rec), ("decoded_pixels_sample", dec.cpu().numpy().astype(np.float32))):
            np.save(os.path.join(out_dir, name + ".npy"), arr if arr.dtype == np.float32 else arr.astype(np.float64))

    def free(self):
        self.frames = self.stream_buf = self.decoded = None


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_ours(a):
    import torch
    import torch.distributed as dist
    import synth
    pkg = importlib.import_module("dbce-video-cpp_b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the DBDE B200 codec has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    codec = pkg.Codec(local)
    Ww, Hh, N = a.width, a.height, a.frames
    px = Ww * Hh
    shard = importlib.import_module("dbce-video-cpp_b200.shard")
    f0, f1 = shard.frame_range(rank, world, world * N)     # this GPU's contiguous frame range (weak scaling: N each)
    assert f1 - f0 == N
    host_threads = max(1, (os.cpu_count() or 1) // world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident buffers (torch owns the device memory; the codec gets raw pointers), parity gate
    leg = DeviceLeg(torch, synth, codec, dev, a.kind, Ww, Hh, N, f0)
    total, alg_bytes, gate_how = leg.gate(host_threads)
    frames, decoded, sizes, stream_buf = leg.frames, leg.decoded, leg.sizes, leg.stream_buf

    # ---- warm-up, then EXACTLY K timed steps
    sampler = ClockSampler(local) if rank == 0 else None
    tm = leg.timed(a.steps, a.warmup, barrier)
    clocks = sampler.stop(*tm["t_host"]) if sampler else None
    if a.dump_outputs and rank == 0:
        leg.dump(a.dump_outputs)        # before the end-to-end leg below reuses the device buffers
    launches, enc_ms, dec_ms = tm["launches"], tm["enc_ms"], tm["dec_ms"]
    t = torch.tensor([tm["elapsed_ms"], enc_ms, dec_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, enc_ms_max, dec_ms_max = [float(x) for x in t.tolist()]
    ms_per_step = elapsed_ms / a.steps
    value = world * 2 * N * px / (ms_per_step * 1e-3) / 1e9

    # ---- end to end through the C ABI with HOST buffers (pinned), copies inside the timed region.
    # A step is still "encode N frames + decode N frames", but the two directions run CONCURRENTLY on
    # two contexts driven by two host threads (the C ABI's contract: one context per thread), so the
    # encoder's H2D of raw frames overlaps the decoder's D2H of raw frames on the full-duplex PCIe
    # link.  Step k decodes the stream step k-1 encoded (same bytes every step).  The strictly
    # sequential figure (encode_host, then decode_host, one context) is reported next to it, and so is
    # the CEILING: the same bytes moved by plain cudaMemcpy with no codec, all ranks at once.
    e2e = None
    if not a.no_e2e:
        from concurrent.futures import ThreadPoolExecutor
        codec2 = pkg.Codec(local)
        # pinned host memory: frames + decoded frames + two stream buffers.  Use the whole N-frame batch
        # when the box can pin it for every rank, else the largest prefix that fits in a third of
        # MemAvailable (throughput is steady-state either way).
        Ne = N
        try:
            avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0]
            per_frame = 2 * px + 2 * codec.stream_bound(Ww, Hh, 1)
            Ne = max(16, min(N, int(avail / 3 / max(world, 1) / per_frame)))
            if a.e2e_frames > 0:
                Ne = min(N, a.e2e_frames)
        except Exception:
            pass
        N_full, N = N, Ne                              # the e2e leg below runs on the first Ne frames
        total = int(sizes[:N].sum().item())
        # the stream buffers are sized from the records' real bytes (known from the device leg) plus slack,
        # not from the 66*wh worst case; ONE pinned arena per process, carved into the four buffers
        cap = (total + total // 8 + (1 << 20) + 4095) // 4096 * 4096
        fb = (N * px + 4095) // 4096 * 4096
        arena = codec.pinned(2 * fb + 2 * cap)

        class View:
            def __init__(self, off, n):
                self.ptr, self.array = arena.ptr + off, arena.array[off:off + n]

        h_frames, h_dec = View(0, N * px), View(fb, N * px)
        h_streams = [View(2 * fb, cap), View(2 * fb + cap, cap)]
        h_offs = [np.zeros(N + 1, dtype=np.uint64), np.zeros(N + 1, dtype=np.uint64)]
        h_status = np.zeros(N, dtype=np.uint32)
        torch.cuda.synchronize()
        lib = codec.lib
        lib.dbde_b200_memcpy_d2h(codec.h, h_frames.ptr, frames.data_ptr(), N * px)

        # ceiling: one step's bytes per direction (raw frames + records) as plain asynchronous copies on
        # two streams, H2D || D2H, no codec -- what the link and the host side give this many ranks at once
        pool = ThreadPoolExecutor(2)
        s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
        t_frames, t_dec = torch.from_numpy(h_frames.array), torch.from_numpy(h_dec.array)
        t_s0, t_s1 = torch.from_numpy(h_streams[0].array[:total]), torch.from_numpy(h_streams[1].array[:total])
        assert t_frames.is_pinned() and t_s1.is_pinned(), "arena is not page-locked"
        dt_ceiling = 1e30
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s_up):
                decoded[:N * px].copy_(t_frames, non_blocking=True)
                decoded[:total].copy_(t_s0, non_blocking=True)
            with torch.cuda.stream(s_dn):
                t_dec.copy_(frames[:N * px], non_blocking=True)
                t_s1.copy_(stream_buf[:total], non_blocking=True)
            s_up.synchronize(); s_dn.synchronize()
            dt_ceiling = min(dt_ceiling, time.perf_counter() - t0)
        del t_frames, t_dec, t_s0, t_s1

        def enc_host(k):
            codec.encode_host_raw(h_frames.ptr, Ww, Hh, f0, N, h_streams[k % 2].ptr, cap, h_offs[k % 2].ctypes.data)

        def dec_host(k, c=None):
            (c or codec2).decode_host_raw(h_streams[k % 2].ptr, int(h_offs[k % 2][N]), h_offs[k % 2].ctypes.data, Ww, Hh, N,
                                          h_dec.ptr, h_status.ctypes.data, None)

        # warm-up (allocates the staging slots of both contexts) + correctness of the host path
        enc_host(0); enc_host(1); dec_host(1); dec_host(0, codec)
        assert int(h_offs[0][N]) == total and int(h_offs[1][N]) == total and not h_status.any()
        assert np.array_equal(h_dec.array, h_frames.array), "e2e round trip differs"
        # sequential: one context, encode then decode
        barrier()
        t0 = time.perf_counter()
        for k in range(a.e2e_steps):
            enc_host(k); dec_host(k, codec)
        dt_seq = time.perf_counter() - t0
        # concurrent: encode(k) || decode(k-1)
        barrier()
        t0 = time.perf_counter()
        for k in range(a.e2e_steps):
            fe, fd = pool.submit(enc_host, k), pool.submit(dec_host, k + 1)
            fe.result(); fd.result()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        pool.shutdown()
        assert not h_status.any() and np.array_equal(h_dec.array, h_frames.array), "e2e round trip differs"
        te = torch.tensor([dt, dt_seq, dt_ceiling], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dt, dt_seq, dt_ceiling = [float(x) for x in te.tolist()]
        e2e_value = world * 2 * N * px * a.e2e_steps / dt / 1e9
        ceiling = world * 2 * N * px / dt_ceiling / 1e9
        e2e = {"value": e2e_value, "unit": UNIT,
               "h2d_bytes_per_step": int(N * px + total + 8 * N), "d2h_bytes_per_step": int(total + 8 * (N + 1) + N * px + 4 * N),
               "steps": a.e2e_steps, "ms_per_step": 1000 * dt / a.e2e_steps, "frames_per_gpu_per_step": int(N),
               "ceiling": ceiling, "frac": e2e_value / ceiling,
               "ceiling_how": "the same bytes per direction (raw frames + records) as four plain cudaMemcpyAsync copies on pinned memory, "
                              "H2D || D2H on two streams, every rank at once, no codec; best of 3, max over ranks",
               "sequential": {"value": world * 2 * N * px * a.e2e_steps / dt_seq / 1e9, "ms_per_step": 1000 * dt_seq / a.e2e_steps},
               "path": "dbde_b200_encode_host || dbde_b200_decode_host on pinned host buffers: two contexts on two host "
                       "threads, each chunked through 3 device staging slots; step k decodes the stream of step k-1"}
        h_frames = h_dec = h_streams = None
        arena.free()
        codec2.close()
        N = N_full
        total = int(sizes[:N].sum().item())

    # ---- the other single-GPU BASELINE configs, device-resident, in the same run (N = 1 only)
    peak, peak_src = hbm_peak()
    extra = []
    if world == 1 and not a.no_extra:
        for name, kind, ew, eh, en in [("BASELINE config 3: odd-size 1001x1003 depth mix", "mix", 1001, 1003, 1000),
                                       ("BASELINE config 4: 4096x4096 low entropy", "low", 4096, 4096, 300)]:
            try:
                xl = DeviceLeg(torch, synth, codec, dev, kind, ew, eh, en, 0)
                xt, xalg, xhow = xl.gate(host_threads)
                xm = xl.timed(a.extra_steps, 3, barrier)
                eg, dg = xalg / (xm["enc_ms"] * 1e-3) / 1e9, xalg / (xm["dec_ms"] * 1e-3) / 1e9
                extra.append({"workload": "%s ('%s' generator, %d frames per launch, %d steps)" % (name, kind, en, a.extra_steps),
                              "width": ew, "height": eh, "frames": en, "generator": kind,
                              "encode": {"ms": xm["enc_ms"], "GBps": eg, "frac": eg / peak, "fps": en / (xm["enc_ms"] * 1e-3)},
                              "decode": {"ms": xm["dec_ms"], "GBps": dg, "frac": dg / peak, "fps": en / (xm["dec_ms"] * 1e-3)},
                              "raw_pixel_GBps": 2 * en * ew * eh / (xm["elapsed_ms"] / a.extra_steps * 1e-3) / 1e9,
                              "algorithmic_bytes_per_launch": int(xalg), "compressed_ratio": xt / float(en * ew * eh),
                              "parity": xhow})
                xl.free()
                del xl
                torch.cuda.empty_cache()
            except Exception as ex:            # an extra config must never take the headline line down
                extra.append({"workload": name, "error": repr(ex)})

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (algorithmic bytes / CUDA-event duration)
    enc_gbs, dec_gbs = alg_bytes / (enc_ms * 1e-3) / 1e9, alg_bytes / (dec_ms * 1e-3) / 1e9
    dom = "encode" if enc_ms >= dec_ms else "decode"
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))      # ncu dram__bytes_read+write per launch, captured for ONE workload
            if tj.get("workload") == {"kind": a.kind, "width": Ww, "height": Hh, "frames": N}:
                traffic = tj.get(dom, {}).get("dram_bytes_per_launch")
                traffic_src = "profiles/roofline_traffic.json (ncu --set full capture of this workload, %s; not re-measured in this run)" \
                              % tj.get("capture", "see profiles/README.md")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "dbde_%s_kernel" % dom, "achieved": enc_gbs if dom == "encode" else dec_gbs,
                "peak": peak, "unit": "GB/s", "frac": (enc_gbs if dom == "encode" else dec_gbs) / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": int(alg_bytes),
                "encode": {"ms": enc_ms, "GBps": enc_gbs, "frac": enc_gbs / peak},
                "decode": {"ms": dec_ms, "GBps": dec_gbs, "frac": dec_gbs / peak,
                           "note": "scan pre-pass + unpack kernel, timed together"}}

    # ---- the reference's CPU path on this box's host cores, bounded sample
    cpu = None
    if not a.no_cpu_baseline:
        try:
            threads = os.cpu_count() or 1
            ns = min(N, 64)
            sample = frames[:ns * px].cpu().numpy().reshape(ns, Hh, Ww)
            r = cpu_reference_rates(sample, threads, target_s=1.0)
            cpu = {"value": r["value"], "unit": UNIT, "cores": threads, "kind": r["kind"],
                   "sample": "first %d frames of this rank's batch, %s, ~1 s per direction (%.0f core-seconds)"
                             % (ns, CPU_CODECS[r["kind"]], r["cpu_seconds"]),
                   "encode_fps": r["encode_fps"], "decode_fps": r["decode_fps"]}
        except Exception as ex:            # the baseline must never take the bench line down
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": None, "sample": "failed: %s" % ex}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": workload_config(a),
            "encode_fps": world * N / (enc_ms_max * 1e-3), "decode_fps": world * N / (dec_ms_max * 1e-3),
            "encode_raw_GBps": world * N * px / (enc_ms_max * 1e-3) / 1e9,
            "decode_raw_GBps": world * N * px / (dec_ms_max * 1e-3) / 1e9,
            "compressed_ratio": total / float(N * px), "parity_gate": gate_how, "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches),
            "gpu_launches_note": "per step: 1 encode kernel + 2 decode kernels (scan, unpack); memset excluded",
            "roofline": roofline, "cpu_baseline": cpu, "extra_configs": extra}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    codec.close()
    return 0


if __name__ == "__main__":
    args = parse()
    sys.exit(run_reference(args) if args.impl == "reference" else run_ours(args))
