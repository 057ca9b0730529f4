"""bench.py contract checks: the reference arm (the reference's own CPU code through oracle/_ref,
or the oracle port) prints one JSON line with the keys a caller reads, our arm refuses to run
without a CUDA device (there is no CPU path to fall back to), and on a B200 --dump-outputs saves
what the timed steps computed."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                          timeout=600, cwd=ROOT, env=e)


def test_reference_arm_prints_the_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--frames", "4", "--width", "256", "--height", "256"])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["unit"] == "GB/s"
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["dtype"] == "u8"
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--frames", "4", "--width", "64", "--height", "64"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return          # on a GPU box this is covered by the gpu tests / the bench itself
    r = _run(["--steps", "1", "--warmup", "1", "--frames", "2", "--width", "64", "--height", "64", "--no-e2e"])
    assert r.returncode != 0
    assert "no CUDA device" in (r.stdout + r.stderr) or "no CPU" in (r.stdout + r.stderr)


def test_zero_steps_is_refused():
    r = _run(["--impl", "reference", "--steps", "0", "--frames", "4", "--width", "64", "--height", "64"])
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_steps_results(tmp_path):
    """--dump-outputs: the timed path's records and decoded pixels (seeded samples) and per-frame sizes, offsets
    and status, all float32/float64 and under 64 MB, equal to what the oracle port computes for the same seeded
    frames; --steps sets the number of timed steps (3 launches each: encode, decode scan, unpack)"""
    import importlib
    import numpy as np
    import oracle
    import synth
    N, W, H = 10, 1001, 1003
    r = _run(["--steps", "3", "--warmup", "1", "--frames", str(N), "--width", str(W), "--height", str(H), "--kind", "mix",
              "--no-e2e", "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3 * 3
    d = {f[:-4]: np.load(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values()) and sum(a.nbytes for a in d.values()) <= 64 << 20
    frames = synth.gen_frames("mix", N, W, H, seed=42)
    want, sizes = oracle.port.pack_frames(frames, 0)
    starts = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    stride = importlib.import_module("dbce-video-cpp_b200").load().dbde_b200_slot_stride(W, H)
    assert d["per_frame_index"].tolist() == list(range(N)) and d["record_sizes"].tolist() == sizes.tolist()
    assert d["record_offsets"].tolist() == [i * stride for i in range(N)] and not d["decode_status"].any()
    fidx, bpos, ppos = (d[k].astype(np.int64) for k in ("sample_frame_index", "sample_byte_position", "sample_pixel_position"))
    assert len(fidx) == 8 and len(bpos) == len(ppos) == 1 << 19
    for j, f in enumerate(fidx):
        rec = want[starts[f]:starts[f + 1]].astype(np.float32)
        assert (d["record_bytes_sample"][j] == np.where(bpos < len(rec), rec[np.minimum(bpos, len(rec) - 1)], -1)).all(), f
    assert (d["decoded_pixels_sample"] == frames.reshape(N, -1)[fidx][:, ppos]).all()
