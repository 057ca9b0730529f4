"""Generate tests/golden/golden_differential.json: what the port-vs-reference comparisons in tests/test_oracle.py
compare against, stored so that they run where the reference (oracle/_ref) is not built.

  * differential: 60 seeded frames of 1..69 x 1..49 pixels (all depth classes, noise, flat), one record each
  * variants: 5 shapes x 3 styles x 2 frames with DBDE_INVERT_ENDIAN + DBDE_HZ_AS_INTEGER, and one video header

The records come from the unmodified reference (oracle.ref / oracle.ref_variants) when oracle/_ref is built,
otherwise from the port (oracle.port / oracle.port_variants()); "source" in the file says which.  The tests
check the port, the CUDA library and, where it is built, the reference against these vectors.
      python tests/golden/make_golden_differential.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, ".."))
import oracle  # noqa: E402
from conftest import rand_frame  # noqa: E402

VARIANT_SHAPES = [(8, 8), (10, 10), (17, 23), (64, 40), (1001, 24)]
STYLES = ("classes", "noise", "flat")
HEADER = (3, 480, 640, 29.97)          # u64s, height, width, frame rate of the stored variant video header


def differential_frames():
    """-> [(frame index, W, H, image)] in the order the comparison uses"""
    rng = np.random.default_rng(3)
    out = []
    for i in range(60):
        W, H = int(rng.integers(1, 70)), int(rng.integers(1, 50))
        out.append((i, W, H, rand_frame(rng, W, H, STYLES[i % 3])))
    return out


def variant_frames():
    """-> [(W, H, style, frames (2,H,W))] in the order the comparison uses"""
    rng = np.random.default_rng(77)
    return [(W, H, style, np.stack([rand_frame(rng, W, H, style) for _ in range(2)]))
            for W, H in VARIANT_SHAPES for style in STYLES]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint8).tobytes()).hexdigest()


if __name__ == "__main__":
    plain = oracle.ref if oracle.ref is not None else oracle.port
    variants = oracle.ref_variants if oracle.ref_variants is not None else oracle.port_variants()
    out = {"source": "reference (oracle/_ref)" if oracle.ref is not None else "oracle port (oracle/_ref not built)",
           "differential": [], "variants": {"first_index": 5, "cases": []}}
    for i, W, H, img in differential_frames():
        rec = plain.pack_frame(i, img)
        out["differential"].append({"index": i, "W": W, "H": H, "image_sha256": sha(img), "record_len": len(rec),
                                    "record_sha256": sha(rec)})
    for W, H, style, fr in variant_frames():
        stream, sizes = variants.pack_frames(fr, 5)
        out["variants"]["cases"].append({"W": W, "H": H, "style": style, "frames_sha256": sha(fr),
                                         "sizes": [int(s) for s in sizes], "stream_sha256": sha(stream)})
    out["variants"]["video_header"] = {"args": list(HEADER), "hex": variants.pack_video_header(*HEADER).tobytes().hex()}
    path = os.path.join(HERE, "golden_differential.json")
    json.dump(out, open(path, "w"), indent=1)
    print("wrote", path, "from", out["source"])
