"""Generates tests/golden/gif_encode_golden.npz from the REFERENCE ITSELF (oracle/_ref): complete
GIF -> GIF ImageOps.Transform outputs (decode, composite, fit / resize, palette mapping with the
reference's order-dependent memo, giflib LZW) for the GIF fixtures already in golden.npz.
GIF encoding is deterministic integer work: the device path must reproduce these BYTES.

Run in the build container:  python tests/golden/make_golden_gif_encode.py
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lilliput_b200 import abi  # noqa: E402
from tests import golden as golden_set  # noqa: E402

TIMEOUT_NS = 600 * 10**9  # ops.go:368,435: a zero EncodeTimeout times out after the first frame

CASES = [  # (fixture, label, options)
    ("party-discord", "fit16", dict(Width=16, Height=16, ResizeMethod=abi.ImageOpsFit)),
    ("party-discord", "noresize", dict(Width=0, Height=0, ResizeMethod=abi.ImageOpsNoResize)),
    ("party-discord", "resize40x30", dict(Width=40, Height=30, ResizeMethod=abi.ImageOpsResize)),
    ("no-loop", "fit64", dict(Width=64, Height=64, ResizeMethod=abi.ImageOpsFit)),
    ("dispose_bgnd", "noresize", dict(Width=0, Height=0, ResizeMethod=abi.ImageOpsNoResize)),
    ("dispose_bgnd", "fit50", dict(Width=50, Height=50, ResizeMethod=abi.ImageOpsFit)),
    ("duplicate_number_of_loops", "fit20", dict(Width=20, Height=20, ResizeMethod=abi.ImageOpsFit)),
    ("no_gce_first_frame", "noresize", dict(Width=0, Height=0, ResizeMethod=abi.ImageOpsNoResize)),
    ("restore_previous", "fit32", dict(Width=32, Height=32, ResizeMethod=abi.ImageOpsFit)),
    ("ferry_sunset", "fit100", dict(Width=100, Height=100, ResizeMethod=abi.ImageOpsFit)),
    ("syn_interlaced", "noresize", dict(Width=0, Height=0, ResizeMethod=abi.ImageOpsNoResize)),
    ("syn_offsets", "noresize", dict(Width=0, Height=0, ResizeMethod=abi.ImageOpsNoResize)),
    ("syn_local_palettes", "fit48", dict(Width=48, Height=48, ResizeMethod=abi.ImageOpsFit)),
    ("syn_dispose3", "noresize", dict(Width=0, Height=0, ResizeMethod=abi.ImageOpsNoResize)),
    ("syn_wide", "resize120x20", dict(Width=120, Height=20, ResizeMethod=abi.ImageOpsResize)),
    ("party-discord", "maxframes3", dict(Width=16, Height=16, ResizeMethod=abi.ImageOpsFit, MaxEncodeFrames=3)),
]


def main():
    ref = abi.load_reference()
    g = golden_set.load("golden")
    out, names = {}, []
    for fixture, label, kw in CASES:
        data = g[f"gif_{fixture}"].tobytes()
        name = f"{fixture}__{label}"
        try:
            enc = ref.transform(data, abi.ImageOptions(FileType=".gif", EncodeTimeout_ns=TIMEOUT_NS, **kw))
            rc = 0
        except abi.LilliputError as e:
            enc, rc = b"", e.code
        names.append(name)
        out[f"rc_{name}"] = np.array(rc, np.int64)
        out[f"sha_{name}"] = np.array(hashlib.sha256(enc).hexdigest())
        out[f"len_{name}"] = np.array(len(enc), np.int64)
        if len(enc) <= 48 * 1024:
            out[f"out_{name}"] = np.frombuffer(enc, np.uint8)
        print(f"{name:44s} rc={rc} {len(enc):7d} B")
    out["names"] = np.array(names)
    path = os.path.join(ROOT, "tests", "golden", "gif_encode_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path))


if __name__ == "__main__":
    main()
