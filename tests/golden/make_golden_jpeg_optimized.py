"""Generates tests/golden/jpeg_optimized_golden.npz from the REFERENCE ITSELF (oracle/_ref):
baseline (sequential, single-scan) JPEGs whose Huffman tables were optimised for the image
(libjpeg optimize_coding through the OpenCV and Pillow writers) -- code-length distributions the
Annex K tables never show: few symbols, codes of every length up to 16, long codes behind other
prefixes than the standard tables' all-ones run -- each with the pixels the reference decodes.

Run in the build container:  python tests/golden/make_golden_jpeg_optimized.py
"""
import hashlib
import io
import os
import sys

import cv2
import numpy as np
from PIL import Image, ImageFile

ImageFile.MAXBLOCK = 1 << 24  # optimize=True buffers the whole file; random pixels at q100 exceed the default

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lilliput_b200 import abi  # noqa: E402
from lilliput_b200.synth import synth_image  # noqa: E402
from tests import golden as golden_set  # noqa: E402


def cases():
    out = {}
    k = 0
    shapes = [(64, 48, 3), (257, 131, 3), (33, 17, 1), (1, 1, 3), (640, 360, 3), (1024, 300, 3)]
    for i, (w, h, ch) in enumerate(shapes):
        for noise, q, samp in [(2.0, 20, 0x221111), (12.0, 75, 0x221111), (40.0, 100, 0x111111), (25.0, 92, 0x211111),
                               (60.0, 98, 0x221111)]:
            if ch == 1 and samp != 0x221111:
                continue
            img = synth_image(700 + 10 * i + k % 7, w, h, ch, noise=noise)
            if ch == 1:
                img = img.reshape(h, w)
            opts = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_OPTIMIZE, 1]
            if ch == 3:
                opts += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp]
            ok, enc = cv2.imencode(".jpg", img, opts)
            assert ok
            k += 1
            if len(enc) > 300 * 1024:  # keep the fixture small
                continue
            out[f"opt{k - 1:02d}_{w}x{h}c{ch}q{q}n{int(noise)}"] = enc.tobytes()
    # random pixels: every run/size symbol shows up, the optimised tables use the whole length range
    rng = np.random.default_rng(77)
    rnd = rng.integers(0, 256, (240, 320, 3), dtype=np.uint8)
    for name, kw in [("pil_rand_q100_444", dict(optimize=True, quality=100, subsampling=0)),
                     ("pil_rand_q95_420", dict(optimize=True, quality=95, subsampling=2)),
                     ("pil_rand_q30_422", dict(optimize=True, quality=30, subsampling=1))]:
        bio = io.BytesIO()
        Image.fromarray(rnd).save(bio, "JPEG", **kw)
        out[name] = bio.getvalue()
    flat = np.full((96, 160, 3), 131, np.uint8)  # two or three symbols per table
    bio = io.BytesIO()
    Image.fromarray(flat).save(bio, "JPEG", optimize=True, quality=90)
    out["pil_flat"] = bio.getvalue()
    return out


def main():
    ref = abi.load_reference()
    out, names = {}, []
    for name, data in cases().items():
        assert b"\xff\xc2" not in data[:600], "expected a sequential file"
        px = ref.decode(data)
        names.append(name)
        out[f"jpg_{name}"] = np.frombuffer(data, np.uint8)
        out[f"sha_{name}"] = np.array(hashlib.sha256(px.tobytes()).hexdigest())
        out[f"shape_{name}"] = np.array(px.shape, np.int64)
        if px.size <= 48 * 1024:
            out[f"px_{name}"] = px
        print(f"{name:32s} {len(data):7d} B -> {px.shape}")
    out["names"] = np.array(names)
    golden_set.save("jpeg_optimized_golden", out)
    print("wrote", len(out), "arrays")


if __name__ == "__main__":
    main()
