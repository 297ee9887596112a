"""Probe (not collected by pytest): throws mutated files at every device decoder through the C ABI.
The calls may fail (that is the point) but must return -- no hang, no crash, no sticky CUDA error.
Run under `timeout` on the GPU box:  timeout 900 python tests/fuzz_probe.py [iterations]"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lilliput_b200 import abi  # noqa: E402
from tests import golden as golden_set  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def corpus():
    g = golden_set.load("golden")
    w = np.load(os.path.join(ROOT, "tests", "golden", "webp_golden.npz"))
    j = np.load(os.path.join(ROOT, "tests", "golden", "jpeg_multiscan_golden.npz"))
    a = np.load(os.path.join(ROOT, "tests", "golden", "png_adam7_golden.npz"))
    out = []
    for k in g.files:
        if k.startswith(("gif_", "png_")) and g[k].dtype == np.uint8 and g[k].ndim == 1 and g[k].size < 40000:
            out.append((k, g[k].tobytes()))
        if k.startswith("jpeg_") and g[k].dtype == np.uint8 and g[k].ndim == 1 and g[k].size < 40000:
            out.append((k, g[k].tobytes()))
    for k in w.files:
        if k.startswith("webp_") and k != "webp_names" and w[k].size < 40000:
            out.append((k, w[k].tobytes()))
    for k in list(j.files)[:40]:
        if k.startswith("jpg_") and j[k].size < 40000:
            out.append((k, j[k].tobytes()))
    for k in list(a.files)[:60]:
        if k.startswith("png_") and a[k].size < 20000:
            out.append((k, a[k].tobytes()))
    return out


def mutate(rng, data: bytes) -> bytes:
    b = bytearray(data)
    mode = rng.integers(0, 5)
    if mode == 0 and len(b) > 20:  # truncate
        return bytes(b[: rng.integers(10, len(b))])
    n = 1 + int(rng.integers(0, 8))
    for _ in range(n):
        i = int(rng.integers(min(12, len(b) - 1), len(b)))
        if mode == 1:
            b[i] ^= 1 << int(rng.integers(0, 8))
        elif mode == 2:
            b[i] = int(rng.integers(0, 256))
        elif mode == 3:
            b[i] = 0xFF
        else:
            b[i] = 0
    return bytes(b)


def main():
    iters = int(sys.argv[1]) if len(sys.argv) > 1 else 400
    lib = abi.load_cuda()
    files = corpus()
    print(len(files), "seed files", flush=True)
    rng = np.random.default_rng(12345)
    ok = fail = 0
    t0 = time.time()
    for it in range(iters):
        name, data = files[int(rng.integers(0, len(files)))]
        m = mutate(rng, data)
        try:
            if name.startswith("webp_"):
                _, frames, _, rc = lib.webp_frames(m)
                ok += rc == 0
                fail += rc != 0
            elif name.startswith("gif_"):
                _, _, _, rc = lib.gif_frames(m, max_frames=64)
                ok += rc == 0
                fail += rc != 0
            else:
                lib.decode(m)
                ok += 1
        except abi.LilliputError:
            fail += 1
        if it % 50 == 49:
            print(f"{it + 1} mutations: {ok} decoded, {fail} refused, {time.time() - t0:.0f} s", flush=True)
    # the device must still be healthy: a clean decode works
    name, data = next(f for f in files if f[0].startswith("png_"))
    lib.decode(data)
    print("device healthy after fuzzing:", ok, "decoded,", fail, "refused")


if __name__ == "__main__":
    main()
