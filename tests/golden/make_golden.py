"""Generates tests/golden/golden.npz from the REFERENCE ITSELF (oracle/_ref: lilliput's own
opencv.cpp shims linked against its vendored OpenCV/libjpeg-turbo), so the restated oracle
(oracle/*.c) and the CUDA path can be pinned on machines where /root/reference is absent.

Run in the build container:  python tests/golden/make_golden.py
Inputs are either regenerated from seeds (lilliput_b200.synth) or stored in the file.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lilliput_b200 import abi  # noqa: E402
from lilliput_b200.synth import synth_image  # noqa: E402
from tests import golden as golden_set  # noqa: E402

RESIZE_CASES = [  # (seed, src_w, src_h, ch, crop(x,y,w,h) or None, dst_w, dst_h, interpolation)
    (11, 1920, 1080, 3, (420, 0, 1080, 1080), 256, 256, 3),   # BASELINE config 2 geometry
    (12, 800, 297, 3, (251, 0, 297, 297), 256, 256, 3),       # config 1 geometry
    (13, 721, 1283, 3, None, 257, 255, 3),
    (14, 300, 200, 3, None, 299, 199, 3),
    (15, 640, 480, 4, (80, 0, 480, 480), 160, 160, 3),        # integer scale 3
    (16, 512, 512, 3, None, 256, 256, 3),                     # 2x2 fast path
    (17, 1024, 512, 4, None, 256, 128, 3),                    # 4x4 fast path
    (18, 100, 100, 3, None, 250, 250, 3),                     # upscale: area-mode bilinear
    (19, 100, 200, 4, None, 50, 300, 3),                      # mixed
    (20, 333, 217, 3, None, 120, 97, 1),                      # INTER_LINEAR
    (21, 64, 48, 1, None, 23, 17, 3),
    (22, 1300, 1942, 3, (0, 321, 1300, 1300), 512, 512, 3),
]
JPEG_CASES = [  # (seed, w, h, ch, quality)
    (31, 256, 256, 3, 85), (32, 800, 297, 3, 85), (33, 17, 33, 3, 90), (34, 1, 1, 3, 85),
    (35, 9, 16, 3, 50), (36, 15, 7, 4, 100), (37, 100, 97, 1, 85), (38, 255, 257, 4, 30),
    (39, 640, 360, 3, 90), (40, 23, 49, 3, 1),
]
ORIENT_SRC = np.arange(6, dtype=np.uint8).reshape(2, 3)
BLEND_CASES = [  # (src BGRA, dst BGRA) from SURVEY Appendix D + random
    ((10, 20, 30, 0), (0, 0, 0, 0)), ((10, 20, 30, 0), (100, 110, 120, 255)),
    ((10, 20, 30, 255), (100, 110, 120, 255)), ((10, 20, 30, 128), (100, 110, 120, 255)),
    ((10, 20, 30, 128), (100, 110, 120, 0)), ((200, 100, 50, 64), (20, 40, 60, 128)),
    ((255, 255, 255, 1), (0, 0, 0, 254)),
]


PNG_NAMES = ["rgb", "rgba", "gray", "la", "pal37", "pal16", "pal2", "bit1", "gray16", "rgba16",
             "pal_trns", "rgb_trns", "stored", "level9", "filters", "wide", "ref_enc", "ref_enc_rgba",
             "fixture_ferry", "fixture_16bit_alpha"]


def png_cases(ref):
    import io
    from PIL import Image
    rng = np.random.default_rng(7)
    arr = synth_image(51, 53, 37, 3, noise=10.0)[:, :, ::-1].copy()  # RGB for PIL

    def enc(im, **kw):
        bio = io.BytesIO()
        im.save(bio, "PNG", **kw)
        return bio.getvalue()
    cases = {
        "rgb": enc(Image.fromarray(arr)),
        "rgba": enc(Image.fromarray(np.dstack([arr, arr[:, :, 0]]))),
        "gray": enc(Image.fromarray(arr[:, :, 0])),
        "la": enc(Image.fromarray(np.ascontiguousarray(arr[:, :, :2]), "LA")),
        "pal37": enc(Image.fromarray(arr).quantize(37)),
        "pal16": enc(Image.fromarray(arr).quantize(16)),
        "pal2": enc(Image.fromarray(arr).quantize(2)),
        "bit1": enc(Image.fromarray(arr[:, :, 0] > 128)),
        "gray16": enc(Image.fromarray(arr[:, :, 0].astype(np.uint16) * 257 + 3)),
        "pal_trns": enc(Image.fromarray(arr).quantize(20), transparency=3),
        "rgb_trns": enc(Image.fromarray(arr), transparency=tuple(int(v) for v in arr[0, 0])),
        "stored": enc(Image.fromarray(arr), compress_level=0),
        "level9": enc(Image.fromarray(synth_image(52, 200, 120, 3, noise=2.0)), compress_level=9),
        "wide": enc(Image.fromarray(rng.integers(0, 256, (3, 700, 4), dtype=np.uint8))),
    }
    import cv2
    big = synth_image(53, 320, 200, 4, noise=4.0)
    cases["filters"] = cv2.imencode(".png", big, [cv2.IMWRITE_PNG_COMPRESSION, 6])[1].tobytes()
    r16 = (synth_image(54, 40, 30, 4, noise=10.0).astype(np.uint16) << 8) | 0x5A
    cases["rgba16"] = cv2.imencode(".png", r16)[1].tobytes()
    cases["ref_enc"] = ref.encode(".png", synth_image(55, 97, 61, 3), {abi.PngCompression: 7})
    cases["ref_enc_rgba"] = ref.encode(".png", synth_image(56, 64, 64, 4), {abi.PngCompression: 1})
    cases["fixture_ferry"] = open("/root/reference/testdata/ferry_sunset.png", "rb").read()
    cases["fixture_16bit_alpha"] = open("/root/reference/data/firefox-16bit-alpha.png", "rb").read()
    assert sorted(cases) == sorted(PNG_NAMES)
    return [(k, cases[k]) for k in PNG_NAMES]


GIF_NAMES = ["dispose_bgnd", "duplicate_number_of_loops", "ferry_sunset", "no-loop", "no_gce_first_frame",
             "party-discord", "restore_previous", "syn_interlaced", "syn_offsets", "syn_local_palettes",
             "syn_dispose3", "syn_wide"]


def gif_cases():
    import io
    from PIL import Image
    cases = {}
    for n in GIF_NAMES[:7]:
        cases[n] = open(f"/root/reference/testdata/{n}.gif", "rb").read()
    rng = np.random.default_rng(3)

    def frames_to_gif(frames, **kw):
        bio = io.BytesIO()
        frames[0].save(bio, "GIF", save_all=True, append_images=frames[1:], **kw)
        return bio.getvalue()
    base = [Image.fromarray(synth_image(60 + i, 90, 70, 3, noise=3.0)[:, :, ::-1].copy()).quantize(64) for i in range(4)]
    cases["syn_interlaced"] = frames_to_gif(base, duration=70, loop=3, interlace=True, optimize=False)
    # PIL writes minimal bounding-box sub-frames when frames differ little: offsets + transparency
    a = np.zeros((60, 80, 3), np.uint8) + 200
    seq = []
    for i in range(5):
        b = a.copy()
        b[10 + 5 * i:25 + 5 * i, 15 + 8 * i:40 + 8 * i] = (30 * i, 255 - 40 * i, 90)
        seq.append(Image.fromarray(b))
    cases["syn_offsets"] = frames_to_gif(seq, duration=[50, 0, 10, 200, 30], loop=0, disposal=1, optimize=True)
    cases["syn_local_palettes"] = frames_to_gif(
        [Image.fromarray(synth_image(70 + i, 64, 48, 3, noise=8.0)[:, :, ::-1].copy()).quantize(256 if i % 2 else 16)
         for i in range(3)], duration=40, loop=1, optimize=False)
    cases["syn_dispose3"] = frames_to_gif(seq, duration=30, loop=0, disposal=[3, 2, 3, 1, 2], transparency=0,
                                          optimize=False)
    cases["syn_wide"] = frames_to_gif([Image.fromarray(rng.integers(0, 256, (5, 700, 3), dtype=np.uint8)).quantize(128)
                                       for _ in range(2)], duration=20)
    assert sorted(cases) == sorted(GIF_NAMES)
    return [(k, cases[k]) for k in GIF_NAMES]


def main():
    ref = abi.load_reference()
    out = {}
    for (seed, sw, sh, ch, crop, dw, dh, interp) in RESIZE_CASES:
        img = synth_image(seed, sw, sh, ch, noise=12.0)
        out[f"resize_{seed}"] = ref.resize(img, dw, dh, crop=crop, interpolation=interp)
    enc_sha = {}
    for (seed, w, h, ch, q) in JPEG_CASES:
        img = synth_image(seed, w, h, ch, noise=8.0)
        data = ref.encode(".jpeg", img, {abi.JpegQuality: q})
        enc_sha[f"{seed}"] = hashlib.sha256(data).hexdigest()
        out[f"jpeg_{seed}"] = np.frombuffer(data, dtype=np.uint8)
        out[f"jpegdec_{seed}"] = ref.decode(data)
    out["jpeg_sha"] = np.array([f"{k}:{v}" for k, v in enc_sha.items()])
    # other chroma layouts and restart intervals (made with cv2's libjpeg; decoded by the reference)
    import cv2
    img = synth_image(41, 203, 151, 3, noise=8.0)
    for sf, name in [(0x111111, "444"), (0x211111, "422"), (0x121111, "440"), (0x411111, "411"),
                     (0x221111, "420")]:
        for rst in (0, 3):
            ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 88,
                                                cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf,
                                                cv2.IMWRITE_JPEG_RST_INTERVAL, rst])
            data = buf.tobytes()
            out[f"jpegvar_{name}_{rst}"] = np.frombuffer(data, dtype=np.uint8)
            out[f"jpegvardec_{name}_{rst}"] = ref.decode(data)
    for o in range(1, 9):
        out[f"orient_{o}"] = ref.orient(ORIENT_SRC, o)
    img = synth_image(42, 37, 23, 3, noise=10.0)
    for o in range(1, 9):
        out[f"orient3_{o}"] = ref.orient(img, o)
    # end-to-end config 1: the reference's own fixture through Transform
    c1 = open("/root/reference/testdata/ferry_sunset.jpg", "rb").read()
    opt = abi.ImageOptions(FileType=".jpeg", Width=256, Height=256, ResizeMethod=abi.ImageOpsFit,
                           NormalizeOrientation=True, EncodeOptions={abi.JpegQuality: 85})
    out["c1_input"] = np.frombuffer(c1, dtype=np.uint8)
    out["c1_output"] = np.frombuffer(ref.transform(c1, opt), dtype=np.uint8)
    # an EXIF-rotated fixture (orientation 6) through Transform
    c6 = open("/root/reference/data/sunrise.jpg", "rb").read()
    opt6 = abi.ImageOptions(FileType=".jpeg", Width=64, Height=64, ResizeMethod=abi.ImageOpsFit,
                            NormalizeOrientation=True, EncodeOptions={abi.JpegQuality: 85})
    out["c6_input"] = np.frombuffer(c6, dtype=np.uint8)
    out["c6_output"] = np.frombuffer(ref.transform(c6, opt6), dtype=np.uint8)
    out["c6_decoded"] = ref.decode(c6)
    # PNG decode (lossless): files made by PIL / the reference encoder, decoded by the reference
    for name, data in png_cases(ref):
        out[f"png_{name}"] = np.frombuffer(data, dtype=np.uint8)
        out[f"pngdec_{name}"] = ref.decode(data)
    # GIF decode: reference fixtures + synthetic animations; frames pinned by SHA-256 (full canvas BGRA)
    for name, data in gif_cases():
        info = ref.gif_info(data)
        frames, delays, disposals, rc = ref.gif_frames(data)
        out[f"gif_{name}"] = np.frombuffer(data, dtype=np.uint8)
        out[f"gifmeta_{name}"] = np.array([info["width"], info["height"], info["frame_count"], info["loop_count"],
                                           info["duration_ms"], info["background_color"], rc, len(frames)],
                                          dtype=np.int64)
        out[f"gifdelay_{name}"] = np.array(delays, dtype=np.int64)
        out[f"gifdisp_{name}"] = np.array(disposals, dtype=np.int64)
        out[f"gifsha_{name}"] = np.array([hashlib.sha256(f.tobytes()).hexdigest() for f in frames])
        if frames.nbytes <= 200000:
            out[f"gifframes_{name}"] = frames
    golden_set.save("golden", out)
    print("wrote", len(out), "arrays")


if __name__ == "__main__":
    main()
