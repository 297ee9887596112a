"""CPU: bench.py's --dump-outputs writer.  Two builds are compared output for output through these files, so they must
hold every item's status / length / CRC, split back into the sampled files exactly, pick the same items whatever the
outputs are, and stay under 64 MB at the largest batch and output capacity any config runs."""
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_dump_round_trips_the_sampled_files(tmp_path):
    rng = np.random.default_rng(5)
    n = 40
    ins = [rng.integers(0, 256, 50 + i, dtype=np.uint8) for i in range(n)]
    outs = [rng.integers(0, 256, int(rng.integers(0, 300)), dtype=np.uint8).tobytes() for _ in range(n)]
    status = [0] * (n - 1) + [-2]
    bench.dump_outputs(str(tmp_path / "a"), ins, outs, status, 1 << 20)
    d = {p.stem: np.load(p) for p in (tmp_path / "a").glob("*.npy")}
    assert set(d) == {"status", "out_len", "out_crc32", "input_crc32", "sample_index", "sample_bytes"}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert d["status"].tolist() == status
    assert d["out_crc32"].tolist() == [zlib.crc32(o) for o in outs]
    assert d["input_crc32"].tolist() == [zlib.crc32(x) for x in ins]
    k = d["sample_index"].astype(int)
    assert 0 < len(k) < n and (np.diff(k) > 0).all()
    lens = d["out_len"].astype(int)
    parts = np.split(d["sample_bytes"].astype(np.uint8), np.cumsum(lens[k])[:-1])
    assert [p.tobytes() for p in parts] == [outs[i] for i in k]
    # other outputs, same item count and capacity: the same items are sampled
    bench.dump_outputs(str(tmp_path / "b"), ins, [b"x"] * n, status, 1 << 20)
    assert np.array_equal(np.load(tmp_path / "b" / "sample_index.npy"), d["sample_index"])


def test_dump_stays_under_64_mb_with_every_output_at_capacity():
    for n, out_cap in ((4096, 65536), (2048, 1 << 20), (256, 8 << 20), (8192, 1 << 17), (1, 8 << 20)):
        k = len(bench.dump_sample(n, out_cap))
        assert k >= 1
        assert 4 * k * out_cap + 8 * (4 * n + k) < 64 << 20, (n, out_cap)
