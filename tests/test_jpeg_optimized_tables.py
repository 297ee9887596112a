"""Baseline JPEGs with image-optimised Huffman tables (libjpeg optimize_coding): the oracle restatement
(CPU) and the device decoders (GPU: the parallel kernel through the per-image ABI) against pixels the
reference itself decoded (tests/golden/jpeg_optimized_golden.npz).  Bit-exact.  These tables exercise
what the Annex K tables never do: codes of every length, long codes behind several prefixes, tables
with two or three symbols."""
import hashlib

import numpy as np
import pytest

from lilliput_b200 import abi
from tests import golden as golden_set

G = golden_set.load("jpeg_optimized_golden")
NAMES = [str(n) for n in G["names"]]


def _check(px, name):
    assert list(px.shape) == [int(v) for v in G[f"shape_{name}"]]
    assert hashlib.sha256(np.ascontiguousarray(px).tobytes()).hexdigest() == str(G[f"sha_{name}"])
    if f"px_{name}" in G.files:
        assert np.array_equal(px, G[f"px_{name}"])


@pytest.mark.parametrize("name", NAMES)
def test_oracle_optimized_tables_match_reference(oracle, name):
    px, _ = oracle.jpeg_decode(G[f"jpg_{name}"].tobytes())
    _check(px, name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_device_optimized_tables_match_reference(cuda_lib, name):
    _check(cuda_lib.decode(G[f"jpg_{name}"].tobytes()), name)


@pytest.mark.gpu
def test_optimized_source_through_transform(cuda_lib, oracle):
    """Optimised-table JPEG -> Fit -> baseline JPEG through lp_transform, against the oracle pipeline."""
    name = next(n for n in NAMES if "640x360" in n and "q98" in n)
    data = G[f"jpg_{name}"].tobytes()
    src, _ = oracle.jpeg_decode(data)
    out = cuda_lib.transform(data, abi.ImageOptions(FileType=".jpeg", Width=200, Height=200,
                                                    ResizeMethod=abi.ImageOpsFit,
                                                    EncodeOptions={abi.JpegQuality: 85}))
    assert out == oracle.jpeg_encode(oracle.fit(src, 200, 200), 85)
