"""Golden vectors.  No stored file exceeds 1 MB: a set larger than that is kept as <name>.npz, <name>_2.npz,
<name>_3.npz, ... (arrays in their original order, split between whole arrays); load() merges the parts back."""
import io
import os
import re

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PART_BYTES = 900_000


class Golden(dict):
    """The merged arrays; `.files` lists the names in stored order, as on an NpzFile."""

    @property
    def files(self):
        return list(self)


def _parts(name):
    found = [f for f in os.listdir(HERE) if f == f"{name}.npz" or re.fullmatch(rf"{re.escape(name)}_\d+\.npz", f)]
    return sorted(found, key=lambda f: 1 if f == f"{name}.npz" else int(f[len(name) + 1:-4]))


def load(name):
    parts = _parts(name)
    if not parts:
        raise FileNotFoundError(os.path.join(HERE, f"{name}.npz"))
    out = Golden()
    for f in parts:
        with np.load(os.path.join(HERE, f)) as z:
            out.update((k, z[k]) for k in z.files)
    return out


def save(name, arrays):
    """Write `arrays` (a mapping) as compressed parts of at most PART_BYTES each, replacing any earlier parts."""
    for f in _parts(name):
        os.remove(os.path.join(HERE, f))
    groups, size = [[]], 0
    for k, v in arrays.items():
        b = io.BytesIO()
        np.savez_compressed(b, **{k: v})
        n = b.tell()
        if groups[-1] and size + n > PART_BYTES:
            groups.append([])
            size = 0
        groups[-1].append(k)
        size += n
    for i, keys in enumerate(groups):
        path = os.path.join(HERE, f"{name}.npz" if i == 0 else f"{name}_{i + 1}.npz")
        np.savez_compressed(path, **{k: arrays[k] for k in keys})
