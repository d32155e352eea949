"""Golden sets stored as `<name>.npz` plus `<name>.<k>.npz` parts (k = 2, 3, ...), each file under 1 MB.

save() packs the arrays of one set into as many compressed parts as needed; load() merges them back into one dict,
so a test reads a set the same way however many files hold it."""
import glob
import io
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PART_BYTES = 900_000


def _compressed(arrays):
    buf = io.BytesIO()
    np.savez_compressed(buf, **arrays)
    return buf.getvalue()


def save(name, directory=HERE, **arrays):
    for old in [os.path.join(directory, f"{name}.npz")] + glob.glob(os.path.join(directory, f"{name}.*.npz")):
        if os.path.exists(old):
            os.remove(old)
    parts, cur = [], {}
    for key, value in arrays.items():
        if cur and len(_compressed({**cur, key: value})) > PART_BYTES:
            parts.append(cur)
            cur = {}
        cur[key] = value
    parts.append(cur)
    paths = []
    for k, part in enumerate(parts, start=1):
        blob = _compressed(part)
        if len(blob) > PART_BYTES:
            raise ValueError(f"{name}: {sorted(part)} alone compresses to {len(blob)} bytes (> {PART_BYTES})")
        paths.append(os.path.join(directory, f"{name}.npz" if k == 1 else f"{name}.{k}.npz"))
        with open(paths[-1], "wb") as f:
            f.write(blob)
    return paths


def load(directory, name):
    paths = [os.path.join(directory, f"{name}.npz")] + sorted(glob.glob(os.path.join(directory, f"{name}.*.npz")))
    out = {}
    for p in paths:
        with np.load(p) as z:
            for key in z.files:
                out[key] = z[key]
    return out
