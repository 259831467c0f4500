"""Golden arrays kept as compressed parts of under 1 MB each, tests/golden/<name>.<i>.npz (i = 0, 1, ...), so that no file of the
repository is large.  save() cuts an array too large for one part along its first axis; load() joins the pieces again, so what a
test reads is bit for bit what the generator saved."""
import io
import os
import zipfile

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAX_FILE_BYTES = 1_000_000
PART_BYTES = 800_000  # packing target: the deflate estimate below is close to, not exactly, what np.savez_compressed writes


def part_paths(name):
    paths = []
    while os.path.exists(os.path.join(GOLD, f"{name}.{len(paths)}.npz")):
        paths.append(os.path.join(GOLD, f"{name}.{len(paths)}.npz"))
    return paths


def load(name):
    """name -> dict of arrays, the pieces of an array that was cut joined along axis 0"""
    paths = part_paths(name)
    if not paths:
        raise FileNotFoundError(os.path.join(GOLD, name + ".0.npz"))
    pieces = {}
    for p in paths:
        with np.load(p) as z:
            for k in z.files:
                pieces.setdefault(k, []).append(z[k])
    return {k: v[0] if len(v) == 1 else np.concatenate(v, axis=0) for k, v in pieces.items()}


def _deflated_bytes(a):
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w", compression=zipfile.ZIP_DEFLATED) as z:
        with z.open("a.npy", "w") as f:
            np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)
    return buf.tell()


def save(name, arrays):
    """write arrays (name -> array) as tests/golden/<name>.<i>.npz, replacing the parts written before"""
    items = []
    for k, a in arrays.items():
        a = np.asarray(a)
        est = _deflated_bytes(a)
        n = 1 if a.ndim == 0 else min(a.shape[0], -(-est // PART_BYTES))
        items += [(k, c, _deflated_bytes(c) if n > 1 else est) for c in (np.array_split(a, n, axis=0) if n > 1 else [a])]
    parts, cur, size = [], {}, 0
    for k, c, est in items:
        if cur and (size + est > PART_BYTES or k in cur):
            parts.append(cur)
            cur, size = {}, 0
        cur[k] = c
        size += est
    parts.append(cur)
    for p in part_paths(name):
        os.remove(p)
    for i, part in enumerate(parts):
        path = os.path.join(GOLD, f"{name}.{i}.npz")
        np.savez_compressed(path, **part)
        assert os.path.getsize(path) < MAX_FILE_BYTES, (path, os.path.getsize(path))
    return [os.path.join(GOLD, f"{name}.{i}.npz") for i in range(len(parts))]
