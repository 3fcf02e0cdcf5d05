"""Golden vectors stored as several compressed .npz parts, none larger than PART_LIMIT bytes, so that no committed file
exceeds 1 MB.  `<dir>/<stem>.npz` is written as `<dir>/<stem>.part0.npz`, `<stem>.part1.npz`, ...; an array too large for
one part is cut along its first axis and its pieces are concatenated again, in part order, by load()."""
import glob
import io
import os
import re

import numpy as np

PART_LIMIT = 900 * 1024


def _compressed_size(arrays):
    buf = io.BytesIO()
    np.savez_compressed(buf, **arrays)
    return buf.tell()


def _pieces(key, a):
    """(key, array) pieces of `a`, each compressing to under PART_LIMIT on its own."""
    n = 1
    while a.ndim > 0 and n < a.shape[0] and max(_compressed_size({key: p}) for p in np.array_split(a, n)) > PART_LIMIT:
        n += 1
    return [(key, p) for p in (np.array_split(a, n) if n > 1 else [a])]


def part_paths(path):
    stem = path[:-len(".npz")]
    found = glob.glob(glob.escape(stem) + ".part*.npz")
    index = lambda p: int(re.search(r"\.part(\d+)\.npz$", p).group(1))
    return sorted((p for p in found if re.search(r"\.part\d+\.npz$", p)), key=index)


def save(path, arrays):
    """Writes `arrays` (name -> array) as the parts of `path` (which must end in .npz), replacing any earlier parts."""
    for p in part_paths(path):
        os.remove(p)
    parts, cur = [], {}
    for key in arrays:
        for k, piece in _pieces(key, np.asarray(arrays[key])):
            if k in cur or (cur and _compressed_size(dict(cur, **{k: piece})) > PART_LIMIT):
                parts.append(cur)
                cur = {}
            cur[k] = piece
    parts.append(cur)
    stem = path[:-len(".npz")]
    for i, part in enumerate(parts):
        np.savez_compressed("%s.part%d.npz" % (stem, i), **part)


def load(path):
    """name -> array, read back from the parts save() wrote for `path`."""
    paths = part_paths(path)
    if not paths:
        raise FileNotFoundError("no parts of %s" % path)
    out = {}
    for p in paths:
        with np.load(p) as d:
            for k in d.files:
                out.setdefault(k, []).append(d[k])
    return {k: (v[0] if len(v) == 1 else np.concatenate(v, axis=0)) for k, v in out.items()}
