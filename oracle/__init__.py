"""CPU oracle for the neural-tape-modeling recurrent forward pass.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs -- never by the product package.
"""
import io
import os

import numpy as np

PART_BYTES = 900_000        # every stored golden file stays under 1 MB


def save_golden(path, **arrays):
    """np.savez_compressed(path, **arrays), split into path-minus-.npz + ".1.npz", ".2.npz", ... (keys in order, each part
    under PART_BYTES) when one file would be larger; tests/conftest.py load_golden() merges the parts."""
    base = path[:-len(".npz")]
    sizes = {}
    for k, v in arrays.items():
        buf = io.BytesIO()
        np.savez_compressed(buf, **{k: v})
        sizes[k] = len(buf.getvalue())
    parts, cur = [], {}
    for k, v in arrays.items():
        if cur and sum(sizes[c] for c in cur) + sizes[k] > PART_BYTES:
            parts.append(cur)
            cur = {}
        cur[k] = v
    parts.append(cur)
    stale = [path] + [f"{base}.{i}.npz" for i in range(1, 100)]
    for p in stale:
        if os.path.exists(p):
            os.remove(p)
    if len(parts) == 1:
        np.savez_compressed(path, **arrays)
        return [path]
    out = [f"{base}.{i + 1}.npz" for i in range(len(parts))]
    for p, part in zip(out, parts):
        np.savez_compressed(p, **part)
    return out
