import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def load_ckpt(tag):
    """state_dict (torch tensors) of one of the three BASELINE.json checkpoints, from tests/golden."""
    import torch
    z = np.load(os.path.join(GOLD, f"ckpt_{tag}.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files if k not in ("model_type", "weights_dir")}


class Golden(dict):
    """Arrays of one golden set by name, like the np.load of a .npz (`.files`, `g[key]`)."""

    @property
    def files(self):
        return list(self)


def load_golden(name):
    """tests/golden/<name>.npz, or its parts <name>.1.npz, <name>.2.npz, ... merged (oracle.save_golden keeps every file
    under 1 MB)."""
    parts = sorted(glob.glob(os.path.join(GOLD, f"{name}.[0-9]*.npz")), key=lambda p: int(p.split(".")[-2]))
    g = Golden()
    for p in parts or [os.path.join(GOLD, f"{name}.npz")]:
        with np.load(p) as z:
            g.update({k: z[k] for k in z.files})
    return g


SIGNALS = ("sweepnoise", "sweepnoise_lo", "noise", "pulse", "sine", "sine1k", "silence")
