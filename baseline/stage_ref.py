#!/usr/bin/env python3
"""Stage the UNMODIFIED reference files the CPU arm of bench.py runs (`bench.py --impl reference`) under baseline/_ref/.

baseline/_ref/ is git-ignored (reference sources never enter this repository's history) but travels to the GPU box with
the working tree.  Run in the build container (where /root/reference exists); __graft_entry__.build() calls it.

    code/model.py  code/networks/unet_1d.py  code/utilities/utilities.py      the reference's RNN / DiffDelRNN classes
    weights/<the three BASELINE.json checkpoints>/best.pth                     ~53 KB each

The reference is a script tree, not a package (no setup.py / pyproject: `pip install /root/reference` has nothing to
install), and `import model` needs soundfile / librosa, which are absent here and on the GPU box: load_reference() below
registers two empty stub modules for them (only plotting / audio-IO helpers of utilities.py use them; SURVEY.md 9.2)."""
import os
import shutil
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
SRC = os.environ.get("NTM_REFERENCE_ROOT", "/root/reference")
FILES = ["code/model.py", "code/networks/unet_1d.py", "code/utilities/utilities.py",
         "code/test-model.py"]       # (test-model.py is never imported: it is the caller code that
                                     # tests/test_caller_contract_gpu.py restates against the drop-in classes)
CKPTS = {
    "cfg1": "GRU-HS[64]-L[ESR]-DS[ReelToReel_Dataset_MiniPulse100_CHOWTAPE]_BEST",
    "cfg2": "GRU-HS[64]-L[DCPreESR]-DS[ReelToReel_Dataset_MiniPulse100_AKAI_IPS[7.5]_MAXELL]_BEST",
    "cfg3": "DiffDelGRU-HS[64]-L[DCPreESR]-DS[ReelToReel_Dataset_MiniPulse100_CHOWTAPE_WOWFLUTTER]_BEST",
}


def stage():
    """Copy the files if the reference tree is present; returns True if baseline/_ref is usable afterwards."""
    if os.path.isdir(SRC):
        for rel in FILES + [f"weights/{d}/best.pth" for d in CKPTS.values()]:
            dst = os.path.join(DST, rel)
            os.makedirs(os.path.dirname(dst), exist_ok=True)
            shutil.copyfile(os.path.realpath(os.path.join(SRC, rel)), dst)
    return available()


def available():
    return all(os.path.exists(os.path.join(DST, rel)) for rel in FILES) and \
        os.path.exists(os.path.join(DST, "weights", CKPTS["cfg2"], "best.pth"))


def load_reference():
    """-> the reference's `model` module (code/model.py, unmodified), imported from baseline/_ref."""
    for name in ("soundfile", "librosa", "librosa.filters"):
        m = types.ModuleType(name)
        if name == "librosa.filters":
            m.mel = None
        sys.modules.setdefault(name, m)
    code = os.path.join(DST, "code")
    if code not in sys.path:
        sys.path.insert(0, code)
    import model as refmodel
    return refmodel


def load_checkpoint(tag):
    import torch
    return torch.load(os.path.join(DST, "weights", CKPTS[tag], "best.pth"), map_location="cpu", weights_only=True)


if __name__ == "__main__":
    print("baseline/_ref staged" if stage() else "reference tree not found; baseline/_ref not staged")
