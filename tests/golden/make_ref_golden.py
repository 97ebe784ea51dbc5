"""Mint ``tests/golden/ref_outputs.npz`` by EXECUTING the reference's own modules.

    python tests/golden/make_ref_golden.py

Runs the original ``script/mfcc.py`` and ``script/calc.py`` unmodified, from the checkout at ``reference_path``
of ``BASELINE.json`` (``$MMF_REFERENCE_ROOT`` overrides it; imported by
``oracle/ref_loader.py`` with stub modules for the five third-party packages this image lacks; the one
arithmetic step served by a stub is ``librosa.feature.mfcc`` -> the restated chain of ``oracle.mfcc``) over
every case of ``tests/ref_cases.py`` and stores each returned array.  The original project is not part of
this repository, which is why the outputs are committed.
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref_loader  # noqa: E402
import ref_cases  # noqa: E402


def main():
    mods = {"mfcc": ref_loader.ref_mfcc(), "calc": ref_loader.ref_calc()}
    out = {}
    for name in ref_cases.CASES:
        for i, a in enumerate(ref_cases.run_case(mods, name)):
            out[f"{name}__{i}"] = a
    path = os.path.join(HERE, "ref_outputs.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(ref_cases.CASES)} cases, {len(out)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
