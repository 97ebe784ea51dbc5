"""Mint tests/golden/filter_bits.npz: SHA-256 digests of the 'fir' and 'sg' output filters' outputs, to pin their bytes.

Three kinds of case, each a name and its float64 output:
- ('fir', seed, n_taps, T, rows, f32): Plan.fir_filtfilt (scipy.signal.filtfilt(b, 1, x)) of `rows` rows of T samples
  with n_taps seeded random taps.  The lengths sit at 3 * n_taps + 1 (the shortest that filtfilt takes) and on either
  side of a 256-output boundary of the input and of the odd-extended signal (T + 6 * n_taps).
- ('sg', seed, window, polyorder, T, rows, f32): Plan.stencil with the savgol_filter(mode='interp') stencil, as
  applyFilter's 'sg' branch builds it.
- ('vel', seed, method, difference, param, T, f32): get_velocity(x, 100.0, ...) of one trajectory: 'gradient' with
  `difference` passes, 'finDiff' with accOrder = param, 'sg' with width = param (polyOrder 2 unless the width is 3).

f32: the input is float32 (widened to float64 by the wrappers).  The digest is over the C-contiguous float64 output.

    python tests/golden/make_filter_bits.py [out.npz]     # needs a GPU; writes tests/golden/filter_bits.npz
"""

import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

FIR = [  # (seed, n_taps, T, rows, f32)
    (1, 1, 4, 1, 0),
    (2, 1, 255, 3, 0),
    (3, 1, 256, 2, 0),
    (4, 1, 257, 2, 0),
    (5, 2, 7, 2, 0),
    (6, 2, 500, 2, 0),        # L = 512
    (7, 2, 501, 1, 0),
    (8, 6, 19, 3, 0),
    (9, 6, 476, 2, 0),        # L = 512
    (10, 6, 477, 2, 1),
    (11, 6, 1000, 4, 0),
    (12, 7, 22, 2, 0),
    (13, 7, 511, 2, 0),
    (14, 7, 512, 2, 1),
    (15, 7, 513, 2, 0),
    (16, 21, 64, 2, 0),
    (17, 21, 1024, 3, 0),
    (18, 21, 1025, 1, 1),
    (19, 64, 193, 2, 0),
    (20, 64, 640, 2, 0),      # L = 1024
    (21, 64, 2000, 2, 0),
    (22, 513, 1540, 1, 0),
    (23, 513, 4096, 2, 0),
    (24, 513, 5000, 1, 1),
    (25, 4096, 12289, 1, 0),
    (26, 4096, 20000, 2, 0),
    (27, 21, 360001, 1, 0),   # cfg4's curve: 360 s at a 1 kHz frame rate
]
SG = [  # (seed, window, polyorder, T, rows, f32)
    (40, 3, 1, 3, 2, 0),
    (41, 3, 2, 256, 2, 0),
    (42, 5, 2, 5, 1, 0),
    (43, 5, 3, 255, 3, 0),
    (44, 5, 2, 257, 2, 1),
    (45, 6, 2, 6, 2, 0),
    (46, 6, 3, 512, 2, 0),
    (47, 11, 3, 11, 1, 0),
    (48, 11, 2, 511, 2, 0),
    (49, 11, 5, 1000, 3, 1),
    (50, 31, 3, 31, 1, 0),
    (51, 31, 4, 513, 2, 0),
    (52, 31, 7, 4097, 2, 0),
    (53, 11, 3, 360001, 1, 0),
]
VEL = [  # (seed, method, difference, param, T, f32)
    (60, "gradient", 1, 0, 2, 0),
    (61, "gradient", 1, 0, 256, 0),
    (62, "gradient", 2, 0, 1000, 1),
    (63, "finDiff", 1, 2, 257, 0),
    (64, "finDiff", 2, 2, 300, 0),
    (65, "finDiff", 1, 4, 513, 1),
    (66, "finDiff", 2, 4, 64, 0),
    (67, "sg", 1, 3, 256, 0),
    (68, "sg", 1, 7, 500, 0),
    (69, "sg", 2, 11, 1000, 1),
]


def cases():
    return [("fir",) + c for c in FIR] + [("sg",) + c for c in SG] + [("vel",) + c for c in VEL]


def case_name(c) -> str:
    return "-".join(str(v) for v in c)


def signal(seed: int, rows: int, T: int, f32: int) -> np.ndarray:
    """A smooth curve plus noise, as the change and envelope curves look: [rows, T] float64 (float32 when f32)."""
    rng = np.random.default_rng(seed)
    t = np.arange(T) / 100.0
    x = np.stack([np.sin(2 * np.pi * (0.7 + r) * t) + 0.3 * rng.standard_normal(T) for r in range(rows)])
    return x.astype(np.float32) if f32 else x


def fir_taps(seed: int, n_taps: int) -> np.ndarray:
    b = np.random.default_rng(seed + 1000).standard_normal(n_taps)
    return b / np.abs(b).sum()


def run_case(plan, c):
    """The float64 output of case c, as a host array."""
    import torch

    import modulation_mfcc_b200 as mm
    from modulation_mfcc_b200.api import _savgol_stencil

    dev = plan.device
    if c[0] == "fir":
        _, seed, n_taps, T, rows, f32 = c
        x = torch.as_tensor(signal(seed, rows, T, f32)).to(dev)
        return plan.fir_filtfilt(x, fir_taps(seed, n_taps)).cpu().numpy()
    if c[0] == "sg":
        _, seed, window, poly, T, rows, f32 = c
        x = torch.as_tensor(signal(seed, rows, T, f32)).to(dev)
        return plan.stencil(x, *_savgol_stencil(window, poly, 0)).cpu().numpy()
    _, seed, method, diff, param, T, f32 = c
    x = signal(seed, 1, T, f32)[0]
    if method == "finDiff":
        return mm.get_velocity(x, 100.0, diff, "finDiff", accOrder=param)
    if method == "sg":
        return mm.get_velocity(x, 100.0, diff, "sg", width=param, polyOrder=2 if param > 3 else 1)
    return mm.get_velocity(x, 100.0, diff, "gradient")


def digest(a: np.ndarray) -> bytes:
    return hashlib.sha256(np.ascontiguousarray(a, np.float64).tobytes()).hexdigest().encode()


def main():
    import modulation_mfcc_b200 as mm

    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "filter_bits.npz")
    plan = mm.get_plan(mm.MfccConfig(16000.0))
    names, digests = [], []
    for c in cases():
        names.append(case_name(c))
        digests.append(digest(run_case(plan, c)))
        print(names[-1], digests[-1].decode(), flush=True)
    np.savez(out, names=np.array(names), sha256=np.array(digests, "S64"))


if __name__ == "__main__":
    main()
