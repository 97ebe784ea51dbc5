"""Mint tests/golden/hilbert_bits.npz: SHA-256 digests of mmf_hilbert_envelope outputs, to pin its bytes.

Each case is (seed, n, n_clips): the input is synth_clip(seed + i, n, 16000) for i < n_clips, stacked, and the digest
is over the whole float32 [n_clips, n] output of Plan.hilbert_envelope.  The lengths cover even, odd and prime n,
powers of two, 4097 (the first length on the FFT path), batches of several clips, both sides of the two / three
pass-group boundary of the batched FFT (2^21 and 2^21 + 1) and lengths of 2^22 and more, up to the 2^26 limit.

    python tests/golden/make_hilbert_bits.py [out.npz]     # needs a GPU; writes tests/golden/hilbert_bits.npz
"""

import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

SR = 16000
# (seed, n, n_clips)
CASES = [
    (1, 4097, 1),
    (2, 4099, 1),         # prime
    (3, 5000, 1),
    (4, 12345, 1),
    (5, 16384, 1),        # 2^14
    (6, 65536, 1),        # 2^16
    (7, 65537, 1),        # prime
    (8, 100003, 1),       # prime
    (9, 160000, 1),       # 10 s at 16 kHz
    (10, 262144, 1),      # 2^18: M = 2^19
    (11, 262145, 1),      # M = 2^20
    (20, 30011, 3),
    (30, 4098, 5),
    (40, 199999, 2),
    (50, 1 << 21, 1),     # M = 2^22: the most that two pass groups take
    (51, (1 << 21) + 1, 1),  # M = 2^23: three groups
    (52, (1 << 22) + 7, 1),  # M = 2^24
    (53, 10_000_019, 1),  # M = 2^25, prime
    (54, 1 << 26, 1),     # the longest clip: M = 2^27
]


def digest(a: np.ndarray) -> bytes:
    return hashlib.sha256(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest().encode()


def inputs(seed: int, n: int, n_clips: int) -> np.ndarray:
    from modulation_mfcc_b200.synth import synth_clip

    return np.stack([synth_clip(seed + i, n, SR) for i in range(n_clips)])


def main():
    import modulation_mfcc_b200 as mm

    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "hilbert_bits.npz")
    plan = mm.get_plan(mm.MfccConfig(SR, 512, 400, 160, 40, 13, 0.0, SR / 2))
    digests = []
    for seed, n, n_clips in CASES:
        digests.append(digest(plan.hilbert_envelope(inputs(seed, n, n_clips)).cpu().numpy()))
        print(seed, n, n_clips, digests[-1].decode(), flush=True)
    np.savez(out, cases=np.array(CASES, np.int64), sr=np.int64(SR), sha256=np.array(digests, "S64"))


if __name__ == "__main__":
    main()
