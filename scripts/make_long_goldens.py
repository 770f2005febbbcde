"""Generates the long-clip reference fixtures (tests/golden/vid73x64.pt, vid261x64.pt, vae_vid73x64.pt) with the
recipe of oracle/make_golden.py: the unmodified reference on seeded synthetic weights and inputs.

    OMT_REFERENCE_ROOT=<checkout> python -m scripts.make_long_goldens [fixture names]

The clips are long enough to cross the latent-frame ranges of the kernels: T' = 19 > 17 runs the chunked temporal
attention kernel, and T' = 66 also takes PEG past the v4 kernel's T' <= 64 (the v3 fallback).  The fixtures only append
to make_golden's case list, so the existing fixtures are neither touched nor regenerated.
"""
import sys

from oracle import make_golden as mg

LONG_CASES = [
    # name, argv extras, input shape, weight seed, input seed
    ("vid73x64", [], (1, 3, 73, 64, 64), 5, 1241),
    ("vid261x64", [], (1, 3, 261, 64, 64), 5, 1242),
    ("vae_vid73x64", ["--use_vae"], (1, 3, 73, 64, 64), 2, 1243),
]


def main(names=()):
    names = list(names) or [c[0] for c in LONG_CASES]
    unknown = set(names) - {c[0] for c in LONG_CASES}
    if unknown:
        raise SystemExit(f"unknown long-clip fixtures {sorted(unknown)}")
    mg.CASES = mg.CASES + [c for c in LONG_CASES if c[0] not in {m[0] for m in mg.CASES}]
    mg.main(names)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
