"""TEST INFRASTRUCTURE — writes tests/golden/dv3_pin.pt by EXECUTING THE REAL REFERENCE (container only):

    python -m oracle.make_golden_pin

The second pin of the oracle (tests/test_oracle_pin.py): the dv3_tiny_a configuration from another initialisation
(reference `build_agent` under seed 3, perturbed), two `train()` steps.  Batches and noise are regenerated from their
seeds by the consumer (oracle/make_golden.py:build_case draws them the same way), so the fixture holds only the
initial state and what the unmodified reference produced: post-step parameters and Moments.
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.make_golden import FIXTURES, GOLDEN, build_case  # noqa: E402

SPEC, SEED = "dv3_tiny_a", 3


def main():
    _, _, sd, _, _, after, metrics, moments, _ = build_case(dict(FIXTURES[SPEC]), seed=SEED)
    path = os.path.join(GOLDEN, "dv3_pin.pt")
    torch.save({"spec": SPEC, "seed": SEED, "init": sd, "after": after, "moments": moments}, path)
    print(f"wrote {path}: {os.path.getsize(path)} bytes", {k: round(v, 5) for k, v in metrics[-1].items()})


if __name__ == "__main__":
    main()
