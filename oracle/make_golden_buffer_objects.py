"""TEST INFRASTRUCTURE — writes tests/golden/buffer_objects.pt by EXECUTING THE REAL REFERENCE buffers (container only):

    python -m oracle.make_golden_buffer_objects

For each buffer of tests/test_buffer_checkpoint_cpu.py: the reference object `to_reference` builds from it after a
pickle round trip (what a reference checkpoint holds as `state["rb"]`), recorded as its attributes with the Generator
as its bit-generator state, and what that object's `sample()` returned.  Memmap-backed objects hold the same arrays
and sample the same rows; that is checked here rather than stored twice.
"""
from __future__ import annotations

import io
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness  # noqa: E402
from tests.test_buffer_checkpoint_cpu import KINDS, _make  # noqa: E402


def _record(obj):
    st = {}
    for k, v in obj.__dict__.items():
        if k == "_rng":
            v = v.bit_generator.state
        elif k == "_buf" and isinstance(v, dict):
            v = {key: np.array(a) for key, a in v.items()}
        elif k == "_buf":
            v = [_record(ring) for ring in v]
        st[k] = v
    return {"class": type(obj).__name__, "attrs": st}


def _pickled(ref):
    bio = io.BytesIO()
    torch.save({"rb": ref}, bio)
    bio.seek(0)
    return torch.load(bio, weights_only=False)["rb"]


def main():
    ref_harness.install()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        for kind in KINDS:
            mine, kw = _make(kind)
            ref = _pickled(mine.to_reference())
            obj = _record(ref)
            want = ref.sample(**kw)
            mm = _pickled(mine.to_reference(memmap=True, memmap_dir=os.path.join(tmp, kind)))
            got = mm.sample(**kw)
            assert all(np.array_equal(np.asarray(want[k]), np.asarray(got[k])) for k in want), kind
            out[kind] = {"object": obj, "sample_kwargs": kw, "sample": {k: np.asarray(v) for k, v in want.items()}}
    path = os.path.join(ROOT, "tests", "golden", "buffer_objects.pt")
    torch.save(out, path)
    print(f"wrote {path}: {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
