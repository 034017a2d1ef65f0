"""Buffer checkpoints (SURVEY §8f-2 / f-3): the device rings pickle like the reference's buffer objects
(`state["rb"] = rb`, utils/callback.py:37-41), `CheckpointCallback` mirrors the reference's truncated fix-up, and
buffers convert to / from the reference's own classes (objects recorded from the executed reference,
tests/golden/buffer_objects.pt) with identical subsequent samples."""
import io
import os

import numpy as np
import pytest
import torch

from oracle.ops_emul import EmulOps
from sheeprl_b200.data import buffers as RB
from sheeprl_b200.utils.callback import CheckpointCallback, load_replay_buffer
from tests.buffer_scenarios import seed_rngs, synth_rows


KINDS = ("uniform", "sequential", "env_independent")


def _rows(length, n_envs, seed):
    d = synth_rows(length, n_envs, seed)
    d["truncated"] = np.zeros((length, n_envs, 1))
    return d


def _make(kind, device="cpu", ops=None):
    ops = ops or EmulOps()
    if kind == "uniform":
        rb = RB.ReplayBuffer(12, 2, device=device, ops=ops)
        rb.add(_rows(9, 2, 1)), rb.add(_rows(7, 2, 2))                       # wrapped, full
        kw = dict(batch_size=6, sample_next_obs=True, n_samples=2)
    elif kind == "sequential":
        rb = RB.SequentialReplayBuffer(16, 2, device=device, ops=ops)
        rb.add(_rows(11, 2, 3))                                              # not full
        kw = dict(batch_size=5, sequence_length=4, n_samples=2)
    else:
        rb = RB.EnvIndependentReplayBuffer(16, 3, buffer_cls=RB.SequentialReplayBuffer, device=device, ops=ops)
        rb.add(_rows(11, 3, 4)), rb.add(_rows(9, 2, 5), indices=[0, 2])      # two of the three rings wrapped
        kw = dict(batch_size=8, sequence_length=4, n_samples=2)
    seed_rngs(rb, 77)
    return rb, kw


def _heads(rb):
    rings = rb.buffer if isinstance(rb, RB.EnvIndependentReplayBuffer) else [rb]
    return [(r._pos, r._full) for r in rings]


def _same_samples(a, b, kw):
    sa, sb = a.sample(**kw), b.sample(**kw)
    assert sorted(sa) == sorted(sb)
    for k in sa:
        assert sa[k].dtype == sb[k].dtype and np.array_equal(sa[k], sb[k]), k


@pytest.mark.parametrize("kind", KINDS)
def test_pickle_round_trip_continues_identically(kind):
    a, kw = _make(kind)
    bio = io.BytesIO()
    torch.save({"rb": a}, bio)
    bio.seek(0)
    b = load_replay_buffer(torch.load(bio, weights_only=False)["rb"], device="cpu", ops=EmulOps())
    assert type(b) is type(a) and _heads(a) == _heads(b)
    _same_samples(a, b, kw)
    extra = _rows(5, a.n_envs, 9)                                            # both keep working after the restore
    a.add(extra), b.add(extra)
    assert _heads(a) == _heads(b)
    _same_samples(a, b, kw)


class _Fabric:
    world_size, global_rank, is_global_zero = 1, 0, True

    def save(self, path, state):
        torch.save(state, path)


@pytest.mark.parametrize("kind", ["uniform", "env_independent"])
def test_checkpoint_callback_marks_the_last_step_truncated_only_in_the_file(kind, tmp_path):
    rb, kw = _make(kind)
    rings = rb.buffer if kind == "env_independent" else [rb]
    before = [r["truncated"].clone() for r in rings]
    cb = CheckpointCallback(keep_last=2)
    for i in range(3):
        cb.on_checkpoint_coupled(_Fabric(), str(tmp_path / f"ckpt_{i}.ckpt"), {"iter_num": i}, rb)
        os.utime(tmp_path / f"ckpt_{i}.ckpt", (i + 1, i + 1))
    assert sorted(p.name for p in tmp_path.glob("*.ckpt")) == ["ckpt_1.ckpt", "ckpt_2.ckpt"]          # keep_last
    for r, t in zip(rings, before):
        assert torch.equal(r["truncated"], t)                                # live buffer untouched afterwards
    state = torch.load(tmp_path / "ckpt_2.ckpt", weights_only=False)
    saved = load_replay_buffer(state["rb"], device="cpu", ops=EmulOps())
    for r, s in zip(rings, saved.buffer if kind == "env_independent" else [saved]):
        row = (r._pos - 1) % r.buffer_size
        assert bool((s["truncated"][row] == 1).all())                        # the episode ends in the checkpoint
        mask = torch.ones(r.buffer_size, dtype=torch.bool)
        mask[row] = False
        assert torch.equal(s["truncated"][mask], r["truncated"][mask])


def _reference_object(rec):
    """a reference buffer object as recorded by oracle/make_golden_buffer_objects.py: the reference's class name and
    attributes (what `load_replay_buffer` and `from_reference` see of it), without the reference's code"""
    attrs = dict(rec["attrs"])
    st = attrs["_rng"]
    attrs["_rng"] = np.random.Generator(getattr(np.random, st["bit_generator"])())
    attrs["_rng"].bit_generator.state = st
    if isinstance(attrs["_buf"], list):
        attrs["_buf"] = [_reference_object(r) for r in attrs["_buf"]]
    obj = type(rec["class"], (), {})()
    obj.__dict__.update(attrs)
    return obj


@pytest.mark.parametrize("kind", KINDS)
def test_conversion_to_and_from_the_reference_classes(kind, golden_dir):
    """ours -> reference: the object the reference's class built from this buffer (`to_reference`, through its pickle)
    holds our rows, write heads and Generator state; reference -> ours: adopting that object (as found in a reference
    checkpoint) samples exactly what the reference sampled from it."""
    rec = torch.load(os.path.join(golden_dir, "buffer_objects.pt"), weights_only=False)[kind]
    mine, kw = _make(kind)
    assert kw == rec["sample_kwargs"]
    ref = _reference_object(rec["object"])
    assert type(ref).__name__ == type(mine).__name__
    rings = mine.buffer if isinstance(mine, RB.EnvIndependentReplayBuffer) else [mine]
    ref_rings = ref._buf if isinstance(mine, RB.EnvIndependentReplayBuffer) else [ref]
    assert [(r._pos, r._full) for r in ref_rings] == _heads(mine)
    for r, theirs in zip(rings, ref_rings):
        assert sorted(theirs._buf) == sorted(r._buf)
        rows = r.buffer_size if r._full else r._pos                         # rows past the write head hold no data
        for k, v in theirs._buf.items():
            ours = r[k].cpu().numpy()
            assert v.dtype == ours.dtype and v.shape == ours.shape and np.array_equal(v[:rows], ours[:rows]), k
        assert theirs._rng.bit_generator.state == r._rng.bit_generator.state
    assert ref._rng.bit_generator.state == mine._rng.bit_generator.state
    back = load_replay_buffer(ref, device="cpu", ops=EmulOps())
    assert type(back) is type(mine) and _heads(back) == _heads(mine)
    got = back.sample(**kw)
    assert sorted(got) == sorted(rec["sample"])
    for k, want in rec["sample"].items():
        assert want.dtype == got[k].dtype and np.array_equal(want, got[k]), (kind, k)
