"""Pins the oracle against the executed reference from a second initialisation (tests/golden/dv3_pin.pt, written by
oracle/make_golden_pin.py from the unmodified reference train())."""
import os

import pytest
import torch

from oracle import dv3_oracle as O
from tests.helpers import GOLDEN


def test_oracle_equals_live_reference_two_steps():
    from oracle.make_golden import FIXTURES
    from sheeprl_b200.configs import make_dv3_cfg
    from tests.helpers import assert_params_close

    fx = torch.load(os.path.join(GOLDEN, "dv3_pin.pt"), weights_only=False)
    spec = FIXTURES[fx["spec"]]
    cfg, adim, steps = make_dv3_cfg(**spec["cfg"]), tuple(spec["actions_dim"]), spec["steps"]
    a, w = cfg.algo, cfg.algo.world_model
    T, B, H = a.per_rank_sequence_length, a.per_rank_batch_size, a.horizon
    cp = [{k: v.clone() for k, v in fx["init"][n].items()} for n in ("wm", "actor", "critic", "target")]
    opts = [O.AdamState(cp[0], w.optimizer.lr, w.optimizer.eps), O.AdamState(cp[1], a.actor.optimizer.lr, a.actor.optimizer.eps),
            O.AdamState(cp[2], a.critic.optimizer.lr, a.critic.optimizer.eps)]
    ms = {"low": torch.zeros(()), "high": torch.zeros(())}
    for s in range(steps):                       # the batches and noise the reference ran on (make_golden.build_case)
        data = O.make_batch(cfg, adim, seed=1 + s)
        noise = O.draw_noise(T, B, H, w.stochastic_size, w.discrete_size, adim, seed=10 + s)
        O.dv3_train_step(cfg, *cp, *opts, data, noise, ms, adim, condition_margin=1e-3)
    for i, n in enumerate(("wm", "actor", "critic")):
        assert_params_close(cp[i], fx["after"][n], 1e-4, 2, label=n)
    assert float(ms["low"]) == pytest.approx(float(fx["moments"]["low"]), rel=1e-5, abs=1e-7)


def test_reference_multinomial_is_argmax_p_over_exp():
    """SURVEY App. B: torch.multinomial(p,1,True) == argmax(p / Exp(1)) on the same generator state."""
    g = torch.Generator().manual_seed(7)
    p = torch.softmax(torch.randn(64, 32, generator=g), -1)
    st = g.get_state()
    idx = torch.multinomial(p, 1, True, generator=g)
    g.set_state(st)
    q = torch.empty_like(p).exponential_(1, generator=g)
    assert torch.equal(idx.squeeze(-1), (p / q).argmax(-1))
