"""Why the B200 engine accepts only `distribution.type` = auto / scaled_normal for continuous Dreamer-V3 actions: the
REFERENCE's own train() does not run with the other two values (executed here, container only).

  * tanh_normal: the entropy of the transformed distribution is not implemented, the fallback at dreamer_v3.py:294-297
    builds a `[H, N, 1, 1]` tensor and the broadcast against the `[H, N, 1]` objective fails;
  * normal: `Normal(mean, std)` is built from the raw head output (agent.py:812-814), i.e. with negative scales.

`DV3Engine` raises NotImplementedError for both instead of silently training something else."""
import copy

import pytest
import torch

from oracle import dv3_oracle as O
from oracle import ref_harness
from tests.helpers import load_fixture

# the first two execute the reference itself; the engine test below needs nothing outside the repository
needs_reference = pytest.mark.skipif(not ref_harness.reference_available(), reason="reference tree not present")


def _setup(dist_type):
    fx, cfg = load_fixture("dv3_tiny_c")
    cfg = copy.deepcopy(cfg)
    cfg.distribution.type = dist_type
    cfg.distribution.validate_args = True        # torch's own argument checks, as a user debugging this would set
    return fx, cfg


@needs_reference
@pytest.mark.parametrize("dist_type", ["tanh_normal", "normal"])
def test_reference_train_fails_with_this_distribution(dist_type):
    from oracle import ref_run

    fx, cfg = _setup(dist_type)
    adim = fx["actions_dim"]
    data = [{k: v.float() for k, v in fx["data"][0].items()}]
    with pytest.raises((RuntimeError, ValueError, NotImplementedError)):
        ref_run.run_reference_train(cfg, adim, data, [fx["noise"][0]], n_steps=1, state=fx["init"], is_continuous=True)


@needs_reference
def test_reference_train_runs_with_the_supported_distribution():
    """control: the same harness and fixture DO run with scaled_normal (what the fixture was generated with)"""
    from oracle import ref_run

    fx, cfg = _setup("scaled_normal")
    data = [{k: v.float() for k, v in fx["data"][0].items()}]
    _, metrics, _ = ref_run.run_reference_train(cfg, fx["actions_dim"], data, [fx["noise"][0]], n_steps=1, state=fx["init"],
                                                is_continuous=True)
    assert all(torch.isfinite(torch.tensor(v)) for v in metrics[0].values())


@pytest.mark.parametrize("dist_type", ["tanh_normal", "normal"])
def test_engine_refuses_the_same_distributions(dist_type):
    from oracle.ops_emul import EmulOps
    from sheeprl_b200.engine import DV3Engine

    fx, cfg = _setup(dist_type)
    with pytest.raises(NotImplementedError):
        DV3Engine(cfg, fx["actions_dim"], in_channels=3, device="cpu", ops=EmulOps(), is_continuous=True)
