"""The configurations the oracle is compared on with the original MARL-LLM code (tests/test_oracle_vs_reference.py,
tests/test_replay_oracle.py: obs_dim 188, no prior, the rule / llm controllers, swarm sizes 1 to 200, periodic walls, the
replay buffer's rollover and sample), pinned without it: the restatement's outputs on seeded inputs, digest for digest, against
tests/golden/oracle_pins.npz (recorded when it matched the original on these configurations; see tests/oracle_cases.py).
CPU only: this is what keeps the oracle the GPU tests and smoke() compare with tied to the original on any machine."""
import os

import numpy as np
import pytest

from tests import oracle_cases as oc
from tests.helpers import GOLDEN

PINS = np.load(os.path.join(GOLDEN, "oracle_pins.npz"))
GROUPS = ("p/dp", "obs/reward/a_prior", "neighbor_index/in_flags/sensed_index/occupied_index")


@pytest.mark.parametrize("name", list(oc.ENV_CASES))
def test_oracle_rollout_matches_pinned_outputs(name):
    got, st = oc.run_env_case(name)
    want = PINS["env_" + name]
    assert got.shape == want.shape
    for t in range(len(want)):
        for g, what in enumerate(GROUPS):
            assert np.array_equal(got[t, g], want[t, g]), f"{what} differs from the pinned outputs at step {t - 1} ({name})"
    n_a, seed, mode, steps, self_state, method = oc.ENV_CASES[name]
    if mode == "goal" and n_a == 30 and self_state and method == "llm_rl":     # the in-shape branches were exercised
        assert st["in_shape"] > 500 and st["subsampled"] >= 1 and st["occupied"] > 1000 and st["reward"] > 0, st
    if not self_state or method != "llm_rl":
        assert st["in_shape"] > 50 or mode == "random", st
    if mode == "drift":
        assert st["wrapped"] > 10, st


def test_oracle_without_prior_leaves_a_prior_zero():
    """training_method != 'llm_rl' (assembly.py:605, 666): the prior is never computed."""
    ob = oc.start(30, 31, want_prior=False)
    ob.step(np.random.RandomState(0).uniform(-1, 1, (1, 2, 30)).astype(np.float32))
    assert not ob.a_prior.any()


@pytest.mark.parametrize("name", list(oc.STRATEGY_CASES))
def test_strategy_actions_match_pinned_outputs(name):
    got, st = oc.run_strategy_case(name)
    want = PINS["strategy_" + name]
    assert got.shape == want.shape
    for t in range(len(want)):
        assert np.array_equal(got[t], want[t]), f"{name} actions differ from the pinned ones at step {t}"
    assert st["in_shape"] > 0 and st["n_free"] > 120, st      # the directed state is far above the cap of 80 cells


def test_replay_oracle_matches_pinned_buffers_and_sample():
    got, want = oc.run_replay_case(), PINS["replay"]
    for k, what in enumerate(oc.REPLAY_FIELDS + ("cursors", "sample")):
        assert np.array_equal(got[k], want[k]), what
