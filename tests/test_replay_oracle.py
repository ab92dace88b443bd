"""Pins oracle/replay_oracle.py to the reference's own ReplayBufferAgent (imported from the checkout of the original project that
oracle/live_reference.py locates, when present; tests/test_oracle_pins.py keeps the pin where it is not)."""
import os
import sys

import numpy as np
import pytest

from oracle.live_reference import REF_ROOT
from oracle.replay_oracle import ReplayOracle

REF = os.path.join(REF_ROOT, "marl_llm", "algorithm", "utils")


def _ref_class():
    if not os.path.isdir(REF):
        pytest.skip("reference checkout not present on this box")
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_buffer_agent", os.path.join(REF, "buffer_agent.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    return m.ReplayBufferAgent


def test_replay_oracle_matches_reference_push_rollover_and_sample():
    Ref = _ref_class()
    n_a, D, A, max_steps = 30, 12, 2, 10007          # 300 210 rows: just above the 3e5 window of BUF:147
    idx = slice(0, n_a)
    ref, orc = Ref(max_steps, n_a, idx, D, A), ReplayOracle(max_steps, n_a, idx, D, A)
    rng = np.random.RandomState(0)
    # jump the cursors close to the end so that the step-back branch (BUF:96-99) and the wrap to 0 are exercised
    for b in (ref, orc):
        b.curr_i = b.filled_i = b.total_length - 3 * n_a - 7
    for t in range(6):
        obs, nxt = rng.randn(D, n_a), rng.randn(D, n_a)
        act, prior = rng.uniform(-1, 1, (A, n_a)).astype(np.float32), rng.uniform(-1, 1, (A, n_a))
        rew, done = rng.rand(1, n_a), rng.rand(1, n_a) > 0.5
        ref.push(obs, act, rew, nxt, done, idx, prior)
        orc.push(obs, act, rew, nxt, done, idx, prior)
        assert (ref.curr_i, ref.filled_i) == (orc.curr_i, orc.filled_i), t
    for name in ("obs_buffs", "ac_buffs", "ac_prior_buffs", "rew_buffs", "next_obs_buffs", "done_buffs", "log_pi_buffs"):
        assert np.array_equal(getattr(ref, name), getattr(orc, name)), name
    np.random.seed(5); got_ref = ref.sample(64, to_gpu=False, is_prior=True)
    np.random.seed(5); got_orc, _ = orc.sample(64, is_prior=True)
    for a, b in zip(got_ref, got_orc):
        assert (a is None) == (b is None)
        if a is not None:
            assert np.array_equal(a.numpy(), b)


def test_batched_push_equals_sequential_single_env_pushes():
    n_a, D, A, E = 5, 8, 2, 7
    idx = slice(0, n_a)
    one, many = ReplayOracle(100, n_a, idx, D, A), ReplayOracle(100, n_a, idx, D, A)
    rng = np.random.RandomState(1)
    obs, nxt = rng.randn(E, D, n_a), rng.randn(E, D, n_a)
    act, prior = rng.randn(E, A, n_a), rng.randn(E, A, n_a)
    rew, done = rng.rand(E, 1, n_a), rng.rand(E, 1, n_a) > 0.5
    many.push(obs, act, rew, nxt, done, idx, prior)
    for e in range(E):
        one.push(obs[e], act[e], rew[e], nxt[e], done[e], idx, prior[e])
    for name in ("obs_buffs", "ac_buffs", "ac_prior_buffs", "rew_buffs", "next_obs_buffs", "done_buffs"):
        assert np.array_equal(getattr(one, name), getattr(many, name)), name
    assert (one.curr_i, one.filled_i) == (many.curr_i, many.filled_i)
