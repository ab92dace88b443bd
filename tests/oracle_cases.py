"""The configurations tests/test_oracle_vs_reference.py and tests/test_replay_oracle.py compare with the original MARL-LLM code,
restated on seeded inputs so that they run without it (test infrastructure).

Each case runs the C restatement (oracle/) and returns, per step, 8-byte BLAKE2b digests of three groups of outputs: state (p, dp),
observation outputs (obs, reward, a_prior) and index outputs (neighbor_index, in_flags, sensed_index, occupied_index); strategy
cases digest the controller's actions, the replay case the buffers and a sample() after the rollover.  tests/golden/
make_oracle_pins.py stored these digests in tests/golden/oracle_pins.npz from the restatement as it stood when it matched the
original bit for bit on these configurations (and the strategies to 1e-12); tests/test_oracle_pins.py recomputes them, so a
change to the restatement that would break that agreement shows up on any machine.  Initial states come from
tests.helpers.reset_like_reference, not from the original's reset(), so these are not the original's own trajectories."""
import hashlib

import numpy as np

from oracle import oracle as orc
from tests.helpers import goal_seeking_action, load_shapes, reset_like_reference

# name -> (n_a, seed, mode, steps, is_con_self_state, training_method); modes as in test_oracle_vs_reference.py
ENV_CASES = {
    "random_a30_s226": (30, 226, "random", 200, True, "llm_rl"),
    "random_a30_s1": (30, 1, "random", 200, True, "llm_rl"),
    "random_a30_s2": (30, 2, "random", 200, True, "llm_rl"),
    "goal_a30_s226": (30, 226, "goal", 200, True, "llm_rl"),
    "goal_a30_s3": (30, 3, "goal", 200, True, "llm_rl"),
    "goal_a1_s12": (1, 12, "goal", 20, True, "llm_rl"),
    "goal_a2_s13": (2, 13, "goal", 50, True, "llm_rl"),
    "goal_a10_s21": (10, 21, "goal", 100, True, "llm_rl"),
    "goal_a64_s75": (64, 75, "goal", 60, True, "llm_rl"),
    "goal_a200_s211": (200, 211, "goal", 10, True, "llm_rl"),
    "noself_goal_a30_s21": (30, 21, "goal", 150, False, "llm_rl"),
    "noself_goal_a31_s22": (31, 22, "goal", 100, False, "llm_rl"),
    "noself_goal_a7_s23": (7, 23, "goal", 100, False, "llm_rl"),
    "noself_random_a30_s24": (30, 24, "random", 100, False, "llm_rl"),
    "noprior_manual_rl_a30_s31": (30, 31, "goal", 120, True, "manual_rl"),
    "noprior_irl_noself_a30_s31": (30, 31, "goal", 120, False, "irl"),
    "periodic_a30_s7": (30, 7, "drift", 150, True, "llm_rl"),
    "periodic_a30_s8": (30, 8, "drift", 150, True, "llm_rl"),
}
# name -> (strategy, n_a, seed); 150 steps each, then one directed state for the 80-cell subsample of the controllers
STRATEGY_CASES = {"rule_a30_s4": ("rule", 30, 4), "rule_a12_s9": ("rule", 12, 9), "llm_a30_s6": ("llm", 30, 6), "llm_a8_s2": ("llm", 8, 2)}


def digest(*arrays):
    h = hashlib.blake2b(digest_size=8)
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def start(n_a, seed, **param_kw):
    shapes = load_shapes()
    k, grid, p, dp = reset_like_reference(np.random.RandomState(seed), n_a, shapes)
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    ob = orc.OracleBatch([orc.make_params(n_a, grid.shape[1], float(shapes["l_cell"][k]), r_avoid, **param_kw)])
    ob.set_grid(0, grid)
    ob.p[0], ob.dp[0] = p, dp
    ob.observe()
    return ob


def _groups(ob):
    return np.stack([digest(ob.p[0], ob.dp[0]), digest(ob.obs[0], ob.reward[0], ob.a_prior[0]),
                     digest(ob.neighbor_index[0], ob.in_flags[0], ob.sensed_index[0], ob.occupied_index[0])])


def run_env_case(name):
    """-> (digests [steps + 1, 3, 8] uint8, stats of the branches the rollout went through)"""
    n_a, seed, mode, steps, self_state, method = ENV_CASES[name]
    ob = start(n_a, seed, is_con_self_state=self_state, want_prior=method == "llm_rl", is_periodic=mode == "drift")
    out = [_groups(ob)]
    rng = np.random.RandomState(seed + 1)
    stats = dict(in_shape=0, subsampled=0, occupied=0, reward=0.0, wrapped=0)
    for t in range(steps):
        if mode == "random":
            a = rng.uniform(-1, 1, (2, n_a)).astype(np.float32)
        elif mode == "drift":                                 # outward drift: agents cross the box edges and wrap
            a = np.clip(0.8 * np.sign(ob.p[0]) + rng.normal(0, 0.5, (2, n_a)), -1, 1).astype(np.float32)
        else:
            a = goal_seeking_action(ob.obs[0], ob.dp[0], rng, target_row=28 if self_state else 24)
        before = ob.p[0].copy()
        ob.step(a[None])
        out.append(_groups(ob))
        stats["in_shape"] += int(ob.in_flags.sum())
        stats["occupied"] += int((ob.occupied_index >= 0).sum())
        stats["subsampled"] += int(((ob.sensed_index[0] >= 0).sum(1) == 80).sum())
        stats["reward"] += float(ob.reward.sum())
        stats["wrapped"] += int((np.abs(ob.p[0] - before) > 2.0).sum())
    return np.stack(out), stats


def run_strategy_case(name):
    """-> (digests [150 + 1, 8] uint8: the actions of every step, then those of the directed state, stats).  The state is
    advanced by the restatement with the controller's actions rounded to float32 (the action type of its step)."""
    kind, n_a, seed = STRATEGY_CASES[name]
    ob = start(n_a, seed)
    out, in_shape = [], 0
    for t in range(150):
        u = orc.strategy_actions(ob, kind)
        out.append(digest(u))
        ob.step(u.astype(np.float32))
        in_shape += int(ob.in_flags.sum())
    # agents on cells deep inside the shape with a small avoidance radius keep far more than 80 free cells in range
    grid = ob.grid_of(0).copy()
    P2 = orc.make_params(n_a, grid.shape[1], float(ob.params[0].l_cell), 0.05, d_sen=0.6)
    ob2 = orc.OracleBatch([P2])
    ob2.set_grid(0, grid)
    order = np.argsort(np.linalg.norm(grid - grid.mean(axis=1, keepdims=True), axis=0))[:n_a * 3:3]
    ob2.p[0] = grid[:, order] + np.random.RandomState(seed).normal(0, 0.004, (2, n_a))
    ob2.dp[0] = np.random.RandomState(seed + 1).uniform(-0.2, 0.2, (2, n_a))
    ob2.observe()                                             # neighbour list for the 'llm' controller
    out.append(digest(orc.strategy_actions(ob2, kind)))
    n_free = max(int((np.linalg.norm(grid - ob2.p[0][:, [i]], axis=0) < 0.6).sum()) for i in range(n_a))
    return np.stack(out), dict(in_shape=in_shape, n_free=n_free)


REPLAY_FIELDS = ("obs_buffs", "ac_buffs", "ac_prior_buffs", "rew_buffs", "next_obs_buffs", "done_buffs", "log_pi_buffs")


def run_replay_case():
    """Pushes that run past the end of a 300 210-row buffer (step-back branch and wrap to 0), then sample(64, is_prior=True)
    -> digests [len(REPLAY_FIELDS) + 2, 8] uint8: every buffer, the cursors, the sampled tensors."""
    from oracle.replay_oracle import ReplayOracle
    n_a, D, A, max_steps = 30, 12, 2, 10007
    idx = slice(0, n_a)
    b = ReplayOracle(max_steps, n_a, idx, D, A)
    b.curr_i = b.filled_i = b.total_length - 3 * n_a - 7
    rng = np.random.RandomState(0)
    for t in range(6):
        obs, nxt = rng.randn(D, n_a), rng.randn(D, n_a)
        act, prior = rng.uniform(-1, 1, (A, n_a)).astype(np.float32), rng.uniform(-1, 1, (A, n_a))
        rew, done = rng.rand(1, n_a), rng.rand(1, n_a) > 0.5
        b.push(obs, act, rew, nxt, done, idx, prior)
    out = [digest(getattr(b, name)) for name in REPLAY_FIELDS]
    out.append(digest(np.array([b.curr_i, b.filled_i], dtype=np.int64)))
    np.random.seed(5)
    got, _ = b.sample(64, is_prior=True)
    out.append(digest(*[np.asarray(x) for x in got if x is not None], np.array([x is None for x in got])))
    return np.stack(out)
