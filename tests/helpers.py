"""Shared helpers for the parity tests (test infrastructure)."""
import os

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")


def load_shapes():
    z = np.load(os.path.join(GOLDEN, "shapes.npz"))
    n_g = z["n_g"]
    return dict(l_cell=z["l_cell"].copy(), n_g=n_g.copy(),
                grid_origin=[np.ascontiguousarray(z["grid_coords"][k, :n_g[k]].T) for k in range(len(n_g))])


def goal_seeking_action(obs, dp, rng, noise=0.3, target_row=28):
    """Noisy PD controller towards the target cell (obs rows 28:30 = target - p; 24:26 without the self-state column): drives
    agents into the shape so the in-shape / occupancy / subsample / reward branches are exercised."""
    a = 3.0 * obs[..., target_row:target_row + 2, :] - 1.0 * dp + rng.normal(0, noise, dp.shape)
    return np.clip(a, -1, 1).astype(np.float32)


def expected_grids(info, shapes):
    """Grids of a device reset rebuilt from its draws (rows of reset_info): grid_center = R.origin + offset with the reference's
    separately rounded products and sums (assembly.py:175-187)."""
    grids = []
    for row in info:
        k, c, s, ox, oy = int(row[0]), row[1], row[2], row[3], row[4]
        g = shapes["grid_origin"][k]
        gx = (c * g[0] + s * g[1]) + ox
        gy = ((-s) * g[0] + c * g[1]) + oy
        grids.append(np.stack([gx, gy]))
    return grids


def oracle_follow_reset(ob, sim, shapes, rows, pick=None):
    """After sim.reset / reset_envs: rebuild the oracle's envs `rows` from sim.reset_info (n_g, l_cell and grid from the shape
    library `shapes`; p / dp from the simulator, whose values are the reference's map of the draws) and re-observe.  Oracle env k
    is simulator env pick[k] (all envs in order without pick).  The oracle's observe must leave every other env's outputs as
    they were: asserted."""
    import torch
    rows = np.asarray(rows, dtype=np.int64)
    envs = rows if pick is None else np.asarray(pick)[rows]
    te = torch.as_tensor(envs, device=sim.device)
    info = sim.reset_info[te].cpu().numpy()
    for k, row, g in zip(rows, info, expected_grids(info, shapes)):
        ob.params[k].n_g = g.shape[1]
        ob.params[k].l_cell = float(shapes["l_cell"][int(row[0])])
        ob.set_grid(k, g)
    ob.p[rows], ob.dp[rows] = sim.p[te].cpu().numpy(), sim.dp[te].cpu().numpy()
    keep = np.setdiff1d(np.arange(ob.E), rows)
    names = ("obs", "neighbor_index", "in_flags", "sensed_index", "occupied_index")
    before = [getattr(ob, n)[keep].copy() for n in names]
    ob.observe()
    for n, b in zip(names, before):
        assert np.array_equal(getattr(ob, n)[keep], b), f"oracle observe is not idempotent on {n}"


def reset_like_reference(rng, n_a, shapes, half=2.4):
    """Domain randomisation in the spirit of assembly.py:156-223 (own RNG stream, not NumPy-global)."""
    k = int(rng.randint(0, len(shapes["l_cell"])))
    ang = np.pi * rng.uniform(-1, 1)
    R = np.array([[np.cos(ang), np.sin(ang)], [-np.sin(ang), np.cos(ang)]])
    off = rng.uniform(-half + 1, half - 1, (2, 1))
    grid = np.dot(R, shapes["grid_origin"][k]) + off
    if rng.uniform(-1, 1) > 0:
        p = rng.uniform(-half, half, (2, n_a))
    else:
        p = rng.uniform(-1, 1, (2, n_a)) + rng.uniform(-half + 1, half - 1, (2, 1))
    dp = rng.uniform(-0.5, 0.5, (2, n_a))
    return k, np.ascontiguousarray(grid), p, dp


import hashlib  # noqa: E402


def sha(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


GOLDEN_CASES = ["a30_random_s226", "a30_goal_s3", "a10_goal_s15", "a64_goal_s75", "a30_periodic_s7"]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, f"traj_{name}.npz"))
    return {k: z[k] for k in z.files}


def replay_golden(g, reset_fn, step_fn, atol=0.0, obs_cast=None):
    """Replays a golden trajectory through an implementation and compares every recorded field.

    reset_fn(g) -> dict(obs, nbr, in_flags, sensed, occupied) after observing the golden initial state
    step_fn(act[2,n_a] f32) -> dict(p, dp, obs, reward, a_prior, nbr, in_flags, sensed, occupied)
    atol == 0 demands bit-exact floating point (integer fields are always exact).
    obs_cast: optional dtype the implementation emits obs/reward/prior in (golden is cast the same way).
    """
    def feq(a, b, what, t):
        b = np.asarray(b)
        if obs_cast is not None and what in ("obs", "reward", "a_prior"):
            b = b.astype(obs_cast)
        a = np.asarray(a).reshape(b.shape)
        if atol == 0.0:
            assert np.array_equal(a, b, equal_nan=True), f"{what} not bit-exact at step {t}: max|d|={np.nanmax(np.abs(a - b))}"
        else:
            assert np.allclose(a, b, rtol=atol, atol=atol, equal_nan=True), f"{what} differs at step {t}"

    def ieq(a, b, what, t):
        assert np.array_equal(np.asarray(a).reshape(np.asarray(b).shape).astype(np.int64), np.asarray(b).astype(np.int64)), \
            f"{what} differs at step {t}"

    r = reset_fn(g)
    feq(r["obs"], g["obs0"], "obs", -1)
    ieq(r["nbr"], g["nbr0"], "neighbor_index", -1)
    ieq(r["in_flags"], g["in_flags0"], "in_flags", -1)
    ieq(r["sensed"], g["sensed0"], "sensed_index", -1)
    ieq(r["occupied"], g["occupied0"], "occupied_index", -1)
    full = {int(t): k for k, t in enumerate(g["full_steps"])}
    for t in range(int(g["steps"])):
        s = step_fn(g["act"][t])
        feq(s["p"], g["p"][t], "p", t)
        feq(s["dp"], g["dp"][t], "dp", t)
        feq(s["reward"], g["reward"][t], "reward", t)
        feq(s["a_prior"], g["a_prior"][t], "a_prior", t)
        ieq(s["nbr"], g["neighbor_index"][t], "neighbor_index", t)
        ieq(s["in_flags"], g["in_flags"][t], "in_flags", t)
        if obs_cast is None and atol == 0.0:
            assert sha(np.asarray(s["obs"], dtype=np.float64)) == g["sha_obs"][t], f"obs digest differs at step {t}"
        assert sha(np.asarray(s["sensed"], dtype=np.int32)) == g["sha_sensed"][t], f"sensed_index digest differs at step {t}"
        assert sha(np.asarray(s["occupied"], dtype=np.int32)) == g["sha_occupied"][t], f"occupied_index digest differs at step {t}"
        if t in full:
            k = full[t]
            feq(s["obs"], g["full_obs"][k], "obs", t)
            ieq(s["sensed"], g["full_sensed"][k], "sensed_index", t)
            ieq(s["occupied"], g["full_occupied"][k], "occupied_index", t)
