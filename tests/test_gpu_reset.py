"""On-device reset() (SURVEY.md §8 f3): the domain randomisation of assembly.py:156-223 from a device-resident shape library.
The random draws are the device generator's; everything derived from them must be the reference's arithmetic: the test
reads the drawn (shape, cos, sin, offset) back, rebuilds grid_center = R.origin + offset with NumPy (separately rounded
products and sums, like np.dot on a 2x2 by 2xN without FMA would give) and requires the device grid, the first observation and
a rollout from that state to be bit-identical to the oracle's."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.helpers import expected_grids, goal_seeking_action, load_shapes

pytestmark = pytest.mark.gpu


def make(E, n_a=30, **kw):
    from marl_llm_b200.batched import BatchedAssemblySim
    shapes = load_shapes()
    ngm = int(shapes["n_g"].max())
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    sim = BatchedAssemblySim(E, n_a, ngm, r_avoid, out_dtype=torch.float64, emit_indices=True, **kw)
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    return sim, shapes, r_avoid, ngm


def test_reset_state_is_the_reference_map_of_the_draws_and_rollout_matches_oracle():
    E, n_a = 96, 30
    sim, shapes, r_avoid, ngm = make(E, n_a)
    sim.reset(seed=226, episode=0)
    info = sim.reset_info.cpu().numpy()
    k = info[:, 0].astype(int)
    assert k.min() >= 0 and k.max() < 7 and len(np.unique(k)) >= 5
    assert np.allclose(info[:, 1] ** 2 + info[:, 2] ** 2, 1.0, atol=1e-12)
    assert (np.abs(info[:, 3:5]) <= 1.4).all() and set(np.unique(info[:, 5])) <= {0.0, 1.0}
    grids = expected_grids(info, shapes)
    dev_grid = sim._grid.cpu().numpy()            # [E, n_g_pad, 2] cell-major internal copy
    n_g = sim._n_g.cpu().numpy()
    for e in range(E):
        assert n_g[e] == grids[e].shape[1]
        assert np.array_equal(dev_grid[e, :n_g[e]].T, grids[e]), e
        assert (dev_grid[e, n_g[e]:] == 1e30).all()
    p, dp = sim.p.cpu().numpy(), sim.dp.cpu().numpy()
    assert (np.abs(p) <= 2.4 + 1e-12).all() and (np.abs(dp) <= 0.5).all()
    wide = info[:, 5] > 0
    assert wide.any() and (~wide).any()
    assert (np.ptp(p[~wide], axis=2) <= 2.0).all()            # clustered spawn: U(-1,1) around a centre (assembly.py:207)
    # p / dp rebuilt exactly from the generator's draws with the reference's map (assembly.py:202-208, 215)
    env_id, ia = np.arange(E)[:, None], np.arange(n_a)[None, :]
    ux, uy = orc.reset_uniform(226, 0, env_id, 16 + ia), orc.reset_uniform(226, 0, env_id, 16 + n_a + ia)
    px = np.where(wide[:, None], -2.4 + 2.0 * 2.4 * ux, (-1.0 + 2.0 * ux) + info[:, 6:7])
    py = np.where(wide[:, None], -2.4 + 2.0 * 2.4 * uy, (-1.0 + 2.0 * uy) + info[:, 7:8])
    assert np.array_equal(p[:, 0], px) and np.array_equal(p[:, 1], py)
    assert np.array_equal(dp[:, 0], -0.5 + orc.reset_uniform(226, 0, env_id, 16 + 2 * n_a + ia))
    assert np.array_equal(dp[:, 1], -0.5 + orc.reset_uniform(226, 0, env_id, 16 + 3 * n_a + ia))
    assert np.array_equal(info[:, 0], np.minimum((orc.reset_uniform(226, 0, np.arange(E), 0) * 7).astype(int), 6))   # randint(0, 7)
    assert np.array_equal(info[:, 3], (-2.4 + 1.0) + (2.0 * 2.4 - 2.0) * orc.reset_uniform(226, 0, np.arange(E), 2))
    # the oracle, started from the same state, must agree on the first observation and on a rollout
    params = [orc.make_params(n_a, grids[e].shape[1], float(shapes["l_cell"][k[e]]), r_avoid) for e in range(E)]
    ob = orc.OracleBatch(params, nthreads=8, ng_max=ngm)
    for e in range(E):
        ob.set_grid(e, grids[e])
    ob.p[:], ob.dp[:] = p, dp
    ob.observe()
    assert np.array_equal(sim.obs.cpu().numpy(), ob.obs)
    assert np.array_equal(sim.sensed_index.cpu().numpy(), ob.sensed_index)
    rng = np.random.RandomState(0)
    for t in range(25):
        a = goal_seeking_action(ob.obs, ob.dp, rng)
        sim.step(torch.from_numpy(a).cuda()); ob.step(a)
        for name, got, ref in (("p", sim.p, ob.p), ("obs", sim.obs, ob.obs), ("reward", sim.reward, ob.reward),
                               ("a_prior", sim.a_prior, ob.a_prior), ("occupied", sim.occupied_index, ob.occupied_index)):
            assert np.array_equal(got.cpu().numpy(), ref), (name, t)


def test_reset_is_deterministic_per_key_and_maskable():
    E = 64
    sim, shapes, _, _ = make(E)
    sim.reset(seed=5, episode=3)
    p1, g1, o1 = sim.p.clone(), sim._grid.clone(), sim.obs.clone()
    sim.reset(seed=5, episode=4)
    assert not torch.equal(sim.p, p1)
    sim.reset(seed=5, episode=3)
    assert torch.equal(sim.p, p1) and torch.equal(sim._grid, g1) and torch.equal(sim.obs, o1)
    # env_offset shifts the key: envs [32, 64) of an offset-0 batch == envs [0, 32) of an offset-32 batch (sharding)
    sim.reset(seed=5, episode=3, env_offset=32)
    assert torch.equal(sim.p[:32], p1[32:])
    # masked reset: only the selected envs change
    sim.reset(seed=5, episode=3)
    mask = torch.zeros(E, dtype=torch.bool); mask[::4] = True
    sim.reset(seed=5, episode=9, env_mask=mask)
    same = (sim.p == p1).flatten(1).all(1).cpu()
    assert same[~mask].all() and not same[mask].any()


def test_shape_and_spawn_statistics():
    E = 4096
    sim, shapes, _, _ = make(E)
    sim.reset(seed=1)
    info = sim.reset_info.cpu().numpy()
    hist = np.bincount(info[:, 0].astype(int), minlength=7) / E
    assert np.abs(hist - 1 / 7).max() < 0.03                       # randint(0, 7)
    ang = np.arctan2(info[:, 2], info[:, 1])
    assert abs(ang.mean()) < 0.15 and ang.min() < -3.0 and ang.max() > 3.0     # pi * U(-1, 1)
    assert abs(info[:, 5].mean() - 0.5) < 0.05                     # U(-1, 1) > 0
    dp = sim.dp.cpu().numpy()
    assert abs(dp.mean()) < 0.01 and abs(dp.std() - 1 / np.sqrt(12)) < 0.01


def test_set_grid_pose_builds_the_host_grid_bit_for_bit_and_rollout_matches_oracle():
    """swarm_set_grid_pose: the device applies grid = R.origin + off itself (assembly.py:175-187).  The stored cells equal the
    host's separately rounded evaluation bit for bit; the pose is then known exactly (fast_path == 2: cells recomputed from
    the shape library) and a goal-seeking rollout follows the oracle on every output, as does the same batch fed through
    set_grid (pose detected, fast_path == 1) and through the general scan (no shape library)."""
    from marl_llm_b200.batched import BatchedAssemblySim
    E, n_a = 64, 30
    sim, shapes, r_avoid, ngm = make(E, n_a)
    rng = np.random.RandomState(12)
    k = rng.randint(0, 7, E)
    ang = np.pi * rng.uniform(-1, 1, E)
    cs, sn, off = np.cos(ang), np.sin(ang), rng.uniform(-1.4, 1.4, (E, 2))
    grids = [BatchedAssemblySim.grid_from_pose(shapes["grid_origin"][k[e]], cs[e], sn[e], off[e, 0], off[e, 1]) for e in range(E)]
    sim.set_grid_pose(k, cs, sn, off[:, 0], off[:, 1])
    assert sim.fast_path == 2
    dev_grid, n_g = sim._grid.cpu().numpy(), sim._n_g.cpu().numpy()
    for e in range(E):
        assert n_g[e] == grids[e].shape[1] and np.array_equal(dev_grid[e, :n_g[e]].T, grids[e]), e
    detected = BatchedAssemblySim(E, n_a, ngm, r_avoid, out_dtype=torch.float64, emit_indices=True)
    detected.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    general = BatchedAssemblySim(E, n_a, ngm, r_avoid, out_dtype=torch.float64, emit_indices=True)
    blocks, ng = sim.pack_grids(grids, ngm)
    for other in (detected, general):
        other.set_grid(blocks, ng, [float(shapes["l_cell"][k[e]]) for e in range(E)])
    assert detected.fast_path == 1 and general.fast_path == 0
    params = [orc.make_params(n_a, grids[e].shape[1], float(shapes["l_cell"][k[e]]), r_avoid) for e in range(E)]
    ob = orc.OracleBatch(params, nthreads=8, ng_max=ngm)
    for e in range(E):
        ob.set_grid(e, grids[e])
        c = rng.choice(grids[e].shape[1], n_a // 2, replace=False)      # half of each swarm starts on cells: in-shape from the start
        ob.p[e] = rng.uniform(-2.4, 2.4, (2, n_a)); ob.p[e][:, :n_a // 2] = grids[e][:, c] + rng.normal(0, 0.01, (2, n_a // 2))
    ob.dp[:] = rng.uniform(-0.5, 0.5, ob.dp.shape)
    for s_ in (sim, detected, general):
        s_.set_state(ob.p, ob.dp); s_.observe()
    ob.observe(with_reward=True)
    for t in range(60):
        a = goal_seeking_action(ob.obs, ob.dp, rng)
        ob.step(a)
        for s_ in (sim, detected, general):
            s_.step(torch.from_numpy(a).cuda())
            for name, got, ref in (("p", s_.p, ob.p), ("obs", s_.obs, ob.obs), ("reward", s_.reward, ob.reward), ("a_prior", s_.a_prior, ob.a_prior),
                                   ("nbr", s_.neighbor_index, ob.neighbor_index), ("in_flags", s_.in_flags, ob.in_flags),
                                   ("sensed", s_.sensed_index, ob.sensed_index), ("occupied", s_.occupied_index, ob.occupied_index)):
                assert np.array_equal(got.cpu().numpy(), ref), (name, t, s_.fast_path)
    assert ob.in_flags.sum() > 500 and ob.reward.sum() > 0
