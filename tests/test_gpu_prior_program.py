"""Prior programs on the device (swarm_set_prior_program / swarm_prior_program_actions, marl_llm_b200.prior_program).

The shipped program (marl_llm_b200/priors/reference_prior.cu) restates the reference's robotPolicy; installed on a handle it
must give the built-in prior bit for bit, and leave every other output of the step as it was.  A second program that reads the
rest of the view (neighbour velocities, cells, in_thresh, env and agent ids, clamped indices) is compared with a NumPy restatement
in the same operation order.  Every comparison is bit for bit."""
import argparse
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

import bench
from marl_llm_b200 import _lib
from marl_llm_b200._lib import SwarmError
from marl_llm_b200.prior_program import PriorProgram, reference_prior_source
from marl_llm_b200.state_store import StateStore
from oracle import oracle as orc
from tests.helpers import REPO, load_shapes

pytestmark = pytest.mark.gpu

SHAPES = load_shapes()
NGM = int(max(SHAPES["n_g"]))
PATHS = ("exact", "detected", "nolib", "brute")   # device reset / uploaded library grids / no library / brute-force scan
OUT = ("p", "dp", "obs", "reward", "a_prior", "neighbor_index", "in_flags", "sensed_index", "occupied_index")

# reads neighbour velocities, cells within d_sen, in_thresh, in_shape, the env / agent ids and two out-of-range indices
SECOND = r"""#include "swarm_prior_api.cuh"
__device__ void robot_policy(const swarm_agent &a, double out[2]) {
    double sx = 0.0, sy = 0.0;
    for (int q = 0; q < a.count; ++q) {
        const swarm_xy v = a.vel(a.neighbor(q));
        sx += (v.x - a.vx) * (double)(q + 1);
        sy += v.y - a.vy;
    }
    int near = 0;
    for (int k = 0; k < a.n_g(); ++k) {
        const swarm_xy c = a.cell(k);
        const double dx = c.x - a.x, dy = c.y - a.y;
        if (dx * dx + dy * dy < a.d_sen * a.d_sen) near++;
    }
    const swarm_xy far_agent = a.pos(a.n_a + 5), first_cell = a.cell(-3);
    out[0] = sx + (a.in_shape ? 0.5 : -0.5) + (double)near * 1e-3 + (double)a.env * 1e-6 + far_agent.x;
    out[1] = sy * a.in_thresh + (double)a.id * 1e-7 + first_cell.y + (a.nearest == 0 ? 1.0 : 0.0) * a.cell_x;
}
"""


def second_numpy(p, dp, grid, n_g, in_thresh, nbr, d_sen):
    """SECOND restated for every env and agent ([E, 2, n_a] float64), with the nearest cell scanned (first minimum)."""
    E, _, n_a = p.shape
    out = np.zeros((E, 2, n_a))
    for e in range(E):
        g = grid[e, :n_g[e]]
        for i in range(n_a):
            x, y, vx, vy = p[e, 0, i], p[e, 1, i], dp[e, 0, i], dp[e, 1, i]
            sx = sy = 0.0
            ids = [j for j in nbr[e, i] if j >= 0]
            for q, j in enumerate(ids):
                sx = sx + (dp[e, 0, j] - vx) * float(q + 1)
                sy = sy + (dp[e, 1, j] - vy)
            dx, dy = g[:, 0] - x, g[:, 1] - y
            s = dx * dx + dy * dy
            near = int(np.sum(s < d_sen * d_sen))
            bc = int(np.argmin(s))                            # first minimum
            in_shape = s[bc] < in_thresh[e]
            out[e, 0, i] = sx + (0.5 if in_shape else -0.5) + float(near) * 1e-3 + float(e) * 1e-6 + p[e, 0, n_a - 1]
            out[e, 1, i] = sy * in_thresh[e] + float(i) * 1e-7 + g[0, 1] + (1.0 if bc == 0 else 0.0) * g[bc, 0]
    return out


@pytest.fixture(scope="module")
def ref_prog():
    return PriorProgram(reference_prior_source())


@pytest.fixture(scope="module")
def second_prog():
    return PriorProgram(SECOND)


def bits(t):
    return t.view({8: torch.int64, 4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def make_sim(E, n_a, path="exact", parity=False, **kw):
    from marl_llm_b200.batched import BatchedAssemblySim
    sim = BatchedAssemblySim(E, n_a, NGM, orc.r_avoid_for(n_a, SHAPES["n_g"], SHAPES["l_cell"]),
                             out_dtype=torch.float64 if parity else torch.float32, emit_indices=parity,
                             brute_force_scan=path == "brute", **kw)
    if path != "nolib":
        sim.set_shapes(SHAPES["grid_origin"], SHAPES["l_cell"])
    return sim


def start(sim, path, seed=3):
    if path in ("exact", "brute"):
        sim.reset(seed=seed)
    else:
        blocks, n_g, l_cell, p, dp = bench.synth_batch(sim.E, sim.n_a, SHAPES, seed, "random")
        sim.set_grid(blocks, n_g, l_cell)
        sim.set_state(p, dp)
        sim.observe()


def actions(E, n_a, seed, t):
    return torch.from_numpy(orc.fill_actions(E, n_a, seed, t)).cuda()


def outputs(sim, rows=None):
    d = {n: getattr(sim, n) for n in OUT}
    return {k: bits(v if rows is None else v[rows]).clone() for k, v in d.items() if v is not None}


def assert_same(a, b, what):
    for k in a:
        assert torch.equal(a[k], b[k]), (k, what)


def twin_pair(E, n_a, path, parity, prog, seed=3, **kw):
    sim, twin = make_sim(E, n_a, path, parity, **kw), make_sim(E, n_a, path, parity, **kw)
    start(sim, path, seed); start(twin, path, seed)
    sim.set_prior_program(prog)
    return sim, twin


# ---- 1. the shipped program against the built-in prior --------------------------------------------------------------------
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("parity", [False, True], ids=["f32", "f64"])
@pytest.mark.parametrize("n_a", [1, 7, 30, 33, 64, 100, 1024])
def test_shipped_program_equals_the_builtin_prior_over_rollouts(ref_prog, n_a, parity, path):
    E = 4 if n_a < 1024 else 2
    sim, twin = twin_pair(E, n_a, path, parity, ref_prog)
    for t in range(200):
        if path != "nolib" and t in (70, 140):             # staggered auto-resets in the middle of the run
            ids = torch.tensor([1, E - 1] if t == 70 else [0], dtype=torch.int32, device="cuda")
            sim.reset_envs(ids, seed=11, episode=t); twin.reset_envs(ids, seed=11, episode=t)
        a = actions(E, n_a, 5, t)
        sim.step(a); twin.step(a)
        assert_same(outputs(sim), outputs(twin), t)


# ---- 2. the scanned nearest cell --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_a", [30, 100])
def test_scanned_nearest_cell_after_state_and_grid_changes(ref_prog, n_a):
    from marl_llm_b200.batched import BatchedAssemblySim
    E = 6
    sim, twin = twin_pair(E, n_a, "exact", True, ref_prog)
    rng = np.random.RandomState(2)
    for t in range(24):
        kind = t % 4
        if kind == 1:                                      # set_state: the stored nearest cell is stale
            p = sim.p.cpu().numpy() + rng.uniform(-0.05, 0.05, (E, 2, n_a))
            dp = sim.dp.cpu().numpy()
            sim.set_state(p, dp); twin.set_state(p, dp)
        elif kind == 2:                                    # set_grid: another grid under the same agents
            k = rng.randint(0, len(SHAPES["n_g"]), E)
            grids = [BatchedAssemblySim.grid_from_pose(SHAPES["grid_origin"][kk], np.cos(0.3 * t), np.sin(0.3 * t), 0.1, -0.2) for kk in k]
            blocks, n_g = BatchedAssemblySim.pack_grids(grids, NGM)
            sim.set_grid(blocks, n_g, SHAPES["l_cell"][k]); twin.set_grid(blocks, n_g, SHAPES["l_cell"][k])
        elif kind == 3:                                    # set_grid_pose on a subset
            ids = rng.randint(0, len(SHAPES["n_g"]), 3)
            args = (ids, np.cos(0.7 * t), np.sin(0.7 * t), -0.3, 0.25)
            sim.set_grid_pose(*args, env0=2); twin.set_grid_pose(*args, env0=2)
        a = actions(E, n_a, 9, t)
        sim.step(a); twin.step(a)
        assert_same(outputs(sim), outputs(twin), t)


# ---- 3. the program as actions, against the oracle --------------------------------------------------------------------------
def test_program_actions_equal_the_oracle_prior(ref_prog):
    E, n_a = 4, 30
    sim = make_sim(E, n_a, "nolib", True, want_prior=False)
    blocks, n_g, l_cell, p, dp = bench.synth_batch(E, n_a, SHAPES, 8, "random")
    sim.set_grid(blocks, n_g, l_cell); sim.set_state(p, dp); sim.observe()
    r_avoid = orc.r_avoid_for(n_a, SHAPES["n_g"], SHAPES["l_cell"])
    ob = orc.OracleBatch([orc.make_params(n_a, int(n_g[e]), float(l_cell[e]), r_avoid) for e in range(E)], ng_max=NGM)
    for e in range(E):
        ob.set_grid(e, blocks[e, :2 * n_g[e]].reshape(2, n_g[e]))
    ob.p[:], ob.dp[:] = p, dp
    ob.observe()
    for t in range(60):
        got = ref_prog.actions(sim).cpu().numpy()
        a = orc.fill_actions(E, n_a, 4, t)
        ob.step(a)                                       # ob.a_prior: orc_prior of the pre-step state (ENV:613-624)
        assert np.array_equal(got, ob.a_prior), t
        sim.step(torch.from_numpy(a).cuda())
        assert np.array_equal(sim.p.cpu().numpy(), ob.p), t


# ---- 4. a second program against its NumPy restatement ------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["exact", "nolib"])
def test_second_program_equals_its_numpy_restatement(second_prog, path):
    E, n_a = 5, 33
    sim = make_sim(E, n_a, path, True)
    start(sim, path, seed=6)
    sim.set_prior_program(second_prog)
    for t in range(12):
        host = [v.cpu().numpy() for v in (sim.p, sim.dp, sim._grid, sim._n_g, sim._in_thresh, sim.neighbor_index)]
        want = second_numpy(*host, sim.d_sen)
        got_act = second_prog.actions(sim).cpu().numpy()
        assert np.array_equal(got_act, want), t
        sim.step(actions(E, n_a, 3, t))
        assert np.array_equal(sim.a_prior.cpu().numpy(), want), t
    # the built-in prior is different: the library runs the program, not the built-in prior
    twin = make_sim(E, n_a, path, True)
    start(twin, path, seed=6)
    want = second_numpy(*[v.cpu().numpy() for v in (twin.p, twin.dp, twin._grid, twin._n_g, twin._in_thresh, twin.neighbor_index)],
                        twin.d_sen)
    twin.step(actions(E, n_a, 3, 0))
    assert not np.array_equal(twin.a_prior.cpu().numpy(), want)


# ---- 5. install, then remove ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["exact", "nolib"])
def test_removing_a_program_restores_the_builtin_prior(second_prog, path):
    E, n_a = 4, 30
    sim, twin = twin_pair(E, n_a, path, True, second_prog)
    for t in range(8):
        a = actions(E, n_a, 2, t)
        sim.step(a); twin.step(a)
        assert not torch.equal(sim.a_prior, twin.a_prior)
    sim.set_prior_program(None)
    for t in range(8, 20):
        a = actions(E, n_a, 2, t)
        sim.step(a); twin.step(a)
        assert_same(outputs(sim), outputs(twin), t)


# ---- 6. state store in both directions ----------------------------------------------------------------------------------------
def test_state_store_in_both_directions(ref_prog, second_prog):
    E, n_a = 4, 30
    prog_sim, ref = twin_pair(E, n_a, "exact", True, second_prog)
    for t in range(5):
        a = actions(E, n_a, 1, t)
        prog_sim.step(a); ref.step(a)
    envs = list(range(E))
    store = StateStore(prog_sim, E)
    store.save(envs, envs)                                   # saved under a program ...
    builtin = make_sim(E, n_a, "exact", True)
    start(builtin, "exact", seed=99)
    builtin.step(actions(E, n_a, 7, 0))                      # a valid prior of its own state, which the load must not keep
    store.load(envs, envs, sim=builtin)                      # ... continued by the built-in prior
    for t in range(5, 12):
        a = actions(E, n_a, 1, t)
        builtin.step(a); ref.step(a)
        assert_same(outputs(builtin), outputs(ref), t)
    store2 = StateStore(ref, E)
    store2.save(envs, envs)                                  # saved under the built-in prior ...
    with_prog = make_sim(E, n_a, "exact", True)
    start(with_prog, "exact", seed=98)
    with_prog.set_prior_program(ref_prog)
    with_prog.step(actions(E, n_a, 7, 0))
    store2.load(envs, envs, sim=with_prog)                  # ... continued by the shipped program
    for t in range(12, 20):
        a = actions(E, n_a, 1, t)
        with_prog.step(a); ref.step(a)
        assert_same(outputs(with_prog), outputs(ref), t)


# ---- 7. launch counts and guard zones -------------------------------------------------------------------------------------------
def test_one_extra_launch_per_step_and_nothing_written_outside(ref_prog):
    E, n_a = 4, 30
    sim, twin = twin_pair(E, n_a, "exact", False, ref_prog, guard_bytes=4096)
    a = actions(E, n_a, 1, 0)
    sim.step(a); twin.step(a)
    c0, d0 = sim.launch_count, twin.launch_count
    for t in range(1, 6):
        a = actions(E, n_a, 1, t)
        sim.step(a); twin.step(a)
    per_prog, per_builtin = (sim.launch_count - c0) / 5, (twin.launch_count - d0) / 5
    assert per_prog == per_builtin + 1, (per_prog, per_builtin)
    sim.set_prior_program(None)
    c1 = sim.launch_count
    sim.step(a)                                              # the first step after removal recomputes the prior with k_prior
    c2 = sim.launch_count
    sim.step(a)
    assert c2 - c1 == per_builtin + 1 and sim.launch_count - c2 == per_builtin
    assert sim.check_guards()
    g = 4096
    raw = torch.full((g + E * 2 * n_a * 8 + g,), 0xA5, dtype=torch.uint8, device="cuda")
    out = raw[g:g + E * 2 * n_a * 8].view(torch.float64).view(E, 2, n_a)
    c3 = sim.launch_count
    ref_prog.actions(sim, out=out)
    assert sim.launch_count == c3 + 1
    assert bool((raw[:g] == 0xA5).all()) and bool((raw[-g:] == 0xA5).all())
    assert torch.isfinite(out).all()


# ---- 8. errors ------------------------------------------------------------------------------------------------------------------
def test_errors_leave_the_handle_unchanged(ref_prog):
    from marl_llm_b200.flocking import BatchedFlockingSim
    lib = _lib.load()
    E, n_a = 3, 30
    sim, twin = twin_pair(E, n_a, "exact", True, ref_prog)
    sim.set_prior_program(None); twin.step(actions(E, n_a, 1, 0)); sim.step(actions(E, n_a, 1, 0))
    no_prior = make_sim(E, n_a, "exact", True, want_prior=False)
    no_prior.reset(seed=3)
    assert lib.swarm_set_prior_program(no_prior._h, ref_prog.handle) == _lib.SWARM_ERR_INVALID
    assert b"want_prior" in lib.swarm_last_error()
    out = torch.empty(E, 2, n_a, dtype=torch.float64, device="cuda")
    ref_prog.actions(no_prior, out=out)                     # the program as actions stays legal there
    flock = BatchedFlockingSim(2, 20)
    assert lib.swarm_set_prior_program(flock._h, ref_prog.handle) == _lib.SWARM_ERR_UNSUPPORTED
    assert lib.swarm_prior_program_actions(flock._h, ref_prog.handle, C.c_void_p(out.data_ptr()), None) == _lib.SWARM_ERR_UNSUPPORTED
    assert lib.swarm_set_prior_program(None, ref_prog.handle) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_prior_program_actions(sim._h, None, C.c_void_p(out.data_ptr()), None) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_prior_program_actions(sim._h, ref_prog.handle, None, None) == _lib.SWARM_ERR_INVALID
    with pytest.raises(SwarmError):
        PriorProgram("this is not C++")
    fresh = make_sim(E, n_a, "exact", True)                 # never observed: no neighbour list yet
    assert lib.swarm_prior_program_actions(fresh._h, ref_prog.handle, C.c_void_p(out.data_ptr()), None) == _lib.SWARM_ERR_INVALID
    if torch.cuda.device_count() > 1:
        other = PriorProgram(reference_prior_source(), device=1)
        assert lib.swarm_set_prior_program(sim._h, other.handle) == _lib.SWARM_ERR_INVALID
    # after every rejected call: the handle still runs the built-in prior, like its twin
    for t in range(1, 6):
        a = actions(E, n_a, 1, t)
        sim.step(a); twin.step(a)
        assert_same(outputs(sim), outputs(twin), t)


# ---- 9. the drop-in env -------------------------------------------------------------------------------------------------------------
def test_dropin_env_takes_its_prior_from_the_program_and_keeps_it_across_a_regrow(second_prog):
    sys.path.insert(0, os.path.join(REPO, "marl_llm_b200", "compat"))
    try:
        from marl_llm_b200.assembly_env import AssemblySwarmEnv
        blob = {"l_cell": [float(v) for v in SHAPES["l_cell"]], "grid_coords": [np.ascontiguousarray(g.T) for g in SHAPES["grid_origin"]],
                "binary_image": [np.zeros((1, 1)) for _ in SHAPES["l_cell"]], "shape_bound_points": [np.zeros(4) for _ in SHAPES["l_cell"]]}
        order = np.argsort(SHAPES["n_g"])
        small = [int(k) for k in order[:3]]
        blob = {key: [val[k] for k in small] for key, val in blob.items()}
        args = argparse.Namespace(n_a=30, is_boundary=True, is_con_self_state=True, is_feature_norm=False, dynamics_mode="Cartesian",
                                  render_traj=False, traj_len=15, agent_strategy="input", training_method="llm_rl", is_collected=False,
                                  results_file=blob, video=False)
        env = AssemblySwarmEnv()
        env.__reinit__(args)
        env.set_prior_program(second_prog)
        np.random.seed(4)
        env.reset()
        cap0 = env._n_g_cap
        rng = np.random.RandomState(1)
        for t in range(8):
            if t == 4:                                        # a shape larger than the handle: the env rebuilds it
                k = int(order[-1])
                env.l_cell = float(SHAPES["l_cell"][k])
                env.grid_center_origin = SHAPES["grid_origin"][k]
                env.n_g = SHAPES["grid_origin"][k].shape[1]
                env.grid_center = SHAPES["grid_origin"][k].copy() + np.array([[0.3], [-0.2]])
            env.step(rng.uniform(-1, 1, (2, 30)).astype(np.float32))
            sim = env._sim
            assert sim.prior_program is second_prog, t
            # the program's actions on the post-step state equal what the next step returns as its prior
            nxt = second_prog.actions(sim).cpu().numpy()[0]
            _, _, _, _, prior2 = env.step(np.zeros((2, 30), np.float32))
            assert np.array_equal(prior2, nxt), t
        assert env._n_g_cap > cap0
        env.set_prior_program(None)
        assert env._sim.prior_program is None
    finally:
        sys.path.remove(os.path.join(REPO, "marl_llm_b200", "compat"))


# ---- 10. full size ---------------------------------------------------------------------------------------------------------------
def test_full_size_batch(ref_prog):
    E, n_a = 65536, 30
    sim, twin = twin_pair(E, n_a, "exact", False, ref_prog, seed=17)
    rows = torch.from_numpy(np.random.RandomState(0).choice(E, 128, replace=False)).cuda()
    act = torch.empty(E, 2, n_a, dtype=torch.float32, device="cuda")
    for t in range(20):
        sim.fill_actions(act, seed=3, step=t)
        sim.step(act); twin.step(act)
        assert_same(outputs(sim, rows), outputs(twin, rows), t)
