"""Prior populations on the device (swarm_prior_population_*, swarm_set_prior_population, marl_llm_b200.prior_program
PriorPopulation / evaluate_priors): K programs in one batch, each on its own envs.

The yardstick is a twin handle per program, in the same state, with that program alone installed: env e of the population
handle must give, bit for bit, what env e of program k's twin gives, for the k assigned to e.  Envs never interact, so every
other output must equal a twin without any program.  Output buffers are filled with NaN before each call, so a skipped env or
agent cannot pass."""
import ctypes as C

import numpy as np
import pytest
import torch

from marl_llm_b200 import _lib
from marl_llm_b200.prior_program import PriorPopulation, PriorProgram, evaluate_priors, reference_prior_source
from marl_llm_b200.state_store import StateStore
from tests.test_gpu_prior_program import SECOND, actions, assert_same, bits, make_sim, outputs, start

pytestmark = pytest.mark.gpu

# the nearest cell's offset, the neighbour count and the velocity: differs from the other programs in every env and agent
THIRD = r"""#include "swarm_prior_api.cuh"
__device__ void robot_policy(const swarm_agent &a, double out[2]) {
    out[0] = (a.cell_x - a.x) * 0.75 - a.vx * 0.25 + (double)a.count * 1e-3;
    out[1] = (a.cell_y - a.y) * 0.75 - a.vy * 0.25 + (a.in_shape ? 0.125 : -0.125);
}
"""
# program k writes (k * 2048 + agent id, env id): which program wrote a row, and for which env and agent, can be read off it
TAG = r"""#include "swarm_prior_api.cuh"
__device__ void robot_policy(const swarm_agent &a, double out[2]) {
    out[0] = (double)(%d * 2048 + a.id);
    out[1] = (double)a.env;
}
"""


@pytest.fixture(scope="module")
def progs():
    return [PriorProgram(reference_prior_source()), PriorProgram(SECOND), PriorProgram(THIRD)]


@pytest.fixture(scope="module")
def tags():
    return [PriorProgram(TAG % k) for k in range(16)]


def spread(E, K, seed):
    """a random assignment env -> program in which every program has at least one env (E >= K)"""
    return np.random.RandomState(seed).permutation(np.arange(E) % K).astype(np.int32)


def nan_prior(sim):
    for b in sim._a_prior:
        b.fill_(float("nan"))


def nan_like(sim):
    return torch.full((sim.E, 2, sim.n_a), float("nan"), dtype=torch.float64, device="cuda")


def rows(assign, k):
    return torch.from_numpy(np.flatnonzero(assign == k)).cuda()


# ---- 1. prior mode against one twin per program -----------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["exact", "nolib"])
@pytest.mark.parametrize("parity", [False, True], ids=["f32", "f64"])
@pytest.mark.parametrize("n_a", [1, 30, 33, 100, 1024])
def test_population_prior_equals_each_programs_twin_over_rollouts(progs, n_a, parity, path):
    E = 8 if n_a < 1024 else 4
    assign = spread(E, len(progs), n_a)
    sim, plain = make_sim(E, n_a, path, parity), make_sim(E, n_a, path, parity)
    twins = [make_sim(E, n_a, path, parity) for _ in progs]
    for h in [sim, plain] + twins:
        start(h, path)
    sim.set_prior_population(PriorPopulation(progs, assign))
    for tw, p in zip(twins, progs):
        tw.set_prior_program(p)
    groups = [rows(assign, k) for k in range(len(progs))]
    for t in range(200):
        if path != "nolib" and t in (70, 140):             # staggered auto-resets in the middle of the run
            ids = torch.tensor([1, E - 1] if t == 70 else [0], dtype=torch.int32, device="cuda")
            for h in [sim, plain] + twins:
                h.reset_envs(ids, seed=11, episode=t)
        a = actions(E, n_a, 5, t)
        nan_prior(sim)
        for h in [sim, plain] + twins:
            h.step(a)
        for k, g in enumerate(groups):
            assert torch.equal(bits(sim.a_prior[g]), bits(twins[k].a_prior[g])), (t, k)
        got, want = outputs(sim), outputs(plain)
        del got["a_prior"], want["a_prior"]
        assert_same(got, want, t)


# ---- 2. tag programs: each (env, agent) holds its own program's tag ----------------------------------------------------------------
def check_tags(tags, E, n_a, assign):
    K = int(assign.max()) + 1
    sim = make_sim(E, n_a, "exact", False)
    start(sim, "exact")
    pop = PriorPopulation(tags[:K], assign)
    want = torch.empty(E, 2, n_a, dtype=torch.float64)
    want[:, 0, :] = torch.from_numpy(assign.astype(np.float64))[:, None] * 2048 + torch.arange(n_a, dtype=torch.float64)[None, :]
    want[:, 1, :] = torch.arange(E, dtype=torch.float64)[:, None]
    out = nan_like(sim)
    pop.actions(sim, out=out)
    assert torch.equal(out.cpu(), want)
    sim.set_prior_population(pop)
    for t in range(2):
        nan_prior(sim)
        sim.step(sim.fill_actions(torch.empty(E, 2, n_a, device="cuda"), seed=1, step=t))
        assert torch.equal(sim.a_prior.cpu().double(), want), t
        out = nan_like(sim)
        pop.actions(sim, out=out)
        assert torch.equal(out.cpu(), want), t


def test_sixteen_tag_programs_on_65536_envs(tags):
    E = 65536
    check_tags(tags, E, 30, np.random.RandomState(7).randint(0, 16, E).astype(np.int32))


@pytest.mark.parametrize("layout", ["one_env_each", "blocks", "empty_program", "single"])
def test_tag_programs_on_other_assignments(tags, layout):
    E = {"one_env_each": 16, "blocks": 40, "empty_program": 24, "single": 12}[layout]
    if layout == "one_env_each":
        assign = np.random.RandomState(1).permutation(16).astype(np.int32)
    elif layout == "blocks":
        assign = np.repeat(np.arange(5), 8).astype(np.int32)
    elif layout == "empty_program":
        assign = (np.arange(E) % 3).astype(np.int32)
        assign[assign == 1] = 3                               # program 1 of 4 has no envs
    else:
        assign = np.zeros(E, np.int32)
    check_tags(tags, E, 33, assign)


# ---- 3. a population of one is set_prior_program -----------------------------------------------------------------------------------
def test_population_of_one_equals_set_prior_program(progs):
    E, n_a = 6, 30
    sim, twin = make_sim(E, n_a, "exact", True), make_sim(E, n_a, "exact", True)
    start(sim, "exact"); start(twin, "exact")
    sim.set_prior_population(PriorPopulation([progs[1]], np.zeros(E, np.int32)))
    twin.set_prior_program(progs[1])
    c0, d0 = sim.launch_count, twin.launch_count
    for t in range(40):
        a = actions(E, n_a, 2, t)
        sim.step(a); twin.step(a)
        assert_same(outputs(sim), outputs(twin), t)
    assert sim.launch_count - c0 == twin.launch_count - d0


# ---- 4. actions -----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["exact", "nolib"])
def test_population_actions_equal_each_programs_actions(progs, path):
    E, n_a = 9, 33
    assign = spread(E, 3, 4)
    sim = make_sim(E, n_a, path, True, want_prior=False)      # actions need no want_prior
    start(sim, path)
    pop = PriorPopulation(progs, assign)
    for t in range(6):
        got = pop.actions(sim, out=nan_like(sim))
        for k, p in enumerate(progs):
            g = rows(assign, k)
            assert torch.equal(got[g], p.actions(sim, out=nan_like(sim))[g]), (t, k)
        sim.step(got)


# ---- 5. evaluate_priors ------------------------------------------------------------------------------------------------------------------
def test_evaluate_priors_equals_the_reduction_over_single_program_twins(progs):
    E, n_a, steps, seed = 12, 30, 30, 21
    assign = spread(E, 3, 5)
    sim = make_sim(E, n_a, "exact", False)
    got = evaluate_priors(sim, PriorPopulation(progs, assign), steps, seed)
    assert set(got) == {"reward", "coverage_rate", "distribution_uniformity", "voronoi_based_uniformity"}
    for k, p in enumerate(progs):
        tw = make_sim(E, n_a, "exact", False)
        tw.reset(seed)
        reward = torch.zeros(E, dtype=torch.float64, device="cuda")
        for _ in range(steps):
            _, rew, _, _, _ = tw.step(p.actions(tw))
            reward += rew.reshape(E, n_a).to(torch.float64).sum(1)
        g = rows(assign, k)
        met = tw.metrics()
        assert torch.equal(got["reward"][k], reward[g].sum() / (g.numel() * steps * n_a)), k
        for j, name in enumerate(("coverage_rate", "distribution_uniformity", "voronoi_based_uniformity")):
            assert torch.equal(got[name][k], met[g, j].sum() / g.numel()), (k, name)
    assert torch.isfinite(got["reward"]).all()


# ---- 6. switching -------------------------------------------------------------------------------------------------------------------------
def test_switching_between_population_program_and_builtin(progs):
    E, n_a = 8, 30
    assign = spread(E, 3, 6)
    pop = PriorPopulation(progs, assign)
    sim, pop_tw, prog_tw, plain = (make_sim(E, n_a, "exact", True) for _ in range(4))
    for h in (sim, pop_tw, prog_tw, plain):
        start(h, "exact")
    pop_tw.set_prior_population(pop)
    prog_tw.set_prior_program(progs[2])
    t = 0

    def step_all(twin, n=3):
        nonlocal t
        for _ in range(n):
            a = actions(E, n_a, 8, t)
            for h in (sim, pop_tw, prog_tw, plain):
                h.step(a)
            assert_same(outputs(sim), outputs(twin), t)
            t += 1

    sim.set_prior_population(pop)
    step_all(pop_tw)
    sim.set_prior_program(progs[2])
    assert sim.prior_population is None
    step_all(prog_tw)
    sim.set_prior_population(pop)
    step_all(pop_tw)
    sim.set_prior_population(None)                          # the built-in prior again, through k_prior
    assert sim.prior_population is None and sim.prior_program is None
    c0, d0 = sim.launch_count, plain.launch_count
    step_all(plain, 1)
    assert sim.launch_count - c0 == plain.launch_count - d0 + 1
    step_all(plain, 2)
    sim.set_prior_population(pop)
    step_all(pop_tw)


# ---- 7. state store ----------------------------------------------------------------------------------------------------------------------------
def test_state_store_under_a_population(progs):
    E, n_a = 6, 30
    assign = spread(E, 3, 7)
    pop = PriorPopulation(progs, assign)
    sim, plain, pop_tw = (make_sim(E, n_a, "exact", True) for _ in range(3))
    for h in (sim, plain, pop_tw):
        start(h, "exact")
    sim.set_prior_population(pop)
    pop_tw.set_prior_population(pop)
    for t in range(5):
        a = actions(E, n_a, 1, t)
        for h in (sim, plain, pop_tw):
            h.step(a)
    envs = list(range(E))
    store = StateStore(sim, E)
    store.save(envs, envs)                                  # saved under the population ...
    builtin = make_sim(E, n_a, "exact", True)
    start(builtin, "exact", seed=99)
    builtin.step(actions(E, n_a, 7, 0))                     # a valid prior of its own state, which the load must not keep
    store.load(envs, envs, sim=builtin)                     # ... continued by the built-in prior
    other = make_sim(E, n_a, "exact", True)
    start(other, "exact", seed=98)
    other.set_prior_population(pop)
    other.step(actions(E, n_a, 7, 0))
    store.load(envs, envs, sim=other)                       # ... and by the population
    for t in range(5, 12):
        a = actions(E, n_a, 1, t)
        for h in (builtin, plain, other, pop_tw):
            h.step(a)
        assert_same(outputs(builtin), outputs(plain), t)
        assert_same(outputs(other), outputs(pop_tw), t)


# ---- 8. launch counts and guard zones ------------------------------------------------------------------------------------------------------------
def test_one_launch_per_program_with_envs_and_nothing_written_outside(progs):
    E, n_a = 8, 30
    assign = np.array([0, 3, 0, 1, 3, 3, 1, 0], np.int32)  # program 2 of 4 has no envs
    pop = PriorPopulation(progs + [progs[0]], assign)
    sim, twin = make_sim(E, n_a, "exact", False, guard_bytes=4096), make_sim(E, n_a, "exact", False)
    start(sim, "exact"); start(twin, "exact")
    sim.set_prior_population(pop)
    a = actions(E, n_a, 1, 0)
    sim.step(a); twin.step(a)
    c0, d0 = sim.launch_count, twin.launch_count
    for t in range(1, 6):
        a = actions(E, n_a, 1, t)
        sim.step(a); twin.step(a)
    assert sim.launch_count - c0 == (twin.launch_count - d0) + 5 * 3
    assert sim.check_guards()
    g = 4096
    raw = torch.full((g + E * 2 * n_a * 8 + g,), 0xA5, dtype=torch.uint8, device="cuda")
    out = raw[g:g + E * 2 * n_a * 8].view(torch.float64).view(E, 2, n_a)
    out.fill_(float("nan"))
    c1 = sim.launch_count
    pop.actions(sim, out=out)
    assert sim.launch_count == c1 + 3
    assert bool((raw[:g] == 0xA5).all()) and bool((raw[-g:] == 0xA5).all())
    assert torch.isfinite(out).all()


# ---- 9. errors --------------------------------------------------------------------------------------------------------------------------------------
def raw_create(lib, device, E, progs, assign):
    handles = (C.c_void_p * max(len(progs), 1))(*[p.handle.value if p is not None else None for p in progs])
    a = np.ascontiguousarray(assign, dtype=np.int32)
    h = C.c_void_p()
    rc = lib.swarm_prior_population_create(device, E, len(progs), handles, C.c_void_p(a.ctypes.data), C.byref(h))
    return rc, h


def test_errors_return_their_code_and_leave_the_installed_prior(progs):
    from marl_llm_b200.flocking import BatchedFlockingSim
    lib = _lib.load()
    E, n_a = 4, 30
    assign = np.array([0, 1, 2, 1], np.int32)
    for args in ((0, E, [], assign), (0, E, [progs[0], None], assign % 2), (0, 0, progs, assign), (0, E, progs, [0, 1, 3, 1]),
                 (0, E, progs, [0, -1, 2, 1])):
        rc, h = raw_create(lib, *args)
        assert rc == _lib.SWARM_ERR_INVALID and h.value is None, args
    if torch.cuda.device_count() > 1:
        other = PriorProgram(reference_prior_source(), device=1)
        assert raw_create(lib, 0, E, [progs[0], other], assign % 2)[0] == _lib.SWARM_ERR_INVALID
    pop = PriorPopulation(progs, assign)
    pop8 = PriorPopulation(progs, np.arange(8) % 3)
    out = torch.empty(E, 2, n_a, dtype=torch.float64, device="cuda")
    no_prior = make_sim(E, n_a, "exact", True, want_prior=False)
    no_prior.reset(seed=3)
    assert lib.swarm_set_prior_population(no_prior._h, pop.handle) == _lib.SWARM_ERR_INVALID
    assert b"want_prior" in lib.swarm_last_error()
    pop.actions(no_prior, out=out)                          # actions stay legal there
    flock = BatchedFlockingSim(2, 20)
    assert lib.swarm_set_prior_population(flock._h, pop.handle) == _lib.SWARM_ERR_UNSUPPORTED
    assert lib.swarm_set_prior_population(None, pop.handle) == _lib.SWARM_ERR_INVALID
    fresh = make_sim(E, n_a, "exact", True)                  # never observed
    assert lib.swarm_prior_population_actions(fresh._h, pop.handle, C.c_void_p(out.data_ptr()), None) == _lib.SWARM_ERR_INVALID
    for installed in ("builtin", "program", "population"):
        sim, twin = make_sim(E, n_a, "exact", True), make_sim(E, n_a, "exact", True)
        start(sim, "exact"); start(twin, "exact")
        for h in (sim, twin):
            if installed == "program":
                h.set_prior_program(progs[1])
            elif installed == "population":
                h.set_prior_population(pop)
        sim.step(actions(E, n_a, 1, 0)); twin.step(actions(E, n_a, 1, 0))
        assert lib.swarm_set_prior_population(sim._h, pop8.handle) == _lib.SWARM_ERR_INVALID      # made for 8 envs
        assert b"number of envs" in lib.swarm_last_error()
        assert lib.swarm_prior_population_actions(sim._h, pop8.handle, C.c_void_p(out.data_ptr()), None) == _lib.SWARM_ERR_INVALID
        assert lib.swarm_prior_population_actions(sim._h, None, C.c_void_p(out.data_ptr()), None) == _lib.SWARM_ERR_INVALID
        assert lib.swarm_prior_population_actions(sim._h, pop.handle, None, None) == _lib.SWARM_ERR_INVALID
        for t in range(1, 5):
            a = actions(E, n_a, 1, t)
            sim.step(a); twin.step(a)
            assert_same(outputs(sim), outputs(twin), (installed, t))
