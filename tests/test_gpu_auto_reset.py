"""Auto-reset against the oracle: reset_envs (the partial reset bench.py's random regime runs inside its timed region) and the
masked reset, on every scan path.

swarm_reset_envs runs k_reset over an env LIST, then observes only those envs (k_step maps CTA b to env_list[b]); that observe
writes the reset state's prior into the a_prior buffer the next step returns.  A reset also decides which second-half kernel
the next observe / step runs (sim.fast_path), from the host's record of which envs hold a shape with a lookup table.  Every
test here compares bit for bit: with the C oracle rebuilt from the draws (reset_info), or with a twin simulator."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from marl_llm_b200._lib import SwarmError
from oracle import oracle as orc
from tests.helpers import REPO, goal_seeking_action, load_shapes, oracle_follow_reset

pytestmark = pytest.mark.gpu

ALL = ("p", "dp", "obs", "reward", "a_prior", "neighbor_index", "in_flags", "sensed_index", "occupied_index")
AFTER_RESET = ("p", "dp", "obs", "neighbor_index", "in_flags", "sensed_index", "occupied_index")   # a reset returns no reward
FAST_PATH = {"exact": 2, "detected": 1, "culled": 0, "brute": 0}


def make_sim(E, n_a, layout="parity", shapes=None, **kw):
    from marl_llm_b200.batched import BatchedAssemblySim
    shapes = shapes or load_shapes()
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    parity = layout == "parity"
    sim = BatchedAssemblySim(E, n_a, int(max(shapes["n_g"])), r_avoid, out_dtype=torch.float64 if parity else torch.float32,
                             emit_indices=parity, **kw)
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    return sim


def make_oracle(sim, shapes, n_envs, **kw):
    """An oracle batch of n_envs envs with the simulator's constants; grids / states are filled in by the caller."""
    ngm = int(max(shapes["n_g"]))
    P = orc.make_params(sim.n_a, ngm, float(shapes["l_cell"][0]), sim.r_avoid, **kw)
    return orc.OracleBatch([P] * n_envs, nthreads=8, ng_max=ngm)


def assert_matches(sim, ob, fields, what, rows=None, pick=None):
    """Simulator env pick[k] equals oracle env k, for every k in rows (default: all), bit for bit."""
    cast = np.float64 if sim.out_dtype == torch.float64 else np.float32
    rows = np.arange(ob.E) if rows is None else np.asarray(rows)
    envs = rows if pick is None else np.asarray(pick)[rows]
    te = torch.as_tensor(envs, device=sim.device)
    for name in fields:
        got = getattr(sim, name)
        if got is None:                  # production layout: no sensed / occupied index arrays
            continue
        ref = getattr(ob, name)[rows]
        if name in ("obs", "reward", "a_prior"):
            ref = ref.astype(cast)
        assert np.array_equal(got[te].cpu().numpy(), ref), (name, what)


def bits(t):
    return t.view({8: torch.int64, 4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def all_buffers(sim):
    """Every device buffer (bit patterns); the two a_prior buffers as the one the last step returned and the one the next returns."""
    d = dict(p=sim.p, dp=sim.dp, grid=sim._grid, n_g=sim._n_g, in_thresh=sim._in_thresh, word_box=sim._word_box, frame=sim._frame,
             nearest_cell=sim.nearest_cell, reset_info=sim.reset_info, obs=sim.obs, reward=sim.reward, a_prior_last=sim.a_prior,
             a_prior_next=pending_prior(sim), neighbor_index=sim.neighbor_index, in_flags=sim.in_flags, sensed_index=sim.sensed_index,
             occupied_index=sim.occupied_index)
    return {k: bits(v) for k, v in d.items() if v is not None}


def pending_prior(sim):
    """The a_prior buffer the next step returns (the one the last step did not)."""
    return sim._a_prior[1] if sim.a_prior.data_ptr() == sim._a_prior[0].data_ptr() else sim._a_prior[0]


# ------------------------------------------------------------------------------------------------------------------
# 1. reset_envs == the full reset, restricted to the listed envs
LISTED = ("p", "dp", "grid", "n_g", "in_thresh", "word_box", "frame", "nearest_cell", "reset_info", "obs", "neighbor_index",
          "in_flags", "sensed_index", "occupied_index")


@pytest.mark.parametrize("layout", ["parity", "production"])
@pytest.mark.parametrize("n_a", [7, 30, 64, 100])
def test_reset_envs_is_the_full_reset_restricted_to_the_listed_envs(n_a, layout):
    E, OFF = 40, 24
    A, B, C, C_off = (make_sim(E, n_a, layout) for _ in range(4))
    C.reset(seed=9, episode=4)
    C_off.reset(seed=9, episode=4, env_offset=OFF)
    # env_offset shifts the key: env e of an offset batch is env OFF + e of a larger batch without offset (sharding)
    C_big = make_sim(OFF + E, n_a, layout)
    C_big.reset(seed=9, episode=4)
    shifted, off_bufs = torch.arange(OFF, OFF + E, device="cuda"), all_buffers(C_off)
    for name, b in all_buffers(C_big).items():
        if name in LISTED:
            assert torch.equal(off_bufs[name], b[shifted]), name
    act = torch.empty(E, 2, n_a, dtype=torch.float32, device="cuda")

    def prepare(s):                      # the same full reset and a few steps for A and B
        s.reset(seed=1, episode=0)
        for t in range(3):
            s.step(s.fill_actions(act, seed=5, step=t))
    prepare(B)
    ref_b = {k: v.clone() for k, v in all_buffers(B).items()}
    lists = {"unsorted": ([17, 3, 29, 8, 0, 22], 0), "single": ([5], 0), "last": ([E - 1], 0),
             "all": (list(np.random.RandomState(0).permutation(E)), 0), "offset": ([2, 11, 37, 20], OFF)}
    for case, (ids, off) in lists.items():
        prepare(A)
        assert torch.equal(bits(A.p), ref_b["p"]) and torch.equal(bits(A.obs), ref_b["obs"]), case
        A.reset_envs(torch.tensor(ids, dtype=torch.int32, device="cuda"), seed=9, episode=4, env_offset=off)
        assert A.fast_path == C.fast_path == 2, case
        got, want = all_buffers(A), all_buffers(C_off if off else C)
        listed = torch.tensor(sorted(ids), device="cuda")
        unlisted = torch.tensor(sorted(set(range(E)) - set(ids)), dtype=torch.int64, device="cuda")
        for name in LISTED:
            if name in got:
                assert torch.equal(got[name][listed], want[name][listed]), (case, name)
        for name, b in ref_b.items():
            assert torch.equal(got[name][unlisted], b[unlisted]), (case, name)


# ------------------------------------------------------------------------------------------------------------------
# 2. / 3. bench's stationary auto-reset schedule at small scale, every env against the oracle at every step
def start(path, E, n_a, shapes, monkeypatch, **kw):
    """Simulator and oracle in the same first state, with the second-half kernel of scan path `path` active."""
    if path == "culled":
        monkeypatch.setenv("SWARM_NO_LOOKUP_SCAN", "1")           # read by set_shapes: the library is kept, the tables are not
    sim = make_sim(E, n_a, shapes=shapes, brute_force_scan=path == "brute", is_con_self_state=kw.get("is_con_self_state", True),
                   want_prior=kw.get("want_prior", True))
    monkeypatch.delenv("SWARM_NO_LOOKUP_SCAN", raising=False)
    for b in sim._a_prior:
        b.fill_(-123.0)
    ob = make_oracle(sim, shapes, E, **kw)
    # grids from set_grid: poses recognised, not known.  The other paths reset from there, so the word boxes / frames of the
    # culled scan are those of other grids unless the reset rebuilds them
    blocks, n_g, l_cell, p, dp = bench.synth_batch(E, n_a, shapes, 11, "random")
    sim.set_grid(blocks, n_g, l_cell)
    if path == "detected":
        sim.set_state(p, dp); sim.observe()
        for e in range(E):
            ob.params[e].n_g, ob.params[e].l_cell = int(n_g[e]), float(l_cell[e])
            ob.set_grid(e, blocks[e, :2 * n_g[e]].reshape(2, n_g[e]))
        ob.p[:], ob.dp[:] = p, dp
        ob.observe()
    else:
        sim.reset(seed=3, episode=0)
        oracle_follow_reset(ob, sim, shapes, np.arange(E))
    assert sim.fast_path == FAST_PATH[path]
    assert_matches(sim, ob, AFTER_RESET, "first observation")
    return sim, ob


def run_schedule(sim, ob, shapes, how, steps=120, C=8, EP=40, target_row=28):
    """Cohort e % C is reset (reset_envs, or reset with a mask) after step t when t = (EP / C) * cohort (mod EP), episode 1 + t;
    half of the envs seek their shape.  Compared with the oracle after every step and every reset; the envs a reset leaves
    alone keep every output, and the prior their next step returns."""
    E, stride = sim.E, EP // C
    want_prior = sim.want_prior
    fields = ALL if want_prior else tuple(f for f in ALL if f != "a_prior")
    rng = np.random.RandomState(17)
    goal = np.arange(E) % 2 == 0
    untouched = None
    for t in range(steps):
        a = orc.fill_actions(E, sim.n_a, 31, t)
        a[goal] = goal_seeking_action(ob.obs[goal], ob.dp[goal], rng, target_row=target_row)
        sim.step(torch.from_numpy(a).cuda()); ob.step(a)
        assert_matches(sim, ob, fields, ("step", t))
        if untouched is not None and want_prior:                  # the step after a reset returns the prior kept for them
            keep, prior = untouched
            assert torch.equal(bits(sim.a_prior[keep]), prior), ("prior of untouched envs", t)
        untouched = None
        if t % stride:
            continue
        due = np.arange((t % EP) // stride, E, C)
        keep = torch.as_tensor(np.setdiff1d(np.arange(E), due), device=sim.device)
        before = {n: bits(getattr(sim, n)[keep]) for n in ALL if n != "a_prior" and getattr(sim, n) is not None}
        untouched = (keep, bits(pending_prior(sim)[keep]))
        if how == "list":
            sim.reset_envs(torch.as_tensor(due, dtype=torch.int32, device=sim.device), seed=226, episode=1 + t)
        else:
            mask = torch.zeros(E, dtype=torch.bool)
            mask[due] = True
            sim.reset(seed=226, episode=1 + t, env_mask=mask)
        for n, b in before.items():
            assert torch.equal(bits(getattr(sim, n)[keep]), b), (n, "changed by the reset of other envs", t)
        oracle_follow_reset(ob, sim, shapes, due)
        assert_matches(sim, ob, AFTER_RESET, ("reset", t), rows=due)
    if not want_prior:
        for b in sim._a_prior:
            assert bool((b == -123.0).all())
    assert ob.in_flags.sum() > 0 and ob.reward.sum() > 0


@pytest.mark.parametrize("path,n_a,kw", [(p, n, {}) for n in (30, 100) for p in FAST_PATH] +
                         [("exact", 30, dict(is_con_self_state=False)), ("exact", 30, dict(want_prior=False))])
def test_auto_reset_follows_the_oracle_at_every_step(path, n_a, kw, monkeypatch):
    shapes = load_shapes()
    sim, ob = start(path, 512, n_a, shapes, monkeypatch, **kw)
    run_schedule(sim, ob, shapes, "list", target_row=28 if kw.get("is_con_self_state", True) else 24)
    assert sim.fast_path == FAST_PATH[path]


@pytest.mark.parametrize("path,n_a", [(p, 30) for p in FAST_PATH] + [("exact", 100)])
def test_masked_reset_follows_the_oracle_at_every_step(path, n_a, monkeypatch):
    shapes = load_shapes()
    sim, ob = start(path, 512, n_a, shapes, monkeypatch)
    run_schedule(sim, ob, shapes, "mask")
    assert sim.fast_path == FAST_PATH[path]


# ------------------------------------------------------------------------------------------------------------------
# 4. a library in which some shapes have no lookup table
def mixed_library():
    """The 7 reference shapes, one of them rotated by 0.5 rad (a lattice, but not an axis-aligned one) and another jittered by
    1e-3: the last two get no lookup table, their envs need the general scan."""
    shapes = load_shapes()
    c, s = np.cos(0.5), np.sin(0.5)
    g0, g1 = shapes["grid_origin"][0], shapes["grid_origin"][1]
    rotated = np.ascontiguousarray(np.array([[c, -s], [s, c]]) @ g0)
    jittered = g1 + np.random.RandomState(5).normal(0, 1e-3, g1.shape)
    return dict(l_cell=np.append(shapes["l_cell"], shapes["l_cell"][:2]), n_g=np.append(shapes["n_g"], shapes["n_g"][:2]),
                grid_origin=shapes["grid_origin"] + [rotated, jittered])


def drawn_shapes(seed, episode, envs, n_shapes):
    return np.minimum((orc.reset_uniform(seed, episode, np.asarray(envs), 0) * n_shapes).astype(int), n_shapes - 1)


def find_seed(episode, envs, n_shapes, untabled):
    """A seed whose draws for `envs` include a shape without a table (untabled=True) or only shapes with one."""
    for seed in range(100000):
        k = drawn_shapes(seed, episode, envs, n_shapes)
        if bool((k >= 7).any()) == untabled:
            return seed
    raise AssertionError("no seed found")


@pytest.mark.parametrize("how", ["full", "list", "mask"])
def test_resets_keep_the_lookup_scan_off_envs_whose_shape_has_no_table(how):
    E, n_a = 16, 30
    shapes = mixed_library()
    S = len(shapes["l_cell"])
    sim = make_sim(E, n_a, shapes=shapes)
    rng = np.random.RandomState(8)
    held = rng.randint(0, 7, E)                                    # shapes with tables only
    ang = np.pi * rng.uniform(-1, 1, E)
    off = rng.uniform(-1.4, 1.4, (E, 2))
    sim.set_grid_pose(held, np.cos(ang), np.sin(ang), off[:, 0], off[:, 1])
    p, dp = rng.uniform(-2.4, 2.4, (E, 2, n_a)), rng.uniform(-0.5, 0.5, (E, 2, n_a))
    sim.set_state(p, dp); sim.observe()
    assert sim.fast_path == 2
    ob = make_oracle(sim, shapes, E)
    for e in range(E):
        g = sim.grid_from_pose(shapes["grid_origin"][held[e]], np.cos(ang[e]), np.sin(ang[e]), off[e, 0], off[e, 1])
        ob.params[e].n_g, ob.params[e].l_cell = g.shape[1], float(shapes["l_cell"][held[e]])
        ob.set_grid(e, g)
    ob.p[:], ob.dp[:] = p, dp
    ob.observe()
    assert_matches(sim, ob, AFTER_RESET, "set_grid_pose")
    listed = np.array([3, 9, 14, 0, 7, 12])
    t = 0
    for phase, untabled in enumerate((True, False)):
        episode = 10 + phase
        if how == "full":
            envs = np.arange(E)
        elif phase == 0:
            envs = listed
        else:                                                      # reset the envs that now hold an untabled shape once more
            envs = np.nonzero(held >= 7)[0]
        seed = find_seed(episode, envs + 0, S, untabled)
        if how == "full":
            sim.reset(seed=seed, episode=episode)
        elif how == "list":
            sim.reset_envs(torch.as_tensor(envs, dtype=torch.int32, device="cuda"), seed=seed, episode=episode)
        else:
            mask = torch.zeros(E, dtype=torch.bool)
            mask[envs] = True
            sim.reset(seed=seed, episode=episode, env_mask=mask)
        held[envs] = sim.reset_info[torch.as_tensor(envs, device="cuda"), 0].cpu().numpy().astype(int)
        assert np.array_equal(held[envs], drawn_shapes(seed, episode, envs, S))
        assert bool((held >= 7).any()) == untabled
        assert (sim.fast_path == 0) == bool((held >= 7).any()), (phase, sim.fast_path)
        oracle_follow_reset(ob, sim, shapes, envs)
        assert_matches(sim, ob, AFTER_RESET, ("reset", phase))
        for _ in range(10):
            a = orc.fill_actions(E, n_a, 3, t)
            a[::2] = goal_seeking_action(ob.obs[::2], ob.dp[::2], rng)
            sim.step(torch.from_numpy(a).cuda()); ob.step(a)
            assert_matches(sim, ob, ALL, ("step", t))
            t += 1
    assert sim.fast_path == 2


# ------------------------------------------------------------------------------------------------------------------
# 5. the benchmarked workload: bench.py's random regime, same schedule
def bench_schedule(sim, EP=200, C=25, ring=16):
    """bench.py's step_random: ring of fill_actions(226, r), cohort e % C reset after step t when t = (EP / C) * cohort (mod EP)
    with episode 1 + t.  Returns step(t), reset(t) -> the envs reset after step t (or None), and the action ring."""
    acts = torch.empty(ring, sim.E, 2, sim.n_a, dtype=torch.float32, device="cuda")
    for r in range(ring):
        sim.fill_actions(acts[r], seed=226, step=r)
    stride = EP // C
    lists = {ph: torch.arange(ph // stride, sim.E, C, dtype=torch.int32, device="cuda") for ph in range(0, EP, stride)}

    def step(t):
        sim.step(acts[t % ring])

    def reset(t):
        due = lists.get(t % EP)
        if due is not None:
            sim.reset_envs(due, seed=226, episode=1 + t)
        return due
    return step, reset, acts


def test_bench_random_regime_full_size_follows_the_oracle():
    """65 536 envs x 30 agents, production layout, bench.py's exact schedule for a 200-step pre-roll and 40 steps more: 128 envs
    drawn from every cohort follow the oracle at every step, and a twin simulator gives identical tensors."""
    E, n_a, C = 65536, 30, 25
    shapes = load_shapes()
    sims = [make_sim(E, n_a, "production") for _ in range(2)]
    schedules = []
    for s_ in sims:
        s_.reset(seed=226, episode=0)
        step, reset, acts = bench_schedule(s_)
        schedules.append((step, reset))
    rng = np.random.RandomState(0)
    pick = np.sort(np.concatenate([rng.choice(np.arange(c, E, C), 6 if c < 3 else 5, replace=False) for c in range(C)]))
    assert len(pick) == 128
    tp = torch.as_tensor(pick, device="cuda")
    for r in range(acts.shape[0]):
        assert np.array_equal(acts[r][tp].cpu().numpy(), orc.fill_actions(E, n_a, 226, r)[pick])
    ob = make_oracle(sims[0], shapes, len(pick))
    oracle_follow_reset(ob, sims[0], shapes, np.arange(len(pick)), pick)
    assert_matches(sims[0], ob, AFTER_RESET, "reset", pick=pick)
    assert sims[0].fast_path == 2
    outputs = ("p", "dp", "obs", "reward", "a_prior", "neighbor_index", "in_flags", "nearest_cell")
    for t in range(240):
        l0 = sims[0].launch_count
        for step, _ in schedules:
            step(t)
        ob.step(acts[t % 16][tp].cpu().numpy())
        assert_matches(sims[0], ob, ALL, ("step", t), pick=pick)
        dues = [reset(t) for _, reset in schedules]
        # a step is 2 launches; reset_envs adds k_reset and the two-launch observe of the listed envs
        assert sims[0].launch_count - l0 == (2 if dues[0] is None else 5), t
        if dues[0] is not None:
            rows = np.nonzero(np.isin(pick, dues[0].cpu().numpy()))[0]
            assert len(rows) >= 5
            oracle_follow_reset(ob, sims[0], shapes, rows, pick)
            assert_matches(sims[0], ob, AFTER_RESET, ("reset", t), rows=rows, pick=pick)
        for name in outputs:
            assert torch.equal(bits(getattr(sims[0], name)), bits(getattr(sims[1], name))), (name, t)
    assert sims[0].fast_path == 2
    assert ob.in_flags.sum() > 0


def test_bench_dump_equals_the_in_process_replay(tmp_path):
    """bench.py --dump-outputs of the random regime (reset, 200 pre-roll + 2 warm-up + 7 timed steps of the auto-reset schedule)
    equals the same 209 steps replayed here, row for row."""
    E = 4096
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--regime", "random", "--envs-per-gpu", str(E), "--steps", "7",
                        "--warmup", "2", "--no-e2e", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path)],
                       cwd=REPO, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 7
    sim = make_sim(E, 30, "production")
    sim.reset(seed=226, episode=0)
    step, reset, _ = bench_schedule(sim)
    for t in range(209):
        step(t)
        reset(t)
    files = sorted(f for f in os.listdir(tmp_path) if f.startswith("random_"))
    assert {"random_obs.npy", "random_a_prior.npy", "random_p.npy", "random_neighbor_index.npy"} <= set(files)
    for f in files:
        dump = np.load(tmp_path / f)
        name = f[len("random_"):-len(".npy")]
        pick = np.sort(np.random.RandomState(0).choice(E, dump.shape[0], replace=False))
        got = getattr(sim, name)[torch.as_tensor(pick, device="cuda")].cpu().numpy().astype(dump.dtype)
        assert np.array_equal(got, dump), f


# ------------------------------------------------------------------------------------------------------------------
# 6. errors and memory safety
def test_reset_envs_rejects_bad_calls_without_launching():
    from marl_llm_b200.batched import BatchedAssemblySim
    E, n_a = 16, 30
    shapes = load_shapes()
    ids = torch.arange(4, dtype=torch.int32, device="cuda")
    bare = BatchedAssemblySim(E, n_a, int(shapes["n_g"].max()), orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"]))
    sim = make_sim(E, n_a, "production")
    for s_, bad in ((bare, ids), (sim, ids)):                      # before set_shapes; before a first observe
        l0 = s_.launch_count
        with pytest.raises(SwarmError):
            s_.reset_envs(bad, seed=1)
        assert s_.launch_count == l0
    sim.reset(seed=1)
    l0 = sim.launch_count
    for bad in (ids[:0], torch.arange(E + 1, dtype=torch.int32, device="cuda")):      # count 0 (valid pointer); count > E
        with pytest.raises(SwarmError):
            sim.reset_envs(bad, seed=1)
    assert sim.launch_count == l0


@pytest.mark.parametrize("n_a", [30, 100])
def test_reset_envs_writes_nothing_outside_its_buffers(n_a):
    E = 37
    sim = make_sim(E, n_a, guard_bytes=65536)
    sim.reset(seed=3)
    act = torch.empty(E, 2, n_a, dtype=torch.float32, device="cuda")
    lists = ([E - 1], [0], list(range(E - 1, -1, -1)), [5, 36, 17])
    for t, ids in enumerate(lists):
        sim.step(sim.fill_actions(act, seed=2, step=t))
        sim.reset_envs(torch.tensor(ids, dtype=torch.int32, device="cuda"), seed=4, episode=t, env_offset=7 * t)
    mask = torch.zeros(E, dtype=torch.bool); mask[-3:] = True
    sim.reset(seed=4, episode=9, env_mask=mask)
    sim.step(sim.fill_actions(act, seed=2, step=9))
    torch.cuda.synchronize()
    assert sim.check_guards()
