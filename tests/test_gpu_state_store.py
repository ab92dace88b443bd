"""State store (swarm_state_save / swarm_state_load, marl_llm_b200.state_store): save envs, disturb the handle, load them back,
and every following step is bit-identical to a twin handle that was never disturbed.

A slot holds an env's whole state: p / dp, grid row, word boxes, frame, n_g, in_thresh, library pose and shape id, nearest cell,
neighbour list, in_flags, obs, reward, the two priors and the index arrays.  The store also records the source's match record
(which decides the scan kernel), whether its prior was valid, and the fingerprint of its shape library.  Every comparison here is
bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

import bench
from marl_llm_b200 import _lib
from marl_llm_b200._lib import SwarmError
from marl_llm_b200.state_store import StateStore
from oracle import oracle as orc
from tests.helpers import load_shapes

pytestmark = pytest.mark.gpu

SHAPES = load_shapes()
NGM = int(max(SHAPES["n_g"]))
PATHS = {"exact": 2, "detected": 1, "nolib": 0, "brute": 0}   # start of each scan path and the swarm_fast_path it gives
OUT = ("p", "dp", "obs", "reward", "a_prior", "neighbor_index", "in_flags", "sensed_index", "occupied_index")


def bits(t):
    return t.view({8: torch.int64, 4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def make_sim(E, n_a, path="exact", layout="production", shapes=SHAPES, **kw):
    from marl_llm_b200.batched import BatchedAssemblySim
    parity = layout == "parity"
    sim = BatchedAssemblySim(E, n_a, NGM, orc.r_avoid_for(n_a, SHAPES["n_g"], SHAPES["l_cell"]),
                             out_dtype=torch.float64 if parity else torch.float32, emit_indices=parity,
                             brute_force_scan=path == "brute", **kw)
    if path != "nolib":
        sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    return sim


def start(sim, path, seed=3):
    """The first state of scan path `path`: a device reset (exact poses) or uploaded grids (poses detected / no library)."""
    if path in ("exact", "brute"):
        sim.reset(seed=seed)
    else:
        blocks, n_g, l_cell, p, dp = bench.synth_batch(sim.E, sim.n_a, SHAPES, seed, "random")
        sim.set_grid(blocks, n_g, l_cell)
        sim.set_state(p, dp)
        sim.observe()
    assert sim.fast_path == PATHS[path]


def actions(E, n_a, seed, t):
    return torch.from_numpy(orc.fill_actions(E, n_a, seed, t)).cuda()


def pending_prior(sim):
    return sim._a_prior[1] if sim.a_prior.data_ptr() == sim._a_prior[0].data_ptr() else sim._a_prior[0]


def stored(sim):
    """Bit patterns of every buffer a slot holds (the two priors: the one the next step returns and the last one returned)."""
    d = dict(p=sim.p, dp=sim.dp, grid=sim._grid, n_g=sim._n_g, in_thresh=sim._in_thresh, word_box=sim._word_box, frame=sim._frame,
             nearest_cell=sim.nearest_cell, neighbor_index=sim.neighbor_index, in_flags=sim.in_flags, obs=sim.obs, reward=sim.reward,
             sensed_index=sim.sensed_index, occupied_index=sim.occupied_index)
    if sim.want_prior:
        d.update(prior_next=pending_prior(sim), prior_last=sim.a_prior)
    return {k: bits(v).clone() for k, v in d.items() if v is not None}


def outputs(sim):
    d = {n: getattr(sim, n) for n in OUT if n != "a_prior"}
    d["a_prior"] = sim.a_prior if sim.want_prior else None
    return {k: bits(v).clone() for k, v in d.items() if v is not None}


def assert_rows_equal(a, b, rows_a, rows_b, what):
    ra, rb = (torch.as_tensor(np.asarray(r, dtype=np.int64), device="cuda") for r in (rows_a, rows_b))
    for k in a:
        assert torch.equal(a[k][ra], b[k][rb]), (k, what)


def continue_equal(sim, twin, steps, seed, rows=None, twin_rows=None):
    """`steps` steps of both handles; row rows[k] of sim gets the actions of row twin_rows[k] of the twin; outputs compared."""
    rows = np.arange(sim.E) if rows is None else np.asarray(rows)
    twin_rows = rows if twin_rows is None else np.asarray(twin_rows)
    for t in range(steps):
        at = actions(twin.E, twin.n_a, seed, t)
        a = actions(sim.E, sim.n_a, seed + 1000, t)
        a[torch.as_tensor(rows, device="cuda")] = at[torch.as_tensor(twin_rows, device="cuda")]
        sim.step(a); twin.step(at)
        assert_rows_equal(outputs(sim), outputs(twin), rows, twin_rows, ("step", t))


def jittered_grids(sim, envs, seed):
    """Grids for `envs`: library shapes in other poses, the last one jittered by 1e-6 (no library shape matches it)."""
    from marl_llm_b200.batched import BatchedAssemblySim
    rng = np.random.RandomState(seed)
    grids, l_cell = [], []
    for i, e in enumerate(envs):
        k = (i + 1) % len(SHAPES["n_g"])
        ang = rng.uniform(-np.pi, np.pi)
        g = BatchedAssemblySim.grid_from_pose(SHAPES["grid_origin"][k], np.cos(ang), np.sin(ang), *rng.uniform(-1, 1, 2))
        if i == len(envs) - 1:
            g = g + rng.uniform(-1e-6, 1e-6, g.shape)
        grids.append(g); l_cell.append(SHAPES["l_cell"][k])
    blocks, n_g = BatchedAssemblySim.pack_grids(grids, NGM)
    return blocks, n_g, np.array(l_cell)


def disturb(sim, path, seed=5):
    """Everything a saved env's state must survive: other grids (one of them unmatched), an observation-buffer swap, resets,
    steps with other actions."""
    blocks, n_g, l_cell = jittered_grids(sim, range(2, 8), seed)
    sim.set_grid(blocks, n_g, l_cell, env0=2)
    assert sim.fast_path == 0
    sim.set_obs_buffer(torch.full_like(sim.obs, 7.0))
    if path != "nolib":
        sim.reset_envs(torch.tensor([9, 1, 4], dtype=torch.int32, device="cuda"), seed=77, episode=3)
    for t in range(2):
        sim.step(actions(sim.E, sim.n_a, seed + 50, t))


# ------------------------------------------------------------------------------------------------------------------
CASES = [(p, n, lay, {}) for p in PATHS for n in (30, 100) for lay in ("production", "parity")] + [
    ("exact", 30, "production", dict(obs_layout="agent_major")), ("detected", 100, "parity", dict(obs_layout="agent_major")),
    ("exact", 30, "parity", dict(is_periodic=True)), ("nolib", 30, "production", dict(is_periodic=True)),
    ("exact", 30, "production", dict(is_con_self_state=False)), ("detected", 30, "parity", dict(want_prior=False)),
    ("exact", 100, "production", dict(want_prior=False))]


@pytest.mark.parametrize("path,n_a,layout,kw", CASES)
def test_continuation_after_load_equals_the_uninterrupted_run(path, n_a, layout, kw):
    E = 48
    A, T = make_sim(E, n_a, path, layout, **kw), make_sim(E, n_a, path, layout, **kw)
    if not A.want_prior:
        for s in (A, T):
            for b in s._a_prior:
                b.fill_(-123.0)
    for s in (A, T):
        start(s, path)
        for t in range(3):
            s.step(actions(E, n_a, 1, t))
    perm = np.random.RandomState(0).permutation(E)
    store = StateStore(A, E)
    store.save(perm, slots=np.arange(E)[::-1])
    saved = stored(A)
    disturb(A, path)
    store.load(np.arange(E)[::-1], perm)
    now = stored(A)
    for k, v in saved.items():
        assert torch.equal(now[k], v), k
    assert A.fast_path == T.fast_path == PATHS[path]
    assert np.array_equal(A.n_g, T.n_g) and np.array_equal(A.l_cell, T.l_cell)
    la, lt = A.launch_count, T.launch_count
    continue_equal(A, T, 4, seed=2)
    assert A.launch_count - la == T.launch_count - lt
    if not A.want_prior:
        for s in (A, T):
            for b in s._a_prior:
                assert bool((b == -123.0).all())


def test_partial_loads_leave_other_envs_alone():
    E = 40
    A, T = make_sim(E, 30, "exact", "parity"), make_sim(E, 30, "exact", "parity")
    for s in (A, T):
        start(s, "exact")
        for t in range(3):
            s.step(actions(E, 30, 1, t))
    store = StateStore(A, 8)
    lists = [[17, 3, 29, 8, 0, 22], [5], [E - 1]]
    store.save(sum(lists, []))
    saved = stored(A)
    disturb(A, "exact")
    k0 = 0
    for ids in lists:
        before = stored(A)
        store.load(np.arange(k0, k0 + len(ids)), ids)
        k0 += len(ids)
        after = stored(A)
        others = np.setdiff1d(np.arange(E), ids)
        assert_rows_equal(after, before, others, others, ("untouched", ids))
        assert_rows_equal(after, saved, ids, ids, ("loaded", ids))
    loaded = sum(lists, [])
    continue_equal(A, T, 4, seed=2, rows=loaded)


def test_clone_one_env_into_seventeen_and_follow_the_oracle():
    E = 32
    A = make_sim(E, 30, "detected", "parity")
    start(A, "detected")                           # set_grid keeps the host mirrors n_g / l_cell the load must carry over
    for t in range(3):
        A.step(actions(E, 30, 1, t))
    src, clones = 7, [e for e in range(18) if e != 7][:17]
    store = StateStore(A, 1)
    store.save([src])
    store.load([0] * len(clones), clones)
    group = np.array([src] + clones)
    ng, lc = int(A.n_g[src]), float(A.l_cell[src])
    assert ng > 0 and (A.n_g[group] == ng).all() and (A.l_cell[group] == lc).all()
    # the oracle rebuilt from the saved state (grid, n_g, l_cell, p, dp), as oracle_follow_reset does after a reset
    c = clones[-1]
    ob = orc.OracleBatch([orc.make_params(30, NGM, lc, A.r_avoid)], nthreads=1, ng_max=NGM)
    ob.params[0].n_g, ob.params[0].l_cell = ng, lc
    ob.set_grid(0, np.ascontiguousarray(A._grid[c, :ng].cpu().numpy().T))
    ob.p[0], ob.dp[0] = A.p[c].cpu().numpy(), A.dp[c].cpu().numpy()
    ob.observe()
    for name in ("obs", "neighbor_index", "in_flags", "sensed_index", "occupied_index"):
        assert np.array_equal(getattr(A, name)[c].cpu().numpy(), getattr(ob, name)[0]), name
    for t in range(20):
        a = actions(E, 30, 4, t)
        a[torch.as_tensor(group, device="cuda")] = a[src].clone()
        A.step(a); ob.step(a[c:c + 1].cpu().numpy())
        out = outputs(A)
        for k, v in out.items():
            assert bool((v[torch.as_tensor(group, device="cuda")] == v[src]).all()), (k, t)
        for name in OUT:
            assert np.array_equal(getattr(A, name)[c].cpu().numpy(), getattr(ob, name)[0]), (name, t)


def test_mirror_follows_the_slots_records():
    E = 24
    D = make_sim(E, 30, "detected")                  # poses detected: records DETECTED
    start(D, "detected")
    D.step(actions(E, 30, 1, 0))
    store = StateStore(D, E)
    store.save(range(E))
    X = make_sim(E, 30, "exact")
    start(X, "exact", seed=8)
    store.load([3, 4], [10, 11], sim=X)
    assert X.fast_path == 1                          # two detected envs among exact ones
    store.load(range(E), range(E), sim=X)
    assert X.fast_path == 1
    X.reset(seed=9)
    assert X.fast_path == 2


def test_unmatched_slot_turns_the_fast_path_off_and_a_full_reset_restores_it():
    E = 24
    A, T = make_sim(E, 30, "exact"), make_sim(E, 30, "exact")
    blocks, n_g, l_cell = jittered_grids(A, [5], seed=1)
    for s in (A, T):
        start(s, "exact")
        s.step(actions(E, 30, 1, 0))
        s.set_grid(blocks, n_g, l_cell, env0=5)
        s.step(actions(E, 30, 1, 1))
        assert s.fast_path == 0
    store = StateStore(A, E)
    store.save(range(E))
    A.reset(seed=8)
    assert A.fast_path == 2
    store.load([5], [5])
    assert A.fast_path == 0
    store.load(range(E), range(E))
    assert A.fast_path == 0
    continue_equal(A, T, 3, seed=2)
    A.reset(seed=9)
    assert A.fast_path == 2


def test_launches_after_a_load_and_the_prior_of_a_dirty_slot():
    E = 24
    A, T = make_sim(E, 30, "exact"), make_sim(E, 30, "exact")
    for s in (A, T):
        start(s, "exact")
        s.step(actions(E, 30, 1, 0))
    l0 = T.launch_count
    T.step(actions(E, 30, 1, 1))
    per_step = T.launch_count - l0
    A.step(actions(E, 30, 1, 1))
    # a slot saved with a valid prior: the step after the load launches what a step launches
    store = StateStore(A, E)
    store.save(range(E))
    A.step(actions(E, 30, 9, 0))
    n = A.launch_count
    store.load(range(E), range(E))
    assert A.launch_count == n + 1
    n = A.launch_count
    A.step(actions(E, 30, 1, 2)); T.step(actions(E, 30, 1, 2))
    assert A.launch_count - n == per_step
    assert_rows_equal(outputs(A), outputs(T), range(E), range(E), "valid prior")
    # right after set_state the prior is stale: a slot saved then makes the next step after its load run k_prior
    for s in (A, T):
        s.set_state(s.p.clone(), s.dp.clone())
    store.save(range(E))
    A.step(actions(E, 30, 9, 1))
    store.load(range(E), range(E))
    n, m = A.launch_count, T.launch_count
    A.step(actions(E, 30, 1, 3)); T.step(actions(E, 30, 1, 3))
    assert A.launch_count - n == per_step + 1 == T.launch_count - m
    assert_rows_equal(outputs(A), outputs(T), range(E), range(E), "dirty prior")
    continue_equal(A, T, 2, seed=5)


def test_across_handles():
    E = 64
    A, T = make_sim(E, 30, "exact", "parity"), make_sim(E, 30, "exact", "parity")
    for s in (A, T):
        start(s, "exact")
        for t in range(3):
            s.step(actions(E, 30, 1, t))
    store = StateStore(A, E)
    store.save(range(E))
    # a 512-env handle of the same configuration
    B = make_sim(512, 30, "exact", "parity")
    start(B, "exact", seed=11)
    B.step(actions(512, 30, 3, 0))
    rows = np.arange(511, 511 - 2 * E, -2)
    store.load(range(E), rows, sim=B)
    assert B.fast_path == 2
    # the same shapes in another order: another library, the envs come back unmatched
    rev = dict(grid_origin=SHAPES["grid_origin"][::-1], l_cell=SHAPES["l_cell"][::-1].copy(), n_g=SHAPES["n_g"][::-1].copy())
    R = make_sim(E, 30, "exact", "parity", shapes=rev)
    start(R, "exact", seed=12)
    store.load(range(E), range(E), sim=R)
    assert R.fast_path == 0
    # a handle that was never observed takes a load of every env
    U = make_sim(E, 30, "exact", "parity")
    assert not U.observed
    store.load(range(E), range(E), sim=U)
    assert U.observed and U.fast_path == 2
    for t in range(4):
        at = actions(E, 30, 2, t)
        ab = actions(512, 30, 7, t)
        ab[torch.as_tensor(rows, device="cuda")] = at
        T.step(at); B.step(ab); R.step(at); U.step(at)
        want = outputs(T)
        assert_rows_equal(outputs(B), want, rows, range(E), ("512-env handle", t))
        assert_rows_equal(outputs(R), want, range(E), range(E), ("reordered library", t))
        assert_rows_equal(outputs(U), want, range(E), range(E), ("unobserved handle", t))
    for other in (make_sim(E, 31, "exact", "parity"), make_sim(E, 30, "exact", "production")):
        start(other, "exact")
        with pytest.raises(SwarmError, match="code 1"):
            store.load([0], [0], sim=other)


def test_reset_envs_after_a_load_equals_the_reset_without_it():
    E = 40
    A, T = make_sim(E, 30, "exact", "parity"), make_sim(E, 30, "exact", "parity")
    for s in (A, T):
        start(s, "exact")
        for t in range(3):
            s.step(actions(E, 30, 1, t))
    store = StateStore(A, E)
    store.save(range(E))
    disturb(A, "exact")
    store.load(range(E), range(E))
    ids = torch.tensor([13, 2, 30, 7], dtype=torch.int32, device="cuda")
    for s in (A, T):
        s.reset_envs(ids, seed=5, episode=9)
    assert A.fast_path == T.fast_path
    assert_rows_equal(stored(A), stored(T), range(E), range(E), "after reset_envs")
    continue_equal(A, T, 4, seed=3)


def test_full_batch_save_and_load():
    E = 65536
    A, T = make_sim(E, 30, "exact"), make_sim(E, 30, "exact")
    for s in (A, T):
        start(s, "exact")
        for t in range(3):
            s.step(actions(E, 30, 1, t))
    store = StateStore(A, E)
    store.save(range(E))
    saved = stored(A)
    for t in range(5):
        A.step(actions(E, 30, 9, t))
    store.load(range(E), range(E))
    now = stored(A)
    for k, v in saved.items():
        assert torch.equal(now[k], v), k
    del now, saved
    continue_equal(A, T, 5, seed=2)


def test_guard_zones_and_more_pairs_than_one_launch():
    E = 2100
    A = make_sim(E, 30, "exact", guard_bytes=4096)
    B = make_sim(E, 30, "exact", guard_bytes=4096)
    for s, seed in ((A, 3), (B, 4)):
        start(s, "exact", seed=seed)
        s.step(actions(E, 30, 1, 0))
    store = StateStore(A, E)
    n = A.launch_count
    store.save(range(E))
    assert A.launch_count == n + 2
    saved = stored(A)
    perm = np.random.RandomState(1).permutation(E)
    store.load(perm, range(E), sim=B)
    got = stored(B)
    assert_rows_equal(got, saved, range(E), perm, "loaded across handles")
    assert A.check_guards() and B.check_guards()


def test_every_invalid_argument_leaves_handle_and_store_unchanged():
    E = 16
    lib = _lib.load()
    A = make_sim(E, 30, "exact", "parity")
    start(A, "exact")
    A.step(actions(E, 30, 1, 0))
    store = StateStore(A, 4)
    store.save([3, 5], [0, 1])
    saved = {k: v[[3, 5]] for k, v in stored(A).items()}
    A.step(actions(E, 30, 1, 1))
    before, launches, fast = stored(A), A.launch_count, A.fast_path
    fresh = make_sim(E, 30, "exact", "parity")
    other = make_sim(E, 30, "exact", "production")
    start(other, "exact")

    def ids(v):
        return np.ascontiguousarray(v, dtype=np.int32)

    def call(fn, sim, st, a, b, count=None):
        a, b = ids(a), ids(b)
        n = len(a) if count is None else count
        return fn(sim, st, C.c_void_p(a.ctypes.data), C.c_void_p(b.ctypes.data), n, A._stream())

    s, h = lib.swarm_state_save, lib.swarm_state_load
    bad = [
        ("null handle", lambda: call(s, None, store._h, [0], [0])),
        ("null store", lambda: call(h, A._h, None, [0], [0])),
        ("null env ids", lambda: s(A._h, store._h, None, C.c_void_p(ids([0]).ctypes.data), 1, A._stream())),
        ("null slots", lambda: h(A._h, store._h, None, C.c_void_p(ids([0]).ctypes.data), 1, A._stream())),
        ("count 0", lambda: call(s, A._h, store._h, [0], [2], count=0)),
        ("negative count", lambda: call(h, A._h, store._h, [0], [0], count=-1)),
        ("env id -1", lambda: call(s, A._h, store._h, [-1], [2])),
        ("env id E", lambda: call(h, A._h, store._h, [0], [E])),
        ("slot -1", lambda: call(s, A._h, store._h, [0], [-1])),
        ("slot capacity", lambda: call(h, A._h, store._h, [4], [0])),
        ("save: repeated slot", lambda: call(s, A._h, store._h, [0, 1], [2, 2])),
        ("load: repeated env", lambda: call(h, A._h, store._h, [0, 1], [6, 6])),
        ("load: empty slot", lambda: call(h, A._h, store._h, [0, 2], [6, 7])),
        ("save: never observed", lambda: call(s, fresh._h, store._h, [0], [2])),
        ("load: partial into a never observed handle", lambda: call(h, fresh._h, store._h, [0], [0])),
        ("save: other configuration", lambda: call(s, other._h, store._h, [0], [2])),
        ("load: other configuration", lambda: call(h, other._h, store._h, [0], [0])),
    ]
    for what, f in bad:
        assert f() == _lib.SWARM_ERR_INVALID, what
        assert A.launch_count == launches and A.fast_path == fast, what
        now = stored(A)
        for k, v in before.items():
            assert torch.equal(now[k], v), (what, k)
    assert not fresh.observed
    out = C.c_void_p()
    assert lib.swarm_state_store_create(A._h, 0, C.byref(out)) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_state_store_create(None, 4, C.byref(out)) == _lib.SWARM_ERR_INVALID
    from marl_llm_b200.flocking import BatchedFlockingSim
    fl = BatchedFlockingSim(4, 30)
    assert lib.swarm_state_store_create(fl._h, 4, C.byref(out)) == _lib.SWARM_ERR_UNSUPPORTED
    assert call(s, fl._h, store._h, [0], [2]) == _lib.SWARM_ERR_UNSUPPORTED
    # the store is unchanged: its two slots still hold what was saved, the others are still empty
    store.load([0, 1], [3, 5])
    now = stored(A)
    for k, v in saved.items():
        assert torch.equal(now[k][[3, 5]], v), k
    assert call(h, A._h, store._h, [2], [0]) == _lib.SWARM_ERR_INVALID
    assert store.slot_bytes % 128 == 0 and lib.swarm_state_slot_bytes(None) == 0
