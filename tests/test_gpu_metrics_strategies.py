"""The wrapper's evaluation metrics (swarm_metrics / k_metrics, assembly_wrapper.py:48-129) and the reference env's host
strategies (swarm_strategy_actions / k_strategy, assembly.py:524-601, 876-941) against plain references: at swarm sizes on
both sides of every block-size boundary of the two kernels, on batches whose envs hold grids of different sizes, after each
way a grid can be installed, and at constructed edges where the statistics are decided (distance ties, the strict coverage
radius, coincident agents, the in-shape threshold).

Every device output buffer is filled with NaN before the call, so an env or agent the kernel skips cannot pass."""
import numpy as np
import pytest
import torch

from oracle import metrics_oracle
from oracle import oracle as orc
from oracle.oracle import OracleBatch
from tests.helpers import goal_seeking_action, load_shapes, oracle_follow_reset, reset_like_reference

pytestmark = pytest.mark.gpu

NGM = 560                 # larger than every library shape (487-536 cells): every env has padding cells


@pytest.fixture(scope="module")
def shapes():
    return load_shapes()


def new_sim(E, n_a, r_avoid, d_sen=0.4, n_g_max=NGM):
    from marl_llm_b200.batched import BatchedAssemblySim
    return BatchedAssemblySim(E, n_a, n_g_max, r_avoid, out_dtype=torch.float64, d_sen=d_sen)


def posed_grid(rng, shapes, k):
    """Library shape k under a random pose (assembly.py:175-187), rounded like set_grid_pose / reset() round it."""
    from marl_llm_b200.batched import BatchedAssemblySim
    ang = np.pi * rng.uniform(-1, 1)
    off = rng.uniform(-1.4, 1.4, 2)
    return BatchedAssemblySim.grid_from_pose(shapes["grid_origin"][k], np.cos(ang), np.sin(ang), off[0], off[1])


def sq(px, py, gx, gy):
    """Squared distance as the reference and the kernels evaluate it: difference, products and sum each rounded."""
    dx, dy = px - gx, py - gy
    return dx * dx + dy * dy


def thresh_lt(d):
    """Smallest double T with sqrt(T) >= d (rounded), so that sqrt(s) < d <=> s < T."""
    t = d * d
    while np.sqrt(t) >= d:
        t = np.nextafter(t, -np.inf)
    while np.sqrt(np.nextafter(t, np.inf)) < d:
        t = np.nextafter(t, np.inf)
    return np.nextafter(t, np.inf)


def at_squared_distance(rng, gx, gy, target, direction=None):
    """A position whose squared distance from (gx, gy) evaluates to exactly `target`: points on the circle of radius
    sqrt(target) (within 0.05 rad of `direction`, or at random angles), moved by up to 12 ulps per coordinate until one
    hits it."""
    ang = rng.uniform(0, 2 * np.pi, 128) if direction is None else direction + rng.uniform(-0.05, 0.05, 128)
    bx, by = gx + np.sqrt(target) * np.cos(ang), gy + np.sqrt(target) * np.sin(ang)
    ks = np.arange(-12, 13)
    px = bx[:, None, None] + ks[None, :, None] * np.spacing(bx)[:, None, None]
    py = by[:, None, None] + ks[None, None, :] * np.spacing(by)[:, None, None]
    px, py = (a.ravel() for a in np.broadcast_arrays(px, py))
    hit = np.flatnonzero(sq(px, py, gx, gy) == target)
    assert hit.size, "no position found at the requested squared distance"
    return px[hit[0]], py[hit[0]]


# ---------------------------------------------------------------------------------------------------------------------
# metrics references
def ratio_in_kernel_order(v):
    """(var(v) - min(v)) / (max(v) - min(v)) evaluated the way k_metrics does: sequential sums, mean = sum / n,
    var = sum((v - mean)^2) / n, every operation rounded separately."""
    v = [np.float64(x) for x in v]
    n = np.float64(len(v))
    s = np.float64(0.0)
    for x in v:
        s += x
    mean = s / n
    var = np.float64(0.0)
    for x in v:
        d = x - mean
        var += d * d
    var /= n
    lo, hi = min(v), max(v)
    with np.errstate(divide="ignore", invalid="ignore"):
        return (var - lo) / (hi - lo)


def voronoi_counts(p, grid, rounded=True):
    """Cells per agent, each cell going to the first agent at the smallest distance (rounded=True: the reference's
    np.argmin of the norms) or at the smallest squared distance (rounded=False)."""
    s = sq(p[0][None, :], p[1][None, :], grid[0][:, None], grid[1][:, None])          # [n_g, n_a]
    return np.bincount(np.argmin(np.sqrt(s) if rounded else s, axis=1), minlength=p.shape[1])


def kernel_order_metrics(p, grid, r_avoid):
    """k_metrics restated in its own order: coverage and Voronoi counts exact, nearest non-coincident distances exact, the
    two ratios by ratio_in_kernel_order.  The device must match this bit for bit."""
    s = sq(p[0][None, :], p[1][None, :], grid[0][:, None], grid[1][:, None])
    cov = int((np.sqrt(s) < r_avoid / 2).any(axis=1).sum()) / grid.shape[1]
    pp = sq(p[0][None, :], p[1][None, :], p[0][:, None], p[1][:, None])
    mins = np.sqrt(np.where(pp != 0, pp, np.inf).min(axis=1))
    return np.array([cov, ratio_in_kernel_order(mins), ratio_in_kernel_order(voronoi_counts(p, grid))])


def device_metrics(sim):
    sim.metrics()
    sim._metrics.fill_(float("nan"))
    return sim.metrics().cpu().numpy()


def check_metrics(sim, grids, r_avoid):
    """Device metrics of every env against the kernel-order restatement (bit for bit) and the wrapper's formulas
    (metrics_oracle: coverage exact, the ratios to 1e-12, NumPy's np.var summing pairwise).  Returns the latter."""
    got = device_metrics(sim)
    p = sim.p.cpu().numpy()
    mine = np.stack([kernel_order_metrics(p[e], grids[e], r_avoid) for e in range(sim.E)])
    ref = np.stack([metrics_oracle.all_metrics(p[e], grids[e], r_avoid) for e in range(sim.E)])
    assert not np.isnan(mine).any()
    bad = np.flatnonzero(~(got == mine).all(axis=1))
    assert bad.size == 0, (bad, got[bad], mine[bad])
    assert np.array_equal(got[:, 0], ref[:, 0])
    np.testing.assert_allclose(got[:, 1:], ref[:, 1:], rtol=1e-12, atol=0)
    return ref


# ---------------------------------------------------------------------------------------------------------------------
# strategies
def oracle_batch(E, n_a, r_avoid, d_sen, grids=None, l_cells=None):
    params = [orc.make_params(n_a, 1 if grids is None else grids[e].shape[1], 0.0 if l_cells is None else float(l_cells[e]),
                              r_avoid, d_sen=d_sen) for e in range(E)]
    ob = OracleBatch(params, nthreads=8, ng_max=NGM)
    for e in range(E if grids is not None else 0):
        ob.set_grid(e, grids[e])
    return ob


def check_strategies(sim, ob):
    """'llm' bit-identical to the C restatement, 'rule' within 1e-13 (the cosine weights may differ in the last bit), for
    the state the simulator holds and the neighbour list of its last observation."""
    ob.p[:], ob.dp[:] = sim.p.cpu().numpy(), sim.dp.cpu().numpy()
    ob.observe()
    assert np.array_equal(sim.neighbor_index.cpu().numpy(), ob.neighbor_index)
    for kind in ("llm", "rule"):
        out = torch.full((sim.E, 2, sim.n_a), float("nan"), dtype=torch.float64, device=sim.device)
        got = sim.strategy_actions(kind, out=out).cpu().numpy()
        want = orc.strategy_actions(ob, kind)
        assert not np.isnan(got).any(), kind
        if kind == "llm":
            assert np.array_equal(got, want)
        else:
            assert np.abs(got - want).max() < 1e-13, np.abs(got - want).max()


def check_installed(sim, ob, r_avoid):
    """Metrics and both strategies against references built from the grids the oracle holds for each env."""
    check_strategies(sim, ob)
    check_metrics(sim, [ob.grid_of(e) for e in range(ob.E)], r_avoid)


def rollout(sim, rng, steps):
    for _ in range(steps):
        a = goal_seeking_action(sim.obs.cpu().numpy(), sim.dp.cpu().numpy(), rng)
        sim.step(torch.from_numpy(a).to(sim.device))


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_a", [2, 7, 31, 32, 33, 100, 127, 128, 129, 257, 1024])
def test_metrics_on_batches_of_different_shapes(shapes, n_a):
    """k_metrics runs 128 threads per env: cells always take several turns of its loop, agents from 129 on.  Every env of
    the batch holds a different library shape (n_g differs, padding cells behind every grid).  States: the random spawn; a
    third of the agents placed on cells (shared cells: coincident agents, piled-up counts); a goal-seeking rollout."""
    E = 7 if n_a <= 257 else 3
    rng = np.random.RandomState(n_a)
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    ks = rng.permutation(len(shapes["n_g"]))[:E]
    grids = [posed_grid(rng, shapes, k) for k in ks]
    assert len({g.shape[1] for g in grids}) == E
    sim = new_sim(E, n_a, r_avoid)
    blocks, n_g = sim.pack_grids(grids, NGM)
    sim.set_grid(blocks, n_g, shapes["l_cell"][ks])
    spawn = [reset_like_reference(rng, n_a, shapes)[2:] for _ in range(E)]
    P, DP = np.stack([s[0] for s in spawn]), np.stack([s[1] for s in spawn])
    sim.set_state(P, DP)
    check_metrics(sim, grids, r_avoid)

    on = P.copy()
    m = max(1, n_a // 3)
    for e in range(E):
        cells = rng.randint(0, grids[e].shape[1], max(1, m // 2))
        on[e][:, :m] = grids[e][:, rng.choice(cells, m)]
    assert m < 2 or all(np.unique(on[e][:, :m], axis=1).shape[1] < m for e in range(E))
    sim.set_state(on, DP)
    check_metrics(sim, grids, r_avoid)

    sim.set_state(P, DP)
    sim.observe()
    rollout(sim, rng, 40)
    ref = check_metrics(sim, grids, r_avoid)
    assert ref[:, 0].max() > 0.3, ref[:, 0]


def install(sim, ob, path, rng, shapes):
    """Install grids on `sim` through `path`, and make `ob` hold the grid, n_g and l_cell each env should then have."""
    from marl_llm_b200.batched import BatchedAssemblySim
    E, n_a = sim.E, sim.n_a
    ks = rng.randint(0, len(shapes["n_g"]), E)
    l_cells = shapes["l_cell"][ks]

    def hold(grids):
        for e in range(E):
            ob.params[e].n_g, ob.params[e].l_cell = grids[e].shape[1], float(l_cells[e])
            ob.set_grid(e, grids[e])

    def set_grid(grids):
        blocks, n_g = sim.pack_grids(grids, NGM)
        sim.set_grid(blocks, n_g, l_cells)
        hold(grids)

    def spawn():
        s = [reset_like_reference(rng, n_a, shapes)[2:] for _ in range(E)]
        sim.set_state(np.stack([x[0] for x in s]), np.stack([x[1] for x in s]))
        sim.observe()
        ob.p[:], ob.dp[:] = sim.p.cpu().numpy(), sim.dp.cpu().numpy()
        ob.observe()

    if path == "set_grid":
        set_grid([posed_grid(rng, shapes, k) for k in ks])
        spawn()
    elif path == "set_grid_pose":
        ang = np.pi * rng.uniform(-1, 1, E)
        cs, sn, off = np.cos(ang), np.sin(ang), rng.uniform(-1.4, 1.4, (E, 2))
        sim.set_grid_pose(ks, cs, sn, off[:, 0], off[:, 1])
        hold([BatchedAssemblySim.grid_from_pose(shapes["grid_origin"][ks[e]], cs[e], sn[e], off[e, 0], off[e, 1]) for e in range(E)])
        spawn()
    elif path == "reset":
        sim.reset(seed=31, episode=2)
        oracle_follow_reset(ob, sim, shapes, np.arange(E))
    elif path == "reset_envs":
        set_grid([posed_grid(rng, shapes, k) for k in ks])
        spawn()
        ids = rng.permutation(E)[:E // 3]
        sim.reset_envs(torch.as_tensor(ids, dtype=torch.int32, device=sim.device), seed=7, episode=1)
        oracle_follow_reset(ob, sim, shapes, ids)
    elif path == "smaller_after_larger":
        large = [posed_grid(rng, shapes, k) for k in ks]
        set_grid(large)
        small = []
        for g in large:
            c0 = rng.randint(0, g.shape[1] - 120)
            small.append(np.ascontiguousarray(g[:, c0:c0 + rng.randint(3, 120)]))
        set_grid(small)
        spawn()
    else:
        raise ValueError(path)


@pytest.mark.parametrize("n_a", [31, 129])
@pytest.mark.parametrize("path", ["set_grid", "set_grid_pose", "reset", "reset_envs", "smaller_after_larger"])
def test_metrics_and_strategies_follow_the_grid_each_env_holds(shapes, path, n_a):
    """Each way of installing grids: set_grid; set_grid_pose (the device evaluates the pose); the device reset and
    reset_envs on a subset (grids rebuilt from reset_info); set_grid with smaller grids after larger ones (cells beyond an
    env's n_g must not count).  Checked right after the installation and after a goal-seeking rollout."""
    E = 12
    rng = np.random.RandomState(100 + n_a)
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    sim = new_sim(E, n_a, r_avoid)
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    ob = oracle_batch(E, n_a, r_avoid, 0.4)
    install(sim, ob, path, rng, shapes)
    assert len({ob.params[e].n_g for e in range(E)}) > 1
    check_installed(sim, ob, r_avoid)
    rollout(sim, rng, 25)
    check_installed(sim, ob, r_avoid)
    assert ob.in_flags.sum() > 0


# ---------------------------------------------------------------------------------------------------------------------
# constructed edges of the metrics
FAR = [(-1.6, -1.6), (-1.6, 1.6), (1.6, -1.6), (1.6, 1.6), (0.0, 1.9)]      # agents 2.. sit on cells of their own here


def tie_env(g, p0, p1, owner, extra):
    """Agents 0 and 1 at p0, p1 near the cell g; three more cells behind the `owner` agent (on the ray from g through it,
    at 2, 3 and 4 times its offset: nearer to it than to anyone else); agents 2..6 on cells of their own far away, agent 2
    also owning `extra` cells next to its own (so that n_g differs between envs)."""
    po = (p0, p1)[owner]
    cells = [g] + [(g[0] + k * (po[0] - g[0]), g[1] + k * (po[1] - g[1])) for k in (2, 3, 4)] + FAR
    cells += [(FAR[0][0] + 0.01 * (j + 1), FAR[0][1]) for j in range(extra)]
    p = np.array([p0, p1] + FAR).T
    return p, np.array(cells).T


def check_tie_edge(sim, envs, r_avoid, other_counts):
    """Installs the tie envs and checks their construction: the counts the kernel must produce (the reference's) differ
    from `other_counts` of each env, and so does the statistic."""
    grids = [g for _, g in envs]
    for (p, g), other in zip(envs, other_counts):
        want = voronoi_counts(p, g)
        assert not np.array_equal(want, other) and ratio_in_kernel_order(want) != ratio_in_kernel_order(other)
    blocks, n_g = sim.pack_grids(grids, 16)
    sim.set_grid(blocks, n_g, [0.06] * len(envs))
    sim.set_state(np.stack([p for p, _ in envs]), np.zeros((len(envs), 2, 7)))
    check_metrics(sim, grids, r_avoid)


def rounded_tie_partner(g, x0, y0):
    """A position at a smaller squared distance from g than (x0, y0) whose square root rounds to the same double: the offset
    of (x0, y0) turned by 90 degrees, moved by up to 3 ulps per coordinate.  None if there is none."""
    s0 = sq(x0, y0, *g)
    bx, by = g[0] - (y0 - g[1]), g[1] + (x0 - g[0])
    for kx in range(-3, 4):
        for ky in range(-3, 4):
            x1, y1 = bx + kx * np.spacing(bx), by + ky * np.spacing(by)
            s1 = sq(x1, y1, *g)
            if s1 < s0 and np.sqrt(s1) == np.sqrt(s0):
                return x1, y1
    return None


def test_voronoi_count_takes_the_first_minimum_of_the_rounded_distances():
    """Agents 0 and 1 at different squared distances s0 > s1 from a cell whose square roots round to the same double: the
    reference's np.argmin of the norms gives the cell to agent 0.  Agent 0 (even envs) or agent 1 (odd envs) owns three
    more cells, so the choice changes the multiset of counts: (4, 0) against (3, 1), or (1, 3) against (0, 4)."""
    rng = np.random.RandomState(5)
    envs = []
    while len(envs) < 4:
        g = tuple(rng.uniform(-0.5, 0.5, 2))
        ang, r = rng.uniform(0, 2 * np.pi), 0.05 * rng.uniform(0.5, 1.0)
        x0, y0 = g[0] + r * np.cos(ang), g[1] + r * np.sin(ang)
        p1 = rounded_tie_partner(g, x0, y0)
        if p1 is not None:
            envs.append(tie_env(g, (x0, y0), p1, owner=len(envs) % 2, extra=len(envs)))
    sim = new_sim(4, 7, 0.26, n_g_max=16)
    check_tie_edge(sim, envs, 0.26, [voronoi_counts(p, g, rounded=False) for p, g in envs])


def test_voronoi_count_gives_an_exact_tie_to_the_lower_index():
    """Agents 0 and 1 at exactly the same squared distance from a cell (offsets (a, b) and (-b, a), all dyadic): the cell
    goes to agent 0.  Giving it to agent 1 would change the multiset of counts (see the rounded-tie test)."""
    envs, others = [], []
    for e, (g, a, b) in enumerate((((0.75, -0.5), 0.0625, 0.03125), ((-0.25, 0.375), 0.046875, -0.015625),
                                   ((0.125, 0.25), -0.03125, 0.0390625), ((-0.5, -0.125), 0.02734375, 0.0546875))):
        p0, p1 = (g[0] + a, g[1] + b), (g[0] - b, g[1] + a)
        assert sq(*p0, *g) == sq(*p1, *g)
        p, grid = tie_env(g, p0, p1, owner=e % 2, extra=e)
        other = voronoi_counts(p, grid)
        other[0] -= 1; other[1] += 1                              # the tied cell given to agent 1 instead
        envs.append((p, grid)); others.append(other)
    sim = new_sim(4, 7, 0.26, n_g_max=16)
    check_tie_edge(sim, envs, 0.26, others)


def test_coverage_radius_is_strict_at_the_last_double():
    """A cell counts as covered when an agent is strictly within r_avoid/2 (rounded norms).  With T the smallest double whose
    square root is >= r_avoid/2 (the kernel tests s < T), one agent per cell sits at squared distance exactly T (not
    covered), at the double below T (covered), and at the double above T, whose square root is r_avoid/2 exactly as well
    (not covered); the other cells have no agent near them."""
    r_avoid = 0.26
    h = r_avoid / 2
    T = thresh_lt(h)
    U = np.nextafter(T, np.inf)
    assert np.sqrt(np.nextafter(T, 0)) < h <= np.sqrt(T) and np.sqrt(U) == h
    rng = np.random.RandomState(3)
    cells = np.array([(-1.5, -1.5), (-1.5, 1.5), (1.5, -1.5), (1.5, 1.5), (0.37, -0.81)]).T
    targets = (T, np.nextafter(T, 0), U, T, U)
    E, n_a = 3, 7
    P = np.zeros((E, 2, n_a))
    for e in range(E):
        order = rng.permutation(5)                                # which cell gets which kind of agent
        for i in range(5):
            c = order[i]
            P[e][:, i] = at_squared_distance(rng, cells[0, c], cells[1, c], targets[i])
        P[e][:, 5:] = [[0.0, 0.1], [0.3, 0.4]]                    # far from every cell
        s = sq(P[e][0][None, :], P[e][1][None, :], cells[0][:, None], cells[1][:, None])
        assert sorted(s.min(axis=1)) == sorted(targets)
        covered = (np.sqrt(s) < h).any(axis=1)
        assert covered.sum() == 1 and ((s <= T).any(axis=1).sum() == 3)     # '<=' would cover two more cells
    sim = new_sim(E, n_a, r_avoid, n_g_max=16)
    blocks, n_g = sim.pack_grids([cells] * E, 16)
    sim.set_grid(blocks, n_g, [0.06] * E)
    sim.set_state(P, np.zeros_like(P))
    ref = check_metrics(sim, [cells] * E, r_avoid)
    assert (ref[:, 0] == 0.2).all()


def test_coincident_agents_are_not_each_others_nearest(shapes):
    """Agents at the same position are left out of each other's nearest distance (the reference keeps the norms != 0):
    pairs and triples of coincident agents, each with some other agent elsewhere."""
    rng = np.random.RandomState(8)
    E, n_a = 4, 9
    P = rng.uniform(-1.5, 1.5, (E, 2, n_a))
    for e in range(E):
        P[e][:, 1] = P[e][:, 0]
        P[e][:, 3:3 + 2 + e % 2] = P[e][:, [2]]
    grids = [posed_grid(rng, shapes, e) for e in range(E)]
    for e in range(E):
        pp = sq(P[e][0][None, :], P[e][1][None, :], P[e][0][:, None], P[e][1][:, None])
        assert (pp == 0).sum() > n_a and ((pp != 0).any(axis=1)).all()
    sim = new_sim(E, n_a, 0.3)
    blocks, n_g = sim.pack_grids(grids, NGM)
    sim.set_grid(blocks, n_g, [0.06] * E)
    sim.set_state(P, np.zeros_like(P))
    check_metrics(sim, grids, 0.3)


# ---------------------------------------------------------------------------------------------------------------------
def place_edge_agent(rng, grid, target):
    """A position whose nearest cell is a cell of `grid` at squared distance exactly `target` (0: on the cell).  The cell
    is the outermost one along a random direction u and the agent lies beyond it along u, so that cell is the unique
    nearest."""
    ang = rng.uniform(0, 2 * np.pi)
    c = int(np.argmax(grid[0] * np.cos(ang) + grid[1] * np.sin(ang)))
    if target == 0:
        return grid[0, c], grid[1, c]
    return at_squared_distance(rng, grid[0, c], grid[1, c], target, direction=ang)


@pytest.mark.parametrize("n_a", [1, 2, 31, 33, 100, 256, 257, 1024])
@pytest.mark.parametrize("d_sen", [0.4, 0.6])
def test_strategies_match_the_oracle_at_every_swarm_size(shapes, n_a, d_sen):
    """k_strategy runs min(round32(n_a), 256) threads per env, so from 257 agents on its agent loop takes several turns.
    Each env holds a different library shape.  The first state places, in turn over the envs, agents exactly on a cell
    (the 'llm' direction term is skipped at distance 0), exactly at the in-shape threshold T_in (squared distance T_in:
    not in the shape) and at the double below it (in the shape); a single agent has no neighbours.  Then a goal-seeking
    rollout.  d_sen = 0.6 comes with a small r_avoid: some agent keeps more than 80 sensed cells ('rule' takes the
    half-even subsample of them)."""
    E = 7 if n_a <= 100 else (3 if n_a <= 257 else 2)
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"]) if d_sen == 0.4 else 0.05
    rng = np.random.RandomState(17 + n_a)
    ks = rng.permutation(len(shapes["n_g"]))[:E]
    grids = [posed_grid(rng, shapes, k) for k in ks]
    l_cells = shapes["l_cell"][ks]
    spawn = [reset_like_reference(rng, n_a, shapes)[2:] for _ in range(E)]
    P, DP = np.stack([s[0] for s in spawn]), np.stack([s[1] for s in spawn])
    for e in range(E):
        T_in = thresh_lt(np.sqrt(2.0) * l_cells[e] / 2)           # in_flag: nearest norm < sqrt(2) l_cell / 2
        edges = (0.0, T_in, np.nextafter(T_in, 0))
        for i in range(min(n_a, 3)):
            target = edges[(i + e) % 3]
            P[e][:, i] = place_edge_agent(rng, grids[e], target)
            s = sq(P[e][0, i], P[e][1, i], grids[e][0], grids[e][1])
            assert s.min() == target and (np.sqrt(s.min()) < np.sqrt(2.0) * l_cells[e] / 2) == (target < T_in)
    sim = new_sim(E, n_a, r_avoid, d_sen=d_sen)
    blocks, n_g = sim.pack_grids(grids, NGM)
    sim.set_grid(blocks, n_g, l_cells)
    sim.set_state(P, DP)
    sim.observe()
    ob = oracle_batch(E, n_a, r_avoid, d_sen, grids, l_cells)
    in_shape, most_kept = 0, 0
    for t in (0, 15, 30):
        if t:
            rollout(sim, rng, 15)
        check_strategies(sim, ob)
        in_shape += int(ob.in_flags.sum())
        for e in range(E):
            d = np.sqrt(sq(ob.p[e][0][None, :], ob.p[e][1][None, :], grids[e][0][:, None], grids[e][1][:, None]))
            uncovered = ~(d <= r_avoid / 2).any(axis=1)          # kept by 'rule' for every agent that senses them
            most_kept = max(most_kept, int(((d < d_sen) & uncovered[:, None]).sum(axis=0).max()))
    assert in_shape > 0
    if d_sen == 0.6:
        assert most_kept > 80
