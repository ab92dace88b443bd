"""swarm_render (include/swarm_b200.h) against render_reference, its NumPy statement (marl_llm_b200/render.py): every pixel of
every frame bit for bit, over agent counts, frame sizes, views, layer subsets, trail rings, periodic wraps and the flocking
handle; env lists; no side effects on the simulator; guard zones; argument errors; the drop-in env's render("rgb_array")."""
import ctypes as C

import numpy as np
import pytest

from marl_llm_b200 import _lib
from marl_llm_b200.build import build_library
from marl_llm_b200.render import AGENT_IN, AGENT_OUT, AGENTS, CELLS, TRAILS, SwarmRenderer, palette, render_reference
from tests.helpers import load_shapes

ALL = CELLS | AGENTS | TRAILS
BEYOND_WALLS = (-3.5, 3.0, 2.9, -3.2)


def test_render_rejects_a_null_handle_without_a_gpu():
    build_library()
    lib = _lib.load()
    a = _lib.SwarmRenderArgs()
    a.struct_size = C.sizeof(_lib.SwarmRenderArgs)
    assert lib.swarm_render(None, C.byref(a), None) == _lib.SWARM_ERR_INVALID
    assert lib.swarm_render(None, None, None) == _lib.SWARM_ERR_INVALID
    assert b"null" in lib.swarm_last_error()
    pal = palette()
    assert pal.shape == (6, 3) and pal.dtype == np.uint8 and len({tuple(c) for c in pal}) == 6


# ------------------------------------------------------------------------------------------------------------------- helpers
def make_sim(E, n_a, seed=3, rule_steps=12, **kw):
    """E envs reset on the device from the library shapes, then `rule_steps` steps of the expert controller (agents move into the
    shapes, so both agent colours occur)."""
    import torch
    from marl_llm_b200.batched import BatchedAssemblySim, r_avoid_for
    sh = load_shapes()
    sim = BatchedAssemblySim(E, n_a, int(sh["n_g"].max()), r_avoid_for(n_a, sh["n_g"], sh["l_cell"]), **kw)
    sim.set_shapes(sh["grid_origin"], sh["l_cell"])
    sim.reset(seed=seed)
    for _ in range(rule_steps):
        sim.step(sim.strategy_actions("rule"))
    torch.cuda.synchronize()
    return sim


def arena(sim):
    return tuple(sim.cfg.boundary_pos)


def reference(sim, e, W, H, view=None, flags=ALL, trail=None):
    """render_reference for env e of an assembly handle, from the handle's own buffers"""
    bp = arena(sim)
    n_g = int(sim._n_g[e])
    return render_reference(W, H, bp if view is None else view, bp, sim.p[e].cpu().numpy(), sim.cfg.size_a,
                            in_flags=sim.in_flags[e].cpu().numpy(), cells=sim._grid[e, :n_g].cpu().numpy().T,
                            in_thresh=float(sim._in_thresh[e]), trail=trail, half=((bp[2] - bp[0]) / 2, (bp[1] - bp[3]) / 2),
                            flags=flags)


def assert_frame(got, want, what):
    got = got.cpu().numpy() if hasattr(got, "cpu") else got
    bad = np.any(got != want, axis=-1)
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} pixels differ, first at {np.argwhere(bad)[0]}"


def zoom_view(sim, e):
    """a view onto env e's shape, with some margin"""
    n_g = int(sim._n_g[e])
    g = sim._grid[e, :n_g].cpu().numpy()
    return (g[:, 0].min() - 0.1, g[:, 1].max() + 0.1, g[:, 0].max() + 0.1, g[:, 1].min() - 0.1)


def rendered(sim, ids, W, H, view=None, flags=ALL):
    r = SwarmRenderer(sim, ids, W, H, view=view)
    return r.render(cells=bool(flags & CELLS), agents=bool(flags & AGENTS), trails=bool(flags & TRAILS)).cpu().numpy()


# ------------------------------------------------------------------------------------------------------------- bit-exactness
@pytest.mark.gpu
@pytest.mark.parametrize("n_a", [1, 7, 30, 100, 1024])
def test_frames_equal_the_reference_for_library_resets(n_a):
    import torch
    E = 2 if n_a == 1024 else 3
    sim = make_sim(E, n_a, seed=10 + n_a)
    if n_a == 30:
        assert sim.fast_path == 2                      # device resets onto library shapes: the lookup-scan envs
    # trails: 15 recorded steps of the expert controller
    rend = SwarmRenderer(sim, np.arange(E), 97, 61, trail_len=15)
    samples = []
    for _ in range(15):
        sim.step(sim.strategy_actions("rule"))
        rend.record()
        samples.append(sim.p.cpu().numpy())
    samples = np.stack(samples)                        # [15, E, 2, n_a]
    flags_in = int(sim.in_flags.sum())
    assert n_a == 1 or 0 < flags_in, "the expert controller should bring some agents into their shapes"
    for W, H in [(97, 61), (480, 480)]:
        for view in [None, zoom_view(sim, 0), BEYOND_WALLS]:
            r = SwarmRenderer(sim, np.arange(E), W, H, view=view, trail_len=15)
            r.trail.copy_(rend.trail)
            r.trail_len, r.trail_head = rend.trail_len, rend.trail_head
            got = r.render().cpu().numpy()
            for e in range(E):
                assert_frame(got[e], reference(sim, e, W, H, view, trail=samples[:, e]), f"n_a {n_a}, {W}x{H}, view {view}, env {e}")
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (97, 61), (480, 480), (1024, 768)])
def test_frame_sizes(W, H):
    sim = make_sim(2, 30, seed=5)
    got = rendered(sim, [0, 1], W, H)
    for e in range(2):
        assert_frame(got[e], reference(sim, e, W, H), f"{W}x{H} env {e}")


@pytest.mark.gpu
def test_every_layer_subset():
    sim = make_sim(2, 30, seed=6)
    r = SwarmRenderer(sim, [1], 300, 200, trail_len=4)
    samples = []
    for _ in range(4):
        sim.step(sim.strategy_actions("rule"))
        r.record()
        samples.append(sim.p[1].cpu().numpy())
    frames = set()
    for flags in range(8):
        got = r.render(cells=bool(flags & CELLS), agents=bool(flags & AGENTS), trails=bool(flags & TRAILS)).cpu().numpy()
        assert_frame(got[0], reference(sim, 1, 300, 200, flags=flags, trail=np.stack(samples)), f"flags {flags}")
        frames.add(got.tobytes())
    assert len(frames) == 8, "every layer should change the frame"


@pytest.mark.gpu
def test_arbitrary_grids_from_set_grid():
    import torch
    rng = np.random.RandomState(4)
    sim = make_sim(3, 30, seed=8, rule_steps=0)
    grids = [rng.uniform(-2.6, 2.6, (2, n)) for n in (1, 57, sim.n_g_max)]      # scattered cells, one outside the arena
    blocks, n_g = sim.pack_grids(grids, sim.n_g_max)
    sim.set_grid(blocks, n_g, [0.05, 0.13, 0.2])
    sim.observe()
    torch.cuda.synchronize()
    assert sim.fast_path == 0
    for view in [None, BEYOND_WALLS]:
        got = rendered(sim, [0, 1, 2], 333, 257, view=view)
        for e in range(3):
            assert_frame(got[e], reference(sim, e, 333, 257, view), f"set_grid env {e}, view {view}")


@pytest.mark.gpu
@pytest.mark.parametrize("cap,n_rec", [(0, 0), (1, 3), (15, 0), (15, 1), (15, 5), (15, 15), (15, 40)])
def test_trail_ring(cap, n_rec):
    """trail_len 0 / 1 / 15, a partly filled ring and one whose head has wrapped (40 records into 15 slots)"""
    import torch
    sim = make_sim(2, 30, seed=9, rule_steps=0)
    r = SwarmRenderer(sim, [1, 0], 160, 160, trail_len=cap)
    act = torch.empty(2, 2, 30, dtype=torch.float32, device=sim.device)
    samples = []
    for t in range(n_rec):
        sim.fill_actions(act, seed=2, step=t)
        sim.step(act)
        r.record()
        samples.append(sim.p.cpu().numpy())
    L = min(cap, n_rec)
    assert r.trail_len == L
    got = r.render().cpu().numpy()
    for f, e in enumerate([1, 0]):
        tr = np.stack(samples[n_rec - L:])[:, e] if L else None
        assert_frame(got[f], reference(sim, e, 160, 160, trail=tr), f"cap {cap}, {n_rec} records, frame {f}")
    if L >= 2:
        r.clear()
        assert_frame(r.render().cpu().numpy()[0], reference(sim, 1, 160, 160), "cleared trail")


@pytest.mark.gpu
def test_periodic_wraps_are_not_drawn():
    import torch
    sim = make_sim(2, 30, seed=12, rule_steps=0, is_periodic=True)
    rng = np.random.RandomState(0)
    p = np.stack([np.stack([rng.uniform(2.0, 2.4, 30), rng.uniform(-2.4, 2.4, 30)])] * 2)
    dp = np.zeros_like(p)
    dp[:, 0], dp[:, 1] = 0.8, 0.3
    sim.set_state(p, dp)
    act = torch.zeros(2, 2, 30, dtype=torch.float32, device=sim.device)
    act[:, 0], act[:, 1] = 1.0, 0.4
    r = SwarmRenderer(sim, [0, 1], 256, 256, trail_len=12)
    samples = []
    for _ in range(12):
        sim.step(act)
        r.record()
        samples.append(sim.p.cpu().numpy())
    s = np.stack(samples)
    assert (np.abs(np.diff(s[:, 0, 0], axis=0)) > 2.4).any(), "no agent crossed the border"
    got = r.render().cpu().numpy()
    bp = arena(sim)
    for e in range(2):
        want = reference(sim, e, 256, 256, trail=s[:, e])
        assert_frame(got[e], want, f"periodic env {e}")
        n_g = int(sim._n_g[e])
        drawn = render_reference(256, 256, bp, bp, sim.p[e].cpu().numpy(), sim.cfg.size_a, in_flags=sim.in_flags[e].cpu().numpy(),
                                 cells=sim._grid[e, :n_g].cpu().numpy().T, in_thresh=float(sim._in_thresh[e]), trail=s[:, e])
        assert not np.array_equal(drawn, want), "drawing the wrapped segments should change the frame"


@pytest.mark.gpu
def test_flocking_handle():
    import torch
    from marl_llm_b200.flocking import BatchedFlockingSim
    sim = BatchedFlockingSim(3, 40)
    sim.reset(seed=1)
    r = SwarmRenderer(sim, [2, 0], 200, 150, trail_len=6)
    act = torch.empty(3, 2, 40, dtype=torch.float32, device=sim.device)
    samples = []
    for t in range(8):
        act.uniform_(-1, 1)
        sim.step(act)
        r.record()
        samples.append(sim.p.cpu().numpy())
    sim.in_flags.fill_(1)                         # a flocking handle has no shape: the flags must not colour its agents
    got = r.render().cpu().numpy()
    bp = (-2.4, 2.4, 2.4, -2.4)
    for f, e in enumerate([2, 0]):
        want = render_reference(200, 150, bp, bp, sim.p[e].cpu().numpy(), 0.035, trail=np.stack(samples[-6:])[:, e], half=(2.4, 2.4))
        assert_frame(got[f], want, f"flocking frame {f}")


@pytest.mark.gpu
def test_overlapping_agents_largest_index_wins():
    """agents 0..5 of env 1 in a tight cluster with alternating in-shape flags: where discs overlap, the largest index shows"""
    import torch
    sim = make_sim(2, 30, seed=18, rule_steps=0)
    p = sim.p.cpu().numpy()
    p[1, :, :6] = np.array([[0.0, 0.02, 0.04, 0.0, 0.02, 0.04], [0.0, 0.0, 0.0, 0.02, 0.02, 0.02]]) + 0.3
    sim.set_state(p, sim.dp.cpu().numpy())
    sim.in_flags[1, :6] = torch.tensor([1, 0, 1, 0, 1, 0], dtype=torch.int32, device=sim.device)
    view = (0.2, 0.45, 0.45, 0.2)
    got = rendered(sim, [1], 250, 250, view=view)[0]
    assert_frame(got, reference(sim, 1, 250, 250, view), "overlapping agents")
    pal = palette()
    # pixel (row, col) of a point: X = 0.2 + (c + 0.5) * 0.001, Y = 0.45 - (r + 0.5) * 0.001
    assert np.array_equal(got[130, 110], pal[AGENT_OUT])      # (0.31, 0.32): covered by agents 0, 1, 3, 4 and 5
    assert np.array_equal(got[149, 89], pal[AGENT_OUT])       # (0.29, 0.30): agents 0, 1 and 3 -> 3, outside
    assert np.array_equal(got[150, 109], pal[AGENT_IN])       # (0.31, 0.30): agents 0..4 -> 4, inside


# ------------------------------------------------------------------------------------------------------------------ env lists
@pytest.mark.gpu
def test_env_lists_permute_and_repeat():
    sim = make_sim(5, 30, seed=13)
    base = rendered(sim, np.arange(5), 120, 90)
    perm = [3, 0, 4, 1, 2]
    assert np.array_equal(rendered(sim, perm, 120, 90), base[perm])
    dup = rendered(sim, [2, 2, 4, 2], 120, 90)
    assert np.array_equal(dup, base[[2, 2, 4, 2]])
    assert len({base[e].tobytes() for e in range(5)}) == 5


@pytest.mark.gpu
def test_more_frames_than_one_launch_carries():
    """2048 env ids travel with one launch: 2050 frames take two, and the second launch draws the right envs"""
    sim = make_sim(7, 7, seed=14, rule_steps=2)
    ids = (np.arange(2050) * 5) % 7
    base = rendered(sim, np.arange(7), 16, 12)
    before = sim.launch_count
    got = rendered(sim, ids, 16, 12)
    assert sim.launch_count - before == 2
    assert np.array_equal(got, base[ids])


# ------------------------------------------------------------------------------------------------------------ no side effects
def sim_buffers(sim):
    names = ["p", "dp", "_grid", "_n_g", "_in_thresh", "_word_box", "_frame", "nearest_cell", "obs", "reward", "done",
             "neighbor_index", "in_flags", "sensed_index", "occupied_index"]
    out = {n: getattr(sim, n).clone() for n in names}
    out["a_prior0"], out["a_prior1"] = sim._a_prior[0].clone(), sim._a_prior[1].clone()
    return out


@pytest.mark.gpu
def test_rendering_has_no_side_effects():
    import torch
    sims = [make_sim(4, 30, seed=15, rule_steps=3, emit_indices=True, out_dtype=torch.float64, guard_bytes=4096) for _ in range(2)]
    a, b = sims
    r = SwarmRenderer(a, [0, 3, 1], 200, 200, trail_len=5)
    act = torch.empty(4, 2, 30, dtype=torch.float32, device=a.device)
    for t in range(20):
        before, launches = sim_buffers(a), a.launch_count
        r.record()
        r.render()
        assert a.launch_count - launches == 1
        for k, v in sim_buffers(a).items():
            assert torch.equal(v, before[k]), f"render changed {k}"
        for s in sims:
            s.fill_actions(act, seed=4, step=t)
            s.step(act)
        twin = sim_buffers(b)
        for k, v in sim_buffers(a).items():
            assert torch.equal(v, twin[k]), f"step {t}: {k} differs from the twin that never rendered"
    assert a.check_guards()


# ------------------------------------------------------------------------------------------------------------ memory safety
def guarded(nbytes, device, gb=4096):
    import torch
    raw = torch.full((gb + nbytes + gb,), 0xA5, dtype=torch.uint8, device=device)
    return raw, raw[gb:gb + nbytes]


def raw_render(sim, ids, W, H, frames_ptr, flags=ALL, view=(0.0, 0.0, 0.0, 0.0), trail=0, cap=0, tlen=0, head=0, **over):
    ids = np.ascontiguousarray(ids, dtype=np.int32)
    a = _lib.SwarmRenderArgs()
    a.struct_size = C.sizeof(_lib.SwarmRenderArgs)
    a.width, a.height, a.flags, a.count, a.env_ids = W, H, flags, ids.shape[0], ids.ctypes.data
    a.view[:] = view
    a.trail, a.trail_cap, a.trail_len, a.trail_head, a.frames = trail, cap, tlen, head, frames_ptr
    for k, v in over.items():
        setattr(a, k, v)
    return sim.lib.swarm_render(sim._h, C.byref(a), sim._stream())


@pytest.mark.gpu
@pytest.mark.parametrize("W,H", [(1, 1), (97, 61), (33, 65)])
def test_frames_write_exactly_their_bytes(W, H):
    import torch
    sim = make_sim(3, 30, seed=16, guard_bytes=4096)
    ids = [2, 0]
    n = len(ids) * H * W * 3
    raw, frames = guarded(n, sim.device)
    frames.fill_(1)                                       # 1 is no palette value: every byte must be overwritten
    cap = 6
    traw, trail = guarded(cap * len(ids) * 2 * 30 * 8, sim.device)
    ring = trail.view(torch.float64).view(cap, len(ids), 2, 30)
    samples = []
    for k in range(cap):
        sim.step(sim.strategy_actions("rule"))
        ring[k].copy_(sim.p[torch.tensor(ids, device=sim.device)])
        samples.append(sim.p.cpu().numpy())
    assert raw_render(sim, ids, W, H, frames.data_ptr(), trail=trail.data_ptr(), cap=cap, tlen=cap, head=cap - 1) == 0
    got = frames.view(len(ids), H, W, 3).cpu().numpy()
    for f, e in enumerate(ids):
        assert_frame(got[f], reference(sim, e, W, H, trail=np.stack(samples)[:, e]), f"{W}x{H} frame {f}")
    for g in (raw, traw):
        assert bool((g[:4096] == 0xA5).all()) and bool((g[-4096:] == 0xA5).all()), "guard zone overwritten"
    assert sim.check_guards()


# ------------------------------------------------------------------------------------------------------------ argument errors
@pytest.mark.gpu
def test_invalid_arguments_are_rejected_before_any_launch():
    import torch
    sim = make_sim(3, 30, seed=17, rule_steps=0)
    frames = torch.full((2 * 8 * 8 * 3,), 7, dtype=torch.uint8, device=sim.device)
    trail = torch.zeros(4, 2, 2, 30, dtype=torch.float64, device=sim.device)
    F, T = frames.data_ptr(), trail.data_ptr()
    nan, inf = float("nan"), float("inf")
    cases = {
        "struct_size": dict(struct_size=8),
        "width 0": dict(W=0), "width 8193": dict(W=8193), "height 0": dict(H=0), "height 8193": dict(H=8193),
        "count 0": dict(count=0), "env_ids NULL": dict(env_ids=None), "env -1": dict(ids=[0, -1]), "env E": dict(ids=[3, 0]),
        "unknown flag": dict(flags=8),
        "view nan": dict(view=(nan, 1, 1, -1)), "view inf": dict(view=(-1, inf, 1, -1)), "xmin = xmax": dict(view=(1, 1, 1, -1)),
        "xmin > xmax": dict(view=(2, 1, 1, -1)), "ymin = ymax": dict(view=(-1, 1, 1, 1)), "ymin > ymax": dict(view=(-1, 1, 1, 2)),
        "trail_len < 0": dict(trail=T, cap=4, tlen=-1), "trail_len > cap": dict(trail=T, cap=4, tlen=5),
        "cap > 1024": dict(trail=T, cap=1025, tlen=2), "trail NULL": dict(trail=0, cap=4, tlen=2),
        "head < 0": dict(trail=T, cap=4, tlen=2, head=-1), "head = cap": dict(trail=T, cap=4, tlen=2, head=4),
        "frames NULL": dict(frames=0),
    }
    before = sim.launch_count
    for what, kw in cases.items():
        kw = dict(kw)
        ids = kw.pop("ids", [0, 2])
        W, H, fr = kw.pop("W", 8), kw.pop("H", 8), kw.pop("frames", F)
        rc = raw_render(sim, ids, W, H, fr, **kw)
        assert rc == _lib.SWARM_ERR_INVALID, f"{what}: rc {rc}"
    torch.cuda.synchronize()
    assert sim.launch_count == before
    assert bool((frames == 7).all()), "a rejected call wrote frames"
    assert raw_render(sim, [0, 2], 8, 8, F, trail=T, cap=4, tlen=4, head=3) == 0       # the baseline of the cases is valid
    assert sim.launch_count == before + 1


# ------------------------------------------------------------------------------------------------------------- drop-in env
def env_args(n_a, **kw):
    import argparse
    sh = load_shapes()
    d = dict(n_a=n_a, is_boundary=True, is_con_self_state=True, is_feature_norm=False, dynamics_mode="Cartesian",
             render_traj=False, traj_len=15, agent_strategy="input", training_method="llm_rl", is_collected=False, video=False,
             results_file={"l_cell": [float(v) for v in sh["l_cell"]], "grid_coords": [np.ascontiguousarray(g.T) for g in sh["grid_origin"]],
                           "shape_bound_points": [np.zeros(4) for _ in sh["l_cell"]]})
    d.update(kw)
    return argparse.Namespace(**d)


@pytest.mark.gpu
def test_dropin_env_rgb_array():
    from marl_llm_b200.assembly_env import AssemblySwarmEnv, AssemblySwarmWrapper
    np.random.seed(3)
    env = AssemblySwarmWrapper(AssemblySwarmEnv(), env_args(30))
    env.reset()
    for _ in range(5):
        env.step(np.random.uniform(-1, 1, (2, 30)))
    assert env.render() is None and env.render("human") is None
    frame = env.render("rgb_array")
    assert isinstance(frame, np.ndarray) and frame.shape == (480, 480, 3) and frame.dtype == np.uint8
    sim = env.env._sim
    assert np.array_equal(frame, SwarmRenderer(sim, [0], 480, 480).render().cpu().numpy()[0])
    assert_frame(frame, reference(sim, 0, 480, 480), "drop-in frame")
    env.close()


@pytest.mark.gpu
def test_dropin_env_trails():
    from marl_llm_b200.assembly_env import AssemblySwarmEnv, AssemblySwarmWrapper
    np.random.seed(4)
    env = AssemblySwarmWrapper(AssemblySwarmEnv(), env_args(30, render_traj=True, traj_len=15))
    env.reset()
    samples = [env.p]
    sim = env.env._sim
    for _ in range(22):
        env.step(np.random.uniform(-1, 1, (2, 30)))
        samples.append(env.p)
    frame = env.render("rgb_array")
    assert_frame(frame, reference(sim, 0, 480, 480, trail=np.stack(samples[-15:])), "15 newest samples")
    assert not np.array_equal(frame, reference(sim, 0, 480, 480, trail=np.stack(samples[-16:])))
    env.reset()
    assert_frame(env.render("rgb_array"), reference(env.env._sim, 0, 480, 480, flags=CELLS | AGENTS), "trail after reset()")
    env.close()


@pytest.mark.gpu
def test_dropin_env_vectorised():
    from marl_llm_b200.assembly_env import AssemblySwarmEnv, AssemblySwarmWrapper
    np.random.seed(5)
    env = AssemblySwarmWrapper(AssemblySwarmEnv(num_envs=4), env_args(30))
    env.reset()
    env.step(np.random.uniform(-1, 1, (4, 2, 30)))
    frames = env.render("rgb_array")
    assert frames.shape == (4, 480, 480, 3) and frames.dtype == np.uint8
    for e in range(4):
        assert_frame(frames[e], reference(env.env._sim, e, 480, 480), f"env {e}")
    env.close()

