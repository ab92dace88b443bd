#!/usr/bin/env python
"""bench.py — agent-steps/s of the assembly-env step() hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's fused sm_100a kernel
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path, all host cores
    python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed (sampled envs, .npy)

A "step" = one env.step() of every env of the batch: 30 agents x 65 536 envs per GPU (BASELINE config 3; at N=1
it is the single-GPU instance of the configuration the metric is quoted on).  Envs are independent, so N GPUs run N
shards with no data-path collective ("weak" scaling: per-GPU work is fixed); the only exchange is the max-over-ranks
of the elapsed time.  One JSON line is printed by rank 0.

    value     device-resident throughput: actions already in HBM, CUDA events around exactly K steps
    e2e       same metric through the host-buffer C-ABI call (swarm_step_host): pinned host actions H2D, step,
              obs + reward + a_prior D2H, every step, inside the timed region
    roofline  algorithmic bytes per launch (DESIGN.md §4) / mean launch duration vs the measured HBM copy peak
    cpu_baseline  the reference's C++ (oracle/_ref) + NumPy glue timed on this box's host cores (rank 0, N=1)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

METRIC = "agent_steps_per_sec"
UNIT = "agent-steps/s"


def load_shapes():
    z = np.load(os.path.join(REPO, "tests", "golden", "shapes.npz"))
    n_g = z["n_g"]
    return dict(l_cell=z["l_cell"].copy(), n_g=n_g.copy(),
                grid_origin=[np.ascontiguousarray(z["grid_coords"][k, :n_g[k]].T) for k in range(len(n_g))])


def synth_batch(E, n_a, shapes, seed, regime, with_pose=False):
    """Vectorised domain randomisation in the spirit of assembly.py:156-223 (shape, rotation, offset, initial p/dp).
    regime 'random': the reference's reset distribution.  'converged': agents start on cells of their shape so the
    in-shape / occupancy / subsample / reward branches are the common case."""
    rng = np.random.RandomState(seed)
    S = len(shapes["l_cell"])
    ngm = int(shapes["n_g"].max())
    k = rng.randint(0, S, E)
    ang = np.pi * rng.uniform(-1, 1, E)
    off = rng.uniform(-1.4, 1.4, (E, 2))
    blocks = np.zeros((E, 2 * ngm))
    n_g = shapes["n_g"][k].astype(np.int32)
    l_cell = shapes["l_cell"][k]
    c, s = np.cos(ang), np.sin(ang)
    p = np.empty((E, 2, n_a))
    for sid in range(S):
        sel = np.nonzero(k == sid)[0]
        if sel.size == 0:
            continue
        g = shapes["grid_origin"][sid]                         # [2, ng]
        ng = g.shape[1]
        gx = c[sel, None] * g[0][None] + s[sel, None] * g[1][None] + off[sel, 0:1]
        gy = -s[sel, None] * g[0][None] + c[sel, None] * g[1][None] + off[sel, 1:2]
        blocks[sel, :ng] = gx
        blocks[sel, ng:2 * ng] = gy
        if regime == "converged":
            pick = np.stack([rng.choice(ng, n_a, replace=n_a > ng) for _ in sel])
            p[sel, 0] = np.take_along_axis(gx, pick, 1) + rng.normal(0, 0.01, pick.shape)
            p[sel, 1] = np.take_along_axis(gy, pick, 1) + rng.normal(0, 0.01, pick.shape)
    if regime != "converged":
        wide = rng.uniform(-1, 1, E) > 0
        p_wide = rng.uniform(-2.4, 2.4, (E, 2, n_a))
        p_clu = rng.uniform(-1, 1, (E, 2, n_a)) + rng.uniform(-1.4, 1.4, (E, 2, 1))
        p = np.where(wide[:, None, None], p_wide, p_clu)
        dp = rng.uniform(-0.5, 0.5, (E, 2, n_a))
    else:
        dp = rng.uniform(-0.05, 0.05, (E, 2, n_a))
    if with_pose:      # (shape, cos, sin, off_x, off_y) per env: the grids above are exactly grid_from_pose of these
        return blocks, n_g, l_cell, p, dp, (k.astype(np.int32), c, s, off[:, 0].copy(), off[:, 1].copy())
    return blocks, n_g, l_cell, p, dp


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._stop_evt = gpu_index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


DUMP_BYTES = 60 * 10**6     # all files of one --dump-outputs run, below 64 MB with the .npy headers


def dump_outputs(out_dir, tag, arrays, budget):
    """Writes the [E, ...] device arrays of `arrays` as <out_dir>/<tag>_<name>.npy so that two builds can be compared output for
    output: the same seeded sample of envs for every array (as many as `budget` bytes allow), float64 arrays as float64, all
    others (integer and bool ones too: their values are exact there) as float32."""
    import torch
    arrays = {k: v for k, v in arrays.items() if v is not None}
    E = next(iter(arrays.values())).shape[0]
    per_env = sum(t[0].numel() * (8 if t.dtype == torch.float64 else 4) for t in arrays.values())
    n = max(1, min(E, budget // per_env))
    pick = np.sort(np.random.RandomState(0).choice(E, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.index_select(0, torch.as_tensor(pick, device=t.device)).cpu().numpy()
        np.save(os.path.join(out_dir, f"{tag}_{name}.npy"), a.astype(np.float64 if a.dtype == np.float64 else np.float32))


def measured_hbm_peak():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------
def reference_arm(args, rank, world):
    """The reference's CPU implementation of the path on this box's host cores (rank 0 only)."""
    if rank != 0:
        return
    from oracle import ref_glue
    shapes = load_shapes()
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, args.ref_procs or cores))
    K = args.steps                          # env.step() calls per env inside the timed region
    if not ref_glue.available():
        # the reference C++ was not compiled here: fall back to the C port of it (never to the product)
        from oracle import oracle as orc
        res = port_rollouts(orc, shapes, args.n_a, procs, args.ref_envs, K)
        kind, sample = "port", f"{res['envs']} envs x {K} steps, oracle C port, {procs} OpenMP threads"
    else:
        for _ in range(max(0, min(args.warmup, 1))):
            ref_glue.timed_rollouts(args.n_a, shapes, procs, 1, 20)
        res = ref_glue.timed_rollouts(args.n_a, shapes, procs, 1, K)
        kind = "reference"
        sample = (f"{procs} processes x {K} steps x {args.n_a} agents, one env each "
                  f"(reference AssemblyEnv.cpp via oracle/_ref + its NumPy glue), env.step() time only")
    value, secs = res["value"], res["seconds"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"assembly env, {args.n_a} agents, reference CPU path (single env per process; the reference has no vector env)",
                   "n_a": args.n_a, "processes": procs},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def port_rollouts(orc, shapes, n_a, threads, envs, steps):
    r_avoid = orc.r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    blocks, n_g, l_cell, p, dp = synth_batch(envs, n_a, shapes, 226, "random")
    params = [orc.make_params(n_a, int(n_g[e]), float(l_cell[e]), r_avoid) for e in range(envs)]
    ob = orc.OracleBatch(params, nthreads=threads, ng_max=int(shapes["n_g"].max()))
    ob.grid[:] = 0
    for e in range(envs):
        ob.grid[e, :2 * n_g[e]] = blocks[e, :2 * n_g[e]]
    ob.p[:], ob.dp[:] = p, dp
    ob.observe()
    acts = [orc.fill_actions(envs, n_a, 226, t) for t in range(steps)]
    t0 = time.perf_counter()
    for t in range(steps):
        ob.step(acts[t])
    dt = time.perf_counter() - t0
    return dict(value=envs * steps * n_a / dt, envs=envs, seconds=dt)


def widened_path_numbers(torch, sim, act, hbm_peak, shapes):
    """Device-timed numbers of the rows built next to the step path (DESIGN.md §9): k_rollout_push against the HBM roofline,
    the policy MLP (fp32 exact path and tcgen05 fp16 path), and the rollout loop policy -> step -> push with nothing on the host."""
    import torch.nn as nn
    from marl_llm_b200.policy import DevicePolicy
    from marl_llm_b200.rollout import ReplayBufferAgent
    E, n_a, D, A, H = sim.E, sim.n_a, sim.obs_dim, 2, 180

    def timed(fn, k):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k):
            fn()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / k

    torch.manual_seed(0)
    sd = {}
    for name, (o, i) in (("fc1", (H, D)), ("fc2", (H, H)), ("fc3", (H, H)), ("fc4", (A, H))):
        lin = nn.Linear(i, o); sd[name + ".weight"] = lin.weight; sd[name + ".bias"] = lin.bias
    pol = DevicePolicy(D, A, H, noise_scale=0.5).load_state_dict(sd)
    buf = ReplayBufferAgent(4, E * n_a, slice(0, n_a), D, A)
    obs_prev, act2 = sim.obs.clone(), torch.empty_like(act)
    obs_pair = [sim.obs, torch.empty_like(sim.obs)]
    idx = slice(0, n_a)
    rows = E * n_a
    push_ms = timed(lambda: buf.push(obs_prev, act, sim.reward, sim.obs, sim.done, idx, sim.a_prior), 10)
    push_bytes = rows * (2 * D * 4 * 2 + 2 * A * 4 * 2 + 4 * 2 + 1 + 4)
    pol_fp32_ms = timed(lambda: pol.step(obs_prev, explore=True, out=act2, want_log_pi=False), 3)
    pol.set_precision("f16x3_tc")
    pol_tc3_ms = timed(lambda: pol.step(obs_prev, explore=True, out=act2, want_log_pi=False), 20)
    pol.set_precision("f16_tc")
    pol_tc_ms = timed(lambda: pol.step(obs_prev, explore=True, out=act2, want_log_pi=False), 20)

    def loop_step():                       # the simulator's obs output alternates between two buffers: no copy
        prev, spare = obs_pair
        _, lp = pol.step(prev, explore=True, out=act2)
        sim.set_obs_buffer(spare)
        nxt, rew, done, _, prior = sim.step(act2)
        buf.push(prev, act2, rew, nxt, done, idx, prior, lp)
        obs_pair[0], obs_pair[1] = spare, prev
    loop_ms = timed(loop_step, 20)

    from marl_llm_b200.episode_ring import EpisodeRing
    del buf
    ring = EpisodeRing(4, E, n_a, D, A)
    state = {"t": 0}

    def ring_step():                       # time-indexed ring: the policy kernel writes the replay rows, only small arrays are pushed
        prev, spare = obs_pair
        if state["t"] == ring.T:
            ring.begin(); state["t"] = 0
        _, lp = pol.step(prev, explore=True, out=act2, rows_out=ring.slot(state["t"]))
        sim.set_obs_buffer(spare)
        nxt, rew, done, _, prior = sim.step(act2)
        ring.record(state["t"], act2, rew, done, prior, lp)
        state["t"] += 1
        obs_pair[0], obs_pair[1] = spare, prev
    ring_ms = timed(ring_step, 20)
    # the same loop with an agent-major simulator writing straight into the ring slots (no observation copy at all)
    direct_ms = None
    try:
        from marl_llm_b200.batched import BatchedAssemblySim
        del ring
        sim2 = BatchedAssemblySim(E, n_a, sim.n_g_max, sim.r_avoid, device=sim.device.index, obs_layout="agent_major")
        sim2.set_shapes(shapes["grid_origin"], shapes["l_cell"])
        sim2.reset(seed=226)
        ring2 = EpisodeRing(8, E, n_a, D, A)      # the wrap copies slot T back to slot 0: once per 8 steps, inside the timed loop
        ring2.begin_direct(sim2)
        st2 = {"t": 0}

        def direct_step():
            if st2["t"] == ring2.T:
                ring2.slot_env(0).copy_(ring2.slot_env(ring2.T)); sim2.set_obs_buffer(ring2.slot_env(0)); ring2.begin(); st2["t"] = 0
            t = st2["t"]
            _, lp = pol.step(ring2.slot_env(t), explore=True, out=act2, agent_major=True)
            sim2.set_obs_buffer(ring2.slot_env(t + 1))
            _, rew, done, _, prior = sim2.step(act2)
            ring2.record(t, act2, rew, done, prior, lp)
            st2["t"] = t + 1
        direct_ms = timed(direct_step, 20)
        pol_am_ms = timed(lambda: pol.step(ring2.slot_env(0), explore=True, out=act2, want_log_pi=False, agent_major=True), 20)
        step_am_ms = timed(lambda: sim2.step(act2), 20)
        del sim2, ring2
    except Exception as ex:
        direct_ms = None; pol_am_ms = step_am_ms = None
        direct_err = f"{type(ex).__name__}: {ex}"
    flop = 2.0 * rows * (D * H + 2 * H * H + H * A)
    return {
        "rollout_push": {"kernel": "swarm::k_rollout_push_tma", "ms": push_ms, "GBps": push_bytes / push_ms / 1e6,
                         "frac_of_hbm_peak": push_bytes / push_ms / 1e6 / hbm_peak, "rows": rows},
        "policy_fp32": {"kernel": "swarm::k_policy_mlp", "ms": pol_fp32_ms, "TFLOPs": flop / pol_fp32_ms / 1e9},
        "policy_f16x3_tc": {"kernel": "swarm::k_policy_mlp_tc3 (tcgen05, fp16 hi/lo split, fp32-accurate)", "ms": pol_tc3_ms,
                            "TFLOPs_useful": flop / pol_tc3_ms / 1e9, "TFLOPs_issued": 3 * flop / pol_tc3_ms / 1e9},
        "policy_f16_tc": {"kernel": "swarm::k_policy_mlp_tc (tcgen05, TMEM)", "ms": pol_tc_ms, "TFLOPs": flop / pol_tc_ms / 1e9},
        "device_rollout_loop": {"stages": "policy(f16_tc) -> step -> push, obs double-buffered", "ms_per_step": loop_ms,
                                "agent_steps_per_s": rows / loop_ms * 1e3},
        "device_rollout_loop_ring": {"stages": "policy(f16_tc, writes the replay rows) -> step -> small-array push (time-indexed ring)",
                                     "ms_per_step": ring_ms, "agent_steps_per_s": rows / ring_ms * 1e3},
        "device_rollout_loop_direct": ({"stages": "agent-major simulator writes obs straight into the ring slot; policy(f16_tc) reads contiguous rows; small-array push",
                                        "ms_per_step": direct_ms, "agent_steps_per_s": rows / direct_ms * 1e3,
                                        "policy_f16_tc_ms": pol_am_ms, "policy_TFLOPs": flop / pol_am_ms / 1e9, "step_ms": step_am_ms}
                                       if direct_ms else {"error": direct_err}),
    }


def flocking_line(args, torch, rank, world, local_rank, barrier, max_over_ranks):
    """BASELINE config 5 (flocking): the variant specified in VARIANTS.md on the shared pair core.  HBM roofline with its own
    algorithmic bytes: action 8 + p/dp read + write 64 + obs 28 x 4 + reward 4 + neighbor_index 24 = 212 B per agent-step."""
    from marl_llm_b200.flocking import BatchedFlockingSim
    E, n_a, K, W = args.envs_per_gpu, min(args.n_a, 128), args.steps, args.warmup
    sim = BatchedFlockingSim(E, n_a, device=local_rank)
    sim.reset(seed=226 + rank)
    g = torch.Generator(device="cuda").manual_seed(rank)
    acts = torch.rand(16, E, 2, n_a, device="cuda", generator=g) * 2 - 1
    for t in range(max(W, 3)):
        sim.step(acts[t % 16])
    barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for t in range(K):
        sim.step(acts[t % 16])
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1), device="cuda")
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "flocking", dict(obs=sim.obs, reward=sim.reward, done=sim.done, p=sim.p, dp=sim.dp), DUMP_BYTES)
    peak, peak_src = measured_hbm_peak()
    b = 8 + 64 + sim.obs_dim * 4 + 4 + 24
    achieved = b * E * n_a / (ms / K * 1e-3) / 1e9
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": world * E * n_a * K / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"flocking variant (VARIANTS.md 3; no reference source: parity unpinned), {n_a} agents x {E} envs per GPU (BASELINE config 5)",
                       "n_a": n_a, "envs_per_gpu": E, "actions": "U(-1,1), ring of 16 device buffers", "l2": "working set per step >> 126 MB L2"},
            "clocks": clocks, "gpu_launches": 2 * K, "e2e": None, "cpu_baseline": None,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_agent_step": b,
                         "kernel": "swarm::k_step<PH=1> (shared with the assembly env) + swarm::k_flock_reward"}}), flush=True)


def predator_prey_line(args, torch, rank, world, local_rank, barrier, max_over_ranks):
    """BASELINE config 5 (predator-prey): the variant specified in VARIANTS.md 4, 1/4 pursuers.  HBM roofline with its own algorithmic
    bytes: action 8 + p/dp read + write 64 + obs 52 x 4 + reward 4 + neighbor_index 48 = 332 B per agent-step."""
    from marl_llm_b200.predator_prey import BatchedPredatorPreySim
    E, n, K, W = args.envs_per_gpu, min(args.n_a, 128), args.steps, args.warmup
    n_p = max(1, n // 4)
    sim = BatchedPredatorPreySim(E, n_p, n - n_p, device=local_rank)
    sim.reset(seed=226 + rank)
    g = torch.Generator(device="cuda").manual_seed(rank)
    acts = torch.rand(16, E, 2, n, device="cuda", generator=g) * 2 - 1
    for t in range(max(W, 3)):
        sim.step(acts[t % 16])
    barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for t in range(K):
        sim.step(acts[t % 16])
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1), device="cuda")
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "predator_prey", dict(obs=sim.obs, reward=sim.reward, done=sim.done, p=sim.p, dp=sim.dp),
                     DUMP_BYTES)
    peak, peak_src = measured_hbm_peak()
    b = 8 + 64 + sim.obs_dim * 4 + 4 + 48
    achieved = b * E * n / (ms / K * 1e-3) / 1e9
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": world * E * n * K / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"predator-prey variant (VARIANTS.md 4; no reference source: parity unpinned), {n_p} pursuers + {n - n_p} escapers x {E} envs per GPU (BASELINE config 5)",
                       "n_a": n, "envs_per_gpu": E, "actions": "U(-1,1) for both types, ring of 16 device buffers", "l2": "working set per step >> 126 MB L2"},
            "clocks": clocks, "gpu_launches": K, "e2e": None, "cpu_baseline": None,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_agent_step": b, "kernel": "swarm::k_pp_step"}}), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--n-a", dest="n_a", type=int, default=30)
    ap.add_argument("--layout", default="production", choices=["production", "parity"],
                    help="production: fp64 state, fp32 obs/reward/prior; parity: everything fp64 + index arrays")
    ap.add_argument("--regime", default="both", choices=["both", "random", "converged"],
                    help="headline = the first regime run (random: U(-1,1) actions, staggered 200-step episodes with auto-reset)")
    ap.add_argument("--episode-length", type=int, default=200, help="CFG:181")
    ap.add_argument("--reset-cohorts", type=int, default=25, help="envs are auto-reset in this many staggered cohorts (<= episode length)")
    ap.add_argument("--brute-force-scan", action="store_true", help="A/B: disable the word-box culling of the grid scan")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the rollout-storage / policy / device-loop measurements")
    ap.add_argument("--variant", default="assembly", choices=["assembly", "flocking", "predator_prey"],
                    help="flocking / predator_prey: the variants specified in VARIANTS.md (BASELINE config 5; no reference source, no CPU baseline)")
    ap.add_argument("--ref-procs", type=int, default=0)
    ap.add_argument("--ref-envs", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of each regime, write what its last step computed (rank 0's envs; a fixed, seeded "
                         "sample of them) as DIR/<regime or variant>_<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from marl_llm_b200.batched import BatchedAssemblySim, r_avoid_for
    from marl_llm_b200.sharding import all_reduce_stats, episode_stats, max_over_ranks, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device: the simulator has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.variant != "assembly":
        (flocking_line if args.variant == "flocking" else predator_prey_line)(args, torch, rank, world, local_rank, barrier, max_over_ranks)
        if world > 1:
            dist.destroy_process_group()
        return

    shapes = load_shapes()
    E, n_a = args.envs_per_gpu, args.n_a
    ngm = int(shapes["n_g"].max())
    r_avoid = r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"])
    parity = args.layout == "parity"
    sim = BatchedAssemblySim(E, n_a, ngm, r_avoid, device=local_rank,
                             out_dtype=torch.float64 if parity else torch.float32, emit_indices=parity,
                             brute_force_scan=args.brute_force_scan)
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    env0, _ = shard_range(world * E, rank, world)                       # this rank's global env ids: [env0, env0 + E)
    sim.n_g[:] = int(np.mean(shapes["n_g"]))                            # mean cell count (roofline bytes); per-env counts live on the device

    K, W = args.steps, args.warmup
    ring = 16
    acts = torch.empty(ring, E, 2, n_a, dtype=torch.float32, device="cuda")
    for r in range(ring):
        sim.fill_actions(acts[r], seed=226, step=r, env_offset=env0)
    EP = args.episode_length
    # auto-reset cohorts: env e belongs to cohort e mod C and is reset when t = (EP / C) * cohort (mod EP): every episode lasts
    # exactly EP steps, the batch holds C evenly spaced episode ages at any time
    C_ = max(1, min(args.reset_cohorts, EP))
    stride = EP // C_
    lists = [torch.arange(ph // stride, E, C_, dtype=torch.int32, device="cuda") if (ph % stride == 0 and ph // stride < C_)
             else torch.empty(0, dtype=torch.int32, device="cuda") for ph in range(EP)]
    clock = {"t": 0}
    peak, peak_src = measured_hbm_peak()

    def step_random():
        """One step of the 'random' regime: U(-1,1) actions (BASELINE config 1/3) for every env, then the auto-reset of the
        envs whose 200-step episode (CFG:181) just ended.  The envs form 25 cohorts whose episodes start 8 steps apart, so the
        batch is a stationary mixture of episode ages and the measured rate does not depend on where the timed window starts
        or how long it is (a cohort's reset + first observation are two small extra launches inside the timed region)."""
        t = clock["t"]
        sim.step(acts[t % ring])
        due = lists[t % EP]
        if due.numel():
            sim.reset_envs(due, seed=226, episode=1 + t, env_offset=env0)
        clock["t"] = t + 1

    def step_converged():
        """One step of the 'converged' regime: every agent follows the prior policy from a state in which the swarm already
        fills its shape (what training converges to): all agents in-shape, ~75 sensed cells, occupancy filter and psi sums live."""
        sim.step(sim.a_prior)

    def timed(step_fn, k, w):
        for _ in range(w):
            step_fn()
        barrier()
        l0 = sim.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(k):
            step_fn()
        ev1.record()
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1), device="cuda"), sim.launch_count - l0

    def measured_traffic(regime):
        prof = os.path.join(REPO, "profiles", "traffic.json")
        try:
            return json.load(open(prof)).get(f"{args.layout}_{regime}_bytes_per_launch") if n_a == 30 and E == 65536 else None
        except Exception:
            return None

    def roofline_of(ms_per_step, regime):
        """SURVEY.md 8(d): HBM for the 30-agent configurations (algorithmic bytes: 1126 B per agent-step in the production
        layout at n_g = 512), the FP32 pipe for the O(n_a^2) large-swarm configuration (6 n_a + 6 n_g flops per agent-step)."""
        if n_a <= 128:
            b = sim.algorithmic_bytes_per_agent_step(survey=True)
            achieved = b * E * n_a / (ms_per_step * 1e-3) / 1e9
            ext = sim.algorithmic_bytes_per_agent_step(survey=False)
            return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": measured_traffic(regime),
                    "algorithmic_bytes_per_launch": b * E * n_a,
                    "peak_source": peak_src, "launch_ms": ms_per_step, "algorithmic_bytes_per_agent_step": b,
                    "bytes_per_agent_step_incl_neighbor_index_and_seed": ext,
                    "frac_incl_neighbor_index_and_seed": ext * E * n_a / (ms_per_step * 1e-3) / 1e9 / peak,
                    "kernel": ("swarm::k_step<PH=1> + swarm::k_step<PH=2, FAST=%d> (one step = two launches; the second, the lookup-scan "
                               "kernel, is the dominant one)" % sim.fast_path) if sim.fast_path else
                              "swarm::k_step<PH=1> + swarm::k_step<PH=2> (one step = two launches; the second is the dominant one)"}
        f32, f64 = sim.measure_fma_peak()
        flops = 6.0 * n_a + 6.0 * float(np.mean(shapes["n_g"]))
        achieved = flops * E * n_a / (ms_per_step * 1e-3) / 1e12
        return {"bound": "fp32", "achieved": achieved, "peak": f32, "unit": "TFLOP/s", "frac": achieved / f32, "traffic": None,
                "peak_source": "measured here: register-resident FMA loop (swarm_measure_fma_peak)", "fp64_peak_tflops": f64,
                "launch_ms": ms_per_step, "algorithmic_flops_per_agent_step": flops,
                "note": "pair loops run an fp32 filter pass + exact fp64 on the survivors; flops = SURVEY 8(d) count (selection excluded)",
                "kernel": "swarm::k_step<PH=0, MAXT=1024, FAST=%d>" % sim.fast_path}

    regimes = {}
    sampler = ClockSampler(local_rank); sampler.start()
    want = ["random", "converged"] if args.regime == "both" else [args.regime]
    for regime in want:
        if regime == "random":
            sim.reset(seed=226, episode=0, env_offset=env0)              # assembly.py:156-223 on the device
            for _ in range(EP):                                          # untimed pre-roll: one full cycle -> uniform episode ages
                step_random()
            ms, launches = timed(step_random, K, W)
        else:
            blocks, n_g, l_cell, p, dp, pose = synth_batch(E, n_a, shapes, 226 + rank, "converged", with_pose=True)
            sim.set_grid_pose(*pose)                                     # the device applies grid = R.origin + off itself
            sim.set_state(p, dp)
            sim.observe()
            sim.step(acts[0])                                            # produces the first prior action
            for _ in range(20):
                step_converged()
            ms, launches = timed(step_converged, K, W)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, regime,
                         dict(obs=sim.obs, reward=sim.reward, done=sim.done, a_prior=sim.a_prior, p=sim.p, dp=sim.dp,
                              neighbor_index=sim.neighbor_index, in_flags=sim.in_flags, sensed_index=sim.sensed_index,
                              occupied_index=sim.occupied_index), DUMP_BYTES // len(want))
        stats = all_reduce_stats(episode_stats(sim.reward, sim.in_flags)).tolist()   # episode statistics (not timed)
        regimes[regime] = {"ms_per_step": ms / K, "value": world * E * n_a * K / (ms * 1e-3), "gpu_launches": int(launches),
                           "roofline": roofline_of(ms / K, regime),
                           "mean_reward": stats[0] / stats[2], "in_shape_fraction": stats[1] / stats[2]}
    clocks = sampler.stop()
    head = regimes[want[0]]
    ms, launches, value, roofline = head["ms_per_step"] * K, head["gpu_launches"], head["value"], head["roofline"]
    bytes_per_launch = sim.algorithmic_bytes_per_agent_step(survey=True) * E * n_a

    # ---- end to end through host buffers ----
    e2e = None
    if not args.no_e2e:
        sim.reset(seed=226, episode=0, env_offset=env0)                  # the e2e loop runs from the reference's reset distribution
        osz = 8 if parity else 4
        act_h = torch.empty(ring, E, 2, n_a, dtype=torch.float32).pin_memory()
        act_h.copy_(acts.cpu())
        obs_h = torch.empty(E, sim.obs_dim, n_a, dtype=sim.out_dtype).pin_memory()
        rew_h = torch.empty(E, 1, n_a, dtype=sim.out_dtype).pin_memory()
        pri_h = torch.empty(E, 2, n_a, dtype=sim.out_dtype).pin_memory()
        for t in range(min(W, 3)):
            sim.step_host(act_h[t % ring], obs_h, rew_h, pri_h)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for t in range(K):
            sim.step_host(act_h[(W + t) % ring], obs_h, rew_h, pri_h)
        e1.record()
        barrier()
        ems = e0.elapsed_time(e1)
        ems = max_over_ranks(ems, device="cuda")
        # what the host side can take: a plain pinned D2H copy of the same observation buffer, all ranks at once (no kernels)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(5):
            obs_h.copy_(sim.obs, non_blocking=True)
        c1.record()
        barrier()
        cms = max_over_ranks(c0.elapsed_time(c1), device="cuda") / 5
        d2h = E * n_a * (sim.obs_dim + 1 + 2) * osz
        e2e = {"value": world * E * n_a * K / (ems * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": E * 2 * n_a * 4, "d2h_bytes_per_step": d2h,
               "ms_per_step": ems / K, "api": "swarm_step_host (C ABI, pinned host buffers)",
               "achieved_d2h_gbs_per_rank": d2h / (ems / K * 1e-3) / 1e9,
               "host_copy_ceiling_gbs_per_rank": obs_h.numel() * osz / (cms * 1e-3) / 1e9,
               "host_copy_ceiling_note": f"plain cudaMemcpyAsync D2H of the obs buffer into pinned memory, {world} rank(s) concurrently"}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import ref_glue
        cores = os.cpu_count() or 1
        if ref_glue.available():
            r = ref_glue.timed_rollouts(n_a, shapes, cores, 2, 200)
            r1 = ref_glue.timed_rollouts(n_a, shapes, 1, 1, 200)          # BASELINE config 1: one env, one core, 200 steps
            cpu = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "reference",
                   "sample": f"{cores} processes x 2 episodes x 200 steps x {n_a} agents (reference C++ via oracle/_ref + NumPy glue)",
                   "single_core_value": r1["value"]}
        else:
            from oracle import oracle as orc
            r = port_rollouts(orc, shapes, n_a, cores, 64 * cores, 50)
            cpu = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{r['envs']} envs x 50 steps, oracle C port, {cores} OpenMP threads"}

    # ---- widened path (SURVEY 8 f1): replay push, on-device policy, whole device-resident rollout loop (rank 0, N=1) ----
    extras = None
    if rank == 0 and world == 1 and not args.no_extras and not parity and n_a == 30:
        try:
            extras = widened_path_numbers(torch, sim, acts[0], peak, shapes)
        except Exception as ex:            # the widened-path numbers must never cost the main line
            extras = {"error": f"{type(ex).__name__}: {ex}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": (f"assembly env, {n_a} agents x {E} envs per GPU, env-sharded (BASELINE config 3)" if n_a == 30 else
                                    f"large swarm: {n_a} agents x {E} envs per GPU (BASELINE config 4)"),
                       "n_a": n_a, "envs_per_gpu": E, "layout": args.layout, "regime": want[0],
                       "episodes": f"{EP}-step episodes, auto-reset (swarm_reset_envs) in {C_} cohorts whose episodes start {stride} steps apart; the reset launches are inside the timed region, reset envs are not counted as extra agent-steps",
                       "out_dtype": "f64" if parity else "f32", "state_dtype": "f64",
                       "grid_scan": "all-pairs" if args.brute_force_scan else ("lookup (per-shape bin table + lattice rows)" if sim.fast_path else "word-box culled"),
                       "l2": f"working set per step {bytes_per_launch / 1e6:.0f} MB >> 126 MB L2 (no flush needed)",
                       "actions": f"ring of {ring} pre-generated device buffers"},
            "regimes": regimes,
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "widened_path": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
