"""Times prior populations (marl_llm_b200.prior_program.PriorPopulation, DESIGN.md §12) and prints one JSON line per case.

K distinct programs (marl_llm_b200/priors/reference_prior.cu, each with a comment naming its k, so each is its own compile and
CUBIN) are assigned to envs interleaved, env e -> e % K.  Production layout (fp32 outputs), device reset, U(-1,1) actions.
  config 3 (65 536 envs x 30 agents), K in {1, 4, 16, 64}:
    step_builtin_ms      one step with the built-in (fused) prior
    step_program_ms      one step with reference_prior.cu installed alone (swarm_set_prior_program)
    step_pop<K>_ms       one step with the population installed: K program launches over 65 536 / K envs each, then the step
    actions_program_ms / actions_pop<K>_ms   the program / the population as actions (swarm_prior_*_actions, fp64 out)
  config 4 (1024 envs x 1024 agents), K = 16 (64 envs per program): the same, for K = 16.
Times are CUDA events around `--reps` calls after `--warmup` calls, median of 5 windows; the step variants alternate between
windows.  `compile` reports the host time of compiling and loading each program (NVRTC, no cache; the first compile also
opens NVRTC).

    python tools/bench_prior_population.py [--reps 50] [--warmup 10]
    python tools/bench_prior_population.py --profile DIR [--k 16]   # torch.profiler trace of config-3 steps with K programs
                                                                    # (K = 1: the launches of one installed program): kernel
                                                                    # times and the gaps between the launches of one step
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from marl_llm_b200.batched import BatchedAssemblySim, r_avoid_for  # noqa: E402
from marl_llm_b200.prior_program import PriorPopulation, PriorProgram, reference_prior_source  # noqa: E402
from tests.helpers import load_shapes  # noqa: E402
from tools.bench_prior_program import gpu_info, timed  # noqa: E402

KS = (1, 4, 16, 64)


def candidates(n):
    src = reference_prior_source()
    return [src + f"\n// candidate {k}\n" for k in range(n)]


def make(E, n_a, shapes):
    ngm = int(shapes["n_g"].max())
    sim = BatchedAssemblySim(E, n_a, ngm, r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"]))
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    sim.reset(seed=1)
    return sim


def run_case(name, sim, variants, reps, warmup, info):
    """variants: {label: installer}; steps alternate between variants window by window"""
    E, n_a = sim.E, sim.n_a
    acts = [sim.fill_actions(torch.empty(E, 2, n_a, dtype=torch.float32, device="cuda"), seed=2, step=t) for t in range(4)]
    k = [0]

    def step():
        sim.step(acts[k[0] % 4]); k[0] += 1

    res = {v: [] for v in variants}
    for v, install in variants.items():
        install()
        for _ in range(warmup):
            step()
    for _ in range(5):
        for v, install in variants.items():
            install()
            step()                                             # the first step after a switch may run k_prior
            res[v].append(timed(step, reps))
    sim.set_prior_program(None)
    step()                                                     # the actions below then see a stored nearest cell, as in a rollout
    line = {"case": name, "envs": E, "n_a": n_a}
    for v in variants:
        line[f"step_{v}_ms"] = round(float(np.median(res[v])), 4)
    for v in variants:
        if v != "builtin":
            line[f"ratio_{v}_to_program"] = round(line[f"step_{v}_ms"] / line["step_program_ms"], 4)
    line["windows"] = {v: [round(x, 4) for x in res[v]] for v in variants}
    line["gpu"] = info
    return line


def actions_times(sim, runners, reps, warmup):
    out = torch.empty(sim.E, 2, sim.n_a, dtype=torch.float64, device="cuda")
    t = {}
    for label, fn in runners.items():
        for _ in range(warmup):
            fn(sim, out=out)
        t[f"actions_{label}_ms"] = round(float(np.median([timed(lambda: fn(sim, out=out), reps) for _ in range(5)])), 4)
    return t


def profile(out_dir, K, info):
    """kernel durations and launch gaps of config-3 steps with K programs (torch.profiler, CUDA activity)"""
    from torch.profiler import ProfilerActivity, profile as tprofile
    shapes = load_shapes()
    progs = [PriorProgram(s) for s in candidates(K)]
    sim = make(65536, 30, shapes)
    sim.set_prior_population(PriorPopulation(progs, np.arange(sim.E) % K))
    act = sim.fill_actions(torch.empty(sim.E, 2, 30, dtype=torch.float32, device="cuda"), seed=2, step=0)
    for _ in range(10):
        sim.step(act)
    torch.cuda.synchronize()
    steps = 10
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            sim.step(act)
        torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    prof.export_chrome_trace(os.path.join(out_dir, f"prior_population_k{K}.json"))
    ev = sorted([e for e in prof.events() if e.device_type.name == "CUDA"], key=lambda e: e.time_range.start)
    kinds = {}
    for e in ev:
        kinds.setdefault("program" if e.name.startswith("swarm_prior") else e.name[:40], []).append(e.time_range.end - e.time_range.start)
    gaps = [b.time_range.start - a.time_range.end for a, b in zip(ev, ev[1:])]
    span = (ev[-1].time_range.end - ev[0].time_range.start) / steps
    print(json.dumps({"case": f"profile_k{K}", "kernels_per_step": len(ev) / steps, "span_per_step_us": round(span, 2),
                      "kernel_us_per_step": {k: round(sum(v) / steps, 2) for k, v in kinds.items()},
                      "kernel_us_median": {k: round(float(np.median(v)), 2) for k, v in kinds.items()},
                      "gap_us_median": round(float(np.median(gaps)), 2), "gap_us_per_step": round(sum(gaps) / steps, 2),
                      "gpu": info}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--profile", metavar="DIR")
    ap.add_argument("--k", type=int, default=16)
    args = ap.parse_args()
    info = gpu_info()
    if args.profile:
        profile(args.profile, args.k, info)
        return
    srcs = candidates(max(KS))
    progs, secs = [], []
    for s in srcs:
        t0 = time.perf_counter()
        progs.append(PriorProgram(s))
        secs.append(time.perf_counter() - t0)
    print(json.dumps({"case": "compile", "programs": len(progs), "compile_and_load_s_first": round(secs[0], 3),
                      "compile_and_load_s_median": round(float(np.median(secs)), 3),
                      "compile_and_load_s_total": round(sum(secs), 2), "each_s": [round(x, 3) for x in secs], "gpu": info}), flush=True)
    shapes = load_shapes()
    for name, E, n_a, ks in (("config3", 65536, 30, KS), ("config4", 1024, 1024, (16,))):
        sim = make(E, n_a, shapes)
        pops = {K: PriorPopulation(progs[:K], np.arange(E) % K) for K in ks}
        variants = {"builtin": lambda: sim.set_prior_program(None), "program": lambda: sim.set_prior_program(progs[0])}
        for K in ks:
            variants[f"pop{K}"] = (lambda p: lambda: sim.set_prior_population(p))(pops[K])
        line = run_case(name, sim, variants, args.reps, args.warmup, info)
        runners = {"program": progs[0].actions}
        runners.update({f"pop{K}": pops[K].actions for K in ks})
        line.update(actions_times(sim, runners, args.reps, args.warmup))
        print(json.dumps(line), flush=True)
        sim.close()


if __name__ == "__main__":
    main()
