"""Times prior programs (marl_llm_b200.prior_program, DESIGN.md §12) and prints one JSON line per case.

For BASELINE config 3 (65 536 envs x 30 agents) and config 4 (1024 envs x 1024 agents), production layout (fp32 outputs),
device reset, U(-1,1) actions:
  step_builtin_ms   one step with the built-in (fused) prior
  step_program_ms   one step with marl_llm_b200/priors/reference_prior.cu installed (its a_prior kernel + the step kernel)
  program_actions_ms  the program's kernel alone, as swarm_prior_actions (the a_prior kernel's body, fp64 output), repeated
  floor_*_ms        byte floors: per agent p, dp (32 B), the neighbour list (24 B), nearest cell and in_flags (8 B), one cell
                    (16 B) and the prior written (8 B as fp32 a_prior, 16 B as fp64 actions), at the HBM bandwidth this project
                    measured on a B200 (6452.5 GB/s, DESIGN.md §4.3)
Times are CUDA events around `--reps` calls after `--warmup` calls, median of 5 windows; the two step variants alternate
between windows.  The host compile time of the shipped program (NVRTC, no cache) is printed too.

    python tools/bench_prior_program.py [--reps 50] [--warmup 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from marl_llm_b200.batched import BatchedAssemblySim, r_avoid_for  # noqa: E402
from marl_llm_b200.prior_program import PriorProgram, compile_source, reference_prior_source  # noqa: E402
from tests.helpers import load_shapes  # noqa: E402

HBM_GBS = 6452.5
BYTES_PER_AGENT = 32 + 24 + 8 + 16 + 8


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    info = gpu_info()
    t0 = time.perf_counter()
    compile_source(reference_prior_source())
    print(json.dumps({"case": "compile", "host_compile_s": round(time.perf_counter() - t0, 3), "gpu": info}), flush=True)
    prog = PriorProgram(reference_prior_source())
    shapes = load_shapes()
    ngm = int(shapes["n_g"].max())
    for name, E, n_a in (("config3", 65536, 30), ("config4", 1024, 1024)):
        sim = BatchedAssemblySim(E, n_a, ngm, r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"]))
        sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
        sim.reset(seed=1)
        acts = [sim.fill_actions(torch.empty(E, 2, n_a, dtype=torch.float32, device="cuda"), seed=2, step=t) for t in range(4)]
        k = [0]

        def step():
            sim.step(acts[k[0] % 4]); k[0] += 1

        res = {"builtin": [], "program": []}
        for which in ("builtin", "program"):
            sim.set_prior_program(prog if which == "program" else None)
            for _ in range(args.warmup):
                step()
        for w in range(5):
            for which in ("builtin", "program"):
                sim.set_prior_program(prog if which == "program" else None)
                step()                                         # the first step after a switch may run k_prior
                res[which].append(timed(step, args.reps))
        # the program's kernel alone, as actions (the a_prior kernel's body with fp64 output, stored nearest cell), repeated
        out = torch.empty(E, 2, n_a, dtype=torch.float64, device="cuda")
        for _ in range(args.warmup):
            prog.actions(sim, out=out)
        t_act = float(np.median([timed(lambda: prog.actions(sim, out=out), args.reps) for _ in range(5)]))
        sb, sp = float(np.median(res["builtin"])), float(np.median(res["program"]))
        floor = E * n_a * BYTES_PER_AGENT / (HBM_GBS * 1e9) * 1e3
        floor_act = E * n_a * (BYTES_PER_AGENT + 8) / (HBM_GBS * 1e9) * 1e3
        print(json.dumps({"case": name, "envs": E, "n_a": n_a, "step_builtin_ms": round(sb, 4), "step_program_ms": round(sp, 4),
                          "ratio": round(sp / sb, 4), "program_actions_ms": round(t_act, 4),
                          "floor_a_prior_ms": round(floor, 4), "floor_actions_ms": round(floor_act, 4),
                          "windows_builtin": [round(v, 4) for v in res["builtin"]], "windows_program": [round(v, 4) for v in res["program"]],
                          "gpu": info}), flush=True)
        sim.close()


if __name__ == "__main__":
    main()
