"""Times swarm_render (SwarmRenderer.render) with CUDA events after a warm-up and prints one JSON line per case:
  64 and 1024 envs x 30 agents on the library shapes, 512 x 512, without and with 15-sample trails;
  one BASELINE config-4 env (1024 agents) at 1024 x 1024.
Each line has the time per batch of frames, Mpixel/s, the write-bandwidth floor (frame bytes / 7.7 TB/s, the HBM3e bandwidth of
NVIDIA's B200 data sheet) and, as a measured yardstick, the time torch's fill of the same frames tensor takes.  The GPU name and
power limit, read in the same run, come first.  The swarms are driven by the expert controller first, so cells, trails and both
agent colours are on the frames.

    python tools/bench_render.py [--reps 50] [--out results.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_llm_b200.batched import BatchedAssemblySim, r_avoid_for   # noqa: E402
from marl_llm_b200.render import SwarmRenderer                     # noqa: E402
from tests.helpers import load_shapes                              # noqa: E402

HBM_BYTES_PER_S = 7.7e12
CASES = [  # name, envs, agents, pixels per side, trail samples
    ("64 envs x 30 agents, 512x512", 64, 30, 512, 0),
    ("64 envs x 30 agents, 512x512, 15-sample trails", 64, 30, 512, 15),
    ("1024 envs x 30 agents, 512x512", 1024, 30, 512, 0),
    ("1024 envs x 30 agents, 512x512, 15-sample trails", 1024, 30, 512, 15),
    ("config 4: 1 env x 1024 agents, 1024x1024", 1, 1024, 1024, 0),
]


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0), "power_limit_w": "not measured"}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out)
    except (OSError, ValueError, subprocess.SubprocessError):
        pass
    return info


def timed(fn, reps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def run_case(name, E, n_a, side, trail, reps, shapes):
    sim = BatchedAssemblySim(E, n_a, int(shapes["n_g"].max()), r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"]))
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    sim.reset(seed=1)
    r = SwarmRenderer(sim, np.arange(E), side, side, trail_len=trail)
    for _ in range(30):
        sim.step(sim.strategy_actions("rule"))
        r.record()
    for _ in range(3):
        r.render()
    torch.cuda.synchronize()
    ms = timed(r.render, reps)
    fill_ms = timed(lambda: r.frames.fill_(0), reps)
    nbytes = r.frames.numel()
    pixels = E * side * side
    res = {"case": name, "envs": E, "agents": n_a, "width": side, "height": side, "trail_samples": trail, "reps": reps,
           "ms_per_batch": round(ms, 4), "mpixel_per_s": round(pixels / ms / 1e3, 1), "frame_bytes": nbytes,
           "write_floor_ms_datasheet": round(nbytes / HBM_BYTES_PER_S * 1e3, 4), "torch_fill_ms": round(fill_ms, 4),
           "in_shape_agents": int(sim.in_flags.bitwise_and(1).sum())}
    sim.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_render.py needs a CUDA device")
    shapes = load_shapes()
    lines = [gpu_info()] + [run_case(*c, args.reps, shapes) for c in CASES]
    for ln in lines:
        print(json.dumps(ln), flush=True)
    if args.out:
        with open(args.out, "a") as f:
            f.writelines(json.dumps(ln) + "\n" for ln in lines)


if __name__ == "__main__":
    main()
