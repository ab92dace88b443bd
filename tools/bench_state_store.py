"""Times swarm_state_save / swarm_state_load (marl_llm_b200.state_store.StateStore) and prints one JSON line per case.

Each case is timed with CUDA events around one save or load call, 30 repetitions after two warm-up calls; before every timed call
a 512 MB buffer is overwritten, which evicts the 126 MB L2, so every pass reads from HBM.  `ms` times the kernels alone (the
device sleeps while the host enqueues the call), `ms_call` the call as a caller sees it (host-side checks and launches
included).  `bytes` counts what a copy must move: every stored row of every pair, read once and written once (slot padding
excluded).  `hbm_share` = that over the time, divided by the HBM bandwidth this project measured on a B200 (6452.5 GB/s,
DESIGN.md §4.3).

    python tools/bench_state_store.py [--reps 30] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from marl_llm_b200.batched import BatchedAssemblySim, r_avoid_for  # noqa: E402
from marl_llm_b200.state_store import StateStore  # noqa: E402
from tests.helpers import load_shapes  # noqa: E402

HBM_GBS = 6452.5


def row_bytes(sim):
    """Bytes of one env's stored rows (the slot layout of DESIGN.md §11 without padding)."""
    n, osz = sim.n_a, 4 if sim.out_dtype == torch.float32 else 8
    b = 2 * 16 * n + 16 * sim.n_g_pad + 16 * (sim.n_g_pad // 32) + 16 + 4 + 8 + 32 + 4   # p, dp, grid, word boxes, frame .. shape id
    b += 4 * n + 24 * n + 4 * n + sim.obs_dim * n * osz + n * osz                         # nearest, neighbours, in_flags, obs, reward
    if sim.want_prior:
        b += 2 * 2 * n * osz
    if sim.emit_indices:
        b += (80 + 200) * 4 * n
    return b


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return name, q


def make(E, n_a, parity):
    shapes = load_shapes()
    sim = BatchedAssemblySim(E, n_a, int(shapes["n_g"].max()), r_avoid_for(n_a, shapes["n_g"], shapes["l_cell"]),
                             out_dtype=torch.float64 if parity else torch.float32, emit_indices=parity)
    sim.set_shapes(shapes["grid_origin"], shapes["l_cell"])
    sim.reset(seed=1)
    act = torch.empty(E, 2, n_a, dtype=torch.float32, device="cuda")
    for t in range(2):                        # stepped: the load writes both priors
        sim.step(sim.fill_actions(act, seed=1, step=t))
    return sim


def time_call(fn, reps, flush, queued):
    """Median, min and max ms.  queued: the device idles (a sleep kernel) while the host enqueues the call's launches, so the
    events time the kernels alone; otherwise they time the call as a caller sees it, host-side checks and launches included."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for _ in range(2):
        fn()
    for a, b in ev:
        flush.fill_(1)
        if queued:
            torch.cuda._sleep(20_000_000)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    return float(np.median(ms)), float(ms.min()), float(ms.max())


def timed(fn, reps, flush):
    return time_call(fn, reps, flush, True), time_call(fn, reps, flush, False)


def report(case, sim, pairs, times, extra=None):
    nbytes = 2 * pairs * row_bytes(sim)
    (med, lo, hi), (call, _, _) = times
    out = dict(case=case, pairs=pairs, n_a=sim.n_a, bytes=nbytes, ms=round(med, 4), ms_min=round(lo, 4), ms_max=round(hi, 4),
               gbs=round(nbytes / med / 1e6, 1), hbm_share=round(nbytes / med / 1e6 / HBM_GBS, 3), ms_call=round(call, 4))
    out.update(extra or {})
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--quick", action="store_true", help="small sizes (a functional check, not a measurement)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_state_store needs a CUDA device")
    name, q = device_info()
    print(json.dumps(dict(device=name, nvidia_smi_name_power_limit=q, hbm_gbs_measured=HBM_GBS, reps=args.reps,
                          l2="evicted before every timed call (512 MB overwrite)")), flush=True)
    flush = torch.empty(128 * 2**20, dtype=torch.float32, device="cuda")
    E = 2048 if args.quick else 65536
    big_n = 64 if args.quick else 1024
    for layout in ("production", "parity"):
        sim = make(E, 30, layout == "parity")
        st = StateStore(sim, E)
        ids = np.arange(E)
        report(f"save all, {layout}", sim, E, timed(lambda: st.save(ids), args.reps, flush), dict(slot_bytes=st.slot_bytes))
        report(f"load all, {layout}", sim, E, timed(lambda: st.load(ids, ids), args.reps, flush))
        if layout == "production":
            rng = np.random.RandomState(0)
            few = rng.choice(E, 1024, replace=False)
            slots = rng.choice(E, 1024, replace=False)
            report("save 1024 scattered envs", sim, 1024, timed(lambda: st.save(few, slots), args.reps, flush))
            report("load 1024 scattered envs", sim, 1024, timed(lambda: st.load(slots, few), args.reps, flush))
            st.save([0])
            rest = np.arange(1, E)
            zeros = np.zeros(E - 1, dtype=np.int64)
            report("clone one env into all others (load)", sim, E - 1, timed(lambda: st.load(zeros, rest), args.reps, flush),
                   dict(note="the one slot is read from L2 after the first CTAs"))
        st.close()
        del sim, st
        torch.cuda.empty_cache()
    sim = make(big_n, 1024, False)
    st = StateStore(sim, big_n)
    ids = np.arange(big_n)
    report("save all, 1024 agents", sim, big_n, timed(lambda: st.save(ids), args.reps, flush), dict(slot_bytes=st.slot_bytes))
    report("load all, 1024 agents", sim, big_n, timed(lambda: st.load(ids, ids), args.reps, flush))
    report("save one env, 1024 agents", sim, 1, timed(lambda: st.save([5]), args.reps, flush))


if __name__ == "__main__":
    main()
