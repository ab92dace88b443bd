"""Times one policy kernel at the BASELINE config-3 shape (65536 envs x 30 agents) with CUDA events (profiling aid).

usage: bench_policy.py [fp32 | f16_tc | f16x3_tc] [am]
The precision picks k_policy_mlp, k_policy_mlp_tc or k_policy_mlp_tc3; `am` passes agent-major observation rows."""
import json, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from marl_llm_b200.policy import DevicePolicy
import torch.nn as nn
E, n_a, D, H, A = 65536, 30, 192, 180, 2
sd = {}
for name, (o, i) in (("fc1", (H, D)), ("fc2", (H, H)), ("fc3", (H, H)), ("fc4", (A, H))):
    l = nn.Linear(i, o); sd[name + ".weight"] = l.weight; sd[name + ".bias"] = l.bias
prec = sys.argv[1] if len(sys.argv) > 1 else "fp32"
AM = len(sys.argv) > 2 and sys.argv[2] == "am"      # agent-major observation rows [E, n_a, D]
pol = DevicePolicy(D, A, H, precision=prec).load_state_dict(sd)
obs = torch.randn(E, n_a, D, device="cuda") if AM else torch.randn(E, D, n_a, device="cuda")
act = torch.empty(E, A, n_a, device="cuda")
for _ in range(30): pol.step(obs, explore=True, out=act, want_log_pi=False, agent_major=AM)     # also lets the clocks ramp up
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
K = 20
ev[0].record()
for _ in range(K): pol.step(obs, explore=True, out=act, want_log_pi=False, agent_major=AM)
ev[1].record(); torch.cuda.synchronize()
ms = ev[0].elapsed_time(ev[1]) / K
per = []
for _ in range(4):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); pol.step(obs, explore=True, out=act, want_log_pi=False, agent_major=AM); b.record(); torch.cuda.synchronize()
    per.append(round(a.elapsed_time(b), 3))
print("single launches ms:", per, file=sys.stderr)
import time
torch.cuda.synchronize(); t0 = time.perf_counter()
for _ in range(5): pol.step(obs, explore=True, out=act, want_log_pi=False, agent_major=AM)
t1 = time.perf_counter(); torch.cuda.synchronize(); t2 = time.perf_counter()
print(f"host time per call {(t1 - t0) / 5 * 1e3:.3f} ms, total per call incl. drain {(t2 - t0) / 5 * 1e3:.3f} ms", file=sys.stderr)
flop = 2.0 * E * n_a * (D * H + H * H * 2 + H * A)
flop_padded = 2.0 * E * n_a * (192 * 192 * 3 + 192 * A)
print(json.dumps({"layout": "agent_major" if AM else "reference", "kernel": "k_policy_mlp" + ("_tc" if prec == "f16_tc" else "_tc3" if prec == "f16x3_tc" else ""), "agents": E * n_a, "ms": ms, "agent_forwards_per_s": E * n_a / ms * 1e3,
                  "useful_TFLOPs": flop / ms / 1e9, "issued_TFLOPs": flop_padded / ms / 1e9}))
