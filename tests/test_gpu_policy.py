"""On-device rollout policy (C ABI group 4) against a plain torch fp32 restatement of the reference network
(marl_llm/algorithm/utils/networks.py:22-44: four nn.Linear, F.leaky_relu, tanh output) and of DDPGAgent.step's
exploration (utils/agents.py:82-93, utils/noise.py:24-37).  Floating point: rtol 1e-5 / atol 2e-6 (fp32 sums in a
different order than a GEMM library's; the north star's tolerance for floating point is 1e-5 relative).  The reference values
are the same network evaluated in float64 and rounded to fp32 (`exact_forward`): torch's own fp32 CPU GEMM differs from box to
box (on some hosts of the GPU pool it is 5e-5 away from the float64 result, which failed the former fp32-vs-fp32 comparison)."""
import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from marl_llm_b200.policy import DevicePolicy

pytestmark = pytest.mark.gpu


class RefMLP(nn.Module):                                   # networks.py:6-44 with constrain_out=True
    def __init__(self, i, o, h):
        super().__init__()
        self.fc1, self.fc2, self.fc3, self.fc4 = nn.Linear(i, h), nn.Linear(h, h), nn.Linear(h, h), nn.Linear(h, o)

    def forward(self, x):
        return torch.tanh(self.fc4(F.leaky_relu(self.fc3(F.leaky_relu(self.fc2(F.leaky_relu(self.fc1(x))))))))


def exact_forward(ref, x):
    """The fp32-parameter network evaluated in float64, rounded to fp32: what every fp32 implementation approximates."""
    import copy
    with torch.no_grad():
        return copy.deepcopy(ref).double()(x.double()).float()


@pytest.mark.parametrize("E,n_a,D,H,A", [(64, 30, 192, 180, 2), (3, 7, 188, 180, 2), (1, 1, 192, 180, 2), (5, 100, 192, 64, 3),
                                         (2, 1024, 192, 180, 2)])
def test_policy_matches_torch_fp32(E, n_a, D, H, A):
    torch.manual_seed(E + n_a)
    ref = RefMLP(D, A, H)
    with torch.no_grad():                                   # weights large enough to leave the linear region of tanh
        for p in ref.parameters():
            p.mul_(3.0)
    obs = torch.randn(E, D, n_a) * 0.7
    obs[:, 32:, :] *= (torch.rand(E, D - 32, n_a) < 0.2)   # sparse sensed-cell rows like the env's
    pol = DevicePolicy(D, A, H).load_state_dict(ref.state_dict())
    act, log_pi = pol.step(obs.cuda(), explore=False)
    with torch.no_grad():
        want = exact_forward(ref, obs.permute(0, 2, 1).reshape(E * n_a, D)).reshape(E, n_a, A).permute(0, 2, 1)   # agents.py:79,95 (.t())
    assert act.shape == (E, A, n_a)
    torch.testing.assert_close(act.cpu(), want, rtol=1e-5, atol=4e-6)
    assert torch.all(log_pi == 0)                           # agents.py:82: -dim * log(1)
    # reference-shaped 2-D call (TRAIN:97-98): [obs_dim, n_a] -> [act_dim, n_a]
    a2, lp2 = pol.step(obs[0].cuda())
    assert a2.shape == (A, n_a) and lp2.shape == (1, n_a) and torch.equal(a2, act[0])
    assert pol.launch_count == 2


PRECISIONS = ["fp32", "f16_tc", "f16x3_tc"]


def test_exploration_noise_statistics_and_log_prob():
    _check_exploration("fp32")


@pytest.mark.parametrize("prec", ["f16_tc", "f16x3_tc"])
def test_exploration_noise_statistics_and_log_prob_tensor_cores(prec):
    """The tensor-core kernels' own exploration tail, held to the fp32 kernel's statistics and tolerances."""
    _check_exploration(prec)


def _check_exploration(prec):
    E, n_a, D, H, A = 2048, 30, 192, 180, 2
    torch.manual_seed(0)
    ref = RefMLP(D, A, H)
    obs = torch.randn(E, D, n_a, device="cuda") * 0.3
    pol = DevicePolicy(D, A, H, noise_scale=0.1, epsilon=0.0, seed=7, precision=prec).load_state_dict(ref.state_dict())
    clean, _ = pol.step(obs)
    noisy, log_pi = pol.step(obs, explore=True)
    noise = (noisy - clean).double()
    inside = (noisy.abs() < 1).all(dim=1, keepdim=True)     # columns the clamp did not touch
    assert inside.float().mean() > 0.99
    assert abs(float(noise.mean())) < 1e-3 and abs(float(noise.std()) - 0.1) < 1e-3
    z = noise / 0.1
    assert abs(float((z ** 4).mean()) - 3.0) < 0.05         # Gaussian kurtosis
    want_lp = -0.5 * (z ** 2).sum(dim=1, keepdim=True) - A * np.log(0.1 * np.sqrt(2 * np.pi))      # noise.py:32-37
    sel = inside.expand_as(want_lp)
    assert torch.allclose(log_pi.double()[sel], want_lp[sel], atol=2e-3)
    again, _ = pol.step(obs, explore=True)
    assert not torch.equal(again, noisy)                     # the step counter advances the stream
    # epsilon branch (agents.py:86-88): uniform actions for the whole batch, log_pi = -dim * log 2
    pol.epsilon = 1.0
    uni, lp = pol.step(obs, explore=True)
    assert float(uni.min()) >= -1 and float(uni.max()) <= 1 and abs(float(uni.mean())) < 2e-3
    assert abs(float(uni.double().var()) - 1 / 3) < 2e-3 and torch.allclose(lp, torch.full_like(lp, -A * np.log(2.0)))


@pytest.mark.parametrize("A", [2, 3])
def test_exploration_draws_are_identical_across_kernels(A):
    """The epsilon branch's actions and log_pi and the Gaussian branch's log_pi do not depend on the network: the generator
    is keyed by (seed, step, column, component) and every kernel sums the squared draws in the same order.  So all three
    kernels must write the same bits."""
    E, n_a, D, H = 67, 30, 192, 180
    torch.manual_seed(5)
    ref = RefMLP(D, A, H)
    obs = torch.randn(E, D, n_a, device="cuda")
    got = {}
    for prec in PRECISIONS:
        pol = DevicePolicy(D, A, H, noise_scale=0.2, epsilon=0.0, seed=3, precision=prec).load_state_dict(ref.state_dict())
        _, lp_gauss = pol.step(obs, explore=True)          # step 0: Gaussian branch
        pol.epsilon = 1.0
        uni, lp_uni = pol.step(obs, explore=True)          # step 1: epsilon branch
        got[prec] = (lp_gauss, uni, lp_uni)
    for prec in PRECISIONS[1:]:
        for want, have in zip(got["fp32"], got[prec]):
            assert torch.equal(want, have), prec
    assert not torch.equal(got["fp32"][1][:, 0], got["fp32"][1][:, 1])     # components draw different numbers


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("agent_major", [False, True])
@pytest.mark.parametrize("E,n_a,D", [(67, 30, 192), (5, 7, 190), (2, 33, 100), (700, 30, 188)])
def test_rows_out_is_the_transposed_observation(prec, agent_major, E, n_a, D):
    """swarm_policy_rows_out: every agent's observation row, bit for bit, for both input layouts.  obs_dim 190 (not a multiple
    of 4) and 100 (not a multiple of 32) take the loaders' scalar tails; 700 x 30 agents = 165 tiles > 148 SMs.  Writing the
    rows does not change the actions."""
    H, A = 180, 2
    torch.manual_seed(E + D)
    ref = RefMLP(D, A, H)
    obs = torch.randn(E, D, n_a, device="cuda")
    rows_want = obs.transpose(1, 2).reshape(E * n_a, D)
    x = rows_want.reshape(E, n_a, D).contiguous() if agent_major else obs
    pol = DevicePolicy(D, A, H, precision=prec).load_state_dict(ref.state_dict())
    rows = torch.full((E * n_a, D), float("nan"), device="cuda")
    act, _ = pol.step(x, rows_out=rows, agent_major=agent_major)
    act = act.clone()
    assert torch.equal(rows, rows_want)
    act_plain, _ = pol.step(x, agent_major=agent_major)
    assert torch.equal(act, act_plain)


def _f16_pipeline(ref, x):
    """torch emulation of the tensor-core path: fp16 operands, fp32 accumulation, fp16 re-rounding of h1/h2, fp32 tail."""
    r = lambda t: t.half().float()     # noqa: E731
    h = x
    for k, fc in enumerate((ref.fc1, ref.fc2, ref.fc3)):
        h = F.leaky_relu(r(h).double() @ r(fc.weight).double().t() + fc.bias.double()).float()
    return torch.tanh(h.double() @ ref.fc4.weight.double().t() + ref.fc4.bias.double()).float()


@pytest.mark.parametrize("E,n_a", [(64, 30), (5, 7), (1, 1), (3, 1024), (300, 30)])
def test_tensor_core_policy_layer1_and_outputs(E, n_a):
    """tcgen05 path: (1) its raw layer-1 accumulators equal fc1 on fp16-rounded operands (fp32 accumulation: 1e-4),
    which pins the UMMA descriptors / TMEM operand layout; (2) the actions equal a torch emulation of the fp16 pipeline
    to 5e-4 and the fp32 network to 5e-3 (documented fast-mode deviation)."""
    D, H, A = 192, 180, 2
    torch.manual_seed(11 + n_a)
    ref = RefMLP(D, A, H)
    with torch.no_grad():
        for p in ref.parameters():
            p.mul_(2.0)
    obs = torch.randn(E, D, n_a) * 0.7
    pol = DevicePolicy(D, A, H, precision="f16_tc").load_state_dict(ref.state_dict())
    dbg = torch.full((E * n_a, 192), float("nan"), device="cuda")
    pol.lib.swarm_policy_debug_buffer(pol._h, dbg.data_ptr())
    act, _ = pol.step(obs.cuda())
    pol.lib.swarm_policy_debug_buffer(pol._h, None)
    x = obs.permute(0, 2, 1).reshape(E * n_a, D)
    with torch.no_grad():
        want1 = (x.half().double() @ ref.fc1.weight.half().double().t()).float()
        torch.testing.assert_close(dbg.cpu()[:, :H], want1, rtol=1e-4, atol=1e-4)
        assert torch.all(dbg[:, H:] == 0)                       # zero-padded outputs
        emu = _f16_pipeline(ref, x).reshape(E, n_a, A).permute(0, 2, 1)
        exact = exact_forward(ref, x).reshape(E, n_a, A).permute(0, 2, 1)
    torch.testing.assert_close(act.cpu(), emu, rtol=0, atol=5e-4)   # fp16 re-rounding of h1/h2 can flip at ties
    torch.testing.assert_close(act.cpu(), exact, rtol=0, atol=5e-3)
    # same handle, exact path again
    pol.set_precision("fp32")
    act32, _ = pol.step(obs.cuda())
    torch.testing.assert_close(act32.cpu(), exact, rtol=1e-5, atol=4e-6)


@pytest.mark.parametrize("E,n_a", [(64, 30), (5, 7), (1, 1), (3, 1024), (700, 30)])
def test_split_fp16_tensor_core_policy_is_fp32_accurate(E, n_a):
    """'f16x3_tc': operands split into fp16 hi + lo, three tcgen05.mma per k-step, weights streamed through a 3-slot ring
    (700 x 30 agents = 165 tiles > 148 SMs: CTAs loop, the ring wraps).  Same tolerance as the exact FFMA path."""
    D, H, A = 192, 180, 2
    torch.manual_seed(23 + n_a)
    ref = RefMLP(D, A, H)
    with torch.no_grad():
        for p in ref.parameters():
            p.mul_(3.0)
    obs = torch.randn(E, D, n_a) * 0.7
    obs[:, 32:, :] *= (torch.rand(E, D - 32, n_a) < 0.2)
    pol = DevicePolicy(D, A, H, precision="f16x3_tc").load_state_dict(ref.state_dict())
    dbg = torch.full((E * n_a, 192), float("nan"), device="cuda")
    pol.lib.swarm_policy_debug_buffer(pol._h, dbg.data_ptr())
    act, _ = pol.step(obs.cuda())
    pol.lib.swarm_policy_debug_buffer(pol._h, None)
    x = obs.permute(0, 2, 1).reshape(E * n_a, D)
    with torch.no_grad():
        want1 = (x.double() @ ref.fc1.weight.double().t()).float()
        exact = exact_forward(ref, x).reshape(E, n_a, A).permute(0, 2, 1)
    torch.testing.assert_close(dbg.cpu()[:, :H], want1, rtol=2e-6, atol=2e-5)
    # the dropped lo x lo products are 2^-22 relative per term: with pre-activations of O(10) that is a few 1e-6 absolute
    torch.testing.assert_close(act.cpu(), exact, rtol=1e-5, atol=1e-5)   # 1e-5 of the (-1, 1) action range; observed max 6e-6
    act2, _ = pol.step(obs.cuda())
    assert torch.equal(act, act2)                               # deterministic


@pytest.mark.parametrize("prec,atol", [("f16x3_tc", 1e-5), ("f16_tc", 5e-3)])
@pytest.mark.parametrize("E,n_a,D,H,A", [(9, 30, 188, 180, 2), (4, 50, 192, 64, 3), (2, 33, 100, 192, 4), (1, 5, 16, 8, 1)])
def test_tensor_core_paths_with_other_network_sizes(prec, atol, E, n_a, D, H, A):
    """Zero padding of the tensor-core paths: obs_dim < 192 (is_con_self_state=False gives 188), hidden < 192, act_dim 1..4
    (partial outputs exchanged between the two epilogue warps of a row)."""
    torch.manual_seed(E * 100 + A)
    ref = RefMLP(D, A, H)
    with torch.no_grad():
        for p in ref.parameters():
            p.mul_(2.0)
    obs = torch.randn(E, D, n_a) * 0.6
    pol = DevicePolicy(D, A, H, precision=prec).load_state_dict(ref.state_dict())
    act, _ = pol.step(obs.cuda())
    with torch.no_grad():
        want = exact_forward(ref, obs.permute(0, 2, 1).reshape(E * n_a, D)).reshape(E, n_a, A).permute(0, 2, 1)
    torch.testing.assert_close(act.cpu(), want, rtol=1e-5 if prec == "f16x3_tc" else 0, atol=atol)


def test_tensor_core_path_rejects_wide_actions():
    from marl_llm_b200._lib import SwarmError
    pol = DevicePolicy(192, 6, 180)
    with pytest.raises(SwarmError):
        pol.set_precision("f16_tc")


@pytest.mark.parametrize("prec,atol", [("fp32", 0.0), ("f16x3_tc", 0.0), ("f16_tc", 0.0)])
def test_agent_major_observations_give_identical_actions(prec, atol):
    """swarm_policy_obs_layout: the same observations as agent-major rows [E, n_a, obs_dim] (what an agent-major simulator or
    a replay-ring slot holds) must give bit-identical actions for every policy kernel — only the loaders' addresses differ."""
    import torch.nn as nn
    from marl_llm_b200.policy import DevicePolicy
    E, n_a, D = 67, 30, 192
    torch.manual_seed(1)
    sd = {}
    for name, (o, i) in (("fc1", (180, D)), ("fc2", (180, 180)), ("fc3", (180, 180)), ("fc4", (2, 180))):
        l = nn.Linear(i, o); sd[name + ".weight"] = l.weight; sd[name + ".bias"] = l.bias
    pol = DevicePolicy(D, 2, 180, precision=prec).load_state_dict(sd)
    obs = torch.randn(E, D, n_a, device="cuda")
    a_ref, _ = pol.step(obs)
    a_ref = a_ref.clone()
    a_am, _ = pol.step(obs.transpose(1, 2).contiguous(), agent_major=True)
    assert torch.equal(a_ref, a_am)
    a_back, _ = pol.step(obs)                       # the layout switch is per call
    assert torch.equal(a_ref, a_back)
