"""Prior policies as programs (include/swarm_b200.h group 6, DESIGN.md §12).

A prior program is a `robot_policy` written against include/swarm_prior_api.cuh, compiled at run time for sm_100a by NVRTC and
run on the device as the simulator's prior (the fifth output of step()) or as actions:

    prog = PriorProgram(open("my_prior.cu").read())
    sim.set_prior_program(prog)          # the following steps' a_prior come from prog; None = the built-in prior again
    act = prog.actions(sim)              # [E, 2, n_a] float64: prog as the controller, from the current state

A population runs a different program on each group of envs of one batch, so K candidate priors share one step:

    pop = PriorPopulation([prog_a, prog_b], env_program=torch.arange(sim.E) % 2)
    sim.set_prior_population(pop)        # env e's a_prior comes from programs[env_program[e]]
    act = pop.actions(sim)               # every env driven by its own program
    scores = evaluate_priors(sim, pop, steps=200, seed=1)   # per-program mean reward and final metrics

marl_llm_b200/priors/reference_prior.cu is the reference's own policy written this way (the template for generated ones).
"""
import ctypes as C
import os
import threading

import numpy as np

from . import _lib
from ._lib import SwarmError, check

PRIORS_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "priors")
LOG_CAP = 1 << 16
_cache = {}                 # (source, device) -> PriorProgram
_lock = threading.Lock()


def reference_prior_source():
    """Source of marl_llm_b200/priors/reference_prior.cu: the reference's robotPolicy (AssemblyEnv.cpp:1121-1196)."""
    with open(os.path.join(PRIORS_DIR, "reference_prior.cu")) as f:
        return f.read()


def nvrtc_candidates():
    """Where NVRTC is looked for, in order: $CUDA_HOME/lib64, /usr/local/cuda/lib64, torch's nvidia/cuda_nvrtc/lib."""
    dirs = []
    if os.environ.get("CUDA_HOME"):
        dirs.append(os.path.join(os.environ["CUDA_HOME"], "lib64"))
    dirs.append("/usr/local/cuda/lib64")
    try:
        import nvidia
        dirs += [os.path.join(p, "cuda_nvrtc", "lib") for p in nvidia.__path__]
    except ImportError:
        pass
    return [os.path.join(d, "libnvrtc.so.12") for d in dirs]


def find_nvrtc():
    """Path of libnvrtc.so.12, or None."""
    for p in nvrtc_candidates():
        if os.path.isfile(p):
            return p
    return None


def compile_source(source, nvrtc_path=None):
    """source -> (sm_100a CUBIN bytes, NVRTC log).  Host only: needs NVRTC, not a GPU.  Raises SwarmError with the log when the
    source does not compile."""
    lib = _lib.load()
    path = nvrtc_path or find_nvrtc()
    if path is None:
        raise SwarmError("NVRTC (libnvrtc.so.12) not found; tried: " + ", ".join(nvrtc_candidates()))
    src, p = source.encode(), path.encode()
    size, log = C.c_int64(0), C.create_string_buffer(LOG_CAP)
    rc = lib.swarm_prior_compile(src, p, None, 0, C.byref(size), log, LOG_CAP)
    if rc != _lib.SWARM_OK:
        check(rc, "swarm_prior_compile")
    image = C.create_string_buffer(size.value)
    check(lib.swarm_prior_compile(src, p, image, size.value, C.byref(size), log, LOG_CAP), "swarm_prior_compile")
    return image.raw[:size.value], log.value.decode("utf-8", "replace")


class PriorProgram:
    """A robot_policy compiled and loaded on one device.  Programs are cached per (source, device): constructing the same one
    twice returns the loaded program.  Keep it alive while a simulator uses it (set_prior_program keeps a reference)."""

    def __new__(cls, source, device=0):
        key = (source, int(device))
        with _lock:
            prog = _cache.get(key)
            if prog is None:
                prog = super().__new__(cls)
                prog._load(source, int(device))
                _cache[key] = prog
        return prog

    def __init__(self, source, device=0):
        pass

    def _load(self, source, device):
        self.lib = _lib.load()
        self.source, self.device = source, device
        self.image, self.log = compile_source(source)
        h = C.c_void_p()
        check(self.lib.swarm_prior_program_create(device, self.image, len(self.image), C.byref(h)), "swarm_prior_program_create")
        self._h = h

    @property
    def handle(self):
        return self._h

    def actions(self, sim, out=None):
        """The program as the controller: [E, 2, n_a] float64 CUDA tensor of its output for sim's current state and the
        neighbour list of its last observation (pass it to sim.step())."""
        import torch
        if out is None:
            out = torch.empty(sim.E, 2, sim.n_a, dtype=torch.float64, device=sim.device)
        assert out.is_cuda and out.dtype == torch.float64 and out.is_contiguous() and out.numel() == sim.E * 2 * sim.n_a
        check(self.lib.swarm_prior_program_actions(sim._h, self._h, C.c_void_p(out.data_ptr()), sim._stream()),
              "swarm_prior_program_actions")
        return out


class PriorPopulation:
    """K loaded programs and the program env_program[e] of every env e of a handle with E = len(env_program) envs
    (include/swarm_b200.h swarm_prior_population_create).  Each program runs on its own envs only.  The population keeps
    references to its programs; install it with sim.set_prior_population(pop)."""

    def __init__(self, programs, env_program, device=0):
        import torch
        self.lib = _lib.load()
        self.programs = list(programs)
        if isinstance(env_program, torch.Tensor):
            env_program = env_program.cpu().numpy()
        self.env_program = np.ascontiguousarray(env_program, dtype=np.int32).reshape(-1)
        self.device, self.E, self.K = int(device), int(self.env_program.shape[0]), len(self.programs)
        handles = (C.c_void_p * max(self.K, 1))(*[p.handle.value if p is not None else None for p in self.programs])
        h = C.c_void_p()
        check(self.lib.swarm_prior_population_create(self.device, self.E, self.K, handles, C.c_void_p(self.env_program.ctypes.data),
                                                     C.byref(h)), "swarm_prior_population_create")
        self._h = h

    @property
    def handle(self):
        return self._h

    def close(self):
        if getattr(self, "_h", None):
            self.lib.swarm_prior_population_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def actions(self, sim, out=None):
        """Every env's program as its controller: [E, 2, n_a] float64 CUDA tensor, env e's rows from programs[env_program[e]],
        for sim's current state and the neighbour list of its last observation."""
        import torch
        if out is None:
            out = torch.empty(sim.E, 2, sim.n_a, dtype=torch.float64, device=sim.device)
        assert out.is_cuda and out.dtype == torch.float64 and out.is_contiguous() and out.numel() == sim.E * 2 * sim.n_a
        check(self.lib.swarm_prior_population_actions(sim._h, self._h, C.c_void_p(out.data_ptr()), sim._stream()),
              "swarm_prior_population_actions")
        return out


def evaluate_priors(sim, population, steps, seed):
    """Ranks the population's programs by how well they drive the swarm: sim.reset(seed), then `steps` times
    sim.step(population.actions(sim)).  Returns a dict of [K] float64 CUDA tensors, per program: `reward`, the mean reward over
    the steps and the program's envs and agents (accumulated in float64), and `coverage_rate`, `distribution_uniformity`,
    `voronoi_based_uniformity`, the means over the program's envs of sim.metrics() after the last step (NaN for a program
    without envs).  Everything stays on the device."""
    import torch
    dev = sim.device
    groups = [torch.from_numpy(np.flatnonzero(population.env_program == k)).to(dev) for k in range(population.K)]
    sim.reset(seed)
    act = torch.empty(sim.E, 2, sim.n_a, dtype=torch.float64, device=dev)
    reward = torch.zeros(sim.E, dtype=torch.float64, device=dev)           # per env, summed over agents and steps
    for _ in range(steps):
        population.actions(sim, out=act)
        _, rew, _, _, _ = sim.step(act)
        reward += rew.reshape(sim.E, sim.n_a).to(torch.float64).sum(1)
    met = sim.metrics()
    # per program a sum over its envs in ascending env id (no atomics: the result is a function of those envs alone)
    res = {"reward": torch.stack([reward[g].sum() / (g.numel() * steps * sim.n_a) for g in groups])}
    for j, name in enumerate(("coverage_rate", "distribution_uniformity", "voronoi_based_uniformity")):
        res[name] = torch.stack([met[g, j].sum() / g.numel() for g in groups])
    return res
