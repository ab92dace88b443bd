"""Prior policies as programs (include/swarm_b200.h group 6, DESIGN.md §12).

A prior program is a `robot_policy` written against include/swarm_prior_api.cuh, compiled at run time for sm_100a by NVRTC and
run on the device as the simulator's prior (the fifth output of step()) or as actions:

    prog = PriorProgram(open("my_prior.cu").read())
    sim.set_prior_program(prog)          # the following steps' a_prior come from prog; None = the built-in prior again
    act = prog.actions(sim)              # [E, 2, n_a] float64: prog as the controller, from the current state

marl_llm_b200/priors/reference_prior.cu is the reference's own policy written this way (the template for generated ones).
"""
import ctypes as C
import os
import threading

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
