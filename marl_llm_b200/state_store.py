"""Save env states of a BatchedAssemblySim on the device and load them back (`swarm_state_*`, include/swarm_b200.h).

    store = StateStore(sim, capacity=64)
    store.save([3, 7])                 # slots 0, 1 <- envs 3, 7
    ...                                # step, reset, install other grids
    store.load([0, 0, 1], [3, 4, 7])   # envs 3 and 4 <- the saved env 3, env 7 <- the saved env 7

Every step after a load is bit-identical to the run the saved envs would have continued (DESIGN.md §11).  A store serves every
handle of the configuration it was created for (`load(..., sim=other)`), whatever its num_envs.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import check


def _ids(v):
    return np.ascontiguousarray(np.asarray(v, dtype=np.int64).reshape(-1), dtype=np.int32)


class StateStore:
    """`capacity` slots of device memory on sim's device, each holding one env's complete state."""

    def __init__(self, sim, capacity):
        self.sim, self.lib = sim, _lib.load()
        self.capacity = int(capacity)
        h = C.c_void_p()
        check(self.lib.swarm_state_store_create(sim._h, self.capacity, C.byref(h)), "swarm_state_store_create")
        self._h = h
        # host mirrors of the handle (BatchedAssemblySim.n_g / l_cell) for the saved envs
        self._n_g = np.zeros(self.capacity, dtype=np.int32)
        self._l_cell = np.zeros(self.capacity)

    @property
    def slot_bytes(self):
        return int(self.lib.swarm_state_slot_bytes(self._h))

    def save(self, env_ids, slots=None):
        """Slot slots[k] <- env env_ids[k] of the store's handle (slots distinct; default 0 .. count - 1).  Stream-ordered."""
        env_ids = _ids(env_ids)
        slots = np.arange(env_ids.shape[0], dtype=np.int32) if slots is None else _ids(slots)
        if slots.shape != env_ids.shape:
            raise ValueError("env_ids and slots must have the same length")
        check(self.lib.swarm_state_save(self.sim._h, self._h, C.c_void_p(env_ids.ctypes.data), C.c_void_p(slots.ctypes.data),
                                        int(env_ids.shape[0]), self.sim._stream()), "swarm_state_save")
        self._n_g[slots] = self.sim.n_g[env_ids]
        self._l_cell[slots] = self.sim.l_cell[env_ids]

    def load(self, slots, env_ids, sim=None):
        """Env env_ids[k] <- slot slots[k] (env ids distinct, slots may repeat: one state into many envs), into the store's
        handle or `sim`, another handle of the same configuration.  Stream-ordered."""
        sim = self.sim if sim is None else sim
        slots, env_ids = _ids(slots), _ids(env_ids)
        if slots.shape != env_ids.shape:
            raise ValueError("slots and env_ids must have the same length")
        check(self.lib.swarm_state_load(sim._h, self._h, C.c_void_p(slots.ctypes.data), C.c_void_p(env_ids.ctypes.data),
                                        int(env_ids.shape[0]), sim._stream()), "swarm_state_load")
        sim.n_g[env_ids] = self._n_g[slots]
        sim.l_cell[env_ids] = self._l_cell[slots]

    def close(self):
        if getattr(self, "_h", None):
            self.lib.swarm_state_store_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
