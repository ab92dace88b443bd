#!/usr/bin/env python
"""Record tests/golden/oracle_pins.npz: the digests of tests/oracle_cases.py, computed by the C restatement (oracle/).

TEST/FIXTURE INFRASTRUCTURE.  Rerun only after the restatement has been compared with the original MARL-LLM code again
(tests/test_oracle_vs_reference.py, tests/test_replay_oracle.py, where a checkout of it is available) and agreed:

    python tests/golden/make_oracle_pins.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests import oracle_cases as oc          # noqa: E402

if __name__ == "__main__":
    out = {}
    for name in oc.ENV_CASES:
        out["env_" + name], st = oc.run_env_case(name)
        print(name, st)
    for name in oc.STRATEGY_CASES:
        out["strategy_" + name], st = oc.run_strategy_case(name)
        print(name, st)
    out["replay"] = oc.run_replay_case()
    path = os.path.join(HERE, "oracle_pins.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")
