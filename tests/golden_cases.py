"""The golden model cases (tests/golden/model_<name>.npz, made by tests/golden/make_golden.py) as dicts of arrays.

Most cases store everything.  model_c0 (BASELINE config 0) would take 1.9 MB of incompressible float32 that way, so it
stores its outputs only: the inputs are rebuilt here from the seeds the reference run used - the input batch from
torch.Generator, the initial parameters from torch.manual_seed and the constructor, whose initialisation
oracle.bigru_oracle.OracleBiGRU repeats - and must hash to the reference's bytes; the parameters after the step ("q:")
are stored as their difference from the initial ones ("dq:"), which adds back exactly.
"""
import hashlib
import os

import numpy as np


def inputs_sha256(x, params):
    """SHA-256 of the input batch and the initial parameters (state_dict order), as float32 bytes."""
    h = hashlib.sha256(np.ascontiguousarray(x, np.float32).tobytes())
    for p in params:
        h.update(np.ascontiguousarray(p, np.float32).tobytes())
    return h.hexdigest()


def load(golden_dir, name):
    z = np.load(os.path.join(golden_dir, f"model_{name}.npz"))
    case = {k: z[k] for k in z.files}
    if "inputs_sha256" in case:
        _rebuild_inputs(case)
    return case


def _rebuild_inputs(case):
    import torch
    from oracle import bigru_oracle as bo
    B, T, F, H, L, C, bidir = [int(v) for v in case["meta"]]
    param_seed, input_seed = [int(v) for v in case["input_seeds"]]
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(param_seed)
        sd = bo.OracleBiGRU(H, F, C, L, 50, 0.0, False, bool(bidir)).state_dict()
    x = torch.randn(B, T, F, generator=torch.Generator().manual_seed(input_seed)).numpy()
    params = {k: v.numpy().copy() for k, v in sd.items()}
    assert inputs_sha256(x, params.values()) == str(case["inputs_sha256"]), \
        "rebuilt inputs differ from the reference run's (torch's CPU random streams changed?)"
    case["x"] = x
    for k, p in params.items():
        case["p:" + k] = p
        case["q:" + k] = p + case.pop("dq:" + k)
