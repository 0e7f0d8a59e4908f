"""Shared helpers for the parity tests: golden loading, seeded weights/inputs, error measures."""
import os

import numpy as np
import torch

from sepreformer_b200.configs import MODEL_SHAPES
from sepreformer_b200.params import ParamTree, separator_spec, seeded_state, state_shapes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# the runnable copy of the reference's model files (oracle/install_reference.py, run by build(); git-ignored)
REF_COPY = os.path.join(os.path.dirname(os.path.dirname(GOLDEN)), "oracle", "_ref")
REF_DIR = REF_COPY if os.path.isdir(os.path.join(REF_COPY, "models")) else None


def reference_model_module(name):
    """Import ``models.<name>.model`` of the reference (from oracle/_ref) with its logger silenced."""
    import importlib
    import sys
    if REF_DIR is None:
        raise RuntimeError("reference files not available")
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    from loguru import logger
    logger.remove()
    return importlib.import_module(f"models.{name}.model")


def reference_model_config(name):
    import yaml
    return yaml.full_load(open(os.path.join(REF_DIR, "models", name, "configs.yaml")))["config"]["model"]

_state_cache = {}


def seeded_input(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def model_state(model_name, wseed):
    """The seeded separator state_dict for ``model_name`` (cached; ~56-220 MB each)."""
    key = (model_name, wseed)
    if key not in _state_cache:
        shape = MODEL_SHAPES[model_name]
        _state_cache[key] = seeded_state(state_shapes(ParamTree(separator_spec(shape))), seed=wseed)
    return _state_cache[key]


def load_golden(tag):
    z = np.load(os.path.join(GOLDEN, tag + ".npz"))
    return {k: z[k] for k in z.files}


def check_generator_stable(gold, sd, x=None):
    """Guard: the stored checksums must match what this machine's generator produces."""
    if "wsum" in gold:
        for k, s in zip(gold["wkeys"], gold["wsum"]):
            got = float(sd[str(k)].double().abs().sum())
            assert abs(got - float(s)) <= 1e-6 * max(1.0, abs(float(s))), f"seeded weights drifted at {k}"
    if x is not None and "xsum" in gold:
        got = float(x.double().abs().sum())
        assert abs(got - float(gold["xsum"])) <= 1e-6 * float(gold["xsum"]), "seeded input drifted"


def rel_l2(a, b):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    return float((a - b).norm() / b.norm())


def max_rel(a, b):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    return float((a - b).abs().max() / b.abs().max())
