"""TEST INFRASTRUCTURE ONLY -- imports an unmodified checkout of the reference from $CCVPE_REFERENCE_ROOT.

This module exists solely so that `oracle/make_golden.py` can execute the real reference (tudelft-iv/CCVPE, GPL-3,
not part of this repository) to pin the oracle restatement in `oracle/ccvpe_oracle.py`.  The tests, smoke() and
bench.py never need the reference checkout.

Two shims, no edits to the reference (SURVEY.md section 8(c)):
  * models.py:8-9 import IPython / matplotlib which are not installed -> empty stub modules.
  * efficientnet_pytorch/model.py:407 downloads ImageNet weights -> no-op ("random-init").
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("CCVPE_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "models.py"))


def load_reference_models():
    """Returns the reference `models` module (CVM_VIGOR, CVM_VIGOR_ori_prior, CVM_KITTI, CVM_OxfordRobotCar)."""
    if not available():
        raise RuntimeError("reference checkout not present at %s" % REFERENCE_ROOT)
    for name in ("IPython", "IPython.display", "matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["IPython.display"].Image = object
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import torch

    rng_state = torch.get_rng_state()
    import efficientnet_pytorch.model as ref_effnet_model  # noqa: E402  (the reference's vendored encoder)

    ref_effnet_model.load_pretrained_weights = lambda *a, **k: None
    # the reference's top-level module is also called "models"; load it under a private name so
    # it can never shadow anything of ours.
    import importlib.util

    spec = importlib.util.spec_from_file_location("_ccvpe_reference_models", os.path.join(REFERENCE_ROOT, "models.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["_ccvpe_reference_models"] = mod
    spec.loader.exec_module(mod)  # NB: reseeds torch(17)/numpy(0) at import (models.py:16-17)
    torch.set_rng_state(rng_state)
    return mod
