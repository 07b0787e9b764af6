"""TEST INFRASTRUCTURE — generator of tests/golden/pose_resnet_epipolar_sampler.json.  Needs the reference source tree
(oracle/ref_harness.py, EPI_REFERENCE_ROOT):
    python -m oracle.make_golden_dropin
Builds the UNMODIFIED reference PoseResNet (modeling/backbones/resnet.py:257-305) at the
configs/epipolar/keypoint_h36m_zresidual_fixed.yaml shape and freezes what a drop-in `Epipolar` has to match there: the
names, shapes and dtypes of the `epipolar_sampler.*` entries of the model's state dict, and the parameter names of the
reference `Epipolar.forward` that the model calls (resnet.py:385-387)."""
from __future__ import annotations

import importlib
import inspect
import json
import os
import sys
import tempfile
import types
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh      # noqa: E402

PREFIX = "epipolar_sampler."


def import_reference_resnet():
    warnings.filterwarnings("ignore")
    _, ref_cfg = rh.load_reference()
    import PIL
    if not hasattr(PIL, "PILLOW_VERSION"):               # the reference targets Pillow < 7 (data/transforms/image.py:6)
        PIL.PILLOW_VERSION = PIL.__version__
    R = rh.REFERENCE_ROOT
    for name, sub in (("modeling.backbones", ("modeling", "backbones")), ("data", ("data",)),
                      ("data.transforms", ("data", "transforms")), ("utils", ("utils",))):
        if name not in sys.modules:                      # leaf packages only: modeling/__init__.py pulls the whole model zoo
            pkg = types.ModuleType(name)
            pkg.__path__ = [os.path.join(R, *sub)]
            sys.modules[name] = pkg
    ref_cfg.FOLDER_NAME = tempfile.mkdtemp()             # resnet.py:16 opens a log file there at import time
    return importlib.import_module("modeling.backbones.resnet"), ref_cfg


def main():
    import torch
    import epipolar_transformers_b200 as epi
    rn, ref_cfg = import_reference_resnet()
    rh.apply_cfg(ref_cfg, epi.cfg_h36m_r50_256())
    ref_cfg.BACKBONE.BODY = "epipolarposeR-50"
    m = rn.PoseResNet(rn.Bottleneck, [3, 4, 6, 3], ref_cfg)                # resnet.py:299-305 instantiates Epipolar()
    sd = m.state_dict()
    out = {"meta": "reference PoseResNet(Bottleneck, [3, 4, 6, 3]) with BODY=epipolarposeR-50 at the cfg_h36m_r50_256 shape, "
                   "torch %s" % torch.__version__.split("+")[0],
           "sampler_state": {k[len(PREFIX):]: {"shape": list(v.shape), "dtype": str(v.dtype).replace("torch.", "")}
                             for k, v in sd.items() if k.startswith(PREFIX)},
           "forward_params": list(inspect.signature(type(m.epipolar_sampler).forward).parameters)[1:]}
    path = os.path.join(ROOT, "tests", "golden", "pose_resnet_epipolar_sampler.json")
    json.dump(out, open(path, "w"), indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
