"""CPU: the drop-in really drops in.  INTEGRATION.md section 2 re-binds the `Epipolar` name of the reference's PoseResNet
(modeling/backbones/resnet.py:257-305) to ours; a checkpoint of the reference-built model must then load strictly and the
model's call (resnet.py:385-387) must find the same forward parameters.  What the reference model expects of its
`epipolar_sampler` is frozen in tests/golden/pose_resnet_epipolar_sampler.json by oracle/make_golden_dropin.py."""
import inspect
import json
import os

import torch

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pose_resnet_epipolar_sampler.json")))


def test_epipolar_drops_into_reference_pose_resnet():
    import epipolar_transformers_b200 as epi
    ours = epi.cfg_h36m_r50_256()                        # configs/epipolar/keypoint_h36m_zresidual_fixed.yaml shape
    m_new = epi.Epipolar(cfg=ours)
    want = GOLD["sampler_state"]
    assert set(m_new.state_dict()) == set(want)                          # identical parameter / buffer names
    # a state dict shaped like the reference model's `epipolar_sampler.*` entries, with values to check the load
    gen = torch.Generator().manual_seed(0)
    sd = {k: (torch.randn(v["shape"], generator=gen).to(getattr(torch, v["dtype"])) if v["dtype"].startswith("float")
              else torch.full(v["shape"], 7, dtype=getattr(torch, v["dtype"])))
          for k, v in want.items()}
    res = m_new.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in m_new.state_dict().items():
        assert v.dtype == sd[k].dtype and torch.equal(v, sd[k]), k
    for k in ("z.weight", "z.bias", "bn.weight", "bn.bias", "bn.running_mean", "bn.running_var"):
        assert list(getattr_path(m_new, k).shape) == want[k]["shape"]
    # the forward signature the caller uses (resnet.py:385-387): positional feats/KRTs + camera kwargs
    params = list(inspect.signature(m_new.forward).parameters)
    assert params[:4] == ["feat1", "feat2", "P1", "P2"] and "camera" in params and "other_camera" in params
    assert params == GOLD["forward_params"]


def getattr_path(obj, path):
    for part in path.split("."):
        obj = getattr(obj, part)
    return obj
