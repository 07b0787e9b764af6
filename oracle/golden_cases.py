"""TEST INFRASTRUCTURE — the golden-vector case list shared by oracle/make_golden.py (which
runs the reference in the build container) and tests/ (which replay the frozen outputs).

Inputs are never stored: they are regenerated from seeds by
epipolar_transformers_b200.synthetic (numpy PCG64, platform independent).  Small cases freeze
every output tensor; the BASELINE-sized cases freeze a per-item subsample of pixels (the
reference's own sample locations, attention weights, fused feature and correspondence at
those pixels) plus float64 checksums.
"""
from __future__ import annotations

import numpy as np

from epipolar_transformers_b200 import config, synthetic as syn

# name -> spec.  cams: 'ring' | 'ring_jitter' | 'randn'.  img = image side the ring cameras see
# (= feature side * DOWNSAMPLE * resize).  full=True stores all outputs.
CASES = {
    # --- small, every tensor frozen -------------------------------------------------------
    "tiny_ring_z": dict(N=2, C=16, H=16, W=16, K=16, cams="ring", feats="randn", correct=True,
                        z=True, zres=True, full=True),
    "tiny_randn_krt": dict(N=2, C=8, H=12, W=20, K=8, cams="randn", feats="randn", correct=False,
                           z=False, zres=False, full=True),
    "tiny_relu_znores": dict(N=1, C=32, H=16, W=16, K=32, cams="ring_jitter", feats="relu_smooth",
                             correct=True, z=True, zres=False, full=True),
    "tiny_k85": dict(N=3, C=4, H=8, W=8, K=85, cams="ring_jitter", feats="randn", correct=False,
                     z=False, zres=False, full=True),
    "tiny_ds8_resize": dict(N=2, C=8, H=10, W=14, K=12, cams="ring_jitter", feats="randn", correct=True,
                            z=False, zres=False, full=True, ds=8, image_resize=2.0, predict_resize=0.5),
    "tiny_zero_query": dict(N=1, C=8, H=8, W=8, K=8, cams="ring", feats="randn", correct=True,
                            z=False, zres=False, full=True, zero_query=True),
    # --- BASELINE.json shapes, subsampled -------------------------------------------------
    "cfg1_randn_krt": dict(N=2, C=64, H=64, W=64, K=32, cams="randn", feats="randn", correct=False,
                           z=False, zres=False, full=False),
    "cfg1_ring": dict(N=2, C=64, H=64, W=64, K=32, cams="ring", feats="randn", correct=True,
                      z=False, zres=False, full=False),
    "cfg2_r50_256": dict(N=4, C=256, H=64, W=64, K=64, cams="ring", feats="relu_smooth", correct=True,
                         z=True, zres=True, full=False),
    "cfg2_r50_256_randn": dict(N=4, C=256, H=64, W=64, K=64, cams="ring", feats="randn", correct=True,
                               z=True, zres=True, full=False),
    "cfg3_r152_384": dict(N=4, C=256, H=96, W=96, K=64, cams="ring", feats="relu_smooth", correct=False,
                          z=False, zres=False, full=False),
}

SUBSAMPLE = 48     # pixels per item frozen for the big cases
DENSE = 128        # pixels per item of the dense fixtures (<case>_dense.npz) of the BASELINE-sized cases below;
                   # sized so that each fixture stays under 1 MB
DENSE_CASES = ("cfg2_r50_256_randn", "cfg3_r152_384")


def case_cfg(spec):
    par = ("z",) if spec["z"] else ()
    return config.make_cfg(
        BACKBONE=dict(DOWNSAMPLE=spec.get("ds", 4)),
        KEYPOINT=dict(HEATMAP_SIZE=(spec["H"], spec["W"]), NFEATS=spec["C"]),
        DATASETS=dict(IMAGE_RESIZE=spec.get("image_resize", 1.0), PREDICT_RESIZE=spec.get("predict_resize", 1.0)),
        EPIPOLAR=dict(SAMPLESIZE=spec["K"], PARAMETERIZED=par, ZRESIDUAL=spec["zres"],
                      USE_CORRECT_NORMALIZE=spec["correct"]),
    )


def case_seed(name):
    return sum(ord(ch) * (i + 1) for i, ch in enumerate(name)) % 100003


def build_inputs(name):
    """-> cfg, feat_ref, feat_src (float32 NCHW), P_ref, P_src (float32 [N,3,4]), params|None."""
    spec = CASES[name]
    seed = case_seed(name)
    cfg = case_cfg(spec)
    N, C, H, W = spec["N"], spec["C"], spec["H"], spec["W"]
    img = int(max(H, W) * spec.get("ds", 4) * spec.get("image_resize", 1.0) * spec.get("predict_resize", 1.0))
    if spec["cams"] == "randn":
        P1, P2 = syn.random_krt(N, seed)
    else:
        jitter = 300.0 if spec["cams"] == "ring_jitter" else 0.0
        P1, P2 = syn.pairs_from_ring(max(N, 2), img, seed=seed, jitter=jitter)
        P1, P2 = P1[:N], P2[:N]
    f1 = syn.features(N, C, H, W, spec["feats"], seed + 1)
    f2 = syn.features(N, C, H, W, spec["feats"], seed + 2)
    if spec.get("zero_query"):
        f1[:, :, 2:4, 3:6] = 0.0          # all-zero query pixels: every sim == 0 -> uniform softmax
    params = syn.z_bn_params(C, seed) if spec["z"] else None
    # the reference receives float32 KRTs (modeling/model.py:183-195)
    return cfg, f1, f2, P1.astype(np.float32), P2.astype(np.float32), params


def subsample_pixels(name):
    """Deterministic [N, SUBSAMPLE, 2] (y, x) pixel picks for the big cases."""
    spec = CASES[name]
    rng = np.random.default_rng(case_seed(name) + 5)
    ys = rng.integers(0, spec["H"], size=(spec["N"], SUBSAMPLE))
    xs = rng.integers(0, spec["W"], size=(spec["N"], SUBSAMPLE))
    return np.stack([ys, xs], -1)


def dense_pixels(name):
    """Deterministic [N, DENSE, 2] (y, x) picks WITHOUT repetition for the dense fixtures."""
    spec = CASES[name]
    rng = np.random.default_rng(case_seed(name) + 11)
    out = np.zeros((spec["N"], DENSE, 2), dtype=np.int64)
    for n in range(spec["N"]):
        flat = rng.choice(spec["H"] * spec["W"], size=DENSE, replace=False)
        out[n, :, 0] = flat // spec["W"]
        out[n, :, 1] = flat % spec["W"]
    return out
