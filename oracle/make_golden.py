"""TEST INFRASTRUCTURE — freezes outputs of the UNMODIFIED reference module as golden vectors.

Run in the build container only (needs /root/reference):
    python -m oracle.make_golden            # writes tests/golden/<case>.npz

The reference has no tests or fixtures for this path (SURVEY.md section 4); these files are
the pin for oracle/epipolar_oracle.py, oracle/epi_oracle.c and for the CUDA path.  Each file
records the reference commit and the torch version that produced it (the numerics live in
torch: F.grid_sample default align_corners=False, softmax, pinverse).
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import golden_cases as gc   # noqa: E402
from oracle import ref_harness as rh    # noqa: E402


def main(names=None):
    import torch
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    meta = {"torch": torch.__version__, "reference_commit": "unknown"}
    sub = os.path.join(rh.REFERENCE_ROOT, ".SUBMODULES.json")
    if os.path.exists(sub):
        try:
            meta["reference_commit"] = json.load(open(sub)).get("commit", "unknown")
        except Exception:
            pass
    for name in (names or gc.CASES):
        spec = gc.CASES[name]
        cfg, f1, f2, P1, P2, params = gc.build_inputs(name)
        r = rh.run_reference(cfg, f1, f2, P1, P2, params=params)
        H, W = spec["H"], spec["W"]
        locs64 = rh.reference_sample_locs(cfg, P1, P2, H, W, dtype="float64")   # T2 truth (fp64 geometry)
        rec = {"meta": json.dumps(dict(meta, case=name, spec=spec))}
        for k in ("out", "attn", "corr_pos"):
            rec["sum_" + k] = np.float64(r[k].astype(np.float64).sum())
            rec["abssum_" + k] = np.float64(np.abs(r[k].astype(np.float64)).sum())
        if spec["full"]:
            rec.update(out=r["out"], attn=r["attn"], corr_pos=r["corr_pos"],
                       sample_locs=r["sample_locs"], sample_locs_fp64=locs64.astype(np.float64))
        else:
            px = gc.subsample_pixels(name)                      # [N,S,2] (y,x)
            n_idx = np.arange(spec["N"])[:, None]
            yy, xx = px[..., 0], px[..., 1]
            rec.update(
                pixels=px,
                out=r["out"][n_idx, :, yy, xx],                 # [N,S,C]
                attn=r["attn"][n_idx, :, yy, xx],               # [N,S,K]
                corr_pos=r["corr_pos"][n_idx, yy, xx],          # [N,S,2]
                sample_locs=r["sample_locs"].transpose(1, 2, 3, 0, 4)[n_idx, yy, xx],        # [N,S,K,2]
                sample_locs_fp64=locs64.transpose(1, 2, 3, 0, 4)[n_idx, yy, xx],
            )
        path = os.path.join(out_dir, name + ".npz")
        np.savez_compressed(path, **rec)
        print("%-22s %8.1f KB  out|max|=%.4g" % (name, os.path.getsize(path) / 1024, np.abs(r["out"]).max()))
        if name in gc.DENSE_CASES:                              # DENSE pixels per item: T1/T3 at BASELINE shapes with real coverage
            px = gc.dense_pixels(name)
            n_idx = np.arange(spec["N"])[:, None]
            yy, xx = px[..., 0], px[..., 1]
            dense = dict(meta=rec["meta"], pixels=px, out=r["out"][n_idx, :, yy, xx], attn=r["attn"][n_idx, :, yy, xx],
                         corr_pos=r["corr_pos"][n_idx, yy, xx],
                         sample_locs=r["sample_locs"].transpose(1, 2, 3, 0, 4)[n_idx, yy, xx],
                         out_absmax=np.float64(np.abs(r["out"]).max()))
            path = os.path.join(out_dir, name + "_dense.npz")
            np.savez_compressed(path, **dense)
            print("%-22s %8.1f KB  (dense)" % (name, os.path.getsize(path) / 1024))


if __name__ == "__main__":
    main(sys.argv[1:] or None)
