"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI, against
(a) golden vectors frozen from the reference and (b) the CPU oracle on the same seeded inputs.

Protocol (SURVEY.md section 8c; fp32, tolerance 1e-4 relative to max|ref| as north_star states):
  T1  inject the reference's own sample locations -> out / attn / corr_pos vs reference
  T2  fused geometry vs the reference's geometry evaluated in fp64 (feature-pixel error)
  T3  end to end: kernel's own locations are emitted, the oracle consumes them, strict compare
"""
import numpy as np
import pytest
import torch

import epipolar_transformers_b200 as epi
from oracle import c_oracle, epipolar_oracle as eo, golden_cases as gc
from tests.util import load_golden, px_err, rel_max

pytestmark = pytest.mark.gpu
TOL = 1e-4
FULL = [n for n, s in gc.CASES.items() if s["full"]]
BIG = [n for n, s in gc.CASES.items() if not s["full"]]
VARIANTS = ["warp", "auto"]          # auto = the pipelined tensor-core kernel wherever the shape allows
DENSE = list(gc.DENSE_CASES)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def fold_params(params, zres, bn_eps=1e-5):
    s = params["bn.weight"] / np.sqrt(params["bn.running_var"] + bn_eps)
    wf = (s[:, None] * params["z.weight"].reshape(len(s), -1)).astype(np.float32)
    bf = (s * (params["z.bias"] - params["bn.running_mean"]) + params["bn.bias"]).astype(np.float32)
    return dev(wf), dev(bf)


def run_kernel(name, locs_in=None, variant="auto", want_locs=True, channels_last=False, **kw):
    cfg, f1, f2, P1, P2, params = gc.build_inputs(name)
    spec = gc.CASES[name]
    t1, t2 = dev(f1), dev(f2)
    if channels_last:
        t1 = t1.contiguous(memory_format=torch.channels_last)
        t2 = t2.contiguous(memory_format=torch.channels_last)
    zf = fold_params(params, spec["zres"]) if params else None
    out, corr, attn, locs = epi.epipolar_fusion(
        t1, t2, dev(P1), dev(P2), K=spec["K"], downsample=cfg.BACKBONE.DOWNSAMPLE,
        img_scale=cfg.DATASETS.IMAGE_RESIZE * cfg.DATASETS.PREDICT_RESIZE, softmax_scale=cfg.EPIPOLAR.SOFTMAXSCALE,
        correct_normalize=spec["correct"], z_folded=zf, z_residual=spec["zres"],
        sample_locs_in=dev(locs_in) if locs_in is not None else None, want_locs=want_locs, variant=variant, **kw)
    torch.cuda.synchronize()
    return (cfg, f1, f2, P1, P2, params), dict(out=out.cpu().numpy(), corr_pos=corr.cpu().numpy(), attn=attn.cpu().numpy(),
                                               sample_locs=locs.cpu().numpy() if locs is not None else None)


def corr_agree(got, want):
    """fraction of pixels whose arg-max correspondence is identical (ties between equal softmax
    weights may legitimately resolve to another sample)."""
    return float((np.abs(got - want).max(-1) < 1e-3).mean())


def assert_corr_exact_or_tie(got_corr, ref_corr, ref_attn, ref_locs, H, W, correct, rel=1e-6):
    """Index work is judged exactly: every pixel's correspondence must equal the reference's, except where the
    reference's own attention row has a near-tie between the two samples (|a[k_ours] - a[k_ref]| <= rel * max a),
    which fp32 summation order can legitimately resolve either way.
    got_corr/ref_corr [...,2]; ref_attn [...,K]; ref_locs [...,K,2] (normalised grid coordinates)."""
    got_corr = np.asarray(got_corr, np.float64).reshape(-1, 2)
    ref_corr = np.asarray(ref_corr, np.float64).reshape(-1, 2)
    K = ref_attn.shape[-1]
    ref_attn = np.asarray(ref_attn, np.float64).reshape(-1, K)
    locs = np.asarray(ref_locs, np.float64).reshape(-1, K, 2)
    bad = np.nonzero(np.abs(got_corr - ref_corr).max(-1) >= 1e-3)[0]
    size = np.array([W, H], np.float64)
    for i in bad:
        cand = (locs[i] + 1) * (size - 1) / 2 if correct else (locs[i] + 1) * size / 2 - 0.5       # de_normalize, multiview.py:39-57
        k_ours = int(np.abs(cand - got_corr[i]).max(-1).argmin())
        assert np.abs(cand[k_ours] - got_corr[i]).max() < 1e-3, "correspondence %s is not a sample of the line" % (got_corr[i],)
        k_ref = int(ref_attn[i].argmax())
        gap = abs(ref_attn[i, k_ours] - ref_attn[i, k_ref])
        assert gap <= rel * ref_attn[i].max(), "pixel %d: arg-max %d vs reference %d is not a tie (gap %.3g)" % (i, k_ours, k_ref, gap)
    return len(bad)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", FULL)
def test_T1_golden_full(name, variant):
    g = load_golden(name)
    _, r = run_kernel(name, locs_in=g["sample_locs"], variant=variant)
    assert rel_max(r["out"], g["out"]) < TOL
    assert rel_max(r["attn"], g["attn"]) < TOL
    spec = gc.CASES[name]
    assert_corr_exact_or_tie(r["corr_pos"], g["corr_pos"], g["attn"].transpose(0, 2, 3, 1),
                             g["sample_locs"].transpose(1, 2, 3, 0, 4), spec["H"], spec["W"], spec["correct"])
    np.testing.assert_array_equal(r["sample_locs"], g["sample_locs"])     # pass-through of injected locations


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", BIG)
def test_T1_golden_subsampled(name, variant):
    """BASELINE-sized shapes: the reference's frozen locations are injected at the frozen pixels
    (the kernel's own geometry everywhere else) and compared there."""
    g = load_golden(name)
    spec = gc.CASES[name]
    _, own = run_kernel(name, variant=variant)
    locs = own["sample_locs"].copy()
    px = g["pixels"]; n_idx = np.arange(spec["N"])[:, None]
    locs.transpose(1, 2, 3, 0, 4)[n_idx, px[..., 0], px[..., 1]] = g["sample_locs"]
    _, r = run_kernel(name, locs_in=locs, variant=variant)
    assert rel_max(r["out"][n_idx, :, px[..., 0], px[..., 1]], g["out"]) < TOL
    assert rel_max(r["attn"][n_idx, :, px[..., 0], px[..., 1]], g["attn"]) < TOL
    assert_corr_exact_or_tie(r["corr_pos"][n_idx, px[..., 0], px[..., 1]], g["corr_pos"], g["attn"], g["sample_locs"],
                             spec["H"], spec["W"], spec["correct"])


@pytest.mark.parametrize("name", DENSE)
def test_T1_T3_dense_baseline_shapes(name, capsys):
    """BASELINE shapes with real coverage: 128 frozen pixels per item (3.1 % / 1.4 % of the cfg2 / cfg3 maps).
    T1: reference locations injected there -> out / attn within 1e-4, correspondences exact up to reference ties.
    T3 (SURVEY.md 8c): the three norms  |kernel - ref_fp32|, |kernel - oracle(fp64 locs)|, |ref_fp32 - oracle(fp64 locs)|
    on those pixels; the kernel's own geometry must be at least as close to the fp64-geometry oracle as the reference is."""
    from tests.util import rel_l2
    gd = load_golden(name + "_dense")
    spec = gc.CASES[name]
    H, W = spec["H"], spec["W"]
    px = gd["pixels"]; n_idx = np.arange(spec["N"])[:, None]
    pick = lambda t, ch_axis=True: (t[n_idx, :, px[..., 0], px[..., 1]] if ch_axis else t[n_idx, px[..., 0], px[..., 1]])
    (cfg, f1, f2, P1, P2, params), own = run_kernel(name)
    locs = own["sample_locs"].copy()
    locs.transpose(1, 2, 3, 0, 4)[n_idx, px[..., 0], px[..., 1]] = gd["sample_locs"]
    _, r = run_kernel(name, locs_in=locs)
    ref_scale = float(gd["out_absmax"])
    e_out = float(np.abs(pick(r["out"]) - gd["out"]).max() / ref_scale)
    assert e_out < TOL, e_out
    assert rel_max(pick(r["attn"]), gd["attn"]) < TOL
    nties = assert_corr_exact_or_tie(pick(r["corr_pos"], False), gd["corr_pos"], gd["attn"], gd["sample_locs"], H, W, spec["correct"])
    # ---- T3: fp64-geometry oracle on the same inputs ----
    locs64 = eo.sample_locs(cfg, P1, P2, H, W, dtype=np.float64).astype(np.float32)
    o64 = c_oracle.forward(cfg, f1, f2, P1, P2, locs=locs64)
    out64 = eo.z_epilogue(o64["out"], params, cfg.EPIPOLAR.ZRESIDUAL) if params else o64["out"]
    k_ref = rel_l2(pick(own["out"]), gd["out"]); k_64 = rel_l2(pick(own["out"]), pick(out64)); r_64 = rel_l2(gd["out"], pick(out64))
    with capsys.disabled():
        print("\nT3 %-20s rel-L2 on %d px: |kernel-ref_fp32| %.3e  |kernel-oracle_fp64locs| %.3e  |ref_fp32-oracle_fp64locs| %.3e  "
              "(T1 max-rel out %.2e, corr ties %d)" % (name, px.shape[0] * px.shape[1], k_ref, k_64, r_64, e_out, nties))
    assert k_64 <= max(r_64, 1e-4)
    if spec["feats"] == "relu_smooth":
        assert k_64 < 1e-4


@pytest.mark.parametrize("name", FULL + BIG)
def test_T2_geometry_vs_fp64(name):
    """Fused fp32 geometry must be at least as close to the fp64 truth as the reference's own
    fp32 locations are (and < 1e-3 feature px on camera-like KRTs)."""
    g = load_golden(name)
    spec = gc.CASES[name]
    H, W = spec["H"], spec["W"]
    cfg, _, _, P1, P2, _ = gc.build_inputs(name)
    locs = epi.sample_locs(dev(P1), dev(P2), H, W, spec["K"], cfg.BACKBONE.DOWNSAMPLE,
                           cfg.DATASETS.IMAGE_RESIZE * cfg.DATASETS.PREDICT_RESIZE, spec["correct"]).cpu().numpy()
    _, r = run_kernel(name, variant="warp")
    # both entry points share the device code (FMA contraction may differ by an ulp between kernels)
    np.testing.assert_allclose(locs, r["sample_locs"], rtol=1e-5, atol=1e-5)
    if not spec["full"]:
        px = g["pixels"]; n_idx = np.arange(spec["N"])[:, None]
        locs = locs.transpose(1, 2, 3, 0, 4)[n_idx, px[..., 0], px[..., 1]]
    err, far_ok = px_err(locs, g["sample_locs_fp64"], H, W)
    ref_err, _ = px_err(g["sample_locs"], g["sample_locs_fp64"], H, W)
    assert far_ok
    if spec["cams"] == "randn":
        assert err < 5e-3, (err, ref_err)
    else:
        assert err < 1e-3 and err <= max(ref_err, 1e-4), (err, ref_err)


@pytest.mark.parametrize("variant", ["warp", "auto", "tile", "sector"])
@pytest.mark.parametrize("name", FULL + BIG)
def test_T3_end_to_end_vs_oracle(name, variant):
    """Own geometry end to end: the locations the kernel sampled are fed to the C oracle.
    ('auto' = epipolar-sector tiles where the shape allows, 'tile' = 4x8 block tiles, 'warp' = CUDA-core kernel.)"""
    if variant in ("tile", "sector") and gc.CASES[name]["C"] % 8 != 0:
        pytest.skip("tensor-core kernel needs C % 8 == 0")
    (cfg, f1, f2, P1, P2, params), r = run_kernel(name, variant=variant)
    o = c_oracle.forward(cfg, f1, f2, P1, P2, locs=r["sample_locs"])
    out = eo.z_epilogue(o["out"], params, cfg.EPIPOLAR.ZRESIDUAL) if params else o["out"]
    assert rel_max(r["out"], out) < TOL
    assert rel_max(r["attn"], o["attn"]) < TOL
    assert corr_agree(r["corr_pos"], o["corr_pos"]) > 0.99
    s = r["attn"].sum(1)
    assert np.abs(s - 1).max() < 1e-5


@pytest.mark.parametrize("name", ["tiny_ring_z", "tiny_randn_krt", "cfg1_ring"])
def test_channels_last_and_residual(name):
    """channels_last strides (zero-copy source) and the fused caller residual give the same numbers."""
    _, base = run_kernel(name)
    (_, f1, _, _, _, _), cl = run_kernel(name, channels_last=True)
    assert rel_max(cl["out"], base["out"]) < 1e-6
    assert rel_max(cl["attn"], base["attn"]) < 1e-6
    _, res = run_kernel(name, add_ref_residual=True)
    assert rel_max(res["out"], base["out"] + f1) < 1e-6


@pytest.mark.parametrize("name", ["tiny_ring_z", "tiny_ds8_resize"])
def test_align_corners_true(name):
    """torch<=1.2 grid_sample semantics as a kernel parameter (SURVEY fact 9), vs the numpy oracle."""
    (cfg, f1, f2, P1, P2, params), r = run_kernel(name, align_corners=True)
    o = eo.forward(cfg, f1, f2, P1, P2, params=params, locs=r["sample_locs"], align_corners=True)
    assert rel_max(r["out"], o["out"]) < TOL
    assert rel_max(r["attn"], o["attn"]) < TOL


def test_module_contract_and_state_dict():
    """nn.Module drop-in: reference parameter names load, 4-tuple contract, eval fold == oracle."""
    name = "tiny_ring_z"
    cfg, f1, f2, P1, P2, params = gc.build_inputs(name)
    cfg.VIS.EPIPOLAR_LINE = True
    m = epi.Epipolar(cfg=cfg).cuda().eval()
    sd = {k: torch.from_numpy(v) for k, v in params.items()}
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and set(missing.missing_keys) <= {"bn.num_batches_tracked"}
    with torch.no_grad():
        out, corr, attn, locs_t = m(dev(f1), dev(f2), dev(P1), dev(P2), camera=None, other_camera=None)
    N, C, H, W = f1.shape
    K = cfg.EPIPOLAR.SAMPLESIZE
    assert out.shape == (N, C, H, W) and corr.shape == (N, H, W, 2) and attn.shape == (N, K, H, W)
    assert locs_t.shape == (N, K, H, W, 2)
    locs = locs_t.transpose(0, 1).contiguous().cpu().numpy()
    o = eo.forward(cfg, f1, f2, P1, P2, params=params, locs=locs)
    assert rel_max(out.cpu().numpy(), o["out"]) < TOL
    # default zero-init BN: z branch contributes nothing, finalout == out (epipolar.py:249-253, BN.py:48-52)
    m0 = epi.Epipolar(cfg=cfg).cuda().eval()
    with torch.no_grad():
        out0 = m0(dev(f1), dev(f2), dev(P1), dev(P2))[0]
    o0 = c_oracle.forward(cfg, f1, f2, P1, P2, locs=locs)
    assert rel_max(out0.cpu().numpy(), o0["out"]) < TOL
    # train mode keeps conv/BN in PyTorch (batch statistics)
    m.train()
    with torch.no_grad():
        out_tr = m(dev(f1), dev(f2), dev(P1), dev(P2))[0]
    pre = torch.from_numpy(o0["out"]).cuda()
    ref_tr = torch.nn.functional.batch_norm(torch.nn.functional.conv2d(pre, m.z.weight, m.z.bias), None, None,
                                            m.bn.weight, m.bn.bias, True, 0.1, 1e-5) + pre
    assert rel_max(out_tr.cpu().numpy(), ref_tr.detach().cpu().numpy()) < 1e-3


@pytest.mark.parametrize("C", [64, 128, 192, 320, 512])
def test_z_epilogue_tensor_core_channel_counts(C):
    """z conv + BN(eval) + ZRESIDUAL on the tensor-core GEMM for every supported channel count (weight box = min(C, 256) rows;
    two blocks of output channels above 256) behind the pipelined kernel (forced: an unsupported shape would be EINVAL)."""
    from epipolar_transformers_b200 import synthetic as syn
    N, H, W, K = 2, 24, 24, 16
    cfg = epi.make_cfg(KEYPOINT=dict(HEATMAP_SIZE=(H, W), NFEATS=C),
                       EPIPOLAR=dict(SAMPLESIZE=K, USE_CORRECT_NORMALIZE=True, PARAMETERIZED=("z",), ZRESIDUAL=True))
    P1, P2 = syn.pairs_from_ring(N, 4 * H)
    P1, P2 = P1.astype(np.float32), P2.astype(np.float32)
    f1, f2 = syn.features(N, C, H, W, "randn", 21), syn.features(N, C, H, W, "randn", 22)
    params = syn.z_bn_params(C, 5)
    out, corr, attn, locs = epi.epipolar_fusion(dev(f1), dev(f2), dev(P1), dev(P2), K=K, correct_normalize=True, want_locs=True,
                                                z_folded=fold_params(params, True), z_residual=True, add_ref_residual=True, variant="pipe")
    torch.cuda.synchronize()
    o = c_oracle.forward(cfg, f1, f2, P1, P2, locs=locs.cpu().numpy())
    want = eo.z_epilogue(o["out"], params, True) + f1
    assert rel_max(out.cpu().numpy(), want) < TOL


def test_fused_caller_residual_module():
    """Epipolar(fuse_ref_residual=True) + fused_other_feat == the reference caller's `ret + feat`
    (modeling/backbones/resnet.py:377-388), with and without the z epilogue; other_features=None passes feat through."""
    for name in ("tiny_ring_z", "cfg1_ring"):
        cfg, f1, f2, P1, P2, params = gc.build_inputs(name)
        base = epi.Epipolar(cfg=cfg).cuda().eval()
        fused = epi.Epipolar(cfg=cfg, fuse_ref_residual=True).cuda().eval()
        if params:
            sd = {k: torch.from_numpy(v) for k, v in params.items()}
            base.load_state_dict(sd, strict=False); fused.load_state_dict(sd, strict=False)
        t1, t2, p1, p2 = dev(f1), dev(f2), dev(P1), dev(P2)
        with torch.no_grad():
            want = epi.fused_other_feat(t1, t2, p1, p2, base)            # unfused sampler: helper adds feat itself
            got = epi.fused_other_feat(t1, t2, p1, p2, fused)            # fused sampler: the kernel already added it
            plain = base(t1, t2, p1, p2)[0]
        assert rel_max(want[0].cpu().numpy(), (plain + t1).cpu().numpy()) < 1e-6
        assert rel_max(got[0].cpu().numpy(), want[0].cpu().numpy()) < 1e-6
        assert torch.equal(got[2], want[2]) and torch.equal(got[1], want[1])
        same = epi.fused_other_feat(t1, None, p1, p2, fused)
        assert same[0] is t1 and same[1] is None


@pytest.mark.parametrize("name", ["cfg1_ring", "tiny_ring_z", "cfg2_r50_256_randn"])
def test_persistent_cache_is_transparent(name):
    """FusionState (persistent workspace + camera-keyed cache of pixel order, pair constants and the fused kernel's work
    items): miss, hit, changed cameras, and back — every call must equal the stateless call bit for bit."""
    cfg, f1, f2, P1, P2, params = gc.build_inputs(name)
    spec = gc.CASES[name]
    kw = dict(K=spec["K"], downsample=cfg.BACKBONE.DOWNSAMPLE, img_scale=cfg.DATASETS.IMAGE_RESIZE * cfg.DATASETS.PREDICT_RESIZE,
              softmax_scale=cfg.EPIPOLAR.SOFTMAXSCALE, correct_normalize=spec["correct"], want_locs=True)
    if params:
        kw.update(z_folded=fold_params(params, spec["zres"]), z_residual=spec["zres"])
    t1, t2 = dev(f1), dev(f2)
    PA = (dev(P1), dev(P2))
    PB = (dev(P1[::-1].copy()), dev(P2[::-1].copy()))               # other cameras in every batch slot
    want = {k: epi.epipolar_fusion(t1, t2, *P, **kw) for k, P in (("A", PA), ("B", PB))}
    state = epi.FusionState()
    for which in ("A", "A", "B", "B", "A"):                          # miss, hit, miss (epoch bump), hit, miss
        got = epi.epipolar_fusion(t1, t2, *(PA if which == "A" else PB), state=state, **kw)
        for g, w in zip(got, want[which]):
            assert torch.equal(g, w), which


def test_errors_are_loud():
    cfg = epi.make_cfg(EPIPOLAR=dict(ATTENTION="max"))
    with pytest.raises(NotImplementedError):
        epi.Epipolar(cfg=cfg)
    m = epi.Epipolar(cfg=epi.make_cfg(KEYPOINT=dict(HEATMAP_SIZE=(8, 8), NFEATS=8), EPIPOLAR=dict(SAMPLESIZE=8)))
    x = torch.zeros(1, 8, 8, 8)
    with pytest.raises(RuntimeError):
        m(x, x, torch.zeros(1, 3, 4), torch.zeros(1, 3, 4))             # CPU tensors: no CPU path
    with pytest.raises(RuntimeError):
        epi.epipolar_fusion(x.cuda(), x.cuda(), torch.zeros(1, 3, 4), torch.zeros(1, 3, 4), K=1)   # EPI_EINVAL


# ---- size-independent properties at BASELINE.json's full shapes --------------------------------
@pytest.mark.parametrize("shape", [(4, 256, 64, 64, 64), (4, 256, 96, 96, 64)])
def test_full_size_properties(shape):
    N, C, H, W, K = shape
    from epipolar_transformers_b200 import synthetic as syn
    P1, P2 = syn.pairs_from_ring(N, 4 * H)
    f1 = dev(syn.features(N, C, H, W, "randn", 3)); f2 = dev(syn.features(N, C, H, W, "randn", 4))
    kw = dict(K=K, correct_normalize=True, want_locs=True)
    out, corr, attn, locs = epi.epipolar_fusion(f1, f2, dev(P1), dev(P2), **kw)
    # (a) softmax weights sum to one; correspondences of pixels with a valid line lie in the map
    #     (pixels whose epipolar line misses the source image keep the reference's far sentinel)
    assert (attn.sum(1) - 1).abs().max().item() < 1e-5
    valid = (locs.abs() < 50).all(-1).all(0)                            # [N,H,W]
    assert valid.float().mean().item() > 0.5
    cv = corr[valid]
    assert cv.min().item() > -1.0 and cv[..., 0].max().item() < W and cv[..., 1].max().item() < H
    # (b) run-to-run determinism, bit exact
    out2 = epi.epipolar_fusion(f1, f2, dev(P1), dev(P2), **kw)[0]
    assert torch.equal(out, out2)
    # (c) pairs are independent: permuting the batch permutes the outputs, bit exact
    perm = torch.tensor([2, 0, 3, 1], device="cuda")
    outp = epi.epipolar_fusion(f1[perm].contiguous(), f2[perm].contiguous(), dev(P1)[perm], dev(P2)[perm], **kw)[0]
    assert torch.equal(outp, out[perm])
    # (d) a spatially constant source map is reproduced wherever all K samples are in bounds
    v = torch.randn(1, C, 1, 1, device="cuda")
    #     (USE_CORRECT_NORMALIZE=False + align_corners=False maps border pixel centres onto border taps exactly)
    kwd = dict(kw, correct_normalize=False)
    outc, _, _, locs = epi.epipolar_fusion(f1, v.expand(N, C, H, W).contiguous(), dev(P1), dev(P2), **kwd)
    lim = torch.tensor([1 - 1.0 / W, 1 - 1.0 / H], device="cuda") + 1e-5
    inb = (locs.abs() <= lim).all(-1).all(0)                            # [N,H,W]: every sample inside the map
    assert inb.float().mean().item() > 0.2
    err = (outc - v).abs().amax(1)[inb].max().item()
    assert err < 1e-4 * v.abs().max().item()
    # (e) linear in the source "values" when the logits are unchanged: zero query => uniform attention
    outz, _, attnz, _ = epi.epipolar_fusion(torch.zeros_like(f1), f2, dev(P1), dev(P2), **kw)
    assert (attnz - 1.0 / K).abs().max().item() < 1e-7
    outz2 = epi.epipolar_fusion(torch.zeros_like(f1), 2 * f2, dev(P1), dev(P2), **kw)[0]
    assert (outz2 - 2 * outz).abs().max().item() < 1e-5


def test_host_streamer_matches_direct_call():
    """pinned-host front end (three-stream pipeline) returns exactly what the direct device call returns."""
    name = "cfg1_ring"
    cfg, f1, f2, P1, P2, _ = gc.build_inputs(name)
    m = epi.Epipolar(cfg=cfg).cuda().eval()
    with torch.no_grad():
        out, corr, attn, _ = m(dev(f1), dev(f2), dev(P1), dev(P2))
    hs = epi.HostStreamer(m, "cuda", depth=2)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h = [pin(f1), pin(f2), pin(P1), pin(P2)]
    outs = [(torch.empty_like(out, device="cpu").pin_memory(), torch.empty_like(attn, device="cpu").pin_memory(),
             torch.empty_like(corr, device="cpu").pin_memory()) for _ in range(5)]
    for o, a_, c in outs:
        hs(h[0], h[1], h[2], h[3], o, a_, c)
    hs.synchronize()
    for o, a_, c in outs:
        assert torch.equal(o, out.cpu()) and torch.equal(a_, attn.cpu()) and torch.equal(c, corr.cpu())


SWEEP = [  # (N, C, H, W, K)   BASELINE config 5 corners + map sizes on both sides of the tensor-core kernel's limits
    (1, 64, 64, 64, 16), (1, 128, 64, 64, 32), (1, 256, 64, 64, 128), (1, 512, 32, 32, 64),   # C=512: two query-panel halves
    (2, 512, 64, 64, 128), (1, 384, 48, 40, 32), (1, 264, 40, 40, 16),                         # wide corners, C % 64 != 0 above 256
    (1, 64, 128, 128, 32),                                                                       # H*W = 16384: largest tile-kernel map
    (1, 32, 160, 96, 16),                                                                        # non-square
    (1, 16, 144, 144, 16), (2, 24, 100, 400, 64), (1, 8, 300, 100, 16),                          # H*W > 16384: row-windowed union; H > 256 -> warp kernel
    (2, 40, 24, 40, 48),                                                                         # C % 32 != 0, partial tiles
    (1, 64, 256, 256, 16),                                                                       # literal 256x256 feature-map reading
]


@pytest.mark.parametrize("shape", SWEEP)
def test_sweep_shapes_vs_oracle(shape):
    """K/C/map-size sweep (BASELINE config 5): default kernel selection, end to end vs the C oracle."""
    N, C, H, W, K = shape
    from epipolar_transformers_b200 import synthetic as syn
    cfg = epi.make_cfg(KEYPOINT=dict(HEATMAP_SIZE=(H, W), NFEATS=C), EPIPOLAR=dict(SAMPLESIZE=K, USE_CORRECT_NORMALIZE=True))
    P1, P2 = syn.pairs_from_ring(max(N, 2), 4 * max(H, W), seed=K)
    P1, P2 = P1[:N].astype(np.float32), P2[:N].astype(np.float32)
    f1 = syn.features(N, C, H, W, "randn", 5); f2 = syn.features(N, C, H, W, "randn", 6)
    # the documented limits of the pipelined tensor-core kernel (DESIGN.md 3.2): inside them the kernel is FORCED, so a shape
    # that silently fell back to another kernel would fail with EINVAL instead of passing
    map_ok = H * W <= 16384 or (H <= 256 and W <= 1024 and H * W <= 65536)            # above 16384 pixels: row-windowed union bitmap
    pipe_ok = C % 8 == 0 and 8 <= C <= 512 and map_ok and K <= 128 and min(4 * K, 4 * max(H, W)) <= 256
    out, corr, attn, locs = epi.epipolar_fusion(dev(f1), dev(f2), dev(P1), dev(P2), K=K, correct_normalize=True, want_locs=True,
                                                variant="pipe" if pipe_ok else "auto")
    torch.cuda.synchronize()
    o = c_oracle.forward(cfg, f1, f2, P1, P2, locs=locs.cpu().numpy())
    assert rel_max(out.cpu().numpy(), o["out"]) < TOL
    assert rel_max(attn.cpu().numpy(), o["attn"]) < TOL
    assert corr_agree(corr.cpu().numpy(), o["corr_pos"]) > 0.99
