#!/usr/bin/env python
"""bench.py — headline benchmark of the epipolar fusion path (BASELINE.json metric).

A "step" = one forward of the fusion layer over one batch of synthetic (ref, src) feature-map pairs.  Default workload
= BASELINE.json configs[1]: H36M 4-view ResNet-50 256x256 -> N=4 pairs, C=256, 64x64 feature map, K=64
(configs/epipolar/keypoint_h36m_zresidual_fixed.yaml shape, 'z' + ZRESIDUAL, eval).  metric = views/s (= pairs/s);
ms_per_step = forward ms.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload cfg2|cfg3|cfg4|cfg4_256|sweep] [--exchange peer|p2p|allgather] [--dump-outputs DIR]

N>1 (torchrun, one rank per GPU = one camera view per GPU): every rank owns `pairs_per_gpu` frames of its view, the ranks
exchange feature maps inside the timed region (ViewParallelFusion: peer-mapped reads over NVLink, NCCL send/recv, or NCCL
all-gather) and every rank fuses its view against its nearest-neighbour view.  Weak scaling.

`--impl reference` times the reference's own CPU op sequence (oracle/torch_port.py, same ATen operators incl. its torch
geometry) on the host cores with the same config / steps / warmup keys; the N=1 line of our arm also carries `cpu_baseline`
(bounded sample of that) and `gpu_reference` (the same op sequence on the same B200: BASELINE.md B2, the >=10x target's denominator).

`--dump-outputs DIR` writes what the last timed step returned (the module's out / corr_pos / attn, and sample_locs when the
config emits them; rank 0's at N>1; the last K x C shape's for the sweep) as DIR/<name>.npy.  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    "cfg2": dict(N=4, C=256, H=64, W=64, K=64, cfg="cfg_h36m_r50_256",
                 desc="H36M 4-view ResNet-50 256x256 (feature 64x64) C=256 K=64, z+ZRESIDUAL eval"),
    "cfg3": dict(N=4, C=256, H=96, W=96, K=64, cfg="cfg_h36m_r152_384",
                 desc="H36M 4-view ResNet-152 384x384 (feature 96x96) C=256 K=64"),
    "cfg4": dict(N=1, C=256, H=64, W=64, K=64, cfg="cfg_h36m_r50_256",
                 desc="8-view synthetic 256x256 (feature 64x64) C=256 K=64, one view (1 frame) per GPU, z+ZRESIDUAL eval"),
    "cfg4_256": dict(N=1, C=256, H=256, W=256, K=64, cfg="cfg_h36m_r50_256",
                     desc="8-view synthetic, literal 256x256 feature map, C=256 K=64, one view (1 frame) per GPU, z+ZRESIDUAL eval"),
}
SWEEP_K, SWEEP_C = (16, 32, 64, 128), (64, 128, 256, 512)
L2_BYTES = 126 * 1024 * 1024
METRIC = "epipolar_fusion_forward_views_per_sec"
OUTPUT_NAMES = ("out", "corr_pos", "attn", "sample_locs")          # the 4-tuple Epipolar.forward returns
DUMP_BYTES = 64 * 10 ** 6                                          # --dump-outputs writes at most this much in all


def algorithmic_bytes(N, C, H, W, K, attn=True, corr=True):
    """SURVEY.md 8(d): read feat_ref + feat_src, write out (+KRTs, + emitted attn / corr_pos)."""
    b = 3 * 4 * N * C * H * W + 96 * N
    if attn:
        b += 4 * N * K * H * W
    if corr:
        b += 8 * N * H * W
    return b


def dump_outputs(out_dir, outputs):
    """Writes each output tensor as <out_dir>/<name>.npy in float32.  When they add up to more than DUMP_BYTES, each is cut
    to its share by a fixed, seeded sample of its flattened elements (sorted flat indices), so that runs with the same
    arguments write the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in zip(OUTPUT_NAMES, outputs) if v is not None}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = int(a.size * (DUMP_BYTES - 4096) / total)                 # 4096: room for the .npy headers
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, size=keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def make_config(args, wl, world):
    """The `config` object: identical for both arms (the reference arm runs the same workload on the host CPU)."""
    N = wl["N"]
    set_bytes = 2 * N * wl["C"] * wl["H"] * wl["W"] * 4
    n_sets = min(24, max(2, int(np.ceil(3.0 * L2_BYTES / set_bytes))))
    par = "single GPU"
    if world > 1:
        par = "1 view per GPU, exchange of per-view feature maps: %s" % {
            "allgather": "NCCL all-gather", "p2p": "NCCL send/recv (each rank receives only its source view)",
            "peer": "symmetric memory, the staging kernel reads the source view from the neighbour GPU over NVLink"}[args.exchange]
    return {"workload": wl["desc"], "pairs_per_gpu": N, "C": wl["C"], "feat_hw": [wl["H"], wl["W"]], "K": wl["K"],
            "parallelism": par,
            "l2": "rotating %d input sets (%.0f MB > 126 MB L2), no reuse between consecutive steps" % (n_sets, n_sets * set_bytes / 1e6),
            "outputs": "finalout + attn + corr_pos", "variant": args.variant}, n_sets


class ClockSampler:
    """Polls SM clock / throttle reasons through NVML while the timed regions run."""

    def __init__(self, index=0, period=0.02):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self.index, self.period = index, period
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    _BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
             0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self._BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=1.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------
# the reference's own op composition (oracle/torch_port.py): host-CPU arm, cpu_baseline, same-GPU baseline
# ----------------------------------------------------------------------------------------------
def reference_inputs(wl):
    import torch
    import epipolar_transformers_b200 as epi
    from epipolar_transformers_b200 import synthetic as syn
    cfg = getattr(epi, wl["cfg"])()
    cfg.EPIPOLAR.SAMPLESIZE = wl["K"]
    N, C, H, W = wl["N"], wl["C"], wl["H"], wl["W"]
    P1, P2 = syn.pairs_from_ring(max(N, 2), 4 * H)
    f1 = torch.from_numpy(syn.features(N, C, H, W, "relu_smooth", 11))
    f2 = torch.from_numpy(syn.features(N, C, H, W, "relu_smooth", 12))
    params = syn.z_bn_params(C) if "z" in cfg.EPIPOLAR.PARAMETERIZED else None
    return cfg, f1, f2, P1[:N].astype(np.float32), P2[:N].astype(np.float32), params, N


def time_cpu_port(wl, steps, warmup, threads=None, budget_s=240.0):
    """`steps` timed + `warmup` untimed forwards of the reference op sequence on the host cores.  A step is the whole
    workload when that fits the time budget, else a bounded sample of it (fewer pairs; views/s is per pair anyway)."""
    import torch
    from oracle import torch_port
    cfg, f1, f2, P1, P2, params, n = reference_inputs(wl)
    geo = torch_port.TorchGeometry(cfg, wl["H"], wl["W"])
    fwd = lambda a, b, p1, p2: torch_port.forward(cfg, a, b, p1, p2, params=params, geometry=geo)
    if not threads:
        # "all the host threads it can use": ATen's intra-op pool stops scaling (then regresses) well before a 100+-core
        # host is full, so the pool size is the fastest of a few candidates (one pair, one forward each).
        ncpu = os.cpu_count() or 1
        best = None
        for t in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True):
            torch.set_num_threads(t)
            fwd(f1[:1], f2[:1], P1[:1], P2[:1])
            t0 = time.perf_counter()
            fwd(f1[:1], f2[:1], P1[:1], P2[:1])
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, t)
        threads, per_pair = best[1], best[0]
    else:
        torch.set_num_threads(threads)
        t0 = time.perf_counter(); fwd(f1[:1], f2[:1], P1[:1], P2[:1]); per_pair = time.perf_counter() - t0
    torch.set_num_threads(threads)
    pairs = n
    while pairs > 1 and per_pair * pairs * (steps + warmup) > budget_s:
        pairs -= 1
    a, b, p1, p2 = f1[:pairs], f2[:pairs], P1[:pairs], P2[:pairs]
    for _ in range(warmup):
        fwd(a, b, p1, p2)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fwd(a, b, p1, p2)
        ts.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.mean(ts)) * (n / pairs)                     # scaled to the whole workload's pairs
    return {"ms_per_step": ms, "views_per_s": n / (ms * 1e-3), "cores": threads,
            "sample": "%d timed + %d warm-up forwards of %d of the %d pairs of [%s], oracle/torch_port.py (the reference's ATen "
                      "operator sequence incl. its torch geometry), %d host threads" % (steps, warmup, pairs, n, wl["desc"], threads)}


def time_gpu_reference(wl, dev, iters=10, warmup=3):
    """The reference's op sequence on the SAME GPU (BASELINE.md B2): fp32, TF32 off, CUDA events."""
    import torch
    from oracle import torch_port
    cfg, f1, f2, P1, P2, params, n = reference_inputs(wl)
    tf = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False; torch.backends.cudnn.allow_tf32 = False
    try:
        geo = torch_port.TorchGeometry(cfg, wl["H"], wl["W"])
        d1, d2 = f1.to(dev), f2.to(dev)
        pd = {k: torch.from_numpy(v).to(dev) for k, v in params.items()} if params else None
        for _ in range(warmup):
            torch_port.forward(cfg, d1, d2, P1, P2, params=pd, geometry=geo)
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in evs:
            a.record(); torch_port.forward(cfg, d1, d2, P1, P2, params=pd, geometry=geo); b.record()
        torch.cuda.synchronize()
        ms = float(np.median([a.elapsed_time(b) for a, b in evs]))
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf
    return {"ms_per_step": ms, "value": n / (ms * 1e-3), "unit": "views/s", "iters": iters,
            "how": "oracle/torch_port.py on CUDA tensors: the reference's ATen operator sequence incl. its torch geometry "
                   "(per-item pinverse, boolean-mask indexing), fp32, TF32 off, median of CUDA-event timings"}


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cfgd, _ = make_config(args, wl, world)
    r = time_cpu_port(wl, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["views_per_s"], "unit": "views/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfgd, "device": "host CPU",
        "cpu_baseline": {"value": r["views_per_s"], "unit": "views/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["views_per_s"], "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def build_model(epi, syn, torch, wl, dev, variant):
    cfg = getattr(epi, wl["cfg"])()
    cfg.EPIPOLAR.SAMPLESIZE = wl["K"]
    model = epi.Epipolar(cfg=cfg, variant=variant).to(dev).eval()
    if "z" in cfg.EPIPOLAR.PARAMETERIZED:
        model.load_state_dict({k: torch.from_numpy(v) for k, v in syn.z_bn_params(wl["C"]).items()}, strict=False)
    return cfg, model


def run_sweep(args):
    """BASELINE config 5: K x C sweep at the 64x64 feature map, one JSON line; value = geometric mean of views/s."""
    import torch
    import epipolar_transformers_b200 as epi
    from epipolar_transformers_b200 import synthetic as syn, _lib
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    peak, peak_src = measured_peaks()
    rows = []
    N, H, W = 4, 64, 64
    steps, warmup = args.steps, max(3, min(args.warmup, 10))
    for K in SWEEP_K:
        for C in SWEEP_C:
            cfg = epi.make_cfg(KEYPOINT=dict(HEATMAP_SIZE=(H, W), NFEATS=C), EPIPOLAR=dict(SAMPLESIZE=K, USE_CORRECT_NORMALIZE=True))
            m = epi.Epipolar(cfg=cfg, variant=args.variant).to(dev).eval()
            P1, P2 = syn.pairs_from_ring(N, 4 * H)
            P1 = torch.from_numpy(P1.astype(np.float32)).to(dev); P2 = torch.from_numpy(P2.astype(np.float32)).to(dev)
            n_sets = min(24, max(2, int(np.ceil(3.0 * L2_BYTES / (2 * N * C * H * W * 4)))))
            refs = [torch.relu(torch.randn(N, C, H, W, device=dev)) for _ in range(n_sets)]
            srcs = [torch.relu(torch.randn(N, C, H, W, device=dev)) for _ in range(n_sets)]
            with torch.no_grad():
                for i in range(warmup):
                    m(refs[i % n_sets], srcs[i % n_sets], P1, P2)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for i in range(steps - 1):
                    m(refs[i % n_sets], srcs[i % n_sets], P1, P2)
                last = m(refs[(steps - 1) % n_sets], srcs[(steps - 1) % n_sets], P1, P2)
                e1.record(); torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / steps
                lib.epi_kernel_timing_enable(1)
                ks = []
                for i in range(5):
                    m(refs[i % n_sets], srcs[i % n_sets], P1, P2)
                    ks.append(float(lib.epi_kernel_timing_last_ms()))
                lib.epi_kernel_timing_enable(0)
            kms = float(np.median(ks))
            balg = algorithmic_bytes(N, C, H, W, K)
            rows.append({"K": K, "C": C, "ms_per_step": ms, "views_per_s": N / (ms * 1e-3), "kernel_ms": kms,
                         "achieved_gbs": balg / (kms * 1e-3) / 1e9, "frac": balg / (kms * 1e-3) / 1e9 / peak})
            del refs, srcs, m
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    gm = float(np.exp(np.mean([np.log(r["views_per_s"]) for r in rows])))
    print(json.dumps({"metric": METRIC, "value": gm, "unit": "views/s", "n_gpus": 1, "steps": steps, "warmup": warmup,
                      "ms_per_step": float(np.mean([r["ms_per_step"] for r in rows])), "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "K x C sweep (BASELINE config 5) at a 64x64 feature map, N=4 pairs; value = geometric mean",
                                 "variant": args.variant}, "peak": peak, "peak_source": peak_src, "sweep": rows}), flush=True)


def run_ours(args, wl):
    # stdout must carry exactly one JSON line: native libraries (NCCL prints its version with printf when
    # NCCL_DEBUG=VERSION is set on the box) write to fd 1, so fd 1 points at stderr until the line is printed.
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    import epipolar_transformers_b200 as epi
    from epipolar_transformers_b200 import synthetic as syn, _lib
    from epipolar_transformers_b200.distributed import ViewParallelFusion

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    N, C, H, W, K = wl["N"], wl["C"], wl["H"], wl["W"], wl["K"]
    cfg, model = build_model(epi, syn, torch, wl, dev, args.variant)
    cfgd, n_sets = make_config(args, wl, world)

    # cameras.  N=1 GPU: the 4 pairs are (cam v, nearest cam) of one H36M-like 4-camera ring (the test-time batch, SURVEY fact 5).
    # N>1: the same ring geometry at every N so per-GPU work does not change (weak scaling): rank r owns camera r % 4 of its
    # group of 4 ranks (`pairs_per_gpu` frames of it); cfg4 uses a literal `world`-camera ring.
    if world == 1:
        ring = syn.ring_cameras(4, 4 * H)
        src_ix = syn.nearest_source(ring)
        take = np.arange(N) % 4
        P_ref = torch.from_numpy(ring[take].astype(np.float32)).to(dev)
        P_src = torch.from_numpy(ring[src_ix[take]].astype(np.float32)).to(dev)
        vp = None
    else:
        if args.workload.startswith("cfg4"):
            KRT_all = syn.ring_cameras(world, 4 * H)
        else:
            ring = syn.ring_cameras(4, 4 * H)
            KRT_all = ring[np.arange(world) % 4].copy()
            for g in range(1, world // 4 + 1):                  # other groups of 4: the same rig translated by 100 m per group,
                sl = slice(4 * g, min(world, 4 * g + 4))        # so the nearest-camera pairing stays inside a group
                if sl.start < world:
                    T = np.eye(4); T[0, 3] = -1e5 * g
                    KRT_all[sl] = KRT_all[sl] @ T
        vp = ViewParallelFusion(KRT_all, sampler=model, exchange=args.exchange)

    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    mk = lambda: torch.relu(torch.randn(N, C, H, W, device=dev, generator=gen))
    if vp is not None and args.exchange == "peer":
        ok = torch.tensor([1], device=dev)
        refs = None
        try:
            refs = vp.alloc_view_buffers((N, C, H, W), torch.float32, dev, count=n_sets)     # the "backbone output" lives in peer-mapped memory
            for t in refs:
                t.copy_(mk())
        except Exception as e:                            # no peer mapping on this box: fall back to the collective
            ok = torch.tensor([0], device=dev)
            sys.stderr.write("bench.py: symmetric memory unavailable (%r), using all-gather\n" % (e,))
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            args.exchange = "allgather"
            vp = ViewParallelFusion(KRT_all, sampler=model, exchange="allgather")
            cfgd, _ = make_config(args, wl, world)
            refs = [mk() for _ in range(n_sets)]
    else:
        refs = [mk() for _ in range(n_sets)]
    srcs = [mk() for _ in range(n_sets)] if world == 1 else None

    def step(i):
        with torch.no_grad():
            if vp is None:
                return model(refs[i % n_sets], srcs[i % n_sets], P_ref, P_src)
            return vp(refs[i % n_sets], slot=i % n_sets)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warmup = max(3, args.warmup)
    sampler = ClockSampler(local) if rank == 0 else None
    for i in range(warmup):
        step(i)
    launches_per_step = lib.epi_last_launch_count()
    barrier()
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps - 1):
        step(warmup + i)
    last = step(warmup + args.steps - 1)
    ev1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    t = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps

    # ---- correctness at N>1: the exchanged source map must give the same result as a local recompute, bit for bit ----
    parity = None
    if vp is not None:
        with torch.no_grad():
            got = vp(refs[0], slot=0)
            src_local = vp.gather(refs[0])[vp.src].clone()                       # independent path: NCCL all-gather
            want = model(refs[0], src_local, vp.P_ref_dev(N, dev), vp.P_src_dev(N, dev))
        same = all(torch.equal(a, b) for a, b in zip(got[:3], want[:3]))
        flag = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = {"exchange_vs_local_recompute_bit_exact": bool(int(flag.item()))}

    # ---- per-launch-group durations of the same call (CUDA events recorded inside the C ABI call, launching stream) ----
    groups, call = [], []
    lib.epi_kernel_timing_enable(1)
    buf3 = (ctypes.c_float * 3)()
    for i in range(max(5, min(args.steps, 20))):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); step(i + 3); b.record()
        lib.epi_kernel_timing_last3(buf3)
        groups.append([float(buf3[0]), float(buf3[1]), float(buf3[2])])
        torch.cuda.synchronize()
        call.append(a.elapsed_time(b))
    lib.epi_kernel_timing_enable(0)
    g = np.median(np.array(groups), 0)
    kern_ms, call_ms = float(g[1]), float(np.median(call))
    breakdown = {"staging_ms": float(g[0]), "fused_kernel_ms": kern_ms, "epilogue_ms": float(g[2]),
                 "exchange_and_host_ms": max(0.0, call_ms - float(g.sum())), "synchronised_call_ms": call_ms}

    # ---- end to end through the public module call with HOST buffers (pinned), copies inside the timed region ----
    # The pinned buffers are allocated (and the copies driven) from the CPUs of the GPU's own NUMA node: host memory one socket
    # away costs 20-40 % of the PCIe rate on these boxes (run-to-run spread of e2e before this: 0.71-1.27 ms/step).
    numa = epi.bind_host_to_gpu(dev.index if dev.index is not None else 0)
    h_ref = [refs[i].cpu().pin_memory() for i in range(2)]
    h_src = [srcs[i].cpu().pin_memory() for i in range(2)] if world == 1 else None
    h_out = torch.empty((N, C, H, W), dtype=torch.float32).pin_memory()
    h_attn = torch.empty((N, K, H, W), dtype=torch.float32).pin_memory()
    h_corr = torch.empty((N, H, W, 2), dtype=torch.float32).pin_memory()
    if world == 1:
        h_P1, h_P2 = P_ref.cpu().pin_memory(), P_src.cpu().pin_memory()
        streamer = epi.HostStreamer(model, dev, depth=2)
        e2e_how = "pinned host buffers -> HostStreamer(Epipolar) -> pinned host buffers; H2D of step i+1 overlaps kernels + D2H of step i"

        def e2e_step(i):
            streamer(h_ref[i % 2], h_src[i % 2], h_P1, h_P2, h_out, h_attn, h_corr)

        def e2e_drain():
            torch.cuda.current_stream().wait_stream(streamer.s_run); torch.cuda.current_stream().wait_stream(streamer.s_out)
    else:
        s_in = torch.cuda.Stream(dev)
        e2e_how = ("pinned host -> this rank's exchange buffer (upload stream) -> ViewParallelFusion (same exchange mode as the headline) "
                   "-> pinned host; the upload of step i+1 overlaps step i")
        up_done = [torch.cuda.Event() for _ in range(2)]
        used = [torch.cuda.Event() for _ in range(2)]

        def e2e_step(i):
            k = i % 2
            with torch.cuda.stream(s_in):
                s_in.wait_event(used[k])
                refs[k].copy_(h_ref[k], non_blocking=True)                       # straight into the (peer-mapped) view buffer
                up_done[k].record(s_in)
            torch.cuda.current_stream().wait_event(up_done[k])
            with torch.no_grad():
                o, c, a_, _ = vp(refs[k], slot=k)
            used[k].record()
            h_out.copy_(o, non_blocking=True); h_attn.copy_(a_, non_blocking=True); h_corr.copy_(c, non_blocking=True)

        def e2e_drain():
            pass

    e2e_steps = max(5, min(args.steps, 50))
    for i in range(3):
        e2e_step(i)
    e2e_drain(); barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        e2e_step(i)
    e2e_drain()
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([max(e0.elapsed_time(e1), 0.0)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item()) / e2e_steps
    clocks = sampler.stop() if sampler else None
    if numa.get("previous") is not None:
        try:
            os.sched_setaffinity(0, numa["previous"])
        except OSError:
            pass
    h2d = (2 if world == 1 else 1) * N * C * H * W * 4 + (2 * N * 48 if world == 1 else 0)
    d2h = N * C * H * W * 4 + N * K * H * W * 4 + N * H * W * 8

    if rank == 0:
        peak, peak_src = measured_peaks()
        balg = algorithmic_bytes(N, C, H, W, K)
        achieved = balg / (kern_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get(wl["name"], {}).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": world * N / (ms_step * 1e-3), "unit": "views/s",
            "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfgd, "clocks": clocks,
            "e2e": {"value": world * N / (e2e_ms * 1e-3), "unit": "views/s", "ms_per_step": e2e_ms, "wall_ms_per_step": wall_ms / e2e_steps,
                    "how": e2e_how, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "host_numa": {"node": numa.get("node"), "cpus_bound": numa.get("cpus"), "rebound": numa.get("previous") is not None}},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "hbm", "kernel": "epi_fusion_pipe_kernel: fused epipolar attention (geometry + taps + softmax + AV)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "algorithmic_bytes": balg, "kernel_ms": kern_ms,
                         "timing": "CUDA events recorded inside the C ABI call on the launching stream around each launch group (median)",
                         "peak_source": peak_src},
            "breakdown": breakdown,
        }
        if parity is not None:
            line["parity"] = parity
        if world == 1 and not args.no_gpu_reference and H * W <= 128 * 128:
            try:
                line["gpu_reference"] = time_gpu_reference(wl, dev)
                line["gpu_reference"]["speedup_device_step"] = line["gpu_reference"]["ms_per_step"] / ms_step
            except Exception as e:                                  # never lose the headline line to a baseline leg
                line["gpu_reference"] = {"unavailable": repr(e)[:200]}
        if world == 1 and not args.no_cpu_baseline:
            r = time_cpu_port(wl, args.cpu_steps, 1, budget_s=40.0)
            line["cpu_baseline"] = {"value": r["views_per_s"], "unit": "views/s", "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"], "ms_per_step": r["ms_per_step"]}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS) + ["sweep"])
    ap.add_argument("--variant", default="auto", choices=["auto", "warp", "tile", "sector", "pipe"])
    ap.add_argument("--exchange", default="peer", choices=["peer", "p2p", "allgather"], help="multi-GPU exchange of per-view feature maps")
    ap.add_argument("--cpu-steps", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.workload == "sweep":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the sweep workload has no reference arm (use cfg2/cfg3)"}))
            return
        run_sweep(args)
        return
    wl = dict(WORKLOADS[args.workload], name=args.workload)
    if args.impl == "reference":
        run_reference_arm(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
