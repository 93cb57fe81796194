#!/usr/bin/env python
"""Contract benchmark of the RAG stereo hot path (cost volume + disparity regression) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload infer|train|router|sweep192|sweep288] [--impl reference]
                    [--dump-outputs DIR]

A step = one pass of the hot path over one batch of synthetic stereo pairs.  Default workload
(BASELINE.json configs[1]): inference batch 8 per GPU at DrivingStereo half-res 400x880, which the
reference pads to 480x960 at eval (dataloaders/stereo_dataset.py:95-96; its Feature Net cannot run
400x880) -> features [8,12,160,320], volume [8,24,64,160,320], head input [8,1,64,160,320],
maxdisp 192.  `--workload train` is configs[2]: fwd+bwd, batch 4 per GPU at 288x576.

Prints ONE JSON line (rank 0).  Top level:
  value / ms_per_step   K steps of the workload on the two-stream schedule (`schedule: "overlapped"`,
                        rag_b200.pipeline.OverlappedPath / OverlappedTrainPath: the HBM-bound volume kernels share the SMs
                        with the FP32-bound head kernels), inputs resident in HBM, CUDA events, max over ranks;
  value_serial          the same K steps with the kernels back to back on ONE stream -- what a single caller of
                        CostVolume / Disp gets; the per-kernel durations and `roofline` come from this pass;
  roofline              the dominant kernel (cost-volume forward) against the measured HBM peak;
  path                  whole-path algorithmic bytes / time for both schedules;
  train                 (default workload only) the same measurements for BASELINE configs[2] (fwd+bwd B=4 288x576), so the
                        driver-run line carries the training step too;
  parity                one pair of this workload checked in-run against the reference (bit-exactness of the volume and its
                        gradient, max |disp - ref| and the fraction of pixels above 1e-4 px, the reference's own deviation
                        from the fp64 evaluation, gradient max-norm errors);
  e2e                   the same metric through rag_b200.pipeline.HostPipeline (HostTrainPipeline for `train`): pinned HOST
                        buffers, ONE host->device and ONE device->host copy per step inside the timed region, and the box's
                        host->device ceiling measured in the same run (`frac_of_h2d_ceiling`);
  cpu_baseline          the UNMODIFIED reference (oracle/_ref, tools/install_ref.sh) timed on this box's host cores
                        (kind "reference"; "port" = the oracle restatement when oracle/_ref is absent);
  torch_cuda_reference  the same unmodified reference modules run by PyTorch eager on this GPU (the honest GPU bar);
  next_rows             the SURVEY.md section 8f rows (fused stem, last_3_3d conv, ...) beside the headline.
`--impl reference` times the reference's own CPU implementation on the same config (rank 0 only).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "stereo pairs/s (cost vol + disp regression)"
WORKLOADS = {
    # name: (B per GPU, C, Hf, Wf, Df, maxdisp, backward?, description)
    "infer": (8, 12, 160, 320, 64, 192, False, "inference batch 8/GPU at 400x880 padded to 480x960 (reference eval pad), maxdisp 192"),
    "train": (4, 12, 96, 192, 64, 192, True, "training step fwd+bwd batch 4/GPU at 288x576 crop, maxdisp 192"),
    # configs[3]: 32 pairs routed over 4 grown scene paths = 4 sub-batches of 8 per step (the hot path is path-independent)
    "router": (32, 12, 160, 320, 64, 192, False, "scene-router inference, 32 pairs/GPU at 480x960 as 4 path sub-batches of 8, maxdisp 192"),
    # configs[4]: resolution / disparity sweep
    "sweep192": (4, 12, 128, 416, 64, 192, False, "inference batch 4/GPU at 384x1248, maxdisp 192"),
    "sweep288": (4, 12, 128, 416, 96, 288, False, "inference batch 4/GPU at 384x1248, maxdisp 288"),
}


def config_dict(workload):
    """Identical in both arms (the driver compares the two lines' `config`)."""
    b, c, hf, wf, df, md, bwd, desc = WORKLOADS[workload]
    cvb, hfb, hbb = alg_bytes(c, hf, wf, df)
    step_bytes = (cvb + hfb + ((cvb + hbb) if bwd else 0)) * b
    return {"workload": workload, "desc": desc, "pairs_per_gpu": b, "features": [b, c, hf, wf],
            "volume": [b, 2 * c, df, hf, wf], "head_in": [b, 1, df, hf, wf], "maxdisp": md,
            "direction": "fwd+bwd" if bwd else "fwd",
            "l2": "no explicit flush: every step streams %.2f GB (>> 126 MB L2) through HBM" % (step_bytes / 1e9),
            "sharding": "stereo pairs across ranks, no data-path collective"}


def alg_bytes(c, hf, wf, df):
    """Algorithmic bytes per pair (SURVEY.md section 8d)."""
    cv = 4 * (2 * c * hf * wf + 2 * c * df * hf * wf)
    head_f = 4 * (df * hf * wf + 9 * hf * wf)
    head_b = 4 * (2 * df * hf * wf + 9 * hf * wf)
    return cv, head_f, head_b


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram read+write bytes per launch of the dominant kernel from the committed ncu capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


# --------------------------------------------------------------------------------------------
# the reference: the unmodified modules from oracle/_ref when installed, else the oracle port
# --------------------------------------------------------------------------------------------
class Reference:
    """Callable view of the reference's hot path.  kind == "reference": rag_model.Network.forward's own lines 375-383
    (driven through stub feature/matching callables, as tests/golden/make_golden.py does) and rag_model.Disp, imported
    unmodified from oracle/_ref; kind == "port": oracle/rag_oracle.py (the same op sequence restated)."""

    def __init__(self, cpu: bool):
        import types

        from oracle import refimport as R

        self.kind = "port"
        self.ref = None
        self.cpu = cpu
        self._R = R
        if R.available():
            try:
                self.ref = R.import_reference(cpu_patch=cpu)
                self.kind = "reference"
                self._types = types
            except Exception as e:  # noqa: BLE001
                print(f"bench.py: reference import failed ({e}); using the oracle port", file=sys.stderr)
        if self.ref is None:
            from oracle import rag_oracle as O

            self.O = O

    def cost_volume(self, x, y, md):
        if self.ref is None:
            return self.O.cost_volume_ref(x, y, md)
        holder = {}
        stub = self._types.SimpleNamespace(maxdisp=md)
        feats = iter([x, y])
        stub.feature = lambda img, task_arch, path: next(feats)
        stub.matching = lambda cost, task_arch, path: holder.setdefault("cost", cost)
        stub.disp = lambda c: c
        self.ref.rag_model.Network.forward(stub, None, None, 0)
        return holder["cost"]

    def head(self, cl, md):
        if self.ref is None:
            return self.O.disp_head_ref(cl, md)
        key = ("disp", md)
        if not hasattr(self, "_disp") or self._disp[0] != key:
            self._disp = (key, self.ref.rag_model.Disp(md))
        return self._disp[1](cl)

    def step(self, x, y, cl, md, bwd, gcost=None, gdisp=None):
        if self.cpu and self.ref is not None:
            with self._R.on_cpu():          # rag_model.py:26 names "the current CUDA device"; CPU tensors need 'cpu'
                return self._step(x, y, cl, md, bwd, gcost, gdisp)
        return self._step(x, y, cl, md, bwd, gcost, gdisp)

    def _step(self, x, y, cl, md, bwd, gcost=None, gdisp=None):
        import torch

        if not bwd:
            with torch.no_grad():
                return self.cost_volume(x, y, md), self.head(cl, md)
        xr, yr, cr = x.clone().requires_grad_(True), y.clone().requires_grad_(True), cl.clone().requires_grad_(True)
        cost = self.cost_volume(xr, yr, md)
        cost.backward(gcost if gcost is not None else torch.ones_like(cost))
        d = self.head(cr, md)
        d.backward(gdisp if gdisp is not None else torch.ones_like(d))
        return cost.detach(), d.detach(), cr.grad, xr.grad, yr.grad


def seeded_pair(workload, device=None):
    import torch

    b, c, hf, wf, df, md, bwd, _ = WORKLOADS[workload]
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(1, c, hf, wf, generator=g)
    y = torch.randn(1, c, hf, wf, generator=g)
    cl = torch.randn(1, 1, df, hf, wf, generator=g)
    gcost = torch.randn(1, 2 * c, df, hf, wf, generator=g)
    gdisp = torch.randn(1, 3 * hf, 3 * wf, generator=g) * (torch.rand(1, 3 * hf, 3 * wf, generator=g) < 0.3)
    ts = (x, y, cl, gcost, gdisp)
    return tuple(t.to(device) for t in ts) if device is not None else ts


def cpu_reference(workload, warmup=1, steps=3, budget_s=25.0):
    """Time the reference's CPU path: `steps` single-pair steps after `warmup`, stopping early once `budget_s` is spent
    (never fewer than 2 timed steps).  Returns (cpu_baseline dict, list of step times)."""
    import torch

    b, c, hf, wf, df, md, bwd, _ = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    refm = Reference(cpu=True)
    x, y, cl, gcost, gdisp = seeded_pair(workload)
    t_start = time.perf_counter()
    for _ in range(max(1, warmup)):
        refm.step(x, y, cl, md, bwd, gcost, gdisp)
        if time.perf_counter() - t_start > budget_s / 3:
            break
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < steps and (len(times) < 2 or time.perf_counter() < t_end):
        t0 = time.perf_counter()
        refm.step(x, y, cl, md, bwd, gcost, gdisp)
        times.append(time.perf_counter() - t0)
    mean = sum(times) / len(times)
    return {
        "value": 1.0 / mean, "unit": "pairs/s", "cores": cores, "kind": refm.kind, "best_pairs_per_s": 1.0 / min(times), "steps_timed": len(times),
        "sample": f"1 pair of the {workload} workload per step ({3*hf}x{3*wf}, maxdisp {md}, {'fwd+bwd' if bwd else 'fwd'}), mean of {len(times)} steps after warm-up, "
                  f"torch {torch.__version__} CPU, {torch.get_num_threads()} threads; pairs are independent, so pairs/s does not depend on the batch "
                  "(the reference head needs ~1.8 GB of temporaries per pair at 480x960)",
        "what": ("unmodified reference: models.rag_model.Network.forward lines 375-383 + models.rag_model.Disp from oracle/_ref" if refm.kind == "reference"
                 else "oracle port of rag_model.py:375-383,18-44 (oracle/_ref not installed)"),
    }, times


def config1_full_network_cpu(budget_s=20.0):
    """BASELINE.json configs[0] / BASELINE.md section 4.5: the reference's full Network.forward (Feature Net + cost volume +
    Matching Net + head), synthetic 1x3x288x576, maxdisp 192, on the host cores.  Needs oracle/_ref."""
    import torch

    from oracle import refimport as R

    if not R.available():
        return None
    try:
        ref = R.import_reference(cpu_patch=True)
        torch.manual_seed(0)
        net = ref.rag_model.Network(R.make_genotype(ref, 0), "cpu").eval()
        g = torch.Generator().manual_seed(1234)
        left, right = torch.randn(1, 3, 288, 576, generator=g), torch.randn(1, 3, 288, 576, generator=g)
        parts = {}

        def timed(name, fn):
            def wrapped(*a, **k):
                t0 = time.perf_counter()
                out = fn(*a, **k)
                parts[name] = parts.get(name, 0.0) + time.perf_counter() - t0
                return out
            return wrapped

        net.feature = timed("feature_x2", net.feature)
        net.matching = timed("matching", net.matching)
        net.disp.forward = timed("head", net.disp.forward)
        times = []
        with torch.no_grad(), R.on_cpu():
            net(left, right, 0, net.arch_init)
            parts.clear()
            t_end = time.perf_counter() + budget_s
            while len(times) < 3 and (not times or time.perf_counter() < t_end):
                t0 = time.perf_counter()
                net(left, right, 0, net.arch_init)
                times.append(time.perf_counter() - t0)
        n = len(times)
        total = sum(times) / n
        br = {k: round(v / n, 4) for k, v in parts.items()}
        br["cost_volume"] = round(total - sum(br.values()), 4)
        return {"what": "unmodified reference Network.forward (rag_model.py:369-387), random genotype, 1x3x288x576, maxdisp 192, CPU",
                "s_per_pair": round(total, 4), "pairs_per_s": round(1.0 / total, 4), "runs": n, "cores": os.cpu_count(), "breakdown_s": br}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    b, c, hf, wf, df, md, bwd, desc = WORKLOADS[args.workload]
    base, times = cpu_reference(args.workload, warmup=args.warmup, steps=args.steps, budget_s=float("inf"))   # exactly --steps
    v = base["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": len(times), "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.workload),
        "note": "each step = one pair of the workload on all host cores (a bounded sample; the batch is a loop over independent pairs); value = mean over the timed steps",
        "cpu_baseline": base,
        "config1_full_network_cpu": config1_full_network_cpu() if not args.no_cpu_baseline else None,
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# clocks sampler (NVML, in-process: the timed region is far shorter than nvidia-smi's period)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml as nv

            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def torch_cuda_reference(workload, dev, reps=5):
    """The UNMODIFIED reference modules (oracle/_ref; oracle port if absent) run by PyTorch eager ON THE SAME GPU: the
    honest GPU baseline (SURVEY.md section 8d).  One pair per call (its temporaries are ~1.8 GB/pair at 480x960)."""
    import torch

    b, c, hf, wf, df, md, bwd, _ = WORKLOADS[workload]
    refm = Reference(cpu=False)
    x, y, cl, gcost, gdisp = seeded_pair(workload, dev)
    refm.step(x, y, cl, md, bwd, gcost, gdisp)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        refm.step(x, y, cl, md, bwd, gcost, gdisp)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    torch.cuda.empty_cache()
    return {"value": 1e3 / ms, "unit": "pairs/s", "ms_per_pair": ms, "kind": refm.kind,
            "what": "reference modules (rag_model.py:375-383,18-44) through PyTorch eager CUDA kernels on this GPU, 1 pair per call"}


def parity_record(workload, dev):
    """One seeded pair of the workload through our kernels and through the reference ON THIS GPU (checker only)."""
    import torch

    from oracle import rag_oracle as O
    from rag_b200 import functional as F_

    b, c, hf, wf, df, md, bwd, _ = WORKLOADS[workload]
    refm = Reference(cpu=False)
    x, y, cl, gcost, gdisp = seeded_pair(workload, dev)
    out = {"pair": f"1 seeded pair of the {workload} workload, sigma = 1 matching cost", "reference": refm.kind + " on CUDA (torch %s)" % torch.__version__}
    cost = F_.cost_volume_forward(x, y, df)
    disp, stats = F_.disp_head_forward(cl, md, want_stats=True)
    with torch.no_grad():
        cost_ref = refm.cost_volume(x, y, md)
        out["cv_bit_exact"] = bool(torch.equal(cost, cost_ref))
        del cost_ref
        disp_ref = refm.head(cl, md)
    d64, _ = O.disp_head_f64_torch(cl[:, 0], md)
    err = (disp - disp_ref).abs()
    ref_dev = (disp_ref.double() - d64).abs()
    out["disp_max_abs_err"] = float(err.max())
    out["disp_frac_gt_1e-4"] = float((err > 1e-4).double().mean())
    out["disp_own_vs_fp64_max"] = float((disp.double() - d64).abs().max())
    out["ref_vs_fp64_max"] = float(ref_dev.max())
    out["disp_max_excess_over_ref_noise"] = float((err.double() - ref_dev).max())    # <= 1e-4 is the per-pixel bound the tests assert
    del d64, err, ref_dev, disp_ref, cost
    torch.cuda.empty_cache()
    if bwd:
        gcl = F_.disp_head_backward(cl, gdisp, disp, stats, md)
        gx, gy = F_.cost_volume_backward(gcost, c)
        _, _, gcl_ref, gx_ref, gy_ref = refm.step(x, y, cl, md, True, gcost, gdisp)
        out["cv_grad_bit_exact"] = bool(torch.equal(gx, gx_ref) and torch.equal(gy, gy_ref))
        _, g64 = O.disp_head_f64_torch(cl[:, 0], md, gdisp)
        den = float(g64.abs().max())
        out["grad_maxnorm_rel"] = float((gcl[:, 0].double() - g64).abs().max()) / den
        out["grad_maxnorm_rel_vs_ref"] = float((gcl - gcl_ref).abs().max()) / float(gcl_ref.abs().max())
        out["ref_grad_vs_fp64_maxnorm_rel"] = float((gcl_ref[:, 0].double() - g64).abs().max()) / den
    torch.cuda.empty_cache()
    return out


def next_rows_record(x, y, df, md, sub):
    """SURVEY.md section 8f rows reported beside the headline, not part of `value`."""
    import torch

    from rag_b200 import functional as F_
    from rag_b200.fused_stem import cv_stem_forward

    dev = x.device
    xs, ys = x[:sub], y[:sub]
    c = x.shape[1]
    g = torch.Generator(device=dev).manual_seed(11)
    conv = torch.nn.Conv3d(2 * c, c, 3, padding=1, bias=False).to(dev)
    bn = torch.nn.BatchNorm3d(c).to(dev).eval()

    def t(fn, n):
        fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n

    rows = {}
    with torch.no_grad():
        bn.running_mean.normal_(0, 0.3, generator=g)
        bn.running_var.uniform_(0.5, 2.0, generator=g)
        scale = bn.weight * torch.rsqrt(bn.running_var + bn.eps)
        shift = bn.bias - bn.running_mean * scale
        fused = t(lambda: cv_stem_forward(xs, ys, conv.weight, scale, shift, True, md), 10)
        ref = t(lambda: torch.relu_(bn(conv(F_.cost_volume_forward(xs, ys, df)))), 3)
        a = cv_stem_forward(xs[:1], ys[:1], conv.weight, scale, shift, True, md)
        old = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        b_ = torch.relu_(bn(conv(F_.cost_volume_forward(xs[:1], ys[:1], df))))
        torch.backends.cudnn.allow_tf32 = old
        err = ((a - b_).abs().max() / b_.abs().max()).item()
        rows["stem3d0"] = {"what": "cost volume + stem3d0 (Conv3d 24->12 3x3x3 + BN(eval) + ReLU), %d pairs" % sub,
                           "fused_ms": round(fused, 4), "cost_volume_plus_cudnn_tf32_ms": round(ref, 4), "speedup": round(ref / fused, 1),
                           "max_rel_err_vs_fp32_cudnn": err}
        del a, b_
        # rank 2: last_3_3d (Conv3d C -> 1, 3x3x3), the producer of the head's input
        from rag_b200.last_conv import conv3d_c1_forward
        feat = torch.randn(sub, c, df, x.shape[2], x.shape[3], device=dev, generator=g)
        last = torch.nn.Conv3d(c, 1, 3, padding=1, bias=False).to(dev)
        lc = t(lambda: conv3d_c1_forward(feat, last.weight), 10)
        lc_ref = t(lambda: last(feat), 3)
        torch.backends.cudnn.allow_tf32 = False
        lc_err = ((conv3d_c1_forward(feat[:1], last.weight) - last(feat[:1])).abs().max() / last(feat[:1]).abs().max()).item()
        torch.backends.cudnn.allow_tf32 = old
        rows["last_3_3d"] = {"what": "last_3_3d (Conv3d %d->1 3x3x3, fp32 direct convolution), %d pairs" % (c, sub),
                             "ms": round(lc, 4), "cudnn_tf32_ms": round(lc_ref, 4), "speedup": round(lc_ref / lc, 1),
                             "max_rel_err_vs_fp32_cudnn": lc_err}
        del feat
    torch.cuda.empty_cache()
    for name, fn in EXTRA_NEXT_ROWS:
        try:
            rows[name] = fn(dev)
        except Exception as e:  # noqa: BLE001
            rows[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    return rows


def stem_train_row(dev):
    """SURVEY.md section 8f rank 1, training: cost volume + stem3d0 = Conv3d(24->12) + BatchNorm3d(train) + ReLU, forward + backward
    at BASELINE configs[2] (B=4, 288x576).  Fused (rag_b200.fused_stem.FusedStemFn: no volume, no volume gradient, no conv output)
    vs the reference composition on the materialised volume through cuDNN (TF32, its default)."""
    import torch

    from rag_b200.functional import cost_volume
    from rag_b200.fused_stem import VirtualCostVolume, stem_forward

    class Layer(torch.nn.Module):                       # the fields of the reference's ConvBR_3d (operations_3d.py:31-47)
        def __init__(self):
            super().__init__()
            self.relu, self.use_bn = True, True
            self.conv = torch.nn.Conv3d(24, 12, 3, 1, 1, bias=False)
            self.bn = torch.nn.BatchNorm3d(12)

    b, hf, wf, md = 4, 96, 192, 192
    g = torch.Generator(device=dev).manual_seed(3)
    layer = Layer().to(dev).train()
    x = torch.randn(b, 12, hf, wf, device=dev, generator=g, requires_grad=True)
    y = torch.randn(b, 12, hf, wf, device=dev, generator=g, requires_grad=True)
    gout = torch.randn(b, 12, md // 3, hf, wf, device=dev, generator=g)

    def fused():
        stem_forward(layer, VirtualCostVolume(x, y, md)).backward(gout)

    def ref():
        torch.relu(layer.bn(layer.conv(cost_volume(x, y, md)))).backward(gout)

    def t(fn, n):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n, (torch.cuda.max_memory_allocated(dev) - base) / 2**20

    f_ms, f_mem = t(fused, 10)
    r_ms, r_mem = t(ref, 3)
    return {"what": "cost volume + stem3d0 (Conv3d 24->12 3x3x3 + BatchNorm3d(train) + ReLU), forward + backward, B=4 288x576",
            "fused_ms": round(f_ms, 4), "cost_volume_plus_cudnn_tf32_ms": round(r_ms, 4), "speedup": round(r_ms / f_ms, 1),
            "fused_peak_extra_MiB": round(f_mem), "cudnn_peak_extra_MiB": round(r_mem),
            "parity": "tests/test_fused_stem_gpu.py: every gradient within 1e-5 max-norm of the fp64 evaluation (ReLU mask fixed)"}


def tail_rows(dev):
    """SURVEY.md section 8f rank 2, training: upsample_6 (trilinear, align_corners=True) forward + backward and the backward of
    last_3_3d at BASELINE configs[2] (B=4, 288x576), beside ATen / cuDNN (TF32 default)."""
    import torch
    import torch.nn.functional as F

    from rag_b200.last_conv import Conv3dC1Fn
    from rag_b200.upsample import trilinear_resize

    b, c, d, h, w = 4, 12, 64, 96, 192
    g = torch.Generator(device=dev).manual_seed(4)

    def t(fn, n):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / n

    x = torch.randn(b, c, d // 2, h // 2, w // 2, device=dev, generator=g, requires_grad=True)
    go = torch.randn(b, c, d, h, w, device=dev, generator=g)
    ours = t(lambda: trilinear_resize(x, (d, h, w), True).backward(go), 10)
    aten = t(lambda: F.interpolate(x, (d, h, w), mode="trilinear", align_corners=True).backward(go), 5)
    feat = torch.randn(b, c, d, h, w, device=dev, generator=g, requires_grad=True)
    wt = (torch.randn(1, c, 3, 3, 3, device=dev, generator=g) * 0.1).requires_grad_(True)
    g1 = torch.randn(b, 1, d, h, w, device=dev, generator=g)
    conv_ours = t(lambda: Conv3dC1Fn.apply(feat, wt).backward(g1), 10)
    conv_ref = t(lambda: F.conv3d(feat, wt, padding=1).backward(g1), 3)
    return {"upsample_6": {"what": "nn.Upsample trilinear align_corners=True [4,12,32,48,96] -> [4,12,64,96,192], forward + backward",
                           "ms": round(ours, 4), "aten_ms": round(aten, 4), "speedup": round(aten / ours, 1),
                           "note": "backward is a deterministic gather (ATen: atomicAdd scatter)"},
            "last_3_3d_train": {"what": "last_3_3d (Conv3d 12->1 3x3x3) forward + backward (data + weight gradient), B=4 288x576",
                                "ms": round(conv_ours, 4), "cudnn_tf32_ms": round(conv_ref, 4), "speedup": round(conv_ref / conv_ours, 1)}}


EXTRA_NEXT_ROWS = [("stem3d0_train", stem_train_row), ("tail_train", tail_rows)]     # (name, fn(dev) -> dict)

DUMP_BYTES = 60 * 2**20         # --dump-outputs: all arrays together stay under 64 MB, .npy headers included
DUMP_ARRAY_BYTES = 16 * 2**20   # an output larger than its share is stored as a sample of its elements
DUMP_SEED = 20240601


def sample_outputs(outputs):
    """{name: [device tensor per call]} (the calls' results concatenated along dim 0 are the output) -> {name: (float32 numpy
    array, description)}.  An output of at most min(DUMP_ARRAY_BYTES, DUMP_BYTES / #outputs) bytes is kept whole; a larger
    one becomes `<name>_sample`: its elements at sorted flat indices (row-major over the concatenated shape) drawn with
    DUMP_SEED, which depend only on the shape, so two builds run with the same arguments compare element for element."""
    import torch

    cap = min(DUMP_ARRAY_BYTES, DUMP_BYTES // len(outputs))
    out = {}
    for name, parts in outputs.items():
        shape = [sum(p.shape[0] for p in parts)] + list(parts[0].shape[1:])
        per = parts[0].numel()
        total = per * len(parts)
        if total * 4 <= cap:
            out[name] = (torch.cat([p.float().cpu() for p in parts]).numpy(), {"shape": shape, "stored": "all"})
            continue
        g = torch.Generator().manual_seed(DUMP_SEED)
        idx = torch.unique(torch.randint(total, (cap // 4,), generator=g))      # sorted, no repeats
        vals = torch.empty(idx.numel(), dtype=torch.float32)
        for j, p in enumerate(parts):
            sel = (idx >= j * per) & (idx < (j + 1) * per)
            vals[sel] = p.reshape(-1)[(idx[sel] - j * per).to(p.device)].float().cpu()
        out[name + "_sample"] = (vals.numpy(), {"shape": shape, "stored": "%d elements at seeded flat indices (seed %d)" % (idx.numel(), DUMP_SEED)})
    return out


def write_outputs(sampled, out_dir):
    """Write sample_outputs()' arrays as out_dir/<name>.npy; returns their description for the JSON line."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, (arr, _) in sampled.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    return {"dir": out_dir, "step": "last timed step of the overlapped pass", "dtype": "float32",
            "arrays": {name: desc for name, (_, desc) in sampled.items()}}


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from rag_b200 import _cabi
    from rag_b200 import dist as D
    from rag_b200 import functional as F_
    from rag_b200.pipeline import HostPipeline, HostTrainPipeline, OverlappedPath, OverlappedTrainPath

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    numa = D.bind_to_gpu_numa(local)        # before any pinned allocation (first-touch placement); a no-op on single-socket hosts
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    K, Wm = args.steps, max(args.warmup, 3)
    peak, peak_src = measured_peak()
    sampler = ClockSampler(local) if rank == 0 else None

    def measure(workload, with_clocks, dump=False):
        """Serial pass (kernels back to back on one stream, events around each) + overlapped pass (two streams).  With
        `dump`, the record's "outputs" holds sample_outputs() of the timed pass's last step."""
        b, c, hf, wf, df, md, bwd, desc = WORKLOADS[workload]
        # identical bits for CPU reference and GPU: generate on the host with a fixed seed, then copy
        g = torch.Generator().manual_seed(1234 + rank)
        x = torch.randn(b, c, hf, wf, generator=g).to(dev)
        y = torch.randn(b, c, hf, wf, generator=g).to(dev)
        cl = torch.randn(b, 1, df, hf, wf, generator=g).to(dev)
        gcost = gdisp = None
        if bwd:
            gcost = torch.randn(b, 2 * c, df, hf, wf, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
            gdisp = (torch.randn(b, 3 * hf, 3 * wf, generator=g) * (torch.rand(b, 3 * hf, 3 * wf, generator=g) < 0.3)).to(dev)
        marks = [[ev() for _ in range(5)] for _ in range(K)]
        sub = 8 if workload == "router" else b   # router: one call per scene path
        n_sub = b // sub

        def step(mk=None):
            if mk: mk[0].record()
            if not bwd:
                cost = [F_.cost_volume_forward(x[i:i + sub], y[i:i + sub], df) for i in range(0, b, sub)]
                if mk: mk[1].record()
                disp = [F_.disp_head_forward(cl[i:i + sub], md, want_stats=False)[0] for i in range(0, b, sub)]
                if mk: mk[2].record()
                return cost, disp
            cost = F_.cost_volume_forward(x, y, df)
            if mk: mk[1].record()
            disp, stats = F_.disp_head_forward(cl, md, want_stats=True)
            if mk: mk[2].record()
            gcl = F_.disp_head_backward(cl, gdisp, disp, stats, md)
            if mk: mk[3].record()
            gx, gy = F_.cost_volume_backward(gcost, c)
            if mk: mk[4].record()
            return cost, disp, gcl, gx, gy

        def serial_pass():
            for _ in range(Wm):
                out = step()
            barrier()
            t0, t1 = ev(), ev()
            t0.record()
            for k in range(K):
                out = step(marks[k])
            t1.record()
            torch.cuda.synchronize()
            del out
            return t0.elapsed_time(t1)

        opath = OverlappedTrainPath(md, dev, schedule=args.schedule) if bwd else OverlappedPath(md, dev, schedule=args.schedule)

        def overlapped_step():
            if bwd:
                return opath.step(x, y, cl, gcost, gdisp)
            return [opath.step(x[i:i + sub], y[i:i + sub], cl[i:i + sub]) for i in range(0, b, sub)]

        def overlapped_pass():
            for _ in range(Wm):
                outs = overlapped_step()
            opath.join()
            barrier()
            t0, t1 = ev(), ev()
            t0.record()
            for k in range(K):
                outs = overlapped_step()
            opath.join()
            t1.record()
            torch.cuda.synchronize()
            return t0.elapsed_time(t1), outs

        def graph_pass():
            """The same two-stream step captured ONCE into a CUDA graph (fork/join included) and replayed K times."""
            if bwd:
                graphs = [opath.capture(x, y, cl, gcost, gdisp)]
            else:
                graphs = [opath.capture(x[i:i + sub], y[i:i + sub], cl[i:i + sub]) for i in range(0, b, sub)]
            for _ in range(Wm):
                for gr, _o in graphs:
                    gr.replay()
            barrier()
            t0, t1 = ev(), ev()
            t0.record()
            for k in range(K):
                for gr, _o in graphs:
                    gr.replay()
            t1.record()
            torch.cuda.synchronize()
            del graphs
            return t0.elapsed_time(t1)

        serial_ms = serial_pass()
        barrier()
        n0 = _cabi.launch_count()
        eager_ms = overlapped_pass()[0]    # untimed for `value`: a second, independent sample of the same schedule
        barrier()
        n0 = _cabi.launch_count()
        if with_clocks and sampler: sampler.start()
        total_ms, outs = overlapped_pass()
        clocks = sampler.stop() if (with_clocks and sampler) else None
        # what the caller of the timed path received in its last step, reduced to host arrays before anything else runs
        names = ("cost", "disp", "gcl", "gx", "gy") if bwd else ("cost", "disp")
        parts = [outs] if bwd else outs            # inference: one (cost, disp, stats) per sub-batch call
        dumped = sample_outputs({n: [p[i] for p in parts] for i, n in enumerate(names)}) if dump else None
        del outs, parts
        # --graph: additionally time the same two-stream step captured ONCE into a CUDA graph and replayed (one host launch per
        # step).  Reported beside the headline, never as it: the launch order of the two branches inside a graph is not
        # defined, and the SM-sharing only works when the persistent volume kernel is dispatched first (0.42 or 0.53 ms per
        # step on the inference workload depending on the replay; profiles/r2_overlap_graph.md).
        graph_ms = graph_pass() if args.graph else None
        used_graph = False
        per_step = (4 if bwd else 2 * n_sub)
        launches = K * per_step            # kernels of ours per timed step (a graph replay launches the captured ones)
        barrier()
        total_ms, serial_ms, eager_ms, graph_ms = max_over_ranks([total_ms, serial_ms, eager_ms, graph_ms if graph_ms is not None else 0.0])
        n_seg = 4 if bwd else 2
        seg_ms = [sum(marks[k][i].elapsed_time(marks[k][i + 1]) for k in range(K)) / K for i in range(n_seg)]
        cvb, hfb, hbb = alg_bytes(c, hf, wf, df)
        cv_ms = seg_ms[0] / n_sub                       # average duration of ONE cost-volume launch
        achieved = cvb * sub / (cv_ms * 1e-3) / 1e9
        lean = wf % 4 == 0
        kname = "cv_fwd_lean_kernel<256,1,true>" if lean else "cv_fwd_kernel"
        roofline = {
            "bound": "hbm", "kernel": kname + " (cost-volume forward)",
            "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
            "traffic": (ncu_traffic("cv_fwd_lean_kernel" if lean else "cv_fwd_kernel") if workload in ("infer", "router")
                        else ncu_traffic("cv_fwd_lean_kernel@B4_288x576") if (workload == "train" and lean) else None),
            "peak_source": peak_src, "alg_bytes_per_launch": cvb * sub, "avg_launch_ms": round(cv_ms, 5),
            "timed_in": "serial pass of %d steps in this run (kernels back to back on one stream, CUDA events around each)" % K,
            "note": "a write-only stream: the measured peak is a COPY (read+write) figure, a pure fill of the same bytes runs at ~7.45 TB/s",
        }
        path_bytes = (cvb + hfb + ((cvb + hbb) if bwd else 0)) * b
        kernels = {"cv_fwd_ms": seg_ms[0], "head_fwd_ms": seg_ms[1]}
        if bwd:
            kernels.update({"head_bwd_ms": seg_ms[2], "cv_bwd_ms": seg_ms[3]})
        kfrac = {"cv_fwd": cvb * b / (seg_ms[0] * 1e-3) / 1e9 / peak, "head_fwd": hfb * b / (seg_ms[1] * 1e-3) / 1e9 / peak}
        if bwd:
            kfrac.update({"head_bwd": hbb * b / (seg_ms[2] * 1e-3) / 1e9 / peak, "cv_bwd": cvb * b / (seg_ms[3] * 1e-3) / 1e9 / peak})
        step_ms, sstep_ms = total_ms / K, serial_ms / K

        def frac(ms):
            return round(path_bytes / (ms * 1e-3) / 1e9 / peak, 4)

        path = {
            "alg_bytes_per_step": path_bytes,
            "overlapped": {"ms_per_step": round(step_ms, 5), "pairs_per_s": round(world * b / (step_ms * 1e-3), 1), "frac_of_hbm_peak": frac(step_ms),
                           "launched_as": "one CUDA graph replay per step (the two-stream step captured once)" if used_graph else "eager launches on two free-running streams"},
            "overlapped_graph": ({"ms_per_step": round(graph_ms / K, 5), "pairs_per_s": round(world * b * K / (graph_ms * 1e-3), 1), "frac_of_hbm_peak": frac(graph_ms / K)} if graph_ms else None),
            "overlapped_first_sample": {"ms_per_step": round(eager_ms / K, 5), "pairs_per_s": round(world * b * K / (eager_ms * 1e-3), 1), "frac_of_hbm_peak": frac(eager_ms / K)},
            "serial": {"ms_per_step": round(sstep_ms, 5), "pairs_per_s": round(world * b / (sstep_ms * 1e-3), 1), "frac_of_hbm_peak": frac(sstep_ms)},
            "kernel_ms": {k: round(v, 5) for k, v in kernels.items()},
            "kernel_frac_of_hbm_peak": {k: round(v, 4) for k, v in kfrac.items()},
            "kernel_schedule": {"name": args.schedule, "variants(cv_fwd, head_fwd, cv_bwd, head_bwd)": list(opath.variants)},
            "schedule_note": ("overlapped = the volume kernels on one stream and the head kernels on another (rag_b200.pipeline.%s, schedule '%s': "
                              "'coresident' = all kernels as persistent grids whose CTAs fit an SM together -- the volume kernel in a quarter of the "
                              "register file, its in-flight reads in shared memory, three head CTAs in the rest -- so they share the SMs whichever "
                              "is launched first; 'launch-order' = persistent volume kernels launched before plain head grids); the kernels of a step "
                              "have no data dependence on each other (in the network the Matching Net sits between them), so a stream of batches "
                              "overlaps them; serial = back to back on one stream" % (type(opath).__name__, args.schedule)),
            "note": "the head kernels are FP32-pipe bound (one exp2 + 7-12 FP32 ops per pixel per low-res bin), not HBM bound; see DESIGN.md",
        }
        rec = {"value": world * b * K / (total_ms * 1e-3), "value_serial": world * b * K / (serial_ms * 1e-3), "ms_per_step": step_ms,
               "ms_per_step_serial": sstep_ms, "schedule": "overlapped, CUDA-graph replay" if used_graph else "overlapped, eager two-stream", "roofline": roofline, "path": path, "gpu_launches": int(launches), "clocks": clocks,
               "outputs": dumped}
        return rec, (x, y, cl, gcost, gdisp)

    main, tensors = measure(args.workload, with_clocks=True, dump=args.dump_outputs is not None and rank == 0)
    b, c, hf, wf, df, md, bwd, desc = WORKLOADS[args.workload]
    x, y, cl, gcost, gdisp = tensors

    # ---- e2e: HOST buffers through the public pipeline (ONE H2D + kernels + ONE D2H per step) ----
    pipe = HostTrainPipeline(md, dev) if bwd else HostPipeline(md, dev)
    Ke = K
    gh = torch.Generator().manual_seed(99 + rank)

    def host_step():
        slot = pipe.acquire((b, c, hf, wf), (b, 1, df, hf, wf))
        return pipe.submit(slot, gcost) if bwd else pipe.submit(slot)

    for _ in range(pipe.depth):              # fill every slot's pinned staging buffer once (the data loader's job), untimed
        slot = pipe.acquire((b, c, hf, wf), (b, 1, df, hf, wf))
        for k, v in slot.host.items():
            v.normal_(generator=gh)
            if k == "gdisp":
                v.mul_((torch.rand(v.shape, generator=gh) < 0.3).float())
        pipe.submit(slot, gcost) if bwd else pipe.submit(slot)
    for _ in range(3):
        host_step()
    pipe.drain()
    barrier()
    e0, e1 = ev(), ev()
    e0.record()
    for _ in range(Ke):
        last = host_step()
    pipe.drain()
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1)
    barrier()
    h2d, d2h = last.h2d_bytes, last.d2h_bytes
    # the box's copy ceiling with the same ranks active: the same bytes, one plain pinned copy per direction, no kernels
    def copy_floor(h2d_bytes, d2h_bytes):
        """What the box's PCIe fabric allows for one step's copies with the same ranks active: the step's H2D bytes as ONE plain
        pinned copy (`h2d_ms`), and the H2D and D2H copies of a step issued together on two streams as the pipeline does
        (`both_ms`: the duplex floor of a step), each the MEDIAN of 12 repetitions timed individually with CUDA events (the
        uplink is shared with the other GPUs of the box and with whoever else is on it: profiles/r2_h2d_ceiling.md)."""
        hin = torch.empty(h2d_bytes // 4, dtype=torch.float32).pin_memory(); hin.zero_()
        din = torch.empty(h2d_bytes // 4, dtype=torch.float32, device=dev)
        hout = torch.empty(d2h_bytes // 4, dtype=torch.float32).pin_memory(); hout.zero_()
        dout = torch.zeros(d2h_bytes // 4, dtype=torch.float32, device=dev)
        sa, sb = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        cur = torch.cuda.current_stream(dev)

        def h2d_only():
            din.copy_(hin, non_blocking=True)

        def both():
            sa.wait_stream(cur); sb.wait_stream(cur)
            with torch.cuda.stream(sa):
                din.copy_(hin, non_blocking=True)
            with torch.cuda.stream(sb):
                hout.copy_(dout, non_blocking=True)
            cur.wait_stream(sa); cur.wait_stream(sb)

        res = []
        for fn in (h2d_only, both):
            for _ in range(2):
                fn()
            barrier()
            ts = []
            for _ in range(12):
                c0, c1 = ev(), ev()
                c0.record(); fn(); c1.record()
                torch.cuda.synchronize()
                ts.append(c0.elapsed_time(c1))
            barrier()
            res.append(sorted(ts)[len(ts) // 2])
        return res

    h2d_ms, both_ms = copy_floor(h2d, d2h)
    e2e_ms, h2d_ms, both_ms = max_over_ranks([e2e_ms, h2d_ms, both_ms])
    checksum = float(last.result["disp"].double().mean())
    e2e_step = e2e_ms / Ke
    e2e = {"value": world * b * Ke / (e2e_ms * 1e-3), "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": Ke, "ms_per_step": e2e_step, "copies_per_step": {"h2d": 1, "d2h": 1},
           "mode": ("forward + backward (training step) through rag_b200.pipeline.HostTrainPipeline" if bwd else "forward (inference) through rag_b200.pipeline.HostPipeline")
                   + ": one coalesced pinned staging buffer per direction, one cudaMemcpyAsync each way per step, double-buffered against the kernels",
           "h2d_GBps_per_rank": round(h2d / (e2e_step * 1e-3) / 1e9, 2),
           # a pipeline cannot beat the link: if the plain-copy sample came out slower than the pipeline's own sustained rate
           # (a neighbour on the shared uplink during the sample), the pipeline's rate IS the better estimate of the ceiling
           "h2d_ceiling_GBps_per_rank": round(max(h2d / (h2d_ms * 1e-3), h2d / (e2e_step * 1e-3)) / 1e9, 2),
           "h2d_plain_copy_sample_GBps": round(h2d / (h2d_ms * 1e-3) / 1e9, 2),
           "frac_of_h2d_ceiling": round(min(1.0, h2d_ms / e2e_step), 4),
           "copy_floor_ms_per_step": round(both_ms, 4), "frac_of_copy_floor": round(min(1.0, both_ms / e2e_step), 4),
           "ceiling_note": "h2d ceiling = the step's H2D bytes as one plain pinned cudaMemcpyAsync on every rank at once; copy floor = the step's H2D and D2H "
                           "copies issued together on two streams, no kernels; medians of 12, slowest rank, measured in this run.  The box's PCIe "
                           "fabric, not the kernels, bounds e2e (profiles/r2_h2d_ceiling.md)",
           "numa_binding": numa, "mean_disp": checksum}
    del pipe
    torch.cuda.empty_cache()

    train = None
    if args.workload == "infer" and not args.no_train_record:
        del tensors
        keep = (x, y)
        trec, ttens = measure("train", with_clocks=False)
        del ttens
        train = {"config": config_dict("train"), "value": trec["value"], "value_serial": trec["value_serial"], "unit": "pairs/s",
                 "ms_per_step": trec["ms_per_step"], "ms_per_step_serial": trec["ms_per_step_serial"], "schedule": trec["schedule"],
                 "roofline": trec["roofline"], "path": trec["path"], "gpu_launches": trec["gpu_launches"], "steps": K, "warmup": Wm}
        torch.cuda.empty_cache()

    cpu = torch_gpu = next_rows = parity = config1 = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        parity = parity_record(args.workload, dev)
        if train is not None:
            train["parity"] = parity_record("train", dev)
            train["torch_cuda_reference"] = torch_cuda_reference("train", dev, reps=3)
            train["cpu_baseline"], _ = cpu_reference("train", warmup=1, steps=3, budget_s=10.0)
        torch_gpu = torch_cuda_reference(args.workload, dev)
        if not bwd:
            next_rows = next_rows_record(x, y, df, md, 8 if args.workload == "router" else b)
        cpu, _ = cpu_reference(args.workload, warmup=1, steps=20, budget_s=15.0)
        if args.workload == "infer":
            config1 = config1_full_network_cpu(budget_s=12.0)

    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_dict(args.workload),
            "schedule": main["schedule"], "value_serial": main["value_serial"], "ms_per_step_serial": main["ms_per_step_serial"],
            "roofline": main["roofline"], "path": main["path"], "train": train, "parity": parity,
            "cpu_baseline": cpu, "config1_full_network_cpu": config1, "torch_cuda_reference": torch_gpu, "next_rows": next_rows,
            "e2e": e2e, "gpu_launches": main["gpu_launches"], "clocks": main["clocks"],
        }
        if args.dump_outputs is not None:
            line["dump_outputs"] = write_outputs(main["outputs"], args.dump_outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="infer")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the host-side legs (cpu_baseline, parity, torch_cuda_reference, next_rows)")
    ap.add_argument("--schedule", choices=["coresident", "launch-order", "slim-volume"], default="coresident",
                    help="kernel variants of the two-stream schedule (rag_b200.pipeline.SCHEDULES)")
    ap.add_argument("--graph", action="store_true", help="additionally time the two-stream step as CUDA-graph replays (path.overlapped_graph)")
    ap.add_argument("--no-train-record", action="store_true", help="default workload only: skip the configs[2] training sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float32; see sample_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
