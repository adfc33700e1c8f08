"""Dual-class Grad-CAM cost: two single-class calls against one K = 2 call (bcad_predict_explain_classes), canonical network.

    python tools/multiclass_probe.py [--steps 20] [--out profiles/r03_multiclass_1gpu.json]

512 distinct 256x256x1 images stay on the device (134 MB, more than the 126 MB L2).  Handles: fp16 with refinement (the headline
handle) and fp16x3.  Per handle, after a 2-s pre-heat and a warm-up, the variants run alternated in the same process, each step
timed with CUDA events around the whole call:
  (a) two bcad_predict_explain calls, classes 0 and 1
  (b) one bcad_predict_explain_classes call, K = 2
  (c) one bcad_predict_explain call (the single-class cost)
A separate profiled call of (b) and (c) gives the tail kernels' times; achieved GB/s counts the algorithmic bytes of the tail
(the activation map A read once, 2 bytes a value and plane -- fp16x3 stores hi + lo planes -- plus K fp32 heat-maps written).
Prints one JSON line (and writes it to --out when given)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from util import engine_from, ocnn  # noqa: E402

HBM_MEASURED_GBS = 6550.0       # the measured HBM copy rate of the B200 the project states its shares against (DESIGN.md §4)
HBM_DATASHEET_GBS = 7700.0      # NVIDIA HGX B200 data sheet, one GPU


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except Exception as e:          # noqa: BLE001 (the measurement stands without it; say why it is missing)
        return f"unavailable: {e}"


def stats(ts):
    a = np.asarray(ts)
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()),
            "p10_ms": float(np.percentile(a, 10)), "p90_ms": float(np.percentile(a, 90))}


def run_handle(precision, x, cfg, p, steps):
    B = x.shape[0]
    H, W = cfg.input_shape[:2]
    eng = engine_from(cfg, p, precision=precision, max_batch=B)
    c0 = torch.zeros(B, dtype=torch.int32, device="cuda")
    c1 = torch.ones(B, dtype=torch.int32, device="cuda")
    heat_a = torch.empty((2, B, H, W), device="cuda")
    heat_b = torch.empty((B, 2, H, W), device="cuda")
    heat_c = torch.empty((B, H, W), device="cuda")
    out = {}

    def va():
        out["a0"] = eng.predict_explain(x, c0, "logit", out_heat=heat_a[0])
        out["a1"] = eng.predict_explain(x, c1, "logit", out_heat=heat_a[1])

    def vb():
        out["b"] = eng.predict_explain_classes(x, (0, 1), "logit", out_heat=heat_b)

    def vc():
        out["c"] = eng.predict_explain(x, c0, "logit", out_heat=heat_c)

    variants = {"a_two_calls": va, "b_classes_k2": vb, "c_one_class": vc}
    t_end = time.time() + 2.0
    while time.time() < t_end:                                  # pre-heat (clocks up, modules loaded)
        for f in variants.values():
            f()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(steps):
        for name, f in variants.items():
            ev[0].record()
            f()
            ev[1].record()
            ev[1].synchronize()
            times[name].append(ev[0].elapsed_time(ev[1]))
    torch.cuda.synchronize()
    equal = (torch.equal(heat_b[:, 0], heat_a[0]) and torch.equal(heat_b[:, 1], heat_a[1])
             and all(torch.equal(out["b"][i], out["a0"][i]) and torch.equal(out["b"][i], out["a1"][i]) for i in range(3)))
    res = {k: stats(v) for k, v in times.items()}
    for k in res:
        kcls = 1 if k == "c_one_class" else 2
        res[k]["images_classes_per_s"] = B * kcls / (res[k]["median_ms"] * 1e-3)
    res["speedup_a_over_b"] = res["a_two_calls"]["median_ms"] / res["b_classes_k2"]["median_ms"]
    res["outputs_equal_a_b"] = bool(equal)
    # kernel times of one profiled call each (a run of its own, after the timed window)
    C, h, w = 64, 128, 128                                      # the canonical target map (second conv block)
    planes = 2 if precision == "fp16x3" else 1
    kern = {}
    eng.set_profiling(True)
    for name, f, tail, K in (("b", vb, "tail_fused_classes", 2), ("c", vc, "tail_fused", 1)):
        f()
        torch.cuda.synchronize()
        prof = eng.last_profile()
        ms = sum(t for n, t in prof if n == tail)
        nbytes = B * (C * h * w * 2 * planes + K * H * W * 4)
        gbs = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else None
        kern[name] = {"kernel": tail, "ms": ms, "algorithmic_bytes": nbytes, "achieved_GBps": gbs,
                      "share_of_measured_6550GBps": gbs / HBM_MEASURED_GBS if gbs else None,
                      "share_of_datasheet_7700GBps": gbs / HBM_DATASHEET_GBS if gbs else None,
                      "profile": [[n, round(t, 4)] for n, t in prof]}
    eng.set_profiling(False)
    res["tail_kernels"] = kern
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multiclass_probe needs a CUDA device (B200)")
    cfg = ocnn.NetConfig.torch_flavour((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.0)
    x = torch.from_numpy(ocnn.synth_images(a.batch, (256, 256, 1), seed=20251018)).cuda()
    line = {"probe": "multiclass_probe", "card": card(), "batch": a.batch, "steps": a.steps,
            "network": "canonical 256x256x1, conv 32-64, dense 256-128-2, torch flavour",
            "timing": "CUDA events around each whole call, variants alternated per step, inputs device-resident (134 MB > L2)"}
    for precision in ("fp16", "fp16x3"):
        line[precision] = run_handle(precision, x, cfg, p, a.steps)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
