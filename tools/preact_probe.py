"""Grad-CAM of the pre-activation target (set_explain_target("conv_preact")) on the tensor paths against the post-activation target and
the fp32 handle that used to be the only way to get it.  Canonical torch network (256x256, 32/64 filters, hidden 256/128), 512
distinct images.

    python tools/preact_probe.py [--steps 20] [--batch 512] [--out-prefix profiles/r07_preact]

After a 2-s pre-heat, the variants of one table run alternated in one process, each step timed with CUDA events around the whole
device-buffer call:
  predict_explain          one class per image, fp16 (refinement on) and fp16x3 handles: post vs pre
  predict_explain_classes  classes 0 and 1 from one forward, same handles: post vs pre
  fp32 handle              the pre-activation call on an fp32 handle (what ADCNNM.predict_explain_batch(target="conv_preact") runs)
  overlays host call       bcad_gradcam_overlays_classes_host, 512x512 grey 8-bit images, classes 0 and 1, fp16 handle: post vs pre
                           (pinned input and outputs)
Kernel times come from one profiled call per handle in a run of their own (CUDA events between launches).  alpha_preact_tcgen05 is
reported against the data-sheet floors from shapes: FLOP = 2 B units flat x (MMAs issued per product: 2 fp16 -- dz1 as hi + lo --,
3 fp16x3); bytes = the W1 tiles
once per 128-image tile row (134 MB fp16 / 268 MB fp16x3 at hidden 256; the four m-tiles of a split run together and share them through
the L2, so the HBM figure counts them once) + the pooled-map mask (m_pad x flat x 2 B, twice in fp16x3).  Writes
<prefix>_fp16.json, <prefix>_fp16x3.json."""
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

import bcad_b200  # noqa: E402,F401
from util import engine_from, ocnn  # noqa: E402

HBM_DATASHEET_GBS = 7700.0        # NVIDIA HGX B200 data sheet, one GPU
F16_DATASHEET_TFLOPS = 2250.0     # dense FP16, one GPU
PRE = "conv_preact"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:          # noqa: BLE001 (the measurement stands without it; say why it is missing)
        return f"unavailable: {e}"


def stats(ts):
    a = np.asarray(ts)
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()), "n": int(a.size)}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def run_table(variants, steps):
    """variants: {name: (engine, target, fn)} -> {name: stats}; alternated step by step after a 2-s pre-heat of all of them."""
    t_end = time.perf_counter() + 2.0
    while time.perf_counter() < t_end:
        for eng, tgt, fn in variants.values():
            eng.set_explain_target(tgt)
            fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in variants}
    for _ in range(steps):
        for k, (eng, tgt, fn) in variants.items():
            eng.set_explain_target(tgt)
            ts[k].append(timed(fn))
    return {k: stats(v) for k, v in ts.items()}


def profile_of(eng, tgt, fn):
    eng.set_explain_target(tgt)
    fn()
    torch.cuda.synchronize()
    eng.set_profiling(True)
    fn()
    torch.cuda.synchronize()
    prof = eng.last_profile()
    eng.set_profiling(False)
    return prof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--out-prefix", default=os.path.join(ROOT, "profiles", "r07_preact"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "preact_probe measures on the GPU"
    B = a.batch
    cfg = ocnn.NetConfig.torch_flavour((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    x = torch.from_numpy(ocnn.synth_images(B, (256, 256, 1), seed=20251022)).cuda()
    ci = torch.from_numpy((np.arange(B) % 2).astype(np.int32)).cuda()
    rng = np.random.default_rng(5)
    g512 = np.clip(rng.normal(110, 40, size=(B, 512, 512)), 0, 255).astype(np.uint8)
    g512_pinned = torch.from_numpy(g512).pin_memory().numpy()
    ov_out = torch.empty((B, 2, 512, 512, 3), dtype=torch.uint8).pin_memory().numpy()       # pinned outputs: the copies run async
    hu_out = torch.empty((B, 2, 512, 512), dtype=torch.uint8).pin_memory().numpy()
    units, flat = cfg.hidden_units[0], 64 * 64 * 64
    m_pad = -(-B // 128) * 128
    fp32 = engine_from(cfg, p, precision="fp32", max_batch=B)
    for prec in ("fp16", "fp16x3"):
        eng = engine_from(cfg, p, precision=prec, max_batch=B)
        res = {"card": card(), "batch": B, "precision": prec, "refine_margin": eng.refine_margin, "steps": a.steps,
               "network": "torch flavour 256x256x1, conv 32/64, hidden 256/128", "timing": "CUDA events around each call, variants alternated"}
        one = lambda: eng.predict_explain(x, ci, "logit")                                      # noqa: E731
        two = lambda: eng.predict_explain_classes(x, (0, 1), "logit")                          # noqa: E731
        table = {"predict_explain_post": (eng, "conv", one), "predict_explain_pre": (eng, PRE, one),
                 "classes01_post": (eng, "conv", two), "classes01_pre": (eng, PRE, two)}
        if prec == "fp16":
            table["fp32_handle_pre"] = (fp32, PRE, lambda: fp32.predict_explain(x, ci, "logit"))
            ov = lambda: eng.gradcam_overlays_classes_host(g512_pinned, (0, 1), "logit", True, ov_out, hu_out)  # noqa: E731
            table["overlays_host_512_post"] = (eng, "conv", ov)
            table["overlays_host_512_pre"] = (eng, PRE, ov)
        res["calls"] = run_table(table, a.steps)
        # outputs: the pre-activation maps against the fp32 handle's (where a pooled value lies within the path's conv error of 0,
        # LeakyReLU' of that window can switch: tests/test_gpu_preact_tensor.py counts those windows) and against the post-activation maps
        eng.set_explain_target(PRE)
        h_pre = eng.predict_explain(x, ci, "logit")[3]
        fp32.set_explain_target(PRE)
        h_ref = fp32.predict_explain(x, ci, "logit")[3]
        eng.set_explain_target("conv")
        h_post = eng.predict_explain(x, ci, "logit")[3]
        res["max_abs_vs_fp32_handle_pre"] = float((h_pre - h_ref).abs().max())
        res["max_abs_pre_vs_post"] = float((h_pre - h_post).abs().max())
        prof = {"predict_explain_pre": profile_of(eng, PRE, one), "predict_explain_post": profile_of(eng, "conv", one),
                "classes01_pre": profile_of(eng, PRE, two)}
        res["profile"] = {k: [[n, round(t, 4)] for n, t in v] for k, v in prof.items()}
        kt = [t for n, t in prof["predict_explain_pre"] if n == "alpha_preact_tcgen05"]
        mmas = 3 if prec == "fp16x3" else 2            # dz1 enters as hi + lo fp16 parts in both modes (x3: and W1 as hi + lo)
        flop = 2.0 * B * units * flat * mmas
        parts = 2 if prec == "fp16x3" else 1
        w_bytes = flat * units * 2 * parts
        mask_bytes = m_pad * flat * 2 * parts
        hbm_bytes = w_bytes + mask_bytes
        if kt:
            t = kt[0] * 1e-3
            floor_c = flop / (F16_DATASHEET_TFLOPS * 1e12)
            floor_m = hbm_bytes / (HBM_DATASHEET_GBS * 1e9)
            res["alpha_preact_tcgen05"] = {
                "ms": kt[0], "flop": flop, "hbm_bytes": hbm_bytes, "w1_bytes_per_m_tile": w_bytes, "mask_bytes": mask_bytes,
                "achieved_tflops": flop / t / 1e12, "achieved_hbm_gbs": hbm_bytes / t / 1e9,
                "floor_compute_ms": floor_c * 1e3, "floor_hbm_ms": floor_m * 1e3,
                "bound": "compute" if floor_c > floor_m else "hbm", "share_of_floor": max(floor_c, floor_m) / t}
        eng.set_explain_target("conv")
        out = f"{a.out_prefix}_{prec}.json"
        os.makedirs(os.path.dirname(out), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f)
        print(json.dumps(res))
        eng.close()
    fp32.close()


if __name__ == "__main__":
    main()
