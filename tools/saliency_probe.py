"""Dual-class input-gradient saliency cost (bcad_predict_saliency_classes), canonical networks, one GPU.

    python tools/saliency_probe.py [--steps 10] [--out profiles/r04_saliency_1gpu.json]

Both canonical flavours: NumPy (valid conv, tie-duplicating pool, softmax head: the reference's saliency network) and torch (pad 1).
512 distinct 256x256x1 images stay on the device (134 MB, more than the 126 MB L2).  Per flavour, fp32 handles with every activation
kept (max_batch 64), fast training off and on.  After a 2-s pre-heat, per handle and step, alternated in one process and timed with
CUDA events around each whole call:
  (a) two K = 1 calls, classes 0 and 1
  (b) one K = 2 call, classes (0, 1)
(b)'s maps are checked bitwise against (a)'s.  One profiled K = 2 call per handle gives the kernel times; saliency_conv0 is set against
the bytes it has to move (reads the block-0 output y and pooled gradient, writes the saliency map).
The reference-shaped loop -- explainability.generate_dual_class_overlays image by image, PNG writes included, on the NumPy mirror's
compat handle -- is timed over 64 images with a host clock (each image ends in device-to-host copies) and reported per image.
Prints one JSON line (and writes it to --out when given)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from util import engine_from, ocnn  # noqa: E402

HBM_DATASHEET_GBS = 7700.0      # NVIDIA HGX B200 data sheet, one GPU
SHAPE = (256, 256, 1)
MB = 64


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


def conv0_bytes(cfg):
    """Bytes saliency_conv0 moves per image and class: y [Ho][Wo][32] and the pooled gradient read, the saliency map written."""
    h, w, _ = cfg.input_shape
    ho, wo = h + 2 * cfg.pad - 2, w + 2 * cfg.pad - 2
    return 4 * (ho * wo * 32 + (ho // 2) * (wo // 2) * 32 + h * w)


def run_handle(cfg, p, x, fast, steps):
    B = x.shape[0]
    eng = engine_from(cfg, p, precision="fp32", max_batch=MB, keep_all_activations=True)
    if fast:
        eng.set_fast_training(True)
    out = {}
    variants = {
        "a_two_k1_calls": lambda: out.__setitem__("a", [eng.predict_saliency_classes(x, (k,), "softmax_ce") for k in (0, 1)]),
        "b_one_k2_call": lambda: out.__setitem__("b", eng.predict_saliency_classes(x, (0, 1), "softmax_ce")),
    }
    t_end = time.time() + 2.0
    while time.time() < t_end:                                  # pre-heat (clocks up, modules loaded, buffers allocated)
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
    res = {k: stats(v) for k, v in times.items()}
    for k in res:
        res[k]["image_classes_per_s"] = B * 2 / (res[k]["median_ms"] * 1e-3)
    res["speedup_a_over_b"] = res["a_two_k1_calls"]["median_ms"] / res["b_one_k2_call"]["median_ms"]
    res["k2_maps_equal_k1_maps"] = bool(all(torch.equal(out["b"][3][:, k], out["a"][k][3][:, 0]) for k in (0, 1)))
    eng.set_profiling(True)
    variants["b_one_k2_call"]()
    torch.cuda.synchronize()
    prof = eng.last_profile()
    eng.set_profiling(False)
    kern = {}
    for n, t in prof:
        if n != "end":
            kern.setdefault(n, [0, 0.0])
            kern[n][0] += 1
            kern[n][1] += t
    res["kernels_k2_call"] = {n: {"launches": c, "ms": round(t, 4)} for n, (c, t) in kern.items()}
    res["profiled_k2_call_ms"] = sum(t for n, t in prof)
    if "saliency_conv0" in kern:
        ms = kern["saliency_conv0"][1]
        nbytes = B * 2 * conv0_bytes(cfg)
        gbs = nbytes / (ms * 1e-3) / 1e9
        res["saliency_conv0"] = {"ms_all_launches": ms, "bytes": nbytes, "achieved_GBps": gbs,
                                 "share_of_datasheet_7700GBps": gbs / HBM_DATASHEET_GBS}
    eng.close()
    return res


def reference_loop(n_images):
    """generate_dual_class_overlays image by image on the NumPy mirror (the reference's per-image call shape)."""
    from bcad_b200.CNNModel import CNNModel
    from bcad_b200 import explainability as E
    np.random.seed(7)
    m = CNNModel(SHAPE, 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[256, 128])
    X = ocnn.synth_images(n_images, SHAPE, seed=20251018, kind="mammo")
    with tempfile.TemporaryDirectory() as d:
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            E.generate_dual_class_overlays(m, X[0], [0, 1], d)       # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(n_images):
                E.generate_dual_class_overlays(m, X[i], [0, 1], d)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
    return {"images": n_images, "ms_per_image": dt / n_images * 1e3, "image_classes_per_s": 2 * n_images / dt,
            "timing": "host clock around the loop; every image ends in device-to-host copies; includes the two PNG writes per class"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--loop-images", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("saliency_probe needs a CUDA device (B200)")
    line = {"probe": "saliency_probe", "card": card(), "batch": a.batch, "steps": a.steps, "max_batch": MB,
            "network": "canonical 256x256x1, conv 32-64, dense 256-128-2",
            "timing": "CUDA events around each whole call, variants alternated per step, inputs device-resident (134 MB > L2)"}
    for flavour in ("numpy", "torch"):
        mk = ocnn.NetConfig.numpy_flavour if flavour == "numpy" else ocnn.NetConfig.torch_flavour
        cfg = mk(SHAPE, 2, [(32, 3), (64, 3)], [256, 128], 0.01)
        p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
        x = torch.from_numpy(ocnn.synth_images(a.batch, SHAPE, seed=20251018, kind="mammo" if flavour == "numpy" else "gauss")).cuda()
        line[flavour] = {("fast_training" if fast else "fp32_kernels"): run_handle(cfg, p, x, fast, a.steps) for fast in (False, True)}
        del x
    line["numpy"]["reference_loop_generate_dual_class_overlays"] = reference_loop(a.loop_images)
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
