"""The dual-class saliency overlays end to end from host buffers: the Python composition a caller needs today and the device composition
against the one-call host path (bcad_saliency_overlays_classes_host), canonical networks, 512 grey 8-bit images, classes 0 and 1.

    python tools/saliency_overlays_probe.py [--steps 10] [--batch 512] [--out-prefix profiles/r06_saliency_overlays]

Per flavour (NumPy: the reference's saliency network; torch) on an fp32 handle with every activation kept, max_batch 64 and fast
training on (what a model's saliency_engine is), and per image size (256x256 = the model's size, 512x512 = the app's), after a 2-s
pre-heat, the variants run alternated in one process, each step timed with the host clock around the whole call:
  host_call_pinned      one bcad_saliency_overlays_classes_host call, pinned input and outputs
  host_call_pageable    the same call from a pageable input array (pinned outputs)
  device_composition    pageable H2D, gray_resize_preprocess, predict_saliency_classes, saliency_overlay_resized, .cpu() of the results
  device_only           predict_saliency_classes + saliency_overlay_resized on a resident CNN input and image, results left on the
                        device (the compute the host call has to hide its copies behind)
  python_composition    cv2.resize(img / 255) and standardisation on the host, explainability.generate_dual_class_overlays_batch
                        (which colours the maps at the model's size on a blend base nobody can read), then per map cv2.resize of its
                        heat-map to the image's size and addWeighted with the grey image, as generate_saliency_overlay does
                        (fewer steps: it takes seconds)
  sharded_<N>gpu        ShardedEngine over N = 2, 4, 8 GPUs where available (pinned input, driver-owned pinned outputs)
Bytes moved = the 8-bit images in + K BGR overlays and K BGR heat-maps out; the copy ceiling is a pinned H2D of the input bytes and a
D2H of the output bytes on two streams at once, measured in the same process.  The colouring kernel is timed with CUDA events over
repeated launches on one 64-image chunk and reported against HBM.  The host call's outputs are checked against the other variants'
(the Python composition resizes its input with cv2 in float32, a few ulp from the device's resize: its differing bytes are counted).
Writes one JSON file per flavour: <prefix>_<flavour>.json."""
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

import bcad_b200  # noqa: E402
from bcad_b200 import engine as E, explainability as X  # noqa: E402
from util import engine_from, ocnn, spec_from_cfg  # noqa: E402

HBM_DATASHEET_GBS = 7700.0      # NVIDIA HGX B200 data sheet, one GPU
K = 2
MB = 64
PY_STEPS = 2


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:          # noqa: BLE001 (the measurement stands without it; say why it is missing)
        return f"unavailable: {e}"


def stats(ts):
    a = np.asarray(ts)
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max()), "steps": len(ts)}


def copy_ceiling(in_bytes, out_bytes, reps=5):
    h_in = torch.empty(in_bytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(in_bytes, dtype=torch.uint8, device="cuda")
    d_out = torch.empty(out_bytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    ts = []
    for _ in range(reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    t = float(np.median(ts[1:]))
    return {"ms": t * 1e3, "GBps": (in_bytes + out_bytes) / t / 1e9}


def device_composition(eng, g):
    h, w, c = eng.spec.input_shape
    gd = torch.from_numpy(g).to(eng.tdev)
    x = E.gray_resize_preprocess(gd, (h, w), c, True)
    cls, probs, _, sal, _ = eng.predict_saliency_classes(x, [0, 1], "softmax_ce")
    ov, hm = E.saliency_overlay_resized(gd, sal)
    return cls.cpu().numpy(), probs.cpu().numpy(), ov.cpu().numpy(), hm.cpu().numpy()


def python_composition(eng, g):
    """What a caller holding grey images of another size does without the host call."""
    import cv2
    h, w, _ = eng.spec.input_shape
    x = np.empty((g.shape[0], h, w, 1), np.float32)
    for b in range(g.shape[0]):
        r = cv2.resize((g[b] / 255.0).astype(np.float32), (w, h), interpolation=cv2.INTER_LINEAR)
        x[b, ..., 0] = (r - r.mean()) / (r.std() + 1e-8)
    model = type("M", (), {"saliency_engine": eng})()
    cls, probs, _, _, heat = X.generate_dual_class_overlays_batch(model, x, [0, 1])
    B, ih, iw = g.shape
    ov = np.empty((B, K, ih, iw, 3), np.uint8)
    hm = np.empty((B, K, ih, iw, 3), np.uint8)
    for b in range(B):
        g3 = np.repeat(g[b][..., None], 3, axis=-1)
        for k in range(K):
            hm[b, k] = cv2.resize(heat[b, k], (iw, ih))
            ov[b, k] = cv2.addWeighted(g3, 0.5, hm[b, k], 0.5, 0)
    return cls, probs, ov, hm


def colouring_kernel_time(hw, n=MB, reps=20):
    g = torch.randint(0, 256, (n, hw, hw), dtype=torch.uint8, device="cuda")
    sal = torch.rand((n, K, 256, 256), device="cuda")
    for _ in range(3):
        E.saliency_overlay_resized(g, sal)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        E.saliency_overlay_resized(g, sal)
    ev[1].record()
    ev[1].synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    nbytes = n * (hw * hw + K * 256 * 256 * 4 + 2 * K * hw * hw * 3)      # image and maps read once, two BGR outputs written once
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"images": n, "image_hw": hw, "ms": ms, "algorithmic_bytes": nbytes, "achieved_GBps": gbs,
            "share_of_datasheet_7700GBps": gbs / HBM_DATASHEET_GBS}


def run_flavour(cfg, p, batch, steps):
    out = {}
    eng = engine_from(cfg, p, precision="fp32", max_batch=MB, keep_all_activations=True)
    eng.set_fast_training(True)
    ngpu = torch.cuda.device_count()
    shard = {}
    for n in (2, 4, 8):
        if n <= ngpu:
            shard[n] = bcad_b200.ShardedEngine(spec_from_cfg(cfg), list(range(n)), precision="fp32", max_batch=MB, keep_all_activations=True)
            shard[n].set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
            shard[n].set_fast_training(True)
    h, w, c = eng.spec.input_shape
    for hw in (256, 512):
        rng = np.random.default_rng(hw)
        g = rng.integers(0, 256, size=(batch, hw, hw), dtype=np.uint8)
        g_pin = torch.from_numpy(g).pin_memory().numpy()
        ov = torch.empty((batch, K, hw, hw, 3), dtype=torch.uint8).pin_memory().numpy()
        hm = torch.empty((batch, K, hw, hw, 3), dtype=torch.uint8).pin_memory().numpy()
        ov2 = torch.empty((batch, K, hw, hw, 3), dtype=torch.uint8).pin_memory().numpy()
        hm2 = torch.empty((batch, K, hw, hw, 3), dtype=torch.uint8).pin_memory().numpy()
        gd = torch.from_numpy(g).cuda()
        xd = E.gray_resize_preprocess(gd, (h, w), c, True)
        results = {}
        variants = {
            "host_call_pinned": lambda: results.__setitem__("pin", eng.saliency_overlays_classes_host(g_pin, (0, 1), "softmax_ce", True, ov, hm)),
            "host_call_pageable": lambda: results.__setitem__("page", eng.saliency_overlays_classes_host(g, (0, 1), "softmax_ce", True, ov2, hm2)),
            "device_composition": lambda: results.__setitem__("dev", device_composition(eng, g)),
            "device_only": lambda: E.saliency_overlay_resized(gd, eng.predict_saliency_classes(xd, [0, 1], "softmax_ce")[3]),
        }
        for n, s in shard.items():
            variants[f"sharded_{n}gpu"] = (lambda s=s, n=n: results.__setitem__(f"sh{n}", s.saliency_overlays_classes_host(g_pin, (0, 1))))
        t_end = time.time() + 2.0
        while time.time() < t_end:                              # pre-heat (clocks up, modules loaded, buffers allocated)
            for f in variants.values():
                f()
        variants["python_composition"] = lambda: results.__setitem__("py", python_composition(eng, g))
        times = {k: [] for k in variants}
        for step in range(steps):
            for name, f in variants.items():
                if name == "python_composition" and step >= PY_STEPS:
                    continue
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                times[name].append((time.perf_counter() - t0) * 1e3)
        in_bytes, out_bytes = batch * hw * hw, batch * K * hw * hw * 3 * 2
        ceil = copy_ceiling(in_bytes, out_bytes)
        res = {"image_hw": hw, "bytes_in": in_bytes, "bytes_out": out_bytes, "copy_ceiling_1gpu": ceil}
        for k, v in times.items():
            r = stats(v)
            r["images_per_s"] = batch / (r["median_ms"] * 1e-3)
            if k != "device_only":
                r["host_GBps"] = (in_bytes + out_bytes) / (r["median_ms"] * 1e-3) / 1e9
            if k.startswith("host_call"):
                r["share_of_copy_ceiling"] = r["host_GBps"] / ceil["GBps"]
            res[k] = r
        res["host_call_over_device_only"] = res["host_call_pinned"]["median_ms"] / res["device_only"]["median_ms"]
        res["speedup_host_call_over_python_composition"] = res["python_composition"]["median_ms"] / res["host_call_pinned"]["median_ms"]
        res["speedup_host_call_over_device_composition"] = res["device_composition"]["median_ms"] / res["host_call_pinned"]["median_ms"]
        c0, p0, _, o0, h0, _ = results["pin"]
        dev, page, py = results["dev"], results["page"], results["py"]
        eq = {
            "host_call_equals_device_composition": bool(np.array_equal(c0, dev[0]) and np.array_equal(p0, dev[1]) and
                                                        np.array_equal(o0, dev[2]) and np.array_equal(h0, dev[3])),
            "pinned_equals_pageable": bool(np.array_equal(c0, page[0]) and np.array_equal(o0, page[3]) and np.array_equal(h0, page[4])),
            "python_composition_classes_equal": bool(np.array_equal(c0, py[0])),
            "python_composition_differing_overlay_bytes": int((o0 != py[2]).sum()),
            "python_composition_differing_heat_bytes": int((h0 != py[3]).sum()),
            "output_bytes_per_kind": int(o0.size),
        }
        for n in shard:
            sc = results[f"sh{n}"]
            eq[f"sharded_{n}gpu_equals_host_call"] = bool(np.array_equal(sc[0], c0) and np.array_equal(sc[3], o0) and np.array_equal(sc[4], h0))
        res["outputs"] = eq
        res["colouring_kernel"] = colouring_kernel_time(hw)
        out[f"{hw}x{hw}"] = res
        del gd, xd
    for s in shard.values():
        s.close()
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--out-prefix", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("saliency_overlays_probe needs a CUDA device (B200)")
    for flavour in ("numpy", "torch"):
        mk = ocnn.NetConfig.numpy_flavour if flavour == "numpy" else ocnn.NetConfig.torch_flavour
        cfg = mk((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
        p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
        line = {"probe": "saliency_overlays_probe", "card": card(), "gpus_visible": torch.cuda.device_count(), "flavour": flavour,
                "batch": a.batch, "classes": [0, 1], "steps": a.steps, "max_batch": MB, "fast_training": True,
                "network": f"canonical 256x256x1, conv 32-64, dense 256-128-2, {flavour} flavour",
                "timing": "host clock around each whole call (outputs in host memory except device_only), variants alternated per step"}
        line.update(run_flavour(cfg, p, a.batch, a.steps))
        s = json.dumps(line)
        print(s, flush=True)
        if a.out_prefix:
            os.makedirs(os.path.dirname(os.path.abspath(a.out_prefix)), exist_ok=True)
            with open(f"{a.out_prefix}_{flavour}.json", "w") as f:
                f.write(s + "\n")


if __name__ == "__main__":
    main()
