"""The dual-class overlay call end to end from host buffers: today's Python composition and two single-class host calls against the
one-call host path (bcad_gradcam_overlays_classes_host), canonical network, 512 grey 8-bit images, classes 0 and 1.

    python tools/overlays_classes_probe.py [--steps 10] [--batch 512] [--out-prefix profiles/r05_overlays_classes]

Per handle (fp16 with refinement, fp16x3) and image size (256x256 = the model's size, 512x512 = the deployed call's), after a 2-s
pre-heat, the variants run alternated in one process, each step timed with the host clock around the whole call (every variant ends
with its outputs in host memory):
  python_composition   today's composition (model size only): pageable H2D, gray_preprocess, predict_explain_classes, the expanded
                       [B*K,H,W] base image, overlay, two pageable .cpu() copies
  two_single_class     two bcad_gradcam_overlays_host calls, classes 0 and 1 (model size only)
  host_call_pinned     one bcad_gradcam_overlays_classes_host call, pinned input and outputs
  host_call_pageable   the same call from a pageable input array (pinned outputs)
  sharded_<N>gpu       ShardedEngine over N = 1, 2, 4, 8 GPUs where available (pinned input, driver-owned pinned outputs)
Bytes moved = the 8-bit images in + K RGB overlays and K heatmap_uint8 out; the copy ceiling is a pinned H2D of the input bytes and a
D2H of the output bytes on two streams at once, measured in the same process.  The two new kernels are timed with CUDA events over
repeated launches of one 128-image chunk (device buffers larger than the L2) and reported against HBM.  Writes one JSON file per
handle: <prefix>_<precision>.json."""
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
from bcad_b200 import engine as E  # noqa: E402
from util import engine_from, ocnn, spec_from_cfg  # noqa: E402

HBM_DATASHEET_GBS = 7700.0      # NVIDIA HGX B200 data sheet, one GPU
K = 2


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:          # noqa: BLE001 (the measurement stands without it; say why it is missing)
        return f"unavailable: {e}"


def stats(ts):
    a = np.asarray(ts)
    return {"median_ms": float(np.median(a)), "min_ms": float(a.min()), "max_ms": float(a.max())}


def python_composition(eng, g, standardise=True):
    """GRADCAM.generate_dual_class_gradcam_overlays_batch before the one-call host path (model-size images only)."""
    h, w, c = eng.spec.input_shape
    B = g.shape[0]
    img01, x = E.gray_preprocess(torch.from_numpy(g).to(eng.tdev), c, standardise)
    cls, probs, _, heat = eng.predict_explain_classes(x, [0, 1], "logit")
    img_k = img01[:, None].expand(B, K, h, w).reshape(B * K, h, w)
    ov, hu = E.overlay(img_k, heat.reshape(B * K, h, w))
    return (cls.cpu().numpy().astype(np.int64), probs.cpu().numpy(), ov.reshape(B, K, h, w, 3).cpu().numpy(),
            hu.reshape(B, K, h, w).cpu().numpy())


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


def kernel_times(hw, c_in=1, n=128, reps=20):
    """CUDA-event times of the two new kernels on one chunk; algorithmic bytes (each input read once, each output written once)."""
    g = torch.randint(0, 256, (n, hw, hw), dtype=torch.uint8, device="cuda")
    cams = torch.rand((n, K, hw, hw), device="cuda")
    res = {}
    for name, f, nbytes in (
            ("gray_resize_preprocess_to_256", lambda: E.gray_resize_preprocess(g, (256, 256), c_in, True), n * (hw * hw + 256 * 256 * 4 * c_in)),
            ("overlay_classes_k2", lambda: E.overlay_classes(g, cams), n * (hw * hw + K * hw * hw * (4 + 3 + 1)))):
        for _ in range(3):
            f()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(reps):
            f()
        ev[1].record()
        ev[1].synchronize()
        ms = ev[0].elapsed_time(ev[1]) / reps
        gbs = nbytes / (ms * 1e-3) / 1e9
        res[name] = {"images": n, "image_hw": hw, "ms": ms, "algorithmic_bytes": nbytes, "achieved_GBps": gbs,
                     "share_of_datasheet_7700GBps": gbs / HBM_DATASHEET_GBS}
    return res


def run_handle(precision, cfg, p, batch, steps):
    out = {}
    eng = engine_from(cfg, p, precision=precision, max_batch=batch)
    ngpu = torch.cuda.device_count()
    worlds = [n for n in (1, 2, 4, 8) if n <= ngpu]
    shard = {n: bcad_b200.ShardedEngine(spec_from_cfg(cfg), list(range(n)), precision=precision, max_batch=batch) for n in worlds}
    for s in shard.values():
        s.set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
    for hw in (256, 512):
        rng = np.random.default_rng(hw)
        g = rng.integers(0, 256, size=(batch, hw, hw), dtype=np.uint8)
        g_pin = torch.from_numpy(g).pin_memory().numpy()
        ov = torch.empty((batch, K, hw, hw, 3), dtype=torch.uint8).pin_memory().numpy()
        hu = torch.empty((batch, K, hw, hw), dtype=torch.uint8).pin_memory().numpy()
        ov1 = [torch.empty((batch, hw, hw, 3), dtype=torch.uint8).pin_memory().numpy() for _ in range(K)]
        hu1 = [torch.empty((batch, hw, hw), dtype=torch.uint8).pin_memory().numpy() for _ in range(K)]
        results = {}
        variants = {}
        if hw == 256:
            variants["python_composition"] = lambda: results.__setitem__("py", python_composition(eng, g))
            variants["two_single_class"] = lambda: results.__setitem__("two", [eng.gradcam_overlays_host(g_pin, k, "logit", True, ov1[k], hu1[k])
                                                                              for k in range(K)])
        variants["host_call_pinned"] = lambda: results.__setitem__("pin", eng.gradcam_overlays_classes_host(g_pin, (0, 1), "logit", True, ov, hu))
        variants["host_call_pageable"] = lambda: eng.gradcam_overlays_classes_host(g, (0, 1), "logit", True, ov, hu)
        for n, s in shard.items():
            variants[f"sharded_{n}gpu"] = (lambda s=s, n=n: results.__setitem__(f"sh{n}", s.gradcam_overlays_classes_host(g_pin, (0, 1))))
        t_end = time.time() + 2.0
        while time.time() < t_end:                              # pre-heat (clocks up, modules loaded, buffers allocated)
            for f in variants.values():
                f()
        times = {k: [] for k in variants}
        for _ in range(steps):
            for name, f in variants.items():
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                times[name].append((time.perf_counter() - t0) * 1e3)
        in_bytes, out_bytes = batch * hw * hw, batch * K * hw * hw * 4
        ceil = copy_ceiling(in_bytes, out_bytes)
        res = {"image_hw": hw, "bytes_in": in_bytes, "bytes_out": out_bytes, "copy_ceiling_1gpu": ceil}
        for k, v in times.items():
            r = stats(v)
            r["images_per_s"] = batch / (r["median_ms"] * 1e-3)
            r["host_GBps"] = (in_bytes + out_bytes) / (r["median_ms"] * 1e-3) / 1e9
            if not k.startswith("sharded") or k == "sharded_1gpu":
                r["share_of_copy_ceiling"] = r["host_GBps"] / ceil["GBps"]
            res[k] = r
        c, pr, _, o, h = results["pin"]
        eq = {}
        if hw == 256:
            py = results["py"]
            eq["host_call_equals_python_composition"] = bool(np.array_equal(c, py[0]) and np.array_equal(pr, py[1]) and
                                                             np.array_equal(o, py[2]) and np.array_equal(h, py[3]))
            eq["host_call_equals_two_single_class"] = bool(all(np.array_equal(o[:, k], ov1[k]) and np.array_equal(h[:, k], hu1[k])
                                                               for k in range(K)))
        for n in shard:
            sc = results[f"sh{n}"]
            eq[f"sharded_{n}gpu_equals_host_call"] = bool(np.array_equal(sc[0], c) and np.array_equal(sc[3], o) and np.array_equal(sc[4], h))
        res["outputs_equal"] = eq
        if hw == 256 and "python_composition" in res:
            res["speedup_host_call_over_python_composition"] = res["python_composition"]["median_ms"] / res["host_call_pinned"]["median_ms"]
            res["speedup_host_call_over_two_single_class"] = res["two_single_class"]["median_ms"] / res["host_call_pinned"]["median_ms"]
        out[f"{hw}x{hw}"] = res
    out["kernels"] = {f"{hw}x{hw}": kernel_times(hw) for hw in (256, 512)}
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
        raise SystemExit("overlays_classes_probe needs a CUDA device (B200)")
    cfg = ocnn.NetConfig.torch_flavour((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.0)
    for precision in ("fp16", "fp16x3"):
        line = {"probe": "overlays_classes_probe", "card": card(), "gpus_visible": torch.cuda.device_count(), "precision": precision,
                "batch": a.batch, "classes": [0, 1], "steps": a.steps,
                "network": "canonical 256x256x1, conv 32-64, dense 256-128-2, torch flavour",
                "timing": "host clock around each whole call (outputs in host memory), variants alternated per step"}
        line.update(run_handle(precision, cfg, p, a.batch, a.steps))
        s = json.dumps(line)
        print(s, flush=True)
        if a.out_prefix:
            os.makedirs(os.path.dirname(os.path.abspath(a.out_prefix)), exist_ok=True)
            with open(f"{a.out_prefix}_{precision}.json", "w") as f:
                f.write(s + "\n")


if __name__ == "__main__":
    main()
