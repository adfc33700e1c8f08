#!/usr/bin/env python
"""Benchmark of the hot path: batched predict + Grad-CAM images/s at 256x256 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of predict + Grad-CAM over one batch of synthetic images that is already resident
in HBM (value) or sits in pinned host memory (e2e, through the host-buffer C-ABI call).  Workload at N=1 is
BASELINE.json configs[1]: the ADCNNM-flavour CNN (conv 32,64 k3 pad1 / fc 256,128 / 2 classes, random init)
on 512 synthetic 256x256x1 images; at N>1 each rank runs that same batch on its own GPU (weak scaling, no
collective on the data path); rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "predict+Grad-CAM images/sec at 256x256"
UNIT = "images/s"
INPUT_SHAPE = (256, 256, 1)
CONV_LAYERS = [(32, 3), (64, 3)]
HIDDEN = [256, 128]
NUM_CLASSES = 2
FLAVOUR = "torch"          # "numpy": the reference's NumPy CNN (valid conv, HWC flatten, tie-duplicating pool, softmax) -- secondary line


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# algorithmic work per image (SURVEY 8d), same-pad ADCNNM flavour at 256x256x1
# ------------------------------------------------------------------------------------------------
def algorithmic_flops_per_image():
    h, w, c = INPUT_SHAPE
    fl = {}
    cin = c
    for i, (f, k) in enumerate(CONV_LAYERS):
        if FLAVOUR == "numpy":
            h, w = h - k + 1, w - k + 1                       # valid conv
        fl[f"conv{i}"] = 2.0 * h * w * f * k * k * cin       # (same-pad: output map == input map)
        h, w, cin = h // 2, w // 2, f
    flat = h * w * cin
    prev, dense = flat, 0.0
    for u in HIDDEN + [NUM_CLASSES]:
        dense += 2.0 * prev * u
        prev = u
    fl["dense_fwd"] = dense
    fl["dense_bwd"] = dense
    return fl


def tail_bytes_per_image(elem_size):
    h, w = INPUT_SHAPE[0] // 2, INPUT_SHAPE[1] // 2      # last conv map (128x128x64 at 256x256)
    k = CONV_LAYERS[-1][0]
    return 2.0 * k * h * w * elem_size + INPUT_SHAPE[0] * INPUT_SHAPE[1] * 4.0


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "25"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def start_under_load(self, step, sync, max_s=3.0):
        """Start the sampler and keep the device busy with `step` until its first line is in: nvidia-smi's start-up (NVML initialisation
        takes driver-wide locks) otherwise stalls the first launches of a short timed region."""
        self.start()
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < max_s:
            for _ in range(10):
                step()
            sync()
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY 8d) -- generated HERE, not by oracle/: the product arm never touches the oracle except for the
# untimed `check` below (the checker) and the cpu_baseline leg
# ------------------------------------------------------------------------------------------------
def synth_weights(seed=7):
    """Random-init weights of the ADCNNM-flavour network with the reference's own initialisers (He-normal conv
    Classes/CNNModel.py:94, Glorot-uniform dense :131-132, zero biases), seeded.  Layouts: conv (F,k,k,C), dense (units, C*H*W)."""
    rng = np.random.default_rng(seed)
    conv_w, conv_b, dense_w, dense_b = [], [], [], []
    h, w, c = INPUT_SHAPE
    for f, k in CONV_LAYERS:
        conv_w.append(rng.standard_normal((f, k, k, c)) * np.sqrt(2.0 / (k * k * c)))
        conv_b.append(np.zeros(f))
        if FLAVOUR == "numpy":
            h, w = h - k + 1, w - k + 1                       # valid conv
        h, w, c = h // 2, w // 2, f                           # (same-pad conv for the torch flavour) + 2x2 pool
    prev = h * w * c
    for units in HIDDEN + [NUM_CLASSES]:
        lim = np.sqrt(6.0 / (prev + units))
        dense_w.append(rng.uniform(-lim, lim, (units, prev)))
        dense_b.append(np.zeros(units))
        prev = units
    return conv_w, conv_b, dense_w, dense_b


def synth_images(n, shape, seed):
    """Per-image standardised float32 [n,H,W,C] (the reference normalises its inputs: Classes/ImageSegmentation.py:229-232)."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n,) + tuple(shape)).astype(np.float32)
    mean = x.mean(axis=(1, 2, 3), keepdims=True)
    std = x.std(axis=(1, 2, 3), keepdims=True)
    return ((x - mean) / std).astype(np.float32)


DUMP_HEAT_BYTES = 32 << 20        # --dump-outputs: heat-map share of the dump (the whole dump stays under 64 MB)


def dump_sample(n_images, pixels_per_map):
    """Sorted indices of the images whose heat-maps --dump-outputs writes: all of them when they fit DUMP_HEAT_BYTES,
    else a fixed seeded sample, so that two runs with the same arguments dump the same images."""
    k = min(n_images, DUMP_HEAT_BYTES // (4 * pixels_per_map))
    if k == n_images:
        return np.arange(n_images)
    return np.sort(np.random.default_rng(0).choice(n_images, k, replace=False))


def write_dump(out_dir, arrays):
    """--dump-outputs: every array as <out_dir>/<name>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] outputs of the last timed step: {', '.join(f'{k}{list(v.shape)}' for k, v in arrays.items())} -> {out_dir}")


def oracle_setup():
    """Checker / CPU-baseline legs only: the oracle's view (config + Params) of the same synthetic weights."""
    from oracle import cnn as ocnn
    mk = ocnn.NetConfig.numpy_flavour if FLAVOUR == "numpy" else ocnn.NetConfig.torch_flavour
    cfg = mk(INPUT_SHAPE, NUM_CLASSES, CONV_LAYERS, HIDDEN, 0.01)
    params = ocnn.Params(*synth_weights())
    return ocnn, cfg, params


_ALL_CPUS = None


def bind_to_gpu_numa_node(gpu_index):
    """Pin this rank's host thread (and therefore its pinned staging buffers, first-touched next) to the CPUs NVML reports as
    local to the GPU: with several ranks per node the host<->device copies of the e2e leg stay off the inter-socket link."""
    global _ALL_CPUS
    try:
        import pynvml
        if _ALL_CPUS is None:
            _ALL_CPUS = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * i + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1} & _ALL_CPUS
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception as e:                                  # affinity is an optimisation, never a requirement
        log(f"[bench] NUMA binding skipped: {e}")
    return None


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU baseline is meant to use every host core."""
    import torch
    if _ALL_CPUS is not None:
        try:
            os.sched_setaffinity(0, _ALL_CPUS)
        except Exception:
            pass
    n = os.cpu_count() or 1
    try:
        torch.set_num_threads(n)
    except Exception:
        pass
    return torch.get_num_threads()


def cpu_reference_rate(n_images, batch=32, repeats=1):
    """The reference's CPU path (oracle port of ADCNNM + autograd Grad-CAM + NumPy tail) on the host cores."""
    import torch
    from oracle import cpu_port
    use_all_host_threads()
    _, cfg, params = oracle_setup()
    rate, secs = cpu_port.time_predict_gradcam(cfg, params, n_images, batch=batch, repeats=repeats)
    return rate, secs, torch.get_num_threads()


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the reference is
    Python and cannot travel to the GPU box).  Rank 0 alone runs and prints."""
    if rank != 0:
        return
    import torch
    use_all_host_threads()
    n_per_step = args.ref_images
    _, cfg, params = oracle_setup()
    from oracle import cpu_port
    from oracle import cnn as ocnn
    model = cpu_port.build(cfg, params)
    x = torch.from_numpy(synth_images(n_per_step, INPUT_SHAPE, seed=20251018))

    def step():
        for s in range(0, n_per_step, 32):
            cpu_port.predict_gradcam(model, x[s:s + 32])

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = n_per_step * args.steps / dt
    sample = f"{n_per_step} synthetic {'x'.join(map(str, INPUT_SHAPE))} images per step in batches of 32 (bounded sample of the batch-512 workload)"
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.batch, "cpu"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


def workload_config(batch, precision, total_batch=0, refine_margin=0.0):
    d = _workload_config(batch, precision)
    if total_batch:
        d["total_batch"] = total_batch
        d["workload"] += f" (strong scaling: {total_batch} images per step split over the GPUs, BASELINE cfg 4)"
    if refine_margin:
        d["refine_margin"] = refine_margin
        d["workload"] += f"; images with a top-2 logit gap < {refine_margin} re-run at fp32 grade inside the call"
    d["inputs"] = "every image of the batch distinct"
    return d


def _workload_config(batch, precision):
    h, w, c = INPUT_SHAPE
    tag = "cfg2" if INPUT_SHAPE == (256, 256, 1) else "secondary shape (SURVEY 8d)"
    if FLAVOUR == "numpy":
        return {"workload": f"secondary line: NumPy-flavour CNN of Classes/CNNModel.py (conv 32,64 k3 valid; HWC flatten; tie-duplicating "
                            f"pool; softmax head; fc 256,128; random init) predict+Grad-CAM(last conv, predicted class, softmax-CE top "
                            f"gradient), {h}x{w}x{c} fp32 NHWC, batch {batch} per GPU",
                "batch_per_gpu": batch, "precision_path": precision, "l2_policy": "inputs + activations per step exceed the 126 MB L2"}
    return {"workload": f"{tag}: ADCNNM-flavour CNN (conv 32,64 k3 pad1; fc 256,128; {NUM_CLASSES} classes; random init) "
                        f"predict+Grad-CAM(last conv, predicted class), {h}x{w}x{c} fp32 NHWC, batch {batch} per GPU",
            "batch_per_gpu": batch, "precision_path": precision,
            "l2_policy": "inputs + activations per step (>= 134 MB input, GBs of activations) exceed the 126 MB L2"}


# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import bcad_b200

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        bind_to_gpu_numa_node(local_rank)
    conv_w, conv_b, dense_w, dense_b = synth_weights()
    B = args.batch
    if args.total_batch:
        if args.total_batch % world:
            raise SystemExit(f"--total-batch {args.total_batch} is not a multiple of {world} GPUs")
        B = args.total_batch // world
    MB = min(B, 512)                                # handle workspace: larger steps run as 512-image chunks
    mk_spec = bcad_b200.NetSpec.numpy_flavour if FLAVOUR == "numpy" else bcad_b200.NetSpec.torch_flavour
    spec = mk_spec(INPUT_SHAPE, NUM_CLASSES, CONV_LAYERS, HIDDEN, 0.01)
    precision = args.precision
    eng = None
    if precision in ("auto", "fp16", "fp16x3"):
        want = ("fp16x3" if FLAVOUR == "numpy" else "fp16") if precision == "auto" else precision
        try:
            eng = bcad_b200.Engine(spec, precision=want, max_batch=MB, device=local_rank, refine_margin=args.refine_margin)
            precision = want
        except ValueError as e:
            if args.precision != "auto":
                raise
            log(f"[bench] fp16 tensor path unavailable ({e}); using the fp32 CUDA-core path")
    if eng is None:
        eng = bcad_b200.Engine(spec, precision="fp32", max_batch=MB, device=local_rank)
        precision = "fp32"
    eng.set_weights(conv_w, conv_b, dense_w, dense_b)

    # synthetic inputs: B distinct images per rank (seed + rank); generated once, resident in HBM for `value`
    x_host = torch.from_numpy(synth_images(B, INPUT_SHAPE, seed=20251018 + rank)).pin_memory()
    x_dev = x_host.to(dev)
    heat_dev = torch.empty((B, INPUT_SHAPE[0], INPUT_SHAPE[1]), device=dev, dtype=torch.float32)
    heat_host = torch.empty((B, INPUT_SHAPE[0], INPUT_SHAPE[1]), dtype=torch.float32).pin_memory()
    heat8_host = torch.empty((B, INPUT_SHAPE[0], INPUT_SHAPE[1]), dtype=torch.uint8).pin_memory()
    x8_host = torch.from_numpy(np.clip(np.rint(x_host.numpy() * 255.0), 0, 255).astype(np.uint8)).pin_memory()

    GRAD = "softmax_ce" if FLAVOUR == "numpy" else "logit"       # the top gradient each reference API uses

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def preheat(fn, seconds):
        """Full duty for `seconds` before a timed region, so a short --steps run is a sample of the SUSTAINED state (clocks
        and power settled under the 1 kW cap), not of a cold burst."""
        t0 = time.perf_counter()
        n = 0
        while time.perf_counter() - t0 < seconds:
            for _ in range(25):
                fn()
            torch.cuda.synchronize(dev)
            n += 25
        return n

    def measure(e):
        """One engine through every leg: device-resident `value`, host-buffer e2e legs, per-kernel profile under load."""
        def step_dev():
            return e.predict_explain(x_dev, None, GRAD, out_heat=heat_dev)

        def step_host():
            return e.predict_explain_host(x_host.numpy(), None, GRAD, heat_out=heat_host.numpy())

        def step_host_u8():      # same call, heat-maps as heatmap_uint8 (GRADCAM.py:70): informational, NOT the headline e2e
            return e.predict_explain_host(x_host.numpy(), None, GRAD, heat_out=heat8_host.numpy(), heat_dtype=np.uint8)

        def step_host_u8io():    # 8-bit pixels in (normalised /255 on the device, app.py:71), heatmap_uint8 out: informational as well
            return e.predict_explain_host(x8_host.numpy(), None, GRAD, heat_out=heat8_host.numpy(), heat_dtype=np.uint8)

        r = {}
        # ---- device-resident throughput (value)
        for _ in range(args.warmup):
            step_dev()
        barrier()
        r["preheat_steps"] = preheat(step_dev, args.preheat)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start_under_load(step_dev, lambda: torch.cuda.synchronize(dev))
        for _ in range(10):
            step_dev()                                            # the sampler's first lines already see the load
        l0 = e.launch_count
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(args.steps):
            out = step_dev()
        ev1.record()
        barrier()
        r["launches"] = e.launch_count - l0
        r["ms_total"] = ev0.elapsed_time(ev1)
        r["out"] = out
        if args.dump_outputs and e is eng:    # copied now: every later call rewrites heat_dev
            cls, probs, logits, heat = out
            rows = torch.from_numpy(dump_sample(B, INPUT_SHAPE[0] * INPUT_SHAPE[1])).to(dev)
            r["dump"] = {"classes": cls.cpu().numpy().astype(np.float32), "probs": probs.cpu().numpy(),
                         "logits": logits.cpu().numpy(), "heatmaps": heat.index_select(0, rows).cpu().numpy()}
        # ---- per-kernel device times (CUDA events before every kernel) taken UNDER LOAD: profiled steps run back to back
        # right behind the timed region and only the last call of each group is read
        e.set_profiling(True)
        prof, nprof = {}, 3
        for _ in range(nprof):
            for _ in range(8):
                step_dev()
            torch.cuda.synchronize(dev)
            for i, (name, ms) in enumerate(e.last_profile()):
                key = f"{i:02d}:{name}"
                prof[key] = prof.get(key, 0.0) + ms / nprof
        # the same step with the two conv blocks as separate kernels (the fused kernel is the production default because the
        # whole step is faster; the stand-alone second block is the cleaner tensor-core roofline point)
        prof2 = {}
        if rank == 0 and any("conv01" in k for k in prof) and "BCAD_TWO_CONV_KERNELS" not in os.environ and not args.only_value:
            os.environ["BCAD_TWO_CONV_KERNELS"] = "1"
            try:
                for _ in range(nprof):
                    for _ in range(8):
                        step_dev()
                    torch.cuda.synchronize(dev)
                    for i, (name, ms) in enumerate(e.last_profile()):
                        prof2[name] = prof2.get(name, 0.0) + ms / nprof
            finally:
                del os.environ["BCAD_TWO_CONV_KERNELS"]
        e.set_profiling(False)
        r["prof"], r["prof2"] = prof, prof2
        if args.only_value:                       # profiling runs (ncu): the device-resident leg only
            r["clocks"] = sampler.stop() if rank == 0 else None
            r["e2e_ms"] = r["e2e_u8_ms"] = r["e2e_u8io_ms"] = float("nan")
            return r
        # ---- end to end through the host-buffer C-ABI call (e2e)
        for _ in range(max(1, min(args.warmup, 3))):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host()
        torch.cuda.synchronize(dev)
        r["e2e_s"] = time.perf_counter() - t0
        barrier()
        r["clocks"] = sampler.stop() if rank == 0 else None
        step_host_u8()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host_u8()
        torch.cuda.synchronize(dev)
        r["e2e_u8_s"] = time.perf_counter() - t0
        barrier()
        step_host_u8io()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host_u8io()
        torch.cuda.synchronize(dev)
        r["e2e_u8io_s"] = time.perf_counter() - t0
        barrier()
        tt = torch.tensor([r["ms_total"], r["e2e_s"] * 1e3, r["e2e_u8_s"] * 1e3, r["e2e_u8io_s"] * 1e3], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        r["ms_total"], r["e2e_ms"], r["e2e_u8_ms"], r["e2e_u8io_ms"] = (float(v) for v in tt)
        return r

    def host_copy_probe(iters=8):
        """The ceiling of the e2e leg on this box: every rank moves the step's bytes (pinned H2D of the input batch and pinned D2H
        of the heat-maps, two streams, both directions at once) with NO compute in between -> aggregate GB/s over all ranks."""
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        def once():
            with torch.cuda.stream(s_in):
                x_dev.copy_(x_host, non_blocking=True)
            with torch.cuda.stream(s_out):
                heat_host.copy_(heat_dev, non_blocking=True)
        once()
        barrier()
        t0 = time.perf_counter()
        for _ in range(iters):
            once()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        nbytes = (x_host.numel() + heat_host.numel()) * 4 * iters * world
        return nbytes / float(tt[0]) / 1e9, float(tt[0]) / iters * 1e3

    def measure_api():
        """End to end through the reference-shaped Python surface: GRADCAM.generate_gradcam_overlays_batch on a drop-in
        ADCNNM.CNNModel with DEFAULT settings (precision auto): uint8 grey images in pinned host memory in, uint8 RGB overlays
        (show_cam_on_image) + heatmap_uint8 out (GRADCAM.py:31-81), everything in between on the device."""
        from bcad_b200 import ADCNNM as A, GRADCAM as G
        model = A.CNNModel(INPUT_SHAPE, NUM_CLASSES, conv_layers=CONV_LAYERS, hidden_units=HIDDEN, max_batch=MB, device_index=local_rank).eval()
        sd = {}
        for i, (w, b) in enumerate(zip(conv_w, conv_b)):
            sd[f"convs.{i}.weight"] = torch.tensor(np.ascontiguousarray(w.transpose(0, 3, 1, 2)), dtype=torch.float32)
            sd[f"convs.{i}.bias"] = torch.tensor(b, dtype=torch.float32)
        for j, (w, b) in enumerate(zip(dense_w, dense_b)):
            sd[f"fc.{3 * j}.weight"] = torch.tensor(w, dtype=torch.float32)
            sd[f"fc.{3 * j}.bias"] = torch.tensor(b, dtype=torch.float32)
        model.load_state_dict(sd)
        g8 = x8_host.numpy().reshape(B, INPUT_SHAPE[0], INPUT_SHAPE[1])
        ov_host = torch.empty((B, INPUT_SHAPE[0], INPUT_SHAPE[1], 3), dtype=torch.uint8).pin_memory()
        def step():
            return G.generate_gradcam_overlays_batch(g8, None, model=model, overlay_out=ov_host.numpy(), heat_out=heat8_host.numpy())
        for _ in range(3):
            step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        prec = model.engine.precision
        model.engine.close()
        return {"value": world * B * args.steps / float(tt[0]), "unit": UNIT, "ms_per_step": float(tt[0]) / args.steps * 1e3,
                "h2d_bytes_per_step": int(g8.size), "d2h_bytes_per_step": int(ov_host.numel() + heat8_host.numel() + B * (2 * NUM_CLASSES * 4 + 4)),
                "precision_path": prec,
                "api": "GRADCAM.generate_gradcam_overlays_batch(uint8 [B,H,W], model=ADCNNM.CNNModel(...)) with the mirror's DEFAULT precision: "
                       "uint8 grey images in -> uint8 RGB show_cam_on_image overlays + heatmap_uint8 out (GRADCAM.py:31-81), one "
                       "bcad_gradcam_overlays_host call per step"}

    main = measure(eng)
    ceiling_gbs, ceiling_ms = (float("nan"), float("nan")) if args.only_value else host_copy_probe()
    api = None
    if FLAVOUR == "torch" and INPUT_SHAPE[2] == 1 and not args.no_api and not args.only_value:
        try:
            api = measure_api()
        except Exception as e:                                      # the API leg must not take the headline down with it
            log(f"[bench] e2e_api leg failed: {e!r}")
    # ---- the same workload at fp32 grade (hi+lo split operands, 3 MMAs per product): the mode the drop-in mirrors default to
    eng3, grade = None, None
    if precision == "fp16" and not args.no_fp32_grade:
        try:
            eng3 = bcad_b200.Engine(spec, precision="fp16x3", max_batch=MB, device=local_rank)
            eng3.set_weights(conv_w, conv_b, dense_w, dense_b)
            grade = measure(eng3)
        except ValueError as e:
            log(f"[bench] fp16x3 not available for this shape ({e})")
    if rank != 0:
        return
    ms_total, e2e_ms, e2e_u8_ms, e2e_u8io_ms = main["ms_total"], main["e2e_ms"], main["e2e_u8_ms"], main["e2e_u8io_ms"]
    launches, prof, prof2, clocks = main["launches"], main["prof"], main["prof2"], main["clocks"]

    # ---- the result against the oracle on EVERY one of the first --check-images images (not timed): a fast wrong answer is
    # not a result.  oracle/compare.py: classes, logits, heat-maps per image; LeakyReLU-kink handling as in the tests
    check, check3 = None, None
    if not args.no_check:
        from oracle.compare import compare_all_images
        ocnn, cfg, params = oracle_setup()
        k = min(B, args.check_images)
        bounds = {"fp16": (1e-2, 1e-2, 1.5e-2), "fp16x3": (2e-4, 5e-4, 5e-4), "fp32": (1e-4, 1e-4, 1e-4)}
        engs = [(eng, bounds[precision][2])] + ([(eng3, bounds["fp16x3"][2])] if eng3 is not None else [])
        res = compare_all_images(cfg, params, x_host[:k].numpy(), engs, [(None, GRAD)], tau=None)

        def summarise(r, prec, e):
            tol_l, tol_h, tau = bounds[prec]
            scale = max(1.0, float(r["logit_absmax"].max()))
            d = {"images": k, "vs": "float64 oracle (oracle/cnn.py + oracle/gradcam.py), every image compared (oracle/compare.py)",
                 "class_mismatches": int((~r["cls_equal"]).sum()), "classes_equal": bool(r["cls_equal"].all()),
                 "max_logit_err": float(r["logit_err"].max()), "logit_tol": tol_l * scale,
                 "max_heat_err": float(r["heat_err"].max()), "heat_tol": tol_h,
                 "maps_out_of_tolerance": int((r["heat_err"] > tol_h).sum()),
                 "hidden_units_on_the_other_leaky_branch_with_abs_z_above_tau": int(r["mask_violations"]), "tau": tau,
                 "images_with_a_near_kink_branch_override": int(r["overridden"].sum())}
            if e.refine_margin > 0:
                refined, overflow = e.refine_stats()
                d["refine"] = {"margin": e.refine_margin, "images_rerun_at_fp32_grade_since_creation": refined, "overflowed": overflow}
            return d
        check = summarise(res[0][0], precision, eng)
        if eng3 is not None:
            check3 = summarise(res[1][0], "fp16x3", eng3)
    pk = peaks()
    fl = algorithmic_flops_per_image()
    step_ms = ms_total / args.steps
    value = world * B * args.steps / (ms_total * 1e-3)
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)

    def kernel_table(prof):
        tot = max(1e-9, sum(prof.values()))
        return [{"kernel": key, "ms": round(ms, 4), "share": round(ms / tot, 4)} for key, ms in sorted(prof.items())]

    def roofline_of(prof, prof2, prec):
        """Dominant kernel of a profile -> roofline object (`frac` against the SUSTAINED measured peak: the kernel times are
        taken under load; `frac_burst` against the burst peak)."""
        dom_key = max(prof, key=prof.get)
        dom_ms = prof[dom_key]
        name = dom_key.split(":", 1)[1]
        def tensor(flops, extra=None):
            ach = flops / (dom_ms * 1e-3) / 1e12
            d = {"bound": "tensor", "kernel": name, "ms": dom_ms, "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                 "frac": ach / pk["bf16_tflops_sustained"], "peak_burst": pk["bf16_tflops"], "frac_burst": ach / pk["bf16_tflops"],
                 "traffic": None, "peak_source": pk["source"] + " (bf16 cuBLAS: sustained for `frac` -- kernel timed under load after a "
                 f"{args.preheat:.0f} s pre-heat --, burst for `frac_burst`)", "algorithmic_flops_per_launch": flops}
            if extra:
                d.update(extra)
            return d
        def hbm(nbytes):
            ach = nbytes / (dom_ms * 1e-3) / 1e9
            return {"bound": "hbm", "kernel": name, "ms": dom_ms, "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / pk["hbm_gbs"], "traffic": None, "peak_source": pk["source"], "algorithmic_bytes_per_launch": nbytes}
        if name.startswith("conv"):
            if name.startswith("conv01"):                     # both conv blocks in one kernel
                roof = tensor((fl["conv0"] + fl["conv1"]) * B)
                if "conv1_igemm_tcgen05" in prof2:
                    t1, t0 = prof2["conv1_igemm_tcgen05"], prof2.get("conv0_first_tcgen05", 0.0)
                    a1 = fl["conv1"] * B / (t1 * 1e-3) / 1e12
                    roof["two_kernel_variant"] = {"conv1_igemm_ms": t1, "conv0_first_ms": t0, "conv1_achieved_tflops": a1,
                                                  "conv1_frac": a1 / pk["bf16_tflops_sustained"], "conv1_frac_burst": a1 / pk["bf16_tflops"],
                                                  "both_frac": (fl["conv0"] + fl["conv1"]) * B / ((t0 + t1) * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
                                                  "measured": "same run, BCAD_TWO_CONV_KERNELS=1, CUDA events"}
                roof["note"] = ("both conv blocks in ONE kernel (conv_fused2_kernel, sm100_fused2.cu: patch-union first block on tcgen05, tensor-map TMA input "
                                "boxes; BCAD_FUSED_V1=1 = the first generation): algorithmic FLOPs of block 1 (9 taps) + block 2 over the kernel's time; "
                                "`two_kernel_variant` has the stand-alone kernels of the same run")
            else:
                li = 0 if "conv0" in name else 1
                roof = tensor(fl[f"conv{li}"] * B)
                if prec == "fp16x3":
                    roof["note"] = ("split-operand mode: every product is 3 tensor-core MMAs (x_hi w_hi + x_lo w_hi + x_hi w_lo); `achieved` counts "
                                    "the ALGORITHMIC FLOPs once, so the tensor pipe does 3x that")
        elif "sgemm" in name or "fc" in name:
            roof = tensor(2.0 * (INPUT_SHAPE[0] // 4) * (INPUT_SHAPE[1] // 4) * CONV_LAYERS[-1][0] * HIDDEN[0] * B)
        elif name == "input_to_c8":
            h, w, c = INPUT_SHAPE
            roof = hbm(float(h * w * (c * 4 + ((c + 15) // 16 * 16) * 2)) * B)      # fp32 NHWC read + fp16 C8-planar write
        else:
            roof = hbm(tail_bytes_per_image(2 if prec.startswith("fp16") else 4) * B)
        return roof

    def tail_roofline(prof, prec):
        # Grad-CAM tail roofline (always reported beside the dominant kernel).  `achieved` counts the bytes THIS path has to move
        # (read A once, write the fp32 map: alpha comes from the shortcut, dA never exists; the low-res cam stays in shared
        # memory); the dense definition of SURVEY 8d (read A, read dA, write the map) is quoted next to it.
        tail_ms = sum(ms for k, ms in prof.items() if k.split(":", 1)[1] in ("cam", "cam_c8", "upsample_norm", "alpha_from_pool_grad", "tail_fused"))
        esz = 2 if prec == "fp16" else 4          # fp16x3 stores A as hi+lo halves = 4 bytes per element
        hc, wc, kc = INPUT_SHAPE[0] // 2, INPUT_SHAPE[1] // 2, CONV_LAYERS[-1][0]
        fused = any(k.endswith("tail_fused") for k in prof)
        own_bytes = (kc * hc * wc * esz + (0 if fused else 2 * hc * wc * 4) + INPUT_SHAPE[0] * INPUT_SHAPE[1] * 4.0) * B
        dense_bytes = tail_bytes_per_image(esz) * B
        ach = own_bytes / max(1e-9, tail_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernels": "Grad-CAM tail (cam channel reduction + min-max/bilinear/min-max)", "ms": tail_ms,
                "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                "algorithmic_bytes_per_launch": own_bytes,
                "dense_definition": {"bytes_per_launch": dense_bytes,
                                     "equivalent_GBps": dense_bytes / max(1e-9, tail_ms * 1e-3) / 1e9,
                                     "note": "SURVEY 8d dense figure (read A, read dA, write fp32 map); this path derives alpha "
                                             "from dz1 and never materialises dA, so it moves fewer bytes than that"}}

    roof = roofline_of(prof, prof2, precision)
    tail_roof = tail_roofline(prof, precision)
    for tfile in ("r02_traffic.json", "r01d_traffic.json"):
        traffic_file = os.path.join(ROOT, "profiles", tfile)
        if roof is not None and os.path.exists(traffic_file) and B == 512 and INPUT_SHAPE == (256, 256, 1) and precision == "fp16":
            tr = json.load(open(traffic_file))
            ncu_name = {"conv1_igemm_tcgen05": "conv_igemm_kernel<32, 64, 0>", "conv01_fused_tcgen05": "conv_fused_kernel<1>",
                        "conv0_first_tcgen05": "conv_first_tc_kernel<32, 0, 0>"}.get(roof["kernel"])
            if roof["kernel"] == "conv01_fused_tcgen05" and os.environ.get("BCAD_FUSED_V1") is None:
                ncu_name = next((k for k in tr if "conv_fused2_kernel" in k), ncu_name)      # the second-generation kernel (sm100_fused2.cu)
            if ncu_name in tr:
                roof["traffic"] = tr[ncu_name]
                roof["traffic_source"] = (f"profiles/{tfile} [{ncu_name}] (ncu --set full, dram__bytes_read.sum + "
                                          "dram__bytes_write.sum, per launch)")
                break

    cpu = None
    if not args.no_cpu_baseline:
        rate, secs, cores = cpu_reference_rate(args.cpu_images)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{args.cpu_images} of the workload's synthetic {'x'.join(map(str, INPUT_SHAPE))} images in batches of 32 "
                         f"({secs:.1f} s), oracle port of ADCNNM + autograd Grad-CAM + NumPy tail"}
    scaling = "strong" if args.total_batch else "weak"
    dtype_of = {"fp16": "f16", "fp16x3": "f16x3 (hi+lo split, fp32-grade)"}
    out_json = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": dtype_of.get(precision, "f32"), "data": "synthetic",
        "config": workload_config(B, precision, args.total_batch, eng.refine_margin),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(x_host.numel() * 4),
                "d2h_bytes_per_step": int(heat_host.numel() * 4 + B * (2 * NUM_CLASSES * 4 + 4)),
                "ms_per_step": e2e_ms / args.steps, "api": "bcad_predict_explain_host (pinned host buffers)",
                "host_ceiling_gbs": ceiling_gbs, "host_ceiling_ms_per_step": ceiling_ms,
                "achieved_gbs": world * (x_host.numel() + heat_host.numel()) * 4 / (e2e_ms / args.steps * 1e-3) / 1e9,
                "host_ceiling_note": "all ranks copying the step's bytes both ways at once with no compute (same pinned buffers): what the "
                                     "host side of this box can move; the e2e leg is bound by it when achieved_gbs is close"},
        "e2e_api": api,
        "e2e_u8_heatmaps": {"value": world * B * args.steps / (e2e_u8_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_u8_ms / args.steps,
                            "d2h_bytes_per_step": int(heat8_host.numel() + B * (2 * NUM_CLASSES * 4 + 4)),
                            "api": "bcad_predict_explain_host_u8: same call, heat-maps as heatmap_uint8 (GRADCAM.py:70) -- informational, "
                                   "the headline e2e above returns float32 maps"},
        "e2e_u8_in_out": {"value": world * B * args.steps / (e2e_u8io_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_u8io_ms / args.steps,
                          "h2d_bytes_per_step": int(x8_host.numel()),
                          "d2h_bytes_per_step": int(heat8_host.numel() + B * (2 * NUM_CLASSES * 4 + 4)),
                          "api": "bcad_predict_explain_host_u8in: 8-bit pixels in (x = u8 / 255 on the device, app.py:71), heatmap_uint8 "
                                 "out -- what the reference's callers hold and write; informational"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "preheat": {"seconds": args.preheat, "steps": main["preheat_steps"],
                    "note": "untimed full-duty steps right before the timed region: the timed steps sample the sustained state"},
        "roofline": roof,
        "roofline_tail": tail_roof,
        "kernels": kernel_table(prof),
        "cpu_baseline": cpu,
        "check": check,
        "tensor_path": bool(eng.uses_tensor_path),
    }
    if grade is not None:
        g_ms = grade["ms_total"] / args.steps
        out_json["fp32_grade"] = {
            "what": "the SAME workload on the split-operand tensor path (precision fp16x3: fp32-grade logits / heat-maps; the default of the "
                    "drop-in mirrors ADCNNM.CNNModel / CNNModel), measured in the same run",
            "value": world * B * args.steps / (grade["ms_total"] * 1e-3), "unit": UNIT, "ms_per_step": g_ms,
            "e2e": {"value": world * B * args.steps / (grade["e2e_ms"] * 1e-3), "unit": UNIT, "ms_per_step": grade["e2e_ms"] / args.steps,
                    "api": "bcad_predict_explain_host (pinned host buffers, float32 in / float32 maps out)"},
            "e2e_u8_in_out": {"value": world * B * args.steps / (grade["e2e_u8io_ms"] * 1e-3), "unit": UNIT,
                              "ms_per_step": grade["e2e_u8io_ms"] / args.steps},
            "gpu_launches": int(grade["launches"]), "clocks": grade["clocks"],
            "roofline": roofline_of(grade["prof"], {}, "fp16x3"), "roofline_tail": tail_roofline(grade["prof"], "fp16x3"),
            "kernels": kernel_table(grade["prof"]), "check": check3}
    if args.dump_outputs:
        write_dump(args.dump_outputs, main["dump"])
    emit(out_json)


def run_sharded(args):
    """Secondary line: the in-process batch-sharded driver (bcad_b200.ShardedEngine: one handle + one host thread per GPU, no
    torchrun, no collective) -- end-to-end images/s from ONE pinned host batch to pinned host heat-maps over --gpus GPUs."""
    import torch
    import bcad_b200
    n = min(args.gpus, torch.cuda.device_count())
    B = args.total_batch if args.total_batch else args.batch * n
    spec = bcad_b200.NetSpec.torch_flavour(INPUT_SHAPE, NUM_CLASSES, CONV_LAYERS, HIDDEN, 0.01)
    prec = "fp16" if args.precision == "auto" else args.precision
    sh = bcad_b200.ShardedEngine(spec, list(range(n)), precision=prec, max_batch=min(512, max(1, B // n)))
    sh.set_weights(*synth_weights())
    out = {}
    for name, dt in (("float32", np.float32), ("uint8", np.uint8)):
        if dt == np.uint8:
            x = torch.from_numpy(np.clip(np.rint(synth_images(B, INPUT_SHAPE, seed=5) * 255.0), 0, 255).astype(np.uint8)).pin_memory().numpy()
        else:
            x = torch.from_numpy(synth_images(B, INPUT_SHAPE, seed=5)).pin_memory().numpy()
        for _ in range(3):
            sh.predict_explain_host(x, None, "logit", heat_dtype=dt)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            sh.predict_explain_host(x, None, "logit", heat_dtype=dt)
        dt_s = time.perf_counter() - t0
        out[name] = {"value": B * args.steps / dt_s, "unit": UNIT, "ms_per_step": dt_s / args.steps * 1e3}
    emit({"metric": METRIC + " (in-process ShardedEngine, end to end)", "value": out["float32"]["value"], "unit": UNIT, "n_gpus": n,
          "steps": args.steps, "warmup": 3, "ms_per_step": out["float32"]["ms_per_step"], "higher_is_better": True,
          "scaling": "strong" if args.total_batch else "weak", "vs_baseline": None, "dtype": "f16" if prec == "fp16" else prec, "data": "synthetic",
          "config": {"workload": f"ShardedEngine.predict_explain_host: {B} images per step split over {n} GPUs by one process "
                                 f"(one handle + one host thread per GPU), pinned host buffers both ways", "images_per_step": B},
          "e2e": dict(out["float32"], h2d_bytes_per_step=B * INPUT_SHAPE[0] * INPUT_SHAPE[1] * INPUT_SHAPE[2] * 4,
                      d2h_bytes_per_step=B * INPUT_SHAPE[0] * INPUT_SHAPE[1] * 4),
          "e2e_u8_in_out": out["uint8"]})
    sh.close()


def run_pipeline(args, rank, world, local_rank):
    """Secondary line, BASELINE config 3: FULL pipeline at batch 256 per GPU -- 8-bit grey image -> per-image standardisation ->
    tiny U-Net encoder (Classes/unet.py:61-73: the "ROI" front) -> average_pool(3) (Classes/ImageSegmentation.py:182) -> CNN classify on
    the (22,22,64) features -> Grad-CAM (last conv block) scaled to the 256x256 image (GRADCAM.py:46-64) -> show_cam_on_image
    overlay + heatmap_uint8 (GRADCAM.py:67,70).  U-Net conv2/conv3 and the CNN's convs / fc1 on tcgen05 (fp16 operands)."""
    import torch
    import torch.distributed as dist
    import bcad_b200
    from bcad_b200 import unet as U
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch if args.batch != 512 else 256
    H, W = INPUT_SHAPE[0], INPUT_SHAPE[1]
    rng = np.random.default_rng(11)
    # the reference draws randn(std 1) kernels inside tiny_unet_numpy; scaled here so the features stay O(1) for the random-init CNN
    ks = [rng.standard_normal(shp) * sc for shp, sc in (((3, 3, 1, 16), 0.3), ((3, 3, 16, 32), 0.08), ((3, 3, 32, 64), 0.06))]
    front = U.UnetFront(H, W, ks, max_batch=B, device=local_rank)
    fh, fw, fc = front.out_shape(3)
    cnn_shape = (fh, fw, fc)
    spec = bcad_b200.NetSpec.torch_flavour(cnn_shape, NUM_CLASSES, CONV_LAYERS, HIDDEN, 0.01)
    eng = bcad_b200.Engine(spec, precision="fp16" if args.precision == "auto" else args.precision, max_batch=B, device=local_rank)
    cw, cb, dw, db = synth_weights_for(cnn_shape)
    eng.set_weights(cw, cb, dw, db)
    g8_host = torch.from_numpy(np.clip(synth_images(B, (H, W, 1), seed=31 + rank)[..., 0] * 48 + 128, 0, 255).astype(np.uint8)).pin_memory()
    ov_host = torch.empty((B, H, W, 3), dtype=torch.uint8).pin_memory()
    hu_host = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
    g8_dev = g8_host.to(dev)
    heat = torch.empty((B, H, W), device=dev, dtype=torch.float32)
    feat = torch.empty((B, fh, fw, fc), device=dev, dtype=torch.float32)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_dev(g8):
        img01, x = bcad_b200.gray_preprocess(g8, 1, True)
        front.forward(x, 3, out=feat)
        cls, probs, logits, _ = eng.predict_explain(feat, None, "logit", out_heat=heat, out_hw=(H, W))
        ov, hu = bcad_b200.overlay(img01, heat)
        return cls, logits, ov, hu

    def step_e2e():
        cls, logits, ov, hu = step_dev(g8_host.to(dev, non_blocking=True))
        ov_host.copy_(ov, non_blocking=True)
        hu_host.copy_(hu, non_blocking=True)
        return cls.cpu()

    for _ in range(max(3, args.warmup)):
        step_dev(g8_dev)
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < args.preheat:
        for _ in range(10):
            step_dev(g8_dev)
        torch.cuda.synchronize(dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start_under_load(lambda: step_dev(g8_dev), lambda: torch.cuda.synchronize(dev))
    for _ in range(10):
        step_dev(g8_dev)
    l0 = eng.launch_count + front.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out = step_dev(g8_dev)
    ev1.record()
    barrier()
    launches = eng.launch_count + front.launch_count - l0 + 2 * args.steps          # + gray_preprocess and overlay per step
    ms_total = ev0.elapsed_time(ev1)
    for _ in range(3):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize(dev)
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    tt = torch.tensor([ms_total, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms = float(tt[0]), float(tt[1])
    # per-kernel times under load: the two handles' own marks, torch events around the two stand-alone stages
    front.set_profiling(True)
    eng.set_profiling(True)
    prof = {}
    nprof = 3
    for _ in range(nprof):
        for _ in range(5):
            step_dev(g8_dev)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        img01, x = bcad_b200.gray_preprocess(g8_dev, 1, True)
        e[1].record()
        front.forward(x, 3, out=feat)
        eng.predict_explain(feat, None, "logit", out_heat=heat, out_hw=(H, W))
        e[2].record()
        bcad_b200.overlay(img01, heat)
        e[3].record()
        torch.cuda.synchronize(dev)
        items = [("gray_preprocess", e[0].elapsed_time(e[1]))] + front.last_profile() + [("cnn_" + n, ms) for n, ms in eng.last_profile()] + \
                [("overlay", e[2].elapsed_time(e[3]))]
        for i, (name, ms) in enumerate(items):
            key = f"{i:02d}:{name}"
            prof[key] = prof.get(key, 0.0) + ms / nprof
    front.set_profiling(False)
    eng.set_profiling(False)
    if rank != 0:
        return
    pk = peaks()
    # algorithmic work of the front per image (true conv areas; quirk rows are zeros, not work)
    H1, W1, H2, W2 = H // 2, W // 2, H // 4 + 1, W // 4 + 1
    flops = {"unet_conv2_igemm_tcgen05": 2.0 * H1 * W1 * 32 * 9 * 16, "unet_conv3_igemm_tcgen05": 2.0 * H2 * W2 * 64 * 9 * 32,
             "cnn_conv0_wide_tcgen05": 2.0 * fh * fw * 32 * 9 * fc, "cnn_conv1_igemm_tcgen05": 2.0 * (fh // 2) * (fw // 2) * 64 * 9 * 32}
    nbytes = {"gray_preprocess": H * W * (1 + 4 + 4.0), "unet_conv1_first_pool": H * W * 4 + H1 * W1 * 16 * 2.0,
              "unet_out_avgpool": H2 * W2 * 64 * 2 + fh * fw * fc * 4.0, "overlay": H * W * (4 + 4 + 3 + 1.0),
              "cnn_upsample_norm": (fh // 2) * (fw // 2) * 4 + H * W * 4.0, "cnn_tail_fused": (fh // 2) * (fw // 2) * 64 * 2 + H * W * 4.0}
    dom_key = max(prof, key=prof.get)
    dom = dom_key.split(":", 1)[1]
    dom_ms = prof[dom_key]
    if dom in flops:
        ach = flops[dom] * B / (dom_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": dom, "ms": dom_ms, "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["bf16_tflops_sustained"], "frac_burst": ach / pk["bf16_tflops"], "traffic": None,
                "algorithmic_flops_per_launch": flops[dom] * B, "peak_source": pk["source"]}
    else:
        nb = nbytes.get(dom, 0.0) * B
        ach = nb / (dom_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "kernel": dom, "ms": dom_ms, "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                "traffic": None, "algorithmic_bytes_per_launch": nb, "peak_source": pk["source"]}
    tot = max(1e-9, sum(prof.values()))
    kernels = [{"kernel": k, "ms": round(v, 4), "share": round(v / tot, 4)} for k, v in sorted(prof.items())]
    for kr in kernels:
        n = kr["kernel"].split(":", 1)[1]
        if n in flops:
            kr["tflops"] = round(flops[n] * B / (kr["ms"] * 1e-3) / 1e12, 1)
        elif n in nbytes:
            kr["GBps"] = round(nbytes[n] * B / (kr["ms"] * 1e-3) / 1e9, 1)
    # untimed check of the first images against the float64 oracle of the whole pipeline
    check = None
    if not args.no_check:
        from oracle import cnn as ocnn, gradcam as ogc, unet as ou
        k = min(B, 16)
        g8 = g8_host[:k].numpy()
        img01 = (g8 / 255.0).astype(np.float32)
        xs = np.stack([((im - im.mean()) / (im.std() + 1e-8)).astype(np.float32) for im in img01])[..., None]
        f64 = ou.average_pool(ou.tiny_unet(xs.astype(np.float64), ks), 3)
        cfg = ocnn.NetConfig.torch_flavour(cnn_shape, NUM_CLASSES, CONV_LAYERS, HIDDEN, 0.01)
        params = ocnn.Params(cw, cb, dw, db)
        cache = ocnn.forward(cfg, params, f64)
        o_cls = cache.logits.argmax(dim=-1).numpy()
        cag, _, _ = ocnn.backward(cfg, params, cache, ocnn.top_gradient(cache, o_cls, "logit"), through_input=False)
        o_heat = ogc.gradcam_tail_nhwc(cache.conv_out[-1].numpy().astype(np.float32), cag[1].numpy().astype(np.float32), (H, W))
        cls, logits, ov, hu = out
        d_feat = feat[:k].cpu().numpy()
        lg = cache.logits.numpy()
        want_hu = np.stack([ogc.heatmap_u8(o_heat[i]) for i in range(k)]).astype(np.int32)
        want_ov = np.stack([ogc.show_cam_on_image(np.stack([img01[i]] * 3, -1), o_heat[i]) for i in range(k)]).astype(np.int32)
        margin = np.abs(lg[:, 0] - lg[:, 1])
        check = {"images": k, "vs": "float64 oracle of the whole pipeline (oracle/unet.py + oracle/cnn.py + oracle/gradcam.py)",
                 "feature_rel_err": float(np.abs(d_feat - f64).max() / max(1.0, np.abs(f64).max())),
                 "class_mismatches": int((cls[:k].cpu().numpy() != o_cls).sum()), "smallest_logit_margin": float(margin.min()),
                 "max_logit_err": float(np.abs(logits[:k].cpu().numpy() - lg).max()), "logit_scale": float(np.abs(lg).max()),
                 "heatmap_u8_max_abs_diff": int(np.abs(hu[:k].cpu().numpy().astype(np.int32) - want_hu).max()),
                 "overlay_u8_frac_pixels_off_by_more_than_1": float((np.abs(ov[:k].cpu().numpy().astype(np.int32) - want_ov) > 1).mean())}
    emit({"metric": "full pipeline (U-Net front -> CNN classify -> Grad-CAM overlay) images/sec at 256x256", "value": world * B * args.steps / (ms_total * 1e-3),
          "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps,
          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
          "config": {"workload": f"cfg3: uint8 grey {H}x{W} images -> standardise -> tiny U-Net encoder (1->16->32->64, ReLU, pools; conv2d 'same' "
                                 f"quirk kept) -> average_pool(3) -> ADCNNM-flavour CNN on ({fh},{fw},{fc}) (conv 32,64 k3 pad1; fc 256,128; random "
                                 f"init) -> Grad-CAM(last conv, predicted class) scaled to {H}x{W} -> JET overlay + heatmap_uint8; batch {B} per GPU",
                     "batch_per_gpu": B, "l2_policy": "image batch + intermediate maps per step (> 300 MB) exceed the 126 MB L2"},
          "e2e": {"value": world * B * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / args.steps,
                  "h2d_bytes_per_step": int(g8_host.numel()), "d2h_bytes_per_step": int(ov_host.numel() + hu_host.numel() + B * 4),
                  "api": "uint8 images in pinned host memory -> bcad_gray_preprocess, bcad_unet_forward, bcad_predict_explain_sized, bcad_overlay -> "
                         "uint8 overlays + heat-maps in pinned host memory + classes"},
          "gpu_launches": int(launches), "clocks": clocks, "preheat": {"seconds": args.preheat}, "roofline": roof, "kernels": kernels, "check": check})
    front.close()
    eng.close()


def synth_weights_for(shape):
    """synth_weights() for another input shape (the pipeline's CNN sees the U-Net features)."""
    global INPUT_SHAPE
    keep = INPUT_SHAPE
    INPUT_SHAPE = tuple(shape)
    try:
        return synth_weights()
    finally:
        INPUT_SHAPE = keep


def run_train(args, rank, world, local_rank):
    """Secondary line (SURVEY 8 row f4 / BASELINE config 5): data-parallel training step, images/s.  fp32 forward +
    backward + weight gradients in libbcad, ONE bucketed NCCL all-reduce of the flat gradient, Adam on the device."""
    import torch
    import torch.distributed as dist
    import bcad_b200
    from bcad_b200.training import DataParallelTrainer

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.train_batch
    spec = bcad_b200.NetSpec.torch_flavour(INPUT_SHAPE, NUM_CLASSES, CONV_LAYERS, HIDDEN, 0.01)
    eng = bcad_b200.Engine(spec, precision="fp32", max_batch=B, keep_all_activations=True, device=local_rank)
    eng.set_weights(*synth_weights())
    if args.train_kernels == "tensor":
        eng.set_fast_training(True)          # second conv block: forward / dgrad / wgrad as split-operand tcgen05 GEMMs (sm100_train.cu)
    tr = DataParallelTrainer(eng, opt="adam", lr=1e-4)
    x_host = torch.from_numpy(synth_images(B, INPUT_SHAPE, seed=777 + rank)).pin_memory()
    y_host = torch.from_numpy((np.arange(B) % 2).astype(np.int32)).pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        tr.step(x_dev, y_dev)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        t0 = time.perf_counter()
        while sampler.proc is not None and not sampler.lines and time.perf_counter() - t0 < 3.0:
            time.sleep(0.02)              # nvidia-smi start-up stalls launches: let it pass before the timed region (the steps hold a collective)
    barrier()
    for _ in range(3):
        tr.step(x_dev, y_dev)
    l0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        loss = tr.step(x_dev, y_dev)
    ev1.record()
    barrier()
    launches = eng.launch_count - l0
    ms_total = ev0.elapsed_time(ev1)
    # what the overlap buys: the same steps with the all-reduce AFTER the whole backward, and the all-reduce of the flat gradient alone
    ms_serial, ar_ms = None, None
    if world > 1:
        tr.overlap = False
        for _ in range(2):
            tr.step(x_dev, y_dev)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            tr.step(x_dev, y_dev)
        e1.record()
        barrier()
        ms_serial = e0.elapsed_time(e1) / args.steps
        tr.overlap = True
        gbuf = torch.zeros((eng.grad_elems(),), device=dev, dtype=torch.float32)
        for _ in range(2):
            dist.all_reduce(gbuf)
        barrier()
        e0.record()
        for _ in range(10):
            dist.all_reduce(gbuf)
        e1.record()
        barrier()
        ar_ms = e0.elapsed_time(e1) / 10
        t2 = torch.tensor([ms_serial, ar_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ms_serial, ar_ms = float(t2[0]), float(t2[1])
    # end to end: inputs and labels from pinned host memory, the step's mean loss read back (2 untimed steps first: torch
    # loads its reduction kernel lazily)
    def step_e2e():
        loss = tr.step(x_host.to(dev, non_blocking=True), y_host.to(dev, non_blocking=True))
        return float(loss.mean())
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        mean_loss = step_e2e()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    tt = torch.tensor([ms_total, e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms = float(tt[0]), float(tt[1])
    eng.set_profiling(True)
    prof = {}
    eng.predict(x_dev)
    torch.cuda.synchronize(dev)
    for i, (name, ms) in enumerate(eng.last_profile()):
        prof[f"fwd{i:02d}:{name}"] = ms
    g, _ = eng.train_backward(x_dev, y_dev)
    torch.cuda.synchronize(dev)
    for i, (name, ms) in enumerate(eng.last_profile()):
        prof[f"bwd{i:02d}:{name}"] = ms
    eng.apply_update(g, "adam", lr=0.0)
    torch.cuda.synchronize(dev)
    for i, (name, ms) in enumerate(eng.last_profile()):
        prof[f"upd{i:02d}:{name}"] = prof.get(f"upd{i:02d}:{name}", 0.0) + ms
    eng.set_profiling(False)
    if rank != 0:
        return
    tot = max(1e-9, sum(prof.values()))
    kernels = [{"kernel": k, "ms": round(v, 4), "share": round(v / tot, 4)} for k, v in sorted(prof.items()) if v / tot >= 0.005]
    grad_bytes = eng.grad_elems() * 4
    emit({
        "metric": "training throughput (forward + backward + gradient all-reduce + Adam), images/s", "value": world * B * args.steps / (ms_total * 1e-3),
        "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (second conv block: split-operand tcgen05, fp32 in/out)" if args.train_kernels == "tensor" else "f32", "data": "synthetic",
        "config": {"workload": f"train: ADCNNM-flavour CNN {INPUT_SHAPE} conv{CONV_LAYERS} fc{HIDDEN}, {B} images/GPU/step, Adam, "
                               f"one {grad_bytes / 1e6:.0f} MB gradient all-reduce per step (secondary line, BASELINE config 5)",
                   "images_per_gpu": B, "l2": "activations >> 126 MB L2 per step", "train_kernels": args.train_kernels},
        "e2e": {"value": world * B * args.steps / (e2e_ms * 1e-3), "unit": "images/s", "h2d_bytes_per_step": int(x_host.numel() * 4 + B * 4),
                "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps, "last_mean_loss": mean_loss},
        "gpu_launches": int(launches), "clocks": clocks, "kernels": kernels, "grad_bytes": grad_bytes,
        "comm": None if world == 1 else {
            "allreduce_alone_ms": ar_ms, "allreduce_busbw_GBps": grad_bytes * 2 * (world - 1) / world / (ar_ms * 1e-3) / 1e9,
            "ms_per_step_overlapped": ms_total / args.steps, "ms_per_step_allreduce_after_backward": ms_serial,
            "allreduce_share_of_step_if_serial": ar_ms / ms_serial,
            "note": "overlapped = the dense (fc1) bucket is all-reduced while the conv blocks' backward runs (bcad_train_backward_part)"},
    })


_JSON_FD = None


def claim_stdout():
    """Rank 0 must print exactly ONE JSON line: route everything else that lands on fd 1 (NCCL's version banner,
    library chatter) to stderr and keep a private handle for the result line."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="images per GPU per step")
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "fp16", "fp16x3"])
    ap.add_argument("--cpu-images", type=int, default=1024, help="bounded CPU-baseline sample (~10 s of CPU work on 16 cores)")
    ap.add_argument("--ref-images", type=int, default=64, help="images per step of the --impl reference arm")
    ap.add_argument("--workload", default="explain", choices=["explain", "train", "sharded", "pipeline"],
                    help="explain = the headline path (predict + Grad-CAM); train = the secondary training-step line")
    ap.add_argument("--train-batch", type=int, default=64, help="images per GPU per training step")
    ap.add_argument("--flavour", default="torch", choices=["torch", "numpy"],
                    help="numpy = SECONDARY line on the reference's NumPy CNN (tie-duplicating pool): fp16x3 tensor path + fp32 tail")
    ap.add_argument("--input-shape", default=None, help="H,W,C of a SECONDARY shape (SURVEY 8d: 256,256,64 or 64,256,256); "
                                                        "the headline line uses the default 256,256,1")
    ap.add_argument("--total-batch", type=int, default=0, help="STRONG scaling (BASELINE cfg 4: 8192): images per step over ALL GPUs, "
                                                               "split evenly; 0 = weak scaling with --batch images per GPU")
    ap.add_argument("--train-kernels", default="tensor", choices=["tensor", "fp32"], help="--workload train: the second conv block on the tensor "
                                                                                         "cores (bcad_set_fast_training) or every kernel fp32")
    ap.add_argument("--preheat", type=float, default=2.0, help="seconds of untimed full-duty steps before each timed region")
    ap.add_argument("--check-images", type=int, default=256, help="images of the batch compared one by one with the oracle (untimed)")
    ap.add_argument("--refine-margin", type=float, default=None, help="fp16 path: top-2 logit gap below which an image is re-run at fp32 "
                                                                    "grade (default: the engine's; 0 switches the refinement off)")
    ap.add_argument("--only-value", action="store_true", help="device-resident leg only (for runs under ncu)")
    ap.add_argument("--no-api", action="store_true", help="skip the e2e_api leg (the mirrors' Python surface)")
    ap.add_argument("--no-fp32-grade", action="store_true", help="skip the second measurement of the workload in fp16x3 mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the (untimed) oracle check of the first images")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what rank 0's last timed step returned as DIR/<name>.npy (float32): classes, probs, logits and the "
                         "heat-maps of every image, or of a fixed seeded sample of them when all would exceed 32 MB; "
                         "explain workload of --impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "explain"):
        ap.error("--dump-outputs writes the outputs of the explain workload of --impl ours")
    global FLAVOUR
    FLAVOUR = args.flavour
    if args.input_shape:
        global INPUT_SHAPE
        INPUT_SHAPE = tuple(int(v) for v in args.input_shape.split(","))
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.workload == "sharded":
        if rank == 0:
            run_sharded(args)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import torch
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    elif args.gpus > 1:
        log(f"[bench] --gpus {args.gpus} without torchrun: launch with torch.distributed.run; running 1 rank")
    try:
        {"train": run_train, "pipeline": run_pipeline}.get(args.workload, run_ours)(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
