"""Drop-in for ``WebApplicationPrototype/GRADCAM.py``.

The reference runs third-party ``pytorch_grad_cam.GradCAM`` on an ImageNet ResNet50 (GRADCAM.py:16,52-53) --
not on its own CNN.  Here the same call surface drives Grad-CAM on the project's CNN (last conv block,
post-LeakyReLU output, ``ClassifierOutputTarget`` = gradient of the raw class logit), computed by libbcad:
forward + backward-to-target + tail (alpha GAP, weighted sum, ReLU, min-max, cv2-bilinear upsample, min-max)
+ ``show_cam_on_image`` / ``heatmap_uint8`` (GRADCAM.py:64-70), all on the GPU.

Set the model once (``GRADCAM.model = my_cnn``) or pass ``model=``; no network download happens at import.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import engine as _engine

model = None          # module-level model, as in the reference (GRADCAM.py:16)


def default_preprocess(img01: np.ndarray, input_shape) -> np.ndarray:
    """(H,W) in [0,1] -> model input (H,W,C): per-image standardisation as the reference does for its CNN
    inputs (app.py:179-182), the single channel replicated to C."""
    x = img01.astype(np.float32)
    x = (x - x.mean()) / (x.std() + 1e-8)
    return np.repeat(x[..., None], input_shape[2], axis=-1)


def generate_dual_class_gradcam_overlays_pytorch(img, classes_to_test=[0, 1], save_folder="explainability",
                                                 model=None, preprocess=default_preprocess, write_png=True):
    """GRADCAM.py:31-81 -> ``{class_idx: (overlay_rgb_u8 (H,W,3), heatmap_u8 (H,W))}`` and the four PNGs.

    ``img``: grayscale (H,W) scaled 0-255, of ANY size: like pytorch_grad_cam, the heat-map is the low-resolution cam scaled to
    the size of ``img`` (the reference hands a 512x512 image over whatever its CNN was fed, app.py:649-657); when ``img`` is not
    the model's input size the CNN sees ``cv2.resize(img / 255, model size)``.  ``classes_to_test=None`` uses the predicted
    class (:60-61)."""
    mdl = model if model is not None else globals()["model"]
    if mdl is None:
        raise RuntimeError("GRADCAM.model is not set: assign a CNNModel (bcad_b200.CNNModel / ADCNNM) first")
    eng = getattr(mdl, "fast_engine", None) or mdl.engine     # NumPy mirror: the batched (tensor-core) handle
    os.makedirs(save_folder, exist_ok=True)
    overlays = {}
    img = np.asarray(img)
    if img.ndim != 2:
        raise ValueError(f"img must be a grayscale (H,W) array, got shape {img.shape}")
    H, W, _ = eng.spec.input_shape
    img01 = (img / 255.0).astype(np.float32)                       # GRADCAM.py:46
    net01 = img01
    if img.shape != (H, W):
        import cv2
        net01 = cv2.resize(img01, (W, H), interpolation=cv2.INTER_LINEAR)
    x = preprocess(net01, eng.spec.input_shape)
    if classes_to_test is None:
        cls, _, _ = eng.predict(x[None])
        classes_to_test = [int(cls[0])]                            # GRADCAM.py:56-61
    n = len(classes_to_test)
    xb = np.repeat(x[None], n, axis=0)
    _, _, _, heat = eng.predict_explain(xb, np.asarray(classes_to_test, dtype=np.int32), "logit",
                                        out_hw=None if img.shape == (H, W) else img.shape)               # :64
    img_dev = torch.from_numpy(img01).to(heat.device)[None].expand(n, *img.shape)
    ov, hu = _engine.overlay(img_dev, heat)                        # :67, :70
    ov, hu = ov.cpu().numpy(), hu.cpu().numpy()
    for i, class_idx in enumerate(classes_to_test):
        if write_png:
            import cv2
            cv2.imwrite(os.path.join(save_folder, f"gradcam_overlay_class_{class_idx}.png"),
                        cv2.cvtColor(ov[i], cv2.COLOR_RGB2BGR))    # :73-76
            cv2.imwrite(os.path.join(save_folder, f"gradcam_heatmap_class_{class_idx}.png"), hu[i])
        overlays[class_idx] = (ov[i], hu[i])
        print(f"Saved Grad-CAM overlay and heatmap for class {class_idx} in {save_folder}")
    return overlays


def generate_gradcam_overlays_batch(imgs_u8, class_idx=None, model=None, standardise=True, overlay_out=None, heat_out=None):
    """The same outputs for a BATCH of 8-bit grey images [B,H,W] at the model's input size, through ONE host-buffer C-ABI call
    (``bcad_gradcam_overlays_host``: uint8 in, uint8 RGB overlays + ``heatmap_uint8`` out; normalisation, CNN, Grad-CAM, JET
    overlay all on the device).  ``class_idx``: None = each image's predicted class (GRADCAM.py:60-61), an int, or one per image.
    -> (classes int64 [B], probs [B,nc], overlays uint8 [B,H,W,3], heatmaps uint8 [B,H,W])."""
    mdl = model if model is not None else globals()["model"]
    if mdl is None:
        raise RuntimeError("GRADCAM.model is not set: assign a CNNModel (bcad_b200.CNNModel / ADCNNM) first")
    eng = getattr(mdl, "fast_engine", None) or mdl.engine
    cls, probs, _, ov, hu = eng.gradcam_overlays_host(imgs_u8, class_idx, "logit", standardise, overlay_out, heat_out)
    return cls.astype(np.int64), probs, ov, hu


def generate_dual_class_gradcam_overlays_batch(imgs_u8, classes_to_test=[0, 1], model=None, standardise=True, overlay_out=None,
                                               heat_out=None):
    """The batched form of the deployed dual-class call (app.py:649-657 -> GRADCAM.py:31-81): 8-bit grey images [B,H,W] of any size
    (the CNN sees ``cv2.resize(img / 255, model size)``, the maps have the image's size, as in the single-image call above), ONE
    forward per image for all of ``classes_to_test`` (K <= 8), through ONE host-buffer C-ABI call (bcad_gradcam_overlays_classes_host),
    no PNGs.  ``overlay_out`` / ``heat_out``: optional C-contiguous uint8 arrays to write into (pinned ones make the copies asynchronous).
    -> (classes int64 [B], probs [B,nc], overlays uint8 [B,K,H,W,3], heatmaps uint8 [B,K,H,W]); at the model's input size ``[:, k]`` is
    byte for byte what ``generate_gradcam_overlays_batch(imgs_u8, class_idx=classes_to_test[k])`` returns."""
    mdl = model if model is not None else globals()["model"]
    if mdl is None:
        raise RuntimeError("GRADCAM.model is not set: assign a CNNModel (bcad_b200.CNNModel / ADCNNM) first")
    eng = getattr(mdl, "fast_engine", None) or mdl.engine
    g = np.asarray(imgs_u8)
    if g.dtype != np.uint8:
        raise ValueError("imgs_u8 must be uint8 (0-255 grey levels)")
    cls, probs, _, ov, hu = eng.gradcam_overlays_classes_host(g, list(classes_to_test), "logit", standardise, overlay_out, heat_out)
    return cls.astype(np.int64), probs, ov, hu
