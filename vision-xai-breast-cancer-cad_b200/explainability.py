"""Drop-in for ``WebApplicationPrototype/explainability.py`` (custom-CNN explainability).

``compute_backprops_for_explainability(model, y_true)`` returns ``(grads, d_input, conv_act_grads)`` like
the reference (explainability.py:13-68); the activation-gradient chain (dense W^T dz with the LeakyReLU'
mask, tie-duplicating un-pool, conv input gradients) runs in libbcad.  ``grads`` holds the weight gradients of
the same backward pass -- ``{'dW','db'}`` per dense / output layer (explainability.py:25,33), ``{'dF','db_conv'}``
per conv layer (:63), ``None`` for pool layers (:42) -- from ``bcad_train_backward`` (the cross-entropy gradient of one
sample with label c IS the reference's ``probs - y_true`` backward); ``want_weight_grads=False`` skips them, as
``generate_dual_class_overlays`` does (explainability.py:94 drops them).
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import engine as _engine


def _class_of(y_true, num_classes):
    y = np.asarray(y_true, dtype=np.float64).reshape(-1)
    if y.shape[0] != num_classes or not np.all((y == 0) | (y == 1)) or y.sum() != 1:
        raise ValueError("y_true must be a one-hot vector of length num_classes")
    return int(np.argmax(y))


def compute_backprops_for_explainability(model, y_true, want_weight_grads=True):
    """Differentiates the model's latest ``forward(x, ...)`` (the reference reads that forward's caches out of ``model.layers``);
    if something else has used the handle since, the forward is repeated first (never a silently different image)."""
    c = _class_of(y_true, model.num_classes)
    conv_idx = [i for i, l in enumerate(model.layers) if l["type"] == "conv"]
    masks = model._last_masks
    if masks is None:
        eng = model._cache_ready()
    else:
        # a training forward: its dropout multipliers stay set on the handle for the whole backward (the weight gradients see the
        # dropped activations, Classes/CNNModel.py:186-188), so the forward is replayed under them first
        if model._last_x is None:
            raise RuntimeError("no forward() has been run on this model yet")
        eng = model.engine
        eng.set_dropout_masks(masks, mask_backward=False)
    try:
        if masks is not None:
            eng.predict(model._last_x[None])
        outs, d_in = eng.explain_backward(1, c, "softmax_ce", want_conv=range(len(conv_idx)), want_input=True)
        conv_act_grads = {li: outs[bi][0].double().cpu().numpy() for bi, li in enumerate(conv_idx)}
        d_input = d_in[0].double().cpu().numpy()
        grads = [None] * len(model.layers)
        if want_weight_grads:
            flat, _ = eng.train_backward(model._last_x[None], [c])
            g = eng.unpack_grads(flat)
            dense_idx = [i for i, l in enumerate(model.layers) if l["type"] in ("dense", "output")]
            for bi, li in enumerate(conv_idx):
                grads[li] = {"dF": g["conv_w"][bi].astype(np.float64), "db_conv": g["conv_b"][bi].astype(np.float64)}
            for di, li in enumerate(dense_idx):
                grads[li] = {"dW": g["dense_w"][di].astype(np.float64), "db": g["dense_b"][di].astype(np.float64)}
    finally:
        if masks is not None:
            eng.set_dropout_masks(None)
            eng.cache_tag = None
    return grads, d_input, conv_act_grads


def saliency_map(d_input):
    """explainability.py:72-73: |d_input|.max(-1), min-max with 1e-8."""
    saliency = np.abs(d_input).max(axis=-1)
    return (saliency - saliency.min()) / (saliency.max() - saliency.min() + 1e-8)


def generate_saliency_overlay(img, d_input):
    """explainability.py:71-78 -> (overlay u8 BGR, heatmap u8 BGR)."""
    import cv2
    saliency = np.uint8(saliency_map(d_input) * 255)
    heatmap = cv2.applyColorMap(saliency, cv2.COLORMAP_JET)
    heatmap = cv2.resize(heatmap, (img.shape[1], img.shape[0]))
    overlay = cv2.addWeighted(img.astype(np.uint8), 0.5, heatmap, 0.5, 0)
    return overlay, heatmap


def generate_dual_class_overlays(model, img, classes_to_test=[0, 1], save_folder="explainability"):
    """explainability.py:81-108.  ``img``: (H,W,C) model input; the overlay needs a 3-channel uint8-like
    image (cv2.addWeighted), so 1-channel inputs are replicated to 3 channels for the blend only."""
    import cv2
    os.makedirs(save_folder, exist_ok=True)
    overlays = {}
    model.forward(img, training=False)          # once: only the top gradient differs per class
    for class_idx in classes_to_test:
        y_true = np.zeros(model.layers[-1]["biases"].shape, dtype=np.float32)
        y_true[class_idx] = 1.0
        grads, d_input, conv_act_grads = compute_backprops_for_explainability(model, y_true, want_weight_grads=False)
        vis = img if img.shape[-1] == 3 else np.repeat(img[..., :1], 3, axis=-1)
        overlay, heatmap = generate_saliency_overlay(vis, d_input)
        cv2.imwrite(os.path.join(save_folder, f"overlay_class_{class_idx}.png"), overlay)
        cv2.imwrite(os.path.join(save_folder, f"heatmap_class_{class_idx}.png"), heatmap)
        overlays[class_idx] = (overlay, heatmap)
        print(f"Saved overlay and heatmap for class {class_idx} in {save_folder}")
    return overlays


def generate_dual_class_overlays_batch(model, X, classes_to_test=[0, 1]):
    """``generate_dual_class_overlays`` for a batch, without the PNGs: one forward per chunk of images, one backward per class, the
    colouring on the GPU.  ``X``: (B,H,W,C) or (H,W,C) model inputs; the blend base is ``X.astype(np.uint8)`` with 1-channel (or
    other non-3-channel) inputs replicated from channel 0, as the single-image mirror builds ``vis``.  Runs on
    ``model.saliency_engine``.  -> (classes int64 [B], probs [B,nc], saliency float32 [B,K,H,W], overlays uint8 [B,K,H,W,3],
    heatmaps uint8 [B,K,H,W,3]); overlays and heat-maps are BGR, as cv2 returns them."""
    X = np.asarray(X)
    if X.ndim == 3:
        X = X[None]
    base = X.astype(np.uint8)
    if base.shape[-1] != 3:
        base = base[..., :1]
    eng = model.saliency_engine
    cls, probs, _, sal, _ = eng.predict_saliency_classes(X.astype(np.float32), list(classes_to_test), "softmax_ce")
    overlay, heat = _engine.saliency_overlay(torch.from_numpy(np.ascontiguousarray(base)), sal)
    return (cls.cpu().numpy().astype(np.int64), probs.cpu().numpy(), sal.cpu().numpy(), overlay.cpu().numpy(), heat.cpu().numpy())
