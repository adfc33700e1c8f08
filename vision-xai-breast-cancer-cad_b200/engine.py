"""Host-side engine over the libbcad handle: batched predict / predict+Grad-CAM, sharding.

PyTorch is used only to own device memory and streams; every computation happens inside
libbcad.so (hand-written sm_100a CUDA) through the C-ABI in include/bcad.h.
"""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib


@dataclass
class NetSpec:
    """Constructor arguments of the reference CNNs + the flavour switches (SURVEY section 0)."""
    input_shape: Tuple[int, int, int]
    num_classes: int
    conv_layers: Sequence[Tuple[int, int]]
    hidden_units: Sequence[int]
    alpha_conv: float = 0.01
    alpha_dense: float = 0.01
    pad: int = 0
    flatten: str = "hwc"
    pool_ties: str = "dup"
    head: str = "softmax"

    @staticmethod
    def numpy_flavour(input_shape, num_classes, conv_layers, hidden_units, leaky_alpha=0.01):
        """Classes/CNNModel.py:68 -- valid conv, HWC flatten, tie-duplicating pool, softmax head."""
        return NetSpec(tuple(input_shape), int(num_classes), [tuple(map(int, c)) for c in conv_layers],
                       [int(u) for u in hidden_units], float(leaky_alpha), float(leaky_alpha), 0, "hwc", "dup", "softmax")

    @staticmethod
    def torch_flavour(input_shape, num_classes, conv_layers, hidden_units, leaky_alpha=0.01):
        """ADCNNM.py:35-78 -- Conv2d(padding=1), F.leaky_relu default slope on convs, CHW flatten, logits."""
        return NetSpec(tuple(input_shape), int(num_classes), [tuple(map(int, c)) for c in conv_layers],
                       [int(u) for u in hidden_units], 0.01, float(leaky_alpha), 1, "chw", "first", "logits")

    def shapes(self):
        h, w, c = self.input_shape
        out = []
        for f, k in self.conv_layers:
            ch, cw = h + 2 * self.pad - k + 1, w + 2 * self.pad - k + 1
            out.append(((ch, cw, f), (ch // 2, cw // 2, f)))
            h, w, c = ch // 2, cw // 2, f
        return out, h * w * c


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        return C.c_void_p(t.data_ptr())
    if isinstance(t, np.ndarray):
        return C.c_void_p(t.ctypes.data)
    raise TypeError(type(t))


def _f32c(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a), dtype=np.float32)


def _stream_of(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _gray_batch(gray_u8) -> np.ndarray:
    """uint8 grey images [B,H,W] or [H,W] -> a C-contiguous uint8 [B,H,W] array."""
    g = np.ascontiguousarray(gray_u8)
    if g.dtype != np.uint8:
        raise ValueError("gray_u8 must be uint8 (0-255 grey levels)")
    if g.ndim == 2:
        g = g[None]
    if g.ndim != 3:
        raise ValueError(f"gray_u8 must be [B,H,W] or [H,W], got shape {g.shape}")
    return g


def _out_array(out, shape, dtype, name):
    a = out if out is not None else np.empty(shape, dtype)
    if a.dtype != dtype or a.shape != shape or not a.flags["C_CONTIGUOUS"]:
        raise ValueError(f"{name} must be a C-contiguous {np.dtype(dtype).name} array of shape {shape}")
    return a


def _host_class_idx(class_idx, B, nc):
    """class_idx of the single-class host calls (None, one class or one per image) -> C-contiguous int32 [B] array or None."""
    if class_idx is None:
        return None
    ci = np.ascontiguousarray(np.broadcast_to(np.asarray(class_idx, dtype=np.int32).reshape(-1), (B,)))
    if ci.min() < 0 or ci.max() >= nc:
        raise ValueError("class_idx out of range")
    return ci


def _host_class_rows(classes, B, nc):
    """classes of the host multi-class calls -> (K, C-contiguous int32 [B,K] array or None = column k is class k)."""
    if classes is None:
        K, ci = nc, None
    else:
        ci = np.asarray(classes, dtype=np.int32)
        if ci.ndim == 1:
            ci = np.broadcast_to(ci[None], (B, ci.shape[0]))
        if ci.ndim != 2 or ci.shape[0] != B:
            raise ValueError(f"classes must be a length-K sequence or a [{B},K] array, got shape {ci.shape}")
        K = ci.shape[1]
        if K >= 1 and (int(ci.min()) < 0 or int(ci.max()) >= nc):
            raise ValueError("classes out of range")
        ci = np.ascontiguousarray(ci)
    if not 1 <= K <= _lib.MAX_EXPLAIN_CLASSES:
        raise ValueError(f"{K} target classes per image; 1..{_lib.MAX_EXPLAIN_CLASSES} are supported")
    return K, ci


class Engine:
    """One libbcad handle on one GPU."""

    #: default of ``refine_margin`` on the fp16 path: ~3x the largest 16-bit logit-gap error seen on the canonical network
    #: (tools/kink_stats.py); about 1 % of random-init images fall below it
    DEFAULT_REFINE_MARGIN = 1e-2

    def __init__(self, spec: NetSpec, precision: str = "fp32", max_batch: int = 64,
                 keep_all_activations: bool = False, device: int = 0, refine_margin: Optional[float] = None,
                 refine_capacity: int = 0):
        """precision "fp16": ``refine_margin`` (None = DEFAULT_REFINE_MARGIN where the shape allows, 0 = off) re-runs images
        whose two largest logits are closer than the margin through the fp32-grade split-operand kernels inside the same call,
        so the predicted classes are the fp32-grade ones (include/bcad.h ``refine_margin``)."""
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("libbcad needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.spec = spec
        self.device = int(device)
        self.precision = precision
        self.max_batch = int(max_batch)
        self.keep_all_activations = bool(keep_all_activations)
        cfg = _lib.Config()
        cfg.in_h, cfg.in_w, cfg.in_c = spec.input_shape
        cfg.num_classes = spec.num_classes
        if len(spec.conv_layers) > _lib.MAX_CONV or len(spec.hidden_units) >= _lib.MAX_DENSE:
            raise ValueError("too many layers")
        cfg.n_conv = len(spec.conv_layers)
        for i, (f, k) in enumerate(spec.conv_layers):
            cfg.conv_filters[i], cfg.conv_ksize[i] = int(f), int(k)
        cfg.n_hidden = len(spec.hidden_units)
        for j, u in enumerate(spec.hidden_units):
            cfg.hidden_units[j] = int(u)
        cfg.alpha_conv, cfg.alpha_dense = spec.alpha_conv, spec.alpha_dense
        cfg.pad = spec.pad
        cfg.flatten_order = _lib.FLATTEN[spec.flatten]
        cfg.pool_ties = _lib.TIES[spec.pool_ties]
        cfg.head = _lib.HEAD[spec.head]
        cfg.precision = _lib.PRECISION[precision]
        cfg.max_batch = self.max_batch
        cfg.keep_all_activations = 1 if keep_all_activations else 0
        cfg.device = self.device
        cfg.refine_capacity = int(refine_capacity)
        self._h = C.c_void_p()
        if precision == "fp16" and refine_margin is None:
            cfg.refine_margin = self.DEFAULT_REFINE_MARGIN
            if self.lib.bcad_create(C.byref(cfg), C.byref(self._h)) != _lib.OK:     # shape outside the split-operand path
                cfg.refine_margin = 0.0
                _lib.check(self.lib.bcad_create(C.byref(cfg), C.byref(self._h)))
        else:
            cfg.refine_margin = float(refine_margin or 0.0)
            _lib.check(self.lib.bcad_create(C.byref(cfg), C.byref(self._h)))
        self.refine_margin = float(cfg.refine_margin)
        self._committed = False
        self.tdev = torch.device("cuda", self.device)
        #: whoever fills the handle's activation cache for later reads (the mirrors' lazy ``layers[*]`` getters, explain_backward)
        #: stamps it here; every forward of this engine resets it, so a stale read is detectable instead of silently wrong
        self.cache_tag = None
        self.explain_target = "conv"

    # ------------------------------------------------------------------ lifetime / weights
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.bcad_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_weights(self, conv_w, conv_b, dense_w, dense_b, batchnorm=None):
        """conv_w[i]: (F,k,k,C); dense_w[j]: (units,in) with fc1 columns in spec.flatten order."""
        for i, (w, b) in enumerate(zip(conv_w, conv_b)):
            f, k = self.spec.conv_layers[i]
            w = _f32c(w)
            if w.shape[0] != f or w.shape[1] != k or w.shape[2] != k:
                raise ValueError(f"conv {i}: filters shape {w.shape} does not match ({f},{k},{k},C)")
            b = _f32c(b)
            _lib.check(self.lib.bcad_set_conv_weights(self._h, i, _ptr(w), _ptr(b)))
            if batchnorm and batchnorm.get(i) is not None:
                # keep the converted arrays alive across the call (ctypes only sees raw addresses)
                bn = [_f32c(v) for v in batchnorm[i][:4]]
                _lib.check(self.lib.bcad_fold_batchnorm(self._h, i, _ptr(bn[0]), _ptr(bn[1]), _ptr(bn[2]), _ptr(bn[3]),
                                                        float(batchnorm[i][4])))
        _, prev = self.spec.shapes()
        units = list(self.spec.hidden_units) + [self.spec.num_classes]
        if len(dense_w) != len(units):
            raise ValueError(f"expected {len(units)} dense matrices, got {len(dense_w)}")
        for j, (w, b) in enumerate(zip(dense_w, dense_b)):
            w = _f32c(w)
            b = _f32c(b)
            if w.shape != (units[j], prev):
                raise ValueError(f"dense {j}: weights shape {w.shape} does not match {(units[j], prev)}")
            _lib.check(self.lib.bcad_set_dense_weights(self._h, j, _ptr(w), _ptr(b)))
            prev = units[j]
        _lib.check(self.lib.bcad_commit(self._h))
        self._committed = True

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return _stream_of(self.tdev)

    def _as_device_input(self, x) -> torch.Tensor:
        h, w, c = self.spec.input_shape
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        if x.dim() == 3:
            x = x[None]
        if tuple(x.shape[1:]) != (h, w, c):
            raise ValueError(f"input shape {tuple(x.shape)} does not match [B,{h},{w},{c}]")
        return x.to(device=self.tdev, dtype=torch.float32, non_blocking=True).contiguous()

    @property
    def uses_tensor_path(self) -> bool:
        return bool(self.lib.bcad_uses_tensor_path(self._h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.bcad_launch_count(self._h))

    def set_explain_target(self, target: str = "conv"):
        """"conv": the last conv block's post-LeakyReLU output (default; explainability.py:64).  "conv_preact": the conv module's own
        output before the activation -- what pytorch_grad_cam sees when it hooks ``model.convs[-1]`` of ADCNNM.CNNModel (ADCNNM.py:76).
        Every precision runs it: on the tensor paths the channel weights come from a masked fc1 input-gradient GEMM on tcgen05, which
        with first-index pooling needs a first dense layer of a multiple of 64 units (ValueError otherwise: use an fp32 engine).
        A handle with ``refine_margin`` passes the target to its refinement twin."""
        _lib.check(self.lib.bcad_set_explain_target(self._h, _lib.TARGET[target]))
        self.explain_target = target

    def refine_stats(self):
        """(images re-run at fp32 grade, flagged images beyond ``refine_capacity``) since creation; synchronises."""
        a, b = C.c_int64(), C.c_int64()
        _lib.check(self.lib.bcad_refine_stats(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def set_profiling(self, on: bool):
        _lib.check(self.lib.bcad_set_profiling(self._h, 1 if on else 0))

    def last_profile(self):
        """[(kernel name, ms)] of the last device-buffer call (needs set_profiling(True) before it)."""
        n = int(self.lib.bcad_profile_count(self._h))
        out = []
        for i in range(n):
            buf = C.create_string_buffer(64)
            ms = C.c_float()
            _lib.check(self.lib.bcad_profile_get(self._h, i, buf, 64, C.byref(ms)))
            out.append((buf.value.decode(), float(ms.value)))
        return out

    # ------------------------------------------------------------------ hot path, device tensors
    def predict(self, x):
        """-> (cls int32 [B], probs fp32 [B,nc], logits fp32 [B,nc]) as CUDA tensors."""
        self.cache_tag = None
        x = self._as_device_input(x)
        B, nc = x.shape[0], self.spec.num_classes
        with torch.cuda.device(self.tdev):
            logits = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            probs = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            cls = torch.empty((B,), device=self.tdev, dtype=torch.int32)
            _lib.check(self.lib.bcad_predict(self._h, _ptr(x), B, _ptr(logits), _ptr(probs), _ptr(cls), self._stream()))
        return cls, probs, logits

    def predict_explain(self, x, class_idx=None, grad_mode: str = "logit", out_heat: Optional[torch.Tensor] = None,
                        out_hw: Optional[Tuple[int, int]] = None):
        """-> (cls, probs, logits, heatmaps fp32 [B,H,W]) as CUDA tensors.  ``out_hw``: heat-maps resized to that size instead
        of the model's input size (pytorch_grad_cam scales the cam to the image it explains: GRADCAM.py:46-64 with a 512x512
        image, app.py:649-657)."""
        self.cache_tag = None
        x = self._as_device_input(x)
        B, nc = x.shape[0], self.spec.num_classes
        h, w, _ = self.spec.input_shape
        if out_hw is not None:
            h, w = int(out_hw[0]), int(out_hw[1])
        with torch.cuda.device(self.tdev):
            logits = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            probs = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            cls = torch.empty((B,), device=self.tdev, dtype=torch.int32)
            heat = out_heat if out_heat is not None else torch.empty((B, h, w), device=self.tdev, dtype=torch.float32)
            if tuple(heat.shape) != (B, h, w) or heat.dtype != torch.float32 or not heat.is_contiguous():
                raise ValueError(f"out_heat must be a contiguous float32 [{B},{h},{w}] tensor")
            ci = self._class_idx(class_idx, B)
            if out_hw is None:
                _lib.check(self.lib.bcad_predict_explain(self._h, _ptr(x), B, _ptr(ci), _lib.GRAD_MODE[grad_mode],
                                                         _ptr(logits), _ptr(probs), _ptr(cls), _ptr(heat), self._stream()))
            else:
                _lib.check(self.lib.bcad_predict_explain_sized(self._h, _ptr(x), B, _ptr(ci), _lib.GRAD_MODE[grad_mode],
                                                               _ptr(logits), _ptr(probs), _ptr(cls), h, w, _ptr(heat), self._stream()))
        return cls, probs, logits, heat

    def predict_explain_classes(self, x, classes=None, grad_mode: str = "logit", out_hw: Optional[Tuple[int, int]] = None,
                                out_heat: Optional[torch.Tensor] = None):
        """Grad-CAM for K target classes per image from one forward (the dual-class explanation of app.py:649-657 -> GRADCAM.py:63-64)
        -> (cls, probs, logits, heatmaps fp32 [B,K,H,W]) as CUDA tensors.  ``classes``: None = every class (K = num_classes), a
        length-K sequence shared by the batch, or a [B,K] array; K <= 8.  ``heat[:, k]`` is bitwise what ``predict_explain`` returns
        for class column k."""
        self.cache_tag = None
        x = self._as_device_input(x)
        B, nc = x.shape[0], self.spec.num_classes
        h, w, _ = self.spec.input_shape
        if out_hw is not None:
            h, w = int(out_hw[0]), int(out_hw[1])
            if h < 1 or w < 1:
                raise ValueError(f"out_hw must be positive, got {out_hw}")
        K, ci = self._class_rows(classes, B)
        with torch.cuda.device(self.tdev):
            logits = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            probs = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            cls = torch.empty((B,), device=self.tdev, dtype=torch.int32)
            heat = out_heat if out_heat is not None else torch.empty((B, K, h, w), device=self.tdev, dtype=torch.float32)
            if tuple(heat.shape) != (B, K, h, w) or heat.dtype != torch.float32 or not heat.is_contiguous():
                raise ValueError(f"out_heat must be a contiguous float32 [{B},{K},{h},{w}] tensor")
            if ci is not None:
                ci = ci.to(self.tdev).contiguous()
            oh, ow = (h, w) if out_hw is not None else (0, 0)
            _lib.check(self.lib.bcad_predict_explain_classes(self._h, _ptr(x), B, K, _ptr(ci), _lib.GRAD_MODE[grad_mode],
                                                             _ptr(logits), _ptr(probs), _ptr(cls), oh, ow, _ptr(heat), self._stream()))
        return cls, probs, logits, heat

    def predict_saliency_classes(self, x, classes=None, grad_mode: str = "softmax_ce", want_d_input: bool = False):
        """Input-gradient saliency (explainability.py:44-73) for K target classes per image from one forward -> (cls, probs, logits,
        saliency fp32 [B,K,H,W] in [0,1], d_input fp32 [B,K,H,W,C] or None) as CUDA tensors.  ``classes`` as in
        ``predict_explain_classes``.  fp32 engines with ``keep_all_activations``; with ``set_fast_training(True)`` the eligible blocks'
        input gradients run on the tensor cores (bcad_predict_saliency_classes)."""
        self.cache_tag = None
        x = self._as_device_input(x)
        B, nc = x.shape[0], self.spec.num_classes
        h, w, c = self.spec.input_shape
        K, ci = self._class_rows(classes, B)
        with torch.cuda.device(self.tdev):
            logits = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            probs = torch.empty((B, nc), device=self.tdev, dtype=torch.float32)
            cls = torch.empty((B,), device=self.tdev, dtype=torch.int32)
            sal = torch.empty((B, K, h, w), device=self.tdev, dtype=torch.float32)
            d_in = torch.empty((B, K, h, w, c), device=self.tdev, dtype=torch.float32) if want_d_input else None
            if ci is not None:
                ci = ci.to(self.tdev).contiguous()
            _lib.check(self.lib.bcad_predict_saliency_classes(self._h, _ptr(x), B, K, _ptr(ci), _lib.GRAD_MODE[grad_mode], _ptr(logits),
                                                              _ptr(probs), _ptr(cls), _ptr(sal), _ptr(d_in), self._stream()))
        return cls, probs, logits, sal, d_in

    def _class_rows(self, classes, B):
        """classes of the multi-class calls -> (K, int32 [B,K] tensor or None = column k is class k)."""
        nc = self.spec.num_classes
        if classes is None:
            K, ci = nc, None
        else:
            ci = torch.as_tensor(classes, dtype=torch.int32)
            if ci.dim() == 1:
                ci = ci[None].expand(B, -1)
            if ci.dim() != 2 or ci.shape[0] != B:
                raise ValueError(f"classes must be a length-K sequence or a [{B},K] array, got shape {tuple(ci.shape)}")
            K = ci.shape[1]
            if K >= 1 and (int(ci.min()) < 0 or int(ci.max()) >= nc):
                raise ValueError("classes out of range")
        if not 1 <= K <= _lib.MAX_EXPLAIN_CLASSES:
            raise ValueError(f"{K} target classes per image; 1..{_lib.MAX_EXPLAIN_CLASSES} are supported")
        return K, ci

    def _class_idx(self, class_idx, B):
        if class_idx is None:
            return None
        ci = torch.as_tensor(class_idx, dtype=torch.int32).reshape(-1)
        if ci.numel() == 1:
            ci = ci.expand(B)
        if ci.numel() != B:
            raise ValueError(f"class_idx has {ci.numel()} entries for a batch of {B}")
        if int(ci.min()) < 0 or int(ci.max()) >= self.spec.num_classes:
            raise ValueError("class_idx out of range")
        return ci.to(self.tdev).contiguous()

    def explain_backward(self, B: int, class_idx, grad_mode: str = "softmax_ce",
                         want_conv: Sequence[int] = (), want_input: bool = False):
        """After predict() of the same B: ({conv_block: dA [B,h,w,F]}, d_input [B,H,W,C] | None)."""
        shapes, _ = self.spec.shapes()
        n_conv = len(shapes)
        with torch.cuda.device(self.tdev):
            ptrs = (C.c_void_p * n_conv)()
            outs = {}
            for i in want_conv:
                ch, cw, f = shapes[i][0]
                outs[i] = torch.empty((B, ch, cw, f), device=self.tdev, dtype=torch.float32)
                ptrs[i] = outs[i].data_ptr()
            d_in = None
            if want_input:
                d_in = torch.empty((B,) + tuple(self.spec.input_shape), device=self.tdev, dtype=torch.float32)
            ci = self._class_idx(class_idx, B)
            _lib.check(self.lib.bcad_explain_backward(self._h, B, _ptr(ci), _lib.GRAD_MODE[grad_mode],
                                                      ptrs, _ptr(d_in), self._stream()))
        return outs, d_in

    def get_tensor(self, kind: int, index: int, B: int) -> torch.Tensor:
        per = int(self.lib.bcad_tensor_elems(self._h, kind, index))
        if per <= 0:
            raise ValueError(f"no such tensor ({kind},{index})")
        with torch.cuda.device(self.tdev):
            out = torch.empty((B, per), device=self.tdev, dtype=torch.float32)
            _lib.check(self.lib.bcad_get_tensor(self._h, kind, index, B, _ptr(out), self._stream()))
        return out

    # ------------------------------------------------------------------ training step (SURVEY 8 row f4)
    def grad_elems(self) -> int:
        return int(self.lib.bcad_grad_elems(self._h))

    def grad_layout(self, is_dense: bool, index: int):
        vals = [C.c_int64() for _ in range(4)]
        _lib.check(self.lib.bcad_grad_layout(self._h, 1 if is_dense else 0, index, *[C.byref(v) for v in vals]))
        return tuple(int(v.value) for v in vals)          # (w_off, w_elems, b_off, b_elems)

    def train_backward(self, x: torch.Tensor, labels, grads: Optional[torch.Tensor] = None, part: int = 0,
                       loss: Optional[torch.Tensor] = None):
        """After ``predict(x)`` of the same batch (fp32 engine, keep_all_activations=True):
        -> (flat gradient of the MEAN cross-entropy [grad_elems], per-sample loss [B]) as CUDA tensors.
        ``part``: 0 everything; 1 the loss + dense layers only (their slice of ``grads`` is final afterwards); 2 the conv blocks
        (after part 1 of the same batch) -- the split a data-parallel step uses to all-reduce fc1 while the convs run."""
        x = self._as_device_input(x)
        B = x.shape[0]
        lab = torch.as_tensor(labels, dtype=torch.int32).reshape(-1).to(self.tdev).contiguous()
        if lab.numel() != B:
            raise ValueError("one label per image")
        with torch.cuda.device(self.tdev):
            if grads is None:
                grads = torch.zeros((self.grad_elems(),), device=self.tdev, dtype=torch.float32)   # gaps between tensors stay 0
            if loss is None:
                loss = torch.empty((B,), device=self.tdev, dtype=torch.float32)
            _lib.check(self.lib.bcad_train_backward_part(self._h, _ptr(x), _ptr(lab), B, _ptr(grads), _ptr(loss), int(part), self._stream()))
        return grads, loss

    def set_fast_training(self, on: bool = True):
        """Training step on the tensor cores where the shape allows (bcad_set_fast_training): the 32 -> 64 conv block's forward, input
        gradient and weight gradient as split-operand tcgen05 GEMMs (~1e-4 relative against the fp32 kernels).  fp32 handles only."""
        _lib.check(self.lib.bcad_set_fast_training(self._h, 1 if on else 0))

    def set_dropout_masks(self, masks, mask_backward: bool = True):
        """masks [B, sum(hidden_units)] multipliers (0 or 1/(1-rate)) for the next forwards of exactly B images; None = off.
        mask_backward=False restates the NumPy reference, whose backward ignores the mask (Classes/CNNModel.py:307-316)."""
        if masks is None:
            _lib.check(self.lib.bcad_set_dropout_masks(self._h, None, 0, 1, self._stream()))
            return
        mk = torch.as_tensor(masks, dtype=torch.float32).to(self.tdev).contiguous()
        if mk.dim() != 2 or mk.shape[1] != sum(self.spec.hidden_units):
            raise ValueError(f"dropout masks must be [B, {sum(self.spec.hidden_units)}], got {tuple(mk.shape)}")
        with torch.cuda.device(self.tdev):
            _lib.check(self.lib.bcad_set_dropout_masks(self._h, _ptr(mk), mk.shape[0], 1 if mask_backward else 0, self._stream()))
            torch.cuda.current_stream(self.tdev).synchronize()      # mk may be freed on return

    def apply_update(self, grads: torch.Tensor, opt: str = "sgd_clip", lr: float = 0.01, max_norm: float = 5.0,
                     betas=(0.9, 0.999), eps: float = 1e-8):
        """opt "sgd_clip": Classes/CNNModel.py:372-394; opt "adam": torch.optim.Adam as ADCNNM.py:88."""
        code = {"sgd_clip": 0, "sgd": 0, "adam": 1}[opt]
        with torch.cuda.device(self.tdev):
            _lib.check(self.lib.bcad_apply_update(self._h, _ptr(grads), code, float(lr), float(max_norm if opt != "sgd" else 0.0),
                                                  float(betas[0]), float(betas[1]), float(eps), self._stream()))

    def get_weights(self):
        """Current device weights in the reference layouts: ([F,k,k,C]), ([F]), ([units,in] fc1 in spec.flatten order), ([units])."""
        conv_w, conv_b, dense_w, dense_b = [], [], [], []
        cin = self.spec.input_shape[2]
        for i, (f, k) in enumerate(self.spec.conv_layers):
            w, b = np.empty((f, k, k, cin), np.float32), np.empty((f,), np.float32)
            _lib.check(self.lib.bcad_get_conv_weights(self._h, i, _ptr(w), _ptr(b)))
            conv_w.append(w); conv_b.append(b)
            cin = f
        _, prev = self.spec.shapes()
        for j, u in enumerate(list(self.spec.hidden_units) + [self.spec.num_classes]):
            w, b = np.empty((u, prev), np.float32), np.empty((u,), np.float32)
            _lib.check(self.lib.bcad_get_dense_weights(self._h, j, _ptr(w), _ptr(b)))
            dense_w.append(w); dense_b.append(b)
            prev = u
        return conv_w, conv_b, dense_w, dense_b

    def unpack_grads(self, grads: torch.Tensor):
        """Flat device-layout gradient -> reference layouts (dict like oracle.train.mean_grads)."""
        g = grads.detach().cpu().numpy()
        out = {"conv_w": [], "conv_b": [], "dense_w": [], "dense_b": []}
        cin = self.spec.input_shape[2]
        shapes, prev = self.spec.shapes()
        for i, (f, k) in enumerate(self.spec.conv_layers):
            wo, we, bo, be = self.grad_layout(False, i)
            cpad = be
            pk = g[wo:wo + we].reshape(k * k, cin, cpad)[:, :, :f]                      # [tap][c][f]
            out["conv_w"].append(np.ascontiguousarray(pk.transpose(2, 0, 1)).reshape(f, k, k, cin))
            out["conv_b"].append(g[bo:bo + f].copy())
            cin = f
        ph, pw, pc = shapes[-1][1]
        for j, u in enumerate(list(self.spec.hidden_units) + [self.spec.num_classes]):
            wo, we, bo, be = self.grad_layout(True, j)
            w = g[wo:wo + we].reshape(u, prev)
            if j == 0 and self.spec.flatten == "chw":                                   # device order is (h,w,c)
                w = w.reshape(u, ph, pw, pc).transpose(0, 3, 1, 2).reshape(u, -1)
            out["dense_w"].append(np.ascontiguousarray(w))
            out["dense_b"].append(g[bo:bo + be].copy())
            prev = u
        return out

    # ------------------------------------------------------------------ hot path, host buffers (end to end)
    def predict_explain_host(self, x: np.ndarray, class_idx: Optional[np.ndarray] = None, grad_mode: str = "logit",
                             heat_out: Optional[np.ndarray] = None, want_heat: bool = True, heat_dtype=np.float32):
        """x: float32 [B,H,W,C] host array (pinned memory makes the copies asynchronous), or uint8 [B,H,W,C] 0-255 pixels,
        which the device normalises as ``float32(x) / 255`` (app.py:71, GRADCAM.py:46): a quarter of the host->device bytes.
        -> (cls int32 [B], probs [B,nc], logits [B,nc], heat [B,H,W]) as host arrays.
        heat_dtype=np.uint8 returns ``heatmap_uint8 = (cam * 255).astype(uint8)`` (GRADCAM.py:70) instead of the float32 map:
        a quarter of the device->host bytes of a PCIe-bound call."""
        self.cache_tag = None
        u8 = np.dtype(heat_dtype) == np.uint8
        h, w, c = self.spec.input_shape
        x8 = x.dtype == np.uint8
        if x8:
            x = np.ascontiguousarray(x)
        elif x.dtype != np.float32 or not x.flags["C_CONTIGUOUS"]:
            x = np.ascontiguousarray(x, dtype=np.float32)
        if x.ndim == 3:
            x = x[None]
        if x.shape[1:] != (h, w, c):
            raise ValueError(f"input shape {x.shape} does not match [B,{h},{w},{c}]")
        B, nc = x.shape[0], self.spec.num_classes
        logits, probs, cls = np.empty((B, nc), np.float32), np.empty((B, nc), np.float32), np.empty((B,), np.int32)
        heat = _out_array(heat_out, (B, h, w), np.uint8 if u8 else np.float32, "heat_out") if want_heat else None
        ci = _host_class_idx(class_idx, B, nc)
        if x8:
            hf, h8 = (None, heat) if u8 else (heat, None)
            _lib.check(self.lib.bcad_predict_explain_host_u8in(self._h, _ptr(x), B, _ptr(ci), _lib.GRAD_MODE[grad_mode], _ptr(logits),
                                                               _ptr(probs), _ptr(cls), _ptr(hf), _ptr(h8)))
            return cls, probs, logits, heat
        fn = self.lib.bcad_predict_explain_host_u8 if (u8 and want_heat) else self.lib.bcad_predict_explain_host
        _lib.check(fn(self._h, _ptr(x), B, _ptr(ci), _lib.GRAD_MODE[grad_mode], _ptr(logits), _ptr(probs), _ptr(cls), _ptr(heat)))
        return cls, probs, logits, heat

    def gradcam_overlays_host(self, gray_u8: np.ndarray, class_idx=None, grad_mode: str = "logit", standardise: bool = True,
                              overlay_out: Optional[np.ndarray] = None, heat_out: Optional[np.ndarray] = None,
                              want_overlay: bool = True, want_heat: bool = True):
        """The GRADCAM.py call surface for a batch, end to end through one C-ABI call (bcad_gradcam_overlays_host): uint8 grey
        images [B,H,W] (model input size) -> (cls int32 [B], probs [B,nc], logits [B,nc], overlay uint8 RGB [B,H,W,3] =
        show_cam_on_image, heatmap_uint8 [B,H,W]).  ``standardise``: the CNN input is the per-image standardised img/255 (the
        reference's CNN-input normalisation, app.py:179-182), else img/255 itself.  Pinned host arrays make the copies asynchronous."""
        self.cache_tag = None
        h, w, _ = self.spec.input_shape
        g = _gray_batch(gray_u8)
        if g.shape[1:] != (h, w):
            raise ValueError(f"image shape {g.shape} does not match [B,{h},{w}]")
        B, nc = g.shape[0], self.spec.num_classes
        logits, probs, cls = np.empty((B, nc), np.float32), np.empty((B, nc), np.float32), np.empty((B,), np.int32)
        ov = _out_array(overlay_out, (B, h, w, 3), np.uint8, "overlay_out") if want_overlay else None
        hu = _out_array(heat_out, (B, h, w), np.uint8, "heat_out") if want_heat else None
        ci = _host_class_idx(class_idx, B, nc)
        _lib.check(self.lib.bcad_gradcam_overlays_host(self._h, _ptr(g), B, _ptr(ci), _lib.GRAD_MODE[grad_mode], 1 if standardise else 0,
                                                       _ptr(logits), _ptr(probs), _ptr(cls), _ptr(ov), _ptr(hu)))
        return cls, probs, logits, ov, hu

    def gradcam_overlays_classes_host(self, gray_u8: np.ndarray, classes=(0, 1), grad_mode: str = "logit", standardise: bool = True,
                                      overlay_out: Optional[np.ndarray] = None, heat_out: Optional[np.ndarray] = None,
                                      want_overlay: bool = True, want_heat: bool = True):
        """The deployed dual-class call (app.py:649-657 -> GRADCAM.py:31-81) for a batch, end to end through one C-ABI call
        (bcad_gradcam_overlays_classes_host): uint8 grey images [B,h,w] of ANY size -> (cls int32 [B], probs [B,nc], logits [B,nc],
        overlay uint8 RGB [B,K,h,w,3] = show_cam_on_image, heatmap_uint8 [B,K,h,w]).  The CNN sees cv2.resize(img / 255, model size)
        (standardised per image when ``standardise``); the maps have the size of the image.  ``classes``: a length-K sequence shared by
        the batch, a [B,K] array or None (every class); K <= 8.  Pinned host arrays make the copies asynchronous."""
        self.cache_tag = None
        g = _gray_batch(gray_u8)
        B, h, w = g.shape
        nc = self.spec.num_classes
        K, ci = _host_class_rows(classes, B, nc)
        logits, probs, cls = np.empty((B, nc), np.float32), np.empty((B, nc), np.float32), np.empty((B,), np.int32)
        ov = _out_array(overlay_out, (B, K, h, w, 3), np.uint8, "overlay_out") if want_overlay else None
        hu = _out_array(heat_out, (B, K, h, w), np.uint8, "heat_out") if want_heat else None
        _lib.check(self.lib.bcad_gradcam_overlays_classes_host(self._h, _ptr(g), B, h, w, K, _ptr(ci), _lib.GRAD_MODE[grad_mode],
                                                               1 if standardise else 0, _ptr(logits), _ptr(probs), _ptr(cls), _ptr(ov),
                                                               _ptr(hu)))
        return cls, probs, logits, ov, hu

    def saliency_overlays_classes_host(self, gray_u8: np.ndarray, classes=(0, 1), grad_mode: str = "softmax_ce", standardise: bool = True,
                                       overlay_out: Optional[np.ndarray] = None, heat_out: Optional[np.ndarray] = None,
                                       saliency_out: Optional[np.ndarray] = None, want_overlay: bool = True, want_heat: bool = True,
                                       want_saliency: bool = False):
        """The dual-class input-gradient saliency overlays (explainability.py:81-108) for a batch, end to end through one C-ABI call
        (bcad_saliency_overlays_classes_host): uint8 grey images [B,h,w] of ANY size -> (cls int32 [B], probs [B,nc], logits [B,nc],
        overlays uint8 BGR [B,K,h,w,3], heat-maps uint8 BGR [B,K,h,w,3], saliency fp32 [B,K,H,W] at the model's size or None).  The CNN
        sees the input ``gradcam_overlays_classes_host`` builds (cv2.resize(img / 255, model size), standardised per image when
        ``standardise``); each map is coloured with JET, resized to the image's size as cv2.resize does on 8-bit BGR, and blended 50/50 with
        the grey image.  ``classes`` as in ``gradcam_overlays_classes_host``; ``grad_mode`` defaults to the reference's softmax
        cross-entropy gradient.  fp32 engines with ``keep_all_activations`` (a model's ``saliency_engine``).  The saliency maps are copied
        back only when ``want_saliency`` or ``saliency_out`` is given.  Pinned host arrays make the copies asynchronous."""
        self.cache_tag = None
        g = _gray_batch(gray_u8)
        B, h, w = g.shape
        H, W, _ = self.spec.input_shape
        nc = self.spec.num_classes
        K, ci = _host_class_rows(classes, B, nc)
        logits, probs, cls = np.empty((B, nc), np.float32), np.empty((B, nc), np.float32), np.empty((B,), np.int32)
        ov = _out_array(overlay_out, (B, K, h, w, 3), np.uint8, "overlay_out") if want_overlay else None
        hm = _out_array(heat_out, (B, K, h, w, 3), np.uint8, "heat_out") if want_heat else None
        sal = _out_array(saliency_out, (B, K, H, W), np.float32, "saliency_out") if (want_saliency or saliency_out is not None) else None
        _lib.check(self.lib.bcad_saliency_overlays_classes_host(self._h, _ptr(g), B, h, w, K, _ptr(ci), _lib.GRAD_MODE[grad_mode],
                                                                1 if standardise else 0, _ptr(logits), _ptr(probs), _ptr(cls), _ptr(sal),
                                                                _ptr(ov), _ptr(hm)))
        return cls, probs, logits, ov, hm, sal


def gradcam_tail(A: torch.Tensor, dA: torch.Tensor, out_hw: Tuple[int, int]) -> torch.Tensor:
    """Stand-alone Grad-CAM tail on NHWC CUDA tensors [B,h,w,K] (fp32 or bf16) -> fp32 [B,H,W]."""
    lib = _lib.load()
    if A.shape != dA.shape or A.dtype != dA.dtype or A.dim() != 4:
        raise ValueError("A and dA must be NHWC tensors of the same shape and dtype")
    if A.dtype not in (torch.float32, torch.bfloat16):
        raise ValueError("fp32 or bf16 only")
    A, dA = A.contiguous(), dA.contiguous()
    B, h, w, K = A.shape
    H, W = out_hw
    out = torch.empty((B, H, W), device=A.device, dtype=torch.float32)
    with torch.cuda.device(A.device):
        _lib.check(lib.bcad_gradcam_tail(_ptr(A), _ptr(dA), B, K, h, w, H, W, 0 if A.dtype == torch.float32 else 1,
                                         _ptr(out), _stream_of(A.device)))
    return out


def gray_preprocess(gray_u8: torch.Tensor, channels: int = 1, standardise: bool = True):
    """uint8 grey images [B,H,W] on the GPU -> (img01 fp32 [B,H,W] = u8 / 255, x fp32 [B,H,W,channels] = the CNN input)."""
    lib = _lib.load()
    g = gray_u8.contiguous()
    if g.dtype != torch.uint8 or g.dim() != 3 or not g.is_cuda:
        raise ValueError("gray_u8 must be a CUDA uint8 tensor [B,H,W]")
    B, H, W = g.shape
    img01 = torch.empty((B, H, W), device=g.device, dtype=torch.float32)
    x = torch.empty((B, H, W, channels), device=g.device, dtype=torch.float32)
    with torch.cuda.device(g.device):
        _lib.check(lib.bcad_gray_preprocess(_ptr(g), B, H, W, int(channels), 1 if standardise else 0, _ptr(img01), _ptr(x),
                                            _stream_of(g.device)))
    return img01, x


def gray_resize_preprocess(gray_u8: torch.Tensor, out_hw: Tuple[int, int], channels: int = 1, standardise: bool = True) -> torch.Tensor:
    """uint8 grey images [B,h,w] of any size on the GPU -> the CNN input x fp32 [B,H,W,channels] = cv2.resize(u8 / 255, (W, H),
    INTER_LINEAR), standardised per image (mean / std of the resized image) when ``standardise``; ``out_hw`` = (H, W)."""
    lib = _lib.load()
    g = gray_u8.contiguous()
    if g.dtype != torch.uint8 or g.dim() != 3 or not g.is_cuda:
        raise ValueError("gray_u8 must be a CUDA uint8 tensor [B,H,W]")
    B, h, w = g.shape
    H, W = int(out_hw[0]), int(out_hw[1])
    x = torch.empty((B, H, W, channels), device=g.device, dtype=torch.float32)
    with torch.cuda.device(g.device):
        _lib.check(lib.bcad_gray_resize_preprocess(_ptr(g), B, h, w, H, W, int(channels), 1 if standardise else 0, _ptr(x),
                                                   _stream_of(g.device)))
    return x


def overlay_classes(gray_u8: torch.Tensor, cams: torch.Tensor, want_overlay=True, want_heat_u8=True):
    """show_cam_on_image + heatmap_uint8 for K maps per grey image on CUDA tensors: ``gray_u8`` uint8 [B,H,W] (img01 = u8 / 255, read
    once for the K maps), ``cams`` fp32 [B,K,H,W] -> (u8 [B,K,H,W,3], u8 [B,K,H,W]); map k is byte for byte ``overlay(u8 / 255, cams[:, k])``."""
    lib = _lib.load()
    g = gray_u8.contiguous()
    cam = cams.to(torch.float32).contiguous()
    if cam.dim() != 4:
        raise ValueError(f"cams must be [B,K,H,W], got shape {tuple(cam.shape)}")
    B, K, H, W = cam.shape
    if g.dtype != torch.uint8 or tuple(g.shape) != (B, H, W) or g.device != cam.device:
        raise ValueError(f"gray_u8 must be a uint8 [{B},{H},{W}] tensor on the cams' device")
    ov = torch.empty((B, K, H, W, 3), device=cam.device, dtype=torch.uint8) if want_overlay else None
    hu = torch.empty((B, K, H, W), device=cam.device, dtype=torch.uint8) if want_heat_u8 else None
    with torch.cuda.device(cam.device):
        _lib.check(lib.bcad_overlay_classes(_ptr(g), _ptr(cam), B, K, H, W, _ptr(ov), _ptr(hu),
                                            _stream_of(cam.device)))
    return ov, hu


def overlay(img01: torch.Tensor, cam: torch.Tensor, want_overlay=True, want_heat_u8=True):
    """show_cam_on_image + heatmap_uint8 (GRADCAM.py:67,70) on CUDA tensors [B,H,W] -> (u8 [B,H,W,3], u8 [B,H,W])."""
    lib = _lib.load()
    img01 = img01.to(torch.float32).contiguous()
    cam = cam.to(torch.float32).contiguous()
    B, H, W = cam.shape
    ov = torch.empty((B, H, W, 3), device=cam.device, dtype=torch.uint8) if want_overlay else None
    hu = torch.empty((B, H, W), device=cam.device, dtype=torch.uint8) if want_heat_u8 else None
    with torch.cuda.device(cam.device):
        _lib.check(lib.bcad_overlay(_ptr(img01), _ptr(cam), B, H, W, _ptr(ov), _ptr(hu),
                                    _stream_of(cam.device)))
    return ov, hu


def saliency_overlay(base_u8, saliency: torch.Tensor):
    """generate_saliency_overlay's colouring (explainability.py:74-77) for [B,K] maps on the GPU: ``base_u8`` uint8 [B,H,W], [B,H,W,1]
    (grey, replicated) or [B,H,W,3] (BGR), shared by an image's K maps; ``saliency`` fp32 [B,K,H,W] in [0,1]
    -> (overlay u8 [B,K,H,W,3], heat-map u8 [B,K,H,W,3]), both BGR as cv2 returns them."""
    lib = _lib.load()
    sal = saliency.to(torch.float32).contiguous()
    if sal.dim() != 4:
        raise ValueError(f"saliency must be [B,K,H,W], got shape {tuple(sal.shape)}")
    B, K, H, W = sal.shape
    base = torch.as_tensor(base_u8).to(device=sal.device)
    if base.dim() == 3:
        base = base[..., None]
    if base.dtype != torch.uint8 or base.dim() != 4 or tuple(base.shape[:3]) != (B, H, W) or base.shape[3] not in (1, 3):
        raise ValueError(f"base_u8 must be uint8 [{B},{H},{W}] or [{B},{H},{W},1|3], got {base.dtype} {tuple(base.shape)}")
    base = base.contiguous()
    ov = torch.empty((B, K, H, W, 3), device=sal.device, dtype=torch.uint8)
    heat = torch.empty((B, K, H, W, 3), device=sal.device, dtype=torch.uint8)
    with torch.cuda.device(sal.device):
        _lib.check(lib.bcad_saliency_overlay(_ptr(base), int(base.shape[3]), _ptr(sal), B, K, H, W, _ptr(ov), _ptr(heat),
                                             _stream_of(sal.device)))
    return ov, heat


def saliency_overlay_resized(gray_u8: torch.Tensor, saliency: torch.Tensor, want_overlay=True, want_heat=True):
    """generate_saliency_overlay (explainability.py:74-77) at the image's size for [B,K] maps on CUDA tensors: ``gray_u8`` uint8 [B,h,w]
    (the blend base, replicated to 3 channels, read once for the K maps), ``saliency`` fp32 [B,K,H,W] in [0,1] at any (model) size
    -> (overlay u8 [B,K,h,w,3], heat-map u8 [B,K,h,w,3]), both BGR: heat = cv2.resize(applyColorMap(uint8(s * 255), JET), (w, h)) with
    OpenCV's 8-bit INTER_LINEAR arithmetic, overlay = addWeighted(grey3, 0.5, heat, 0.5, 0)."""
    lib = _lib.load()
    g = gray_u8.contiguous()
    sal = saliency.to(torch.float32).contiguous()
    if sal.dim() != 4:
        raise ValueError(f"saliency must be [B,K,H,W], got shape {tuple(sal.shape)}")
    B, K, H, W = sal.shape
    if g.dtype != torch.uint8 or g.dim() != 3 or g.shape[0] != B or g.device != sal.device:
        raise ValueError(f"gray_u8 must be a uint8 [{B},h,w] tensor on the saliency maps' device")
    h, w = g.shape[1:]
    ov = torch.empty((B, K, h, w, 3), device=sal.device, dtype=torch.uint8) if want_overlay else None
    heat = torch.empty((B, K, h, w, 3), device=sal.device, dtype=torch.uint8) if want_heat else None
    with torch.cuda.device(sal.device):
        _lib.check(lib.bcad_saliency_overlay_resized(_ptr(g), _ptr(sal), B, K, H, W, h, w, _ptr(ov), _ptr(heat),
                                                     _stream_of(sal.device)))
    return ov, heat


# --------------------------------------------------------------------------------------------------
# batch sharding (SURVEY 8e): contiguous split, replicated weights, no collective on this path
# --------------------------------------------------------------------------------------------------
def shard_bounds(n: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous near-equal split of n images over `world` ranks: [(start, stop)] (empty shards allowed)."""
    base, rem = divmod(n, world)
    out, s = [], 0
    for r in range(world):
        e = s + base + (1 if r < rem else 0)
        out.append((s, e))
        s = e
    return out


class ShardedEngine:
    """Single-process driver over several GPUs of one box (north_star (d)): one Engine + one host thread per GPU, contiguous
    batch split, replicated weights, NO collective.  Results land in PINNED host arrays owned by the driver (reused from call to
    call while the batch size stays the same), so every shard's device->host copies are asynchronous and overlap the other
    shards' work; pass a pinned ``x`` (``torch.Tensor.pin_memory().numpy()``) for the same on the way in."""

    def __init__(self, spec: NetSpec, devices: Sequence[int], **kw):
        self.engines = [Engine(spec, device=d, **kw) for d in devices]
        self.spec = spec
        self._out = None

    def set_weights(self, *a, **k):
        for e in self.engines:
            e.set_weights(*a, **k)

    def _pinned(self, key, specs):
        """The driver's pinned output arrays for ``key``, one per (shape, torch dtype) of ``specs``.  One set is kept: a call with
        another key replaces it."""
        if self._out is None or self._out[0] != key:
            self._out = (key, tuple(torch.empty(shape, dtype=dt).pin_memory() for shape, dt in specs))
        return tuple(t.numpy() for t in self._out[1])

    def _fan_out(self, B, work):
        """work(engine, start, stop) on one host thread per engine over shard_bounds(B), empty shards skipped; raises the first error
        once every thread has joined."""
        errs = []

        def run(e, s, t):
            try:
                work(e, s, t)
            except Exception as ex:  # surfaced after join
                errs.append(ex)

        ths = [threading.Thread(target=run, args=(e, s, t))
               for e, (s, t) in zip(self.engines, shard_bounds(B, len(self.engines))) if t > s]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errs:
            raise errs[0]

    def predict_explain_host(self, x: np.ndarray, class_idx=None, grad_mode="logit", heat_dtype=np.float32):
        """-> (cls, probs, logits, heat) host arrays over the whole batch.  The arrays are the driver's pinned buffers: they are
        overwritten by the next call with the same batch size (copy what must outlive it)."""
        B = x.shape[0]
        h, w, _ = self.spec.input_shape
        nc = self.spec.num_classes
        heat_t = torch.uint8 if np.dtype(heat_dtype) == np.uint8 else torch.float32
        cls, probs, logits, heat = self._pinned((B, np.dtype(heat_dtype).str), [((B,), torch.int32), ((B, nc), torch.float32),
                                                                                ((B, nc), torch.float32), ((B, h, w), heat_t)])
        ci = _host_class_idx(class_idx, B, nc)

        def work(e, s, t):
            cls[s:t], probs[s:t], logits[s:t], _ = e.predict_explain_host(x[s:t], None if ci is None else ci[s:t], grad_mode,
                                                                          heat_out=heat[s:t], heat_dtype=heat_dtype)

        self._fan_out(B, work)
        return cls, probs, logits, heat

    def gradcam_overlays_classes_host(self, gray_u8: np.ndarray, classes=(0, 1), grad_mode="logit", standardise=True):
        """Engine.gradcam_overlays_classes_host over the GPUs of the box: contiguous split, one host thread per GPU
        -> (cls, probs, logits, overlays [B,K,h,w,3], heatmap_uint8 [B,K,h,w]).  The arrays are the driver's pinned buffers: they are
        overwritten by the next call of the same shape (copy what must outlive it)."""
        g = _gray_batch(gray_u8)
        B, h, w = g.shape
        nc = self.spec.num_classes
        K, ci = _host_class_rows(classes, B, nc)
        cls, probs, logits, ov, hu = self._pinned(("classes", B, K, h, w), [((B,), torch.int32), ((B, nc), torch.float32),
                                                                             ((B, nc), torch.float32), ((B, K, h, w, 3), torch.uint8),
                                                                             ((B, K, h, w), torch.uint8)])

        def work(e, s, t):
            cls[s:t], probs[s:t], logits[s:t], _, _ = e.gradcam_overlays_classes_host(g[s:t], None if ci is None else ci[s:t], grad_mode,
                                                                                      standardise, overlay_out=ov[s:t], heat_out=hu[s:t])

        self._fan_out(B, work)
        return cls, probs, logits, ov, hu

    def set_fast_training(self, on: bool = True):
        """Engine.set_fast_training on every GPU's engine (a model's ``saliency_engine`` has it on where the shape allows)."""
        for e in self.engines:
            e.set_fast_training(on)

    def set_explain_target(self, target: str = "conv"):
        """Engine.set_explain_target on every GPU's engine (they share one network shape: all accept the target or the first refuses)."""
        for e in self.engines:
            e.set_explain_target(target)

    def saliency_overlays_classes_host(self, gray_u8: np.ndarray, classes=(0, 1), grad_mode="softmax_ce", standardise=True,
                                       want_saliency=False):
        """Engine.saliency_overlays_classes_host over the GPUs of the box (fp32 engines with ``keep_all_activations``): contiguous
        split, one host thread per GPU -> (cls, probs, logits, overlays [B,K,h,w,3], heat-maps [B,K,h,w,3], saliency [B,K,H,W] or
        None).  The arrays are the driver's pinned buffers: they are overwritten by the next call of the same shape (copy what must
        outlive it)."""
        g = _gray_batch(gray_u8)
        B, h, w = g.shape
        H, W, _ = self.spec.input_shape
        nc = self.spec.num_classes
        K, ci = _host_class_rows(classes, B, nc)
        specs = [((B,), torch.int32), ((B, nc), torch.float32), ((B, nc), torch.float32), ((B, K, h, w, 3), torch.uint8),
                 ((B, K, h, w, 3), torch.uint8)] + ([((B, K, H, W), torch.float32)] if want_saliency else [])
        cls, probs, logits, ov, hm, *rest = self._pinned(("saliency", B, K, h, w, bool(want_saliency)), specs)
        sal = rest[0] if want_saliency else None

        def work(e, s, t):
            cls[s:t], probs[s:t], logits[s:t], _, _, _ = e.saliency_overlays_classes_host(
                g[s:t], None if ci is None else ci[s:t], grad_mode, standardise, overlay_out=ov[s:t], heat_out=hm[s:t],
                saliency_out=None if sal is None else sal[s:t])

        self._fan_out(B, work)
        return cls, probs, logits, ov, hm, sal

    def close(self):
        for e in self.engines:
            e.close()
