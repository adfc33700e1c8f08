"""Drop-in for ``Classes/CNNModel.py`` (== WebApplicationPrototype/CNNModel.py, CNNM.py): the NumPy CNN.

Same constructor, ``layers`` list-of-dicts, ``forward`` / ``predict`` / ``load_weights`` /
``save_model`` as the reference (Classes/CNNModel.py:30-60, 67-198, 524-555) -- but ``forward`` runs
on the GPU through libbcad instead of Python loops.  None of the reference's import-time side effects
(stdout hijack :28, log file :10, Windows-path weight load :587) are reproduced.

Added batched entry points the reference only hints at (``Classes/Model.py:43 predict_batch``):
``predict_batch(X)`` and ``predict_explain_batch(X, class_idx=None)``.
"""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from . import _lib
from .engine import Engine, NetSpec


class _Lazy:
    __slots__ = ("fn",)

    def __init__(self, fn):
        self.fn = fn


class _Layer(dict):
    """layer dict whose cached activations are fetched from the device on first access."""

    def __getitem__(self, key):
        v = dict.__getitem__(self, key)
        if isinstance(v, _Lazy):
            v = v.fn()
            dict.__setitem__(self, key, v)
        return v

    def get(self, key, default=None):
        return self[key] if key in self else default


def load_weights(cls, path="trained_model/cnn_model.npz"):
    """Classes/CNNModel.py:30-60: ``.npz`` with a JSON ``config`` and ``W{i}``/``b{i}`` keyed by layer index."""
    data = np.load(path, allow_pickle=True)
    config = json.loads(str(data["config"]))
    model = cls(
        input_shape=tuple(config["input_shape"]),
        num_classes=config["num_classes"],
        conv_layers=config["conv_layers"],
        hidden_units=config["hidden_units"],
        dropout_rate=config["dropout_rate"],
        leaky_alpha=config.get("leaky_alpha", 0.01),
    )
    for i, layer in enumerate(model.layers):
        if layer["type"] == "conv":
            layer["filters"] = data[f"W{i}"]
            layer["biases"] = data[f"b{i}"]
        elif layer["type"] in ["dense", "output"]:
            layer["weights"] = data[f"W{i}"]
            layer["biases"] = data[f"b{i}"]
    print(f"[INFO] Model loaded from {path}")
    return model


class CNNModel:
    """Two handles behind one model (created on first use):

    * the COMPAT handle -- fp32 CUDA-core path, every activation kept -- serves ``forward`` / ``predict`` (single sample, with the
      reference's ``layers[*]`` caches), ``compute_backprops_for_explainability`` and training;
    * the FAST handle serves the batched entry points ``predict_batch`` / ``predict_explain_batch``: ``precision="auto"``
      (default) takes the fp32-grade split-operand tensor-core path (``fp16x3``) where the network's shape allows and the
      compat handle otherwise; ``"fp32"`` forces the compat handle, ``"fp16x3"`` raises if the shape is not covered."""

    def __init__(self, input_shape, num_classes, conv_layers=[(8, 3), (16, 3)], hidden_units=[128, 64],
                 dropout_rate=0.3, leaky_alpha=0.01, *, precision="auto", max_batch=32, device=0,
                 keep_all_activations=True):
        self.input_shape = input_shape
        self.num_classes = num_classes
        self.conv_layers_config = conv_layers
        self.hidden_units = hidden_units
        self.dropout_rate = dropout_rate
        self.leaky_alpha = leaky_alpha
        self.layers = []
        self.epoch_accuracy = []
        self._precision, self._max_batch, self._device = precision, max_batch, device
        self._keep_all = keep_all_activations
        self._engine = None             # compat handle
        self._weights_key = None
        self._fast = None               # fast handle (None: not created yet; the compat handle itself when the shape is not covered)
        self._fast_key = None
        self._gen = 0                   # forward() generation: the lazy layer caches and the explain backward check it
        self._last_x = None
        self._last_masks = None
        self._dirty = False             # a training step moved the compat handle's weights ahead of ``layers`` (until _pull_weights)
        self._build_model()

    # ------------------------------------------------------------------ build (Classes/CNNModel.py:88-157)
    def _build_model(self):
        in_shape = tuple(self.input_shape)
        for num_filters, ksize in self.conv_layers_config:
            filters = np.random.randn(num_filters, ksize, ksize, in_shape[2]) * np.sqrt(2.0 / (ksize * ksize * in_shape[2]))
            out_h, out_w = in_shape[0] - ksize + 1, in_shape[1] - ksize + 1
            self.layers.append(_Layer({
                "type": "conv", "filters": filters, "biases": np.zeros(num_filters),
                "input_shape": in_shape, "output_shape": (out_h, out_w, num_filters),
                "ksize": ksize, "num_filters": num_filters, "input": None, "output": None}))
            in_shape = (out_h, out_w, num_filters)
            pool_h, pool_w = in_shape[0] // 2, in_shape[1] // 2
            self.layers.append(_Layer({
                "type": "pool", "input_shape": in_shape, "output_shape": (pool_h, pool_w, in_shape[2]),
                "input": None, "output": None, "switches": None}))
            in_shape = (pool_h, pool_w, in_shape[2])
        prev_units = int(np.prod(in_shape))
        for units in self.hidden_units:
            limit = np.sqrt(6.0 / (prev_units + units))
            self.layers.append(_Layer({
                "type": "dense", "weights": np.random.uniform(-limit, limit, (units, prev_units)),
                "biases": np.zeros(units), "input_shape": (prev_units,), "input": None, "z": None,
                "output_shape": (units,)}))
            prev_units = units
        limit = np.sqrt(6.0 / (prev_units + self.num_classes))
        self.layers.append(_Layer({
            "type": "output", "weights": np.random.uniform(-limit, limit, (self.num_classes, prev_units)),
            "biases": np.zeros(self.num_classes), "input_shape": (prev_units,), "input": None, "z": None,
            "output_shape": (self.num_classes,)}))

    # ------------------------------------------------------------------ engine plumbing
    def _spec(self) -> NetSpec:
        return NetSpec.numpy_flavour(self.input_shape, self.num_classes, self.conv_layers_config,
                                     self.hidden_units, self.leaky_alpha)

    def _conv_layers(self):
        return [l for l in self.layers if l["type"] == "conv"]

    def _dense_layers(self):
        return [l for l in self.layers if l["type"] in ("dense", "output")]

    def _key(self):
        convs, denses = self._conv_layers(), self._dense_layers()
        return tuple(id(dict.__getitem__(l, k)) for l in convs for k in ("filters", "biases")) + \
            tuple(id(dict.__getitem__(l, k)) for l in denses for k in ("weights", "biases"))

    def _upload(self, eng):
        convs, denses = self._conv_layers(), self._dense_layers()
        eng.set_weights([l["filters"] for l in convs], [l["biases"] for l in convs],
                        [l["weights"] for l in denses], [l["biases"] for l in denses])

    def sync_weights(self, force=True):
        """Upload ``layers[*]['filters'|'weights'|'biases']`` to the device.  Called automatically when a
        weight array OBJECT is replaced (as ``load_weights`` does); call it yourself after in-place edits."""
        key = self._key()
        if self._engine is None:
            self._engine = Engine(self._spec(), precision="fp32", max_batch=self._max_batch,
                                  keep_all_activations=self._keep_all, device=self._device)
            force = True
        if force or key != self._weights_key:
            self._upload(self._engine)
            self._weights_key = key
            if force:
                self._fast_key = None
        return self._engine

    @property
    def engine(self) -> Engine:
        """The compat handle (fp32, every activation kept)."""
        return self.sync_weights(force=False)

    @property
    def fast_engine(self) -> Engine:
        """The handle of the batched entry points (see the class docstring)."""
        if self._fast is None:
            if self._precision in ("auto", "fp16x3"):
                try:
                    self._fast = Engine(self._spec(), precision="fp16x3", max_batch=self._max_batch, device=self._device)
                except ValueError:
                    if self._precision != "auto":
                        raise
            if self._fast is None:
                self._fast = self.engine
        if self._fast is self._engine:
            return self.engine
        key = self._key()
        if key != self._fast_key:
            self._upload(self._fast)
            self._fast_key = key
        return self._fast

    # ------------------------------------------------------------------ forward / predict
    def forward(self, x, training=True):
        """Classes/CNNModel.py:162-198 (single sample (H,W,C) -> probs (num_classes,) float64).

        Caches ``layer['input'|'output'|'switches'|'z']`` like the reference (fetched lazily from the device).
        ``training=True`` (the reference's default) applies inverted dropout after every hidden dense layer (:186-188); the
        multipliers are drawn from the global ``np.random`` stream exactly as the reference draws them (one ``rand(units)`` per
        hidden layer, in layer order), so a seeded call follows the reference's random numbers."""
        x = np.asarray(x)
        eng = self.engine
        masks = None
        if training and self.dropout_rate > 0.0 and len(self.hidden_units) > 0:
            masks = self._draw_dropout(1)
            eng.set_dropout_masks(masks, mask_backward=False)
        try:
            cls, probs, logits = eng.predict(x[None].astype(np.float32))
        finally:
            if masks is not None:
                eng.set_dropout_masks(None)
        self._gen += 1
        eng.cache_tag = (id(self), self._gen)
        self._last_x, self._last_masks = np.array(x, dtype=np.float32), masks
        self._fill_caches(x)
        self._last_logits = logits
        return probs[0].double().cpu().numpy()

    def _cache_ready(self):
        """The compat handle still holds the activations of THIS model's latest forward(); anything run on it since (predict,
        a batched call, another model sharing nothing but the device...) has reset the tag -> the forward is repeated."""
        eng = self.engine
        if self._last_x is None:
            raise RuntimeError("no forward() has been run on this model yet")
        if eng.cache_tag != (id(self), self._gen):
            if self._last_masks is not None:
                eng.set_dropout_masks(self._last_masks, mask_backward=False)
            try:
                eng.predict(self._last_x[None])
            finally:
                if self._last_masks is not None:
                    eng.set_dropout_masks(None)
            eng.cache_tag = (id(self), self._gen)
        return eng

    def _fill_caches(self, x):
        gen = self._gen
        ci = di = 0
        for idx, layer in enumerate(self.layers):
            t = layer["type"]
            if t == "conv":
                layer["input"] = x if ci == 0 else _Lazy(self._getter(_lib.T_POOL_OUT, ci - 1, self.layers[idx - 1]["output_shape"], gen))
                layer["output"] = _Lazy(self._getter(_lib.T_CONV_OUT, ci, layer["output_shape"], gen))
            elif t == "pool":
                layer["input"] = _Lazy(self._getter(_lib.T_CONV_OUT, ci, layer["input_shape"], gen))
                layer["output"] = _Lazy(self._getter(_lib.T_POOL_OUT, ci, layer["output_shape"], gen))
                layer["switches"] = _Lazy(self._switch_getter(idx))
                ci += 1
            else:
                layer["z"] = _Lazy(self._getter(_lib.T_DENSE_Z, di, layer["output_shape"], gen))
                layer["input"] = _Lazy(self._dense_input_getter(idx, di))
                di += 1

    def _getter(self, kind, index, shape, gen):
        def fn():
            if gen != self._gen:
                raise RuntimeError("this layer cache belongs to an earlier forward(); read model.layers[...] again")
            return self._cache_ready().get_tensor(kind, index, 1)[0].double().cpu().numpy().reshape(shape)
        return fn

    def _switch_getter(self, idx):
        def fn():                                              # Classes/CNNModel.py:260 (every tie marked)
            x, p = self.layers[idx]["input"], self.layers[idx]["output"]
            h2, w2 = p.shape[0], p.shape[1]
            sw = np.zeros_like(x, dtype=bool)
            up = np.repeat(np.repeat(p, 2, axis=0), 2, axis=1)
            sw[:2 * h2, :2 * w2] = x[:2 * h2, :2 * w2] == up
            return sw
        return fn

    def _dense_input_getter(self, idx, di):
        def fn():                                              # flat.copy() (Classes/CNNModel.py:179,192)
            prev = self.layers[idx - 1]
            if prev["type"] == "pool":
                return prev["output"].flatten()
            z = prev["z"]
            h = np.where(z > 0, z, self.leaky_alpha * z)
            if self._last_masks is not None:                  # training forward: the dropped activations (Classes/CNNModel.py:186-188)
                off = sum(self.hidden_units[:di - 1])
                h = h * self._last_masks[0, off:off + h.shape[0]].astype(np.float64)
            return h
        return fn

    def _softmax(self, z):
        """Classes/CNNModel.py:203-212 (host helper kept for explainability-style callers)."""
        z = np.array(z, dtype=np.float64)
        z = np.clip(z, -50.0, 50.0)
        z = z - np.max(z)
        exps = np.exp(z)
        s = np.sum(exps)
        if s == 0:
            return np.ones_like(z) / len(z)
        return exps / (s + 1e-12)

    def predict(self, X):
        """Classes/CNNModel.py:524-526: (argmax, probs)."""
        probs = self.forward(X, training=False)
        return np.argmax(probs), probs

    # ------------------------------------------------------------------ batched entry points (new)
    def _batch_engine(self):
        # between a training step and the next _pull_weights() only the compat handle has the current weights
        return self.engine if self._dirty else self.fast_engine

    def predict_batch(self, X):
        """X [B,H,W,C] -> (classes int64 [B], probs float32 [B,nc])."""
        cls, probs, _ = self._batch_engine().predict(np.asarray(X, dtype=np.float32))
        return cls.cpu().numpy().astype(np.int64), probs.cpu().numpy()

    def predict_explain_batch(self, X, class_idx=None, grad_mode="softmax_ce"):
        """X [B,H,W,C] -> (classes [B], probs [B,nc], Grad-CAM heatmaps float32 [B,H,W] in [0,1])."""
        X = np.asarray(X)
        if X.dtype != np.uint8:
            X = np.asarray(X, dtype=np.float32)
        cls, probs, _, heat = self._batch_engine().predict_explain_host(X, class_idx, grad_mode)
        return cls.astype(np.int64), probs, heat

    def predict_explain_classes_batch(self, X, classes=(0, 1), grad_mode="softmax_ce"):
        """X [B,H,W,C] -> (classes [B], probs [B,nc], Grad-CAM heatmaps float32 [B,K,H,W] in [0,1]) for K target classes per image
        from one forward.  ``classes``: a length-K sequence shared by the batch, a [B,K] array, or None = every class."""
        X = np.asarray(X)
        if X.dtype == np.uint8:
            X = X.astype(np.float32) / np.float32(255.0)
        cls, probs, _, heat = self._batch_engine().predict_explain_classes(np.asarray(X, dtype=np.float32), classes, grad_mode)
        return cls.cpu().numpy().astype(np.int64), probs.cpu().numpy(), heat.cpu().numpy()

    # ------------------------------------------------------------------ persistence (Classes/CNNModel.py:530-555)
    def save_model(self, path="trained_model/cnn_model.npz"):
        d = os.path.dirname(path)
        if d:
            os.makedirs(d, exist_ok=True)
        config = {"input_shape": list(self.input_shape), "num_classes": self.num_classes,
                  "conv_layers": [list(c) for c in self.conv_layers_config], "hidden_units": list(self.hidden_units),
                  "dropout_rate": self.dropout_rate, "leaky_alpha": self.leaky_alpha}
        weights = {}
        for i, layer in enumerate(self.layers):
            if layer["type"] == "conv":
                weights[f"W{i}"], weights[f"b{i}"] = layer["filters"], layer["biases"]
            elif layer["type"] in ["dense", "output"]:
                weights[f"W{i}"], weights[f"b{i}"] = layer["weights"], layer["biases"]
        np.savez(path, config=json.dumps(config), **weights)
        print(f"[INFO] Model saved to {path}")

    # ------------------------------------------------------------------ training (Classes/CNNModel.py:399-512)
    def _training_engine(self, batch_size):
        """The handle the training step runs on: fp32, every activation kept, max_batch >= batch_size."""
        eng = self._engine
        if eng is None or not eng.keep_all_activations or eng.max_batch < batch_size:
            if eng is not None:
                if self._fast is eng:
                    self._fast = None
                eng.close()
            self._engine, self._keep_all = None, True
            self._max_batch = max(self._max_batch, int(batch_size))
        return self.sync_weights(force=False)

    def _pull_weights(self):
        """Device weights -> ``layers[*]`` (float64 arrays like the reference's), without triggering a re-upload."""
        cw, cb, dw, db = self._engine.get_weights()
        for l, w, b in zip(self._conv_layers(), cw, cb):
            l["filters"], l["biases"] = w.astype(np.float64), b.astype(np.float64)
        for l, w, b in zip(self._dense_layers(), dw, db):
            l["weights"], l["biases"] = w.astype(np.float64), b.astype(np.float64)
        self._weights_key = self._key()
        self._dirty = False

    def _draw_dropout(self, n_samples):
        """The multipliers the reference would draw for n samples: np.random.rand(units) per hidden layer, sample by
        sample (Classes/CNNModel.py:186-188) -- same global stream, same order."""
        rows = []
        for _ in range(n_samples):
            rows.append(np.concatenate([(np.random.rand(u) > self.dropout_rate).astype(np.float32) / (1.0 - self.dropout_rate)
                                        for u in self.hidden_units]))
        return np.stack(rows)

    def train_batch(self, X_batch, y_batch, lr):
        """One mini-batch of ``train``: averaged gradients (:438-464) + ``_apply_grads`` (:372-394) on the device.
        Under an initialised torch.distributed group the gradients are averaged over the ranks first.  -> summed loss."""
        from .training import allreduce_mean_
        X_batch = np.asarray(X_batch, dtype=np.float32)
        y_batch = np.asarray(y_batch)
        labels = y_batch.argmax(axis=1) if y_batch.ndim == 2 else y_batch
        eng = self._training_engine(len(X_batch))
        drop = self.dropout_rate > 0.0 and len(self.hidden_units) > 0
        if drop:
            eng.set_dropout_masks(self._draw_dropout(len(X_batch)), mask_backward=False)
        try:
            eng.predict(X_batch)
            grads, loss = eng.train_backward(X_batch, labels)
        finally:
            if drop:
                eng.set_dropout_masks(None)
        allreduce_mean_(grads)
        eng.apply_update(grads, "sgd_clip", lr=lr, max_norm=5.0)
        self._dirty = True
        return float(loss.sum())

    def train(self, X, y_onehot, X_test, y_test, epochs=10, lr=0.01, batch_size=8, eval_every_batch=True):
        """Same loop as the reference: shuffle per epoch (np.random), one clipped-SGD update per mini-batch of averaged
        gradients, test accuracy after every batch, lr *= 0.98 per epoch, best-accuracy weights restored at the end.
        ``y_onehot`` one-hot rows (the reference's cross_entropy / probs - y_true)."""
        X, y_onehot = np.asarray(X), np.asarray(y_onehot)
        dataset_size = len(X)
        best_acc, best_weights = 0.0, None
        print("[Training Params] :")
        print("       Learning Rate:", lr)
        print("       Drop Out Rate:", self.dropout_rate)
        print("       Num Epochs:", epochs)
        print("       Batch size:", batch_size)
        self._training_engine(batch_size)
        for epoch in range(epochs):
            indices = np.arange(dataset_size)
            np.random.shuffle(indices)
            X_shuf, y_shuf = X[indices], y_onehot[indices]
            accuracy, total_loss = 0, 0.0
            for i in range(0, dataset_size, batch_size):
                xb, yb = X_shuf[i:i + batch_size], y_shuf[i:i + batch_size]
                batch_loss = self.train_batch(xb, yb, lr)
                total_loss += batch_loss
                if eval_every_batch or i + batch_size >= dataset_size:
                    accuracy = self.get_training_metrics(X_test, y_test, verbose=False)
                print(f"[EPOCH {epoch+1}/{epochs}, BATCH {i//batch_size+1}] BatchLoss={batch_loss/ max(1, len(xb)):.4f}  Accuracy={accuracy}")
            self._pull_weights()
            print(f"\n[EPOCH {epoch+1}] Loss={total_loss / dataset_size:.4f}, Acc={accuracy:.4f}")
            self.epoch_accuracy.append(accuracy)
            if accuracy > best_acc:
                best_acc = accuracy
                best_weights = [{k: np.copy(dict.__getitem__(l, k)) for k in ("weights", "biases", "filters") if k in l}
                                for l in self.layers]
            lr *= 0.98
        print(f"[TRAIN] Best accuracy: {best_acc:.4f}")
        if best_weights is not None:
            for layer, saved in zip(self.layers, best_weights):
                for key in saved:
                    layer[key] = saved[key]
            self.sync_weights(force=True)

    def get_training_metrics(self, X_test, Y_test, verbose=True):
        """Accuracy of ``predict`` over a test set (Classes/CNNModel.py:560-585; the reference reads undefined globals for
        the labels -- here they come from ``Y_test``: one-hot rows or integer labels)."""
        Y_test = np.asarray(Y_test)
        y_true = Y_test.argmax(axis=1) if Y_test.ndim == 2 else Y_test
        y_pred, _ = self.predict_batch(np.asarray(X_test, dtype=np.float32))
        y_pred = np.asarray(y_pred)
        acc = float((y_pred == y_true).mean())
        if verbose:
            print(f"\n[Test Accuracy] {acc:.4f}")
            cm = np.zeros((self.num_classes, self.num_classes), dtype=np.int64)
            np.add.at(cm, (y_true, y_pred), 1)
            print("\nConfusion Matrix:")
            print(cm)
        return acc
