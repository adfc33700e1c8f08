"""Drop-in for ``WebApplicationPrototype/ADCNNM.py``: the PyTorch CNN.

``CNNModel`` keeps the reference's constructor, parameter names (``convs.{i}.weight/bias``,
``fc.{0,3,6..}.weight/bias`` -- so ``load_state_dict(torch.load(...))`` of a reference checkpoint works),
``forward(x[B,H,W,C]) -> logits`` (ADCNNM.py:72-78) and ``load_trained_model`` (ADCNNM.py:155-202).
The modules only HOLD the parameters; ``forward`` runs in libbcad (Conv2d(padding=1) + leaky_relu(0.01) +
MaxPool2d(2), CHW flatten handled by permuting fc1's columns at load time, Linear + LeakyReLU(alpha)).
``forward`` returns logits without an autograd graph; training goes through ``train_model`` (forward, backward and
Adam all on the device, SURVEY 8 row f4).

``precision="auto"`` (default) picks the fastest path that is fp32-grade for the network's shape: the split-operand tensor-core
path ``fp16x3`` where it is covered (single-channel inputs, conv 32/64: logits within 2e-4 of float64), else the 16-bit tensor
path ``fp16`` (multi-channel inputs such as the deployed [64,256,256] model, app.py:584: logits within 1e-2), else the fp32
CUDA-core path.  A model in train mode (the reference's state after construction) runs ``forward`` with dropout, like
``nn.Dropout`` (ADCNNM.py:62): the multipliers are drawn with ``torch.rand`` on the device.
"""
from __future__ import annotations

import json

import numpy as np
import torch
import torch.nn as nn

from .engine import Engine, NetSpec


class CNNModel(nn.Module):
    def __init__(self, input_shape, num_classes, conv_layers=[(32, 3), (64, 3)], hidden_units=[256, 128],
                 dropout_rate=0.3, leaky_alpha=0.01, *, precision="auto", max_batch=64, device_index=0):
        super().__init__()
        H, W, C = input_shape                      # ADCNNM.py:42
        self._spec = NetSpec.torch_flavour((H, W, C), num_classes, conv_layers, hidden_units, leaky_alpha)
        self.convs = nn.ModuleList()
        self.pools = nn.ModuleList()
        in_channels = C
        for out_channels, ksize in conv_layers:
            self.convs.append(nn.Conv2d(in_channels, out_channels, ksize, padding=1))   # ADCNNM.py:48
            self.pools.append(nn.MaxPool2d(2))
            in_channels = out_channels
        _, flatten_size = self._spec.shapes()
        layers = []
        in_units = flatten_size
        for units in hidden_units:
            layers += [nn.Linear(in_units, units), nn.LeakyReLU(leaky_alpha), nn.Dropout(dropout_rate)]
            in_units = units
        layers.append(nn.Linear(in_units, num_classes))
        self.fc = nn.Sequential(*layers)
        self._precision, self._max_batch, self._device_index = precision, max_batch, device_index
        self._engine = None
        self._versions = None
        self._train_eng = None           # fp32 handle of the train-mode forward (dropout lives on the fp32 path)
        self._train_versions = None

    # ------------------------------------------------------------------ engine plumbing
    def _make_engine(self):
        if self._precision != "auto":
            return Engine(self._spec, precision=self._precision, max_batch=self._max_batch, device=self._device_index)
        for prec in ("fp16x3", "fp16"):
            try:
                return Engine(self._spec, precision=prec, max_batch=self._max_batch, device=self._device_index)
            except ValueError:
                continue
        return Engine(self._spec, precision="fp32", max_batch=self._max_batch, device=self._device_index)

    def _host_weights(self):
        conv_w = [c.weight.detach().cpu().numpy().transpose(0, 2, 3, 1) for c in self.convs]   # (F,C,k,k)->(F,k,k,C)
        conv_b = [c.bias.detach().cpu().numpy() for c in self.convs]
        lin = [m for m in self.fc if isinstance(m, nn.Linear)]
        return conv_w, conv_b, [l.weight.detach().cpu().numpy() for l in lin], [l.bias.detach().cpu().numpy() for l in lin]

    def _param_versions(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def sync_weights(self, force=True):
        ver = self._param_versions()
        if self._engine is None:
            self._engine = self._make_engine()
            force = True
        if force or ver != self._versions:
            self._engine.set_weights(*self._host_weights())
            self._versions = ver
        return self._engine

    @property
    def engine(self) -> Engine:
        return self.sync_weights(force=False)

    # ------------------------------------------------------------------ forward (ADCNNM.py:72-78)
    def forward(self, x):
        rates = [m.p for m in self.fc if isinstance(m, nn.Dropout)]
        if self.training and any(r > 0 for r in rates):
            logits = self._forward_train(x, rates)
        else:
            cls, probs, logits = self.engine.predict(x)
        return logits.to(x.device) if isinstance(x, torch.Tensor) else logits

    def _forward_train(self, x, rates, masks=None):
        """ADCNNM.py:72-78 with the module in train mode: nn.Dropout(p) after every hidden LeakyReLU (ADCNNM.py:62).  ``masks``
        [B, sum(hidden_units)] (0 or 1/(1-p)) may be injected; by default they are drawn with torch.rand on the device."""
        eng = self._engine
        if eng is None or eng.uses_tensor_path:
            ver = self._param_versions()
            if self._train_eng is None:
                self._train_eng = Engine(self._spec, precision="fp32", max_batch=self._max_batch, device=self._device_index)
                self._train_versions = None
            if ver != self._train_versions:
                self._train_eng.set_weights(*self._host_weights())
                self._train_versions = ver
            eng = self._train_eng
        else:
            eng = self.engine
        n = int(x.shape[0]) if hasattr(x, "shape") and len(x.shape) == 4 else 1
        units = list(self._spec.hidden_units)
        out = []
        for s0 in range(0, n, eng.max_batch):                   # masks are per forward of exactly B images
            s1 = min(n, s0 + eng.max_batch)
            if masks is None:
                mk = torch.cat([(torch.rand(s1 - s0, u, device=eng.tdev) >= r).float() / (1.0 - r) if r < 1.0 else
                                torch.zeros(s1 - s0, u, device=eng.tdev) for u, r in zip(units, rates)], dim=1)
            else:
                mk = torch.as_tensor(masks)[s0:s1]
            eng.set_dropout_masks(mk, mask_backward=True)
            try:
                out.append(eng.predict(x[s0:s1] if n > 1 or (hasattr(x, "shape") and len(x.shape) == 4) else x)[2])
            finally:
                eng.set_dropout_masks(None)
        return out[0] if len(out) == 1 else torch.cat(out, dim=0)

    # ------------------------------------------------------------------ batched entry points (new)
    def predict_batch(self, x):
        """-> (classes int64 [B], probs [B,nc]) -- torch.max / torch.softmax of app.py:589-593."""
        cls, probs, _ = self.engine.predict(x)
        return cls.long(), probs

    def predict_explain_batch(self, x, class_idx=None, grad_mode="logit", target="conv"):
        """-> (classes [B], logits [B,nc], Grad-CAM heatmaps fp32 [B,H,W]) on the GPU.
        ``target="conv"``: the last block's post-LeakyReLU map (default).  ``target="conv_preact"``: the ``nn.Conv2d`` module's own
        output -- what ``GradCAM(model, target_layers=[model.convs[-1]])`` of pytorch_grad_cam would hook on the reference model,
        whose activation is functional (ADCNNM.py:76); runs on an fp32 handle (it needs the dense pooled gradient)."""
        if target == "conv":
            cls, probs, logits, heat = self.engine.predict_explain(x, class_idx, grad_mode)
            return cls.long(), logits, heat
        if target != "conv_preact":
            raise ValueError(f"unknown target {target!r} (conv | conv_preact)")
        ver = self._param_versions()
        if self._train_eng is None:
            self._train_eng = Engine(self._spec, precision="fp32", max_batch=self._max_batch, device=self._device_index)
            self._train_versions = None
        if ver != self._train_versions:
            self._train_eng.set_weights(*self._host_weights())
            self._train_versions = ver
        eng = self._train_eng
        eng.set_explain_target("conv_preact")
        try:
            cls, probs, logits, heat = eng.predict_explain(x, class_idx, grad_mode)
        finally:
            eng.set_explain_target("conv")
        return cls.long(), logits, heat

    def predict_explain_classes_batch(self, x, classes=(0, 1), grad_mode="logit"):
        """Grad-CAM for several target classes per image from one forward (the dual-class call of app.py:649-657)
        -> (classes [B], logits [B,nc], heatmaps fp32 [B,K,H,W]) on the GPU.  ``classes``: a length-K sequence shared by the batch,
        a [B,K] array, or None = every class; ``heat[:, k]`` equals ``predict_explain_batch(x, classes[:, k])``'s heat-maps."""
        cls, probs, logits, heat = self.engine.predict_explain_classes(x, classes, grad_mode)
        return cls.long(), logits, heat


def _pull_into_modules(model, eng):
    """Weights of the training handle -> the nn.Parameters (state_dict layout); the inference handle re-uploads on its next use."""
    cw, cb, dw, db = eng.get_weights()
    lin = [m for m in model.fc if isinstance(m, nn.Linear)]
    with torch.no_grad():
        for c, w, b in zip(model.convs, cw, cb):
            c.weight.copy_(torch.from_numpy(np.ascontiguousarray(w.transpose(0, 3, 1, 2))))
            c.bias.copy_(torch.from_numpy(b))
        for l, w, b in zip(lin, dw, db):
            l.weight.copy_(torch.from_numpy(w))
            l.bias.copy_(torch.from_numpy(b))
    model._train_versions = model._param_versions()


def train_model(model, train_loader, test_loader, epochs=10, lr=0.001, device="cuda",
                save_path="trained_model/cnn_model_Advanced.pth", tensor_cores=False):
    """ADCNNM.py:86-153 on the device: Adam(lr) on the mean cross-entropy, nn.Dropout after every hidden layer, validation
    accuracy per epoch, best state_dict saved to ``save_path`` -> (history, best_val_acc).

    Forward, backward and the Adam update all run in libbcad; under an initialised torch.distributed group each rank
    feeds its own loader shard and the flat gradient is averaged with one bucketed all-reduce per step.
    ``tensor_cores=True`` (an addition to the reference's signature): the second conv block and the first dense layer run their
    forward / backward GEMMs on tcgen05 with split operands (``Engine.set_fast_training``; gradients agree with the fp32 kernels to
    ~1e-5 relative, a 64-image step takes 2.0 instead of 8.2 ms); ValueError when the network has no eligible block."""
    import os

    from .training import DataParallelTrainer
    first = next(iter(train_loader))[0]
    bs = int(first.shape[0])
    eng = model._train_eng
    if eng is None or not eng.keep_all_activations or eng.max_batch < bs:
        if eng is not None:
            eng.close()
        eng = model._train_eng = Engine(model._spec, precision="fp32", max_batch=max(bs, model._max_batch), keep_all_activations=True,
                                        device=model._device_index)
        model._train_versions = None
    if model._param_versions() != model._train_versions:
        eng.set_weights(*model._host_weights())
        model._train_versions = model._param_versions()
    eng.set_fast_training(bool(tensor_cores)) if tensor_cores else None
    trainer = DataParallelTrainer(eng, opt="adam", lr=lr)
    rates = [m.p for m in model.fc if isinstance(m, nn.Dropout)]
    units = list(model._spec.hidden_units)
    best_val_acc, history = 0.0, []
    for epoch in range(epochs):
        model.train()
        total_loss, correct, total = 0.0, 0, 0
        for X, y in train_loader:
            n = int(X.shape[0])
            if any(r > 0 for r in rates):
                mk = torch.cat([(torch.rand(n, u, device=eng.tdev) >= r).float() / (1.0 - r) for u, r in zip(units, rates)], dim=1)
                eng.set_dropout_masks(mk, mask_backward=True)
            try:
                loss = trainer.step(X, y)
                cls = trainer.last_classes
            finally:
                eng.set_dropout_masks(None)
            total_loss += float(loss.mean())
            correct += int((cls.cpu() == torch.as_tensor(y).cpu().int()).sum())
            total += n
        train_acc = correct / max(1, total)
        avg_loss = total_loss / max(1, len(train_loader))
        print(f"[EPOCH {epoch+1}] Loss={avg_loss:.4f}, Acc={train_acc:.4f}")
        model.eval()
        val_correct, val_total = 0, 0
        for X, y in test_loader:
            cls, _, _ = eng.predict(X)
            val_correct += int((cls.cpu() == torch.as_tensor(y).cpu().int()).sum())
            val_total += int(X.shape[0])
        val_acc = val_correct / max(1, val_total)
        print(f"[VAL] Acc={val_acc:.4f}")
        history.append({"epoch": epoch + 1, "loss": avg_loss, "val_acc": val_acc})
        if val_acc > best_val_acc:
            best_val_acc = val_acc
            _pull_into_modules(model, eng)
            d = os.path.dirname(save_path)
            if d:
                os.makedirs(d, exist_ok=True)
            torch.save(model.state_dict(), save_path)
            print(f" Saved best model at epoch {epoch+1} with val_acc={val_acc:.4f}")
    _pull_into_modules(model, eng)
    return history, best_val_acc


def load_trained_model(json_path, weight_path, **engine_kw):
    """ADCNNM.py:155-202: JSON config + ``.pth`` state_dict -> eval-mode model (same exceptions)."""
    with open(json_path, "r") as f:
        config = json.load(f)
    input_shape = tuple(config["dataset"]["input_shape"])
    num_classes = config["dataset"]["num_classes"]
    conv_layers = [tuple(layer) for layer in config["model"]["conv_layers"]]
    hidden_units = config["model"]["hidden_units"]
    dropout_rate = config["model"]["dropout_rate"]
    model = CNNModel(input_shape=input_shape, num_classes=num_classes, conv_layers=conv_layers,
                     hidden_units=hidden_units, dropout_rate=dropout_rate, **engine_kw)
    try:
        state_dict = torch.load(weight_path, map_location="cpu")
        model.load_state_dict(state_dict)
        model.eval()
        model.sync_weights()
        print(f" Model loaded successfully from '{weight_path}' on device: cuda")
    except FileNotFoundError:
        raise FileNotFoundError(f" Could not find weight file at '{weight_path}'")
    except Exception as e:
        raise RuntimeError(f" Failed to load model weights: {e}")
    return model
