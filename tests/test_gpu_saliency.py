"""Input-gradient saliency for several target classes per image from one forward (bcad_predict_saliency_classes /
Engine.predict_saliency_classes) and its overlay (bcad_saliency_overlay).

Every comparison of the gradients is anchored to ``explain_backward(want_input=True)`` after ``predict`` on the SAME handle, so both sides
read the same cached forward: pool switches and LeakyReLU' branches are identical by construction, and only the summation order (fp32
kernels) or the split-operand products (fast training) differ."""
import ctypes as C

import numpy as np
import pytest
import torch

from util import engine_from, load_numpy_golden, ocnn

pytestmark = pytest.mark.gpu


def _norm(s):
    """explainability.py:72-73 per image: (s - min) / (max - min + 1e-8) over the last two axes."""
    mn = s.min(axis=(-2, -1), keepdims=True)
    mx = s.max(axis=(-2, -1), keepdims=True)
    return (s - mn) / (mx - mn + 1e-8)


def _cols(classes, B, K):
    if classes is None:
        return np.tile(np.arange(K, dtype=np.int32), (B, 1))
    c = np.asarray(classes, dtype=np.int32)
    return np.ascontiguousarray(np.broadcast_to(c, (B, K)) if c.ndim == 1 else c)


def _anchor(eng, x, cols, mode="softmax_ce"):
    """d_input [B,K,H,W,C] of predict + explain_backward, chunk by chunk, on the same handle."""
    B, K = cols.shape
    out = []
    for b0 in range(0, B, eng.max_batch):
        xb = x[b0:b0 + eng.max_batch]
        n = xb.shape[0]
        eng.predict(xb)
        per_k = []
        for k in range(K):
            _, d_in = eng.explain_backward(n, cols[b0:b0 + n, k].copy(), mode, want_input=True)
            per_k.append(d_in.cpu().numpy())
        out.append(np.stack(per_k, axis=1))
    return np.concatenate(out, axis=0)


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. reference fixtures (generic first blocks: 2-channel inputs, ties, k = 5): the conv_fp32 + saliency_absmax route
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["ref_numpy_small", "ref_numpy_odd", "ref_numpy_ties", "ref_numpy_k5"])
def test_reference_fixtures_inside_a_chunked_batch(name):
    g, cfg, p, _, _ = load_numpy_golden(name)
    shape = tuple(cfg.input_shape)
    x = ocnn.synth_images(7, shape, seed=3).astype(np.float32)
    at = 5                                                       # the fixture image, in the second chunk
    x[at] = g["x"].astype(np.float32)
    eng = engine_from(cfg, p, precision="fp32", max_batch=4, keep_all_activations=True)
    cls, probs, logits, sal, d_in = eng.predict_saliency_classes(x, (0, 1), "softmax_ce", want_d_input=True)
    assert sal.shape == (7, 2) + shape[:2] and d_in.shape == (7, 2) + shape
    for c in (0, 1):
        np.testing.assert_allclose(d_in[at, c].cpu().numpy(), g[f"d_input_c{c}"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(sal[at, c].cpu().numpy(), g[f"saliency_c{c}"], rtol=0, atol=1e-4)
    assert int(cls[at]) == int(g["pred_class"])
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. same-handle anchor on the fused first-block kernel's shape (1 -> 32 -> 64, 3x3), chunked and ragged
# ---------------------------------------------------------------------------------------------------------------------------------
FLAVOURS = ["torch", "numpy"]


def _net(kind, shape, hidden, nc=2, seed=7):
    mk = ocnn.NetConfig.torch_flavour if kind == "torch" else ocnn.NetConfig.numpy_flavour
    cfg = mk(shape, nc, [(32, 3), (64, 3)], hidden, 0.01)
    p = ocnn.init_params(cfg, seed=seed, bias_std=0.05)
    return cfg, p


def _images(kind, B, shape, seed):
    return ocnn.synth_images(B, shape, seed=seed, kind="gauss" if kind == "torch" else "mammo")


@pytest.mark.parametrize("kind", FLAVOURS)
@pytest.mark.parametrize("shape,hidden", [((67, 61, 1), [64, 32]), ((256, 256, 1), [256, 128])])
@pytest.mark.parametrize("fast", [False, True])
def test_same_handle_anchor(kind, shape, hidden, fast):
    cfg, p = _net(kind, shape, hidden)
    B = 70
    x = _images(kind, B, shape, seed=11)
    eng = engine_from(cfg, p, precision="fp32", max_batch=32, keep_all_activations=True)
    if fast:
        eng.set_fast_training(True)
    cols = _cols((0, 1), B, 2)
    cls, probs, logits, sal, d_in = eng.predict_saliency_classes(x, (0, 1), "softmax_ce", want_d_input=True)
    ref = _anchor(eng, x, cols)
    d_tol, s_tol = (1e-3, 2e-3) if fast else (1e-5, 1e-4)
    got = d_in.cpu().numpy()
    for b in range(B):
        for k in range(2):
            scale = max(1e-30, np.abs(ref[b, k]).max())
            err = np.abs(got[b, k] - ref[b, k]).max()
            assert err <= d_tol * scale, f"image {b} class {k}: d_input err {err:.3e} vs max {scale:.3e}"
    s_ref = _norm(np.abs(ref).max(axis=-1))
    s_err = np.abs(sal.cpu().numpy() - s_ref).max()
    assert s_err <= s_tol, f"saliency err {s_err:.3e}"
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. multi-class contract
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fast", [False, True])
def test_classes_equal_single_class_calls_and_predict(fast):
    shape, nc, B = (64, 64, 1), 3, 70
    cfg, p = _net("torch", shape, [64, 32], nc=nc)
    x = torch.from_numpy(_images("torch", B, shape, seed=5)).cuda()
    eng = engine_from(cfg, p, precision="fp32", max_batch=32, keep_all_activations=True)
    if fast:
        eng.set_fast_training(True)
    rng = np.random.default_rng(1)
    for classes in [(2, 0), rng.integers(0, nc, size=(B, 3)), None, rng.integers(0, nc, size=(B, 1)), rng.integers(0, nc, size=(B, 8))]:
        cls, probs, logits, sal, d_in = eng.predict_saliency_classes(x, classes, "softmax_ce", want_d_input=True)
        K = sal.shape[1]
        cols = _cols(classes, B, K)
        c0, p0, l0 = eng.predict(x)
        assert torch.equal(cls, c0) and torch.equal(probs, p0) and torch.equal(logits, l0)
        for k in range(K):
            _, _, _, s1, d1 = eng.predict_saliency_classes(x, cols[:, k:k + 1].copy(), "softmax_ce", want_d_input=True)
            assert torch.equal(sal[:, k], s1[:, 0]), f"K={K} column {k}: saliency differs"
            assert torch.equal(d_in[:, k], d1[:, 0]), f"K={K} column {k}: d_input differs"
    a = eng.predict_saliency_classes(x, (0, 1), "logit", want_d_input=True)
    b = eng.predict_saliency_classes(x, (0, 1), "logit", want_d_input=True)
    assert all(torch.equal(u, v) for u, v in zip(a, b)), "two identical calls differ"
    # new weights take effect (tensor-core dgrad weight images included): same results as a fresh handle created with them
    _, p2 = _net("torch", shape, [64, 32], nc=nc, seed=99)
    eng.set_weights(p2.conv_w, p2.conv_b, p2.dense_w, p2.dense_b)
    fresh = engine_from(cfg, p2, precision="fp32", max_batch=32, keep_all_activations=True)
    if fast:
        fresh.set_fast_training(True)
    got = eng.predict_saliency_classes(x, (0, 1), "softmax_ce", want_d_input=True)
    want = fresh.predict_saliency_classes(x, (0, 1), "softmax_ce", want_d_input=True)
    assert not torch.equal(got[4], b[4]) and not torch.equal(got[3], a[3])
    assert all(torch.equal(u, v) for u, v in zip(got, want)), "weights set between calls did not take effect"
    eng.close()
    fresh.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 4. overlay: byte-identical to cv2 on the device's own saliency
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("base_c", [1, 3])
def test_overlay_matches_cv2(base_c):
    import cv2
    from bcad_b200 import engine as E
    shape, B = (67, 61, 1), 6
    cfg, p = _net("numpy", shape, [32, 16])
    eng = engine_from(cfg, p, precision="fp32", max_batch=8, keep_all_activations=True)
    _, _, _, sal, _ = eng.predict_saliency_classes(_images("numpy", B, shape, seed=2), (0, 1))
    base = np.random.default_rng(base_c).integers(0, 256, size=(B,) + shape[:2] + (base_c,), dtype=np.uint8)
    ov, heat = E.saliency_overlay(base, sal)
    ov, heat, s = ov.cpu().numpy(), heat.cpu().numpy(), sal.cpu().numpy()
    assert ov.shape == heat.shape == (B, 2) + shape[:2] + (3,)
    for b in range(B):
        base3 = base[b] if base_c == 3 else np.repeat(base[b], 3, axis=-1)
        for k in range(2):
            want_heat = cv2.applyColorMap(np.uint8(s[b, k] * 255), cv2.COLORMAP_JET)
            assert np.array_equal(heat[b, k], want_heat)
            assert np.array_equal(ov[b, k], cv2.addWeighted(base3, 0.5, want_heat, 0.5, 0))
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. mirrors
# ---------------------------------------------------------------------------------------------------------------------------------
def test_dual_class_overlays_batch_matches_the_single_image_mirror(tmp_path):
    from bcad_b200.CNNModel import CNNModel
    from bcad_b200 import explainability as E
    shape, B = (67, 61, 1), 12
    np.random.seed(4)
    m = CNNModel(shape, 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[32, 16], max_batch=8)
    X = (3.0 * _images("numpy", B, shape, seed=8)).astype(np.float32)
    cls, probs, sal, ov, heat = E.generate_dual_class_overlays_batch(m, X, [0, 1])
    assert sal.shape == (B, 2) + shape[:2] and ov.shape == heat.shape == (B, 2) + shape[:2] + (3,) and ov.dtype == np.uint8
    for b in range(B):
        out = E.generate_dual_class_overlays(m, X[b], [0, 1], str(tmp_path / f"img{b}"))
        p1 = m.forward(X[b], training=False)
        assert int(cls[b]) == int(np.argmax(p1))
        for k in (0, 1):
            o1, h1 = out[k]
            _, d_input, _ = E.compute_backprops_for_explainability(m, np.eye(2, dtype=np.float32)[k], want_weight_grads=False)
            s1 = E.saliency_map(d_input)
            assert np.abs(sal[b, k] - s1).max() <= 2e-3
            i_batch, i_ref = np.uint8(sal[b, k] * 255).astype(int), np.uint8(s1 * 255).astype(int)
            assert np.abs(i_batch - i_ref).max() <= 1
            same = i_batch == i_ref
            assert np.array_equal(heat[b, k][same], h1[same]) and np.array_equal(ov[b, k][same], o1[same])
    c2, p2, s2 = m.predict_saliency_classes_batch(X, (0, 1))
    c3, p3, _, s3, _ = m.saliency_engine.predict_saliency_classes(X, (0, 1), "softmax_ce")
    assert np.array_equal(c2, c3.cpu().numpy()) and np.array_equal(p2, p3.cpu().numpy()) and np.array_equal(s2, s3.cpu().numpy())
    assert np.array_equal(s2, sal)


def test_torch_mirror_saliency_batch_returns_the_engine_call():
    from bcad_b200 import ADCNNM as A
    shape, B = (64, 48, 1), 20
    cfg, p = _net("torch", shape, [32, 16], seed=6)
    model = A.CNNModel(shape, 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[32, 16], max_batch=16).eval()
    model.load_state_dict(ocnn.params_to_state_dict(cfg, p))
    x = torch.from_numpy(_images("torch", B, shape, seed=9)).cuda()
    cls, logits, sal = model.predict_saliency_classes_batch(x, (1, 0))
    c1, p1, l1, s1, _ = model.saliency_engine.predict_saliency_classes(x, (1, 0), "logit")
    assert torch.equal(cls, c1.long()) and torch.equal(logits, l1) and torch.equal(sal, s1)
    with torch.no_grad():                                        # a weight change is picked up
        model.convs[0].bias.add_(0.1)
    _, _, sal2 = model.predict_saliency_classes_batch(x, (1, 0))
    assert not torch.equal(sal2, sal)


# ---------------------------------------------------------------------------------------------------------------------------------
# 6. launch pattern: one forward per chunk, the fused first-block kernel once per class and chunk, no fp32 conv
# ---------------------------------------------------------------------------------------------------------------------------------
def test_launch_pattern_canonical_network():
    shape = (256, 256, 1)
    cfg, p = _net("torch", shape, [256, 128])
    x = torch.from_numpy(_images("torch", 128, shape, seed=4)).cuda()
    eng = engine_from(cfg, p, precision="fp32", max_batch=64, keep_all_activations=True)
    eng.set_fast_training(True)
    eng.set_profiling(True)
    eng.predict_saliency_classes(x, (0, 1))
    names = [n for n, _ in eng.last_profile()]
    eng.set_profiling(False)
    assert names.count("conv0_fwd_fused") == 2, names
    assert names.count("saliency_conv0") == 4, names
    assert [n for n in names if n.startswith("conv") and n.endswith("fp32")] == [], names
    eng.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 7. errors
# ---------------------------------------------------------------------------------------------------------------------------------
def test_errors_and_the_handle_stays_usable():
    from bcad_b200 import _lib
    shape, B = (32, 32, 1), 4
    cfg, p = _net("torch", shape, [32])
    x = torch.from_numpy(_images("torch", B, shape, seed=1)).cuda()
    tp = engine_from(cfg, p, precision="fp16x3", max_batch=8)
    with pytest.raises(ValueError, match="runs on the fp32 path"):
        tp.predict_saliency_classes(x, (0, 1))
    tp.close()
    lean = engine_from(cfg, p, precision="fp32", max_batch=8)
    with pytest.raises(ValueError, match="keep_all_activations"):
        lean.predict_saliency_classes(x, (0, 1))
    lean.close()
    eng = engine_from(cfg, p, precision="fp32", max_batch=8, keep_all_activations=True)
    eng.set_dropout_masks(np.ones((B, 32), np.float32))
    with pytest.raises(ValueError, match="dropout"):
        eng.predict_saliency_classes(x, (0, 1))
    eng.set_dropout_masks(None)
    lib, h, s = eng.lib, eng._h, eng._stream()
    sal = torch.empty((B, 9, 32, 32), device="cuda")
    ci = torch.zeros((B, 9), dtype=torch.int32, device="cuda")

    def call(K, classes, out):
        return lib.bcad_predict_saliency_classes(h, C.c_void_p(x.data_ptr()), B, K, classes, 1, None, None, None, out, None, s)

    sp, cp = C.c_void_p(sal.data_ptr()), C.c_void_p(ci.data_ptr())
    for K in (0, 9):
        assert call(K, cp, sp) == _lib.ERR_INVALID and "out of range" in _lib.last_error()
    assert call(3, None, sp) == _lib.ERR_INVALID                    # classes 0..2 of a 2-class model
    assert call(2, cp, None) == _lib.ERR_INVALID and "saliency" in _lib.last_error()
    with pytest.raises(ValueError, match="out of range"):
        eng.predict_saliency_classes(x, (0, 2))
    with pytest.raises(ValueError, match="1..8"):
        eng.predict_saliency_classes(x, [0] * 9)
    cls, probs, logits, s1, _ = eng.predict_saliency_classes(x, (0, 1))    # still usable
    c0, p0, l0 = eng.predict(x)
    assert torch.equal(cls, c0) and torch.equal(logits, l0) and bool(torch.isfinite(s1).all())
    eng.close()
