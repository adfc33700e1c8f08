"""The dual-class input-gradient saliency overlays as one batched host-buffer call for 8-bit grey images of any size
(bcad_saliency_overlays_classes_host / Engine.saliency_overlays_classes_host / explainability.generate_dual_class_saliency_overlays_batch).

Every output of the host call is byte for byte the device composition gray_resize_preprocess -> predict_saliency_classes ->
saliency_overlay_resized.  The colouring stage is byte for byte generate_saliency_overlay's cv2 calls on the device's own saliency maps:
applyColorMap, cv2.resize of the 8-bit BGR heat-map to the image's size, addWeighted with the grey image.  Its resize follows OpenCV's
fixed-point INTER_LINEAR for 8-bit data, emulated below in NumPy (the CPU reference, checked against cv2.resize without a GPU)."""
import ctypes as C

import numpy as np
import pytest
import torch

from util import engine_from, ocnn

SIZES = [(256, 256), (512, 512), (300, 260), (200, 180)]


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU reference: cv2.resize(u8 image, (dw, dh), INTER_LINEAR)
# ---------------------------------------------------------------------------------------------------------------------------------
def _cv_linear_coeffs(n_src, n_dst, clamp_weight):
    """Source indices and 11-bit weights of OpenCV's 8-bit INTER_LINEAR along one axis.  Columns (clamp_weight) clamp the coordinate at
    both borders; rows keep the weights and clamp only the indices."""
    scale = 1.0 / (n_dst / n_src)
    f = ((np.arange(n_dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if clamp_weight:
        lo = s < 0
        f[lo], s[lo] = 0, 0
        hi = s >= n_src - 1
        f[hi], s[hi] = 0, n_src - 1
        i0, i1 = s, np.minimum(s + 1, n_src - 1)
    else:
        i0, i1 = np.clip(s, 0, n_src - 1), np.clip(s + 1, 0, n_src - 1)
    w0 = np.rint((np.float32(1) - f) * np.float32(2048)).astype(np.int64)
    w1 = np.rint(f * np.float32(2048)).astype(np.int64)
    return i0, i1, w0, w1


def cv_resize_u8(src, dh, dw):
    """src uint8 [h,w,C] -> [dh,dw,C]: horizontal S[x0] * c0 + S[x1] * c1 in integers, then the vertical step
    ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2, saturated."""
    h, w = src.shape[:2]
    x0, x1, c0, c1 = _cv_linear_coeffs(w, dw, True)
    y0, y1, b0, b1 = _cv_linear_coeffs(h, dh, False)
    S = src.astype(np.int64)
    hor = S[:, x0] * c0[None, :, None] + S[:, x1] * c1[None, :, None]
    out = (((b0[:, None, None] * (hor[y0] >> 4)) >> 16) + ((b1[:, None, None] * (hor[y1] >> 4)) >> 16) + 2) >> 2
    return np.clip(out, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("src_hw,dst_hw", [
    ((256, 256), (512, 512)), ((256, 256), (300, 260)), ((256, 256), (200, 180)), ((256, 256), (1024, 768)), ((125, 125), (512, 512)),
    ((64, 48), (97, 333)), ((254, 254), (512, 512)), ((256, 256), (255, 257)), ((67, 61), (13, 7)), ((5, 3), (2, 11)), ((1, 1), (4, 3)),
    ((3, 1), (9, 5)), ((256, 256), (256, 256)),
])
def test_resize_emulation_equals_cv2(src_hw, dst_hw):
    import cv2
    rng = np.random.default_rng(src_hw[0] * 1000 + dst_hw[1])
    for _ in range(3):
        src = rng.integers(0, 256, size=src_hw + (3,), dtype=np.uint8)
        want = cv2.resize(src, (dst_hw[1], dst_hw[0]), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(cv_resize_u8(src, *dst_hw), want)


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _net(kind, shape=(256, 256, 1), hidden=(256, 128), seed=7):
    mk = ocnn.NetConfig.torch_flavour if kind == "torch" else ocnn.NetConfig.numpy_flavour
    cfg = mk(shape, 2, [(32, 3), (64, 3)], list(hidden), 0.01)
    return cfg, ocnn.init_params(cfg, seed=seed, bias_std=0.05)


def _imgs(B, h, w, seed):
    """8-bit grey images with structure (the mammography-like synthetic images) plus pixel noise."""
    rng = np.random.default_rng(seed)
    base = ocnn.synth_images(B, (h, w, 1), seed=seed, kind="mammo")[..., 0]
    base = (base - base.min()) / (base.max() - base.min() + 1e-12)
    return np.clip(base * 200 + rng.integers(0, 56, size=(B, h, w)), 0, 255).astype(np.uint8)


def _saliency_engine(cfg, p, **kw):
    return engine_from(cfg, p, precision="fp32", keep_all_activations=True, **kw)


def _device_composition(eng, imgs, classes, grad_mode, standardise):
    from bcad_b200 import engine as E
    h, w, c = eng.spec.input_shape
    g = torch.from_numpy(imgs).cuda()
    x = E.gray_resize_preprocess(g, (h, w), c, standardise)
    cls, probs, logits, sal, _ = eng.predict_saliency_classes(x, classes, grad_mode)
    ov, hm = E.saliency_overlay_resized(g, sal)
    return [t.cpu().numpy() for t in (cls, probs, logits, ov, hm, sal)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["numpy", "torch"])
@pytest.mark.parametrize("img_hw", SIZES)
def test_host_call_equals_device_composition(kind, img_hw, monkeypatch):
    cfg, p = _net(kind)
    eng = _saliency_engine(cfg, p, max_batch=64)
    B = 7
    imgs = _imgs(B, img_hw[0], img_hw[1], seed=img_hw[1])
    rng = np.random.default_rng(3)
    per_image = rng.integers(0, 2, size=(B, 2)).astype(np.int32)
    for fast in (False, True):
        eng.set_fast_training(fast)
        for grad_mode in ("softmax_ce", "logit"):
            for standardise in (True, False):
                for classes in ((1,), (0, 1), (1, 0, 1), per_image, None):
                    got = eng.saliency_overlays_classes_host(imgs, classes, grad_mode, standardise, want_saliency=True)
                    want = _device_composition(eng, imgs, classes, grad_mode, standardise)
                    K = got[3].shape[1]
                    assert got[3].shape == got[4].shape == (B, K) + img_hw + (3,) and got[5].shape == (B, K, 256, 256)
                    for name, a, b in zip(("cls", "probs", "logits", "overlays", "heat-maps", "saliency"), got, want):
                        assert np.array_equal(a, b), f"{name} differ ({fast=}, {grad_mode=}, {standardise=}, {classes=})"
                    if classes is not None and len(np.shape(classes)) == 1 and list(classes) == [1, 0, 1]:
                        assert np.array_equal(got[3][:, 0], got[3][:, 2]) and np.array_equal(got[5][:, 0], got[5][:, 2])
        # chunks of 3, 3, 1 against one chunk of 7 (the handle's buffers were sized by the unchunked calls above)
        full = eng.saliency_overlays_classes_host(imgs, per_image, "softmax_ce", True, want_saliency=True)
        monkeypatch.setenv("BCAD_HOST_CHUNK", "3")
        chunked = eng.saliency_overlays_classes_host(imgs, per_image, "softmax_ce", True, want_saliency=True)
        monkeypatch.delenv("BCAD_HOST_CHUNK")
        for a, b in zip(full, chunked):
            assert np.array_equal(a, b), f"chunked call differs ({fast=})"
    eng.close()


@pytest.mark.gpu
def test_max_batch_below_the_batch():
    """Chunks bounded by a small max_batch (4, 3 of 7 images) against the device composition."""
    cfg, p = _net("numpy", (64, 48, 1), (32, 16))
    eng = _saliency_engine(cfg, p, max_batch=4)
    imgs = _imgs(7, 90, 70, seed=5)
    got = eng.saliency_overlays_classes_host(imgs, (0, 1), want_saliency=True)
    want = _device_composition(eng, imgs, (0, 1), "softmax_ce", True)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    eng.close()


def _cv2_overlay(gray, s):
    import cv2
    h, w = gray.shape
    heat = cv2.resize(cv2.applyColorMap((s * 255).astype(np.uint8), cv2.COLORMAP_JET), (w, h))
    return cv2.addWeighted(np.repeat(gray[..., None], 3, axis=-1), 0.5, heat, 0.5, 0), heat


@pytest.mark.gpu
@pytest.mark.parametrize("img_hw", SIZES + [(97, 333)])
def test_colouring_equals_cv2_on_the_device_saliency(img_hw):
    from bcad_b200 import engine as E
    cfg, p = _net("numpy")
    eng = _saliency_engine(cfg, p, max_batch=64)
    eng.set_fast_training(True)
    B = 4
    imgs = _imgs(B, img_hw[0], img_hw[1], seed=9)
    _, _, _, ov, hm, sal = eng.saliency_overlays_classes_host(imgs, (0, 1), want_saliency=True)
    import cv2
    for b in range(B):
        for k in range(2):
            o1, h1 = _cv2_overlay(imgs[b], sal[b, k])
            assert np.array_equal(hm[b, k], h1), (img_hw, b, k)
            assert np.array_equal(ov[b, k], o1), (img_hw, b, k)
            jet = cv2.applyColorMap((sal[b, k] * 255).astype(np.uint8), cv2.COLORMAP_JET)
            assert np.array_equal(cv_resize_u8(jet, *img_hw), h1)
    if img_hw == (256, 256):                                     # the model's size: exactly bcad_saliency_overlay with base_c = 1
        o2, h2 = E.saliency_overlay(torch.from_numpy(imgs).cuda(), torch.from_numpy(sal).cuda())
        assert np.array_equal(o2.cpu().numpy(), ov) and np.array_equal(h2.cpu().numpy(), hm)
    eng.close()


@pytest.mark.gpu
def test_colouring_kernel_on_odd_sizes_equals_cv2():
    """bcad_saliency_overlay_resized alone: random maps, K up to 8, sizes that are not multiples of 4, up- and down-scaling."""
    from bcad_b200 import engine as E
    rng = np.random.default_rng(5)
    for (B, K, H, W, h, w) in ((3, 3, 33, 31, 65, 97), (2, 8, 17, 12, 5, 7), (2, 1, 64, 48, 64, 49), (1, 2, 40, 40, 333, 97)):
        g = rng.integers(0, 256, size=(B, h, w), dtype=np.uint8)
        s = rng.random((B, K, H, W), dtype=np.float32)
        ov, hm = E.saliency_overlay_resized(torch.from_numpy(g).cuda(), torch.from_numpy(s).cuda())
        ov, hm = ov.cpu().numpy(), hm.cpu().numpy()
        for b in range(B):
            for k in range(K):
                o1, h1 = _cv2_overlay(g[b], s[b, k])
                assert np.array_equal(hm[b, k], h1) and np.array_equal(ov[b, k], o1), (B, K, H, W, h, w, b, k)


@pytest.mark.gpu
def test_outputs_are_independent():
    cfg, p = _net("torch", (64, 48, 1), (32, 16))
    eng = _saliency_engine(cfg, p, max_batch=64)
    imgs = _imgs(5, 100, 90, seed=2)
    cls, probs, logits, ov, hm, sal = eng.saliency_overlays_classes_host(imgs, (1, 0), want_saliency=True)
    r = eng.saliency_overlays_classes_host(imgs, (1, 0), want_overlay=False)
    assert r[3] is None and r[5] is None and np.array_equal(r[4], hm) and np.array_equal(r[0], cls)
    r = eng.saliency_overlays_classes_host(imgs, (1, 0), want_heat=False)
    assert r[4] is None and np.array_equal(r[3], ov) and np.array_equal(r[1], probs)
    r = eng.saliency_overlays_classes_host(imgs, (1, 0), want_overlay=False, want_heat=False, want_saliency=True)
    assert r[3] is None and r[4] is None and np.array_equal(r[5], sal) and np.array_equal(r[2], logits)
    ov_out = torch.empty(ov.shape, dtype=torch.uint8).pin_memory().numpy()
    sal_out = np.empty(sal.shape, np.float32)
    r = eng.saliency_overlays_classes_host(imgs, (1, 0), overlay_out=ov_out, saliency_out=sal_out)
    assert r[3] is ov_out and r[5] is sal_out and np.array_equal(ov_out, ov) and np.array_equal(sal_out, sal)
    eng.close()


@pytest.mark.gpu
def test_mirrors_batch_call_returns_the_engine_call():
    from bcad_b200 import ADCNNM as A, explainability as X
    from bcad_b200.CNNModel import CNNModel
    shape = (64, 48, 1)
    cfg, p = _net("torch", shape, (32, 16), seed=6)
    torch_model = A.CNNModel(shape, 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[32, 16], max_batch=16).eval()
    torch_model.load_state_dict(ocnn.params_to_state_dict(cfg, p))
    np.random.seed(4)
    numpy_model = CNNModel(shape, 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[32, 16], max_batch=8)
    imgs = _imgs(11, 120, 80, seed=12)
    for model in (torch_model, numpy_model):
        cls, probs, ov, hm, sal = X.generate_dual_class_saliency_overlays_batch(model, imgs, [0, 1], want_saliency=True)
        assert cls.dtype == np.int64 and ov.shape == hm.shape == (11, 2, 120, 80, 3) and sal.shape == (11, 2) + shape[:2]
        c2, p2, _, o2, h2, s2 = model.saliency_engine.saliency_overlays_classes_host(imgs, (0, 1), "softmax_ce", True, want_saliency=True)
        assert np.array_equal(cls, c2) and np.array_equal(probs, p2) and np.array_equal(ov, o2) and np.array_equal(hm, h2)
        assert np.array_equal(sal, s2)
        assert X.generate_dual_class_saliency_overlays_batch(model, imgs[0], [1])[4] is None
    with pytest.raises(ValueError, match="uint8"):
        X.generate_dual_class_saliency_overlays_batch(numpy_model, imgs.astype(np.float32), [0, 1])


@pytest.mark.gpu
def test_sharded_equals_single_gpu_call():
    import bcad_b200
    from util import spec_from_cfg
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"ShardedEngine needs two or more GPUs, {n} visible")
    cfg, p = _net("numpy")
    single = _saliency_engine(cfg, p, max_batch=64)
    single.set_fast_training(True)
    B = 37
    imgs = _imgs(B, 300, 260, seed=8)
    want = single.saliency_overlays_classes_host(imgs, (0, 1), want_saliency=True)
    for world in sorted({2, 4, 8, n} & set(range(2, n + 1))):
        sh = bcad_b200.ShardedEngine(spec_from_cfg(cfg), list(range(world)), precision="fp32", max_batch=64, keep_all_activations=True)
        sh.set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
        sh.set_fast_training(True)
        got = sh.saliency_overlays_classes_host(imgs, (0, 1), want_saliency=True)
        for a, b in zip(got, want):
            assert np.array_equal(a, b), f"{world} GPUs"
        sh.close()
    single.close()


@pytest.mark.gpu
def test_errors():
    from bcad_b200 import _lib
    cfg, p = _net("torch", (32, 32, 1), (32,))
    eng = _saliency_engine(cfg, p, max_batch=8)
    lib = eng.lib
    B, hh, ww = 3, 40, 36
    imgs = np.zeros((B, hh, ww), np.uint8)
    ov = np.empty((B, 9, hh, ww, 3), np.uint8)
    hm = np.empty((B, 9, hh, ww, 3), np.uint8)
    sal = np.empty((B, 9, 32, 32), np.float32)
    ci = np.zeros((B, 9), np.int32)
    P = lambda a: C.c_void_p(a.ctypes.data) if a is not None else None  # noqa: E731

    def call(K, classes, o, h, s=None, handle=eng._h, Bn=B, ih=hh, iw=ww):
        return lib.bcad_saliency_overlays_classes_host(handle, P(imgs), Bn, ih, iw, K, P(classes), 1, 1, None, None, None, P(s), P(o), P(h))

    assert call(0, ci, ov, hm) == _lib.ERR_INVALID
    assert call(9, ci, ov, hm) == _lib.ERR_INVALID
    assert call(3, None, ov, hm) == _lib.ERR_INVALID                 # classes 0..2 of a 2-class model
    bad = np.zeros((B, 2), np.int32)
    bad[1, 1] = 2
    assert call(2, bad, ov, hm) == _lib.ERR_INVALID
    bad[1, 1] = -1
    assert call(2, bad, ov, hm) == _lib.ERR_INVALID
    assert call(2, ci, None, None) == _lib.ERR_INVALID               # all three outputs NULL
    assert call(2, ci, ov, hm, Bn=0) == _lib.ERR_INVALID
    assert call(2, ci, ov, hm, ih=0) == _lib.ERR_INVALID
    assert call(2, ci, ov, hm, iw=16385) == _lib.ERR_INVALID
    assert call(2, ci, ov, hm) == _lib.OK
    assert call(2, None, None, None, s=sal) == _lib.OK
    # handles run_saliency refuses are refused before any copy
    tensor = engine_from(*_net("torch", (64, 48, 1), (32, 16)), precision="fp16x3", max_batch=8)
    assert call(2, ci, ov, hm, handle=tensor._h) == _lib.ERR_INVALID and "fp32" in _lib.last_error()
    lean = engine_from(cfg, p, precision="fp32", max_batch=8)
    assert call(2, ci, ov, hm, handle=lean._h) == _lib.ERR_INVALID and "keep_all_activations" in _lib.last_error()
    eng.set_dropout_masks(np.ones((B, 32), np.float32))
    assert call(2, ci, ov, hm) == _lib.ERR_INVALID and "dropout" in _lib.last_error()
    eng.set_dropout_masks(None)
    assert call(2, ci, ov, hm) == _lib.OK
    with pytest.raises(ValueError, match="uint8"):
        eng.saliency_overlays_classes_host(imgs.astype(np.float32), (0, 1))
    with pytest.raises(ValueError, match="out of range"):
        eng.saliency_overlays_classes_host(imgs, (0, 2))
    with pytest.raises(ValueError):
        eng.saliency_overlays_classes_host(imgs, [0] * 9)
    with pytest.raises(ValueError):
        eng.saliency_overlays_classes_host(imgs, (0, 1), heat_out=np.empty((B, 2, hh, ww), np.uint8))
    dev = torch.zeros((B, hh, ww), dtype=torch.uint8, device="cuda")
    smap = torch.zeros((B, 9, 32, 32), device="cuda")
    out = torch.empty((B, 9, hh, ww, 3), dtype=torch.uint8, device="cuda")
    s = eng._stream()
    D = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    assert lib.bcad_saliency_overlay_resized(D(dev), D(smap), B, 9, 32, 32, hh, ww, D(out), None, s) == _lib.ERR_INVALID
    assert lib.bcad_saliency_overlay_resized(D(dev), D(smap), 0, 2, 32, 32, hh, ww, D(out), None, s) == _lib.ERR_INVALID
    assert lib.bcad_saliency_overlay_resized(D(dev), D(smap), B, 2, 32, 32, 0, ww, D(out), None, s) == _lib.ERR_INVALID
    torch.cuda.synchronize()
    for e in (tensor, lean, eng):
        e.close()
