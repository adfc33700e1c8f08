"""The deployed dual-class overlay call as one batched host-buffer call for 8-bit grey images of any size
(bcad_gradcam_overlays_classes_host / Engine.gradcam_overlays_classes_host / GRADCAM.generate_dual_class_gradcam_overlays_batch).

At the model's input size every map is byte for byte the single-class host call's; at other sizes the host call is byte for byte the
device composition gray_resize_preprocess -> predict_explain_classes(out = image size) -> overlay_classes, whose overlay stage is
byte for byte bcad_overlay on img01 = u8 / 255 and whose resize stage is bcad_bottleneck_resize's one-channel arithmetic."""
import ctypes as C

import numpy as np
import pytest
import torch

from util import engine_from, ocnn

pytestmark = pytest.mark.gpu

# cv2.resize (OpenCV 4.13) of u8 / 255 against the kernel's arithmetic (double coordinate, float weight): a few ulp apart on many
# pixels.  Measured on a B200 at 512x512, 300x260 and 200x180 -> 256x256: <= 1.2e-7 on the resized image, <= 9.5e-7 after standardisation
RESIZE_TOL = 5e-7
STANDARDISED_TOL = 5e-6


def _canonical(shape=(256, 256, 1), hidden=(256, 128), seed=7):
    cfg = ocnn.NetConfig.torch_flavour(shape, 2, [(32, 3), (64, 3)], list(hidden), 0.01)
    return cfg, ocnn.init_params(cfg, seed=seed, bias_std=0.05)


def _imgs(B, h, w, seed):
    """8-bit grey images with structure (the mammography-like synthetic images) plus pixel noise."""
    rng = np.random.default_rng(seed)
    base = ocnn.synth_images(B, (h, w, 1), seed=seed, kind="mammo")[..., 0]
    base = (base - base.min()) / (base.max() - base.min() + 1e-12)
    return np.clip(base * 200 + rng.integers(0, 56, size=(B, h, w)), 0, 255).astype(np.uint8)


def _cols(classes, B, K):
    if classes is None:
        return np.tile(np.arange(K, dtype=np.int32), (B, 1))
    c = np.asarray(classes, dtype=np.int32)
    return np.broadcast_to(c, (B, K)) if c.ndim == 1 else c


@pytest.mark.parametrize("shape,hidden,precision,B,mb", [
    ((256, 256, 1), (256, 128), "fp16", 70, 64),     # the canonical network on the headline handle; chunks 32, 32, 6
    ((64, 48, 1), (32, 16), "fp32", 45, 16),          # odd model size, fp32 path, max_batch below the chunk
    ((64, 48, 1), (32, 16), "fp16x3", 37, 64),
])
def test_model_size_maps_equal_single_class_host_calls(shape, hidden, precision, B, mb):
    cfg, p = _canonical(shape, hidden)
    eng = engine_from(cfg, p, precision=precision, max_batch=mb)
    imgs = _imgs(B, shape[0], shape[1], seed=B)
    rng = np.random.default_rng(1)
    for standardise in (True, False):
        for classes in ((0,), (0, 1), rng.integers(0, 2, size=(B, 3)), None):
            cls, probs, logits, ov, hu = eng.gradcam_overlays_classes_host(imgs, classes, "logit", standardise)
            K = ov.shape[1]
            assert ov.shape == (B, K) + shape[:2] + (3,) and hu.shape == (B, K) + shape[:2]
            cols = _cols(classes, B, K)
            for k in range(K):
                c1, p1, l1, ov1, hu1 = eng.gradcam_overlays_host(imgs, cols[:, k].copy(), "logit", standardise)
                assert np.array_equal(cls, c1) and np.array_equal(probs, p1) and np.array_equal(logits, l1)
                assert np.array_equal(ov[:, k], ov1), f"overlay of column {k} differs ({standardise=}, {classes=})"
                assert np.array_equal(hu[:, k], hu1), f"heatmap_uint8 of column {k} differs ({standardise=}, {classes=})"
    eng.close()


def _device_composition(eng, imgs, classes, standardise):
    from bcad_b200 import engine as E
    h, w, c = eng.spec.input_shape
    g = torch.from_numpy(imgs).cuda()
    x = E.gray_resize_preprocess(g, (h, w), c, standardise)
    cls, probs, logits, heat = eng.predict_explain_classes(x, classes, "logit", out_hw=imgs.shape[1:])
    ov, hu = E.overlay_classes(g, heat)
    return g, heat, cls, probs, logits, ov, hu


@pytest.mark.parametrize("img_hw", [(512, 512), (300, 260), (200, 180)])
def test_other_sizes_equal_device_composition(img_hw, monkeypatch):
    from bcad_b200 import engine as E
    cfg, p = _canonical()
    eng = engine_from(cfg, p, precision="fp16", max_batch=64)
    B = 5
    imgs = _imgs(B, img_hw[0], img_hw[1], seed=img_hw[1])
    classes = np.array([[0, 1], [1, 0], [1, 1], [0, 1], [0, 0]], np.int32)
    for standardise in (True, False):
        cls, probs, logits, ov, hu = eng.gradcam_overlays_classes_host(imgs, classes, "logit", standardise)
        g, heat, c2, p2, l2, ov2, hu2 = _device_composition(eng, imgs, classes, standardise)
        assert np.array_equal(cls, c2.cpu().numpy()) and np.array_equal(probs, p2.cpu().numpy()) and np.array_equal(logits, l2.cpu().numpy())
        assert np.array_equal(ov, ov2.cpu().numpy()) and np.array_equal(hu, hu2.cpu().numpy())
        img01 = torch.from_numpy(imgs.astype(np.float32) / np.float32(255.0)).cuda()   # IEEE division, as the kernels divide
        for k in range(2):                                       # every map: bcad_overlay on img01 = u8 / 255
            ov1, hu1 = E.overlay(img01, heat[:, k])
            assert torch.equal(ov2[:, k], ov1) and torch.equal(hu2[:, k], hu1)
        monkeypatch.setenv("BCAD_HOST_CHUNK", "2")              # chunks of 2, 2, 1 against one chunk of 5
        cc, pc, lc, ovc, huc = eng.gradcam_overlays_classes_host(imgs, classes, "logit", standardise)
        monkeypatch.delenv("BCAD_HOST_CHUNK")
        assert np.array_equal(cls, cc) and np.array_equal(probs, pc) and np.array_equal(ov, ovc) and np.array_equal(hu, huc)
        ho, hh = eng.gradcam_overlays_classes_host(imgs, classes, "logit", standardise, want_overlay=False)[3:]
        assert ho is None and np.array_equal(hh, hu)
        ho, hh = eng.gradcam_overlays_classes_host(imgs, classes, "logit", standardise, want_heat=False)[3:]
        assert hh is None and np.array_equal(ho, ov)
    eng.close()


def _emulate_resize(u8, H, W):
    """The kernel's arithmetic on the CPU: coordinate in float64, weight float32(frac), float32 products and sums without FMA."""
    def coord(n_dst, ns):
        sd = (np.arange(n_dst, dtype=np.float64) + 0.5) * (ns / n_dst) - 0.5
        i0 = np.floor(sd).astype(np.int64)
        f = (sd - i0).astype(np.float32)
        f[i0 < 0] = 0
        i0[i0 < 0] = 0
        f[i0 >= ns - 1] = 0
        i0[i0 >= ns - 1] = ns - 1
        return i0, np.minimum(i0 + 1, ns - 1), f
    src = u8.astype(np.float32) / np.float32(255.0)
    x0, x1, fx = coord(W, u8.shape[-1])
    y0, y1, fy = coord(H, u8.shape[-2])
    gx, gy = np.float32(1) - fx, np.float32(1) - fy
    top = src[:, y0][:, :, x0] * gx + src[:, y0][:, :, x1] * fx
    bot = src[:, y1][:, :, x0] * gx + src[:, y1][:, :, x1] * fx
    return top * gy[:, None] + bot * fy[:, None]


@pytest.mark.parametrize("img_hw", [(512, 512), (300, 260), (200, 180), (256, 256)])
def test_resized_input_against_bottleneck_resize_and_cv2(img_hw):
    import cv2
    from bcad_b200 import _lib, engine as E
    H, W = 256, 256
    B = 3
    imgs = _imgs(B, img_hw[0], img_hw[1], seed=3)
    g = torch.from_numpy(imgs).cuda()
    x0 = E.gray_resize_preprocess(g, (H, W), 1, False)[..., 0]
    x1 = E.gray_resize_preprocess(g, (H, W), 3, True)
    assert torch.equal(x1[..., 0], x1[..., 2])
    x1 = x1[..., 0]
    # bit for bit bcad_bottleneck_resize (one channel, HWC) of the same unit-range image, and its CPU emulation
    src = torch.from_numpy(imgs.astype(np.float32) / np.float32(255.0))[..., None].cuda()   # IEEE division, as the kernels divide
    ref = torch.empty((B, H, W, 1), device="cuda")
    _lib.check(_lib.load().bcad_bottleneck_resize(C.c_void_p(src.data_ptr()), B, 1, img_hw[0], img_hw[1], 1, H, W,
                                                  C.c_void_p(ref.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert torch.equal(x0, ref[..., 0])
    assert np.array_equal(x0.cpu().numpy(), _emulate_resize(imgs, H, W))
    if img_hw == (H, W):                                         # the model's size: exactly gray_preprocess
        _, xp = E.gray_preprocess(g, 1, True)
        assert torch.equal(x1, xp[..., 0])
    worst_r = worst_s = 0.0
    for b in range(B):
        r = cv2.resize((imgs[b] / 255.0).astype(np.float32), (W, H), interpolation=cv2.INTER_LINEAR)
        s = (r - r.mean()) / (r.std() + 1e-8)
        worst_r = max(worst_r, float(np.abs(x0[b].cpu().numpy() - r).max()))
        worst_s = max(worst_s, float(np.abs(x1[b].cpu().numpy() - s).max()))
    print(f"\nresize {img_hw} -> {(H, W)}: largest difference to cv2 {worst_r:.3e} (resized), {worst_s:.3e} (standardised)")
    assert worst_r <= RESIZE_TOL and worst_s <= STANDARDISED_TOL


def test_overlay_classes_equals_overlay_on_odd_sizes():
    from bcad_b200 import engine as E
    rng = np.random.default_rng(5)
    for (B, K, H, W) in ((3, 3, 33, 31), (2, 8, 17, 12), (4, 1, 64, 48)):
        g = torch.from_numpy(rng.integers(0, 256, size=(B, H, W), dtype=np.uint8)).cuda()
        cams = torch.from_numpy(rng.random((B, K, H, W), dtype=np.float32)).cuda()
        cams[:, :, 0, 0] = 1.0
        ov, hu = E.overlay_classes(g, cams)
        for k in range(K):
            ov1, hu1 = E.overlay(torch.from_numpy(g.cpu().numpy().astype(np.float32) / np.float32(255.0)).cuda(), cams[:, k])
            assert torch.equal(ov[:, k], ov1) and torch.equal(hu[:, k], hu1), (B, K, H, W, k)


def test_gradcam_batch_against_single_image_mirror_512():
    """GRADCAM.generate_dual_class_gradcam_overlays_batch on 512x512 images against the single-image mirror, which resizes with cv2
    and standardises in float32 NumPy: the classes agree; heat-maps and overlays differ by a few levels in a counted number of pixels."""
    from bcad_b200 import ADCNNM as A, GRADCAM as G
    cfg, p = _canonical()
    model = A.CNNModel((256, 256, 1), 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[256, 128], max_batch=64).eval()
    model.load_state_dict(ocnn.params_to_state_dict(cfg, p))
    B = 4
    imgs = _imgs(B, 512, 512, seed=11)
    cls, probs, ov, hu = G.generate_dual_class_gradcam_overlays_batch(imgs, [0, 1], model=model)
    assert ov.shape == (B, 2, 512, 512, 3) and hu.shape == (B, 2, 512, 512) and cls.dtype == np.int64
    n_heat = n_ov = 0
    d_heat = d_ov = 0
    for b in range(B):
        one = G.generate_dual_class_gradcam_overlays_pytorch(imgs[b], [0, 1], model=model, write_png=False)
        for k in (0, 1):
            o1, h1 = one[k]
            dh = np.abs(hu[b, k].astype(np.int32) - h1)
            do = np.abs(ov[b, k].astype(np.int32) - o1)
            n_heat += int((dh > 0).sum()); n_ov += int((do > 0).any(-1).sum())
            d_heat = max(d_heat, int(dh.max())); d_ov = max(d_ov, int(do.max()))
    print(f"\n512x512 against the single-image mirror: heatmap_uint8 differs in {n_heat} of {B * 2 * 512 * 512} pixels (at most {d_heat}), "
          f"overlays in {n_ov} (at most {d_ov})")
    import cv2
    eng = getattr(model, "fast_engine", None) or model.engine      # the mirror's input, predicted on the same handle
    x = np.stack([G.default_preprocess(cv2.resize((im / 255.0).astype(np.float32), (256, 256), interpolation=cv2.INTER_LINEAR),
                                       (256, 256, 1)) for im in imgs])
    assert np.array_equal(cls, eng.predict(x)[0].cpu().numpy())
    assert d_heat <= 1 and n_heat <= 0.01 * B * 2 * 512 * 512
    assert d_ov <= 4 and n_ov <= 0.01 * B * 2 * 512 * 512          # a heat level across a JET step moves the colour by a few levels


def test_gradcam_batch_any_size_and_output_arrays():
    from bcad_b200 import ADCNNM as A, GRADCAM as G
    shape = (64, 48, 1)
    cfg, p = _canonical(shape, (32, 16), seed=6)
    model = A.CNNModel(shape, 2, conv_layers=[(32, 3), (64, 3)], hidden_units=[32, 16], max_batch=64).eval()
    model.load_state_dict(ocnn.params_to_state_dict(cfg, p))
    B = 9
    imgs = _imgs(B, 100, 90, seed=2)
    ov_out = torch.empty((B, 3, 100, 90, 3), dtype=torch.uint8).pin_memory().numpy()
    hu_out = np.empty((B, 3, 100, 90), np.uint8)
    cls, probs, ov, hu = G.generate_dual_class_gradcam_overlays_batch(imgs, [1, 0, 1], model=model, overlay_out=ov_out, heat_out=hu_out)
    assert ov is ov_out and hu is hu_out
    eng = getattr(model, "fast_engine", None) or model.engine
    c2, p2, _, ov2, hu2 = eng.gradcam_overlays_classes_host(imgs, (1, 0, 1))
    assert np.array_equal(cls, c2) and np.array_equal(probs, p2) and np.array_equal(ov, ov2) and np.array_equal(hu, hu2)
    assert np.array_equal(ov[:, 0], ov[:, 2]) and np.array_equal(hu[:, 0], hu[:, 2])
    with pytest.raises(ValueError):
        G.generate_dual_class_gradcam_overlays_batch(imgs.astype(np.float32), [0, 1], model=model)


def test_errors():
    from bcad_b200 import _lib
    cfg, p = _canonical((32, 32, 1), (32,))
    eng = engine_from(cfg, p, precision="fp32", max_batch=8)
    lib, h = eng.lib, eng._h
    B, hh, ww = 3, 40, 36
    imgs = np.zeros((B, hh, ww), np.uint8)
    ov = np.empty((B, 9, hh, ww, 3), np.uint8)
    hu = np.empty((B, 9, hh, ww), np.uint8)
    ci = np.zeros((B, 9), np.int32)
    P = lambda a: C.c_void_p(a.ctypes.data) if a is not None else None  # noqa: E731

    def call(K, classes, o, u, img=imgs, Bn=B, ih=hh, iw=ww):
        return lib.bcad_gradcam_overlays_classes_host(h, P(img), Bn, ih, iw, K, P(classes), 0, 1, None, None, None, P(o), P(u))

    assert call(0, ci, ov, hu) == _lib.ERR_INVALID
    assert call(9, ci, ov, hu) == _lib.ERR_INVALID
    assert call(3, None, ov, hu) == _lib.ERR_INVALID                 # classes 0..2 of a 2-class model
    bad = np.zeros((B, 2), np.int32)
    bad[1, 1] = 2
    assert call(2, bad, ov, hu) == _lib.ERR_INVALID
    bad[1, 1] = -1
    assert call(2, bad, ov, hu) == _lib.ERR_INVALID
    assert call(2, ci, None, None) == _lib.ERR_INVALID
    assert call(2, ci, ov, hu, Bn=0) == _lib.ERR_INVALID
    assert call(2, ci, ov, hu, ih=0) == _lib.ERR_INVALID
    assert call(2, ci, ov, hu) == _lib.OK
    assert call(2, None, None, hu) == _lib.OK
    with pytest.raises(ValueError, match="uint8"):
        eng.gradcam_overlays_classes_host(imgs.astype(np.float32), (0, 1))
    with pytest.raises(ValueError, match="out of range"):
        eng.gradcam_overlays_classes_host(imgs, (0, 2))
    with pytest.raises(ValueError):
        eng.gradcam_overlays_classes_host(imgs, [0] * 9)
    with pytest.raises(ValueError):
        eng.gradcam_overlays_classes_host(imgs, (0, 1), overlay_out=np.empty((B, 2, hh, ww), np.uint8))
    dev = torch.zeros((B, hh, ww), dtype=torch.uint8, device="cuda")
    cam = torch.zeros((B, 9, hh, ww), device="cuda")
    s = eng._stream()
    assert lib.bcad_overlay_classes(C.c_void_p(dev.data_ptr()), C.c_void_p(cam.data_ptr()), B, 9, hh, ww, C.c_void_p(dev.data_ptr()), None, s) == _lib.ERR_INVALID
    assert lib.bcad_overlay_classes(C.c_void_p(dev.data_ptr()), C.c_void_p(cam.data_ptr()), B, 2, hh, ww, None, None, s) == _lib.ERR_INVALID
    torch.cuda.synchronize()
    eng.close()


def test_sharded_equals_single_gpu_call():
    import bcad_b200
    from util import spec_from_cfg
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"ShardedEngine needs two or more GPUs, {n} visible")
    cfg, p = _canonical()
    single = engine_from(cfg, p, precision="fp16", max_batch=64)
    B = 37
    imgs = _imgs(B, 300, 260, seed=8)
    want = single.gradcam_overlays_classes_host(imgs, (0, 1))
    for world in sorted({2, 4, 8, n} & set(range(2, n + 1))):
        sh = bcad_b200.ShardedEngine(spec_from_cfg(cfg), list(range(world)), precision="fp16", max_batch=64)
        sh.set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
        got = sh.gradcam_overlays_classes_host(imgs, (0, 1))
        for a, b in zip(got, want):
            assert np.array_equal(a, b), f"{world} GPUs"
        sh.close()
    single.close()
