"""The pre-activation Grad-CAM target (``set_explain_target("conv_preact")``: the nn.Conv2d output that pytorch_grad_cam hooks on the
reference's torch CNN, ADCNNM.py:76) on the tensor-core paths.

With first-index pooling the channel weights come from the masked fc1 input-gradient GEMM on tcgen05 (alpha_preact_tcgen05); the tails
undo the activation, z = a > 0 ? a : a / slope.  The tie-duplicating (NumPy) flavour keeps its dense pooled gradient and gains the
LeakyReLU' factor in alpha_ties_c8.  Checked: every image of the canonical network against the float64 oracle, odd shapes against
the fp32 handle, the bitwise contracts (K classes, chunking, host buffers, overlays), the refinement twin, target switching,
refusals and several GPUs."""
import dataclasses

import numpy as np
import pytest
import torch

from util import engine_from, ocnn

pytestmark = pytest.mark.gpu

# fp16 handles, pre-activation target: the fp16 conv output's error (<= 8.3e-3 on |z| <= 12, measured) reaches this map unattenuated --
# the post-activation map scales negative z by the slope, 0.01 -- and a map whose positive part is small against |z| turns it into up to
# 1.4e-2 after min-max (2 of 128 canonical images, 1.8e-2 on one 64x48 image).  The fp16x3 handle stays within X3_TOL.
F16_PRE_TOL = 3e-2
F16_TAU = 1.5e-2         # the 16-bit path's bound on its hidden dense pre-activation error (test_gpu_tensor_path.py)
X3_TOL = 5e-4
X3_TAU = 5e-4
FP32_TOL = 1e-4
# bounds on the error of the last conv block's pooled output, where LeakyReLU' of a window's maximum switches: largest seen on the
# canonical network and the 64x48 one, fp16 8.3e-3, fp16x3 1.7e-5, fp32 1.1e-5 (|P| up to 12)
F16_CONV_TAU = 1.5e-2
X3_CONV_TAU = 5e-4
FP32_CONV_TAU = 1e-4
PRE = "conv_preact"


def _np(t):
    return t.detach().cpu().numpy()


def compare_preact(cfg, params, x, engs, modes, batch=64):
    """oracle.compare.compare_all_images for the pre-activation target: every image of `x` on each engine of `engs`
    [(engine, tau, conv_tau)] (target already set) against the float64 oracle map of Z = A > 0 ? A : A / slope with
    dZ = dA * (A > 0 ? 1 : slope), nothing excluded.

    Two discontinuities get the device's branch where the oracle value lies within the path's error bound of the kink, and are
    counted: a hidden dense unit whose |z| <= tau (as compare_all_images does: `mask_violations` counts the rest), and -- new with
    this target -- LeakyReLU' of a pool window's maximum, where the oracle pooled value |P| <= conv_tau: the oracle then takes the
    sign of the device's pooled value, read back with get_tensor(BCAD_T_CONV_OUT).  Windows whose sign differs although |P| >
    conv_tau are `conv_mask_violations`; the overridden ones are `conv_overrides`.  Returns, per engine, one dict per mode as
    compare_all_images does."""
    from oracle import gradcam as ogc
    B = x.shape[0]
    n_hidden = len(cfg.hidden_units)
    last = len(cfg.conv_layers) - 1
    s = cfg.alpha_conv
    out = [[dict(cls_equal=np.zeros(B, bool), heat_err=np.zeros(B), mask_violations=0, conv_mask_violations=0, conv_overrides=0)
            for _ in modes] for _ in engs]
    mb = min(e.max_batch for e, _, _ in engs)
    for s0 in range(0, B, mb):
        s1 = min(B, s0 + mb)
        dev, dev_a = [], []
        for e, _, _ in engs:
            per_mode = []
            for class_idx, mode in modes:
                ci = None if class_idx is None else np.asarray(class_idx)[s0:s1]
                cls, _, _, heat = e.predict_explain(x[s0:s1], ci, mode)
                zs = [_np(e.get_tensor(2, j, s1 - s0)) for j in range(n_hidden)]        # BCAD_T_DENSE_Z
                per_mode.append((_np(cls), _np(heat), zs))
            dev.append(per_mode)
            dev_a.append(_np(e.get_tensor(0, last, s1 - s0)))                          # BCAD_T_CONV_OUT (the last forward's)
        for b0 in range(s0, s1, batch):
            b1 = min(s1, b0 + batch)
            sl = slice(b0 - s0, b1 - s0)
            cache = ocnn.forward(cfg, params, x[b0:b1])
            score = cache.probs if cfg.head == "softmax" else cache.logits
            o_cls = score.argmax(dim=-1).numpy()
            z_or = [cache.z[j].clone() for j in range(n_hidden)]
            A = cache.conv_out[last].numpy().astype(np.float32)
            n_, h_, w_, c_ = A.shape
            hp, wp = h_ // 2, w_ // 2

            def pool(t):
                return t[:, :2 * hp, :2 * wp].reshape(n_, hp, 2, wp, 2, c_).max(axis=(2, 4))
            po = pool(A.astype(np.float64))
            for ei, (e, e_tau, e_ctau) in enumerate(engs):
                pd = pool(dev_a[ei][sl].reshape(A.shape).astype(np.float64))
                for mi, (class_idx, mode) in enumerate(modes):
                    d_cls, d_heat, d_z = dev[ei][mi]
                    r = out[ei][mi]
                    for j in range(n_hidden):
                        zo = z_or[j].numpy()
                        differ = (zo > 0) != (d_z[j][sl] > 0)
                        r["mask_violations"] += int((differ & (np.abs(zo) > e_tau)).sum())
                        zj = zo.copy()
                        zj[differ] = np.where(d_z[j][sl][differ] > 0, 1e-300, -1e-300)
                        cache.z[j] = torch.as_tensor(zj)
                    ci = o_cls if class_idx is None else np.asarray(class_idx)[b0:b1]
                    cag, _, _ = ocnn.backward(cfg, params, cache, ocnn.top_gradient(cache, ci, mode), through_input=False)
                    for j in range(n_hidden):
                        cache.z[j] = z_or[j]
                    fac = np.where(A > 0, 1.0, s)
                    differ = (po > 0) != (pd > 0)
                    r["conv_mask_violations"] += int((differ & (np.abs(po) > e_ctau)).sum())
                    ov = differ & (np.abs(po) <= e_ctau)
                    r["conv_overrides"] += int(ov.sum())
                    if ov.any():           # the device's LeakyReLU' for the whole window (only its maximum carries a gradient)
                        big = np.repeat(np.repeat(ov, 2, axis=1), 2, axis=2)
                        fdev = np.repeat(np.repeat(np.where(pd > 0, 1.0, s), 2, axis=1), 2, axis=2)
                        sub = fac[:, :2 * hp, :2 * wp]
                        sub[big] = fdev[big]
                    Z = np.where(A > 0, A, A / s).astype(np.float32)
                    dZ = (cag[last].numpy() * fac).astype(np.float32)
                    o_heat = ogc.gradcam_tail_nhwc(Z, dZ, cfg.input_shape[:2])
                    r["cls_equal"][b0:b1] = d_cls[sl] == o_cls
                    r["heat_err"][b0:b1] = np.abs(d_heat[sl] - o_heat).reshape(b1 - b0, -1).max(axis=1)
    return out


def _canonical():
    cfg = ocnn.NetConfig.torch_flavour((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
    return cfg, ocnn.init_params(cfg, seed=7, bias_std=0.05)


def test_canonical_network_every_image_against_the_oracle():
    """512 distinct images, both grad modes, fp16 (refinement on) and fp16x3 against one oracle sweep of the pre-activation target."""
    cfg, p = _canonical()
    B = 512
    x = ocnn.synth_images(B, (256, 256, 1), seed=20251022)
    e16 = engine_from(cfg, p, precision="fp16", max_batch=256)
    e3 = engine_from(cfg, p, precision="fp16x3", max_batch=256)
    assert e16.uses_tensor_path and e3.uses_tensor_path and e16.refine_margin > 0
    e16.set_explain_target(PRE)
    e3.set_explain_target(PRE)
    modes = [(None, "logit"), (np.arange(B) % 2, "softmax_ce")]
    res = compare_preact(cfg, p, x, [(e16, F16_TAU, F16_CONV_TAU), (e3, X3_TAU, X3_CONV_TAU)], modes)
    for (eng, tol), rr in zip(((e16, F16_PRE_TOL), (e3, X3_TOL)), res):
        for r in rr:
            assert r["mask_violations"] == 0 and r["conv_mask_violations"] == 0
            assert r["cls_equal"].all(), f"classes differ on images {np.flatnonzero(~r['cls_equal'])}"
            assert r["heat_err"].max() <= tol, f"{eng.precision}: heat-map err {r['heat_err'].max()} (tol {tol})"
    e16.close()
    e3.close()


@pytest.mark.parametrize("flavour,precision,tol,tau,conv_tau", [("torch", "fp16", F16_PRE_TOL, F16_TAU, F16_CONV_TAU),
                                                                 ("torch", "fp16x3", X3_TOL, X3_TAU, X3_CONV_TAU),
                                                                 ("numpy", "fp16x3", X3_TOL, X3_TAU, X3_CONV_TAU)])
def test_odd_shapes_against_the_fp32_handle(flavour, precision, tol, tau, conv_tau):
    """64x48 inputs, hidden 64/16, 150 images on handles of 160 (rows not a multiple of 128), the tensor handle and an fp32 handle with
    the same weights and target.  Torch flavour: both against one oracle sweep, within their tolerances.  NumPy flavour (tie rule, exact
    zero background): the tie structure is the device's own (test_gpu_tensor_path.py), so the maps are compared with the fp32 handle's
    directly.  Then the post-activation maps differ."""
    mk = ocnn.NetConfig.numpy_flavour if flavour == "numpy" else ocnn.NetConfig.torch_flavour
    cfg = mk((64, 48, 1), 2, [(32, 3), (64, 3)], [64, 16], 0.01)
    p = ocnn.init_params(cfg, seed=4, bias_std=0.05)
    B = 150
    x = ocnn.synth_images(B, (64, 48, 1), seed=17, kind="mammo" if flavour == "numpy" else "gauss")
    ci = (np.arange(B) % 2).astype(np.int32)
    ref = engine_from(cfg, p, precision="fp32", max_batch=160)
    eng = engine_from(cfg, p, precision=precision, max_batch=160)
    ref.set_explain_target(PRE)
    eng.set_explain_target(PRE)
    if flavour == "numpy":
        for mode in ("logit", "softmax_ce"):
            want = _np(ref.predict_explain(x, ci, mode)[3])
            got = _np(eng.predict_explain(x, ci, mode)[3])
            assert np.abs(got - want).max() <= tol, f"{mode}: max err {np.abs(got - want).max()}"
    else:
        modes = [(ci, "logit"), (None, "softmax_ce")]
        res = compare_preact(cfg, p, x, [(ref, FP32_TOL, FP32_CONV_TAU), (eng, tau, conv_tau)], modes)
        for rr, t in zip(res, (FP32_TOL, tol)):
            for r in rr:
                assert r["mask_violations"] == 0 and r["conv_mask_violations"] == 0 and r["cls_equal"].all()
                assert r["heat_err"].max() <= t, f"heat-map err {r['heat_err'].max()} (tol {t})"
    want = _np(ref.predict_explain(x, ci, "logit")[3])
    eng.set_explain_target("conv")
    post = _np(eng.predict_explain(x, ci, "logit")[3])
    assert np.abs(post - want).max() > 1e-2                            # the two targets really differ
    ref.close()
    eng.close()


def _assert_classes_equal_single(eng, x, classes, mode, out_hw=None):
    cls, probs, logits, heat = eng.predict_explain_classes(x, classes, mode, out_hw=out_hw)
    B, K = heat.shape[:2]
    cols = np.broadcast_to(np.asarray(classes, np.int32), (B, K)) if classes is not None else np.tile(np.arange(K, dtype=np.int32), (B, 1))
    for k in range(K):
        c1, p1, l1, h1 = eng.predict_explain(x, cols[:, k].copy(), mode, out_hw=out_hw)
        assert torch.equal(heat[:, k], h1), f"class column {k} differs"
        assert torch.equal(cls, c1) and torch.equal(logits, l1)
    return heat


@pytest.mark.parametrize("precision,mb", [("fp16", 64), ("fp16x3", 48), ("fp16", 16)])
def test_bitwise_contracts_under_the_pre_activation_target(precision, mb):
    """K-class columns == single-class calls (K = 1, 2, 3, duplicates, [B,K]); a call of 70 images == its max_batch chunks called one
    by one; host call == device call.
    max_batch 16 takes the two-launch tail."""
    cfg = ocnn.NetConfig.torch_flavour((64, 64, 1), 2, [(32, 3), (64, 3)], [128, 32], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    B = 70
    x = ocnn.synth_images(B, (64, 64, 1), seed=5)
    eng = engine_from(cfg, p, precision=precision, max_batch=mb)
    eng.set_explain_target(PRE)
    rng = np.random.default_rng(3)
    for mode in ("logit", "softmax_ce"):
        for classes in (rng.integers(0, 2, size=(B, 1)), (0, 1), (1, 0, 1), rng.integers(0, 2, size=(B, 3)), None):
            _assert_classes_equal_single(eng, x, classes, mode)
    ci = (np.arange(B) % 2).astype(np.int32)
    whole = eng.predict_explain(x, ci, "logit")[3]
    for b0 in range(0, B, mb):
        part = eng.predict_explain(x[b0:b0 + mb], ci[b0:b0 + mb], "logit")[3]
        assert torch.equal(part, whole[b0:b0 + mb]), "chunked != unchunked"
    hc, hp, hl, hh = eng.predict_explain_host(x, ci, "logit")
    assert np.array_equal(hh, _np(whole)), "host call != device call"
    eng.close()


def _imgs(B, h, w, seed):
    """8-bit grey images with structure plus pixel noise (as test_gpu_overlays_classes_host.py)."""
    rng = np.random.default_rng(seed)
    base = ocnn.synth_images(B, (h, w, 1), seed=seed, kind="mammo")[..., 0]
    base = (base - base.min()) / (base.max() - base.min() + 1e-12)
    return np.clip(base * 200 + rng.integers(0, 56, size=(B, h, w)), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("img_hw", [(512, 512), (300, 260)])
def test_overlays_classes_host_equals_device_composition(img_hw):
    from bcad_b200 import engine as E
    import bcad_b200.GRADCAM as G
    cfg, p = _canonical()
    eng = engine_from(cfg, p, precision="fp16", max_batch=64)
    imgs = _imgs(37, *img_hw, seed=2)
    eng.set_explain_target(PRE)
    cls, probs, logits, ov, hu = eng.gradcam_overlays_classes_host(imgs, (0, 1), "logit", True)
    h, w, c = eng.spec.input_shape
    g = torch.from_numpy(imgs).cuda()
    xd = E.gray_resize_preprocess(g, (h, w), c, True)
    _, _, _, heat = eng.predict_explain_classes(xd, (0, 1), "logit", out_hw=img_hw)
    ovd, hud = E.overlay_classes(g, heat)
    assert np.array_equal(ov, _np(ovd)) and np.array_equal(hu, _np(hud))
    eng.set_explain_target("conv")
    post_hu = eng.gradcam_overlays_classes_host(imgs, (0, 1), "logit", True)[4]
    assert not np.array_equal(post_hu, hu)

    class M:                                                             # the GRADCAM mirror's keyword sets and restores the target
        engine = eng
        fast_engine = None
    c2, p2, ov2, hu2 = G.generate_dual_class_gradcam_overlays_batch(imgs, [0, 1], model=M, target=PRE)
    assert np.array_equal(hu2, hu) and np.array_equal(ov2, ov)
    assert eng.explain_target == "conv"
    assert np.array_equal(G.generate_dual_class_gradcam_overlays_batch(imgs, [0, 1], model=M)[3], post_hu)
    eng.close()


def test_refinement_twin_explains_the_same_target():
    """refine_margin 1e3 flags every image: all maps come from the fp16x3 twin and must match an fp16x3 handle."""
    cfg = ocnn.NetConfig.torch_flavour((64, 64, 1), 2, [(32, 3), (64, 3)], [64, 32], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    B = 24
    x = ocnn.synth_images(B, (64, 64, 1), seed=12)
    ci = (np.arange(B) % 2).astype(np.int32)
    eng = engine_from(cfg, p, precision="fp16", max_batch=64, refine_margin=1e3, refine_capacity=B)
    x3 = engine_from(cfg, p, precision="fp16x3", max_batch=64)
    post = _np(eng.predict_explain(x, ci, "logit")[3])
    eng.set_explain_target(PRE)
    x3.set_explain_target(PRE)
    r0 = eng.refine_stats()[0]
    got = _np(eng.predict_explain(x, ci, "logit")[3])
    assert eng.refine_stats()[0] - r0 == B
    want = _np(x3.predict_explain(x, ci, "logit")[3])
    assert np.abs(got - want).max() <= X3_TOL
    assert np.abs(got - post).max() > 1e-2
    eng.close()
    x3.close()


@pytest.mark.parametrize("precision", ["fp16", "fp16x3"])
def test_target_switching_leaves_no_state(precision):
    cfg = ocnn.NetConfig.torch_flavour((64, 64, 1), 2, [(32, 3), (64, 3)], [64, 32], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    x = ocnn.synth_images(20, (64, 64, 1), seed=8)
    eng = engine_from(cfg, p, precision=precision, max_batch=32)
    before = eng.predict_explain_classes(x, (0, 1), "softmax_ce")
    eng.set_explain_target(PRE)
    eng.predict_explain_classes(x, (0, 1), "softmax_ce")
    eng.predict_explain(x, None, "logit")
    eng.set_explain_target("conv")
    after = eng.predict_explain_classes(x, (0, 1), "softmax_ce")
    for a, b in zip(before, after):
        assert torch.equal(a, b)
    eng.close()


def test_refusals_name_the_fp32_path():
    from util import spec_from_cfg
    import bcad_b200
    cfg = ocnn.NetConfig.torch_flavour((32, 32, 1), 2, [(32, 3), (64, 3)], [96, 16], 0.01)          # 96 units: not a multiple of 64
    for precision in ("fp16", "fp16x3"):
        eng = bcad_b200.Engine(spec_from_cfg(cfg), precision=precision)
        with pytest.raises(ValueError, match="fp32 path"):
            eng.set_explain_target(PRE)
        eng.close()
    cfg = dataclasses.replace(ocnn.NetConfig.torch_flavour((32, 32, 1), 2, [(32, 3), (64, 3)], [64, 16]), alpha_conv=0.0)
    eng = bcad_b200.Engine(spec_from_cfg(cfg), precision="fp16")
    with pytest.raises(ValueError, match="fp32 path"):
        eng.set_explain_target(PRE)
    eng.close()


def test_sharded_equals_one_gpu():
    import bcad_b200
    from util import spec_from_cfg
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"ShardedEngine needs two or more GPUs, {n} visible")
    cfg, p = _canonical()
    single = engine_from(cfg, p, precision="fp16", max_batch=64)
    single.set_explain_target(PRE)
    imgs = _imgs(37, 300, 260, seed=8)
    want = single.gradcam_overlays_classes_host(imgs, (0, 1))
    sh = bcad_b200.ShardedEngine(spec_from_cfg(cfg), list(range(min(n, 4))), precision="fp16", max_batch=64)
    sh.set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
    sh.set_explain_target(PRE)
    got = sh.gradcam_overlays_classes_host(imgs, (0, 1))
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    sh.close()
    single.close()
