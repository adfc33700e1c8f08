"""Pin the oracle to the reference's own outputs (tests/golden/*.npz, made by make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import cnn as ocnn
from oracle import gradcam as ogc

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _numpy_case(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    cfg = ocnn.NetConfig.numpy_flavour(tuple(int(v) for v in g["input_shape"]), 2,
                                       [tuple(int(a) for a in r) for r in g["conv_layers"]],
                                       [int(v) for v in g["hidden"]], float(g["alpha"]))
    n_conv = len(cfg.conv_layers)
    conv_idx = [2 * i for i in range(n_conv)]                       # layers index incl. pools
    dense_idx = [2 * n_conv + j for j in range(len(cfg.hidden_units) + 1)]
    p = ocnn.Params([g[f"W{i}"] for i in conv_idx], [g[f"b{i}"] for i in conv_idx],
                    [g[f"W{i}"] for i in dense_idx], [g[f"b{i}"] for i in dense_idx])
    return g, cfg, p, conv_idx, dense_idx


@pytest.mark.parametrize("name", ["ref_numpy_small", "ref_numpy_odd", "ref_numpy_ties", "ref_numpy_k5"])
def test_numpy_flavour_forward_and_explain(name):
    g, cfg, p, conv_idx, dense_idx = _numpy_case(name)
    cache = ocnn.forward(cfg, p, g["x"])
    tol = dict(rtol=0, atol=1e-11)
    np.testing.assert_allclose(cache.probs[0].numpy(), g["probs"], **tol)
    assert int(cache.probs[0].argmax()) == int(g["pred_class"])
    for bi, li in enumerate(conv_idx):
        np.testing.assert_allclose(cache.conv_out[bi][0].numpy(), g[f"conv_out{li}"], **tol)
        np.testing.assert_allclose(cache.pool_out[bi][0].numpy(), g[f"pool_out{li + 1}"], **tol)
        assert np.array_equal(cache.switches[bi][0].numpy() > 0, g[f"switches{li + 1}"])
    for j, li in enumerate(dense_idx):
        np.testing.assert_allclose(cache.z[j][0].numpy(), g[f"z{li}"], **tol)
    for c in (0, 1):
        d_top = ocnn.top_gradient(cache, c, "softmax_ce")
        cag, d_input, wg = ocnn.backward(cfg, p, cache, d_top, want_wgrads=True)
        np.testing.assert_allclose(d_input[0].numpy(), g[f"d_input_c{c}"], **tol)
        for bi, li in enumerate(conv_idx):
            np.testing.assert_allclose(cag[bi][0].numpy(), g[f"conv_act_grads{li}_c{c}"], **tol)
            np.testing.assert_allclose(wg["conv"][bi][0][0].numpy(), g[f"grad{li}_dF_c{c}"], **tol)
            np.testing.assert_allclose(wg["conv"][bi][1][0].numpy(), g[f"grad{li}_db_conv_c{c}"], **tol)
        for j, li in enumerate(dense_idx):
            np.testing.assert_allclose(wg["dense"][j][0][0].numpy(), g[f"grad{li}_dW_c{c}"], **tol)
            np.testing.assert_allclose(wg["dense"][j][1][0].numpy(), g[f"grad{li}_db_c{c}"], **tol)
        sal, _ = ogc.saliency_map(d_input[0].numpy())
        np.testing.assert_allclose(sal, g[f"saliency_c{c}"], **tol)


def test_ties_fixture_really_has_ties():
    g, cfg, p, conv_idx, _ = _numpy_case("ref_numpy_ties")
    sw = g[f"switches{conv_idx[0] + 1}"]
    h2, w2 = sw.shape[0] // 2, sw.shape[1] // 2
    per_window = sw[:2 * h2, :2 * w2].reshape(h2, 2, w2, 2, -1).sum(axis=(1, 3))
    assert per_window.max() == 4 and per_window.min() >= 1


def _torch_case(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    cfg = ocnn.NetConfig.torch_flavour(tuple(int(v) for v in g["input_shape"]), 2,
                                       [tuple(int(a) for a in r) for r in g["conv_layers"]],
                                       [int(v) for v in g["hidden"]], float(g["alpha"]))
    n_conv, n_dense = len(cfg.conv_layers), len(cfg.hidden_units) + 1
    p = ocnn.Params([g[f"sd.convs.{i}.weight"].transpose(0, 2, 3, 1) for i in range(n_conv)],
                    [g[f"sd.convs.{i}.bias"] for i in range(n_conv)],
                    [g[f"sd.fc.{3 * j}.weight"] for j in range(n_dense)],
                    [g[f"sd.fc.{3 * j}.bias"] for j in range(n_dense)])
    return g, cfg, p


@pytest.mark.parametrize("name", ["ref_torch_small", "ref_torch_odd"])
def test_torch_flavour_forward_and_gradients(name):
    g, cfg, p = _torch_case(name)
    cache = ocnn.forward(cfg, p, g["x"])                       # fp64 oracle vs fp32 reference
    np.testing.assert_allclose(cache.logits.numpy(), g["logits"], rtol=0, atol=2e-6)
    np.testing.assert_allclose(cache.probs.numpy(), g["probs"], rtol=0, atol=2e-6)
    assert np.array_equal(cache.logits.argmax(dim=1).numpy(), g["pred_class"])
    np.testing.assert_allclose(cache.conv_out[-1].permute(0, 3, 1, 2).numpy(), g["A_last"], rtol=0, atol=2e-6)
    for c in (0, 1):
        cag, _, _ = ocnn.backward(cfg, p, cache, ocnn.top_gradient(cache, c, "logit"))
        for i in range(len(cfg.conv_layers)):
            np.testing.assert_allclose(cag[i].permute(0, 3, 1, 2).numpy(), g[f"dA{i}_logit_c{c}"],
                                       rtol=0, atol=2e-6)


def test_state_dict_converter_roundtrip():
    """NumPy-layout params (HWC fc1 columns) -> ADCNNM state_dict -> same function."""
    cfg_np = ocnn.NetConfig((10, 12, 2), 2, [(3, 3), (4, 3)], [5], 0.01, 0.01, 1, "hwc", "first", "logits")
    p = ocnn.init_params(cfg_np, seed=5, bias_std=0.1)
    sd = ocnn.params_to_state_dict(cfg_np, p)
    cfg_t = ocnn.NetConfig.torch_flavour((10, 12, 2), 2, [(3, 3), (4, 3)], [5])
    p_t = ocnn.Params([sd[f"convs.{i}.weight"].numpy().transpose(0, 2, 3, 1) for i in range(2)],
                      [sd[f"convs.{i}.bias"].numpy() for i in range(2)],
                      [sd[f"fc.{3 * j}.weight"].numpy() for j in range(2)],
                      [sd[f"fc.{3 * j}.bias"].numpy() for j in range(2)])
    x = ocnn.synth_images(3, (10, 12, 2), seed=1)
    a = ocnn.forward(cfg_np, p, x).logits.numpy()
    b = ocnn.forward(cfg_t, p_t, x).logits.numpy()
    np.testing.assert_allclose(a, b, rtol=0, atol=1e-6)


def test_bilinear_equals_cv2_fixture():
    g = np.load(os.path.join(GOLDEN, "cv2_resize.npz"))
    i = 0
    while f"src{i}" in g:
        dst = g[f"dst{i}"]
        got = ogc.bilinear_resize(g[f"src{i}"], dst.shape[0], dst.shape[1])
        np.testing.assert_allclose(got, dst, rtol=0, atol=1.3e-7)   # <= 1 ulp at 1.0
        i += 1
    assert i >= 6


def test_jet_lut_fixture():
    lut = ogc.jet_lut_bgr()
    assert lut.shape == (256, 3) and lut.dtype == np.uint8
    assert lut[0].tolist() == [128, 0, 0] and lut[255].tolist() == [0, 0, 128]      # SURVEY P12


def test_tail_known_answers():
    """Known-answer micro-tests the reference lacks (SURVEY section 4)."""
    rng = np.random.default_rng(0)
    A = rng.standard_normal((2, 4, 6, 6)).astype(np.float32)
    # constant map: min == max => 0/(1e-7) path => all zeros
    out = ogc.gradcam_tail(np.ones_like(A), np.ones_like(A), (12, 12))
    assert np.all(out == 0)
    # all-negative cam => ReLU => zeros
    out = ogc.gradcam_tail(np.abs(A), -np.ones_like(A), (12, 12))
    assert np.all(out == 0)
    # generic: range [0,1], max hits ~1 after the second normalisation
    out = ogc.gradcam_tail(A, rng.standard_normal(A.shape).astype(np.float32), (12, 12))
    assert out.dtype == np.float32 and out.min() == 0 and abs(out.max() - 1) < 1e-5


@pytest.mark.parametrize("name", ["ref_numpy_small", "ref_numpy_odd", "ref_numpy_ties", "ref_numpy_k5"])
def test_oracle_predict_against_reference_fixture(name):
    """oracle.cnn.predict vs the reference's own ``CNNModel.predict`` (class, probs) as make_golden.py recorded it."""
    g, cfg, p, _, _ = _numpy_case(name)
    c, pr, _ = ocnn.predict(cfg, p, g["x"])
    assert int(c[0]) == int(g["pred_class"])
    np.testing.assert_allclose(pr[0], g["probs"], rtol=0, atol=1e-12)


def test_cpu_port_matches_reference_fixture():
    """oracle.cpu_port (the timed CPU baseline) reproduces the reference ADCNNM logits and gradients."""
    from oracle import cpu_port
    g, cfg, p = _torch_case("ref_torch_small")
    model = cpu_port.build(cfg, p)
    x = torch.from_numpy(g["x"])
    cls, logits, heat = cpu_port.predict_gradcam(model, x, class_idx=[0, 0, 0])
    np.testing.assert_allclose(logits, g["logits"], rtol=0, atol=1e-6)
    assert np.array_equal(cls, g["pred_class"])
    want = ogc.gradcam_tail(g["A_last"], g["dA1_logit_c0"], (16, 16))
    np.testing.assert_allclose(heat, want, rtol=0, atol=2e-6)


@pytest.mark.parametrize("name,c", [("ref_unet_small", 1), ("ref_unet_odd", 2)])
def test_unet_oracle_matches_reference_fixture(name, c):
    """oracle.unet vs Classes/unet.py outputs (padded-size 'same' conv quirk, pools, kernel stream order)."""
    from oracle import unet as ou
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    ks = ou.draw_kernels(c, int(g["seed"]))
    c1 = ou.conv2d_same_quirk(g["x"], ks[0])
    assert c1.shape == g["c1"].shape == (g["x"].shape[0], g["x"].shape[1] + 2, g["x"].shape[2] + 2, 16)
    assert np.all(c1[:, -2:] == 0) and np.all(c1[:, :, -2:] == 0)            # the quirk: trailing rows/cols are zero
    np.testing.assert_allclose(c1, g["c1"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(ou.max_pool(ou.relu(c1)), g["p1"], rtol=0, atol=1e-12)
    bn = ou.tiny_unet(g["x"], ks)
    np.testing.assert_allclose(bn, g["bn"], rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(ou.average_pool(bn, 3), g["avg3"], rtol=1e-12, atol=1e-9)


def test_training_oracle_matches_reference_fixture():
    """oracle.train (mean gradients, SGD + per-tensor clip) vs the reference's _compute_sample_grads / _apply_grads."""
    from oracle import train as otr
    g = np.load(os.path.join(GOLDEN, "ref_numpy_train.npz"))
    cfg = ocnn.NetConfig.numpy_flavour((12, 12, 2), 2, [(3, 3), (4, 3)], [6, 5], 0.01)
    p = ocnn.Params([g["W0"], g["W2"]], [g["b0"], g["b2"]], [g["W4"], g["W5"], g["W6"]], [g["b4"], g["b5"], g["b6"]])
    gr, loss = otr.mean_grads(cfg, p, g["X"], g["labels"])
    np.testing.assert_allclose(loss, g["losses"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(gr["conv_w"][0], g["grad0_dF"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(gr["conv_w"][1], g["grad2_dF"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(gr["conv_b"][1], g["grad2_db_conv"], rtol=0, atol=1e-12)
    for j, li in enumerate((4, 5, 6)):
        np.testing.assert_allclose(gr["dense_w"][j], g[f"grad{li}_dW"], rtol=0, atol=1e-12)
    assert max(np.linalg.norm(x) for x in gr["conv_w"] + gr["dense_w"]) > 5.0          # the clip branch is exercised
    newp = otr.sgd_clip_step(p, gr, float(g["lr"]))
    np.testing.assert_allclose(newp.conv_w[1], g["newW2"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(newp.dense_w[0], g["newW4"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(newp.dense_b[2], g["newb6"], rtol=0, atol=1e-12)


def test_training_oracle_dropout_matches_reference_fixture():
    """forward(training=True) with dropout + _compute_sample_grads: the reference's backward does NOT mask the gradient."""
    from oracle import train as otr
    g = np.load(os.path.join(GOLDEN, "ref_numpy_train_dropout.npz"))
    cfg = ocnn.NetConfig.numpy_flavour((12, 12, 2), 2, [(3, 3), (4, 3)], [8, 6], 0.01)
    p = ocnn.Params([g["W0"], g["W2"]], [g["b0"], g["b2"]], [g["W4"], g["W5"], g["W6"]], [g["b4"], g["b5"], g["b6"]])
    mk = g["dropout_masks"]
    gr, loss = otr.mean_grads(cfg, p, g["X"], g["labels"], dropout=[mk[:, :8], mk[:, 8:]], dropout_in_backward=False)
    np.testing.assert_allclose(loss, g["losses"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(gr["conv_w"][0], g["grad0_dF"], rtol=0, atol=1e-12)
    for j, li in enumerate((4, 5, 6)):
        np.testing.assert_allclose(gr["dense_w"][j], g[f"grad{li}_dW"], rtol=0, atol=1e-12)
    masked, _ = otr.mean_grads(cfg, p, g["X"], g["labels"], dropout=[mk[:, :8], mk[:, 8:]], dropout_in_backward=True)
    assert np.abs(masked["dense_w"][0] - g["grad4_dW"]).max() > 1e-3       # the autograd rule is a different function


def test_bottleneck_resize_oracle_matches_reference_fixture():
    """oracle.gradcam.process_bottleneck_features vs the reference's app.py:466-489 (cv2's > 4-channel float32-coordinate path
    and the <= 4-channel double-coordinate path are different arithmetic; both pinned)."""
    from oracle import gradcam as ogc
    g = np.load(os.path.join(GOLDEN, "ref_bottleneck.npz"))
    for i, rs in enumerate([(8, 8), (11, 7), (9, 10)]):
        assert np.array_equal(ogc.process_bottleneck_features(g[f"feat{i}"], rs), g[f"out{i}"])
