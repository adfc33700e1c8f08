"""Grad-CAM for several target classes per image from one forward (bcad_predict_explain_classes / Engine.predict_explain_classes).

The contract is bit-identity: ``heat[:, k]``, logits, probabilities and classes equal what ``predict_explain`` returns on the same
handle with class column k, on every path (fp32, fp16x3, fp16 with and without refinement, both pool tie rules, both grad modes,
fused and two-launch tails, chunked batches, resized heat-maps)."""
import ctypes as C

import numpy as np
import pytest
import torch

from util import engine_from, oracle_heatmaps, ocnn

pytestmark = pytest.mark.gpu

X3_HEAT_TOL = 5e-4          # the fp16x3 path's heat-map tolerance against the float64 oracle (test_gpu_tensor_path.py)


def _cols(classes, B, K):
    if classes is None:
        return np.tile(np.arange(K, dtype=np.int32), (B, 1))
    c = np.asarray(classes, dtype=np.int32)
    return np.broadcast_to(c, (B, K)) if c.ndim == 1 else c


def _assert_matches_single_class_calls(eng, x, classes, mode, out_hw=None):
    cls, probs, logits, heat = eng.predict_explain_classes(x, classes, mode, out_hw=out_hw)
    B, K = heat.shape[:2]
    cols = _cols(classes, B, K)
    for k in range(K):
        c1, p1, l1, h1 = eng.predict_explain(x, cols[:, k].copy(), mode, out_hw=out_hw)
        assert torch.equal(heat[:, k], h1), f"class column {k}: heat-maps differ on images {torch.nonzero((heat[:, k] != h1).flatten(1).any(1)).flatten().tolist()}"
        assert torch.equal(logits, l1) and torch.equal(probs, p1) and torch.equal(cls, c1), f"class column {k}: forward outputs differ"
    return cls, probs, logits, heat


def _class_sets(B, nc, seed):
    rng = np.random.default_rng(seed)
    return [rng.integers(0, nc, size=(B, 1)),                      # K = 1, per image
            (0, 1),                                                # the deployed dual-class call
            rng.integers(0, nc, size=(B, 3)),                      # K = 3: duplicates within rows
            None]                                                  # every class


TORCH = ("torch", (64, 64, 1), [64, 32])
NUMPY = ("numpy", (48, 48, 1), [48, 16])


@pytest.mark.parametrize("flavour,precision,refine,B,mb", [
    (TORCH, "fp32", None, 20, 8),             # fp32 path, chunked
    (TORCH, "fp16x3", None, 70, 48),          # fused K-class tail on split operands, chunked
    (TORCH, "fp16", None, 70, 64),            # the headline handle (refinement on), chunked
    (TORCH, "fp16", 0.0, 140, 256),           # refinement off, B not a multiple of 128
    (TORCH, "fp16", None, 20, 16),            # max_batch <= 32: the two-launch tail
    (NUMPY, "fp32", None, 6, 8),              # tie-duplicating rule, exact-zero background
    (NUMPY, "fp16x3", None, 40, 48),
])
def test_classes_equal_single_class_calls(flavour, precision, refine, B, mb):
    kind, shape, hidden = flavour
    if kind == "torch":
        cfg = ocnn.NetConfig.torch_flavour(shape, 2, [(32, 3), (64, 3)], hidden, 0.01)
        x = ocnn.synth_images(B, shape, seed=5)
    else:
        cfg = ocnn.NetConfig.numpy_flavour(shape, 2, [(32, 3), (64, 3)], hidden, 0.01)
        x = ocnn.synth_images(B, shape, seed=31, kind="mammo")
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    kw = {} if refine is None else {"refine_margin": refine}
    eng = engine_from(cfg, p, precision=precision, max_batch=mb, **kw)
    for mode in ("logit", "softmax_ce"):
        for classes in _class_sets(B, 2, seed=len(mode)):
            _assert_matches_single_class_calls(eng, x, classes, mode)
    eng.close()


def test_classes_canonical_network_resized_heatmaps():
    """The canonical 256x256 network on the headline handle, heat-maps scaled to 512x512 (the deployed call's image size)."""
    cfg = ocnn.NetConfig.torch_flavour((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.0)
    x = ocnn.synth_images(6, (256, 256, 1), seed=20251018)
    eng = engine_from(cfg, p, precision="fp16", max_batch=64)
    _, _, _, heat = _assert_matches_single_class_calls(eng, x, (0, 1), "logit", out_hw=(512, 512))
    assert heat.shape == (6, 2, 512, 512)
    _assert_matches_single_class_calls(eng, x, None, "softmax_ce")
    eng.close()


def test_classes_pre_activation_target_on_fp32():
    cfg = ocnn.NetConfig.torch_flavour((40, 40, 1), 2, [(16, 3), (32, 3)], [32], 0.01)
    p = ocnn.init_params(cfg, seed=3, bias_std=0.05)
    x = ocnn.synth_images(5, (40, 40, 1), seed=9)
    eng = engine_from(cfg, p, precision="fp32", max_batch=8)
    eng.set_explain_target("conv_preact")
    for mode in ("logit", "softmax_ce"):
        _assert_matches_single_class_calls(eng, x, np.array([[0, 1, 1]] * 5), mode)
    eng.close()


def test_classes_refinement_twin_runs_once_per_chunk():
    """A huge margin flags every image; a capacity of 3 refines some and lets the rest overflow.  The maps stay bit-identical and
    the refinement counters grow by what ONE single-class call of the batch adds (the flag does not depend on the class)."""
    cfg = ocnn.NetConfig.torch_flavour((64, 64, 1), 2, [(32, 3), (64, 3)], [64, 32], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    x = ocnn.synth_images(10, (64, 64, 1), seed=12)
    eng = engine_from(cfg, p, precision="fp16", max_batch=64, refine_margin=1e3, refine_capacity=3)
    r0 = eng.refine_stats()
    eng.predict_explain(x, np.zeros(10, np.int32), "logit")
    r1 = eng.refine_stats()
    eng.predict_explain_classes(x, (0, 1), "logit")
    r2 = eng.refine_stats()
    assert (r1[0] - r0[0], r1[1] - r0[1]) == (3, 7)
    assert (r2[0] - r1[0], r2[1] - r1[1]) == (r1[0] - r0[0], r1[1] - r0[1])
    for mode in ("logit", "softmax_ce"):
        _assert_matches_single_class_calls(eng, x, np.array([[1, 0, 1]] * 10), mode)
        _assert_matches_single_class_calls(eng, x, (0, 1), mode, out_hw=(100, 90))
    eng.close()


def test_classes_one_forward_per_chunk():
    """Profiled K = 2 call on the canonical fp16 handle: one conv launch per chunk, one K-class tail launch per chunk."""
    cfg = ocnn.NetConfig.torch_flavour((256, 256, 1), 2, [(32, 3), (64, 3)], [256, 128], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.0)
    x = torch.from_numpy(ocnn.synth_images(256, (256, 256, 1), seed=4)).cuda()
    eng = engine_from(cfg, p, precision="fp16", max_batch=128)
    eng.set_profiling(True)
    eng.predict_explain_classes(x, (0, 1), "logit")
    names = [n for n, _ in eng.last_profile()]
    eng.set_profiling(False)
    assert sum(n.startswith("conv") for n in names) == 2, names            # two chunks of 128
    assert names.count("conv01_fused_tcgen05") == 2, names
    assert names.count("tail_fused_classes") == 2 and "tail_fused" not in names, names
    eng.close()


def test_classes_against_the_oracle():
    cfg = ocnn.NetConfig.torch_flavour((64, 64, 1), 2, [(32, 3), (64, 3)], [64, 32], 0.01)
    p = ocnn.init_params(cfg, seed=7, bias_std=0.05)
    x = ocnn.synth_images(40, (64, 64, 1), seed=21)
    eng = engine_from(cfg, p, precision="fp16x3", max_batch=64)
    cls, probs, logits, heat = eng.predict_explain_classes(x, (0, 1), "logit")
    for k in (0, 1):
        o_cls, cache, A, dA, o_heat = oracle_heatmaps(cfg, p, x, np.full(40, k), "logit")
        assert np.array_equal(cls.cpu().numpy(), o_cls)
        assert np.abs(heat[:, k].cpu().numpy() - o_heat).max() <= X3_HEAT_TOL
    eng.close()


def test_dual_class_overlays_batch_equals_class_by_class_calls():
    from bcad_b200 import ADCNNM as A, GRADCAM as G
    shape, convs, hidden, B = (64, 48, 1), [(32, 3), (64, 3)], [32, 16], 70
    cfg = ocnn.NetConfig.torch_flavour(shape, 2, convs, hidden, 0.01)
    p = ocnn.init_params(cfg, seed=6, bias_std=0.05)
    model = A.CNNModel(shape, 2, conv_layers=convs, hidden_units=hidden, max_batch=64).eval()
    model.load_state_dict(ocnn.params_to_state_dict(cfg, p))
    imgs = np.random.default_rng(3).integers(0, 256, size=(B,) + shape[:2], dtype=np.uint8)
    for standardise in (True, False):
        cls, probs, ov, hu = G.generate_dual_class_gradcam_overlays_batch(imgs, [0, 1], model=model, standardise=standardise)
        assert ov.shape == (B, 2) + shape[:2] + (3,) and hu.shape == (B, 2) + shape[:2] and ov.dtype == hu.dtype == np.uint8
        for k in (0, 1):
            c1, p1, ov1, hu1 = G.generate_gradcam_overlays_batch(imgs, k, model=model, standardise=standardise)
            assert np.array_equal(cls, c1) and np.array_equal(probs, p1)
            assert np.array_equal(ov[:, k], ov1) and np.array_equal(hu[:, k], hu1)
    x = torch.from_numpy((imgs / 255.0).astype(np.float32)[..., None]).cuda()
    c, lg, heat = model.predict_explain_classes_batch(x, (1, 0))
    for k, ck in enumerate((1, 0)):
        c1, l1, h1 = model.predict_explain_batch(x, np.full(B, ck))
        assert torch.equal(heat[:, k], h1) and torch.equal(lg, l1) and torch.equal(c, c1)


def test_numpy_mirror_classes_batch():
    from bcad_b200 import CNNModel as M
    cfg = ocnn.NetConfig.numpy_flavour((48, 48, 1), 2, [(32, 3), (64, 3)], [48, 16], 0.01)
    p = ocnn.init_params(cfg, seed=11, bias_std=0.05)
    x = ocnn.synth_images(9, (48, 48, 1), seed=2, kind="mammo")
    eng = engine_from(cfg, p, precision="fp32", max_batch=16)
    model = M.CNNModel.__new__(M.CNNModel)
    model._batch_engine = lambda: eng
    cls, probs, heat = model.predict_explain_classes_batch(x, (0, 1))
    assert heat.shape == (9, 2, 48, 48) and cls.dtype == np.int64
    for k in (0, 1):
        c1, p1, l1, h1 = eng.predict_explain(x, np.full(9, k, np.int32), "softmax_ce")
        assert np.array_equal(heat[:, k], h1.cpu().numpy()) and np.array_equal(probs, p1.cpu().numpy())
    eng.close()


def test_classes_errors():
    from bcad_b200 import _lib
    cfg = ocnn.NetConfig.torch_flavour((32, 32, 1), 2, [(32, 3), (64, 3)], [32], 0.01)
    p = ocnn.init_params(cfg, seed=1, bias_std=0.05)
    B = 4
    x = torch.from_numpy(ocnn.synth_images(B, (32, 32, 1), seed=1)).cuda()
    eng = engine_from(cfg, p, precision="fp32", max_batch=8, keep_all_activations=True)
    lib, h, s = eng.lib, eng._h, eng._stream()
    heat = torch.empty((B, 9, 32, 32), device="cuda")
    ci = torch.zeros((B, 9), dtype=torch.int32, device="cuda")

    def call(K, classes, out, oh=0, ow=0):
        return lib.bcad_predict_explain_classes(h, C.c_void_p(x.data_ptr()), B, K, classes, 0, None, None, None, oh, ow, out, s)

    hp, cp = C.c_void_p(heat.data_ptr()), C.c_void_p(ci.data_ptr())
    assert call(0, cp, hp) == _lib.ERR_INVALID
    assert call(9, cp, hp) == _lib.ERR_INVALID
    assert call(3, None, hp) == _lib.ERR_INVALID                     # classes 0..2 of a 2-class model
    assert call(2, cp, None) == _lib.ERR_INVALID
    assert call(2, cp, hp, 0, 16) == _lib.ERR_INVALID
    assert call(2, None, hp) == _lib.OK
    torch.cuda.synchronize()
    buf = torch.empty((B, 64), device="cuda")
    for kind in (_lib.T_ALPHA, _lib.T_CAM_LOWRES):
        assert lib.bcad_get_tensor(h, kind, 0, B, C.c_void_p(buf.data_ptr()), s) == _lib.ERR_STATE
    assert lib.bcad_get_tensor(h, _lib.T_DENSE_Z, 0, B, C.c_void_p(buf.data_ptr()), s) == _lib.OK
    eng.predict_explain(x, None, "logit")                           # a single-class call makes the caches valid again
    assert lib.bcad_get_tensor(h, _lib.T_ALPHA, 0, B, C.c_void_p(buf.data_ptr()), s) == _lib.OK
    eng.set_dropout_masks(np.ones((B, 32), np.float32))
    assert call(2, cp, hp) == _lib.ERR_INVALID
    eng.set_dropout_masks(None)
    with pytest.raises(ValueError, match="out of range"):
        eng.predict_explain_classes(x, (0, 2))
    with pytest.raises(ValueError, match="out of range"):
        eng.predict_explain_classes(x, np.full((B, 2), -1))
    with pytest.raises(ValueError):
        eng.predict_explain_classes(x, [0] * 9)
    with pytest.raises(ValueError):
        eng.predict_explain_classes(x, np.zeros((B + 1, 2)))
    torch.cuda.synchronize()
    eng.close()
