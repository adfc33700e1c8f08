"""The chunk schedule of the host-buffer calls and the multi-GPU driver's fan-out, on one GPU.

A single-class host-buffer call runs its batch in chunks of a quarter of the batch, rounded up to a multiple of 32, between 32 images
and a cap: 64 for float32 images, 128 for 8-bit pixels and grey images.  Each chunk is one device-buffer predict + Grad-CAM of that many
images, so a call's launch count is the sum of those of device calls of its chunk sizes.  ShardedEngine's fan-out runs on two engines
of the same GPU here, so that a one-GPU box exercises it too."""
import numpy as np
import pytest

from util import engine_from, ocnn, spec_from_cfg

pytestmark = pytest.mark.gpu

SHAPE = (64, 48, 1)

# B -> (chunks of a float32-input call, chunks of an 8-bit-input call) on a handle with max_batch=128
SCHEDULE = {
    512: ([64] * 8, [128] * 4),
    200: ([64, 64, 64, 8], [64, 64, 64, 8]),
    40: ([32, 8], [32, 8]),
    1: ([1], [1]),
}


def _net(seed=3):
    cfg = ocnn.NetConfig.torch_flavour(SHAPE, 2, [(32, 3), (64, 3)], [32, 16], 0.01)
    return cfg, ocnn.init_params(cfg, seed=seed, bias_std=0.05)


def _grey(B, h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, size=(B, h, w), dtype=np.uint8)


def test_chunk_schedule(monkeypatch):
    monkeypatch.delenv("BCAD_HOST_CHUNK", raising=False)
    cfg, p = _net()
    eng = engine_from(cfg, p, precision="fp16", max_batch=128)
    x = ocnn.synth_images(max(SCHEDULE), SHAPE, seed=5)
    x8 = np.clip(np.rint(x * 255.0), 0, 255).astype(np.uint8)
    calls = {
        "float32": lambda B: eng.predict_explain_host(x[:B], None, "logit"),
        "uint8": lambda B: eng.predict_explain_host(x8[:B], None, "logit", heat_dtype=np.uint8),
        "grey": lambda B: eng.gradcam_overlays_host(x8[:B, ..., 0], None, "logit"),
    }
    per_chunk = {}

    def device_launches(n):                     # launches of one device-buffer call of n images
        if n not in per_chunk:
            eng.predict_explain(x[:n], None, "logit")
            before = eng.launch_count
            eng.predict_explain(x[:n], None, "logit")
            per_chunk[n] = eng.launch_count - before
        return per_chunk[n]

    for call in calls.values():                  # first use allocates the slots
        call(1)
    for B, (f32_chunks, u8_chunks) in SCHEDULE.items():
        for name, call in calls.items():
            chunks = f32_chunks if name == "float32" else u8_chunks
            assert sum(chunks) == B
            before = eng.launch_count
            call(B)
            got = eng.launch_count - before
            want = sum(device_launches(n) for n in chunks)
            assert got == want, f"{name} input, B={B}: {got} launches, chunks {chunks} make {want}"
    eng.close()


def test_sharded_driver_on_one_gpu_equals_single_engine():
    import bcad_b200
    cfg, p = _net()
    B = 37
    x = ocnn.synth_images(B, SHAPE, seed=9)
    imgs = _grey(B, 100, 90, seed=4)

    single = engine_from(cfg, p, precision="fp16", max_batch=128)
    sh = bcad_b200.ShardedEngine(spec_from_cfg(cfg), [0, 0], precision="fp16", max_batch=128)
    sh.set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
    ci = (np.arange(B) % 2).astype(np.int32)
    for got, want in ((sh.predict_explain_host(x, ci, "logit"), single.predict_explain_host(x, ci, "logit")),
                      (sh.gradcam_overlays_classes_host(imgs, (0, 1)), single.gradcam_overlays_classes_host(imgs, (0, 1)))):
        assert len(got) == len(want)
        for a, b in zip(got, want):
            assert np.array_equal(a, b)
    again = sh.gradcam_overlays_classes_host(imgs, (1, 0))
    assert all(np.shares_memory(a, b) for a, b in zip(again, got))       # the same shape reuses the driver's pinned arrays
    sh.close()
    single.close()

    single = engine_from(cfg, p, precision="fp32", max_batch=128, keep_all_activations=True)
    sh = bcad_b200.ShardedEngine(spec_from_cfg(cfg), [0, 0], precision="fp32", max_batch=128, keep_all_activations=True)
    sh.set_weights(p.conv_w, p.conv_b, p.dense_w, p.dense_b)
    got = sh.saliency_overlays_classes_host(imgs, (0, 1), want_saliency=True)
    want = single.saliency_overlays_classes_host(imgs, (0, 1), want_saliency=True)
    assert len(got) == len(want) and got[5] is not None
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    sh.close()
    single.close()
