"""Pins the CPU oracle (oracle/openpose_oracle.py) against outputs of the REAL reference that
oracle/make_golden.py recorded in tests/golden/ (the reference ships no fixtures of its own)."""
import numpy as np
import pytest
import torch

from oracle import openpose_oracle as O
from oracle.make_golden import THREADS, smooth_noise_maps


@pytest.fixture(autouse=True, scope="module")
def recorded_thread_count():
    """oneDNN partitions the fp32 convolutions by the intra-op thread count, which reorders their sums and changes the
    last bits of the network outputs: the oracle computes with the count the fixtures were recorded with
    (make_golden.THREADS), whatever the host's core count."""
    n = torch.get_num_threads()
    torch.set_num_threads(THREADS)
    yield
    torch.set_num_threads(n)


def test_network_matches_reference_modules(golden):
    g = golden("net_default_init")
    x = torch.rand(*g["x_shape"].tolist(), generator=torch.Generator().manual_seed(int(g["x_seed"]))) - 0.5
    paf, heat = O.body_net(x, O.make_weights("body", int(g["seed"])))
    assert np.array_equal(paf.numpy(), g["body_paf"])
    assert np.array_equal(heat.numpy(), g["body_heat"])
    assert heat.min().item() >= 0.0          # stage-6 L2 ReLU quirk (src/model.py:30-33)
    hm = O.hand_net(x, O.make_weights("hand", int(g["seed"])))
    assert np.array_equal(hm.numpy(), g["hand_heat"])


def test_body_call_matches_reference(golden):
    g = golden("body_call_default_init")
    img = np.random.default_rng(int(g["img_seed"])).integers(0, 256, tuple(g["img_shape"]), dtype=np.uint8)
    sd = O.make_weights("body", int(g["weight_seed"]))
    for tag, scales in (("s1", (0.5,)), ("s2", (0.5, 1.0))):
        cand, sub = O.body_call(img, sd, scales, use_cv2=True)
        assert np.array_equal(cand, g["cand_" + tag])
        assert sub.shape == g["subset_" + tag].shape and np.array_equal(sub, g["subset_" + tag])


def test_hand_call_matches_reference(golden):
    g = golden("hand_call_kaiming")
    peaks = O.hand_call(g["crop"], O.make_weights("hand", int(g["weight_seed"]), "kaiming"))
    assert peaks.shape == (21, 3)
    assert (g["peaks"][:, 2] > 0).sum() >= 3          # the fixture is not degenerate
    assert np.array_equal(peaks, g["peaks"])


@pytest.mark.parametrize("tag,H,W,grid", [("p1", 240, 320, (1, 1)), ("p8", 360, 640, (4, 2)),
                                          ("p50", 720, 1280, (10, 5))])
def test_body_postproc_scenes(golden, tag, H, W, grid):
    g = golden("body_postproc")
    heat, paf, _ = O.synthetic_scene(H, W, grid, seed=0)
    cand, sub = O.body_postprocess(heat, paf, H)
    assert np.array_equal(cand, g["cand_" + tag])
    assert np.array_equal(sub, g["subset_" + tag])
    hands = np.array([[x, y, w, int(l)] for x, y, w, l in O.hand_detect(cand, sub, H, W)]).reshape(-1, 4)
    assert np.array_equal(hands, g["hands_" + tag])


def test_body_postproc_noise(golden):
    g = golden("body_postproc")
    heat = smooth_noise_maps(240, 320, 19, 4, 0.12, 11)
    paf = smooth_noise_maps(240, 320, 38, 6, 0.30, 12)
    cand, sub = O.body_postprocess(heat, paf, 240)
    assert len(cand) > 1000
    assert np.array_equal(cand, g["cand_noise"])
    assert np.array_equal(sub, g["subset_noise"])


def test_hand_postproc(golden):
    hm = smooth_noise_maps(184, 184, 22, 5, 0.03, 21)
    hm[:, :, 3] = -1.0
    peaks = O.hand_postprocess(hm)
    assert np.array_equal(peaks, golden("hand_postproc")["peaks"])
    assert np.array_equal(peaks[3], [0, 0, 0])


def test_thirdparty_restatements(golden):
    g = golden("thirdparty")
    rng = np.random.default_rng(int(g["seed"]))
    small = rng.integers(0, 256, (45, 70, 3), dtype=np.uint8)
    for i, f in enumerate((0.38333333333333336, 0.7666666666666667, 1.0222222222222221, 2.0444444444444443)):
        mine = O.resize_cubic_u8(small, f)
        assert np.array_equal(mine, g["u8_%d" % i]), "open-source cv2 path must be bit-exact"
        ipp = g["u8ipp_%d" % i].astype(int)
        assert np.abs(mine.astype(int) - ipp).max() <= 1, "IPP path differs by at most 1 LSB"
    fm = rng.standard_normal((6, 9, 5)).astype(np.float32)
    up = O.resize_cubic_f32(fm, f=8)
    assert np.abs(up - g["f32_up"]).max() < 2e-6
    full = O.resize_cubic_f32(up[:45, :70], dsize=(161, 97))
    assert np.abs(full - g["f32_full"]).max() < 4e-6
    # composite 1-D operators reproduce the two-pass result
    My = O.composite_upsample_matrix(6, 45, 97)
    Mx = O.composite_upsample_matrix(9, 70, 161)
    comp = np.einsum("yh,hwc,xw->yxc", My, fm.astype(np.float64), Mx)
    assert np.abs(comp - g["f32_full"]).max() < 1e-5
    gm = rng.random((40, 33)).astype(np.float32).astype(np.float64)
    assert np.array_equal(O.gaussian_sigma3(gm), g["gauss"]), "gaussian must be bit-exact with scipy"


# ---- batched estimators (srcmx/Batch_model.py, SURVEY.md 8f row N2) ------------------------------------------------
def _flat(c):
    return np.asarray(c, dtype=np.float64).reshape(-1, 4)


def test_batch_body_call_matches_reference(golden):
    from oracle.make_golden import batch_frames
    g = golden("batch_model")
    out = O.batch_body_call(batch_frames(2, 120, 160, 31), O.make_weights("body", 0))
    for f, (cand, sub) in enumerate(out):
        assert len(g["body_cand_%d" % f]) > 10
        assert np.array_equal(_flat(cand), _flat(g["body_cand_%d" % f]))
        assert np.array_equal(sub, g["body_subset_%d" % f])


def test_batch_hand_call_matches_reference(golden):
    from oracle.make_golden import batch_frames
    g = golden("batch_model")
    peaks = O.batch_hand_call(batch_frames(2, 96, 96, 32), O.make_weights("hand", 5, "kaiming"))
    assert (g["hand_peaks"][:, :, 2] > 0).sum() >= 6
    assert np.array_equal(peaks, g["hand_peaks"])


@pytest.mark.parametrize("tag,H,W,grid", [("p1", 240, 320, (1, 1)), ("p8", 360, 640, (4, 2)),
                                          ("p50", 720, 1280, (10, 5))])
def test_batch_body_postproc_scenes(golden, tag, H, W, grid):
    """Peaks found and scored on the 5x5-blurred map + FindBody_frame, vs the reference's own code on the same maps."""
    g = golden("batch_model")
    heat, paf, _ = O.synthetic_scene(H, W, grid, seed=0)
    cand, sub = O.batch_body_postprocess(O.blur5_fixed_order(heat), paf.astype(np.float32))
    assert len(sub) >= grid[0] * grid[1]
    assert np.array_equal(_flat(cand), _flat(g["post_cand_" + tag]))
    assert np.array_equal(sub, g["post_subset_" + tag])


def test_batch_hand_postproc(golden):
    hm = O.blur5_fixed_order(smooth_noise_maps(184, 184, 22, 5, 0.03, 21))
    hm[:, :, 3] = -1.0
    peaks = O.batch_hand_postprocess(hm)
    assert np.array_equal(peaks, golden("batch_model")["post_hand_peaks"][0])
    assert np.array_equal(peaks[3], [0, 0, 0]) and (peaks[:, 2] > 0).sum() >= 10
