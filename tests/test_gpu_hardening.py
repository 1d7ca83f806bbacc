"""Parity hardening (round-2 review): tests that separate "kernel wrong" from "bf16 inherent", that are not vacuous on
flat default-init maps, and that exercise the true drop-in path (checkpoint FILE -> Body / Hand, `src.*` shim)."""
import os
import sys

import numpy as np
import pytest

from oracle import openpose_oracle as O

pytestmark = pytest.mark.gpu


def _match_rate(cand_a, cand_b):
    """Fraction of the key points in `cand_b` that have a key point of `cand_a` within 1 px (Chebyshev)."""
    a, b = np.asarray(cand_a).reshape(-1, 4), np.asarray(cand_b).reshape(-1, 4)
    if len(b) == 0:
        return 1.0
    if len(a) == 0:
        return 0.0
    d = np.abs(b[:, None, :2] - a[None, :, :2]).max(-1)
    return float((d.min(1) <= 1.0).mean())


def _kaiming_scene():
    import cv2
    sd = O.make_weights("body", 2, "kaiming")
    img = cv2.GaussianBlur(np.random.default_rng(21).integers(0, 256, (240, 320, 3), dtype=np.uint8), (0, 0), 3)
    return sd, img, (0.5, 1.0)


def test_body_keypoints_vs_bf16_emulating_oracle():
    """north_star (3), split by cause.  The device computes in bf16 with fp32 accumulation; `O.body_call(bf16=True)` is
    the CPU restatement with the SAME roundings (weights and every stored activation to bf16, fp32 accumulation) but
    another summation ORDER.  Two bf16 implementations are not bit-reproducible against each other: a different
    fp32 summation order moves a sum across a bf16 rounding boundary here and there (4e-3 relative each), and ~50
    layers with ReLU amplify that like any other perturbation (measured: maps 1e-2 apart, half the bf16-vs-fp32
    distance).  So the check is relative: the device must be CLOSER to the bf16 emulation than the emulation is to
    fp32, for the maps and for the key points -- a kernel defect would add to the device's distance and not to the
    emulation's.  (Per-layer exactness is established separately: tests/test_gpu_net_layers.py compares every launch of
    the networks' execution plans, problem by problem, with an fp64 convolution of the device's own bf16 inputs.)"""
    from pytorch_openpose_b200 import Body
    sd, img, scales = _kaiming_scene()
    body = Body(sd, scale_search=list(scales))
    cand, subset = body(img)
    heat, paf = body.last_maps(img.shape)
    c16, s16, h16, p16 = O.body_call(img, sd, scales, use_cv2=False, bf16=True, return_maps=True)
    c32, s32, h32, p32 = O.body_call(img, sd, scales, use_cv2=True, return_maps=True)
    dev_vs_emul = min(_match_rate(cand, c16), _match_rate(c16, cand))
    emul_vs_fp32 = min(_match_rate(c16, c32), _match_rate(c32, c16))
    dev_vs_fp32 = min(_match_rate(cand, c32), _match_rate(c32, cand))
    rel = lambda a, b: float(np.abs(a - b).max() / np.abs(b).max())
    print("key points within 1 px: device vs bf16-emulating CPU %.1f %% | bf16-emulating CPU vs fp32 CPU %.1f %% | "
          "device vs fp32 CPU %.1f %%   (%d / %d / %d key points)" % (100 * dev_vs_emul, 100 * emul_vs_fp32,
                                                                     100 * dev_vs_fp32, len(cand), len(c16), len(c32)))
    print("maps, max|d|/max|ref|: device vs emulation heat %.2e paf %.2e | emulation vs fp32 heat %.2e paf %.2e" %
          (rel(heat, h16), rel(paf, p16), rel(h16, h32), rel(p16, p32)))
    assert rel(heat, h16) <= 0.75 * rel(h16, h32) and rel(paf, p16) <= 0.75 * rel(p16, p32)
    assert rel(heat, h16) <= 2e-2 and rel(paf, p16) <= 2e-2
    assert dev_vs_emul >= 0.9 and dev_vs_emul >= emul_vs_fp32
    assert dev_vs_fp32 >= emul_vs_fp32 - 0.03          # the device is as good a bf16 implementation as the emulation


def test_default_init_maps_structure_not_only_level():
    """With PyTorch's default init the maps are a constant (the last bias) plus ~1e-4 of spatial structure, so
    max|d|/max|ref| <= 1e-2 alone mostly checks the bias.  Here the per-channel mean is removed first: the spatial
    structure of the device maps must correlate with the fp32 CPU maps', and the device must be as close to the
    bf16-emulating restatement as that restatement's own distance to fp32."""
    from pytorch_openpose_b200 import Body
    sd = O.make_weights("body", 0)
    img = np.random.default_rng(0).integers(0, 256, (480, 640, 3), dtype=np.uint8)
    body = Body(sd)
    body(img)
    heat, paf = body.last_maps(img.shape)
    _, _, h32, p32 = O.body_call(img, sd, (0.5,), use_cv2=True, return_maps=True)
    _, _, h16, p16 = O.body_call(img, sd, (0.5,), use_cv2=False, bf16=True, return_maps=True)

    def structure(a, ref):
        """per channel with structure: (correlation of the mean-removed maps, rms of the mean-removed error / std)"""
        out = []
        for c in range(ref.shape[2]):
            r = ref[..., c] - ref[..., c].mean()
            if r.std() < 1e-6:
                continue
            d = a[..., c] - a[..., c].mean()
            out.append((float(np.corrcoef(d.ravel(), r.ravel())[0, 1]), float(np.sqrt(((d - r) ** 2).mean()) / r.std())))
        return np.array(out)

    for name, dev, emul, ref in (("heat", heat, h16, h32), ("paf", paf, p16, p32)):
        s_dev, s_emul, s_de = structure(dev, ref), structure(emul, ref), structure(dev, emul)
        print("%s structure (corr min / median, rms err / std median): device vs fp32 %.3f / %.3f, %.3f | emulation vs "
              "fp32 %.3f / %.3f, %.3f | device vs emulation %.3f / %.3f, %.3f" %
              (name, s_dev[:, 0].min(), np.median(s_dev[:, 0]), np.median(s_dev[:, 1]), s_emul[:, 0].min(),
               np.median(s_emul[:, 0]), np.median(s_emul[:, 1]), s_de[:, 0].min(), np.median(s_de[:, 0]),
               np.median(s_de[:, 1])))
        assert len(s_dev) >= 10
        assert np.median(s_dev[:, 0]) >= 0.95 and s_dev[:, 0].min() >= 0.8          # the structure is there ...
        assert np.median(s_dev[:, 1]) <= 0.4                                          # ... to a fraction of its own size
        assert np.median(s_de[:, 1]) <= np.median(s_emul[:, 1]) + 0.05               # and bf16 explains the rest


def test_body_and_hand_from_checkpoint_files(tmp_path):
    """The reference's constructor takes a PATH (src/body.py:16-22, src/hand.py:17-23): torch.load + util.transfer."""
    import torch
    from pytorch_openpose_b200 import Body, Hand
    sd_b, sd_h = O.make_weights("body", 0), O.make_weights("hand", 0)
    pb, ph = str(tmp_path / "body_pose_model.pth"), str(tmp_path / "hand_pose_model.pth")
    torch.save(sd_b, pb)
    torch.save(sd_h, ph)
    img = np.random.default_rng(5).integers(0, 256, (120, 160, 3), dtype=np.uint8)
    c1, s1 = Body(pb)(img)
    c2, s2 = Body(sd_b)(img)
    assert np.array_equal(c1, c2) and np.array_equal(s1, s2) and len(c1) > 0
    crop = img[:64, :64]
    assert np.array_equal(Hand(ph)(crop), Hand(sd_h)(crop))
    with pytest.raises(FileNotFoundError):
        Body(str(tmp_path / "missing.pth"))
    broken = dict(sd_b)
    del broken["conv4_2.weight"]
    torch.save(broken, pb)
    with pytest.raises(KeyError):
        Body(pb)


def test_install_as_src_runs_the_reference_callers_imports(tmp_path):
    """`from src.body import Body; from src.hand import Hand; from src import util, model` -- the import lines of
    srcmx/MotionEstimation.py:12-19 -- resolve to this package, and the module-level singletons built from checkpoint
    paths run the per-frame caller's sequence: body -> util.handDetect -> crops -> hand."""
    import torch
    import pytorch_openpose_b200
    saved = {k: sys.modules.get(k) for k in ("src", "src.body", "src.hand", "src.util", "src.model")}
    try:
        pytorch_openpose_b200.install_as_src()
        from src.body import Body
        from src.hand import Hand
        from src import util, model          # noqa: F401
        pb, ph = str(tmp_path / "b.pth"), str(tmp_path / "h.pth")
        torch.save(O.make_weights("body", 0), pb)
        torch.save(O.make_weights("hand", 5, "kaiming"), ph)
        body_estimation, hand_estimation = Body(pb), Hand(ph)                    # MotionEstimation.py:18-19
        oriImg = np.random.default_rng(3).integers(0, 256, (240, 320, 3), dtype=np.uint8)
        candidate, subset = body_estimation(oriImg)
        assert candidate.dtype == np.float64 and subset.shape[1:] == (20,)
        # one synthetic person so that handDetect yields boxes (random weights find none)
        candidate = np.array([[100., 60., 1., 0.], [80., 90., 1., 1.], [70., 140., 1., 2.], [120., 90., 1., 3.],
                              [130., 140., 1., 4.], [135., 185., 1., 5.], [72., 190., 1., 6.]])
        person = -np.ones(20)
        person[[2, 3, 4, 5, 6, 7]] = [1, 2, 6, 3, 4, 5]
        hands = util.handDetect(candidate, person[None], oriImg)
        assert len(hands) == 2
        for x, y, w, is_left in hands:
            peaks = hand_estimation(oriImg[y:y + w, x:x + w, :])
            assert peaks.shape == (21, 3) and peaks.dtype == np.float64
            peaks[:, 0] = np.where(peaks[:, 0] == 0, peaks[:, 0], peaks[:, 0] + x)     # caller mutates in place (:187-188)
        assert hasattr(model, "bodypose_model") and hasattr(model, "handpose_model")
        assert callable(util.padRightDownCorner) and callable(util.transfer) and callable(util.npmax)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_multiscale_average_in_float32_is_a_tolerance_level_deviation():
    """The reference adds float32(heatmap / n) of every scale into a float64 map (src/body.py:67-68) after two cv2
    resizes per scale; the device applies one composite operator per axis and accumulates the scales in float32.  The
    maps differ at the 1e-6 level, so discrete results can only differ where two smoothed values tie to ~1e-7.  Here the
    oracle post-processes maps built the reference's way (cv2 two-pass resize, float64 accumulation) from the DEVICE's own
    per-scale net outputs: key points must agree (positions identical, scores to 1e-5)."""
    from pytorch_openpose_b200 import Body
    from tests import gpu_util as G
    sd, img, _ = _kaiming_scene()
    scales = (0.5, 1.0, 1.5, 2.0)
    body = Body(sd, scale_search=list(scales))
    cand, subset = body(img)
    heat_dev, paf_dev = body.last_maps(img.shape)
    H, W = img.shape[:2]
    plan = O.scale_plan(H, W, scales)
    heats, pafs = [], []
    for p, s in zip(plan, scales):
        pre, _ = G.preprocess(img, s)
        paf, heat = G.net_forward(body.net.session(), pre[None])
        heats.append(np.ascontiguousarray(heat[0].transpose(2, 0, 1)))
        pafs.append(np.ascontiguousarray(paf[0].transpose(2, 0, 1)))
    heat_ref = O.upsample_avg(heats, plan, H, W, use_cv2=True)
    paf_ref = O.upsample_avg(pafs, plan, H, W, use_cv2=True)
    print("composite float32 maps vs cv2 two-pass float64 maps: heat %.2e paf %.2e (max abs)" %
          (np.abs(heat_dev - heat_ref).max(), np.abs(paf_dev - paf_ref).max()))
    assert np.abs(heat_dev - heat_ref).max() <= 1e-5 and np.abs(paf_dev - paf_ref).max() <= 1e-5
    rc, rs = O.body_postprocess(heat_ref, paf_ref, H)
    rc = rc.reshape(-1, 4)
    cand = cand.reshape(-1, 4)
    dev = {(x, y): s for x, y, s, _ in cand}
    hit = [(x, y) in dev for x, y, _, _ in rc]
    frac = float(np.mean(hit)) if len(rc) else 1.0
    print("key points: device %d, reference-style maps %d, identical positions: %.1f %%" % (len(cand), len(rc), 100 * frac))
    assert len(rc) > 100 and abs(len(rc) - len(cand)) <= max(2, len(rc) // 50)
    assert frac >= 0.98                                  # a differing peak needs two smoothed values within ~1e-7
    for (x, y, s, _), h in zip(rc, hit):
        if h:
            assert abs(dev[(x, y)] - s) <= 1e-5


def test_fuzz_random_sizes_and_scales():
    """tests/tools/fuzz_body.py (random frame sizes 12..520, scale lists, single frames and batches, structured and flat
    weights): discrete results equal the oracle's post-processing of the device maps in every case."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "tools", "fuzz_body.py"), "10", "5"], cwd=root,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "10 cases, 0 mismatches" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_graft_entry_smoke():
    """The driver's smoke check (one small Body and Hand call against the oracle) stays green with the rest."""
    import __graft_entry__ as entry
    entry.smoke()
