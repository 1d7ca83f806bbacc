"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the REAL reference
(/root/reference, imported through oracle/reference_loader.py) in the build container.

    python oracle/make_golden.py            # rewrites every fixture

The fixtures hold only small OUTPUT arrays (and, where inputs cannot be regenerated from a seed, small
inputs).  Inputs are regenerated at test time from the recorded seeds with numpy / torch CPU generators,
which are deterministic for the pinned numpy 2.3 / torch 2.11 of this image.  Versions used to generate
are stored in each file under `versions`.
"""
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import reference_loader as RL          # noqa: E402
from oracle import openpose_oracle as O            # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
# torch intra-op threads the fixtures are recorded with.  oneDNN partitions the fp32 convolutions by this count, so
# it fixes the order of their sums and with it the last bits of the stored network outputs; the stored files were
# made on an 8-core host at torch's default count, and 8 reproduces them on hosts with other core counts.
THREADS = 8


def versions():
    import cv2
    import scipy
    import torch
    return np.array(["numpy=%s" % np.__version__, "torch=%s" % torch.__version__, "cv2=%s" % cv2.__version__,
                     "scipy=%s" % scipy.__version__])


def smooth_noise_maps(h, w, c, sigma, std, seed):
    """Deterministic smooth random maps (fp32-representable float64)."""
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    m = np.stack([gaussian_filter(rng.standard_normal((h, w)), sigma) for _ in range(c)], -1)
    return (m / m.std() * std).astype(np.float32).astype(np.float64)


def batch_frames(n, h, w, seed):
    """Deterministic structured float frames in [0,1], NCHW float32 (what transforms.ToTensor yields)."""
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    x = np.stack([gaussian_filter(rng.random((3, h, w)), (0, 3, 3)) for _ in range(n)])
    x = (x - x.min()) / (x.max() - x.min())
    return x.astype(np.float32)


def main():
    import cv2
    import torch
    from scipy.ndimage import gaussian_filter
    torch.set_num_threads(THREADS)
    os.makedirs(OUT, exist_ok=True)
    ns = RL.load()
    tmp = tempfile.mkdtemp()
    v = versions()

    # ---- 1. networks: reference nn.Modules on tiny inputs ---------------------------------------
    torch.manual_seed(0)
    body = ns.model.bodypose_model().eval()
    torch.manual_seed(0)
    hand = ns.model.handpose_model().eval()
    g = torch.Generator().manual_seed(1)
    x = torch.rand(1, 3, 48, 64, generator=g) - 0.5
    with torch.no_grad():
        paf, heat = body(x)
        hm = hand(x)
    np.savez_compressed(os.path.join(OUT, "net_default_init.npz"), versions=v, seed=0, x_seed=1,
                        x_shape=np.array(x.shape), body_paf=paf.numpy(), body_heat=heat.numpy(),
                        hand_heat=hm.numpy())

    # ---- 2. Body.__call__ end to end, default init, tiny frame, 1 and 2 scales ------------------
    sd = RL.save_checkpoint(body, os.path.join(tmp, "body.pth"))
    B = ns.Body(os.path.join(tmp, "body.pth"))
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (120, 160, 3), dtype=np.uint8)
    out = {}
    for tag, scales in (("s1", [0.5]), ("s2", [0.5, 1.0])):
        B.scale_search = scales
        cand, sub = B(img.copy())
        out["cand_" + tag], out["subset_" + tag] = cand, sub
    np.savez_compressed(os.path.join(OUT, "body_call_default_init.npz"), versions=v, weight_seed=0, img_seed=0,
                        img_shape=np.array(img.shape), **out)

    # ---- 3. Hand.__call__ end to end (Kaiming weights so that peaks exist) ----------------------
    sdh = O.make_weights("hand", seed=5, init="kaiming")
    torch.save(sdh, os.path.join(tmp, "hand.pth"))
    Hd = ns.Hand(os.path.join(tmp, "hand.pth"))
    crop = np.random.default_rng(2).integers(0, 256, (40, 40, 3), dtype=np.uint8)
    crop = cv2.GaussianBlur(crop, (0, 0), 3)
    peaks = Hd(crop.copy())
    np.savez_compressed(os.path.join(OUT, "hand_call_kaiming.npz"), versions=v, weight_seed=5, img_seed=2,
                        crop=crop, peaks=peaks)

    # ---- 4. body post-processing on injected maps: synthetic scenes + smooth noise --------------
    pp = RL.body_postproc()
    out = {}
    for tag, (H, W, grid) in {"p1": (240, 320, (1, 1)), "p8": (360, 640, (4, 2)), "p50": (720, 1280, (10, 5))}.items():
        heatm, pafm, _ = O.synthetic_scene(H, W, grid, seed=0)
        cand, sub = pp(heatm.copy(), pafm.copy(), np.zeros((H, W, 3), np.uint8))
        out["cand_" + tag], out["subset_" + tag] = cand, sub
        out["hands_" + tag] = np.array([[x, y, w, int(l)] for x, y, w, l in
                                        ns.util.handDetect(cand, sub, np.zeros((H, W, 3), np.uint8))]).reshape(-1, 4)
    heatm = smooth_noise_maps(240, 320, 19, 4, 0.12, 11)
    pafm = smooth_noise_maps(240, 320, 38, 6, 0.30, 12)
    cand, sub = pp(heatm.copy(), pafm.copy(), np.zeros((240, 320, 3), np.uint8))
    out["cand_noise"], out["subset_noise"] = cand, sub
    np.savez_compressed(os.path.join(OUT, "body_postproc.npz"), versions=v, **out)

    # ---- 5. hand post-processing on injected maps ---------------------------------------------
    hp = RL.hand_postproc()
    hmaps = smooth_noise_maps(184, 184, 22, 5, 0.03, 21)
    hmaps[:, :, 3] = -1.0
    np.savez_compressed(os.path.join(OUT, "hand_postproc.npz"), versions=v, peaks=hp(hmaps.copy()))

    # ---- 6. third-party numerics: cv2 (IPP off = open-source path) and scipy -------------------
    rng = np.random.default_rng(7)
    small = rng.integers(0, 256, (45, 70, 3), dtype=np.uint8)
    cv2.setUseOptimized(False)
    u8 = {("u8_%d" % i): cv2.resize(small, (0, 0), fx=f, fy=f, interpolation=cv2.INTER_CUBIC)
          for i, f in enumerate((0.38333333333333336, 0.7666666666666667, 1.0222222222222221, 2.0444444444444443))}
    cv2.setUseOptimized(True)
    u8_ipp = {("u8ipp_%d" % i): cv2.resize(small, (0, 0), fx=f, fy=f, interpolation=cv2.INTER_CUBIC)
              for i, f in enumerate((0.38333333333333336, 0.7666666666666667, 1.0222222222222221, 2.0444444444444443))}
    fm = rng.standard_normal((6, 9, 5)).astype(np.float32)
    up = cv2.resize(fm, (0, 0), fx=8, fy=8, interpolation=cv2.INTER_CUBIC)
    full = cv2.resize(up[:45, :70], (161, 97), interpolation=cv2.INTER_CUBIC)
    gm = rng.random((40, 33)).astype(np.float32).astype(np.float64)
    np.savez_compressed(os.path.join(OUT, "thirdparty.npz"), versions=v, seed=7, f32_up=up, f32_full=full,
                        gauss=gaussian_filter(gm, sigma=3), **u8, **u8_ipp)
    # ---- 7. batched estimators (srcmx/Batch_model.py): end to end + their post-processing on injected maps ----
    RLb = RL.load_batch()
    out = {}
    torch.save(sd, os.path.join(tmp, "body.pth"))
    bb = RLb.Batch_body(os.path.join(tmp, "body.pth"))
    frames = batch_frames(2, 120, 160, 31)
    for f, (cand, sub) in enumerate(bb(torch.from_numpy(frames))):
        out["body_cand_%d" % f], out["body_subset_%d" % f] = np.asarray(cand, dtype=np.float64), sub
    bh = RLb.Batch_hand(os.path.join(tmp, "hand.pth"))
    out["hand_peaks"] = bh(torch.from_numpy(batch_frames(2, 96, 96, 32)))
    bpp, hpp = RL.batch_body_postproc(), RL.batch_hand_postproc()
    for tag, (H, W, grid) in {"p1": (240, 320, (1, 1)), "p8": (360, 640, (4, 2)), "p50": (720, 1280, (10, 5))}.items():
        heatm, pafm, _ = O.synthetic_scene(H, W, grid, seed=0)
        blurred = O.blur5_fixed_order(heatm)
        (cand, sub), = bpp(bb, torch.from_numpy(blurred.transpose(2, 0, 1)[None].copy()),
                           pafm.astype(np.float32).transpose(2, 0, 1)[None].copy())
        out["post_cand_" + tag], out["post_subset_" + tag] = np.asarray(cand, dtype=np.float64), sub
    hm = O.blur5_fixed_order(smooth_noise_maps(184, 184, 22, 5, 0.03, 21))
    hm[:, :, 3] = -1.0
    out["post_hand_peaks"] = hpp(bh, hm[None].copy())
    np.savez_compressed(os.path.join(OUT, "batch_model.npz"), versions=v, **out)

    print("wrote", sorted(os.listdir(OUT)))
    for f in sorted(os.listdir(OUT)):
        print("  %-32s %8d bytes" % (f, os.path.getsize(os.path.join(OUT, f))))


if __name__ == "__main__":
    main()
