"""Live check of the oracle against the reference itself -- only where /root/reference exists (the build
container).  Skipped on the GPU box."""
import numpy as np
import pytest
import torch

from oracle import openpose_oracle as O
from oracle import reference_loader as RL

pytestmark = pytest.mark.skipif(not RL.available(), reason="needs a checkout of the original project (set OPENPOSE_REFERENCE_ROOT)")


def test_weights_follow_reference_rng_stream():
    ns = RL.load()
    for kind, ctor in (("body", ns.model.bodypose_model), ("hand", ns.model.handpose_model)):
        torch.manual_seed(4)
        ref = {k.split(".", 1)[1]: v for k, v in ctor().state_dict().items()}
        mine = O.make_weights(kind, 4)
        assert sorted(ref) == sorted(mine)
        assert all(torch.equal(ref[k], mine[k]) for k in ref)


def test_body_call_live(tmp_path):
    ns = RL.load()
    sd = O.make_weights("body", 1)
    torch.save(sd, tmp_path / "b.pth")
    B = ns.Body(str(tmp_path / "b.pth"))
    B.scale_search = [0.5, 1.5]
    img = np.random.default_rng(5).integers(0, 256, (96, 128, 3), dtype=np.uint8)
    cand_ref, sub_ref = B(img.copy())
    cand, sub = O.body_call(img, sd, (0.5, 1.5))
    assert np.array_equal(cand, cand_ref) and np.array_equal(sub, sub_ref)


def test_postproc_live():
    pp = RL.body_postproc()
    heat, paf, _ = O.synthetic_scene(300, 400, (3, 1), seed=3)
    cand_ref, sub_ref = pp(heat.copy(), paf.copy(), np.zeros((300, 400, 3), np.uint8))
    cand, sub = O.body_postprocess(heat, paf, 300)
    assert len(sub_ref) >= 3
    assert np.array_equal(cand, cand_ref) and np.array_equal(sub, sub_ref)


def test_batch_estimators_live(tmp_path):
    """srcmx/Batch_model.py Batch_body / Batch_hand (row N2) run from the reference checkout vs the restatement."""
    from oracle.make_golden import batch_frames
    b = RL.load_batch()
    sd = O.make_weights("body", 3)
    torch.save(sd, tmp_path / "b.pth")
    frames = batch_frames(2, 96, 136, 8)
    ref = b.Batch_body(str(tmp_path / "b.pth"))(torch.from_numpy(frames))
    for (rc, rs), (mc, ms) in zip(ref, O.batch_body_call(frames, sd)):
        assert np.array_equal(np.asarray(rc, dtype=np.float64).reshape(-1, 4), mc.reshape(-1, 4)) and np.array_equal(rs, ms)
    sdh = O.make_weights("hand", 3, "kaiming")
    torch.save(sdh, tmp_path / "h.pth")
    crops = batch_frames(2, 64, 64, 9)
    ref = b.Batch_hand(str(tmp_path / "h.pth"))(torch.from_numpy(crops))
    assert np.array_equal(ref, O.batch_hand_call(crops, sdh))
    # the reference's own post-processing on injected maps
    heat, paf, _ = O.synthetic_scene(300, 400, (3, 1), seed=3)
    blurred = O.blur5_fixed_order(heat)
    est = b.Batch_body(str(tmp_path / "b.pth"))
    (rc, rs), = RL.batch_body_postproc()(est, torch.from_numpy(blurred.transpose(2, 0, 1)[None].copy()),
                                         paf.astype(np.float32).transpose(2, 0, 1)[None].copy())
    mc, ms = O.batch_body_postprocess(blurred, paf.astype(np.float32))
    assert len(rs) == 3 and np.array_equal(np.asarray(rc, dtype=np.float64), mc) and np.array_equal(rs, ms)
