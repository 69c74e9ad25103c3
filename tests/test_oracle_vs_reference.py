"""CPU: the oracle restatements against what the UNMODIFIED reference outputs on the same inputs, stored in
tests/golden/reference_parity.npz (written from the reference by `python -m oracle.make_goldens parity`)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN


@pytest.fixture(scope="module")
def parity():
    return np.load(os.path.join(GOLDEN, "reference_parity.npz"))


def _scene_index(g, scene_kw, n_frames):
    for i in range(int(g['n_scenes'])):
        if str(g[f's{i}_scene_kw']) == repr(scene_kw) and int(g[f's{i}_n_frames']) == n_frames:
            return i
    raise KeyError(f"no reference golden for {scene_kw!r}, {n_frames} frames")


@pytest.mark.parametrize("scene_kw,n_frames", [
    (dict(n_objects=40, seed=9), 17),
    (dict(n_objects=30, seed=4, overlap=True), 12),
    (dict(n_objects=64, seed=1), 22),                     # config-1 size; scripted drop-outs on frames 10 / 15 -> aging,
                                                          # IoU stage and re-identification from the history
    (dict(n_objects=50, seed=7, bounce_radius=8), 31),    # direction reversals (benchmark scene motion model)
    (dict(n_objects=30, seed=12, dropout_frames=(10,), dropout_every=1), 22),       # a detector frame with NO detections
    (dict(n_objects=30, seed=13, dropout_frames=(5, 10, 15), dropout_every=2), 22),  # half the objects never confirm
])
def test_oracle_tracker_full_pipeline_identical(parity, scene_kw, n_frames):
    """OracleTracker + OracleFlow (cv2) vs reference MultiTracker + Flow: identical ids and boxes per frame."""
    from fastmot_b200.synth import SyntheticScene
    from oracle.run import run_oracle_tracker
    i = _scene_index(parity, scene_kw, n_frames)
    got, otrk = run_oracle_tracker(SyntheticScene(**scene_kw), n_frames)
    for t in range(n_frames):
        assert np.array_equal(parity[f's{i}_ids_{t}'], got[t]['ids']), t
        assert np.array_equal(parity[f's{i}_tlbr_{t}'], got[t]['tlbr']), t
    ref_ids = parity[f's{i}_track_ids']
    assert ref_ids.tolist() == list(otrk.tracks.keys())
    np.testing.assert_allclose(parity[f's{i}_homography'], otrk.homography, atol=1e-12)
    for k, mean in zip(ref_ids.tolist(), parity[f's{i}_mean']):
        np.testing.assert_allclose(mean, otrk.tracks[k].mean, atol=1e-6)


def test_detect_oracle_against_reference_functions(parity):
    from oracle import detect
    assert int(parity['n_nms']) == 6
    for trial in range(6):
        tlwh, sc = parity[f'nms_tlwh_{trial}'], parity[f'nms_score_{trial}']
        assert np.array_equal(parity[f'nms_keep_{trial}'], detect.diou_nms(tlwh, sc, 0.5))
