"""GPU parity at the BENCHMARKED configurations (BASELINE.json configs[1] and configs[2]): the whole `MOT.step`
data flow with the real conv stacks -- YOLO pipeline at full cost, ReID crops from the frame, OSNet embeddings into
the association kernels, KLT on -- in lock step with the oracle tracker (bit-identical to the reference's
MultiTracker, tests/test_oracle_vs_reference.py).  The oracle is fed the same scripted detections and the embeddings
the GPU produced (tapped after OSNet), so every visible track id must agree frame by frame and boxes within +-1 px
(KLT tier T3, SURVEY.md 8c); the embeddings themselves are pinned to the fp32 oracle network in
tests/test_gpu_osnet_fused.py / test_gpu_nets.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(yolo, reid, n_obj, skip, n_frames, overlap=False, seed=3):
    from types import SimpleNamespace as NS
    from fastmot_b200 import MOT, DET_DTYPE, models
    from fastmot_b200.config import default_tracker_cfg
    from fastmot_b200.synth import SyntheticScene
    from oracle.run import default_tracker_cfg as oracle_cfg
    from oracle.tracker import OracleTracker
    scene = SyntheticScene(n_obj, seed=seed, label=0, dropout_frames=(), bounce_radius=16, overlap=overlap)
    tapped = {}

    def dets(t):
        tl, lb, cf, _ = scene.detections(t)
        d = np.zeros(len(tl), DET_DTYPE)
        d['tlbr'], d['label'], d['conf'] = tl, lb, cf
        return d.view(np.recarray)

    def tap(t, d, emb):
        tapped[t] = np.asarray(emb, np.float32).copy()

    mot = MOT(scene.size, detector_frame_skip=skip, class_ids=(0,),
              yolo_detector_cfg=NS(model=yolo, conf_thresh=0.25, nms_thresh=0.5, max_area=800000, min_aspect_ratio=1.2),
              feature_extractor_cfgs=(NS(model=reid, batch_size=16),), tracker_cfg=NS(**default_tracker_cfg()),
              detections_override=dets, embeddings_tap=tap)
    mot.reset(1 / 30.)
    metric = models.ReID.get_model(reid).METRIC
    ora = OracleTracker(scene.size, metric, **oracle_cfg())
    ora.reset(1 / 30.)
    exact = total = 0
    for t in range(n_frames):
        frame = scene.frame(t)
        mot.step(frame)
        tl, lb, cf, ids = scene.detections(t)
        if t == 0:
            ora.init(frame, tl, lb)
        else:
            ora.compute_flow(frame)
            ora.apply_kalman()
            if t % skip == 0:
                assert t in tapped, t
                emb = tapped[t]
                assert emb.shape == (len(tl), 512)
                np.testing.assert_allclose(np.linalg.norm(emb, axis=1), 1.0, atol=1e-3)
                ora.update(t, tl, lb, cf, emb)
        got = {trk.trk_id: trk.tlbr for trk in mot.visible_tracks()}
        want = dict(ora.visible())
        assert set(got) == set(want), (t, sorted(set(got) ^ set(want)))
        for k in got:
            d = float(np.abs(got[k] - np.asarray(want[k])).max())
            assert d <= 1.0, (t, k, got[k], want[k])
            exact += d == 0
            total += 1
    return exact / max(total, 1), len(got)


def test_config3_mot_step_200_tracks_real_osnet_embeddings_ids_match_oracle():
    frac, n = _run('YOLOv4CSP', 'OSNet10', 200, 5, 12)
    assert n == 200
    assert frac > 0.7, frac          # ratchet: exact-box fraction with the GPU LK (not bit-identical to OpenCV's)
    print(f"config 3: exact boxes {frac:.3f}")


def test_config2_detector_every_frame_tiny_x025():
    frac, n = _run('YOLOv4Tiny', 'OSNet025', 50, 1, 8, seed=5)
    assert n == 50
    assert frac > 0.7, frac


def test_bench_dump_outputs_repeatable_and_taken_after_the_last_timed_step(tmp_path):
    """`bench.py --dump-outputs`: the same arguments give the same arrays (float32 / float64, within the 64 MB
    budget); one more timed step moves the tracks."""
    import json
    import os
    import subprocess
    import sys
    from conftest import ROOT
    names = {"track_ids", "track_tlbr", "track_label", "track_mean", "track_cov", "track_feature"}

    def run(steps, tag):
        out = tmp_path / tag
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", str(steps),
                            "--warmup", "2", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == steps and line["repeats"]["windows"] == 1
        assert {p.stem for p in out.iterdir()} == names
        arrays = {n: np.load(out / f"{n}.npy") for n in names}
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        return arrays, line

    a, line = run(3, "a")
    n = len(a["track_ids"])
    assert n == line["config"]["visible_tracks_last_step"] > 0
    assert a["track_tlbr"].shape == (n, 4) and a["track_cov"].shape == (n, 8, 8)
    assert a["track_feature"].shape == (n, 512)
    b, _ = run(3, "b")
    for k in names:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    c, _ = run(4, "c")
    assert not np.array_equal(a["track_mean"], c["track_mean"])
