"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by running the UNMODIFIED reference
(imported from /root/reference through oracle/refshim.py) on the deterministic synthetic scene.
Run in the build container:  python -m oracle.make_goldens
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from fastmot_b200.synth import SyntheticScene  # noqa: E402
from oracle.refshim import load_reference  # noqa: E402
from oracle.ref_run import run_reference_tracker  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def sequence_golden(name, scene_kw, n_frames, frame_skip=5, metric='cosine'):
    """Per-frame visible ids/boxes + the KLT outputs (so Kalman/association can be replayed with KLT
    bypassed) + full per-track records at the last frame."""
    fm = load_reference()
    scene = SyntheticScene(**scene_kw)
    rec = {}

    assoc_calls = []
    orig_la = fm.tracker.linear_assignment

    def spy_la(cost, row_ids, col_ids):
        res = orig_la(cost, row_ids, col_ids)
        assoc_calls.append((np.array(cost, np.float64), list(map(int, row_ids)), list(map(int, col_ids)), res))
        return res

    fm.tracker.linear_assignment = spy_la

    def capture(t, trk, phase):
        if phase == 'flow':
            ids = np.array(list(trk.klt_bboxes.keys()), np.int64)
            rec[f'klt_ids_{t}'] = ids
            rec[f'klt_tlbr_{t}'] = np.array([trk.klt_bboxes[k] for k in ids], np.float64).reshape(-1, 4)
            rec[f'klt_ratio_{t}'] = np.array([trk.tracks[k].inlier_ratio for k in ids], np.float64)
            rec[f'H_{t}'] = np.zeros((0,)) if trk.homography is None else np.array(trk.homography, np.float64)
        elif phase == 'kalman':
            ids = np.array(list(trk.tracks.keys()), np.int64)
            rec[f'kal_ids_{t}'] = ids
            rec[f'kal_tlbr_{t}'] = np.array([trk.tracks[k].tlbr for k in ids], np.float64).reshape(-1, 4)
            rec[f'kal_mean_{t}'] = np.array([trk.tracks[k].state[0] for k in ids], np.float64).reshape(-1, 8)
        elif phase == 'update':
            ids = np.array(list(trk.tracks.keys()), np.int64)
            rec[f'upd_ids_{t}'] = ids
            rec[f'upd_age_{t}'] = np.array([trk.tracks[k].age for k in ids], np.int64)
            rec[f'upd_hits_{t}'] = np.array([trk.tracks[k].hits for k in ids], np.int64)
            rec[f'upd_hist_{t}'] = np.array(list(trk.hist_tracks.keys()), np.int64)

    try:
        out, trk = run_reference_tracker(scene, n_frames, frame_skip, metric, capture=capture)
    finally:
        fm.tracker.linear_assignment = orig_la
    for t, o in enumerate(out):
        rec[f'vis_ids_{t}'] = o['ids']
        rec[f'vis_tlbr_{t}'] = o['tlbr']
    ids = np.array(list(trk.tracks.keys()), np.int64)
    rec['final_ids'] = ids
    rec['final_mean'] = np.array([trk.tracks[k].state[0] for k in ids]).reshape(-1, 8)
    rec['final_cov'] = np.array([trk.tracks[k].state[1] for k in ids]).reshape(-1, 8, 8)
    rec['final_cnt'] = np.array([trk.tracks[k].avg_feat.count for k in ids], np.int64)
    rec['final_avg'] = np.array([trk.tracks[k].avg_feat() if trk.tracks[k].avg_feat.count else np.zeros(512)
                                 for k in ids], np.float32)
    rec['n_frames'] = np.int64(n_frames)
    rec['frame_skip'] = np.int64(frame_skip)
    rec['scene_kw'] = np.array(repr(scene_kw))
    rec['metric'] = np.array(metric)
    # keep a handful of (cost, assignment) pairs as LSA known-answer vectors
    keep = [c for c in assoc_calls if c[0].size > 0][:6]
    rec['n_lsa'] = np.int64(len(keep))
    for i, (cost, rid, cid, res) in enumerate(keep):
        rec[f'lsa_cost_{i}'] = cost
        rec[f'lsa_rid_{i}'] = np.array(rid, np.int64)
        rec[f'lsa_cid_{i}'] = np.array(cid, np.int64)
        rec[f'lsa_matches_{i}'] = np.array(res[0], np.int64).reshape(-1, 2)
        rec[f'lsa_urow_{i}'] = np.array(res[1], np.int64)
        rec[f'lsa_ucol_{i}'] = np.array(res[2], np.int64)
    np.savez_compressed(os.path.join(OUT, name), **rec)
    print(name, 'frames', n_frames, 'final tracks', len(ids), 'lsa', len(keep))


def primitive_golden():
    """Known-answer vectors for the association primitives straight from the reference functions."""
    fm = load_reference()
    rng = np.random.default_rng(7)
    rec = {}
    kf = fm.KalmanFilter()
    kf.reset_dt(1 / 30)
    MT = fm.kalman_filter.MeasType
    n = 64
    tl = rng.uniform(0, 1500, (n, 2))
    wh = rng.uniform(20, 200, (n, 2))
    tlbr = np.rint(np.concatenate([tl, tl + wh], 1))
    H = np.eye(3)
    H[:2, :2] += rng.normal(0, 0.01, (2, 2))
    H[:2, 2] = [1.3, -0.7]
    H[2, :2] = rng.normal(0, 1e-5, 2)
    z_flow = tlbr + rng.normal(0, 2, (n, 4))
    z_det = np.rint(tlbr + rng.normal(0, 3, (n, 4)))
    mult = rng.uniform(1, 3, n)
    m0, c0, m1, c1, m2, c2, md = [], [], [], [], [], [], []
    for i in range(n):
        m, c = kf.create(tlbr[i])
        m0.append(m); c0.append(c)
        m, c = kf.warp(m, c, H)
        m, c = kf.predict(m, c)
        m, c = kf.update(m, c, z_flow[i], MT.FLOW, mult[i])
        m1.append(m); c1.append(c)
        md.append(kf.motion_distance(m, c, z_det))
        m, c = kf.update(m, c, z_det[i], MT.DETECTOR)
        m2.append(m); c2.append(c)
    rec.update(kf_tlbr=tlbr, kf_H=H, kf_zflow=z_flow, kf_zdet=z_det, kf_mult=mult,
               kf_m0=np.array(m0), kf_c0=np.array(c0), kf_m1=np.array(m1), kf_c1=np.array(c1),
               kf_m2=np.array(m2), kf_c2=np.array(c2), kf_maha=np.array(md))
    # cdist / iou / occlusion
    XA = rng.normal(size=(64, 512))
    XA /= np.linalg.norm(XA, axis=1, keepdims=True)
    XA = XA.astype(np.float32)
    XB = (XA[rng.permutation(64)[:50]] + rng.normal(0, 0.02, (50, 512))).astype(np.float32)
    mask = rng.uniform(size=(64, 50)) < 0.1
    Met = fm.utils.distance.Metric
    rec['cd_XA'], rec['cd_XB'], rec['cd_mask'] = XA, XB, mask
    rec['cd_cos'] = fm.utils.distance.cdist(XA.astype(np.float64), XB, Met.COSINE, mask, 0.9)
    rec['cd_euc'] = fm.utils.distance.cdist(XA.astype(np.float64), XB, Met.EUCLIDEAN, mask, 0.9)
    b2 = np.rint(tlbr[:50] + rng.normal(0, 15, (50, 4)))
    rec['iou_a'], rec['iou_b'] = tlbr, b2
    rec['iou_dist'] = fm.utils.distance.iou_dist(tlbr, b2)
    allb = np.concatenate([tlbr, b2])
    rec["occ_thresh"] = np.float64(0.4567)  # not a ratio of small ints: the reference is @njit(fastmath) and its
    # result at inter/area == thresh exactly depends on LLVM reciprocal tricks (seen: 748/1496 >= 0.5 -> False)
    rec["occ_in"] = allb
    rec['occ_out'] = fm.utils.rect.find_occluded(allb, 0.4567)
    # assignment known answers (ties, gated, rectangular)
    k = 0
    for trial in range(24):
        nr, nc = rng.integers(1, 70, 2)
        mode = trial % 4
        if mode == 0:
            C = rng.uniform(0, 1, (nr, nc))
        elif mode == 1:
            C = rng.integers(0, 4, (nr, nc)).astype(float)
        elif mode == 2:
            C = np.where(rng.uniform(size=(nr, nc)) < 0.5, 1e5, rng.uniform(0, 1, (nr, nc)))
        else:
            C = np.where(rng.uniform(size=(nr, nc)) < 0.7, 1e5, np.round(rng.uniform(0, 1, (nr, nc)), 1))
        rid = [int(x) for x in rng.permutation(500)[:nr]]
        cid = [int(x) for x in rng.permutation(500)[:nc]]
        a = fm.utils.matching.linear_assignment(C, rid, cid)
        g = fm.utils.matching.greedy_match(C.copy(), rid, cid, 0.5)
        rec[f'la_cost_{k}'] = C
        rec[f'la_rid_{k}'] = np.array(rid, np.int64)
        rec[f'la_cid_{k}'] = np.array(cid, np.int64)
        rec[f'la_m_{k}'] = np.array(a[0], np.int64).reshape(-1, 2)
        rec[f'la_ur_{k}'] = np.array(a[1], np.int64)
        rec[f'la_uc_{k}'] = np.array(a[2], np.int64)
        rec[f'gr_m_{k}'] = np.array(g[0], np.int64).reshape(-1, 2)
        rec[f'gr_ur_{k}'] = np.array(g[1], np.int64)
        rec[f'gr_uc_{k}'] = np.array(g[2], np.int64)
        k += 1
    rec['n_la'] = np.int64(k)
    np.savez_compressed(os.path.join(OUT, 'assoc_primitives.npz'), **rec)
    print('assoc_primitives', k)


# scenes of tests/test_oracle_vs_reference.py (same order, same frame counts)
PARITY_SCENES = [
    (dict(n_objects=40, seed=9), 17),
    (dict(n_objects=30, seed=4, overlap=True), 12),
    (dict(n_objects=64, seed=1), 22),
    (dict(n_objects=50, seed=7, bounce_radius=8), 31),
    (dict(n_objects=30, seed=12, dropout_frames=(10,), dropout_every=1), 22),
    (dict(n_objects=30, seed=13, dropout_frames=(5, 10, 15), dropout_every=2), 22),
]

# det.txt of tests/test_public_detector.py
PUBLIC_DET_TXT = """1,-1,100.4,200.6,50.5,120.2,0.9,-1,-1,-1
1,-1,1800.0,900.0,200.0,300.0,0.4,-1,-1,-1
2,-1,10,20,30,40,1,-1,-1,-1
6,-1,640.5,360.5,11,21,1,-1,-1,-1
6,-1,0,0,1919,1079,1,-1,-1,-1
"""
PUBLIC_SIZES = ((1280, 720), (1920, 1080), (640, 360))


def parity_golden():
    """What the reference itself outputs for the oracle-parity tests: the full tracker (MultiTracker + Flow) on the
    PARITY_SCENES, DIoU-NMS on random boxes and the MOT Challenge public-detection reader."""
    import tempfile
    fm = load_reference()
    rec = {'n_scenes': np.int64(len(PARITY_SCENES))}
    for i, (scene_kw, n_frames) in enumerate(PARITY_SCENES):
        out, trk = run_reference_tracker(SyntheticScene(**scene_kw), n_frames)
        rec[f's{i}_scene_kw'] = np.array(repr(scene_kw))
        rec[f's{i}_n_frames'] = np.int64(n_frames)
        for t, o in enumerate(out):
            rec[f's{i}_ids_{t}'] = o['ids']
            rec[f's{i}_tlbr_{t}'] = o['tlbr']
        keys = np.array(list(trk.tracks.keys()), np.int64)
        rec[f's{i}_track_ids'] = keys
        rec[f's{i}_homography'] = np.array(trk.homography, np.float64)
        rec[f's{i}_mean'] = np.array([trk.tracks[k].state[0] for k in keys], np.float64).reshape(-1, 8)
    rng = np.random.default_rng(3)
    rec['n_nms'] = np.int64(6)
    for k in range(6):
        n = int(rng.integers(5, 150))
        tlwh = np.concatenate([rng.uniform(0, 300, (n, 2)), rng.uniform(10, 120, (n, 2))], 1).astype(np.float32)
        sc = rng.uniform(0.3, 1, n).astype(np.float32)
        rec[f'nms_tlwh_{k}'], rec[f'nms_score_{k}'] = tlwh, sc
        rec[f'nms_keep_{k}'] = np.array(fm.utils.rect.diou_nms(tlwh, sc, 0.5), np.int64)
    rec['pub_det_txt'] = np.array(PUBLIC_DET_TXT)
    with tempfile.TemporaryDirectory() as tmp:
        seq = os.path.join(tmp, 'MOT-TEST')
        os.makedirs(os.path.join(seq, 'det'))
        with open(os.path.join(seq, 'seqinfo.ini'), 'w') as f:
            f.write("[Sequence]\nname=MOT-TEST\nimWidth=1920\nimHeight=1080\n")
        with open(os.path.join(seq, 'det', 'det.txt'), 'w') as f:
            f.write(PUBLIC_DET_TXT)
        for j, size in enumerate(PUBLIC_SIZES):
            det = fm.detector.PublicDetector(size, (1,), 5, sequence_path=seq, conf_thresh=0.5, max_area=800000)
            for c in range(3):
                d = det.postprocess()
                rec[f'pub_tlbr_{j}_{c}'] = np.array(d.tlbr, np.float64).reshape(-1, 4)
                rec[f'pub_label_{j}_{c}'] = np.array(d.label, np.int64)
                rec[f'pub_conf_{j}_{c}'] = np.array(d.conf, np.float64)
    np.savez_compressed(os.path.join(OUT, 'reference_parity.npz'), **rec)
    print('reference_parity', len(PARITY_SCENES), 'scenes')


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ['prim', 'seq64', 'seq200', 'seqovl', 'parity']
    if 'parity' in which:
        parity_golden()
    if 'prim' in which:
        primitive_golden()
    if 'seq64' in which:
        sequence_golden('seq_T64.npz', dict(n_objects=64, seed=3), 22)
    if 'seq200' in which:
        sequence_golden('seq_T200.npz', dict(n_objects=200, seed=0), 32)
    if 'seqovl' in which:
        sequence_golden('seq_T70_overlap.npz', dict(n_objects=70, seed=5, overlap=True), 27)


def detect_golden():
    """_filter_dets (detector.py:322-365) known answers from the reference's own Numba function."""
    fm = load_reference()
    rng = np.random.default_rng(21)
    rec = {}
    cases = [(2500, False, (1920, 1920), (0., 420.)), (1200, True, (1920, 1080), (0., 0.)),
             (6000, False, (1920, 1920), (0., 420.))]
    for k, (K, two_cls, size, off) in enumerate(cases):
        det = np.zeros((K, 7), np.float32)
        det[:, :2] = rng.uniform(0, 0.9, (K, 2))
        det[:, 2:4] = rng.uniform(0.01, 0.15, (K, 2)) * [1, 2.2]
        det[:, 4] = rng.uniform(0, 1, K)
        det[:, 5] = rng.integers(0, 2, K) if two_cls else 0
        det[:, 6] = rng.uniform(0.2, 1, K)
        lm = np.array([True, True]) if two_cls else np.array([True])
        ref = fm.detector.YOLODetector._filter_dets(det.copy(), np.array(size), np.array(off), lm, 0.25, 0.5,
                                                    800000, 1.2)
        rec[f'det_{k}'] = det
        rec[f'size_{k}'] = np.array(size)
        rec[f'off_{k}'] = np.array(off)
        rec[f'lm_{k}'] = lm
        rec[f'tlbr_{k}'] = np.array([r[0] for r in ref]).reshape(-1, 4)
        rec[f'label_{k}'] = np.array([r[1] for r in ref], np.int64)
        rec[f'conf_{k}'] = np.array([r[2] for r in ref], np.float64)
        print('detect case', k, K, '->', len(ref))
    rec['n'] = np.int64(len(cases))
    np.savez_compressed(os.path.join(OUT, 'detect_filter.npz'), **rec)


if __name__ == '__main__' and 'detect' in (sys.argv[1:] or ['detect']):
    detect_golden()
