"""SURVEY.md §8(f) row 2: MOT Challenge public-detection reader and result writer (host-side formats either side of
the hot path).  The reader is checked against hand-computed rows and against the rows the reference's own
`PublicDetector` returned for the same det.txt (tests/golden/reference_parity.npz)."""
import io
import os

import numpy as np

DET_TXT = """1,-1,100.4,200.6,50.5,120.2,0.9,-1,-1,-1
1,-1,1800.0,900.0,200.0,300.0,0.4,-1,-1,-1
2,-1,10,20,30,40,1,-1,-1,-1
6,-1,640.5,360.5,11,21,1,-1,-1,-1
6,-1,0,0,1919,1079,1,-1,-1,-1
"""


def _make_sequence(tmp_path, w=1920, h=1080):
    seq = tmp_path / "MOT-TEST"
    (seq / "det").mkdir(parents=True)
    (seq / "seqinfo.ini").write_text(f"[Sequence]\nname=MOT-TEST\nimWidth={w}\nimHeight={h}\n")
    (seq / "det" / "det.txt").write_text(DET_TXT)
    return seq


def test_public_detector_rows(tmp_path):
    from fastmot_b200 import PublicDetector, DET_DTYPE
    seq = _make_sequence(tmp_path)
    det = PublicDetector((1280, 720), (1,), 5, sequence_path=str(seq), conf_thresh=0.5, max_area=800000)
    d0 = det(None)
    assert d0.dtype == DET_DTYPE and len(d0) == 2
    # to_tlbr: rint(100.4)=100, rint(200.6)=201, rint(100.4+50.5-1)=150, rint(200.6+120.2-1)=320, then x 2/3 and rint
    np.testing.assert_array_equal(d0.tlbr[0], np.rint(np.array([100, 201, 150, 320]) * (2 / 3)))
    assert list(d0.label) == [1, 1] and list(d0.conf) == [1.0, 1.0]     # confidences are forced to 1 (reference)
    d5 = det(None)                                                        # frame index 5 = file frame 6
    assert len(d5) == 1                                                   # the full-frame box exceeds max_area
    np.testing.assert_array_equal(d5.tlbr[0], np.rint(np.rint(np.array([640.5, 360.5, 650.5, 380.5])) * (2 / 3)))
    assert len(det(None)) == 0                                            # frame 10: nothing
    # a larger max_area keeps the full-frame box (1280 x 720 inclusive pixels)
    det2 = PublicDetector((1280, 720), (1,), 5, sequence_path=str(seq), max_area=1000000)
    det2(None)
    d5b = det2(None)
    assert len(d5b) == 2
    np.testing.assert_array_equal(d5b.tlbr[1], [0, 0, 1279, 719])


def test_public_detector_matches_reference(tmp_path, golden_dir):
    from fastmot_b200 import PublicDetector
    g = np.load(os.path.join(golden_dir, "reference_parity.npz"))
    assert str(g["pub_det_txt"]) == DET_TXT
    seq = _make_sequence(tmp_path, 1920, 1080)
    for j, size in enumerate(((1280, 720), (1920, 1080), (640, 360))):
        ours = PublicDetector(size, (1,), 5, sequence_path=str(seq), conf_thresh=0.5, max_area=800000)
        for c in range(3):
            a = ours.postprocess()
            assert len(a) == len(g[f"pub_tlbr_{j}_{c}"])
            np.testing.assert_array_equal(a.tlbr, g[f"pub_tlbr_{j}_{c}"])
            np.testing.assert_array_equal(a.label, g[f"pub_label_{j}_{c}"])
            np.testing.assert_array_equal(a.conf, g[f"pub_conf_{j}_{c}"])


def test_mot_result_line_format():
    from fastmot_b200.utils.mot_io import mot_result_line, write_mot_results

    class _T:
        def __init__(self, i, tlbr):
            self.trk_id, self.tlbr = i, np.asarray(tlbr, float)

    class _M:
        frame_count = 6

        def visible_tracks(self):
            return iter([_T(1, [136, 541, 222, 719]), _T(2, [233, 542, 307, 719])])

    line = mot_result_line(6, 1, [136, 541, 222, 719], (1280, 720), (1920, 1080))
    assert line == "6,1,204.000000,811.500000,130.000000,268.000000,-1,-1,-1\n"   # eval/results/MOT20-01.txt:1
    buf = io.StringIO()
    write_mot_results(buf, _M(), (1280, 720), (1920, 1080))
    assert buf.getvalue().splitlines()[1] == "6,2,349.500000,813.000000,112.000000,266.500000,-1,-1,-1"
