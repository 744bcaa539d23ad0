"""not-gpu: the post-processing oracle (oracle/postprocess_ref.py) against the picks of the reference's own
`_detect_peaks`, stored in tests/golden/reference_checks.npz (tests/golden/make_reference_checks.py)."""
import os

import numpy as np
import pytest

import reference_inputs as I
from oracle import postprocess_ref as PR

REF = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz"))


@pytest.mark.parametrize("topk,mpd", I.PICK_CASES)
def test_pick_phase_matches_reference_detect_peaks(topk, mpd):
    x = I.pick_traces(topk, mpd)
    assert np.array_equal(I.probe(x), REF[f"pick.{topk}_{mpd}.x_probe"]), "seeded input changed"
    for thr in I.PICK_THRESHOLDS:
        mine = PR.pick_phase(x, thr, mpd, topk)
        ref = REF[f"pick.{topk}_{mpd}.{thr}"]
        for i in range(x.shape[0]):
            want = ref[i][ref[i] != PR.PAD_PHASE]
            got = mine[i][mine[i] != PR.PAD_PHASE]
            assert np.array_equal(got, want), (i, thr, got, want)
            assert (mine[i][got.size:] == PR.PAD_PHASE).all()


def test_detect_event_runs_and_padding():
    x = np.zeros((3, 64), dtype=np.float32)
    x[0, 5:9] = 0.9
    x[0, 20:40] = 0.7
    x[0, 63] = 0.9                      # run of one sample touching the end
    x[1, :] = 0.9                       # one run covering everything
    out = PR.detect_event(x, 0.5, 2)
    assert out[0].tolist() == [20, 39, 5, 8]
    assert out[1].tolist() == [0, 63, 1, 0]
    assert out[2].tolist() == [1, 0, 1, 0]
    assert PR.detect_event(x, 0.5, 1)[0].tolist() == [20, 39]
    x[2, 10:14] = 0.6
    x[2, 30:34] = 0.6                   # equal lengths: the earlier run first (stable sort)
    assert PR.detect_event(x, 0.5, 2)[2].tolist() == [10, 13, 30, 33]
    assert PR.detect_event(np.full((1, 8), 0.5, np.float32), 0.5, 1)[0].tolist() == [1, 0]     # strict >


def test_counters():
    t = np.array([[100], [200], [-10000000], [300]])
    p = np.array([[103], [260], [50], [-10000000]])
    c = PR.pick_counters(t, p, 8192, 5)
    assert (c["tp"], c["predp"], c["possp"], c["data_size"]) == (1, 3, 3, 4)
    assert c["sum_res"] == -3.0 and c["sum_abs_res"] == 3.0 and c["sum_squ_res"] == 9.0
    d = PR.det_counters(np.array([[10, 19], [1, 0]]), np.array([[15, 30], [5, 6]]), 64)
    assert (d["tp"], d["predp"], d["possp"]) == (5, 18, 10)
