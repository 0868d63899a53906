"""Tracker parity (SURVEY.md §8f N2): the C++ OC-SORT behind clearcam_b200.ocsort_tracker against golden vectors that
oracle/make_golden_ocsort.py produced by running the reference's own tracker (ocsort_tracker/ocsort.py) — on the
reference's fixture test/tracks.pkl (the sequence its test/test_ocsort.py asserts on) and on three synthetic scenes with
other constructor arguments.  Host code only: runs without a GPU."""
from pathlib import Path

import numpy as np
import pytest

from clearcam_b200.ocsort_tracker import ocsort
from clearcam_b200.ocsort_tracker.STrack import STrack

GOLD = Path(__file__).parent / "golden"


def _as_rows(tracks):
    return np.array([[*t.tlwh, t.score, t.class_id, t.track_id, t.tracklet_len, t.speed] for t in tracks], np.float64).reshape(-1, 9)


def _replay(frames, rows, offs, thr, **kw):
    trk = ocsort.OCSort(**kw)
    for i in range(len(frames)):
        got = _as_rows(trk.update(frames[i], thr))
        exp = rows[offs[i]:offs[i + 1]]
        assert got.shape == exp.shape, f"frame {i}: {got.shape[0]} tracks, reference has {exp.shape[0]}"
        # the reference's own test compares xyxy, score, class at rtol 1e-5 (test/test_ocsort.py:12-14); ids, lengths
        # and speeds are held to the same bar here
        np.testing.assert_allclose(got, exp, rtol=1e-5, atol=1e-9, err_msg=f"frame {i}")
    return trk


def test_reference_fixture_sequence():
    g = np.load(GOLD / "ocsort_mot16.npz")
    trk = _replay(g["frames"], g["rows"], g["offsets"], float(g["det_thresh"]), max_age=int(g["max_age"]))
    assert trk.frame_count == 1501 and len(trk) > 0


@pytest.mark.parametrize("scene", ["a", "b", "c"])
def test_synthetic_scenes_other_arguments(scene):
    s = np.load(GOLD / "ocsort_synth.npz")
    a = s[f"{scene}_args"]
    _replay(s[f"{scene}_frames"], s[f"{scene}_rows"], s[f"{scene}_offsets"], float(a[0]), max_age=int(a[1]), min_hits=int(a[2]),
            iou_threshold=float(a[3]), delta_t=int(a[4]), inertia=float(a[5]), use_byte=bool(a[6]))


def _replay_up_to_relabelling(frames, rows, offs, thr, **kw):
    """Every frame: the same rows (as a set) in everything but the track id, ids equal up to ONE consistent bijection."""
    trk, ids = ocsort.OCSort(**kw), {}
    for i in range(len(frames)):
        got, exp = _as_rows(trk.update(frames[i], thr)), rows[offs[i]:offs[i + 1]]
        assert got.shape == exp.shape, f"frame {i}"
        key = lambda a: np.lexsort((a[:, 3], a[:, 2], a[:, 1], a[:, 0]))       # noqa: E731
        got, exp = got[key(got)], exp[key(exp)]
        cols = [0, 1, 2, 3, 4, 5, 7, 8]
        np.testing.assert_array_equal(got[:, cols], exp[:, cols], err_msg=f"frame {i}")
        for a, b in zip(exp[:, 6], got[:, 6]):
            assert ids.setdefault(a, b) == b, f"frame {i}: track {a} relabelled inconsistently"
    assert len(set(ids.values())) == len(ids)
    return ids


@pytest.mark.parametrize("variant", ["a", "b"])
def test_street_scene_from_the_reference_second_fixture(variant):
    """test/tracker_inputs.pkl (1500 frames of real detections, mostly cars; unused by the reference's scripts) through the
    reference tracker with the product's settings (a: max_age=100, threshold 0.5, clearcam.py:239,584) and with BYTE on
    (b).  Bit-equal in every field of every frame; of ~250-320 tracks one or two born in the same frame as another get
    the other's number (the reference's argsort leaves the order of exactly tied costs unspecified)."""
    g = np.load(GOLD / "ocsort_street.npz")
    a = g[f"{variant}_args"]
    ids = _replay_up_to_relabelling(g["frames"], g[f"{variant}_rows"], g[f"{variant}_offsets"], float(a[0]), max_age=int(a[1]),
                                    use_byte=bool(a[2]))
    assert len(ids) > 200 and sum(x != y for x, y in ids.items()) <= 6


def test_batched_cameras_equal_single_calls():
    """update_many on B cameras (threaded inside the library) == B independent trackers stepped one by one."""
    s = np.load(GOLD / "ocsort_synth.npz")
    seqs = [s["a_frames"], s["b_frames"], s["c_frames"]] * 4          # 12 cameras -> 3 worker threads
    B, n = len(seqs), 120
    single = [ocsort.OCSort(max_age=20) for _ in range(B)]
    many = [ocsort.OCSort(max_age=20) for _ in range(B)]
    many[5] = None                                                      # a camera without a tracker
    for f in range(n):
        batch = np.stack([q[f] for q in seqs])
        got = ocsort.update_many(many, batch, 0.25)
        for b in range(B):
            exp = _as_rows(single[b].update(batch[b], 0.25))
            if many[b] is None:
                assert got[b] == []
            else:
                np.testing.assert_array_equal(_as_rows(got[b]), exp)


def test_contract_edges():
    trk = ocsort.OCSort(max_age=100)                                   # clearcam.py:239
    assert trk.update(None).shape == (0, 5)                            # ocsort.py:185-186
    assert trk.update(np.zeros((300, 6), np.float32), 0.5) == []       # a frame without detections still advances time
    rows = np.zeros((300, 6), np.float32)
    rows[0] = [10, 20, 110, 220, 0.9, 2]
    rows[1] = [400, 50, 460, 200, 0.2, 0]                              # below threshold: never starts a track
    out = trk.update(rows, 0.5)
    assert len(out) == 1 and isinstance(out[0], STrack)
    t = out[0]
    np.testing.assert_allclose(t.tlwh, [10, 20, 100, 200], rtol=1e-6)
    np.testing.assert_allclose(t.tlbr, [10, 20, 110, 220], rtol=1e-6)
    assert int(t.class_id) == 2 and int(t.track_id) == 1 and abs(t.score - 0.9) < 1e-6
    assert len(trk) == 1
    with pytest.raises(ValueError):
        trk.update(np.zeros((4, 5), np.float32))
    with pytest.raises(ValueError):
        ocsort.OCSort(asso_func="giou")
    # anything with .numpy() is accepted, like the detector's result object
    class R:
        def numpy(self): return rows
    assert len(trk.update(R(), 0.5)) == 1


def test_live_against_the_reference_tracker_on_random_scenes():
    """Twelve seeded random scenes with randomly drawn constructor arguments against the reference tracker's output on them
    (ocsort_random.npz, from oracle/make_golden_ocsort.py; the frames are regenerated here from the seeds).  Everything must
    agree frame by frame except the *numbering* of tracks born in the same frame: that order comes from how the reference's
    np.argsort happens to order exactly equal costs (zero-cost pairs of non-overlapping boxes), which numpy leaves unspecified
    and which differs between CPUs (SIMD sort dispatch).  So ids are compared up to one consistent relabelling per scene,
    rows as sets."""
    import sys
    sys.path.insert(0, str(Path(__file__).parent.parent / "oracle"))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from make_golden_ocsort import RANDOM_SEEDS, random_scene
        gold = np.load(GOLD / "ocsort_random.npz")
        relabelled = 0
        for seed in RANDOM_SEEDS:
            frames, thr, kw = random_scene(seed)
            assert frames.astype(np.float64).sum() == gold[f"{seed}_frames_sum"], f"seed {seed}: synthetic_scene changed"
            rows, offs = gold[f"{seed}_rows"].astype(np.float64), gold[f"{seed}_offsets"]
            trk, ids = ocsort.OCSort(**kw), {}
            for i in range(len(frames)):
                got = _as_rows(trk.update(frames[i], thr))
                exp = rows[offs[i]:offs[i + 1]]
                assert got.shape == exp.shape, f"seed {seed} frame {i}"
                key = lambda a: np.lexsort((a[:, 3], a[:, 2], a[:, 1], a[:, 0]))       # noqa: E731
                got, exp = got[key(got)], exp[key(exp)]
                cols = [0, 1, 2, 3, 4, 5, 7, 8]
                np.testing.assert_allclose(got[:, cols], exp[:, cols], rtol=1e-5, atol=1e-9, err_msg=f"seed {seed} frame {i}")
                for a, b in zip(exp[:, 6], got[:, 6]):
                    assert ids.setdefault(a, b) == b, f"seed {seed} frame {i}: track {a} relabelled inconsistently"
            assert len(set(ids.values())) == len(ids)                                    # one-to-one
            relabelled += any(a != b for a, b in ids.items())
        assert relabelled <= 3                                                            # rare: needs a tie in a frame that births two tracks
