"""Golden vectors for the tracker that consumes the detector output (SURVEY.md §8f N2).

TEST INFRASTRUCTURE, not product code.  Runs the *reference's own* tracker (ocsort_tracker/ocsort.py:163-308, imported
from /root/reference — only possible in the build container) and stores inputs and outputs as plain arrays:

  tests/golden/ocsort_mot16.npz     the reference's fixture test/tracks.pkl (1501 frames of (300,6) detector rows and the
                                    tracks its test/test_ocsort.py:8-14 expects), re-run through the reference here with
                                    OCSort(max_age=60), det_thresh 0.25, and checked equal to the pickle's expectation
  tests/golden/ocsort_street.npz    the reference's unused second fixture test/tracker_inputs.pkl (1500 frames of a street
                                    scene) through the reference with the product's settings (max_age=100, threshold 0.5)
                                    and with the BYTE stage on
  tests/golden/ocsort_synth.npz     three seeded synthetic scenes (crossing boxes, drop-outs, low-score rows, class flips)
                                    through the reference with other constructor arguments (use_byte, max_age, delta_t)
  tests/golden/ocsort_random.npz    twelve shorter seeded scenes, each with randomly drawn constructor arguments, through
                                    the reference; only the outputs are stored, the test regenerates the frames from the
                                    seeds with synthetic_scene()

Per frame the stored output rows are [tl_x, tl_y, w, h, score, class_id, track_id, tracklet_len, speed] (float64; float32
in ocsort_random.npz).

    python oracle/make_golden_ocsort.py
"""
import pickle
import sys
from pathlib import Path

import numpy as np

REF = Path("/root/reference")
OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def run_reference(frames, det_thresh, **kw):
    sys.path.insert(0, str(REF))
    from ocsort_tracker import ocsort
    trk = ocsort.OCSort(**kw)
    rows, offs = [], [0]
    for f in frames:
        out = trk.update(f, det_thresh)
        for x in out:
            t = x.tlwh
            rows.append([t[0], t[1], t[2], t[3], x.score, x.class_id, x.track_id, x.tracklet_len, x.speed])
        offs.append(len(rows))
    return np.asarray(rows, np.float64).reshape(-1, 9), np.asarray(offs, np.int64)


def synthetic_scene(seed, n_frames=240, n_obj=14, W=1280, H=720):
    """Boxes on straight/curved paths that cross each other, with detector-like jitter, drop-outs (occlusions of 1-40
    frames), low-confidence stretches (0.1 < s < 0.25, the BYTE band), class flips and a few false positives."""
    g = np.random.default_rng(seed)
    pos = g.uniform([100, 100], [W - 100, H - 100], (n_obj, 2))
    vel = g.uniform(-6, 6, (n_obj, 2))
    size = g.uniform([30, 60], [120, 220], (n_obj, 2))
    cls = g.integers(0, 6, n_obj)
    born = g.integers(0, n_frames // 3, n_obj)
    born[: n_obj // 2] = 0
    gone_until = np.zeros(n_obj, int)
    frames = []
    for f in range(n_frames):
        vel += g.normal(0, 0.15, vel.shape)
        pos += vel
        bounce = (pos < 40) | (pos > [W - 40, H - 40])
        vel[bounce] *= -1
        rows = []
        for i in range(n_obj):
            if f < born[i]:
                continue
            if f >= gone_until[i] and g.random() < 0.03:
                gone_until[i] = f + g.integers(1, 41)
            if f < gone_until[i]:
                continue
            wh = size[i] * (1 + g.normal(0, 0.02, 2))
            c = pos[i] + g.normal(0, 1.0, 2)
            s = g.uniform(0.3, 0.95) if g.random() > 0.12 else g.uniform(0.11, 0.249)
            k = cls[i] if g.random() > 0.08 else g.integers(0, 6)
            rows.append([c[0] - wh[0] / 2, c[1] - wh[1] / 2, c[0] + wh[0] / 2, c[1] + wh[1] / 2, s, k])
        for _ in range(g.poisson(0.3)):
            c, wh = g.uniform([50, 50], [W - 50, H - 50]), g.uniform(20, 90, 2)
            rows.append([c[0] - wh[0] / 2, c[1] - wh[1] / 2, c[0] + wh[0] / 2, c[1] + wh[1] / 2, g.uniform(0.26, 0.5), g.integers(0, 80)])
        rows.sort(key=lambda r: -r[4])                      # the detector emits rows by descending confidence
        a = np.zeros((300, 6), np.float32)
        if rows:
            a[: len(rows)] = np.asarray(rows, np.float32)
        frames.append(a)
    return np.stack(frames)


RANDOM_SEEDS = range(100, 112)


def random_scene(seed):
    """(frames, det_thresh, OCSort kwargs) of the random scene `seed`: constructor arguments, threshold and object count
    are drawn from the seed too."""
    g = np.random.default_rng(seed)
    kw = dict(max_age=int(g.choice([5, 30, 100])), min_hits=int(g.choice([1, 3])), iou_threshold=float(g.choice([0.2, 0.3, 0.5])),
              delta_t=int(g.choice([1, 2, 3])), inertia=float(g.choice([0.0, 0.2, 0.4])), use_byte=bool(g.integers(0, 2)))
    thr = float(g.choice([0.25, 0.4, 0.5]))
    return synthetic_scene(seed, n_frames=100, n_obj=int(g.integers(3, 25))), thr, kw


def make_random_scenes():
    out = {}
    for seed in RANDOM_SEEDS:
        frames, thr, kw = random_scene(seed)
        rows, offs = run_reference(frames, thr, **kw)
        out[f"{seed}_rows"], out[f"{seed}_offsets"] = rows.astype(np.float32), offs.astype(np.int32)     # float32: far below rtol 1e-5
        out[f"{seed}_frames_sum"] = frames.astype(np.float64).sum()      # detects a change of synthetic_scene's output
    np.savez_compressed(OUT / "ocsort_random.npz", **out)


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    sys.path.insert(0, str(REF))
    tracks = pickle.load(open(REF / "test" / "tracks.pkl", "rb"))
    frames = np.stack([t[0] for t in tracks]).astype(np.float32)
    rows, offs = run_reference(frames, 0.25, max_age=60)
    # the pickle's own expectation (test/test_ocsort.py:12-14), same comparison the reference test makes
    for i, t in enumerate(tracks):
        exp = np.array([[x.tlwh[0], x.tlwh[1], x.tlwh[0] + x.tlwh[2], x.tlwh[1] + x.tlwh[3], x.score, x.class_id] for x in t[1]])
        got = rows[offs[i]:offs[i + 1]]
        got = np.stack([got[:, 0], got[:, 1], got[:, 0] + got[:, 2], got[:, 1] + got[:, 3], got[:, 4], got[:, 5]], 1) if len(got) else got
        np.testing.assert_allclose(got.reshape(-1, 6), exp.reshape(-1, 6), rtol=1e-5)
    np.savez_compressed(OUT / "ocsort_mot16.npz", frames=frames, rows=rows, offsets=offs, det_thresh=0.25, max_age=60)
    print("mot16:", frames.shape, rows.shape)

    scenes = {}
    for name, seed, thr, kw in [("a", 11, 0.25, dict(max_age=100)),
                                ("b", 12, 0.4, dict(max_age=8, min_hits=2, delta_t=2, use_byte=True)),
                                ("c", 13, 0.25, dict(max_age=30, iou_threshold=0.2, inertia=0.4, use_byte=True))]:
        fr = synthetic_scene(seed)
        rows, offs = run_reference(fr, thr, **kw)
        scenes[f"{name}_frames"], scenes[f"{name}_rows"], scenes[f"{name}_offsets"] = fr, rows, offs
        scenes[f"{name}_args"] = np.array([thr, kw.get("max_age", 30), kw.get("min_hits", 3), kw.get("iou_threshold", 0.3),
                                           kw.get("delta_t", 3), kw.get("inertia", 0.2), float(kw.get("use_byte", False))])
        print(name, fr.shape, rows.shape, "ids up to", rows[:, 6].max())
    np.savez_compressed(OUT / "ocsort_synth.npz", **scenes)

    # the reference's second, unused fixture: 1500 frames of recorded detections from another (street, mostly cars) video
    real = np.stack(pickle.load(open(REF / "test" / "tracker_inputs.pkl", "rb"))).astype(np.float32)
    out = {"frames": real}
    for name, thr, kw in [("a", 0.5, dict(max_age=100)), ("b", 0.25, dict(max_age=30, use_byte=True))]:   # a = clearcam.py:239,584
        rows, offs = run_reference(real, thr, **kw)
        out[f"{name}_rows"], out[f"{name}_offsets"] = rows, offs
        out[f"{name}_args"] = np.array([thr, kw["max_age"], float(kw.get("use_byte", False))])
        print("tracker_inputs", name, rows.shape, "ids up to", rows[:, 6].max())
    np.savez_compressed(OUT / "ocsort_street.npz", **out)
    make_random_scenes()


if __name__ == "__main__":
    main()
