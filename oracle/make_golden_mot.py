"""The reference's end-to-end known answer for the detector -> tracker chain (test/run_mot.py:14-51): YOLOv9-t at res 960
on every frame of test/videos/MOT16-03.mp4 (float32 frames), OCSort(max_age=60).update(pred, 0.25), count the distinct
person tracks with tracklet_len >= 1 and speed >= 2.5 -> the reference asserts 156.

TEST INFRASTRUCTURE.  The reference's detector cannot run here (tinygrad) and its weights are fetched from HuggingFace;
this script runs the ORACLE detector with the YOLOv9-t weights recovered from the reference's iOS model blob
(oracle/extract_ios_weights.py -> tests/golden/yolov9t_mot16.npz) on the reference's own video and stores the (1501,300,6)
detections in tests/golden/mot16_oracle_dets.npz for tests/test_oracle_cpu.py.  bgr_swap=False: the configuration that also
reproduces the detections recorded in test/tracks.pkl (SURVEY.md D10: the reference's fixtures were recorded by a detector
revision without the BGR->RGB swap of detection/yolov9.py:378; either that, or the blob's first conv is stored in BGR order).

Measured here: 156 people tracks = the reference's known answer.  The statistic is sensitive at the +-2 % level: the same
chain gives 159 with the channel swap, 155 with the bf16-mirror oracle and 153 from the older-revision detections stored
in test/tracks.pkl.

    CLEARCAM_B200_MOT_VIDEO=<the reference's test/videos/MOT16-03.mp4> python oracle/make_golden_mot.py    # ~100 s on 8 cores
"""
import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
VIDEO = os.environ.get("CLEARCAM_B200_MOT_VIDEO", "")


def count_people(dets, tracker):
    ppl = set()
    for pred in dets:
        for x in tracker.update(pred, 0.25):
            if x.tracklet_len < 1 or x.speed < 2.5:          # run_mot.py:41
                continue
            if x.class_id == 0:
                ppl.add(x.track_id)                            # run_mot.py:42
    return len(ppl)


def main():
    import cv2
    from oracle import yolov9 as o
    g = np.load(ROOT / "tests" / "golden" / "yolov9t_mot16.npz")
    P = {k[2:]: torch.from_numpy(g[k]) for k in g.keys() if k.startswith("w:")}
    cap = cv2.VideoCapture(VIDEO)
    dets = []
    while True:
        ret, im = cap.read()
        if not ret:
            break
        with torch.no_grad():
            dets.append(o.detect("t", P, torch.from_numpy(im).float()[None], 960, bgr_swap=False)[0].numpy())
    dets = np.stack(dets)
    sys.path.insert(0, "/root/reference")
    from ocsort_tracker import ocsort as ref_ocsort           # the reference's own tracker on the same detections
    n_ref = count_people(dets, ref_ocsort.OCSort(max_age=60))
    print("frames", len(dets), "people tracks (reference tracker):", n_ref)
    np.savez_compressed(ROOT / "tests" / "golden" / "mot16_oracle_dets.npz", dets=dets, people=n_ref, expected=156)


def make_frame1():
    """mot16_frame1.npz: frame 1 of the video as its difference from frame 0 (the frame stored in yolov9t_mot16.npz); the
    camera is static, so the difference compresses to a few KB.  tests/test_oracle_cpu.py runs the oracle on frames 0 and 1
    and compares with the stored detections."""
    import cv2
    f0 = np.load(ROOT / "tests" / "golden" / "yolov9t_mot16.npz")["frame"]
    cap = cv2.VideoCapture(VIDEO)
    ok0, im0 = cap.read()
    ok1, im1 = cap.read()
    assert ok0 and ok1 and np.array_equal(im0, f0)
    d = im1.astype(np.int16) - f0
    assert np.abs(d).max() < 128
    np.savez_compressed(ROOT / "tests" / "golden" / "mot16_frame1.npz", delta_from_frame0=d.astype(np.int8))


if __name__ == "__main__":
    main()
    make_frame1()
