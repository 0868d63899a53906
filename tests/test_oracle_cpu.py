"""CPU tests (no GPU): the oracle against the reference's own fixtures / identities, the tokenizer against the
reference tokenizer's recorded ids, host logic, and the C-ABI library surface."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import yolov9 as o
from oracle import clip as oc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ------------------------------------------------------------------------------------------------ graph identities
@pytest.mark.parametrize("size,convs,params_m,gflop", [("t", 185, 2.00, 7.71), ("c", 144, 25.29, 102.14), ("e", 261, 57.35, 188.95)])
def test_graph_matches_published_counts(size, convs, params_m, gflop):
    """SURVEY.md §6: the restated graphs reproduce the published YOLOv9 parameter/FLOP numbers."""
    tab = o.conv_table(size)
    assert len(tab) == convs
    n = sum(co * (ci // g) * k * k + co for _, ci, co, k, s, g, a in tab) + 16
    assert abs(n / 1e6 - params_m) < 0.01
    assert abs(o.conv_flops(size, 640, 640) / 1e9 - gflop) < 0.01


def test_clip_flops_identities():
    assert abs(oc.flops_image(oc.VIT_L_14) / 1e9 - 162.03) < 0.01 and abs(oc.flops_text(oc.VIT_L_14) / 1e9 - 13.30) < 0.01
    assert abs(oc.flops_image(oc.VIT_B_32) / 1e9 - 8.82) < 0.01 and abs(oc.flops_text(oc.VIT_B_32) / 1e9 - 5.96) < 0.01


# ------------------------------------------------------------------------------------------------ reference fixture
def test_oracle_reproduces_reference_recorded_detections():
    """Real YOLOv9-t weights (from the reference's iOS bundle) + frame 0 of its MOT16-03 test video vs the detector
    output the reference recorded in test/tracks.pkl (older revision without the BGR swap, SURVEY D10)."""
    z = np.load(os.path.join(GOLD, "yolov9t_mot16.npz"))
    P = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    frame, ref = torch.from_numpy(z["frame"]), torch.from_numpy(z["ref_preds"])
    assert o.count_params(P) == 2001840
    out = o.detect("t", P, frame, 960, bgr_swap=False)[0]
    A, Bq = ref[ref[:, 4] > 0], out[out[:, 4] > 0]
    d = (A[:, None, :4] - Bq[None, :, :4]).abs().max(-1)[0] + (A[:, None, 5] != Bq[None, :, 5]) * 1e6
    md, mi = d.min(1)
    ok = md < 3.0
    assert len(A) == 34 and int(ok.sum()) >= 32
    assert float(md[ok].median()) < 0.5
    assert float((A[ok, 4] - Bq[mi[ok], 4]).abs().max()) < 0.06


# ------------------------------------------------------------------------------------------------ semantics units
def test_letterbox_params_match_reference_examples():
    # 1080p @ res 640 -> 360x640 resized, pad 12/12 -> 384x640 (SURVEY D8); square stays identity
    assert o.letterbox_params(1080, 1920, 640) == (640, 360, 0, 12)
    assert o.letterbox_params(640, 640, 640) == (640, 640, 0, 0)
    assert o.letterbox_params(540, 960, 960) == (960, 540, 0, 2)
    img = torch.zeros(1080, 1920, 3, dtype=torch.uint8)
    assert o.preprocess(img, 640).shape == (384, 640, 3)


def test_resize_identity_and_dtype():
    img = (torch.arange(6 * 8 * 3) % 251).reshape(6, 8, 3).to(torch.uint8)
    assert torch.equal(o.resize(img, (8, 6)), img)
    up = o.resize(img, (16, 12))
    assert up.dtype == torch.uint8 and up.shape == (12, 16, 3)
    upf = o.resize(img.float(), (16, 12))
    assert upf.dtype == torch.float32 and (upf - up.float()).abs().max() <= 2.0


def test_postprocess_one_shot_suppression_and_stable_order():
    """A box is zeroed iff ANY higher-ranked same-class box overlaps it > 0.45, even a suppressed one
    (detection/yolov9.py:453-458); ties keep ascending anchor order."""
    A = 400
    raw = torch.zeros(1, 84, A)
    raw[0, 2:4] = 1.0
    def put(i, x, y, w, h, cls, p):
        raw[0, 0, i], raw[0, 1, i], raw[0, 2, i], raw[0, 3, i] = x, y, w, h
        raw[0, 4 + cls, i] = p
    put(10, 100, 100, 50, 50, 3, 0.9)
    put(20, 104, 100, 50, 50, 3, 0.8)     # suppressed by #10
    put(30, 112, 100, 50, 50, 3, 0.7)     # IoU with #10 < 0.45? (0.63 -> suppressed) and with #20 (0.72)
    put(40, 300, 300, 20, 20, 3, 0.6)     # far away: kept
    put(50, 100, 100, 50, 50, 5, 0.5)     # other class: kept
    put(7, 200, 200, 10, 10, 1, 0.5)      # same conf as #50, lower index -> ranked first
    out = o.postprocess(raw)[0]
    assert out.shape == (300, 6)
    assert out[0, 4] == pytest.approx(0.9) and out[1].abs().sum() == 0 and out[2].abs().sum() == 0
    assert out[3, 4] == pytest.approx(0.6)
    assert out[4, 5] == 1 and out[5, 5] == 5          # stable tie order
    assert (out[6:, 4] == 0).all()


def test_scale_boxes_uses_float_pad_and_clips():
    p = torch.tensor([[[10.0, 20.0, 700.0, 400.0, 0.9, 1.0]]])
    s = o.scale_boxes((384, 640), p, (1080, 1920))
    gain = min(384 / 1080, 640 / 1920)
    assert s[0, 0, 0] == pytest.approx((10 - 0) / gain) and s[0, 0, 2] == 1920
    assert s[0, 0, 1] == pytest.approx((20 - (384 - 1080 * gain) / 2) / gain)


def test_bf16_mirror_differs_only_by_rounding():
    P = o.synthetic_weights("t", seed=1)
    x = o.synthetic_frames(1, 128, 160, seed=2).flip(-1).permute(0, 3, 1, 2).float() / 255
    with torch.no_grad():
        a, b = o.forward_raw("t", P, x), o.forward_raw("t", P, x, quant="bf16")
    assert (a[:, 4:] - b[:, 4:]).abs().max() < 0.1 and not torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ tokenizer
def test_tokenizer_matches_reference_ids():
    from clearcam_b200.utils.clip_tokenizer import SimpleTokenizer
    gold = json.load(open(os.path.join(GOLD, "clip_tokens.json")))
    tok = SimpleTokenizer()
    for p, ids in zip(gold["prompts"], gold["ids"]):
        assert tok.encode(p) == ids, p
    assert tok.encode("ferrari f40") == [9606, 325, 275, 271]          # SURVEY §2 known answer
    assert oc.pad_tokens([tok.encode("ferrari f40")])[0, :6].tolist() == [49406, 9606, 325, 275, 271, 49407]


def test_clip_oracle_shapes_and_norms():
    cfg = oc.VIT_TINY
    P = oc.synthetic_weights(cfg, 0)
    e = oc.encode_image(cfg, P, oc.synthetic_images(3, cfg.image_size))
    t = oc.encode_text_ids(cfg, P, oc.pad_tokens([[1, 2, 3], [5]]))
    assert e.shape == (3, cfg.embed_dim) and t.shape == (2, cfg.embed_dim)
    assert (e.norm(dim=-1) - 1).abs().max() < 1e-5 and (t.norm(dim=-1) - 1).abs().max() < 1e-5
    with pytest.raises(ValueError):
        oc.pad_tokens([list(range(80))])                               # the reference does not truncate


# ------------------------------------------------------------------------------------------------ C-ABI surface
def test_library_exports_every_declared_symbol():
    from clearcam_b200._lib import lib, declared_symbols, LIB_PATH
    hdr = open(os.path.join(ROOT, "include", "clearcam_b200.h")).read()
    declared = set(re.findall(r"\b(cc_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"cc_clip_config"}
    h = ctypes.CDLL(LIB_PATH)
    for name in sorted(declared):
        assert hasattr(h, name), f"{name} declared in include/clearcam_b200.h but not exported"
    assert declared == set(declared_symbols()), "ctypes signature table out of sync with the header"
    assert lib().cc_version() == 1


def test_product_path_fails_loudly_without_gpu():
    """No CPU fallback: on a box without a B200 the drop-ins raise instead of computing something."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from clearcam_b200 import CCError
    from clearcam_b200.detection.yolov9 import YOLOv9
    from clearcam_b200.models.objects import OpenCLIP
    with pytest.raises(CCError):
        YOLOv9("t", 320, weights={})
    with pytest.raises(CCError):
        OpenCLIP(weights={}, arch="ViT-tiny")


def test_shard_range_partitions():
    from clearcam_b200.parallel import shard_range
    for n in (0, 1, 7, 32, 128, 1001):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, world, r) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_fp32_noise_floor_of_the_reference_arithmetic():
    """The north-star bar (boxes within 1e-3 px of the fp32 path) is below what fp32 arithmetic itself reproduces:
    the SAME oracle on the reference's real YOLOv9-t weights and a real frame moves boxes by more than 1e-3 px when
    only the summation precision/order changes (fp32 vs fp64 accumulate).  Class probabilities stay within 1e-4."""
    z = np.load(os.path.join(GOLD, "yolov9t_mot16.npz"))
    P = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    pre = o.preprocess(torch.from_numpy(z["frame"]), 640)
    x = pre.flip(-1).permute(2, 0, 1).unsqueeze(0).float() / 255
    with torch.no_grad():
        r32 = o.forward_raw("t", P, x)
        r64 = o.forward_raw("t", {k: v.double() for k, v in P.items()}, x.double())
    d = (r32.double() - r64).abs()
    assert d[:, :4].max() > 1e-3, "fp32 and fp64 evaluation agree to 1e-3 px?"
    assert d[:, :4].mean() < 1e-3 and d[:, 4:].max() < 1e-4


@pytest.mark.parametrize("size", ["t", "m"])
def test_zero_padded_equivalent_computes_the_same_function(size):
    """YOLOv9-t / -m run on the GPU as their zero-padded equivalents (widths rounded up to multiples of 16, weights scattered
    by clearcam_b200/detection/padding.py).  The oracle evaluates both the reference-shaped and the padded model: the
    head tensors and the detections agree to fp32 summation order."""
    from clearcam_b200.detection.padding import pad_state_dict, padded_size, layer_channel_maps, PADDED
    torch.set_num_threads(min(8, torch.get_num_threads()))
    fr = o.synthetic_frames(2, 128, 160, seed=3)
    x = fr.flip(-1).permute(0, 3, 1, 2).float() / 255
    P = o.synthetic_weights(size, seed=1, calib=x[:1])
    P16 = {k: torch.from_numpy(np.asarray(v)) for k, v in pad_state_dict(size, {k: v.numpy() for k, v in P.items()}).items()}
    taps, taps16 = [], []
    with torch.no_grad():
        y = o.forward_raw(size, P, x, taps=taps)
        y16 = o.forward_raw(padded_size(size), P16, x, taps=taps16)
    assert float((y - y16).abs().max()) <= 2e-5 * float(y.abs().max())
    maps = layer_channel_maps(size)
    for i, idx in enumerate(maps):                      # every layer: real channels equal, padding channels exactly zero
        a, b = taps[i], taps16[i]
        assert torch.allclose(b[:, torch.from_numpy(idx)], a, rtol=1e-4, atol=1e-4 * float(a.abs().max())), f"layer {i}"
        pad = torch.ones(b.shape[1], dtype=torch.bool)
        pad[torch.from_numpy(idx)] = False
        assert float(b[:, pad].abs().max()) == 0.0 if pad.any() else True
    assert all(v % 16 == 0 for k, v in zip("abcdefghijklmnpqrstuvw", PADDED[size]) if k not in "p")
    d, d16 = o.detect(size, P, fr, 128), o.detect(padded_size(size), P16, fr, 128)
    assert float((d - d16).abs().max()) < 1e-2


def test_tokenizer_live_against_the_reference_on_random_text():
    """300 generated texts — mixed case, digits, punctuation, apostrophe forms, runs of spaces, accented and non-Latin
    characters, emoji, html entities — against the ids the reference's own tokenizer module gave for them
    (clip_tokens_random.json, from oracle/make_golden.py)."""
    from clearcam_b200.utils.clip_tokenizer import SimpleTokenizer
    tok = SimpleTokenizer()
    gold = json.load(open(os.path.join(GOLD, "clip_tokens_random.json")))
    assert len(gold["texts"]) == 300
    for text, ids in zip(gold["texts"], gold["ids"]):
        assert tok.encode(text) == ids, repr(text)


def test_reference_known_answer_156_people_tracks_on_mot16():
    """test/run_mot.py:14-51, the reference's end-to-end check of detector + tracker: YOLOv9-t (res 960) on every frame of
    MOT16-03.mp4 -> OCSort(max_age=60) -> 156 distinct moving person tracks.  The detections are the ORACLE's (with the
    YOLOv9-t weights recovered from the reference's iOS blob, channel swap off as for test/tracks.pkl; oracle/make_golden_mot.py), the tracker is the product's C++
    one: the chain lands on the reference's number exactly.  (The statistic moves by +-2 % with rounding: see the script.)"""
    from clearcam_b200.ocsort_tracker import ocsort
    g = np.load(os.path.join(GOLD, "mot16_oracle_dets.npz"))
    dets = g["dets"]
    assert dets.shape == (1501, 300, 6) and int(g["expected"]) == 156
    trk, ppl = ocsort.OCSort(max_age=60), set()
    for pred in dets:
        for x in trk.update(pred, 0.25):
            if x.tracklet_len < 1 or x.speed < 2.5:
                continue
            if x.class_id == 0:
                ppl.add(x.track_id)
    assert len(ppl) == 156
    # tie the stored detections to the oracle code: its detections on the video's first two frames
    w = np.load(os.path.join(GOLD, "yolov9t_mot16.npz"))
    P = {k[2:]: torch.from_numpy(w[k]) for k in w.keys() if k.startswith("w:")}
    f0 = w["frame"]
    f1 = (f0 + np.load(os.path.join(GOLD, "mot16_frame1.npz"))["delta_from_frame0"]).astype(np.uint8)
    for i, im in enumerate((f0, f1)):
        with torch.no_grad():
            pred = o.detect("t", P, torch.from_numpy(im).float()[None], 960, bgr_swap=False)[0].numpy()
        live = dets[i][:, 4] > 0
        assert (pred[:, 4] > 0).sum() == live.sum()
        np.testing.assert_allclose(pred[live], dets[i][live], rtol=0, atol=2e-2)
