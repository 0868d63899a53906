"""Generates the committed golden fixtures under tests/golden/ from the REFERENCE tree (run here, where
/root/reference exists; the GPU box only sees the fixtures).  Usage: python oracle/make_golden.py

  yolov9t_mot16.npz: real YOLOv9-t weights + one real frame + the reference's recorded detections (see below)
  clip_tokens.json : token ids of fixed prompts from the reference's own utils/clip_tokenizer.py (imported, not copied)
                     -> pins clearcam_b200/utils/clip_tokenizer.py (tests/test_tokenizer_cpu.py)
  clip_tokens_random.json: the same for 300 generated texts (tests/test_oracle_cpu.py)
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference"
PROMPTS = [
    "ferrari f40", "text here", "a photo of a cat", "person riding a bicycle at night", "Red TRUCK, parked!!",
    "it's 3 o'clock &amp; raining", "naïve café — déjà vu", "  multiple   spaces\tand\nnewlines ", "don't we've I'll he'd",
    "email@example.com 12345 #hashtag", "日本語のテキスト", "emoji 😀 test", "<start_of_text> weird <end_of_text>", "a" * 40,
    "white van with ladder on roof", "delivery driver carrying a box", "dog", "UPS", "x",
    "a man in a yellow jacket walking a large black dog past a parked silver car on a rainy evening",
]


def main():
    sys.path.insert(0, REF)
    from utils.clip_tokenizer import SimpleTokenizer  # the reference's tokenizer
    tok = SimpleTokenizer()
    out = {"source": "reference utils/clip_tokenizer.py SimpleTokenizer.encode", "prompts": PROMPTS,
           "ids": [tok.encode(p) for p in PROMPTS]}
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    with open(os.path.join(ROOT, "tests", "golden", "clip_tokens.json"), "w") as f:
        json.dump(out, f, ensure_ascii=True, indent=0)
    print("wrote clip_tokens.json:", len(PROMPTS), "prompts")


WORDS = ["person", "Ferrari", "F40", "don't", "it's", "we'll", "I'M", "dog's", "naïve", "café", "Zürich", "北京", "мотоцикл", "🚗", "😀",
         "&amp;", "&lt;b&gt;", "3.14", "1080p", "a", "THE", "x-ray", "e-mail", "#tag", "@home", "100%", "(red)", "white/blue", "...",
         "  ", "\t", "van", "ladder", "night-time", "ＦＵＬＬ", "ﬁre", "o'clock", "10:30", "$5", "état", "straße"]


def make_random_tokens():
    """clip_tokens_random.json: 300 generated texts (mixed case, digits, punctuation, apostrophe forms, runs of spaces,
    accented and non-Latin characters, emoji, html entities) and the reference tokenizer's ids for them."""
    import numpy as np
    sys.path.insert(0, REF)
    from utils.clip_tokenizer import SimpleTokenizer
    tok = SimpleTokenizer()
    rng = np.random.default_rng(0)
    texts = [" ".join(WORDS[int(i)] for i in rng.integers(0, len(WORDS), int(rng.integers(1, 9)))) for _ in range(300)]
    out = {"source": "reference utils/clip_tokenizer.py SimpleTokenizer.encode", "texts": texts, "ids": [tok.encode(t) for t in texts]}
    with open(os.path.join(ROOT, "tests", "golden", "clip_tokens_random.json"), "w") as f:
        json.dump(out, f, ensure_ascii=True, separators=(",", ":"))



def make_yolov9t_fixture():
    """yolov9t_mot16.npz: the reference's REAL YOLOv9-t weights (recovered from ios/clearcam/yolov9t by
    oracle/extract_ios_weights.py), frame 0 of test/videos/MOT16-03.mp4 (cv2 decode, BGR uint8 540x960) and the
    reference's own recorded detector output for that frame, test/tracks.pkl[0][0] (300,6) — recorded by an older
    detector revision without the BGR->RGB swap (SURVEY.md D10), so it pins the oracle only loosely
    (tests/test_oracle_cpu.py: >= 32/34 boxes within 3 px, confidences within 0.06)."""
    import pickle
    import cv2
    import numpy as np
    sys.path.insert(0, ROOT)
    from oracle.extract_ios_weights import extract
    P, used, total = extract()
    assert used == total
    cap = cv2.VideoCapture(os.path.join(REF, "test/videos/MOT16-03.mp4"))
    ok, frame = cap.read()
    assert ok and frame.shape == (540, 960, 3)
    tracks = pickle.load(open(os.path.join(REF, "test/tracks.pkl"), "rb"))
    ref = np.asarray(tracks[0][0], dtype=np.float32)
    arrays = {"w:" + k: v.numpy() for k, v in P.items()}
    arrays["frame"] = frame
    arrays["ref_preds"] = ref
    path = os.path.join(ROOT, "tests", "golden", "yolov9t_mot16.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, os.path.getsize(path) / 1e6, "MB")


if __name__ == "__main__":
    main()
    make_random_tokens()
    make_yolov9t_fixture()
