"""Generate the golden vectors under tests/golden/ (run in the authoring container; cv2 4.13 is the third-party library the
reference calls for these primitives, the reference binary itself cannot be built here -- see DESIGN.md section 4).

    python tools/gen_golden.py

cv2_primitives.npz  cv::resize / cv::FAST / cv::GaussianBlur 7x7 + 5x5 / cv::Sobel / cv::fastAtan2 on a seeded image
cv2_lsd.npz         cv::LineSegmentDetector(1, 0.5, 0.6, 2, 22.5, 1, 0.6, 1024) segments on two seeded images
orb_mirror.npz      orb_extractor::extract with every third-party stage done by cv2 (tests/test_orb_oracle.py mirror)
line_extract.npz    LineFeatureTracker::extract_LSD_LBD output of the oracle (whose LSD stage is pinned to cv2 above)
The images are regenerated from their seeds by the tests; only the outputs are stored.

    python tools/gen_golden.py --reference <Structure-PLP-SLAM source tree>

writes, instead, the fixtures taken from the reference's own data files (too large to store whole):
orb_vocab_sample.npz  orb_vocab/orb_vocab.dbow2: its header, every node a descent of the 16 test descriptors visits or
                      compares against (the children of each node on their paths), and transform()'s answers on the
                      whole file
equirectangular_image_00{1,2}_band.png
                      test/data/equirectangular_image_00{1,2}.jpg, grayscale, resized to 640x480, rows 120-359"""
import argparse
import sys
from pathlib import Path

import cv2
import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
import bow_data  # noqa: E402
import oracle_api  # noqa: E402
import synth  # noqa: E402
import test_orb_oracle  # noqa: E402

OUT = ROOT / "tests" / "golden"


def reference_fixtures(ref: Path, orc):
    # ---- the shipped vocabulary, pruned to the subtree the test descents touch
    path = ref / "orb_vocab" / "orb_vocab.dbow2"
    raw = np.fromfile(path, np.uint8)
    header, rec = raw[:24].copy(), raw[24:].reshape(-1, 41)
    vocab = dict(k=10, L=6, parent=rec[:, :4].copy().view("<i4").ravel(), desc=rec[:, 4:36],
                 weight=rec[:, 36:40].copy().view("<f4").ravel(), is_leaf=rec[:, 40])
    rng = np.random.default_rng(0)
    queries = np.concatenate([synth.rand_desc(rng, 8),
                              synth.flip_bits(rng, vocab["desc"][rng.integers(0, len(rec), 8)], 12)])
    v = orc.bow_vocab_load(path)
    info = orc.bow_vocab_info(v)
    word, node, w = orc.bow_transform(v, queries, 4)
    orc.bow_vocab_destroy(v)
    assert [(int(a), int(b), float(c)) for a, b, c in zip(word, node, w)] == bow_data.transform_numpy(vocab, queries, 4)
    n_nodes = len(vocab["parent"]) + 1
    by_parent = np.argsort(vocab["parent"], kind="stable") + 1                 # node ids, grouped by parent, file order
    first_child = np.searchsorted(vocab["parent"][by_parent - 1], np.arange(n_nodes + 1))
    bits = np.unpackbits(vocab["desc"], axis=1)
    keep = set()
    for q in np.unpackbits(queries, axis=1):
        cur = 0
        while first_child[cur] < first_child[cur + 1]:
            ch = by_parent[first_child[cur]:first_child[cur + 1]]
            keep.update(ch.tolist())
            cur = int(ch[np.argmin((bits[ch - 1] != q).sum(1))])
    ids = np.array(sorted(keep), np.int32)
    word_of = np.cumsum(vocab["is_leaf"], dtype=np.int64) - 1
    np.savez_compressed(OUT / "orb_vocab_sample.npz", header=header,
                        info=np.array([info["k"], info["L"], info["num_nodes"], info["num_words"]], np.int32),
                        ids=ids, parent=vocab["parent"][ids - 1], desc=vocab["desc"][ids - 1],
                        weight=vocab["weight"][ids - 1], is_leaf=vocab["is_leaf"][ids - 1],
                        word_id=np.where(vocab["is_leaf"][ids - 1] > 0, word_of[ids - 1], -1).astype(np.int32),
                        queries=queries, word=word, node=node, node_weight=w)
    # ---- the reference's test images at the resolution of the LSD tests; the central band keeps the file small
    for i in (1, 2):
        img = cv2.imread(str(ref / "test" / "data" / f"equirectangular_image_00{i}.jpg"), cv2.IMREAD_GRAYSCALE)
        cv2.imwrite(str(OUT / f"equirectangular_image_00{i}_band.png"), cv2.resize(img, (640, 480))[120:360],
                    [cv2.IMWRITE_PNG_COMPRESSION, 9])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", type=Path, default=None, help="Structure-PLP-SLAM source tree")
    args = ap.parse_args()
    OUT.mkdir(exist_ok=True)
    orc = oracle_api.Oracle()
    if args.reference is not None:
        reference_fixtures(args.reference, orc)
        return
    tex = synth.make_texture(4321, 240, 320, n_rect=120, n_blob=500)      # the image of __graft_entry__.smoke()
    lines = synth.make_line_image(7, 240, 320, n_patch=16)
    # ---- third-party primitives
    lv1 = cv2.resize(tex, (267, 200), interpolation=cv2.INTER_LINEAR)      # round(320 / 1.2) x round(240 / 1.2)
    lv2 = cv2.resize(lv1, (222, 167), interpolation=cv2.INTER_LINEAR)
    roi = np.ascontiguousarray(tex[19:89, 83:153])
    fast = {}
    for thr in (20, 7):
        kk = cv2.FastFeatureDetector_create(thr, True).detect(roi)
        fast[thr] = np.array([(k.pt[0], k.pt[1], k.response) for k in kk], np.float32).reshape(-1, 3)
    blur7 = cv2.GaussianBlur(tex, (7, 7), 2, sigmaY=2, borderType=cv2.BORDER_REFLECT_101)
    blur5 = cv2.GaussianBlur(lines, (5, 5), 1.0)
    dx = cv2.Sobel(blur5, cv2.CV_16S, 1, 0, ksize=3)
    dy = cv2.Sobel(blur5, cv2.CV_16S, 0, 1, ksize=3)
    yy, xx = np.meshgrid(np.arange(-40, 41, 5, dtype=np.float32), np.arange(-40, 41, 5, dtype=np.float32), indexing="ij")
    at = np.array([cv2.fastAtan2(float(y), float(x)) for y, x in zip(yy.ravel(), xx.ravel())], np.float32)
    np.savez_compressed(OUT / "cv2_primitives.npz", resize1=lv1, resize2=lv2, fast20=fast[20], fast7=fast[7], blur7=blur7,
                        blur5=blur5, sobel_dx=dx, sobel_dy=dy, atan2_y=yy.ravel(), atan2_x=xx.ravel(), atan2=at,
                        cv2_version=np.array(cv2.__version__))
    # ---- LSD
    lsd = cv2.createLineSegmentDetector(1, 0.5, 0.6, 2.0, 22.5, 1.0, 0.6, 1024)
    seg = {}
    for name, img in (("lines", lines), ("texture", tex)):
        r = lsd.detect(img)[0]
        seg[name] = np.zeros((0, 4), np.float32) if r is None else r.reshape(-1, 4)
    np.savez_compressed(OUT / "cv2_lsd.npz", lines=seg["lines"], texture=seg["texture"])
    # ---- ORB through the cv2-driven mirror of orb_extractor.cc
    p = oracle_api.orb_params(500)
    kps, desc, _ = test_orb_oracle._cv2_mirror_extract(orc, p, tex)
    np.savez_compressed(OUT / "orb_mirror.npz", kps=kps, desc=desc)
    # ---- line extraction (oracle, LSD pinned to cv2)
    kl, lbd, fn = orc.line_extract(lines)
    np.savez_compressed(OUT / "line_extract.npz", keylines=kl, lbd=lbd, line_functions=fn)
    for f in sorted(OUT.glob("*.npz")):
        print(f.name, f.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
