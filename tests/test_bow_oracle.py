"""CPU tests: the oracle's DBoW2 vocabulary (binary loader + transform) against an independent numpy restatement, a
synthetic .dbow2 round trip and a sample of the shipped orb_vocab.dbow2 (tests/golden/orb_vocab_sample.npz, see
tools/gen_golden.py); the oracle's match::bow_tree against a line-by-line Python restatement."""
import struct
from pathlib import Path

import numpy as np
import pytest

import bow_data
import synth

VOCAB_SAMPLE = Path(__file__).resolve().parent / "golden" / "orb_vocab_sample.npz"


@pytest.mark.parametrize("k,L,levelsup", [(10, 3, 1), (4, 5, 4), (20, 2, 4), (10, 4, 2)])
def test_transform_matches_numpy_restatement(orc, tmp_path, k, L, levelsup):
    vocab = bow_data.make_vocab(k * 100 + L, k=k, L=L)
    rng = np.random.default_rng(L)
    leaves = vocab["desc"][vocab["is_leaf"] > 0]
    desc = np.concatenate([synth.rand_desc(rng, 60),
                           synth.flip_bits(rng, leaves[rng.integers(0, len(leaves), 140)], rng.integers(0, 30, 140))])
    v = orc.bow_vocab_create(k, L, vocab["parent"], vocab["desc"], vocab["weight"], vocab["is_leaf"])
    info = orc.bow_vocab_info(v)
    assert info == dict(k=k, L=L, num_nodes=len(vocab["parent"]) + 1, num_words=int(vocab["is_leaf"].sum()))
    word, node, w = orc.bow_transform(v, desc, levelsup)
    want = bow_data.transform_numpy(vocab, desc, levelsup)
    assert [(int(a), int(b), float(c)) for a, b, c in zip(word, node, w)] == want
    nid_level = L - levelsup
    if nid_level > 0:
        reached = node > 0
        assert np.all(vocab["level"][node[reached] - 1] == nid_level)
    else:
        assert np.all(node == 0)
    # the binary file round trip gives the same vocabulary
    path = tmp_path / "v.dbow2"
    bow_data.write_dbow2(path, vocab)
    v2 = orc.bow_vocab_load(path)
    assert orc.bow_vocab_info(v2) == info
    w2 = orc.bow_transform(v2, desc, levelsup)
    assert all(np.array_equal(a, b) for a, b in zip((word, node, w), w2))
    orc.bow_vocab_destroy(v)
    orc.bow_vocab_destroy(v2)


def test_shipped_orb_vocabulary(orc, tmp_path):
    """The file the reference loads (system.cc:82): header, tree consistency and a few descents.  The sample keeps every
    node the descents of its 16 descriptors compare against, so the subtree written back as a .dbow2 file descends
    exactly like the whole file did; its answers are mapped back to the whole file's node and word ids."""
    g = np.load(VOCAB_SAMPLE)
    n_nodes, node_size, k, L, scoring, weighting = struct.unpack("<IIiiii", g["header"].tobytes())
    assert (n_nodes, node_size, k, L) == (1082073, 41, 10, 6)
    assert g["info"].tolist() == [10, 6, 1082073, 971814]      # orc.bow_vocab_info of the whole file
    ids = g["ids"]
    assert np.all(np.diff(ids) > 0) and np.all(g["parent"] < ids)
    new_id = {0: 0, **{int(i): j + 1 for j, i in enumerate(ids)}}
    vocab = dict(k=k, L=L, parent=np.array([new_id[int(p)] for p in g["parent"]], np.int32), desc=g["desc"],
                 weight=g["weight"], is_leaf=g["is_leaf"])
    path = tmp_path / "orb_vocab_sample.dbow2"
    bow_data.write_dbow2(path, vocab, scoring, weighting)
    v = orc.bow_vocab_load(path)
    assert orc.bow_vocab_info(v) == dict(k=10, L=6, num_nodes=len(ids) + 1, num_words=int(g["is_leaf"].sum()))
    word, node, w = orc.bow_transform(v, g["queries"], 4)
    orc.bow_vocab_destroy(v)
    assert [(int(a), int(b), float(c)) for a, b, c in zip(word, node, w)] == \
        bow_data.transform_numpy(vocab, g["queries"], 4)
    leaf_ids = np.flatnonzero(g["is_leaf"])
    assert np.array_equal(g["word_id"][leaf_ids[word]], g["word"])
    assert np.array_equal(ids[node - 1], g["node"]) and np.array_equal(w, g["node_weight"])
    parent_of = dict(zip(ids.tolist(), g["parent"].tolist()))
    for nd in g["node"].tolist():                       # the feature-vector nodes sit at level L - levelsup = 2
        assert nd > 0 and parent_of[nd] > 0 and parent_of[parent_of[nd]] == 0


@pytest.mark.parametrize("seed", range(4))
def test_bow_tree_oracle_matches_python_restatement(orc, seed):
    s1, s2, truth = bow_data.make_bow_sides(seed, n1=300, n2=340, num_nodes=30)
    for ratio, check, use_valid2 in [(0.7, True, False), (0.75, True, True), (0.9, False, True)]:
        b = dict(s2)
        if not use_valid2:
            b.pop("valid")          # match_frame_and_keyframe: every frame keypoint is a candidate
        o = orc.bow_tree_match(s1, b, ratio, check)
        p = bow_data.bow_tree_match_python(s1, b, ratio, check)
        assert np.array_equal(o[0], p[0]) and np.array_equal(o[1], p[1]) and o[2] == p[2]
        assert o[2] > 40
        hit = o[0] >= 0
        assert (o[0][hit] == truth[hit]).mean() > 0.9
        assert np.all(o[0][s1["valid"] == 0] == -1)


def test_fold_bow_is_l1_normalised(plp):
    word = np.array([5, 2, 5, 9, 2, 7], np.int32)
    node = np.array([11, 12, 11, 13, 12, 11], np.int32)
    w = np.array([1.5, 0.5, 1.5, 0.0, 0.5, 2.0], np.float32)
    words, vals, fv = plp.capi.fold_bow(word, node, w)
    assert words.tolist() == [2, 5, 7] and abs(vals.sum() - 1.0) < 1e-15
    assert np.allclose(vals, np.array([1.0, 3.0, 2.0]) / 6.0)
    assert fv[0].tolist() == [11, 12] and fv[1].tolist() == [0, 3, 5] and fv[2].tolist() == [0, 2, 5, 1, 4]
