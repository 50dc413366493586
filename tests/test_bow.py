"""DBoW3 vocabulary (SURVEY 8f rows 1-2): loader, Vocabulary::transform / Frame::ComputeBoW, Matcher::SearchByBoW.

The oracle (oracle/bow.cpp) follows the vendored DBoW3 source; here it is checked against an independent numpy descent
written from the file format and the transform's text (Vocabulary.cpp:706-832, 1180-1225), on synthetic vocabularies in the
same binary format and on the part of the reference's own vocab/ORBvoc.bin that real descriptors descend through
(tests/golden/orbvoc_subtree.npz).  The GPU tests compare the CUDA path with the oracle: word / node / match indices exact,
values 1e-14.
"""
import struct
from pathlib import Path

import numpy as np
import pytest

from oracle.pyoracle import Oracle
from ygz_slam_b200 import synth

GOLD_VOC = Path(__file__).resolve().parent / "golden" / "orbvoc_subtree.npz"
REC = np.dtype([("parent", "<i4"), ("desc", "u1", 32), ("w", "<f4"), ("leaf", "u1")])


def parse(data: bytes):
    nb, size, k, L, scoring, weighting = struct.unpack("<IIiiii", data[:24])
    assert size == 41
    rec = np.frombuffer(data[24:], dtype=REC)
    assert len(rec) == nb - 1
    return rec, k, L, scoring, weighting


def numpy_transform(data: bytes, desc: np.ndarray, levelsup: int):
    """Independent restatement: returns word, node, weight per descriptor and the BowVector (dict word -> value)."""
    rec, k, L, scoring, weighting = parse(data)
    n_rec = len(rec)
    # the reference's eof() loop appends a copy of the last record as node n_rec + 1
    parent = np.r_[rec["parent"], rec["parent"][-1]]
    vdesc = np.concatenate([rec["desc"], rec["desc"][-1:]])
    w = np.r_[rec["w"], rec["w"][-1]].astype(np.float64)
    leaf = np.r_[rec["leaf"], rec["leaf"][-1]].astype(bool)
    word_of = np.full(n_rec + 2, -1)
    word_of[1:][leaf] = np.arange(int(leaf.sum()))
    order = np.argsort(parent, kind="stable")             # children of a node in file order
    starts = np.searchsorted(parent[order], np.arange(n_rec + 3))
    bits = np.unpackbits(vdesc, axis=1)
    words, nodes, weights = [], [], []
    nid_level = L - levelsup
    for f in np.asarray(desc, np.uint8).reshape(-1, 32):
        fb = np.unpackbits(f)
        cur, level, nid = 0, 0, (0 if nid_level <= 0 else None)
        while True:
            ch = order[starts[cur]:starts[cur + 1]] + 1       # node ids of the children
            if len(ch) == 0:
                break
            level += 1
            d = (bits[ch - 1] != fb).sum(1)
            cur = int(ch[int(np.argmin(d))])                  # first minimum
            if level == nid_level:
                nid = cur
        if nid is None:
            nid = cur
        words.append(int(word_of[cur]))
        weights.append(float(w[cur - 1]))
        nodes.append(nid if w[cur - 1] > 0 else -1)
    bow = {}
    for wd, wt in zip(words, weights):
        if wt <= 0:
            continue
        if wd in bow:
            if weighting in (0, 1):
                bow[wd] += wt
        else:
            bow[wd] = wt
    must, l2 = scoring != 5, scoring == 1
    if weighting in (0, 1) and bow and not must:
        bow = {a: b / len(bow) for a, b in bow.items()}
    if must:
        vals = [bow[a] for a in sorted(bow)]
        norm = 0.0
        for v in vals:
            norm += v * v if l2 else abs(v)
        if l2:
            norm = np.sqrt(norm)
        if norm > 0:
            bow = {a: b / norm for a, b in bow.items()}
    return np.array(words), np.array(nodes), np.array(weights), bow


def random_descriptors(data: bytes, n: int, seed: int):
    """Descriptors near the vocabulary's own centres (so descents spread over the tree) plus pure noise."""
    rec = parse(data)[0]
    rng = np.random.default_rng(seed)
    base = rec["desc"][rng.integers(0, len(rec), n)].copy()
    for d in base[: n * 3 // 4]:
        for b in rng.integers(0, 256, int(rng.integers(0, 30))):
            d[b >> 3] ^= np.uint8(1 << (b & 7))
    base[n * 3 // 4:] = rng.integers(0, 256, (n - n * 3 // 4, 32), dtype=np.uint8)
    return base


@pytest.fixture(scope="module")
def ora():
    return Oracle()


@pytest.mark.parametrize("scoring,weighting", [(0, 0), (1, 0), (5, 0), (0, 1), (0, 2), (5, 3)])
def test_oracle_transform_vs_numpy(ora, scoring, weighting):
    data = synth.make_vocabulary(k=5, L=4, seed=3 + scoring, scoring=scoring, weighting=weighting)
    rec, k, L, _, _ = parse(data)
    v = ora.vocab_load(data)
    info = ora.vocab_info(v)
    assert (info["k"], info["L"], info["scoring"], info["weighting"]) == (5, 4, scoring, weighting)
    assert info["nodes"] == len(rec) + 2                                   # root + records + the eof() repeat
    assert info["words"] == int(rec["leaf"].sum()) + int(rec["leaf"][-1])
    desc = random_descriptors(data, 300, 1)
    for levelsup in (2, 4, 1):
        word, node, weight, bw, bv = ora.bow_transform(v, desc, levelsup)
        nw, nn, nwt, nbow = numpy_transform(data, desc, levelsup)
        assert np.array_equal(word, nw) and np.array_equal(node, nn) and np.array_equal(weight, nwt)
        assert list(bw) == sorted(nbow)
        assert np.allclose(bv, [nbow[a] for a in sorted(nbow)], rtol=1e-15, atol=0)
    assert (node < 0).any() and (node >= 0).any()                           # stopped words are exercised
    ora.vocab_free(v)


def test_loader_rejects_malformed(ora):
    data = synth.make_vocabulary(k=4, L=3, seed=1)
    with pytest.raises(ValueError):
        ora.vocab_load(data[:24 + 41 * 3 + 7])                               # truncated record / wrong count
    bad = bytearray(data)
    bad[24:28] = struct.pack("<i", 7)                                        # first record points at a later parent
    with pytest.raises(ValueError):
        ora.vocab_load(bytes(bad))


def test_oracle_on_reference_vocabulary(ora):
    """The reference's vocab/ORBvoc.bin, reduced to the nodes that the descents of 150 real ORB descriptors (synthetic frame 2)
    compare against (tools/make_orbvoc_fixture.py): the oracle and the numpy descent agree on the reduced tree, and mapped back
    to the whole file's node and word ids they give what the whole file gave."""
    g = np.load(GOLD_VOC)
    assert tuple(g["info"]) == (10, 6, 0, 0, 1082075, 971816)                  # the whole file: k, L, L1_NORM, TF_IDF, nodes, words
    data = g["vocab"].tobytes()
    rec = parse(data)[0]
    v = ora.vocab_load(data)
    info = ora.vocab_info(v)
    assert (info["k"], info["L"], info["scoring"], info["weighting"]) == (10, 6, 0, 0)
    assert info["nodes"] == len(rec) + 2 and info["words"] == int(rec["leaf"].sum()) + int(rec["leaf"][-1])
    # real ORB descriptors of a synthetic frame
    img, _, _ = synth.stream_frame(2)
    pyr = ora.build_pyramid(img, 3)
    f = ora.detect(pyr, n_levels=3)
    desc = ora.describe(pyr, 640, 480, 3, f["px"], f["py"], f["level"])[1][:150]
    assert np.array_equal(desc, g["desc"])
    word, node, weight, bw, bv = ora.bow_transform(v, desc, int(g["levelsup"]))
    nw, nn, nwt, nbow = numpy_transform(data, desc, int(g["levelsup"]))
    assert np.array_equal(word, nw) and np.array_equal(node, nn) and np.array_equal(weight, nwt)
    assert list(bw) == sorted(nbow) and np.allclose(bv, [nbow[a] for a in sorted(nbow)], rtol=1e-15, atol=0)
    assert np.array_equal(g["word_id"][word], g["word"]) and np.array_equal(np.where(node >= 0, g["node_id"][node], -1), g["node"])
    assert np.array_equal(weight, g["weight"]) and (g["node"] >= 0).sum() > 100
    assert np.array_equal(g["word_id"][bw], g["bow_words"]) and np.allclose(bv, g["bow_values"], rtol=1e-15, atol=0)
    assert abs(bv.sum() - 1.0) < 1e-12
    ora.vocab_free(v)


def numpy_search_by_bow(desc1, node1, angle1, desc2, node2, angle2, th_low, ratio, check):
    """Matcher.cpp:196-292 walked the reference's way: common nodes ascending, index lists ascending."""
    b1, b2 = np.unpackbits(desc1, axis=1), np.unpackbits(desc2, axis=1)
    match = np.full(len(node1), -1)
    hist = [[] for _ in range(30)]
    cnt = 0
    for nd in sorted(set(node1[node1 >= 0]) & set(node2[node2 >= 0])):
        i2 = np.flatnonzero(node2 == nd)
        for i in np.flatnonzero(node1 == nd):
            best1, best2, bi = 256, 256, -1
            for j in i2:
                d = int((b1[i] != b2[j]).sum())
                if d < best1:
                    best2, best1, bi = best1, d, j
                elif d < best2:
                    best2 = d
            if best1 < th_low and np.float32(best1) < np.float32(ratio) * np.float32(best2):
                match[i] = bi
                if check:
                    rot = np.float32(angle1[i]) - np.float32(angle2[bi])
                    if rot < 0:
                        rot = np.float32(rot + np.float32(360))
                    x = np.float32(rot * np.float32(1.0 / 30))
                    b = int(np.floor(x + 0.5)) if x >= 0 else int(np.ceil(x - 0.5))   # C round(): half away from zero
                    if b == 30:
                        b = 0
                    hist[b].append(bi)
                cnt += 1
    if check:
        sizes = [len(h) for h in hist]
        m1 = m2 = m3 = 0
        i1 = i2_ = i3 = -1
        for i, s in enumerate(sizes):
            if s > m1:
                m3, m2, m1 = m2, m1, s
                i3, i2_, i1 = i2_, i1, i
            elif s > m2:
                m3, m2 = m2, s
                i3, i2_ = i2_, i
            elif s > m3:
                m3, i3 = s, i
        if m2 < np.float32(0.1) * np.float32(m1):
            i2_ = i3 = -1
        elif m3 < np.float32(0.1) * np.float32(m1):
            i3 = -1
        cnt -= sum(s for i, s in enumerate(sizes) if i not in (i1, i2_, i3))
    return match, cnt


def bow_pair(seed, n1=260, n2=300, n_nodes=12):
    rng = np.random.default_rng(seed)
    if n2 == 0:   # a key-frame 2 without features: nothing can match
        return (rng.integers(0, 256, (n1, 32), dtype=np.uint8), rng.integers(0, n_nodes, n1).astype(np.int32),
                rng.uniform(0, 360, n1).astype(np.float32), np.zeros((0, 32), np.uint8), np.zeros(0, np.int32), np.zeros(0, np.float32))
    desc2 = rng.integers(0, 256, (n2, 32), dtype=np.uint8)
    src = rng.integers(0, n2, n1)
    desc1 = desc2[src].copy()
    for d in desc1:
        for b in rng.integers(0, 256, int(rng.integers(0, 70))):
            d[b >> 3] ^= np.uint8(1 << (b & 7))
    node2 = rng.integers(0, n_nodes, n2).astype(np.int32)
    node1 = node2[src].copy()
    node1[rng.random(n1) < 0.1] = -1
    node2[rng.random(n2) < 0.05] = -1
    node1[rng.random(n1) < 0.1] = n_nodes + 3                       # a node key-frame 2 does not have
    angle2 = rng.uniform(0, 360, n2).astype(np.float32)
    angle1 = ((angle2[src] + np.where(rng.random(n1) < 0.7, 12.0, rng.uniform(0, 360, n1))) % 360).astype(np.float32)
    return desc1, node1, angle1, desc2, node2, angle2


@pytest.mark.parametrize("check", [False, True])
def test_oracle_search_by_bow_vs_numpy(ora, check):
    d1, n1, a1, d2, n2, a2 = bow_pair(5)
    m, cnt = ora.search_by_bow(d1, n1, a1, d2, n2, a2, th_low=50, knn_ratio=0.9, check_orientation=check)
    nm, ncnt = numpy_search_by_bow(d1, n1, a1, d2, n2, a2, 50, 0.9, check)
    assert np.array_equal(m, nm) and cnt == ncnt
    assert (m >= 0).sum() > 50
    if check:
        assert cnt < (m >= 0).sum()


# ---- CUDA path -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("scoring,weighting", [(0, 0), (1, 0), (5, 0), (0, 1), (0, 2), (5, 3)])
def test_gpu_transform_matches_oracle(ora, scoring, weighting):
    from ygz_slam_b200 import Context
    data = synth.make_vocabulary(k=10, L=4, seed=11 + scoring, scoring=scoring, weighting=weighting)
    ov = ora.vocab_load(data)
    ctx = Context(0)
    voc = ctx.vocabulary(data)
    assert voc.info() == ora.vocab_info(ov)
    sizes = [700, 0, 1, 1300, 33]
    offsets = np.r_[0, np.cumsum(sizes)].astype(np.int32)
    desc = random_descriptors(data, int(offsets[-1]), 4)
    for levelsup in (2, 4):
        word, node, weight, bows = voc.transform(offsets, desc, levelsup)
        for f in range(len(sizes)):
            a, b = offsets[f], offsets[f + 1]
            ow, on, owt, obw, obv = ora.bow_transform(ov, desc[a:b], levelsup)
            assert np.array_equal(word[a:b], ow) and np.array_equal(node[a:b], on) and np.array_equal(weight[a:b], owt)
            assert np.array_equal(bows[f][0], obw)
            assert np.allclose(bows[f][1], obv, rtol=1e-14, atol=0)
    voc.close()
    ctx.close()
    ora.vocab_free(ov)


@pytest.mark.gpu
def test_gpu_vocab_rejects_malformed():
    from ygz_slam_b200 import Context, YgzbError
    data = synth.make_vocabulary(k=4, L=3, seed=1)
    ctx = Context(0)
    with pytest.raises(YgzbError):
        ctx.vocabulary(data[:24 + 41 * 3 + 7])
    bad = bytearray(data)
    bad[24:28] = struct.pack("<i", 7)
    with pytest.raises(YgzbError):
        ctx.vocabulary(bytes(bad))
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("check", [False, True])
def test_gpu_search_by_bow_matches_oracle(ora, check):
    from ygz_slam_b200 import Context
    pairs = [bow_pair(s, n1, n2) for s, n1, n2 in ((1, 260, 300), (2, 1, 40), (3, 500, 129), (4, 90, 0))]
    off1 = np.r_[0, np.cumsum([len(p[1]) for p in pairs])].astype(np.int32)
    off2 = np.r_[0, np.cumsum([len(p[4]) for p in pairs])].astype(np.int32)
    cat = [np.concatenate([p[i] for p in pairs]) for i in range(6)]
    ctx = Context(0)
    m, cnt = ctx.search_by_bow(off1, off2, cat[0], cat[1], cat[2], cat[3], cat[4], cat[5], th_low=50, knn_ratio=0.9, check_orientation=check)
    for q, p in enumerate(pairs):
        om, ocnt = ora.search_by_bow(*p, th_low=50, knn_ratio=0.9, check_orientation=check)
        assert np.array_equal(m[off1[q]:off1[q + 1]], om)
        assert cnt[q] == ocnt
    ctx.close()


@pytest.mark.gpu
def test_gpu_transform_feeds_search_for_triangulation(ora):
    """ComputeBoW's node ids are what SearchForTriangulation / SearchByBoW consume (Frame::_feature_vec)."""
    from ygz_slam_b200 import Context
    data = synth.make_vocabulary(k=8, L=5, seed=2)
    ctx = Context(0)
    voc = ctx.vocabulary(data)
    d1 = random_descriptors(data, 400, 8)
    d2 = d1[np.random.default_rng(1).permutation(400)]
    _, node, _, _ = voc.transform([0, 400, 800], np.concatenate([d1, d2]), 4)
    m, cnt = ctx.search_by_bow([0, 400], [0, 400], d1, node[:400], None, d2, node[400:], None, th_low=50, knn_ratio=0.9)
    ok = m >= 0
    assert ok.sum() == cnt[0] and ok.sum() > 200
    assert np.array_equal(d1[ok], d2[m[ok]])                                  # identical descriptors find each other
    voc.close()
    ctx.close()


@pytest.mark.gpu
def test_gpu_transform_properties_on_a_large_vocabulary():
    """Size-independent properties on a ~100k-node vocabulary and a full frame load (no oracle in the loop): the reported node is
    the word's ancestor at level L - levelsup, BowVectors are sorted, unique and L1-normalised, stopped words appear nowhere,
    and the transform is a function of the descriptor alone (same descriptor -> same word in every frame)."""
    from ygz_slam_b200 import Context
    data = synth.make_vocabulary(k=10, L=6, seed=5, early_leaf=0.02)
    rec = parse(data)[0]
    n_rec = len(rec)
    parent = np.r_[0, rec["parent"], rec["parent"][-1]]                       # node id -> parent (root = 0; the eof() repeat last)
    leaf = np.r_[False, rec["leaf"].astype(bool), bool(rec["leaf"][-1])]
    word_node = np.flatnonzero(leaf)                                             # word id -> node id
    depth = np.zeros(n_rec + 2, np.int32)
    for i in range(1, n_rec + 2):
        depth[i] = depth[parent[i]] + 1
    ctx = Context(0)
    voc = ctx.vocabulary(data)
    sizes = [3072, 2500, 3072]
    offsets = np.r_[0, np.cumsum(sizes)].astype(np.int32)
    desc = random_descriptors(data, int(offsets[-1]), 9)
    desc[offsets[1]:offsets[1] + 500] = desc[:500]                             # the same descriptors in another frame
    word, node, weight, bows = voc.transform(offsets, desc, 4)
    assert np.array_equal(word[offsets[1]:offsets[1] + 500], word[:500]) and np.array_equal(node[offsets[1]:offsets[1] + 500], node[:500])
    stopped = weight <= 0
    assert np.array_equal(node < 0, stopped) and stopped.any() and (~stopped).any()
    lvl = 6 - 4
    for i in np.flatnonzero(~stopped)[::7]:
        a = int(word_node[word[i]])
        while depth[a] > lvl:
            a = int(parent[a])
        assert a == node[i], i                                                  # ancestor at level 2 (or the leaf itself if shallower)
    for f, (bw, bv) in enumerate(bows):
        seg = slice(offsets[f], offsets[f + 1])
        assert np.all(np.diff(bw) > 0) and abs(bv.sum() - 1.0) < 1e-12 and np.all(bv > 0)
        assert set(bw) == set(word[seg][~stopped[seg]])
    voc.close()
    ctx.close()
