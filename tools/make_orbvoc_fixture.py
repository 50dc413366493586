#!/usr/bin/env python3
"""Generates tests/golden/orbvoc_subtree.npz: the part of the reference's vocab/ORBvoc.bin (44 MB, DBoW3 binary format, k = 10,
L = 6) that the descents of 150 real ORB descriptors touch, and what Vocabulary::transform gives for them on the whole file.

A descent compares the descriptor with every child of the node it stands on and moves to the closest one.  Keeping, for each
descriptor, all children of every node on its path (in file order, parents re-indexed) gives a vocabulary in the same format on
which every descent takes the same path and ends on a record with the same weight; only node and word ids are renumbered, and
`node_id` / `word_id` map them back.  A kept node that is not on any path loses its children, so it is flagged a leaf (the loader
requires a childless node to be a word); no descent ends there, and its word maps to -1.  tests/test_bow.py runs the oracle and
its numpy restatement on the sub-tree and compares with the whole-file results stored here.

usage: python tools/make_orbvoc_fixture.py <path to the reference's vocab/ORBvoc.bin>"""
import struct
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from oracle.pyoracle import Oracle  # noqa: E402
from test_bow import numpy_transform, parse  # noqa: E402
from ygz_slam_b200 import synth  # noqa: E402

LEVELSUP = 4


def subtree(data: bytes, desc: np.ndarray):
    """Sorted original node ids (1-based) of all children of every node on the descents of `desc`."""
    rec = parse(data)[0]
    parent = rec["parent"]
    order = np.argsort(parent, kind="stable")
    starts = np.searchsorted(parent[order], np.arange(len(rec) + 2))
    bits = np.unpackbits(rec["desc"], axis=1)
    keep = set()
    for f in desc:
        fb = np.unpackbits(f)
        cur = 0
        while True:
            ch = order[starts[cur]:starts[cur + 1]] + 1
            if len(ch) == 0:
                break
            keep.update(ch.tolist())
            cur = int(ch[int(np.argmin((bits[ch - 1] != fb).sum(1)))])
    return np.array(sorted(keep))


def main(path: str) -> None:
    data = Path(path).read_bytes()
    rec, k, L, scoring, weighting = parse(data)
    ora = Oracle()
    g, _, _ = synth.stream_frame(2)
    pyr = ora.build_pyramid(g, 3)
    f = ora.detect(pyr, n_levels=3)
    desc = ora.describe(pyr, 640, 480, 3, f["px"], f["py"], f["level"])[1][:150]

    # the whole file: the oracle and the independent numpy descent must agree before anything is stored
    v = ora.vocab_load(data)
    info = ora.vocab_info(v)
    word, node, weight, bw, bv = ora.bow_transform(v, desc, LEVELSUP)
    ora.vocab_free(v)
    nw, nn, nwt, nbow = numpy_transform(data, desc, LEVELSUP)
    assert np.array_equal(word, nw) and np.array_equal(node, nn) and np.array_equal(weight, nwt)
    assert list(bw) == sorted(nbow) and np.allclose(bv, [nbow[a] for a in sorted(nbow)], rtol=1e-15, atol=0)

    keep = subtree(data, desc)
    new_of = np.zeros(len(rec) + 1, np.int64)
    new_of[keep] = np.arange(1, len(keep) + 1)
    sub = rec[keep - 1].copy()
    assert np.all((sub["parent"] == 0) | (new_of[sub["parent"]] > 0))
    sub["parent"] = new_of[sub["parent"]]
    leaf_rank = np.cumsum(rec["leaf"].astype(np.int64)) - 1          # original word id of every leaf record
    orig_word = np.where(sub["leaf"] > 0, leaf_rank[keep - 1], -1)
    childless = ~np.isin(np.arange(1, len(keep) + 1), sub["parent"])
    sub["leaf"][childless] = 1
    sub_bytes = struct.pack("<IIiiii", len(keep) + 1, 41, k, L, scoring, weighting) + sub.tobytes()
    out = dict(vocab=np.frombuffer(sub_bytes, np.uint8), desc=desc, levelsup=np.int32(LEVELSUP),
               node_id=np.r_[0, keep].astype(np.int32), word_id=orig_word[sub["leaf"] > 0].astype(np.int32),
               info=np.array([info[n] for n in ("k", "L", "scoring", "weighting", "nodes", "words")], np.int32),
               word=word, node=node, weight=weight, bow_words=bw, bow_values=bv)
    dst = ROOT / "tests" / "golden" / "orbvoc_subtree.npz"
    np.savez_compressed(dst, **out)
    print("wrote", dst, dst.stat().st_size, "bytes;", len(keep), "of", len(rec), "records")


if __name__ == "__main__":
    main(sys.argv[1])
