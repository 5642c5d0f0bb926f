"""Generates the committed golden fixtures under tests/golden/.

There is no runnable reference here (Rust toolchain absent), so the vectors come from the C
oracle (oracle/pbx_oracle.c) and are accepted into the fixture only when the independent numpy
restatement (tests/np_restatement.py) and, for top-k cases, the SQLite-level oracle running the
verbatim SQL of src/engine.rs:375-382 agree bit for bit.  Run:  python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402
from tests import np_restatement as npr  # noqa: E402
from tests import sqlite_oracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def bits(x) -> int:
    return int(np.float32(x).view(np.uint32))


def clustered_corpus(rng, n, d, ncent, noise):
    cent = rng.integers(0, 256, size=(ncent, d))
    which = rng.integers(0, ncent, size=n)
    x = cent[which] + rng.integers(-noise, noise + 1, size=(n, d))
    return np.clip(x, 0, 255).astype(np.uint8)


def make_pairs():
    rng = np.random.default_rng(20260101)
    pairs = []
    # upstream KATs (src/engine.rs:705-707) and README example bytes (README.md:54)
    fixed = [([255, 0], [255, 0]), ([0, 255], [0, 255]), ([255, 0], [0, 255]),
             ([0x00, 0xFF, 0x80, 0x8C], [0x00, 0xFF, 0x80, 0x8C]), ([0x00, 0xFF, 0x80, 0x8C], [0x8C, 0x80, 0xFF, 0x00]),
             ([127], [128]), ([128], [128]), ([127] * 8, [128] * 8), ([0] * 8, [255] * 8), ([0] * 8, [0] * 8)]
    for a, b in fixed:
        pairs.append((np.array(a, np.uint8), np.array(b, np.uint8)))
    for d in (1, 2, 3, 8, 16, 63, 64, 100, 256, 1024):
        for t in range(12):
            a = rng.integers(0, 256, d, dtype=np.uint8)
            if t % 4 == 0:
                b = np.clip(a.astype(int) + rng.integers(-2, 3, d), 0, 255).astype(np.uint8)   # near duplicate
            elif t % 4 == 1:
                b = (255 - a).astype(np.uint8)                                               # anti-correlated -> plateau
            elif t % 4 == 2:
                b = rng.integers(126, 130, d, dtype=np.uint8)                                 # tiny magnitudes
            else:
                b = rng.integers(0, 256, d, dtype=np.uint8)
            pairs.append((a, b))
    out = []
    for a, b in pairs:
        c = oracle.cosine_distance(a, b)
        p = npr.cosine_distance(a, b)
        assert bits(c) == bits(p), (a, b, c, p)
        dot, nq, nr = oracle.int_terms(a, b)
        out.append({"a": bytes(a).hex(), "b": bytes(b).hex(), "dist_bits": bits(c), "dist": float(c),
                    "dot": dot, "norm2_a": nq, "norm2_b": nr})
    with open(os.path.join(HERE, "cosine_pairs.json"), "w") as f:
        json.dump(out, f, indent=0)
    print("cosine_pairs.json:", len(out))


def make_topk():
    rng = np.random.default_rng(20260102)
    cases = {}
    # row counts keep the fixture under 1 MB: its corpora are random bytes and do not compress
    specs = [("uniform_d8", 300, 8, None), ("uniform_d64", 1200, 64, None), ("uniform_d256", 1000, 256, None),
             ("cluster_d256", 1000, 256, (40, 3)), ("cluster_d64_ties", 2000, 64, (10, 0)), ("cluster_d1024", 220, 1024, (8, 2))]
    for name, n, d, cl in specs:
        corpus = rng.integers(0, 256, size=(n, d), dtype=np.uint8) if cl is None else clustered_corpus(rng, n, d, *cl)
        ids = np.sort(rng.choice(np.arange(1, 10 * n), size=n, replace=False)).astype(np.int64)
        queries = np.stack([corpus[int(rng.integers(0, n))],                                   # right-click "find similar"
                            np.clip(corpus[int(rng.integers(0, n))].astype(int) + rng.integers(-9, 10, d), 0, 255).astype(np.uint8),
                            rng.integers(0, 256, d, dtype=np.uint8)])
        conn = sqlite_oracle.make_db(":memory:", ids, corpus)
        for qi, q in enumerate(queries):
            for k, md in ((10, 1e3), (50, 1e3), (100, 1e3), (100, 0.5), (100, 1e7)):
                o_ids, o_dist, o_dot, o_n2 = oracle.topk(corpus, ids, q, k, md)
                sql = sqlite_oracle.query(conn, bytes(q), md, k)
                assert [r[0] for r in sql] == list(o_ids), (name, qi, k, md)
                assert [bits(r[1]) for r in sql] == [bits(x) for x in o_dist], (name, qi, k, md)
                cases[f"{name}/q{qi}/k{k}/md{md:g}/ids"] = o_ids
                cases[f"{name}/q{qi}/k{k}/md{md:g}/dist_bits"] = o_dist.view(np.uint32)
                cases[f"{name}/q{qi}/k{k}/md{md:g}/dot"] = o_dot
                cases[f"{name}/q{qi}/k{k}/md{md:g}/norm2"] = o_n2
        cases[f"{name}/corpus"] = corpus
        cases[f"{name}/ids"] = ids
        cases[f"{name}/queries"] = queries
    np.savez_compressed(os.path.join(HERE, "topk_small.npz"), **cases)
    print("topk_small.npz:", len(cases), "arrays")


if __name__ == "__main__":
    make_pairs()
    make_topk()
