"""Pins oracle/mgoracle.c (plain-C restatement) against the golden vectors generated from the unmodified reference,
and against the reference library itself (or its stored results) on seeded random inputs."""
import ctypes as C
import json
import os
import random
import subprocess

import pytest

import mgtest as T

GOLD = os.path.join(T.REPO, "tests", "golden", "vectors.json")


@pytest.fixture(scope="module")
def orc():
    return T.load_oracle()


orc_sketch = T.orc_sketch


def orc_sort(orc, arr):
    n = len(arr)
    x, y = (C.c_uint64 * n)(*[a[0] for a in arr]), (C.c_uint64 * n)(*[a[1] for a in arr])
    orc.orc_radix_sort_128x(x, y, n)
    return [x[i] for i in range(n)], [y[i] for i in range(n)]


def test_sketch_golden(orc):
    gold = json.load(open(GOLD))
    assert len(gold["sketch"]) >= 18
    for c in gold["sketch"]:
        assert orc_sketch(orc, c["seq"].encode(), c["w"], c["k"], c["rid"]) == c["mz"], (c["name"], c["w"], c["k"])


def test_radix_sort_golden_tie_order(orc):
    gold = json.load(open(GOLD))
    for c in gold["sort"]:
        xs, ys = orc_sort(orc, c["in"])
        assert xs == sorted(a[0] for a in c["in"])
        assert ys == c["out_y"], "tie order differs from klib's unstable radix sort (n=%d)" % len(c["in"])


def test_against_reference_random(orc):
    rng = random.Random(7)
    for it in range(60):
        n = rng.choice([30, 200, 1000, 5000])
        alpha = rng.choice(["ACGT", "ACGTN", "AC", "ACGTacgtnN"])
        s = "".join(rng.choice(alpha) for _ in range(n)).encode()
        w, k = rng.choice([(11, 17), (10, 19), (3, 7), (20, 28)])
        assert orc_sketch(orc, s, w, k, 5) == T.ref_sketch(s, w, k, 5), (it, w, k)
    for it in range(40):
        n = rng.choice([3, 64, 65, 500, 4000])
        nk = rng.choice([2, 10, 1000, 2 ** 50])
        arr = [[rng.randrange(nk) << rng.choice([0, 8, 33]), i] for i in range(n)]
        xs, ys = orc_sort(orc, arr)
        assert list(zip(xs, ys)) == T.ref_radix_sort([tuple(a) for a in arr]), it


def test_name_hash(orc):
    # kh_hash_str (X31) known answers: h("") = 0, h("a") = 97, h("ab") = 97*31 + 98
    assert orc.orc_hash_str(b"") == 0 and orc.orc_hash_str(b"a") == 97 and orc.orc_hash_str(b"ab") == 97 * 31 + 98


def test_index_matches_oracle_sketch(orc):
    """the product's index (built from the device sketch of every segment) holds exactly the occurrence lists that the
    oracle's sketch of the segments implies (reference: index.c:115-165)"""
    lib = T.load_hostsim()
    check_index(lib, orc)


def check_index(lib, orc):
    from minigraph_b200 import options
    gfa = os.path.join(T.FIX, "MT.gfa")
    g = lib.mgb_gfa_read(gfa.encode())
    io, mo = options.opt_set("lr")
    gi = lib.mg_index(g, C.byref(io), 1, C.byref(mo))
    assert gi
    want = {}
    for sid in range(g.contents.n_seg):
        seg = g.contents.seg[sid]
        s = C.string_at(seg.seq, seg.len)
        for x, y in orc_sketch(orc, s, io.w, io.k, sid):
            want.setdefault(x >> 8, []).append(y)
    n = C.c_int(0)
    for key, ys in want.items():
        p = lib.mg_idx_get(gi, key, C.byref(n))
        assert n.value == len(ys) and [p[i] for i in range(n.value)] == sorted(ys), hex(key)
    assert not lib.mg_idx_get(gi, 12345, C.byref(n)) and n.value == 0
    lib.mg_idx_destroy(gi)
    lib.mgb_gfa_destroy(g)
