"""Pins the plain index references of tests/index_ref.py (CPU only): the vectorised sort equals the stable Python sort
on adversarial short keys, and the dedup reference equals the oracle's ResolveDuplicates in both §Q1 tail shapes."""
import random

import numpy as np
import pytest

from oracle import oracle as orc
from tests.index_ref import from_values, key_words, ref_dedup, ref_gather, ref_order, ref_order_np, values

EDGE = [b"", b"\x00", b"\x00\x00", b"\x00a", b"a", b"a\x00", b"a\x00\x00", b"a\x01", b"ab", b"a\xff", b"\x7f", b"\x80",
        b"\xff", b"\xff\xff", b"\xff" * 8, b"\x00" * 8, b"abcdefgh", b"abcdefg", b"abcdefg\x00", b"abcdefg\xff"]


def _random_short(rng, n):
    alphabet = b"\x00\x01a\x7f\x80\xff"
    out = []
    for _ in range(n):
        if rng.random() < 0.3:
            v = rng.choice(EDGE)
        else:
            v = bytes(rng.choice(alphabet) for _ in range(rng.randrange(0, 9)))
            if rng.random() < 0.3:
                v = (v + b"\x00" * rng.randrange(1, 4))[:8]  # NUL tails
        out.append(v)
    return out


def test_ref_order_edges_pinned():
    cols = {"k": list(EDGE)}
    got = [EDGE[i] for i in ref_order(cols, ["k"])]
    assert got == [b"", b"\x00", b"\x00\x00", b"\x00" * 8, b"\x00a", b"a", b"a\x00", b"a\x00\x00", b"a\x01", b"ab",
                   b"abcdefg", b"abcdefg\x00", b"abcdefgh", b"abcdefg\xff", b"a\xff", b"\x7f", b"\x80", b"\xff",
                   b"\xff\xff", b"\xff" * 8]
    # composite keys never compare as their concatenation; ties keep input order
    cols = {"p": [b"ab", b"a", b"a", b"", b"a", b"a"], "q": [b"c", b"bc", b"", b"abc", b"b", b""]}
    assert ref_order(cols, ["p", "q"]) == [3, 2, 5, 4, 1, 0]
    assert ref_order(cols, ["q", "p"]) == [2, 5, 3, 4, 1, 0]


@pytest.mark.parametrize("seed", range(4))
def test_ref_order_np_equals_ref_order(seed):
    rng = random.Random(seed)
    n = 4000
    a, b = _random_short(rng, n), _random_short(rng, n)
    # pairs that concatenate to the same bytes
    for i in range(0, n, 97):
        a[i], b[i] = b"ab", b"c"
        a[i + 1], b[i + 1] = b"a", b"bc"
    lists = {"a": a, "b": b}
    arrs = {k: from_values(v) for k, v in lists.items()}
    for keys in (["a"], ["b"], ["a", "b"], ["b", "a"]):
        want = ref_order(lists, keys)
        got = ref_order_np(arrs, keys)
        assert got.tolist() == want, keys
    w, ln = key_words(*arrs["a"])
    assert (w[a.index(b"a")], ln[a.index(b"a")]) != (w[a.index(b"a\x00")], ln[a.index(b"a\x00")])


def test_ref_gather():
    rng = random.Random(7)
    vals = [bytes(rng.randrange(256) for _ in range(rng.randrange(0, 20))) for _ in range(500)]
    off, data = from_values(vals)
    perm = [rng.randrange(500) for _ in range(700)]  # a selection may repeat or leave out rows
    go, gd = ref_gather(off, data, perm)
    assert values(go, gd) == [vals[p] for p in perm]
    go, gd = ref_gather(off, data, [])
    assert go.tolist() == [0] and gd.size == 0


def _rows(seed, n, tail):
    """orders-like rows with ~half the keys in duplicate groups and repeated order ids (the resolver's tie rule matters:
    qty tells tied rows apart); tail: the greatest key is a singleton ("single") or a group ("group")"""
    rng = random.Random(seed)
    side = int((1.44 * n) ** 0.5)
    rows = [{"cust_id": str(rng.randrange(side)), "prod_id": str(rng.randrange(side)), "order_id": str(rng.randrange(n // 2)),
             "qty": str(i)} for i in range(n)]
    for k in range(1 if tail == "single" else 3):
        rows.insert(rng.randrange(len(rows) + 1), {"cust_id": "~", "prod_id": "~", "order_id": str(k), "qty": "t%d" % k})
    return rows


@pytest.mark.parametrize("tail", ["single", "group"])
def test_ref_dedup_vs_oracle(tail):
    rows = _rows(11, 3000, tail)
    cols = {c: from_values([r[c].encode() for r in rows]) for c in ("cust_id", "prod_id", "order_id", "qty")}
    keys = ["cust_id", "prod_id"]
    perm = ref_order_np(cols, keys)
    sorted_cols = {c: ref_gather(*cols[c], perm) for c in cols}
    oi = orc.take_rows(rows).index_on(*keys)
    o = oi.rows()
    for c in cols:  # the reference sort is the oracle's stable sort
        assert np.array_equal(o.column(c)[0], sorted_cols[c][0]) and np.array_equal(o.column(c)[1], sorted_cols[c][1]), c
    sk = [a for k in keys for a in key_words(*sorted_cols[k])]
    lo, hi, keep, kept = ref_dedup(sk, key_words(*sorted_cols["order_id"]))
    assert 0.3 * len(rows) < int((hi - lo).sum()) < 0.7 * len(rows)
    assert bool(hi[-1] == len(rows)) == (tail == "group")
    oi.dedup("min", "order_id")
    o = oi.rows()
    assert len(o) == len(kept) == len(rows) - int((hi - lo).sum()) + len(lo) - (tail == "single")
    for c in cols:
        go, gd = ref_gather(*sorted_cols[c], kept)
        assert np.array_equal(o.column(c)[0], go) and np.array_equal(o.column(c)[1], gd), c
    # without the §Q1 loss only the trailing singleton comes back
    _, _, _, kept2 = ref_dedup(sk, key_words(*sorted_cols["order_id"]), bug_compatible=False)
    want = np.append(kept, len(rows) - 1) if tail == "single" else kept
    assert kept2.tolist() == want.tolist()


def test_ref_dedup_small_cases():
    def run(keys, by=None, bug=True):
        k = np.frombuffer(keys.encode(), np.uint8)
        by = np.zeros(len(keys), np.int64) if by is None else np.asarray(by)
        lo, hi, keep, rows = ref_dedup([k], [by], bug)
        return lo.tolist(), hi.tolist(), keep.tolist(), rows.tolist()
    assert run("abc") == ([], [], [], [0, 1, 2])  # no group: nothing is lost
    assert run("aab") == ([0], [2], [0], [0])
    assert run("aab", bug=False) == ([0], [2], [0], [0, 2])
    assert run("abb") == ([1], [3], [1], [0, 1])
    assert run("abbcdde", by=[0, 5, 4, 0, 3, 3, 0]) == ([1, 4], [3, 6], [2, 4], [0, 2, 3, 4])
