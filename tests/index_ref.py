"""Plain references of IndexOn / ResolveDuplicates for the index tests, independent of the CUDA code and of the oracle.

Columns are (offsets int64[n+1], bytes uint8[]) pairs, the shape Table.column() returns, or lists of `bytes` for
ref_order.  Order is per key column bytewise (Python's `bytes` ordering is exactly Go's strings.Compare), columns left to
right, ties in input order: the order IndexOn defines (the reference's sort.Sort is unstable, SURVEY §Q2)."""
from __future__ import annotations

import numpy as np


def ref_order(cols, keys) -> list[int]:
    """the stable sort permutation of the rows by `keys`; cols: name -> list[bytes]"""
    kc = [cols[k] for k in keys]
    return sorted(range(len(kc[0])), key=lambda r: tuple(c[r] for c in kc))


def values(off, data) -> list[bytes]:
    d = np.asarray(data, np.uint8).tobytes()
    return [d[off[i]:off[i + 1]] for i in range(len(off) - 1)]


def from_values(vals) -> tuple[np.ndarray, np.ndarray]:
    """list[bytes] -> (offsets, data)"""
    off = np.zeros(len(vals) + 1, np.int64)
    off[1:] = np.cumsum([len(v) for v in vals])
    return off, np.frombuffer(b"".join(vals), np.uint8).copy()


def key_words(off, data) -> tuple[np.ndarray, np.ndarray]:
    """values of at most 8 bytes -> (big-endian uint64 of the zero-padded value, length): comparing the pairs compares the
    values bytewise.  (numpy `S` strings would not do: they drop trailing NUL bytes, so b"a" == b"a\\x00" there.)"""
    off = np.asarray(off, np.int64)
    data = np.asarray(data, np.uint8)
    ln = off[1:] - off[:-1]
    assert int(ln.max(initial=0)) <= 8, "key_words takes values of at most 8 bytes"
    w = np.zeros(len(ln), np.uint64)
    for b in range(8):
        m = ln > b
        w[m] |= data[off[:-1][m] + b].astype(np.uint64) << np.uint64(8 * (7 - b))
    return w, ln


def ref_order_np(cols, keys) -> np.ndarray:
    """ref_order for key values of at most 8 bytes, vectorised; cols: name -> (offsets, data)"""
    parts = []
    for k in keys:
        parts += list(key_words(*cols[k]))
    n = len(parts[0])
    return np.lexsort([np.arange(n)] + parts[::-1])  # last key of lexsort = most significant


def ref_gather(off, data, perm) -> tuple[np.ndarray, np.ndarray]:
    """(offsets, data) of a column after the row permutation / selection `perm`"""
    off = np.asarray(off, np.int64)
    perm = np.asarray(perm, np.int64)
    start = off[:-1][perm]
    ln = off[1:][perm] - start
    noff = np.zeros(len(perm) + 1, np.int64)
    np.cumsum(ln, out=noff[1:])
    src = np.repeat(start - noff[:-1], ln) + np.arange(int(noff[-1]), dtype=np.int64)
    return noff, np.asarray(data, np.uint8)[src]


def ref_dedup(sorted_keys, resolve_by, bug_compatible=True):
    """indexImpl.dedup (csvplus.go:810-867) with the tie-order-independent resolver "keep the row with the smallest
    resolve_by value, the first such row on ties" (SURVEY §8d cfg 5).

    sorted_keys: arrays over the rows in sorted order; two rows have the same key iff they are equal in every array.
    resolve_by: arrays over the same rows, compared lexicographically (e.g. key_words of order_id).
    Returns (lo, hi, keep, rows): the [lo, hi) sorted positions of every run of >= 2 rows with equal keys, the position
    kept for each run, and the sorted positions the index holds afterwards.  With bug_compatible the last sorted row is
    lost when it is a singleton and at least one run exists (SURVEY §Q1, :851-864)."""
    n = len(sorted_keys[0])
    head = np.ones(n, bool)
    if n > 1:
        same = np.ones(n - 1, bool)
        for a in sorted_keys:
            same &= a[1:] == a[:-1]
        head[1:] = ~same
    starts = np.flatnonzero(head)
    ends = np.append(starts[1:], n)
    grouped = ends - starts >= 2
    lo, hi = starts[grouped], ends[grouped]
    run = np.repeat(np.arange(len(starts)), ends - starts)
    order = np.lexsort([np.arange(n)] + list(resolve_by)[::-1] + [run])  # runs stay contiguous, best row first
    keep = order[starts][grouped]
    rows = np.sort(np.concatenate([starts[~grouped], keep]))
    if bug_compatible and len(lo) and not grouped[-1]:
        rows = rows[:-1]
    return lo, hi, keep, rows
