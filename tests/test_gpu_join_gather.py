"""Join gather edge cases: the row-slot build (slot_lens / slot_fill) and copy (slot_copy), the per-column gather
(gather_copy) and the probe key packing, each against the oracle's mergeRows output (csvplus.go:545-583).

Covers what a random join hits only by chance: every value length 0..64 at every slot size, row counts that leave a
partial warp, a warp group too long for the shared-memory stage, source values at every residue mod 8 (row-range views),
a value ending at the last byte of its buffer, and probe keys that are empty or longer than the index width, single- and
two-column, for every probe table a large index uses."""
from __future__ import annotations

import random

import pytest

from oracle import oracle as orc
from tests.helpers import assert_table_equals_oracle

pytestmark = pytest.mark.gpu

ALPHA = "abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789_-."


def _csv(header, rows):
    return (",".join(header) + "\n" + "".join(",".join(r) + "\n" for r in rows)).encode()


def _word(rng, n):
    return "".join(rng.choice(ALPHA) for _ in range(n))


def _split(rng, total, nc):
    """nc lengths summing to total, in random proportions"""
    cuts = sorted(rng.randrange(total + 1) for _ in range(nc - 1))
    return [b - a for a, b in zip([0] + cuts, cuts + [total])]


def _index_both(data, on, *, unique, drop=0):
    import csvplus_b200 as cp
    src, osrc = cp.Take(cp.FromBytes(data)), orc.reader_rows(data)
    if drop:
        src, osrc = src.Drop(drop), osrc.drop(drop)
    return (src.UniqueIndexOn(*on) if unique else src.IndexOn(*on)), osrc.index_on(*on, unique=unique)


def _check_join(pdata, idx, oidx, on, drop=0):
    import csvplus_b200 as cp
    src, osrc = cp.Take(cp.FromBytes(pdata)), orc.reader_rows(pdata)
    if drop:
        src, osrc = src.Drop(drop), osrc.drop(drop)
    tp, err = src._table()
    assert err is None
    assert_table_equals_oracle(tp.join(idx, *on), osrc.join(oidx, *on))


@pytest.mark.parametrize("S", [16, 32, 48, 64])
@pytest.mark.parametrize("nc", [1, 2, 3, 4])
@pytest.mark.parametrize("unique", [True, False], ids=["source_order", "sorted_order"])
def test_row_slots_every_length(nc, S, unique):
    """every row length 0..S split over nc output columns (so every value length 0..S occurs for column 0), the
    longest row exactly S; identity probes and probes with misses / repeats, at partial-warp row counts"""
    rng = random.Random(1000 * nc + S + unique)
    hdr = ["k"] + [f"v{c}" for c in range(nc)]
    rows = []
    for i in range(3 * (S + 1) + 5):
        tot = i % (S + 1)
        lens = [tot] + [0] * (nc - 1) if i < S + 1 else _split(rng, tot, nc)
        rows.append([f"{i:05d}"] + [_word(rng, n) for n in lens])
    rng.shuffle(rows)
    nidx = len(rows)
    idata = _csv(hdr, rows)
    for drop, nprobe in ((0, nidx + 13), (3, nidx + 45)):
        idx, oidx = _index_both(idata, ["k"], unique=unique, drop=drop)
        # identity: every probe row matches once -> the slots are built and slot_copy runs alone
        keys = [rows[rng.randrange(drop, nidx)][0] for _ in range(nprobe)]
        _check_join(_csv(["pid", "k"], [[str(j), k] for j, k in enumerate(keys)]), idx, oidx, ["k"])
        # misses: expand_pairs, slot_copy of the matches, gather_copy of the probe side
        keys = [rows[rng.randrange(drop, nidx)][0] if j % 7 else "nope%d" % j for j in range(nprobe)]
        _check_join(_csv(["pid", "k"], [[str(j), k] for j, k in enumerate(keys)]), idx, oidx, ["k"])
        # fewer than 32 rows
        _check_join(_csv(["pid", "k"], [[str(j), rows[(j * 11) % nidx][0]] for j in range(19)]), idx, oidx, ["k"])


def test_row_slots_direct_path():
    """64-byte rows in 64-byte slots, the destination of a warp group not 16-byte aligned: 32 x 64 bytes plus the
    head do not fit the stage, the group is written straight to global memory"""
    rng = random.Random(7)
    rows = [[f"{i:05d}", _word(rng, 59 if i == 0 else 64)] for i in range(300)]
    idata = _csv(["k", "v"], rows)
    keys = [rows[0][0]] + [rows[1 + (j % 299)][0] for j in range(1000)]
    for unique in (True, False):
        idx, oidx = _index_both(idata, ["k"], unique=unique)
        _check_join(_csv(["pid", "k"], [[str(j), k] for j, k in enumerate(keys)]), idx, oidx, ["k"])


@pytest.mark.parametrize("drop", range(8))
def test_gather_copy_source_residues(drop):
    """row-range views shift every source value by `drop` rows: IndexOn(...).table() (gather_copy of the sorted
    rows), a join through the per-column gather (values > 255 bytes: no row slots) including groups too long for the
    stage, and the probe-side gather of a join with misses"""
    rng = random.Random(50 + drop)
    rows = [[_word(rng, rng.randrange(0, 6)), _word(rng, rng.randrange(0, 40)), _word(rng, 300 if i % 97 == 5 else rng.randrange(0, 90))]
            for i in range(1000 + drop)]
    data = _csv(["k", "a", "b"], rows)
    idx, oidx = _index_both(data, ["k"], unique=False, drop=drop)
    assert_table_equals_oracle(idx.table(), oidx.rows())
    keys = [rows[rng.randrange(len(rows))][0] if j % 5 else "zz" for j in range(1501)]
    _check_join(_csv(["pid", "k", "pad"], [[str(j), k, _word(rng, rng.randrange(0, 120))] for j, k in enumerate(keys)]),
                idx, oidx, ["k"], drop=drop)


@pytest.mark.parametrize("total", [4096, 4095])
def test_value_ends_at_buffer_end(total):
    """the bytes of a column total a multiple of 512 (or one less), so its last value ends at the end of a 512-byte
    block of the buffer: the copies must not read past the aligned word holding that byte"""
    rng = random.Random(total)
    lens = []
    while sum(lens) < total - 64:
        lens.append(rng.randrange(1, 64))
    lens.append(total - sum(lens))
    rows = [[f"{i:04d}", _word(rng, n)] for i, n in enumerate(lens)]
    data = _csv(["k", "v"], rows)
    for unique in (True, False):
        idx, oidx = _index_both(data, ["k"], unique=unique)
        assert_table_equals_oracle(idx.table(), oidx.rows())
        keys = [rows[-1][0]] * 40 + [rows[rng.randrange(len(rows))][0] for _ in range(400)]
        _check_join(_csv(["pid", "k"], [[str(j), k] for j, k in enumerate(keys)]), idx, oidx, ["k"])


@pytest.mark.parametrize("width", [3, 8, 11, 12, 15, 16, 20, 30, "two_columns"])
def test_probe_key_packing(width):
    """large indices (probe tables in global memory): key images of up to 12 bytes (16-byte slots), up to 24 bytes
    (32-byte slots) and wider; probe keys that are empty, longer than the index width, or absent must behave as in the
    reference"""
    rng = random.Random(str(width))
    n = 24_000
    two = width == "two_columns"
    w = 6 if two else width
    keys = {("x" * w, "x" if two else ""), ("", "")}
    while len(keys) < n:
        keys.add((_word(rng, rng.randrange(1, w + 1)), _word(rng, rng.randrange(0, 4)) if two else ""))
    keys = sorted(keys)
    rng.shuffle(keys)
    on = ["k", "k2"] if two else ["k"]
    rows = [[k, k2, _word(rng, rng.randrange(0, 12))] if two else [k, _word(rng, rng.randrange(0, 12))] for k, k2 in keys]
    idata = _csv(on + ["v"], rows)
    probe = []
    for j in range(n + 1001):
        r = j % 9
        pk = ("", "") if r == 0 else ("x" * w + "y", "") if r == 1 else (keys[rng.randrange(n)][0] + "~", "q") if r == 2 \
            else keys[rng.randrange(n)]
        probe.append([str(j), pk[0], pk[1]] if two else [str(j), pk[0]])
    pdata = _csv(["pid"] + on, probe)
    for unique in (True, False):
        idx, oidx = _index_both(idata, on, unique=unique)
        _check_join(pdata, idx, oidx, on)
