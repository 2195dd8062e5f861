"""Exact parity of IndexOn / UniqueIndexOn / Find / SubIndex / ResolveDuplicates at the sizes where every part of the
index build runs, against the plain references of tests/index_ref.py (GPU only).

The radix sort gives each block ceil(tiles / min(tiles, 4 * SMs)) tiles of 2048 rows, so a block walks more than one
tile, and carries its digit bases from one tile to the next, only above T = 4 * SMs * 2048 rows (1,212,416 on a 148-SM
B200).  The tables here are built around T, taken from the device.  Every table carries a row-number column `i` (eight
digits), so the `i` column of a sorted table is the permutation the sort chose: it is compared exactly with the stable
reference order, and every other column with the reference gather."""
import bisect
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as orc
from tests.helpers import gpu_ctx
from tests.index_ref import from_values, key_words, ref_dedup, ref_gather, ref_order, ref_order_np, values

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0xC5B200
ALPHA = b"\x00\x01a\x7f\x80\xff"
RS_TILE = 2048  # rows of one radix tile (sort.cu RS_THREADS * RS_ITEMS)


def _multi_tile_rows():
    """T: the smallest row count above which a radix block sorts two or more tiles"""
    import torch
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count * RS_TILE


# ------------------------------------------------------------------ inputs
def _ids(n, base=0):
    """(offsets, data) of the eight-digit row numbers base .. base + n - 1"""
    v = np.arange(base, base + n, dtype=np.int64)
    digits = (v[:, None] // 10 ** np.arange(7, -1, -1, dtype=np.int64)) % 10 + 48
    return np.arange(n + 1, dtype=np.int64) * 8, digits.astype(np.uint8).ravel()


def _decode_ids(off, data):
    assert np.all(np.diff(off) == 8)
    return (np.asarray(data, np.int64).reshape(-1, 8) - 48) @ 10 ** np.arange(7, -1, -1, dtype=np.int64)


def _rand_keys(rng, n, lens, alphabet=ALPHA):
    """(offsets, data) of n values with the given lengths, bytes drawn from `alphabet`"""
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    return off, np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), int(off[-1]))]


def _csv(cols):
    """header + one record per row, the values of `cols` (name -> (offsets, data)) joined by ','; the values hold no
    ',', '"', CR or LF, so every field is written as it is"""
    names = list(cols)
    n = len(cols[names[0]][0]) - 1
    lens = [np.diff(cols[c][0]) for c in names]
    hdr = np.frombuffer((",".join(names) + "\n").encode(), np.uint8)
    start = np.zeros(n + 1, np.int64)
    np.cumsum(sum(lens) + len(names), out=start[1:])
    buf = np.empty(len(hdr) + int(start[-1]), np.uint8)
    buf[:len(hdr)] = hdr
    pos = start[:-1] + len(hdr)
    for k, c in enumerate(names):
        off, data = cols[c]
        buf[np.repeat(pos - off[:-1], lens[k]) + np.arange(int(off[-1]), dtype=np.int64)] = data
        pos = pos + lens[k]
        buf[pos] = ord("\n") if k == len(names) - 1 else ord(",")
        pos = pos + 1
    return buf


def _parse(cols):
    import csvplus_b200 as cp
    t, err = cp.parse_csv(gpu_ctx(), _csv(cols))
    assert err is None and len(t) == len(next(iter(cols.values()))[0]) - 1
    return t


# ------------------------------------------------------------------ checks
def _same(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    if not np.array_equal(got, want):
        bad = np.flatnonzero(got[:min(len(got), len(want))] != want[:min(len(got), len(want))])
        raise AssertionError(f"{what}: lengths {len(got)} / {len(want)}, first difference at {bad[:1].tolist()}")


def _check_sorted(table, cols, perm):
    """the sorted table holds the rows perm[0], perm[1], ... of `cols`: its i column (if any), then every column exactly"""
    if "i" in cols:
        _same(_decode_ids(*table.column("i")), _decode_ids(*ref_gather(*cols["i"], perm)), "row order (i column)")
    for c, (off, data) in cols.items():
        go, gd = table.column(c)
        wo, wd = ref_gather(off, data, perm)
        _same(go, wo, f"offsets of {c}")
        _same(gd, wd, f"bytes of {c}")


def _rows_of(ds):
    t, err = ds._table()
    assert err is None
    return _decode_ids(*t.column("i")) if t is not None and len(t) else np.empty(0, np.int64)


def _check_find(ix, sorted_keys, sorted_ids, probes):
    """Find(*probe) returns exactly the reference's [lower, upper) range of the probe among the sorted keys"""
    prefixes = {}
    for probe in probes:
        m = len(probe)
        if m not in prefixes:
            prefixes[m] = [k[:m] for k in sorted_keys]
        lo, hi = bisect.bisect_left(prefixes[m], probe), bisect.bisect_right(prefixes[m], probe)
        _same(_rows_of(ix.Find(*probe)), sorted_ids[lo:hi], f"Find{probe!r:.80}")


def _stats_of(build):
    ctx = gpu_ctx()
    ctx.stats(enable=True, reset=True)
    try:
        out = build()
        st = ctx.stats()
    finally:
        ctx.stats(enable=False, reset=True)
    return out, st


# ------------------------------------------------------------------ multi-tile radix sort
def test_multi_tile_short_keys():
    """(a) T + 1 rows: one tile more than one per block, so half the blocks get two tiles and the others none; keys
    of 0-6 bytes over NUL, 0x01, 'a', 0x7f, 0x80, 0xff, with long runs of equal keys"""
    n = _multi_tile_rows() + 1
    rng = np.random.default_rng(1)
    cols = {"k": _rand_keys(rng, n, rng.integers(0, 7, n)), "i": _ids(n)}
    ix = _parse(cols).index_on("k")
    kv = values(*cols["k"])
    perm = np.asarray(ref_order({"k": kv}, ["k"]))
    _check_sorted(ix.table(), cols, perm)
    sk = [(kv[p],) for p in perm]
    assert sk[0] == (b"",)
    _check_find(ix, sk, perm, [sk[0], sk[-1], sk[n // 2], (b"b",), (b"a\x02",), (b"\xff" * 7,), (sk[-1][0] + b"\x00",),
                               (b"a" * 7,)])


def test_multi_tile_three_keys_long_runs():
    """(b) ~3 M rows and three distinct keys: every run of equal keys spans many blocks, so the order inside a run is
    the input order only if the scatter is stable across tiles and blocks"""
    n = max(3_000_000, 2 * _multi_tile_rows() + 3)
    keys = [b"m", b"m\x00", b"\x80m"]
    rng = np.random.default_rng(2)
    pick = rng.integers(0, 3, n)
    cols = {"k": ref_gather(*from_values(keys), pick), "i": _ids(n)}
    ix = _parse(cols).index_on("k")
    perm = ref_order_np(cols, ["k"])
    _same(perm, np.argsort(pick, kind="stable"), "reference order")
    _check_sorted(ix.table(), cols, perm)
    sk = [(keys[p],) for p in pick[perm]]
    _check_find(ix, sk, perm, [(b"m",), (b"m\x00",), (b"\x80m",), (b"l",), (b"\x81",), (b"m\x01",), (b"m\x00\x00",), (b"",)])


def _composite_cols(n, rng):
    k1 = b"\x01a\x80\xff\x00z\x7f8"  # one constant 8-byte value: image word 0 is the same on every row
    ln = rng.integers(0, 10, n)
    ln[0] = 9
    off, data = _rand_keys(rng, n, ln, b"\x00\x01a\xff")
    cut = np.repeat(rng.integers(0, 10, n), ln)  # NUL tails: bytes past a random cut are zero
    data = np.where(np.arange(len(data)) - np.repeat(off[:-1], ln) >= cut, 0, data).astype(np.uint8)
    return k1, {"k1": ref_gather(*from_values([k1]), np.zeros(n, np.int64)), "k2": (off, data), "i": _ids(n)}


def test_multi_tile_composite_constant_word():
    """(c) (k1, k2): k1 one constant 8-byte value, k2 0-9 bytes with NUL tails.  The image is 19 bytes = 3 words and
    word 0 (k1's bytes) is constant, so it is skipped: sort_gather_word runs once per remaining word"""
    n = _multi_tile_rows() + 1
    k1, cols = _composite_cols(n, np.random.default_rng(3))
    t = _parse(cols)
    ix, st = _stats_of(lambda: t.index_on("k1", "k2"))
    assert st["sort_gather_word"]["launches"] == 3 - 1, st.get("sort_gather_word")
    k2 = values(*cols["k2"])
    perm = np.asarray(ref_order({"k1": [k1] * n, "k2": k2}, ["k1", "k2"]))
    _check_sorted(ix.table(), cols, perm)
    sk = [(k1, k2[p]) for p in perm]
    _check_find(ix, sk, perm, [sk[0], sk[-1], sk[n // 3], (k1,), (k1, b"a\x00"), (k1, b"b"), (k1, b"\xff" * 10),
                               (k1 + b"\x00",), (k1[:3],), (b"\x00",), (b"\x02",), (k1, b"")])
    # SubIndex on the constant prefix covers every row (> T): its rows and its Find are the same ranges
    import csvplus_b200 as cp
    sub = ix.SubIndex(k1)
    _same(_rows_of(cp.Take(sub)), perm, "SubIndex rows")
    sk2 = [(k2[p],) for p in perm]
    _check_find(sub, sk2, perm, [sk2[0], sk2[-1], sk2[n // 2], (b"a",), (b"\xff" * 10,), (b"b",)])


@pytest.mark.parametrize("width", [254, 255, 256])
def test_key_width_length_field(width):
    """(d) the length field of the image is one byte below width 255 and two from 255: values of 0..width bytes that
    share long prefixes, differing in their last byte and in NUL tails"""
    rng = random.Random(width)
    bases = [bytes(rng.choice(b"\x00a\xff") for _ in range(width)) for _ in range(3)]
    vals = []
    for r in range(50_000):
        L = width if r == 0 else rng.choice([0, 1, width // 2, width - 2, width - 1, width, width, rng.randrange(width + 1)])
        v = rng.choice(bases)[:L]
        if v and rng.random() < 0.5:
            v = v[:-1] + bytes([rng.choice(b"\x00\x01a\xff")])
        vals.append(v)
    cols = {"k": from_values(vals), "i": _ids(len(vals))}
    ix = _parse(cols).index_on("k")
    perm = np.asarray(ref_order({"k": vals}, ["k"]))
    _check_sorted(ix.table(), cols, perm)
    sk = [(vals[p],) for p in perm]
    _check_find(ix, sk, perm, [sk[0], sk[-1], sk[len(sk) // 2], (bases[0],), (bases[1][:-1],), (bases[2] + b"\x00",)])


def test_all_constant_key():
    """(e) one key value on every row: no radix pass runs and the order is the input order"""
    n = 200_000
    cols = {"k": ref_gather(*from_values([b"same\x00"]), np.zeros(n, np.int64)), "i": _ids(n)}
    t = _parse(cols)
    ix, st = _stats_of(lambda: t.index_on("k"))
    assert "radix_pass" not in st and "sort_gather_word" not in st, st
    _check_sorted(ix.table(), cols, np.arange(n))
    _same(_rows_of(ix.Find(b"same\x00")), np.arange(n), "Find")
    assert len(_rows_of(ix.Find(b"same"))) == 0


def test_multi_tile_row_range_view():
    """(f) the index of a row-range view (Drop(k)): the rows start inside the source's buffers"""
    import csvplus_b200 as cp
    drop = 777
    n = _multi_tile_rows() + 1 + drop
    rng = np.random.default_rng(6)
    cols = {"k": _rand_keys(rng, n, rng.integers(0, 7, n)), "i": _ids(n)}
    t = _parse(cols)
    ix = cp.TakeTable(t).Drop(drop).IndexOn("k")
    kv = values(*cols["k"])[drop:]
    perm = drop + np.asarray(ref_order({"k": kv}, ["k"]))
    _check_sorted(ix.table(), cols, perm)


# ------------------------------------------------------------------ the unique check, on every probe table
# (key column width, rows): pbytes = ka width + 1 + kb width 2 + 1
UNIQUE_TABLES = {
    "slot16": (6, 100_000),    # pbytes 10 <= 12: the 128-bit CAS insert sees the duplicate
    "slot32": (18, 100_000),   # pbytes 22 <= 24: 32-byte slots, self-probe
    "global": (40, 100_000),   # pbytes 44: ordinal slots + heads + image in global memory, self-probe
    "shared": (6, 10_000),     # (nslots + n + 1) * 4 <= 200 KB: the table staged in shared memory, self-probe
}


def _unique_rows(width, n, case, rng):
    """n distinct keys (ka, kb) with ka of width-1 digits, plus near-duplicates that are distinct keys: ka vs ka + NUL,
    and (x + "7", "c") vs (x, "7c"), whose concatenations are equal; then the planted duplicates of `case`"""
    ids = list(range(n))
    rng.shuffle(ids)
    rows = [(b"%0*d" % (width - 1, u), b"c") for u in ids]
    x, y = rows[10][0], rows[20][0]
    for extra in [(x + b"\x00", b"c"), (y + b"7", b"c"), (y, b"7c")]:
        rows.insert(rng.randrange(len(rows) + 1), extra)
    if case == "adjacent":
        p = rng.randrange(len(rows))
        rows.insert(p + 1, rows[p])
    elif case == "ends":
        rows.append(rows[0])
    elif case == "thousand":
        r = rows[rng.randrange(len(rows))]
        for _ in range(999):
            rows.insert(rng.randrange(len(rows) + 1), r)
    elif case == "several":
        for r in rng.sample(rows, 6):
            rows.insert(rng.randrange(len(rows) + 1), r)
    return rows


@pytest.mark.parametrize("case", ["none", "adjacent", "ends", "thousand", "several"])
@pytest.mark.parametrize("table", list(UNIQUE_TABLES))
def test_unique_check_every_probe_table(table, case):
    """UniqueIndexOn's duplicate check on each of its four probe tables, in a fresh index per case; a duplicate is
    reported with the oracle's message (the key that comes first in sort order), near-duplicates are not"""
    import csvplus_b200 as cp
    width, n = UNIQUE_TABLES[table]
    rng = random.Random(f"{table}/{case}")
    rows = _unique_rows(width, n, case, rng)
    ka, kb = [r[0] for r in rows], [r[1] for r in rows]
    cols = {"ka": from_values(ka), "kb": from_values(kb), "i": _ids(len(rows))}
    data = _csv(cols)
    t = _parse(cols)
    if case != "none":
        with pytest.raises(cp.CsvPlusError) as e:
            t.index_on("ka", "kb", unique=True)
        with pytest.raises(orc.OracleError) as oe:
            orc.reader_rows(data).unique_index_on("ka", "kb")
        assert str(e.value) == str(oe.value)
        return
    ix, st = _stats_of(lambda: t.index_on("ka", "kb", unique=True))
    assert ("join_probe" in st) == (table != "slot16"), sorted(st)  # the self-probe runs unless the CAS insert checked
    # a full-key join first (probes the table built over the unsorted rows), then Find and iteration (sort)
    where = {r: i for i, r in enumerate(rows)}
    x = rows[0][0]
    probe = [rows[rng.randrange(len(rows))] for _ in range(3000)] + [(b"x", b"c"), (x, b""), (x + b"\x00\x00", b"c")]
    rng.shuffle(probe)
    pcols = {"pa": from_values([p[0] for p in probe]), "pb": from_values([p[1] for p in probe]), "j": _ids(len(probe))}
    j = _parse(pcols).join(ix, "pa", "pb")
    hit = [k for k, p in enumerate(probe) if p in where]
    _same(_decode_ids(*j.column("j")), hit, "join: probe rows")
    _same(_decode_ids(*j.column("i")), [where[probe[k]] for k in hit], "join: index rows")
    perm = np.asarray(ref_order({"ka": ka, "kb": kb}, ["ka", "kb"]))
    sk = [rows[p] for p in perm]
    y = rows[[r[1] for r in rows].index(b"7c")][0]
    _check_find(ix, sk, perm, [sk[0], sk[-1], sk[len(sk) // 2], (y,), (y + b"7",), (y, b"7c"), (y + b"7", b"c"),
                               (rows[5][0],), (rows[5][0] + b"\x00",), (b"x",)])
    _check_sorted(ix.table(), cols, perm)


# ------------------------------------------------------------------ configs[4] at its full size
def _check_index_and_resolve(tab, keys, names, bug_compatible_too):
    import bench
    cols = {c: tab.column(c) for c in names}
    perm = ref_order_np(cols, keys)
    ix = tab.index_on(*keys)
    _check_sorted(ix.table(), cols, perm)
    scols = {c: ref_gather(*cols[c], perm) for c in names}
    sk = [a for k in keys for a in key_words(*scols[k])]
    by = key_words(*scols["order_id"])
    lo, hi, keep, kept = ref_dedup(sk, by)
    glo, ghi = ix.dup_groups()
    _same(glo, lo, "dup_groups lo")
    _same(ghi, hi, "dup_groups hi")
    gkeep = bench.min_id_resolver(ix.table(), glo, ghi)
    _same(gkeep, keep, "min_id_resolver")
    ix.dedup_apply(gkeep)
    _check_sorted(ix.table(), scols, kept)
    if bug_compatible_too:
        _, _, _, kept2 = ref_dedup(sk, by, bug_compatible=False)
        assert len(kept2) == len(kept) + 1
        ix2 = tab.index_on(*keys)
        l2, h2 = ix2.dup_groups()
        ix2.dedup_apply(bench.min_id_resolver(ix2.table(), l2, h2), bug_compatible=False)
        _check_sorted(ix2.table(), scols, kept2)
    return int((hi - lo).sum()), len(lo)


def test_configs4_full_size_vs_reference():
    """BASELINE configs[4] at its own size (10 M rows; CPB_INDEX_FULL_ROWS shrinks it): the bench's input,
    IndexOn(cust_id, prod_id) against the stable reference order, dup_groups and ResolveDuplicates(min order_id)
    through bench.min_id_resolver against ref_dedup, in both §Q1 tail shapes, and once with bug_compatible=False"""
    import bench
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    n = int(os.environ.get("CPB_INDEX_FULL_ROWS", "10000000"))
    side = bench.index_sides(n)
    t, err = cp.parse_csv(ctx, ctx.gen_csv("orders", (0, n), seed=SEED, n_cust=side, n_prod=side), spec=bench.INDEX_COLS)
    assert err is None and len(t) == n
    names, keys = [c for c, _ in bench.INDEX_COLS], ("cust_id", "prod_id")
    shapes = set()
    tab = t
    for _ in range(40):
        ix = tab.index_on(*keys)
        lo, hi = ix.dup_groups()
        in_group = bool(len(hi) and hi[-1] == len(ix))
        del ix
        if in_group not in shapes:
            shapes.add(in_group)
            grouped, groups = _check_index_and_resolve(tab, keys, names, bug_compatible_too=not in_group)
            assert 0.35 * len(tab) < grouped < 0.65 * len(tab) and groups > 0
            if len(shapes) == 2:
                break
        tab = bench.without_greatest_key(tab, keys)
    assert shapes == {True, False}


class _Columns:
    """columns (name -> (offsets, data)) behind the Table.column(name, lo, hi) interface bench.dump_table reads"""

    def __init__(self, cols):
        self.cols = cols
        self.columns = list(cols)

    def __len__(self):
        return len(next(iter(self.cols.values()))[0]) - 1

    def column(self, name, lo, hi):
        off, data = self.cols[name]
        return off[lo:hi + 1] - off[lo], data[off[lo]:off[hi]]


def test_bench_index_dump_matches_reference(tmp_path):
    """bench.py --dump-outputs with the index_on leg just above T rows: its sample of the sorted table equals the same
    sample of the reference sort of the same generated input"""
    import bench
    n = _multi_tile_rows() + 1
    out = tmp_path / "gpu"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--orders", "40000",
                        "--customers", "10000", "--products", "500", "--people", "30000", "--index-rows", str(n),
                        "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    side = bench.index_sides(n)
    raw = gpu_ctx().gen_csv("orders", (0, n), seed=SEED, n_cust=side, n_prod=side, header=True).to_host()
    names = [c for c, _ in bench.INDEX_COLS]
    o = orc.reader_rows(raw, select=names)
    cols = {c: o.column(c)[:2] for c in names}
    perm = ref_order_np(cols, ["cust_id", "prod_id"])
    want = tmp_path / "ref"
    bench.dump_table(str(want), "index_on", _Columns({c: ref_gather(*cols[c], perm) for c in names}))
    got = sorted(p.name for p in out.iterdir() if p.name.startswith("index_on."))
    assert got == sorted(p.name for p in want.iterdir())
    assert np.load(want / "index_on.num_rows.npy").tolist() == [n]
    for f in got:
        assert np.array_equal(np.load(out / f), np.load(want / f)), f


# ------------------------------------------------------------------ limits
def test_key_column_count_and_image_size_limits():
    """16 key columns work and 17 are refused; an image of exactly 4096 bytes works and 4097 bytes is refused"""
    import csvplus_b200 as cp
    rng = np.random.default_rng(9)
    n = 5000
    cols = {f"k{c}": from_values([b"", b"a", b"b", b"ab"]) for c in range(16)}
    cols = {c: ref_gather(*v, rng.integers(0, 4, n)) for c, v in cols.items()}
    cols["i"] = _ids(n)
    t = _parse(cols)
    keys = [f"k{c}" for c in range(16)]
    perm = np.asarray(ref_order({k: values(*cols[k]) for k in keys}, keys))
    _check_sorted(t.index_on(*keys).table(), cols, perm)
    with pytest.raises(cp.CsvPlusError) as e:
        t.index_on(*keys, "i")
    assert e.value.status == 4  # CPB_ERR_UNSUPPORTED
    # one key column: width + 2 length bytes (width >= 255) = 4096 -> 512 image words; one byte more is refused
    r = random.Random(9)
    for width, ok in ((4094, True), (4095, False)):
        vals = []
        for k in range(300):
            L = width if k == 0 else r.choice([0, 1, 2000, width - 1, width])
            v = b"p" * L
            if L and r.random() < 0.7:
                p = r.choice([0, L // 2, L - 1])
                v = v[:p] + bytes([r.choice(b"\x00a\xff")]) + v[p + 1:]
            vals.append(v)
        cols = {"k": from_values(vals), "i": _ids(len(vals))}
        t = _parse(cols)
        if ok:
            _check_sorted(t.index_on("k").table(), cols, np.asarray(ref_order({"k": vals}, ["k"])))
        else:
            with pytest.raises(cp.CsvPlusError) as e:
                t.index_on("k")
            assert e.value.status == 4 and "4 KiB" in str(e.value)


def test_oversized_key_refused_before_packing():
    """one 5000-byte key value in 200 k rows: UNSUPPORTED, and no key image is packed (or allocated: words * n * 8
    bytes, ~1 GB here) before the refusal"""
    import csvplus_b200 as cp
    n = 200_000
    vals = [b"%07d" % k for k in range(n)]
    vals[n // 2] = b"q" * 5000
    cols = {"k": from_values(vals), "i": _ids(n)}
    t = _parse(cols)

    def build():
        with pytest.raises(cp.CsvPlusError) as e:
            t.index_on("k")
        return e.value
    err, st = _stats_of(build)
    assert err.status == 4 and "4 KiB" in str(err)
    assert "key_pack" not in st, st.get("key_pack")
