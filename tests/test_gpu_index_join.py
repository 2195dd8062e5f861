"""GPU parity of IndexOn / UniqueIndexOn / Find / SubIndex / ResolveDuplicates / Join / Except / ToCsv
against the CPU oracle.  Mirrors csvplus_test.go: TestIndexImpl (:198-246), TestSimpleUniqueJoin (:368-452),
TestSorted (:454-514), TestMultiIndex (:573-649), TestExcept (:651-693), TestResolver (:695-752),
TestErrors (:808-909), TestWriteFile (:172-196), TestLongChain (:248-366).

Tie order: the reference's sort.Sort is unstable (SURVEY §Q2); the CUDA sort and the oracle (stable=True)
both keep input order inside equal-key runs, so sorted outputs are compared exactly."""
import io
import random

import numpy as np
import pytest

from oracle import oracle as orc
from tests.helpers import assert_table_equals_oracle, gpu_ctx, people_csv, random_csv
from tests.index_ref import ref_gather, ref_order_np

pytestmark = pytest.mark.gpu


def _orders_csv(n, ncust, nprod, seed=3):
    rng = random.Random(seed)
    rows = [b"order_id,cust_id,prod_id,qty,ts"]
    for i in range(n):
        rows.append(b"%d,%d,%d,%d,2016-09-14T08:%02d:%02d+01:00" % (i, rng.randrange(ncust), rng.randrange(nprod), 1 + rng.randrange(100),
                                                                    rng.randrange(60), rng.randrange(60)))
    return b"\n".join(rows) + b"\n"


STOCK = b"prod_id,product,price\n" + b"".join(b"%d,%s,%0.2f\n" % (i, n, 0.01 * (i + 1)) for i, n in enumerate(
    [b"banana", b"apple", b"orange", b"pea", b"tomato", b"potato", b"cucumber", b"iPhone"]))


def test_index_impl_kat():
    # csvplus_test.go:198-246
    import csvplus_b200 as cp
    rows = [
        {"x": "1", "y": "2", "z": "3", "junk": "zzz"}, {"x": "5", "y": "6", "z": "8", "junk": "nnn"},
        {"x": "0", "y": "5", "z": "3", "junk": "xxx"}, {"x": "8", "y": "9", "z": "1", "junk": "aaa"},
        {"x": "7", "y": "4", "z": "0", "junk": "bbb"}, {"x": "5", "y": "6", "z": "9", "junk": "iii"},
        {"x": "2", "y": "6", "z": "7", "junk": "mmm"},
    ]
    index = cp.TakeRows(rows).IndexOn("x", "y", "z")
    r = index.Find("1", "2", "3").ToRows()
    assert r == [{"x": "1", "y": "2", "z": "3", "junk": "zzz"}]
    r = index.Find("5", "6", "8").ToRows()
    assert len(r) == 1 and r[0]["junk"] == "nnn"
    r = index.Find("5", "6").ToRows()
    assert len(r) == 2 and all(x["x"] == "5" and x["y"] == "6" for x in r)
    assert [x["x"] for x in cp.Take(index).ToRows()] == ["0", "1", "2", "5", "5", "7", "8"]
    assert index.Find("9").ToRows() == [] and index.Find("4", "4").ToRows() == []
    assert len(index.Find().ToRows()) == 7
    with pytest.raises(ValueError):
        index.SubIndex("a", "b", "c")


def test_sort_order_is_bytewise_and_stable():
    import csvplus_b200 as cp
    vals = ["10", "9", "a", "a\x00", "", "ab", "a b", "B", "\xff", "\x7f", "aa", "a", "10", "100", "é", "z" * 300, "z" * 299 + "y"]
    rows = [{"k": v, "i": str(i)} for i, v in enumerate(vals)]
    ix = cp.TakeRows(rows).IndexOn("k")
    o = orc.take_rows(rows).index_on("k")
    assert_table_equals_oracle(ix.table(), o.rows())
    # composite keys cannot be concatenated: ("ab","c") vs ("a","bc")
    rows = [{"p": "ab", "q": "c"}, {"p": "a", "q": "bc"}, {"p": "a", "q": ""}, {"p": "", "q": "abc"}, {"p": "a", "q": "b"}]
    ix = cp.TakeRows(rows).IndexOn("p", "q")
    assert_table_equals_oracle(ix.table(), orc.take_rows(rows).index_on("p", "q").rows())
    ix = cp.TakeRows(rows).IndexOn("q", "p")
    assert_table_equals_oracle(ix.table(), orc.take_rows(rows).index_on("q", "p").rows())


@pytest.mark.parametrize("seed", range(3))
def test_index_random_vs_oracle(seed):
    import csvplus_b200 as cp
    rng = random.Random(seed)
    n = 30000
    rows = [{"a": "".join(rng.choice("abc") for _ in range(rng.randrange(0, 4))), "b": str(rng.randrange(50)), "i": str(i)}
            for i in range(n)]
    t = cp.Table.from_rows(gpu_ctx(), rows)
    o = orc.take_rows(rows)
    for keys in (("a",), ("b", "a"), ("a", "b", "i")):
        ix = t.index_on(*keys)
        assert_table_equals_oracle(ix.table(), o.index_on(*keys).rows())
    # Find / SubIndex on the composite index (csvplus_test.go:573-649)
    ix = t.index_on("a", "b")
    oi = o.index_on("a", "b")
    for probe in (("abc",), ("a", "7"), ("", "0"), ("zz",), ("c", "49")):
        assert ix.Find(*probe).ToRows() == [{k.decode(): v.decode() for k, v in r.items()} for r in oi.find(*probe).to_dicts()]
    sub = ix.SubIndex("ab")
    got = cp.Take(sub).ToRows()
    want = [{k.decode(): v.decode() for k, v in r.items()} for r in oi.find("ab").to_dicts()]
    assert got == want
    assert sub.Find("7").ToRows() == [r for r in want if r["b"] == "7"]


def test_unique_index_and_errors():
    # csvplus_test.go:826-841
    import csvplus_b200 as cp
    data = people_csv(120)
    source = cp.Take(cp.FromBytes(data).SelectColumns("id", "name", "surname"))
    with pytest.raises(cp.DataSourceError) as e:
        source.IndexOn("name", "xxx")
    assert str(e.value).endswith('missing column "xxx" while creating an index')
    with pytest.raises(cp.CsvPlusError) as e:
        source.UniqueIndexOn("name")
    o = orc.reader_rows(data, select=["id", "name", "surname"])
    with pytest.raises(orc.OracleError) as oe:
        o.unique_index_on("name")
    assert str(e.value) == str(oe.value)
    assert "duplicate value while creating unique index:" in str(e.value)
    ix = source.UniqueIndexOn("id")
    assert_table_equals_oracle(ix.table(), o.unique_index_on("id").rows())
    with pytest.raises(ValueError):
        source.IndexOn()
    with pytest.raises(ValueError):
        source.IndexOn("id", "id")


def test_sorted_iteration():
    # csvplus_test.go:454-514: byte-lexicographic order of names, then (surname, name)
    import csvplus_b200 as cp
    data = people_csv(120)
    people = cp.Take(cp.FromBytes(data).ExpectHeader({"name": 1, "surname": 2}))
    idx = people.IndexOn("name")
    rows = cp.Take(idx).ToRows()
    assert all(r["name"] == "Amelia" for r in rows[:12]) and rows[12]["name"] == "Ava"
    idx = people.UniqueIndexOn("surname", "name")
    rows = cp.Take(idx).ToRows()
    assert all(r["surname"] == "Brown" for r in rows[:10]) and rows[10]["surname"] == "Davies"
    assert [r["name"] for r in rows[:3]] == ["Amelia", "Ava", "Charlie"]
    o = orc.reader_rows(data, expect={"name": 1, "surname": 2})
    assert_table_equals_oracle(idx.table(), o.unique_index_on("surname", "name").rows())


def test_resolve_duplicates():
    # csvplus_test.go:845-863 and :695-752, plus both tail shapes of SURVEY §Q1
    import csvplus_b200 as cp
    data = people_csv(120)
    source = cp.Take(cp.FromBytes(data).SelectColumns("id", "name", "surname"))
    index = source.IndexOn("name")
    calls = []

    def resolve(rows):
        calls.append(len(rows))
        return rows[0]
    index.ResolveDuplicates(resolve)
    assert calls == [12] * 10 and len(index) == 10

    def keys_after(keys, mode="first"):
        rows = [{"k": k, "v": str(i)} for i, k in enumerate(keys)]
        ix = cp.TakeRows(rows).IndexOn("k")
        ix.ResolveDuplicates((lambda g: g[0]) if mode == "first" else (lambda g: {}))
        oi = orc.take_rows(rows).index_on("k"); oi.dedup("first" if mode == "first" else "drop")
        got = cp.Take(ix).ToRows()
        assert got == [{k.decode(): v.decode() for k, v in r.items()} for r in oi.rows().to_dicts()]
        return [r["k"] for r in got]
    assert keys_after("aab") == ["a"]
    assert keys_after("aabc") == ["a", "b"]
    assert keys_after("abbcdde") == ["a", "b", "c", "d"]
    assert keys_after("abb") == ["a", "b"]
    assert keys_after("abbcdd") == ["a", "b", "c", "d"]
    assert keys_after("abc") == ["a", "b", "c"]
    assert keys_after("abbcdde", "drop") == ["a", "c"]
    # tie-order independent resolver: keep the smallest id (SURVEY §8d config 5)
    rng = random.Random(5)
    rows = [{"surname": rng.choice("ABCDEFGH") * 3, "name": rng.choice("xyzw"), "id": "%05d" % i} for i in range(5000)]
    ix = cp.TakeRows(rows).IndexOn("surname", "name")
    ix.ResolveDuplicates(lambda g: min(g, key=lambda r: r["id"]))
    oi = orc.take_rows(rows).index_on("surname", "name"); oi.dedup("min", "id")
    assert_table_equals_oracle(ix.table(), oi.rows())
    # keeping something after dedup: the index is still searchable
    assert len(ix.Find("AAA").ToRows()) == len(oi.find("AAA"))


def test_simple_unique_join():
    # csvplus_test.go:368-452
    import csvplus_b200 as cp
    pdata = people_csv(120)
    odata = _orders_csv(10000, 120, 8)
    people = cp.Take(cp.FromBytes(pdata).SelectColumns("id", "name", "surname"))
    orders = cp.Take(cp.FromBytes(odata).SelectColumns("order_id", "cust_id", "qty"))
    idx = people.UniqueIndexOn("id")
    joined = orders.Join(idx, "cust_id").ToRows()
    op = orc.reader_rows(pdata, select=["id", "name", "surname"])
    oo = orc.reader_rows(odata, select=["order_id", "cust_id", "qty"])
    oj = oo.join(op.unique_index_on("id"), "cust_id")
    assert len(joined) == len(oj) == 10000
    assert all(len(r) == 6 and r["id"] == r["cust_id"] for r in joined)
    t, _ = orders._table()
    assert_table_equals_oracle(t.join(idx, "cust_id"), oj)


def test_join_duplicates_prefix_natural_and_except():
    import csvplus_b200 as cp
    odata = _orders_csv(3000, 40, 8)
    o_orders = orc.reader_rows(odata)
    orders = cp.Take(cp.FromBytes(odata))
    # non-unique index, prefix join on 1 of 2 key columns (csvplus_test.go:1161-1186 shape)
    idx = orders.IndexOn("cust_id", "prod_id")
    oidx = o_orders.index_on("cust_id", "prod_id")
    people = b"id,name\n" + b"".join(b"%d,n%d\n" % (i, i) for i in range(0, 60, 2))
    probe = cp.Take(cp.FromBytes(people))
    t, _ = probe._table()
    oj = orc.reader_rows(people).join(oidx, "id")
    assert_table_equals_oracle(t.join(idx, "id"), oj)
    assert len(oj) > 1000
    # natural join on the index columns; probe value wins name collisions (mergeRows)
    stock_idx = cp.Take(cp.FromBytes(STOCK)).UniqueIndexOn("prod_id")
    o_stock_idx = orc.reader_rows(STOCK).unique_index_on("prod_id")
    to, _ = orders._table()
    assert_table_equals_oracle(to.join(stock_idx), o_orders.join(o_stock_idx))
    collide = b"prod_id,product\n3,override\n99,none\n"
    tc, _ = cp.Take(cp.FromBytes(collide))._table()
    assert_table_equals_oracle(tc.join(stock_idx), orc.reader_rows(collide).join(o_stock_idx))
    # Except (csvplus_test.go:651-693)
    assert_table_equals_oracle(t.join(idx, "id", anti=True), orc.reader_rows(people).except_(oidx, "id"))
    assert_table_equals_oracle(tc.join(stock_idx, anti=True), orc.reader_rows(collide).except_(o_stock_idx))
    # missing join column and too many columns
    with pytest.raises(cp.DataSourceError) as e:
        probe.Join(idx, "nope").ToRows()
    assert str(e.value).endswith('missing column "nope"')
    with pytest.raises(ValueError):
        probe.Join(stock_idx, "id", "name")
    # values longer than any index key never match
    long_probe = b"id\n" + b"7" * 40 + b"\n7\n"
    tl, _ = cp.Take(cp.FromBytes(long_probe))._table()
    assert_table_equals_oracle(tl.join(idx, "id"), orc.reader_rows(long_probe).join(oidx, "id"))


def test_join_large_index_global_hash_path():
    """index too large for the shared-memory table: global-memory probe"""
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    ncust = 300_000
    cust = ctx.gen_csv("customers", (0, ncust), n_cust=ncust, permute=True)
    orders = ctx.gen_csv("orders", (0, 400_000), n_cust=ncust + 1000, n_prod=100)
    tc, _ = cp.parse_csv(ctx, cust, spec=[("id", -1), ("name", -1), ("surname", -1)])
    to, _ = cp.parse_csv(ctx, orders, spec=[("cust_id", -1), ("prod_id", -1), ("qty", -1), ("ts", -1)])
    idx = tc.index_on("id", unique=True)
    j = to.join(idx, "cust_id")
    oc = orc.reader_rows(cust.to_host(), select=["id", "name", "surname"])
    oo = orc.reader_rows(orders.to_host(), select=["cust_id", "prod_id", "qty", "ts"])
    oj = oo.join(oc.unique_index_on("id"), "cust_id")
    assert 390_000 < len(oj) < 400_000  # ids >= ncust find no customer
    assert_table_equals_oracle(j, oj)
    assert_table_equals_oracle(idx.table(), oc.unique_index_on("id").rows())


def test_to_csv_roundtrip_and_quoting():
    # csvplus_test.go:172-196 + SURVEY App. B
    import csvplus_b200 as cp
    data = people_csv(120)
    src = cp.Take(cp.FromBytes(data).SelectColumns("id", "name", "surname", "born"))
    buf = io.BytesIO()
    src.ToCsv(buf, "id", "name", "surname", "born")
    assert buf.getvalue().strip() == data.strip()
    nasty = random_csv(11, nrows=2000, ncols=4, quoted_p=0.5, crlf_p=0.2)
    t, err = cp.parse_csv(gpu_ctx(), nasty)
    assert err is None
    want, oerr = orc.reader_rows(nasty).to_csv("c3", "c0", "c1")
    assert oerr is None and t.to_csv("c3", "c0", "c1") == want
    rows = [{"a": 'x"y', "b": " lead"}, {"a": "", "b": "p,q"}, {"a": "\\.", "b": " nbsp"}, {"a": "　x", "b": "\r"}]
    assert cp.Table.from_rows(gpu_ctx(), rows).to_csv("a", "b") == orc.take_rows(rows).to_csv("a", "b")[0]
    with pytest.raises(cp.DataSourceError) as e:
        src.ToCsv(io.BytesIO(), "id", "nope")
    assert str(e.value).endswith('missing column "nope"')
    with pytest.raises(ValueError):
        src.ToCsv(io.BytesIO())


def test_long_chain():
    # csvplus_test.go:248-366 — opaque Python closures sit at host boundaries between device stages
    import csvplus_b200 as cp
    odata = _orders_csv(10000, 120, 8)
    pdata = people_csv(120)
    orders = cp.Take(cp.FromBytes(odata).SelectColumns("order_id", "cust_id", "prod_id", "qty", "ts")).IndexOn("cust_id")
    products = cp.Take(cp.FromBytes(STOCK).SelectColumns("prod_id", "product", "price")).UniqueIndexOn("prod_id")
    people = cp.Take(cp.FromBytes(pdata).SelectColumns("id", "name", "surname", "born"))
    out = (people.Filter(lambda row: int(row["born"]) > 1970)
           .SelectColumns("id", "name", "surname")
           .Join(orders, "id")
           .DropColumns("ts", "order_id", "cust_id")
           .Join(products)
           .DropColumns("prod_id")
           .Map(lambda row: {**row, "name": "Julia"} if row["name"] == "Amelia" else row)
           .Filter(cp.Like({"surname": "Smith"}))
           .Top(10)
           .DropColumns("id")).ToRows()
    assert 0 < len(out) <= 10
    for row in out:
        assert row["surname"] == "Smith" and row["name"] != "Amelia"
        assert sorted(row) == ["name", "price", "product", "qty", "surname"]
    assert len(cp.Take(orders).ToRows()) == 10000
    assert len(cp.Take(products).ToRows()) == 8


def _kv_csv(header, rows):
    return (",".join(header) + "\n" + "".join(",".join(r) + "\n" for r in rows)).encode()


@pytest.mark.parametrize("shape", ["slots4", "slots1_empty", "too_wide", "too_long_value", "five_cols"])
def test_join_row_slot_path_and_fallbacks(shape):
    """gather of index rows: fixed-size row slots (<= 4 output columns, values <= 255 bytes, row <= 64 bytes) and
    the per-column fallback must both reproduce mergeRows (csvplus.go:571-583) exactly"""
    import csvplus_b200 as cp
    rng = random.Random(sum(shape.encode()))
    nidx, nprobe = 257, 1999

    def word(maxlen):
        return "".join(rng.choice("abcxyz01") for _ in range(rng.randrange(0, maxlen + 1)))
    if shape == "slots4":
        hdr = ["k", "a", "b", "c"]; mk = lambda i: [str(i), word(20), word(20), word(18)]
    elif shape == "slots1_empty":
        hdr = ["k"]; mk = lambda i: [str(i)]
    elif shape == "too_wide":
        hdr = ["k", "a", "b"]; mk = lambda i: [str(i), word(40), word(40)]
    elif shape == "too_long_value":
        hdr = ["k", "a"]; mk = lambda i: [str(i), "q" * 300 if i == 77 else word(5)]
    else:
        hdr = ["k", "a", "b", "c", "d"]; mk = lambda i: [str(i), word(3), word(3), word(3), word(3)]
    # non-unique index: every third key appears twice
    irows = [mk(i) for i in range(nidx)] + [mk(i) for i in range(0, nidx, 3)]
    rng.shuffle(irows)
    idata = _kv_csv(hdr, irows)
    pdata = _kv_csv(["pid", "k2"], [[str(j), str(rng.randrange(nidx + 20))] for j in range(nprobe)])
    idx = cp.Take(cp.FromBytes(idata)).IndexOn("k")
    oidx = orc.reader_rows(idata).index_on("k")
    tp, _ = cp.Take(cp.FromBytes(pdata))._table()
    op = orc.reader_rows(pdata)
    oj = op.join(oidx, "k2")
    assert len(oj) > nprobe
    assert_table_equals_oracle(tp.join(idx, "k2"), oj)
    # second probe of the same index with fewer rows than the index (cached slots are reused)
    small = _kv_csv(["pid", "k2"], [[str(j), str(j * 7 % nidx)] for j in range(33)])
    ts, _ = cp.Take(cp.FromBytes(small))._table()
    assert_table_equals_oracle(ts.join(idx, "k2"), orc.reader_rows(small).join(oidx, "k2"))
    # unique index: identity fast path (every probe row matches exactly once)
    udata = _kv_csv(hdr, [mk(i) for i in range(nidx)])
    uidx = cp.Take(cp.FromBytes(udata)).UniqueIndexOn("k")
    exact = _kv_csv(["pid", "k2"], [[str(j), str(rng.randrange(nidx))] for j in range(nprobe)])
    te, _ = cp.Take(cp.FromBytes(exact))._table()
    assert_table_equals_oracle(te.join(uidx, "k2"), orc.reader_rows(exact).join(orc.reader_rows(udata).unique_index_on("k"), "k2"))


@pytest.mark.parametrize("shape", ["nonunique_slot32", "wide_key_generic"])
def test_join_large_index_other_probe_tables(shape):
    """large indices that cannot use the 16-byte unique-key slots: non-unique keys (32-byte slots with run lengths)
    and key prefixes wider than 24 bytes (slot -> heads -> image probe in global memory)"""
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    ncust = 120_000
    cust = ctx.gen_csv("customers", (0, ncust), n_cust=ncust, permute=True)
    orders = ctx.gen_csv("orders", (0, 200_000), n_cust=ncust, n_prod=100)
    tc, _ = cp.parse_csv(ctx, cust, spec=[("id", -1), ("name", -1), ("surname", -1)])
    to, _ = cp.parse_csv(ctx, orders, spec=[("cust_id", -1), ("prod_id", -1), ("qty", -1), ("ts", -1)])
    oc = orc.reader_rows(cust.to_host(), select=["id", "name", "surname"])
    oo = orc.reader_rows(orders.to_host(), select=["cust_id", "prod_id", "qty", "ts"])
    if shape == "nonunique_slot32":
        idx = to.index_on("cust_id")
        j = tc.join(idx, "id")
        oj = oc.join(oo.index_on("cust_id"), "id")
        assert len(oj) > 150_000
    else:
        idx = to.index_on("ts", "cust_id", "prod_id")
        probe, _ = cp.parse_csv(ctx, orders, spec=[("ts", -1), ("cust_id", -1), ("prod_id", -1), ("order_id", -1)])
        j = probe.join(idx, "ts", "cust_id", "prod_id")
        op = orc.reader_rows(orders.to_host(), select=["ts", "cust_id", "prod_id", "order_id"])
        oj = op.join(oo.index_on("ts", "cust_id", "prod_id"), "ts", "cust_id", "prod_id")
        assert len(oj) >= 200_000
    assert_table_equals_oracle(j, oj)


def test_join_scale_property_id_equals_cust_id():
    """BASELINE-size shape at 20 M x 2 M rows (too large for the oracle): size-independent properties of a
    foreign-key join — every probe row survives in order (the probe columns are shared, not copied), and the
    index-side key column gathered through the row slots is byte-identical to the probe key column"""
    import torch
    import csvplus_b200 as cp
    from csvplus_b200.dist import _as_tensor
    ctx = gpu_ctx()
    ncust, nord = 2_000_000, 20_000_000
    cust = ctx.gen_csv("customers", (0, ncust), n_cust=ncust, permute=True)
    orders = ctx.gen_csv("orders", (0, nord), n_cust=ncust, n_prod=1000)
    tc, _ = cp.parse_csv(ctx, cust, spec=[("id", -1), ("name", -1), ("surname", -1)])
    to, _ = cp.parse_csv(ctx, orders, spec=[("cust_id", -1), ("prod_id", -1), ("qty", -1), ("ts", -1)])
    assert len(tc) == ncust and len(to) == nord
    idx = tc.index_on("id", unique=True)
    j = to.join(idx, "cust_id")
    assert len(j) == nord
    ctx.sync()

    def col(t, name):
        po, pd = t.device_column(name)
        off = _as_tensor(po, 4 * (len(t) + 1)).view(torch.int32)
        return off, _as_tensor(pd, int(off[-1].item()))
    oi, di = col(j, "id")
    oc, dc = col(j, "cust_id")
    assert torch.equal(oi, oc) and torch.equal(di, dc)
    # the probe columns of an exact-once join are the probe table's own buffers
    assert j.device_column("ts") == to.device_column("ts")
    # sorted index (2 M rows: blocks of the radix sort walk several tiles): exactly the reference's bytewise order
    ids = tc.column("id")
    want = ref_gather(*ids, ref_order_np({"id": ids}, ["id"]))
    so, sd = idx.table().column("id")
    assert np.array_equal(so, want[0]) and np.array_equal(sd, want[1])
