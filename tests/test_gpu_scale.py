"""Parity of the configurations BASELINE.json names, through the public API / C ABI (GPU only):
  * configs[1] at FULL size (people 100 M rows, parse + SelectColumns + Filter(Like)) against the oracle, chunk by chunk;
  * configs[3] pattern (orders x customers x products three-way Join, README.md:34-56) against the oracle, incl. the ToCsv sink;
  * the gathered build side of the multi-GPU path: shards -> cpb_table_from_device -> cpb_table_concat -> index -> join;
  * configs[4]: composite-key IndexOn + ResolveDuplicates(min order_id) with both §Q1 tail shapes, via the resolver of bench.py;
  * (>= 2 GPUs only) a 2-rank torchrun run of the all-gathered three-way join.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as orc
from tests.helpers import assert_table_equals_oracle, gpu_ctx

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0xC5B200


def test_full_size_parse_filter_vs_oracle_chunked():
    """BASELINE configs[1] at its full size: one GPU parse of the whole file, compared with the oracle on consecutive
    row ranges of the same generator (every chunk is the exact byte range of those rows of the big file)"""
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    n = int(os.environ.get("CPB_FULL_ROWS", "100000000"))
    chunk = 5_000_000
    big = ctx.gen_csv("people", (0, n), seed=SEED)
    t, err = cp.parse_csv(ctx, big, spec=[("name", -1), ("surname", -1), ("id", -1)], pred=cp.Like({"name": "Amelia"}))
    assert err is None
    cols = {c: t.column(c) for c in ("name", "surname", "id")}
    row = 0
    pos = 0
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        part = ctx.gen_csv("people", (lo, hi), seed=SEED, header=(lo == 0)).to_host()
        # the chunk is byte-identical to its range of the big buffer
        if lo in (0, chunk * (n // chunk // 2)):
            assert np.array_equal(part[:4096], big.to_host(4096, pos))
        pos += part.size
        if lo == 0:
            o = orc.reader_rows(part, select=["name", "surname", "id"], pred=orc.Like({"name": "Amelia"}))
        else:
            o = orc.reader_rows(part, assume={"id": 0, "name": 1, "surname": 2}, pred=orc.Like({"name": "Amelia"}),
                                opts=orc.Opts(fields_per_record=6))
        k = len(o)
        for c in ("name", "surname", "id"):
            go, gd = cols[c]
            oo, od, pres = o.column(c)
            assert pres.all()
            assert np.array_equal(go[row:row + k + 1] - go[row], oo), (c, lo)
            assert np.array_equal(gd[go[row]:go[row + k]], od), (c, lo)
        row += k
    assert pos == big.nbytes and row == len(t)
    assert 0.09 * n < row < 0.11 * n


def _three_way(ctx, n_orders, n_cust, n_prod, cust_parts=1):
    import csvplus_b200 as cp
    prod = ctx.gen_csv("products", (0, n_prod), seed=SEED, n_prod=n_prod, permute=True)
    orders = ctx.gen_csv("orders", (0, n_orders), seed=SEED, n_cust=n_cust, n_prod=n_prod)
    shards = []
    for r in range(cust_parts):
        lo, hi = r * n_cust // cust_parts, (r + 1) * n_cust // cust_parts
        shards.append(ctx.gen_csv("customers", (lo, hi), seed=SEED, n_cust=n_cust, permute=True, header=True))
    return prod, orders, shards


def _oracle_three_way(prod, orders, cust_all):
    cidx = orc.reader_rows(cust_all, select=["id", "name", "surname"]).unique_index_on("id")
    pidx = orc.reader_rows(prod, select=["prod_id", "product", "price"]).unique_index_on("prod_id")
    return orc.reader_rows(orders, select=["cust_id", "prod_id", "qty", "ts"]).join(cidx, "cust_id").join(pidx)


def test_three_way_join_vs_oracle_with_gathered_build_side():
    """configs[3] pattern; the customers side arrives as 4 separately parsed shards that are re-imported through
    cpb_table_from_device and concatenated with cpb_table_concat, exactly what the all-gather of the multi-GPU path
    hands to the index build"""
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    n_orders, n_cust, n_prod = 300_000, 100_000, 10_000
    prod, orders, shards = _three_way(ctx, n_orders, n_cust, n_prod, cust_parts=4)
    parts = []
    for s in shards:
        t, err = cp.parse_csv(ctx, s, spec=[("id", -1), ("name", -1), ("surname", -1)])
        assert err is None
        ctx.sync()
        imported = cp.Table.from_device_columns(ctx, t.columns, [t.device_column(c) for c in t.columns], len(t))
        ctx.sync()
        parts.append(imported)
        del t
    tc = cp.Table.concat(parts)
    assert len(tc) == n_cust
    cidx = tc.index_on("id", unique=True)
    tp, err = cp.parse_csv(ctx, prod, spec=[("prod_id", -1), ("product", -1), ("price", -1)])
    pidx = tp.index_on("prod_id", unique=True)
    to, err = cp.parse_csv(ctx, orders, spec=[("cust_id", -1), ("prod_id", -1), ("qty", -1), ("ts", -1)])
    j = to.join(cidx, "cust_id").join(pidx)
    # oracle: one customers file = header + the rows of all shards
    hosts = [s.to_host() for s in shards]
    hdr = len(b"id,name,surname,born,city,score\n")
    cust_all = np.concatenate([hosts[0]] + [h[hdr:] for h in hosts[1:]])
    oj = _oracle_three_way(prod.to_host(), orders.to_host(), cust_all)
    assert len(j) == n_orders
    assert_table_equals_oracle(j, oj)
    sink = ("name", "surname", "qty", "product", "price", "ts")  # README.md:59-64
    assert j.to_csv(*sink) == oj.to_csv(*sink)[0]
    # the streamed sink of bench.py's e2e leg: batches into one pinned buffer, header once
    hb = ctx.host_alloc(len(oj.to_csv(*sink)[0]) + 64)
    w = j.slice(0, 100_000).to_csv_into(hb, 0, *sink, header=True)
    w += j.slice(100_000, n_orders).to_csv_into(hb, w, *sink, header=False)
    assert bytes(hb.array()[:w]) == oj.to_csv(*sink)[0]


def test_sliced_table_survives_reimport():
    """a row-range view (Top/Drop/Find) exported by device pointers: offsets do not start at 0 (ADVICE r1)"""
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    t, _ = cp.parse_csv(ctx, ctx.gen_csv("people", (0, 5000), seed=SEED), spec=[("id", -1), ("name", -1)])
    v = t.slice(1000, 3000)
    ctx.sync()
    m = cp.Table.from_device_columns(ctx, v.columns, [v.device_column(c) for c in v.columns], len(v))
    for c in v.columns:
        a, b = v.column(c), m.column(c)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("n_rows", [300_000])
def test_composite_index_and_resolve_duplicates_vs_oracle(n_rows):
    """configs[4] shape: IndexOn(cust_id, prod_id) with ~50 % of the rows in duplicate groups, then
    ResolveDuplicates(min order_id) through dup_groups / dedup_apply and bench.py's vectorised resolver; both §Q1
    tail shapes (last sorted row in a group / a singleton) are searched for and compared with the oracle"""
    import bench
    import csvplus_b200 as cp
    ctx = gpu_ctx()
    side = bench.index_sides(n_rows)
    raw = ctx.gen_csv("orders", (0, n_rows), seed=SEED, n_cust=side, n_prod=side)
    t, err = cp.parse_csv(ctx, raw, spec=bench.INDEX_COLS)
    assert err is None
    host = raw.to_host()
    shapes = set()
    tab, cur = t, host
    for attempt in range(40):
        n = len(tab)
        ix = tab.index_on("cust_id", "prod_id")
        lo, hi = ix.dup_groups()
        in_group = bool(len(hi) and hi[-1] == n)
        if in_group not in shapes:
            shapes.add(in_group)
            grouped = int((hi - lo).sum())
            assert 0.35 * n < grouped < 0.65 * n
            orows = orc.reader_rows(cur, select=[c for c, _ in bench.INDEX_COLS])
            oi = orows.index_on("cust_id", "prod_id")
            # (order inside equal-key groups is an artefact of the sort: compare after the tie-free dedup)
            keep = bench.min_id_resolver(ix.table(), lo, hi)
            ix.dedup_apply(keep)
            oi.dedup("min", "order_id")
            assert len(ix) == len(oi) == n - grouped + len(lo) - (0 if in_group or len(lo) == 0 else 1)
            assert_table_equals_oracle(ix.table(), oi.rows())
            if len(shapes) == 2:
                break
        # the other tail shape: drop every row carrying the greatest key; the next greatest key takes the last position
        tab = bench.without_greatest_key(tab, ("cust_id", "prod_id"))
        cur = tab.to_csv(*[c for c, _ in bench.INDEX_COLS])
    assert shapes == {True, False}


class _OracleTable:
    """oracle rows behind the Table.column(name, lo, hi) interface bench.dump_table reads"""

    def __init__(self, rows):
        self.n = len(rows)
        self.columns = [c.decode() for c in rows.header(0)]
        self.cols = {c: rows.column(c)[:2] for c in self.columns}

    def __len__(self):
        return self.n

    def column(self, name, lo, hi):
        off, data = self.cols[name]
        return off[lo:hi + 1] - off[lo], data[off[lo]:off[hi]]


def test_bench_dump_outputs_match_oracle(tmp_path):
    """bench.py --dump-outputs at a small size: the samples of the joined and the filtered table it writes equal the
    oracle's results on the same generated inputs, written by the same dump"""
    import bench
    n_orders, n_cust, n_prod, n_people = 40_000, 10_000, 500, 30_000
    out = tmp_path / "gpu"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--orders", str(n_orders),
                        "--customers", str(n_cust), "--products", str(n_prod), "--people", str(n_people), "--index-rows", "20000",
                        "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    files = sorted(p.name for p in out.iterdir())
    assert sum(p.stat().st_size for p in out.iterdir()) <= bench.DUMP_LIMIT_BYTES
    for f in files:
        assert np.load(out / f).dtype in (np.float32, np.float64), f
    assert np.load(out / "index_on.num_rows.npy").tolist() == [20_000]

    ctx = gpu_ctx()
    cust = ctx.gen_csv("customers", (0, n_cust), seed=SEED, n_cust=n_cust, permute=True, header=True).to_host()
    prod = ctx.gen_csv("products", (0, n_prod), seed=SEED, n_prod=n_prod, permute=True, header=True).to_host()
    orders = ctx.gen_csv("orders", (0, n_orders), seed=SEED, n_cust=n_cust, n_prod=n_prod, header=True).to_host()
    people = ctx.gen_csv("people", (0, n_people), seed=SEED, header=True).to_host()
    want = tmp_path / "oracle"
    bench.dump_table(str(want), "join", _OracleTable(_oracle_three_way(prod, orders, cust)))
    bench.dump_table(str(want), "csv_parse", _OracleTable(orc.reader_rows(people, select=[c for c, _ in bench.PEOPLE_COLS],
                                                                          pred=orc.Like({"name": "Amelia"}))))
    assert np.load(want / "join.num_rows.npy").tolist() == [n_orders]
    assert {f for f in files if f.startswith(("join.", "csv_parse."))} == {p.name for p in want.iterdir()}
    for p in sorted(want.iterdir()):
        assert np.array_equal(np.load(out / p.name), np.load(p)), p.name


def test_two_rank_allgathered_three_way_join():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", os.path.join(ROOT, "tests", "dist_gpu_worker.py")], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "RANK0_OK" in r.stdout and "RANK1_OK" in r.stdout
