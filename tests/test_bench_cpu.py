"""Host-side helpers of bench.py that must not depend on a GPU: the ncu traffic reader behind roofline.traffic, the
NUMA binding (best effort, never raises) and the clock-sample filter."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_ncu_traffic_reads_committed_profile():
    t, src = bench.ncu_traffic([os.path.join(ROOT, "profiles", "does_not_exist.csv"), os.path.join(ROOT, "profiles", "r1_traffic_csv_scan.csv")])
    # mean of the customers (0.69 GB) and orders (10.87 GB) csv_scan launches of one round-1 join step
    assert t is not None and 5.5e9 < t < 6.1e9 and src.endswith("r1_traffic_csv_scan.csv")
    assert bench.ncu_traffic([os.path.join(ROOT, "profiles", "does_not_exist.csv")]) == (None, None)


def test_ncu_traffic_units_and_kernel_filter(tmp_path):
    p = tmp_path / "t.csv"
    hdr = '"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"\n'
    row = '"{i}","1","p","h","{k}","1","7","(256, 1, 1)","(444, 1, 1)","0","10.0","s","{m}","{u}","{v}"\n'
    p.write_text("==PROF== noise\n" + hdr
                 + row.format(i=0, k="void csv_scan_kernel<4, 1, 0>(ParseParams)", m="dram__bytes_read.sum", u="Gbyte", v="1.5")
                 + row.format(i=0, k="void csv_scan_kernel<4, 1, 0>(ParseParams)", m="dram__bytes_write.sum", u="Mbyte", v="500")
                 + row.format(i=0, k="void csv_scan_kernel<4, 1, 0>(ParseParams)", m="gpu__time_duration.sum", u="ns", v="9000")
                 + row.format(i=1, k="other_kernel()", m="dram__bytes_read.sum", u="byte", v="7")
                 + row.format(i=2, k="void csv_scan_kernel<3, 1, 0>(ParseParams)", m="dram__bytes_read.sum", u="byte", v="1000000000"))
    assert bench.ncu_traffic([str(p)])[0] == (2.0e9 + 1.0e9) / 2


def test_numa_binding_is_best_effort():
    before = os.sched_getaffinity(0)
    assert bench.bind_to_gpu_numa_node(0) is None or isinstance(bench.bind_to_gpu_numa_node(0), int)
    assert os.sched_getaffinity(0) <= before  # never widens, never raises without a GPU


def test_workload_config_names_the_baseline_configs():
    cfg = bench.workload_config(1)
    assert "workload" in cfg and "model" not in cfg and cfg["orders_rows_per_gpu"] == 125_000_000
    assert cfg["customers_rows"] == 100_000_000 and cfg["products_rows"] == 1_000_000  # BASELINE configs[3] at --gpus 8
    assert "NCCL" in bench.workload_config(4)["parallelism"]
    ref = bench.workload_config(1, ref=(2_000_000, 1_600_000, 100_000))  # the reference arm states the sample it ran
    assert ref["orders_rows_per_gpu"] == 2_000_000 and ref["customers_rows"] == 1_600_000


def test_min_id_resolver_keeps_bytewise_smallest():
    import numpy as np

    class FakeTable:
        def __init__(self, vals):
            self.vals = vals

        def column(self, name):
            off = np.zeros(len(self.vals) + 1, np.int64); off[1:] = np.cumsum([len(v) for v in self.vals])
            return off, np.frombuffer(b"".join(self.vals), np.uint8)
    vals = [b"7", b"10", b"9", b"100", b"3", b"21", b"2", b"20", b"5"]
    lo, hi = np.array([1, 5], np.int64), np.array([4, 8], np.int64)  # groups [1,4) and [5,8)
    keep = bench.min_id_resolver(FakeTable(vals), lo, hi)
    # bytewise: "10" < "100" < "9" ; "2" < "20" < "21"
    assert keep.tolist() == [1, 6]
    assert bench.index_sides(10_000_000) == 3794


def test_dump_sample_is_fixed_and_covers_both_ends():
    n = 125_000_000
    blocks = bench.dump_sample_blocks(n)
    assert blocks == bench.dump_sample_blocks(n) and len(blocks) == bench.DUMP_BLOCKS
    assert blocks[0] == (0, bench.DUMP_BLOCK_ROWS) and blocks[-1][1] == n
    assert all(a[1] <= b[0] for a, b in zip(blocks, blocks[1:]))
    assert bench.dump_sample_blocks(1000) == [(0, 256), (256, 512), (512, 768), (768, 1000)]
    assert bench.dump_sample_blocks(0) == []


def test_dump_table_writes_float_byte_matrices(tmp_path):
    import numpy as np

    class FakeTable:  # Table.column(name, lo, hi): offsets rebased to 0 and the bytes of rows [lo, hi)
        columns = ["a", "b"]
        vals = {"a": [b"x%d" % i for i in range(600)], "b": [b"" if i % 3 else b"\xff\x00" * (i % 5) for i in range(600)]}

        def __len__(self):
            return 600

        def column(self, name, lo, hi):
            v = self.vals[name][lo:hi]
            off = np.zeros(len(v) + 1, np.int64); off[1:] = np.cumsum([len(x) for x in v])
            return off, np.frombuffer(b"".join(v), np.uint8)
    t = FakeTable()
    written = bench.dump_table(str(tmp_path), "t", t)
    files = sorted(p.name for p in tmp_path.iterdir())
    assert files == ["t.a.npy", "t.b.npy", "t.num_rows.npy", "t.sample_rows.npy"]
    assert written == sum(p.stat().st_size for p in tmp_path.iterdir())
    assert np.load(tmp_path / "t.num_rows.npy").tolist() == [600.0]
    rows = np.load(tmp_path / "t.sample_rows.npy")
    assert rows.dtype == np.float64 and rows.tolist() == list(range(600))
    for c in t.columns:
        m = np.load(tmp_path / f"t.{c}.npy")
        assert m.dtype == np.float32 and m.shape == (600, max(len(v) for v in t.vals[c]))
        for i in (0, 1, 3, 4, 599):
            v = t.vals[c][i]
            assert m[i, :len(v)].tolist() == list(v) and (m[i, len(v):] == -1).all()
