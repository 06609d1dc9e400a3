"""bench.py's host-side arithmetic, checked without a GPU: the roofline blocks (which ceiling binds, that `frac` is
t_roof / t_measured, that measured DRAM traffic is reported per launch) and the JSON line of the reference arm."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO]
import bench  # noqa: E402

CEIL = {"gather_gbs": {"8MB_64B_independent": 8000.0, "8MB_32B_independent": 9000.0, "1GB_64B_independent": 1400.0,
                       "1GB_32B_independent": 1350.0},
        "issue_tops": {"fadd_fmul": 36.0}}


def counters(segments, launches, extend_ms, shade_ms=100.0, paths=None):
    return {"segments": segments, "paths": paths if paths is not None else segments // 4, "extend_launches": launches,
            "extend_ms": extend_ms, "shade_ms": shade_ms}


def test_roofline_l2_resident_tree_is_bound_by_the_gather_ceiling():
    c = counters(400_000_000, 8, 8 * 6.0)                       # 50 M segments per 6 ms launch
    ci = {"segments": 1000, "node_visits": 7000, "tri_tests": 4500}
    r = bench.extend_roofline(c, ci, CEIL, "config2", 6_600_000, 1000.0, None, 4)
    bvh_b = 7.0 * 64 + 4.5 * 48
    assert r["bvh_resident_in"] == "L2" and r["bound"] == "l2_gather" and r["node_bytes"] == 64
    assert r["bvh_bytes_per_segment"] == pytest.approx(bvh_b) and r["bytes_per_segment"] == pytest.approx(bvh_b + 96)
    t_gather = bvh_b * 50e6 / 8000e9
    assert r["frac"] == pytest.approx(t_gather / 6.0e-3)
    assert r["achieved"] == pytest.approx(bvh_b * 50e6 / 6.0e-3 * 1e-9) and r["peak"] == 8000.0
    assert r["frac_by_ceiling"]["fp32"] == pytest.approx((7.0 * 4 * 24 + 4.5 * 56) * 50e6 / 36e12 / 6.0e-3)
    assert r["frac_by_ceiling"]["hbm"] == pytest.approx(96 * 50e6 / (r["peaks"]["hbm_gbs"] * 1e9) / 6.0e-3)
    assert max(r["frac_by_ceiling"].values()) == pytest.approx(r["frac"]) and r["frac"] < 1.2
    assert r["extend_share_of_step"] == pytest.approx(48.0 / 1000.0)


def test_roofline_hbm_resident_tree_is_charged_to_the_copy_peak_and_reports_measured_dram():
    c = counters(800_000_000, 2, 2 * 80.0)
    ci = {"segments": 1000, "node_visits": 9700, "tri_tests": 4900}
    r = bench.extend_roofline(c, ci, CEIL, "config4", 658_000_000, None, None, 4)
    assert r["bvh_resident_in"] == "HBM" and r["bound"] == "hbm" and "hbm_gather" not in r["t_roof_ms"]
    b = 9.7 * 64 + 4.9 * 48 + 96
    assert r["frac"] == pytest.approx(b * 400e6 / (r["peaks"]["hbm_gbs"] * 1e9) / 80e-3)
    tr = bench.load_traffic("config4")
    if tr is not None:   # committed ncu pass: traffic is per LAUNCH, the diagnostic compares it with both HBM rates
        assert r["traffic"] == pytest.approx(tr["dram_bytes_per_segment"] * 400e6)
        d = r["dram_measured"]
        assert d["gbs"] == pytest.approx(r["traffic"] / 80e-3 * 1e-9)
        assert d["frac_of_hbm_random_gather_peak"] == pytest.approx(d["gbs"] / 1400.0)
        assert 0.0 < d["algorithmic_bytes_served_on_chip"] < 1.0


def test_binary_tree_uses_32_byte_nodes_and_two_boxes_per_visit():
    c = counters(1000, 1, 1.0)
    ci = {"segments": 10, "node_visits": 240, "tri_tests": 40}
    r = bench.extend_roofline(c, ci, None, "config1", 5000, 2.0, {"sm_mhz": 1965.0}, 2)
    assert r["node_bytes"] == 32 and r["flops_per_segment"] == pytest.approx(24 * 2 * 24 + 4 * 56)
    assert r["peaks"]["fp32_source"].startswith("estimate") and "l2_gather" not in r["t_roof_ms"]


def test_shade_roofline_counts_the_streamed_records():
    c = counters(4_000_000, 1, 1.0, shade_ms=2.0, paths=1_000_000)
    r = bench.shade_roofline(c, 10.0)
    total = 64.0 * 4e6 + 48.0 * 3e6 + 80.0 * 1e6
    assert r["achieved"] == pytest.approx(total / 2e-3 * 1e-9) and r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    assert r["share_of_step"] == pytest.approx(0.2)
    assert bench.shade_roofline(counters(0, 1, 1.0), 1.0) is None


def test_committed_traffic_table_matches_its_raw_csv():
    """profiles/extend_traffic.json is derived data: recompute one entry from the committed ncu CSV."""
    import csv
    t = json.load(open(os.path.join(REPO, "profiles", "extend_traffic.json")))
    for name, e in t.items():
        raw = os.path.join(REPO, "profiles", f"r2_traffic_{name}.csv")
        if not os.path.exists(raw):
            continue
        rows = list(csv.reader(open(raw)))
        hi = next(i for i, r in enumerate(rows) if "Kernel Name" in r)
        col = {h: i for i, h in enumerate(rows[hi])}
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        total = 0.0
        for r in rows[hi + 1:]:
            if len(r) >= len(col) and "k_extend" in r[col["Kernel Name"]] and r[col["Metric Name"]].startswith("dram__bytes"):
                total += float(r[col["Metric Value"]].replace(",", "")) * scale[r[col["Metric Unit"]]]
        assert e["dram_bytes_per_segment"] == pytest.approx(total / e["segments"], rel=1e-6), name


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` on the smallest workload: one JSON line with impl, metric, cpu_baseline and an e2e
    block without copies (the CPU arm needs no GPU and may run here)."""
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--workload", "config1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "Mrays/s" and d["unit"] == "Mrays/s" and d["value"] > 0
    assert d["higher_is_better"] is True and d["scaling"] == "strong" and d["steps"] == 1 and d["warmup"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["name"] == "config1" and "workload" in d["config"]


def test_dump_outputs_is_a_fixed_sample_within_64_mb(tmp_path):
    """--dump-outputs: a small image is written whole; a 4K one as the same seeded pixel sample every time, under
    64 MB in all, each stored value the image's own."""
    import numpy as np
    small = np.arange(6 * 5 * 3, dtype=np.uint8).reshape(6, 5, 3)
    bench.dump_outputs(str(tmp_path / "s"), small)
    assert np.array_equal(np.load(tmp_path / "s" / "screenshot.npy"), small.reshape(-1, 3).astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "s" / "screenshot_pixel_index.npy"), np.arange(30, dtype=np.float64))
    shot = np.random.default_rng(1).integers(0, 256, (2160, 3840, 3), dtype=np.uint8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), shot)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["screenshot.npy", "screenshot_pixel_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    for f in files:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
    rgb, idx = np.load(tmp_path / "a" / "screenshot.npy"), np.load(tmp_path / "a" / "screenshot_pixel_index.npy")
    assert rgb.dtype == np.float32 and idx.dtype == np.float64 and rgb.shape == (bench.DUMP_PIXELS, 3)
    assert np.all(np.diff(idx) > 0) and np.array_equal(rgb, shot.reshape(-1, 3)[idx.astype(np.int64)])


def test_microbench_library_is_built_by_build():
    """bench.py's `ceilings` block (the L2 / HBM gather and FP32-issue rates the roofline is measured against) needs
    tools/libmicrobench.so; __graft_entry__.build() must compile it, and it must export what bench.microbench binds."""
    import ctypes
    path = os.path.join(REPO, "tools", "libmicrobench.so")
    if not os.path.exists(path):
        subprocess.check_call(["make", "-C", os.path.join(REPO, "tools"), "all"])
    src = open(os.path.join(REPO, "__graft_entry__.py")).read()
    assert '"tools"), "all"' in src, "build() does not compile tools/libmicrobench.so"
    L = ctypes.CDLL(path)
    for sym in ("mb_gather_gbs", "mb_issue_tops", "mb_stream_gbs"):
        assert hasattr(L, sym), sym
