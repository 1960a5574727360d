"""CPU: bench.py's synthetic-data helpers (the matrix must not depend on thread count or rank count)."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import refapi  # noqa: E402


def test_gen_bins_is_slice_and_thread_invariant():
    a = bench.gen_bins(70000, 300, 44, threads=1)
    b = bench.gen_bins(70000, 300, 44, col_lo=96, col_hi=290, threads=5)
    assert a.dtype == np.uint8 and a.max() <= 254
    assert np.array_equal(a[:, 96:290], b)
    assert not np.array_equal(a, bench.gen_bins(70000, 300, 45))


def test_gen_bins_row_ranges_tile_the_matrix():
    a = bench.gen_bins(200000, 160, 7)
    b = bench.gen_bins(200000, 160, 7, row_lo=65536, row_hi=150000)
    assert np.array_equal(a[65536:150000], b)
    c = bench.gen_bins(200000, 160, 7, col_lo=128, col_hi=160, row_lo=131072)
    assert np.array_equal(a[131072:, 128:], c)


def test_effective_cores_is_sane():
    n = bench.effective_cores()
    assert 1 <= n <= (os.cpu_count() or 1)


@pytest.mark.skipif(not refapi.available(), reason="times the reference library itself: needs oracle/_ref (oracle/Makefile.ref)")
def test_reference_arm_prints_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C2", "--rows", "20000",
                        "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "iters/sec" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0
    # the arm trains on exactly the workload it prints: no sampling, no scaling
    assert "20000 rows" in d["config"]["workload"] and "all 20000 rows" in d["cpu_baseline"]["sample"]
    assert abs(d["value"] * d["ms_per_step"] - 1e3) < 1e-6 * 1e3


def test_dump_outputs_writes_the_tree_and_a_fixed_score_sample(tmp_path):
    from lightgbm_b200.tree_learner import SPLIT_DTYPE, Tree
    sp = np.zeros(2, SPLIT_DTYPE)
    sp["feature"] = [3, 7]; sp["gain"] = [1.5, 0.25]
    t = Tree(3, sp, np.array([0.1, -0.2, 0.3]), np.ones(3), np.array([5, 6, 7], np.int32), np.array([1, 2, 2], np.int32), 0.0, 18.0)
    scores = np.random.default_rng(1).normal(size=bench.DUMP_SCORE_ROWS + 5)
    bench.dump_outputs(str(tmp_path / "a"), t, scores)
    bench.dump_outputs(str(tmp_path / "b"), t, scores)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(p.name for p in (tmp_path / "b").iterdir())
    assert sum((tmp_path / "a" / n).stat().st_size for n in names) <= 64 << 20
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and np.array_equal(a, b)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "tree_split_feature.npy"), [3, 7])
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "tree_leaf_count.npy"), [5, 6, 7])
    rows = np.load(tmp_path / "a" / "score_rows.npy").astype(np.int64)
    assert len(rows) == bench.DUMP_SCORE_ROWS and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "scores.npy"), scores[rows])


def test_c4_generator_raw_and_bundled_views_agree():
    """C4: the raw sparse features (fed to the reference arms) and the EFB-bundled columns (this repo's arm) describe the
    same matrix, features of a block of 4 are mutually exclusive, and any 64K-aligned row range / column range of the
    bundled view equals the corresponding slice."""
    wl = dict(bench.WORKLOADS["C4"], rows=140000, cols=512)
    cols = bench.gen_columns(wl)
    raw = bench.gen_efb4(wl["rows"], wl["cols"], wl["seed"], raw=True)
    assert cols.shape == (140000, 128) and raw.shape == (140000, 512) and cols.max() <= 252
    assert (raw.reshape(len(raw), -1, 4) > 0).sum(axis=2).max() == 1
    r, c = np.nonzero(raw)
    assert np.array_equal(cols[r, c // 4], 1 + bench.EFB_VALUES * (c % 4) + raw[r, c] - 1)
    assert np.array_equal((cols > 0), (raw.reshape(len(raw), -1, 4) > 0).any(axis=2))
    assert abs((cols > 0).mean() - (1 - (1 - bench.EFB_P) ** 4)) < 3e-3
    part = bench.gen_columns(wl, 32, 96, row_lo=65536)
    assert np.array_equal(part, cols[65536:, 32:96])
    y = bench.gen_label_wl(wl, cols[:, :bench.LABEL_COLS["efb4"]])
    assert set(np.unique(y)) == {0.0, 1.0} and 0.3 < y.mean() < 0.7


def test_c5_generator_and_row_sliced_labels():
    wl = dict(bench.WORKLOADS["C5"], rows=150000)
    h = bench.gen_columns(wl)
    assert h.shape == (150000, 28) and h.max() <= 254
    assert np.array_equal(h[:, 21], ((h[:, 0].astype(int) + h[:, 1] + h[:, 2]) // 3).astype(np.uint8))
    y = bench.gen_label_wl(wl, h)
    assert np.array_equal(y[65536:], bench.gen_label_wl(wl, h[65536:], row_lo=65536))     # a rank's row slice gets the same labels


def test_c4_reference_dataset_bundles_like_the_generator():
    """The reference's own Dataset construction (cuda rules, sampled-column API + PushRows) turns the raw C4 features into
    exactly the bundled columns the generator writes directly (same bundles, offsets 1 + 63 j, most-frequent bin elided).
    The Dataset the reference built from the 70000 x 64 workload is recorded in tests/golden/reference/c4_dataset_70k_x64.npz
    (its layout, and the SHA-1 of its stored bytes)."""
    from oracle.refapi import Layout
    wl = dict(bench.WORKLOADS["C4"], rows=70000, cols=64)
    rec = np.load(os.path.join(ROOT, "tests", "golden", "reference", "c4_dataset_70k_x64.npz"))
    lay = Layout.from_npz_dict(rec)
    assert lay.num_data == wl["rows"] and lay.num_columns == 16 and lay.num_features == 64
    raw = bench.gen_efb4(wl["rows"], wl["cols"], wl["seed"], raw=True)
    bins = np.zeros((lay.num_data, lay.num_columns), np.uint8)        # zero where every feature of a bundle is zero
    for f in range(lay.num_features):
        rf = int(lay.feat_real_index[f])
        assert lay.feat_num_bin[f] == bench.EFB_VALUES + 1 and lay.feat_mfb[f] == 0
        nz = np.nonzero(raw[:, rf])[0]
        assert not bins[nz, lay.feat_column[f]].any()                 # exclusive inside the bundle
        bins[nz, lay.feat_column[f]] = lay.feat_lo[f] + raw[nz, rf] - 1
    assert hashlib.sha1(bins.tobytes()).hexdigest() == str(rec["bins_sha1"]), "not the bytes the reference stored"
