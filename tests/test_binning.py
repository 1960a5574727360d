"""Dataset construction (SURVEY.md §8 f-3) against Datasets built by the unmodified reference.

tests/golden/binning_*.npz hold float matrices and what LGBM_DatasetCreateFromMat (device_type=cuda Dataset rules) made of
them: per-feature layout, bin upper bounds, every stored byte (tests/golden/make_binning_golden.py).

CPU part (no GPU): LGBMB200_BinnerFit — row sample, BinMapper::FindBin, feature bundling — must reproduce the layout and
the bounds EXACTLY (float64 bounds compared bitwise).
GPU part: LGBMB200_BinnerTransform must reproduce every stored byte, from host and from device-resident input, and a tree
trained on the device-made matrix must equal the tree trained on the reference-made matrix."""
import glob
import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "binning_*.npz")))
RECORDED = os.path.join(ROOT, "tests", "golden", "reference")
META = (("feat_column", "feat_column"), ("feat_lo", "feat_lo"), ("feat_num_bin", "feat_num_bin"), ("feat_most_freq_bin", "feat_mfb"),
        ("feat_default_bin", "feat_default_bin"), ("feat_missing_type", "feat_missing"), ("feat_real_index", "feat_real_index"))


def _load(path):
    d = np.load(path)
    params = json.loads(bytes(d["params"]).decode())
    ub, o = [], 0
    for nb in d["feat_num_bin"]:
        ub.append(d["ub_concat"][o:o + nb]); o += nb
    return d, params, ub


def test_fixtures_present():
    assert len(GOLD) >= 11


@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[8:-4] for p in GOLD])
def test_fit_reproduces_reference_mappers_and_bundles(built_lib, path):
    import lightgbm_b200 as lgb
    d, params, ref_ub = _load(path)
    b = lgb.Binner(params).fit(d["X"])
    m = b.layout_meta()
    assert (m["num_data"], m["num_columns"], m["num_features"]) == tuple(int(v) for v in d["dims"][:3])
    for mine, ref in META:
        np.testing.assert_array_equal(m[mine], d[ref], err_msg=mine)
    ub = b.bin_upper_bounds()
    for f in range(m["num_features"]):
        assert ub[f].tobytes() == np.asarray(ref_ub[f], np.float64).tobytes(), f"bin upper bounds of inner feature {f}"


def test_row_sample_is_the_reference_generator(built_lib):
    """Random::Sample (utils/random.h:70-105), both branches, against the indices LGBM_SampleIndices of the compiled
    reference returned for seed 7, N=20000, K=3000 (tests/golden/reference/sample_indices.npz)."""
    import lightgbm_b200 as lgb
    X = np.zeros((20000, 1), np.float32); X[::2] = 1.0
    got = lgb.Binner(dict(bin_construct_sample_cnt=3000, data_random_seed=7)).fit(X).sample_indices()
    assert len(got) == 3000 and np.all(np.diff(got) > 0) and got[-1] < 20000
    np.testing.assert_array_equal(got, np.load(os.path.join(RECORDED, "sample_indices.npz"))["indices"])


def test_rejects_what_it_does_not_implement(built_lib):
    import lightgbm_b200 as lgb
    with pytest.raises(RuntimeError, match="max_bin"):
        lgb.Binner(dict(max_bin=1000)).fit(np.zeros((10, 2), np.float32))
    with pytest.raises(RuntimeError, match="more than one bin"):
        lgb.Binner({}).fit(np.ones((100, 3), np.float32))
    with pytest.raises(TypeError):
        lgb.Binner({}).fit(np.zeros((10, 2), np.int32))


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLD, ids=[os.path.basename(p)[8:-4] for p in GOLD])
def test_transform_reproduces_every_stored_byte(built_lib, path):
    import lightgbm_b200 as lgb
    from lightgbm_b200.tree_learner import DeviceArray
    d, params, _ = _load(path)
    X = np.ascontiguousarray(d["X"])
    b = lgb.Binner(params).fit(X)
    host_out, _ = b.transform(X, to_device=False)
    np.testing.assert_array_equal(host_out, d["bins"])
    dev_out, _ = b.transform(X, to_device=True)
    np.testing.assert_array_equal(dev_out.download(), d["bins"])
    dx = DeviceArray(X.nbytes).upload(X)                                   # input already in HBM
    dev2, ms = b.transform((dx, X.dtype), to_device=True, data_rows=X.shape[0])
    np.testing.assert_array_equal(dev2.download(), d["bins"])
    assert ms > 0


@pytest.mark.gpu
def test_tree_on_device_binned_matrix_equals_tree_on_reference_binned_matrix(built_lib):
    """raw floats -> Dataset (device pass, matrix stays in HBM) -> Train  ==  reference-made bins -> Train."""
    import lightgbm_b200 as lgb
    path = [p for p in GOLD if p.endswith("binning_efb_mixed_dense_sparse.npz")][0]
    d, params, ref_ub = _load(path)
    X = np.ascontiguousarray(d["X"])
    r = np.random.default_rng(5)
    y = (X[:, 0] + 0.1 * X[:, 5] - 0.2 * X[:, 9] + 0.3 * r.normal(size=len(X))).astype(np.float32)
    g = (float(y.mean()) - y).astype(np.float32); h = np.ones_like(g)
    ds = lgb.Dataset(X, label=y, params=params).construct()
    assert hasattr(ds.layout.bins, "ptr")                                  # never came back to the host
    L1 = lgb.B200TreeLearner(lgb.Config(num_leaves=31)); L1.init(ds.layout, is_constant_hessian=True)
    t1 = L1.train(g, h)
    ref_layout = lgb.Layout(np.ascontiguousarray(d["bins"]), *[np.ascontiguousarray(d[k], np.int32) for _, k in META], bin_upper_bound=ref_ub)
    L2 = lgb.B200TreeLearner(lgb.Config(num_leaves=31)); L2.init(ref_layout, is_constant_hessian=True)
    t2 = L2.train(g, h)
    assert t1.num_leaves == t2.num_leaves == 31
    assert t1.splits.tobytes() == t2.splits.tobytes()
    np.testing.assert_array_equal(t1.leaf_value, t2.leaf_value)


@pytest.mark.gpu
def test_full_size_properties_1m_x_256(built_lib):
    """At benchmark scale (C2-shaped float matrix) through properties the reference's definition gives: every value lies in
    (upper[bin - 1], upper[bin]] of its feature; the device result does not depend on chunking or on where the input lives."""
    import lightgbm_b200 as lgb
    r = np.random.default_rng(9)
    n, f = 1_000_000, 256
    X = r.normal(size=(n, f)).astype(np.float32)
    X[r.random(n) < 0.01, 3] = np.nan
    b = lgb.Binner(dict(min_data_in_bin=3)).fit(X)
    out, ms = b.transform(X, to_device=False)
    m = b.layout_meta(); ub = b.bin_upper_bounds()
    assert out.shape == (n, m["num_columns"])
    rows = r.choice(n, 20000, replace=False)
    for fi in range(0, m["num_features"], 7):
        col, lo, mfb, real = int(m["feat_column"][fi]), int(m["feat_lo"][fi]), int(m["feat_most_freq_bin"][fi]), int(m["feat_real_index"][fi])
        stored = out[rows, col].astype(np.int64)
        v = X[rows, real].astype(np.float64)
        bins = np.where(stored == 0, mfb, stored - lo + (1 if mfb == 0 else 0))       # one feature per column here
        nan = np.isnan(v)
        if nan.any():
            assert np.all(bins[nan] == m["feat_num_bin"][fi] - 1)
        u = ub[fi]
        ok = ~nan
        assert np.all(v[ok] <= u[bins[ok]])
        prev = np.where(bins[ok] > 0, u[np.maximum(bins[ok] - 1, 0)], -np.inf)
        assert np.all(v[ok] > prev)
    half, _ = b.transform(np.ascontiguousarray(X[: n // 2]), to_device=False)
    np.testing.assert_array_equal(half, out[: n // 2])
    print(f"1M x 256 float32 -> bins: {ms:.1f} ms device time incl. H2D/D2H ({n * f * 5 / ms / 1e6:.1f} GB/s)")


# ---------------------------------------------------------------------------------------------------- C4-shaped EFB at 200 K x 256
def _efb4():
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_golden
    d = np.load(os.path.join(ROOT, "tests", "golden", "efb4_200k_x256.npz"))
    _, raw, _, _, _ = make_golden.efb4_inputs()
    X = np.ascontiguousarray(raw, dtype=np.float32)
    params = dict(max_bin=255, min_data_in_bin=1, feature_pre_filter="false", enable_bundle="true")
    return d, X, params


def test_fit_reproduces_the_reference_bundles_of_the_c4_fixture(built_lib):
    """tests/golden/efb4_200k_x256.npz: the layout the UNMODIFIED reference built from the bench generator's C4-shaped data (256
    sparse features, exclusive in blocks of 4 -> 64 bundled columns, through LGBM_DatasetCreateFromSampledColumn + PushRows).
    The binner must arrive at the same 64 columns: same members, same order inside a column, same offsets."""
    import lightgbm_b200 as lgb
    d, X, params = _efb4()
    m = lgb.Binner(params).fit(X).layout_meta()
    assert (m["num_columns"], m["num_features"]) == (64, 256) == (int(d["dims"][1]), int(d["dims"][2]))
    for mine, ref in META:
        np.testing.assert_array_equal(m[mine], d[ref], err_msg=mine)


@pytest.mark.gpu
def test_transform_reproduces_the_reference_bytes_of_the_c4_fixture(built_lib):
    import lightgbm_b200 as lgb
    d, X, params = _efb4()
    bins = lgb.Binner(params).fit(X).transform(X, to_device=True)[0].download()
    cs = np.array([int(bins.astype(np.uint64).sum()), int((bins.astype(np.uint64) * (np.arange(bins.shape[1], dtype=np.uint64) + 1)).sum())], np.uint64)
    np.testing.assert_array_equal(cs, d["bins_checksum"])


def _sha1(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def random_small_case(seed):
    """Seeded random float matrix and Dataset parameters of test_random_small_shapes_against_the_live_reference."""
    r = np.random.default_rng(1000 + seed)
    n, f = int(r.integers(40, 3000)), int(r.integers(1, 71))
    X = r.normal(size=(n, f)).astype(np.float32 if seed % 2 == 0 else np.float64)
    for j in range(f):
        kind = r.integers(0, 5)
        if kind == 0:
            X[r.random(n) < 0.9, j] = 0.0
        elif kind == 1:
            X[:, j] = r.integers(-3, 4, n)
        elif kind == 2:
            X[r.random(n) < 0.2, j] = np.nan
        elif kind == 3:
            X[:, j] = np.where(r.random(n) < 0.97, 0.0, r.integers(1, 30, n))
    params = dict(max_bin=int(r.choice([15, 63, 255])), min_data_in_bin=int(r.choice([1, 3])), min_data_in_leaf=int(r.choice([1, 20])),
                  bin_construct_sample_cnt=int(r.choice([200000, max(20, n // 2)])), data_random_seed=int(r.integers(1, 100)),
                  feature_pre_filter="true", use_missing="true", zero_as_missing=str(bool(r.integers(0, 2))).lower(), enable_bundle="true")
    return X, params


@pytest.mark.gpu
def test_random_small_shapes_against_the_live_reference(built_lib):
    """Eight seeded random configurations (1 .. 70 columns, 40 .. 3000 rows, mixed dense / sparse / NaN / few-valued columns,
    random Dataset parameters) through the binner + device pass against what the compiled reference built from the same
    matrices (tests/golden/reference/binning_random_small.npz): same layout, same bounds, same bytes (SHA-1 of the
    reference's) — or the same refusal when no feature survives."""
    import lightgbm_b200 as lgb
    from oracle.refapi import Layout
    rec = np.load(os.path.join(RECORDED, "binning_random_small.npz"))
    checked = 0
    for seed in range(8):
        X, params = random_small_case(seed)
        assert _sha1(X) == str(rec[f"s{seed}_x_sha1"]), f"seed {seed}: not the recorded input"
        if not bool(rec[f"s{seed}_built"]):
            with pytest.raises(RuntimeError):
                lgb.Binner(params).fit(X)
            continue
        p = f"s{seed}_"
        ref = Layout.from_npz_dict({k[len(p):]: rec[k] for k in rec.files if k.startswith(p)})
        b = lgb.Binner(params).fit(X)
        m = b.layout_meta()
        assert (m["num_columns"], m["num_features"]) == (ref.num_columns, ref.num_features), seed
        for mine, theirs in META:
            np.testing.assert_array_equal(m[mine], getattr(ref, theirs), err_msg=f"seed {seed} {mine}")
        for fi, ub in enumerate(b.bin_upper_bounds()):
            assert ub.tobytes() == np.asarray(ref.bin_upper_bound[fi], np.float64).tobytes(), (seed, fi)
        out = b.transform(np.ascontiguousarray(X), to_device=False)[0]
        assert out.dtype == np.uint8 and out.shape == (X.shape[0], ref.num_columns)
        assert _sha1(out) == str(rec[f"s{seed}_bins_sha1"]), f"seed {seed}: stored bytes differ from the reference's"
        checked += 1
    assert checked >= 5
