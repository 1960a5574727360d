"""Model text writer / reader and device prediction (SURVEY.md §8 f-4) against the unmodified reference.

tests/golden/model_*.npz: model texts TRAINED AND WRITTEN by the reference, a test matrix (NaN, zeros, +-1e30 rows) and the
reference's own LGBM_BoosterPredictForMat results (tests/golden/make_model_golden.py).

CPU: reader -> writer reproduces the reference's text byte for byte (header keys, every tree block, feature importances);
     a text written by this repo loads in the reference and predicts the same.
GPU: raw scores from the device predictor are BIT-identical to the reference's; transformed outputs within 1e-15;
     float raw data -> device binning -> device boosting -> model text -> reference load -> reference predict agrees with
     this repo's predict bit for bit (the whole f-3 + path + f-4 chain through the reference's own reader).
What the compiled reference made of texts and matrices the tests generate is recorded under tests/golden/reference/
(tests/golden/make_reference_golden.py); where oracle/_ref is built, the texts written now are also loaded live."""
import glob
import hashlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "model_*.npz")))
IDS = [os.path.basename(p)[6:-4] for p in GOLD]
RECORDED = os.path.join(ROOT, "tests", "golden", "reference")


def _load(path):
    d = np.load(path)
    return bytes(d["model"]).decode(), d["X"], d["raw"], d["out"]


def test_fixtures_present():
    assert len(GOLD) >= 5


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_reader_then_writer_reproduces_the_reference_text(path):
    from lightgbm_b200.model import Model
    text, _, _, _ = _load(path)
    m = Model.from_string(text)
    mine = m.to_string()
    # everything up to and including the feature importances is byte-identical; the `parameters:` section is carried over
    ref_main = text.split("\nparameters:\n")[0]
    my_main = mine.split("\nparameters:\n")[0]
    assert my_main == ref_main
    assert m.parameters and m.parameters in text
    # and a second pass is a fixed point
    assert Model.from_string(mine).to_string() == mine


@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_written_text_loads_in_the_reference(path):
    """The text written for each fixture is the one the reference loaded and scored exactly as the fixture records (its
    SHA-1 is in tests/golden/reference/written_model_texts.npz); with oracle/_ref built, it is also loaded and scored live."""
    from lightgbm_b200.model import Model
    from oracle import refapi
    text, X, raw, out = _load(path)
    m = Model.from_string(text)
    m.parameters = ""                                   # a model of this repo carries no reference parameter dump
    m.feature_infos = []                                # nor bin ranges: "none" placeholders
    written = m.to_string()
    rec = np.load(os.path.join(RECORDED, "written_model_texts.npz"))
    assert hashlib.sha1(written.encode()).hexdigest() == str(rec[os.path.basename(path)[:-4]])
    if refapi.available():
        loaded = refapi.RefLoadedBooster(written)
        np.testing.assert_array_equal(loaded.predict(X, raw_score=True), raw)
        np.testing.assert_array_equal(loaded.predict(X, raw_score=False), out)
        loaded.free()


def test_tree_replay_matches_tree_split_bookkeeping():
    """ModelTree.from_learner_tree on a hand-made 3-leaf tree: children / parents / internal values as Tree::Split leaves them."""
    import lightgbm_b200 as lgb
    from lightgbm_b200.tree_learner import SPLIT_DTYPE
    sp = np.zeros(2, SPLIT_DTYPE)
    sp[0] = (0, 1, 3, 1, 60, 40, 12.5, 0, 60.0, -0.5, 0, 40.0, 0.75)
    sp[1] = (1, 0, 1, 0, 30, 10, 2.25, 0, 30.0, 0.25, 0, 10.0, 1.5)
    t = lgb.Tree(3, sp, np.array([-0.05, 0.025, 0.15]), np.array([60.0, 30.0, 10.0]), np.array([60, 30, 10], np.int32), np.array([1, 2, 2], np.int32), 0.0, 100.0)
    t.shrink = 0.1
    lay = lgb.Layout(np.zeros((1, 2), np.uint8), *[np.array(a, np.int32) for a in ([0, 1], [1, 1], [4, 6], [0, 0], [0, 0], [0, 2], [5, 7])],
                     bin_upper_bound=[np.array([0.5, 1.5, 2.5, np.inf]), np.array([-1.0, 0.0, 1.0, 2.0, np.inf, 2.0])])
    mt = lgb.ModelTree.from_learner_tree(t, lay, shrinkage=0.1)
    assert list(mt.split_feature) == [7, 5] and list(mt.threshold) == [2.0, 1.5]
    assert list(mt.decision_type) == [2 | (2 << 2), 0]                  # default-left + NaN missing; plain
    assert list(mt.left_child) == [-1, -2] and list(mt.right_child) == [1, -3]
    np.testing.assert_allclose(mt.internal_value, [0.0, 0.075]); assert list(mt.internal_count) == [100, 40]
    np.testing.assert_allclose(mt.internal_weight, [100.0, 40.0])
    s = mt.to_string()
    assert "split_gain=12.5 2.25\n" in s and "threshold=2 1.5\n" in s and "shrinkage=0.1\n" in s and s.endswith("\n\n")


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLD, ids=IDS)
def test_device_predict_is_bit_identical_to_the_reference(built_lib, path):
    from lightgbm_b200.model import Model
    text, X, raw, out = _load(path)
    m = Model.from_string(text)
    mine = m.predict_raw(X)
    assert mine.tobytes() == raw.tobytes()
    assert m.predict_raw(X.astype(np.float64)).tobytes() == raw.tobytes()
    np.testing.assert_allclose(m.predict(X), out, rtol=1e-15, atol=1e-15)
    # more rows than one chunk / one tile, ragged last tile
    big = np.tile(X, (40, 1))[:-7]
    assert m.predict_raw(big).tobytes() == np.tile(raw, 40)[:-7].tobytes()


def raw_float_data(objective):
    """Training matrix, labels and test matrix of test_raw_floats_to_model_text_to_reference_predict."""
    r = np.random.default_rng(3)
    n, f = 50_000, 20
    X = r.normal(size=(n, f)).astype(np.float32)
    X[r.random((n, f)) < 0.03] = np.nan
    X[:, 5] = np.where(r.random(n) < 0.7, 0.0, X[:, 5])
    s = np.nan_to_num(X[:, 0]) * 2 - np.nan_to_num(X[:, 3]) + np.sin(np.nan_to_num(X[:, 7]) * 2)
    y = (s + 0.2 * r.normal(size=n)).astype(np.float32) if objective == "regression" else (s > 0).astype(np.float32)
    Xt = r.normal(size=(5000, f)).astype(np.float32); Xt[r.random((5000, f)) < 0.05] = np.nan
    return X, y, Xt


@pytest.mark.gpu
@pytest.mark.parametrize("objective", ["regression", "binary"])
def test_raw_floats_to_model_text_to_reference_predict(built_lib, objective):
    """The reference's scores for the text this repo trained are recorded in tests/golden/reference/raw_floats_*.npz."""
    import lightgbm_b200 as lgb
    from oracle import refapi
    X, y, Xt = raw_float_data(objective)
    bst = lgb.train(dict(objective=objective, num_leaves=31, learning_rate=0.1, min_data_in_leaf=20), lgb.Dataset(X, label=y), num_boost_round=10)
    m = bst.to_model()
    text = m.to_string()
    mine = m.predict_raw(Xt)
    # the training scores the booster kept on the device are the model's predictions on the training matrix
    np.testing.assert_allclose(m.predict_raw(X), bst.scores(), rtol=1e-12, atol=1e-12)
    assert lgb.Model.from_string(text).predict_raw(Xt).tobytes() == mine.tobytes()
    rec = np.load(os.path.join(RECORDED, f"raw_floats_{objective}.npz"))
    assert rec["raw"].tobytes() == mine.tobytes()
    np.testing.assert_allclose(rec["out"], m.predict(Xt), rtol=1e-15, atol=1e-15)
    if refapi.available():
        loaded = refapi.RefLoadedBooster(text)
        assert loaded.num_iterations == 10
        assert loaded.predict(Xt, raw_score=True).tobytes() == mine.tobytes()
        np.testing.assert_allclose(loaded.predict(Xt, raw_score=False), m.predict(Xt), rtol=1e-15, atol=1e-15)
        loaded.free()


def single_leaf_data():
    """Rows and parameters on which the reference grows only single-leaf trees (no split satisfies min_data_in_leaf)."""
    r = np.random.default_rng(0)
    X = r.normal(size=(500, 4)).astype(np.float32); y = r.normal(size=500).astype(np.float32)
    return X, y, dict(objective="regression", num_leaves=7, min_data_in_leaf=400, verbosity=-1, num_threads=2)


def _single_leaf_model():
    """The model the reference wrote after 3 iterations on single_leaf_data(), those rows, and its raw scores for them
    (tests/golden/reference/single_leaf_model.npz)."""
    d = np.load(os.path.join(RECORDED, "single_leaf_model.npz"))
    X, _, _ = single_leaf_data()
    assert d["X"].tobytes() == X.tobytes()
    return bytes(d["model"]).decode(), X, d["raw"]


def test_single_leaf_tree_text_round_trips():
    from lightgbm_b200.model import Model
    text, _, _ = _single_leaf_model()
    m = Model.from_string(text)
    assert [t.num_leaves for t in m.trees] == [1]
    assert m.to_string().split("\nparameters:\n")[0] == text.split("\nparameters:\n")[0]


@pytest.mark.gpu
def test_single_leaf_tree_and_tiny_inputs_predict(built_lib):
    from lightgbm_b200.model import Model
    text, X, raw = _single_leaf_model()
    m = Model.from_string(text)
    for rows in (1, 2, 31, 33, 500):
        assert m.predict_raw(X[:rows]).tobytes() == raw[:rows].tobytes()
    # a real model on 1 .. 65 rows (less than one tile, exactly one, one more)
    d = np.load([p for p in GOLD if p.endswith("model_regression_missing_nan.npz")][0])
    m2 = Model.from_string(bytes(d["model"]).decode())
    for rows in (1, 7, 63, 64, 65):
        assert m2.predict_raw(d["X"][:rows]).tobytes() == d["raw"][:rows].tobytes()
