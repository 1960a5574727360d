"""GPU parity at BENCHMARK scale (VERDICT r1 item 2): the CUDA path against the oracle — and, for C2, against a tree
grown by the compiled reference itself — on the bench generator's own data, with the FULL split sequence compared.

  C2          : 1 000 000 x 256, 63 leaves  (bench.py --workload C2, seed 42)  vs oracle and vs the reference library
  C3-shaped   : 2 000 000 x 1024, 127 leaves (bench generator, seed 44)        vs oracle

Pass rule (helpers.compare_trees): every split equal to the oracle's (leaf, feature, threshold bin, default_left,
child counts exact; gains / sums / outputs within 1e-4 relative) unless the ORACLE's own best-vs-runner-up margin at the
first differing split is below 1e-5 relative; accepted divergences are printed and counted.
The oracle's histogram loop is threaded over columns for these sizes (bit-identical to its single-thread result)."""
import os
import sys
import time

import numpy as np
import pytest

from helpers import DIVERGENCES, compare_trees

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _workload(rows, cols, seed):
    import bench
    bins = bench.gen_bins(rows, cols, seed)
    y = bench.gen_label(rows, cols, seed, bins[:, :32])
    return bins, y


def _boost(lgb, orc, lay, y, leaves, iters, const_hess):
    """`iters` boosting iterations of L2 regression (lr 0.1) where every tree is grown by BOTH the CUDA path and the
    oracle from the same gradients; the score follows the ORACLE's tree so that a tolerated divergence cannot
    propagate into the next comparison.  Returns the number of splits compared."""
    n = lay.num_data
    L = lgb.B200TreeLearner(lgb.Config(num_leaves=leaves, min_data_in_leaf=20))
    L.init(lay, is_constant_hessian=const_hess)
    score = np.full(n, float(np.mean(y, dtype=np.float64)))
    h = np.ones(n, np.float32)
    total = 0
    for it in range(iters):
        g = (score - y).astype(np.float32)
        t0 = time.time()
        t = L.train(g, h)
        t1 = time.time()
        o = orc.train_tree(lay, g, h, num_leaves=leaves, min_data_in_leaf=20)
        t2 = time.time()
        matched, diverged = compare_trees(t, o, 1e-5)
        print(f"iter {it}: {matched}/{o.num_leaves - 1} splits identical, diverged={diverged}, "
              f"cuda {1e3 * (t1 - t0):.0f} ms, oracle {t2 - t1:.1f} s")
        assert diverged or matched == o.num_leaves - 1
        total += matched
        for leaf in range(o.num_leaves):
            rows = o.indices[o.leaf_begin[leaf]:o.leaf_begin[leaf] + o.leaf_count[leaf]]
            score[rows] += 0.1 * o.leaf_value[leaf]
    return total


@pytest.mark.parametrize("const_hess", [True, False])
def test_c2_full_split_sequence_matches_oracle(built_lib, const_hess):
    import lightgbm_b200 as lgb
    from oracle import oracle_py
    bins, y = _workload(1_000_000, 256, 42)
    lay = lgb.Layout.identity(bins)
    before = len(DIVERGENCES)
    total = _boost(lgb, oracle_py, lay, y, leaves=63, iters=2, const_hess=const_hess)
    print(f"C2 const_hess={const_hess}: {total} splits compared, {len(DIVERGENCES) - before} accepted near-tie divergences")
    assert total >= 62


def c2_reference_inputs():
    """C2 bins, labels, first-iteration gradients, and the reference Dataset / Booster parameters of
    test_c2_first_tree_matches_the_compiled_reference."""
    rows, cols, leaves = 1_000_000, 256, 63
    bins, y = _workload(rows, cols, 42)
    dsp = dict(max_bin=255, min_data_in_bin=1, enable_bundle="false", feature_pre_filter="false", verbosity=-1,
               num_threads=min(32, os.cpu_count() or 8))
    bp = dict(dsp, objective="custom", num_leaves=leaves, min_data_in_leaf=20, learning_rate=1.0, device_type="cpu",
              force_col_wise="true", deterministic="true")
    g = (float(np.mean(y, dtype=np.float64)) - y).astype(np.float32)
    h = np.ones(rows, np.float32)
    return bins, y, g, h, dsp, bp


def test_c2_first_tree_matches_the_compiled_reference(built_lib):
    """The same C2 matrix through the UNMODIFIED reference library (oracle/_ref, LGBM_BoosterUpdateOneIterCustom with the
    same gradients, serial col-wise deterministic CPU learner; its tree is recorded in tests/golden/reference/c2_first_tree.npz)
    and through the CUDA path: same split features, same real-valued thresholds (bin upper bounds), same child counts, for
    every split of the first tree."""
    import lightgbm_b200 as lgb
    bins, y, g, h, _, bp = c2_reference_inputs()
    leaves = bp["num_leaves"]
    ref = np.load(os.path.join(ROOT, "tests", "golden", "reference", "c2_first_tree.npz"))

    L = lgb.B200TreeLearner(lgb.Config(num_leaves=leaves, min_data_in_leaf=20))
    L.init(lgb.Layout.identity(bins), is_constant_hessian=True)
    t = L.train(g, h)
    assert t.num_leaves == int(ref["num_leaves"]) == leaves
    np.testing.assert_array_equal(t.splits["leaf"], ref["split_leaf"])
    np.testing.assert_array_equal(t.splits["feature"], ref["split_feature"])
    # identity bins: value v has bin v, bin upper bound = v + 0.5 (bin.cpp: midpoints of consecutive distinct values)
    np.testing.assert_allclose(ref["threshold"], t.splits["threshold"] + 0.5, atol=1e-6)
    np.testing.assert_array_equal(t.splits["left_count"] + t.splits["right_count"], ref["internal_count"])
    np.testing.assert_array_equal(t.leaf_count, ref["leaf_count"])
    np.testing.assert_allclose(t.splits["gain"], ref["split_gain"], rtol=2e-5)     # the model text stores float32 gains
    np.testing.assert_allclose(t.leaf_value, ref["leaf_value"], rtol=1e-6, atol=1e-9)


def test_c3_shaped_2m_x_1024_matches_oracle(built_lib):
    import lightgbm_b200 as lgb
    from oracle import oracle_py
    bins, y = _workload(2_000_000, 1024, 44)
    lay = lgb.Layout.identity(bins)
    before = len(DIVERGENCES)
    total = _boost(lgb, oracle_py, lay, y, leaves=127, iters=1, const_hess=True)
    print(f"2M x 1024: {total} splits compared, {len(DIVERGENCES) - before} accepted near-tie divergences")
    assert total >= 100
