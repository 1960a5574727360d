"""Records, under tests/golden/reference/, what the tests that once called the compiled reference library at test time
compare against, so that they run from the repository alone.  Every fixture is produced by RUNNING THE UNMODIFIED
REFERENCE (oracle/_ref, built by oracle/Makefile.ref) on the inputs the test itself generates from its seeds.

  sample_indices.npz           test_binning.py::test_row_sample_is_the_reference_generator      LGBM_SampleIndices
  binning_random_small.npz     test_binning.py::test_random_small_shapes_against_the_live_reference
                               per seed: the reference Dataset's layout and bounds, the SHA-1 of its stored bytes (or
                               that it built none)
  written_model_texts.npz      test_model.py::test_written_text_loads_in_the_reference
                               SHA-1 of the texts this repo writes for tests/golden/model_*.npz, each of which the
                               reference loaded and scored exactly as the fixture records
  single_leaf_model.npz        test_model.py single-leaf tests: a text the reference wrote + its raw scores
  raw_floats_<objective>.npz   test_model.py::test_raw_floats_to_model_text_to_reference_predict: the model text this
                               repo trained (step `texts`, needs a GPU) and the reference's scores for it
  c4_dataset_70k_x64.npz       test_bench_helpers.py::test_c4_reference_dataset_bundles_like_the_generator: the layout
                               and the SHA-1 of the stored bytes
  c2_first_tree.npz            test_gpu_scale.py::test_c2_first_tree_matches_the_compiled_reference

Usage:  python tests/golden/make_reference_golden.py texts   (GPU machine: trains the raw_floats models)
        python tests/golden/make_reference_golden.py         (needs oracle/_ref: everything else)
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _save(name, **arrays):
    path = os.path.join(OUT, name)
    np.savez_compressed(path, **arrays)
    print(f"{name}: {os.path.getsize(path)} B")


def _text(a):
    return np.frombuffer(a.encode(), np.uint8)


def sha1(a):
    """digest that stands in for a large array or text in a fixture"""
    return np.array(hashlib.sha1(a.encode() if isinstance(a, str) else np.ascontiguousarray(a).tobytes()).hexdigest())


def sample_indices(refapi):
    import ctypes as C
    out = np.zeros(3000, np.int32); n = C.c_int32(0)
    refapi._check(refapi.lib().LGBM_SampleIndices(C.c_int32(20000), b"bin_construct_sample_cnt=3000 data_random_seed=7",
                                                   out.ctypes.data_as(C.c_void_p), C.byref(n)))
    assert n.value == 3000
    _save("sample_indices.npz", indices=out)


def binning_random_small(refapi):
    from test_binning import random_small_case
    d = {}
    for seed in range(8):
        X, params = random_small_case(seed)
        d[f"s{seed}_x_sha1"] = sha1(X)
        try:
            ds = refapi.RefDataset(X, None, dict(params, device_type="cuda", verbosity=-1))
        except RuntimeError:
            ds = None
        lay = ds.layout() if ds is not None else None
        if ds is not None:
            ds.free()
        built = lay is not None and lay.num_features > 0
        d[f"s{seed}_built"] = np.array(built)
        if built:
            d.update({f"s{seed}_{k}": v for k, v in lay.to_npz_dict(with_bins=False).items()})
            d[f"s{seed}_bins_sha1"] = sha1(lay.bins)
    _save("binning_random_small.npz", **d)


def written_model_texts(refapi):
    import glob
    from lightgbm_b200.model import Model
    d = {}
    for path in sorted(glob.glob(os.path.join(HERE, "model_*.npz"))):
        g = np.load(path)
        m = Model.from_string(bytes(g["model"]).decode())
        m.parameters = ""
        m.feature_infos = []
        text = m.to_string()
        loaded = refapi.RefLoadedBooster(text)
        assert loaded.predict(g["X"], raw_score=True).tobytes() == g["raw"].tobytes(), path
        assert loaded.predict(g["X"], raw_score=False).tobytes() == g["out"].tobytes(), path
        loaded.free()
        d[os.path.basename(path)[:-4]] = sha1(text)
    _save("written_model_texts.npz", **d)


def single_leaf_model(refapi):
    from test_model import single_leaf_data
    X, y, p = single_leaf_data()
    ds = refapi.RefDataset(X, y, p); b = refapi.RefBooster(ds, p)
    for _ in range(3):
        b.update()
    text = b.model_string()
    b.free(); ds.free()
    loaded = refapi.RefLoadedBooster(text)
    raw = loaded.predict(X, raw_score=True)
    for rows in (1, 2, 31, 33):
        assert loaded.predict(X[:rows], raw_score=True).tobytes() == raw[:rows].tobytes()
    loaded.free()
    _save("single_leaf_model.npz", model=_text(text), X=X, raw=raw)


def raw_floats_texts():
    import lightgbm_b200 as lgb
    from test_model import raw_float_data
    os.makedirs(OUT, exist_ok=True)
    for objective in ("regression", "binary"):
        X, y, Xt = raw_float_data(objective)
        bst = lgb.train(dict(objective=objective, num_leaves=31, learning_rate=0.1, min_data_in_leaf=20), lgb.Dataset(X, label=y),
                        num_boost_round=10)
        _save(f"raw_floats_{objective}.npz", model=_text(bst.to_model().to_string()))


def raw_floats_predict(refapi):
    from test_model import raw_float_data
    for objective in ("regression", "binary"):
        text = bytes(np.load(os.path.join(OUT, f"raw_floats_{objective}.npz"))["model"]).decode()
        _, _, Xt = raw_float_data(objective)
        loaded = refapi.RefLoadedBooster(text)
        assert loaded.num_iterations == 10
        raw, out = loaded.predict(Xt, raw_score=True), loaded.predict(Xt, raw_score=False)
        loaded.free()
        _save(f"raw_floats_{objective}.npz", model=_text(text), raw=raw, out=out)


def c4_dataset(refapi):
    import bench
    wl = dict(bench.WORKLOADS["C4"], rows=70000, cols=64)
    dsp, _ = bench._ref_params(wl, 2, "cpu")
    ds, _ = bench._ref_dataset(refapi, wl, wl["rows"], dsp, 2)
    lay = ds.layout()
    ds.free()
    _save("c4_dataset_70k_x64.npz", bins_sha1=sha1(lay.bins), **lay.to_npz_dict(with_bins=False))


def c2_first_tree(refapi):
    from test_gpu_scale import c2_reference_inputs
    bins, y, g, h, dsp, bp = c2_reference_inputs()
    ds = refapi.RefDatasetStreamed(lambda lo, hi: bins[lo:hi].astype(np.float32), len(bins), bins.shape[1], y, dsp, block_rows=262144)
    bst = refapi.RefBooster(ds, bp)
    bst.update_custom(g, h)
    t = bst.trees()[0]
    bst.free(); ds.free()
    _save("c2_first_tree.npz", num_leaves=np.int64(t.num_leaves), split_leaf=t.split_leaf(), split_feature=t.split_feature,
          threshold=t.threshold, internal_count=t.internal_count, leaf_count=t.leaf_count, split_gain=t.split_gain,
          leaf_value=t.leaf_value)


def main():
    if sys.argv[1:] == ["texts"]:
        raw_floats_texts()
        return
    from oracle import refapi
    os.makedirs(OUT, exist_ok=True)
    sample_indices(refapi)
    binning_random_small(refapi)
    written_model_texts(refapi)
    single_leaf_model(refapi)
    raw_floats_predict(refapi)
    c4_dataset(refapi)
    c2_first_tree(refapi)


if __name__ == "__main__":
    main()
