"""CPU-only tests: the host logic above the C ABI, the API contract of the reference, the shared
library's exports, and the oracle's forest evaluator against scikit-learn."""
import ctypes
import os
import re

import numpy as np
import pandas as pd
import pytest

import parity_utils  # noqa: F401  (sys.path)
from conftest import GOLDEN, ROOT


# ------------------------------------------------------------------ C ABI
def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "b200repair.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(dr_[a-z0-9_]+)\s*\(", hdr)))


def test_library_exports_every_declared_symbol():
    from repair import _native
    lib = _native.load_library()
    declared = _declared_symbols()
    assert len(declared) >= 30
    for sym in declared:
        assert hasattr(lib, sym), "missing export: " + sym
    assert sorted(_native.EXPORTED_SYMBOLS) == declared
    assert lib.dr_abi_version() == 4
    raw = ctypes.CDLL(_native.LIB_PATH)
    for sym in declared:
        getattr(raw, sym)


def test_engine_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from repair import RepairModel
    from repair._native import NativeError
    df = pd.read_csv(os.path.join(GOLDEN, "adult.csv"))
    with pytest.raises(NativeError, match="no CPU fallback"):
        RepairModel().setInput(df).setRowId("tid").run()


# ------------------------------------------------------------------ API contract (tests/test_model.py:98-317)
def test_invalid_params():
    from repair import RepairModel
    from repair.costs import Levenshtein
    df = pd.read_csv(os.path.join(GOLDEN, "adult.csv"))
    msg = "`setInput` and `setRowId` should be called before repairing"
    for f in (lambda: RepairModel().run(), lambda: RepairModel().setTableName("dummyTab").run(),
              lambda: RepairModel().setInput("dummyTab").run()):
        with pytest.raises(ValueError, match=msg):
            f()
    with pytest.raises(ValueError, match="Can not specify a database name when input is `DataFrame`"):
        RepairModel().setInput(df).setDbName("default")
    with pytest.raises(ValueError, match="`setRepairDelta` should be called when enabling maximal likelihood"):
        RepairModel().setTableName("dummyTab").setRowId("dummyId").run(maximal_likelihood_repair=True)
    with pytest.raises(ValueError, match="`setUpdateCostFunction` should be called when enabling maximal"):
        RepairModel().setInput("dummyTab").setRowId("dummyId").setRepairDelta(3).run(maximal_likelihood_repair=True)
    with pytest.raises(ValueError, match="`UpdateCostFunction.targets` cannot be used when enabling maximal"):
        RepairModel().setInput("dummyTab").setRowId("dummyId").setRepairDelta(3) \
            .setUpdateCostFunction(Levenshtein(targets=["non-existent"])).run(maximal_likelihood_repair=True)
    with pytest.raises(ValueError, match="`attrs` should have at least one attribute"):
        RepairModel().setTargets([])
    with pytest.raises(ValueError, match="`thres` should be bigger than 1, got 0"):
        RepairModel().setDiscreteThreshold(0)
    with pytest.raises(ValueError, match="`table_name` should have at least character"):
        RepairModel().setTableName("")
    with pytest.raises(ValueError, match="`table_name` should have at least character"):
        RepairModel().setInput("")
    with pytest.raises(ValueError, match="`row_id` should have at least character"):
        RepairModel().setRowId("")
    with pytest.raises(ValueError, match="Repair delta should be positive, got -1"):
        RepairModel().setRepairDelta(-1)
    with pytest.raises(ValueError, match="`error_cells` should have at least character"):
        RepairModel().setErrorCells("")
    with pytest.raises(ValueError, match="`setRowId` should be called before specifying error cells"):
        RepairModel().setErrorCells(df)
    with pytest.raises(ValueError, match="Error cells should have `tid` and `attribute` in columns"):
        RepairModel().setInput(df).setRowId("tid").setErrorCells(df)


def test_exclusive_params():
    from repair import RepairModel
    api = RepairModel().setTableName("dummyTab").setRowId("dummyId")
    for kw in ({"detect_errors_only": True, "compute_repair_candidate_prob": True},
               {"detect_errors_only": True, "repair_data": True},
               {"compute_repair_candidate_prob": True, "repair_data": True},
               {"compute_repair_candidate_prob": True, "compute_repair_prob": True},
               {"compute_repair_candidate_prob": True, "compute_repair_score": True}):
        with pytest.raises(ValueError, match="cannot be set to true simultaneously"):
            api.run(**kw)


def test_argtype_check():
    from repair import RepairModel
    cases = [
        (lambda: RepairModel().setDbName(1), "`db_name` should be provided as str, got int"),
        (lambda: RepairModel().setTableName(1), "`table_name` should be provided as str, got int"),
        (lambda: RepairModel().setDiscreteThreshold("a"), "`thres` should be provided as int, got str"),
        (lambda: RepairModel().setInput(1), "`input` should be provided as str/DataFrame, got int"),
        (lambda: RepairModel().setTargets(1), "`attrs` should be provided as list[str], got int"),
        (lambda: RepairModel().setTargets(["a", 1]), "`attrs` should be provided as list[str], got int in elements"),
        (lambda: RepairModel().setErrorDetectors(1), "`detectors` should be provided as list[ErrorDetector], got int"),
        (lambda: RepairModel().setErrorDetectors([1]),
         "`detectors` should be provided as list[ErrorDetector], got int in elements"),
        (lambda: RepairModel().setUpdateCostFunction(1), "`cf` should be provided as UpdateCostFunction, got int"),
        (lambda: RepairModel().setUpdateCostFunction([1]), "`cf` should be provided as UpdateCostFunction, got list"),
    ]
    for f, msg in cases:
        with pytest.raises(TypeError, match=re.escape(msg)):
            f()


def test_options():
    from repair import RepairModel
    with pytest.raises(ValueError, match="Non-existent key specified: key=non-existent"):
        RepairModel().option("non-existent", "1")
    keys = [("error.domain_threshold_alpha", "0.0"), ("error.domain_threshold_beta", "0.7"),
            ("error.max_attrs_to_compute_pairwise_stats", "3"), ("error.max_attrs_to_compute_domains", "2"),
            ("error.attr_freq_ratio_threshold", "0.0"), ("error.pairwise_freq_ratio_threshold", "0.05"),
            ("model.max_training_row_num", "100000"), ("model.max_training_column_num", "65536"),
            ("model.small_domain_threshold", "12"), ("model.rule.repair_by_nearest_values.disabled", "1"),
            ("model.rule.merge_threshold", "2.0"), ("model.rule.repair_by_regex.disabled", ""),
            ("model.rule.repair_by_functional_deps.disabled", ""), ("model.rule.max_domain_size", "1000"),
            ("repair.pmf.cost_weight", "0.1"), ("repair.pmf.prob_threshold", "0.0"), ("repair.pmf.prob_top_k", "80"),
            ("model.lgb.boosting_type", "gbdt"), ("model.lgb.class_weight", "balanced"),
            ("model.lgb.learning_rate", "0.01"), ("model.lgb.max_depth", "7"), ("model.lgb.max_bin", "255"),
            ("model.lgb.reg_alpha", "0.0"), ("model.lgb.min_split_gain", "0.0"), ("model.lgb.n_estimators", "300"),
            ("model.lgb.importance_type", "gain"), ("model.cv.n_splits", "3"), ("model.hp.timeout", "0"),
            ("model.hp.max_evals", "10000000"), ("model.hp.no_progress_loss", "50")]
    for k, v in keys:
        RepairModel().option(k, v)


def test_option_value_parsing(monkeypatch):
    from repair.utils import get_option_value
    assert get_option_value({}, "k", 3, int) == 3
    assert get_option_value({"k": "5"}, "k", 3, int, lambda v: v >= 2, "`{}` should be greater than 1") == 5
    monkeypatch.delenv("SPARK_TESTING", raising=False)
    assert get_option_value({"k": "x"}, "k", 3, int) == 3                       # warn + default
    assert get_option_value({"k": "1"}, "k", 3, int, lambda v: v >= 2, "`{}` bad") == 3
    monkeypatch.setenv("SPARK_TESTING", "1")
    with pytest.raises(ValueError, match='Failed to cast "invalid" into float data: key=error.attr_freq'):
        get_option_value({"error.attr_freq": "invalid"}, "error.attr_freq", 0.0, float)
    with pytest.raises(ValueError, match="`k` should be greater than 1, got 1"):
        get_option_value({"k": "1"}, "k", 3, int, lambda v: v >= 2, "`{}` should be greater than 1")
    assert get_option_value({"b": ""}, "b", True, bool) is False  # bool("") is False (test_model.py:248)


def test_detector_constructors_and_strings():
    from repair.errors import (ConstraintErrorDetector, DomainValues, GaussianOutlierErrorDetector,
                               NullErrorDetector, RegExErrorDetector)
    assert str(NullErrorDetector()) == "NullErrorDetector()"
    assert str(DomainValues("a", ["x"], False, 3)) == 'DomainValues(attr="a",size=1,autofill=False,min_count_thres=3)'
    assert DomainValues("a", ["x"], autofill=True).values == []
    assert str(RegExErrorDetector("a", "b.*")) == 'RegExErrorDetector(pattern="b.*")'
    assert str(GaussianOutlierErrorDetector(True)) == "GaussianOutlierErrorDetector(approx_enabled=True)"
    with pytest.raises(ValueError, match="At least one of `constraint_path` or `constraints` should be specified"):
        ConstraintErrorDetector()
    d = ConstraintErrorDetector(constraints="X->Y", targets=["Y"]).setUp("tid", "t", [], ["X", "Y", "Z"])
    assert d._targets == ["Y"]
    d = NullErrorDetector().setUp("tid", "t", [], ["X", "Y"])
    assert d._targets == ["X", "Y"]


# ------------------------------------------------------------------ host logic vs oracle
def test_constraint_parser_matches_oracle():
    from oracle import detect as OD
    from repair import constraints as PC
    stmts = ['t1&EQ(t1.v1,"abc")&EQ(t1.v2,"def")', "t1&t2&EQ(t1.v1,t2.v1)&IQ(t1.v2,t2.v2)",
             "t1&t2&LT(t1.v1,t2.v1)&GT(t1.v2,t2.v2)&EQ(t1.v1,t2.v1)", ' t1 & EQ ( t1.v1 , "abc") & EQ ( t1.v2 , "def" ) ',
             "X->Y", "v1 -> v2", 'EQ(t1.v1,"abc")', "t1&", "t1", "a&b&", "k1&k2", "X=>Y", "", 't1&EQ(t1.v1,"abc")',
             't1&t2&GT(t3.v0,"abc")&EQ(t1.v1,t2.v1)&IQ(t1.v2,t2.v2)']
    for s in stmts:
        try:
            try:
                want = OD.parse(s)
            except Exception:
                want = OD.parse_alt(s)
            want = [(p.sign, p.left, p.right, p.right_kind == "attr") for p in want]
        except Exception:
            want = "error"
        try:
            try:
                got = PC.parse_denial_constraint(s)
            except Exception:
                got = PC.parse_fd_sugar(s)
            got = [tuple(p) for p in got]
        except Exception:
            got = "error"
        assert got == want, s
    lines = PC.load_statements(os.path.join(GOLDEN, "hospital_constraints.txt"), "A->B;;C->D")
    assert len(lines) == 17
    preds = PC.parse_and_verify(lines, ["tid", "HospitalName", "ZipCode", "A", "B"])
    assert len(preds) == 2
    assert PC.classify(preds[0])[0] == "FD" and PC.classify(preds[1]) == ("FD", (["A"], "B"))
    assert PC.classify(PC.parse_denial_constraint('t1&EQ(t1.Sex,"Female")&EQ(t1.Relationship,"Husband")'))[0] == "CONST"
    assert PC.classify(PC.parse_denial_constraint("t1&t2&EQ(t1.a,t2.a)&EQ(t1.b,t2.b)"))[0] == "EQ_ONLY"
    assert PC.classify(PC.parse_denial_constraint("t1&t2&EQ(t1.a,t2.a)&LT(t1.b,t2.b)")) == ("INEQ", (["a"], "LT", "b"))
    assert PC.classify(PC.parse_denial_constraint("t1&t2&GT(t1.b,t2.b)&EQ(t1.g,t2.g)")) == ("INEQ", (["g"], "GT", "b"))
    assert PC.classify(PC.parse_denial_constraint("t1&t2&LT(t1.a,t2.a)&GT(t1.b,t2.b)"))[0] == "OTHER"
    assert PC.classify(PC.parse_denial_constraint("t1&t2&EQ(t1.a,t2.a)&LT(t1.b,t2.c)"))[0] == "OTHER"
    assert PC.classify(PC.parse_denial_constraint("t1&t2&EQ(t1.a,t2.b)&IQ(t1.c,t2.c)"))[0] == "OTHER"


def _counts(codes_x, dx, codes_y=None, dy=None):
    if codes_y is None:
        return np.bincount(codes_x.astype(np.int64) + 1, minlength=dx + 1)
    idx = (codes_x.astype(np.int64) + 1) * (dy + 1) + codes_y + 1
    return np.bincount(idx, minlength=(dx + 1) * (dy + 1)).reshape(dx + 1, dy + 1)


@pytest.mark.parametrize("having_thr", [0.0, 0.02])
def test_entropies_and_pair_selection_match_oracle(having_thr):
    from oracle import stats as OS
    from oracle.table import OTable
    from repair import stats_host as SH
    rng = np.random.default_rng(3)
    n, doms = 4000, [3, 5, 8, 4, 6]
    cols = [rng.integers(0, d, size=n) for d in doms]
    cols[1] = (cols[2] * 3 % 5)
    for c in cols:
        c[rng.random(n) < 0.04] = -1
    names = ["a", "b", "c", "d", "e"]
    otbl = OTable(["tid"] + names, ["int"] + ["str"] * 5, [np.arange(n, dtype=np.float64)] + cols)
    ndv = {nm: len(np.unique(c[c >= 0])) for nm, c in zip(names, cols)}
    targets = ["b", "d"]
    fs, want_stats, want_pairs = OS.compute_attr_stats(otbl, "tid", targets, ndv, having_thr, 1.0, 2)
    # product host logic on dense counts
    hist = {nm: _counts(c, d) for nm, c, d in zip(names, cols, doms)}
    cands = SH.candidate_pairs(targets, names)
    col_of = dict(zip(names, zip(cols, doms)))
    nnz = {frozenset(p): int(np.count_nonzero(_counts(col_of[p[0]][0], col_of[p[0]][1], col_of[p[1]][0], col_of[p[1]][1])))
           for t in targets for p in cands[t]}
    pairs = [p for t in targets for p in SH.select_scored(cands[t], nnz, ndv, 1.0, 2)]
    assert pairs == want_pairs
    tables = {p: _counts(col_of[p[0]][0], col_of[p[0]][1], col_of[p[1]][0], col_of[p[1]][1]) for p in pairs}
    got = SH.pairwise_entropies(n, hist, tables, pairs, ndv, SH.having_threshold(n, having_thr))
    assert set(got) == {k for k, v in want_stats.items() if v}
    for t in got:
        assert [a for a, _ in got[t]] == [a for a, _ in want_stats[t]]
        for (_, h1), (_, h2) in zip(got[t], want_stats[t]):
            assert abs(h1 - h2) < 1e-12
    # lower bounds only ever exclude what the exact counts exclude
    lower = {k: max(1, v // 2) for k, v in nnz.items()}
    for t in targets:
        und = SH.undecided(cands[t], lower, ndv, 0.9)
        assert set(SH.select_scored(cands[t], nnz, ndv, 0.9, 2)) <= set(und)


def test_tau_and_discretize_params_match_oracle():
    from oracle import stats as OS
    from repair import stats_host as SH
    assert SH.tau_for(0.5, 1000, 7, 9) == int(0.5 * (1000 // 63))
    for kind, lo, hi in (("float", 0.00632, 88.9762), ("float", 1e-5, 3.5), ("int", 0, 711), ("float", 0.5, 3.2),
                         ("float", 187.0, 2.5e7)):
        assert SH.discretize_params(kind, lo, hi) == OS.discretize_params(kind, lo, hi)


def test_double_to_string_matches_oracle():
    from oracle.table import spark_double_to_string
    from repair.utils import double_to_string
    rng = np.random.default_rng(0)
    vals = [1.0, 3.2, 0.5, 1000.0, 1e7, 1.5e7, 0.001, 0.0001, 123456.789, -2.5e-5, 9999999.0, 0.0, -0.0, 1e-3, 1e22,
            5e-324, 1.7976931348623157e308] + list(rng.normal(size=200) * 10.0 ** rng.integers(-8, 12, size=200))
    for v in vals:
        assert double_to_string(v) == spark_double_to_string(v), v
    assert double_to_string(1e7) == "1.0E7" and double_to_string(0.0001) == "1.0E-4" and double_to_string(100.0) == "100.0"


def test_encoders_match_oracle():
    from oracle.forest import encode_rows
    from repair.forest import encode_matrix, first_seen
    rng = np.random.default_rng(1)
    n = 300
    dict_size = {"s": 4, "o": 15}
    train = {"s": rng.integers(-1, 4, size=n), "o": rng.integers(-1, 12, size=n)}     # codes, -1 = NULL
    train["s"][train["s"] == 2] = 1                                                 # value 2 unseen in training
    test = {"s": rng.integers(-1, 4, size=n), "o": rng.integers(-1, 15, size=n)}
    vals = {"x": np.where(rng.random(n) < 0.1, np.nan, rng.normal(size=n))}
    for null_in_training in (True, False):
        tr = {k: (v if null_in_training else np.where(v < 0, 0, v)) for k, v in train.items()}
        p_enc = [{"attr": "s", "type": "sum", "categories": first_seen(tr["s"])},
                 {"attr": "x", "type": "cont"},
                 {"attr": "o", "type": "ordinal", "categories": first_seen(tr["o"])}]
        o_enc = [dict(e, categories=[None if c < 0 else int(c) for c in e["categories"]]) if "categories" in e else e
                 for e in p_enc]
        got = encode_matrix(p_enc, test, vals, dict_size)
        cols = {"s": [None if c < 0 else int(c) for c in test["s"]], "o": [None if c < 0 else int(c) for c in test["o"]],
                "x": [None if v != v else float(v) for v in vals["x"]]}
        want = encode_rows(o_enc, cols)
        assert got.shape == want.shape
        assert np.all((got == want) | (np.isnan(got) & np.isnan(want)))


def test_select_features_matches_oracle():
    from oracle.repair import select_features as o_sel
    from repair.model import select_features as p_sel
    stats = {"y": [("a", -0.1), ("b", 0.3), ("c", 0.0), ("d", 0.7)]}
    feats = ["a", "b", "c", "d", "e"]
    for m in (2, 3, 4, 10):
        assert p_sel(stats, "y", feats, m) == o_sel(stats, "y", feats, m)
    assert p_sel({}, "y", feats, 2) == feats


# ------------------------------------------------------------------ forest: oracle vs scikit-learn
@pytest.mark.parametrize("kind", ["binary", "multiclass", "regression"])
def test_oracle_forest_matches_sklearn(kind):
    """Pins the oracle's flat-forest evaluator to an independent implementation: margins are
    bit-identical to HistGradientBoosting's own raw predictions, labels to its predict()."""
    from oracle.forest import forest_margins, forest_predict, forest_proba
    from repair.train import build_model
    rng = np.random.default_rng(0)
    n = 1500
    X = rng.integers(0, 6, size=(n, 7)).astype(float)
    X[rng.random(X.shape) < 0.08] = np.nan
    base = np.nan_to_num(X[:, 0]) + np.nan_to_num(X[:, 3]) * 2
    opts = {"model.lgb.n_estimators": "40", "model.lgb.learning_rate": "0.1", "model.hp.max_evals": "1"}
    from sklearn.ensemble import HistGradientBoostingClassifier, HistGradientBoostingRegressor
    common = dict(learning_rate=0.1, max_iter=40, max_depth=7, max_leaf_nodes=31, min_samples_leaf=20, max_bins=255,
                  l2_regularization=0.0, early_stopping=False, random_state=42)
    Xt = rng.integers(-1, 7, size=(500, 7)).astype(float)
    Xt[Xt < 0] = np.nan
    if kind == "regression":
        y = base + rng.normal(size=n)
        forest, classes = build_model(X, y, False, 0, opts)
        est = HistGradientBoostingRegressor(**common).fit(X, y)
        assert classes is None
        assert np.array_equal(forest_predict(forest, Xt), est.predict(Xt))
        return
    y = (base.astype(int) % (2 if kind == "binary" else 5))
    forest, classes = build_model(X, y, True, len(set(y)), opts)
    est = HistGradientBoostingClassifier(class_weight="balanced", **common).fit(X, y)
    assert classes == sorted(set(y.tolist()))
    raw = est._raw_predict(Xt)
    assert np.array_equal(forest_margins(forest, Xt), raw)
    pred = np.asarray(classes)[forest_predict(forest, Xt)]
    assert np.array_equal(pred, est.predict(Xt))
    assert np.allclose(forest_proba(forest, Xt), est.predict_proba(Xt), atol=1e-12)


def test_pack_nodes_roundtrip():
    from repair.forest import LEAF, pack_nodes
    from tools.randforest import random_forest
    rng = np.random.default_rng(0)
    f = random_forest(10, 3, 5, [[0.5, 1.5]] * 10, rng)
    thr, meta = pack_nodes(f)
    leaf = f["feature"] < 0
    assert np.array_equal((meta & 0xFFF) == LEAF, leaf)
    assert np.array_equal((meta & 0xFFF)[~leaf], f["feature"][~leaf])
    assert np.array_equal(((meta >> 13) & 0x1FF)[~leaf], f["left"][~leaf])
    assert np.array_equal(((meta >> 22) & 0x1FF)[~leaf], f["right"][~leaf])
    assert np.array_equal(((meta >> 12) & 1), f["missing_left"])
    assert np.array_equal(thr[leaf], f["value"][leaf]) and np.array_equal(thr[~leaf], f["threshold"][~leaf])
    sizes = np.diff(f["tree_offset"])
    assert sizes.max() <= 61 and len(sizes) == 15


# ------------------------------------------------------------------ ingest + synthetic data
def test_ingest_encoding():
    from repair.table import EncodedTable
    from repair.utils import AnalysisException
    df = pd.DataFrame({"tid": [10, 11, 12, 13], "s": ["b", None, "a", "b"], "i": [3, 1, None, 3],
                       "f": [0.5, None, 2.5, 0.5]})
    t = EncodedTable.from_pandas(df, "tid")
    assert t.names == ["s", "i", "f"] and t.continuous_attrs == ["i", "f"]
    s, i, f = t.columns
    assert list(s.dictionary) == ["a", "b"] and s.codes.tolist() == [1, -1, 0, 1]
    assert i.kind == "float" and i.codes.tolist() == [1, 0, -1, 1]  # pandas float column (NULL present)
    assert f.strings() == ["0.5", "2.5"] and f.decode([1, -1]) == ["2.5", None]
    assert s.code_of("b") == 1 and s.code_of("zz") == -2 and s.rank_bounds("aa") == (1, 1)
    df["b"] = [True, False, True, False]
    with pytest.raises(AnalysisException, match="unsupported ones found: boolean"):
        EncodedTable.from_pandas(df, "tid")
    sh = t.shard(1, 2)
    assert sh.n_rows == 2 and sh.row_offset == 2 and sh.n_rows_global == 4 and sh.columns[0].codes.tolist() == [0, 1]


def test_synthetic_generator_is_shardable_and_deterministic():
    import torch
    from repair import synth
    spec = synth.SynthSpec.c4(50000, 16, seed=3)
    full = synth.generate_numpy(spec)
    part = synth.generate_numpy(spec, 12345, 23456)
    assert all(np.array_equal(part[i], full[i][12345:23456]) for i in range(16))
    t = synth.generate_torch(spec, "cpu", 1000, 9000, chunk=3000)
    assert all(np.array_equal(t[i, :8000].numpy(), full[i][1000:9000]) for i in range(16))
    assert all(full[i].max() < spec.dom[i] and full[i].min() >= -1 for i in range(16))
    assert all((full[i] < 0).sum() == 0 for i in (4, 5, 12, 13)) and (full[0] < 0).mean() > 0.005
    dep, det = full[4], full[5]
    clean = det < spec.dom[5] - 3
    assert all(len(set(dep[(det == v)].tolist())) == 1 for v in np.unique(det[clean]))
    assert any(len(set(dep[(det == v)].tolist())) > 1 for v in range(spec.dom[5] - 3, spec.dom[5]))


def _image_margins(spec, dict_sizes, codes):
    from ranked_emul import eval_image
    from repair.forest import group_by_sequence, rank_code, ranked_image
    rk = rank_code(spec, dict_sizes)
    off, order = group_by_sequence(spec["forest"])
    img = ranked_image(rk, order, off)
    return rk, img, off, order, eval_image(rk, img, spec["forest"]["baseline"], codes)


def test_rank_coded_forest_makes_the_same_decisions():
    from oracle.forest import forest_margins
    from repair.forest import encode_matrix, encoder_width, rank_code
    from tools.randforest import random_forest
    rng = np.random.default_rng(4)
    dict_sizes = {"a": 5, "b": 14, "c": 3}
    encoders = [{"attr": "a", "type": "sum", "categories": [2, -1, 0, 4]},
                {"attr": "b", "type": "ordinal", "categories": list(range(13))},
                {"attr": "c", "type": "sum", "categories": [1, 0, 2]}]
    n_feat = sum(encoder_width(e) for e in encoders)
    thr = [[-1.5, -0.5, 0.5, 1.5]] * 3 + [[-3.0, -1.0, 0.5, 3.5, 7.5, 12.5, 20.0]] + [[-0.5, 0.5]] * 2
    forest = random_forest(n_feat, 3, 6, thr, rng, leaf_scale=0.2)
    spec = {"forest": forest, "encoders": encoders, "class_codes": [0, 1, 2]}
    n = 200
    codes = {a: rng.integers(-1, d + 1, size=n) for a, d in dict_sizes.items()}   # d = "unknown category"
    rk, img, _, _, got = _image_margins(spec, dict_sizes, codes)
    assert rk is not None and rk["max_depth"] <= 7 and 1 <= rk["n_slots"] <= 2 * n_feat
    inr = {a: np.where(codes[a] < dict_sizes[a], codes[a], 0) for a in codes}
    X = encode_matrix(encoders, inr, {}, dict_sizes)
    j = 0
    for e in encoders:  # a code outside the dictionary encodes to NaN in every column of its encoder
        w = encoder_width(e)
        X[codes[e["attr"]] >= dict_sizes[e["attr"]], j:j + w] = np.nan
        j += w
    assert np.array_equal(got, forest_margins(forest, X))
    spec["encoders"] = encoders + [{"attr": "x", "type": "cont"}]
    assert rank_code(spec, dict_sizes) is None  # continuous feature -> generic kernel


def test_rank_slots_only_for_tested_feature_directions():
    """One slot per (feature, NaN direction) that a node tests; a forest whose nodes all send NaN the
    same way needs one slot per tested feature."""
    from oracle.forest import forest_margins
    from repair.forest import encode_matrix, rank_code
    from tools.randforest import random_forest
    rng = np.random.default_rng(11)
    dict_sizes = {"a": 9, "b": 30}
    encoders = [{"attr": "a", "type": "sum", "categories": list(range(9))},
                {"attr": "b", "type": "ordinal", "categories": list(range(28))}]   # codes 28, 29 unseen -> NaN
    thr = [[-0.5, 0.5]] * 8 + [[j + 0.5 for j in range(1, 28)]]
    forest = random_forest(9, 4, 10, thr, rng)
    forest["missing_left"][:] = 0
    forest["feature"] = np.where(forest["feature"] == 3, 4, forest["feature"]).astype(np.int32)  # feature 3 unused
    spec = {"forest": forest, "encoders": encoders, "class_codes": [0, 1, 2, 3]}
    rk = rank_code(spec, dict_sizes)
    used = set(int(f) for f in forest["feature"] if f >= 0)
    assert 3 not in used and rk["n_slots"] == len(used)
    codes = {a: rng.integers(-1, d, size=300) for a, d in dict_sizes.items()}
    got = _image_margins(spec, dict_sizes, codes)[4]
    assert np.array_equal(got, forest_margins(forest, encode_matrix(encoders, codes, {}, dict_sizes)))
    forest["missing_left"][::3] = 1                              # both directions now -> more slots
    assert rank_code(spec, dict_sizes)["n_slots"] > len(used)
    got = _image_margins(spec, dict_sizes, codes)[4]
    assert np.array_equal(got, forest_margins(forest, encode_matrix(encoders, codes, {}, dict_sizes)))


def test_ranked_image_padding_and_chunks():
    from oracle.forest import forest_margins
    from repair.forest import (RANKED_CHUNK_LEAVES, RANKED_CHUNK_NODES, RANKED_CHUNK_TREES, RANKED_GROUP,
                               encode_matrix, encoder_width)
    from tools.randforest import random_forest
    rng = np.random.default_rng(8)
    dict_sizes = {"a": 6, "b": 20}
    encoders = [{"attr": "a", "type": "sum", "categories": [0, 1, 2, 3, 4, 5]},
                {"attr": "b", "type": "ordinal", "categories": list(range(20))}]
    n_feat = sum(encoder_width(e) for e in encoders)
    forest = random_forest(n_feat, 7, 120, [[-0.5, 0.5]] * 5 + [[j + 0.5 for j in range(1, 20)]], rng)
    spec = {"forest": forest, "encoders": encoders, "class_codes": list(range(7))}
    n = 40
    codes = {a: rng.integers(-1, d, size=n) for a, d in dict_sizes.items()}
    rk, img, off, order, got = _image_margins(spec, dict_sizes, codes)
    cto, cs = img["chunk_tree_off"], img["chunk_seq"]
    cn, cl, ch = img["chunk_node_off"], img["chunk_leaf_off"], img["chunk_hdr_off"]
    assert np.all(cn % 4 == 0) and np.all(cl % 4 == 0) and np.all(ch % 2 == 0)
    # the device form of the leaf table: per chunk the low words of its float64 values, then the high words
    sp = img["leaf_split"]
    assert sp.dtype == np.uint32 and len(sp) == 2 * len(img["leaf"])
    for c in range(len(cs)):
        a, b = int(cl[c]), int(cl[c + 1])
        back = (sp[2 * a + (b - a):2 * b].astype(np.uint64) << np.uint64(32)) | sp[2 * a:2 * a + (b - a)].astype(np.uint64)
        assert np.array_equal(back.view(np.float64), img["leaf"][a:b])
    assert cto[0] == 0 and cto[-1] == len(order) and np.all(np.diff(cto) > 0) and len(cs) == len(cto) - 1
    for c in range(len(cs)):
        assert off[cs[c]] <= cto[c] and cto[c + 1] <= off[cs[c] + 1]                    # inside one sequence
        assert cn[c + 1] - cn[c] <= RANKED_CHUNK_NODES and cl[c + 1] - cl[c] <= RANKED_CHUNK_LEAVES
        assert cto[c + 1] - cto[c] <= RANKED_CHUNK_TREES
        assert (cto[c + 1] - cto[c]) % RANKED_GROUP == 0 or cto[c + 1] == off[cs[c] + 1]
    assert list(cs) == sorted(cs) and set(cs) == set(range(7))
    # every leaf of a tree sits in the tail its values are stored for; few slots are wasted on internal nodes
    toff, first = rk["tree_offset"], rk["first_leaf"]
    for t in range(len(first)):
        w = rk["word"][toff[t]:toff[t + 1]]
        leaves = np.nonzero((w & 0xFF) == 0)[0]
        assert leaves.min() == first[t] and np.array_equal((w[leaves] >> 8) & 0xFFFF, leaves)
    n_leaves = int(((rk["word"] & 0xFF) == 0).sum())
    assert n_leaves <= len(rk["leaf_value"]) <= 1.35 * n_leaves
    # walking the chunked image (chunk-absolute child indices, root words and value biases in the
    # headers) gives the oracle's margins
    assert np.array_equal(got, forest_margins(forest, encode_matrix(encoders, codes, {}, dict_sizes)))


def test_ranked_image_of_stumps_and_single_leaf_trees():
    """Depth 0 / 1 forests and mixed shapes: the walk's last level is the only level."""
    from oracle.forest import forest_margins
    from repair.forest import encode_matrix
    from tools.randforest import random_forest
    rng = np.random.default_rng(3)
    dict_sizes = {"a": 4, "b": 17}
    encoders = [{"attr": "a", "type": "sum", "categories": [0, 1, 2, 3]},
                {"attr": "b", "type": "ordinal", "categories": list(range(17))}]
    thr = [[-0.5, 0.5]] * 3 + [[j + 0.5 for j in range(1, 17)]]
    codes = {a: rng.integers(-1, d, size=64) for a, d in dict_sizes.items()}
    X = encode_matrix(encoders, codes, {}, dict_sizes)
    for max_depth, max_leaves in ((0, 1), (1, 2), (2, 3), (7, 31)):
        forest = random_forest(4, 3, 9, thr, rng, max_depth=max_depth, max_leaves=max_leaves)
        spec = {"forest": forest, "encoders": encoders, "class_codes": [0, 1, 2]}
        rk, img, _, _, got = _image_margins(spec, dict_sizes, codes)
        assert rk["max_depth"] <= max_depth
        assert np.array_equal(got, forest_margins(forest, X)), max_depth


def test_misc_repair_applies_updates_like_the_reference():
    """RepairMiscSuite.scala:125-155 (repairAttrsFrom) known answers + misc.py:87-89 option check."""
    import pandas as pd
    from repair import delphi
    from repair.utils import AnalysisException
    inp = pd.DataFrame({"tid": [1, 2, 3], "x": pd.array([None, None, 1], dtype="Int64"),
                        "y": ["test-1", None, "test-2"], "z": [1.0, 2.0, None]})
    upd = pd.DataFrame({"tid": [1, 2, 2, 3], "attribute": ["x", "x", "y", "z"],
                        "repaired": ["2.4", "2.6", "test-3", "3.1D"]})
    delphi.register_table("inputView", inp)
    delphi.register_table("repairUpdates", upd)
    out = delphi.misc.options({"repair_updates": "repairUpdates", "table_name": "inputView", "row_id": "tid"}).repair()
    assert out["tid"].tolist() == [1, 2, 3] and out["x"].tolist() == [2, 3, 1]
    assert out["y"].tolist() == ["test-1", "test-3", "test-2"] and out["z"].tolist() == [1.0, 2.0, 3.1]
    assert inp["y"].isna().tolist() == [False, True, False]         # the input is left alone
    with pytest.raises(AnalysisException, match="Table 'inputView' must have 'tid', 'attribute', and 'repaired' columns"):
        delphi.misc.options({"repair_updates": "inputView", "table_name": "inputView", "row_id": "tid"}).repair()
    with pytest.raises(ValueError, match="Required options not found: repair_updates, table_name, row_id"):
        delphi.misc.option("table_name", "inputView").repair()


def test_regex_structure_repair_matches_the_oracle_on_random_patterns():
    """Product scanner (repair/regex_structure.py) vs the oracle's restatement of RegexBase.g4 +
    RegexStructureRepair.scala: same tokens, same verdict (lexer error / outside the grammar / ok),
    same repaired strings -- on the reference's patterns and on random ones."""
    import random
    import re
    from oracle.regex_repair import RegexStructureRepair as Oracle
    from oracle.regex_repair import lex
    from repair.regex_structure import LexError, StructureRepair, tokenize
    rnd = random.Random(1)
    pats = ["^[0-9]{1,3} patients$", "^[0-9]{1,3}%", "^[0-9]{2}-[0-9]{2}-[0-9]{2}-[0-9]{2}$", "[a-z]{2,}[0-9]{,3}xy",
            "^ab[0-9]{2}.*cd$", "[a-c0-9A-Z]{3}--[x]{1}%", "ab|cd[0-9]{1}", "[0-9]+ab", "^[0-9]{1,", "a{2}bc",
            "x[0-9]{2}", "[a-b-c]{2}zz", "[0-9]{2}?ab", "", "^$", "[z-a]{2}ab"]
    alphabet = "ab0-9[]{},^$ %-xyz.*+?|"
    pats += ["".join(rnd.choice(alphabet) for _ in range(rnd.randint(1, 10))) for _ in range(1500)]
    vals = ["32 patxxnts", "1xx patients", "23.39.23.11", "ab12zzcd", "aa123xy", "9AZ--x%", "ab", "cd5", "55ab", "xx", ""]
    n_ok = 0
    for p in pats:
        try:
            want_tokens = [t[1] for t in lex(p)]
        except ValueError:
            want_tokens = None
        try:
            got_tokens = [t[1] for t in tokenize(p)]
        except LexError:
            got_tokens = None
        assert got_tokens == want_tokens, p

        def verdict(make):
            try:
                return make(p), "ok"
            except NotImplementedError:
                return None, "outside the grammar"
            except re.error:
                return None, "does not compile"
            except ValueError:
                return None, "lexer error"
        o, ov = verdict(Oracle)
        g, gv = verdict(StructureRepair)
        assert ov == gv, (p, ov, gv)
        if o is not None:
            n_ok += 1
            assert [o(v) for v in vals] == [g(v) for v in vals], p
    assert n_ok > 50


def test_nearest_value_lut_and_functional_deps_host_logic(tmp_path):
    """Host halves of the rule-based repairs against the oracle (no GPU involved)."""
    from oracle import repair as OR
    from oracle.table import from_rows
    from repair import RepairModel
    from repair import rules as RU
    from repair.costs import Levenshtein
    from repair.errors import ConstraintErrorDetector, NullErrorDetector
    from repair.table import EncodedTable
    import pandas as pd
    df = pd.DataFrame({"tid": [1, 3, 4, 5, 6], "v0": ["100%", "32%", "1xx%", "100x", "12x"],
                       "v1": [100, 101, 1, 2, 300], "v2": ["a", "b", "a", "b", "a"]})
    enc = EncodedTable.from_pandas(df, "tid")
    # v0: error cells 1xx% / 100x / 12x, domain {100%, 32%}
    col = enc.by_name["v0"]
    cur = [col.code_of(v) for v in ("1xx%", "100x", "12x")]
    dom = [col.code_of(v) for v in ("100%", "32%")]
    lut = RU.nearest_value_lut(col, cur, dom, Levenshtein(), 2.0)
    assert [col.dictionary[lut[c + 1]] for c in cur] == ["100%", "100%", "32%"] and (lut >= 0).sum() == 3
    # v1 (integers): 101 -> 100, 2 -> 1, 300 -> 100; a zero in the domain has a NULL cost (costs.py:33-34)
    col = enc.by_name["v1"]
    cur = [col.code_of(v) for v in (101, 2, 300)]
    lut = RU.nearest_value_lut(col, cur, [col.code_of(100), col.code_of(1)], Levenshtein(), 2.0)
    assert [int(col.dictionary[lut[c + 1]]) for c in cur] == [100, 1, 100]
    # ties and far values repair nothing
    col = enc.by_name["v2"]
    assert (RU.nearest_value_lut(col, [0], [0, 1], Levenshtein(), 0.5) >= 0).sum() == 1      # 'a' itself, cost 0
    assert (RU.nearest_value_lut(enc.by_name["v0"], [enc.by_name["v0"].code_of("12x")], dom, Levenshtein(), 1.0)
            >= 0).sum() == 0
    # functional dependencies: same map as the oracle (DepGraphSuite.scala:230-266)
    import os
    from conftest import GOLDEN
    hosp = pd.read_csv(os.path.join(GOLDEN, "hospital.csv"), dtype=str).astype({"tid": int})
    henc = EncodedTable.from_pandas(hosp, "tid")
    rm = RepairModel()
    rm.setRepairByRules(True)
    path = os.path.join(GOLDEN, "hospital_constraints.txt")
    rm.setErrorDetectors([NullErrorDetector(), ConstraintErrorDetector(path, "City->ZipCode")])
    targets = ["HospitalOwner", "Condition", "CountyName", "HospitalName", "EmergencyService", "ZipCode", "MeasureCode"]
    assert RU.functional_deps(rm, henc, targets) == OR.functional_deps(henc.names, path, "City->ZipCode", targets)
    rm.option("model.rule.repair_by_functional_deps.disabled", "1")
    assert RU.functional_deps(rm, henc, targets) is None
    order = RU.resolve_prediction_order([("a", ("fd", "b")), ("b", ("fd", "c")), ("c", ("forest",)), ("d", ("fd", "z"))],
                                        ["a", "b", "c", "d"])
    assert [y for y, _ in order] == ["c", "b", "d", "a"]
    del from_rows, tmp_path


def test_arrow_ingest_matches_pandas_ingest_and_arrow_egress(tmp_path):
    """EncodedTable.from_arrow (plain, chunked and Parquet-dictionary-page input) == from_pandas on the
    reference's fixtures; cells_to_arrow decodes like Column.decode."""
    import pandas as pd
    import pyarrow as pa
    import pyarrow.parquet as pq
    from conftest import GOLDEN
    from repair import RepairModel
    from repair.table import EncodedTable, cells_to_arrow
    from repair.utils import AnalysisException

    def same(a, b):
        assert a.names == b.names and np.array_equal(a.row_ids, b.row_ids) and a.row_id_kind == b.row_id_kind
        for ca, cb in zip(a.columns, b.columns):
            assert ca.kind == cb.kind and list(ca.dictionary) == list(cb.dictionary), ca.name
            assert np.array_equal(ca.codes, cb.codes), ca.name
            assert (ca.values is None) == (cb.values is None)
            if ca.values is not None:
                assert np.array_equal(ca.values, cb.values, equal_nan=True)

    for name in ("adult.csv", "hospital.csv", "boston.csv"):
        df = pd.read_csv(os.path.join(GOLDEN, name), dtype=str if name == "hospital.csv" else None)
        if name == "hospital.csv":
            df = df.astype({"tid": int})
        want = EncodedTable.from_pandas(df, "tid")
        t = pa.Table.from_pandas(df, preserve_index=False)
        same(EncodedTable.from_arrow(t, "tid"), want)
        path = str(tmp_path / (name + ".parquet"))
        pq.write_table(t, path, row_group_size=max(len(df) // 3, 1))
        strs = [f.name for f in t.schema if pa.types.is_string(f.type) or pa.types.is_large_string(f.type)]
        t2 = pq.read_table(path, read_dictionary=strs)                       # dictionary pages, several chunks
        assert not strs or any(pa.types.is_dictionary(f.type) for f in t2.schema)
        same(EncodedTable.from_arrow(t2, "tid"), want)
    # the type gate and the row-id check speak like checkInputTable (RepairApi.scala:34-67)
    bad = pa.table({"tid": [1, 2], "x": [True, False], "y": ["a", "b"]})
    with pytest.raises(AnalysisException, match="unsupported ones found: boolean"):
        EncodedTable.from_arrow(bad, "tid")
    with pytest.raises(AnalysisException, match="Uniqueness does not hold in column 'tid'"):
        EncodedTable.from_arrow(pa.table({"tid": [1, 1], "x": ["a", "b"], "y": ["a", "b"]}), "tid")
    assert RepairModel().setArrowInput(t).input is t
    with pytest.raises(TypeError, match="should be provided as str/DataFrame"):
        RepairModel().setInput(t)
    # egress: dictionary arrays over the column dictionaries
    enc = EncodedTable.from_pandas(pd.read_csv(os.path.join(GOLDEN, "adult.csv")), "tid")
    cells = [("Sex", np.array([3, 7, 12]), np.array([-1, -1, 0], dtype=np.int32), np.array([1, 0, -1], dtype=np.int32)),
             ("Age", np.array([5]), np.array([-1], dtype=np.int32), np.array([2], dtype=np.int32))]
    frame = cells_to_arrow(enc, cells)
    assert pa.types.is_dictionary(frame.schema.field("repaired").type)
    got = frame.to_pylist()
    sex, age = enc.by_name["Sex"].strings(), enc.by_name["Age"].strings()
    assert got == [{"tid": enc.row_ids[3], "attribute": "Sex", "current_value": None, "repaired": sex[1]},
                   {"tid": enc.row_ids[7], "attribute": "Sex", "current_value": None, "repaired": sex[0]},
                   {"tid": enc.row_ids[12], "attribute": "Sex", "current_value": sex[0], "repaired": None},
                   {"tid": enc.row_ids[5], "attribute": "Age", "current_value": None, "repaired": age[2]}]
    assert cells_to_arrow(enc, []).num_rows == 0


def test_invalid_running_modes_are_refused_before_any_gpu_work():
    # tests/test_model.py:231-266 (all raised on the host, before an engine exists)
    import pandas as pd
    from repair import RepairModel
    from repair.costs import Levenshtein
    mixed = pd.DataFrame({"tid": range(6), "v1": [1, 2, 3, 2, None, 2], "v2": ["a", "b", "a", None, "a", "b"],
                          "v3": [1.0, 1.5, None, 1.4, 1.1, 1.2]})
    m = RepairModel().setInput(mixed).setRowId("tid").setRepairDelta(1).setUpdateCostFunction(Levenshtein())
    with pytest.raises(ValueError, match="Cannot enable the maximal likelihood repair mode when continous attributes found"):
        m.run(maximal_likelihood_repair=True)
    adult = pd.read_csv(os.path.join(GOLDEN, "adult.csv"))
    m = RepairModel().setInput(adult).setRowId("tid").setRepairByRules(True).setUpdateCostFunction(Levenshtein()) \
        .setRepairDelta(3).option("model.rule.repair_by_nearest_values.disabled", "")
    msg = "Cannot repair data by nearest values when enabling `maximal_likelihood_repair`, " \
          "`compute_repair_candidate_prob`, `compute_repair_prob`, or `compute_repair_score`"
    for mode in ("maximal_likelihood_repair", "compute_repair_candidate_prob", "compute_repair_prob",
                 "compute_repair_score"):
        with pytest.raises(ValueError, match=msg):
            m.run(**{mode: True})



def test_training_data_rebalancing_restates_smoten_and_random_under_sampling():
    """repair/rebalance.py (train.py:242-293): every class ends at the median class size -- larger classes keep
    a subset of their rows, smaller ones (with more than k = 5 rows) get synthetic rows whose every feature
    value is the mode of the k nearest class members under the value difference metric."""
    from repair.rebalance import K_NEIGHBORS, rebalance
    rng = np.random.default_rng(4)
    n = 600
    y = rng.choice([0, 1, 2, 3, 4], size=n, p=[0.55, 0.25, 0.12, 0.075, 0.005])
    y[:3] = 4                                        # a class too small to over-sample
    codes = np.stack([(y * 2 + rng.integers(0, 2, n)) % 7, rng.integers(-1, 5, n), (y + rng.integers(0, 3, n)) % 4],
                     axis=1).astype(np.int32)
    src, out_codes, out_y = rebalance(codes, y)
    counts = np.bincount(y, minlength=5)
    median = int(np.median(counts))
    got = np.bincount(out_y, minlength=5)
    for c in range(5):
        want = median if counts[c] > K_NEIGHBORS else counts[c]
        assert got[c] == want, (c, counts[c], got[c])
    real = src >= 0
    assert np.array_equal(out_codes[real], codes[src[real]]) and np.array_equal(out_y[real], y[src[real]])
    assert len(np.unique(src[real])) == real.sum()                      # under-sampling draws without replacement
    for c in range(5):                                                  # synthetic rows only use the class's own values
        synth = out_codes[(~real) & (out_y == c)]
        for j in range(codes.shape[1]):
            assert set(synth[:, j].tolist()) <= set(codes[y == c][:, j].tolist())
    # deterministic (seeded)
    again = rebalance(codes, y)
    assert all(np.array_equal(a, b) for a, b in zip(again, (src, out_codes, out_y)))


def test_row_id_joins_are_vectorised_and_string_compatible():
    """utils.row_positions (setErrorCells / misc.repair / maximal-likelihood repair_data): ids are compared like
    the reference's CAST(.. AS STRING) joins, without a Python dict over the table."""
    from repair.utils import row_positions
    pos, found = row_positions(np.array([3, 5, 9, 12]), ["5", "12", "7", 9, "x"])
    assert list(found) == [True, True, False, True, False] and list(pos[found]) == [1, 3, 2]
    pos, found = row_positions(np.array([9, 3, 12, 5]), [5, 12, 7, 9])            # unordered integer ids
    assert list(found) == [True, True, False, True] and list(pos[found]) == [3, 2, 0]
    pos, found = row_positions(np.array(["a", "b", "c"], dtype=object), ["c", "z", "a"])
    assert list(found) == [True, False, True] and list(pos[found]) == [2, 0]
    pos, found = row_positions(np.zeros(0, dtype=np.int64), [1])
    assert list(found) == [False]


def test_search_keeps_the_defaults_unless_a_configuration_wins_by_one_standard_error():
    """search.search: trial 0 = LightGBM's defaults; max_evals = 1 does not evaluate at all; a better mean CV
    loss only wins when it beats the defaults by more than the standard error of the defaults' folds."""
    from repair import search as HS
    assert HS.search(lambda p: 1 / 0, 1, 50, 0) == (dict(HS.DEFAULTS), None, 0)
    calls = []

    def noisy(p):          # every configuration 2 % better than the defaults, whose folds scatter by 10 %
        calls.append(p)
        return (1.0, [0.9, 1.0, 1.1]) if p == HS.DEFAULTS else (0.98, [0.98] * 3)
    best, loss, n = HS.search(noisy, 6, 50, 0)
    assert calls[0] == HS.DEFAULTS and n == 6 and best == HS.DEFAULTS and loss == 1.0

    def clear(p):          # a clear win is taken
        return (1.0, [0.99, 1.0, 1.01]) if p == HS.DEFAULTS else (0.5, [0.5] * 3)
    best, loss, n = HS.search(clear, 4, 50, 0)
    assert best != HS.DEFAULTS and loss == 0.5
    # plain floats (no fold losses) fall back to hyperopt's argmin; exceptions count as loss 0.0 (train.py:176-180)
    best, loss, _ = HS.search(lambda p: 1.0 if p == HS.DEFAULTS else 0.9, 3, 50, 0)
    assert best != HS.DEFAULTS and loss == 0.9
    # early stop after `no_progress_loss` evaluations without improvement
    assert HS.search(lambda p: 1.0, 100, 5, 0)[2] == 6


def test_gpu_trainer_bins_high_cardinality_features_like_max_bin():
    """gbdt.bin_sample: more than 254 distinct encoded values -> adjacent values share a bin (about equal sample
    counts), every row's value lies inside its bin, thresholds fall between bins (train.py:106 max_bin = 255)."""
    from repair import gbdt as G
    from repair.forest import encoder_lut, first_seen
    rng = np.random.default_rng(0)
    k = 600
    codes = rng.integers(-1, k, size=5000)
    enc = [{"attr": "a", "type": "ordinal", "categories": first_seen(codes)},
           {"attr": "b", "type": "ordinal", "categories": list(range(10))}]
    small = rng.integers(0, 10, size=5000)
    bins, n_bins, values = G.bin_sample(enc, {"a": codes, "b": small}, {"a": k, "b": 10})
    assert bins.dtype == np.uint8 and n_bins[0] <= G.MAX_BINS + 1 and n_bins[1] in (11, 12)   # 10 values (+ "unseen") + missing
    hi, lo = values[0]
    assert np.all(lo <= hi) and np.all(hi[:-1] < lo[1:])                 # disjoint, ordered value ranges
    e = encoder_lut(enc[0], k)[:, 0][codes + 1]
    ok = ~np.isnan(e)
    b = bins[:, 0].astype(np.int64)
    assert np.all(b[~ok] == n_bins[0] - 1)                               # missing bin
    assert np.all((e[ok] >= lo[b[ok]]) & (e[ok] <= hi[b[ok]]))
    assert np.bincount(b[ok]).max() <= 3 * len(e) // G.MAX_BINS + 3      # roughly equal-count bins
    assert np.ndim(values[1]) == 1                                       # the small feature keeps one bin per value
    # thresholds: midway between the split bin's largest and the next bin's smallest value
    nodes = np.zeros((1, 1, G.MAX_NODES), dtype=G.NODE_DTYPE)
    nodes[0, 0, 0] = (0, 3, 0, 1, 2, (0, 0), 0.0)
    nodes[0, 0, 1] = (-1, 0, 0, 0, 0, (0, 0), -1.0)
    nodes[0, 0, 2] = (-1, 0, 0, 0, 0, (0, 0), 1.0)
    f = G.flatten(nodes, np.array([[3]]), np.zeros(1), values, 2, 1)
    assert f["threshold"][0] == (hi[3] + lo[4]) / 2.0


def test_presence_map_decodes_pairs_on_demand():
    """engine._PresenceMap: the packed presence bits of a pair launch, unpacked per pair only when asked."""
    from repair.engine import _PresenceMap
    dom = {"x": 3, "y": 5, "z": 2}
    pairs = [("x", "y"), ("z", "x")]
    rng = np.random.default_rng(1)
    mats = [rng.random((dom[a] + 1, dom[b] + 1)) < 0.4 for a, b in pairs]
    words, offs = [], [0]
    for m in mats:
        bits = np.zeros((m.size + 31) // 32 * 32, dtype=np.uint8)
        bits[:m.size] = m.reshape(-1)
        words.append(np.packbits(bits, bitorder="little").view(np.uint32))
        offs.append(offs[-1] + len(words[-1]))
    pm = _PresenceMap(pairs, offs, np.concatenate(words), dom)
    assert ("x", "y") in pm and ("y", "x") not in pm and pm.get(("y", "x")) is None
    assert np.array_equal(pm[("x", "y")], mats[0]) and np.array_equal(pm.get(("z", "x")), mats[1])


def test_bench_frame_comparison_catches_differences():
    """bench.frames_equal (the e2e leg's check of the API's Arrow frame against the resident pass)."""
    import sys
    import pyarrow as pa
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    from repair.table import EncodedTable
    names = ["a", "b", "c"]
    table = EncodedTable.from_codes("tid", names, [np.zeros(4, dtype=np.int32)] * 3, [3, 2, 2])
    out = [("a", np.array([1, 3], dtype=np.int32), np.array([-1, 2], dtype=np.int32), np.array([0, 1], dtype=np.int32)),
           ("c", np.array([0], dtype=np.int32), np.array([1], dtype=np.int32), np.array([-1], dtype=np.int32))]

    def frame(rep_a=(0, 1), ids_a=(101, 103)):
        def dic(codes, attr):
            strs = pa.array(table.by_name[attr].strings(), type=pa.string())
            codes = np.asarray(codes, dtype=np.int32)
            return pa.DictionaryArray.from_arrays(pa.array(codes, mask=codes < 0), strs)
        attr_names = pa.array(["a", "b", "c"], type=pa.string())
        att = [pa.DictionaryArray.from_arrays(pa.array(np.array([0, 0], dtype=np.int32)), attr_names),
               pa.DictionaryArray.from_arrays(pa.array(np.array([2], dtype=np.int32)), attr_names)]
        return pa.table({"tid": pa.chunked_array([pa.array(np.array(ids_a, dtype=np.int64)), pa.array(np.array([100], dtype=np.int64))]),
                         "attribute": pa.chunked_array(att),
                         "current_value": pa.chunked_array([dic([-1, 2], "a"), dic([1], "c")]),
                         "repaired": pa.chunked_array([dic(list(rep_a), "a"), dic([-1], "c")])})
    assert bench.frames_equal(frame(), out, 100, names, table)
    assert not bench.frames_equal(frame(rep_a=(0, 2)), out, 100, names, table)        # a repaired value differs
    assert not bench.frames_equal(frame(ids_a=(101, 102)), out, 100, names, table)    # a row id differs
    assert not bench.frames_equal(frame(), out[:1], 100, names, table)                # an attribute is missing


def test_bench_dump_outputs_is_float64_bounded_and_order_independent(tmp_path):
    """bench.dump_outputs (--dump-outputs): whole-frame counts and per-attribute code histograms, plus every cell of
    the seeded row sample sorted by (attribute, tid); the frame's order does not change the files."""
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    import bench
    names, dom, n = ["a", "b", "c"], [3, 2, 4], 10
    out = [("a", np.array([1, 3], dtype=np.int32), np.array([-1, 2], dtype=np.int32), np.array([0, 1], dtype=np.int32)),
           ("c", np.array([0, 9], dtype=np.int32), np.array([1, 3], dtype=np.int32), np.array([-1, 2], dtype=np.int32))]
    info = bench.dump_outputs(str(tmp_path / "x"), out, names, dom, n)
    got = {f[:-4]: np.load(str(tmp_path / "x" / f)) for f in os.listdir(str(tmp_path / "x"))}
    assert info["frame_cells"] == 4 and info["sampled_cells"] == 4      # 10 rows: the sample is the whole table
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["cells_per_attribute"].tolist() == [2, 0, 2]
    assert got["current_hist"].shape == (3, 5) and got["current_hist"][0].tolist() == [1, 0, 0, 1, 0]
    assert got["repaired_hist"][2].tolist() == [1, 0, 0, 1, 0]
    assert got["tid"].tolist() == [1, 3, 0, 9] and got["attribute"].tolist() == [0, 0, 2, 2]
    assert got["current_value"].tolist() == [-1, 2, 1, 3] and got["repaired"].tolist() == [0, 1, -1, 2]
    bench.dump_outputs(str(tmp_path / "y"), [(a, r[::-1], c[::-1], p[::-1]) for a, r, c, p in out[::-1]], names, dom, n)
    assert all(np.array_equal(a, np.load(str(tmp_path / "y" / (k + ".npy")))) for k, a in got.items())
    # a larger table: the sample is a fixed subset of DUMP_SAMPLE_ROWS rows, the same in every run
    big = bench.DUMP_SAMPLE_ROWS * 4
    rows = np.arange(0, big, 2, dtype=np.int32)
    zeros = np.zeros(len(rows), dtype=np.int32)
    i1 = bench.dump_outputs(str(tmp_path / "p"), [("a", rows, zeros, zeros)], names, dom, big)
    i2 = bench.dump_outputs(str(tmp_path / "q"), [("a", rows, zeros, zeros)], names, dom, big)
    assert 0 < i1["sampled_cells"] < bench.DUMP_SAMPLE_ROWS and i1 == dict(i2, dir=i1["dir"])
    assert np.array_equal(np.load(str(tmp_path / "p" / "tid.npy")), np.load(str(tmp_path / "q" / "tid.npy")))
