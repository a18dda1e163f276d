"""LOFOutlierErrorDetector / ScikitLearnBackedErrorDetector without a GPU: the host definition of the
one-dimensional LOF against scikit-learn and against the reference's known-answer table, and the
detector classes' constructors."""
import warnings

import numpy as np
import pytest

import parity_utils  # noqa: F401  (sys.path)
from lof_reference import LOF_K, lof_flags, lof_scores_1d


def _tie_free(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=n)
    if n >= 21:
        x[rng.choice(n, 3, replace=False)] = [9.5, -11.25, 17.0]
    assert len(np.unique(x)) == n
    return x


@pytest.mark.parametrize("n", [2, 3, 21, 22, 5000])
def test_oracle_matches_sklearn_on_tie_free_data(n):
    from sklearn.neighbors import LocalOutlierFactor
    x = _tie_free(n, seed=n)
    got = lof_scores_1d(x, min(LOF_K, n - 1))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = LocalOutlierFactor(novelty=False)
        labels = m.fit_predict(x[:, None])
    want = -m.negative_outlier_factor_
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    assert np.array_equal(lof_flags(x), labels < 0)


def _kat_columns(nrows):
    ids = np.r_[np.arange(nrows), [1000000, 1000001, 1000002]]
    v1 = np.r_[np.arange(nrows) % 2, [1, 1000, np.nan]].astype(np.float64)
    v2 = np.r_[np.arange(nrows) % 3, [1000, 1, np.nan]].astype(np.float64)
    return ids, {"v1": v1, "v2": v2}


@pytest.mark.parametrize("nrows", [3000, 10000])
def test_reference_kat_through_the_oracle(nrows):
    # test_errors.py:236-267: LOFOutlierErrorDetector on id, id % 2, id % 3 plus three dirty rows
    ids, cols = _kat_columns(nrows)
    flagged = {a: set(ids[lof_flags(v)].tolist()) for a, v in cols.items()}
    for targets, want in [(["v1", "v2"], [(1000000, "v2"), (1000001, "v1")]),
                          (["v1"], [(1000001, "v1")]),
                          (["Unknown", "v1"], [(1000001, "v1")]),
                          (["Non-existent"], [])]:
        got = sorted((int(r), a) for a in cols if a in targets for r in flagged[a])
        assert got == want, targets


def test_oracle_edge_cases():
    assert np.isnan(lof_scores_1d([np.nan, np.nan, np.nan], 2)).all()
    assert np.isnan(lof_scores_1d([1.0], 1)).all()
    assert not lof_flags([5.0]).any()
    # a constant column: every reach distance is 0, every lrd 1e10, every lof exactly 1
    assert (lof_scores_1d(np.full(50, 3.0), 20) == 1.0).all()
    # -0.0 and +0.0 are one value; NULLs take the median
    a = lof_scores_1d([-0.0, 0.0, 1.0, 2.0, np.nan, 40.0], 2)
    b = lof_scores_1d([0.0, 0.0, 1.0, 2.0, 1.0, 40.0], 2)
    assert np.array_equal(a, b)


def test_constructors_and_lowering():
    from repair import LOFOutlierErrorDetector, ScikitLearnBackedErrorDetector
    from repair.errors import ScikitLearnBasedErrorDetector
    from sklearn.neighbors import LocalOutlierFactor

    with pytest.raises(ValueError, match="`num_parallelism` must be positive, got 0"):
        LOFOutlierErrorDetector(5000, num_parallelism=0)
    with pytest.raises(ValueError, match="`num_parallelism` must be positive, got 0"):
        ScikitLearnBackedErrorDetector(lambda: LocalOutlierFactor(novelty=False), 5000, 0)
    with pytest.raises(ValueError, match="`error_detector_cls` should be callable"):
        ScikitLearnBackedErrorDetector(1, 5000, 1)
    with pytest.raises(ValueError, match="An instance that `error_detector_cls` returns should have a "
                                         "`fit_predict` method"):
        ScikitLearnBackedErrorDetector(lambda: 1, 5000, 1)
    with pytest.raises(TypeError):
        ScikitLearnBasedErrorDetector()

    lof = LOFOutlierErrorDetector()
    assert str(lof) == "LOFOutlierErrorDetector()"
    assert lof.spec() == {"type": "lof"}
    assert (lof.parallel_mode_threshold, lof.num_parallelism) == (10000, None)
    assert isinstance(lof._outlier_detector_impl(), LocalOutlierFactor)

    factory = lambda: LocalOutlierFactor(novelty=False)  # noqa: E731
    sk = ScikitLearnBackedErrorDetector(factory, parallel_mode_threshold=5000, num_parallelism=2)
    assert str(sk) == "ScikitLearnBackedErrorDetector()"
    spec = sk.spec()
    assert spec["type"] == "sklearn" and isinstance(spec["factory"](), LocalOutlierFactor)
    assert (sk.parallel_mode_threshold, sk.num_parallelism) == (5000, 2)

    sk.setUp("id", "tbl", ["v1", "v2"], ["v1", "Unknown"])
    assert sk._targets == ["v1", "Unknown"]
