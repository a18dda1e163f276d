"""LOFOutlierErrorDetector on the device: ``dr_lof_flag`` bit for bit against the host definition
(``lof_reference.lof_scores_1d``), the reference's known-answer tests through the public protocol,
pipeline parity with the oracle, the scikit-learn-backed detector, and a 2-rank sharded run equal to the
one-GPU run."""
import os
import socket
import warnings

import numpy as np
import pandas as pd
import pytest

import parity_utils as PU
from conftest import GOLDEN
from lof_reference import lof_scores_1d, with_lof

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _lof_gpu(values, k, row_begin=0, row_count=None):
    """-> (flag bits of rows [row_begin, row_begin + row_count), scores in row order, flagged count)."""
    from repair._native import Context
    ctx = Context.acquire(0)
    try:
        n = len(values)
        row_count = n - row_begin if row_count is None else row_count
        col = torch.tensor(np.asarray(values, dtype=np.float64), device="cuda")
        bm = torch.zeros(row_count // 32 + 1, dtype=torch.int32, device="cuda")
        out = torch.empty(n, dtype=torch.float64, device="cuda")
        ws = torch.empty(max(ctx.lof_workspace_bytes(n), 1), dtype=torch.uint8, device="cuda")
        cnt = ctx.lof_flag(col, n, k, row_begin, row_count, bm, ws, out_lof=out, count=True)
        bits = np.unpackbits(bm.cpu().numpy().view(np.uint8), bitorder="little")
        assert not bits[row_count:].any()
        return bits[:row_count].astype(bool), out.cpu().numpy(), cnt
    finally:
        Context.release(ctx)


def _check(values, k, row_begin=0, row_count=None):
    n = len(values)
    row_count = n - row_begin if row_count is None else row_count
    bits, got, cnt = _lof_gpu(values, k, row_begin, row_count)
    want = lof_scores_1d(values, k)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    mismatch = np.nonzero(got[~nan].view(np.int64) != want[~nan].view(np.int64))[0]
    assert len(mismatch) == 0, "{} scores differ, first at {}: {!r} vs {!r}".format(
        len(mismatch), mismatch[0], got[~nan][mismatch[0]], want[~nan][mismatch[0]])
    with np.errstate(invalid="ignore"):
        flags = (want > 1.5)[row_begin:row_begin + row_count]
    assert np.array_equal(bits, flags)
    assert cnt == int(flags.sum())
    return flags


def _gauss(n, seed, outliers=True):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=n)
    if outliers and n >= 100:
        x[rng.choice(n, max(3, n // 1000), replace=False)] = rng.uniform(8, 40, max(3, n // 1000))
    return x


def test_gaussian_1m():
    assert _check(_gauss(1_000_000, 1), 20).sum() > 0


@pytest.mark.parametrize("kind", ["mod2", "mod3", "constant"])
def test_heavy_duplicates(kind):
    n = 30_000
    ids = np.arange(n)
    x = {"mod2": ids % 2, "mod3": ids % 3, "constant": np.zeros(n)}[kind].astype(np.float64)
    x[[17, 29_000]] = [1000.0, -7.0]
    _check(x, 20)


def test_signed_zeros():
    rng = np.random.default_rng(2)
    x = rng.choice([-0.0, 0.0, 1.0, -1.0, 2.5], size=5000)
    x[10] = 60.0
    bits, got, _ = _lof_gpu(x, 20)
    _check(x, 20)
    y = np.where(x == 0.0, 0.0, x)
    assert np.array_equal(_lof_gpu(y, 20)[1], got)


@pytest.mark.parametrize("n_valid", [4001, 4000])
def test_nulls_take_the_median(n_valid):
    x = np.round(_gauss(6000, n_valid), 1)
    x[np.random.default_rng(3).permutation(6000)[:6000 - n_valid]] = np.nan
    _check(x, 20)


@pytest.mark.parametrize("n", [2, 20, 21])
def test_tiny_columns(n):
    x = _gauss(n, n)
    x[0] = 50.0
    _check(x, min(20, n - 1))


def test_all_null_and_single_row():
    for x in (np.full(100, np.nan), np.array([3.0])):
        bits, got, cnt = _lof_gpu(x, 1)
        assert not bits.any() and cnt == 0 and np.isnan(got).all()


@pytest.mark.parametrize("k", [1, 5, 20, 64])
def test_k(k):
    rng = np.random.default_rng(k)
    x = rng.integers(0, 300, size=50_000).astype(np.float64)    # many ties
    x[rng.choice(50_000, 40, replace=False)] = rng.uniform(1e3, 1e4, 40)
    x[rng.choice(50_000, 500, replace=False)] = np.nan
    _check(x, k)


def test_several_tiles_per_cta():
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    n = 3 * sm * 4 * 1024 + 333      # >= 3 tiles of 1024 positions per CTA, not a multiple of the tile
    x = np.round(_gauss(n, 5), 3)
    _check(x, 20)


def test_row_range():
    x = _gauss(20_000, 6)
    x[1500] = 99.0
    flags = _check(x, 20, row_begin=1000, row_count=5000)
    assert flags[500]


# ---- the reference's KATs through the public protocol (test_errors.py:236-340) -----------------------
def _kat_frame(nrows):
    ids = np.r_[np.arange(nrows), [1000000, 1000001, 1000002]]
    v1 = np.r_[np.arange(nrows) % 2, [1, 1000, np.nan]].astype(np.float64)
    v2 = np.r_[np.arange(nrows) % 3, [1000, 1, np.nan]].astype(np.float64)
    return pd.DataFrame({"id": ids, "v1": v1, "v2": v2})


def _cells(frame, row_id):
    return sorted((int(r), a) for r, a in zip(frame[row_id], frame["attribute"]))


@pytest.mark.parametrize("nrows", [3000, 10000])
@pytest.mark.parametrize("which", ["lof", "sklearn"])
def test_reference_kat(nrows, which):
    from repair import LOFOutlierErrorDetector, ScikitLearnBackedErrorDetector
    from sklearn.neighbors import LocalOutlierFactor
    df = _kat_frame(nrows)

    def make():
        if which == "lof":
            return LOFOutlierErrorDetector(5000, num_parallelism=1)
        return ScikitLearnBackedErrorDetector(lambda: LocalOutlierFactor(novelty=False), 5000, 1)

    with pytest.raises(ValueError, match="`num_parallelism` must be positive, got 0"):
        LOFOutlierErrorDetector(5000, num_parallelism=0)
    with pytest.raises(ValueError, match="`error_detector_cls` should be callable"):
        ScikitLearnBackedErrorDetector(1, 5000, 1)
    with pytest.raises(ValueError, match="should have a `fit_predict` method"):
        ScikitLearnBackedErrorDetector(lambda: 1, 5000, 1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")     # scikit-learn warns about the duplicate values
        for targets, want in [(["v1", "v2"], [(1000000, "v2"), (1000001, "v1")]),
                              (["v1"], [(1000001, "v1")]),
                              (["Unknown", "v1"], [(1000001, "v1")]),
                              (["Non-existent"], [])]:
            got = _cells(make().setUp("id", df, ["v1", "v2"], targets).detect(), "id")
            assert got == want, targets


# ---- pipeline parity with the oracle ------------------------------------------------------------------
def _boston():
    df = pd.read_csv(os.path.join(GOLDEN, "boston.csv"))
    df["CHAS"] = df["CHAS"].map(lambda v: None if v != v else str(v))
    df["RAD"] = df["RAD"].map(lambda v: None if v != v else str(int(v)) if float(v).is_integer() else str(v))
    return df


@pytest.fixture
def lof_aware(monkeypatch):
    """parity_utils / the oracle pipeline, taught the {"type": "lof"} detector."""
    from oracle import repair as OR
    from repair import LOFOutlierErrorDetector
    monkeypatch.setattr(OR, "run_detectors", with_lof(OR.run_detectors))
    make = PU.make_detectors
    monkeypatch.setattr(PU, "make_detectors", lambda specs: [
        LOFOutlierErrorDetector() if s["type"] == "lof" else make([s])[0] for s in specs])


SPECS = [{"type": "null"}, {"type": "lof"}]


def test_boston_detect_parity(lof_aware):
    got, want, _ = PU.run_both_frame(_boston(), "tid", SPECS, mode="detect")
    assert got == want
    assert sum(1 for g in got if g[2] is not None) > 20      # LOF cells beyond the NULL cells


def test_boston_repair_parity(lof_aware):
    got, want, _ = PU.run_both_frame(_boston(), "tid", SPECS, opts={"model.lgb.n_estimators": 20})
    assert got == want
    assert len(got) > 0


def test_boston_arrow_input_equals_pandas_input():
    import pyarrow as pa
    from repair import LOFOutlierErrorDetector, NullErrorDetector, RepairModel
    df = _boston()
    want = PU.frame_tuples(RepairModel().setInput(df).setRowId("tid").setErrorDetectors(
        [NullErrorDetector(), LOFOutlierErrorDetector()]).run(detect_errors_only=True), "tid")
    out = RepairModel().setArrowInput(pa.Table.from_pandas(df, preserve_index=False)).setRowId("tid") \
        .setErrorDetectors([NullErrorDetector(), LOFOutlierErrorDetector()]).run(detect_errors_only=True)
    got = PU.frame_tuples(out.to_pandas() if hasattr(out, "to_pandas") else out, "tid")
    assert got == want and len(got) > 0


def test_sklearn_backed_equals_lof_on_tie_free_data():
    from repair import LOFOutlierErrorDetector, RepairModel, ScikitLearnBackedErrorDetector
    from sklearn.neighbors import LocalOutlierFactor
    n = 5000
    rng = np.random.default_rng(11)
    df = pd.DataFrame({"tid": np.arange(n), "x": _gauss(n, 12), "y": rng.exponential(size=n),
                       "s": rng.choice(["a", "b", "c"], size=n)})
    runs = []
    for det in (LOFOutlierErrorDetector(), ScikitLearnBackedErrorDetector(lambda: LocalOutlierFactor(novelty=False))):
        runs.append(PU.frame_tuples(RepairModel().setInput(df).setRowId("tid").setErrorDetectors([det])
                                    .run(detect_errors_only=True), "tid"))
    assert runs[0] == runs[1]
    assert {t[1] for t in runs[0]} == {"x", "y"}


def test_reference_example_runs_unchanged():
    # resources/examples/error-detectors.py: delphi.repair.setInput(df).setRowId(..).setErrorDetectors([..]).run()
    from repair import LOFOutlierErrorDetector, delphi
    out = delphi.repair.setInput(_boston()).setRowId("tid").setErrorDetectors([LOFOutlierErrorDetector()]) \
        .option("model.hp.max_evals", "1").run()
    assert len(out) > 0


# ---- 2 ranks == 1 GPU ---------------------------------------------------------------------------------
N_DIST = 60_000


def _dist_frame():
    rng = np.random.default_rng(21)
    x = np.round(rng.normal(size=N_DIST), 2)              # ties; both shards cover the same value range
    x[rng.choice(N_DIST, 30, replace=False)] = rng.uniform(10, 50, 30)
    x[N_DIST // 2 + rng.choice(N_DIST // 2, 700, replace=False)] = np.nan   # NULLs in the second shard only
    y = rng.normal(size=N_DIST) * 3
    return pd.DataFrame({"tid": np.arange(N_DIST), "x": x, "y": y, "s": rng.choice(["p", "q"], size=N_DIST)})


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _dets(which):
    from repair import LOFOutlierErrorDetector, NullErrorDetector, ScikitLearnBackedErrorDetector
    from sklearn.neighbors import LocalOutlierFactor
    if which == "lof":
        return [NullErrorDetector(), LOFOutlierErrorDetector()]
    return [ScikitLearnBackedErrorDetector(lambda: LocalOutlierFactor(novelty=False))]


def _dist_worker(rank, world, port, backend, out_dir):
    import torch.distributed as td
    from repair import RepairModel
    from repair.table import EncodedTable
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    td.init_process_group(backend, rank=rank, world_size=world)
    df = _dist_frame()
    lo, hi = (N_DIST * rank) // world, (N_DIST * (rank + 1)) // world
    shard = EncodedTable.from_pandas(df.iloc[lo:hi].reset_index(drop=True), "tid")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for which in ("lof", "sklearn"):
            out = RepairModel().setEncodedInput(shard).setErrorDetectors(_dets(which)) \
                .setDistributed(True, dev).run(detect_errors_only=True)
            got = PU.frame_tuples(out, "tid")
            assert all(lo <= int(t[0]) < hi for t in got)
            gathered = [None] * world
            td.all_gather_object(gathered, got)
            if rank == 0:
                union = sorted((t for part in gathered for t in part), key=lambda t: (int(t[0]), t[1]))
                full = RepairModel().setInput(df).setRowId("tid").setErrorDetectors(_dets(which)) \
                    .run(detect_errors_only=True)
                want = sorted(PU.frame_tuples(full, "tid"), key=lambda t: (int(t[0]), t[1]))
                assert sum(1 for t in want if t[1] == "x" and t[2] is not None) > 10
                assert union == want, which
    td.barrier()
    open(os.path.join(out_dir, "ok%d" % rank), "w").write("ok")
    td.destroy_process_group()


def test_two_rank_lof_equals_one_gpu(tmp_path):
    import torch.multiprocessing as mp
    backend = "nccl" if torch.cuda.device_count() >= 2 else "gloo"
    mp.spawn(_dist_worker, args=(2, _free_port(), backend, str(tmp_path)), nprocs=2, join=True)
    assert sorted(os.listdir(tmp_path)) == ["ok0", "ok1"]
