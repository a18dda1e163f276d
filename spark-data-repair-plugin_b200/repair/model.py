"""``RepairModel``: the reference's builder-style API (``python/repair/model.py:103-1537``) in front of
the B200 pipeline.  Setter names, argument checks, option keys, error messages, running modes and
the output schema ``(row_id, attribute, current_value, repaired)`` are the reference's; the work
behind ``run()`` is ``engine.Engine`` (CUDA) instead of Spark SQL + pandas UDFs.

Inputs: a pandas ``DataFrame`` (a pyspark ``DataFrame`` is collected once with ``toPandas()``), a
``pyarrow.Table`` (``setArrowInput``: device-side ingest, Arrow frame out), the name of a table
registered in ``repair.catalog``, or a pre-encoded ``EncodedTable``.  Every running mode of the
reference is implemented: default, ``detect_errors_only``, ``repair_data``, the pmf / prob / score modes
and maximal-likelihood repair.
"""
import logging
import time
from typing import Any, Dict, List, Optional, Union

import numpy as np
import pandas as pd
from pandas import DataFrame

from . import catalog
from . import rules as R
from .costs import UpdateCostFunction
from .errors import ErrorDetector, ErrorModelOptions, default_detectors
from .forest import DeviceModel, encode_matrix, encoder_type, first_seen
from .table import EncodedTable
from .train import build_model, train_option_keys, validate_options
from .utils import argtype_check, cell_to_string, get_option_value, row_positions, to_list_str

_logger = logging.getLogger("repair")

_MODEL_OPTS = [
    ("model.max_training_row_num", 10000, int, lambda v: v >= 10, "`{}` should be greater than and equal to 10"),
    ("model.max_training_column_num", 65536, int, lambda v: v >= 2, "`{}` should be greater than 1"),
    ("model.small_domain_threshold", 12, int, lambda v: v >= 3, "`{}` should be greater than 2"),
    ("model.rule.repair_by_regex.disabled", True, bool, None, None),
    ("model.rule.repair_by_nearest_values.disabled", True, bool, None, None),
    ("model.rule.merge_threshold", 2.0, float, None, None),
    ("model.rule.repair_by_functional_deps.disabled", False, bool, None, None),
    ("model.rule.max_domain_size", 1000, int, lambda v: v > 10, "`{}` should be greater than 10"),
    ("repair.pmf.cost_weight", 0.1, float, lambda v: v > 0.0, "`{}` should be positive"),
    ("repair.pmf.prob_threshold", 0.0, float, None, None),
    ("repair.pmf.prob_top_k", 32, int, lambda v: v >= 3, "`{}` should be greater than 2"),
]
_MODEL_OPT = {o[0]: o for o in _MODEL_OPTS}


def _is_spark_df(obj):
    return type(obj).__module__.startswith("pyspark.") and type(obj).__name__ == "DataFrame"


def _as_encoded(obj, row_id, name="input"):
    if isinstance(obj, EncodedTable):
        return obj
    if _is_spark_df(obj):
        obj = obj.toPandas()
    if _is_arrow_table(obj):
        return EncodedTable.from_arrow(obj, row_id, name)
    return EncodedTable.from_pandas(obj, row_id, name)


def _is_arrow_table(obj):
    return type(obj).__module__.startswith("pyarrow") and hasattr(obj, "schema")


def _maybe_arrow(frame, arrow_io):
    """Arrow in -> Arrow out (modes whose frame is assembled with pandas are converted at the end)."""
    if not arrow_io or _is_arrow_table(frame):
        return frame
    import pyarrow as pa
    return pa.Table.from_pandas(frame, preserve_index=False)


def select_features(pairwise_stats, y, features, max_training_column_num):
    """Keeps the features most correlated with y when there are too many (model.py:677-699)."""
    if max_training_column_num < len(features) and y in pairwise_stats:
        ranked = sorted((float(h), f) for f, h in pairwise_stats[y] if f in features)
        kept = []
        for h, f in ranked:
            if len(kept) <= 1 or (h >= 0.0 and len(kept) < max_training_column_num):
                kept.append(f)
        return kept
    return features


class RepairModel():
    """Interface to detect error cells in given input data and repair them (drop-in for
    ``repair.model.RepairModel``)."""

    option_keys = set([o[0] for o in _MODEL_OPTS]) | set(ErrorModelOptions.option_keys) | set(train_option_keys)

    def __init__(self) -> None:
        self.db_name: str = ""
        self.input: Optional[Union[str, DataFrame, EncodedTable]] = None
        self.row_id: Optional[str] = None
        self.targets: List[str] = []
        self.error_cells: Optional[Union[str, DataFrame]] = None
        self.error_detectors: List[ErrorDetector] = []
        self.discrete_thres: int = 80
        self.parallel_stat_training_enabled: bool = False
        self.training_data_rebalancing_enabled: bool = False
        self.repair_by_rules: bool = False
        self.repair_delta: Optional[int] = None
        self.cf: Optional[UpdateCostFunction] = None
        self.opts: Dict[str, str] = {}
        # engine knobs (not part of the reference API)
        self.device_index: int = 0
        self.model_provider = None   # callable(ctx) -> model spec; default: _fit (GPU GBDT / scikit-learn)
        self.trainer = "gpu"         # "gpu": dr_gbdt_train when eligible; "sklearn": always train.build_model
        self.distributed = None      # torch.distributed process group (or True = default group): row-sharded run
        self.frozen_models = None    # models of an earlier run() (setFrozenModels): skips the training phase
        self.borrow_encoded_output = False   # encoded result arrays may alias a reusable pinned buffer (bench loop)
        self.last_run: Dict[str, Any] = {}

    # ---- setters (same names / checks / messages as the reference) -------------------------------
    @argtype_check
    def setDbName(self, db_name: str) -> "RepairModel":
        if isinstance(self.input, DataFrame) or _is_spark_df(self.input):
            raise ValueError("Can not specify a database name when input is `DataFrame`")
        self.db_name = db_name
        return self

    @argtype_check
    def setTableName(self, table_name: str) -> "RepairModel":
        if not table_name:
            raise ValueError("`table_name` should have at least character")
        self.input = table_name
        return self

    @argtype_check
    def setInput(self, input: Union[str, DataFrame]) -> "RepairModel":
        if type(input) is str:
            self.setTableName(input)
        else:
            self.db_name = ""
            self.input = input
        return self

    def setArrowInput(self, table: Any) -> "RepairModel":
        """A ``pyarrow.Table`` as input (``spark_df.toArrow()``, ``pyarrow.parquet.read_table(path,
        read_dictionary=[...])``): dictionary-encoded by Arrow, no Python object per cell
        (EncodedTable.from_arrow).  ``setInput`` keeps the reference's str / DataFrame contract."""
        if not (type(table).__module__.startswith("pyarrow") and hasattr(table, "schema")):
            raise TypeError("`table` should be provided as pyarrow.Table, got {}".format(type(table).__name__))
        self.db_name = ""
        self.input = table
        return self

    def setFrozenModels(self, models: Any) -> "RepairModel":
        """Reuse the repair models an earlier ``run()`` trained (``model.last_run["models"]``) instead of
        training again: inference-only passes over new batches of the same table (same columns and
        dictionaries).  The reference retrains on every run (model.py:1001-1052); not part of its API."""
        self.frozen_models = models
        return self

    def setEncodedInput(self, table: EncodedTable) -> "RepairModel":
        """Pre-encoded input (label-encoded int32 columns + dictionaries); sets the row id too."""
        if not isinstance(table, EncodedTable):
            raise TypeError("`table` should be provided as EncodedTable, got {}".format(type(table).__name__))
        self.db_name = ""
        self.input = table
        self.row_id = table.row_id
        return self

    def setDistributed(self, group: Any = True, device_index: Optional[int] = None) -> "RepairModel":
        """Row-sharded run over the ranks of a ``torch.distributed`` process group (one process per GPU,
        NCCL): every rank passes ITS rows to ``setInput`` and gets the repairs of its rows back.  The
        shards exchange dictionaries once at ingest and count tensors (one collective per pass phase)
        during detection; models are trained on the same global sample on every rank, so the union of
        the per-rank results equals the one-GPU result (not part of the reference API)."""
        self.distributed = group
        if device_index is not None:
            self.device_index = int(device_index)
        return self

    @argtype_check
    def setRowId(self, row_id: str) -> "RepairModel":
        if not row_id:
            raise ValueError("`row_id` should have at least character")
        self.row_id = row_id
        return self

    @argtype_check
    def setTargets(self, attrs: List[str]) -> "RepairModel":
        if len(attrs) == 0:
            raise ValueError("`attrs` should have at least one attribute")
        self.targets = attrs
        return self

    @argtype_check
    def setErrorCells(self, error_cells: Union[str, DataFrame]) -> "RepairModel":
        if type(error_cells) is str and not error_cells:
            raise ValueError("`error_cells` should have at least character")
        if self.row_id is None:
            raise ValueError("`setRowId` should be called before specifying error cells")
        df = error_cells if isinstance(error_cells, DataFrame) else catalog.table(str(error_cells))
        if not all(c in df.columns for c in [str(self.row_id), "attribute"]):
            raise ValueError("Error cells should have `{}` and `attribute` in columns".format(self.row_id))
        self.error_cells = error_cells
        return self

    @argtype_check
    def setErrorDetectors(self, detectors: List[ErrorDetector]) -> "RepairModel":
        self.error_detectors = detectors
        return self

    @argtype_check
    def setDiscreteThreshold(self, thres: int) -> "RepairModel":
        if int(thres) < 2:
            raise ValueError("`thres` should be bigger than 1, got {}".format(thres))
        self.discrete_thres = thres
        return self

    @argtype_check
    def setParallelStatTrainingEnabled(self, enabled: bool) -> "RepairModel":
        self.parallel_stat_training_enabled = enabled
        return self

    @argtype_check
    def setTrainingDataRebalancingEnabled(self, enabled: bool) -> "RepairModel":
        self.training_data_rebalancing_enabled = enabled
        return self

    @argtype_check
    def setRepairByRules(self, enabled: bool) -> "RepairModel":
        self.repair_by_rules = enabled
        return self

    @argtype_check
    def setRepairDelta(self, delta: int) -> "RepairModel":
        if delta <= 0:
            raise ValueError("Repair delta should be positive, got {}".format(delta))
        self.repair_delta = int(delta)
        return self

    @argtype_check
    def setUpdateCostFunction(self, cf: UpdateCostFunction) -> "RepairModel":
        self.cf = cf
        return self

    @argtype_check
    def option(self, key: str, value: str) -> "RepairModel":
        if key not in self.option_keys:
            raise ValueError("Non-existent key specified: key={}".format(key))
        self.opts[key] = value
        return self

    # ---- helpers ---------------------------------------------------------------------------------
    def _opt(self, key):
        return get_option_value(self.opts, *_MODEL_OPT[key])

    @property
    def _repair_by_nearest_values_enabled(self) -> bool:
        return not bool(self._opt("model.rule.repair_by_nearest_values.disabled")) \
            and self.repair_by_rules and self.cf is not None

    def _resolve_input(self):
        if isinstance(self.input, str):
            name = "{}.{}".format(self.db_name, self.input) if self.db_name else self.input
            return _as_encoded(catalog.table(name), str(self.row_id), name), name
        return _as_encoded(self.input, str(self.row_id)), "input"

    def _given_cells(self, table):
        """setErrorCells frame -> (row positions, attrs) restricted like errors.py:434-446."""
        if self.error_cells is None:
            return None
        df = self.error_cells if isinstance(self.error_cells, DataFrame) else catalog.table(str(self.error_cells))
        keep = set(self.targets) if self.targets else set(table.names) | {table.row_id}
        attr = df["attribute"].to_numpy(dtype=object)
        pos, found = row_positions(table.row_ids, df[str(self.row_id)].to_numpy())
        ok = found & np.array([a in keep and a in table.by_name for a in attr.tolist()], dtype=bool)
        return pos[ok].tolist(), attr[ok].tolist()

    # ---- run -------------------------------------------------------------------------------------
    def run(self, detect_errors_only: bool = False, compute_repair_candidate_prob: bool = False,
            compute_repair_prob: bool = False, compute_repair_score: bool = False,
            repair_data: bool = False, maximal_likelihood_repair: bool = False) -> DataFrame:
        if self.input is None or self.row_id is None:
            raise ValueError("`setInput` and `setRowId` should be called before repairing")
        if maximal_likelihood_repair and self.repair_delta is None:
            raise ValueError("`setRepairDelta` should be called when enabling maximal likelihood repairing")
        if maximal_likelihood_repair and self.cf is None:
            raise ValueError("`setUpdateCostFunction` should be called when enabling maximal likelihood repairing")
        if maximal_likelihood_repair and len(self.cf.targets) > 0:  # type: ignore
            raise ValueError("`UpdateCostFunction.targets` cannot be used when enabling "
                             "maximal likelihood repairing")
        exclusive = [("detect_errors_only", detect_errors_only),
                     ("compute_repair_candidate_prob", compute_repair_candidate_prob),
                     ("compute_repair_prob", compute_repair_prob),
                     ("compute_repair_score", compute_repair_score),
                     ("repair_data", repair_data)]
        chosen = [n for n, v in exclusive if v]
        if len(chosen) > 1:
            raise ValueError("{} cannot be set to true simultaneously".format(to_list_str(chosen, sep="/", quote=True)))
        if self._repair_by_nearest_values_enabled and \
                (maximal_likelihood_repair or compute_repair_candidate_prob or compute_repair_prob
                 or compute_repair_score):
            raise ValueError("Cannot repair data by nearest values when enabling "
                             "`maximal_likelihood_repair`, `compute_repair_candidate_prob`, "
                             "`compute_repair_prob`, or `compute_repair_score`")
        if compute_repair_prob or compute_repair_score:
            compute_repair_candidate_prob = True
        if compute_repair_score:
            maximal_likelihood_repair = True

        t0 = time.time()
        from ._native import Context
        from .engine import Dist, Engine
        ctx = dt = table = None
        launches0 = 0
        ingest: Dict[str, Any] = {}
        arrow_io = _is_arrow_table(self.input)
        if arrow_io:
            # raw Arrow buffers -> device, encoded there (no per-row host work); None = needs the host path
            import torch
            ctx = Context.acquire(self.device_index)
            launches0 = ctx.launch_count
            try:
                got = EncodedTable.from_arrow_device(self.input, str(self.row_id), ctx,
                                                     torch.device("cuda", self.device_index), timings=ingest)
            except Exception:
                Context.release(ctx)
                raise
            if got is not None:
                table, dt = got
                input_name = "input"
        if table is None:
            table, input_name = self._resolve_input()
        ingest.setdefault("ingest_total_s", time.time() - t0)
        continuous = table.continuous_attrs
        _logger.info("input_table: {} ({} rows x {} columns)".format(input_name, table.n_rows, len(table.columns)))
        if maximal_likelihood_repair and len(continuous) != 0:
            raise ValueError("Cannot enable the maximal likelihood repair mode when continous attributes found")
        if self.targets and len(set(self.targets) & (set(table.names) | {table.row_id})) == 0:
            raise ValueError("Target attributes not found in {}: {}".format(input_name, to_list_str(self.targets)))
        err_opts = ErrorModelOptions.resolve(self.opts)
        validate_options(self.opts)
        for key in _MODEL_OPT:
            self._opt(key)

        dist = None
        if self.distributed is not None and self.distributed is not False:
            dist = Dist(None if self.distributed is True else self.distributed)
            table = table.unify(dist, dt, ctx)
        engine = Engine(table, self.device_index, dist=dist, device_table=dt, ctx=ctx)
        ingest["engine_ready_s"] = time.time() - t0
        try:
            detectors = self.error_detectors or default_detectors(self.targets, table.names)
            _logger.info("[Error Detection Phase] Used error detectors: {}".format(to_list_str(detectors)))
            res = engine.detect([d.spec() for d in detectors], self.targets, self.discrete_thres, err_opts,
                                self._given_cells(table))
            self.last_run = {"detect": res, "elapsed_detect": time.time() - t0}
            self.last_run.update(ingest)
            self.last_run["detect_done_s"] = time.time() - t0
            if detect_errors_only:
                return _maybe_arrow(self._cells_frame(engine, table, res), arrow_io)
            if sum((res.n_cells_global or res.n_cells).values()) == 0:
                _logger.info("Any error cell not found, so the input data is already clean")
                return _maybe_arrow(self._input_frame(table) if repair_data else
                                    self._empty_frame(table, repaired=True), arrow_io)
            if len(res.target_columns) == 0:
                raise ValueError("At least one valid discretizable feature is needed to repair error cells, "
                                 "but no such feature found")
            if compute_repair_candidate_prob or maximal_likelihood_repair:
                out = self._run_pmf_modes(engine, table, res, continuous, compute_repair_prob, compute_repair_score,
                                          repair_data, maximal_likelihood_repair)
            elif arrow_io and not repair_data and not self.repair_by_rules and not engine.dt.cont_index:
                # Arrow in, Arrow out: the frame is assembled from device-side arrays, no Python object per cell
                t1 = time.time()
                models = self.frozen_models if self.frozen_models is not None else \
                    build_models(self, engine, table, res, continuous)
                self.last_run["models"] = models
                self.last_run["elapsed_training"] = time.time() - t1
                out = repair_cells_encoded(self, engine, table, res, models, arrow=True)
                self.last_run["repair_done_s"] = time.time() - t0
            else:
                out = repair_cells(self, engine, table, res, continuous, repair_data, models=self.frozen_models)
            _logger.info("!!!Total Processing time is {}(s)!!!".format(time.time() - t0))
            return _maybe_arrow(out, arrow_io)
        finally:
            self.last_run["gpu_launches"] = engine.launches + (engine._launches0 - launches0 if ctx is not None else 0)
            engine.close()
            self.last_run["total_s"] = time.time() - t0

    # ---- pmf / score / maximal-likelihood modes (model.py:1350-1390) -------------------------------
    def _run_pmf_modes(self, engine, table, res, continuous, compute_repair_prob, compute_repair_score,
                       repair_data, maximal_likelihood_repair):
        from . import pmf as P
        cells = repair_cells_pmf(self, engine, table, res, continuous)
        opts = {k: self._opt(k) for k in ("repair.pmf.cost_weight", "repair.pmf.prob_threshold",
                                          "repair.pmf.prob_top_k")}
        shaped = P.shape_pmf(cells, opts, self.cf)
        rid = table.row_id
        if not maximal_likelihood_repair:
            if compute_repair_prob:
                return DataFrame({rid: [c[0] for c in shaped], "attribute": [c[1] for c in shaped],
                                  "current_value": pd.array([c[2][0] for c in shaped], dtype=object),
                                  "repaired": pd.array([c[3][0][0] if c[3] else None for c in shaped], dtype=object),
                                  "prob": [c[3][0][1] if c[3] else None for c in shaped]})
            return DataFrame({rid: [c[0] for c in shaped], "attribute": [c[1] for c in shaped],
                              "current_value": pd.array([c[2][0] for c in shaped], dtype=object),
                              "pmf": [[{"class": k, "prob": p} for k, p in c[3]] for c in shaped]})
        assert self.cf is not None
        scored = P.compute_score(shaped, self.cf)
        if compute_repair_score:
            return DataFrame({rid: [c[0] for c in scored], "attribute": [c[1] for c in scored],
                              "current_value": pd.array([c[2] for c in scored], dtype=object),
                              "repaired": pd.array([c[3] for c in scored], dtype=object),
                              "score": [c[4] for c in scored]})
        top = P.maximal_likelihood_repair(scored, int(self.repair_delta))
        if repair_data:
            frame = self._input_frame(table)
            pos, _ = row_positions(table.row_ids, [r for r, _, _, _ in top])
            by_attr: Dict[str, Any] = {}
            for p_, (_, a, _, rep) in zip(pos.tolist(), top):
                by_attr.setdefault(a, []).append((p_, rep))
            for a, cells in by_attr.items():
                col = frame[a].to_numpy(dtype=object, copy=True)
                for p_, rep in cells:
                    col[p_] = rep
                frame[a] = col
            return frame
        return DataFrame({rid: [c[0] for c in top], "attribute": [c[1] for c in top],
                          "current_value": pd.array([c[2] for c in top], dtype=object),
                          "repaired": pd.array([c[3] for c in top], dtype=object)})

    # ---- frames ----------------------------------------------------------------------------------
    def _empty_frame(self, table, repaired=False):
        cols = [table.row_id, "attribute", "current_value"] + (["repaired"] if repaired else [])
        return DataFrame({c: [] for c in cols})

    def _input_frame(self, table):
        data = {table.row_id: table.row_ids}
        for c in table.columns:
            if c.continuous:
                data[c.name] = c.values if c.kind == "float" else pd.array(
                    [None if v != v else int(v) for v in c.values], dtype="Int64")
            else:
                data[c.name] = c.decode(c.codes)
        return DataFrame(data)

    def _cells_frame(self, engine, table, res):
        ids, attrs, curs = [], [], []
        for a, rows, cur in engine.cells_of(res):
            ids.append(table.row_ids[rows])
            attrs += [a] * len(rows)
            curs += table.by_name[a].decode(cur)
        if not ids:
            return self._empty_frame(table)
        return DataFrame({table.row_id: np.concatenate(ids), "attribute": attrs,
                          "current_value": pd.array(curs, dtype=object)})


def _fit(rm, engine, encoders, codes, tile_col, features, dict_sizes, X, y_values, is_discrete, num_class, y=None):
    """Model producer: the GPU histogram GBDT (gbdt.py) when every feature is discrete, else
    scikit-learn's (train.py).  Both use the reference's fixed parameters (train.py:102-115) and the
    tuned ones found by search.py (train.py:133-229: TPE-style search under k-fold CV, budget options
    model.hp.* / model.cv.n_splits)."""
    from . import gbdt as G
    from . import search as HS
    from .train import _get, search_options
    binned = None
    if rm.trainer != "sklearn" and is_discrete:
        binned = G.bin_sample(encoders, {f: codes[:, tile_col[f]] for f in features}, dict_sizes)
    if binned is not None and int(binned[1].sum()) * 12 <= 200 * 1024:
        bins, n_bins, values = binned
        classes = sorted(set(int(v) for v in y_values.tolist()))
        y_idx = np.searchsorted(np.asarray(classes), y_values).astype(np.int64)
        balanced = _get(rm.opts, "model.lgb.class_weight") == "balanced"
        depth = _get(rm.opts, "model.lgb.max_depth")

        def train(params, rows=None):
            b, yi = (bins, y_idx) if rows is None else (np.ascontiguousarray(bins[rows]), y_idx[rows])
            w = G.class_weights(yi, len(classes), balanced)
            return G.train_gpu(engine.ctx, engine.device, b, n_bins, values, yi, len(classes), w,
                               _get(rm.opts, "model.lgb.n_estimators"), _get(rm.opts, "model.lgb.learning_rate"),
                               depth if depth > 0 else 31,
                               num_leaves=int(min(max(params["num_leaves"], 2), 32)),   # the trainer's node budget
                               min_data_in_leaf=int(max(params["min_child_samples"], 1)),
                               min_sum_hessian=float(params["min_child_weight"]),
                               reg_lambda=float(params["reg_lambda"]),
                               colsample_bytree=float(params["colsample_bytree"]),
                               subsample=float(params["subsample"]), subsample_freq=int(params["subsample_freq"]))

        max_evals, no_progress, timeout, n_splits = search_options(rm.opts)
        params = dict(HS.DEFAULTS)
        if max_evals > 1 and y is not None:
            folds = HS.cv_folds(y_idx, True, n_splits)
            tile = engine.torch.from_numpy(np.ascontiguousarray(codes, dtype=np.int32)).to(engine.device)
            K = codes.shape[1]

            def evaluate(p):
                scores = []
                for tr, va in folds:
                    spec = {"forest": train(p, tr), "encoders": encoders, "class_codes": classes, "integral": False}
                    dm = DeviceModel(spec, tile_col, dict_sizes, {}, engine.device)
                    work = tile.clone()
                    cells = engine.torch.from_numpy(np.ascontiguousarray(va, dtype=np.int32)).to(engine.device)
                    dm.predict(engine.ctx, work, K, None, 0, cells, len(va), tile_col[y])
                    pred = work[cells.to(engine.torch.int64), tile_col[y]].cpu().numpy()
                    scores.append(HS.score(y_values[va], pred, True))
                return -float(np.mean(scores)), [-float(v) for v in scores]

            params, _, n_eval = HS.search(evaluate, max_evals, no_progress, timeout)
            rm.last_run.setdefault("search", {})[y] = {"evals": n_eval, "params": params}
        return {"forest": train(params), "class_codes": classes}
    forest, classes = build_model(X, y_values, is_discrete, num_class, rm.opts)
    return None if forest is None else {"forest": forest, "class_codes": classes}


def _train_model(rm, engine, table, res, y, continuous, tile_col, fdeps=None):
    """Bookkeeping of _build_repair_models for one target (model.py:1001-1052, 768-815).
    -> ("const", code or None) | ("fd", x, lut, map) | ("forest", DeviceModel, info)"""
    col = table.by_name[y]
    is_discrete = not col.continuous
    input_columns = [c for c in table.names if c != y]
    if is_discrete:
        counts = np.asarray(engine.raw_value_counts(y), dtype=np.int64).copy()
        if y in res.bitmaps and (res.n_cells_global or res.n_cells).get(y, 0):
            masked = engine.torch.zeros(len(counts), dtype=engine.torch.int64, device=engine.device)
            if res.n_cells.get(y, 0):
                rows = engine.bitmap_rows(res.bitmaps[y])
                cur = engine.torch.empty(int(rows.numel()), dtype=engine.torch.int32, device=engine.device)
                engine.ctx.gather(engine.dt.col(y), rows, int(rows.numel()), cur)
                masked += engine.torch.bincount((cur + 1).to(engine.torch.int64), minlength=len(counts))
            engine.exchange([(masked, "sum")])
            counts -= masked.cpu().numpy()
        present = np.nonzero(counts[1:] > 0)[0]
        num_class = len(present)
        if num_class <= 1:
            return ("const", int(present[0]) if num_class == 1 else None)
    else:
        num_class = 0
    if fdeps is not None and y in fdeps:  # model.py:1018-1029: y follows a clean attribute by rule
        fx = [x for x in fdeps[y] if int(res.domain_stats[x]) < int(rm._opt("model.rule.max_domain_size"))]
        if fx:
            _logger.info("Building model... type=rule(FD: X->y) y={} X={}".format(y, fx[0]))
            return R.build_fd_model(engine, table, res, fx[0], y)
    features = select_features(res.pairwise_stats, y, input_columns, rm._opt("model.max_training_column_num"))
    rows_local, rows, n_valid = engine.valid_training_rows(res, y, rm._opt("model.max_training_row_num"))
    if n_valid == 0:
        return ("const", None)
    codes, vals = engine.sample_rows_masked(res, res.target_columns, rows_local)
    cont_idx = engine.dt.cont_index
    encoders = []
    dict_sizes = {c.name: c.dict_size for c in table.columns}
    for f in features:
        kind = encoder_type(f, continuous, res.domain_stats, rm._opt("model.small_domain_threshold"))
        e = {"attr": f, "type": kind}
        if kind != "cont":
            e["categories"] = first_seen(codes[:, tile_col[f]])
        encoders.append(e)
    if rm.training_data_rebalancing_enabled and is_discrete:
        # train.py:901-903: the classes of a discrete target are brought to the median class size before
        # training; like SMOTEN, every feature is taken as nominal (numeric ones by their distinct values)
        from .rebalance import rebalance
        fcols = [tile_col[f] for f in features]
        src, fcodes, y_new = rebalance(codes[:, fcols], codes[:, tile_col[y]])
        codes2 = np.full((len(src), codes.shape[1]), -1, dtype=codes.dtype)
        codes2[:, fcols] = fcodes
        codes2[:, tile_col[y]] = y_new
        if vals is not None:
            vals2 = np.full((len(src), vals.shape[1]), np.nan, dtype=np.float64)
            for f in features:
                if f in cont_idx:
                    d = np.r_[np.asarray(table.by_name[f].dictionary, dtype=np.float64), np.nan]
                    vals2[:, cont_idx[f]] = d[codes2[:, tile_col[f]]]      # code -1 -> NaN (last slot)
            vals = vals2
        codes = codes2
        rows = np.where(src >= 0, np.asarray(rows)[np.maximum(src, 0)], -1)   # -1 = synthetic row
    X = encode_matrix(encoders, {f: codes[:, tile_col[f]] for f in features},
                      {f: vals[:, cont_idx[f]] for f in features if f in cont_idx} if vals is not None else {},
                      dict_sizes)
    y_values = codes[:, tile_col[y]] if is_discrete else vals[:, cont_idx[y]]
    ctx = {"y": y, "features": features, "encoders": encoders, "X": X, "y_values": y_values,
           "is_discrete": is_discrete, "num_class": num_class, "train_rows": rows, "opts": rm.opts}
    _logger.info("Building model... type={} y={} features={} #rows={}".format(
        "classfier" if is_discrete else "regressor", y, to_list_str(features), len(rows)))
    if rm.model_provider is not None:
        spec = rm.model_provider(ctx)
    else:
        spec = _fit(rm, engine, encoders, codes, tile_col, features, dict_sizes, X, y_values, is_discrete, num_class, y)
    if spec is None:
        return ("const", None)
    if "const" in spec:
        return ("const", spec["const"])
    full = {"forest": spec["forest"], "encoders": encoders,
            "class_codes": [int(c) for c in spec["class_codes"]] if is_discrete else None,
            "integral": (not is_discrete) and col.kind == "int"}
    dm = DeviceModel(full, tile_col, dict_sizes, cont_idx, engine.device)
    return ("forest", dm, {"spec": full, "ctx": ctx})


def build_models(rm, engine, table, res, continuous):
    """Training phase: one model per target column, in target order (model.py:1001-1052)."""
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    fdeps = R.functional_deps(rm, table, res.target_columns)
    models = [(y, _train_model(rm, engine, table, res, y, continuous, tile_col, fdeps)) for y in res.target_columns]
    if any(m[0] == "fd" for _, m in models):
        models = R.resolve_prediction_order(models, res.target_columns)
    return models


def run_chain(engine, table, models, tile, ctile, D):
    """Repair phase proper: the sequential chain over the targets on the dirty-row tile, in place
    (the reference's `repair` pandas UDF, model.py:1096-1135)."""
    torch = engine.torch
    K = len(table.columns)
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    cont_idx = engine.dt.cont_index
    n_cc = len(cont_idx)
    words = (D + 31) // 32 + 1
    nullbits = torch.zeros(words, dtype=torch.int32, device=engine.device)
    # NULL cells of every discrete column in one pass (a model only fills its own column)
    all_null = engine.tile_nulls  # [K][words], produced by build_dirty_tile together with the tile
    assert tuple(all_null.shape) == (K, words)
    # a model only fills its own column, so the work-list sizes can all be taken now, in one round trip
    null_counts = engine.ctx.bitmap_count_many([all_null[i] for i in range(K)], D)
    engine.mark("chain:null bitmaps")
    # the work lists of all discrete targets in one batched compaction (three launches instead of 2-3 per model)
    disc = [y for y, _ in models if not table.by_name[y].continuous and null_counts[tile_col[y]] > 0]
    lists = {}
    if disc:
        sizes = [null_counts[tile_col[y]] for y in disc]
        flat = torch.empty(sum(sizes), dtype=torch.int32, device=engine.device)
        outs, o = [], 0
        for sz in sizes:
            outs.append(flat[o:o + sz])
            o += sz
        engine.ctx.bitmaps_to_rows_many([all_null[tile_col[y]] for y in disc], D, outs, sizes)
        lists = dict(zip(disc, outs))
    empty = torch.zeros(0, dtype=torch.int32, device=engine.device)
    for y, m in models:
        ycol = table.by_name[y]
        if ycol.continuous:
            engine.ctx.tile_null_bitmap(ctile, D, n_cc, cont_idx[y], nullbits, f64=True)
            todo = engine.bitmap_rows(nullbits, D)
        else:
            todo = lists.get(y, empty)
        n = int(todo.numel())
        engine.mark("chain:cells of " + y)
        if n == 0:
            continue
        if m[0] == "const":
            if m[1] is not None and not ycol.continuous:
                engine.ctx.tile_fill(tile, K, tile_col[y], todo, n, int(m[1]))
            continue
        if m[0] == "fd":  # FunctionalDepModel.predict (model.py:86-87)
            engine.ctx.tile_lut_fill(tile, K, tile_col[m[1]], tile_col[y], todo, n, m[2], int(m[2].numel()))
            continue
        m[1].predict(engine.ctx, tile, K, ctile, n_cc, todo, n, cont_idx[y] if ycol.continuous else tile_col[y])
        engine.mark("chain:predict " + y)


def repair_cells_pmf(rm, engine, table, res, continuous):
    """pmf variant of the repair phase (model.py:1104-1128): discrete targets keep the class margins of
    every predicted cell, and the cell itself becomes "neither NULL nor a known category" for the
    later models (the reference parks a JSON string there).
    -> [(row id, attribute, current_value, classes or None, probs or value string)]"""
    _, undo = R.apply_rules(rm, engine, table, res) if rm.repair_by_rules else ([], [])  # model.py:1326-1328
    try:
        return _repair_cells_pmf(rm, engine, table, res, continuous)
    finally:
        R.restore(engine, undo)


def _repair_cells_pmf(rm, engine, table, res, continuous):
    from . import pmf as P
    torch = engine.torch
    targets = res.target_columns
    K = len(table.columns)
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    cont_idx = engine.dt.cont_index
    n_cc = len(cont_idx)
    cells = engine.cells_of(res, targets)
    if not cells:
        return []
    models = build_models(rm, engine, table, res, continuous)
    rm.last_run["models"] = models
    drows, tile, ctile = engine.build_dirty_tile(res, targets)
    D = int(drows.numel())
    words = (D + 31) // 32 + 1
    nullbits = torch.zeros(words, dtype=torch.int32, device=engine.device)
    all_null = engine.tile_nulls  # [K][words], produced by build_dirty_tile together with the tile
    assert tuple(all_null.shape) == (K, words)
    kept = {}
    for y, m in models:
        ycol = table.by_name[y]
        if ycol.continuous:
            engine.ctx.tile_null_bitmap(ctile, D, n_cc, cont_idx[y], nullbits, f64=True)
            todo = engine.bitmap_rows(nullbits, D)
            if int(todo.numel()) and m[0] == "forest":
                m[1].predict(engine.ctx, tile, K, ctile, n_cc, todo, int(todo.numel()), cont_idx[y])
            continue
        todo = engine.bitmap_rows(all_null[tile_col[y]], D)
        n = int(todo.numel())
        if n == 0:
            continue
        if m[0] == "const":
            kept[y] = (todo.cpu().numpy(), None, [m[1]])
        elif m[0] == "fd":  # FunctionalDepModel.predict_proba (model.py:89-100): one-hot, or nothing
            xs = torch.empty(n, dtype=torch.int32, device=engine.device)
            engine.ctx.tile_gather(tile, K, tile_col[m[1]], todo, n, xs)
            pred = torch.empty(n, dtype=torch.int32, device=engine.device)
            # an x that is itself a parked pmf cell (code = dict size) maps to nothing
            engine.ctx.gather(m[2][1:], torch.where(xs < int(m[2].numel()) - 1, xs, torch.full_like(xs, -1)), n, pred)
            kept[y] = (todo.cpu().numpy(), ("onehot", pred.cpu().numpy()), sorted(set(m[3].values())))
        else:
            dm = m[1]
            margins = torch.empty((n, dm.n_seq), dtype=torch.float64, device=engine.device)
            dm.predict(engine.ctx, tile, K, ctile, n_cc, todo, n, tile_col[y], margins)
            kept[y] = (todo.cpu().numpy(), margins.cpu().numpy(), m[2]["spec"]["class_codes"])
        engine.ctx.tile_fill(tile, K, tile_col[y], todo, n, ycol.dict_size)  # unknown category from here on
    out = []
    for a, rows, cur in cells:
        col = table.by_name[a]
        d_rows = torch.from_numpy(rows.astype(np.int32)).to(engine.device)
        dpos = torch.empty(len(rows), dtype=torch.int32, device=engine.device)
        engine.ctx.lookup_sorted(drows, D, d_rows, len(rows), dpos)
        ids = table.row_ids[rows].tolist()
        cur_s = col.decode(cur)
        if col.continuous:
            vals = torch.empty(len(rows), dtype=torch.float64, device=engine.device)
            engine.ctx.tile_gather(ctile, n_cc, cont_idx[a], dpos, len(rows), vals, f64=True)
            for i, v in enumerate(vals.cpu().numpy().tolist()):
                out.append((ids[i], a, cur_s[i], None, cell_to_string(col.kind, v)))
            continue
        todo_h, margins_h, class_codes = kept[a]
        at = np.searchsorted(todo_h, dpos.cpu().numpy())
        if margins_h is None:
            classes = [None if class_codes[0] is None else col.strings()[class_codes[0]]]
            for i in range(len(rows)):
                out.append((ids[i], a, cur_s[i], classes, [1.0]))
        elif isinstance(margins_h, tuple):
            strs = col.strings()
            classes = [strs[c] for c in class_codes]
            for i, p in enumerate(margins_h[1][at].tolist()):
                if p < 0:
                    out.append((ids[i], a, cur_s[i], [], []))
                else:
                    out.append((ids[i], a, cur_s[i], classes, [1.0 if c == p else 0.0 for c in class_codes]))
        else:
            probs = P.probabilities(margins_h[at])
            strs = col.strings()
            classes = [strs[c] for c in class_codes]
            for i in range(len(rows)):
                out.append((ids[i], a, cur_s[i], classes, probs[i].tolist()))
    return out


def _arrow_cells_frame(engine, table, seg, idx, n_keep, rows_all, cur_all, rep_all):
    """The filtered (row id, attribute, current_value, repaired) frame as a ``pyarrow.Table`` built from
    device-side arrays: row ids gathered on the device, dictionary indices + Arrow validity bits copied
    into fresh host buffers (dr_d2h_copy) that the Arrow arrays wrap without another copy; string
    columns are dictionary arrays over the column dictionaries (one chunk per attribute)."""
    import pyarrow as pa
    torch = engine.torch
    dev = engine.device
    m = max(n_keep, 1)
    words = (m + 31) // 32
    rows_k = torch.empty(m, dtype=torch.int32, device=dev)
    codes_k = torch.empty((2, m), dtype=torch.int32, device=dev)
    bits_k = torch.zeros((2, words), dtype=torch.int32, device=dev)
    ids_k = None
    if n_keep:
        engine.ctx.gather(rows_all, idx, n_keep, rows_k)
        engine.ctx.gather(cur_all, idx, n_keep, codes_k[0])
        engine.ctx.gather(rep_all, idx, n_keep, codes_k[1])
        engine.ctx.valid_bits(codes_k[0], n_keep, bits_k[0])
        engine.ctx.valid_bits(codes_k[1], n_keep, bits_k[1])
        if engine.dt.ids is not None:
            ids_k = torch.empty(m, dtype=torch.int64, device=dev)
            engine.ctx.gather_i64(engine.dt.ids, rows_k, n_keep, ids_k)
    # where each attribute's cells start among the kept ones
    starts = torch.tensor([o for _, o, _ in seg] + [sum(n for _, _, n in seg)], dtype=torch.int32, device=dev)
    bounds = torch.searchsorted(idx[:n_keep].contiguous(), starts).cpu().numpy() if n_keep else \
        np.zeros(len(seg) + 1, dtype=np.int64)
    h_codes = np.empty((2, m), dtype=np.int32)
    h_bits = np.empty((2, words), dtype=np.uint32)
    src, dst, size = [codes_k, bits_k], [h_codes.ctypes.data, h_bits.ctypes.data], [h_codes.nbytes, h_bits.nbytes]
    if ids_k is not None:
        h_ids = np.empty(m, dtype=np.int64)
        src.append(ids_k); dst.append(h_ids.ctypes.data); size.append(h_ids.nbytes)
    else:
        h_rows = np.empty(m, dtype=np.int32)
        src.append(rows_k); dst.append(h_rows.ctypes.data); size.append(h_rows.nbytes)
    engine.ctx.d2h_copy(src, dst, size)
    if ids_k is None:
        h_ids = np.asarray(table.row_ids)[h_rows[:n_keep].astype(np.int64)]
    ids = pa.array(h_ids[:n_keep])
    big = [pa.Array.from_buffers(pa.int32(), n_keep, [pa.py_buffer(h_bits[j]), pa.py_buffer(h_codes[j])])
           for j in range(2)]
    names = pa.array([a for a, _, _ in seg], type=pa.string())
    attr, cur, rep = [], [], []
    for i, ((a, _, _), lo, hi) in enumerate(zip(seg, bounds[:-1], bounds[1:])):
        lo, hi = int(lo), int(hi)
        if hi == lo:
            continue
        strs = pa.array(table.by_name[a].strings(), type=pa.string())
        attr.append(pa.DictionaryArray.from_arrays(pa.array(np.full(hi - lo, i, dtype=np.int32)), names, safe=False))
        cur.append(pa.DictionaryArray.from_arrays(big[0].slice(lo, hi - lo), strs, safe=False))
        rep.append(pa.DictionaryArray.from_arrays(big[1].slice(lo, hi - lo), strs, safe=False))
    if not cur:
        empty = pa.array([], type=pa.string())
        return pa.table({table.row_id: ids, "attribute": empty, "current_value": empty, "repaired": empty})
    # (one chunk per attribute in every column: chunk layouts must agree)
    offs = [0] + [int(b) for b in np.cumsum([len(c) for c in cur])]
    id_chunks = [ids.slice(lo, hi - lo) for lo, hi in zip(offs[:-1], offs[1:])]
    return pa.table({table.row_id: pa.chunked_array(id_chunks), "attribute": pa.chunked_array(attr),
                     "current_value": pa.chunked_array(cur), "repaired": pa.chunked_array(rep)})


def repair_cells_encoded(rm, engine, table, res, models, arrow=False):
    """Default-mode repair of an all-discrete table with frozen models, everything device-side:
    -> [(attr, row positions int32, current codes, repaired codes)] already filtered like
    model.py:1401.  One D2H of the result at the end (pinned), no per-attribute host round trips.
    arrow: -> the same frame as a ``pyarrow.Table`` (_arrow_cells_frame)."""
    torch = engine.torch
    targets = res.target_columns
    K = len(table.columns)
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    attrs = [a for a in table.names if a in targets and res.n_cells.get(a, 0) > 0]
    E = sum(res.n_cells[a] for a in attrs)
    rm.last_run["n_error_cells"] = E
    if E == 0:
        rm.last_run["n_dirty_rows"] = 0
        if arrow:
            import pyarrow as pa
            return pa.Table.from_pandas(rm._empty_frame(table, repaired=True), preserve_index=False)
        return []
    engine.mark("repair:start")
    rows_all = torch.empty(E, dtype=torch.int32, device=engine.device)
    cur_all = torch.empty(E, dtype=torch.int32, device=engine.device)
    rep_all = torch.empty(E, dtype=torch.int32, device=engine.device)
    seg, off = [], 0
    for a in attrs:
        seg.append((a, off, res.n_cells[a]))
        off += res.n_cells[a]
    engine.ctx.bitmaps_to_rows_many([res.bitmaps[a] for a in attrs], engine.n_rows,
                                    [rows_all[o:o + n] for _, o, n in seg], [n for _, _, n in seg])
    for a, o, n in seg:
        engine.ctx.gather(engine.dt.col(a), rows_all[o:o + n], n, cur_all[o:o + n])
    engine.mark("repair:cell lists")
    drows, tile, ctile = engine.build_dirty_tile(res, targets)
    D = int(drows.numel())
    rm.last_run["n_dirty_rows"] = D
    engine.mark("repair:dirty tile")
    chain = [(y, m) for y, m in models if y in targets]
    run_chain(engine, table, chain, tile, ctile, D)
    engine.mark("repair:chain")
    # kept until the next pass for after-the-fact checks (bench.py --verify): the filled tile, its rows,
    # the NULL state of every tile column BEFORE the chain and the order the models ran in
    engine.last_repair = {"tile": tile, "drows": drows, "D": D, "nulls": engine.tile_nulls,
                          "chain": [y for y, _ in chain]}
    dpos = torch.empty(E, dtype=torch.int32, device=engine.device)
    engine.ctx.lookup_sorted(drows, D, rows_all, E, dpos)
    for a, o, n in seg:
        engine.ctx.tile_gather(tile, K, tile_col[a], dpos[o:o + n], n, rep_all[o:o + n])
    keep = torch.zeros((E + 31) // 32 + 1, dtype=torch.int32, device=engine.device)
    engine.ctx.changed_bitmap(cur_all, rep_all, E, keep)
    idx = engine.bitmap_rows(keep, E)
    n_keep = int(idx.numel())
    if arrow:
        t_e = time.time()
        frame = _arrow_cells_frame(engine, table, seg, idx, n_keep, rows_all, cur_all, rep_all)
        rm.last_run["egress_s"] = time.time() - t_e
        rm.last_run["n_out_cells"] = n_keep
        return frame
    host = engine.pinned_i32(4 * max(n_keep, 1)).view(4, max(n_keep, 1))  # reused across runs
    packed = torch.empty((4, max(n_keep, 1)), dtype=torch.int32, device=engine.device)
    if n_keep:
        packed[0, :n_keep].copy_(idx)
        engine.ctx.gather(rows_all, idx, n_keep, packed[1])
        engine.ctx.gather(cur_all, idx, n_keep, packed[2])
        engine.ctx.gather(rep_all, idx, n_keep, packed[3])
    engine.mark("repair:collect")
    host.copy_(packed, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    engine.mark("repair:d2h")
    h = host.numpy()
    out = []
    # (int32 needles: a wider type would make numpy convert the whole 10^7-element haystack first)
    bounds = np.searchsorted(h[0, :n_keep], np.asarray([o for _, o, _ in seg] + [E], dtype=np.int32))
    # The arrays are copies unless the caller asked to borrow the engine's pinned staging buffer
    # (rm.borrow_encoded_output: valid until the next pass on the same engine -- bench.py's timed loop).
    borrow = getattr(rm, "borrow_encoded_output", False)
    for (a, _, _), lo, hi in zip(seg, bounds[:-1], bounds[1:]):
        part = (h[1, lo:hi], h[2, lo:hi], h[3, lo:hi])
        out.append((a,) + (part if borrow else tuple(np.array(x) for x in part)))
    return out


def repair_cells(rm, engine, table, res, continuous, repair_data=False, models=None, encoded_output=False):
    """Phases 2-3 of RepairModel._run (model.py:1311-1408) on the device.

    models: frozen output of build_models (skips the training phase).
    encoded_output: return [(attr, row positions, current codes, repaired codes)] -- the
    (tid, attribute, current_value, repaired) frame in dictionary-encoded form, already filtered --
    instead of materialising Python strings."""
    torch = engine.torch
    targets = res.target_columns
    K = len(table.columns)
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    cont_idx = engine.dt.cont_index
    if encoded_output and models is not None and not engine.dt.cont_index:
        return repair_cells_encoded(rm, engine, table, res, models)
    by_rules, undo = R.apply_rules(rm, engine, table, res) if rm.repair_by_rules else ([], [])  # model.py:1326-1328
    try:
        return _repair_cells(rm, engine, table, res, continuous, repair_data, models, encoded_output, by_rules)
    finally:
        R.restore(engine, undo)


def _rule_repairs_frame(table, by_rules):
    """Cells decided by a rule as output rows: appended unfiltered (model.py:1403-1404)."""
    ids, attrs, curs, reps = [], [], [], []
    for a, rows, old, new in by_rules:
        col = table.by_name[a]
        ids.append(table.row_ids[rows])
        attrs += [a] * len(rows)
        curs += col.decode(old)
        reps += col.decode(new)
    return DataFrame({table.row_id: np.concatenate(ids) if ids else [], "attribute": attrs,
                      "current_value": pd.array(curs, dtype=object), "repaired": pd.array(reps, dtype=object)})


def _repair_cells(rm, engine, table, res, continuous, repair_data, models, encoded_output, by_rules):
    torch = engine.torch
    targets = res.target_columns
    K = len(table.columns)
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    cont_idx = engine.dt.cont_index
    cells = engine.cells_of(res, targets)           # (attr, rows, current codes), table order
    if not cells and engine.dist is None:           # (a shard without cells still takes part in the training collectives)
        if by_rules and not repair_data:
            return _rule_repairs_frame(table, by_rules)
        if by_rules:
            return _apply_repairs(rm, table, _rule_cells_for_apply(table, by_rules))
        return rm._input_frame(table) if repair_data else rm._empty_frame(table, repaired=True)
    # models (training phase)
    t0 = time.time()
    if models is None:
        models = build_models(rm, engine, table, res, continuous)
        rm.last_run["models"] = models
        rm.last_run["elapsed_training"] = time.time() - t0
    models = [(y, m) for y, m in models if y in targets]
    # repair phase: sequential chain over the targets on the dirty-row tile
    t0 = time.time()
    drows, tile, ctile = engine.build_dirty_tile(res, targets)
    D = int(drows.numel())
    n_cc = len(cont_idx)
    run_chain(engine, table, models, tile, ctile, D)
    # output: (row id, attribute, current_value, repaired) for the error cells
    ids, attrs, curs, reps = [], [], [], []
    repaired_cells = []
    for a, rows, cur in cells:
        col = table.by_name[a]
        d_rows = torch.from_numpy(rows.astype(np.int32)).to(engine.device)
        dpos = torch.empty(len(rows), dtype=torch.int32, device=engine.device)
        engine.ctx.lookup_sorted(drows, D, d_rows, len(rows), dpos)
        if encoded_output and not col.continuous:
            out = torch.empty(len(rows), dtype=torch.int32, device=engine.device)
            engine.ctx.tile_gather(tile, K, tile_col[a], dpos, len(rows), out)
            codes = out.cpu().numpy()
            keep = (codes < 0) | (codes != cur)
            repaired_cells.append((a, rows[keep], cur[keep], codes[keep]))
            continue
        cur_s = col.decode(cur)
        if col.continuous:
            out = torch.empty(len(rows), dtype=torch.float64, device=engine.device)
            engine.ctx.tile_gather(ctile, n_cc, cont_idx[a], dpos, len(rows), out, f64=True)
            vals = out.cpu().numpy()
            rep_s = [cell_to_string(col.kind, v) for v in vals.tolist()]
            repaired_cells.append((a, rows, vals))
        else:
            out = torch.empty(len(rows), dtype=torch.int32, device=engine.device)
            engine.ctx.tile_gather(tile, K, tile_col[a], dpos, len(rows), out)
            codes = out.cpu().numpy()
            rep_s = col.decode(codes)
            repaired_cells.append((a, rows, codes))
        ids.append(table.row_ids[rows])
        attrs += [a] * len(rows)
        curs += cur_s
        reps += rep_s
    rm.last_run["elapsed_repair"] = time.time() - t0
    rm.last_run["n_error_cells"] = sum(len(r) for _, r, _ in cells)
    rm.last_run["n_dirty_rows"] = D
    if encoded_output:
        return repaired_cells
    if repair_data:
        return _apply_repairs(rm, table, repaired_cells + _rule_cells_for_apply(table, by_rules))
    frame = DataFrame({table.row_id: np.concatenate(ids) if ids else table.row_ids[:0], "attribute": attrs,
                       "current_value": pd.array(curs, dtype=object), "repaired": pd.array(reps, dtype=object)})
    # repaired IS NULL OR NOT(current_value <=> repaired)   (model.py:1401)
    cur_a, rep_a = frame["current_value"].to_numpy(dtype=object), frame["repaired"].to_numpy(dtype=object)
    keep = np.array([r is None or c is None or c != r for c, r in zip(cur_a, rep_a)], dtype=bool)
    frame = frame[keep].reset_index(drop=True)
    if by_rules:
        frame = pd.concat([frame, _rule_repairs_frame(table, by_rules)], ignore_index=True)
    return frame


def _rule_cells_for_apply(table, by_rules):
    """(attr, rows, repaired) in the form _apply_repairs takes: codes for discrete attributes, values
    for numeric ones."""
    out = []
    for a, rows, _, new in by_rules:
        col = table.by_name[a]
        out.append((a, rows, np.asarray(col.dictionary, dtype=np.float64)[new] if col.continuous else new))
    return out


def _apply_repairs(rm, table, repaired_cells):
    """repair_data=True: the input table with every error cell replaced by its repair."""
    frame = rm._input_frame(table)
    for a, rows, vals in repaired_cells:
        col = table.by_name[a]
        series = frame[a].to_numpy(dtype=object, copy=True) if not col.continuous or col.kind == "int" \
            else frame[a].to_numpy(copy=True)
        if col.continuous:
            for r, v in zip(rows.tolist(), vals.tolist()):
                series[r] = (None if v != v else int(v)) if col.kind == "int" else v
        else:
            dec = col.decode(vals)
            for r, v in zip(rows.tolist(), dec):
                series[r] = v
        frame[a] = pd.array(series, dtype="Int64") if col.continuous and col.kind == "int" else series
    return frame


def detect_with(detector):
    """``ErrorDetector.setUp(...).detect()`` standalone (errors.py:78-82): -> (row_id, attribute)."""
    from .engine import Engine
    src = detector.qualified_input_name
    df = catalog.table(src) if isinstance(src, str) else src
    table = _as_encoded(df, detector.row_id)
    engine = Engine(table, 0)
    try:
        spec = dict(detector.spec())
        spec.pop("targets", None)  # already folded into _targets by setUp
        targets = [t for t in detector._targets if t in table.by_name]
        if not targets:
            return DataFrame({table.row_id: [], "attribute": []})
        engine.discretize(80)
        bitmaps, fused = {}, {}
        kind = spec["type"]
        if kind == "null":
            engine.detect_null(targets, bitmaps, fused)
            engine.scan_hist(list(fused.keys()), fused)
        elif kind == "regex":
            engine.detect_regex(spec["attr"], spec["regex"], targets, bitmaps)
        elif kind == "domain":
            if spec["attr"] in targets:
                rx = engine.domain_values_regex(spec["attr"], spec["values"], spec["autofill"],
                                                spec["min_count_thres"])
                if rx is not None:
                    engine.detect_regex(spec["attr"], rx, targets, bitmaps)
        elif kind == "constraint":
            engine.detect_constraints(spec["path"], spec["constraints"], targets, bitmaps)
        elif kind == "outlier":
            engine.detect_outliers(targets, bitmaps, spec.get("approx", False))
        elif kind == "lof":
            engine.detect_lof(targets, bitmaps)
        elif kind == "sklearn":
            engine.detect_sklearn(targets, bitmaps, spec["factory"])
        ids, attrs = [], []
        for a in table.names:
            if a in bitmaps:
                rows = engine.bitmap_rows(bitmaps[a]).cpu().numpy().astype(np.int64)
                ids.append(table.row_ids[rows])
                attrs += [a] * len(rows)
        if not attrs:
            return DataFrame({table.row_id: [], "attribute": []})
        return DataFrame({table.row_id: np.concatenate(ids), "attribute": attrs})
    finally:
        engine.close()
