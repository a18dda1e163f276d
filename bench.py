#!/usr/bin/env python
"""bench.py -- one "step" = one pass of the hot path (error detection -> attribute statistics ->
weak-label domain analysis -> repair-model inference -> (tid, attribute, current, repaired) frame) over
one synthetic N x K categorical table (config C4 of SURVEY.md section 8d).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--rows R] [--cols C] [--scaling strong|weak]
                  [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL).  Default = STRONG scaling: ONE R-row table,
rows sharded R/N per GPU (BASELINE config 4); --scaling weak keeps R rows per GPU.  The only exchange
is the packed count-tensor collective of each pass phase.  `value` times the pass with the shard
resident in HBM; `e2e` times RepairModel().setArrowInput(host table).run() -> host Arrow frame.
Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "spark-data-repair-plugin_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "rows scanned/sec through the full detect+stats+repair pass (cells repaired/sec alongside) " \
         "on synthetic N x K categorical table"
N_ESTIMATORS = 300  # train.py:54-56


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rows", type=int, default=100_000_000,
                    help="rows of the table (strong scaling: sharded over the GPUs; weak scaling: per GPU)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): ONE --rows table sharded rows/N per GPU (BASELINE config 4); "
                         "weak: --rows per GPU of a N x --rows table")
    ap.add_argument("--cols", type=int, default=32)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-rows", type=int, default=0,
                    help="rows of the CPU arm's sample (0 = as many as fit the time budget, 20k..200k)")
    ap.add_argument("--configs", default="auto",
                    help="extra wall-clock rows for BASELINE configs: comma list of c2,c3,c5, 'none', or 'auto' "
                         "(all three on a 1-GPU run of the default size)")
    ap.add_argument("--forests", default="trained", choices=["trained", "random"],
                    help="trained: dr_gbdt_train on the real 10k-row samples (default); random: random-init "
                         "forests of the same architecture")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-calls", action="store_true", help="print the per-call timing table to stderr")
    ap.add_argument("--no-verify", action="store_true",
                    help="skip the after-the-fact self-check of the last timed step (histograms, cell counts, "
                         "a seeded sample of repaired cells re-evaluated by the oracle's C forest)")
    ap.add_argument("--verify-cells", type=int, default=50000)
    ap.add_argument("--trace", action="store_true",
                    help="one extra step with device-synchronised split points of the repair phase on stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the frame of the last one as DIR/<name>.npy (float64; see "
                         "dump_outputs) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1 or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs writes the frame of the b200 arm on one GPU: --impl b200 --gpus 1, no torchrun")
    return args


# ---------------------------------------------------------------------------------------------
# model producer used by both arms: random-init forests of the reference's architecture
# (300 boosting rounds x one tree per class, depth <= 7, <= 31 leaves) on the REAL encoders of a
# real training sample -- no data of this size can be fitted inside the benchmark's time budget,
# and the timed region is inference only (SURVEY.md section 8d).
# ---------------------------------------------------------------------------------------------
def _thresholds_for(ctx):
    out = []
    for e in ctx["encoders"]:
        if e["type"] == "cont":
            out.append([0.0])
        elif e["type"] == "ordinal":
            k = len(e["categories"])
            out.append([-0.5] + [j + 0.5 for j in range(1, max(k, 2))])
        else:
            k = len(e["categories"])
            out += [[-0.5, 0.5]] * (k - 1 if k >= 2 else 0)
    return out


def random_forest_provider(n_iter):
    cache = {}

    def provider(ctx):
        from tools.randforest import random_forest
        n_feat = ctx["X"].shape[1]
        if ctx["is_discrete"]:
            classes = sorted(set(int(v) for v in np.asarray(ctx["y_values"]).tolist()))
            n_classes = len(classes)
        else:
            classes, n_classes = None, 1
        seed = sum(ord(ch) * (i + 1) for i, ch in enumerate(ctx["y"]))
        thr = _thresholds_for(ctx)
        key = (ctx["y"], n_feat, tuple(classes or ()), tuple(len(t) for t in thr))
        if key not in cache:  # building the forest is the model producer's cost, not inference
            cache[key] = random_forest(n_feat, n_classes, n_iter, thr, np.random.default_rng(seed), leaf_scale=0.05)
        return {"forest": cache[key], "class_codes": classes}
    return provider


def detector_specs(n_cols):
    from repair import synth
    specs = [{"type": "null"}]
    fds = synth.fd_constraints(n_cols)
    if fds:
        specs.append({"type": "constraint", "constraints": fds})
    return specs


# model.hp.max_evals=1: fixed parameters, no search -- SURVEY.md 8(d) "trained once per target ... with fixed params"
OPTS = {"error.pairwise_freq_ratio_threshold": "1.0", "model.hp.max_evals": "1"}


# ---------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port on a bounded sample of the same workload
# ---------------------------------------------------------------------------------------------
_ORACLE_RF = {}


def gpu_trained_specs(args):
    """The frozen models of the b200 arm for the CPU arm: same table, same detect pass, same global 10k-row
    training samples, same deterministic trainer (dr_gbdt_train) -> {target: model spec}.  Untimed setup;
    needs a GPU (the CPU arm falls back to random-init forests of the same architecture without one)."""
    import torch
    from repair import RepairModel, synth
    from repair.engine import Engine
    from repair.errors import ErrorModelOptions
    from repair.model import build_models
    from repair.table import DeviceTable, EncodedTable
    k = args.cols
    total_rows = args.rows if args.scaling == "strong" else args.rows * max(args.gpus, 1)
    device = torch.device("cuda", 0)
    spec = synth.SynthSpec.c4(total_rows, k)
    codes_dev = synth.generate_torch(spec, device, 0, total_rows)
    names = synth.column_names(k)
    table = EncodedTable.from_codes("tid", names, [np.zeros(0, dtype=np.int32)] * k, spec.dom,
                                    row_ids=np.arange(total_rows, dtype=np.int64))
    table.n_rows = table.n_rows_global = total_rows
    engine = Engine(table, 0, device_table=DeviceTable(table, device, codes=codes_dev))
    rm = RepairModel()
    rm.opts = dict(OPTS)
    res = engine.detect(detector_specs(k), [], 80, ErrorModelOptions.resolve(rm.opts))
    models = build_models(rm, engine, table, res, [])
    out = {y: (m[2]["spec"] if m[0] == "forest" else {"const": m[1]}) for y, m in models}
    engine.close()
    del engine, codes_dev, models
    torch.cuda.empty_cache()
    return out


def run_oracle_sample(n_rows, n_cols, n_iter, trained=None):
    """One pass of the oracle pipeline over the first `n_rows` rows of the C4 table.
    trained: {target: spec} of gpu_trained_specs -- the oracle then evaluates the SAME forests as the b200
    arm, under the encoders they were trained with; else random-init forests of the same architecture.
    -> (seconds, rows, error cells, seconds of the detect phase, threads used, repaired cells, fallbacks)"""
    from oracle import ckernels
    from oracle import forest as OF
    from oracle import repair as OR
    from oracle.table import OTable
    from repair import synth
    threads = 1
    if ckernels.available():
        OF.forest_margins = ckernels.forest_margins  # compiled, OpenMP; checked in tests/test_oracle_c.py
        threads = ckernels.use_all_cores()           # (torchrun exports OMP_NUM_THREADS=1)
    spec = synth.SynthSpec.c4(n_rows, n_cols)
    codes = synth.generate_numpy(spec)
    names = synth.column_names(n_cols)
    tbl = OTable(["tid"] + names, ["int"] + ["str"] * n_cols,
                 [np.arange(n_rows, dtype=np.float64)] + [c.astype(np.int64) for c in codes])
    rf = _ORACLE_RF.setdefault(n_iter, random_forest_provider(n_iter))  # forests are built once
    fallbacks = []

    def provider(ctx):
        t = (trained or {}).get(ctx["y"])
        if t is not None and "const" in t:
            return {"const": t["const"]}
        if t is not None:
            # (the sample may have seen fewer categories than the training sample of the full table -- e.g. no
            # NULL in a column -- which is harmless: the forest is evaluated under ITS encoders)
            same = len(t["encoders"]) == len(ctx["encoders"]) and all(
                pe["attr"] == oe["attr"] and pe["type"] == oe["type"] for pe, oe in zip(t["encoders"], ctx["encoders"]))
            if same:
                for pe, oe in zip(t["encoders"], ctx["encoders"]):   # the encoders the forest was trained with
                    if pe["type"] != "cont":
                        oe["categories"] = [None if c < 0 else int(c) for c in pe["categories"]]
                return {"forest": t["forest"], "classes": [int(c) for c in t["class_codes"]]}
            fallbacks.append(ctx["y"])   # different features / encoder types: random-init stand-in
        octx = dict(ctx)
        octx["encoders"] = [dict(e) for e in ctx["encoders"]]
        spec_ = rf(octx)
        return {"forest": spec_["forest"], "classes": spec_["class_codes"]}

    o_opts = {"error.pairwise_freq_ratio_threshold": 1.0}
    t0 = time.time()
    cells = OR.run(tbl, "tid", detector_specs(n_cols), None, 80, None, o_opts, provider, detect_errors_only=True)
    t_detect = time.time() - t0
    t0 = time.time()
    out = OR.run(tbl, "tid", detector_specs(n_cols), None, 80, None, o_opts, provider)
    t_full = time.time() - t0
    return t_full, n_rows, len(cells), t_detect, threads, len(out), fallbacks


def reference_arm(args):
    """The reference's CPU path (restated: oracle/, NumPy + OpenMP C) on a bounded sample of the b200 arm's
    workload: the first R rows of the same table, the same detectors and options, the same frozen forests.
    R is chosen so that the whole --steps/--warmup run stays within minutes; the pass has a fixed cost
    (pair statistics over the 32 x 31 attribute pairs), so a 10k-row pass is timed as well and the line
    reports the marginal rate of the linear fit next to the plain rows / seconds of the sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    trained, forests = None, "random-init (no GPU to train them on)"
    try:
        import torch
        if args.forests == "trained" and torch.cuda.is_available():
            t0 = time.time()
            trained = gpu_trained_specs(args)
            forests = "the b200 arm's frozen forests (dr_gbdt_train, {:.0f} s of untimed setup)".format(time.time() - t0)
    except Exception as e:  # noqa: BLE001
        forests = "random-init (training them failed: {}: {})".format(type(e).__name__, e)
    small = 10000
    run_oracle_sample(small, args.cols, N_ESTIMATORS, trained)          # untimed: builds / loads the forests
    t_small = run_oracle_sample(small, args.cols, N_ESTIMATORS, trained)[0]
    rows = args.ref_rows
    if rows <= 0:   # auto: as many rows as (steps + warmup) passes fit into ~3 minutes, assuming ~half of the
        budget = 180.0 / max(args.steps + args.warmup, 1)                # small pass is fixed cost
        rows = int(small * max(1.0, (budget - 0.5 * t_small) / max(0.5 * t_small, 1e-3)))
        rows = int(min(max(rows, 2 * small), 200000) // 1000 * 1000)
    times, info = [], None
    for i in range(args.warmup + args.steps):
        info = run_oracle_sample(rows, args.cols, N_ESTIMATORS, trained)
        if i >= args.warmup:
            times.append(info[0])
    t = float(np.mean(times))
    value = info[1] / t
    per_row = (t - t_small) / max(rows - small, 1)
    fixed = t_small - per_row * small
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "int32 codes / f64 margins", "data": "synthetic",
        "config": {"workload": "C4 synthetic: first {} rows (bounded sample) of the {}-row x {}-col table, 1% NULLs + 4 FD "
                               "denial constraints, NULL + Constraint detectors, pairwise_freq_ratio_threshold=1.0, "
                               "{}".format(info[1], args.rows, args.cols, forests),
                   "rows_total": args.rows, "rows_in_sample": info[1], "cols": args.cols},
        "cells_repaired_per_sec": info[2] / max(t - info[3], 1e-9),
        "rows_scanned_per_sec": info[1] / info[3],
        "fit": {"rows": [small, rows], "seconds": [t_small, t], "fixed_s": fixed,
                "marginal_rows_per_sec": (1.0 / per_row) if per_row > 0 else None,
                "note": "seconds(rows) = fixed_s + rows / marginal_rows_per_sec; extrapolated to the full table the "
                        "CPU pass tends to the marginal rate"},
        "targets_on_random_forests": info[6],
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": info[4], "kind": "port",
                         "sample": "first {} rows of the C4 table; oracle (NumPy + OpenMP C forest) full pass".format(
                             info[1])},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md): ONE
    `nvidia-smi -lms 200` process started before the region and stopped after it (spawning a process per
    sample from a parent with GBs of pinned memory stalls the launching thread for tens of ms)."""

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
            "clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            try:
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=5)
                rows = [[x.strip() for x in ln.split(",")] for ln in out.splitlines() if ln.strip()]
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}



# ---------------------------------------------------------------------------------------------
# --verify: after the timed region, re-derive what the last step produced by independent means
# ---------------------------------------------------------------------------------------------
def verify_step(engine, table, res, out, models, k, n_sample, dist, seed=12345):
    """Independent re-computation of the last pass (untimed):
      * every column histogram vs torch.bincount of the resident codes (all-reduced when sharded);
      * per-attribute error-cell counts (before the weak-label pruning) vs NULL counts + a torch
        restatement of the FD constraints (per-key min/max through scatter_reduce);
      * a seeded sample of the emitted repairs: the cell's feature vector as the chain saw it (later
        targets' error cells still NULL, earlier ones already filled) is encoded on the host and
        evaluated by the ORACLE's C forest (oracle/c, float64 thresholds, generic layout) -- label must
        equal the code the CUDA chain wrote.
    -> dict for the JSON line."""
    import torch
    from oracle import ckernels
    from repair import synth
    from repair.forest import encode_matrix
    dev = engine.device
    names = table.names
    n = engine.n_rows
    if ckernels.available():
        ckernels.use_all_cores()   # (torchrun exports OMP_NUM_THREADS=1; the rank is bound to its GPU's NUMA node)
    info = {"hist_columns_checked": 0, "hist_mismatches": 0, "cell_count_attrs_checked": 0,
            "cell_count_mismatches": 0, "cells_checked": 0, "mismatches": 0}
    # ---- histograms ----
    for a in names:
        col = engine.dt.col(a)[:n]
        d = table.by_name[a].dict_size
        h = torch.bincount((col + 1).to(torch.int64), minlength=d + 1)
        if dist is not None:
            dist.sum_(h)
        got = engine._hist_cache.get(a)
        info["hist_columns_checked"] += 1
        if got is None or not np.array_equal(np.asarray(got), h.cpu().numpy()):
            info["hist_mismatches"] += 1
    # ---- error-cell counts of the detect phase (local shard; the FD tables are global) ----
    flagged = {}
    fds = synth.fd_constraints(k)
    for stmt in [x for x in fds.split(";") if x]:
        xname, yname = stmt.split("->")
        x, y = engine.dt.col(xname)[:n], engine.dt.col(yname)[:n]
        dx = table.by_name[xname].dict_size
        key = (x + 1).to(torch.int64)
        lo = torch.full((dx + 1,), 2 ** 31 - 1, dtype=torch.int32, device=dev)
        hi = torch.full((dx + 1,), -2 ** 31, dtype=torch.int32, device=dev)
        lo.scatter_reduce_(0, key, y + 1, reduce="amin")
        hi.scatter_reduce_(0, key, y + 1, reduce="amax")
        if dist is not None:
            dist.min_(lo)
            dist.max_(hi)
        viol = (lo != hi)[key]
        for a in (xname, yname):
            flagged[a] = viol if a not in flagged else (flagged[a] | viol)
    for a in names:
        want = (engine.dt.col(a)[:n] < 0)
        if a in flagged:
            want = want | flagged[a]
        want = int(want.sum().item())
        info["cell_count_attrs_checked"] += 1
        if int(res.n_cells_detected.get(a, 0)) != want:
            info["cell_count_mismatches"] += 1
    # ---- sampled repairs through the oracle's forest ----
    lr = getattr(engine, "last_repair", None)
    if lr is None or not out or not ckernels.available():
        info["note"] = "no repaired cells to sample" if ckernels.available() else "oracle/c not built"
        return info
    chain = lr["chain"]
    pos_in_chain = {y: i for i, y in enumerate(chain)}
    tile_col = {c.name: i for i, c in enumerate(table.columns)}
    dict_sizes = {c.name: c.dict_size for c in table.columns}
    by_attr = {a: (rows, cur, rep) for a, rows, cur, rep in out}
    forest_of = {y: m for y, m in models if m[0] == "forest"}
    sizes = np.asarray([len(by_attr[a][0]) if a in forest_of and a in by_attr else 0 for a in names], dtype=np.int64)
    total = int(sizes.sum())
    if total == 0:
        return info
    rng = np.random.default_rng(seed)
    pick = np.sort(rng.choice(total, size=min(n_sample, total), replace=False))
    bounds = np.r_[0, np.cumsum(sizes)]
    drows = lr["drows"]
    K = len(names)
    for ai, a in enumerate(names):
        sel = pick[(pick >= bounds[ai]) & (pick < bounds[ai + 1])] - bounds[ai]
        if len(sel) == 0:
            continue
        rows, _, rep = by_attr[a]
        rows_s, rep_s = np.asarray(rows)[sel], np.asarray(rep)[sel]
        d_rows = torch.from_numpy(np.ascontiguousarray(rows_s, dtype=np.int32)).to(dev)
        dpos = torch.searchsorted(drows[:lr["D"]], d_rows).to(torch.int64)
        assert bool((drows[dpos] == d_rows).all())
        codes = lr["tile"][dpos].cpu().numpy().astype(np.int64)                    # [m, K] final tile rows
        was_null = ((lr["nulls"][:, dpos >> 5] >> (dpos & 31).to(torch.int32)) & 1).cpu().numpy().astype(bool)  # [K, m]
        assert np.array_equal(codes[:, tile_col[a]], rep_s.astype(np.int64))       # the frame reports the tile
        for c in names:   # state of the row when model `a` ran
            j = tile_col[c]
            if c == a or (c in pos_in_chain and pos_in_chain[c] > pos_in_chain[a]):
                codes[was_null[j], j] = -1
        spec = forest_of[a][2]["spec"]
        X = encode_matrix(spec["encoders"], {e["attr"]: codes[:, tile_col[e["attr"]]] for e in spec["encoders"]}, {},
                          dict_sizes)
        m = ckernels.forest_margins(spec["forest"], X)
        lab = (m[:, 0] > 0).astype(np.int64) if m.shape[1] == 1 else np.argmax(m, axis=1)
        want = np.asarray(spec["class_codes"], dtype=np.int64)[lab]
        info["cells_checked"] += int(len(sel))
        info["mismatches"] += int((want != rep_s.astype(np.int64)).sum())
    return info


DUMP_SAMPLE_ROWS = 1 << 22
DUMP_MAX_CELLS = 1_500_000   # 4 float64 arrays of 48 MB at most: a dump stays under 64 MB
DUMP_SEED = 20261017


def dump_outputs(path, out, names, dom, n_rows):
    """Writes the (tid, attribute, current_value, repaired) frame that one pass handed its caller, in
    dictionary codes (-1 = NULL), as float64 arrays under `path`:
      cells_per_attribute [K]          cells of the whole frame per attribute (table column order);
      current_hist, repaired_hist [K, max(dom) + 1]
                                       the whole frame's counts of each code per attribute (column 0 = NULL);
      tid, attribute, current_value, repaired [m]
                                       every cell of a fixed sample of DUMP_SAMPLE_ROWS table rows (drawn with
                                       DUMP_SEED, so the same for every run of the same --rows), ordered by
                                       (attribute, tid), at most DUMP_MAX_CELLS of them.
    Inputs are seeded, so two builds that compute the same frame write identical files."""
    os.makedirs(path, exist_ok=True)
    k, width = len(names), max(dom) + 1
    sampled = np.zeros(n_rows, dtype=bool)
    sampled[np.random.default_rng(DUMP_SEED).choice(n_rows, size=min(DUMP_SAMPLE_ROWS, n_rows), replace=False)] = True
    counts = np.zeros(k)
    cur_hist, rep_hist = np.zeros((k, width)), np.zeros((k, width))
    parts = []
    col_of = {a: i for i, a in enumerate(names)}
    for a, rows, cur, rep in out:
        i = col_of[a]
        rows, cur, rep = np.asarray(rows, dtype=np.int64), np.asarray(cur, dtype=np.int64), np.asarray(rep, dtype=np.int64)
        counts[i] += len(rows)
        cur_hist[i] += np.bincount(cur + 1, minlength=width)
        rep_hist[i] += np.bincount(rep + 1, minlength=width)
        keep = sampled[rows]
        parts.append(np.stack([rows[keep], np.full(int(keep.sum()), i), cur[keep], rep[keep]]))
    cells = np.concatenate(parts, axis=1) if parts else np.zeros((4, 0), dtype=np.int64)
    cells = cells[:, np.lexsort((cells[0], cells[1]))][:, :DUMP_MAX_CELLS]
    arrays = {"cells_per_attribute": counts, "current_hist": cur_hist, "repaired_hist": rep_hist,
              "tid": cells[0], "attribute": cells[1], "current_value": cells[2], "repaired": cells[3]}
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))
    return {"dir": path, "sampled_cells": int(cells.shape[1]), "frame_cells": int(counts.sum())}


# ---------------------------------------------------------------------------------------------
# NUMA: a rank's host threads (Arrow ingest workers, the pinned chunk ring they fill) belong on the
# CPU socket its GPU hangs off; 8 ranks sharing one socket's memory controllers is what cost the
# end-to-end leg 10 % at N=8 in round 1
# ---------------------------------------------------------------------------------------------
_FULL_AFFINITY = None


def bind_to_gpu_numa_node(local):
    global _FULL_AFFINITY
    info = {"bound": False}
    try:
        import pynvml
        _FULL_AFFINITY = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else local
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = "/sys/bus/pci/devices/{}/numa_node".format(bus.lower()[-12:])
        node = int(open(path).read().strip())
        if node >= 0:
            cpus = set()
            for part in open("/sys/devices/system/node/node{}/cpulist".format(node)).read().strip().split(","):
                a, _, b = part.partition("-")
                cpus |= set(range(int(a), int(b or a) + 1))
            cpus &= _FULL_AFFINITY
            if cpus:
                os.sched_setaffinity(0, cpus)
                info = {"bound": True, "node": node, "cpus": len(cpus)}
    except Exception as e:  # no NVML / sysfs entry / permission: run unbound
        info["why"] = "{}: {}".format(type(e).__name__, e)
    return info


def restore_affinity():
    if _FULL_AFFINITY:
        try:
            os.sched_setaffinity(0, _FULL_AFFINITY)
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------
# the other BASELINE.json configs: wall clock through the public API
# ---------------------------------------------------------------------------------------------
def other_configs(want, local, steps):
    import pandas as pd
    import torch
    from repair import (ConstraintErrorDetector, GaussianOutlierErrorDetector, NullErrorDetector, RepairModel, synth)
    golden = os.path.join(ROOT, "tests", "golden")
    out = {}

    def timed_run(make, **kw):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m = make()
        frame = m.run(**kw)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, frame, m

    if "c2" in want:   # hospital.csv + hospital_constraints.txt, Null + Constraint detectors (BASELINE config 2)
        df = pd.read_csv(os.path.join(golden, "hospital.csv"), dtype=str)
        make = lambda: RepairModel().setInput(df).setRowId("tid").setErrorDetectors(  # noqa: E731
            [NullErrorDetector(), ConstraintErrorDetector(os.path.join(golden, "hospital_constraints.txt"))]) \
            .option("model.hp.max_evals", "1")
        timed_run(make, detect_errors_only=True)                        # warm-up (library load, allocator)
        t_det, cells, _ = timed_run(make, detect_errors_only=True)
        t_all, frame, m = timed_run(make)
        frozen = m.last_run["models"] if "models" in m.last_run else None
        t_inf = None
        if frozen is not None:
            t_inf, _, _ = timed_run(lambda: make().setFrozenModels(frozen))
        out["C2_hospital"] = {"rows": len(df), "cols": len(df.columns) - 1, "error_cells": int(len(cells)),
                              "repaired_cells": int(len(frame)), "detect_only_s": round(t_det, 4),
                              "full_run_with_training_s": round(t_all, 3),
                              "training_s": round(m.last_run.get("elapsed_training", 0.0), 3),
                              "full_run_frozen_models_s": None if t_inf is None else round(t_inf, 4),
                              "how": "RepairModel.run() wall clock, pandas in / pandas out, 300-round models "
                                     "trained inside the call (no hyper-parameter search)"}
    if "c5" in want:   # boston.csv: numeric outlier detector + regressor predict (BASELINE config 5)
        df = pd.read_csv(os.path.join(golden, "boston.csv"))
        make = lambda: RepairModel().setInput(df).setRowId("tid").setErrorDetectors(  # noqa: E731
            [NullErrorDetector(), GaussianOutlierErrorDetector(approx_enabled=False)]).option("model.hp.max_evals", "1")
        timed_run(make, detect_errors_only=True)
        t_det, cells, _ = timed_run(make, detect_errors_only=True)
        t_all, frame, m = timed_run(make)
        out["C5_boston"] = {"rows": len(df), "cols": len(df.columns) - 1, "error_cells": int(len(cells)),
                            "repaired_cells": int(len(frame)), "detect_only_s": round(t_det, 4),
                            "full_run_with_training_s": round(t_all, 3),
                            "training_s": round(m.last_run.get("elapsed_training", 0.0), 3),
                            "how": "RepairModel.run() wall clock; continuous features: scikit-learn histogram GBDT "
                                   "trainer, generic float64 forest kernel"}
    if "c3" in want:   # synthetic 10M x 16, 1% NULLs, NullErrorDetector (BASELINE config 3)
        n, k = 10_000_000, 16
        spec = synth.SynthSpec.c3(n, k)
        dev = torch.device("cuda", local)
        codes = synth.generate_torch(spec, dev, 0, n)
        from repair._native import Context
        ctx = Context(local)
        tbl = host_arrow_shard(ctx, codes, n, 0, synth.column_names(k), spec.dom)
        ctx.close()
        del codes
        make = lambda: RepairModel().setArrowInput(tbl).setRowId("tid").setErrorDetectors([NullErrorDetector()]) \
            .option("model.hp.max_evals", "1")  # noqa: E731
        t_det, cells, _ = timed_run(make, detect_errors_only=True)
        t_det, cells, _ = timed_run(make, detect_errors_only=True)
        t_all, frame, m = timed_run(make)
        frozen = m.last_run["models"]
        timed_run(lambda: make().setFrozenModels(frozen))
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            t_inf, frame, mi = timed_run(lambda: make().setFrozenModels(frozen))
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
        out["C3_10Mx16"] = {"rows": n, "cols": k, "error_cells": int(cells.num_rows),
                            "repaired_cells": int(frame.num_rows), "detect_only_s": round(t_det, 4),
                            "full_run_with_training_s": round(t_all, 3),
                            "training_s": round(m.last_run.get("elapsed_training", 0.0), 3),
                            "ms_per_pass_frozen_models": round(ms, 2), "rows_per_sec": n / (ms / 1e3),
                            "ingest_s": round(mi.last_run.get("ingest_total_s", 0.0), 4),
                            "egress_s": round(mi.last_run.get("egress_s", 0.0), 4),
                            "how": "RepairModel().setArrowInput(host pyarrow.Table).run() -> pyarrow.Table, "
                                   "host buffers in / host frame out every pass"}
    return out


def host_arrow_shard(ctx, codes_dev, n, lo, names, dom):
    """The collected shard as the host holds it before ingest: a pyarrow.Table in ordinary (pageable)
    memory -- int64 `tid`, one dictionary<int8, string> column per attribute ("v%03d" entries), NULLs as
    Arrow nulls -- what `pyarrow.parquet.read_table(..., read_dictionary=...)` hands over."""
    import pyarrow as pa
    import torch
    words = (n + 31) // 32
    cols = {"tid": pa.array(np.arange(lo, lo + n, dtype=np.int64))}
    bits = torch.empty(words, dtype=torch.int32, device=codes_dev.device)
    for i, nm in enumerate(names):
        col = codes_dev[i][:n]
        idx = torch.clamp(col, min=0).to(torch.int8).cpu().numpy()
        ctx.valid_bits(col, n, bits)
        valid = bits.cpu().numpy().view(np.uint8)
        indices = pa.Array.from_buffers(pa.int8(), n, [pa.py_buffer(valid), pa.py_buffer(idx)])
        d = pa.array(["v%03d" % c for c in range(int(dom[i]))], type=pa.string())
        cols[nm] = pa.DictionaryArray.from_arrays(indices, d, safe=False)
    return pa.table(cols)


def api_detectors(n_cols):
    from repair import ConstraintErrorDetector, NullErrorDetector, synth
    dets = [NullErrorDetector()]
    fds = synth.fd_constraints(n_cols)
    if fds:
        dets.append(ConstraintErrorDetector(constraints=fds))
    return dets


def frames_equal(arrow_frame, out, lo, names, table):
    """The API's Arrow frame == the encoded frame of the resident-table pass (row ids, attribute, current and
    repaired dictionary entries), compared attribute chunk by attribute chunk."""
    by_attr = {a: (np.asarray(rows), np.asarray(cur), np.asarray(rep)) for a, rows, cur, rep in out}
    if arrow_frame.num_rows != sum(len(v[0]) for v in by_attr.values()):
        return False
    pos = 0
    seen = set()
    for k in range(arrow_frame["attribute"].num_chunks):
        att = arrow_frame["attribute"].chunk(k)
        if len(att) == 0:
            continue
        a = att.dictionary[att.indices[0].as_py()].as_py()
        seen.add(a)
        rows, cur, rep = by_attr[a]
        m = len(rows)
        ids = arrow_frame["tid"].chunk(k).to_numpy()
        if len(att) != m or not np.array_equal(ids, rows.astype(np.int64) + lo):
            return False
        strs = table.by_name[a].strings()
        for chunk, codes in ((arrow_frame["current_value"].chunk(k), cur), (arrow_frame["repaired"].chunk(k), rep)):
            d = chunk.dictionary.to_pylist()
            idx = chunk.indices.fill_null(-1).to_numpy(zero_copy_only=False).astype(np.int64)
            want = np.asarray(codes, dtype=np.int64)
            if not np.array_equal(idx < 0, want < 0):
                return False
            ok = idx >= 0
            lut = np.array([strs.index(v) for v in d], dtype=np.int64) if d else np.zeros(0, dtype=np.int64)
            if ok.any() and not np.array_equal(lut[idx[ok]], want[ok]):
                return False
        pos += m
    return seen == {a for a, v in by_attr.items() if len(v[0])}


def b200_arm(args):
    import torch
    from repair import RepairModel, synth
    from repair._native import profile_summary
    from repair.engine import Dist, Engine
    from repair.errors import ErrorModelOptions
    from repair.model import build_models, repair_cells
    from repair.table import DeviceTable, EncodedTable

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as td
        # NCCL's own log lines (e.g. "NCCL version ...") belong on stderr: stdout carries ONE JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        td.init_process_group("nccl", device_id=device)
        dist = Dist()
    k = args.cols
    total_rows = args.rows if args.scaling == "strong" else args.rows * world
    spec = synth.SynthSpec.c4(total_rows, k)
    lo, hi = (total_rows * rank) // world, (total_rows * (rank + 1)) // world
    n = hi - lo

    # ---- setup (untimed): the shard resident in HBM ------------------------------------------------
    codes_dev = synth.generate_torch(spec, device, lo, hi)
    n_pad = codes_dev.shape[1]
    names = synth.column_names(k)
    host_np = [np.zeros(0, dtype=np.int32) for i in range(k)]
    table = EncodedTable.from_codes("tid", names, host_np, spec.dom, row_ids=np.arange(lo, hi, dtype=np.int64))
    table.n_rows = n
    table.row_offset, table.n_rows_global = lo, total_rows
    dt = DeviceTable(table, device, codes=codes_dev)
    engine = Engine(table, local, dist=dist, device_table=dt)
    rm = RepairModel()
    rm.opts = dict(OPTS)
    rm.borrow_encoded_output = True   # the step reads its frame in place; verify / e2e take copies below
    if args.forests == "random":
        rm.model_provider = random_forest_provider(N_ESTIMATORS)
    err_opts = ErrorModelOptions.resolve(rm.opts)
    specs = detector_specs(k)
    continuous = []

    # frozen models: trained ONCE on the global 10k-row sample (every rank draws the same sample and trains
    # the same deterministic forests -- engine.valid_training_rows / sample_rows_masked)
    res = engine.detect(specs, [], 80, err_opts)
    torch.cuda.synchronize()
    t_train = time.time()
    models = build_models(rm, engine, table, res, continuous)
    torch.cuda.synchronize()
    t_train = time.time() - t_train
    n_trees = sum(m[1].n_trees for _, m in models if m[0] == "forest")
    from repair.forest import forest_shape_stats
    shape = {y: forest_shape_stats(m[2]["spec"]["forest"]) for y, m in models if m[0] == "forest"}

    stats = {}
    res_cells = {}

    def step():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        engine.mark("step:begin")
        engine.reset()
        r = engine.detect(specs, [], 80, err_opts)
        ev[1].record()
        engine.mark("step:detect")
        out = repair_cells(rm, engine, table, r, continuous, models=models, encoded_output=True)
        ev[2].record()
        engine.mark("step:repair returned")
        for a_, n_ in r.n_cells.items():
            res_cells[a_] = n_
        stats["cells"] = rm.last_run["n_error_cells"]
        stats["dirty"] = rm.last_run["n_dirty_rows"]
        stats["out_rows"] = sum(len(x[1]) for x in out)
        stats["last"] = (r, out)
        stats["d2h"] = sum(x[1].nbytes + x[2].nbytes + x[3].nbytes for x in out)
        return ev

    def barrier():
        if dist is not None:
            dist.td.barrier()
        torch.cuda.synchronize()

    def timed(steps, warmup):
        for _ in range(warmup):
            step()
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
            time.sleep(0.3)  # let nvidia-smi finish initialising before the timed region starts
        barrier()
        l0 = engine.ctx.launch_count
        x0 = dist.n_exchanges if dist is not None else 0
        evs = [step() for _ in range(steps)]
        barrier()
        clocks = sampler.stop() if sampler else None
        tot = evs[0][0].elapsed_time(evs[-1][2]) / steps   # whole span: gaps between steps count too
        det = sum(e[0].elapsed_time(e[1]) for e in evs) / steps
        t = torch.tensor([tot, det], dtype=torch.float64, device=device)
        if dist is not None:
            dist.max_(t)
        xs = ((dist.n_exchanges - x0) / steps) if dist is not None else 0
        return float(t[0]), float(t[1]), (engine.ctx.launch_count - l0), clocks, xs

    ms, ms_det, launches, clocks, exchanges = timed(args.steps, args.warmup)
    # before any further pass: the frame of the last timed step borrows a staging buffer the next pass reuses
    dumped = dump_outputs(args.dump_outputs, stats["last"][1], names, spec.dom, n) if args.dump_outputs else None
    cells = torch.tensor([stats["cells"], stats["out_rows"]], dtype=torch.int64, device=device)
    if dist is not None:
        dist.sum_(cells)
    line = {
        "metric": METRIC, "value": total_rows / (ms / 1e3), "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "int32 codes / f64 margins", "data": "synthetic",
        "config": {"workload": "C4 synthetic {} rows x {} cols in total, {} rows per GPU ({} scaling), 1% NULLs + 4 FD "
                               "denial constraints, NULL + Constraint detectors, pairwise_freq_ratio_threshold=1.0, "
                               "{} frozen repair models ({} trees: 300 rounds x classes, {}), "
                               "inputs > L2 (no flush needed)".format(
                                   total_rows, k, n, args.scaling, len(models), n_trees,
                                   "trained by dr_gbdt_train on 10k-row samples" if args.forests == "trained"
                                   else "random-init"),
                   "rows_total": total_rows, "rows_per_gpu": n, "cols": k,
                   "parallelism": "rows sharded x{}".format(world)},
        "rows_scanned_per_sec": total_rows / (ms_det / 1e3),
        "cells_repaired_per_sec": int(cells[0]) / max((ms - ms_det) / 1e3, 1e-9),
        "error_cells": int(cells[0]), "repaired_cells_emitted": int(cells[1]),
        "ms_detect_phase": ms_det, "ms_repair_phase": ms - ms_det,
        "gpu_launches": launches, "clocks": clocks,
        "model_training_s": t_train, "forests": args.forests,
    }
    line["numa"] = numa
    if dumped:
        line["dump_outputs"] = dumped
    if dist is not None:
        line["exchanges_per_step"] = exchanges

    # ---- self-check of the last timed step (untimed) -------------------------------------------
    if not args.no_verify:
        t_v = time.time()
        r_last, out_last = stats["last"]
        # copies: the result arrays are views of a pinned staging buffer the next pass reuses
        out_last = [(a, np.array(x), np.array(c), np.array(rp)) for a, x, c, rp in out_last]
        v = verify_step(engine, table, r_last, out_last, models, k, args.verify_cells, dist)
        cnt = torch.tensor([v["hist_mismatches"], v["cell_count_mismatches"], v["cells_checked"], v["mismatches"]],
                           dtype=torch.int64, device=device)
        if dist is not None:
            dist.sum_(cnt)
            v["hist_mismatches"], v["cell_count_mismatches"] = int(cnt[0]), int(cnt[1])
            v["cells_checked"], v["mismatches"] = int(cnt[2]), int(cnt[3])
        v["seconds"] = round(time.time() - t_v, 2)
        v["how"] = "torch.bincount histograms; NULL + torch scatter_reduce FD cell counts; sampled repairs " \
                   "re-evaluated by oracle/c forest_margins on host-encoded feature vectors"
        line["verify"] = v

    # ---- per-kernel timing (CUDA events on the launching stream) and rooflines ------------------
    engine.ctx.profile = []
    step()
    prof = profile_summary(engine.ctx)
    engine.ctx.profile = None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    n_disc = k
    alg = {
        "scan_hist": 4.0 * n_disc * n,                               # every code read once (SURVEY 8d)
        # SURVEY 8(d): per error cell 4*F bytes of feature gather (F = K - 1) + 4 bytes written + 16 bytes of
        # output record = 144 B/cell at K = 32
        "forest_predict": stats["cells"] * (4.0 * (k - 1) + 4.0 + 16.0),
        "forest_predict_ranked": stats["cells"] * (4.0 * (k - 1) + 4.0 + 16.0),
        "gather_rows_masked": stats["dirty"] * 4.0 * k * 2,          # dirty rows in, tile out
        "cooc": None, "dc_fd_build": None, "dc_fd_flag": None, "domain_score": None,
    }
    kernels = {}
    for name, (cnt, tms) in sorted(prof.items(), key=lambda kv: -kv[1][1]):
        entry = {"calls": cnt, "ms": round(tms, 3)}
        if alg.get(name):
            gbs = alg[name] / (tms / 1e3) / 1e9
            entry.update({"algorithmic_gb": round(alg[name] / 1e9, 3), "achieved_gbs": round(gbs, 1),
                          "frac_of_hbm_peak": round(gbs / peak, 4)})
        kernels[name] = entry
    dominant = max(prof.items(), key=lambda kv: kv[1][1])[0] if prof else None
    line["kernels"] = kernels
    fp = [v for kname, v in prof.items() if kname.startswith("forest_predict")]
    ncu = {}
    try:  # per-launch figures taken from ncu --set full captures of this very command (profiles/)
        ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_per_launch.json")))
    except Exception:
        pass

    def ncu_for(kernel):
        e = ncu.get(kernel)
        ok = e and e.get("rows_per_gpu") == n and e.get("cols") == k
        return e if ok else None
    if fp:
        # forest inference is bounded by the shared-memory pipe, not HBM (profiles/r1_ncu_forest_*.md): the
        # roofline that explains it counts shared-memory wavefronts.  Algorithmic minimum per warp: two
        # loads per tree level (rank, node word; the last level only the rank) + per tree one header
        # broadcast and the leaf value (two 32-bit loads); peak = one wavefront per cycle per SM.
        f_ms = sum(v[1] for v in fp)
        levels = sum((m[1].n_trees * (m[1].ranked.max_depth if m[1].ranked is not None else 5)) *
                     res_cells.get(y, 0) for y, m in models if m[0] == "forest")
        tree_cells = sum(m[1].n_trees * res_cells.get(y, 0) for y, m in models if m[0] == "forest")
        line["forest_tree_levels_per_sec"] = levels / (f_ms / 1e3)
        # how much of the fixed-depth walk the trained trees need (weights: trees x cells of each model)
        wsum = sum(shape[y]["n_trees"] * res_cells.get(y, 0) for y in shape) or 1
        wavg = (lambda key: sum(shape[y][key] * shape[y]["n_trees"] * res_cells.get(y, 0) for y in shape) / wsum)
        line["forest_stats"] = {
            "levels_walked_per_tree": levels / max(tree_cells, 1), "mean_tree_depth": wavg("mean_tree_depth"),
            "mean_leaf_depth": wavg("mean_leaf_depth"), "mean_leaves": wavg("mean_leaves"),
            "single_leaf_tree_frac": wavg("single_leaf_tree_frac"),
            "max_depth_by_model": {y: shape[y]["max_depth"] for y in shape}}
        sm_hz = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
        sm_count = torch.cuda.get_device_properties(device).multi_processor_count
        # per warp and tree: 2 loads per level except the last (rank only) + header broadcast (1) + leaf value
        # (two 32-bit loads) = 2 * depth + 2
        wf = (2.0 * levels + 2.0 * tree_cells) / 32.0
        e = ncu_for("k_forest_predict_ranked")
        line["roofline_forest"] = {
            "kernel": "k_forest_predict_ranked", "bound": "shared-memory wavefronts",
            "achieved": wf / (f_ms / 1e3) / 1e9, "peak": sm_count * sm_hz / 1e9, "unit": "Gwavefront/s",
            "frac": wf / (f_ms / 1e3) / (sm_count * sm_hz),
            "measured_pipe_utilisation": e.get("smem_wavefronts_per_cycle_per_sm") if e else None,
            "note": "achieved = algorithmic wavefronts (2 per warp-level + 2 per warp-tree) / kernel time; "
                    "measured_pipe_utilisation is ncu's wavefront count (conflict replays and the tile fill "
                    "included) per cycle and SM"}
    if dominant:
        d = kernels[dominant]
        ach = d.get("achieved_gbs")
        e = ncu_for("k_" + dominant)
        line["roofline"] = {"kernel": dominant, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                            "frac": (ach / peak) if ach else None,
                            "traffic": e.get("dram_bytes_per_launch") if e else None, "peak_source": peak_src,
                            "note": "this kernel is not HBM bound, see roofline_forest; the HBM-bound kernel of "
                                    "the path is k_scan_hist (roofline_scan)"
                            if dominant.startswith("forest_predict") else None}
    sh = kernels.get("scan_hist")
    if sh:
        e = ncu_for("k_scan_hist")
        line["roofline_scan"] = {"kernel": "k_scan_hist", "bound": "hbm", "achieved": sh.get("achieved_gbs"),
                                 "peak": peak, "unit": "GB/s", "frac": sh.get("frac_of_hbm_peak"),
                                 "traffic": e.get("dram_bytes_per_launch") if e else None,
                                 "peak_source": peak_src}
    if args.profile_calls and rank == 0:
        for kname, v in kernels.items():
            print(kname, v, file=sys.stderr)
    if args.trace:
        engine.trace = []
        step()
        if rank == 0:
            for label, dt_s in engine.trace:
                print("trace %-24s %8.2f ms" % (label, dt_s * 1e3), file=sys.stderr)
        engine.trace = None

    # ---- end to end THROUGH THE PUBLIC API: host Arrow table in, host Arrow frame out, every step ----------
    if not args.no_e2e:
        r_last, out_last = stats["last"]
        out_resident = [(a, np.array(x), np.array(c), np.array(rp)) for a, x, c, rp in out_last]
        arrow_tbl = host_arrow_shard(engine.ctx, codes_dev, n, lo, names, spec.dom)
        h2d = sum(c.nbytes for c in arrow_tbl.columns)   # indices + validity bits + row ids (dictionaries are tiny)
        last = {}

        def api_step():
            m = RepairModel().setArrowInput(arrow_tbl).setRowId("tid").setErrorDetectors(api_detectors(k)) \
                .setFrozenModels(models)
            for kk, vv in OPTS.items():
                m.option(kk, vv)
            m.device_index = local
            if args.forests == "random":
                m.model_provider = rm.model_provider
            if dist is not None:
                m.setDistributed(True, local)
            t0 = time.perf_counter()
            frame = m.run()
            last.update({"frame": frame, "rm": m, "wall": time.perf_counter() - t0})
            return frame

        api_step()                       # warm-up: allocator pools, the pinned chunk ring, page faults
        e_steps = args.steps
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        t0 = time.perf_counter()
        parts = {"ingest_s": 0.0, "egress_s": 0.0, "ingest_copy_s": 0.0, "ingest_encode_s": 0.0,
                 "engine_ready_s": 0.0, "detect_done_s": 0.0, "repair_done_s": 0.0, "total_s": 0.0}
        for _ in range(e_steps):
            api_step()
            lr = last["rm"].last_run
            parts["ingest_s"] += lr.get("ingest_total_s", 0.0)
            parts["ingest_copy_s"] += lr.get("ingest_copy_s", 0.0)
            parts["ingest_encode_s"] += lr.get("ingest_encode_s", 0.0)
            parts["egress_s"] += lr.get("egress_s", 0.0)
            for kk in ("engine_ready_s", "detect_done_s", "repair_done_s", "total_s"):
                parts[kk] += lr.get(kk, 0.0)
        ev1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3 / e_steps
        t = torch.tensor([ev0.elapsed_time(ev1) / e_steps, wall_ms] + [v / e_steps for v in parts.values()],
                         dtype=torch.float64, device=device)
        if dist is not None:
            dist.max_(t)
        e_ms = float(t[0])
        frame = last["frame"]
        d2h = sum(c.nbytes for c in frame.columns)
        same = frames_equal(frame, out_resident, lo, names, table)
        flag = torch.tensor([0 if same else 1], dtype=torch.int64, device=device)
        if dist is not None:
            dist.sum_(flag)
        line["e2e"] = {"value": total_rows / (e_ms / 1e3), "unit": "rows/s", "ms_per_step": e_ms,
                       "wall_ms_per_step": float(t[1]), "steps": e_steps,
                       "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "ingest_s": float(t[2]), "egress_s": float(t[3]),
                       "ingest_copy_s": float(t[4]), "ingest_encode_s": float(t[5]),
                       "stamps_s": {"engine_ready": float(t[6]), "detect_done": float(t[7]), "repair_done": float(t[8]),
                                    "run_returned": float(t[9])},
                       "ingest_detail_rank0_last_step": {kk: lr.get(kk) for kk in ("ingest_ids_s", "ingest_encode_phases")},
                       "frame_rows": int(frame.num_rows), "frame_equals_resident_pass": int(flag[0]) == 0,
                       "call": "RepairModel().setArrowInput(pyarrow.Table in pageable host memory).setRowId('tid')"
                               ".setErrorDetectors([NullErrorDetector(), ConstraintErrorDetector(..)])"
                               ".setFrozenModels(models).run() -> pyarrow.Table (tid, attribute, current_value, "
                               "repaired); CUDA events around the calls, max over ranks",
                       "note": "ingest = Arrow dictionary indices (int8) + validity bits + int64 row ids through the "
                               "pinned chunk ring (dr_h2d_copy), dictionaries re-encoded on the device; egress = row "
                               "ids gathered on the device, dictionary indices + validity bits copied back and "
                               "wrapped as Arrow arrays; models frozen (training is not part of the step)"}
        del arrow_tbl, frame
        last.clear()

    # ---- the other BASELINE configs: wall clock through the public API (untimed setup excluded) ------------
    want = [] if args.configs == "none" else (["c2", "c3", "c5"] if args.configs == "auto" else
                                              [c.strip() for c in args.configs.split(",") if c.strip()])
    if args.configs == "auto" and (world != 1 or args.rows != 100_000_000):
        want = []
    if want and rank == 0:
        line["other_configs"] = other_configs(want, local, args.steps)

    # ---- CPU baseline (rank 0, single GPU run only) -----------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        restore_affinity()   # the CPU leg gets every host core
        trained = {y: (m[2]["spec"] if m[0] == "forest" else {"const": m[1]}) for y, m in models} \
            if args.forests == "trained" else None
        rows_cpu = args.ref_rows if args.ref_rows > 0 else 20000
        run_oracle_sample(10000, k, N_ESTIMATORS, trained)  # untimed: first touch of the forests, thread pool
        t_full, rows, ncells, t_det, threads, _, fb = run_oracle_sample(rows_cpu, k, N_ESTIMATORS, trained)
        line["cpu_baseline"] = {"value": rows / t_full, "unit": "rows/s", "cores": threads, "kind": "port",
                                "sample": "first {} rows of the C4 table with the same frozen forests, oracle full "
                                          "pass in {:.1f} s (detect phase {:.1f} s)".format(rows, t_full, t_det),
                                "cells_repaired_per_sec": ncells / max(t_full - t_det, 1e-9),
                                "targets_on_random_forests": fb}
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.td.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == "__main__":
    main()
