"""Benchmark of LOFOutlierErrorDetector's kernel (dr_lof_flag) on one resident float64 column.

  python tools/bench_lof.py [--rows 100000000] [--verify-rows 10000000] [--sklearn-rows 1000000] [--out F]

Prints one JSON line:
  * CUDA-event time of dr_lof_flag on a --rows column (1 % NULLs, 0.01 % far values), rows/s;
  * per-phase kernel time (fill: keys + median + place, sort: CUB radix sort, kdist, lrd, score) from one
    call under torch.profiler, with the algorithmic bytes of each phase and their rate against the
    device-to-device copy rate measured in the same run;
  * verify: flags and float64 scores of a --verify-rows column against the host definition
    (tests/lof_reference.py), as mismatch counts;
  * context: LocalOutlierFactor.fit_predict on a --sklearn-rows host sample (wall clock).
Needs a CUDA device; there is no CPU fallback.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "spark-data-repair-plugin_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

K = 20
SORT_PASSES = 8   # CUB's onesweep radix sort of 64-bit keys: 8 digit passes of 8 bits


def phase_bytes(n):
    """Algorithmic bytes per phase (each array read or written once; the halo re-reads are not counted)."""
    return {
        "fill": n * (8 + 8 + 4) + n * (8 + 4 + 8 + 4),   # keys: col -> key, row; place: key, row -> s, perm
        "sort": SORT_PASSES * n * 2 * (8 + 4),           # every pass reads and writes (key, row)
        "kdist": n * (8 + 8 + 1),                        # s -> kdist, window offset
        "lrd": n * (8 + 8 + 1 + 8),                      # s, kdist, offset -> lrd
        "score": n * (8 + 1 + 4) + n // 8,               # lrd, offset, perm -> bitmap
    }


def phase_of(name):
    for key, phase in (("k_lof_keys", "fill"), ("k_lof_median", "fill"), ("k_lof_place", "fill"),
                       ("k_lof_kdist", "kdist"), ("k_lof_lrd", "lrd"), ("k_lof_score", "score")):
        if key in name:
            return phase
    if "Radix" in name or "radix" in name or "Onesweep" in name or "cub" in name:
        return "sort"
    return None


def make_column(torch, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
    u = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
    x = torch.where(u < 1e-4, x * 50.0 + 40.0, x)               # far values
    x = torch.where((u >= 1e-4) & (u < 1e-4 + 0.01), torch.full_like(x, float("nan")), x)   # 1 % NULLs
    return x


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--verify-rows", type=int, default=10_000_000)
    ap.add_argument("--sklearn-rows", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_lof.py needs a CUDA device")
    from repair._native import Context
    ctx = Context.acquire(0)
    n = args.rows
    res = {"bench": "lof_1d", "rows": n, "k": K, "gpu": gpu_info()}

    # device-to-device copy rate (read + write bytes) as the HBM reference point
    a = torch.empty(1 << 28, dtype=torch.float64, device="cuda")    # 2 GiB, far beyond L2
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    copy_gbs = 10 * 2 * a.numel() * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    res["copy_GBps"] = round(copy_gbs, 1)
    del a, b

    col = make_column(torch, n, seed=1)
    words = torch.zeros((n + 31) // 32, dtype=torch.int32, device="cuda")
    ws = torch.empty(ctx.lof_workspace_bytes(n), dtype=torch.uint8, device="cuda")
    res["workspace_bytes"] = int(ws.numel())
    for _ in range(args.warmup):
        ctx.lof_flag(col, n, K, 0, n, words, ws)
    times = []
    for _ in range(args.reps):
        words.zero_()
        e0.record()
        ctx.lof_flag(col, n, K, 0, n, words, ws)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    res["lof_flag_ms"] = {"median": round(float(np.median(times)), 3), "min": round(min(times), 3),
                          "max": round(max(times), 3), "reps": args.reps}
    res["rows_per_s"] = round(n / (float(np.median(times)) * 1e-3), 1)
    res["flagged"] = int(ctx.lof_flag(col, n, K, 0, n, words.zero_(), ws, count=True))

    # per-phase kernel time from one profiled call
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.lof_flag(col, n, K, 0, n, words, ws)
        torch.cuda.synchronize()
    phase_us = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        ph = phase_of(ev.name)
        if ph is not None:
            phase_us[ph] = phase_us.get(ph, 0.0) + ev.device_time
    nbytes = phase_bytes(n)
    res["phases"] = {ph: {"ms": round(phase_us.get(ph, 0.0) / 1e3, 3), "bytes": nbytes[ph],
                          "GBps": round(nbytes[ph] / (phase_us[ph] * 1e-6) / 1e9, 1) if phase_us.get(ph) else None,
                          "of_copy": round(nbytes[ph] / (phase_us[ph] * 1e-6) / 1e9 / copy_gbs, 3)
                          if phase_us.get(ph) else None}
                     for ph in ("fill", "sort", "kdist", "lrd", "score")}
    del col, ws, words
    torch.cuda.empty_cache()

    # verify against the host definition
    from lof_reference import lof_scores_1d
    nv = args.verify_rows
    col = make_column(torch, nv, seed=2)
    words = torch.zeros((nv + 31) // 32 + 1, dtype=torch.int32, device="cuda")
    out = torch.empty(nv, dtype=torch.float64, device="cuda")
    ws = torch.empty(ctx.lof_workspace_bytes(nv), dtype=torch.uint8, device="cuda")
    ctx.lof_flag(col, nv, K, 0, nv, words, ws, out_lof=out)
    got = out.cpu().numpy()
    bits = np.unpackbits(words.cpu().numpy().view(np.uint8), bitorder="little")[:nv].astype(bool)
    t0 = time.time()
    want = lof_scores_1d(col.cpu().numpy(), K)
    host_s = time.time() - t0
    res["verify"] = {"rows": nv, "flag_mismatches": int((bits != (want > 1.5)).sum()),
                     "score_bit_mismatches": int((got.view(np.int64) != want.view(np.int64)).sum()),
                     "flagged": int(bits.sum()), "host_definition_s": round(host_s, 2)}

    # context: scikit-learn on a host sample
    from sklearn.neighbors import LocalOutlierFactor
    ns = args.sklearn_rows
    x = col[:ns].cpu().numpy()
    x = np.where(np.isnan(x), np.median(x[~np.isnan(x)]), x)
    t0 = time.time()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        LocalOutlierFactor(novelty=False).fit_predict(x[:, None])
    sk_s = time.time() - t0
    res["sklearn_fit_predict"] = {"rows": ns, "s": round(sk_s, 2), "rows_per_s": round(ns / sk_s, 1),
                                  "host_cpus": os.cpu_count()}
    Context.release(ctx)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
