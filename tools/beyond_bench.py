"""What the beyond-accuracy metrics (novelty / avg_popularity / diversity) cost: device-resident calls of BASELINE configs 2, 4
and 5 without them, with Novelty + AvgPop, with ILD, and with all three; each new kernel on its own; the bytes
beyond_accuracy_kernel gathers and its achieved bandwidth; and item_popularity from a host CSR and from a DeviceCSR next to
numpy.bincount.

    python tools/beyond_bench.py [--configs 2 4 5] [--reps 5] [--out FILE]

Calls are timed with a host clock around a call that ends in a device synchronise, the four variants alternating.  Kernel
times come from a separate torch.profiler run of one call per variant.  Prints one JSON document and, with --out, writes it to
FILE as well.  Needs a CUDA device: there is no CPU path to measure."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_TBPS = 7.7          # NVIDIA's data-sheet HBM3e bandwidth of one B200
KERNELS = ("beyond_accuracy_kernel", "unit_rows_kernel", "popularity_table_kernel", "item_popularity_kernel")
VARIANTS = {"plain": {}, "nov_avg": dict(novelty=True, avg_popularity=True), "ild": dict(diversity=True),
            "all": dict(novelty=True, avg_popularity=True, diversity=True)}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4, 5])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import recometrics_b200 as rb
    from tools import synth

    if not torch.cuda.is_available() or rb.device_count() == 0:
        raise SystemExit("beyond_bench.py: no CUDA device -- nothing to measure")
    dev = torch.device("cuda", 0)
    doc = {"gpu": gpu_info(), "reps": args.reps, "hbm_tbps_datasheet": HBM_TBPS, "configs": {}}
    for cfg_id in args.configs:
        cfg = synth.CONFIGS[cfg_id]
        d = synth.make(cfg_id)
        m, n = d["X_test"].shape
        p = d["A"].shape[1]
        A, B = torch.from_numpy(d["A"]).to(dev), torch.from_numpy(d["B"]).to(dev)
        bias = None if d["item_biases"] is None else torch.from_numpy(d["item_biases"]).to(dev)
        Xtr = rb.DeviceCSR.from_scipy(d["X_train"], 0, cfg.dtype, with_data=False)
        Xte = rb.DeviceCSR.from_scipy(d["X_test"], 0, cfg.dtype)
        names = dict(p="precision", tp="trunc_precision", r="recall", ap="average_precision", tap="trunc_average_precision",
                     ndcg="ndcg", hit="hit", rr="rr", roc="roc_auc", pr="pr_auc")
        kw = dict(k=cfg.k, item_biases=bias, break_ties_with_noise=False, cumulative=cfg.cumulative, min_pos_test=cfg.min_pos_test,
                  **{name: q in cfg.metrics for q, name in names.items()})
        pop = rb.item_popularity(Xtr, m=m)         # once, as a caller evaluating several models would

        def call(variant):
            extra = dict(VARIANTS[variant])
            if extra.get("novelty"):
                extra["item_popularity"] = pop
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = rb.calc_reco_metrics_device(Xtr, Xte, A, B, means_only=True, **kw, **extra)
            torch.cuda.synchronize()
            return r, (time.perf_counter() - t0) * 1e3

        for v in VARIANTS:                        # warm-up: modules, workspace cache
            call(v)
        wall = {v: [] for v in VARIANTS}
        total = {v: [] for v in VARIANTS}
        last = {}
        for _ in range(args.reps):
            for v in VARIANTS:
                r, w = call(v)
                wall[v].append(round(w, 2)); total[v].append(round(r.timing["total_ms"], 2))
                last[v] = r
        kernels = {}
        for v in ("nov_avg", "ild", "all"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(v)
            kernels[v] = {}
            for kname in KERNELS:
                ev = [e for e in prof.events() if kname in e.name]
                if ev:
                    kernels[v][kname] = {"ms": round(sum(e.device_time for e in ev) / 1e3, 4), "launches": len(ev)}
        cnt = last["all"].counts["Novelty@K"]
        users = int(cnt[-1] if np.ndim(cnt) else cnt)
        item = np.dtype(cfg.dtype).itemsize
        pitch = -(-p // (16 // item)) * (16 // item)
        entries = users * cfg.k
        ild_bytes = entries * (pitch * item + 4)            # one unit row and one id per listed item
        ild_ms = kernels["ild"]["beyond_accuracy_kernel"]["ms"]
        # item popularity: host CSR (upload + count), DeviceCSR, numpy.bincount of the same rows
        Xh = d["X_train"]
        ip = {}
        for what, f in (("host_csr", lambda: rb.item_popularity(Xh, m=m)), ("device_csr", lambda: rb.item_popularity(Xtr, m=m)),
                        ("numpy_bincount", lambda: np.bincount(Xh.indices[: Xh.indptr[m]], minlength=n))):
            f()
            ts = []
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = f()
                torch.cuda.synchronize()
                ts.append(round((time.perf_counter() - t0) * 1e3, 2))
            ip[what] = ts
        assert np.array_equal(rb.item_popularity(Xh, m=m), np.bincount(Xh.indices[: Xh.indptr[m]], minlength=n))
        med = lambda x: float(np.median(x))
        c = {"shape": cfg.name, "m": m, "n": n, "p": p, "k": cfg.k, "dtype": np.dtype(cfg.dtype).name, "cumulative": cfg.cumulative,
             "scoring_path": int(last["plain"].timing["scoring_path"]), "users_with_a_list": users, "train_nnz": int(Xh.indptr[m]),
             "call_ms": wall, "total_ms": total,
             "median_overhead_ms": {v: round(med(wall[v]) - med(wall["plain"]), 3) for v in VARIANTS if v != "plain"},
             "kernels": kernels,
             "ild_gathered_bytes": ild_bytes, "ild_bound_ms_at_datasheet": round(ild_bytes / (HBM_TBPS * 1e12) * 1e3, 3),
             "ild_achieved_tbps": round(ild_bytes / (ild_ms * 1e-3) / 1e12, 3) if ild_ms > 0 else None,
             "ild_share_of_datasheet": round(ild_bytes / (ild_ms * 1e-3) / 1e12 / HBM_TBPS, 3) if ild_ms > 0 else None,
             "item_popularity_ms": ip}
        doc["configs"]["cfg%d" % cfg_id] = c
        print(json.dumps({"cfg%d" % cfg_id: c}), flush=True)
        del A, B, bias, Xtr, Xte, d, pop, last
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
