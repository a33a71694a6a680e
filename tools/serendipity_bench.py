"""What Unexpectedness@K / Serendipity@K (unexpectedness / serendipity) cost: device-resident means_only calls of BASELINE
configs 4, 5 and 2 without any beyond-accuracy row, with the two new rows, with ILD alone and with ILD plus the new rows;
history_distance_kernel on its own; the bytes it gathers and its achieved bandwidth.

    python tools/serendipity_bench.py [--configs 4 5 2] [--reps 5] [--out FILE]

Calls are timed with a host clock around a call that ends in a device synchronise, the four variants alternating.  Kernel
times come from a separate torch.profiler run of one call per variant.  Prints one JSON document and, with --out, writes it to
FILE as well.  Needs a CUDA device: there is no CPU path to measure."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.beyond_bench import HBM_TBPS, gpu_info  # noqa: E402

KERNELS = ("history_distance_kernel", "beyond_accuracy_kernel", "unit_rows_kernel")
VARIANTS = {"plain": {}, "hist": dict(unexpectedness=True, serendipity=True), "ild": dict(diversity=True),
            "ild_hist": dict(diversity=True, unexpectedness=True, serendipity=True)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[4, 5, 2])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import recometrics_b200 as rb
    from tools import synth

    if not torch.cuda.is_available() or rb.device_count() == 0:
        raise SystemExit("serendipity_bench.py: no CUDA device -- nothing to measure")
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

        def call(variant, **more):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = rb.calc_reco_metrics_device(Xtr, Xte, A, B, means_only=True, **kw, **VARIANTS[variant], **more)
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
        for v in ("hist", "ild", "ild_hist"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                call(v)
            kernels[v] = {}
            for kname in KERNELS:
                ev = [e for e in prof.events() if kname in e.name]
                if ev:
                    kernels[v][kname] = {"ms": round(sum(e.device_time for e in ev) / 1e3, 4), "launches": len(ev)}
        # the rows the kernel gathers: the history of every user with a list (the kernel reads no more for a user without
        # history), and the listed rows of the users it evaluates
        status = call("plain", return_status=True)[0].status.cpu().numpy()
        ntrain = np.diff(d["X_train"].indptr)[:m].astype(np.int64)
        listed = status == 0
        defined = listed & (ntrain > 0)
        cnt = last["hist"].counts["Unexpectedness@K"]
        users = int(cnt[-1] if np.ndim(cnt) else cnt)
        assert users == int(defined.sum())
        hist_rows, list_rows = int(ntrain[defined].sum()), users * cfg.k
        item = np.dtype(cfg.dtype).itemsize
        pitch = -(-p // (16 // item)) * (16 // item)
        hist_bytes = (hist_rows + list_rows) * pitch * item
        hist_ms = kernels["hist"]["history_distance_kernel"]["ms"]
        med = lambda x: float(np.median(x))
        c = {"shape": cfg.name, "m": m, "n": n, "p": p, "k": cfg.k, "dtype": np.dtype(cfg.dtype).name, "cumulative": cfg.cumulative,
             "scoring_path": int(last["plain"].timing["scoring_path"]), "users_defined": users,
             "history_rows": hist_rows, "listed_rows": list_rows, "call_ms": wall, "total_ms": total,
             "median_call_ms": {v: round(med(wall[v]), 3) for v in VARIANTS},
             "median_overhead_ms": {v: round(med(wall[v]) - med(wall["plain"]), 3) for v in VARIANTS if v != "plain"},
             "kernels": kernels,
             "history_gathered_bytes": hist_bytes, "history_bound_ms_at_datasheet": round(hist_bytes / (HBM_TBPS * 1e12) * 1e3, 3),
             "history_achieved_tbps": round(hist_bytes / (hist_ms * 1e-3) / 1e12, 3) if hist_ms > 0 else None,
             "history_share_of_datasheet": round(hist_bytes / (hist_ms * 1e-3) / 1e12 / HBM_TBPS, 3) if hist_ms > 0 else None}
        doc["configs"]["cfg%d" % cfg_id] = c
        print(json.dumps({"cfg%d" % cfg_id: c}), flush=True)
        del A, B, bias, Xtr, Xte, d, last
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
