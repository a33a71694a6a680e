"""What item exposure (return_exposure) costs: a device-resident call of BASELINE configs 2, 3 and 4 with and without it,
exposure_count_kernel on its own, and the host route it replaces (top-K ids and scores copied to the host, numpy.bincount).

    python tools/exposure_bench.py [--configs 2 3 4] [--reps 5] [--out FILE]

Calls are timed with a host clock around a call that ends in a device synchronise (plus the call's own timing.total_ms),
alternating the two variants.  The kernel alone comes from a separate torch.profiler run of one call.  Prints one JSON document
and, with --out, writes it to FILE as well.  Needs a CUDA device: there is no CPU path to measure."""
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 3, 4])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()

    import torch
    import recometrics_b200 as rb
    from tools import synth

    if not torch.cuda.is_available() or rb.device_count() == 0:
        raise SystemExit("exposure_bench.py: no CUDA device -- nothing to measure")
    dev = torch.device("cuda", 0)
    doc = {"gpu": gpu_info(), "reps": args.reps, "configs": {}}
    for cfg_id in args.configs:
        cfg = synth.CONFIGS[cfg_id]
        d = synth.make(cfg_id)
        m, n = d["X_test"].shape
        A, B = torch.from_numpy(d["A"]).to(dev), torch.from_numpy(d["B"]).to(dev)
        bias = None if d["item_biases"] is None else torch.from_numpy(d["item_biases"]).to(dev)
        Xtr = rb.DeviceCSR.from_scipy(d["X_train"], 0, cfg.dtype, with_data=False)
        Xte = rb.DeviceCSR.from_scipy(d["X_test"], 0, cfg.dtype)
        names = dict(p="precision", tp="trunc_precision", r="recall", ap="average_precision", tap="trunc_average_precision",
                     ndcg="ndcg", hit="hit", rr="rr", roc="roc_auc", pr="pr_auc")
        kw = dict(k=cfg.k, item_biases=bias, break_ties_with_noise=False, cumulative=cfg.cumulative, min_pos_test=cfg.min_pos_test,
                  **{name: q in cfg.metrics for q, name in names.items()})

        def call(**extra):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = rb.calc_reco_metrics_device(Xtr, Xte, A, B, means_only=True, **kw, **extra)
            torch.cuda.synchronize()
            return r, (time.perf_counter() - t0) * 1e3

        def host_route():
            # what a user does without the feature: the ranked lists (ids and scores) to the host, then numpy.bincount
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = rb.calc_reco_metrics_device(Xtr, Xte, A, B, means_only=True, return_topk=True, **kw)
            ids, _ = r.topk_items.cpu().numpy(), r.topk_scores.cpu().numpy()
            counts = np.bincount(ids[ids >= 0], minlength=n)
            return counts, (time.perf_counter() - t0) * 1e3

        call(), call(return_exposure=True)            # warm-up: modules, workspace cache
        rows = {"plain": [], "exposure": [], "plain_total_ms": [], "exposure_total_ms": []}
        for _ in range(args.reps):
            r0, w0 = call()
            r1, w1 = call(return_exposure=True)
            rows["plain"].append(w0); rows["plain_total_ms"].append(r0.timing["total_ms"])
            rows["exposure"].append(w1); rows["exposure_total_ms"].append(r1.timing["total_ms"])
        host = [host_route() for _ in range(2)]
        assert np.array_equal(host[-1][0], r1.exposure.cpu().numpy()), "host route and the library count differently"
        # the kernel alone, from a profiled call of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(return_exposure=True)
        ks = [e for e in prof.events() if "exposure_count_kernel" in e.name]
        kernel_ms = sum(e.device_time for e in ks) / 1e3
        med = lambda v: float(np.median(v))
        c = {"shape": cfg.name, "m": m, "n": n, "k": cfg.k, "scoring_path": int(r1.timing["scoring_path"]),
             "entries": r1.catalogue["entries"], "users": r1.catalogue["users"], "catalogue": r1.catalogue,
             "call_ms_plain": [round(x, 2) for x in rows["plain"]], "call_ms_exposure": [round(x, 2) for x in rows["exposure"]],
             "total_ms_plain": [round(x, 2) for x in rows["plain_total_ms"]],
             "total_ms_exposure": [round(x, 2) for x in rows["exposure_total_ms"]],
             "median_overhead_ms": round(med(rows["exposure"]) - med(rows["plain"]), 3),
             "median_overhead_pct": round(100 * (med(rows["exposure"]) / med(rows["plain"]) - 1), 2),
             "exposure_count_kernel_ms": round(kernel_ms, 3), "exposure_count_kernel_launches": len(ks),
             "host_route_ms": [round(h[1], 1) for h in host]}
        doc["configs"]["cfg%d" % cfg_id] = c
        print(json.dumps({"cfg%d" % cfg_id: c}), flush=True)
        del A, B, bias, Xtr, Xte, d
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
