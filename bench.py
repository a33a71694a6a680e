#!/usr/bin/env python
"""bench.py -- evaluated users/sec of the per-user evaluation path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle/_ref)

A "step" is one pass of the hot path (one calc_metrics call) over one batch of synthetic input: the
users of the configuration named in config.workload (default: BASELINE configs[3], the 1M x 1M
catalogue the north-star quotes its target on; it fits one B200).  One process per GPU; under
torchrun the configuration's users are block-partitioned over the ranks ("strong" scaling, the default:
BASELINE configs[3] is "1M users x 1M items, user-sharded at 1/2/4/8 B200") or, with `--scaling weak`,
every rank evaluates its own `--users` users; either way against its own replica of B and with no
data-path collective: the path has no exchange step.

  value     users/s with A, B, the CSR matrices and the outputs resident in HBM when the timed
            region starts (C-ABI call with inputs_on_device=1), CUDA events, max over ranks.
  e2e       the same call through the reference-facing API with HOST (pinned) buffers: host->device
            copies of that step's inputs and device->host copies of its metric rows inside the timed
            region.
  roofline  of the dominant scoring kernel: algorithmic flops 2*p'*sum_eligible(n-ntrain) (SURVEY 8(d)) / the kernel's
            CUDA-event time.  Top-K-only workloads run the tensor-core candidate filter (filter_select_kernel, fp16 MMAs):
            bound "tensor", peak = the driver-measured sustained bf16 figure of MEASURED_PEAKS.json.  Rank counting
            (ROC/PR-AUC) runs the FMA tiles (score_select_kernel): bound "fp32_fma"/"fp64_fma", peak = the FMA
            microbenchmark run live before the timed region.  traffic = DRAM bytes of one launch from the committed ncu
            capture (profiles/roofline_traffic.json).
  e2e_pageable  e2e with ordinary (pageable) numpy buffers -- what the reference's callers pass: the library's
            host-thread upload pipeline is then inside the timed region.
  cpu_baseline  the reference's own OpenMP/SIMD implementation (oracle/_ref; the C port if absent)
            on this box's host cores, on a bounded prefix of the same users.
  parity    the metric rows the CPU baseline computed for that prefix against the rows the timed e2e call wrote for the
            same users: {users, rows compared, mismatches beyond 1e-6 / NaN pattern, largest difference}.

`--dump-outputs DIR` writes the metric rows of the last timed step as DIR/<metric>.npy, the defined values, and
DIR/<metric>_defined.npy, where they are defined (see dump_outputs), so that two builds can be compared output for output:
with the same arguments the inputs are the same from run to run.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (it may be read-only)
from tools import synth  # noqa: E402

METRIC = "evaluated_users_per_sec"
UNIT = "users/s"
DUMP_BYTES = 60 << 20      # --dump-outputs: array bytes of all files, under 64 MB with the .npy headers
METRIC_FLAGS = dict(p="precision", tp="trunc_precision", r="recall", ap="average_precision",
                    tap="trunc_average_precision", ndcg="ndcg", hit="hit", rr="rr", roc="roc_auc", pr="pr_auc")


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def workload_name(cfg, users_total, gpus, scaling):
    return "%s; %d users in all, block-partitioned over %d GPU(s) (%s scaling)" % (cfg.name, users_total, gpus, scaling)


def dump_outputs(out_dir, rows, rank, world):
    """Write this rank's metric rows (name -> (users,) or (users, K) array) to out_dir, every file finite: a metric is NaN
    where the reference leaves it undefined (a user without test items or with too few candidates), so <name>.npy holds
    the defined values in user order and <name>_defined.npy (float32, the rows' shape) 1 where a value is defined and 0
    where the caller gets NaN.  Under torchrun the names end in _rank<r>.  The ranks share DUMP_BYTES; when the files
    would be larger, the same seeded sample of users is kept in every file."""
    os.makedirs(out_dir, exist_ok=True)
    m = next(iter(rows.values())).shape[0]
    row_bytes = sum((v.nbytes + 4 * v.size) // max(m, 1) for v in rows.values())
    keep = min(m, DUMP_BYTES // world // max(row_bytes, 1))
    users = None if keep == m else np.sort(np.random.default_rng(12345 + rank).choice(m, keep, replace=False))
    tail = "" if world == 1 else "_rank%d" % rank
    for name, v in rows.items():
        v = v if users is None else v[users]
        defined = np.isfinite(v)
        np.save(os.path.join(out_dir, name + tail + ".npy"), v[defined])
        np.save(os.path.join(out_dir, name + "_defined" + tail + ".npy"), defined.astype(np.float32))


# ----------------------------------------------------------------------------- CPU arms
def cpu_arm_callable():
    """The CPU implementation to time: the compiled reference when it travelled, else the C port."""
    import oracle
    oracle.build()
    if oracle.have_ref():
        oracle.use_best_ref_build_for_timing()      # the build closest to -march=native on this host (BASELINE.md section 3)
        return "reference", oracle
    return "port", oracle


def run_cpu(kind, oracle, d, cfg, nthreads, want_rows=False):
    A, B = synth.fold_biases(d["A"], d["B"], d["item_biases"])   # what the reference front-end does
    kw = dict(metrics=cfg.metrics, cumulative=cfg.cumulative, nthreads=nthreads, min_pos_test=cfg.min_pos_test,
              dtype=cfg.dtype)
    t0 = time.perf_counter()
    if kind == "reference":
        rows = oracle.ref_calc(A, B, d["X_train"], d["X_test"], cfg.k, **kw)
    else:
        rows = oracle.oracle_calc(A, B, d["X_train"], d["X_test"], cfg.k, fix_quirks=False, **kw)
    if want_rows:
        return time.perf_counter() - t0, rows
    return time.perf_counter() - t0


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def sources_hash(name=None):
    """Identifies the kernel source the committed ncu traffic figure was captured on (profiles/roofline_traffic.json)."""
    h = hashlib.sha1()
    src = os.path.join(ROOT, "recometrics_b200", "csrc")
    for fn in sorted(os.listdir(src)):
        if (name is None and fn.endswith((".cu", ".cuh"))) or fn == name:
            h.update(open(os.path.join(src, fn), "rb").read())
    return h.hexdigest()[:12]


def cpu_sample_size(kind, oracle, cfg, cores, target_s, n_items):
    """Pilot on a few users, then size the sample for ~target_s seconds of CPU work."""
    pilot = max(2 * cores, 16)
    d = synth.make(cfg.cfg_id, m=pilot, n=n_items)
    dt = max(run_cpu(kind, oracle, d, cfg, cores), 1e-4)
    users = int(min(max(pilot, target_s * pilot / dt), 200000))
    users = max(cores, (users // cores) * cores)
    return users


def reference_arm(args, cfg, rank):
    """--impl reference: the reference's CPU path, all host threads, bounded sample per step."""
    if rank != 0:
        return
    kind, oracle = cpu_arm_callable()
    cores = os.cpu_count() or 1
    users = cpu_sample_size(kind, oracle, cfg, cores, 4.0, args.items)
    d = synth.make(cfg.cfg_id, m=users, n=args.items)
    for _ in range(args.warmup):
        run_cpu(kind, oracle, d, cfg, cores)
    t = [run_cpu(kind, oracle, d, cfg, cores) for _ in range(args.steps)]
    sec = float(np.mean(t))
    value = users / sec
    sample = "first %d users of the workload per step (users are independent; OpenMP schedule(dynamic))" % users
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32" if cfg.dtype == np.float32 else "f64", "data": "synthetic",
        "config": {"workload": workload_name(cfg, args.users_total, args.gpus, args.scaling), "items": args.items, "k_metrics": cfg.k,
                   "factors": cfg.p, "metrics": list(cfg.metrics), "cpu_sample_users_per_step": users},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "cpu": cpu_model(),
                         "build": getattr(oracle, "ref_build_note", lambda: None)()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        if os.environ.get("RMB200_BENCH_NO_SAMPLER") == "1":       # developer: is the sampler itself visible in the timing?
            return
        try:
            fd, self.path = tempfile.mkstemp(prefix="rmb200_clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], [], set(), []
        try:
            for ln in open(self.path):
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            hot = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
            out = {"sm_mhz": float(np.median(hot)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                   "samples": len(sm), "power_w_max": float(max(power))}
        return out


# ----------------------------------------------------------------------------- product arm
def product_arm(args, cfg, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import recometrics_b200 as rb
    from recometrics_b200 import _capi

    if not torch.cuda.is_available() or rb.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path to measure")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    T = cfg.dtype
    tdt = torch.float32 if T == np.float32 else torch.float64
    # this rank's block of the workload's users (strong: the configuration's users split over the ranks; weak: --users each);
    # rank r draws its users from its own streams, the item factors are the same on every rank (B is replicated)
    users = args.users_total * (rank + 1) // world - args.users_total * rank // world
    d = synth.make(cfg.cfg_id, m=users, n=args.items, seed_shift=rank, shared_items=True)
    A, B, bias = d["A"], d["B"], d["item_biases"]
    Xtr, Xte = d["X_train"], d["X_test"]
    if args.zero_users > 0:
        # users unseen in training have all-zero factors (every score equal -> NaN row): the tensor-core filter settles them
        # without scoring and nobody else's batch pays for them (VERDICT r01: one such row used to send its whole batch to the FMA tiles)
        zr = np.random.default_rng(99 + rank).random(A.shape[0]) < args.zero_users
        A[zr] = 0
    m, n, p = A.shape[0], B.shape[0], A.shape[1]
    K = cfg.k
    flops = synth.algorithmic_flops(cfg, Xtr, Xte, has_ndcg="ndcg" in cfg.metrics)
    rs = K if cfg.cumulative else 1

    def pinned(x):
        t = torch.from_numpy(np.ascontiguousarray(x))
        try:
            return t.pin_memory()
        except Exception:
            return t

    # host side (pinned) for e2e; device side for `value`
    hA, hB = pinned(A), pinned(B)
    hb = pinned(bias) if bias is not None else None
    htrp, htri, htep, htei = pinned(Xtr.indptr), pinned(Xtr.indices), pinned(Xte.indptr), pinned(Xte.indices)
    htev = pinned(Xte.data.astype(T))
    houts = {q: pinned(np.empty(m * (rs if q in _capi.TOPK_METRICS else 1), dtype=T)) for q in cfg.metrics}
    dA, dB = hA.to(dev), hB.to(dev)
    db = hb.to(dev) if hb is not None else None
    dtrp, dtri, dtep, dtei, dtev = (x.to(dev) for x in (htrp, htri, htep, htei, htev))
    douts = {q: torch.empty(m * (rs if q in _capi.TOPK_METRICS else 1), dtype=tdt, device=dev) for q in cfg.metrics}

    def call(on_device, timing):
        ex = _capi.make_extra(device=local_rank, inputs_on_device=on_device, timing=timing)
        if on_device:
            ptr = lambda t: t.data_ptr() if t is not None else None
            outs = {q: v.data_ptr() for q, v in douts.items()}
            rc = _capi.calc_metrics(T, ptr(dA), p, ptr(dB), p, m, n, p, ptr(dtrp), ptr(dtri), ptr(dtep), ptr(dtei), ptr(dtev),
                                    K, cfg.cumulative, False, outs, True, 2, cfg.min_pos_test, item_biases=ptr(db), extra=ex)
        else:
            npv = lambda t: t.numpy() if t is not None else None
            outs = {q: v.numpy() for q, v in houts.items()}
            rc = _capi.calc_metrics(T, npv(hA), p, npv(hB), p, m, n, p, npv(htrp), npv(htri), npv(htep), npv(htei), npv(htev),
                                    K, cfg.cumulative, False, outs, True, 2, cfg.min_pos_test, item_biases=npv(hb), extra=ex)
        _capi.raise_for_status(rc)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # measured FMA peak (roofline denominator) -- before the timed region
    peak_tflops, _ = _capi.measure_fma_peak(local_rank, T)

    # ---- device-resident timing: W warm-up steps, then exactly K timed steps
    tm = _capi.Timing()
    for _ in range(args.warmup):
        call(True, tm)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms, launches, path, fallbacks, retry_rows = 0.0, 0, 0, 0, 0
    phases = {}
    wall_calls_ms = 0.0
    e0.record()
    for _ in range(args.steps):
        t_w = time.perf_counter()
        call(True, tm)
        wall_calls_ms += (time.perf_counter() - t_w) * 1e3
        kernel_ms += tm.dominant_kernel_ms
        launches += tm.kernel_launches
        for f in ("total_ms", "prep_ms", "score_select_ms", "metrics_ms"):
            phases[f] = phases.get(f, 0.0) + getattr(tm, f) / args.steps
        path, fallbacks = int(tm.scoring_path), fallbacks + int(tm.filter_fallback_batches)
        retry_rows += int(tm.filter_retry_rows)
    e1.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:
        # the rows the last timed step wrote (the e2e and pageable legs below write their own buffers)
        dump_outputs(args.dump_outputs, {METRIC_FLAGS[q]: v.cpu().numpy().reshape(m, -1) if cfg.cumulative and q in _capi.TOPK_METRICS
                                         else v.cpu().numpy() for q, v in douts.items()}, rank, world)
    dev_ms = e0.elapsed_time(e1)
    per_rank = None
    if world > 1:
        mine = torch.tensor([dev_ms, phases.get("total_ms", 0.0), kernel_ms / args.steps, wall_calls_ms / args.steps], dtype=torch.float64, device=dev)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"ms_per_step": [round(float(x[0]) / args.steps, 2) for x in allr], "call_total_ms": [round(float(x[1]), 2) for x in allr],
                    "kernel_ms": [round(float(x[2]), 2) for x in allr], "host_wall_ms_per_call": [round(float(x[3]), 2) for x in allr]}
        t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    value = args.users_total * args.steps / (dev_ms * 1e-3)

    # ---- end-to-end through the host-pointer C-ABI (H2D of inputs + D2H of metric rows inside)
    call(False, tm)   # one warm-up
    barrier()
    t0 = time.perf_counter()
    h2d = d2h = 0
    for _ in range(args.steps):
        call(False, tm)
        h2d, d2h = tm.h2d_bytes, tm.d2h_bytes
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = args.users_total * args.steps / e2e_s

    # ---- the same with ordinary (pageable) numpy buffers, what the reference's callers pass (upload pipeline inside)
    def call_pageable():
        ex = _capi.make_extra(device=local_rank, inputs_on_device=False, timing=tm)
        rc = _capi.calc_metrics(T, A, p, B, p, m, n, p, Xtr.indptr, Xtr.indices, Xte.indptr, Xte.indices, pg_tev,
                                K, cfg.cumulative, False, pg_outs, True, 2, cfg.min_pos_test, item_biases=bias, extra=ex)
        _capi.raise_for_status(rc)
    pg_tev = np.ascontiguousarray(Xte.data, dtype=T)
    pg_outs = {q: np.empty(m * (rs if q in _capi.TOPK_METRICS else 1), dtype=T) for q in cfg.metrics}
    call_pageable()
    barrier()
    t0 = time.perf_counter()
    pg_steps = args.steps
    for _ in range(pg_steps):
        call_pageable()
    barrier()
    pg_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([pg_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pg_s = float(t.item())
    e2e_pageable = {"value": args.users_total * pg_steps / pg_s, "unit": UNIT, "ms_per_step": pg_s * 1e3 / pg_steps, "steps": pg_steps,
                    "note": "host inputs and outputs in pageable numpy memory (the reference's callers): the library's host-thread upload pipeline is inside"}

    # ---- roofline of the dominant kernel (score_select): algorithmic flops / CUDA-event kernel time
    ach = flops * args.steps / (kernel_ms * 1e-3) / 1e12
    traffic, traffic_note, captured_users = None, None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(str(cfg.cfg_id))
            if isinstance(traffic, dict):      # DRAM bytes of one launch of the dominant kernel, from the committed ncu capture
                traffic_note = "%s; %s" % (traffic.get("per"), traffic.get("source"))
                now = sources_hash(traffic.get("kernel_source"))
                if traffic.get("sources_hash") not in (None, now):
                    traffic_note += "; NOTE: captured on %s %s, this build has %s (the kernel source changed since the capture)" % (
                        traffic.get("kernel_source", "sources"), traffic.get("sources_hash"), now)
                captured_users = traffic.get("users_per_launch")
                traffic = int(traffic["dram_bytes_read"]) + int(traffic["dram_bytes_write"])
        except Exception:
            traffic = None
    big = path == 2 and (-(-n // 128) * 128) * (-(-(p + (1 if bias is not None else 0)) // 16) * 16) * 2 > (160 << 20)
    batches = -(-m // ((4 if big else 8) * 148 * 128))      # (api.cu: a user batch is 8 waves of 148 CTAs x 128 users, 4 on very large catalogues)
    users_per_launch = min(m, (4 if big else 8) * 148 * 128)
    try:
        if traffic is not None and captured_users and int(captured_users) != users_per_launch:
            # every wave of 148 CTAs streams the item image once: DRAM bytes of a launch go with its number of waves
            traffic = int(round(traffic * users_per_launch / int(captured_users)))
            traffic_note = (traffic_note or "") + "; scaled by %d/%d: the capture was a launch of %d users, a launch of this run has %d" % (
                users_per_launch, int(captured_users), int(captured_users), users_per_launch)
    except Exception:       # noqa: BLE001  (bookkeeping must never fail the bench)
        pass
    if path == 2:
        # tensor-core filter: every (user, item) score is an MMA on fp16 copies of the factors (tcgen05 kind::f16 runs
        # fp16 and bf16 operands at the same rate); the measured denominator is the driver's cuBLAS bf16 figure
        # (sustained: the kernel IS the long step)
        try:
            mp0 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            tpeak, tsrc = float(mp0["bf16_tflops_sustained"]), "MEASURED_PEAKS.json bf16_tflops_sustained (of measured); burst %.1f" % mp0["bf16_tflops"]
        except Exception:
            tpeak, tsrc = 1400.0, "fallback 1.4 PFLOP/s sustained bf16 (B200_PROFILING.md; of fallback)"
        roofline = {
            "bound": "tensor", "achieved": ach, "peak": tpeak, "unit": "TFLOP/s", "frac": ach / tpeak, "traffic": traffic,
            "kernel": "filter_select_kernel (tcgen05 fp16 candidate filter, fp32 accumulation in TMEM; survivors re-scored exactly in %s by exact_topk_kernel)" % ("fp32" if T == np.float32 else "fp64"),
            "kernel_ms_per_step": kernel_ms / args.steps, "kernel_share_of_step": kernel_ms / dev_ms if world == 1 else None,
            "algorithmic_flops_per_step": flops, "launches_per_step": batches, "peak_source": tsrc,
            "fma_peak_tflops_live": peak_tflops, "filter_fallback_batches": fallbacks, "filter_retry_rows": retry_rows,
        }
    else:
        roofline = {
            "bound": "fp32_fma" if T == np.float32 else "fp64_fma", "achieved": ach, "peak": peak_tflops, "unit": "TFLOP/s",
            "frac": ach / peak_tflops if peak_tflops > 0 else None, "traffic": traffic,
            "kernel": "score_select_kernel", "kernel_ms_per_step": kernel_ms / args.steps,
            "kernel_share_of_step": kernel_ms / dev_ms if world == 1 else None,
            "algorithmic_flops_per_step": flops, "launches_per_step": batches,
            "peak_source": "FMA microbenchmark run live on this GPU (rmb200_measure_fma_peak): MEASURED_PEAKS.json holds "
                           "HBM and bf16-tensor peaks only; nominal %s" % ("74.4 TFLOP/s FP32" if T == np.float32 else "37.2 TFLOP/s FP64"),
        }
    if traffic_note:
        roofline["traffic_note"] = traffic_note
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        roofline["hbm_peak_gbs_measured"] = mp.get("hbm_gbs")
    except Exception:
        pass

    # ---- CPU baseline: the reference's implementation on this box's cores (rank 0, N=1 only)
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        kind, oracle = cpu_arm_callable()
        cores = os.cpu_count() or 1
        cu = cpu_sample_size(kind, oracle, cfg, cores, 12.0, args.items)
        cu = min(cu, m)
        dd = synth.make(cfg.cfg_id, m=cu, n=args.items)
        sec, cpu_rows = run_cpu(kind, oracle, dd, cfg, cores, want_rows=True)
        cpu = {"value": cu / sec, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model(),
               "build": getattr(oracle, "ref_build_note", lambda: None)(),
               "sample": "first %d users of the workload, %d threads, %.1f s" % (cu, cores, sec)}
        # the rows the timed e2e call wrote for the same users (synth is block-reproducible: the prefix is bit-identical)
        bad_users = np.zeros(cu, dtype=bool)
        worst, rows_cmp = 0.0, 0
        for q in cfg.metrics:
            w = rs if q in _capi.TOPK_METRICS else 1
            g = houts[q].numpy()[: cu * w].reshape(cu, w).astype(np.float64)
            c = np.asarray(cpu_rows[q]).reshape(cu, w).astype(np.float64)
            both_nan = np.isnan(g) & np.isnan(c)
            diff = np.where(both_nan, 0.0, np.abs(g - c))
            diff = np.where(np.isnan(diff), np.inf, diff)          # NaN on one side only
            bad_users |= (diff > 1e-6).any(axis=1)
            worst = max(worst, float(diff.max()) if diff.size else 0.0)
            rows_cmp += cu
        # the north-star's exception: two scores within a 1e-6 relative gap where their order matters (float64 re-scoring decides;
        # "relative" to the user's score scale, tests/parity_utils.py).  Every mismatching user must be such a user.
        unexplained, checked = 0, 0
        bad_idx = np.nonzero(bad_users)[0][:400]
        if bad_idx.size:
            B64 = dd["B"].astype(np.float64)
            b64 = None if dd["item_biases"] is None else dd["item_biases"].astype(np.float64)
            for u in bad_idx:
                sc = dd["A"][u].astype(np.float64) @ B64.T
                if b64 is not None:
                    sc = sc + b64
                tr = dd["X_train"].indices[dd["X_train"].indptr[u]:dd["X_train"].indptr[u + 1]]
                te = dd["X_test"].indices[dd["X_test"].indptr[u]:dd["X_test"].indptr[u + 1]]
                sc[tr] = -np.inf
                order = np.sort(sc[np.isfinite(sc)])[::-1]
                tol = 1e-6 * max(abs(order[0]), abs(order[-1]))
                near = bool(np.any(np.abs(np.diff(order[: K + 1])) <= tol))
                if not near and ("roc" in cfg.metrics or "pr" in cfg.metrics):
                    asc = order[::-1]
                    for it in te:
                        lo, hi = np.searchsorted(asc, sc[it] - tol, "left"), np.searchsorted(asc, sc[it] + tol, "right")
                        if hi - lo > 1:
                            near = True
                            break
                checked += 1
                unexplained += 0 if near else 1
        parity = {"users": int(cu), "metric_rows": int(rows_cmp), "mismatched_users": int(bad_users.sum()), "tolerance": 1e-6,
                  "mismatched_users_checked_in_float64": int(checked), "mismatched_users_without_a_1e-6_near_tie": int(unexplained),
                  "max_abs_diff": worst, "nan_rows_cpu": int(np.isnan(np.asarray(cpu_rows[cfg.metrics[0]]).reshape(cu, -1)[:, 0]).sum()),
                  "against": "cpu_baseline rows (%s) vs the rows of the timed e2e call, same users" % kind}

    split = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        split = split_block()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if T == np.float32 else "f64", "data": "synthetic",
            "config": {"workload": workload_name(cfg, args.users_total, world, args.scaling), "users_total": args.users_total,
                       "users_per_gpu": m, "items": n, "factors": p,
                       "k_metrics": K, "metrics": list(cfg.metrics), "cumulative": bool(cfg.cumulative),
                       "l2": "inputs (A+B+CSR = %.0f MB) larger than the 126 MB L2; no flush" % (
                           (A.nbytes + B.nbytes + Xtr.indices.nbytes + Xte.indices.nbytes) / 1e6),
                       "scoring_path": {1: "fma", 2: "tensor filter + exact re-score", 3: "full order"}.get(path, "?"),
                       **({"zero_factor_users": args.zero_users} if args.zero_users > 0 else {}),
                       "parallelism": "users block-partitioned, B replicated, no data-path collective"},
            "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world,
                    "ms_per_step": e2e_s * 1e3 / args.steps, "host_buffers": "pinned"},
            "e2e_pageable": e2e_pageable,
            "gpu_launches": int(launches) * world, "clocks": clocks, "per_rank": per_rank,
            "phases_ms_per_step": {k: round(v, 3) for k, v in phases.items()},
            "split": split,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def split_block():
    """A side measurement, NOT part of the headline: the step before the evaluation (SURVEY section 8 row f-4), one train/test
    split of a MovieLens-20M-shaped matrix through the C-ABI (host buffers in, host arrays out) beside the reference's own
    splitter on one host thread (it is sequential), outputs compared entry for entry.  Never fails the bench."""
    try:
        from recometrics_b200 import _capi
        from tools.split_once import power_law_matrix
        import oracle
        m, n = 138493, 26744
        p, i, v = power_law_matrix(m, n, 144.0)
        best, res = None, None
        for _ in range(4):
            t0 = time.perf_counter()
            res = _capi.split("all", p, i, v, m, n, test_fraction=0.3, seed=1)
            ms = (time.perf_counter() - t0) * 1e3
            best = ms if best is None else min(best, ms)
        out = {"workload": "split_reco_train_test(split_type='all'): %d users x %d items, %d entries, f32" % (m, n, i.size),
               "ms": round(best, 2), "entries_per_s": round(i.size / (best * 1e-3)), "library_timing": res["timing"]}
        if oracle.have_ref():
            t0 = time.perf_counter()
            r = oracle.ref_split(p, i, v, m, n, split_type="all", test_fraction=0.3, seed=1)
            out["reference_ms"] = round((time.perf_counter() - t0) * 1e3, 2)
            out["identical_to_reference"] = bool(all(np.array_equal(x, y) for key in ("train", "test") for x, y in zip(r[key], res[key][:3])))
        return out
    except Exception as e:      # noqa: BLE001
        return {"error": "%s: %s" % (type(e).__name__, e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=4, help="BASELINE.json configs index + 1 (default 4: 1M x 1M, K=100)")
    ap.add_argument("--users", type=int, default=0, help="users: in all (strong scaling) / per GPU (weak); default: the configuration's m")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: split the configuration's users over the GPUs (strong, default) or give every GPU that many (weak)")
    ap.add_argument("--items", type=int, default=0, help="items (default: the configuration's n)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--zero-users", type=float, default=0.0, help="fraction of users whose factors are set to zero (robustness line)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the metric rows of the last timed step as DIR/<metric>.npy (the defined values) and "
                         "DIR/<metric>_defined.npy (1 where defined, 0 where NaN); at most 64 MB in all: larger outputs "
                         "as a fixed seeded sample of users")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what this repository's CUDA path computed (--impl b200)")

    cfg = synth.CONFIGS[args.config]
    args.users = args.users or cfg.m
    args.items = args.items or cfg.n
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    args.users_total = args.users * (max(world, args.gpus) if args.scaling == "weak" else 1)
    if world == 1 and args.gpus > 1 and args.impl == "b200":
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    if args.impl == "reference":
        reference_arm(args, cfg, rank)
    else:
        product_arm(args, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
