#!/usr/bin/env python
"""Benchmark of the audit-sweep hot path (BASELINE.json: constraint x object evaluations / second).

  python bench.py --gpus N --steps K --warmup W              # this framework, one rank per GPU (torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...    # the reference's CPU path (C++ restatement) on the host cores
  python bench.py --config 4|5 [--scaling strong]            # the other BASELINE.json sweep configs (default: 2 = configs[1])
  python bench.py --config 3                                 # admission replay: 64-request micro-batches x 200 constraints
  python bench.py ... --dump-outputs DIR                     # also write the last timed step's results to DIR/*.npy

Workload (config.workload), default: BASELINE.json configs[1] -- "audit sweep: 10 templates, 50 constraints, 1M synthetic
Pods on 1 B200".  Weak scaling: every rank evaluates its own 1M-Pod shard of the cluster and the violation bitmaps are
exchanged once per step (the one exchange the path has, SURVEY.md 8(e)); `--scaling strong` keeps the total at --objects.

One step = one pass of the hot path over the batch: the fused match-prefilter + predicate kernel over the column-wise batch
resident in HBM, producing the violation/error bitmaps and per-constraint totals, plus (N > 1) the exchange.  `value` is
device-timed (CUDA events, max over ranks) with inputs resident; `e2e` goes through the public API (gk_review_blob) with the
raw JSON of a DIFFERENT page of objects in pinned host memory every step: H2D of the JSON -> device ingest (tokenise, extract
columns) -> kernel -> D2H of the bitmaps and totals.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "constraint_object_evals_per_sec_audit_sweep"
UNIT = "evals/s"
L2_BYTES = 126 * 1024 * 1024


def env_int(k, d):
    try:
        return int(os.environ.get(k, d))
    except ValueError:
        return d


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc = None
        self.lines = []
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ workloads
def workload(cfg: int):
    """(templates, constraints, namespaces, synth mode, objects per GPU by default, label)"""
    from gatekeeper_b200 import workloads as W
    if cfg == 2:
        tm, cons = W.config2()
        return tm, cons, W.synth_namespaces(), 0, 1_000_000, "audit sweep: 10 gatekeeper in-tree templates, 50 constraints, 1M synthetic Pods per GPU (BASELINE.json configs[1])"
    if cfg == 4:
        tm, cons = W.config4()
        return tm, cons, W.synth_namespaces(), 1, 1_250_000, "K8sPSP* suite (5 templates) x mixed-GVK objects, 10M over 8 GPUs = 1.25M per GPU (BASELINE.json configs[3])"
    if cfg == 5:
        tm, cons = W.config5()
        return tm, cons, W.synth_namespaces(), 0, 625_000, "K8sAllowedRepos prefix lists + namespace / name wildcards x Pods, 5M over 8 GPUs = 625k per GPU (BASELINE.json configs[4])"
    raise SystemExit("bench.py: --config must be 2, 3, 4 or 5")


# ------------------------------------------------------------------------------------------------ CPU legs (test / bench infrastructure)
def cpu_ref_engine(cfg):
    from oracle.cpu_ref import CpuRef
    tm, cons, nss, mode, _, _ = workload(cfg)
    ref = CpuRef()
    for k, r, *rest in tm:
        ref.add_template(k, r)
    for c in cons:
        ref.add_constraint(c)
    for ns in nss:
        ref.add_namespace(ns)
    return ref, len(cons), mode


def python_oracle_rate(cfg, sample=300):
    """single-core Python oracle (oracle/k8s.py + oracle/rego.py), for the record beside the C++ restatement"""
    from gatekeeper_b200 import workloads as W
    from oracle import k8s
    tm, cons, nss, mode, _, _ = workload(cfg)
    c = k8s.Client()
    for k, r, *rest in tm:
        c.add_template(k, r)
    for x in cons:
        c.add_constraint(x)
    nsd = {n["metadata"]["name"]: n for n in nss}
    for n in nss:
        c.add_namespace(n)
    blob = W.synth_objects(0, sample, mode=mode, threads=1)
    t0 = time.perf_counter()
    for i in range(sample):
        obj = json.loads(blob.get(i))
        c.review(k8s.Review(obj=obj, ns=nsd.get((obj.get("metadata") or {}).get("namespace", "")), source="Original"), k8s.AUDIT_EP)
    return sample * len(cons) / (time.perf_counter() - t0)


def cpu_baseline(cfg, sample_objects):
    from gatekeeper_b200 import workloads as W
    from gatekeeper_b200.hostinfo import host_cpus
    from oracle import k8s
    ref, C, mode = cpu_ref_engine(cfg)
    cores = max(1, host_cpus())
    blob = W.synth_objects(0, sample_objects, mode=mode)
    ref.review_blob(blob, k8s.AUDIT_EP, cores)                      # warm-up (thread-private copies, allocator)
    _, nres, _, secs = ref.review_blob(blob, k8s.AUDIT_EP, cores)
    py = python_oracle_rate(cfg, 200)
    ref.close()
    return {"value": sample_objects * C / secs, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"oracle/cpu_ref.cpp: C++ restatement of Client.Review (match pre-filter + one Rego evaluation per matching constraint x object, "
                      f"one JSON parse per object) on {cores} host threads, first {sample_objects} objects of the workload x {C} constraints, {secs:.2f} s, "
                      f"{nres} results; the single-core Python oracle (oracle/k8s.py) does {py:.0f} evals/s on the same objects"}


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    from gatekeeper_b200 import workloads as W
    from gatekeeper_b200.hostinfo import host_cpus
    from oracle import k8s
    cfg = args.config if args.config != 3 else 2
    ref, C, mode = cpu_ref_engine(cfg)
    cores = max(1, host_cpus())
    per = args.ref_objects_per_step
    steps, warm = args.steps, max(1, args.warmup)
    blobs = [W.synth_objects(k * per, per, mode=mode) for k in range(min(4, steps + warm))]
    for k in range(warm):
        ref.review_blob(blobs[k % len(blobs)], k8s.AUDIT_EP, cores)
    total_t, total_n = 0.0, 0
    for k in range(steps):
        pairs, _, _, secs = ref.review_blob(blobs[(warm + k) % len(blobs)], k8s.AUDIT_EP, cores)
        total_t += secs
        total_n += per
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [[pairs.get(key, 0) for key in ref.constraints()]])
    value = total_n * C / total_t
    tm, cons, nss, mode, n_default, label = workload(cfg)
    sample = (f"oracle/cpu_ref.cpp (C++ restatement of the reference's Client.Review loop: JSON parse, spec.match pre-filter, one Rego evaluation per matching "
              f"constraint x object) on {cores} host threads (= usable CPUs: affinity + cgroup quota of a {os.cpu_count()}-thread host); each step reviews {per} "
              f"synthetic objects x {C} constraints (a bounded sample of the workload; objects are independent so throughput is size-independent)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * total_t / max(1, steps), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int",
            "data": "synthetic", "config": {"workload": label, "objects_per_step": per, "constraints": C},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))
    ref.close()
    return 0


# ------------------------------------------------------------------------------------------------ output dump (--dump-outputs)
DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, totals, viol=None, err=None):
    """What the last timed step handed its caller, as .npy files that two builds can be compared with:
      totals.npy      float64 [k, C]     per-constraint totals (audit sweep / admission: [violations, matcher errors];
                                         reference arm: [violating objects])
      violations.npy  float32 [rows, C]  1 where object row violates constraint c (the uint32 bitmap `viol`, bit c of word c // 32,
                                         unpacked; with N > 1 the rows of every rank, as gathered)
      errors.npy      float32 [rows', C] 1 where the matcher errored (`err`: the caller's own rows, the first of viol's)
      rows.npy        float64 [rows]     the object index of each row
    Unpacked bits make any difference a whole 1.0.  When every row does not fit in 64 MB, the rows are a fixed seeded sample."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    totals = np.asarray(totals, dtype=np.float64)
    np.save(os.path.join(out_dir, "totals.npy"), totals)
    if viol is None:
        return
    C = totals.shape[1]
    per_row = 2 * 4 * C + 8
    keep = (DUMP_BYTES - totals.nbytes - 4096) // per_row
    n_rows = len(viol)
    rows = np.arange(n_rows) if n_rows <= keep else np.sort(np.random.default_rng(0).choice(n_rows, keep, replace=False))
    cols = np.arange(C)

    def bits(words, idx):
        w = np.asarray(words).view(np.uint32)[idx]
        return ((w[:, cols // 32] >> (cols % 32).astype(np.uint32)) & 1).astype(np.float32)

    np.save(os.path.join(out_dir, "violations.npy"), bits(viol, rows))
    np.save(os.path.join(out_dir, "errors.npy"), bits(err, rows[rows < len(err)]))
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


# ------------------------------------------------------------------------------------------------ GPU arm: audit sweeps
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from gatekeeper_b200 import driver as D
    from gatekeeper_b200 import workloads as W

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback (use --impl reference for the CPU path)")
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # (NCCL's version banner goes to stdout: the bench prints ONE line there)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    tm, cons, nss, mode, n_default, label = workload(args.config)
    from gatekeeper_b200.hostinfo import host_cpus
    host_threads = max(1, host_cpus() // max(1, world))
    drv = D.Driver(device=local, threads=host_threads)
    for k, r, *rest in tm:
        drv.add_template(k, r)
    for c in cons:
        drv.AddConstraint(c)
    for ns in nss:
        drv.AddData("admission.k8s.gatekeeper.sh", ["cluster", "v1", "Namespace", ns["metadata"]["name"]], ns)
    C = len(drv.constraints())
    words = (C + 31) // 32
    n_total = args.objects if args.objects else n_default
    n = n_total // world if args.scaling == "strong" else n_total        # objects of this rank
    shard0 = rank * n
    ingest_mode = drv.Dump().splitlines()[1].strip()
    t0 = time.perf_counter()
    blob = W.synth_objects(shard0, n, mode=mode, threads=host_threads)
    gen_s = time.perf_counter() - t0
    drv.pin_blob(blob)
    rb = drv.upload_blob(blob)                       # ingest once: inputs resident for the `value` leg
    alg_in = rb.alg_bytes
    alg_bytes = alg_in + n * words * 4 * 2           # + violation and error planes written

    from gatekeeper_b200.sweep import ShardedSweep
    sweep = ShardedSweep(drv, rb, n, C, dev, world)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if alg_in < 2 * L2_BYTES else None
    ep = D.AUDIT_EP
    stream = torch.cuda.current_stream()

    def step(e0=None, e1=None):
        if flush is not None:
            flush.fill_(1)                            # evict L2 between iterations when the batch could fit in it
        if e0 is not None:
            e0.record(stream)
        sweep.evaluate(ep, stream)                    # the fused match + predicate kernel over the resident shard
        if e1 is not None:
            e1.record(stream)
        sweep.exchange()                              # N > 1: bitmap + totals exchange

    W_ = max(3, args.warmup)
    for _ in range(W_):
        step()
    torch.cuda.synchronize()
    launches0 = rb.eval(ep, D.F_NO_COPY_BACK).stats["gpu_launches"]     # engine launch counter before the timed region
    if world > 1:
        dist.barrier()
    K = args.steps
    e0 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    e1 = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    torch.cuda.synchronize()
    ev_a.record(stream)
    for k in range(K):
        step(e0[k], e1[k])
    ev_b.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if args.dump_outputs and rank == 0:
        viol = sweep.viol if sweep.gathered is None else sweep.gathered.reshape(-1, words)
        dump_outputs(args.dump_outputs, sweep.tot[:, :C].cpu().numpy(), viol.cpu().numpy(), sweep.err.cpu().numpy())
    total_ms = ev_a.elapsed_time(ev_b)
    kern_ms = sum(a.elapsed_time(b) for a, b in zip(e0, e1)) / K
    t = torch.tensor([total_ms, kern_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = float(t[0]), float(t[1])
    ms_per_step = total_ms / K
    value = world * n * C / (ms_per_step / 1e3)
    launches = rb.eval(ep, D.F_NO_COPY_BACK).stats["gpu_launches"] - launches0 - 1   # minus this probe's own launch
    totals_host = sweep.tot[0].tolist()              # after the exchange: summed over ranks
    sweep.evaluate(ep, stream)                       # this rank's own totals again (untimed), to check the e2e path against
    torch.cuda.synchronize()
    totals_local = sweep.tot_local[0].tolist()
    if world > 1:
        ref = sweep.tot_local.clone()
        dist.all_reduce(ref)
        assert torch.equal(ref, sweep.tot), "exchanged totals differ from the all-reduced local totals"
        g = sweep.gathered.contiguous().view(world * n, words)
        bit0 = int(((g[:, 0] & 1) != 0).sum())
        assert bit0 == int(sweep.tot[0, 0]), "gathered bitmap and exchanged totals disagree"

    # ---- in-run spot check against the oracle (a few hundred objects of this rank's shard, rank 0)
    spot = None
    spot_bits = None
    if rank == 0 and args.spot_check > 0:
        from oracle import k8s
        orc = k8s.Client()
        for k, r, *rest in tm:
            orc.add_template(k, r)
        for c in cons:
            orc.add_constraint(c)
        for ns in nss:
            orc.add_namespace(ns)
        m = min(n, args.spot_check)
        sub = W.PyBlob([blob.get(i) for i in range(m)])
        got = drv.ReviewBlob(sub, ep, with_results=False)
        want = set()
        for i in range(m):
            for x in orc.review(k8s.Review(obj=json.loads(blob.get(i)), source="Original"), ep):
                if not x.get("autoreject"):
                    want.add((i, "%s/%s" % x["constraint"]))
        have = got.pairs()
        assert have == want, "spot check against the oracle failed: %d / %d pairs differ" % (len(have ^ want), len(want))
        spot = {"objects": m, "violating_pairs": len(want), "identical_to_oracle": True, "kernel": drv.last_kernel()}
        spot_bits = np.array(got.viol_bits[:m], copy=True)   # (a batch this small runs on the netlist interpreter)

    # ---- e2e: public API, raw JSON in pinned host memory in, bitmaps + totals out; a DIFFERENT page of objects every step
    e2e_steps = max(1, min(K, args.e2e_steps))
    e2e_warm = 2
    pages = []
    for k in range(e2e_warm + e2e_steps):
        pg = blob if k == 0 else W.synth_objects((world * (k + 1) + rank) * n, n, mode=mode, threads=host_threads)
        if k:
            drv.pin_blob(pg)
        pages.append(pg)
    resp = None
    for k in range(e2e_warm):   # (same call as the timed loop: the result buffers of two pages in flight come from the engine's page-locked pool)
        resp = drv.ReviewBlob(pages[k], ep, with_results=False, zero_copy=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    stats = []
    t0 = time.perf_counter()
    drv.prefetch_blob(pages[e2e_warm])                 # (inside the timed region: every page's copy is)
    for k in range(e2e_steps):
        if k + 1 < e2e_steps:
            drv.prefetch_blob(pages[e2e_warm + k + 1])  # the next page streams in while this one is extracted and evaluated
        resp = drv.ReviewBlob(pages[e2e_warm + k], ep, with_results=False, zero_copy=True)   # (bitmaps read in place, as a C / Go caller does)
        stats.append(resp.stats)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.barrier()
    e2e_s = float(te[0])
    clocks = sampler.stop() if rank == 0 else None
    first = drv.ReviewBlob(blob, ep, with_results=False)
    assert first.totals == totals_local[:len(first.totals)], "e2e path and resident path disagree"
    if spot_bits is not None and first.viol_bits is not None:
        # the same objects as rows of the full page: evaluated by the kernel generated for the constraint set (a large batch), while the
        # spot-check batch above ran on the interpreter and was compared with the oracle -- the rows must be identical
        assert np.array_equal(np.asarray(first.viol_bits[:len(spot_bits)]), spot_bits), "the page's rows differ from the spot-check batch (oracle-checked)"
        spot["page_rows_identical"] = True
        spot["page_kernel"] = drv.last_kernel()
    blob_bytes = pages[-1].total_bytes()
    e2e = {"value": world * n * C / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(stats[-1]["h2d_bytes"]) * world,
           "d2h_bytes_per_step": int(stats[-1]["d2h_bytes"] + 16 * C) * world, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s,
           "json_bytes_per_step": blob_bytes * world, "ingest": ingest_mode,
           "breakdown_ms": {k: round(sum(s[k] for s in stats) / len(stats), 3) for k in ("flatten_ms", "h2d_ms", "kernel_ms", "d2h_ms")},
           "breakdown_note": "h2d_ms = chunked copy of the JSON overlapped with the tokeniser; flatten_ms = the rest of the device ingest (count, scan, extract) + host glue",
           "pages": "every timed step reviews a page of objects it has not seen before (pinned host memory); page k+1 is prefetched (gk_blob_prefetch: "
                    "copy + tokenise on their own streams) while page k is extracted and evaluated -- all copies inside the timed region"}

    # the same call asked to also render every violation's {msg, details} (what Client.Review returns in the reference):
    # measured on a bounded sample, reported beside the decision-only figure
    msg_n = min(n, args.msg_sample)
    e2e_msgs = None
    if msg_n > 0 and rank == 0:
        sub = W.synth_objects(shard0, msg_n, mode=mode, threads=host_threads)
        r2 = drv.ReviewBlob(sub, ep, flags=D.F_MATERIALIZE, with_results=False)   # results stay in the engine's buffers: not converted to Python
        dt = sum(r2.stats[k] for k in ("flatten_ms", "h2d_ms", "kernel_ms", "d2h_ms", "materialize_ms")) / 1e3
        e2e_msgs = {"value": msg_n * C / dt, "unit": UNIT, "objects": msg_n, "results_rendered": r2.stats["n_violations"],
                    "materialize_ms": round(r2.stats["materialize_ms"], 1), "flatten_ms": round(r2.stats["flatten_ms"], 1)}
        del r2
    # the audit sweep proper: one page through gk_batch_upload_blob + gk_audit_add_batch -- totals per constraint and the K smallest
    # violations with their messages (pkg/audit/manager.go:886-1041).  Pairs with one result are counted from the bitmaps (the
    # ambiguity netlist runs on the device); the host evaluates what can still enter a list and the pairs that may have several.
    e2e_audit = None
    if args.config == 2 and not args.no_audit and rank == 0:   # (host-side aggregation: one rank's page is the measurement)
        ta = time.perf_counter()
        audit_rb = drv.upload_blob(pages[1])
        audit_run = D.AuditRun(drv, violations_limit=20)
        audit_run.add_batch(audit_rb, ep)
        rep = audit_run.report()
        dta = time.perf_counter() - ta
        e2e_audit = {"value": n * C / dta, "unit": UNIT, "objects": n, "ms": round(1e3 * dta, 1), "results": rep["results"],
                     "pairs_counted_on_device": rep["pairsCounted"], "pairs_evaluated_on_host": rep["pairsEvaluated"], "violations_limit": 20}
        del audit_rb, audit_run
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9
    # gk_spec_kernel: CUDA C++ generated from the constraint set's netlist, compiled by NVRTC at the first large batch (outside the
    # timed region); the netlist interpreter gk_eval_kernel is launched behind it for the tiles it hands over (none on this workload)
    kernel_name = drv.last_kernel()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and args.config == 2:
        try:
            traffic = json.load(open(tp)).get(drv.last_kernel(), {}).get("dram_bytes_per_launch")   # (one ncu --set full capture per kernel)
        except Exception:
            traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W_,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int (u32 ids / u8 bytes / i64)",
        "data": "synthetic",
        "config": {"workload": label, "objects_per_gpu": n, "constraints": C, "evals_per_step": world * n * C,
                   "l2": ("inputs larger than L2: %.0f MB of columns per GPU" % (alg_in / 1e6)) if flush is None else "explicit 256 MB L2 flush between steps",
                   "parallelism": (f"objects sharded over {world} GPU(s); exchange per step: " +
                                   ("fused into the kernel -- bitmap words and totals stored straight into every peer's buffer over NVLink, one device-side barrier"
                                    if sweep.p2p is not None else "one NCCL all-gather (bitmap shard + totals)")) if world > 1 else "single GPU",
                   "violating_pairs_per_step": int(sum(totals_host)), "violating_density": round(sum(totals_host) / max(1, world * n * C), 4),
                   "synth_s": round(gen_s, 2), "ingest_ms_once": round(rb.stats["flatten_ms"] + rb.stats["h2d_ms"], 1), "spot_check": spot},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "kernel": kernel_name, "kernel_ms": kern_ms, "alg_bytes_per_launch": alg_bytes, "peak_source": peak_src},
        "e2e": dict(e2e, with_messages=e2e_msgs, audit=e2e_audit), "gpu_launches": int(launches), "clocks": clocks,
    }
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(args.config, args.cpu_sample)
    if os.environ.get("GK_BENCH_NOTE"):
        line["note"] = os.environ["GK_BENCH_NOTE"]
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------------ GPU arm: admission replay (configs[2])
def run_admission(args):
    """64-request UPDATE micro-batches against 200 cloned PSP constraints (pkg/webhook/policy_benchmark_test.go:191-249): latency per
    micro-batch through gk_review_batch with messages rendered, p50 / p99 (metrics.py percentiles)."""
    import torch
    from gatekeeper_b200 import driver as D
    from gatekeeper_b200 import workloads as W
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    tm, cons, pods = W.config3(200)
    drv = D.Driver(device=0)
    for k, r in tm:
        drv.add_template(k, r)
    for c in cons:
        drv.AddConstraint(c)
    C = len(drv.constraints())
    import copy
    import random
    rnd = random.Random(3)
    batch = 64

    def make_batch(seed):
        revs = []
        for i in range(batch):
            p = copy.deepcopy(pods[(seed + i) % len(pods)])
            p["metadata"]["name"] = "pod-%d-%d" % (seed, i)
            old = copy.deepcopy(p)
            old["metadata"].setdefault("labels", {})["rev"] = str(rnd.randrange(1000))
            revs.append(D.Review(object=p, old_object=old, operation="UPDATE", source="Original"))
        return revs
    batches = [make_batch(s) for s in range(32)]
    for b in batches[:4]:
        drv.ReviewBatch(b, D.WEBHOOK_EP)
    # the timed call is gk_review_batch itself on pre-marshalled requests (what the Go shim's cgo call costs): building the
    # ctypes structs and converting 12 800 results per batch into Python objects is the mirror's overhead, not the engine's
    marshalled = [drv._marshal(b) for b in batches]
    sampler = ClockSampler(0)
    sampler.start()
    lat, kern = [], []
    K = args.steps
    t_all = time.perf_counter()
    for k in range(K):
        arr, nb, _keep = marshalled[k % len(marshalled)]
        t0 = time.perf_counter()
        resp = drv.review_marshalled(arr, nb, D.WEBHOOK_EP, D.F_MATERIALIZE)
        lat.append((time.perf_counter() - t0) * 1e3)
        kern.append(resp.stats["kernel_ms"])
    total_s = time.perf_counter() - t_all
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [resp.totals, resp.err_totals], resp.viol_bits, resp.err_bits)
    def pct(v, p):   # linear interpolation at rank p/100 * (n-1), as gatekeeper_b200/metrics.py (pkg/gator/bench/metrics.go:37-59)
        v = sorted(v)
        r = (p / 100.0) * (len(v) - 1)
        lo = int(r)
        hi = min(lo + 1, len(v) - 1)
        return v[lo] + (v[hi] - v[lo]) * (r - lo)
    p50, p99 = pct(lat, 50), pct(lat, 99)
    line = {"metric": "admission_review_latency_ms_per_64_request_batch", "value": p99, "unit": "ms (p99)", "n_gpus": 1, "steps": K, "warmup": 4,
            "ms_per_step": 1e3 * total_s / K, "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "int", "data": "synthetic",
            "config": {"workload": "admission Review replay: 64-request UPDATE micro-batches, 200 cloned PSP constraints, messages rendered (BASELINE.json configs[2])",
                       "constraints": C, "batch": batch},
            "latency_ms": {"p50": p50, "p99": p99, "mean": sum(lat) / len(lat), "per_request_p50": p50 / batch, "per_request_p99": p99 / batch},
            "kernel_ms_mean": sum(kern) / len(kern), "evals_per_s": batch * C * K / total_s,
            "e2e": {"value": batch * C * K / total_s, "unit": UNIT, "h2d_bytes_per_step": int(resp.stats["h2d_bytes"]), "d2h_bytes_per_step": int(resp.stats["d2h_bytes"])},
            "gpu_launches": K, "clocks": clocks}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 50 for --config 3, 20 otherwise)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json workload: 2 = configs[1] (default), 3 = admission replay, 4 = PSP x mixed GVK, 5 = wildcards")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: --objects per GPU; strong: --objects in total")
    ap.add_argument("--objects", type=int, default=0, help="objects per GPU (weak) / in total (strong); 0 = the config's size")
    ap.add_argument("--e2e-steps", type=int, default=8, help="pages of the pipelined end-to-end sweep (each is a fresh 1M-object page in pinned host memory)")
    ap.add_argument("--cpu-sample", type=int, default=30_000, help="objects reviewed by the C++ CPU restatement leg (all host threads)")
    ap.add_argument("--no-audit", action="store_true", help="skip the audit-aggregation measurement (e2e.audit)")
    ap.add_argument("--msg-sample", type=int, default=50_000, help="objects of the sample whose messages are all rendered (e2e.with_messages)")
    ap.add_argument("--spot-check", type=int, default=300, help="objects of the shard checked against the Python oracle inside the run")
    ap.add_argument("--ref-objects-per-step", type=int, default=40_000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 50 if args.config == 3 and args.impl == "ours" else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        sys.exit(run_reference(args))
    if args.config == 3:
        sys.exit(run_admission(args))
    # Single-GPU runs: if an in-run check fails while the kernel generated for the constraint set is in use, the run is repeated once on
    # the netlist interpreter alone (GK_SPEC=0) and the line says so -- a measured interpreter figure instead of no figure.  (With
    # several ranks a failure is fatal: the ranks could not agree on the retry without a collective.)
    failure = None
    try:
        rc = run_ours(args)
    except AssertionError as e:
        if env_int("WORLD_SIZE", 1) > 1 or os.environ.get("GK_SPEC") == "0":
            raise
        failure = str(e)
    if failure is None:
        sys.exit(rc)
    sys.stderr.write("bench.py: in-run check failed with the generated kernel enabled (%s); repeating with GK_SPEC=0\n" % failure)
    os.environ["GK_SPEC"] = "0"
    os.environ["GK_BENCH_NOTE"] = "first attempt failed an in-run check with the generated kernel enabled (%s); this line was measured with GK_SPEC=0" % failure
    sys.exit(run_ours(args))


if __name__ == "__main__":
    main()
