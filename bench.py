#!/usr/bin/env python
"""bench.py -- EMAT log-lik evals/s + SPR candidates scored/s + MCMC steps/s on B200 (BASELINE.json metric).

Workload at N = 1: a forest of `--chains` independent synthetic 100k-tip x 29,903-site EMATs (BASELINE.json configs[3] shape,
the shape the target is quoted on; 16 chains so that the forest exceeds the 126 MB L2 and the timed kernels stream from HBM).
One "step" = `--evals-per-step` log-G evaluations (calc_lambda_i + calc_log_root_prior + calc_log_G_below_root, SURVEY.md
section 8d) of every EMAT of the forest; K steps are enqueued back to back between two CUDA events on the launching stream.

  value               = log-lik evals/s, inputs resident in HBM (whole job, all ranks)
  roofline            = algorithmic bytes of one evaluation / its CUDA-event duration vs the measured HBM peak
                        (+ achieved_dram_frac: the DRAM bytes ncu measured for the same launch, same duration)
  spr_candidates_per_s, roofline_spr   = full SPR regraft studies (the metric's second figure), timed the same way
  loglik_general_schedule              = the per-event schedule (the one site-rate heterogeneity needs)
  configs             = the same two figures for BASELINE.json configs[1], [2], [4] (parity-test shapes; secondary)
  model_change_cycle  = evals/s when every evaluation follows a model change (set_evo + eval + read-back)
  partitioned         = ONE 100k-tip tree cut into parts spread over the ranks: per cycle new mu -> every part re-evaluated ->
                        packed tallies -> ONE NCCL all-reduce (strong scaling; SURVEY.md section 8e)
  e2e                 = the log-lik metric through the C ABI with HOST buffers (upload + eval + download per step)
  mcmc                = MCMC steps/s of the reference's own CLI with the hot path substituted at link time
                        (delphy_b200/adapter/_build/delphy_b200_cli); `--impl reference` runs the stock build of the same sources
  cpu_baseline        = the reference's own CPU code (oracle/_ref, compiled from /root/reference) on the box's host cores

`--impl reference` times the reference's CPU implementation (oracle/_ref) on the same workload and prints the same keys; it
loads no product code (inputs come from libdphy_synth.so).

`--dump-outputs DIR` writes, after the timed steps, what the timed evaluation and SPR batch computed in their last step (log G
terms and lambda_i of every chain, the batch's study summaries and regions; float64, a fixed seeded sample of any array larger
than DUMP_MAX_ELEMS) as DIR/<name>.npy.  The inputs are seeded, so two builds run with the same arguments can be compared
output for output.

Multi-GPU (torchrun): the headline shards independent EMATs over ranks with no data-path collective (weak scaling); the
`partitioned` section is the one place with a real exchange.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "EMAT log-lik evals/s (+ spr_candidates_per_s, mcmc steps/s)"
UNIT = "evals/s"
SHAPES = {1: "200-tip x 29,903-site", 2: "1,600-tip x 18,959-site (nu_l on, missations)", 3: "10k-tip x 29,903-site",
          4: "100k-tip x 29,903-site", 5: "50k-tip x 197,000-site (heavy missing, 2 partitions)"}
SECONDARY = {2: 256, 3: 64, 5: 8}        # config -> chains per GPU (forest > L2 where the shape allows it)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, help="synthetic shape: 1..5 == BASELINE.json configs[0..4]")
    ap.add_argument("--chains", type=int, default=16, help="independent EMATs per GPU (forest must exceed L2)")
    ap.add_argument("--evals-per-step", type=int, default=32, help="log-G evaluations of the whole forest per step (timed region >= 50 ms)")
    ap.add_argument("--spr-studies", type=int, default=128, help="full SPR studies per batch (0 disables)")
    ap.add_argument("--spr-batches-per-step", type=int, default=4)
    ap.add_argument("--e2e-chains", type=int, default=16)
    ap.add_argument("--e2e-threads", type=int, default=2, help="host threads (one context each) that take the e2e steps in turn")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="CPU baseline budget per figure")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs 2/3/5 figures")
    ap.add_argument("--no-partitioned", action="store_true")
    ap.add_argument("--no-mcmc", action="store_true")
    ap.add_argument("--parts-per-gpu", type=int, default=2)
    ap.add_argument("--mcmc-tips", type=int, default=10000, help="tips of the second MCMC alignment (config 3 shape)")
    ap.add_argument("--mcmc-steps", type=int, default=200000)
    ap.add_argument("--mcmc-threads-per-gpu", type=int, default=1)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed log-G and SPR steps computed in their last step to DIR/<name>.npy (float64, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


DUMP_MAX_ELEMS = 1 << 19      # per array: a fixed, seeded sample beyond this keeps a dump of ~30 MB at the default workload (<= 64 MB)


def dump_sample(a):
    """`a` as float64, or a fixed seeded sample of DUMP_MAX_ELEMS of its elements (in order) when it is larger."""
    a = np.asarray(a, np.float64).ravel()
    if a.size <= DUMP_MAX_ELEMS:
        return a
    idx = np.sort(np.random.default_rng(20251017).choice(a.size, DUMP_MAX_ELEMS, replace=False))
    return a[idx]


def write_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= 64 << 20, f"output dump of {total} bytes exceeds 64 MB"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def config_block(args):
    """Identical for both arms: names the workload, nothing implementation specific."""
    return {"workload": f"synthetic {SHAPES.get(args.config, 'small')} EMAT x {args.chains} independent chains per GPU",
            "chains_per_gpu": args.chains, "evals_per_step": args.evals_per_step,
            "step": f"{args.evals_per_step} log-G evaluations (lambda_i + root prior + log G below root) of every EMAT of the forest",
            "spr_studies_per_batch": args.spr_studies, "l2": "inputs larger than L2 (forest > 126 MB)",
            "parallelism": f"chains x{args.gpus}"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel, cfg, chains):
    """DRAM bytes (read + write) per launch of `kernel` from the committed ncu --set full capture of this workload
    (profiles/traffic.json), or None when no capture matches."""
    try:
        best = None
        for row in json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))):
            if row["kernel"] == kernel and row["config"] == cfg and row["chains"] == chains:
                best = row["dram_bytes_per_launch"]
        return best
    except Exception:
        return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---- the reference's own CPU code (oracle/_ref), or the oracle port when it is absent ------------------------------------------
def _oracle_modules():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    from helpers import to_oracle
    return ol, to_oracle


def cpu_log_G(emat, sites, budget_s, threads):
    """calc_lambda_i + calc_log_root_prior + calc_log_G_below_root on `threads` replicas of one tree, one per thread."""
    import ctypes as C
    ol, to_oracle = _oracle_modules()
    e, s = to_oracle(emat, sites)
    es, ss = e.as_struct(), s.as_struct()
    if not ol.ref_available():
        o = ol.Oracle("oracle")
        cq = o.cum_Q_l(s)
        t0 = time.perf_counter(); n = 0
        while time.perf_counter() - t0 < budget_s or n < 2:
            lam = o.lambda_i(e, s, cq); o.log_root_prior(e, s); o.log_G_below_root(e, s, lam); n += 1
        t = time.perf_counter() - t0
        return dict(value=n / t, unit=UNIT, cores=1, kind="port", seconds=t, sample=f"{n} evals of one {emat.num_nodes}-node EMAT, 1 thread, {t:.1f} s")
    lib = ol.ref()
    lg = C.c_double()
    t1 = lib.ref_bench_log_G(C.byref(es), C.byref(ss), 2, threads, C.byref(lg))      # calibration
    reps = max(2, int(budget_s / max(t1 / 2, 1e-6)))
    t = lib.ref_bench_log_G(C.byref(es), C.byref(ss), reps, threads, C.byref(lg))
    return dict(value=threads * reps / t, unit=UNIT, cores=threads, kind="reference", log_G=lg.value, seconds=t,
                sample=f"{reps} evals/thread x {threads} threads of one {emat.num_nodes}-node EMAT "
                       f"(calc_lambda_i + calc_log_root_prior + calc_log_G_below_root), {t:.1f} s")


def cpu_log_G_partitioned(db, emat, sites, budget_s, threads):
    """The reference's own multithreaded scheme (core/run.cpp:682-693): the tree cut into `threads` parts, one per worker thread."""
    import ctypes as C
    ol, to_oracle = _oracle_modules()
    if not ol.ref_available():
        return None
    lib = ol.ref()
    part = db.Partition(emat, sites, threads, seed=20251017, host_only=True)
    pes = [to_oracle(p, sites)[0] for p in part.parts]
    _, s = to_oracle(emat, sites)
    structs = [pe.as_struct() for pe in pes]
    arr = (C.POINTER(type(structs[0])) * len(structs))(*[C.pointer(x) for x in structs])
    ss = s.as_struct()
    lib.ref_bench_log_G_parts.restype = C.c_double
    lg = C.c_double()
    t1 = lib.ref_bench_log_G_parts(arr, len(structs), C.byref(ss), 2, C.byref(lg))
    reps = max(2, int(budget_s / max(t1 / 2, 1e-6)))
    t = lib.ref_bench_log_G_parts(arr, len(structs), C.byref(ss), reps, C.byref(lg))
    n_parts = len(structs)
    part.close()
    return dict(value=reps / t, unit="whole-tree evals/s", cores=n_parts, kind="reference", log_G=lg.value, seconds=t,
                sample=f"one {emat.num_nodes}-node EMAT cut into {n_parts} parts (generate_random_partition_stencil), one part per thread, "
                       f"{reps} evaluations of every part, {t:.1f} s")


def cpu_spr(emat, sites, xs, budget_s, threads, t_max_tip):
    import ctypes as C
    ol, to_oracle = _oracle_modules()
    if not ol.ref_available() or xs is None or len(xs) == 0:
        return None
    lib = ol.ref()
    e, s = to_oracle(emat, sites)
    es, ss = e.as_struct(), s.as_struct()
    xs = np.ascontiguousarray(xs, np.int32)
    nreg = C.c_int64()
    n0 = min(len(xs), threads)
    t0 = lib.ref_bench_spr(C.byref(es), C.byref(ss), xs.ctypes.data_as(ol.i32p), n0, threads, 0.8, t_max_tip, C.byref(nreg))
    n_x = int(min(len(xs), max(threads, budget_s / max(t0, 1e-9) * n0)))
    t = lib.ref_bench_spr(C.byref(es), C.byref(ss), xs.ctypes.data_as(ol.i32p), n_x, threads, 0.8, t_max_tip, C.byref(nreg))
    return dict(value=nreg.value / t, unit="candidates/s", cores=threads, kind="reference", seconds=t,
                sample=f"{n_x} full SPR studies (reconstruct_missing_sites_at + seed_fill_from + Spr_study), {nreg.value} regions, {t:.1f} s")


def cpu_api_tree_read(buf):
    """api_tree_and_tree_info_to_phylo_tree (core/api.cpp:127-186, fix_up_missations included) on one buffer, one thread: the compiled
    reference when it travelled, else the oracle's restatement."""
    ol, _ = _oracle_modules()
    kind = "reference" if ol.ref_available() else "port"
    t0 = time.perf_counter()
    ol.api_tree_read(buf, "ref" if kind == "reference" else "oracle")
    return {"load_ms_per_tree": (time.perf_counter() - t0) * 1e3, "kind": kind, "cores": 1,
            "sample": "one buffer -> Phylo_tree (-> flat arrays), single thread"}


def pick_spr_nodes(emat, n, seed=1234):
    rng = np.random.default_rng(seed)
    cand = np.array([v for v in rng.permutation(emat.num_nodes)[: 8 * n + 8] if v != emat.root and emat.parent[v] != emat.root], np.int32)
    return cand[:n]


# ---- MCMC through the reference's own CLI (stock build or link-time drop-in) ------------------------------------------------------
def mcmc_figures(db, args, which, n_gpus):
    """steps/s of the reference's CLI on two synthetic alignments: configs[0] (200 tips, 1 M steps -- the reference's own
    CPU-runnable case) and a config-3-shaped one (`--mcmc-tips` tips).  `which`: "dropin" | "stock"."""
    from delphy_b200 import mcmc
    from delphy_b200.maple import write_maple
    binary = mcmc.DROPIN_CLI if which == "dropin" else mcmc.STOCK_CLI
    if not os.path.exists(binary):
        return {"unavailable": f"{os.path.relpath(binary, ROOT)} not built (needs the reference checkout at build time)"}
    tmp = os.path.join("/tmp", f"dphy_bench_{os.getpid()}")
    os.makedirs(tmp, exist_ok=True)
    threads = max(1, args.mcmc_threads_per_gpu * n_gpus)
    out = {"binary": os.path.relpath(binary, ROOT), "host_threads": threads, "n_gpus": n_gpus if which == "dropin" else 0}
    cases = [("cfg1_200_tips", db.synth_params(1), 1000000), (f"cfg3_{args.mcmc_tips}_tips", db.synth_params(3, num_tips=args.mcmc_tips), args.mcmc_steps)]
    for name, params, steps in cases:
        emat, sites, info = db.synth_generate(params)
        path = os.path.join(tmp, name + ".maple")
        write_maple(emat, sites, path, info["t_max_tip"])
        r = mcmc.run_cli(binary, path, steps, threads=threads, seed=20251017, log_every=max(1, steps // 10),
                         env={"DPHY_DEVICES": n_gpus, "DPHY_DROPIN_STATS": 1}, timeout=900)
        last = r["samples"][-1] if r["samples"] else {}
        out[name] = {"steps_per_s": r["steps_per_s"], "steps": steps, "mcmc_seconds": r["mcmc_s"], "init_seconds": r["init_s"],
                     "returncode": r["returncode"], "final": {k: last.get(k) for k in ("log_G", "num_muts", "t_MRCA", "mu", "n0")},
                     "tips": (emat.num_nodes + 1) // 2}
        if r["returncode"] != 0:
            out[name]["stderr_tail"] = r["stderr_tail"][-4:]
        last_case = (name, path, steps)
    if n_gpus > 1:
        # weak scaling (BASELINE.json configs[4]: independent chains, replicas only): one CLI process per GPU, one worker thread each,
        # different seeds, all at once; steps/s summed.  The figures above are the strong-scaling ones (ONE chain, its tree cut into
        # n_gpus parts, a worker thread and a GPU per part).
        name, path, steps = last_case
        res = [None] * n_gpus

        def one(i):
            env = {"DPHY_DEVICES": 1, "DPHY_DROPIN_STATS": 0}
            if which == "dropin":
                env["CUDA_VISIBLE_DEVICES"] = i
            res[i] = mcmc.run_cli(binary, path, steps, threads=1, seed=20251017 + 1 + i, log_every=max(1, steps // 10), env=env, timeout=900)
        def guarded(i):
            try:
                one(i)
            except Exception as ex:          # a failed side figure must not cost the whole line
                res[i] = {"returncode": -1, "steps_per_s": None, "error": repr(ex)[:200]}
        ths = [threading.Thread(target=guarded, args=(i,)) for i in range(n_gpus)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        ok = all(r is not None and r["returncode"] == 0 and r["steps_per_s"] for r in res)
        out[name + "_independent_chains"] = {"chains": n_gpus, "steps_per_s": sum(r["steps_per_s"] for r in res) if ok else None,
                                             "per_chain_steps_per_s": [r["steps_per_s"] if r else None for r in res], "steps_per_chain": steps,
                                             "returncodes": [r["returncode"] if r else None for r in res]}
    return out


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner at communicator
    creation), so file descriptor 1 is pointed at stderr for the whole run and the line goes to a private duplicate of the
    original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def reference_arm(db, args, rank):
    """The reference's own CPU implementation of the path on all host threads; rank 0 only.  Loads libdphy_synth.so (inputs)
    and oracle/_ref -- no product code."""
    if rank != 0:
        return 0
    threads = host_cores()
    emat, sites, info = db.synth_generate(db.synth_params(args.config))
    spr_xs = pick_spr_nodes(emat, max(args.spr_studies, threads)) if args.spr_studies > 0 else None
    # a step = a bounded sample of the workload: as many evaluations as fit the per-step budget, measured, not assumed
    per_step = max(0.25, min(args.cpu_seconds, 100.0 / max(1, args.steps + args.warmup)))
    vals, secs, last = [], [], None
    for i in range(args.warmup + args.steps):
        r = cpu_log_G(emat, sites, per_step, threads)
        if i >= args.warmup:
            vals.append(r["value"]); secs.append(r["seconds"])
        last = r
    v = float(np.mean(vals))
    spr = cpu_spr(emat, sites, spr_xs, args.cpu_seconds, threads, info["t_max_tip"]) if spr_xs is not None else None
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_block(args),
            "spr_candidates_per_s": spr["value"] if spr else None,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": last["kind"], "sample": last["sample"], "spr": spr},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.no_partitioned:
        line["partitioned"] = cpu_log_G_partitioned(db, emat, sites, args.cpu_seconds, threads)
    if not args.no_secondary:
        # the wire format on the reference's side: its own writer, then its own reader (api_tree_and_tree_info_to_phylo_tree incl.
        # fix_up_missations), one thread -- what `wire_format.load_ms_per_tree` of our arm replaces
        ol, to_oracle = _oracle_modules()
        if ol.ref_available():
            e, s = to_oracle(emat, sites)
            t0 = time.perf_counter()
            buf = ol.api_tree_write(e, s.ref, "ref", s)
            wr_ms = (time.perf_counter() - t0) * 1e3
            wf = cpu_api_tree_read(buf)
            wf.update({"format": "delphy.api.Tree (FlatBuffers; core/api.fbs:13-49)", "buffer_bytes_per_tree": len(buf), "write_ms_per_tree": wr_ms})
            line["wire_format"] = wf
    if not args.no_mcmc:
        line["mcmc"] = mcmc_figures(db, args, "stock", args.gpus)
    emit_line(line)
    return 0


def main():
    args = parse_args()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import delphy_b200 as db

    if args.impl == "reference":
        return reference_arm(db, args, rank)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = db.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    peak, peak_src = measured_peak()
    R = max(1, args.evals_per_step)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def max_over_ranks(vals):
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def make_forest(cfg, chains):
        emats, tables, infos = [], [], []
        base_seed = 20251017 + 1000 * rank + 100000 * cfg
        for c in range(chains):
            e, s, info = db.synth_generate(db.synth_params(cfg, seed=base_seed + c))
            emats.append(e); infos.append(info)
            tables.append(db.DeviceSites(ctx, s))
        return emats, tables, infos, db.Forest(ctx, emats, tables, sites_index=np.arange(chains))

    def time_evals(forest, steps, reps):
        """ms per step of `reps` evaluations of the forest each, K steps back to back between two events on the launching stream."""
        a, b = ev(), ev()
        barrier()
        a.record(stream)
        h0 = time.perf_counter()
        for _ in range(steps * reps):
            forest.eval_log_G()
        host_ms = (time.perf_counter() - h0) * 1e3 / steps
        b.record(stream)
        barrier()
        return a.elapsed_time(b) / steps, host_ms

    # ---- headline workload --------------------------------------------------------------------------------------------------------------
    emats, tables, infos, forest = make_forest(args.config, args.chains)
    host_sites = [t.host for t in tables]
    alg_bytes = forest.log_G_algorithmic_bytes
    spr_reqs = None
    spr_xs = pick_spr_nodes(emats[0], args.spr_studies) if args.spr_studies > 0 else np.zeros(0, np.int32)
    if args.spr_studies > 0:
        forest.eval_log_G()
        spr_reqs = db.spr_requests_for_attached(emats[0], 0, spr_xs, forest.lambda_i(0), infos[0]["t_max_tip"])

    def spr_batch(keep=False):
        b = forest.spr_study_batch(spr_reqs)
        if keep:
            return b
        b.close()                    # stream-ordered free: the memory is reused by the next batch

    for _ in range(max(args.warmup, 3)):
        for _ in range(R):
            forest.eval_log_G()
        if spr_reqs is not None:
            spr_batch()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launches
    logg_ms, host_enqueue_ms = time_evals(forest, args.steps, R)
    launches = ctx.launches - launches0
    rp, br, lg = forest.log_G()      # checksum of the timed work: log G of every chain
    dumped = {}
    if args.dump_outputs:
        # what a caller of the timed evaluation reads back: per chain the three log-G terms and lambda_i of every node
        dumped.update(log_root_prior=rp, log_G_below_root=br, log_G=lg,
                      lambda_i=dump_sample(np.concatenate([forest.lambda_i(k) for k in range(args.chains)])))

    spr_ms, spr_regions, spr_launches = None, 0, 0
    if spr_reqs is not None:
        SB = max(1, args.spr_batches_per_step)
        l0 = ctx.launches
        a, b = ev(), ev()
        barrier()
        a.record(stream)
        n_batches = args.steps * SB
        for i in range(n_batches):
            last = spr_batch(keep=bool(args.dump_outputs) and i == n_batches - 1)      # --dump-outputs reads the last timed batch back
        ctx.join_side_streams()       # the last batches' normalisation passes run on the library's tail stream: inside the timed region
        b.record(stream)
        barrier()
        spr_ms = a.elapsed_time(b) / (args.steps * SB)        # per batch
        spr_launches = ctx.launches - l0
        if args.dump_outputs:
            sm = last.summaries()
            for k in ("mu", "log_Wmax", "sum_W_over_Wmax", "num_regions"):
                dumped["spr_summary_" + k] = np.array([getattr(s, k) for s in sm], np.float64)
            regs = last.regions()
            for k in ("branch", "mut_idx", "min_muts", "t_min", "t_max", "log_W_over_Wmax", "W_over_Wmax"):
                dumped["spr_region_" + k] = dump_sample(regs[k])
            del regs
            last.close()
        bt = forest.spr_study_batch(spr_reqs)
        spr_regions = bt.total_regions()
        bt.close()

    # the general schedule (every mutation / missation / from-state list re-read per evaluation)
    ctx.set_log_G_path("general")
    for _ in range(3):
        forest.eval_log_G()
    gen_ms, _ = time_evals(forest, args.steps, R)
    _, _, lg_gen = forest.log_G()
    if args.dump_outputs:
        dumped["log_G_general_schedule"] = lg_gen
    ctx.set_log_G_path("auto")
    assert np.allclose(lg_gen, lg, rtol=1e-11), "folded and general log-G schedules disagree"
    clocks = sampler.stop() if rank == 0 else None
    logg_ms_max, spr_ms_max, gen_ms_max = max_over_ranks([logg_ms, spr_ms or 0.0, gen_ms])

    # ---- the reference's global-move cycle: new mu on every chain's site table, re-evaluate every chain, read log G back --------
    mc_steps = max(3, min(args.steps, 20))
    mus = [t.host.mu.copy() for t in tables]

    def model_change_cycle(i):
        # Run::push_global_params_to_subruns (core/run.cpp:267-275): the new model goes to every chain's table -- one launch for all
        db.sites_set_evo_many(ctx, tables, mus=[mus[k] * (1.0 + 1e-3 * ((i % 7) + 1)) for k in range(len(tables))])
        forest.eval_log_G()
        return forest.log_G()
    for i in range(2):
        model_change_cycle(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(mc_steps):
        model_change_cycle(i)
    torch.cuda.synchronize()
    mc_s = time.perf_counter() - t0
    for k, t in enumerate(tables):
        t.set_evo(mu=mus[k])
    forest.eval_log_G()
    assert np.allclose(forest.log_G()[2], lg, rtol=1e-12), "restoring the model does not restore log G"
    (mc_s,) = max_over_ranks([mc_s])

    # ---- edit + eval (SURVEY.md section 8f row 1): per step one branch reform per chain (the mutation times of one branch redrawn,
    # core/subrun.cpp:316-319) shipped as rows -> dphy_forest_apply_rows -> evaluation -> log G read back.  Only the rows cross PCIe.
    edit_rng = np.random.default_rng(99 + rank)
    edit_steps = max(3, min(args.steps, 10))
    edit_nodes = []
    for e in emats:
        has = np.nonzero((np.diff(e.mut_off) > 0) & (e.parent >= 0))[0]
        edit_nodes.append(has[edit_rng.integers(len(has), size=edit_steps + 2)])

    def edit_step(i):
        rows, nbytes = [], 0
        for k, e in enumerate(emats):
            v = int(edit_nodes[k][i]); m0, m1 = int(e.mut_off[v]), int(e.mut_off[v + 1])
            lo, hi = e.t[e.parent[v]], e.t[v]
            e.mut_t[m0:m1] = np.sort(lo + (hi - lo) * edit_rng.random(m1 - m0))
            r = db.node_row(k, e, v)
            rows.append(r)
            nbytes += C_sizeof_row + 14 * r.n_muts + 8 * r.n_miss + 5 * r.n_fs
        forest.apply_rows(rows)
        forest.eval_log_G()
        return forest.log_G(), nbytes
    import ctypes as _C
    C_sizeof_row = _C.sizeof(db.NodeRow)
    for i in range(2):
        edit_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(edit_steps):
        edit_out, edit_bytes = edit_step(2 + i)
    torch.cuda.synchronize()
    (edit_s,) = max_over_ranks([time.perf_counter() - t0])
    fresh = db.Forest(ctx, emats, tables, sites_index=np.arange(args.chains))     # the edited trees, uploaded afresh
    fresh.eval_log_G()
    assert np.allclose(fresh.log_G()[2], edit_out[2], rtol=1e-12), "edited forest differs from a fresh upload"
    fresh.close()
    lg_timed, lg = lg, edit_out[2]          # the e2e leg below uploads the edited trees

    # ---- e2e: host buffers -> C ABI -> host scalars, copies inside the timed region ------------------------------
    n_e2e = min(args.e2e_chains, args.chains)
    e2e_emats = [e.pinned(ctx) for e in emats[:n_e2e]]        # page-locked caller arrays (dphy_host_alloc): DMA'd from where they lie
    e2e_steps = max(3, min(args.steps, 10))
    h2d = sum(getattr(e, k).nbytes for e in e2e_emats for k in db.HostEmat.FIELDS_I32 + db.HostEmat.FIELDS_U8 + db.HostEmat.FIELDS_F64)
    d2h = n_e2e * 3 * 8

    # `--e2e-threads` host threads, each with its own context (stream, arena, pinned slab -- the per-thread handles the reference's
    # threading model asks for, SURVEY.md section 8b "Threading"), take the steps in turn: while one thread's forest is being
    # flattened / evaluated / read back, the other thread's arrays are crossing PCIe.  Every step still uploads all its inputs.
    n_thr = max(1, args.e2e_threads)
    e2e_ctxs = [ctx] + [db.Context(local_rank) for _ in range(n_thr - 1)]
    e2e_tables = [tables[:n_e2e]] + [[db.DeviceSites(c, host_sites[k]) for k in range(n_e2e)] for c in e2e_ctxs[1:]]

    def e2e_step(w=0):
        fo = db.Forest(e2e_ctxs[w], e2e_emats, e2e_tables[w], sites_index=np.arange(n_e2e))
        fo.eval_log_G()
        out = fo.log_G()
        fo.close()
        return out

    def e2e_run(total_steps):
        """total_steps steps shared by the worker threads (a common counter); returns the last result of every thread"""
        lock, nxt, outs = threading.Lock(), [0], [None] * n_thr

        def worker(w):
            torch.cuda.set_device(local_rank)
            while True:
                with lock:
                    if nxt[0] >= total_steps:
                        return
                    nxt[0] += 1
                outs[w] = e2e_step(w)
        ths = [threading.Thread(target=worker, args=(w,)) for w in range(1, n_thr)]
        for t in ths:
            t.start()
        worker(0)
        for t in ths:
            t.join()
        for c in e2e_ctxs:
            c.synchronize()
        return [o for o in outs if o is not None]
    e2e_run(2 * n_thr)
    barrier()
    t0 = time.perf_counter()
    e2e_outs = e2e_run(e2e_steps)
    torch.cuda.synchronize()
    (e2e_s,) = max_over_ranks([time.perf_counter() - t0])
    for e2e_out in e2e_outs:
        assert np.allclose(e2e_out[2], lg[:n_e2e], rtol=1e-12)
    for c, tb in zip(e2e_ctxs[1:], e2e_tables[1:]):
        for t in tb:
            t.close()
        c.close()
    del e2e_emats
    # ---- the reference's wire format (delphy.api.Tree, core/api.fbs) straight to the device and back --------------------------------------------
    wire = None
    wire_buf0 = None
    if not args.no_secondary:
        n_w = min(4, args.chains)
        forest.write_api_tree(0)                                               # (warm-up: the context's pinned slab grows once)
        t0 = time.perf_counter()
        bufs = [forest.write_api_tree(k) for k in range(n_w)]                  # phylo_tree_to_api_tree of the resident trees
        wr_ms = (time.perf_counter() - t0) * 1e3 / n_w
        wire_buf0 = bufs[0]
        db.Forest.from_api_trees(ctx, bufs, tables[:n_w], sites_index=np.arange(n_w)).close()
        reps_w = 3
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps_w):
            fw = db.Forest.from_api_trees(ctx, bufs, tables[:n_w], sites_index=np.arange(n_w))
            lgw = fw.log_G()[2]
            fw.close()
        torch.cuda.synchronize()
        (ld_s,) = max_over_ranks([time.perf_counter() - t0])
        # the trees went device -> float32 times -> device: same integers, log G close to the resident trees' (times rounded to float32)
        assert np.allclose(lgw, lg[:n_w], rtol=1e-4)
        wire = {"format": "delphy.api.Tree (FlatBuffers; core/api.fbs:13-49)", "trees_per_call": n_w, "buffer_bytes_per_tree": len(bufs[0]),
                "load_ms_per_tree": ld_s / reps_w / n_w * 1e3, "write_ms_per_tree": wr_ms,
                "note": "load: host buffer -> dphy_forest_upload_api_trees (struct vectors DMA'd as they lie; SoA split, CSR offsets, from_states "
                        "reconstruction, two flattens on the device) -> first evaluation -> log G read back, wall clock; write: "
                        "dphy_forest_write_api_tree (pack on the device + D2H)"}
    forest_bytes = forest.device_bytes
    nodes0, info0 = emats[0].num_nodes, infos[0]
    whole_emat, whole_sites = emats[0], host_sites[0]
    forest.close()
    for tb in tables[1:]:
        tb.close()

    # ---- secondary shapes: BASELINE.json configs[1], [2], [4] ------------------------------------------------------------------------------------
    secondary = {}
    if not args.no_secondary:
        for cfg, chains in SECONDARY.items():
            if cfg == args.config:
                continue
            se, st, si, sf = make_forest(cfg, chains)
            for _ in range(3):
                sf.eval_log_G()
            reps = 8
            ms, _ = time_evals(sf, max(3, args.steps // 2), reps)
            (ms,) = max_over_ranks([ms])
            ab = sf.log_G_algorithmic_bytes
            uniform = bool(np.all(st[0].host.nu_l == st[0].host.nu_l[0]))
            entry = {"workload": f"synthetic {SHAPES[cfg]} EMAT x {chains} chains per GPU", "value": chains * reps * world / (ms * 1e-3), "unit": UNIT,
                     "ms_per_eval": ms / reps, "schedule": "folded (uniform nu)" if uniform else "general (site-rate heterogeneity)",
                     "forest_device_bytes": sf.device_bytes, "l2": "larger than L2" if sf.device_bytes > 130e6 else "fits in L2",
                     "roofline": {"bound": "hbm", "achieved": ab / (ms / reps * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                  "frac": ab / (ms / reps * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": ab,
                                  "traffic": measured_traffic("emat_log_G_folded_kernel" if uniform else "emat_log_G_tile_kernel", cfg, chains)}}
            if spr_reqs is not None:
                # 32 full studies on each of up to 32 trees of the forest in ONE batch (one group of the event-scan path per tree):
                # small trees only fill the GPU when many chains ask at once
                sf.eval_log_G()
                rq = []
                for k in range(min(chains, 32)):
                    xs2 = pick_spr_nodes(se[k], 32, seed=1234 + k)
                    rq += db.spr_requests_for_attached(se[k], k, xs2, sf.lambda_i(k), si[k]["t_max_tip"])
                for _ in range(2):
                    sf.spr_study_batch(rq).close()
                a, b = ev(), ev()
                nb = max(4, args.steps)
                barrier(); a.record(stream)
                for _ in range(nb):
                    sf.spr_study_batch(rq).close()
                ctx.join_side_streams()
                b.record(stream); barrier()
                (sms,) = max_over_ranks([a.elapsed_time(b) / nb])
                bt = sf.spr_study_batch(rq); nreg = bt.total_regions(); bt.close()
                entry["spr_studies_per_batch"] = len(rq)
                entry["spr_candidates_per_s"] = nreg * world / (sms * 1e-3)
                entry["spr_roofline_frac"] = nreg * 60 / (sms * 1e-3) / 1e9 / peak
            secondary[str(cfg)] = entry
            sf.close()
            for tb in st:
                tb.close()

    # ---- one tree, parts spread over the ranks, one all-reduce per cycle -----------------------------------------------------------------
    partitioned = None
    if not args.no_partitioned:
        from delphy_b200 import partitioned as pp
        # every rank cuts the SAME tree (same seed) and keeps the parts i % world == rank
        pe, ps, pinfo = db.synth_generate(db.synth_params(args.config, seed=20251017))
        pt = pp.PartitionedTree(ctx, pe, ps, world, rank, parts_per_rank=args.parts_per_gpu, dist=dist if world > 1 else None,
                                torch=torch, device=dev)
        pt.cycle(1.0)
        got = pt.totals()
        want = pp.whole_tree_totals(ctx, pe, ps, torch, dev, 1.0)
        pp.check_totals(got, want)                 # Run::check_global_and_local_totals_match (core/run.cpp:340-357)
        psteps = max(20, args.steps * 4)
        cyc_ms, cyc_host_ms = pp.timed_cycles(pt, psteps, torch, reduce=True, barrier=barrier)
        nored_ms, _ = pp.timed_cycles(pt, psteps, torch, reduce=False, barrier=barrier)
        cyc_ms, nored_ms = max_over_ranks([cyc_ms, nored_ms])
        t0 = time.perf_counter()
        merged = pt.partition.reassemble()
        reasm_ms = (time.perf_counter() - t0) * 1e3
        assert merged.root == pe.root and np.array_equal(merged.parent, pe.parent) and np.array_equal(merged.mut_t, pe.mut_t)
        partitioned = {"workload": f"ONE synthetic {SHAPES[args.config]} EMAT cut into {pt.num_parts} parts, parts i % {world} on rank i",
                       "parallelism": "partition parts", "scaling": "strong", "parts": pt.num_parts, "parts_on_rank0": len(pt.mine),
                       "cycle": "set_evo(new mu) + log G / T / num_muts / num_muts_ab / Ttwiddle_beta_a of every local part + ONE all-reduce of 23 doubles",
                       "value": 1e3 / cyc_ms, "unit": "whole-tree cycles/s", "ms_per_cycle": cyc_ms, "ms_per_cycle_without_allreduce": nored_ms,
                       "allreduce_ms": max(0.0, cyc_ms - nored_ms), "collective": "NCCL all_reduce(sum), 23 x f64" if world > 1 else "none (1 rank)",
                       "host_enqueue_ms_per_cycle": cyc_host_ms, "totals_match_whole_tree": True, "log_G": float(got[0]),
                       "reassemble_ms_host": reasm_ms}
        pt.close()

    if rank == 0:
        value = args.chains * R * world / (logg_ms_max * 1e-3)
        eval_ms = logg_ms_max / R
        achieved = alg_bytes / (eval_ms * 1e-3) / 1e9
        traffic = measured_traffic("emat_log_G_folded_kernel", args.config, args.chains)
        cfg = config_block(args)          # identical in both arms (the driver compares them); what is specific to this arm goes beside it
        detail = {"nodes_per_chain": nodes0, "mutations_per_chain": info0["num_mutations"], "missation_intervals_per_chain": info0["num_intervals"],
                  "max_depth": info0["max_depth"], "forest_device_bytes": forest_bytes}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": logg_ms_max, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg, "workload_detail": detail,
            "roofline": {"kernel": "emat_log_G_folded_kernel (+ emat_log_G_folded_tree_kernel)", "bound": "hbm", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": eval_ms,
                         "achieved_dram_frac": (traffic / (eval_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "note": "algorithmic bytes = SURVEY 8(d) per-event figure; this schedule reads per-branch folded weights instead of the "
                                 "missation / from-state lists, so its DRAM traffic (traffic, achieved_dram_frac) is below the algorithmic bytes"},
            "loglik_general_schedule": {"value": args.chains * R * world / (gen_ms_max * 1e-3), "unit": UNIT, "launch_ms": gen_ms_max / R,
                                        "achieved": alg_bytes / (gen_ms_max / R * 1e-3) / 1e9, "frac": alg_bytes / (gen_ms_max / R * 1e-3) / 1e9 / peak,
                                        "traffic": measured_traffic("emat_log_G_tile_kernel", args.config, args.chains),
                                        "note": "every mutation / missation / from-state list re-read per evaluation (also refreshes nsmn and the num_muts tallies)"},
            "model_change_cycle": {"value": args.chains * mc_steps * world / mc_s, "unit": UNIT, "ms_per_cycle": mc_s / mc_steps * 1e3,
                                   "note": "dphy_sites_set_evo_many(new mu on every chain's site table, one launch) + evaluation of every chain + log G read back, wall clock"},
            "spr_candidates_per_s": (spr_regions * world / (spr_ms_max * 1e-3)) if spr_ms else None,
            "spr_regions_per_batch": spr_regions, "spr_ms_per_batch": spr_ms_max if spr_ms else None,
            "e2e": {"value": n_e2e * e2e_steps * world / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "chains_per_step": n_e2e, "steps": e2e_steps, "host_threads": n_thr,
                    "note": "per step: page-locked host arrays of every chain -> dphy_forest_upload (DMA + device-side flatten) -> evaluation -> log G read back"},
            "e2e_edit": {"value": args.chains * edit_steps * world / edit_s, "unit": UNIT, "h2d_bytes_per_step": int(edit_bytes), "d2h_bytes_per_step": int(args.chains * 3 * 8),
                         "ms_per_step": edit_s / edit_steps * 1e3, "chains_per_step": args.chains,
                         "note": "per step: one branch reform per chain shipped as rows (dphy_forest_apply_rows: resident host-order arrays patched and "
                                 "re-flattened on the device) + evaluation of every chain + log G read back; checked against a fresh upload of the edited trees"},
            "host_enqueue_ms_per_step": host_enqueue_ms, "gpu_launches": int(launches), "gpu_launches_spr": int(spr_launches), "clocks": clocks,
            "log_G_checksum": float(np.sum(lg_timed)),
        }
        if spr_ms:
            spr_alg = spr_regions * 60
            line["roofline_spr"] = {"bound": "hbm", "achieved": spr_alg / (spr_ms_max * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                    "frac": spr_alg / (spr_ms_max * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_candidate": 60,
                                    "launch_ms": spr_ms_max}
        if secondary:
            line["configs"] = secondary
        if partitioned:
            line["partitioned"] = partitioned
        if wire:
            line["wire_format"] = wire
        if world == 1 and not args.no_cpu_baseline:
            threads = host_cores()
            cb = cpu_log_G(whole_emat, whole_sites, args.cpu_seconds, threads)
            cb["spr"] = cpu_spr(whole_emat, whole_sites, spr_xs if spr_reqs is not None else None, args.cpu_seconds, threads, info0["t_max_tip"])
            if not args.no_partitioned:
                cb["partitioned"] = cpu_log_G_partitioned(db, whole_emat, whole_sites, args.cpu_seconds / 2, threads)
            if wire_buf0 is not None:
                cb["wire_format"] = cpu_api_tree_read(wire_buf0)
            line["cpu_baseline"] = cb
    tables[0].close()
    ctx.close()
    # MCMC steps/s through the reference's own driver with the hot path substituted at link time: one process (the driver's own
    # thread pool, one Subrun per thread, threads spread round-robin over the N GPUs), run by rank 0 while the other ranks wait
    if not args.no_mcmc:
        if rank == 0:
            line["mcmc"] = mcmc_figures(db, args, "dropin", world)
        if world > 1:
            dist.barrier()
    if rank == 0:
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dumped)
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
