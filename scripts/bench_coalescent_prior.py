#!/usr/bin/env python
"""Time the exponential-growth coalescent log-prior of a resident forest (Forest.log_coalescent_prior, one synchronous call) against
the host round trip it replaces: the forest's node times copied device -> host, then a vectorised numpy evaluation per tree.

Forests have bench.py's shapes (tips per tree x trees per GPU): 200 x 1, 1,600 x 256, 10k x 64, 50k x 8, 100k x 16.  Only node times
enter the prior, so the synthetic trees are generated with short sequences (--sites) to keep set-up short.  Each figure is the
median of --reps timed calls after --warmup untimed ones, host wall clock around work that ends in a device synchronisation.  Both
paths must agree (rtol 1e-9).  Prints one JSON line per shape plus one with the device's name and power limit."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = [(1, 1), (2, 256), (3, 64), (5, 8), (4, 16)]     # (synthetic config, trees per forest), as in bench.py


def host_prior(t, tip, n0, g, t0):
    order = np.argsort(t, kind="stable")
    ts = t[order]
    k = 1 + np.cumsum(np.where(tip[order], -1, 1))
    a, d, kk = ts[:-1], np.diff(ts), k[:-1].astype(np.float64)
    gd = g * d
    with np.errstate(divide="ignore", invalid="ignore"):
        w = np.where(gd == 0.0, d, -np.expm1(-gd) / g)
    keep = (d > 0) & (kk >= 2)
    intervals = 0.5 * kk[keep] * (kk[keep] - 1) * np.exp(-g * (a[keep] - t0)) / n0 * w[keep]
    return -np.sum(np.log(n0) + g * (t[~tip] - t0)) - np.sum(intervals)


def median_ms(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        h0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - h0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--sites", type=int, default=2000)
    ap.add_argument("--configs", default=",".join(str(c) for c, _ in SHAPES), help="subset of the synthetic configs above")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    args = ap.parse_args()

    import torch
    import delphy_b200 as db
    if not torch.cuda.is_available():
        raise SystemExit("bench_coalescent_prior.py: no CUDA device")
    lines = []
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    lines.append(dict(device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1]))
    n0, g, t0 = 3.0, 10.0, 0.0
    wanted = {int(c) for c in args.configs.split(",")}
    with db.Context(0) as ctx:
        for cfg, chains in SHAPES:
            if cfg not in wanted:
                continue
            trees = [db.synth_generate(db.synth_params(cfg, num_sites=args.sites, seed=20251017 + 100000 * cfg + c)) for c in range(chains)]
            emats = [e for e, _, _ in trees]
            tables = [db.DeviceSites(ctx, s) for _, s, _ in trees]
            fo = db.Forest(ctx, emats, tables, sites_index=np.arange(chains))
            tips = [e.child0 < 0 for e in emats]
            bounds = np.cumsum([0] + [e.num_nodes for e in emats])
            t_dev = torch.tensor(np.concatenate([e.t for e in emats]), dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()

            def host():
                t = t_dev.cpu().numpy()
                return np.array([host_prior(t[bounds[k]:bounds[k + 1]], tips[k], n0, g, t0) for k in range(chains)])

            gpu = fo.log_coalescent_prior(n0, g, t0)
            np.testing.assert_allclose(gpu, host(), rtol=1e-9, atol=0)
            dev_ms = median_ms(lambda: fo.log_coalescent_prior(n0, g, t0), args.warmup, args.reps)
            host_ms = median_ms(host, args.warmup, args.reps)
            lines.append(dict(shape=f"{chains} x {emats[0].num_nodes // 2 + 1}-tip trees", nodes=int(bounds[-1]),
                              device_call_ms_median=round(dev_ms[0], 4), device_call_ms_min_max=[round(x, 4) for x in dev_ms[1:]],
                              host_round_trip_ms_median=round(host_ms[0], 4), host_round_trip_ms_min_max=[round(x, 4) for x in host_ms[1:]],
                              host_over_device=round(host_ms[0] / dev_ms[0], 2)))
            print(json.dumps(lines[-1]), flush=True)
            fo.close()
            for t in tables:
                t.close()
    print(json.dumps(lines[0]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
