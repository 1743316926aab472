"""Clade tables (dphy_clade_table_*) on forests of 16 trees of 100k tips (config 4's tree shape; mutation lists left empty: clades
depend only on topology and times), at the two extremes: 16 copies of one tree (every clade shared) and 16 independent trees (almost
every clade new).  Reported, host call to host result (every call ends in a stream synchronise): trees added per second into an empty
table and into a table already holding 48 trees, scores per second, table bytes after 64 trees, the device time per kernel of one add
and one score (torch.profiler, a separate pass), and a host baseline on the same trees: numpy clade keys (levels of the tree, deepest
first) and sort-based grouping into counts and time sums, single process.
usage: python tools/clade_timing.py [--out profiles/clade_timing.json] [--quick]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np

import delphy_b200 as db


def bare_tree(cfg, seed, **kw):
    e, _, _ = db.synth_generate(db.synth_params(cfg, seed=seed, muts_per_tip=0.0, missing_mean_intervals_per_tip=0.0, num_sites=100, **kw))
    z = np.zeros(e.num_nodes + 1, np.int32)
    return db.HostEmat(e.root, parent=e.parent, child0=e.child0, child1=e.child1, t=e.t, mut_off=z, mut_site=[], mut_from=[], mut_to=[],
                       mut_t=[], miss_off=z, miss_start=[], miss_end=[], fs_off=z, fs_site=[], fs_from=[])


def tiny_sites(L=8):
    q = np.full((4, 4), 1.0 / 3.0)
    np.fill_diagonal(q, -1.0)
    return db.HostSites(np.zeros(L, np.uint8), np.zeros(L, np.int32), np.ones(L), [1.0], [0.25] * 4, q)


def wall(fn, reps):
    fn()                                               # warm-up of this shape
    ws = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ws.append(time.perf_counter() - t0)
    return float(np.median(ws)), ws


# ---- host baseline ----------------------------------------------------------------------------------------------------------------------
def splitmix64(x):
    x = x + np.uint64(0x9e3779b97f4a7c15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
    return x ^ (x >> np.uint64(31))


def host_keys(e):
    """the library's clade keys of every node, in numpy: depth by pointer jumping, then children into parents level by level"""
    parent = e.parent.astype(np.int64)
    d = (parent >= 0).astype(np.int64)
    a = parent.copy()
    while True:
        m = a >= 0
        if not m.any():
            break
        d[m] += d[a[m]]
        a[m] = a[a[m]]
    tip = e.child0 < 0
    idx = np.arange(e.num_nodes, dtype=np.uint64)
    with np.errstate(over="ignore"):
        k = np.zeros((e.num_nodes, 2), np.uint64)
        k[tip, 0] = splitmix64(idx[tip] << np.uint64(1))
        k[tip, 1] = splitmix64(idx[tip] << np.uint64(1) | np.uint64(1))
        order = np.argsort(-d, kind="stable")
        bounds = np.flatnonzero(np.diff(d[order])) + 1
        for lvl in np.split(order, bounds):
            lvl = lvl[parent[lvl] >= 0]
            np.add.at(k, parent[lvl], k[lvl])
    return k


def host_group(keys, t):
    """counts and time sums per distinct key (sort-based)"""
    o = np.lexsort((keys[:, 1], keys[:, 0]))
    ks = keys[o]
    head = np.ones(len(ks), bool)
    head[1:] = np.any(ks[1:] != ks[:-1], axis=1)
    starts = np.flatnonzero(head)
    counts = np.diff(np.append(starts, len(ks)))
    sums = np.add.reduceat(t[o], starts)
    return counts, sums


def host_baseline(trees):
    t0 = time.perf_counter()
    keys = np.concatenate([host_keys(e) for e in trees])
    t1 = time.perf_counter()
    counts, _ = host_group(keys, np.concatenate([e.t for e in trees]))
    t2 = time.perf_counter()
    return dict(keys_s=t1 - t0, group_s=t2 - t1, total_s=t2 - t0, trees_per_s=len(trees) / (t2 - t0), num_clades=int(len(counts)))


# ---- device -----------------------------------------------------------------------------------------------------------------------------
def kernel_ms(fn):
    """device time per kernel name over one call (torch.profiler)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        name = ev.name if "clade_" in ev.name else ev.name.split("<")[0].split("(")[0][:60]
        out[name] = out.get(name, 0.0) + (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def table_with(ctx, forests):
    tab = db.CladeTable(ctx)
    for f in forests:
        tab.add(f)
    return tab


def workload(ctx, forests, reps):
    """forests: four forests of 16 trees; the first is the one timed"""
    fo = forests[0]
    res = dict(trees_per_forest=fo.num_trees, nodes_per_tree=fo.emats[0].num_nodes)
    ms, _ = wall(lambda: table_with(ctx, [fo]).close(), reps)
    res.update(add_empty_ms=ms * 1e3, add_empty_trees_per_s=fo.num_trees / ms)
    times = []
    for _ in range(reps + 1):                          # each: a 48-tree table, then the timed add of the 16 (the first is a warm-up)
        t48 = table_with(ctx, forests[1:])
        t0 = time.perf_counter(); t48.add(fo); times.append(time.perf_counter() - t0)
        t48.close()
    ms = float(np.median(times[1:]))
    res.update(add_after_48_ms=ms * 1e3, add_after_48_trees_per_s=fo.num_trees / ms)
    full = table_with(ctx, forests[1:] + [fo])
    res["table_after_64"] = dict(num_trees=full.num_trees, num_clades=full.num_clades, device_bytes=full.device_bytes)
    ms, _ = wall(lambda: full.score(fo), reps)
    res.update(score_ms=ms * 1e3, scores_per_s=fo.num_trees / ms)
    t48 = table_with(ctx, forests[1:])
    res["clades_after_48"] = t48.num_clades
    res["kernels_add_after_48_ms"] = kernel_ms(lambda: t48.add(fo))
    res["kernels_score_ms"] = kernel_ms(lambda: full.score(fo))
    t48.close(); full.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "clade_timing.json"))
    ap.add_argument("--quick", action="store_true", help="2k-tip trees, few repetitions (a rehearsal)")
    a = ap.parse_args()
    cfg, reps = (0, 2) if a.quick else (4, 5)
    kw = dict(num_tips=2000) if a.quick else {}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    gpu = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown (nvidia-smi failed)"

    t0 = time.perf_counter()
    independent = [bare_tree(cfg, 5000 + k, **kw) for k in range(64)]
    gen_s = time.perf_counter() - t0
    same = [independent[0]] * 64
    out = dict(tool="tools/clade_timing.py", gpu=gpu, config=cfg, quick=a.quick, tree_generation_s=gen_s,
               note="wall time of each synchronous call, median of %d after a warm-up" % reps)
    with db.Context(0) as ctx:
        ds = db.DeviceSites(ctx, tiny_sites())
        for name, trees in (("identical", same), ("independent", independent)):
            forests = [db.Forest(ctx, trees[16 * i:16 * (i + 1)], [ds]) for i in range(4)]
            out[name] = workload(ctx, forests, reps)
            out[name]["host_baseline"] = host_baseline(trees[:16])
            dev = db.CladeTable(ctx)
            dev.add(forests[0])
            assert dev.num_clades == out[name]["host_baseline"]["num_clades"], (dev.num_clades, out[name]["host_baseline"])
            dev.close()
            for f in forests:
                f.close()
        ds.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
