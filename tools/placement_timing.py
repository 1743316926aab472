"""Placement of new samples (dphy_forest_place_samples) on the synthetic trees of BASELINE.json: placements/s from host arrays to host
results, the placement kernel's device time (torch.profiler), the one-off index build, the existing route (one full REL_REF study per
sample through dphy_spr_study_batch, batches of 128, lambda_X = 0, regions left on the device: a lower bound of that route) and the
C oracle's single-thread rate.  Samples are the trees' own tips -- their missing intervals are the synthetic missing-data model's --
with 0-3 random extra deltas each.
usage: python tools/placement_timing.py [--out profiles/placement_timing.json] [--quick]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import delphy_b200 as db
from delphy_b200 import maple
from helpers import to_oracle
from oracle_lib import Oracle

INF = 2**31 - 1
DBL_MAX = np.finfo(np.float64).max


def tip_samples(emat, sites, n, rng):
    tips = list(maple.tip_sequences(emat, sites))
    order = rng.permutation(len(tips))
    L = sites.num_sites
    out = []
    for k in range(n):
        _, diffs, missing = tips[order[k % len(tips)]]
        d = list(diffs.items()) + [(int(rng.integers(L)), int(rng.integers(4))) for _ in range(int(rng.integers(0, 4)))]
        out.append((d, missing))
    return out


def sample_set(samples):
    d_off = np.zeros(len(samples) + 1, np.int32)
    m_off = np.zeros(len(samples) + 1, np.int32)
    d_off[1:] = np.cumsum([len(d) for d, _ in samples])
    m_off[1:] = np.cumsum([len(iv) for _, iv in samples])
    return dict(delta_off=d_off, delta_site=np.array([l for d, _ in samples for l, _ in d], np.int32),
                delta_to=np.array([t for d, _ in samples for _, t in d], np.uint8), miss_off=m_off,
                miss_start=np.array([a for _, iv in samples for a, _ in iv], np.int32),
                miss_end=np.array([b for _, iv in samples for _, b in iv], np.int32))


def size_of_A(emat, sites, samples):
    """|A| per sample (mutations of the tree at its delta and missing sites, duplicates counted once)"""
    L = sites.num_sites
    per_site = np.bincount(emat.mut_site, minlength=L)
    out = []
    for d, iv in samples:
        mask = np.zeros(L, bool)
        for a, b in iv:
            mask[a:b] = True
        for l, _ in d:
            mask[l] = True
        out.append(int(per_site[mask].sum()))
    return np.array(out)


def rel_ref_inputs(emat, sites, sample):
    ref = np.asarray(sites.ref, np.uint8)
    root = int(emat.root)
    rs = ref.copy()
    for i in range(int(emat.mut_off[root]), int(emat.mut_off[root + 1])):
        rs[int(emat.mut_site[i])] = int(emat.mut_to[i])
    d, iv = sample
    x = ref.copy()
    for l, t in d:
        x[l] = t
    miss = np.zeros(len(ref), bool)
    for a, b in iv:
        miss[a:b] = True
    return rs, x, miss


def kernel_ms(fo, arrays):
    """device time of the placement kernels in one call (torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fo.place_samples(arrays)
        torch.cuda.synchronize()
    tot = 0.0
    for ev in prof.events():
        if "place_samples_kernel" in ev.name:
            tot += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    return tot / 1e3


def workload(ctx, orc, cfg, sample_counts, rng, study_samples, oracle_samples):
    emat, sites, info = db.synth_generate(db.synth_params(cfg))
    ds = db.DeviceSites(ctx, sites)
    fo = db.Forest(ctx, [emat], [ds])
    R = emat.num_nodes + int(emat.mut_off[-1]) - int(emat.mut_off[emat.root + 1] - emat.mut_off[emat.root])
    res = dict(config=cfg, num_tips=int((emat.child0 < 0).sum()), num_sites=sites.num_sites, num_mutations=int(emat.mut_off[-1]), regions=R)
    all_samples = tip_samples(emat, sites, max(sample_counts), rng)
    A = size_of_A(emat, sites, all_samples[:2000])
    res["A_per_sample"] = dict(mean=float(A.mean()), median=float(np.median(A)), p99=float(np.percentile(A, 99)), max=int(A.max()))
    one = sample_set(all_samples[:1])
    t0 = time.perf_counter(); fo.place_samples(one); t1 = time.perf_counter()
    fo.place_samples(one); t2 = time.perf_counter()
    res["index_build_ms"] = ((t1 - t0) - (t2 - t1)) * 1e3
    res["index_first_call_ms"] = (t1 - t0) * 1e3
    res["runs"] = []
    for S in sample_counts:
        arrays = sample_set(all_samples[:S])
        fo.place_samples(arrays)                       # warm-up of this shape
        walls = []
        for _ in range(3):
            t0 = time.perf_counter(); got = fo.place_samples(arrays); walls.append(time.perf_counter() - t0)
        w = float(np.median(walls))
        km = kernel_ms(fo, arrays)
        res["runs"].append(dict(samples=S, wall_s=w, wall_all_s=walls, placements_per_s=S / w, kernel_ms=km,
                                kernel_us_per_sample=km * 1e3 / S, mean_min_muts=float(got["min_muts"].mean()),
                                mean_num_best=float(got["num_best"].mean())))
        print(f"config {cfg}: {S} samples  {w * 1e3:9.1f} ms wall  {S / w:10.0f} placements/s  kernel {km:8.2f} ms", flush=True)
    # the existing route: one full study per sample, 128 per batch, regions left on the device
    sub = all_samples[:study_samples]
    root = int(emat.root)
    n_root = int(emat.mut_off[root + 1] - emat.mut_off[root])
    reqs = []
    for smp in sub:
        rs, x, miss = rel_ref_inputs(emat, sites, smp)
        d, iv = smp
        reqs.append(db.spr_request(0, -1, DBL_MAX, root, n_root, int((~miss & (rs != x)).sum()), 0.0, info["t_max_tip"], INF, True,
                                   x_deltas=d, x_missing=([a for a, _ in iv], [b for _, b in iv]), x_state_mode=db.SPR_X_REL_REF))
    batches = [reqs[i:i + 128] for i in range(0, len(reqs), 128)]
    for br in batches:                                 # warm-up: the batches' device blocks reach their steady state
        b = fo.spr_study_batch(br); b.close()
    ctx.join_side_streams(); ctx.synchronize()
    t0 = time.perf_counter()
    for br in batches:
        b = fo.spr_study_batch(br); b.close()
    ctx.join_side_streams(); ctx.synchronize()
    ws = time.perf_counter() - t0
    res["study_route"] = dict(samples=len(sub), batch=128, wall_s=ws, samples_per_s=len(sub) / ws)
    print(f"config {cfg}: study route {len(sub)} samples {ws * 1e3:9.1f} ms  {len(sub) / ws:10.0f} samples/s", flush=True)
    # the C oracle, one thread: the builder's whole study per sample (the ctypes call only)
    e, s = to_oracle(emat, sites)
    tt = 0.0
    for smp in sub[:oracle_samples]:
        rs, x, miss = rel_ref_inputs(emat, sites, smp)
        miss2 = np.concatenate([[False], miss, [False]]).astype(np.int8)
        ed = np.diff(miss2)
        ms, me = np.nonzero(ed == 1)[0].astype(np.int32), np.nonzero(ed == -1)[0].astype(np.int32)
        idx = np.nonzero(~miss & (rs != x))[0]
        init = [(int(l), int(rs[l]), int(x[l])) for l in idx]
        t0 = time.perf_counter()
        orc.spr_study(e, s, -1, DBL_MAX, (ms, me), root, n_root, init, INF, True)
        tt += time.perf_counter() - t0
    res["oracle_cpu"] = dict(samples=oracle_samples, s_per_sample=tt / oracle_samples, samples_per_s=oracle_samples / tt)
    print(f"config {cfg}: C oracle {oracle_samples / tt:8.1f} samples/s on one thread", flush=True)
    fo.close(); ds.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "placement_timing.json"))
    ap.add_argument("--quick", action="store_true", help="small sample counts (a rehearsal)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("placement_timing: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=smi.stdout.strip(), workloads=[])
    ctx = db.Context(0)
    orc = Oracle("oracle")
    rng = np.random.default_rng(2026)
    if a.quick:
        out["workloads"].append(workload(ctx, orc, 1, [100], rng, 128, 4))
    else:
        out["workloads"].append(workload(ctx, orc, 4, [10000, 100000], rng, 1024, 20))
        out["workloads"].append(workload(ctx, orc, 5, [10000], rng, 512, 10))
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
