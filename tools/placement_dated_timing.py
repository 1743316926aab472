"""Dated placement of new samples (dphy_forest_place_dated_samples) on the synthetic trees of BASELINE.json, config 4 (100k tips) and
config 5 (50k tips x 197k sites, heavy missing data).  Samples are the trees' own tips, each with its own time as the date limit.
Reported, host arrays to host results: dated placements/s; the undated call on the same samples; the study route with the same
limits (one full REL_REF study per sample through dphy_spr_study_batch, batches of 128, lambda_X = 0, regions left on the device:
a lower bound of that route).  Also the placement kernel's device time per sample (torch.profiler), the dated index's build time
(first dated call minus a repeat, on a fresh tree and again after dphy_forest_set_node_times) and its resident bytes.
usage: python tools/placement_dated_timing.py [--out profiles/placement_dated_timing.json] [--quick]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
import torch

import delphy_b200 as db
from delphy_b200 import maple
from placement_timing import INF, rel_ref_inputs, sample_set

DBL_MAX = np.finfo(np.float64).max


def kernel_ms(fo, arrays, t_X):
    """device time of the placement kernel in one call (torch.profiler)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fo.place_samples(arrays, t_X=t_X)
        torch.cuda.synchronize()
    tot = 0.0
    for ev in prof.events():
        if "place_samples_kernel" in ev.name:
            tot += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
    return tot / 1e3


def wall(fn, reps=3):
    fn()                                               # warm-up of this shape
    ws = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ws.append(time.perf_counter() - t0)
    return float(np.median(ws)), ws


def workload(ctx, cfg, S, study_samples, rng):
    emat, sites, info = db.synth_generate(db.synth_params(cfg))
    ds = db.DeviceSites(ctx, sites)
    fo = db.Forest(ctx, [emat], [ds])
    R = emat.num_nodes + int(emat.mut_off[-1]) - int(emat.mut_off[emat.root + 1] - emat.mut_off[emat.root])
    res = dict(config=cfg, num_tips=int((emat.child0 < 0).sum()), num_sites=sites.num_sites, num_mutations=int(emat.mut_off[-1]), regions=R)
    tips = list(maple.tip_sequences(emat, sites))
    order = rng.permutation(len(tips))
    picked = [tips[order[k % len(tips)]] for k in range(S)]
    samples = [(list(d.items()), iv) for _, d, iv in picked]
    t_X = np.array([float(emat.t[v]) for v, _, _ in picked])
    arrays = sample_set(samples)
    one, one_t = sample_set(samples[:1]), np.array([float(np.median(emat.t))])
    # index builds: the undated part first, then the dated part (cold minus warm, on one sample whose limit drops regions)
    fo.place_samples(one)
    b0 = fo.device_bytes
    t0 = time.perf_counter(); fo.place_samples(one, t_X=one_t); t1 = time.perf_counter()
    fo.place_samples(one, t_X=one_t); t2 = time.perf_counter()
    res["dated_index_bytes"] = fo.device_bytes - b0
    res["dated_index_build_ms"] = ((t1 - t0) - (t2 - t1)) * 1e3
    v = picked[0][0]
    fo.set_node_times(0, [v], [emat.t[v]])             # same time: the dated part is stale all the same
    t0 = time.perf_counter(); fo.place_samples(one, t_X=one_t); t1 = time.perf_counter()
    fo.place_samples(one, t_X=one_t); t2 = time.perf_counter()
    res["dated_index_rebuild_ms"] = ((t1 - t0) - (t2 - t1)) * 1e3
    assert fo.device_bytes - b0 == res["dated_index_bytes"]
    # dated and undated calls on the same samples, alternated
    wd, wd_all = wall(lambda: fo.place_samples(arrays, t_X=t_X))
    wu, wu_all = wall(lambda: fo.place_samples(arrays))
    wd2, wd2_all = wall(lambda: fo.place_samples(arrays, t_X=t_X))
    got = fo.place_samples(arrays, t_X=t_X)
    und = fo.place_samples(arrays)
    kd, ku = kernel_ms(fo, arrays, t_X), kernel_ms(fo, arrays, None)
    res["dated"] = dict(samples=S, wall_s=min(wd, wd2), wall_all_s=wd_all + wd2_all, placements_per_s=S / min(wd, wd2), kernel_ms=kd,
                        kernel_us_per_sample=kd * 1e3 / S, mean_min_muts=float(got["min_muts"].mean()),
                        mean_num_best=float(got["num_best"].mean()))
    res["undated"] = dict(samples=S, wall_s=wu, wall_all_s=wu_all, placements_per_s=S / wu, kernel_ms=ku, kernel_us_per_sample=ku * 1e3 / S,
                          mean_min_muts=float(und["min_muts"].mean()), mean_num_best=float(und["num_best"].mean()))
    print(f"config {cfg}: {S} samples  dated {S / min(wd, wd2):10.0f}/s (kernel {kd:8.2f} ms)  undated {S / wu:10.0f}/s "
          f"(kernel {ku:8.2f} ms)  dated index {res['dated_index_bytes'] / 1e6:.1f} MB, build {res['dated_index_build_ms']:.2f} ms, "
          f"rebuild {res['dated_index_rebuild_ms']:.2f} ms", flush=True)
    # the study route with the same limits: one full study per sample, 128 per batch, regions left on the device
    root = int(emat.root)
    n_root = int(emat.mut_off[root + 1] - emat.mut_off[root])
    reqs = []
    for smp, tX in zip(samples[:study_samples], t_X[:study_samples]):
        rs, x, miss = rel_ref_inputs(emat, sites, smp)
        d, iv = smp
        reqs.append(db.spr_request(0, -1, float(tX), root, n_root, int((~miss & (rs != x)).sum()), 0.0, info["t_max_tip"], INF, True,
                                   x_deltas=d, x_missing=([a for a, _ in iv], [b for _, b in iv]), x_state_mode=db.SPR_X_REL_REF))
    batches = [reqs[i:i + 128] for i in range(0, len(reqs), 128)]

    def studies():
        for br in batches:
            b = fo.spr_study_batch(br); b.close()
        ctx.join_side_streams(); ctx.synchronize()
    ws, ws_all = wall(studies, 2)
    n = len(reqs)
    res["study_route"] = dict(samples=n, batch=128, wall_s=ws, wall_all_s=ws_all, samples_per_s=n / ws)
    print(f"config {cfg}: study route {n} samples {ws * 1e3:9.1f} ms  {n / ws:10.0f} samples/s", flush=True)
    fo.close(); ds.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "placement_dated_timing.json"))
    ap.add_argument("--quick", action="store_true", help="small sample counts (a rehearsal)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("placement_dated_timing: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    out = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=smi.stdout.strip(), workloads=[])
    ctx = db.Context(0)
    rng = np.random.default_rng(2026)
    if a.quick:
        out["workloads"].append(workload(ctx, 1, 100, 128, rng))
    else:
        out["workloads"].append(workload(ctx, 4, 10000, 2048, rng))
        out["workloads"].append(workload(ctx, 5, 10000, 1024, rng))
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
