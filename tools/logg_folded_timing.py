"""Folded log-G schedule on a 16 x 100k-tip forest: evaluation time back to back, the tile kernel's in-stream time, and its bytes.

usage: python tools/logg_folded_timing.py OUT.json [chains] [cfg]

Every figure comes from a child process of its own, because the launcher reads DPHY_FOLDED_REPEAT (tile kernel launched n times
per evaluation) once.  The tile kernel's in-stream time is
(t(repeat = 9) - t(repeat = 1)) / 8 of back-to-back evaluations: what one more launch adds in a saturated queue.  Its bytes per
evaluation are counted from the shapes: per node parent_pos, t, mut_off (4 + 8 + 4), the state-count row (4 * 4P) and lambda_i
written (8); per non-root mutation its code and time (1 + 8); per tile its two partials (16).  The parent's time is a gather of a
nearby node and is not counted again."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(chains, cfg):
    import numpy as np
    import torch
    import delphy_b200 as db
    ctx = db.Context(0)
    ems, tabs, P = [], [], 1
    for c in range(chains):
        e, s, _ = db.synth_generate(db.synth_params(cfg, seed=20251017 + c))
        ems.append(e); tabs.append(db.DeviceSites(ctx, s)); P = max(P, s.num_partitions)
    fo = db.Forest(ctx, ems, tabs, sites_index=np.arange(chains))
    st = torch.cuda.ExternalStream(ctx.stream)
    for _ in range(10):
        fo.eval_log_G()
    ctx.synchronize()
    reps, best = 200, None
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(reps):
            fo.eval_log_G()
        b.record(st); ctx.synchronize()
        us = a.elapsed_time(b) / reps * 1e3
        best = us if best is None else min(best, us)
    N = sum(e.num_nodes for e in ems)
    M = sum(int(e.mut_off[e.num_nodes]) - int(e.mut_off[e.root + 1] - e.mut_off[e.root]) for e in ems)
    tiles = sum((e.num_nodes + 511) // 512 for e in ems)
    nbytes = N * (4 + 8 + 4 + 16 * P + 8) + M * (1 + 8) + tiles * 16
    print(json.dumps({"eval_us": best, "nodes": N, "nonroot_mutations": M, "partitions": P, "tile_kernel_bytes": nbytes,
                      "log_G0": float(fo.log_G()[2][0])}))


def run(repeat, chains, cfg):
    env = dict(os.environ, DPHY_FOLDED_REPEAT=str(repeat))
    out = subprocess.run([sys.executable, __file__, "--child", str(chains), str(cfg)], env=env, check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def main():
    if sys.argv[1] == "--child":
        child(int(sys.argv[2]), int(sys.argv[3]))
        return
    out = sys.argv[1]
    chains = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    cfg = int(sys.argv[3]) if len(sys.argv) > 3 else 4
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    r1, r9 = run(1, chains, cfg), run(9, chains, cfg)
    tile_us = (r9["eval_us"] - r1["eval_us"]) / 8
    res = {"workload": f"{chains} x synthetic config {cfg} EMATs, folded log-G schedule", "gpu": gpu,
           "nodes": r1["nodes"], "nonroot_mutations": r1["nonroot_mutations"], "partitions": r1["partitions"],
           "eval_us": r1["eval_us"], "tile_kernel_in_stream_us": tile_us, "tile_kernel_bytes": r1["tile_kernel_bytes"],
           "tile_kernel_gb_s": r1["tile_kernel_bytes"] / (tile_us * 1e-6) / 1e9, "log_G0": r1["log_G0"]}
    print(json.dumps(res), flush=True)
    with open(out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
