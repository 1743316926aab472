"""Folded log-G timing (back-to-back evaluations between two events).  usage: python tools/logg_occ.py [chains] [cfg]"""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import delphy_b200 as db
chains = int(sys.argv[1]) if len(sys.argv) > 1 else 16
cfg = int(sys.argv[2]) if len(sys.argv) > 2 else 4
ctx = db.Context(0)
ems, tabs = [], []
for c in range(chains):
    e, s, info = db.synth_generate(db.synth_params(cfg, seed=20251017 + c))
    ems.append(e); tabs.append(db.DeviceSites(ctx, s))
fo = db.Forest(ctx, ems, tabs, sites_index=np.arange(chains))
st = torch.cuda.ExternalStream(ctx.stream)
for path in ("auto", "general"):
    ctx.set_log_G_path(path)
    for _ in range(5): fo.eval_log_G()
    ctx.synchronize()
    a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
    a.record(st); t0 = time.perf_counter()
    for _ in range(200): fo.eval_log_G()
    t1 = time.perf_counter(); b.record(st); ctx.synchronize()
    print(f"path={path} eval={a.elapsed_time(b)/200*1e3:8.1f} us  host_enqueue={(t1-t0)/200*1e6:6.1f} us  logG0={fo.log_G()[2][0]:.9f}")
