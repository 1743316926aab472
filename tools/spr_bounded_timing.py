"""Bounded (max_muts_from_start = limit) vs full SPR studies on a 100k-tip tree: device time per batch of 64, and the reference's
own CPU time for the same studies (oracle/_ref, one thread per study).  usage: python tools/spr_bounded_timing.py [limit] [studies]"""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np, torch
import delphy_b200 as db
limit = int(sys.argv[1]) if len(sys.argv) > 1 else 2
nstudies = int(sys.argv[2]) if len(sys.argv) > 2 else 64
ctx = db.Context(0)
e, s, info = db.synth_generate(db.synth_params(4))
ds = db.DeviceSites(ctx, s); fo = db.Forest(ctx, [e], [ds])
lam = fo.lambda_i(0)
rng = np.random.default_rng(1234)
xs = [int(v) for v in rng.permutation(e.num_nodes)[:8 * nstudies] if v != e.root and e.parent[v] != e.root][:nstudies]
st = torch.cuda.ExternalStream(ctx.stream)
for name, lim in ((("full", 2**31 - 1),) if nstudies <= 64 else ()) + ((f"limit={limit}", limit),):
    reqs = db.spr_requests_for_attached(e, 0, xs, lam, info["t_max_tip"], lim, True)
    for _ in range(3):
        b = fo.spr_study_batch(reqs); b.close()
    a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(20):
        b = fo.spr_study_batch(reqs); b.close()
    c.record(st); ctx.synchronize()
    b = fo.spr_study_batch(reqs); n = b.total_regions(); b.close()
    print(f"{name:10s}: {a.elapsed_time(c)/20*1e3:8.1f} us per batch of {len(xs)} studies ({a.elapsed_time(c)/20/len(xs)*1e3:.1f} us per study), {n} regions")
try:
    if nstudies > 64: raise RuntimeError('large batch: device timing only')
    import ctypes as C
    import oracle_lib as ol
    from helpers import to_oracle
    if ol.ref_available():
        eo, so = to_oracle(e, s)
        o = ol.Oracle("ref")
        lam_o = o.lambda_i(eo, so)
        for name, lim in (("full", 2**31 - 1), (f"limit={limit}", limit)):
            t0 = time.perf_counter(); n = 0
            for X in xs[:16]:
                regs, _ = o.spr_study_from_attached(eo, so, X, lam_o, lim, True, 0.8, info["t_max_tip"]); n += len(regs)
            t = time.perf_counter() - t0
            print(f"reference CPU {name:10s}: {t/16*1e6:8.1f} us per study on one thread (incl. ctypes marshalling), {n} regions in 16 studies")
except Exception as ex:
    print("reference timing skipped:", ex)
