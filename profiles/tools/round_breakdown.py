import sys,time,importlib,os; sys.path.insert(0,os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
pkg=importlib.import_module("batch-scheduler_b200")
import numpy as np
S=pkg.snapshot
def bench(name, snap, flags):
    eng=pkg.Engine(snap.lanes, 0, **flags); eng.upload(snap)
    for _ in range(5): eng.evaluate()
    n=50
    t0=time.perf_counter()
    for _ in range(n): eng.evaluate_async()
    eng.sync(); dt=(time.perf_counter()-t0)/n
    eng.set_profiling(True)
    acc={}
    for _ in range(10):
        eng.evaluate_async(); eng.sync()
        for k,(ms,nl) in eng.kernel_ms().items(): acc[k]=acc.get(k,0)+ms/10
    print(f"{name:24s} P={snap.pods.n:7d} N={snap.nodes.n:6d} step {dt*1e3:7.3f} ms | "+" ".join(f"{k}={v*1e3:.0f}us" for k,v in acc.items() if v>0), flush=True)
    eng.close()
dec=dict(fit_bitmap=False, score=False); full=dict(fit_bitmap=True, score=True)
bench("readme", S.readme_scenario(), full)
bench("cfg2 full", S.config(2), full)
bench("cfg4 x0.1", S.config(4,0.1), dec)
bench("cfg4 x0.16", S.config(4,0.16), dec)
bench("cfg3 x0.1", S.config(3,0.1), dec)
