import sys,time,importlib,os; sys.path.insert(0,os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
pkg=importlib.import_module("batch-scheduler_b200")
import numpy as np
S=pkg.snapshot
def bench(name, snap, flags):
    eng=pkg.Engine(snap.lanes, 0, **flags); eng.upload(snap)
    for _ in range(5): eng.evaluate()
    n=50
    ta=tb=tc=0.0
    for _ in range(n):
        t0=time.perf_counter(); eng.evaluate_async(); t1=time.perf_counter(); eng.sync(); t2=time.perf_counter(); r=eng.fetch(); t3=time.perf_counter()
        ta+=t1-t0; tb+=t2-t1; tc+=t3-t2
    t0=time.perf_counter()
    for _ in range(n): eng.evaluate_async()
    eng.sync(); dt=(time.perf_counter()-t0)/n
    print(f"{name:28s} P={snap.pods.n:7d} N={snap.nodes.n:6d} async {ta/n*1e3:7.3f} ms  sync {tb/n*1e3:7.3f}  fetch {tc/n*1e3:7.3f}  | back-to-back step {dt*1e3:7.3f} ms  launches/step {eng.launch_count()//(2*n+5)}", flush=True)
    eng.close()
full=dict(fit_bitmap=True, score=True); dec=dict(fit_bitmap=False, score=False)
bench("readme", S.readme_scenario(), full)
bench("cfg2 full outputs", S.config(2), full)
bench("cfg2 decisions", S.config(2), dec)
bench("cfg4 x0.1 decisions", S.config(4,0.1), dec)
bench("cfg4 full outputs", S.config(4), full)
bench("cfg4 decisions", S.config(4), dec)
