import sys, time, torch
sys.path.insert(0, '.')
from vexautonomousplanner_b200 import synth
from vexautonomousplanner_b200.engine import Engine
B = int(sys.argv[1]); N = int(sys.argv[2]) if len(sys.argv) > 2 else 8
packed = synth.random_paths(B, N, seed=1)
for vi, ti in (("chunked", "split"), ("serial", "serial")):
    eng = Engine("cuda:0", velocity_impl=vi, time_impl=ti)
    db = eng.upload(packed)
    for _ in range(2):
        res = eng.profile(db, reuse_plan=True)
    torch.cuda.synchronize()
    eng.stage_events = []
    t0 = time.perf_counter()
    for _ in range(3):
        res = eng.profile(db, reuse_plan=True)
    torch.cuda.synchronize()
    el = (time.perf_counter() - t0) / 3
    st = {}
    for name, s, e in eng.stage_events:
        st[name] = st.get(name, 0.0) + s.elapsed_time(e) / 3
    print(f"B={B} N={N} velocity={vi} time={ti}: {el*1e3:.2f} ms/step -> {B/el:.0f} paths/s", {k: round(v, 2) for k, v in st.items()})
    del eng, db, res
    torch.cuda.empty_cache()
