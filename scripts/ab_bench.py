"""A/B of tuning switches in ONE process: device time of a lock-step solve and its stage split per (config, env).
usage: ab_bench.py B reps CONFIG[:ENV=VAL[,ENV=VAL]] ...      e.g.  ab_bench.py 65536 2 C4 C4:TG_QP_STAGED=0"""
import sys, os, ctypes, torch, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from trajectory_generator_b200 import batch as tgb, synthetic as syn, _native
B = int(sys.argv[1]); reps = int(sys.argv[2])
dev = torch.device("cuda:0")
lib = _native.lib()
cache = {}
for item in sys.argv[3:]:
    name, _, envs = item.partition(":")
    mode = "fd"
    sets = {}
    for kv in filter(None, envs.split(",")):
        k, v = kv.split("=")
        if k == "mode": mode = v
        else: sets[k] = v
    for k, v in sets.items(): os.environ[k] = v
    if name not in cache:
        bt = syn.make(name, B)
        cache[name] = (bt, torch.from_numpy(bt.par).to(dev), torch.from_numpy(bt.x0).to(dev), tgb.SolveBuffers(bt.spec, B, dev))
    bt, par, x0, bufs = cache[name]
    if bufs.ws.numel() < lib.tg_solve_workspace_bytes(bufs.sp, B):      # a switch that adds workspace slots (TG_QP_FAR=1)
        bufs = tgb.SolveBuffers(bt.spec, B, dev)
        cache[name] = (bt, par, x0, bufs)
    ts = []
    for r in range(reps + 1):
        x = x0.clone()
        s = torch.cuda.Event(enable_timing=True); e = torch.cuda.Event(enable_timing=True)
        s.record(); out = tgb.solve(bt.spec, par, x, jacobian=mode, buffers=bufs); e.record(); torch.cuda.synchronize()
        if r: ts.append(s.elapsed_time(e))
    lib.tg_set_stage_timing(1)
    x = x0.clone(); tgb.solve(bt.spec, par, x, jacobian=mode, buffers=bufs); torch.cuda.synchronize()
    lib.tg_set_stage_timing(0)
    st = (ctypes.c_double * 6)(); lib.tg_last_solve_stats(st, 6)
    print("%-28s %s B=%d: %.1f ms (min %.1f) ls+der %.1f qp %.1f (%.3g flop) | status0 %.4f nit %.2f xsum %.10e -> %.0f traj/s" % (
        item, mode, B, np.mean(ts), np.min(ts), st[0], st[1], st[2], (out["status"] == 0).float().mean().item(),
        out["nit"].float().mean().item(), out["x"].double().sum().item(), B / np.min(ts) * 1e3), flush=True)
    for k in sets: os.environ.pop(k, None)
