import os, sys, json, torch
sys.path.insert(0, os.getcwd())
import bench
import kgc_gcn_b200 as k
orc = bench.oracle()
dev = torch.device('cuda', 0)
flush = bench.Flusher(dev)
for wl in sys.argv[1:]:
    case = bench.LayerCase(k, orc, wl, dev)
    roof, out = bench.kernel_rooflines(case, flush)
    print(wl, {n: round(v['ms'], 4) for n, v in out.items()}, {n: round(v['ms'], 4) for n, v in roof['passes'].items() if isinstance(v, dict)})
    del case
    k.plan._PLAN_CACHE.clear(); torch.cuda.empty_cache()
