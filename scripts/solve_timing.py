import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, scipy.sparse as sp
import conicip_b200 as cb
from conicip_b200 import problems as P
prob = P.config4_device(n=8192, m=16384, seed=4)
eng = cb.Engine(sp.diags(prob["qdiag"].cpu().numpy()).tocsr(), prob["At"].t(), None, prob["cone_dims"])
eng._bind_stream()
for rep in range(4):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    y, w, v, info = eng.ipm_solve(prob["c"], prob["b"], None, optTol=1e-8)
    torch.cuda.synchronize(); print(rep, time.perf_counter() - t0, info["seconds"], info["Iter"], info["factors"], info["solves"], flush=True)
