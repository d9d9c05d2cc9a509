"""Cholesky alone (cip_factor_H after cip_form_H) at several n: CUDA-event time and TFLOP/s.
usage: python scripts/chol_timing.py [n ...]   (env CIP_CHOL_OUTER selects the outer panel width)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, scipy.sparse as sp
import conicip_b200 as cb

for n in [int(a) for a in sys.argv[1:]] or [1000, 4096, 8192, 16384]:
    m = 2 * n
    g = torch.Generator(device="cuda"); g.manual_seed(n)
    At = torch.randn((n, m), generator=g, dtype=torch.float64, device="cuda") / n ** 0.5
    q = 1.0 + torch.rand(n, generator=g, dtype=torch.float64, device="cuda")
    eng = cb.Engine(sp.diags(q.cpu().numpy()).tocsr(), At.t(), None, [("R", m)])
    eng._bind_stream()
    v = torch.rand(m, generator=g, dtype=torch.float64, device="cuda") + 0.5
    s = torch.rand(m, generator=g, dtype=torch.float64, device="cuda") + 0.5
    eng.nt_scaling(v, s)
    ts = []
    for rep in range(6):
        eng.form_H()
        assert eng.factor_H() == 0
        ts.append(eng.stats()["ms_chol"])
    best = min(ts[1:])
    print(f"n={n}: cholesky {best:.3f} ms  {n**3/3/(best*1e-3)/1e12:.2f} TFLOP/s", flush=True)
    eng.close()
