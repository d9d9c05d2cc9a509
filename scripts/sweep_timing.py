"""Triangular sweeps alone (cip_solve_H): correctness against the factor read back, and CUDA-event timing.
usage: python scripts/sweep_timing.py [n ...]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, scipy.sparse as sp
import conicip_b200 as cb

for n in [int(a) for a in sys.argv[1:]] or [1000, 4096, 8192, 16384]:
    m = 2048
    g = torch.Generator(device="cuda"); g.manual_seed(n)
    At = torch.randn((n, m), generator=g, dtype=torch.float64, device="cuda") / n ** 0.5
    q = 1.0 + torch.rand(n, generator=g, dtype=torch.float64, device="cuda")
    eng = cb.Engine(sp.diags(q.cpu().numpy()).tocsr(), At.t(), None, [("R", m)])
    eng._bind_stream()
    v = torch.rand(m, generator=g, dtype=torch.float64, device="cuda") + 0.5
    s = torch.rand(m, generator=g, dtype=torch.float64, device="cuda") + 0.5
    eng.factor_from_point(v, s)
    rhs = torch.randn(n, generator=g, dtype=torch.float64, device="cuda")
    x = eng.solve_H(rhs)
    # H x = rhs with H = Q + A' diag(v/s) A evaluated independently
    Hx = q * x + At @ ((v / s) * (At.t() @ x))
    err = float(torch.linalg.vector_norm(Hx - rhs) / torch.linalg.vector_norm(rhs))
    x2 = eng.solve_H(rhs)
    for _ in range(5):
        eng.solve_H(rhs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    e0.record()
    for _ in range(reps):
        eng.solve_H(rhs)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    npad = (n + 127) // 128 * 128
    gb = 2 * 8 * npad * (npad + 128) / 2 / 1e9          # lower triangle of L read once per sweep
    print(f"n={n}: residual {err:.2e} deterministic={bool(torch.equal(x, x2))} fwd+bwd {ms*1e3:.1f} us  "
          f"({gb / (ms * 1e-3) / 1e3:.2f} TB/s on the lower triangle of L; {2*8*npad*npad/1e9/(ms*1e-3)/1e3:.2f} TB/s counting the square)", flush=True)
    eng.close()
