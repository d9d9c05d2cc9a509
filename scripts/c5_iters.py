"""C5-shaped LP (R rows + one S(64) block + sparse equalities): iteration counts of the device path with and
without the H + rho G'G augmentation, against the oracle's 29 (kktsolver_qr and kktsolver_chol agree)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import conicip_b200 as cb
from conicip_b200 import problems as P
prob = P.config5(n=2200, k=64, p=60)
for rho in (-1.0, 0.0, 1e-3, 100.0):
    eng = cb.Engine(prob["Q"], prob["A"], prob["G"], prob["cone_dims"], aug_rho=rho)
    s = cb.conicIP_native(prob["Q"], prob["c"], prob["A"], prob["b"], prob["cone_dims"], prob["G"], prob["d"],
                          optTol=1e-8, engine=eng, verbose=(rho == -1.0))
    print("aug_rho", rho, s.status, s.Iter, s.solves, s.pobj, flush=True)
    eng.close()
