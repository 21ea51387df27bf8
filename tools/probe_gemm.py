#!/usr/bin/env python
"""GPU probe: the batched GEMM alone on BASELINE-shaped problems (f16x2 path), mean device time per launch."""
import json, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cnmf_b200.engine import Engine

eng = Engine(0)
rng = np.random.RandomState(0)
out = {}
for name, (M, N, K, sp) in {"c2_W_half": (1000, 20000, 2000, 1), "c2_H_half": (1000, 2000, 20000, 5),
                            "mid_W_half": (4096, 16384, 2000, 1), "mid_H_half": (4096, 2000, 16384, 4),
                            "tail_H_half": (128, 2000, 20000, 5)}.items():
    A = np.abs(rng.standard_normal((M, K))).astype(np.float32)
    B = rng.poisson(1.5, size=(N, K)).astype(np.float32)
    C, ms = eng.gemm_abt(A, B, precision="f16x2", splits=sp, reps=20)
    ref = A[:64].astype(np.float64) @ B.astype(np.float64).T
    err = float(np.linalg.norm(C[:64] - ref) / np.linalg.norm(ref))
    tail = A[-64:].astype(np.float64) @ B.astype(np.float64).T
    err2 = float(np.linalg.norm(C[-64:] - tail) / np.linalg.norm(tail))
    out[name] = {"ms": round(ms, 4), "tflops": round(2.0 * M * N * K / (ms * 1e-3) / 1e12, 1), "rel_err_first_rows": err, "rel_err_last_rows": err2}
print(json.dumps(out))
