"""Time loo() at the C2 and C4 shapes on seeded synthetic histories, one JSON line per (shape, path).

    python tools/loo_bench.py [--reps 3] [--shapes c2,c4] [--out FILE]

The shapes are those of tools/waic_bench.py.  C2: the K3_N1000_P5 data (32 distinct rows), K = 3, 1024 chains x 1800
draws (the long-row regime: a Pareto tail of 4073 draws per row).  C4: 1e7 bit-packed random rows, P = 64, K = 32, one
chain x 90 draws (the many-short-rows regime: a tail of 18 draws).  `kernel_ms` is the device time of the call's kernels
(CUDA events around the tables, the log-likelihood matrix and the PSIS kernels of every chunk, after a warm-up call of the
same shape); `call_ms` is the whole call, host de-duplication and copies included.  The card's name, power limit and
maximum SM clock are read with a read-only nvidia-smi query."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bmm_mcmc_b200 as B  # noqa: E402
from bmm_mcmc_b200 import _lib  # noqa: E402
from tools.waic_bench import card, shape  # noqa: E402


def run(X, fit, no_tensor, reps):
    B.loo(fit, X, no_tensor=no_tensor)                          # warm-up: module load, device buffers
    ks, cs = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = B.loo(fit, X, no_tensor=no_tensor)
        cs.append((time.perf_counter() - t0) * 1e3)
        ms, t = C.c_float(), C.c_int32()
        _lib.check(_lib.lib().bmm_loo_kernel_ms(C.byref(ms), C.byref(t)))
        ks.append(ms.value)
    return r, ("tensor" if t.value else "fp64"), ks, cs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="c2,c4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if _lib.lib().bmm_device_count() < 1:
        sys.exit("loo_bench: no CUDA device")
    info = card()
    lines = []
    for name in a.shapes.split(","):
        X, fit, dims = shape(name)
        res = {}
        for no_tensor in (False, True):
            r, path, ks, cs = run(X, fit, no_tensor, a.reps)
            if path in res:
                continue                                        # the default already took the fp64 kernel
            res[path] = r
            line = dict(shape=name, path=path, default=not no_tensor, **dims, reps=a.reps,
                        kernel_ms=[round(v, 3) for v in ks], call_ms=[round(v, 1) for v in cs],
                        kernel_ms_min=round(min(ks), 3), call_ms_min=round(min(cs), 1),
                        elpd_loo=r["elpd_loo"], p_loo=r["p_loo"], max_pareto_k=float(np.max(r["pareto_k"])),
                        n_k_very_bad=r["n_k_very_bad"], **info)
            lines.append(line)
            print(json.dumps(line), flush=True)
        if len(res) == 2:
            t, f = res["tensor"], res["fp64"]
            fin = np.isfinite(f["pareto_k"])
            line = dict(shape=name, compare="tensor-vs-fp64",
                        max_abs_d_pointwise_elpd_loo=float(np.abs(t["pointwise_elpd_loo"] - f["pointwise_elpd_loo"]).max()),
                        max_abs_d_pointwise_p_loo=float(np.abs(t["pointwise_p_loo"] - f["pointwise_p_loo"]).max()),
                        max_abs_d_pareto_k=float(np.abs(t["pareto_k"][fin] - f["pareto_k"][fin]).max()),
                        rel_d_elpd_loo=abs(t["elpd_loo"] / f["elpd_loo"] - 1), **info)
            lines.append(line)
            print(json.dumps(line), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
