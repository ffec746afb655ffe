"""Time waic() at the C2 and C4 shapes on seeded synthetic histories, one JSON line per (shape, path).

    python tools/waic_bench.py [--reps 3] [--shapes c2,c4] [--out FILE]

C2: the K3_N1000_P5 data (32 distinct rows), K = 3, 1024 chains x 1800 draws.  C4: 1e7 bit-packed random rows, P = 64,
K = 32, one chain x 90 draws.  `kernel_ms` is the device time of the call's kernels (CUDA events around tables, WAIC pass
and merge, after a warm-up call of the same shape); `call_ms` is the whole call, host de-duplication and copies included.
The card's name, power limit and maximum SM clock are read with a read-only nvidia-smi query."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bmm_mcmc_b200 as B  # noqa: E402
from bmm_mcmc_b200 import _lib  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = [v.strip() for v in r.stdout.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers are still reported, marked as from an unidentified card
        return {"gpu": "unknown (%s)" % e}


def shape(name):
    rng = np.random.default_rng(20261021)
    if name == "c2":
        X, K, Cn, S = B.load_dataset("K3_N1000_P5"), 3, 1024, 1800
    else:
        X = B.PackedX(rng.integers(0, 2 ** 32, (10_000_000, 2), dtype=np.uint32), 64)
        K, Cn, S = 32, 1, 90
    P = X.shape[1]
    th = rng.uniform(1e-3, 1 - 1e-3, (Cn, K, P, S))
    pi = rng.dirichlet(np.ones(K), (Cn, S))
    fit = {"theta": th, "pi": pi} if Cn > 1 else {"theta": th[0], "pi": pi[0]}
    return X, fit, dict(N=X.shape[0], P=P, K=K, C=Cn, S=S)


def run(X, fit, no_tensor, reps):
    B.waic(fit, X, no_tensor=no_tensor)                         # warm-up: module load, device buffers
    ks, cs = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = B.waic(fit, X, no_tensor=no_tensor)
        cs.append((time.perf_counter() - t0) * 1e3)
        ms, t = C.c_float(), C.c_int32()
        _lib.check(_lib.lib().bmm_waic_kernel_ms(C.byref(ms), C.byref(t)))
        ks.append(ms.value)
    return r, ("tensor" if t.value else "fp64"), ks, cs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="c2,c4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if _lib.lib().bmm_device_count() < 1:
        sys.exit("waic_bench: no CUDA device")
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
                        waic=r["waic"], p_waic=r["p_waic"], **info)
            lines.append(line)
            print(json.dumps(line), flush=True)
        if len(res) == 2:
            t, f = res["tensor"], res["fp64"]
            line = dict(shape=name, compare="tensor-vs-fp64",
                        max_abs_d_pointwise_lppd=float(np.abs(t["pointwise_lppd"] - f["pointwise_lppd"]).max()),
                        max_abs_d_pointwise_p_waic=float(np.abs(t["pointwise_p_waic"] - f["pointwise_p_waic"]).max()),
                        max_rel_d_loglik=float(np.abs(t["loglik"] / f["loglik"] - 1).max()),
                        rel_d_lppd=abs(t["lppd"] / f["lppd"] - 1), rel_d_p_waic=abs(t["p_waic"] / f["p_waic"] - 1), **info)
            lines.append(line)
            print(json.dumps(line), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
