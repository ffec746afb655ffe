#!/usr/bin/env python3
"""Per-phase cycle accounting of the chain-per-block kernels at the C2 shape (gibbs_full, K3_N1000_P5, K = 3,
1024 chains, relabelling with burnin 200 / burnrelabel 50).

Builds libbmm_b200_phases.so -- kern_full.cu compiled with -DBMM_CHAIN_PHASE_CLOCKS, linked with the other objects of
the default build (tools/jobs/build_variant.sh) -- then runs the C2 shape once with full_chain_kernel
(BMM_CHAIN_KERNEL=generic) and once with chain_sweep_kernel, and prints the mean cycles per sweep of every phase on
each warp, averaged over all chains.  A phase's cycles include the wait at the barrier that closes it, except for E and
F, which run side by side on warps 1 and 0: their wait has a row of its own.

    python -m bmm_mcmc_b200.build && python tools/chain_phases.py [--sweeps 600] [--json out.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHASES = ["A log tables", "B row table", "C allocations", "D histogram fold", "E relabelling", "F parameter draws",
          "history write", "wait after E / F"]
NPH, NW, MAXC = 9, 4, 4096


def build_variant():
    subprocess.run(["sh", "tools/jobs/build_variant.sh", "phases", "kern_full.cu", "-DBMM_CHAIN_PHASE_CLOCKS"], cwd=ROOT,
                   check=True, stdout=subprocess.DEVNULL)
    return os.path.join(ROOT, "bmm_mcmc_b200", "libbmm_b200_phases.so")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=600, help="nsamples of the run (burnin 200 of them)")
    ap.add_argument("--chains", type=int, default=1024)
    ap.add_argument("--json", default=None)
    ap.add_argument("--no-build", action="store_true", help="use an existing libbmm_b200_phases.so")
    a = ap.parse_args()
    lib = os.path.join(ROOT, "bmm_mcmc_b200", "libbmm_b200_phases.so") if a.no_build else build_variant()
    os.environ["BMM_LIB"] = lib
    sys.path.insert(0, ROOT)
    import numpy as np
    import bmm_mcmc_b200 as B
    from bmm_mcmc_b200 import _lib
    L = _lib.lib()
    X = B.load_dataset("K3_N1000_P5")
    buf = (C.c_uint64 * (MAXC * NW * NPH))()
    _lib.check(L.bmm_debug_chain_phases(buf, len(buf)))            # clear
    out = {}
    for name, env in (("full_chain_kernel", "generic"), ("chain_sweep_kernel", None)):
        if env:
            os.environ["BMM_CHAIN_KERNEL"] = env
        else:
            os.environ.pop("BMM_CHAIN_KERNEL", None)
        B.gibbs_full(X, a.sweeps, 3, burnin=200, relabel=True, burnrelabel=50, chains=a.chains, seed=2025, compact_z=True)
        picked = L.bmm_debug_chain_kernel()
        _lib.check(L.bmm_debug_chain_phases(buf, len(buf)))
        t = np.frombuffer(buf, dtype=np.uint64).reshape(MAXC, NW, NPH)[:min(a.chains, MAXC)].astype(np.float64)
        sweeps = t[:, :, NPH - 1].sum(0)                          # per warp
        per = t[:, :, :NPH - 1].sum(0) / np.maximum(sweeps, 1)[:, None]
        warps = [w for w in range(NW) if sweeps[w] > 0]
        out[name] = {"kernel_id": int(picked), "sweeps_per_chain": float(sweeps[0] / t.shape[0]),
                     "cycles_per_sweep": {PHASES[ph]: {"warp%d" % w: round(per[w, ph], 1) for w in warps} for ph in range(NPH - 1)},
                     "total_per_sweep": {"warp%d" % w: round(per[w].sum(), 1) for w in warps}}
        print("\n%s (kernel id %d), %d chains, %.0f sweeps per chain: mean cycles per sweep" % (
            name, picked, t.shape[0], sweeps[0] / t.shape[0]))
        print("| phase | " + " | ".join("warp %d" % w for w in warps) + " |")
        print("|---|" + "---:|" * len(warps))
        for ph in range(NPH - 1):
            print("| %s | " % PHASES[ph] + " | ".join("%.0f" % per[w, ph] for w in warps) + " |")
        print("| total | " + " | ".join("%.0f" % per[w].sum() for w in warps) + " |")
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
