#!/usr/bin/env python3
"""Benchmark of the allocation-sampling hot path (BASELINE.json metric: allocation updates/sec =
N * chains * sweeps / second).

Workload (config[1] of BASELINE.json, "C2"): gibbs_full on the bundled K3_N1000_P5 data, K = 3,
1024 independent chains per GPU, Stephens relabelling on (burnrelabel 50), all histories returned in
the reference's list layout.  One step = one complete run of `nsamples` sweeps for every chain.
  value : device-resident (plan created once, inputs in HBM), timed with CUDA events on the
          launching stream inside the library, max over ranks.
  e2e   : the public call `bmm_mcmc_b200.gibbs_full(...)` = C ABI bmm_gibbs_full with host
          buffers: upload, all sweeps, relabelling, layout conversion, download into pinned host
          memory, every step.
Chains are independent units, so multi-GPU runs split them with no collective ("weak": 1024
chains per GPU).  `--impl reference` times the CPU oracle (the restatement of the reference's
Rcpp samplers + the reference's own lp_solve) on all host cores, one chain per core.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "allocation updates/sec (N*chains*sweeps/s)"

# Chain-parallel workloads (independent chains, split across GPUs with no collective).
# "c2" is BASELINE.json configs[1] and the default; the others are the remaining chain configs.
WORKLOADS = {
    "c2": dict(sampler="full", dataset="K3_N1000_P5", K=3, chains=1024, nsamples=2000, burnin=200, burnrelabel=50,
               relabel=True, label="C2: gibbs_full K3_N1000_P5 (N=1000,P=5) K=3"),
    "collapsed": dict(sampler="collapsed", dataset="K3_N1000_P5", K=3, chains=1024, nsamples=300, burnin=30,
                      burnrelabel=10, relabel=False, label="gibbs_collapsed K3_N1000_P5 (N=1000,P=5) K=3 (north_star 100x target)"),
    "c1": dict(sampler="collapsed", dataset="K2_N100_P5", K=2, chains=1, nsamples=10000, burnin=1000,
               burnrelabel=50, relabel=False, label="C1: gibbs_collapsed K2_N100_P5 (N=100,P=5) K=2, 1 chain, 10k iters"),
    "c3": dict(sampler="dp", dataset="K2_N1000_P5", K=64, chains=4096, nsamples=300, burnin=30, burnrelabel=10,
               relabel=False, label="C3: gibbs_dp K2_N1000_P5 (N=1000,P=5) maxK=64"),
}
WL = WORKLOADS["c2"]
DATASET, K = WL["dataset"], WL["K"]
CHAINS_PER_GPU = WL["chains"]
NSAMPLES, BURNIN, BURNRELABEL = WL["nsamples"], WL["burnin"], WL["burnrelabel"]


def select_workload(name):
    global WL, DATASET, K, CHAINS_PER_GPU, NSAMPLES, BURNIN, BURNRELABEL
    WL = WORKLOADS[name]
    DATASET, K = WL["dataset"], WL["K"]
    CHAINS_PER_GPU = WL["chains"]
    NSAMPLES, BURNIN, BURNRELABEL = WL["nsamples"], WL["burnin"], WL["burnrelabel"]


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []
        self.t0 = self.t1 = None

    def launch(self):
        """Start nvidia-smi (it needs a few hundred ms to come up: call before the warm-up)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def start(self):
        """Open the timed window; only samples that arrive inside it are reported."""
        if self.proc is None:
            self.launch()
        self.t0 = time.perf_counter()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        self.t1 = time.perf_counter()
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        inside = [ln for (t, ln) in self.lines if self.t0 <= t <= self.t1 + 0.03]
        if not inside and self.lines:      # a timed region shorter than one sampling period: the nearest sample
            inside = [min(self.lines, key=lambda x: abs(x[0] - self.t1))[1]]
        sm, mx, reasons = [], None, set()
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def init_states(chains, P, seed):
    """Initial pi / theta exactly as R/utils.R:68-74 draws them (R-compatible Mersenne-Twister)."""
    from bmm_mcmc_b200.rcompat import RRng
    rng = RRng(seed)
    u = rng.runif(chains * (K + K * P)).reshape(chains, K + K * P)
    ip = np.exp(u[:, :K]); ip /= ip.sum(1, keepdims=True)
    th = u[:, K:].reshape(chains, P, K)
    return np.ascontiguousarray(ip), np.ascontiguousarray(th)


def cpu_kind():
    """'reference' when oracle/_ref/libbmm_ref.so (the reference's own src/*.cpp, compiled unmodified against the
    header shim, oracle/build_ref.sh) is present, else 'port' (the oracle restatement)."""
    try:
        from oracle import pyref
        return "reference" if pyref.available() else "port"
    except Exception:
        return "port"


def cpu_chain(args):
    """One CPU chain of the bench workload through the reference's own compiled sampler (its registered .Call
    symbol) -- or the oracle port when that library is absent; returns (updates, seconds)."""
    seed, nsamples, burnin, br = args
    import bmm_mcmc_b200 as B
    from bmm_mcmc_b200.rcompat import RRng
    X = B.load_dataset(DATASET)
    N, P = X.shape
    ref = cpu_kind() == "reference"
    if ref:
        from oracle import pyref as R
        R.lib()
    else:
        from oracle import pyoracle as O
        kw = dict(burnin=burnin, relabel=WL["relabel"], burnrelabel=br, seed=seed, use_ref=O.has_ref(), probes=False)
    rel = WL["relabel"]
    if WL["sampler"] == "full":
        ip, th = init_states(1, P, 1000 + seed)
        t0 = time.perf_counter()
        if ref:
            R.gibbs_cpp(X, ip[0], th[0].T, nsamples, K, 0.0, 0.5, 0.5, 1.0, 1.0, burnin, rel, br, seed=seed)
        else:
            O.gibbs_full(X, ip[0], th[0].T, nsamples, K, **kw)
    elif WL["sampler"] == "collapsed":
        iz = RRng(1000 + seed).sample_int(K, N)
        t0 = time.perf_counter()
        if ref:
            R.collapsed_gibbs_cpp(X, iz, nsamples, K, 0.0, 0.5, 0.5, 1.0, 1.0, burnin, rel, br, seed=seed)
        else:
            O.gibbs_collapsed(X, iz, nsamples, K, **kw)
    else:
        t0 = time.perf_counter()
        if ref:
            R.collapsed_gibbs_dp_cpp(X, nsamples, 0.0, 0.5, 0.5, 1.0, 1.0, burnin, rel, br, K, seed=seed)
        else:
            O.gibbs_dp(X, nsamples, maxK=K, **kw)
    return N * (nsamples - 1), time.perf_counter() - t0


CPU_NOTE = {
    "reference": "the reference's own src/*.cpp compiled unmodified (g++ -O2, R's default level) against a header-only "
                 "Rcpp/Armadillo stand-in, called through its registered .Call symbol, console output sunk",
    "port": "oracle/oracle.cpp, the line-faithful restatement (compiled reference library absent)",
}


def cpu_sample_shape():
    """Sweeps of one CPU sample chain: the workload's own, capped so one chain stays within seconds
    (the collapsed reference is O(N^2 P) per sweep; per-update cost does not depend on the sweep count)."""
    ns = NSAMPLES if WL["sampler"] == "full" else min(NSAMPLES, 120)
    burnin = min(BURNIN, max(2, ns // 10))
    return ns, burnin, min(BURNRELABEL, burnin)


def cpu_baseline_single(budget_s=12.0):
    """Oracle on one host core, bounded sample of the same workload."""
    ns, burnin, br = cpu_sample_shape()
    upd, sec, chains = 0, 0.0, 0
    while sec < budget_s and chains < 16:
        u, s = cpu_chain((chains, ns, burnin, br))
        upd += u; sec += s; chains += 1
    return {"value": upd / sec, "unit": "allocation updates/s", "cores": 1,
            "kind": cpu_kind(), "assignment": "reference lp_solve",
            "sample": "%d chain(s) x %d sweeps of %s, relabel=%s burnrelabel=%d, %.1f s; %s"
                      % (chains, ns - 1, WL["label"], WL["relabel"], br, sec, CPU_NOTE[cpu_kind()])}


def run_reference(a):
    """--impl reference: the CPU oracle on all host cores (one chain per core per step)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    select_workload(a.workload)
    ns, burnin, br = cpu_sample_shape()
    kind = cpu_kind()
    if kind == "reference":
        from oracle import pyref
        pyref.lib()
    else:
        from oracle import pyoracle as O
        O.lib()
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(cores) as pool:
        for step in range(a.warmup + a.steps):
            t0 = time.perf_counter()
            res = pool.map(cpu_chain, [(step * cores + c, ns, burnin, br) for c in range(cores)])
            dt = time.perf_counter() - t0
            if step >= a.warmup:
                times.append((sum(r[0] for r in res), dt))
    upd = sum(t[0] for t in times); sec = sum(t[1] for t in times)
    val = upd / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "allocation updates/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * sec / max(a.steps, 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "bundled %s (regenerated from set.seed(17))" % DATASET,
        "config": {"workload": "%s, relabel=%s burnrelabel=%d; CPU sample: %d chains x %d sweeps per step"
                               % (WL["label"], WL["relabel"], br, cores, ns - 1)},
        "cpu_baseline": {"value": val, "unit": "allocation updates/s", "cores": cores,
                         "kind": kind, "assignment": "reference lp_solve",
                         "sample": "one chain per core, %d cores x %d sweeps per step (the reference is single-threaded); %s"
                                   % (cores, ns - 1, CPU_NOTE[kind])},
        "e2e": {"value": val, "unit": "allocation updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---- grid workloads: one uncollapsed chain over many observations, N-sharded across GPUs ----------
GRID_WORKLOADS = {
    # BASELINE.json configs[3]: strong scaling, total N fixed, counts all-reduced every sweep
    "c4": dict(sampler="stickbreaking", N=10_000_000, P=64, K=32, nsamples=101, burnin=11, alpha=1.0,
               precision="fp32", cpu_N=60_000, cpu_ns=6,
               label="C4: gibbs_stickbreaking synthetic N=1e7 P=64 maxK=32, alpha=1"),
    # the same with online Stephens relabelling after the burn-in (SURVEY 8d: "relabel off and on")
    "c4relabel": dict(sampler="stickbreaking", N=10_000_000, P=64, K=32, nsamples=41, burnin=5, alpha=1.0, relabel=True,
                      burnrelabel=1, precision="fp32", cpu_N=60_000, cpu_ns=6,
                      label="C4 + Stephens relabelling: gibbs_stickbreaking synthetic N=1e7 P=64 maxK=32, alpha=1"),
    # BASELINE.json configs[4]
    "c5": dict(sampler="full", N=1_000_000, P=4096, K=128, nsamples=41, burnin=5, alpha=1.0, relabel=True, burnrelabel=1,
               precision="fp32", cpu_N=150, cpu_ns=3, stabilise=True,
               label="C5: gibbs_full synthetic N=1e6 P=4096 K=128 (large-P tcgen05 contraction) + Stephens relabelling (Hungarian)"),
    "c5small": dict(sampler="full", N=100_000, P=4096, K=128, nsamples=21, burnin=5, alpha=1.0, relabel=True, burnrelabel=1,
                    precision="fp32", cpu_N=150, cpu_ns=3, stabilise=True,
                    label="C5 shape at N=1e5 (smoke size) + relabelling"),
    "c5norelabel": dict(sampler="full", N=1_000_000, P=4096, K=128, nsamples=21, burnin=3, alpha=1.0,
                        precision="fp32", cpu_N=150, cpu_ns=3, stabilise=True,
                        label="C5 shape, relabel=FALSE (sweep kernels only)"),
    "c4small": dict(sampler="stickbreaking", N=1_000_000, P=64, K=32, nsamples=21, burnin=3, alpha=1.0,
                    precision="fp32", cpu_N=20_000, cpu_ns=4,
                    label="C4 shape at N=1e6 (smoke size)"),
}


def synth_rows(lo, hi, P, K_true, seed=17, chunk=None):
    """Rows [lo, hi) of the synthetic data set (SURVEY 8d): pi* uniform, theta* ~ U(0.1, 0.9),
    x_id ~ Bernoulli(theta*[z*_i, d]); generated chunk by chunk so any shard sees the same rows."""
    from bmm_mcmc_b200 import PackedX
    chunk = chunk or (500_000 if P <= 64 else 16_384)
    th = np.random.default_rng([seed, 0]).uniform(0.1, 0.9, (K_true, P)).astype(np.float32)
    thq = np.clip(np.round(th * 256.0), 1, 255).astype(np.uint8)      # 8-bit thresholds, 1 B of randomness per bit
    W = (P + 31) // 32
    out = np.zeros((hi - lo, W), dtype=np.uint32)
    c0 = lo // chunk
    while c0 * chunk < hi:
        a0, a1 = c0 * chunk, (c0 + 1) * chunk
        rng = np.random.default_rng([seed, 1 + c0])
        z = rng.integers(0, K_true, chunk)
        x = rng.integers(0, 256, (chunk, P), dtype=np.uint8) < thq[z]
        s0, s1 = max(a0, lo), min(a1, hi)
        out[s0 - lo:s1 - lo] = PackedX.pack(x[s0 - a0:s1 - a0]).bits
        c0 += 1
    return PackedX(out, P)


def grid_init(K, P):
    from bmm_mcmc_b200.rcompat import RRng
    rng = RRng(1)
    ip = np.exp(rng.runif(K)); ip /= ip.sum()                  # R/utils.R:98-100
    th = rng.runif(K * P).reshape(P, K)                        # matrix(runif(K*P), nrow=K), column-major
    return np.ascontiguousarray(ip[None]), np.ascontiguousarray(th[None])


def grid_cpu_baseline(w):
    """One reduced CPU chain of a grid workload: the compiled reference where it can run the shape (C4), the
    oracle port with a stabilised softmax where the reference underflows to NaN (C5, SURVEY App. D quirk 13)."""
    N, ns, K, P = w["cpu_N"], w["cpu_ns"], w["K"], w["P"]
    X = synth_rows(0, N, P, K)
    Xi = ((X.bits[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(N, -1)[:, :P].astype(np.int32)
    ip, th = grid_init(K, P)
    kind = "port" if w.get("stabilise") else cpu_kind()
    if kind == "reference":
        from oracle import pyref as R
        f = R.gibbs_stickbreaking_cpp if w["sampler"] == "stickbreaking" else R.gibbs_cpp
        R.lib()
        t0 = time.perf_counter()
        f(Xi, ip[0], th[0].T, ns, K, w["alpha"], 0.5, 0.5, 1.0, 1.0, 1, False, 1, seed=3)
    else:
        from oracle import pyoracle as O
        f = O.gibbs_stickbreaking if w["sampler"] == "stickbreaking" else O.gibbs_full
        t0 = time.perf_counter()
        f(Xi, ip[0], th[0].T, ns, K, alpha=w["alpha"], burnin=1, seed=3, probes=False, **({"stabilise": True} if w.get("stabilise") else {}))
    sec = time.perf_counter() - t0
    return {"value": N * (ns - 1) / sec, "unit": "allocation updates/s", "cores": 1, "kind": kind,
            "sample": "%s reduced to N=%d, %d sweeps (the reference's N x K x nsamples double cube cannot hold N=%g; "
                      "per-update cost of the uncollapsed sampler does not depend on N), %.1f s; %s"
                      % (w["label"], N, ns - 1, w["N"], sec, CPU_NOTE[kind])}, sec


def run_grid_reference(a):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    import multiprocessing as mp
    w = GRID_WORKLOADS[a.workload]
    cores = os.cpu_count() or 1
    kind = "port" if w.get("stabilise") else cpu_kind()
    ctx = mp.get_context("fork")
    tot_u, tot_s = 0, 0.0
    with ctx.Pool(cores) as pool:
        for step in range(a.warmup + a.steps):
            t0 = time.perf_counter()
            pool.map(grid_cpu_baseline, [w] * cores)
            dt = time.perf_counter() - t0
            if step >= a.warmup:
                tot_u += cores * w["cpu_N"] * (w["cpu_ns"] - 1); tot_s += dt
    val = tot_u / tot_s
    sample = "one independent reduced chain per core: %d cores x N=%d x %d sweeps per step" % (cores, w["cpu_N"], w["cpu_ns"] - 1)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "allocation updates/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot_s / max(a.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic (seed 17)",
        "config": {"workload": w["label"] + "; CPU sample: " + sample},
        "cpu_baseline": {"value": val, "unit": "allocation updates/s", "cores": cores, "kind": kind,
                         "sample": sample + "; " + CPU_NOTE[kind]},
        "e2e": {"value": val, "unit": "allocation updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))
    return 0


def run_grid(a):
    w = dict(GRID_WORKLOADS[a.workload])
    if a.nsamples:
        w["nsamples"] = a.nsamples
    if a.n:
        w["N"] = a.n
    if a.precision:
        w["precision"] = a.precision
    rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import bmm_mcmc_b200 as B
    from bmm_mcmc_b200 import _lib, api, dist as bdist
    L = _lib.lib()
    assert L.bmm_device_count() > local, "no CUDA device: the product path has no CPU fallback"
    p2p = bdist.init(rank, world, local)
    N, P, K, ns, burnin = w["N"], w["P"], w["K"], w["nsamples"], w["burnin"]
    lo, hi = bdist.shard_rows(N, world, rank)
    X = synth_rows(lo, hi, P, K)
    ip, th = grid_init(K, P)
    sid = _lib.SAMPLER_STICKBREAKING if w["sampler"] == "stickbreaking" else _lib.SAMPLER_FULL
    kname = "big_sweep_ws_kernel" if (K <= 32 and P <= 112) else "lp_table + lp_sweep + cnt_* kernels"
    tkey = "big_sweep_ws_kernel" if (K <= 32 and P <= 112) else "lp_sweep_kernel"
    shard = dict(n_global=N, row_offset=lo) if world > 1 else {}
    relabel, br = bool(w.get("relabel")), int(w.get("burnrelabel", 0))
    kw = dict(alpha=w["alpha"], beta=0.5, gamma=0.5, a=1.0, b=1.0, burnin=burnin, relabel=relabel, burnrelabel=br)

    def barrier():
        if dist:
            dist.barrier()

    plan = api.Plan(sid, X, ns, K, chains=1, seed=2026, device=local, init_pi=ip, init_theta=th,
                    precision=w["precision"], compact_z=True, grid_path=True, **shard, **kw)
    clocks = ClockSampler(local)
    clocks.launch()
    for _ in range(a.warmup):
        plan.run(); plan.sync()
    barrier(); plan.sync()
    clocks.start()
    l0 = L.bmm_launch_count()
    t0 = time.perf_counter()
    dev_ms, kern = 0.0, np.zeros(4)
    for _ in range(a.steps):
        plan.run(); plan.sync()
        dev_ms += plan.elapsed_ms()[0]
        kern += np.array(plan.kernel_ms())
    plan.sync(); barrier()
    wall_s = time.perf_counter() - t0
    launches = int(L.bmm_launch_count() - l0)
    clk = clocks.stop()
    plan.check()      # a chain that stopped with an error status invalidates the timing
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, plan.fetch())
    plan.close()

    # e2e: the public call with host buffers (bit-packed rows in, uint8 allocation history out)
    bufs = api._alloc_out(sid, 1, hi - lo, P, K, ns, burnin, relabel, True, (), True)
    d2h = api.out_nbytes(bufs[0])
    h2d = X.nbytes + ip.nbytes + th.nbytes
    fn = B.gibbs_stickbreaking if w["sampler"] == "stickbreaking" else B.gibbs_full

    def e2e_step():
        return fn(X, ns, K, alpha=w["alpha"], burnin=burnin, seed=2026, device=local, initial_pi=ip,
                  initial_theta=th.transpose(0, 2, 1), precision=w["precision"], compact_z=True, grid_path=True,
                  relabel=relabel, burnrelabel=br, out_bufs=bufs, **shard)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        r = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    assert 1 <= int(r["z"][-1].max()) <= K

    tm = np.array([dev_ms / 1e3, wall_s, e2e_s])
    if dist:
        import torch
        t = torch.tensor(tm, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tm = t.cpu().numpy()
    total_updates = N * (ns - 1) * a.steps
    pk, pk_src = peaks()
    n_local = hi - lo
    bytes_per_update = (P + 7) // 8 + 1
    dur_s = kern[0] / a.steps / (ns - 1) / 1e3
    achieved = n_local * bytes_per_update / dur_s / 1e9
    traffic = None   # dram bytes of the dominant kernel's launch from the committed ncu --set full capture (same rows per GPU)
    ncu_pipes = None  # ... and its issue-slot / MUFU / tensor-pipe utilisation from the same capture
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f).get(tkey, {})
        if not tr:
            with open(os.path.join(ROOT, "profiles", "r01_traffic.json")) as f:
                tr = json.load(f).get(tkey, {})
        if tr.get("n") == n_local and tr.get("dram_bytes_read") is not None:
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            ncu_pipes = tr.get("ncu")
    except Exception:
        pass
    roof = {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "peak_source": pk_src,
            "kernel": "%s (%d rows, %d B/update)" % (kname, n_local, bytes_per_update),
            "kernel_ms": dur_s * 1e3, "kernel_share_of_step": float(kern[0] / max(kern[:3].sum() + kern[3], 1e-9))}
    if ncu_pipes:
        roof["ncu"] = ncu_pipes
    if relabel and kern[2] > 0:
        # with relabelling the dominant kernel is the single-pass relabelling kernel: Q once in, once out (fp32) plus the
        # packed row per update (SURVEY 8d: 2*K*4 + ceil(P/8) bytes), HBM-bound
        rb = 2 * K * 4 + (P + 7) // 8
        rdur = kern[2] / a.steps / (ns - burnin) / 1e3
        racc = n_local * rb / rdur / 1e9
        rtraffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                tr = json.load(f).get("big_relabel_ws_kernel", {})
            if tr.get("n") == n_local:
                rtraffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
                ncu_pipes = tr.get("ncu")
        except Exception:
            pass
        roof = {"bound": "hbm", "achieved": racc, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": racc / pk["hbm_gbs"],
                "traffic": rtraffic, "peak_source": pk_src,
                "kernel": "big_relabel_ws_kernel (%d rows, %d B/update: Q read + Q written in fp32, packed row)" % (n_local, rb),
                "kernel_ms": rdur * 1e3, "kernel_share_of_step": float(kern[2] / max(kern[:3].sum() + kern[3], 1e-9)),
                "sweep_kernel_ms": dur_s * 1e3}
        if ncu_pipes:
            roof["ncu"] = ncu_pipes
    elif 2 * K * P / bytes_per_update > 1e3 * pk["bf16_tflops_sustained"] / pk["hbm_gbs"]:
        # arithmetic intensity above the ridge (C5: 2044 flop/B vs 216): the tensor pipe bounds it
        flops = 2.0 * K * P * n_local          # algorithmic: one K x P contraction per update (SURVEY 8d)
        tf = flops / dur_s / 1e12
        roof.update(bound="tensor", achieved=tf, peak=pk["bf16_tflops_sustained"], unit="TFLOP/s",
                    frac=tf / pk["bf16_tflops_sustained"],
                    kernel="%s (%d rows, %d algorithmic flop/update; the kernel issues 2x that: D = hi + lo in fp16)"
                           % (kname, n_local, 2 * K * P))
    line = {
        "metric": METRIC, "value": total_updates / tm[0], "unit": "allocation updates/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tm[0] / a.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32" if w["precision"] == "fp32" else "f64",
        "data": "synthetic (seed 17): pi* uniform, theta* ~ U(0.1,0.9), bit-packed rows",
        "config": {"workload": "%s, nsamples=%d (one step = %d sweeps), relabel=%s burnrelabel=%d"
                               % (w["label"], ns, ns - 1, relabel, br),
                   "N": N, "rows_per_gpu": n_local,
                   "parallelism": ("rows block-partitioned over GPUs; int32 counts all-reduced every sweep by %s"
                                   % ("a one-shot push over IPC-mapped NVLink peer memory" if p2p else "NCCL"))
                                  if world > 1 else "single GPU",
                   "l2": "per-sweep input (%.0f MB of packed rows + allocations) vs 126 MB L2; sweeps alternate "
                         "history rows" % (n_local * bytes_per_update / 1e6)},
        "clocks": clk,
        "e2e": {"value": total_updates / tm[2], "unit": "allocation updates/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * tm[2] / a.steps,
                "api": "bmm_mcmc_b200.gibbs_%s(PackedX, ...) -> bmm_gibbs_%s (C ABI), pinned host output buffers"
                       % (w["sampler"], w["sampler"])},
        "gpu_launches": launches,
        "roofline": roof,
        "extra": {"wall_ms_per_step": 1e3 * tm[1] / a.steps,
                  "kernels_ms": {"sweep_kernels": kern[0] / a.steps, "relabel_kernels": kern[2] / a.steps,
                                 "params_allreduce_assign_other": kern[1] / a.steps, "finalize_layout": kern[3] / a.steps}},
    }
    if rank == 0 and world == 1 and not a.no_cpu:
        line["cpu_baseline"] = grid_cpu_baseline(w)[0]
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line))
    bdist.finalize()
    if dist:
        dist.destroy_process_group()
    return 0


DUMP_LIMIT = 64 * 10 ** 6


def dump_outputs(dirname, res):
    """--dump-outputs: the arrays a caller of the timed path receives from its last step, one DIR/<name>.npy each, in the
    returned layout (float64 as computed, integer arrays as float32, which holds labels exactly).  When together they
    exceed 64 MB, every array keeps the same fraction of its elements, taken at seeded positions that depend only on
    the array's name and shape: element i of the file is element idx[i] of the row-major flattened array, idx sorted.
    Two builds run with the same arguments therefore write files that compare element for element."""
    import zlib
    os.makedirs(dirname, exist_ok=True)
    res = {k: np.asarray(v) for k, v in res.items()}
    size = lambda v: v.size * (8 if v.dtype == np.float64 else 4)
    total = sum(size(v) for v in res.values())
    frac = min(1.0, (DUMP_LIMIT - 4096 * len(res)) / max(total, 1))       # 4 KB per file for the .npy header
    for name, v in sorted(res.items()):
        if frac < 1.0:
            m = max(1, int(v.size * frac))
            idx = np.sort(np.random.default_rng([zlib.crc32(name.encode()), *v.shape]).choice(v.size, m, replace=False))
            v = v[np.unravel_index(idx, v.shape)]
        np.save(os.path.join(dirname, name + ".npy"), v.astype(np.float64 if v.dtype == np.float64 else np.float32))
    print("bench: wrote %d arrays to %s (%s of every array)" % (len(res), dirname, "all" if frac == 1.0 else "%.3g" % frac),
          file=sys.stderr)


def _max_over_ranks(x, dist):
    if not dist:
        return x
    import torch
    t = torch.tensor([float(x)], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def ncu_record(key, n_rows):
    """Issue-slot / MUFU / tensor-pipe utilisation and DRAM bytes of one launch of `key` from the committed ncu --set full
    capture (profiles/r02_traffic.json), when it was taken at this many rows per GPU; else None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f).get(key, {})
        if tr.get("n") == n_rows and tr.get("ncu"):
            return dict(tr["ncu"], dram_bytes=tr["dram_bytes_read"] + tr["dram_bytes_write"], source=tr.get("source"))
    except Exception:
        pass
    return None


def sharded_leg(rank, world, local, dist, steps=3, warmup=2):
    """The path that communicates (BASELINE configs[3], north_star's multi-GPU deliverable): ONE stick-breaking chain
    over N = 1e7 observations, rows block-partitioned over the ranks, per-sweep count exchange (stickbreaking.cpp:164-194
    counts summed over ranks).  Short runs, relabelling off and on; device-timed, max over ranks."""
    from bmm_mcmc_b200 import _lib, api, dist as bdist
    L = _lib.lib()
    w = GRID_WORKLOADS["c4"]
    N, P, K = w["N"], w["P"], w["K"]
    p2p = bdist.init(rank, world, local)
    lo, hi = bdist.shard_rows(N, world, rank)
    X = synth_rows(lo, hi, P, K)
    ip, th = grid_init(K, P)
    shard = dict(n_global=N, row_offset=lo) if world > 1 else {}
    pk, _ = peaks()
    out = {"workload": "C4: gibbs_stickbreaking synthetic N=1e7 P=64 maxK=32, alpha=1, rows sharded over %d GPU(s)" % world,
           "rows_per_gpu": hi - lo, "scaling": "strong",
           "exchange": ("tagged 8-byte words pushed over IPC-mapped NVLink peer memory by the sweep kernel's last CTA, "
                        "summed by the parameter-update kernel" if p2p else ("NCCL all-reduce" if world > 1 else "none (one GPU)")),
           "comm_nranks": world}
    for name, ns, burnin, relabel, br in (("relabel_off", 31, 1, False, 0), ("relabel_on", 62, 2, True, 1)):
        plan = api.Plan(_lib.SAMPLER_STICKBREAKING, X, ns, K, chains=1, seed=2026, device=local, init_pi=ip, init_theta=th,
                        precision="fp32", compact_z=True, grid_path=True, alpha=w["alpha"], beta=0.5, gamma=0.5, a=1.0, b=1.0,
                        burnin=burnin, relabel=relabel, burnrelabel=br, **shard)
        clocks = ClockSampler(local)
        clocks.launch()
        t_w = 0.0
        for _ in range(warmup):
            plan.run(); plan.sync()
            t_w = plan.elapsed_ms()[0]
        # at 8 GPUs a step lasts a few milliseconds: repeat it until the timed region covers ~1.5 s, so that the clock
        # sampler (one nvidia-smi query per ~0.2 s) sees it; every rank derives the same count from the max step time
        t_w = _max_over_ranks(t_w, dist)
        nrep = int(min(400, max(steps, np.ceil(1500.0 / max(t_w, 1e-3)))))
        if dist:
            dist.barrier()
        clocks.start()
        l0 = L.bmm_launch_count()
        dev_ms, kern = 0.0, np.zeros(4)
        for _ in range(nrep):
            plan.run(); plan.sync()
            dev_ms += plan.elapsed_ms()[0]
            kern += np.array(plan.kernel_ms())
        if dist:
            dist.barrier()
        clk = clocks.stop()
        launches = int(L.bmm_launch_count() - l0)
        plan.check()
        plan.close()
        dev_ms = _max_over_ranks(dev_ms, dist)
        sweeps = (ns - 1) * nrep
        sweep_us = 1e3 * kern[0] / sweeps
        other_us = 1e3 * (kern[1]) / sweeps
        relabel_us = 1e3 * kern[2] / ((ns - burnin) * nrep) if relabel else 0.0
        n_local = hi - lo
        bytes_upd = (P + 7) // 8 + 1 + (2 * K * 4 if relabel else 0)       # SURVEY 8d: X row + z (+ Q read and write)
        out[name] = {
            "value": N * sweeps / (dev_ms / 1e3), "unit": "allocation updates/s", "nsamples": ns, "burnin": burnin,
            "steps": nrep, "ms_per_sweep": dev_ms / sweeps, "sweep_kernel_us": sweep_us,
            "exchange_us": other_us, "exchange_note": "everything of a sweep that is neither the z-sweep kernel nor the relabelling "
            "kernel: count exchange + parameter update" + (" + cost all-reduce, assignment, batch initialisation of Q (amortised)"
                                                          if relabel else "") + ", per sweep, this rank",
            "relabel_kernel_us": relabel_us,
            "hbm_frac": n_local * bytes_upd / (dev_ms / 1e3 / sweeps) / 1e9 / pk["hbm_gbs"],
            "hbm_bytes_per_update": bytes_upd,
            "tensor_frac": 2.0 * K * P * n_local / (sweep_us * 1e-6) / 1e12 / pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
            "gpu_launches": launches, "clocks": clk}
        rec = ncu_record("big_relabel_ws_kernel" if relabel else "big_sweep_ws_kernel", n_local)
        if rec:
            out[name]["ncu_dominant_kernel"] = rec
    bdist.finalize()
    return out


def collapsed_leg(rank, world, local, dist, steps=3, warmup=2):
    """north_star's >= 100x target workload: gibbs_collapsed on K3_N1000_P5, 1024 chains per GPU, device-timed."""
    import bmm_mcmc_b200 as B
    from bmm_mcmc_b200 import _lib, api
    from bmm_mcmc_b200.rcompat import RRng
    w = WORKLOADS["collapsed"]
    X = B.load_dataset(w["dataset"])
    N, P = X.shape
    Kc, C_, ns, burnin = w["K"], w["chains"], w["nsamples"], w["burnin"]
    iz = np.ascontiguousarray(np.random.default_rng(1 + rank).integers(1, Kc + 1, (C_, N)), dtype=np.int32)
    iz[0] = RRng(1 + rank).sample_int(Kc, N)
    plan = api.Plan(_lib.SAMPLER_COLLAPSED, X, ns, Kc, chains=C_, seed=2026, device=local, chain_offset=rank * C_, init_z=iz,
                    alpha=0.0, beta=0.5, gamma=0.5, a=1.0, b=1.0, burnin=burnin, relabel=False, burnrelabel=w["burnrelabel"])
    for _ in range(warmup):
        plan.run(); plan.sync()
    if dist:
        dist.barrier()
    dev_ms = 0.0
    for _ in range(steps):
        plan.run(); plan.sync()
        dev_ms += plan.elapsed_ms()[0]
    plan.check()
    plan.close()
    dev_ms = _max_over_ranks(dev_ms, dist)
    val = N * C_ * (ns - 1) * steps * world / (dev_ms / 1e3)
    out = {"workload": "%s, %d chains/GPU, nsamples=%d" % (w["label"], C_, ns), "value": val, "unit": "allocation updates/s",
           "ms_per_step": dev_ms / steps, "scaling": "weak"}
    if rank == 0 and world == 1:
        global WL, DATASET, K, NSAMPLES, BURNIN, BURNRELABEL
        keep = (WL, DATASET, K, NSAMPLES, BURNIN, BURNRELABEL)
        select_workload("collapsed")
        cpu = cpu_baseline_single(budget_s=6.0)
        WL, DATASET, K, NSAMPLES, BURNIN, BURNRELABEL = keep
        out["cpu_baseline"] = cpu
        out["ratio_vs_one_cpu_core"] = val / cpu["value"]
        out["ratio_vs_all_host_cores_ideal"] = val / (cpu["value"] * (os.cpu_count() or 1))
        try:        # SURVEY 8a5: "most of the >= 100x target is algorithmic" -- the count-maintaining sampler on the host cores
            from oracle import pyoracle as O
            cores = os.cpu_count() or 1
            O.opt_cpu_collapsed_gibbs(X, Kc, 20, cores, cores)
            s1 = O.opt_cpu_collapsed_gibbs(X, Kc, ns, 4, 1)
            chains = 16 * cores
            sa = O.opt_cpu_collapsed_gibbs(X, Kc, ns, chains, cores)
            one, allc = N * (ns - 1) * 4 / s1, N * (ns - 1) * chains / sa
            out["cpu_optimised"] = {"value": allc, "unit": "allocation updates/s", "cores": cores, "one_core": one, "kind": "port-optimised",
                                    "sample": "%d chains x %d sweeps on %d threads (%.2f s): counts maintained, product-form conditional, "
                                              "fixed alpha, byte-wide history (oracle/opt_cpu.cpp)" % (chains, ns - 1, cores, sa),
                                    "algorithmic_gain_per_core": one / cpu["value"], "gpu_over_all_cores": val / allc}
        except Exception as e:
            out["cpu_optimised"] = {"unavailable": repr(e)[:200]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS) + sorted(GRID_WORKLOADS))
    ap.add_argument("--n", type=int, default=None, help="grid workloads: override N")
    ap.add_argument("--precision", default=None, choices=["fp32", "fp64"])
    ap.add_argument("--chains", type=int, default=None)
    ap.add_argument("--nsamples", type=int, default=None)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip extra.sharded / extra.collapsed_1024 on the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step as DIR/<name>.npy (rank 0; sampled to 64 MB "
                         "after fetching the whole list into host memory, 15 GB at the C2 size)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm only times the CPU oracle")
    if a.workload in GRID_WORKLOADS:
        if a.impl == "reference":
            return run_grid_reference(a)
        a.warmup = max(a.warmup, 3)
        return run_grid(a)
    if a.impl == "reference":
        return run_reference(a)
    a.warmup = max(a.warmup, 3)
    select_workload(a.workload)
    a.chains = a.chains or CHAINS_PER_GPU
    a.nsamples = a.nsamples or NSAMPLES

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import bmm_mcmc_b200 as B
    from bmm_mcmc_b200 import _lib, api
    L = _lib.lib()
    assert L.bmm_device_count() > local, "no CUDA device: the product path has no CPU fallback"
    X = B.load_dataset(DATASET)
    N, P = X.shape
    C_, ns = a.chains, a.nsamples
    burnin = BURNIN if ns > 2 * BURNIN else max(2, ns // 10)
    br = min(BURNRELABEL, burnin)
    relabel = WL["relabel"]
    S = ns - burnin
    smp = WL["sampler"]
    sid = {"full": _lib.SAMPLER_FULL, "collapsed": _lib.SAMPLER_COLLAPSED, "dp": _lib.SAMPLER_DP}[smp]
    kw = dict(alpha=0.0, beta=0.5, gamma=0.5, a=1.0, b=1.0, burnin=burnin, relabel=relabel, burnrelabel=br)
    updates_per_step = N * C_ * (ns - 1)
    init_kw, h2d = {}, X.nbytes
    if smp == "full":
        ip, th = init_states(C_, P, 1 + rank)
        init_kw = dict(init_pi=ip, init_theta=th)
        h2d += ip.nbytes + th.nbytes
    elif smp == "collapsed":
        from bmm_mcmc_b200.rcompat import RRng
        iz = np.ascontiguousarray(np.random.default_rng(1 + rank).integers(1, K + 1, (C_, N)), dtype=np.int32)
        iz[0] = RRng(1 + rank).sample_int(K, N)   # chain 0 exactly as R/utils.R:42 draws it
        init_kw = dict(init_z=iz)
        h2d += iz.nbytes

    def barrier():
        if dist:
            dist.barrier()

    # The e2e arm, and --dump-outputs before it, receive the reference's list layout: S x N int32 allocation matrices,
    # 15 GB per rank at the C2 size -- never drive the box out of memory for it; checked before anything is allocated
    need = (2 if relabel else 1) * C_ * S * N * 4 * int(os.environ.get("LOCAL_WORLD_SIZE", world))
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = None
    if avail is not None and need > 0.8 * avail:
        raise SystemExit("bench: the e2e leg needs %.0f GB of host memory for the returned histories, %.0f GB available"
                         % (need / 1e9, avail / 1e9))

    # ---- device-resident arm (value) --------------------------------------------------------
    plan = api.Plan(sid, X, ns, K, chains=C_, seed=2026, device=local, chain_offset=rank * C_, **init_kw, **kw)
    clocks = ClockSampler(local)
    clocks.launch()
    for _ in range(a.warmup):
        plan.run(); plan.sync()
    barrier(); plan.sync()
    clocks.start()
    l0 = L.bmm_launch_count()
    t0 = time.perf_counter()
    dev_ms, kern = 0.0, np.zeros(4)
    for _ in range(a.steps):
        plan.run(); plan.sync()
        dev_ms += plan.elapsed_ms()[0]
        kern += np.array(plan.kernel_ms())
    plan.sync(); barrier()
    wall_s = time.perf_counter() - t0
    launches = int(L.bmm_launch_count() - l0)
    clk = clocks.stop()
    plan.check()      # a chain that stopped with an error status invalidates the timing
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, plan.fetch())
    plan.close()

    # ---- end-to-end arm (e2e): the public call with host buffers, every step ------------------
    bufs = api._alloc_out(sid, C_, N, P, K, ns, burnin, relabel, False, (), True)  # pinned
    host_out = api.out_nbytes(bufs[0])
    # bytes that actually cross PCIe: int32 z matrices above 8M allocations travel as 1 B per allocation and
    # are widened by the library on the host (bmm_plan_fetch)
    zbytes = sum(v.nbytes for k, v in bufs[0].items() if k in ("z", "z_original"))
    d2h = host_out - (zbytes - zbytes // 4 if C_ * S * N >= (8 << 20) else 0)
    common = dict(chains=C_, seed=2026, device=local, chain_offset=rank * C_, out_bufs=bufs, alpha=None,
                  burnin=burnin, relabel=relabel, burnrelabel=br)

    def e2e_step():
        if smp == "full":
            return B.gibbs_full(X, ns, K, initial_pi=ip, initial_theta=th.transpose(0, 2, 1), **common)
        if smp == "collapsed":
            return B.gibbs_collapsed(X, ns, K, initial_K=iz, **common)
        return B.gibbs_dp(X, ns, maxK=K, **common)
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        r = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    d2h = int(_lib.lib().bmm_fetch_bytes())     # counted by the library over the last call's device-to-host copies
    zmax = int(r["z"][0, -1].max())
    assert 1 <= zmax <= K

    # ---- reduce over ranks (max time) --------------------------------------------------------
    tm = np.array([dev_ms / 1e3, wall_s, e2e_s])
    if dist:
        import torch
        t = torch.tensor(tm, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tm = t.cpu().numpy()
    total_updates = updates_per_step * a.steps * world
    value = total_updates / tm[0]
    e2e_val = total_updates / tm[2]

    pk, pk_src = peaks()
    # dominant kernel: full_chain_kernel over sweeps burnin..nsamples-1 (kern[2]).  Algorithmic HBM
    # bytes per allocation update: 1 B appended to the allocation history; per sweep and chain
    # theta, theta_rel (K*P*8 each), pi (K*8), alpha (8), permutations (K*4).
    sweeps2 = (ns - burnin) if relabel else (ns - 1)
    per_sweep_hist = (2 if relabel else 1) * K * P * 8 + K * 8 + 8 + (K * 4 if relabel else 0)
    bytes_launch = C_ * (sweeps2 * N * 1 + S * per_sweep_hist)
    dur_s = kern[2] / a.steps / 1e3
    kname = {"full": "full_chain_kernel", "collapsed": "collapsed_prod_kernel", "dp": "dp_kernel"}[smp]
    achieved = bytes_launch / dur_s / 1e9
    traffic = None   # dram bytes of the dominant launch from the committed ncu --set full capture of this configuration
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f).get(kname, {})
        if tr.get("workload") == a.workload and tr.get("chains") == C_ and tr.get("nsamples") == ns:
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
            if tr.get("sweeps_in_launch"):       # the capture is one segment launch: scale to the step's post-burn-in sweeps
                traffic = int(traffic * sweeps2 / tr["sweeps_in_launch"])
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "algorithmic_bytes": int(bytes_launch),
                "peak_source": pk_src,
                "kernel": "%s (sweeps %d..%d, %d chains; launched per download segment, the segments' layout kernels "
                          "are inside kernel_ms)" % (kname, burnin if relabel else 1, ns - 1, C_),
                "kernel_ms": dur_s * 1e3, "kernel_share_of_step": float(kern[2] / max(kern.sum(), 1e-9)),
                "note": "C1-C3 are on-chip (issue/latency) bound by construction: chain state lives in shared "
                        "memory and only the 1 B/update history reaches HBM (SURVEY 8d); see extra.kernels_ms"}
    line = {
        "metric": METRIC, "value": value, "unit": "allocation updates/s", "n_gpus": world, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * tm[0] / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "bundled %s regenerated from set.seed(17) (bit-identical to data/%s.RData)" % (DATASET, DATASET),
        "config": {"workload": "%s, %d chains/GPU, nsamples=%d burnin=%d, relabel=%s burnrelabel=%d"
                               % (WL["label"], C_, ns, burnin, relabel, br),
                   "chains_per_gpu": C_, "nsamples": ns, "parallelism": "chains split across GPUs, no collective",
                   "l2": "per-step histories (%.1f GB written on the device) exceed the 126 MB L2; no explicit flush" % (2 * C_ * ns * N / 1e9)},
        "clocks": clk,
        "e2e": {"value": e2e_val, "unit": "allocation updates/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "host_output_bytes_per_step": int(host_out),
                "ms_per_step": 1e3 * tm[2] / a.steps,
                "api": "bmm_mcmc_b200.gibbs_%s -> bmm_gibbs_%s (C ABI), pinned host output buffers; d2h bytes counted by the "
                       "library: the allocations cross PCIe as one byte each, sweep segment by sweep segment while the later "
                       "sweeps run, and the host widens them to the two int32 matrices (z = perm[z_original])" % (smp, smp)},
        "gpu_launches": launches,
        "roofline": roofline,
        "extra": {"wall_ms_per_step": 1e3 * tm[1] / a.steps,
                  "kernels_ms": {"sweeps_pre_burnin": kern[0] / a.steps, "stephens_batch": kern[1] / a.steps,
                                 "sweeps_post_burnin": kern[2] / a.steps, "finalize_layout": kern[3] / a.steps}},
    }
    if a.workload == "c2" and not a.no_extra:
        # the other two north_star workloads ride on every default line, so the driver's 1 -> 8 runs carry them
        import gc
        del bufs, r
        gc.collect()
        L.bmm_release_cache()
        line["extra"]["sharded"] = sharded_leg(rank, world, local, dist)
        line["extra"]["collapsed_1024"] = collapsed_leg(rank, world, local, dist)
    if rank == 0 and world == 1 and not a.no_cpu:
        line["cpu_baseline"] = cpu_baseline_single()
        if a.workload == "c2":
            line["extra"]["cpu_optimised"] = cpu_optimised(value, e2e_val)
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()
    return 0


def cpu_optimised(gpu_value, gpu_e2e):
    """SURVEY 8d's optional row: the GPU path's ALGORITHM (de-duplicated rows, hoisted log tables, count histograms, one
    uniform per allocation, online relabelling on the patterns) on the host cores (oracle/opt_cpu.cpp, -O3), so that the
    algorithmic and the hardware share of the speed-up over the reference can be told apart."""
    try:
        import bmm_mcmc_b200 as B
        from oracle import pyoracle as O
        X = B.load_dataset(DATASET)
        N = X.shape[0]
        cores = os.cpu_count() or 1
        O.opt_cpu_full_gibbs(X, K, 50, 5, cores, cores)                      # warm-up: threads, page faults
        s1 = O.opt_cpu_full_gibbs(X, K, NSAMPLES, BURNIN, 2, 1)
        one = N * (NSAMPLES - 1) * 2 / s1
        chains = 32 * cores
        sa = O.opt_cpu_full_gibbs(X, K, NSAMPLES, BURNIN, chains, cores)
        allc = N * (NSAMPLES - 1) * chains / sa
        return {"value": allc, "unit": "allocation updates/s", "cores": cores, "one_core": one, "kind": "port-optimised",
                "sample": "%d chains x %d sweeps on %d threads (%.2f s); keeps the byte-wide allocation history per chain, "
                          "returns no int32 matrices" % (chains, NSAMPLES - 1, cores, sa),
                "gpu_device_over_all_cores": gpu_value / allc, "gpu_e2e_over_all_cores": gpu_e2e / allc}
    except Exception as e:      # a baseline that cannot be built must not take the bench line with it
        return {"unavailable": repr(e)[:200]}


def _guarded_main():
    """Exactly one JSON line reaches stdout: everything else a library prints there while the bench runs (the
    NCCL version banner, for one) is sent to stderr by pointing fd 1 at fd 2 until the line is ready."""
    import io
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    buf = io.StringIO()
    py_stdout, sys.stdout = sys.stdout, buf
    try:
        rc = main()
    finally:
        sys.stdout = py_stdout
        sys.stdout.flush()
        os.dup2(real, 1)
        os.close(real)
    lines = buf.getvalue().splitlines()
    js = [ln for ln in lines if ln.startswith("{")]
    for ln in lines:
        if ln not in js[-1:]:
            print(ln, file=sys.stderr)
    if js:
        print(js[-1], flush=True)
    return rc


if __name__ == "__main__":
    sys.exit(_guarded_main())
