#!/usr/bin/env python
"""bench.py -- leapfrog-steps/sec (all chains) of the B200-native HMC hot path, with the HBM
roofline of the vectorised leapfrog kernel and the CPU baseline timed beside it.

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun launches N>1)
    python bench.py --impl reference --gpus N --steps K ...   # reference arm: CPU oracle twin
    python bench.py ... --dump-outputs DIR                     # also write the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over every chain of the workload: one HMC transition (L leapfrogs), one NUTS
transition (config 3), or one complete 200-step window-adaptation warm-up (config 4).  `value` counts executed
leapfrogs with the chain state resident in HBM; `e2e` is the same metric through the public API with HOST buffers
(pinned host -> device copy of the step's positions and keys, init, one step, device -> host copy of the new positions
and acceptance rates, all inside the timed region).  See DESIGN.md section "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# NCCL writes its banner / debug lines to stdout by default; stdout carries exactly one JSON line, so send them to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "leapfrog-steps/sec (all chains)"
UNIT = "leapfrog-steps/s"

WORKLOADS = {
    # BASELINE configs[1]: HMC, 1024-D correlated Gaussian (Sigma = Q diag(logspace(-1,1)) Q^T), 65536 chains,
    # dense mass matrix M^-1 = Sigma, 50 leapfrog steps, 1 GPU (SURVEY section 8d fixed inputs: eps 0.5, q0 = 0.1 N(0,1))
    "hmc_dense_gaussian_65536x1024_L50": dict(C=65536, D=1024, L=50, eps=0.5, dense=True),
    # the same chains x dims x L with a diagonal mass matrix / diagonal Gaussian: the HBM-bound leapfrog shape the
    # north star's ">= 60 % of HBM roofline at 65k chains x 1024 dims" names
    "hmc_diag_gaussian_65536x1024_L50": dict(C=65536, D=1024, L=50, eps=0.1, dense=False),
    # BASELINE configs[0]: the reference's own CPU-runnable case
    "hmc_iso_gaussian_1024x100_L10": dict(C=1024, D=100, L=10, eps=0.2, dense=False),
    # BASELINE configs[2]: NUTS, Neal's funnel (D=128), 65536 chains, diag mass, max_tree_depth=10 (SURVEY 8d: eps 0.1,
    # q0 = 0.1 N(0,1)); a step is one NUTS transition, value counts the leapfrogs the trees actually executed
    # block: NUTS transitions per bench step, run by bjx_nuts_sample (the native run_inference_algorithm) with the chains
    # decoupled across transitions; block=1 times single bjx_nuts_step calls (BJX_BENCH_NUTS_BLOCK overrides)
    "nuts_funnel_65536x128": dict(C=65536, D=128, eps=0.1, nuts=True, depth=10, block=32),
    # BASELINE configs[3]: NUTS + window adaptation (dual averaging + diagonal mass matrix, ONE step size / metric for all
    # chains of all GPUs), 512-D Gaussian with std = logspace(-1,1), 32768 chains per GPU (262144 over 8), eps0 = 1.0,
    # target 0.8; a step is one complete 200-step warm-up: per warm-up step one NUTS transition, the block statistics,
    # ONE NCCL all-gather and the device-side merge / dual averaging
    "nuts_window_adaptation_512": dict(C=32768, D=512, adapt=True, warmup_steps=200, depth=10),
    # BASELINE configs[4]: HMC, hierarchical logistic regression (synthetic, 10000 parameters: G = 9996 group intercepts,
    # 8 Bernoulli-logit observations per group with 2 covariates), 20 leapfrog steps, diag mass, chains sharded over the
    # GPUs (32768 per GPU here; 131072 per GPU = 1M over 8 also fits).  Start in the typical set, eps = 0.005: the origin
    # start with eps = 0.02 pencilled in by SURVEY 8d is unstable for this centred model (acceptance 0).
    "hmc_hier_logit_32768x10000_L20": dict(C=32768, D=10000, L=20, eps=0.005, dense=False, hier=True),
}
DEFAULT_WORKLOAD = "hmc_dense_gaussian_65536x1024_L50"


def target_scale(D):
    import numpy as np
    return np.ones(D) if D == 100 else np.logspace(-0.5, 0.5, D)


def dense_matrices(D):
    """Synthetic inputs of configs[1]: Sigma = Q diag(logspace(-1, 1, D)) Q^T with Q from the QR of a
    default_rng(0) normal matrix (recipe of tests/mcmc/test_mclmc_lrd.py:68-90); returns (cov, precision) float32."""
    import numpy as np
    rng = np.random.default_rng(0)
    Q, _ = np.linalg.qr(rng.standard_normal((D, D)))
    eigs = np.logspace(-1.0, 1.0, D)
    cov = (Q * eigs) @ Q.T
    prec = (Q / eigs) @ Q.T
    return (0.5 * (cov + cov.T)).astype(np.float32), (0.5 * (prec + prec.T)).astype(np.float32)


# ------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks DURING the timed region")
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        if os.environ.get("BJX_BENCH_NO_CLOCKS"):   # diagnosis only: does the nvidia-smi poller disturb short launches?
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU arm: the restated oracle's C twin (the reference itself needs jax, which cannot be installed here)
# ------------------------------------------------------------------------------------------------------
def cpu_hmc_rate(wl, budget_s=12.0, steps=1, warmup=0):
    """leapfrog-steps/s of the C/pthreads oracle twin on all host cores, on a bounded chain sample of the
    same workload (same D, L, eps, target)."""
    import numpy as np
    from oracle import cport, prng
    D, L, eps = wl["D"], wl["L"], wl["eps"]
    cores = cport.num_threads()
    if wl.get("dense"):
        cov, prec = dense_matrices(D)
        msqrt = cport.dense_mass_sqrt(cov)

        def run(Cs, n):
            rs = np.random.default_rng(0)
            q = (0.1 * rs.standard_normal((Cs, D))).astype(np.float32)
            g = (-(q @ prec.T)).astype(np.float32)
            logp = (0.5 * (q * g).sum(1)).astype(np.float32)
            keys = prng.split(prng.key(0), Cs)
            t0 = time.perf_counter()
            for _ in range(n):
                cport.hmc_dense_step(prec, cov, keys, q, logp, g, eps, L, msqrt=msqrt)
            return time.perf_counter() - t0
    else:
        s = target_scale(D)
        inv_var = (1.0 / s ** 2).astype(np.float32)
        imm = (s ** 2).astype(np.float32)

        def run(Cs, n):
            rs = np.random.default_rng(0)
            q = (rs.standard_normal((Cs, D)) * s).astype(np.float32)
            g = (-q * inv_var).astype(np.float32)
            logp = (-0.5 * (q * q * inv_var).sum(1)).astype(np.float32)
            keys = prng.split(prng.key(0), Cs)
            t0 = time.perf_counter()
            for _ in range(n):
                cport.hmc_step(0, inv_var, imm, keys, q, logp, g, eps, L)
            return time.perf_counter() - t0

    # the dense twin works on blocks of 48 chains (its GEMM micro-kernel): keep every thread on whole blocks
    gran = cores * (48 if wl.get("dense") else 1)
    probe_c = max(gran if wl.get("dense") else cores * 4, 64)
    run(probe_c, 1)
    t = run(probe_c, 1)
    per_chain = t / probe_c
    n_steps = max(1, steps)
    Cs = int(min(wl["C"], max(probe_c, budget_s / max(per_chain * (n_steps + warmup), 1e-9))))
    Cs = max(gran, (Cs // gran) * gran)
    Cs = min(Cs, max(gran, (wl["C"] // gran) * gran)) if wl["C"] >= gran else wl["C"]
    if steps <= 1:  # cpu_baseline leg: fill the ~budget_s of CPU work with more transitions when all chains fit
        n_steps = int(max(1, min(200, budget_s / max(per_chain * Cs, 1e-9))))
    if warmup:
        run(Cs, warmup)
    # three repeats, median: worker threads are pinned (oracle/c/oracle_hmc.c) and the thread count follows the cgroup
    # CPU quota, so the repeats agree to a few per cent instead of swinging with the box's scheduler
    n_steps = max(1, n_steps // 3) if steps <= 1 else n_steps
    ts = sorted(run(Cs, n_steps) for _ in range(3))
    t = ts[1]
    rate = Cs * L * n_steps / t
    extra = {"repeats_s": [round(x, 3) for x in ts]}
    if wl.get("dense"):  # two D x D matvecs per leapfrog per chain
        extra["gflops"] = round(4.0 * D * D * rate / 1e9, 1)
    sample = f"{Cs} of {wl['C']} chains x {D} dims x L={L}, {n_steps} transition(s) x 3 repeats (median {t:.2f} s)"
    return rate, cores, sample, t / n_steps * 1e3, extra


def _cpu_nuts_worker(args):
    """One process of the NUTS CPU arm: the restated numpy oracle (oracle/nuts.py, oracle/adaptation.py) on its own chain
    sample, numpy's own threading off (one process per granted core).  Returns (leapfrogs, seconds, repetitions)."""
    wl, budget_s, seed = args
    import numpy as np
    from oracle import adaptation as oadapt, hmc as ohmc, nuts as onuts, prng, targets as otargets
    D = wl["D"]
    F = np.float32
    rs = np.random.default_rng(seed)
    if wl.get("adapt"):
        tgt = otargets.DiagGaussian(np.logspace(-1, 1, D))
        Cs, T = 64, 12
        q = rs.standard_normal((Cs, D)).astype(F)
        count = {"n": 0}

        def kernel(keys, state, target, eps, imm, **kw):
            st, info = onuts.nuts_kernel(keys, state, target, eps, imm, wl["depth"])
            count["n"] += int(info.num_integration_steps.sum())
            return st, info
        t0 = time.perf_counter()
        oadapt.window_adaptation_run(kernel, tgt, prng.key(11 + seed), q, T, shared=True)
        return count["n"], time.perf_counter() - t0, T
    tgt = otargets.Funnel(D)
    Cs = 256
    q = (0.1 * rs.standard_normal((Cs, D))).astype(F)
    st = ohmc.init(q, tgt)
    imm = np.ones(D, F)
    n, t0, reps = 0, time.perf_counter(), 0
    while time.perf_counter() - t0 < budget_s and reps < 20:
        st, info = onuts.nuts_kernel(prng.split(prng.fold_in(prng.key(1 + seed), reps), Cs), st, tgt, F(wl["eps"]), imm, wl["depth"])
        n += int(info.num_integration_steps.sum())
        reps += 1
    return n, time.perf_counter() - t0, reps


def cpu_nuts_rate(wl, budget_s=12.0):
    """leapfrog-steps/s of the restated numpy oracle on a bounded chain sample of the NUTS workloads: one process per core
    this job may use (scheduler affinity and cgroup quota, as for the C twin), each on its own chains; value = all
    leapfrogs / the slowest process's time."""
    import multiprocessing as mp
    from oracle import cport
    cores = max(1, min(cport.num_threads(), 32))   # (32 processes bound the arm's memory and start-up time on big hosts)
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.setdefault(v, "1")           # inherited by the spawned workers: one thread per process
    jobs = [(wl, budget_s, s) for s in range(cores)]
    if cores == 1:
        res = [_cpu_nuts_worker(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(cores) as pool:
            res = pool.map(_cpu_nuts_worker, jobs)
    n = sum(r[0] for r in res)
    t = max(r[1] for r in res)
    reps = res[0][2]
    D = wl["D"]
    if wl.get("adapt"):
        sample = f"{cores} x 64 of {wl['C']} chains x {D} dims, first {reps} of {wl['warmup_steps']} warm-up steps ({t:.1f} s)"
    else:
        sample = f"{cores} x 256 of {wl['C']} chains x {D} dims, {reps} NUTS transition(s) each ({t:.1f} s)"
    return n / t, cores, sample, t / max(reps, 1) * 1e3, {}


def cpu_hier_rate(wl, budget_s=12.0):
    """leapfrog-steps/s of the C/pthreads oracle twin (oracle/c/oracle_hmc.c, target kind 2 = oracle/targets.py HierLogit
    with the library's exact expf / log1pf) on all host cores it may use, on a bounded chain sample of config 5."""
    import numpy as np
    from blackjax_b200.targets import HierLogit
    from oracle import cport, hmc as ohmc, prng, targets as otargets
    D, L = wl["D"], wl["L"]
    F = np.float32
    x, bits = HierLogit.synthetic_data(D - 4, seed=1)
    cores = cport.num_threads()
    Cs = max(cores, 8)
    rs = np.random.default_rng(0)
    q = np.empty((Cs, D), F)
    q[:, :4] = [0.5, np.log(0.7), 1.0, -0.5]
    q[:, 4:] = 0.5 + 0.7 * rs.standard_normal((Cs, D - 4))
    st = ohmc.init(q, otargets.HierLogit(x, bits))
    qc, lc, gc = q.copy(), st.logdensity.copy(), st.logdensity_grad.copy()
    imm = np.ones(D, F)

    def run(n):
        t0 = time.perf_counter()
        for r in range(n):
            cport.hmc_hier_step(x, bits, imm, prng.split(prng.fold_in(prng.key(1), r), Cs), qc, lc, gc, wl["eps"], L)
        return time.perf_counter() - t0
    t1 = run(1)
    n = int(max(1, min(50, budget_s / 3.0 / max(t1, 1e-9))))
    ts = sorted(run(n) for _ in range(3))
    t = ts[1]
    sample = f"{Cs} of {wl['C']} chains x {D} dims x L={L}, {n} transition(s) x 3 repeats (median {t:.2f} s)"
    return Cs * L * n / t, cores, sample, t / n * 1e3, {"repeats_s": [round(v, 3) for v in ts]}


def cpu_rate(wl, budget_s, steps=1, warmup=0):
    if wl.get("nuts") or wl.get("adapt"):
        return cpu_nuts_rate(wl, budget_s)
    if wl.get("hier"):
        return cpu_hier_rate(wl, budget_s)
    return cpu_hmc_rate(wl, budget_s, steps, warmup)


def run_reference(args, wl_name, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rate, cores, sample, ms, extra = cpu_rate(wl, budget_s=20.0, steps=args.steps, warmup=min(args.warmup, 1))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl_name, **{k: v for k, v in wl.items()},
                   "note": "baseline/_ref (BlackJAX on JAX) was tried first and cannot be installed in this image (no jax / "
                           "jaxlib wheel, no network); this arm times the restated oracle instead: the C/pthreads twin of "
                           "oracle/hmc.py (HMC workloads, config 5's hierarchical model included) or the numpy oracle (NUTS workloads)"},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, **extra},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel at its benchmark shape, from the committed
    `ncu --set full` capture summaries (profiles/r02_traffic.json, written by scripts/ncu_traffic.py from the .ncu-rep of the
    same command); None when no capture of that kernel is committed."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        e = t.get(kernel_key)
        return (float(e["dram_bytes"]), e["source"]) if e else (None, None)
    except Exception:
        return None, None


# payload cap of --dump-outputs; with the .npy headers the files stay under 64 MB
DUMP_BYTES = 60 * 10 ** 6


def dump_outputs(out_dir, per_chain, shared=None):
    """--dump-outputs: writes what the timed path returned in its last step as out_dir/<name>.npy, float32.  per_chain maps
    names to tensors with the chains on axis 0.  When they exceed DUMP_BYTES, every one of them keeps the same seeded sample
    of chains; chain_index.npy (float64) holds the chain indices kept.  shared holds the arrays that are not per chain."""
    import numpy as np
    import torch
    shared = {k: torch.as_tensor(v) for k, v in (shared or {}).items()}
    C = next(iter(per_chain.values())).shape[0]
    row_bytes = 8 + sum(4 * v[0].numel() for v in per_chain.values())
    n = min(C, (DUMP_BYTES - sum(4 * v.numel() for v in shared.values())) // row_bytes)
    idx = np.arange(C) if n == C else np.sort(np.random.default_rng(0).choice(C, n, replace=False))
    out = {"chain_index": idx.astype(np.float64)}
    for k, v in per_chain.items():
        out[k] = v.index_select(0, torch.from_numpy(idx).to(v.device)).float().cpu().numpy()
    for k, v in shared.items():
        out[k] = v.float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_nuts_workload(args, wl, dev, dist, world, rank, local_rank):
    """BASELINE configs[2] (NUTS on the funnel) and configs[3] (NUTS + shared window adaptation).  value = leapfrogs the
    trees actually executed (sum of num_integration_steps over chains, steps and ranks) / max-over-ranks CUDA-event time."""
    import numpy as np
    import torch

    import blackjax_b200 as bj

    C, D, depth = wl["C"], wl["D"], wl["depth"]
    K, W = args.steps, args.warmup
    adapt = bool(wl.get("adapt"))
    BLK = 1 if adapt else int(os.environ.get("BJX_BENCH_NUTS_BLOCK", wl.get("block", 1)))
    n_gpus = world
    key0 = bj.random.key(7, dev)
    # global chain c starts at normal(split(key, C_global)[c]): the same chains whatever the GPU count
    chain_keys = bj.random.split(key0, C * world)[rank * C:(rank + 1) * C]
    if adapt:
        tgt = bj.targets.DiagGaussian(np.logspace(-1, 1, D))
        q0 = bj.random.normal(chain_keys, (D,))
        T = wl["warmup_steps"]
        warm = bj.window_adaptation(bj.nuts, tgt, shared=True, initial_step_size=1.0, target_acceptance_rate=0.8,
                                    max_num_doublings=depth)
    else:
        tgt = bj.targets.Funnel(D)
        q0 = 0.1 * bj.random.normal(chain_keys, (D,))
        imm = torch.ones(D, device=dev)
        kern = bj.nuts.build_kernel(inplace=True, chain_offset=rank * C, max_tree_depth=depth)
    step_keys = bj.random.split(bj.random.key(0, dev), W + K + 16)
    lf = torch.zeros(1, dtype=torch.int64, device=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if adapt:
        def one_step(t, count):
            (st, params), hist = warm.run(step_keys[t], q0, T, _leapfrog_counter=count)
            return st, params, hist
        state = None
    else:
        state = bj.nuts.init(q0.clone(), tgt)

        def one_step(t, count):
            nonlocal state
            if BLK > 1:
                state, _, acc, n_int = bj.sample_nuts_native(step_keys[t], state, tgt, wl["eps"], imm, BLK,
                                                              max_num_doublings=depth, keep_history=False, chain_offset=rank * C)
                if count is not None:
                    count += n_int.sum()
                return state, acc, n_int
            state, info = kern(step_keys[t], state, tgt, wl["eps"], imm, depth)
            if count is not None:
                count += info.num_integration_steps.sum()
            return state, info
    for t in range(W):   # warm-up runs the SAME code as the timed steps (the leapfrog counter's kernels load lazily)
        out = one_step(t, lf)
    lf.zero_()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(W, W + K):
        out = one_step(t, lf)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    if dist is not None:
        allc = [None] * world
        dist.all_gather_object(allc, clocks)
        ok = [c for c in allc if c and c.get("sm_mhz")]
        if ok:
            clocks = {"sm_mhz": min(c["sm_mhz"] for c in ok), "sm_max_mhz": max(c["sm_max_mhz"] for c in ok),
                      "reasons": sorted(set(r for c in ok for r in c["reasons"])),
                      "per_rank_sm_mhz": [c["sm_mhz"] for c in ok], "samples": sum(c.get("samples", 0) for c in ok)}
    if args.dump_outputs and rank == 0:
        if adapt:
            st, params, hist = out
            dump_outputs(args.dump_outputs, st._asdict(), {"step_size": [params["step_size"]],
                                                           "inverse_mass_matrix": params["inverse_mass_matrix"],
                                                           "step_size_history": hist})
        elif BLK > 1:   # acceptance rates and tree sizes of the step's BLK transitions, chains first
            st, acc, n_int = out
            dump_outputs(args.dump_outputs, {**st._asdict(), "acceptance_rate": acc.T, "num_integration_steps": n_int.T})
        else:
            st, info = out
            dump_outputs(args.dump_outputs, {**st._asdict(), **{k: v for k, v in info._asdict().items() if torch.is_tensor(v)}})

    # ---- end to end with HOST buffers: positions in from pinned memory, one step, positions + a per-chain result out -----
    q_host = torch.empty(C, D, dtype=torch.float32).pin_memory()
    q_host.copy_(q0 if adapt else state.position)
    out_host = torch.empty(C, D, dtype=torch.float32).pin_memory()
    acc_host = torch.empty(C, dtype=torch.float32).pin_memory()
    q_dev = torch.empty(C, D, device=dev)
    lf_e2e = torch.zeros(1, dtype=torch.int64, device=dev)
    K_e2e = max(1, min(K, 5))

    def e2e_step(t, count):
        q_dev.copy_(q_host, non_blocking=True)
        if adapt:
            (st, params), hist = warm.run(step_keys[t], q_dev, T, _leapfrog_counter=count)
            out_host.copy_(st.position, non_blocking=True)
            acc_host.copy_(st.logdensity, non_blocking=True)
        else:
            st = bj.nuts.init(q_dev, tgt)
            if BLK > 1:
                st, _, acc, n_int = bj.sample_nuts_native(step_keys[t], st, tgt, wl["eps"], imm, BLK, max_num_doublings=depth,
                                                          keep_history=False, chain_offset=rank * C)
                count += n_int.sum()
                out_host.copy_(st.position, non_blocking=True)
                acc_host.copy_(acc[-1], non_blocking=True)
            else:
                st, info = kern(step_keys[t], st, tgt, wl["eps"], imm, depth)
                count += info.num_integration_steps.sum()
                out_host.copy_(st.position, non_blocking=True)
                acc_host.copy_(info.acceptance_rate, non_blocking=True)
    e2e_step(0, lf_e2e)
    lf_e2e.zero_()
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for t in range(K_e2e):
        e2e_step(W + t, lf_e2e)
    g1.record()
    barrier()
    ms_e2e = g0.elapsed_time(g1)

    tot = torch.tensor([float(lf.item()), float(lf_e2e.item())], dtype=torch.float64, device=dev)
    times = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tot)
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    n_lf, n_lf_e2e = float(tot[0]), float(tot[1])
    ms_total, ms_e2e = float(times[0]), float(times[1])
    if rank != 0:
        return
    peaks = load_peaks()
    peak = float(peaks.get("hbm_gbs", 6650.0))
    value = n_lf / (ms_total * 1e-3)
    transitions = K * (T if adapt else BLK)
    # The HBM roofline of the path is that of the vectorised one-step leapfrog kernel (24*D bytes per chain per launch,
    # SURVEY 8d) at this workload's chains x dims, timed live below; the tree kernel keeps (q, p, g, p_sum) in registers
    # across the leaves of a launch, so its own figure is reported as an equivalent (what 24*D per executed leapfrog would
    # amount to) next to it, not as a fraction of the HBM peak.
    from blackjax_b200 import _engine
    dtgt = bj.targets.DiagGaussian(np.ones(D))
    deng = _engine.Engine(dev, C, D, dtgt)
    deng.set_metric(torch.ones(D, device=dev))
    q1 = torch.randn(C, D, device=dev)
    p1 = deng.sample_momentum(step_keys[0], chain_offset=rank * C)
    lp1, g1 = deng.init_state(q1)
    for _ in range(3):
        deng.leapfrog_(q1, p1, lp1, g1, 0.05, 1)
    torch.cuda.synchronize()
    n1 = 40
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(n1):
        deng.leapfrog_(q1, p1, lp1, g1, 0.05, 1)
    f1.record()
    torch.cuda.synchronize()
    ms_1step = f0.elapsed_time(f1) / n1
    achieved = 24.0 * C * D / (ms_1step * 1e-3) / 1e9
    del q1, p1, g1, deng
    traffic, traffic_src = ncu_traffic(f"k_leapfrog_diag_{C}x{D}")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "chains_per_gpu": C, "dims": D, "max_tree_depth": depth,
                   "mass_matrix": "diag", "step": ("one %d-step window-adaptation warm-up (NUTS transition + block statistics "
                                                   "+ one NCCL all-gather + device-side merge / dual averaging per warm-up step)" % T)
                   if adapt else ("one NUTS transition" if BLK == 1 else
                                  "%d NUTS transitions of every chain in one bjx_nuts_sample call (the native run_inference_algorithm; "
                                  "chains decoupled across transitions, k_nuts_chains)" % BLK),
                   "parallelism": (f"chains sharded x{n_gpus}; one NCCL all-gather of {(C // 4096) * (2 + 2 * D) * 4} bytes per rank "
                                   "per warm-up step (bjx_allgather_stats)") if adapt
                   else f"chains sharded x{n_gpus}, no data-path collective",
                   "l2": "state arrays %.0f MB per GPU (workspace rows 9 + 2*depth); inputs exceed L2" % (C * D * 4 / 1e6),
                   "mean_tree_size": n_lf / (n_gpus * C * transitions), "ms_per_transition": ms_total / transitions},
        "roofline": {"bound": "hbm", "kernel": "k_leapfrog (diag metric, 1 step/launch, 24*D B per chain) at this workload's chains x dims",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": traffic_src, "avg_launch_ms": ms_1step, "launches_timed": n1,
                     "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"},
        "tree_kernel": {"kernel": "k_nuts_doubling (one launch for doublings 0-3 over all chains, then one per further doubling over "
                        "the compacted list; row counts stay on the device: no host round trip)" if (adapt or BLK == 1) else
                        "k_nuts_chains (persistent grid; every warp takes whole chains through all transitions of the call)",
                        "equivalent_GBps_at_24D_per_leapfrog": 24.0 * D * value / n_gpus / 1e9,
                        "bound": "dependent-instruction latency / issue slots (rows are register-resident inside a launch); "
                                 "ncu issue-slot figures: profiles/r02_ncu_nuts.md"},
        "e2e": {"value": n_lf_e2e / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": C * D * 4 + 8,
                "d2h_bytes_per_step": C * D * 4 + C * 4, "steps": K_e2e, "ms_per_step": ms_e2e / K_e2e},
        "gpu_launches": K * ((T * 7 + 2) if adapt else (4 if BLK == 1 else 3)),
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and n_gpus == 1:
        rate, cores, sample, _, extra_cpu = cpu_rate(wl, budget_s=12.0)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                "note": "restated numpy oracle, not JAX (no jax wheel in this image)", **extra_cpu}
    print(json.dumps(line), flush=True)



# ------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=4, help="chain slices (streams) of the end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0's chains) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, args.workload, wl)
        return

    import numpy as np
    import torch

    import blackjax_b200 as bj
    from blackjax_b200 import _engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: blackjax_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    if wl.get("nuts") or wl.get("adapt"):
        run_nuts_workload(args, wl, dev, dist, world, rank, local_rank)
        if dist is not None:
            dist.destroy_process_group()
        return

    C, D, L, eps = wl["C"], wl["D"], wl["L"], wl["eps"]
    K, W = args.steps, args.warmup
    dense = bool(wl.get("dense"))
    s = target_scale(D)
    diag_tgt = bj.targets.DiagGaussian(s)
    diag_imm = torch.from_numpy((s ** 2).astype(np.float32)).to(dev)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    # chains are sharded over GPUs: this rank owns global chains [rank*C, (rank+1)*C)  (weak scaling)
    hier = bool(wl.get("hier"))
    if dense:
        cov, prec = dense_matrices(D)
        tgt = bj.targets.DenseGaussian(prec)
        imm = torch.from_numpy(cov).to(dev)
        q0 = 0.1 * torch.randn(C, D, device=dev, generator=gen)
    elif hier:
        tgt = bj.targets.HierLogit(*bj.targets.HierLogit.synthetic_data(D - 4, seed=1))
        imm = torch.ones(D, device=dev)
        q0 = torch.empty(C, D, device=dev)
        q0[:, 0], q0[:, 1], q0[:, 2], q0[:, 3] = 0.5, float(np.log(0.7)), 1.0, -0.5
        q0[:, 4:] = 0.5 + 0.7 * torch.randn(C, D - 4, device=dev, generator=gen)
    else:
        tgt, imm = diag_tgt, diag_imm
        q0 = torch.randn(C, D, device=dev, generator=gen) * torch.from_numpy(s.astype(np.float32)).to(dev)
    # one step key per transition; chain c of this rank uses split(step_key, C_global)[rank*C + c], derived inside the
    # transition kernel (bjx_set_key_mode), so results do not depend on the GPU count
    kernel = bj.hmc.build_kernel(inplace=True, chain_offset=rank * C)
    state = bj.hmc.init(q0.clone(), tgt)
    step_keys = bj.random.split(bj.random.key(0, dev), W + K + 1)

    def chain_keys(t):
        return step_keys[t]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for t in range(W):
        state, info = kernel(chain_keys(t), state, tgt, eps, imm, L)
    sampler = ClockSampler(local_rank)
    sampler.start()  # every rank samples its own GPU
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(W, W + K):
        state, info = kernel(chain_keys(t), state, tgt, eps, imm, L)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    # our kernels per step: (diag) k_hmc_transition | (dense) 2L+3 products (bjx::k_gemm_f16x3), 2L-1 window checks, normal
    # draw, 2 exact operand splits, 2 energies, the opening and the closing row kernel, accept
    launches = K * (1 if not dense else (4 * L + 10))
    acc_mean = float(info.acceptance_rate.mean())
    clocks = sampler.stop()
    if dist is not None:  # rank 0 reports the slowest GPU's median SM clock and the union of throttle reasons
        all_clocks = [None] * world
        dist.all_gather_object(all_clocks, clocks)
        if rank == 0:
            ok = [c for c in all_clocks if c and c.get("sm_mhz")]
            if ok:
                clocks = {"sm_mhz": min(c["sm_mhz"] for c in ok), "sm_max_mhz": max(c["sm_max_mhz"] for c in ok),
                          "reasons": sorted(set(r for c in ok for r in c["reasons"])),
                          "per_rank_sm_mhz": [c["sm_mhz"] for c in ok], "samples": sum(c.get("samples", 0) for c in ok)}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {**state._asdict(), **{k: v for k, v in info._asdict().items() if torch.is_tensor(v)}})

    # ---- the vectorised single-step leapfrog kernel: the HBM roofline the north star names -------------
    eng = _engine.get_engine(state.position, tgt)
    ms_gemm = 0.0
    n_prod = 0
    if dense:
        # The dominant kernel of the dense workload: bjx::k_gemm_f16x3 in its fused form (Cin + lincomb / double kick + Y +
        # operand planes of Y), timed where it runs: inside a run of leapfrog steps on the engine's stream.  n_lf steps =
        # 2 n_lf products (2 n_lf - 1 fused + the closing gradient product) + one opening and one closing row kernel +
        # the 3 us window checks; the average below charges all of that to the products (conservative).
        pv = eng.sample_momentum(chain_keys(W + K), chain_offset=rank * C)
        qv, lv, gv = state.position.clone(), state.logdensity.clone(), state.logdensity_grad.clone()
        n_lf = 20
        eng.leapfrog_(qv, pv, lv, gv, 0.01, n_lf)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(2):
            eng.leapfrog_(qv, pv, lv, gv, 0.01, n_lf)
        f1.record()
        torch.cuda.synchronize()
        n_prod = 2 * 2 * n_lf
        ms_gemm = f0.elapsed_time(f1) / n_prod
        del pv, qv, lv, gv
    # the vectorised one-step leapfrog kernel (diagonal metric) at the same chains x dims: the HBM roofline kernel
    qd = torch.randn(C, D, device=dev, generator=gen)
    deng = _engine.Engine(dev, C, D, diag_tgt)
    deng.set_metric(diag_imm)
    p = deng.sample_momentum(chain_keys(W + K), chain_offset=rank * C)
    lp1, g1 = deng.init_state(qd)
    q1 = qd
    for _ in range(3):
        deng.leapfrog_(q1, p, lp1, g1, 0.1, 1)
    torch.cuda.synchronize()
    n1 = 40
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(n1):
        deng.leapfrog_(q1, p, lp1, g1, 0.1, 1)
    f1.record()
    torch.cuda.synchronize()
    ms_1step = f0.elapsed_time(f1) / n1
    del q1, p, g1, qd, deng

    # ---- end to end through the public API with HOST buffers ----------------------------------------------
    q_host = torch.empty(C, D, dtype=torch.float32).pin_memory()
    q_host.copy_(state.position)
    out_host = torch.empty(C, D, dtype=torch.float32).pin_memory()
    acc_host = torch.empty(C, dtype=torch.float32).pin_memory()
    key_host = torch.empty(2, dtype=torch.int32).pin_memory()
    key_host.copy_(chain_keys(0).view(torch.int32))
    q_dev = torch.empty(C, D, device=dev)
    k_dev = torch.empty(2, dtype=torch.int32, device=dev)
    K_e2e = max(1, min(K, 10))
    # The batch goes through the public API as n_chunks chain slices, each on its own stream, so that one slice's
    # host->device / device->host copies run beside another slice's kernels.  Slicing is invisible in the results:
    # every chain's key derives from the step key and its GLOBAL chain index (chain_offset).
    n_chunks = args.e2e_chunks if (args.e2e_chunks > 0 and C % (8 * args.e2e_chunks) == 0) else 1
    Cc = C // n_chunks
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_chunks)]
    kernels_e2e = [bj.hmc.build_kernel(inplace=True, chain_offset=rank * C + k * Cc) for k in range(n_chunks)]

    def e2e_step():
        main = torch.cuda.current_stream()
        for k, s_ in enumerate(streams):
            s_.wait_stream(main)
            with torch.cuda.stream(s_):
                rows = slice(k * Cc, (k + 1) * Cc)
                q_dev[rows].copy_(q_host[rows], non_blocking=True)
                if k == 0:
                    k_dev.copy_(key_host, non_blocking=True)
                    key_ready = torch.cuda.Event()
                    key_ready.record(s_)
                else:
                    s_.wait_event(key_ready)
                st = bj.hmc.init(q_dev[rows], tgt)
                st, inf = kernels_e2e[k](k_dev.view(torch.uint32), st, tgt, eps, imm, L)
                out_host[rows].copy_(st.position, non_blocking=True)
                acc_host[rows].copy_(inf.acceptance_rate, non_blocking=True)
        for s_ in streams:
            main.wait_stream(s_)

    for _ in range(2):
        e2e_step()
    barrier()
    g0, g1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(K_e2e):
        e2e_step()
    g1e.record()
    barrier()
    ms_e2e = g0.elapsed_time(g1e)

    # ---- max over ranks ---------------------------------------------------------------------------------------
    times = torch.tensor([ms_total, ms_e2e, ms_1step, ms_gemm], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_1step, ms_gemm = [float(x) for x in times]
    value = n_gpus * C * L * K / (ms_total * 1e-3)
    e2e_value = n_gpus * C * L * K_e2e / (ms_e2e * 1e-3)

    if rank == 0:
        peaks = load_peaks()
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        bytes_1step = 24.0 * C * D
        achieved = bytes_1step / (ms_1step * 1e-3) / 1e9
        ms_step = ms_total / K
        traffic_leapfrog, src_leapfrog = ncu_traffic("k_leapfrog_diag_65536x1024") if (C, D) == (65536, 1024) else (None, None)
        traffic_gemm, src_gemm = ncu_traffic("k_gemm_f16x3_fused_65536x1024") if (C, D) == (65536, 1024) else (None, None)
        hbm_roofline = {"bound": "hbm", "kernel": "k_leapfrog (diag metric, 1 step/launch, 24*D B per chain)",
                        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                        "traffic": traffic_leapfrog, "traffic_source": src_leapfrog,
                        "peak_source": peak_src, "avg_launch_ms": ms_1step, "launches_timed": n1}
        if dense:
            burst = float(peaks.get("bf16_tflops", 1590.0))
            tpeak = float(peaks.get("bf16_tflops_sustained", 1400.0))
            tf_achieved = 2.0 * C * D * D / (ms_gemm * 1e-3) / 1e12
            roofline = {"bound": "tensor",
                        "kernel": "bjx::k_gemm_f16x3, fused form (hand-written tcgen05.mma.cta_group::2 + TMA; epilogue: Cin, per-row "
                                  "lincomb / double kick, Y, operand planes of Y for the next product); float32-accurate: 3 fp16 "
                                  "products per float32 product (ceiling frac = 1/3)",
                        "achieved": tf_achieved, "peak": tpeak, "unit": "TFLOP/s", "frac": tf_achieved / tpeak,
                        "frac_of_burst_peak": tf_achieved / burst, "burst_peak": burst,
                        "traffic": traffic_gemm, "traffic_source": src_gemm,
                        "algorithmic_bytes": 16.0 * C * D,
                        "peak_source": ("measured sustained bf16 (MEASURED_PEAKS.json bf16_tflops_sustained): the kernel is timed inside "
                                        "a run of leapfrog steps under the power cap" if "bf16_tflops_sustained" in peaks
                                        else "fallback 1400 TFLOP/s sustained"),
                        "avg_launch_ms": ms_gemm, "launches_timed": n_prod,
                        "note": "algorithmic float32 flops 2*C*D^2 per launch; CUDA events on the engine's stream around 2 x 20 "
                                "leapfrog steps = 80 products, row kernels and window checks of those steps charged to the products",
                        "gemms_per_step": 2 * L + 3, "gemm_share_of_step": (2 * L + 3) * ms_gemm / ms_step}
            extra = {"roofline_hbm_leapfrog": hbm_roofline}
        else:
            roofline = hbm_roofline
            extra = {"fused_transition": {"kernel": ("k_big_hmc (CTA per chain, row resident in shared memory)" if D > 1024 else
                                                     "k_hmc_transition (L leapfrogs/launch, row resident in registers)"),
                                          "hbm_bytes_per_launch": 16.0 * C * D + 20.0 * C,
                                          "equivalent_GBps_at_24D_per_leapfrog": 24.0 * C * D * L / (ms_step * 1e-3) / 1e9,
                                          "speedup_vs_1step_launches": (ms_1step * L) / ms_step}}
            if hier:  # the transition kernel is bound by the model's transcendental work, not by HBM: report it beside
                n_obs = 8.0 * (D - 4)
                mufu = (2.0 * (L - 1) + 3.0) * n_obs * C  # ex2 + rcp per observation; + lg2 where the log-density is live
                extra["model_compute"] = {"sigmoid_evals_per_s": n_obs * C * L / (ms_step * 1e-3),
                                          "mufu_per_s": mufu / (ms_step * 1e-3),
                                          "mufu_peak_per_s": 148 * 16 * 1.965e9,
                                          "note": "16 MUFU lanes/clk/SM x 148 SMs at the maximum SM clock"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "chains_per_gpu": C, "dims": D, "leapfrogs_per_step": L,
                       "step_size": eps, "mass_matrix": "dense" if dense else "diag",
                       "parallelism": f"chains sharded x{n_gpus}, no data-path collective",
                       "l2": "inputs larger than L2 (q,g = 2 x %.0f MB per GPU)" % (C * D * 4 / 1e6),
                       "mean_acceptance": acc_mean},
            "roofline": roofline, **extra,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": C * D * 4 + 8,
                    "d2h_bytes_per_step": C * D * 4 + C * 4, "steps": K_e2e, "ms_per_step": ms_e2e / K_e2e,
                    "pipeline": f"{n_chunks} chain slices on {n_chunks} streams through the public API "
                                "(hmc.init + kernel per slice); copies of one slice overlap kernels of another"},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if not args.no_cpu_baseline and n_gpus == 1:
            rate, cores, sample, _, extra_cpu = cpu_rate(wl, budget_s=12.0)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "note": "restated oracle (C/pthreads twin or numpy), not JAX (no jax wheel in this image)",
                                    **extra_cpu}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
