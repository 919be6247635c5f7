#!/usr/bin/env python
"""Benchmark of the CAVI sweep hot path: SNP x trait updates/s (BASELINE.json's metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one full VB iteration of the BASELINE config as `atlasqtl()` would run it: the host
q-/p-sized algebra, the fused sweep kernel (coreDualLoop + its reductions), the row sums of Z, the
all-reduce (N > 1) and the table refresh (+ ELBO part once annealing is over).

  value  updates/s with everything resident in HBM: p*q*K / (device time of the K steps' kernels,
         CUDA events on the library's stream, max over ranks)
  e2e    the same K steps through the public host API / C ABI with HOST buffers (per-step H2D of the
         per-trait vectors and theta/zeta, D2H of the column / row sums), wall clock between
         barrier + device synchronize, max over ranks
  N > 1  traits are sharded over ranks (strong scaling: the total q is fixed), one NCCL all-reduce per sweep.

`--impl reference` times the reference's own coreDualLoop (oracle/_ref: src/coreLoop.cpp compiled
unmodified) on the host cores, on a bounded sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, what the timed path returned after its last step as DIR/<name>.npy
(float64): gam_vb, beta_vb, theta_vb, zeta_vb (the reference arm: its gam_vb, mu_beta_vb, beta_vb).  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.  A p x q output too large for
DUMP_BYTES in all is written as a fixed, seeded sample of its entries, <name>_sample.npy, with their column-major
positions in pq_sample_index.npy.  With N > 1 ranks each rank writes its own trait slab, with the suffix .rank<r>.
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

# roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the sweep kernel, taken from the ncu
# `--set full` capture recorded in profiles/ncu_traffic.json by tools/profile_c2.sh.  The record carries the hash of the
# kernel sources it was captured from; it is reported only while that hash matches the sources of the library being
# benchmarked -- otherwise the field is null and `traffic_source` says which capture is stale.  Never a constant.
TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")


def kernel_source_hash():
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "atlasqtl_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(config, world):
    try:
        rec = json.load(open(TRAFFIC_FILE))[config][str(world)]
    except (OSError, KeyError, ValueError):
        return None, "no ncu capture recorded for this config / GPU count (profiles/ncu_traffic.json)"
    if rec.get("src_hash") != kernel_source_hash():
        return None, f"stale: {rec.get('source')} was captured from other kernel sources ({rec.get('src_hash')})"
    return rec["bytes"], rec.get("source")

FP64_PEAK_TFLOPS = 37.05  # measured DMMA m8n8k4 peak on this pool's B200 (profiles/r2_fp64_peaks_microbench.txt, with a clock record);
                          # MEASURED_PEAKS.json has no fp64 entry (bf16 / HBM only)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


DUMP_BYTES = 64 << 20       # --dump-outputs: at most this much in all (over all ranks)
DUMP_SAMPLE = 1 << 21       # entries kept of each large p x q output (split over the ranks)


def dump_outputs(dirname, arrays, rank=0, world=1):
    """Write `arrays` (name -> vector or p x q matrix) as float64 .npy files under `dirname` (see the module doc)."""
    os.makedirs(dirname, exist_ok=True)
    suffix = f".rank{rank}" if world > 1 else ""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    mats = {k: v for k, v in arrays.items() if v.ndim == 2}
    if world * sum(v.nbytes for v in arrays.values()) > DUMP_BYTES and mats:
        shape = next(iter(mats.values())).shape
        size = shape[0] * shape[1]
        idx = np.sort(np.random.default_rng([123, rank]).choice(size, min(size, DUMP_SAMPLE // world), replace=False))
        np.save(os.path.join(dirname, f"pq_sample_index{suffix}.npy"), idx.astype(np.float64))
        for k, v in mats.items():
            assert v.shape == shape
            arrays.pop(k)
            arrays[k + "_sample"] = v.ravel(order="F")[idx]
    for k, v in arrays.items():
        np.save(os.path.join(dirname, f"{k}{suffix}.npy"), v)


# ----------------------------------------------------------------------------- workload
# X larger than this is generated as packed 2-bit calls and standardised on the device
PACKED_ABOVE_BYTES = int(float(os.environ.get("AQ_BENCH_PACKED_ABOVE_GB", "4")) * (1 << 30))


def make_workload(name, k_first, k_last, seed=123, threads=None, force_dense=False):
    """Synthetic data + default hyper / init of BASELINE config `name` for the trait slab [k_first, k_last).

    Returns (cfg, X, Y, hyper, init).  X is the standardised n x p matrix (Fortran) -- or, when it would exceed
    PACKED_ABOVE_BYTES (C3: 4.8 GB, C5: 20 GB per rank), a dict(packed=uint8 [p][ceil(n/4)], n=n) of 2-bit genotype calls
    that the library standardises on the device (aq_prep_geno, R/prepare_atlasqtl.R:57), with Y then RAW (centred there)."""
    from concurrent.futures import ThreadPoolExecutor

    from scipy import special as sp

    from atlasqtl_b200 import hyper_init, synthetic
    from atlasqtl_b200.device import pack_genotypes
    cfg = dict(synthetic.CONFIGS[name])
    n, p, q = cfg["n"], cfg["p"], cfg["q"]
    threads = threads or host_threads()
    packed = (not force_dense) and 8.0 * n * p > PACKED_ABOVE_BYTES
    rng = np.random.default_rng(seed)
    p_act = cfg.get("p_act", cfg.get("hotspots", 20))
    q_act = cfg.get("q_act", q)
    act = np.sort(rng.choice(p, size=p_act, replace=False))
    traits_act = rng.choice(q, size=q_act, replace=False)
    beta = np.zeros((p_act, q))
    pat = rng.random((p_act, q_act)) < 0.2
    beta[:, traits_act] = pat * rng.normal(0.0, cfg.get("beta_sd", 1.0), size=(p_act, q_act))
    maf = 0.25
    chunk_cols = 8192
    starts = list(range(0, p, chunk_cols))
    X = None if packed else np.empty((n, p), order="F")
    G_packed = np.empty((p, (n + 3) // 4), dtype=np.uint8) if packed else None
    X_act = np.empty((n, p_act))

    def gen(j0):   # genotypes of one column chunk (its own generator stream: the same data whatever the thread count)
        j1 = min(p, j0 + chunk_cols)
        G = np.random.default_rng([seed, 11, j0]).binomial(2, maf, size=(n, j1 - j0)).astype(np.float64)
        sd = G.std(axis=0, ddof=1)
        bad = sd == 0   # constant columns are re-drawn rather than dropped so that p stays as named
        if bad.any():
            G[:2, bad] = [[0.0], [1.0]]
            sd = G.std(axis=0, ddof=1)
        Z = (G - G.mean(axis=0)) / sd
        if packed:
            G_packed[j0:j1] = pack_genotypes(G)
        else:
            X[:, j0:j1] = Z
        lo, hi = np.searchsorted(act, [j0, j1])
        X_act[:, lo:hi] = Z[:, act[lo:hi] - j0]

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(gen, starts))
    ql = k_last - k_first
    # Everything per-trait is drawn on a FIXED global grid of trait chunks (each with its own generator stream), so that the
    # data do not depend on how the traits are sharded: the `check` values of runs at different GPU counts are comparable.
    tchunk = 64

    def trait_chunks():
        for c0 in range((k_first // tchunk) * tchunk, k_last, tchunk):
            lo, hi = max(c0, k_first), min(c0 + tchunk, k_last, q)
            yield c0, lo - c0, hi - c0, lo - k_first, hi - k_first   # chunk start, columns inside it, columns of the slab

    Y = np.empty((n, ql), order="F")
    gam = np.empty((p, ql), order="F")
    mu = np.empty((p, ql), order="F")
    e_p = max(1.0, float(pat.sum(axis=0).mean()))
    p0 = (e_p, max(10.0, 2.0 * e_p))  # (mean, variance) of the prior number of active SNPs per trait
    t02 = hyper_init._solve_t02(p, p0)
    n0 = float(hyper_init.get_mu(p0[0], t02, p))
    sd0 = 1e-4 + t02

    def fill(ch):
        c0, a, b, lo, hi = ch
        r = np.random.default_rng([seed, 7, c0])
        noise = r.standard_normal((tchunk, n))   # auto_set_init_ distributions (R/set_hyper_init.R:388-405) below
        Y[:, lo:hi] = X_act @ beta[:, k_first + lo:k_first + hi] + noise[a:b].T
        for k in range(tchunk):   # one trait at a time: bounded scratch whatever p is
            z = r.standard_normal(p, dtype=np.float32)
            m = r.standard_normal(p, dtype=np.float32)
            if a <= k < b:
                gam[:, lo + k - a] = sp.ndtr(n0 + sd0 * z)
                mu[:, lo + k - a] = m

    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(fill, list(trait_chunks())))
    if not packed:
        Y -= Y.mean(axis=0)   # (packed path: centred on the device, like scale(Y, scale = FALSE) R/prepare_atlasqtl.R:83)
    tau0 = 1.0  # ~ 1 / median var(Y_k) of the recipe (unit noise); fixed so that every rank uses the same value
    hyper = hyper_init.set_hyper(q, p, tau0, 1.0, n0, 1e-2, 1.0, t02)
    r = np.random.default_rng(seed + 3)
    sig02_inv = float(r.gamma(shape=max(p, q), scale=1.0))
    init = dict(q_init=q, p_init=p, gam_vb=gam, mu_beta_vb=mu, sig02_inv_vb=sig02_inv,
                sig2_beta_vb=1 / r.gamma(shape=2.0, scale=1e-2 * tau0, size=q),
                sig2_theta_vb=1 / (q + r.gamma(shape=sig02_inv * q, scale=1.0, size=p)),
                tau_vb=np.full(q, tau0), theta_vb=r.normal(0.0, 1 / np.sqrt(sig02_inv * q), size=p),
                zeta_vb=r.normal(n0, np.sqrt(t02), size=q))
    return cfg, (dict(packed=G_packed, n=n) if packed else X), Y, hyper, init


def host_threads():
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return max(1, min(32, ncpu // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) == 6 and r[0].isdigit()]
        if not rows:
            return None
        sm = sorted(int(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": reasons, "samples": len(rows)}


# ----------------------------------------------------------------------------- CPU arms
def reference_sample(cfg, X, Y, hyper, init, p_s=8192, traits_per_thread=1, threads=None, steps=2, warmup=1):
    """Time the reference's own coreDualLoop on a bounded sample: the first p_s SNPs (its p x p Gram of the full
    p does not fit / cannot be formed in minutes) x `threads * traits_per_thread` traits, one disjoint sample_q
    range per host thread (traits are independent, so concurrent calls on disjoint columns are valid)."""
    from concurrent.futures import ThreadPoolExecutor

    from scipy import special as sp

    from oracle import native
    threads = threads or (os.cpu_count() or 1)
    n, p = cfg["n"], cfg["p"]
    p_s = min(p, p_s)
    q_s = min(Y.shape[1], threads * traits_per_thread)
    Xs = dense_columns(X, 0, p_s)
    Ys = np.asfortranarray(Y[:, :q_s] - Y[:, :q_s].mean(axis=0))
    kind = "reference" if native.ref_available() else "port"
    impl = "reference" if kind == "reference" else "oracle"
    t0 = time.time()
    cp_X = np.asfortranarray(Xs.T @ Xs)
    cp_Y_X = np.asfortranarray(Ys.T @ Xs)
    gam = np.asfortranarray(init["gam_vb"][:p_s, :q_s].copy())
    mu = np.asfortranarray(init["mu_beta_vb"][:p_s, :q_s].copy())
    beta = np.asfortranarray(gam * mu)
    cbx = np.asfortranarray(cp_X @ beta)
    setup_s = time.time() - t0
    u = init["theta_vb"][:p_s, None] + init["zeta_vb"][None, :q_s]
    lp, lq = np.asfortranarray(sp.log_ndtr(u)), np.asfortranarray(sp.log_ndtr(-u))
    tau = np.ascontiguousarray(init["tau_vb"][:q_s])
    sig2 = 1.0 / ((n - 1 + 1.0) * tau)
    log_tau = np.log(tau)
    order = np.arange(p_s, dtype=np.int32)
    ranges = [np.arange(t * q_s // threads, (t + 1) * q_s // threads, dtype=np.int32) for t in range(threads)]
    ranges = [r for r in ranges if len(r)]

    def one(rng_q):
        native.core_dual_loop(cp_X, cp_Y_X, gam, lp, lq, 0.0, log_tau, beta, cbx, mu, sig2, tau, order, rng_q,
                              c=1.0, impl=impl)

    times = []
    with ThreadPoolExecutor(len(ranges)) as ex:
        for s in range(warmup + steps):
            t0 = time.time()
            list(ex.map(one, ranges))
            dt = time.time() - t0
            if s >= warmup:
                times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = p_s * q_s / (ms / 1e3)
    return dict(value=value, unit="SNPxtrait updates/s", cores=len(ranges), kind=kind, ms_per_step=ms,
                outputs=dict(gam_vb=gam, mu_beta_vb=mu, beta_vb=beta),
                sample=f"coreDualLoop (dual/Gram form, as the reference runs it), n={n}, first {p_s} of {p} SNPs x "
                       f"{q_s} traits, {len(ranges)} host threads on disjoint sample_q ranges; Gram set-up {setup_s:.1f} s "
                       f"not timed; dual-form cost per update grows with p, so at the full p this is ~{p_s / p:.3g}x",
                value_at_full_p_est=value * p_s / p)


def dense_columns(X, j0, j1):
    """Standardised columns [j0, j1) of the workload's X as a dense Fortran matrix (unpacks 2-bit calls if need be)."""
    if not isinstance(X, dict):
        return np.asfortranarray(X[:, j0:j1])
    g = X["packed"][j0:j1]
    n = X["n"]
    G = np.stack([(g >> s) & 3 for s in (0, 2, 4, 6)], axis=2).reshape(g.shape[0], -1)[:, :n].T.astype(np.float64)
    return np.asfortranarray((G - G.mean(axis=0)) / G.std(axis=0, ddof=1))


def port_sample(X, Y, init, threads=None, target_s=6.0):
    """Best-effort CPU (ours, primal form, all host threads) on a q-slice of the full-n, full-p workload."""
    from scipy import special as sp

    from oracle import native
    threads = threads or (os.cpu_count() or 1)
    if isinstance(X, dict):
        raise ValueError("port_sample needs the dense X")
    n, p = X.shape
    q_s = min(Y.shape[1], max(threads, int(target_s * threads * 1.5e9 / (4.0 * n * p))))
    Ys = np.asfortranarray(Y[:, :q_s])
    gam = np.asfortranarray(init["gam_vb"][:, :q_s].copy())
    mu = np.asfortranarray(init["mu_beta_vb"][:, :q_s].copy())
    beta = np.asfortranarray(gam * mu)
    R = native.residual(X, Ys, beta)
    xn = np.asfortranarray(np.sum(X ** 2, axis=0))
    u = init["theta_vb"][:, None] + init["zeta_vb"][None, :q_s]
    lp, lq = np.asfortranarray(sp.log_ndtr(u)), np.asfortranarray(sp.log_ndtr(-u))
    tau = np.ascontiguousarray(init["tau_vb"][:q_s])
    sig2 = 1.0 / ((n - 1 + 1.0) * tau)
    t0 = time.time()
    native.sweep_primal(X, xn, R, gam, lp, lq, 0.0, np.log(tau), beta, mu, sig2, tau, np.arange(p, dtype=np.int32),
                        c=1.0, nthreads=threads)
    dt = time.time() - t0
    return dict(value=p * q_s / dt, unit="SNPxtrait updates/s", cores=threads, kind="port",
                sample=f"oracle primal sweep, n={n}, p={p}, {q_s} traits, {threads} threads, {dt:.1f} s")


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C2")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--na-frac", type=float, default=0.0,
                    help="fraction of missing responses (NaN in Y): times the coreDualMisLoop path instead of coreDualLoop")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path computed in its last step to DIR/<name>.npy (see the module doc)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    # stdout carries the ONE JSON line and nothing else: whatever libraries print there (NCCL's version banner, ...) is
    # sent to stderr by pointing fd 1 at fd 2 for the run; the line itself goes to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    W, K = args.warmup, args.steps

    from atlasqtl_b200 import synthetic
    from atlasqtl_b200.dist import slab_bounds
    cfg0 = synthetic.CONFIGS[args.config]
    n, p, q = cfg0["n"], cfg0["p"], cfg0["q"]
    anneal = cfg0.get("anneal")
    config = {"workload": f"{args.config}: synthetic n={n}, p={p} SNPs, q={q} traits, anneal={anneal}, fp64; "
                          f"first {W}+{K} VB iterations", "n": n, "p": p, "q": q,
              "l2": "inputs larger than L2 (p x q arrays stream from HBM every step)",
              "parallelism": f"traits sharded over {world} GPU(s), X replicated"}
    if args.na_frac > 0:
        config["workload"] += f"; {100 * args.na_frac:g} % of the responses missing at random (coreDualMisLoop path)"
        config["na_frac"] = args.na_frac

    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import native
        native.build()
        ncpu = os.cpu_count() or 1
        ws = make_workload(args.config, 0, min(q, 4 * ncpu))
        res = reference_sample(*ws, steps=K, warmup=W)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res["outputs"])
        # the reference's dual form needs the p x p Gram matrix (20 GB at C2) and O(p) work per update: it is timed on a
        # bounded SAMPLE of the workload, and the line says so where the config is named
        config["workload"] += f" -- REFERENCE ARM TIMES A SAMPLE: {res['sample']}"
        line = {"impl": "reference", "metric": "SNPxtrait CAVI updates/s", "value": res["value"],
                "unit": "updates/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": res["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "value_at_full_p_est": res["value_at_full_p_est"],
                "e2e": {"value": res["value"], "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    from atlasqtl_b200 import core
    from atlasqtl_b200.device import PreparedPredictors, SweepContext
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the hot path")
    torch.cuda.set_device(local_rank)
    comm = None
    if world > 1:
        import torch.distributed as dist
        from atlasqtl_b200.dist import TorchComm
        # NCCL writes its debug output (the version banner at NCCL_DEBUG=VERSION / WARN) to stdout: send it to stderr so
        # that stdout carries the ONE JSON line only
        # (NCCL honours NCCL_DEBUG_FILE only above the VERSION level)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        comm = TorchComm()
    k0, k1 = slab_bounds(q, rank, world)
    ql = k1 - k0
    # memory plan of this rank (bytes): five p x q_local arrays + X (tiled; the untiled copy is released) -- refuse early
    # rather than drive the GPU out of memory
    need = 5 * 8.0 * p * ql + 1.15 * 8.0 * n * p * 2 + 16.0 * n * ql
    free_b, total_b = torch.cuda.mem_get_info()
    if need > 0.97 * free_b:
        raise SystemExit(f"{args.config} on {world} GPU(s) needs ~{need / 2**30:.0f} GiB per GPU, {free_b / 2**30:.0f} GiB free: "
                         "use more GPUs (the traits are sharded, X is replicated)")
    # ... and the host: every rank builds its slab's initial state (two p x q_local matrices) and X in host memory
    try:
        import psutil
        avail = psutil.virtual_memory().available
        local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
        host_need = (2 * 8.0 * p * ql * 1.3 + min(8.0 * n * p, PACKED_ABOVE_BYTES) + 0.3 * n * p) * local_world
        if host_need > 0.85 * avail:
            raise SystemExit(f"{args.config} on {world} GPU(s) needs ~{host_need / 2**30:.0f} GiB of host memory to build the "
                             f"synthetic state, {avail / 2**30:.0f} GiB available")
    except ImportError:
        pass
    t_setup = time.time()
    cfg, X, Y, hyper, init = make_workload(args.config, k0, k1)
    log(f"[rank {rank}] workload built in {time.time() - t_setup:.1f} s (slab {k0}:{k1}, "
        f"X {'packed 2-bit calls' if isinstance(X, dict) else 'dense'})")

    def barrier_sync():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
            torch.cuda.synchronize()

    marks, launches = {}, {}
    sampler = ClockSampler(local_rank)

    def hook(it, ctx):
        if it == W + 1:
            ctx.sync()
            barrier_sync()
            if rank == 0:
                sampler.start()
            launches["t0"] = ctx.launch_count()
            marks["t0"] = time.perf_counter()
        if it == W + K + 1:
            ctx.sync()
            barrier_sync()
            marks["t1"] = time.perf_counter()
            launches["t1"] = ctx.launch_count()

    if args.na_frac > 0:
        if isinstance(X, dict):
            raise SystemExit("--na-frac needs a dense-X config (C1, C2, C4)")
        # the same entries whatever the sharding: drawn per global chunk of 64 traits
        for c0 in range((k0 // 64) * 64, k1, 64):
            m = np.random.default_rng([123, 13, c0]).uniform(size=(64, n)) < args.na_frac
            lo, hi = max(c0, k0), min(c0 + 64, k1)
            Y[:, lo - k0:hi - k0][m[lo - c0:hi - c0].T] = np.nan
    trace = []
    t_up = time.time()
    if isinstance(X, dict):
        prep = PreparedPredictors(packed=X["packed"], n=X["n"], device=local_rank)
        if prep.p != p:
            raise SystemExit(f"device pre-processing kept {prep.p} of {p} SNPs (duplicates in the synthetic genotypes)")
        ctx = SweepContext.from_prepared(prep, Y)
        prep.close()
        Xarg = prep   # the core only asks for .shape
        if world > 1:
            X["packed"] = None   # (kept at N = 1 for the CPU baseline's sample)
    else:
        ctx = SweepContext(X, np.where(np.isnan(Y), 0.0, Y) if args.na_frac > 0 else Y, device=local_rank)
        Xarg = X
    log(f"[rank {rank}] context created in {time.time() - t_up:.1f} s")
    try:
        result = core.atlasqtl_global_local_core_(Y, Xarg, q, anneal, 1, 1e-300, W + K, 0, hyper, init, debug=False,
                                                  comm=comm, slab=(k0, k1), ctx=ctx, trace=trace, iter_hook=hook,
                                                  release_x=True)
        clocks = sampler.stop() if rank == 0 else None
        timed = [r for r in trace if W < r["it"] <= W + K]
        if len(timed) != K or "t1" not in marks:
            raise SystemExit(f"the run stopped after {result['it']} of {W + K} iterations: {len(timed)} of {K} steps timed")
        seg_keys = list(timed[0].get("host_ms", {})) if timed else []
        host_ms = np.array([np.mean([r["host_ms"].get(k, 0.0) for r in timed]) for k in seg_keys])
        dev_ms = sum(r["sweep_ms"] + r["rows_ms"] + r["tables_ms"] for r in timed)
        per = np.array([np.mean([r[k] for r in timed]) for k in ("sweep_ms", "rows_ms", "tables_ms")])
        wall_ms = 1e3 * (marks["t1"] - marks["t0"])
        red = np.concatenate([[dev_ms, wall_ms], per, host_ms])
        if world > 1:
            t = torch.tensor(red, device="cuda")
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            red = t.cpu().numpy()
        dev_ms, wall_ms = float(red[0]), float(red[1])
        sweep_ms, rows_ms, tables_ms = (float(v) for v in red[2:5])
        host_ms = red[5:]
        if rank == 0 and seg_keys:
            log("[host wall-clock per step, ms, max over ranks] " + ", ".join(f"{k}={v:.2f}" for k, v in zip(seg_keys, host_ms)))
        dims = ctx.dims()
        plan = ctx.sweep_plan()
        dev_reduce = world > 1 and callable(getattr(comm, "allreduce_sum_device", None))
        # per step: H2D tau / log_tau / sig2_beta (q_local each), theta (p), zeta (q_local) [+ the all-reduce message];
        # D2H the five column-sum vectors, the row sums (p), the ELBO scalar [+ the all-reduce result]
        h2d = 8 * (3 * ql + p + ql) + (8 * 2 if dev_reduce else (8 * (p + 2) if world > 1 else 0))
        d2h = 8 * (5 * dims["q_pad"] + p + 1) + (8 * 2 if dev_reduce else (8 * (p + 2) if world > 1 else 0))
        n_launch = launches["t1"] - launches["t0"]
        lbs = [r["lb"] for r in trace if r["lb"] is not None]
        check = {"lb_last": lbs[-1] if lbs else None, "lb_it": max((r["it"] for r in trace if r["lb"] is not None), default=None),
                 "sum_gam": trace[-1]["sum_gam"], "it": trace[-1]["it"],
                 "note": "global quantities after the last step (all-reduced over ranks): lines of the same config at "
                         "different GPU counts must agree to ~1e-10 relative"}
    finally:
        ctx.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: result[k] for k in ("gam_vb", "beta_vb", "zeta_vb")}
                     | ({"theta_vb": result["theta_vb"]} if rank == 0 else {}), rank, world)
    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    flops_per_sweep = 4.0 * n * p * ql  # algorithmic: 2n (X_j'r) + 2n (rank-1 update) per SNP x trait, this rank
    achieved = flops_per_sweep / (sweep_ms * 1e-3) / 1e12
    traffic, traffic_src = ncu_traffic(args.config, world)
    line = {"metric": "SNPxtrait CAVI updates/s", "value": p * q * K / (dev_ms * 1e-3), "unit": "updates/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "e2e": {"value": p * q * K / (wall_ms * 1e-3), "unit": "updates/s", "ms_per_step": wall_ms / K,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(n_launch),
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                         "frac": achieved / FP64_PEAK_TFLOPS,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "traffic_algorithmic": 56.0 * p * ql + 8.0 * n * p + 16.0 * n * ql,
                         "kernel": "sweep_kernel (fp64 DMMA m8n8k4), one sweep of this rank's trait slab"
                                   + (" -- missing-response variant (masked accumulators, per-trait Gram band)" if args.na_frac > 0 else ""),
                         "ms": sweep_ms, "plan": plan,
                         "peak_source": "measured fp64 DMMA peak, tools/microbench/fp64_peaks.cu on this pool "
                                        "(MEASURED_PEAKS.json has no fp64 entry)",
                         "algorithmic": "4*n flops per SNPxtrait update; HBM: 56 B per update (read gam, mu, D, W, I0; write "
                                        "gam, mu: one table more than the reference's 48 B, W / I0 replace its two log-CDF "
                                        "tables plus the Z pass) + X once + residual in / out"},
            "clocks": clocks, "check": check,
            "per_step_ms": {"sweep": sweep_ms, "rowsums": rows_ms, "tables": tables_ms,
                            "host": {k: float(v) for k, v in zip(seg_keys, host_ms)}, "over_ranks": "max"}}
    if args.na_frac > 0:
        line["cpu_baseline"] = {"skipped": "the CPU arm times coreDualLoop (no missing responses); see the default run"}
    elif world == 1 and not args.no_cpu_baseline:
        try:
            from oracle import native
            native.build()
            ref = reference_sample(cfg, X, Y, hyper, init, steps=2, warmup=1)
            line["cpu_baseline"] = {k: ref[k] for k in ("value", "unit", "cores", "kind", "sample")}
            line["cpu_baseline"]["value_at_full_p_est"] = ref["value_at_full_p_est"]
            if not isinstance(X, dict):
                line["cpu_port"] = port_sample(X, Y, init)
        except Exception as e:  # the baseline is a report, never the product path
            line["cpu_baseline"] = {"error": repr(e)}
    emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
