"""Stored outputs of the reference's own sweep loop (src/coreLoop.cpp's coreDualLoop) for the test problems that
are compared against it, so that those tests need nothing outside the repository.

    python tests/reference_runs.py        # rewrites tests/golden/reference_runs.npz

Inputs are not stored: every case rebuilds them from tests/problems.py exactly as its test does, and `in_check`
(checksums of the inputs) lets a test tell "inputs drifted" from "results differ".  The loop that runs is the
reference's library (oracle/_ref) where it is present; elsewhere it is the dual restatement in oracle/cavi_oracle.c,
and only after the restatement has reproduced the reference's committed outputs (tests/golden/coredualloop_*.npz)
bit for bit.  `source` in the file says which one ran.

A p x q matrix of more than SAMPLE_ABOVE entries (a residual: more than SAMPLE) is kept as a fixed, seeded sample
of SAMPLE entries (column-major positions in `index` / `R_index`) so that the file stays small; the selection sets
({gam_vb > 0.5}, {bFDR < 0.05}), the column / row sums and the ELBO trajectory are kept whole.
"""
import glob
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
if os.path.dirname(HERE) not in sys.path:
    sys.path.insert(0, os.path.dirname(HERE))
PATH = os.path.join(HERE, "golden", "reference_runs.npz")
SAMPLE_ABOVE = 1024
SAMPLE = 512
LOG_SQRT_2PI = 0.5 * np.log(2 * np.pi)

HOST_ANNEALS = [None, (1, 2, 10), (2, 3, 5), (3, 2, 4)]
FULL_RUNS = [(100, 75, 20, (1, 2, 10)), (100, 75, 20, None), (200, 300, 200, (1, 2, 10))]
SWEEPS = [(100, 75, 20, 1.0, False), (100, 75, 20, 0.6, True), (200, 300, 200, 0.8, True)]


def key(*parts):
    return "_".join("-".join(map(str, x)) if isinstance(x, tuple) else str(x) for x in parts)


def in_check(X, Y, init=None):
    """Checksums of a case's inputs (sums of magnitudes: none of them is close to zero)."""
    v = [np.abs(X).sum(), (X ** 2).sum(), np.abs(Y).sum(), (Y ** 2).sum()]
    if init is not None:
        v += [np.abs(init[k]).sum() for k in ("gam_vb", "mu_beta_vb", "theta_vb", "zeta_vb")]
    return np.array(v)


# ----------------------------------------------------------------------------- what the tests compare against
def oracle_sweep(native, X, Y, si, order, form):
    """One sweep on the CPU: "reference" / "dual" (the reference's coreDualLoop / its restatement, Gram form) or
    "primal" (sample space).  Returns gam_vb, mu_beta_vb, beta_vb and the residual Y - X beta_vb."""
    gam, mu = si["gam"].copy(order="F"), si["mu"].copy(order="F")
    beta = np.asfortranarray(gam * mu)
    q = Y.shape[1]
    if form in ("reference", "dual"):
        cp_X = np.asfortranarray(X.T @ X)
        cp_Y_X = np.asfortranarray(Y.T @ X)
        cbx = np.asfortranarray(cp_X @ beta)
        native.core_dual_loop(cp_X, cp_Y_X, gam, si["log_Phi"], si["log_1_min_Phi"], si["log_sig2_inv"], si["log_tau"],
                              beta, cbx, mu, si["sig2_beta"], si["tau"], order, np.arange(q, dtype=np.int32),
                              c=si["c"], impl="reference" if form == "reference" else "oracle")
        R = np.asfortranarray(Y - X @ beta)
    else:
        R = native.residual(X, Y, beta)
        xn = np.asfortranarray(np.sum(X ** 2, axis=0))
        native.sweep_primal(X, xn, R, gam, si["log_Phi"], si["log_1_min_Phi"], si["log_sig2_inv"], si["log_tau"], beta,
                            mu, si["sig2_beta"], si["tau"], order, c=si["c"], nthreads=4)
    return gam, mu, beta, R


def zparts(si, gam):
    """Column and row sums of the gam-dependent part of Z (R/update_vb.R:219-229) after a sweep."""
    from scipy import special as sp
    u = si["theta"][:, None] + si["zeta"][None, :]
    sc = 1.0 if abs(si["c"] - 1) < 1.5e-8 else np.sqrt(si["c"])
    U = sc * u
    lp, lq = sp.log_ndtr(U), sp.log_ndtr(-U)
    m1 = np.exp(-U ** 2 / 2 - LOG_SQRT_2PI - lp)
    m1 = np.where(m1 < -U, -U, m1)
    m0 = -np.exp(-U ** 2 / 2 - LOG_SQRT_2PI - lq)
    m0 = np.where(m0 > -U, -U, m0)
    zp = gam * (m1 - m0) + m0
    return zp.sum(axis=0), zp.sum(axis=1)


def sample_index(shape, seed=0, above=SAMPLE_ABOVE):
    size = int(np.prod(shape))
    if size <= above:
        return None
    return np.sort(np.random.default_rng(seed).choice(size, SAMPLE, replace=False)).astype(np.int32)


def _picker(index):
    if index is None:
        return lambda a: np.asarray(a)
    return lambda a: np.asarray(a).ravel(order="F")[index]


def sweep_summary(si, gam, mu, beta, R, sample=True):
    """What a test of one sweep compares: the entries of gam / mu / beta (all, or a sample) and a sample of R, the
    largest |mu|, |beta| and the per-trait / per-SNP sums the sweep returns."""
    zc, zr = zparts(si, gam)
    d = dict(colsum_gam=gam.sum(axis=0), colsum_beta2=(beta ** 2).sum(axis=0), colsum_gam_mu2=(gam * mu ** 2).sum(axis=0),
             resid_sq=(R ** 2).sum(axis=0), colsum_zpart=zc, rowsum_zpart=zr, mu_absmax=np.abs(mu).max(),
             beta_absmax=np.abs(beta).max())
    idx = sample_index(gam.shape) if sample else None
    d.update(gam=_picker(idx)(gam), mu=_picker(idx)(mu), beta=_picker(idx)(beta))
    r_idx = sample_index(R.shape, above=SAMPLE) if sample else None
    d["R"] = _picker(r_idx)(R)
    for name, i in (("index", idx), ("R_index", r_idx)):
        if i is not None:
            d[name] = i
    return d


def run_summary(out, trace, sample=True, beta=True):
    """What a test of a full run compares: iteration count, ELBO trajectory, final parameters (gam_vb / beta_vb
    entries: all or a sample; beta_vb only if `beta`) and the selection sets."""
    from oracle import vb_oracle
    gam = out["gam_vb"]
    d = dict(it=out["it"], converged=out["converged"], trace_it=np.array([r["it"] for r in trace]),
             trace_c=np.array([r["c"] for r in trace]),
             trace_lb=np.array([np.nan if r["lb"] is None else r["lb"] for r in trace]),
             theta_vb=out["theta_vb"], zeta_vb=out["zeta_vb"], sel=gam > 0.5, sel_bfdr=vb_oracle.assign_bFDR(gam) < 0.05)
    idx = sample_index(gam.shape) if sample else None
    d["gam_vb"] = _picker(idx)(gam)
    if beta:
        d["beta_vb"] = _picker(idx)(out["beta_vb"])
    if idx is not None:
        d["index"] = idx
    return d


def with_views(d):
    """`pick` / `pick_R` (full matrix -> the stored entries of the p x q outputs / of the residual) and `trace` (the
    oracle's per-iteration records)."""
    d = dict(d)
    d["pick"] = _picker(d.get("index"))
    d["pick_R"] = _picker(d.get("R_index"))
    if "trace_it" in d:
        d["trace"] = [dict(it=int(i), c=float(c), lb=None if np.isnan(lb) else float(lb))
                      for i, c, lb in zip(d["trace_it"], d["trace_c"], d["trace_lb"])]
    return d


def load(*parts):
    """The stored case `key(*parts)` as a dict (see run_summary / sweep_summary), with `pick` and `trace`."""
    name = key(*parts)
    with np.load(PATH) as f:
        d = {k[len(name) + 2:]: f[k] for k in f.files if k.startswith(name + "__")}
    if not d:
        raise KeyError(f"{name} is not in {PATH}")
    return with_views(d)


# ----------------------------------------------------------------------------- the cases
def host_problem():
    from problems import make_problem
    return make_problem(100, 75, 20, p_act=10, q_act=20, maf=0.2, p0=(5, 25))


def order_problem():
    from problems import make_problem
    return make_problem(100, 60, 12, p_act=6, q_act=12)


def order_perm(it, p):
    return np.random.default_rng(it).permutation(p).astype(np.int32)


def saturated_inputs():
    """The sweep driven into saturation (test_gpu_logistic.py): theta + zeta at +-30, effects scaled by 40."""
    from scipy import special as sp

    from problems import make_problem, sweep_inputs
    X, Y, hyper, init = make_problem(120, 60, 24)
    p, q = X.shape[1], Y.shape[1]
    Y = np.asfortranarray(Y * 40.0)
    si = sweep_inputs(X, Y, init, c=1.0)
    rng = np.random.default_rng(3)
    si["theta"] = rng.choice([-30.0, 0.0, 9.0], size=p)
    si["zeta"] = rng.choice([-8.0, 0.0, 3.0], size=q)
    u = si["theta"][:, None] + si["zeta"][None, :]
    si["log_Phi"], si["log_1_min_Phi"] = np.asfortranarray(sp.log_ndtr(u)), np.asfortranarray(sp.log_ndtr(-u))
    return X, Y, si, np.arange(p, dtype=np.int32)


def generate(form):
    from oracle import native, vb_oracle
    from problems import make_problem, sweep_inputs
    cases = {}

    def run(name, X, Y, hyper, init, anneal, maxit, beta=True, **kw):
        tr = []
        out = vb_oracle.atlasqtl_global_local_core_(Y, X, Y.shape[1], anneal, 1, 0.1, maxit, hyper, init, sweep=form,
                                                    trace=tr, **kw)
        cases[name] = dict(run_summary(out, tr, beta=beta), in_check=in_check(X, Y, init))
        print(name, "it", out["it"], flush=True)

    for anneal in HOST_ANNEALS:
        run(key("host", anneal), *host_problem(), anneal, 1000, beta=False)
    X, Y, hyper, init = order_problem()
    run(key("order", "perm"), X, Y, hyper, init, None, 50, beta=False, perm_fn=order_perm)
    run(key("order", "identity"), X, Y, hyper, init, None, 50, beta=False)
    for n, p, q, anneal in FULL_RUNS:
        run(key("full", n, p, q, anneal), *make_problem(n, p, q), anneal, 1000)
    for n, p, q, c, shuffle in SWEEPS:
        X, Y, hyper, init = make_problem(n, p, q)
        si = sweep_inputs(X, Y, init, c=c)
        order = (np.random.default_rng(5).permutation(X.shape[1]) if shuffle else np.arange(X.shape[1])).astype(np.int32)
        cases[key("sweep", n, p, q, c, shuffle)] = dict(sweep_summary(si, *oracle_sweep(native, X, Y, si, order, form)),
                                                        in_check=in_check(X, Y, init))
    X, Y, si, order = saturated_inputs()
    cases[key("saturated")] = dict(sweep_summary(si, *oracle_sweep(native, X, Y, si, order, form)), in_check=in_check(X, Y))
    return cases


def certify_restatement():
    """The dual restatement must reproduce every committed output of the reference's coreDualLoop bit for bit."""
    from oracle import native
    paths = sorted(glob.glob(os.path.join(HERE, "golden", "coredualloop_*.npz")))
    assert paths
    for path in paths:
        d = dict(np.load(path))
        X, Y = d["X"], d["Y"]
        gam, mu = np.array(d["gam"], order="F"), np.array(d["mu"], order="F")
        beta = np.asfortranarray(gam * mu)
        cp_X, cp_Y_X = np.asfortranarray(X.T @ X), np.asfortranarray(Y.T @ X)
        cbx = np.asfortranarray(cp_X @ beta)
        native.core_dual_loop(cp_X, cp_Y_X, gam, np.asfortranarray(d["log_Phi"]), np.asfortranarray(d["log_1_min_Phi"]),
                              float(d["log_sig2_inv"]), d["log_tau"], beta, cbx, mu, d["sig2_beta"], d["tau"], d["order"],
                              np.arange(Y.shape[1], dtype=np.int32), c=float(d["c"]), impl="oracle")
        for a, b in ((gam, "out_gam"), (mu, "out_mu"), (beta, "out_beta"), (cbx, "out_cp_betaX_X")):
            if not np.array_equal(a, d[b]):
                raise SystemExit(f"the dual restatement no longer reproduces {os.path.basename(path)}:{b}")


def main():
    from oracle import native
    native.build()
    if native.ref_available():
        form, source = "reference", "the reference's coreDualLoop (oracle/_ref)"
    else:
        certify_restatement()
        form, source = "dual", ("oracle/cavi_oracle.c's dual restatement of the reference's coreDualLoop, bit-exact on "
                                "tests/golden/coredualloop_*.npz")
    cases = generate(form)
    flat = {f"{name}__{k}": np.asarray(v) for name, d in cases.items() for k, v in d.items()}
    np.savez_compressed(PATH, source=source, **flat)
    print(f"wrote {PATH} ({os.path.getsize(PATH)} bytes) from {source}")


if __name__ == "__main__":
    main()
