"""Golden vectors of the reference's OWN R code (outer loop, ELBO, pre-processing, bFDR) -- TEST INFRASTRUCTURE ONLY.

  python tests/golden/make_rlite_golden.py            -> tests/golden/rlite_*.npz

R is not installed in this image, so the reference's R sources are executed, unmodified and from where they lie
under /root/reference/R, by the small R evaluator in oracle/rlite (parser + evaluator + the base / stats / gsl
functions those files call, SciPy standing in for nmath / gsl); `.Call(_atlasqtl_coreDualLoop / coreDualMisLoop)` is
the reference's own src/coreLoop.cpp (oracle/_ref).  Every statement executed is the reference's; this script only
supplies inputs and stores outputs.  The inputs are stored in the files, so the fixtures do not depend on any
generator stream.  The GPU box has no /root/reference: it only reads the .npz.

Files
  rlite_core_<case>.npz   atlasqtl_global_local_core_ (R/atlasqtl_global_local_core.R:8-433) run to convergence:
                          inputs, ELBO at every evaluation (elbo_global_local_, :440-495), it, converged, lb_opt,
                          diff_lb, gam_vb, beta_vb, theta_vb, zeta_vb and the full_output internals
  rlite_atlasqtl_top.npz  atlasqtl() (R/atlasqtl.R:179-322) on RAW X / Y with constant and duplicated columns and
                          missing responses: prepare_data_ outputs + the run
  rlite_functions.npz     function-level probes: get_annealing_ladder_, Q_approx_vec, update_annealed_lam2_inv_vb_,
                          inv_mills_ratio_, update_Z_, log_one_plus_exp_, assign_bFDR, auto_set_hyper_, e_* ELBO terms
  rlite_c1.npz            BASELINE config C1 (n=200, p=500, q=1000, no annealing) through the same route: ELBO
                          sequence, it, probes -- the existing c1_trajectory.npz (made by oracle/vb_oracle.py) must
                          agree with it (tests/test_rlite.py)
  rlite_c4.npz            BASELINE config C4 (n=500, p=10000, q=5000, 20 hotspots, annealing; `c4`, not in the default
                          list: ~1.5 h with RLITE_REF_THREADS=8) -- same check against c4_trajectory.npz, incl. the
                          {bFDR < 0.05} set formed by the reference's own assign_bFDR
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
HERE = os.path.dirname(os.path.abspath(__file__))

HYPER_KEYS = ("q_hyper", "p_hyper", "A2_inv", "eta", "kappa", "m0", "n0", "nu", "rho", "t02")
INIT_KEYS = ("q_init", "p_init", "gam_vb", "mu_beta_vb", "sig02_inv_vb", "sig2_beta_vb", "sig2_theta_vb", "tau_vb",
             "theta_vb", "zeta_vb")

# name: (n, p, q, anneal, thinned_elbo_eval, NA fraction, tol, seed)
CORE_CASES = {
    "a_noanneal": (100, 75, 20, None, True, 0.0, 0.1, 11),
    "b_geometric": (100, 75, 20, (1, 2, 10), True, 0.0, 0.1, 12),
    "c_harmonic_unthinned": (120, 60, 24, (2, 3, 7), False, 0.0, 0.1, 13),
    "d_linear": (90, 50, 16, (3, 2.5, 6), True, 0.0, 0.01, 14),
    "e_missing_anneal": (100, 60, 18, (1, 2, 5), True, 0.07, 0.1, 15),
    "f_missing_noanneal": (80, 40, 12, None, True, 0.15, 0.1, 16),
    "g_wide": (200, 300, 120, (1, 2, 10), True, 0.0, 0.1, 17),
}


def plain(d, keys):
    return {k: d[k] for k in keys}


def core_case(name):
    from problems import make_problem
    n, p, q, anneal, thinned, na, tol, seed = CORE_CASES[name]
    X, Y, hyper, init = make_problem(n, p, q, seed=seed)
    if na > 0:
        Y = Y.copy()
        Y[np.random.default_rng(seed).uniform(size=Y.shape) < na] = np.nan
        Y = np.asfortranarray(Y - np.nanmean(Y, axis=0))
    return X, Y, plain(hyper, HYPER_KEYS), plain(init, INIT_KEYS), anneal, thinned, tol


def run_core(it, X, Y, hyper, init, anneal, thinned, tol, maxit=1000):
    from oracle.rlite import reference as R
    q = Y.shape[1]
    lbs = []
    out = R.global_local_core(Y, X, q, anneal, 1, tol, maxit, hyper, init, it=it, hook=lambda n, v: lbs.append(v),
                              thinned_elbo_eval=bool(thinned), debug=True)
    full = R.global_local_core(Y, X, q, anneal, 1, tol, maxit, hyper, init, it=it, thinned_elbo_eval=bool(thinned),
                               debug=True, full_output=True)
    res = dict(lb=np.array(lbs), it=int(out["it"][0]), converged=bool(out["converged"][0]),
               lb_opt=float(out["lb_opt"][0]), diff_lb=float(out["diff_lb"][0]), gam_vb=out["gam_vb"],
               beta_vb=out["beta_vb"], theta_vb=out["theta_vb"], zeta_vb=out["zeta_vb"])
    for k in ("eta_vb", "kappa_vb", "lam2_inv_vb", "nu_s0_vb", "nu_vb", "rho_s0_vb", "rho_vb", "rho_xi_inv_vb",
              "sig02_inv_vb", "sig2_beta_vb", "sig2_inv_vb", "sig2_theta_vb", "sig2_zeta_vb", "tau_vb", "xi_inv_vb"):
        res["full_" + k] = np.asarray(full[k], dtype=np.float64)
    assert np.array_equal(full["gam_vb"], out["gam_vb"])
    return res


MAX_FILE_BYTES = 1_000_000
SPLIT_KEYS = ("init_gam_vb", "init_mu_beta_vb")


def save(name, **arrays):
    dest = os.path.join(HERE, name)
    np.savez_compressed(dest, **arrays)
    if name.startswith("rlite_core_") and os.path.getsize(dest) > MAX_FILE_BYTES:
        # keep every file under 1 MB: the initial p x q matrices go to rlite_init_<case>.npz (tests/rlite_cases.py
        # merges it back)
        save("rlite_init_" + name[len("rlite_core_"):], **{k: arrays[k] for k in SPLIT_KEYS})
        np.savez_compressed(dest, **{k: v for k, v in arrays.items() if k not in SPLIT_KEYS})
    print(f"wrote {dest} ({os.path.getsize(dest) / 1024:.0f} KiB)", flush=True)


def flat_inputs(X, Y, hyper, init, anneal, thinned, tol):
    d = dict(X=X, Y=Y, anneal=np.array([np.nan] if anneal is None else anneal, dtype=np.float64),
             thinned=bool(thinned), tol=float(tol))
    d.update({"hyper_" + k: np.asarray(v) for k, v in hyper.items()})
    d.update({"init_" + k: np.asarray(v) for k, v in init.items()})
    return d


def make_core(it):
    for name in CORE_CASES:
        t0 = time.time()
        X, Y, hyper, init, anneal, thinned, tol = core_case(name)
        res = run_core(it, X, Y, hyper, init, anneal, thinned, tol)
        assert res["converged"], name
        print(f"  {name}: it={res['it']} evaluations={len(res['lb'])} lb_opt={res['lb_opt']:.6f} "
              f"warnings={len(it.warnings)} [{time.time() - t0:.1f} s]", flush=True)
        save(f"rlite_core_{name}.npz", **flat_inputs(X, Y, hyper, init, anneal, thinned, tol), **res)


def raw_problem(seed=21, n=90, p_raw=70, q=14):
    """Raw genotype calls with constant and duplicated columns (one triplicate), raw responses with NAs."""
    rng = np.random.default_rng(seed)
    G = rng.binomial(2, 0.25, size=(n, p_raw)).astype(np.float64)
    G[:, 5] = 1.0                   # constant
    G[:, 40] = 0.0                  # constant
    G[:, 12] = G[:, 3]              # duplicate of an earlier column
    G[:, 33] = 2 - G[:, 3]          # NOT a duplicate after scaling (sign flips)
    G[:, 50] = G[:, 20]
    G[:, 61] = G[:, 20]             # triplicate
    G[:, 66] = 2 * G[:, 7]          # equal to column 7 once standardised, up to rounding: may or may not be bitwise equal
    beta = np.zeros((p_raw, q))
    act = rng.choice(p_raw, size=8, replace=False)
    beta[act] = rng.normal(0, 0.6, size=(8, q)) * (rng.uniform(size=(8, q)) < 0.5)
    Y = G @ beta + rng.normal(size=(n, q)) + 3.0
    Y[rng.uniform(size=Y.shape) < 0.05] = np.nan
    return np.asfortranarray(G), np.asfortranarray(Y)


def make_top(it):
    from atlasqtl_b200 import hyper_init
    from oracle.rlite import reference as R
    from oracle.rlite.values import from_py, to_py
    X, Y = raw_problem()
    prep = it.call("prepare_data_", R._copy_in(Y), R._copy_in(X), from_py(0.1), from_py(1000.0), None, from_py(0.0),
                   None, None)
    Xp, Yp = prep.get("X").a, prep.get("Y").a
    p, q = Xp.shape[1], Yp.shape[1]
    p0 = (3.0, 10.0)
    hyper = plain(hyper_init.auto_set_hyper_(Yp, p, p0), HYPER_KEYS)
    init = plain(hyper_init.auto_set_init_(Yp, p, p0, q, user_seed=5), INIT_KEYS)
    rm_coll = prep.get("rmvd_coll_x")
    lbs = []
    orig = it.globalenv.vars["elbo_global_local_"]
    from oracle.rlite.values import Builtin

    def traced(it_, pos, named):
        v = it_.apply(orig, pos, named, it_.globalenv)
        lbs.append(float(v.a[0]))
        return v
    it.globalenv.vars["elbo_global_local_"] = Builtin(traced, "elbo_global_local_")
    anneal = (1, 2, 5)
    out = it.call("atlasqtl", Y=R._copy_in(Y), X=R._copy_in(X), p0=None, anneal=from_py(np.array(anneal, float)),
                  tol=from_py(0.1), maxit=from_py(1000.0), verbose=from_py(0.0),
                  list_hyper=R.with_class(R._copy_in(hyper), "out_hyper"),
                  list_init=R.with_class(R._copy_in(init), "out_init"))
    it.globalenv.vars["elbo_global_local_"] = orig
    o = to_py(out)
    assert bool(o["converged"][0])
    # the same call with add_collinear_back = TRUE (add_collinear_back_, R/utils.R:680-735): one row per non-constant
    # predictor again, a removed duplicate carrying the rows of the predictor it duplicates
    cb = it.call("atlasqtl", Y=R._copy_in(Y), X=R._copy_in(X), p0=None, anneal=from_py(np.array(anneal, float)),
                 tol=from_py(0.1), maxit=from_py(1000.0), verbose=from_py(0.0),
                 list_hyper=R.with_class(R._copy_in(hyper), "out_hyper"),
                 list_init=R.with_class(R._copy_in(init), "out_init"), add_collinear_back=from_py(True))
    cb_names = np.array(cb.get("gam_vb").dimnames[0], dtype="U")
    assert list(cb.get("theta_vb").names) == list(cb_names)
    print(f"  atlasqtl(): p_raw={X.shape[1]} -> p={p}, removed constant {list(prep.get('rmvd_cst_x').a)}, collinear "
          f"{list(rm_coll.a)} (kept {rm_coll.names}); it={int(o['it'][0])}", flush=True)
    save("rlite_atlasqtl_top.npz", X_raw=X, Y_raw=Y, anneal=np.array(anneal, float), tol=0.1,
         prep_X=Xp, prep_Y=Yp, prep_bool_rmvd_x=prep.get("bool_rmvd_x").a,
         prep_rmvd_cst_x=np.array(list(prep.get("rmvd_cst_x").a), dtype="U"),
         prep_rmvd_coll_x=np.array(list(rm_coll.a), dtype="U"), prep_rmvd_coll_kept=np.array(rm_coll.names, dtype="U"),
         prep_initial_colnames_X=np.array(list(prep.get("initial_colnames_X").a), dtype="U"),
         names_x=np.array(out.get("gam_vb").dimnames[0], dtype="U"), names_y=np.array(out.get("gam_vb").dimnames[1], dtype="U"),
         **{"hyper_" + k: np.asarray(v) for k, v in hyper.items()}, **{"init_" + k: np.asarray(v) for k, v in init.items()},
         lb=np.array(lbs), it=int(o["it"][0]), converged=True, lb_opt=float(o["lb_opt"][0]), diff_lb=float(o["diff_lb"][0]),
         gam_vb=o["gam_vb"], beta_vb=o["beta_vb"], theta_vb=o["theta_vb"], zeta_vb=o["zeta_vb"],
         cb_names_x=cb_names, cb_gam_vb=cb.get("gam_vb").a, cb_beta_vb=cb.get("beta_vb").a, cb_theta_vb=cb.get("theta_vb").a)


def make_functions(it):
    from oracle.rlite.values import from_py
    rng = np.random.default_rng(31)
    out = {}
    ladders = [(1, 2, 10), (2, 3, 7), (3, 2.5, 6), (1, 5, 100), (2, 1.5, 3)]
    out["ladder_args"] = np.array(ladders, dtype=np.float64)
    for i, a in enumerate(ladders):
        out[f"ladder_{i}"] = it.call("get_annealing_ladder_", from_py(np.array(a, float)), from_py(0.0)).a
    x = np.concatenate([10.0 ** rng.uniform(-12, 0, 40), [1.0], 1 + 10.0 ** rng.uniform(-6, 4, 60)])
    out["q_x"] = x
    out["q_vec"] = it.call("Q_approx_vec", from_py(x)).a                 # vector-wide stop (R/utils.R:402)
    out["q_lower_only"] = it.call("Q_approx_vec", from_py(x[:41])).a
    out["q_scalar"] = np.array([it.call("Q_approx", from_py(float(v))).a[0] for v in x])
    L = 10.0 ** rng.uniform(-8, 3, 80)
    out["lam_L"] = L
    for i, c in enumerate((0.5, 0.5946035575013605, 0.8408964152537145, 0.9)):
        out[f"lam_c{i}"] = np.array(c)
        out[f"lam_{i}"] = it.call("update_annealed_lam2_inv_vb_", from_py(L), from_py(c), from_py(1.0)).a
    U = np.asfortranarray(np.concatenate([rng.normal(0, 3, 150), [-38.0, -20.0, 8.0, 20.0, 37.0, 0.0]]).reshape(26, 6))
    out["imr_U"] = U
    lp = it.call("pnorm", from_py(U), **{"log.p": from_py(True)})
    l1p = it.call("pnorm", from_py(U), **{"log.p": from_py(True), "lower.tail": from_py(False)})
    out["imr_logp"], out["imr_log1p"] = lp.a, l1p.a
    out["imr_1"] = it.call("inv_mills_ratio_", from_py(1.0), from_py(U), l1p, lp).a
    out["imr_0"] = it.call("inv_mills_ratio_", from_py(0.0), from_py(U), l1p, lp).a
    gam = np.asfortranarray(rng.uniform(size=U.shape) ** 3)
    out["z_gam"] = gam
    out["z_c1"] = it.call("update_Z_", from_py(gam), from_py(U), l1p, lp, c=from_py(1.0)).a
    out["z_c07"] = it.call("update_Z_", from_py(gam), from_py(U), l1p, lp, c=from_py(0.7)).a
    xs = np.concatenate([rng.normal(0, 50, 60), [-800.0, -745.0, -37.0, 0.0, 37.0, 709.0, 745.0, 800.0]])
    out["l1pe_x"] = xs
    out["l1pe"] = it.call("log_one_plus_exp_", from_py(xs)).a
    ppi = np.asfortranarray(rng.uniform(size=(40, 17)) ** 4)
    ppi[3, 2] = ppi[7, 9] = ppi[20, 1] = 0.83   # ties
    ppi[0, 0] = 1.0
    ppi[1, 1] = 0.0
    out["fdr_ppi"] = ppi
    out["fdr"] = it.call("assign_bFDR", from_py(ppi)).a
    Yh = np.asfortranarray(rng.normal(size=(60, 9)) * rng.uniform(0.5, 3, size=9))
    Yh[rng.uniform(size=Yh.shape) < 0.05] = np.nan
    out["hyper_Y"] = Yh
    hyp = []
    p0s = [(5.0, 25.0, 75.0), (2.0, 10.0, 500.0), (10.0, 50.0, 10000.0), (1.0, 2.0, 40.0)]
    for E, Vv, p in p0s:
        h = it.call("auto_set_hyper_", from_py(Yh), from_py(p), from_py(np.array([E, Vv])))
        hyp.append([h.get("t02").a[0], h.get("n0").a[0], h.get("eta").a[0], h.get("nu").a[0], h.get("rho").a[0]])
    out["hyper_p0"] = np.array(p0s)
    out["hyper_out"] = np.array(hyp)
    save("rlite_functions.npz", **out)


def make_c1(it):
    import make_trajectory as mt
    t0 = time.time()
    X, Y, hyper, init, anneal = mt.problem("C1")
    res = run_core_light(it, X, Y, plain(hyper, HYPER_KEYS), plain(init, INIT_KEYS), anneal, 0.1)
    print(f"  C1: it={res['it']} evaluations={len(res['lb'])} [{time.time() - t0:.0f} s]", flush=True)
    save("rlite_c1.npz", in_check=mt.input_checksums(X, Y, hyper, init), **res)


def make_c4(it):
    """BASELINE config C4 (n=500, p=10000, q=5000, 20 hotspots, anneal=c(1,2,10), tol = 30 as c4_trajectory.npz) through
    the reference's own R code and its own dual-form loop: ~50 M pair updates of p-long axpys per iteration, run with
    RLITE_REF_THREADS concurrent calls on disjoint sample_q ranges (about 1.5 h on 8 cores)."""
    import make_trajectory as mt
    t0 = time.time()
    X, Y, hyper, init, anneal = mt.problem("C4")
    print(f"  C4 inputs in {time.time() - t0:.0f} s", flush=True)
    res = run_core_light(it, X, Y, plain(hyper, HYPER_KEYS), plain(init, INIT_KEYS), anneal, 30.0, t0=t0, with_fdr=it)
    print(f"  C4: it={res['it']} evaluations={len(res['lb'])} [{time.time() - t0:.0f} s]", flush=True)
    save("rlite_c4.npz", in_check=mt.input_checksums(X, Y, hyper, init), **res)


def run_core_light(it, X, Y, hyper, init, anneal, tol, t0=None, with_fdr=None):
    from oracle.rlite import reference as R
    from oracle.rlite.values import from_py
    lbs = []

    def hook(n, v):
        lbs.append(v)
        if t0 is not None:
            print(f"    ELBO evaluation {len(lbs)}: {v!r} [{time.time() - t0:.0f} s]", flush=True)
    out = R.global_local_core(Y, X, Y.shape[1], anneal, 1, tol, 1000, hyper, init, it=it, hook=hook, debug=True)
    gam = out["gam_vb"].flatten(order="F")
    probe = np.random.default_rng(5).integers(0, gam.size, size=20000)
    res = dict(lb=np.array(lbs), it=int(out["it"][0]), converged=bool(out["converged"][0]),
               lb_opt=float(out["lb_opt"][0]), probe_idx=probe, probe_gam=gam[probe],
               probe_beta=out["beta_vb"].flatten(order="F")[probe], theta_vb=out["theta_vb"], zeta_vb=out["zeta_vb"],
               sum_gam=float(gam.sum()), sel_ppi=np.flatnonzero(gam > 0.5))
    if with_fdr is not None:   # the reference's own assign_bFDR (R/summarise_output.R:207-223) on the final gam_vb
        fdr = with_fdr.call("assign_bFDR", from_py(out["gam_vb"])).a
        res["sel_fdr"] = np.flatnonzero(fdr.flatten(order="F") < 0.05)
    return res


def main():
    from oracle import native
    from oracle.rlite import reference as R
    native.build()
    if not R.available():
        raise SystemExit("needs /root/reference (R sources) and oracle/_ref (the reference's coreLoop.cpp)")
    it = R.load()
    what = sys.argv[1:] or ["functions", "core", "top", "c1"]
    for w in what:
        print(w, flush=True)
        {"functions": make_functions, "core": make_core, "top": make_top, "c1": make_c1, "c4": make_c4}[w](it)
    if it.warnings:
        print("R warnings raised during the runs:", sorted(set(it.warnings)))


if __name__ == "__main__":
    main()
