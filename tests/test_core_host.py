"""CPU tests of the host driver (atlasqtl_b200.core) with the oracle-backed test double in place of the
CUDA context: the re-expression of the R updates through per-trait / per-SNP sums must reproduce the
line-by-line restatement of the R loop (oracle/vb_oracle.py), iteration by iteration; with the reference's own
sweep, its stored runs (tests/reference_runs.py)."""
import numpy as np
import pytest

import reference_runs
from atlasqtl_b200 import core
from fake_context import OracleSweepContext
from oracle import vb_oracle
from problems import make_problem


@pytest.mark.parametrize("anneal", [None, (1, 2, 10), (2, 3, 5), (3, 2, 4)])
def test_host_loop_matches_restated_r_loop(oracle_built, anneal):
    X, Y, hyper, init = reference_runs.host_problem()
    q = Y.shape[1]
    tr_c = []
    ref = reference_runs.load("host", anneal)   # the restated R loop with the reference's own sweep
    tr_o = ref["trace"]
    np.testing.assert_allclose(reference_runs.in_check(X, Y, init), ref["in_check"], rtol=1e-12)
    out = core.atlasqtl_global_local_core_(Y, X, q, anneal, 1, 0.1, 1000, 0, hyper, init, debug=True,
                                           context_factory=lambda X_, Y_: OracleSweepContext(X_, Y_), trace=tr_c)
    assert ref["converged"] and out["converged"]
    assert out["it"] == ref["it"]
    assert len(tr_o) == len(tr_c)
    for a, b in zip(tr_o, tr_c):
        assert a["it"] == b["it"] and abs(a["c"] - b["c"]) < 1e-15
        assert (a["lb"] is None) == (b["lb"] is None)
        if a["lb"] is not None:
            assert abs(a["lb"] - b["lb"]) <= 1e-10 * abs(a["lb"])
    assert np.abs(ref["pick"](out["gam_vb"]) - ref["gam_vb"]).max() <= 1e-10
    assert np.array_equal(out["gam_vb"] > 0.5, ref["sel"])
    np.testing.assert_allclose(out["theta_vb"], ref["theta_vb"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(out["zeta_vb"], ref["zeta_vb"], rtol=1e-9, atol=1e-10)


def test_order_fn_is_honoured(oracle_built):
    X, Y, hyper, init = reference_runs.order_problem()
    q = Y.shape[1]
    ref = reference_runs.load("order", "perm")   # the restated R loop with the reference's own sweep, shuffled order
    np.testing.assert_allclose(reference_runs.in_check(X, Y, init), ref["in_check"], rtol=1e-12)
    out = core.atlasqtl_global_local_core_(Y, X, q, None, 1, 0.1, 50, 0, hyper, init, debug=True,
                                           order_fn=reference_runs.order_perm,
                                           context_factory=lambda X_, Y_: OracleSweepContext(X_, Y_))
    assert out["it"] == ref["it"]
    assert np.abs(ref["pick"](out["gam_vb"]) - ref["gam_vb"]).max() <= 1e-10
    ident = reference_runs.load("order", "identity")
    assert np.abs(ident["gam_vb"] - ref["gam_vb"]).max() > 1e-8  # the order really changes the trajectory


def test_rejects_what_this_build_does_not_cover():
    X, Y, hyper, init = make_problem(50, 20, 5)
    with pytest.raises(ValueError):
        core.atlasqtl_global_local_core_(Y, X, 5, None, 1, 0.1, 5, 0, hyper, init, batch="0")
    with pytest.raises(NotImplementedError):
        core.atlasqtl_global_local_core_(Y, X, 5, None, 1, 0.1, 5, 0, hyper, init, trace_path="/tmp/x")


@pytest.mark.parametrize("background", [False, True])
def test_checkpoints_and_resume(oracle_built, tmp_path, background):
    """checkpoint_ / checkpoint_clean_up_ (R/utils.R:571-627): files every `rate` iterations with the reference's fields,
    only the last two kept, removed at the end; and (extension) a run restarted from a checkpoint lands on the same
    optimum.  background: the context offers snapshot / snapshot_fetch, so the files are written on a worker thread."""
    import glob
    from fake_context import SnapshotOracleSweepContext
    X, Y, hyper, init = make_problem(100, 75, 20, p_act=10, q_act=20, maf=0.2, p0=(5, 25))
    q = Y.shape[1]
    base = str(tmp_path) + "/"
    made = []

    def fac(X_, Y_):
        made.append((SnapshotOracleSweepContext if background else OracleSweepContext)(X_, Y_))
        return made[-1]
    ref = core.atlasqtl_global_local_core_(Y, X, q, None, 1, 0.1, 1000, 0, hyper, init, context_factory=fac)
    out = core.atlasqtl_global_local_core_(Y, X, q, None, 1, 0.1, 1000, 0, hyper, init, checkpoint_path=base,
                                           checkpoint_rate=10, keep_checkpoints=True, context_factory=fac)
    assert np.array_equal(out["gam_vb"], ref["gam_vb"])            # checkpointing does not perturb the run
    if background:
        ctx = made[1]
        assert ctx.snapshots == out["it"] // 10 and ctx._ckpt_future is None     # every writer has been joined
        assert all(not name.startswith("MainThread") for name in ctx.fetch_threads)
    files = sorted(glob.glob(base + "tmp_output_it_*.npz"), key=lambda f: int(f.split("_it_")[1][:-4]))
    its = [int(f.split("_it_")[1][:-4]) for f in files]
    assert its == [i for i in range(10, out["it"] + 1, 10)][-2:]   # only the last two are kept
    d = np.load(files[0])
    for key in ("beta_vb", "gam_vb", "theta_vb", "zeta_vb", "converged", "it", "lb_new", "diff_lb", "lam2_inv_vb",
                "sig02_inv_vb"):
        assert key in d.files
    assert d["gam_vb"].shape == (X.shape[1], q) and int(d["it"]) == its[0]
    init2 = core.init_from_checkpoint(files[0], init)
    res = core.atlasqtl_global_local_core_(Y, X, q, None, 1, 0.1, 1000, 0, hyper, init2, checkpoint_path=base,
                                           checkpoint_rate=10, context_factory=fac)
    assert res["converged"]
    assert np.abs(res["gam_vb"] - ref["gam_vb"]).max() <= 1e-2 and abs(res["lb_opt"] - ref["lb_opt"]) <= 1.0  # tol = 0.1 on the ELBO
    assert glob.glob(base + "tmp_output_it_*.npz") == []           # cleaned up at the end by default


@pytest.mark.parametrize("anneal", [None, (1, 2, 5)])
def test_host_loop_with_missing_responses_matches_restated_r_loop(oracle_built, anneal):
    """NaN responses: the host loop written against the per-trait sums of aq_set_state_mis / aq_sweep_mis
    (R/update_vb.R:131, :149-154, R/elbo.R:28-30, :141) reproduces the restated R loop with mis_pat / X_norm_sq."""
    X, Y, hyper, init = make_problem(100, 75, 20, p_act=10, q_act=20, maf=0.2, p0=(5, 25))
    q = Y.shape[1]
    Ym = Y.copy()
    Ym[np.random.default_rng(3).uniform(size=Y.shape) < 0.06] = np.nan
    tr_o, tr_c = [], []
    ref = vb_oracle.atlasqtl_global_local_core_(Ym, X, q, anneal, 1, 0.1, 1000, hyper, init, trace=tr_o)
    out = core.atlasqtl_global_local_core_(Ym, X, q, anneal, 1, 0.1, 1000, 0, hyper, init, debug=True,
                                           context_factory=lambda X_, Y_: OracleSweepContext(X_, Y_), trace=tr_c)
    assert ref["converged"] and out["converged"] and out["it"] == ref["it"]
    for a, b in zip(tr_o, tr_c):
        assert (a["lb"] is None) == (b["lb"] is None)
        if a["lb"] is not None:
            assert abs(a["lb"] - b["lb"]) <= 1e-10 * abs(a["lb"])
    assert np.abs(out["gam_vb"] - ref["gam_vb"]).max() <= 1e-10
