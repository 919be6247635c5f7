"""GPU: full VB runs through the C ABI against the restated R loop on the CPU oracle
(sweep = the reference's own coreLoop.cpp where its p x p inputs are feasible: its stored runs, tests/reference_runs.py)."""
import numpy as np
import pytest

import reference_runs
from problems import make_problem

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,p,q,anneal,form", [
    (100, 75, 20, (1, 2, 10), "reference"),
    (100, 75, 20, None, "reference"),
    (200, 300, 200, (1, 2, 10), "reference"),
    (500, 400, 150, (1, 2, 10), "primal"),
    (1500, 200, 90, (1, 2, 10), "primal"),   # 2-CTA cluster
    (3000, 120, 40, None, "primal"),          # 4-CTA cluster
])
def test_trajectory_parity(oracle_built, n, p, q, anneal, form):
    from atlasqtl_b200 import core, summarise
    from oracle import vb_oracle
    X, Y, hyper, init = make_problem(n, p, q)
    q = Y.shape[1]
    tr_g = []
    if form == "reference":
        ref = reference_runs.load("full", n, p, q, anneal)
        np.testing.assert_allclose(reference_runs.in_check(X, Y, init), ref["in_check"], rtol=1e-12)
    else:
        tr_o = []
        run = vb_oracle.atlasqtl_global_local_core_(Y, X, q, anneal, 1, 0.1, 1000, hyper, init, sweep=form, trace=tr_o,
                                                    nthreads=4)
        ref = reference_runs.with_views(reference_runs.run_summary(run, tr_o, sample=False))
    out = core.atlasqtl_global_local_core_(Y, X, q, anneal, 1, 0.1, 1000, 0, hyper, init, debug=True, trace=tr_g)
    assert out["converged"] and ref["converged"]
    assert out["it"] == ref["it"]
    for a, b in zip(ref["trace"], tr_g):
        if a["lb"] is not None:
            assert abs(a["lb"] - b["lb"]) <= 1e-10 * abs(a["lb"]), (a["it"], a["lb"], b["lb"])
    pick = ref["pick"]   # every entry, or the stored sample of the reference's run
    assert np.abs(pick(out["gam_vb"]) - ref["gam_vb"]).max() <= 1e-8
    assert np.abs(pick(out["beta_vb"]) - ref["beta_vb"]).max() <= 1e-8
    # integer outputs: selection sets must be identical
    assert np.array_equal(out["gam_vb"] > 0.5, ref["sel"])
    assert np.array_equal(summarise.assign_bFDR(out["gam_vb"]) < 0.05, ref["sel_bfdr"])
