"""GPU parity of one sweep through the C ABI against the CPU oracle (and, at dual-feasible sizes,
against the reference's own coreLoop.cpp: its stored outputs, tests/reference_runs.py).  Tolerances: max|d gam_vb| <= 1e-8
(north_star), tighter in practice."""
import numpy as np
import pytest

import reference_runs
from problems import make_problem, sweep_inputs

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,p,q,c,form,shuffle", [
    (100, 75, 20, 1.0, "reference", False),
    (100, 75, 20, 0.6, "reference", True),
    (200, 300, 200, 0.8, "reference", True),
    (500, 203, 70, 1.0, "primal", True),
    (1000, 120, 50, 0.5, "primal", False),
    # one full round of the persistent grid (148 tiles) + a tail launch: the row sums come from the per-tile partials
    # the helper warps leave (main launch) plus one streamed row (tail traits)
    (1000, 21, 2500, 0.5, "primal", True),    # 16-trait tiles, 17 tail tiles of 8
    (100, 24, 4776, 0.7, "primal", True),     # 32-trait tiles (one trait per helper lane), 5 tail tiles
    (600, 19, 3552 + 3, 1.0, "primal", False),  # 24-trait tiles, q not a multiple of 8
])
def test_single_sweep_parity(oracle_built, n, p, q, c, form, shuffle):
    from atlasqtl_b200.device import SweepContext
    native = oracle_built
    X, Y, hyper, init = make_problem(n, p, q)
    p = X.shape[1]
    si = sweep_inputs(X, Y, init, c=c)
    order = (np.random.default_rng(5).permutation(p) if shuffle else np.arange(p)).astype(np.int32)
    if form == "reference":
        ref = reference_runs.load("sweep", n, p, q, c, shuffle)
        np.testing.assert_allclose(reference_runs.in_check(X, Y, init), ref["in_check"], rtol=1e-12)
    else:
        ref = reference_runs.with_views(reference_runs.sweep_summary(
            si, *reference_runs.oracle_sweep(native, X, Y, si, order, form), sample=False))
    pick = ref["pick"]   # every entry, or the stored sample of the reference's sweep

    with SweepContext(X, Y) as ctx:
        ctx.set_order(order)
        st0 = ctx.set_state(si["gam"], si["mu"])
        beta0 = si["gam"] * si["mu"]
        np.testing.assert_allclose(st0["colsum_gam"], si["gam"].sum(axis=0), rtol=1e-12)
        np.testing.assert_allclose(st0["colsum_beta2"], (beta0 ** 2).sum(axis=0), rtol=1e-12)
        np.testing.assert_allclose(st0["colsum_gam_mu2"], (si["gam"] * si["mu"] ** 2).sum(axis=0), rtol=1e-12)
        R0 = Y - X @ beta0
        np.testing.assert_allclose(ctx.get_residual(), R0, atol=1e-10)
        np.testing.assert_allclose(st0["resid_sq"], (R0 ** 2).sum(axis=0), rtol=1e-11)

        ctx.refresh_tables(si["theta"], si["zeta"], c_next=c)
        out = ctx.sweep(c, si["log_sig2_inv"], si["tau"], si["log_tau"], si["sig2_beta"])
        st = ctx.get_state()
        R = ctx.get_residual()
        rows = ctx.rowsums_zpart()

    assert np.abs(pick(st["gam_vb"]) - ref["gam"]).max() <= 1e-9
    assert np.abs(pick(st["mu_beta_vb"]) - ref["mu"]).max() <= 1e-9 * max(1.0, ref["mu_absmax"])
    assert np.abs(pick(st["beta_vb"]) - ref["beta"]).max() <= 1e-9
    np.testing.assert_allclose(ref["pick_R"](R), ref["R"], atol=1e-9)
    np.testing.assert_allclose(out["colsum_gam"], ref["colsum_gam"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(out["colsum_beta2"], ref["colsum_beta2"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(out["colsum_gam_mu2"], ref["colsum_gam_mu2"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(out["resid_sq"], ref["resid_sq"], rtol=1e-9)
    np.testing.assert_allclose(out["colsum_zpart"], ref["colsum_zpart"], rtol=1e-9, atol=1e-8)
    np.testing.assert_allclose(rows, ref["rowsum_zpart"], rtol=1e-9, atol=1e-8)
