"""GPU: the sweep's annealed logistic (aq_common.cuh logistic_neg == exp(-logOnePlusExp(x)), src/coreLoop.cpp:28-33,
:75-77) evaluated on the device by the very routine the chain warp uses, over its whole range including the selects
beyond +-700 and saturated gam_vb; and a sweep driven into saturation."""
import mpmath as mp
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("variant", [0, 1])
def test_logistic_neg_full_range(variant):
    from atlasqtl_b200.compat import logistic_neg_device as _dev
    logistic_neg_device = lambda x: _dev(x, variant=variant)
    x = np.concatenate([np.linspace(-750, 750, 3001), [-700.0, 700.0, np.nextafter(700.0, 800), np.nextafter(-700.0, -800),
                                                        -1e308, 1e308, -np.inf, np.inf, 0.0, -0.0, 1e-320, 36.7, -36.7,
                                                        709.78, -709.78, 745.2, -745.2],
                        np.random.default_rng(0).normal(scale=30, size=5000)])
    got = logistic_neg_device(x)
    assert got.shape == x.shape and np.isnan(logistic_neg_device(np.array([np.nan]))[0])
    mp.mp.dps = 40
    for xi, gi in zip(x, got):
        if not np.isfinite(xi) or abs(xi) > 700:
            assert gi == (0.0 if xi > 0 else 1.0), xi   # 1/(1+e^x) < 1e-304 resp. 1 - 1e-304: the reference gives 0 / 1 too
            continue
        want = 1 / (1 + mp.exp(mp.mpf(float(xi))))
        err = abs(mp.mpf(float(gi)) - want)
        # relative: a few ulp where the value matters; the one-constant argument reduction adds |x| / ln2 * 5.5e-17 (6e-14 at
        # |x| = 700, where the value is 1e-304).  Absolute: never above an ulp of 1 (the bound on gam_vb is 1e-8).
        assert err <= (5e-16 + (1e-16 * abs(xi) if variant == 1 else 0.0)) * want, (xi, gi)
        assert err <= 2.5e-16, (xi, gi)
    assert np.all((got >= 0) & (got <= 1))
    # monotone non-increasing over the grid part
    assert np.all(np.diff(got[:3001]) <= 0)


def test_sweep_with_saturated_probabilities(oracle_built):
    """theta + zeta driven to +-30 and huge effects: gam_vb saturates at 0 and 1 (logistic arguments beyond +-700);
    the CUDA sweep must agree with the reference's own loop there too."""
    import reference_runs
    from atlasqtl_b200.device import SweepContext
    # strong signals (Y scaled by 40: mu^2 / (2 sig2_beta) in the thousands), theta + zeta at +-30 / +-8
    X, Y, si, _ = reference_runs.saturated_inputs()
    ref = reference_runs.load("saturated")   # the reference's own loop on these inputs
    np.testing.assert_allclose(reference_runs.in_check(X, Y), ref["in_check"], rtol=1e-12)
    pick, g_ref, b_ref = ref["pick"], ref["gam"], ref["beta"]
    assert (g_ref == 0).any() or (g_ref < 1e-300).any()
    assert (g_ref == 1).any()
    with SweepContext(X, Y) as ctx:
        ctx.set_state(si["gam"], si["mu"])
        ctx.refresh_tables(si["theta"], si["zeta"], c_next=1.0)
        ctx.sweep(1.0, si["log_sig2_inv"], si["tau"], si["log_tau"], si["sig2_beta"])
        st = ctx.get_state()
    assert np.isfinite(st["gam_vb"]).all() and np.isfinite(st["mu_beta_vb"]).all()
    assert np.abs(pick(st["gam_vb"]) - g_ref).max() <= 1e-9
    assert np.abs(pick(st["beta_vb"]) - b_ref).max() <= 1e-9 * max(1.0, ref["beta_absmax"])
