"""GPU: the segmented sweep (SNP blocks of every tile cut into segments that different CTAs process in turn, DESIGN.md
section 4.1) against the CPU oracle and against the unsegmented launch of the same state.

The segmented launch hands a tile's residual and column sums from CTA to CTA through global memory (release / acquire
on a per-tile counter); results must not depend on the number of segments beyond the summation order of the column sums."""
import numpy as np
import pytest

from problems import make_problem, sweep_inputs
from reference_runs import oracle_sweep, zparts

pytestmark = pytest.mark.gpu


def _sweep(monkeypatch, X, Y, si, order, env):
    from atlasqtl_b200.device import SweepContext
    for k in ("AQ_NSEG", "AQ_NO_SEG", "AQ_NO_TAIL"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    with SweepContext(X, Y) as ctx:
        ctx.set_order(order)
        st0 = ctx.set_state(si["gam"], si["mu"])
        ctx.refresh_tables(si["theta"], si["zeta"], c_next=si["c"])
        out = ctx.sweep(si["c"], si["log_sig2_inv"], si["tau"], si["log_tau"], si["sig2_beta"])
        plan = ctx.sweep_plan()
        out2 = ctx.sweep(si["c"], si["log_sig2_inv"], si["tau"], si["log_tau"], si["sig2_beta"])   # a second sweep on top
        st = ctx.get_state()
        R = ctx.get_residual()
        rows = ctx.rowsums_zpart()
    return dict(st0=st0, out=out, out2=out2, st=st, R=R, rows=rows, plan=plan)


@pytest.mark.parametrize("n,p,q,nseg,cluster", [
    (100, 400, 4800 + 5, 3, None),    # 32-trait tiles (151 of them on 148 SMs), 50 blocks in 3 segments
    (1000, 256, 2400 + 16, 2, None),  # the C2 configuration (16-trait tiles, 9 sample tiles per warp): 151 tiles, 2 segments
    (600, 520, 3600, 4, None),        # 24-trait tiles: 150 tiles, 65 blocks in 4 segments (last one shorter)
    (1500, 256, 1620, 2, None),       # 3-CTA clusters of 32-trait tiles: 51 tiles on 49 resident clusters
    (3000, 256, 560, 2, 4),           # 4-CTA clusters of 16-trait tiles (forced): 35 tiles on 33 resident clusters
])
def test_segmented_sweep_matches_oracle_and_unsegmented(oracle_built, monkeypatch, n, p, q, nseg, cluster):
    if cluster:
        monkeypatch.setenv("AQ_FORCE_CLUSTER", str(cluster))
    X, Y, hyper, init = make_problem(n, p, q)
    p = X.shape[1]
    si = sweep_inputs(X, Y, init, c=0.8)
    order = np.random.default_rng(5).permutation(p).astype(np.int32)
    seg = _sweep(monkeypatch, X, Y, si, order, {"AQ_NSEG": str(nseg)})
    one = _sweep(monkeypatch, X, Y, si, order, {"AQ_NO_SEG": "1", "AQ_NO_TAIL": "1"})
    assert seg["plan"]["nseg"] == nseg and one["plan"]["nseg"] == 1
    assert seg["plan"]["ntiles"] > seg["plan"]["groups"]
    # segmented vs unsegmented, two sweeps each: the same mathematics, but not bit for bit -- the first block of a segment
    # forms S from the fully updated residual, where the unsegmented sweep corrects a look-ahead S by the cross Gram block
    # (S_{b+1} = X_{b+1}' R_{b-1} - G_{b+1,b} Delta_b), and the column sums are added in segment order
    assert np.abs(seg["st"]["gam_vb"] - one["st"]["gam_vb"]).max() <= 1e-12
    assert np.abs(seg["st"]["mu_beta_vb"] - one["st"]["mu_beta_vb"]).max() <= 1e-12 * max(1.0, np.abs(one["st"]["mu_beta_vb"]).max())
    np.testing.assert_allclose(seg["R"], one["R"], atol=1e-11)
    for key in ("colsum_gam", "colsum_gam_mu2", "colsum_beta2", "colsum_zpart", "resid_sq"):
        np.testing.assert_allclose(seg["out2"][key], one["out2"][key], rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(seg["rows"], one["rows"], rtol=1e-11, atol=1e-11)
    # the state set-up (mode 1 of the kernel) is segmented as well
    for key in ("colsum_gam", "colsum_gam_mu2", "colsum_beta2", "resid_sq"):
        np.testing.assert_allclose(seg["st0"][key], one["st0"][key], rtol=1e-13, atol=1e-13)
    # against the CPU oracle (one sweep)
    g_ref, m_ref, b_ref, R_ref = oracle_sweep(oracle_built, X, Y, si, order, "primal")
    np.testing.assert_allclose(seg["out"]["colsum_gam"], g_ref.sum(axis=0), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(seg["out"]["colsum_beta2"], (b_ref ** 2).sum(axis=0), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(seg["out"]["colsum_gam_mu2"], (g_ref * m_ref ** 2).sum(axis=0), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(seg["out"]["resid_sq"], (R_ref ** 2).sum(axis=0), rtol=1e-9)
    zc, _ = zparts(si, g_ref)
    np.testing.assert_allclose(seg["out"]["colsum_zpart"], zc, rtol=1e-9, atol=1e-8)


def test_plan_prefers_segments_over_a_partly_filled_round(monkeypatch):
    """q_local = 2500 traits at n = 1000 (C2 on 8 GPUs): 157 tiles on 148 SMs.  Unsegmented that is one full round plus
    a tail launch; the plan cuts the SNPs into segments so that the 9 extra tiles cost 1 / nseg of a round."""
    from atlasqtl_b200.device import SweepContext
    for k in ("AQ_NSEG", "AQ_NO_SEG", "AQ_NO_TAIL"):
        monkeypatch.delenv(k, raising=False)
    rng = np.random.default_rng(0)
    n, p, q = 1000, 2048, 2500
    X = np.asfortranarray(rng.normal(size=(n, p)))
    Y = np.asfortranarray(rng.normal(size=(n, q)))
    with SweepContext(X, Y) as ctx:
        ctx.set_state(np.asfortranarray(rng.uniform(size=(p, q)) * 1e-3), np.asfortranarray(rng.normal(size=(p, q)) * 1e-2))
        ctx.refresh_tables(np.zeros(p), np.full(q, -2.0))
        ctx.sweep(1.0, 0.0, np.ones(q), np.zeros(q), np.full(q, 1e-3))
        plan = ctx.sweep_plan()
    assert plan["ntiles"] == 157 and plan["groups"] == 148
    slots = -(-plan["ntiles"] * plan["nseg"] // plan["groups"])
    assert plan["nseg"] >= 8 and slots / plan["nseg"] <= 1.13   # vs 1.68 rounds (full round + 8-trait tail round)
