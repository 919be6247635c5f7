"""The table pass (tables_kernel, atlasqtl_b200/csrc/aq_stream.cuh) entry by entry against the mathematical functions.

Every entry of D = log(1 - Phi(u)) - log Phi(u), W = imr1 - imr0 and I0 = imr0 (inv_mills_ratio_, R/utils.R:172-191)
is compared with a 40-digit mpmath evaluation at the double the kernel sees: u = fl(theta_j + zeta_k), and for W and
I0 while annealing U = fl(fl(sqrt(c)) u) (update_Z_, R/update_vb.R:219-224; R evaluates at the same doubles).  D is
checked on both of its code paths (the ELBO iterations' log Phi / log(1 - Phi) and the one-log log-odds of the other
iterations) and the two paths against each other.  The p x q part of ELBO term B (R/elbo.R:19-26) is pinned through
sums over bands of u, so that no region is swamped by another.  The row and column sums of the Z part are compared
with exact sums of the downloaded tables.

Bars, with eps = 2^-52 (a CPU emulation of the kernel's formulas, with SciPy's erfcx in place of CUDA's, reaches
5.5 eps on D, 2.5 eps on W and 246 eps on I0 at U = -35):
  D (both paths)                                  |d| <= 16 eps max(1, |D|);  the two paths apart: 8 eps max(1, |D|)
  W                                               |d| <= 16 eps |W|
  I0 for U >= 0 (about -U there)                  |d| <= 16 eps |I0|
  exponentially small values: I0 for U < 0,       |d| <= (16 + U^2) eps |value|, or 1e-300 where |value| < 1e-290.
  log Phi(u) for u > 0, log(1 - Phi(u)) for u < 0
The U^2 is not slack: exp(-U^2 / 2) from a U * U rounded once carries a relative error of about (U^2 / 2) eps.
"""
import functools
import math
import os

import mpmath as mp
import numpy as np
import pytest

from problems import mis_inputs, sweep_inputs

EPS = 2.0 ** -52
ELBO_EPS = 1.8189894035458565e-12   # .Machine$double.eps^0.75 (R/elbo.R:15)
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "rlite_functions.npz")


# ----------------------------------------------------------------------------- the 40-digit reference
@functools.lru_cache(maxsize=None)
def ref_point(u):
    """log Phi(u), log(1 - Phi(u)), phi(u) / Phi(u), -phi(u) / (1 - Phi(u)) at the double u, to 40 digits (mpf).
    The side of the tail mass t = Phi(-|u|) that is close to 1 is taken as log1p(-t), which needs no more digits than
    t itself (log Phi(38) = -3e-316 read as log(Phi(38)) would need 400)."""
    with mp.workdps(40):
        x = mp.mpf(u)
        t = mp.ncdf(-abs(x))
        log_tail, log_body = mp.log(t), mp.log1p(-t)
        ph = mp.npdf(x)
        r_tail, r_body = ph / t, ph / (1 - t)
        if u >= 0:
            lp, lq, m1, m0 = log_body, log_tail, r_body, -r_tail
        else:
            lp, lq, m1, m0 = log_tail, log_body, r_tail, -r_body
        # the clamps of R/utils.R:179, :184 (never active in exact arithmetic: phi / Phi > -U > -phi / (1 - Phi))
        return lp, lq, max(m1, -x), min(m0, -x)


def _split(v):
    """mpf -> (hi, lo) doubles with hi + lo = v to about 2^-106 relative."""
    hi = float(v)
    return hi, float(v - mp.mpf(hi))


@functools.lru_cache(maxsize=None)
def _ref_split(u):
    lp, lq, m1, m0 = ref_point(u)
    with mp.workdps(40):
        return _split(lp) + _split(lq) + _split(lq - lp) + _split(m1 - m0) + _split(m0)


def ref_arrays(u):
    """Arrays of u's shape: hi / lo parts of lp, lq, D, W, I0 (W and I0 at the argument u itself)."""
    uniq, inv = np.unique(np.asarray(u, dtype=np.float64).ravel(), return_inverse=True)
    tab = np.array([_ref_split(float(v)) for v in uniq]).reshape(len(uniq), 5, 2)[inv]
    names = ("lp", "lq", "D", "W", "I0")
    return {nm: (tab[:, i, 0].reshape(np.shape(u)), tab[:, i, 1].reshape(np.shape(u))) for i, nm in enumerate(names)}


def _err(k, ref):
    hi, lo = ref
    return np.abs((k - hi) - lo)


def _small_bar(value, x):
    """Bar of an exponentially small value at argument x."""
    return np.where(np.abs(value) < 1e-290, 1e-300, (16 + x * x) * EPS * np.abs(value))


def arg_U(u, c):
    """The argument of W and I0: the kernel's c_is_one switch (isTRUE(all.equal(c, 1)), R/update_vb.R:219)."""
    return u if abs(c - 1.0) < 1.5e-8 else np.sqrt(c) * u


def check_tables(tab, u, c, what=""):
    """Every entry of D, W, I0 (any may be None) against the reference; returns the worst error of each in units of its
    bar's eps multiple, for the record."""
    u = np.asarray(u, dtype=np.float64)
    U = arg_U(u, c)
    r = ref_arrays(u)
    rU = r if U is u else ref_arrays(U)
    worst = {}
    if tab.get("D") is not None:
        e, scale = _err(tab["D"], r["D"]), np.maximum(1.0, np.abs(r["D"][0]))
        bad = ~(e <= 16 * EPS * scale)
        assert not bad.any(), (what, "D", u[bad][:5], tab["D"][bad][:5], r["D"][0][bad][:5])
        worst["D"] = float((e / (EPS * scale)).max())
    if tab.get("W") is not None:
        e, scale = _err(tab["W"], rU["W"]), np.abs(rU["W"][0])
        bad = ~(e <= 16 * EPS * scale)
        assert not bad.any(), (what, "W", c, U[bad][:5], tab["W"][bad][:5], rU["W"][0][bad][:5])
        worst["W"] = float((e / (EPS * scale)).max())
    if tab.get("I0") is not None:
        i0 = rU["I0"][0]
        e = _err(tab["I0"], rU["I0"])
        bar = np.where(U >= 0, 16 * EPS * np.abs(i0), _small_bar(i0, U))
        bad = ~(e <= bar)
        assert not bad.any(), (what, "I0", c, U[bad][:5], tab["I0"][bad][:5], i0[bad][:5])
        pos = U >= 0
        worst["I0+"] = float((e[pos] / (EPS * np.abs(i0[pos]))).max(initial=0.0))
        neg = (U < 0) & (np.abs(i0) >= 1e-290)
        worst["I0-"] = float((e[neg] / (EPS * np.abs(i0[neg]))).max(initial=0.0))
    return worst


@functools.lru_cache(maxsize=None)
def _entropy(g):
    """g log(fl(g + eps)) + fl(1 - g) log(fl(fl(1 - g) + eps)) at the doubles the kernel forms, to 40 digits."""
    g1 = 1.0 - g
    with mp.workdps(40):
        return (float(mp.mpf(g) * mp.log(mp.mpf(g + ELBO_EPS))), float(mp.mpf(g1) * mp.log(mp.mpf(g1 + ELBO_EPS))))


def elbo_reference(u, gam):
    """(fsum of the terms, the bar): terms g lp + (1 - g) lq - g log(g + eps) - (1 - g) log(1 - g + eps) per pair.
    Bar: the per-term bars of lp and lq weighted by g and 1 - g, plus 64 eps times the sum of the absolute values of
    the four products (this also covers the rounding of the reference's own products, at most eps / 2 each)."""
    u = np.asarray(u, dtype=np.float64).ravel()
    g = np.asarray(gam, dtype=np.float64).ravel()
    g1 = 1.0 - g
    r = ref_arrays(u)
    uniq, inv = np.unique(g, return_inverse=True)
    ent = np.array([_entropy(float(v)) for v in uniq]).reshape(len(uniq), 2)[inv]
    lp, lq = r["lp"][0] + r["lp"][1], r["lq"][0] + r["lq"][1]
    prods = [g * r["lp"][0], g * r["lp"][1], g1 * r["lq"][0], g1 * r["lq"][1], -ent[:, 0], -ent[:, 1]]
    total = math.fsum(np.concatenate(prods).tolist())
    bar_lp = np.where(u > 0, _small_bar(lp, u), 16 * EPS * np.maximum(1.0, np.abs(lp)))
    bar_lq = np.where(u < 0, _small_bar(lq, u), 16 * EPS * np.maximum(1.0, np.abs(lq)))
    mag = np.abs(g * lp) + np.abs(g1 * lq) + np.abs(ent[:, 0]) + np.abs(ent[:, 1])
    return total, math.fsum((g * bar_lp + g1 * bar_lq).tolist()) + 64 * EPS * math.fsum(mag.tolist())


# ----------------------------------------------------------------------------- arguments
GRID = np.arange(-40 * 64, 40 * 64 + 1) / 64.0            # dense, step 2^-6 on [-40, 40]
BAND = 37.5 + np.arange(0, 308) / 256.0                   # exp(-u^2 / 2) goes subnormal, then to zero: 37.5 .. 38.7
EDGES = np.array([1e-300, 1e-12, 1e-6, 100.0, 1e3])
POINTS = np.unique(np.concatenate([GRID, BAND, -BAND, EDGES, -EDGES]))
GAM_VALUES = np.array([0.0, 1.0, 5e-324, 1e-300, 1.8e-12, 0.5, 1 - 2.0 ** -53, 0.25, 0.9, 1e-3, 0.999, 1.0 / 3])
C_VALUES = [1.0, 1 + 1e-9, 1 - 1e-9, 1 - 1e-7, 0.7, 0.05]


def ladder():
    from atlasqtl_b200.core import get_annealing_ladder_
    return [float(c) for c in get_annealing_ladder_((1, 2, 10)) if c != 1.0]


def grid_theta(p, seed):
    """theta_j / zeta_k on the 2^-6 grid in [-20, 20]: every u = theta_j + zeta_k is exact and lies in GRID."""
    j = np.arange(p)
    return ((j * 37 + seed) % 2561 - 1280) / 64.0


def _context(n, p, q, seed=0):
    from atlasqtl_b200.device import SweepContext
    rng = np.random.default_rng(seed)
    return SweepContext(np.asfortranarray(rng.normal(size=(n, p))), np.asfortranarray(rng.normal(size=(n, q))))


def _both_paths(ctx, theta, zeta, c):
    """Tables without the ELBO part (log-odds path of D) and with it (log Phi / log(1 - Phi) path): (tabs, tabs, part)."""
    ctx.refresh_tables(theta, zeta, c_next=c, want_elbo=False)
    t0 = ctx.get_tables()
    part = ctx.refresh_tables(theta, zeta, c_next=c, want_elbo=True)
    t1 = ctx.get_tables()
    return t0, t1, part


def _check_paths_agree(t0, t1, what=""):
    scale = np.maximum(1.0, np.abs(t1["D"]))
    bad = ~(np.abs(t0["D"] - t1["D"]) <= 8 * EPS * scale)
    assert not bad.any(), (what, t0["D"][bad][:5], t1["D"][bad][:5])
    return float((np.abs(t0["D"] - t1["D"]) / (EPS * scale)).max())


# ----------------------------------------------------------------------------- CPU: the reference itself
def test_reference_matches_direct_400_digit_log_ncdf():
    """log Phi via log1p(-Phi(-u)) at 40 digits equals the direct log(ncdf(u)) at 400 digits, in both tails (400 digits
    resolve 1 - Phi(u) up to |u| of about 42)."""
    for u in (-38.6, -37.9, -30.0, -20.0, -5.0, -1e-6, 1e-12, 0.5, 8.0, 20.0, 37.9, 38.6):
        lp, lq, _, _ = ref_point(u)
        with mp.workdps(400):
            x = mp.mpf(u)
            want_p, want_q = mp.log(mp.ncdf(x)), mp.log(mp.ncdf(-x))
            assert abs(lp - want_p) <= mp.mpf("1e-36") * abs(want_p), u
            assert abs(lq - want_q) <= mp.mpf("1e-36") * abs(want_q), u


def test_reference_ratios_and_bars_are_self_consistent():
    """The reference's inverse Mills ratios satisfy the identities W = phi / (Phi (1 - Phi)) and I0 -> -U for large U,
    and the relative bars of the small values are what the module docstring states."""
    for u in (-38.0, -3.0, 0.0, 2.5, 30.0):
        _, _, m1, m0 = ref_point(u)
        with mp.workdps(40):
            x = mp.mpf(u)
            w = mp.npdf(x) / (mp.ncdf(x) * mp.ncdf(-x))
            assert abs((m1 - m0) - w) <= mp.mpf("1e-35") * w, u
    assert abs(float(ref_point(30.0)[3]) + 30.0) < 0.04
    assert _small_bar(np.array([1e-295]), np.array([38.0]))[0] == 1e-300
    assert _small_bar(np.array([1e-100]), np.array([3.0]))[0] == 25 * EPS * 1e-100


# ----------------------------------------------------------------------------- GPU: pointwise
@pytest.mark.gpu
def test_get_tables_call_order_and_null_pointers():
    from atlasqtl_b200 import _lib
    with _context(10, 9, 5) as ctx:
        with pytest.raises(_lib.AtlasqtlB200Error, match="before aq_refresh_tables"):
            ctx.get_tables()
        theta, zeta = grid_theta(9, 3), grid_theta(5, 7)
        ctx.refresh_tables(theta, zeta)
        full = ctx.get_tables()
        only_w = ctx.get_tables(D=False, I0=False)
    assert only_w["D"] is None and only_w["I0"] is None
    np.testing.assert_array_equal(only_w["W"], full["W"])
    check_tables(full, theta[:, None] + zeta[None, :], 1.0)


@pytest.mark.gpu
def test_tables_pointwise_dense_grid_and_edges():
    """u on a 2^-6 grid over [-40, 40], the band 37.5 .. 38.7 at 2^-8, +-0.0, +-1e-300, +-1e-12, +-1e-6, +-100, +-1e3;
    every c of C_VALUES and of the annealing ladder get_annealing_ladder_((1, 2, 10)).  zeta = (0.0, -0.0) gives u = +0.0
    and -0.0 from theta = -0.0."""
    theta = np.concatenate([POINTS, [-0.0]])
    zeta = np.array([0.0, -0.0])
    u = theta[:, None] + zeta[None, :]
    assert np.signbit(u[-1, 1]) and not np.signbit(u[-1, 0])
    worst = {}
    base = None
    with _context(4, len(theta), 2) as ctx:
        ctx.set_state(np.full((len(theta), 2), 0.5), np.zeros((len(theta), 2)))
        for c in C_VALUES + ladder():
            t0, t1, _ = _both_paths(ctx, theta, zeta, c)
            for tab in (t0, t1):
                for k, v in check_tables(tab, u, c, what=f"c={c}").items():
                    worst[k] = max(worst.get(k, 0.0), v)
            worst["D paths"] = max(worst.get("D paths", 0.0), _check_paths_agree(t0, t1, what=f"c={c}"))
            if c == 1.0:
                base = (t0, t1)
            elif abs(c - 1.0) < 1.5e-8:   # 1 +- 1e-9 takes the unannealed branch: bit-identical to c = 1
                for t, b in zip((t0, t1), base):
                    np.testing.assert_array_equal(t["W"], b["W"])
                    np.testing.assert_array_equal(t["I0"], b["I0"])
            else:                          # 1 - 1e-7 and below: evaluated at sqrt(c) u
                assert not np.array_equal(t1["W"], base[1]["W"]), c
            if c != 1.0:                   # D does not depend on c
                np.testing.assert_array_equal(t0["D"], base[0]["D"])
                np.testing.assert_array_equal(t1["D"], base[1]["D"])
    print("worst errors in eps:", {k: round(v, 2) for k, v in worst.items()})


@pytest.mark.gpu
@pytest.mark.parametrize("q", [1, 95, 96, 97, 255, 256, 257, 513])
@pytest.mark.parametrize("p", [1, 7, 8, 9, 4097])
def test_tables_every_entry_at_ragged_shapes(p, q):
    """Partial 8-row blocks, partial and several 256-trait column blocks, q_pad padding: every entry on both D paths,
    and the ELBO part against an exact sum.  c alternates between 1 and 0.7 over the shapes."""
    c = 1.0 if (p + q) % 2 else 0.7
    theta, zeta = grid_theta(p, 11), grid_theta(q, 5)
    u = theta[:, None] + zeta[None, :]
    idx = (np.arange(p)[:, None] * 7 + np.arange(q)[None, :] * 3) % len(GAM_VALUES)
    gam = np.asfortranarray(GAM_VALUES[idx])
    with _context(6, p, q, seed=p + q) as ctx:
        ctx.set_state(gam, np.zeros((p, q)))
        t0, t1, part = _both_paths(ctx, theta, zeta, c)
    check_tables(t0, u, c, what=(p, q))
    check_tables(t1, u, c, what=(p, q))
    _check_paths_agree(t0, t1, what=(p, q))
    want, bar = elbo_reference(u, gam)
    assert abs(part - want) <= bar, (part, want, bar)


@pytest.mark.gpu
def test_tables_past_the_row_grid_limit():
    """p = 524,289: more 8-row blocks than gridDim.y can hold (65,535), so the pass takes two launches.  The first and
    last 64 rows of every table, and the ELBO part over all rows."""
    p, q = 524289, 1
    theta, zeta = grid_theta(p, 11), np.array([0.25])
    u = theta[:, None] + zeta[None, :]
    gam = np.asfortranarray(GAM_VALUES[np.arange(p) % len(GAM_VALUES)][:, None])
    rows = np.r_[0:64, p - 64:p]
    with _context(2, p, q) as ctx:
        ctx.set_state(gam, np.zeros((p, q)))
        before = ctx.launch_count()
        ctx.refresh_tables(theta, zeta, c_next=1.0, want_elbo=False)
        assert ctx.launch_count() - before == 2   # 65,535 + 2 row blocks
        t0 = ctx.get_tables()
        part = ctx.refresh_tables(theta, zeta, c_next=0.5, want_elbo=True)
        t1 = ctx.get_tables()
        again = ctx.refresh_tables(theta, zeta, c_next=0.5, want_elbo=True)
    check_tables({k: v[rows] for k, v in t0.items()}, u[rows], 1.0, what="p=524289 c=1")
    check_tables({k: v[rows] for k, v in t1.items()}, u[rows], 0.5, what="p=524289 c=0.5")
    # the rows in between were written too: D does not depend on c, and both paths agree everywhere
    _check_paths_agree(t0, t1, what="p=524289")
    want, bar = elbo_reference(u, gam)
    assert abs(part - want) <= bar, (part, want, bar)
    assert part == again


# ----------------------------------------------------------------------------- GPU: the ELBO part, region by region
ELBO_BANDS = {
    "negative_tail": np.concatenate([np.arange(-40 * 16, -5 * 16 + 1) / 16.0, -BAND, [-100.0, -1e3]]),
    "central": np.concatenate([np.arange(-63, 64) / 64.0, [0.0, -0.0, 1e-300, -1e-300, 1e-12, -1e-12, 1e-6, -1e-6]]),
    "positive_tail": np.concatenate([np.arange(5 * 16, 40 * 16 + 1) / 16.0, BAND, [100.0, 1e3]]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("band", list(ELBO_BANDS))
def test_elbo_part_by_band(band):
    """One context per band of u, so that the large terms of one region cannot hide the errors of another: gam = 1
    everywhere gives sum lp, gam = 0 gives sum lq (plus the entropy terms of gam = 1 / 0).  Twice on the same inputs is
    bit-identical."""
    u = ELBO_BANDS[band]
    p = len(u)
    with _context(3, p, 1) as ctx:
        for g in (1.0, 0.0):
            gam = np.full((p, 1), g)
            ctx.set_state(gam, np.zeros((p, 1)))
            part = ctx.refresh_tables(u, np.zeros(1), want_elbo=True)
            assert ctx.refresh_tables(u, np.zeros(1), want_elbo=True) == part
            want, bar = elbo_reference(u[:, None], gam)
            assert abs(part - want) <= bar, (band, g, part, want, bar)


@pytest.mark.gpu
def test_elbo_part_entropy_terms():
    """gam at the edges of the entropy terms with eps = .Machine$double.eps^0.75 ~ 1.82e-12: 0, 1, the smallest
    subnormal, 1e-300, 1.8e-12 (about eps), 0.5 and 1 - 2^-53, on |u| < 1 where lp and lq are O(1)."""
    gvals = np.array([0.0, 1.0, 5e-324, 1e-300, 1.8e-12, 0.5, 1 - 2.0 ** -53])
    theta = np.arange(-48, 49) / 64.0
    p, q = len(theta), len(gvals)
    gam = np.asfortranarray(np.tile(gvals, (p, 1)))
    u = theta[:, None] + np.zeros(q)[None, :]
    with _context(3, p, q) as ctx:
        ctx.set_state(gam, np.zeros((p, q)))
        part = ctx.refresh_tables(theta, np.zeros(q), want_elbo=True)
        assert ctx.refresh_tables(theta, np.zeros(q), want_elbo=True) == part
    want, bar = elbo_reference(u, gam)
    assert abs(part - want) <= bar, (part, want, bar)
    # the bar resolves eps itself: log(1 + eps) of the gam = 1 column alone adds p eps
    assert p * ELBO_EPS > 10 * bar


# ----------------------------------------------------------------------------- GPU: against the reference's own R code
@pytest.mark.gpu
def test_tables_match_r_inv_mills_ratio_and_update_z():
    """tests/golden/rlite_functions.npz: inv_mills_ratio_ and update_Z_ of the reference at 156 points (including -38,
    -20, 8, 20, 37 and 0).  R forms imr0 as exp(-U^2/2 - log sqrt(2 pi) - log Phi(U)), which loses about 3e-13 relative
    at U = -38; that loss is in R's value, not the kernel's, and sets the 1e-12 bar.  z = (gam W + I0) / sqrt(c) + u
    cancels (z = -9.6e-4 at u = 3.09 from terms of size 3.7, where R's own z is 1.4e-12 off the exact value), so its bar
    is 1e-12 relative to the size of the terms it adds."""
    g = np.load(GOLDEN)
    U = g["imr_U"].ravel(order="F")
    gam = g["z_gam"].ravel(order="F")
    zeta = np.zeros(1)
    with _context(3, len(U), 1) as ctx:
        for c, z_want in ((1.0, g["z_c1"]), (0.7, g["z_c07"])):
            ctx.refresh_tables(U, zeta, c_next=c)
            t = ctx.get_tables(D=False)
            W, I0 = t["W"][:, 0], t["I0"][:, 0]
            if c == 1.0:
                np.testing.assert_allclose(I0, g["imr_0"].ravel(order="F"), rtol=1e-12, atol=0)
                np.testing.assert_allclose(W, (g["imr_1"] - g["imr_0"]).ravel(order="F"), rtol=1e-12, atol=0)
            z = (gam * W + I0) / np.sqrt(c) + U
            size = (np.abs(gam * W) + np.abs(I0)) / np.sqrt(c) + np.abs(U)
            bad = ~(np.abs(z - z_want.ravel(order="F")) <= 1e-12 * size)
            assert not bad.any(), (c, U[bad], z[bad], z_want.ravel(order="F")[bad])


# ----------------------------------------------------------------------------- GPU: row and column sums of the Z part
def _exact_zsums(gam, W, I0):
    """Exact (fsum) row and column sums of gam W + I0, and their bars 64 eps sum(|gam W| + |I0|)."""
    gw = gam * W
    mag = np.abs(gw) + np.abs(I0)
    rows = np.array([math.fsum(np.concatenate([gw[j], I0[j]]).tolist()) for j in range(gw.shape[0])])
    cols = np.array([math.fsum(np.concatenate([gw[:, k], I0[:, k]]).tolist()) for k in range(gw.shape[1])])
    return rows, 64 * EPS * mag.sum(axis=1), cols, 64 * EPS * mag.sum(axis=0)


def _clear_overrides(monkeypatch):
    for k in ("AQ_NSEG", "AQ_NO_SEG", "AQ_NO_TAIL", "AQ_FORCE_CLUSTER", "AQ_MIS_KERNEL"):
        monkeypatch.delenv(k, raising=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n,p,q,no_tail,missing", [
    (100, 16, 4776, True, False),    # single CTA, more tiles than one round: the sweep's per-tile partials only
    (100, 16, 4777, False, False),   # partials of the full rounds + one streamed row for the 8-trait tail (odd width)
    (64, 9, 33, False, False),       # all traits in 8-trait tail tiles; odd q through the streamed pass
    (1100, 20, 71, False, False),    # sample-split clusters: streamed
    (200, 24, 41, False, True),      # missing responses: streamed
], ids=["partials", "partials_tail", "odd_q", "cluster", "missing"])
def test_zpart_row_and_column_sums_are_exact_sums_of_the_tables(monkeypatch, n, p, q, no_tail, missing):
    """rowsum_zpart after a sweep (whichever route the sweep left), after a fresh refresh of the same tables (the
    streamed rowsums_kernel), and the sweep's colsum_zpart, each against fsum of gam_new W + I0 over the downloaded
    state and tables."""
    from atlasqtl_b200.device import SweepContext
    _clear_overrides(monkeypatch)
    if no_tail:
        monkeypatch.setenv("AQ_NO_TAIL", "1")
    c = 0.8
    rng = np.random.default_rng(n + p + q)
    X = rng.normal(size=(n, p))
    X = np.asfortranarray((X - X.mean(0)) / X.std(0, ddof=1))
    Y = rng.normal(size=(n, q))
    Y = np.asfortranarray(Y - Y.mean(0))
    si = sweep_inputs(X, Y, None, c=c)
    si["theta"] = si["theta"] - 3.0 * (np.arange(p) % 3)   # some pairs deep in the negative tail, I0 exponentially small
    with SweepContext(X, Y) as ctx:
        if missing:
            mi = mis_inputs(X, Y, si)
            ctx.set_missing(mi["mis"])
            ctx.set_state_mis(si["gam"], si["mu"])
            ctx.refresh_tables(si["theta"], si["zeta"], c_next=c)
            out = ctx.sweep_mis(c, si["log_sig2_inv"], mi["sig2_inv"], si["tau"], si["log_tau"])
        else:
            ctx.set_state(si["gam"], si["mu"])
            ctx.refresh_tables(si["theta"], si["zeta"], c_next=c)
            out = ctx.sweep(c, si["log_sig2_inv"], si["tau"], si["log_tau"], si["sig2_beta"])
            plan = ctx.sweep_plan()
            if q > 4000:
                assert plan["ntiles"] > plan["groups"], plan
        rows_sweep = ctx.rowsums_zpart()
        gam = ctx.get_state(mu=False, beta=False)["gam_vb"]
        tabs = ctx.get_tables(D=False)
        ctx.refresh_tables(si["theta"], si["zeta"], c_next=c)   # same tables; drops the sweep's partials
        rows_streamed = ctx.rowsums_zpart()
        again = ctx.get_tables(D=False)
    np.testing.assert_array_equal(again["W"], tabs["W"])
    rows, rbar, cols, cbar = _exact_zsums(gam, tabs["W"], tabs["I0"])
    for name, got in (("sweep", rows_sweep), ("streamed", rows_streamed)):
        bad = ~(np.abs(got - rows) <= rbar)
        assert not bad.any(), (name, np.flatnonzero(bad)[:5], got[bad][:5], rows[bad][:5])
    bad = ~(np.abs(out["colsum_zpart"] - cols) <= cbar)
    assert not bad.any(), (np.flatnonzero(bad)[:5], out["colsum_zpart"][bad][:5], cols[bad][:5])
