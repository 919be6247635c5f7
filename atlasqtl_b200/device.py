"""`SweepContext`: Python face of one aq_ctx (one GPU, one slab of traits)."""
import ctypes

import numpy as np

from . import _lib


class SweepContext:
    """Owns the device state of the CAVI sweep for q_local traits (include/atlasqtl_b200.h)."""

    def __init__(self, X, Y, device=0):
        self._lib = _lib.load()
        X = _lib.fmat(X)
        Y = _lib.fmat(Y)
        if X.shape[0] != Y.shape[0]:
            raise ValueError("X and Y must have the same number of rows")
        self.n, self.p = X.shape
        self.q = Y.shape[1]
        self._ctx = ctypes.c_void_p()
        _lib.check(self._lib.aq_create(ctypes.byref(self._ctx), ctypes.c_int(device), self.n, self.p, self.q,
                                       _lib.dptr(X), _lib.dptr(Y)))
        self.device = device

    @classmethod
    def from_prepared(cls, prep, Y_raw):
        """Context over the kept, device-standardised columns of `prep` (aq_create_prepared): Y_raw is centred on the
        device over its observed entries (NaN = missing, set to 0); `n_obs` holds the observed counts per trait."""
        self = cls.__new__(cls)
        self._lib = _lib.load()
        Y = _lib.fmat(Y_raw)
        if Y.shape[0] != prep.n:
            raise ValueError("X and Y must have the same number of samples.")
        self.n, self.p, self.q = prep.n, prep.p, Y.shape[1]
        self._ctx = ctypes.c_void_p()
        self.n_obs = np.empty(self.q)
        _lib.check(self._lib.aq_create_prepared(ctypes.byref(self._ctx), prep._prep, self.q, _lib.dptr(Y),
                                                _lib.dptr(self.n_obs)))
        self.device = prep.device
        return self

    def get_x(self):
        X = np.empty((self.n, self.p), order="F")
        _lib.check(self._lib.aq_get_x(self._ctx, _lib.dptr(X)))
        return X

    def release_x(self):
        """Free the untiled device copy of X (aq_release_x): fixed sweep order, no missing responses from here on."""
        _lib.check(self._lib.aq_release_x(self._ctx))

    def get_y(self):
        Y = np.empty((self.n, self.q), order="F")
        _lib.check(self._lib.aq_get_y(self._ctx, _lib.dptr(Y)))
        return Y

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.aq_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def dims(self):
        v = [ctypes.c_int() for _ in range(5)]
        _lib.check(self._lib.aq_dims(self._ctx, *[ctypes.byref(x) for x in v]))
        return dict(zip(("n", "p", "q", "p_pad", "q_pad"), (x.value for x in v)))

    def set_order(self, shuffled_ind=None):
        arr = None if shuffled_ind is None else np.ascontiguousarray(shuffled_ind, dtype=np.int32)
        if arr is not None and arr.shape != (self.p,):
            raise ValueError("shuffled_ind must have length p")
        _lib.check(self._lib.aq_set_order(self._ctx, _lib.iptr(arr)))

    def _qvecs(self, k):
        return [np.empty(self.q) for _ in range(k)]

    def set_state(self, gam_vb, mu_beta_vb):
        g, m = _lib.fmat(gam_vb), _lib.fmat(mu_beta_vb)
        if g.shape != (self.p, self.q) or m.shape != (self.p, self.q):
            raise ValueError("gam_vb / mu_beta_vb must be p x q")
        o = self._qvecs(4)
        _lib.check(self._lib.aq_set_state(self._ctx, _lib.dptr(g), _lib.dptr(m), *[_lib.dptr(x) for x in o]))
        return dict(colsum_gam=o[0], colsum_gam_mu2=o[1], colsum_beta2=o[2], resid_sq=o[3])

    def get_state(self, gam=True, mu=True, beta=True):
        outs = [np.empty((self.p, self.q), order="F") if f else None for f in (gam, mu, beta)]
        _lib.check(self._lib.aq_get_state(self._ctx, *[_lib.dptr(x) for x in outs]))
        return dict(gam_vb=outs[0], mu_beta_vb=outs[1], beta_vb=outs[2])

    def snapshot(self):
        """Freeze gam_vb / mu_beta_vb on the device in stream order (aq_snapshot); later sweeps do not disturb it."""
        _lib.check(self._lib.aq_snapshot(self._ctx))

    def snapshot_fetch(self, gam=True, mu=True, beta=True):
        """Download the frozen state (aq_snapshot_fetch) on the copy stream; may run on another thread while this
        context keeps sweeping."""
        outs = [np.empty((self.p, self.q), order="F") if f else None for f in (gam, mu, beta)]
        _lib.check(self._lib.aq_snapshot_fetch(self._ctx, *[_lib.dptr(x) for x in outs]))
        return dict(gam_vb=outs[0], mu_beta_vb=outs[1], beta_vb=outs[2])

    def get_residual(self):
        r = np.empty((self.n, self.q), order="F")
        _lib.check(self._lib.aq_get_residual(self._ctx, _lib.dptr(r)))
        return r

    def refresh_tables(self, theta_vb, zeta_vb, c_next=1.0, want_elbo=False):
        th = np.ascontiguousarray(theta_vb, dtype=np.float64)
        ze = np.ascontiguousarray(zeta_vb, dtype=np.float64)
        if th.shape != (self.p,) or ze.shape != (self.q,):
            raise ValueError("theta_vb must have length p and zeta_vb length q_local")
        out = ctypes.c_double()
        _lib.check(self._lib.aq_refresh_tables(self._ctx, _lib.dptr(th), _lib.dptr(ze), ctypes.c_double(c_next),
                                               ctypes.byref(out) if want_elbo else None))
        return out.value if want_elbo else None

    def get_tables(self, D=True, W=True, I0=True):
        """The tables of the last refresh_tables (aq_get_tables), p x q_local: D = log(1 - Phi(u)) - log Phi(u), W and I0."""
        outs = [np.empty((self.p, self.q), order="F") if f else None for f in (D, W, I0)]
        _lib.check(self._lib.aq_get_tables(self._ctx, *[_lib.dptr(x) for x in outs]))
        return dict(D=outs[0], W=outs[1], I0=outs[2])

    def sweep(self, c, log_sig2_inv_vb, tau_vb, log_tau_vb, sig2_beta_vb):
        vecs = [np.ascontiguousarray(v, dtype=np.float64) for v in (tau_vb, log_tau_vb, sig2_beta_vb)]
        for v in vecs:
            if v.shape != (self.q,):
                raise ValueError("per-trait vectors must have length q_local")
        o = self._qvecs(5)
        _lib.check(self._lib.aq_sweep(self._ctx, ctypes.c_double(c), ctypes.c_double(log_sig2_inv_vb),
                                      *[_lib.dptr(v) for v in vecs], *[_lib.dptr(x) for x in o]))
        return dict(colsum_gam=o[0], colsum_gam_mu2=o[1], colsum_beta2=o[2], resid_sq=o[3], colsum_zpart=o[4])

    # ---- missing responses (coreDualMisLoop; include/atlasqtl_b200.h)
    def set_missing(self, mis_pat):
        """mis_pat: n x q_local, 1 where y is observed, 0 where missing.  Returns colSums(mis_pat)."""
        m = _lib.fmat(mis_pat)
        if m.shape != (self.n, self.q):
            raise ValueError("mis_pat must be n x q_local")
        n_obs = np.empty(self.q)
        _lib.check(self._lib.aq_set_missing(self._ctx, _lib.dptr(m), _lib.dptr(n_obs)))
        return n_obs

    def set_state_mis(self, gam_vb, mu_beta_vb):
        g, m = _lib.fmat(gam_vb), _lib.fmat(mu_beta_vb)
        if g.shape != (self.p, self.q) or m.shape != (self.p, self.q):
            raise ValueError("gam_vb / mu_beta_vb must be p x q")
        o = self._qvecs(7)
        _lib.check(self._lib.aq_set_state_mis(self._ctx, _lib.dptr(g), _lib.dptr(m), *[_lib.dptr(x) for x in o]))
        return dict(zip(("colsum_gam", "colsum_gam_mu2", "colsum_beta2", "resid_sq", "colsum_xn_gam",
                         "colsum_xn_gam_mu2", "colsum_xn_beta2"), o))

    def sweep_mis(self, c, log_sig2_inv_vb, sig2_inv_vb, tau_vb, log_tau_vb):
        vecs = [np.ascontiguousarray(v, dtype=np.float64) for v in (tau_vb, log_tau_vb)]
        for v in vecs:
            if v.shape != (self.q,):
                raise ValueError("per-trait vectors must have length q_local")
        o = self._qvecs(9)
        _lib.check(self._lib.aq_sweep_mis(self._ctx, ctypes.c_double(c), ctypes.c_double(log_sig2_inv_vb),
                                          ctypes.c_double(sig2_inv_vb), *[_lib.dptr(v) for v in vecs],
                                          *[_lib.dptr(x) for x in o]))
        return dict(zip(("colsum_gam", "colsum_gam_mu2", "colsum_sig2b_gam", "colsum_xn_gam_mu2", "colsum_xn_sig2b_gam",
                         "colsum_xn_beta2", "resid_sq", "colsum_zpart", "colsum_gam_logsig2b"), o))

    # ---- selection sets on the device (R/summarise_output.R:99-106, :207-223)
    def ppi_count_sum(self, t):
        """(#{1 - gam_vb <= t}, sum of those 1 - gam_vb) over this slab."""
        cnt, tot = ctypes.c_double(), ctypes.c_double()
        _lib.check(self._lib.aq_ppi_count_sum(self._ctx, ctypes.c_double(t), ctypes.byref(cnt), ctypes.byref(tot)))
        return cnt.value, tot.value

    def ppi_next_above(self, t):
        nxt = ctypes.c_double()
        _lib.check(self._lib.aq_ppi_next_above(self._ctx, ctypes.c_double(t), ctypes.byref(nxt)))
        return nxt.value

    def ppi_collect(self, mode, lo, hi, capacity):
        """Pairs with lo < 1 - gam_vb <= hi (mode 0) or gam_vb > lo (mode 1): (j, k_local, gam_vb, n_found), sorted by
        column-major index."""
        cap = int(capacity)
        j, k, g = np.empty(max(cap, 1), np.int32), np.empty(max(cap, 1), np.int32), np.empty(max(cap, 1))
        n = ctypes.c_int64()
        _lib.check(self._lib.aq_ppi_collect(self._ctx, ctypes.c_int(mode), ctypes.c_double(lo), ctypes.c_double(hi),
                                            ctypes.c_int64(cap), _lib.iptr(j), _lib.iptr(k), _lib.dptr(g), ctypes.byref(n)))
        m = min(n.value, cap)
        o = np.lexsort((j[:m], k[:m]))
        return j[:m][o], k[:m][o], g[:m][o], n.value

    def rowsums_zpart(self):
        r = np.empty(self.p)
        _lib.check(self._lib.aq_rowsums_zpart(self._ctx, _lib.dptr(r)))
        return r

    def rowsums_zpart_dev(self):
        ptr = _lib._DP()
        _lib.check(self._lib.aq_rowsums_zpart_dev(self._ctx, ctypes.byref(ptr)))
        return ctypes.cast(ptr, ctypes.c_void_p).value

    def launch_count(self):
        return int(self._lib.aq_launch_count(self._ctx))

    def sweep_plan(self):
        """How the last sweep spread its trait tiles over the GPU (aq_sweep_plan)."""
        v = [ctypes.c_int() for _ in range(4)]
        _lib.check(self._lib.aq_sweep_plan(self._ctx, *[ctypes.byref(x) for x in v]))
        return dict(zip(("traits_per_tile", "ntiles", "groups", "nseg"), (x.value for x in v)))

    def last_sweep_ms(self):
        ms = ctypes.c_float()
        _lib.check(self._lib.aq_last_sweep_ms(self._ctx, ctypes.byref(ms)))
        return ms.value

    def last_ms(self, which):
        """Device time (ms) of the last sweep (0), row-sum (1) or table (2) kernel group."""
        ms = ctypes.c_float()
        _lib.check(self._lib.aq_last_ms(self._ctx, ctypes.c_int(which), ctypes.byref(ms)))
        return ms.value

    def sync(self):
        _lib.check(self._lib.aq_sync(self._ctx))


def pack_genotypes(G):
    """n x p matrix of calls 0 / 1 / 2 -> the packed form aq_prep_geno reads: uint8 [p][ceil(n / 4)], sample i of a
    column in bits 2 (i % 4) .. 2 (i % 4) + 1 of byte i / 4."""
    G = np.asarray(G)
    if G.ndim != 2:
        raise ValueError("G must be a matrix")
    if ((G < 0) | (G > 2) | (G != np.floor(G))).any():
        raise ValueError("genotype calls must be 0, 1 or 2")
    n, p = G.shape
    nb = (n + 3) // 4
    g = np.zeros((p, nb * 4), dtype=np.uint8)
    g[:, :n] = G.T
    g = g.reshape(p, nb, 4)
    return np.ascontiguousarray(g[:, :, 0] | (g[:, :, 1] << 2) | (g[:, :, 2] << 4) | (g[:, :, 3] << 6))


class PreparedPredictors:
    """Predictors pre-processed on the device (aq_prep_x / aq_prep_geno): scale(X), constant and duplicated columns
    dropped (R/prepare_atlasqtl.R:57-72).  Stands in for the standardised X matrix in the core: `.shape` is (n, p_kept)
    and `.context(Y_raw)` creates the sweep context whose X is materialised from the raw input on the device."""

    def __init__(self, X_raw=None, *, packed=None, n=None, device=0):
        self._lib = _lib.load()
        self._prep = ctypes.c_void_p()
        self.device = device
        kept = ctypes.c_int()
        if (X_raw is None) == (packed is None):
            raise ValueError("give either X_raw or packed genotype calls")
        if X_raw is not None:
            X = _lib.fmat(X_raw)
            if X.ndim != 2:
                raise ValueError("X must be a matrix")
            self.n, self.p_raw = X.shape
            _lib.check(self._lib.aq_prep_x(ctypes.byref(self._prep), ctypes.c_int(device), self.n, self.p_raw,
                                           _lib.dptr(X), ctypes.byref(kept)))
        else:
            g = np.ascontiguousarray(packed, dtype=np.uint8)
            if g.ndim != 2 or n is None or g.shape[1] < (n + 3) // 4:
                raise ValueError("packed must be uint8 [p][>= ceil(n / 4)] and n must be given")
            self.n, self.p_raw = int(n), g.shape[0]
            _lib.check(self._lib.aq_prep_geno(ctypes.byref(self._prep), ctypes.c_int(device), self.n, self.p_raw,
                                              g.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
                                              ctypes.c_int64(g.shape[1]), ctypes.byref(kept)))
        self.p = kept.value
        self.status = np.empty(self.p_raw, np.uint8)
        self.dup_of = np.empty(self.p_raw, np.int32)
        self.mean, self.sd = np.empty(self.p_raw), np.empty(self.p_raw)
        _lib.check(self._lib.aq_prep_result(self._prep, self.status.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
                                            _lib.iptr(self.dup_of), _lib.dptr(self.mean), _lib.dptr(self.sd)))

    @property
    def shape(self):
        return (self.n, self.p)

    def context(self, Y_raw):
        return SweepContext.from_prepared(self, Y_raw)

    def launch_count(self):
        return int(self._lib.aq_prep_launch_count(self._prep))

    def close(self):
        if getattr(self, "_prep", None) is not None and self._prep:
            self._lib.aq_prep_destroy(self._prep)
            self._prep = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
