"""Loader of the tests/golden/rlite_*.npz fixtures (inputs + outputs of the reference's R code, see
tests/golden/make_rlite_golden.py), shared by the CPU and GPU tests."""
import glob
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CORE_FILES = sorted(glob.glob(os.path.join(GOLD, "rlite_core_*.npz")))
CORE_IDS = [os.path.basename(f)[11:-4] for f in CORE_FILES]
HYPER_KEYS = ("q_hyper", "p_hyper", "A2_inv", "eta", "kappa", "m0", "n0", "nu", "rho", "t02")
INIT_KEYS = ("q_init", "p_init", "gam_vb", "mu_beta_vb", "sig02_inv_vb", "sig2_beta_vb", "sig2_theta_vb", "tau_vb",
             "theta_vb", "zeta_vb")


def hyper_init_of(g):
    hyper = {k: (g["hyper_" + k] if g["hyper_" + k].ndim else g["hyper_" + k].item()) for k in HYPER_KEYS}
    init = {k: (g["init_" + k] if g["init_" + k].ndim else g["init_" + k].item()) for k in INIT_KEYS}
    return hyper, init


def load_case(path):
    g = dict(np.load(path))
    init_part = os.path.join(GOLD, "rlite_init_" + os.path.basename(path)[len("rlite_core_"):])
    if os.path.exists(init_part):   # a fixture over 1 MB keeps its initial p x q matrices there
        g.update(np.load(init_part))
    hyper, init = hyper_init_of(g)
    anneal = None if np.isnan(g["anneal"][0]) else tuple(float(a) for a in g["anneal"])
    return g, hyper, init, anneal
