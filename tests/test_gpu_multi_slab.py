"""GPU: the multi-GPU path on hardware.

 (1) Two (three) trait slabs as separate CUDA contexts on ONE device, driven by the real core loop in one thread each with
     an in-process all-reduce (tests/thread_comm.py): every slab runs the real kernels; the only thing replaced is NCCL.
     Traits are independent inside a sweep (reference src/coreLoop.cpp:58-85) and coupled only through rowSums(Z)
     (R/update_vb.R:179), so the sharded run must reproduce the single-context run.
 (2) The same through torch.distributed / NCCL with one process per GPU (torchrun), when the box has >= 2 GPUs."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from problems import make_problem

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _nan(Y, frac):
    if not frac:
        return Y
    Ym = Y.copy()
    Ym[np.random.default_rng(3).uniform(size=Y.shape) < frac] = np.nan
    return Ym


@pytest.mark.parametrize("n,p,q,world,anneal,nan_frac", [
    (200, 300, 203, 2, (1, 2, 10), 0.0),
    (500, 400, 150, 3, None, 0.0),
    (1000, 320, 2500, 2, (1, 2, 5), 0.0),    # 79 tiles per slab (+ ragged last tile); one context: 157 tiles on 148 SMs
    (150, 120, 61, 2, (1, 2, 5), 0.06),      # missing responses: per-slab masks, X_norm_sq, n_obs
])
def test_slabs_on_one_device_reproduce_single_context(n, p, q, world, anneal, nan_frac):
    from atlasqtl_b200 import core, summarise
    from atlasqtl_b200.device import SweepContext
    from atlasqtl_b200.dist import slab_bounds
    from thread_comm import ThreadGroup
    X, Y, hyper, init = make_problem(n, p, q)
    Y = _nan(Y, nan_frac)
    q = Y.shape[1]
    p = X.shape[1]
    tr1 = []
    with SweepContext(X, np.where(np.isnan(Y), 0.0, Y)) as ctx1:
        one = core.atlasqtl_global_local_core_(Y, X, q, anneal, 1, 0.1, 60, 0, hyper, init, debug=True, trace=tr1, ctx=ctx1)
        sel1 = summarise.select_bFDR_device(ctx1, 0.05)
    group = ThreadGroup(world)
    res, traces, sels, errs = [None] * world, [[] for _ in range(world)], [None] * world, []

    def work(rank):
        try:
            k0, k1 = slab_bounds(q, rank, world)
            Ys = np.asfortranarray(Y[:, k0:k1])
            comm = group.comm(rank)
            with SweepContext(X, np.where(np.isnan(Ys), 0.0, Ys)) as ctx:
                res[rank] = core.atlasqtl_global_local_core_(Ys, X, q, anneal, 1, 0.1, 60, 0, hyper, init, debug=True,
                                                             comm=comm, slab=(k0, k1), trace=traces[rank], ctx=ctx)
                sels[rank] = summarise.select_bFDR_device(ctx, 0.05, comm=comm, k_first=k0, p=p)
        except BaseException as e:   # do not leave the peers stuck in the barrier
            errs.append(e)
            group.barrier.abort()

    th = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    assert all(r["it"] == one["it"] and r["converged"] == one["converged"] for r in res)
    gam = np.concatenate([r["gam_vb"] for r in res], axis=1)
    beta = np.concatenate([r["beta_vb"] for r in res], axis=1)
    # the all-reduce adds the slabs' row sums in another order than one context does: agreement to rounding, not bitwise
    assert np.abs(gam - one["gam_vb"]).max() <= 1e-10
    assert np.abs(beta - one["beta_vb"]).max() <= 1e-10
    np.testing.assert_allclose(res[0]["theta_vb"], one["theta_vb"], rtol=1e-9, atol=1e-11)
    np.testing.assert_allclose(np.concatenate([r["zeta_vb"] for r in res]), one["zeta_vb"], rtol=1e-9, atol=1e-11)
    for a, b in zip(tr1, traces[0]):
        assert (a["lb"] is None) == (b["lb"] is None)
        if a["lb"] is not None:
            assert abs(a["lb"] - b["lb"]) <= 1e-11 * abs(a["lb"])
        assert abs(a["sum_gam"] - b["sum_gam"]) <= 1e-9 * max(1.0, abs(a["sum_gam"]))
    # every rank saw the same replicated quantities
    for r in range(1, world):
        assert np.array_equal(res[r]["theta_vb"], res[0]["theta_vb"])
        assert [t["lb"] for t in traces[r]] == [t["lb"] for t in traces[0]]
    # selection over slabs == selection in one context
    got = np.zeros((p, q), bool)
    for rows, cols, nsel in sels:
        got[rows, cols] = True
        assert nsel == sel1[2]
    want = np.zeros((p, q), bool)
    want[sel1[0], sel1[1]] = True
    assert np.array_equal(got, want)


def test_nccl_two_ranks_reproduce_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from atlasqtl_b200 import core
    out = tmp_path / "nccl.npz"
    port = 29600 + (os.getpid() % 1000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "nccl_worker.py"), str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    d = np.load(out)
    X, Y, hyper, init = make_problem(300, 240, 2500, seed=7)
    q = Y.shape[1]
    tr = []
    one = core.atlasqtl_global_local_core_(Y, X, q, (1, 2, 5), 1, 0.1, 40, 0, hyper, init, debug=True, trace=tr)
    assert int(d["it"]) == one["it"]
    lbs = np.array([t["lb"] for t in tr if t["lb"] is not None])
    np.testing.assert_allclose(d["lbs"], lbs, rtol=1e-11)
    assert np.abs(d["gam"] - one["gam_vb"]).max() <= 1e-10
    np.testing.assert_allclose(d["theta"], one["theta_vb"], rtol=1e-9, atol=1e-11)
    # default (unseeded) initialisation under a communicator: every rank must have drawn the same replicated state
    assert bool(d["default_init_consistent"])
