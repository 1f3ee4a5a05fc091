"""The row-stripe sharded driver (solver.LRSPnP + StripeComm) over gloo, world_size 2 and 3, on CPU.
The compute backend is substituted by the NumPy oracle (test infrastructure) so that what is
exercised here is the host logic of the N>1 path: partition, halo reduce, Gram all-reduce, halo
refresh, coverage weights of the full geometry on a stripe.  The sharded result must equal the
unsharded oracle run."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from lrs_pnp_dip_b200 import solver, synth
from oracle import lrs_oracle as orc


class OracleBackend:
    """Same five methods as solver.CudaBackend, on CPU tensors, computed by the oracle."""

    def __init__(self, Y, MtM, D, prm):
        self.Y, self.MtM, self.D, self.prm = Y.numpy(), MtM.numpy(), D, prm
        self.oprm = orc.Params(gamma=prm.gamma, mu_1=prm.mu_1, mu_2=prm.mu_2, lambda_ista=prm.lambda_ista, Nit=prm.Nit,
                               bb=prm.bb, slidingDis=prm.slidingDis, step=prm.step)

    def imout(self, X, lambda_1):
        phi, _ = orc.sparse_step(X.numpy(), lambda_1.numpy(), self.Y, self.D, self.oprm)
        R, C = self.Y.shape
        return torch.from_numpy(orc.col2im_accumulate(phi, R, C, self.prm.bb, self.prm.slidingDis))

    def gram(self, X, lambda_2, c, rows):
        Z = (X.numpy()[:rows] + np.float32(c) * lambda_2.numpy()[:rows]).astype(np.float64)
        return torch.from_numpy(Z.T @ Z)

    def svt_apply(self, X, lambda_2, c, G, tau, rows):
        Z = (X.numpy()[:rows] + np.float32(c) * lambda_2.numpy()[:rows]).astype(np.float32)
        ev, V = np.linalg.eigh(G.numpy())
        sig = np.sqrt(np.maximum(ev, 0))
        w = np.where(sig > tau, 1 - tau / np.maximum(sig, 1e-300), 0)
        return torch.from_numpy((Z.astype(np.float64) @ ((V * w[None]) @ V.T)).astype(np.float32))

    def axpy(self, X, L, c, rows):
        return torch.from_numpy((X.numpy()[:rows] + np.float32(c) * L.numpy()[:rows]).astype(np.float32))

    def admm_update(self, IMout, U, lambda_1, lambda_2, rows, row_offset, R_total):
        C = self.Y.shape[1]
        W = orc.coverage_weight(R_total, C, self.prm.bb, self.prm.slidingDis)[row_offset:row_offset + rows]
        l1 = lambda_1.numpy()[:rows]
        l1s = np.zeros_like(l1)
        for t in range(int(W.max())):
            l1s = np.where(W > t, l1s + l1, l1s).astype(np.float32)
        Xn, l1n, l2n = orc.admm_update(None, l1, lambda_2.numpy()[:rows], self.Y[:rows], self.MtM[:rows],
                                       IMout.numpy()[:rows], W, U.numpy()[:rows], l1s, self.oprm)
        lambda_1[:rows] = torch.from_numpy(l1n)
        lambda_2[:rows] = torch.from_numpy(l2n)
        return torch.from_numpy(Xn)


def _problem(H=10, W=9):
    B = 14
    clean, noisy = synth.synthetic_cube(H, W, B, rank=3, seed=5)
    pm = synth.pixel_mask(H, W, "bernoulli", keep=0.65, seed=6)
    Y = synth.observe(noisy, pm)
    MtM = np.repeat(pm.astype(np.float32)[:, None], B, axis=1)
    D = synth.synthetic_dictionary(64, 48, seed=0)
    prm = solver.Params(mu_1=0.15, mu_2=0.9, Nit=15, bb=8, slidingDis=1, step="frob4")
    return Y, MtM, D, prm


DUMP_TEST_BYTES = 30 * 3 * 14 * 4          # bench.DUMP_BYTES that makes the 90 x 14 state of _problem() a 30-row sample


def _worker(rank, world, port, iters, out_dir, H=10, W=9, dump=False):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.set_num_threads(1)
        Y, MtM, D, prm = _problem(H, W)
        st = solver.make_stripe(Y.shape[0], prm.bb, rank, world)
        Yl = torch.from_numpy(Y[st.row_slice].copy())
        Ml = torch.from_numpy(MtM[st.row_slice].copy())
        be = OracleBackend(Yl, Ml, D, prm)
        sol = solver.LRSPnP(Yl, Ml, D, prm, stripe=st, backend=be)
        sol.run(iters)
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), X=sol.X.numpy()[:st.rows_owned], a=st.a,
                 l1=sol.lambda_1.numpy()[:st.rows_owned], l2=sol.lambda_2.numpy()[:st.rows_owned],
                 halo_X=sol.X.numpy()[st.rows_owned:])
        if dump:                                         # what bench.py --dump-outputs gathers on N ranks
            import bench

            bench.DUMP_BYTES = DUMP_TEST_BYTES
            got = bench.state_rows(torch, dist, sol, st, bench.dump_rows(*Y.shape), rank, world)
            if rank == 0:
                np.savez(os.path.join(out_dir, "dump.npz"), **got)
            else:
                assert got is None
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_equals_unsharded(world, tmp_path):
    iters = 2
    mp.spawn(_worker, args=(world, _free_port(), iters, str(tmp_path)), nprocs=world, join=True)
    Y, MtM, D, prm = _problem()
    oprm = orc.Params(gamma=prm.gamma, mu_1=prm.mu_1, mu_2=prm.mu_2, lambda_ista=prm.lambda_ista, Nit=prm.Nit, bb=prm.bb,
                      slidingDis=prm.slidingDis, step=prm.step)
    ref = orc.run(Y, MtM, D, oprm, iteration_num=iters)
    X = np.zeros_like(Y)
    l1 = np.zeros_like(Y)
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        a = int(z["a"])
        X[a:a + z["X"].shape[0]] = z["X"]
        l1[a:a + z["l1"].shape[0]] = z["l1"]
        # the refreshed halo equals the right neighbour's owned rows
        if r + 1 < world:
            h = z["halo_X"].shape[0]
            assert h == prm.bb - 1
    err = np.linalg.norm(X - ref.X) / np.linalg.norm(ref.X)
    assert err < 2e-5, err
    assert np.linalg.norm(l1 - ref.lambda_1) / np.linalg.norm(ref.lambda_1) < 1e-4


def test_bench_dump_gathers_sampled_rows_over_stripes(tmp_path, monkeypatch):
    """bench.py --dump-outputs on N ranks: the fixed row sample (forced here by a small DUMP_BYTES) is gathered on rank 0
    from the stripes that own its rows, the last rank's trailing bb-1 rows included, in row order and unchanged."""
    import bench

    world = 3
    mp.spawn(_worker, args=(world, _free_port(), 2, str(tmp_path), 10, 9, True), nprocs=world, join=True)
    Y, _, _, prm = _problem()
    R, C = Y.shape
    monkeypatch.setattr(bench, "DUMP_BYTES", DUMP_TEST_BYTES)
    rows = bench.dump_rows(R, C)
    assert len(rows) == 30 and rows[-1] >= R - (prm.bb - 1)
    full = {n: np.full_like(Y, np.nan) for n in bench.STATE}
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        a = int(z["a"])
        for n, key in zip(bench.STATE, ("X", "l1", "l2")):
            full[n][a:a + z[key].shape[0]] = z[key]
    got = np.load(tmp_path / "dump.npz")
    for n in bench.STATE:
        assert got[n].dtype == np.float32 and np.array_equal(got[n], full[n][rows]), n


def test_stripes_as_narrow_as_the_halo(tmp_path):
    """Boundary of the neighbour-only halo exchange: 14 patch rows over 2 ranks = 7 per stripe = bb-1, the narrowest
    stripe whose halo lies entirely inside the immediate neighbour's owned rows.  One row fewer must be refused."""
    iters, world, H, W = 2, 2, 3, 7                      # R = 21 unfolded rows
    mp.spawn(_worker, args=(world, _free_port(), iters, str(tmp_path), H, W), nprocs=world, join=True)
    Y, MtM, D, prm = _problem(H, W)
    oprm = orc.Params(gamma=prm.gamma, mu_1=prm.mu_1, mu_2=prm.mu_2, lambda_ista=prm.lambda_ista, Nit=prm.Nit, bb=prm.bb,
                      slidingDis=prm.slidingDis, step=prm.step)
    ref = orc.run(Y, MtM, D, oprm, iteration_num=iters)
    X = np.zeros_like(Y)
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        X[int(z["a"]):int(z["a"]) + z["X"].shape[0]] = z["X"]
    assert np.linalg.norm(X - ref.X) / np.linalg.norm(ref.X) < 2e-5
    with pytest.raises(ValueError, match="narrower than the halo"):
        solver.make_stripe(20, 8, 0, 2)                  # 13 patch rows -> stripes of 6 and 7
    with pytest.raises(ValueError, match="narrower than the halo"):
        solver.make_stripe(90, 8, 1, 12)


def test_unsharded_driver_with_oracle_backend_matches_oracle_run():
    Y, MtM, D, prm = _problem()
    be = OracleBackend(torch.from_numpy(Y), torch.from_numpy(MtM), D, prm)
    sol = solver.LRSPnP(torch.from_numpy(Y.copy()), torch.from_numpy(MtM), D, prm, backend=be)
    sol.run(2)
    oprm = orc.Params(gamma=prm.gamma, mu_1=prm.mu_1, mu_2=prm.mu_2, lambda_ista=prm.lambda_ista, Nit=prm.Nit, bb=prm.bb,
                      slidingDis=prm.slidingDis, step=prm.step)
    ref = orc.run(Y, MtM, D, oprm, iteration_num=2)
    assert np.linalg.norm(sol.X.numpy() - ref.X) / np.linalg.norm(ref.X) < 2e-5
