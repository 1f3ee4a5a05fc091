"""The row-stripe sharded solver on ONE GPU, stripe by stripe, against the whole-cube run and fp64.

A sharded run gives each rank a stripe of patch row-starts plus the bb-1 halo rows that follow, runs every kernel on the
stripe's own geometry, completes the overlap sums of the first bb-1 owned rows with the left neighbour's partial sums,
all-reduces the band Gram matrix and refreshes the halo rows of X and lambda_1.  None of that needs several GPUs:

A. Stripe-local kernels (one process): the Phi_z columns of every stripe against the same columns of the whole cube (all
   fused engines, the explicit engine, every step mode), the stripe-local overlap sum after an emulated halo reduce
   against the whole-cube overlap sum (bit-exact off the seams, within the reassociation bound on them), and the low-rank
   kernels and the X / multiplier update with rows = rows_owned and NaN in every halo row they must not read.
B. The driver over W = 2, 3, 4 processes sharing the device: gloo between them, the halo rows and the Gram matrix staged
   through host memory (HostStagedComm).  Each case against the unsharded GPU run and the fp64 oracle after 1 and 3
   outer iterations, the reduced overlap sum bit for bit off the seams, the refreshed halos, the same G and W on every
   rank; and a diverged state that every rank must report.
C. CPU self-checks of the helpers above: HostStagedComm against StripeComm with the NumPy backend over gloo, and the
   patch index map, seam rows and reassociation bound on a stripe of the oracle's overlap sum.

GPU tests: pytest -m gpu tests/test_sharded_one_gpu.py.  All inputs come from seeded generators.
"""
import functools
import os
from datetime import timedelta

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from lrs_pnp_dip_b200 import _lib, ops, solver, synth
from oracle import lrs_oracle as orc
from tests.test_ista_edges import ista_plan
from tests.test_kernel_edges import F32_EPS, _check_apply, _check_gram, rel, svt_weights_fp64
from tests.test_sharded_gloo import OracleBackend, _free_port
from tests.test_sharded_gloo import _problem as gloo_problem

WORLDS = (2, 3, 4)
F32 = np.float32
MU1, MU2 = 0.15, 0.9


def gpu_test(fn):
    """Marked gpu (pytest -m gpu on the B200 box) and skipped where no CUDA device is present."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(fn))


# ================================================================ helpers (host)
class HostStagedComm(solver.StripeComm):
    """StripeComm whose messages travel through host memory, so that gloo can carry them and several ranks can share one
    device: each tensor to exchange and the Gram matrix are copied to the host, the StripeComm operation runs on the
    copies, and the result is copied back on the current stream."""

    def _exchange(self, send_to_right, send_to_left, like):
        host = lambda t: None if t is None else t.cpu()                               # noqa: E731
        from_left, from_right = super()._exchange(host(send_to_right), host(send_to_left),
                                                  torch.empty(tuple(like.shape), dtype=like.dtype))
        back = lambda t: None if t is None else t.to(like.device)                     # noqa: E731
        return back(from_left), back(from_right)

    def allreduce_sum(self, t):
        h = super().allreduce_sum(t.cpu())
        if h is not t:
            t.copy_(h)
        return t


def local_patch_columns(st: solver.Stripe, C: int) -> np.ndarray:
    """Global patch number of every patch of stripe ``st`` (stride 1, patch order row-start fastest): local patch
    ci*nR_loc + (ri - a) is global patch ci*nR + ri."""
    nR, nC = st.R_total - st.bb + 1, C - st.bb + 1
    return (np.arange(nC)[:, None] * nR + np.arange(st.a, st.b)[None, :]).reshape(-1)


def seam_rows(st: solver.Stripe) -> np.ndarray:
    """Local owned rows whose overlap sum is completed by the left neighbour's partial sum: the first bb-1 owned rows of
    every rank after rank 0."""
    return np.arange(st.halo) if st.rank > 0 else np.arange(0)


def overlap_fp64(phi, R: int, C: int, bb: int):
    """The overlap sum of ``phi`` [bb², P] in fp64, the overlap sum of |phi| (stride 1), and the number k of patches
    covering each element."""
    x, y = orc.patch_index(R, C, bb, 1)
    k = np.arange(bb * bb)
    rr = x[None, :] + (k % bb)[:, None]
    cc = y[None, :] + (k // bb)[:, None]
    phi = np.asarray(phi, np.float64)
    s, a = np.zeros((R, C)), np.zeros((R, C))
    np.add.at(s, (rr, cc), phi)
    np.add.at(a, (rr, cc), np.abs(phi))
    return s, a, orc.coverage_weight(R, C, bb, 1).astype(np.float64)


def reassociation_bound(abs_sum, k):
    """|fl32(any order of k addends) - exact| <= gamma_{k-1} sum |addend|, gamma_m = m u / (1 - m u), u = 2^-24."""
    g = np.maximum(k - 1, 0) * F32_EPS
    return g / (1 - g) * abs_sum


def emulate_halo_reduce(parts, stripes):
    """StripeComm.halo_reduce on a list of per-rank overlap sums: every rank's last bb-1 local rows (its partial sums of
    the right neighbour's first owned rows) are added to the right neighbour's first bb-1 rows, own sum first."""
    sends = [p[st.rows_local - st.halo:].copy() for p, st in zip(parts, stripes)]
    for r in range(1, len(parts)):
        parts[r][:stripes[r].halo] += sends[r - 1]
    return parts


def check_reduced_stripe(got, st, whole32, s64, bound):
    """Owned rows of one rank's reduced overlap sum: bit-exact against the whole-cube fp32 sum off the seams, within the
    reassociation bound of the fp64 sum on the seams.  Returns the number of seam elements that differ from whole32."""
    own = np.arange(st.rows_owned)
    seam = seam_rows(st)
    inner = np.setdiff1d(own, seam)
    bad = np.argwhere(got[inner] != whole32[st.a + inner])
    assert bad.size == 0, (st.rank, [(int(st.a + inner[i]), int(j)) for i, j in bad[:8]])
    err = np.abs(got[seam].astype(np.float64) - s64[st.a + seam])
    assert np.all(err <= bound[st.a + seam]), (st.rank, float((err - bound[st.a + seam]).max()))
    return int((got[seam] != whole32[st.a + seam]).sum())


def make_problem(R, C, K, bb=8, seed=0, elementwise=False, dead_rows=None):
    """(Y_observed, MtM, D): a rank-3 cube plus noise, rows (pixels) observed with probability 0.7, with ``elementwise``
    also per element; ``dead_rows``: a boolean row mask of pixels never observed."""
    rng = np.random.default_rng(seed)
    X = (rng.random((R, 3)) @ rng.random((3, C)) / 3 + 0.05 * rng.standard_normal((R, C))).astype(F32)
    M = np.repeat((rng.random(R) < 0.7)[:, None], C, axis=1)
    if elementwise:
        M &= rng.random((R, C)) < 0.8
    if dead_rows is not None:
        M[dead_rows] = False
    Y = np.where(M, X, 0).astype(F32)
    Y[M & (Y == 0)] = F32(1e-12)
    return Y, M.astype(F32), synth.synthetic_dictionary(bb * bb, K, seed=K + bb)


def state_near(Y, seed):
    """A non-trivial (X, lambda_1, lambda_2) next to Y."""
    rng = np.random.default_rng(seed)
    X = (Y + 0.3 + 0.1 * rng.standard_normal(Y.shape)).astype(F32)
    L1 = (0.01 * rng.standard_normal(Y.shape)).astype(F32)
    L2 = (0.01 * rng.standard_normal(Y.shape)).astype(F32)
    return X, L1, L2


def oracle_step_mode(step):
    return "frob4" if step == "frob4" else "spectral"       # the table and the per-patch constants are both ||M_p D||_2^2


# ================================================================ C. CPU self-checks
def _comm_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=120))
    try:
        torch.set_num_threads(1)
        Y, MtM, D, prm = gloo_problem()
        st = solver.make_stripe(Y.shape[0], prm.bb, rank, world)
        out = {}
        for name, comm in (("plain", solver.StripeComm), ("staged", HostStagedComm)):
            Yl, Ml = torch.from_numpy(Y[st.row_slice].copy()), torch.from_numpy(MtM[st.row_slice].copy())
            sol = solver.LRSPnP(Yl, Ml, D, prm, stripe=st, backend=OracleBackend(Yl, Ml, D, prm))
            sol.comm = comm(st, None)
            sol.run(2)
            for k in ("X", "lambda_1", "lambda_2"):
                out[f"{name}_{k}"] = getattr(sol, k).numpy().copy()
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), **out)
    finally:
        dist.destroy_process_group()


def test_host_staged_comm_equals_stripe_comm_on_the_oracle(tmp_path):
    """HostStagedComm (the communicator of the one-GPU driver tests below) with the NumPy backend over gloo gives
    exactly what StripeComm gives: the same halo reduce, Gram all-reduce and halo refresh, bit for bit, on every row a
    rank holds."""
    world = 3
    mp.spawn(_comm_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        z = np.load(tmp_path / f"rank{r}.npz")
        for k in ("X", "lambda_1", "lambda_2"):
            assert np.isfinite(z[f"plain_{k}"][:solver.make_stripe(90, 8, r, world).rows_owned]).all(), (r, k)
            assert np.array_equal(z[f"staged_{k}"], z[f"plain_{k}"], equal_nan=True), (r, k)


@pytest.mark.parametrize("R,C,bb", [(40, 12, 8), (31, 10, 6), (21, 9, 8)])
def test_stripe_helpers_on_the_oracle_overlap_sum(R, C, bb):
    """The host helpers of the stripe-local kernel tests, on the oracle: the local-to-global patch map matches the oracle's
    patch index; the seam rows are exactly the owned rows that a patch of another rank covers; after the emulated halo
    reduce, a stripe's oracle overlap sum equals the whole-cube sum bit for bit off the seams and stays within the
    reassociation bound on them; without the reduce the seam rows break that bound (the bound is not vacuous)."""
    rng = np.random.default_rng(R * C + bb)
    P = (R - bb + 1) * (C - bb + 1)
    phi = (rng.standard_normal((bb * bb, P)) * 10.0 ** rng.uniform(-3, 3, (1, P))).astype(F32)
    whole = orc.col2im_accumulate(phi, R, C, bb, 1)
    s64, a64, k = overlap_fp64(phi, R, C, bb)
    bound = reassociation_bound(a64, k)
    assert np.all(np.abs(whole - s64) <= bound)                      # the bound holds for the sequential order itself
    xg, yg = orc.patch_index(R, C, bb, 1)
    for world in (w for w in WORLDS if (R - bb + 1) >= w * (bb - 1)):
        stripes = [solver.make_stripe(R, bb, r, world) for r in range(world)]
        parts, cols_seen = [], []
        for st in stripes:
            cols = local_patch_columns(st, C)
            xl, yl = orc.patch_index(st.rows_local, C, bb, 1)
            assert np.array_equal(xg[cols], xl + st.a) and np.array_equal(yg[cols], yl)
            cols_seen.append(cols)
            # seam rows from the geometry: owned rows covered by a patch row-start below the stripe's first
            g = st.a + np.arange(st.rows_owned)
            covered_from_left = np.maximum(g - bb + 1, 0) < st.a
            assert np.array_equal(np.flatnonzero(covered_from_left), seam_rows(st)), (world, st.rank)
            assert len(seam_rows(st)) == (0 if st.rank == 0 else bb - 1)
            parts.append(orc.col2im_accumulate(phi[:, cols], st.rows_local, C, bb, 1))
        assert np.array_equal(np.sort(np.concatenate(cols_seen)), np.arange(P))   # every patch in exactly one stripe
        unreduced = [p.copy() for p in parts]
        emulate_halo_reduce(parts, stripes)
        differ = sum(check_reduced_stripe(p, st, whole, s64, bound) for p, st in zip(parts, stripes))
        assert differ > 0, world                                     # the seams really are summed in another order
        for p, st in zip(unreduced[1:], stripes[1:]):
            seam = seam_rows(st)
            assert np.any(np.abs(p[seam] - s64[st.a + seam]) > bound[st.a + seam]), (world, st.rank)


# ================================================================ A. stripe-local kernels against the whole cube
def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


@pytest.fixture(scope="module")
def lib():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return _lib.lib()


# engine kind -> (SparseCoder engine, bb, K): fused engines at bb = 8, K = 256; the explicit engine at K = 96 and bb = 6
KERNEL_ENGINES = {"tc": ("tc", 8, 256), "simt": ("simt", 8, 256), "explicit-K96": ("auto", 8, 96),
                  "explicit-bb6": ("auto", 6, 72)}
STEP_MODES = ("spectral", "spectral_patch", "frob4")
A_R, A_C, A_NIT = 300, 20, 12                  # 293 row starts (prime): ragged stripes, tiles cut at other lanes


def _kernel_inputs(kind, step, seed=3):
    _, bb, K = KERNEL_ENGINES[kind]
    # the row-pattern table needs masks replicated over the bands; the other modes take per-element masks
    Y, _, D = make_problem(A_R, A_C, K, bb=bb, seed=seed, elementwise=step != "spectral")
    X, L, _ = state_near(Y, seed + 1)
    return X, L, Y, D, solver.Params(mu_1=MU1, mu_2=MU2, Nit=A_NIT, bb=bb, slidingDis=1, step=step)


@pytest.mark.parametrize("step", STEP_MODES)
@pytest.mark.parametrize("kind", list(KERNEL_ENGINES))
@pytest.mark.usefixtures("lib")
@gpu_test
def test_stripe_phi_z_columns_equal_the_whole_cube(kind, step):
    """Every stripe's Phi_z (W = 2, 3, 4) equals the same columns of the whole cube's Phi_z bit for bit: the fused tcgen05
    and FFMA engines and the dynamically dealt tcgen05 instance (a patch sits at another lane of its 128-row-start tile
    inside a stripe), and the explicit engine (im2col, ISTA, same launch plan for the stripe's patch count), in the
    row-pattern table, per-patch spectral and frob4 modes.  The whole cube against the fp64 oracle: rel-L2 <= 1e-4."""
    engine, bb, K = KERNEL_ENGINES[kind]
    X, L, Y, D, prm = _kernel_inputs(kind, step)
    Dd = cu(D)
    whole = solver.SparseCoder(cu(Y), Dd, prm, engine=engine)
    assert whole.fused == (kind in ("tc", "simt"))
    want = whole.phi_z(cu(X), cu(L)).cpu().numpy()
    assert np.isfinite(want).all()
    oprm = orc.Params(mu_1=MU1, lambda_ista=prm.lambda_ista, Nit=A_NIT, bb=bb, slidingDis=1, step=oracle_step_mode(step))
    ref, _ = orc.sparse_step(X, L, Y, D, oprm, dtype=np.float64)
    assert rel(want, ref) <= 1e-4
    nR = A_R - bb + 1
    for world in WORLDS:
        for r in range(world):
            st = solver.make_stripe(A_R, bb, r, world)
            cols = local_patch_columns(st, A_C)
            sc = solver.SparseCoder(cu(Y[st.row_slice]), Dd, prm, engine=engine)
            Xl, Ll = cu(X[st.row_slice]), cu(L[st.row_slice])
            got = {"static": sc.phi_z(Xl, Ll).cpu().numpy()}
            if kind == "tc":
                got["dynamic"] = sc._fused_range(Xl, Ll, 0, sc.P, dynamic=True).cpu().numpy()
            if not sc.fused:                   # the explicit engine's launch plan depends on the patch count: the same here
                assert ista_plan(bb * bb, K, sc.P) == ista_plan(bb * bb, K, whole.P), (world, r)
            for inst, phi in got.items():
                assert phi.shape == (bb * bb, len(cols))
                diff = np.flatnonzero((phi != want[:, cols]).any(axis=0))
                lanes = [(int(cols[p] % nR), int(cols[p] // nR), int(p % (st.b - st.a)) % 128, int(cols[p] % nR) % 128)
                         for p in diff[:8]]                             # (row start, column start, lane here, lane in the cube)
                assert diff.size == 0, (world, r, inst, diff.size, lanes)


IMOUT_ENGINES = {"tc": ("tc", "spectral", 256), "simt": ("simt", "frob4", 64), "explicit-K96": ("auto", "spectral_patch", 96)}


@pytest.mark.parametrize("kind", list(IMOUT_ENGINES))
@pytest.mark.usefixtures("lib")
@gpu_test
def test_stripe_overlap_sum_after_halo_reduce(kind):
    """SparseCoder.imout of every stripe (fused engines: the column-range pipe with at least 3 ranges, with and without the
    short dynamically dealt first range), reduced over the seams as StripeComm.halo_reduce does: bit-exact against the
    whole cube's IMout on every owned row off the seams; on the seam rows (first bb-1 owned rows of ranks > 0) within
    (k-1) 2^-24 sum|phi| of the fp64 overlap sum of the same Phi_z."""
    engine, step, K = IMOUT_ENGINES[kind]
    bb = 8
    Y, _, D = make_problem(A_R, A_C, K, seed=11, elementwise=step != "spectral")
    X, L, _ = state_near(Y, 12)
    prm = solver.Params(mu_1=MU1, mu_2=MU2, Nit=A_NIT, bb=bb, slidingDis=1, step=step)
    Dd = cu(D)
    whole = solver.SparseCoder(cu(Y), Dd, prm, engine=engine)
    want = whole.imout(cu(X), cu(L)).cpu().numpy()
    s64, a64, k = overlap_fp64(whole.phi_z(cu(X), cu(L)).cpu().numpy(), A_R, A_C, bb)
    bound = reassociation_bound(a64, k)
    assert k.max() == 64
    for world in WORLDS:
        stripes = [solver.make_stripe(A_R, bb, r, world) for r in range(world)]
        coders = []
        for st in stripes:
            sc = solver.SparseCoder(cu(Y[st.row_slice]), Dd, prm, engine=engine)
            if sc.fused:
                sc.CHUNK_BYTES = 4 * (st.b - st.a) * 64 * 4          # 4 column starts per range: 13 starts in 4 ranges
                assert sc._chunk_cols() == 4 and len(sc._ranges(False)) >= 3 and len(sc._ranges(True)) >= 3
            coders.append(sc)
        for shared_start in ((False, True) if whole.fused else (False,)):
            parts = [sc.imout(cu(X[st.row_slice]), cu(L[st.row_slice]), shared_start=shared_start).cpu().numpy()
                     for sc, st in zip(coders, stripes)]
            assert all(np.isfinite(p).all() for p in parts)
            emulate_halo_reduce(parts, stripes)
            for p, st in zip(parts, stripes):
                check_reduced_stripe(p, st, want, s64, bound)


@pytest.mark.parametrize("C", [29, 224])
@pytest.mark.usefixtures("lib")
@gpu_test
def test_low_rank_kernels_and_update_on_owned_rows(C):
    """The kernels the driver calls with rows = rows_owned, on stripes whose halo rows of X, lambda_2, IMout, U and
    lambda_1 hold NaN: the per-stripe Gram matrices summed equal Z^T Z of the whole cube to 1e-12 |Z|^T|Z|; svt_apply,
    axpy and admm_update (row_offset = a, R_total = R) are finite on the owned rows and equal the same rows of the
    whole-cube calls bit for bit; the recomposition also against fp64; no halo row of lambda_1, lambda_2 or X is
    written."""
    R, bb = A_R, 8
    rng = np.random.default_rng(C)
    f = lambda *s: rng.standard_normal(s).astype(F32)                               # noqa: E731
    Y, MtM, D = make_problem(R, C, 64, seed=C)
    Xw, L2w, IMw, Uw, L1w = f(R, C), f(R, C), f(R, C) * 8, f(R, C), f(R, C)
    prm = solver.Params(mu_1=MU1, mu_2=MU2, Nit=5, bb=bb, slidingDis=1, step="frob4")
    c, tau = 1.0 / MU2, 1.0 / MU2
    Z = (Xw + F32(c) * L2w).astype(F32)
    W = svt_weights_fp64(Z, 0.3 * float(np.linalg.norm(Z, 2))).astype(F32)   # keeps part of the spectrum
    Wd = cu(W)
    be = solver.CudaBackend(cu(Y), cu(MtM), cu(D), prm)
    U_whole = be.svt_apply(cu(Xw), cu(L2w), c, None, tau, R, W=Wd).cpu().numpy()
    A_whole = be.axpy(cu(Xw), cu(L2w), c, R).cpu().numpy()
    l1d, l2d = cu(L1w), cu(L2w)
    X_whole = be.admm_update(cu(IMw), cu(Uw), l1d, l2d, R, 0, R).cpu().numpy()
    l1_whole, l2_whole = l1d.cpu().numpy(), l2d.cpu().numpy()
    assert np.abs(A_whole - Z).max() <= 2 * F32_EPS * np.abs(Z).max()
    for world in WORLDS:
        G = torch.zeros((C, C), dtype=torch.float64, device="cuda")
        for r in range(world):
            st = solver.make_stripe(R, bb, r, world)
            sl, own, a = st.row_slice, st.rows_owned, st.a
            assert own < st.rows_local or r == world - 1

            def loc(A):
                t = A[sl].copy()
                t[own:] = np.nan
                return cu(t)

            bl = solver.CudaBackend(cu(Y[sl]), cu(MtM[sl]), cu(D), prm)
            Xl, L2l = loc(Xw), loc(L2w)
            G += bl.gram(Xl, L2l, c, own)
            U = bl.svt_apply(Xl, L2l, c, None, tau, own, W=Wd).cpu().numpy()
            assert U.shape == (own, C) and np.isfinite(U).all(), (world, r)
            assert np.array_equal(U, U_whole[a:a + own]), (world, r)
            _check_apply(U, Z[a:a + own], W)
            Ax = bl.axpy(Xl, L2l, c, own).cpu().numpy()
            assert np.isfinite(Ax).all() and np.array_equal(Ax, A_whole[a:a + own]), (world, r)
            l1l, l2l = loc(L1w), loc(L2w)
            Xout = torch.full((st.rows_local, C), float("nan"), device="cuda")
            bl.admm_update(loc(IMw), loc(Uw), l1l, l2l, own, a, R, out=Xout[:own])
            Xo, l1o, l2o = Xout.cpu().numpy(), l1l.cpu().numpy(), l2l.cpu().numpy()
            for name, got, want in (("X", Xo, X_whole), ("lambda_1", l1o, l1_whole), ("lambda_2", l2o, l2_whole)):
                assert np.isfinite(got[:own]).all(), (world, r, name)
                assert np.array_equal(got[:own], want[a:a + own]), (world, r, name)
                assert np.isnan(got[own:]).all(), (world, r, name)            # halo rows untouched
        _check_gram(G.cpu().numpy(), Z)


# ================================================================ B. the driver over W processes on one device
STEPS_CHECKED = (1, 3)
B_R, B_C, B_NIT = 150, 29, 15                  # 143 row starts: stripes of 71/72, 47/48, 35/36

# name -> what the case sets; every case runs tc / spectral table / K = 256 / C = 29 unless it says otherwise
CASES = {
    "tc-table-K256": dict(),
    "simt-frob4-K64": dict(engine="simt", step="frob4", K=64, elementwise=True),
    "tc-patch-K128": dict(step="spectral_patch", K=128, elementwise=True),
    "explicit-bb8-K96": dict(engine="auto", K=96),
    "explicit-bb6": dict(engine="auto", bb=6, K=72, step="frob4", elementwise=True),
    "narrowest-stripes": dict(narrow=True),
    "small-chunks": dict(chunk_cols=3),
    "hidden-eig-C224": dict(C=224, R=60, hide=True),
    "sequential-eig-C224": dict(C=224, R=60, hide=False),
    "from-host": dict(K=128, from_host=True),
    "low-rank-callable": dict(K=64, low_rank=True),
    "dead-stripe": dict(dead=True),
    "lambda2-halo-nan": dict(l2_halo_nan=True),
}


def case_spec(name):
    spec = dict(engine="tc", step="spectral", K=256, bb=8, C=B_C, R=B_R, elementwise=False)
    spec.update(CASES[name])
    return spec


def case_key(name, world):
    """The problem of a case depends on the world size only where the stripes shape it."""
    s = case_spec(name)
    return (name, world if s.get("narrow") or s.get("dead") else 0)


@functools.lru_cache(maxsize=None)
def case_problem(name, world):
    """(Y, MtM, D, Params, initial state or None) of a case: deterministic, the same in every process."""
    s = case_spec(name)
    bb, R, C = s["bb"], s["R"], s["C"]
    if s.get("narrow"):
        R = world * (bb - 1) + bb - 1            # R - bb + 1 = W (bb-1): every stripe exactly as wide as the halo
    dead = None
    if s.get("dead"):
        dead = np.zeros(R, bool)
        st1 = solver.make_stripe(R, bb, 1, world)
        dead[st1.row_slice] = True               # rank 1 holds no observed pixel at all
        a_last = solver.make_stripe(R, bb, world - 1, world).a
        dead[a_last - 6:a_last + 6] = True       # a run of missing rows across the last seam
    Y, MtM, D = make_problem(R, C, s["K"], bb=bb, seed=R + C + s["K"], elementwise=s["elementwise"], dead_rows=dead)
    prm = solver.Params(mu_1=MU1, mu_2=MU2, Nit=B_NIT, bb=bb, slidingDis=1, step=s["step"])
    state = state_near(Y, 5) if s.get("from_host") else None
    return Y, MtM, D, prm, state


def row_map(C):
    """The stand-in low-rank step of the low_rank case: a fixed per-row linear map U = Z A (fp32)."""
    rng = np.random.default_rng(C)
    return (np.eye(C) * 0.9 + 0.02 * rng.standard_normal((C, C))).astype(F32)


def _instrument(sol):
    """Record what a step produces: the overlap sum (halo_reduce later completes it in place), the all-reduced G, W."""
    rec = {"imout": [], "G": [], "W": []}

    def keep(lst, fn):
        def wrapped(*a, **k):
            out = fn(*a, **k)
            lst.append(out)
            return out
        return wrapped

    sol.be.imout = keep(rec["imout"], sol.be.imout)
    sol.comm.allreduce_sum = keep(rec["G"], sol.comm.allreduce_sum)
    sol.be.svt_weights = keep(rec["W"], sol.be.svt_weights)
    return rec


def _build(name, world, dev, stripe=None, group=None):
    """The solver of a case: one rank of a sharded run (``stripe``) or the unsharded run."""
    s = case_spec(name)
    Y, MtM, D, prm, state = case_problem(name, world)
    sl = stripe.row_slice if stripe is not None else slice(None)
    shapes = []
    low_rank = None
    if s.get("low_rank"):
        A = torch.from_numpy(row_map(Y.shape[1])).to(dev)

        def low_rank(Z):
            shapes.append(tuple(Z.shape))
            return Z @ A

    kw = dict(engine=s["engine"], low_rank=low_rank, device=dev)
    if stripe is not None:
        kw["stripe"] = stripe
    if s.get("from_host"):
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a[sl])).pin_memory()   # noqa: E731
        sol = solver.LRSPnP.from_host(pin(Y), pin(MtM), torch.from_numpy(D).to(dev), prm,
                                      state=tuple(pin(t) for t in state), **kw)
    else:
        sol = solver.LRSPnP(Y[sl].copy(), MtM[sl].copy(), D, prm, **kw)
    if stripe is not None:
        sol.comm = HostStagedComm(stripe, group)
    if "hide" in s:
        sol.hide_eigensolver = s["hide"]
    return sol, shapes


def _run_case(sol, stripe, l2_halo_nan=False, chunk_cols=None):
    """Three outer iterations; the state after the 1st and the 3rd, the step-1 overlap sum, G and W of every step."""
    own = sol.rows_owned
    if chunk_cols:
        n_rows = sol.Y.shape[0] - sol.prm.bb + 1                 # patch row-starts of this stripe
        sol.be.coder.CHUNK_BYTES = chunk_cols * n_rows * sol.be.coder.n * 4
        assert sol.be.coder._chunk_cols() == chunk_cols
    if l2_halo_nan:
        sol.lambda_2[own:] = float("nan")
    rec = _instrument(sol)
    out = {"hide": sol.hide_eigensolver, "rows_owned": own}
    if sol.be.coder.fused:
        out["n_ranges"] = len(sol.be.coder._ranges(shared_start=True))
    for t in range(1, STEPS_CHECKED[-1] + 1):
        sol.step()
        if t in STEPS_CHECKED:
            torch.cuda.synchronize()
            for k, v in (("X", sol.X), ("l1", sol.lambda_1), ("l2", sol.lambda_2)):
                a = v.cpu().numpy()
                out[f"{k}{t}"] = a[:own]
                if stripe is not None and k != "l2":
                    out[f"{k}{t}_halo"] = a[own:]
    sol.validate()
    out["imout1"] = rec["imout"][0].cpu().numpy()[:own]
    for k in ("G", "W"):
        if rec[k]:
            out[k] = np.stack([g.cpu().numpy() for g in rec[k]])
    return out


def _driver_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=timedelta(seconds=120))
    try:
        torch.set_num_threads(1)
        dev = torch.device("cuda", rank % torch.cuda.device_count())
        torch.cuda.set_device(dev)
        for name in CASES:
            s = case_spec(name)
            Y = case_problem(name, world)[0]
            st = solver.make_stripe(Y.shape[0], s["bb"], rank, world)
            sol, shapes = _build(name, world, dev, stripe=st)
            out = _run_case(sol, st, l2_halo_nan=s.get("l2_halo_nan", False), chunk_cols=s.get("chunk_cols"))
            out["low_rank_shapes"] = np.array(shapes, dtype=np.int64).reshape(-1, 2)
            np.savez(os.path.join(out_dir, f"{name}-rank{rank}.npz"), **out)
        # a diverged state: NaN in the owned lambda_2 rows of rank 1 reaches every rank through the all-reduced G
        st = solver.make_stripe(B_R, 8, rank, world)
        sol, _ = _build("tc-table-K256", world, dev, stripe=st)
        if rank == 1:
            sol.lambda_2[:st.rows_owned] = float("nan")
        sol.step()
        msg = ""
        try:
            sol.validate()
        except _lib.LrsError as e:
            msg = str(e)
        np.savez(os.path.join(out_dir, f"diverged-rank{rank}.npz"), msg=np.array(msg))
    finally:
        dist.destroy_process_group()


@functools.lru_cache(maxsize=None)
def unsharded_reference(key):
    name, world = key
    sol, shapes = _build(name, world, torch.device("cuda", 0))
    out = _run_case(sol, None, chunk_cols=None)
    out["low_rank_shapes"] = shapes
    return out


@functools.lru_cache(maxsize=None)
def oracle_reference(key):
    """The fp64 oracle (sparse step in fp64, the rest as the reference computes it) from the case's initial state."""
    name, world = key
    s = case_spec(name)
    Y, MtM, D, prm, state = case_problem(name, world)
    oprm = orc.Params(gamma=prm.gamma, mu_1=prm.mu_1, mu_2=prm.mu_2, lambda_ista=prm.lambda_ista, Nit=prm.Nit, bb=prm.bb,
                      slidingDis=1, step=oracle_step_mode(prm.step))
    X0, L10, L20 = state if state is not None else (Y.copy(), np.zeros_like(Y), np.zeros_like(Y))
    st = orc.State(X=X0.copy(), lambda_1=L10.copy(), lambda_2=L20.copy())
    a = orc.step_constants_batched(D.astype(np.float64), orc.patch_masks(orc.get_image_block(Y, prm.bb, 1)[0]), oprm.step)
    A = row_map(Y.shape[1]) if s.get("low_rank") else None
    low_rank = (lambda Z: (Z @ A).astype(F32)) if A is not None else None
    out = {}
    s32 = orc.State(X=X0.copy(), lambda_1=L10.copy(), lambda_2=L20.copy())
    for t in range(1, STEPS_CHECKED[-1] + 1):
        st = orc.outer_iteration(st, Y, MtM, D, oprm, a=a, low_rank=low_rank, dtype=np.float64)
        s32 = orc.outer_iteration(s32, Y, MtM, D, oprm, a=a.astype(F32), low_rank=low_rank, dtype=F32)
        out[t] = {"X": st.X, "l1": st.lambda_1, "l2": st.lambda_2}
        # what rounding alone changes on this cube: the same iteration with an fp32 sparse step
        out[t]["drift"] = {k: rel(v, out[t][k]) for k, v in (("X", s32.X), ("l1", s32.lambda_1), ("l2", s32.lambda_2))}
    return out


@pytest.fixture(scope="module", params=WORLDS, ids=[f"W{w}" for w in WORLDS])
def sharded(request, tmp_path_factory):
    """One spawn per world size: every case runs in the same W processes; the parent asserts them one by one."""
    world = request.param
    _lib.lib()                                   # built and loadable before the ranks start
    out = tmp_path_factory.mktemp(f"sharded-w{world}")
    mp.spawn(_driver_worker, args=(world, _free_port(), str(out)), nprocs=world, join=True)
    return world, out


@pytest.mark.parametrize("name", list(CASES))
@gpu_test
def test_sharded_driver_on_one_gpu(sharded, name):
    """One case of the sharded driver on W ranks sharing the device: X, lambda_1, lambda_2 on the owned rows after 1 and 3
    outer iterations against the unsharded GPU run (rel-L2 <= 2e-5, or twice the drift rounding alone causes on the
    cube) and the fp64 oracle (<= 1e-4, or the unsharded run's own distance plus that allowance); the step-1 overlap
    sum after the halo reduce bit-exact against the unsharded one on every owned row off the seams; the refreshed halo
    rows of X and lambda_1 equal the right neighbour's first owned rows; G and W identical on every rank; all finite."""
    world, out_dir = sharded
    s = case_spec(name)
    key = case_key(name, world)
    Y, MtM, D, prm, state = case_problem(name, world)
    R, C, bb = Y.shape[0], Y.shape[1], prm.bb
    stripes = [solver.make_stripe(R, bb, r, world) for r in range(world)]
    recs = [dict(np.load(out_dir / f"{name}-rank{r}.npz")) for r in range(world)]
    ref = unsharded_reference(key)
    orf = oracle_reference(key)
    # the case is what it claims to be
    if s.get("narrow"):
        assert all(st.b - st.a == bb - 1 for st in stripes)
    if s.get("dead"):
        assert not Y[stripes[1].row_slice].any()
    if "hide" in s:
        assert C > ops.JACOBI_AUTO_C and all(bool(z["hide"]) == s["hide"] for z in recs)
    if s.get("chunk_cols"):
        assert all(int(z["n_ranges"]) >= 3 for z in recs)
    if s.get("low_rank"):
        for z, st in zip(recs, stripes):
            assert [tuple(v) for v in z["low_rank_shapes"]] == [(st.rows_owned, C)] * STEPS_CHECKED[-1]
    for z, st in zip(recs, stripes):
        assert int(z["rows_owned"]) == st.rows_owned
    for t in STEPS_CHECKED:
        for k in ("X", "l1", "l2"):
            full = np.full((R, C), np.nan, F32)
            for z, st in zip(recs, stripes):
                full[st.a:st.a + st.rows_owned] = z[f"{k}{t}"]
            assert np.isfinite(full).all(), (t, k)
            # The ADMM iteration amplifies rounding: on the spectral-step cubes the fp32 oracle is 1e-7 from the fp64 one
            # after 1 step and 2-4e-5 after 3.  A sharded run sums G in another order, so it may differ from the unsharded
            # run by 2e-5 or twice that drift, and be no farther from fp64 than the unsharded run plus that much.
            tol = max(2e-5, 2.0 * orf[t]["drift"][k])
            d_ref, d_orc, d_unsh = rel(full, ref[f"{k}{t}"]), rel(full, orf[t][k]), rel(ref[f"{k}{t}"], orf[t][k])
            assert d_ref <= tol, (t, k, d_ref, tol)
            assert d_orc <= max(1e-4, d_unsh + tol), (t, k, d_orc, d_unsh, tol)
        for r in range(world - 1):
            h = stripes[r].halo
            for k in ("X", "l1"):
                halo = recs[r][f"{k}{t}_halo"]
                assert halo.shape == (h, C) and np.array_equal(halo, recs[r + 1][f"{k}{t}"][:h]), (t, k, r)
    for z, st in zip(recs, stripes):
        im = z["imout1"]
        assert np.isfinite(im).all()
        inner = np.setdiff1d(np.arange(st.rows_owned), seam_rows(st))
        assert np.array_equal(im[inner], ref["imout1"][st.a + inner]), st.rank
    for k in ("G", "W"):
        if s.get("low_rank"):
            assert all(k not in z for z in recs)
            continue
        assert recs[0][k].shape[0] == STEPS_CHECKED[-1] and np.isfinite(recs[0][k]).all(), k
        for z in recs[1:]:
            assert np.array_equal(z[k], recs[0][k]), k


@gpu_test
def test_sharded_driver_every_rank_reports_a_diverged_state(sharded):
    """NaN in the owned lambda_2 rows of one rank: after one step every rank's validate() raises 'diverged', because the
    all-reduced Gram matrix carries the NaN to every rank's eigensolver."""
    world, out_dir = sharded
    for r in range(world):
        msg = str(np.load(out_dir / f"diverged-rank{r}.npz")["msg"])
        assert "diverged" in msg, (r, msg)
