"""The batched path (LRSPnPBatch and the lrs_*_batch_* entry points) cube by cube against plain references: the fp32
oracle bit for bit for the geometry kernels and the X / multiplier update, fp64 restatements for the low-rank kernels,
and the fp64 oracle for whole runs, at the edges of the batch itself: stride-1 kernels with a cube index above 0, band
counts above JACOBI_AUTO_C (the library eigensolver), row counts that need a second recomposition launch per cube,
batches that mix empty, rank-1 and 2^+-20-scaled cubes, and B up to LRS_MAX_BATCH.

Every cube of every batch has its own seed and its own scale, so a kernel that read cube b - 1's data (or cube 0's)
would fail; the CPU self-check at the bottom shows that each per-cube comparator here rejects the neighbouring cube's
reference.  Run on the B200 box: pytest -m gpu tests/test_batch_edges.py.
"""
import ctypes
import functools
import zlib

import numpy as np
import pytest
import torch

from lrs_pnp_dip_b200 import _lib, ops, synth
from lrs_pnp_dip_b200.solver import LRSPnP, LRSPnPBatch, Params
from oracle import lrs_oracle as orc
from tests.test_kernel_edges import (F32_EPS, _check_apply, _check_gram, _check_weights, _gram_ref, per_patch_err, rel,
                                     shrink_weights, svt_fp64)

gpu = pytest.mark.gpu
C_OVER_MU2 = np.float32(1 / 0.9)


# ================================================================ helpers (CPU)
def cube_rng(*key):
    """The generator of one cube: seeded by the test's key and the cube index (strings through crc32: reproducible)."""
    return np.random.default_rng([zlib.crc32(k.encode()) if isinstance(k, str) else int(k) for k in key])


def cube_scale(b):
    """A different scale for every cube (powers of two and an odd factor, so no two cubes share one)."""
    return float(2.0 ** ((b % 7) - 3) * (1.0 + b / 64.0))


def check_cubes(check, got, refs):
    """check(got[b], refs[b]) for every cube b; a failure names its cube."""
    assert len(got) == len(refs)
    for b in range(len(refs)):
        try:
            check(got[b], refs[b])
        except AssertionError as e:
            raise AssertionError(f"cube {b}: {e}") from None


def same_bits(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape and np.array_equal(got, ref), int((got != ref).sum())


def close_rel(tol):
    def check(got, ref):
        r = rel(got, ref)
        assert r <= tol, r
    return check


def z32(X, L, c):
    """Z exactly as the kernels form it: fl32(X + fl32(c * L))."""
    return X if L is None else (X + np.float32(c) * L).astype(np.float32)


def b_form_weights(lam, tau):
    """Weights of the B form (column k of V = lambda_k v_k): shrink / lambda_k^2, 0 at or below 1e-12 lambda_max."""
    lam = np.asarray(lam, np.float64)
    cut = max(lam.max(), 0.0) * 1e-12
    return np.where(lam > cut, shrink_weights(lam, tau) / np.where(lam > cut, lam, 1.0) ** 2, 0.0)


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def stream():
    return torch.cuda.current_stream().cuda_stream


def L():
    return _lib.lib()


# ================================================================ A. geometry kernels against the oracle, bit for bit
# name -> (R, C, bb, s); the kernel branch each one reaches
GEOMS = {
    "s1-bb8": (40, 23, 8, 1),            # im2col_s1_kernel + col2im_s1_kernel
    "s1-bb6": (30, 37, 6, 1),            # im2col_s1_kernel + generic col2im_kernel
    "s1-bb36": (45, 40, 36, 1),          # im2col_s1_kernel (window 43 KB) + generic col2im_kernel
    "s1-bb41": (50, 43, 41, 1),          # window (256 + 40) x 42 floats > 48 KB: generic im2col_kernel
    "s1-bb8-C65543": (8, 65543, 8, 1),   # 65536 column starts > 65535: generic im2col_kernel; col2im_s1_kernel
    "s3-appended": (42, 31, 8, 3),       # appended last starts on both axes
    "s9-above-bb5": (50, 29, 5, 9),      # coverage gaps, appended last column start
    "s5-bb6": (33, 65, 6, 5),            # R, C neither multiples of 4 nor of 32
}


@functools.lru_cache(maxsize=8)               # the cases run geometry by geometry: B = 1, 2, 7 share their cubes
def _geom_cube(name, b):
    """Cube b of a geometry case and its oracle results: (inputs, im2col, im2col of X + L/mu, col2im, update)."""
    R, C, bb, s = GEOMS[name]
    rng = cube_rng("geom", name, b)
    sc = np.float32(cube_scale(b))
    f = lambda *shape: (sc * rng.standard_normal(shape)).astype(np.float32)       # noqa: E731
    X, Lm = f(R, C), f(R, C)
    P = len(orc.patch_index(R, C, bb, s)[0])
    blocks = f(bb * bb, P)
    Y = np.where(rng.random((R, C)) < 0.3, 0, f(R, C)).astype(np.float32)
    MtM = np.where(rng.random((R, C)) < 0.3, 0, rng.random((R, C))).astype(np.float32)
    IM, U, l1, l2 = f(R, C) * 8, f(R, C), f(R, C), f(R, C)
    mu = np.float32(0.15)
    V = (X + Lm / mu).astype(np.float32)
    oprm = orc.Params(gamma=0.5, mu_1=0.15, mu_2=0.9, bb=bb, slidingDis=s)
    upd = orc.admm_update(None, l1, l2, Y, MtM, IM, orc.coverage_weight(R, C, bb, s), U,
                          orc.lambda1_summation(l1, R, C, bb, s), oprm)
    inputs = dict(X=X, L=Lm, blocks=blocks, Y=Y, MtM=MtM, IM=IM, U=U, l1=l1, l2=l2)
    return inputs, orc.get_image_block(X, bb, s)[0], orc.get_image_block(V, bb, s)[0], \
        orc.col2im_accumulate(blocks, R, C, bb, s), upd


GEOM_CASES = [(g, B) for g in GEOMS for B in (1, 2, 7)]


@gpu
@pytest.mark.parametrize("name,B", GEOM_CASES, ids=[f"{g}-B{B}" for g, B in GEOM_CASES])
def test_geometry_kernels_batch_vs_oracle_bit_exact(name, B):
    """ops.im2col_batch without and with lambda_1/mu_1, ops.col2im_batch and lrs_admm_update_batch_f32 against
    orc.get_image_block, orc.col2im_accumulate and orc.admm_update (with orc.lambda1_summation) on each cube: all three are
    sequential fp32 in the reference's order, so every cube must match bit for bit."""
    R, C, bb, s = GEOMS[name]
    cubes = [_geom_cube(name, b) for b in range(B)]
    P = ops.patch_count(R, C, bb, s)
    stack = lambda key: cu(np.stack([c[0][key] for c in cubes]))                  # noqa: E731
    X, Lm = stack("X"), stack("L")
    got = ops.im2col_batch(X, bb, s).cpu().numpy()
    check_cubes(same_bits, [got[:, b * P:(b + 1) * P] for b in range(B)], [c[1] for c in cubes])
    got = ops.im2col_batch(X, bb, s, Lm, 0.15).cpu().numpy()
    check_cubes(same_bits, [got[:, b * P:(b + 1) * P] for b in range(B)], [c[2] for c in cubes])
    blocks = cu(np.concatenate([c[0]["blocks"] for c in cubes], axis=1))
    check_cubes(same_bits, ops.col2im_batch(blocks, B, R, C, bb, s).cpu().numpy(), [c[3] for c in cubes])
    Y, M, IM, U, l1, l2 = (stack(k) for k in ("Y", "MtM", "IM", "U", "l1", "l2"))
    Xo = torch.full_like(X, float("nan"))
    _lib.check(L().lrs_admm_update_batch_f32(Y.data_ptr(), M.data_ptr(), IM.data_ptr(), U.data_ptr(), l1.data_ptr(),
                                             l2.data_ptr(), Xo.data_ptr(), 0.5, 0.15, 0.9, B, R, C, bb, s, stream()))
    for k, t in enumerate((Xo, l1, l2)):
        check_cubes(same_bits, t.cpu().numpy(), [c[4][k] for c in cubes])


# ================================================================ B. low-rank kernels against fp64
# (R, C, B): the Gram kernel's row chunking is sms*4 / (pairs*B), so the same R, C run different chunks at different B
GRAM_CASES = [(1, 1, 600), (1, 256, 5), (17, 65, 150), (17, 256, 600), (17, 191, 2), (4099, 65, 5), (4099, 224, 2),
              (4099, 1, 600), (65536, 191, 2), (65536, 256, 1)] + [(65536, 1, B) for B in (1, 2, 5, 150, 600)]


def _xl_cubes(key, B, R, C):
    X = np.empty((B, R, C), np.float32)
    Lm = np.empty((B, R, C), np.float32)
    for b in range(B):
        rng = cube_rng(key, R, C, b)
        sc = np.float32(cube_scale(b))
        X[b] = sc * rng.standard_normal((R, C), dtype=np.float32)
        Lm[b] = sc * rng.standard_normal((R, C), dtype=np.float32)
    return X, Lm


@gpu
@pytest.mark.parametrize("R,C,B", GRAM_CASES)
def test_gram_batch_vs_fp64(R, C, B):
    """lrs_gram_batch_f64 with the lambda term against Z_b^T Z_b in fp64 for every cube (1e-12 of |Z|^T |Z|
    elementwise); a second call into the same G doubles every cube's matrix."""
    X, Lm = _xl_cubes("gram", B, R, C)
    Xd, Ld = cu(X), cu(Lm)
    G = torch.zeros((B, C, C), dtype=torch.float64, device="cuda")
    _lib.check(L().lrs_gram_batch_f64(Xd.data_ptr(), Ld.data_ptr(), float(C_OVER_MU2), B, R, C, G.data_ptr(), stream()))
    G1 = G.cpu().numpy()
    _lib.check(L().lrs_gram_batch_f64(Xd.data_ptr(), Ld.data_ptr(), float(C_OVER_MU2), B, R, C, G.data_ptr(), stream()))
    G2 = G.cpu().numpy()
    Z = [z32(X[b], Lm[b], C_OVER_MU2) for b in range(B)]
    check_cubes(_check_gram, G1, Z)
    check_cubes(lambda g, z: _check_gram(g, z, mult=2.0), G2, Z)


def _eig_problems(C, rng):
    """The problems of test_sym_eig_jacobi_vs_lapack plus the zero matrix and matrices scaled by 2^+-40."""
    Z = rng.standard_normal((max(4 * C, 64), C)) * np.logspace(0, -5, C)[None, :]
    yield "decaying", Z.T @ Z
    r = max(1, C // 4)
    Zr = rng.standard_normal((300, r)) @ rng.standard_normal((r, C))
    rank_def = Zr.T @ Zr
    yield "rank-deficient", rank_def
    yield "identity", np.eye(C)
    yield "diagonal", np.diag(np.arange(1, C + 1, dtype=np.float64) ** 2)
    Q, _ = np.linalg.qr(rng.standard_normal((C, C)))
    lam = np.repeat(np.array([100.0, 1.5, 1.5 - 1e-9, 1e-3]), -(-C // 4))[:C]       # clustered eigenvalues
    clustered = (Q * lam[None, :]) @ Q.T
    yield "clustered", clustered
    yield "zero", np.zeros((C, C))
    yield "clustered-2^40", clustered * 2.0 ** 40
    yield "rank-deficient-2^-40", rank_def * 2.0 ** -40


@gpu
@pytest.mark.parametrize("C", [2, 31, 128, 192, 256])
def test_jacobi_batch_of_different_problems(C):
    """ops.sym_eig_jacobi_batch on one batch of different problems (decaying, rank-deficient, identity, diagonal,
    clustered, zero, scaled by 2^40 and 2^-40): each cube within the bounds of test_sym_eig_jacobi_vs_lapack, and each
    cube's status word (sweep count included) and results equal to its single-problem solve."""
    rng = np.random.default_rng(C + 1000)
    names, Gs = zip(*[(n, 0.5 * (G + G.T)) for n, G in _eig_problems(C, rng)])
    Gd = cu(np.stack(Gs))
    lam, Bt, st = ops.sym_eig_jacobi_batch(Gd)
    lam, Bt, st = lam.cpu().numpy(), Bt.cpu().numpy(), st.cpu().numpy()
    for b, (name, G) in enumerate(zip(names, Gs)):
        l1, B1, s1 = ops.sym_eig_jacobi(Gd[b])
        assert np.array_equal(st[b], s1.cpu().numpy()), (name, st[b], s1.cpu().numpy())
        assert np.array_equal(lam[b], l1.cpu().numpy()) and np.array_equal(Bt[b], B1.cpu().numpy()), name
        assert st[b, 1] == 0 and st[b, 2] == 0 and st[b, 0] < 30, (name, st[b])
        ref = np.linalg.eigvalsh(G)
        scale = max(ref.max(), 1e-300)
        assert np.abs(np.sort(lam[b]) - np.clip(ref, 0, None)).max() <= 1e-10 * scale, name
        assert np.abs(Bt[b] @ Bt[b].T - np.diag(lam[b] ** 2)).max() <= 3e-8 * scale ** 2, name
        assert np.abs(Bt[b] @ G - lam[b][:, None] * Bt[b]).max() <= 3e-8 * scale ** 2, name
    assert len(set(st[:, 0].tolist())) > 1, st[:, 0]          # the clusters stopped after different sweep counts
    assert not lam[names.index("zero")].any() and not Bt[names.index("zero")].any()


WEIGHT_CS = [96, 128, 135, 191, 192, 193, 224, 256]


def _edge_spectrum(C, tau, rng, scale):
    """Eigenvalues with sigma == tau exactly, tau (1 +- 1e-12), a tiny negative value and 0 up front, the rest spread
    over four decades of ``scale``."""
    lam = scale * 10 ** rng.uniform(-2, 2, C)
    t2 = tau * tau
    edges = np.array([t2, (tau * (1 + 1e-12)) ** 2, (tau * (1 - 1e-12)) ** 2, -1e-14, 0.0])
    lam[:5] = edges
    return rng.permutation(lam)


def _weights_batch(lam, V, strides, C, n, tau, b_form):
    B = lam.shape[0]
    lam_d, V_d = cu(np.asarray(lam, np.float64)), cu(np.asarray(V, np.float64))
    W = torch.full((B, C, C), float("nan"), dtype=torch.float32, device="cuda")
    _lib.check(L().lrs_svt_weights_batch_f64(lam_d.data_ptr(), V_d.data_ptr(), *strides, B, C, n, float(tau), int(b_form),
                                             W.data_ptr(), stream()), "lrs_svt_weights_batch_f64")
    return W.cpu().numpy()


@gpu
@pytest.mark.parametrize("C", WEIGHT_CS)
def test_svt_weights_batch_kernel_edges(C):
    """lrs_svt_weights_batch_f64 on given eigenpairs, three cubes with their own V and spectrum: plain form with V read
    row-major and through the strides (C*C, 1, C) of a batched eigh, at sigma == tau, tau (1 +- 1e-12) and tau = 0; B form
    with lambda_max differing by 1e20 between cubes, each cube's directions at and below its OWN 1e-12 lambda_max cut."""
    B = 3
    rng = np.random.default_rng(C + 77)
    Q = np.stack([np.linalg.qr(rng.standard_normal((C, C)))[0] for _ in range(B)])
    for tau in (0.0, 2.0):
        lam = np.stack([_edge_spectrum(C, tau, rng, cube_scale(b) * max(tau * tau, 1.0)) for b in range(B)])
        w = [shrink_weights(lam[b], tau) for b in range(B)]
        check = lambda W, ref: _check_weights(W, *ref)                               # noqa: E731
        refs = [(Q[b], w[b]) for b in range(B)]
        check_cubes(check, _weights_batch(lam, Q, (C * C, C, 1), C, C, tau, 0), refs)            # V[b,i,k] at b*C*C + i*C + k
        check_cubes(check, _weights_batch(lam, np.swapaxes(Q, 1, 2), (C * C, 1, C), C, C, tau, 0), refs)   # ... + k*C + i
    # B form: row k of Bt_b = lambda_k v_k, read with strides (C*C, 1, C); lambda_max = 1, 1e20, 1e-10
    lam = np.empty((B, C))
    for b, top in enumerate((1.0, 1e20, 1e-10)):
        l = top * 10 ** rng.uniform(-3, 0, C)
        l[0] = top
        l[1:6] = top * np.array([1e-12, 0.5e-12, 2e-12, -1e-14, 0.0])       # at the cut, below, above, negative, zero
        lam[b] = rng.permutation(l)
    Bt = lam[:, :, None] * np.swapaxes(Q, 1, 2)
    for tau in (0.0, 0.5):
        refs = [(Bt[b].T, b_form_weights(lam[b], tau)) for b in range(B)]
        check_cubes(lambda W, ref: _check_weights(W, *ref), _weights_batch(lam, Bt, (C * C, 1, C), C, C, tau, 1), refs)


def _psd_cubes(C, B, seed):
    """Gram matrices of B cubes, each with its own scale and a decaying spectrum (every one full rank)."""
    Gs = []
    for b in range(B):
        rng = cube_rng("psd", C, seed, b)
        Z = rng.standard_normal((3 * C, C)) * np.logspace(0, -2, C)[None, :] * cube_scale(b)
        Gs.append(Z.T @ Z)
    return np.stack(Gs)


@gpu
@pytest.mark.parametrize("C", WEIGHT_CS)
def test_svt_weights_batch_both_solvers_vs_fp64(C):
    """ops.svt_weights_batch with the Jacobi solver (B form) and the library solver (batched eigh, V read through the
    strides (C*C, 1, C), no zero border) against V diag(w) V^T in fp64 on the eigenpairs each solver produced; the
    library batch also against the single-cube library path (zero-bordered for C in [96, 136)) and the fp64 SVT weights."""
    B = 3
    Gs = _psd_cubes(C, B, 1)
    Gd = cu(Gs)
    lam_top = np.linalg.eigvalsh(Gs)
    tau = float(np.sqrt(np.median(lam_top[0])))                     # mid-spectrum of cube 0, elsewhere in the others
    lam, Bt, _ = ops.sym_eig_jacobi_batch(Gd)
    Wj = ops.svt_weights_batch(Gd, tau, solver="jacobi").cpu().numpy()
    lam, Bt = lam.cpu().numpy(), Bt.cpu().numpy()
    check_cubes(lambda W, ref: _check_weights(W, *ref), Wj, [(Bt[b].T, b_form_weights(lam[b], tau)) for b in range(B)])
    evals, V = torch.linalg.eigh(Gd)
    assert V.stride() == (C * C, 1, C)
    Wl = ops.svt_weights_batch(Gd, tau, solver="library").cpu().numpy()
    evals, V = evals.cpu().numpy(), V.cpu().numpy()
    check_cubes(lambda W, ref: _check_weights(W, *ref), Wl, [(V[b], shrink_weights(evals[b], tau)) for b in range(B)])
    for b in range(B):
        lam64, V64 = np.linalg.eigh(Gs[b])
        ref = (V64 * shrink_weights(lam64, tau)) @ V64.T
        one = ops.svt_weights(Gd[b], tau, solver="library").cpu().numpy()
        for W in (Wj[b], Wl[b], one):
            assert np.abs(W - ref).max() <= 3e-6 * max(np.abs(ref).max(), 1.0), b
        assert np.abs(Wl[b] - one).max() <= 3e-6 * max(np.abs(one).max(), 1.0), b


@gpu
@pytest.mark.parametrize("C", [128, 224])
def test_svt_weights_batch_library_names_the_non_finite_cube(C):
    """A NaN in one cube's Gram matrix: the library path raises naming exactly that cube."""
    Gd = cu(_psd_cubes(C, 4, 2))
    Gd[2, 5, 9] = float("nan")
    Gd[2, 9, 5] = float("nan")
    with pytest.raises(_lib.LrsError, match=r"cube\(s\) \[2\]:"):
        ops.svt_weights_batch(Gd, 0.5, solver="library")


def _apply_batch(Xd, Ld, c, Wd):
    B, R, C = Xd.shape
    U = torch.full_like(Xd, float("nan"))
    _lib.check(L().lrs_svt_apply_batch_f32(Xd.data_ptr(), _lib.ptr(Ld), float(c), Wd.data_ptr(), B, R, C, U.data_ptr(),
                                           stream()), "lrs_svt_apply_batch_f32")
    return U.cpu().numpy()


@gpu
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("R,C", [(1, 17), (65, 17), (300, 256), (64, 224), (4099, 191)])
def test_svt_apply_batch_vs_fp64(R, C, B):
    """lrs_svt_apply_batch_f32: U_b = (X_b + c L_b) W_b with a non-symmetric W per cube, L absent and present,
    within 2 C 2^-24 (|Z| |W|) elementwise of fp64 for every cube."""
    X, Lm = _xl_cubes("apply", B, R, C)
    W = np.stack([(cube_rng("W", C, b).standard_normal((C, C)) / np.sqrt(C) * cube_scale(b + 3)).astype(np.float32)
                  for b in range(B)])
    Xd, Ld, Wd = cu(X), cu(Lm), cu(W)
    check_cubes(lambda U, zw: _check_apply(U, *zw), _apply_batch(Xd, None, 0.0, Wd), [(X[b], W[b]) for b in range(B)])
    check_cubes(lambda U, zw: _check_apply(U, *zw), _apply_batch(Xd, Ld, C_OVER_MU2, Wd),
                [(z32(X[b], Lm[b], C_OVER_MU2), W[b]) for b in range(B)])


@gpu
def test_svt_apply_batch_second_launch():
    """B = 2 cubes of 65535*64 + 77 rows: each cube needs the second launch, whose row offset is combined with the cube
    stride R*C."""
    B, R, C = 2, 65535 * 64 + 77, 3
    X, Lm = _xl_cubes("apply2", B, R, C)
    W = np.stack([cube_rng("W2", b).standard_normal((C, C)).astype(np.float32) for b in range(B)])
    U = _apply_batch(cu(X), cu(Lm), C_OVER_MU2, cu(W))
    check_cubes(lambda u, zw: _check_apply(u, *zw, chunk=1 << 20), U, [(z32(X[b], Lm[b], C_OVER_MU2), W[b]) for b in range(B)])


def _low_rank_cubes(R, C):
    """X, lambda_2 of five cubes: rank-8 plus noise; zero; rank-1; rank-8 plus noise x 2^20; x 2^-20."""
    X = np.zeros((5, R, C), np.float32)
    L2 = np.zeros((5, R, C), np.float32)
    for b, kind in enumerate(("noisy", "zero", "rank1", "noisy", "noisy")):
        rng = cube_rng("lowrank", R, C, b)
        if kind == "noisy":
            X[b] = rng.standard_normal((R, 8), dtype=np.float32) @ rng.standard_normal((8, C), dtype=np.float32)
            X[b] += np.float32(0.05) * rng.standard_normal((R, C), dtype=np.float32)
            L2[b] = np.float32(0.05) * rng.standard_normal((R, C), dtype=np.float32)
        elif kind == "rank1":
            X[b] = 3.0 * np.outer(rng.standard_normal(R), rng.standard_normal(C)).astype(np.float32)
    X[3] *= np.float32(2.0 ** 20)
    L2[3] *= np.float32(2.0 ** 20)
    X[4] *= np.float32(2.0 ** -20)
    L2[4] *= np.float32(2.0 ** -20)
    return X, L2


@gpu
@pytest.mark.parametrize("C", [191, 192, 193, 224, 256])
def test_batch_low_rank_step_vs_fp64(C, monkeypatch):
    """LRSPnPBatch._low_rank() (batched Gram -> eigensolver -> weights -> recomposition) on a prepared state of five
    different cubes, on both eigensolvers at every C, against svt_fp64(X_b + lambda2_b/mu_2, 1/mu_2) per cube: rel-L2
    <= 1e-5, no row off by more than 1e-4 of its norm, and exactly 0 where the fp64 result is 0."""
    R = 400
    X, L2 = _low_rank_cubes(R, C)
    prm = Params(bb=4, slidingDis=4, step="frob4", Nit=1)
    sol = LRSPnPBatch(X, np.ones_like(X), np.random.default_rng(0).standard_normal((16, 20)).astype(np.float32), prm)
    sol.X.copy_(cu(X))
    sol.lambda_2.copy_(cu(L2))
    tau = 1.0 / prm.mu_2
    refs = [svt_fp64(z32(X[b], L2[b], C_OVER_MU2), tau) for b in range(5)]
    assert not refs[1].any() and not refs[4].any() and all(r.any() for r in (refs[0], refs[2], refs[3]))

    def check(U, ref):
        if not ref.any():
            assert not U.any(), float(np.abs(U).max())
            return
        assert rel(U, ref) <= 1e-5, rel(U, ref)
        assert per_patch_err(U.T, ref.T).max() <= 1e-4, float(per_patch_err(U.T, ref.T).max())

    for auto_c in (ops.JACOBI_MAX_C, 0):                 # the cluster Jacobi kernel, the library eigh
        monkeypatch.setattr(ops, "JACOBI_AUTO_C", auto_c)
        check_cubes(check, sol._low_rank().cpu().numpy(), refs)
        sol.validate()


# ================================================================ C. the whole solver against the fp64 oracle
def _stride1_cubes():
    """Six 60 x 24 cubes: row masks (two of them scaled x1e3 and x1e-3), a per-element mask, fully observed,
    all missing."""
    H, W, R, C = 6, 10, 60, 24
    Y = np.zeros((6, R, C), np.float32)
    M = np.zeros((6, R, C), np.float32)
    for b, kind in enumerate(("rows", "rows", "element", "full", "missing", "rows")):
        _, noisy = synth.synthetic_cube(H, W, C, rank=4, seed=300 + b)
        rng = cube_rng("s1", b)
        if kind == "rows":
            m = np.repeat((rng.random(R) < 0.6)[:, None], C, axis=1)
        elif kind == "element":
            m = rng.random((R, C)) < 0.7
        else:
            m = np.full((R, C), kind == "full")
        Y[b] = np.where(m, noisy, 0)
        M[b] = m
    Y[1] *= np.float32(1e3)
    Y[5] *= np.float32(1e-3)
    return Y, M


def _vs_oracle(sol, Y, M, D, oprm, cubes, tol=1e-4):
    for b in cubes:
        ref = orc.run(Y[b], M[b], D, oprm, 2, dtype=np.float64)
        for name in ("X", "lambda_1", "lambda_2"):
            got = getattr(sol, name)[b].cpu().numpy()
            r = rel(got, getattr(ref, name))
            assert r <= tol, (b, name, r)


@gpu
def test_batch_stride1_explicit_vs_oracle():
    """bb = 8, s = 1, K = 96 (explicit engine), six different cubes against orc.run in fp64, cube by cube; the all-missing
    cube comes back exactly 0 with finite multipliers."""
    Y, M = _stride1_cubes()
    D = synth.synthetic_dictionary(64, 96, seed=96)
    sol = LRSPnPBatch(Y, M, D, Params(Nit=20, bb=8, slidingDis=1)).run(2)
    assert not sol.X[4].any() and bool(torch.isfinite(sol.lambda_1[4]).all()) and bool(torch.isfinite(sol.lambda_2[4]).all())
    _vs_oracle(sol, Y, M, D, orc.Params(Nit=20, bb=8, slidingDis=1), range(6))


@gpu
def test_batch_stride1_nlm_patches_vs_pnp_ista_nlm():
    """The same batch with the plug-and-play NLM denoiser: after two outer iterations, the sparse step of patches of two
    different cubes against orc.pnp_ista_nlm (one patch vector at a time, the solver's own step constant)."""
    Y, M = _stride1_cubes()
    D = synth.synthetic_dictionary(64, 96, seed=96)
    prm = Params(Nit=20, bb=8, slidingDis=1, denoiser="nlm")
    sol = LRSPnPBatch(Y, M, D, prm).run(2)
    assert bool(torch.isfinite(sol.X).all())
    phi = sol.coder.phi_z(sol.X, sol.lambda_1).cpu().numpy()
    a = sol.coder.a_patch.cpu().numpy()
    P = sol.coder.P
    for b in (1, 2):
        V = (sol.X[b].cpu().numpy() + sol.lambda_1[b].cpu().numpy() / np.float32(prm.mu_1)).astype(np.float32)
        blocks = orc.get_image_block(V, 8, 1)[0]
        mask = orc.patch_masks(orc.get_image_block(Y[b], 8, 1)[0])
        live = np.flatnonzero(mask.any(axis=0))
        for p in cube_rng("nlm", b).choice(live, 4, replace=False):
            m = mask[:, p]
            x = orc.pnp_ista_nlm(blocks[m, p], D[m], prm.lambda_ista, prm.Nit, float(a[b * P + p]), h_scale=prm.nlm_h_scale)
            assert rel(phi[:, b * P + p], (D.astype(np.float64) @ x).ravel()) < 2e-4, (b, p)


@gpu
def test_batch_above_192_bands_vs_oracle():
    """bb = 6, s = 3 with appended starts, C = 224 > JACOBI_AUTO_C: the library eigensolver and the lr_async = False
    ordering of LRSPnPBatch._step, three cubes against orc.run in fp64."""
    R, C, B = 50, 224, 3
    Y = np.zeros((B, R, C), np.float32)
    M = np.zeros((B, R, C), np.float32)
    for b in range(B):
        _, noisy = synth.synthetic_cube(5, 10, C, rank=4, seed=400 + b)
        m = np.repeat((cube_rng("b224", b).random(R) < 0.7)[:, None], C, axis=1)
        Y[b] = np.where(m, noisy * np.float32(cube_scale(b)), 0)
        M[b] = m
    D = synth.synthetic_dictionary(36, 48, seed=48)
    prm = Params(Nit=20, bb=6, slidingDis=3)
    sol = LRSPnPBatch(Y, M, D, prm)
    assert C > ops.JACOBI_AUTO_C
    sol.step()
    assert not sol._pending                                 # the library path hands no Jacobi status words on
    sol.run(1)
    _vs_oracle(sol, Y, M, D, orc.Params(Nit=20, bb=6, slidingDis=3), range(B))


def _cfg1_cubes(B, masks=4):
    """B cfg 1 cubes (1296 x 128): rank-4 plus noise, each with its own seed and scale (cube 1 x 2^-20, the last x 2^20),
    row masks from a pool of ``masks`` (so the spectral step constants cost a few hundred eigensolves)."""
    R, C = 1296, 128
    pool = [np.random.default_rng(900 + k).random(R) < 0.7 for k in range(masks)]
    Y = np.zeros((B, R, C), np.float32)
    M = np.zeros((B, R, C), np.float32)
    for b in range(B):
        rng = cube_rng("cfg1", b)
        Z = rng.standard_normal((R, 4), dtype=np.float32) @ rng.standard_normal((4, C), dtype=np.float32)
        Z += np.float32(0.1) * rng.standard_normal((R, C), dtype=np.float32)
        sc = cube_scale(b) * (2.0 ** -20 if b == 1 else 2.0 ** 20 if b == B - 1 else 1.0)
        m = np.repeat(pool[b % masks][:, None], C, axis=1)
        Y[b] = np.where(m, Z * np.float32(sc), 0)
        M[b] = m
    return Y, M


@gpu
def test_large_explicit_tc_batch_vs_separate_solvers_and_oracle():
    """cfg 1 geometry, K = 324, Nit = 12, B = 64 (9216 ISTA columns on the tcgen05 engine): every cube against its own
    LRSPnP (a_patch bit for bit, the state within 1e-5), the first and the last cube against orc.run in fp64."""
    B = 64
    Y, M = _cfg1_cubes(B)
    D = synth.synthetic_dictionary(1296, 324, seed=0)
    Dd = cu(D)                                                # one device dictionary: its step-constant memo is shared
    prm = Params(Nit=12)
    sol = LRSPnPBatch(Y, M, Dd, prm).run(2)
    P = sol.coder.P
    assert B * P == 9216
    for b in range(B):
        one = LRSPnP(Y[b], M[b], Dd, prm)
        assert torch.equal(sol.coder.a_patch[b * P:(b + 1) * P], one.be.coder.a_patch), b
        one.run(2)
        for name in ("X", "lambda_1", "lambda_2"):
            r = rel(getattr(sol, name)[b].cpu().numpy(), getattr(one, name).cpu().numpy())
            assert r <= 1e-5, (b, name, r)
    _vs_oracle(sol, Y, M, D, orc.Params(Nit=12), (0, B - 1))


# ================================================================ D. the largest batches
@gpu
def test_max_batch_tiny_cubes_every_kernel():
    """B = LRS_MAX_BATCH = 65535 cubes of 3 x 3 (bb = 2, s = 1): im2col, col2im, the update, Gram, Jacobi, weights and
    recomposition once each, against vectorised references over all cubes."""
    B, R, C, bb, s = _lib.MAX_BATCH, 3, 3, 2, 1
    rng = np.random.default_rng(65535)
    sc = (2.0 ** rng.integers(-8, 9, B) * (1 + rng.random(B))).astype(np.float32)[:, None, None]    # a scale per cube
    f = lambda: (sc * rng.standard_normal((B, R, C))).astype(np.float32)                             # noqa: E731
    X, Lm, IM, U, l1, l2, Y = f(), f(), f(), f(), f(), f(), f()
    MtM = (rng.random((B, R, C)) < 0.7).astype(np.float32)
    xs, ys = orc.patch_index(R, C, bb, s)
    P, n = len(xs), bb * bb
    k = np.arange(n)
    # im2col: blocks[k, b*P + p] = V_b[x_p + k % bb, y_p + k // bb]
    V = (X + Lm / np.float32(0.15)).astype(np.float32)
    want = V[:, xs[None, :] + (k % bb)[:, None], ys[None, :] + (k // bb)[:, None]]          # [B, n, P]
    got = ops.im2col_batch(cu(X), bb, s, cu(Lm), 0.15).cpu().numpy()
    assert np.array_equal(got, want.transpose(1, 0, 2).reshape(n, B * P))
    # col2im: every element sums its covering patches in ascending patch order, in fp32
    blocks = (sc.reshape(1, B, 1) * rng.standard_normal((n, B, P))).astype(np.float32)
    want = np.zeros((B, R, C), np.float32)
    for p in range(P):
        for kk in range(n):
            want[:, xs[p] + kk % bb, ys[p] + kk // bb] += blocks[kk, :, p]
    assert np.array_equal(ops.col2im_batch(cu(blocks.reshape(n, B * P)), B, R, C, bb, s).cpu().numpy(), want)
    # X / multiplier update (the oracle's elementwise formulas broadcast over the cubes)
    oprm = orc.Params(gamma=0.5, mu_1=0.15, mu_2=0.9, bb=bb, slidingDis=s)
    Xr, l1r, l2r = orc.admm_update(None, l1, l2, Y, MtM, IM, orc.coverage_weight(R, C, bb, s), U,
                                   orc.lambda1_summation(l1, R, C, bb, s), oprm)
    Yd, Md, IMd, Ud, l1d, l2d = (cu(a) for a in (Y, MtM, IM, U, l1, l2))
    Xo = torch.empty_like(Yd)
    _lib.check(L().lrs_admm_update_batch_f32(Yd.data_ptr(), Md.data_ptr(), IMd.data_ptr(), Ud.data_ptr(), l1d.data_ptr(),
                                             l2d.data_ptr(), Xo.data_ptr(), 0.5, 0.15, 0.9, B, R, C, bb, s, stream()))
    assert np.array_equal(Xo.cpu().numpy(), Xr)
    assert np.array_equal(l1d.cpu().numpy(), l1r) and np.array_equal(l2d.cpu().numpy(), l2r)
    # Gram
    Xd, Ld = cu(X), cu(Lm)
    G = torch.zeros((B, C, C), dtype=torch.float64, device="cuda")
    _lib.check(L().lrs_gram_batch_f64(Xd.data_ptr(), Ld.data_ptr(), float(C_OVER_MU2), B, R, C, G.data_ptr(), stream()))
    Z = z32(X, Lm, C_OVER_MU2).astype(np.float64)
    Gr = np.einsum("bri,brj->bij", Z, Z)
    bound = np.einsum("bri,brj->bij", np.abs(Z), np.abs(Z))
    assert np.all(np.abs(G.cpu().numpy() - Gr) <= 1e-12 * bound)
    # Jacobi (C = 3)
    lam, Bt, st = ops.sym_eig_jacobi_batch(G)
    lam, Bt, st = lam.cpu().numpy(), Bt.cpu().numpy(), st.cpu().numpy()
    assert not st[:, 1:].any() and st[:, 0].max() < 30
    ref = np.linalg.eigvalsh(Gr)
    scale = ref.max(axis=1, keepdims=True)
    assert np.all(np.abs(np.sort(lam, axis=1) - np.clip(ref, 0, None)) <= 1e-10 * scale)
    assert np.all(np.abs(np.einsum("bki,bli->bkl", Bt, Bt) - lam[:, :, None] ** 2 * np.eye(C)) <= 3e-8 * scale[:, :, None] ** 2)
    # weights (B form) and recomposition
    tau = float(C_OVER_MU2)
    Wd = torch.empty((B, C, C), dtype=torch.float32, device="cuda")
    lam_d, Bt_d = cu(lam), cu(Bt)
    _lib.check(L().lrs_svt_weights_batch_f64(lam_d.data_ptr(), Bt_d.data_ptr(), C * C, 1, C, B, C, C, tau, 1, Wd.data_ptr(),
                                             stream()))
    cut = np.maximum(lam.max(axis=1, keepdims=True), 0) * 1e-12
    w = np.where(lam > cut, shrink_weights(lam, tau) / np.where(lam > cut, lam, 1.0) ** 2, 0.0)
    Wr = np.einsum("bki,bk,bkj->bij", Bt, w, Bt)
    Wb = np.einsum("bki,bk,bkj->bij", np.abs(Bt), np.abs(w), np.abs(Bt))
    W = Wd.cpu().numpy()
    assert np.all(np.abs(W - Wr) <= 2 * F32_EPS * np.abs(Wr) + 1e-13 * Wb)
    U = _apply_batch(Xd, Ld, C_OVER_MU2, Wd)
    Z32 = z32(X, Lm, C_OVER_MU2).astype(np.float64)
    W64 = W.astype(np.float64)
    Ur = np.einsum("bri,bij->brj", Z32, W64)
    assert np.all(np.abs(U - Ur) <= 2 * C * F32_EPS * np.einsum("bri,bij->brj", np.abs(Z32), np.abs(W64)))


@gpu
def test_batch_of_2048_small_cubes():
    """LRSPnPBatch with B = 2048 cubes of 20 x 12 (bb = 4, s = 2): everything finite, a seeded sample of 8 cubes against
    separate LRSPnP solvers (1e-5) and orc.run in fp64 (1e-4)."""
    B, R, C = 2048, 20, 12
    pool = [np.random.default_rng(2048 + k).random(R) < 0.7 for k in range(8)]
    Y = np.zeros((B, R, C), np.float32)
    M = np.zeros((B, R, C), np.float32)
    for b in range(B):
        rng = cube_rng("b2048", b)
        Z = rng.standard_normal((R, 3)) @ rng.standard_normal((3, C)) + 0.1 * rng.standard_normal((R, C))
        m = np.repeat(pool[b % 8][:, None], C, axis=1)
        Y[b] = np.where(m, Z * cube_scale(b), 0)
        M[b] = m
    D = synth.synthetic_dictionary(16, 24, seed=24)
    Dd = cu(D)
    prm = Params(Nit=10, bb=4, slidingDis=2)
    sol = LRSPnPBatch(Y, M, Dd, prm).run(2)
    assert all(bool(torch.isfinite(getattr(sol, k)).all()) for k in ("X", "lambda_1", "lambda_2"))
    sample = np.sort(np.random.default_rng(8).choice(B, 8, replace=False))
    for b in sample:
        one = LRSPnP(Y[b], M[b], Dd, prm).run(2)
        for name in ("X", "lambda_1", "lambda_2"):
            r = rel(getattr(sol, name)[b].cpu().numpy(), getattr(one, name).cpu().numpy())
            assert r <= 1e-5, (b, name, r)
    _vs_oracle(sol, Y, M, D, orc.Params(Nit=10, bb=4, slidingDis=2), sample)


# ================================================================ the spectral step constants' pattern limit
@gpu
def test_batch_beyond_the_spectral_pattern_limit():
    """29 cfg 1 cubes with per-element masks have 29 x 144 = 4176 distinct patch patterns, more than the 4096 that
    spectral step constants serve: construction raises with advice that applies to a batch; step='frob4' runs."""
    B, R, C = 29, 1296, 128
    Y = np.zeros((B, R, C), np.float32)
    M = np.zeros((B, R, C), np.float32)
    for b in range(B):
        rng = cube_rng("limit", b)
        m = rng.random((R, C)) < 0.7
        Y[b] = np.where(m, rng.standard_normal((R, C)) * cube_scale(b), 0)
        M[b] = m
    D = synth.synthetic_dictionary(1296, 324, seed=0)
    assert B * ops.patch_count(R, C, 36, 36) > ops.MAX_SPECTRAL_PATTERNS
    with pytest.raises(_lib.LrsError, match=r"batch of 29 cubes: 4176 distinct mask patterns.*step='frob4', or fewer cubes"):
        LRSPnPBatch(Y, M, D, Params(Nit=5))
    sol = LRSPnPBatch(Y, M, D, Params(Nit=5, step="frob4")).run(1)
    assert sol.iterations == 1 and bool(torch.isfinite(sol.X).all())


# ================================================================ E. CPU only
BATCH_ENTRY_POINTS = {
    # name -> arguments with the cube count B at index i (dummy non-null pointers, a valid geometry otherwise)
    "lrs_im2col_batch_f32": lambda p, B: (p, None, 1.0, B, 8, 8, 2, 1, p, None),
    "lrs_col2im_accum_batch_f32": lambda p, B: (p, B, 8, 8, 2, 1, p, None),
    "lrs_gram_batch_f64": lambda p, B: (p, None, 0.0, B, 8, 8, p, None),
    "lrs_sym_eig_jacobi_batch_f64": lambda p, B: (p, B, 8, p, p, p, None),
    "lrs_svt_weights_batch_f64": lambda p, B: (p, p, 64, 8, 1, B, 8, 8, 0.5, 0, p, None),
    "lrs_svt_apply_batch_f32": lambda p, B: (p, None, 0.0, p, B, 8, 8, p, None),
    "lrs_admm_update_batch_f32": lambda p, B: (p, p, p, p, p, p, p, 0.5, 0.15, 0.9, B, 8, 8, 2, 1, None),
}


@pytest.mark.parametrize("B", [0, _lib.MAX_BATCH + 1])
@pytest.mark.parametrize("name", list(BATCH_ENTRY_POINTS))
def test_batched_entry_points_refuse_batch_size(name, B):
    """Every batched entry point returns LRS_E_ARG for B = 0 and B = LRS_MAX_BATCH + 1, naming LRS_MAX_BATCH.  Each
    launcher checks B before it touches a pointer or the device, so host dummies stand in for the device buffers."""
    buf = ctypes.create_string_buffer(64)
    lib = L()
    assert getattr(lib, name)(*BATCH_ENTRY_POINTS[name](ctypes.addressof(buf), B)) == -1        # LRS_E_ARG
    msg = lib.lrs_last_error().decode()
    assert msg.startswith(name) and "LRS_MAX_BATCH" in msg, msg


def test_per_cube_comparators_tell_cubes_apart():
    """Each per-cube comparator of this file passes a cube against its own reference and fails it against the next
    cube's (check_cubes with the references rolled by one)."""
    B, (R, C, bb, s) = 3, GEOMS["s3-appended"]
    roll = lambda refs: refs[1:] + refs[:1]                                        # noqa: E731

    def tells_apart(check, got, refs):
        check_cubes(check, got, refs)
        with pytest.raises(AssertionError, match="cube 0"):
            check_cubes(check, got, roll(refs))

    cubes = [_geom_cube("s3-appended", b) for b in range(B)]
    tells_apart(same_bits, [c[1] for c in cubes], [c[1] for c in cubes])             # im2col
    tells_apart(same_bits, [c[3] for c in cubes], [c[3] for c in cubes])             # col2im
    tells_apart(same_bits, [c[4][0] for c in cubes], [c[4][0] for c in cubes])       # update
    X, Lm = _xl_cubes("self-check", B, 40, 17)
    Z = [z32(X[b], Lm[b], C_OVER_MU2) for b in range(B)]
    tells_apart(_check_gram, [_gram_ref(z)[0] for z in Z], Z)
    W = [cube_rng("self-check-W", b).standard_normal((17, 17)).astype(np.float32) for b in range(B)]
    U = [(z.astype(np.float64) @ w.astype(np.float64)).astype(np.float32) for z, w in zip(Z, W)]
    tells_apart(lambda u, zw: _check_apply(u, *zw), U, list(zip(Z, W)))
    rng = np.random.default_rng(1)
    Q = [np.linalg.qr(rng.standard_normal((17, 17)))[0] for _ in range(B)]
    w = [shrink_weights(10 ** rng.uniform(-2, 2, 17), 1.0) for _ in range(B)]
    Wt = [((q * ww) @ q.T).astype(np.float32) for q, ww in zip(Q, w)]
    tells_apart(lambda W_, ref: _check_weights(W_, *ref), Wt, list(zip(Q, w)))
    # the whole-solver comparison: two cubes of the same batch after two oracle iterations
    Y, M = _stride1_cubes()
    D = np.random.default_rng(2).standard_normal((64, 32)).astype(np.float32)
    oprm = orc.Params(Nit=3, bb=8, slidingDis=1)
    Xs = [orc.run(Y[b], M[b], D, oprm, 1).X for b in (0, 2, 3)]
    tells_apart(close_rel(1e-4), Xs, Xs)
    # the low-rank step's comparison, given the fp64 results of three cubes
    Xl, L2 = _low_rank_cubes(60, 12)
    refs = [svt_fp64(z32(Xl[b], L2[b], C_OVER_MU2), 1 / 0.9) for b in (0, 2, 3)]
    tells_apart(close_rel(1e-5), refs, refs)
