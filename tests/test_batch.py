"""LRSPnPBatch: B same-shape cubes in one ADMM loop (explicit engine).

CPU: every refusal of the host layer (no device needed), the (image, mask) pairs of the ``lrs_pnp_batch`` driver
subcommand and the cross-mask construction of its cubes.
GPU: each batched entry point slice by slice against its single-cube entry point (bit for bit where the single call is
deterministic), the batch against the stored literal-loop goldens, the batch against B separate LRSPnP solvers, cube
isolation, and a step without host synchronisation.
"""
import numpy as np
import pytest
import torch

from lrs_pnp_dip_b200 import _lib, drivers, matio, metrics, ops, synth
from lrs_pnp_dip_b200.solver import LRSPnP, LRSPnPBatch, Params

gpu = pytest.mark.gpu
IMAGES = ("base", "img2", "img3", "img4", "img5")
MASK_OWNERS = ("base", "img2", "img3", "img4")          # the pixel masks of these images are the four distinct masks


def rel(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def bundled(golden, tag):
    g = golden("bundled_inputs_r2" if tag in ("img3", "img4") else "bundled_inputs")
    return g[f"{tag}_Y"], g[f"{tag}_pixmask"], g[f"{tag}_clean"].astype(np.float32)


def cross_cubes(golden):
    """The 20 cubes (image i, mask m): Y_i with the rows of mask m also zeroed (synth.cross_masked)."""
    out = []
    for img in IMAGES:
        Y, _, _ = bundled(golden, img)
        for owner in MASK_OWNERS:
            out.append((img, owner) + synth.cross_masked(Y, bundled(golden, owner)[1]))
    return out


# ================================================================ CPU: host-layer refusals, pairs, cube construction
def _inputs(B=2, R=40, C=12, n=36, K=50, dtype=np.float32):
    rng = np.random.default_rng(0)
    Y = rng.standard_normal((B, R, C)).astype(dtype)
    return Y, np.ones_like(Y), rng.standard_normal((n, K)).astype(np.float32)


def test_refuses_mismatched_shapes_and_dtypes():
    Y, M, D = _inputs()
    prm = Params(bb=6, slidingDis=6)
    with pytest.raises(ValueError, match="both be"):
        LRSPnPBatch(Y, M[:, :-1], D, prm)
    with pytest.raises(ValueError, match="both be"):
        LRSPnPBatch(Y[0], M[0], D, prm)                           # 2-D: not a batch
    with pytest.raises(ValueError, match="dtype"):
        LRSPnPBatch(Y, M.astype(np.float64), D, prm)
    with pytest.raises(ValueError, match="dtype"):
        LRSPnPBatch(Y.astype(np.int32), M.astype(np.int32), D, prm)
    with pytest.raises(ValueError, match="dictionary has"):
        LRSPnPBatch(Y, M, D[:30], prm)


def test_refuses_bad_geometry():
    Y, M, D = _inputs(R=5)
    with pytest.raises(ValueError, match="geometry"):
        LRSPnPBatch(Y, M, D, Params(bb=6, slidingDis=6))            # bb > R
    Y, M, D = _inputs()
    with pytest.raises(ValueError, match="geometry"):
        LRSPnPBatch(Y, M, D, Params(bb=6, slidingDis=0))


def test_refuses_batch_size_out_of_range():
    Y, M, D = _inputs()
    with pytest.raises(ValueError, match="1..65535"):
        LRSPnPBatch(Y[:0], M[:0], D, Params(bb=6, slidingDis=6))
    big = torch.zeros((_lib.MAX_BATCH + 1, 6, 6))                  # shape checks come before any copy or device work
    with pytest.raises(ValueError, match="1..65535"):
        LRSPnPBatch(big, big, D, Params(bb=6, slidingDis=6))


@pytest.mark.parametrize("K", [64, 128, 192, 256])
def test_refuses_fused_capable_shapes(K):
    Y, M, D = _inputs(n=64, K=K)
    with pytest.raises(_lib.LrsError, match="one LRSPnP per cube"):
        LRSPnPBatch(Y, M, D, Params(bb=8, slidingDis=1))


def test_fused_shape_with_explicit_denoiser_or_other_K_is_not_refused_by_the_fused_rule():
    """bb = 8 with the NLM denoiser, or with K outside the fused set, is served by the explicit engine: the host layer
    lets it through to the device (without one, the refusal is the missing device, not the fused rule)."""
    for K, den in ((64, "nlm"), (96, "soft")):
        Y, M, D = _inputs(n=64, K=K)
        try:
            LRSPnPBatch(Y, M, D, Params(bb=8, slidingDis=1, denoiser=den))
        except _lib.LrsError as e:
            assert "one LRSPnP per cube" not in str(e) and not torch.cuda.is_available()


def test_refuses_low_rank_callables_and_spectral_patch():
    Y, M, D = _inputs()
    with pytest.raises(_lib.LrsError, match="low_rank callable"):
        LRSPnPBatch(Y, M, D, Params(bb=6, slidingDis=6), low_rank=lambda Z: Z)
    with pytest.raises(_lib.LrsError, match="spectral_patch"):
        LRSPnPBatch(Y, M, D, Params(bb=6, slidingDis=6, step="spectral_patch"))
    with pytest.raises(ValueError, match="engine"):
        LRSPnPBatch(Y, M, D, Params(bb=6, slidingDis=6), engine="fast")


def test_driver_batch_pairs():
    pairs = drivers.batch_pairs()
    assert len(pairs) == 20 and len(set(pairs)) == 20
    assert {i for i, _ in pairs} == set(drivers.PAIRS) and {m for _, m in pairs} == set(drivers.BATCH_MASKS)
    # the four distinct masks of the pair table, img5 sharing img4's
    assert {drivers.PAIRS[i][2][:-4] for i in drivers.PAIRS} == set(drivers.BATCH_MASKS)
    assert drivers.batch_pairs("base:fourth_mask.mat, img5:second_mask") == [("base", "fourth_mask"), ("img5", "second_mask")]
    for bad in ("base", "img9:second_mask", "base:fifth_mask", ""):
        with pytest.raises(ValueError):
            drivers.batch_pairs(bad)
    with pytest.raises(ValueError, match="bad pair"):              # the subcommand parses its pairs before loading
        drivers.main(["lrs_pnp_batch", "--data-dir", "unused", "--pairs", "base:fifth_mask"])


def test_cross_masked_cubes(golden):
    cubes = cross_cubes(golden)
    assert len(cubes) == 20
    for img, owner, Y, M in cubes:
        Yi, pm_i, _ = bundled(golden, img)
        keep = (pm_i != 0) & (bundled(golden, owner)[1] != 0)
        assert np.array_equal((Y != 0).any(axis=1), keep) and np.array_equal(M[:, 0] != 0, keep)
        assert (M == M[:, :1]).all() and np.array_equal(Y[keep], Yi[keep])
    # a cube against its own mask is the bundled cube
    Y0, _, _ = bundled(golden, "img2")
    assert np.array_equal(cubes[IMAGES.index("img2") * 4 + 1][2], Y0)


# ================================================================ GPU 1: kernel by kernel, cube by cube
GEOMS = {"cfg1": (1296, 128, 36, 36), "s3-appended": (42, 31, 8, 3), "b191-s3-appended": (46, 191, 6, 3)}


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def stream():
    return torch.cuda.current_stream().cuda_stream


@gpu
@pytest.mark.parametrize("name", list(GEOMS))
def test_batched_entry_points_equal_single_calls(name):
    R, C, bb, s = GEOMS[name]
    B, L = 5, _lib.lib()
    rng = np.random.default_rng(11)
    X = cu(rng.standard_normal((B, R, C)).astype(np.float32))
    Lam = cu((0.1 * rng.standard_normal((B, R, C))).astype(np.float32))
    P, n = ops.patch_count(R, C, bb, s), bb * bb
    # im2col, without and with the multiplier term
    for lam in (None, Lam):
        got = ops.im2col_batch(X, bb, s, lam, 0.15)
        for b in range(B):
            one = ops.im2col(X[b], bb, s, None if lam is None else lam[b], 0.15)
            assert torch.equal(got[:, b * P:(b + 1) * P], one), (name, b)
    # col2im
    blocks = cu(rng.standard_normal((n, B * P)).astype(np.float32))
    got = ops.col2im_batch(blocks, B, R, C, bb, s)
    for b in range(B):
        assert torch.equal(got[b], ops.col2im(blocks[:, b * P:(b + 1) * P].contiguous(), R, C, bb, s)), (name, b)
    # Gram: fp64 atomics; bit-identical where the single call is deterministic (one row chunk)
    c = 1.0 / 0.9
    G = torch.zeros((B, C, C), dtype=torch.float64, device="cuda")
    _lib.check(L.lrs_gram_batch_f64(X.data_ptr(), Lam.data_ptr(), c, B, R, C, G.data_ptr(), stream()))
    for b in range(B):
        G1 = torch.zeros((C, C), dtype=torch.float64, device="cuda")
        _lib.check(L.lrs_gram_f64(X[b].data_ptr(), Lam[b].data_ptr(), c, R, C, G1.data_ptr(), stream()))
        Z = (X[b].cpu().numpy() + np.float32(c) * Lam[b].cpu().numpy()).astype(np.float64)
        assert rel(G[b].cpu(), Z.T @ Z) < 1e-12 and rel(G[b].cpu(), G1.cpu()) < 1e-12
        if R <= 256:
            assert torch.equal(G[b], G1), (name, b)
    # Jacobi eigensolver, given the same G
    lam, Bt, st = ops.sym_eig_jacobi_batch(G)
    for b in range(B):
        l1, B1, s1 = ops.sym_eig_jacobi(G[b])
        assert torch.equal(lam[b], l1) and torch.equal(Bt[b], B1) and torch.equal(st[b], s1), (name, b)
        assert int(s1[1]) == 0 and int(s1[2]) == 0
    # weights: B form (Jacobi) and eigenvector form (library eigh, column-major V)
    tau = 0.9
    W = torch.empty((B, C, C), dtype=torch.float32, device="cuda")
    _lib.check(L.lrs_svt_weights_batch_f64(lam.data_ptr(), Bt.data_ptr(), C * C, 1, C, B, C, C, tau, 1, W.data_ptr(), stream()))
    evals, V = torch.linalg.eigh(G)
    W2 = torch.empty_like(W)
    _lib.check(L.lrs_svt_weights_batch_f64(evals.data_ptr(), V.data_ptr(), V.stride(0), V.stride(1), V.stride(2), B, C, C, tau,
                                           0, W2.data_ptr(), stream()))
    for b in range(B):
        w1 = torch.empty((C, C), dtype=torch.float32, device="cuda")
        _lib.check(L.lrs_svt_weights_f64(lam[b].data_ptr(), Bt[b].data_ptr(), 1, C, C, C, tau, 1, w1.data_ptr(), stream()))
        assert torch.equal(W[b], w1), (name, b)
        Vb = V[b]
        _lib.check(L.lrs_svt_weights_f64(evals[b].data_ptr(), Vb.data_ptr(), Vb.stride(0), Vb.stride(1), C, C, tau, 0,
                                         w1.data_ptr(), stream()))
        assert torch.equal(W2[b], w1), (name, b)
    # recomposition
    U = torch.empty_like(X)
    _lib.check(L.lrs_svt_apply_batch_f32(X.data_ptr(), Lam.data_ptr(), c, W.data_ptr(), B, R, C, U.data_ptr(), stream()))
    for b in range(B):
        u1 = torch.empty((R, C), dtype=torch.float32, device="cuda")
        _lib.check(L.lrs_svt_apply_f32(X[b].data_ptr(), Lam[b].data_ptr(), c, W[b].data_ptr(), R, C, u1.data_ptr(), stream()))
        assert torch.equal(U[b], u1), (name, b)
    # X / multiplier update
    Y = cu(rng.standard_normal((B, R, C)).astype(np.float32))
    M = cu((rng.random((B, R, 1)) < 0.7).astype(np.float32).repeat(C, axis=2))
    IM = cu(rng.standard_normal((B, R, C)).astype(np.float32))
    l1, l2 = Lam.clone(), cu((0.1 * rng.standard_normal((B, R, C))).astype(np.float32))
    l1_ref, l2_ref = l1.clone(), l2.clone()
    Xo = torch.empty_like(X)
    _lib.check(L.lrs_admm_update_batch_f32(Y.data_ptr(), M.data_ptr(), IM.data_ptr(), U.data_ptr(), l1.data_ptr(),
                                           l2.data_ptr(), Xo.data_ptr(), 0.5, 0.15, 0.9, B, R, C, bb, s, stream()))
    for b in range(B):
        x1 = torch.empty((R, C), dtype=torch.float32, device="cuda")
        _lib.check(L.lrs_admm_update_f32(Y[b].data_ptr(), M[b].data_ptr(), IM[b].data_ptr(), U[b].data_ptr(),
                                         l1_ref[b].data_ptr(), l2_ref[b].data_ptr(), x1.data_ptr(), 0.5, 0.15, 0.9, R, 0, R, C,
                                         bb, s, stream()))
        assert torch.equal(Xo[b], x1) and torch.equal(l1[b], l1_ref[b]) and torch.equal(l2[b], l2_ref[b]), (name, b)


def _psd_batch(B, C, seed):
    rng = np.random.default_rng(seed)
    Z = rng.standard_normal((B, 3 * C, C))
    return cu(np.einsum("brc,brd->bcd", Z, Z))


@gpu
def test_jacobi_batch_larger_than_the_gpu():
    """B = 24 at C = 128: 192 CTAs (24 clusters of 8), more than the 148 SMs hold at once."""
    G = _psd_batch(24, 128, 3)
    lam, Bt, st = ops.sym_eig_jacobi_batch(G)
    for b in range(24):
        l1, B1, s1 = ops.sym_eig_jacobi(G[b])
        assert torch.equal(lam[b], l1) and torch.equal(Bt[b], B1) and torch.equal(st[b], s1), b
    assert int(st[:, 1:].abs().sum()) == 0
    ref = np.linalg.eigvalsh(G.cpu().numpy())
    assert rel(np.sort(lam.cpu().numpy(), axis=1), ref) < 1e-12


@gpu
def test_jacobi_batch_flags_only_the_non_finite_cube():
    G = _psd_batch(5, 31, 4)
    G[2, 3, 7] = float("nan")
    G[2, 7, 3] = float("nan")
    lam, Bt, st = ops.sym_eig_jacobi_batch(G)
    st = st.cpu().numpy()
    assert st[2, 2] == 1 and (st[[0, 1, 3, 4], 1:] == 0).all()
    assert ops.eig_status_failures(st) == ([2], [])
    for b in (0, 1, 3, 4):
        l1, B1, _ = ops.sym_eig_jacobi(G[b])
        assert torch.equal(lam[b], l1) and torch.equal(Bt[b], B1)


# ================================================================ GPU 2/3: pinned to the stored literal-loop goldens
def ref_metrics(clean, X):
    c = torch.from_numpy(matio.fold_cube(clean, 36, 36))
    x = torch.from_numpy(matio.fold_cube(np.asarray(X, np.float32), 36, 36))
    return metrics.mpsnr(c, x), metrics.ssim(c, x)


@gpu
def test_batch_base_img5_against_literal_loop_goldens(golden):
    ge, gc = golden("e2e_bundled"), golden("e2e_configs")
    assert int(ge["K"][0]) == int(gc["K_bundled"][0])
    cases = [bundled(golden, t) for t in ("base", "img5")]
    Y = np.stack([c[0] for c in cases])
    M = np.stack([np.repeat(c[1].astype(np.float32)[:, None], 128, axis=1) for c in cases])
    D = synth.synthetic_dictionary(1296, int(ge["K"][0]), seed=0)
    sol = LRSPnPBatch(Y, M, D, Params())
    sol.step()
    X1 = sol.X.cpu().numpy()
    assert rel(X1[0], ge["X1"]) < 1e-4 and rel(X1[1], gc["cfg1_X1"]) < 1e-4
    sol.step()
    sol.validate()
    X2 = sol.X.cpu().numpy()
    assert rel(X2[0], ge["X2"]) < 1e-4 and rel(X2[1], gc["cfg1_X2"]) < 1e-4
    mp, ms = ref_metrics(cases[1][2], X2[1])
    assert abs(mp - gc["cfg1_mpsnr_mssim_2"][0]) < 0.01 and abs(ms - gc["cfg1_mpsnr_mssim_2"][1]) < 1e-4


@gpu
def test_batch_dip_parameters_first_phi_z(golden):
    gc = golden("e2e_configs")
    tags = ("img2", "img3", "img4", "img5")
    cases = [bundled(golden, t) for t in tags]
    Y = np.stack([c[0] for c in cases])
    M = np.stack([np.repeat(c[1].astype(np.float32)[:, None], 128, axis=1) for c in cases])
    D = synth.synthetic_dictionary(1296, int(gc["K_bundled"][0]), seed=0)
    prm = Params(gamma=0.5, mu_1=0.1, mu_2=0.1, lambda_ista=0.1, Nit=100, bb=36, slidingDis=36, step="frob4")
    sol = LRSPnPBatch(Y, M, D, prm)
    phi = sol.coder.phi_z(sol.X, sol.lambda_1).cpu().numpy()
    P = sol.coder.P
    assert phi.shape == (1296, 4 * P)
    for b, t in enumerate(tags):
        assert rel(phi[:, b * P:(b + 1) * P][::9, ::5], gc[f"cfg23_{t}_Phi_z1_sample"]) < 1e-4, t


# ================================================================ GPU 4: batch == separate solvers
@gpu
def test_batch_equals_separate_solvers_on_twenty_cubes(golden):
    cubes = cross_cubes(golden)
    D = synth.synthetic_dictionary(1296, 324, seed=0)
    prm = Params()
    Y = np.stack([c[2] for c in cubes])
    M = np.stack([c[3] for c in cubes])
    sol = LRSPnPBatch(Y, M, D, prm).run(2)
    P = sol.coder.P
    for b, (img, owner, Yb, Mb) in enumerate(cubes):
        one = LRSPnP(Yb, Mb, D, prm)
        assert torch.equal(sol.coder.a_patch[b * P:(b + 1) * P], one.be.coder.a_patch), (img, owner)
        one.run(2)
        for name in ("X", "lambda_1", "lambda_2"):
            assert rel(getattr(sol, name)[b].cpu().numpy(), getattr(one, name).cpu().numpy()) < 1e-5, (img, owner, name)


# ================================================================ GPU 5/6: isolation, no host synchronisation
def _four(golden):
    cubes = cross_cubes(golden)[::5]                             # four cubes, four different masks
    return np.stack([c[2] for c in cubes]), np.stack([c[3] for c in cubes]), synth.synthetic_dictionary(1296, 324, seed=0)


@gpu
def test_cubes_do_not_interact(golden):
    Y, M, D = _four(golden)
    clean = LRSPnPBatch(Y, M, D, Params())
    bad = LRSPnPBatch(Y, M, D, Params())
    clean.step()
    bad.step()
    clean.validate()
    bad.X[2, 100, 5] = float("nan")
    clean.step()
    bad.step()
    with pytest.raises(_lib.LrsError, match=r"cube\(s\) \[2\]"):
        bad.validate()
    for b in (0, 1, 3):
        for name in ("X", "lambda_1", "lambda_2"):
            assert torch.equal(getattr(bad, name)[b], getattr(clean, name)[b]), (b, name)


@gpu
def test_step_does_not_synchronise_with_the_host(golden):
    Y, M, D = _four(golden)
    sol = LRSPnPBatch(Y, M, D, Params())
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        sol.step()
        sol.step()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    sol.validate()
    assert sol.iterations == 2 and bool(torch.isfinite(sol.X).all())
    sol.reset()
    assert torch.equal(sol.X, sol.Y) and sol.iterations == 0 and not bool(sol.lambda_1.any())
