"""Pin the CPU oracle (oracle/lrs_oracle.py) against

 * the committed golden fixtures produced by the reference's own functions
   (tests/golden/make_golden.py), and
 * the literal reference functions themselves when /root/reference is present
   (build container only).
"""
import numpy as np
import pytest

from oracle import lrs_oracle as orc
from oracle import ref_extract as rx

needs_ref = pytest.mark.skipif(not rx.reference_available(), reason="reference checkout not present")


def rel(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ---------------------------------------------------------------- geometry
def test_index_kat_bit_exact(golden):
    g = golden("index_kat")
    for ci in range(int(g["ncases"][0])):
        R, C, bb, s = (int(v) for v in g[f"c{ci}_geom"])
        x, y = orc.patch_index(R, C, bb, s)
        assert np.array_equal(x, g[f"c{ci}_x"]), (R, C, bb, s)
        assert np.array_equal(y, g[f"c{ci}_y"]), (R, C, bb, s)
        assert orc.idx_mat(R, C, bb, s).sum() == g[f"c{ci}_idxsum"][0]
        blocks, x2, y2, idx = orc.get_image_block(g[f"c{ci}_X"], bb, s)
        assert blocks.dtype == np.float32 and x2.dtype == np.int64
        # the reference's x, y are the argwhere of its 0/1 idx_Mat: with the stored sum they fix every 1 of idx_Mat
        assert idx.shape == (R - bb + 1, C - bb + 1) and np.isin(idx, (0, 1)).all()
        assert (idx[g[f"c{ci}_x"], g[f"c{ci}_y"]] == 1).all() and idx.sum() == g[f"c{ci}_idxsum"][0] == len(x)
        if f"c{ci}_blocks" in g:
            assert np.array_equal(blocks, g[f"c{ci}_blocks"])
        else:
            assert np.array_equal(blocks[:, ::7], g[f"c{ci}_blocks_sample"])


def test_shipped_geometry_kat():
    # SURVEY §8c: P = 144, cols {0,36,72,92}, rows 0..1260 step 36
    x, y = orc.patch_index(1296, 128, 36, 36)
    assert len(x) == 144
    assert sorted(set(y.tolist())) == [0, 36, 72, 92]
    assert sorted(set(x.tolist())) == list(range(0, 1261, 36))
    # row start varies fastest (column-major patch order)
    assert x[:3].tolist() == [0, 36, 72] and y[:36].tolist() == [0] * 36
    # (64,41,8,3): 64 % 8 == 0 → last row start 56 is NOT appended
    x, y = orc.patch_index(64, 41, 8, 3)
    assert x.max() == 54 and y.max() == 33


@needs_ref
@pytest.mark.parametrize("geom", [(40, 23, 8, 1), (33, 17, 4, 3), (36, 36, 6, 6), (29, 31, 5, 4), (16, 64, 8, 2)])
def test_get_image_block_vs_literal(geom):
    import torch

    R, C, bb, s = geom
    gib = rx.extract("main_LRS_PnP.py")["get_image_block"]
    X = np.random.default_rng(sum(geom)).standard_normal((R, C)).astype(np.float32)
    b_ref, x_ref, y_ref, idx_ref = gib(torch.tensor(X), bb, s)
    b, x, y, idx = orc.get_image_block(X, bb, s)
    assert np.array_equal(b, b_ref.numpy())
    assert np.array_equal(x, x_ref) and np.array_equal(y, y_ref)
    assert np.array_equal(idx, idx_ref.numpy())


def test_weight_and_col2im_roundtrip():
    rng = np.random.default_rng(0)
    for R, C, bb, s in [(40, 23, 8, 1), (64, 41, 8, 3), (1296, 128, 36, 36), (30, 30, 5, 2)]:
        X = rng.standard_normal((R, C)).astype(np.float32)
        blocks, x, y, _ = orc.get_image_block(X, bb, s)
        W = orc.coverage_weight(R, C, bb, s)
        ones = orc.col2im_accumulate(np.ones_like(blocks), R, C, bb, s)
        assert np.array_equal(ones, W)
        acc = orc.col2im_accumulate(blocks, R, C, bb, s)
        np.testing.assert_allclose(acc, W * X, rtol=2e-6, atol=2e-6)


# ---------------------------------------------------------------- prox / SVT
def test_prox_kat(golden):
    g = golden("prox_kat")
    thr = np.float32(g["thr"][0])
    for key in ("shrink", "soft_thresh", "l1_prox"):
        assert np.array_equal(orc.soft(g["v"], thr), g[key]), key
    assert rel(orc.svt(g["Z"], float(g["tau"][0])), g["svt"]) < 2e-6


# ---------------------------------------------------------------- ISTA
def test_ista_kat(golden):
    g = golden("ista_kat")
    for i in range(int(g["nprobs"][0])):
        H, y, Nit = g[f"p{i}_H"], g[f"p{i}_y"], int(g[f"p{i}_Nit"][0])
        a_s = orc.step_constant(H, "spectral")
        a_f = orc.step_constant(H, "frob4")
        assert abs(a_s - g[f"p{i}_a_spectral"][0]) / a_s < 1e-5
        assert abs(a_f - g[f"p{i}_a_frob4"][0]) / a_f < 1e-5
        x = orc.ista_soft(y, H, 0.1, Nit, "spectral")
        assert rel(x, g[f"p{i}_x_spectral_soft"]) < 2e-5, i
        x = orc.ista_soft(y, H, 0.1, Nit, "frob4")
        assert rel(x, g[f"p{i}_x_frob4_soft"]) < 2e-5, i
        # batched masked form == single-patch form (no missing rows)
        A = orc.ista_soft_batched(y.reshape(-1, 1), np.ones((H.shape[0], 1), bool), H,
                                  np.array([a_s], np.float32), 0.1, Nit)
        assert rel(A, g[f"p{i}_x_spectral_soft"]) < 2e-5


def test_masked_form_equals_row_deletion():
    rng = np.random.default_rng(3)
    n, K, P = 64, 96, 7
    D = rng.standard_normal((n, K)).astype(np.float32) / 8
    blocks = rng.standard_normal((n, P)).astype(np.float32)
    mask = rng.random((n, P)) < 0.6
    mask[:, 0] = True
    for mode in ("spectral", "frob4"):
        a = orc.step_constants_batched(D, mask, mode)
        A = orc.ista_soft_batched(blocks, mask, D, a, 0.1, 40)
        for p in range(P):
            x = orc.ista_soft(blocks[mask[:, p], p], D[mask[:, p]], 0.1, 40, mode)
            assert rel(A[:, p:p + 1], x) < 3e-5, (mode, p)


def test_all_missing_patch_is_defined_zero():
    D = np.eye(4, 6, dtype=np.float32)
    blocks = np.ones((4, 2), np.float32)
    mask = np.array([[1, 0]] * 4, bool)
    a = orc.step_constants_batched(D, mask, "frob4")
    A = orc.ista_soft_batched(blocks, mask, D, a, 0.1, 5)
    assert np.all(A[:, 1] == 0) and np.isfinite(A).all()


# ---------------------------------------------------------------- end to end
@pytest.mark.parametrize("variant", ["spectral", "frob4"])
def test_e2e_small_vs_literal_loop(golden, variant):
    g = golden("e2e_small")
    Y, D, pm = g["Y"], g["D"], g["pixmask"]
    MtM = np.repeat(pm.astype(np.float32)[:, None], Y.shape[1], axis=1)
    mu1, mu2 = (0.15, 0.9) if variant == "spectral" else (0.1, 0.1)
    prm = orc.Params(mu_1=mu1, mu_2=mu2, Nit=80, bb=8, slidingDis=1, step=variant)
    low_rank = None if variant == "spectral" else (lambda Z: Z.copy())
    st = orc.State(X=Y.copy(), lambda_1=np.zeros_like(Y), lambda_2=np.zeros_like(Y))
    for it in (1, 2):
        if it == 1:
            Phi, _ = orc.sparse_step(st.X, st.lambda_1, Y, D, prm)
            assert rel(Phi, g[f"{variant}_Phi_z_1"]) < 2e-5
            assert np.array_equal(orc.coverage_weight(*Y.shape, 8, 1), g[f"{variant}_Weight_1"])
        st = orc.outer_iteration(st, Y, MtM, D, prm, low_rank=low_rank)
        assert rel(st.X, g[f"{variant}_X_{it}"]) < 3e-5, it
        assert rel(st.lambda_1, g[f"{variant}_lambda_1_{it}"]) < 1e-4, it
        assert rel(st.lambda_2, g[f"{variant}_lambda_2_{it}"]) < 1e-4, it


def test_admm_update_and_lam1sum_bit_exact_given_same_inputs(golden):
    # With the literal loop's own IMout/U the elementwise tail must reproduce bit for bit.
    g = golden("e2e_small")
    Y, pm = g["Y"], g["pixmask"]
    MtM = np.repeat(pm.astype(np.float32)[:, None], Y.shape[1], axis=1)
    prm = orc.Params(mu_1=0.15, mu_2=0.9, bb=8, slidingDis=1)
    l1s = orc.lambda1_summation(g["spectral_lambda_1_1"], *Y.shape, 8, 1)
    assert np.array_equal(l1s, g["spectral_lam1sum_2"])
    X2, l1, l2 = orc.admm_update(g["spectral_X_1"], g["spectral_lambda_1_1"], g["spectral_lambda_2_1"], Y, MtM,
                                 g["spectral_IMout_2"], g["spectral_Weight_2"], g["spectral_U_2"], l1s, prm)
    assert np.array_equal(X2, g["spectral_X_2"])
    assert np.array_equal(l1, g["spectral_lambda_1_2"])
    assert np.array_equal(l2, g["spectral_lambda_2_2"])


def test_e2e_bundled_vs_literal_loop(golden):
    gi, ge = golden("bundled_inputs"), golden("e2e_bundled")
    from lrs_pnp_dip_b200 import synth

    Y, pm = gi["base_Y"], gi["base_pixmask"]
    assert ((Y == 0).all(axis=1) == (pm == 0)).all()          # '== 0' ⇔ mask (SURVEY §8c)
    MtM = np.repeat(pm.astype(np.float32)[:, None], 128, axis=1)
    D = synth.synthetic_dictionary(1296, int(ge["K"][0]), seed=0)
    prm = orc.Params()
    st = orc.run(Y, MtM, D, prm, iteration_num=1)
    assert rel(st.X, ge["X1"]) < 3e-5
    st = orc.outer_iteration(st, Y, MtM, D, prm)
    assert rel(st.X, ge["X2"]) < 5e-5


def test_input_mpsnr_kat(golden):
    # list_MPSNR = [33.074]  (main_LRS_PnP_DIP_pro.py:344)
    from lrs_pnp_dip_b200 import matio

    gi = golden("bundled_inputs")
    noisy = matio.fold_cube(gi["base_Y"], 36, 36)
    clean = matio.fold_cube(gi["base_clean"], 36, 36)
    assert abs(orc.mpsnr_ref(clean, noisy) - 33.074) < 1e-3


# ---------------------------------------------------------------- NLM restatement (parity unpinned: no MATLAB here)
def test_nlm_restatement_properties():
    kw = orc.nlm_kernel_rowsums(3)
    assert abs(kw.sum() - 1) < 1e-12 and np.allclose(kw, kw[::-1])
    assert np.allclose(kw, [1 / 21, 4 / 35, 71 / 315, 71 / 315, 71 / 315, 4 / 35, 1 / 21])
    rng = np.random.default_rng(0)
    x = rng.standard_normal(40)
    # h -> 0: every weight underflows and the filter returns its input (NLmeansfilter.m:80-84)
    assert np.array_equal(orc.nlm_column(x, 3, 3, 1e-6), x)
    # constant signal is a fixed point; huge h = plain average over the +-3 search window
    assert np.allclose(orc.nlm_column(np.full(20, 2.5), 3, 3, 0.1), 2.5)
    big = orc.nlm_column(x, 3, 3, 1e6)
    assert abs(big[10] - x[7:14].mean()) < 1e-6


def test_literal_loop_port_matches_reference_and_oracle():
    """oracle/literal_loop.py (the per-patch B0 baseline of bench.py) against the vectorised oracle, and — when the
    checkout is present — against the reference's own ista / delete_element executed literally."""
    from oracle import literal_loop as ll, ref_extract as rx

    rng = np.random.default_rng(2)
    n, K, P = 36, 50, 7
    D = rng.standard_normal((n, K)).astype(np.float32)
    D /= np.linalg.norm(D, axis=0, keepdims=True)
    blocks = rng.standard_normal((n, P)).astype(np.float32)
    mask = rng.random((n, P)) < 0.7
    mask[:, 2] = True
    bc = np.where(mask, blocks + 3.0, 0).astype(np.float32)
    for step in ("spectral", "frob4"):
        phi, dt = ll.sparse_step_literal(blocks, bc, D, 0.1, 30, step)
        a = orc.step_constants_batched(D, mask, step)
        want = D @ orc.ista_soft_batched(blocks, mask, D, a, 0.1, 30)
        assert rel(phi, want) < 2e-5 and dt > 0
        sub, _ = ll.sparse_step_literal(blocks, bc, D, 0.1, 30, step, patches=np.array([5, 1]))
        assert np.array_equal(sub, phi[:, [5, 1]])
    if rx.reference_available():
        import torch

        ns = rx.extract("main_LRS_PnP.py")
        ns["denoise_nl_means"] = rx.soft_shim(10.0)
        phi, _ = ll.sparse_step_literal(blocks, bc, D, 0.1, 30, "spectral")
        for jj in range(P):
            miss = np.where(bc[:, jj] == 0)[0]
            y, H = torch.tensor(blocks[:, jj]).view(-1, 1), torch.tensor(D)
            if len(miss):
                y, H = ns["delete_element"](y, miss.tolist()), ns["delete_element"](H, miss.tolist())
            lit = torch.mm(torch.tensor(D), ns["ista"](y, H, 0.1, 0, 30)).flatten().numpy()
            assert rel(phi[:, jj], lit) < 1e-5, jj


def test_svt_through_the_b_form_of_a_one_sided_jacobi_sweep():
    """The math behind lrs_sym_eig_jacobi_f64 + lrs_svt_weights_f64 (DESIGN 3.3), on the CPU: orthogonalising the columns of
    the band Gram matrix G = Z^T Z by plane rotations gives B = G V with column k = lambda_k v_k, and
    W = sum_k b_k b_k^T max(1 - tau/sqrt(lambda_k), 0) / lambda_k^2 reproduces SVT(Z, tau) = Z W (main_LRS_PnP.py:118-124)."""
    rng = np.random.default_rng(3)
    Z = (rng.standard_normal((400, 4)) @ rng.standard_normal((4, 24)) + 0.05 * rng.standard_normal((400, 24))).astype(np.float32)
    G = Z.astype(np.float64).T @ Z.astype(np.float64)
    B = G.copy()
    for _ in range(12):                                   # cyclic one-sided Jacobi (any order that meets every pair works)
        worst = 0.0
        for p in range(24):
            for q in range(p + 1, 24):
                a, b, g = B[:, p] @ B[:, p], B[:, q] @ B[:, q], B[:, p] @ B[:, q]
                if g * g <= 1e-22 * a * b:
                    continue
                worst = max(worst, g * g / (a * b))
                d, h = b - a, 2.0 * g
                t = (h if d >= 0 else -h) / (abs(d) + np.sqrt(d * d + h * h))
                c = 1.0 / np.sqrt(1.0 + t * t)
                s = c * t
                B[:, p], B[:, q] = c * B[:, p] - s * B[:, q], s * B[:, p] + c * B[:, q]
        if worst <= 1e-9:
            break
    lam = np.linalg.norm(B, axis=0)
    assert np.abs(np.sort(lam) - np.linalg.eigvalsh(G)).max() <= 1e-9 * lam.max()
    for tau in (1.0 / 0.9, 3.0):
        sigma = np.sqrt(lam)
        w = np.where((sigma > tau) & (lam > 1e-12 * lam.max()), (1.0 - tau / np.maximum(sigma, 1e-300)) / lam ** 2, 0.0)
        W = (B * w[None, :]) @ B.T
        got = Z.astype(np.float64) @ W
        want = orc.svt(Z, tau)
        assert np.linalg.norm(got - want) <= 1e-5 * np.linalg.norm(want)


# ---------------------------------------------------------------- helpers of tests/test_kernel_edges.py (CPU self-checks)
def test_de_bruijn_rows_carry_every_row_pattern_once():
    """The de Bruijn row mask of the fused-step edge test: its 2^n row starts see every n-row validity pattern once."""
    from tests.test_kernel_edges import de_bruijn_rows, row_patterns

    for n in (3, 8):
        rows = de_bruijn_rows(n)
        assert rows.shape == ((1 << n) + n - 1,)
        pats = row_patterns(rows, np.arange(1 << n), bb=n)
        assert sorted(pats.tolist()) == list(range(1 << n)), n


def test_svt_fp64_restatement_vs_svd():
    """The fp64 SVT restatement (Gram matrix, eigh, max(1 - tau/sigma, 0), recomposition) equals U soft(S, tau) V^T of an
    fp64 SVD, with tau at 0, mid-spectrum, exactly at a singular value and above the largest one."""
    from tests.test_kernel_edges import svt_fp64

    rng = np.random.default_rng(5)
    Z = rng.standard_normal((300, 5)) @ rng.standard_normal((5, 17)) + 0.05 * rng.standard_normal((300, 17))
    U, S, Vt = np.linalg.svd(Z, full_matrices=False)
    for tau in (0.0, float(np.median(S)), float(S[2]), 2.0 * float(S[0])):
        want = (U * np.maximum(S - tau, 0.0)) @ Vt
        assert np.abs(svt_fp64(Z, tau) - want).max() <= 1e-10 * np.abs(Z).max(), tau
