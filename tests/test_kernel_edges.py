"""Each kernel by itself against a plain fp64 restatement, at the shapes and values where kernels go wrong: the low-rank
kernels (Gram matrix, shrinkage weights, recomposition) at every band count the configurations run, the step-constant
table for all 256 row patterns, the fused sparse step at the edges of its tile schedule (compared patch by patch), and
the X / multiplier update across geometries and row stripes.  Run on the B200 box: pytest -m gpu.

All inputs come from seeded generators.  The helpers at the top are also used by CPU-only self-checks in
tests/test_oracle.py.
"""
import numpy as np
import pytest
import torch

from lrs_pnp_dip_b200 import _lib, ops, synth
from oracle import lrs_oracle as orc

pytestmark = pytest.mark.gpu

F32_EPS = 2.0 ** -24          # unit roundoff of fp32


# ---------------------------------------------------------------- helpers (CPU)
def per_patch_err(got, ref, floor=1e-30):
    """||got_p - ref_p|| / max(||ref_p||, floor) for every column p."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    return np.linalg.norm(got - ref, axis=0) / np.maximum(np.linalg.norm(ref, axis=0), floor)


def rel(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def de_bruijn_rows(n=8):
    """Linearised binary de Bruijn sequence B(2, n) as a bool array of 2^n + n - 1 entries: its 2^n windows of n
    consecutive entries are all different, so they carry every n-bit pattern exactly once."""
    a = [0] * (2 * n)
    seq = []

    def db(t, p):
        if t > n:
            if n % p == 0:
                seq.extend(a[1:p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, 2):
                a[t] = j
                db(t + 1, t)

    db(1, 1)
    return np.array(seq + seq[:n - 1], dtype=bool)


def row_patterns(row_obs, starts, bb=8):
    """Bit i set iff unfolded row start + i is observed: the index of the step-constant table."""
    return sum(row_obs[starts + i].astype(np.int64) << i for i in range(bb))


def shrink_weights(lam, tau):
    """w_k = max(1 - tau/sigma_k, 0) with sigma_k = sqrt(max(lambda_k, 0)); 0 where sigma_k <= tau (also sigma = tau = 0)."""
    sigma = np.sqrt(np.maximum(np.asarray(lam, np.float64), 0.0))
    keep = sigma > tau
    return np.where(keep, 1.0 - tau / np.where(keep, sigma, 1.0), 0.0)


def svt_weights_fp64(Z, tau):
    """W = V diag(w) V^T from the fp64 Gram matrix of Z, so that SVT(Z, tau) = Z W."""
    Z = np.asarray(Z, np.float64)
    lam, V = np.linalg.eigh(Z.T @ Z)
    return (V * shrink_weights(lam, tau)) @ V.T


def svt_fp64(Z, tau):
    """SVT(Z, tau) = U soft(S, tau) V^T restated in fp64: Gram matrix, eigh, shrinkage weights, recomposition."""
    return np.asarray(Z, np.float64) @ svt_weights_fp64(Z, tau)


# ---------------------------------------------------------------- device plumbing
@pytest.fixture(scope="module")
def lrs():
    import lrs_pnp_dip_b200 as m

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m._lib.lib()
    return m


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


# ================================================================ A. step-constant table
def _coherent_dictionary():
    rng = np.random.default_rng(12)
    D = rng.standard_normal((64, 1)) + 0.1 * rng.standard_normal((64, 256))
    return (D / np.linalg.norm(D, axis=0, keepdims=True)).astype(np.float32)


def _orthonormal_rows():
    Q, _ = np.linalg.qr(np.random.default_rng(7).standard_normal((128, 64)))
    return (1.5 * Q.T).astype(np.float32)                   # D D^T = 2.25 I: every masked Gram matrix is a multiple of a projector


def _near_degenerate_top():
    rng = np.random.default_rng(8)
    U, _ = np.linalg.qr(rng.standard_normal((64, 64)))
    V, _ = np.linalg.qr(rng.standard_normal((256, 64)))
    s = np.r_[1.0, 1.0 - 1e-7, np.linspace(0.5, 0.01, 62)]
    return ((U * s) @ V.T).astype(np.float32)


def _dominant_top():
    D = synth.synthetic_dictionary(64, 256, seed=4)
    D[:, :40] += 0.6 * D[:, [0]]                            # coherent atoms: a dominant singular value
    return D


TABLE_DICTIONARIES = {
    **{f"gaussian-K{K}": (lambda K=K: synth.synthetic_dictionary(64, K, seed=K)) for K in (64, 128, 192, 256)},
    "orthonormal-rows": _orthonormal_rows,
    "near-degenerate-top": _near_degenerate_top,
    "coherent": _coherent_dictionary,
    "dominant-top": _dominant_top,
    "rank-16": lambda: synth.synthetic_dictionary(64, 16, seed=16),
    "scale-2^-20": lambda: synth.synthetic_dictionary(64, 256, seed=3) * np.float32(2.0 ** -20),
    "scale-2^20": lambda: synth.synthetic_dictionary(64, 256, seed=3) * np.float32(2.0 ** 20),
}


@pytest.mark.parametrize("name", list(TABLE_DICTIONARIES))
def test_step_constant_table_every_pattern(lrs, name):
    """The row-pattern table (lrs_spectral_patterns_f32 on the 256 row-pattern words) for all 256 row-validity patterns
    against np.linalg.norm(D[valid], 2)**2 and 4||D[valid]||_F^2 in fp64; the empty pattern gives exactly 0."""
    D = TABLE_DICTIONARIES[name]()
    Dd = cu(D)
    tab_s = ops._row_pattern_table(Dd, 8, "spectral").cpu().numpy()
    tab_f = ops._row_pattern_table(Dd, 8, "frob4").cpu().numpy()
    assert tab_s[0] == 0.0 and tab_f[0] == 0.0
    k_rows = np.arange(64) % 8
    bad = []
    for pat in range(1, 256):
        H = D[((pat >> k_rows) & 1).astype(bool)].astype(np.float64)
        ref_s = np.linalg.norm(H, 2) ** 2
        ref_f = 4.0 * (H ** 2).sum()
        if not abs(tab_s[pat] - ref_s) <= 2e-6 * ref_s or not abs(tab_f[pat] - ref_f) <= 2e-6 * ref_f:
            bad.append((pat, float(tab_s[pat]), ref_s, float(tab_f[pat]), ref_f))
    assert not bad, bad[:8]


@pytest.mark.parametrize("name", ["coherent", "near-degenerate-top", "gaussian-K256"])
def test_step_constant_table_is_repeatable(lrs, name):
    """The table is a deterministic function of the dictionary: three calls return the same bits."""
    Dd = cu(TABLE_DICTIONARIES[name]())
    for step in ("spectral", "frob4"):
        first = ops._row_pattern_table(Dd, 8, step)
        for _ in range(2):
            assert torch.equal(ops._row_pattern_table(Dd, 8, step), first), step


def test_step_constant_table_built_without_host_sync(lrs):
    """Building the solver in the table mode, with the table not yet cached, does not synchronise with the host."""
    H, W, B = 12, 12, 20
    _, noisy = synth.synthetic_cube(H, W, B, rank=4, seed=1)
    Y = synth.observe(noisy, synth.pixel_mask(H, W, keep=0.6, seed=2))
    Yd, Md, Dd = cu(Y), cu((Y != 0).astype(np.float32)), cu(synth.synthetic_dictionary(64, 256, seed=0))
    prm = lrs.Params(bb=8, slidingDis=1, step="spectral")
    ops._TABLE_CACHE.clear()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        sol = lrs.LRSPnP(Yd, Md, Dd, prm)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert sol.be.coder.a_table is not None and len(ops._TABLE_CACHE) == 1


# ================================================================ B. fused sparse step at the geometry edges
MU1, LAM, NIT = 0.15, 0.1, 30

# name -> (R, C, s); "debruijn": rows observed after a de Bruijn sequence, 256 row starts = every 8-row pattern once
FUSED_GEOMS = {
    "P1": (8, 8, 1),
    "one-full-tile": (135, 9, 1),
    "full-tile-plus-one": (136, 8, 1),
    "debruijn": (263, 12, 1),
    "tiny-tiles-many-columns": (15, 300, 1),
    "s3-appended-starts": (301, 30, 3),
    "s5-two-tiles": (1031, 17, 5),
    "s-equals-bb": (64, 64, 8),
    "s-above-bb": (50, 9, 20),
}
FUSED_MODES = ("table", "a_patch", "frob4", "frob4-elementwise")
FUSED_CASES = [(g, 256, FUSED_MODES) for g in FUSED_GEOMS] + \
              [(g, K, ("table", "a_patch")) for g in ("debruijn", "s3-appended-starts") for K in (64, 128, 192)]


def _fused_inputs(name, K, elementwise):
    R, C, s = FUSED_GEOMS[name]
    rng = np.random.default_rng(R * 1000 + C + K)
    X = (rng.standard_normal((R, C)) * 0.3 + 0.5).astype(np.float32)
    L = (rng.standard_normal((R, C)) * 0.01).astype(np.float32)
    if name == "debruijn":
        row_obs = de_bruijn_rows(8)
    else:
        row_obs = rng.random(R) < 0.6
        row_obs[0] = True                                    # P = 1 must not be a dead patch
        if R >= 40:
            row_obs[R // 3:R // 3 + 10] = False              # a run of missing rows: patches with no observed entry
    M = np.repeat(row_obs[:, None], C, axis=1)
    if elementwise:
        M = M & (rng.random((R, C)) < 0.7)
    Y = np.where(M, X + 0.01, 0).astype(np.float32)
    Y[M & (Y == 0)] = 1e-12
    return X, L, Y, M, row_obs, synth.synthetic_dictionary(64, K, seed=K + 5)


@pytest.mark.parametrize("name,K,modes", FUSED_CASES, ids=[f"{g}-K{K}" for g, K, _ in FUSED_CASES])
def test_fused_step_geometry_edges_per_patch(lrs, name, K, modes):
    """lrs_sparse_step_fused_f32, both engines and the dynamically dealt tcgen05 instance, in every step-constant mode,
    against the fp64 oracle given the same step constants: global rel-L2, the worst single patch (allowed 4x the fp32
    oracle's own per-patch error, at least 1e-3), dead patches exactly 0, tc against FFMA per patch, and the dynamic
    instance bit-identical to the static one."""
    R, C, s = FUSED_GEOMS[name]
    xs, ys = orc.patch_index(R, C, 8, s)
    P = len(xs)
    assert P <= 3000
    if name == "debruijn":
        pats = row_patterns(de_bruijn_rows(8), orc.axis_starts(R, 8, s))
        assert sorted(pats.tolist()) == list(range(256))
    oprm = orc.Params(mu_1=MU1, lambda_ista=LAM, Nit=NIT, bb=8, slidingDis=s)
    for mode in modes:
        X, L, Y, M, row_obs, D = _fused_inputs(name, K, mode == "frob4-elementwise")
        Xd, Ld, Yd, Dd = cu(X), cu(L), cu(Y), cu(D)
        mask = orc.patch_masks(orc.get_image_block(Y, 8, s)[0])
        dead = ~mask.any(axis=0)
        a_patch_d = a_table_d = None
        if mode == "table":
            a_table_d = ops._row_pattern_table(Dd, 8, "spectral")
            a = a_table_d.cpu().numpy()[row_patterns(row_obs, xs)]
        elif mode == "a_patch":
            a = orc.step_constants_batched(D, mask, "spectral")
            a_patch_d = cu(a)
        else:
            a = orc.step_constants_batched(D, mask, "frob4")
        ref64, _ = orc.sparse_step(X, L, Y, D, oprm, a=a.astype(np.float64), dtype=np.float64)
        ref32, _ = orc.sparse_step(X, L, Y, D, oprm, a=a.astype(np.float32), dtype=np.float32)
        assert np.all(ref64[:, dead] == 0)
        floor = 1e-6 * float(np.linalg.norm(ref64, axis=0).max())
        allow = max(1e-3, 4.0 * float(per_patch_err(ref32, ref64, floor).max()))

        def call(engine):
            phi = torch.full((64, P), float("nan"), dtype=torch.float32, device="cuda")
            _lib.check(_lib.lib().lrs_sparse_step_fused_f32(
                _lib.ptr(Xd), _lib.ptr(Ld), MU1, _lib.ptr(Yd), _lib.ptr(Dd), K, _lib.ptr(a_patch_d), _lib.ptr(a_table_d),
                LAM, NIT, R, C, 8, s, 0, P, _lib.ptr(phi), engine, _lib.stream_ptr()), "lrs_sparse_step_fused_f32")
            return phi.cpu().numpy()

        out = {"simt": call(_lib.ENGINE_SIMT), "tc": call(_lib.ENGINE_TC)}
        dyn = call(_lib.ENGINE_TC | _lib.ENGINE_DYNAMIC_TILES)
        for engine, phi in out.items():
            where = (mode, engine)
            assert np.isfinite(phi).all(), where
            assert rel(phi, ref64) <= 1e-4, where
            err = per_patch_err(phi, ref64, floor)
            assert err.max() <= allow, (where, int(err.argmax()), float(err.max()), allow)
            assert np.all(phi[:, dead] == 0), where
        tc_simt = per_patch_err(out["tc"], out["simt"], floor)
        assert tc_simt.max() <= 1e-4, (mode, int(tc_simt.argmax()), float(tc_simt.max()))
        assert np.array_equal(dyn, out["tc"]), mode


def test_fused_simt_rejects_unsupported_dictionary_width(lrs):
    """The FFMA engine is instantiated for K in {64, 128, 192, 256} only: K = 96 is an argument error with a message."""
    R, C, K = 40, 12, 96
    rng = np.random.default_rng(0)
    X = cu(rng.standard_normal((R, C)).astype(np.float32))
    D = cu(rng.standard_normal((64, K)).astype(np.float32))
    P = (R - 7) * (C - 7)
    phi = torch.empty((64, P), dtype=torch.float32, device="cuda")
    L = _lib.lib()
    rc = L.lrs_sparse_step_fused_f32(_lib.ptr(X), None, MU1, _lib.ptr(X), _lib.ptr(D), K, None, None, LAM, 5, R, C, 8, 1, 0, P,
                                     _lib.ptr(phi), _lib.ENGINE_SIMT, _lib.stream_ptr())
    assert rc == -1                                           # LRS_E_ARG
    assert b"K in {64,128,192,256}" in L.lrs_last_error()


# ================================================================ C. low-rank kernels
C_OVER_MU2 = np.float32(1 / 0.9)


def _z32(X, L, c):
    """Z exactly as the kernels form it: fl32(X + fl32(c * L))."""
    return X if L is None else (X + np.float32(c) * L).astype(np.float32)


def _gram(X, L=None, c=0.0, G=None):
    R, C = X.shape
    if G is None:
        G = torch.zeros((C, C), dtype=torch.float64, device="cuda")
    _lib.check(_lib.lib().lrs_gram_f64(_lib.ptr(X), _lib.ptr(L), float(c), R, C, _lib.ptr(G), _lib.stream_ptr()), "lrs_gram_f64")
    return G


def _gram_ref(Z, chunk=1 << 16):
    """(Z^T Z, |Z|^T |Z|) in fp64, summed over row chunks (bounded temporaries at a million rows)."""
    C = Z.shape[1]
    G, A = np.zeros((C, C)), np.zeros((C, C))
    for r0 in range(0, Z.shape[0], chunk):
        z = Z[r0:r0 + chunk].astype(np.float64)
        G += z.T @ z
        A += np.abs(z).T @ np.abs(z)
    return G, A


def _check_gram(G, Z, mult=1.0):
    ref, bound = _gram_ref(Z)
    err = np.abs(G - mult * ref)
    assert np.all(err <= 1e-12 * mult * bound), (float(err.max()), np.unravel_index(int(np.argmax(err - 1e-12 * mult * bound)), err.shape))


GRAM_CASES = [(R, C) for C in (1, 63, 64, 65, 128, 191, 224, 256) for R in (1, 15, 16, 17, 255, 257, 4099)] + \
             [(262144, 191), (1048576, 224)]


@pytest.mark.parametrize("R,C", GRAM_CASES)
def test_gram_vs_fp64(lrs, R, C):
    """lrs_gram_f64 without and with the lambda term (c = 1/mu_2) against Z^T Z in fp64.  Products of fp32 numbers are
    exact in fp64, so only the order of the sums differs: 1e-12 of |Z|^T |Z| elementwise.  A dropped row or a misplaced
    tile is an O(1) error."""
    rng = np.random.default_rng(R + 7 * C)
    X = rng.standard_normal((R, C), dtype=np.float32)
    L = rng.standard_normal((R, C), dtype=np.float32)
    Xd, Ld = cu(X), cu(L)
    _check_gram(_gram(Xd).cpu().numpy(), X)
    _check_gram(_gram(Xd, Ld, C_OVER_MU2).cpu().numpy(), _z32(X, L, C_OVER_MU2))


@pytest.mark.parametrize("C", [65, 224])
def test_gram_accumulates_into_g(lrs, C):
    """G is accumulated INTO: a second call doubles it, and the Gram matrices of row stripes summed into one G give the
    whole matrix's (the sharded all-reduce relies on both)."""
    R = 4099
    rng = np.random.default_rng(C)
    X = rng.standard_normal((R, C), dtype=np.float32)
    L = rng.standard_normal((R, C), dtype=np.float32)
    Z = _z32(X, L, C_OVER_MU2)
    Xd, Ld = cu(X), cu(L)
    G = _gram(Xd, Ld, C_OVER_MU2)
    _gram(Xd, Ld, C_OVER_MU2, G)
    _check_gram(G.cpu().numpy(), Z, mult=2.0)
    G = torch.zeros((C, C), dtype=torch.float64, device="cuda")
    for a, b in ((0, 1000), (1000, 1001), (1001, 1017), (1017, R)):
        _gram(Xd[a:b], Ld[a:b], C_OVER_MU2, G)
    _check_gram(G.cpu().numpy(), Z)


def _weights(lam, V, sr, sk, C, n, tau, b_form):
    lam_d = torch.as_tensor(np.ascontiguousarray(lam, np.float64)).cuda()
    V_d = torch.as_tensor(np.ascontiguousarray(V, np.float64)).cuda()
    W = torch.full((C, C), float("nan"), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib().lrs_svt_weights_f64(_lib.ptr(lam_d), _lib.ptr(V_d), sr, sk, C, n, float(tau), int(b_form), _lib.ptr(W),
                                              _lib.stream_ptr()), "lrs_svt_weights_f64")
    return W.cpu().numpy()


def _check_weights(W, Vl, w):
    """W (fp32) against Vl diag(w) Vl^T in fp64 (Vl = the C x n matrix the kernel addresses)."""
    ref = (Vl * w) @ Vl.T
    bound = (np.abs(Vl) * np.abs(w)) @ np.abs(Vl).T
    err = np.abs(W.astype(np.float64) - ref)
    assert np.isfinite(W).all()
    assert np.all(err <= 2 * F32_EPS * np.abs(ref) + 1e-13 * bound), float((err - 2 * F32_EPS * np.abs(ref)).max())


def _spectra(C, tau, rng):
    """Eigenvalues with the shrinkage edges in front: sigma == tau exactly, tau (1 +- 1e-12), a tiny negative value and 0
    (clamped to sigma = 0), one well above tau; the rest spread over four decades.  C < 6: one spectrum per edge group."""
    t2 = tau * tau
    edges = np.array([t2, (tau * (1 + 1e-12)) ** 2, (tau * (1 - 1e-12)) ** 2, -1e-14, 0.0, 9 * t2 + 1])
    base = max(t2, 1.0) * 10 ** rng.uniform(-2, 2, C)
    for i in range(0, len(edges), C):
        lam = base.copy()
        e = edges[i:i + C]
        lam[:len(e)] = e
        yield rng.permutation(lam)


@pytest.mark.parametrize("C", [1, 15, 16, 17, 191, 224, 256])
def test_svt_weights_vs_fp64(lrs, C):
    """lrs_svt_weights_f64 against V diag(max(1 - tau/sigma, 0)) V^T in fp64: plain form with V row- and column-major, at
    sigma == tau and within 1e-12 of it, tiny negative eigenvalues, tau = 0 (zero eigenvalues keep weight 0); B form
    (column k = lambda_k v_k, weights / lambda_k^2) with directions at and below the 1e-12 lambda_max cut."""
    rng = np.random.default_rng(C)
    Q, _ = np.linalg.qr(rng.standard_normal((C, C)))
    for tau in (0.0, 2.0):
        for lam in _spectra(C, tau, rng):
            w = shrink_weights(lam, tau)
            _check_weights(_weights(lam, Q, C, 1, C, C, tau, 0), Q, w)                      # V[i,k] at i*C + k
            _check_weights(_weights(lam, Q.T, 1, C, C, C, tau, 0), Q, w)                    # V[i,k] at k*C + i
    # B form: row k of Bt = lambda_k v_k (what lrs_sym_eig_jacobi_f64 returns), read with strides (1, C)
    lam = 10 ** rng.uniform(-3, 0, C)
    lam[0] = 1.0
    edges = np.array([1e-12, 0.5e-12, 2e-12, -1e-14, 0.0])    # at the cut, below it, just above it, negative, zero
    lam[1:1 + min(C - 1, len(edges))] = edges[:C - 1]
    lam = rng.permutation(lam)
    Bt = lam[:, None] * Q.T
    cut = max(lam.max(), 0.0) * 1e-12
    for tau in (0.0, 0.5):
        w = np.where(lam > cut, shrink_weights(lam, tau) / np.where(lam > cut, lam, 1.0) ** 2, 0.0)
        _check_weights(_weights(lam, Bt, 1, C, C, C, tau, 1), Bt.T, w)


def test_svt_weights_zero_bordered_problem(lrs):
    """n_eig > C: the leading C x C block of a zero-bordered eigenproblem (what ops.svt_weights solves for C in [96, 136)),
    a rank-deficient Gram matrix whose zero eigenvalues meet the border's; V in both storage orders.  For tau > 0 the
    block equals the shrinkage matrix of the unbordered problem."""
    C, n = 100, 136
    rng = np.random.default_rng(100)
    Z = rng.standard_normal((400, 30)) @ rng.standard_normal((30, C))
    G = np.zeros((n, n))
    G[:C, :C] = Z.T @ Z
    lam, V = np.linalg.eigh(G)
    for tau in (0.0, 1 / 0.9, 40.0):
        w = shrink_weights(lam, tau)
        for Wd in (_weights(lam, V, n, 1, C, n, tau, 0), _weights(lam, V.T, 1, n, C, n, tau, 0)):
            _check_weights(Wd, V[:C], w)
            if tau > 0:
                ref = svt_weights_fp64(Z, tau)
                assert np.abs(Wd - ref).max() <= 1e-6 * np.abs(ref).max(), tau


def _apply(Xd, Ld, c, Wd):
    R, C = Xd.shape
    U = torch.full((R, C), float("nan"), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib().lrs_svt_apply_f32(_lib.ptr(Xd), _lib.ptr(Ld), float(c), _lib.ptr(Wd), R, C, _lib.ptr(U), _lib.stream_ptr()),
               "lrs_svt_apply_f32")
    return U.cpu().numpy()


def _check_apply(U, Z, W, chunk=1 << 16):
    """|U - Z W| <= 2 C 2^-24 (|Z| |W|) elementwise, Z W in fp64 (row chunks)."""
    C = W.shape[0]
    W64 = W.astype(np.float64)
    for r0 in range(0, Z.shape[0], chunk):
        z = Z[r0:r0 + chunk].astype(np.float64)
        err = np.abs(U[r0:r0 + chunk] - z @ W64)
        bound = 2 * C * F32_EPS * (np.abs(z) @ np.abs(W64))
        assert np.isfinite(U[r0:r0 + chunk]).all(), r0
        assert np.all(err <= bound), (r0, float((err - bound).max()))


@pytest.mark.parametrize("C", [1, 17, 64, 65, 191, 224, 256])
def test_svt_apply_vs_fp64(lrs, C):
    """lrs_svt_apply_f32: U = (X + c L) W with a NON-symmetric W (a transposed operand shows), L absent and present."""
    rng = np.random.default_rng(C)
    W = (rng.standard_normal((C, C)) / np.sqrt(C)).astype(np.float32)
    Wd = cu(W)
    for R in (1, 63, 64, 65, 262144):
        X = rng.standard_normal((R, C), dtype=np.float32)
        L = rng.standard_normal((R, C), dtype=np.float32)
        Xd, Ld = cu(X), cu(L)
        _check_apply(_apply(Xd, None, 0.0, Wd), X, W)
        _check_apply(_apply(Xd, Ld, C_OVER_MU2, Wd), _z32(X, L, C_OVER_MU2), W)


def test_svt_apply_second_launch(lrs):
    """More rows than one launch covers (65535 blocks x 64 rows): the second launch starts at row 65535*64 of X, L and U."""
    R, C = 65535 * 64 + 77, 3
    rng = np.random.default_rng(3)
    X = rng.standard_normal((R, C), dtype=np.float32)
    L = rng.standard_normal((R, C), dtype=np.float32)
    W = rng.standard_normal((C, C)).astype(np.float32)
    U = _apply(cu(X), cu(L), C_OVER_MU2, cu(W))
    _check_apply(U, _z32(X, L, C_OVER_MU2), W, chunk=1 << 20)


@pytest.mark.parametrize("R,C", [(262144, 191), (1048576, 224)])
def test_svt_device_full_size_vs_fp64(lrs, R, C, monkeypatch):
    """The whole low-rank step (ops.svt_device: Gram -> eigensolver -> weights -> recomposition) at the cfg 4 and cfg 5
    sizes on a rank-8 signal plus noise, tau at the median singular value and at one singular value exactly, against
    the fp64 restatement: rel-L2 <= 1e-5 and no row off by more than 1e-4 of its norm.  At 224 bands both eigensolvers:
    the cluster Jacobi kernel and the library eigh."""
    rng = np.random.default_rng(R + C)
    X = rng.standard_normal((R, 8), dtype=np.float32) @ rng.standard_normal((8, C), dtype=np.float32)
    X += np.float32(0.05) * rng.standard_normal((R, C), dtype=np.float32)
    L = np.float32(0.05) * rng.standard_normal((R, C), dtype=np.float32)
    Z = _z32(X, L, C_OVER_MU2)
    G, _ = _gram_ref(Z)
    lam, V = np.linalg.eigh(G)
    sigma = np.sqrt(np.maximum(lam, 0.0))                   # ascending
    Xd, Ld = cu(X), cu(L)
    # JACOBI_AUTO_C decides which eigensolver svt_device takes: 256 -> the Jacobi kernel, 0 -> the library eigh
    solvers = {"jacobi": ops.JACOBI_MAX_C} if C <= ops.JACOBI_AUTO_C else {"jacobi": ops.JACOBI_MAX_C, "library": 0}
    for tau in (float(np.median(sigma)), float(sigma[-10])):  # mid-spectrum; the 10th largest (noise level) exactly
        got = {}
        for solver, auto_c in solvers.items():
            monkeypatch.setattr(ops, "JACOBI_AUTO_C", auto_c)
            got[solver] = ops.svt_device(Xd, tau, Ld, float(C_OVER_MU2)).cpu().numpy()
        W = (V * shrink_weights(lam, tau)) @ V.T
        sq = {k: 0.0 for k in got}
        worst = {k: 0.0 for k in got}
        ref_sq = 0.0
        for r0 in range(0, R, 1 << 16):
            ref = Z[r0:r0 + (1 << 16)].astype(np.float64) @ W
            ref_sq += float((ref ** 2).sum())
            for k, U in got.items():
                u = U[r0:r0 + (1 << 16)]
                sq[k] += float(((u - ref) ** 2).sum())
                worst[k] = max(worst[k], float(per_patch_err(u.T, ref.T).max()))
        for k in got:
            assert np.sqrt(sq[k] / ref_sq) <= 1e-5, (k, tau, np.sqrt(sq[k] / ref_sq))
            assert worst[k] <= 1e-4, (k, tau, worst[k])


# ================================================================ D. X / multiplier update
ADMM_GEOMS = [(40, 23, 8, 1), (64, 41, 8, 3), (1296, 128, 36, 36), (30, 30, 5, 2), (8, 8, 8, 1), (257, 70, 8, 1), (100, 12, 6, 4),
              (9, 8, 8, 5), (50, 9, 8, 20), (33, 31, 1, 1), (41, 64, 8, 5), (20, 20, 3, 7), (8, 300, 8, 1), (3, 20, 1, 1)]


@pytest.mark.parametrize("geom", ADMM_GEOMS)
def test_admm_update_geometries_and_stripes_bit_exact(lrs, geom):
    """lrs_admm_update_f32 bit-exact against the oracle's update (coverage Weight, lambda_1 added once per covering patch)
    on every geometry class — coverage gaps, bb = 36, fewer than / not a multiple of 4 rows — and on row stripes of 1, 2,
    3, 5 and the remaining rows at offsets 1, 3, 6, 11 (not multiples of 4): each equals the same rows of the full update."""
    R, C, bb, s = geom
    rng = np.random.default_rng(R * 31 + C)
    f = lambda *shape: rng.standard_normal(shape).astype(np.float32)       # noqa: E731
    Y = np.where(rng.random((R, C)) < 0.3, 0, f(R, C)).astype(np.float32)
    MtM = np.where(rng.random((R, C)) < 0.3, 0, rng.random((R, C))).astype(np.float32)
    IM, U, l1, l2 = f(R, C) * 8, f(R, C), f(R, C), f(R, C)
    oprm = orc.Params(gamma=0.5, mu_1=0.15, mu_2=0.9, bb=bb, slidingDis=s)
    Xr, l1r, l2r = orc.admm_update(None, l1, l2, Y, MtM, IM, orc.coverage_weight(R, C, bb, s), U,
                                   orc.lambda1_summation(l1, R, C, bb, s), oprm)
    prm = lrs.Params(gamma=0.5, mu_1=0.15, mu_2=0.9, bb=bb, slidingDis=s)
    Yd, Md, IMd, Ud = cu(Y), cu(MtM), cu(IM), cu(U)
    l1d, l2d = cu(l1), cu(l2)
    Xd = lrs.admm_update(Yd, Md, IMd, Ud, l1d, l2d, prm)
    assert np.array_equal(Xd.cpu().numpy(), Xr)
    assert np.array_equal(l1d.cpu().numpy(), l1r) and np.array_equal(l2d.cpu().numpy(), l2r)
    bounds = [b for b in (0, 1, 3, 6, 11) if b < R] + [R]
    for a, b in zip(bounds[:-1], bounds[1:]):
        l1s, l2s = cu(l1[a:b]), cu(l2[a:b])
        Xs = lrs.admm_update(Yd[a:b].contiguous(), Md[a:b].contiguous(), IMd[a:b].contiguous(), Ud[a:b].contiguous(), l1s, l2s,
                             prm, rows=b - a, row_offset=a, R_total=R)
        assert torch.equal(Xs, Xd[a:b]), (a, b)
        assert torch.equal(l1s, l1d[a:b]) and torch.equal(l2s, l2d[a:b]), (a, b)
