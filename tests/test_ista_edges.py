"""The explicit ISTA path (lrs_ista_pnp_f32) column by column against fp64, on both of its engines: the split-K tcgen05
GEMMs with the 3-pass fp16 operand split (csrc/ista_tc.cu) and the fp32 FFMA GEMMs (csrc/ista_generic.cu).

A batch of patches is only right if every column is right, so every comparison here is per column:
    err_p = ||got_p - ref_p|| / max(||ref_p||, floor_p) <= 1e-4      (2e-4 with the NLM denoiser)
with floor_p = 1e-3 ||m_p . y_p|| / sqrt(a_p) for the coefficients and 1e-3 ||m_p . y_p|| for Phi_z = D alpha (the same
floor in Phi_z's units: ||D||_2 ~ sqrt(a)).  Columns with a_p <= 0, NaN or +inf must come out exactly 0, and every
output must be finite.

The shapes are chosen by the launch plan: `ista_plan` below restates make_plan / choose_splits (ista_tc.cu) and the
FFMA engine's split-K and row-tile choices (ista_generic.cu), the CPU tests pin that restatement to the library's own
host replay (lrs_debug_ista_plan, diagnostics build) and check that the shape table reaches every branch.  The GPU
tests (pytest -m gpu) then run those shapes, column-scale edges, column independence, the FFMA engine's own edges,
sentinel-guarded output and workspace tails, and the NLM denoiser at small K.  All inputs come from seeded generators.
"""
import numpy as np
import pytest
import torch

from lrs_pnp_dip_b200 import _lib
from oracle import lrs_oracle as orc
from tests.test_kernel_edges import per_patch_err, rel

F64 = np.float64
SMS = 148                     # PLAN_SMS of ista_tc.cu; the FFMA row-tile choice is replayed for the same SM count
TC_MAX_P = 65535 * 256


# ================================================================ the launch plan, restated
def _ru(x, m):
    return (x + m - 1) // m * m


def _tc_splits(Mp, Kp, ntiles):
    """choose_splits: split k only as far as one wave of CTAs allows.  Returns (S, k blocks per split, last split's)."""
    nkb = Kp // 64
    s = min(max(SMS // (Mp // 128 * ntiles), 1), nkb)
    kb = -(-nkb // s)
    S = -(-nkb // kb)
    return S, kb, nkb - (S - 1) * kb


def _ffma_splits(M, N, Kd):
    sp = -(-592 // (-(-M // 32) * -(-N // 48)))
    return max(1, min(sp, Kd // 128, 8))


def _ffma_row_tile(M, N, splits):
    return 32 if splits > 1 or -(-M // 64) * -(-N // 48) < 2 * SMS else 64


def ista_plan(n, K, P):
    """The 15 values of lrs_debug_ista_plan (include/lrs_pnp_diag.h) for an [n, K] dictionary and P patches."""
    out = [0] * 15
    if n >= 128 and K >= 128 and 8 <= P <= TC_MAX_P:
        Np = _ru(P, 16)
        nt = -(-Np // 256)
        stage = 2 * (128 * 64 * 2) + 2 * min(Np, 256) * 64 * 2             # A pieces + B pieces of one stage, bytes
        S1, kb1, l1 = _tc_splits(_ru(n, 128), _ru(K, 64), nt)
        S2, kb2, l2 = _tc_splits(_ru(K, 128), _ru(n, 64), nt)
        out[:11] = [1, Np, nt, Np - (nt - 1) * 256, 3 if 3 * stage <= 220 * 1024 else 2, S1, kb1, S2, kb2, l1, l2]
    s1, s2 = _ffma_splits(n, P, K), _ffma_splits(K, P, n)
    out[11:] = [s1, s2, _ffma_row_tile(n, P, s1), _ffma_row_tile(K, P, s2)]
    return out


# (n, K, P) of the tensor-core engine and the plan branch each one reaches
TC_SHAPES = [(128, 128, 8),          # smallest tensor-core shape; S = 2
             (129, 130, 9),          # padding in every dimension; P % 4 = 1
             (300, 200, 160),        # last shape with 3 stages
             (300, 200, 161),        # first shape with 2 stages
             (640, 4000, 8),         # S1 = 21, last split 3 of 3: the 8-wide reduce4 loop runs
             (257, 1000, 1795),      # 8 patch tiles, last one 16 wide; S1 = 6 with a short last split; P % 4 = 3
             (1296, 2592, 144),      # the bundled cfg 1 shape: S1 = 11, S2 = 7
             (1296, 2592, 2880),     # the 20-cube cfg 1 batch: 12 tiles, S = 1
             (200, 500, 10241)]      # 41 tiles, last one 16 wide
# FFMA-engine shapes (the shape alone picks that engine)
FFMA_SHAPES = [(64, 1024, 20),       # 8 k-splits on the residual GEMM
               (64, 100, 14400),     # 64-row tiles
               (100, 130, 17), (36, 80, 33),     # ragged
               (127, 4000, 50),      # n just below the tensor-core limit
               (128, 127, 50),       # K just below it
               (128, 128, 7)]        # P just below it: the engine switch


def _diag_plan(L, n, K, P):
    out = np.zeros(15, dtype=np.int64)
    assert L.lrs_debug_ista_plan(n, K, P, out.ctypes.data) == 0, L.lrs_last_error()
    return out.tolist()


# ================================================================ CPU: plan replay and branch coverage
def test_plan_restatement_matches_host_replay():
    L = _lib.diag_lib()
    rng = np.random.default_rng(0)
    shapes = list(TC_SHAPES) + list(FFMA_SHAPES) + [(128, 128, TC_MAX_P), (128, 128, TC_MAX_P + 1)]
    for _ in range(400):
        n, K = (int(np.exp(rng.uniform(0, np.log(5000)))) for _ in range(2))
        shapes.append((n, K, int(np.exp(rng.uniform(0, np.log(40000))))))
    for s in shapes:
        assert _diag_plan(L, *s) == ista_plan(*s), s
    assert L.lrs_debug_ista_plan(0, 5, 5, np.zeros(15, np.int64).ctypes.data) != 0


def test_shape_tables_reach_every_plan_branch():
    pl = {s: ista_plan(*s) for s in TC_SHAPES}
    assert all(p[0] == 1 for p in pl.values())
    assert {p[4] for p in pl.values()} == {2, 3}                                     # stage counts
    assert pl[(300, 200, 160)][4] == 3 and pl[(300, 200, 161)][4] == 2              # the stage switch itself
    assert any(p[2] == 1 for p in pl.values()) and any(p[2] > 1 and p[3] == 16 for p in pl.values())
    S = [x for p in pl.values() for x in (p[5], p[7])]
    assert 1 in S and any(2 <= x <= 8 for x in S) and any(x >= 9 for x in S)        # reduce4 without / with its 8-wide loop
    assert any(p[9] < p[6] or p[10] < p[8] for p in pl.values())                    # a short last split
    assert {s[2] % 4 for s in TC_SHAPES} >= {0, 1, 3}                               # vector and scalar epilogues
    assert pl[(640, 4000, 8)][5:7] + [pl[(640, 4000, 8)][9]] == [21, 3, 3]
    assert pl[(1296, 2592, 144)][5] == 11 and pl[(1296, 2592, 144)][7] == 7
    assert pl[(1296, 2592, 2880)][2] == 12 and pl[(1296, 2592, 2880)][5] == pl[(1296, 2592, 2880)][7] == 1
    assert pl[(200, 500, 10241)][2:4] == [41, 16] and pl[(257, 1000, 1795)][2:4] == [8, 16]
    ff = {s: ista_plan(*s) for s in FFMA_SHAPES}
    assert all(p[0] == 0 for p in ff.values())
    assert ff[(64, 1024, 20)][11] == 8
    assert ff[(64, 100, 14400)][13:] == [64, 64]
    assert any(p[13] == 32 and p[11] == 1 for p in ff.values())                     # 32-row tiles without split-K


def test_engine_switch_sits_at_the_tensor_core_limits():
    for s, tc in [((128, 128, 8), 1), ((127, 128, 8), 0), ((128, 127, 8), 0), ((128, 128, 7), 0),
                  ((128, 128, TC_MAX_P), 1), ((128, 128, TC_MAX_P + 1), 0)]:
        assert ista_plan(*s)[0] == tc, s


# ================================================================ fp64 references (CPU)
def nlm_columns_fp64(G, h):
    """orc.nlm_column(G[:, p], 3, 3, h[p]) for every column p at once (same padding, taps and weights)."""
    G = np.asarray(G, F64)
    K, P = G.shape
    kw = orc.nlm_kernel_rowsums(3)
    Gp = np.pad(G, ((3, 3), (0, 0)), mode="symmetric")
    win = np.stack([Gp[u:u + K] for u in range(7)])                  # [7, K, P]: window of row i, tap u
    h2 = np.asarray(h, F64) ** 2
    wmax, avg, sw = np.zeros((K, P)), np.zeros((K, P)), np.zeros((K, P))
    for dr in (-3, -2, -1, 1, 2, 3):
        i = np.arange(K)
        ok = (i + dr >= 0) & (i + dr < K)
        r = np.clip(i + dr, 0, K - 1)
        d = np.einsum("u,ukp->kp", kw, (win - win[:, r]) ** 2)
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            w = np.where(h2 > 0, np.exp(-d / np.where(h2 > 0, h2, 1.0)), (d == 0).astype(F64))
        w = np.where(ok[:, None], w, 0.0)
        wmax = np.maximum(wmax, w)
        sw += w
        avg += w * G[r]
    avg += wmax * G
    sw += wmax
    return np.where(sw > 0, avg / np.where(sw > 0, sw, 1.0), G)


def ista_fp64(Y, mask, D, a, lam, Nit, denoiser="soft", h_scale=0.1):
    """fp64 column-batched ISTA on fp64 copies of the fp32 inputs: soft (orc.ista_soft_batched), identity (the same
    loop without the threshold) or NLM (the identity step, then NLmeansfilter(g, 3, 3, h_scale T) on each column)."""
    D = np.asarray(D, F64)
    a = np.asarray(a, F64)
    Y = np.where(mask, np.asarray(Y, F64), 0.0)                # unobserved entries do not enter the masked residual
    ok = (a > 0) & np.isfinite(a)
    if denoiser == "soft":
        A = orc.ista_soft_batched(Y, mask, D, np.where(ok, a, 0.0), lam, Nit)
    else:
        inv_a = np.where(ok, 1.0 / np.where(ok, a, 1.0), 0.0)
        T = lam * inv_a / 2
        m = mask.astype(F64)
        A = np.zeros((D.shape[1], Y.shape[1]))
        for _ in range(Nit):
            A = A + (D.T @ (m * (Y - D @ A))) * inv_a
            if denoiser == "nlm":
                A = nlm_columns_fp64(A, h_scale * T)
    A[:, ~ok] = 0.0
    return A


def column_errors(got, ref, floor):
    """per_patch_err with a per-column floor; a column whose reference and floor are both 0 must be exactly 0."""
    got, ref = np.asarray(got, F64), np.asarray(ref, F64)
    num = np.linalg.norm(got - ref, axis=0)
    den = np.maximum(np.linalg.norm(ref, axis=0), floor)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(den > 0, num / np.where(den > 0, den, 1.0), np.where(num == 0, 0.0, np.inf))


def test_nlm_reference_is_the_oracle_filter():
    rng = np.random.default_rng(5)
    for K in list(range(1, 17)) + [40]:
        G = rng.standard_normal((K, 6))
        G[:, 1] = np.round(G[:, 1])                             # repeated values: zero distances
        h = np.array([0.05, 0.5, 2.0, 0.0, 1e-3, 10.0])
        want = np.stack([orc.nlm_column(G[:, p], 3, 3, h[p]) for p in range(6)], axis=1)
        assert np.allclose(nlm_columns_fp64(G, h), want, rtol=1e-13, atol=1e-15), K


def test_column_errors_criterion():
    ref = np.array([[1.0, 0.0, 0.0], [0.0, 0.0, 0.0]])
    got = np.array([[1.0 + 1e-6, 1e-9, 0.0], [0.0, 0.0, 0.0]])
    e = column_errors(got, ref, np.array([0.0, 1e-3, 0.0]))
    assert np.allclose(e, [1e-6, 1e-6, 0.0])
    assert np.isinf(column_errors(got[:, 1:2], ref[:, 1:2], np.zeros(1)))[0]
    assert np.allclose(per_patch_err(got, ref)[0], 1e-6)


# ================================================================ device plumbing
@pytest.fixture(scope="module")
def lrs():
    import lrs_pnp_dip_b200 as m

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m._lib.lib()
    return m


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def run(lrs, monkeypatch, engine, Y, bc, D, a, lam, Nit, denoiser="soft", h_scale=0.1):
    """lrs_ista_pnp_f32 on host arrays; engine 'tc' / 'simt' sets LRS_ISTA_ENGINE, 'auto' leaves it unset."""
    if engine == "auto":
        monkeypatch.delenv("LRS_ISTA_ENGINE", raising=False)
    else:
        monkeypatch.setenv("LRS_ISTA_ENGINE", engine)
    c, p = lrs.ista_batched(cu(Y), cu(bc), cu(D), cu(a), lam, Nit, want_coefs=True, denoiser=denoiser, h_scale=h_scale)
    torch.cuda.synchronize()
    return c.cpu().numpy(), p.cpu().numpy()


def make_problem(n, K, P, seed, atom_norms=None):
    """Gaussian D with unit-scale atoms, Gaussian data, three mask patterns and one all-missing column (column 1)."""
    rng = np.random.default_rng(seed)
    D = rng.standard_normal((n, K)) / np.sqrt(n)
    if atom_norms is not None:
        D = D / np.linalg.norm(D, axis=0) * atom_norms
    D = D.astype(np.float32)
    Y = rng.standard_normal((n, P)).astype(np.float32)
    mask = (rng.random((n, 3)) < 0.7)[:, rng.integers(0, 3, P)]
    mask[:, 1 % P] = False
    return D, Y, mask


def bc_of(mask):
    return np.where(mask, np.float32(1.5), np.float32(0)).astype(np.float32)


def sample_columns(P, seed, count=300):
    """All columns of small problems; else ~count columns: the first and last of every 256-wide patch tile plus random."""
    if P <= count:
        return np.arange(P)
    edges = np.r_[np.arange(0, P, 256), np.minimum(np.arange(255, P + 255, 256), P - 1), [1]]
    rng = np.random.default_rng(seed)
    return np.unique(np.r_[edges, rng.choice(P, max(count - len(edges), 0), replace=False)])


def check_against_fp64(got, Y, mask, D, a, lam, Nit, denoiser, cols, what, h_scale=0.1, bound=None):
    """The per-column criterion of the module docstring on the columns `cols` (a_p <= 0, NaN, +inf: exactly 0 on all)."""
    coefs, phi = got
    bound = bound or (2e-4 if denoiser == "nlm" else 1e-4)
    assert np.isfinite(coefs).all() and np.isfinite(phi).all(), what
    a = np.asarray(a, np.float32)
    dead = ~((a > 0) & np.isfinite(a))
    assert not coefs[:, dead].any() and not phi[:, dead].any(), (what, np.flatnonzero(dead))
    cols = np.asarray([c for c in cols if not dead[c]])
    ref = ista_fp64(Y[:, cols], mask[:, cols], D, a[cols], lam, Nit, denoiser, h_scale)
    my = np.linalg.norm(np.where(mask[:, cols], Y[:, cols].astype(F64), 0.0), axis=0)
    ec = column_errors(coefs[:, cols], ref, 1e-3 * my / np.sqrt(a[cols].astype(F64)))
    ep = column_errors(phi[:, cols], np.asarray(D, F64) @ ref, 1e-3 * my)
    for name, e in (("coefs", ec), ("phi", ep)):
        bad = np.flatnonzero(~(e <= bound))
        assert bad.size == 0, f"{what} {name}: {bad.size} columns above {bound:g}, worst " \
                              f"{[(int(cols[i]), float(e[i])) for i in bad[np.argsort(-e[bad])][:8]]}"
    return ec, ep


# ================================================================ 1. plan-edge shapes, both engines
@pytest.mark.gpu
@pytest.mark.parametrize("shape", TC_SHAPES, ids=[f"{n}x{K}x{P}" for n, K, P in TC_SHAPES])
def test_tc_plan_edges_per_column(lrs, shape, monkeypatch):
    n, K, P = shape
    big = n * K * P > 5e8
    Nit, lam = (12 if big else 30), 0.05
    D, Y, mask = make_problem(n, K, P, seed=n + K + P)
    cols = sample_columns(P, seed=P)
    bc = bc_of(mask)
    for step in ("spectral", "frob4"):
        a = orc.step_constants_batched(D.astype(F64), mask, step).astype(np.float32)
        assert a[1] == 0
        for denoiser in ("soft", "identity"):
            for engine in ("tc", "simt"):
                got = run(lrs, monkeypatch, engine, Y, bc, D, a, lam, Nit, denoiser)
                check_against_fp64(got, Y, mask, D, a, lam, Nit, denoiser, cols, (engine, step, denoiser))


# ================================================================ 2. column-scale edges inside one call
def _scale_edge_problem(n=256, K=192, P=40, atom_norms=None):
    D, Y, mask = make_problem(n, K, P, seed=77, atom_norms=atom_norms)
    mask[:, 1] = mask[:, 0]                                   # column 1 is not all-missing here
    Y = Y.astype(F64)
    cases = {}
    for j, k in zip((2, 3, 4), (12, 16, 20)):                 # unobserved entries 2^k times the observed ones
        Y[~mask[:, j], j] *= 2.0 ** k
        cases[f"unobserved x2^{k}"] = j
    Y[mask[:, 5], 5] = 0.0                                    # observed all zero, unobserved nonzero
    cases["observed zero"] = 5
    for j in (6, 15):                                         # observed entries all fp32 subnormals
        Y[:, j] = np.where(mask[:, j], np.sign(Y[:, j]) * 1e-40 * (1 + np.abs(Y[:, j])), Y[:, j])
    Y[~mask[:, 6], 6] = 0.0                                   # ... with nothing else in the column
    cases["observed subnormal"] = 6
    cases["observed subnormal, unobserved normal"] = 15
    Y[:, 7] *= 1e-30
    Y[:, 8] *= 1e30
    Y[:, 9] *= 2.0 ** 40
    Y[:, 10] *= 2.0 ** -40
    cases.update({"1e-30": 7, "1e30": 8, "2^40": 9, "2^-40": 10})
    Y = Y.astype(np.float32)
    assert 0 < np.abs(Y[mask[:, 6], 6]).max() < 1.17549435e-38 and 0 < np.abs(Y[mask[:, 15], 15]).max() < 1.17549435e-38
    a = orc.step_constants_batched(D.astype(F64), mask, "spectral").astype(np.float32)
    a[11], a[12], a[13], a[14] = 0.0, -1.0, np.nan, np.inf    # must all give exactly 0
    return D, Y, mask, a, cases


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["tc", "simt"])
def test_column_scale_edges_per_column(lrs, engine, monkeypatch):
    D, Y, mask, a, cases = _scale_edge_problem()
    lam, Nit = 0.01, 30
    coefs, phi = run(lrs, monkeypatch, engine, Y, bc_of(mask), D, a, lam, Nit)
    subs = [cases["observed subnormal"], cases["observed subnormal, unobserved normal"]]
    ref_sub = ista_fp64(Y[:, subs], mask[:, subs], D, a[subs], lam, Nit)
    assert np.isfinite(coefs[:, subs]).all() and np.isfinite(phi[:, subs]).all()
    assert np.abs(coefs[:, subs] - ref_sub).max() <= 1e-37 and np.abs(phi[:, subs] - D.astype(F64) @ ref_sub).max() <= 1e-37
    assert not coefs[:, cases["observed zero"]].any() and not phi[:, cases["observed zero"]].any()
    cols = [p for p in range(Y.shape[1]) if p not in subs]
    ec, ep = check_against_fp64((coefs, phi), Y, mask, D, a, lam, Nit, "soft", cols, engine)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["tc", "simt"])
def test_wide_atom_norms_per_column(lrs, engine, monkeypatch):
    """Atom norms from 2^-8 to 1: the fp16 pieces of the small atoms sit far below D's largest entry."""
    n, K, P = 256, 192, 40
    norms = 2.0 ** -np.random.default_rng(3).uniform(0, 8, K)
    norms[:2] = [1.0, 2.0 ** -8]
    D, Y, mask = make_problem(n, K, P, seed=78, atom_norms=norms)
    a = orc.step_constants_batched(D.astype(F64), mask, "spectral").astype(np.float32)
    for lam, denoiser in ((0.01, "soft"), (0.0, "identity")):
        got = run(lrs, monkeypatch, engine, Y, bc_of(mask), D, a, lam, 30, denoiser)
        check_against_fp64(got, Y, mask, D, a, lam, 30, denoiser, range(P), (engine, denoiser))


# ================================================================ 3. column independence and determinism
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["tc", "simt"])
def test_columns_are_independent_and_deterministic(lrs, engine, monkeypatch):
    """Same call twice: bit-identical.  Every other column replaced by random data, huge values, NaN or zeros (n, K, P
    and D fixed, so the launch plan is the same): the chosen columns stay bit-identical."""
    n, K, P = 257, 1000, 1795
    D, Y, mask = make_problem(n, K, P, seed=9)
    a = orc.step_constants_batched(D.astype(F64), mask, "frob4").astype(np.float32)
    bc = bc_of(mask)
    keep = np.array([0, 2, 3, 255, 256, 511, 1279, 1280, 1790, 1791, 1792, 1793, 1794])   # last tile = 1792..1794
    others = np.setdiff1d(np.arange(P), keep)
    base = run(lrs, monkeypatch, engine, Y, bc, D, a, 0.05, 12)
    again = run(lrs, monkeypatch, engine, Y, bc, D, a, 0.05, 12)
    assert np.array_equal(base[0], again[0]) and np.array_equal(base[1], again[1])
    rng = np.random.default_rng(10)
    for kind in ("random", "huge", "nan", "zero"):
        Y2, bc2, a2 = Y.copy(), bc.copy(), a.copy()
        if kind == "random":
            Y2[:, others] = rng.standard_normal((n, others.size)) * 10.0 ** rng.uniform(-6, 6, others.size)
            bc2[:, others] = bc_of(rng.random((n, others.size)) < 0.5)
            a2[others] = rng.uniform(0.1, 50.0, others.size)
        elif kind == "huge":
            Y2[:, others] = 3e38
            a2[others] = 1e-30
        elif kind == "nan":
            Y2[:, others] = np.nan
            a2[others] = np.nan
        else:
            Y2[:, others] = 0.0
            bc2[:, others] = 0.0
            a2[others] = 0.0
        got = run(lrs, monkeypatch, engine, Y2, bc2, D, a2, 0.05, 12)
        for g, b, name in ((got[0], base[0], "coefs"), (got[1], base[1], "phi")):
            diff = [int(p) for p in keep if not np.array_equal(g[:, p], b[:, p])]
            assert not diff, (kind, name, diff)


# ================================================================ 4. FFMA-engine edges
@pytest.mark.gpu
@pytest.mark.parametrize("shape", FFMA_SHAPES, ids=[f"{n}x{K}x{P}" for n, K, P in FFMA_SHAPES])
def test_ffma_edges_per_column(lrs, shape, monkeypatch):
    n, K, P = shape
    D, Y, mask = make_problem(n, K, P, seed=n * K + P)
    cols = sample_columns(P, seed=P)
    bc = bc_of(mask)
    nlm_cols = cols[:6]
    for step in ("spectral", "frob4"):
        a = orc.step_constants_batched(D.astype(F64), mask, step).astype(np.float32)
        # NLM with the spectral step only: with frob4's larger a, h = 40 lambda / (2a) puts d / h^2 in the hundreds, where
        # the weights exp(-d / h^2) amplify the fp32 rounding of their input by that factor (no fp32 pipeline meets 2e-4)
        for denoiser in ("soft", "identity", "nlm") if step == "spectral" else ("soft", "identity"):
            h = 40.0 if denoiser == "nlm" else 0.1
            got = run(lrs, monkeypatch, "auto", Y, bc, D, a, 0.05, 30, denoiser, h_scale=h)
            check_against_fp64(got, Y, mask, D, a, 0.05, 30, denoiser, nlm_cols if denoiser == "nlm" else cols,
                               (step, denoiser), h_scale=h)


# ================================================================ 5. writes stay in bounds
TAIL = 64 * 1024
BOUNDS_CASES = [(128, 128, 8, "auto", "soft"), (129, 130, 9, "auto", "nlm"), (300, 200, 161, "auto", "identity"),
                (640, 4000, 8, "auto", "soft"), (257, 1000, 1795, "auto", "nlm"), (200, 500, 10241, "auto", "soft"),
                (257, 1000, 1795, "simt", "soft"), (64, 1024, 20, "auto", "soft"), (64, 100, 14400, "auto", "nlm"),
                (100, 130, 17, "auto", "identity"), (127, 4000, 50, "auto", "soft"), (128, 128, 7, "auto", "nlm")]


@pytest.mark.gpu
@pytest.mark.parametrize("n,K,P,engine,denoiser", BOUNDS_CASES)
def test_writes_stay_inside_outputs_and_workspace(lrs, n, K, P, engine, denoiser, monkeypatch):
    """Workspace, coefs and Phi_z each get a 64 KB tail filled with a sentinel pattern; the call must leave every tail
    unchanged (NLM's G buffer is the last region of the tensor-core workspace)."""
    if engine == "auto":
        monkeypatch.delenv("LRS_ISTA_ENGINE", raising=False)
    else:
        monkeypatch.setenv("LRS_ISTA_ENGINE", engine)
    D, Y, mask = make_problem(n, K, P, seed=11)
    Yd, bcd, Dd = cu(Y), cu(bc_of(mask)), cu(D)
    a = lrs.step_constants(bcd, Dd, "frob4")
    L = _lib.lib()
    need = L.lrs_ista_workspace_bytes(n, K, P)
    bufs = {name: torch.full((size + TAIL,), fill, dtype=torch.uint8, device="cuda")
            for name, size, fill in (("ws", need, 0xA5), ("coefs", K * P * 4, 0x5A), ("phi", n * P * 4, 0xC3))}
    rc = L.lrs_ista_pnp_f32(_lib.ptr(Yd), _lib.ptr(bcd), _lib.ptr(Dd), _lib.ptr(a), 0.05, 3, n, K, P,
                            _lib.DENOISERS[denoiser], 0.1, _lib.ptr(bufs["coefs"]), _lib.ptr(bufs["phi"]),
                            _lib.ptr(bufs["ws"]), need, _lib.stream_ptr())
    _lib.check(rc, "lrs_ista_pnp_f32")
    torch.cuda.synchronize()
    for name, fill in (("ws", 0xA5), ("coefs", 0x5A), ("phi", 0xC3)):
        tail = bufs[name][-TAIL:]
        changed = torch.nonzero(tail != fill).flatten()
        assert changed.numel() == 0, (name, int(changed[0]), changed.numel())
    coefs = bufs["coefs"][:K * P * 4].view(torch.float32).reshape(K, P)
    assert bool(torch.isfinite(coefs).all())


# ================================================================ 6. NLM at small K
@pytest.mark.gpu
@pytest.mark.parametrize("K", range(1, 17))
def test_nlm_small_K_vs_oracle(lrs, K):
    rng = np.random.default_rng(100 + K)
    n, Nit = 24, 12
    H = (rng.standard_normal((n, K)) / np.sqrt(n)).astype(np.float32)
    y = (H @ rng.standard_normal((K, 1)) + 0.05 * rng.standard_normal((n, 1))).astype(np.float32)
    a = orc.step_constant(H.astype(F64), "spectral")
    for h_scale in (0.1, 40.0):
        ref = orc.pnp_ista_nlm(y, H, 0.1, Nit, a, h_scale=h_scale)
        x = lrs.ista(torch.tensor(y), torch.tensor(H), 0.1, 0, Nit, denoiser="nlm", h_scale=h_scale).numpy()
        assert per_patch_err(x, ref, 1e-3 * np.linalg.norm(y) / np.sqrt(a))[0] < 2e-4, h_scale
    # one filter application: H = I, so that g = v and x1 = NLM(v) with h = h_scale * lambda / 2
    v = np.r_[np.zeros(2), np.ones(3), np.linspace(0, 1, 5), rng.standard_normal(6) * 0.1][:K].astype(np.float32)
    v[-1] += 0.25
    for h_scale in (0.5, 40.0):
        x1 = lrs.ista(torch.tensor(v.reshape(-1, 1)), torch.tensor(np.eye(K, dtype=np.float32)), 0.1, 0, 1, denoiser="nlm",
                      h_scale=h_scale).numpy().ravel()
        assert rel(x1, orc.nlm_column(v, 3, 3, h_scale * 0.05)) < 1e-5, h_scale
