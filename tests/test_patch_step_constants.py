"""step='spectral_patch': the reference's spectral step constant np.linalg.norm(H, 2)**2 (main_LRS_PnP.py:134) for every
patch of ANY observation mask, from the patch's own 64-bit validity word.  The validity words and the per-pattern values
are checked against fp64 NumPy, the on-device merging of equal words against the unmerged kernel, and the sparse step
and the solver against the oracle.  GPU tests run on the B200 box (pytest -m gpu); the last three tests need no GPU.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import lrs_pnp_dip_b200 as lrs
from lrs_pnp_dip_b200 import _lib, ops, synth
from oracle import lrs_oracle as orc
from tests.test_kernel_edges import FUSED_GEOMS, TABLE_DICTIONARIES, rel, row_patterns

HERE = os.path.dirname(os.path.abspath(__file__))
gpu = pytest.mark.gpu


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


# ---------------------------------------------------------------- fp64 references (CPU)
def pack_words(mask):
    """mask [n, P] bool -> int64 view of the uint64 words, bit k = element k."""
    w = np.zeros(mask.shape[1], np.uint64)
    for k in range(mask.shape[0]):
        w |= mask[k].astype(np.uint64) << np.uint64(k)
    return w.view(np.int64)


def unpack_words(words, n=64):
    w = np.asarray(words).view(np.uint64)
    return ((w[None, :] >> np.arange(n, dtype=np.uint64)[:, None]) & np.uint64(1)).astype(bool)   # [n, P]


def spectral_fp64(D, mask, chunk=2048):
    """lambda_max(D_S D_S^T) = ||D_S||_2^2 for every column of mask [n, P], fp64 (zero-bordered Gram matrices)."""
    G = D.astype(np.float64) @ D.astype(np.float64).T
    out = np.empty(mask.shape[1])
    for p0 in range(0, mask.shape[1], chunk):
        m = mask[:, p0:p0 + chunk].T
        A = G[None] * (m[:, :, None] & m[:, None, :])
        out[p0:p0 + chunk] = np.maximum(np.linalg.eigvalsh(A)[:, -1], 0.0)
    return out


def frob4_fp64(D, mask):
    return 4.0 * ((D.astype(np.float64) ** 2).sum(1) @ mask.astype(np.float64))


# ---------------------------------------------------------------- device calls
def words_dev(Y, bb, s, p0=0, p1=None):
    Yd = cu(Y)
    R, C = Y.shape
    p1 = ops.patch_count(R, C, bb, s) if p1 is None else p1
    out = torch.full((p1 - p0,), 0x5A5A5A5A, dtype=torch.int64, device="cuda")
    _lib.check(_lib.lib().lrs_patch_mask_words_u64(_lib.ptr(Yd), R, C, bb, s, p0, p1, _lib.ptr(out), _lib.stream_ptr()),
               "lrs_patch_mask_words_u64")
    return out.cpu().numpy()


def patterns_dev(D, words, step="spectral", count=None):
    Dd = cu(D)
    n, K = D.shape
    w = cu(np.asarray(words, np.int64))
    a = torch.full((len(w),), float("nan"), dtype=torch.float32, device="cuda")
    L = _lib.lib()
    nb = L.lrs_spectral_patterns_workspace_bytes(n)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    cnt = None if count is None else torch.tensor([count], dtype=torch.int64, device="cuda")
    mode = {"spectral": _lib.STEP_SPECTRAL, "frob4": _lib.STEP_FROB4}[step]
    _lib.check(L.lrs_spectral_patterns_f32(_lib.ptr(Dd), n, K, _lib.ptr(w), len(w), _lib.ptr(cnt), mode, _lib.ptr(a),
                                           _lib.ptr(ws), nb, _lib.stream_ptr()), "lrs_spectral_patterns_f32")
    return a.cpu().numpy()


def masked_matrix(rng, R, C, keep=0.6, signed_zero_nan=False):
    """Per-element observed matrix: missing entries are 0.0 (some -0.0), a few observed entries NaN."""
    Y = (rng.standard_normal((R, C)) * 0.3 + 0.5).astype(np.float32)
    Y[Y == 0] = 1e-12
    miss = rng.random((R, C)) >= keep
    Y[miss] = 0.0
    if signed_zero_nan:
        Y[miss & (rng.random((R, C)) < 0.5)] = -0.0
        Y[~miss & (rng.random((R, C)) < 0.05)] = np.nan
    return Y


# ================================================================ 1. validity words
WORD_CASES = [(8,) + g for g in FUSED_GEOMS.values()] + \
             [(4, 37, 19, 3), (4, 50, 23, 1), (5, 64, 41, 4), (5, 33, 12, 7), (8, 300, 40, 2), (4, 9, 9, 1)]


@gpu
@pytest.mark.parametrize("bb,R,C,s", WORD_CASES, ids=[f"bb{c[0]}-{c[1]}x{c[2]}-s{c[3]}" for c in WORD_CASES])
def test_mask_words_match_oracle(bb, R, C, s):
    """Every patch's word equals the oracle's validity mask (get_image_block of Y_observed != 0) packed bit k = element
    k; -0.0 counts as missing and NaN as observed.  Sub-ranges that start and end off the 256-row-start tiles give the
    same words as the whole launch."""
    rng = np.random.default_rng(R * 31 + C * 7 + s + bb)
    Y = masked_matrix(rng, R, C, signed_zero_nan=True)
    ref = pack_words(orc.patch_masks(orc.get_image_block(Y, bb, s)[0]))
    whole = words_dev(Y, bb, s)
    assert np.array_equal(whole, ref)
    P = len(ref)
    ranges = {(0, 1), (P - 1, P), (min(1, P - 1), P), (P // 3, P // 3 + 1)}
    ranges |= {(p0, min(P, p0 + 300)) for p0 in (255, 257, 511) if p0 < P}
    for _ in range(4):
        p0 = int(rng.integers(0, P))
        ranges.add((p0, int(rng.integers(p0 + 1, P + 1))))
    for p0, p1 in sorted(ranges):
        assert np.array_equal(words_dev(Y, bb, s, p0, p1), ref[p0:p1]), (p0, p1)


# ================================================================ 2. per-pattern values
def _check_close(got, ref, tol=2e-6):
    got = np.asarray(got, np.float64)
    bad = np.flatnonzero(~(np.abs(got - ref) <= tol * np.abs(ref)))
    assert bad.size == 0, [(int(i), float(got[i]), float(ref[i])) for i in bad[:8]]


@gpu
@pytest.mark.parametrize("name", list(TABLE_DICTIONARIES))
def test_pattern_values_every_dictionary(name):
    """Single elements (= ||D_i||^2), the full pattern (= ||D||_2^2), the empty pattern (exactly 0), all 256
    band-replicated patterns (equal, bit for bit, to the row-pattern table) and random patterns at keep 0.5 / 0.9:
    spectral and frob4 within 2e-6 of fp64."""
    D = TABLE_DICTIONARIES[name]()
    rng = np.random.default_rng(1)
    k_rows = np.arange(64) % 8
    single = np.eye(64, dtype=bool)
    full = np.ones((64, 1), bool)
    rows = ((np.arange(256)[None, :] >> k_rows[:, None]) & 1).astype(bool)
    rand = np.concatenate([rng.random((64, 500)) < keep for keep in (0.5, 0.9)], axis=1)
    mask = np.concatenate([single, full, rows, rand], axis=1)
    words = pack_words(mask)
    a = patterns_dev(D, words)
    ref = spectral_fp64(D, mask)
    Dd = D.astype(np.float64)
    assert a[65] == 0.0                                            # row pattern 0: the empty pattern
    _check_close(a[:64], (Dd ** 2).sum(1))
    _check_close(a[64:65], [np.linalg.norm(Dd, 2) ** 2])
    nz = ref > 0
    _check_close(a[nz], ref[nz])
    assert np.all(a[~nz] == 0.0)
    assert np.array_equal(a[65:65 + 256], ops._row_pattern_table(cu(D), 8, "spectral").cpu().numpy())
    f = patterns_dev(D, words, "frob4")
    fref = frob4_fp64(D, mask)
    _check_close(f[fref > 0], fref[fref > 0])
    assert f[65] == 0.0 and np.all(f[fref == 0] == 0.0)


@gpu
def test_pattern_values_random_keep_rates_and_repeatable():
    """About 20 000 random patterns at keep 0.1 / 0.5 / 0.9 / 1.0 on the Gaussian K = 256 dictionary within 2e-6 of fp64;
    equal words in different positions give the same bits, three calls give the same bits, and a device count limits
    the launch to the leading words."""
    D = TABLE_DICTIONARIES["gaussian-K256"]()
    rng = np.random.default_rng(2)
    mask = np.concatenate([rng.random((64, 5000)) < keep for keep in (0.1, 0.5, 0.9, 1.0)], axis=1)
    words = pack_words(mask)
    words = np.concatenate([words, words[::-1][:3000]])               # duplicates, sharing warps with other patterns
    mask = unpack_words(words)
    a = patterns_dev(D, words)
    ref = spectral_fp64(D, mask)
    nz = ref > 0
    _check_close(a[nz], ref[nz])
    assert np.all(a[~nz] == 0.0)
    assert np.array_equal(a[20000:], a[:20000][::-1][:3000])
    for _ in range(2):
        assert np.array_equal(patterns_dev(D, words), a)
    part = patterns_dev(D, words, count=777)
    assert np.array_equal(part[:777], a[:777]) and np.isnan(part[777:]).all()
    f = patterns_dev(D, words, "frob4")
    fref = frob4_fp64(D, mask)
    _check_close(f[fref > 0], fref[fref > 0])


# ================================================================ 3. merging equal words
@gpu
@pytest.mark.parametrize("kind", ["few-patterns", "all-distinct"])
def test_merged_constants_equal_unmerged_kernel(kind, monkeypatch):
    """ops.patch_step_constants (sort, run starts, cumsum, scatter of the representatives, gather back) is bit-identical
    to the pattern kernel run on every patch's word, whole and on a sub-range, also when the merge runs in many passes."""
    rng = np.random.default_rng(3)
    R, C, s = 600, 40, 1
    if kind == "few-patterns":
        Y = np.repeat((rng.random(R) < 0.6)[:, None], C, axis=1) * np.float32(0.5)
    else:
        Y = masked_matrix(rng, R, C, keep=0.5)
    D = TABLE_DICTIONARIES["gaussian-K128"]()
    words = words_dev(Y, 8, s)
    assert (len(np.unique(words)) <= 256) == (kind == "few-patterns")
    if kind == "all-distinct":
        assert len(np.unique(words)) > 0.99 * len(words)
    ref = patterns_dev(D, words)
    Yd, Dd = cu(Y), cu(D)
    a = ops.patch_step_constants(Yd, Dd, 8, s).cpu().numpy()
    assert np.array_equal(a, ref)
    P = len(words)
    assert np.array_equal(ops.patch_step_constants(Yd, Dd, 8, s, p_begin=1000, p_end=P - 77).cpu().numpy(), ref[1000:P - 77])
    monkeypatch.setattr(ops, "PATCH_CONSTANTS_CHUNK", 4099)
    assert np.array_equal(ops.patch_step_constants(Yd, Dd, 8, s).cpu().numpy(), ref)
    fr = ops.patch_step_constants(Y, D, 8, s, step="frob4")                     # host inputs: host result
    assert isinstance(fr, np.ndarray) and np.array_equal(fr, patterns_dev(D, words, "frob4"))


# ================================================================ 4. sparse step
MU1, LAM, NIT = 0.15, 0.1, 25


def _cube_inputs(kind, H=8, W=12, B=20, seed=0):
    clean, noisy = synth.synthetic_cube(H, W, B, rank=4, seed=seed)
    rng = np.random.default_rng(seed + 11)
    if kind == "bernoulli":
        m = (rng.random((H * W, B)) < 0.6).astype(np.uint8)
    elif kind == "band":
        m = synth.band_mask(H, W, B, keep=0.7, band_frac=0.4, dead_frac=0.3, seed=seed + 5)
    else:
        m = synth.pixel_mask(H, W, "bernoulli", keep=0.6, seed=seed + 5)
    m = m.reshape(H * W, -1) if m.ndim > 1 else m
    if m.ndim == 2:
        m[30:45] = 0                                             # 15 unfolded rows with nothing observed: dead patches
    Y = synth.observe(noisy, m)
    L = (rng.standard_normal(Y.shape) * 0.01).astype(np.float32)
    X = (clean + 0.05 * rng.standard_normal(Y.shape)).astype(np.float32)
    return X, L, Y, m


@gpu
@pytest.mark.parametrize("kind", ["bernoulli", "band"])
@pytest.mark.parametrize("s", [1, 3])
def test_sparse_step_per_element_masks_vs_oracle(kind, s):
    """The fused sparse step in 'spectral_patch' mode against the oracle's 'spectral' (one SVD per distinct pattern):
    Phi_z rel-L2 <= 1e-4 for every fused dictionary width and both engines; patches with nothing observed are 0."""
    X, L, Y, m = _cube_inputs(kind)
    mask = orc.patch_masks(orc.get_image_block(Y, 8, s)[0])
    dead = ~mask.any(axis=0)
    obs = Y != 0
    assert dead.any() and (obs != obs[:, :1]).any()                 # not band-replicated: the row-pattern table cannot serve it
    for K in (64, 128, 192, 256):
        D = synth.synthetic_dictionary(64, K, seed=K)
        ref, _ = orc.sparse_step(X, L, Y, D, orc.Params(mu_1=MU1, lambda_ista=LAM, Nit=NIT, bb=8, slidingDis=s))
        prm = lrs.Params(mu_1=MU1, lambda_ista=LAM, Nit=NIT, bb=8, slidingDis=s, step="spectral_patch")
        for engine in ("simt", "tc"):
            sc = lrs.SparseCoder(cu(Y), cu(D), prm, engine=engine)
            assert sc.fused and sc.a_table is None and sc.a_patch is not None
            phi = sc.phi_z(cu(X), cu(L)).cpu().numpy()
            assert rel(phi, ref) <= 1e-4, (K, engine)
            assert np.all(phi[:, dead] == 0.0), (K, engine)


@gpu
def test_spectral_patch_equals_table_on_replicated_masks():
    """On band-replicated masks every patch's constant equals, bit for bit, the 256-entry table's entry for the patch's
    row pattern, and the two give the same sparse step (<= 1e-5: the kernels' table and per-patch paths round
    differently)."""
    X, L, Y, _ = _cube_inputs("replicated", H=10, W=16, B=24, seed=4)
    D = synth.synthetic_dictionary(64, 256, seed=2)
    sc, out = {}, {}
    for step in ("spectral", "spectral_patch"):
        prm = lrs.Params(mu_1=MU1, lambda_ista=LAM, Nit=NIT, bb=8, slidingDis=1, step=step)
        sc[step] = lrs.SparseCoder(cu(Y), cu(D), prm)
        out[step] = sc[step].phi_z(cu(X), cu(L)).cpu().numpy()
    xs, _ = orc.patch_index(Y.shape[0], Y.shape[1], 8, 1)
    table = sc["spectral"].a_table.cpu().numpy()
    assert np.array_equal(sc["spectral_patch"].a_patch.cpu().numpy(), table[row_patterns(Y[:, 0] != 0, xs)])
    assert rel(out["spectral_patch"], out["spectral"]) <= 1e-5


@gpu
def test_ranges_and_rangewise_overlap_sum_bit_exact():
    """phi_z_range pieces and the range-wise overlap sum (small ranges forced through CHUNK_BYTES) equal the whole launch
    bit for bit in 'spectral_patch' mode."""
    X, L, Y, _ = _cube_inputs("band", H=12, W=20, B=30, seed=6)
    D = synth.synthetic_dictionary(64, 128, seed=1)
    prm = lrs.Params(mu_1=MU1, lambda_ista=LAM, Nit=NIT, bb=8, slidingDis=1, step="spectral_patch")
    sc = lrs.SparseCoder(cu(Y), cu(D), prm, engine="tc")
    Xd, Ld = cu(X), cu(L)
    whole = sc.phi_z(Xd, Ld)
    cuts = [0, 1, 255, 256, 1000, 1777, sc.P]
    pieces = torch.cat([sc.phi_z_range(Xd, Ld, a, b) for a, b in zip(cuts[:-1], cuts[1:])], dim=1)
    assert torch.equal(pieces, whole)
    full = ops.col2im(whole, sc.R, sc.C, 8, 1)
    sc.CHUNK_BYTES = 3 * (sc.R - 7) * 64 * 4                    # three column starts per range
    assert sc._chunk_cols() == 3 < sc.C - 7
    assert torch.equal(sc.imout(Xd, Ld), full)
    assert torch.equal(sc.imout(Xd, Ld, shared_start=True), full)


# ================================================================ 5. solver
@gpu
def test_solver_two_iterations_vs_oracle_without_host_sync():
    """Two outer iterations of LRSPnP in 'spectral_patch' mode on a per-element masked cube equal the oracle's run with
    'spectral' (X within 1e-4), built from device tensors (eigensolver hidden beside the sparse step) and through
    from_host; neither construction synchronises with the host."""
    H, W, B, K = 12, 12, 20, 256
    clean, noisy = synth.synthetic_cube(H, W, B, rank=4, seed=1)
    m = synth.band_mask(H, W, B, keep=0.6, band_frac=0.5, dead_frac=0.3, seed=2).reshape(H * W, B)
    Y = synth.observe(noisy, m)
    MtM = m.astype(np.float32)
    D = synth.synthetic_dictionary(64, K, seed=0)
    prm = lrs.Params(Nit=20, bb=8, slidingDis=1, step="spectral_patch")
    ref = orc.run(Y, MtM, D, orc.Params(Nit=20, bb=8, slidingDis=1, step="spectral"), iteration_num=2)
    Yd, Md, Dd = cu(Y), cu(MtM), cu(D)
    pin = lambda a: torch.from_numpy(a).pin_memory()                        # noqa: E731
    hY, hM = pin(Y), pin(MtM)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        direct = lrs.LRSPnP(Yd, Md, Dd, prm)
        staged = lrs.LRSPnP.from_host(hY, hM, Dd, prm)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert direct.hide_eigensolver
    for sol in (direct, staged):
        sol.run(2)
        assert rel(sol.X.cpu().numpy(), ref.X) <= 1e-4


# ================================================================ 6. full size
@gpu
def test_cfg4_per_element_bernoulli_full_size():
    """The cfg-4 cube (512 x 512 x 191) with a per-element Bernoulli(0.5) mask, about every patch distinct: 10 000 random
    patches' constants within 2e-6 of fp64, and one outer iteration gives a finite X."""
    H, W, B = 512, 512, 191
    _, noisy = synth.synthetic_cube(H, W, B, rank=8, seed=0)
    rng = np.random.default_rng(9)
    Y = synth.observe(noisy, (rng.random((H * W, B)) < 0.5).astype(np.uint8))
    del noisy
    D = synth.synthetic_dictionary(64, 256, seed=0)
    prm = lrs.Params(bb=8, slidingDis=1, step="spectral_patch")
    Yd, Dd = cu(Y), cu(D)
    sol = lrs.LRSPnP(Yd, (Yd != 0).float(), Dd, prm)
    a = sol.be.coder.a_patch
    nR = H * W - 7
    p = rng.choice(sol.be.coder.P, 10000, replace=False)
    ri, ci = p % nR, p // nR
    k = np.arange(64)
    mask = (Y[ri[None, :] + (k % 8)[:, None], ci[None, :] + (k // 8)[:, None]] != 0)
    ref = spectral_fp64(D, mask)
    _check_close(a[torch.as_tensor(p, device="cuda")].cpu().numpy(), ref)
    sol.step()
    assert bool(torch.isfinite(sol.X).all())


# ================================================================ 7. several GPUs
@gpu
def test_sharded_nccl_spectral_patch_equals_single_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29611", os.path.join(HERE, "_sharded_patch_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "sharded-vs-unsharded" in out.stdout


# ================================================================ 8. host side (no GPU needed)
def test_params_accept_spectral_patch():
    assert lrs.Params(step="spectral_patch").step == "spectral_patch"


def test_spectral_patch_rejects_bb_above_8():
    with pytest.raises(ValueError, match="'spectral'"):
        lrs.SparseCoder(torch.zeros(40, 20), torch.zeros(81, 64), lrs.Params(bb=9, slidingDis=1, step="spectral_patch"))
    with pytest.raises(ValueError, match="bb <= 8"):
        ops.patch_step_constants(np.ones((40, 20), np.float32), np.ones((81, 64), np.float32), 9, 1)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
def test_patch_constants_refuse_without_device():
    with pytest.raises(lrs.LrsError):
        ops.patch_step_constants(np.ones((40, 20), np.float32), np.ones((64, 64), np.float32), 8, 1)
    with pytest.raises(lrs.LrsError):
        lrs.SparseCoder(torch.ones(40, 20), torch.ones(64, 64), lrs.Params(bb=8, slidingDis=1, step="spectral_patch"))
    L = _lib.lib()
    assert L.lrs_patch_mask_words_u64(1, 40, 20, 8, 1, 0, 33 * 13, 1, None) == -2 and b"CUDA" in L.lrs_last_error()
    assert L.lrs_spectral_patterns_f32(1, 64, 64, 1, 10, None, 0, 1, 1, 1 << 15, None) == -2
    assert L.lrs_spectral_patterns_workspace_bytes(65) == 0
