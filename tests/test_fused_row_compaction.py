"""The tcgen05 fused sparse step in the step-constant table mode orders the row starts by their row-validity pattern
and runs GEMM-B and the residual over each tile's observed window rows only.  The host half replays that tile order
(diagnostics build, no GPU); the GPU half runs row masks at every compaction edge against the fp64 oracle, the FFMA
engine, the dynamically dealt instance and the same launch in the per-patch constant mode (identity tile order)."""
import numpy as np
import pytest
import torch

from lrs_pnp_dip_b200 import _lib, ops, synth
from oracle import lrs_oracle as orc
from tests.test_kernel_edges import de_bruijn_rows, per_patch_err, rel, row_patterns


def gray_rank(w):
    w = np.asarray(w, np.int64)
    w = w ^ (w >> 1)
    w = w ^ (w >> 2)
    return w ^ (w >> 4)


# ================================================================ host: the ordered tile walk
def test_ordered_tile_walk_covers_every_patch_once():
    """lrs_debug_tile_walk_ordered replays the table mode's tile walk on the host: the order is a permutation of the row
    starts, sorted by the Gray rank of their 8-row validity word and ascending within a word, and every patch of the
    range is owned by exactly one valid lane, for random masks, strides with appended starts, sub-ranges cutting
    through columns and SM counts from 1 to 200."""
    L = _lib.diag_lib()
    rng = np.random.default_rng(7)
    cases = [(300, 20, 1, 148), (263, 12, 1, 148), (64, 41, 3, 148), (1500, 30, 1, 7), (262144 // 64, 30, 1, 148),
             (9, 8, 5, 3), (8, 8, 1, 1), (50, 9, 20, 200), (301, 30, 3, 200)]
    for _ in range(30):
        cases.append((int(rng.integers(8, 900)), int(rng.integers(8, 40)), int(rng.integers(1, 6)),
                      int(rng.integers(1, 201))))
    for R, Cc, s, sms in cases:
        kind = int(rng.integers(0, 3))
        if kind == 0:
            row_obs = rng.random(R) < rng.uniform(0.1, 0.9)
        elif kind == 1:
            row_obs = (np.arange(R) % int(rng.integers(2, 9))) == 0
        else:
            row_obs = rng.random(R) < 0.5
            g = int(rng.integers(0, R))
            row_obs[g:g + 140] = False                               # a run of unobserved rows longer than a tile
        row_obs = np.ascontiguousarray(row_obs.astype(np.uint8))
        starts = orc.axis_starts(R, 8, s)
        nR = len(starts)
        keys = gray_rank(row_patterns(row_obs.astype(bool), starts))
        P = ops.patch_count(R, Cc, 8, s)
        ranges = [(0, P)]
        if P > 1:
            a = int(rng.integers(0, P))
            ranges += [(a, int(rng.integers(a + 1, P + 1))), (P - 1, P), (0, 1), (nR // 2, P - nR // 3)]
        for b, e in ranges:
            if not 0 <= b < e <= P:
                continue
            visits = np.zeros(e - b, dtype=np.int32)
            tiles = np.zeros(1, dtype=np.int64)
            order = np.full(nR, -1, dtype=np.int32)
            rc = L.lrs_debug_tile_walk_ordered(R, Cc, 8, s, b, e, sms, row_obs.ctypes.data, visits.ctypes.data,
                                               tiles.ctypes.data, order.ctypes.data)
            assert rc == 0, (L.lrs_last_error(), R, Cc, s, b, e, sms)
            assert visits.min() == 1 and visits.max() == 1, (R, Cc, s, b, e, sms)
            assert np.array_equal(np.sort(order), np.arange(nR)), (R, Cc, s)
            assert np.array_equal(order, np.argsort(keys, kind="stable")), (R, Cc, s)
            cols = (e - 1) // nR - b // nR + 1
            assert tiles[0] == cols * ((nR + 127) // 128), (R, Cc, s, b, e, sms)


# ================================================================ GPU: compaction edges in the table mode
MU1, LAM = 0.15, 0.1
R_ROWS, C_COLS = 400, 12


def _row_mask(name):
    rng = np.random.default_rng(11)
    r = np.arange(R_ROWS)
    if name == "all":
        return np.ones(R_ROWS, bool)
    if name == "none":
        return np.zeros(R_ROWS, bool)
    if name == "one-in-eight":
        return r % 8 == 3
    if name == "alternate":
        return r % 2 == 0
    if name == "long-gaps":
        m = rng.random(R_ROWS) < 0.5
        m[40:180] = False
        m[250:390] = False
        return m
    if name == "random":
        return rng.random(R_ROWS) < 0.5
    return de_bruijn_rows(8)                                     # "debruijn": every 8-row pattern once, R = 263


MASKS = ("all", "none", "one-in-eight", "alternate", "long-gaps", "random", "debruijn")


@pytest.fixture(scope="module")
def lrs():
    import lrs_pnp_dip_b200 as m

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    m._lib.lib()
    return m


def cu(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("K", [64, 128, 192, 256])
@pytest.mark.parametrize("mask", MASKS)
def test_fused_tc_table_mode_row_compaction_edges(lrs, mask, K):
    """Table mode (row-pattern tile order, compacted GEMM-B and residual) against the fp64 oracle and the FFMA engine
    per patch, dead patches exactly 0, the dynamic instance bit-identical to the static one, and the same launch in the
    per-patch constant mode (identity tile order: other tiles, other row sets) within 1e-5 per patch, Nit in {1, 3, 80}."""
    row_obs = _row_mask(mask)
    R, C, s = len(row_obs), C_COLS, 1
    rng = np.random.default_rng(R + K)
    X = (rng.standard_normal((R, C)) * 0.3 + 0.5).astype(np.float32)
    L = (rng.standard_normal((R, C)) * 0.01).astype(np.float32)
    M = np.repeat(row_obs[:, None], C, axis=1)
    Y = np.where(M, X + 0.01, 0).astype(np.float32)
    Y[M & (Y == 0)] = 1e-12
    D = synth.synthetic_dictionary(64, K, seed=K + 5)
    xs, _ = orc.patch_index(R, C, 8, s)
    P = len(xs)
    Xd, Ld, Yd, Dd = cu(X), cu(L), cu(Y), cu(D)
    a_table_d = ops._row_pattern_table(Dd, 8, "spectral")
    a = a_table_d.cpu().numpy()[row_patterns(row_obs, xs)]
    a_patch_d = cu(a.astype(np.float32))
    mask_p = orc.patch_masks(orc.get_image_block(Y, 8, s)[0])
    dead = ~mask_p.any(axis=0)
    for nit in (1, 3, 80):
        oprm = orc.Params(mu_1=MU1, lambda_ista=LAM, Nit=nit, bb=8, slidingDis=s)
        ref64, _ = orc.sparse_step(X, L, Y, D, oprm, a=a.astype(np.float64), dtype=np.float64)
        ref32, _ = orc.sparse_step(X, L, Y, D, oprm, a=a.astype(np.float32), dtype=np.float32)
        floor = 1e-6 * max(float(np.linalg.norm(ref64, axis=0).max()), 1e-30)
        allow = max(1e-3, 4.0 * float(per_patch_err(ref32, ref64, floor).max()))

        def call(engine, a_patch=None, a_table=None):
            phi = torch.full((64, P), float("nan"), dtype=torch.float32, device="cuda")
            _lib.check(_lib.lib().lrs_sparse_step_fused_f32(
                _lib.ptr(Xd), _lib.ptr(Ld), MU1, _lib.ptr(Yd), _lib.ptr(Dd), K, _lib.ptr(a_patch), _lib.ptr(a_table),
                LAM, nit, R, C, 8, s, 0, P, _lib.ptr(phi), engine, _lib.stream_ptr()), "lrs_sparse_step_fused_f32")
            return phi.cpu().numpy()

        tc = call(_lib.ENGINE_TC, a_table=a_table_d)
        simt = call(_lib.ENGINE_SIMT, a_table=a_table_d)
        dyn = call(_lib.ENGINE_TC | _lib.ENGINE_DYNAMIC_TILES, a_table=a_table_d)
        ident = call(_lib.ENGINE_TC, a_patch=a_patch_d)
        where = (mask, K, nit)
        for name, phi in (("tc", tc), ("simt", simt)):
            assert np.isfinite(phi).all(), (where, name)
            assert np.all(phi[:, dead] == 0), (where, name)
            if ref64.any():
                assert rel(phi, ref64) <= 1e-4, (where, name)
            err = per_patch_err(phi, ref64, floor)
            assert err.max() <= allow, (where, name, int(err.argmax()), float(err.max()), allow)
        if mask == "none":
            assert not tc.any(), where
        assert per_patch_err(tc, simt, floor).max() <= 1e-4, where
        assert np.array_equal(dyn, tc), where
        iso = per_patch_err(tc, ident, floor)
        assert iso.max() <= 1e-5, (where, int(iso.argmax()), float(iso.max()))
