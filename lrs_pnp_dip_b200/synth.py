"""Seeded synthetic inputs for the configurations BASELINE.json names
(SURVEY §8d): dictionary, hyperspectral cube, per-pixel masks.  Host-side
NumPy only; the arrays are uploaded by the caller.

The dictionary file the reference loads (``trained_dictionary.mat``,
main_LRS_PnP.py:159-165) is not part of the checkout, so every run that does
not find it uses :func:`synthetic_dictionary`.
"""
from __future__ import annotations

import numpy as np

F32 = np.float32


def synthetic_dictionary(n: int, K: int, seed: int = 0) -> np.ndarray:
    """Gaussian ``D ∈ R^{n×K}``, columns ℓ2-normalised as columnNormalise.m:1-4."""
    rng = np.random.default_rng(seed)
    D = rng.standard_normal((n, K)).astype(F32)
    D /= np.sqrt((D.astype(np.float64) ** 2).sum(0, keepdims=True)).astype(F32)
    return np.ascontiguousarray(D)


def _smooth_fields(rng, H, W, k, sigma):
    from scipy.ndimage import gaussian_filter

    f = rng.standard_normal((k, H, W)).astype(F32)
    for i in range(k):
        f[i] = gaussian_filter(f[i], sigma=sigma, mode="wrap")
        f[i] /= max(float(f[i].std()), 1e-12)
    return f


def synthetic_cube(H: int, W: int, B: int, rank: int = 8, noise_sigma: float = 0.12, seed: int = 0):
    """Rank-``rank`` linear mixture ``clip(A·E, 0, 1)`` + N(0, σ²) noise, unfolded
    with row = i*W + j.  Returns ``(clean [H*W,B], noisy [H*W,B])`` f32.
    σ = 0.12 is the reference's noise level (main_LRS_PnP.m:23)."""
    rng_a = np.random.default_rng(seed)
    rng_e = np.random.default_rng(seed + 1)
    rng_n = np.random.default_rng(seed + 2)
    fields = _smooth_fields(rng_a, H, W, rank, sigma=6.0) * F32(2.0)
    fields -= fields.max(0, keepdims=True)
    A = np.exp(fields)
    A /= A.sum(0, keepdims=True)
    A = A.reshape(rank, H * W).T.astype(F32)                       # [R, rank]
    E = np.cumsum(rng_e.standard_normal((rank, B)), axis=1)
    E -= E.min(1, keepdims=True)
    E /= np.maximum(E.max(1, keepdims=True), 1e-12)
    clean = np.clip(A @ E.astype(F32), 0, 1).astype(F32)
    noisy = clean.copy()
    step = 1 << 16
    for r0 in range(0, H * W, step):                                # chunked: keeps peak RAM low
        noisy[r0:r0 + step] += (noise_sigma * rng_n.standard_normal((min(step, H * W - r0), B))).astype(F32)
    return clean, noisy


def pixel_mask(H: int, W: int, kind: str = "bernoulli", keep: float = 0.5, seed: int = 3) -> np.ndarray:
    """Per-pixel 0/1 mask ``[H*W]`` (uint8), replicated over bands by the caller
    (main_LRS_PnP.m:42-44).  'bernoulli': keep with probability ``keep``;
    'stripe+bernoulli': every third image column dropped (like fourth_mask)
    ∪ Bernoulli(keep)."""
    rng = np.random.default_rng(seed)
    m = (rng.random((H, W)) < keep)
    if kind == "stripe+bernoulli":
        m[:, 2::3] = False
    elif kind != "bernoulli":
        raise ValueError(kind)
    return m.reshape(-1).astype(np.uint8)


def band_mask(H: int, W: int, B: int, keep: float = 0.7, band_frac: float = 0.25, dead_frac: float = 0.05,
              seed: int = 5) -> np.ndarray:
    """Per-element 0/1 mask ``[H, W, B]`` (uint8) with band-dependent missing data: a per-pixel Bernoulli(``keep``) mask
    replicated over the bands, and in a random ``band_frac`` of the bands, each its own random ``dead_frac`` of the
    image columns dropped (dead detector lines / stripes that affect only some bands).  Not band-replicated, but an 8 x 8
    patch meets at most one dead column per band, so the distinct patch patterns stay moderate in number."""
    rng = np.random.default_rng(seed)
    m = np.repeat((rng.random((H, W)) < keep)[:, :, None], B, axis=2)
    bands = np.flatnonzero(rng.random(B) < band_frac)
    for b in bands:
        m[:, rng.random(W) < dead_frac, b] = False
    return m.astype(np.uint8)


def observe(noisy: np.ndarray, pix_mask: np.ndarray) -> np.ndarray:
    """Apply the mask the way the reference detects it: missing entries are
    exactly 0.0 (main_LRS_PnP.py:276-278), and an observed exact zero is nudged
    to 1e-12 so that ``== 0`` ⇔ masked.  ``pix_mask``: per pixel ``[H*W]``
    (replicated over the bands), or per element ``[H*W, B]`` / ``[H, W, B]``."""
    Y = noisy.astype(F32).copy()
    Y[Y == 0] = F32(1e-12)
    if pix_mask.ndim == 1:
        Y[pix_mask == 0, :] = 0
    else:
        Y[pix_mask.reshape(Y.shape) == 0] = 0
    return Y


def cross_masked(Y: np.ndarray, pix_mask: np.ndarray):
    """Cube (i, m) of the batched experiments: the observed cube ``Y [R, C]`` of image i (already zero on its own
    missing pixels) with the pixels missing in mask m (``pix_mask [R]``, 0 = missing, unfolded pixel order) zeroed too.
    Returns ``(Y_im [R, C] f32, MtM [R, C] f32)``; MtM is the row indicator of the pixels still observed (a row of Y
    that is not all zero, and kept by mask m), replicated over the bands."""
    Y = np.asarray(Y, dtype=F32)
    keep = (np.asarray(pix_mask).reshape(-1) != 0) & (Y != 0).any(axis=1)
    Yim = np.where(keep[:, None], Y, F32(0)).astype(F32)
    return np.ascontiguousarray(Yim), np.ascontiguousarray(np.repeat(keep.astype(F32)[:, None], Y.shape[1], axis=1))
