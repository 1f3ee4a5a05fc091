"""The reference's own call signatures, served by the sm_100a library.

Every public function here has the name, positional arguments, return arity,
shapes, dtypes and orderings of the function it replaces in
main_LRS_PnP.py / main_LRS_PnP_DIP_*.py / admm_utils.py (cited per function),
so the scripts' bodies can call them unchanged.  Inputs may live on the CPU
(as in the reference, which is CPU-only on this path) or on a CUDA device;
outputs come back on the input's device.  All arithmetic runs in
liblrs_pnp.so on the GPU — there is no CPU fallback.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import check, lib, ptr, require_cuda, stream_ptr


# ------------------------------------------------------------------ helpers
def _to_dev(x, dtype=torch.float32) -> Tuple[torch.Tensor, torch.device, bool]:
    """→ (contiguous CUDA tensor, original device, was_numpy)."""
    require_cuda()
    was_np = isinstance(x, np.ndarray)
    t = torch.as_tensor(x)
    src = t.device
    if t.device.type != "cuda":
        t = t.to("cuda", non_blocking=False)
    if t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous(), src, was_np


def _back(t: torch.Tensor, src: torch.device, was_np: bool = False):
    if was_np:
        return t.cpu().numpy()
    return t if src.type == "cuda" else t.to(src)


def patch_grid(R: int, C: int, bb: int, s: int) -> Tuple[np.ndarray, np.ndarray]:
    """Selected row / column starts (host, int64) — the product set behind
    idx_Mat, main_LRS_PnP.py:76-91."""
    L = lib()
    out = []
    for length in (R, C):
        n = L.lrs_axis_count(length, bb, s)
        if n < 0:
            raise _lib.LrsError(f"invalid geometry: length={length} bb={bb} stride={s}")
        buf = (_lib.C.c_int64 * n)()
        check(L.lrs_axis_starts(length, bb, s, buf, n), "lrs_axis_starts")
        out.append(np.frombuffer(buf, dtype=np.int64).copy())
    return out[0], out[1]


def patch_count(R: int, C: int, bb: int, s: int) -> int:
    L = lib()
    nr, nc = L.lrs_axis_count(R, bb, s), L.lrs_axis_count(C, bb, s)
    if nr < 0 or nc < 0:
        raise _lib.LrsError(f"invalid geometry: R={R} C={C} bb={bb} stride={s}")
    return int(nr * nc)


# ------------------------------------------------------------------ get_image_block
def im2col(X: torch.Tensor, bb: int, s: int, lambda_1: Optional[torch.Tensor] = None, mu_1: float = 1.0) -> torch.Tensor:
    """Device-side patch matrix of ``X`` (or of ``X + lambda_1/mu_1``) ``[bb², P]``."""
    R, C = X.shape
    P = patch_count(R, C, bb, s)
    out = torch.empty((bb * bb, P), dtype=torch.float32, device=X.device)
    check(lib().lrs_im2col_f32(ptr(X), ptr(lambda_1), float(mu_1), R, C, bb, s, ptr(out), stream_ptr()), "lrs_im2col_f32")
    return out


def get_image_block(input_img, block_size, slidingDis):
    """main_LRS_PnP.py:73-107 → ``(blocks [bb²,P] f32, x_index [P] int64 ndarray,
    y_index [P] int64 ndarray, idx_Mat [R-bb+1, C-bb+1] f32)``."""
    X, src, _ = _to_dev(input_img)
    if X.dim() != 2:
        raise ValueError("get_image_block expects a 2-D (pixels x bands) matrix")
    bb, s = int(block_size), int(slidingDis)
    R, C = X.shape
    with torch.cuda.device(X.device):
        P = patch_count(R, C, bb, s)
        blocks = im2col(X, bb, s)
        xi = torch.empty(P, dtype=torch.int64, device=X.device)
        yi = torch.empty(P, dtype=torch.int64, device=X.device)
        idx = torch.empty((R - bb + 1, C - bb + 1), dtype=torch.float32, device=X.device)
        check(lib().lrs_patch_index_i64(R, C, bb, s, ptr(xi), ptr(yi), ptr(idx), stream_ptr()), "lrs_patch_index_i64")
    return _back(blocks, src), xi.cpu().numpy(), yi.cpu().numpy(), _back(idx, src)


def col2im(blocks: torch.Tensor, R: int, C: int, bb: int, s: int) -> torch.Tensor:
    """Overlap sum of ``blocks [bb²,P]`` in ascending patch order
    (main_LRS_PnP.py:332-339), bit-exact with the sequential loop."""
    blocks = blocks.contiguous()
    if tuple(blocks.shape) != (bb * bb, patch_count(R, C, bb, s)):
        raise ValueError(f"blocks has shape {tuple(blocks.shape)}, geometry needs {(bb * bb, patch_count(R, C, bb, s))}")
    out = torch.empty((R, C), dtype=torch.float32, device=blocks.device)
    check(lib().lrs_col2im_accum_f32(ptr(blocks), R, C, bb, s, ptr(out), stream_ptr()), "lrs_col2im_accum_f32")
    return out


def im2col_batch(X: torch.Tensor, bb: int, s: int, lambda_1: Optional[torch.Tensor] = None, mu_1: float = 1.0) -> torch.Tensor:
    """Patch matrices of B cubes ``X [B, R, C]`` (or of ``X + lambda_1/mu_1``) side by side: ``[bb², B*P]``, cube b in
    columns ``[b*P, (b+1)*P)``."""
    B, R, C = X.shape
    P = patch_count(R, C, bb, s)
    out = torch.empty((bb * bb, B * P), dtype=torch.float32, device=X.device)
    check(lib().lrs_im2col_batch_f32(ptr(X), ptr(lambda_1), float(mu_1), B, R, C, bb, s, ptr(out), stream_ptr()),
          "lrs_im2col_batch_f32")
    return out


def col2im_batch(blocks: torch.Tensor, B: int, R: int, C: int, bb: int, s: int) -> torch.Tensor:
    """Overlap sums ``[B, R, C]`` of ``blocks [bb², B*P]`` (cube b in columns ``[b*P, (b+1)*P)``), each bit-exact with
    :func:`col2im` on its own columns."""
    blocks = blocks.contiguous()
    if tuple(blocks.shape) != (bb * bb, B * patch_count(R, C, bb, s)):
        raise ValueError(f"blocks has shape {tuple(blocks.shape)}, geometry needs {(bb * bb, B * patch_count(R, C, bb, s))}")
    out = torch.empty((B, R, C), dtype=torch.float32, device=blocks.device)
    check(lib().lrs_col2im_accum_batch_f32(ptr(blocks), B, R, C, bb, s, ptr(out), stream_ptr()), "lrs_col2im_accum_batch_f32")
    return out


def coverage_weight(R: int, C: int, bb: int, s: int, device="cuda") -> torch.Tensor:
    """``Weight`` of main_LRS_PnP.py:341."""
    require_cuda()
    out = torch.empty((R, C), dtype=torch.float32, device=device)
    check(lib().lrs_coverage_weight_f32(R, C, bb, s, ptr(out), stream_ptr()), "lrs_coverage_weight_f32")
    return out


# ------------------------------------------------------------------ soft threshold family
def _soft(x, tau):
    t, src, was_np = _to_dev(x)
    out = torch.empty_like(t)
    with torch.cuda.device(t.device):
        check(lib().lrs_soft_f32(ptr(t), float(tau), ptr(out), t.numel(), stream_ptr()), "lrs_soft_f32")
    return _back(out, src, was_np)


def soft_thresh(x, l):
    """main_LRS_PnP.py:128-129."""
    return _soft(x, l)


def Shrinkage_Operator(X, tau):
    """main_LRS_PnP.py:112-116."""
    return _soft(X, tau)


def l1_prox(input, lamda):
    """admm_utils.py:72-75."""
    return _soft(input, lamda)


def delete_element(tensor, indices):
    """main_LRS_PnP.py:152-155 — row deletion (index bookkeeping only, no arithmetic)."""
    mask = torch.ones(tensor.size(0), dtype=torch.bool, device=tensor.device)
    mask[torch.as_tensor(indices, dtype=torch.long, device=tensor.device)] = False
    return tensor[mask].view((-1, tensor.size()[1]))


# ------------------------------------------------------------------ step constants
def spectral_norm_sq(H: torch.Tensor) -> float:
    """``np.linalg.norm(H,2)**2`` (main_LRS_PnP.py:134) as λmax of the smaller Gram matrix, fp64 on
    the device (one-off setup, library eigensolver)."""
    Hd = H.to(torch.float64)
    G = Hd @ Hd.T if Hd.shape[0] <= Hd.shape[1] else Hd.T @ Hd
    if G.numel() == 0:
        return 0.0
    return float(torch.linalg.eigvalsh(G)[-1].clamp_min(0))


def step_constants(blocks_copy: torch.Tensor, D: torch.Tensor, step: str) -> torch.Tensor:
    """a[p] for explicit patch matrices; mask = (blocks_copy != 0), main_LRS_PnP.py:276-280.
    'frob4': main_LRS_PnP_DIP_pro.py:190 ; 'spectral': main_LRS_PnP.py:134 (one eigensolve per
    DISTINCT mask pattern instead of one SVD per patch per outer iteration)."""
    n, P = blocks_copy.shape
    K = D.shape[1]
    a = torch.empty(P, dtype=torch.float32, device=blocks_copy.device)
    if step == "frob4":
        check(lib().lrs_step_frob4_f32(ptr(blocks_copy), ptr(D), n, K, P, ptr(a), stream_ptr()), "lrs_step_frob4_f32")
        return a
    if step != "spectral":
        raise ValueError(f"unknown step mode {step!r}")
    m = (blocks_copy != 0).T.contiguous()                         # [P, n] bool
    # distinct patterns through two independent 64-bit hashes per patch (torch.unique(dim=0) sorts whole rows: ~10 ms for
    # 144 x 1296); equal patterns hash equal, and the representatives are compared bit by bit below
    gen = torch.Generator(device="cpu").manual_seed(0x5EED)
    w = torch.randint(-(1 << 62), 1 << 62, (2, n), generator=gen, dtype=torch.int64).to(m.device)
    h = torch.empty((P, 2), dtype=torch.int64, device=m.device)   # wrapping int64 arithmetic
    chunk = max(1, (4 << 20) // max(n, 1))                        # bounded temporaries whatever P is
    for p0 in range(0, P, chunk):
        mm = m[p0:p0 + chunk].to(torch.int64)
        h[p0:p0 + chunk, 0] = (mm * w[0]).sum(1)
        h[p0:p0 + chunk, 1] = (mm * w[1]).sum(1)
    _, inv = torch.unique(h, dim=0, return_inverse=True)
    inv = inv.reshape(-1)
    n_u = int(inv.max()) + 1
    rep = torch.full((n_u,), P, dtype=torch.int64, device=m.device).scatter_reduce(
        0, inv, torch.arange(P, device=m.device), reduce="amin")
    uniq = m[rep]
    if not bool((uniq[inv] == m).all()):                          # a hash collision merged two patterns: exact fallback
        uniq, inv = torch.unique(m, dim=0, return_inverse=True)
    if uniq.shape[0] > MAX_SPECTRAL_PATTERNS:
        raise _lib.LrsError(f"{uniq.shape[0]} distinct mask patterns: spectral step constants need one eigensolve "
                            "each; use step='frob4' or pass explicit step constants")
    # One eigensolve per distinct pattern AND dictionary, ever: the value depends on (D, pattern) only, the reference pays an
    # SVD for it per patch per outer iteration, and an eigensolve of a 1296 x 1296 Gram matrix is ~10 ms — five outer
    # iterations of configuration 1.  Memoised per dictionary TENSOR (address, in-place version, shape: as the row-pattern
    # table below) and pattern bytes; the patterns travel to the host once (U x n bits).
    dkey = (D.data_ptr(), D._version, tuple(D.shape), tuple(D.stride()), str(D.device))
    packed = np.packbits(uniq.cpu().numpy(), axis=1)
    vals = []
    for u in range(uniq.shape[0]):
        key = (dkey, packed[u].tobytes())
        hit = _SPECTRAL_CACHE.get(key)
        if hit is None:
            if len(_SPECTRAL_CACHE) > 4096:
                _SPECTRAL_CACHE.clear()
            hit = _SPECTRAL_CACHE[key] = (D, spectral_norm_sq(D[uniq[u]]))
        vals.append(hit[1])
    vals = torch.tensor(vals, dtype=torch.float32, device=a.device)
    return vals[inv.reshape(-1)].contiguous()


_SPECTRAL_CACHE: dict = {}
MAX_SPECTRAL_PATTERNS = 4096             # distinct mask patterns step_constants solves (one eigensolve each)


def row_pattern_table(D: torch.Tensor, bb: int, step: str) -> torch.Tensor:
    """a for each of the 2^bb validity patterns of a patch's pixel rows (band-replicated masks:
    window element (i, j) is valid iff unfolded row r+i is observed).  bb = 8 → 256 entries."""
    n, K = D.shape
    assert n == bb * bb
    # The table depends on the dictionary only; the reference recomputes it per patch per outer iteration
    # (main_LRS_PnP.py:134).  Cached per dictionary TENSOR: the key is (storage address, in-place version counter,
    # shape, device) and the entry keeps a reference to the tensor, so the address cannot be recycled while the entry
    # lives and any in-place write to D invalidates it.  No device synchronisation on a hit or a miss.
    key = (D.data_ptr(), D._version, tuple(D.shape), tuple(D.stride()), str(D.device), bb, step)
    hit = _TABLE_CACHE.get(key)
    if hit is not None:
        return hit[1]
    out = _row_pattern_table(D, bb, step)
    if len(_TABLE_CACHE) > 16:
        _TABLE_CACHE.clear()
    _TABLE_CACHE[key] = (D, out)
    return out


_TABLE_CACHE: dict = {}

# patches whose words are merged in one pass of patch_step_constants: bounds its transient memory (~80 B per patch of a
# pass: the words, the sort's keys, indices and scratch, the group numbers and representatives) whatever P is
PATCH_CONSTANTS_CHUNK = 1 << 25


_STEP_MODES = {"spectral": _lib.STEP_SPECTRAL, "frob4": _lib.STEP_FROB4}


def _spectral_patterns(D: torch.Tensor, words: torch.Tensor, step: str, count: Optional[torch.Tensor] = None):
    """a[i] = the step constant of pattern word words[i] (int64 view of the uint64 word, bit k = row k of the contiguous
    fp32 dictionary D) by lrs_spectral_patterns_f32, on the current stream.  ``count``: a device int64 holding how many
    leading words to process (the rest of a is left unwritten), None = all of them."""
    mode = _STEP_MODES.get(step)
    if mode is None:
        raise ValueError(f"unknown step mode {step!r}")
    n, K = D.shape
    L = lib()
    ws_bytes = L.lrs_spectral_patterns_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=D.device)
    a = torch.empty(words.numel(), dtype=torch.float32, device=D.device)
    check(L.lrs_spectral_patterns_f32(ptr(D), n, K, ptr(words), words.numel(), ptr(count), mode, ptr(a), ptr(ws), ws_bytes,
                                      stream_ptr()), "lrs_spectral_patterns_f32")
    return a


def patch_step_constants(Y_observed, D, bb: int, s: int, step: str = "spectral", p_begin: int = 0,
                         p_end: Optional[int] = None):
    """a[p] = ||M_p D||_2^2 (``step='spectral'``, np.linalg.norm(H, 2)**2 of main_LRS_PnP.py:134) or 4||M_p D||_F^2
    (``'frob4'``) for the patches p in [p_begin, p_end) of the observed matrix, M_p = the patch's own observed entries
    (``Y_observed != 0``, main_LRS_PnP.py:276-289), for ANY mask, bb <= 8.

    Each patch's validity is one 64-bit word (lrs_patch_mask_words_u64).  The word IS the pattern, so equal patterns are
    merged exactly, on the device and without a host synchronisation: sort, mark where a run of equal words starts,
    cumsum for the group number, scatter one representative per group.  lrs_spectral_patterns_f32 then runs once per
    distinct word (it reads the number of groups on the device) and the values are gathered back to the patches."""
    bb, s = int(bb), int(s)
    if not 1 <= bb <= 8:
        raise ValueError(f"per-patch step constants pack a patch's mask into 64 bits: bb <= 8 (got bb = {bb})")
    if step not in _STEP_MODES:
        raise ValueError(f"unknown step mode {step!r}")
    Y, src, was_np = _to_dev(Y_observed)
    if Y.dim() != 2:
        raise ValueError("Y_observed must be a 2-D (pixels x bands) matrix")
    R, C = Y.shape
    Dd = torch.as_tensor(D).to(device=Y.device, dtype=torch.float32).contiguous()
    n = Dd.shape[0]
    if n != bb * bb:
        raise ValueError(f"dictionary has {n} rows, bb² = {bb * bb}")
    P = patch_count(R, C, bb, s)
    p_end = P if p_end is None else int(p_end)
    p_begin = int(p_begin)
    if not 0 <= p_begin <= p_end <= P:
        raise ValueError(f"patch range [{p_begin}, {p_end}) outside [0, {P}]")
    L = lib()
    with torch.cuda.device(Y.device):
        a = torch.empty(p_end - p_begin, dtype=torch.float32, device=Y.device)
        for c0 in range(p_begin, p_end, PATCH_CONSTANTS_CHUNK):
            c1 = min(p_end, c0 + PATCH_CONSTANTS_CHUNK)
            m = c1 - c0
            words = torch.empty(m, dtype=torch.int64, device=Y.device)
            check(L.lrs_patch_mask_words_u64(ptr(Y), R, C, bb, s, c0, c1, ptr(words), stream_ptr()), "lrs_patch_mask_words_u64")
            sw, order = torch.sort(words)                  # int64 order of the uint64 words: any order groups equal words
            del words
            start = torch.ones(m, dtype=torch.bool, device=Y.device)
            torch.ne(sw[1:], sw[:-1], out=start[1:])
            group = torch.cumsum(start, 0, dtype=torch.int64).sub_(1)     # group number of each sorted word
            del start
            uniq = torch.empty_like(sw).scatter_(0, group, sw)    # the words of a group are equal: any writer is right
            count = group[-1:] + 1                                 # number of distinct words, stays on the device
            vals = _spectral_patterns(Dd, uniq, step, count)
            a[c0 - p_begin:c1 - p_begin].index_copy_(0, order, vals.index_select(0, group))
            del sw, order, group, uniq, vals
    return _back(a, src, was_np)


def _row_pattern_table(D: torch.Tensor, bb: int, step: str) -> torch.Tensor:
    """The pattern values of the 2^bb row-pattern words: row pattern r is the word with bit k set iff bit k % bb of r
    is set (element k of a patch sits in pixel row k % bb), the word of a patch whose rows are observed in all bands
    or in none."""
    if not 1 <= bb <= 8:
        raise _lib.LrsError(f"row-pattern step-constant tables exist for bb <= 8 (got bb = {bb})")
    with torch.cuda.device(D.device):
        r = torch.arange(1 << bb, dtype=torch.int64, device=D.device)
        k = torch.arange(bb * bb, dtype=torch.int64, device=D.device)
        words = (((r[:, None] >> (k % bb)) & 1) << k).sum(1)      # distinct bits: the sum is their OR (bit 63 = sign)
        return _spectral_patterns(D.contiguous(), words, step)


# ------------------------------------------------------------------ ista
def ista_batched(blocks: torch.Tensor, blocks_copy: torch.Tensor, D: torch.Tensor, a: torch.Tensor, lambda_ista: float,
                 Nit: int, want_coefs: bool = False, want_phi: bool = True, denoiser: str = "soft", h_scale: float = 0.1):
    """All patches at once (explicit patch matrices, any n / K / P).  Returns (coefs [K,P] | None,
    phi_z [n,P] | None).  Replaces the jj loop main_LRS_PnP.py:270-303.  ``denoiser``: 'soft' (ista.m:23),
    'nlm' (NLmeansfilter(g,3,3,h_scale*T), pnp_ista.m:30) or 'identity'."""
    n, P = blocks.shape
    K = D.shape[1]
    L = lib()
    ws_bytes = L.lrs_ista_workspace_bytes(n, K, P)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=blocks.device)
    coefs = torch.empty((K, P), dtype=torch.float32, device=blocks.device) if want_coefs else None
    phi = torch.empty((n, P), dtype=torch.float32, device=blocks.device) if want_phi else None
    if denoiser not in _lib.DENOISERS:
        raise ValueError(f"unknown denoiser {denoiser!r}")
    check(L.lrs_ista_pnp_f32(ptr(blocks), ptr(blocks_copy), ptr(D), ptr(a), float(lambda_ista), int(Nit), n, K, P,
                             _lib.DENOISERS[denoiser], float(h_scale), ptr(coefs), ptr(phi), ptr(ws), ws_bytes,
                             stream_ptr()), "lrs_ista_pnp_f32")
    return coefs, phi


def ista(y, H, lambda_ista, alpha, Nit, *, denoiser: str = "soft", step: str = "spectral", h_scale: float = 0.1):
    """main_LRS_PnP.py:131-149 / main_LRS_PnP_DIP_pro.py:188-201 / ista.m:1-24 / pnp_ista.m:1-32.
    ``alpha`` is ignored and recomputed exactly as the reference does (``step='spectral'``:
    ‖H‖₂² ; ``'frob4'``: 4‖H‖_F²).  ``denoiser='soft'`` is the MATLAB twin's soft(g, T) (ista.m:23);
    ``'nlm'`` is the in-repo MATLAB NLmeansfilter(g, 3, 3, h_scale*T) (pnp_ista.m:30) — the skimage
    ``denoise_nl_means`` of the Python scripts is a different third-party algorithm and is not reproduced."""
    Hd, src, _ = _to_dev(H)
    yd, _, _ = _to_dev(y)
    yd = yd.reshape(-1, 1)
    with torch.cuda.device(Hd.device):
        ones = torch.ones_like(yd)
        if step == "spectral":
            a = torch.tensor([spectral_norm_sq(Hd)], dtype=torch.float32, device=Hd.device)
        else:
            a = step_constants(ones, Hd, step)
        coefs, _ = ista_batched(yd, ones, Hd, a, lambda_ista, Nit, want_coefs=True, want_phi=False, denoiser=denoiser,
                                h_scale=h_scale)
    return _back(coefs, src)


# ------------------------------------------------------------------ SVT
_EIGH_PAD_FROM, _EIGH_PAD_TO = 96, 136     # library path: band counts in [96, 136) are solved as a zero-bordered order-136 problem
JACOBI_MAX_C = 256                         # lrs_sym_eig_jacobi_f64: one cluster, columns in distributed shared memory
JACOBI_AUTO_C = 192                        # solver='auto' takes the Jacobi kernel up to this order (scripts/jacobi_time.py:
#                                            0.19 / 0.35 / 0.83 / 1.61 ms against 0.34 / 1.00 / 1.14-1.22 / 1.72 ms of syevd at C = 31 / 64 / 128 / 191,
#                                            and no host synchronisation; at C = 224 / 256 the library is faster: 2.33 / 2.96 vs 2.06 / 2.42 ms)

_DIVERGED = ("SVT: the band Gram matrix of X + lambda_2/mu_2 is not finite — the ADMM state has diverged "
             "(the reference's update lambda_1 += mu_1*(X - IMout) uses the overlap SUM, main_LRS_PnP.py:346,361; "
             "with stride-1 overlap it grows geometrically and overflows fp32 after ~20 outer iterations)")


def raise_for_eig_status(status) -> None:
    """``status`` = the three host ints of lrs_sym_eig_jacobi_f64: sweeps, not-converged flag, non-finite flag."""
    sweeps, unconverged, nonfinite = (int(v) for v in status)
    if nonfinite:
        raise _lib.LrsError(_DIVERGED)
    if unconverged:
        raise _lib.LrsError(f"SVT: the Jacobi eigensolver still rotated after {sweeps} sweeps")


def sym_eig_jacobi(G: torch.Tensor):
    """(lam [C], Bt [C, C], status [3] int32) of lrs_sym_eig_jacobi_f64 for a symmetric PSD fp64 matrix on the device:
    row k of Bt is lam[k] * v_k.  No host synchronisation."""
    C = G.shape[0]
    if G.dtype != torch.float64 or G.shape != (C, C) or not 1 <= C <= JACOBI_MAX_C:
        raise ValueError("sym_eig_jacobi needs a square fp64 matrix of order 1..256")
    G = G.contiguous()
    lam = torch.empty(C, dtype=torch.float64, device=G.device)
    Bt = torch.empty((C, C), dtype=torch.float64, device=G.device)
    status = torch.empty(3, dtype=torch.int32, device=G.device)
    check(lib().lrs_sym_eig_jacobi_f64(ptr(G), C, ptr(lam), ptr(Bt), ptr(status), stream_ptr()), "lrs_sym_eig_jacobi_f64")
    return lam, Bt, status


def sym_eig_jacobi_batch(G: torch.Tensor):
    """(lam [B, C], Bt [B, C, C], status [B, 3] int32) of lrs_sym_eig_jacobi_batch_f64 for B symmetric PSD fp64 matrices
    ``G [B, C, C]``; slice b is what :func:`sym_eig_jacobi` gives for ``G[b]``.  No host synchronisation."""
    B, C = G.shape[0], G.shape[-1]
    if G.dtype != torch.float64 or G.dim() != 3 or G.shape[1] != C or not 1 <= C <= JACOBI_MAX_C:
        raise ValueError("sym_eig_jacobi_batch needs [B, C, C] fp64 matrices of order 1..256")
    G = G.contiguous()
    lam = torch.empty((B, C), dtype=torch.float64, device=G.device)
    Bt = torch.empty((B, C, C), dtype=torch.float64, device=G.device)
    status = torch.empty((B, 3), dtype=torch.int32, device=G.device)
    check(lib().lrs_sym_eig_jacobi_batch_f64(ptr(G), B, C, ptr(lam), ptr(Bt), ptr(status), stream_ptr()),
          "lrs_sym_eig_jacobi_batch_f64")
    return lam, Bt, status


def eig_status_failures(status) -> Tuple[list, list]:
    """Cubes (indices) whose eigensolve met a non-finite Gram matrix, and those that did not converge, from the host
    status words ``[B, 3]`` of :func:`sym_eig_jacobi_batch`."""
    st = np.asarray(status).reshape(-1, 3)
    return [int(b) for b in np.flatnonzero(st[:, 2])], [int(b) for b in np.flatnonzero((st[:, 1] != 0) & (st[:, 2] == 0))]


def svt_weights_batch(G: torch.Tensor, tau: float, solver: str = "auto", status_sink=None) -> torch.Tensor:
    """W [B, C, C] of :func:`svt_weights` for each of the B Gram matrices ``G [B, C, C]``.  'jacobi' (auto up to
    JACOBI_AUTO_C): one launch of the batched cluster eigensolver, status words [B, 3] handed to ``status_sink`` (None:
    checked here); 'library': torch.linalg.eigh on the batch (synchronises)."""
    B, C = G.shape[0], G.shape[-1]
    if solver == "auto":
        solver = "jacobi" if C <= JACOBI_AUTO_C else "library"
    W = torch.empty((B, C, C), dtype=torch.float32, device=G.device)
    if solver == "jacobi":
        lam, Bt, status = sym_eig_jacobi_batch(G)
        check(lib().lrs_svt_weights_batch_f64(ptr(lam), ptr(Bt), C * C, 1, C, B, C, C, float(tau), 1, ptr(W), stream_ptr()),
              "lrs_svt_weights_batch_f64")
        if status_sink is None:
            raise_for_batch_status(status.cpu())
        else:
            status_sink(status)
        return W
    if solver != "library":
        raise ValueError(solver)
    try:
        evals, V = torch.linalg.eigh(G)
    except RuntimeError as e:
        fin = torch.isfinite(G).flatten(1).all(1).cpu()
        bad = [b for b in range(B) if not bool(fin[b])]
        raise _lib.LrsError(f"cube(s) {bad}: {_DIVERGED}" if bad else f"SVT: batched eigh failed: {e}") from e
    fin = torch.isfinite(evals).all(1).cpu()              # eigh has synchronised on its status words already
    bad = [b for b in range(B) if not bool(fin[b])]
    if bad:
        raise _lib.LrsError(f"cube(s) {bad}: {_DIVERGED}")
    check(lib().lrs_svt_weights_batch_f64(ptr(evals), ptr(V), V.stride(0), V.stride(1), V.stride(2), B, C, C, float(tau), 0,
                                          ptr(W), stream_ptr()), "lrs_svt_weights_batch_f64")
    return W


def raise_for_batch_status(status) -> None:
    """Raise naming the cubes of a batch whose eigensolve met a non-finite Gram matrix or did not converge (host status
    words [B, 3])."""
    nonfinite, unconverged = eig_status_failures(status)
    if nonfinite:
        raise _lib.LrsError(f"cube(s) {nonfinite}: {_DIVERGED}")
    if unconverged:
        raise _lib.LrsError(f"cube(s) {unconverged}: SVT: the Jacobi eigensolver did not converge")


def svt_weights(G: torch.Tensor, tau: float, solver: str = "auto", status_sink=None) -> torch.Tensor:
    """W = V diag(max(1 - tau/sigma, 0)) Vᵀ from the fp64 Gram matrix (σ² = eig).

    ``solver``: 'jacobi' = the cluster Jacobi kernel (C <= 256, one launch, no host synchronisation), 'library' =
    torch.linalg.eigh (cuSOLVER syevd, synchronises on its status word), 'auto' = jacobi up to JACOBI_AUTO_C bands.
    ``status_sink``: with the Jacobi solver the device status words are handed to this callable instead of being read
    back here (the ADMM driver looks at them later, without stalling the step); None = check now (one small copy)."""
    C = G.shape[0]
    if solver == "auto":
        solver = "jacobi" if C <= JACOBI_AUTO_C else "library"
    W = torch.empty((C, C), dtype=torch.float32, device=G.device)
    if solver == "jacobi":
        lam, Bt, status = sym_eig_jacobi(G)
        check(lib().lrs_svt_weights_f64(ptr(lam), ptr(Bt), 1, C, C, C, float(tau), 1, ptr(W), stream_ptr()), "lrs_svt_weights_f64")
        if status_sink is None:
            raise_for_eig_status(status.cpu())
        else:
            status_sink(status)
        return W
    if solver != "library":
        raise ValueError(solver)
    G0 = G
    if _EIGH_PAD_FROM <= C < _EIGH_PAD_TO:
        # cuSOLVER's syevd back-transforms the eigenvectors of orders <= ~128 with unblocked gemv/gerc pairs (126 pairs,
        # 1.3 of the 2.1 ms at C = 128, scripts/eigh_time.py); from order 136 on it takes the blocked path (1.1 ms).  A
        # zero border adds decoupled zero eigenvalues, whose weight is 0 (sigma = 0 <= tau): W's leading block is unchanged.
        Gp = torch.zeros((_EIGH_PAD_TO, _EIGH_PAD_TO), dtype=G.dtype, device=G.device)
        Gp[:C, :C] = G
        G = Gp
    try:
        evals, V = torch.linalg.eigh(G)
    except RuntimeError as e:                       # torch.linalg.LinAlgError is a RuntimeError
        if not bool(torch.isfinite(G0).all()):      # name the real cause
            raise _lib.LrsError(_DIVERGED) from e
        raise _lib.LrsError(f"SVT: eigh of the {C}x{C} band Gram matrix failed: {e}") from e
    # eigh has synchronised on its status word: the eigenvalues are ready, reading them back costs one small copy
    if not bool(torch.isfinite(evals.cpu()).all()):
        raise _lib.LrsError(_DIVERGED)
    check(lib().lrs_svt_weights_f64(ptr(evals), ptr(V), V.stride(0), V.stride(1), C, G.shape[0], float(tau), 0, ptr(W),
                                    stream_ptr()), "lrs_svt_weights_f64")
    return W


def svt_device(X: torch.Tensor, tau: float, lambda_2: Optional[torch.Tensor] = None, c: float = 0.0,
               gram_reduce=None) -> torch.Tensor:
    """SVT(X + c*lambda_2, tau) for tall-skinny matrices: fp64 Gram (lrs_gram_f64) → eigh of the
    C×C matrix → fused recomposition (lrs_svt_apply_f32).  ``gram_reduce`` (optional) is applied
    to the Gram matrix before the eigh — the all-reduce hook of the sharded driver."""
    R, Cc = X.shape
    G = torch.zeros((Cc, Cc), dtype=torch.float64, device=X.device)
    check(lib().lrs_gram_f64(ptr(X), ptr(lambda_2), float(c), R, Cc, ptr(G), stream_ptr()), "lrs_gram_f64")
    if gram_reduce is not None:
        G = gram_reduce(G)
    W = svt_weights(G, float(tau))
    U = torch.empty_like(X)
    check(lib().lrs_svt_apply_f32(ptr(X), ptr(lambda_2), float(c), ptr(W), R, Cc, ptr(U), stream_ptr()), "lrs_svt_apply_f32")
    return U


def SVT(X, tau):
    """main_LRS_PnP.py:118-124."""
    Xd, src, _ = _to_dev(X)
    with torch.cuda.device(Xd.device):
        U = svt_device(Xd, float(tau))
    return _back(U, src)
