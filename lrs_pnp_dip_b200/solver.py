"""Batched fast path of the ADMM outer iteration (the script body
main_LRS_PnP.py:244-362, identical in main_LRS_PnP_DIP_pro.py:355-456 and
main_LRS_PnP_DIP_1-LiP.py:347-448) on one B200, or on a row-stripe shard of
the unfolded matrix per rank (one process per GPU).

    coder  = SparseCoder(Y_observed, D, prm)           # once: masks, step constants
    solver = LRSPnP(Y_observed, MtM, D, prm)           # X = Y_observed, λ1 = λ2 = 0   (:218-229)
    solver.step()                                      # one outer iteration           (:250-362)

The low-rank step is SVT (main_LRS_PnP.py:315) by default; the DIP variants pass
``low_rank=callable(Z) -> U`` and keep their PyTorch network (out of scope here).

Sharding (SURVEY §8e): contiguous stripes of patch row-starts, each rank holding its
rows plus the ``bb-1`` rows of read halo that follow.  Per outer iteration: one
neighbour halo *reduce* of the partial overlap sums, one all-reduce of the C×C band
Gram matrix for the SVT, one neighbour halo *refresh* of X and λ1.  Stripes are
supported for ``slidingDis == 1`` (the multi-GPU configurations BASELINE.json
names); other strides run unsharded.
"""
from __future__ import annotations

import contextlib
from dataclasses import dataclass
from typing import Callable, Optional, Tuple

import numpy as np
import torch

from . import _lib, ops
from ._lib import check, lib, ptr, stream_ptr

FUSED_K = (64, 128, 192, 256)


def _on(t):
    """The C library launches on the CURRENT CUDA device and stream: make the tensor's device current."""
    if isinstance(t, torch.Tensor) and t.device.type == "cuda":
        return torch.cuda.device(t.device)
    return contextlib.nullcontext()


@dataclass
class Params:
    """Hyper-parameters, SURVEY Appendix C.  Defaults = main_LRS_PnP.py:218-238;
    DIP variants: mu_1 = mu_2 = 0.1, Nit = 100, step = 'frob4' (main_LRS_PnP_DIP_pro.py:324-341,190).

    ``step`` — the ISTA step constant a_p of each patch:
      'spectral'        ||M_p D||_2^2 (main_LRS_PnP.py:134).  On the fused engines it comes from the 256-entry row-pattern
                        table, which needs masks replicated over the bands (per-element masks are refused).
      'spectral_patch'  the same value from each patch's own 64-bit validity pattern, for ANY mask (bb <= 8): one fp64
                        Lanczos run per distinct pattern at construction (ops.patch_step_constants), 4 B per patch kept.
      'frob4'           4||M_p D||_F^2 (main_LRS_PnP_DIP_pro.py:190), a different step rule."""
    gamma: float = 0.5
    mu_1: float = 0.15
    mu_2: float = 0.15 * 6
    lambda_ista: float = 0.1
    Nit: int = 80
    bb: int = 36
    slidingDis: int = 36
    step: str = "spectral"
    denoiser: str = "soft"      # 'soft' (ista.m:23) | 'nlm' (pnp_ista.m:30, explicit engine only) | 'identity'
    nlm_h_scale: float = 0.1    # h = nlm_h_scale * T


# --------------------------------------------------------------------------------------------------
# stripe partition (host logic, no device)
# --------------------------------------------------------------------------------------------------
def stripe_bounds(R: int, bb: int, world: int) -> np.ndarray:
    """Balanced split of the R-bb+1 patch row-starts (stride 1) into ``world`` contiguous stripes;
    returns world+1 boundaries a_0=0 < ... < a_world = R-bb+1."""
    n = R - bb + 1
    if n < world:
        raise ValueError(f"cannot split {n} patch rows over {world} ranks")
    return np.array([(n * g) // world for g in range(world + 1)], dtype=np.int64)


@dataclass
class Stripe:
    rank: int
    world: int
    R_total: int
    bb: int
    a: int          # first owned patch row-start (= first owned matrix row)
    b: int          # one past the last owned patch row-start

    @property
    def halo(self) -> int:            # rows read beyond the owned patch starts
        return self.bb - 1

    @property
    def rows_local(self) -> int:      # rows held: [a, b + bb - 1)
        return self.b - self.a + self.bb - 1

    @property
    def rows_owned(self) -> int:      # rows whose X/λ this rank updates
        return (self.R_total - self.a) if self.rank == self.world - 1 else (self.b - self.a)

    @property
    def row_slice(self) -> slice:
        return slice(self.a, self.a + self.rows_local)


def make_stripe(R: int, bb: int, rank: int, world: int) -> Stripe:
    bd = stripe_bounds(R, bb, world)
    if world > 1 and int(np.diff(bd).min()) < bb - 1:
        # halo_reduce / halo_refresh exchange the bb-1 halo rows with the IMMEDIATE neighbour only: a stripe that owns
        # fewer rows than the halo would need a multi-hop exchange (contributions would be lost silently otherwise)
        raise ValueError(f"row stripes of {int(np.diff(bd).min())} patch rows are narrower than the halo (bb-1 = {bb - 1}): "
                         f"use at most {(R - bb + 1) // (bb - 1)} ranks for R = {R}")
    return Stripe(rank=rank, world=world, R_total=R, bb=bb, a=int(bd[rank]), b=int(bd[rank + 1]))


# --------------------------------------------------------------------------------------------------
# sparse-coding step
# --------------------------------------------------------------------------------------------------
class _RangePipe:
    """Per-device resources of the range-wise overlap sum (SparseCoder.imout): two side streams and two Phi_z range
    buffers, shared by every SparseCoder on the device.  Buffer i is only ever touched on stream i, so stream order
    alone serialises successive users; nothing is allocated or created per call."""

    def __init__(self, device):
        self.device = device
        self.streams = [torch.cuda.Stream(device=device) for _ in range(2)]
        self.bufs = None

    def buffers(self, numel: int):
        if self.bufs is None or self.bufs[0].numel() < numel:
            for st in self.streams:              # growing (rare): pending work on the old buffers must finish first
                st.synchronize()
            self.bufs = None
            self.bufs = [torch.empty(numel, dtype=torch.float32, device=self.device) for _ in range(2)]
        return self.bufs


_RANGE_PIPES: dict = {}


def _range_pipe(device) -> _RangePipe:
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _RANGE_PIPES:
        _RANGE_PIPES[key] = _RangePipe(torch.device("cuda", key))
    return _RANGE_PIPES[key]


_SIDE_STREAMS: dict = {}


def _side_stream(device) -> "torch.cuda.Stream":
    """One extra stream per device for the low-rank step that runs beside the explicit sparse step (LRSPnP._step)."""
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _SIDE_STREAMS:
        # high priority: its few CTAs (the 8-CTA eigensolver cluster) are placed before the sparse step's persistent grid
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=torch.device("cuda", key), priority=-1)
    return _SIDE_STREAMS[key]


class SparseCoder:
    """Everything of the sparse step that depends only on (Y_observed, D, geometry): the per-patch
    validity masks (``blocks_copy == 0``, main_LRS_PnP.py:244,276-280) and the ISTA step constants,
    which the reference recomputes for every patch in every outer iteration (:134)."""

    def __init__(self, Y_observed: torch.Tensor, D: torch.Tensor, prm: Params, engine: str = "auto",
                 defer_validation: bool = False):
        """``defer_validation``: do not wait for the device-side input test (band-replicated masks for the
        spectral table) at construction; its verdict is checked around the launches and by :meth:`validate`."""
        with _on(Y_observed):
            self._init(Y_observed, D, prm, engine)
            if not defer_validation:
                self.validate()

    def _init(self, Y_observed: torch.Tensor, D: torch.Tensor, prm: Params, engine: str):
        if prm.step == "spectral_patch" and prm.bb > 8:
            raise ValueError(f"step='spectral_patch' packs a patch's mask into 64 bits and needs bb <= 8 (got bb = {prm.bb}); "
                             "use step='spectral' for explicit patch matrices")
        _lib.require_cuda()
        if Y_observed.device.type != "cuda" or D.device.type != "cuda":
            raise _lib.LrsError("SparseCoder needs CUDA tensors")
        self.Y = Y_observed.contiguous().float()
        self.D = D.contiguous().float()
        self.prm = prm
        self.R, self.C = self.Y.shape
        self.n, self.K = self.D.shape
        if self.n != prm.bb * prm.bb:
            raise ValueError(f"dictionary has {self.n} rows, bb² = {prm.bb * prm.bb}")
        self.P = ops.patch_count(self.R, self.C, prm.bb, prm.slidingDis)
        self.engine = _lib.ENGINES[engine]
        self.fused = prm.bb == 8 and self.K in FUSED_K and prm.denoiser == "soft"
        self.a_patch = self.a_table = self.blocks_copy = None
        self._bad_event = self._bad_host = None
        if self.fused:
            if prm.step == "spectral":
                # The 256-entry table is indexed by the validity of the patch's 8 unfolded ROWS, which needs masks
                # replicated over the bands (main_LRS_PnP.py:188-192).  The test runs on the device and its verdict
                # travels to pinned host memory asynchronously: no host synchronisation here; the flag is looked at
                # (without waiting) around every launch and (waiting) by validate().
                obs = self.Y != 0
                self._bad_host = torch.empty((), dtype=torch.bool).pin_memory()
                self._bad_host.copy_((obs != obs[:, :1]).any(), non_blocking=True)
                self._bad_event = torch.cuda.Event()
                self._bad_event.record()
                self.a_table = ops.row_pattern_table(self.D, prm.bb, "spectral")
            elif prm.step == "spectral_patch":
                # any mask: one value per patch (the kernels' a_patch_dev, indexed by the global patch number)
                self.a_patch = ops.patch_step_constants(self.Y, self.D, prm.bb, prm.slidingDis, "spectral")
            elif prm.step != "frob4":
                raise ValueError(prm.step)
        else:
            self.blocks_copy = ops.im2col(self.Y, prm.bb, prm.slidingDis)
            if prm.step == "spectral_patch":
                self.a_patch = ops.patch_step_constants(self.Y, self.D, prm.bb, prm.slidingDis, "spectral")
            else:
                self.a_patch = ops.step_constants(self.blocks_copy, self.D, prm.step)

    def validate(self, wait: bool = True) -> None:
        """Raise if the construction-time mask test failed.  ``wait=False`` only looks at a verdict that has
        already arrived (no synchronisation)."""
        ev = self._bad_event
        if ev is None:
            return
        if wait:
            ev.synchronize()
        elif not ev.query():
            return
        self._bad_event = None
        if bool(self._bad_host):
            raise _lib.LrsError("spectral step constants on the fused path need band-replicated masks "
                                "(one validity flag per unfolded row); use step='spectral_patch' (the same spectral "
                                "constant per patch, for any mask) or step='frob4' (a different step rule)")

    def phi_z(self, X: torch.Tensor, lambda_1: Optional[torch.Tensor]) -> torch.Tensor:
        """Phi_z [n, P] of main_LRS_PnP.py:259-303 for V = X + lambda_1/mu_1."""
        with _on(X):
            self.validate(wait=False)
            out = self._phi_z(X, lambda_1)
            self.validate(wait=False)
            return out

    def _phi_z(self, X: torch.Tensor, lambda_1: Optional[torch.Tensor]) -> torch.Tensor:
        prm = self.prm
        if self.fused:
            return self._fused_range(X, lambda_1, 0, self.P)
        blocks = ops.im2col(X, prm.bb, prm.slidingDis, lambda_1, prm.mu_1)
        _, phi = ops.ista_batched(blocks, self.blocks_copy, self.D, self.a_patch, prm.lambda_ista, prm.Nit,
                                  denoiser=prm.denoiser, h_scale=prm.nlm_h_scale)
        return phi

    def _fused_range(self, X, lambda_1, p_begin: int, p_end: int, out: Optional[torch.Tensor] = None,
                     dynamic: bool = False) -> torch.Tensor:
        prm = self.prm
        if out is None:
            out = torch.empty((self.n, p_end - p_begin), dtype=torch.float32, device=X.device)
        check(lib().lrs_sparse_step_fused_f32(ptr(X), ptr(lambda_1), float(prm.mu_1), ptr(self.Y), ptr(self.D), self.K,
                                              ptr(self.a_patch), ptr(self.a_table), float(prm.lambda_ista), int(prm.Nit),
                                              self.R, self.C, prm.bb, prm.slidingDis, p_begin, p_end, ptr(out),
                                              self.engine | (_lib.ENGINE_DYNAMIC_TILES if dynamic else 0), stream_ptr()),
              "lrs_sparse_step_fused_f32")
        return out

    def phi_z_range(self, X: torch.Tensor, lambda_1: Optional[torch.Tensor], p_begin: int, p_end: int) -> torch.Tensor:
        """Phi_z columns [p_begin, p_end) only (patch numbering of main_LRS_PnP.py:94-99; fused engines)."""
        if not self.fused:
            raise _lib.LrsError("patch sub-ranges are served by the fused engines (bb = 8, K in 64/128/192/256, soft denoiser)")
        if not 0 <= p_begin < p_end <= self.P:
            raise ValueError(f"patch range [{p_begin}, {p_end}) outside [0, {self.P})")
        with _on(X):
            self.validate(wait=False)
            return self._fused_range(X, lambda_1, int(p_begin), int(p_end))

    # ---- overlap sum without materialising Phi_z ----
    # Patch order is column-start-outer (main_LRS_PnP.py:94-99), so the sequential fp32 overlap sum (:332-339) can be
    # continued range by range of column starts (lrs_col2im_accum_range_f32): only two ranges of Phi_z exist at a time.
    # Two streams alternate: the fused kernel of range k+1 starts on the SMs range k frees while the overlap sum of
    # range k runs; the sums themselves are chained by events because consecutive ranges share output columns.
    CHUNK_BYTES = 768 << 20          # per Phi_z range buffer (two buffers): cfg 4 -> 12 column starts, cfg 5 -> 3

    def _chunk_cols(self) -> int:
        nR = self.R - self.prm.bb + 1
        return max(1, int(self.CHUNK_BYTES // (nR * self.n * 4)))

    # A launch that shares the GPU with the eigensolver (shared_start) uses the dynamically dealt kernel instance, which
    # needs ~4 % more cycles: that first range is kept just long enough to cover the eigensolver (~2 ms), judged by the
    # kernel's rate on a B200.
    SHARED_START_SECONDS = 2.5e-3
    FUSED_PATCH_ITERS_PER_S = 6.7e9

    def _ranges(self, shared_start: bool = False):
        """Column-start ranges [(c0, c1), ...] of one sparse step, ascending and contiguous."""
        prm = self.prm
        nR, nC, cpc = self.R - prm.bb + 1, self.C - prm.bb + 1, self._chunk_cols()
        out, c0 = [], 0
        if shared_start:
            first = int(np.ceil(self.SHARED_START_SECONDS * self.FUSED_PATCH_ITERS_PER_S / (nR * max(prm.Nit, 1))))
            c0 = min(nC, max(1, min(cpc, first)))
            out.append((0, c0))
        while c0 < nC:
            out.append((c0, min(nC, c0 + cpc)))
            c0 += cpc
        return out

    def imout(self, X: torch.Tensor, lambda_1: Optional[torch.Tensor], shared_start: bool = False) -> torch.Tensor:
        """Overlap sum of the reconstructed patches (main_LRS_PnP.py:332-339).  ``shared_start``: another kernel holds a
        few SMs while the first launch starts (the eigensolver of the low-rank step): that launch claims its work items
        dynamically, so the CTAs that start late take fewer of them."""
        prm = self.prm
        with _on(X):
            nC = self.C - prm.bb + 1
            if not (self.fused and prm.slidingDis == 1) or self._chunk_cols() >= nC:
                self.validate(wait=False)
                phi = self._fused_range(X, lambda_1, 0, self.P, dynamic=shared_start) if self.fused else self._phi_z(X, lambda_1)
                return ops.col2im(phi, self.R, self.C, prm.bb, prm.slidingDis)
            self.validate(wait=False)
            nR, cpc = self.R - prm.bb + 1, self._chunk_cols()
            pipe = _range_pipe(X.device)
            bufs, streams = pipe.buffers(self.n * cpc * nR), pipe.streams
            out = torch.empty((self.R, self.C), dtype=torch.float32, device=X.device)
            main = torch.cuda.current_stream()
            ready = torch.cuda.Event()
            ready.record(main)
            prev_sum = None
            for k, (c0, c1) in enumerate(self._ranges(shared_start)):
                st = streams[k & 1]
                if k < 2:
                    st.wait_event(ready)                      # inputs (and `out`) are ready on the caller's stream
                with torch.cuda.stream(st):
                    buf = bufs[k & 1][:self.n * (c1 - c0) * nR].view(self.n, (c1 - c0) * nR)
                    self._fused_range(X, lambda_1, c0 * nR, c1 * nR, out=buf,   # buffer k&1 was released by sum k-2 (same stream)
                                      dynamic=shared_start and k == 0)
                    if prev_sum is not None:
                        st.wait_event(prev_sum)               # running sum: range k continues where range k-1 stopped
                    check(lib().lrs_col2im_accum_range_f32(ptr(buf), self.R, self.C, prm.bb, prm.slidingDis, c0, c1, ptr(out),
                                                           stream_ptr()), "lrs_col2im_accum_range_f32")
                    prev_sum = torch.cuda.Event()
                    prev_sum.record(st)
            for st in streams:
                main.wait_stream(st)
            self.validate(wait=False)
            return out


def sparse_step(X, lambda_1, mu_1, Y_observed, D, bb, slidingDis, lambda_ista, Nit, step="spectral", engine="auto",
                return_phi=False):
    """Functional form: (IMout, Weight[, Phi_z]) for one call (builds a SparseCoder each time)."""
    prm = Params(mu_1=mu_1, lambda_ista=lambda_ista, Nit=Nit, bb=bb, slidingDis=slidingDis, step=step)
    sc = SparseCoder(Y_observed, D, prm, engine)
    phi = sc.phi_z(X, lambda_1)
    im = ops.col2im(phi, sc.R, sc.C, bb, slidingDis)
    W = ops.coverage_weight(sc.R, sc.C, bb, slidingDis, device=X.device)
    return (im, W, phi) if return_phi else (im, W)


def admm_update(Y_observed, MtM, IMout, U, lambda_1, lambda_2, prm: Params, rows=None, row_offset=0, R_total=None, out=None):
    """X / λ update (main_LRS_PnP.py:346,361-362).  λ1, λ2 are updated in place; returns X (written into ``out`` — a
    contiguous [rows, C] fp32 tensor, e.g. the previous iterate, which the update does not read — when given)."""
    R, C = Y_observed.shape
    rows = R if rows is None else rows
    R_total = R if R_total is None else R_total
    if out is not None and (out.shape != (rows, C) or out.dtype != torch.float32 or not out.is_contiguous()):
        raise ValueError("out must be a contiguous float32 tensor of shape [rows, C]")
    X = out if out is not None else torch.empty((rows, C), dtype=torch.float32, device=Y_observed.device)
    check(lib().lrs_admm_update_f32(ptr(Y_observed), ptr(MtM), ptr(IMout), ptr(U), ptr(lambda_1), ptr(lambda_2), ptr(X),
                                    float(prm.gamma), float(prm.mu_1), float(prm.mu_2), rows, row_offset, R_total, C,
                                    prm.bb, prm.slidingDis, stream_ptr()), "lrs_admm_update_f32")
    return X


# --------------------------------------------------------------------------------------------------
# communication shim: the three exchanges of a sharded outer iteration
# --------------------------------------------------------------------------------------------------
class StripeComm:
    """Neighbour halo exchange + Gram all-reduce over torch.distributed (NCCL on GPUs, gloo in the
    CPU tests).  world == 1 → every method is a no-op."""

    def __init__(self, stripe: Stripe, group=None):
        self.st = stripe
        self.group = group

    def _exchange(self, send_to_right: Optional[torch.Tensor], send_to_left: Optional[torch.Tensor],
                  like: torch.Tensor) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
        """Send tensors to the right / left neighbour; returns (from_left, from_right)."""
        import torch.distributed as dist

        st = self.st
        ops_, from_left, from_right = [], None, None
        if send_to_right is not None and st.rank + 1 < st.world:
            ops_.append(dist.P2POp(dist.isend, send_to_right.contiguous(), st.rank + 1, self.group))
        if send_to_right is not None and st.rank > 0:
            from_left = torch.empty_like(like)
            ops_.append(dist.P2POp(dist.irecv, from_left, st.rank - 1, self.group))
        if send_to_left is not None and st.rank > 0:
            ops_.append(dist.P2POp(dist.isend, send_to_left.contiguous(), st.rank - 1, self.group))
        if send_to_left is not None and st.rank + 1 < st.world:
            from_right = torch.empty_like(like)
            ops_.append(dist.P2POp(dist.irecv, from_right, st.rank + 1, self.group))
        if ops_:
            for w in dist.batch_isend_irecv(ops_):
                w.wait()
        return from_left, from_right

    def halo_reduce(self, imout_local: torch.Tensor) -> None:
        """Partial overlap sums of the halo rows go to the right neighbour, which owns them."""
        st = self.st
        if st.world == 1 or st.halo == 0:
            return
        h = st.halo
        send = imout_local[st.rows_local - h:] if st.rank + 1 < st.world else None
        if st.rank + 1 < st.world or st.rank > 0:
            from_left, _ = self._exchange(send if send is not None else imout_local[:0], None, imout_local[:h])
            if from_left is not None:
                imout_local[:h] += from_left

    def halo_refresh(self, *arrays: torch.Tensor) -> None:
        """Owned first rows travel to the LEFT neighbour's halo (X and λ1 after the update): all arrays in ONE
        exchange (stacked into one message per neighbour)."""
        st = self.st
        if st.world == 1 or st.halo == 0 or not arrays:
            return
        h = st.halo
        send = torch.stack([arr[:h] for arr in arrays]) if st.rank > 0 else None
        like = torch.empty((len(arrays), h) + tuple(arrays[0].shape[1:]), dtype=arrays[0].dtype, device=arrays[0].device)
        _, from_right = self._exchange(None, send if send is not None else like[:0], like)
        if from_right is not None:
            for i, arr in enumerate(arrays):
                arr[st.rows_local - h:] = from_right[i]

    def allreduce_sum(self, t: torch.Tensor) -> torch.Tensor:
        if self.st.world > 1:
            import torch.distributed as dist

            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t


# --------------------------------------------------------------------------------------------------
# compute backend of one stripe (CUDA).  The CPU tests of the sharded driver substitute their own
# object with the same five methods; the product never does.
# --------------------------------------------------------------------------------------------------
class CudaBackend:
    def __init__(self, Y_local: torch.Tensor, MtM_local: torch.Tensor, D: torch.Tensor, prm: Params, engine="auto"):
        self.prm = prm
        self.Y, self.MtM = Y_local, MtM_local
        self.coder = SparseCoder(Y_local, D, prm, engine, defer_validation=True)
        self._pending: list = []

    def imout(self, X, lambda_1, shared_start=False):
        return self.coder.imout(X, lambda_1, shared_start=shared_start)

    def gram(self, X, lambda_2, c, rows):
        C = X.shape[1]
        G = torch.zeros((C, C), dtype=torch.float64, device=X.device)
        check(lib().lrs_gram_f64(ptr(X), ptr(lambda_2), float(c), rows, C, ptr(G), stream_ptr()), "lrs_gram_f64")
        return G

    def _defer_status(self, status: torch.Tensor) -> None:
        """Status words of the Jacobi eigensolver travel to pinned host memory behind the kernels that produced them;
        check_status() looks at them later (LRSPnP: at the next step and in validate()), so no step waits on the host."""
        host = torch.empty(3, dtype=torch.int32).pin_memory()
        host.copy_(status, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pending.append((host, ev))

    def check_status(self, wait: bool = False) -> None:
        while self._pending:
            host, ev = self._pending[0]
            if wait:
                ev.synchronize()
            elif not ev.query():
                return
            self._pending.pop(0)
            ops.raise_for_eig_status(host)

    def svt_weights(self, G, tau, solver="auto"):
        return ops.svt_weights(G, tau, solver=solver, status_sink=self._defer_status)

    def svt_apply(self, X, lambda_2, c, G, tau, rows, W=None):
        if W is None:
            W = self.svt_weights(G, tau)
        U = torch.empty((rows, X.shape[1]), dtype=torch.float32, device=X.device)
        check(lib().lrs_svt_apply_f32(ptr(X), ptr(lambda_2), float(c), ptr(W), rows, X.shape[1], ptr(U), stream_ptr()),
              "lrs_svt_apply_f32")
        return U

    def axpy(self, X, L, c, rows):
        out = torch.empty((rows, X.shape[1]), dtype=torch.float32, device=X.device)
        check(lib().lrs_axpy_f32(ptr(X), ptr(L), float(c), ptr(out), out.numel(), stream_ptr()), "lrs_axpy_f32")
        return out

    def admm_update(self, IMout, U, lambda_1, lambda_2, rows, row_offset, R_total, out=None):
        return admm_update(self.Y, self.MtM, IMout, U, lambda_1, lambda_2, self.prm, rows, row_offset, R_total, out=out)


class LRSPnP:
    """ADMM driver.  ``Y_observed`` / ``MtM`` are this rank's LOCAL rows (the whole matrix when
    unsharded).  ``low_rank``: None → SVT with τ = 1/μ2 (main_LRS_PnP.py:315); or a callable
    ``U = low_rank(Z)`` on this rank's owned rows (the DIP variants' network, kept in PyTorch)."""

    def __init__(self, Y_observed, MtM, D, prm: Params, low_rank: Optional[Callable] = None, engine: str = "auto",
                 stripe: Optional[Stripe] = None, group=None, backend=None, device=None):
        if backend is None:
            _lib.require_cuda()
            device = torch.device(device if device is not None else "cuda")
            Y_observed = torch.as_tensor(Y_observed, dtype=torch.float32).to(device).contiguous()
            MtM = torch.as_tensor(MtM, dtype=torch.float32).to(device).contiguous()
            D = torch.as_tensor(D, dtype=torch.float32).to(device).contiguous()
            backend = CudaBackend(Y_observed, MtM, D, prm, engine)
        self.be = backend
        self.prm = prm
        self.Y = Y_observed
        R_loc = Y_observed.shape[0]
        self.stripe = stripe if stripe is not None else Stripe(0, 1, R_loc, prm.bb, 0, R_loc - prm.bb + 1)
        if self.stripe.world > 1 and prm.slidingDis != 1:
            raise _lib.LrsError("row-stripe sharding is implemented for slidingDis == 1")
        if self.stripe.world > 1 and R_loc != self.stripe.rows_local:
            raise ValueError("Y_observed must hold exactly this rank's stripe rows (owned + halo)")
        self.comm = StripeComm(self.stripe, group)
        self.low_rank = low_rank
        self.X = Y_observed.clone()                      # X = Y_observed          (:229)
        self.lambda_1 = torch.zeros_like(Y_observed)     # (:219)
        self.lambda_2 = torch.zeros_like(Y_observed)     # (:220)
        self.iterations = 0
        # The low-rank step reads (X, λ2) and the sparse step reads (X, λ1): the two are independent until the X / λ
        # update (SURVEY §1, L2 ‖ L3).  With the explicit engine (a chain of short launches that leaves SMs idle) the
        # low-rank step — Gram, eigh, recomposition, or the caller's network — runs on a second stream beside it.  The
        # fused engines keep every SM busy with persistent CTAs (nothing could run beside them): sequential there.
        coder = getattr(backend, "coder", None)
        self.overlap_low_rank = (isinstance(backend, CudaBackend) and coder is not None and not coder.fused
                                 and self.stripe.world == 1)
        self._side = None
        self._late_inputs = None                         # from_host(): MtM / λ2 uploads still in flight on the side stream
        # Fused engines: the persistent grid leaves no SM for a whole low-rank step, but the Jacobi eigensolver needs only
        # 8 — it is launched (high-priority stream) right before the sparse step's first kernel and runs beside it; the
        # fused kernel claims its work items dynamically, so the 8 CTAs that start late just take fewer of them.
        # (Hidden, the Jacobi kernel is taken for every order it supports: beside a sparse step its 2.3 ms at 224 bands
        # cost nothing, the library's 2.1 ms plus a host synchronisation did.)
        self.hide_eigensolver = (isinstance(backend, CudaBackend) and coder is not None and coder.fused
                                 and low_rank is None and Y_observed.shape[1] <= ops.JACOBI_MAX_C)

    @classmethod
    def from_host(cls, Y_observed, MtM, D, prm: Params, state=None, device=None, **kw) -> "LRSPnP":
        """Solver for HOST inputs (pinned CPU tensors; ``state`` = optional ``(X, lambda_1, lambda_2)`` to resume from).
        What the sparse step needs (Y_observed, X, λ1) is uploaded on the caller's stream; MtM and λ2, which only the
        low-rank step and the X / λ update read, travel on a second stream while the sparse step already runs
        (:meth:`_step` waits for them where they are first used)."""
        _lib.require_cuda()
        device = torch.device(device if device is not None else "cuda")
        as_f32 = lambda t: torch.as_tensor(t, dtype=torch.float32)          # noqa: E731
        hY, hM = as_f32(Y_observed), as_f32(MtM)
        with torch.cuda.device(device):
            main = torch.cuda.current_stream()
            side = _side_stream(device)
            dY = hY.to(device, non_blocking=True)
            dM = torch.empty(hM.shape, dtype=torch.float32, device=device)
            side.wait_stream(main)                       # the blocks just handed out may have pending work of a former owner
            with torch.cuda.stream(side):
                dM.copy_(hM, non_blocking=True)
            self = cls(dY, dM, D, prm, device=device, **kw)
            if state is not None:
                hX, hL1, hL2 = (as_f32(t) for t in state)
                self.X.copy_(hX, non_blocking=True)
                self.lambda_1.copy_(hL1, non_blocking=True)
                side.wait_stream(main)                   # the constructor zero-filled λ2 on the caller's stream
                with torch.cuda.stream(side):
                    self.lambda_2.copy_(hL2, non_blocking=True)
            self._late_inputs = torch.cuda.Event()
            self._late_inputs.record(side)
        return self

    def to_host(self, X_out, lambda_1_out=None, lambda_2_out=None) -> None:
        """Asynchronous copies of the state into (pinned) host tensors on the current stream."""
        with _on(self.X):
            X_out.copy_(self.X, non_blocking=True)
            if lambda_1_out is not None:
                lambda_1_out.copy_(self.lambda_1, non_blocking=True)
            if lambda_2_out is not None:
                lambda_2_out.copy_(self.lambda_2, non_blocking=True)

    @property
    def rows_owned(self) -> int:
        return self.stripe.rows_owned if self.stripe.world > 1 else self.Y.shape[0]

    def reset(self) -> None:
        """Back to the reference's initial state: X = Y_observed, λ1 = λ2 = 0 (main_LRS_PnP.py:219-220,229).
        Three device copies/memsets on the current stream, no allocation."""
        with _on(self.X):
            self.X.copy_(self.Y)
            self.lambda_1.zero_()
            self.lambda_2.zero_()
        self.iterations = 0

    def step(self) -> None:
        with _on(self.X):
            self._step()

    def _step(self) -> None:
        prm, st, be = self.prm, self.stripe, self.be
        if hasattr(be, "check_status"):
            be.check_status(wait=False)                  # deferred eigensolver verdicts of earlier steps (no stall)
        own = self.rows_owned
        row_off = st.a if st.world > 1 else 0
        c = 1.0 / prm.mu_2

        def low_rank_step():
            # low-rank step on Z = X + (1/mu_2) lambda_2 (:315)
            if self.low_rank is None:
                G = self.comm.allreduce_sum(be.gram(self.X, self.lambda_2, c, own))
                return be.svt_apply(self.X, self.lambda_2, c, G, 1.0 / prm.mu_2, own)
            return self.low_rank(be.axpy(self.X, self.lambda_2, c, own))

        if self.overlap_low_rank:
            main = torch.cuda.current_stream()
            if self._side is None:
                self._side = _side_stream(self.X.device)
            self._side.wait_stream(main)                 # X, λ2 as the previous iteration left them
            # The SVT through the Jacobi kernel never blocks the host: it is enqueued first and runs from the start of the
            # sparse step.  A caller's network or the library eigensolver may block (early stop, status word): then the
            # sparse step is enqueued first.
            lr_async = self.low_rank is None and self.X.shape[1] <= ops.JACOBI_AUTO_C
            if lr_async:
                with torch.cuda.stream(self._side):
                    U = low_rank_step()                  # (the side stream also carried the late uploads: in order)
            IMout = be.imout(self.X, self.lambda_1)
            if not lr_async:
                with torch.cuda.stream(self._side):
                    U = low_rank_step()
            main.wait_stream(self._side)
            U.record_stream(main)                        # allocated on the side stream, consumed on the caller's
        elif self.hide_eigensolver and self.low_rank is None and self._late_inputs is None:
            # Gram (+ all-reduce) first, then the eigensolver on the side stream beside the whole sparse step; the
            # recomposition follows the sparse step on the caller's stream.  (Right after from_host() λ2 is still being
            # uploaded beside the sparse step: that one iteration keeps the sequential order below.)
            main = torch.cuda.current_stream()
            if self._side is None:
                self._side = _side_stream(self.X.device)
            G = self.comm.allreduce_sum(be.gram(self.X, self.lambda_2, c, own))
            self._side.wait_stream(main)
            with torch.cuda.stream(self._side):
                W = be.svt_weights(G, 1.0 / prm.mu_2, solver="jacobi")
            IMout = be.imout(self.X, self.lambda_1, shared_start=True)   # first launch behind the eigensolver's: dynamic deal
            self.comm.halo_reduce(IMout)
            main.wait_stream(self._side)
            W.record_stream(main)
            U = be.svt_apply(self.X, self.lambda_2, c, G, 1.0 / prm.mu_2, own, W=W)
        else:
            # sparse step + overlap sum on the local rows (:259-303, :332-339)
            IMout = be.imout(self.X, self.lambda_1)
            self.comm.halo_reduce(IMout)
            if self._late_inputs is not None:
                torch.cuda.current_stream().wait_event(self._late_inputs)     # MtM, λ2 of from_host()
            U = low_rank_step()
        # closed-form X, multipliers (:346, :361-362) on the owned rows
        self._late_inputs = None                         # every later use is ordered behind this step on the caller's stream
        if isinstance(be, CudaBackend):                 # the new iterate goes straight into X (the update never reads X)
            be.admm_update(IMout, U, self.lambda_1, self.lambda_2, own, row_off, st.R_total, out=self.X[:own])
        else:
            self.X[:own] = be.admm_update(IMout, U, self.lambda_1, self.lambda_2, own, row_off, st.R_total)
        self.comm.halo_refresh(self.X, self.lambda_1)
        self.iterations += 1

    def validate(self) -> None:
        """Wait for and check the deferred device-side input tests (see SparseCoder.validate)."""
        coder = getattr(self.be, "coder", None)
        if coder is not None:
            coder.validate()
        if hasattr(self.be, "check_status"):
            self.be.check_status(wait=True)

    def run(self, iteration_num: int) -> "LRSPnP":
        for _ in range(iteration_num):
            self.step()
        self.validate()
        return self


# --------------------------------------------------------------------------------------------------
# a batch of same-shape cubes in one ADMM loop (explicit engine)
# --------------------------------------------------------------------------------------------------
def _batch_inputs(Y_observed, MtM, D, prm: Params, low_rank, engine: str):
    """Host-side checks of LRSPnPBatch's inputs (no device needed): returns (Y, MtM, D) as tensors, not yet moved."""
    if low_rank is not None:
        raise _lib.LrsError("LRSPnPBatch runs the SVT low-rank step only; a low_rank callable (a DIP network) needs one "
                            "LRSPnP per cube")
    if prm.step == "spectral_patch":
        raise _lib.LrsError("LRSPnPBatch serves explicit patch matrices: step='spectral_patch' (bb <= 8 fused engines) is "
                            "not supported; use step='spectral' or 'frob4', or one LRSPnP per cube")
    if prm.step not in ("spectral", "frob4"):
        raise ValueError(f"unknown step mode {prm.step!r}")
    if prm.denoiser not in _lib.DENOISERS:
        raise ValueError(f"unknown denoiser {prm.denoiser!r}")
    if engine not in _lib.ENGINES:
        raise ValueError(f"unknown engine {engine!r}")
    Y, M, Dt = (torch.as_tensor(a) for a in (Y_observed, MtM, D))
    if Y.dim() != 3 or tuple(M.shape) != tuple(Y.shape):
        raise ValueError(f"Y_observed and MtM must both be [B, R, C] (got {tuple(Y.shape)} and {tuple(M.shape)})")
    if Y.dtype != M.dtype or not Y.dtype.is_floating_point:
        raise ValueError(f"Y_observed and MtM must share one floating-point dtype (got {Y.dtype} and {M.dtype})")
    if Dt.dim() != 2 or not Dt.dtype.is_floating_point:
        raise ValueError("D must be a floating-point [bb², K] matrix")
    B, R, C = Y.shape
    if not 1 <= B <= _lib.MAX_BATCH:
        raise ValueError(f"a batch holds 1..{_lib.MAX_BATCH} cubes (got B = {B})")
    if prm.bb < 1 or prm.slidingDis < 1 or prm.bb > min(R, C):
        raise ValueError(f"invalid geometry: R={R} C={C} bb={prm.bb} stride={prm.slidingDis}")
    if Dt.shape[0] != prm.bb * prm.bb:
        raise ValueError(f"dictionary has {Dt.shape[0]} rows, bb² = {prm.bb * prm.bb}")
    if prm.bb == 8 and Dt.shape[1] in FUSED_K and prm.denoiser == "soft":
        raise _lib.LrsError(f"bb = 8, K = {Dt.shape[1]} with the soft denoiser runs on the fused engines, which fill the GPU "
                            "from one cube: use one LRSPnP per cube (LRSPnPBatch serves the explicit engine)")
    return Y, M, Dt


class BatchSparseCoder:
    """The sparse step of B cubes of one geometry as ONE explicit-engine problem: the patch matrices of all cubes side by
    side ([n, B*P], cube b in columns [b*P, (b+1)*P)), one ISTA call over all B*P columns, one overlap sum per cube.
    Step constants come from the concatenated observed patches (patterns shared between cubes: one eigensolve)."""

    def __init__(self, Y_observed: torch.Tensor, D: torch.Tensor, prm: Params):
        self.Y, self.D, self.prm = Y_observed, D, prm
        self.B, self.R, self.C = Y_observed.shape
        self.n, self.K = D.shape
        self.P = ops.patch_count(self.R, self.C, prm.bb, prm.slidingDis)
        self.fused = False
        self.blocks_copy = ops.im2col_batch(self.Y, prm.bb, prm.slidingDis)
        try:
            self.a_patch = ops.step_constants(self.blocks_copy, self.D, prm.step)
        except _lib.LrsError as e:        # too many distinct patterns; a batch takes no explicit step constants
            raise _lib.LrsError(f"a batch of {self.B} cubes: {e.args[0].split(':')[0]}, more than the "
                                f"{ops.MAX_SPECTRAL_PATTERNS} that spectral step constants serve (one eigensolve each); use "
                                "step='frob4', or fewer cubes per batch") from e

    def phi_z(self, X: torch.Tensor, lambda_1: Optional[torch.Tensor]) -> torch.Tensor:
        """Phi_z [n, B*P] of main_LRS_PnP.py:259-303 for V = X + lambda_1/mu_1 of every cube."""
        prm = self.prm
        with _on(X):
            blocks = ops.im2col_batch(X, prm.bb, prm.slidingDis, lambda_1, prm.mu_1)
            _, phi = ops.ista_batched(blocks, self.blocks_copy, self.D, self.a_patch, prm.lambda_ista, prm.Nit,
                                      denoiser=prm.denoiser, h_scale=prm.nlm_h_scale)
            return phi

    def imout(self, X: torch.Tensor, lambda_1: Optional[torch.Tensor]) -> torch.Tensor:
        """Overlap sums [B, R, C] (main_LRS_PnP.py:332-339) of every cube."""
        with _on(X):
            return ops.col2im_batch(self.phi_z(X, lambda_1), self.B, self.R, self.C, self.prm.bb, self.prm.slidingDis)


class LRSPnPBatch:
    """ADMM driver for B cubes that share one dictionary, one Params and one geometry: ``Y_observed``, ``MtM`` are
    [B, R, C] and so are ``X``, ``lambda_1``, ``lambda_2``.  Cube b evolves as ``LRSPnP`` would evolve it alone; the
    batch runs each kernel of an outer iteration once for all cubes.  Served on the explicit engine (shapes where
    ``SparseCoder.fused`` is false) with the SVT low-rank step, on one GPU."""

    def __init__(self, Y_observed, MtM, D, prm: Params, engine: str = "auto", device=None, low_rank=None):
        Y, M, Dt = _batch_inputs(Y_observed, MtM, D, prm, low_rank, engine)
        _lib.require_cuda()
        device = torch.device(device if device is not None else "cuda")
        self.prm, self.engine = prm, engine
        with torch.cuda.device(device):
            self.Y = Y.to(device=device, dtype=torch.float32).contiguous()
            self.MtM = M.to(device=device, dtype=torch.float32).contiguous()
            self.D = Dt.to(device=device, dtype=torch.float32).contiguous()
            self.coder = BatchSparseCoder(self.Y, self.D, prm)
            self.X = self.Y.clone()                          # X = Y_observed          (:229)
            self.lambda_1 = torch.zeros_like(self.Y)         # (:219)
            self.lambda_2 = torch.zeros_like(self.Y)         # (:220)
        self.B, self.R, self.C = self.Y.shape
        self.iterations = 0
        self._side = None
        self._pending: list = []

    def reset(self) -> None:
        """Every cube back to X = Y_observed, λ1 = λ2 = 0 (main_LRS_PnP.py:219-220,229), on the current stream."""
        with _on(self.X):
            self.X.copy_(self.Y)
            self.lambda_1.zero_()
            self.lambda_2.zero_()
        self.iterations = 0

    def _defer_status(self, status: torch.Tensor) -> None:
        """Jacobi status words [B, 3] travel to pinned host memory behind the kernels that produced them (no stall)."""
        host = torch.empty(tuple(status.shape), dtype=torch.int32).pin_memory()
        host.copy_(status, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pending.append((host, ev))

    def _check_status(self, wait: bool) -> None:
        while self._pending:
            host, ev = self._pending[0]
            if wait:
                ev.synchronize()
            elif not ev.query():
                return
            self._pending.pop(0)
            ops.raise_for_batch_status(host.numpy())

    def _low_rank(self) -> torch.Tensor:
        """SVT of Z_b = X_b + λ2_b/μ2 with τ = 1/μ2 for every cube (main_LRS_PnP.py:315) on the current stream."""
        c = 1.0 / self.prm.mu_2
        B, R, C = self.B, self.R, self.C
        G = torch.zeros((B, C, C), dtype=torch.float64, device=self.X.device)
        check(lib().lrs_gram_batch_f64(ptr(self.X), ptr(self.lambda_2), float(c), B, R, C, ptr(G), stream_ptr()),
              "lrs_gram_batch_f64")
        W = ops.svt_weights_batch(G, c, status_sink=self._defer_status)
        U = torch.empty_like(self.X)
        check(lib().lrs_svt_apply_batch_f32(ptr(self.X), ptr(self.lambda_2), float(c), ptr(W), B, R, C, ptr(U), stream_ptr()),
              "lrs_svt_apply_batch_f32")
        return U

    def step(self) -> None:
        """One outer iteration (main_LRS_PnP.py:259-362) of every cube."""
        with _on(self.X):
            self._step()

    def _step(self) -> None:
        prm = self.prm
        self._check_status(wait=False)                   # deferred eigensolver verdicts of earlier steps (no stall)
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = _side_stream(self.X.device)
        # as LRSPnP's explicit path: the low-rank step runs on the side stream beside the sparse step; with the Jacobi
        # eigensolver it never blocks the host and is enqueued first, the library eigensolver synchronises and goes second
        self._side.wait_stream(main)
        lr_async = self.C <= ops.JACOBI_AUTO_C
        if lr_async:
            with torch.cuda.stream(self._side):
                U = self._low_rank()
        IMout = self.coder.imout(self.X, self.lambda_1)
        if not lr_async:
            with torch.cuda.stream(self._side):
                U = self._low_rank()
        main.wait_stream(self._side)
        U.record_stream(main)
        check(lib().lrs_admm_update_batch_f32(ptr(self.Y), ptr(self.MtM), ptr(IMout), ptr(U), ptr(self.lambda_1),
                                              ptr(self.lambda_2), ptr(self.X), float(prm.gamma), float(prm.mu_1),
                                              float(prm.mu_2), self.B, self.R, self.C, prm.bb, prm.slidingDis, stream_ptr()),
              "lrs_admm_update_batch_f32")
        self.iterations += 1

    def validate(self) -> None:
        """Wait for the deferred eigensolver verdicts; raise naming the cube(s) whose eigensolve met a non-finite Gram
        matrix (a diverged state) or did not converge."""
        self._check_status(wait=True)

    def run(self, iteration_num: int) -> "LRSPnPBatch":
        for _ in range(iteration_num):
            self.step()
        self.validate()
        return self
