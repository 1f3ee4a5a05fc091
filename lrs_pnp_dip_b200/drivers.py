"""Drivers mirroring the reference's three entry scripts (SURVEY §8f-4), with arguments instead of the
hard-coded ``/home/s1809498/...`` paths:

    python -m lrs_pnp_dip_b200.drivers lrs_pnp  --data-dir <ref>/data --image img5 --mask fourth_mask
    python -m lrs_pnp_dip_b200.drivers lrs_pnp_dip --net skip   --reference-root <ref> ...
    python -m lrs_pnp_dip_b200.drivers lrs_pnp_dip --net 1lip   --reference-root <ref> ...
    python -m lrs_pnp_dip_b200.drivers lrs_pnp_batch --data-dir <ref>/data [--pairs base:fourth_mask,img2:second_mask]

``lrs_pnp_batch`` runs the same loop for many (image, mask) pairs at once (:class:`LRSPnPBatch`, one kernel of each
kind per outer iteration for all cubes): by default every bundled image against each of the four distinct masks.
``lrs_pnp`` is main_LRS_PnP.py:159-451 (ADMM with the sparse step, SVT and the closed-form X update on the
GPU, metrics printed per outer iteration).  ``lrs_pnp_dip`` is main_LRS_PnP_DIP_pro.py / _1-LiP.py: the same
loop with the low-rank step replaced by a deep image prior that stays the REFERENCE's own PyTorch module
(``models.skip`` / ``models.my_Lipschitz_Unet``, imported from ``--reference-root``); this package only
provides the training loop around it (:func:`dip_low_rank`, restating get_DIP_out :211-272 with its
variance-based early stop :74-102) and keeps every tensor on the device.

The dictionary ``trained_dictionary.mat`` is not part of the reference checkout; pass ``--dictionary`` or a
seeded synthetic one (K atoms) is used.  ``learn_dict`` trains a substitute on the patches of a clean cube
(:mod:`lrs_pnp_dip_b200.dictlearn`) and writes it in the format the scripts load:

    python -m lrs_pnp_dip_b200.drivers learn_dict --data-dir <ref>/data --image base --out trained_dictionary.mat
"""
from __future__ import annotations

import argparse
import os
import sys
from typing import Callable, List, Optional, Tuple

import numpy as np
import torch

from . import matio, metrics, synth
from .solver import LRSPnP, LRSPnPBatch, Params

PAIRS = {"base": ("low_rank_sparsity_noisy.mat", "low_rank_sparsity_clean.mat", "low_rank_sparsity_mask.mat"),
         "img2": ("low_rank_sparsity_noisy_img2.mat", "low_rank_sparsity_clean_img2.mat", "second_mask.mat"),
         "img3": ("low_rank_sparsity_noisy_img3.mat", "low_rank_sparsity_clean_img3.mat", "third_mask.mat"),
         "img4": ("low_rank_sparsity_noisy_img4.mat", "low_rank_sparsity_clean_img4.mat", "fourth_mask.mat"),
         "img5": ("low_rank_sparsity_noisy_img5.mat", "low_rank_sparsity_clean_img5.mat", "fourth_mask.mat")}


# the distinct masks of PAIRS (img5 shares img4's fourth mask), in the order of the images that own them
BATCH_MASKS = ("low_rank_sparsity_mask", "second_mask", "third_mask", "fourth_mask")


def batch_pairs(spec: Optional[str] = None) -> List[Tuple[str, str]]:
    """(image, mask) pairs of ``lrs_pnp_batch``: ``spec`` = "image:mask,image:mask,..." (mask names with or without
    ``.mat``), or None = every image of PAIRS against each of BATCH_MASKS (5 x 4 = 20 cubes, image-major)."""
    if spec is None:
        return [(img, m) for img in PAIRS for m in BATCH_MASKS]
    out = []
    for item in spec.split(","):
        img, sep, m = item.strip().partition(":")
        m = m[:-4] if m.endswith(".mat") else m
        if not sep or img not in PAIRS or m not in BATCH_MASKS:
            raise ValueError(f"bad pair {item!r}: expected image:mask with image in {sorted(PAIRS)} and mask in {BATCH_MASKS}")
        out.append((img, m))
    if not out:
        raise ValueError("no (image, mask) pair given")
    return out


def load_case(data_dir: str, image: str, mask: Optional[str] = None):
    """→ (noisy cube [1,B,d2,d3], clean cube, msk (1,1,d2,d3) uint8) as numpy arrays (main_LRS_PnP.py:170-192)."""
    noisy_f, clean_f, mask_f = PAIRS[image]
    if mask:
        mask_f = mask if mask.endswith(".mat") else mask + ".mat"
    noisy = matio.load_cube(os.path.join(data_dir, noisy_f))
    clean = matio.load_cube(os.path.join(data_dir, clean_f))
    msk = np.asarray(matio.loadmat_any(os.path.join(data_dir, mask_f))["msk"], dtype=np.uint8)
    return noisy, clean, msk


def load_dictionary(path: Optional[str], n: int, K: int) -> np.ndarray:
    """``Dictionary`` of trained_dictionary.mat (main_LRS_PnP.py:159-165) or the seeded synthetic stand-in."""
    if path and os.path.isfile(path):
        D = np.asarray(matio.loadmat_any(path)["Dictionary"], dtype=np.float32)
        if D.shape[0] != n:
            raise ValueError(f"dictionary has {D.shape[0]} rows, expected bb^2 = {n}")
        return np.ascontiguousarray(D)
    return synth.synthetic_dictionary(n, K, seed=0)


class EarlyStop:
    """Windowed-variance early stop of the DIP fit (main_LRS_PnP_DIP_pro.py:74-102): keep the last ``size``
    outputs; stop when their mean squared deviation from the window mean has not decreased for ``patience``
    checks."""

    def __init__(self, size: int = 30, patience: int = 60):
        self.size, self.patience = size, patience
        self.window: list = []
        self.best, self.wait = float("inf"), 0

    def update(self, out: torch.Tensor) -> bool:
        self.window.append(out.detach().reshape(-1).clone())
        if len(self.window) > self.size:
            self.window.pop(0)
        if len(self.window) < self.size:
            return False
        stack = torch.stack(self.window)
        var = float(((stack - stack.mean(0, keepdim=True)) ** 2).mean())      # mean_i myMetric(ave, img_i), :105-106
        if var < self.best:
            self.best, self.wait = var, 0
            return False
        self.wait += 1
        return self.wait >= self.patience


def dip_low_rank(net_factory: Callable[[], torch.nn.Module], target_cube: torch.Tensor, mask_bkg: torch.Tensor, d2: int,
                 d3: int, num_iter: int = 5000, lr: float = 0.1, buffer_size: int = 30, patience: int = 60):
    """``U = low_rank(Z)`` hook for :class:`LRSPnP` restating get_DIP_out (main_LRS_PnP_DIP_pro.py:211-272): a
    FRESH network per outer iteration, Adam(lr), loss = MSE(target*mask, net(Z_img)*mask), early stop on the
    windowed output variance.  Unlike the reference it returns the last output when the early stop never
    triggers within ``num_iter`` (the reference returns None there and crashes, SURVEY §3.4)."""

    def low_rank(Z: torch.Tensor) -> torch.Tensor:
        z_img = metrics.fold(Z, d2, d3)                                        # :412  (device, no CPU bounce)
        net = net_factory().to(Z.device)
        opt = torch.optim.Adam(net.parameters(), lr)
        es = EarlyStop(buffer_size, patience)
        out = z_img
        for _ in range(num_iter):
            opt.zero_grad()
            out = net(z_img)
            loss = torch.nn.functional.mse_loss(target_cube * mask_bkg, out * mask_bkg)   # :242
            loss.backward()
            opt.step()
            if es.update(out):
                break
        return metrics.unfold(out.detach())                                    # :419

    return low_rank


def reference_net_factory(reference_root: str, kind: str, bands: int) -> Callable[[], torch.nn.Module]:
    """The reference's own DIP modules (out of scope of this package): ``skip(128,128,[128]*5,...)``
    (main_LRS_PnP_DIP_pro.py:215-221) or ``my_Lipschitz_Unet(128,128,ln_lambda=1)`` (main_LRS_PnP_DIP_1-LiP.py:212-214)."""
    if not os.path.isdir(os.path.join(reference_root, "models")):
        raise FileNotFoundError(f"{reference_root}/models not found: the DIP networks are the reference's own modules")
    if reference_root not in sys.path:
        sys.path.insert(0, reference_root)
    if kind == "skip":
        from models.skip import skip  # type: ignore

        return lambda: skip(bands, bands, num_channels_down=[128] * 5, num_channels_up=[128] * 5, num_channels_skip=[128] * 5,
                            filter_size_up=3, filter_size_down=3, upsample_mode="nearest", filter_skip_size=1,
                            need_sigmoid=True, need_bias=True, pad="reflection", act_fun="LeakyReLU")
    if kind == "1lip":
        from models.my_Lipschitz_Unet import my_Lipschitz_Unet  # type: ignore

        return lambda: my_Lipschitz_Unet(bands, bands, ln_lambda=1)
    raise ValueError(kind)


def run(noisy: np.ndarray, clean: np.ndarray, msk: np.ndarray, D: np.ndarray, prm: Params, iteration_num: int,
        low_rank_factory=None, engine: str = "auto", device="cuda", log=print):
    """The outer loop of the scripts (main_LRS_PnP.py:250-451) with per-iteration MPSNR / MSSIM / state distances."""
    dev = torch.device(device)
    _, B, d2, d3 = noisy.shape
    Y = matio.unfold_cube(noisy)
    MtM = matio.unfold_mask(msk, B)
    clean_t, noisy_t = torch.from_numpy(clean).to(dev), torch.from_numpy(noisy).to(dev)
    low_rank = low_rank_factory(dev, noisy_t, torch.from_numpy(msk.astype(np.float32)).to(dev), d2, d3) if low_rank_factory else None
    sol = LRSPnP(Y, MtM, D, prm, low_rank=low_rank, engine=engine, device=dev)
    history = []
    log(f"input MPSNR {metrics.mpsnr(clean_t, noisy_t):.4f}  MSSIM {metrics.ssim(clean_t, noisy_t):.4f}")
    for itr in range(iteration_num):
        Xp, l1p, l2p = sol.X.clone(), sol.lambda_1.clone(), sol.lambda_2.clone()
        sol.step()
        img = metrics.fold(sol.X, d2, d3)
        rec = dict(iteration=itr, mpsnr=metrics.mpsnr(clean_t, img), mssim=metrics.ssim(clean_t, img),
                   dX=metrics.state_convergence(sol.X, Xp), dl1=metrics.state_convergence(sol.lambda_1, l1p),
                   dl2=metrics.state_convergence(sol.lambda_2, l2p))
        history.append(rec)
        log("Outer-Loop Iteration {iteration}: MPSNR {mpsnr:.4f}  MSSIM {mssim:.4f}  log|dX| {dX:.3f}  log|dλ1| {dl1:.3f}  "
            "log|dλ2| {dl2:.3f}".format(**rec))
    return sol, history


def load_pair(data_dir: str, image: str, mask: str):
    """Cube (image, mask) of a batch: the image's observed cube with the pixels missing in ``mask`` also zeroed
    (:func:`synth.cross_masked`) → (Y [R, C], MtM [R, C], clean cube [1, B, d2, d3])."""
    noisy, clean, _ = load_case(data_dir, image)
    msk = np.asarray(matio.loadmat_any(os.path.join(data_dir, mask + ".mat"))["msk"], dtype=np.uint8)
    Y, MtM = synth.cross_masked(matio.unfold_cube(noisy), matio.unfold_mask(msk, 1)[:, 0])
    return Y, MtM, clean


def run_batch(cases, D: np.ndarray, prm: Params, iteration_num: int, engine: str = "auto", device="cuda", log=print):
    """The outer loop for a batch of cubes of one shape: ``cases`` = [(label, Y [R, C], MtM [R, C], clean [1, B, d2, d3])],
    e.g. from :func:`batch_pairs` / :func:`load_pair`.  One :class:`LRSPnPBatch` runs them together; MPSNR / MSSIM of every
    cube are logged after each outer iteration.  Returns (solver, history) with history[it][b] = {mpsnr, mssim}."""
    dev = torch.device(device)
    labels = [c[0] for c in cases]
    Y = np.stack([c[1] for c in cases])
    MtM = np.stack([c[2] for c in cases])
    cleans = [torch.from_numpy(np.asarray(c[3], dtype=np.float32)).to(dev) for c in cases]
    _, _, d2, d3 = cases[0][3].shape
    sol = LRSPnPBatch(Y, MtM, D, prm, engine=engine, device=dev)
    history = []
    for itr in range(iteration_num):
        sol.step()
        rec = []
        for b, lab in enumerate(labels):
            img = metrics.fold(sol.X[b], d2, d3)
            rec.append(dict(cube=lab, mpsnr=metrics.mpsnr(cleans[b], img), mssim=metrics.ssim(cleans[b], img)))
        history.append(rec)
        log(f"Outer-Loop Iteration {itr}: " + "  ".join(f"{r['cube']} {r['mpsnr']:.4f}/{r['mssim']:.4f}" for r in rec))
    sol.validate()
    return sol, history


def main(argv=None):
    ap = argparse.ArgumentParser(prog="lrs_pnp_dip_b200.drivers", description=__doc__.split("\n\n")[0])
    sub = ap.add_subparsers(dest="cmd", required=True)
    for name in ("lrs_pnp", "lrs_pnp_dip"):
        p = sub.add_parser(name)
        p.add_argument("--data-dir", required=True)
        p.add_argument("--image", default="img5" if name == "lrs_pnp" else "base", choices=sorted(PAIRS))
        p.add_argument("--mask", default=None)
        p.add_argument("--dictionary", default=None)
        p.add_argument("--atoms", type=int, default=2592)
        p.add_argument("--iterations", type=int, default=2 if name == "lrs_pnp" else 250)
        p.add_argument("--engine", default="auto")
        p.add_argument("--denoiser", default="soft", choices=["soft", "nlm", "identity"])
        if name == "lrs_pnp_dip":
            p.add_argument("--net", default="skip", choices=["skip", "1lip"])
            p.add_argument("--reference-root", required=True)
            p.add_argument("--dip-iterations", type=int, default=5000)
    p = sub.add_parser("lrs_pnp_batch")
    p.add_argument("--data-dir", required=True)
    p.add_argument("--pairs", default=None, help="image:mask,... (default: every image x each of the four masks)")
    p.add_argument("--dictionary", default=None)
    p.add_argument("--atoms", type=int, default=2592)
    p.add_argument("--iterations", type=int, default=2)
    p.add_argument("--engine", default="auto")
    p.add_argument("--denoiser", default="soft", choices=["soft", "nlm", "identity"])
    p = sub.add_parser("learn_dict")
    p.add_argument("--data-dir", required=True)
    p.add_argument("--image", default="base", choices=sorted(PAIRS))
    p.add_argument("--out", required=True)
    p.add_argument("--atoms", type=int, default=2592)
    p.add_argument("--bb", type=int, default=36)
    p.add_argument("--stride", type=int, default=4)
    p.add_argument("--rounds", type=int, default=10)
    p.add_argument("--lambda-ista", type=float, default=0.1)
    p.add_argument("--iterations", type=int, default=40, help="ISTA iterations per round")
    a = ap.parse_args(argv)
    if a.cmd == "learn_dict":
        from . import dictlearn

        _, clean, _ = load_case(a.data_dir, a.image)
        Y = torch.tensor(matio.unfold_cube(clean)).cuda()
        patches = dictlearn.training_patches(Y, a.bb, a.stride)
        D, hist = dictlearn.learn_dictionary(patches, a.atoms, a.lambda_ista, a.iterations, a.rounds)
        dictlearn.save_dictionary(a.out, D)
        print(f"learned {tuple(D.shape)} dictionary from {patches.shape[1]} patches; relative error per round: "
              + " ".join(f"{h:.4f}" for h in hist))
        return
    bb = 36
    if a.cmd == "lrs_pnp_batch":
        cases = [(f"{img}+{m}",) + load_pair(a.data_dir, img, m) for img, m in batch_pairs(a.pairs)]
        D = load_dictionary(a.dictionary or os.path.join(a.data_dir, "trained_dictionary.mat"), bb * bb, a.atoms)
        run_batch(cases, D, Params(denoiser=a.denoiser), a.iterations, engine=a.engine)
        return
    noisy, clean, msk = load_case(a.data_dir, a.image, a.mask)
    D = load_dictionary(a.dictionary or os.path.join(a.data_dir, "trained_dictionary.mat"), bb * bb, a.atoms)
    if a.cmd == "lrs_pnp":
        prm = Params(denoiser=a.denoiser)                                      # main_LRS_PnP.py:218-238
        run(noisy, clean, msk, D, prm, a.iterations, engine=a.engine)
    else:
        prm = Params(mu_1=0.1, mu_2=0.1, Nit=100, step="frob4", denoiser=a.denoiser)   # main_LRS_PnP_DIP_pro.py:324-341
        factory = reference_net_factory(a.reference_root, a.net, noisy.shape[1])
        lrf = lambda dev, target, mask_bkg, d2, d3: dip_low_rank(factory, target, mask_bkg, d2, d3, a.dip_iterations)  # noqa: E731
        run(noisy, clean, msk, D, prm, a.iterations, low_rank_factory=lrf, engine=a.engine)


if __name__ == "__main__":
    main()
