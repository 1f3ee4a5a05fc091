"""lrs_pnp_dip_b200 — B200 (sm_100a) implementation of the data-parallel hot path of
shuoli0708/LRS-PnP-DIP: patch extraction → masked soft-ISTA against a dictionary →
overlap-sum reconstruction → closed-form ADMM update (+ SVT), behind the reference's own
Python call signatures.  Kernels live in ``csrc/`` (C ABI: ``include/lrs_pnp.h``).

Drop-in names (same signatures as main_LRS_PnP.py / admm_utils.py):
    get_image_block, ista, delete_element, soft_thresh, Shrinkage_Operator, SVT, l1_prox
Batched fast path replacing the script body of the outer iteration:
    SparseCoder, sparse_step, admm_update, LRSPnP, Params
B same-shape cubes in one ADMM loop (explicit engine):
    LRSPnPBatch
Metrics on the device (reference formulas): metrics.mpsnr / ssim / state_convergence.
Drivers mirroring the three entry scripts: python -m lrs_pnp_dip_b200.drivers {lrs_pnp,lrs_pnp_dip,learn_dict}.
"""
from ._lib import LIB_PATH, LrsError  # noqa: F401
from .ops import (SVT, Shrinkage_Operator, col2im, col2im_batch, coverage_weight, delete_element, get_image_block, im2col, im2col_batch,  # noqa: F401
                  ista, ista_batched, l1_prox, patch_count, patch_grid, soft_thresh, step_constants, svt_device)
from .solver import LRSPnP, LRSPnPBatch, Params, SparseCoder, Stripe, admm_update, make_stripe, sparse_step, stripe_bounds  # noqa: F401

from . import dictlearn, drivers, matio, metrics, synth  # noqa: E402,F401

__version__ = "0.1.0"
