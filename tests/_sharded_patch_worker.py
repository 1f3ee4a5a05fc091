"""torchrun worker for tests/test_patch_step_constants.py: sharded LRSPnP (NCCL) with per-element masks in
step='spectral_patch' == unsharded on rank 0.  Each rank builds the step constants of its own stripe."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lrs_pnp_dip_b200 as lrs  # noqa: E402
from lrs_pnp_dip_b200 import synth  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    H, W, B = 40, 33, 29
    clean, noisy = synth.synthetic_cube(H, W, B, rank=4, seed=7)
    m = synth.band_mask(H, W, B, keep=0.6, band_frac=0.5, dead_frac=0.2, seed=8).reshape(H * W, B)
    Y = synth.observe(noisy, m)
    MtM = m.astype(np.float32)
    D = synth.synthetic_dictionary(64, 256, seed=0)
    prm = lrs.Params(Nit=30, bb=8, slidingDis=1, step="spectral_patch")
    st = lrs.make_stripe(Y.shape[0], 8, rank, world)
    sol = lrs.LRSPnP(Y[st.row_slice].copy(), MtM[st.row_slice].copy(), D, prm, stripe=st, device=dev)
    sol.run(3)
    own = sol.X[:st.rows_owned].contiguous()
    sizes = [lrs.make_stripe(Y.shape[0], 8, r, world).rows_owned for r in range(world)]
    mx = max(sizes)
    pad = torch.zeros((mx, B), device=dev)
    pad[:own.shape[0]] = own
    bufs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    ok = True
    if rank == 0:
        Xs = torch.cat([b[:n] for b, n in zip(bufs, sizes)]).cpu().numpy()
        ref = lrs.LRSPnP(Y, MtM, D, prm, device=dev).run(3).X.cpu().numpy()
        err = float(np.linalg.norm(Xs - ref) / np.linalg.norm(ref))
        print(f"sharded-vs-unsharded rel-L2 = {err:.3e} (world {world}, spectral_patch)", flush=True)
        ok = err < 2e-5
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
