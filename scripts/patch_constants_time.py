"""Cost of step='spectral_patch' at cfg 4 and cfg 5 on one GPU: for the bench's band-replicated mask, synth.band_mask and a
per-element Bernoulli(0.5) mask, the number of distinct patch patterns, the set-up time of SparseCoder (CUDA events
around the construction), its peak extra device memory, and ms per outer iteration of LRSPnP beside the same cube with
the bench's mask in the row-pattern table mode (step='spectral').

    python scripts/patch_constants_time.py --out profiles/r03_patch_constants.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lrs_pnp_dip_b200 as lrs  # noqa: E402
from lrs_pnp_dip_b200 import ops, synth  # noqa: E402

# copied from bench.py (name: H, W, bands, mask kind, keep) and its K / Nit
WORKLOADS = {
    "cfg4": (512, 512, 191, "bernoulli", 0.5),
    "cfg5": (1024, 1024, 224, "stripe+bernoulli", 0.75),
}
K_ATOMS, NIT = 256, 80


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                     # noqa: BLE001
        return f"unknown ({e})"


def distinct_patterns(Yd, bb=8, s=1, chunk=1 << 26):
    R, C = Yd.shape
    P = ops.patch_count(R, C, bb, s)
    words = torch.empty(P, dtype=torch.int64, device=Yd.device)
    for c0 in range(0, P, chunk):
        c1 = min(P, c0 + chunk)
        lrs._lib.check(lrs._lib.lib().lrs_patch_mask_words_u64(lrs._lib.ptr(Yd), R, C, bb, s, c0, c1,
                                                              lrs._lib.ptr(words[c0:c1]), lrs._lib.stream_ptr()))
    n = int(torch.unique(words).numel())
    del words
    return n, P


def time_setup(Yd, Dd, prm, reps=3):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sc = lrs.SparseCoder(Yd, Dd, prm, defer_validation=True)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
        peak = torch.cuda.max_memory_allocated() - base
        resident = torch.cuda.memory_allocated() - base
        del sc
    return float(np.median(ts)), ts, int(peak), int(resident)


def ms_per_iteration(Yd, Md, Dd, prm, warmup=1, steps=3):
    sol = lrs.LRSPnP(Yd, Md, Dd, prm)
    for _ in range(warmup):
        sol.step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        sol.step()
    e1.record()
    sol.validate()
    torch.cuda.synchronize()
    finite = bool(torch.isfinite(sol.X).all())
    del sol
    return e0.elapsed_time(e1) / steps, finite


def run(workload):
    H, W, B, kind, keep = WORKLOADS[workload]
    _, noisy = synth.synthetic_cube(H, W, B, rank=8, seed=0)
    D = synth.synthetic_dictionary(64, K_ATOMS, seed=0)
    Dd = torch.as_tensor(D).cuda()
    masks = {
        "replicated": np.repeat(synth.pixel_mask(H, W, kind, keep=keep, seed=3)[:, None], B, axis=1),
        "band_mask": synth.band_mask(H, W, B).reshape(H * W, B),
        "bernoulli0.5": (np.random.default_rng(11).random((H * W, B), dtype=np.float32) < 0.5).astype(np.uint8),
    }
    out = {"workload": workload, "shape": [H * W, B], "K": K_ATOMS, "Nit": NIT, "masks": {}}
    table_ms = None
    for name, m in masks.items():
        Yd = torch.as_tensor(synth.observe(noisy, m)).cuda()
        Md = torch.as_tensor(m.astype(np.float32)).cuda()
        del m
        n_distinct, P = distinct_patterns(Yd)
        prm = lrs.Params(Nit=NIT, bb=8, slidingDis=1, step="spectral_patch")
        lrs.SparseCoder(Yd[:4096].contiguous(), Dd, prm)                       # module load / first launches
        setup_ms, setup_all, peak, resident = time_setup(Yd, Dd, prm)
        ms, finite = ms_per_iteration(Yd, Md, Dd, prm)
        rec = {"patches": P, "distinct_patterns": n_distinct, "setup_ms": setup_ms, "setup_ms_all": setup_all,
               "peak_extra_bytes": peak, "resident_bytes": resident, "ms_per_iteration_spectral_patch": ms,
               "finite": finite}
        if name == "replicated":
            table_ms, tfin = ms_per_iteration(Yd, Md, Dd, lrs.Params(Nit=NIT, bb=8, slidingDis=1, step="spectral"))
            rec["ms_per_iteration_table"] = table_ms
        rec["vs_table_mode"] = rec["ms_per_iteration_spectral_patch"] / table_ms
        out["masks"][name] = rec
        print(workload, name, json.dumps(rec), flush=True)
        del Yd, Md
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--workloads", nargs="+", default=["cfg4", "cfg5"], choices=sorted(WORKLOADS))
    ap.add_argument("--out", default=None, help="JSON output path")
    a = ap.parse_args()
    lrs._lib.require_cuda()
    res = {"gpu": gpu_name(), "torch": torch.__version__, "runs": [run(w) for w in a.workloads]}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
