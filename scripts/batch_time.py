"""Time LRSPnPBatch against the same B cubes stepped one after another by B separate LRSPnP solvers, on cfg 1's settings
(bundled 36x36x128 crops, 36x36 blocks at stride 36, synthetic dictionary K = 2592 seed 0, Nit = 80, default Params).

The cubes are the 20 (image, mask) pairs of the bundled crops: images base, img2..img5 against the pixel masks of base,
img2, img3 and img4 (synth.cross_masked); a batch of B takes the first B of them.  For every B the two arms are warmed
up, then alternated (ABAB) over --rounds rounds of --steps outer iterations each, timed with CUDA events, the state reset
every 2 iterations as bench.py does.  The sparse step (im2col + ISTA) is timed with events on the caller's stream; its
GEMM floor is the fp16 MMA work of the 3-pass operand split at the data-sheet dense rate, a bound never reached on a
power-capped card.

    python scripts/batch_time.py --out profiles/r04_batch_cfg1.json [--profile profiles/r04_batch_cfg1_profile.txt]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import lrs_pnp_dip_b200 as lrs  # noqa: E402
from lrs_pnp_dip_b200 import synth  # noqa: E402

K, NIT, BB = 2592, 80, 36
FP16_DENSE_FLOPS = 2.25e15        # B200 data sheet, dense fp16, one GPU (1,000 W)
IMAGES = ("base", "img2", "img3", "img4", "img5")
MASK_OWNERS = ("base", "img2", "img3", "img4")


def bundled(tag):
    g = np.load(os.path.join(ROOT, "tests", "golden", "bundled_inputs_r2.npz" if tag in ("img3", "img4") else "bundled_inputs.npz"))
    return g[f"{tag}_Y"], g[f"{tag}_pixmask"]


def cubes():
    out = []
    for img in IMAGES:
        Y, _ = bundled(img)
        for owner in MASK_OWNERS:
            out.append((f"{img}+{owner}",) + synth.cross_masked(Y, bundled(owner)[1]))
    return out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


class Arm:
    """One way of stepping B cubes: one LRSPnPBatch, or B LRSPnP solvers one after another.  ``sparse`` collects event
    pairs around every sparse step (im2col + ISTA) on the caller's stream."""

    def __init__(self, kind, cases, D, prm):
        self.kind, self.sparse, self.n_done = kind, [], 0
        if kind == "batch":
            Y = np.stack([c[1] for c in cases])
            M = np.stack([c[2] for c in cases])
            self.solvers = [lrs.LRSPnPBatch(Y, M, D, prm)]
            coders = [self.solvers[0].coder]
        else:
            self.solvers = [lrs.LRSPnP(c[1], c[2], D, prm) for c in cases]
            coders = [s.be.coder for s in self.solvers]
        # the call a step makes for its Phi_z: BatchSparseCoder.imout -> phi_z, SparseCoder.imout -> _phi_z
        name = "phi_z" if kind == "batch" else "_phi_z"
        for co in coders:
            orig = getattr(co, name)

            def timed(X, l1, orig=orig):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = orig(X, l1)
                e1.record()
                self.sparse.append((e0, e1))
                return out

            setattr(co, name, timed)

    def step(self):
        if self.n_done % 2 == 0:
            for s in self.solvers:
                s.reset()
        for s in self.solvers:
            s.step()
        self.n_done += 1

    def timed(self, steps):
        torch.cuda.synchronize()
        self.n_done, self.sparse = 0, []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        torch.cuda.synchronize()
        for s in self.solvers:
            s.validate()
        return e0.elapsed_time(e1) / steps, sum(a.elapsed_time(b) for a, b in self.sparse) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--profile", default=None, help="write a torch.profiler table of one batched step (B = 20) here")
    ap.add_argument("--sizes", default="1,2,4,8,16,20")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_time.py: no CUDA device")
    info = card()
    all_cases = cubes()
    D = torch.from_numpy(synth.synthetic_dictionary(BB * BB, K, seed=0)).cuda()   # one tensor: step constants memoised once
    prm = lrs.Params()
    n = BB * BB
    P = lrs.patch_count(1296, 128, BB, BB)
    rows = []
    for B in (int(v) for v in a.sizes.split(",")):
        cases = all_cases[:B]
        arms = {k: Arm(k, cases, D, prm) for k in ("batch", "separate")}
        for arm in arms.values():
            for _ in range(a.warmup):
                arm.step()
        res = {k: {"ms": [], "sparse_ms": []} for k in arms}
        for _ in range(a.rounds):
            for k, arm in arms.items():                         # A B A B ...
                ms, sp = arm.timed(a.steps)
                res[k]["ms"].append(ms)
                res[k]["sparse_ms"].append(sp)
        floor_ms = 1e3 * (2 * NIT + 1) * 2 * n * K * P * B * 3 / FP16_DENSE_FLOPS
        row = {"B": B, "gemm_floor_ms": floor_ms}
        for k, r in res.items():
            med, med_sp = float(np.median(r["ms"])), float(np.median(r["sparse_ms"]))
            row[k] = {"ms_per_outer_iteration": med, "ms_per_cube": med / B, "runs_ms": r["ms"],
                      "spread_pct": 100 * (max(r["ms"]) - min(r["ms"])) / med, "sparse_step_ms": med_sp,
                      "sparse_runs_ms": r["sparse_ms"], "sparse_over_floor": med_sp / floor_ms}
        row["speedup_batch_vs_separate"] = row["separate"]["ms_per_outer_iteration"] / row["batch"]["ms_per_outer_iteration"]
        rows.append(row)
        print(json.dumps({"B": B, "batch_ms": row["batch"]["ms_per_outer_iteration"],
                          "separate_ms": row["separate"]["ms_per_outer_iteration"],
                          "speedup": row["speedup_batch_vs_separate"]}), flush=True)
        del arms
    out = {"card": info, "workload": f"cfg1 settings: bundled 36x36x128 crops (image x mask pairs), bb=36 stride 36, P={P}, "
                                      f"n={n}, K={K} synthetic seed 0, Nit={NIT}, default Params",
           "timing": f"CUDA events, {a.rounds} alternated rounds of {a.steps} outer iterations per arm, reset every 2, "
                     f"{a.warmup} warm-up iterations per arm and shape; medians, spread = (max - min) / median",
           "gemm_floor": "(2 Nit + 1) GEMMs x 2 n K P B FLOP x 3 fp16 passes at 2,250 TFLOP/s (data sheet, dense fp16)",
           "rows": rows}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    if a.profile:
        from torch.profiler import ProfilerActivity, profile

        arm = Arm("batch", all_cases, D, prm)
        for _ in range(a.warmup):
            arm.step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            arm.solvers[0].step()
            torch.cuda.synchronize()
        with open(a.profile, "w") as f:
            f.write(f"# one LRSPnPBatch step, B = {len(all_cases)}, cfg1 settings; card: {json.dumps(info)}\n")
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))


if __name__ == "__main__":
    main()
