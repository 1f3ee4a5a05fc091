"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys, and the
GPU arm refuses to run without a device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "mini",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len(out.stdout.strip().splitlines()) == 1          # stdout carries the one JSON line and nothing else
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "ista_patch_iters_per_s" and line["unit"] == "patch-iters/s"
    assert line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]
    # every step is a MEASURED pass over the fixed sample: ms_per_step is that pass, not an extrapolation
    assert line["config"]["extrapolated"] is False
    assert line["config"]["patches_per_step"] == 185 * 25
    assert abs(line["value"] - line["config"]["patches_per_step"] * 80 / (line["ms_per_step"] * 1e-3)) < 1e-6 * line["value"]


def test_bench_state_schedule_stays_finite_on_the_oracle():
    """bench.py re-initialises the ADMM state every 2 steps.  The oracle shows why: the reference's literal update
    (overlap SUM in lambda_1 += mu_1 (X - IMout), main_LRS_PnP.py:346,361) diverges geometrically at stride 1, so the
    driver's 5 warm-up + 20 timed steps from one state overflow fp32, while the reset schedule stays finite."""
    import numpy as np

    from lrs_pnp_dip_b200 import synth
    from oracle import lrs_oracle as orc

    H, W, B = 10, 10, 12
    _, noisy = synth.synthetic_cube(H, W, B, rank=3, seed=1)
    pm = synth.pixel_mask(H, W, "bernoulli", keep=0.6, seed=2)
    Y = synth.observe(noisy, pm)
    MtM = np.repeat(pm.astype(np.float32)[:, None], B, axis=1)
    D = synth.synthetic_dictionary(64, 32, seed=0)
    prm = orc.Params(Nit=5, bb=8, slidingDis=1, step="frob4")
    a = orc.step_constants_batched(D, orc.patch_masks(orc.get_image_block(Y, 8, 1)[0]), "frob4")
    fresh = lambda: orc.State(X=Y.copy(), lambda_1=np.zeros_like(Y), lambda_2=np.zeros_like(Y))
    st, peak = fresh(), 0.0
    for i in range(25):                                   # the bench schedule
        if i % 2 == 0:
            st = fresh()
        st = orc.outer_iteration(st, Y, MtM, D, prm, a=a)
        peak = max(peak, float(np.abs(st.X).max()))
    assert np.isfinite(st.X).all() and peak < 2.0
    st = fresh()
    with np.errstate(all="ignore"):
        g = []
        for i in range(12):                               # one state, no reset: geometric growth
            st = orc.outer_iteration(st, Y, MtM, D, prm, a=a)
            g.append(float(np.abs(st.X).max()))
    assert g[-1] > 100 * g[1] and all(g[i + 1] > 1.5 * g[i] for i in range(5, 11))


def test_reference_arm_dumps_its_last_pass(tmp_path):
    """--dump-outputs: the reference arm writes the Phi_z of its last timed pass over the fixed sample, in float32."""
    import numpy as np

    import bench
    from oracle import lrs_oracle as orc

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "mini",
                          "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    phi = np.load(tmp_path / "Phi_z.npy")
    Y, _, D = bench.make_inputs("mini")
    sub = bench.cpu_sample(Y)
    oprm = orc.Params(Nit=bench.NIT, bb=bench.BB, slidingDis=bench.STRIDE, step="spectral")
    want, _ = orc.sparse_step(sub, np.zeros_like(sub), sub, D, oprm)
    assert phi.dtype == np.float32 and phi.shape == want.shape
    assert np.linalg.norm(phi - want) <= 1e-6 * np.linalg.norm(want)


def test_dump_row_sample_is_fixed_and_fits():
    import numpy as np

    import bench

    for R, C in ((262144, 191), (1048576, 224)):
        rows = bench.dump_rows(R, C)
        assert len(rows) * C * 4 * len(bench.STATE) <= bench.DUMP_BYTES and len(rows) > 10000
        assert np.all(np.diff(rows) > 0) and rows[-1] < R
        assert np.array_equal(rows, bench.dump_rows(R, C))
    assert np.array_equal(bench.dump_rows(4096, 32), np.arange(4096))         # small states are written whole


def test_reference_arm_other_ranks_exit_silently():
    """Under torchrun (N > 1) rank 0 alone runs the CPU reference arm; the other ranks exit 0 without work."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "mini",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_gpu_arm_fails_loudly_without_a_device():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "mini", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0
    assert "no CUDA device" in (out.stderr + out.stdout)
