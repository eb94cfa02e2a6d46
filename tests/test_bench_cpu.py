"""bench.py pieces that run without a GPU: the algorithmic work tables the roofline figures are computed from
(DESIGN.md section 5, SURVEY.md section 8d), the per-launch byte / FLOP model of the instrumented backend, the peak
table, and the JSON contract of the reference arm's helpers."""
import json
import os
import subprocess
import sys

import pytest
import torch

import bench
from conftest import ROOT


def test_block_table_adds_up_to_the_step_totals():
    gf = sum(v[0] for v in bench.VNET96_BLOCKS.values())
    mb = sum(v[1] for v in bench.VNET96_BLOCKS.values())
    w = bench.WORKLOADS["vnet3d96"]
    assert abs(gf - w["gflop"]) / w["gflop"] < 1e-3 and abs(mb - w["mb"]) / w["mb"] < 1e-3
    # SURVEY 8d per-voxel figures x voxels of the step
    vox = 2 * 96 ** 3
    assert abs(244768 * vox / 1e9 - w["gflop"]) < 0.5 and abs(1831 * vox / 1e6 - w["mb"]) < 1.0


def test_peaks_have_the_fields_the_roofline_uses():
    p = bench.load_peaks()
    assert p["hbm_gbs"] > 1000 and p["bf16_tflops_burst"] >= p["bf16_tflops"] > 100 and p["source"]


def test_per_launch_work_model():
    """conv: e(|X|+|Y|+|W|) bytes, 2*|Y|*Cin*taps FLOPs; wgrad: e(|X|+|dY|)+4|W| bytes, same product"""
    x = torch.zeros(2, 8, 8, 8, 16, dtype=torch.bfloat16)
    y = torch.zeros(2, 8, 8, 8, 32, dtype=torch.bfloat16)
    from pytorchdeeplearing_b200._abi import BF16, PackedWeight
    w = torch.zeros(27, 16, 32, dtype=torch.bfloat16)
    by, fl = bench.TimedBackend._work("conv", (0, 3, x, PackedWeight(w, BF16, None, 0, "fwd", 3), None, y, None, None))
    assert by == 2 * (x.numel() + y.numel() + w.numel()) and fl == 2.0 * y.numel() * 16 * 27
    dwp = torch.zeros(27, 16, 32, dtype=torch.float32)
    by, fl = bench.TimedBackend._work("wgrad", (0, 3, x, y, dwp))
    assert by == 2 * (x.numel() + y.numel()) + 4 * dwp.numel() and fl == 2.0 * (y.numel() // 32) * dwp.numel()
    assert bench.TimedBackend._describe("wgrad", (0, 3, x, y, dwp)) == "wgrad[k0] 16x32@(8, 8, 8)"
    by, fl = bench.TimedBackend._work("apply_gn", (y, None, None, None, None, y))
    assert by == 2 * 2 * y.numel() and fl == 0.0


def test_workload_selection_and_batches():
    try:
        for name, w in bench.WORKLOADS.items():
            bench.select_workload(name)
            assert bench.voxels_per_sample() > 0
            x, y = bench.make_batch(1, 2)                       # rank 1 of 2: its rows of the global batch
            assert tuple(x.shape) == (w["batch"], 1) + tuple(w["spatial"]) and y.shape[0] == w["batch"]
            xg, _ = bench.make_batch(0, 2)
            assert not torch.equal(x, xg)
    finally:
        bench.select_workload("vnet3d96")


def test_dump_outputs_writes_loss_dice_and_every_gradient(tmp_path):
    import numpy as np
    m = torch.nn.Sequential(torch.nn.Conv3d(1, 2, 3), torch.nn.GroupNorm(1, 2))
    m(torch.randn(1, 1, 4, 4, 4)).sum().backward()
    out = bench.step_outputs(torch.tensor(0.5), torch.tensor(0.25, dtype=torch.float64), m)
    bench.write_outputs(str(tmp_path / "d"), out)
    names = {"loss", "dice"} | {"grad." + n for n, _ in m.named_parameters()}
    assert {p.name for p in (tmp_path / "d").iterdir()} == {n + ".npy" for n in names}
    for n, p in m.named_parameters():
        a = np.load(tmp_path / "d" / f"grad.{n}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, p.grad.numpy())
    dice = np.load(tmp_path / "d" / "dice.npy")
    assert dice.shape == () and dice.dtype == np.float32 and float(dice) == 0.25
    big = {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)}
    with pytest.raises(SystemExit):
        bench.write_outputs(str(tmp_path / "e"), big)
    assert not (tmp_path / "e").exists()


def test_b200_arm_refuses_to_run_without_a_gpu():
    """no CPU fallback: the product arm exits with an error when there is no CUDA device (SURVEY 8c, tier rule 3)"""
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode != 0 and "CUDA" in (r.stderr + r.stdout)
    assert not any(l.startswith("{") and "voxels" in l for l in r.stdout.splitlines())
