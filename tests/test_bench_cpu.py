"""bench.py's host-side pieces that can run without a GPU: the FLOP bookkeeping behind `roofline`, the output dump of
`--dump-outputs`, and the torch-eager
training comparator (SURVEY.md 8d config 3) exercised on the CPU at a toy size (on the GPU box it runs on cuda:0)."""
import os
import sys
from functools import partial

import torch
import torch.nn as nn

from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_flop_bookkeeping_matches_the_survey_numbers():
    # SURVEY.md 8d: 370.806 GFLOP per base sequence at T = 243; Lite 142.093 / 45.080 / 14.773 at T = 243 / 81 / 27
    assert abs(bench.flops_per_sequence(512, 1024, 243) / 1e9 - 370.806) < 0.01
    for t, g in ((243, 142.093), (81, 45.080), (27, 14.773)):
        assert abs(bench.flops_per_sequence(256, 1024, t) / 1e9 - g) < 0.01
    assert bench.gemm_flops_per_sequence(512, 1024, 243) < bench.flops_per_sequence(512, 1024, 243)


def test_dump_outputs_writes_float32_within_the_size_cap_and_samples_the_same_rows(monkeypatch, tmp_path):
    import numpy as np
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 16)
    big = torch.arange(1000 * 32, dtype=torch.float64).reshape(1000, 32)
    arrays = {"loss_parts": torch.tensor([1.0, 2.0, 3.0, 6.0]), "pose_3d": big}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    a = {f.stem: np.load(f) for f in (tmp_path / "a").iterdir()}
    b = {f.stem: np.load(f) for f in (tmp_path / "b").iterdir()}
    assert sorted(a) == ["loss_parts", "pose_3d"] and all(v.dtype == np.float32 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 1 << 16
    assert np.array_equal(a["loss_parts"], [1, 2, 3, 6])
    rows = a["pose_3d"][:, 0] / 32                                   # whole rows of the batch, in order
    assert 0 < len(rows) < 1000 and np.all(np.diff(rows) > 0) and np.array_equal(a["pose_3d"], big.float().numpy()[rows.astype(int)])
    assert all(np.array_equal(a[k], b[k]) for k in a)
    bench.dump_outputs(str(tmp_path / "r"), {"pose_3d": big[:10]}, rank=1, world=2)
    assert [f.name for f in (tmp_path / "r").iterdir()] == ["pose_3d_rank1.npy"]


def test_eager_training_comparator_runs_a_real_optimizer_step(monkeypatch):
    from motionbert_b200 import DSTformer
    torch.manual_seed(0)
    m = DSTformer(dim_in=3, dim_out=3, dim_feat=256, dim_rep=512, depth=5, num_heads=8, mlp_ratio=4,
                  norm_layer=partial(nn.LayerNorm, eps=1e-6), maxlen=243, num_joints=17)
    monkeypatch.setattr(bench, "synthetic_clips",
                        lambda B, T, seed: torch.rand(B, T, 17, 3, generator=torch.Generator().manual_seed(seed)))
    before = {k: v.detach().clone() for k, v in m.state_dict().items()}
    r = bench.gpu_eager_train_baseline(m, "lite", 5, torch.device("cpu"), batch=2, iters=1)
    for k in ("bf16_autocast", "tf32"):
        assert r[k]["value"] > 0 and r[k]["unit"] == "sequences/sec"
    # the comparator trains its OWN copy of the parameters: the module it was handed is untouched
    assert all(torch.equal(before[k], v) for k, v in m.state_dict().items())
