"""CPU tests of the host-side pieces: layout conversion, synthetic generators, metric."""
import os

import numpy as np
import pytest
import torch

from gaussianformer_b200.metric import MeanIoU
from gaussianformer_b200.ops.deformable_aggregation import feature_maps_format
from gaussianformer_b200.synthetic import (inverse_covariance, make_daf_inputs, make_splat_inputs, quat_to_rotmat,
                                          voxel_centers)


def test_feature_maps_format_round_trip_and_layout():
    fms = [torch.randn(2, 3, 8, h, w) for h, w in ((6, 10), (3, 5), (2, 2))]
    col, shape, start = feature_maps_format(fms)
    assert col.shape == (2, 3, 60 + 15 + 4, 8)
    assert shape.dtype == torch.int64 and shape.tolist() == [[6, 10], [3, 5], [2, 2]] and start.tolist() == [0, 60, 75]
    # row (start_l + y*w + x) of camera m holds the channel vector of pixel (y, x) of level l
    assert torch.equal(col[1, 2, 60 + 2 * 5 + 3], fms[1][1, 2, :, 2, 3])
    back = feature_maps_format([col, shape, start], inverse=True)
    for a, b in zip(back, fms):
        assert torch.equal(a, b)


def test_voxel_centres_are_x_major_and_in_their_voxel():
    dims, pc_min, gs = (5, 4, 3), (-1.0, 2.0, 0.5), 0.5
    xyz = voxel_centers(dims, pc_min, gs)
    assert xyz.shape == (5, 4, 3, 3)
    flat = xyz.reshape(-1, 3)
    idx = ((flat - torch.tensor(pc_min)) / gs).to(torch.int)
    n = (idx[:, 0] * 4 + idx[:, 1]) * 3 + idx[:, 2]
    assert torch.equal(n, torch.arange(60, dtype=n.dtype))


def test_inverse_covariance_is_spd_and_matches_closed_form():
    g = torch.Generator().manual_seed(0)
    s = 0.1 + torch.rand(50, 3, generator=g)
    q = torch.randn(50, 4, generator=g)
    inv = inverse_covariance(s, q)
    R = quat_to_rotmat(q)
    closed = R.transpose(-1, -2) @ torch.diag_embed(1 / s ** 2) @ R
    assert torch.allclose(inv, closed, rtol=2e-3, atol=1e-3)
    assert (torch.linalg.eigvalsh(closed.double()) > 0).all()


def test_rotation_matrix_equals_reference_helper():
    """tests/golden/ref_rotation_matrix.npz: the reference's get_rotation_matrix on 64 seeded quaternions."""
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_rotation_matrix.npz"))
    q = torch.randn(64, 4, generator=torch.Generator().manual_seed(1))
    assert torch.equal(q, torch.from_numpy(gold["quaternions"]))
    assert torch.allclose(quat_to_rotmat(q), torch.from_numpy(gold["rotation"]), atol=1e-6)


def test_synthetic_shapes_and_determinism():
    kw, inp, variant = make_splat_inputs("tiny", seed=3)
    kw2, inp2, _ = make_splat_inputs("tiny", seed=3)
    assert all(torch.equal(inp[k], inp2[k]) for k in inp)
    assert inp["pts"].shape == (1, 50 * 50 * 4, 3) and inp["cov"].shape == (1, 256, 3, 3) and variant == "base"
    fms, loc, w = make_daf_inputs(num_anchor=10, num_pts=3, levels=((4, 4), (2, 2)), embed_dims=8, num_groups=2)
    assert loc.shape == (1, 30, 6, 2) and w.shape == (1, 30, 6, 2, 2)
    s = w.reshape(1, 10, 3 * 6 * 2, 2).sum(2)          # joint softmax over (pts, cams, levels) per group
    assert torch.all((s - 1).abs().lt(1e-5) | s.abs().lt(1e-6))


def test_mean_iou_definition():
    m = MeanIoU([1, 2], empty_label=0)
    pred = torch.tensor([1, 1, 2, 0, 2, 0])
    gt = torch.tensor([1, 2, 2, 0, 0, 1])
    m.after_step(pred, gt)
    miou, iou = m.after_epoch()
    # class 1: correct 1, seen 2, positive 2 -> 1/3 ; class 2: correct 1, seen 2, positive 2 -> 1/3
    assert abs(miou - 100 / 3) < 1e-9
    # occupancy: seen 4 (gt != 0), positive 4, correct 3 -> 3/5
    assert abs(iou - 60.0) < 1e-9


def test_miou_parity_recipe_on_the_oracle():
    """SURVEY.md 8(d) mIoU parity recipe, exercised on the CPU: fp32 vs fp64 oracle logits of the tiny config give
    the same mIoU against the seeded noisy labels up to the voxels whose top two classes tie numerically (each such
    flip moves a class IoU of this 10 000-voxel grid by ~1e-3; at the full 640 000-voxel shape bench.py reports the
    figure); a deliberately damaged prediction does not."""
    import numpy as np
    import helpers as h
    from gaussianformer_b200.metric import miou_parity, synthetic_labels
    kw, inp, variant = h.splat_case("tiny", 0, False)
    ref64 = h.oracle_forward(kw, inp, variant, precision="f64")["logits"]
    ref32 = h.oracle_forward(kw, inp, variant, precision="f32")["logits"]
    C = ref64.shape[1]
    labels, mask = synthetic_labels(ref64, C)
    assert 0.05 < float((labels != torch.as_tensor(ref64).argmax(1)).float().mean()) < 0.15
    r = miou_parity(ref32.argmax(1), ref64.argmax(1), labels, mask, C)
    flips = int((ref32.argmax(1) != ref64.argmax(1)).sum())
    assert flips <= 20 and r["abs_diff"] <= 0.01 * max(flips, 1) and r["ref"][0] > 50.0
    bad = ref64.argmax(1).copy()
    bad[: bad.shape[0] // 4] = 3
    assert miou_parity(bad, ref64.argmax(1), labels, mask, C)["abs_diff"] > 1.0


def test_fused_sampling_entry_point_rejects_cpu_tensors_and_bad_shapes():
    """The opt-in fused caller path has no CPU fallback either, and validates its shapes before touching the library."""
    from gaussianformer_b200.ops import deformable_aggregation_fused
    from gaussianformer_b200.synthetic import make_daf_fused_inputs
    from gaussianformer_b200.ops.deformable_aggregation import feature_maps_format
    fms, loc, logits, pm, _ = make_daf_fused_inputs(num_anchor=6, num_pts=2, batch=1, num_cams=2, embed_dims=8,
                                                    num_groups=2, levels=((4, 4),), seed=1)
    feat, shape, start = feature_maps_format(fms)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        deformable_aggregation_fused(feat.contiguous(), shape, start, loc, logits, pm)
    with pytest.raises(ValueError, match="weight_logits must be"):
        deformable_aggregation_fused(feat.contiguous(), shape, start, loc, logits.flatten(1, 2), pm)


def test_fused_reference_composition_matches_masked_softmax_definition():
    """synthetic.reference_fused_composition (the PyTorch route the fused op replaces, used by bench.py and the GPU
    tests) against a direct per-anchor evaluation: softmax over the unmasked (key point, camera, level) entries of each
    group, zero weights for a group with every entry masked."""
    from gaussianformer_b200.synthetic import reference_fused_composition
    B, A, K, M, L, Gr, C = 1, 3, 2, 2, 2, 2, 4
    gen = torch.Generator().manual_seed(0)
    logits = torch.randn(B, A, K, M, L, Gr, generator=gen, dtype=torch.float64)
    pm = torch.rand(B, A, K, M, generator=gen) > 0.4
    pm[0, 1] = False
    vals = torch.randn(B, A * K, M, L, C, generator=gen, dtype=torch.float64)     # stand-in for the sampled features

    def fake_daf(feat, shape, start, loc, w):                                      # out[b,p,c] = sum_{m,l} w * val
        return (w.repeat_interleave(C // Gr, dim=-1) * vals).sum(dim=(2, 3))
    out = reference_fused_composition(fake_daf, None, None, None, None, logits, pm)
    want = torch.zeros(B, A, C, dtype=torch.float64)
    for a in range(A):
        for g in range(Gr):
            on = pm[0, a][:, :, None].expand(K, M, L)
            if on.any():
                w = torch.where(on, logits[0, a, ..., g], torch.tensor(-float("inf"), dtype=torch.float64)).flatten().softmax(0).reshape(K, M, L)
                for c in range(g * (C // Gr), (g + 1) * (C // Gr)):
                    want[0, a, c] = (w * vals[0].reshape(A, K, M, L, C)[a, ..., c]).sum()
    assert torch.allclose(out, want, atol=1e-12)
    assert torch.all(out[0, 1] == 0)


def test_grid_points_are_the_reference_loaders_voxel_centres():
    """LocalAggregator.grid_points reproduces LoadOccupancySurroundOcc.get_meshgrid (dataset/transform_3d.py:487-499)
    bit for bit: arange * reso + 0.5 * reso + min in fp32, stacked x-major."""
    import local_aggregate
    m = local_aggregate.LocalAggregator(3, 200, 200, 16, [-50.0, -50.0, -5.0], 0.5)
    got = m.grid_points("cpu")
    reso, grid, ranges = 0.5, [200, 200, 16], [-50, -50, -5.0]
    xxx = torch.arange(grid[0], dtype=torch.float) * reso + 0.5 * reso + ranges[0]
    yyy = torch.arange(grid[1], dtype=torch.float) * reso + 0.5 * reso + ranges[1]
    zzz = torch.arange(grid[2], dtype=torch.float) * reso + 0.5 * reso + ranges[2]
    want = torch.stack([xxx[:, None, None].expand(*grid), yyy[None, :, None].expand(*grid),
                        zzz[None, None, :].expand(*grid)], dim=-1).reshape(1, -1, 3)
    assert got.shape == (1, 640000, 3) and torch.equal(got, want)
    assert m.grid_points("cpu") is got                       # cached
