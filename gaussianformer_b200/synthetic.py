"""Seeded synthetic inputs shaped like the reference's SurroundOcc configs (no dataset needed).

Distributions follow SURVEY.md §8(d):

* grid / voxel centres — ``dataset/transform_3d.py:484-499`` (x-major, z fastest);
* scales ``lo + (hi-lo)*sigmoid(N(0,1))`` with the config's ``scale_range``
  (``config/nuscenes_gs25600_solid.py:70``, ``config/nuscenes_gs144000.py:70``,
  ``config/prob/nuscenes_gs6400.py:88``);
* inverse covariance built like ``model/head/gaussian_head.py:111-119``
  (``S``, ``R`` -> ``M = S R`` -> ``Cov = M^T M`` -> ``Cov.inverse()``), rotation from a unit
  quaternion (``model/utils/utils.py:20-69``);
* the "empty" Gaussian of the solid config — ``model/head/gaussian_head.py:43-48,96-102`` with
  ``config/nuscenes_gs25600_solid.py:179-184``.

Everything is generated on the CPU with a ``torch.Generator`` so the same seed gives the same
bytes on every box.
"""
from __future__ import annotations

import math

import torch

SPLAT_CONFIGS = {
    # name: (G, grid dims, pc_min, grid_size, scale_range, scale_multiplier, variant, empty, opa, sem)
    "tiny": dict(G=256, dims=(50, 50, 4), pc_min=(-12.5, -12.5, -1.0), grid_size=0.5,
                 scale_range=(0.08, 0.64), scale_multiplier=3, variant="base", with_empty=False,
                 include_opa=True, sem="softplus17"),
    "gs25600_solid": dict(G=25600, dims=(200, 200, 16), pc_min=(-50.0, -50.0, -5.0), grid_size=0.5,
                          scale_range=(0.08, 0.64), scale_multiplier=3, variant="base",
                          with_empty=True, include_opa=True, sem="softplus17"),
    "gs144000": dict(G=144000, dims=(200, 200, 16), pc_min=(-50.0, -50.0, -5.0), grid_size=0.5,
                     scale_range=(0.08, 0.32), scale_multiplier=3, variant="base",
                     with_empty=False, include_opa=False, sem="normal18"),
    "prob_gs6400": dict(G=6400, dims=(200, 200, 16), pc_min=(-50.0, -50.0, -5.0), grid_size=0.5,
                        scale_range=(0.01, 3.2), scale_multiplier=4, variant="prob",
                        with_empty=False, include_opa=True, sem="softmax17"),
    "tiny_prob": dict(G=192, dims=(40, 36, 8), pc_min=(-10.0, -9.0, -2.0), grid_size=0.5,
                      scale_range=(0.05, 1.2), scale_multiplier=4, variant="prob",
                      with_empty=False, include_opa=True, sem="softmax17"),
}


def voxel_centers(dims, pc_min, grid_size):
    """[H,W,D,3] voxel-centre coordinates, the ``occ_xyz`` of the reference loader."""
    H, W, D = dims
    xs = torch.arange(H, dtype=torch.float) * grid_size + 0.5 * grid_size + pc_min[0]
    ys = torch.arange(W, dtype=torch.float) * grid_size + 0.5 * grid_size + pc_min[1]
    zs = torch.arange(D, dtype=torch.float) * grid_size + 0.5 * grid_size + pc_min[2]
    return torch.stack([xs[:, None, None].expand(H, W, D), ys[None, :, None].expand(H, W, D),
                        zs[None, None, :].expand(H, W, D)], dim=-1).contiguous()


def quat_to_rotmat(q):
    """Unit-quaternion (w,x,y,z) -> 3x3 rotation, same matrix as the reference's helper."""
    q = torch.nn.functional.normalize(q, dim=-1)
    w, x, y, z = q.unbind(-1)
    rows = [
        torch.stack([w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)], -1),
        torch.stack([2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)], -1),
        torch.stack([2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z], -1),
    ]
    return torch.stack(rows, dim=-2)


def inverse_covariance(scales, rotations):
    """``CovInv`` of ``GaussianHead.prepare_gaussian_args`` (computed on the CPU, like the reference)."""
    S = torch.diag_embed(scales)
    R = quat_to_rotmat(rotations)
    M = torch.matmul(S, R)
    cov = torch.matmul(M.transpose(-1, -2), M)
    return torch.linalg.inv(cov.cpu())


def make_splat_inputs(name="gs25600_solid", seed=0, perturb=False, overrides=None):
    """Returns (module_kwargs, inputs) with ``inputs`` = dict(pts, means, opa, sem, scales, cov)
    each carrying the reference's leading batch dimension of 1 (CPU float32)."""
    cfg = dict(SPLAT_CONFIGS[name])
    if overrides:
        cfg.update(overrides)
    gen = torch.Generator().manual_seed(seed)
    G = cfg["G"]
    dims, pc_min, gs = cfg["dims"], cfg["pc_min"], cfg["grid_size"]
    lo, hi = cfg["scale_range"]
    pc_min_t = torch.tensor(pc_min, dtype=torch.float)
    extent = torch.tensor(dims, dtype=torch.float) * gs

    pts = voxel_centers(dims, pc_min, gs).reshape(-1, 3)
    if perturb:  # dataset/transform_3d.py:522-525
        jitter = torch.clamp(torch.randn(pts.shape, generator=gen) / 6, -0.5, 0.5) * 0.49
        pts = pts + jitter
    means = pc_min_t + torch.rand(G, 3, generator=gen) * extent * (1 - 1e-3)
    scales = lo + (hi - lo) * torch.sigmoid(torch.randn(G, 3, generator=gen))
    rots = torch.randn(G, 4, generator=gen)
    if cfg["include_opa"]:
        opa = torch.sigmoid(torch.randn(G, generator=gen))
    else:
        opa = torch.ones(G)
    kind = cfg["sem"]
    if kind == "softplus17":
        sem = torch.nn.functional.softplus(torch.randn(G, 17, generator=gen))
        sem = torch.cat([sem, torch.zeros(G, 1)], dim=-1)
    elif kind == "softmax17":
        sem = torch.softmax(torch.randn(G, 17, generator=gen), dim=-1)
        sem = torch.cat([sem, torch.zeros(G, 1)], dim=-1)
    elif kind == "normal18":
        sem = torch.randn(G, 18, generator=gen)
    else:
        raise ValueError(kind)
    if cfg["with_empty"]:
        means = torch.cat([means, torch.tensor([[0.0, 0.0, -1.0]])], 0)
        scales = torch.cat([scales, torch.tensor([[100.0, 100.0, 8.0]])], 0)
        rots = torch.cat([rots, torch.tensor([[1.0, 0.0, 0.0, 0.0]])], 0)
        empty_sem = torch.zeros(1, 18)
        empty_sem[0, 17] = 10.0
        sem = torch.cat([sem, empty_sem], 0)
        opa = torch.cat([opa, torch.ones(1)], 0)
    cov = inverse_covariance(scales, rots)
    module_kwargs = dict(scale_multiplier=cfg["scale_multiplier"], H=dims[0], W=dims[1], D=dims[2],
                         pc_min=list(pc_min), grid_size=gs)
    inputs = dict(pts=pts[None].contiguous(), means=means[None].contiguous(),
                  opa=opa[None].contiguous(), sem=sem[None].contiguous(),
                  scales=scales[None].contiguous(), cov=cov[None].contiguous().float())
    return module_kwargs, inputs, cfg["variant"]


DAF_LEVELS_1600x864 = ((108, 200), (54, 100), (27, 50), (14, 25))


def make_daf_inputs(num_anchor=25600, num_pts=9, batch=1, num_cams=6, embed_dims=128, num_groups=4,
                    levels=DAF_LEVELS_1600x864, visible_p=0.22, seed=0):
    """Feature pyramid + sampling locations + masked-softmax weights shaped like
    ``DeformableFeatureAggregation.forward`` hands them to the op
    (``model/encoder/gaussian_encoder/deformable_module.py:161-228``)."""
    gen = torch.Generator().manual_seed(seed)
    feature_maps = [torch.randn(batch, num_cams, embed_dims, h, w, generator=gen) for h, w in levels]
    P = num_anchor * num_pts
    L = len(levels)
    inside = torch.rand(batch, P, num_cams, generator=gen) < visible_p
    loc_in = torch.rand(batch, P, num_cams, 2, generator=gen) * 0.998 + 0.001
    loc_out = 1.0 + torch.rand(batch, P, num_cams, 2, generator=gen) * 0.5
    flip = torch.rand(batch, P, num_cams, 2, generator=gen) < 0.5
    loc_out = torch.where(flip, -loc_out + 1.0, loc_out)
    loc = torch.where(inside[..., None], loc_in, loc_out).contiguous()
    # joint softmax over (pts, cams, levels) per anchor and group with invisible cams masked out
    raw = torch.randn(batch, num_anchor, num_pts, num_cams, L, num_groups, generator=gen)
    mask = inside.reshape(batch, num_anchor, num_pts, num_cams)[..., None, None].expand_as(raw)
    all_miss = mask.sum(dim=[2, 3, 4], keepdim=True) == 0
    raw = raw.masked_fill(~mask, -math.inf)
    raw = torch.where(all_miss.expand_as(raw), torch.zeros_like(raw), raw)
    w = raw.flatten(2, 4).softmax(dim=-2).reshape(batch, P, num_cams, L, num_groups)
    w = w * (1 - all_miss.expand(-1, -1, num_pts, -1, -1, -1).reshape(batch, P, 1, 1, num_groups).float())
    return feature_maps, loc, w.contiguous()


def make_daf_inputs_projected(num_anchor=25600, num_pts=9, batch=1, num_cams=6, embed_dims=128, num_groups=4,
                              levels=DAF_LEVELS_1600x864, seed=0, image_wh=(1600.0, 864.0), kp_sigma=0.3):
    """A CORRELATED sampling workload: what ``DeformableFeatureAggregation`` really feeds the op.  Anchors are 3-D
    points in the nuScenes volume; each anchor has ``num_pts`` key points scattered ``kp_sigma`` metres around it
    (``SparseGaussian3DKeyPointsGenerator``: fixed + learnable offsets scaled by the Gaussian, deformable_module.py:17-90);
    the key points are projected into ``num_cams`` pinhole cameras that look outward at 360/num_cams degree steps and
    normalised by the image size (``project_points``, deformable_module.py:287-305).  A camera sees a key point when it
    lies in front of it and inside the image; the other cameras get a location outside (0, 1) like the reference's.
    Key points of one anchor therefore land a few pixels apart (and on the same rows of the coarse levels), unlike
    ``make_daf_inputs`` whose locations are independent uniform draws.  Returns (feature_maps, loc, weights)."""
    gen = torch.Generator().manual_seed(seed)
    feature_maps = [torch.randn(batch, num_cams, embed_dims, h, w, generator=gen) for h, w in levels]
    W_img, H_img = image_wh
    P = num_anchor * num_pts
    L = len(levels)
    anchors = torch.rand(batch, num_anchor, 3, generator=gen) * torch.tensor([100.0, 100.0, 8.0]) + torch.tensor([-50.0, -50.0, -5.0])
    kps = anchors[:, :, None, :] + torch.randn(batch, num_anchor, num_pts, 3, generator=gen) * kp_sigma
    kps = kps.reshape(batch, P, 3)
    focal = 0.8 * W_img
    locs, vis = [], []
    for m in range(num_cams):
        yaw = 2 * math.pi * m / num_cams
        fwd = torch.tensor([math.cos(yaw), math.sin(yaw), 0.0])
        right = torch.tensor([math.sin(yaw), -math.cos(yaw), 0.0])
        up = torch.tensor([0.0, 0.0, 1.0])
        rel = kps - torch.tensor([0.0, 0.0, -3.2])                 # camera 1.8 m above the ground plane of the volume
        depth = (rel * fwd).sum(-1)
        u = focal * (rel * right).sum(-1) / depth.clamp(min=1e-5) + 0.5 * W_img
        v = -focal * (rel * up).sum(-1) / depth.clamp(min=1e-5) + 0.5 * H_img
        xy = torch.stack([u / W_img, v / H_img], -1)
        ok = (depth > 1e-5) & (xy > 0).all(-1) & (xy < 1).all(-1)
        xy = torch.where(ok[..., None], xy, torch.full_like(xy, 2.0))
        locs.append(xy)
        vis.append(ok)
    loc = torch.stack(locs, 2).contiguous()                          # [B, P, M, 2]
    inside = torch.stack(vis, 2)                                     # [B, P, M]
    raw = torch.randn(batch, num_anchor, num_pts, num_cams, L, num_groups, generator=gen)
    mask = inside.reshape(batch, num_anchor, num_pts, num_cams)[..., None, None].expand_as(raw)
    all_miss = mask.sum(dim=[2, 3, 4], keepdim=True) == 0
    raw = raw.masked_fill(~mask, -math.inf)
    raw = torch.where(all_miss.expand_as(raw), torch.zeros_like(raw), raw)
    w = raw.flatten(2, 4).softmax(dim=-2).reshape(batch, P, num_cams, L, num_groups)
    w = w * (1 - all_miss.expand(-1, -1, num_pts, -1, -1, -1).reshape(batch, P, 1, 1, num_groups).float())
    return feature_maps, loc, w.contiguous()


def make_daf_fused_inputs(num_anchor=25600, num_pts=9, batch=1, num_cams=6, embed_dims=128, num_groups=4,
                          levels=DAF_LEVELS_1600x864, visible_p=0.22, seed=0, attn_drop=0.0):
    """Inputs of the fused caller path (``ops.deformable_aggregation_fused``): the same pyramid and sampling
    locations as ``make_daf_inputs`` plus what ``DeformableFeatureAggregation.forward`` holds BEFORE its softmax
    (``deformable_module.py:177-212``): raw weights ``[B, A, K, M, L, Gr]``, the projection mask
    ``[B, A, K, M]`` (a camera sees the key point) and, for ``attn_drop > 0``, the training-time weight mask."""
    feature_maps, loc, _ = make_daf_inputs(num_anchor, num_pts, batch, num_cams, embed_dims, num_groups, levels,
                                           visible_p, seed)
    gen = torch.Generator().manual_seed(seed + 1000)
    L = len(levels)
    logits = torch.randn(batch, num_anchor, num_pts, num_cams, L, num_groups, generator=gen)
    point_mask = ((loc > 0) & (loc < 1)).all(-1).reshape(batch, num_anchor, num_pts, num_cams).contiguous()
    weight_mask = None
    if attn_drop > 0:
        weight_mask = torch.rand(logits.shape, generator=gen) > attn_drop
    return feature_maps, loc, logits, point_mask, weight_mask


def reference_fused_composition(daf_apply, feat, shape, start, loc, logits, point_mask=None, weight_mask=None):
    """``deformable_module.py:213-228`` + ``:242`` in PyTorch around an op call ``daf_apply`` — what the fused entry
    point replaces (used by the tests and by bench.py to time the unfused route on the same GPU)."""
    B, A, K, M, L, Gr = logits.shape
    mask = torch.ones_like(logits, dtype=torch.bool)
    if point_mask is not None:
        mask = point_mask[..., None, None] & mask
    if weight_mask is not None:
        mask = mask & weight_mask
    all_miss = mask.sum(dim=[2, 3, 4], keepdim=True) == 0
    all_miss = all_miss.expand(-1, -1, K, M, L, -1)
    weights = logits.clone()
    weights[~mask] = -torch.inf
    weights[all_miss] = 0.
    weights = weights.flatten(2, 4).softmax(dim=-2).reshape(B, A * K, M, L, Gr)
    weights = weights * (1 - all_miss.flatten(1, 2).float())
    features = daf_apply(feat, shape, start, loc, weights).reshape(B, A, K, -1)
    return features.sum(dim=2)


OCC_LOSS_CASES = {
    # name: (B, N, C, use_softmax)
    "small": (2, 3001, 18, True),
    "small_prob": (2, 3001, 18, False),
    "cfg2": (1, 200 * 200 * 16, 18, True),            # config 2's grid, one sample
    "cfg2_prob": (1, 200 * 200 * 16, 18, False),
    "cfg5": (4, 200 * 200 * 16, 18, True),            # config 5: four samples per GPU
}


def make_occ_loss_inputs(name="small", seed=0, empty_label=17, empty_frac=0.8, overrides=None):
    """Seeded CPU inputs of the occupancy loss shaped like ``GaussianHead`` hands them over: ``pred [B,C,N]`` (logits,
    or probabilities for the ``*_prob`` cases), ``labels [B,N]`` int64 (about ``empty_frac`` of them ``empty_label``, the
    rest uniform over the other classes), ``occ_mask = labels != 0`` (dataset/transform_3d.py:509) and class weights
    drawn from [0.5, 1.3].  Logits are moderate (N(0, 1.5^2)), so Lovász errors are tie-free."""
    B, N, C, use_softmax = OCC_LOSS_CASES[name]
    if overrides:
        B, N, C, use_softmax = (overrides.get(k, v) for k, v in zip(("B", "N", "C", "use_softmax"), (B, N, C, use_softmax)))
    gen = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, C, N, generator=gen) * 1.5
    pred = logits if use_softmax else torch.softmax(logits, dim=1)
    other = torch.randint(0, C - 1, (B, N), generator=gen)
    other = other + (other >= empty_label).long()                  # any class but the empty one
    labels = torch.where(torch.rand(B, N, generator=gen) < empty_frac, torch.full_like(other, empty_label), other)
    weights = 0.5 + 0.8 * torch.rand(C, generator=gen)
    return dict(pred=pred.contiguous(), labels=labels, occ_mask=labels != 0, class_weights=weights,
                use_softmax=use_softmax)


def reference_occupancy_loss(pred, labels, occ_mask=None, class_weights=None, *, use_softmax=True, ce_weight=10.0,
                             lovasz_weight=1.0, lovasz_ignore=17, ignore_empty=False, empty_label=17):
    """The reference's composition in PyTorch, as ``OccupancyLoss.loss_voxel`` runs it for one prediction
    (loss/occupancy_loss.py:102-149): boolean-mask selects of the labels and the logits, ``nn.CrossEntropyLoss`` or
    ``nll_loss(log(clamp(p)))``, then the Lovász-softmax of loss/utils/lovasz_softmax.py:157-204 -- a loop over the
    classes with one ``fg.sum() == 0`` host check and one ``torch.sort`` each.  Differentiable; the timing baseline of
    tools/time_loss.py and the end-to-end comparison of the tests.  Returns (loss, ce part, lovasz part)."""
    F = torch.nn.functional
    if ignore_empty:
        keep = labels != empty_label
        occ_mask = keep if occ_mask is None else keep & occ_mask.flatten(1)
    if occ_mask is not None:
        occ_mask = occ_mask.flatten(1)
        labels = labels[occ_mask][None]
        pred = pred.transpose(1, 2)[occ_mask][None].transpose(1, 2)
    labels = labels.long()
    w = None if class_weights is None else class_weights.to(pred)
    if use_softmax:
        ce = F.cross_entropy(pred, labels, weight=w, ignore_index=255)
        probas = torch.softmax(pred, dim=1)
    else:
        ce = F.nll_loss(torch.log(torch.clamp(pred, 1e-6, 1. - 1e-6)), labels, w, ignore_index=255)
        probas = pred
    probas = probas.transpose(1, 2).flatten(0, 1)
    flat = labels.flatten()
    if lovasz_ignore is not None:
        keep = flat != lovasz_ignore
        probas, flat = probas[keep], flat[keep]
    losses = []
    if probas.numel() > 0:
        for c in range(probas.shape[1]):
            fg = (flat == c).float()
            if fg.sum() == 0:                                   # a host sync per class, as in the reference
                continue
            err = (fg - probas[:, c]).abs()
            err_sorted, perm = torch.sort(err, 0, descending=True)
            fg_sorted = fg[perm]
            gts = fg_sorted.sum()
            inter = gts - fg_sorted.cumsum(0)
            union = gts + (1 - fg_sorted).cumsum(0)
            jac = 1. - inter / union
            jac = torch.cat([jac[:1], jac[1:] - jac[:-1]])
            losses.append(torch.dot(err_sorted, jac))
    lov = torch.stack(losses).mean() if losses else pred.new_zeros(())
    return ce_weight * ce + lovasz_weight * lov, ce_weight * ce, lovasz_weight * lov
