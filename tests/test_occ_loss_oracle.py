"""CPU-only: the fp64 occupancy-loss oracle against the reference's own loss code (tests/golden/ref_occ_loss_*.npz),
its edge cases, the tie-order invariants, the C-ABI struct layout and the host-side behaviour of the module."""
import os
import re

import numpy as np
import pytest
import torch

import helpers as h
from gaussianformer_b200.synthetic import make_occ_loss_inputs
from oracle import occ_loss as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
FIXTURES = [("ref_occ_loss_small", "small"), ("ref_occ_loss_small_prob", "small_prob"), ("ref_occ_loss_cfg2", "cfg2")]


def oracle_pair(d, **kw):
    args = (d["pred"].numpy(), d["labels"].numpy(), d["occ_mask"].numpy(), d["class_weights"].numpy())
    kw.setdefault("use_softmax", d["use_softmax"])
    return O.occ_loss(*args, **kw), O.occ_loss(*args, precision="f32", **kw)


def rows_of(grad_bcn):
    """[B,C,N] -> [B*N, C], the row layout the fixtures store"""
    return np.asarray(grad_bcn).transpose(0, 2, 1).reshape(-1, grad_bcn.shape[1])


def check_loss_parts(got, o64, o32, what):
    for k in ("loss", "ce", "lovasz"):
        floor = abs(o32[k] - o64[k])
        tol = max(h.ATOL + h.RTOL * abs(o64[k]), h.K_FLOOR * floor)
        assert abs(float(got[k]) - o64[k]) <= tol, f"{what} {k}: {float(got[k])!r} vs {o64[k]!r} (tol {tol:.3e})"


@pytest.mark.parametrize("fixture,case", FIXTURES)
def test_oracle_matches_reference_loss_code(fixture, case):
    g = np.load(os.path.join(GOLDEN, fixture + ".npz"))
    d = make_occ_loss_inputs(case, int(g["seed"]))
    o64, o32 = oracle_pair(d)
    check_loss_parts(g, o64, o32, fixture)
    r64, r32 = rows_of(o64["grad"]), rows_of(o32["grad"])
    stride = int(g["row_stride"])
    h.assert_grad_parity(g["grad_rows"], r64[::stride], r32[::stride], what=f"{fixture} grad rows")
    if "top_rows" in g:
        top = g["top_rows"]
        h.assert_grad_parity(g["grad_top"], r64[top], r32[top], what=f"{fixture} largest grad rows")
        floor = np.abs(r32.sum(0) - r64.sum(0)).max()
        h.assert_grad_parity(g["grad_colsum"], r64.sum(0), r64.sum(0) + floor, what=f"{fixture} grad column sums")


def test_no_present_class_gives_zero_lovasz():
    d = make_occ_loss_inputs("small", 3)
    d["labels"] = torch.where(d["labels"] % 2 == 0, torch.full_like(d["labels"], 17), torch.full_like(d["labels"], 255))
    o = O.occ_loss(d["pred"].numpy(), d["labels"].numpy(), None, None)
    assert o["lovasz"] == 0.0 and o["present"] == []
    assert np.isfinite(o["ce"]) and o["ce"] > 0


def test_single_point():
    pred = np.array([[[0.3], [-1.0], [2.0]] + [[0.0]] * 15], np.float32)    # [1, 18, 1]
    o = O.occ_loss(pred, np.array([[2]]), None, None, ce_weight=1.0)
    z = pred[0, :, 0].astype(np.float64)
    p = np.exp(z - z.max()) / np.exp(z - z.max()).sum()
    assert abs(o["ce"] - (-np.log(p[2]))) < 1e-12
    # one foreground element: dJ = 1 / g = 1, loss = e = 1 - p[2]
    assert abs(o["lovasz"] - (1 - p[2])) < 1e-12 and o["present"] == [2]


def test_empty_mask_gives_nan_ce_zero_lovasz_zero_grad():
    d = make_occ_loss_inputs("small", 4)
    o = O.occ_loss(d["pred"].numpy(), d["labels"].numpy(), np.zeros(d["labels"].shape, bool), d["class_weights"].numpy())
    assert np.isnan(o["ce"]) and o["lovasz"] == 0.0 and not o["grad"].any()


def test_closed_form_lovasz_grad_equals_jaccard_differences():
    rng = np.random.default_rng(0)
    fg = (rng.random(500) < 0.3).astype(np.int64)
    g = fg.sum()
    inter = g - np.cumsum(fg)
    union = g + np.cumsum(1 - fg)
    jac = 1.0 - inter / union
    ref = np.concatenate([jac[:1], np.diff(jac)])
    assert np.allclose(O.lovasz_grad_closed(fg), ref, rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize("mixed", [False, True])
def test_tie_permutation_keeps_loss_and_tie_group_gradient_sums(mixed):
    """Reordering tied errors keeps the loss and the sum of dL/de over each tie group.  When a group holds one
    foreground status (mixed=False) that sum is that status's; when it mixes both, only the group total is fixed."""
    rng = np.random.default_rng(1)
    n = 400
    fg = (rng.random(n) < 0.4).astype(np.int64)
    if mixed:
        e = rng.choice([0.0, 0.25, 0.5, 0.75, 1.0], size=n)
    else:
        e = np.where(fg == 1, rng.choice([0.1, 0.3, 0.6], size=n), rng.choice([0.0, 0.2, 0.3 + 1e-3, 0.9], size=n))
    loss, dlde = O.lovasz_class(e, fg)
    for seed in range(3):
        perm = np.random.default_rng(10 + seed).permutation(n)
        loss_p, dlde_p = O.lovasz_class(e[perm], fg[perm])
        assert abs(loss - loss_p) < 1e-12
        for v in np.unique(e):
            assert abs(dlde[e == v].sum() - dlde_p[e[perm] == v].sum()) < 1e-12


def test_occ_loss_struct_follows_the_header():
    from gaussianformer_b200 import _lib
    src = open(os.path.join(ROOT, "include", "gf_b200.h")).read()
    body = re.search(r"typedef struct gf_occ_loss_desc \{(.*?)\} gf_occ_loss_desc;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in filter(None, (s.strip() for s in body.split(";"))):
        first, *rest = decl.split(",")
        fields += [first.split()[-1]] + [r.strip() for r in rest]
    assert fields == [f[0] for f in _lib.OccLossDesc._fields_]


def test_module_kwargs_and_refusals():
    from gaussianformer_b200.loss import OccupancyLoss, occupancy_loss
    w = [1.0, 2.0] + [1.0] * 16
    m = OccupancyLoss(empty_label=17, num_classes=18, balance_cls_weight=True, use_sem_geo_scal_loss=False,
                      multi_loss_weights=dict(loss_voxel_ce_weight=10.0, loss_voxel_lovasz_weight=1.0),
                      lovasz_ignore=17, manual_class_weight=w)
    ref = 18 * torch.tensor(w) / sum(w)                      # num_classes * F.normalize(w, 1, -1), occupancy_loss.py:88
    assert torch.allclose(m.class_weights, ref) and m.loss_voxel_ce_weight == 10.0
    for kw in (dict(use_focal_loss=True), dict(use_dice_loss=True), dict(use_sem_geo_scal_loss=True),
               dict(use_sem_geo_scal_loss=False, balance_cls_weight=True)):
        with pytest.raises(NotImplementedError):
            OccupancyLoss(**kw)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        occupancy_loss(torch.zeros(1, 18, 4), torch.zeros(1, 4, dtype=torch.long))
