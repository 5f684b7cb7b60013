"""Generates tests/golden/ref_occ_loss_*.npz from the REFERENCE's own loss code, on the CPU.

    python tests/golden/make_golden_loss.py [outdir]

Needs the reference tree (oracle/build_ref.REF).  loss/utils/lovasz_softmax.py is loaded by file path (pure PyTorch);
the cross-entropy terms are ``nn.CrossEntropyLoss`` / ``F.nll_loss`` called with the arguments of ``CE_ssc_loss`` /
``CE_wo_softmax`` (loss/occupancy_loss.py:164-183; that module itself imports mmcv / mmseg and is not loaded), and the
masking / weighting of ``OccupancyLoss.loss_voxel`` (:102-149) is spelled out around them.  Gradients come from
autograd.  Inputs are NOT stored: they are re-created from (case name, seed) by
``gaussianformer_b200.synthetic.make_occ_loss_inputs``.  The full-size case keeps every ROW_STRIDE-th gradient row,
the fp64 column sums of all rows and the TOP_ROWS rows with the largest |gradient|.
"""
import importlib.util
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from gaussianformer_b200.synthetic import make_occ_loss_inputs  # noqa: E402
from oracle import build_ref  # noqa: E402

CASES = [  # (fixture, case, seed, full gradient)
    ("ref_occ_loss_small", "small", 0, True),
    ("ref_occ_loss_small_prob", "small_prob", 1, True),
    ("ref_occ_loss_cfg2", "cfg2", 2, False),
]
CE_WEIGHT, LOVASZ_WEIGHT, LOVASZ_IGNORE = 10.0, 1.0, 17   # the shipped configs' multi_loss_weights / lovasz_ignore
ROW_STRIDE = 61
TOP_ROWS = 512


def load_lovasz():
    path = os.path.join(build_ref.REF, "loss", "utils", "lovasz_softmax.py")
    spec = importlib.util.spec_from_file_location("ref_lovasz_softmax", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def reference_loss(lv, pred, labels, occ_mask, weights, use_softmax):
    """loss_voxel for one prediction with the shipped configs' options (no focal / dice / sem-geo-scal terms)."""
    occ_mask = occ_mask.flatten(1)
    lab = labels[occ_mask][None]
    sem = pred.transpose(1, 2)[occ_mask][None].transpose(1, 2)
    if use_softmax:
        ce = torch.nn.CrossEntropyLoss(weight=weights, ignore_index=255, reduction="mean")(sem, lab.long())
        lov_in = torch.softmax(sem, dim=1)
    else:
        ce = torch.nn.functional.nll_loss(torch.log(torch.clamp(sem, 1e-6, 1. - 1e-6)), lab, weights, ignore_index=255)
        lov_in = sem
    lov = lv.lovasz_softmax(lov_in.transpose(1, 2).flatten(0, 1), lab.flatten(), ignore=LOVASZ_IGNORE)
    return CE_WEIGHT * ce, LOVASZ_WEIGHT * lov


def run(lv, name, case, seed, full, outdir):
    d = make_occ_loss_inputs(case, seed)
    pred = d["pred"].clone().requires_grad_()
    ce, lov = reference_loss(lv, pred, d["labels"], d["occ_mask"], d["class_weights"], d["use_softmax"])
    (ce + lov).backward()
    g = pred.grad.transpose(1, 2).reshape(-1, pred.shape[1]).numpy()     # [B*N, C] rows
    arrays = dict(seed=np.int64(seed), loss=np.float64((ce + lov).item()), ce=np.float64(ce.item()),
                  lovasz=np.float64(lov.item()))
    if full:
        arrays["grad_rows"] = g
        arrays["row_stride"] = np.int64(1)
    else:
        arrays["grad_rows"] = g[::ROW_STRIDE].copy()
        arrays["row_stride"] = np.int64(ROW_STRIDE)
        arrays["grad_colsum"] = g.astype(np.float64).sum(0)
        top = np.sort(np.argsort(np.abs(g).max(1))[-TOP_ROWS:])
        arrays["top_rows"] = top
        arrays["grad_top"] = g[top]
    np.savez_compressed(os.path.join(outdir, name + ".npz"), **arrays)
    print(name, {k: getattr(v, "shape", v) for k, v in arrays.items()})


if __name__ == "__main__":
    outdir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    lv = load_lovasz()
    for case in CASES:
        run(lv, *case, outdir)
