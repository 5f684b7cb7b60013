"""ORACLE — TEST INFRASTRUCTURE ONLY.  numpy restatement of the occupancy loss (include/gf_b200.h, gf_occ_loss_desc).

Written from the semantics, citing the reference (paths relative to its tree):

* masking and the pooled set — ``OccupancyLoss.loss_voxel``, loss/occupancy_loss.py:105-116 (``ignore_empty``
  :105-107); the B samples are flattened into one set;
* cross-entropy — ``CE_ssc_loss`` :164-178 (``nn.CrossEntropyLoss(weight, ignore_index=255)``, weighted mean) and
  ``CE_wo_softmax`` :180-183 (``nll_loss(log(clamp(p, 1e-6, 1 - 1e-6)))``);
* Lovász-softmax — ``lovasz_softmax(classes='present', per_image=False, ignore=lovasz_ignore)`` on ``softmax(pred)``
  or ``pred`` (occupancy_loss.py:135-141), loss/utils/lovasz_softmax.py:157-204 with ``lovasz_grad`` :22-34 and
  ``mean`` :311-329 (0 for an empty list).

``precision="f64"`` is the truth: closed-form Lovász gradient from integer counts, stable descending sort (ties in
ascending point index, the op's order).  ``precision="f32"`` follows the reference's arithmetic (fp32 softmax, fp32
Jaccard differences, fp32 dot products) and serves to measure the fp32 floor the GPU tests gate on.
"""
from __future__ import annotations

import numpy as np

IGNORE_INDEX = 255


def _softmax(z, rt):
    z = z.astype(rt)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return e / e.sum(axis=1, keepdims=True)


def lovasz_grad_closed(fg_sorted):
    """dJ per sorted position from integer counts: foreground 1/(g+B); background (g-F)/((g+B-1)(g+B)), with g the
    foreground total, F the foreground count before the position, B the background count up to and including it."""
    fg = np.asarray(fg_sorted, np.int64)
    g = float(fg.sum())
    F_incl = np.cumsum(fg)
    F_before = (F_incl - fg).astype(np.float64)
    Bc = (np.cumsum(1 - fg)).astype(np.float64)
    fg_term = 1.0 / (g + Bc)
    with np.errstate(divide="ignore", invalid="ignore"):
        bg_term = (g - F_before) / ((g + Bc - 1.0) * (g + Bc))
    return np.where(fg == 1, fg_term, bg_term)


def lovasz_grad_f32(fg_sorted):
    """The reference's ``lovasz_grad`` in fp32: differences of consecutive Jaccard values."""
    fg = np.asarray(fg_sorted, np.float32)
    g = fg.sum(dtype=np.float32)
    inter = g - np.cumsum(fg, dtype=np.float32)
    union = g + np.cumsum(np.float32(1) - fg, dtype=np.float32)
    jac = (np.float32(1) - inter / union).astype(np.float32)
    if jac.size > 1:
        jac[1:] = jac[1:] - jac[:-1]
    return jac


def lovasz_class(e, fg, precision="f64"):
    """One class: (loss, dL/de per element in the input order).  Errors sorted descending, ties by index."""
    order = np.argsort(-np.asarray(e, np.float64), kind="stable")
    if precision == "f64":
        dj = lovasz_grad_closed(fg[order])
        loss = float(np.dot(np.asarray(e, np.float64)[order], dj))
    else:
        dj = lovasz_grad_f32(fg[order])
        loss = float(np.dot(np.asarray(e, np.float32)[order], dj))
    dlde = np.empty_like(dj)
    dlde[order] = dj
    return loss, dlde


def occ_loss(pred, labels, occ_mask=None, class_weights=None, *, use_softmax=True, ce_weight=10.0, lovasz_weight=1.0,
             lovasz_ignore=17, ignore_empty=False, empty_label=17, lovasz=True, precision="f64"):
    """``pred [B,C,N]``, ``labels [B,N]``, ``occ_mask [B,N]`` or None, ``class_weights [C]`` or None.
    Returns dict(loss, ce, lovasz (both weighted), grad [B,C,N], present [list], dlde {class: [M]}, set_rows [M],
    the flat indices of the Lovász set)."""
    rt = np.float64 if precision == "f64" else np.float32
    pred = np.asarray(pred, np.float32)
    B, C, N = pred.shape
    z = pred.transpose(0, 2, 1).reshape(B * N, C)
    y = np.asarray(labels).reshape(B * N).astype(np.int64)
    w = np.ones(C, rt) if class_weights is None else np.asarray(class_weights, np.float32).astype(rt)
    active = np.ones(B * N, bool) if occ_mask is None else np.asarray(occ_mask, bool).reshape(B * N)
    if ignore_empty:
        active &= y != empty_label
    in_range = y < C
    ce_rows = active & in_range & (y != IGNORE_INDEX)
    set_rows = active & (in_range | (y == IGNORE_INDEX))
    if lovasz_ignore is not None and lovasz_ignore >= 0:
        set_rows &= y != lovasz_ignore
    q = _softmax(z, rt) if use_softmax else z.astype(rt)
    grad_q = np.zeros((B * N, C), np.float64)   # d loss / d q, Lovász part
    grad_z = np.zeros((B * N, C), np.float64)

    # cross-entropy
    yc = y[ce_rows]
    if use_softmax:
        zz = z[ce_rows].astype(rt)
        m = zz.max(axis=1, keepdims=True)
        lse = (m + np.log(np.exp(zz - m).sum(axis=1, keepdims=True)))[:, 0]
        nll = lse - zz[np.arange(yc.size), yc]
    else:
        lo, hi = rt(np.float32(1e-6)), rt(np.float32(1 - 1e-6))
        py = q[ce_rows, yc] if yc.size else np.zeros(0, rt)
        nll = -np.log(np.clip(py, lo, hi))
    wy = w[yc]
    den = float(wy.astype(np.float64).sum())
    num = float((wy.astype(np.float64) * nll.astype(np.float64)).sum())
    ce = num / den if den != 0 else float("nan")
    if yc.size:
        scale = ce_weight * wy.astype(np.float64) / den
        rows = np.nonzero(ce_rows)[0]
        if use_softmax:
            grad_z[rows] += scale[:, None] * q[ce_rows].astype(np.float64)
            grad_z[rows, yc] -= scale
        else:
            p = q[ce_rows, yc].astype(np.float64)
            inside = (py >= lo) & (py <= hi)
            grad_q[rows, yc] += np.where(inside, -scale / np.where(p == 0, 1, p), 0.0)

    # Lovász-softmax
    lov = 0.0
    present, dlde_all = [], {}
    set_idx = np.nonzero(set_rows)[0] if lovasz else np.zeros(0, np.int64)
    if set_idx.size:
        ys = y[set_idx]
        qs = q[set_idx]
        losses = []
        for c in range(C):
            fg = (ys == c).astype(np.int64)
            if fg.sum() == 0:
                continue
            present.append(c)
            e = np.abs(fg.astype(rt) - qs[:, c])
            lc, dlde = lovasz_class(e, fg, precision)
            losses.append(lc)
            dlde_all[c] = dlde
        if losses:
            lov = float(np.sum(losses)) / len(losses)
            for c in present:
                fg = (ys == c)
                diff = fg.astype(np.float64) - qs[:, c].astype(np.float64)
                # e = |fg - q|: de/dq = -sign(fg - q), abs'(0) = 0
                grad_q[set_idx, c] += lovasz_weight / len(present) * dlde_all[c] * -np.sign(diff)
    if use_softmax:
        qd = q.astype(np.float64)
        grad_z += qd * (grad_q - (qd * grad_q).sum(axis=1, keepdims=True))
    else:
        grad_z += grad_q
    grad = grad_z.reshape(B, N, C).transpose(0, 2, 1)
    return dict(loss=ce_weight * ce + lovasz_weight * lov, ce=ce_weight * ce, lovasz=lovasz_weight * lov, grad=grad,
                present=present, dlde=dlde_all, set_rows=set_idx)
