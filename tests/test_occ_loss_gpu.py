"""GPU: the occupancy loss op (gaussianformer_b200.loss) against the fp64 oracle and the reference's own loss code,
over shapes, masks, ignore labels, ties, determinism, sync-freedom, graph capture, the splat end to end and the
drop-in module."""
import os

import numpy as np
import pytest
import torch

import helpers as h
from gaussianformer_b200.loss import OccupancyLoss, occupancy_loss
from gaussianformer_b200.synthetic import make_occ_loss_inputs, reference_occupancy_loss
from oracle import occ_loss as O

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def run_op(d, mask="from_inputs", validate=True, **kw):
    kw.setdefault("use_softmax", d["use_softmax"])
    pred = d["pred"].cuda().requires_grad_()
    m = d["occ_mask"] if mask == "from_inputs" else mask
    loss, parts = occupancy_loss(pred, d["labels"].cuda(), None if m is None else m.cuda(),
                                 d["class_weights"].cuda(), validate=validate, **kw)
    loss.backward()
    return dict(loss=loss.item(), ce=parts["loss_voxel_ce"].item(), lovasz=parts["loss_voxel_lovasz"].item(),
                grad=pred.grad.cpu().numpy())


def run_oracle(d, mask="from_inputs", **kw):
    kw.setdefault("use_softmax", d["use_softmax"])
    m = d["occ_mask"] if mask == "from_inputs" else mask
    args = (d["pred"].numpy(), d["labels"].numpy(), None if m is None else m.numpy(), d["class_weights"].numpy())
    return O.occ_loss(*args, **kw), O.occ_loss(*args, precision="f32", **kw)


def check(got, o64, o32, what):
    for k in ("loss", "ce", "lovasz"):
        if np.isnan(o64[k]):
            assert np.isnan(got[k]), f"{what} {k}: {got[k]} is not NaN"
            continue
        tol = max(h.ATOL + h.RTOL * abs(o64[k]), h.K_FLOOR * abs(o32[k] - o64[k]))
        assert abs(got[k] - o64[k]) <= tol, f"{what} {k}: {got[k]!r} vs {o64[k]!r}"
    h.assert_grad_parity(got["grad"], o64["grad"], o32["grad"], what=f"{what} grad")


def op_vs_oracle(d, what, **kw):
    got = run_op(d, **kw)
    o64, o32 = run_oracle(d, **kw)
    check(got, o64, o32, what)
    return got, o64


@pytest.mark.parametrize("fixture,case", [("ref_occ_loss_small", "small"), ("ref_occ_loss_small_prob", "small_prob"),
                                          ("ref_occ_loss_cfg2", "cfg2")])
def test_fixtures(fixture, case):
    g = np.load(os.path.join(GOLDEN, fixture + ".npz"))
    d = make_occ_loss_inputs(case, int(g["seed"]))
    got, o64 = op_vs_oracle(d, fixture)
    _, o32 = run_oracle(d)
    rows = lambda a: a.transpose(0, 2, 1).reshape(-1, a.shape[1])   # noqa: E731
    mine, r64, r32 = rows(got["grad"]), rows(o64["grad"]), rows(o32["grad"])
    sel = np.arange(0, mine.shape[0], int(g["row_stride"]))
    if "top_rows" in g:
        sel = np.concatenate([sel, g["top_rows"]])
        gold = np.concatenate([g["grad_rows"], g["grad_top"]])
    else:
        gold = g["grad_rows"]
    # against the reference's own result, with the golden's measured distance from the fp64 oracle as extra slack
    h.assert_grad_parity(mine[sel], gold, r32[sel], what=f"{fixture} vs reference grad",
                         extra_floor=float(np.abs(gold - r64[sel]).max()))
    for k in ("loss", "ce", "lovasz"):
        slack = max(abs(float(g[k]) - o64[k]), abs(o32[k] - o64[k]))
        assert abs(got[k] - float(g[k])) <= max(h.ATOL + h.RTOL * abs(float(g[k])), (h.K_FLOOR + 1) * slack), k


@pytest.mark.parametrize("B", [1, 2, 3])
@pytest.mark.parametrize("C", [16, 18, 20])
@pytest.mark.parametrize("use_softmax", [True, False])
def test_shapes(B, C, use_softmax):
    d = make_occ_loss_inputs("small", 10 * B + C, empty_label=C - 1,
                             overrides=dict(B=B, N=4099 + 17 * B, C=C, use_softmax=use_softmax))
    op_vs_oracle(d, f"B={B} C={C}", lovasz_ignore=C - 1, empty_label=C - 1)


@pytest.mark.parametrize("use_softmax", [True, False])
def test_single_point(use_softmax):
    d = make_occ_loss_inputs("small", 5, overrides=dict(B=1, N=1, use_softmax=use_softmax))
    d["labels"][:] = 3
    op_vs_oracle(d, "N=1", mask=None)


@pytest.mark.parametrize("mask", ["none", "all_false", "partial"])
def test_masks(mask):
    d = make_occ_loss_inputs("small", 6)
    m = {"none": None, "all_false": torch.zeros_like(d["occ_mask"]),
         "partial": torch.rand(d["labels"].shape, generator=torch.Generator().manual_seed(0)) < 0.3}[mask]
    got, _ = op_vs_oracle(d, f"mask={mask}", mask=m)
    if mask == "all_false":
        assert np.isnan(got["ce"]) and got["lovasz"] == 0.0 and not got["grad"].any()


@pytest.mark.parametrize("use_softmax", [True, False])
def test_ignore_empty_and_ignore_labels(use_softmax):
    d = make_occ_loss_inputs("small", 7, overrides=dict(use_softmax=use_softmax))
    d["labels"][:, ::7] = 255
    op_vs_oracle(d, "ignore_empty", ignore_empty=True)
    op_vs_oracle(d, "labels 255")
    op_vs_oracle(d, "no lovasz_ignore", lovasz_ignore=None)


def test_out_of_range_labels_set_the_status_bit():
    d = make_occ_loss_inputs("small", 8)
    d["labels"][0, 5] = 30
    d["occ_mask"][0, 5] = True
    with pytest.raises(ValueError, match="labels outside"):
        run_op(d, validate=True)
    got = run_op(d, validate=False)                                  # the row contributes nothing
    check(got, *run_oracle(d), "out of range, validate off")


def test_every_point_one_class():
    d = make_occ_loss_inputs("small", 9)
    d["labels"][:] = 4
    got, o64 = op_vs_oracle(d, "one class", mask=None)
    assert o64["present"] == [4]


@pytest.mark.parametrize("use_softmax", [False, True])
def test_exact_ties(use_softmax):
    gen = torch.Generator().manual_seed(11)
    d = make_occ_loss_inputs("small", 11, overrides=dict(use_softmax=use_softmax))
    levels = torch.tensor([0.0, 0.25, 0.5, 0.75, 1.0]) if not use_softmax else torch.tensor([-1.0, 0.0, 1.0])
    d["pred"] = levels[torch.randint(0, len(levels), d["pred"].shape, generator=gen)]
    if use_softmax:   # identical rows give identical probabilities: exact ties within each class
        d["pred"][:, :, 1::2] = d["pred"][:, :, 0:-1:2]
    got, o64 = op_vs_oracle(d, "ties")
    # both order ties by point index, so the gradient agrees elementwise; the tie-group sums then agree a fortiori
    assert abs(got["lovasz"] - o64["lovasz"]) <= 1e-5 * max(1.0, abs(o64["lovasz"]))


def test_deterministic():
    d = make_occ_loss_inputs("cfg2", 12)
    a, b = run_op(d), run_op(d)
    assert a["loss"] == b["loss"] and a["ce"] == b["ce"] and a["lovasz"] == b["lovasz"]
    assert np.array_equal(a["grad"].view(np.uint32), b["grad"].view(np.uint32))


def test_no_host_sync():
    d = make_occ_loss_inputs("small", 13)
    pred = d["pred"].cuda().requires_grad_()
    lab, m, w = d["labels"].cuda(), d["occ_mask"].cuda(), d["class_weights"].cuda()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss, _ = occupancy_loss(pred, lab, m, w, validate=False)
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.isfinite(pred.grad).all()


def test_cuda_graph_replay_equals_eager():
    d0, d1 = make_occ_loss_inputs("small", 14), make_occ_loss_inputs("small", 15)
    pred = d0["pred"].cuda().requires_grad_()
    lab, m, w = d0["labels"].cuda(), d0["occ_mask"].cuda(), d0["class_weights"].cuda()

    def step():
        loss, _ = occupancy_loss(pred, lab, m, w, validate=False)
        return loss, torch.autograd.grad(loss, pred)[0]

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        loss_s, grad_s = step()
    with torch.no_grad():
        pred.copy_(d1["pred"].cuda())
    lab.copy_(d1["labels"].cuda())
    m.copy_(d1["occ_mask"].cuda())
    w.copy_(d1["class_weights"].cuda())
    g.replay()
    torch.cuda.synchronize()
    eager = run_op(d1)
    assert loss_s.item() == eager["loss"]
    assert np.array_equal(grad_s.cpu().numpy(), eager["grad"])


def _splat_then_loss(variant, loss_fn):
    """GaussianHead's order: splat -> [1, C, N] prediction -> loss -> backward; returns the Gaussians' gradients."""
    cfg = "tiny" if variant == "base" else "tiny_prob"
    kw, inp, var = h.splat_case(cfg, 3, False)
    m = h.make_module(kw, var)
    t = h.to_dev(inp, requires_grad=True)
    out = m(t["pts"], t["means"], t["opa"], t["sem"], t["scales"], t["cov"])
    if var == "base":
        pred = out[None].transpose(1, 2)
    else:   # the GF-2 geosem composition, model/head/gaussian_head.py:165-172
        logits, binl, _ = out
        geosem = torch.cat([logits[:, :-1] * binl.unsqueeze(-1), 1 - binl.unsqueeze(-1)], dim=-1)
        pred = geosem[None].transpose(1, 2)
        assert float(pred.min()) >= 0.0 and float(pred.max()) <= 1.0
    N = pred.shape[2]
    d = make_occ_loss_inputs("small", 21, overrides=dict(B=1, N=N))
    loss = loss_fn(pred, d["labels"].cuda(), d["occ_mask"].cuda(), d["class_weights"].cuda(), var == "base")
    loss.backward()
    return {k: t[k].grad.cpu().numpy() for k in ("means", "opa", "sem", "cov")}


@pytest.mark.parametrize("variant", ["base", "prob"])
def test_end_to_end_through_the_splat(variant):
    mine = _splat_then_loss(variant, lambda p, y, m, w, sm: occupancy_loss(p, y, m, w, use_softmax=sm)[0])
    ref = _splat_then_loss(variant, lambda p, y, m, w, sm: reference_occupancy_loss(p, y, m, w, use_softmax=sm)[0])
    for k in mine:
        scale = max(1.0, float(np.abs(ref[k]).max()))
        h.assert_close(mine[k], ref[k], rtol=1e-4, atol=1e-5 * scale, what=f"{variant} grad {k}")


@pytest.mark.parametrize("use_softmax", [True, False])
def test_drop_in_module_matches_reference_composition(use_softmax):
    manual = (0.5 + 0.8 * torch.rand(18, generator=torch.Generator().manual_seed(5))).tolist()
    mod = OccupancyLoss(weight=1.0, empty_label=17, num_classes=18, use_focal_loss=False, use_dice_loss=False,
                        balance_cls_weight=True, multi_loss_weights=dict(loss_voxel_ce_weight=10.0,
                                                                         loss_voxel_lovasz_weight=1.0),
                        use_sem_geo_scal_loss=False, use_lovasz_loss=True, lovasz_ignore=17,
                        manual_class_weight=manual, lovasz_use_softmax=use_softmax).cuda()
    d = [make_occ_loss_inputs("small", 30 + i, overrides=dict(B=1, use_softmax=use_softmax)) for i in range(2)]
    lab, m = d[0]["labels"].cuda(), d[0]["occ_mask"].cuda()
    preds = [x["pred"].cuda().requires_grad_() for x in d]
    loss = mod({"pred_occ": preds, "sampled_xyz": None, "sampled_label": lab, "occ_mask": m})
    loss.backward()
    refs = [x["pred"].cuda().requires_grad_() for x in d]
    ref = sum(reference_occupancy_loss(p, lab, m, mod.class_weights, use_softmax=use_softmax)[0] for p in refs) / 2
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 1e-5 + 1e-4 * abs(ref.item())
    for p, r in zip(preds, refs):
        g, gr = p.grad.cpu().numpy(), r.grad.cpu().numpy()
        h.assert_close(g, gr, rtol=1e-4, atol=1e-5 * max(1.0, float(np.abs(gr).max())), what="module grad")
