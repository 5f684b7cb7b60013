"""Parity of the sm_100a deformable-aggregation kernels against the oracle, torch.grid_sample
(the reference's own fallback path) and the committed reference-op golden."""
import os

import numpy as np
import pytest
import torch

import helpers as h
import oracle
from gaussianformer_b200.ops import DeformableAggregationFunction as DAF
from gaussianformer_b200.synthetic import make_daf_inputs

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _run(fms, loc, w, backward_seed=None):
    feat, shape, start = DAF.feature_maps_format([f.cuda() for f in fms])
    feat = feat.contiguous().requires_grad_(backward_seed is not None)
    loc_d = loc.cuda().requires_grad_(backward_seed is not None)
    w_d = w.cuda().requires_grad_(backward_seed is not None)
    out = DAF.apply(feat, shape, start, loc_d, w_d)
    grads = None
    if backward_seed is not None:
        g = torch.randn(out.shape, generator=torch.Generator().manual_seed(backward_seed))
        out.backward(g.cuda())
        grads = (g, feat.grad, loc_d.grad, w_d.grad)
    return feat, shape, start, out, grads


@pytest.mark.parametrize("embed,groups,levels", [
    (128, 4, ((12, 20), (6, 10), (3, 5))),        # vectorised path (C % 128 == 0)
    (256, 8, ((9, 7), (5, 4))),                   # two channel slices per warp
    (16, 4, ((7, 12), (4, 6), (2, 3))),           # scalar fallback path
    (24, 3, ((5, 5),)),
])
def test_daf_forward_backward_vs_oracle(embed, groups, levels):
    fms, loc, w = make_daf_inputs(num_anchor=64, num_pts=5, batch=2, num_cams=3, embed_dims=embed,
                                  num_groups=groups, levels=levels, visible_p=0.5, seed=3)
    loc[0, 0, 0] = torch.tensor([0.0, 0.5]); loc[0, 1, 0] = torch.tensor([1.0, 0.5])
    loc[0, 2, 0] = torch.tensor([0.004, 0.996]); loc[0, 3, 1] = torch.tensor([0.999, 0.001])
    loc[1, 4, 2] = torch.tensor([float("nan"), 0.5])
    feat, shape, start, out, (g, gf, gl, gw) = _run(fms, loc, w, backward_seed=11)
    f_np, s_np, st_np = feat.detach().cpu().numpy(), shape.cpu().numpy(), start.cpu().numpy()
    ref = oracle.daf_forward(f_np, s_np, st_np, loc.numpy(), w.numpy(), "f64")
    h.assert_close(out.detach().cpu().numpy(), ref, what="daf out")
    rf, rl, rw = oracle.daf_backward(f_np, s_np, st_np, loc.numpy(), w.numpy(), g.numpy(), "f64")
    rf32, rl32, rw32 = oracle.daf_backward(f_np, s_np, st_np, loc.numpy(), w.numpy(), g.numpy(), "f32")
    # BASELINE gate, else K x the measured fp32 floor of the oracle's own arithmetic (helpers.assert_grad_parity)
    h.assert_grad_parity(gf.cpu().numpy(), rf, rf32, what="grad feat")
    h.assert_grad_parity(gw.cpu().numpy(), rw, rw32, what="grad weights")
    h.assert_grad_parity(gl.cpu().numpy(), rl, rl32, what="grad loc")


def test_daf_matches_reference_golden():
    path = os.path.join(GOLD, "ref_daf_small.npz")
    if not os.path.exists(path):
        pytest.skip("golden fixture not generated yet")
    gold = np.load(path)
    levels = ((12, 20), (6, 10), (3, 5))
    fms, loc, w = make_daf_inputs(num_anchor=96, num_pts=5, batch=2, num_cams=3, embed_dims=128, num_groups=4,
                                  levels=levels, visible_p=0.5, seed=4)
    _, _, _, out, (g, gf, gl, gw) = _run(fms, loc, w, backward_seed=int(gold["grad_seed"]))
    h.assert_close(out.detach().cpu().numpy(), gold["out"], what="daf out vs reference op")
    # both are fp32 atomically-accumulated sums: the slack is the golden's own measured distance from the fp64 oracle
    feat_t, shape_t, start_t = DAF.feature_maps_format(fms)
    r64 = oracle.daf_backward(feat_t.contiguous().numpy(), shape_t.numpy(), start_t.numpy(), loc.numpy(), w.numpy(), g.numpy(), "f64")
    rows = slice(None, None, int(gold["feat_row_stride"]))      # the golden keeps every stride-th feature row
    for name, mine, ref, truth in (("feat", gf[:, :, rows], gold["grad_feat_rows"], r64[0][:, :, rows]),
                                   ("loc", gl, gold["grad_loc"], r64[1]), ("w", gw, gold["grad_weights"], r64[2])):
        floor = float(np.abs(ref.astype(np.float64) - truth).max())
        err = np.abs(mine.cpu().numpy().astype(np.float64) - ref)
        tol = np.maximum(h.ATOL + h.RTOL * np.abs(ref), (h.K_FLOOR + 1.0) * floor)
        assert (err <= tol).all(), f"grad {name} vs reference op: max err {err.max():.3e}, reference floor {floor:.3e}"


def test_daf_full_size_properties():
    """BASELINE config-2 shape (P = 25600*9, 6 cams, 4 levels, C = 128): linearity in the weights
    and agreement with a sampled oracle subset (the full oracle would take minutes)."""
    fms, loc, w = make_daf_inputs(num_anchor=25600, num_pts=9, seed=0)
    feat, shape, start, out, _ = _run(fms, loc, w)
    out2 = DAF.apply(feat.detach(), shape, start, loc.cuda(), (2 * w).cuda())
    h.assert_close(out2.cpu().numpy(), 2 * out.detach().cpu().numpy(), what="weight linearity")
    sel = torch.randperm(loc.shape[1], generator=torch.Generator().manual_seed(1))[:4096]
    ref = oracle.daf_forward(feat.detach().cpu().numpy(), shape.cpu().numpy(), start.cpu().numpy(),
                             loc[:, sel].contiguous().numpy(), w[:, sel].contiguous().numpy(), "f64")
    h.assert_close(out.detach()[:, sel.cuda()].cpu().numpy(), ref, what="daf sampled subset")


@pytest.mark.parametrize("channels,levels", [
    (128, ((108, 200), (54, 100), (27, 50), (14, 25))),    # BASELINE config-2 maps (1 sample x 6 cameras)
    (24, ((5, 7), (3, 3), (1, 1))),                         # ragged: nothing divides the tile or vector sizes
    (130, ((9, 13),)),
])
def test_feature_maps_format_is_the_reference_layout(channels, levels):
    """The fused table kernel is a pure data movement: bit-exact against the reference's
    reshape + cat + permute (ops/deformable_aggregation.py:78-95), and its gradient is the inverse
    scatter (what autograd derives for the reference's view ops)."""
    gen = torch.Generator().manual_seed(5)
    bs, cams = (1, 6) if channels == 128 else (2, 3)
    maps = [torch.randn(bs, cams, channels, h_, w_, generator=gen).cuda().requires_grad_(True) for h_, w_ in levels]
    col, shape, start = DAF.feature_maps_format(maps)
    assert col.is_contiguous() and col.shape == (bs, cams, sum(h_ * w_ for h_, w_ in levels), channels)
    ref_col = torch.cat([m.detach().reshape(bs, cams, channels, -1) for m in maps], dim=-1).permute(0, 1, 3, 2)
    assert torch.equal(col.detach(), ref_col)
    assert shape.tolist() == [list(l) for l in levels]
    assert start.tolist() == [int(s) for s in np.cumsum([0] + [h_ * w_ for h_, w_ in levels])[:-1]]
    g = torch.randn(col.shape, generator=gen).cuda()
    col.backward(g)
    back = DAF.feature_maps_format([g, shape, start], inverse=True)      # the reference's inverse: views of g
    for m, b in zip(maps, back):
        assert torch.equal(m.grad, b.contiguous())


# ------------------------------------------------------------------------------ fused caller path (SURVEY.md 8f-2)
from gaussianformer_b200.ops import deformable_aggregation_fused, fused_supported  # noqa: E402
from gaussianformer_b200.synthetic import make_daf_fused_inputs, reference_fused_composition  # noqa: E402


@pytest.mark.parametrize("embed,groups,levels,masks", [
    (128, 4, ((12, 20), (6, 10), (3, 5)), "both"),
    (128, 4, ((12, 20), (6, 10), (3, 5)), "point"),
    (128, 4, ((12, 20), (6, 10), (3, 5)), "none"),
    (256, 8, ((9, 7), (5, 4)), "both"),                 # two channel slices per warp, 8 groups
    (128, 1, ((5, 5),), "point"),                       # one group = the whole warp
])
def test_daf_fused_forward_backward_vs_oracle(embed, groups, levels, masks):
    B, A, K, M = 2, 40, 5, 3
    fms, loc, logits, pm, wm = make_daf_fused_inputs(num_anchor=A, num_pts=K, batch=B, num_cams=M, embed_dims=embed,
                                                     num_groups=groups, levels=levels, visible_p=0.5, seed=21,
                                                     attn_drop=0.15)
    loc[0, 2, 0] = torch.tensor([0.004, 0.996]); loc[0, 3, 1] = torch.tensor([0.999, 0.001])
    loc[1, 4, 2] = torch.tensor([float("nan"), 0.5])
    pm = ((loc > 0) & (loc < 1)).all(-1).reshape(B, A, K, M).contiguous()
    pm[0, 0] = False                                     # an anchor no camera sees
    wm[0, 1, :, :, :, 0] = False                         # a group with every entry dropped
    logits[1, 2, 0, 0, 0, 0] = 30.0                      # a dominant entry (softmax range)
    if masks == "point":
        wm = None
    elif masks == "none":
        pm = wm = None
    assert fused_supported(embed, groups, M, len(levels))
    feat, shape, start = DAF.feature_maps_format([f.cuda() for f in fms])
    feat = feat.contiguous().requires_grad_()
    loc_d = loc.cuda().requires_grad_()
    lg_d = logits.cuda().requires_grad_()
    out = deformable_aggregation_fused(feat, shape, start, loc_d, lg_d, None if pm is None else pm.cuda(),
                                       None if wm is None else wm.cuda())
    assert out.shape == (B, A, embed)
    f_np, s_np, st_np = feat.detach().cpu().numpy(), shape.cpu().numpy(), start.cpu().numpy()
    pm_np = None if pm is None else pm.numpy()
    wm_np = None if wm is None else wm.numpy()
    ref = oracle.daf_fused_forward(f_np, s_np, st_np, loc.numpy(), logits.numpy(), pm_np, wm_np, "f64")
    h.assert_close(out.detach().cpu().numpy(), ref, what="fused daf out")
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(5))
    out.backward(g.cuda())
    rf, rl, rw = oracle.daf_fused_backward(f_np, s_np, st_np, loc.numpy(), logits.numpy(), g.numpy(), pm_np, wm_np, "f64")
    rf32, rl32, rw32 = oracle.daf_fused_backward(f_np, s_np, st_np, loc.numpy(), logits.numpy(), g.numpy(), pm_np, wm_np, "f32")
    h.assert_grad_parity(feat.grad.cpu().numpy(), rf, rf32, what="fused grad feat")
    h.assert_grad_parity(lg_d.grad.cpu().numpy(), rw, rw32, what="fused grad logits")
    h.assert_grad_parity(loc_d.grad.cpu().numpy(), rl, rl32, what="fused grad loc")
    if pm is not None:
        assert torch.all(out[0, 0] == 0) and torch.all(lg_d.grad[0, 0] == 0)


def test_daf_fused_rejects_unsupported_shapes():
    assert not fused_supported(16, 4, 3, 3)              # C % 128 != 0
    assert not fused_supported(128, 4, 6, 8)             # more than 32 (camera, level) pairs
    fms, loc, logits, pm, _ = make_daf_fused_inputs(num_anchor=8, num_pts=2, batch=1, num_cams=2, embed_dims=16,
                                                    num_groups=4, levels=((4, 4),), seed=1)
    feat, shape, start = DAF.feature_maps_format([f.cuda() for f in fms])
    with pytest.raises(Exception, match="not supported"):
        deformable_aggregation_fused(feat.contiguous(), shape, start, loc.cuda(), logits.cuda(), pm.cuda())


def test_daf_fused_full_size_equals_the_unfused_route():
    """BASELINE config-2 shape (25 600 anchors x 9 key points, 6 cameras, 4 levels, C = 128): the fused entry
    point against the reference's composition (PyTorch masked softmax -> our drop-in op -> sum over key points)
    on the same GPU, forward and backward."""
    fms, loc, logits, pm, _ = make_daf_fused_inputs(seed=0)
    feat, shape, start = DAF.feature_maps_format([f.cuda() for f in fms])
    feat = feat.contiguous()
    outs, grads = [], []
    g = torch.randn(1, 25600, 128, generator=torch.Generator().manual_seed(2)).cuda()
    for fused in (True, False):
        f = feat.detach().clone().requires_grad_()
        l = loc.cuda().requires_grad_()
        w = logits.cuda().requires_grad_()
        if fused:
            out = deformable_aggregation_fused(f, shape, start, l, w, pm.cuda())
        else:
            out = reference_fused_composition(DAF.apply, f, shape, start, l, w, pm.cuda())
        out.backward(g)
        outs.append(out.detach().cpu().numpy())
        grads.append([t.grad.cpu().numpy() for t in (f, l, w)])
    h.assert_close(outs[0], outs[1], what="fused vs unfused out")
    for name, a, b in zip(("feat", "loc", "logits"), grads[0], grads[1]):
        h.assert_close(a, b, rtol=1e-3, atol=h.grad_tolerance(b), what="fused vs unfused grad " + name)


def test_tma_corner_box_variant_is_bit_identical():
    """The TMA experiment (gf_debug_daf_forward_tma, include/gf_b200_debug.h): one cp.async.bulk.tensor box {C,2,2,1} per
    visible (camera, level) pair with hardware zero fill for corners outside the map -- the same products in the same
    order as the product kernel, so the outputs are equal bit for bit (incl. locations on and beyond the map border)."""
    import ctypes
    from gaussianformer_b200 import _lib
    from gaussianformer_b200.ops.deformable_aggregation import _desc
    levels = ((12, 20), (6, 10), (3, 5))
    fms, loc, w = make_daf_inputs(num_anchor=80, num_pts=5, batch=2, num_cams=3, embed_dims=128, num_groups=4,
                                  levels=levels, visible_p=0.6, seed=7)
    loc[0, 0, 0] = torch.tensor([0.004, 0.996]); loc[0, 1, 1] = torch.tensor([0.999, 0.001]); loc[1, 2, 2] = torch.tensor([0.5, 0.0])
    feat, shape, start = DAF.feature_maps_format([f.cuda() for f in fms])
    feat = feat.contiguous()
    loc_d, w_d = loc.cuda(), w.cuda()
    ref = DAF.apply(feat, shape, start, loc_d, w_d)
    d = _desc(feat, shape, loc_d, w_d)
    hs = (ctypes.c_int32 * (2 * len(levels)))(*[v for hw in levels for v in hw])
    hst = (ctypes.c_int32 * len(levels))(*[int(v) for v in start.cpu().tolist()])
    out = torch.empty_like(ref)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().gf_debug_daf_forward_tma(ctypes.byref(d), ctypes.c_void_p(feat.data_ptr()), hs, hst,
                                                  ctypes.c_void_p(loc_d.data_ptr()), ctypes.c_void_p(w_d.data_ptr()),
                                                  ctypes.c_void_p(out.data_ptr()), stream))
    torch.cuda.synchronize()
    assert torch.equal(out, ref)
