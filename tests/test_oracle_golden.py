"""Pins the CPU oracle to the reference itself: tests/golden/ref_*.npz were produced by the
reference CUDA ops (built from /root/reference by oracle/build_ref.py) on a B200 with
tests/golden/make_golden_ref.py; inputs are regenerated from (config, seed)."""
import os

import numpy as np
import pytest
import torch

import helpers as h
import oracle
from gaussianformer_b200.ops.deformable_aggregation import feature_maps_format
from gaussianformer_b200.synthetic import make_daf_inputs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = [
    ("ref_splat_base_tiny", "tiny", 0, False, False),
    ("ref_splat_base_tiny_perturb", "tiny", 1, True, False),
    ("ref_splat_prob_tiny", "tiny_prob", 0, False, False),
    ("ref_splat_probfast_tiny", "tiny_prob", 2, True, True),
]


@pytest.mark.parametrize("fixture,cfg,seed,perturb,per_axis", CASES)
def test_splat_oracle_matches_reference_op(fixture, cfg, seed, perturb, per_axis):
    gold = np.load(os.path.join(GOLD, fixture + ".npz"))
    kw, inp, variant = h.splat_case(cfg, seed, perturb, per_axis=per_axis)
    gen = torch.Generator().manual_seed(int(gold["grad_seed"]))
    N = inp["pts"].shape[1]
    for precision in ("f32", "f64"):
        fwd = h.oracle_forward(kw, inp, variant, precision)
        assert fwd["num_pairs"] == int(gold["num_pairs"])          # identical inclusion sets
        if variant == "base":
            h.assert_close(fwd["logits"], gold["logits"], what="logits")
        else:
            z = gold["probability"]
            stable = np.abs(z - 1e-9) > 1e-10
            h.assert_close(fwd["logits"][stable], gold["logits"][stable], what="logits")
            # exact fallback rows: 1/17 on the first 17 channels, untouched zero on the last
            fb = z <= 1e-9
            if fb.any():
                assert np.all(gold["logits"][fb][:, 17] == 0) and np.allclose(gold["logits"][fb][:, :17], 1 / 17)
            for k in ("bin_logits", "density", "probability"):
                h.assert_close(fwd[k], gold[k], what=k)
    gen = torch.Generator().manual_seed(int(gold["grad_seed"]))
    if variant == "base":
        grads = (torch.randn(N, 18, generator=gen).numpy(),)
        saved = None
    else:
        grads = (torch.randn(N, 18, generator=gen).numpy(), torch.randn(N, generator=gen).numpy(),
                 torch.randn(N, generator=gen).numpy())
        saved = dict(logits=gold["logits"], bin_logits=gold["bin_logits"], probability=gold["probability"])
    for precision in ("f32", "f64"):
        gm, go, gs, gc = h.oracle_backward(kw, inp, variant, grads, saved, precision)
        for name, mine, ref in (("means", gm, gold["means_grad"]), ("opa", go, gold["opacity_grad"]),
                                ("sem", gs, gold["semantics_grad"]), ("cov", gc, gold["cov_grad"])):
            h.assert_close(mine, ref, rtol=2e-3, atol=5 * h.grad_tolerance(ref), what=f"{precision} grad {name}")


def test_splat_oracle_matches_reference_op_mid_size():
    """2000 Gaussians + the whole-grid "empty" one on the full 200 x 200 x 16 grid (config 2's grid): identical pair
    count, the sampled logits rows and the column sums of ALL rows, and the complete gradients of the reference op."""
    path = os.path.join(GOLD, "ref_splat_base_mid.npz")
    if not os.path.exists(path):
        pytest.skip("mid-size golden not generated yet")
    gold = np.load(path)
    kw, inp, variant = h.splat_case("gs25600_solid", 7, False, dict(G=2000))
    stride = int(gold["row_stride"])
    fwd = h.oracle_forward(kw, inp, variant, "f64")
    assert fwd["num_pairs"] == int(gold["num_pairs"])
    h.assert_close(fwd["logits"][::stride], gold["logits_rows"], what="sampled logits rows")
    # column sums over all 640 000 rows: the fp32 reference rows sum to the fp64 oracle's within their elementwise gate
    tol = h.ATOL * fwd["logits"].shape[0] + h.RTOL * gold["logits_abs_colsum"]
    assert np.all(np.abs(fwd["logits"].sum(0) - gold["logits_colsum"]) <= tol)
    N = inp["pts"].shape[1]
    g = torch.randn(N, 18, generator=torch.Generator().manual_seed(int(gold["grad_seed"]))).numpy()
    g64, g32 = h.oracle_grads(kw, inp, variant, (g,))
    ref = {"means": gold["means_grad"], "opa": gold["opacity_grad"], "sem": gold["semantics_grad"],
           "cov": oracle.cov6_grad_to_3x3(gold["cov_grad"])}
    for name in ref:   # the reference op is an fp32 evaluation: gate, else K x the fp32 oracle's own floor
        h.assert_grad_parity(ref[name], g64[name], g32[name], what="reference-op golden grad " + name)


def test_daf_oracle_matches_reference_op():
    gold = np.load(os.path.join(GOLD, "ref_daf_small.npz"))
    levels = ((12, 20), (6, 10), (3, 5))
    fms, loc, w = make_daf_inputs(num_anchor=96, num_pts=5, batch=2, num_cams=3, embed_dims=128, num_groups=4,
                                  levels=levels, visible_p=0.5, seed=4)
    feat, shape, start = feature_maps_format(fms)
    args = (feat.contiguous().numpy(), shape.numpy(), start.numpy(), loc.numpy(), w.numpy())
    h.assert_close(oracle.daf_forward(*args, "f32"), gold["out"], what="daf out")
    g = torch.randn(gold["out"].shape, generator=torch.Generator().manual_seed(int(gold["grad_seed"]))).numpy()
    gf, gl, gw = oracle.daf_backward(*args, g, "f64")
    rows = slice(None, None, int(gold["feat_row_stride"]))      # the golden keeps every stride-th feature row
    for name, mine, ref in (("feat", gf[:, :, rows], gold["grad_feat_rows"]), ("loc", gl, gold["grad_loc"]),
                            ("w", gw, gold["grad_weights"])):
        h.assert_close(mine, ref, rtol=1e-3, atol=h.grad_tolerance(ref), what="grad " + name)
