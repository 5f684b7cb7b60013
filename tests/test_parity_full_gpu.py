"""Op-vs-op parity at the FULL BASELINE.json sizes (configs 2, 3, 4): the sm_100a path (public module -> C ABI)
against (a) the UNMODIFIED reference CUDA op and (b) the fp64 C oracle, on the same seeded inputs: forward, all four
gradients, arg-max agreement and MeanIoU.  The reference op's side is read from tests/golden/ref_parity_full_<case>.npz
(made on a B200 by tests/golden/make_golden_ref.py): its pair count, its forward outputs on a seeded sample of voxels
and its gradient rows of a seeded sample of Gaussians, its whole-tensor distance from the fp64 oracle per gradient,
and its arg-max wherever that differs from the fp64 oracle's, i.e. its arg-max on every voxel.

Gates (BASELINE.md "Parity gates"):

* forward outputs: ``|new - ref| <= 1e-5 + 1e-4*|ref|`` elementwise, against the reference op AND the fp64 oracle;
* gradients: the same elementwise gate wherever it holds.  A gradient entry is a sum of 10^2..10^6 signed fp32
  terms, so where the gate cannot hold the bound is the MEASURED fp32 floor of the reference itself on the same
  tensor: ``K_FLOOR x max(|reference op - fp64 oracle|, |fp32 oracle - fp64 oracle|)`` (printed per tensor and
  written to gpurun_out/parity_full_*.json); the new op must be no further from fp64 truth than K_FLOOR times the
  reference's own fp32 arithmetic is;
* arg-max: identical on >= 99.99 % of the voxels, every difference confined to voxels whose top two classes are
  within the elementwise tolerance of each other (numerical ties);
* MeanIoU (misc/metric_util.py:35-111, labels per SURVEY.md 8d): equal within 1e-4 points on the voxels whose arg-max
  is numerically decided; the raw figure over all voxels is reported next to the reference op's own distance from the
  fp64 oracle and must stay within K_FLOOR x that floor (+ 1e-4).
"""
import json
import os

import numpy as np
import pytest
import torch

import helpers as h

pytestmark = pytest.mark.gpu

K_FLOOR = 4.0
GRAD_SEED = 4242   # + the case's seed: the upstream gradients
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def _np(x):
    return x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)


def _gate(err, ref):
    return err <= h.ATOL + h.RTOL * np.abs(ref)


def _tie_mask(ref_logits):
    """voxels whose top two classes (of the fp64 oracle) are within twice the elementwise tolerance"""
    srt = np.sort(ref_logits, axis=1)
    return (srt[:, -1] - srt[:, -2]) <= 2 * (h.ATOL + h.RTOL * np.abs(srt[:, -1]))


CASES = [
    # id, config, seed, perturb, per_axis
    ("cfg2_gs25600_solid", "gs25600_solid", 0, False, False),
    ("cfg2_gs25600_solid_perturbed", "gs25600_solid", 1, True, False),
    ("cfg3_gs144000", "gs144000", 0, False, False),
    ("cfg4_prob_gs6400", "prob_gs6400", 0, False, False),
    ("cfg4_probfast_gs6400", "prob_gs6400", 1, True, True),
]


@pytest.mark.parametrize("case,cfg,seed,perturb,per_axis", CASES, ids=[c[0] for c in CASES])
def test_full_size_vs_reference_op_and_fp64_oracle(case, cfg, seed, perturb, per_axis):
    import oracle
    from gaussianformer_b200.metric import miou_parity, synthetic_labels

    kw, inp, variant = h.splat_case(cfg, seed, perturb, per_axis=per_axis)
    prob = variant != "base"
    gold = np.load(os.path.join(GOLD, f"ref_parity_full_{case}.npz"))
    rows, gaussians = gold["rows"], gold["gaussians"]
    report = {"case": case, "G": int(inp["means"].shape[1]), "N": int(inp["pts"].shape[1]), "variant": variant,
              "reference_op": f"stored: {rows.size} voxels, {gaussians.size} Gaussians",
              "gate": f"{h.ATOL} + {h.RTOL}*|ref|", "k_floor": K_FLOOR}

    # ---- the op under test ------------------------------------------------------------------------------------------
    m = h.make_module(kw, variant)
    t = h.to_dev(inp, requires_grad=True)
    out = m(t["pts"], t["means"], t["opa"], t["sem"], t["scales"], t["cov"])
    outs = (out,) if not prob else tuple(out)
    gen = torch.Generator().manual_seed(GRAD_SEED + seed)
    grads = tuple(torch.randn(o.shape, generator=gen) for o in outs)
    torch.autograd.backward(list(outs), [g.cuda() for g in grads])
    new = {"logits": _np(outs[0])}
    if prob:
        new.update(bin_logits=_np(outs[1]), density=_np(outs[2]))
    new_g = {"means": _np(t["means"].grad[0]), "opa": _np(t["opa"].grad[0]), "sem": _np(t["sem"].grad[0]),
             "cov": _np(t["cov"].grad[0])}
    assert float(np.abs(new_g["cov"].reshape(-1, 9)[:, [3, 6, 7]]).max()) == 0.0   # lower triangle: no gradient
    del out, outs, t, m
    torch.cuda.empty_cache()

    # ---- fp64 and fp32 C oracle -------------------------------------------------------------------------------------
    g_np = tuple(g.numpy() for g in grads)
    o64 = h.oracle_forward(kw, inp, variant, "f64")
    o32 = h.oracle_forward(kw, inp, variant, "f32")
    report["pairs"] = int(o64["num_pairs"])

    def oracle_grads(fw, precision):
        saved = None if not prob else dict(logits=fw["logits"], bin_logits=fw["bin_logits"], probability=fw["probability"])
        gm, go, gs, gc = h.oracle_backward(kw, inp, variant, g_np, saved, precision)
        return {"means": gm, "opa": go, "sem": gs, "cov": oracle.cov6_grad_to_3x3(gc)}
    g64, g32 = oracle_grads(o64, "f64"), oracle_grads(o32, "f32")

    # ---- the reference CUDA op (stored) -------------------------------------------------------------------------------
    assert int(gold["num_pairs"]) == int(o64["num_pairs"])                 # identical inclusion sets
    ref = {k: gold[k + "_rows"] for k in (("logits", "bin_logits", "density") if prob else ("logits",))}
    ref_g = {k: gold[k + "_grad_rows"] for k in ("means", "opa", "sem", "cov")}

    # ---- forward: BASELINE gate against both -------------------------------------------------------------------------
    stable = np.ones(new["logits"].shape[0], bool)
    if prob:   # voxels sitting on the Z > 1e-9 fallback switch may take either branch (localagg_prob/src/forward.cu:92)
        stable = np.abs(o64["probability"] - 1e-9) > 1e-10
        stable[gold["unstable_rows"]] = False
    report["forward"] = {}
    for name in new:
        sel = stable if name == "logits" else np.ones_like(stable)
        on = sel[rows]                                                      # the stored voxels among them
        entry = {}
        for against, got, want in (("fp64_oracle", new[name][sel], o64[name][sel]),
                                   ("reference_op", new[name][rows][on], ref[name][on])):
            err = np.abs(got.astype(np.float64) - want)
            entry[against] = {"max_abs_err": float(err.max()), "outside_gate": int((~_gate(err, want)).sum())}
        entry["reference_op_vs_fp64"] = float(np.abs(ref[name][on].astype(np.float64) - o64[name][rows][on]).max())
        report["forward"][name] = entry
    for name, entry in report["forward"].items():
        for against in ("fp64_oracle", "reference_op"):
            assert entry[against]["outside_gate"] == 0, (case, name, against, entry)

    # ---- gradients: BASELINE gate, else K_FLOOR x the reference's own measured fp32 floor ---------------------------------
    report["gradients"] = {}
    for name in ("means", "opa", "sem", "cov"):
        want = np.asarray(g64[name], np.float64)
        err = np.abs(new_g[name].astype(np.float64) - want)
        floor32 = float(np.abs(np.asarray(g32[name], np.float64) - want).max())
        floor_ref = float(gold[name + "_grad_floor"])
        floor = max(floor32, floor_ref)
        ok = _gate(err, want) | (err <= K_FLOOR * floor)
        entry = {"max_abs_ref": float(np.abs(want).max()), "max_abs_err_vs_fp64": float(err.max()),
                 "outside_baseline_gate": int((~_gate(err, want)).sum()), "of": int(err.size),
                 "fp32_oracle_floor": floor32, "reference_op_floor": floor_ref, "outside_k_floor": int((~ok).sum())}
        e2 = np.abs(new_g[name][gaussians].astype(np.float64) - ref_g[name])
        entry["max_abs_err_vs_reference_op"] = float(e2.max())
        # the two fp32 ops against each other: the gate, else both within their floors of the truth
        ok2 = _gate(e2, ref_g[name]) | (e2 <= (K_FLOOR + 1.0) * floor)
        entry["outside_vs_reference_op"] = int((~ok2).sum())
        report["gradients"][name] = entry
    for name, entry in report["gradients"].items():
        assert entry["outside_k_floor"] == 0, (case, name, entry)
        assert entry["outside_vs_reference_op"] == 0, (case, name, entry)

    # ---- arg-max agreement and MeanIoU --------------------------------------------------------------------------------------
    truth = o64["logits"]
    C = truth.shape[1]
    tie = _tie_mask(truth)
    am_new, am_64 = new["logits"].argmax(1), truth.argmax(1)
    am_ref = am_64.copy()
    am_ref[gold["argmax_flip_rows"]] = gold["argmax_flip_class"]
    against = "reference_op"
    diff = am_new != am_ref
    labels, mask = synthetic_labels(truth, C)
    r_all = miou_parity(am_new, am_ref, labels, mask, C)
    decided = torch.as_tensor(~tie)
    r_dec = miou_parity(am_new, am_ref, labels, mask & decided, C)
    floor_all = miou_parity(am_ref, am_64, labels, mask, C)          # the reference's own distance from fp64 truth
    report["argmax"] = {"against": against, "differences": int(diff.sum()), "differences_on_decided_voxels": int((diff & ~tie).sum()),
                        "tie_voxels": int(tie.sum()), "agreement": float(1.0 - diff.mean()),
                        "reference_vs_fp64_differences": int((am_ref != am_64).sum())}
    report["miou"] = {"new": r_all["new"], "ref": r_all["ref"], "abs_diff_all_voxels": r_all["abs_diff"],
                      "abs_diff_decided_voxels": r_dec["abs_diff"], "reference_vs_fp64_abs_diff": floor_all["abs_diff"]}
    out_dir = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, f"parity_full_{case}.json"), "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))
    assert report["argmax"]["differences_on_decided_voxels"] == 0, report["argmax"]
    # >= 99.99 % agreement; where the reference op itself disagrees with the fp64 oracle on more voxels than that
    # (far-tail voxels whose top two classes tie within rounding), the bound is K_FLOOR x the reference's own rate
    ref_rate = report["argmax"]["reference_vs_fp64_differences"] / truth.shape[0]
    assert report["argmax"]["agreement"] >= min(0.9999, 1.0 - K_FLOOR * ref_rate), report["argmax"]
    assert 1.0 - float((diff & ~tie).mean()) >= 0.9999
    assert r_dec["abs_diff"] <= 1e-4, report["miou"]
    assert r_all["abs_diff"] <= 1e-4 + K_FLOOR * floor_all["abs_diff"], report["miou"]
