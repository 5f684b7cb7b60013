"""Generates tests/golden/ref_*.npz from the REFERENCE CUDA ops themselves.

Run on a B200 box (the reference kernels are CUDA-only):

    gpurun -- 'python tests/golden/make_golden_ref.py gpurun_out/golden'

then copy gpurun_out/golden/*.npz into tests/golden/.  Inputs are NOT stored: they are re-created
bit-identically from (config name, seed) by gaussianformer_b200.synthetic on the CPU.  oracle/ref_op.py
restates the reference's Python host preparation with torch ops on the GPU, as the reference does
(model/head/localagg/local_aggregate/__init__.py:137-143), around the unmodified native op.
The mid-size fixture (2000 Gaussians + the whole-grid one on the full 200 x 200 x 16 grid) stores every 61st logits
row, the fp64 column sums of all rows and the complete gradients (0.9 MB instead of 46 MB).
The DAF fixture stores every FEAT_ROW_STRIDE-th feature row of the feature gradient.
The full-size parity fixtures (ref_parity_full_<case>.npz, the cases of tests/test_parity_full_gpu.py) store what that
test compares with the reference op: see run_parity_full.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gaussianformer_b200.synthetic import make_daf_inputs, make_splat_inputs  # noqa: E402
from gaussianformer_b200.ops.deformable_aggregation import feature_maps_format  # noqa: E402
from oracle import build_ref  # noqa: E402

SPLAT_CASES = [  # (fixture, config, seed, overrides, module, per_axis, perturb)
    ("ref_splat_base_tiny", "tiny", 0, None, "gf_ref_localagg", False, False),
    ("ref_splat_base_tiny_perturb", "tiny", 1, None, "gf_ref_localagg", False, True),
    ("ref_splat_prob_tiny", "tiny_prob", 0, None, "gf_ref_localagg_prob", False, False),
    ("ref_splat_probfast_tiny", "tiny_prob", 2, None, "gf_ref_localagg_prob_fast", True, True),
]
# mid-size: 2000 Gaussians + the whole-grid "empty" one on the FULL 200 x 200 x 16 grid (config 2's grid)
MID_CASE = ("ref_splat_base_mid", "gs25600_solid", 7, dict(G=2000), "gf_ref_localagg", False, False)


MID_STRIDE = 61   # the mid-size golden keeps every 61st logits row (the full 640000 x 18 tensor would be 46 MB)
FEAT_ROW_STRIDE = 4   # the DAF golden keeps every 4th feature row of grad_feat (all of it would be 0.97 MB)
PARITY_ROWS = 256     # voxels and Gaussians (at most) stored by each full-size parity fixture
PARITY_WORST = 32     # of which chosen by the reference op's distance from the fp64 oracle, the rest seeded


def run_splat(name, cfg, seed, overrides, modname, per_axis, perturb, outdir, row_stride=1):
    """One sample through the UNMODIFIED reference op (oracle/ref_op.py restates its Python host preparation)."""
    from oracle import ref_op
    kw, inp, variant = make_splat_inputs(cfg, seed=seed, perturb=perturb, overrides=overrides)
    if per_axis:
        variant = "prob_fast"
    gen = torch.Generator().manual_seed(1000 + seed)
    N = inp["pts"].shape[1]
    grads = (torch.randn(N, 18, generator=gen),)
    if variant != "base":
        grads = grads + (torch.randn(N, generator=gen), torch.randn(N, generator=gen))
    r = ref_op.splat(kw, inp, variant, grads)
    save = {k: v for k, v in r.items() if k != "num_pairs"}
    arrays = {k: v.detach().cpu().numpy() for k, v in save.items()}
    arrays["num_pairs"] = np.int64(r["num_pairs"])
    arrays["grad_seed"] = np.int64(1000 + seed)
    if row_stride > 1:   # mid-size fixture: a row sample of the logits + per-class column sums of ALL rows (fp64)
        full = arrays.pop("logits")
        arrays["logits_rows"] = full[::row_stride].copy()
        arrays["row_stride"] = np.int64(row_stride)
        arrays["logits_colsum"] = full.astype(np.float64).sum(0)
        arrays["logits_abs_colsum"] = np.abs(full.astype(np.float64)).sum(0)
    np.savez_compressed(os.path.join(outdir, name + ".npz"), **arrays)
    print(name, {k: getattr(v, "shape", v) for k, v in arrays.items()})


def run_daf(outdir):
    mod = build_ref.load_ref("gf_ref_daf")
    dev = torch.device("cuda")
    levels = ((12, 20), (6, 10), (3, 5))
    fms, loc, w = make_daf_inputs(num_anchor=96, num_pts=5, batch=2, num_cams=3, embed_dims=128, num_groups=4,
                                  levels=levels, visible_p=0.5, seed=4)
    feat, shape, start = feature_maps_format(fms)
    feat, loc, w = feat.contiguous().to(dev), loc.to(dev), w.to(dev)
    shape_i, start_i = shape.int().to(dev), start.int().to(dev)
    out = mod.deformable_aggregation_forward(feat, shape_i, start_i, loc, w)
    g = torch.randn(out.shape, generator=torch.Generator().manual_seed(2004)).to(dev)
    gf, gl, gw = torch.zeros_like(feat), torch.zeros_like(loc), torch.zeros_like(w)
    mod.deformable_aggregation_backward(feat, shape_i, start_i, loc, w, g, gf, gl, gw)
    torch.cuda.synchronize()
    np.savez_compressed(os.path.join(outdir, "ref_daf_small.npz"), out=out.cpu().numpy(),
                        grad_feat_rows=gf[:, :, ::FEAT_ROW_STRIDE].cpu().numpy(), feat_row_stride=np.int64(FEAT_ROW_STRIDE),
                        grad_loc=gl.cpu().numpy(), grad_weights=gw.cpu().numpy(), grad_seed=np.int64(2004))
    print("ref_daf_small", out.shape)


def run_rotation(outdir):
    """The reference's quaternion -> rotation helper (model/utils/utils.py, CPU) on the quaternions of
    tests/test_host_logic.py::test_rotation_matrix_equals_reference_helper."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_utils", os.path.join(build_ref.REF, "model", "utils", "utils.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    q = torch.randn(64, 4, generator=torch.Generator().manual_seed(1))
    np.savez_compressed(os.path.join(outdir, "ref_rotation_matrix.npz"), quaternions=q.numpy(),
                        rotation=ref.get_rotation_matrix(q).numpy())


def run_parity_full(case, cfg, seed, perturb, per_axis, outdir):
    """What tests/test_parity_full_gpu.py compares with the reference op, for one of its full-size cases, with the same
    inputs and upstream gradients: the pair count; the forward outputs on PARITY_ROWS voxels and the gradient rows of
    PARITY_ROWS Gaussians; per gradient, the reference op's largest distance from the fp64 oracle over
    the whole tensor; the voxels whose reference arg-max differs from the fp64 oracle's, with the reference's class
    there; for the prob variants, the voxels whose reference probability sits on the Z = 1e-9 fallback switch."""
    import helpers as h
    import oracle
    from oracle import ref_op
    from test_parity_full_gpu import GRAD_SEED
    kw, inp, variant = h.splat_case(cfg, seed, perturb, per_axis=per_axis)
    prob = variant != "base"
    N, G = inp["pts"].shape[1], inp["means"].shape[1]
    gen = torch.Generator().manual_seed(GRAD_SEED + seed)
    grads = (torch.randn(N, 18, generator=gen),) + ((torch.randn(N, generator=gen), torch.randn(N, generator=gen)) if prob else ())
    r = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else v) for k, v in ref_op.splat(kw, inp, variant, grads).items()}
    o64 = h.oracle_forward(kw, inp, variant, "f64")
    saved = dict(logits=o64["logits"], bin_logits=o64["bin_logits"], probability=o64["probability"]) if prob else None
    gm, go, gs, gc = h.oracle_backward(kw, inp, variant, tuple(g.numpy() for g in grads), saved, "f64")
    g64 = {"means": gm, "opa": go, "sem": gs, "cov": oracle.cov6_grad_to_3x3(gc)}
    ref_g = {"means": r["means_grad"], "opa": r["opacity_grad"], "sem": r["semantics_grad"],
             "cov": oracle.cov6_grad_to_3x3(r["cov_grad"])}
    # seeded samples, plus the rows where the reference op is farthest from the fp64 oracle (PARITY_WORST of them: for the
    # voxels by their logits, for the Gaussians a quarter by each gradient), which are where two fp32 ops can part most
    def worst(dev, k):
        return np.argsort(dev.reshape(dev.shape[0], -1).max(1))[-k:]
    rng = np.random.default_rng(seed)
    rows = np.unique(np.concatenate([rng.choice(N, PARITY_ROWS - PARITY_WORST, replace=False),
                                     worst(np.abs(r["logits"] - o64["logits"]), PARITY_WORST)]))
    gaussians = np.unique(np.concatenate([rng.choice(G, PARITY_ROWS - PARITY_WORST, replace=False)]
                                         + [worst(np.abs(v - g64[k]), PARITY_WORST // 4) for k, v in ref_g.items()]))
    am_ref = r["logits"].argmax(1)
    flips = np.nonzero(am_ref != o64["logits"].argmax(1))[0]
    arrays = dict(num_pairs=np.int64(r["num_pairs"]), rows=rows, gaussians=gaussians, argmax_flip_rows=flips,
                  argmax_flip_class=am_ref[flips])
    for k in ("logits", "bin_logits", "density") if prob else ("logits",):
        arrays[k + "_rows"] = r[k][rows]
    if prob:
        arrays["unstable_rows"] = np.nonzero(np.abs(r["probability"].astype(np.float64) - 1e-9) <= 1e-10)[0]
    for k, v in ref_g.items():
        arrays[k + "_grad_rows"] = v[gaussians]
        arrays[k + "_grad_floor"] = np.float64(np.abs(v.astype(np.float64) - g64[k]).max())
    np.savez_compressed(os.path.join(outdir, f"ref_parity_full_{case}.npz"), **arrays)
    print("ref_parity_full_" + case, {k: getattr(v, "shape", v) for k, v in arrays.items()})


if __name__ == "__main__":
    from test_parity_full_gpu import CASES
    outdir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden")
    os.makedirs(outdir, exist_ok=True)
    for case in SPLAT_CASES:
        run_splat(*case, outdir)
    run_splat(*MID_CASE, outdir, row_stride=MID_STRIDE)
    run_daf(outdir)
    run_rotation(outdir)
    for case in CASES:
        run_parity_full(*case, outdir)
