"""Times the occupancy loss op against the reference composition (forward + backward), on one GPU.

    python tools/time_loss.py [--iters 20] [--json out.json]

CUDA events around ``iters`` forward + backward steps of each side, warmed up, the two sides alternated, median of
three regions.  Sizes: config 2's grid (200 x 200 x 16, one sample) with logits (GaussianFormer-1) and with
probabilities (GaussianFormer-2), and config 5's four samples per GPU.  For scale, the splat's forward + backward on
config 2's Gaussians at the same batch.  Prints the card and its power limit with the numbers, and the compulsory bytes
of the op: pred read, gradient written, labels, mask, and the sort's key traffic (3 passes, key + payload read and
written, over the present classes).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gaussianformer_b200.loss import occupancy_loss  # noqa: E402
from gaussianformer_b200.synthetic import make_occ_loss_inputs, reference_occupancy_loss  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        out = f"nvidia-smi unavailable ({e})"
    return out or torch.cuda.get_device_name(0)


def timed(fn, iters):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / iters


def compulsory_bytes(d):
    B, C, N = d["pred"].shape
    T = B * N
    in_set = (d["occ_mask"] & (d["labels"] != 17)).sum().item()
    present = len(set(d["labels"][d["occ_mask"] & (d["labels"] != 17)].unique().tolist()))
    return dict(pred_read=4 * T * C, grad_write=4 * T * C, labels=T, mask=T,
                sort_keys=3 * 2 * 8 * in_set * present, lovasz_set=in_set, present_classes=present)


def loss_sides(d):
    dev = torch.device("cuda")
    pred = d["pred"].to(dev).requires_grad_()
    lab, m, w = d["labels"].to(dev), d["occ_mask"].to(dev), d["class_weights"].to(dev)
    sm = d["use_softmax"]

    def op():
        loss, _ = occupancy_loss(pred, lab, m, w, use_softmax=sm, validate=False)
        loss.backward()

    def ref():
        loss = reference_occupancy_loss(pred, lab, m, w, use_softmax=sm)[0]
        loss.backward()

    return op, ref


def splat_side(B):
    import helpers as h
    kw, inp, var = h.splat_case("gs25600_solid", 0, False)
    m = h.make_module(kw, var, validate=False)
    t = {k: v.cuda().expand(B, *v.shape[1:]).contiguous() for k, v in inp.items()}
    for k in ("means", "opa", "sem", "cov"):
        t[k].requires_grad_(True)
    g = torch.randn(B, t["pts"].shape[1], 18, device="cuda")

    def step():
        out = m(t["pts"][0], t["means"], t["opa"], t["sem"], t["scales"], t["cov"])
        out.backward(g[0] if B == 1 else g)
    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "time_loss.py measures on the GPU; there is no CPU mode"
    info = card()
    print(f"card: {info}")
    results = []
    for case, B in (("cfg2", 1), ("cfg2_prob", 1), ("cfg5", 4)):
        d = make_occ_loss_inputs(case, 0)
        op, ref = loss_sides(d)
        splat = splat_side(B)
        for fn in (op, ref, splat):
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        t = {"op": [], "reference": [], "splat": []}
        for _ in range(3):
            t["op"].append(timed(op, a.iters))
            t["reference"].append(timed(ref, a.iters))
            t["splat"].append(timed(splat, a.iters))
        med = {k: sorted(v)[1] for k, v in t.items()}
        row = dict(case=case, batch=B, card=info, ms=med, ms_all=t, speedup=med["reference"] / med["op"],
                   bytes=compulsory_bytes(d))
        results.append(row)
        print(f"{case:10s} B={B}  op {med['op']:.3f} ms  reference {med['reference']:.3f} ms  "
              f"({row['speedup']:.1f}x)  splat fwd+bwd {med['splat']:.3f} ms  bytes {row['bytes']}")
    if a.json:
        with open(a.json, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
