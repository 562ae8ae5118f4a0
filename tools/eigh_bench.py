"""Time ard_sym_eigh (linalg.sym_eigh: eigenvalues and eigenvectors) beside the routes it replaces, alternating the arms in one
process:

  batched   a  28 covariances 4096 x 4096 (decaying spectrum, 64 exact zeros: the covariance heads of layers 0-2)
            b  32 Gram matrices 1152 x 1152 of centred softmax-row maps (the layer-3 heads)
            c  32 Gram matrices 2000 x 2000
            d  one covariance 4096 x 4096 (HeadPCA.finalize on a single head)
            against the per-head torch.linalg.eigh loop on the device;
  single    one covariance at each HTSAT-tiny / -base layer width (96, 128, 192, 256, 384, 512, 768, 1024), the solve behind
            compute_pca_components, against the host route it replaces (copy to the host + numpy.linalg.eigh) and against
            torch.linalg.eigh on the device.

Device arms: CUDA events around the call (sym_eigh ends with its one host synchronisation, reading the convergence flags). Host
arm: a host clock around copy + numpy.linalg.eigh. Median over `--rounds` rounds; the library works in place, so each round first
copies its inputs (outside the timed window). Also recorded: max |eigenvalue difference| / top eigenvalue against torch, the
largest residual max_m ||A z_m - w_m z_m|| / max|w| and orthogonality error of the library's vectors, the card name and power limit.

    python tools/eigh_bench.py [--rounds 3] [--only a b c d single] [--out profiles/eigh_bench.json]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from audio_residual_b200 import lib as L  # noqa: E402
from audio_residual_b200.linalg import sym_eigh  # noqa: E402
from eig_bench import card, covariances, grams, timed  # noqa: E402

WIDTHS = (96, 128, 192, 256, 384, 512, 768, 1024)


def quality(mats, w, Q, ref_w):
    res = orth = dw = 0.0
    for b in range(mats.shape[0]):
        M, q, wb = mats[b], Q[b], w[b]
        scale = wb.abs().max().clamp_min(1e-300)
        res = max(res, float(torch.linalg.vector_norm(M @ q - q * wb[None, :], dim=0).max() / scale))
        orth = max(orth, float((q.mT @ q - torch.eye(M.shape[0], device=M.device, dtype=M.dtype)).abs().max()))
        dw = max(dw, float((wb - ref_w[b]).abs().max() / ref_w[b].abs().max().clamp_min(1e-300)))
    return {"max_residual_over_top": res, "max_orthogonality_error": orth, "max_abs_eigval_diff_over_top": dw}


def batched(what, mats, rounds):
    batch, D = mats.shape[0], mats.shape[1]
    work = mats.clone()
    sym_eigh(work, overwrite=True)                        # warm-up both arms at this shape
    torch.linalg.eigh(mats[0])
    lib = L.load()
    c0 = lib.ard_launch_counter_read()
    work.copy_(mats)
    sym_eigh(work, overwrite=True)
    launches = lib.ard_launch_counter_read() - c0
    ours, loop = [], []
    for _ in range(rounds):
        work.copy_(mats)
        torch.cuda.synchronize()
        t, (w, Q) = timed(lambda: sym_eigh(work, overwrite=True))
        ours.append(t)
        t, ref = timed(lambda: [torch.linalg.eigh(m) for m in mats])
        loop.append(t)
    rec = {"workload": what, "batch": batch, "D": D, "ard_sym_eigh_s": statistics.median(ours),
           "eigh_loop_s": statistics.median(loop), "ard_sym_eigh_all_s": ours, "eigh_loop_all_s": loop,
           "speedup": statistics.median(loop) / statistics.median(ours), "launches_per_call": int(launches)}
    rec.update(quality(mats, w, Q, torch.stack([r[0] for r in ref])))
    print(json.dumps({k: v for k, v in rec.items() if not k.endswith("all_s")}), flush=True)
    return rec


def single(rounds):
    out = []
    for D in WIDTHS:
        mats = covariances(1, D, 100 + D)
        work = mats.clone()
        sym_eigh(work, overwrite=True)
        torch.linalg.eigh(mats[0])
        np.linalg.eigh(mats[0].cpu().numpy())
        ours, dev, host = [], [], []
        for _ in range(rounds):
            work.copy_(mats)
            torch.cuda.synchronize()
            t, (w, Q) = timed(lambda: sym_eigh(work, overwrite=True))
            ours.append(t)
            dev.append(timed(lambda: torch.linalg.eigh(mats[0]))[0])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            np.linalg.eigh(mats[0].cpu().numpy())
            host.append(time.perf_counter() - t0)
        rec = {"D": D, "ard_sym_eigh_s": statistics.median(ours), "torch_eigh_device_s": statistics.median(dev),
               "host_numpy_eigh_s": statistics.median(host)}
        rec["library_fastest"] = rec["ard_sym_eigh_s"] < min(rec["torch_eigh_device_s"], rec["host_numpy_eigh_s"])
        rec.update(quality(mats, w, Q, torch.linalg.eigvalsh(mats)))
        print(json.dumps(rec), flush=True)
        out.append(rec)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", nargs="+", default=["a", "b", "c", "d", "single"])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eigh_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eigh_bench needs a GPU")
    L.load()
    res = {"card": card(), "timing": "CUDA events (device arms) / host clock (host arm) around one solve of the whole workload, "
                                      "median of alternating rounds", "runs": {}}
    work = {
        "a": ("28 PCA-like covariances 4096^2 (decaying spectrum, 64 exact zeros)", lambda: covariances(28, 4096, 1)),
        "b": ("32 Gram matrices 1152^2 (centred softmax-row maps)", lambda: grams(32, 1152, 2)),
        "c": ("32 Gram matrices 2000^2 (centred softmax-row maps)", lambda: grams(32, 2000, 3)),
        "d": ("1 PCA-like covariance 4096^2", lambda: covariances(1, 4096, 4)),
    }
    for k in args.only:
        if k == "single":
            res["single"] = single(args.rounds)
            continue
        what, make = work[k]
        mats = make()
        res["runs"][k] = batched(what, mats, args.rounds)
        del mats
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
