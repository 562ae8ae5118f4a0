"""Time ard_sym_eigvals (one batched call) beside the per-head torch.linalg.eigvalsh loop it replaces in run_PCA's finalize,
alternating the two in one process, on the finalize's workloads:

  a  28 covariances 4096 x 4096: decaying spectrum, the last 64 eigenvalues exactly zero (the covariance heads of layers 0-2)
  b  32 Gram matrices 1152 x 1152 of centred softmax-row maps (the layer-3 heads: one window per clip)
  c  32 Gram matrices 2000 x 2000 (the same at 2000 clips)
  d  one covariance 4096 x 4096 (HeadPCA.finalize on a single head: no batch to amortise the column steps over)

and a crossover sweep: D in {64, 256, 1152, 2000, 4096} x batch in {1, 2, 4, 8, 16} (Gram matrices of centred softmax-row maps), the
data behind analyze_attention._LIB_MIN_BATCH, which sends a group of heads to the library only from the batch where it wins.

Each timing is CUDA events around the solve on the default stream, the median over `--rounds` alternating rounds. The solver
works in place, so each of its rounds first copies the inputs (outside the timed window). Also recorded: the largest
|eigenvalue difference| / top eigenvalue between the two routes, the launch count of one call, the card name and power limit.

    python tools/eig_bench.py [--rounds 3] [--only a b c d] [--sweep-rounds 2] [--out profiles/eig_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from audio_residual_b200 import lib as L  # noqa: E402
from audio_residual_b200.linalg import sym_eigvals  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:   # the timing stands without it; say why it is missing
        info["power_limit"] = f"unread ({e})"
    return info


def covariances(n, D, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty(n, D, D, device="cuda", dtype=torch.float64)
    lam = torch.exp(-8.0 * torch.arange(D, device="cuda", dtype=torch.float64) / D)
    lam[D - 64:] = 0.0
    for k in range(n):
        Q, _ = torch.linalg.qr(torch.randn(D, D, generator=g, device="cuda", dtype=torch.float64))
        C = Q @ (lam[:, None] * Q.t())
        out[k] = 0.5 * (C + C.t())
    return out


def grams(n, rows, seed, D=4096):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty(n, rows, rows, device="cuda", dtype=torch.float64)
    for k in range(n):
        X = torch.softmax(3.0 * torch.randn(rows, D // 64, 64, generator=g, device="cuda"), dim=-1).reshape(rows, D).double()
        Xc = X - X.mean(0, keepdim=True)
        out[k] = Xc @ Xc.t() / (rows - 1)
    return out


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, r


def run(name, what, mats, rounds):
    batch, D = mats.shape[0], mats.shape[1]
    ours, loop, err = [], [], 0.0
    work = mats.clone()
    sym_eigvals(work, overwrite=True)                      # warm-up both routes at this shape
    torch.linalg.eigvalsh(mats[0])
    lib = L.load()
    c0 = lib.ard_launch_counter_read()
    work.copy_(mats)
    sym_eigvals(work, overwrite=True)
    launches = lib.ard_launch_counter_read() - c0
    for _ in range(rounds):
        work.copy_(mats)
        torch.cuda.synchronize()
        t, w = timed(lambda: sym_eigvals(work, overwrite=True))
        ours.append(t)
        t, ref = timed(lambda: torch.stack([torch.linalg.eigvalsh(m) for m in mats]))
        loop.append(t)
        err = max(err, float(((w - ref).abs().amax(1) / ref.abs().amax(1).clamp_min(1e-300)).max()))
    rec = {"workload": what, "batch": batch, "D": D, "ard_sym_eigvals_s": statistics.median(ours),
           "eigvalsh_loop_s": statistics.median(loop), "ard_sym_eigvals_all_s": ours, "eigvalsh_loop_all_s": loop,
           "speedup": statistics.median(loop) / statistics.median(ours), "max_abs_diff_over_top": err,
           "launches_per_call": int(launches)}
    print(json.dumps({k: v for k, v in rec.items() if not k.endswith("all_s")}), flush=True)
    return rec


def sweep(rounds, sizes=(64, 256, 1152, 2000, 4096), batches=(1, 2, 4, 8, 16)):
    out = []
    for D in sizes:
        one = grams(1, D, 10 + D)
        for b in batches:
            mats = one.expand(b, D, D).contiguous()
            work = mats.clone()
            sym_eigvals(work, overwrite=True)
            torch.linalg.eigvalsh(mats[0])
            ours, loop = [], []
            for _ in range(rounds):
                work.copy_(mats)
                torch.cuda.synchronize()
                ours.append(timed(lambda: sym_eigvals(work, overwrite=True))[0])
                loop.append(timed(lambda: [torch.linalg.eigvalsh(m) for m in mats])[0])
            rec = {"D": D, "batch": b, "ard_sym_eigvals_s": statistics.median(ours), "eigvalsh_loop_s": statistics.median(loop)}
            rec["library_wins"] = rec["ard_sym_eigvals_s"] < rec["eigvalsh_loop_s"]
            print(json.dumps(rec), flush=True)
            out.append(rec)
            del mats, work
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--only", nargs="+", default=["a", "b", "c", "d"])
    ap.add_argument("--sweep-rounds", type=int, default=2, help="0: skip the crossover sweep")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "eig_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eig_bench needs a GPU")
    L.load()
    res = {"card": card(), "timing": "CUDA events around one solve of the whole workload, median of alternating rounds", "runs": {}}
    work = {
        "a": ("28 PCA-like covariances 4096^2 (decaying spectrum, 64 exact zeros)", lambda: covariances(28, 4096, 1)),
        "b": ("32 Gram matrices 1152^2 (centred softmax-row maps)", lambda: grams(32, 1152, 2)),
        "c": ("32 Gram matrices 2000^2 (centred softmax-row maps)", lambda: grams(32, 2000, 3)),
        "d": ("1 PCA-like covariance 4096^2", lambda: covariances(1, 4096, 4)),
    }
    for k in args.only:
        what, make = work[k]
        mats = make()
        res["runs"][k] = run(k, what, mats, args.rounds)
        del mats
        torch.cuda.empty_cache()
    if args.sweep_rounds > 0:
        res["crossover"] = sweep(args.sweep_rounds)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
