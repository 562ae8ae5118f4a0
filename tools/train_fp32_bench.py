"""Time the fp32-grade training step (train_precision="fp32") beside the bf16 step on the same handle, alternating.

One step = src/training.py:21-33 on the mirror API: get_audio_embedding_from_data (forward with the tape), zero-shot
similarities + CrossEntropyLoss, loss.backward() into the ResiDual lambdas, Adam. HTSAT-tiny with a ResiDual in every layer,
synthetic weights / clips (weights.py). Per batch and precision: ms per step (median over rounds, each round a host clock
around `--steps` steps ending in a device synchronise) and clips/s; ard_workspace_bytes after the bf16 warm-up and again
after the fp32-grade one (the handle's buffers only grow, so the second is what a handle running both holds; the fp32-grade
mode's split weights and forward workspace are not part of it). The card name and its power limit are read in the same run.

    python tools/train_fp32_bench.py [--batches 64 256] [--steps 5] [--rounds 5] [--out profiles/train_fp32_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from audio_residual_b200 import lib as L  # noqa: E402
from audio_residual_b200 import weights as W  # noqa: E402
from audio_residual_b200.clap import build_clap_module  # noqa: E402
from audio_residual_b200.residual import inject_residuals  # noqa: E402


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:   # the timing stands without it; say why it is missing
        info["power_limit"] = f"unread ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[64, 256])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_fp32_bench needs a GPU")
    sd = W.make_state_dict("tiny", seed=0)
    clap = build_clap_module("tiny", sd, device="cuda:0")
    pca, lam = W.make_pca("tiny", seed=0)
    residuals = inject_residuals(clap.model.audio_branch, pca, lam)
    enc = clap.model.audio_branch
    lams = [r.learnable for r in residuals.values()]
    for p in lams:
        p.requires_grad_(True)
    opt = torch.optim.Adam(lams, lr=1e-4)
    text = W.make_text_embeds(50, 512, seed=7).cuda()
    lib = L.load()
    result = {"model": "tiny", "residual_layers": sorted(residuals), "steps_per_round": args.steps, "rounds": args.rounds,
              "timing": "median over rounds of (host clock around steps ending in torch.cuda.synchronize) / steps", "card": card(),
              "results": []}

    def step(wave, labels):
        opt.zero_grad()
        emb = clap.get_audio_embedding_from_data(wave, use_tensor=True)
        loss = torch.nn.functional.cross_entropy(emb @ text.T, labels)
        loss.backward()
        opt.step()

    for B in args.batches:
        wave = W.make_clips(B, seed=1234).cuda()
        labels = torch.randint(0, 50, (B,), generator=torch.Generator().manual_seed(5)).cuda()
        times = {"bf16": [], "fp32": []}
        ws = {}
        for prec in ("bf16", "fp32"):            # warm-up: workspaces, tapes, split weights, first launches
            enc.train_precision = prec
            for _ in range(2):
                step(wave, labels)
            torch.cuda.synchronize()
            ws[prec] = int(lib.ard_workspace_bytes(enc._hb.h))   # buffers only grow: bf16 alone, then with the fp32-grade step
        for _ in range(args.rounds):
            for prec in ("bf16", "fp32"):        # alternating on the same handle
                enc.train_precision = prec
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    step(wave, labels)
                torch.cuda.synchronize()
                times[prec].append((time.perf_counter() - t0) / args.steps * 1e3)
        row = {"B": B}
        for prec in ("bf16", "fp32"):
            ms = statistics.median(times[prec])
            row[prec] = {"ms_per_step": round(ms, 3), "clips_per_s": round(B / ms * 1e3, 1), "ms_all_rounds": [round(t, 3) for t in times[prec]]}
        row["workspace_bytes_bf16_step"] = ws["bf16"]
        row["workspace_bytes_after_fp32_step"] = ws["fp32"]
        row["fp32_over_bf16"] = round(row["fp32"]["ms_per_step"] / row["bf16"]["ms_per_step"], 2)
        result["results"].append(row)
        print(json.dumps(row), flush=True)
        del wave
        torch.cuda.empty_cache()
    text_out = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text_out + "\n")
    print(text_out)


if __name__ == "__main__":
    main()
