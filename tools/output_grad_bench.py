"""Training-step time (forward + backward + Adam over the ResiDual lambdas) for losses on different keys of the HTSAT output dict.

HTSAT-tiny with every layer patched, synthetic weights and clips. In one process, alternating step by step, it times:
  audio_embed  - CE on zero-shot similarities of audio_embed (the c3 step: no tail, no captures)
  clipwise     - BCE on clipwise_output against random AudioSet-style tags (tail backward)
  all_keys     - the sum of BCE on clipwise_output and fixed random linear functionals on framewise_output,
                 fine_grained_embedding, each layers_residuals[l] and each layers_attention[l] (tail + capture gradients)
at B = 256 in bf16 and at B = 64 at fp32 grade. Writes a JSON with the per-step medians and the card's name and power limit.

    python tools/output_grad_bench.py [--steps 5] [--warmup 2] [--out profiles/output_grads_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import gpu_checks as G  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def make_losses(enc, B):
    g = torch.Generator().manual_seed(11)
    dev = "cuda"
    text = G.W.make_text_embeds(50, 512, seed=7).cuda()
    labels = torch.randint(0, 50, (B,), generator=g).cuda()
    tags = (torch.rand(B, 527, generator=g) < 0.1).float().to(dev)
    fw = (torch.randn(B, 1024, 527, generator=g) / 1024).to(dev)
    fine = (torch.randn(B, 1024, enc.num_features, generator=g) / 1024).to(dev)
    res = [(torch.randn(B, enc.depths[l] * (64 >> l) ** 2, enc.embed_dim << l, generator=g) / (64 >> l) ** 2).to(dev) for l in range(4)]
    nw = [max(1, (64 >> l) // 8) ** 2 for l in range(4)]
    att = [(torch.randn(B * nw[l], enc.num_heads[l], 64, 64, generator=g) / nw[l]).to(dev) for l in range(4)]

    def audio_embed(wave):
        emb = enc.encode(waveform=wave, want_audio_embed=True)["audio_embed"]
        return F.cross_entropy(emb @ text.T, labels)

    def clipwise(wave):
        return F.binary_cross_entropy(enc({"waveform": wave})["clipwise_output"], tags)

    def all_keys(wave):
        out = enc({"waveform": wave})
        loss = F.binary_cross_entropy(out["clipwise_output"], tags) + (out["framewise_output"] * fw).sum()
        loss = loss + (out["fine_grained_embedding"] * fine).sum()
        loss = loss + sum((out["layers_residuals"][l] * res[l]).sum() for l in range(4))
        return loss + sum((out["layers_attention"][l] * att[l]).sum() for l in range(4))

    return {"audio_embed": audio_embed, "clipwise": clipwise, "all_keys": all_keys}


def run(precision, B, steps, warmup):
    clap, _, _ = G.make_encoder("tiny", residual=True)
    enc = clap.model.audio_branch
    enc.train_precision = precision
    wave = G.W.make_clips(B, seed=1234).cuda()
    opt = torch.optim.Adam([r.learnable for r in clap._residuals.values()], lr=1e-3)
    losses = make_losses(enc, B)
    times = {k: [] for k in losses}
    for it in range(warmup + steps):
        for name, fn in losses.items():          # alternating: every round times each loss once
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            opt.zero_grad()
            fn(wave).backward()
            opt.step()
            torch.cuda.synchronize()
            if it >= warmup:
                times[name].append(time.perf_counter() - t0)
    return {k: {"median_s": statistics.median(v), "min_s": min(v), "max_s": max(v), "steps": len(v)} for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "output_grads_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("output_grad_bench needs a GPU")
    res = {"card": card(), "model": "HTSAT-tiny, every layer patched", "timing": "host clock around forward + backward + Adam, synchronised",
           "bf16_B256": run("bf16", 256, a.steps, a.warmup), "fp32_B64": run("fp32", 64, a.steps, a.warmup)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
