"""Headline benchmark: HTSAT-tiny + ResiDual (all layers) inference, clips/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): HTSAT-tiny CLAP audio encoder with ResiDual injected in every block of all four
layers (reference-faithful doubled FFN, src/residual.py:91-96), batch 256 synthetic 10 s / 48 kHz clips per GPU,
waveform -> log-mel -> Swin encoder -> audio_projection -> L2-normalised 512-d embedding. One "step" = one batch.
N > 1: launched under torchrun, one rank per GPU, clips batch-sharded (weak scaling, no data-path collective).

JSON line keys follow the task contract: value = device-resident throughput, e2e = through the public
CLAP_Module.get_audio_embedding_from_data API with pinned-host inputs and a host read of the result, roofline = the
tcgen05 GEMM family (dominant kernel class) timed with CUDA events inside this process, cpu_baseline = the oracle port
of the reference timed on the host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "htsat_residual_clips_per_sec"
UNIT = "clips/s"
# Algorithmic FLOPs per clip, HTSAT-tiny + ResiDual on all layers, reference-faithful doubled FFN, FFT front end
# (BASELINE.md §3: 21.10 GF excl. STFT; the ResiDual GEMM pair is folded into the out-projection here, so the GEMM
# family executes 21.10 - 1.812 = 19.29 GF/clip of tensor work; the roofline uses the flops the launches really do).
GF_PER_CLIP_TINY_FAITHFUL = 21.10


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        """Only samples taken after this call are reported (call at the start of the timed region)."""
        self.t_mark = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t_mark = getattr(self, "t_mark", 0.0)
        for ts, r in self.rows:
            if ts < t_mark:
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def synth_clips_device(B, seed, device):
    """0.1*randn + three sinusoids (50..14000 Hz), clamped to [-1,1] — generated on the device (SURVEY §8d)."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    x = 0.1 * torch.randn(B, 480000, generator=g, device=device)
    t = torch.arange(480000, device=device, dtype=torch.float32) / 48000.0
    for _ in range(3):
        f = 50 + (14000 - 50) * torch.rand(B, 1, generator=g, device=device)
        a = 0.05 * (0.2 + 0.8 * torch.rand(B, 1, generator=g, device=device))
        x += a * torch.sin(2 * 3.14159265 * f * t[None, :])
    return x.clamp_(-1.0, 1.0)


# ------------------------------------------------------------------------------------------------- reference / CPU arm
def oracle_setup(model="tiny"):
    import torch
    from audio_residual_b200 import weights as W
    from oracle import htsat_oracle as O
    sd = W.make_state_dict(model, seed=0)
    pca, lam = W.make_pca(model, seed=0)
    ores = {l: (torch.tensor(pca[l]["mean"], dtype=torch.float32), torch.tensor(pca[l]["components"], dtype=torch.float32),
                torch.from_numpy(lam[l])) for l in pca}
    return O, sd, ores


def reference_setup():
    """The reference's OWN modules (clap_module.model.CLAP + src.residual.setup_residual_htsat, imported unmodified through
    oracle/refimport.py from /root/reference or its snapshot oracle/_ref) with the bench's weights and PCA files loaded.
    Returns (ns, clap, residuals, audio_cfg) or None when neither tree is present."""
    try:
        import pickle
        import tempfile
        import numpy as np
        import torch
        from audio_residual_b200 import weights as W
        from oracle import refimport
        from oracle.make_golden import load_into_reference
        if not refimport.available():
            return None
        ns = refimport.load()
        torch.manual_seed(0)
        clap, cfg = refimport.build_clap("tiny")
        load_into_reference(clap, W.make_state_dict("tiny", seed=0))
        pca, lam = W.make_pca("tiny", seed=0)
        tmp = tempfile.mkdtemp()
        files = {}
        for l, d in pca.items():
            files[l] = os.path.join(tmp, f"layer_{l}")
            with open(files[l], "wb") as f:
                pickle.dump({"components": d["components"], "mean": d["mean"]}, f)
        new_htsat, residuals = ns.residual.setup_residual_htsat(clap.audio_branch, files, [0, 1, 2, 3])   # src/training.py:100-103
        clap.audio_branch = new_htsat
        for l, r in residuals.items():
            r.learnable.data = torch.from_numpy(np.array(lam[l])).clone()
        return ns, clap, residuals, cfg["audio_cfg"]
    except Exception as e:  # noqa: BLE001
        sys.stderr.write(f"bench: reference modules unavailable ({type(e).__name__}: {e}); timing the oracle port instead\n")
        return None


def make_cpu_step(wl, B):
    """One step of the reference's CPU path on B clips -> (callable, kind, description). `kind` = "reference" when the real
    reference modules run (hook.py:175-190's per-clip featuriser loop + CLAP.get_audio_embedding, model.py:720-742, with
    src/residual.py's patched blocks), "port" when only the oracle restatement is available."""
    import torch
    torch.set_num_threads(os.cpu_count())
    g = torch.Generator().manual_seed(99)
    wave = (0.1 * torch.randn(B, 480000, generator=g)).clamp_(-1, 1)
    labels = torch.randint(0, 50, (B,), generator=g)
    ref = reference_setup()
    if ref is not None:
        ns, clap, residuals, audio_cfg = ref

        def feats():
            return [ns.get_audio_features({}, x, 480000, data_truncating="rand_trunc", data_filling="repeatpad", audio_cfg=audio_cfg,
                                          require_grad=False) for x in wave]
        if wl == "train":
            torch.manual_seed(0)
            cls = torch.nn.Linear(512, 50)
            opt = torch.optim.Adam([r.learnable for r in residuals.values()] + list(cls.parameters()), lr=1e-3)

            def one():
                opt.zero_grad()
                emb = clap.get_audio_embedding(feats())
                torch.nn.functional.cross_entropy(cls(emb.float()), labels).backward()
                opt.step()
        else:
            def one():
                with torch.no_grad():
                    clap.get_audio_embedding(feats())
        return one, "reference", "the reference's own modules (clap_module.model.CLAP.get_audio_embedding + src/residual.py patched blocks)"
    O, sd, ores = oracle_setup()
    if wl == "train":
        ores = {l: (mu, comp, lam.clone().requires_grad_(True)) for l, (mu, comp, lam) in ores.items()}
        torch.manual_seed(0)
        Wc, bc = (0.02 * torch.randn(50, 512)).requires_grad_(True), torch.zeros(50, requires_grad=True)

        def one():
            loss, _ = O.linear_probe_loss(wave, labels, Wc, bc, sd, O.CONFIGS["tiny"], ores)
            loss.backward()
    else:
        def one():
            with torch.no_grad():
                O.get_audio_embedding(wave, sd, O.CONFIGS["tiny"], ores)
    return one, "port", "oracle port of the reference's PyTorch CPU path (oracle/htsat_oracle.py)"


def cpu_time_batches(nbatch, B, warm=1, wl="infer"):
    """Bounded CPU sample of the workload on all host cores. Returns (clips/s, s/batch, kind, description)."""
    one, kind, desc = make_cpu_step(wl, B)
    times = []
    for i in range(warm + nbatch):
        t0 = time.perf_counter()
        one()
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
    sec = sum(times) / len(times)
    return B / sec, sec, kind, desc


def run_reference(args):
    """--impl reference: the reference's own CPU (PyTorch fp32) implementation of the path on all host cores, each step a bounded
    sample of 8 clips of the batch-256 workload. Runs the real reference modules from oracle/_ref (snapshot made by
    oracle/build_ref.py; /root/reference does not exist on the GPU box), else the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    B = 8
    wl = getattr(args, "workload", "infer")
    if wl not in ("infer", "train"):
        print(json.dumps({"impl": "reference", "unavailable": f"no CPU reference arm for --workload {wl} (only infer and train are timed)"}), flush=True)
        return
    one, kind, desc = make_cpu_step(wl, B)
    warm = max(1, min(args.warmup, 2))
    for _ in range(warm):
        one()
    t0 = time.perf_counter()
    steps = args.steps
    for _ in range(steps):
        one()
    dt = time.perf_counter() - t0
    v = B * steps / dt
    sample = (f"{steps} steps x {B} clips (a bounded sample: the workload's batch is 256 clips per step), {desc}, torch {torch.__version__} CPU fp32, "
              f"{torch.get_num_threads()} threads")
    cfg = config_dict(256, wl)
    cfg["reference_sample"] = {"clips_per_step": B, "steps": steps, "note": "throughput of the CPU arm is per clip; 8-clip steps keep the run bounded"}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def config_dict(B, workload="infer"):
    common = {"batch_per_gpu": B, "clip_samples": 480000,
              "l2_policy": "per-step inputs (492 MB waveform at B=256) and activations (>2 GB) exceed the 126 MB L2",
              "weights": "random-init (seeded), random orthonormal PCA basis, lambda = 1 + 0.1 randn"}
    if workload == "train":
        return dict(common, workload="ResiDual training step (BASELINE configs[2]): HTSAT-tiny frozen, ResiDual on all layers, forward + "
                                     "backward to every lambda + 50-class Linear(512,50) probe on audio_embed, CE loss, one flat gradient "
                                     f"allreduce (27,090 floats), Adam step; batch {B} clips per GPU",
                    parallelism="batch-sharded replicas; one NCCL allreduce of the flat lambda+classifier gradient per step")
    if workload == "pca":
        return dict(common, workload="Head-representation PCA statistics (BASELINE configs[3]): HTSAT-tiny forward with capture, per-layer residual "
                                     "moments (D = 96..768) and per-(layer, head) 4096-d attention-map moments (60 heads) accumulated on the "
                                     f"tensor cores; batch {B} clips per GPU per step",
                    parallelism="clip-sharded; moments summed over ranks once at the end (outside the per-step timing)")
    if workload == "base_fusion":
        return dict(common, workload="HTSAT-base + feature fusion (aff_2d) + ResiDual on all layers, embedding throughput (BASELINE configs[4]): "
                                     f"waveform -> device get_mel x4 -> encoder -> 512-d embedding; batch {B} clips per GPU",
                    parallelism="batch-sharded replicas, no collective")
    return dict(common, workload="HTSAT-tiny + ResiDual injected in all attention blocks of layers 0-3 (reference-faithful doubled FFN), "
                                 f"inference, batch {B} clips per GPU, 10 s 48 kHz synthetic waveform -> 512-d L2-normalised embedding (BASELINE configs[1])",
                parallelism="batch-sharded replicas, no collective")


# ------------------------------------------------------------------------------------------------- our arm
class Workload:
    """One of BASELINE configs[1..4] on this rank's GPU: `step()` is the device-resident step, `e2e_step(host)` the same step
    through the public API from a pinned host batch with a host read of the result."""

    def __init__(self, wl, B, dev, rank, world, precision="bf16"):
        import torch
        from audio_residual_b200 import weights as W
        from audio_residual_b200.clap import build_clap_module
        from audio_residual_b200.residual import inject_residuals
        self.wl, self.B, self.dev, self.world = wl, B, dev, world
        model = "base" if wl == "base_fusion" else "tiny"
        clap = build_clap_module(model, W.make_state_dict(model, seed=0), device=dev, enable_fusion=(wl == "base_fusion"))
        pca, lam = W.make_pca(model, seed=0)
        enc = clap.model.audio_branch
        enc.precision = precision
        self.clap, self.enc = clap, enc
        wave = synth_clips_device(B, 1234 + rank, dev)
        self.wave = wave
        self.comm = None
        if wl != "pca":
            residuals = inject_residuals(enc, pca, lam)
        if wl == "infer":
            self.step = lambda: enc.encode(waveform=wave, want_audio_embed=True)["audio_embed"]
            # the reference's inference route (evaluate_zero_shot, src/evaluation.py:93-95): int16-quantised input, use_tensor=False.
            # The host batch is int16 PCM (what quantize_tensor's output is, and what a wav file holds): 0.96 MB per clip over PCIe.
            self.e2e_step = lambda host: clap.get_audio_embedding_from_data(host, use_tensor=False)
            self.e2e_api = ("CLAP_Module.get_audio_embedding_from_data(x_pinned_host_int16_pcm, use_tensor=False) -> numpy "
                            "(the reference's evaluation route: int16 round trip of the waveform, hook.py:177-179)")
            self.e2e_dtype = torch.int16
        elif wl == "base_fusion":
            self.step = lambda: enc.encode(mel_fusion=clap.fusion_mel(wave), want_audio_embed=True)["audio_embed"]
            self.e2e_step = lambda host: clap.get_audio_embedding_from_data(host, use_tensor=False)
            self.e2e_api = "CLAP_Module(enable_fusion=True).get_audio_embedding_from_data(x_pinned_host_int16_pcm, use_tensor=False) -> numpy"
            self.e2e_dtype = torch.int16
        elif wl == "train":
            from audio_residual_b200.head import cross_entropy, head_logits
            from audio_residual_b200.parallel import flat_grad_allreduce
            for r in residuals.values():
                r.to(dev)
            torch.manual_seed(0)
            cls = torch.nn.Linear(512, 50).to(dev)
            params = [r.learnable for r in residuals.values()] + list(cls.parameters())
            opt = torch.optim.Adam(params, lr=1e-3)
            self.trained = {f"lambda{l}": r.learnable for l, r in residuals.items()}
            self.trained.update(classifier_weight=cls.weight, classifier_bias=cls.bias)
            labels = torch.randint(0, 50, (B,), device=dev, generator=torch.Generator(device=dev).manual_seed(5 + rank))
            self.comm = {"collective": "allreduce(sum) of one flat fp32 buffer: lambda grads + classifier grads",
                         "floats": int(sum(p.numel() for p in params)), "comm_nranks": world}

            def train_step(x):
                opt.zero_grad(set_to_none=False)
                emb = clap.get_audio_embedding_from_data(x, use_tensor=True)
                loss = cross_entropy(head_logits(emb, cls.weight, cls.bias), labels)
                loss.backward()
                flat_grad_allreduce([p.grad for p in params])
                opt.step()
                return loss.detach()
            self.step = lambda: train_step(wave)
            self.e2e_step = lambda host: train_step(host.to(dev, non_blocking=True)).cpu()
            self.e2e_api = ("CLAP_Module.get_audio_embedding_from_data(x.to(device), use_tensor=True) -> head_logits(Linear(512,50)) -> "
                            "cross_entropy -> loss.backward() -> allreduce -> Adam.step(); loss.cpu()")
            self.e2e_dtype = torch.float32
        else:   # pca
            from audio_residual_b200.residual import MomentAccumulator
            res_acc = [MomentAccumulator(96 << l, dev) for l in range(4)]
            heads = [4, 8, 16, 32]
            attn_acc = [[MomentAccumulator(4096, dev) for _ in range(heads[l])] for l in range(4)]
            self.res_acc, self.attn_acc = res_acc, attn_acc
            self.comm = {"collective": "allreduce(sum) of {n, sum x, sum x x^T} per layer and per (layer, head), once per pass (finalize)",
                         "floats": int(sum(a.s1.numel() + a.s2.numel() + 1 for a in res_acc) + 60 * (4096 + 4096 * 4096 + 1)),
                         "comm_nranks": world}

            def pca_step(x):
                out = enc.encode(waveform=x, quantize=True, want_dict=True)
                for l in range(4):
                    r = out["layers_residuals"][l]
                    res_acc[l].update(r.view(-1, r.shape[-1]))
                    a = out["layers_attention"][l]
                    a3 = a.view(a.shape[0], a.shape[1], 4096)
                    for hd in range(a.shape[1]):
                        attn_acc[l][hd].update(a3[:, hd])
                return res_acc[3].s1
            self.step = lambda: pca_step(wave)
            self.e2e_step = lambda host: pca_step(host.to(dev, non_blocking=True)).cpu()
            self.e2e_api = "encode(want_dict=True) + MomentAccumulator.update per layer and per (layer, head); mean vector .cpu()"
            self.e2e_dtype = torch.float32

    def outputs(self, out):
        """What a caller of the step holds after it, given `out` = what step() returned: the audio embeddings; for the training step
        the loss and the updated lambdas and classifier; for the PCA statistics every accumulator's moments {n, sum x, sum x x^T},
        the per-(layer, head) attention moments stacked per layer."""
        import torch
        if self.wl == "train":
            return dict(loss=out, **self.trained)
        if self.wl != "pca":
            return {"audio_embed": out}
        res = {}
        f64 = dict(dtype=torch.float64)
        for l in range(4):
            r, heads = self.res_acc[l], self.attn_acc[l]
            res.update({f"layer{l}_residual_n": torch.tensor(float(r.n), **f64), f"layer{l}_residual_s1": r.s1, f"layer{l}_residual_s2": r.s2,
                        f"layer{l}_attention_n": torch.tensor([float(a.n) for a in heads], **f64),
                        f"layer{l}_attention_s1": torch.stack([a.s1 for a in heads]),
                        f"layer{l}_attention_s2": torch.stack([a.s2 for a in heads])})
        return res

    def host_batch(self):
        """Pinned host copy of this rank's clips in the dtype the e2e route takes (int16 PCM = quantize_tensor's integers)."""
        import torch
        if self.e2e_dtype == torch.int16:
            q = (self.wave.clamp(-1.0, 1.0) * 32767.0).to(torch.int16)
            host = torch.empty(q.shape, dtype=torch.int16).pin_memory()
            host.copy_(q)
            return host
        host = torch.empty(self.wave.shape, dtype=torch.float32).pin_memory()
        host.copy_(self.wave)
        return host


class RankGuard:
    """CPU-side (gloo) agreement between ranks for the EXTRA records: a rank whose CUDA context died (a kernel fault is sticky)
    cannot take part in an NCCL barrier any more, and the healthy ranks would wait in it until the NCCL watchdog fires. The extras
    therefore synchronise through a gloo group: every rank reports whether its phase succeeded, all of them learn the minimum, and
    if any failed they all abandon that record together. The headline measurement keeps the NCCL barrier the contract asks for."""

    def __init__(self, dist, world):
        self.dist, self.world = dist, world
        self.group = dist.new_group(backend="gloo") if world > 1 else None

    def all_ok(self, ok):
        import torch
        if self.world == 1:
            return bool(ok)
        t = torch.tensor([1 if ok else 0], dtype=torch.int32)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN, group=self.group)
        return bool(t.item())

    def max(self, value):
        import torch
        if self.world == 1:
            return float(value)
        t = torch.tensor([float(value)], dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return float(t.item())

    def barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.group)


def measure(wl, B, K, Wm, dev, rank, world, dist, do_e2e=True, do_profile=True, sampler=None, precision="bf16", guard=None,
            dump_dir=None):
    """W warm-up + K timed steps of workload `wl` (CUDA events, barrier + synchronize on both sides, max over ranks), then the
    e2e leg and the per-class launch profile. Returns a dict (same on every rank except the rank-0-only profile). With dump_dir,
    rank 0 writes the outputs of the last timed step there (dump_outputs) before anything else runs on the workload."""
    import torch
    from audio_residual_b200 import lib as L
    if guard is not None:
        return _measure_guarded(wl, B, K, Wm, dev, rank, world, precision, guard)
    w = Workload(wl, B, dev, rank, world, precision)
    grad = wl == "train"
    torch.set_grad_enabled(grad)   # inference workloads run as the reference's evaluate() does (src/training.py:47): no autograd tape
    for _ in range(Wm):
        out = w.step()
    torch.cuda.synchronize()
    L.load().ard_launch_counter_reset()
    w.step()
    torch.cuda.synchronize()
    launches_per_step = L.load().ard_launch_counter_read()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    barrier()
    if sampler is not None:
        sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        out = w.step()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if sampler is not None else None
    ms_total = ms.item()
    res = {"workload": wl, "value": world * B * K / (ms_total / 1e3), "ms_per_step": ms_total / K, "steps": K, "warmup": Wm,
           "launches_per_step": int(launches_per_step), "clocks": clocks, "comm": w.comm,
           "checksum": float(out.double().abs().sum().item()), "precision": precision}
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, w.outputs(out))

    if do_e2e:
        host = w.host_batch()
        for _ in range(8):   # warm-up: first call eager, second captures the per-chunk graphs, then the host-pipeline planner may re-plan
            w.e2e_step(host)   # (at most once every three calls, each re-plan followed by an eager + a capture call): let it settle
        barrier()
        t0 = time.perf_counter()
        Ke = max(2, min(K, 10))
        for _ in range(Ke):
            emb_host = w.e2e_step(host)
        torch.cuda.synchronize()
        t_mine = time.perf_counter() - t0
        te = torch.tensor([t_mine], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        # per-rank view of the e2e leg: wall time of the Ke calls and the pipeline fit (copy ms/clip, encode a + b n) each rank measured
        fit = (getattr(w.clap, "_pipe_rates", {}).get(host.dtype) or {}) if hasattr(w, "clap") else {}
        mine = torch.tensor([t_mine, fit.get("c", 0.0), fit.get("a", 0.0), fit.get("b", 0.0),
                             float(len(getattr(w.clap, "_last_bounds", []) or []))], device=dev, dtype=torch.float64)
        allr = [mine.clone() for _ in range(world)]
        if world > 1:
            dist.all_gather(allr, mine)
        # bare pinned-host -> device copy rate of the same buffer on every rank at once: the floor the e2e step cannot beat
        dst = torch.empty(host.shape, device=dev, dtype=host.dtype)
        barrier()
        t1 = time.perf_counter()
        for _ in range(3):
            dst.copy_(host, non_blocking=True)
        torch.cuda.synchronize()
        gbs = torch.tensor([3 * host.numel() * host.element_size() / (time.perf_counter() - t1) / 1e9], device=dev, dtype=torch.float64)
        per_rank = [gbs.clone() for _ in range(world)]
        if world > 1:
            dist.all_gather(per_rank, gbs)
        per_rank = [round(float(t.item()), 2) for t in per_rank]
        del dst
        nb = host.numel() * host.element_size()
        res["e2e"] = {"value": world * B * Ke / te.item(), "unit": UNIT, "h2d_bytes_per_step": int(nb),
                      "d2h_bytes_per_step": int(getattr(emb_host, "nbytes", 0) or emb_host.numel() * 4), "api": w.e2e_api, "steps": Ke,
                      "host_dtype": str(host.dtype).replace("torch.", ""), "h2d_gbs_measured": min(per_rank), "h2d_gbs_per_rank": per_rank,
                      "h2d_bound_clips_per_s": sum(per_rank) * 1e9 / (nb / B),
                      "per_rank": [{"ms_per_call": round(1e3 * float(t[0]) / Ke, 3), "copy_ms_per_clip": round(float(t[1]), 5),
                                    "enc_fixed_ms": round(float(t[2]), 4), "enc_ms_per_clip": round(float(t[3]), 5), "chunks": int(t[4])} for t in allr],
                      "host_cores_per_rank": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None,
                      "host_chunks_rank0": [hi - lo for lo, hi in getattr(w.clap, "_last_bounds", [])],
                      "host_pipe_fit_rank0": {k: round(float(v), 5) for k, v in (getattr(w.clap, "_pipe_rates", {}).get(host.dtype) or {}).items()
                                              if k in ("c", "a", "b", "predicted_ms")},
                      "host_chunks_note": "chunk sizes (clips) of rank 0's last timed call; each rank fits copy(n) = c n and encode(n) = a + b n (ms) "
                                          "to the CUDA-event timings of its previous call (per_rank); ARD_PIPE_ADAPT=2 also re-plans the chunks from the fit"}
        if wl == "infer":   # the same call with the fp32 host waveform (use_tensor=True): 1.92 MB per clip over PCIe
            hf = torch.empty(w.wave.shape, dtype=torch.float32).pin_memory()
            hf.copy_(w.wave)
            f = lambda: w.clap.get_audio_embedding_from_data(hf, use_tensor=True).cpu()   # noqa: E731
            for _ in range(8):
                f()
            barrier()
            t0 = time.perf_counter()
            for _ in range(Ke):
                f()
            torch.cuda.synchronize()
            tf = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tf, op=dist.ReduceOp.MAX)
            res["e2e"]["fp32_host_waveform"] = {"value": world * B * Ke / tf.item(), "h2d_bytes_per_step": B * 480000 * 4,
                                                "api": "get_audio_embedding_from_data(x_pinned_host_fp32, use_tensor=True).cpu()"}
            del hf

    if do_profile:
        # per-class launch timing: every rank runs the two profiled steps (the training step holds a collective); rank 0 records
        if rank == 0:
            L.profile_enable(True)
        for _ in range(2):
            w.step()
        torch.cuda.synchronize()
        if rank == 0:
            res["profile"] = L.profile_read()
            L.profile_enable(False)
        if world > 1:
            dist.barrier()
    torch.set_grad_enabled(True)
    res["_workload_obj"] = w
    return res


def _measure_guarded(wl, B, K, Wm, dev, rank, world, precision, guard):
    """measure() for the extra records (no e2e / profile legs): same W warm-up + K timed steps with CUDA events and the max over
    ranks, but every synchronisation point is a RankGuard agreement, so one rank's failure ends the record on ALL ranks instead of
    leaving the others in a barrier. (The training step's gradient allreduce and the PCA finalize are NCCL collectives of the
    workload itself and stay what they are.)"""
    import torch
    from audio_residual_b200 import lib as L
    state = {}

    def phase(fn, what):
        ok, err = True, None
        try:
            fn()
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            ok, err = False, f"{type(e).__name__}: {e}"
        if not guard.all_ok(ok):
            raise RuntimeError(f"extra '{wl}' abandoned on every rank: {what} failed on " + ("this rank: " + err[:300] if err else "another rank"))

    def setup():
        if os.environ.get("ARD_BENCH_INJECT_FAULT") == f"{rank}:{wl}":          # test hook: one rank fails its warm-up
            raise RuntimeError("injected failure (ARD_BENCH_INJECT_FAULT)")
        state["w"] = Workload(wl, B, dev, rank, world, precision)
        torch.set_grad_enabled(wl == "train")
        for _ in range(Wm):
            state["w"].step()
        torch.cuda.synchronize()
        L.load().ard_launch_counter_reset()
        state["w"].step()
        torch.cuda.synchronize()
        state["launches"] = L.load().ard_launch_counter_read()

    def timed():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            state["out"] = state["w"].step()
        e1.record()
        torch.cuda.synchronize()
        state["ms"] = e0.elapsed_time(e1)
        state["checksum"] = float(state["out"].double().abs().sum().item())

    try:
        phase(setup, "set-up / warm-up")        # doubles as the barrier in front of the timed region
        phase(timed, "the timed steps")
    finally:
        torch.set_grad_enabled(True)
    ms_total = guard.max(state["ms"])
    w = state["w"]
    return {"workload": wl, "value": world * B * K / (ms_total / 1e3), "ms_per_step": ms_total / K, "steps": K, "warmup": Wm,
            "launches_per_step": int(state["launches"]), "clocks": None, "comm": w.comm, "checksum": state["checksum"],
            "precision": precision, "_workload_obj": w}


DUMP_LIMIT_BYTES = 64 * 10**6      # all files of one dump, .npy headers included
NPY_HEADER_BYTES = 1024            # reserved per file; np.save writes 128 bytes for these shapes


def dump_outputs(path, arrays):
    """Writes each tensor of `arrays` as <path>/<name>.npy, float64 where the workload computes in float64 and float32 otherwise, so
    that two builds run with the same arguments (hence the same seeded inputs and weights) can be compared output for output.
    Smallest first, an array is stored whole when it fits its share of the budget still left; a larger one is replaced by a sample
    of its flattened elements at indices drawn from a fixed seed, so the same elements are stored on every run."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    left = DUMP_LIMIT_BYTES
    todo = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(todo):
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 else t.float()
        fit = (left // (len(todo) - i) - NPY_HEADER_BYTES) // t.element_size()
        if t.numel() > fit:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), fit, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(path, f"{name}.npy"), a)
        left -= a.nbytes + NPY_HEADER_BYTES


def pin_rank_to_cores(local_rank, world):
    """One contiguous block of host cores per rank (torchrun does not pin). Measured on an 8-GPU box with 32 vCPUs: un-pinned, three
    of the eight ranks spent 20 ms per e2e call against 12.4-12.8 ms for the others - their Python threads were what their GPUs
    waited for. No-op when the cores cannot be split evenly."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // max(1, world)
        if world > 1 and per >= 2:
            os.sched_setaffinity(0, set(cores[local_rank * per:(local_rank + 1) * per]))
            return per
    except (AttributeError, OSError):
        pass
    return 0


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cores_per_rank = pin_rank_to_cores(local, world)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, Wm = args.batch, args.steps, max(3, args.warmup)
    wl = args.workload
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler is not None:
        sampler.start()          # started before warm-up so nvidia-smi is already streaming when the timed region begins
    guard = RankGuard(dist, world)
    main = measure(wl, B, K, Wm, dev, rank, world, dist, sampler=sampler, dump_dir=args.dump_outputs)
    main.pop("_workload_obj", None)
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs at this N (a few steps each), so the collectives of c3 / c4 and the c5 model are measured
    # wherever the headline is: training step with the flat-gradient allreduce, PCA statistics with the end-of-pass moment
    # allreduce + head-sharded eigensolve, HTSAT-base fusion throughput, and the fp32-grade inference mode.
    extra = {}
    if wl == "infer" and not args.no_extra:
        Ks = max(2, min(K, 5))
        for name, kw in (("train", dict(wl="train", B=B)), ("pca", dict(wl="pca", B=min(B, 128))),
                         ("infer_fp32", dict(wl="infer", B=min(B, 64), precision="fp32")), ("base_fusion", dict(wl="base_fusion", B=B))):
            try:
                r = measure(kw["wl"], kw["B"], Ks, 3, dev, rank, world, dist, do_e2e=False, do_profile=False, precision=kw.get("precision", "bf16"),
                            guard=guard)
                wobj = r.pop("_workload_obj")
                rec = {"metric": METRIC, "value": r["value"], "unit": UNIT, "ms_per_step": r["ms_per_step"], "steps": r["steps"], "n_gpus": world,
                       "batch_per_gpu": kw["B"], "launches_per_step": r["launches_per_step"], "comm": r["comm"], "precision": r["precision"],
                       "workload": config_dict(kw["B"], kw["wl"])["workload"]}
                if name == "pca":   # end of the pass: sum the moments over ranks (NCCL), eigensolve (heads sharded over ranks)
                    from audio_residual_b200.analyze_attention import finalize_head_spectra
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for acc in wobj.res_acc:
                        acc.allreduce()
                    spectra = finalize_head_spectra([a for row in wobj.attn_acc for a in row], n_components=64)
                    torch.cuda.synchronize()
                    rec["finalize_s"] = time.perf_counter() - t0
                    rec["finalize"] = "allreduce of all moments + 60 head spectra (4096-d covariance eigvalsh, heads sharded over ranks)"
                    rec["spectrum_checksum"] = float(sum(float(s[:8].sum()) for s in spectra))
                del wobj
                extra[name] = rec
            except Exception as e:  # noqa: BLE001  (an extra record must never take the headline line down)
                extra[name] = {"error": f"{type(e).__name__}: {e}"[:400]}
            try:
                torch.cuda.empty_cache()
            except Exception:  # noqa: BLE001  (a dead CUDA context: the remaining extras will report it, the headline is already measured)
                pass

    if rank != 0:
        if world > 1:
            guard.barrier()          # gloo: a rank that lost its CUDA context in an extra can still leave in step with the others
            try:
                dist.destroy_process_group()
            except Exception:  # noqa: BLE001
                pass
        return
    if world > 1:
        guard.barrier()
    peaks = read_peaks()
    prof = main.pop("profile")
    tot_ms = sum(v["ms"] for v in prof.values())
    shares = {k: round(v["ms"] / tot_ms, 4) for k, v in prof.items() if v["launches"]}
    gm = prof["gemm_tc"]
    ff = prof.get("ffn_fused", {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
    at = prof.get("window_attention", {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
    achieved = gm["flops"] / (gm["ms"] * 1e-3) / 1e12
    tc_ms, tc_flops = gm["ms"] + ff["ms"] + at["ms"], gm["flops"] + ff["flops"] + at["flops"]
    peak = peaks["bf16_tflops_sustained"]
    ms_step = main["ms_per_step"]
    executed_gf = tc_flops / 2 / B / 1e9
    roofline = {"kernel": "gemm_tc_kernel (tcgen05 GEMM family: qkv / proj+ResiDual / fc1+GELU / fc2 / merge / head)", "bound": "tensor",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                "launches_per_step": gm["launches"] // 2, "ms_per_step": gm["ms"] / 2, "flops_per_step": gm["flops"] / 2,
                "algorithmic_bytes_per_step": gm["bytes"] / 2, "achieved_hbm_gbs": gm["bytes"] / (gm["ms"] * 1e-3) / 1e9,
                "hbm_frac_of_measured": gm["bytes"] / (gm["ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "all_tensor_core_kernels": {"ms_per_step": tc_ms / 2, "tflops": tc_flops / (tc_ms * 1e-3) / 1e12,
                                            "frac": tc_flops / (tc_ms * 1e-3) / 1e12 / peak,
                                            "ffn_fused_ms_per_step": ff["ms"] / 2, "ffn_fused_launches_per_step": ff["launches"] // 2,
                                            "attention_ms_per_step": at["ms"] / 2, "attention_launches_per_step": at["launches"] // 2},
                "share_of_step_by_class": shares}
    if wl == "infer":
        roofline["whole_step_tensor_frac"] = {
            "algorithmic": (B * GF_PER_CLIP_TINY_FAITHFUL * 1e9) / (ms_step * 1e-3) / 1e12 / peak,
            "algorithmic_gf_per_clip": GF_PER_CLIP_TINY_FAITHFUL,
            "executed": (B * executed_gf * 1e9) / (ms_step * 1e-3) / 1e12 / peak, "executed_gf_per_clip": executed_gf,
            "note": "algorithmic = SURVEY 8d figure incl. the 1.81 GF ResiDual GEMM pair; executed = flops the launches really do "
                    "(the pair is folded into the out-projection weights, so it costs no launch)"}
    traffic_file = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(traffic_file):
        tj = json.load(open(traffic_file))
        roofline["traffic"] = tj.get("dram_bytes_per_launch")
        roofline["traffic_of"] = {"instantiation": tj.get("kernel"), "algorithmic_bytes_per_launch": tj.get("algorithmic_bytes_per_launch"),
                                  "note": "ncu --set full capture of ONE instantiation of the family (the one with the largest share of the "
                                          "step); `achieved` / `frac` above are the whole family measured live"}

    cpu = None
    if world == 1 and not args.no_cpu:
        v, sec, kind, desc = cpu_time_batches(nbatch=2, B=8, warm=1, wl="train" if wl == "train" else "infer")
        import torch as _t
        cpu = {"value": v, "unit": UNIT, "cores": _t.get_num_threads(), "kind": kind,
               "sample": f"2 batches x 8 clips of the same workload ({sec:.2f} s/batch), {desc}, fp32"}

    line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config_dict(B, wl),
            "clocks": main["clocks"], "e2e": main["e2e"], "gpu_launches": main["launches_per_step"] * K, "roofline": roofline, "cpu_baseline": cpu,
            "comm": main["comm"], "extra": extra, "embedding_checksum": main["checksum"]}
    print(json.dumps(line), flush=True)
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="infer", choices=["infer", "train", "pca", "base_fusion"],
                    help="infer = the headline (BASELINE configs[1]); the others measure configs[2..4] with the same JSON contract")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra records (train / pca / base_fusion / fp32 at this N)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
