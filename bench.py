#!/usr/bin/env python
"""MDViT training-throughput benchmark (BASELINE.json metric: MDViT train images/sec at 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch-per-domain B] [--impl reference] [--dump-outputs DIR]

One *step* = the reference's optimizer step (multi_train_MDViT.py:121-213): 4 single-domain mini-batches forward,
BCE+Dice / MKD losses, the two-pass backward, AdamW — on synthetic 256x256 data, random-init weights, dropout 0.1 /
DropPath 0.1 as in the trainer (multi_train_MDViT.py:59).  N>1 is launched by torchrun (one rank per GPU, NCCL).
Prints ONE JSON line on rank 0.  `--impl reference` times the CPU restatement of the reference (oracle/) instead.
`--dump-outputs DIR` writes what the last timed training step returned (losses, logits, updated weights) as DIR/<name>.npy, so
that two builds can be compared output for output on identical seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "mdvit_train_images_per_sec"
UNIT = "images/s"
IMG = 256
F_TRAIN_GFLOP_PER_IMG = 62.3     # SURVEY.md §8(d): 3 x 20.77 GFLOP algorithmic fwd+bwd per image
LINEAR_FUSE_DRAM_BYTES = 557116416 + 236415744   # ncu --set full, profiles/r2_ncu_gemm_linear_fuse_fwd.txt (dram read + write, one launch)
DUMP_SAMPLE = 1 << 20      # --dump-outputs keeps this many elements (a fixed, seeded sample) of a larger output: 4 MB in float32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch-per-domain", type=int, default=32)
    ap.add_argument("--impl", default="mdvit_b200")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of one CUDA graph per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the stock-PyTorch-eager-on-this-GPU baseline leg")
    ap.add_argument("--cpu-batch-per-domain", type=int, default=1)
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="train (default, the headline metric) or infer = BASELINE.json config 5: eval-mode throughput / latency sweep over batch 1..256")
    ap.add_argument("--model", default="MDViT", choices=["MDViT", "BASE", "TransFuse"],
                    help="MDViT (default, the headline metric); BASE = BASELINE.json config 2: no DA, no MKD; TransFuse = config 4: "
                         "TransFuse_S_adapt train step (extras, not the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed training step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.mode == "infer"):
        ap.error("--dump-outputs writes the outputs of the training step of this repository's kernels")
    return args


def dump_outputs(path, trainer, losses):
    """What a caller of the timed training step receives after its last step: the step's losses, the logits of its forward
    (MKDTrainer: main and auxiliary per domain; TransFuseTrainer: map_2 per dataset) and the updated weights (the flat fp32
    parameter buffer), as float32 .npy files.  An output larger than DUMP_SAMPLE elements is written as the same seeded sample
    of its elements on every run."""
    import numpy as np
    import torch
    outs = {"losses": losses}
    logits = trainer.last_logits
    if isinstance(logits[0], tuple):
        outs["logits_out"] = torch.cat([o for o, _ in logits])
        if logits[0][1] is not None:
            outs["logits_aux"] = torch.cat([a for _, a in logits])
    else:
        outs["logits"] = torch.cat(logits)
    outs["params"] = trainer.flat
    os.makedirs(path, exist_ok=True)
    for name, t in outs.items():
        a = t.detach().float().reshape(-1)
        if a.numel() > DUMP_SAMPLE:
            idx = np.random.Generator(np.random.PCG64(0)).integers(0, a.numel(), DUMP_SAMPLE)
            a = a[torch.from_numpy(np.sort(idx)).to(a.device)]
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy().astype(np.float32))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_step_time(batch_per_domain, steps, warmup, threads=None):
    """The reference algorithm on host cores: oracle/mdvit_oracle.py train step (+AdamW) on a bounded sample."""
    import torch
    from mdvit_b200 import synth
    from mdvit_b200.model import MDViT
    from oracle import mdvit_oracle as O
    # torchrun exports OMP_NUM_THREADS=1 to every rank: the CPU arm must use all host cores regardless of the launcher
    torch.set_num_threads(threads or os.cpu_count() or 1)
    torch.manual_seed(0)
    holder = MDViT(img_size=IMG, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")   # parameter container: reference init
    sd = {k: v.detach().clone() for k, v in holder.state_dict().items()}
    for k, v in sd.items():
        if v.is_floating_point() and "running" not in k:
            v.requires_grad_(True)
    for k in list(sd):
        ck = synth.canonical_key(k)
        if ck != k:
            sd[k] = sd[ck]
    names = [k for k, v in sd.items() if v.requires_grad and synth.canonical_key(k) == k]
    m = {k: torch.zeros_like(sd[k]) for k in names}
    v = {k: torch.zeros_like(sd[k]) for k in names}
    times = []
    for it in range(warmup + steps):
        batches = [synth.synth_batch(1234 + it, d, batch_per_domain, IMG, IMG) + (d,) for d in range(4)]
        t0 = time.perf_counter()
        _, grads = O.train_step_grads(sd, batches, drop=0.1, dpr=0.1, drop2d=0.1)
        with torch.no_grad():
            for k in names:
                if grads[k] is not None:
                    O.adamw_step(sd[k], grads[k], m[k], v[k], it + 1)
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return sum(times) / len(times), torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.pop("OMP_NUM_THREADS", None)
    bpd = args.cpu_batch_per_domain
    steps = args.steps          # ~2 s of CPU work per 4-image step
    sec, cores = cpu_oracle_step_time(bpd, steps, min(args.warmup, 1))
    val = 4 * bpd / sec
    sample = f"{4 * bpd} images/step ({bpd}/domain x 4 domains) at {IMG}x{IMG}, fp32, dropout on, {steps} timed steps"
    args.steps = steps
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": min(args.warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"MDViT(Sup, MLPFM) MKD train step, CPU restatement of the reference (oracle port: the reference source is "
                               f"not present on the GPU box), {sample}"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def gpu_eager_baseline(device, B, steps=2, warmup=1):
    """The reference algorithm as stock PyTorch eager on THIS GPU (BASELINE.md section 2's "reference on B200" row): the
    oracle port's MKD train step (4 domain forwards, two backward passes over the retained graphs, torch.optim.AdamW) at
    the bench's batch, timed with CUDA events — in fp32 (torch defaults: cuBLAS fp32, cuDNN TF32 convs) and under bf16
    autocast.  A reported baseline beside the CPU one; nothing of mdvit_b200's kernels runs here."""
    import torch
    from mdvit_b200 import synth
    from mdvit_b200.model import MDViT
    from oracle import mdvit_oracle as O
    out = {"batch_per_domain": B, "what": "oracle port (torch eager restatement of the reference) MKD train step + torch.optim.AdamW, dropout on"}
    for mode in ("fp32", "bf16_autocast"):
        try:
            torch.manual_seed(0)
            holder = MDViT(img_size=IMG, adapt_method="Sup", num_domains=4, decoder_name="MLPFM")
            sd = {k: v.detach().clone().to(device) for k, v in holder.state_dict().items()}
            del holder
            for k, v in sd.items():
                if v.is_floating_point() and "running" not in k:
                    v.requires_grad_(True)
            for k in list(sd):
                ck = synth.canonical_key(k)
                if ck != k:
                    sd[k] = sd[ck]
            names = [k for k, v in sd.items() if v.requires_grad and synth.canonical_key(k) == k]
            opt = torch.optim.AdamW([sd[k] for k in names], lr=1e-4, weight_decay=0.05)
            batches = [tuple(t.to(device) for t in synth.synth_batch(99, d, B, IMG, IMG)) + (d,) for d in range(4)]
            times = []
            for it in range(warmup + steps):
                s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16_autocast")):
                    _, grads = O.train_step_grads(sd, batches, drop=0.1, dpr=0.1, drop2d=0.1)
                for k in names:
                    sd[k].grad = grads[k]
                opt.step()
                opt.zero_grad(set_to_none=True)
                del grads
                t.record()
                t.synchronize()
                if it >= warmup:
                    times.append(s.elapsed_time(t))
            ms = sum(times) / len(times)
            out[mode] = {"images_per_s": 4 * B / (ms * 1e-3), "ms_per_step": ms}
        except torch.cuda.OutOfMemoryError:
            out[mode] = {"error": "out of memory at this batch"}
        except Exception as ex:      # a baseline leg must never take the headline line down
            out[mode] = {"error": str(ex)[:200]}
        finally:
            sd = opt = batches = None
            torch.cuda.empty_cache()
    return out


def _time_launch(fn, device, reps=8, skip=3):
    """Average CUDA-event duration of one launch on the launching stream, L2 flushed (256 MB write) between launches."""
    import torch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    st = torch.cuda.current_stream(device)
    times = []
    for i in range(reps):
        flush.zero_()
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(st)
        fn()
        t.record(st)
        t.synchronize()
        if i >= skip:
            times.append(s.elapsed_time(t))
    return sum(times) / len(times)


def gemm_roofline(peaks, device, M, N, K, out_bf16, what, traffic=None, traffic_source=None):
    """The tcgen05 GEMM (gemm_kernel<NT, 8 epilogue warps>: the kernel with the largest share of the step in
    profiles/r2_launches_step_graph_final.txt) at one of its MLPDecoderFM.linear_fuse shapes, timed alone."""
    import ctypes
    import torch
    from mdvit_b200 import _lib as L
    lib = L.lib()
    A = torch.randn(M, K, device=device).bfloat16()
    W = (torch.randn(N, K, device=device) / K ** 0.5).bfloat16()
    bias = torch.zeros(N, device=device)
    out = torch.empty(M, N, device=device, dtype=torch.bfloat16 if out_bf16 else torch.float32)
    e = L.GemmEpi()
    e.out, e.ldc, e.out_bf16 = L.ptr(out), N, int(out_bf16)
    if not out_bf16:
        e.bias = L.ptr(bias)
    ms = _time_launch(lambda: L.check(lib.mdv_gemm_nt(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e), L.stream()), "mdv_gemm_nt"), device)
    achieved = 2.0 * M * N * K / (ms * 1e-3) / 1e12
    peak = peaks["bf16_tflops"]
    return {"bound": "tensor", "kernel": f"gemm_kernel<NT, 8 epilogue warps, CTA pair> (tcgen05 cta_group::2) @ {what} M={M} N={N} K={K}", "achieved": achieved,
            "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source,
            "algorithmic_flops_per_launch": 2.0 * M * N * K,
            "algorithmic_bytes_per_launch": (M * K + N * K) * 2 + M * N * (2 if out_bf16 else 4),
            "peak_source": peaks["source"] + " (burst)", "ms_per_launch": ms}


def mlp_fused_roofline(peaks, device, backward):
    """The fused fc1-GELU-fc2 kernels (mlp_fused_kernel, csrc/mlp_fused.cu) at the stage-0 shape of the step (M = 128*4096
    tokens, C = 64, hidden = 512): HBM-bound by design (the hidden tile stays on chip; in training hact / u / du still have to
    be written for the weight gradients).  Algorithmic bytes: forward(train) = M*C*(2+4+4) + 2*M*hidden*2; backward =
    M*C*(2+4) + 2*M*hidden*2 (u read, du written)."""
    import torch
    from mdvit_b200 import _lib as L
    lib = L.lib()
    M, C, hidden = 128 * 4096, 64, 512
    a = torch.randn(M, C, device=device).bfloat16()
    w1 = (torch.randn(hidden, C, device=device) / C ** 0.5).bfloat16()
    w2 = (torch.randn(C, hidden, device=device) / hidden ** 0.5).bfloat16()
    b1, b2 = torch.zeros(hidden, device=device), torch.zeros(C, device=device)
    res, out = torch.randn(M, C, device=device), torch.empty(M, C, device=device)
    hact = torch.empty(M, hidden, device=device, dtype=torch.bfloat16)
    u = torch.rand(M, hidden, device=device).bfloat16()
    rng = torch.tensor([1, 2], dtype=torch.int64, device=device)
    cs = torch.zeros(hidden, device=device)
    st = L.stream()
    if backward:
        fn = lambda: L.check(lib.mdv_mlp_bwd(L.ptr(a), L.ptr(w1), L.ptr(u), L.ptr(w2), L.ptr(hact), L.ptr(out), L.ptr(cs), M, C, hidden, st), "mdv_mlp_bwd")  # noqa: E731
        nbytes = M * C * 6 + 2 * M * hidden * 2
        name = "mlp_fused_kernel<backward> du=(dY W2)*u, dX=du W1, du stored + fc1 bias-gradient sums"
        traffic, src = 604202752 + 621095680, "profiles/r2_ncu_mlp_fused_bwd.txt"
    else:
        fn = lambda: L.check(lib.mdv_mlp_fwd(L.ptr(a), L.ptr(w1), L.ptr(b1), L.ptr(w2), L.ptr(b2), L.ptr(res), L.ptr(out), L.ptr(hact), L.ptr(u), M, C,  # noqa: E731
                                             hidden, 0.1, L.ptr(rng), 3, 4, None, 1, st), "mdv_mlp_fwd")
        nbytes = M * C * 10 + 2 * M * hidden * 2
        name = "mlp_fused_kernel<forward, training> fc1-GELU-dropout-fc2-dropout-residual, hact and u stored"
        traffic, src = 201570048 + 1150855000, "profiles/r2_ncu_mlp_fused_fwd_train.txt"
    ms = _time_launch(fn, device)
    achieved = nbytes / (ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": name + f" @ stage 0: M={M} C={C} hidden={hidden}", "achieved": achieved, "peak": peaks["hbm_gbs"],
            "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "traffic_source": "ncu --set full dram bytes, " + src,
            "algorithmic_bytes_per_launch": nbytes, "algorithmic_flops_per_launch": 4.0 * M * C * hidden, "peak_source": peaks["source"],
            "ms_per_launch": ms}


def run_infer(args):
    """BASELINE.json config 5 (multi_train_MDViT.py:351-395 test loop): eval-mode forward, main output only, batch 1..256 on one
    B200, single-domain batches and mixed-domain batches (the DA gate is per sample, so one batch may mix domains: per-domain
    routing needs no regrouping).  One CUDA graph per batch size; BatchNorm (running statistics) is folded into the GEMM
    epilogues, the auxiliary decoder is skipped (only output[0] is used by the reference's test loop), the MLP runs in the
    fused fc1-GELU-fc2 kernel.  `value` = images/s at the best batch size, inputs resident; `e2e` adds the H2D copy of every
    batch from pinned memory and the D2H copy of its logits."""
    import torch
    from mdvit_b200 import _lib as L
    from mdvit_b200.model import MDViT
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = L.lib()
    torch.manual_seed(0)
    model = MDViT(img_size=IMG, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev).eval()
    model.skip_aux_in_eval = True
    sampler = ClockSampler(0)
    sampler.start()
    sweep, launches = [], 0
    steps = args.steps
    for kind in ("single", "mixed"):
        for B in (1, 2, 4, 8, 16, 32, 64, 128, 256):
            g = torch.Generator().manual_seed(B)
            x_host = torch.randn(B, 3, IMG, IMG, generator=g).pin_memory()
            dom = torch.full((B,), 1, dtype=torch.long) if kind == "single" else torch.arange(B) % 4
            dl = torch.nn.functional.one_hot(dom, 4).float().to(dev)
            x = x_host.to(dev)
            out_host = torch.empty(B, 1, IMG, IMG).pin_memory()
            with torch.no_grad():
                side = torch.cuda.Stream(device=dev)
                side.wait_stream(torch.cuda.current_stream(dev))
                with torch.cuda.stream(side):
                    for _ in range(2):
                        model(x, dl, "1")
                torch.cuda.current_stream(dev).wait_stream(side)
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                n0 = lib.mdv_launch_count()
                with torch.cuda.graph(graph):
                    out = model(x, dl, "1")[0]
                per_fwd = lib.mdv_launch_count() - n0
            for _ in range(max(args.warmup, 3)):
                graph.replay()
            torch.cuda.synchronize(dev)
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(steps):
                graph.replay()
            t.record()
            t.synchronize()
            ms = s.elapsed_time(t) / steps
            s.record()
            for _ in range(steps):
                x.copy_(x_host, non_blocking=True)
                graph.replay()
                out_host.copy_(out, non_blocking=True)
            t.record()
            t.synchronize()
            ms_e2e = s.elapsed_time(t) / steps
            launches += per_fwd * steps * 2
            sweep.append({"batch": B, "domains": kind, "latency_ms": ms, "images_per_s": B / (ms * 1e-3), "e2e_latency_ms": ms_e2e,
                          "e2e_images_per_s": B / (ms_e2e * 1e-3), "launches_per_forward": int(per_fwd)})
            del graph, out, x, dl
            torch.cuda.empty_cache()
    clocks = sampler.stop()
    best = max(sweep, key=lambda r: r["images_per_s"])
    best_e2e = max(sweep, key=lambda r: r["e2e_images_per_s"])
    print(json.dumps({
        "metric": "mdvit_infer_images_per_sec", "value": best["images_per_s"], "unit": UNIT, "n_gpus": 1, "steps": steps,
        "warmup": max(args.warmup, 3), "ms_per_step": best["latency_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"MDViT(adapt_method=Sup) eval-mode forward at {IMG}x{IMG}, main output only (aux decoder skipped), BatchNorm folded "
                               "into GEMM epilogues, one CUDA graph per batch size; sweep over batch 1..256, single-domain and mixed-domain batches",
                   "best_batch": best["batch"], "l2": "inputs of batch >= 64 exceed the 126 MB L2; smaller batches are L2-resident between replays (stated)"},
        "e2e": {"value": best_e2e["e2e_images_per_s"], "unit": UNIT, "h2d_bytes_per_step": best_e2e["batch"] * 3 * IMG * IMG * 4,
                "d2h_bytes_per_step": best_e2e["batch"] * IMG * IMG * 4},
        "gpu_launches": int(launches), "sweep": sweep, "clocks": clocks}))


def run_transfuse(args):
    """BASELINE.json config 4: the TransFuse_S_adapt train step of multi_train_TransFuse.py:145-197 (4 datasets x B images, three
    structure losses per dataset, one backward, AdamW).  An extra line, not the headline metric."""
    import torch
    import torch.distributed as dist
    from mdvit_b200 import _lib as L
    from mdvit_b200 import ops, synth
    from mdvit_b200.train_step import TransFuseTrainer
    from mdvit_b200.transfuse import TransFuse_S_adapt
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — mdvit_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.lib()
    B = args.batch_per_domain
    torch.manual_seed(0)
    model = TransFuse_S_adapt(drop_rate=0.2, num_domains=4).to(dev).train()
    ops.manual_seed(1234 + rank, dev)
    trainer = TransFuseTrainer(model, lr=1e-4, weight_decay=0.05)
    host = []
    for d in range(4):
        img, lab = synth.synth_batch(1234 + 17 * rank, d, B, IMG, IMG)
        host.append((img.pin_memory(), lab.to(torch.uint8).pin_memory(), d))
    dev_batches = [(i.to(dev), l.to(dev), d) for i, l, d in host]
    h2d = sum(i.numel() * i.element_size() + l.numel() * l.element_size() for i, l, _ in host)
    use_graph = not args.no_graph
    if use_graph:
        trainer.capture(dev_batches, warmup=1)
        step_resident = lambda: trainer.step_graph(None)      # noqa: E731
        step_e2e = lambda: trainer.step_graph(host)      # noqa: E731  H2D of the step's inputs from pinned memory, then the replay
    else:
        step_resident = lambda: trainer.step(dev_batches)      # noqa: E731
        step_e2e = lambda: trainer.step([(i.to(dev, non_blocking=True), l.to(dev, non_blocking=True), d) for i, l, d in host])      # noqa: E731

    def timed(fn, steps, read_back):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        loss_host = None
        for _ in range(steps):
            losses = fn()
            if read_back:
                loss_host = losses.to("cpu", non_blocking=False)
        t.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([s.elapsed_time(t)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps, loss_host

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.mdv_launch_count()
    ncu_range = bool(int(os.environ.get("MDV_NCU_RANGE", "0")))     # `ncu --profile-from-start off`: capture exactly the timed steps
    if ncu_range:
        torch.cuda.profiler.start()
    ms_res, _ = timed(step_resident, args.steps, False)
    if ncu_range:
        torch.cuda.profiler.stop()
    n1 = lib.mdv_launch_count()
    ms_e2e, loss_host = timed(step_e2e, args.steps, True)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, loss_host)
    launches = trainer.launches_per_step if use_graph else (n1 - n0) // max(args.steps, 1)
    imgs = 4 * B * world
    if rank == 0:
        print(json.dumps({
            "metric": "transfuse_train_images_per_sec", "value": imgs / (ms_res * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_res, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "tf32 forward convs / bf16 transformer and gradient GEMMs, fp32 accumulate", "data": "synthetic",
            "config": {"workload": f"TransFuse_S_adapt train step (BASELINE.json config 4): 4 datasets x {B} images/GPU at {IMG}x{IMG}, Dropout2d 0.2 / 0.1, "
                                   "0.5/0.3/0.2 structure_loss deep supervision, one backward, AdamW",
                       "batch_per_domain_per_gpu": B, "images_per_step": imgs, "parallelism": f"dp{world}", "cuda_graph": use_graph,
                       "l2": "per-step working set (>10 GB) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * 4},
            "gpu_launches": int(launches * args.steps * 2), "launches_per_step": int(launches),
            "model_algorithmic_tflops": imgs / (ms_res * 1e-3) * 71.2 / 1e3,      # SURVEY section 8(d): 3 x 23.72 GFLOP per image
            "clocks": clocks, "final_losses_per_dataset": loss_host.tolist() if loss_host is not None else None,
        }))
    if world > 1:
        torch.cuda.synchronize(dev)
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    if args.mode == "infer":
        return run_infer(args)
    if args.model == "TransFuse":
        return run_transfuse(args)
    import torch
    import torch.distributed as dist
    from mdvit_b200 import _lib as L
    from mdvit_b200 import ops, synth
    from mdvit_b200.model import BASE, MDViT
    from mdvit_b200.train_step import MKDTrainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — mdvit_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.lib()   # fail loudly if the extension is missing
    peaks = load_peaks()
    B = args.batch_per_domain

    torch.manual_seed(0)
    if args.model == "BASE":     # multi_train_BASE.py: BASE(adapt_method=False), seg loss only, one backward
        model = BASE(img_size=IMG, drop_rate=0.1, drop_path_rate=0.1, adapt_method=False).to(dev).train()
    else:
        model = MDViT(img_size=IMG, drop_rate=0.1, drop_path_rate=0.1, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev).train()
    ops.manual_seed(1234 + rank, dev)
    trainer = MKDTrainer(model, lr=1e-4, weight_decay=0.05, with_aux=(args.model != "BASE"))
    # synthetic inputs: per-rank slice of each domain batch, staged in pinned host memory for the e2e arm
    host = []
    for d in range(4):
        img, lab = synth.synth_batch(1234 + 17 * rank, d, B, IMG, IMG)
        host.append((img.pin_memory(), lab.to(torch.uint8).pin_memory(), d))      # binary masks travel as uint8 {0,1}
    dev_batches = [(i.to(dev), l.to(dev), d) for i, l, d in host]
    h2d = sum(i.numel() * i.element_size() + l.numel() * l.element_size() for i, l, _ in host)

    use_graph = not args.no_graph
    if use_graph:
        trainer.capture(dev_batches, warmup=1)
        step_resident = lambda: trainer.step_graph(None)          # noqa: E731  inputs already in the static HBM buffers
        step_e2e = None      # pipelined below: H2D of step i+1 (side stream, staging buffers) overlaps the replay of step i
    else:
        step_resident = lambda: trainer.step(dev_batches)         # noqa: E731
        step_e2e = lambda: trainer.step([(i.to(dev, non_blocking=True), l.to(dev, non_blocking=True), d) for i, l, d in host])  # noqa: E731

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, read_back):
        barrier()
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        loss_host = None
        if fn is None:
            # end to end through MKDTrainer's public API: every step's inputs come from pinned host memory (one H2D per
            # step, all inside the timed region) and its losses are read back to the host
            trainer.prefetch(host)
            for i in range(steps):
                if i + 1 < steps:
                    trainer.prefetch(host)
                losses = trainer.step_graph()
                loss_host = losses.to("cpu", non_blocking=False)
        else:
            for _ in range(steps):
                losses = fn()
                if read_back:
                    loss_host = losses.to("cpu", non_blocking=False)   # device->host read of the step's result, every step
        t.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(t)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps, loss_host

    for _ in range(max(args.warmup, 3)):
        step_resident()
    lib = L.lib()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.mdv_launch_count()
    ncu_range = bool(int(os.environ.get("MDV_NCU_RANGE", "0")))     # `ncu --profile-from-start off`: capture exactly the timed steps
    if ncu_range:
        torch.cuda.profiler.start()
    ms_res, _ = timed(step_resident, args.steps, False)
    if ncu_range:
        torch.cuda.profiler.stop()
    n1 = lib.mdv_launch_count()
    ms_e2e, loss_host = timed(step_e2e, args.steps, True)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, loss_host)
    launches_per_step = trainer.launches_per_step if use_graph else (n1 - n0) // max(args.steps, 1)

    imgs_per_step = 4 * B * world
    value = imgs_per_step / (ms_res * 1e-3)
    e2e = imgs_per_step / (ms_e2e * 1e-3)
    if rank == 0:
        # `roofline`: the time-dominant kernel family of the step (gemm_kernel: 25% of the kernel time over ~350 launches,
        # profiles/r2_launches_step_graph_final.txt) at its heaviest shape, the linear_fuse input-gradient GEMM (8 launches,
        # 2.0 ms per step; CTA-pair instantiation); secondary views: the same kernel at the linear_fuse forward shape (r1's headline view), and the
        # fused MLP kernels that replaced r1's issue-bound GELU / gelu'-epilogue GEMM family (HBM-bound views)
        roof = gemm_roofline(peaks, dev, 32 * 4096, 2112, 512, True, "linear_fuse dgrad", 136420864 + 500927232,
                             "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum, profiles/r2_ncu_gemm_linear_fuse_dgrad.txt")
        extra = {}
        for key, fn in (("roofline_linear_fuse_fwd", lambda: gemm_roofline(peaks, dev, 32 * 4096, 512, 2112, False, "linear_fuse forward", LINEAR_FUSE_DRAM_BYTES,
                                                                             "ncu --set full dram bytes, profiles/r2_ncu_gemm_linear_fuse_fwd.txt")),
                        ("roofline_hbm_kernel", lambda: mlp_fused_roofline(peaks, dev, True)),
                        ("roofline_hbm_kernel_fwd", lambda: mlp_fused_roofline(peaks, dev, False))):
            try:
                extra[key] = fn()
            except Exception as ex:  # never let a secondary view take the headline line down
                extra[key] = {"error": str(ex)[:200]}
        cpu = None
        if world == 1 and not args.no_cpu_baseline and args.model == "MDViT":
            sec, cores = cpu_oracle_step_time(args.cpu_batch_per_domain, 2, 1)
            cpu = {"value": 4 * args.cpu_batch_per_domain / sec, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"oracle (torch fp32 restatement of the reference) train step, {4 * args.cpu_batch_per_domain} images/step "
                             f"at {IMG}x{IMG}, 1 warm-up + 2 timed steps"}
        eager = None
        if world == 1 and not args.no_gpu_eager and args.model == "MDViT":
            del trainer, model
            torch.cuda.empty_cache()
            eager = gpu_eager_baseline(dev, B)
            for k in ("fp32", "bf16_autocast"):
                if "images_per_s" in eager.get(k, {}):
                    eager[k]["speedup_of_this_repo"] = value / eager[k]["images_per_s"]
        model_tflops = value * (34.4 if args.model == "BASE" else F_TRAIN_GFLOP_PER_IMG) / 1e3     # SURVEY §8(d): 3 x fwd GFLOP per image
        if args.model == "BASE":
            workload = (f"BASE(adapt_method=False) train step (BASELINE.json config 2): 4 domains x {B} images/GPU at {IMG}x{IMG}, dropout 0.1, "
                        "DropPath 0.1, BCE+Dice, one backward, AdamW; bf16 tensor-core operands, fp32 accumulate/residual")
        else:
            workload = (f"MDViT(adapt_method=Sup, decoder=MLPFM) MKD train step: 4 domains x {B} images/GPU at {IMG}x{IMG}, "
                        "dropout 0.1, DropPath 0.1, the 4 domain mini-batches stacked through the trunk in one pass (BatchNorm per domain "
                        "group), MKD backward (single-sweep schedule, gradient-equivalent to the reference's two passes), AdamW; "
                        "bf16 tensor-core operands, fp32 accumulate/residual")
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_res, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": workload,
                       "batch_per_domain_per_gpu": B, "images_per_step": imgs_per_step, "parallelism": f"dp{world}",
                       "cuda_graph": use_graph, "l2": "per-step working set (>10 GB) exceeds the 126 MB L2; no explicit flush"},
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * 3 * 4},
            "gpu_launches": int(launches_per_step * args.steps * 2),
            "launches_per_step": int(launches_per_step),
            "model_algorithmic_tflops": model_tflops,
            "roofline": roof, **extra, "cpu_baseline": cpu, "gpu_eager_baseline": eager, "clocks": clocks,
            "final_losses_seg_aux_kt_per_domain": loss_host.tolist() if loss_host is not None else None,
        }))
    if world > 1:
        # the captured step graph holds NCCL work; destroying the process group under it can block: sync, barrier, leave
        torch.cuda.synchronize(dev)
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
