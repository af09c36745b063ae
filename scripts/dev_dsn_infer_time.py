"""Dev: MDViT_DSN inference on mixed-domain batches.  One CUDA graph per (variant, batch size), 256 x 256, eval mode, main
output only:

    mixed      forward_mixed on a mixed batch (sample i from domain i % 4): one pass, per-sample norm sets on the device
    mixed-1d   forward_mixed on a single-domain batch
    grouped    the workaround without forward_mixed: gather each domain's samples, forward(x_d, dl_d, str(d)) per domain,
               scatter the logits back (up to four passes)
    forward    forward(x, dl, d)[0] with skip_aux_in_eval on a single-domain batch (the reference point)

    python scripts/dev_dsn_infer_time.py [ROUNDS]

For every batch size 1, 2, 4 ... 256 all four graphs are captured (after two eager warm-up calls of each), then ROUNDS (default 5)
alternating windows of replays are timed with CUDA events; the script prints the median per-forward latency, images/s and the
library launches per forward, with the GPU name and its power limit.  Inputs of batch >= 64 exceed the 126 MB L2; smaller
batches stay L2-resident between replays.  It then times the stage-0 patch-embedding GEMM (M = B*64*64, N = K = 64, HSWISH) with
one folded BatchNorm set (mdv_gemm_nt_tf32) and with per-sample sets (mdv_gemm_nt_tf32_sets), alternating."""
import ctypes
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from mdvit_b200 import _lib as L
from mdvit_b200 import synth
from mdvit_b200.model import MDViT_DSN

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
IMG = 256
BATCHES = (1, 2, 4, 8, 16, 32, 64, 128, 256)
dev = torch.device("cuda")
lib = L.lib()


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


torch.manual_seed(0)
model = MDViT_DSN(img_size=IMG, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev).eval()
model.load_state_dict(synth.dsn_perturb(model.state_dict()), strict=True)
model.skip_aux_in_eval = True


def variants(B):
    g = torch.Generator().manual_seed(B)
    x = torch.randn(B, 3, IMG, IMG, generator=g).to(dev)
    mixed = torch.arange(B) % 4
    single = torch.full((B,), 1)
    dl_mixed, dl_single = F.one_hot(mixed, 4).float().to(dev), F.one_hot(single, 4).float().to(dev)
    dom_mixed = mixed.to(torch.int32).to(dev)
    dom_single = single.to(torch.int32).to(dev)
    groups = [(d, torch.nonzero(mixed == d).flatten().to(dev)) for d in range(4) if (mixed == d).any()]
    out_grouped = torch.empty(B, 1, IMG, IMG, device=dev)

    def grouped():
        for d, idx in groups:
            out_grouped[idx] = model(x[idx], dl_mixed[idx], str(d))[0]
        return out_grouped

    return {
        "mixed": lambda: model.forward_mixed(x, dl_mixed, dom_mixed),
        "mixed-1d": lambda: model.forward_mixed(x, dl_single, dom_single),
        "grouped": grouped,
        "forward": lambda: model(x, dl_single, "1")[0],
    }


def capture(fn):
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    n0 = lib.mdv_launch_count()
    with torch.cuda.graph(graph):
        out = fn()
    return graph, out, lib.mdv_launch_count() - n0


def window(graph, reps):
    s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        graph.replay()
    t.record()
    t.synchronize()
    return s.elapsed_time(t) / reps


print(f"{torch.cuda.get_device_name()}, power limit {power_limit()}; MDViT_DSN(adapt_method='Sup') eval forward {IMG}x{IMG}, main output, "
      f"one CUDA graph per variant and batch, {ROUNDS} alternating windows", flush=True)
print(f"{'batch':>5s} " + " ".join(f"{v:>26s}" for v in ("mixed", "mixed-1d", "grouped", "forward")))
rows = []
with torch.no_grad():
    for B in BATCHES:
        arms = {}
        for name, fn in variants(B).items():
            graph, out, launches = capture(fn)
            arms[name] = (graph, launches, [], out)
        for graph, *_ in arms.values():
            for _ in range(3):
                graph.replay()
        torch.cuda.synchronize()
        reps = max(5, 160 // B)
        for _ in range(ROUNDS):
            for graph, _, ts, _ in arms.values():
                ts.append(window(graph, reps))
        cells = []
        for name, (graph, launches, ts, _) in arms.items():
            ms = statistics.median(ts)
            rows.append((B, name, ms, B / ms * 1e3, launches, min(ts), max(ts)))
            cells.append(f"{ms:7.3f} ms {B / ms * 1e3:6.0f}/s {launches:4d}L")
        print(f"{B:5d} " + " ".join(f"{c:>26s}" for c in cells), flush=True)
        # the mixed and grouped graphs compute the same logits
        err = ((arms["mixed"][3] - arms["grouped"][3]).abs().max() / arms["grouped"][3].abs().max()).item()
        print(f"      mixed vs grouped max-abs / abs-max {err:.2e}; spread (max-min)/median: " +
              ", ".join(f"{n} {(max(a[2]) - min(a[2])) / statistics.median(a[2]) * 100:.1f}%" for n, a in arms.items()), flush=True)
        del arms
        torch.cuda.empty_cache()

# ---- the stage-0 patch-embedding GEMM alone: one folded set vs per-sample sets
print("\nstage-0 patch-embedding GEMM (M = B*4096, N = K = 64, TF32, folded BatchNorm + HSWISH), alternating windows of 50 launches")
for B in (32, 256):
    M, N, K, S = B * 4096, 64, 64, 4
    A, W = torch.randn(M, K, device=dev), torch.randn(N, K, device=dev) / 8
    sc, sh = 1 + 0.3 * torch.randn(S, N, device=dev), 0.3 * torch.randn(S, N, device=dev)
    ss = (torch.arange(B, device=dev) % S).to(torch.int32)
    out = torch.empty(M, N, device=dev)

    def epi(s, h):
        e = L.GemmEpi()
        e.out, e.ldc, e.colscale, e.bias, e.act = L.ptr(out).value, N, L.ptr(s).value, L.ptr(h).value, L.ACT_HSWISH
        return e

    e1, es = epi(sc[0].contiguous(), sh[0].contiguous()), epi(sc, sh)
    one = lambda: L.check(lib.mdv_gemm_nt_tf32(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(e1), L.stream()), "gemm")  # noqa: E731
    sets = lambda: L.check(lib.mdv_gemm_nt_tf32_sets(L.ptr(A), K, L.ptr(W), K, M, N, K, ctypes.byref(es), L.ptr(ss), 4096, S,  # noqa: E731
                                                     L.stream()), "gemm_sets")
    ts = {"one set": [], "per-sample sets": []}
    for fn in (one, sets):
        for _ in range(10):
            fn()
    torch.cuda.synchronize()
    for _ in range(ROUNDS):
        for name, fn in (("one set", one), ("per-sample sets", sets)):
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(50):
                fn()
            t.record()
            t.synchronize()
            ts[name].append(s.elapsed_time(t) / 50 * 1e3)
    print(f"B={B:3d}: " + "; ".join(f"{n} median {statistics.median(v):.1f} us (min {min(v):.1f}, max {max(v):.1f})" for n, v in ts.items()))
