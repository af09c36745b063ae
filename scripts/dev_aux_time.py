"""Dev: cost of the auxiliary decoder (ops.AuxFn) at the bench shapes, and a per-kernel breakdown of one training step.

    python scripts/dev_aux_time.py [OUT_DIR]

1. CUDA events around MLPDecoderFM forward, backward with weight gradients and backward in da_only mode (B = 32 per domain,
   256 x 256 images: x1 / x5 at 64 x 64, 131072 rows), median of 20 after 5 warm-up calls.
2. torch.profiler (CUDA activities) over one CUDA-graph replay of the MDViT MKD train step as bench.py runs it (4 domains x 32
   images); kernel times aggregated by name, written to OUT_DIR/step_kernels.txt (and the head printed).
Runs unchanged against any tree that has mdvit_b200.model.MLPDecoderFM, so two builds can be compared."""
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mdvit_b200 import ops, synth
from mdvit_b200.model import MDViT, MLPDecoderFM
from mdvit_b200.train_step import MKDTrainer

out_dir = sys.argv[1] if len(sys.argv) > 1 else "."
os.makedirs(out_dir, exist_ok=True)
dev = torch.device("cuda")
B, IMG = 32, 256


def timed(fn, n=20, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        t.record()
        t.synchronize()
        ts.append(s.elapsed_time(t) * 1e3)
    return statistics.median(ts), min(ts), max(ts)


torch.manual_seed(0)
dec = MLPDecoderFM([64, 128, 320, 512], 1, 512).to(dev).train()
sizes = [(64, 64), (32, 32), (16, 16), (8, 8)]
feats = [torch.randn(B, h * w, c, device=dev, requires_grad=True) for (h, w), c in zip(sizes, [64, 128, 320, 512])]
feats.append(torch.randn(B, 64 * 64, 64, device=dev, requires_grad=True))
cot = torch.randn(B, 1, IMG, IMG, device=dev)
holder = {}


def fwd():
    holder["out"] = dec(feats, sizes, (IMG, IMG))


def bwd(mode):
    def run():
        out = dec(feats, sizes, (IMG, IMG))
        torch.cuda.synchronize()
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        with ops.backward_mode(mode):
            out.backward(cot)
        t.record()
        t.synchronize()
        return s.elapsed_time(t) * 1e3
    for _ in range(5):
        run()
    ts = [run() for _ in range(20)]
    return statistics.median(ts), min(ts), max(ts)


lines = []
for name, r in (("aux forward", timed(fwd)), ("aux backward (all)", bwd("all")), ("aux backward (da_only)", bwd("da_only"))):
    lines.append(f"{name:24s} median {r[0]:8.1f} us  (min {r[1]:.1f}, max {r[2]:.1f})")
    print(lines[-1], flush=True)
del holder, feats, dec
torch.cuda.empty_cache()

# one graph replay of the bench's training step under torch.profiler
torch.manual_seed(0)
model = MDViT(img_size=IMG, drop_rate=0.1, drop_path_rate=0.1, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev).train()
ops.manual_seed(1234, dev)
trainer = MKDTrainer(model, lr=1e-4, weight_decay=0.05)
batches = []
for d in range(4):
    img, lab = synth.synth_batch(1234, d, B, IMG, IMG)
    batches.append((img.to(dev), lab.to(torch.uint8).to(dev), d))
trainer.capture(batches, warmup=1)
for _ in range(3):
    trainer.step_graph(None)
torch.cuda.synchronize()
st = timed(lambda: trainer.step_graph(None), n=10, warm=2)
lines.append(f"train step (graph replay) median {st[0] / 1e3:.2f} ms (min {st[1] / 1e3:.2f}, max {st[2] / 1e3:.2f})")
print(lines[-1], flush=True)
from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    trainer.step_graph(None)
    torch.cuda.synchronize()
agg = {}
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
        a = agg.setdefault(e.name, [0, 0.0])
        a[0] += 1
        a[1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
tot = sum(v[1] for v in agg.values())
lines.append(f"one graph replay: {tot / 1e3:.3f} ms of kernel time over {sum(v[0] for v in agg.values())} kernels (profiled, serialised by tracing)")
for n, (c, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    lines.append(f"{us / 1e3:9.3f} ms {100 * us / max(tot, 1e-9):5.1f}%  n={c:4d}  avg {us / c:8.1f} us  {n}")
with open(os.path.join(out_dir, "step_kernels.txt"), "w") as f:
    f.write(torch.cuda.get_device_name() + "\n" + "\n".join(lines) + "\n")
print("\n".join(lines[:45]))
