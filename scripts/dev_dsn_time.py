"""Dev: MDViT_DSN MKD training step, stacked (MKDTrainer(fuse_domains=True): one trunk pass over the 4 domain mini-batches with
per-group norm sets) against the per-domain loop (fuse_domains=False: four trunk passes), both as captured CUDA graphs.

    python scripts/dev_dsn_time.py [ROUNDS]

4 domains x 32 images, 256 x 256, drop_rate = drop_path_rate = 0.1, Sup domain adapter, MLPFM auxiliary decoders (bench.py's
MDViT configuration on the domain-specific-norm model).  Both trainers live in one process; the script alternates ROUNDS
(default 5) windows of 10 replays of each and prints the median and spread of the per-window step times, with the GPU name
and its power limit."""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from mdvit_b200 import ops, synth
from mdvit_b200.model import MDViT_DSN
from mdvit_b200.train_step import MKDTrainer

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
B, IMG, STEPS = 32, 256, 10
dev = torch.device("cuda")


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def trainer(fuse):
    torch.manual_seed(0)
    m = MDViT_DSN(img_size=IMG, drop_rate=0.1, drop_path_rate=0.1, adapt_method="Sup", num_domains=4, decoder_name="MLPFM").to(dev).train()
    m.load_state_dict(synth.dsn_perturb(m.state_dict()), strict=True)
    ops.manual_seed(1234, dev)
    return MKDTrainer(m, lr=1e-4, weight_decay=0.05, fuse_domains=fuse)


def window(tr):
    s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(STEPS):
        tr.step_graph(None)
    t.record()
    t.synchronize()
    return s.elapsed_time(t) / STEPS


batches = []
for d in range(4):
    img, lab = synth.synth_batch(1234, d, B, IMG, IMG)
    batches.append((img.to(dev), lab.to(torch.uint8).to(dev), d))
arms = {}
for name, fuse in (("fused", True), ("per-domain", False)):
    tr = trainer(fuse)
    tr.capture(batches, warmup=2)
    for _ in range(3):
        tr.step_graph(None)
    torch.cuda.synchronize()
    arms[name] = (tr, [])
    print(f"{name}: captured, {tr.launches_per_step} library launches per step, peak memory "
          f"{torch.cuda.max_memory_allocated() / 2**30:.1f} GiB so far", flush=True)
for _ in range(ROUNDS):
    for name, (tr, ts) in arms.items():
        ts.append(window(tr))
print(f"{torch.cuda.get_device_name()}, power limit {power_limit()}; MDViT_DSN MKD step, 4 x {B} images {IMG}x{IMG}, CUDA graph, "
      f"{ROUNDS} alternating windows of {STEPS} steps")
for name, (tr, ts) in arms.items():
    print(f"{name:10s} median {statistics.median(ts):7.2f} ms/step (min {min(ts):.2f}, max {max(ts):.2f}); "
          f"{4 * B / statistics.median(ts) * 1e3:.0f} images/s; last losses {tr._static_losses.sum(0).tolist()}")
