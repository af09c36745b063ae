"""The MDViT training step (multi_train_MDViT.py:121-213) on the B200 kernels, single- or multi-GPU.

One step = 4 domain forwards (each a single-domain mini-batch) -> fused BCE+Dice / MKD losses -> the MKD backward ->
gradient all-reduce -> fused AdamW.

MKD backward schedules (both produce the reference's gradients; tests compare them):
  "reference"     multi_train_MDViT.py:195-207 verbatim: aux.backward(retain_graph) with `domain_layer` frozen, then
                  (alpha*kt + (1-alpha)*seg).backward() — every weight gradient kernel runs twice.
  "single_sweep"  gradients are linear in the loss cotangent, so  grad(non-DA) = d(aux + a*kt + (1-a)*seg)  and
                  grad(DA) = d(aux + a*kt + (1-a)*seg) - d(aux).  Pass 1 back-propagates -aux in ops.backward_mode("da_only")
                  (activation-gradient chain + DA gradients only, no other wgrad kernel), pass 2 back-propagates the total
                  loss once with all weight gradients.  Same result, ~1 trunk wgrad sweep cheaper (SURVEY.md App. F5).

Data parallelism (replaces nn.DataParallel, multi_train_MDViT.py:73-74): one process per GPU; every rank runs all four
domain forwards on its own slice of each domain batch.  The 8 loss partial sums are all-reduced so BCE/Dice are those
of the gathered global batch (what DataParallel computes on GPU0); gradients are then a plain SUM over ranks, all-reduced
in one flat fp32 buffer that the fused AdamW consumes in place.  BatchNorm statistics stay per-replica, as in DataParallel.
"""
import contextlib

import torch
import torch.distributed as dist

from . import _lib as L
from . import ops
from ._lib import check, ptr


def _align(n, a=4):
    return (n + a - 1) // a * a


class GradBucketer:
    """Overlaps the data-parallel gradient all-reduce with the backward pass (replaces nn.DataParallel's gather/reduce,
    multi_train_MDViT.py:73-74; the stock DDP reducer cannot be used because the MKD step back-propagates one graph twice).

    The flat fp32 gradient buffer is cut into contiguous ranges ("buckets") in parameter-registration order; backward
    finishes the FIRST-registered parameters (stem, first patch embedding, stage 0) last, so the first bucket is kept
    small: it is the only one whose all-reduce cannot hide under remaining backward kernels.  Every parameter receives
    contributions from all domain graphs; autograd runs the graph of the domain that was forwarded FIRST last (tag 0), so
    a parameter is final once the Functions of that domain have reported it as many times as they use it (`uses`: 2 for
    the CPE/CRPE shared by a stage's two blocks, 0 for the other domains' aux decoders).  `uses` is recorded per forward
    PATH (stacked multi-domain forward vs per-domain loop): the two paths tag Functions differently, and mixing one path's
    counts with the other's reports would reduce a bucket before its gradients are complete.  When the last parameter of
    a bucket is final the bucket is all-reduced on a side stream behind an event, so NCCL runs under the remaining
    backward kernels.  The autograd-order assumption is CHECKED: a report from another tag after tag 0 started, or a
    report for a bucket that was already reduced, raises.  Device-agnostic (CPU tensors + gloo in the tests)."""

    def __init__(self, flat_grad, param_ranges, n_buckets=8, group=None, comm_stream=None, first_bucket_frac=1.0 / 64):
        self.flat, self.group, self.comm = flat_grad, group, comm_stream
        total = flat_grad.numel()
        n_buckets = max(1, min(n_buckets, len(param_ranges)))
        target = (total + n_buckets - 1) // n_buckets
        first_target = max(1, int(total * first_bucket_frac)) if n_buckets > 2 else target
        self.bucket_of, self.bounds = {}, []
        lo, cur = 0, 0
        for i, (key, (o, n)) in enumerate(param_ranges.items()):
            self.bucket_of[key] = len(self.bounds)
            cur = o + n
            want = first_target if not self.bounds else target
            if cur - lo >= want or i == len(param_ranges) - 1:
                hi = total if i == len(param_ranges) - 1 else _align(cur)
                self.bounds.append((lo, hi))
                lo = hi
        self.uses_by_path = {}      # path key -> {param key -> reports expected from the last-run (tag 0) graph}
        self.uses = None
        self.reduced = []           # bucket ids in the order they were reduced (inspected by the tests)
        self._started = False

    # -- recording of how often each parameter is used by the first-forwarded domain, once per forward path
    def needs_recording(self, path):
        return path not in self.uses_by_path

    def start_recording(self, path):
        self.uses_by_path[path] = {}
        self._rec = self.uses_by_path[path]

    def record_use(self, keys):
        for k in keys:
            if k in self.bucket_of:
                self._rec[k] = self._rec.get(k, 0) + 1

    def begin(self, path=None):
        if path is None and len(self.uses_by_path) == 1:
            path = next(iter(self.uses_by_path))
        assert path in self.uses_by_path, "record_use() must run during one forward of this path first"
        self.uses = self.uses_by_path[path]
        self._left = {k: self.uses.get(k, 0) for k in self.bucket_of}
        self._bucket_left = [0] * len(self.bounds)
        for k, b in self.bucket_of.items():
            if self._left[k] > 0:
                self._bucket_left[b] += 1
        self._started = False
        self.reduced = []

    def _start(self):
        self._started = True
        for b, left in enumerate(self._bucket_left):      # buckets owned entirely by other domains' graphs: already final
            if left == 0:
                self._reduce(b)

    def report(self, keys, tag=0):
        """Parameters `keys` have received their gradient from one Function of the graph tagged `tag`."""
        if tag != 0:
            if self._started:
                raise RuntimeError("GradBucketer: a Function of domain graph %r ran after the first-forwarded graph started "
                                   "reporting; the autograd execution order this reducer relies on does not hold" % (tag,))
            return
        if not self._started:
            self._start()
        for k in keys:
            b = self.bucket_of.get(k)
            if b is None:
                continue
            if b in self.reduced:
                raise RuntimeError("GradBucketer: gradient written after its bucket was all-reduced (forward path changed "
                                   "without re-recording parameter uses?)")
            left = self._left.get(k, 0)
            if left <= 0:
                continue
            self._left[k] = left - 1
            if left == 1:
                self._bucket_left[b] -= 1
                if self._bucket_left[b] == 0:
                    self._reduce(b)

    def _reduce(self, b):
        if b in self.reduced:
            return
        self.reduced.append(b)
        lo, hi = self.bounds[b]
        view = self.flat[lo:hi]
        if self.comm is not None:
            ev = torch.cuda.Event()
            ev.record()
            with torch.cuda.stream(self.comm):
                self.comm.wait_event(ev)
                dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group)
        else:
            dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group)

    def finish(self):
        """Reduce whatever has not been reported final (defensive) and join the side stream."""
        if not self._started:
            self._start()
        for b in range(len(self.bounds)):
            self._reduce(b)
        if self.comm is not None:
            torch.cuda.current_stream().wait_stream(self.comm)


def _copy_inputs(dst, src):
    """Copy the (image, label) of each mini-batch of `src` into the buffers of `dst`, stream-ordered."""
    for (d_img, d_lab, *_), (s_img, s_lab, *_) in zip(dst, src):
        d_img.copy_(s_img, non_blocking=True)
        d_lab.copy_(s_lab, non_blocking=True)


class _FlatAdamWTrainer:
    """What MKDTrainer and TransFuseTrainer share.  Every parameter is a view into one flat fp32 buffer (`flat`; its gradient
    into `grad`; each parameter 4-element aligned), so one fused AdamW launch (mdv_adamw) updates the model and one flat buffer
    carries the gradient all-reduce.  The whole step can be captured into one CUDA graph over static input buffers
    (capture() / step_graph()).  Subclasses provide forward_losses(batches) and backward(losses)."""

    def __init__(self, model, lr, weight_decay, betas, eps, process_group, num_domains):
        self.model = model
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.num_domains = num_domains
        self.params = list(model.parameters())      # (a parameter shared by several modules is listed once)
        self.device = dev = self.params[0].device
        offs, total = [], 0
        for p in self.params:
            offs.append(total)
            total += _align(p.numel())
        self.total = total
        with torch.no_grad():
            self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
            self.grad = torch.zeros(total, dtype=torch.float32, device=dev)
            for p, o in zip(self.params, offs):
                n = p.numel()
                self.flat[o:o + n].copy_(p.data.reshape(-1))
                p.data = self.flat[o:o + n].view(p.shape)
                p.grad = self.grad[o:o + n].view(p.shape)
        # this trainer owns the gradient buffers and their reduction: weight-gradient kernels add straight into them
        ops.enable_inplace_grad_accumulation(self.params)
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        # AdamW hyper-parameters AND the step count live on the device (fp64[8]: lr, b1, b2, eps, wd, t, -, grad scale):
        # mdv_adamw bumps t itself, so a graph replay needs no per-step host input and the host can run ahead freely
        self.hyper = torch.tensor([lr, betas[0], betas[1], eps, weight_decay, 0.0, 0.0, 1.0], dtype=torch.float64, device=dev)
        self._lr = lr
        self.mirror = None
        self._graph = None
        self._labels = {}
        ops.bump_weight_epoch()

    # ------------------------------------------------------------------ hyper-parameters
    @property
    def lr(self):
        return self._lr

    @lr.setter
    def lr(self, value):
        """StepLR (multi_train_MDViT.py:95,327) changes lr between epochs: a stream-ordered device fill, no host race."""
        self._lr = float(value)
        self.hyper[0:1].fill_(self._lr)

    @property
    def t(self):
        """Optimizer steps taken (reads the device counter: synchronises)."""
        return int(self.hyper[5].item())

    # ------------------------------------------------------------------ pieces
    def _domain_labels(self, B, domains):
        """One-hot domain labels [len(domains) * B, num_domains], B rows per domain.  Built once per (B, domains) and reused,
        so a captured step reads them from a buffer that outlives the capture."""
        key = (B, tuple(int(d) for d in domains))
        dl = self._labels.get(key)
        if dl is None:
            dl = torch.zeros((len(domains) * B, self.num_domains), dtype=torch.float32, device=self.device)
            for g, d in enumerate(key[1]):
                dl[g * B:(g + 1) * B, d] = 1.0
            self._labels[key] = dl
        return dl

    def optimizer_step(self):
        with torch.cuda.device(self.device):
            check(L.lib().mdv_adamw(ptr(self.flat), ptr(self.grad), ptr(self.m), ptr(self.v), ptr(self.hyper), self.total, L.stream()),
                  "mdv_adamw")
            ops.rng_bump(self.device)
            if self.mirror is not None and self.mirror.table is not None:
                self.mirror.refresh()          # GEMM operand copies of the updated weights, one launch

    def _step_body(self, batches):
        ops.reset_stream_ids()
        self.grad.zero_()
        # weight-gradient kernels accumulate into the flat views (ops.enable_inplace_grad_accumulation above)
        losses = self.forward_losses(batches)
        self.backward(losses)
        self.optimizer_step()
        return losses.detach()

    # ------------------------------------------------------------------ eager step
    def step(self, batches):
        ops.bump_weight_epoch()
        return self._step_body(batches)

    # ------------------------------------------------------------------ CUDA-graph step
    def _state_tensors(self):
        return [self.flat, self.m, self.v, self.hyper, ops.rng_tensor(self.device)] + list(self.model.buffers())

    def capture(self, example_batches, warmup=2):
        """Capture the whole step into one CUDA graph over static input buffers (launch-bound otherwise: ~1.5k kernels).
        The GEMM operand copies of the weights (bf16 / TF32 layouts, ~200 per step) become persistent buffers refreshed by
        one launch after AdamW (ops.WeightMirror) instead of one conversion launch each.  The warm-up steps that allocator
        and NCCL need before a capture DO run the optimizer on the example batch; parameters, AdamW moments, the step count,
        the dropout counter and the BatchNorm buffers are restored afterwards, so capture() leaves the training state
        exactly as it found it."""
        self.static = [(img.clone(), lab.clone(), d) for img, lab, d in example_batches]
        saved = [t.clone() for t in self._state_tensors()]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        self.mirror = ops.WeightMirror()
        ops.set_weight_mirror(self.mirror)
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                ops.bump_weight_epoch()
                self._step_body(self.static)
            self.mirror.freeze(self.device)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        ops.bump_weight_epoch()
        n0 = L.lib().mdv_launch_count()
        with torch.cuda.graph(graph):
            self._static_losses = self._step_body(self.static)   # ends with AdamW + mirror.refresh()
        self.launches_per_step = L.lib().mdv_launch_count() - n0   # kernels of this library captured per step
        ops.bump_weight_epoch()      # operand copies made inside the capture live in the graph's private pool: never reuse them eagerly
        with torch.no_grad():
            for t, s in zip(self._state_tensors(), saved):
                t.copy_(s)
            self.mirror.refresh()                     # operand copies of the restored weights
        self._graph = graph
        # double-buffered input staging for prefetch(): H2D on a side stream, one D2D into the static buffers
        self._h2d = torch.cuda.Stream(device=self.device)
        self._stage = [[(torch.empty_like(i), torch.empty_like(l)) for i, l, _ in self.static] for _ in range(2)]
        self._ready = [None, None]
        self._consumed = [None, None]
        self._n_pref = self._n_used = 0
        return self

    def prefetch(self, batches):
        """Start the host->device copy of the NEXT step's inputs (pinned host tensors) on a side stream, into one of two
        staging sets, so it overlaps the step that is running; step_graph() then consumes the oldest prefetched set."""
        if self._graph is None:
            raise RuntimeError("prefetch() needs capture() first")
        if self._n_pref - self._n_used >= 2:
            raise RuntimeError("at most two input sets can be in flight")
        k = self._n_pref % 2
        self._n_pref += 1
        with torch.cuda.stream(self._h2d):
            if self._consumed[k] is not None:
                self._h2d.wait_event(self._consumed[k])
            _copy_inputs(self._stage[k], batches)
            ev = torch.cuda.Event()
            ev.record(self._h2d)
        self._ready[k] = ev

    def step_graph(self, batches=None):
        """Replay the captured step.  `batches` (host or device tensors) are copied straight into the static input buffers on
        the current stream; without them the replay consumes the oldest pending prefetch(), or with none pending runs on
        whatever the static buffers hold.  Passing `batches` while a prefetch() is pending raises: one of the two input sets
        would be dropped."""
        if self._graph is None:
            raise RuntimeError("step_graph() needs capture() first")
        pending = self._n_pref > self._n_used
        if batches is not None:
            if pending:
                raise RuntimeError("step_graph(batches) with a prefetch() pending: call step_graph() to consume it first")
            _copy_inputs(self.static, batches)
        elif pending:
            k = self._n_used % 2
            self._n_used += 1
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(self._ready[k])
            _copy_inputs(self.static, self._stage[k])
            ev = torch.cuda.Event()
            ev.record(cur)
            self._consumed[k] = ev
        self._graph.replay()
        return self._static_losses


class MKDTrainer(_FlatAdamWTrainer):
    def __init__(self, model, lr=1e-4, weight_decay=0.05, betas=(0.9, 0.999), eps=1e-8, alpha=0.5, process_group=None,
                 num_domains=4, with_aux=True, schedule="single_sweep", n_buckets=8, fuse_domains=True, track_metrics=False):
        if schedule not in ("single_sweep", "reference"):
            raise ValueError("schedule must be 'single_sweep' or 'reference'")
        super().__init__(model, lr, weight_decay, betas, eps, process_group, num_domains)
        self.schedule = schedule
        self.fuse_domains = fuse_domains      # stack the domain mini-batches into one trunk pass (MDViT.forward_multi)
        self.alpha = alpha
        self.with_aux = with_aux
        # device-side Dice/Jaccard counts per domain for (main, aux) predictions, accumulated every step inside the step
        # (and its CUDA graph) — the trainer's per-domain output.cpu().numpy() + medpy round trip without the host sync
        self.track_metrics = track_metrics
        self.metric_counts = None
        self.da_params = [p for n, p in model.named_parameters() if "domain_layer" in n]
        self.bucketer = None
        self._path = None
        if self.world > 1:
            ranges = {id(p): (p.data.storage_offset(), p.numel()) for p in self.params}      # (offsets into the flat buffer)
            self.bucketer = GradBucketer(self.grad, ranges, n_buckets=n_buckets, group=process_group,
                                         comm_stream=torch.cuda.Stream(device=self.device))

    # ------------------------------------------------------------------ pieces
    def _reduce_sums(self, sums):
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=self.pg)

    def _model_label(self, B, domains):
        """The domain label the model is called with: the one-hot labels for a model with auxiliary branches, or with domain
        adapters and domain-specific norms; None for any other model, which is trained without it as multi_train_BASE.py does."""
        if self.with_aux or (self.da_params and getattr(self.model, "domain_specific_norms", False)):
            return self._domain_labels(B, domains)
        return None

    @contextlib.contextmanager
    def _tagged_forward(self, path):
        """Scope of one forward along `path` ("fused" or "per_domain"): yields tag(i), which marks the Functions that follow as
        domain graph i.  The first forward of a path records for the bucketer how often graph 0 uses each parameter."""
        self._path = path
        recording = self.bucketer is not None and self.bucketer.needs_recording(path)
        if recording:
            self.bucketer.start_recording(path)

        def tag(i):
            ops.set_forward_tag(i)
            if recording:
                ops.set_forward_use_cb((lambda _, params: self.bucketer.record_use([id(p) for p in params if p is not None]))
                                       if i == 0 else None)
        try:
            yield tag
        finally:
            ops.set_forward_use_cb(None)
            ops.set_forward_tag(None)

    def forward_losses(self, batches):
        """batches: list of (img [B,3,H,W], label [B,1,H,W] fp32 or uint8, domain index).  Returns [n_dom, 3] losses
        (seg, aux, kt).  The partial sums of all domains are all-reduced in ONE collective after the last forward."""
        # all domain mini-batches in one trunk pass (same result as the per-domain loop up to dropout masks); with_aux=False
        # on a model WITH auxiliary branches keeps the per-domain loop: its forward_multi would compute them
        fused = (self.fuse_domains and (self.with_aux or getattr(self.model, "decoder_name", None) is None) and len(batches) > 1
                 and hasattr(self.model, "forward_multi") and len({tuple(b[0].shape) for b in batches}) == 1)
        dsn = getattr(self.model, "domain_specific_norms", False)
        with self._tagged_forward("fused" if fused else "per_domain") as tag:
            if fused:
                x = torch.cat([b[0] for b in batches], dim=0)
                label = self._model_label(batches[0][0].shape[0], [b[2] for b in batches])
                tag(0)
                res = self.model.forward_multi(x, label, [str(b[2]) for b in batches])
                outs, auxs = [o for o, _ in res], [a for _, a in res]
            else:
                outs, auxs = [], []
                for i, (img, _, d) in enumerate(batches):
                    tag(i)
                    # (BASE_DSN: the domain key selects the norm set; the label only feeds domain adapters)
                    o = self.model(img, self._model_label(img.shape[0], [d]), str(d)) if self.with_aux or dsn else self.model(img)
                    if self.with_aux:
                        o, a = o
                    else:
                        o, a = (o[0] if isinstance(o, (list, tuple)) else o), None
                    outs.append(o)
                    auxs.append(a)
        labels = [b[1] for b in batches]
        self.last_logits = [(o.detach(), a.detach() if a is not None else None) for o, a in zip(outs, auxs)]
        if self.track_metrics:
            if self.metric_counts is None:
                self.metric_counts = torch.zeros((len(outs), 2, 3), dtype=torch.int64, device=self.device)
            for g, (o, a) in enumerate(self.last_logits):
                ops.seg_counts(o, labels[g], self.metric_counts[g, 0])
                if a is not None:
                    ops.seg_counts(a, labels[g], self.metric_counts[g, 1])
        return ops.seg_losses_multi(outs, auxs, labels, n_total=outs[0].numel() * self.world,
                                    reduce_sums=self._reduce_sums if self.world > 1 else None)

    def metrics(self, reset=True):
        """[(dc_main, jc_main, dc_aux, jc_aux)] per domain since the last reset (one device->host read of 24 integers)."""
        c = self.metric_counts.clone()
        if self.world > 1:
            dist.all_reduce(c, group=self.pg)
        if reset:
            self.metric_counts.zero_()
        return [ops.dice_jaccard(c[g, 0]) + ops.dice_jaccard(c[g, 1]) for g in range(c.shape[0])]

    def _final_backward(self, loss):
        """The last backward call of the step: gradients become final bucket by bucket and are all-reduced as they do."""
        if self.bucketer is None:
            loss.backward()
            return
        bk = self.bucketer
        bk.begin(self._path)
        ops.set_grad_ready_cb(lambda tag, params: bk.report([id(p) for p in params if p is not None], tag))
        try:
            loss.backward()
        finally:
            ops.set_grad_ready_cb(None)
        bk.finish()

    def backward(self, losses):
        """multi_train_MDViT.py:195-207: aux pass with DA frozen (retain_graph), then alpha*kt + (1-alpha)*seg.  (The gradients
        are all-reduced bucket by bucket during the last backward call, see GradBucketer.)"""
        seg, aux, kt = losses[:, 0].sum(), losses[:, 1].sum(), losses[:, 2].sum()
        if self.with_aux and self.schedule == "reference":
            for p in self.da_params:
                p.requires_grad = False
            aux.backward(retain_graph=True)
            for p in self.da_params:
                p.requires_grad = True
            self._final_backward(self.alpha * kt + (1.0 - self.alpha) * seg)
        elif self.with_aux:
            main = self.alpha * kt + (1.0 - self.alpha) * seg
            if self.da_params:
                with ops.backward_mode("da_only"):
                    (-aux).backward(retain_graph=True)
            self._final_backward(aux + main)
        else:
            self._final_backward(seg)


class TransFuseTrainer(_FlatAdamWTrainer):
    """One training step of multi_train_TransFuse.py:145-197 for TransFuse_S_adapt: per dataset one mini-batch -> three logit maps
    -> loss = 0.5 structure_loss(map_2) + 0.3 structure_loss(map_1) + 0.2 structure_loss(map_x); the dataset losses are summed,
    one backward, one AdamW step.  Data parallel: one all-reduce of the flat gradient buffer (the loss is a per-sample mean, so
    the average over ranks is the global-batch gradient)."""

    def __init__(self, model, lr=1e-4, weight_decay=0.05, betas=(0.9, 0.999), eps=1e-8, process_group=None, num_domains=4,
                 fuse_datasets=True):
        super().__init__(model, lr, weight_decay, betas, eps, process_group, num_domains)
        self.fuse_datasets = fuse_datasets      # stack the dataset mini-batches into one pass (TransFuse_S_adapt.forward_multi)
        self._total_loss = None
        self.last_logits = []      # per dataset: map_2 logits of the last forward (detached)

    def forward_losses(self, batches):
        """batches: [(img [B,3,H,W], mask [B,1,H,W] fp32 or uint8, domain index)] -> per-dataset losses [n]"""
        self.last_logits = []
        self._total_loss = None
        if self.fuse_datasets and len(batches) > 1 and len({tuple(b[0].shape) for b in batches}) == 1:
            return self._forward_losses_fused(batches)
        losses = []
        for img, mask, d in batches:
            mask = mask.float()
            map_x, map_1, map_2 = self.model(img, self._domain_labels(img.shape[0], [d]))
            self.last_logits.append(map_2.detach())      # the prediction the trainer scores (multi_train_TransFuse.py:167,175-181)
            weit = ops.structure_weit(mask)      # shared by the three maps
            losses.append(0.5 * ops.structure_loss(map_2, mask, weit) + 0.3 * ops.structure_loss(map_1, mask, weit)
                          + 0.2 * ops.structure_loss(map_x, mask, weit))
        return torch.stack(losses)

    def _forward_losses_fused(self, batches):
        """All dataset mini-batches in one stacked pass (TransFuse_S_adapt.forward_multi); the summed loss of the G datasets is
        G x the mean of the per-sample terms over the whole stack, so each map needs one loss launch; the per-dataset values (for
        logging) are group means of the detached per-sample terms."""
        G, B = len(batches), batches[0][0].shape[0]
        x = torch.cat([b[0] for b in batches], dim=0)
        mask = torch.cat([b[1] for b in batches], dim=0).float()
        map_x, map_1, map_2 = self.model.forward_multi(x, self._domain_labels(B, [b[2] for b in batches]), G)
        self.last_logits = list(map_2.detach().split(B, dim=0))
        weit = ops.structure_weit(mask)
        total, per = 0.0, 0.0
        for c, mp in ((0.5, map_2), (0.3, map_1), (0.2, map_x)):
            l, ps = ops.structure_loss(mp, mask, weit, per_sample=True)
            total = total + c * l
            per = per + c * ps
        self._total_loss = G * total
        return per.view(G, B).mean(dim=1)

    def backward(self, losses):
        (self._total_loss if self._total_loss is not None else losses.sum()).backward()
        if self.world > 1:
            dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=self.pg)
            self.grad.mul_(1.0 / self.world)
