"""Training / evaluation step glue, the device-side counterpart of ``PredictionEngine.train`` / ``.test``
(/root/reference/engine/prediction.py:198-317, :319-430) for the DSTD-GCN hot path.

One ``TrainStep`` call is one iteration of the reference loop body (:215-294):

    outputs = model(tsc(inputs));            loss  = mpjpe(outputs, targets)             (:231-258)
    outputs = model(tsc(inputs_inv));        loss += mpjpe(outputs, targets[:, ::-1])    (:267-287)   if inverse
    loss /= 2;  zero_grad;  loss.backward();  [clip];  optimizer.step()                  (:287-294)

with the differences that make it a B200 data-parallel step:
  * trainable parameters, their gradients and the Adam moments live in flat fp32 buckets (the module's parameters are
    views into the bucket, so ``state_dict()`` / checkpoints are unchanged);
  * the batch is sharded over ranks; the only collective is one ``all_reduce(sum)`` of the flat gradient bucket
    (NCCL over NVLink), with the 1/world scaling folded into the fused Adam kernel;
  * the loss and its gradient come out of one kernel and the loss stays on the device (no per-step ``.item()`` sync,
    cf. prediction.py:264).
BatchNorm statistics are per rank by default (DDP-without-SyncBN semantics).  With ``TrainStep(sync_bn=True)`` and
more than one rank every training-mode BatchNorm normalises with the statistics of the global batch and updates the
running statistics from them, as ``torch.nn.SyncBatchNorm`` does (``ops.sync_batch_norm``): each BN call then
all-gathers 3*C*V fp64 values per rank in its forward and again in its backward, both passes of the step run on one
stream so every rank issues those collectives in the same order, and the step is not captured into a CUDA graph.  The
running statistics stay bit-identical across ranks.
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.distributed as dist

from . import ops


class FlatParams:
    """Re-homes a module's trainable parameters into one contiguous fp32 bucket (and a matching gradient bucket)."""

    def __init__(self, model: torch.nn.Module):
        self.named = [(k, p) for k, p in model.named_parameters() if p.requires_grad]
        total = sum(p.numel() for _, p in self.named)
        dev, dt = self.named[0][1].device, self.named[0][1].dtype     # fp32 in the product; fp64 only in CPU tests
        self.param = torch.empty(total, dtype=dt, device=dev)
        self.grad = torch.zeros(total, dtype=dt, device=dev)
        self.slices = {}
        off = 0
        for k, p in self.named:
            n = p.numel()
            self.param[off:off + n].copy_(p.detach().reshape(-1))
            p.data = self.param[off:off + n].view(p.shape)
            p.grad = self.grad[off:off + n].view(p.shape)
            self.slices[k] = (off, n, tuple(p.shape))
            off += n
        self.numel = total

    def rebind_grads(self):
        """autograd accumulates in place into the views; re-attach them if something detached a ``.grad``."""
        for k, p in self.named:
            off, n, shape = self.slices[k]
            if p.grad is None or p.grad.data_ptr() != self.grad.data_ptr() + self.grad.element_size() * off:
                p.grad = self.grad[off:off + n].view(shape)


class TrainStep:
    """One optimisation step of the reference engine loop on the sm_100a kernels.

    ``inputs``, ``inputs_inv``, ``targets``: raw ``[N, T, D*V]`` fp32 batches already on the device (this rank's shard),
    D coordinates per joint as the model takes them (``model.coords``: input_channels / 2, 3 for xyz).  Returns the (device, 0-dim) loss of this rank's shard.

    ``sync_bn``: synchronised BatchNorm over the ranks of ``process_group`` (see the module docstring); with one rank
    it changes nothing.
    """

    def __init__(self, model, lr=3e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, inverse=True, clip=-1.0,
                 process_group: Optional[dist.ProcessGroup] = None, sync_bn: bool = False):
        self.model = model
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), betas, float(eps), float(weight_decay)
        self.inverse, self.clip = bool(inverse), float(clip)
        self.flat = FlatParams(model)
        self.exp_avg = torch.zeros_like(self.flat.param)
        self.exp_avg_sq = torch.zeros_like(self.flat.param)
        self.step_count = 0
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        self.sync_bn = bool(sync_bn) and self.world > 1
        dev = self.flat.param.device
        # learning rate and step count also live on the device so that a captured CUDA graph of the step stays valid
        # across steps and StepLR updates (engine/prediction.py:193-196,310)
        self.lr_dev = torch.full((1,), self.lr, dtype=self.flat.param.dtype, device=dev)
        self.step_dev = torch.zeros((1,), dtype=torch.int32, device=dev)
        self._grad_tmp = None
        self._side = None
        self._overlap = os.environ.get('DSTD_OVERLAP_PASSES', '1') != '0'     # two-stream passes (A/B switch)
        self.graph = None
        self._graph_has_update = False
        self._static = None
        self._static_loss = None
        if self.world > 1:
            self.sync_state()

    def sync_state(self, src: int = 0):
        """Make every rank start from rank `src`'s replica: parameters, Adam moments, step count, learning rate and the
        model's buffers (BatchNorm running statistics) are broadcast, as DistributedDataParallel does at construction.
        Without it ranks that were seeded differently, or of which only one loaded a checkpoint, would silently train
        diverging replicas (the only other collective is the gradient all-reduce).  Called from ``__init__`` and
        ``load_checkpoint`` when world > 1."""
        if self.world <= 1:
            return
        gsrc = dist.get_global_rank(self.pg, src) if self.pg is not None else src
        for t in (self.flat.param, self.exp_avg, self.exp_avg_sq, self.step_dev, self.lr_dev):
            dist.broadcast(t, gsrc, group=self.pg)
        for p in self.model.parameters():          # frozen parameters (A_s / A_t) live outside the flat bucket
            if not p.requires_grad:
                dist.broadcast(p.data, gsrc, group=self.pg)
        for b in self.model.buffers():
            dist.broadcast(b, gsrc, group=self.pg)
        self.lr = float(self.lr_dev.item())

    def set_lr(self, lr):
        self.lr = float(lr)
        self.lr_dev.fill_(self.lr)

    def grad_of(self, name):
        off, n, shape = self.flat.slices[name]
        return self.flat.grad[off:off + n].view(shape)

    def _pass_grads(self, loss, dst):
        """Gradients of one pass, gathered straight into the flat bucket `dst`.  ``autograd.grad`` hands back one fresh
        tensor per parameter, so the ~250 per-parameter ``grad += g`` launches of ``backward()`` become one batched
        concatenation."""
        params = [p for _, p in self.flat.named]
        gs = torch.autograd.grad(loss, params, allow_unused=True)
        torch.cat([(g if g is not None else torch.zeros_like(p)).reshape(-1) for g, p in zip(gs, params)], out=dst)

    def loss_and_grads(self, inputs, inputs_inv, targets):
        n, t, vc = inputs.shape
        d = coords(self.model)
        v = vc // d
        scale = 0.5 if self.inverse else 1.0
        self.flat.rebind_grads()
        if self.sync_bn:
            # both passes in order on the current stream: every rank issues the BN exchanges in the same order
            with ops.sync_batch_norm(self.pg):
                return self._loss_and_grads_one_stream(inputs, inputs_inv, targets, n, t, v, d, vc, scale)
        if self.inverse and self._overlap and inputs.is_cuda:
            return self._loss_and_grads_two_streams(inputs, inputs_inv, targets, n, t, v, d, vc, scale)
        return self._loss_and_grads_one_stream(inputs, inputs_inv, targets, n, t, v, d, vc, scale)

    def _loss_and_grads_one_stream(self, inputs, inputs_inv, targets, n, t, v, d, vc, scale):
        out = self.model(inputs.view(n, t, v, d))
        loss = ops.mpjpe(out.reshape(n, t, vc), targets, scale, d)
        # the two passes share nothing but the parameters: back-propagate each as soon as its forward is done (the
        # first pass's saved activations are released before the second forward runs)
        self._pass_grads(loss, self.flat.grad)
        loss = loss.detach()
        if self.inverse:
            out_i = self.model(inputs_inv.view(n, t, v, d))
            loss_i = ops.mpjpe(out_i.reshape(n, t, vc), torch.flip(targets, dims=[1]), scale, d)
            if self._grad_tmp is None:
                self._grad_tmp = torch.empty_like(self.flat.grad)
            self._pass_grads(loss_i, self._grad_tmp)
            self.flat.grad.add_(self._grad_tmp)
            loss = loss + loss_i.detach()
        return loss

    def _loss_and_grads_two_streams(self, inputs, inputs_inv, targets, n, t, v, d, vc, scale):
        """The forward pass and the time-reversed pass on two streams (they share nothing but the parameters).  Every hot
        kernel is a persistent one-CTA-per-SM kernel, so the gain is not co-residency but the filling of each kernel's
        tail and set-up with CTAs of the other pass: +9 % on B200 at the H3.6M bench shape (24.7 vs 27.0 ms/step).
        The reference updates the BatchNorm running statistics of the reversed pass after those of the forward pass
        (engine/prediction.py:232,271): the second pass defers them and they are applied after the join."""
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream()
        if self._grad_tmp is None:
            self._grad_tmp = torch.empty_like(self.flat.grad)
        side = self._side
        side.wait_stream(main)
        out = self.model(inputs.view(n, t, v, d))
        loss = ops.mpjpe(out.reshape(n, t, vc), targets, scale, d)
        self._pass_grads(loss, self.flat.grad)
        with torch.cuda.stream(side), ops.defer_bn_updates() as deferred:
            out_i = self.model(inputs_inv.view(n, t, v, d))
            loss_i = ops.mpjpe(out_i.reshape(n, t, vc), torch.flip(targets, dims=[1]), scale, d)
            self._pass_grads(loss_i, self._grad_tmp)
            loss_i = loss_i.detach()
        main.wait_stream(side)
        ops.apply_deferred_bn_updates(deferred)
        self.flat.grad.add_(self._grad_tmp)
        return loss.detach() + loss_i

    def _finish_step(self):
        """All-reduce of the flat gradient bucket (the only collective unless sync_bn), optional clip, fused Adam."""
        if self.world > 1:
            dist.all_reduce(self.flat.grad, op=dist.ReduceOp.SUM, group=self.pg)
        gscale = 1.0 / self.world
        if self.clip > 0:
            gn = torch.linalg.vector_norm(self.flat.grad) * gscale
            self.flat.grad.mul_(torch.clamp(self.clip / (gn + 1e-6), max=1.0))
        self.step_dev.add_(1)
        torch.ops.dstd_b200.adam_step(self.flat.param, self.flat.grad, self.exp_avg, self.exp_avg_sq, self.lr,
                                      self.betas[0], self.betas[1], self.eps, self.weight_decay, gscale, 0,
                                      self.lr_dev, self.step_dev)

    def _eager(self, inputs, inputs_inv, targets):
        loss = self.loss_and_grads(inputs, inputs_inv, targets)
        self._finish_step()
        return loss

    def __call__(self, inputs, inputs_inv, targets):
        self.step_count += 1
        if self.graph is not None and tuple(inputs.shape) == tuple(self._static[0].shape):
            for dst, src in zip(self._static, (inputs, inputs_inv, targets)):
                if dst.data_ptr() != src.data_ptr():
                    dst.copy_(src, non_blocking=True)
            self.graph.replay()
            if not self._graph_has_update:
                self._finish_step()
            return self._static_loss
        return self._eager(inputs, inputs_inv, targets)

    # ------------------------------------------------------------------ CUDA graph of the whole step
    def _snapshot(self):
        bufs = {k: b.clone() for k, b in self.model.named_buffers()}
        return (self.flat.param.clone(), self.exp_avg.clone(), self.exp_avg_sq.clone(), self.step_dev.clone(), bufs,
                torch.cuda.get_rng_state(self.flat.param.device))

    def _restore(self, snap):
        prm, m, v, st, bufs, rng = snap
        self.flat.param.copy_(prm)
        self.exp_avg.copy_(m)
        self.exp_avg_sq.copy_(v)
        self.step_dev.copy_(st)
        for k, b in self.model.named_buffers():
            b.copy_(bufs[k])
        torch.cuda.set_rng_state(rng, self.flat.param.device)

    def capture(self, inputs, inputs_inv, targets, warmup=2):
        """Capture one whole step (both forwards, backward, all-reduce, Adam: several hundred launches) into a CUDA
        graph bound to static input buffers.  The warm-up steps needed before capture are rolled back, so capturing
        does not change the training state.  Later calls with the same batch shape replay the graph."""
        if self.sync_bn:
            raise RuntimeError("TrainStep.capture: steps with synchronised BatchNorm (sync_bn=True, world > 1) run "
                               "eagerly; their BatchNorm exchanges are collectives inside the passes, which are not "
                               "captured")
        self._static = tuple(t.clone() for t in (inputs, inputs_inv, targets))
        snap = self._snapshot()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._eager(*self._static)
        torch.cuda.current_stream().wait_stream(side)
        self._restore(snap)
        torch.cuda.synchronize()
        # single GPU: the whole step is one graph.  Data parallel: the graph ends after the backward pass and the
        # NCCL all-reduce + Adam (3 launches) are issued eagerly behind it, so no collective is captured.
        self._graph_has_update = self.world == 1
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            if self._graph_has_update:
                self._static_loss = self._eager(*self._static)
            else:
                self._static_loss = self.loss_and_grads(*self._static)
        self._restore(snap)       # capture itself does not execute, but keep the invariant explicit
        self.graph = g
        return self


def coords(model):
    """Coordinates per joint of the model's input (``DSTDGCN.coords``: input_channels / 2); 3 (xyz) for a module that
    does not say."""
    return int(getattr(model, "coords", 3))


@torch.no_grad()
def predict(model, inputs):
    """Eval-mode forward on raw ``[N, T, D*V]`` batches (engine/prediction.py:340-353), D = ``coords(model)``."""
    n, t, vc = inputs.shape
    d = coords(model)
    return model(inputs.view(n, t, vc // d, d)).reshape(n, -1, vc)


_EVAL_STREAMS = {}


@torch.no_grad()
def forward_overlapped(model, x, parts=2):
    """Eval-mode forward of ``x [N, T, V, D]`` as ``parts`` independent sub-batches on separate streams.

    In eval mode (BatchNorm on running statistics, engine/prediction.py:340-353) the samples of a batch do not
    interact, so the sub-batches are independent kernel chains: the persistent one-CTA-per-SM kernels of one chain
    fill their tails and set-up phases with CTAs of the other, exactly as the two passes of the training step do.
    Result identical to ``model(x)`` (same kernels per sample).  Capturable in a CUDA graph (fork / join by events)."""
    assert not model.training, "forward_overlapped is an eval-mode path (BatchNorm batch statistics couple the samples)"
    n = x.shape[0]
    parts = max(1, min(parts, n))
    if parts == 1 or not x.is_cuda:
        return model(x)
    main = torch.cuda.current_stream()
    key = (x.device.index, parts)
    if key not in _EVAL_STREAMS:
        _EVAL_STREAMS[key] = [torch.cuda.Stream(device=x.device) for _ in range(parts - 1)]
    bounds = [n * i // parts for i in range(parts + 1)]
    outs = [None] * parts
    for i, st in enumerate(_EVAL_STREAMS[key]):
        st.wait_stream(main)
        with torch.cuda.stream(st):
            outs[i + 1] = model(x[bounds[i + 1]:bounds[i + 2]])
    outs[0] = model(x[bounds[0]:bounds[1]])
    for st in _EVAL_STREAMS[key]:
        main.wait_stream(st)
    for o in outs[1:]:
        o.record_stream(main)
    return torch.cat(outs, dim=0)


@torch.no_grad()
def evaluate(model, batches, input_n, eval_frame, dim_used=None, joint_to_ignore=None, joint_equal=None):
    """Per-frame MPJPE of ``PredictionEngine.test`` (engine/prediction.py:319-430) on the sm_100a forward.

    ``batches`` yields ``(inputs [N, T, D*V], all_seqs [N, T_all, D*J])`` (the 1st and 4th element of the reference's
    dataset tuple) already on the model's device, D = ``coords(model)`` coordinates per joint.  The prediction is scattered into a copy of the ground truth at
    ``dim_used`` (:374-379), ignored joints take the value of their ``joint_equal`` twin (:385-390), and the metric
    at output frame ``eval_frame[k]`` is the batch-size-weighted mean joint distance (:395-406).
    Returns ``(average over all eval frames and batches, per-frame metric)`` like the reference (``t_l.avg, t_metric``)."""
    eval_frame = [int(j) for j in eval_frame]
    d = coords(model)
    was_training = model.training
    model.eval()
    metric = torch.zeros(len(eval_frame), dtype=torch.float64)
    total = 0
    for inputs, all_seqs in batches:
        outputs = predict(model, inputs.float())
        all_seqs = all_seqs.float()
        n, seq_len, _ = all_seqs.shape
        pred = all_seqs.clone()
        tail = outputs.shape[1] != seq_len              # model predicts only the frames after input_n
        if dim_used is not None:
            idx = torch.as_tensor(dim_used, dtype=torch.long, device=pred.device)
            if tail:
                pred[:, input_n:, idx] = outputs
            else:
                pred[:, :, idx] = outputs
        elif tail:
            pred[:, input_n:] = outputs
        else:
            pred[:, :, :] = outputs
        if joint_to_ignore is not None:
            ign = torch.as_tensor(joint_to_ignore, dtype=torch.long, device=pred.device)
            eq = torch.as_tensor(joint_equal, dtype=torch.long, device=pred.device)
            assert ign.shape == eq.shape
            pred[:, :, torch.cat([ign * d + c for c in range(d)])] = pred[:, :, torch.cat([eq * d + c for c in range(d)])]
        p3 = pred.view(n, seq_len, -1, d)[:, input_n:]
        t3 = all_seqs.view(n, seq_len, -1, d)[:, input_n:]
        fr = torch.as_tensor(eval_frame, dtype=torch.long, device=pred.device)
        dist_ = torch.linalg.vector_norm(t3[:, fr] - p3[:, fr], dim=-1).mean(dim=(0, 2))   # one device->host read per batch
        metric += dist_.double().cpu() * n
        total += n
    if was_training:
        model.train()
    metric /= max(total, 1)
    return float(metric.mean()), metric.numpy()


# ====================================================================================== checkpoints (reference format)
class ModelWrapper(torch.nn.Module):
    """Key-prefix twin of the reference's ``ModelWrapper`` (engine/prediction.py:22-101): checkpoints written by
    ``PredictionEngine.save`` (:170-182) hold ``ModelWrapper.state_dict()``, i.e. every key starts with ``model.``."""

    def __init__(self, model):
        super().__init__()
        self.model = model

    def forward(self, x, inverse=False):
        return self.model(x)


def _adam_state_dict(step: "TrainStep"):
    """The flat Adam buckets in ``torch.optim.Adam.state_dict()`` layout (parameter index = position in
    ``model.parameters()``, as the reference's ``optim.Adam(self.model.parameters())`` numbers them)."""
    params = list(step.model.parameters())
    index = {id(p): i for i, p in enumerate(params)}
    state = {}
    nsteps = int(step.step_dev.item())
    for name, p in step.flat.named:
        off, n, shape = step.flat.slices[name]
        if nsteps > 0:
            state[index[id(p)]] = {"step": torch.tensor(float(nsteps)),
                                   "exp_avg": step.exp_avg[off:off + n].view(shape).clone(),
                                   "exp_avg_sq": step.exp_avg_sq[off:off + n].view(shape).clone()}
    group = {"lr": step.lr, "betas": tuple(step.betas), "eps": step.eps, "weight_decay": step.weight_decay,
             "amsgrad": False, "maximize": False, "foreach": None, "capturable": False, "differentiable": False,
             "fused": None, "decoupled_weight_decay": False, "params": list(range(len(params)))}
    return {"state": state, "param_groups": [group]}


def save_checkpoint(path, step: "TrainStep", err=float("inf"), epoch=0, scheduler_state=None):
    """Write ``last.pth``-compatible state (engine/prediction.py:170-182): same top-level keys, ``model.``-prefixed
    weights, Adam state in torch's own layout, so the reference's ``PredictionEngine.recover`` can read it back."""
    state = {"lr": step.lr, "err": err, "model": ModelWrapper(step.model).state_dict(),
             "optimizer": _adam_state_dict(step), "scheduler": scheduler_state or {}, "epoch": epoch}
    torch.save(state, path)
    return state


def load_checkpoint(path_or_state, model, step: Optional["TrainStep"] = None, model_only=False):
    """Counterpart of ``PredictionEngine.recover`` (engine/prediction.py:159-168).  Accepts checkpoints written by the
    reference (keys prefixed ``model.``) as well as bare model state_dicts; strict key / shape matching."""
    state = path_or_state if isinstance(path_or_state, dict) else torch.load(path_or_state, map_location="cpu",
                                                                             weights_only=False)
    sd = state["model"] if "model" in state and isinstance(state["model"], dict) else state
    if all(k.startswith("model.") for k in sd):
        sd = {k[len("model."):]: v for k, v in sd.items()}
    with torch.no_grad():
        own = model.state_dict()
        missing = set(own) - set(sd)
        extra = set(sd) - set(own)
        if missing or extra:
            raise RuntimeError(f"checkpoint does not match the model: missing {sorted(missing)[:3]}, "
                               f"unexpected {sorted(extra)[:3]}")
        for k, v in own.items():            # in place: parameters may be views into the flat bucket
            v.copy_(sd[k].to(v.dtype))
    if step is not None and not model_only and "optimizer" in state and state["optimizer"].get("state"):
        params = list(model.parameters())
        index = {id(p): i for i, p in enumerate(params)}
        ost = state["optimizer"]["state"]
        nsteps = 0
        for name, p in step.flat.named:
            off, n, shape = step.flat.slices[name]
            st = ost.get(index[id(p)])
            if st is None:
                continue
            step.exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1))
            step.exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
            nsteps = max(nsteps, int(float(st["step"])))
        step.step_dev.fill_(nsteps)
        step.set_lr(state.get("lr", step.lr))
    if step is not None and step.world > 1:
        step.sync_state()                   # every rank continues from rank 0's copy of what was loaded
    return state.get("epoch", 0), state.get("err", float("inf"))
