"""Stage-1 training step — the loop body of the reference's train.py:66-97 (before LPIPS starts at epoch 30) — over the
fused kernels, with optional frame-level data parallelism (one process per GPU; the only collective is one all-reduce of
the shared feature-net / geo_feature gradients, SURVEY.md §8e).

    loss = lambda_scale * scale_loss + wdecay_rgl * offset_loss + (1-lambda_dssim) * L1 + lambda_dssim * (1-SSIM) + geo_loss
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist

from .losses import image_loss
from .optim import FusedAdam


def adjust_loss_weights(init_weight, current_epoch, mode="decay", start=400, every=20):
    """Loss-weight schedule of utils/general_utils.py:260-279 as train.py:60 uses it for the offset regulariser:
    constant before `start`, then x0.85 ('decay') or x1.05 ('rise') every `every` epochs."""
    if mode == "binary":
        raise ValueError("mode='binary' leaves the weight undefined in the reference")
    if current_epoch < start:
        return init_weight * 1e-6 if mode == "rise" else init_weight
    if every == 0:
        return init_weight
    factor = 1.05 if mode == "rise" else 0.85
    return init_weight * (factor ** ((current_epoch - start) // every))


def allreduce_gradients(grads, group=None):
    """SUM all-reduce of a list of gradient tensors (asynchronously issued, then waited).  The caller divides by the world
    size (FusedAdam.grad_scale).  Works with any torch.distributed backend (NCCL on the GPUs, gloo in the CPU tests)."""
    works = [dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group, async_op=True) for g in grads if g is not None]
    for w in works:
        w.wait()


class _StepGraph:
    """One captured forward + loss + backward of a stage-1 step and its static input / output tensors."""
    __slots__ = ("graph", "idx", "gt", "cams", "loss", "g_flat", "g_geo", "capacity", "plan", "states", "launches")


class Stage1Trainer:
    """The loop body of train.py:66-97 for either training stage (the name dates from when only stage 1 existed; `AvatarTrainer` is an alias)."""
    def __init__(self, model, fused_adam: bool = True, process_group=None, use_graph=None, perceptual_loss=None):
        self.model = model
        # train.py:26,89-91: after `lpips_start_iter` epochs the reference adds lambda_lpips * LPIPS((image-0.5)*2, (gt-0.5)*2).  LPIPS is
        # an external pretrained network (out of scope, SURVEY.md §2 #6): pass any callable(image, gt) -> scalar here to get the term
        self.perceptual_loss = perceptual_loss
        self._warned_lpips = False
        # whole-step CUDA graph (forward + loss + backward in ONE launch; all-reduce and Adam follow eagerly): on unless GA_STEP_GRAPH=0
        self.use_graph = (os.environ.get("GA_STEP_GRAPH", "1") != "0") if use_graph is None else bool(use_graph)
        self._graphs = {}
        self.host_wait_s = self.host_enqueue_s = 0.0
        self.replayed_launches = 0      # kernels of this library launched through graph replays (ga_launch_count sees only eager launches)
        self.opt = model.opt_parms
        self.world = dist.get_world_size(process_group) if (dist.is_available() and dist.is_initialized()) else 1
        self.group = process_group
        # the caller may already have followed the reference's resume order (training_setup() -> load(), train.py:36-45): keep what it loaded
        prev_opt = model.optimizer.state_dict() if model.optimizer is not None else None
        prev_sched = model.scheduler.state_dict() if model.scheduler is not None else None
        if model.optimizer is None:
            model.training_setup()
        if fused_adam and not isinstance(model.optimizer, FusedAdam):
            # same hyper-parameters / groups / state layout as the torch.optim.Adam the reference builds (avatar_model.py:150-155)
            if getattr(model.model_parms, "train_stage", 1) == 2:
                model.optimizer = FusedAdam([{"params": list(model.net.parameters()), "lr": self.opt.lr_net * 0.1},
                                             {"params": list(model.pose_encoder.parameters()), "lr": self.opt.lr_net}])
            else:
                model.optimizer = FusedAdam([{"params": list(model.net.parameters()), "lr": self.opt.lr_net},
                                             {"params": [model.geo_feature], "lr": self.opt.lr_geomfeat}])
            model.scheduler = torch.optim.lr_scheduler.MultiStepLR(model.optimizer, self.opt.sched_milestones, gamma=0.1)
            if prev_opt is not None and prev_opt.get("state"):
                model.optimizer.load_state_dict(model.translate_optimizer_state(prev_opt))
            if prev_sched is not None and prev_sched.get("last_epoch", 0) > 0:
                model.scheduler.load_state_dict(prev_sched)
        self._comm_stream = None

    def loss(self, batch, iteration: int, epoch: int = 0):
        """Forward only: returns (loss, image) exactly as train.py:70-77 forms them."""
        m, o = self.model, self.opt
        wdecay_rgl = adjust_loss_weights(o.lambda_rgl, epoch, mode="decay", start=self.epoch_start, every=20)   # train.py:60
        if getattr(m.model_parms, "train_stage", 1) == 2:                                                      # train.py:79-86
            image, points, pose_loss, offset_loss = m.train_stage2(batch, iteration)
            loss = wdecay_rgl * offset_loss + image_loss(image, batch["original_image"], o.lambda_dssim) + pose_loss * 10
        else:
            image, points, offset_loss, geo_loss, scale_loss = m.train_stage1(batch, iteration)
            loss = o.lambda_scale * scale_loss + wdecay_rgl * offset_loss + image_loss(image, batch["original_image"], o.lambda_dssim) + geo_loss
        if epoch > o.lpips_start_iter:                   # train.py:89-91
            if self.perceptual_loss is not None:
                gt = batch["original_image"]
                loss = loss + o.lambda_lpips * torch.mean(self.perceptual_loss((image - 0.5) * 2, (gt - 0.5) * 2))
            elif not self._warned_lpips:
                import warnings
                warnings.warn(f"epoch {epoch} > lpips_start_iter {o.lpips_start_iter}: the reference adds lambda_lpips * LPIPS from here on "
                              "(train.py:89-91) but no perceptual_loss callable was given to Stage1Trainer; the term is omitted")
                self._warned_lpips = True
        return loss, image

    epoch_start = 0    # train.py:38-45: 0 unless resuming from a checkpoint

    def sync_gradients(self):
        """Data parallelism: ONE all-reduce(sum) per step over a flat bucket [net.flat.grad | geo_feature.grad | overflow flag]
        (6.2 MB), issued asynchronously on NCCL's stream; the compute stream waits for it in-stream (the host does not), the
        1/world factor is folded into the Adam kernel and the gradients Adam reads are the bucket's views.  The last word
        carries the batched rasterizer's overflow flag, so that every rank skips (and later re-runs) a step any rank could not
        fit.  Pose / transl embedding rows are per-frame and stay rank-local (sparse grads)."""
        if self.world == 1:
            return
        m = self.model
        # the parameters every rank shares: stage 1 = feature net + geo_feature, stage 2 = feature net + pose encoder (avatar_model.py:148-161)
        shared = [m.net.flat] + ([m.geo_feature] if getattr(m.model_parms, "train_stage", 1) != 2 else list(m.pose_encoder.parameters()))
        shared = [p for p in shared if p.grad is not None]
        sizes = [p.grad.numel() for p in shared]
        total = sum(sizes)
        dev = shared[0].grad.device
        bk = getattr(self, "_bucket", None)
        if bk is None or bk.numel() != total + 1:
            bk = self._bucket = torch.zeros(total + 1, dtype=torch.float32, device=dev)
            self._skip = torch.zeros(1, dtype=torch.int32, device=dev)
            self._flag_host = torch.zeros(1, dtype=torch.float32).pin_memory() if dev.type == "cuda" else torch.zeros(1)
            self._flag_event = torch.cuda.Event() if dev.type == "cuda" else None
        off = 0
        for p, n in zip(shared, sizes):
            bk[off:off + n].copy_(p.grad.reshape(-1))
            off += n
        plan = getattr(m, "_last_plan", None)
        if plan is not None:
            bk[total:].copy_(plan.status_dev[1:2])
        else:
            bk[total:].zero_()
        work = dist.all_reduce(bk, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        work.wait()                                   # stream-level wait on CUDA; a host wait only with gloo (CPU tests)
        off = 0
        for p, n in zip(shared, sizes):
            p.grad = bk[off:off + n].view_as(p.grad)
            off += n
        self._skip.copy_(bk[total:] != 0)
        self._flag_host.copy_(bk[total:], non_blocking=True)
        if self._flag_event is not None:
            self._flag_event.record()

    def _step_fitted(self) -> bool:
        """Did the previous step fit the rasterizer's binning buffer — on every rank?  (Grows this rank's buffer if it did not.)"""
        ok = self.model.raster_ok(wait=True)
        if self.world > 1 and getattr(self, "_flag_event", None) is not None:
            self._flag_event.synchronize()
            ok = ok and float(self._flag_host[0]) == 0.0
        return ok

    def step(self, batch, iteration: int, epoch: int = 0):
        """One optimisation step.  The batched rasterizer never makes the host wait for the device: whether the step's binning
        buffer was large enough is known one step later (the device flag also turns that step's Adam launches into no-ops), so
        an overflowed step is detected here, before the next one, and simply run again with the grown buffer."""
        import time as _time
        t0 = _time.perf_counter()
        prev = getattr(self, "_prev", None)
        if prev is not None and not self._step_fitted():
            self._undo_host_step(prev[2])
            self._step_once(*prev)
            if not self._step_fitted():
                raise RuntimeError("batched rasterizer: binning buffer overflowed twice in a row")
        t1 = _time.perf_counter()
        self._prev = (batch, iteration, epoch)
        out = self._step_once(batch, iteration, epoch)
        self.host_wait_s += t1 - t0                      # waiting for the previous step's rasterizer status (the GPU is busy meanwhile)
        self.host_enqueue_s += _time.perf_counter() - t1  # enqueueing this step
        return out

    def finish(self):
        """Settle the last step (re-run it if its binning buffer overflowed).  Returns the loss of the re-run, None if there was none."""
        prev, self._prev = getattr(self, "_prev", None), None
        if prev is not None and not self._step_fitted():
            self._undo_host_step(prev[2])
            out = self._step_once(*prev)
            if not self._step_fitted():
                raise RuntimeError("batched rasterizer: binning buffer overflowed twice in a row")
            return out
        return None

    def _undo_host_step(self, epoch):
        """Host-side bookkeeping of a step the device skipped (Adam step counts, lr schedule)."""
        m = self.model
        for st in m.optimizer.state.values():
            if "step" in st:
                st["step"] = st["step"] - 1
        m.scheduler.last_epoch -= 1
        m.scheduler._step_count -= 1
        for g, lr in zip(m.optimizer.param_groups, m.scheduler._get_closed_form_lr() if hasattr(m.scheduler, "_get_closed_form_lr") else m.scheduler.get_last_lr()):
            g["lr"] = lr

    # ---- whole-step CUDA graph -------------------------------------------------------------------------------------------------
    def sync_pose_gradients(self, epoch):
        """Pose optimisation under data parallelism (epoch > pose_op_start_iter): every rank must apply the SAME sparse update to its
        replica of the pose / transl tables.  The touched rows (this rank's frames) and their gradients are all-gathered, scaled by
        1/world (the global loss is the mean of the ranks' losses) and installed as the sparse gradient SparseAdam steps on."""
        m = self.model
        if self.world == 1 or epoch <= self.opt.pose_op_start_iter:
            return
        for emb in (m.pose, m.transl):
            g = emb.weight.grad
            if g is None:
                continue
            g = g.coalesce()
            idx, val = g.indices()[0].contiguous(), g.values().contiguous()
            n = torch.tensor([idx.numel()], device=idx.device)
            counts = [torch.zeros_like(n) for _ in range(self.world)]
            dist.all_gather(counts, n, group=self.group)
            nmax = int(max(int(c) for c in counts))
            pad_i = torch.zeros(nmax, dtype=idx.dtype, device=idx.device); pad_i[:idx.numel()] = idx
            pad_v = torch.zeros(nmax, val.shape[1], dtype=val.dtype, device=val.device); pad_v[:idx.numel()] = val
            all_i = [torch.zeros_like(pad_i) for _ in range(self.world)]
            all_v = [torch.zeros_like(pad_v) for _ in range(self.world)]
            dist.all_gather(all_i, pad_i, group=self.group)
            dist.all_gather(all_v, pad_v, group=self.group)
            ii = torch.cat([a[:int(c)] for a, c in zip(all_i, counts)])
            vv = torch.cat([a[:int(c)] for a, c in zip(all_v, counts)]) / self.world
            emb.weight.grad = torch.sparse_coo_tensor(ii[None], vv, emb.weight.shape).coalesce()

    def _graph_applicable(self, batch, iteration, epoch) -> bool:
        """The captured step holds no host-dependent value: the scale ramp is over (iteration >= 1000, avatar_model.py:316-319), pose
        optimisation is inactive (its sparse embedding gradients are then never read, avatar_model.py:261-270) and the frames share
        one image size."""
        m = self.model
        img = batch.get("original_image")
        return (self.use_graph and isinstance(m.optimizer, FusedAdam) and getattr(m.model_parms, "train_stage", 1) != 2
                and iteration >= 1000 and epoch <= self.opt.pose_op_start_iter
                and not (self.perceptual_loss is not None and epoch > self.opt.lpips_start_iter)
                and torch.is_tensor(img) and img.is_cuda and img.shape[0] <= 8 and os.environ.get("GA_RASTER_BATCHED", "1") != "0"
                and m._uniform_frames(batch, img.shape[0]))

    def _capture(self, batch, iteration, epoch, key):
        m = self.model
        dev = m.device
        B = batch["original_image"].shape[0]
        G = _StepGraph()
        G.idx = batch["pose_idx"].to(dev).clone()
        G.gt = batch["original_image"].float().contiguous().clone()
        G.cams = m._batch_cameras(batch, B, dev).clone()
        sb = dict(batch)
        sb.update(pose_idx=G.idx, original_image=G.gt, _cams=G.cams, height=m._scalar_list(batch["height"], B),
                  width=m._scalar_list(batch["width"], B))
        m._detach_pose = True
        run_backup = m.net.bn_running.clone()
        states = [(st, st.num_batches_tracked) for st in m.net._states.values()]
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                      # warm-up off the capture: allocator pools, lazy one-time setup in the library
            for _ in range(2):
                loss, _ = self.loss(sb, iteration, epoch)
                m.optimizer.zero_grad(set_to_none=True)
                loss.backward()
        torch.cuda.current_stream().wait_stream(side)
        if not m.raster_ok(wait=True):                      # the warm-up found the binning buffer too small: it has been grown
            pass
        m.optimizer.zero_grad(set_to_none=True)
        from . import _lib
        G.graph = torch.cuda.CUDAGraph()
        l0 = _lib.launch_count()
        with torch.cuda.graph(G.graph):
            loss, _ = self.loss(sb, iteration, epoch)
            loss.backward()
        G.launches = _lib.launch_count() - l0
        G.loss = loss.detach()
        G.g_flat, G.g_geo = m.net.flat.grad, m.geo_feature.grad
        G.plan = m._last_plan
        G.capacity = G.plan.capacity
        m.net.bn_running.copy_(run_backup)                  # warm-up and capture must not count as training iterations
        G.states = [st for st, n in states if st.num_batches_tracked != n] or [st for st in m.net._states.values()
                                                                                 if not any(st is s0 for s0, _ in states)]
        for st in m.net._states.values():
            st.num_batches_tracked = 0
        for st, n in states:
            st.num_batches_tracked = n
        m._detach_pose = False
        self._graphs[key] = G
        return G

    def _step_graphed(self, batch, iteration, epoch):
        m, o = self.model, self.opt
        B = batch["original_image"].shape[0]
        wdecay_rgl = adjust_loss_weights(o.lambda_rgl, epoch, mode="decay", start=self.epoch_start, every=20)
        key = (B, tuple(batch["original_image"].shape[-2:]), float(wdecay_rgl))
        G = self._graphs.get(key)
        if G is not None and G.capacity != G.plan.capacity:      # the rasterizer's buffers were re-allocated: the graph points at freed memory
            G = None
        if G is None:
            G = self._capture(batch, iteration, epoch, key)
        G.idx.copy_(batch["pose_idx"], non_blocking=True)
        G.gt.copy_(batch["original_image"], non_blocking=True)
        G.cams.copy_(m._batch_cameras(batch, B, m.device))
        G.plan.bump_serial()
        G.plan.pending = True
        m._last_plan = G.plan
        G.graph.replay()
        self.replayed_launches += G.launches
        for st in G.states:
            st.num_batches_tracked += 1
        m.net.flat.grad, m.geo_feature.grad = G.g_flat, G.g_geo
        return G.loss

    def _step_once(self, batch, iteration: int, epoch: int = 0):
        """Runs the step on a dedicated non-default stream when the caller sits on the default one: autograd ties each parameter's
        AccumulateGrad node to the stream of its first backward, and a node tied to the legacy default stream makes every later graph
        capture illegal (the engine would have to synchronise with stream 0 inside the capture)."""
        m = self.model
        if self.use_graph and m.device.type == "cuda":
            cur = torch.cuda.current_stream(m.device)
            if cur == torch.cuda.default_stream(m.device):
                if getattr(self, "_stream", None) is None:
                    self._stream = torch.cuda.Stream(device=m.device)
                self._stream.wait_stream(cur)
                with torch.cuda.stream(self._stream):
                    out = self._step_impl(batch, iteration, epoch)
                cur.wait_stream(self._stream)
                return out
        return self._step_impl(batch, iteration, epoch)

    def _step_impl(self, batch, iteration: int, epoch: int = 0):
        m = self.model
        if self._graph_applicable(batch, iteration, epoch):
            loss = self._step_graphed(batch, iteration, epoch)
        else:
            loss, _ = self.loss(batch, iteration, epoch)
            m.zero_grad(epoch)
            loss.backward()
        self.sync_gradients()
        self.sync_pose_gradients(epoch)
        if isinstance(m.optimizer, FusedAdam):
            m.optimizer.grad_scale = 1.0 / self.world
            plan = getattr(m, "_last_plan", None)
            m.optimizer.skip_flag = self._skip if self.world > 1 else (plan.status_dev[1:2] if plan is not None else None)
        elif self.world > 1:
            for group in m.optimizer.param_groups:
                for p in group["params"]:
                    if p.grad is not None:
                        p.grad.div_(self.world)
        m.step(epoch)
        return loss


AvatarTrainer = Stage1Trainer
