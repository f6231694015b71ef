"""Native training step for the HumanRF hot path (the fast path behind bench.py and the data-parallel driver).
Same maths as the reference's Trainer.train_step (humanrf/trainer.py:229-255: random background,
Huber(delta=0.01) + 1e-3 * BCE, Adam lr 1e-2 betas (0.9,0.99) eps 1e-15, lr * lr_decay^(min(step/max,1)),
run.py:101-104), but built so that ONE step never stops the device:

* prune_samples' density pass keeps the composed features of every candidate (64 B/sample); the render pass of the
  survivors runs the two MLPs on those features instead of encoding the survivors a second time
  (`reuse="feat"`; "feat+grid" also keeps the per-grid features for the scatter, "none" is the round-1 flow);
* the survivor count stays on the device (hrf_samples.num_samples_dev): no `.item()` between pruning and the forward;
* loss forward + backward is one kernel (hrf_train_loss), Adam over all tensors is one launch (hrf_adam_multi) with
  device-side step counters / active-segment flags, it refreshes the bf16 shadow tables and the packed MLP blob and
  leaves the gradient bucket zeroed for the next step;
* gradients go straight into ONE flat fp32 bucket (no per-parameter zero-filled tensors, no autograd graph);
* bf16 needs no GradScaler, so the inf-check host sync of trainer.py:250-252 disappears.

Data parallel (SURVEY 8e), one process per GPU, `exchange=`:
  "p2p"  (default) the bucket and the shadow tables live in peer-visible memory; after the backward ONE kernel
         (hrf_dp_reduce_adam) does reduce-scatter + rank-sharded Adam + all-gather of the bf16 shadows over NVLink peer
         memory, bracketed by two tiny NCCL all-reduces that act as barriers (the first also carries the
         active-segment flags).  fp32 masters and moments of the hash tables are sharded 1/world per rank
         (`gather_master_parameters()` re-assembles them for checkpoints);
  "nccl" one all-reduce of the bucket, then the single-GPU Adam on every rank.

The autograd-compatible route (humanrf_b200.volume_rendering.render + torch.optim.Adam) stays available for
running the reference's trainer.py unchanged.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from .parallel import active_segments, grid_major_bucket_layout, shard_bounds
from .scene_representation.grid_layout import MLP_SIGMA_PARAMS, mlp_blob_permutation
from .scene_representation.humanrf import HumanRF
from .volume_rendering import ray_offsets


class _RawCuda:
    """__cuda_array_interface__ view of device memory the C library allocated (peer-visible buffers)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _device_struct_array(items, dev) -> torch.Tensor:
    raw = b"".join(bytes(x) for x in items)
    return torch.from_numpy(np.frombuffer(raw, dtype=np.uint8).copy()).to(dev)


class FusedTrainer:
    def __init__(self, model: HumanRF, lr: float = 1e-2, betas=(0.9, 0.99), eps: float = 1e-15, lr_decay: float = 0.5,
                 max_steps: int = 50001, bce_loss_weight: float = 1e-3, huber_delta: float = 0.01,
                 render_step_size: float = 4e-4, world_size: int = 1, process_group=None, prune: bool = True,
                 seed: int = 123, reuse: str = "feat", exchange: str = "p2p", overlap_exchange: bool = False):
        if reuse not in ("none", "feat", "feat+grid"):
            raise ValueError("reuse must be 'none', 'feat' or 'feat+grid'")
        if exchange not in ("p2p", "nccl"):
            raise ValueError("exchange must be 'p2p' or 'nccl'")
        self.model, self.lr, self.betas, self.eps = model, lr, betas, eps
        self.lr_decay, self.max_steps = lr_decay, max_steps
        self.bce_w, self.delta, self.step_size = bce_loss_weight, huber_delta, render_step_size
        self.world, self.pg, self.prune, self.reuse = world_size, process_group, prune, reuse
        self.exchange = exchange if world_size > 1 else "local"
        # exchange="p2p", optional: run the exchange of hash grid k (barrier + reduce/Adam/shadow kernel on a side stream)
        # while grid k+1 is still being scattered.  Measured on 2 B200s (profiles/r2_dp_2gpu_overlap_ab.txt): the exposed
        # exchange shrinks 0.46 -> 0.39 ms but four per-grid scatter launches cost 0.15 ms more than one: off by default.
        self.overlap_exchange = bool(overlap_exchange) and self.exchange == "p2p"
        self.rank = dist.get_rank(process_group) if world_size > 1 else 0
        self.params: List[torch.nn.Parameter] = model.hot_parameters()
        dev = self.params[0].device
        self.dev = dev
        S = model.num_segments
        # Bucket layout (grid-major: [grid 0 of every segment | grid 1 ... | grid 3 ... | vectors, MLPs, embeddings])
        self.slices, self.regions, self.adam_order = grid_major_bucket_layout([p.numel() for p in self.params], S)
        total = self.regions[-1][1]
        self._peer_ptrs: List[int] = []
        lib = L.lib()
        if self.exchange == "p2p":
            self.grad = self._peer_buffer(total * 4).view(torch.float32)      # peers read it
        else:
            self.grad = torch.zeros(total, dtype=torch.float32, device=dev)   # the all-reduce bucket
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=dev)
        self.grad_views = [self.grad[a:b] for a, b in self.slices]
        self.t = 0                                  # optimiser steps taken (drives the learning-rate schedule)
        self.steps_dev = torch.zeros(len(self.params), dtype=torch.int32, device=dev)   # torch.optim.Adam's state['step']
        self.active_dev = torch.ones(max(S, 1), dtype=torch.int32, device=dev)          # segment touched by this step
        self.gen = torch.Generator(device=dev).manual_seed(seed)
        self.nat = model.native()
        if self.exchange == "p2p":
            self._adopt_peer_shadows()
        sg = (L.SegmentGrads * S)()
        for s_ in range(S):
            for k in range(4):
                sg[s_].grid[k] = self.grad_views[5 * s_ + k].data_ptr()
            sg[s_].vectors = self.grad_views[5 * s_ + 4].data_ptr()
        self.sg_dev = _device_struct_array([sg], dev)
        i = 5 * S
        self.mlp_grad = self.grad[self.slices[i][0]:self.slices[i + 1][1]]   # sigma params then colour params, contiguous
        assert self.mlp_grad.numel() == model.mlp_grad_elems
        self.emb_grad = self.grad_views[i + 2] if model.camera_embedding_dim > 0 else None
        dst, src = mlp_blob_permutation(model.camera_embedding_dim)
        perm = np.zeros(model.mlp_grad_elems, np.int32)
        perm[src] = dst
        self.blob_perm = torch.from_numpy(perm).to(dev)
        self._build_descriptors()
        self.last = {}
        self.profile = False
        self.keep_grad = False       # tests: leave the step's gradient in self.grad (cleared before the next backward instead)
        if self.world > 1:
            self._bar = torch.zeros(1, dtype=torch.float32, device=dev)
            self._side = torch.cuda.Stream(dev)

    # ---------------------------------------------------------------------------------------------- set-up
    def _peer_buffer(self, nbytes: int) -> torch.Tensor:
        p = C.c_void_p()
        L.check(L.lib().hrf_peer_alloc(int(nbytes), C.byref(p)))
        self._peer_ptrs.append(p.value)
        return torch.as_tensor(_RawCuda(p.value, int(nbytes)), device=self.dev)

    def _exchange_handles(self, local: torch.Tensor) -> List[int]:
        """Every rank's device address of the same buffer (CUDA IPC; own entry = local pointer)."""
        lib = L.lib()
        h = (C.c_ubyte * 64)()
        L.check(lib.hrf_peer_export(local.data_ptr(), h))
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(h), group=self.pg)
        out = []
        for r, hb in enumerate(handles):
            if r == self.rank:
                out.append(local.data_ptr())
            else:
                p = C.c_void_p()
                L.check(lib.hrf_peer_open((C.c_ubyte * 64).from_buffer_copy(hb), C.byref(p)))
                out.append(p.value)
        return out

    def _adopt_peer_shadows(self) -> None:
        """Move the bf16 shadow tables into ONE peer-visible buffer (the owners of the slices write into it remotely)."""
        m, nat = self.model, self.nat
        sizes = [g.numel() for fg in m.feature_grids for g in fg.grids()]
        self.shadow_offsets = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)
        self.shadow_flat = self._peer_buffer(int(self.shadow_offsets[-1]) * 2).view(torch.bfloat16)
        views, j = [], 0
        for s_, fg in enumerate(m.feature_grids):
            row = []
            for k in range(4):
                v = self.shadow_flat[int(self.shadow_offsets[j]):int(self.shadow_offsets[j + 1])]
                v.copy_(nat.shadows[s_][k])
                row.append(v)
                j += 1
            views.append(row)
        nat.adopt_shadows(views)
        self.peer_grad = self._exchange_handles(self.grad)
        self.peer_shadow = self._exchange_handles(self.shadow_flat)

    def _build_descriptors(self) -> None:
        m, nat, S = self.model, self.nat, self.model.num_segments
        blob_ptr = nat.blob.data_ptr()
        n_sig = MLP_SIGMA_PARAMS
        p2p = self.exchange == "p2p"
        items, first = [], 0
        for i in self.adam_order:
            p = self.params[i]
            a, b = self.slices[i]
            is_grid = i < 5 * S and i % 5 < 4
            seg_flag = self.active_dev[i // 5:].data_ptr() if (i < 5 * S and S > 1) else None
            step_ptr = self.steps_dev[i:].data_ptr()
            shadow, perm = None, None
            if is_grid:
                shadow = nat.shadows[i // 5][i % 5].data_ptr()
            elif i == 5 * S:
                shadow, perm = blob_ptr, self.blob_perm.data_ptr()
            elif i == 5 * S + 1:
                shadow, perm = blob_ptr, self.blob_perm[n_sig:].data_ptr()
            vt, vr = (nat.vec_t[i // 5].data_ptr(), int(p.shape[1])) if (i < 5 * S and i % 5 == 4) else (None, 0)
            if p2p:
                t = L.DpTensor()
                t.vectors_t, t.vec_res = vt, vr
                t.param, t.exp_avg, t.exp_avg_sq = p.data_ptr(), self.exp_avg[a:b].data_ptr(), self.exp_avg_sq[a:b].data_ptr()
                t.grad_offset, t.n = a, b - a
                t.blob_perm, t.active, t.step = perm, seg_flag, step_ptr
                if is_grid:
                    j = 4 * (i // 5) + i % 5
                    t.sharded, t.shadow_offset, t.local_shadow_bf16 = 1, int(self.shadow_offsets[j]), None
                    t.shard_begin, t.shard_end = shard_bounds(b - a, self.rank, self.world, L.ADAM_BLOCK_ELEMS)
                else:
                    t.sharded, t.shadow_offset, t.local_shadow_bf16 = 0, -1, shadow
                    t.shard_begin, t.shard_end = 0, b - a
                t.first_block = first
                first += (t.shard_end - t.shard_begin + L.ADAM_BLOCK_ELEMS - 1) // L.ADAM_BLOCK_ELEMS
            else:
                t = L.AdamTensor()
                t.vectors_t, t.vec_res = vt, vr
                t.param, t.exp_avg, t.exp_avg_sq = p.data_ptr(), self.exp_avg[a:b].data_ptr(), self.exp_avg_sq[a:b].data_ptr()
                t.grad, t.shadow_bf16, t.blob_perm = self.grad[a:b].data_ptr(), shadow, perm
                t.active, t.step, t.n, t.first_block = seg_flag, step_ptr, b - a, first
                first += (b - a + L.ADAM_BLOCK_ELEMS - 1) // L.ADAM_BLOCK_ELEMS
            items.append(t)
        self.adam_desc = _device_struct_array(items, self.dev)
        self.adam_blocks = int(first)
        # block ranges of the 5 bucket regions (grid 0..3 of every segment, then vectors / MLPs / embeddings) in the
        # descriptor table's block numbering: what one launch of the per-grid exchange covers
        firsts = [int(t.first_block) for t in items] + [int(first)]
        bounds = [firsts[k * S] for k in range(4)] + [firsts[4 * S], int(first)]
        self.region_blocks = [(bounds[k], bounds[k + 1] - bounds[k]) for k in range(5)]
        if p2p:
            self.peers = L.DpPeers()
            for r in range(self.world):
                self.peers.grad[r], self.peers.shadow[r] = self.peer_grad[r], self.peer_shadow[r]
            self.peers.world, self.peers.rank = self.world, self.rank

    @property
    def steps(self) -> List[int]:
        """torch.optim.Adam's per-parameter state['step'], in hot_parameters() order (reads the device counters)."""
        return [int(x) for x in self.steps_dev.cpu().tolist()]

    def gather_master_parameters(self) -> None:
        """exchange="p2p" shards the fp32 masters of the hash tables over the ranks: bring every rank's copy of every
        table up to date (before state_dict() / the autograd route).  Collective."""
        if self.exchange != "p2p":
            return
        S = self.model.num_segments
        with torch.no_grad():
            for i in range(5 * S):
                if i % 5 == 4:
                    continue
                flat = self.params[i].view(-1)
                for r in range(self.world):
                    a, b = shard_bounds(flat.numel(), r, self.world, L.ADAM_BLOCK_ELEMS)
                    if b > a:
                        dist.broadcast(flat[a:b], src=dist.get_global_rank(self.pg, r) if self.pg is not None else r, group=self.pg)

    # ----------------------------------------------------------------------------------------------
    def current_lr(self) -> float:
        """LambdaLR of run.py:102-104 evaluated at the number of COMPLETED steps: the scheduler is stepped after the
        optimiser (trainer.py:251-253), so the first update runs at the full learning rate."""
        return self.lr * self.lr_decay ** min(self.t / self.max_steps, 1.0)

    def step(self, o, d, frames, t, ri, rgba, num_rays: int, kernel_event=None, return_loss: bool = False,
             background: Optional[torch.Tensor] = None, cameras: Optional[torch.Tensor] = None, bwd_events=None):
        """One optimisation step on a ray batch given in InputBatch layout (device tensors; `ri` int64 as in the reference's
        InputBatch.ray_indices, or int32).  Nothing in here reads
        the device back: the step is enqueued and the call returns.  Returns the number of kernels launched, or the
        loss value when return_loss (that one read is the caller's choice)."""
        lib, nat, dev = L.lib(), self.model.native(), t.device
        launches = 0
        marks = [] if self.profile else None

        def mark(name):
            if marks is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((name, e))

        mark("start")
        step = self.step_size
        t = t.reshape(-1)
        if ri.dtype != torch.int64:      # int32 ray indices are accepted (a third of the bytes of a host upload) and widened here
            ri = ri.long()
        S = self.model.num_segments
        cams = cameras if self.model.camera_embedding_dim > 0 else None
        # Segments this batch touches (humanrf.py:162-179): the reference gives the others no gradient, so Adam leaves
        # their parameters, moments and step counters alone.  Decided AND consumed on the device.
        used = None
        if S > 1:
            used = active_segments(self.model.frame_numbers_to_segment_numbers, frames, S)
            if self.world == 1:
                self.active_dev.copy_(used)
            launches += 8
        loss_scale = head_work = None
        if self.world > 1:
            # ONE small all-reduce at the head of the step: the union batch's ray count (each rank weights its loss with
            # world * R_local / R_total so that the summed gradients are those of the union-batch mean,
            # humanrf_b200/parallel.py) and the union of the active-segment flags (a segment takes part iff ANY rank's batch
            # touches it).  Everything stays on the device.
            head = torch.zeros(1 + S, dtype=torch.float32, device=dev)
            head[0] = float(num_rays)
            if used is not None:
                head[1:] = used.float()
            # Asynchronous: the collective runs on NCCL's stream beside the prune pass (measured on 2 B200s: 0.11 ms per step
            # when the prune pass waited for it); its result is first needed by the loss kernel.
            head_work = dist.all_reduce(head, group=self.pg, async_op=True)
            launches += 6
        src = feat_src = None
        n_cap = t.shape[0]
        count = None
        # ---- prune_samples (volume_rendering.py:42-84): jitter, density-only pass, visibility compaction
        if self.prune:
            t = t + torch.rand(t.shape, device=dev, generator=self.gen) * step
            off0 = ray_offsets(ri, num_rays)
            s0 = nat.samples_rays(o, d, frames, t, ri)
            if self.reuse == "none":
                sigma0 = nat.density_early_stop(s0, off0, num_rays, step)
            else:
                sigma0, feat_src = nat.density_early_stop(s0, off0, num_rays, step, save=self.reuse)
            keep = torch.empty(n_cap, dtype=torch.uint8, device=dev)
            kept_off = torch.empty(num_rays + 1, dtype=torch.int32, device=dev)
            t2 = torch.empty(n_cap, dtype=torch.float32, device=dev)
            ri2 = torch.empty(n_cap, dtype=torch.int64, device=dev)
            src = torch.empty(n_cap, dtype=torch.int32, device=dev) if feat_src is not None else None
            count = torch.zeros(1, dtype=torch.int64, device=dev)
            L.check(lib.hrf_prune(sigma0.data_ptr(), t.data_ptr(), ri.data_ptr(), off0.data_ptr(), num_rays, step, 1e-4,
                                  1e-4, keep.data_ptr(), kept_off.data_ptr(), t2.data_ptr(), ri2.data_ptr(), L.ptr(src),
                                  count.data_ptr(), L.stream()))
            t, ri, off = t2, ri2, kept_off                  # hrf_prune's scan IS the ray-offset table of the survivors
            launches += 9
            mark("prune")
        else:
            off = ray_offsets(ri, num_rays)
            launches += 1
        # ---- forward: fused field + compositing (survivor count read from the device by the kernels)
        samples = nat.samples_rays(o, d, frames, t, ri, cams, count_dev=count)
        if feat_src is not None:
            sigma, rgb = nat.forward_from_features(samples, feat_src, src)
            feat, egrid, egrid_stride = feat_src, (feat_src.data_ptr() + 64 * n_cap if self.reuse == "feat+grid" else None), n_cap
        else:
            sigma, _, rgb, feat = nat.forward(samples, 1, want_geo=False, want_feat=True)
            egrid, egrid_stride = feat.data_ptr() + 64 * n_cap, n_cap
        if kernel_event is not None:
            kernel_event.record()
        mark("forward")
        bg = background if background is not None else torch.rand((num_rays, 3), device=dev, generator=self.gen)  # trainer.py:237
        color = torch.empty((num_rays, 3), dtype=torch.float32, device=dev)
        wsum = torch.empty((num_rays, 1), dtype=torch.float32, device=dev)
        L.check(lib.hrf_composite_forward(sigma.data_ptr(), rgb.data_ptr(), t.data_ptr(), off.data_ptr(), num_rays, step,
                                          bg.data_ptr(), color.data_ptr(), wsum.data_ptr(), None, L.stream()))
        # ---- loss (Huber + BCE) and its gradient w.r.t. the [R,3] / [R] outputs in one launch
        d_color = torch.empty((num_rays, 3), dtype=torch.float32, device=dev)
        d_wsum = torch.empty(num_rays, dtype=torch.float32, device=dev)
        loss = torch.zeros(1, dtype=torch.float32, device=dev)
        rgba = rgba if (rgba.dtype == torch.float32 and rgba.is_contiguous()) else rgba.float().contiguous()
        if head_work is not None:
            head_work.wait()           # the current stream waits for the head all-reduce (no host synchronisation)
            loss_scale = (float(self.world * num_rays) / head[:1].clamp(min=1.0)).contiguous()
            if used is not None:
                self.active_dev.copy_(head[1:] > 0)
        L.check(lib.hrf_train_loss(color.data_ptr(), wsum.data_ptr(), rgba.data_ptr(), bg.data_ptr(), num_rays, self.delta,
                                   self.bce_w, L.ptr(loss_scale), d_color.data_ptr(), d_wsum.data_ptr(), loss.data_ptr(),
                                   L.stream()))
        # ---- backward: compositing, then the fused field backward into the flat bucket (clean: Adam re-zeroes it)
        d_sigma = torch.empty(n_cap, dtype=torch.float32, device=dev)
        d_rgb = torch.empty((n_cap, 3), dtype=torch.float32, device=dev)
        L.check(lib.hrf_composite_backward(sigma.data_ptr(), rgb.data_ptr(), t.data_ptr(), off.data_ptr(), num_rays, step,
                                           bg.data_ptr(), d_color.data_ptr(), d_wsum.data_ptr(), d_sigma.data_ptr(),
                                           d_rgb.data_ptr(), L.stream()))
        mark("composite+loss")
        if bwd_events is not None:
            bwd_events[0].record()
        if self.keep_grad:
            self.grad.zero_()
        ws = torch.empty(n_cap * 40, dtype=torch.float32, device=dev)   # 160 B / sample
        L.check(lib.hrf_field_backward_mlp(C.byref(nat.field), C.byref(samples), d_sigma.data_ptr(), d_rgb.data_ptr(), None,
                                           feat.data_ptr(), L.ptr(src), self.mlp_grad.data_ptr(), L.ptr(self.emb_grad),
                                           ws.data_ptr(), L.stream()))
        mark("backward_mlp")
        if self.overlap_exchange:
            launches += self._scatter_and_exchange_overlapped(nat, samples, egrid, src, egrid_stride, ws, mark)
        else:
            L.check(lib.hrf_field_backward_tables(C.byref(nat.field), C.byref(samples), self.sg_dev.data_ptr(), egrid, L.ptr(src),
                                                  egrid_stride, ws.data_ptr(), 0, 4, L.stream()))
            launches += 8
            if bwd_events is not None:
                bwd_events[1].record()
            mark("scatter")
            launches += self._exchange_and_adam()
            mark("exchange+adam")
        self.last = {"samples": count[0] if count is not None else n_cap, "loss": loss[0], "marks": marks}
        if return_loss:
            return float(loss.item())
        return launches

    def _exchange_and_adam(self) -> int:
        lib = L.lib()
        lr = self.current_lr()
        self.t += 1
        b1, b2 = self.betas
        if self.world == 1:
            L.check(lib.hrf_adam_multi(self.adam_desc.data_ptr(), len(self.params), self.adam_blocks, lr, b1, b2, self.eps, 1.0,
                                       0 if self.keep_grad else 1, L.stream()))
            return 2
        if self.exchange == "nccl":
            dist.all_reduce(self.grad, group=self.pg)
            L.check(lib.hrf_adam_multi(self.adam_desc.data_ptr(), len(self.params), self.adam_blocks, lr, b1, b2, self.eps,
                                       1.0 / self.world, 1, L.stream()))
            return 3
        # barrier A: every rank's gradients are complete
        dist.all_reduce(self._bar, group=self.pg)
        L.check(lib.hrf_dp_reduce_adam(C.byref(self.peers), self.adam_desc.data_ptr(), len(self.params), 0, self.adam_blocks, 1, lr,
                                       b1, b2, self.eps, 1.0 / self.world, L.stream()))
        # barrier B: every peer has read this rank's bucket and written this rank's shadow slices
        dist.all_reduce(self._bar, group=self.pg)
        self.grad.zero_()
        return 6

    def _scatter_and_exchange_overlapped(self, nat, samples, egrid, src, egrid_stride, ws, mark) -> int:
        """exchange="p2p", overlapped: the scatter runs one hash grid per launch; as soon as grid k's launch is queued, a side
        stream waits for it, passes a cross-rank barrier (all ranks' gradients of grid k complete) and runs the
        reduce-scatter / Adam / shadow all-gather kernel over grid k's tensors -- while the main stream scatters grid k+1.
        The small tensors follow the last grid; one closing barrier (all shadows written, all buckets read), the bucket is
        cleared, and the main stream waits for the side stream."""
        lib = L.lib()
        lr = self.current_lr()
        self.t += 1
        b1, b2 = self.betas
        main, side = torch.cuda.current_stream(), self._side
        for k in range(4):
            L.check(lib.hrf_field_backward_tables(C.byref(nat.field), C.byref(samples), self.sg_dev.data_ptr(), egrid, L.ptr(src),
                                                  egrid_stride, ws.data_ptr(), k, 1, L.stream()))
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(side):
                side.wait_event(ev)
                dist.all_reduce(self._bar, group=self.pg)
                first, count = self.region_blocks[k]
                L.check(lib.hrf_dp_reduce_adam(C.byref(self.peers), self.adam_desc.data_ptr(), len(self.params), first, count,
                                               1 if k == 0 else 0, lr, b1, b2, self.eps, 1.0 / self.world, side.cuda_stream))
        mark("scatter")
        with torch.cuda.stream(side):
            first, count = self.region_blocks[4]      # vectors (complete after the last scatter launch), MLPs, embeddings
            L.check(lib.hrf_dp_reduce_adam(C.byref(self.peers), self.adam_desc.data_ptr(), len(self.params), first, count, 0, lr, b1,
                                           b2, self.eps, 1.0 / self.world, side.cuda_stream))
            dist.all_reduce(self._bar, group=self.pg)
            self.grad.zero_()
            done = torch.cuda.Event()
            done.record(side)
        main.wait_event(done)
        mark("exchange+adam")
        return 8 + 4 + 5 * 2 + 2

    def close(self) -> None:
        """Releases the peer-visible buffers (exchange="p2p").  Collective-free; call after the last step."""
        if self.exchange == "p2p" and self._peer_ptrs:
            torch.cuda.synchronize()
            lib = L.lib()
            for r in range(self.world):
                if r != self.rank:
                    lib.hrf_peer_close(self.peer_grad[r])
                    lib.hrf_peer_close(self.peer_shadow[r])
            self._peer_ptrs = []      # the buffers themselves stay alive as long as tensors view them (process lifetime)
