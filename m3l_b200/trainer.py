"""Fused VTMAE train step: zero_grad -> forward -> backward -> [gradient all-reduce] ->
clip_grad_norm_(0.5) -> AdamW.step -> bf16 shadow refresh, as one kernel sequence over flat arenas,
optionally replayed from CUDA graphs.  Semantics of /root/reference/models/pretrain_models.py:707-711
with torch.optim.AdamW defaults (:670-676).

Data parallel (one process per GPU): identical replicas, rank-sharded batch; the flat gradient arena
is all-reduced (AVG) in two buckets — heads+decoder as soon as their backward is done, overlapping
the encoder backward on a side stream, then encoder+embeddings (SURVEY.md §8e).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Tuple

import torch

from . import dp, engine, ops
from ._lib import M3LError
from .data import clone_inputs, copy_inputs, input_signature


class FusedAdamW:
    """Minimal optimizer facade (param_groups / state_dict) over the trainer's flat moment arenas.

    Differences from torch.optim.AdamW, by construction of the flat-arena step: ONE step counter serves every
    parameter (torch keeps one per parameter, which only differs for parameters that receive a gradient in some
    steps and not in others, e.g. alternating use_tactile); zero_grad() always zero-fills (the gradient arena is a
    persistent buffer, `set_to_none` is accepted and ignored).  lr / betas / eps / weight_decay may be changed
    through param_groups at any time: they are read from a device buffer at run time, also under graph replay."""

    def __init__(self, trainer, lr, betas, eps, weight_decay):
        self._t = trainer
        self.param_groups = [dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay,
                                  params=[trainer.model.arena.params[n] for n in trainer.model.arena.names])]

    def zero_grad(self, set_to_none: bool = True):
        self._t.gflat.zero_()

    def state_dict(self):
        t = self._t
        return dict(step=float(t.state[0].item()), exp_avg=t.m.clone(), exp_avg_sq=t.v.clone(),
                    param_groups=[{k: v for k, v in self.param_groups[0].items() if k != "params"}])

    def load_state_dict(self, sd):
        t = self._t
        t.state[0] = sd["step"]
        t.m.copy_(sd["exp_avg"]); t.v.copy_(sd["exp_avg_sq"])


class FusedTrainer:
    _MAX_GRAPHS = 4      # captured (modalities, batch) shapes kept alive; oldest evicted first

    def __init__(self, model, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, max_norm=0.5,
                 process_group=None, use_cuda_graph=True):
        self.model = model
        A = model.arena
        dev = A.device
        self.gflat = torch.zeros(A.total, dtype=torch.float32, device=dev)
        self.m = torch.zeros_like(self.gflat)
        self.v = torch.zeros_like(self.gflat)
        self.state = torch.zeros(ops.OPT_STATE_DOUBLES, dtype=torch.float64, device=dev)  # step, sumsq, norm, bias corrections
        self.hyper = torch.zeros(8, dtype=torch.float32, device=dev)   # lr, beta1, beta2, eps, weight_decay, max_norm
        self._hyper_host = None
        self.max_norm = max_norm
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.use_graph = use_cuda_graph
        self.opt = FusedAdamW(self, lr, betas, eps, weight_decay)
        self._graphs: Dict = {}
        self.comm_stream = torch.cuda.Stream(device=dev) if self.world > 1 else None
        # M3L_DP_ONE_GRAPH=0: keep the NCCL calls outside the graphs (four graph replays per step, host-launched
        # all-reduces between them) - the fallback if a NCCL build cannot be stream-captured
        self.one_graph_dp = os.environ.get("M3L_DP_ONE_GRAPH", "1") != "0"
        self.kernel_launches_per_step = None

    def optimizer_facade(self):
        return self.opt

    # ------------------------------------------------------------------------------------
    def _plan(self, geo):
        """(live names, all live ranges, [bucket ranges]) - three buckets in the order their gradients become final:
        heads + decoder, encoder transformer, token embeddings (dp.split_three)."""
        model, A = self.model, self.model.arena
        live = model.live_param_names(geo, True)
        return live, A.ranges(live), [A.ranges(names) for names in dp.split_three(live)]

    def _phase_a(self, xs, noise, geo, box):
        self.gflat.zero_()
        self.state[1:2].zero_()
        loss_acc, ctx = engine.mae_forward(self.model, xs, noise, geo, training=True, gflat=self.gflat)
        engine.mae_backward_decoder(self.model, ctx, self.gflat)
        box["loss"], box["ctx"] = loss_acc, ctx

    def _phase_b(self, box):
        self._phase_b1(box)
        self._phase_b2(box)

    def _phase_b1(self, box):
        box["dx0"] = engine.mae_backward_encoder_stack(self.model, box["ctx"], self.gflat)

    def _phase_b2(self, box):
        engine.mae_backward_embed(self.model, box["ctx"], self.gflat, box["dx0"])

    def _dp_sequence(self, xs, noise, geo, box, ranges, buckets):
        """The data-parallel step as one stream program: each bucket's all-reduce runs on the communication stream
        beside the next phase of the backward (event fork / join, so the whole sequence - NCCL included - can be
        captured into ONE CUDA graph): decoder bucket || encoder-stack backward, encoder-stack bucket || embedding
        backward, embedding bucket, then clip + AdamW on the averaged gradients."""
        main = torch.cuda.current_stream()
        phases = (lambda: self._phase_a(xs, noise, geo, box), lambda: self._phase_b1(box), lambda: self._phase_b2(box))
        for phase, rng in zip(phases, buckets):
            phase()
            if rng:
                self.comm_stream.wait_stream(main)
                with torch.cuda.stream(self.comm_stream):
                    dp.allreduce_ranges(self.gflat, rng, group=self.pg)
        main.wait_stream(self.comm_stream)
        self._phase_c(ranges)

    def _push_hyper(self):
        """Optimizer hyper-parameters -> device buffer (only when they changed): the kernels read them at run time,
        so captured graphs follow param_groups (LR schedules) without re-capture."""
        g = self.opt.param_groups[0]
        vals = (float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]),
                float(self.max_norm if self.max_norm is not None else 0.0))
        if vals != self._hyper_host:
            self.hyper[:6].copy_(torch.tensor(vals, dtype=torch.float32))
            self._hyper_host = vals

    def _phase_c(self, ranges):
        A = self.model.arena
        g = self.opt.param_groups[0]
        for s, e in ranges:
            ops.grad_sumsq(self.gflat[s:e], self.state)
        ops.optimizer_step_begin(self.state, g["betas"], hyper=self.hyper)
        for s, e in ranges:
            ops.clip_adamw(A.flat[s:e], self.gflat[s:e], self.m[s:e], self.v[s:e], self.state, lr=g["lr"],
                           betas=g["betas"], eps=g["eps"], weight_decay=g["weight_decay"], max_norm=self.max_norm,
                           hyper=self.hyper)
        A.refresh_shadows()

    # ------------------------------------------------------------------------------------
    def step(self, x, noise=None, use_vision=True, use_tactile=True):
        model = self.model
        A = model._sync()
        xs, geo, B = model._prep_inputs(x, use_vision, use_tactile)
        if noise is None:
            noise = torch.rand(B, geo.n, device=A.device)
        noise = noise.to(device=A.device, dtype=torch.float32).contiguous()
        live, ranges, buckets = self._plan(geo)
        for k in live:
            p = A.params[k]
            if p.grad is None or p.grad.data_ptr() != A.view(self.gflat, k).data_ptr():
                p.grad = A.view(self.gflat, k)
        self._push_hyper()
        if not self.use_graph:
            box = {}
            if self.world > 1:
                self._dp_sequence(xs, noise, geo, box, ranges, buckets)
            else:
                self._phase_a(xs, noise, geo, box)
                self._phase_b(box)
                self._phase_c(ranges)
            A._version_seen = A.version()
            return box["loss"].reshape(())
        key = (geo.use_vision, geo.nt, B, input_signature(xs), engine.p_drop(model.encoder.transformer))
        g = self._graphs.get(key)
        if g is None:
            while len(self._graphs) >= self._MAX_GRAPHS:       # each capture owns a full activation pool
                self._graphs.pop(next(iter(self._graphs)))
            g = self._capture(xs, noise, geo, ranges, buckets)
            self._graphs[key] = g
        copy_inputs(g["xs"], xs)
        g["noise"].copy_(noise, non_blocking=True)
        if "all" in g:
            g["all"].replay()             # single GPU, or the data-parallel step with its all-reduces captured
        else:
            main = torch.cuda.current_stream()
            for name, rng in zip(("a", "b1", "b2"), buckets):
                g[name].replay()
                if rng:
                    self.comm_stream.wait_stream(main)
                    with torch.cuda.stream(self.comm_stream):
                        dp.allreduce_ranges(self.gflat, rng, group=self.pg)
            main.wait_stream(self.comm_stream)
            g["c"].replay()
        A._version_seen = A.version()
        return g["box"]["loss"].reshape(())

    def _capture(self, xs, noise, geo, ranges, buckets):
        """Warm-up once eagerly (lazy kernel attributes, allocator), then capture."""
        sx = clone_inputs(xs)
        sn = noise.clone()
        # eager warm-up on a side stream must not advance the optimizer: snapshot & restore state
        snap = (self.model.arena.flat.clone(), self.m.clone(), self.v.clone(), self.state.clone())
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            box = {}
            if self.world > 1:
                # the warm-up runs the real data-parallel sequence: NCCL sets up its channels / buffers on the first
                # collective of a communicator (host-side allocation and peer exchange), which must not happen for
                # the first time inside a stream capture
                self._dp_sequence(sx, sn, geo, box, ranges, buckets)
            else:
                self._phase_a(sx, sn, geo, box)
                self._phase_b(box)
                self._phase_c(ranges)
        torch.cuda.current_stream().wait_stream(s)
        if self.world > 1:
            torch.cuda.current_stream().wait_stream(self.comm_stream)
        torch.cuda.synchronize()
        self.model.arena.flat.copy_(snap[0]); self.m.copy_(snap[1]); self.v.copy_(snap[2]); self.state.copy_(snap[3])
        self.model.arena.refresh_shadows()
        out = {"xs": sx, "noise": sn, "box": {}}
        counter = ops.LaunchCounter()
        with engine.capture_guard():
            if self.world == 1:
                g = torch.cuda.CUDAGraph()
                with counter, torch.cuda.graph(g):
                    self._phase_a(sx, sn, geo, out["box"])
                    self._phase_b(out["box"])
                    self._phase_c(ranges)
                out["all"] = g
            elif self.one_graph_dp:
                # NCCL all-reduces captured with the kernels: one graph launch per step, no host in the loop
                g = torch.cuda.CUDAGraph()
                with counter, torch.cuda.graph(g, capture_error_mode="thread_local"):
                    self._dp_sequence(sx, sn, geo, out["box"], ranges, buckets)
                out["all"] = g
            else:
                gs = [torch.cuda.CUDAGraph() for _ in range(4)]
                pool = torch.cuda.graph_pool_handle()
                with counter:
                    with torch.cuda.graph(gs[0], pool=pool):
                        self._phase_a(sx, sn, geo, out["box"])
                    with torch.cuda.graph(gs[1], pool=pool):
                        self._phase_b1(out["box"])
                    with torch.cuda.graph(gs[2], pool=pool):
                        self._phase_b2(out["box"])
                    with torch.cuda.graph(gs[3], pool=pool):
                        self._phase_c(ranges)
                out.update(a=gs[0], b1=gs[1], b2=gs[2], c=gs[3])
        self.kernel_launches_per_step = counter.count
        return out
