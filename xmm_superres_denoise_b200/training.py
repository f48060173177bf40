"""Plain-torch training loop for the RRDB path (what ``lightning.Trainer.fit`` + ``Model.training_step``
+ ``configure_optimizers`` do in the reference: train.py:148-165, models/model.py:51-86,239-247), with the
pieces the reference leaves to Lightning made explicit and B200-native:

* data parallel: one process per GPU, the batch is already sharded by the caller; gradients live in ONE
  flat fp32 buffer that is all-reduced with NCCL in chunks (one per RRDB, released as soon as that RRDB's
  weight gradients have been enqueued) on a side stream, overlapping the rest of the backward pass;
* optimizer: Adam on ONE flat fp32 parameter buffer (single kernel), after which the packed bf16
  tensor-core weight images are rebuilt by the engine's single repack launch on the next forward.

``TrainStep`` talks to the engine directly (no autograd graph); the autograd path
(``loss(model(x)).backward()``) stays available for Lightning / DDP users and is tested to give the same
gradients.
"""
from __future__ import annotations

import gc
import os
from typing import List, Optional, Tuple

import torch
from torch import nn

from . import _lib, determinism, ops


def flatten_parameters(module: nn.Module) -> torch.Tensor:
    """Re-point every parameter of `module` at a slice of one contiguous fp32 buffer (in place:
    Parameter objects, names and shapes are unchanged, so state_dict / optimizers / DDP keep working)."""
    params = list(module.parameters())
    if not params:
        raise ValueError("module has no parameters")
    dev = params[0].device
    if any(p.device != dev or p.dtype != torch.float32 for p in params):
        raise RuntimeError("flatten_parameters needs fp32 parameters on one device")
    flat = torch.empty(sum(p.numel() for p in params), dtype=torch.float32, device=dev)
    off = 0
    with torch.no_grad():
        for p in params:
            n = p.numel()
            view = flat[off:off + n].view(p.shape)
            view.copy_(p.data)
            p.data = view
            off += n
    return flat


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous shard [lo, hi) of n items for `rank` (inference shards images, no collective)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def allreduce_mean_(flat: torch.Tensor, group=None) -> torch.Tensor:
    """In-place mean all-reduce of a flat gradient buffer (NCCL on CUDA tensors, gloo on CPU tensors)."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat.div_(dist.get_world_size(group))
    return flat


class FusedAdam:
    """torch.optim.Adam semantics on a flat parameter buffer (one kernel per step)."""

    def __init__(self, flat_params: torch.Tensor, lr: float = 1e-4, betas=(0.9, 0.999), eps: float = 1e-8,
                 on_update=None) -> None:
        _lib.require_cuda_tensor(flat_params, torch.float32, "FusedAdam parameters")
        self.params = flat_params
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.exp_avg = torch.zeros_like(flat_params)
        self.exp_avg_sq = torch.zeros_like(flat_params)
        self.step_count = 0
        # the kernel writes through raw pointers, which no tensor version counter sees: the owner of packed
        # copies of these parameters (engine.WeightArena) must be told explicitly
        self.on_update = on_update

    def step(self, flat_grads: torch.Tensor, grad_scale: float = 1.0) -> None:
        _lib.require_cuda_tensor(flat_grads, torch.float32, "FusedAdam gradients")
        if flat_grads.numel() != self.params.numel():
            raise RuntimeError("gradient buffer size does not match the parameter buffer")
        self.step_count += 1
        _lib.check(_lib.load().xmm_adam_step(self.params.data_ptr(), flat_grads.data_ptr(), self.exp_avg.data_ptr(),
                                             self.exp_avg_sq.data_ptr(), self.params.numel(), self.lr, self.betas[0],
                                             self.betas[1], self.eps, self.step_count, grad_scale, _lib.stream_ptr()))
        ops._count()
        if self.on_update is not None:
            self.on_update()

    def state_dict(self):
        return {"step": self.step_count, "exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq, "lr": self.lr,
                "betas": self.betas, "eps": self.eps}

    def load_state_dict(self, sd) -> None:
        self.step_count = int(sd["step"])
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.lr = float(sd.get("lr", self.lr))
        self.betas = tuple(float(b) for b in sd.get("betas", self.betas))
        self.eps = float(sd.get("eps", self.eps))


class TrainStep:
    """forward + loss + backward + gradient all-reduce + Adam for one (lr, hr) batch."""

    def __init__(self, model: nn.Module, loss, lr: float = 1e-4, betas=(0.9, 0.999), group=None,
                 overlap_allreduce: bool = True, use_graph: Optional[bool] = None) -> None:
        """use_graph: replay forward + loss + backward (~800 launches, ~95 % GPU-busy when launched through Python) as
        ONE CUDA graph per input shape; Adam and the running loss state stay outside.  Off by default
        (XMM_TRAIN_GRAPH=1 enables): measured on B200 the eager step is already GPU-bound (362 vs 363 img/s, DN
        training, profiles/r01_bench_train_graph_ab.log); it pays with a slow host.  Single-process runs only: with a
        process group the NCCL chunks are issued eagerly."""
        import torch.distributed as dist

        self.model, self.loss, self.group = model, loss, group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.flat = flatten_parameters(model)
        if self.world > 1:
            # Lightning's DDP wrapper broadcasts rank 0's parameters when it wraps the module (train.py:148-155 of the
            # reference): replicas must START identical -- they may have been seeded per rank or loaded from a
            # checkpoint on one rank only -- because only gradients are exchanged afterwards.
            dist.broadcast(self.flat, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        self.engine = model._get_engine(train=True)
        self.engine.arena.invalidate()  # packed bf16 weight images follow the (possibly replaced) parameters
        self.opt = FusedAdam(self.flat, lr, betas, on_update=self.engine.arena.invalidate)
        # XMM_COMM_MODE (experiments): "overlap" (default: chunks released per RRDB on a side stream), "serial" (one
        # all-reduce after the backward pass), "none" (NO gradient exchange -- replicas diverge; only to measure what the
        # collective costs next to the spread between the GPUs of a box)
        self.comm_mode = os.environ.get("XMM_COMM_MODE", "overlap")
        if self.comm_mode not in ("overlap", "serial", "none"):
            raise ValueError(f"XMM_COMM_MODE={self.comm_mode!r}: expected overlap, serial or none")
        overlap_allreduce = overlap_allreduce and self.comm_mode == "overlap"
        self.overlap = overlap_allreduce and self.world > 1
        self.comm_stream = torch.cuda.Stream(device=self.flat.device) if self.overlap else None
        # SMs left to NCCL's kernels while the overlapped all-reduce chunks are in flight (XMM_COMM_SM_RESERVE; 0 = off,
        # the default): the conv / weight-gradient kernels are persistent grids of one CTA per SM whose work is divided
        # for that many CTAs, so CTAs a collective displaces would run as a second wave.  Measured on 8 x B200
        # (profiles/r02_scale_1_vs_8gpu_comm_knobs.log): reserve 0 / 4 / 8 and NCCL_MAX_CTAS 4 / 8 / 32 all give
        # 2622..2635 img/s (SR training) -- the 4 % the step loses at 8 GPUs is not SM contention -- so it stays off.
        self.sm_reserve = int(os.environ.get("XMM_COMM_SM_RESERVE", "0")) if self.overlap else 0
        self._works: List = []
        self._ones = torch.ones(1, dtype=torch.float32, device=self.flat.device)
        # chunk boundaries of the flat buffer: one chunk per RRDB (parameters are registered in module order)
        self._chunks = self._rrdb_chunks()
        if use_graph is None:
            use_graph = os.environ.get("XMM_TRAIN_GRAPH", "0") == "1"
        self.use_graph = bool(use_graph) and self.world == 1
        self._graph = None      # (key, CUDAGraph, static lr, static hr, loss state, flat gradient)
        self._seen_key = None   # shapes of the last eager step (the capture follows one eager step of that shape)

    def _rrdb_chunks(self):
        offs, off = {}, 0
        for name, p in self.model.named_parameters():
            offs[name] = (off, off + p.numel())
            off += p.numel()
        chunks = {}
        for i in range(self.model.num_res_blocks):
            names = [n for n in offs if n.startswith(f"rrdb.{i}.")]
            chunks[i] = (min(offs[n][0] for n in names), max(offs[n][1] for n in names))
        return chunks

    def _allreduce_range(self, flat_grad: torch.Tensor, lo: int, hi: int) -> None:
        import torch.distributed as dist

        if self.world == 1 or hi <= lo or self.comm_mode == "none":
            return
        if self.overlap:
            if self.sm_reserve > 0 and not self._works:
                _lib.load().xmm_set_sm_reserve(self.sm_reserve)
            self.comm_stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.comm_stream):
                self._works.append(dist.all_reduce(flat_grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group,
                                                   async_op=True))
        else:
            dist.all_reduce(flat_grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group)

    def _fwd_bwd(self, lr_img: torch.Tensor, hr_img: torch.Tensor):
        """forward + loss + backward (+ the gradient all-reduce chunks); returns (loss state, flat gradient)."""
        eng = self.engine
        out, bufs = eng.forward_train(lr_img)
        # Model.forward's second clamp (models/model.py:49) is the identity on an output already in [0,1]
        st = self.loss._evaluate(out, hr_img.contiguous().float())
        gout = self.loss._gradient(out, hr_img.contiguous().float(), st, self._ones)
        done = [len(self.flat)]  # upper end of the not-yet-reduced tail of the flat buffer

        def hook(rrdb_index: int, flat_grad: torch.Tensor) -> None:
            lo, _ = self._chunks[rrdb_index]
            self._allreduce_range(flat_grad, lo, done[0])  # this RRDB and everything after it not yet sent
            done[0] = lo

        _, _ = eng.backward(bufs, eng.generation, lr_img, gout, need_x_grad=False,
                            rrdb_done_hook=hook if self.overlap else None)
        flat_grad = eng.last_flat_grad
        self._allreduce_range(flat_grad, 0, done[0])
        for w in self._works:
            w.wait()
        if self._works and self.sm_reserve > 0:
            _lib.load().xmm_set_sm_reserve(0)
        self._works.clear()
        return st, flat_grad

    def __call__(self, lr_img: torch.Tensor, hr_img: torch.Tensor) -> torch.Tensor:
        # (the deterministic mode changes the backward's launches: a graph is captured per mode)
        key = (tuple(lr_img.shape), tuple(hr_img.shape), lr_img.dtype, hr_img.dtype, determinism.enabled())
        if self.use_graph and self._graph is not None and self._graph[0] == key:
            _, graph, s_lr, s_hr, st, flat_grad = self._graph
            s_lr.copy_(lr_img)
            s_hr.copy_(hr_img)
            graph.replay()
        elif self.use_graph and self._seen_key == key and not torch.cuda.is_current_stream_capturing():
            # second step of this shape: every lazily created buffer / tensor map / function attribute exists now
            s_lr, s_hr = lr_img.clone(), hr_img.clone()
            gc.collect()  # nothing may release device memory in mid-capture
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                st, flat_grad = self._fwd_bwd(s_lr, s_hr)
            self._graph = (key, graph, s_lr, s_hr, st, flat_grad)
            graph.replay()
        else:
            self._seen_key = key
            st, flat_grad = self._fwd_bwd(lr_img, hr_img)
        self.loss._merge(st)
        self.opt.step(flat_grad, 1.0 / self.world)
        return st["total"]
