"""Data-parallel wiring of the train_op (reference distributedExample/04, MultiWorkerMirroredStrategy).

The reference marks every accumulator ``aggregation=SUM`` (04:55), so ``assign_add`` all-reduces
every gradient tensor on EVERY micro-step over a gRPC ring (04:58,70,106), and pre-divides the loss
by ``num_workers`` (04:46).  Summation is linear, so here each rank accumulates locally and the
packed accumulator slab is exchanged ONCE per window, on the apply step, over NCCL / NVLink:

    accumulate steps : local kernel only, no communication
    apply step       : a += G (local)  ->  all-reduce(a)  ->  apply kernel without a gradient

Every rank then runs the identical deterministic apply on identical inputs, so replicas stay
bit-identical without an extra norm exchange.  The producer keeps 04's convention of dividing the
loss by ``num_workers``.  (04's second reduction inside ``apply_gradients`` -- SURVEY.md 5.8 -- is
not reproduced.)
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
import torch.distributed as dist


class DataParallelTrainOp:
    """Wraps an engine exposing accumulate_only / apply_only / run / accum / N / global_step."""
    launches_per_apply = 2      # local accumulate + apply (the all-reduce between them is NCCL's kernel)

    def __init__(self, engine, process_group=None):
        self.engine = engine
        self.group = process_group if process_group is not None and process_group is not True else None
        self.world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        self.allreduces = 0

    def state_dict(self):
        """Replicated moments are already complete on every rank; the rank-local accumulators are summed (04:55)."""
        e = self.engine
        if self.world == 1:
            return e.state_dict()
        acc = e.accum.clone()
        dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=self.group)
        saved, e.accum = e.accum, acc
        try:
            return e.state_dict()
        finally:
            e.accum = saved

    def load_state_dict(self, sd, strict: bool = True) -> None:
        self.engine.load_state_dict(sd, strict)
        if self.world > 1 and dist.get_rank(self.group) != 0:
            self.engine.accum.zero_()

    def run(self, grads: Sequence[Optional[torch.Tensor]]) -> bool:
        e = self.engine
        if self.world == 1:
            return e.run(grads)
        g = e.global_step
        if (g % e.N) != 0:                       # optimization.py:91 predicate, accumulate branch
            return e.run(grads)
        e.accumulate_only(grads)                 # 04:58
        dist.all_reduce(e.accum, op=dist.ReduceOp.SUM, group=self.group)   # 04:55, once per window
        self.allreduces += 1
        e.apply_only(None)                       # 04:59-66 on the summed accumulators
        e.global_step = g + 1                    # 04:74
        return True


class FusedDataParallelTrainOp:
    """The data-parallel train_op with the exchange INSIDE the apply kernel (csrc/gaccum_dp.cuh).

    Parameters are moved into one packed slab in NVLink peer-mapped symmetric memory (the tensors
    passed in are re-pointed at views of it, so the model keeps working unchanged); a staging area
    (W-1 shard-sized regions) and a 256-byte control block live there too.  PyTorch's symmetric-memory
    allocator is only the plumbing that maps every rank's buffers into every process -- the kernel does
    the reduce-scatter (peer stores into the owner's staging area), the norm exchange and the
    all-gather (peer stores into every parameter slab) itself, in ONE launch that also performs the
    window's last local ``a += G``.  Accumulate steps are rank-local: zero bytes cross NVLink until
    the apply step (vs one all-reduce per variable per micro-step in 04:55,58,70).

    m / v are sharded: each rank holds valid Adam moments only for the tiles it owns
    (``plan.dp_shard_range``); ``gather_state()`` rebuilds full copies for checkpoints.
    """
    launches_per_apply = 1

    def __init__(self, params: Sequence[torch.Tensor], names: Sequence[str], hp, accum_n: int, lr_fn,
                 process_group=None, exclude_from_weight_decay=("LayerNorm", "layer_norm", "bias"),
                 global_step: int = 0):
        import torch.distributed._symmetric_memory as symm
        from . import _lib
        from .train_op import GaccumTrainOp
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed must be initialised (backend nccl)")
        self.group = process_group if process_group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        if not (2 <= self.world <= _lib.MAX_RANKS):
            raise ValueError(f"fused data parallelism supports 2..{_lib.MAX_RANKS} ranks of one NVLink domain")
        dev = params[0].device
        layout = _lib.Plan([p.numel() for p in params], None, hp, device=-1)
        n = max(layout.padded_size, 32)
        stage_n = layout.dp_stage_elements(self.world)
        self.param_slab = symm.empty(n, dtype=torch.float32, device=dev)
        self.stage = symm.empty(stage_n, dtype=torch.float32, device=dev)
        self.ctrl = symm.empty(_lib.DP_CTRL_BYTES // 4, dtype=torch.int32, device=dev)
        self.param_slab.zero_(); self.stage.zero_(); self.ctrl.zero_()
        with torch.no_grad():
            for p, o in zip(params, layout.offsets):
                view = self.param_slab[o:o + p.numel()].view(p.shape)
                view.copy_(p)
                p.data = view                      # the caller's tensors now alias the packed slab
        gname = self.group.group_name
        self._handles = [symm.rendezvous(t, gname) for t in (self.param_slab, self.stage, self.ctrl)]
        hp_, hs_, hc_ = self._handles
        self.engine = GaccumTrainOp(list(params), names, hp, accum_n, lr_fn, exclude_from_weight_decay, global_step)
        self.plan = self.engine.plan
        self.comm = _lib.DpComm()
        self.comm.rank, self.comm.world = self.rank, self.world
        self.comm.accum = self.engine.accum.data_ptr()        # private: peers never touch the accumulators
        self.comm.stage_elements = stage_n
        for w in range(self.world):
            self.comm.param_peers[w] = int(hp_.buffer_ptrs[w])
            self.comm.stage_peers[w] = int(hs_.buffer_ptrs[w])
            self.comm.ctrl_peers[w] = int(hc_.buffer_ptrs[w])
        # own buffers through their ordinary local mapping, not the peer-aperture alias
        self.comm.param_peers[self.rank] = self.param_slab.data_ptr()
        self.comm.stage_peers[self.rank] = self.stage.data_ptr()
        self.comm.ctrl_peers[self.rank] = self.ctrl.data_ptr()
        self.tile_lo, self.tile_hi, self.owned_elements = self.plan.dp_shard_range(self.world, self.rank)
        self.epoch = 0
        self.exchanges = 0
        torch.cuda.synchronize(dev)
        dist.barrier(group=self.group)              # every rank's buffers are zeroed and mapped

    @property
    def global_step(self) -> int:
        return self.engine.global_step

    def run(self, grads: Sequence[Optional[torch.Tensor]]) -> bool:
        return self.run_bound(self.engine._grad_table(grads))

    def bind(self, grads):
        return self.engine.bind(grads)

    def run_bound(self, grad_table, stream: Optional[int] = None) -> bool:
        e = self.engine
        g = e.global_step
        if (g % e.N) != 0:
            return e.run_bound(grad_table, stream)            # rank-local accumulate (04:58 without the all-reduce)
        if stream is None:
            stream = torch.cuda.current_stream(e.device).cuda_stream
        from ._lib import StepArgs
        lr = e.lr_fn(g)
        self.epoch += 1
        e.plan.apply_dp(self.comm, grad_table, e._m_ptr, e._v_ptr,
                        StepArgs(g, e.N, 0, lr, e.beta1_power, e.beta2_power, 0.0), self.epoch, stream)
        self.exchanges += 1
        e._after(True, lr)
        return True

    # -- checkpoint compatibility under data parallelism (SURVEY.md 8(f) #3; reference 04:55 aggregation=SUM) --------
    def state_dict(self):
        """What the reference's Saver would hold: full adam_m / adam_v (every rank's owned shard gathered) and the
        SUM over ranks of the rank-local accumulators (04:55 declares them aggregation=SUM).  Collective: every rank
        must call it; every rank gets the same dictionary."""
        e = self.engine
        full = self.gather_state()
        acc = e.accum.clone()
        dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=self.group)
        saved = (e.m, e.v, e.accum)
        e.m, e.v, e.accum = full["m"], full["v"], acc
        try:
            return e.state_dict()
        finally:
            e.m, e.v, e.accum = saved

    def load_state_dict(self, sd, strict: bool = True) -> None:
        """Inverse of state_dict(): every rank takes parameters and the full moments (only its shard is ever used);
        the summed accumulators go to rank 0 alone, the others start the rest of the window from zero, so the next
        exchange reproduces the checkpointed sum."""
        e = self.engine
        e.load_state_dict(sd, strict)
        if self.rank != 0:
            e.accum.zero_()
        torch.cuda.synchronize(e.device)
        dist.barrier(group=self.group)

    def gather_state(self):
        """Full m and v slabs (every rank's owned range all-gathered) for checkpointing."""
        out = {}
        for name, slab in (("m", self.engine.m), ("v", self.engine.v)):
            full = slab.clone()
            for w in range(self.world):
                lo, hi, _ = self.plan.dp_shard_range(self.world, w)
                if hi <= lo:
                    continue
                a = self._tile_elem_offset(lo)
                b = self._tile_elem_offset(hi) if hi < self.plan.num_tiles else full.numel()
                dist.broadcast(full[a:b], src=dist.get_global_rank(self.group, w), group=self.group)
            out[name] = full
        return out

    def _tile_elem_offset(self, tile: int) -> int:
        """Slab element offset at which tile index `tile` starts (tiles are laid out tensor by tensor)."""
        t = 0
        for numel, off in zip(self.plan.numels, self.plan.offsets):
            nt = (numel + 2047) // 2048
            if tile < t + nt:
                return off + (tile - t) * 2048
            t += nt
        return self.engine.accum.numel()
