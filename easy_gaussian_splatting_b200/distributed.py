"""View-sharded multi-GPU training step (new capability named by BASELINE.json north_star; the
reference itself is single-GPU, SURVEY.md §2.2 / §8e).

Every rank holds a full replica of the Gaussian parameters, renders its own share of the step's
camera views, and then two collectives make the replicas agree again:

* parameter gradients: one SUM all-reduce over a single flat bucket (59 floats = 236 B per
  Gaussian).  The bucket is the storage of every ``param.grad``, so autograd accumulates straight
  into it and no pack / unpack copy exists;
* densification statistics (/root/reference/model/gaussian.py:56-64,188-197): SUM for
  ``grad_norm_accum`` and ``collecting_counts``, MAX for ``max_radii`` (12 B per Gaussian).  Each
  rank applies the per-view update for its own views to a per-step DELTA (``stages.densify_stats_update``
  on three zeroed rows), the deltas are reduced, and every rank folds the reduced delta into its persistent
  statistics — which equals what one GPU would have accumulated over all views.  When the statistics are
  attached to the gradient bucket (``DensifyStats(n, device, bucket=bucket)``) the delta rows live in the
  same symmetric buffer behind the gradients and travel in the SAME kernel launch (SUM rows with the
  gradients, the MAX row through the kernel's max tail): no NCCL call, no clone, no subtraction.

Works with any torch.distributed backend (NCCL over NVLink on the B200 box, gloo in CPU tests).
"""
from __future__ import annotations

import contextlib
import os
from typing import Dict, Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist
from torch import Tensor


def shard_views(n_views: int, rank: int, world_size: int) -> List[int]:
    """Round-robin view partition: rank r renders {v : v mod R == r} (SURVEY.md §8e)."""
    return [v for v in range(n_views) if v % world_size == rank]


class FlatGradBucket:
    """One contiguous fp32 buffer that backs ``.grad`` of every parameter.

    On CUDA with more than one rank the buffer is allocated in SYMMETRIC memory (every rank's bucket mapped into
    every peer over NVLink) and ``all_reduce()`` runs our own kernels instead of NCCL (csrc/collective.cu): a two-shot
    peer load / peer store all-reduce on 2 GPUs (0.36 ms against NCCL's 0.47 ms for the 236 MB bucket of 1 M
    Gaussians), the in-switch multimem.ld_reduce / multimem.st exchange on more (8 GPUs: 0.59 against 0.63 ms);
    both deliver bit-identical sums to every replica.  A self-check against NCCL at construction, agreed on by all
    ranks, falls back to ``dist.all_reduce`` if symmetric memory is unavailable or the check fails
    (EGS_PEER_ALLREDUCE=0 forces the fallback)."""

    def __init__(self, params: Sequence[Tensor], symmetric: Optional[bool] = None, stats_size: int = 0):
        """``stats_size`` = N reserves three more rows of N floats behind the gradients for the per-step densify-stat
        deltas (two SUM rows, one MAX row) so that they ride in the gradient exchange; see ``DensifyStats``."""
        self.params = list(params)
        # every parameter's slice starts on a 16-byte boundary (4 floats): the fused backward stores float4s into
        # it, and N is arbitrary after the first densify / prune
        total = sum(-(-p.numel() // 4) * 4 for p in self.params)
        ref = self.params[0]
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.grad_floats = -(-total // (4 * max(world, 1))) * (4 * max(world, 1))  # whole float4s per rank slice
        self.stats_size = int(stats_size)
        self.stats_row = -(-self.stats_size // 4) * 4  # each row starts on a 16-byte boundary
        self.n_sum_floats = self.grad_floats + 2 * self.stats_row
        self.n_max_floats = self.stats_row
        padded = self.n_sum_floats + self.n_max_floats
        self.epoch = 0  # number of completed exchanges
        self._symm = None
        self._mode = "nccl"
        if symmetric is None:
            symmetric = os.environ.get("EGS_PEER_ALLREDUCE", "1") != "0"
        # peer memory only makes sense (and its rendezvous only works) with an initialised group of > 1 CUDA ranks
        symmetric = bool(symmetric) and ref.is_cuda and world > 1
        self.flat = self._symmetric_buffer(padded, ref, world) if symmetric else None
        if self.flat is None:
            self.flat = torch.zeros(padded, dtype=ref.dtype, device=ref.device)
        off = 0
        self.views = []
        for p in self.params:
            v = self.flat[off:off + p.numel()].view_as(p)
            p.grad = v
            self.views.append(v)
            off += -(-p.numel() // 4) * 4

    def _symmetric_buffer(self, n: int, ref: Tensor, world: int) -> Optional[Tensor]:
        buf, ok = None, 0
        try:
            import torch.distributed._symmetric_memory as symm_mem
            group = dist.group.WORLD
            if hasattr(symm_mem, "enable_symm_mem_for_group"):
                import warnings
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    try:
                        symm_mem.enable_symm_mem_for_group(group.group_name)
                    except Exception:
                        pass
            buf = symm_mem.empty(n, dtype=torch.float32, device=ref.device)
            hdl = symm_mem.rendezvous(buf, group.group_name)
            mode = "two_shot" if world == 2 else ("multimem" if getattr(hdl, "multicast_ptr", 0) else None)
            if mode is not None and ref.dtype == torch.float32:
                self._symm, self._mode = hdl, mode
                # self-check: rank r contributes (r + 1) * pattern; every rank must read back the NCCL sum
                pattern = torch.arange(n, dtype=torch.float32, device=ref.device).remainder_(977.0).add_(1.0)
                buf.copy_(pattern * float(dist.get_rank() + 1))
                expect = buf.clone()
                dist.all_reduce(expect[:self.n_sum_floats])
                if self.n_max_floats:
                    dist.all_reduce(expect[self.n_sum_floats:], op=dist.ReduceOp.MAX)
                self._peer_all_reduce(buf)
                ok = int(torch.equal(buf, expect))
        except Exception:
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=ref.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)  # every rank takes the same route
        if int(flag.item()) != 1:
            self._symm, self._mode = None, "nccl"
            return None
        buf.zero_()
        return buf

    def _peer_all_reduce(self, buf: Tensor) -> None:
        import ctypes
        from . import _lib
        hdl, world, rank = self._symm, dist.get_world_size(), dist.get_rank()
        st = ctypes.c_void_p(torch.cuda.current_stream(buf.device).cuda_stream)
        hdl.barrier(channel=0)  # every bucket is complete
        lib = _lib.load()
        if self._mode == "two_shot":
            rc = lib.egs_allreduce_f32_peer(world, rank, ctypes.c_void_p(hdl.buffer_ptrs_dev), self.n_sum_floats,
                                            self.n_max_floats, st)
        else:
            rc = lib.egs_allreduce_f32_multimem(world, rank, ctypes.c_void_p(hdl.multicast_ptr), self.n_sum_floats,
                                                self.n_max_floats, st)
        _lib.check(rc, "egs_allreduce_f32")
        hdl.barrier(channel=1)  # every slice has landed everywhere

    @property
    def exchange(self) -> str:
        return {"nccl": "NCCL all-reduce", "two_shot": "hand-written two-shot all-reduce over NVLink peer memory",
                "multimem": "hand-written NVLS (multimem.ld_reduce / multimem.st) all-reduce"}[self._mode]

    @property
    def stats_delta(self) -> Optional[Tensor]:
        """[3, stats_size] view of the statistics rows behind the gradients (SUM, SUM, MAX), or None."""
        if not self.stats_size:
            return None
        return self.flat[self.grad_floats:].view(3, self.stats_row)[:, :self.stats_size]

    def zero_(self) -> None:
        self.flat[:self.grad_floats].zero_()
        for p, v in zip(self.params, self.views):  # an optimizer may have detached .grad
            if p.grad is None or p.grad.data_ptr() != v.data_ptr():
                p.grad = v

    def begin_direct(self) -> None:
        """For a step with ONE backward pass (all of the step's views in one ``rasterization()`` call): every
        parameter's bucket slice is registered as the one-shot gradient target of that parameter, so the fused
        projection backward, which writes every gradient element exactly once, stores straight into the bucket — no
        zero fill before and no accumulate pass after the backward (2 x 236 B/Gaussian of traffic less).  Call
        ``end_direct()`` after ``backward()``."""
        from . import stages
        for p, v in zip(self.params, self.views):
            p.grad = None
            stages.register_grad_target(p, v)

    def end_direct(self) -> None:
        from . import stages
        stages.clear_grad_targets()
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                v.zero_()
            elif p.grad.data_ptr() != v.data_ptr():  # the gradient took another route (e.g. torch ops in front)
                v.copy_(p.grad)
            p.grad = v

    @contextlib.contextmanager
    def direct(self):
        """``with bucket.direct(): loss.backward()`` — begin_direct / end_direct with the registration always removed."""
        self.begin_direct()
        try:
            yield self
        finally:
            self.end_direct()

    def all_reduce(self, group=None, async_op: bool = False):
        """SUM all-reduce of the whole bucket.  Returns ``None`` (``async_op=False``) or a work handle with ``wait()``
        and ``is_completed()``.  The peer-memory kernels are stream ordered like every other kernel of the step, so
        in that mode the handle is already complete; a non-default ``group`` cannot use the WORLD rendezvous of the
        symmetric buffer and is refused rather than silently rerouted."""
        if self._symm is not None:
            if group is not None and group is not dist.group.WORLD:
                raise ValueError("the symmetric-memory bucket was rendezvoused on the WORLD group; build the bucket with "
                                 "symmetric=False to all-reduce over another group")
            self._peer_all_reduce(self.flat)
            self.epoch += 1
            return _CompletedWork() if async_op else None
        self.epoch += 1
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            if self.n_max_floats:  # the MAX row cannot share a SUM collective: reduce it first, synchronously
                dist.all_reduce(self.flat[self.n_sum_floats:], op=dist.ReduceOp.MAX, group=group)
            return dist.all_reduce(self.flat[:self.n_sum_floats], op=dist.ReduceOp.SUM, group=group, async_op=async_op)
        return _CompletedWork() if async_op else None

    @property
    def nbytes(self) -> int:
        return self.flat.numel() * self.flat.element_size()


class _CompletedWork:
    """Stand-in for a torch.distributed work handle when the exchange was stream ordered (or there was nothing to
    exchange): ``wait()`` returns immediately."""

    def wait(self, timeout=None) -> bool:
        return True

    def is_completed(self) -> bool:
        return True


class DensifyStats:
    """``grad_norm_accum`` / ``collecting_counts`` / ``max_radii`` with the reference's semantics
    (/root/reference/model/gaussian.py:56-64, 188-197), kept as the three rows of one ``[3, N]`` buffer.

    One process: ``update_local`` applies every view's contribution to the persistent rows directly.
    View-sharded (``distributed=True``, the default whenever a process group with more than one rank exists): the
    views of a step go to a per-step DELTA — ``begin_step()`` clears it, ``update_local`` accumulates into it,
    ``all_reduce()`` reduces it over the ranks (SUM, SUM, MAX) and folds it into the persistent rows.  With
    ``bucket=`` (a ``FlatGradBucket`` built with ``stats_size=N``) the delta rows ARE the tail of the gradient bucket
    and have already been reduced by ``bucket.all_reduce()`` — call that first; ``all_reduce()`` here then only folds."""

    def __init__(self, n: int, device, bucket: Optional["FlatGradBucket"] = None, distributed: Optional[bool] = None):
        self.buf = torch.zeros(3, n, dtype=torch.float32, device=device)
        if distributed is None:
            distributed = bucket is not None or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1)
        self.bucket = bucket
        self.delta: Optional[Tensor] = None
        self._epoch = 0
        if bucket is not None:
            if bucket.stats_size != n:
                raise ValueError(f"the bucket reserves {bucket.stats_size} statistics slots, need {n}")
            self.delta = bucket.stats_delta
        elif distributed:
            self.delta = torch.zeros(3, n, dtype=torch.float32, device=device)

    @property
    def grad_norm_accum(self) -> Tensor:
        return self.buf[0]

    @property
    def collecting_counts(self) -> Tensor:
        return self.buf[1]

    @property
    def max_radii(self) -> Tensor:
        return self.buf[2]

    @property
    def step_buf(self) -> Tensor:
        """Where the views of the current step accumulate: the delta rows when view-sharded, else the persistent rows."""
        return self.buf if self.delta is None else self.delta

    @property
    def exchange(self) -> str:
        if self.delta is None:
            return "none (one process)"
        if self.bucket is not None:
            return "rides in the gradient exchange (SUM rows + MAX row of the same launch)"
        return "NCCL all-reduce (SUM of the two accumulator deltas, MAX of the max_radii delta)"

    def begin_step(self) -> None:
        if self.delta is not None:
            self.delta.zero_()
            if self.bucket is not None:
                self._epoch = self.bucket.epoch

    def update_local(self, radii: Tensor, absgrad: Tensor, width: int, height: int) -> None:
        """Per-view update for the views this rank rendered (CUDA kernel; no host sync)."""
        from . import stages
        t = self.step_buf
        stages.densify_stats_update(t[2], t[0], t[1], radii, absgrad, width, height)

    def all_reduce(self, group=None) -> None:
        if self.delta is None:
            return
        if self.bucket is not None:
            if self.bucket.epoch == self._epoch:
                raise RuntimeError("statistics attached to a gradient bucket are reduced by bucket.all_reduce(): call it "
                                   "before DensifyStats.all_reduce()")
        elif dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(self.delta[:2], op=dist.ReduceOp.SUM, group=group)
            mr = self.delta[2].contiguous()
            dist.all_reduce(mr, op=dist.ReduceOp.MAX, group=group)
            self.delta[2].copy_(mr)
        self.buf[:2] += self.delta[:2]
        torch.maximum(self.buf[2], self.delta[2], out=self.buf[2])
