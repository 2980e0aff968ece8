"""Data-parallel plumbing for the U-Net hot path (one process per GPU, torch.distributed over NCCL/NVLink).

The reference is single-GPU (train.py:304 `device = "cuda:0"`); batch sharding is the path's natural partition:
each rank runs forward/backward on its own images, and only two things cross ranks
  (i)  BatchNorm statistics (SyncBN): the fp64 [sum, sum^2] (forward) and [sum da, sum da*xhat] (backward) vectors
       are all-reduced between the reduce and the apply kernels, so every rank normalises with global-batch
       statistics (torch.nn.SyncBatchNorm semantics);
  (ii) parameter gradients: written by backward straight into ONE flat fp32 buffer laid out in backward order and
       all-reduced (mean) bucket by bucket on a side stream while backward keeps running.
Works with the gloo backend on CPU tensors for the world_size-2 unit tests of the bucketing logic.
"""
from __future__ import annotations

import ctypes
import os
import warnings
import weakref

import torch
import torch.distributed as dist


def _ptr(t):
    return None if t is None else t.data_ptr()


class FlatGrads:
    def __init__(self, ctx: "DataParallelContext", params, flat=None):
        self.ctx = ctx
        self.params = list(params)
        self.offsets = {}
        total = 0
        for p in self.params:
            self.offsets[p] = total
            total += (p.numel() + 63) // 64 * 64  # keep every view 256-byte aligned
        dev = self.params[0].device
        # `flat`: the buffer of an earlier backward over the same parameters (every element that is read is rewritten by
        # each backward; the alignment padding was zeroed once) - no 124 MB allocation + memset per step
        self.flat = flat if flat is not None else torch.zeros(total, dtype=torch.float32, device=dev)
        self.total = total
        # buckets: contiguous ranges in backward order, closed when >= bucket_bytes
        self.buckets = []
        start, size = 0, 0
        limit = ctx.bucket_bytes // 4
        for p in self.params:
            size += (p.numel() + 63) // 64 * 64
            if size >= limit:
                self.buckets.append((start, start + size))
                start, size = start + size, 0
        if size:
            self.buckets.append((start, start + size))
        self.ready_upto = 0
        self.next_bucket = 0
        self.works = []
        self._pending = set(self.params)
        self._order = list(self.params)
        self._pos = 0

    def view_for(self, p):
        o = self.offsets[p]
        return self.flat[o:o + p.numel()].view(p.shape)

    def mark_ready(self, ps):
        for p in ps:
            self._pending.discard(p)
        # advance the contiguous ready prefix (parameters are produced in the declared order)
        while self._pos < len(self._order) and self._order[self._pos] not in self._pending:
            p = self._order[self._pos]
            self.ready_upto = self.offsets[p] + (p.numel() + 63) // 64 * 64
            self._pos += 1
        while self.next_bucket < len(self.buckets) and self.buckets[self.next_bucket][1] <= self.ready_upto:
            self._launch(self.buckets[self.next_bucket])
            self.next_bucket += 1

    def _launch(self, rng):
        self.ctx.all_reduce_mean_async(self.flat[rng[0]:rng[1]], self.works)

    def finish(self):
        while self.next_bucket < len(self.buckets):
            self._launch(self.buckets[self.next_bucket])
            self.next_bucket += 1
        self.ctx.wait_all(self.works)


class DataParallelContext:
    """Process-wide switch: `enable()` once after init_process_group; UNet picks it up in training mode."""

    _current = None

    def __init__(self, sync_bn=True, bucket_mb=25.0, group=None, graphs=None):
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed is not initialised")
        self.group = group
        self.world_size = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.sync_bn = sync_bn and self.world_size > 1
        self.bucket_bytes = int(bucket_mb * (1 << 20))
        self.comm_stream = torch.cuda.Stream() if torch.cuda.is_available() else None
        # graphs=True / B200UNET_DP_GRAPHS=1: net.enable_cuda_graphs() may replay the data-parallel step as CUDA graphs (the
        # NVLink SyncBN kernels and the NCCL gradient all-reduces are captured with the compute kernels). Opt-in: replay ==
        # eager launches bit for bit on 2 B200 (tests/dp_worker.py); measured on 8 B200: 5431 -> 5448 img/s device-resident,
        # 5272 -> 5347 img/s end to end. Graphs holding NCCL kernels must be dropped before destroy_process_group()
        # (DataParallelContext.disable()). Needs the NVLink SyncBN path (the NCCL fallback would put 36 tiny collectives
        # per step into the graph) - decided after _setup_nvl below.
        env = os.environ.get("B200UNET_DP_GRAPHS", "")
        self._want_graphs = (torch.cuda.is_available() and dist.get_backend() == "nccl"
                             and (env not in ("", "0") if env != "" else bool(graphs)))
        self.graph_capturable = False
        self._graph_owners = weakref.WeakSet()  # engines holding graphs captured under this context
        self._flat_cache = {}                   # parameter-id tuple -> flat gradient buffer of the last backward
        # NCCL averages in the collective itself (ReduceOp.AVG); gloo (CPU tests) sums and scales afterwards
        self._nccl = dist.get_backend(group) == "nccl"
        self.extra_wait_streams = []  # streams (besides the current one) whose work a gradient bucket depends on
        # SyncBN statistics over NVLink peer memory (csrc/nvl_sync.cu): symmetric buffer + peer pointer table
        self._nvl = None
        self._seq = 0
        if (self.sync_bn and torch.cuda.is_available() and group is None and self.world_size <= 8
                and dist.get_backend() == "nccl" and os.environ.get("B200UNET_NVL_SYNCBN", "1") not in ("", "0")):
            self._setup_nvl()
        self.graph_capturable = self._want_graphs and (self._nvl is not None or not self.sync_bn)

    def _setup_nvl(self):
        """Allocate the symmetric buffer and exchange peer pointers. Any failure (no P2P, older torch) leaves the NCCL
        path in place; the decision is made collectively so that all ranks take the same path."""
        ok = 1
        state = None
        try:
            import torch.distributed._symmetric_memory as symm_mem

            from . import _lib

            nbytes = int(_lib.query("b200unet_nvl_buffer_bytes"))
            buf = symm_mem.empty(nbytes, dtype=torch.uint8, device=torch.device("cuda", torch.cuda.current_device()))
            buf.zero_()
            hdl = symm_mem.rendezvous(buf, dist.group.WORLD)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            if len(ptrs) != self.world_size or any(p == 0 for p in ptrs):
                raise RuntimeError("symmetric memory rendezvous returned no peer pointers")
            state = (buf, hdl, (ctypes.c_void_p * self.world_size)(*ptrs))
        except Exception as e:  # noqa: BLE001
            ok = 0
            warnings.warn(f"NVLink SyncBN path unavailable ({type(e).__name__}: {e}); using NCCL all-reduce")
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        torch.cuda.synchronize()  # buffers are zeroed everywhere before any peer can write
        dist.barrier()
        if int(flag.item()) == 1:
            self._nvl = state
            from . import _lib

            # bound on the wait for a peer inside the SyncBN kernel: NCCL-like 10 minutes by default (rank-0-only
            # validation / checkpointing or a stalled data loader must not kill the job); 0 = wait forever
            tmo = float(os.environ.get("B200UNET_NVL_TIMEOUT_S", "600"))
            _lib.call("b200unet_nvl_set_timeout_ms", int(tmo * 1000))

    def check_health(self):
        """Host-side health check of the NVLink SyncBN path (one device->host read + one small all-gather; call it once
        per epoch or when a loss turns NaN). All ranks must issue the same sequence of training forwards/backwards
        (lockstep, as under torch DDP + SyncBatchNorm): raises if a reduction timed out on this rank (naming the ranks that
        never arrived) or if the ranks' reduction counters have diverged."""
        if self._nvl is None:
            return
        from . import _lib

        out = (ctypes.c_int64 * 3)()
        _lib.call("b200unet_nvl_status", ctypes.c_void_p(self._nvl[0].data_ptr()), torch.cuda.current_stream().cuda_stream, out)
        count, failed_seq, mask = int(out[0]), int(out[1]), int(out[2])
        t = torch.tensor([count, failed_seq], dtype=torch.int64, device="cuda")
        all_t = [torch.empty_like(t) for _ in range(self.world_size)]
        dist.all_gather(all_t, t, group=self.group)
        counts = [int(a[0]) for a in all_t]
        fails = [int(a[1]) for a in all_t]
        if failed_seq:
            missing = [r for r in range(self.world_size) if mask >> r & 1]
            raise RuntimeError(f"NVLink SyncBN reduction #{failed_seq} timed out on rank {self.rank}: ranks {missing} never "
                               "arrived (outputs were set to NaN); re-create the DataParallelContext to continue")
        if any(fails) or len(set(counts)) != 1:
            raise RuntimeError(f"NVLink SyncBN state diverged across ranks: reduction counters {counts}, failed reductions "
                               f"{fails} (every rank must run the same training forwards/backwards)")

    @property
    def has_nvl(self):
        return self._nvl is not None

    nvl_max_doubles = 2048  # slot size of the symmetric buffer (csrc/nvl_sync.cu SLOT_DOUBLES); longer vectors go through NCCL

    def bn_sync_finalize(self, sums, global_count, bn, eps, momentum, running_mean, running_var, mean, rstd, scale, shift):
        """All-reduce the fp64 [sum, sum^2] vector over NVLink and finalise BatchNorm in the same kernel (running buffers may
        be None: see ops.bn_train_buffers)."""
        from . import _lib

        c = bn.num_features
        # seq = 0: device-side reduction counter, so the launch can be captured in a CUDA graph and replayed
        _lib.call("b200unet_nvl_bn_sync_finalize", sums.data_ptr(), sums.data_ptr(), self._nvl[2], self.world_size,
                  self.rank, 0, float(global_count), bn.weight.data_ptr(), bn.bias.data_ptr(), float(eps),
                  float(momentum), _ptr(running_mean), _ptr(running_var), mean.data_ptr(), rstd.data_ptr(), scale.data_ptr(),
                  shift.data_ptr(), c, torch.cuda.current_stream().cuda_stream)

    def bn_rows_sync_finalize(self, stats_partial, rows, global_count, bn, eps, momentum, running_mean, running_var,
                              num_batches_tracked, mean, rstd, scale, shift):
        """Forward SyncBN in ONE kernel: reduce this rank's partial statistics rows, exchange them over NVLink, finalise
        BatchNorm (running statistics and num_batches_tracked included; None: not updated)."""
        from . import _lib

        _lib.call("b200unet_nvl_bn_rows_sync_finalize", stats_partial.data_ptr(), int(rows), bn.num_features, self._nvl[2],
                  self.world_size, self.rank, float(global_count), bn.weight.data_ptr(), bn.bias.data_ptr(), float(eps),
                  float(momentum), _ptr(running_mean), _ptr(running_var), _ptr(num_batches_tracked), mean.data_ptr(),
                  rstd.data_ptr(), scale.data_ptr(), shift.data_ptr(), torch.cuda.current_stream().cuda_stream)

    def rows_allreduce(self, partial, rows, c, sums_local, sums_global):
        """Backward SyncBN: block partials [rows][2][c] -> local and all-rank fp64 sums [2c], one kernel over NVLink."""
        from . import _lib

        _lib.call("b200unet_nvl_rows_allreduce", partial.data_ptr(), int(rows), int(c), self._nvl[2], self.world_size, self.rank,
                  sums_local.data_ptr(), sums_global.data_ptr(), torch.cuda.current_stream().cuda_stream)

    def supports_rows(self, c):
        return self._nvl is not None and c <= 2048 and os.environ.get("B200UNET_NVL_ROWS", "1") not in ("", "0")

    # ---- global registration
    @classmethod
    def enable(cls, **kw):
        cls._current = cls(**kw)
        return cls._current

    @classmethod
    def disable(cls):
        """Leave data-parallel mode. CUDA graphs that captured collectives are destroyed first: a live graph holding
        NCCL kernels makes `destroy_process_group()` wait forever (observed with torch 2.11 / NCCL 2.28), so call this
        before tearing the process group down."""
        cur = cls._current
        if cur is not None:
            for eng in list(cur._graph_owners):
                eng._graphs.clear()
            if torch.cuda.is_available():
                torch.cuda.synchronize()
        cls._current = None

    @classmethod
    def current(cls):
        c = cls._current
        if c is None or c.world_size == 1:
            return None
        return c

    # ---- collectives
    def all_reduce_sum(self, t):
        if (self._nvl is not None and t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
                and 0 < t.numel() <= 2048):
            from . import _lib

            _lib.call("b200unet_nvl_allreduce_f64", t.data_ptr(), t.data_ptr(), t.numel(), self._nvl[2], self.world_size,
                      self.rank, 0, torch.cuda.current_stream().cuda_stream)
            return
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)

    def make_flat_grads(self, params):
        """Flat gradient buffer for one backward. Outside CUDA-graph capture the buffer of the previous backward over the
        same parameters is reused once the optimizer has consumed it: the caller's .grad tensors are VIEWS of it, so it is
        only recycled when they have been released (zero_grad(set_to_none=True), torch's default) - otherwise a new one is
        allocated, exactly as before."""
        params = list(params)
        key = tuple(id(p) for p in params)
        flat = None
        capturing = params[0].is_cuda and torch.cuda.is_current_stream_capturing()
        if not capturing:
            old = self._flat_cache.get(key)
            if old is not None and all(p.grad is None or p.grad.untyped_storage().data_ptr() != old.untyped_storage().data_ptr()
                                       for p in params):
                flat = old
        fg = FlatGrads(self, params, flat)
        if not capturing:
            self._flat_cache[key] = fg.flat
        return fg

    def all_reduce_mean_async(self, t, works):
        if t.is_cuda:
            # run the collective on a side stream so the backward kernels that follow keep the SMs busy
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            with torch.cuda.stream(self.comm_stream):
                self.comm_stream.wait_event(ev)
                for st in self.extra_wait_streams:
                    self.comm_stream.wait_stream(st)
                if self._nccl:
                    dist.all_reduce(t, op=dist.ReduceOp.AVG, group=self.group)  # one pass: no separate 1/world scaling
                else:
                    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
                    t.mul_(1.0 / self.world_size)
            works.append(None)
        else:
            w = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            works.append((w, t))

    def wait_all(self, works):
        if self.comm_stream is not None and any(w is None for w in works):
            torch.cuda.current_stream().wait_stream(self.comm_stream)
        for w in works:
            if w is not None:
                w[0].wait()
                w[1].mul_(1.0 / self.world_size)
        works.clear()


def init_from_env(sync_bn=True, bucket_mb=25.0, graphs=None):
    """torchrun-style bring-up: RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* from the environment."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:
        return None
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
        backend = "nccl"
        # Measured on 2 x B200 (scripts/gpu_scale.sh): NCCL's default CTA count next to full-width persistent grids is
        # fastest (23.99 ms/step vs 24.28-24.43 with NCCL_MAX_CTAS=4/8 or with 4/8 SMs kept free of the persistent
        # conv grids), so neither is done.
    else:
        backend = "gloo"
    if not dist.is_initialized():
        kw = {"device_id": torch.device("cuda", local)} if backend == "nccl" else {}
        dist.init_process_group(backend=backend, **kw)
    return DataParallelContext.enable(sync_bn=sync_bn, bucket_mb=bucket_mb, graphs=graphs)
