"""Multi-GPU plumbing for the sharded sample stream (SURVEY.md section 8e).

The stream shards with no data-path exchange: rank r ingests the contiguous
index range shard_range(r, world, n_total) into its own bucket arrays.  The
only collective is one sum all-reduce of the frozen uint64 bucket (and counter)
arrays per snapshot, issued through torch.distributed (NCCL over NVLink on
GPUs, gloo in the CPU tests).  Integer sums are associative, so the reduced
counts are bit-identical to a single-GPU run over the whole stream; uint64
addition and int64 addition produce the same bits, which is why an int64 view
is what gets reduced.
"""
from __future__ import annotations


def shard_range(rank: int, world: int, n_total: int) -> tuple[int, int]:
    """[start, stop) of rank's contiguous slice; the first n_total % world ranks take one extra sample."""
    base, extra = divmod(n_total, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def allreduce_sum_u64(t, group=None):
    """In-place sum all-reduce of a tensor holding uint64 bit patterns (dtype int64 or uint64 view)."""
    import torch
    import torch.distributed as dist
    if t.dtype == torch.uint64:
        t = t.view(torch.int64)
    assert t.dtype == torch.int64
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


class _CudaView:
    """Zero-copy __cuda_array_interface__ wrapper over a raw device pointer."""

    def __init__(self, ptr: int, words: int):
        self.__cuda_array_interface__ = {"shape": (words,), "typestr": "<i8", "data": (ptr, False), "version": 3}


class ShardedEngine:
    """An Engine per rank plus the snapshot-time all-reduce.

    snapshot() = lh_snapshot_begin -> all-reduce of the frozen device arrays on the snapshot stream ->
    lh_snapshot_reduce (+ export) -> lh_snapshot_end, so every rank ends with the global percentiles.
    snapshot_async()/result() is the pipelined form: everything is only enqueued (the snapshot stream
    outranks the ingest stream), the caller launches the next interval's ingest, then collects the result.

    collective:
      "peer"  the library's own peer-memory all-reduce kernel behind the C ABI (lh_comm_* /
              lh_snapshot_allreduce): every rank sums the live window of all peers' frozen arrays over NVLink
              in one small kernel; torch.distributed only carries the 512-byte peer handles at start-up;
      "nccl"  torch.distributed all_reduce (NCCL on GPUs, gloo in the CPU tests) of the dense arrays;
      "none"  single rank.
    """

    def __init__(self, engine, device_index: int, group=None, collective: str = "nccl"):
        import torch.distributed as dist
        self.engine = engine
        self.device_index = device_index
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.collective = collective if self.world > 1 else "none"
        self._views = {}     # device pointer -> cached zero-copy tensor
        self._ext = None
        self._bytes = 0
        self.fallback_reason = None
        if self.collective == "peer":
            self._init_peer(dist)

    def _init_peer(self, dist):
        """Exchange the opaque peer handles (lh_comm_export) with an all_gather and hand them to lh_comm_import."""
        import torch
        eng = self.engine
        mine = eng.comm_export()                                   # bytes
        rank = dist.get_rank(self.group)
        t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).to("cuda:%d" % self.device_index)
        out = [torch.empty_like(t) for _ in range(self.world)]
        dist.all_gather(out, t, group=self.group)
        err = ""
        try:
            eng.comm_import(rank, self.world, b"".join(bytes(o.cpu().numpy().tobytes()) for o in out))
        except Exception as e:                                     # e.g. no peer access / CUDA IPC between two of the devices
            err = str(e)
        # every rank has mapped every peer -- or ALL ranks fall back to NCCL together (a rank must never wait in the
        # peer kernel for a rank that is not going to launch it)
        ok = torch.tensor([0 if err else 1], dtype=torch.int32, device="cuda:%d" % self.device_index)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
        if int(ok.item()) == 0:
            self.collective = "nccl"
            self.fallback_reason = err or "a peer rank could not map this rank's memory"

    def _tensor(self, ptr: int, words: int):
        import torch
        t = self._views.get(ptr)
        if t is None or t.numel() != words:
            t = torch.as_tensor(_CudaView(ptr, words), device="cuda:%d" % self.device_index)
            self._views[ptr] = t
        return t

    def _tensor32(self, ptr: int, words: int):
        import torch
        key = ("i32", ptr)
        t = self._views.get(key)
        if t is None or t.numel() != words:
            view = _CudaView(ptr, words)
            view.__cuda_array_interface__["typestr"] = "<i4"
            t = torch.as_tensor(view, device="cuda:%d" % self.device_index)
            self._views[key] = t
        return t

    def _allreduce_frozen(self, counters: bool):
        """Enqueue the collective for the open snapshot; returns what allreduce_ms() needs to time it."""
        eng = self.engine
        if self.collective == "peer":
            seq = eng.snapshot_allreduce(counters)
            return ("peer", seq)
        import torch
        v = eng.snapshot_device()
        if self._ext is None or self._ext.cuda_stream != int(v.stream):
            self._ext = torch.cuda.ExternalStream(int(v.stream), device=self.device_index)
        ext = self._ext
        self._bytes = int(v.n_bucket_words) * 8 + (int(v.n_counter_words) * 8 if counters else 0)
        with torch.cuda.stream(ext):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            allreduce_sum_u64(self._tensor(int(v.d_buckets), int(v.n_bucket_words)), self.group)
            # the per-histogram flags (0 / 1 / 3) tell the reduction kernels what to scan: OR over ranks == MAX
            import torch.distributed as dist
            dist.all_reduce(self._tensor32(int(v.d_flags), int(v.n_flag_words)), op=dist.ReduceOp.MAX, group=self.group)
            if counters:
                allreduce_sum_u64(self._tensor(int(v.d_counters), int(v.n_counter_words)), self.group)
            e1.record(ext)
        return ("nccl", (e0, e1))

    def snapshot(self, percentiles, export: bool = False, counters: bool = False, window: bool = False):
        """window=True also folds the (all-reduced) snapshot into the engine's window (Engine.window_configure)."""
        eng = self.engine
        eng.snapshot_begin()
        try:
            if self.world > 1:
                self._allreduce_frozen(counters)
            if window:
                eng.window_fold()
            red = eng.snapshot_reduce(percentiles)
            sp = eng.snapshot_export() if export else None
        finally:
            eng.snapshot_end()
        return red, sp

    def snapshot_async(self, percentiles, counters: bool = False, after_swap=None, window: bool = False):
        """begin + all-reduce + reduce + end, all enqueued; returns a handle for result() / allreduce_ms().

        `after_swap` (optional callable) runs right after the buffer swap and before the collective is issued:
        pipelined callers launch the next interval's ingest there, so that it is already queued on the device
        should the collective's host call take time.  window=True folds the snapshot into the engine's window
        after the collective (one snapshot-stream synchronisation)."""
        eng = self.engine
        eng.snapshot_begin()
        ar = None
        try:
            if after_swap is not None:
                after_swap()
            if self.world > 1:
                ar = self._allreduce_frozen(counters)
            if window:
                eng.window_fold()
            h = eng.snapshot_reduce_async(percentiles)
        finally:
            eng.snapshot_end()
        return (h, ar)

    def result(self, handle):
        return self.engine.snapshot_result(handle[0])

    def allreduce_ms(self, handle) -> float:
        """Device time of THIS snapshot's collective (CUDA events around it on the snapshot stream)."""
        ar = handle[1]
        if ar is None:
            return 0.0
        if ar[0] == "peer":
            return self.engine.comm_allreduce_ms(ar[1])
        e0, e1 = ar[1]
        e1.synchronize()
        return float(e0.elapsed_time(e1))

    def allreduce_bytes(self) -> int:
        """Bytes one rank's collective moves per snapshot (dense arrays for nccl; window bytes read from peers)."""
        if self.collective == "peer":
            return self.engine.comm_last_bytes()
        return self._bytes
