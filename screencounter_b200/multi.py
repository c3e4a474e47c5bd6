"""Multi-GPU plumbing: one process per GPU, reads sharded by contiguous range, results combined in ONE exchange step
(SURVEY.md 8.2 row e).  torch.distributed carries the bytes (NCCL over NVLink on the GPUs); the merging itself runs in
this library's kernels.

The reference merges per-thread results in `reduce()` -- a vector add for the dense counters
(handlers/SingleBarcodeSingleEnd.hpp:119-125, handlers/DualBarcodesPairedEnd.hpp:202-208), an append + sort for
combinations (handlers/CombinatorialBarcodesSingleEnd.hpp:268-305), a map merge for random barcodes
(handlers/RandomBarcodeSingleEnd.hpp:197-207).  Across GPUs the same merges are:

  dense outputs    one all-reduce (sum) of the count vector / count matrix, on the device;
  sparse outputs   every GPU sort-reduces its own table on the device (radix sort of the live hash entries), the key space
                   is cut into `world` ranges at splitters taken from rank 0's table (the shards are random samples of one
                   library, so the cut is balanced), one all-to-all moves every range to its owner, the owner merges the
                   `world` sorted runs it received with the merge kernels of runners_random.cu (binary-search ranks, counts
                   of equal keys added), and rank 0 gathers the ranges in rank order -- the concatenation is the sorted table
                   of the whole file.

Results do not depend on how reads are split (SURVEY.md 8.1 T24).  Nothing here computes on the host: without a CUDA
device the sparse path fails loudly; the CPU tests (gloo, world size 2) inject the table operations."""
import ctypes as C

import numpy as np


def shard_range(n, rank, world):
    """Contiguous range [first, first + count) of `n` reads (pairs) owned by `rank` of `world`."""
    first = (n * rank) // world
    last = (n * (rank + 1)) // world
    return first, last - first


def _dist():
    import torch.distributed as dist
    return dist


def _device_for(group=None):
    import torch
    dist = _dist()
    backend = dist.get_backend(group)
    if "nccl" in str(backend):
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def combine_dense(counts, scalars=(), group=None):
    """Sum `counts` (int32 vector) and the integer `scalars` (total, barcode1_only, ...) over all
    ranks with a single all-reduce of one packed buffer.  Returns (counts, [scalars...]).

    `counts` may be a numpy array or a torch tensor (a CUDA tensor stays on the device and the
    all-reduce runs over NCCL); the scalars ride in the same buffer so there is exactly one
    collective per call."""
    import torch
    dist = _dist()
    scalars = [int(s) for s in scalars]
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return counts, scalars
    dev = _device_for(group)
    is_tensor = isinstance(counts, torch.Tensor)
    body = counts.to(device=dev, dtype=torch.int64) if is_tensor else torch.from_numpy(np.asarray(counts, dtype=np.int64)).to(dev)
    # int64 on the wire: per-rank int32 counters cannot overflow the sum of up to 8 ranks
    packed = torch.cat([body.reshape(-1), torch.tensor(scalars, dtype=torch.int64, device=dev)])
    dist.all_reduce(packed, op=dist.ReduceOp.SUM, group=group)
    n = body.numel()
    if int(packed.max().item()) > np.iinfo(np.int32).max:
        raise OverflowError("combined count exceeds the reference's 32-bit counters (SURVEY.md 8.1 T17)")
    out_scalars = [int(v) for v in packed[n:].tolist()]
    if is_tensor:
        return packed[:n].to(dtype=torch.int32).reshape(counts.shape), out_scalars
    return packed[:n].cpu().numpy().astype(np.int32).reshape(np.asarray(counts).shape), out_scalars


# ---------------------------------------------------------------------------------------------------------------------
# sorted (key, count) tables on the device
# ---------------------------------------------------------------------------------------------------------------------
class _DevView:
    """Zero-copy torch view of device memory this library owns (CUDA array interface)."""

    def __init__(self, ptr, shape, typestr):
        shape = (int(shape),) if isinstance(shape, (int, np.integer)) else tuple(int(d) for d in shape)
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (int(ptr), False), "version": 2}


class DeviceTableOps:
    """The table operations of the sparse exchange, on the device through the C ABI (include/scg.h scg_table_*)."""

    def __init__(self, device=None):
        from .rcpp import context, default_device
        self.ctx = context(device)
        if device is None:
            device = default_device()
        # the device the context's tables live on: the first of a multi-device context
        self.device = int(device[0] if isinstance(device, (list, tuple)) else device)

    def from_plan(self, plan):
        from ._lib import lib
        from .rcpp import _check
        h = C.c_void_p()
        _check(plan.ctx, lib().scg_plan_sorted_table(plan.handle, C.byref(h)))
        return h

    def views(self, table):
        """(keys int64 of shape (rows, words), counts int32) torch views of a table's device arrays.  A row's words are in
        the order they sort by (include/scg.h scg_table_keys); every word is below 2^63."""
        import torch
        from ._lib import lib
        n = int(lib().scg_table_rows(table))
        words = int(lib().scg_table_key_words(table))
        if n == 0:
            dev = torch.device("cuda", self.device)
            return torch.empty((0, words), dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.int32, device=dev)
        keys = torch.as_tensor(_DevView(lib().scg_table_keys(table), (n, words), "<i8"), device="cuda")
        counts = torch.as_tensor(_DevView(lib().scg_table_counts(table), n, "<i4"), device="cuda")
        return keys, counts

    def key_len(self, table):
        from ._lib import lib
        return int(lib().scg_table_key_len(table))

    def from_tensors(self, keys, counts, key_len):
        """A table copied from `keys` (int64, (rows, words), or (rows,) when a row has one word) and `counts` (int32, (rows,)),
        both on this context's device.  The library refuses rows that are not a sorted table (include/scg.h)."""
        import torch
        from ._lib import lib
        from .rcpp import _check
        dev = torch.device("cuda", self.device)
        words = 2 if int(key_len) > 21 else 1
        if not isinstance(keys, torch.Tensor) or keys.dtype != torch.int64 or keys.device != dev:
            raise ValueError("table keys must be an int64 tensor on %s" % dev)
        if not isinstance(counts, torch.Tensor) or counts.dtype != torch.int32 or counts.device != dev:
            raise ValueError("table counts must be an int32 tensor on %s" % dev)
        if not (keys.dim() == 2 and keys.shape[1] == words or keys.dim() == 1 and words == 1):
            raise ValueError("table keys of key length %d must have shape (rows, %d)%s, not %s"
                             % (key_len, words, " or (rows,)" if words == 1 else "", tuple(keys.shape)))
        rows = keys.shape[0]
        if counts.dim() != 1 or counts.shape[0] != rows:
            raise ValueError("table counts must have shape (%d,), not %s" % (rows, tuple(counts.shape)))
        keys, counts = keys.contiguous(), counts.contiguous()
        torch.cuda.current_stream(dev).synchronize()   # the tensors were produced on torch's stream, the copy runs on the library's
        h = C.c_void_p()
        _check(self.ctx, lib().scg_table_from_device(self.ctx, C.c_void_p(keys.data_ptr()), C.c_void_p(counts.data_ptr()),
                                                     C.c_longlong(keys.shape[0]), int(key_len), C.byref(h)))
        return h

    def merge(self, a, b):
        from ._lib import lib
        from .rcpp import _check
        h = C.c_void_p()
        _check(self.ctx, lib().scg_table_merge(self.ctx, a, b, C.byref(h)))
        return h

    def free(self, table):
        from ._lib import lib
        if table:
            lib().scg_table_free(table)

    def render(self, table):
        """The table as the file-level call returns it: (int32 rows x 2, freq) for combinations, (S<len> array, freq) for barcodes."""
        from ._lib import lib
        from .rcpp import _check, _table
        h = C.c_void_p()
        _check(self.ctx, lib().scg_table_render(self.ctx, table, C.byref(h)))
        try:
            return _table(h, "random_array" if self.key_len(table) > 0 else "combo")
        finally:
            lib().scg_result_free(h)


def _cut(keys, splitters):
    """Rows of the sorted table `keys` that sort before each splitter row.  Keys of two words per row (random barcodes longer
    than 21 bases) compare lexicographically: word 0 locates the run of rows that share the splitter's word 0, word 1 the
    place inside that run."""
    import torch
    if keys.dim() == 1:
        return torch.searchsorted(keys, splitters)
    w0 = keys[:, 0].contiguous()
    lo = torch.searchsorted(w0, splitters[:, 0].contiguous())
    hi = torch.searchsorted(w0, splitters[:, 0].contiguous(), right=True)
    cuts = [torch.searchsorted(keys[a:b, 1].contiguous(), splitters[j:j + 1, 1].contiguous()) + a
            for j, (a, b) in enumerate(zip(lo.tolist(), hi.tolist()))]
    return torch.cat(cuts) if cuts else torch.empty(0, dtype=torch.int64, device=keys.device)


def merge_tables_across_ranks(ops, local, group=None, gather_to=0):
    """The sparse exchange described at the top of this file.  `local` is this rank's sorted table (an `ops` handle; it is
    consumed).  Returns the merged table of ALL ranks on rank `gather_to` (None elsewhere) and a dict of what moved.
    `ops.views` gives keys of one int64 per row (a vector, or a (rows, 1) matrix) or of two (a (rows, 2) matrix)."""
    import torch
    dist = _dist()
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    keys, counts = ops.views(local)
    if keys.dim() == 2 and keys.shape[1] == 1:
        keys = keys.reshape(-1)   # one word per row: the int64 values are the order
    row = tuple(keys.shape[1:])   # () for one word per row, (2,) for two
    dev = keys.device
    key_len = ops.key_len(local)
    # --- splitters: world - 1 keys at the quantiles of rank 0's table, broadcast ---
    splitters = torch.zeros((max(world - 1, 1),) + row, dtype=torch.int64, device=dev)
    if rank == 0 and keys.shape[0] > 0 and world > 1:
        at = (torch.arange(1, world, device=dev, dtype=torch.int64) * keys.shape[0]) // world
        splitters[: world - 1] = keys[at]
    nrows = torch.tensor([keys.shape[0]], dtype=torch.int64, device=dev)
    dist.broadcast(splitters, src=0, group=group)
    dist.broadcast(nrows, src=0, group=group)
    if int(nrows.item()) == 0:
        splitters.fill_(np.iinfo(np.int64).max)   # rank 0 holds nothing: everything goes to rank 0's range
    # --- cut this rank's table at the splitters (it is sorted: every range is a contiguous slice) ---
    cuts = _cut(keys, splitters[: world - 1]) if world > 1 else torch.empty(0, dtype=torch.int64, device=dev)
    bounds = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), cuts.to(torch.int64),
                        torch.tensor([keys.shape[0]], dtype=torch.int64, device=dev)])
    send_sizes = (bounds[1:] - bounds[:-1]).contiguous()
    recv_sizes = torch.empty_like(send_sizes)
    dist.all_to_all_single(recv_sizes, send_sizes, group=group)
    send_list, recv_list = send_sizes.tolist(), recv_sizes.tolist()
    # --- ONE all-to-all per array: range r of every rank goes to rank r ---
    rkeys = torch.empty((int(sum(recv_list)),) + row, dtype=torch.int64, device=dev)
    rcounts = torch.empty(int(sum(recv_list)), dtype=torch.int32, device=dev)
    dist.all_to_all_single(rkeys, keys.contiguous(), output_split_sizes=recv_list, input_split_sizes=send_list, group=group)
    dist.all_to_all_single(rcounts, counts.contiguous(), output_split_sizes=recv_list, input_split_sizes=send_list, group=group)
    ops.free(local)
    # --- merge the `world` sorted runs received: pairwise, as a tree ---
    runs, at = [], 0
    for size in recv_list:
        runs.append(ops.from_tensors(rkeys[at:at + size], rcounts[at:at + size], key_len))
        at += size
    while len(runs) > 1:
        nxt = []
        for k in range(0, len(runs) - 1, 2):
            nxt.append(ops.merge(runs[k], runs[k + 1]))
            ops.free(runs[k])
            ops.free(runs[k + 1])
        if len(runs) % 2:
            nxt.append(runs[-1])
        runs = nxt
    mine = runs[0]
    # --- the ranges, in rank order, are the sorted table of everything: gathered on one rank ---
    mkeys, mcounts = ops.views(mine)
    mkeys = mkeys.reshape((mkeys.shape[0],) + row)
    sizes = torch.zeros(world, dtype=torch.int64, device=dev)
    sizes[rank] = mkeys.shape[0]
    dist.all_reduce(sizes, group=group)
    size_list = sizes.tolist()
    to_root = [int(mkeys.shape[0]) if r == gather_to else 0 for r in range(world)]
    from_all = [int(s) for s in size_list] if rank == gather_to else [0] * world
    gkeys = torch.empty((int(sum(from_all)),) + row, dtype=torch.int64, device=dev)
    gcounts = torch.empty(int(sum(from_all)), dtype=torch.int32, device=dev)
    dist.all_to_all_single(gkeys, mkeys.contiguous(), output_split_sizes=from_all, input_split_sizes=to_root, group=group)
    dist.all_to_all_single(gcounts, mcounts.contiguous(), output_split_sizes=from_all, input_split_sizes=to_root, group=group)
    ops.free(mine)
    row_bytes = 8 * (row[0] if row else 1) + 4
    info = {"rows_sent": int(sum(send_list)), "rows_owned_after_merge": int(size_list[rank]), "rows_total": int(sum(size_list)),
            "bytes_all_to_all": int(sum(send_list)) * row_bytes}
    if rank != gather_to:
        return None, info
    return ops.from_tensors(gkeys, gcounts, key_len), info


# ---------------------------------------------------------------------------------------------------------------------
# the exchange step of bench.py
# ---------------------------------------------------------------------------------------------------------------------
class Exchange:
    """What the GPUs exchange after a pass over their shards: one all-reduce for dense results, the sorted-table merge for
    sparse ones."""

    def __init__(self, wl, world, dev):
        import torch
        from ._lib import lib
        self.wl, self.world, self.dev = wl, world, dev
        self.merged = None
        self.info = {}
        self.ops = None
        self.tensor = wl.dense_tensor()
        self.kind = "vector"
        if self.tensor is None:
            ptr, cells = C.c_void_p(), C.c_longlong()
            lib().scg_plan_dense_tally(wl.plan.handle, C.byref(ptr), C.byref(cells))
            if ptr.value:
                self.tensor = torch.as_tensor(_DevView(ptr.value, cells.value, "<i4"), device="cuda")
                self.kind = "matrix"
            else:
                self.kind = "table"
                self.ops = DeviceTableOps(dev.index)

    def run(self):
        dist = _dist()
        if self.kind != "table":
            dist.all_reduce(self.tensor)   # one NCCL all-reduce over NVLink
            return
        if self.merged is not None:
            self.ops.free(self.merged)
        self.merged, self.info = merge_tables_across_ranks(self.ops, self.ops.from_plan(self.wl.plan))

    def result(self):
        """The combined result in the shape of Workload.result(); sparse tables only on rank 0 (None elsewhere)."""
        if self.kind == "vector":
            return [self.tensor.cpu().numpy()]
        if self.kind == "matrix":
            return self.wl.result()   # the plan's matrix now holds the sum
        if self.merged is None:
            return None
        return list(self.ops.render(self.merged))

    def describe(self):
        if self.kind == "vector":
            return "count vector (%d int32) combined with one NCCL all-reduce" % self.tensor.numel()
        if self.kind == "matrix":
            return "dense count matrix (%d int32) combined with one NCCL all-reduce" % self.tensor.numel()
        return ("per-GPU tables sort-reduced on the device, key ranges exchanged with one NCCL all-to-all per array, merged on the "
                "device (scg_table_merge), gathered on rank 0; last step moved %s" % json_safe(self.info))


def json_safe(d):
    return {k: (int(v) if isinstance(v, (int, np.integer)) else v) for k, v in d.items()}


def verify_sharded(wl, exchange, first, units, rank, world, local_rank, stream):
    """N > 1 on real NCCL: every rank runs the first `check` units of ITS range and the results are exchanged; rank 0 then
    runs the union of those ranges alone and both must be equal.  Returns a dict for the bench line (rank 0) / None."""
    import torch
    dist = _dist()
    check = int(min(units, 2_000_000))
    firsts = torch.zeros(world, dtype=torch.int64, device=exchange.dev)
    firsts[rank] = first
    dist.all_reduce(firsts)
    mine = wl.resident(first, check, local_rank)
    wl.reset(stream)
    wl.run_slice(mine, stream) if hasattr(wl, "run_slice") else wl.run(mine, stream)
    exchange.run()
    torch.cuda.synchronize()
    combined = exchange.result()
    del mine
    if rank != 0:
        dist.barrier()
        return None
    wl.reset(stream)
    for f in firsts.tolist():
        part = wl.resident(int(f), check, local_rank)
        wl.run(part, stream)
        torch.cuda.synchronize()
        del part
    alone = wl.result()
    equal = len(alone) == len(combined) and all(np.array_equal(np.asarray(a), np.asarray(b)) for a, b in zip(alone, combined))
    dist.barrier()
    assert equal, "the sharded, exchanged result differs from one GPU's result over the union of the ranges"
    return {"equal_to_one_gpu_over_the_union": True, "units_per_rank": check, "ranks": world,
            "rows_or_counters": int(np.asarray(alone[-1]).size)}
