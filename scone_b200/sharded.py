"""Row-sharded tier: a cache table too large for one GPU, split by f-gram id across the ranks of a process group.

New design (the reference's inference path is single-process, single-GPU; SURVEY.md section 8e).  One process per GPU,
``torch.distributed`` (NCCL over NVLink 5 / NVSwitch) for the plumbing:

  * the f-gram INDEX is replicated (128 B / f-gram), so every rank matches its own positions locally and only
    4-byte row numbers travel:  owner(id) = id % W, local row = id // W  (ids are frequency ranks in the reference,
    ``n_gram_extractor.py:98``, so the modulo spreads the hot low ids over all ranks);
  * all-to-all #1 carries the requested local row numbers (int32) to their owners;
  * each owner copies the requested rows VERBATIM -- still quantised -- into a reply buffer (``gather_packed``);
  * all-to-all #2 carries the packed rows back (INT4: 2 112 B instead of 8 192 B per row over NVLink);
  * the requester dequantises the received rows, fills misses from its local fallback table and writes
    ``[B, L, D]`` with ``scone_embed_gather``.  Misses never leave the GPU.
  Optionally the batch is cut into micro-batches of batch rows and these steps are software-pipelined (measured: no gain on
  8 GPUs, see ``ShardedEmbeddingCache``).

The routing arithmetic is plain torch (device-agnostic, exercised on CPU with gloo in tests/test_sharded_cpu.py); the
three compute steps are CUDA kernels of libscone_b200 behind the ``ops`` object.
"""

from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def owner_of(fgram_id: torch.Tensor, world: int) -> torch.Tensor:
    return fgram_id % world


def local_row_of(fgram_id: torch.Tensor, world: int) -> torch.Tensor:
    return torch.div(fgram_id, world, rounding_mode="floor")


def shard_rows(num_fgrams: int, rank: int, world: int) -> int:
    """Number of table rows rank ``rank`` owns (ids rank, rank + W, ...)."""
    return (num_fgrams - rank + world - 1) // world if num_fgrams > rank else 0


@dataclass
class RoutePlan:
    """Routing of one batch, cut into ``micro`` micro-batches of whole batch rows."""
    micro: int                       # number of micro-batches
    bounds: List[Tuple[int, int]]    # [micro] (first position, end position) of each micro-batch in the flattened batch
    order: torch.Tensor              # [n_hit] flat positions of the hits, grouped by (micro-batch, owner), stable
    send_rows: torch.Tensor          # [n_hit] int32 local row numbers, same order
    send_counts: List[List[int]]     # [micro][W] requests this rank sends to each owner
    recv_counts: List[List[int]]     # [micro][W] requests this rank receives from each requester
    slot_of_position: torch.Tensor   # [T] int32: index into ITS micro-batch's reply buffer, -1 for a miss

    def send_offset(self, m: int) -> int:
        return sum(sum(c) for c in self.send_counts[:m])


def make_plan(fgram_id: torch.Tensor, world: int, group=None, micro: int = 1) -> RoutePlan:
    """Bucket the hit positions by (micro-batch, owner) with ONE stable sort and exchange all bucket sizes with ONE small
    all-to-all (the tier's one host synchronisation per batch)."""
    B = fgram_id.shape[0] if fgram_id.dim() == 2 else 1
    flat = fgram_id.reshape(-1)
    T = flat.numel()
    L = T // max(B, 1)
    micro = max(1, min(int(micro), B))
    rows_per = max(1, (B + micro - 1) // micro)
    micro = max(1, (B + rows_per - 1) // rows_per)
    bounds = [(m * rows_per * L, min(B, (m + 1) * rows_per) * L) for m in range(micro)]
    hit = flat >= 0
    mb = torch.div(torch.arange(T, device=flat.device), max(rows_per * L, 1), rounding_mode="floor")
    key = torch.where(hit, mb * world + owner_of(flat.clamp(min=0), world), torch.full_like(mb, micro * world))
    order_all = torch.argsort(key, stable=True)
    counts = torch.bincount(key, minlength=micro * world + 1)[:micro * world].view(micro, world)
    n_hit = int(counts.sum().item())
    order = order_all[:n_hit]
    send_rows = local_row_of(flat[order], world).to(torch.int32)
    send_t = counts.t().contiguous()                 # [W, micro]: what goes to each owner, per micro-batch
    recv_t = torch.empty_like(send_t)                # [W, micro]: what each requester asks of this rank
    dist.all_to_all_single(recv_t, send_t, group=group)
    # position -> slot in its micro-batch's reply buffer
    first_of_mb = torch.cumsum(counts.sum(dim=1), 0) - counts.sum(dim=1)
    slot = torch.full((T,), -1, dtype=torch.int32, device=flat.device)
    slot[order] = (torch.arange(n_hit, device=flat.device) - first_of_mb[mb[order]]).to(torch.int32)
    return RoutePlan(micro, bounds, order, send_rows, counts.tolist(), recv_t.t().tolist(), slot)


def exchange_requests(plan: RoutePlan, m: int = 0, group=None, async_op: bool = False):
    """all-to-all #1 of micro-batch m: local row numbers to their owners.  Returns the int32 rows this rank must serve
    (and the work handle when ``async_op``)."""
    off = plan.send_offset(m)
    send = plan.send_rows[off:off + sum(plan.send_counts[m])]
    req = torch.empty((sum(plan.recv_counts[m]),), dtype=torch.int32, device=send.device)
    work = dist.all_to_all_single(req, send, plan.recv_counts[m], plan.send_counts[m], group=group, async_op=async_op)
    return (req, work) if async_op else req


def exchange_replies(plan: RoutePlan, served: torch.Tensor, m: int = 0, group=None, async_op: bool = False):
    """all-to-all #2 of micro-batch m: packed rows back to the requesters, in request order.  served: [n_recv, row_stride] uint8."""
    reply = torch.empty((sum(plan.send_counts[m]), served.shape[1]), dtype=served.dtype, device=served.device)
    work = dist.all_to_all_single(reply, served, plan.send_counts[m], plan.recv_counts[m], group=group, async_op=async_op)
    return (reply, work) if async_op else reply


class CudaOps:
    """The compute steps, as kernels of libscone_b200."""

    def __init__(self, index, local_table, base_emb: torch.Tensor):
        self.index, self.table, self.base = index, local_table, base_emb

    def match(self, input_ids: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        return self.index.lookup(input_ids)

    def serve(self, local_rows: torch.Tensor) -> torch.Tensor:
        return self.table.gather_packed(local_rows)

    def assemble(self, input_ids: torch.Tensor, reply: torch.Tensor, slot_of_position: torch.Tensor,
                 out: Optional[torch.Tensor]) -> torch.Tensor:
        from .table import embed_gather
        view = self.table.view_of(reply) if reply.shape[0] else self.table.view_of(
            torch.zeros((1, self.table.row_stride), dtype=torch.uint8, device=reply.device))
        return embed_gather(view, self.base, input_ids, slot_of_position.view(input_ids.shape), out=out)


class ShardedEmbeddingCache:
    """``lookup`` over a table row-sharded across the process group, through two all-to-alls (the north star's design).

    ``ops`` supplies match / serve / assemble; the default is :class:`CudaOps` (there is no CPU implementation in the
    product -- tests inject an oracle-backed stand-in to exercise the routing on CPU with gloo).

    One stable sort buckets the whole batch by (micro-batch, owner) and one small all-to-all exchanges every bucket size:
    one host synchronisation per batch.  With ``micro_batches > 1`` the batch is cut into groups of batch rows and
    software-pipelined: while the packed rows of micro-batch m cross NVLink (all-to-all #2, on the communicator's own
    stream), the owner-side gather of micro-batch m+1 and the requester-side dequantising gather of micro-batch m-1 are
    enqueued on the compute stream.  MEASURED (config 4 in full, 8 GPUs; profiles/tune_r02.md section 11): 7.88 ms with one
    micro-batch, 8.16 with four, 8.60 with eight -- the smaller all-to-alls are less efficient and the persistent gather
    kernels do not leave the communicator the SMs to overlap with; the default is therefore ONE micro-batch.
    """

    def __init__(self, ops, group=None, micro_batches: int = 1):
        self.ops = ops
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.micro_batches = max(1, int(micro_batches))
        self.last_plan: Optional[RoutePlan] = None

    def lookup(self, input_ids: torch.Tensor, out: Optional[torch.Tensor] = None):
        fgram_id, match_len = self.ops.match(input_ids)
        B, L = input_ids.shape
        plan = make_plan(fgram_id, self.world, self.group, micro=self.micro_batches)
        self.last_plan = plan
        M = plan.micro
        slot2d = plan.slot_of_position.view(B, L)
        # all-to-all #1 of every micro-batch (a few bytes per position): issued at once, waited for just before its serve
        reqs = [exchange_requests(plan, m, self.group, async_op=True) for m in range(M)]
        parts, replies = [None] * M, [None] * M

        def assemble(m):
            b0, b1 = plan.bounds[m][0] // L, plan.bounds[m][1] // L
            reply, work = replies[m]
            work.wait()
            parts[m] = self.ops.assemble(input_ids[b0:b1], reply, slot2d[b0:b1].reshape(-1), None if out is None else out[b0:b1])

        for m in range(M):
            req, work = reqs[m]
            work.wait()
            served = self.ops.serve(req)                                     # owner side: packed rows, no dequantisation
            replies[m] = exchange_replies(plan, served, m, self.group, async_op=True)   # crosses NVLink while ...
            if m >= 1:
                assemble(m - 1)                                             # ... the previous micro-batch is dequantised
        assemble(M - 1)
        embeds = out if out is not None else (parts[0] if M == 1 else torch.cat(parts, dim=0))
        return embeds, fgram_id, match_len


# ----------------------------------------------------------------------------------------------------------------
# Peer-direct variant: the gather and the exchange are ONE kernel.  Every rank maps every shard (symmetric memory over
# NVLink / NVSwitch); the matcher warps of the fused kernel turn (id % W, id // W) into a peer address and the TMA bulk
# copy pulls the still-quantised row across NVSwitch straight into shared memory.  No request / reply messages, no
# bucketing, no host synchronisation -- the call is CUDA-graph capturable like the single-GPU path.
# ----------------------------------------------------------------------------------------------------------------

class PeerShardedTable:
    """This rank's shard of a table of ``total_rows`` rows, allocated in symmetric memory and mapped by all peers."""

    def __init__(self, total_rows: int, dim: int, quant: str = "fp16", group_size: int = 128, device=None, group=None):
        import torch.distributed._symmetric_memory as symm_mem
        from .table import CacheTable, table_layout
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.total_rows = int(total_rows)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        cap = (self.total_rows + self.world - 1) // self.world
        row_stride, _ = table_layout(quant, dim, group_size)
        storage = symm_mem.empty((max(cap, 1), row_stride), dtype=torch.uint8, device=self.device)
        storage.zero_()
        self._handle = symm_mem.rendezvous(storage, self.group.group_name)
        self.local = CacheTable(max(cap, 1), dim, quant, group_size, self.device, storage=storage)
        self.ptr_table = torch.tensor(list(self._handle.buffer_ptrs), dtype=torch.int64, device=self.device)
        self.rows_owned = shard_rows(self.total_rows, self.rank, self.world)
        self._views = {}

    def shard_view(self, rank: int):
        """Rank ``rank``'s shard as a CacheTable over its peer-mapped buffer (reads cross NVLink; ``rank == self.rank`` is
        the local shard).  Valid after that rank's :meth:`publish`."""
        if rank == self.rank:
            return self.local
        if rank not in self._views:
            buf = self._handle.get_buffer(rank, tuple(self.local.storage.shape), torch.uint8)
            self._views[rank] = self.local.view_of(buf)
        return self._views[rank]

    def store_owned(self, rows_fp32: torch.Tensor, fgram_ids: torch.Tensor) -> None:
        """Quantise and store the rows of the given GLOBAL f-gram ids; ids this rank does not own are ignored."""
        fgram_ids = fgram_ids.to(self.device)
        mine = owner_of(fgram_ids, self.world) == self.rank
        if bool(mine.any()):
            self.local.store(rows_fp32.to(self.device)[mine], local_row_of(fgram_ids[mine], self.world))

    def publish(self) -> None:
        """Make this rank's rows visible to its peers (call once after the last store)."""
        torch.cuda.synchronize(self.device)
        dist.barrier(self.group)


def embed_forward_sharded(index, table: PeerShardedTable, base_emb: torch.Tensor, input_ids: torch.Tensor,
                          pos_emb: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                          status: Optional[torch.Tensor] = None, out_id: Optional[torch.Tensor] = None,
                          out_len: Optional[torch.Tensor] = None):
    """The fused hot path over a peer-mapped, row-sharded table (one kernel, asynchronous, graph-capturable)."""
    import ctypes as C
    from . import _lib
    from .index import _stream_ptr
    from .table import _OUT
    from .table import check_embed_args
    ids = index._check_ids(input_ids)
    B, L = ids.shape
    dev = index.device
    if table.device != dev:
        raise ValueError("index and shard must be on the same device")
    out, out_id, out_len = check_embed_args(dev, table.local.dim, base_emb, pos_emb, (B, L), out, out_id, out_len, True)
    if status is not None and (status.device != dev or status.dtype != torch.int32):
        raise ValueError("status must be an int32 tensor on the index device")
    with torch.cuda.device(dev):
        _lib.check(_lib.load().scone_embed_forward_sharded(
            index.handle, C.byref(table.local.desc), table.ptr_table.data_ptr(), table.world, table.total_rows,
            base_emb.data_ptr(), base_emb.shape[0], pos_emb.data_ptr() if pos_emb is not None else None,
            ids.data_ptr(), B, L, out.data_ptr(), _OUT[base_emb.dtype], out_id.data_ptr(), out_len.data_ptr(),
            status.data_ptr() if status is not None else None, _stream_ptr(dev)))
    return out, out_id, out_len
