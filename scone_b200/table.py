"""Packed cache table in HBM (or device-mapped pinned host memory) + the fused embed call."""

from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from .index import FGramIndex, _require_cuda, _stream_ptr

_OUT = {torch.bfloat16: _lib.OUT_BF16, torch.float16: _lib.OUT_FP16, torch.float32: _lib.OUT_FP32}


def table_layout(quant: str, dim: int, group: int = 128, align: int = 32) -> Tuple[int, int]:
    """(row_stride bytes, scale_offset bytes) of a stored row."""
    if quant not in _lib.QUANT:
        raise ValueError(f"quant must be one of {sorted(_lib.QUANT)}")
    rs, so = C.c_int64(), C.c_int32()
    _lib.check(_lib.load().scone_table_layout(_lib.QUANT[quant], dim, group, align, C.byref(rs), C.byref(so)))
    return int(rs.value), int(so.value)


def _free_host(ptr: int, nbytes: int) -> None:
    try:
        _lib.load().scone_host_free(ptr, nbytes)
    except Exception:
        pass


class CacheTable:
    """N rows of D elements stored as FP32 (unquantised, the reference's own storage) / FP16 / INT8 (per-row scale) /
    INT4 (per-group fp16 scales).

    Row r is the embedding of f-gram id r (reference ``scone/inference/embedding_cache.py:77,99``).
    ``storage`` is a uint8 tensor [N, row_stride]: on the GPU (tier "hbm") or pinned host memory
    mapped into the device address space (tier "host").
    """

    def __init__(self, num_rows: int, dim: int, quant: str = "fp16", group: int = 128, device="cuda", tier: str = "hbm",
                 align: int = 32, storage: Optional[torch.Tensor] = None):
        self.num_rows, self.dim, self.quant, self.group, self.tier = int(num_rows), int(dim), quant, int(group), tier
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("CacheTable lives on a CUDA device: scone_b200 has no CPU path")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.row_stride, self.scale_offset = table_layout(quant, dim, group, align)
        if storage is not None:
            if storage.dtype != torch.uint8 or tuple(storage.shape) != (self.num_rows, self.row_stride):
                raise ValueError("storage must be uint8 [num_rows, row_stride]")
            self.storage = storage
        elif tier == "hbm":
            self.storage = torch.zeros((self.num_rows, self.row_stride), dtype=torch.uint8, device=self.device)
        elif tier == "host":
            self.storage = self._alloc_host(self.num_rows * self.row_stride).view(self.num_rows, self.row_stride)
        else:
            raise ValueError("tier must be 'hbm' or 'host'")
        if tier == "hbm":
            _require_cuda(self.storage, "storage")
            self._dev_ptr = self.storage.data_ptr()
        elif self._host_dev_ptr is not None:
            self._dev_ptr = self._host_dev_ptr
        else:
            if not self.storage.is_pinned():
                raise ValueError("host-tier storage must be pinned")
            # pinned allocations are mapped under UVA: the host pointer is valid on the device
            self._dev_ptr = self.storage.data_ptr()
        self.desc = _lib.TableDesc(self._dev_ptr, self.row_stride, self.num_rows, _lib.QUANT[quant], self.dim, self.group,
                                   self.scale_offset)

    _host_dev_ptr = None

    def _alloc_host(self, nbytes: int) -> torch.Tensor:
        """Zero-filled host memory the GPU reads in place: ``scone_host_alloc`` (huge pages, parallel first touch, registered
        as mapped pinned memory)."""
        import os
        import weakref
        nbytes = max(int(nbytes), 1)
        host, dev = C.c_void_p(), C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_host_alloc(nbytes, min(32, os.cpu_count() or 1), C.byref(host), C.byref(dev)))
        buf = (C.c_uint8 * nbytes).from_address(host.value)
        t = torch.frombuffer(buf, dtype=torch.uint8)
        self._host_dev_ptr = dev.value
        # the region lives as long as this table: ``storage`` (and numpy views of it) must not outlive the CacheTable
        weakref.finalize(self, _free_host, host.value, nbytes)
        return t

    @property
    def bytes(self) -> int:
        return self.num_rows * self.row_stride

    def store(self, rows_fp32: torch.Tensor, row_ids: Optional[torch.Tensor] = None, row_base: int = 0) -> None:
        """Quantise fp32 rows [k, D] on the GPU and write them at ``row_ids`` (or row_base..row_base+k)."""
        _require_cuda(rows_fp32, "rows")
        rows = rows_fp32.to(torch.float32).contiguous()
        if rows.dim() != 2 or rows.shape[1] != self.dim:
            raise ValueError(f"rows must be [k, {self.dim}]")
        k = rows.shape[0]
        ids_ptr = None
        if row_ids is not None:
            row_ids = row_ids.to(device=self.device, dtype=torch.int64).contiguous()
            if row_ids.numel() != k:
                raise ValueError("row_ids and rows disagree on k")
            if k and (int(row_ids.min()) < 0 or int(row_ids.max()) >= self.num_rows):
                raise IndexError("row id out of range")
            ids_ptr = row_ids.data_ptr()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_table_store(C.byref(self.desc), rows.data_ptr(), ids_ptr, int(row_base), k,
                                                     _stream_ptr(self.device)))

    def store_projected(self, rows: torch.Tensor, projection: torch.Tensor, row_ids: Optional[torch.Tensor] = None,
                        row_base: int = 0) -> None:
        """``table[row] = quantise(rows @ projection.T)`` -- the reference's bias-free ``f_gram_projection``
        (``scone/models/language_model.py:172-176, 236``) folded into the table build.  rows [k, H_f], projection [D, H_f]
        (``nn.Linear.weight`` layout); both are rounded to bf16 (RNE) and multiplied on the tensor cores with fp32
        accumulation; the quantise-and-store of :meth:`store` is the GEMM's epilogue (no fp32 [k, D] intermediate)."""
        _require_cuda(rows, "rows")
        _require_cuda(projection, "projection")
        if rows.dim() != 2 or projection.dim() != 2 or projection.shape[0] != self.dim or rows.shape[1] != projection.shape[1]:
            raise ValueError(f"rows must be [k, H_f] and projection [{self.dim}, H_f]")
        if self.tier != "hbm":
            raise ValueError("store_projected writes an HBM-resident table")
        a = rows.to(device=self.device, dtype=torch.bfloat16).contiguous()
        w = projection.detach().to(device=self.device, dtype=torch.bfloat16).contiguous()
        k = a.shape[0]
        ids_ptr = None
        if row_ids is not None:
            row_ids = row_ids.to(device=self.device, dtype=torch.int64).contiguous()
            if row_ids.numel() != k:
                raise ValueError("row_ids and rows disagree on k")
            ids_ptr = row_ids.data_ptr()
        bad = torch.zeros((1,), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_table_store_projected(C.byref(self.desc), a.data_ptr(), w.data_ptr(), int(a.shape[1]), ids_ptr,
                                                               int(row_base), k, bad.data_ptr(), _stream_ptr(self.device)))
        if int(bad.item()):
            raise IndexError("row id out of range")

    def gather(self, row_ids: torch.Tensor, dtype: torch.dtype = torch.float32) -> torch.Tensor:
        """dequant(table[row_ids]) -> [k, D] (the reference's get_embeddings gather)."""
        row_ids = row_ids.to(device=self.device, dtype=torch.int64).contiguous()
        k = row_ids.numel()
        out = torch.empty((k, self.dim), dtype=dtype, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_table_gather(C.byref(self.desc), row_ids.data_ptr(), k, out.data_ptr(), _OUT[dtype],
                                                      None, _stream_ptr(self.device)))
        return out


    def gather_packed(self, row_ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Stored bytes of rows ``row_ids`` (int32) -> uint8 [k, row_stride]; no dequantisation (sharded tier, owner side)."""
        row_ids = row_ids.to(device=self.device, dtype=torch.int32).contiguous()
        k = row_ids.numel()
        if out is None:
            out = torch.empty((k, self.row_stride), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_table_gather_packed(C.byref(self.desc), row_ids.data_ptr(), k, out.data_ptr(), None,
                                                             _stream_ptr(self.device)))
        return out

    def view_of(self, storage: torch.Tensor) -> "CacheTable":
        """A table with this one's format over another [k, row_stride] uint8 buffer (e.g. rows received from a peer)."""
        return CacheTable(storage.shape[0], self.dim, self.quant, self.group, self.device, "hbm", storage=storage)


def check_embed_args(dev: torch.device, dim: int, base_emb: torch.Tensor, pos_emb: Optional[torch.Tensor], shape: Tuple[int, ...],
                     out: Optional[torch.Tensor], out_id: Optional[torch.Tensor] = None, out_len: Optional[torch.Tensor] = None,
                     want_ids: bool = False):
    """Argument checks shared by every fused entry (hbm, host, sharded tiers; resolved-ids gather): a short or mistyped
    ``pos_emb`` / ``out`` would otherwise become an out-of-bounds bulk copy instead of a ValueError.  ``shape`` is the id
    tensor's shape (its last dimension is the sequence length).  Allocates what is missing; returns (out, out_id, out_len)."""
    L = shape[-1] if len(shape) else 1
    n = 1
    for d in shape:
        n *= int(d)
    if base_emb.dtype not in (torch.bfloat16, torch.float16):
        raise ValueError("base_emb must be bf16 or fp16 (it defines the output dtype)")
    if base_emb.device != dev:
        raise ValueError("index, table and base_emb must be on the same device")
    if base_emb.dim() != 2 or base_emb.shape[1] != dim or not base_emb.is_contiguous():
        raise ValueError(f"base_emb must be contiguous [V, {dim}]")
    if pos_emb is not None:
        if pos_emb.dtype != base_emb.dtype or pos_emb.device != dev or not pos_emb.is_contiguous() \
                or pos_emb.dim() != 2 or pos_emb.shape[1] != dim or pos_emb.shape[0] < L:
            raise ValueError(f"pos_emb must be contiguous [>= {L}, {dim}] {base_emb.dtype} on {dev}")
    if out is None:
        out = torch.empty(tuple(shape) + (dim,), dtype=base_emb.dtype, device=dev)
    elif out.dtype != base_emb.dtype or tuple(out.shape) != tuple(shape) + (dim,) or not out.is_contiguous() or out.device != dev:
        raise ValueError(f"out must be contiguous {tuple(shape) + (dim,)} in base_emb.dtype on {dev}")
    if want_ids:
        if out_id is None:
            out_id = torch.empty(tuple(shape), dtype=torch.int32, device=dev)
        if out_len is None:
            out_len = torch.empty(tuple(shape), dtype=torch.uint8, device=dev)
        if out_id.dtype != torch.int32 or out_len.dtype != torch.uint8 or out_id.numel() != n or out_len.numel() != n \
                or not out_id.is_contiguous() or not out_len.is_contiguous() or out_id.device != dev or out_len.device != dev:
            raise ValueError("out_id must be contiguous int32 and out_len uint8, both of the id tensor's shape, on the index device")
    else:
        out_id = out_len = None
    return out, out_id, out_len


def embed_forward(index: FGramIndex, table: CacheTable, base_emb: torch.Tensor, input_ids: torch.Tensor,
                  pos_emb: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                  status: Optional[torch.Tensor] = None, want_ids: bool = True,
                  out_id: Optional[torch.Tensor] = None, out_len: Optional[torch.Tensor] = None, combine: str = "replace",
                  inputs_stable: bool = False):
    """The fused hot path.  Returns (embeds [B, L, D] in base_emb.dtype, fgram_id int32 [B, L], match_len uint8 [B, L]).

    out[b, i] = dequant(table[fgram_id[b, i]]) if an f-gram ends at (b, i) else base_emb[input_ids[b, i]]
    (+ pos_emb[i] when given).  ``combine="add"`` is the reference code's combine instead of Algorithm 2's replacement
    (``scone/models/language_model.py:239-243``): base_emb[input_ids[b, i]] + dequant(row) where an f-gram ends.
    Everything is enqueued on the current stream; nothing synchronises.

    ``inputs_stable=True`` (``SCONE_EMBED_INPUTS_STABLE``): the caller vouches that none of the inputs (ids, table, base /
    position rows) is written by the kernel that precedes this call on the stream -- a serving loop whose ids arrive by
    copy and whose tables are static.  Back-to-back lookups then overlap: the next call's matching and row fetches run
    under this call's tail, only its writes wait.  Same results.
    """
    if combine not in ("replace", "add"):
        raise ValueError("combine must be 'replace' or 'add'")
    ids = index._check_ids(input_ids)
    B, L = ids.shape
    dev = index.device
    if table.device != dev:
        raise ValueError("index, table and base_emb must be on the same device")
    out, out_id, out_len = check_embed_args(dev, table.dim, base_emb, pos_emb, (B, L), out, out_id, out_len, want_ids)
    opts = _lib.EmbedOpts((_lib.EMBED_ADDITIVE if combine == "add" else 0) | (_lib.EMBED_INPUTS_STABLE if inputs_stable else 0))
    with torch.cuda.device(dev):
        _lib.check(_lib.load().scone_embed_forward_ex(
            index.handle, C.byref(table.desc), base_emb.data_ptr(), base_emb.shape[0],
            pos_emb.data_ptr() if pos_emb is not None else None, ids.data_ptr(), B, L, out.data_ptr(), _OUT[base_emb.dtype],
            out_id.data_ptr() if want_ids else None, out_len.data_ptr() if want_ids else None,
            status.data_ptr() if status is not None else None, C.byref(opts), _stream_ptr(dev)))
    return out, out_id, out_len


def embed_gather(table: CacheTable, base_emb: torch.Tensor, input_ids: torch.Tensor, fgram_id: torch.Tensor,
                 pos_emb: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                 status: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Second half of the path with ids already resolved (sharded / staged tiers)."""
    _require_cuda(input_ids, "input_ids")
    ids = input_ids.contiguous()
    fid = fgram_id.contiguous()
    if ids.dtype != torch.int64 or fid.dtype != torch.int32 or ids.shape != fid.shape:
        raise ValueError("input_ids (long) and fgram_id (int32) must have the same shape")
    dev = table.device
    if ids.device != dev or fid.device != dev:
        raise ValueError(f"input_ids and fgram_id must be on the table's device {dev}")
    if status is not None and (status.device != dev or status.dtype != torch.int32):
        raise ValueError("status must be an int32 tensor on the table's device")
    T = ids.numel()
    L = ids.shape[-1] if ids.dim() >= 1 else 1
    out, _, _ = check_embed_args(dev, table.dim, base_emb, pos_emb, tuple(ids.shape), out)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().scone_embed_gather(
            C.byref(table.desc), base_emb.data_ptr(), base_emb.shape[0], pos_emb.data_ptr() if pos_emb is not None else None,
            L, ids.data_ptr(), fid.data_ptr(), T, out.data_ptr(), _OUT[base_emb.dtype],
            status.data_ptr() if status is not None else None, _stream_ptr(dev)))
    return out


def embed_mean_forward(index: FGramIndex, table: CacheTable, input_ids: torch.Tensor, dtype: torch.dtype = torch.float32) -> torch.Tensor:
    """Reference-CODE semantics (``scone/inference/engine.py:235-259``): per position the mean of the rows of all f-grams
    containing it, zeros where none -- the tensor the reference passes as ``f_gram_embeddings``.  [B, L, D] in ``dtype``."""
    ids = index._check_ids(input_ids)
    B, L = ids.shape
    dev = index.device
    work = torch.empty((B, L, index.max_n), dtype=torch.int32, device=dev)
    out = torch.empty((B, L, table.dim), dtype=dtype, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().scone_embed_mean_forward(index.handle, C.byref(table.desc), ids.data_ptr(), B, L, work.data_ptr(),
                                                        out.data_ptr(), _OUT[dtype], _stream_ptr(dev)))
    return out
