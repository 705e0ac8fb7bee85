"""Device-resident f-gram index (thin wrapper over scone_index_* of the C ABI)."""

from __future__ import annotations

import ctypes as C
from typing import Tuple

import torch

from . import _lib


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor: scone_b200 has no CPU path")


# scone_index_info_t::slot_format -> name, in the order of index_plan.h's SlotFormat (kSlotFormats[].name)
SLOT_FORMATS = ("wide32", "compact16", "compact20")


class FGramIndex:
    """Open-addressing hash index of the f-gram vocabulary in HBM.

    Replaces ``NGramExtractor.f_grams`` / ``f_gram_to_id`` (reference
    ``scone/tokenization/n_gram_extractor.py:41-44``) for batched lookups.  Immutable after
    construction, so it can be shared by any number of streams / threads.
    """

    def __init__(self, vocab_tokens: torch.Tensor, vocab_lens: torch.Tensor, load_factor: float = 0.0):
        """vocab_tokens int32 [N, max_n] (reading order, padded with -1), vocab_lens uint8 [N]; id = row.
        load_factor 0 = the library default (0.25).  Compact 16-byte slots are used automatically when all tokens are
        < 65535 and max_n <= 6 (six 16-bit tokens) or < 1048575 and max_n <= 5 (five 20-bit tokens: V = 128 000),
        32-byte slots otherwise (``slot_bytes`` / ``slot_format``).  Vocabularies of up to 48 M f-grams also get a Bloom
        pre-filter (``filter_bytes``: 16 bits per f-gram up to 12 M, 8 bits above) that large batches consult before
        touching a slot."""
        _require_cuda(vocab_tokens, "vocab_tokens")
        _require_cuda(vocab_lens, "vocab_lens")
        if vocab_tokens.dtype != torch.int32 or vocab_lens.dtype != torch.uint8:
            raise ValueError("vocab_tokens must be int32 and vocab_lens uint8")
        if vocab_tokens.dim() != 2 or vocab_lens.dim() != 1 or vocab_tokens.shape[0] != vocab_lens.shape[0]:
            raise ValueError("vocab_tokens must be [N, max_n] and vocab_lens [N]")
        vocab_tokens = vocab_tokens.contiguous()
        vocab_lens = vocab_lens.contiguous()
        self.device = vocab_tokens.device
        self.num_fgrams, self.max_n = int(vocab_tokens.shape[0]), int(vocab_tokens.shape[1])
        self._h = C.c_void_p()
        L = _lib.load()
        with torch.cuda.device(self.device):
            _lib.check(L.scone_index_create(vocab_tokens.data_ptr(), vocab_lens.data_ptr(), self.num_fgrams, self.max_n,
                                            float(load_factor), _stream_ptr(self.device), C.byref(self._h)))
        info = _lib.IndexInfo()
        _lib.check(L.scone_index_info(self._h, C.byref(info)))
        self.capacity, self.bytes = int(info.capacity), int(info.bytes)
        self.len_mask, self.max_probe = int(info.len_mask), int(info.max_probe)
        self.slot_bytes = int(info.slot_bytes)
        self.slot_format = SLOT_FORMATS[int(info.slot_format)]
        self.filter_bytes = int(info.filter_bytes)     # L2-resident pre-filter (0 = none), included in `bytes`

    @property
    def handle(self) -> C.c_void_p:
        if not self._h:
            raise RuntimeError("FGramIndex has been destroyed")
        return self._h

    def close(self) -> None:
        if getattr(self, "_h", None):
            _lib.load().scone_index_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check_ids(self, input_ids: torch.Tensor) -> torch.Tensor:
        _require_cuda(input_ids, "input_ids")
        if input_ids.device != self.device:
            raise ValueError(f"input_ids on {input_ids.device}, index on {self.device}")
        if input_ids.dtype != torch.int64:
            raise ValueError("input_ids must be torch.long")
        if input_ids.dim() != 2:
            raise ValueError("input_ids must be [batch, seq]")
        return input_ids.contiguous()

    def lookup(self, input_ids: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """Longest f-gram ending at each position: (fgram_id int32 [B, L] (-1 none), match_len uint8 [B, L])."""
        ids = self._check_ids(input_ids)
        B, L = ids.shape
        out_id = torch.empty((B, L), dtype=torch.int32, device=self.device)
        out_len = torch.empty((B, L), dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_index_lookup(self.handle, ids.data_ptr(), B, L, out_id.data_ptr(), out_len.data_ptr(),
                                                      _stream_ptr(self.device)))
        return out_id, out_len

    def match_all(self, input_ids: torch.Tensor) -> torch.Tensor:
        """int32 [B, L, max_n]: id of the n-gram ending at each position (slot n-1), -1 if not an f-gram."""
        ids = self._check_ids(input_ids)
        B, L = ids.shape
        out = torch.empty((B, L, self.max_n), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().scone_index_match_all(self.handle, ids.data_ptr(), B, L, out.data_ptr(),
                                                         _stream_ptr(self.device)))
        return out
