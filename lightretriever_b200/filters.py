"""Document bitmaps: deletions and per-request filters inside the exact top-k of K2 and K4.

A bitmap is an int32 tensor holding u32 words indexed by GLOBAL document id (local row + ``id_offset``, the id a search
returns): document ``i`` is allowed when bit ``i & 31`` of word ``i >> 5`` is set — on a little-endian machine the bytes
Faiss's ``IDSelectorBitmap`` reads.  ``live`` ([ld_words], deletions) and a query's row of ``allow`` ([F, ld_words], with
``q_filter`` [Q] int32 choosing the row; -1 = unrestricted, any other value outside [0, F) allows nothing) are ANDed in the
kernels before a document can enter a candidate list, so the result is the exact top-k of the allowed documents (see
include/lr_b200.h).  Words are int32 tensors holding the u32 bit pattern, as impacts are int16 tensors holding u16.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _C
from ._util import require_cuda, stream_ptr


def _pack(bits: torch.Tensor) -> torch.Tensor:
    """bool [n_words * 32] -> int32 [n_words] (bit j of word w = bits[32 w + j])."""
    b = bits.view(-1, 32).to(torch.int64) << torch.arange(32, device=bits.device, dtype=torch.int64)
    w = b.sum(1)
    return torch.where(w >= 1 << 31, w - (1 << 32), w).to(torch.int32)


def _popcount(words: torch.Tensor) -> int:
    w = words.to(torch.int64) & 0xFFFFFFFF
    return int(((w.unsqueeze(1) >> torch.arange(32, device=w.device, dtype=torch.int64)) & 1).sum())


def doc_bitmap(n_ids: int, ids=None, device=None) -> torch.Tensor:
    """Bitmap of ``ceil(n_ids / 32)`` words with the bits of ids ``[0, n_ids)`` set (``ids`` None) or only those of
    ``ids`` (each in ``[0, n_ids)``)."""
    n_ids = int(n_ids)
    if n_ids < 0:
        raise ValueError(f"n_ids ({n_ids}) must be >= 0")
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    n_words = (n_ids + 31) // 32
    if ids is None:
        bits = torch.arange(n_words * 32, device=device) < n_ids
    else:
        idx = torch.as_tensor(ids, dtype=torch.int64).reshape(-1).to(device)
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= n_ids):
            raise ValueError(f"ids must lie in [0, {n_ids})")
        bits = torch.zeros(n_words * 32, dtype=torch.bool, device=device)
        bits[idx] = True
    return _pack(bits)


def doc_bitmap_update(words: torch.Tensor, ids, set: bool) -> None:
    """Set (``set=True``) or clear the bits of ``ids`` in ``words`` in place with ``lr_doc_bitmap_update``, on the current
    stream: no host synchronisation, so it may run between replays of a CUDA graph that reads ``words``.  Ids outside
    the bitmap are ignored."""
    words = require_cuda(words, "words")
    if words.dtype != torch.int32 or words.ndim != 1 or not words.is_contiguous():
        raise ValueError("words must be a contiguous 1-D int32 bitmap")
    dev = words.device
    idx = torch.as_tensor(ids, dtype=torch.int64).reshape(-1).to(dev, non_blocking=True).contiguous()
    lib = _C.load()
    with torch.cuda.device(dev):
        _C.check(lib.lr_doc_bitmap_update(words.data_ptr(), words.numel(), idx.data_ptr(), idx.numel(), int(bool(set)),
                                          stream_ptr(dev)))


def filter_args(live: Optional[torch.Tensor], allow: Optional[torch.Tensor], q_filter: Optional[torch.Tensor], Q: int,
                device) -> Optional[tuple]:
    """(live, allow, ld_words, n_filters, q_filter) arguments of the ``lr_*_filtered`` entry points, or None when no
    filter is given.  Range checks of ``ld_words`` against the shard are the library's (ValueError)."""
    if live is None and allow is None and q_filter is None:
        return None
    ld, n_filters = None, 0
    if live is not None:
        if live.dtype != torch.int32 or live.ndim != 1 or not live.is_contiguous() or live.device != device:
            raise ValueError(f"live must be a contiguous 1-D int32 bitmap on {device}")
        ld = live.numel()
    if allow is not None:
        if allow.ndim == 1:
            allow = allow.unsqueeze(0)
        if allow.dtype != torch.int32 or allow.ndim != 2 or not allow.is_contiguous() or allow.device != device:
            raise ValueError(f"allow must be a contiguous int32 [n_filters, ld_words] table on {device}")
        if ld is not None and allow.shape[1] != ld:
            raise ValueError(f"allow rows ({allow.shape[1]} words) and live ({ld} words) differ in length")
        ld, n_filters = allow.shape[1], allow.shape[0]
    if q_filter is not None:
        if q_filter.dtype != torch.int32 or q_filter.shape != (Q,) or not q_filter.is_contiguous() or q_filter.device != device:
            raise ValueError(f"q_filter must be a contiguous int32 [{Q}] tensor on {device}")
    return (None if live is None else live.data_ptr(), None if allow is None else allow.data_ptr(), int(ld or 0),
            int(n_filters), None if q_filter is None else q_filter.data_ptr())


class DocDeletions:
    """``delete`` / ``restore`` / ``n_live`` of an index whose documents have global ids ``[id_offset, id_offset +
    _live_rows())``.  Ids are in the index's result id space: passage ids when ``_passage_ids`` is set, otherwise global
    ids.  The ``live`` bitmap is created at the first deletion and applied by every later search."""

    _live: Optional[torch.Tensor] = None

    def _live_rows(self) -> int:
        raise NotImplementedError

    def _global_ids(self, ids) -> torch.Tensor:
        ids = np.asarray(torch.as_tensor(ids).cpu(), dtype=np.int64).reshape(-1)
        n = self._live_rows()
        pids = getattr(self, "_passage_ids", None)
        if pids is not None:
            order = np.argsort(pids, kind="stable")
            pos = np.searchsorted(pids[order], ids)
            pos = np.minimum(pos, len(pids) - 1) if len(pids) else pos
            if not len(pids) or not (pids[order][pos] == ids).all():
                raise ValueError("delete/restore: unknown passage id")
            rows = order[pos]
        else:
            rows = ids - self.id_offset
            if ((rows < 0) | (rows >= n)).any():
                raise ValueError(f"delete/restore: ids outside [{self.id_offset}, {self.id_offset + n})")
        return torch.from_numpy(rows + self.id_offset)

    def _range_words(self, lo: int, hi: int) -> torch.Tensor:
        n_words = (self.id_offset + self._live_rows() + 31) // 32
        bits = torch.arange(n_words * 32, device=self.device)
        return _pack((bits >= lo) & (bits < hi))

    def _extend_live(self, old_rows: int) -> None:
        """After rows were appended: the new rows are live."""
        if self._live is None:
            return
        new = self._range_words(self.id_offset + old_rows, self.id_offset + self._live_rows())
        new[:self._live.numel()] |= self._live
        self._live = new

    def delete(self, ids) -> None:
        """Remove documents from every later search (their rows stay in HBM; ``restore`` brings them back)."""
        g = self._global_ids(ids)
        if self._live is None:
            self._live = self._range_words(self.id_offset, self.id_offset + self._live_rows())
        doc_bitmap_update(self._live, g, False)

    def restore(self, ids) -> None:
        g = self._global_ids(ids)
        if self._live is not None:
            doc_bitmap_update(self._live, g, True)

    @property
    def n_live(self) -> int:
        return self._live_rows() if self._live is None else _popcount(self._live)

    @property
    def live_words(self) -> Optional[torch.Tensor]:
        """The index's ``live`` bitmap (None until the first deletion)."""
        return self._live
