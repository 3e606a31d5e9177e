"""Host -> device staging of batch dicts, overlapped with compute.

The reference's loops move every tensor of a batch with a blocking ``batch[k].to(device)`` from pageable memory
right before the forward (fragnet/train/pretrain/pretrain_utils.py:13-14, train/utils.py:335-336): ~40 MB per
1024-molecule batch (19 tensors, int64 indices, one-hot fp32 features), i.e. ~1.2 ms of PCIe time that the GPU spends
idle.  ``DevicePrefetcher`` wraps any iterable of batch dicts (a ``DataLoader`` with ``collate_fn_pt``) and issues
the copies of the NEXT batches on a side stream from pinned memory while the current one is being consumed.

Device memory comes from ``depth`` persistent slots of grow-only flat buffers (one per dtype), so the steady state
performs no allocation and never touches the caching allocator from the copy stream.

Batches in the compact wire format (``dataset.data.compact_batch``: uint8 feature matrices, int32 indices -- a third
of the bytes) are widened on the device right behind their copy, on the copy stream, by one ``fnb_widen_batch`` launch:
the consumer always sees ``collate_fn``'s dtypes and values.  Batches that already live on the device (an
``ArenaLoader``) pass through untouched.
"""
from __future__ import annotations

import collections
import ctypes as C
from typing import Dict, Iterable, Iterator, List

import torch

from .. import _abi
from .data import INDEX_KEYS, ONE_HOT_KEYS

_UNREAD = ("edge_attr", "cnx_attr")


def _wide_dtype(key: str, t: torch.Tensor):
    """dtype the consumer expects for a (possibly narrowed) host tensor."""
    if t.dtype == torch.uint8 and key in ONE_HOT_KEYS:
        return torch.float32
    if t.dtype == torch.int32 and key in INDEX_KEYS:
        return torch.int64
    return t.dtype


def staged_bytes(host: Dict[str, torch.Tensor], hot_path_only: bool = True) -> int:
    """Bytes ``DevicePrefetcher`` moves over PCIe for this host batch."""
    return sum(v.numel() * v.element_size() for k, v in host.items()
               if isinstance(v, torch.Tensor) and not (hot_path_only and (k in _UNREAD or k == "x_frags")))


class _Slot:
    """Grow-only device staging area: one flat buffer per dtype, handed out as aligned views."""

    def __init__(self, device):
        self.device = device
        self.buffers: Dict[torch.dtype, torch.Tensor] = {}
        self.free_event = None          # recorded on the compute stream once the consumer has moved on

    def packed_views(self, blob: torch.Tensor, layout, widen):
        """Device mirror of a ``PackedBatch`` buffer: (device blob, wire views, consumer views, grew).  ``widen`` maps a
        key to the dtype the consumer expects where it differs from the wire dtype."""
        grew = False
        pad = lambda n: (n + 63) // 64 * 64
        need: Dict[object, int] = collections.defaultdict(int)
        need["blob"] = blob.numel()
        for key, dtype, shape, off, nbytes in layout:
            if key in widen:
                need[widen[key]] += pad(nbytes // torch.empty((), dtype=dtype).element_size())
        for dt, n in need.items():
            buf = self.buffers.get(dt)
            if buf is None or buf.numel() < n:
                self.buffers[dt] = torch.empty(int(n * 1.25) + 64, dtype=torch.uint8 if dt == "blob" else dt,
                                               device=self.device)
                grew = True
        dev_blob = self.buffers["blob"][:blob.numel()]
        used: Dict[object, int] = collections.defaultdict(int)
        wire, out = {}, {}
        for key, dtype, shape, off, nbytes in layout:
            wire[key] = dev_blob[off:off + nbytes].view(dtype).view(shape)
            if key in widen:
                n = wire[key].numel()
                o = used[widen[key]]
                used[widen[key]] = o + pad(n)
                out[key] = self.buffers[widen[key]][o:o + n].view(shape)
            else:
                out[key] = wire[key]
        return dev_blob, wire, out, grew

    def views(self, host: Dict[str, torch.Tensor]):
        """(wire views, consumer views, grew): device views shaped like the tensors of ``host`` in their wire dtype and
        in the dtype the consumer expects (the same view where nothing has to be widened)."""
        grew = False
        need: Dict[torch.dtype, int] = collections.defaultdict(int)
        pad = lambda n: (n + 63) // 64 * 64
        for k, v in host.items():
            if isinstance(v, torch.Tensor):
                need[v.dtype] += pad(v.numel())
                if _wide_dtype(k, v) != v.dtype:
                    need[_wide_dtype(k, v)] += pad(v.numel())
        for dt, n in need.items():
            buf = self.buffers.get(dt)
            if buf is None or buf.numel() < n:
                self.buffers[dt] = torch.empty(int(n * 1.25) + 64, dtype=dt, device=self.device)
                grew = True
        used: Dict[torch.dtype, int] = collections.defaultdict(int)

        def take(dt, shape, n):
            o = used[dt]
            used[dt] = o + pad(n)
            return self.buffers[dt][o:o + n].view(shape)
        wire, out = {}, {}
        for k, v in host.items():
            if isinstance(v, torch.Tensor):
                wire[k] = take(v.dtype, v.shape, v.numel())
                wd = _wide_dtype(k, v)
                out[k] = wire[k] if wd == v.dtype else take(wd, v.shape, v.numel())
            else:
                out[k] = v
        return wire, out, grew


class DevicePrefetcher:
    """``for batch in DevicePrefetcher(loader, device): ...`` yields device-resident batch dicts.

    ``depth`` batches are in flight (2 = double buffering).  A yielded batch stays valid until ``depth`` further
    batches have been requested.  Host tensors that are not pinned are pinned first (``DataLoader(pin_memory=True)``
    does that in the loader's workers)."""

    def __init__(self, batches: Iterable[Dict[str, torch.Tensor]], device, depth: int = 2, hot_path_only: bool = False,
                 keep: Iterable[str] = ()):
        """``hot_path_only=True`` moves only what the GAT2 path reads: ``edge_attr`` and ``cnx_attr`` are dropped
        (``FragNet.forward`` never reads them: gat2.py:381-442 takes ``node_features_bonds`` / ``edge_attr_fbonds``),
        and ``x_frags`` -- whose VALUES are overwritten unread by the atom->fragment pooling (gat2.py:234), only its
        row count matters -- arrives as a ``meta`` tensor of the same shape.  ~20 % fewer PCIe bytes per batch.
        ``keep``: entries of those two that are moved all the same (``cnx_attr`` for gat2_edge, gat2_edge.py:167)."""
        self.batches, self.device, self.depth = batches, torch.device(device), max(1, int(depth))
        self.hot_path_only = bool(hot_path_only)
        self._unread = tuple(k for k in _UNREAD if k not in set(keep))
        if self.device.type != "cuda":
            raise ValueError("DevicePrefetcher stages batches onto a CUDA device")
        # copy stream and staging slots are recycled across prefetchers of a device (a training loop makes one per
        # epoch, plus one per validation pass): a new set of slots is ~150 MB of cudaMalloc, i.e. a device-synchronising
        # stall of 100-300 ms whenever the caching allocator has to make room
        self._pool_key = (self.device.type, torch.cuda.current_device() if self.device.index is None else self.device.index,
                          self.depth)
        self._copy_stream, self._slots = None, None      # taken from the pool for the duration of one iteration
        self.last_event = None          # CUDA event after which the tensors of the batch yielded last are complete

    _pool: Dict[tuple, list] = {}

    def _acquire(self):
        pooled = DevicePrefetcher._pool.get(self._pool_key)
        if pooled:
            self._copy_stream, self._slots = pooled.pop()
        else:
            self._copy_stream = torch.cuda.Stream(self.device)
            self._slots = [_Slot(self.device) for _ in range(self.depth + 1)]

    def _release(self):
        """Hand stream and slots to the next prefetcher of this device (their last consumer is ordered by ``free_event``)."""
        if self._slots is not None:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            for s in self._slots:
                s.free_event = ev
            DevicePrefetcher._pool.setdefault(self._pool_key, []).append((self._copy_stream, self._slots))
            self._slots = None

    def _stage(self, host: Dict[str, torch.Tensor], slot: _Slot):
        if all(v.is_cuda for v in host.values() if isinstance(v, torch.Tensor)):
            # already on the device (ArenaLoader): nothing to stage; an overlapped assembly brings its own event
            return host, getattr(host, "ready_event", None), None, None
        shape_only = None
        if self.hot_path_only:
            kept = {k: v for k, v in host.items() if k not in self._unread}
            if getattr(host, "blob", None) is not None:      # a PackedBatch stays one (its buffer holds the hot path only)
                kept = type(host)(kept)
                kept.blob, kept.layout = host.blob, host.layout
            host = kept
            if isinstance(host.get("x_frags"), torch.Tensor):
                shape_only = host.pop("x_frags")
        dev, ev, pinned, slot = self._stage_tensors(host, slot)
        if shape_only is not None:
            dev["x_frags"] = torch.empty(shape_only.shape, dtype=torch.float32, device="meta")
        return dev, ev, pinned, slot

    def _stage_packed(self, host, slot: _Slot):
        """A ``PackedBatch`` (dataset.data.pack_batch): the tensors of the hot path travel as ONE copy of its buffer."""
        packed = host if host.blob.is_pinned() else host.pin_memory()
        blob, layout = packed.blob, packed.layout
        in_blob = {k for k, *_ in layout}
        widen = {k: _wide_dtype(k, packed[k]) for k in in_blob if _wide_dtype(k, packed[k]) != packed[k].dtype}
        dev_blob, wire, dev, grew = slot.packed_views(blob, layout, widen)
        rest = {k: v for k, v in packed.items() if k not in in_blob}     # tensors outside the buffer, non-tensor entries
        cs = self._copy_stream
        if slot.free_event is not None:
            cs.wait_event(slot.free_event)
        if grew:
            cs.wait_stream(torch.cuda.current_stream(self.device))
        keep = [packed]
        with torch.cuda.stream(cs):
            dev_blob.copy_(blob, non_blocking=True)
            jobs = [(wire[k], dev[k], _abi.WIDEN_U8_F32 if wire[k].dtype == torch.uint8 else _abi.WIDEN_I32_I64)
                    for k in widen if wire[k].numel()]
            for c in range(0, len(jobs), _abi.WIDEN_MAX_JOBS):
                chunk = jobs[c:c + _abi.WIDEN_MAX_JOBS]
                arr = (_abi.CWidenJob * len(chunk))(*[_abi.CWidenJob(s.data_ptr(), d.data_ptr(), s.numel(), m)
                                                      for s, d, m in chunk])
                _abi.check(_abi.load().fnb_widen_batch(arr, len(chunk), C.c_void_p(cs.cuda_stream)), "widen_batch")
            dev.update(rest)                   # non-tensor entries (every host tensor is inside the buffer here)
            ev = torch.cuda.Event()
            ev.record(cs)
        return dev, ev, keep, slot

    def _stage_tensors(self, host: Dict[str, torch.Tensor], slot: _Slot):
        if getattr(host, "blob", None) is not None:
            inside = {k for k, *_ in host.layout}
            if not any(isinstance(v, torch.Tensor) and not v.is_cuda for k, v in host.items() if k not in inside):
                return self._stage_packed(host, slot)    # (otherwise: tensor by tensor, like any other dict)
        pinned = {k: (v if (not isinstance(v, torch.Tensor) or v.is_cuda or v.is_pinned()) else v.pin_memory())
                  for k, v in host.items()}
        wire, dev, grew = slot.views(pinned)             # (re)allocation, if any, happens on the current stream
        cs = self._copy_stream
        if slot.free_event is not None:
            cs.wait_event(slot.free_event)               # the previous tenant of this slot has been consumed
        if grew:
            cs.wait_stream(torch.cuda.current_stream(self.device))   # stream-ordered reuse of freed memory
        jobs = []
        with torch.cuda.stream(cs):
            for k, v in pinned.items():
                if isinstance(v, torch.Tensor):
                    if v.is_cuda:
                        cs.wait_stream(torch.cuda.current_stream(self.device))   # its producer runs on the consumer's stream
                    wire[k].copy_(v, non_blocking=True)
                    if wire[k] is not dev[k] and v.numel():
                        jobs.append((wire[k], dev[k], _abi.WIDEN_U8_F32 if v.dtype == torch.uint8 else _abi.WIDEN_I32_I64))
            for c in range(0, len(jobs), _abi.WIDEN_MAX_JOBS):
                chunk = jobs[c:c + _abi.WIDEN_MAX_JOBS]
                arr = (_abi.CWidenJob * len(chunk))(*[_abi.CWidenJob(s.data_ptr(), d.data_ptr(), s.numel(), m)
                                                      for s, d, m in chunk])
                _abi.check(_abi.load().fnb_widen_batch(arr, len(chunk), C.c_void_p(cs.cuda_stream)), "widen_batch")
            ev = torch.cuda.Event()
            ev.record(cs)
        return dev, ev, pinned, slot                     # pinned host tensors stay alive until the copy was waited for

    def __iter__(self) -> Iterator[Dict[str, torch.Tensor]]:
        if self._slots is not None:
            raise RuntimeError("DevicePrefetcher: one iteration at a time")
        self._acquire()
        try:
            yield from self._iterate()
        finally:
            self._release()

    def _iterate(self) -> Iterator[Dict[str, torch.Tensor]]:
        it = iter(self.batches)
        queue = collections.deque()
        done, n_staged, last = False, 0, None
        while True:
            cur = torch.cuda.current_stream(self.device)
            if last is not None:                         # everything the consumer queued on the last batch precedes this
                last.free_event = torch.cuda.Event()
                last.free_event.record(cur)
                last = None
            while not done and len(queue) < self.depth:
                try:
                    host = next(it)
                except StopIteration:
                    done = True
                    break
                queue.append(self._stage(host, self._slots[n_staged % len(self._slots)]))
                n_staged += 1
            if not queue:
                return
            dev, ev, _pinned, slot = queue.popleft()
            if ev is not None:
                cur.wait_event(ev)
            else:                                        # produced on the consumer's stream (ArenaLoader)
                ev = torch.cuda.Event()
                ev.record(cur)
            self.last_event = ev                         # (for consumers that touch the batch from another stream)
            last = slot
            yield dev
