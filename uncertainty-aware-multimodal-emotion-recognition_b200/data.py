"""Batch wire format + device staging around the hot path (SURVEY.md section 8 row f2).

Wire format (reference: src/data/preprocessing.py:461-491 collate dict, src/models/multi_dataset_framework.py:85-103;
the driver's synthetic loader yields 4-tuples, experiments/run_multimodal_deer.py:329-349):

    {"audio_features", "video_features", "text_features", "targets"[, "attention_mask", "linguistic_features",
     "target_mask", "dataset_id"]}           or           (audio, video, text, targets)

"target_mask" (the targets' shape, bool / uint8, nonzero = labelled) marks the targets a partially labelled batch
has; it keeps its dtype on the device.

`DevicePrefetcher` turns any iterable of such HOST batches into device batches whose H2D copies overlap the compute of
the previous step: `depth` rotating sets of STATIC device buffers per batch signature (static addresses, so the
trainer's CUDA graph of a step can be captured once per buffer set and replayed), a dedicated copy stream, pinned
staging, and event edges in both directions (a buffer set is refilled only after the step that read it has finished).
At the BASELINE shapes a B=256 sequence batch is 89 MB: 1.6 ms of PCIe Gen5 time hidden behind a 4 ms step.
"""
from __future__ import annotations

from typing import Dict, Iterable, Iterator, Optional

import torch

BATCH_KEYS = ("audio_features", "video_features", "text_features", "targets")
OPTIONAL_KEYS = ("attention_mask", "linguistic_features", "target_mask", "dataset_id")


def as_batch_dict(batch) -> Dict[str, torch.Tensor]:
    """Normalise the reference's two batch shapes to the dict schema (tensors only)."""
    if isinstance(batch, dict):
        out = {k: v for k, v in batch.items() if torch.is_tensor(v)}
        for short, full in (("audio", "audio_features"), ("video", "video_features"), ("text", "text_features")):
            if short in out and full not in out:
                out[full] = out.pop(short)
        return out
    if isinstance(batch, (tuple, list)) and len(batch) == 4:
        return dict(zip(BATCH_KEYS, batch))
    raise TypeError("deer_b200: a batch is the reference's feature dict or the driver's (audio, video, text, targets)")


class _BufferSet:
    def __init__(self, like: Dict[str, torch.Tensor], device):
        self.tensors = {k: torch.empty(v.shape, dtype=_device_dtype(k, v), device=device) for k, v in like.items()}
        self.ready = torch.cuda.Event()      # H2D copies of the current contents have completed
        self.consumed = torch.cuda.Event()   # the step that read the current contents has completed
        self.consumed.record()


def _device_dtype(key: str, v: torch.Tensor):
    # features / targets / masks travel as fp32 (the kernels' input type); ids stay integer
    return torch.float32 if (v.is_floating_point() or key == "attention_mask") else v.dtype


class DevicePrefetcher:
    """for dev_batch in DevicePrefetcher(loader, device): ...   (dev_batch tensors live in static device buffers).

    Call `release(dev_batch)` (or simply advance the iterator: it releases the previous batch on the CURRENT stream)
    after enqueueing the work that reads the batch.  `bytes_per_batch` is the H2D volume of the last staged batch."""

    def __init__(self, loader: Iterable, device, depth: int = 2, keys: Optional[Iterable[str]] = None):
        self.loader = loader
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("deer_b200.data.DevicePrefetcher stages batches for a CUDA device (no CPU path)")
        self.depth = max(2, int(depth))
        self.keys = None if keys is None else tuple(keys)
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self._sets: Dict[tuple, list] = {}
        self._turn: Dict[tuple, int] = {}
        self._pinned: Dict[tuple, list] = {}
        self.bytes_per_batch = 0

    def __len__(self):
        return len(self.loader)

    # ------------------------------------------------------------------ staging
    def _signature(self, b: Dict[str, torch.Tensor]) -> tuple:
        return tuple(sorted((k, tuple(v.shape), str(v.dtype)) for k, v in b.items()))

    def stage(self, host_batch) -> Dict[str, torch.Tensor]:
        """Enqueue the H2D copies of one host batch on the copy stream; returns the (static) device batch.  The caller
        must `wait(dev_batch)` on its compute stream before reading it."""
        b = as_batch_dict(host_batch)
        if self.keys is not None:
            b = {k: b[k] for k in self.keys if k in b}
        sig = self._signature(b)
        sets = self._sets.get(sig)
        if sets is None:
            sets = self._sets[sig] = [_BufferSet(b, self.device) for _ in range(self.depth)]
            self._turn[sig] = 0
            self._pinned[sig] = [None] * self.depth
        j = self._turn[sig]
        self._turn[sig] = (j + 1) % self.depth
        bs = sets[j]
        nbytes = 0
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(bs.consumed)             # the step that last read these buffers is done
            for k, v in b.items():
                dst = bs.tensors[k]
                src = v if v.dtype == dst.dtype else v.to(dst.dtype)
                if not src.is_pinned():                          # pageable memory would make the copy synchronous
                    pin = self._pinned[sig][j]
                    if pin is None:
                        pin = self._pinned[sig][j] = {}
                    if k not in pin:
                        pin[k] = torch.empty(src.shape, dtype=src.dtype).pin_memory()
                    else:
                        bs.ready.synchronize()                   # the previous H2D copy out of this staging buffer
                    pin[k].copy_(src)
                    src = pin[k]
                dst.copy_(src, non_blocking=True)
                nbytes += dst.numel() * dst.element_size()
            bs.ready.record(self.copy_stream)
        self.bytes_per_batch = nbytes
        out = dict(bs.tensors)
        out["_buffer_set"] = bs
        return out

    @staticmethod
    def wait(dev_batch, stream=None):
        """Make `stream` (default: current) wait for the batch's H2D copies."""
        (stream or torch.cuda.current_stream()).wait_event(dev_batch["_buffer_set"].ready)

    @staticmethod
    def release(dev_batch, stream=None):
        """Record on `stream` (default: current) that everything enqueued so far has read the batch."""
        dev_batch["_buffer_set"].consumed.record(stream or torch.cuda.current_stream())

    @staticmethod
    def tensors(dev_batch) -> Dict[str, torch.Tensor]:
        return {k: v for k, v in dev_batch.items() if k != "_buffer_set"}

    # ------------------------------------------------------------------ iteration: one batch ahead
    def __iter__(self) -> Iterator[Dict[str, torch.Tensor]]:
        it = iter(self.loader)
        try:
            nxt = self.stage(next(it))
        except StopIteration:
            return
        prev = None
        while nxt is not None:
            cur = nxt
            if prev is not None:
                self.release(prev)               # the consumer has enqueued its work on the previous batch by now
            try:
                nxt = self.stage(next(it))       # the next batch's copies run beside the step on `cur`
            except StopIteration:
                nxt = None
            self.wait(cur)
            yield self.tensors(cur)
            prev = cur
        if prev is not None:
            self.release(prev)
