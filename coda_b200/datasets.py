"""Datasets: the reference loader contract (coda/datasets.py:4-23) plus shard-aware variants."""
from __future__ import annotations

import os

import torch

from .synth import shard_range, synth, synth_compact


def keep_fp16_default() -> bool:
    """``CODA_B200_KEEP_FP16=1`` makes ``keep_fp16=True`` the loaders' default (for drivers that build ``Dataset`` with
    the reference's two arguments, e.g. main.py through the ``coda`` shim)."""
    return os.environ.get("CODA_B200_KEEP_FP16", "0") == "1"


def _slab_dtype(t, keep_fp16):
    """fp16 scores stay fp16 with ``keep_fp16`` (the kernels read them as they are and compute in fp32: the run is
    bit-identical to one on the upcast slab, with half the memory); everything else is upcast to fp32 as the reference
    loader does (coda/datasets.py:14).  Nothing is ever rounded."""
    return torch.float16 if (keep_fp16 and t.dtype == torch.float16) else torch.float32


class Dataset:
    """(H, N, C) post-softmax scores from ``filepath`` (+ optional ``*_labels.pt``), forced to fp32
    (coda/datasets.py:12-23) unless ``keep_fp16`` keeps an fp16 file fp16 (default: ``CODA_B200_KEEP_FP16``)."""

    def __init__(self, filepath, device, keep_fp16=None):
        self.device = device
        keep = keep_fp16_default() if keep_fp16 is None else bool(keep_fp16)
        preds = torch.load(filepath, map_location=device)
        self.preds = preds.to(_slab_dtype(preds, keep)).contiguous()
        print("Loaded preds of shape", self.preds.shape)
        self.labels = None
        label_p = filepath.replace(".pt", "_labels.pt")
        if os.path.exists(label_p):
            self.labels = torch.load(label_p, map_location=device)
            print("Loaded labels of shape", self.labels.shape)
        else:
            print("Did not load labels.")


class TensorDataset:
    """Wrap tensors already in memory.  ``n_offset``/``n_global`` describe an N-axis shard."""

    def __init__(self, preds, labels=None, n_offset=0, n_global=None):
        self.preds, self.labels, self.device = preds, labels, preds.device
        self.n_offset = n_offset
        self.n_global = preds.shape[1] if n_global is None else n_global


class ShardedFileDataset(TensorDataset):
    """This rank's contiguous N-range of an (H, N, C) ``.pt`` slab, read through ``torch.load(mmap=True)`` so that
    no rank ever materialises the whole tensor (the reference loader, coda/datasets.py:14, loads all of it onto
    one device).  Labels (``*_labels.pt``, N int64) are small and replicated.  ``keep_fp16`` as for ``Dataset``."""

    def __init__(self, filepath, device, rank=0, world=1, keep_fp16=None):
        keep = keep_fp16_default() if keep_fp16 is None else bool(keep_fp16)
        full = torch.load(filepath, map_location="cpu", mmap=True, weights_only=True)
        if full.dim() != 3:
            raise ValueError(f"{filepath}: expected an (H, N, C) tensor, got shape {tuple(full.shape)}")
        n = int(full.shape[1])
        lo, hi = shard_range(n, rank, world)
        # avoid fp16 precision errors (coda/datasets.py:14): the kernels compute in fp32 whatever the storage type
        preds = full[:, lo:hi].to(_slab_dtype(full, keep)).contiguous().to(device)
        labels = None
        label_p = filepath.replace(".pt", "_labels.pt")
        if os.path.exists(label_p):
            labels = torch.load(label_p, map_location="cpu", weights_only=True)
        super().__init__(preds, labels, n_offset=lo, n_global=n)
        self.labels_host = labels


class SyntheticDataset(TensorDataset):
    """This rank's shard of the synthetic task (SURVEY.md 8d); labels are replicated (N int64)."""

    def __init__(self, H, N, C, seed=0, device="cuda", dense=False, rank=0, world=1, generator_device=None):
        lo, hi = shard_range(N, rank, world)
        gdev = generator_device or device
        preds, _ = synth(H, N, C, seed, device=gdev, dense=dense, n_lo=lo, n_hi=hi)
        _, labels = synth(H, N, C, seed, device=gdev, dense=dense, want_preds=False)
        super().__init__(preds.to(device), labels, n_offset=lo, n_global=N)
        self.labels_host = labels.cpu()


class CompactSlab:
    """Top-K + uniform-remainder form of an (H, N, C) score slab (``csrc/compact.cu``): ``ids`` (H, N, K) int16 holding
    uint16 class ids in descending score order, ``probs`` (H, N, K) float32; every other class of (h, n) gets
    ``(1 - sum_j probs) / (C - K)``.  24 bytes per (model, item) at K = 4 -- BASELINE.json configs[4] is 98 GB this way
    and 16.4 TB dense.  Duck-types the few tensor attributes the selector reads from ``dataset.preds``."""

    def __init__(self, ids: torch.Tensor, probs: torch.Tensor, C: int):
        if ids.shape != probs.shape or ids.dim() != 3 or ids.dtype != torch.int16 or probs.dtype != torch.float32:
            raise TypeError("CompactSlab: ids (H, N, K) int16 and probs (H, N, K) float32 expected")
        if ids.stride() != probs.stride() or ids.stride(2) != 1 or ids.stride(1) != ids.shape[2]:
            raise ValueError("CompactSlab: ids and probs must share strides, items contiguous")
        self.ids, self.probs, self.C = ids, probs, int(C)
        self.K = int(ids.shape[2])
        self.shape = (int(ids.shape[0]), int(ids.shape[1]), self.C)
        self.device = ids.device
        self.is_cuda = ids.is_cuda
        self.dtype = torch.float32

    def numel(self):
        return self.ids.numel() * 2          # what it costs relative to a dense float count (for the auto-shard rule)

    def narrow_items(self, lo, hi):
        return CompactSlab(self.ids[:, lo:hi], self.probs[:, lo:hi], self.C)

    def to(self, device):
        return CompactSlab(self.ids.to(device).contiguous(), self.probs.to(device).contiguous(), self.C)

    def densify(self) -> torch.Tensor:
        """The dense (H, N, C) float32 slab this form stands for (tests / small cases): same fp32 arithmetic for the
        remainder as the kernels (left-to-right sum of the K scores, 1 - s, times fp32(1 / (C - K)))."""
        H, N, C = self.shape
        s = self.probs[..., 0].clone()
        for j in range(1, self.K):
            s = s + self.probs[..., j]
        inv = torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(C - self.K), dtype=torch.float32)
        rest = (1.0 - s) * inv.to(s.device)
        dense = rest[..., None].expand(H, N, C).clone()
        dense.scatter_(2, (self.ids.to(torch.int64) & 0xFFFF), self.probs)
        return dense


class CompactDataset:
    def __init__(self, slab: CompactSlab, labels=None, n_offset=0, n_global=None):
        self.preds, self.labels, self.device = slab, labels, slab.device
        self.n_offset = n_offset
        self.n_global = slab.shape[1] if n_global is None else n_global


class SyntheticCompactDataset(CompactDataset):
    """This rank's shard of the synthetic task generated directly in the compact form (the dense slab never exists)."""

    def __init__(self, H, N, C, K=4, seed=0, device="cuda", rank=0, world=1):
        lo, hi = shard_range(N, rank, world)
        ids, probs, _ = synth_compact(H, N, C, K, seed, device=device, n_lo=lo, n_hi=hi)
        _, _, labels = synth_compact(H, N, C, K, seed, device=device, want_slab=False)
        super().__init__(CompactSlab(ids, probs, C), labels, n_offset=lo, n_global=N)
        self.labels_host = labels.cpu()
