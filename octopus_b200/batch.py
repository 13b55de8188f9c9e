"""Struct-of-arrays packing of haplotypes and reads — the memory layout of include/phmm_b200.h.

A *block* keeps every per-base array concatenated in one contiguous numpy array plus an int64 offset array, i.e.
exactly what ``phmm_haplotypes`` / ``phmm_reads`` point at. Blocks can be moved to the GPU as torch tensors
(``to_device``) so that a call can run on inputs already resident in HBM.
"""
import ctypes as C

import numpy as np

from . import _lib


def _u8(x):
    if isinstance(x, str):
        x = x.encode()
    if isinstance(x, (bytes, bytearray)):
        return np.frombuffer(bytes(x), dtype=np.uint8)
    return np.ascontiguousarray(np.asarray(x)).view(np.uint8).reshape(-1)


def _concat(seqs, dtype):
    off = np.zeros(len(seqs) + 1, dtype=np.int64)
    parts = []
    for i, s in enumerate(seqs):
        a = _u8(s) if dtype == np.uint8 else np.ascontiguousarray(np.asarray(s, dtype=dtype)).reshape(-1)
        parts.append(a)
        off[i + 1] = off[i] + len(a)
    data = np.concatenate(parts) if parts else np.zeros(0, dtype=dtype)
    return np.ascontiguousarray(data.astype(dtype, copy=False)), off


class _Block:
    _fields = ()

    def arrays(self):
        return {f: getattr(self, f) for f in self._fields if getattr(self, f) is not None}

    def to_device(self, device="cuda:0"):
        """Copy of this block whose arrays are torch CUDA tensors (inputs resident in HBM)."""
        import torch
        out = object.__new__(type(self))
        out.__dict__.update(self.__dict__)
        for f in self._fields:
            a = getattr(self, f)
            if a is not None:
                t = torch.from_numpy(np.ascontiguousarray(a))
                setattr(out, f, t.to(device, non_blocking=False))
        out.on_device = True
        return out

    def pin(self):
        """Copy of this block in page-locked host memory (torch pinned tensors viewed as numpy)."""
        import torch
        out = object.__new__(type(self))
        out.__dict__.update(self.__dict__)
        keep = []
        for f in self._fields:
            a = getattr(self, f)
            if a is not None:
                t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
                keep.append(t)
                setattr(out, f, t.numpy())
        out._pinned = keep
        return out


def _ptr(a):
    if a is None:
        return None
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return a.ctypes.data


class HaplotypeBlock(_Block):
    """H haplotypes: what HaplotypeLikelihoodModel::reset computes per haplotype (haplotype_likelihood_model.cpp:60-78)."""
    _fields = ("off", "seq", "snv_mask_fwd", "snv_prior_fwd", "snv_mask_rev", "snv_prior_rev", "gap_open", "gap_extend", "begin")

    def __init__(self, off, seq, snv_mask_fwd, snv_prior_fwd, snv_mask_rev, snv_prior_rev, gap_open, gap_extend, begin=None):
        self.n = len(off) - 1
        self.off = np.ascontiguousarray(off, dtype=np.int64)
        self.seq = np.ascontiguousarray(seq, dtype=np.uint8)
        self.snv_mask_fwd = np.ascontiguousarray(snv_mask_fwd, dtype=np.uint8)
        self.snv_prior_fwd = np.ascontiguousarray(snv_prior_fwd, dtype=np.int8)
        self.snv_mask_rev = np.ascontiguousarray(snv_mask_rev, dtype=np.uint8)
        self.snv_prior_rev = np.ascontiguousarray(snv_prior_rev, dtype=np.int8)
        self.gap_open = np.ascontiguousarray(gap_open, dtype=np.int8)
        self.gap_extend = np.ascontiguousarray(gap_extend, dtype=np.int8)
        self.begin = None if begin is None else np.ascontiguousarray(begin, dtype=np.int64)
        self.on_device = False
        total = int(self.off[-1])
        for f in self._fields[1:8]:
            assert len(getattr(self, f)) == total, f

    def c_struct(self):
        s = _lib.Haplotypes()
        s.n = self.n
        for f in self._fields:
            setattr(s, f, _ptr(getattr(self, f)))
        return s

    def length(self, h):
        return int(self.off[h + 1] - self.off[h])

    def hap(self, h):
        """Host-side view of haplotype h's arrays (dict of numpy slices)."""
        a, b = int(self.off[h]), int(self.off[h + 1])
        return {f: getattr(self, f)[a:b] for f in self._fields[1:8]}


class ReadBlock(_Block):
    """R reads: the AlignedRead fields the path consumes (basics/aligned_read.hpp:36-39,120-146)."""
    _fields = ("off", "bases", "quals", "mapq", "reverse", "begin")

    def __init__(self, off, bases, quals, mapq=None, reverse=None, begin=None):
        self.n = len(off) - 1
        self.off = np.ascontiguousarray(off, dtype=np.int64)
        self.bases = np.ascontiguousarray(bases, dtype=np.uint8)
        self.quals = np.ascontiguousarray(quals, dtype=np.uint8)
        self.mapq = np.full(self.n, 60, dtype=np.uint8) if mapq is None else np.ascontiguousarray(mapq, dtype=np.uint8)
        self.reverse = np.zeros(self.n, dtype=np.uint8) if reverse is None else np.ascontiguousarray(reverse, dtype=np.uint8)
        self.begin = np.zeros(self.n, dtype=np.int64) if begin is None else np.ascontiguousarray(begin, dtype=np.int64)
        self.on_device = False
        assert len(self.bases) == len(self.quals) == int(self.off[-1])

    def c_struct(self):
        s = _lib.Reads()
        s.n = self.n
        for f in self._fields:
            setattr(s, f, _ptr(getattr(self, f)))
        return s

    def length(self, r):
        return int(self.off[r + 1] - self.off[r])

    def read(self, r):
        a, b = int(self.off[r]), int(self.off[r + 1])
        return self.bases[a:b], self.quals[a:b]


def pack_haplotypes(seqs, snv_mask_fwd, snv_prior_fwd, snv_mask_rev, snv_prior_rev, gap_open, gap_extend, begin=None):
    """Lists (one entry per haplotype) → HaplotypeBlock."""
    seq, off = _concat(seqs, np.uint8)
    mf, _ = _concat(snv_mask_fwd, np.uint8)
    pf, _ = _concat(snv_prior_fwd, np.int8)
    mr, _ = _concat(snv_mask_rev, np.uint8)
    pr, _ = _concat(snv_prior_rev, np.int8)
    go, _ = _concat(gap_open, np.int8)
    ge, _ = _concat(gap_extend, np.int8)
    return HaplotypeBlock(off, seq, mf, pf, mr, pr, go, ge, begin)


def pack_reads(bases, quals, mapq=None, reverse=None, begin=None):
    b, off = _concat(bases, np.uint8)
    q, _ = _concat(quals, np.uint8)
    return ReadBlock(off, b, q, mapq, reverse, begin)


def pack_positions(position_lists, H, R):
    """position_lists[h][r] → (off[H*R+1] int64, pos int32) in [H][R] order (phmm_positions)."""
    off = np.zeros(H * R + 1, dtype=np.int64)
    flat = []
    i = 0
    for h in range(H):
        for r in range(R):
            p = position_lists[h][r]
            flat.extend(int(x) for x in p)
            off[i + 1] = off[i] + len(p)
            i += 1
    return off, np.asarray(flat if flat else [0], dtype=np.int32)[:max(len(flat), 1)]


def concat_blocks(hap_blocks, read_blocks):
    """Regions back to back for PairHMMEngine.populate_regions: (HaplotypeBlock, ReadBlock, hap_first, read_first) (host blocks)."""
    def cat_off(blocks):
        off, base = [np.zeros(1, dtype=np.int64)], 0
        for b in blocks:
            off.append(b.off[1:] + base)
            base += int(b.off[-1])
        return np.concatenate(off)
    cat = lambda blocks, f: np.concatenate([getattr(b, f) for b in blocks])     # noqa: E731
    haps = HaplotypeBlock(cat_off(hap_blocks), *[cat(hap_blocks, f) for f in HaplotypeBlock._fields[1:8]],
                          np.concatenate([b.begin if b.begin is not None else np.zeros(b.n, dtype=np.int64) for b in hap_blocks]))
    reads = ReadBlock(cat_off(read_blocks), cat(read_blocks, "bases"), cat(read_blocks, "quals"), cat(read_blocks, "mapq"),
                      cat(read_blocks, "reverse"), cat(read_blocks, "begin"))
    hap_first = np.concatenate([[0], np.cumsum([b.n for b in hap_blocks])]).astype(np.int32)
    read_first = np.concatenate([[0], np.cumsum([b.n for b in read_blocks])]).astype(np.int32)
    return haps, reads, hap_first, read_first


def concat_templates(per_region_template_offs):
    """Templates of regions back to back, matching ``concat_blocks``: region g's template_off (local: from 0 to its read count) →
    (template_off over the concatenated reads, int64; template_first over the regions, int32) — PairHMMEngine.populate_regions'
    ``templates`` argument."""
    offs = [np.asarray(o, dtype=np.int64) for o in per_region_template_offs]
    parts, base = [np.zeros(1, dtype=np.int64)], 0
    for o in offs:
        if len(o) < 2 or o[0] != 0 or (np.diff(o) < 0).any():
            raise ValueError("a region's template offsets must start at 0, be non-decreasing and hold at least one template")
        parts.append(o[1:] + base)
        base += int(o[-1])
    template_first = np.concatenate([[0], np.cumsum([len(o) - 1 for o in offs])]).astype(np.int32)
    return np.concatenate(parts), template_first
