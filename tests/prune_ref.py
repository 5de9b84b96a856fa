"""NumPy statement of the contract of ipr_prune_magnitude_f32 (csrc/prune.cu), shared by the host and GPU tests.

Keys are |w| as 31-bit integers (+-0 share 0, every NaN one key above +inf); the threshold T is the k-th smallest key,
found digit by digit (11 / 10 / 10 bits) as the kernel does; every key < T is pruned, and of the keys == T the
``need`` with the lowest arena index.  A pruned entry becomes w * 0."""
import numpy as np


def magnitude_keys(w):
    k = np.ascontiguousarray(w, dtype=np.float32).view(np.uint32) & np.uint32(0x7fffffff)
    return np.where(k > 0x7f800000, np.uint32(0x7fffffff), k).astype(np.uint32)


def radix_threshold(keys, k):
    """-> (T, need): the k-th smallest key (k >= 1) and how many entries equal to it are pruned."""
    keys = keys.astype(np.int64)
    rank, prefix = k - 1, 0
    for shift, bits in ((20, 11), (10, 10), (0, 10)):
        sel = keys[(keys >> (shift + bits)) == prefix]
        hist = np.bincount((sel >> shift) & ((1 << bits) - 1), minlength=1 << bits)
        cum = np.cumsum(hist)
        b = int(np.searchsorted(cum, rank, side="right"))
        rank -= int(cum[b] - hist[b])
        prefix = (prefix << bits) | b
    return prefix, rank + 1


def segment_index(segments):
    return np.concatenate([np.arange(o, o + c, dtype=np.int64) for o, c in segments])


def prune_mask(w, k):
    """Boolean mask (True = pruned) over the virtual entries w (segment order)."""
    mask = np.zeros(w.shape[0], dtype=bool)
    if k == 0:
        return mask
    keys = magnitude_keys(w)
    T, need = radix_threshold(keys, k)
    mask[keys < T] = True
    mask[np.flatnonzero(keys == T)[:need]] = True
    return mask


def prune_emulate(arena, segments, k):
    """The arena after ipr_prune_magnitude_f32 (float32 copy)."""
    out = np.array(arena, dtype=np.float32, copy=True)
    idx = segment_index(segments)
    w = out[idx]
    m = prune_mask(w, k)
    with np.errstate(invalid="ignore"):
        out[idx[m]] = w[m] * np.float32(0.0)
    return out
