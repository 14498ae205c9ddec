"""Digests that stand in for large golden tensors.

The reference run's weights and logits are megabytes; the oracle regenerates them exactly from a seed, so the fixture keeps
their SHA-256 instead and the tests recompute the tensors and compare digests: still a bit-for-bit comparison, a few bytes stored.
"""
import hashlib

import torch


def tensor_sha256(t: torch.Tensor) -> str:
    """Digest of dtype, shape and raw bytes."""
    t = t.detach().cpu().contiguous()
    h = hashlib.sha256(f"{t.dtype} {tuple(t.shape)}".encode())
    h.update(t.reshape(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()


def state_sha256(module: torch.nn.Module) -> str:
    """Digest of every state_dict entry (name + tensor digest), in name order."""
    h = hashlib.sha256()
    for k, v in sorted(module.state_dict().items()):
        h.update(k.encode())
        h.update(tensor_sha256(v).encode())
    return h.hexdigest()
