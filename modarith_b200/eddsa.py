"""Batched Ed25519 signature verification (RFC 8032 section 5.1.7, pure Ed25519) in one fused kernel per call
(include/modarith_b200_sig.h, mab_ED25519_eddsa_verify).

    ok = verify(messages, signatures, public_keys)          # 64-byte R || S signatures, 32-byte keys
    ok = verify_digest(h, sig, pk)                          # [n, 64] / [n, 64] / [n, 32] uint8 rows

The policy, pinned by the tests: S < L; A decoded strictly (y < p, a square root, not x = 0 with the sign bit);
k = SHA-512(R || A || M) mod L; valid iff the encoding of [S]B - [k]A equals the given R in all 256 bits (the
cofactorless equation: R is never decoded); small-order A and R are accepted where the equation holds.

`verify` hashes on the host with hashlib and makes one GPU call; a row whose signature is not 64 bytes or whose key is
not 32 bytes is not parsed and is False.  `verify_digest` takes the rows as they are: CUDA tensors are used in place
on the current stream, numpy arrays (or CPU tensors) go through the current device.  There is no CPU path.

    python -m modarith_b200.eddsa FILE      # a Wycheproof EddsaVerify file (edwards25519)
"""
from __future__ import annotations

import hashlib
from typing import Sequence

import numpy as np
import torch

from . import lib as _lib

__all__ = ["verify", "verify_digest", "prepare"]

KEY_BYTES = 32
SIG_BYTES = 64
DIGEST_BYTES = 64


def _args(h, sig, pk):
    arrays = [h, sig, pk]
    on_device = all(isinstance(t, torch.Tensor) and t.is_cuda for t in arrays)
    if not on_device:
        if any(isinstance(t, torch.Tensor) and t.is_cuda for t in arrays):
            raise ValueError("mixed host and device arguments")
        arrays = [t.contiguous() if isinstance(t, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(t))
                  for t in arrays]
    n = arrays[0].shape[0] if arrays[0].dim() >= 1 else -1
    for name, t, nb in zip(("h", "sig", "pk"), arrays, (DIGEST_BYTES, SIG_BYTES, KEY_BYTES)):
        if t.dtype != torch.uint8 or t.dim() != 2 or tuple(t.shape) != (n, nb) or not t.is_contiguous():
            raise ValueError("%s must be a contiguous [n, %d] uint8 array (h, sig, pk with the same n)" % (name, nb))
        if t.device != arrays[0].device:
            raise ValueError("arguments live on different devices")
    if not on_device:
        if not torch.cuda.is_available():
            raise _lib.MabError("modarith_b200 needs a CUDA device: there is no CPU fallback")
        arrays = [t.cuda() for t in arrays]
    return arrays, on_device


def verify_digest(h, sig, pk, ok=None):
    """ok[i] = whether sig[i] = R || S is a valid signature under the key pk[i] for h[i] = SHA-512(R || A || M).

    h: [n, 64], sig: [n, 64], pk: [n, 32] uint8 arrays, byte strings as RFC 8032 encodes them.  CUDA tensors give a
    CUDA bool tensor (written into `ok`, a contiguous [n] uint8 or bool CUDA tensor, when one is given); host arrays
    give a numpy bool array.  An all-zero row is not guaranteed to be rejected (the zero encoding is a point of order
    4): rows that did not parse must be masked by the caller, as `verify` does."""
    arrays, on_device = _args(h, sig, pk)
    h = arrays[0]
    n = h.shape[0]
    if ok is None:
        ok = torch.empty(n, dtype=torch.uint8, device=h.device)
    elif not on_device:
        raise ValueError("ok can only be supplied with device tensors (host arguments get a fresh numpy result)")
    elif not isinstance(ok, torch.Tensor) or not ok.is_cuda or ok.dtype not in (torch.uint8, torch.bool) \
            or tuple(ok.shape) != (n,) or ok.device != h.device or not ok.is_contiguous():
        raise ValueError("ok must be a contiguous uint8 or bool CUDA tensor of shape (%d,) on %s" % (n, h.device))
    lib = _lib.load()
    stream = torch.cuda.current_stream(h.device).cuda_stream
    with torch.cuda.device(h.device):
        _lib.check(lib.mab_ED25519_eddsa_verify(*(t.data_ptr() for t in arrays), ok.data_ptr(), n, stream),
                   "mab_ED25519_eddsa_verify")
    ok = ok.view(torch.bool)
    return ok if on_device else ok.cpu().numpy()


def prepare(messages: Sequence[bytes], signatures: Sequence[bytes], public_keys: Sequence[bytes]):
    """The rows `verify` sends to the GPU: (h [n, 64], sig [n, 64], pk [n, 32]) uint8 arrays and parsed[n].  A row
    whose signature is not 64 bytes or whose key is not 32 bytes is all zeros and parsed False."""
    n = len(messages)
    if len(signatures) != n or len(public_keys) != n:
        raise ValueError("messages, signatures and public_keys must have the same length")
    h = np.zeros((n, DIGEST_BYTES), dtype=np.uint8)
    sig = np.zeros((n, SIG_BYTES), dtype=np.uint8)
    pk = np.zeros((n, KEY_BYTES), dtype=np.uint8)
    parsed = np.zeros(n, dtype=bool)
    for i in range(n):
        s, a = bytes(signatures[i]), bytes(public_keys[i])
        if len(s) != SIG_BYTES or len(a) != KEY_BYTES:
            continue
        h[i] = np.frombuffer(hashlib.sha512(s[:32] + a + bytes(messages[i])).digest(), dtype=np.uint8)
        sig[i] = np.frombuffer(s, dtype=np.uint8)
        pk[i] = np.frombuffer(a, dtype=np.uint8)
        parsed[i] = True
    return (h, sig, pk), parsed


def verify(messages: Sequence[bytes], signatures: Sequence[bytes], public_keys: Sequence[bytes]) -> np.ndarray:
    """bool[n]: whether signatures[i] (R || S, 64 bytes) is a valid Ed25519 signature of messages[i] under
    public_keys[i] (32 bytes)."""
    rows, parsed = prepare(messages, signatures, public_keys)
    if len(parsed) == 0:
        return parsed
    return verify_digest(*rows) & parsed


def main(argv=None):
    """`python -m modarith_b200.eddsa FILE`: every edwards25519 test of a Wycheproof EdDSA file through the GPU."""
    import sys
    from .wire import load_eddsa_vectors, run_eddsa_vectors

    argv = sys.argv[1:] if argv is None else argv
    if len(argv) != 1:
        print("usage: python -m modarith_b200.eddsa <wycheproof eddsa file>", file=sys.stderr)
        return 2
    vecs = load_eddsa_vectors(argv[0])
    ok, passed = run_eddsa_vectors(vecs)
    for v, good, p in zip(vecs, ok, passed):
        if not p:
            print("FAILED tcId %d (%s, verified %s): %s" % (v.tc_id, v.result, bool(good), v.comment))
    acc = [bool(good) for v, good in zip(vecs, ok) if v.result == "acceptable"]
    count = lambda kind: sum(1 for v in vecs if v.result == kind)
    npass = lambda kind: sum(1 for v, p in zip(vecs, passed) if v.result == kind and p)
    print("Ed25519: %d tests; valid %d/%d verified, invalid %d/%d rejected, acceptable %d (%d verified)"
          % (len(vecs), npass("valid"), count("valid"), npass("invalid"), count("invalid"), len(acc), sum(acc)))
    return 0 if passed.all() else 1


if __name__ == "__main__":
    raise SystemExit(main())
