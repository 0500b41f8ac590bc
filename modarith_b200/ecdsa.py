"""Batched ECDSA signature verification over P-256 (SEC1 v2 section 4.1.4; the reference's NIST256_VERIFY, nist256.c)
in one fused kernel per call (include/modarith_b200_sig.h, mab_NIST256_ecdsa_verify).

    ok = verify(messages, signatures, public_keys)                       # DER signatures, SHA-256
    ok = verify(messages, signatures, public_keys, hash="sha384", encoding="p1363")
    ok = verify_digest(h, r, s, qx, qy)                                   # [n, 32] uint8 rows, big-endian

`verify` prepares the rows on the host -- hashes with hashlib, keeps the leftmost 256 bits of the digest (bits2int),
decodes strict DER or raw r||s signatures and SEC1 uncompressed public keys (04 || X || Y) -- and makes one GPU call.
A row that does not parse is False.  `verify_digest` takes the prepared rows: CUDA tensors are used in place on the
current stream, numpy arrays (or CPU tensors) go through the current device.  There is no CPU path.

    python -m modarith_b200.ecdsa FILE      # a Wycheproof EcdsaVerify / EcdsaP1363Verify file (secp256r1)
"""
from __future__ import annotations

import hashlib
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import lib as _lib
from .ecn import _args

__all__ = ["verify", "verify_digest", "decode_der", "decode_p1363", "decode_public_key", "digest_int", "prepare"]

NBYTES = 32
ENCODINGS = ("der", "p1363")


def verify_digest(h, r, s, qx, qy, ok=None):
    """ok[i] = whether (r[i], s[i]) is a valid signature of digest h[i] under the key (qx[i], qy[i]).

    Every argument is an [n, 32] uint8 array of big-endian values.  h is the digest already cut to its leftmost 256
    bits.  CUDA tensors give a CUDA bool tensor (written into `ok`, a contiguous [n] uint8 or bool CUDA tensor, when
    one is given); host arrays give a numpy bool array."""
    arrays, on_device = _args("NIST256", [h, r, s, qx, qy])
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
        _lib.check(lib.mab_NIST256_ecdsa_verify(*(t.data_ptr() for t in arrays), ok.data_ptr(), n, stream),
                   "mab_NIST256_ecdsa_verify")
    ok = ok.view(torch.bool)
    return ok if on_device else ok.cpu().numpy()


# ---- host-side preparation ---------------------------------------------------------------------------------------
def _der_length(b: bytes, i: int) -> Tuple[int, int]:
    """A DER definite length at b[i]: (length, index after it).  Long forms are accepted only where the short form
    cannot express the length (X.690 10.1); indefinite length (0x80) is not DER."""
    if i >= len(b):
        raise ValueError("truncated")
    first = b[i]
    if first < 0x80:
        return first, i + 1
    k = first & 0x7F
    if k == 0 or k > 4 or i + 1 + k > len(b):
        raise ValueError("bad length")
    v = int.from_bytes(b[i + 1:i + 1 + k], "big")
    if b[i + 1] == 0 or v < 0x80:
        raise ValueError("non-minimal length")
    return v, i + 1 + k


def _der_uint(b: bytes, i: int) -> Tuple[int, int]:
    if i >= len(b) or b[i] != 0x02:
        raise ValueError("INTEGER expected")
    ln, i = _der_length(b, i + 1)
    v = b[i:i + ln]
    if ln == 0 or len(v) != ln:
        raise ValueError("bad INTEGER")
    if v[0] & 0x80:
        raise ValueError("negative INTEGER")
    if ln > 1 and v[0] == 0 and not v[1] & 0x80:
        raise ValueError("non-minimal INTEGER")
    return int.from_bytes(v, "big"), i + ln


def decode_der(sig: bytes) -> Tuple[int, int]:
    """Ecdsa-Sig-Value ::= SEQUENCE { r INTEGER, s INTEGER } in strict DER: minimal lengths and integers, both
    non-negative, nothing after the sequence.  Raises ValueError otherwise."""
    sig = bytes(sig)
    if len(sig) < 2 or sig[0] != 0x30:
        raise ValueError("SEQUENCE expected")
    ln, i = _der_length(sig, 1)
    if i + ln != len(sig):
        raise ValueError("SEQUENCE length does not match")
    r, i = _der_uint(sig, i)
    s, i = _der_uint(sig, i)
    if i != len(sig):
        raise ValueError("trailing data in SEQUENCE")
    return r, s


def decode_p1363(sig: bytes) -> Tuple[int, int]:
    """IEEE P1363 r || s, 32 big-endian bytes each."""
    sig = bytes(sig)
    if len(sig) != 2 * NBYTES:
        raise ValueError("a P1363 signature over P-256 is 64 bytes")
    return int.from_bytes(sig[:NBYTES], "big"), int.from_bytes(sig[NBYTES:], "big")


def decode_public_key(key: bytes) -> Tuple[int, int]:
    """SEC1 uncompressed point 04 || X || Y (X, Y: 32 bytes each); the values themselves are checked on the GPU."""
    key = bytes(key)
    if len(key) != 1 + 2 * NBYTES or key[0] != 0x04:
        raise ValueError("an uncompressed P-256 key is 04 || X || Y (65 bytes)")
    return int.from_bytes(key[1:1 + NBYTES], "big"), int.from_bytes(key[1 + NBYTES:], "big")


def digest_int(digest: bytes) -> int:
    """bits2int (SEC1 v2 4.1.3 step 5): the leftmost 256 bits of the digest."""
    v = int.from_bytes(digest, "big")
    extra = 8 * len(digest) - 8 * NBYTES
    return v >> extra if extra > 0 else v


def prepare(messages: Sequence[bytes], signatures: Sequence[bytes], public_keys: Sequence[bytes],
            hash: Optional[str] = "sha256", encoding: str = "der"):
    """The rows `verify` sends to the GPU: (h, r, s, qx, qy) as [n, 32] uint8 arrays and parsed[n].  A row whose
    signature or key does not parse, or whose r or s does not fit 256 bits, is all zeros (which the kernel rejects)
    and parsed False.  hash=None: the messages are digests already."""
    if encoding not in ENCODINGS:
        raise ValueError("encoding must be one of %s" % (ENCODINGS,))
    n = len(messages)
    if len(signatures) != n or len(public_keys) != n:
        raise ValueError("messages, signatures and public_keys must have the same length")
    if hash is not None:
        hashlib.new(hash)                                        # unknown names raise here, before any work
    decode = decode_der if encoding == "der" else decode_p1363
    rows = np.zeros((5, n, NBYTES), dtype=np.uint8)
    parsed = np.zeros(n, dtype=bool)
    top = 1 << (8 * NBYTES)
    for i in range(n):
        try:
            r, s = decode(signatures[i])
            qx, qy = decode_public_key(public_keys[i])
        except ValueError:
            continue
        if r >= top or s >= top:
            continue
        d = bytes(messages[i]) if hash is None else hashlib.new(hash, bytes(messages[i])).digest()
        for k, v in enumerate((digest_int(d), r, s, qx, qy)):
            rows[k, i] = np.frombuffer(v.to_bytes(NBYTES, "big"), dtype=np.uint8)
        parsed[i] = True
    return tuple(rows), parsed


def verify(messages: Sequence[bytes], signatures: Sequence[bytes], public_keys: Sequence[bytes], hash: Optional[str] = "sha256",
           encoding: str = "der") -> np.ndarray:
    """bool[n]: whether signatures[i] is a valid ECDSA P-256 signature of messages[i] under public_keys[i].

    hash: a hashlib name ("sha256", "sha384", "sha512", "sha3_256", ...), or None when the messages are digests
    already; encoding: "der" (strict DER Ecdsa-Sig-Value) or "p1363" (r || s); keys: SEC1 uncompressed, 65 bytes."""
    rows, parsed = prepare(messages, signatures, public_keys, hash, encoding)
    if len(parsed) == 0:
        return parsed
    return verify_digest(*rows) & parsed


def main(argv=None):
    """`python -m modarith_b200.ecdsa FILE`: every secp256r1 test of a Wycheproof ECDSA file through the GPU."""
    import sys
    from .wire import load_ecdsa_vectors, run_ecdsa_vectors

    argv = sys.argv[1:] if argv is None else argv
    if len(argv) != 1:
        print("usage: python -m modarith_b200.ecdsa <wycheproof ecdsa file>", file=sys.stderr)
        return 2
    vecs = load_ecdsa_vectors(argv[0])
    ok, passed = run_ecdsa_vectors(vecs)
    for v, good, p in zip(vecs, ok, passed):
        if not p:
            print("FAILED tcId %d (%s, verified %s): %s" % (v.tc_id, v.result, bool(good), v.comment))
    acc = [bool(good) for v, good in zip(vecs, ok) if v.result == "acceptable"]
    count = lambda kind: sum(1 for v in vecs if v.result == kind)
    npass = lambda kind: sum(1 for v, p in zip(vecs, passed) if v.result == kind and p)
    print("ECDSA P-256: %d tests; valid %d/%d verified, invalid %d/%d rejected, acceptable %d (%d verified)"
          % (len(vecs), npass("valid"), count("valid"), npass("invalid"), count("invalid"), len(acc), sum(acc)))
    return 0 if passed.all() else 1


if __name__ == "__main__":
    raise SystemExit(main())
