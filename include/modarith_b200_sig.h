/* modarith_b200_sig.h -- signature verification on top of the batched engine (C ABI).
 *
 * Same conventions as modarith_b200.h: device pointers, n independent rows, an optional cudaStream_t
 * (NULL = default stream), asynchronous calls, 0 or a cudaError_t / MAB_ERR_* value returned.
 */
#ifndef MODARITH_B200_SIG_H
#define MODARITH_B200_SIG_H

#include "modarith_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ECDSA over P-256 (SEC1 v2 section 4.1.4; the reference's NIST256_VERIFY, nist256.c), one signature per row.
 * h, r, s, qx, qy: n big-endian 32-byte strings each, row i at offset 32*i:
 *   h        the message digest, already cut to its leftmost 256 bits (bits2int); h >= n is reduced mod n
 *   r, s     the signature; rows with r or s outside [1, n-1] are invalid
 *   qx, qy   the public key; rows with a coordinate >= p or a point off the curve are invalid
 * ok[i] = 1 if row i is a valid signature, 0 if not.  Every row does the same work whatever its inputs.
 * n = 0 is a no-op. */
MAB_API int mab_NIST256_ecdsa_verify(const char *h, const char *r, const char *s, const char *qx, const char *qy,
                                     unsigned char *ok, size_t n, void *stream);

/* Ed25519 (RFC 8032 section 5.1.7, pure Ed25519, the cofactorless equation), one signature per row; byte strings
 * as RFC 8032 encodes them (little-endian), row i at offset 64*i (h, sig) or 32*i (pk):
 *   h        SHA-512(R || A || M), 64 bytes, reduced mod L here
 *   sig      R || S, 64 bytes; rows with S >= L are invalid; R is compared as bytes with the encoding of
 *            [S]B - [k]A (all 256 bits), never decoded
 *   pk       the public key A, 32 bytes; rows whose A does not decode strictly (y >= p, no square root,
 *            x = 0 with the sign bit set) are invalid
 * Small-order A and R are accepted where the equation holds.  ok[i] = 1 if row i is a valid signature, 0 if not.
 * Every row does the same work whatever its inputs.  n = 0 is a no-op. */
MAB_API int mab_ED25519_eddsa_verify(const char *h, const char *sig, const char *pk, unsigned char *ok,
                                     size_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MODARITH_B200_SIG_H */
