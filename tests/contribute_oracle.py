"""Big-integer restatement of a Powers-of-Tau contribution (powersoftau `compute`, `keypair`, `hash_to_g2`,
`verify_transform`) over the field and curve code of oracle/ptau_oracle.py; the reference for tests/test_contribute.py.

Recalled, not vendored (the crates are not available offline): rand 0.4 ChaChaRng (RFC 7539 ChaCha20 block, 8 key
words, 128-bit block counter in words 12..15 from 0, u32 words in keystream order), rand 0.4's default next_u64 (first
u32 is the HIGH half), pairing 0.14.2 Fq::rand (six u64 limbs least significant first, top 3 bits cleared, rejection
while >= p, the limbs taken as the Montgomery representation) and G2::rand (x = Fq2::rand, greatest = next_u32 as u8
& 1, y with the largest test equal to greatest, times the full cofactor h2, retried while zero)."""
import hashlib

import pairing_oracle as po
import ptau_oracle as o

P, R = o.P, o.R_ORDER
_Z = -o.Z_ABS
H2 = (_Z**8 - 4 * _Z**7 + 5 * _Z**6 - 4 * _Z**4 + 6 * _Z**3 - 4 * _Z**2 - 4 * _Z + 13) // 9
_RINV = pow(1 << 384, -1, P)
# the secrets (tau, alpha, beta, s_tau, s_alpha, s_beta) of tests/golden/n8_contribution.bin (tools/make_golden.py);
# rust/tests/golden.rs states the same values
GOLDEN_SECRETS = (0x2A5F3C91D7E04B86, 0x6C1E9A74B3F2D058, 0x1F8B6E3D5A7C9042, 0x3B7D1F5E9C2A6084, 0x5E2C8A4F1D6B3097,
                  0x7A4E2C6F8B1D5039)
M32 = 0xFFFFFFFF


def _rotl(v, n):
    return ((v << n) | (v >> (32 - n))) & M32


def chacha_block(key_words, counter: int):
    """The ChaCha20 block (RFC 7539 2.3) with rand 0.4's state: constants, key, 128-bit counter, no nonce."""
    st = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574] + list(key_words) + [
        (counter >> (32 * i)) & M32 for i in range(4)]
    x = list(st)

    def qr(a, b, c, d):
        x[a] = (x[a] + x[b]) & M32; x[d] = _rotl(x[d] ^ x[a], 16)
        x[c] = (x[c] + x[d]) & M32; x[b] = _rotl(x[b] ^ x[c], 12)
        x[a] = (x[a] + x[b]) & M32; x[d] = _rotl(x[d] ^ x[a], 8)
        x[c] = (x[c] + x[d]) & M32; x[b] = _rotl(x[b] ^ x[c], 7)

    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    return [(a + b) & M32 for a, b in zip(x, st)]


class ChaChaRng:
    """rand 0.4 ChaChaRng::from_seed(key words)."""

    def __init__(self, key_words):
        self.key = list(key_words)
        self.ctr = 0
        self.buf = []

    def next_u32(self) -> int:
        if not self.buf:
            self.buf = chacha_block(self.key, self.ctr)
            self.ctr += 1
        return self.buf.pop(0)

    def next_u64(self) -> int:
        hi = self.next_u32()
        return (hi << 32) | self.next_u32()


def fq_rand(rng, stats=None) -> int:
    while True:
        v = 0
        for i in range(6):
            v |= rng.next_u64() << (64 * i)
        v &= (1 << 381) - 1
        if v < P:
            return v * _RINV % P
        if stats is not None:
            stats["rejected"] += 1


def hash_to_g2(digest: bytes, stats=None):
    """powersoftau hash_to_g2: affine point (None never: G2::rand retries while zero)."""
    key = [int.from_bytes(digest[4 * i:4 * i + 4], "big") for i in range(8)]
    rng = ChaChaRng(key)
    while True:
        x = (fq_rand(rng, stats), fq_rand(rng, stats))
        greatest = (rng.next_u32() & 0xFF) & 1 == 1
        y = o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2))
        if y is None:
            if stats is not None:
                stats["no_root"] += 1
            continue
        if o.fq2_lex_largest(y) != greatest:
            y = o.fq2_neg(y)
        q = o.g2_mul((x, y), H2)
        if q is not None:
            return q


def _g2_s(digest: bytes, pers: int, g1_s, g1_s_x):
    h = hashlib.blake2b(bytes([pers]) + digest + o.zcash_g1_uncompressed_encode(g1_s)
                        + o.zcash_g1_uncompressed_encode(g1_s_x)).digest()
    return hash_to_g2(h)


def public_key(digest: bytes, secrets) -> bytes:
    """powersoftau keypair with g1_s = [s]G1: 1152 bytes, uncompressed."""
    g1, g2 = [], []
    for i in range(3):
        x, s = secrets[i], secrets[3 + i]
        g1_s = o.g1_mul(o.G1_GEN, s)
        g1_s_x = o.g1_mul(g1_s, x)
        g1 += [g1_s, g1_s_x]
        g2.append(o.g2_mul(_g2_s(digest, i, g1_s, g1_s_x), x))
    return b"".join(o.zcash_g1_uncompressed_encode(q) for q in g1) + b"".join(
        o.zcash_g2_uncompressed_encode(q) for q in g2)


def serialize_challenge(acc: o.Accumulator, prefix: bytes) -> bytes:
    parts = [prefix]
    parts += [o.zcash_g1_uncompressed_encode(q) for q in acc.tau_g1]
    parts += [o.zcash_g2_uncompressed_encode(q) for q in acc.tau_g2]
    parts += [o.zcash_g1_uncompressed_encode(q) for q in acc.alpha_g1]
    parts += [o.zcash_g1_uncompressed_encode(q) for q in acc.beta_g1]
    parts.append(o.zcash_g2_uncompressed_encode(acc.beta_g2))
    return b"".join(parts)


def parse_challenge(data: bytes, n: int) -> o.Accumulator:
    off = 64
    out = []
    for count, size, dec in ((2 * n - 1, 96, o.zcash_g1_uncompressed_decode), (n, 192, o.zcash_g2_uncompressed_decode),
                             (n, 96, o.zcash_g1_uncompressed_decode), (n, 96, o.zcash_g1_uncompressed_decode),
                             (1, 192, o.zcash_g2_uncompressed_decode)):
        out.append([dec(data[off + i * size:off + (i + 1) * size]) for i in range(count)])
        off += count * size
    return o.Accumulator(out[0], out[1], out[2], out[3], out[4][0])


def parse_response(data: bytes, n: int):
    off = 64
    out = []
    for count, size, dec in ((2 * n - 1, 48, o.zcash_g1_compressed_decode), (n, 96, o.zcash_g2_compressed_decode),
                             (n, 48, o.zcash_g1_compressed_decode), (n, 48, o.zcash_g1_compressed_decode),
                             (1, 96, o.zcash_g2_compressed_decode)):
        out.append([dec(data[off + i * size:off + (i + 1) * size]) for i in range(count)])
        off += count * size
    pk = data[off:]
    g1 = [o.zcash_g1_uncompressed_decode(pk[96 * i:96 * i + 96]) for i in range(6)]
    g2 = [o.zcash_g2_uncompressed_decode(pk[576 + 192 * i:576 + 192 * i + 192]) for i in range(3)]
    return o.Accumulator(out[0], out[1], out[2], out[3], out[4][0]), g1, g2


def scalar_of(section: int, i: int, tau: int, alpha: int, beta: int) -> int:
    """The contribution's scalar of point i of a section (0 tau_g1, 1 tau_g2, 2 alpha_g1, 3 beta_g1, 4 beta_g2)."""
    t = pow(tau, i, R)
    return (t, t, alpha * t % R, beta * t % R, beta)[section]


def transform(acc: o.Accumulator, tau: int, alpha: int, beta: int) -> o.Accumulator:
    return o.Accumulator([o.g1_mul(q, scalar_of(0, i, tau, alpha, beta)) for i, q in enumerate(acc.tau_g1)],
                         [o.g2_mul(q, scalar_of(1, i, tau, alpha, beta)) for i, q in enumerate(acc.tau_g2)],
                         [o.g1_mul(q, scalar_of(2, i, tau, alpha, beta)) for i, q in enumerate(acc.alpha_g1)],
                         [o.g1_mul(q, scalar_of(3, i, tau, alpha, beta)) for i, q in enumerate(acc.beta_g1)],
                         o.g2_mul(acc.beta_g2, beta))


def contribute(challenge: bytes, n: int, secrets) -> bytes:
    """The response of powersoftau `compute` with these secrets (tau, alpha, beta, s_tau, s_alpha, s_beta)."""
    digest = hashlib.blake2b(challenge).digest()
    after = transform(parse_challenge(challenge, n), *secrets[:3])
    body = o.serialize_response(after)[64:-o.PUBKEY_SIZE]
    return digest + body + public_key(digest, secrets)


def same_ratio(g1_pair, g2_pair) -> bool:
    """e(a, d) == e(b, c) for ((a, b), (c, d))."""
    (a, b), (c, d) = g1_pair, g2_pair
    nb = None if b is None else (b[0], (-b[1]) % P)
    return po.product_of_pairings([(a, d), (nb, c)]) == po.F12_ONE


def verify_transform(challenge, response: bytes, n: int, powers: bool = True):
    """powersoftau verify_transform: the first failing relation's name, or None.  challenge None: only the key's
    relations (the digest is the response's prefix).  powers=False skips the (slow) powers relations."""
    after, g1, g2 = parse_response(response, n)
    digest = response[:64]
    if challenge is not None:
        if hashlib.blake2b(challenge).digest() != digest:
            return "HASH"
        before = parse_challenge(challenge, n)
    g2_s = [_g2_s(digest, i, g1[2 * i], g1[2 * i + 1]) for i in range(3)]
    for i, name in enumerate(("POK_TAU", "POK_ALPHA", "POK_BETA")):
        if not same_ratio((g1[2 * i], g1[2 * i + 1]), (g2_s[i], g2[i])):
            return name
    if challenge is not None:
        if not same_ratio((before.tau_g1[1], after.tau_g1[1]), (g2_s[0], g2[0])):
            return "CHAIN_TAU"
        if not same_ratio((before.alpha_g1[0], after.alpha_g1[0]), (g2_s[1], g2[1])):
            return "CHAIN_ALPHA"
        if not same_ratio((before.beta_g1[0], after.beta_g1[0]), (g2_s[2], g2[2])):
            return "CHAIN_BETA"
        if not same_ratio((before.beta_g1[0], after.beta_g1[0]), (before.beta_g2, after.beta_g2)):
            return "CHAIN_BETA_G2"
    if powers:
        if after.tau_g1[0] != o.G1_GEN or after.tau_g2[0] != o.G2_GEN:
            return "GENERATORS"
        for name, sec in (("TAU_G1", after.tau_g1), ("ALPHA_G1", after.alpha_g1), ("BETA_G1", after.beta_g1)):
            for i in range(len(sec) - 1):
                if not same_ratio((sec[i], sec[i + 1]), (after.tau_g2[0], after.tau_g2[1])):
                    return name
        for i in range(n - 1):
            if not same_ratio((after.tau_g1[0], after.tau_g1[1]), (after.tau_g2[i], after.tau_g2[i + 1])):
                return "TAU_G2"
        if not same_ratio((after.tau_g1[0], after.beta_g1[0]), (after.tau_g2[0], after.beta_g2)):
            return "BETA_G2"
    return None
