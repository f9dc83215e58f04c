"""A Powers-of-Tau contribution (ptau_contribute, powersoftau `compute`) and its check (ptau_verify_contribution,
powersoftau `verify_transform`).

CPU tests pin the recalled formats (ChaCha20 against `cryptography`, h2, hash_to_g2) and run the product's per-point
code (host build, tests/host_emul/hostemul_contribute.cpp) against the big-integer oracle (tests/contribute_oracle.py).
GPU tests check contributions byte for byte against the oracle and against the generator with composed secrets, and
that verify_contribution accepts them and names the relation or point of each tampering."""
import ctypes
import hashlib
import os
import random

import numpy as np
import pytest

import contribute_oracle as co
import ptau_oracle as o

R = o.R_ORDER
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ZABS = o.Z_ABS
SECRETS = (0x1234567 * 3 + 11, 0xABCDEF12345 % R, 0x0FEDCBA987654321 * 5 % R, 77, 0x5151 * 0x9999 % R, 0xDEADBEEF)


# ---- formats (powersoftau with pairing 0.14.2; restated from memory, pinned only where noted) ---------------------
def test_dagger_challenge_and_response_formats():
    """challenge = 64-byte hash || uncompressed accumulator (tau_g1 2n-1, tau_g2 n, alpha_g1 n, beta_g1 n, beta_g2 1);
    response = BLAKE2b-512(challenge) || compressed accumulator || 1152-byte uncompressed public key in the order
    tau_g1.(s, s tau), alpha_g1.(s, s alpha), beta_g1.(s, s beta), tau_g2, alpha_g2, beta_g2."""
    for n in (2, 8, 1 << 21):
        assert 64 + o.uncompressed_size(n) == 64 + (2 * n - 1) * 96 + n * 192 + 2 * n * 96 + 192
        assert o.response_size(n) == 64 + (2 * n - 1) * 48 + n * 96 + 2 * n * 48 + 96 + 3 * 192 + 6 * 96


def test_dagger_next_u64_first_word_high():
    """rand 0.4 Rng::next_u64 default: ((next_u32 as u64) << 32) | next_u32 -- recalled, not vendored."""
    rng = co.ChaChaRng([0] * 8)
    w0, w1 = co.chacha_block([0] * 8, 0)[:2]
    assert rng.next_u64() == (w0 << 32) | w1


@pytest.fixture(scope="module")
def hostemul():
    d = os.path.join(ROOT, "tests", "host_emul")
    so = os.path.join(d, "libptau_hostemul_contribute.so")
    csrc = os.path.join(ROOT, "kzg_setup_powersoftau_b200", "csrc")
    deps = [os.path.join(d, "hostemul_contribute.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                           if f.endswith((".cuh", ".inc", ".h"))]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        import subprocess

        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                               os.path.join(d, "hostemul_contribute.cpp")])
    return ctypes.CDLL(so)


# ---- 1. ChaCha20 --------------------------------------------------------------------------------------------------
def test_chacha_matches_cryptography(hostemul):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms

    rnd = random.Random(1)
    for _ in range(6):
        key = [rnd.getrandbits(32) for _ in range(8)]
        kb = b"".join(w.to_bytes(4, "little") for w in key)
        ks = Cipher(algorithms.ChaCha20(kb, bytes(16)), mode=None).encryptor().update(bytes(64 * 5))
        want = [int.from_bytes(ks[4 * i:4 * i + 4], "little") for i in range(80)]
        rng = co.ChaChaRng(key)
        assert [rng.next_u32() for _ in range(80)] == want
        out = (ctypes.c_uint32 * 80)()
        hostemul.hostemul_chacha((ctypes.c_uint32 * 8)(*key), out, 80)
        assert list(out) == want


def test_chacha_rfc7539_block():
    """RFC 7539 2.3.2: key 00..1f, counter 1, nonce 00000009 0000004a 00000000 (rand's counter words 13..15)."""
    key = [int.from_bytes(bytes(range(4 * i, 4 * i + 4)), "little") for i in range(8)]
    ctr = 1 | (0x09000000 << 32) | (0x4A000000 << 64)
    blk = co.chacha_block(key, ctr)
    assert b"".join(w.to_bytes(4, "little") for w in blk)[:8].hex() == "10f1e7e4d13b5915"


# ---- 2. h2 --------------------------------------------------------------------------------------------------------
def test_h2_clears_the_cofactor():
    rnd = random.Random(2)
    z = -ZABS
    assert co.H2 * 9 == z**8 - 4 * z**7 + 5 * z**6 - 4 * z**4 + 6 * z**3 - 4 * z**2 - 4 * z + 13
    found = 0
    while found < 3:
        x = (rnd.randrange(o.P), rnd.randrange(o.P))
        y = o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2))
        if y is None:
            continue
        q = o.g2_mul((x, y), co.H2)
        assert q is not None and o.g2_mul(q, R) is None
        found += 1


# ---- 3. hash_to_g2 ------------------------------------------------------------------------------------------------
def test_host_hash_to_g2_matches_oracle(hostemul):
    rejected = no_root = 0
    out = (ctypes.c_uint8 * 192)()
    stats = (ctypes.c_int * 2)()
    for i in range(100):
        d = hashlib.blake2b(b"h2g2" + i.to_bytes(4, "little")).digest()
        st = {"rejected": 0, "no_root": 0}
        want = o.zcash_g2_uncompressed_encode(co.hash_to_g2(d, st))
        hostemul.hostemul_hash_to_g2(d, out, stats)
        assert bytes(out) == want, i
        assert (stats[0], stats[1]) == (st["rejected"], st["no_root"])
        rejected += st["rejected"] > 0
        no_root += st["no_root"] > 0
    assert rejected and no_root


# ---- 4. decomposition and ladder -----------------------------------------------------------------------------------
def _scalars():
    z2 = ZABS**2
    ks = [0, 1, 2, R - 1, R - 2, z2 - 1, z2, z2 + 1, 5 * z2 - 1, 5 * z2 + 1, (z2 - 1) * z2 + z2 - 1]
    for i in (1, 2, 3):
        ks += [ZABS**i - 1, ZABS**i + 1]
    ks += [sum((ZABS - 1) * ZABS**i for i in range(3)) + (R // ZABS**3), 8 * 0x1111111111111111, 0x8888888888888888]
    rnd = random.Random(4)
    ks += [rnd.randrange(R) for _ in range(12)]
    return [k % R for k in ks]


def _int(b):
    return int.from_bytes(bytes(b), "little")


def test_decompositions(hostemul):
    z2 = ZABS**2
    k0, k1 = (ctypes.c_uint8 * 16)(), (ctypes.c_uint8 * 16)()
    d = (ctypes.c_uint8 * 32)()
    for k in _scalars():
        kb = k.to_bytes(32, "little")
        hostemul.hostemul_glv_split_g1(kb, k0, k1)
        assert _int(k0) + _int(k1) * z2 == k and _int(k0) < z2 and _int(k1) < z2
        hostemul.hostemul_zdigits_g2(kb, d)
        ds = [_int(bytes(d)[8 * i:8 * i + 8]) for i in range(4)]
        assert sum(v * ZABS**i for i, v in enumerate(ds)) == k and all(v < ZABS for v in ds)
    e = (ctypes.c_int8 * 33)()
    for s in (0, 1, 7, 8, 15, 16, 0x88888888888888888888888888888888, z2 - 1, 2**128 - 1):
        hostemul.hostemul_recode(s.to_bytes(16, "little"), 2, e, 33)
        assert sum(v * 16**j for j, v in enumerate(e)) == s and all(-8 <= v <= 7 for v in e)


def _enc(group, q):
    if group == 1:
        return q[0].to_bytes(48, "big") + q[1].to_bytes(48, "big")
    (x0, x1), (y0, y1) = q
    return b"".join(v.to_bytes(48, "big") for v in (x0, x1, y0, y1))


@pytest.mark.parametrize("group", [1, 2])
def test_host_ladder_matches_oracle(hostemul, group):
    gen, mul = (o.G1_GEN, o.g1_mul) if group == 1 else (o.G2_GEN, o.g2_mul)
    rnd = random.Random(5 + group)
    bases = [gen, mul(gen, rnd.randrange(1, R)), mul(gen, rnd.randrange(1, R))]
    out = (ctypes.c_uint8 * 192)()
    for bi, base in enumerate(bases):
        for k in _scalars() if bi == 0 else _scalars()[::3]:
            want = mul(base, k)
            fin = hostemul.hostemul_contrib_mul(group, _enc(group, base), k.to_bytes(32, "little"), out)
            if want is None:
                assert fin == 0, k
            else:
                assert fin == 1 and bytes(out)[:96 * group] == _enc(group, want), k


# ---- 5. oracle self-consistency ------------------------------------------------------------------------------------
def test_oracle_contribution_composes():
    n = 2
    t0, a0, b0 = o.derive_scalars(3)
    acc = o.make_accumulator(n, 3)
    chal = co.serialize_challenge(acc, bytes(range(64)))
    sec = SECRETS
    resp = co.contribute(chal, n, sec)
    after, _, _ = co.parse_response(resp, n)
    t, a, b = t0 * sec[0] % R, a0 * sec[1] % R, b0 * sec[2] % R
    assert after.tau_g1 == [o.g1_mul(o.G1_GEN, pow(t, i, R)) for i in range(2 * n - 1)]
    assert after.alpha_g1 == [o.g1_mul(o.G1_GEN, a * pow(t, i, R) % R) for i in range(n)]
    assert after.beta_g2 == o.g2_mul(o.G2_GEN, b)
    assert co.verify_transform(chal, resp, n) is None
    assert co.verify_transform(None, resp, n, powers=False) is None
    bad = bytearray(resp)
    bad[0] ^= 1
    assert co.verify_transform(chal, bytes(bad), n, powers=False) == "HASH"
    pk = len(resp) - o.PUBKEY_SIZE
    for i, name in enumerate(("POK_TAU", "POK_ALPHA", "POK_BETA")):  # swap in another s.x
        bad = bytearray(resp)
        j = (i + 1) % 3
        bad[pk + (2 * i + 1) * 96:pk + (2 * i + 2) * 96] = resp[pk + (2 * j + 1) * 96:pk + (2 * j + 2) * 96]
        assert co.verify_transform(chal, bytes(bad), n, powers=False) == name
    for i, name in enumerate(("CHAIN_TAU", "CHAIN_ALPHA", "CHAIN_BETA")):  # a key of another x, consistent in itself
        other = list(sec)
        other[i] += 1
        assert co.verify_transform(chal, resp[:pk] + co.public_key(resp[:64], other), n, powers=False) == name
    assert co.verify_transform(*_chain_beta_g2_case(acc, chal, resp, n, sec), n, powers=False) == "CHAIN_BETA_G2"
    # the powers relations: one point of a section doubled (the first power of each section is left alone, the chain
    # relations read it)
    off = {"TAU_G1": 64 + 48 * 2, "ALPHA_G1": 64 + 48 * (2 * n - 1) + 96 * n + 48, "BETA_G1": 64 + 48 * (2 * n - 1) + 96 * n
           + 48 * n + 48, "GENERATORS": 64}
    for name, at in off.items():
        q = o.g1_mul(o.zcash_g1_compressed_decode(resp[at:at + 48]), 2)
        assert co.verify_transform(chal, resp[:at] + o.zcash_g1_compressed_encode(q) + resp[at + 48:], n) == name


def _chain_beta_g2_case(acc, chal, resp, n, sec):
    """A challenge whose beta_g2 is not beta_g1's partner, and a response to it that is consistent in itself: the body
    of the original challenge's response under the changed challenge's digest and a key made for that digest.  Only
    CHAIN_BETA_G2 can fail."""
    acc2 = o.Accumulator(acc.tau_g1, acc.tau_g2, acc.alpha_g1, acc.beta_g1, o.g2_mul(acc.beta_g2, 3))
    chal2 = co.serialize_challenge(acc2, chal[:64])
    d2 = hashlib.blake2b(chal2).digest()
    pk = len(resp) - o.PUBKEY_SIZE
    return chal2, d2 + resp[64:pk] + co.public_key(d2, sec)


# ---- the golden contribution (tools/make_golden.py) and the 64-bit section offsets ---------------------------------
def _golden(name):
    with open(os.path.join(ROOT, "tests", "golden", name), "rb") as f:
        return f.read()


def test_golden_contribution_is_the_oracle_contribution():
    prev = _golden("n8_powersoftau.bin")
    chal = _golden("n8_challenge.bin")
    assert chal == hashlib.blake2b(prev).digest() + _golden("n8_powersoftau_uncompressed.bin")
    resp = _golden("n8_contribution.bin")
    assert resp == co.contribute(chal, 8, co.GOLDEN_SECRETS)
    assert co.verify_transform(chal, resp, 8, powers=False) is None


def test_section_offsets_are_64_bit(hostemul):
    hostemul.hostemul_section_offset.restype = ctypes.c_uint64
    hostemul.hostemul_section_offset.argtypes = [ctypes.c_uint64, ctypes.c_int, ctypes.c_int]
    for n in (2, 8, 1 << 21, 1 << 22, 1 << 26, 1 << 40):
        for fmt, g1, g2 in ((1, 96, 192), (2, 48, 96)):
            want = [0, (2 * n - 1) * g1, (2 * n - 1) * g1 + n * g2, (3 * n - 1) * g1 + n * g2, (4 * n - 1) * g1 + n * g2]
            assert [hostemul.hostemul_section_offset(n, fmt, s) for s in range(5)] == want, (n, fmt)


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ptau():
    import kzg_setup_powersoftau_b200 as p

    return p


@pytest.fixture(scope="module")
def ctx(ptau):
    c = ptau.Context(1)
    yield c
    c.close()


def _sec_bytes(sec):
    return b"".join(v.to_bytes(32, "little") for v in sec)


def _gen_challenge(ptau, ctx, n, t, a, b, prefix=bytes(64)):
    """challenge of (t, a, b) from the GPU generator"""
    U = ptau.FMT_ZCASH_UNCOMPRESSED
    parts = [prefix, ctx.generate(1, U, 1, t, 0, 2 * n - 1), ctx.generate(2, U, 1, t, 0, n),
             ctx.generate(1, U, a, t, 0, n), ctx.generate(1, U, b, t, 0, n), ctx.generate(2, U, b, t, 0, 1)]
    return np.concatenate([np.frombuffer(bytes(p), dtype=np.uint8) if isinstance(p, bytes) else p for p in parts])


def _gen_body(ptau, ctx, n, t, a, b):
    C = ptau.FMT_ZCASH_COMPRESSED
    return np.concatenate([ctx.generate(1, C, 1, t, 0, 2 * n - 1), ctx.generate(2, C, 1, t, 0, n),
                           ctx.generate(1, C, a, t, 0, n), ctx.generate(1, C, b, t, 0, n),
                           ctx.generate(2, C, b, t, 0, 1)]).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 8])
def test_contribute_matches_oracle(ptau, ctx, n):
    acc = o.make_accumulator(n, 10 + n)
    chal = co.serialize_challenge(acc, hashlib.blake2b(b"prev").digest())
    got = ctx.contribute(chal, n, secrets=SECRETS).tobytes()
    assert got == co.contribute(chal, n, SECRETS)
    ctx.verify_contribution(chal, got, n)
    ctx.verify_contribution(None, got, n)


@pytest.mark.gpu
def test_contribute_sampled_against_oracle_2p10p1(ptau, ctx):
    n = (1 << 10) + 1
    t0, a0, b0 = o.derive_scalars(9)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0)
    got = ctx.contribute(chal, n, secrets=SECRETS).tobytes()
    t, a, b = SECRETS[:3]
    rnd = random.Random(6)
    off_u, off_c = 64, 64
    for s, (g, cnt) in enumerate(((1, 2 * n - 1), (2, n), (1, n), (1, n), (2, 1))):
        ru, rc = 96 * g, 48 * g
        for i in sorted({i for i in (0, 1, cnt - 1) if i < cnt} | {rnd.randrange(cnt) for _ in range(12)}):
            dec = o.zcash_g1_uncompressed_decode if g == 1 else o.zcash_g2_uncompressed_decode
            p = dec(chal[off_u + i * ru:off_u + (i + 1) * ru].tobytes())
            k = co.scalar_of(s, i, t, a, b)
            q = (o.g1_mul if g == 1 else o.g2_mul)(p, k)
            enc = o.zcash_g1_compressed_encode if g == 1 else o.zcash_g2_compressed_encode
            assert got[off_c + i * rc:off_c + (i + 1) * rc] == enc(q), (s, i)
        off_u += cnt * ru
        off_c += cnt * rc
    assert got[:64] == hashlib.blake2b(chal.tobytes()).digest()
    # and every byte of the body: the generator's records of the composed secrets
    body = _gen_body(ptau, ctx, n, t0 * t % R, a0 * a % R, b0 * b % R)
    assert got[64:64 + len(body)] == body


def _composed(ptau, ctx, n, chunk_ctx=None):
    t0, a0, b0 = o.derive_scalars(21)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0)
    got = (chunk_ctx or ctx).contribute(chal, n, secrets=SECRETS)
    t, a, b = t0 * SECRETS[0] % R, a0 * SECRETS[1] % R, b0 * SECRETS[2] % R
    want = _gen_body(ptau, ctx, n, t, a, b)
    body = got[64:64 + len(want)].tobytes()
    assert body == want
    return chal, got


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1 << 16, 1 << 21])
def test_known_tau_composition(ptau, ctx, n):
    chal, got = _composed(ptau, ctx, n)
    ctx.verify_contribution(chal, got, n)


@pytest.mark.gpu
def test_known_tau_composition_small_chunks(ptau, ctx):
    c = ptau.Context(1, chunk_points=1000)
    try:
        for n in (999, 1000, 1001, 2 * 1000 - 1, 2 * 1000 + 1):
            _composed(ptau, ctx, n, c)
    finally:
        c.close()


@pytest.mark.gpu
def test_two_gpu_context_is_byte_identical(ptau, ctx):
    if ptau._ffi.lib().ptau_device_count() < 2:
        pytest.skip("one GPU")
    n = 1 << 14
    t0, a0, b0 = o.derive_scalars(5)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0)
    c2 = ptau.Context(2)
    try:
        assert c2.contribute(chal, n, secrets=SECRETS).tobytes() == ctx.contribute(chal, n, secrets=SECRETS).tobytes()
    finally:
        c2.close()


@pytest.mark.gpu
def test_public_key_and_random_secrets(ptau, ctx):
    n = 4
    t0, a0, b0 = o.derive_scalars(7)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0)
    got = ctx.contribute(chal, n, secrets=SECRETS).tobytes()
    assert got[-o.PUBKEY_SIZE:] == co.public_key(hashlib.blake2b(chal.tobytes()).digest(), SECRETS)
    r1 = ctx.contribute(chal, n).tobytes()
    r2 = ctx.contribute(chal, n).tobytes()
    assert r1[64:] != r2[64:] and r1[:64] == r2[:64]
    ctx.verify_contribution(chal, r1, n)
    ctx.verify_contribution(chal, r2, n)


@pytest.fixture(scope="module")
def pair8(ptau, ctx):
    n = 8
    t0, a0, b0 = o.derive_scalars(8)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0, prefix=hashlib.blake2b(b"x").digest())
    return n, chal.tobytes(), ctx.contribute(chal, n, secrets=SECRETS).tobytes()


def _rel(ptau, ctx, chal, resp, n):
    with pytest.raises(ptau.PtauError) as e:
        ctx.verify_contribution(chal, resp, n)
    return e.value


@pytest.mark.gpu
def test_verify_contribution_rejects(ptau, ctx, pair8):
    n, chal, resp = pair8
    pk = len(resp) - o.PUBKEY_SIZE
    bad = bytearray(resp)
    bad[3] ^= 1
    assert _rel(ptau, ctx, chal, bytes(bad), n).relation == ptau.REL_HASH
    for i, rel in enumerate((ptau.REL_POK_TAU, ptau.REL_POK_ALPHA, ptau.REL_POK_BETA)):
        j = (i + 1) % 3
        bad = bytearray(resp)
        bad[pk + (2 * i + 1) * 96:pk + (2 * i + 2) * 96] = resp[pk + (2 * j + 1) * 96:pk + (2 * j + 2) * 96]
        assert _rel(ptau, ctx, chal, bytes(bad), n).relation == rel
        assert _rel(ptau, ctx, None, bytes(bad), n).relation == rel
    # a response of another tau that is consistent in itself: only the chain to the challenge fails
    other = ctx.contribute(np.frombuffer(chal, dtype=np.uint8), n, secrets=(SECRETS[0] + 1,) + SECRETS[1:]).tobytes()
    ctx.verify_contribution(None, other, n)
    # the key's tau part (the tau_g1 pair and tau_g2) taken from the other response
    mixed_key = resp[:pk] + other[pk:pk + 2 * 96] + resp[pk + 2 * 96:pk + 576] + other[pk + 576:pk + 768] + \
        resp[pk + 768:]
    assert _rel(ptau, ctx, chal, mixed_key, n).relation == ptau.REL_CHAIN_TAU
    # the key's alpha and beta parts from a response of another alpha / beta
    for i, rel in ((1, ptau.REL_CHAIN_ALPHA), (2, ptau.REL_CHAIN_BETA)):
        sec = list(SECRETS)
        sec[i] += 1
        oth = ctx.contribute(np.frombuffer(chal, dtype=np.uint8), n, secrets=sec).tobytes()
        key = bytearray(resp[pk:])
        key[2 * i * 96:(2 * i + 2) * 96] = oth[pk + 2 * i * 96:pk + (2 * i + 2) * 96]
        key[576 + 192 * i:576 + 192 * (i + 1)] = oth[pk + 576 + 192 * i:pk + 576 + 192 * (i + 1)]
        assert _rel(ptau, ctx, chal, resp[:pk] + bytes(key), n).relation == rel
    # a challenge whose beta_g2 does not match its beta_g1, and a response consistent in itself
    acc = co.parse_challenge(chal, n)
    chal2, resp2 = _chain_beta_g2_case(acc, chal, resp, n, SECRETS)
    assert _rel(ptau, ctx, chal2, resp2, n).relation == ptau.REL_CHAIN_BETA_G2
    # beta_g2 of another beta: the powers relation BETA_G2 of the response fails first
    other_b = ctx.contribute(np.frombuffer(chal, dtype=np.uint8), n, secrets=SECRETS[:2] + (SECRETS[2] + 1,) + SECRETS[3:]).tobytes()
    bg2 = pk - 96
    assert _rel(ptau, ctx, chal, resp[:bg2] + other_b[bg2:pk] + resp[pk:], n).relation == ptau.REL_BETA_G2
    # a tampered power
    off = 64 + 48 * 5
    bad = resp[:off] + resp[off + 48:off + 96] + resp[off:off + 48] + resp[off + 96:]
    assert _rel(ptau, ctx, chal, bad, n).relation == ptau.REL_TAU_G1
    # a bad public-key point (G2 #1 off the curve) and a bad challenge point (beta_g1[0] off the curve)
    bad = bytearray(resp)
    bad[pk + 6 * 96 + 192 + 191] ^= 1
    e = _rel(ptau, ctx, chal, bytes(bad), n)
    assert (e.section, e.index, e.code) == (5, 7, ptau.BAD_NOT_ON_CURVE)
    c = bytearray(chal)
    b0 = 64 + (2 * n - 1) * 96 + n * 192 + n * 96
    c[b0 + 95] ^= 1
    e = _rel(ptau, ctx, bytes(c), resp, n)
    assert (e.section, e.index, e.code) == (6 + 3, 0, ptau.BAD_NOT_ON_CURVE)


@pytest.mark.gpu
def test_end_to_end_files(ptau, ctx, tmp_path):
    n, log2 = 1 << 10, 10
    t0, a0, b0 = o.derive_scalars(12)
    prev = np.concatenate([np.frombuffer(hashlib.blake2b(b"p").digest(), dtype=np.uint8), _gen_body_arr(ptau, ctx, n, t0, a0, b0),
                           np.zeros(o.PUBKEY_SIZE, dtype=np.uint8)])
    (tmp_path / "prev").write_bytes(prev.tobytes())
    digest = ptau.challenge_from_response(str(tmp_path / "prev"), str(tmp_path / "challenge"), log2, ctx=ctx)
    assert digest == hashlib.blake2b(prev.tobytes()).digest()
    with pytest.raises(FileExistsError):
        ptau.challenge_from_response(str(tmp_path / "prev"), str(tmp_path / "challenge"), log2, ctx=ctx)
    h = ptau.contribute(str(tmp_path / "challenge"), str(tmp_path / "response"), log2, ctx=ctx, secrets=SECRETS)
    assert h == hashlib.blake2b((tmp_path / "challenge").read_bytes()).digest()
    ptau.verify_contribution(str(tmp_path / "challenge"), str(tmp_path / "response"), log2, ctx=ctx)
    ptau.verify_contribution(None, str(tmp_path / "response"), log2, ctx=ctx)
    setup = ctx.preprocess(ptau.VARIANT_KGZ, (tmp_path / "response").read_bytes(), n)
    t, a, b = t0 * SECRETS[0] % R, a0 * SECRETS[1] % R, b0 * SECRETS[2] % R
    synth = b"\0" * 64 + _gen_body(ptau, ctx, n, t, a, b) + b"\0" * o.PUBKEY_SIZE
    assert bytes(setup) == bytes(ctx.preprocess(ptau.VARIANT_KGZ, synth, n))


def _gen_body_arr(ptau, ctx, n, t, a, b):
    return np.frombuffer(_gen_body(ptau, ctx, n, t, a, b), dtype=np.uint8)


@pytest.mark.gpu
def test_errors_and_infinity(ptau, ctx):
    L = ptau._ffi.lib()
    n = 4
    t0, a0, b0 = o.derive_scalars(13)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0)
    for bad in ((0,) + SECRETS[1:], SECRETS[:5] + (R,), SECRETS[:2] + (R + 5,) + SECRETS[3:]):
        with pytest.raises(ptau.PtauError) as e:
            ctx.contribute(chal, n, secrets=bad)
        assert e.value.code == ptau._ffi.ERR_ARG
    with pytest.raises(ptau.PtauError) as e:
        ctx.contribute(chal[:-1], n, secrets=SECRETS)
    assert e.value.code == ptau._ffi.ERR_SIZE
    with pytest.raises(ptau.PtauError) as e:
        ctx.contribute(chal, n, secrets=SECRETS, out=np.empty(L.ptau_response_size(n) + 1, dtype=np.uint8))
    assert e.value.code == ptau._ffi.ERR_SIZE
    small = _gen_challenge(ptau, ctx, 1, t0, a0, b0)
    with pytest.raises(ptau.PtauError) as e:
        ctx.contribute(small, 1, secrets=SECRETS)
    assert e.value.code == ptau._ffi.ERR_ARG
    resp = ctx.contribute(chal, n, secrets=SECRETS)
    with pytest.raises(ptau.PtauError) as e:
        ctx.verify_contribution(chal[:-1], resp, n)
    assert e.value.code == ptau._ffi.ERR_SIZE
    with pytest.raises(ptau.PtauError) as e:
        ctx.verify_contribution(chal, resp[:-1], n)
    assert e.value.code == ptau._ffi.ERR_SIZE
    # a bad challenge point: the same (section, index, kind) as preprocess of the same bytes
    c = chal.copy()
    at = 64 + (2 * n - 1) * 96 + 2 * 192 + 191  # tau_g2[2], last byte
    c[at] ^= 1
    with pytest.raises(ptau.PtauError) as e:
        ctx.contribute(c, n, secrets=SECRETS)
    with pytest.raises(ptau.PtauError) as e2:
        ctx.preprocess_uncompressed(ptau.VARIANT_FASTKGZ, c[64:], n)
    assert (e.value.section, e.value.index, e.value.code) == (e2.value.section, e2.value.index, e2.value.code) == \
        (1, 2, ptau.BAD_NOT_ON_CURVE)
    # infinity in the challenge, as the conversion reads an uncompressed record (the reference's read_g1: the flag bits
    # sit in the first byte of y): rejected with CHECKS_STRICT; with CHECKS_DECOMPRESS it stays infinity and every
    # other point of the body is the one of the unmodified challenge
    c = chal.copy()
    at = 64 + 96 * 3
    inf_rec = bytes(48) + bytes([0x40]) + bytes(47)
    assert o.read_g1(inf_rec) is None
    c[at:at + 96] = np.frombuffer(inf_rec, dtype=np.uint8)
    with pytest.raises(ptau.PtauError) as e:
        ctx.contribute(c, n, secrets=SECRETS)
    assert (e.value.section, e.value.index, e.value.code) == (0, 3, ptau.BAD_INFINITY)
    got = ctx.contribute(c, n, secrets=SECRETS, checks=ptau.CHECKS_DECOMPRESS).tobytes()
    ref = resp.tobytes()
    rec = slice(64 + 48 * 3, 64 + 48 * 4)
    assert got[rec] == o.zcash_g1_compressed_encode(None)
    assert got[64:rec.start] == ref[64:rec.start]
    assert got[rec.stop:-o.PUBKEY_SIZE] == ref[rec.stop:-o.PUBKEY_SIZE]


@pytest.mark.gpu
def test_golden_contribution_on_gpu(ptau, ctx, tmp_path):
    chal = _golden("n8_challenge.bin")
    assert ctx.contribute(chal, 8, secrets=co.GOLDEN_SECRETS).tobytes() == _golden("n8_contribution.bin")
    ctx.verify_contribution(chal, _golden("n8_contribution.bin"), 8)
    prev = tmp_path / "prev"
    prev.write_bytes(_golden("n8_powersoftau.bin"))
    ptau.challenge_from_response(str(prev), str(tmp_path / "challenge"), 3, ctx=ctx)
    assert (tmp_path / "challenge").read_bytes() == chal


@pytest.mark.gpu
def test_verify_contribution_past_2gb(ptau, ctx):
    """2^22 powers: the challenge is 2.4 GB, so the offsets of its later sections do not fit in 32 bits."""
    n = 1 << 22
    t0, a0, b0 = o.derive_scalars(22)
    chal = _gen_challenge(ptau, ctx, n, t0, a0, b0)
    resp = ctx.contribute(chal, n, secrets=SECRETS)
    ctx.verify_contribution(chal, resp, n)
    ctx.verify_contribution(None, resp, n)
    # the beta_g2 record read by the chain relation, past 2^31 bytes: off the curve
    at = len(chal) - 1
    chal[at] ^= 1
    e = _rel(ptau, ctx, chal, resp, n)
    assert (e.section, e.index, e.code) == (6 + 4, 0, ptau.BAD_NOT_ON_CURVE)
