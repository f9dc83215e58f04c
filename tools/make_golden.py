#!/usr/bin/env python3
"""Generate tests/golden/* from the Python big-int oracle (oracle/ptau_oracle.py).

The reference holds no usable fixtures for this path (SURVEY.md 8c), so these are
oracle-generated: a synthetic N=8 Powers-of-Tau response with known tau and every
artefact the reference binaries/loaders derive from it, plus a table of malformed
records with the status each check mode must report.  Committed together with this
script; regenerate with `python tools/make_golden.py`.
"""
import hashlib
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ptau_oracle as o  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)
N = 8
SEED = 0xB200


def w(name, data):
    with open(os.path.join(OUT, name), "wb") as f:
        f.write(data)


acc = o.make_accumulator(N, SEED)
resp = o.serialize_response(acc, SEED)
assert len(resp) == o.response_size(N)
unc = o.powersoftau_uncompress(resp, N)
assert len(unc) == o.uncompressed_size(N)
kgz = o.preprocess_kgz(unc, N)
fast = o.preprocess_fastkgz(unc, N)
assert len(kgz) == o.kgz_size(N) and len(fast) == o.fastkgz_size(N)
w("n8_powersoftau.bin", resp)
w("n8_powersoftau_uncompressed.bin", unc)
w("n8_kzg_setup_kgz.bin", kgz)
w("n8_kzg_setup_fastkgz.bin", fast)

pg, pgg, vk = o.load_kzg_setup(kgz, N)
g1 = b"".join(o.g1_mont_record(*p) for p in pg + pgg + [vk[0], vk[1]])
g2 = b"".join(o.g2_mont_record(*p) for p in [vk[2], vk[3]])
w("n8_load_kgz_g1.bin", g1)
w("n8_load_kgz_g2.bin", g2)
pg, pgg, h, bh, bhf, ph = o.load_fastkzg_setup(fast, N)
w("n8_load_fastkgz_g1.bin", b"".join(o.g1_mont_record(*p) for p in pg + pgg))
w("n8_load_fastkgz_g2.bin", b"".join(o.g2_mont_record(*p) for p in [h, bhf] + ph))

# phase1radix2m2-shaped file (m = 4) from the same points
m = 4
ph1 = (o.zcash_g1_uncompressed_encode(acc.alpha_g1[0]) + o.zcash_g1_uncompressed_encode(acc.beta_g1[0])
       + o.zcash_g2_uncompressed_encode(acc.beta_g2)
       + b"".join(o.zcash_g1_uncompressed_encode(q) for q in acc.tau_g1[:m])
       + b"".join(o.zcash_g2_uncompressed_encode(q) for q in acc.tau_g2[:m])
       + b"".join(o.zcash_g1_uncompressed_encode(q) for q in acc.alpha_g1[:m])
       + b"".join(o.zcash_g1_uncompressed_encode(q) for q in acc.beta_g1[:m]))
w("n8_phase1radix2m2.bin", ph1)

# ---- malformed / edge records ------------------------------------------------
rnd = random.Random(SEED)
P = o.P
cases = []
KIND = {None: 0, o.BAD_NON_CANONICAL: 1, o.BAD_FLAGS: 2, o.BAD_INFINITY: 3, o.BAD_NOT_ON_CURVE: 4,
        o.BAD_NOT_IN_SUBGROUP: 5}
STRICT, READ = 2 | 4 | 8, 4


def status_of(fn):
    try:
        fn()
        return 0
    except o.DecodeError as e:
        return KIND[e.kind]


def add(desc, group, in_fmt, rec):
    """expected statuses: strict = on-curve + subgroup + reject-infinity (GPU default);
    read = reference-exact read_g1/read_g2 (subgroup by r-multiplication only)."""
    if in_fmt == 2:  # compressed: pairing decode, then (strict) subgroup
        dec = o.zcash_g1_compressed_decode if group == 1 else o.zcash_g2_compressed_decode
        sub = o.g1_in_subgroup_rmul if group == 1 else o.g2_in_subgroup_rmul

        def strict():
            q = dec(rec)
            if q is None:
                raise o.DecodeError(o.BAD_INFINITY)
            if not sub(q):
                raise o.DecodeError(o.BAD_NOT_IN_SUBGROUP)

        st_strict = status_of(strict)
        st_none = status_of(lambda: dec(rec))
        cases.append({"desc": desc, "group": group, "in_fmt": in_fmt, "rec": rec.hex(), "strict": st_strict,
                      "nocheck": st_none})
        return
    rd = o.read_g1 if group == 1 else o.read_g2
    if in_fmt == 3:
        rd = o.ark_g1_deserialize_uncompressed if group == 1 else o.ark_g2_deserialize_uncompressed
    un = ((lambda b: o.ark_g1_deserialize_unchecked(o.read_g1_bytes(b) if in_fmt == 1 else b)) if group == 1 else
          (lambda b: o.ark_g2_deserialize_unchecked(o.read_g2_bytes(b) if in_fmt == 1 else b)))

    def strict():
        x, y, inf = un(rec)
        if inf:
            raise o.DecodeError(o.BAD_INFINITY)
        rd(rec, True)

    entry = {"desc": desc, "group": group, "in_fmt": in_fmt, "rec": rec.hex(), "strict": status_of(strict),
             "nocheck": status_of(lambda: un(rec))}
    # subgroup-only mode is reference-exact on every input (G1: the GLV test is; G2: off-curve
    # points fall back to the multiplication by r)
    entry["read"] = status_of(lambda: rd(rec, False))
    cases.append(entry)


q1 = acc.tau_g1[3]
q2 = acc.tau_g2[3]
zu1, zc1 = o.zcash_g1_uncompressed_encode(q1), o.zcash_g1_compressed_encode(q1)
zu2, zc2 = o.zcash_g2_uncompressed_encode(q2), o.zcash_g2_compressed_encode(q2)
au1, au2 = o.ark_g1_serialize_uncompressed(q1), o.ark_g2_serialize_uncompressed(q2)


def mod(b, i, v=None, orv=None, andv=None):
    b = bytearray(b)
    if v is not None:
        b[i] = v
    if orv is not None:
        b[i] |= orv
    if andv is not None:
        b[i] &= andv
    return bytes(b)


add("valid", 1, 1, zu1); add("valid", 1, 2, zc1); add("valid", 1, 3, au1)
add("valid", 2, 1, zu2); add("valid", 2, 2, zc2); add("valid", 2, 3, au2)
# zcash infinity encodings
add("zcash infinity (uncompressed) -> x >= p after reversal", 1, 1, o.zcash_g1_uncompressed_encode(None))
add("zcash infinity (uncompressed)", 2, 1, o.zcash_g2_uncompressed_encode(None))
add("zcash infinity (compressed)", 1, 2, o.zcash_g1_compressed_encode(None))
add("zcash infinity (compressed)", 2, 2, o.zcash_g2_compressed_encode(None))
add("infinity with sort bit", 1, 2, mod(o.zcash_g1_compressed_encode(None), 0, orv=0x20))
add("infinity with stray byte", 2, 2, mod(o.zcash_g2_compressed_encode(None), 50, v=1))
add("ark infinity", 1, 3, o.ark_g1_serialize_uncompressed(None))
add("ark infinity", 2, 3, o.ark_g2_serialize_uncompressed(None))
# flag bits
add("compressed without compression bit", 1, 2, mod(zc1, 0, andv=0x7F))
add("compressed without compression bit", 2, 2, mod(zc2, 0, andv=0x7F))
add("uncompressed with compression bit in x", 1, 1, mod(zu1, 0, orv=0x80))
add("uncompressed with sort bit in x", 2, 1, mod(zu2, 0, orv=0x20))
add("y top bit set (ark PositiveY flag: accepted and stripped)", 1, 1, mod(zu1, 48, orv=0x80))
add("y.c1 top bit set (ark PositiveY flag)", 2, 1, mod(zu2, 96, orv=0x80))
add("y both flag bits", 1, 1, mod(zu1, 48, orv=0xC0))
add("y both flag bits", 2, 3, mod(au2, 191, orv=0xC0))
add("y infinity flag with finite coordinates", 1, 1, mod(zu1, 48, orv=0x40))
add("y infinity flag with finite coordinates", 1, 3, mod(au1, 95, orv=0x40))
add("y infinity flag with finite coordinates", 2, 1, mod(zu2, 96, orv=0x40))
add("wrong sort bit: the other root (valid point -q)", 1, 2, mod(zc1, 0, v=zc1[0] ^ 0x20))
add("wrong sort bit: the other root", 2, 2, mod(zc2, 0, v=zc2[0] ^ 0x20))
# non-canonical
add("x = p", 1, 1, P.to_bytes(48, "big") + zu1[48:])
add("y = p", 1, 1, zu1[:48] + P.to_bytes(48, "big"))
add("x = p compressed", 1, 2, mod(P.to_bytes(48, "big"), 0, orv=0x80))
add("x.c0 = p", 2, 1, zu2[:48] + P.to_bytes(48, "big") + zu2[96:])
add("y.c0 = p + 5", 2, 3, au2[:96] + (P + 5).to_bytes(48, "little") + au2[144:])
add("x = 2^381 - 1", 1, 3, ((1 << 381) - 1).to_bytes(48, "little") + au1[48:])
add("x.c1 = p compressed", 2, 2, mod(P.to_bytes(48, "big"), 0, orv=0x80) + zc2[48:])
# off curve
add("y + 1", 1, 1, zu1[:48] + ((q1[1] + 1) % P).to_bytes(48, "big"))
add("y.c0 + 1", 2, 1, zu2[:144] + ((q2[1][0] + 1) % P).to_bytes(48, "big"))
while True:
    x = rnd.randrange(P)
    if o.fq_sqrt((x ** 3 + 4) % P) is None:
        add("x^3+4 is a non-residue", 1, 2, mod(x.to_bytes(48, "big"), 0, orv=0x80))
        break
while True:
    x = (rnd.randrange(P), rnd.randrange(P))
    if o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2)) is None:
        add("x^3+4(1+u) is a non-residue", 2, 2, mod(x[1].to_bytes(48, "big") + x[0].to_bytes(48, "big"), 0, orv=0x80))
        break
# invalid-curve point that the reference accepts: (k^2 x, k^3 y) lies on y^2 = x^3 + 4k^6, is r-torsion there
k = 7
tw = (k * k * q1[0] % P, k ** 3 * q1[1] % P)
add("r-torsion point of the isomorphic curve y^2=x^3+4*7^6 (ark 0.2 accepts; strict rejects)", 1, 1,
    o.zcash_g1_uncompressed_encode(tw))
kk = (5, 3)  # same for G2 with k in Fq2
k2, k3 = o.fq2_sqr(kk), o.fq2_mul(o.fq2_sqr(kk), kk)
tw2 = (o.fq2_mul(k2, q2[0]), o.fq2_mul(k3, q2[1]))
assert not o.g2_on_curve(tw2) and o.g2_in_subgroup_rmul(tw2)
add("r-torsion point of the isomorphic twist y^2=x^3+4(1+u)(5+3u)^6 (ark 0.2 accepts; strict rejects)", 2, 1,
    o.zcash_g2_uncompressed_encode(tw2))
add("same, ark encoding", 2, 3, o.ark_g2_serialize_uncompressed(tw2))
# on curve, outside the subgroup
cnt = 0
while cnt < 4:
    x = rnd.randrange(P)
    y = o.fq_sqrt((x ** 3 + 4) % P)
    if y is None:
        continue
    cnt += 1
    add("random curve point (cofactor component present)", 1, 1, o.zcash_g1_uncompressed_encode((x, y)))
    add("random curve point", 1, 2, o.zcash_g1_compressed_encode((x, y)))
h1 = (o.Z - 1) ** 2 // 3
def point_of_order(mulfn, sample, group_cofactor, small):
    """a point of exact order `small` (small prime dividing the cofactor)."""
    cof = group_cofactor
    while cof % small == 0:
        cof //= small
    for _ in range(200):
        q = sample()
        if q is None:
            continue
        t = mulfn(q, o.R_ORDER * cof)  # lands in the small-primary part
        if t is None:
            continue
        while True:
            nt = mulfn(t, small)
            if nt is None:
                return t
            t = nt
    raise RuntimeError("no point of order %d found" % small)


def sample_g1():
    x = rnd.randrange(P)
    y = o.fq_sqrt((x ** 3 + 4) % P)
    return None if y is None else (x, y)


def sample_g2():
    x = (rnd.randrange(P), rnd.randrange(P))
    y = o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2))
    return None if y is None else (x, y)


for small in (3, 11, 10177):  # points of small order: exercise the exceptional cases of the ladders
    assert h1 % small == 0
    t = point_of_order(o.g1_mul, sample_g1, h1, small)
    add("point of order %d" % small, 1, 1, o.zcash_g1_uncompressed_encode(t))
    add("point of order %d" % small, 1, 3, o.ark_g1_serialize_uncompressed(t))
cnt = 0
while cnt < 3:
    x = (rnd.randrange(P), rnd.randrange(P))
    y = o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2))
    if y is None:
        continue
    cnt += 1
    add("random twist point", 2, 1, o.zcash_g2_uncompressed_encode((x, y)))
    add("random twist point", 2, 2, o.zcash_g2_compressed_encode((x, y)))
    add("random twist point", 2, 3, o.ark_g2_serialize_uncompressed((x, y)))
# G2 small-order: h2 = 13^2 * 23^2 * ...
z = o.Z
h2 = (z ** 8 - 4 * z ** 7 + 5 * z ** 6 - 4 * z ** 4 + 6 * z ** 3 - 4 * z ** 2 - 4 * z + 13) // 9
for small in (13, 23):
    assert h2 % small == 0
    t = point_of_order(o.g2_mul, sample_g2, h2, small)
    add("twist point of order %d" % small, 2, 1, o.zcash_g2_uncompressed_encode(t))
# a1 == 0 special case of the Fq2 square root: x in Fq
while True:
    x = (rnd.randrange(P), 0)
    y = o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2))
    if y is not None:
        add("twist point with x.c1 = 0", 2, 2, o.zcash_g2_compressed_encode((x, y)))
        break

with open(os.path.join(OUT, "edge_cases.json"), "w") as f:
    json.dump({"seed": SEED, "n_powers": N, "scalars": [hex(v) for v in o.derive_scalars(SEED)], "cases": cases}, f,
              indent=1)
# ---- a contribution (powersoftau new_challenge + compute) to the response above, with fixed secrets ------------
sys.path.insert(0, os.path.join(ROOT, "tests"))
import contribute_oracle as co  # noqa: E402

challenge = hashlib.blake2b(resp).digest() + unc
assert len(challenge) == 64 + o.uncompressed_size(N)
w("n8_challenge.bin", challenge)
w("n8_contribution.bin", co.contribute(challenge, N, co.GOLDEN_SECRETS))

print("golden files written:", sorted(os.listdir(OUT)), "edge cases:", len(cases))
