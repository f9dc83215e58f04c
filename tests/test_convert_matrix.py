"""Every per-point conversion instance under every check mask, against the C oracle.

ptau_convert dispatches to 2 groups x 4 input formats x 3 output formats x {light, heavy}
kernel instances, and each instance branches on the three public check bits.  The corpus
below holds, per (group, input format), valid points and every kind of bad record the
decoders distinguish, each re-encoded into every format that can express it.  For every
(group, in, out, mask) cell the product must give the oracle's status per record, its
output bytes on the accepted records and its lowest failing index on the shuffled corpus.

The same matrix runs on the host build of the product's point code (no GPU needed), and
the GPU-only part adds block boundaries, the device entry point, validate-only calls and
the chunk plan of large chunks.
"""
import ctypes as C
import random

import numpy as np
import pytest

import ptau_oracle as o

G1, G2 = 1, 2
ZU, ZC, AU, ML = 1, 2, 3, 4
FMT_NAMES = {ZU: "ZU", ZC: "ZC", AU: "AU", ML: "ML"}
ON_CURVE, SUBGROUP, REJECT_INF = 2, 4, 8
MASKS = [a | b | c for a in (0, ON_CURVE) for b in (0, SUBGROUP) for c in (0, REJECT_INF)]
STRICT = ON_CURVE | SUBGROUP | REJECT_INF
IN_FMTS = (ZU, ZC, AU, ML)
OUT_FMTS = (ZU, AU, ML)
SZ = {G1: {ZU: 96, ZC: 48, AU: 96, ML: 104}, G2: {ZU: 192, ZC: 96, AU: 192, ML: 200}}
P = o.P
NONCANON = (P, P + 1, (1 << 381) - 1)
BLOCK = 128  # PTAU_BLOCK of both groups' convert kernels (kernels.cu)
EDGE_POINTS = 148 * 2 * 128  # kEdgePoints of the chunk plan (capi.cu)


def is_light(in_fmt, checks):
    """launch_one's choice (kernels.cu): compressed input is on the curve by construction,
    so only the subgroup bit makes its instance heavy."""
    if in_fmt == ZC:
        return not (checks & SUBGROUP)
    return not (checks & (ON_CURVE | SUBGROUP))


def chunk_plan(n, chunk):
    """Chunk sizes ptau_convert issues for n points on one GPU (capi.cu): the first and the last
    chunk of a large range are one wave of blocks, so that their copies overlap with work."""
    plan, rem, issued = [], n, 0
    while rem:
        if issued == 0 and rem > 2 * EDGE_POINTS and chunk > EDGE_POINTS:
            k = EDGE_POINTS
        elif rem > chunk + EDGE_POINTS or chunk <= EDGE_POINTS:
            k = min(rem, chunk)
        elif rem > 2 * EDGE_POINTS:
            k = rem - EDGE_POINTS
        else:
            k = min(rem, chunk)
        plan.append(k)
        rem -= k
        issued += 1
    return plan


# ---------------------------------------------------------------------------------------
# encoders from raw coordinate values (any 384-bit value, so non-canonical ones too)
# ---------------------------------------------------------------------------------------
def _be(v):
    return v.to_bytes(48, "big")


def _le(v):
    return v.to_bytes(48, "little")


def mont(v):
    return v * o.MONT_R % P


def enc_unc(g, fmt, x, y, fl=0):
    """ZU / AU record; the two SWFlags bits go to the top of y (G2: y.c1), as the reader sees them."""
    if g == G1:
        yr = y | (fl << 382)
        return _be(x) + _be(yr) if fmt == ZU else _le(x) + _le(yr)
    (x0, x1), (y0, y1) = x, y
    y1r = y1 | (fl << 382)
    return _be(x1) + _be(x0) + _be(y1r) + _be(y0) if fmt == ZU else _le(x0) + _le(x1) + _le(y0) + _le(y1r)


def enc_ml(g, xm, ym, inf=0, pad=bytes(7)):
    """ARK_MONT_LIMBS record from limb values (already Montgomery; may be >= p)."""
    body = _le(xm) + _le(ym) if g == G1 else _le(xm[0]) + _le(xm[1]) + _le(ym[0]) + _le(ym[1])
    return body + bytes([inf]) + pad


def enc_zc(g, x, flags):
    """zcash compressed record: `flags` are the three top bits of the first byte (0x80 compression,
    0x40 infinity, 0x20 sort)."""
    b = bytearray(_be(x) if g == G1 else _be(x[1]) + _be(x[0]))
    b[0] |= flags
    return bytes(b)


def _ml_point(g, q):
    if g == G1:
        return enc_ml(g, mont(q[0]), mont(q[1]))
    return enc_ml(g, (mont(q[0][0]), mont(q[0][1])), (mont(q[1][0]), mont(q[1][1])))


def _largest(g, y):
    return o.fq_lex_largest(y) if g == G1 else o.fq2_lex_largest(y)


def _on_curve(g, q):
    return o.g1_on_curve(q) if g == G1 else o.g2_on_curve(q)


def _decode_raw(g, fmt, rec):
    """Semantic content of a ZU / AU / ZC edge-case record: a finite point (x, y), or None when the
    record has no such content (bad flags, non-canonical, infinity, no square root)."""
    if fmt in (ZU, AU):
        if g == G1:
            f = (lambda b: int.from_bytes(b, "big")) if fmt == ZU else (lambda b: int.from_bytes(b, "little"))
            x, yr = f(rec[:48]), f(rec[48:])
            fl, y = yr >> 382, yr & ((1 << 382) - 1)
            ok = x < P and y < P
        else:
            if fmt == ZU:
                x1, x0, y1r, y0 = (int.from_bytes(rec[48 * i:48 * i + 48], "big") for i in range(4))
            else:
                x0, x1, y0, y1r = (int.from_bytes(rec[48 * i:48 * i + 48], "little") for i in range(4))
            fl, y1 = y1r >> 382, y1r & ((1 << 382) - 1)
            x, y = (x0, x1), (y0, y1)
            ok = max(x0, x1, y0, y1) < P
        return (x, y) if ok and fl == 0 else None
    b = bytearray(rec)
    if b[0] & 0xE0 not in (0x80, 0xA0):
        return None
    greatest = bool(b[0] & 0x20)
    b[0] &= 0x1F
    if g == G1:
        x = int.from_bytes(b, "big")
        if x >= P:
            return None
        y = o.fq_sqrt((x * x * x + o.B_G1) % P)
        if y is None:
            return None
        return (x, y if o.fq_lex_largest(y) == greatest else (-y) % P)
    x = (int.from_bytes(b[48:], "big"), int.from_bytes(b[:48], "big"))
    if max(x) >= P:
        return None
    y = o.fq2_sqrt_alg9(o.fq2_add(o.fq2_mul(o.fq2_sqr(x), x), o.B_G2))
    if y is None:
        return None
    return (x, y if o.fq2_lex_largest(y) == greatest else o.fq2_neg(y))


def _twist_point_real_y(rnd):
    """A point of the G2 curve y^2 = x^3 + 4(1+u) whose y has c1 = 0, so that the compressed sort flag is
    decided by y.c0 (pairing's lexicographic order).  With x = a + bu, x^3 = (a^3 - 3ab^2) + (3a^2 b - b^3)u:
    pick b, solve 3a^2 b - b^3 = -4 for a, and keep x when y^2 = a^3 - 3ab^2 + 4 has a root in Fq."""
    while True:
        b = rnd.randrange(1, P)
        a2 = (b * b * b - 4) * pow(3 * b, -1, P) % P
        a = o.fq_sqrt(a2)
        if a is None:
            continue
        c = (a * a * a - 3 * a * b * b + 4) % P
        y = o.fq_sqrt(c)
        if y is None or y == 0:
            continue
        q = ((a, b), (y, 0))
        assert o.g2_on_curve(q)
        return q


def build_corpus(edge_cases):
    """{(group, in_fmt): [(description, record bytes)]}, deterministic."""
    rnd = random.Random(0x3A7121)
    corpus = {(g, f): [] for g in (G1, G2) for f in IN_FMTS}

    def add(g, f, desc, rec):
        assert len(rec) == SZ[g][f], (desc, len(rec))
        corpus[(g, f)].append((desc, bytes(rec)))

    for g in (G1, G2):
        gen = o.G1_GEN if g == G1 else o.G2_GEN
        mul = o.g1_mul if g == G1 else o.g2_mul
        zero = 0 if g == G1 else (0, 0)
        one = 1 if g == G1 else (1, 0)

        # ---- finite points with one semantic content, in every format that can carry them ----
        points = [("generator", gen)] + [("random subgroup point", mul(gen, rnd.randrange(1, o.R_ORDER)))
                                         for _ in range(3)]
        if g == G2:
            points.append(("twist point with y.c1 = 0", _twist_point_real_y(rnd)))
        seen = {repr(q) for _, q in points}
        for c in edge_cases:
            if c["group"] != g or c["in_fmt"] not in (ZU, AU, ZC):
                continue
            q = _decode_raw(g, c["in_fmt"], bytes.fromhex(c["rec"]))
            if q is not None and repr(q) not in seen:
                seen.add(repr(q))
                points.append(("edge case: " + c["desc"], q))
        # canonical coordinates off the curve
        if g == G1:
            points += [("y + 1", (gen[0], (gen[1] + 1) % P)), ("(0, 0)", (0, 0)), ("(1, 1)", (1, 1)),
                       ("random (x, y)", (rnd.randrange(P), rnd.randrange(P)))]
        else:
            points += [("y.c0 + 1", (gen[0], ((gen[1][0] + 1) % P, gen[1][1]))),
                       ("y.c1 + 1", (gen[0], (gen[1][0], (gen[1][1] + 1) % P))),
                       ("(0, 0)", ((0, 0), (0, 0))),
                       ("random (x, y)", ((rnd.randrange(P), rnd.randrange(P)), (rnd.randrange(P), rnd.randrange(P))))]
        for desc, q in points:
            add(g, ZU, desc, enc_unc(g, ZU, q[0], q[1]))
            add(g, AU, desc, enc_unc(g, AU, q[0], q[1]))
            add(g, ML, desc, _ml_point(g, q))
            if _on_curve(g, q):
                s = 0x20 if _largest(g, q[1]) else 0
                add(g, ZC, desc, enc_zc(g, q[0], 0x80 | s))
                add(g, ZC, desc + ", other sort flag", enc_zc(g, q[0], 0x80 | (s ^ 0x20)))
        # the edge-case records as committed, in their own format (non-residue x, flags, ...)
        for c in edge_cases:
            if c["group"] == g:
                add(g, c["in_fmt"], "edge case record: " + c["desc"], bytes.fromhex(c["rec"]))

        # ---- infinity in every encoding ----
        for f in (ZU, AU):
            add(g, f, "ark infinity flag, zero coordinates", enc_unc(g, f, zero, zero, 1))
            add(g, f, "ark infinity flag, ark zero() coordinates", enc_unc(g, f, zero, one, 1))
            add(g, f, "ark infinity flag, finite coordinates", enc_unc(g, f, gen[0], gen[1], 1))
            add(g, f, "ark infinity flag, y off curve", enc_unc(g, f, gen[0], one, 1))
        zu_inf = bytearray(SZ[g][ZU])
        zu_inf[0] = 0x40
        add(g, ZU, "zcash infinity 0x40", zu_inf)
        zu_inf[0] = 0x60
        add(g, ZU, "zcash infinity + sort bit", zu_inf)
        zu_inf[0], zu_inf[-1] = 0x40, 1
        add(g, ZU, "zcash infinity + stray byte", zu_inf)
        zc_inf = bytearray(SZ[g][ZC])
        zc_inf[0] = 0xC0
        add(g, ZC, "zcash infinity 0xC0", zc_inf)
        zc_inf[0] = 0xE0
        add(g, ZC, "infinity + sort bit", zc_inf)
        zc_inf[0], zc_inf[-1] = 0xC0, 1
        add(g, ZC, "infinity + stray byte", zc_inf)
        zc_inf[0], zc_inf[-1] = 0xC1, 0
        add(g, ZC, "infinity + stray bit in the first byte", zc_inf)
        zc_inf[0] = 0x40
        add(g, ZC, "infinity without compression bit", zc_inf)
        gm = _ml_point(g, gen)
        z = 0 if g == G1 else (0, 0)
        r1 = o.MONT_R if g == G1 else (o.MONT_R, 0)
        add(g, ML, "ML infinity, zero limbs", enc_ml(g, z, z, 1))
        add(g, ML, "ML infinity, ark zero() limbs", enc_ml(g, z, r1, 1))
        add(g, ML, "ML infinity, generator limbs", gm[:-8] + bytes([1]) + bytes(7))
        add(g, ML, "ML infinity byte 0x80, generator limbs", gm[:-8] + bytes([0x80]) + bytes(7))
        add(g, ML, "ML generator, stray padding bytes", gm[:-8] + bytes([0]) + bytes([0xFF] * 7))
        add(g, ML, "ML infinity, stray padding bytes", enc_ml(g, z, r1, 1, bytes([0x5A] * 7)))

        # ---- non-canonical coordinates, in every position ----
        if g == G1:
            slots = {"x": lambda v: (v, gen[1]), "y": lambda v: (gen[0], v)}
        else:
            (gx0, gx1), (gy0, gy1) = gen
            slots = {"x.c0": lambda v: ((v, gx1), gen[1]), "x.c1": lambda v: ((gx0, v), gen[1]),
                     "y.c0": lambda v: (gen[0], (v, gy1)), "y.c1": lambda v: (gen[0], (gy0, v))}
        for name, put in slots.items():
            for v in NONCANON:
                x, y = put(v)
                for f in (ZU, AU):
                    add(g, f, "%s = %#x" % (name, v), enc_unc(g, f, x, y))
                    # both faults: the order x >= p -> flags -> y (G2: y.c1) >= p decides the kind
                    add(g, f, "%s = %#x and flags 11" % (name, v), enc_unc(g, f, x, y, 3))
                    add(g, f, "%s = %#x and infinity flag" % (name, v), enc_unc(g, f, x, y, 1))
            for v in NONCANON + ((1 << 384) - 1,):
                xm, ym = put(v)  # limbs: the value stands for itself, the others are Montgomery of the generator
                if g == G1:
                    xm = xm if name == "x" else mont(xm)
                    ym = ym if name == "y" else mont(ym)
                else:
                    xm = tuple(c if name == "x.c%d" % i else mont(c) for i, c in enumerate(xm))
                    ym = tuple(c if name == "y.c%d" % i else mont(c) for i, c in enumerate(ym))
                add(g, ML, "ML limbs %s = %#x" % (name, v), enc_ml(g, xm, ym))
                add(g, ML, "ML limbs %s = %#x, infinity" % (name, v), enc_ml(g, xm, ym, 1))
        xs = {"x": lambda v: v} if g == G1 else {"x.c0": lambda v: (v, gen[0][1]), "x.c1": lambda v: (gen[0][0], v)}
        for name, put in xs.items():
            for v in NONCANON:
                add(g, ZC, "compressed %s = %#x" % (name, v), enc_zc(g, put(v), 0x80))
                add(g, ZC, "compressed %s = %#x, sort flag" % (name, v), enc_zc(g, put(v), 0xA0))

        # ---- flag bits ----
        for f in (ZU, AU):
            add(g, f, "flags 11 on the generator", enc_unc(g, f, gen[0], gen[1], 3))
            add(g, f, "PositiveY flag on the generator (accepted, stripped)", enc_unc(g, f, gen[0], gen[1], 2))
            xc = gen[0] | (1 << 383) if g == G1 else (gen[0][0], gen[0][1] | (1 << 383))
            add(g, f, "compression bit in an uncompressed x", enc_unc(g, f, xc, gen[1]))
        add(g, ZC, "generator without compression bit", enc_zc(g, gen[0], 0))
        add(g, ZC, "generator without compression bit, sort flag", enc_zc(g, gen[0], 0x20))
    return corpus


def _edge_cases():
    import json
    import os

    from conftest import GOLDEN

    with open(os.path.join(GOLDEN, "edge_cases.json")) as fh:
        return json.load(fh)["cases"]


@pytest.fixture(scope="module")
def corpus():
    return build_corpus(_edge_cases())


def _cells():
    return [(g, fi, fo, m) for g in (G1, G2) for fi in IN_FMTS for fo in OUT_FMTS for m in MASKS]


def _recs(corpus, g, f):
    return b"".join(r for _, r in corpus[(g, f)])


def _shuffled(corpus, g, f, seed):
    recs = list(corpus[(g, f)])
    random.Random(seed).shuffle(recs)
    return recs


# ---------------------------------------------------------------------------------------
# CPU: the corpus itself, the oracle's Montgomery output, and the host build of the kernels
# ---------------------------------------------------------------------------------------
def test_corpus_covers_every_status(corpus, cref):
    """Every (group, input format) corpus holds accepted records and every rejection kind its format can produce
    under the strict mask, so the matrix below compares something in each cell."""
    for (g, f), recs in corpus.items():
        _, st = cref.convert(g, f, b"".join(r for _, r in recs), AU, STRICT)
        _, st0 = cref.convert(g, f, b"".join(r for _, r in recs), AU, 0)
        want = {0, 1, 2, 3, 4, 5}
        if f == ML:
            want -= {2}  # Montgomery records have no flag bits
        assert want <= set(st), (g, f, sorted(set(st)))
        assert 0 in st0 and any(s != 0 for s in st0)
    assert sum(len(v) for v in corpus.values()) >= 250


def test_oracle_direct_ml_equals_via_ark_uncompressed(corpus, cref):
    """The oracle's in -> ARK_MONT_LIMBS equals its in -> ARK_UNCOMPRESSED -> ARK_MONT_LIMBS on every record it
    accepts: both must be ark's in-memory GroupAffine of the same point (infinity = zero() = (0, 1, true))."""
    for (g, f), recs in corpus.items():
        data = b"".join(r for _, r in recs)
        ro = SZ[g][ML]
        for m in MASKS:
            direct, st = cref.convert(g, f, data, ML, m)
            au, st_au = cref.convert(g, f, data, AU, m)
            assert st == st_au, (g, f, m)
            via, _ = cref.convert(g, AU, au, ML, 0)
            for i, (desc, _) in enumerate(recs):
                if st[i] == 0:
                    assert direct[i * ro:(i + 1) * ro] == via[i * ro:(i + 1) * ro], (g, FMT_NAMES[f], m, i, desc)


def test_oracle_ml_infinity_is_ark_zero(cref):
    """Infinity in every input encoding becomes ark's zero() = (0, 1, true) in Montgomery form, as the Python
    oracle's record of it."""
    for g, zero_rec in ((G1, o.g1_mont_record(0, 1, True)), (G2, o.g2_mont_record((0, 0), (1, 0), True))):
        one = 1 if g == G1 else (1, 0)
        zero = 0 if g == G1 else (0, 0)
        zc = bytearray(SZ[g][ZC])
        zc[0] = 0xC0
        for f, rec in ((ZC, bytes(zc)), (ZU, enc_unc(g, ZU, zero, one, 1)), (AU, enc_unc(g, AU, zero, one, 1)),
                       (ML, zero_rec)):
            for m in (0, ON_CURVE, SUBGROUP, ON_CURVE | SUBGROUP):
                out, st = cref.convert(g, f, rec, ML, m)
                assert st == [0] and out == zero_rec, (g, FMT_NAMES[f], m)


def _hostemul_convert(lib, g, fi, data, fo, m):
    n = len(data) // SZ[g][fi]
    out = (C.c_uint8 * max(n * SZ[g][fo], 1))()
    st = (C.c_uint32 * max(n, 1))()
    assert lib.hostemul_convert(g, fi, data, fo, out, C.c_size_t(n), m, st) == 0
    return bytes(out)[:n * SZ[g][fo]], list(st)[:n]


def test_matrix_host_build(corpus, cref, hostemul):
    """The whole (group, in, out, mask) matrix on the host build of the product's point code: per-record status and,
    on the records the oracle accepts, output bytes.  The host build instantiates the heavy instances only (checks
    compiled in; a mask without checks skips them at run time): the light instances exist on the GPU only and are
    covered by the GPU matrix."""
    bad = []
    for g, fi, fo, m in _cells():
        recs = corpus[(g, fi)]
        data = _recs(corpus, g, fi)
        want, wst = cref.convert(g, fi, data, fo, m)
        got, gst = _hostemul_convert(hostemul, g, fi, data, fo, m)
        ro = SZ[g][fo]
        for i, (desc, _) in enumerate(recs):
            if gst[i] != wst[i]:
                bad.append((g, FMT_NAMES[fi], FMT_NAMES[fo], m, desc, "status", gst[i], wst[i]))
            elif wst[i] == 0 and got[i * ro:(i + 1) * ro] != want[i * ro:(i + 1) * ro]:
                bad.append((g, FMT_NAMES[fi], FMT_NAMES[fo], m, desc, "bytes"))
    assert not bad, "%d disagreements, first: %s" % (len(bad), bad[:8])


def test_both_instances_in_every_pair():
    """The masks of the matrix run both the light and the heavy instance of every (group, in, out) kernel."""
    for fi in IN_FMTS:
        assert {is_light(fi, m) for m in MASKS} == {True, False}, fi


def test_chunk_plan_branches():
    """The chunk sizes the large-chunk test expects exercise every branch of the plan (first wave, full chunks,
    the chunk that leaves exactly one wave, the short tail)."""
    assert chunk_plan(75_777, 50_000) == [37_888, 37_889]
    assert chunk_plan(120_000, 50_000) == [37_888, 44_224, 37_888]
    assert chunk_plan(150_017, 50_000) == [37_888, 50_000, 50_000, 12_129]
    assert chunk_plan(1000, 96) == [96] * 10 + [40]
    for n in (1, 75_776, 75_777, 87_888, 113_664, 300_001):
        assert sum(chunk_plan(n, 50_000)) == n


# ---------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------
def _lib():
    from kzg_setup_powersoftau_b200 import _ffi

    return _ffi.lib()


def _raw_convert(ctx, g, fi, data, fo, m, with_out=True):
    """ptau_convert through the C ABI: (rc, bad index, bad kind, output bytes or None)."""
    n = len(data) // SZ[g][fi]
    src = np.frombuffer(data, dtype=np.uint8)
    dst = np.zeros(max(n * SZ[g][fo], 1), dtype=np.uint8) if with_out else None
    bi, bk = C.c_uint64(0), C.c_int(0)
    rc = _lib().ptau_convert(ctx._h, g, fi, src.ctypes.data, fo, dst.ctypes.data if with_out else None, n, m,
                             C.byref(bi), C.byref(bk))
    return rc, (bi.value if rc > 0 else None), (bk.value if rc > 0 else None), \
        (dst[:n * SZ[g][fo]].tobytes() if with_out else None)


def _first_bad(st):
    for i, s in enumerate(st):
        if s:
            return i, s
    return None


@pytest.mark.gpu
def test_matrix_gpu(corpus, cref, ctx):
    """Per cell: each record alone gives the oracle's status (index 0 on failure); one batch of the accepted records
    gives the oracle's bytes; the shuffled corpus gives the oracle's lowest failing (index, kind), with and without an
    output buffer."""
    bad = []
    light = heavy = 0
    for g, fi, fo, m in _cells():
        light += is_light(fi, m)
        heavy += not is_light(fi, m)
        cell = (g, FMT_NAMES[fi], FMT_NAMES[fo], m)
        recs = corpus[(g, fi)]
        ro = SZ[g][fo]
        want, wst = cref.convert(g, fi, _recs(corpus, g, fi), fo, m)
        for i, (desc, r) in enumerate(recs):
            rc, bi, bk, out = _raw_convert(ctx, g, fi, r, fo, m)
            if rc != wst[i] or (rc and (bi, bk) != (0, rc)):
                bad.append(cell + (desc, "status", rc, bi, wst[i]))
            elif rc == 0 and out != want[i * ro:(i + 1) * ro]:
                bad.append(cell + (desc, "single-record bytes"))
        ok = [i for i in range(len(recs)) if wst[i] == 0]
        assert ok, cell
        rc, _, _, out = _raw_convert(ctx, g, fi, b"".join(recs[i][1] for i in ok), fo, m)
        if rc != 0 or out != b"".join(want[i * ro:(i + 1) * ro] for i in ok):
            bad.append(cell + ("batch of accepted records", rc))
        sh = _shuffled(corpus, g, fi, seed=((g * 8 + fi) * 8 + fo) * 16 + m)
        data = b"".join(r for _, r in sh)
        _, sst = cref.convert(g, fi, data, fo, m)
        fb = _first_bad(sst)
        for with_out in (True, False):
            rc, bi, bk, _ = _raw_convert(ctx, g, fi, data, fo, m, with_out)
            got = None if rc == 0 else (bi, bk)
            if got != fb or (rc and rc != bk):
                bad.append(cell + ("shuffled corpus", with_out, got, fb))
    assert not bad, "%d disagreements, first: %s" % (len(bad), bad[:8])
    assert light + heavy == 192 and light > 0 and heavy > 0


def _valid_points(cref, g, fmt, n, seed):
    tau = random.Random(seed).randrange(2, o.R_ORDER)
    zu = cref.generate(g, ZU, 1, tau, 0, n, 8)
    if fmt == ZU:
        return zu
    if fmt == ZC:
        return cref.generate(g, ZC, 1, tau, 0, n, 8)
    out, st = cref.convert(g, ZU, zu, fmt, 0, 8)
    assert not any(st)
    return out


def _inf_record(g, fmt):
    if fmt == ML:
        return enc_ml(g, 0 if g == G1 else (0, 0), o.MONT_R if g == G1 else (o.MONT_R, 0), 1)
    if fmt == ZC:
        return bytes([0xC0]) + bytes(SZ[g][ZC] - 1)
    return enc_unc(g, fmt, 0 if g == G1 else (0, 0), 1 if g == G1 else (1, 0), 1)


def _bad_record(g, fmt, good):
    if fmt == ML:  # x (G2: x.c0) limbs = p
        return _le(P) + good[48:]
    if fmt == ZC:  # no compression bit
        return bytes([good[0] & 0x7F]) + good[1:]
    b = bytearray(good)  # flags 11
    if fmt == ZU:
        b[SZ[g][fmt] // 2] |= 0xC0
    else:
        b[-1] |= 0xC0
    return bytes(b)


@pytest.mark.gpu
@pytest.mark.parametrize("g", [G1, G2])
@pytest.mark.parametrize("fi,fo", [(ML, ML), (ZC, ML), (ZU, AU)])
def test_block_boundaries(ctx, cref, g, fi, fo):
    """Counts around the 128-record blocks, with an infinity record last (an odd count of 104-byte records leaves an
    8-byte staging tail), under the light (0) and the heavy (SUBGROUP) instance; then bad records at 0, 127, 128 and
    n - 1, peeled off lowest first."""
    ri = SZ[g][fi]
    pool = _valid_points(cref, g, fi, 1000, seed=g * 10 + fi)
    for n in (1, BLOCK - 1, BLOCK, BLOCK + 1, 2 * BLOCK - 1, 2 * BLOCK, 2 * BLOCK + 1, 1000):
        recs = [pool[i * ri:(i + 1) * ri] for i in range(n - 1)] + [_inf_record(g, fi)]
        data = b"".join(recs)
        for m in (0, SUBGROUP):
            want, st = cref.convert(g, fi, data, fo, m, 8)
            assert not any(st)
            rc, _, _, out = _raw_convert(ctx, g, fi, data, fo, m)
            assert rc == 0 and out == want, (n, m)
        pos = sorted({p for p in (0, BLOCK - 1, BLOCK, n - 1) if p < n})
        for p in pos:
            recs[p] = _bad_record(g, fi, recs[p])
        for p in pos:
            data = b"".join(recs)
            _, st = cref.convert(g, fi, data, fo, STRICT, 8)
            fb = _first_bad(st)
            assert fb is not None and fb[0] == p
            rc, bi, bk, _ = _raw_convert(ctx, g, fi, data, fo, STRICT)
            assert (rc, bi, bk) == (fb[1], p, fb[1]), (n, p)
            recs[p] = pool[p * ri:(p + 1) * ri] if p < n - 1 else _inf_record(g, fi)


def _status_decode():
    """ptau_status_decode with the header's signature, bound here on a fresh function object."""
    fn = _lib()["ptau_status_decode"]
    fn.restype = C.c_int
    fn.argtypes = [C.c_uint64, C.POINTER(C.c_uint64)]

    def dec(word):
        idx = C.c_uint64(0xDEAD)
        kind = fn(word, C.byref(idx))
        return kind, idx.value

    return dec


@pytest.mark.gpu
def test_device_entry_point(ctx, cref):
    """Three ptau_convert_device launches share one status word (base_index 5000, 1000, 0, launched in that order);
    the word folds to (lowest index << 8) | kind, ptau_status_decode reads it back, the output bytes equal the host
    path's, and malformed arguments are refused."""
    import torch

    from kzg_setup_powersoftau_b200 import _ffi

    L = _lib()
    dec = _status_decode()
    assert dec(_ffi.STATUS_NONE) == (0, 0xDEAD)
    assert dec((77 << 8) | 5) == (5, 77)

    g, fi, fo, m, n = G1, ZU, AU, SUBGROUP, 1000
    ri, ro = SZ[g][fi], SZ[g][fo]
    pool = _valid_points(cref, g, fi, 3 * n, seed=99)
    dev = torch.device("cuda", 0)
    cofactor = next(bytes.fromhex(c["rec"]) for c in _edge_cases()
                    if c["group"] == g and c["in_fmt"] == fi and c["desc"].startswith("random curve point"))
    for bads, want in ((((1000, 7, "flags"), (0, 900, "subgroup")), (900 << 8) | 5),
                       (((5000, 3, "subgroup"), (1000, 20, "flags")), (1020 << 8) | 2)):
        launches = []
        for k, base in enumerate((5000, 1000, 0)):
            recs = [pool[(k * n + i) * ri:(k * n + i + 1) * ri] for i in range(n)]
            for b, j, what in bads:
                if b == base:
                    recs[j] = _bad_record(g, fi, recs[j]) if what == "flags" else cofactor
            launches.append((base, b"".join(recs)))
        status = torch.full((1,), -1, dtype=torch.int64, device=dev)
        outs = []
        for base, data in launches:
            d_in = torch.frombuffer(bytearray(data), dtype=torch.uint8).to(dev)
            d_out = torch.zeros(n * ro, dtype=torch.uint8, device=dev)
            ctx.convert_device(g, fi, d_in.data_ptr(), fo, d_out.data_ptr(), n, m, status.data_ptr(), base_index=base)
            outs.append((d_in, d_out))
        torch.cuda.synchronize()
        word = int(status.item()) & 0xFFFFFFFFFFFFFFFF
        assert word == want
        assert dec(word) == (want & 0xFF, want >> 8)
        for (base, data), (_, d_out) in zip(launches, outs):
            rc, bi, bk, host = _raw_convert(ctx, g, fi, data, fo, m)
            assert bytes(d_out.cpu().numpy()) == host
            _, st = cref.convert(g, fi, data, fo, m, 8)
            fb = _first_bad(st)
            assert (None if rc == 0 else (bi, bk)) == fb

    d_in = torch.frombuffer(bytearray(pool[:16 * ri + 16]), dtype=torch.uint8).to(dev)
    d_out = torch.zeros(16 * SZ[g][ML] + 16, dtype=torch.uint8, device=dev)
    status = torch.full((1,), -1, dtype=torch.int64, device=dev)
    a_in, a_out, a_st = d_in.data_ptr(), d_out.data_ptr(), status.data_ptr()

    def call(gpu=0, group=g, in_ptr=a_in, out_fmt=fo, out_ptr=a_out, st=a_st, in_fmt=fi):
        return L.ptau_convert_device(ctx._h, gpu, group, in_fmt, in_ptr, out_fmt, out_ptr, 16, m, 0, st, None)

    assert call() == 0
    torch.cuda.synchronize()
    assert int(status.item()) == -1
    assert call(in_ptr=a_in + 8) == _ffi.ERR_ARG
    assert call(out_ptr=a_out + 4) == _ffi.ERR_ARG
    assert call(out_fmt=ZC) == _ffi.ERR_ARG
    assert call(out_fmt=0) == _ffi.ERR_ARG
    assert call(in_fmt=5) == _ffi.ERR_ARG
    assert call(group=3) == _ffi.ERR_ARG
    assert call(gpu=ctx.n_gpus) == _ffi.ERR_ARG
    assert call(gpu=-1) == _ffi.ERR_ARG
    assert call(st=None) == _ffi.ERR_ARG
    torch.cuda.synchronize()
    assert int(status.item()) == -1


@pytest.mark.gpu
def test_validate_only_all_valid(ctx, cref):
    """out = NULL on an all-valid batch: success, like the call with a buffer."""
    for g in (G1, G2):
        for fi in IN_FMTS:
            data = _valid_points(cref, g, fi, 300, seed=7 + fi) + _inf_record(g, fi)
            for fo in OUT_FMTS:
                for m in (0, SUBGROUP, ON_CURVE | SUBGROUP):
                    assert _raw_convert(ctx, g, fi, data, fo, m, True)[:3] == (0, None, None)
                    assert _raw_convert(ctx, g, fi, data, fo, m, False)[:3] == (0, None, None)


@pytest.mark.gpu
def test_large_chunk_plan(cref):
    """chunk_points = 50 000 > one wave: the first-wave chunk, full chunks, the chunk that leaves exactly one wave and
    the short tail all run; every output byte equals the oracle's, the launch count is the plan's, and a bad record
    at the first and at the last index of every chunk is the one reported."""
    import kzg_setup_powersoftau_b200 as kz

    rnd = np.random.default_rng(50_000)
    g, fi, fo, chunk = G1, AU, ZU, 50_000
    with kz.Context(1, chunk_points=chunk) as c:
        for n in (75_777, 120_000, 150_017):
            recs = rnd.integers(0, 256, size=(n, 96), dtype=np.uint8)
            recs[:, 47] &= 0x0F  # x < 2^380 < p
            recs[:, 95] &= 0x0F  # y < p, no flag bits
            data = recs.tobytes()
            want, st = cref.convert(g, fi, data, fo, 0, 8)
            assert not any(st)
            out = c.convert(g, fi, recs, fo, 0)
            assert out.tobytes() == want
            plan = chunk_plan(n, chunk)
            assert c.timing()["kernel_launches"] == len(plan)
            starts = np.cumsum([0] + plan)
            for lo, hi in zip(starts[:-1], starts[1:]):
                for i in (int(lo), int(hi) - 1):
                    keep = recs[i, 95]
                    recs[i, 95] |= 0xC0
                    with pytest.raises(kz.PtauError) as e:
                        c.convert(g, fi, recs, fo, 0)
                    assert (e.value.code, e.value.index) == (kz.BAD_FLAGS, i)
                    recs[i, 95] = keep
