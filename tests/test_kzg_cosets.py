"""Coset openings of KZG10 (ptau_kzg_open_cosets / ptau_kzg_check_cosets, KZG10.open_cosets / check_cosets): the
strided quotient scan and the NTT of csrc/kzg_coset.cuh against big-integer division and O(k^2) evaluation on the host
build, a big-integer restatement of the scheme, and the GPU against known-tau setups, open_many and check_many."""
import ctypes
import os
import random

import numpy as np
import pytest

import ptau_oracle as o
from conftest import ROOT

R = o.R_ORDER
ZU, ML = 1, 4
LG_CHUNK = 5           # kKzgLgChunk
LG_CARRY_THREADS = 10  # kKzgLgCarryThreads
OMEGA = 0x16A2A19EDFE81F20D09B681922C813B4B63683508C2280B93829971F439F0D2B


@pytest.fixture(scope="module")
def he():
    """Host build of fr.cuh and the coset items (tests/host_emul/hostemul_coset.cpp)."""
    d = os.path.join(ROOT, "tests", "host_emul")
    so = os.path.join(d, "libptau_hostemul_coset.so")
    csrc = os.path.join(ROOT, "kzg_setup_powersoftau_b200", "csrc")
    deps = [os.path.join(d, "hostemul_coset.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                       if f.endswith((".cuh", ".inc", ".h"))]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        import subprocess

        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                               os.path.join(d, "hostemul_coset.cpp")])
    return ctypes.CDLL(so)


def le(v: int) -> bytes:
    return int(v).to_bytes(32, "little")


def ints(raw: bytes):
    return [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(len(raw) // 32)]


def root(e):
    return pow(OMEGA, 1 << (32 - e), R)


def divide(p, k, c):
    """p = (X^k - c) q + r by big-integer long division: (q, r) with len(r) = k."""
    rem = list(p) + [0] * max(k - len(p), 0)
    q = [0] * max(len(p) - k, 0)
    for i in range(len(p) - 1, k - 1, -1):
        t = rem[i] % R
        q[i - k] = t
        rem[i] = 0
        rem[i - k] = (rem[i - k] + c * t) % R
    return q, [x % R for x in rem[:k]]


def evaluate(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + c) % R
    return acc


# ---------------------------------------------------------------------------------------------- CPU
def test_root_of_unity():
    """omega = 7^((r - 1) / 2^32) has order exactly 2^32; coset_points names k distinct points of h <omega_k>."""
    import kzg_setup_powersoftau_b200 as kz

    assert OMEGA == kz.FR_ROOT_OF_UNITY == pow(7, (R - 1) >> 32, R)
    assert pow(OMEGA, 1 << 32, R) == 1 and pow(OMEGA, 1 << 31, R) == R - 1
    for e in (0, 1, 5, 20):
        pts = kz.coset_points(e, 3)
        assert len(pts) == 1 << e and pts[0] == 3 and len(set(pts)) == 1 << e
        assert all(pow(x, 1 << e, R) == pow(3, 1 << e, R) for x in pts[:64])


def test_fr_sub_and_powers_on_edge_limbs(he):
    """fr_mul (a b R^-1), fr_add, fr_sub, fr_is_canonical, fr_mont_one and fr_pow_bits of csrc/fr.cuh against Python
    integers, on edge limbs."""
    rnd = random.Random(1)
    edges = [0, 1, 2, R - 1, R - 2, 2 ** 32 - 1, 2 ** 32, 2 ** 64 - 1, 2 ** 255 % R, (R - 1) // 2, (R + 1) // 2]
    edges += [sum(0xFFFFFFFF << (32 * i) for i in range(k)) % R for k in range(1, 9)]
    edges += [((R >> (32 * i)) << (32 * i)) - 1 for i in range(1, 8)]
    edges += [rnd.randrange(R) for _ in range(20)]
    out = ctypes.create_string_buffer(32)

    def op(k, a, b):
        he.hostemul_coset_fr_op(k, le(a), le(b), out)
        return int.from_bytes(out.raw, "little")

    rinv = pow(2 ** 256, -1, R)
    for a in edges:
        for b in edges:
            assert op(0, a, b) == (a - b) % R, (a, b)
            assert op(3, a, b) == a * b * rinv % R, (a, b)
            assert op(4, a, b) == (a + b) % R, (a, b)
    for a, canon in ((0, 1), (R - 1, 1), (R, 0), (R + 1, 0), (2 ** 256 - 1, 0), (R | (1 << 255), 0), (2 ** 254, 1)):
        assert op(5, a, 0) == canon, a
    assert op(1, 0, 0) == 2 ** 256 % R
    for a in edges[:12] + edges[-5:]:
        for x in (0, 1, 2, 3, 2 ** 20 - 1, 2 ** 32 + 5, 2 ** 64 - 1, rnd.randrange(2 ** 64)):
            assert op(2, a, x) == pow(a, x, R), (a, x)


def _host_quotient(lib, p, lg_k, c, lg_chunk, lg_threads):
    n, k = len(p), 1 << lg_k
    q = ctypes.create_string_buffer(max(n - k, 1) * 32)
    rem = ctypes.create_string_buffer(k * 32)
    bad = lib.hostemul_coset_quotient(b"".join(le(x) for x in p), ctypes.c_size_t(n), lg_k, le(c), lg_chunk,
                                      lg_threads, q, rem)
    return bad, ints(q.raw[:max(n - k, 0) * 32]), ints(rem.raw)


@pytest.mark.parametrize("lg_k", [0, 1, 5, 10])
@pytest.mark.parametrize("lg_chunk,lg_threads", [(0, 2), (1, 2), (LG_CHUNK, 2), (0, LG_CARRY_THREADS),
                                                 (LG_CHUNK, LG_CARRY_THREADS), (1, LG_CARRY_THREADS)])
def test_strided_quotient_equals_division(he, lg_k, lg_chunk, lg_threads):
    """The strided blocked scan (chunks of 1, 2, 32 rows, a carry segment of at most 4 or 1024 threads) gives exactly
    the quotient and remainder of long division by X^k - c: n around k, multiples of k, the chunk and the block of
    chunks, several runs per carry thread, c = 0, 1, r - 1 and random, p = (X^k - c) s, whose remainder is 0 and
    quotient s, and the constant polynomials 0 and r - 1.  At k = 1 this is synthetic division by X - z, the witness
    polynomial of ptau_kzg_open with r = [p(z)]."""
    rnd = random.Random(lg_k * 101 + lg_chunk * 7 + lg_threads)
    k, L, T = 1 << lg_k, 1 << lg_chunk, 1 << lg_threads
    sizes = {0, 1, 2, max(k - 1, 0), k, k + 1, 3 * k - 1, 3 * k + 1, k * L - 1, k * L, k * L + 1, k * L * T - 1,
             k * L * T, k * L * T + 1}
    if k * L * T < 4096:
        sizes |= {5 * k * L * T + 3, 3 * k * L * T + 5, 17 * k * L * T - 3}  # several runs per carry thread
    for n in sorted(s for s in sizes if s <= 40000):
        p = [rnd.randrange(R) for _ in range(n)]
        for c in (0, 1, R - 1, rnd.randrange(R)):
            bad, q, rem = _host_quotient(he, p, lg_k, c, lg_chunk, lg_threads)
            assert bad == 0 and (q, rem) == divide(p, k, c), (n, c)
        if n > k:
            c = rnd.randrange(R)
            s = [rnd.randrange(R) for _ in range(n - k)]
            pp = [((s[i - k] if i >= k else 0) - c * (s[i] if i < n - k else 0)) % R for i in range(n)]
            bad, q, rem = _host_quotient(he, pp, lg_k, c, lg_chunk, lg_threads)
            assert bad == 0 and q == s and rem == [0] * k, n
    for n in (k * L + 1, k * L * T + 1):
        for v in (0, R - 1):
            if n <= 40000:
                c = rnd.randrange(R)
                assert _host_quotient(he, [v] * n, lg_k, c, lg_chunk, lg_threads) == (0, *divide([v] * n, k, c)), (n, v)


def test_strided_quotient_flags_non_canonical(he):
    """A coefficient >= r first, in the middle or last sets the flag, for k = 1 and k = 32."""
    n = 300
    for lg_k in (0, 5):
        for at in (0, n // 2, n - 1):
            for bad_value in (R, 2 ** 256 - 1):
                p = [7] * n
                p[at] = bad_value
                assert _host_quotient(he, p, lg_k, 3, LG_CHUNK, LG_CARRY_THREADS)[0] == 1, (lg_k, at)
        assert _host_quotient(he, [R - 1] * n, lg_k, 3, LG_CHUNK, LG_CARRY_THREADS)[0] == 0


def _host_ntt(lib, rows, e, w, hs):
    k = 1 << e
    out = ctypes.create_string_buffer(len(rows) * k * 32)
    lib.hostemul_ntt(b"".join(le(x) for row in rows for x in row), ctypes.c_size_t(len(rows)), e, le(w),
                     b"".join(le(h) for h in hs) if hs is not None else None, out)
    vals = ints(out.raw)
    return [vals[i * k:(i + 1) * k] for i in range(len(rows))]


def test_ntt_equals_evaluation_and_interpolation(he):
    """The NTT items give sum_j a_j h^j w^(jm) (evaluation on the coset h <omega_k>, natural order) and, with
    w^-1 and the unscale k^-1 h^-j, the interpolant back, for e = 0..10, on a coset and on the subgroup (h = 1)."""
    rnd = random.Random(3)
    for e in range(11):
        k, w = 1 << e, root(e)
        rows = [[rnd.randrange(R) for _ in range(k)] for _ in range(2)]
        hs = [rnd.randrange(1, R), 1]
        got = _host_ntt(he, rows, e, w, hs)
        for row, h, g in zip(rows, hs, got):
            pts = [h * pow(w, m, R) % R for m in range(k)]
            if e <= 8:
                assert g == [evaluate(row, x) for x in pts], e
            else:
                assert all(g[m] == evaluate(row, pts[m]) for m in rnd.sample(range(k), 12)), e
            inv = _host_ntt(he, [g], e, pow(w, -1, R), None)[0]  # unscaled inverse NTT
            kinv, hinv = pow(k, -1, R), pow(h, -1, R)
            assert [x * kinv * pow(hinv, j, R) % R for j, x in enumerate(inv)] == row, e


def _restated_check(tau, k, items, rhos, tau_k):
    """The check equation of ptau_kzg_check_cosets in the exponent, with G1 points as their discrete logs at a known
    tau: sum rho_i (C_i + c_i pi_i) - sum_j (sum_i rho_i I_ij) tau^j - tau_k sum rho_i pi_i == 0."""
    w = root(k.bit_length() - 1)
    lhs, a = 0, [0] * k
    for (C, h, vals, pi), rho in zip(items, rhos):
        c = pow(h, k, R)
        kinv, hinv = pow(k, -1, R), pow(h, -1, R)
        for j in range(k):
            I = kinv * pow(hinv, j, R) * sum(v * pow(w, -j * m % k, R) for m, v in enumerate(vals)) % R
            a[j] = (a[j] + rho * I) % R
        lhs += rho * (C + c * pi) - tau_k * rho * pi
    return (lhs - evaluate(a, tau)) % R == 0


def test_restated_open_and_check():
    """Big-integer restatement of the scheme at a known tau on the G1 side: the proof q(tau) of each coset opening
    satisfies C + c pi - I(tau) = tau^k pi, the values are p on the coset, and the batched check accepts honest items
    and rejects a false value, a swapped proof and a wrong tau^k."""
    rnd = random.Random(11)
    tau = rnd.randrange(R)
    for e in (0, 2, 4):
        k, w = 1 << e, root(e)
        p = [rnd.randrange(R) for _ in range(3 * k + 5)]
        C = evaluate(p, tau)
        items = []
        for h in (1, pow(root(e + 1), 1, R), rnd.randrange(1, R)):
            q, r = divide(p, k, pow(h, k, R))
            vals = [evaluate([x * pow(h, j, R) % R for j, x in enumerate(r)], pow(w, m, R)) for m in range(k)]
            assert vals == [evaluate(p, h * pow(w, m, R) % R) for m in range(k)]
            items.append((C, h, vals, evaluate(q, tau)))
        rhos = [rnd.randrange(2 ** 127) for _ in items]
        tk = pow(tau, k, R)
        assert _restated_check(tau, k, items, rhos, tk)
        bad = list(items)
        bad[1] = (bad[1][0], bad[1][1], [bad[1][2][0] + 1] + bad[1][2][1:], bad[1][3])
        assert not _restated_check(tau, k, bad, rhos, tk)
        swapped = list(items)
        swapped[0], swapped[2] = items[0][:3] + (items[2][3],), items[2][:3] + (items[0][3],)
        assert not _restated_check(tau, k, swapped, rhos, tk)
        assert not _restated_check(tau, k, items, rhos, tk * tau % R)


# ---------------------------------------------------------------------------------------------- GPU
def _kz():
    import kzg_setup_powersoftau_b200 as kz
    return kz


def rec(k):
    q = o.g1_mul(o.G1_GEN, k % R)
    return o.g1_mont_record(0, 1, True) if q is None else o.g1_mont_record(q[0], q[1], False)


def powers_of(ctx, tau, n):
    return ctx.convert(1, ZU, ctx.generate(1, ZU, 1, tau, 0, n), ML, 0).reshape(n, 104)


def g2_powers(ctx, tau, first, n):
    return ctx.convert(2, ZU, ctx.generate(2, ZU, 1, tau, first, n), ML, 0).reshape(n, 200)


@pytest.fixture(scope="module")
def setup16(ctx):
    """2^16 + 8 G1 powers of a known tau, as an array and resident."""
    kz = _kz()
    tau = o.derive_scalars(0xC05E)[0]
    n = (1 << 16) + 8
    pw = kz.Powers(powers_of_g=powers_of(ctx, tau, n), powers_of_gamma_g=powers_of(ctx, tau, 1))
    return tau, pw, pw.to_device(ctx)


def _proof_scalar(p, k, h, tau):
    q, _ = divide(p, k, pow(h, k, R))
    return evaluate(q, tau)


@pytest.mark.gpu
def test_open_cosets_against_known_tau(ctx, setup16):
    """Each proof is [(p(tau) - r(tau)) / (tau^k - c)]G byte for byte and each value is p(h omega_k^m) (all m for
    small k, a sample otherwise), for n = 0, 1, k - 1, k, k + 1, 2^16 + 3, e = 0, 1, 5, 12, 16, shifts 1, omega_2k and
    random."""
    kz = _kz()
    tau, _, dev = setup16
    rnd = random.Random(4)
    for e in (0, 1, 5, 12, 16):
        k = 1 << e
        for n in sorted({0, 1, max(k - 1, 0), k, k + 1, (1 << 16) + 3}):
            p = [rnd.randrange(R) for _ in range(n)]
            hs = [1, root(e + 1), rnd.randrange(1, R)]
            values, proofs = kz.KZG10.open_cosets(dev, p, e, hs, ctx=ctx)
            assert proofs.shape == (3, 104) and len(values) == 3 and all(len(v) == k for v in values)
            w = root(e)
            for i, h in enumerate(hs):
                q, r = divide(p, k, pow(h, k, R))
                c = pow(h, k, R)
                want = (evaluate(p, tau) - evaluate(r, tau)) * pow((pow(tau, k, R) - c) % R, -1, R)
                assert proofs[i].tobytes() == rec(want) == rec(evaluate(q, tau)), (e, n, i)
                ms = range(k) if k * max(n, 1) <= 1 << 14 else rnd.sample(range(k), min(3, k)) + [0, k - 1]
                for mm in ms:
                    assert values[i][mm] == evaluate(p, h * pow(w, mm, R) % R), (e, n, i, mm)


@pytest.fixture(scope="module")
def vk16(ctx, setup16):
    kz = _kz()
    tau, pw, dev = setup16
    g2 = g2_powers(ctx, tau, 0, 2)
    return kz.VerifierKey(g=pw.powers_of_g[0], gamma_g=pw.powers_of_gamma_g[0], h=g2[0], beta_h=g2[1])


@pytest.mark.gpu
def test_open_cosets_k1_and_small_k_match_open_many(ctx, setup16, vk16):
    """k = 1: proof and value byte-equal to open_many(p, [h]), accepted by check_many and by check_cosets with
    beta_h as [tau]h.  e <= 6: the values equal open_many at coset_points(e, h)."""
    kz = _kz()
    tau, pw, dev = setup16
    rnd = random.Random(5)
    p = [rnd.randrange(R) for _ in range(300)]
    comm = kz.KZG10.commit(dev, p, ctx=ctx)
    hs = [1, 5, rnd.randrange(1, R)]
    values, proofs = kz.KZG10.open_cosets(dev, p, 0, hs, ctx=ctx)
    ov, op, _ = kz.KZG10.open_many(dev, p, hs, ctx=ctx)
    assert [v[0] for v in values] == ov and proofs.tobytes() == op.tobytes()
    assert kz.KZG10.check_many(vk16, [comm] * 3, hs, ov, proofs, ctx=ctx).all()
    assert kz.KZG10.check_cosets(dev.powers_of_g, vk16.h, vk16.beta_h, 0, [comm] * 3, hs, values, proofs, ctx=ctx)
    for e in range(1, 7):
        h = rnd.randrange(1, R)
        values, _ = kz.KZG10.open_cosets(dev, p, e, [h], ctx=ctx)
        assert values[0] == kz.KZG10.open_many(dev, p, kz.coset_points(e, h), ctx=ctx)[0], e


def _batch(kz, ctx, dev, p, e, m, rnd):
    comm = kz.KZG10.commit(dev, p, ctx=ctx)
    hs = [rnd.randrange(1, R) for _ in range(m)]
    values, proofs = kz.KZG10.open_cosets(dev, p, e, hs, ctx=ctx)
    return [comm] * m, hs, values, proofs


@pytest.mark.gpu
def test_check_cosets_accepts_and_rejects(ctx, setup16):
    """check_cosets accepts honest batches (m = 1, 7, 64; e = 0, 4, 12) and rejects one changed value, two swapped
    proofs, a wrong shift, a changed commitment and tau_k_h = [tau^(k +- 1)]h; the same seed gives the same verdict."""
    kz = _kz()
    tau, pw, dev = setup16
    rnd = random.Random(6)
    p = [rnd.randrange(R) for _ in range(9000)]
    for e in (0, 4, 12):
        k = 1 << e
        g2 = g2_powers(ctx, tau, k - 1, 3)  # tau^(k-1), tau^k, tau^(k+1)
        h0 = g2_powers(ctx, tau, 0, 1)[0]
        for m in (1, 7, 64):
            comms, hs, values, proofs = _batch(kz, ctx, dev, p, e, m, rnd)
            seed = bytes(rnd.randrange(256) for _ in range(32))
            assert kz.KZG10.check_cosets(dev.powers_of_g, h0, g2[1], e, comms, hs, values, proofs, seed=seed, ctx=ctx)
            assert kz.KZG10.check_cosets(pw.powers_of_g, h0, g2[1], e, comms, hs, values, proofs, ctx=ctx)
            if m != 7:
                continue
            bad_v = [list(v) for v in values]
            bad_v[3][k // 2] = (bad_v[3][k // 2] + 1) % R
            swapped = proofs.copy()
            swapped[[1, 5]] = proofs[[5, 1]]
            bad_h = list(hs)
            bad_h[6] = (bad_h[6] + 1) % R
            bad_c = [c.copy() for c in comms]
            bad_c[2] = kz.KZG10.commit(dev, p[:-1], ctx=ctx)
            cases = [(comms, hs, bad_v, proofs, g2[1]), (comms, hs, values, swapped, g2[1]),
                     (comms, bad_h, values, proofs, g2[1]), (bad_c, hs, values, proofs, g2[1]),
                     (comms, hs, values, proofs, g2[0]), (comms, hs, values, proofs, g2[2])]
            for j, (c, h, v, w, tk) in enumerate(cases):
                for _ in range(2):  # the same seed, the same verdict
                    assert not kz.KZG10.check_cosets(dev.powers_of_g, h0, tk, e, c, h, v, w, seed=seed, ctx=ctx), (e, j)
                assert not kz.KZG10.check_cosets(dev.powers_of_g, h0, tk, e, c, h, v, w, ctx=ctx), (e, j)


@pytest.mark.gpu
def test_cosets_full_size_polynomial(ctx):
    """A 2^21-coefficient polynomial over a 2^21-power setup: e = 4 and 12 with m = 2 against the known-tau proof
    and sampled values, and e = 20 opened and checked once against [tau^(2^20)]h."""
    kz = _kz()
    n = 1 << 21
    tau = o.derive_scalars(0x2C05)[0]
    dev = kz.ResidentPoints(ctx, powers_of(ctx, tau, n))
    pw = kz.Powers(powers_of_g=dev, powers_of_gamma_g=None)
    raw = np.random.default_rng(21).integers(0, 256, size=(n, 32), dtype=np.uint8)
    raw[:, 31] &= 0x3F  # < 2^254 < r
    p = [int.from_bytes(raw[i].tobytes(), "little") for i in range(n)]
    p_tau = evaluate(p, tau)
    rnd = random.Random(7)
    for e in (4, 12):
        k, w = 1 << e, root(e)
        hs = [rnd.randrange(1, R) for _ in range(2)]
        values, proofs = kz.KZG10.open_cosets(pw, raw, e, hs, ctx=ctx)
        for i, h in enumerate(hs):
            c = pow(h, k, R)
            # r(tau) from the values: r is the interpolant of the values on the coset
            kinv, hinv = pow(k, -1, R), pow(h, -1, R)
            r = [kinv * pow(hinv, j, R) * sum(v * pow(w, -j * mm % k, R) for mm, v in enumerate(values[i])) % R
                 for j in range(k)] if k <= 16 else None
            if r is not None:
                want = (p_tau - evaluate(r, tau)) * pow((pow(tau, k, R) - c) % R, -1, R)
                assert proofs[i].tobytes() == rec(want), (e, i)
            for mm in (0, 1, k - 1):
                assert values[i][mm] == evaluate(p, h * pow(w, mm, R) % R), (e, i, mm)
        comm = dev.msm(raw)
        g2 = g2_powers(ctx, tau, 0, 1)[0]
        tk = g2_powers(ctx, tau, k, 1)[0]
        assert kz.KZG10.check_cosets(dev, g2, tk, e, [comm] * 2, hs, values, proofs, ctx=ctx)
    e, k = 20, 1 << 20
    h = rnd.randrange(1, R)
    values, proofs = kz.KZG10.open_cosets(pw, raw, e, [h], ctx=ctx)
    assert values[0][5] == evaluate(p, h * pow(root(e), 5, R) % R)
    g2 = g2_powers(ctx, tau, 0, 1)[0]
    tk = g2_powers(ctx, tau, k, 1)[0]
    comm = dev.msm(raw)
    assert kz.KZG10.check_cosets(dev, g2, tk, e, [comm], [h], values, proofs, ctx=ctx)
    bad = [list(values[0])]
    bad[0][k - 1] = (bad[0][k - 1] + 1) % R
    assert not kz.KZG10.check_cosets(dev, g2, tk, e, [comm], [h], bad, proofs, ctx=ctx)


@pytest.mark.gpu
def test_cosets_argument_errors(ctx, setup16):
    """PTAU_ERR_ARG for log2_k outside [0, 20], more coefficients than powers, k above the powers for check, a shift 0
    or >= r, a coefficient or value >= r, a handle of another context and NULL outputs; the context keeps working."""
    kz = _kz()
    L = kz._ffi.lib()
    ERR = kz._ffi.ERR_ARG
    tau, pw, dev = setup16
    rnd = random.Random(8)
    n = 3000
    good = np.frombuffer(b"".join(le(rnd.randrange(R)) for _ in range(n)), dtype=np.uint8).reshape(n, 32)
    hs = np.frombuffer(le(5) + le(6), dtype=np.uint8).reshape(2, 32)
    out = np.zeros((2, 104), dtype=np.uint8)
    vals = np.zeros(2 * 16 * 32, dtype=np.uint8)
    g, c, H, P, V = dev.powers_of_g._h, good.ctypes.data, hs.ctypes.data, out.ctypes.data, vals.ctypes.data
    for e in (-1, 21):
        assert L.ptau_kzg_open_cosets(ctx._h, g, c, n, e, H, 2, P, V) == ERR
    assert L.ptau_kzg_open_cosets(ctx._h, g, c, len(pw.powers_of_g) + 1, 4, H, 2, P, V) == ERR
    for bad_h in (0, R, R + 1):
        bh = np.frombuffer(le(5) + le(bad_h), dtype=np.uint8)
        assert L.ptau_kzg_open_cosets(ctx._h, g, c, n, 4, bh.ctypes.data, 2, P, V) == ERR, bad_h
    for at in (0, n // 2, n - 1):
        bad = good.copy()
        bad[at] = np.frombuffer(le(R), dtype=np.uint8)
        assert L.ptau_kzg_open_cosets(ctx._h, g, bad.ctypes.data, n, 4, H, 2, P, V) == ERR, at
    assert L.ptau_kzg_open_cosets(ctx._h, g, c, n, 4, H, 2, None, V) == ERR
    assert L.ptau_kzg_open_cosets(ctx._h, g, c, n, 4, H, 2, P, None) == ERR
    assert L.ptau_kzg_open_cosets(ctx._h, None, c, n, 4, H, 2, P, V) == ERR
    assert L.ptau_kzg_open_cosets(ctx._h, g, c, n, 4, None, 0, None, None) == 0  # m = 0: nothing to do

    values, proofs = kz.KZG10.open_cosets(dev, good, 4, [5, 6], ctx=ctx)
    comm = dev.powers_of_g.msm(good)
    g2 = g2_powers(ctx, tau, 0, 1)[0]
    tk = g2_powers(ctx, tau, 16, 1)[0]
    v = np.frombuffer(b"".join(le(x) for row in values for x in row), dtype=np.uint8).copy()
    cm = np.ascontiguousarray(np.stack([comm, comm]))
    g2b, tkb = np.ascontiguousarray(g2), np.ascontiguousarray(tk)
    ok = np.zeros(1, dtype=np.uint8)
    args = lambda **kw: [kw.get("ctx", ctx._h), kw.get("g", g), kw.get("h", g2b.ctypes.data),
                         kw.get("tk", tkb.ctypes.data), kw.get("e", 4), kw.get("c", cm.ctypes.data),
                         kw.get("s", hs.ctypes.data), kw.get("v", v.ctypes.data), kw.get("w", proofs.ctypes.data),
                         kw.get("m", 2), kw.get("seed", None), kw.get("ok", ok.ctypes.data)]
    assert L.ptau_kzg_check_cosets(*args()) == 0 and ok[0] == 1
    for kw in ({"e": -1}, {"e": 21}, {"ok": None}, {"h": None}, {"tk": None}, {"c": None}, {"v": None}, {"w": None},
               {"s": None}, {"g": None}):
        assert L.ptau_kzg_check_cosets(*args(**kw)) == ERR, kw
    small = kz.ResidentPoints(ctx, pw.powers_of_g[:8])
    assert L.ptau_kzg_check_cosets(*args(g=small._h)) == ERR  # k = 16 > 8 resident powers
    for bad_h in (0, R):
        bh = np.frombuffer(le(5) + le(bad_h), dtype=np.uint8)
        assert L.ptau_kzg_check_cosets(*args(s=bh.ctypes.data)) == ERR, bad_h
    bv = v.copy()
    bv[32 * 17:32 * 18] = np.frombuffer(le(R), dtype=np.uint8)
    assert L.ptau_kzg_check_cosets(*args(v=bv.ctypes.data)) == ERR
    with kz.Context(1) as other:
        foreign = kz.ResidentPoints(other, pw.powers_of_g[:n])
        assert L.ptau_kzg_open_cosets(ctx._h, foreign._h, c, n, 4, H, 2, P, V) == ERR
        assert L.ptau_kzg_check_cosets(*args(g=foreign._h)) == ERR
        del foreign
    # still working
    assert kz.KZG10.open_cosets(dev, good, 4, [5, 6], ctx=ctx)[1].tobytes() == proofs.tobytes()
    assert kz.KZG10.check_cosets(dev.powers_of_g, g2, tk, 4, [comm] * 2, [5, 6], values, proofs, ctx=ctx)


@pytest.mark.gpu
def test_open_cosets_two_gpus():
    """A 2-GPU context splits the cosets in two contiguous ranges: the same values and proofs as one GPU."""
    kz = _kz()
    if kz._ffi.lib().ptau_device_count() < 2:
        pytest.skip("single-GPU box")
    tau = o.derive_scalars(0x2C06)[0]
    rnd = random.Random(9)
    with kz.Context(1) as c1, kz.Context(2) as c2:
        pw = kz.Powers(powers_of_g=powers_of(c1, tau, 5000), powers_of_gamma_g=powers_of(c1, tau, 1))
        d1, d2 = pw.to_device(c1), pw.to_device(c2)
        p = [rnd.randrange(R) for _ in range(4999)]
        for e, m in ((0, 2), (4, 3), (8, 7)):
            hs = [rnd.randrange(1, R) for _ in range(m)]
            a = kz.KZG10.open_cosets(d1, p, e, hs, ctx=c1)
            b = kz.KZG10.open_cosets(d2, p, e, hs, ctx=c2)
            assert a[0] == b[0] and a[1].tobytes() == b[1].tobytes(), (e, m)
            assert c2.timing()["n_gpus"] == 2
