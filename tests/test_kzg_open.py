"""KZG10::open on the GPU (ptau_kzg_open, KZG10.open_many): the openings against the host quotient committed by the
existing MSM, against a known tau, and against KZG10.check_many on the GPU.  The division scan they run is the k = 1
case of the coset openings' and is tested on the host build in test_kzg_cosets.py."""
import random

import numpy as np
import pytest

import ptau_oracle as o

R = o.R_ORDER
ZU, ML = 1, 4


def le(v: int) -> bytes:
    return int(v).to_bytes(32, "little")


def synthetic_division(coeffs, z):
    n = len(coeffs)
    q = [0] * max(n - 1, 0)
    carry = 0
    for i in range(n - 1, 0, -1):
        carry = (coeffs[i] + carry * z) % R
        q[i - 1] = carry
    return ((coeffs[0] if n else 0) + carry * z) % R, q


def evaluate(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + c) % R
    return acc


def _kz():
    import kzg_setup_powersoftau_b200 as kz
    return kz


def rec(k):
    q = o.g1_mul(o.G1_GEN, k % R)
    return o.g1_mont_record(0, 1, True) if q is None else o.g1_mont_record(q[0], q[1], False)


def powers_of(ctx, scale, tau, n):
    return ctx.convert(1, ZU, ctx.generate(1, ZU, scale, tau, 0, n), ML, 0).reshape(n, 104)


@pytest.fixture(scope="module")
def setup16(ctx):
    """2^16 + 8 powers of a known tau (G1 and gamma), as arrays and resident on the context's GPU."""
    kz = _kz()
    tau, alpha, _ = o.derive_scalars(0x0BE7)
    n = (1 << 16) + 8
    pw = kz.Powers(powers_of_g=powers_of(ctx, 1, tau, n), powers_of_gamma_g=powers_of(ctx, alpha, tau, 64))
    return tau, alpha, pw, pw.to_device(ctx)


def _old_open(kz, ctx, pw, coeffs, z, blinding=None):
    """The previous KZG10.open: host quotient (KZG10._quotient) committed by the MSM (KZG10._msm)."""
    value, q = kz.KZG10._quotient([int(c) % R for c in coeffs], int(z) % R)
    pairs = [(pw.powers_of_g, q)]
    random_v = None
    if blinding:
        random_v, rq = kz.KZG10._quotient([int(c) % R for c in blinding], int(z) % R)
        pairs.append((pw.powers_of_gamma_g, rq))
    return value, kz.KZG10._msm(ctx, pairs), random_v


@pytest.mark.gpu
def test_open_parity_across_sizes(ctx, setup16):
    """Each proof equals ptau_kzg_commit of the host quotient byte for byte and [(p(tau) - v) / (tau - z)]G, and each
    value equals p(z), for n from 0 to 2^16 + 3 around the chunk (32) and the block of chunks (32 x 1024)."""
    kz = _kz()
    tau, _, pw, dev = setup16
    rnd = random.Random(4)
    for n in (0, 1, 2, 31, 32, 33, 1023, 1024, 1025, 32767, 32768, 32769, 65536 + 3):
        p = [rnd.randrange(R) for _ in range(n)]
        z = rnd.randrange(R)
        values, proofs, rvs = kz.KZG10.open_many(dev, p, [z], ctx=ctx)
        assert rvs is None and proofs.shape == (1, 104)
        v, q = kz.KZG10._quotient(p, z)
        assert values == [v] and v == evaluate(p, z), n
        assert proofs[0].tobytes() == kz.KZG10.commit(pw, q, ctx=ctx).tobytes(), n
        assert proofs[0].tobytes() == rec((evaluate(p, tau) - v) * pow(tau - z, -1, R)), n


@pytest.mark.gpu
def test_open_full_size_polynomial(ctx):
    """A 2^21-coefficient polynomial over a 2^21-power setup, opened at 3 points: every proof equals the resident MSM
    of the host quotient (ptau_kzg_quotient), every value the host value, one proof the known-tau witness."""
    kz = _kz()
    L = kz._ffi.lib()
    n = 1 << 21
    tau = o.derive_scalars(0x21)[0]
    dev = kz.Powers(powers_of_g=powers_of(ctx, 1, tau, n), powers_of_gamma_g=powers_of(ctx, 1, tau, 1)).to_device(ctx)
    raw = np.random.default_rng(21).integers(0, 256, size=(n, 32), dtype=np.uint8)
    raw[:, 31] &= 0x3F  # < 2^254 < r
    zs = [0, 5, R - 7]
    values, proofs, _ = kz.KZG10.open_many(dev, raw, zs, ctx=ctx)
    for j, z in enumerate(zs):
        q = np.zeros((n - 1) * 32, dtype=np.uint8)
        v = np.zeros(32, dtype=np.uint8)
        assert L.ptau_kzg_quotient(raw.ctypes.data, n, le(z), q.ctypes.data, v.ctypes.data) == 0
        assert values[j] == int.from_bytes(v.tobytes(), "little"), z
        assert proofs[j].tobytes() == dev.powers_of_g.msm(q.reshape(-1, 32)).tobytes(), z
    p = [int.from_bytes(b, "little") for b in (raw[i].tobytes() for i in range(n))]
    assert values[1] == evaluate(p, 5)
    assert proofs[1].tobytes() == rec((evaluate(p, tau) - values[1]) * pow(tau - 5, -1, R))


@pytest.mark.gpu
def test_open_hiding(ctx, setup16):
    """With blinding: random_v = b(z), and the proof equals the single MSM over the concatenated quotients (the
    non-resident commit path), with resident and plain powers, including empty quotients (n, n_b = 0 or 1)."""
    kz = _kz()
    _, _, pw, dev = setup16
    rnd = random.Random(5)
    for n, n_b in ((0, 1), (1, 1), (1, 2), (5, 1), (100, 2), (3000, 40), (40, 64)):
        p = [rnd.randrange(R) for _ in range(n)]
        b = [rnd.randrange(R) for _ in range(n_b)]
        z = rnd.randrange(R)
        v, q = synthetic_division(p, z)
        rv, bq = synthetic_division(b, z)
        want = kz.KZG10._msm(ctx, [(pw.powers_of_g, q), (pw.powers_of_gamma_g, bq)]).tobytes()
        for powers in (dev, pw):
            values, proofs, rvs = kz.KZG10.open_many(powers, p, [z], blinding=b, ctx=ctx)
            assert values == [v] and rvs == [rv] and proofs[0].tobytes() == want, (n, n_b)


@pytest.mark.gpu
def test_open_many_points(ctx, setup16):
    """k = 1, 7, 64 points (repeated points, z = 0) equal k single opens; check_many accepts every opening and rejects
    each one after one tampered byte of its proof or a changed value."""
    kz = _kz()
    tau, alpha, pw, dev = setup16
    g2 = ctx.convert(2, ZU, ctx.generate(2, ZU, 1, tau, 0, 2), ML, 0).reshape(2, 200)
    vk = kz.VerifierKey(g=pw.powers_of_g[0], gamma_g=pw.powers_of_gamma_g[0], h=g2[0], beta_h=g2[1])
    rnd = random.Random(6)
    p = [rnd.randrange(R) for _ in range(777)]
    b = [rnd.randrange(R) for _ in range(3)]
    for blinding in (None, b):
        comm = kz.KZG10.commit(dev, p, blinding=blinding, ctx=ctx)
        for k in (1, 7, 64):
            zs = [rnd.randrange(R) for _ in range(k)]
            if k > 1:
                zs[1] = 0
                zs[-1] = zs[0]
            values, proofs, rvs = kz.KZG10.open_many(dev, p, zs, blinding=blinding, ctx=ctx)
            assert proofs.shape == (k, 104) and len(values) == k and (rvs is None) == (blinding is None)
            for j, z in enumerate(zs):
                v1, w1, r1 = kz.KZG10.open(dev, p, z, blinding=blinding, ctx=ctx)
                assert (values[j], proofs[j].tobytes(), None if rvs is None else rvs[j]) == (v1, w1.tobytes(), r1), (k, j)
            assert kz.KZG10.check_many(vk, [comm] * k, zs, values, proofs, rvs, ctx=ctx).all()
            for j in range(k):
                bad_proofs = proofs.copy()
                bad_proofs[j, 7] ^= 0x10
                bad_values = list(values)
                bad_values[j] = (bad_values[j] + 1) % R
                for pr, vs in ((bad_proofs, values), (proofs, bad_values)):
                    ok = kz.KZG10.check_many(vk, [comm] * k, zs, vs, pr, rvs, ctx=ctx)
                    assert not ok[j] and ok.sum() == k - 1, (k, j)


@pytest.mark.gpu
def test_open_matches_previous_path(ctx, setup16):
    """KZG10.open returns the same (value, proof, random_v) as the previous host-quotient path, with resident and
    plain powers, with and without blinding; the only change is ark's degree rule."""
    kz = _kz()
    _, _, pw, dev = setup16
    rnd = random.Random(7)
    for n in (0, 1, 2, 3, 300, 5000):
        p = [rnd.randrange(2 * R) for _ in range(n)]  # ints are taken mod r, as before
        for blinding in (None, [], [rnd.randrange(R) for _ in range(2)]):
            z = rnd.randrange(R)
            want = _old_open(kz, ctx, pw, p, z, blinding)
            for powers in (pw, dev):
                v, w, rv = kz.KZG10.open(powers, p, z, blinding=blinding, ctx=ctx)
                assert (v, w.tobytes(), rv) == (want[0], want[1].tobytes(), want[2]), (n, blinding)
    small = kz.Powers(powers_of_g=pw.powers_of_g[:10], powers_of_gamma_g=pw.powers_of_gamma_g[:2])
    assert kz.KZG10.open(small, list(range(10)), 3, ctx=ctx)[0] == evaluate(list(range(10)), 3)
    with pytest.raises(kz.PtauError) as e:
        kz.KZG10.open(small, list(range(11)), 3, ctx=ctx)  # len(powers) + 1 coefficients: TooManyCoefficients
    assert e.value.code == kz._ffi.ERR_ARG
    with pytest.raises(kz.PtauError):
        kz.KZG10.open(small, [1], 3, blinding=[1, 2, 3], ctx=ctx)


@pytest.mark.gpu
def test_open_argument_errors(ctx, setup16):
    """PTAU_ERR_ARG for a non-canonical coefficient (first, middle, last, in the blinding), a non-canonical point,
    too many coefficients for the powers or gamma powers, missing gamma powers with blinding, a powers handle of
    another context and NULL outputs; the context keeps working afterwards."""
    kz = _kz()
    L = kz._ffi.lib()
    ERR = kz._ffi.ERR_ARG
    _, _, pw, dev = setup16
    rnd = random.Random(8)
    n = 3000
    good = np.frombuffer(b"".join(le(rnd.randrange(R)) for _ in range(n)), dtype=np.uint8).reshape(n, 32)
    bl = np.frombuffer(b"".join(le(rnd.randrange(R)) for _ in range(3)), dtype=np.uint8).reshape(3, 32)
    for at in (0, n // 2, n - 1):
        bad = good.copy()
        bad[at] = np.frombuffer(le(R), dtype=np.uint8)
        with pytest.raises(kz.PtauError) as e:
            kz.KZG10.open_many(dev, bad, [5, 6], ctx=ctx)
        assert e.value.code == ERR, at
    badb = bl.copy()
    badb[1] = np.frombuffer(le(R + 3), dtype=np.uint8)
    with pytest.raises(kz.PtauError) as e:
        kz.KZG10.open_many(dev, good, [5], blinding=badb, ctx=ctx)
    assert e.value.code == ERR
    zbad = np.frombuffer(le(5) + le(R), dtype=np.uint8).reshape(2, 32)
    with pytest.raises(kz.PtauError) as e:
        kz.KZG10.open_many(dev, good, zbad, ctx=ctx)
    assert e.value.code == ERR
    with pytest.raises(kz.PtauError) as e:
        kz.KZG10.open_many(dev, [1] * (len(pw.powers_of_g) + 1), [5], ctx=ctx)
    assert e.value.code == ERR
    with pytest.raises(kz.PtauError) as e:
        kz.KZG10.open_many(dev, [1], [5], blinding=[1] * (len(pw.powers_of_gamma_g) + 1), ctx=ctx)
    assert e.value.code == ERR

    out = np.zeros((2, 104), dtype=np.uint8)
    vals = np.zeros(64, dtype=np.uint8)
    rvs = np.zeros(64, dtype=np.uint8)
    z = np.frombuffer(le(5) + le(6), dtype=np.uint8)
    P, V, RV = out.ctypes.data, vals.ctypes.data, rvs.ctypes.data
    g, gg, c, b = dev.powers_of_g._h, dev.powers_of_gamma_g._h, good.ctypes.data, bl.ctypes.data
    assert L.ptau_kzg_open(ctx._h, g, None, c, n, b, 3, z.ctypes.data, 2, P, V, RV) == ERR  # gamma powers missing
    assert L.ptau_kzg_open(ctx._h, g, gg, c, n, b, 3, z.ctypes.data, 2, None, V, RV) == ERR
    assert L.ptau_kzg_open(ctx._h, g, gg, c, n, b, 3, z.ctypes.data, 2, P, None, RV) == ERR
    assert L.ptau_kzg_open(ctx._h, g, gg, c, n, b, 3, z.ctypes.data, 2, P, V, None) == ERR
    assert L.ptau_kzg_open(ctx._h, g, gg, c, n, None, 0, z.ctypes.data, 2, P, V, RV) == ERR  # random_v without blinding
    assert L.ptau_kzg_open(ctx._h, None, gg, c, n, None, 0, z.ctypes.data, 2, P, V, None) == ERR
    assert L.ptau_kzg_open(ctx._h, g, gg, c, n, b, 3, None, 0, None, None, None) == 0  # k = 0: nothing to do
    with kz.Context(1) as other:
        foreign = kz.ResidentPoints(other, pw.powers_of_g[:n])
        assert L.ptau_kzg_open(ctx._h, foreign._h, None, c, n, None, 0, z.ctypes.data, 2, P, V, None) == ERR
        assert L.ptau_kzg_open(ctx._h, g, foreign._h, c, n, b, 3, z.ctypes.data, 2, P, V, RV) == ERR
        del foreign
    # still working: the same opening as before the errors
    values, proofs, _ = kz.KZG10.open_many(dev, good, [5, 6], ctx=ctx)
    p = [int.from_bytes(good[i].tobytes(), "little") for i in range(n)]
    for j, zz in enumerate((5, 6)):
        v, q = synthetic_division(p, zz)
        assert values[j] == v and proofs[j].tobytes() == kz.KZG10.commit(pw, q, ctx=ctx).tobytes()


@pytest.mark.gpu
def test_open_two_gpus():
    """A 2-GPU context splits the points in two contiguous ranges, each opened against its own resident copy: the
    same values, proofs and random values as one GPU, with k crossing the split."""
    kz = _kz()
    if kz._ffi.lib().ptau_device_count() < 2:
        pytest.skip("single-GPU box")
    tau, alpha, _ = o.derive_scalars(0x2C)
    rnd = random.Random(9)
    with kz.Context(1) as c1, kz.Context(2) as c2:
        pw = kz.Powers(powers_of_g=powers_of(c1, 1, tau, 5000), powers_of_gamma_g=powers_of(c1, alpha, tau, 8))
        d1, d2 = pw.to_device(c1), pw.to_device(c2)
        p = [rnd.randrange(R) for _ in range(4999)]
        b = [rnd.randrange(R) for _ in range(4)]
        for k in (1, 2, 7):
            zs = [rnd.randrange(R) for _ in range(k)]
            for blinding in (None, b):
                a = kz.KZG10.open_many(d1, p, zs, blinding=blinding, ctx=c1)
                m = kz.KZG10.open_many(d2, p, zs, blinding=blinding, ctx=c2)
                assert a[0] == m[0] and a[2] == m[2] and a[1].tobytes() == m[1].tobytes(), (k, blinding is None)
                assert c2.timing()["n_gpus"] == 2
        assert kz.KZG10.open_many(pw, p, zs, ctx=c2)[1].tobytes() == kz.KZG10.open_many(d1, p, zs, ctx=c1)[1].tobytes()
