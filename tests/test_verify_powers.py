"""ptau_verify_powers and ptau_msm_g2: do the points of a response / kzg_setup hold powers of ONE tau?

CPU tests run the product's per-item code (host build, tests/host_emul) against the oracle and hashlib; GPU tests
build setups with the GPU generator and a known tau and check acceptance, the combinations byte for byte, and that
each kind of corruption is caught by the expected relation."""
import ctypes
import hashlib
import os
import random

import numpy as np
import pytest

import ptau_oracle as o

R = o.R_ORDER
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def hostemul_verify():
    """Host build of the G2 MSM item code and the coefficient code (tests/host_emul/hostemul_verify.cpp)."""
    d = os.path.join(ROOT, "tests", "host_emul")
    so = os.path.join(d, "libptau_hostemul_verify.so")
    csrc = os.path.join(ROOT, "kzg_setup_powersoftau_b200", "csrc")
    deps = [os.path.join(d, "hostemul_verify.cpp")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                        if f.endswith((".cuh", ".inc", ".h"))]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        import subprocess

        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", so,
                               os.path.join(d, "hostemul_verify.cpp")])
    return ctypes.CDLL(so)


def rho(seed: bytes, k: int, i: int) -> int:
    d = hashlib.blake2b(bytes([k]) + i.to_bytes(8, "little"), key=seed, digest_size=16).digest()
    return int.from_bytes(d, "little") & (2**127 - 1)


def g1rec(q):
    return o.g1_mont_record(0, 1, True) if q is None else o.g1_mont_record(q[0], q[1], False)


def g2rec(q):
    return o.g2_mont_record((0, 0), (1, 0), True) if q is None else o.g2_mont_record(q[0], q[1], False)


# ---------------------------------------------------------------------------------------------- CPU
def test_limb_msm_g2_code_vs_known_tau(hostemul_verify):
    """The G2 bucket MSM's per-item code (csrc/msm_g2.cuh) run serially on the host: sum c_i [tau^i]H ==
    [sum c_i tau^i]H at sizes of several window widths, plus repeated points, P + (-P), zero scalars, all scalars
    equal and infinity records."""
    tau = 0xABCDEF123
    rnd = random.Random(21)

    def msm(points, scalars):
        out = ctypes.create_string_buffer(200)
        hostemul_verify.hostemul_msm_g2(b"".join(points), b"".join(int(s).to_bytes(32, "little") for s in scalars),
                                 ctypes.c_size_t(len(scalars)), out)
        return out.raw

    n = 140  # c = 4
    pts, q, tp = [], o.G2_GEN, [1]
    for _ in range(n):
        pts.append(g2rec(q))
        q = o.g2_mul(q, tau)
        tp.append(tp[-1] * tau % R)

    def want(k):
        return g2rec(o.g2_mul(o.G2_GEN, k % R) if k % R else None)

    for m in (1, 7, 33, n):  # c = 3, 3, 3, 4
        sc = [rnd.randrange(R) for _ in range(m)]
        assert msm(pts[:m], sc) == want(sum(c * t for c, t in zip(sc, tp))), m
    assert msm(pts[:40], [R - 1] * 40) == want(-sum(tp[:40]))
    assert msm(pts[:40], [0x1234567] * 40) == want(0x1234567 * sum(tp[:40]))          # all equal: one hot bucket
    assert msm(pts[:30], [0] * 30) == want(0)
    assert msm([pts[3]] * 40, [7] * 40) == want(280 * tp[3])                           # P + P inside a bucket
    assert msm([pts[3]] * 40, [9, R - 9] * 20) == want(0)                               # P + (-P)
    holes = [p if i % 3 else p[:192] + b"\x01" + p[193:] for i, p in enumerate(pts[:60])]
    sc = [rnd.randrange(R) for _ in range(60)]
    assert msm(holes, sc) == want(sum(c * t for i, (c, t) in enumerate(zip(sc, tp)) if i % 3))


def test_ratio_coefficients_match_hashlib(hostemul_verify):
    """The product's coefficient code (blake2b.h: one compression from the keyed chaining value) equals the keyed
    BLAKE2b formula, for several relations, across the 2^32 boundary of the index, for several seeds."""
    for s in range(3):
        seed = hashlib.sha256(b"seed%d" % s).digest()
        for k in (1, 2, 3, 4):
            for first in (0, (1 << 32) - 3, (1 << 56) - 1):
                out = ctypes.create_string_buffer(32 * 6)
                hostemul_verify.hostemul_ratio_coeffs(seed, ctypes.c_uint32(k), ctypes.c_uint64(first), ctypes.c_size_t(6), out)
                got = [int.from_bytes(out.raw[32 * j:32 * j + 32], "little") for j in range(6)]
                assert got == [rho(seed, k, first + j) for j in range(6)], (s, k, first)


def test_blake2b_digest_unchanged_by_the_shared_compression(hostemul_verify):
    """The streaming unkeyed BLAKE2b-512 (the file digest) still matches hashlib around the block boundaries."""
    rnd = random.Random(5)
    for n in (0, 1, 3, 127, 128, 129, 255, 256, 257, 1000, 4096 + 17):
        data = bytes(rnd.randrange(256) for _ in range(n))
        out = ctypes.create_string_buffer(129)
        hostemul_verify.hostemul_blake2b_hex(data, ctypes.c_size_t(n), out)
        assert out.value.decode() == hashlib.blake2b(data).hexdigest(), n


# ---------------------------------------------------------------------------------------------- GPU
ZC, ZU, AU, ML = 2, 1, 3, 4


def _kz():
    import kzg_setup_powersoftau_b200 as kz
    return kz


def response(ctx, n, tau, alpha, beta, scale=1, tau_g2=None, alpha_tau=None, beta_g2=None):
    """Synthetic compressed response: every section from the GPU generator with a known tau."""
    g = lambda grp, s0, t, cnt: ctx.generate(grp, ZC, s0 * scale % R, t, 0, cnt)
    body = np.concatenate([g(1, 1, tau, 2 * n - 1), g(2, 1, tau_g2 or tau, n), g(1, alpha, alpha_tau or tau, n),
                           g(1, beta, tau, n), g(2, beta_g2 or beta, tau, 1)])
    return np.concatenate([np.frombuffer(b"h" * 64, dtype=np.uint8), body, np.zeros(o.PUBKEY_SIZE, dtype=np.uint8)])


def setup(ctx, kind, resp, n):
    kz = _kz()
    return ctx.preprocess(kz.VARIANT_KGZ if kind == kz.POWERS_KGZ else kz.VARIANT_FASTKGZ, resp, n)


def rel_of(ctx, kind, data, n, seed=b"\x07" * 32):
    kz = _kz()
    with pytest.raises(kz.PtauError) as e:
        ctx.verify_powers(kind, data, n, seed=seed)
    assert e.value.code == kz.BAD_NOT_POWERS
    return e.value.relation


def put_g1(data, offset, k, fmt):
    """Replaces the G1 point at byte `offset` by [k]G (a valid subgroup point)."""
    q = o.g1_mul(o.G1_GEN, k % R)
    enc = o.zcash_g1_compressed_encode(q) if fmt == ZC else o.ark_g1_serialize_uncompressed(q)
    out = np.array(data, copy=True)
    out[offset:offset + len(enc)] = np.frombuffer(enc, dtype=np.uint8)
    return out


def put_g2(data, offset, k, fmt):
    q = o.g2_mul(o.G2_GEN, k % R)
    enc = o.zcash_g2_compressed_encode(q) if fmt == ZC else o.ark_g2_serialize_uncompressed(q)
    out = np.array(data, copy=True)
    out[offset:offset + len(enc)] = np.frombuffer(enc, dtype=np.uint8)
    return out


def expected_combos(kind, n, tau, alpha, beta, seed):
    kz = _kz()
    want = np.zeros((8, 200), dtype=np.uint8)
    secs = {kz.POWERS_RESPONSE: [(1, 2 * n - 1, 1, 1), (2, n, 1, 2), (3, n, alpha, 1), (4, n, beta, 1)],
            kz.POWERS_KGZ: [(1, 2 * n - 1, 1, 1), (3, n, alpha, 1)],
            kz.POWERS_FASTKGZ: [(1, 2 * n - 1, 1, 1), (2, n, 1, 2), (3, n, alpha, 1)]}[kind]
    for k, L, s0, grp in secs:
        a = b = 0
        t = s0
        for i in range(L - 1):
            r = rho(seed, k, i)
            a += r * t
            t = t * tau % R
            b += r * t
        for slot, v in ((2 * k - 2, a % R), (2 * k - 1, b % R)):
            rec = g1rec(o.g1_mul(o.G1_GEN, v)) if grp == 1 else g2rec(o.g2_mul(o.G2_GEN, v))
            want[slot, :len(rec)] = np.frombuffer(rec, dtype=np.uint8)
    return want


@pytest.mark.gpu
def test_honest_inputs_pass_and_combos_match_oracle(ctx):
    """Response, kgz and fastkgz at n = 2^10 and 2^16 from a known tau are accepted, and the combinations A_k, B_k
    equal the oracle's [sum rho_{k,i} s_i] records: this pins rho, the MSMs, the slab overlap and the summing."""
    kz = _kz()
    tau, alpha, beta = o.derive_scalars(0x7E51)
    seed = hashlib.sha256(b"honest").digest()
    for lg in (10, 16):
        n = 1 << lg
        resp = response(ctx, n, tau, alpha, beta)
        for kind in (kz.POWERS_RESPONSE, kz.POWERS_KGZ, kz.POWERS_FASTKGZ):
            data = resp if kind == kz.POWERS_RESPONSE else setup(ctx, kind, resp, n)
            got = ctx.verify_powers(kind, data, n, seed=seed, combos=True)
            assert (got == expected_combos(kind, n, tau, alpha, beta, seed)).all(), (lg, kind)
        assert ctx.verify_powers(kz.POWERS_RESPONSE, resp, n) is None  # random seed


@pytest.mark.gpu
def test_each_corruption_is_caught_by_its_relation(ctx):
    kz = _kz()
    n = 1 << 10
    tau, alpha, beta = o.derive_scalars(0x7E52)
    t2 = (tau * 3 + 1) % R
    resp = response(ctx, n, tau, alpha, beta)
    P = kz.POWERS_RESPONSE
    # two tau powers swapped
    sw = np.array(resp, copy=True)
    a, b = 64 + 5 * 48, 64 + 6 * 48
    sw[a:a + 48], sw[b:b + 48] = resp[b:b + 48], resp[a:a + 48]
    assert rel_of(ctx, P, sw, n) == kz.REL_TAU_G1
    # alpha powers made with another tau
    assert rel_of(ctx, P, response(ctx, n, tau, alpha, beta, alpha_tau=t2), n) == kz.REL_ALPHA_G1
    assert rel_of(ctx, kz.POWERS_KGZ, setup(ctx, kz.POWERS_KGZ, response(ctx, n, tau, alpha, beta, alpha_tau=t2), n),
                  n) == kz.REL_ALPHA_G1
    # beta_g2 != [beta]H
    assert rel_of(ctx, P, response(ctx, n, tau, alpha, beta, beta_g2=beta + 1), n) == kz.REL_BETA_G2
    # one beta power replaced
    off = 64 + (2 * n - 1) * 48 + n * 96 + n * 48 + 7 * 48
    assert rel_of(ctx, P, put_g1(resp, off, beta * pow(tau, 7, R) + 1, ZC), n) == kz.REL_BETA_G1
    # the G2 powers of a fastkgz with another tau (h and beta_h = powers_of_h[0..1] kept)
    fast = setup(ctx, kz.POWERS_FASTKGZ, resp, n)
    g2_off = (3 * n - 1) * 96 + 2 * 192
    other = ctx.convert(2, ZU, ctx.generate(2, ZU, 1, t2, 0, n), AU, 0).reshape(n, 192)
    bad = np.array(fast, copy=True)
    bad[g2_off + 2 * 192:g2_off + n * 192] = other[2:].reshape(-1)
    assert rel_of(ctx, kz.POWERS_FASTKGZ, bad, n) == kz.REL_TAU_G2
    # fastkgz: beta_h != powers_of_h[1]
    assert rel_of(ctx, kz.POWERS_FASTKGZ, put_g2(fast, (3 * n - 1) * 96 + 192, tau + 1, AU), n) == kz.REL_KEY
    # kgz: beta_h = [tau']H breaks every G1 ratio; gamma_g != powers_of_gamma_g[0]
    kgz = setup(ctx, kz.POWERS_KGZ, resp, n)
    tail = (3 * n + 1) * 96
    assert rel_of(ctx, kz.POWERS_KGZ, put_g2(kgz, tail + 192, t2, AU), n) == kz.REL_TAU_G1
    assert rel_of(ctx, kz.POWERS_KGZ, put_g1(kgz, (3 * n) * 96, alpha + 1, AU), n) == kz.REL_KEY
    assert rel_of(ctx, kz.POWERS_KGZ, put_g1(kgz, (3 * n - 1) * 96, 2, AU), n) == kz.REL_KEY
    # the whole setup scaled by 5: every ratio holds, only the generators are wrong
    s5 = response(ctx, n, tau, alpha, beta, scale=5)
    for kind in (P, kz.POWERS_KGZ, kz.POWERS_FASTKGZ):
        data = s5 if kind == P else setup(ctx, kind, s5, n)
        assert rel_of(ctx, kind, data, n) == kz.REL_GENERATORS, kind


@pytest.mark.gpu
def test_replaced_power_at_chunk_and_slab_boundaries():
    """A replaced tau power at index 1, at the section's last point, and around the conversion-chunk and MSM-slab
    boundaries of a context with a small chunk (chunk 1024, slab 16 x 1024 pairs) is rejected."""
    kz = _kz()
    n = 1 << 14
    L = 2 * n - 1
    chunk, slab = 1024, 16 * 1024
    tau, alpha, beta = o.derive_scalars(0x7E53)
    with kz.Context(1, chunk_points=chunk) as c:
        resp = response(c, n, tau, alpha, beta)
        kgz = setup(c, kz.POWERS_KGZ, resp, n)
        assert c.verify_powers(kz.POWERS_KGZ, kgz, n, seed=b"\x01" * 32) is None
        for i in (1, L - 1, chunk - 1, chunk, chunk + 1, slab - 1, slab, slab + 1):
            bad = put_g1(kgz, i * 96, pow(tau, i, R) + 1, AU)
            assert rel_of(c, kz.POWERS_KGZ, bad, n) == kz.REL_TAU_G1, i
        # a G2 power of the response at a chunk boundary, and alpha's last point
        g2_at = 64 + L * 48
        assert rel_of(c, kz.POWERS_RESPONSE, put_g2(resp, g2_at + chunk * 96, pow(tau, chunk, R) + 1, ZC), n) == kz.REL_TAU_G2
        a_last = 64 + L * 48 + n * 96 + (n - 1) * 48
        assert rel_of(c, kz.POWERS_RESPONSE, put_g1(resp, a_last, 3, ZC), n) == kz.REL_ALPHA_G1


@pytest.mark.gpu
def test_point_errors_take_precedence(ctx):
    """An invalid point is reported as ptau_preprocess / ptau_load_setup (STRICT) report the same bytes, and wins
    over a broken relation elsewhere in the file."""
    kz = _kz()
    n = 1 << 10
    tau, alpha, beta = o.derive_scalars(0x7E54)
    resp = response(ctx, n, tau, alpha, beta)
    sw = np.array(resp, copy=True)
    sw[64 + 5 * 48:64 + 6 * 48] = resp[64 + 6 * 48:64 + 7 * 48]  # duplicated power: TAU_G1 broken
    for off in (64 + (2 * n - 1) * 48 + n * 96 + 17 * 48,        # alpha_g1[17]
                64 + (2 * n - 1) * 48 + 3 * 96):                  # tau_g2[3]
        bad = np.array(sw, copy=True)
        bad[off + 20] ^= 0x40
        with pytest.raises(kz.PtauError) as want:
            ctx.preprocess(kz.VARIANT_FASTKGZ, bad, n, checks=kz.CHECKS_STRICT)
        with pytest.raises(kz.PtauError) as got:
            ctx.verify_powers(kz.POWERS_RESPONSE, bad, n)
        assert (got.value.code, got.value.section, got.value.index) == (want.value.code, want.value.section, want.value.index)
        assert got.value.code != kz.BAD_NOT_POWERS
    kgz = setup(ctx, kz.POWERS_KGZ, sw, n)
    for off in (40 * 96, (3 * n + 1) * 96 + 192):  # a G1 power, beta_h (G2 index in file order)
        bad = np.array(kgz, copy=True)
        bad[off + 10] ^= 0x20
        with pytest.raises(kz.PtauError) as want:
            ctx.load_setup(kz.VARIANT_KGZ, bad, n, kz.CHECKS_STRICT)
        with pytest.raises(kz.PtauError) as got:
            ctx.verify_powers(kz.POWERS_KGZ, bad, n)
        assert (got.value.code, got.value.index) == (want.value.code, want.value.index)
    with pytest.raises(kz.PtauError) as e:
        ctx.verify_powers(kz.POWERS_KGZ, kgz[:-1], n)
    assert e.value.code == kz._ffi.ERR_SIZE
    with pytest.raises(kz.PtauError) as e:
        ctx.verify_powers(kz.POWERS_RESPONSE, resp[: o.response_size(1)], 1)
    assert e.value.code == kz._ffi.ERR_ARG


@pytest.mark.gpu
def test_combos_deterministic_across_chunk_sizes_and_gpus(ctx):
    kz = _kz()
    n = 1 << 14
    tau, alpha, beta = o.derive_scalars(0x7E55)
    resp = response(ctx, n, tau, alpha, beta)
    seed = b"\x42" * 32
    ref = ctx.verify_powers(kz.POWERS_RESPONSE, resp, n, seed=seed, combos=True)
    with kz.Context(1, chunk_points=1 << 10) as c:
        assert (c.verify_powers(kz.POWERS_RESPONSE, resp, n, seed=seed, combos=True) == ref).all()
    ngpu = kz._ffi.lib().ptau_device_count()
    if ngpu < 2:
        pytest.skip("single-GPU box: multi-GPU part not run")
    with kz.Context(ngpu) as cn, kz.Context(ngpu, chunk_points=1 << 10) as cs:
        assert (cn.verify_powers(kz.POWERS_RESPONSE, resp, n, seed=seed, combos=True) == ref).all()
        assert (cs.verify_powers(kz.POWERS_RESPONSE, resp, n, seed=seed, combos=True) == ref).all()


@pytest.mark.gpu
def test_msm_g2_window_widths_and_adversarial_scalars(ctx):
    """ptau_msm_g2 against the known tau at sizes that select every window width (c = 3 .. 16), with the
    adversarial scalars of the G1 test; scalars >= r give PTAU_ERR_ARG."""
    kz = _kz()
    tau = o.derive_scalars(0xC0FFEF)[0]
    nmax = (1 << 20) + 3
    pts = ctx.convert(2, ZU, ctx.generate(2, ZU, 1, tau, 0, nmax), ML, 0).reshape(nmax, 200)
    tp = [1]
    for _ in range(nmax - 1):
        tp.append(tp[-1] * tau % R)

    def want(sc):
        k = sum(c * t for c, t in zip(sc, tp)) % R
        return g2rec(o.g2_mul(o.G2_GEN, k) if k else None)

    def msm(sc):
        return ctx.msm_g2(pts[:len(sc)], sc).tobytes()

    rnd = random.Random(78)
    widths = set()
    for n in (1, 2, 127, 200, 300, 600, 2048, 4096, 5000, 10_000, 1 << 15, 40_000, (1 << 16) + 1, (1 << 17) + 1,
              (1 << 18) + 5, nmax):
        lg = max(n - 1, 0).bit_length()
        widths.add(min(max(lg - 4, 3), 16))
        sc = [rnd.randrange(R) for _ in range(n)]
        assert msm(sc) == want(sc), n
    assert widths == set(range(3, 17))
    for n in (1000, 100_000):
        lg = (n - 1).bit_length()
        c = min(max(lg - 4, 3), 16)
        W = (256 + c - 1) // c
        a = 256 - (c - 1) * W
        tops = [(w + 1) * c - 1 if w < a else a * c + (w - a + 1) * (c - 1) - 1 for w in range(W - 1)]
        for sc in ([R - 1] * n, [0x1234567] * n, [sum(1 << b for b in tops[:-1])] * n,
                   [sum(1 << b for b in tops[:-1]) + 1] * n, [0] * (n - 1) + [5]):
            assert msm(sc) == want(sc), n
    bad = np.frombuffer(R.to_bytes(32, "little"), dtype=np.uint8).reshape(1, 32)
    with pytest.raises(kz.PtauError) as e:
        ctx.msm_g2(pts[:1], bad)
    assert e.value.code == kz._ffi.ERR_ARG


@pytest.mark.gpu
def test_full_size_fastkgz_file(ctx, tmp_path):
    """A 2^21 fastkgz setup from the generator is accepted through verify_fastkzg_setup(path) (n inferred from the
    file size); the same file with one power replaced is rejected."""
    kz = _kz()
    n = 1 << 21
    tau, alpha, beta = o.derive_scalars(0x7E56)
    fast = setup(ctx, kz.POWERS_FASTKGZ, response(ctx, n, tau, alpha, beta), n)
    path = tmp_path / "kzg_setup"
    fast.tofile(path)
    assert kz.verify_fastkzg_setup(str(path), ctx=ctx) is None
    i = 1_234_567
    put_g1(fast, i * 96, pow(tau, i, R) * 2, AU).tofile(path)
    with pytest.raises(kz.PtauError) as e:
        kz.verify_fastkzg_setup(str(path), ctx=ctx)
    assert e.value.code == kz.BAD_NOT_POWERS and e.value.relation == kz.REL_TAU_G1
