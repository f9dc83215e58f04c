"""GPU parity tests: every call goes through the C ABI (libptau_b200.so) and is
compared bit-for-bit with the oracle (Python big-int / C restatement of the
reference's algorithms), the committed golden fixtures, and -- at BASELINE.json's
full sizes -- size-independent properties."""
import json
import os
import random

import numpy as np
import pytest

import ptau_oracle as o
from conftest import GOLDEN, golden

pytestmark = pytest.mark.gpu

import kzg_setup_powersoftau_b200 as kz  # noqa: E402

SZ = {1: {1: 96, 2: 48, 3: 96, 4: 104}, 2: {1: 192, 2: 96, 3: 192, 4: 200}}
ZU, ZC, AU, ML = kz.FMT_ZCASH_UNCOMPRESSED, kz.FMT_ZCASH_COMPRESSED, kz.FMT_ARK_UNCOMPRESSED, kz.FMT_ARK_MONT_LIMBS
STRICT = kz.CHECKS_STRICT


def test_native_library_is_the_path():
    from kzg_setup_powersoftau_b200 import _ffi

    assert os.path.exists(_ffi.LIB_PATH)
    assert _ffi.lib().ptau_device_count() >= 1
    maps = open("/proc/self/maps").read()
    assert os.path.basename(_ffi.LIB_PATH) in maps  # libptau_b200.so, or the A/B build PTAU_LIB names


def test_field_ops_on_gpu_carry_stress(ctx):
    """The PTX carry chains themselves (IMAD.WIDE rows, dedicated squaring, add/sub) on limb
    patterns that force every carry path, against Python big integers."""
    import ctypes

    P = o.P
    rinv = pow(o.MONT_R, -1, P)
    rnd = random.Random(2026)
    pats = [0, 1, 2, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF, 0xFFFF0000, 0x0000FFFF, 0xAAAAAAAA, 0x55555555]
    vals = []
    for _ in range(3000):
        v = 0
        for i in range(12):
            v |= rnd.choice(pats) << (32 * i)
        vals.append((v & ((1 << 381) - 1)) % P)
    for k in range(1, 12):
        vals += [(1 << (32 * k)) - 1, 1 << (32 * k), (1 << (32 * k)) + 1, P - (1 << (32 * k)), P - (1 << (32 * k)) - 1]
    vals += [0, 1, P - 1, P - 2, o.MONT_R, (P - 1) // 2, (P + 1) // 2] + [rnd.randrange(P) for _ in range(2000)]
    vals = [v % P for v in vals]
    n = len(vals)
    a = vals
    b = [vals[(7 * i + 3) % n] for i in range(n)]
    abuf = b"".join(v.to_bytes(48, "little") for v in a)
    bbuf = b"".join(v.to_bytes(48, "little") for v in b)
    L = kz._ffi.lib()

    def run(op):
        out = ctypes.create_string_buffer(n * 48)
        assert L.ptau_selftest_fq_op(ctx._h, 0, op, abuf, bbuf, out, n) == 0
        return [int.from_bytes(out.raw[i * 48:(i + 1) * 48], "little") for i in range(n)]

    assert run(0) == [x * y * rinv % P for x, y in zip(a, b)]
    assert run(4) == [x * x * rinv % P for x in a]
    assert run(1) == [(x + y) % P for x, y in zip(a, b)]
    assert run(2) == [(x - y) % P for x, y in zip(a, b)]
    assert run(3) == [(-x) % P for x in a]
    # exponentiation chain and Fermat inverse on Montgomery-form inputs
    am = [x * o.MONT_R % P for x in a[:200]]
    abuf2 = b"".join(v.to_bytes(48, "little") for v in am)
    out = ctypes.create_string_buffer(200 * 48)
    assert L.ptau_selftest_fq_op(ctx._h, 0, 5, abuf2, abuf2, out, 200) == 0
    got = [int.from_bytes(out.raw[i * 48:(i + 1) * 48], "little") for i in range(200)]
    assert got == [pow(x, (P - 3) // 4, P) * o.MONT_R % P for x in a[:200]]
    assert L.ptau_selftest_fq_op(ctx._h, 0, 6, abuf2, abuf2, out, 200) == 0
    got = [int.from_bytes(out.raw[i * 48:(i + 1) * 48], "little") for i in range(200)]
    assert got == [(pow(x, -1, P) if x else 0) * o.MONT_R % P for x in a[:200]]


# ---- golden fixtures ----------------------------------------------------------------
@pytest.mark.parametrize("variant,name", [(kz.VARIANT_KGZ, "kgz"), (kz.VARIANT_FASTKGZ, "fastkgz")])
def test_preprocess_golden(ctx, variant, name):
    n = 8
    resp = golden("n8_powersoftau.bin")
    want = golden("n8_kzg_setup_%s.bin" % name)
    # fused path (no intermediate file)
    got = ctx.preprocess(variant, resp, n, STRICT)
    assert bytes(got) == want
    # two-stage path that also emits `powersoftau_uncompressed`
    got, unc = ctx.preprocess(variant, resp, n, STRICT, emit_uncompressed=True)
    assert bytes(got) == want and bytes(unc) == golden("n8_powersoftau_uncompressed.bin")
    # from the uncompressed file (load_powersoftau_accumulator)
    got = ctx.preprocess_uncompressed(variant, golden("n8_powersoftau_uncompressed.bin"), n, kz.CHECKS_READ)
    assert bytes(got) == want
    # wrong size -> the reference panics at preprocess-kgz.rs:83
    with pytest.raises(kz.PtauError) as e:
        ctx.preprocess(variant, resp[:-1], n)
    assert e.value.code == kz._ffi.ERR_SIZE


def test_load_golden(ctx):
    n = 8
    for checks in (kz.CHECKS_LOAD, STRICT):
        g1, g2 = ctx.load_setup(kz.VARIANT_KGZ, golden("n8_kzg_setup_kgz.bin"), n, checks)
        assert g1.tobytes() == golden("n8_load_kgz_g1.bin") and g2.tobytes() == golden("n8_load_kgz_g2.bin")
        g1, g2 = ctx.load_setup(kz.VARIANT_FASTKGZ, golden("n8_kzg_setup_fastkgz.bin"), n, checks)
        assert g1.tobytes() == golden("n8_load_fastkgz_g1.bin") and g2.tobytes() == golden("n8_load_fastkgz_g2.bin")


def test_loader_api_mirrors_reference(ctx, tmp_path):
    n = 8
    (tmp_path / "kzg_setup").write_bytes(golden("n8_kzg_setup_kgz.bin"))
    powers, vk = kz.load_kzg_setup(str(tmp_path / "kzg_setup"), ctx=ctx)
    assert powers.powers_of_g.shape == (2 * n - 1, 104) and powers.powers_of_gamma_g.shape == (n, 104)
    pg, pgg, ovk = o.load_kzg_setup(golden("n8_kzg_setup_kgz.bin"), n)
    assert powers.powers_of_g[5].tobytes() == o.g1_mont_record(*pg[5])
    assert vk.g.tobytes() == o.g1_mont_record(*ovk[0]) and vk.beta_h.tobytes() == o.g2_mont_record(*ovk[3])
    x, y, inf = kz.g1_limbs(vk.gamma_g)
    assert not inf and int.from_bytes(x.tobytes(), "little") == ovk[1][0] * o.MONT_R % o.P
    (tmp_path / "kzg_setup").write_bytes(golden("n8_kzg_setup_fastkgz.bin"))
    params, ph = kz.load_fastkzg_setup(str(tmp_path / "kzg_setup"), ctx=ctx)
    assert ph.shape == (n, 200) and params.beta_h.tobytes() == ph[1].tobytes() == params.prepared_beta_h_src.tobytes()
    assert params.neg_powers_of_h == {}
    # the returned arrays own their pinned memory: still valid after a garbage collection
    import gc

    keep = params.powers_of_g[3].copy()
    del params
    gc.collect()
    assert ph[1].tobytes() == o.g2_mont_record(*o.load_fastkzg_setup(golden("n8_kzg_setup_fastkgz.bin"), n)[5][1])
    assert keep.tobytes() == o.g1_mont_record(*pg[3])
    # validated load of the same file
    kz.load_fastkzg_setup(str(tmp_path / "kzg_setup"), ctx=ctx, checks=STRICT)
    # truncated file: the reference's unwrap() panics
    (tmp_path / "kzg_setup").write_bytes(golden("n8_kzg_setup_kgz.bin")[:-7])
    with pytest.raises(kz.PtauError):
        kz.load_kzg_setup(str(tmp_path / "kzg_setup"), ctx=ctx)


def test_binaries_file_behaviour(ctx, tmp_path):
    n = 8
    (tmp_path / "powersoftau").write_bytes(golden("n8_powersoftau.bin"))
    kz.preprocess_kgz(str(tmp_path), log2_powers=3, expected_digest=None, ctx=ctx)
    assert (tmp_path / "kzg_setup").read_bytes() == golden("n8_kzg_setup_kgz.bin")
    assert (tmp_path / "powersoftau_uncompressed").read_bytes() == golden("n8_powersoftau_uncompressed.bin")
    # create_new(true): an existing intermediate file is an error (preprocess-kgz.rs:113-118)
    with pytest.raises(FileExistsError):
        kz.preprocess_fastkgz(str(tmp_path), log2_powers=3, expected_digest=None, ctx=ctx)
    os.remove(tmp_path / "powersoftau_uncompressed")
    kz.preprocess_fastkgz(str(tmp_path), log2_powers=3, expected_digest=None, ctx=ctx)
    assert (tmp_path / "kzg_setup").read_bytes() == golden("n8_kzg_setup_fastkgz.bin")
    # digest check (preprocess-kgz.rs:33-47) with the synthetic file's own digest, then a wrong one
    dg = o.blake2b_hex(golden("n8_powersoftau.bin"))
    os.remove(tmp_path / "powersoftau_uncompressed")
    kz.preprocess_kgz(str(tmp_path), log2_powers=3, expected_digest=dg, ctx=ctx)
    os.remove(tmp_path / "powersoftau_uncompressed")
    with pytest.raises(IOError):
        kz.preprocess_kgz(str(tmp_path), log2_powers=3, ctx=ctx)  # real ceremony digest cannot match


def test_cli_binaries(tmp_path):
    """The compiled drop-in binaries (csrc/cli_main.cpp): same files in, same files out."""
    import subprocess

    from conftest import ROOT

    bindir = os.path.join(ROOT, "kzg_setup_powersoftau_b200", "bin")
    (tmp_path / "powersoftau").write_bytes(golden("n8_powersoftau.bin"))
    dg = o.blake2b_hex(golden("n8_powersoftau.bin"))
    r = subprocess.run([os.path.join(bindir, "preprocess-kgz"), "--dir", str(tmp_path), "--log2-powers", "3",
                        "--expect-digest", dg], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Done serializing. KZG parameters are stored in kzg_setup" in r.stdout
    assert (tmp_path / "kzg_setup").read_bytes() == golden("n8_kzg_setup_kgz.bin")
    assert (tmp_path / "powersoftau_uncompressed").read_bytes() == golden("n8_powersoftau_uncompressed.bin")
    # second run: the intermediate file exists -> the reference panics (create_new)
    r = subprocess.run([os.path.join(bindir, "preprocess-fastkgz"), "--dir", str(tmp_path), "--log2-powers", "3",
                        "--skip-digest"], capture_output=True, text=True)
    assert r.returncode != 0 and "unable to create `powersoftau_uncompressed`" in r.stderr
    r = subprocess.run([os.path.join(bindir, "preprocess-fastkgz"), "--dir", str(tmp_path), "--log2-powers", "3",
                        "--skip-digest", "--no-uncompressed"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "kzg_setup").read_bytes() == golden("n8_kzg_setup_fastkgz.bin")
    # default digest = the real ceremony file's: a synthetic file fails validation
    r = subprocess.run([os.path.join(bindir, "preprocess-kgz"), "--dir", str(tmp_path), "--log2-powers", "3",
                        "--no-uncompressed"], capture_output=True, text=True)
    assert r.returncode != 0 and "failed validation" in r.stderr
    # wrong size (preprocess-kgz.rs:83)
    r = subprocess.run([os.path.join(bindir, "preprocess-kgz"), "--dir", str(tmp_path), "--log2-powers", "4",
                        "--skip-digest", "--no-uncompressed"], capture_output=True, text=True)
    assert r.returncode != 0 and "something isn't right" in r.stderr
    # a corrupted point: reported with section and index, non-zero exit (the reference panics)
    bad = bytearray(golden("n8_powersoftau.bin"))
    bad[64 + 15 * 48 + 8 * 96 + 2 * 48 + 20] ^= 0x55  # alpha_tau_powers_g1[2]
    (tmp_path / "powersoftau").write_bytes(bytes(bad))
    r = subprocess.run([os.path.join(bindir, "preprocess-kgz"), "--dir", str(tmp_path), "--log2-powers", "3",
                        "--skip-digest", "--no-uncompressed"], capture_output=True, text=True)
    assert r.returncode != 0 and "point 2 of alpha_tau_powers_g1" in r.stderr


def test_file_pipeline_2pow14_multi_slab(ctx, tmp_path):
    """2^14-power response through the file pipeline (tau_g1 spans several chunks) against
    the memory-to-memory pipeline, both variants, and the C++ BLAKE2b against hashlib."""
    import ctypes

    n = 1 << 14
    tau, alpha, beta = o.derive_scalars(0xB201)
    ZCf = kz.FMT_ZCASH_COMPRESSED
    body = np.concatenate([ctx.generate(1, ZCf, 1, tau, 0, 2 * n - 1), ctx.generate(2, ZCf, 1, tau, 0, n),
                           ctx.generate(1, ZCf, alpha, tau, 0, n), ctx.generate(1, ZCf, beta, tau, 0, n),
                           ctx.generate(2, ZCf, beta, tau, 0, 1)])
    resp = o.filler_bytes(2, 64, b"hash") + body.tobytes() + o.filler_bytes(2, o.PUBKEY_SIZE, b"pubkey")
    (tmp_path / "powersoftau").write_bytes(resp)
    hexbuf = ctypes.create_string_buffer(129)
    assert kz._ffi.lib().ptau_blake2b_file(str(tmp_path / "powersoftau").encode(), hexbuf) == 0
    assert hexbuf.value.decode() == o.blake2b_hex(resp)
    want_kgz, want_unc = ctx.preprocess(kz.VARIANT_KGZ, resp, n, emit_uncompressed=True)
    kz.preprocess_kgz(str(tmp_path), log2_powers=14, expected_digest=o.blake2b_hex(resp), ctx=ctx)
    assert (tmp_path / "kzg_setup").read_bytes() == want_kgz.tobytes()
    assert (tmp_path / "powersoftau_uncompressed").read_bytes() == want_unc.tobytes()
    kz.preprocess_fastkgz(str(tmp_path), log2_powers=14, expected_digest=None, emit_uncompressed=False, ctx=ctx)
    assert (tmp_path / "kzg_setup").read_bytes() == ctx.preprocess(kz.VARIANT_FASTKGZ, resp, n).tobytes()
    params, ph = kz.load_fastkzg_setup(str(tmp_path / "kzg_setup"), ctx=ctx)  # n inferred from the size
    assert params.powers_of_g.shape == (2 * n - 1, 104) and ph.shape == (n, 200)


def test_file_pipeline_failure_is_atomic_and_ordered(ctx, tmp_path, monkeypatch):
    """A failed run publishes nothing: an older good `kzg_setup` stays byte-identical, no partial
    `powersoftau_uncompressed`, no temporary files (the reference validates in RAM before it creates `kzg_setup`,
    preprocess-kgz.rs:128-160 then :186).  Errors come in the reference's order of events: decode errors of the
    decompression pass over ALL sections (:105-110), then create_new of the intermediate file (:113-118), then the
    first bad point of the read_g1/read_g2 loops (:140-153) -- with several slabs per section."""
    monkeypatch.setenv("PTAU_SLAB_LOG2", "10")  # floor of the knob: slabs of 1024 points, 2^11-power file below
    meta = json.load(open(os.path.join(GOLDEN, "edge_cases.json")))
    off_subgroup = next(bytes.fromhex(c["rec"]) for c in meta["cases"] if c["group"] == 1 and c["in_fmt"] == 2 and c["strict"] == 5)
    undecodable = next(bytes.fromhex(c["rec"]) for c in meta["cases"] if c["group"] == 1 and c["in_fmt"] == 2 and c["strict"] == 4)
    k = 11
    n = 1 << k
    tau, alpha, beta = o.derive_scalars(0xB202)
    ZCf = kz.FMT_ZCASH_COMPRESSED
    body = np.concatenate([ctx.generate(1, ZCf, 1, tau, 0, 2 * n - 1), ctx.generate(2, ZCf, 1, tau, 0, n),
                           ctx.generate(1, ZCf, alpha, tau, 0, n), ctx.generate(1, ZCf, beta, tau, 0, n),
                           ctx.generate(2, ZCf, beta, tau, 0, 1)])
    good = o.filler_bytes(3, 64, b"hash") + body.tobytes() + o.filler_bytes(3, o.PUBKEY_SIZE, b"pubkey")
    src = tmp_path / "powersoftau"
    src.write_bytes(good)
    kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest=None, emit_uncompressed=False, ctx=ctx)
    want = (tmp_path / "kzg_setup").read_bytes()
    assert want == ctx.preprocess(kz.VARIANT_KGZ, good, n).tobytes()

    def clean_dir():
        assert sorted(p.name for p in tmp_path.iterdir()) == ["kzg_setup", "powersoftau"]
        assert (tmp_path / "kzg_setup").read_bytes() == want

    off_tau = 64 + 3000 * 48                                   # tau_powers_g1[3000]: third slab of section 0
    off_alpha = 64 + (2 * n - 1) * 48 + n * 96 + 1500 * 48     # alpha_tau_powers_g1[1500]: second slab of section 2
    bad = bytearray(good)
    bad[off_tau:off_tau + 48] = off_subgroup
    src.write_bytes(bytes(bad))
    for emit in (False, True):
        with pytest.raises(kz.PtauError) as ei:
            kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest=None, emit_uncompressed=emit, ctx=ctx)
        assert (ei.value.code, ei.value.section, ei.value.index) == (kz.BAD_NOT_IN_SUBGROUP, 0, 3000)
        clean_dir()
    # a later undecodable point wins over the earlier subgroup failure (the decompression pass runs first)
    bad[off_alpha:off_alpha + 48] = undecodable
    src.write_bytes(bytes(bad))
    for emit in (False, True):
        with pytest.raises(kz.PtauError) as ei:
            kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest=None, emit_uncompressed=emit, ctx=ctx)
        assert (ei.value.code, ei.value.section, ei.value.index) == (kz.BAD_NOT_ON_CURVE, 2, 1500)
        clean_dir()
    # ... and over create_new; create_new in turn wins over the read_g1 failure
    (tmp_path / "powersoftau_uncompressed").write_bytes(b"older")
    with pytest.raises(kz.PtauError) as ei:
        kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest=None, ctx=ctx)
    assert ei.value.code == kz.BAD_NOT_ON_CURVE
    bad[off_alpha:off_alpha + 48] = good[off_alpha:off_alpha + 48]
    src.write_bytes(bytes(bad))
    with pytest.raises(FileExistsError):
        kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest=None, ctx=ctx)
    assert (tmp_path / "powersoftau_uncompressed").read_bytes() == b"older"
    os.remove(tmp_path / "powersoftau_uncompressed")
    # a wrong digest wins over everything
    with pytest.raises(IOError):
        kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest="00" * 64, ctx=ctx)
    clean_dir()
    # the good file again, through many slabs, with the intermediate file
    src.write_bytes(good)
    kz.preprocess_kgz(str(tmp_path), log2_powers=k, expected_digest=o.blake2b_hex(good), ctx=ctx)
    assert (tmp_path / "kzg_setup").read_bytes() == want
    assert (tmp_path / "powersoftau_uncompressed").read_bytes() == ctx.preprocess(kz.VARIANT_KGZ, good, n, emit_uncompressed=True)[1].tobytes()
    assert sorted(p.name for p in tmp_path.iterdir()) == ["kzg_setup", "powersoftau", "powersoftau_uncompressed"]


def test_phase1_and_read_g(ctx, tmp_path):
    m = 4
    data = golden("n8_phase1radix2m2.bin")
    (tmp_path / "phase1radix2m2").write_bytes(data)
    ph = kz.load_phase1(2, directory=str(tmp_path), ctx=ctx)
    alpha, beta_g1, beta_g2, c1, c2, ac1, bc1 = o.load_phase1(data, m)
    assert ph.alpha.tobytes() == o.g1_mont_record(*alpha, False)
    assert ph.beta_g2.tobytes() == o.g2_mont_record(*beta_g2, False)
    assert ph.coeffs_g2.tobytes() == b"".join(o.g2_mont_record(*q, False) for q in c2)
    assert ph.beta_coeffs_g1.tobytes() == b"".join(o.g1_mont_record(*q, False) for q in bc1)
    with open(tmp_path / "phase1radix2m2", "rb") as f:
        a = kz.read_g1(f, ctx=ctx)
        b = kz.read_g1(f, ctx=ctx)
        c = kz.read_g2(f, ctx=ctx)
    assert a.tobytes() == ph.alpha.tobytes() and b.tobytes() == ph.beta_g1.tobytes() and c.tobytes() == ph.beta_g2.tobytes()
    import io

    with pytest.raises(EOFError):
        kz.read_g1(io.BytesIO(b"\x00" * 95), ctx=ctx)


# ---- edge cases ------------------------------------------------------------------------
def test_edge_cases(ctx):
    meta = json.load(open(os.path.join(GOLDEN, "edge_cases.json")))
    for cs in meta["cases"]:
        rec = bytes.fromhex(cs["rec"])
        for mode, checks in (("strict", STRICT), ("nocheck", 0), ("read", kz.CHECKS_READ)):
            if mode not in cs:
                continue
            try:
                ctx.convert(cs["group"], cs["in_fmt"], rec, AU, checks)
                st = 0
            except kz.PtauError as e:
                st = e.code
                assert e.index == 0
            assert st == cs[mode], (cs["desc"], mode, st)


def test_mont_limb_input_and_differential_fuzz(ctx, cref):
    """ARK_MONT_LIMBS input (serialize direction) round trips, and mutated / random records of
    every input format in every check mode agree with the C oracle, record by record."""
    n = 8
    kgz = golden("n8_kzg_setup_kgz.bin")
    assert ctx.convert(1, ML, golden("n8_load_kgz_g1.bin"), AU, STRICT).tobytes() == kgz[:(3 * n - 1) * 96] + kgz[-576:-384]
    assert ctx.convert(2, ML, golden("n8_load_kgz_g2.bin"), AU, STRICT).tobytes() == kgz[-384:]
    rnd = random.Random(777)
    P = o.P
    base = []
    for _ in range(4):
        q1 = o.g1_mul(o.G1_GEN, rnd.randrange(1, o.R_ORDER))
        q2 = o.g2_mul(o.G2_GEN, rnd.randrange(1, o.R_ORDER))
        base += [(1, ZU, o.zcash_g1_uncompressed_encode(q1)), (1, ZC, o.zcash_g1_compressed_encode(q1)),
                 (1, AU, o.ark_g1_serialize_uncompressed(q1)), (1, ML, o.g1_mont_record(q1[0], q1[1], False)),
                 (2, ZU, o.zcash_g2_uncompressed_encode(q2)), (2, ZC, o.zcash_g2_compressed_encode(q2)),
                 (2, AU, o.ark_g2_serialize_uncompressed(q2)), (2, ML, o.g2_mont_record(q2[0], q2[1], False))]

    def mutate(rec):
        b = bytearray(rec)
        k = rnd.randrange(4)
        if k == 0:
            b[rnd.randrange(len(b))] ^= 1 << rnd.randrange(8)
        elif k == 1:
            b[0] ^= rnd.choice([0x80, 0x40, 0x20, 0xC0, 0xE0])
        elif k == 2:
            pos = rnd.choice(range(0, len(b) - 47, 48))
            b[pos:pos + 48] = rnd.choice([P, P - 1, P + 1, 0, 1, (1 << 381) - 1, (1 << 384) - 1]).to_bytes(48, "big")
        else:
            b[48 * rnd.randrange(len(b) // 48)] ^= rnd.choice([0x80, 0x40, 0xC0])
        return bytes(b)

    n_bad = 0
    for g, f, rec in base:
        recs = [rec] + [mutate(rec) for _ in range(5)] + [bytes(rnd.randrange(256) for _ in range(len(rec)))]
        for r in recs:
            for checks in (0, kz.CHECKS_READ, STRICT):
                want, st = cref.convert(g, f, r, AU, checks)
                try:
                    got = ctx.convert(g, f, r, AU, checks).tobytes()
                    code = 0
                except kz.PtauError as e:
                    code = e.code
                assert code == st[0], (g, f, checks, r.hex())
                if code == 0:
                    assert got == want
                else:
                    n_bad += 1
    assert n_bad > 100


def test_empty_ragged_and_chunk_boundaries(cref):
    rnd = random.Random(31)
    tau = rnd.randrange(1, o.R_ORDER)
    n = 1000
    zu = cref.generate(1, 1, 1, tau, 0, n, 8)
    want = b"".join(o.read_g1_bytes(zu[i * 96:(i + 1) * 96]) for i in range(n))
    with kz.Context(1, chunk_points=96) as small:  # forces 11 chunks, ragged tail, partial blocks
        assert small.convert(1, ZU, b"", AU, STRICT).size == 0
        for cnt in (1, 2, 127, 128, 129, 255, 257, 1000):
            got = small.convert(1, ZU, zu[:cnt * 96], AU, STRICT)
            assert got.tobytes() == want[:cnt * 96], cnt
        assert small.timing()["kernel_launches"] == 11
        # lowest failing index wins, across chunks, whatever the order of completion
        bad = bytearray(zu)
        for i in (977, 403, 404, 612):
            bad[i * 96 + 95] ^= 0x01
        with pytest.raises(kz.PtauError) as e:
            small.convert(1, ZU, bytes(bad), AU, STRICT)
        assert e.value.index == 403 and e.value.code == kz.BAD_NOT_ON_CURVE
        with pytest.raises(kz.PtauError):
            small.convert(1, ZU, zu[:100], AU, STRICT)  # not a whole number of records


def test_random_batches_vs_c_oracle(ctx, cref):
    """Seeded random sections at a size the CPU oracle finishes in seconds; the oracle
    runs the reference's algorithms (r-multiplication, Algorithm 9)."""
    rnd = random.Random(77)
    tau, alpha = rnd.randrange(1, o.R_ORDER), rnd.randrange(1, o.R_ORDER)
    n1, n2 = 3000, 1200
    zc1 = cref.generate(1, 2, alpha, tau, 0, n1, 16)
    zc2 = cref.generate(2, 2, 1, tau, 0, n2, 16)
    for g, zc in ((1, zc1), (2, zc2)):
        zu_want, st = cref.convert(g, ZC, zc, ZU, 0, 16)
        assert not any(st)
        au_want, st = cref.convert(g, ZU, zu_want, AU, 4, 16)
        assert not any(st)
        ml_want, _ = cref.convert(g, AU, au_want, ML, 0, 16)
        assert ctx.convert(g, ZC, zc, ZU, kz.CHECKS_DECOMPRESS).tobytes() == zu_want
        assert ctx.convert(g, ZC, zc, AU, STRICT).tobytes() == au_want
        assert ctx.convert(g, ZU, zu_want, AU, STRICT).tobytes() == au_want
        assert ctx.convert(g, ZU, zu_want, AU, kz.CHECKS_READ).tobytes() == au_want
        assert ctx.convert(g, AU, au_want, ML, kz.CHECKS_LOAD).tobytes() == ml_want
        assert ctx.convert(g, AU, au_want, ML, STRICT).tobytes() == ml_want
        assert ctx.convert(g, ZU, zu_want, ML, STRICT).tobytes() == ml_want
        assert ctx.convert(g, AU, au_want, ZU, 0).tobytes() == zu_want


def test_configs_1_and_2_input_from_the_c_oracle_2pow16(ctx, cref):
    """BASELINE configs[1] / configs[2] at 2^16 points per group with input that does NOT come from the repository's
    GPU generator: sections built by oracle/cpu_ref.c (6 x 64-bit Montgomery, its own scalar multiplication), expected
    bytes by the same C code running the reference's algorithms (Algorithm-9 Fq2 sqrt, multiplication by r).  A field
    bug shared by the GPU generator and the GPU decompressor cannot cancel here."""
    n = 1 << 16
    th = os.cpu_count() or 1
    rnd = random.Random(0xC0FFEE)
    tau, s0 = rnd.randrange(1, o.R_ORDER), rnd.randrange(1, o.R_ORDER)
    for g in (1, 2):
        zc = cref.generate(g, ZC, s0, tau, 5, n, th)
        zu_want, st = cref.convert(g, ZC, zc, ZU, 0, th)
        assert not any(st)
        au_want, st = cref.convert(g, ZU, zu_want, AU, 4, th)
        assert not any(st)
        assert ctx.convert(g, ZC, zc, AU, STRICT).tobytes() == au_want            # configs[2]: fused compressed path
        assert ctx.convert(g, ZC, zc, ZU, kz.CHECKS_DECOMPRESS).tobytes() == zu_want
        assert ctx.convert(g, ZU, zu_want, AU, STRICT).tobytes() == au_want        # configs[1]: uncompressed path
        # and the GPU generator against the independent one, at this size
        assert ctx.generate(g, ZC, s0, tau, 5, n).tobytes() == zc


def test_config5_known_tau_spot_check_2pow24(ctx):
    """BASELINE configs[4] at 2^24 points per section, slab by slab on the device (generate -> fused compressed ->
    strict -> ark), with 64 random indices per group compared with [s tau^i]G computed by the Python big-int oracle
    (affine formulas, nothing shared with the CUDA field code), plus the boundary indices of every slab."""
    import torch

    n = 1 << 24
    slab = 1 << 22
    tau, alpha, _ = o.derive_scalars(0xB226)
    dev = torch.device("cuda", 0)
    d_in = torch.empty(slab * 96, dtype=torch.uint8, device=dev)
    d_out = torch.empty(slab * 192, dtype=torch.uint8, device=dev)
    status = torch.full((1,), -1, dtype=torch.int64, device=dev)
    rnd = random.Random(24)
    for g, s0, ro, enc, mul, gen in ((kz.G1, alpha, 96, o.ark_g1_serialize_uncompressed, o.g1_mul, o.G1_GEN),
                                     (kz.G2, 1, 192, o.ark_g2_serialize_uncompressed, o.g2_mul, o.G2_GEN)):
        picks = sorted(rnd.randrange(n) for _ in range(64))
        for a in range(0, n, slab):
            ctx.generate_device(g, ZC, s0, tau, a, slab, d_in.data_ptr())
            ctx.convert_device(g, ZC, d_in.data_ptr(), AU, d_out.data_ptr(), slab, STRICT, status.data_ptr(), base_index=a)
            torch.cuda.synchronize()
            for i in [a, a + slab - 1] + [p for p in picks if a <= p < a + slab]:
                got = bytes(d_out[(i - a) * ro:(i - a + 1) * ro].cpu().numpy())
                want = enc(mul(gen, s0 * pow(tau, i, o.R_ORDER) % o.R_ORDER))
                assert got == want, (g, i)
    assert int(status.item()) == -1


def test_generator_vs_oracles(ctx, cref):
    rnd = random.Random(5)
    tau, beta = rnd.randrange(1, o.R_ORDER), rnd.randrange(1, o.R_ORDER)
    got = ctx.generate(1, ZC, beta, tau, 7, 25)
    want = b"".join(o.zcash_g1_compressed_encode(o.g1_mul(o.G1_GEN, beta * pow(tau, 7 + i, o.R_ORDER) % o.R_ORDER))
                    for i in range(25))
    assert got.tobytes() == want
    for g, fmt in ((1, ZU), (2, ZC), (2, ZU)):
        assert ctx.generate(g, fmt, 1, tau, 3, 700).tobytes() == cref.generate(g, fmt, 1, tau, 3, 700, 16)


def test_pipeline_2pow10_vs_c_oracle(ctx, cref):
    """Whole preprocess at N = 2^10 against the C oracle assembling the same layout."""
    n = 1 << 10
    tau, alpha, beta = o.derive_scalars(0xB200)
    secs = [(1, 1, 2 * n - 1), (2, 1, n), (1, alpha, n), (1, beta, n), (2, beta, 1)]
    body = b"".join(cref.generate(g, ZC, s0, tau, 0, cnt, 16) for g, s0, cnt in secs)
    resp = o.filler_bytes(1, 64, b"hash") + body + o.filler_bytes(1, o.PUBKEY_SIZE, b"pubkey")
    assert len(resp) == o.response_size(n)
    off = 0
    ark = []
    for g, _, cnt in secs:
        ln = cnt * SZ[g][ZC]
        zu, _ = cref.convert(g, ZC, body[off:off + ln], ZU, 0, 16)
        au, st = cref.convert(g, ZU, zu, AU, 4, 16)
        assert not any(st)
        ark.append(au)
        off += ln
    kgz = ark[0] + ark[2] + ark[0][:96] + ark[2][:96] + ark[1][:384]
    fast = ark[0] + ark[2] + ark[1][:384] + ark[1]
    assert ctx.preprocess(kz.VARIANT_KGZ, resp, n).tobytes() == kgz
    assert ctx.preprocess(kz.VARIANT_FASTKGZ, resp, n).tobytes() == fast
    # a corrupted point in alpha_g1 is reported with its section and index
    bad = bytearray(resp)
    pos = 64 + (2 * n - 1) * 48 + n * 96 + 17 * 48
    while True:
        bad[pos + 47] = (bad[pos + 47] + 1) & 0xFF
        if o.fq_sqrt((int.from_bytes(bytes([bad[pos] & 0x1F]) + bytes(bad[pos + 1:pos + 48]), "big") ** 3 + 4) % o.P) is not None:
            break
    with pytest.raises(kz.PtauError) as e:
        ctx.preprocess(kz.VARIANT_KGZ, bytes(bad), n)
    assert e.value.section == 2 and e.value.index == 17 and e.value.code == kz.BAD_NOT_IN_SUBGROUP


# ---- full-size properties (BASELINE.json configs 2 and 3) --------------------------------
def _reverse_fields(a: np.ndarray, nfields: int) -> np.ndarray:
    return a.reshape(-1, nfields, 48)[:, :, ::-1]


@pytest.mark.parametrize("log2n", [20])
def test_config2_g1_uncompressed_full_size(ctx, log2n):
    """2^20 uncompressed G1 tau-powers: output must be the byte reversal of each
    coordinate (src/lib.rs:49-50), every point must pass, and the generator's known-tau
    chain ties the points to [tau^i]G."""
    n = 1 << log2n
    tau = o.derive_scalars(0xB200)[0]
    zu = ctx.generate(1, ZU, 1, tau, 0, n)
    au = ctx.convert(1, ZU, zu, AU, STRICT)
    assert np.array_equal(au.reshape(-1, 2, 48), _reverse_fields(zu, 2))
    assert zu[:96].tobytes() == o.zcash_g1_uncompressed_encode(o.G1_GEN)
    for i in (1, 2, n // 3, n - 1):  # spot-check against the big-int oracle
        assert zu[i * 96:(i + 1) * 96].tobytes() == o.zcash_g1_uncompressed_encode(o.g1_mul(o.G1_GEN, pow(tau, i, o.R_ORDER)))
    # idempotence / round trip: ark -> zcash -> ark
    back = ctx.convert(1, AU, au, ZU, 0)
    assert np.array_equal(back, zu)
    # one flipped bit anywhere is caught, with its exact index
    k = 777_777 % n
    zu[k * 96 + 60] ^= 0x10
    with pytest.raises(kz.PtauError) as e:
        ctx.convert(1, ZU, zu, AU, STRICT)
    assert e.value.index == k


def test_config3_compressed_full_size(ctx):
    """2^21 compressed G1 + 2^21 compressed G2 (reduced to 2^19 G2 under PTAU_TEST_FAST):
    decompress(compressed) must equal the independently generated uncompressed stream
    (encode -> decode round trip), and the fused path must equal the two-stage one."""
    n1 = 1 << 21
    n2 = 1 << (19 if os.environ.get("PTAU_TEST_FAST") else 21)
    tau = o.derive_scalars(0xB200)[0]
    for g, n in ((1, n1), (2, n2)):
        zc = ctx.generate(g, ZC, 1, tau, 0, n)
        zu = ctx.generate(g, ZU, 1, tau, 0, n)
        dec = ctx.convert(g, ZC, zc, ZU, kz.CHECKS_DECOMPRESS)
        assert np.array_equal(dec, zu)
        fused = ctx.convert(g, ZC, zc, AU, STRICT)
        staged = ctx.convert(g, ZU, zu, AU, kz.CHECKS_READ)
        assert np.array_equal(fused, staged)
        nf = 2 if g == 1 else 4
        rev = _reverse_fields(zu, nf)
        if g == 2:
            rev = rev[:, [1, 0, 3, 2], :]  # c1|c0 -> c0|c1 (src/lib.rs:64-71)
        assert np.array_equal(fused.reshape(-1, nf, 48), rev)
        # both sort flags occur
        flags = zc.reshape(n, -1)[:, 0] & 0x20
        assert 0.4 < float((flags != 0).mean()) < 0.6


def test_bench_dump_outputs_vs_c_oracle(cref, tmp_path):
    """`bench.py --dump-outputs` at 2^16 points per group: --steps sets the timed steps, the files hold a sorted sample
    of 2^15 distinct indices with their G1 / G2 ark records as float32 bytes, and the records of the sampled indices
    below 2^14 equal the C oracle's conversion of the same [tau^i]G."""
    import subprocess
    import sys

    import bench
    from conftest import ROOT

    n, n_check, th = 1 << 16, 1 << 14, os.cpu_count() or 1
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--log2-points", "16", "--steps", "2",
                        "--warmup", "3", "--no-extra", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])["steps"] == 2
    arrays = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert sorted(arrays) == ["g1_ark_uncompressed", "g2_ark_uncompressed", "index", "status"]
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert arrays["status"].tolist() == [-1.0]
    idx = arrays["index"]
    assert idx.shape == (1 << 15,) and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < n
    assert np.array_equal(idx, idx.astype(np.int64))
    mask = idx < n_check
    for g, name, ro in ((1, "g1_ark_uncompressed", 96), (2, "g2_ark_uncompressed", 192)):
        rec = arrays[name]
        assert rec.shape == (1 << 15, ro) and np.array_equal(rec, rec.astype(np.uint8))
        zc = cref.generate(g, ZC, 1, bench.TAU, 0, n_check, th)
        zu, st = cref.convert(g, ZC, zc, ZU, 0, th)
        assert not any(st)
        want, st = cref.convert(g, ZU, zu, AU, 4, th)
        assert not any(st)
        want = np.frombuffer(want, dtype=np.uint8).reshape(n_check, ro)[idx[mask].astype(np.int64)]
        assert np.array_equal(rec[mask].astype(np.uint8), want)


def test_config4_validated_load(ctx, tmp_path):
    """BASELINE configs[3]: load of a 2^21-power setup (powers_of_g up to degree 2^22-2; 2^17
    powers under PTAU_TEST_FAST), both variants, through the file loaders: validated and
    unchecked loads return identical Montgomery limbs; limbs decode back to the file;
    KZG10 commit sanity with the known tau; a corrupted point deep in the file is found by
    the validated load only."""
    k = 17 if os.environ.get("PTAU_TEST_FAST") else 21
    n = 1 << k
    tau, alpha, _ = o.derive_scalars(0xB200)
    g1 = np.concatenate([ctx.generate(1, ZU, 1, tau, 0, 2 * n - 1), ctx.generate(1, ZU, alpha, tau, 0, n)])
    g1_ark = ctx.convert(1, ZU, g1, AU, 0)
    del g1
    nh = n if k <= 18 else 1 << 18  # powers_of_h of the fastkgz file (kept smaller: 192 B each)
    g2_ark = ctx.convert(2, ZU, ctx.generate(2, ZU, 1, tau, 0, max(nh, 2)), AU, 0)
    kgz = np.concatenate([g1_ark, g1_ark[:96], g1_ark[(2 * n - 1) * 96:(2 * n) * 96], g2_ark[:384]])
    assert kgz.size == o.kgz_size(n)
    path = str(tmp_path / "kzg_setup")
    kgz.tofile(path)
    powers, vk = kz.load_kzg_setup(path, ctx=ctx)                       # reference: unchecked
    powers_v, vk_v = kz.load_kzg_setup(path, ctx=ctx, checks=STRICT)    # validated
    assert powers.powers_of_g.shape == (2 * n - 1, 104) and powers.powers_of_gamma_g.shape == (n, 104)
    assert np.array_equal(powers.powers_of_g, powers_v.powers_of_g)
    assert np.array_equal(powers.powers_of_gamma_g, powers_v.powers_of_gamma_g)
    assert np.array_equal(vk.h, vk_v.h) and np.array_equal(vk.beta_h, vk_v.beta_h)
    assert not powers.powers_of_g[:, 96:].any()
    for i in (0, 1, n, 2 * n - 2):
        x, y, inf = o.ark_g1_deserialize_unchecked(kgz[i * 96:(i + 1) * 96].tobytes())
        assert powers.powers_of_g[i].tobytes() == o.g1_mont_record(x, y, inf)
    assert vk.g.tobytes() == powers.powers_of_g[0].tobytes() and vk.gamma_g.tobytes() == powers.powers_of_gamma_g[0].tobytes()
    # serialize direction: Montgomery limbs -> ark bytes reproduces the file (round trip)
    back = ctx.convert(1, ML, powers.powers_of_g[:4096].reshape(-1), AU, 0)
    assert np.array_equal(back, kgz[:4096 * 96])
    # KZG10 commit sanity with the known tau: sum c_i [tau^i]G == [p(tau)]G
    coeffs = [3, 1, 4, 1, 5, 9, 2, 6]
    pts = []
    for i in range(len(coeffs)):
        x, y, _ = o.ark_g1_deserialize_unchecked(kgz[i * 96:(i + 1) * 96].tobytes())
        pts.append((x, y))
    ptau = sum(c * pow(tau, i, o.R_ORDER) for i, c in enumerate(coeffs)) % o.R_ORDER
    assert o.kzg_commit(pts, coeffs) == o.g1_mul(o.G1_GEN, ptau)
    # corrupt one point deep in the file: validated load finds it, unchecked load does not
    kgz[(2 * n + 5) * 96 + 3] ^= 0x04
    kgz.tofile(path)
    kz.load_kzg_setup(path, ctx=ctx)
    with pytest.raises(kz.PtauError) as e:
        kz.load_kzg_setup(path, ctx=ctx, checks=STRICT)
    assert e.value.index == 2 * n + 5
    del kgz, powers, powers_v
    # UniversalParams variant (load_fastkzg_setup), n_h powers
    m = nh
    fast = np.concatenate([g1_ark[:(2 * m - 1) * 96], g1_ark[(2 * n - 1) * 96:(2 * n - 1 + m) * 96], g2_ark[:384], g2_ark[:m * 192]])
    assert fast.size == o.fastkgz_size(m)
    fast.tofile(path)
    params, ph = kz.load_fastkzg_setup(path, ctx=ctx, checks=STRICT)
    assert params.powers_of_g.shape == (2 * m - 1, 104) and ph.shape == (m, 200)
    assert params.beta_h.tobytes() == ph[1].tobytes() and params.h.tobytes() == ph[0].tobytes()
    x, y, inf = o.ark_g2_deserialize_unchecked(fast[-192:].tobytes())
    assert ph[m - 1].tobytes() == o.g2_mont_record(x, y, inf)


def test_kzg10_commit_open_known_tau(ctx, tmp_path):
    """SURVEY 8f-4, first step: KZG10 commit / open on the GPU, mirroring the reference's
    end_to_end_test_kzg (src/lib.rs:250-289: 10 x 10 random polynomials of degree 2..19,
    hiding_bound 1) but verified without pairings through the known tau:
      C = [p(tau) + alpha b(tau)] G ,   W = [w(tau) + alpha bw(tau)] G ,   p(tau) - v = (tau - z) w(tau)."""
    n = 1 << 10
    tau, alpha, _ = o.derive_scalars(0xB200)
    g1 = np.concatenate([ctx.generate(1, ZU, 1, tau, 0, 2 * n - 1), ctx.generate(1, ZU, alpha, tau, 0, n)])
    g2 = ctx.generate(2, ZU, 1, tau, 0, 2)
    setup = np.concatenate([ctx.convert(1, ZU, g1, AU, 0), ctx.convert(1, ZU, g1[:96], AU, 0),
                            ctx.convert(1, ZU, g1[(2 * n - 1) * 96:(2 * n) * 96], AU, 0), ctx.convert(2, ZU, g2, AU, 0)])
    path = str(tmp_path / "kzg_setup")
    setup.tofile(path)
    powers, vk = kz.load_kzg_setup(path, ctx=ctx)
    R = o.R_ORDER

    def ev(c, x):
        return sum(v * pow(x, i, R) for i, v in enumerate(c)) % R

    def rec(k):
        q = o.g1_mul(o.G1_GEN, k % R)
        return o.g1_mont_record(0, 1, True) if q is None else o.g1_mont_record(q[0], q[1], False)

    rnd = random.Random(20)
    for _ in range(10):
        degree = rnd.randrange(2, 20)
        for _ in range(3):
            p = [rnd.randrange(R) for _ in range(degree + 1)]
            b = [rnd.randrange(R) for _ in range(2)]  # hiding_bound = Some(1)
            comm = kz.KZG10.commit(powers, p, blinding=b, ctx=ctx)
            assert comm.tobytes() == rec(ev(p, tau) + alpha * ev(b, tau))
            z = rnd.randrange(R)
            value, proof, random_v = kz.KZG10.open(powers, p, z, blinding=b, ctx=ctx)
            assert value == ev(p, z) and random_v == ev(b, z)
            _, w = kz.KZG10._quotient(p, z)
            _, bw = kz.KZG10._quotient(b, z)
            assert proof.tobytes() == rec(ev(w, tau) + alpha * ev(bw, tau))
            assert (ev(p, tau) - value) % R == (tau - z) * ev(w, tau) % R
    # device-resident powers (uploaded once; only scalars travel): same commitments and proofs
    dev = powers.to_device(ctx)
    assert len(dev.powers_of_g) == 2 * n - 1 and len(dev.powers_of_gamma_g) == n
    for _ in range(3):
        p = [rnd.randrange(R) for _ in range(rnd.randrange(2, 2 * n - 1))]
        b = [rnd.randrange(R) for _ in range(2)]
        assert kz.KZG10.commit(dev, p, blinding=b, ctx=ctx).tobytes() == kz.KZG10.commit(powers, p, blinding=b, ctx=ctx).tobytes()
        assert kz.KZG10.commit(dev, p, ctx=ctx).tobytes() == rec(ev(p, tau))
        z = rnd.randrange(R)
        v1, w1, r1 = kz.KZG10.open(dev, p, z, blinding=b, ctx=ctx)
        v2, w2, r2 = kz.KZG10.open(powers, p, z, blinding=b, ctx=ctx)
        assert (v1, r1) == (v2, r2) and w1.tobytes() == w2.tobytes()
    assert kz.KZG10.commit(dev, [], ctx=ctx).tobytes() == o.g1_mont_record(0, 1, True)
    with pytest.raises(kz.PtauError):
        kz.KZG10.commit(dev, [1] * (2 * n), ctx=ctx)
    # special cases of the group law inside the MSM
    assert kz.KZG10.commit(powers, [0, 0, 0], ctx=ctx).tobytes() == o.g1_mont_record(0, 1, True)  # zero polynomial
    assert kz.KZG10.commit(powers, [], ctx=ctx).tobytes() == o.g1_mont_record(0, 1, True)
    same = kz.Powers(powers_of_g=np.repeat(powers.powers_of_g[1:2], 16, axis=0), powers_of_gamma_g=powers.powers_of_gamma_g)
    assert kz.KZG10.commit(same, [1, 1], ctx=ctx).tobytes() == rec(2 * tau)               # P + P -> doubling
    assert kz.KZG10.commit(same, [5, R - 5], ctx=ctx).tobytes() == o.g1_mont_record(0, 1, True)  # P + (-P)
    assert kz.KZG10.commit(same, [3] * 16, ctx=ctx).tobytes() == rec(48 * tau)
    assert kz.KZG10.commit(same, [0, 7, 0, 0, 0, 0, 0, 0, 0, 9], ctx=ctx).tobytes() == rec(16 * tau)
    # a full-degree polynomial against p(tau)
    big = [rnd.randrange(R) for _ in range(2 * n - 1)]
    assert kz.KZG10.commit(powers, big, ctx=ctx).tobytes() == rec(ev(big, tau))
    with pytest.raises(kz.PtauError):
        kz.KZG10.commit(powers, [1] * (2 * n), ctx=ctx)  # Error::TooManyCoefficients
    bad = np.frombuffer((R).to_bytes(32, "little"), dtype=np.uint8)
    out = np.zeros(104, dtype=np.uint8)
    assert kz._ffi.lib().ptau_kzg_commit(ctx._h, powers.powers_of_g[:1].ctypes.data, bad.ctypes.data, 1, out.ctypes.data) == kz._ffi.ERR_ARG


def test_msm_bucket_method_window_widths_and_adversarial_scalars(ctx):
    """The bucket (Pippenger) MSM behind KZG10::commit at sizes that select every window width
    (c = 3 .. 16), against the known tau:  sum c_i [tau^i]G == [sum c_i tau^i]G.
    Adversarial scalars: all equal (one hot bucket per window), r - 1 (carries through every signed
    window), digits exactly on the signed-window boundary 2^(cw-1), zero scalars, the same point
    repeated, and records flagged infinity (which must contribute nothing)."""
    R = o.R_ORDER
    tau = o.derive_scalars(0xC0FFEE)[0]
    nmax = (1 << 20) + 3
    pts = ctx.convert(1, ZU, ctx.generate(1, ZU, 1, tau, 0, nmax), ML, 0).reshape(nmax, 104)
    lib = kz._ffi.lib()

    def msm(points, scalars):
        n = len(scalars)
        sc = np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in scalars), dtype=np.uint8)
        out = np.zeros(104, dtype=np.uint8)
        pp = np.ascontiguousarray(points[:n])
        assert lib.ptau_kzg_commit(ctx._h, pp.ctypes.data, sc.ctypes.data, n, out.ctypes.data) == 0
        return out.tobytes()

    def rec(k):
        q = o.g1_mul(o.G1_GEN, k % R)
        return o.g1_mont_record(0, 1, True) if q is None else o.g1_mont_record(q[0], q[1], False)

    tp = [1]
    for _ in range(nmax - 1):
        tp.append(tp[-1] * tau % R)

    def ev(scalars):
        return sum(c * t for c, t in zip(scalars, tp)) % R

    rnd = random.Random(77)
    def geometry(n):  # mirrors msm_g1_plan
        lg = max(n - 1, 0).bit_length()
        c = min(max(lg - 4, 3), 16)
        W = (256 + c - 1) // c
        a = 256 - (c - 1) * W
        return c, W, a

    widths = set()
    for n in (1, 2, 127, 128, 200, 300, 600, 2047, 2048, 4096, 5000, 10_000, (1 << 15) - 1, 1 << 15, 40_000, (1 << 16) + 1,
              (1 << 17) + 1, (1 << 18) + 5, nmax):
        widths.add(geometry(n)[0])
        sc = [rnd.randrange(R) for _ in range(n)]
        assert msm(pts, sc) == rec(ev(sc)), n
    assert widths == set(range(3, 17))
    for n in (100, 1000, 20_000, 100_000, (1 << 18) + 5):
        c, W, a = geometry(n)
        tops = [(w + 1) * c - 1 if w < a else a * c + (w - a + 1) * (c - 1) - 1 for w in range(W - 1)]  # top bit of each window
        for sc in ([R - 1] * n,                                            # = -sum P_i, carries everywhere
                   [0x1234567] * n,                                        # one hot bucket per window
                   [sum(1 << b for b in tops[:-1])] * n,                   # digits on the boundary 2^(cw-1)
                   [sum(1 << b for b in tops[:-1]) + 1] * n,               # ... and just above it (negative digits, carries)
                   [0] * (n - 1) + [5],
                   [rnd.randrange(1 << 20) for _ in range(n)]):            # short scalars: the top windows stay empty
            assert msm(pts, sc) == rec(ev(sc)), (n, c)
    # the same point many times, and P + (-P) inside one bucket
    same = np.repeat(pts[3:4], 5000, axis=0)
    assert msm(same, [7] * 5000) == rec(35_000 * tp[3])
    assert msm(same, [9, R - 9] * 2500) == o.g1_mont_record(0, 1, True)
    # records flagged infinity are skipped
    holes = pts[:3000].copy()
    holes[::3, 96] = 1
    sc = [rnd.randrange(R) for _ in range(3000)]
    assert msm(holes, sc) == rec(sum(c * t for i, (c, t) in enumerate(zip(sc, tp)) if i % 3))


def _g1_rec(q):
    return np.frombuffer(o.g1_mont_record(0, 1, True) if q is None else o.g1_mont_record(q[0], q[1], False), dtype=np.uint8)


def _g2_rec(q):
    z2 = (0, 0)
    return np.frombuffer(o.g2_mont_record(z2, (1, 0), True) if q is None else o.g2_mont_record(q[0], q[1], False), dtype=np.uint8)


def test_pairing_value_vs_oracle(ctx):
    """GPU pairing (tower arithmetic, projective lines, split final exponentiation) against the independent
    CPU restatement (flat Fq12, affine lines in E(Fq12), one plain exponentiation): the 576 GT bytes themselves."""
    import pairing_oracle as po

    rnd = random.Random(5)
    a, b, c, d = (rnd.randrange(1, o.R_ORDER) for _ in range(4))
    P1, Q1, P2, Q2 = o.g1_mul(o.G1_GEN, a), o.g2_mul(o.G2_GEN, b), o.g1_mul(o.G1_GEN, c), o.g2_mul(o.G2_GEN, d)
    negP1 = (P1[0], (-P1[1]) % o.P)
    items = [((P1, Q1), (None, Q2)),           # one pairing, the other slot at infinity
             ((P1, Q1), (P2, Q2)),             # product of two
             ((P1, Q1), (negP1, Q1)),          # = 1
             ((P2, None), (None, None)),       # empty product = 1
             ((o.G1_GEN, o.G2_GEN), (None, None))]
    g1 = np.stack([np.stack([_g1_rec(p) for p, _ in it]) for it in items])
    g2 = np.stack([np.stack([_g2_rec(q) for _, q in it]) for it in items])
    gt, one = kz.KZG10.pairing_product2(g1, g2, ctx=ctx)
    assert list(one) == [False, False, True, True, False]

    def flat(rec):
        coeffs = [int.from_bytes(rec[48 * i:48 * i + 48].tobytes(), "little") for i in range(12)]
        assert all(v < o.P for v in coeffs)
        return po.f12_from_tower(coeffs)

    e11 = po.pairing(P1, Q1)
    assert flat(gt[0]) == e11
    assert flat(gt[1]) == po.f12_mul(e11, po.pairing(P2, Q2))
    assert flat(gt[2]) == po.F12_ONE and flat(gt[3]) == po.F12_ONE
    # bilinearity on the GPU value: e(aG, bH) == e(G, H)^(ab)
    assert e11 == po.f12_pow(flat(gt[4]), a * b % o.R_ORDER)


def test_kzg10_check_mirrors_reference_test(ctx, tmp_path):
    """The reference's end_to_end_test_kzg (src/lib.rs:250-289): random polynomials of degree 2..19, hiding bound 1,
    commit -> open at a random point -> KZG10::check must accept; plus what the reference does not test: a wrong
    value / point / proof / commitment must be rejected, the boolean must equal the CPU restatement's, and
    batch_check must agree."""
    import pairing_oracle as po

    n = 32
    tau, alpha, _ = o.derive_scalars(0xB201)
    g1 = np.concatenate([ctx.generate(1, ZU, 1, tau, 0, 2 * n - 1), ctx.generate(1, ZU, alpha, tau, 0, n)])
    g2 = ctx.generate(2, ZU, 1, tau, 0, 2)
    setup = np.concatenate([ctx.convert(1, ZU, g1, AU, 0), ctx.convert(1, ZU, g1[:96], AU, 0),
                            ctx.convert(1, ZU, g1[(2 * n - 1) * 96:(2 * n) * 96], AU, 0), ctx.convert(2, ZU, g2, AU, 0)])
    path = str(tmp_path / "kzg_setup")
    setup.tofile(path)
    powers, vk = kz.load_kzg_setup(path, ctx=ctx)
    R = o.R_ORDER
    rnd = random.Random(21)
    comms, points, values, proofs, rvs = [], [], [], [], []
    for i in range(20):
        degree = rnd.randrange(2, 20)
        p = [rnd.randrange(R) for _ in range(degree + 1)]
        b = [rnd.randrange(R) for _ in range(2)] if i % 4 else None   # every fourth opening without hiding
        comm = kz.KZG10.commit(powers, p, blinding=b, ctx=ctx)
        z = rnd.randrange(R)
        value, proof, random_v = kz.KZG10.open(powers, p, z, blinding=b, ctx=ctx)
        assert kz.KZG10.check(vk, comm, z, value, proof, random_v, ctx=ctx)          # the reference's assertion
        comms.append(comm); points.append(z); values.append(value); proofs.append(proof); rvs.append(random_v)
    N = len(points)
    assert kz.KZG10.check_many(vk, comms, points, values, proofs, rvs, ctx=ctx).all()
    # tampering: each of the five inputs in turn
    bad_values = [(v + 1) % R for v in values]
    assert not kz.KZG10.check_many(vk, comms, points, bad_values, proofs, rvs, ctx=ctx).any()
    bad_points = [(z + 1) % R for z in points]
    assert not kz.KZG10.check_many(vk, comms, bad_points, values, proofs, rvs, ctx=ctx).any()
    assert not kz.KZG10.check_many(vk, comms, points, values, proofs[1:] + proofs[:1], rvs, ctx=ctx).any()
    assert not kz.KZG10.check_many(vk, comms[1:] + comms[:1], points, values, proofs, rvs, ctx=ctx).any()
    hid = [i for i in range(N) if rvs[i] is not None]
    bad_rv = [None if r is None else (r + 1) % R for r in rvs]
    res = kz.KZG10.check_many(vk, comms, points, values, proofs, bad_rv, ctx=ctx)
    assert not res[hid].any() and res[[i for i in range(N) if rvs[i] is None]].all()
    # the fixed-base tables are cached per verifier key: another key must rebuild them, and going back must too
    vk_g = kz.VerifierKey(g=powers.powers_of_g[1], gamma_g=vk.gamma_g, h=vk.h, beta_h=vk.beta_h)
    assert not kz.KZG10.check_many(vk_g, comms, points, values, proofs, rvs, ctx=ctx).any()
    vk_gg = kz.VerifierKey(g=vk.g, gamma_g=powers.powers_of_g[2], h=vk.h, beta_h=vk.beta_h)
    res = kz.KZG10.check_many(vk_gg, comms, points, values, proofs, rvs, ctx=ctx)
    assert not res[hid].any() and res[[i for i in range(N) if rvs[i] is None]].all()
    g2x = ctx.convert(2, ZU, ctx.generate(2, ZU, 5, tau, 0, 2), ML, 0).reshape(2, 200)   # (5H, 5 tau H): consistent pair
    vk_h = kz.VerifierKey(g=vk.g, gamma_g=vk.gamma_g, h=g2x[0], beta_h=g2x[1])
    assert kz.KZG10.check_many(vk_h, comms, points, values, proofs, rvs, ctx=ctx).all()
    vk_hbad = kz.VerifierKey(g=vk.g, gamma_g=vk.gamma_g, h=g2x[0], beta_h=vk.beta_h)     # (5H, tau H): inconsistent
    assert not kz.KZG10.check_many(vk_hbad, comms, points, values, proofs, rvs, ctx=ctx).any()
    assert kz.KZG10.check_many(vk, comms, points, values, proofs, rvs, ctx=ctx).all()
    # same boolean as the CPU restatement of KZG10::check (slow: a few cases)
    ovk = (o.g1_mul(o.G1_GEN, 1), o.g1_mul(o.G1_GEN, alpha), o.G2_GEN, o.g2_mul(o.G2_GEN, tau))

    def aff(rec):
        x, y, inf = kz.g1_limbs(rec)
        if inf:
            return None
        rinv = pow(o.MONT_R, -1, o.P)
        xi = sum(int(v) << (64 * k) for k, v in enumerate(x)) * rinv % o.P
        yi = sum(int(v) << (64 * k) for k, v in enumerate(y)) * rinv % o.P
        return (xi, yi)

    for i in (0, 1):
        assert po.kzg_check(ovk, aff(comms[i]), points[i], values[i], aff(proofs[i]), rvs[i]) is True
        assert po.kzg_check(ovk, aff(comms[i]), points[i], bad_values[i], aff(proofs[i]), rvs[i]) is False
    # batch_check (ark: r_0 = 1, then u128 randomizers)
    rz = [1] + [rnd.randrange(1 << 128) for _ in range(N - 1)]
    assert kz.KZG10.batch_check(vk, comms, points, values, proofs, rvs, randomizers=rz, ctx=ctx)
    assert not kz.KZG10.batch_check(vk, comms, points, values[:-1] + [bad_values[-1]], proofs, rvs, randomizers=rz, ctx=ctx)
    assert kz.KZG10.batch_check(vk, comms[:3], points[:3], values[:3], proofs[:3], rvs[:3], ctx=ctx)   # own randomizers
    assert po.kzg_batch_check(ovk, [aff(c) for c in comms[:3]], points[:3], values[:3],
                              [(aff(w), r) for w, r in zip(proofs[:3], rvs[:3])], rz[:3]) is True
    # a non-canonical scalar is an argument error, as in ptau_kzg_commit
    bad = np.frombuffer(R.to_bytes(32, "little"), dtype=np.uint8)
    ok = np.zeros(1, dtype=np.uint8)
    g1v = np.ascontiguousarray(np.concatenate([vk.g.reshape(-1), vk.gamma_g.reshape(-1)]))
    g2v = np.ascontiguousarray(np.concatenate([vk.h.reshape(-1), vk.beta_h.reshape(-1)]))
    c0 = np.ascontiguousarray(comms[0])
    assert kz._ffi.lib().ptau_kzg_check(ctx._h, g1v.ctypes.data, g2v.ctypes.data, c0.ctypes.data, bad.ctypes.data, bad.ctypes.data,
                                        c0.ctypes.data, None, 1, ok.ctypes.data) == kz._ffi.ERR_ARG


def test_g2_prepared_on_gpu(ctx):
    """ptau_g2_prepare = ark-ec 0.2 G2Prepared::from (prepared_h / prepared_beta_h, src/lib.rs:223-224): the 68 line
    coefficient triples per point against oracle/pairing_oracle.py, infinity, and the VerifierKey helpers."""
    import pairing_oracle as po

    pts = [o.g2_mul(o.G2_GEN, k) for k in (1, 3, 0xDEADBEEF)] + [None]
    recs = np.frombuffer(b"".join(o.g2_mont_record((0, 0), (1, 0), True) if q is None else o.g2_mont_record(q[0], q[1], False)
                                  for q in pts), dtype=np.uint8).reshape(-1, 200)
    prep = kz.g2_prepare(recs, ctx=ctx)
    rinv = pow(1 << 384, -1, o.P)
    for q, pr in zip(pts, prep):
        want, is_inf = po.g2_prepared_coeffs(q)
        assert pr.infinity == is_inf and pr.ell_coeffs.shape[0] == len(want)
        for t, w in enumerate(want):
            blob = pr.ell_coeffs[t].tobytes()
            vals = [int.from_bytes(blob[48 * k:48 * k + 48], "little") * rinv % o.P for k in range(6)]
            assert ((vals[0], vals[1]), (vals[2], vals[3]), (vals[4], vals[5])) == w
    g1 = np.frombuffer(o.g1_mont_record(o.G1_GEN[0], o.G1_GEN[1], False), dtype=np.uint8)
    vk = kz.VerifierKey(g=g1, gamma_g=g1, h=recs[0], beta_h=recs[1])
    assert vk.prepared_h(ctx).ell_coeffs.tobytes() == prep[0].ell_coeffs.tobytes()
    assert vk.prepared_beta_h(ctx).ell_coeffs.tobytes() == prep[1].ell_coeffs.tobytes()


def test_multi_gpu_sharding_is_invisible(cref):
    """Same bytes and same first-bad-index with 1 GPU and with every GPU of the box."""
    from kzg_setup_powersoftau_b200 import _ffi

    ngpu = _ffi.lib().ptau_device_count()
    if ngpu < 2:
        pytest.skip("single-GPU box")
    tau = o.derive_scalars(7)[0]
    n = 50_001
    with kz.Context(1) as c1, kz.Context(ngpu, chunk_points=4096) as cn:
        zc = c1.generate(2, ZC, 1, tau, 0, n)
        a = c1.convert(2, ZC, zc, AU, STRICT)
        b = cn.convert(2, ZC, zc, AU, STRICT)
        assert np.array_equal(a, b)
        zc[30_000 * 96 + 40] ^= 1
        zc[45_000 * 96 + 40] ^= 1
        codes = []
        for c in (c1, cn):
            with pytest.raises(kz.PtauError) as e:
                c.convert(2, ZC, zc, AU, STRICT)
            codes.append((e.value.index, e.value.code))
        assert codes[0] == codes[1] and codes[0][0] == 30_000


def test_multi_gpu_consumer_ops():
    """KZG10 commit (MSM) and check sharded by index range over every GPU of the box: same commitment bytes and same
    booleans as with one GPU."""
    from kzg_setup_powersoftau_b200 import _ffi

    ngpu = _ffi.lib().ptau_device_count()
    if ngpu < 2:
        pytest.skip("single-GPU box")
    R = o.R_ORDER
    tau = o.derive_scalars(11)[0]
    n = 70_001
    rnd = random.Random(3)
    with kz.Context(1) as c1, kz.Context(ngpu) as cn:
        pts = c1.convert(1, ZU, c1.generate(1, ZU, 1, tau, 0, n), ML, 0).reshape(n, 104)
        sc = [rnd.randrange(R) for _ in range(n)]
        pw = kz.Powers(powers_of_g=pts, powers_of_gamma_g=pts[:1])
        a = kz.KZG10.commit(pw, sc, ctx=c1)
        b = kz.KZG10.commit(pw, sc, ctx=cn)
        assert a.tobytes() == b.tobytes()
        q = o.g1_mul(o.G1_GEN, sum(c * pow(tau, i, R) for i, c in enumerate(sc[:2000])) % R)
        assert kz.KZG10.commit(pw, sc[:2000], ctx=cn).tobytes() == o.g1_mont_record(q[0], q[1], False)   # small: one GPU
        g2p = c1.convert(2, ZU, c1.generate(2, ZU, 1, tau, 0, 2), ML, 0).reshape(2, 200)
        vk = kz.VerifierKey(g=pts[0], gamma_g=pts[5], h=g2p[0], beta_h=g2p[1])
        poly = [rnd.randrange(R) for _ in range(12)]
        comm = kz.KZG10.commit(pw, poly, ctx=c1)
        m = 3000
        zs = [rnd.randrange(R) for _ in range(m)]
        opened = [kz.KZG10.open(pw, poly, z, ctx=c1) for z in zs[:8]]
        vals = [opened[i % 8][0] for i in range(m)]
        prfs = [opened[i % 8][1] for i in range(m)]
        zs = [zs[i % 8] for i in range(m)]
        vals[1234] = (vals[1234] + 1) % R
        vals[2999] = (vals[2999] + 1) % R
        r1 = kz.KZG10.check_many(vk, [comm] * m, zs, vals, prfs, ctx=c1)
        rn = kz.KZG10.check_many(vk, [comm] * m, zs, vals, prfs, ctx=cn)
        assert (r1 == rn).all() and r1.sum() == m - 2 and not r1[1234] and not r1[2999]


def test_pairing_golden_vectors(ctx):
    """tests/golden/pairing_vectors.json through the C ABI on the GPU."""
    import pairing_oracle as po

    with open(os.path.join(GOLDEN, "pairing_vectors.json")) as f:
        vec = json.load(f)
    g1 = np.stack([np.stack([_g1_rec(o.g1_mul(o.G1_GEN, int(s, 16)) if int(s, 16) else None) for s in pv["g1_scalars"]])
                   for pv in vec["products"]])
    g2 = np.stack([np.stack([_g2_rec(o.g2_mul(o.G2_GEN, int(s, 16)) if int(s, 16) else None) for s in pv["g2_scalars"]])
                   for pv in vec["products"]])
    gt, one = kz.KZG10.pairing_product2(g1, g2, ctx=ctx)
    for i, pv in enumerate(vec["products"]):
        flat = po.f12_from_tower([int.from_bytes(gt[i][48 * k:48 * k + 48].tobytes(), "little") for k in range(12)])
        assert flat == [int(v, 16) for v in pv["gt_flat"]] and bool(one[i]) == pv["is_one"]
    tau, alpha, _ = o.derive_scalars(0xB200)
    g2v = ctx.convert(2, ZU, ctx.generate(2, ZU, 1, tau, 0, 2), ML, 0).reshape(2, 200)
    vk = kz.VerifierKey(g=_g1_rec(o.G1_GEN), gamma_g=_g1_rec(o.g1_mul(o.G1_GEN, alpha)), h=g2v[0], beta_h=g2v[1])
    ks = vec["kzg_checks"]
    comms = [_g1_rec(o.g1_mul(o.G1_GEN, int(k["commitment_scalar"], 16))) for k in ks]
    prfs = [_g1_rec(o.g1_mul(o.G1_GEN, int(k["proof_scalar"], 16)) if int(k["proof_scalar"], 16) else None) for k in ks]
    res = kz.KZG10.check_many(vk, comms, [int(k["point"], 16) for k in ks], [int(k["value"], 16) for k in ks], prfs,
                              [None if k["random_v"] is None else int(k["random_v"], 16) for k in ks], ctx=ctx)
    assert list(res) == [k["expect"] for k in ks]
