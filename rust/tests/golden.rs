//! Pins the repository's oracle and golden files to the REFERENCE crate and the crates its path is made of
//! (pairing 0.14.2, ark-* 0.2.0, ark-poly-commit 0.2.0).  SOURCE ONLY: never compiled or run in the build image (no
//! Rust toolchain, no network); one `cargo test` on any machine with cargo turns the "parity unpinned" statement
//! of DESIGN.md section 0 into a green or red answer.  The tests that use `kzg_setup_powersoftau_ref` /
//! arkworks / pairing only (all but the last two) need no GPU and no libptau_b200.so at run time.
//!
//! What is compared (files under ../tests/golden, produced by tools/make_golden.py from oracle/ptau_oracle.py):
//!   * n8_powersoftau.bin (compressed response, N = 8)  --pairing into_affine_unchecked / into_uncompressed-->
//!     n8_powersoftau_uncompressed.bin           [what Accumulator::deserialize(Compressed, No) + serialize(No) do per
//!                                                point; the powersoftau crate itself hard-codes 2^21 powers]
//!   * n8_powersoftau_uncompressed.bin  --reference read_g1 / read_g2 + serialize_uncompressed-->
//!     n8_kzg_setup_kgz.bin, n8_kzg_setup_fastkgz.bin (sections in the order of preprocess-kgz.rs:140-153, :186-194
//!     and preprocess-fastkgz.rs:141-159, :192-208)
//!   * n8_kzg_setup_*.bin  --deserialize_unchecked-->  n8_load_*_g1.bin / _g2.bin (in-memory Montgomery limbs), with
//!     the 576-byte tail through `VerifierKey::deserialize_unchecked` (src/lib.rs:191-192)
//!   * edge_cases.json: every malformed / boundary record with the status the oracle expects in the three check modes;
//!     `read` = what read_g1/read_g2 (ark 0.2 deserialize_uncompressed) answers, `nocheck` = deserialize_unchecked
//!     resp. pairing's into_affine_unchecked.
//!   * n8_challenge.bin -> n8_contribution.bin: a contribution with fixed secrets, checked with the `powersoftau`
//!     crate's hash_to_g2 and PublicKey::deserialize and pairing 0.14.2's pairing (contribution_matches_powersoftau_crate)
//! Each [dagger] assumption of SURVEY.md 8a-3/5/6/7/9 is named at the assertion that would flip if it were wrong;
//! tests/test_dagger_assumptions.py holds the same list on the oracle side.
use ark_bls12_381::Bls12_381;
use ark_ec::PairingEngine;
use ark_poly_commit::kzg10::VerifierKey;
use ark_serialize::{CanonicalDeserialize, CanonicalSerialize};
use kzg_setup_powersoftau_ref as reference;
use pairing::bls12_381::{G1Compressed, G1Uncompressed, G2Compressed, G2Uncompressed};
use pairing::{CurveAffine, EncodedPoint};
use std::fs::File;
use std::io::{BufReader, Write};

type ArkG1Affine = <ark_ec::bls12::Bls12<ark_bls12_381::Parameters> as PairingEngine>::G1Affine;
type ArkG2Affine = <ark_ec::bls12::Bls12<ark_bls12_381::Parameters> as PairingEngine>::G2Affine;

const N: usize = 8;

fn golden(name: &str) -> Vec<u8> {
    std::fs::read(format!("{}/../tests/golden/{}", env!("CARGO_MANIFEST_DIR"), name)).unwrap()
}

/// read_g1 / read_g2 take `&mut BufReader<File>`: the bytes go through a temporary file.
fn reader_over(bytes: &[u8], tag: &str) -> BufReader<File> {
    let path = std::env::temp_dir().join(format!("ptau_golden_{}_{}", std::process::id(), tag));
    File::create(&path).unwrap().write_all(bytes).unwrap();
    BufReader::new(File::open(&path).unwrap())
}

fn g1_limbs(p: &ArkG1Affine) -> Vec<u8> {
    let mut r = Vec::new();
    for f in [&p.x, &p.y].iter() {
        for l in (f.0).0.iter() {
            r.extend_from_slice(&l.to_le_bytes());
        }
    }
    r.extend_from_slice(&[p.infinity as u8, 0, 0, 0, 0, 0, 0, 0]);
    r
}

fn g2_limbs(p: &ArkG2Affine) -> Vec<u8> {
    let mut r = Vec::new();
    for f in [&p.x.c0, &p.x.c1, &p.y.c0, &p.y.c1].iter() {
        for l in (f.0).0.iter() {
            r.extend_from_slice(&l.to_le_bytes());
        }
    }
    r.extend_from_slice(&[p.infinity as u8, 0, 0, 0, 0, 0, 0, 0]);
    r
}

/// [dagger 8a-3] zcash compressed encoding, sign choice ("largest": Fq2 ordered by c1 then c0) and the
/// uncompressed layout x.c1|x.c0|y.c1|y.c0 -- everything the oracle's decompression restates.
#[test]
fn decompression_matches_pairing_crate() {
    let resp = golden("n8_powersoftau.bin");
    let want = golden("n8_powersoftau_uncompressed.bin");
    let mut off = 64; // challenge hash
    let mut out = Vec::new();
    let sections: [(bool, usize); 5] = [(true, 2 * N - 1), (false, N), (true, N), (true, N), (false, 1)];
    for (is_g1, count) in sections.iter() {
        for _ in 0..*count {
            if *is_g1 {
                let mut c = G1Compressed::empty();
                c.as_mut().copy_from_slice(&resp[off..off + 48]);
                off += 48;
                out.extend_from_slice(c.into_affine_unchecked().unwrap().into_uncompressed().as_ref());
            } else {
                let mut c = G2Compressed::empty();
                c.as_mut().copy_from_slice(&resp[off..off + 96]);
                off += 96;
                out.extend_from_slice(c.into_affine_unchecked().unwrap().into_uncompressed().as_ref());
            }
        }
    }
    assert_eq!(out, want, "oracle decompression differs from pairing 0.14.2");
}

/// The reference's own read_g1 / read_g2 over the uncompressed golden file, re-serialized the way its main() does:
/// must reproduce both golden `kzg_setup` files byte for byte.
/// [dagger 8a-5] serialize_uncompressed layout (x LE | y LE, G2 c0 then c1); [dagger 8a-9] VerifierKey written as
/// g, gamma_g, h, beta_h = 576 bytes; [dagger 8a-7] subgroup check accepts these points.
#[test]
fn reference_read_and_serialize_reproduce_golden_setups() {
    let unc = golden("n8_powersoftau_uncompressed.bin");
    let mut rd = reader_over(&unc, "unc");
    let tau_g1: Vec<ArkG1Affine> = (0..2 * N - 1).map(|_| reference::read_g1(&mut rd).unwrap()).collect();
    let tau_g2: Vec<ArkG2Affine> = (0..N).map(|_| reference::read_g2(&mut rd).unwrap()).collect();
    let alpha_g1: Vec<ArkG1Affine> = (0..N).map(|_| reference::read_g1(&mut rd).unwrap()).collect();
    let beta_g1: Vec<ArkG1Affine> = (0..N).map(|_| reference::read_g1(&mut rd).unwrap()).collect();
    assert_eq!(beta_g1.len(), N);

    // preprocess-kgz.rs:186-194
    let mut kgz = Vec::new();
    for g in tau_g1.iter().chain(alpha_g1.iter()) {
        g.serialize_uncompressed(&mut kgz).unwrap();
    }
    let vk = VerifierKey::<Bls12_381> {
        g: tau_g1[0],
        gamma_g: alpha_g1[0],
        h: tau_g2[0],
        beta_h: tau_g2[1],
        prepared_h: tau_g2[0].into(),
        prepared_beta_h: tau_g2[1].into(),
    };
    vk.serialize_uncompressed(&mut kgz).unwrap();
    assert_eq!(kgz, golden("n8_kzg_setup_kgz.bin"));

    // preprocess-fastkgz.rs:192-208
    let mut fast = Vec::new();
    for g in tau_g1.iter().chain(alpha_g1.iter()) {
        g.serialize_uncompressed(&mut fast).unwrap();
    }
    tau_g2[0].serialize_uncompressed(&mut fast).unwrap();
    tau_g2[1].serialize_uncompressed(&mut fast).unwrap();
    for p in tau_g2.iter() {
        p.serialize_uncompressed(&mut fast).unwrap();
    }
    assert_eq!(fast, golden("n8_kzg_setup_fastkgz.bin"));
}

/// [dagger 8a-6] deserialize_unchecked reads the uncompressed form and yields these in-memory limbs;
/// [dagger 8a-9] VerifierKey::deserialize_unchecked consumes exactly the 576-byte tail (src/lib.rs:191-192).
#[test]
fn unchecked_loads_match_golden_limbs() {
    let kgz = golden("n8_kzg_setup_kgz.bin");
    let want_g1 = golden("n8_load_kgz_g1.bin");
    let want_g2 = golden("n8_load_kgz_g2.bin");
    let mut cur = &kgz[..];
    let mut got_g1 = Vec::new();
    for _ in 0..(3 * N - 1) {
        got_g1.extend(g1_limbs(&ArkG1Affine::deserialize_unchecked(&mut cur).unwrap()));
    }
    assert_eq!(cur.len(), 576);
    let vk = VerifierKey::<Bls12_381>::deserialize_unchecked(&mut cur).unwrap();
    assert!(cur.is_empty(), "VerifierKey did not consume the whole tail");
    got_g1.extend(g1_limbs(&vk.g));
    got_g1.extend(g1_limbs(&vk.gamma_g));
    assert_eq!(got_g1, want_g1);
    let mut got_g2 = g2_limbs(&vk.h);
    got_g2.extend(g2_limbs(&vk.beta_h));
    assert_eq!(got_g2, want_g2);

    let fast = golden("n8_kzg_setup_fastkgz.bin");
    let mut cur = &fast[..];
    let mut got_g1 = Vec::new();
    for _ in 0..(3 * N - 1) {
        got_g1.extend(g1_limbs(&ArkG1Affine::deserialize_unchecked(&mut cur).unwrap()));
    }
    let mut got_g2 = Vec::new();
    for _ in 0..(N + 2) {
        got_g2.extend(g2_limbs(&ArkG2Affine::deserialize_unchecked(&mut cur).unwrap()));
    }
    assert!(cur.is_empty());
    assert_eq!(got_g1, golden("n8_load_fastkgz_g1.bin"));
    assert_eq!(got_g2, golden("n8_load_fastkgz_g2.bin"));
}

/// Every record of tests/golden/edge_cases.json against the real primitives.  `read` (zcash-uncompressed records,
/// in_fmt 1): the reference's read_g1 / read_g2 -- [dagger 8a-7] no on-curve check in ark 0.2, infinity / flag bits /
/// non-canonical coordinates rejected.  `nocheck`: in_fmt 3 = deserialize_unchecked -- [dagger 8a-6] x needs empty
/// flags, y's top bits are SWFlags with (1,0) accepted and (1,1) refused; in_fmt 2 = pairing's into_affine_unchecked.
#[test]
fn edge_cases_match_real_primitives() {
    let meta: serde_json::Value = serde_json::from_slice(&golden("edge_cases.json")).unwrap();
    for (i, c) in meta["cases"].as_array().unwrap().iter().enumerate() {
        let group = c["group"].as_i64().unwrap();
        let in_fmt = c["in_fmt"].as_i64().unwrap();
        let rec = hex::decode(c["rec"].as_str().unwrap()).unwrap();
        let desc = c["desc"].as_str().unwrap();
        match in_fmt {
            1 => {
                if let Some(want) = c.get("read").and_then(|v| v.as_i64()) {
                    let ok = if group == 1 {
                        reference::read_g1(&mut reader_over(&rec, &format!("e{}", i))).is_ok()
                    } else {
                        reference::read_g2(&mut reader_over(&rec, &format!("e{}", i))).is_ok()
                    };
                    assert_eq!(ok, want == 0, "case {} ({}): read_g{} disagrees with the oracle", i, desc, group);
                }
            }
            2 => {
                let want = c["nocheck"].as_i64().unwrap();
                let ok = if group == 1 {
                    let mut e = G1Compressed::empty();
                    e.as_mut().copy_from_slice(&rec);
                    e.into_affine_unchecked().is_ok()
                } else {
                    let mut e = G2Compressed::empty();
                    e.as_mut().copy_from_slice(&rec);
                    e.into_affine_unchecked().is_ok()
                };
                assert_eq!(ok, want == 0, "case {} ({}): into_affine_unchecked disagrees with the oracle", i, desc);
            }
            3 => {
                let want = c["nocheck"].as_i64().unwrap();
                let ok = if group == 1 {
                    ArkG1Affine::deserialize_unchecked(&rec[..]).is_ok()
                } else {
                    ArkG2Affine::deserialize_unchecked(&rec[..]).is_ok()
                };
                assert_eq!(ok, want == 0, "case {} ({}): deserialize_unchecked disagrees with the oracle", i, desc);
                if let Some(read) = c.get("read").and_then(|v| v.as_i64()) {
                    let ok = if group == 1 {
                        ArkG1Affine::deserialize_uncompressed(&rec[..]).is_ok()
                    } else {
                        ArkG2Affine::deserialize_uncompressed(&rec[..]).is_ok()
                    };
                    assert_eq!(ok, read == 0, "case {} ({}): deserialize_uncompressed disagrees with the oracle", i, desc);
                }
            }
            _ => unreachable!(),
        }
    }
}

/// pairing's uncompressed encoding of the points the oracle calls zcash-uncompressed is what read_g1 expects:
/// [dagger 8a-1/2] the byte shuffles of src/lib.rs:49-50, :64-76 map it onto ark's x LE | y LE (G2: c0 | c1).
#[test]
fn zcash_uncompressed_layout_is_pairing_layout() {
    let unc = golden("n8_powersoftau_uncompressed.bin");
    let mut e1 = G1Uncompressed::empty();
    e1.as_mut().copy_from_slice(&unc[96..192]); // tau_g1[1]
    let p = e1.into_affine().unwrap();
    assert_eq!(p.into_uncompressed().as_ref(), &unc[96..192]);
    let off = (2 * N - 1) * 96 + 192; // tau_g2[1]
    let mut e2 = G2Uncompressed::empty();
    e2.as_mut().copy_from_slice(&unc[off..off + 192]);
    let q = e2.into_affine().unwrap();
    assert_eq!(q.into_uncompressed().as_ref(), &unc[off..off + 192]);
}

// ---- the shim itself against the reference (these two need libptau_b200.so and a B200) ---------------------------

/// kzg_setup_powersoftau (this crate) and the reference return the same points for the same bytes.
#[test]
#[ignore = "needs a B200 and libptau_b200.so"]
fn shim_read_g1_read_g2_equal_reference() {
    let unc = golden("n8_powersoftau_uncompressed.bin");
    let (mut a, mut b) = (reader_over(&unc, "shim_a"), reader_over(&unc, "shim_b"));
    for _ in 0..(2 * N - 1) {
        assert_eq!(kzg_setup_powersoftau::read_g1(&mut a).unwrap(), reference::read_g1(&mut b).unwrap());
    }
    for _ in 0..N {
        assert_eq!(kzg_setup_powersoftau::read_g2(&mut a).unwrap(), reference::read_g2(&mut b).unwrap());
    }
}

/// G2Prepared line coefficients computed on the GPU equal ark-ec's `G2Prepared::from` (src/lib.rs:223-224).
#[test]
#[ignore = "needs a B200 and libptau_b200.so"]
fn shim_g2_prepare_equals_ark() {
    let unc = golden("n8_powersoftau_uncompressed.bin");
    let mut rd = reader_over(&unc[(2 * N - 1) * 96..], "prep");
    let pts: Vec<ArkG2Affine> = (0..N).map(|_| reference::read_g2(&mut rd).unwrap()).collect();
    let got = kzg_setup_powersoftau::kzg::g2_prepare(&pts);
    for (p, (coeffs, inf)) in pts.iter().zip(got.iter()) {
        let want: <Bls12_381 as PairingEngine>::G2Prepared = (*p).into();
        assert_eq!(want.infinity, *inf);
        assert_eq!(&want.ell_coeffs, coeffs);
    }
}

/// The golden contribution (tests/golden/n8_challenge.bin -> n8_contribution.bin, tools/make_golden.py) against the
/// real `powersoftau` crate and pairing 0.14.2: its prefix is BLAKE2b of the challenge, its public key deserializes
/// with the crate's strict checks, every G2 element is [x] hash_to_g2(BLAKE2b(personalization || digest || g1_s ||
/// g1_s_x)) computed by the crate's own `hash_to_g2` (rand 0.4 ChaChaRng, `G2::rand`), the proofs of knowledge hold
/// by pairing, and the transformed accumulator is the challenge's times the known secrets.  This is what pins the
/// recalled rand 0.4 / `Fq::rand` / `G2::rand` behaviour of csrc/contribute.cuh; the crate's `verify_transform` is
/// fixed at 2^21 powers and cannot take N = 8.
#[test]
fn contribution_matches_powersoftau_crate() {
    use pairing::bls12_381::{Fr, FrRepr, G1Affine, G2Affine};
    use pairing::{CurveProjective, Field, PrimeField};
    // tau, alpha, beta, s_tau, s_alpha, s_beta: tests/contribute_oracle.py GOLDEN_SECRETS
    const SECRETS: [u64; 6] = [0x2A5F3C91D7E04B86, 0x6C1E9A74B3F2D058, 0x1F8B6E3D5A7C9042, 0x3B7D1F5E9C2A6084,
                               0x5E2C8A4F1D6B3097, 0x7A4E2C6F8B1D5039];
    let fr = |v: u64| Fr::from_repr(FrRepr([v, 0, 0, 0])).unwrap();
    let chal = golden("n8_challenge.bin");
    let resp = golden("n8_contribution.bin");
    let digest = blake2b_simd::blake2b(&chal);
    assert_eq!(&resp[..64], digest.as_bytes());
    let pk = &resp[resp.len() - powersoftau::PUBLIC_KEY_SIZE..];
    powersoftau::PublicKey::deserialize(&mut &pk[..]).expect("strict public key");
    let g1 = |i: usize| {
        let mut e = G1Uncompressed::empty();
        e.as_mut().copy_from_slice(&pk[96 * i..96 * (i + 1)]);
        e.into_affine().unwrap()
    };
    let g2 = |i: usize| {
        let mut e = G2Uncompressed::empty();
        e.as_mut().copy_from_slice(&pk[576 + 192 * i..576 + 192 * (i + 1)]);
        e.into_affine().unwrap()
    };
    for i in 0..3 {
        let (s, sx, x_g2s) = (g1(2 * i), g1(2 * i + 1), g2(i));
        let (x, sv) = (fr(SECRETS[i]), fr(SECRETS[3 + i]));
        assert_eq!(s, G1Affine::one().mul(sv).into_affine());
        assert_eq!(sx, s.mul(x).into_affine());
        let mut h = blake2b_simd::State::new();
        h.update(&[i as u8]);
        h.update(digest.as_bytes());
        h.update(s.into_uncompressed().as_ref());
        h.update(sx.into_uncompressed().as_ref());
        let g2_s: G2Affine = powersoftau::hash_to_g2(h.finalize().as_bytes()).into_affine();
        assert_eq!(x_g2s, g2_s.mul(x).into_affine(), "hash_to_g2 of key pair {}", i);
        assert_eq!(s.pairing_with(&x_g2s), sx.pairing_with(&g2_s), "proof of knowledge {}", i);
    }
    // the body: tau_g1[i] * tau^i ... beta_g2 * beta, section by section (decompressed with pairing's own code)
    let (tau, alpha, beta) = (fr(SECRETS[0]), fr(SECRETS[1]), fr(SECRETS[2]));
    let (mut off_u, mut off_c) = (64usize, 64usize);
    for (sec, count) in [(0usize, 2 * N - 1), (1, N), (2, N), (3, N), (4, 1)].iter() {
        let mut t = Fr::one();
        for _ in 0..*count {
            let mut k = t;
            if *sec == 2 {
                k.mul_assign(&alpha);
            } else if *sec >= 3 {
                k.mul_assign(&beta);
            }
            if *sec == 1 || *sec == 4 {
                let mut u = G2Uncompressed::empty();
                u.as_mut().copy_from_slice(&chal[off_u..off_u + 192]);
                let mut c = G2Compressed::empty();
                c.as_mut().copy_from_slice(&resp[off_c..off_c + 96]);
                assert_eq!(c.into_affine().unwrap(), u.into_affine().unwrap().mul(k).into_affine());
                off_u += 192;
                off_c += 96;
            } else {
                let mut u = G1Uncompressed::empty();
                u.as_mut().copy_from_slice(&chal[off_u..off_u + 96]);
                let mut c = G1Compressed::empty();
                c.as_mut().copy_from_slice(&resp[off_c..off_c + 48]);
                assert_eq!(c.into_affine().unwrap(), u.into_affine().unwrap().mul(k).into_affine());
                off_u += 96;
                off_c += 48;
            }
            t.mul_assign(&tau);
        }
    }
    assert_eq!(off_c + powersoftau::PUBLIC_KEY_SIZE, resp.len());
}
