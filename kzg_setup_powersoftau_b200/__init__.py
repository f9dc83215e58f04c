"""kzg_setup_powersoftau_b200 -- host-side mirror of the `kzg_setup_powersoftau`
crate's public surface on top of libptau_b200.so (CUDA, sm_100a).

Same names, argument meaning and error behaviour as the reference
(/root/reference/src/lib.rs): KZG_SETUP_FILE, read_g1, read_g2, load_phase1,
download_kzg_setup, download_fastkzg_setup, load_kzg_setup, load_fastkzg_setup,
plus the two binaries' main() as preprocess_kgz / preprocess_fastkgz
(/root/reference/src/bin/*.rs).  Sizes that the reference hard-codes to 2^21
powers (src/lib.rs:23-24) are run-time parameters defaulting to 21.

Everything that touches a curve point goes through the C ABI; this package holds
no arithmetic.  It raises if the CUDA library is missing or no B200 is present.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
from dataclasses import dataclass, field
from typing import Dict, Optional, Tuple

import numpy as np

from . import _ffi
from ._ffi import (  # noqa: F401  (re-exported constants)
    BAD_FLAGS, BAD_INFINITY, BAD_NAMES, BAD_NON_CANONICAL, BAD_NOT_IN_SUBGROUP, BAD_NOT_ON_CURVE,
    CHECK_ON_CURVE, CHECK_REJECT_INFINITY, CHECK_SUBGROUP, CHECKS_DECOMPRESS, CHECKS_LOAD, CHECKS_READ,
    CHECKS_STRICT, FMT_ARK_MONT_LIMBS, FMT_ARK_UNCOMPRESSED, FMT_ZCASH_COMPRESSED, FMT_ZCASH_UNCOMPRESSED,
    G1, G2, STATUS_NONE, VARIANT_FASTKGZ, VARIANT_KGZ,
    BAD_NOT_POWERS, POWERS_FASTKGZ, POWERS_KGZ, POWERS_RESPONSE, REL_ALPHA_G1, REL_BETA_G1, REL_BETA_G2,
    REL_GENERATORS, REL_KEY, REL_NAMES, REL_TAU_G1, REL_TAU_G2,
    REL_HASH, REL_POK_TAU, REL_POK_ALPHA, REL_POK_BETA, REL_CHAIN_TAU, REL_CHAIN_ALPHA, REL_CHAIN_BETA, REL_CHAIN_BETA_G2,
)

# ---- reference constants (src/lib.rs:20-28, src/bin/preprocess-kgz.rs:18-23) --
KZG_SETUP_FILE = "kzg_setup"
KZG_SETUP_FILE_DIGEST = (
    "87932f626204ab9a5d4be67ef2ee479471baf942364ada2f89840a2afec8925911fb88cb77024e66d759b4970b25cf2a"
    "7b03d1fc8c15768e021220b8ba21efcf"
)
FASTKZG_SETUP_FILE_DIGEST = (
    "d177841ad145c0d526e56a8d2cde473f09e85944f5c5d6b72d8063e4a199f8a6fca0b0f6ee91ef79df48518b5edd8165"
    "bbdecf0fe4eb0d29809032878f8b17ce"
)
POWERSOFTAU_DIGEST = (
    "88dc1dc6914e44568e8511eace177e6ecd9da9a9bd8f67e4c0c9f215b517db4d1d54a755d051978dbb85ef947918193c"
    "93cd4cf4c99c0dc5a767d4eeb10047a4"
)
KZG_SETUP_URL = "https://heliax-ferveo-v1.s3-eu-west-1.amazonaws.com/ferveo-dkg-kzg-setup"
FASTKZG_SETUP_URL = "https://heliax-ferveo-v1.s3-eu-west-1.amazonaws.com/ferveo-dkg-fastkzg-setup"
POWERSOFTAU_FILE = "powersoftau"
POWERSOFTAU_UNCOMPRESSED_FILE = "powersoftau_uncompressed"
DEFAULT_LOG2_POWERS = 21  # TAU_POWERS_LENGTH = 1 << 21

SECTION_NAMES = ("tau_powers_g1", "tau_powers_g2", "alpha_tau_powers_g1", "beta_tau_powers_g1", "beta_g2")


class PtauError(Exception):
    """Data or runtime error from the C ABI.  The reference panics at this point
    (`unwrap()` at src/bin/preprocess-kgz.rs:142, src/lib.rs:180, ...)."""

    def __init__(self, code: int, index: Optional[int] = None, section: Optional[int] = None, detail: str = "",
                 relation: Optional[int] = None):
        self.code = code
        self.kind = BAD_NAMES.get(code)
        self.index = index
        self.section = section
        self.relation = relation  # verify_powers: the lowest failing relation (REL_*)
        msg = _ffi.strerror(code)
        if index is not None:
            msg += " at point %d" % index
        if section is not None and 0 <= section < len(SECTION_NAMES):
            msg += " of section %s" % SECTION_NAMES[section]
        if relation is not None and 0 <= relation < len(REL_NAMES):
            msg += " (relation %s)" % REL_NAMES[relation]
        if detail:
            msg += " (%s)" % detail
        super().__init__(msg)


# ---- pinned host buffers ---------------------------------------------------------
class PinnedBuffer:
    """Page-locked host memory from ptau_host_alloc, exposed as a numpy u8 array.  The
    memory is returned with ptau_host_free when the last numpy view of it is gone (the
    finalizer hangs on the ctypes object every view keeps alive), so slices handed to
    callers stay valid after the PinnedBuffer itself is dropped."""

    def __init__(self, nbytes: int):
        import weakref

        self.nbytes = int(nbytes)
        L = _ffi.lib()
        ptr = L.ptau_host_alloc(max(self.nbytes, 1))
        if not ptr:
            raise PtauError(_ffi.ERR_NOMEM, detail="ptau_host_alloc(%d)" % nbytes)
        self._ptr = ptr
        cobj = (C.c_uint8 * max(self.nbytes, 1)).from_address(ptr)
        weakref.finalize(cobj, L.ptau_host_free, ptr)
        self.array = np.ctypeslib.as_array(cobj)[: self.nbytes]

    @property
    def ptr(self) -> int:
        return self._ptr

    def free(self):
        """Drop this object's reference; the memory goes away with the last view."""
        self.array = None
        self._ptr = None


def _as_u8(data) -> np.ndarray:
    if isinstance(data, PinnedBuffer):
        return data.array
    if isinstance(data, np.ndarray):
        a = data.view(np.uint8).reshape(-1) if data.dtype != np.uint8 or data.ndim != 1 else data
        return np.ascontiguousarray(a)
    return np.frombuffer(bytes(data) if not isinstance(data, (bytes, bytearray, memoryview)) else data, dtype=np.uint8)


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


# ---- context ---------------------------------------------------------------------
class Context:
    """Owns per-GPU streams and device double buffers (ptau_create / ptau_destroy)."""

    def __init__(self, n_gpus: int = 1, device_ids=None, chunk_points: int = 0):
        L = _ffi.lib()
        h = C.c_void_p()
        ids = None
        if device_ids is not None:
            ids = (C.c_int * len(device_ids))(*device_ids)
            n_gpus = len(device_ids)
        rc = L.ptau_create(C.byref(h), n_gpus, ids, chunk_points)
        if rc != 0:
            raise PtauError(rc, detail="ptau_create(n_gpus=%d): a CUDA sm_100 device is required" % n_gpus)
        self._h = h
        self.n_gpus = n_gpus

    def close(self):
        if getattr(self, "_h", None):
            _ffi.lib().ptau_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _raise(self, rc, index=None, section=None):
        detail = ""
        if rc == _ffi.ERR_CUDA:
            detail = _ffi.lib().ptau_last_error(self._h).decode()
        raise PtauError(rc, index, section, detail)

    def timing(self) -> dict:
        t = _ffi.Timing()
        _ffi.lib().ptau_last_timing(self._h, C.byref(t))
        n = t.n_gpus
        return {
            "n_gpus": n,
            "wall_ms": t.wall_ms,
            "gpu_ms": list(t.gpu_ms)[:n],
            "kernel_ms": list(t.kernel_ms)[:n],
            "h2d_bytes": list(t.h2d_bytes)[:n],
            "d2h_bytes": list(t.d2h_bytes)[:n],
            "kernel_launches": int(t.kernel_launches),
        }

    # -- the per-point path --
    def convert(self, group: int, in_fmt: int, data, out_fmt: int, checks: int = CHECKS_STRICT, out=None) -> np.ndarray:
        """ptau_convert on host buffers.  Returns the output bytes as a numpy u8
        array (or fills `out`).  Raises PtauError with the lowest failing index."""
        L = _ffi.lib()
        src = _as_u8(data)
        ri = L.ptau_record_size(group, in_fmt)
        ro = L.ptau_record_size(group, out_fmt)
        if ri == 0 or ro == 0 or src.size % ri:
            raise PtauError(_ffi.ERR_SIZE, detail="input is not a whole number of %d-byte records" % ri)
        n = src.size // ri
        dst = _as_u8(out) if out is not None else np.empty(n * ro, dtype=np.uint8)
        if dst.size != n * ro:
            raise PtauError(_ffi.ERR_SIZE, detail="output buffer must hold %d bytes" % (n * ro))
        bad_i, bad_k = C.c_uint64(0), C.c_int(0)
        rc = L.ptau_convert(self._h, group, in_fmt, _ptr(src), out_fmt, _ptr(dst), n, checks, C.byref(bad_i),
                            C.byref(bad_k))
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None)
        return dst

    def convert_device(self, group, in_fmt, d_in: int, out_fmt, d_out: int, n_points: int, checks: int,
                       d_status: int, base_index: int = 0, stream: int = 0, gpu: int = 0):
        """ptau_convert_device: one asynchronous kernel launch on device pointers."""
        rc = _ffi.lib().ptau_convert_device(self._h, gpu, group, in_fmt, d_in, out_fmt, d_out, n_points, checks,
                                            base_index, d_status, stream)
        if rc != 0:
            self._raise(rc)

    def generate(self, group: int, fmt: int, scalar0: int, step: int, first: int, n_points: int, out=None) -> np.ndarray:
        """Synthetic section: points [scalar0 * step^(first+i)] G, i < n_points."""
        L = _ffi.lib()
        ro = L.ptau_record_size(group, fmt)
        dst = _as_u8(out) if out is not None else np.empty(n_points * ro, dtype=np.uint8)
        rc = L.ptau_generate(self._h, group, fmt, int(scalar0).to_bytes(32, "little"),
                             int(step).to_bytes(32, "little"), first, n_points, _ptr(dst))
        if rc != 0:
            self._raise(rc)
        return dst

    def generate_device(self, group, fmt, scalar0: int, step: int, first: int, n_points: int, d_out: int,
                        stream: int = 0, gpu: int = 0):
        rc = _ffi.lib().ptau_generate_device(self._h, gpu, group, fmt, int(scalar0).to_bytes(32, "little"),
                                             int(step).to_bytes(32, "little"), first, n_points, d_out, stream)
        if rc != 0:
            self._raise(rc)

    # -- whole-file pipelines (memory to memory) --
    def preprocess(self, variant: int, response, n_powers: int, checks: int = CHECKS_STRICT,
                   emit_uncompressed: bool = False, out=None, uncompressed_out=None):
        L = _ffi.lib()
        src = _as_u8(response)
        setup = _as_u8(out) if out is not None else np.empty(L.ptau_setup_size(variant, n_powers), dtype=np.uint8)
        unc = None
        if emit_uncompressed or uncompressed_out is not None:
            unc = _as_u8(uncompressed_out) if uncompressed_out is not None else np.empty(
                L.ptau_uncompressed_size(n_powers), dtype=np.uint8)
        bad_i, bad_k, bad_s = C.c_uint64(0), C.c_int(0), C.c_int(-1)
        rc = L.ptau_preprocess(self._h, variant, _ptr(src), src.size, n_powers, _ptr(setup), setup.size,
                               _ptr(unc) if unc is not None else None, unc.size if unc is not None else 0, checks,
                               C.byref(bad_i), C.byref(bad_k), C.byref(bad_s))
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None, bad_s.value if rc > 0 else None)
        return (setup, unc) if unc is not None else setup

    def preprocess_uncompressed(self, variant: int, uncompressed, n_powers: int, checks: int = CHECKS_STRICT, out=None):
        L = _ffi.lib()
        src = _as_u8(uncompressed)
        setup = _as_u8(out) if out is not None else np.empty(L.ptau_setup_size(variant, n_powers), dtype=np.uint8)
        bad_i, bad_k, bad_s = C.c_uint64(0), C.c_int(0), C.c_int(-1)
        rc = L.ptau_preprocess_uncompressed(self._h, variant, _ptr(src), src.size, n_powers, _ptr(setup), setup.size,
                                            checks, C.byref(bad_i), C.byref(bad_k), C.byref(bad_s))
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None, bad_s.value if rc > 0 else None)
        return setup

    def load_setup(self, variant: int, setup, n_powers: int, checks: int = CHECKS_LOAD):
        """-> (g1_records u8[n_g1,104], g2_records u8[n_g2,200]) in file order."""
        L = _ffi.lib()
        src = _as_u8(setup)
        fast = variant == VARIANT_FASTKGZ
        n_g1 = 3 * n_powers - 1 + (0 if fast else 2)
        n_g2 = n_powers + 2 if fast else 2
        g1 = np.empty(n_g1 * 104, dtype=np.uint8)
        g2 = np.empty(n_g2 * 200, dtype=np.uint8)
        bad_i, bad_k = C.c_uint64(0), C.c_int(0)
        rc = L.ptau_load_setup(self._h, variant, _ptr(src), src.size, n_powers, checks, _ptr(g1), g1.size, _ptr(g2),
                               g2.size, C.byref(bad_i), C.byref(bad_k))
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None)
        return g1.reshape(n_g1, 104), g2.reshape(n_g2, 200)

    def load_phase1(self, data, m: int, checks: int = CHECKS_READ):
        L = _ffi.lib()
        src = _as_u8(data)
        g1 = np.empty((2 + 3 * m) * 104, dtype=np.uint8)
        g2 = np.empty((1 + m) * 200, dtype=np.uint8)
        bad_i, bad_k = C.c_uint64(0), C.c_int(0)
        rc = L.ptau_load_phase1(self._h, _ptr(src), src.size, m, checks, _ptr(g1), g1.size, _ptr(g2), g2.size,
                                C.byref(bad_i), C.byref(bad_k))
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None)
        return g1.reshape(-1, 104), g2.reshape(-1, 200)

    def verify_powers(self, kind: int, data, n_powers: int, seed: Optional[bytes] = None, combos: bool = False):
        """ptau_verify_powers: are the points of a response (POWERS_RESPONSE) or kzg_setup (POWERS_KGZ /
        POWERS_FASTKGZ) powers of one tau?  Raises PtauError: a bad point as ptau_preprocess / ptau_load_setup
        report it, or BAD_NOT_POWERS with `.relation`.  seed: 32 bytes (None: random).  combos=True returns the
        8 x 200-byte combinations (A_k, B_k of ratio relation k in slots 2k-2, 2k-1), else None."""
        src = _as_u8(data)
        if seed is not None and len(seed) != 32:
            raise PtauError(_ffi.ERR_ARG, detail="seed must be 32 bytes")
        out = np.zeros((8, 200), dtype=np.uint8) if combos else None
        bad_i, bad_k, bad_s, bad_r = C.c_uint64(0), C.c_int(0), C.c_int(-1), C.c_int(-1)
        rc = _ffi.lib().ptau_verify_powers(self._h, kind, _ptr(src), src.size, n_powers,
                                           bytes(seed) if seed is not None else None, C.byref(bad_i), C.byref(bad_k),
                                           C.byref(bad_s), C.byref(bad_r), _ptr(out) if combos else None)
        if rc == BAD_NOT_POWERS:
            raise PtauError(rc, relation=bad_r.value)
        if rc != 0:
            section = bad_s.value if (rc > 0 and kind == POWERS_RESPONSE) else None
            self._raise(rc, bad_i.value if rc > 0 else None, section)
        return out

    def contribute(self, challenge, n_powers: int, secrets=None, checks: int = CHECKS_STRICT, out=None) -> np.ndarray:
        """ptau_contribute: the response of powersoftau `compute` on a challenge (64-byte hash + uncompressed
        accumulator).  secrets: None (drawn from the OS) or (tau, alpha, beta, s_tau, s_alpha, s_beta) as ints in
        (0, r), or their 192 bytes (6 x 32, little-endian).  The library wipes its own copies of the secrets before it
        returns; the Python objects passed in (and the bytes built from them here) are not wiped.  Returns the response
        bytes (or fills `out`).  A bad
        challenge point raises PtauError with its section and index, as preprocess reports it."""
        L = _ffi.lib()
        src = _as_u8(challenge)
        sec = None
        if secrets is not None:
            sec = bytes(secrets) if isinstance(secrets, (bytes, bytearray)) else b"".join(
                int(v).to_bytes(32, "little") if 0 <= int(v) < (1 << 256) else b"" for v in secrets)
            if len(sec) != 192:
                raise PtauError(_ffi.ERR_ARG, detail="secrets must be six scalars")
        size = L.ptau_response_size(n_powers)
        dst = _as_u8(out) if out is not None else np.empty(size, dtype=np.uint8)
        bad_i, bad_k, bad_s = C.c_uint64(0), C.c_int(0), C.c_int(-1)
        rc = L.ptau_contribute(self._h, _ptr(src), src.size, n_powers, sec, checks, _ptr(dst), dst.size,
                               C.byref(bad_i), C.byref(bad_k), C.byref(bad_s))
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None, bad_s.value if rc > 0 else None)
        return dst

    def verify_contribution(self, challenge, response, n_powers: int, seed: Optional[bytes] = None) -> None:
        """ptau_verify_contribution (powersoftau verify_transform).  challenge None: the response's own relations only
        (public key and powers).  Raises PtauError: a bad point with .section (0-4 response, 5 public key, 6 + s the
        challenge's section s) and .index, or BAD_NOT_POWERS with .relation."""
        resp = _as_u8(response)
        chal = _as_u8(challenge) if challenge is not None else None
        if seed is not None and len(seed) != 32:
            raise PtauError(_ffi.ERR_ARG, detail="seed must be 32 bytes")
        bad_i, bad_k, bad_s, bad_r = C.c_uint64(0), C.c_int(0), C.c_int(-1), C.c_int(-1)
        rc = _ffi.lib().ptau_verify_contribution(self._h, _ptr(chal) if chal is not None else None,
                                                 chal.size if chal is not None else 0, _ptr(resp), resp.size, n_powers,
                                                 bytes(seed) if seed is not None else None, C.byref(bad_i),
                                                 C.byref(bad_k), C.byref(bad_s), C.byref(bad_r))
        if rc == BAD_NOT_POWERS:
            raise PtauError(rc, relation=bad_r.value)
        if rc != 0:
            self._raise(rc, bad_i.value if rc > 0 else None, bad_s.value if rc > 0 else None)

    def msm_g2(self, points, scalars) -> np.ndarray:
        """sum_i scalars[i] * points[i] over G2 (ptau_msm_g2): points [n, 200] Montgomery-limb records, scalars ints
        (taken mod r) or a [n, 32] u8 array of little-endian scalars < r.  Returns one 200-byte record."""
        pts = np.ascontiguousarray(np.asarray(points, dtype=np.uint8).reshape(-1, 200))
        sc = KZG10._scalars(scalars)
        n = sc.size // 32
        if pts.shape[0] < n:
            raise PtauError(_ffi.ERR_ARG, detail="more scalars than points")
        out = np.zeros(200, dtype=np.uint8)
        rc = _ffi.lib().ptau_msm_g2(self._h, _ptr(pts) if n else None, _ptr(sc) if n else None, n, _ptr(out))
        if rc != 0:
            self._raise(rc)
        return out

    def microbench(self, kind: int, iters: int, gpu: int = 0) -> Tuple[float, float]:
        ms, ops = C.c_double(0), C.c_double(0)
        rc = _ffi.lib().ptau_microbench(self._h, gpu, kind, iters, C.byref(ms), C.byref(ops))
        if rc != 0:
            self._raise(rc)
        return ms.value, ops.value


R_ORDER = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001  # Fr modulus
# 7^((r - 1) / 2^32) mod r: a root of unity of order 2^32 (ark-bls12-381 Fr TWO_ADIC_ROOT_OF_UNITY, GENERATOR 7)
FR_ROOT_OF_UNITY = 0x16A2A19EDFE81F20D09B681922C813B4B63683508C2280B93829971F439F0D2B


def coset_points(log2_k: int, h: int) -> list:
    """The points h omega_k^m, m < k = 2^log2_k, of the coset KZG10.open_cosets opens, in its order."""
    w = pow(FR_ROOT_OF_UNITY, 1 << (32 - log2_k), R_ORDER)
    pts, x = [], int(h) % R_ORDER
    for _ in range(1 << log2_k):
        pts.append(x)
        x = x * w % R_ORDER
    return pts


class KZG10:
    """SURVEY 8f-4: ark-poly-commit 0.2 `KZG10` on the GPU (the reference's consumer usage,
    src/lib.rs:266-286): `commit` / `open` (bucket MSM), `check` / `batch_check` (pairings).
    Polynomials are lists of coefficients (ints mod r, low degree first).  Hiding: ark draws a
    random polynomial of degree `hiding_bound`; here the caller passes its coefficients
    (`blinding`) so results are reproducible, and `batch_check` takes its randomizers as an
    argument for the same reason (ark draws u128s from the caller's rng)."""

    @staticmethod
    def _msm(ctx, pairs) -> np.ndarray:
        if any(isinstance(p, ResidentPoints) for p, _ in pairs):
            # device-resident operands: one MSM per (points, scalars) pair, partial results added by a two-term MSM
            parts = []
            for p, c in pairs:
                if not len(c):
                    continue
                if isinstance(p, ResidentPoints):
                    parts.append(p.msm(c))
                else:
                    parts.append(KZG10._msm(ctx, [(p, c)]))
            if not parts:
                return KZG10._msm(ctx, [])
            if len(parts) == 1:
                return parts[0]
            return KZG10._msm(ctx, [(np.stack(parts), [1] * len(parts))])
        pts = np.concatenate([np.ascontiguousarray(p[: len(c)]).reshape(-1) for p, c in pairs if len(c)] or
                             [np.zeros(0, dtype=np.uint8)])
        sc = b"".join((int(v) % R_ORDER).to_bytes(32, "little") for _, c in pairs for v in c)
        n = len(sc) // 32
        out = np.zeros(104, dtype=np.uint8)
        scb = np.frombuffer(sc, dtype=np.uint8) if n else np.zeros(0, dtype=np.uint8)
        rc = _ffi.lib().ptau_kzg_commit(ctx._h, _ptr(pts) if n else None, _ptr(scb) if n else None, n, _ptr(out))
        if rc != 0:
            ctx._raise(rc)
        return out

    @staticmethod
    def commit(powers: "Powers", coeffs, blinding=None, ctx: Optional["Context"] = None) -> np.ndarray:
        """KZG10::commit: sum c_i powers_of_g[i] (+ sum b_i powers_of_gamma_g[i] when hiding).
        Returns the commitment as a 104-byte Montgomery-limb record."""
        ctx = ctx or default_context()
        if len(coeffs) > len(powers.powers_of_g) or (blinding and len(blinding) > len(powers.powers_of_gamma_g)):
            raise PtauError(_ffi.ERR_ARG, detail="polynomial degree exceeds the supported degree")  # Error::TooManyCoefficients
        pairs = [(powers.powers_of_g, list(coeffs))]
        if blinding:
            pairs.append((powers.powers_of_gamma_g, list(blinding)))
        return KZG10._msm(ctx, pairs)

    @staticmethod
    def _quotient(coeffs, z):
        """(p(X) - p(z)) / (X - z) by synthetic division; returns (p(z), quotient coefficients).
        Long polynomials go through the library's host routine (ptau_kzg_quotient)."""
        n = len(coeffs)
        if n >= 256:
            cb = np.frombuffer(b"".join((int(c) % R_ORDER).to_bytes(32, "little") for c in coeffs), dtype=np.uint8)
            zb = np.frombuffer((int(z) % R_ORDER).to_bytes(32, "little"), dtype=np.uint8)
            qb = np.zeros((n - 1) * 32, dtype=np.uint8)
            vb = np.zeros(32, dtype=np.uint8)
            rc = _ffi.lib().ptau_kzg_quotient(_ptr(cb), n, _ptr(zb), _ptr(qb), _ptr(vb))
            if rc != 0:
                raise PtauError(rc)
            raw = qb.tobytes()
            return int.from_bytes(vb.tobytes(), "little"), [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(n - 1)]
        q = [0] * max(n - 1, 0)
        carry = 0
        for i in range(n - 1, 0, -1):
            carry = (coeffs[i] + carry * z) % R_ORDER
            q[i - 1] = carry
        value = ((coeffs[0] if n else 0) + carry * z) % R_ORDER
        return value, q

    @staticmethod
    def open(powers: "Powers", coeffs, point: int, blinding=None, ctx: Optional["Context"] = None):
        """KZG10::open: witness commitment w = commit((p - p(z)) / (X - z)) (+ the blinding
        polynomial's witness on powers_of_gamma_g).  Returns (value p(z), proof record,
        random_v = blinding(z) or None).  One point of open_many."""
        values, proofs, random_vs = KZG10.open_many(powers, coeffs, [point], blinding=blinding, ctx=ctx)
        return values[0], proofs[0], None if random_vs is None else random_vs[0]

    @staticmethod
    def open_many(powers: "Powers", coeffs, points, blinding=None, ctx: Optional["Context"] = None):
        """KZG10::open of one polynomial at every point of `points` in one call (ptau_kzg_open): the witness
        polynomials are computed on the GPU and committed to there, point after point, with no host round trip.
        coeffs / points / blinding: ints (taken mod r) or [m, 32] u8 arrays of little-endian scalars < r.  powers:
        Powers of arrays (the first len(coeffs) / len(blinding) powers are uploaded for the call) or
        Powers.to_device().  Returns (values: list of p(z_j), proofs: u8 [k, 104], random_vs: list of b(z_j) or
        None without blinding).  More coefficients than powers raises PtauError (ark: TooManyCoefficients)."""
        ctx = ctx or default_context()
        c, z = KZG10._scalars(coeffs), KZG10._scalars(points)
        b = KZG10._scalars(blinding) if blinding is not None and len(blinding) else None
        n, k, n_b = c.size // 32, z.size // 32, 0 if b is None else b.size // 32

        def resident(pts, m):
            if isinstance(pts, ResidentPoints):
                return pts
            if m > len(pts):
                raise PtauError(_ffi.ERR_ARG, detail="polynomial degree exceeds the supported degree")  # TooManyCoefficients
            return ResidentPoints(ctx, np.asarray(pts)[:m])

        pg = resident(powers.powers_of_g, n)
        gg = resident(powers.powers_of_gamma_g, n_b) if n_b else None
        proofs = np.zeros((k, 104), dtype=np.uint8)
        vals = np.zeros(k * 32, dtype=np.uint8)
        rvs = np.zeros(k * 32, dtype=np.uint8) if n_b else None
        rc = _ffi.lib().ptau_kzg_open(ctx._h, pg._h, gg._h if n_b else None, _ptr(c) if n else None, n,
                                      _ptr(b) if n_b else None, n_b, _ptr(z) if k else None, k,
                                      _ptr(proofs) if k else None, _ptr(vals) if k else None,
                                      _ptr(rvs) if (n_b and k) else None)
        if rc != 0:
            ctx._raise(rc)

        def ints(a):
            raw = a.tobytes()
            return [int.from_bytes(raw[32 * i:32 * i + 32], "little") for i in range(k)]

        return ints(vals), proofs, None if rvs is None else ints(rvs)

    @staticmethod
    def open_cosets(powers: "Powers", coeffs, log2_k: int, shifts, ctx: Optional["Context"] = None):
        """Open one polynomial on whole cosets {h omega_k^m : m < k}, k = 2^log2_k (0 <= log2_k <= 20), one proof per
        shift h (ptau_kzg_open_cosets): the proof commits to q with p = (X^k - h^k) q + r, the values are p at the
        coset's points in natural order (coset_points(log2_k, h)).  powers: Powers of arrays (the first len(coeffs)
        powers_of_g are uploaded for the call) or Powers.to_device().  coeffs / shifts: ints or [m, 32] u8 arrays.
        Returns (values: m lists of k ints, proofs: u8 [m, 104])."""
        ctx = ctx or default_context()
        c, h = KZG10._scalars(coeffs), KZG10._scalars(shifts)
        n, m, k = c.size // 32, h.size // 32, 1 << log2_k if 0 <= log2_k <= 20 else 0
        pg = powers.powers_of_g
        if not isinstance(pg, ResidentPoints):
            if n > len(pg):
                raise PtauError(_ffi.ERR_ARG, detail="polynomial degree exceeds the supported degree")  # TooManyCoefficients
            pg = ResidentPoints(ctx, np.asarray(pg)[:n])
        proofs = np.zeros((m, 104), dtype=np.uint8)
        vals = np.zeros(m * k * 32, dtype=np.uint8)
        rc = _ffi.lib().ptau_kzg_open_cosets(ctx._h, pg._h, _ptr(c) if n else None, n, log2_k, _ptr(h) if m else None, m,
                                             _ptr(proofs) if m else None, _ptr(vals) if m else None)
        if rc != 0:
            ctx._raise(rc)
        raw = vals.tobytes()
        return [[int.from_bytes(raw[32 * (i * k + j):32 * (i * k + j + 1)], "little") for j in range(k)]
                for i in range(m)], proofs

    @staticmethod
    def check_cosets(powers_of_g, h, tau_k_h, log2_k: int, comms, shifts, values, proofs, seed: Optional[bytes] = None,
                     ctx: Optional["Context"] = None) -> bool:
        """Batched check of coset openings with one k = 2^log2_k (ptau_kzg_check_cosets): item i is (comms[i],
        shifts[i], values[i] (k ints or a [k, 32] u8 array), proofs[i]).  powers_of_g: >= k G1 powers as an array
        (its first k are uploaded for the call) or ResidentPoints; h, tau_k_h: 200-byte G2 records h and [tau^k] h
        (fastkgz powers_of_h[0] and powers_of_h[k]).  One random linear combination of the items (127-bit
        randomizers from the 32-byte seed, or from getrandom when None) and one pairing product decide: a false item
        passes with probability at most 2^-127."""
        ctx = ctx or default_context()
        m, k = len(shifts), 1 << log2_k if 0 <= log2_k <= 20 else 0
        if not isinstance(powers_of_g, ResidentPoints):
            if k > len(powers_of_g):
                raise PtauError(_ffi.ERR_ARG, detail="fewer powers than the coset size")
            powers_of_g = ResidentPoints(ctx, np.asarray(powers_of_g)[:k])
        c = np.ascontiguousarray(np.asarray(comms, dtype=np.uint8).reshape(m, 104))
        w = np.ascontiguousarray(np.asarray(proofs, dtype=np.uint8).reshape(m, 104))
        z = KZG10._scalars(shifts)
        if isinstance(values, np.ndarray) and values.dtype == np.uint8:
            v = np.ascontiguousarray(values).reshape(-1)
        else:
            v = KZG10._scalars([x for row in values for x in row])
        if v.size != m * k * 32:
            raise PtauError(_ffi.ERR_ARG, detail="expected k values per item")
        g2 = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.uint8).reshape(-1),
                                                  np.asarray(tau_k_h, dtype=np.uint8).reshape(-1)]))
        if seed is not None and len(seed) != 32:
            raise PtauError(_ffi.ERR_ARG, detail="seed must be 32 bytes")
        ok = np.zeros(1, dtype=np.uint8)
        rc = _ffi.lib().ptau_kzg_check_cosets(ctx._h, powers_of_g._h, _ptr(g2), _ptr(g2[200:]), log2_k,
                                              _ptr(c) if m else None, _ptr(z) if m else None, _ptr(v) if m else None,
                                              _ptr(w) if m else None, m, seed, _ptr(ok))
        if rc != 0:
            ctx._raise(rc)
        return bool(ok[0])

    @staticmethod
    def _scalars(vals) -> np.ndarray:
        if isinstance(vals, np.ndarray) and vals.dtype == np.uint8 and vals.ndim == 2 and vals.shape[1] == 32:
            return np.ascontiguousarray(vals).reshape(-1)  # already 32-byte LE scalars (must be < r)
        b = b"".join((int(v) % R_ORDER).to_bytes(32, "little") for v in vals)
        return np.frombuffer(b, dtype=np.uint8) if b else np.zeros(0, dtype=np.uint8)

    @staticmethod
    def check_many(vk: "VerifierKey", comms, points, values, proofs, random_vs=None, ctx: Optional["Context"] = None) -> np.ndarray:
        """KZG10::check for many openings at once (one GPU thread per opening).  comms / proofs: arrays of
        104-byte records; points / values / random_vs: ints.  Returns a bool array."""
        ctx = ctx or default_context()
        n = len(points)
        c = np.ascontiguousarray(np.asarray(comms, dtype=np.uint8).reshape(n, 104))
        w = np.ascontiguousarray(np.asarray(proofs, dtype=np.uint8).reshape(n, 104))
        g1 = np.ascontiguousarray(np.concatenate([vk.g.reshape(-1), vk.gamma_g.reshape(-1)]))
        g2 = np.ascontiguousarray(np.concatenate([vk.h.reshape(-1), vk.beta_h.reshape(-1)]))
        z, v = KZG10._scalars(points), KZG10._scalars(values)
        rv = KZG10._scalars([0 if r is None else r for r in random_vs]) if random_vs is not None else None
        ok = np.zeros(n, dtype=np.uint8)
        rc = _ffi.lib().ptau_kzg_check(ctx._h, _ptr(g1), _ptr(g2), _ptr(c) if n else None, _ptr(z) if n else None,
                                       _ptr(v) if n else None, _ptr(w) if n else None,
                                       _ptr(rv) if (rv is not None and n) else None, n, _ptr(ok) if n else None)
        if rc != 0:
            ctx._raise(rc)
        return ok.astype(bool)

    @staticmethod
    def check(vk: "VerifierKey", comm, point: int, value: int, proof, random_v=None, ctx: Optional["Context"] = None) -> bool:
        """KZG10::check(&vk, &comm, point, value, &proof): e(C - [v]g - [rv]gamma_g, h) == e(w, beta_h - [z]h)."""
        return bool(KZG10.check_many(vk, [comm], [point], [value], [proof], None if random_v is None else [random_v], ctx=ctx)[0])

    @staticmethod
    def pairing_product2(g1_pairs: np.ndarray, g2_pairs: np.ndarray, ctx: Optional["Context"] = None):
        """prod_{k<2} e(P_ik, Q_ik) for n items: g1_pairs [n, 2, 104], g2_pairs [n, 2, 200] Montgomery-limb records.
        Returns (gt [n, 576] canonical little-endian Fq12 coefficients in arkworks order, is_one [n] bool)."""
        ctx = ctx or default_context()
        a = np.ascontiguousarray(np.asarray(g1_pairs, dtype=np.uint8).reshape(-1, 2, 104))
        b = np.ascontiguousarray(np.asarray(g2_pairs, dtype=np.uint8).reshape(-1, 2, 200))
        n = a.shape[0]
        gt = np.zeros((n, 576), dtype=np.uint8)
        one = np.zeros(n, dtype=np.uint8)
        if n:
            rc = _ffi.lib().ptau_pairing_product2(ctx._h, _ptr(a), _ptr(b), n, _ptr(gt), _ptr(one))
            if rc != 0:
                ctx._raise(rc)
        return gt, one.astype(bool)

    @staticmethod
    def batch_check(vk: "VerifierKey", comms, points, values, proofs, random_vs=None, randomizers=None,
                    ctx: Optional["Context"] = None) -> bool:
        """KZG10::batch_check: with randomizers r_i (ark: r_0 = 1, then u128s from the rng),
            total_c = sum r_i (C_i + [z_i] w_i) - [sum r_i v_i] g - [sum r_i rv_i] gamma_g,   total_w = sum r_i w_i,
            e(-total_w, beta_h) * e(total_c, h) == 1.
        Both sums are one multi-scalar multiplication each (ptau_kzg_commit), followed by one pairing product."""
        ctx = ctx or default_context()
        n = len(points)
        if randomizers is None:
            randomizers = [1] + [int.from_bytes(os.urandom(16), "little") for _ in range(n - 1)]
        c = np.asarray(comms, dtype=np.uint8).reshape(n, 104)
        w = np.asarray(proofs, dtype=np.uint8).reshape(n, 104)
        rvs = [0] * n if random_vs is None else [0 if r is None else int(r) for r in random_vs]
        gm = sum(r * int(v) for r, v in zip(randomizers, values)) % R_ORDER
        ggm = sum(r * rv for r, rv in zip(randomizers, rvs)) % R_ORDER
        pts_c = np.concatenate([c, w, vk.g.reshape(1, 104), vk.gamma_g.reshape(1, 104)])
        sc_c = [r % R_ORDER for r in randomizers] + [r * int(z) % R_ORDER for r, z in zip(randomizers, points)] + \
               [(-gm) % R_ORDER, (-ggm) % R_ORDER]
        total_c = KZG10._msm(ctx, [(pts_c, sc_c)])
        total_w = KZG10._msm(ctx, [(w, [(-r) % R_ORDER for r in randomizers])])  # = -sum r_i w_i
        g1 = np.stack([total_w, total_c]).reshape(1, 2, 104)
        g2 = np.stack([vk.beta_h.reshape(-1), vk.h.reshape(-1)]).reshape(1, 2, 200)
        return bool(KZG10.pairing_product2(g1, g2, ctx=ctx)[1][0])


G2_PREPARED_COEFFS = 68  # PTAU_G2_PREPARED_COEFFS


@dataclass
class G2Prepared:
    """ark-ec 0.2 `G2Prepared { ell_coeffs, infinity }` (prepared_h / prepared_beta_h, src/lib.rs:223-224):
    ell_coeffs as a u8 array [68, 3, 96] -- per Miller-loop step the triple (c0, c1, c2) of Fq2 in ark-ff's in-memory
    Montgomery limbs (c0-part | c1-part); empty for the point at infinity, as in ark."""
    ell_coeffs: np.ndarray
    infinity: bool


def g2_prepare(points, ctx: Optional["Context"] = None) -> list:
    """`G2Prepared::from(q)` for each 200-byte G2 record, computed on the GPU (ptau_g2_prepare)."""
    ctx = ctx or default_context()
    pts = np.ascontiguousarray(np.asarray(points, dtype=np.uint8).reshape(-1, 200))
    n = pts.shape[0]
    coeffs = np.zeros((n, G2_PREPARED_COEFFS, 3, 96), dtype=np.uint8)
    inf = np.zeros(n, dtype=np.uint8)
    rc = _ffi.lib().ptau_g2_prepare(ctx._h, _ptr(pts) if n else None, n, _ptr(coeffs) if n else None, _ptr(inf) if n else None)
    if rc != 0:
        ctx._raise(rc)
    return [G2Prepared(ell_coeffs=coeffs[i] if not inf[i] else coeffs[i][:0], infinity=bool(inf[i])) for i in range(n)]


class ResidentPoints:
    """G1 powers kept on the GPU(s) of a context (ptau_kzg_powers_upload): commitments then send only the scalars.
    Behaves like the array it was made from as far as KZG10.commit / open are concerned (len, prefix use)."""

    def __init__(self, ctx: "Context", points: np.ndarray):
        import weakref

        pts = np.ascontiguousarray(np.asarray(points, dtype=np.uint8).reshape(-1, 104))
        self._ctx = ctx
        self._n = pts.shape[0]
        h = C.c_void_p()
        rc = _ffi.lib().ptau_kzg_powers_upload(ctx._h, _ptr(pts) if self._n else None, self._n, C.byref(h))
        if rc != 0:
            ctx._raise(rc)
        self._h = h
        weakref.finalize(self, _ffi.lib().ptau_kzg_powers_free, h)

    def __len__(self) -> int:
        return self._n

    def msm(self, scalars) -> np.ndarray:
        """sum_i scalars[i] * points[i] over the first len(scalars) resident points -> 104-byte record."""
        n = len(scalars)
        if n > self._n:
            raise PtauError(_ffi.ERR_ARG, detail="more scalars than resident points")
        sc = KZG10._scalars(scalars)
        out = np.zeros(104, dtype=np.uint8)
        rc = _ffi.lib().ptau_kzg_commit_resident(self._ctx._h, self._h, _ptr(sc) if n else None, n, _ptr(out))
        if rc != 0:
            self._ctx._raise(rc)
        return out


_default_ctx: Optional[Context] = None


def default_context() -> Context:
    global _default_ctx
    if _default_ctx is None:
        n = int(os.environ.get("PTAU_GPUS", "1"))
        _default_ctx = Context(n_gpus=n)
    return _default_ctx


# ---- containers returned by the loaders (ark-poly-commit 0.2 kzg10 types) --------
# A point array is a numpy u8 array [n, 104] (G1) or [n, 200] (G2) of
# PTAU_FMT_ARK_MONT_LIMBS records: the limbs ark-ff keeps in memory.
def g1_limbs(rec: np.ndarray):
    """(x, y, infinity) of one 104-byte record; x, y as 6 x u64 Montgomery limbs."""
    r = np.ascontiguousarray(rec).view(np.uint8).reshape(-1)
    return r[0:48].view("<u8").copy(), r[48:96].view("<u8").copy(), bool(r[96])


def g2_limbs(rec: np.ndarray):
    r = np.ascontiguousarray(rec).view(np.uint8).reshape(-1)
    x = (r[0:48].view("<u8").copy(), r[48:96].view("<u8").copy())
    y = (r[96:144].view("<u8").copy(), r[144:192].view("<u8").copy())
    return x, y, bool(r[192])


@dataclass
class Powers:
    """kzg10::Powers { powers_of_g, powers_of_gamma_g } (src/lib.rs:186-189)."""
    powers_of_g: np.ndarray
    powers_of_gamma_g: np.ndarray

    def to_device(self, ctx: Optional["Context"] = None) -> "Powers":
        """The same powers kept resident on the context's GPU(s): KZG10.commit / open then upload only scalars."""
        ctx = ctx or default_context()
        return Powers(powers_of_g=ResidentPoints(ctx, self.powers_of_g),
                      powers_of_gamma_g=ResidentPoints(ctx, self.powers_of_gamma_g))


@dataclass
class VerifierKey:
    """kzg10::VerifierKey { g, gamma_g, h, beta_h } (src/lib.rs:191-192).  prepared_h /
    prepared_beta_h are Miller-loop line coefficients that ark derives from h and beta_h
    when it reads the key; KZG10.check / batch_check here compute the same lines inside
    their Miller loops (csrc/pairing.cuh), so the key keeps only the four points."""
    g: np.ndarray
    gamma_g: np.ndarray
    h: np.ndarray
    beta_h: np.ndarray

    def prepared_h(self, ctx: Optional["Context"] = None) -> "G2Prepared":
        return g2_prepare(self.h, ctx)[0]

    def prepared_beta_h(self, ctx: Optional["Context"] = None) -> "G2Prepared":
        return g2_prepare(self.beta_h, ctx)[0]


@dataclass
class UniversalParams:
    """kzg10::UniversalParams (src/lib.rs:217-225).  powers_of_gamma_g is the
    BTreeMap<usize, G1Affine> with keys 0..n-1 stored as an array indexed by key."""
    powers_of_g: np.ndarray
    powers_of_gamma_g: np.ndarray
    h: np.ndarray
    beta_h: np.ndarray            # = powers_of_h[1] (src/lib.rs:221)
    prepared_beta_h_src: np.ndarray  # the file's beta_h, source of prepared_beta_h (src/lib.rs:224)
    neg_powers_of_h: Dict[int, np.ndarray] = field(default_factory=dict)

    def prepared_h(self, ctx: Optional["Context"] = None) -> "G2Prepared":
        return g2_prepare(self.h, ctx)[0]

    def prepared_beta_h(self, ctx: Optional["Context"] = None) -> "G2Prepared":
        """`beta_h.into()` of the FILE's beta_h, not of the `beta_h` field (= powers_of_h[1]): src/lib.rs:221 vs :224."""
        return g2_prepare(self.prepared_beta_h_src, ctx)[0]


@dataclass
class Phase1Parameters:
    """src/lib.rs:30-39."""
    alpha: np.ndarray
    beta_g1: np.ndarray
    beta_g2: np.ndarray
    coeffs_g1: np.ndarray
    coeffs_g2: np.ndarray
    alpha_coeffs_g1: np.ndarray
    beta_coeffs_g1: np.ndarray


# ---- the crate's pub fns ------------------------------------------------------------
def read_g1(reader, ctx: Optional[Context] = None, checks: int = CHECKS_READ) -> np.ndarray:
    """src/lib.rs:41-54.  Reads one 96-byte zcash-uncompressed G1 point from a
    binary file object and returns its 104-byte Montgomery record.  A short read
    raises (the reference `unwrap()`s read_exact); an invalid point raises
    PtauError (the reference returns Err(SerializationError))."""
    buf = reader.read(96)
    if len(buf) != 96:
        raise EOFError("failed to fill whole buffer")
    ctx = ctx or default_context()
    return ctx.convert(G1, FMT_ZCASH_UNCOMPRESSED, buf, FMT_ARK_MONT_LIMBS, checks)


def read_g2(reader, ctx: Optional[Context] = None, checks: int = CHECKS_READ) -> np.ndarray:
    """src/lib.rs:56-80."""
    buf = reader.read(192)
    if len(buf) != 192:
        raise EOFError("failed to fill whole buffer")
    ctx = ctx or default_context()
    return ctx.convert(G2, FMT_ZCASH_UNCOMPRESSED, buf, FMT_ARK_MONT_LIMBS, checks)


def load_phase1(exp: int, directory: str = "..", ctx: Optional[Context] = None,
                checks: int = CHECKS_READ) -> Phase1Parameters:
    """src/lib.rs:82-121: reads `../phase1radix2m{exp}`."""
    m = 2 ** exp
    path = os.path.join(directory, "phase1radix2m%d" % exp)
    try:
        data = np.fromfile(path, dtype=np.uint8)
    except OSError as e:
        raise RuntimeError("Couldn't load phase1radix2m%d: %r" % (exp, e))
    ctx = ctx or default_context()
    g1, g2 = ctx.load_phase1(data, m, checks)
    return Phase1Parameters(
        alpha=g1[0], beta_g1=g1[1], beta_g2=g2[0], coeffs_g1=g1[2:2 + m], coeffs_g2=g2[1:1 + m],
        alpha_coeffs_g1=g1[2 + m:2 + 2 * m], beta_coeffs_g1=g1[2 + 2 * m:2 + 3 * m],
    )


def _check_file_hash(data, digest: str) -> bool:
    """blake2b_simd::State::new().update(data).finalize().to_hex() (src/lib.rs:128-131)."""
    return hashlib.blake2b(data).hexdigest() == digest


def _download_setup(file_url: str, file_digest: str, check_digest: bool, directory: str = "."):
    """src/lib.rs:123-164.  Kept as-is; with no network the download branch raises."""
    path = os.path.join(directory, KZG_SETUP_FILE)
    if os.path.exists(path):
        if check_digest:
            print("Checking existing %s file..." % KZG_SETUP_FILE)
            with open(path, "rb") as f:
                if _check_file_hash(f.read(), file_digest):
                    print("Checking passed, using existing %s file." % KZG_SETUP_FILE)
                    return
        return
    print("Downloading %s" % file_url)
    import urllib.request

    data = urllib.request.urlopen(file_url).read()  # raises offline, like minreq::Error
    if not _check_file_hash(data, file_digest):
        raise IOError("failed validation (expected: %s, fetched %d bytes)" % (file_digest, len(data)))
    with open(path, "wb") as f:
        f.write(data)


def download_kzg_setup(check_digest: bool, directory: str = "."):
    """src/lib.rs:166-168."""
    return _download_setup(KZG_SETUP_URL, KZG_SETUP_FILE_DIGEST, check_digest, directory)


def download_fastkzg_setup(check_digest: bool, directory: str = "."):
    """src/lib.rs:170-172."""
    return _download_setup(FASTKZG_SETUP_URL, FASTKZG_SETUP_FILE_DIGEST, check_digest, directory)


def _n_from_setup_size(variant: int, size: int) -> int:
    if variant == VARIANT_KGZ:  # (3n-1)*96 + 576
        q, r = divmod(size - 576 + 96, 288)
    else:  # (3n-1)*96 + 384 + n*192
        q, r = divmod(size - 384 + 96, 480)
    if r or q < 2:
        raise PtauError(_ffi.ERR_SIZE, detail="%d bytes is not a kzg_setup size" % size)
    return q


def _load_setup_file(variant: int, path: str, log2_powers: Optional[int], ctx: Optional["Context"], checks: int):
    """ptau_load_setup_file: the file is streamed through pinned slabs in C++; the records
    land in the returned arrays."""
    L = _ffi.lib()
    ctx = ctx or default_context()
    if not os.path.exists(path):
        raise FileNotFoundError(path)  # File::open(KZG_SETUP_FILE).unwrap()
    n_in = (1 << log2_powers) if log2_powers is not None else 0
    n_out, bad_i, bad_k = C.c_uint64(0), C.c_uint64(0), C.c_int(0)
    rc = L.ptau_load_setup_file(ctx._h, variant, path.encode(), n_in, checks, None, 0, None, 0, C.byref(n_out),
                                C.byref(bad_i), C.byref(bad_k))
    if rc != 0:
        raise PtauError(rc, detail="%s: %d bytes is not a kzg_setup of this variant/size" % (path, os.path.getsize(path)))
    n = n_out.value
    fast = variant == VARIANT_FASTKGZ
    n_g1, n_g2 = 3 * n - 1 + (0 if fast else 2), (n + 2 if fast else 2)
    # plain (pageable) arrays: pinning 650 MB of output costs more (~0.5 ms per MB) than the staged copy it would save
    b1, b2 = np.empty(n_g1 * 104, dtype=np.uint8), np.empty(n_g2 * 200, dtype=np.uint8)
    rc = L.ptau_load_setup_file(ctx._h, variant, path.encode(), n, checks, _ptr(b1), b1.size, _ptr(b2), b2.size,
                                C.byref(n_out), C.byref(bad_i), C.byref(bad_k))
    if rc != 0:
        ctx._raise(rc, bad_i.value if rc > 0 else None)
    return n, b1.reshape(n_g1, 104), b2.reshape(n_g2, 200)


def load_kzg_setup(path: str = KZG_SETUP_FILE, log2_powers: Optional[int] = None, ctx: Optional[Context] = None,
                   checks: int = CHECKS_LOAD) -> Tuple[Powers, VerifierKey]:
    """src/lib.rs:174-195.  log2_powers None infers n from the file size (the
    reference hard-codes 21).  checks=CHECKS_STRICT gives the validated load."""
    n, g1, g2 = _load_setup_file(VARIANT_KGZ, path, log2_powers, ctx, checks)
    powers = Powers(powers_of_g=g1[: 2 * n - 1], powers_of_gamma_g=g1[2 * n - 1: 3 * n - 1])
    vk = VerifierKey(g=g1[3 * n - 1], gamma_g=g1[3 * n], h=g2[0], beta_h=g2[1])
    return powers, vk


def load_fastkzg_setup(path: str = KZG_SETUP_FILE, log2_powers: Optional[int] = None, ctx: Optional[Context] = None,
                       checks: int = CHECKS_LOAD) -> Tuple[UniversalParams, np.ndarray]:
    """src/lib.rs:197-228."""
    n, g1, g2 = _load_setup_file(VARIANT_FASTKGZ, path, log2_powers, ctx, checks)
    powers_of_h = g2[2:]
    params = UniversalParams(
        powers_of_g=g1[: 2 * n - 1], powers_of_gamma_g=g1[2 * n - 1: 3 * n - 1], h=g2[0], beta_h=powers_of_h[1],
        prepared_beta_h_src=g2[1],
    )
    return params, powers_of_h


# ---- are the powers powers of one tau? (ptau_verify_powers) --------------------------------------
def _verify_file(kind: int, path: str, n: int, ctx: Optional[Context], seed: Optional[bytes]) -> None:
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    data = np.memmap(path, dtype=np.uint8, mode="r")
    try:
        (ctx or default_context()).verify_powers(kind, data, n, seed=seed)
    finally:
        del data


def verify_kzg_setup(path: str = KZG_SETUP_FILE, log2_powers: Optional[int] = None, ctx: Optional[Context] = None,
                     seed: Optional[bytes] = None) -> None:
    """Checks that a preprocess-kgz `kzg_setup` holds powers of one tau (strict point checks, then the ratio
    relations by pairing).  n from log2_powers, or inferred from the file size.  Raises PtauError on failure."""
    n = (1 << log2_powers) if log2_powers is not None else _n_from_setup_size(VARIANT_KGZ, os.path.getsize(path))
    _verify_file(POWERS_KGZ, path, n, ctx, seed)


def verify_fastkzg_setup(path: str = KZG_SETUP_FILE, log2_powers: Optional[int] = None, ctx: Optional[Context] = None,
                         seed: Optional[bytes] = None) -> None:
    """verify_kzg_setup for a preprocess-fastkgz `kzg_setup` (its powers_of_h are checked too)."""
    n = (1 << log2_powers) if log2_powers is not None else _n_from_setup_size(VARIANT_FASTKGZ, os.path.getsize(path))
    _verify_file(POWERS_FASTKGZ, path, n, ctx, seed)


def verify_powersoftau(path: str = POWERSOFTAU_FILE, log2_powers: int = DEFAULT_LOG2_POWERS, ctx: Optional[Context] = None,
                       seed: Optional[bytes] = None) -> None:
    """Checks that a `powersoftau` response holds powers of one tau: tau, alpha and beta powers, both groups."""
    _verify_file(POWERS_RESPONSE, path, 1 << log2_powers, ctx, seed)


# ---- the two binaries (src/bin/preprocess-kgz.rs, preprocess-fastkgz.rs) -------------
def _preprocess_main(variant: int, directory: str, log2_powers: int, expected_digest: Optional[str],
                     emit_uncompressed: bool, checks: int, ctx: Optional[Context]):
    """Both binaries' main(): everything (size check, BLAKE2b digest check, create_new of
    the intermediate file, streaming through pinned slabs, section table) happens in
    ptau_preprocess_files (csrc/files.cu); this wrapper only maps return codes onto the
    reference's panics/messages."""
    L = _ffi.lib()
    n = 1 << log2_powers
    src_path = os.path.join(directory, POWERSOFTAU_FILE)
    unc_path = os.path.join(directory, POWERSOFTAU_UNCOMPRESSED_FILE)
    out_path = os.path.join(directory, KZG_SETUP_FILE)
    if not os.path.exists(src_path):
        raise FileNotFoundError("unable open `%s` in this directory" % POWERSOFTAU_FILE)
    flags = 0
    if expected_digest is None:
        flags |= _ffi.FILE_SKIP_DIGEST
    else:
        print("Checking existing %s file..." % POWERSOFTAU_FILE)
    if not emit_uncompressed:
        flags |= _ffi.FILE_NO_UNCOMPRESSED
    ctx = ctx or default_context()
    print("Started deserializing compressed Powers of Tau...")
    bad_i, bad_k, bad_s = C.c_uint64(0), C.c_int(0), C.c_int(-1)
    rc = L.ptau_preprocess_files(ctx._h, variant, src_path.encode(), out_path.encode(), unc_path.encode(), log2_powers,
                                 expected_digest.encode() if expected_digest else None, flags, checks,
                                 C.byref(bad_i), C.byref(bad_k), C.byref(bad_s))
    if rc == _ffi.ERR_SIZE:  # preprocess-kgz.rs:83-90
        raise PtauError(rc, detail="The size of `%s` should be %d, but it's %d, so something isn't right."
                        % (POWERSOFTAU_FILE, L.ptau_response_size(n), os.path.getsize(src_path)))
    if rc == _ffi.ERR_EXISTS:  # create_new(true), preprocess-kgz.rs:113-118
        raise FileExistsError("unable to create `%s`" % POWERSOFTAU_UNCOMPRESSED_FILE)
    if rc == _ffi.ERR_DIGEST:
        raise IOError("failed validation (expected: %s); download impossible offline" % expected_digest)
    if rc != 0:
        ctx._raise(rc, bad_i.value if rc > 0 else None, bad_s.value if rc > 0 else None)
    print("Done serializing. KZG parameters are stored in %s" % KZG_SETUP_FILE)
    return out_path


def preprocess_kgz(directory: str = ".", log2_powers: int = DEFAULT_LOG2_POWERS,
                   expected_digest: Optional[str] = POWERSOFTAU_DIGEST, emit_uncompressed: bool = True,
                   checks: int = CHECKS_STRICT, ctx: Optional[Context] = None) -> str:
    """main() of src/bin/preprocess-kgz.rs:162-200: `powersoftau` ->
    (`powersoftau_uncompressed`) -> `kzg_setup` in `directory`."""
    return _preprocess_main(VARIANT_KGZ, directory, log2_powers, expected_digest, emit_uncompressed, checks, ctx)


def preprocess_fastkgz(directory: str = ".", log2_powers: int = DEFAULT_LOG2_POWERS,
                       expected_digest: Optional[str] = POWERSOFTAU_DIGEST, emit_uncompressed: bool = True,
                       checks: int = CHECKS_STRICT, ctx: Optional[Context] = None) -> str:
    """main() of src/bin/preprocess-fastkgz.rs:180-214."""
    return _preprocess_main(VARIANT_FASTKGZ, directory, log2_powers, expected_digest, emit_uncompressed, checks, ctx)


# ---- a Powers-of-Tau contribution (powersoftau compute / verify_transform / new_challenge) -------------------------
def _write_new(path: str, size: int, fill) -> None:
    """Creates `path` atomically: `fill` writes a memory-mapped temporary file of `size` bytes in the same directory,
    which is then linked to `path` (never replacing an existing file: FileExistsError) and removed."""
    if os.path.exists(path):
        raise FileExistsError(path)
    tmp = "%s.tmp-%d" % (path, os.getpid())
    try:
        with open(tmp, "wb") as f:
            f.truncate(size)
        m = np.memmap(tmp, dtype=np.uint8, mode="r+", shape=(size,))
        try:
            fill(m)
            m.flush()
        finally:
            del m
        os.link(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.unlink(tmp)


def _read_map(path: str) -> np.ndarray:
    if not os.path.exists(path):
        raise FileNotFoundError(path)
    return np.memmap(path, dtype=np.uint8, mode="r")


def challenge_from_response(response_path: str, challenge_path: str, log2_powers: int = DEFAULT_LOG2_POWERS,
                            ctx: Optional[Context] = None, checks: int = CHECKS_STRICT) -> bytes:
    """powersoftau new_challenge: writes BLAKE2b(response) || the response's accumulator in uncompressed records to
    `challenge_path` (created new).  This is how a downloaded response becomes the challenge of one's own
    contribution.  Returns the new challenge's 64-byte prefix."""
    L = _ffi.lib()
    n = 1 << log2_powers
    ctx = ctx or default_context()
    resp = _read_map(response_path)
    if resp.size != L.ptau_response_size(n):
        raise PtauError(_ffi.ERR_SIZE, detail="%s is not a response of 2^%d powers" % (response_path, log2_powers))
    hx = C.create_string_buffer(129)
    rc = L.ptau_blake2b_file(response_path.encode(), hx)
    if rc != 0:
        raise PtauError(rc, detail=response_path)
    digest = bytes.fromhex(hx.value.decode())

    def fill(m):
        m[:64] = np.frombuffer(digest, dtype=np.uint8)
        ri, ro = 64, 64
        for s, (group, count) in enumerate(((G1, 2 * n - 1), (G2, n), (G1, n), (G1, n), (G2, 1))):
            ci, cu = L.ptau_record_size(group, FMT_ZCASH_COMPRESSED), L.ptau_record_size(group, FMT_ZCASH_UNCOMPRESSED)
            try:
                ctx.convert(group, FMT_ZCASH_COMPRESSED, resp[ri:ri + count * ci], FMT_ZCASH_UNCOMPRESSED, checks,
                            out=m[ro:ro + count * cu])
            except PtauError as e:
                e.section = s
                raise
            ri += count * ci
            ro += count * cu

    try:
        _write_new(challenge_path, L.ptau_challenge_size(n), fill)
    finally:
        del resp
    return digest


def contribute(challenge_path: str, response_path: str, log2_powers: int = DEFAULT_LOG2_POWERS,
               ctx: Optional[Context] = None, secrets=None, checks: int = CHECKS_STRICT) -> bytes:
    """powersoftau compute: reads `challenge_path`, writes the response to `response_path` (created new) and returns
    the response's 64-byte prefix (BLAKE2b of the challenge).  secrets: None draws them from the OS inside the
    library, which wipes its copies before returning; secrets passed in as Python ints or bytes stay in the caller's
    objects, which Python cannot wipe."""
    L = _ffi.lib()
    n = 1 << log2_powers
    ctx = ctx or default_context()
    chal = _read_map(challenge_path)
    if chal.size != L.ptau_challenge_size(n):
        raise PtauError(_ffi.ERR_SIZE, detail="%s is not a challenge of 2^%d powers" % (challenge_path, log2_powers))
    try:
        _write_new(response_path, L.ptau_response_size(n),
                   lambda m: ctx.contribute(chal, n, secrets=secrets, checks=checks, out=m))
    finally:
        del chal
    with open(response_path, "rb") as f:
        return f.read(64)


def verify_contribution(challenge_path: Optional[str], response_path: str, log2_powers: int = DEFAULT_LOG2_POWERS,
                        ctx: Optional[Context] = None, seed: Optional[bytes] = None) -> None:
    """powersoftau verify_transform of `response_path` against `challenge_path` (None: the response's public key and
    powers only).  Raises PtauError on failure."""
    n = 1 << log2_powers
    ctx = ctx or default_context()
    resp = _read_map(response_path)
    chal = _read_map(challenge_path) if challenge_path is not None else None
    try:
        ctx.verify_contribution(chal, resp, n, seed=seed)
    finally:
        del resp, chal
