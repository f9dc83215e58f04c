// File-to-file pipelines of libptau_b200.so: the two reference binaries' main()
// (/root/reference/src/bin/preprocess-kgz.rs:162-200,
//  /root/reference/src/bin/preprocess-fastkgz.rs:180-214) as one streaming pass.
//
// The reference holds every section in RAM as Vec<GroupAffine> (O(N) memory, and
// download_parameters even slurps the whole file to hash it, preprocess-kgz.rs:41-42).
// Here the `powersoftau` file is streamed slab by slab through pinned host buffers:
// a reader thread prefetches slab k+1, the GPUs convert slab k (ptau_convert shards it
// by index range), a writer thread flushes slab k-1.  Memory is O(slab).
#include <errno.h>
#include <fcntl.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <unistd.h>

#include <chrono>
#include <future>
#include <string>
#include <vector>

#include "../../include/ptau_b200.h"
#include "blake2b.h"
#include "layout.h"

namespace {

const char* kPowersoftauDigest =  // preprocess-kgz.rs:19
    "88dc1dc6914e44568e8511eace177e6ecd9da9a9bd8f67e4c0c9f215b517db4d1d54a755d051978dbb85ef947918193c"
    "93cd4cf4c99c0dc5a767d4eeb10047a4";

bool pread_all(int fd, void* buf, size_t len, uint64_t off) {
  uint8_t* p = (uint8_t*)buf;
  while (len) {
    ssize_t r = pread(fd, p, len, (off_t)off);
    if (r <= 0) {
      if (r < 0 && errno == EINTR) continue;
      return false;
    }
    p += r;
    off += (uint64_t)r;
    len -= (size_t)r;
  }
  return true;
}
bool pwrite_all(int fd, const void* buf, size_t len, uint64_t off) {
  const uint8_t* p = (const uint8_t*)buf;
  while (len) {
    ssize_t r = pwrite(fd, p, len, (off_t)off);
    if (r <= 0) {
      if (r < 0 && errno == EINTR) continue;
      return false;
    }
    p += r;
    off += (uint64_t)r;
    len -= (size_t)r;
  }
  return true;
}

// A slab goes to the page cache in parallel parts: one thread copies ~2 GB/s into fresh pages, which is slower than
// the GPUs produce records.
bool pwrite_parts(int fd, const void* buf, size_t len, uint64_t off) {
  const size_t kPart = 8u << 20;
  if (len <= 2 * kPart) return pwrite_all(fd, buf, len, off);
  const int parts = len / kPart > 4 ? 4 : (int)(len / kPart);
  const size_t each = ((len / parts) + 4095) & ~(size_t)4095;
  std::future<bool> f[4];
  for (int i = 1; i < parts; i++) {
    const size_t lo = each * i, n = i == parts - 1 ? len - lo : each;
    f[i] = std::async(std::launch::async, pwrite_all, fd, (const void*)((const uint8_t*)buf + lo), n, off + lo);
  }
  bool ok = pwrite_all(fd, buf, each, off);
  for (int i = 1; i < parts; i++) ok = f[i].get() && ok;
  return ok;
}

// PTAU_TRACE=1: wall-clock marks of the file pipelines on stderr
struct Trace {
  bool on;
  std::chrono::steady_clock::time_point t0, last;
  Trace() : on(getenv("PTAU_TRACE") != nullptr), t0(std::chrono::steady_clock::now()), last(t0) {}
  void mark(const char* what) {
    if (!on) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[ptau trace] %-24s +%.1f ms (total %.1f ms)\n", what,
            std::chrono::duration<double, std::milli>(now - last).count(),
            std::chrono::duration<double, std::milli>(now - t0).count());
    last = now;
  }
};

struct Pinned {
  void* p = nullptr;
  explicit Pinned(size_t n) { p = ptau_host_alloc(n); }
  ~Pinned() { ptau_host_free(p); }
  uint8_t* u8() { return (uint8_t*)p; }
};

}  // namespace

extern "C" {

int ptau_blake2b_file(const char* path, char out_hex[129]) {
  int fd = open(path, O_RDONLY);
  if (fd < 0) return PTAU_ERR_IO;
  ptau::Blake2b h;
  std::vector<uint8_t> buf(8 << 20);
  for (;;) {
    ssize_t r = read(fd, buf.data(), buf.size());
    if (r < 0) {
      if (errno == EINTR) continue;
      close(fd);
      return PTAU_ERR_IO;
    }
    if (r == 0) break;
    h.update(buf.data(), (size_t)r);
  }
  close(fd);
  std::string s = h.hexdigest();
  memcpy(out_hex, s.c_str(), 129);
  return PTAU_OK;
}

// Outputs are written under temporary names next to their final paths and published only when the whole job
// succeeded (`kzg_setup`: rename(), replacing an older file atomically; `powersoftau_uncompressed`: link(), which
// keeps the reference's create_new semantics); on any error they are unlinked.  The reference validates everything
// in RAM before it creates `kzg_setup` (preprocess-kgz.rs:128-160 then :186), so a bad input never leaves a partial
// or truncated file behind there either.
//
// Error precedence = the reference's order of events: BLAKE2b digest (preprocess-kgz.rs:33-47), then any decode error
// of the decompression pass over ALL sections (:105-110), then create_new of the intermediate file (:113-118), then
// the first bad point of the read_g1 / read_g2 loops (:140-153).  The slabs still make one pass: a stage-2 error is
// remembered while the remaining slabs are only decompressed, and the digest is computed by a thread of its own
// while the GPUs work.
int ptau_preprocess_files(ptau_ctx* ctx, int variant, const char* response_path, const char* setup_path,
                          const char* uncompressed_path, unsigned log2_powers, const char* expected_digest_hex,
                          unsigned flags, unsigned checks, uint64_t* bad_index, int* bad_kind, int* bad_section) {
  if (!ctx || !response_path || !setup_path || log2_powers < 1 || log2_powers > 30) return PTAU_ERR_ARG;
  if (variant != PTAU_VARIANT_KGZ && variant != PTAU_VARIANT_FASTKGZ) return PTAU_ERR_ARG;
  const uint64_t n = 1ull << log2_powers;
  const bool fast = variant == PTAU_VARIANT_FASTKGZ;
  const bool emit_unc = uncompressed_path && !(flags & PTAU_FILE_NO_UNCOMPRESSED);
  Trace trace;

  int fd_in = open(response_path, O_RDONLY);
  if (fd_in < 0) return PTAU_ERR_IO;
  struct stat st;
  if (fstat(fd_in, &st) != 0) {
    close(fd_in);
    return PTAU_ERR_IO;
  }
  // preprocess-kgz.rs:83: size must equal CONTRIBUTION_BYTE_SIZE
  if ((uint64_t)st.st_size != ptau_response_size(n)) {
    close(fd_in);
    return PTAU_ERR_SIZE;
  }
  // download_parameters (preprocess-kgz.rs:38-47): digest of the existing file.  A mismatch sends the reference to
  // the network; offline that is an error.  Hashing 604 MB takes as long as the GPUs need for the points, so it
  // runs beside them and is checked before anything is published.
  std::future<int> digest;
  char digest_hex[129] = {0};
  if (!(flags & PTAU_FILE_SKIP_DIGEST))
    digest = std::async(std::launch::async, ptau_blake2b_file, response_path, digest_hex);

  const std::string tmp_tag = ".tmp." + std::to_string((long)getpid());
  const std::string setup_tmp = std::string(setup_path) + tmp_tag;
  const std::string unc_tmp = emit_unc ? std::string(uncompressed_path) + tmp_tag : std::string();
  bool unc_exists = false;
  int fd_unc = -1, fd_out = -1;
  auto fail = [&](int code) {
    if (digest.valid()) digest.wait();
    close(fd_in);
    if (fd_unc >= 0) close(fd_unc);
    if (fd_out >= 0) close(fd_out);
    if (fd_out >= 0) unlink(setup_tmp.c_str());
    if (fd_unc >= 0) unlink(unc_tmp.c_str());
    return code;
  };
  if (emit_unc) {
    struct stat su;
    unc_exists = lstat(uncompressed_path, &su) == 0;  // create_new(true) will fail (preprocess-kgz.rs:113-118)
    if (!unc_exists) {
      fd_unc = open(unc_tmp.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
      if (fd_unc < 0) return fail(PTAU_ERR_IO);
    }
  }
  fd_out = open(setup_tmp.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0644);
  if (fd_out < 0) return fail(PTAU_ERR_IO);

  const auto secs = ptau::response_sections(n);
  const ptau::SetupLayout L = ptau::setup_layout(variant, n);
  // offset of each section's ark output in `kzg_setup`, -1 = checked but not written
  const int64_t out_off[5] = {
      (int64_t)L.g1(0),                          // tau_g1 -> powers_of_g
      fast ? (int64_t)L.g2(L.powers_of_h) : -1,  // tau_g2 -> powers_of_h (fast)
      (int64_t)L.g1(L.gamma_g),                  // alpha_g1 -> powers_of_gamma_g
      -1, -1};
  const bool process[5] = {
      true, true, true,
      fast || emit_unc,  // beta_g1: fastkgz reads+checks+drops it (:156-159); kgz never reads it
      emit_unc,          // beta_g2: only ever decompressed into `powersoftau_uncompressed`
  };
  // points per slab: pinned memory is paid for by the page (allocation time), so no more than the pipeline needs
  unsigned slab_log2 = 18;
  if (const char* e = getenv("PTAU_SLAB_LOG2")) slab_log2 = (unsigned)atoi(e) < 10 ? 10 : (unsigned)atoi(e) > 22 ? 22 : (unsigned)atoi(e);
  const size_t slab = (size_t)((2 * n) < (1ull << slab_log2) ? (2 * n) : (1ull << slab_log2));
  Pinned in0(slab * 96), in1(slab * 96), out0(slab * 192), out1(slab * 192);
  Pinned unc0(emit_unc ? slab * 192 : 16), unc1(emit_unc ? slab * 192 : 16);
  if (!in0.p || !in1.p || !unc0.p || !unc1.p || !out0.p || !out1.p) return fail(PTAU_ERR_NOMEM);
  trace.mark("open + pinned slabs");
  uint8_t* inb[2] = {in0.u8(), in1.u8()};
  uint8_t* uncb[2] = {unc0.u8(), unc1.u8()};
  uint8_t* outb[2] = {out0.u8(), out1.u8()};
  uint8_t first_g1[96], first_alpha[96], first_g2[384];
  memset(first_g2, 0, sizeof(first_g2));

  int rc = PTAU_OK;
  // first stage-2 (read_g1 / read_g2) error, reported only if the decompression of everything after it is clean
  int s2_rc = PTAU_OK, s2_kind = 0, s2_sec = -1;
  uint64_t s2_index = 0;
  uint64_t in_off = ptau::kResponseHash;  // skip the 64-byte challenge hash (:96-101)
  uint64_t unc_off = 0;
  std::future<bool> wr[2], wu[2];
  for (int s = 0; s < 5 && rc == PTAU_OK; s++) {
    const ptau::Section& sec = secs[s];
    const size_t rc_in = ptau_record_size(sec.group, PTAU_FMT_ZCASH_COMPRESSED);
    const size_t r_unc = ptau_record_size(sec.group, PTAU_FMT_ZCASH_UNCOMPRESSED);
    const size_t r_out = ptau_record_size(sec.group, PTAU_FMT_ARK_UNCOMPRESSED);
    const bool only_decompress = (s == 3 && !fast) || s == 4;  // sections the binaries never validate
    if (process[s]) {
      const uint64_t nslab = (sec.count + slab - 1) / slab;
      std::future<bool> rd = std::async(std::launch::async, pread_all, fd_in, inb[0],
                                        (size_t)((sec.count < slab ? sec.count : slab) * rc_in), in_off);
      for (uint64_t k = 0; k < nslab && rc == PTAU_OK; k++) {
        const int b = (int)(k & 1);
        const uint64_t lo = k * slab;
        const size_t cnt = (size_t)(sec.count - lo < slab ? sec.count - lo : slab);
        if (!rd.get()) rc = PTAU_ERR_IO;
        if (k + 1 < nslab) {
          const uint64_t lo2 = (k + 1) * slab;
          const size_t cnt2 = (size_t)(sec.count - lo2 < slab ? sec.count - lo2 : slab);
          rd = std::async(std::launch::async, pread_all, fd_in, inb[b ^ 1], cnt2 * rc_in, in_off + lo2 * rc_in);
        }
        if (wr[b].valid() && !wr[b].get()) rc = PTAU_ERR_IO;  // buffer b is free again
        if (wu[b].valid() && !wu[b].get()) rc = PTAU_ERR_IO;
        if (rc != PTAU_OK) break;
        uint64_t bi = 0;
        int bk = 0;
        const bool stage2 = !only_decompress && s2_rc == PTAU_OK;
        // sections that are checked but not written (kgz: tau_g2 beyond its first slab;
        // fastkgz: beta_g1) are validated on the GPU without copying results back
        uint8_t* dst = (out_off[s] >= 0 || k == 0) ? outb[b] : nullptr;
        int rc2 = PTAU_OK;
        if (emit_unc) {
          // stage 1: decompress (CheckForCorrectness::No) -> `powersoftau_uncompressed`
          rc = ptau_convert(ctx, sec.group, PTAU_FMT_ZCASH_COMPRESSED, inb[b], PTAU_FMT_ZCASH_UNCOMPRESSED, uncb[b], cnt,
                            PTAU_CHECKS_DECOMPRESS, &bi, &bk);
          if (rc == PTAU_OK && fd_unc >= 0)
            wu[b] = std::async(std::launch::async, pwrite_parts, fd_unc, (const void*)uncb[b], cnt * r_unc,
                               unc_off + lo * r_unc);
          // stage 2: read_g1 / read_g2 on the uncompressed bytes
          if (rc == PTAU_OK && stage2)
            rc2 = ptau_convert(ctx, sec.group, PTAU_FMT_ZCASH_UNCOMPRESSED, uncb[b], PTAU_FMT_ARK_UNCOMPRESSED, dst, cnt,
                               checks, &bi, &bk);
        } else if (stage2) {
          // fused: a decode error of the decompression and a failed check are told apart by the kind, and the kernel
          // reports the lowest bad index of the slab -- same precedence within a slab only if nothing later fails to
          // decode, so a check failure is re-examined below
          rc2 = ptau_convert(ctx, sec.group, PTAU_FMT_ZCASH_COMPRESSED, inb[b], PTAU_FMT_ARK_UNCOMPRESSED, dst, cnt, checks,
                             &bi, &bk);
          if (rc2 == PTAU_BAD_NOT_IN_SUBGROUP || rc2 == PTAU_BAD_INFINITY) {
            // stage-2 kinds; is there a stage-1 (decode) error anywhere in this slab?
            uint64_t bi1 = 0;
            int bk1 = 0;
            int rc1 = ptau_convert(ctx, sec.group, PTAU_FMT_ZCASH_COMPRESSED, inb[b], PTAU_FMT_ZCASH_UNCOMPRESSED, nullptr, cnt,
                                   PTAU_CHECKS_DECOMPRESS, &bi1, &bk1);
            if (rc1 != PTAU_OK) {
              rc = rc1;
              bi = bi1;
              bk = bk1;
              rc2 = PTAU_OK;
            }
          } else if (rc2 != PTAU_OK) {  // decode error (or a runtime error): stage 1
            rc = rc2;
            rc2 = PTAU_OK;
          }
        } else if (!only_decompress || emit_unc) {
          // a stage-2 error is pending: only look for decode errors from here on
          rc = ptau_convert(ctx, sec.group, PTAU_FMT_ZCASH_COMPRESSED, inb[b], PTAU_FMT_ZCASH_UNCOMPRESSED, nullptr, cnt,
                            PTAU_CHECKS_DECOMPRESS, &bi, &bk);
        }
        if (rc > 0) {
          if (bad_index) *bad_index = lo + bi;
          if (bad_kind) *bad_kind = bk;
          if (bad_section) *bad_section = s;
          break;
        }
        if (rc != PTAU_OK) break;
        if (rc2 < 0) {
          rc = rc2;
          break;
        }
        if (rc2 > 0) {
          s2_rc = rc2;
          s2_kind = bk;
          s2_sec = s;
          s2_index = lo + bi;
          continue;
        }
        if (stage2) {
          if (k == 0) {
            if (s == 0) memcpy(first_g1, outb[b], 96);
            if (s == 2) memcpy(first_alpha, outb[b], 96);
            if (s == 1) memcpy(first_g2, outb[b], 384);  // n >= 2
          }
          if (out_off[s] >= 0)
            wr[b] = std::async(std::launch::async, pwrite_parts, fd_out, (const void*)outb[b], cnt * r_out,
                               (uint64_t)out_off[s] + lo * r_out);
        }
      }
      if (rd.valid()) rd.wait();
    }
    in_off += sec.count * rc_in;
    unc_off += sec.count * r_unc;
  }
  for (int b = 0; b < 2; b++) {
    if (wr[b].valid() && !wr[b].get() && rc == PTAU_OK) rc = PTAU_ERR_IO;
    if (wu[b].valid() && !wu[b].get() && rc == PTAU_OK) rc = PTAU_ERR_IO;
  }
  trace.mark("sections");
  // precedence: digest, decode errors (rc), create_new, first read_g1/read_g2 error
  if (digest.valid()) {
    int drc = digest.get();
    if (drc != PTAU_OK) return fail(drc);
    if (strcmp(digest_hex, expected_digest_hex ? expected_digest_hex : kPowersoftauDigest) != 0) return fail(PTAU_ERR_DIGEST);
  }
  trace.mark("digest join");
  if (rc != PTAU_OK) return fail(rc);
  if (unc_exists) return fail(PTAU_ERR_EXISTS);
  if (s2_rc != PTAU_OK) {
    if (bad_index) *bad_index = s2_index;
    if (bad_kind) *bad_kind = s2_kind;
    if (bad_section) *bad_section = s2_sec;
    return fail(s2_rc);
  }
  if (!fast) {  // VerifierKey tail: g, gamma_g, h, beta_h (preprocess-kgz.rs:177-194)
    uint8_t tail[576];
    memcpy(tail, first_g1, 96);
    memcpy(tail + 96, first_alpha, 96);
    memcpy(tail + 192, first_g2, 384);
    if (!pwrite_all(fd_out, tail, sizeof(tail), L.g1(L.vk_g))) return fail(PTAU_ERR_IO);
  } else {  // h, beta_h in front of powers_of_h (preprocess-fastkgz.rs:199-208)
    if (!pwrite_all(fd_out, first_g2, 384, L.g2(0))) return fail(PTAU_ERR_IO);
  }
  if (flags & PTAU_FILE_FSYNC) {
    if (fsync(fd_out) != 0 || (fd_unc >= 0 && fsync(fd_unc) != 0)) return fail(PTAU_ERR_IO);
  }
  // publish
  if (fd_unc >= 0) {
    if (close(fd_unc) != 0) {
      fd_unc = -1;
      unlink(unc_tmp.c_str());
      return fail(PTAU_ERR_IO);
    }
    fd_unc = -1;
    if (link(unc_tmp.c_str(), uncompressed_path) != 0) {  // create_new: never replaces an existing file
      const int code = errno == EEXIST ? PTAU_ERR_EXISTS : PTAU_ERR_IO;
      unlink(unc_tmp.c_str());
      return fail(code);
    }
    unlink(unc_tmp.c_str());
  }
  const int crc = close(fd_out);
  fd_out = -1;
  if (crc != 0 || rename(setup_tmp.c_str(), setup_path) != 0) {
    unlink(setup_tmp.c_str());
    if (emit_unc) unlink(uncompressed_path);
    return fail(PTAU_ERR_IO);
  }
  close(fd_in);
  trace.mark("publish");
  return PTAU_OK;
}

// load_kzg_setup / load_fastkzg_setup (/root/reference/src/lib.rs:174-228) from the file:
// `kzg_setup` is streamed through pinned slabs; records land in the caller's buffers
// (pin them with ptau_host_alloc for full PCIe speed).  n_powers == 0 infers n from the file
// size (the reference hard-codes 2^21).
int ptau_load_setup_file(ptau_ctx* ctx, int variant, const char* setup_path, uint64_t n_powers, unsigned checks,
                         void* g1_out, uint64_t g1_out_len, void* g2_out, uint64_t g2_out_len, uint64_t* n_powers_out,
                         uint64_t* bad_index, int* bad_kind) {
  if (!ctx || !setup_path) return PTAU_ERR_ARG;
  if (variant != PTAU_VARIANT_KGZ && variant != PTAU_VARIANT_FASTKGZ) return PTAU_ERR_ARG;
  const bool fast = variant == PTAU_VARIANT_FASTKGZ;
  int fd = open(setup_path, O_RDONLY);
  if (fd < 0) return PTAU_ERR_IO;
  struct stat st;
  if (fstat(fd, &st) != 0) {
    close(fd);
    return PTAU_ERR_IO;
  }
  uint64_t n = n_powers;
  if (n == 0) {  // kgz: (3n-1)*96 + 576 ; fastkgz: (3n-1)*96 + 384 + n*192
    const uint64_t sz = (uint64_t)st.st_size;
    const uint64_t num = fast ? sz + 96 - 384 : sz + 96 - 576, den = fast ? 480 : 288;
    if (sz < 1000 || num % den) {
      close(fd);
      return PTAU_ERR_SIZE;
    }
    n = num / den;
  }
  if (n_powers_out) *n_powers_out = n;
  if ((uint64_t)st.st_size != ptau_setup_size(variant, n)) {  // the reference's unwrap() panics on a short file
    close(fd);
    return PTAU_ERR_SIZE;
  }
  const ptau::SetupLayout L = ptau::setup_layout(variant, n);
  if (!g1_out || !g2_out) {  // size query
    close(fd);
    return (g1_out_len == 0 && g2_out_len == 0) ? PTAU_OK : PTAU_ERR_ARG;
  }
  if (g1_out_len != L.n_g1 * ptau::kMontG1 || g2_out_len != L.n_g2 * ptau::kMontG2) {
    close(fd);
    return PTAU_ERR_SIZE;
  }
  // pinned memory costs ~0.5 ms per MB to allocate: two slabs of 2^18 records (the G1 sections are 96-byte records;
  // the few G2 slabs of a fastkgz file go through the same buffers at half the count)
  Trace trace;
  const size_t slab_bytes = (size_t)96 << 18;
  Pinned b0(slab_bytes), b1(slab_bytes);
  if (!b0.p || !b1.p) {
    close(fd);
    return PTAU_ERR_NOMEM;
  }
  trace.mark("load: pinned slabs");
  uint8_t* buf[2] = {b0.u8(), b1.u8()};
  const struct {
    int group;
    uint64_t count;
    uint8_t* out;
  } secs[2] = {{PTAU_G1, L.n_g1, (uint8_t*)g1_out}, {PTAU_G2, L.n_g2, (uint8_t*)g2_out}};
  int rc = PTAU_OK;
  uint64_t off = 0, base = 0;
  for (int s = 0; s < 2 && rc == PTAU_OK; s++) {
    const size_t ri = ptau_record_size(secs[s].group, PTAU_FMT_ARK_UNCOMPRESSED);
    const size_t ro = ptau_record_size(secs[s].group, PTAU_FMT_ARK_MONT_LIMBS);
    const size_t slab = slab_bytes / ri;
    const uint64_t cnt = secs[s].count, nslab = (cnt + slab - 1) / slab;
    std::future<bool> rd = std::async(std::launch::async, pread_all, fd, buf[0], (size_t)((cnt < slab ? cnt : slab) * ri), off);
    for (uint64_t k = 0; k < nslab && rc == PTAU_OK; k++) {
      const int b = (int)(k & 1);
      const uint64_t lo = k * slab;
      const size_t c = (size_t)(cnt - lo < slab ? cnt - lo : slab);
      if (!rd.get()) rc = PTAU_ERR_IO;
      if (k + 1 < nslab) {
        const uint64_t lo2 = (k + 1) * slab;
        rd = std::async(std::launch::async, pread_all, fd, buf[b ^ 1], (size_t)((cnt - lo2 < slab ? cnt - lo2 : slab) * ri),
                        off + lo2 * ri);
      }
      if (rc != PTAU_OK) break;
      uint64_t bi = 0;
      int bk = 0;
      rc = ptau_convert(ctx, secs[s].group, PTAU_FMT_ARK_UNCOMPRESSED, buf[b], PTAU_FMT_ARK_MONT_LIMBS, secs[s].out + lo * ro, c,
                        checks, &bi, &bk);
      if (rc > 0) {
        if (bad_index) *bad_index = base + lo + bi;  // index over all points in file order
        if (bad_kind) *bad_kind = bk;
      }
    }
    if (rd.valid()) rd.wait();
    off += cnt * ri;
    base += cnt;
  }
  close(fd);
  trace.mark("load: sections");
  return rc;
}

}  // extern "C"
