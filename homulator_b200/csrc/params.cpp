#include "params.h"

namespace hml {

typedef unsigned __int128 u128;

u64 h_mulmod(u64 a, u64 b, u64 m) { return (u64)(((u128)a * b) % m); }
u64 h_powmod(u64 a, u64 e, u64 m) {
  u64 r = 1 % m;
  a %= m;
  for (; e; e >>= 1) {
    if (e & 1) r = h_mulmod(r, a, m);
    a = h_mulmod(a, a, m);
  }
  return r;
}
u64 h_invmod(u64 a, u64 m) { return h_powmod(a % m, m - 2, m); }

bool h_is_prime(u64 n) {
  // deterministic Miller-Rabin for 64-bit n (first twelve prime bases)
  static const u64 B[12] = {2, 3, 5, 7, 11, 13, 17, 19, 23, 29, 31, 37};
  if (n < 2) return false;
  for (u64 b : B) {
    if (n == b) return true;
    if (n % b == 0) return false;
  }
  u64 d = n - 1;
  int s = 0;
  while (!(d & 1)) { d >>= 1; ++s; }
  for (u64 b : B) {
    u64 x = h_powmod(b, d, n);
    if (x == 1 || x == n - 1) continue;
    bool witness = true;
    for (int r = 1; r < s && witness; ++r) {
      x = h_mulmod(x, x, n);
      if (x == n - 1) witness = false;
    }
    if (witness) return false;
  }
  return true;
}

uint32_t h_bitrev(uint32_t x, uint32_t bits) {
  uint32_t r = 0;
  for (uint32_t i = 0; i < bits; ++i, x >>= 1) r = (r << 1) | (x & 1);
  return r;
}

bool Params::init(uint32_t N_, uint32_t wb, uint32_t bs, uint32_t ml, uint32_t al, std::string &err) {
  if (N_ < 16 || (N_ & (N_ - 1)) || N_ > (1u << 16)) { err = "N must be a power of two in [16, 65536]"; return false; }
  if (wb < 20 || wb > 36) { err = "elementBitWidth must be in [20, 36] (FP64 datapath, see modarith.cuh)"; return false; }
  if (ml == 0 || al == 0) { err = "maxLevel and alpha must be positive"; return false; }
  if (ml + al > 512) { err = "maxLevel + alpha > 512 not supported"; return false; }
  if (bs == 0 || N_ % bs) { err = "batchSize must divide N"; return false; }
  N = N_; word_bits = wb; batch_size = bs; max_level = ml; alpha = al;
  logN = 0;
  while ((1u << logN) < N) ++logN;
  const u64 step = 2ull * N, top = 1ull << wb, floor_ = 1ull << (wb - 1);
  mod.clear();
  for (u64 c = ((top - 2) / step) * step + 1; c > floor_ && mod.size() < n_mod(); c -= step)
    if (h_is_prime(c)) mod.push_back(c);
  if (mod.size() < n_mod()) { err = "not enough primes = 1 (mod 2N) below 2^elementBitWidth"; return false; }
  psi.resize(n_mod()); psi_inv.resize(n_mod()); n_inv.resize(n_mod());
  for (uint32_t i = 0; i < n_mod(); ++i) {
    const u64 m = mod[i];
    u64 root = 0;
    for (u64 x = 2; x < m && !root; ++x) {
      u64 c = h_powmod(x, (m - 1) / step, m);
      if (h_powmod(c, N, m) == m - 1) root = c;  // c^N = -1 <=> order exactly 2N
    }
    psi[i] = root;
    psi_inv[i] = h_invmod(root, m);
    n_inv[i] = h_invmod(N % m, m);
  }
  return true;
}

void Params::twiddles(uint32_t mi, bool inverse, std::vector<u64> &out) const {
  out.resize(N);
  const u64 m = mod[mi], base = inverse ? psi_inv[mi] : psi[mi];
  u64 pw = 1;
  for (uint32_t e = 0; e < N; ++e) {
    out[h_bitrev(e, logN)] = pw;
    pw = h_mulmod(pw, base, m);
  }
}

u64 Params::p_inv(uint32_t i) const {
  const u64 q = mod[i];
  u64 P = 1;
  for (uint32_t j = 0; j < alpha; ++j) P = h_mulmod(P, mod[max_level + j] % q, q);
  return h_invmod(P, q);
}

u64 Params::modup_scale(uint32_t L, uint32_t i) const {
  const uint32_t lo = i / alpha * alpha, hi = lo + digit_size(L, i / alpha);
  const u64 q = mod[i];
  u64 hat = 1;
  for (uint32_t t = lo; t < hi; ++t)
    if (t != i) hat = h_mulmod(hat, mod[t] % q, q);
  return h_mulmod(n_inv[i], h_invmod(hat, q), q);
}

u64 Params::moddown_scale(uint32_t j) const {
  const u64 q = mod[max_level + j];
  u64 hat = 1;
  for (uint32_t t = 0; t < alpha; ++t)
    if (t != j) hat = h_mulmod(hat, mod[max_level + t] % q, q);
  return h_mulmod(n_inv[max_level + j], h_invmod(hat, q), q);
}

u64 Params::ql_inv(uint32_t L, uint32_t l) const { return h_invmod(mod[L - 1] % mod[l], mod[l]); }

void make_bconv_table(const Params &p, const std::vector<uint32_t> &src, const std::vector<uint32_t> &dst, BConvTable &out) {
  out.src = src; out.dst = dst;
  const size_t ns = src.size(), nd = dst.size();
  out.hat_inv.assign(ns, 0);
  out.hat.assign(ns * nd, 0);
  for (size_t i = 0; i < ns; ++i) {
    const u64 si = p.mod[src[i]];
    u64 a = 1;
    for (size_t j = 0; j < ns; ++j)
      if (j != i) a = h_mulmod(a, p.mod[src[j]] % si, si);
    out.hat_inv[i] = h_invmod(a, si);
    for (size_t t = 0; t < nd; ++t) {
      const u64 m = p.mod[dst[t]];
      u64 b = 1;
      for (size_t j = 0; j < ns; ++j)
        if (j != i) b = h_mulmod(b, p.mod[src[j]] % m, m);
      out.hat[i * nd + t] = b;
    }
  }
}

}  // namespace hml
