// RNS-CKKS parameter set on the host: moduli, roots of unity, NTT twiddle tables and the per-level
// base-conversion constants.  The reference has none of this (it never computes values); the rules
// are those of SURVEY.md Appendix A and are restated independently by oracle/oracle.c.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace hml {

typedef unsigned long long u64;

u64 h_mulmod(u64 a, u64 b, u64 m);
u64 h_powmod(u64 a, u64 e, u64 m);
u64 h_invmod(u64 a, u64 m);  // m prime
bool h_is_prime(u64 n);
uint32_t h_bitrev(uint32_t x, uint32_t bits);

struct Params {
  uint32_t N = 0, logN = 0, word_bits = 0, batch_size = 0, max_level = 0, alpha = 0;
  uint32_t bconv_high = 2, bconv_width = 6;  // reference config_4.cfg:36-37 defaults
  std::vector<u64> mod;      // q_0..q_{maxLevel-1}, p_0..p_{alpha-1}
  std::vector<u64> psi;      // primitive 2N-th root per modulus
  std::vector<u64> psi_inv;
  std::vector<u64> n_inv;

  uint32_t n_mod() const { return max_level + alpha; }
  uint32_t beta(uint32_t L) const { return (L + alpha - 1) / alpha; }
  uint32_t digit_size(uint32_t L, uint32_t j) const { uint32_t r = L - j * alpha; return r > alpha ? alpha : r; }
  // modulus index of extended-basis limb e at level L: (q_0..q_{L-1}, p_0..p_{alpha-1})
  uint32_t ext_mod(uint32_t L, uint32_t e) const { return e < L ? e : max_level + (e - L); }

  // Generates moduli and roots.  Moduli: all primes = 1 (mod 2N) in (2^(w-1), 2^w), scanned downward.
  // psi: x^((q-1)/2N) for the smallest x >= 2 where that power has order exactly 2N.
  bool init(uint32_t N, uint32_t word_bits, uint32_t batch_size, uint32_t max_level, uint32_t alpha, std::string &err);

  // psi^bitrev(i) (forward) or psi^-bitrev(i) (inverse), i < N, for modulus index mi
  void twiddles(uint32_t mi, bool inverse, std::vector<u64> &out) const;

  // Constants of the key switch and the rescale at level L (SURVEY.md Appendix A), P = p_0 * .. * p_{alpha-1}:
  u64 p_inv(uint32_t i) const;                    // P^-1 mod q_i
  u64 modup_scale(uint32_t L, uint32_t i) const;  // N^-1 * (D_j / q_i)^-1 mod q_i, D_j the product of the digit j = i / alpha
  u64 moddown_scale(uint32_t j) const;            // N^-1 * (P / p_j)^-1 mod p_j
  u64 ql_inv(uint32_t L, uint32_t l) const;       // q_{L-1}^-1 mod q_l
};

// Base-conversion constants for source moduli S (product D) and destination moduli T:
//   hat_inv[i]  = (D/s_i)^-1 mod s_i            (step 1)
//   hat[i][t]   = (D/s_i) mod T_t               (step 2), row-major [n_src][n_dst]
struct BConvTable {
  std::vector<uint32_t> src, dst;
  std::vector<u64> hat_inv;
  std::vector<u64> hat;
};
void make_bconv_table(const Params &p, const std::vector<uint32_t> &src, const std::vector<uint32_t> &dst, BConvTable &out);

}  // namespace hml
