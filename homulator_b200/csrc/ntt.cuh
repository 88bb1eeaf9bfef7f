// Negacyclic NTT / inverse NTT per RNS limb on B200 (sm_100a), FP64 datapath (see modarith.cuh).
//
// Executes the reference's NTT / INTT instruction classes (InsGen::GenNTT, reference
// src/InsGen.cpp:17-44; simulated unit NTTU, reference src/Components.cpp:380-569 — which is itself a
// two-phase + transpose structure, :397-431) on real data.
//
// Algorithm: merged-psi Cooley-Tukey (forward, natural in -> bit-reversed out) / Gentleman-Sande
// (inverse), split 4-step style into TWO passes over 4096-point tiles (256 threads x 16 points):
//   forward  pass 1 "columns": the first log2(R1) stages couple elements R2 apart (R2 = 256, R1 = N/256);
//            a CTA owns C = 4096/R1 adjacent columns (>= 128 B contiguous per row -> full-line accesses).
//   forward  pass 2 "rows":    the last 8 stages stay inside contiguous 256-element rows; a CTA owns 16 rows.
//   inverse  = the mirror image (rows first, then columns).
// Every thread keeps 16 points in registers and runs FOUR radix-2 stages per round (one 16-point network with
// a 15-entry twiddle heap), so a pass needs a single exchange through shared memory.  Tiles reach shared
// memory by asynchronous 16-byte copies (cp.async), double buffered: the next tile / item is in flight while
// the current one is transformed.  Twiddles are single doubles (the quotient estimate uses 1/q, see
// mulmod_var); the row pass reads them from a per-tile blob laid out for conflict-free vector loads
// (ntt_permute_row_twiddles) that arrives by ONE bulk copy (TMA engine) per CTA.
// The buffer between the passes holds raw signed-lazy doubles (no conversion / reduction cost).
#pragma once
#include "modarith.cuh"

namespace hml {

constexpr int NTT_TILE = 4096;     // elements per CTA tile
constexpr int NTT_THREADS = 256;   // 16 elements per thread
constexpr int NTT_ROW_LOG = 8;     // R2 = 256: contiguous row length handled by the row pass
constexpr int NTT_SMALL_LOG = 12;  // N <= 4096: one CTA per limb, all stages in shared memory
constexpr int NTT_MAX_LIMBS = 128; // limbs (x polys) per launch

struct LimbMap {
  uint16_t mod[NTT_MAX_LIMBS];  // modulus index of each limb of the launch
  uint16_t pos[NTT_MAX_LIMBS];  // NTT launches: limb slot inside the buffer (address = base + pos * limb_stride)
  uint8_t skip[NTT_MAX_LIMBS];  // NTT launches: poly index NOT to transform for this limb (0xFF = none); used by
                                // ModUp, where digit j's own limbs stay as they are
};

// Twiddle tables, one double per entry (w = psi^(+-bitrev)), per modulus N entries.
//   fwd / inv          natural "heap" order: the butterflies of stage s, group g use entry (1 << s) + g
//   fwd_rows/inv_rows  the same values permuted per 16-row tile for the row pass (null when N <= 4096)
struct NttTables {
  const double *fwd, *inv;            // [n_mod][N]
  const double *fwd_rows, *inv_rows;  // [n_mod][N / 4096][4096]
  const ModConst *mc;                 // [n_mod]
  // tile queue of the column passes (ntt.cu, ColQueue): two zero-initialised words; null: static split.  Launches that may run
  // CONCURRENTLY need distinct counters.
  unsigned *col_ctr;
};

// Host: permute one modulus' natural table (N entries) into the row-pass layout.  Per 16-row tile (rows r = 16 *
// tile + rr, thread slot ts = rr * 16 + l) a 4096-entry blob:
//   [   0 +  rr*16 + h ]            h = 1..15: heap of the row's first four stages (t = 128..16), h = (1 << s) + g
//   [ 256 +  ts ]                   stage 4 (t = 8):  entry ((R1 + r) << 4) + l
//   [ 512 +  ts*2 + x ]             stage 5 (t = 4):  entry ((R1 + r) << 5) + 2l + x
//   [1024 + k*512 + ts*2 + x ]      stage 6 (t = 2):  entry ((R1 + r) << 6) + 4l + 2k + x,  k < 2
//   [2048 + k*512 + ts*2 + x ]      stage 7 (t = 1):  entry ((R1 + r) << 7) + 8l + 2k + x,  k < 4
// so that every 16-byte load instruction of a warp covers 512 contiguous bytes.
void ntt_permute_row_twiddles(const double *nat, int logN, double *out);

// Optional fused epilogue of a FORWARD transform (ModDownSub + add, reference src/Operation.cpp:548-590, :967-1005, and
// Rescale sub + mul, :825-911): instead of storing y = NTT(in) the row pass writes
//   dst = (x - y) * cst[limb] (+ z)              mod q, canonical,      or, when cst2 is given (merged ModDown + Rescale
//   dst = ((x * cst[limb] + z) - y) * cst2[limb]  mod q, canonical       of hmult, see context.cu),
// so the transform's output never round-trips HBM.  Items are (b, c) = (idx / n_c, idx % n_c) with idx the launch's
// poly index (n_batch must be 1); every operand is addressed as base + c * c_stride + b * b_stride + limb * N.
struct NttFuse {
  const u64 *x, *z;             // x = null: no fusion;  z may be null
  u64 *dst;
  long long x_c_stride, x_b_stride, z_c_stride, z_b_stride, dst_c_stride, dst_b_stride;
  const double2 *cst;           // [n_limbs] (c, RN(c/q))
  const double2 *cst2;          // [n_limbs] or null
  int n_c;
  unsigned z_mask;              // z is added for component c iff bit c is set
  int x_packed, z_packed;       // x / z hold packed limbs (modarith.cuh: 5 bytes per coefficient inside the 8N-byte slot)
  unsigned z_galois;            // != 0: z is read through the automorphism X -> X^g, z'[k] = z[sigma_g(k)] (hrotate's sigma(c0)
                                // addend, reference src/Operation.cpp:1302-1319 + :1339-1357; z must hold plain words).  In
                                // evaluation order the automorphism maps every 256-slot row onto ONE source row (RowSigma)
};

// Optional key-switch inner product fused into the ModUp transform's row pass — the GPU counterpart of the reference's HPIP
// unit, which multiplies the transformed digits by the key as they leave the NTT (InsGen::GenHPIP reference src/InsGen.cpp:356-406,
// unit HPIP src/Components.cpp:571-668; inner product itself: KeySwitch::InnerProduceOperation src/Operation.cpp:294-414).
// The launch transforms the beta extended digits (polys) of n_batch ciphertexts; instead of storing NTT(t_j)[e] the row pass
// accumulates   acc_c[b][e] (+)= NTT(t_j)[e] * evk[j][c][key_pos[e]]   for c = 0, 1, so the transformed digits never reach
// memory.  The member of (b, e) with the smallest digit index starts the sum (and adds the own-digit term
// d[b][e] * evk[own][c][..] when e is a Q-limb), the others read-modify-write the 8-byte accumulator slots (lazy doubles,
// L2-resident between members: one CTA handles all members of a (b, e, tile)), the last one stores canonical words.
struct NttMac {
  const u64 *evk;               // [beta][2][evk_limbs][N]; null: no fusion
  int evk_packed;               // the key's limb slots hold packed limbs (hml_key_pack)
  const u64 *d;                 // the untouched evaluation-form input, [>= L][N] per ciphertext
  u64 *acc;                     // accumulators [n_batch][2][..][N], 8-byte slots
  long long d_batch_stride, acc_batch_stride, acc_comp_stride;
  int evk_limbs;
  uint16_t key_pos[NTT_MAX_LIMBS];
  // hmult's merged ModDown + Rescale: see InnerArgs::u_limb
  int u_limb, u_slot;
  const u64 *u_add;
  long long u_add_comp_stride, u_add_batch_stride;
  double2 u_cst;
};

// ---- launch descriptors (host side, ntt.cu)
struct NttLaunch {
  const u64 *in;        // [n_polys][n_limbs][N] (poly stride / limb stride in elements below)
  u64 *out;
  long long in_poly_stride, in_limb_stride;    // in_limb_stride = 0 broadcasts one source limb (rescale)
  long long out_poly_stride, out_limb_stride;
  int n_limbs, n_polys;
  int n_batch;                                  // independent ciphertexts: item (b, p) lives at base + b * batch_stride + p * poly_stride
  long long in_batch_stride, out_batch_stride;
  // inverse only: per-limb post-scale constant c (folded with N^-1 on the host): out = INTT(in) * c, canonical.
  const double2 *post_scale;  // [n_limbs] (c*ninv mod q, RN(that / q)) or nullptr for plain N^-1
  NttFuse fuse;               // forward only
  NttMac mac;                 // forward only, two-pass rings, no fused epilogue: see NttMac (n_polys = beta, LimbMap::skip = own digit)
  // inverse only, two-pass rings, n_polys == 1: the input is read through the automorphism X -> X^in_galois (hrotate's
  // sigma(c1), the key-switch input) while the row pass loads it, and the permuted limbs are also written to side_out
  // ([n_batch] items side_batch_stride apart, limb slots like `out`) for the inner product's own-digit term.
  // in_ginv8 = in_galois^-1 mod 256.  0: plain load.
  unsigned in_galois, in_ginv8;
  u64 *side_out;
  long long side_batch_stride;
  int in_f64;                 // forward only, two-pass rings: `in` holds signed doubles |v| <= q (BConvArgs::out_f64)
  int out_f64;                // forward only, two-pass rings, no fused epilogue: leave the raw lazy sums (|v| < 10 q) as doubles
                              // in `out` instead of canonical words (consumer: InnerArgs::ext_f64)
  // inverse only, two-pass rings, n_polys == 1, no in_galois: the row pass transforms in * in_mul mod q (canonical words,
  // same limb and batch strides as `in`) — the batched hmult squares its ciphertexts' c1 (d2 = a1 * b1) on load.  null: off.
  const u64 *in_mul;
};

void launch_ntt_forward(const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s);
void launch_ntt_inverse(const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s);

}  // namespace hml
