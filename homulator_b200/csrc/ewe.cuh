// Element-wise (EWE), automorphism and base-conversion kernels.  sm_100a, FP64 datapath (modarith.cuh).
//
// Reference instruction classes executed here:
//   MULT         InsGen::GenEWE   reference src/InsGen.cpp:77-125   (unit EWE,   src/Components.cpp:8-169)
//   AUTO         InsGen::GenAUTO  reference src/InsGen.cpp:46-71    (unit AUTOU, src/Components.cpp:173-266)
//   BCONV_STEP2  InsGen::GenBCONV reference src/InsGen.cpp:263-313  (unit BCONVU, src/Components.cpp:268-362)
#pragma once
#include <vector>

#include "modarith.cuh"
#include "ntt.cuh"

namespace hml {

// out = x1*x2 (+|-) x3*x4 per limb; null operands as in hml_ewe().  All [n_limbs][N].  n_comp > 1 runs the components
// of a ciphertext op in one launch: operand k advances by comp_strides[k] words per component (x1, x2, x3, x4, out;
// 0 repeats a plaintext).
void launch_ewe(const ModConst *mc, const LimbMap &lm, int N, int n_limbs, const u64 *x1, const u64 *x2, const u64 *x3,
                const u64 *x4, int subtract, u64 *out, cudaStream_t s, int n_comp = 1, const long long *comp_strides = nullptr);

// TensorCompute (reference src/Operation.cpp:592-739): d0 = a0*b0, d1 = a0*b1 + a1*b0, d2 = a1*b1; limbs 0..L-1
// n_batch ciphertext pairs: inputs advance by in_stride words per pair, outputs by out_stride.
// pack01: d0 and d1 are stored as packed limbs (modarith.cuh), d2 always as words.
void launch_tensor3(const ModConst *mc, int N, int L, const u64 *a0, const u64 *a1, const u64 *b0, const u64 *b1,
                    u64 *d0, u64 *d1, u64 *d2, int n_batch, long long in_stride, long long out_stride, cudaStream_t s, int pack01 = 0);

// Key-switch inner product (reference src/Operation.cpp:294-414, emitted as MULT) over n_ext extended limbs:
//   acc[c][e] = sum_j t_j[e] * evk[j][c][lm.pos[e]],   modulus lm.mod[e]
// t_j[e] is d[e] (the untouched evaluation-form input) when digit j owns limb e (j == lm.skip[e]), else ext[j][e].
struct InnerArgs {
  const u64 *d;     // [>= number of owned Q-limbs][N]
  const u64 *ext;   // [beta][n_ext][N]
  const u64 *evk;   // [beta][2][evk_limbs][N]
  int evk_packed;   // the key's limb slots hold packed limbs (hml_key_pack: 5 of every 8 bytes are read)
  u64 *acc;         // [2][n_ext][N]
  int N, n_ext, beta, evk_limbs;   // beta <= 8
  int n_batch;                     // ciphertexts sharing the key: d / ext / acc advance by the strides below
  long long d_batch_stride, ext_batch_stride, acc_batch_stride;
  long long acc_comp_stride;       // words between the two accumulators of a ciphertext (0 = n_ext * N)
  int ext_f64;                     // 1: `ext` holds the forward NTT's raw signed doubles (NttLaunch::out_f64), |v| < 2^41
  int acc_pack_limbs;              // the accumulators of extended limbs e < acc_pack_limbs are stored as packed limbs
  // hoisted rotations: galois != 0 applies the automorphism X -> X^galois to every digit ON LOAD (t_j[k] is read at the
  // slot k' the automorphism kernel would have fetched, 2*brv(k')+1 = galois*(2*brv(k)+1) mod 2N), so one ModUp serves many
  // rotations and the rotated digits never exist in memory.  The key is read in place.
  unsigned galois;
  int logN;
  // hmult's merged ModDown + Rescale (context.cu, hmult_run): for extended limb e == u_limb the kernel ALSO stores
  //   u_c = acc_c[e] * u_cst + u_add_c[e]   (canonical words)   into limb slot u_slot of accumulator c,
  // u_add_c = u_add + c * u_add_comp_stride + b * u_add_batch_stride (packed limbs).  u_limb < 0: off.
  int u_limb, u_slot;
  const u64 *u_add;
  long long u_add_comp_stride, u_add_batch_stride;
  double2 u_cst;
  // the batched hmult's tensor product (context.cu, hmult_run), n_batch > 1 and ct_a != null: the launch covers Q-limbs
  // only; the kernel reads the ciphertext pair instead of d and forms d0 = a0*b0, d1 = a0*b1 + a1*b0 and d2 = a1*b1
  // itself.  d2 is the own-digit term, and the stored accumulators are acc_c + d_c * P mod q_e
  // (tensor_pmod[e] = (P mod q_e, RN(that / q_e))), so a consumer's acc * P^-1 already holds the d_c term.
  // a_c = ct_a + b * ct_batch_stride + c * ct_comp_stride (limb slots of N words), likewise b_c.  d is not read.
  const u64 *ct_a, *ct_b;
  long long ct_comp_stride, ct_batch_stride;
  const double2 *tensor_pmod;
};
// n_limbs > 0: only the extended limbs e < n_limbs of lm (grid.y = n_limbs instead of n_ext)
void launch_inner_product(const ModConst *mc, const LimbMap &lm, const InnerArgs &a, cudaStream_t s, int n_limbs = 0);

// The same inner product for up to IP_MAX_ROT hoisted rotations of one ciphertext in ONE launch (grid.z = rotation): every
// rotation reads the same digits d / ext, through its own automorphism (as InnerArgs::galois), and multiplies them by its own
// key (8-byte words).  Rotation r writes acc + r * acc_rot_stride, [2][n_ext][N] words.  The digits of one launch are read
// from L2 after the first rotation.
constexpr int IP_MAX_ROT = 16;
struct InnerRotArgs {
  const u64 *d;                    // [>= number of owned Q-limbs][N], read through the automorphism like ext
  const u64 *ext;                  // [beta][n_ext][N]
  u64 *acc;
  long long acc_rot_stride;
  int N, n_ext, beta, evk_limbs, logN;  // beta <= 8
  int ext_f64;                     // as InnerArgs::ext_f64
  const u64 *evk[IP_MAX_ROT];      // [beta][2][evk_limbs][N] per rotation
  unsigned galois[IP_MAX_ROT];     // galois element mod 2N per rotation; 0 = identity
};
void launch_inner_product_rot(const ModConst *mc, const LimbMap &lm, const InnerRotArgs &a, int n_rot, cudaStream_t s);

// Double-hoisted rotation sum (context.cu, hrot_sum_hoisted_run): the inner product of up to IP_MAX_ROT rotations of one
// ciphertext, each weighted by its plaintext in the extended basis and summed before any ModDown.  One thread serves one
// coefficient pair of extended limb e (grid (N/2/256, n_ext)) and loops over the rotations r < n_rot:
//   acc[c][e] (+)= sum_r pt_r[e] * sum_j sigma_r(t_j)[e] * evk_r[j][c][lm.pos[e]]        (words, [2][n_ext][N])
//   z[e]      (+)= sum_r pt_r[e] * sigma_r(c0)[e]                          for e < L      (words, [L][N])
// t_j as in InnerArgs (d for the digit's own limbs, else ext), read through sigma_r like InnerRotArgs.  pt_r[e] is row
// e < L ? e : pt_q_limbs + (e - L) of pt[r].  accumulate = 1 adds to what acc / z hold (the later groups of one op).
struct InnerRotSumArgs {
  const u64 *d;                    // [>= number of owned Q-limbs][N] (c1)
  const u64 *ext;                  // [beta][n_ext][N]
  const u64 *c0;                   // [L][N]
  u64 *acc, *z;
  int N, n_ext, L, beta, evk_limbs, pt_q_limbs, logN;  // beta <= 8
  int ext_f64;                     // as InnerArgs::ext_f64
  int evk_packed;                  // as InnerArgs::evk_packed
  int accumulate, n_rot;           // n_rot <= IP_MAX_ROT
  const u64 *evk[IP_MAX_ROT];      // [beta][2][evk_limbs][N] per rotation
  const u64 *pt[IP_MAX_ROT];       // [pt_q_limbs + alpha][N] per rotation
  unsigned galois[IP_MAX_ROT];     // galois element mod 2N per rotation; 0 = identity
};
void launch_inner_product_rot_sum(const ModConst *mc, const LimbMap &lm, const InnerRotSumArgs &a, cudaStream_t s);

// The two inner products of a double-hoisted baby-step / giant-step linear transform (context.cu, hrot_bsgs_hoisted_run), as
// InnerRotSumArgs with:
//   baby  (giant = false): an entry with evk[r] == null is the identity without a key switch.  It loads no digit and no key
//         and adds pt_r[e] * c0[e] to z and pt_r[e] * d[e] (c1) to z1, on the Q-limbs only.  z1 is stored like z.
//   giant (giant = true):  no plaintext is read and the sums are unweighted, acc (+)= sum_j sigma_r(t_j) * evk_r[j],
//         z (+)= sigma_r(c0); z1 is not touched.
struct InnerBsgsArgs : InnerRotSumArgs {
  u64 *z1;                         // [L][N] (baby only)
};
void launch_inner_product_bsgs(const ModConst *mc, const LimbMap &lm, const InnerBsgsArgs &a, bool giant, cudaStream_t s);

// A sum of up to IP_MAX_ROT tensor products (context.cu, hmult_sum_run and shard_tensor_sum), L limb slots, grid
// (N/2/256, L, n_batch):
//   d0 (+)= sum_k a_k0*b_k0,   d1 (+)= sum_k (a_k0*b_k1 + a_k1*b_k0),   d2 (+)= sum_k a_k1*b_k1        k < n_pairs
// a[k] / b[k] are [n_batch][2][L][N]: component c at + c * comp_stride, batch entry z at + z * in_stride; d0 / d1 / d2 advance
// by out_stride per batch entry.  Limb slot l has modulus q_{mod0 + l * mod_step}: 0 and 1 for a whole ciphertext, rank and
// world for a limb-sharded one.  A pair with a[k] == b[k] (a square) loads one ciphertext.  The outputs have launch_tensor3's
// formats (pack01: d0 / d1 packed limbs); accumulate = 1 adds to what d0 / d1 / d2 hold (the later groups of one op).
struct TensorSumArgs {
  const u64 *a[IP_MAX_ROT], *b[IP_MAX_ROT];
  u64 *d0, *d1, *d2;
  long long comp_stride, in_stride, out_stride;
  int N, n_pairs, accumulate, pack01;
  int mod0, mod_step;
};
void launch_tensor_sum(const ModConst *mc, int L, int n_batch, const TensorSumArgs &a, cudaStream_t s);

// out = (x - y) * c (+ z) per limb:  ModDownSub (+ HMULT add)  reference src/Operation.cpp:548-590, :967-1005
// and Rescale sub+mul  reference src/Operation.cpp:825-911.  cst[limb] = (c, RN(c/q)).  n_polys via strides.
struct SubMulArgs {
  const u64 *x, *y, *z;   // y and z may be null (y = 0: out = x * c + z)
  u64 *out;
  long long x_poly_stride, y_poly_stride, z_poly_stride, out_poly_stride;
  const double2 *cst;     // [n_limbs]
  int N, n_limbs, n_polys;
  int x_packed, z_packed; // x / z hold packed limbs (modarith.cuh)
  unsigned z_mask;        // 0: z is added for every poly; else only for the polys whose bit is set (poly < 32)
};
void launch_sub_mul_add(const ModConst *mc, const LimbMap &lm, const SubMulArgs &a, cudaStream_t s);

// out[k] = in[k'],  2*brv(k')+1 = g*(2*brv(k)+1) mod 2N, for n_limbs limbs
void launch_automorph(int logN, int n_limbs, const u64 *in, u64 *out, u64 g, cudaStream_t s);

// words [n_limbs][N] -> packed limbs inside slots of the same size (modarith.cuh st_packed2); out must not overlap in
void launch_pack_limbs(int N, size_t n_limbs, const u64 *in, u64 *out, cudaStream_t s);

// Fast base conversion.  in [n_src][N] coefficient form.  If step1 != nullptr the per-source scaling
// y_i = in_i * hat_inv_i mod s_i is applied inside (step1[i] = (hat_inv_i, RN(hat_inv_i / s_i)));
// otherwise `in` must already hold y_i (the fused pipeline folds it into the preceding INTT).
// The matrix (D/s_i mod t), split into three 12-bit pieces as doubles, lives in device memory, zero-padded:
//   mat[(i * n_dst_pad + t) * 3 + k],  i < n_src_pad = bconv_pad_src(n_src),  t < n_dst_pad = bconv_pad_dst(n_dst)
struct BConvArgs {
  const u64 *in;
  u64 *out;
  long long in_batch_stride, out_batch_stride;  // grid.y batches (e.g. the two key-switch accumulators)
  const double2 *step1;   // [n_src] or null
  int N, n_src, n_dst, n_batches;
  // optional pre-pass on the staged tile (hmult's merged ModDown + Rescale, context.cu): the LAST source row is replaced by
  //   row_last + sum_{i < n_src-1} y_i * fold_i   mod q_{fold_mod}   (canonical)
  // before the conversion; fold = [n_src-1][3] 12-bit pieces of the per-source constants, or null
  const double *fold;
  int fold_mod;
  // 1: store the centred remainder as a double (|v| <= q/2) instead of the canonical word — the hand-off format to a
  // forward NTT launched with NttLaunch::in_f64 (saves the canonicalisation here and the integer -> double conversion there)
  int out_f64;
  // optional (tcgen05 kernel only): word offset of every source limb relative to `in`, replacing src_lm.pos[i] * N.  The
  // limb-sharded key switch points these at the PEER GPUs' buffers (NVLink loads inside the conversion, no all-gather).
  const long long *src_off;   // device array [n_src] or null
};
// int8 operand image of a conversion matrix for the tcgen05 path (bconv_umma.cu): img == null -> the DMMA kernel runs
struct BConvImage {
  const uint8_t *img = nullptr;   // device, K * NP bytes in the kernel's shared-memory layout
  int K = 0, NP = 0, ND = 0, n16 = 0, fold = 0;
};
// One conversion of a multi-conversion launch (tcgen05 kernel): everything that differs between the conversions lives in a
// device-resident table built once (context.cu), so the three ModUp digits of a key switch run as ONE launch — CTA c serves
// job c % n_jobs for its whole life (per-CTA matrix image, target table and source offsets stay constant).
struct BConvJob {
  uint16_t src_pos[48];       // limb slot of source i inside the job's input (relative to in + in_off)
  uint16_t dst_mod[48], dst_pos[48];
  const uint8_t *img;         // operand image (device)
  int K, NP, ND;
  int n_src, n_dst;
  long long in_off, out_off;  // words, added to BConvArgs::in / out
  const long long *src_off;   // optional device array [n_src]: word offset of every source relative to BConvArgs::in (peer buffers)
};
// host: eligibility (n_src <= 48, 5 * pad8(n_dst + fold) <= 256) and image construction; see bconv_umma.cu
bool bconv_image_shape(int n_src, int n_dst, int fold, BConvImage &im);
bool bconv_image_build(const u64 *hat, int n_src, int n_dst, const u64 *dst_q, const u64 *fold, u64 fold_q, std::vector<uint8_t> &img,
                       BConvImage &im);
void launch_bconv_umma(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const BConvImage &im, cudaStream_t s);
// n_jobs conversions in one launch: `a` carries what they share (N, n_batches, batch strides, out_f64; in / out are the bases the
// jobs' offsets are added to; no step 1, no fold, no peer offsets), d_jobs the device table, ims the host copies of the image
// shapes.  Returns false (nothing launched) when the jobs cannot share a launch (different slab counts, N % 128 != 0).
bool launch_bconv_umma_multi(const ModConst *mc, const BConvJob *d_jobs, const BConvImage *ims, const int *n_dst, int n_jobs, const BConvArgs &a,
                             cudaStream_t s);
// HML_BCONV_UMMA=0 keeps every conversion on the DMMA kernel
int bconv_umma_enabled();
inline int bconv_pad_src(int n_src) { return (n_src + 3) & ~3; }   // k-steps of 4 sources
inline int bconv_pad_dst(int n_dst) { return (n_dst + 7) & ~7; }   // target blocks of 8 (one warp each); n_dst <= 128
// Source limb i is read at in + src_lm.pos[i] * N (modulus src_lm.mod[i], used by step 1 only); output limb t is
// written at out + dst_lm.pos[t] * N with modulus dst_lm.mod[t].  N >= 16.
// `im` (optional): the same matrix as an int8 operand image; when it is usable for this launch (N a multiple of 128,
// image built with / without the fold as the launch asks) the conversion runs on tcgen05 (bconv_umma.cu) instead.
void launch_bconv(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const double *mat, cudaStream_t s,
                  const BConvImage *im = nullptr);

}  // namespace hml
