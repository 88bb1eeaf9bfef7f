// Internal (non-ABI) interface of context.cu: the op compositions and helpers that shard.cu / replay.cu / hostpath.cu build on.
#pragma once
#include <string>

#include "context.h"

#define HML_CU_TRY(ctx, call)                                                                      \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                             \
      return HML_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)

int fail(hml_ctx *ctx, int code, const std::string &msg);
int ensure_ws(hml_ctx *ctx, size_t words);
int check_level(hml_ctx *ctx, uint32_t L, uint32_t min_level);
int shard_check(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world);

// A galois element mod 2N, and the inner-product kernels' form of it: 0 for the identity (InnerArgs::galois)
inline unsigned galois_mod(uint64_t g, size_t N) { return (unsigned)(g & (2ull * N - 1)); }
inline unsigned inner_galois(uint64_t g, size_t N) { const unsigned r = galois_mod(g, N); return r == 1 ? 0 : r; }

size_t hmult_ws_words(const hml::Params &p, uint32_t L, uint32_t nb);
size_t hrot_ws_words(const hml::Params &p, uint32_t L, uint32_t nb);

int hmult_run(hml_ctx *ctx, uint32_t L, uint32_t nb, const hml::u64 *ct_a, const hml::u64 *ct_b, const hml::u64 *evk, uint32_t evk_q_limbs,
              hml::u64 *ct_out, hml::u64 *ws, cudaStream_t s);
int hrot_run(hml_ctx *ctx, uint32_t L, uint32_t nb, const hml::u64 *ct, const hml::u64 *rk, uint32_t evk_q_limbs, hml::u64 g, hml::u64 *ct_out,
             hml::u64 *ws, cudaStream_t s);

// limb-sharded building blocks beyond the ABI's phase entry points (shard.cu)
// peer-direct ModDown of accumulator pair r of a hoisted group of H (r = 0, H = 1: the key switch), sources from slot r
// (slot_words apart) of the owners' gather buffers 2, plus the addends (add0 read through add0_galois when it is not 0)
int shard_end_p2p(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers2, uint64_t *out0_own,
                  uint64_t *out1_own, const uint64_t *add0_own, const uint64_t *add1_own, cudaStream_t s, uint32_t r = 0, uint32_t H = 1,
                  size_t slot_words = 0, uint64_t add0_galois = 0);
int shard_prepare(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers1, const uint64_t *const *peers2,
                  uint32_t max_rot);
// hoisted rotations of one sharded ciphertext, H = the shard's rotation capacity (context.cu)
int shard_hoist_inner(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t H, const uint64_t *const *peers1, const uint64_t *c1_own,
                      uint32_t n, const uint64_t *const *keys, const uint64_t *galois, cudaStream_t s);
int shard_hoist_intt(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t n, uint64_t *g2_own, size_t slot_words, cudaStream_t s);
// the sharded sums' limb-local stages (context.cu): the rotation sum's ModUp + weighted inner product (z_own [nq][N] = the c0
// term), and the product sum's tensor-product sum into d0 | d1 | d2 [nq][N]
int shard_rot_sum_inner(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers1, const uint64_t *ct_own,
                        uint32_t n_rot, const uint64_t *const *keys, const uint64_t *galois, const uint64_t *const *pts, uint64_t *z_own,
                        cudaStream_t s);
int shard_tensor_sum(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t n, const uint64_t *const *a_own,
                     const uint64_t *const *b_own, uint64_t *d0, uint64_t *d1, uint64_t *d2, cudaStream_t s);
