// Internal (non-ABI) interface of context.cu: the op compositions and helpers that shard.cu / replay.cu build on.
#pragma once
#include <string>

#include "context.h"

// Strided view of `nb` independent polynomials / ciphertext halves: item b lives at ptr + b * stride (words).
struct BatchPtr {
  const hml::u64 *ptr;
  long long stride;
};
struct BatchOut {
  hml::u64 *ptr;
  long long stride;
};

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
int check_launch(hml_ctx *ctx, const char *what);
int check_level(hml_ctx *ctx, uint32_t L, uint32_t min_level);
void clear_map(hml::LimbMap &lm);
void id_map(hml::LimbMap &lm, const uint32_t *mod_idx, uint32_t n);
int get_level(hml_ctx *ctx, uint32_t L, hml::LevelConsts **out);
int get_shard_plan(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, hml::ShardPlan **out);
int shard_check(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world);

size_t ks_ws_words(const hml::Params &p, uint32_t L);
size_t rs_ws_words(const hml::Params &p, uint32_t L, uint32_t n_polys);
size_t hmult_ws_words(const hml::Params &p, uint32_t L, uint32_t nb);
size_t hrot_ws_words(const hml::Params &p, uint32_t L, uint32_t nb);
size_t shard_ws_words(const hml::Params &p, const hml::ShardPlan &sp);

// hrotate on two-pass rings: the automorphism rides on the key switch's loads instead of a kernel of its own.  d and add0 are
// the RAW polynomials; the ModUp INTT reads d through sigma_g and leaves sigma_g(d) in sigma_d (item b at + b * sigma_stride)
// for the inner product's own-digit term; the ModDown epilogue reads add0 through sigma_g.
struct KsAuto {
  hml::u64 g;
  hml::u64 *sigma_d;
  long long sigma_stride;
};

// hmult's merged ModDown + Rescale: the addend d_c[L-1] of u[L-1] = acc_c[L-1] * P^-1 + d_c[L-1] (packed limbs; component c at
// add + c * comp_stride, ciphertext b at + b * batch_stride)
struct MergedU {
  const hml::u64 *add;
  long long comp_stride, batch_stride;
};

// K1..K7 of nb key switches sharing one key (ModUp, inner product, INTT of the P-limbs); see context.cu
int ks_front(hml_ctx *ctx, hml::LevelConsts *lc, uint32_t L, uint32_t nb, BatchPtr d, const hml::u64 *evk, uint32_t evk_q_limbs, hml::u64 *yb,
             hml::u64 *ext, hml::u64 *acc, uint32_t AL, cudaStream_t s, const MergedU *mu = nullptr, const KsAuto *au = nullptr);
int ks_modup(hml_ctx *ctx, hml::LevelConsts *lc, uint32_t L, uint32_t nb, BatchPtr d, hml::u64 *yb, hml::u64 *ext, cudaStream_t s,
             const hml::NttMac *mac = nullptr, const KsAuto *au = nullptr);
bool ks_uses_hpip(const hml_ctx *ctx, uint32_t L, uint32_t nb);
int ks_inner(hml_ctx *ctx, hml::LevelConsts *lc, uint32_t L, uint32_t nb, BatchPtr d, const hml::u64 *evk, uint32_t evk_q_limbs, const hml::u64 *ext,
             hml::u64 *acc, uint32_t AL, hml::u64 galois, cudaStream_t s, const MergedU *mu = nullptr, bool ip_done = false);
int ks_tail(hml_ctx *ctx, hml::LevelConsts *lc, uint32_t L, uint32_t nb, hml::u64 *acc, hml::u64 *vb, BatchOut out0, BatchOut out1, BatchPtr add0,
            BatchPtr add1, cudaStream_t s, bool acc_packed, hml::u64 add0_galois = 0);
int hrot_hoisted_run(hml_ctx *ctx, uint32_t L, const hml::u64 *ct, uint32_t n_rot, const uint64_t *const *rotkeys, uint32_t evk_q_limbs,
                     const uint64_t *galois, uint64_t *const *outs, hml::u64 *ws, cudaStream_t s);
int ks_run(hml_ctx *ctx, uint32_t L, uint32_t nb, BatchPtr d, const hml::u64 *evk, uint32_t evk_q_limbs, BatchOut out0, BatchOut out1,
           BatchPtr add0, BatchPtr add1, hml::u64 *ws, cudaStream_t s, const KsAuto *au = nullptr);
int rescale_run(hml_ctx *ctx, uint32_t L, const hml::u64 *in, long long in_poly_stride, uint32_t n_polys, hml::u64 *out,
                long long out_poly_stride, hml::u64 *ws, cudaStream_t s);
int hmult_run(hml_ctx *ctx, uint32_t L, uint32_t nb, const hml::u64 *ct_a, const hml::u64 *ct_b, const hml::u64 *evk, uint32_t evk_q_limbs,
              hml::u64 *ct_out, hml::u64 *ws, cudaStream_t s);
int hrot_run(hml_ctx *ctx, uint32_t L, uint32_t nb, const hml::u64 *ct, const hml::u64 *rk, uint32_t evk_q_limbs, hml::u64 g, hml::u64 *ct_out,
             hml::u64 *ws, cudaStream_t s);

// limb-sharded building blocks beyond the ABI's phase entry points (shard.cu)
int shard_end_p2p_add(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers2, uint64_t *out0_own,
                      uint64_t *out1_own, const uint64_t *add0_own, const uint64_t *add1_own, cudaStream_t s);
int shard_prepare(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers1, const uint64_t *const *peers2,
                  uint32_t max_rot);
// hoisted rotations of one sharded ciphertext, H = the shard's rotation capacity (context.cu)
size_t shard_hoist_ws_words(const hml::Params &p, const hml::ShardPlan &sp, uint32_t H);
int shard_hoist_inner(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t H, const uint64_t *const *peers1, const uint64_t *c1_own,
                      uint32_t n, const uint64_t *const *keys, const uint64_t *galois, cudaStream_t s);
int shard_hoist_intt(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t n, uint64_t *g2_own, size_t slot_words, cudaStream_t s);
int shard_hoist_end(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t H, const uint64_t *const *peers2, size_t slot_words,
                    uint32_t r, const uint64_t *add0, uint64_t add0_galois, uint64_t *out0, uint64_t *out1, cudaStream_t s);
