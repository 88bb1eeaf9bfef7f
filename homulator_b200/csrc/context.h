// Internal definition of hml_ctx: device tables, per-level constants, workspace, op composition.
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/homulator_b200.h"
#include "config.h"
#include "ewe.cuh"
#include "ntt.cuh"
#include "params.h"

namespace hml {

// A base conversion prepared for launch: the 12-bit-split matrix in device memory (zero-padded to whole k-steps and
// target blocks, see ewe.cuh) and the destination limb map.
struct HostBConv {
  int n_src = 0, n_dst = 0;
  double *d_mat = nullptr;   // [bconv_pad_src(n_src)][bconv_pad_dst(n_dst)][3]
  uint8_t *d_img = nullptr;  // the same matrix as the tcgen05 kernel's int8 operand image (null: shape not eligible)
  BConvImage im;
  LimbMap dst_lm;
  bool empty() const { return n_dst == 0; }
};

// Per-level constants of the key-switch / rescale pipeline (SURVEY.md Appendix A "Constant tables").
struct LevelConsts {
  uint32_t L = 0, beta = 0, E = 0;
  // K1+K2 fused: INTT post-scale  N^-1 * (D_j/q_i)^-1 mod q_i  for every input limb i (digit j = i / alpha)
  double2 *modup_scale = nullptr;            // [L]
  // K3: per digit, the conversion to the E - a_j other limbs (matrix in 12-bit pieces, kernel-parameter resident)
  std::vector<HostBConv> up;                 // [beta]
  std::vector<LimbMap> up_src;               // [beta] source map of each digit's conversion (q_lm: the digit sits at yb + j * alpha)
  BConvJob *up_jobs = nullptr;               // [beta] device table of the one-launch form (null: digits launch one by one)
  // K4: limbs = the E extended limbs, polys = the beta digits, skip = the digit that owns the limb
  LimbMap ext_lm;
  // K6+K7 fused: INTT post-scale N^-1 * (P/p_j)^-1 mod p_j;  K8 matrix [alpha][L][3];  K10 constant P^-1 mod q_i
  double2 *moddown_scale = nullptr;          // [alpha]
  double2 *moddown_scale_u = nullptr;        // [alpha + 1]: the same + plain N^-1 mod q_{L-1} for hmult's extra limb (slot E)
  LimbMap pu_lm;                             // p_lm + limb alpha -> modulus q_{L-1}, pos = E
  double2 pinv_last{};                       // P^-1 mod q_{L-1} (host copy, kernel parameter of the inner product)
  HostBConv down;
  double2 *pinv = nullptr;                   // [L]
  double2 *pmod = nullptr;                   // [L]: P mod q_i (the batched hmult's tensor fold, InnerArgs::tensor_pmod)
  // Rescale: q_{L-1}^-1 mod q_l
  double2 *qlinv = nullptr;                  // [L-1]
  // hmult only (L >= 2): ModDown merged with Rescale by linearity of the NTT (context.cu, hmult_run).  Sources = the alpha
  // P-limbs of an accumulator (slots L + j) plus one extra coefficient-form limb in slot E holding INTT(u[L-1]).  The
  // conversion first folds r = slot_E - v[L-1] * P^-1 (mod q_{L-1}) on its staged tile (`merged_fold`: the constants
  // -(P/p_j mod q_{L-1}) * P^-1 in 12-bit pieces), then produces w_l = v_l * P^-1 + [r]_{q_l} for l < L-1 (`merged_rest`).
  HostBConv merged_rest;
  double *merged_fold = nullptr;             // [alpha][3]
  LimbMap merged_src, last_lm;
  LimbMap q_lm;                              // limbs 0..L-1 -> moduli q_0..q_{L-1}, pos = limb
  LimbMap p_lm;                              // limbs 0..alpha-1 -> moduli p_j, pos = L + j (inside an [E][N] buffer)
};

// Plan of the limb-sharded key switch for one (level, rank, world): owned limbs, gather-buffer positions, constants.
struct ShardPlan {
  uint32_t L = 0, world = 1, rank = 0, beta = 0;
  uint32_t gq = 0, gp = 0;                 // limb slots per rank in gather buffer 1 (Q) and 2 (P, per accumulator)
  std::vector<uint32_t> own_q, own_p;      // owned Q-limb indices i, owned P-limb indices j (extended limb L + j)
  LimbMap q_lm, p_lm, e_lm;                // owned Q / owned P (pos = nq + k inside the local [ne][N] buffers) / owned extended
  double2 *scale1 = nullptr, *scale2 = nullptr, *pinv = nullptr;
  std::vector<HostBConv> up;               // [beta]
  std::vector<LimbMap> up_src;             // positions of the digit's limbs inside gather buffer 1
  HostBConv down;
  LimbMap down_src;                        // positions of the P-limbs inside gather buffer 2 (accumulator 0)
  // rank r's owned P-limbs are the extended limbs e = L + j with e % world == r; its first such e sits at slot
  // floor(e / world) counted over ALL its limbs, so subtract the number of Q-limbs it owns
  static uint32_t first_p_slot(uint32_t r, uint32_t L, uint32_t world) { return L > r ? (L - r + world - 1) / world : 0; }
  // peer-direct mode (hml_keyswitch_shard_*_p2p): per-source word offsets into the OWNERS' gather buffers, relative to this
  // rank's own buffer, rebuilt whenever the peer pointers change
  std::vector<long long *> d_off1;         // [beta] device arrays [a_j]
  BConvJob *up_jobs = nullptr;             // [beta] one-launch form of the ModUp conversions (rebuilt with d_off1), or null
  long long *d_off2 = nullptr;             // device array [alpha]
  std::vector<const void *> peers1_sig, peers2_sig;
  // sharded rescale (hml_rescale_shard_*): q_{L-1}^-1 mod q_l for the owned limbs l < L - 1
  double2 *qlinv_own = nullptr;
};

struct DevBConv {  // cached tables of an arbitrary (src, dst) conversion for the primitive entry point
  double2 *step1 = nullptr;
  HostBConv host;
};

// Per-kernel-class device time of the ops executed between hml_profile_begin / hml_profile_end: the counterpart of the
// reference's per-unit busy statistics (NTT_(c), BCONV_(c), EWE_(c), AUTO_(c); reference include/Staistics.h:6-40).  While
// it is on, every launch group is followed by an event record (which also serialises the programmatic dependent launches).
struct Prof {
  bool on = false;
  cudaEvent_t start = nullptr;
  std::vector<std::pair<int, cudaEvent_t>> marks;
};

}  // namespace hml

struct hml_ctx {
  hml::Params p;
  int device = 0;
  std::string err;
  hml::CfgFile cfg;
  bool has_cfg = false;

  double *tw_fwd = nullptr, *tw_inv = nullptr, *tw_fwd_rows = nullptr, *tw_inv_rows = nullptr;
  hml::ModConst *mc = nullptr;
  hml::NttTables tabs{};
  unsigned *col_ctr = nullptr;  // tabs.col_ctr: the column passes' tile queue (two-pass rings)

  std::map<uint32_t, hml::LevelConsts> levels;
  std::map<std::vector<uint32_t>, hml::DevBConv> bconv_cache;
  std::map<uint64_t, hml::ShardPlan> shard_plans;

  hml::u64 *ws = nullptr;  // workspace, grown on demand
  size_t ws_words = 0;

  hml_exec_counts exec{};

  // host-buffer API: staging buffers + streams
  cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
  hml::u64 *stage = nullptr;
  size_t stage_words = 0;

  // Ops share ONE workspace.  The stream the workspace was last used on is remembered; an op arriving on a different
  // stream first waits (device-side, through ev_ws) for everything queued on the previous one.
  cudaStream_t last_stream = nullptr;
  bool have_last = false;
  cudaEvent_t ev_ws = nullptr;

  hml::Prof prof;
};

namespace hml {
// order the workspace between caller streams (see hml_ctx::last_stream); call at the start of every op that touches ctx->ws
void ws_enter(hml_ctx *ctx, cudaStream_t s);
// profiling mark after a launch group of class cls (HML_CLS_*); no-op unless hml_profile_begin was called
void prof_mark(hml_ctx *ctx, int cls, cudaStream_t s);
}  // namespace hml
