// Limb-sharded operations behind the C ABI (SURVEY.md 8e mode 2, BASELINE.json configs[4]).
//
// One ciphertext, its L + alpha extended limbs partitioned over `world` GPUs of one node: extended limb e lives on rank
// e % world — the rule the reference uses to map limbs to its compute clusters (reference include/Driver.h:158,:178), whose
// inter-cluster NoC fetch (reference include/mem.h:612-621, src/mem.cpp:78-100) becomes NVLink loads issued from inside the
// base-conversion kernel (bconv_umma.cu, BConvArgs::src_off).  An `hml_shard` is one rank's view of the group: its own
// peer-visible buffers (two gather buffers, a rescale buffer, a flag block), the mappings of every peer's, and the scratch the
// composite ops need.  Ranks are either one process per GPU (buffers exchanged as cudaIpc handles: hml_shard_handles /
// hml_shard_connect_ipc) or several devices driven by one process (hml_shard_connect_local; the CLI's [cluster] argument).
//
// Every op is a list of limb-local PHASES separated by EXCHANGES (all ranks' phase outputs become visible to every rank):
//   keyswitch  begin | X0 | mid | X1 | end                          reference src/Operation.cpp:9-54
//   hrotate    automorphism + begin | X0 | mid | X1 | end (+ add)   reference src/Operation.cpp:1271-1358
//   hmult      tensor + begin | X0 | mid | X1 | end (+ add) + rescale begin | X2 | rescale end      :913-1023
//   rescale    begin | X2 | end                                      reference src/Operation.cpp:741-911
// An exchange is ONE launch per rank (k_shard_sync: release this rank's epoch into every peer's flag block, then acquire-spin
// until every peer's epoch has arrived), with the epochs kept in device memory, so a whole op sequence can be captured in a
// CUDA graph and replayed.  hml_group_* drives all ranks of a group from one host thread, phase by phase; when several ranks
// share a device (tests on a one-GPU box) it uses separate signal / wait launches on ONE stream, so that no kernel ever
// spins on a flag that a not-yet-launched kernel has to write.
#include <algorithm>
#include <cstring>

#include "ops.h"

using namespace hml;

struct hml_shard {
  hml_ctx *ctx = nullptr;
  uint32_t rank = 0, world = 1, max_L = 0;
  uint32_t max_rot = 1;                    // hoisted rotations per group: gather buffer 2 holds max_rot slots of n2 words
  size_t n1 = 0, n2 = 0, nf = 0, nr = 0;   // words of the own buffers (n2: one slot of gather buffer 2)
  uint64_t *g1 = nullptr, *g2 = nullptr, *fl = nullptr, *rb = nullptr;
  std::vector<uint64_t *> p1, p2, pf, pr;       // every rank's buffers as pointers valid on this device (own at [rank])
  uint64_t **pf_dev = nullptr;                  // device copy of pf
  std::vector<uint64_t *> ipc_maps;
  bool connected = false;
  uint64_t *scratch = nullptr;                  // [5][nq_max][N]: sigma(ct) / d0 d1 d2 / the un-rescaled hmult result
  uint64_t host_epoch[3] = {0, 0, 0};      // used only when signal and wait are separate launches (emulated ranks)
  bool rb_dirty = false;                   // peers may still be reading the rescale buffer of the previous rescale
};

// SOP_ROT_SUM and SOP_HMULT_SUM are internal kinds (hml_group_op serves 0..3): the double-hoisted rotation sum has the key
// switch's phases, the product sum hmult's
enum ShardOpKind { SOP_KEYSWITCH = 0, SOP_HROTATE = 1, SOP_HMULT = 2, SOP_RESCALE = 3, SOP_ROT_SUM = 4, SOP_HMULT_SUM = 5 };
struct ShardOp {
  int kind;
  uint32_t L;
  const uint64_t *a, *b, *key;   // keyswitch: a = d_own; hrotate, rotation sum: a = ct_own; hmult: a, b = ct_own; rescale: a = x_own
  uint64_t *out0, *out1;         // keyswitch: both outputs; others: out0 = the result ciphertext
  uint64_t g;
  // the term table of the sums (n entries): rotation sum ta = key slices, tb = plaintext slices, gs = galois elements;
  // product sum ta[i] (x) tb[i]
  uint32_t n = 0;
  const uint64_t *const *ta = nullptr, *const *tb = nullptr;
  const uint64_t *gs = nullptr;
};
static int op_phases(int kind) { return kind == SOP_HMULT || kind == SOP_HMULT_SUM ? 4 : kind == SOP_RESCALE ? 2 : 3; }
// exchange group (= flag slot group) after phase `ph`
static int op_exchange(int kind, int ph) { return kind == SOP_RESCALE ? 2 : ph; }

static int sfail(hml_shard *sh, int code, const std::string &msg) { return fail(sh->ctx, code, msg); }

static uint32_t own_q_count(uint32_t L, uint32_t rank, uint32_t world) { return L > rank ? (L - rank + world - 1) / world : 0; }

// ------------------------------------------------------------------------------------------------ lifetime
extern "C" int hml_shard_create_ex(hml_ctx *ctx, uint32_t max_L, uint32_t rank, uint32_t world, uint32_t max_rot, hml_shard **out) {
  if (!ctx || !out) return HML_ERR_INVALID;
  *out = nullptr;
  int rc = shard_check(ctx, max_L, rank, world);
  if (rc) return rc;
  if (max_rot < 1 || max_rot > IP_MAX_ROT) return fail(ctx, HML_ERR_INVALID, "max_rot must be in [1, 16]");
  HML_CU_TRY(ctx, cudaSetDevice(ctx->device));
  hml_shard *sh = new hml_shard();
  sh->ctx = ctx; sh->rank = rank; sh->world = world; sh->max_L = max_L; sh->max_rot = max_rot;
  const size_t N = ctx->p.N, A = ctx->p.alpha;
  const size_t gq = (max_L + world - 1) / world, gp = (A + world - 1) / world;
  sh->n1 = (size_t)world * gq * N; sh->n2 = (size_t)world * 2 * gp * N; sh->nf = 3 * (size_t)world + 8; sh->nr = 2 * N;
  auto alloc = [&](uint64_t **p, size_t words) -> cudaError_t {
    cudaError_t e = cudaMalloc((void **)p, words * 8);
    return e == cudaSuccess ? cudaMemset(*p, 0, words * 8) : e;
  };
  cudaError_t e = alloc(&sh->g1, sh->n1);
  if (e == cudaSuccess) e = alloc(&sh->g2, sh->n2 * max_rot);
  if (e == cudaSuccess) e = alloc(&sh->fl, sh->nf);
  if (e == cudaSuccess) e = alloc(&sh->rb, sh->nr);
  if (e == cudaSuccess) e = alloc(&sh->scratch, 5 * std::max<size_t>(1, own_q_count(max_L, rank, world)) * N);
  if (e == cudaSuccess) e = cudaMalloc((void **)&sh->pf_dev, world * sizeof(uint64_t *));
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    ctx->err = std::string("hml_shard_create: ") + cudaGetErrorString(e);
    cudaFree(sh->g1); cudaFree(sh->g2); cudaFree(sh->fl); cudaFree(sh->rb); cudaFree(sh->scratch); cudaFree(sh->pf_dev);
    delete sh;
    return HML_ERR_CUDA;
  }
  sh->p1.assign(world, nullptr); sh->p2.assign(world, nullptr); sh->pf.assign(world, nullptr); sh->pr.assign(world, nullptr);
  sh->p1[rank] = sh->g1; sh->p2[rank] = sh->g2; sh->pf[rank] = sh->fl; sh->pr[rank] = sh->rb;
  if (world == 1) {
    HML_CU_TRY(ctx, cudaMemcpy(sh->pf_dev, sh->pf.data(), sizeof(uint64_t *), cudaMemcpyHostToDevice));
    sh->connected = true;
  }
  *out = sh;
  return HML_OK;
}

extern "C" int hml_shard_create(hml_ctx *ctx, uint32_t max_L, uint32_t rank, uint32_t world, hml_shard **out) {
  return hml_shard_create_ex(ctx, max_L, rank, world, 1, out);
}

extern "C" int hml_shard_destroy(hml_shard *sh) {
  if (!sh) return HML_OK;
  cudaSetDevice(sh->ctx->device);
  cudaDeviceSynchronize();
  for (uint64_t *m : sh->ipc_maps) cudaIpcCloseMemHandle(m);
  cudaFree(sh->g1); cudaFree(sh->g2); cudaFree(sh->fl); cudaFree(sh->rb); cudaFree(sh->scratch); cudaFree(sh->pf_dev);
  delete sh;
  return HML_OK;
}

extern "C" int hml_shard_handles(hml_shard *sh, unsigned char *out_4x64) {
  if (!sh || !out_4x64) return HML_ERR_INVALID;
  HML_CU_TRY(sh->ctx, cudaSetDevice(sh->ctx->device));
  uint64_t *bufs[4] = {sh->g1, sh->g2, sh->fl, sh->rb};
  for (int k = 0; k < 4; ++k) {
    cudaIpcMemHandle_t h;
    HML_CU_TRY(sh->ctx, cudaIpcGetMemHandle(&h, bufs[k]));
    memcpy(out_4x64 + 64 * k, &h, 64);
  }
  return HML_OK;
}

static int finish_connect(hml_shard *sh) {
  HML_CU_TRY(sh->ctx, cudaMemcpy(sh->pf_dev, sh->pf.data(), sh->world * sizeof(uint64_t *), cudaMemcpyHostToDevice));
  sh->connected = true;
  return HML_OK;
}

extern "C" int hml_shard_connect_ipc(hml_shard *sh, const unsigned char *handles_world_4x64) {
  if (!sh || !handles_world_4x64) return HML_ERR_INVALID;
  HML_CU_TRY(sh->ctx, cudaSetDevice(sh->ctx->device));
  for (uint32_t r = 0; r < sh->world; ++r) {
    if (r == sh->rank) continue;
    uint64_t **dst[4] = {&sh->p1[r], &sh->p2[r], &sh->pf[r], &sh->pr[r]};
    for (int k = 0; k < 4; ++k) {
      cudaIpcMemHandle_t h;
      memcpy(&h, handles_world_4x64 + ((size_t)r * 4 + k) * 64, 64);
      void *p = nullptr;
      HML_CU_TRY(sh->ctx, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
      *dst[k] = (uint64_t *)p;
      sh->ipc_maps.push_back((uint64_t *)p);
    }
  }
  return finish_connect(sh);
}

extern "C" int hml_shard_connect_local(hml_shard *const *group, uint32_t world) {
  if (!group || world == 0) return HML_ERR_INVALID;
  for (uint32_t r = 0; r < world; ++r)
    if (!group[r] || group[r]->world != world || group[r]->rank != r) return HML_ERR_INVALID;
  for (uint32_t r = 1; r < world; ++r)  // slot r of every gather buffer 2 sits r * n2 words in: all ranks need the same layout
    if (group[r]->max_rot != group[0]->max_rot) return sfail(group[r], HML_ERR_INVALID, "every rank of a shard group must use the same max_rot");
  for (uint32_t r = 0; r < world; ++r) {
    hml_shard *sh = group[r];
    HML_CU_TRY(sh->ctx, cudaSetDevice(sh->ctx->device));
    for (uint32_t q = 0; q < world; ++q) {
      if (q == r) continue;
      const int pd = group[q]->ctx->device;
      if (pd != sh->ctx->device) {
        int can = 0;
        HML_CU_TRY(sh->ctx, cudaDeviceCanAccessPeer(&can, sh->ctx->device, pd));
        if (!can) return sfail(sh, HML_ERR_UNSUPPORTED, "devices of the shard group cannot access each other's memory");
        cudaError_t e = cudaDeviceEnablePeerAccess(pd, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) HML_CU_TRY(sh->ctx, e);
        cudaGetLastError();
      }
      sh->p1[q] = group[q]->g1; sh->p2[q] = group[q]->g2; sh->pf[q] = group[q]->fl; sh->pr[q] = group[q]->rb;
    }
    int rc = finish_connect(sh);
    if (rc) return rc;
  }
  return HML_OK;
}

extern "C" int hml_shard_prepare(hml_shard *sh, uint32_t L) {
  if (!sh) return HML_ERR_INVALID;
  if (!sh->connected) return sfail(sh, HML_ERR_INVALID, "shard group not connected");
  if (L > sh->max_L) return sfail(sh, HML_ERR_INVALID, "level above the shard's maximum");
  return shard_prepare(sh->ctx, L, sh->rank, sh->world, (const uint64_t *const *)sh->p1.data(), (const uint64_t *const *)sh->p2.data(), sh->max_rot);
}

extern "C" int hml_shard_status(hml_ctx *ctx, const uint64_t *flags, uint32_t world, void *stream);
extern "C" int hml_shard_check(hml_shard *sh, void *stream) {
  if (!sh) return HML_ERR_INVALID;
  return hml_shard_status(sh->ctx, sh->fl, sh->world, stream);
}

extern "C" int hml_shard_own_limbs(const hml_shard *sh, uint32_t L, uint32_t *n_own_q, uint32_t *n_own_q_after_rescale) {
  if (!sh || L == 0) return HML_ERR_INVALID;
  const uint32_t nq = own_q_count(L, sh->rank, sh->world);
  if (n_own_q) *n_own_q = nq;
  if (n_own_q_after_rescale) *n_own_q_after_rescale = nq - ((L - 1) % sh->world == sh->rank ? 1 : 0);
  return HML_OK;
}

// ------------------------------------------------------------------------------------------------ phases
// the sums' operands, checked on every rank before anything is enqueued
static int sum_check(hml_shard *sh, const ShardOp &op) {
  const bool rot = op.kind == SOP_ROT_SUM;
  if (op.n == 0) return sfail(sh, HML_ERR_INVALID, rot ? "n_rot must be at least 1" : "n_terms must be at least 1");
  if (!op.out0 || (rot && (!op.a || !op.gs)) || (!rot && (!op.ta || !op.tb))) return sfail(sh, HML_ERR_INVALID, "null buffer");
  const size_t N = sh->ctx->p.N;
  const uint32_t nq = own_q_count(op.L, sh->rank, sh->world);
  const bool own_ext = nq > 0 || own_q_count(op.L + sh->ctx->p.alpha, sh->rank, sh->world) > 0;
  const uint32_t n_out = rot ? nq : nq - ((op.L - 1) % sh->world == sh->rank ? 1 : 0);
  const size_t in_w = 2 * (size_t)std::max<uint32_t>(nq, 1) * N, out_w = 2 * (size_t)std::max<uint32_t>(n_out, 1) * N;
  auto overlaps = [&](const uint64_t *in) { return op.out0 < in + in_w && in < op.out0 + out_w; };
  if (rot && overlaps(op.a)) return sfail(sh, HML_ERR_INVALID, "the output overlaps the input");
  if (!rot && own_ext && !op.key) return sfail(sh, HML_ERR_INVALID, "null key on a rank that owns extended limbs");
  for (uint32_t i = 0; i < op.n; ++i) {
    if (rot) {
      if (!(op.gs[i] & 1)) return sfail(sh, HML_ERR_INVALID, "galois element must be odd");
      if (own_ext && (!op.ta || !op.ta[i])) return sfail(sh, HML_ERR_INVALID, "null rotation key on a rank that owns extended limbs");
      if (own_ext && (!op.tb || !op.tb[i])) return sfail(sh, HML_ERR_INVALID, "null plaintext on a rank that owns extended limbs");
    } else {
      if (!op.ta[i] || !op.tb[i]) return sfail(sh, HML_ERR_INVALID, "null ciphertext");
      if (overlaps(op.ta[i]) || overlaps(op.tb[i])) return sfail(sh, HML_ERR_INVALID, "the output overlaps an input");
    }
  }
  return HML_OK;
}

static int op_check(hml_shard *sh, const ShardOp &op) {
  if (!sh->connected) return sfail(sh, HML_ERR_INVALID, "shard group not connected");
  int rc = check_level(sh->ctx, op.L, op.kind == SOP_HMULT || op.kind == SOP_RESCALE || op.kind == SOP_HMULT_SUM ? 2 : 1);
  if (rc) return rc;
  if (op.L > sh->max_L) return sfail(sh, HML_ERR_INVALID, "level above the shard's maximum");
  if (op.kind == SOP_HROTATE && !(op.g & 1)) return sfail(sh, HML_ERR_INVALID, "galois element must be odd");
  if (op.kind == SOP_ROT_SUM || op.kind == SOP_HMULT_SUM) return sum_check(sh, op);
  return HML_OK;
}

static int run_phase(hml_shard *sh, const ShardOp &op, int ph, cudaStream_t s) {
  hml_ctx *ctx = sh->ctx;
  const uint32_t L = op.L, rank = sh->rank, world = sh->world;
  const size_t N = ctx->p.N;
  const uint32_t nq = own_q_count(L, rank, world);
  const bool own_ext = nq > 0 || own_q_count(L + ctx->p.alpha, rank, world) > 0;
  std::vector<uint32_t> own(nq);
  for (uint32_t k = 0; k < nq; ++k) own[k] = rank + k * world;
  uint64_t *sc = sh->scratch;
  void *st = (void *)s;
  int rc = HML_OK;
  auto peers = [](const std::vector<uint64_t *> &v) { return (const uint64_t *const *)v.data(); };
  switch (op.kind) {
    case SOP_KEYSWITCH:
      if (ph == 0) return hml_keyswitch_shard_begin(ctx, L, rank, world, op.a, sh->g1, st);
      if (ph == 1) return own_ext ? hml_keyswitch_shard_mid_p2p(ctx, L, rank, world, op.a, peers(sh->p1), op.key, sh->g2, st) : HML_OK;
      return hml_keyswitch_shard_end_p2p(ctx, L, rank, world, peers(sh->p2), op.out0, op.out1, st);
    case SOP_HROTATE: {
      uint64_t *sig = sc;  // [2][nq][N]
      if (ph == 0) {
        if (nq && (rc = hml_automorph(ctx, op.a, sig, op.g, 2 * nq, st))) return rc;
        return hml_keyswitch_shard_begin(ctx, L, rank, world, sig + (size_t)nq * N, sh->g1, st);
      }
      if (ph == 1) return own_ext ? hml_keyswitch_shard_mid_p2p(ctx, L, rank, world, sig + (size_t)nq * N, peers(sh->p1), op.key, sh->g2, st) : HML_OK;
      // (sigma(c0) + ks0, ks1): the addend rides in the ModDown epilogue
      return shard_end_p2p(ctx, L, rank, world, peers(sh->p2), op.out0, op.out0 + (size_t)nq * N, sig, nullptr, s);
    }
    case SOP_ROT_SUM: {
      // begin(c1) | X0 | ModUp, weighted inner products, P-limb INTT | X1 | one ModDown with addend z = sum_r pt_r * sigma_r(c0)
      uint64_t *z = sc;  // [nq][N]
      if (ph == 0) return hml_keyswitch_shard_begin(ctx, L, rank, world, op.a + (size_t)nq * N, sh->g1, st);
      if (ph == 1) {
        if (!own_ext) return HML_OK;
        if ((rc = shard_rot_sum_inner(ctx, L, rank, world, peers(sh->p1), op.a, op.n, op.ta, op.gs, op.tb, z, s))) return rc;
        return shard_hoist_intt(ctx, L, rank, world, 1, sh->g2, sh->n2, s);
      }
      return shard_end_p2p(ctx, L, rank, world, peers(sh->p2), op.out0, op.out0 + (size_t)nq * N, z, nullptr, s);
    }
    case SOP_HMULT:
    case SOP_HMULT_SUM: {
      uint64_t *d0 = sc, *d1 = d0 + (size_t)nq * N, *d2 = d1 + (size_t)nq * N, *c = d2 + (size_t)nq * N;  // c [2][nq][N]
      const size_t PL = (size_t)nq * N;
      if (ph == 0) {
        if (op.kind == SOP_HMULT_SUM) {  // the sums of the terms' tensor products: everything after them is hmult's
          if ((rc = shard_tensor_sum(ctx, L, rank, world, op.n, op.ta, op.tb, d0, d1, d2, s))) return rc;
        } else if (nq) {  // TensorCompute on the owned limbs (reference src/Operation.cpp:592-739)
          if ((rc = hml_ewe(ctx, op.a, op.b, nullptr, nullptr, 0, d0, own.data(), nq, st))) return rc;
          if ((rc = hml_ewe(ctx, op.a, op.b + PL, op.a + PL, op.b, 0, d1, own.data(), nq, st))) return rc;
          if ((rc = hml_ewe(ctx, op.a + PL, op.b + PL, nullptr, nullptr, 0, d2, own.data(), nq, st))) return rc;
        }
        return hml_keyswitch_shard_begin(ctx, L, rank, world, d2, sh->g1, st);
      }
      if (ph == 1) return own_ext ? hml_keyswitch_shard_mid_p2p(ctx, L, rank, world, d2, peers(sh->p1), op.key, sh->g2, st) : HML_OK;
      if (ph == 2) {
        if ((rc = shard_end_p2p(ctx, L, rank, world, peers(sh->p2), c, c + PL, d0, d1, s))) return rc;
        return hml_rescale_shard_begin(ctx, L, rank, world, c, sh->rb, st);
      }
      return hml_rescale_shard_end(ctx, L, rank, world, c, sh->pr[(L - 1) % world], op.out0, st);
    }
    case SOP_RESCALE:
      if (ph == 0) return hml_rescale_shard_begin(ctx, L, rank, world, op.a, sh->rb, st);
      return hml_rescale_shard_end(ctx, L, rank, world, op.a, sh->pr[(L - 1) % world], op.out0, st);
  }
  return HML_ERR_INVALID;
}

static int fused_sync(hml_shard *sh, int grp, cudaStream_t s) {
  return hml_shard_sync(sh->ctx, (uint64_t *const *)sh->pf_dev, grp * sh->world + sh->rank, sh->fl, grp * sh->world, 0, sh->world, (void *)s);
}

static int hoist_prepare(hml_shard *sh, uint32_t L);

// one rank per GPU: phases with one fused exchange launch between them
static int run_op(hml_shard *sh, const ShardOp &op, cudaStream_t s) {
  int rc = op_check(sh, op);
  if (rc) return rc;
  HML_CU_TRY(sh->ctx, cudaSetDevice(sh->ctx->device));
  if (op.kind >= SOP_ROT_SUM && (rc = hoist_prepare(sh, op.L))) return rc;  // a no-op after hml_shard_prepare(L)
  if ((op.kind == SOP_RESCALE) && sh->rb_dirty && (rc = fused_sync(sh, 2, s))) return rc;  // write-after-read on the rescale buffer
  const int n = op_phases(op.kind);
  for (int ph = 0; ph < n; ++ph) {
    if ((rc = run_phase(sh, op, ph, s))) return rc;
    if (ph + 1 < n && (rc = fused_sync(sh, op_exchange(op.kind, ph), s))) return rc;
  }
  sh->rb_dirty = op.kind == SOP_RESCALE || op.kind == SOP_HMULT ? (op.kind == SOP_RESCALE) : false;
  return HML_OK;
}

extern "C" int hml_keyswitch_sharded(hml_shard *sh, uint32_t L, const uint64_t *d_own, const uint64_t *evk_own, uint64_t *out0_own,
                                     uint64_t *out1_own, void *stream) {
  if (!sh || !d_own || !out0_own || !out1_own) return HML_ERR_INVALID;
  return run_op(sh, ShardOp{SOP_KEYSWITCH, L, (const uint64_t *)d_own, nullptr, (const uint64_t *)evk_own, (uint64_t *)out0_own, (uint64_t *)out1_own, 0}, (cudaStream_t)stream);
}
extern "C" int hml_hrotate_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, const uint64_t *rotkey_own, uint64_t galois_elt,
                                   uint64_t *out_own, void *stream) {
  if (!sh || !ct_own || !out_own) return HML_ERR_INVALID;
  return run_op(sh, ShardOp{SOP_HROTATE, L, (const uint64_t *)ct_own, nullptr, (const uint64_t *)rotkey_own, (uint64_t *)out_own, nullptr, galois_elt}, (cudaStream_t)stream);
}
extern "C" int hml_hmult_sharded(hml_shard *sh, uint32_t L, const uint64_t *a_own, const uint64_t *b_own, const uint64_t *evk_own,
                                 uint64_t *out_own, void *stream) {
  if (!sh || !a_own || !b_own || !out_own) return HML_ERR_INVALID;
  return run_op(sh, ShardOp{SOP_HMULT, L, (const uint64_t *)a_own, (const uint64_t *)b_own, (const uint64_t *)evk_own, (uint64_t *)out_own, nullptr, 0}, (cudaStream_t)stream);
}
extern "C" int hml_rescale_sharded(hml_shard *sh, uint32_t L, const uint64_t *x_own, uint64_t *out_own, void *stream) {
  if (!sh || !x_own || !out_own) return HML_ERR_INVALID;
  return run_op(sh, ShardOp{SOP_RESCALE, L, (const uint64_t *)x_own, nullptr, nullptr, (uint64_t *)out_own, nullptr, 0}, (cudaStream_t)stream);
}

// limb-local ciphertext ops on the owned limbs: kind 0 = hadd (b = ct [2][nq][N]), 1 = pmult, 2 = padd (b = pt [nq][N]),
// 3 = pmult + hadd in one pass (out = a * b + out: `out_own` is also the addend)
extern "C" int hml_ew_sharded(hml_shard *sh, uint32_t L, int kind, const uint64_t *a_own, const uint64_t *b_own, uint64_t *out_own, void *stream) {
  if (!sh || !a_own || !b_own || !out_own || kind < 0 || kind > 3) return HML_ERR_INVALID;
  int rc = check_level(sh->ctx, L, 1);
  if (rc) return rc;
  const uint32_t nq = own_q_count(L, sh->rank, sh->world);
  if (!nq) return HML_OK;
  const size_t PL = (size_t)nq * sh->ctx->p.N;
  std::vector<uint32_t> own(nq);
  for (uint32_t k = 0; k < nq; ++k) own[k] = sh->rank + k * sh->world;
  for (int c = 0; c < 2; ++c) {
    const uint64_t *a = a_own + c * PL, *b = kind == 0 ? b_own + c * PL : b_own;
    rc = kind == 1   ? hml_ewe(sh->ctx, a, b, nullptr, nullptr, 0, out_own + c * PL, own.data(), nq, stream)
         : kind == 3 ? hml_ewe(sh->ctx, a, b, out_own + c * PL, nullptr, 0, out_own + c * PL, own.data(), nq, stream)
                     : hml_ewe(sh->ctx, a, nullptr, b, nullptr, 0, out_own + c * PL, own.data(), nq, stream);
    if (rc) return rc;
  }
  return HML_OK;
}

// ------------------------------------------------------------------------------------------------ hoisted rotations
// n_rot rotations of ONE sharded ciphertext sharing one ModUp of c1 (the sharded form of hml_hrotate_hoisted, bit-identical to
// it on the owned limbs).  The rotations run in groups of up to max_rot; a group shares one inner-product launch, one P-limb
// INTT and one exchange, and uses slots 0.. of every rank's gather buffer 2:
//   begin | X0 | ModUp, IP(0), INTT(0) | X1 | end(0) | IP(1) | X1 | INTT(1) | X1 | end(1) | ...
// begin and X0 run once per op.  The extra X1 in front of a later group's INTT orders its writes to gather buffer 2 after every
// peer's ModDown reads of the previous group.  end(k) is one ModDown per rotation of the group, with sigma_r(c0) as its addend:
// gathered by the fused epilogue on two-pass rings, an automorphism kernel into the shard scratch on single-pass rings.
enum HoistStepKind { HS_BEGIN, HS_INNER, HS_INTT, HS_END, HS_X0, HS_X1 };
struct HoistStep {
  int kind;
  uint32_t group;
};
struct HoistOp {
  uint32_t L, n_rot;
  const uint64_t *ct;            // [2][nq][N]
  const uint64_t *const *keys;   // [n_rot] owned key slices (may be null on a rank that owns no extended limb)
  const uint64_t *galois;        // [n_rot]
  uint64_t *const *outs;         // [n_rot] [2][nq][N]
};

static std::vector<HoistStep> hoist_steps(uint32_t n_rot, uint32_t H) {
  std::vector<HoistStep> v{{HS_BEGIN, 0}, {HS_X0, 0}};
  for (uint32_t k = 0; k * H < n_rot; ++k) {
    v.push_back({HS_INNER, k});
    if (k) v.push_back({HS_X1, k});
    v.push_back({HS_INTT, k});
    v.push_back({HS_X1, k});
    v.push_back({HS_END, k});
  }
  return v;
}

static int hoist_check(hml_shard *sh, const HoistOp &op) {
  hml_ctx *ctx = sh->ctx;
  if (!sh->connected) return sfail(sh, HML_ERR_INVALID, "shard group not connected");
  int rc = check_level(ctx, op.L, 1);
  if (rc) return rc;
  if (op.L > sh->max_L) return sfail(sh, HML_ERR_INVALID, "level above the shard's maximum");
  if (!op.ct || !op.galois || !op.outs) return sfail(sh, HML_ERR_INVALID, "null buffer");
  const uint32_t nq = own_q_count(op.L, sh->rank, sh->world);
  const bool own_ext = nq > 0 || own_q_count(op.L + ctx->p.alpha, sh->rank, sh->world) > 0;
  const size_t words = 2 * (size_t)std::max<uint32_t>(nq, 1) * ctx->p.N;
  for (uint32_t r = 0; r < op.n_rot; ++r) {
    const uint64_t *o = op.outs[r];
    if (!o) return sfail(sh, HML_ERR_INVALID, "null output");
    if (o < op.ct + words && op.ct < o + words) return sfail(sh, HML_ERR_INVALID, "an output aliases the input");
    if (!(op.galois[r] & 1)) return sfail(sh, HML_ERR_INVALID, "galois element must be odd");
    if (own_ext && (!op.keys || !op.keys[r])) return sfail(sh, HML_ERR_INVALID, "null rotation key on a rank that owns extended limbs");
  }
  return HML_OK;
}

static int hoist_prepare(hml_shard *sh, uint32_t L) {
  HML_CU_TRY(sh->ctx, cudaSetDevice(sh->ctx->device));
  return shard_prepare(sh->ctx, L, sh->rank, sh->world, (const uint64_t *const *)sh->p1.data(), (const uint64_t *const *)sh->p2.data(), sh->max_rot);
}

static int hoist_phase(hml_shard *sh, const HoistOp &op, const HoistStep &st, cudaStream_t s) {
  hml_ctx *ctx = sh->ctx;
  const uint32_t L = op.L, rank = sh->rank, world = sh->world, H = sh->max_rot;
  const size_t N = ctx->p.N;
  const uint32_t nq = own_q_count(L, rank, world);
  const uint64_t *c1 = op.ct + (size_t)nq * N;
  const uint32_t lo = st.group * H, n = std::min(H, op.n_rot - lo);
  auto peers = [](const std::vector<uint64_t *> &v) { return (const uint64_t *const *)v.data(); };
  switch (st.kind) {
    case HS_BEGIN: return hml_keyswitch_shard_begin(ctx, L, rank, world, c1, sh->g1, (void *)s);
    case HS_INNER:
      return shard_hoist_inner(ctx, L, rank, world, H, st.group == 0 ? peers(sh->p1) : nullptr, c1, n, op.keys ? op.keys + lo : nullptr,
                               op.galois + lo, s);
    case HS_INTT: return shard_hoist_intt(ctx, L, rank, world, n, sh->g2, sh->n2, s);
    case HS_END:
      for (uint32_t r = 0; r < n && nq; ++r) {
        const uint64_t g = galois_mod(op.galois[lo + r], N);
        uint64_t *o = op.outs[lo + r];
        const uint64_t *add = op.ct;  // g = 1: sigma(c0) is c0 itself
        uint64_t add_g = 0;
        if (g != 1 && ctx->p.logN > NTT_SMALL_LOG) {
          add_g = g;
          ctx->exec.automorph_limbs += nq;
        } else if (g != 1) {
          int rc = hml_automorph(ctx, op.ct, sh->scratch, g, nq, (void *)s);
          if (rc) return rc;
          add = sh->scratch;
        }
        int rc = shard_end_p2p(ctx, L, rank, world, peers(sh->p2), o, o + (size_t)nq * N, add, nullptr, s, r, H, sh->n2, add_g);
        if (rc) return rc;
      }
      return HML_OK;
  }
  return HML_ERR_INVALID;
}

extern "C" int hml_hrotate_hoisted_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, uint32_t n_rot, const uint64_t *const *rotkeys_own,
                                           const uint64_t *galois_elts, uint64_t *const *outs_own, void *stream) {
  if (!sh) return HML_ERR_INVALID;
  if (n_rot == 0) return HML_OK;
  const HoistOp op{L, n_rot, ct_own, rotkeys_own, galois_elts, outs_own};
  int rc = hoist_check(sh, op);
  if (rc || (rc = hoist_prepare(sh, L))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  for (const HoistStep &st : hoist_steps(n_rot, sh->max_rot)) {
    rc = st.kind == HS_X0 ? fused_sync(sh, 0, s) : st.kind == HS_X1 ? fused_sync(sh, 1, s) : hoist_phase(sh, op, st, s);
    if (rc) return rc;
  }
  sh->rb_dirty = false;  // no rescale buffer written; X0 ordered this op after every peer's earlier reads of it
  return HML_OK;
}

// ------------------------------------------------------------------------------------------------ group driver
// All ranks of a group driven from one host thread, phase by phase.  Arrays are indexed by rank; streams[r] is rank r's stream.
// Ranks that share a device MUST share one stream; they are then ordered by that stream and use separate signal / wait
// launches (host-side epochs) instead of the fused exchange.
static int group_setup(hml_shard *const *group, uint32_t world, void *const *streams, bool *emulate) {
  *emulate = false;
  for (uint32_t r = 0; r < world; ++r) {
    if (!group[r] || group[r]->world != world || group[r]->rank != r) return HML_ERR_INVALID;
    for (uint32_t q = 0; q < r; ++q)
      if (group[q]->ctx->device == group[r]->ctx->device) {
        *emulate = true;
        if ((streams ? streams[q] : nullptr) != (streams ? streams[r] : nullptr))
          return fail(group[r]->ctx, HML_ERR_INVALID, "ranks that share a device must share one stream");
      }
  }
  return HML_OK;
}

static cudaStream_t group_stream(void *const *streams, uint32_t r) { return (cudaStream_t)(streams ? streams[r] : nullptr); }

static int group_exchange(hml_shard *const *group, uint32_t world, bool emulate, void *const *streams, int grp) {
  int rc;
  if (!emulate) {
    for (uint32_t r = 0; r < world; ++r) {
      cudaSetDevice(group[r]->ctx->device);
      if ((rc = fused_sync(group[r], grp, group_stream(streams, r)))) return rc;
    }
    return HML_OK;
  }
  for (uint32_t r = 0; r < world; ++r) {
    hml_shard *sh = group[r];
    cudaSetDevice(sh->ctx->device);
    if ((rc = hml_shard_signal(sh->ctx, (uint64_t *const *)sh->pf_dev, grp * world + r, ++sh->host_epoch[grp], world, (void *)group_stream(streams, r)))) return rc;
  }
  for (uint32_t r = 0; r < world; ++r) {
    hml_shard *sh = group[r];
    cudaSetDevice(sh->ctx->device);
    if ((rc = hml_shard_wait(sh->ctx, sh->fl, grp * world, sh->host_epoch[grp], world, (void *)group_stream(streams, r)))) return rc;
  }
  return HML_OK;
}

// ops[r] (one kind) on every rank of the group, phase by phase
static int group_run(hml_shard *const *group, uint32_t world, void *const *streams, const std::vector<ShardOp> &ops) {
  bool emulate;
  int rc = group_setup(group, world, streams, &emulate);
  if (rc) return rc;
  const int op_kind = ops[0].kind;
  for (uint32_t r = 0; r < world; ++r)
    if ((rc = op_check(group[r], ops[r]))) return rc;
  if (op_kind >= SOP_ROT_SUM)  // before the first exchange: nothing may allocate or synchronise while a rank waits
    for (uint32_t r = 0; r < world; ++r)
      if ((rc = hoist_prepare(group[r], ops[r].L))) return rc;
  if (op_kind == SOP_RESCALE && group[0]->rb_dirty && (rc = group_exchange(group, world, emulate, streams, 2))) return rc;
  const int n = op_phases(op_kind);
  for (int ph = 0; ph < n; ++ph) {
    for (uint32_t r = 0; r < world; ++r) {
      cudaSetDevice(group[r]->ctx->device);
      if ((rc = run_phase(group[r], ops[r], ph, group_stream(streams, r)))) return rc;
    }
    if (ph + 1 < n && (rc = group_exchange(group, world, emulate, streams, op_exchange(op_kind, ph)))) return rc;
  }
  for (uint32_t r = 0; r < world; ++r) group[r]->rb_dirty = op_kind == SOP_RESCALE;
  return HML_OK;
}

// op: 0 keyswitch (a = d_own, out0/out1), 1 hrotate (a = ct_own, out0), 2 hmult (a, b, out0), 3 rescale (a, out0).
extern "C" int hml_group_op(hml_shard *const *group, uint32_t world, int op_kind, uint32_t L, const uint64_t *const *a, const uint64_t *const *b,
                            const uint64_t *const *key, uint64_t *const *out0, uint64_t *const *out1, uint64_t galois_elt, void *const *streams) {
  if (!group || world == 0 || !a || !out0 || op_kind < 0 || op_kind > 3) return HML_ERR_INVALID;
  std::vector<ShardOp> ops(world);
  for (uint32_t r = 0; r < world; ++r)
    ops[r] = ShardOp{op_kind, L, (const uint64_t *)a[r], b ? (const uint64_t *)b[r] : nullptr, key ? (const uint64_t *)key[r] : nullptr, (uint64_t *)out0[r],
                     out1 ? (uint64_t *)out1[r] : nullptr, galois_elt};
  return group_run(group, world, streams, ops);
}

// hml_hrotate_hoisted_sharded for every rank of a local group; rotkeys_own / outs_own are rank-major ([rank * n_rot + i])
extern "C" int hml_group_hrotate_hoisted(hml_shard *const *group, uint32_t world, uint32_t L, const uint64_t *const *ct_own, uint32_t n_rot,
                                         const uint64_t *const *rotkeys_own, const uint64_t *galois_elts, uint64_t *const *outs_own,
                                         void *const *streams) {
  if (!group || world == 0 || !ct_own) return HML_ERR_INVALID;
  bool emulate;
  int rc = group_setup(group, world, streams, &emulate);
  if (rc) return rc;
  if (n_rot == 0) return HML_OK;
  if (!outs_own) return fail(group[0]->ctx, HML_ERR_INVALID, "null output");
  std::vector<HoistOp> ops(world);
  for (uint32_t r = 0; r < world; ++r) {
    if (group[r]->max_rot != group[0]->max_rot) return fail(group[r]->ctx, HML_ERR_INVALID, "every rank of a shard group must use the same max_rot");
    ops[r] = HoistOp{L, n_rot, ct_own[r], rotkeys_own ? rotkeys_own + (size_t)r * n_rot : nullptr, galois_elts, outs_own + (size_t)r * n_rot};
    if ((rc = hoist_check(group[r], ops[r]))) return rc;
  }
  for (uint32_t r = 0; r < world; ++r)  // before the first exchange: nothing may allocate or synchronise while a rank waits
    if ((rc = hoist_prepare(group[r], L))) return rc;
  for (const HoistStep &st : hoist_steps(n_rot, group[0]->max_rot)) {
    if (st.kind == HS_X0 || st.kind == HS_X1) {
      if ((rc = group_exchange(group, world, emulate, streams, st.kind == HS_X0 ? 0 : 1))) return rc;
      continue;
    }
    for (uint32_t r = 0; r < world; ++r) {
      cudaSetDevice(group[r]->ctx->device);
      if ((rc = hoist_phase(group[r], ops[r], st, group_stream(streams, r)))) return rc;
    }
  }
  for (uint32_t r = 0; r < world; ++r) group[r]->rb_dirty = false;
  return HML_OK;
}

// ------------------------------------------------------------------------------------------------ sums
// The double-hoisted rotation sum and the lazily relinearised product sum on the owned limbs, with the exchanges of ONE key
// switch (rotation sum) or ONE hmult (product sum) whatever the number of terms: every term's work is limb-local.
extern "C" int hml_hrotate_sum_hoisted_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, uint32_t n_rot, const uint64_t *const *rotkeys_own,
                                               const uint64_t *galois_elts, const uint64_t *const *pts_own, uint64_t *out_own, void *stream) {
  if (!sh) return HML_ERR_INVALID;
  ShardOp op{SOP_ROT_SUM, L, ct_own, nullptr, nullptr, out_own, nullptr, 0};
  op.n = n_rot; op.ta = rotkeys_own; op.tb = pts_own; op.gs = galois_elts;
  return run_op(sh, op, (cudaStream_t)stream);
}

extern "C" int hml_group_hrotate_sum_hoisted(hml_shard *const *group, uint32_t world, uint32_t L, const uint64_t *const *ct_own, uint32_t n_rot,
                                             const uint64_t *const *rotkeys_own, const uint64_t *galois_elts, const uint64_t *const *pts_own,
                                             uint64_t *const *out_own, void *const *streams) {
  if (!group || world == 0 || !ct_own || !out_own) return HML_ERR_INVALID;
  std::vector<ShardOp> ops(world);
  for (uint32_t r = 0; r < world; ++r) {
    ops[r] = ShardOp{SOP_ROT_SUM, L, ct_own[r], nullptr, nullptr, out_own[r], nullptr, 0};
    ops[r].n = n_rot; ops[r].gs = galois_elts;
    ops[r].ta = rotkeys_own ? rotkeys_own + (size_t)r * n_rot : nullptr;
    ops[r].tb = pts_own ? pts_own + (size_t)r * n_rot : nullptr;
  }
  return group_run(group, world, streams, ops);
}

extern "C" int hml_hmult_sum_sharded(hml_shard *sh, uint32_t L, uint32_t n_terms, const uint64_t *const *a_own, const uint64_t *const *b_own,
                                     const uint64_t *evk_own, uint64_t *out_own, void *stream) {
  if (!sh) return HML_ERR_INVALID;
  ShardOp op{SOP_HMULT_SUM, L, nullptr, nullptr, evk_own, out_own, nullptr, 0};
  op.n = n_terms; op.ta = a_own; op.tb = b_own;
  return run_op(sh, op, (cudaStream_t)stream);
}

extern "C" int hml_group_hmult_sum(hml_shard *const *group, uint32_t world, uint32_t L, uint32_t n_terms, const uint64_t *const *a_own,
                                   const uint64_t *const *b_own, const uint64_t *const *evk_own, uint64_t *const *out_own, void *const *streams) {
  if (!group || world == 0 || !a_own || !b_own || !out_own) return HML_ERR_INVALID;
  std::vector<ShardOp> ops(world);
  for (uint32_t r = 0; r < world; ++r) {
    ops[r] = ShardOp{SOP_HMULT_SUM, L, nullptr, nullptr, evk_own ? evk_own[r] : nullptr, out_own[r], nullptr, 0};
    ops[r].n = n_terms; ops[r].ta = a_own + (size_t)r * n_terms; ops[r].tb = b_own + (size_t)r * n_terms;
  }
  return group_run(group, world, streams, ops);
}
