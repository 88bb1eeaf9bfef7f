// Op-sequence replay behind the C ABI (BASELINE.json configs[4]; SURVEY.md 8f rank 3).
//
// The reference simulates ONE operation per run and cannot chain them ("NotSuppotr the continuous operation simulate",
// reference src/Operation.cpp:636,675,714); its tree holds no application trace.  A trace here is a list of the five operations
// the reference's CLI accepts (reference bench_test/bench_micro24.cpp:29-48) over numbered ciphertext slots; the input enters
// at level L and every hmult lowers its result by one level, which later ops of the trace may go on using (keys bound in a
// layout with evk_q_limbs >= L serve every level; a plaintext's first limbs serve the lower levels).  A trace runs on one GPU
// (hml_ctx) or limb-sharded over a group (hml_shard), as plain launches or as ONE captured CUDA graph,
// and optionally with hoisted rotations: consecutive hrotate ops that read the same slot share one ModUp
// (hml_hrotate_hoisted on one GPU, hml_hrotate_hoisted_sharded over a shard group).  On one GPU such a run whose outputs are
// summed with plaintext weights right after it may also become one double-hoisted sum (hml_hrotate_sum_hoisted), and a chain
// of products summed as they are formed one lazily relinearised sum (hml_hmult_sum).
#include <algorithm>
#include <cstring>
#include <map>

#include "ops.h"

using namespace hml;

extern "C" int hml_hrotate_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, const uint64_t *rotkey_own, uint64_t galois_elt,
                                   uint64_t *out_own, void *stream);
extern "C" int hml_hmult_sharded(hml_shard *sh, uint32_t L, const uint64_t *a_own, const uint64_t *b_own, const uint64_t *evk_own,
                                 uint64_t *out_own, void *stream);
extern "C" int hml_ew_sharded(hml_shard *sh, uint32_t L, int kind, const uint64_t *a_own, const uint64_t *b_own, uint64_t *out_own, void *stream);
extern "C" int hml_shard_own_limbs(const hml_shard *sh, uint32_t L, uint32_t *n_own_q, uint32_t *n_own_q_after_rescale);
extern "C" int hml_shard_prepare(hml_shard *sh, uint32_t L);
extern "C" int hml_hrotate_hoisted_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, uint32_t n_rot, const uint64_t *const *rotkeys_own,
                                           const uint64_t *galois_elts, uint64_t *const *outs_own, void *stream);

struct hml_replay {
  hml_ctx *ctx = nullptr;
  hml_shard *sh = nullptr;
  uint32_t L = 0, flags = 0, n_slots = 0;
  uint32_t nq = 0, nk = 0;                 // limbs per polynomial of a slot at level L / of an hmult result (owned limbs when sharded)
  std::vector<hml_trace_op> ops;
  std::vector<uint64_t *> slot;            // device buffers, slot 0 = the bound input
  std::vector<uint8_t> owned;              // allocated here
  std::vector<uint32_t> op_level;          // level every op runs at (= the level of its sources when it is reached)
  std::vector<uint32_t> final_level;       // level of every slot after the whole trace (0: never written)
  // bindings
  const uint64_t *x = nullptr, *evk = nullptr;
  std::vector<const uint64_t *> pts, keys;
  std::map<uint32_t, uint32_t> key_of_rot;
  uint32_t evk_q_limbs = 0;
  bool bound = false;
  // graph
  cudaStream_t cap_stream = nullptr;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  bool warm = false;
};

static int rfail(hml_replay *rp, int code, const std::string &m) { return fail(rp->ctx, code, m); }

extern "C" int hml_replay_create(hml_ctx *ctx, hml_shard *sh, uint32_t L, const hml_trace_op *ops, uint32_t n_ops, uint32_t flags,
                                 hml_replay **out) {
  if (!ctx || !ops || !out || n_ops == 0) return HML_ERR_INVALID;
  *out = nullptr;
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (sh && (flags & HML_REPLAY_HOIST_SUM)) return fail(ctx, HML_ERR_UNSUPPORTED, "HML_REPLAY_HOIST_SUM has no limb-sharded op");
  if (sh && (flags & HML_REPLAY_HMULT_SUM)) return fail(ctx, HML_ERR_UNSUPPORTED, "HML_REPLAY_HMULT_SUM has no limb-sharded op");
  hml_replay *rp = new hml_replay();
  rp->ctx = ctx; rp->sh = sh; rp->L = L; rp->flags = flags;
  rp->ops.assign(ops, ops + n_ops);
  uint32_t ns = 1;
  for (const hml_trace_op &o : rp->ops) ns = std::max(ns, std::max(o.dst, o.a) + 1);
  for (const hml_trace_op &o : rp->ops)
    if (o.kind == HML_OP_HADD || o.kind == HML_OP_HMULT) ns = std::max(ns, o.b + 1);
  rp->n_slots = ns;
  rp->slot.assign(ns, nullptr); rp->owned.assign(ns, 0); rp->final_level.assign(ns, 0);
  rp->nq = L; rp->nk = L - 1;
  if (sh && (rc = hml_shard_own_limbs(sh, L, &rp->nq, &rp->nk))) { delete rp; return rc; }
  // walk the trace once: slot 0 is the input at level L; a source must have been written; the two sources of hadd / hmult
  // must sit at the same level; hmult lowers its result by one level and cannot run in place
  std::vector<uint32_t> &lvl = rp->final_level;
  lvl[0] = L;
  auto bad = [&](const char *m) { delete rp; return fail(ctx, HML_ERR_INVALID, std::string("trace: ") + m); };
  for (const hml_trace_op &o : rp->ops) {
    if (o.kind > HML_OP_HMULT) return bad("unknown operation");
    if (o.dst == 0) return bad("slot 0 is the input and cannot be overwritten");
    if (!lvl[o.a]) return bad("source slot not yet written");
    const uint32_t la = lvl[o.a];
    if (o.kind == HML_OP_HADD || o.kind == HML_OP_HMULT) {
      if (!lvl[o.b]) return bad("second source slot not yet written");
      if (lvl[o.b] != la) return bad("the two sources sit at different levels");
    }
    if (o.kind == HML_OP_HMULT) {
      if (la < 2) return bad("hmult needs a source level >= 2");
      if (o.dst == o.a || o.dst == o.b) return bad("hmult cannot run in place");
    }
    rp->op_level.push_back(la);
    lvl[o.dst] = o.kind == HML_OP_HMULT ? la - 1 : la;
    // limb-sharded traces stay at one level: the owner of P-limb j is (level + j) % world, so a rank's key slice is level-specific
    if (sh && la != L) { delete rp; return fail(ctx, HML_ERR_UNSUPPORTED, "limb-sharded traces cannot go on from an hmult result (key slices are per level)"); }
  }
  cudaSetDevice(ctx->device);
  const size_t N = ctx->p.N;
  for (uint32_t i = 1; i < ns; ++i) {
    if (!lvl[i]) continue;
    const size_t words = 2 * (size_t)std::max<uint32_t>(1, rp->nq) * N;   // sized for the top level: every lower level fits
    if (cudaMalloc((void **)&rp->slot[i], words * 8) != cudaSuccess) {
      for (uint32_t k = 1; k < ns; ++k) cudaFree(rp->slot[k]);
      delete rp;
      return fail(ctx, HML_ERR_CUDA, "replay: out of device memory for the ciphertext slots");
    }
    rp->owned[i] = 1;
  }
  *out = rp;
  return HML_OK;
}

extern "C" int hml_replay_destroy(hml_replay *rp) {
  if (!rp) return HML_OK;
  cudaSetDevice(rp->ctx->device);
  cudaDeviceSynchronize();
  if (rp->exec) cudaGraphExecDestroy(rp->exec);
  if (rp->graph) cudaGraphDestroy(rp->graph);
  if (rp->cap_stream) cudaStreamDestroy(rp->cap_stream);
  for (uint32_t i = 0; i < rp->n_slots; ++i)
    if (rp->owned[i]) cudaFree(rp->slot[i]);
  delete rp;
  return HML_OK;
}

extern "C" int hml_replay_bind(hml_replay *rp, const uint64_t *x, const uint64_t *const *plaintexts, uint32_t n_plaintexts,
                               const uint32_t *rot_amounts, const uint64_t *const *rot_keys, uint32_t n_rot_keys, const uint64_t *evk,
                               uint32_t evk_q_limbs) {
  if (!rp || !x) return HML_ERR_INVALID;
  rp->x = x; rp->slot[0] = const_cast<uint64_t *>(x);
  rp->pts.assign(plaintexts, plaintexts + (plaintexts ? n_plaintexts : 0));
  rp->keys.assign(rot_keys, rot_keys + (rot_keys ? n_rot_keys : 0));
  rp->key_of_rot.clear();
  for (uint32_t k = 0; k < rp->keys.size(); ++k) rp->key_of_rot[rot_amounts[k]] = k;
  rp->evk = evk; rp->evk_q_limbs = evk_q_limbs;
  for (const hml_trace_op &o : rp->ops) {
    if ((o.kind == HML_OP_PMULT || o.kind == HML_OP_PADD) && (o.b >= rp->pts.size() || !rp->pts[o.b])) return rfail(rp, HML_ERR_INVALID, "trace uses a plaintext that is not bound");
    if ((o.kind == HML_OP_HROTATE || o.kind == HML_OP_HMULT) && rp->sh && (evk_q_limbs & HML_KEY_PACKED))
      return rfail(rp, HML_ERR_UNSUPPORTED, "limb-sharded traces take word keys (no HML_KEY_PACKED)");
    if ((o.kind == HML_OP_HROTATE || o.kind == HML_OP_HMULT) && (evk_q_limbs & ~HML_KEY_PACKED) < rp->L) return rfail(rp, HML_ERR_INVALID, "keys must be laid out for at least the trace's top level (evk_q_limbs >= L)");
    if (o.kind == HML_OP_HROTATE && (!rp->key_of_rot.count(o.b) || !rp->keys[rp->key_of_rot[o.b]]) && !(rp->sh && rp->nq == 0 && rp->key_of_rot.count(o.b)))
      return rfail(rp, HML_ERR_INVALID, "trace uses a rotation whose key is not bound");
    if (o.kind == HML_OP_HMULT && !evk && !(rp->sh && rp->nq == 0)) return rfail(rp, HML_ERR_INVALID, "trace has an hmult but no relinearisation key is bound");
  }
  rp->bound = true;
  // new pointers invalidate a captured graph
  if (rp->exec) { cudaGraphExecDestroy(rp->exec); rp->exec = nullptr; }
  if (rp->graph) { cudaGraphDestroy(rp->graph); rp->graph = nullptr; }
  rp->warm = false;
  return HML_OK;
}

static uint64_t galois_of(const hml_ctx *ctx, uint32_t r) {
  const uint64_t m = 2ull * ctx->p.N;
  uint64_t g = 1;
  for (uint32_t i = 0; i < r; ++i) g = (g * 5) % m;
  return g;
}

// true when `slot` is dead from op `from` on: its next access, if any, is a write
static bool dead_from(const std::vector<hml_trace_op> &ops, size_t from, uint32_t slot) {
  for (size_t k = from; k < ops.size(); ++k) {
    const hml_trace_op &q = ops[k];
    if (q.a == slot || ((q.kind == HML_OP_HADD || q.kind == HML_OP_HMULT) && q.b == slot)) return false;
    if (q.dst == slot) return true;
  }
  return true;
}

// HML_REPLAY_HOIST_SUM: the rotations ops[i, j) of one source are followed directly by
//   pmult(y, d, pt), then n - 1 times  pmult(t, d, pt); hadd(y, y, t) (or hadd(y, t, y)),
// consuming every rotation output d exactly once, with y neither the source nor a rotation output, t none of y, the source or
// a rotation output, and every d and t dead afterwards.  On a match: *end = the op after the chain, *y = its slot and
// pt_of[k] = the plaintext that weights rotation i + k.
static bool match_rot_sum(const std::vector<hml_trace_op> &ops, size_t i, size_t j, size_t *end, uint32_t *y, std::vector<uint32_t> &pt_of) {
  const size_t n = j - i;
  const uint32_t src = ops[i].a, none = ~0u;
  auto rot_of = [&](uint32_t slot) -> size_t {
    for (size_t k = 0; k < n; ++k)
      if (ops[i + k].dst == slot) return k;
    return n;
  };
  pt_of.assign(n, none);
  size_t k = j;
  if (k >= ops.size() || ops[k].kind != HML_OP_PMULT) return false;
  const uint32_t acc = ops[k].dst;
  size_t r = rot_of(ops[k].a);
  if (r == n || acc == src || rot_of(acc) != n) return false;
  pt_of[r] = ops[k].b;
  std::vector<uint32_t> temps;
  for (k = j + 1; temps.size() + 1 < n; k += 2) {
    if (k + 1 >= ops.size()) return false;
    const hml_trace_op &pm = ops[k], &ad = ops[k + 1];
    if (pm.kind != HML_OP_PMULT || ad.kind != HML_OP_HADD) return false;
    const uint32_t t = pm.dst;
    r = rot_of(pm.a);
    if (r == n || pt_of[r] != none || t == acc || t == src || rot_of(t) != n) return false;
    if (ad.dst != acc || !((ad.a == acc && ad.b == t) || (ad.a == t && ad.b == acc))) return false;
    pt_of[r] = pm.b;
    temps.push_back(t);
  }
  for (size_t q = 0; q < n; ++q)
    if (!dead_from(ops, k, ops[i + q].dst)) return false;
  for (uint32_t t : temps)
    if (!dead_from(ops, k, t)) return false;
  *end = k;
  *y = acc;
  return true;
}

// HML_REPLAY_HMULT_SUM: ops[i] = hmult(y, a_0, b_0) is followed by n - 1 >= 1 pairs  hmult(t, a_k, b_k); hadd(y, y, t) (or
// hadd(y, t, y)), every product at the level of the first, y and every t neither a source of any product of the chain nor each
// other, and every t dead afterwards.  On a match: *end = the op after the chain and srcs[k] = the sources of product k.
static bool match_hmult_sum(const std::vector<hml_trace_op> &ops, const std::vector<uint32_t> &level, size_t i, size_t *end,
                            std::vector<std::pair<uint32_t, uint32_t>> &srcs) {
  const uint32_t y = ops[i].dst;
  srcs.assign(1, {ops[i].a, ops[i].b});
  std::vector<uint32_t> temps;
  size_t k = i + 1;
  for (; k + 1 < ops.size(); k += 2) {
    const hml_trace_op &mu = ops[k], &ad = ops[k + 1];
    if (mu.kind != HML_OP_HMULT || ad.kind != HML_OP_HADD || level[k] != level[i]) break;
    const uint32_t t = mu.dst;
    if (t == y || ad.dst != y || !((ad.a == y && ad.b == t) || (ad.a == t && ad.b == y))) break;
    srcs.push_back({mu.a, mu.b});
    temps.push_back(t);
  }
  if (temps.empty()) return false;
  for (const auto &s : srcs) {
    if (s.first == y || s.second == y) return false;
    for (uint32_t t : temps)
      if (s.first == t || s.second == t) return false;
  }
  for (uint32_t t : temps)
    if (!dead_from(ops, k, t)) return false;
  *end = k;
  return true;
}

static int enqueue(hml_replay *rp, cudaStream_t s) {
  hml_ctx *ctx = rp->ctx;
  void *st = (void *)s;
  int rc = HML_OK;
  for (size_t i = 0; i < rp->ops.size() && rc == HML_OK; ++i) {
    const hml_trace_op &o = rp->ops[i];
    const uint32_t L = rp->op_level[i];
    uint64_t *dst = rp->slot[o.dst];
    const uint64_t *a = rp->slot[o.a];
    switch (o.kind) {
      case HML_OP_HROTATE: {
        if (rp->flags & (HML_REPLAY_HOIST | HML_REPLAY_HOIST_SUM)) {
          // the run of consecutive rotations of the same source (none of which overwrites it) shares one ModUp
          size_t j = i;
          std::vector<const uint64_t *> keys;
          std::vector<uint64_t> gs;
          std::vector<uint64_t *> outs;
          while (j < rp->ops.size() && rp->ops[j].kind == HML_OP_HROTATE && rp->ops[j].a == o.a && rp->ops[j].dst != o.a && rp->op_level[j] == L) {
            bool dup = false;
            for (size_t k = i; k < j; ++k) dup |= rp->ops[k].dst == rp->ops[j].dst;
            if (dup) break;
            keys.push_back(rp->keys[rp->key_of_rot[rp->ops[j].b]]);
            gs.push_back(galois_of(ctx, rp->ops[j].b));
            outs.push_back(rp->slot[rp->ops[j].dst]);
            ++j;
          }
          size_t end;
          uint32_t y;
          std::vector<uint32_t> pt_of;
          if (outs.size() >= 2 && (rp->flags & HML_REPLAY_HOIST_SUM) && match_rot_sum(rp->ops, i, j, &end, &y, pt_of)) {
            std::vector<const uint64_t *> pts;
            for (uint32_t b : pt_of) pts.push_back(rp->pts[b]);
            rc = hml_hrotate_sum_hoisted(ctx, L, a, (uint32_t)outs.size(), keys.data(), rp->evk_q_limbs, gs.data(), pts.data(), rp->L,
                                         rp->slot[y], st);
            i = end - 1;
            break;
          }
          if (outs.size() >= 2 && (rp->flags & HML_REPLAY_HOIST)) {
            rc = rp->sh ? hml_hrotate_hoisted_sharded(rp->sh, L, a, (uint32_t)outs.size(), keys.data(), gs.data(), outs.data(), st)
                        : hml_hrotate_hoisted(ctx, L, a, (uint32_t)outs.size(), keys.data(), rp->evk_q_limbs, gs.data(), outs.data(), st);
            i = j - 1;
            break;
          }
        }
        const uint64_t *key = rp->keys[rp->key_of_rot[o.b]];
        rc = rp->sh ? hml_hrotate_sharded(rp->sh, L, a, key, galois_of(ctx, o.b), dst, st)
                    : hml_hrotate(ctx, L, a, key, rp->evk_q_limbs, galois_of(ctx, o.b), dst, st);
        break;
      }
      case HML_OP_PMULT: {
        // peephole: "t = a * pt; d = d + t" with t dead afterwards (its next access, if any, is a write) is ONE element-wise
        // pass d = a * pt + d (hml_pmult_add): the accumulation loops of rotation-heavy traces are made of exactly this pair
        if (i + 1 < rp->ops.size()) {
          const hml_trace_op &n = rp->ops[i + 1];
          const bool pair = n.kind == HML_OP_HADD && n.dst != o.dst && rp->op_level[i + 1] == L && ((n.a == n.dst && n.b == o.dst) || (n.b == n.dst && n.a == o.dst)) && o.a != n.dst;
          if (pair && dead_from(rp->ops, i + 2, o.dst)) {
            uint64_t *acc = rp->slot[n.dst];
            rc = rp->sh ? hml_ew_sharded(rp->sh, L, 3, a, rp->pts[o.b], acc, st) : hml_pmult_add(ctx, L, a, rp->pts[o.b], acc, acc, st);
            ++i;
            break;
          }
        }
        rc = rp->sh ? hml_ew_sharded(rp->sh, L, 1, a, rp->pts[o.b], dst, st) : hml_pmult(ctx, L, a, rp->pts[o.b], dst, st);
        break;
      }
      case HML_OP_PADD:
        rc = rp->sh ? hml_ew_sharded(rp->sh, L, 2, a, rp->pts[o.b], dst, st) : hml_padd(ctx, L, a, rp->pts[o.b], dst, st);
        break;
      case HML_OP_HADD:
        rc = rp->sh ? hml_ew_sharded(rp->sh, L, 0, a, rp->slot[o.b], dst, st) : hml_hadd(ctx, L, a, rp->slot[o.b], dst, st);
        break;
      case HML_OP_HMULT: {
        size_t end;
        std::vector<std::pair<uint32_t, uint32_t>> srcs;
        if ((rp->flags & HML_REPLAY_HMULT_SUM) && match_hmult_sum(rp->ops, rp->op_level, i, &end, srcs)) {
          std::vector<const uint64_t *> as, bs;
          for (const auto &s : srcs) { as.push_back(rp->slot[s.first]); bs.push_back(rp->slot[s.second]); }
          rc = hml_hmult_sum(ctx, L, (uint32_t)srcs.size(), as.data(), bs.data(), 1, rp->evk, rp->evk_q_limbs, dst, st);
          i = end - 1;
          break;
        }
        rc = rp->sh ? hml_hmult_sharded(rp->sh, L, a, rp->slot[o.b], rp->evk, dst, st)
                    : hml_hmult(ctx, L, a, rp->slot[o.b], rp->evk, rp->evk_q_limbs, dst, st);
        break;
      }
      default: rc = HML_ERR_INVALID;
    }
  }
  return rc;
}

extern "C" int hml_replay_run(hml_replay *rp, void *stream) {
  if (!rp) return HML_ERR_INVALID;
  if (!rp->bound) return rfail(rp, HML_ERR_INVALID, "hml_replay_bind has not been called");
  hml_ctx *ctx = rp->ctx;
  HML_CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaStream_t user = (cudaStream_t)stream;
  if (!(rp->flags & HML_REPLAY_GRAPH)) return enqueue(rp, user);
  int rc;
  if (!rp->exec) {
    if (!rp->cap_stream) HML_CU_TRY(ctx, cudaStreamCreateWithFlags(&rp->cap_stream, cudaStreamNonBlocking));
    // order the private stream after the caller's (inputs), then warm up outside the capture: builds every per-level table,
    // sizes the workspace, maps the peers — nothing may allocate or synchronise while the stream is capturing
    cudaEvent_t ev;
    HML_CU_TRY(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaEventRecord(ev, user);
    cudaStreamWaitEvent(rp->cap_stream, ev, 0);
    cudaEventDestroy(ev);
    if (rp->sh) {  // every level the trace runs at: tables, peer offsets, workspace — nothing may allocate during the capture
      for (uint32_t l : rp->op_level)
        if ((rc = hml_shard_prepare(rp->sh, l))) return rc;
    }
    if (!rp->warm) {
      if ((rc = enqueue(rp, rp->cap_stream))) return rc;
      rp->warm = true;
    }
    HML_CU_TRY(ctx, cudaStreamSynchronize(rp->cap_stream));
    ctx->have_last = false;  // everything has completed; the capture must not wait on an event of another stream
    HML_CU_TRY(ctx, cudaStreamBeginCapture(rp->cap_stream, cudaStreamCaptureModeThreadLocal));
    rc = enqueue(rp, rp->cap_stream);
    cudaError_t e = cudaStreamEndCapture(rp->cap_stream, &rp->graph);
    ctx->have_last = false;
    if (rc) { if (rp->graph) { cudaGraphDestroy(rp->graph); rp->graph = nullptr; } return rc; }
    if (e != cudaSuccess) return rfail(rp, HML_ERR_CUDA, std::string("replay: graph capture failed: ") + cudaGetErrorString(e));
    HML_CU_TRY(ctx, cudaGraphInstantiate(&rp->exec, rp->graph, 0));
  }
  ws_enter(ctx, user);
  HML_CU_TRY(ctx, cudaGraphLaunch(rp->exec, user));
  return HML_OK;
}

extern "C" int hml_replay_slot(hml_replay *rp, uint32_t slot, uint64_t **ptr, uint32_t *n_limbs) {
  if (!rp || slot >= rp->n_slots || !rp->slot[slot] || !rp->final_level[slot]) return HML_ERR_INVALID;
  if (ptr) *ptr = rp->slot[slot];
  if (n_limbs) {  // limbs per polynomial of the slot's final content (the rank's owned limbs when sharded)
    uint32_t nq = rp->final_level[slot];
    if (rp->sh) {
      int rc = hml_shard_own_limbs(rp->sh, rp->final_level[slot], &nq, nullptr);
      if (rc) return rc;
    }
    *n_limbs = nq;
  }
  return HML_OK;
}

extern "C" int hml_replay_slot_level(hml_replay *rp, uint32_t slot, uint32_t *level) {
  if (!rp || !level || slot >= rp->n_slots || !rp->final_level[slot]) return HML_ERR_INVALID;
  *level = rp->final_level[slot];
  return HML_OK;
}
