// hml_ctx: tables, per-level constants, workspace, and the composition of the reference's ops out of the
// kernels in ntt.cu / ewe.cu.  Stage order follows the reference's constructors:
//   KeySwitch  reference src/Operation.cpp:9-54      Rescale  :741-911
//   HMULT      :913-1023      HROTATE :1271-1358      HADD :1114-1176   PMULT :1453-1523   PADD :1618-1680
#include "context.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "launch.h"
#include "ops.h"
#include "planner.h"

using namespace hml;

// Strided view of `nb` independent polynomials / ciphertext halves: item b lives at ptr + b * stride (words).
struct BatchPtr {
  const u64 *ptr;
  long long stride;
};
struct BatchOut {
  u64 *ptr;
  long long stride;
};

// hrotate on two-pass rings: the automorphism rides on the key switch's loads instead of a kernel of its own.  d and add0 are
// the RAW polynomials; the ModUp INTT reads d through sigma_g and leaves sigma_g(d) in sigma_d (item b at + b * sigma_stride)
// for the inner product's own-digit term; the ModDown epilogue reads add0 through sigma_g.
struct KsAuto {
  u64 g;
  u64 *sigma_d;
  long long sigma_stride;
};

// hmult's merged ModDown + Rescale: the addend d_c[L-1] of u[L-1] = acc_c[L-1] * P^-1 + d_c[L-1] (packed limbs; component c at
// add + c * comp_stride, ciphertext b at + b * batch_stride)
struct MergedU {
  const u64 *add;
  long long comp_stride, batch_stride;
};

// The batched hmult's ciphertext pairs (a, b), component c of pair b at a + b * batch_stride + c * comp_stride: the key switch
// squares c1 on the ModUp transform's load (d2 = a1 * b1, NttLaunch::in_mul) and forms the tensor product in the inner
// product (InnerArgs::ct_a), so that d0, d1 and d2 never reach memory.
struct KsTensor {
  const u64 *a, *b;
  long long comp_stride, batch_stride;
};

static thread_local std::string g_create_err;

#define CU_TRY(ctx, call)                                                                          \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                             \
      return HML_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)

int fail(hml_ctx *ctx, int code, const std::string &msg) {
  ctx->err = msg;
  return code;
}

namespace hml {
void ws_enter(hml_ctx *ctx, cudaStream_t s) {
  if (ctx->have_last && ctx->last_stream != s) {
    // everything queued so far on the previous stream (a superset of the ops that used the workspace) precedes this op
    if (!ctx->ev_ws) cudaEventCreateWithFlags(&ctx->ev_ws, cudaEventDisableTiming);
    if (ctx->ev_ws && cudaEventRecord(ctx->ev_ws, ctx->last_stream) == cudaSuccess) cudaStreamWaitEvent(s, ctx->ev_ws, 0);
    else cudaGetLastError();  // the previous stream no longer exists: nothing of it can still be running
  }
  ctx->last_stream = s;
  ctx->have_last = true;
}
void prof_mark(hml_ctx *ctx, int cls, cudaStream_t s) {
  if (!ctx->prof.on) return;
  cudaEvent_t e = nullptr;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, s);
  ctx->prof.marks.emplace_back(cls, e);
}
}  // namespace hml

extern "C" int hml_profile_begin(hml_ctx *ctx, void *stream) {
  if (!ctx) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (auto &m : ctx->prof.marks) cudaEventDestroy(m.second);
  ctx->prof.marks.clear();
  if (!ctx->prof.start) CU_TRY(ctx, cudaEventCreate(&ctx->prof.start));
  CU_TRY(ctx, cudaEventRecord(ctx->prof.start, (cudaStream_t)stream));
  ctx->prof.on = true;
  return HML_OK;
}
extern "C" int hml_profile_end(hml_ctx *ctx, hml_profile *out) {
  if (!ctx || !out) return HML_ERR_INVALID;
  if (!ctx->prof.on) return fail(ctx, HML_ERR_INVALID, "hml_profile_end without hml_profile_begin");
  ctx->prof.on = false;
  memset(out, 0, sizeof(*out));
  cudaEvent_t prev = ctx->prof.start;
  cudaError_t e = cudaSuccess;
  static const bool dump = getenv("HML_PROFILE_DUMP") != nullptr;  // per-launch-group times on stderr (tuning aid)
  static const char *cls_name[HML_CLS_COUNT] = {"NTT", "INTT", "BCONV", "EWE", "AUTO"};
  int idx = 0;
  for (auto &m : ctx->prof.marks) {
    if (e == cudaSuccess) e = cudaEventSynchronize(m.second);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, prev, m.second);
    if (dump && e == cudaSuccess) fprintf(stderr, "[hml profile] %2d %-5s %8.2f us\n", idx, m.first >= 0 && m.first < HML_CLS_COUNT ? cls_name[m.first] : "?", ms * 1e3);
    ++idx;
    if (e == cudaSuccess && m.first >= 0 && m.first < HML_CLS_COUNT) {
      out->us[m.first] += ms * 1e3;
      out->launches[m.first]++;
      out->total_us += ms * 1e3;
    }
    prev = m.second;
  }
  for (auto &m : ctx->prof.marks) cudaEventDestroy(m.second);
  ctx->prof.marks.clear();
  if (e != cudaSuccess) return fail(ctx, HML_ERR_CUDA, std::string("profile: ") + cudaGetErrorString(e));
  return HML_OK;
}

static double2 mk_cst(u64 c, u64 q) { return make_double2((double)c, (double)c / (double)q); }

template <class T>
static int upload(hml_ctx *ctx, const std::vector<T> &h, T **dev) {
  CU_TRY(ctx, cudaMalloc((void **)dev, std::max<size_t>(1, h.size()) * sizeof(T)));
  if (!h.empty()) CU_TRY(ctx, cudaMemcpy(*dev, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  return HML_OK;
}

// A base conversion prepared for launch: the matrix in 12-bit pieces, zero-padded, uploaded once; the destination LimbMap.
// dst_pos[t] = limb slot (in the output buffer) of destination t.
// fold_c (optional): the constants of BConvArgs::fold as integers, modulus index fold_mod; the tcgen05 image then carries the
// fold as a virtual target (bconv_umma.cu) while the DMMA kernel keeps using the caller's 12-bit pieces.
static int prepare_bconv(hml_ctx *ctx, const BConvTable &bt, const std::vector<uint32_t> &dst_pos, hml::HostBConv &out,
                         const std::vector<u64> *fold_c = nullptr, uint32_t fold_mod = 0) {
  const int ns = (int)bt.src.size(), nd = (int)bt.dst.size();
  const int nsp = bconv_pad_src(ns), ndp = bconv_pad_dst(nd);
  out.n_src = ns; out.n_dst = nd;
  memset(&out.dst_lm, 0, sizeof(out.dst_lm));
  std::vector<double> m((size_t)nsp * ndp * 3, 0.0);
  for (int t = 0; t < nd; ++t) {
    out.dst_lm.mod[t] = (uint16_t)bt.dst[t];
    out.dst_lm.pos[t] = (uint16_t)dst_pos[t];
    for (int i = 0; i < ns; ++i) {
      const u64 h = bt.hat[(size_t)i * nd + t];
      double *d = &m[((size_t)i * ndp + t) * 3];
      d[0] = (double)(h & 0xFFF);
      d[1] = (double)((h >> 12) & 0xFFF);
      d[2] = (double)(h >> 24);
    }
  }
  {
    std::vector<u64> dq(nd);
    for (int t = 0; t < nd; ++t) dq[t] = ctx->p.mod[bt.dst[t]];
    std::vector<uint8_t> img;
    BConvImage im;
    if (bconv_image_build(bt.hat.data(), ns, nd, dq.data(), fold_c ? fold_c->data() : nullptr, fold_c ? ctx->p.mod[fold_mod] : 0, img, im)) {
      int rc = upload(ctx, img, &out.d_img);
      if (rc) return rc;
      im.img = out.d_img;
      out.im = im;
    }
  }
  return upload(ctx, m, &out.d_mat);
}

static void run_bconv(hml_ctx *ctx, const hml::HostBConv &hb, const LimbMap &src_lm, BConvArgs a, cudaStream_t s) {
  a.n_src = hb.n_src; a.n_dst = hb.n_dst;
  launch_bconv(ctx->mc, src_lm, hb.dst_lm, a, hb.d_mat, s, &hb.im);
  prof_mark(ctx, HML_CLS_BCONV, s);
  ctx->exec.kernel_launches++;
  ctx->exec.bconv_limb_macs += (uint64_t)hb.n_src * hb.n_dst * a.n_batches;
}

// A forward or inverse transform and its counters: n_batch x the (poly, limb) pairs that the map does not skip
static void run_ntt(hml_ctx *ctx, bool inverse, const LimbMap &lm, const NttLaunch &l, cudaStream_t s) {
  if (inverse) launch_ntt_inverse(ctx->tabs, ctx->p.logN, lm, l, s);
  else launch_ntt_forward(ctx->tabs, ctx->p.logN, lm, l, s);
  prof_mark(ctx, inverse ? HML_CLS_INTT : HML_CLS_NTT, s);
  uint64_t limbs = 0;
  for (int poly = 0; poly < l.n_polys; ++poly)
    for (int k = 0; k < l.n_limbs; ++k) limbs += lm.skip[k] != poly;
  (inverse ? ctx->exec.intt_limbs : ctx->exec.ntt_limbs) += limbs * l.n_batch;
  ctx->exec.kernel_launches += ctx->p.logN <= NTT_SMALL_LOG ? 1 : 2;
}

// K9 + K10 of a ModDown, and the transform + subtract of a rescale: the forward transform of l, then for every poly
// p = b * n_c + c of it  dst_c[b] = (x_c[b] - NTT(in)_p) * cst (+ z_c[b] when bit c of z_mask is set), as l.fuse describes.
// Two-pass rings run it as the transform's fused epilogue.  Single-pass rings store the transform in l.out and run
// k_sub_mul_add over the same description: one launch when n_b = 1 (the components are its polys), else one per component.
static int ntt_sub_mul(hml_ctx *ctx, const LimbMap &lm, NttLaunch l, cudaStream_t s) {
  const NttFuse f = l.fuse;
  if (ctx->p.logN > NTT_SMALL_LOG) {
    run_ntt(ctx, false, lm, l, s);
    return HML_OK;
  }
  if (f.z_galois) return fail(ctx, HML_ERR_INVALID, "automorphism on the addend needs the fused ModDown epilogue");
  l.fuse = NttFuse{};
  run_ntt(ctx, false, lm, l, s);
  SubMulArgs a{};
  a.cst = f.cst; a.N = ctx->p.N; a.n_limbs = l.n_limbs; a.x_packed = f.x_packed; a.z_packed = f.z_packed;
  const int n_b = l.n_polys / f.n_c;
  if (n_b == 1) {
    a.x = f.x; a.x_poly_stride = f.x_c_stride;
    a.y = l.out; a.y_poly_stride = l.out_poly_stride;
    a.z = f.z_mask ? f.z : nullptr; a.z_poly_stride = f.z_c_stride; a.z_mask = f.z_mask;
    a.out = f.dst; a.out_poly_stride = f.dst_c_stride; a.n_polys = f.n_c;
    launch_sub_mul_add(ctx->mc, lm, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.kernel_launches++;
    return HML_OK;
  }
  for (int c = 0; c < f.n_c; ++c) {
    a.x = f.x + c * f.x_c_stride; a.x_poly_stride = f.x_b_stride;
    a.y = l.out + c * l.out_poly_stride; a.y_poly_stride = f.n_c * l.out_poly_stride;
    a.z = (f.z_mask >> c) & 1u ? f.z + c * f.z_c_stride : nullptr; a.z_poly_stride = f.z_b_stride;
    a.out = f.dst + c * f.dst_c_stride; a.out_poly_stride = f.dst_b_stride; a.n_polys = n_b;
    launch_sub_mul_add(ctx->mc, lm, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.kernel_launches++;
  }
  return HML_OK;
}

// Device job table of the one-launch ModUp: digit j reads its sources at in + j * in_step (slots 0.., or through
// (*src_off)[j]) and writes at out + j * out_step.  Left null for one digit or a digit the multi-conversion form cannot take.
static int upload_up_jobs(hml_ctx *ctx, const std::vector<HostBConv> &up, long long in_step, long long out_step,
                          const std::vector<long long *> *src_off, BConvJob **out) {
  *out = nullptr;
  if (up.size() < 2) return HML_OK;
  std::vector<BConvJob> jobs(up.size());
  for (size_t j = 0; j < up.size(); ++j) {
    const HostBConv &hb = up[j];
    if (!hb.d_img || hb.n_src > 48 || hb.n_dst > 48) return HML_OK;
    BConvJob &jb = jobs[j];
    memset(&jb, 0, sizeof(jb));
    for (int i = 0; i < hb.n_src; ++i) jb.src_pos[i] = (uint16_t)i;
    for (int t = 0; t < hb.n_dst; ++t) { jb.dst_mod[t] = hb.dst_lm.mod[t]; jb.dst_pos[t] = hb.dst_lm.pos[t]; }
    jb.img = hb.d_img; jb.K = hb.im.K; jb.NP = hb.im.NP; jb.ND = hb.im.ND; jb.n_src = hb.n_src; jb.n_dst = hb.n_dst;
    jb.in_off = (long long)j * in_step; jb.out_off = (long long)j * out_step; jb.src_off = src_off ? (*src_off)[j] : nullptr;
  }
  return upload(ctx, jobs, out);
}

// The ModUp conversions (K3) of every digit j: up[j] from `a.in + j * in_step` (source map src_lm[j], offsets (*src_off)[j]
// when given) to `a.out + j * out_step`.  ONE launch for all digits when a job table is given and the tcgen05 kernel's
// multi-conversion form takes it (every CTA serves one digit), else one launch per digit that has targets.
static void run_modup_bconv(hml_ctx *ctx, const std::vector<HostBConv> &up, const std::vector<LimbMap> &src_lm, const BConvJob *jobs,
                            const std::vector<long long *> *src_off, const BConvArgs &a, long long in_step, long long out_step, cudaStream_t s) {
  const int beta = (int)up.size();
  if (jobs) {
    std::vector<BConvImage> ims(beta);
    std::vector<int> nd(beta);
    for (int j = 0; j < beta; ++j) { ims[j] = up[j].im; nd[j] = up[j].n_dst; }
    if (launch_bconv_umma_multi(ctx->mc, jobs, ims.data(), nd.data(), beta, a, s)) {
      prof_mark(ctx, HML_CLS_BCONV, s);
      ctx->exec.kernel_launches++;
      for (int j = 0; j < beta; ++j) ctx->exec.bconv_limb_macs += (uint64_t)up[j].n_src * up[j].n_dst * a.n_batches;
      return;
    }
  }
  for (int j = 0; j < beta; ++j) {
    if (up[j].empty()) continue;
    BConvArgs aj = a;
    aj.in = a.in + j * in_step; aj.out = a.out + j * out_step; aj.src_off = src_off ? (*src_off)[j] : nullptr;
    run_bconv(ctx, up[j], src_lm[j], aj, s);
  }
}

// ------------------------------------------------------------------------------------------------ creation
static int ctx_init_device(hml_ctx *ctx) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    ctx->err = std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e);
    return HML_ERR_CUDA;
  }
  if (ctx->device < 0 || ctx->device >= ndev) return fail(ctx, HML_ERR_INVALID, "device index out of range");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const Params &p = ctx->p;
  const size_t N = p.N, nm = p.n_mod();
  const bool two_pass = p.logN > NTT_SMALL_LOG;
  std::vector<double> f(nm * N), iv(nm * N), fr(two_pass ? nm * N : 0), ir(two_pass ? nm * N : 0);
  std::vector<ModConst> mc(nm);
  std::vector<u64> tw;
  for (uint32_t i = 0; i < nm; ++i) {
    const u64 q = p.mod[i];
    const double qd = (double)q;
    p.twiddles(i, false, tw);
    for (size_t k = 0; k < N; ++k) f[i * N + k] = (double)tw[k];
    p.twiddles(i, true, tw);
    for (size_t k = 0; k < N; ++k) iv[i * N + k] = (double)tw[k];
    if (two_pass) {
      ntt_permute_row_twiddles(&f[i * N], (int)p.logN, &fr[i * N]);
      ntt_permute_row_twiddles(&iv[i * N], (int)p.logN, &ir[i * N]);
    }
    mc[i].q = qd; mc[i].qinv = 1.0 / qd;
    mc[i].ninv = (double)p.n_inv[i]; mc[i].ninv_q = (double)p.n_inv[i] / qd;
    mc[i].qi = q; mc[i].pad = 0;
  }
  int rc;
  if ((rc = upload(ctx, f, &ctx->tw_fwd))) return rc;
  if ((rc = upload(ctx, iv, &ctx->tw_inv))) return rc;
  if ((rc = upload(ctx, fr, &ctx->tw_fwd_rows))) return rc;
  if ((rc = upload(ctx, ir, &ctx->tw_inv_rows))) return rc;
  if ((rc = upload(ctx, mc, &ctx->mc))) return rc;
  ctx->tabs.fwd_rows = ctx->tw_fwd_rows; ctx->tabs.inv_rows = ctx->tw_inv_rows;
  ctx->tabs.fwd = ctx->tw_fwd; ctx->tabs.inv = ctx->tw_inv; ctx->tabs.mc = ctx->mc;
  if (two_pass) {
    CU_TRY(ctx, cudaMalloc((void **)&ctx->col_ctr, 2 * sizeof(unsigned)));
    CU_TRY(ctx, cudaMemset(ctx->col_ctr, 0, 2 * sizeof(unsigned)));
    ctx->tabs.col_ctr = ctx->col_ctr;
  }
  return HML_OK;
}

extern "C" int hml_ctx_create_params(uint32_t N, uint32_t element_bit_width, uint32_t batch_size, uint32_t max_level,
                                     uint32_t alpha, int device, hml_ctx **out) {
  if (!out) { g_create_err = "out is null"; return HML_ERR_INVALID; }
  *out = nullptr;
  hml_ctx *ctx = new hml_ctx();
  ctx->device = device;
  std::string err;
  if (!ctx->p.init(N, element_bit_width, batch_size, max_level, alpha, err)) {
    g_create_err = err; delete ctx; return HML_ERR_UNSUPPORTED;
  }
  if (max_level + alpha > NTT_MAX_LIMBS) {
    g_create_err = "maxLevel + alpha > 128 is not supported"; delete ctx; return HML_ERR_UNSUPPORTED;
  }
  int rc = ctx_init_device(ctx);
  if (rc) { g_create_err = ctx->err; hml_ctx_destroy(ctx); return rc; }
  *out = ctx;
  return HML_OK;
}

extern "C" int hml_ctx_create(const char *cfg_path, uint32_t max_level, uint32_t alpha, int device, hml_ctx **out) {
  if (!out || !cfg_path) { g_create_err = "null argument"; return HML_ERR_INVALID; }
  *out = nullptr;
  CfgFile cfg;
  std::string err;
  if (!cfg.load(cfg_path, err)) { g_create_err = err; return HML_ERR_CONFIG; }
  uint32_t N, bs, w;
  if (!cfg.get("N", N) || !cfg.get("batchSize", bs) || !cfg.get("elementBitWidth", w)) {
    g_create_err = "Can not find this key! (N, batchSize and elementBitWidth are required)";
    return HML_ERR_CONFIG;
  }
  int rc = hml_ctx_create_params(N, w, bs, max_level, alpha, device, out);
  if (rc) return rc;
  (*out)->cfg = cfg; (*out)->has_cfg = true;
  (*out)->p.bconv_high = cfg.get_or("bconv_num_high", 2);
  (*out)->p.bconv_width = cfg.get_or("bconv_num_width", 6);
  return HML_OK;
}

static void free_level(LevelConsts &lc) {
  cudaFree(lc.modup_scale); cudaFree(lc.moddown_scale); cudaFree(lc.moddown_scale_u); cudaFree(lc.pinv); cudaFree(lc.pmod); cudaFree(lc.qlinv);
  for (auto &u : lc.up) { cudaFree(u.d_mat); cudaFree(u.d_img); }
  cudaFree(lc.down.d_mat); cudaFree(lc.merged_rest.d_mat); cudaFree(lc.merged_fold);
  cudaFree(lc.down.d_img); cudaFree(lc.merged_rest.d_img); cudaFree(lc.up_jobs);
}

extern "C" void hml_ctx_destroy(hml_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (auto &kv : ctx->levels) free_level(kv.second);
  for (auto &kv : ctx->bconv_cache) { cudaFree(kv.second.step1); cudaFree(kv.second.host.d_mat); cudaFree(kv.second.host.d_img); }
  for (auto &kv : ctx->shard_plans) {
    cudaFree(kv.second.scale1); cudaFree(kv.second.scale2); cudaFree(kv.second.pinv); cudaFree(kv.second.down.d_mat); cudaFree(kv.second.down.d_img);
    cudaFree(kv.second.d_off2); cudaFree(kv.second.qlinv_own); cudaFree(kv.second.up_jobs);
    for (auto *o : kv.second.d_off1) cudaFree(o);
    for (auto &u : kv.second.up) { cudaFree(u.d_mat); cudaFree(u.d_img); }
  }
  cudaFree(ctx->tw_fwd); cudaFree(ctx->tw_inv); cudaFree(ctx->tw_fwd_rows); cudaFree(ctx->tw_inv_rows); cudaFree(ctx->mc); cudaFree(ctx->ws); cudaFree(ctx->stage); cudaFree(ctx->col_ctr);
  if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
  if (ctx->s_comp) cudaStreamDestroy(ctx->s_comp);
  if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
  if (ctx->ev_ws) cudaEventDestroy(ctx->ev_ws);
  if (ctx->prof.start) cudaEventDestroy(ctx->prof.start);
  for (auto &m : ctx->prof.marks) cudaEventDestroy(m.second);
  delete ctx;
}

extern "C" const char *hml_last_error(const hml_ctx *ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }
extern "C" const char *hml_last_create_error(void) { return g_create_err.c_str(); }
extern "C" uint32_t hml_ring_degree(const hml_ctx *ctx) { return ctx->p.N; }
extern "C" uint32_t hml_n_moduli(const hml_ctx *ctx) { return ctx->p.n_mod(); }
extern "C" int hml_get_moduli(const hml_ctx *ctx, uint64_t *out, uint32_t cap) {
  if (!ctx || !out || cap < ctx->p.n_mod()) return HML_ERR_INVALID;
  for (uint32_t i = 0; i < ctx->p.n_mod(); ++i) out[i] = ctx->p.mod[i];
  return HML_OK;
}
extern "C" int hml_get_roots(const hml_ctx *ctx, uint64_t *out, uint32_t cap) {
  if (!ctx || !out || cap < ctx->p.n_mod()) return HML_ERR_INVALID;
  for (uint32_t i = 0; i < ctx->p.n_mod(); ++i) out[i] = ctx->p.psi[i];
  return HML_OK;
}

// ------------------------------------------------------------------------------------------------ memory helpers
extern "C" int hml_dev_alloc(hml_ctx *ctx, uint64_t n_words, uint64_t **out) {
  if (!ctx || !out) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaMalloc((void **)out, std::max<uint64_t>(1, n_words) * 8));
  return HML_OK;
}
extern "C" int hml_dev_free(hml_ctx *ctx, uint64_t *ptr) { CU_TRY(ctx, cudaFree(ptr)); return HML_OK; }
extern "C" int hml_h2d(hml_ctx *ctx, uint64_t *dst, const uint64_t *src, uint64_t n, void *stream) {
  CU_TRY(ctx, cudaMemcpyAsync(dst, src, n * 8, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return HML_OK;
}
extern "C" int hml_d2h(hml_ctx *ctx, uint64_t *dst, const uint64_t *src, uint64_t n, void *stream) {
  CU_TRY(ctx, cudaMemcpyAsync(dst, src, n * 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  return HML_OK;
}
extern "C" int hml_sync(hml_ctx *ctx, void *stream) { CU_TRY(ctx, cudaStreamSynchronize((cudaStream_t)stream)); return HML_OK; }
extern "C" int hml_host_alloc_pinned(hml_ctx *ctx, uint64_t n_words, uint64_t **out) {
  CU_TRY(ctx, cudaMallocHost((void **)out, std::max<uint64_t>(1, n_words) * 8));
  return HML_OK;
}
extern "C" int hml_host_free_pinned(hml_ctx *ctx, uint64_t *ptr) { CU_TRY(ctx, cudaFreeHost(ptr)); return HML_OK; }

int ensure_ws(hml_ctx *ctx, size_t words) {
  if (ctx->ws_words >= words) return HML_OK;
  // growing the workspace must not race with work already queued on it
  CU_TRY(ctx, cudaDeviceSynchronize());
  if (ctx->ws) CU_TRY(ctx, cudaFree(ctx->ws));
  ctx->ws = nullptr; ctx->ws_words = 0;
  CU_TRY(ctx, cudaMalloc((void **)&ctx->ws, words * 8));
  ctx->ws_words = words;
  return HML_OK;
}

static int check_launch(hml_ctx *ctx, const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { ctx->err = std::string(what) + ": " + cudaGetErrorString(e); return HML_ERR_CUDA; }
  return HML_OK;
}

static void clear_map(LimbMap &lm) {
  memset(&lm, 0, sizeof(lm));
  memset(lm.skip, 0xFF, sizeof(lm.skip));
}

static void id_map(LimbMap &lm, const uint32_t *mod_idx, uint32_t n) {
  clear_map(lm);
  for (uint32_t i = 0; i < n; ++i) { lm.mod[i] = (uint16_t)mod_idx[i]; lm.pos[i] = (uint16_t)i; }
}

// ------------------------------------------------------------------------------------------------ per-level constants
static int get_level(hml_ctx *ctx, uint32_t L, LevelConsts **out) {
  auto it = ctx->levels.find(L);
  if (it != ctx->levels.end()) { *out = &it->second; return HML_OK; }
  const Params &p = ctx->p;
  const uint32_t A = p.alpha, E = L + A, beta = p.beta(L);
  LevelConsts lc;
  lc.L = L; lc.beta = beta; lc.E = E;
  clear_map(lc.q_lm); clear_map(lc.p_lm); clear_map(lc.ext_lm);
  for (uint32_t i = 0; i < L; ++i) { lc.q_lm.mod[i] = i; lc.q_lm.pos[i] = i; }
  for (uint32_t j = 0; j < A; ++j) { lc.p_lm.mod[j] = p.max_level + j; lc.p_lm.pos[j] = L + j; }
  int rc;
  // ---- ModUp
  std::vector<double2> up_scale(L);
  for (uint32_t i = 0; i < L; ++i) up_scale[i] = mk_cst(p.modup_scale(L, i), p.mod[i]);
  for (uint32_t e = 0; e < E; ++e) {
    lc.ext_lm.mod[e] = p.ext_mod(L, e); lc.ext_lm.pos[e] = e;
    lc.ext_lm.skip[e] = e < L ? (uint8_t)(e / A) : 0xFF;  // digit j owns limbs [j*alpha, j*alpha + a_j)
  }
  for (uint32_t j = 0; j < beta; ++j) {
    const uint32_t lo = j * A, aj = p.digit_size(L, j);
    std::vector<uint32_t> src, dst, dst_pos;
    for (uint32_t i = 0; i < aj; ++i) src.push_back(lo + i);
    for (uint32_t e = 0; e < E; ++e) {
      if (e >= lo && e < lo + aj) continue;
      dst.push_back(p.ext_mod(L, e));
      dst_pos.push_back(e);
    }
    BConvTable bt;
    make_bconv_table(p, src, dst, bt);
    lc.up.emplace_back();
    lc.up_src.push_back(lc.q_lm);
    if ((rc = prepare_bconv(ctx, bt, dst_pos, lc.up.back()))) return rc;
  }
  if ((rc = upload(ctx, up_scale, &lc.modup_scale))) return rc;
  // the merged ModUp launch: sources at yb + j * alpha limbs, targets at ext + j * E limbs
  if ((rc = upload_up_jobs(ctx, lc.up, (long long)A * p.N, (long long)E * p.N, nullptr, &lc.up_jobs))) return rc;
  // ---- ModDown
  {
    std::vector<uint32_t> src, dst;
    for (uint32_t j = 0; j < A; ++j) src.push_back(p.max_level + j);
    for (uint32_t i = 0; i < L; ++i) dst.push_back(i);
    BConvTable bt;
    make_bconv_table(p, src, dst, bt);
    std::vector<double2> sc(A), pinv(L);
    for (uint32_t j = 0; j < A; ++j) sc[j] = mk_cst(p.moddown_scale(j), p.mod[p.max_level + j]);
    std::vector<double2> pmod(L);
    for (uint32_t i = 0; i < L; ++i) {
      pinv[i] = mk_cst(p.p_inv(i), p.mod[i]);
      u64 pm = 1;
      for (uint32_t j = 0; j < A; ++j) pm = h_mulmod(pm, p.mod[p.max_level + j] % p.mod[i], p.mod[i]);
      pmod[i] = mk_cst(pm, p.mod[i]);
    }
    if ((rc = prepare_bconv(ctx, bt, dst, lc.down))) return rc;
    if ((rc = upload(ctx, sc, &lc.moddown_scale))) return rc;
    if ((rc = upload(ctx, pinv, &lc.pinv))) return rc;
    if ((rc = upload(ctx, pmod, &lc.pmod))) return rc;
    // hmult's merged path: the P-limbs plus slot E (modulus q_{L-1}, plain N^-1) in one INTT launch
    lc.pu_lm = lc.p_lm;
    lc.pu_lm.mod[A] = (uint16_t)(L - 1); lc.pu_lm.pos[A] = (uint16_t)E;
    sc.push_back(mk_cst(p.n_inv[L - 1], p.mod[L - 1]));
    if ((rc = upload(ctx, sc, &lc.moddown_scale_u))) return rc;
    lc.pinv_last = pinv[L - 1];
  }
  // ---- hmult: ModDown merged with Rescale (matrices with P^-1 folded in and a unit row for the extra source)
  if (L >= 2) {
    std::vector<uint32_t> src, dst;
    for (uint32_t j = 0; j < A; ++j) src.push_back(p.max_level + j);
    for (uint32_t i = 0; i < L; ++i) dst.push_back(i);
    BConvTable bt;
    make_bconv_table(p, src, dst, bt);
    std::vector<u64> pinv_i(L);
    for (uint32_t i = 0; i < L; ++i) pinv_i[i] = p.p_inv(i);
    clear_map(lc.merged_src); clear_map(lc.last_lm);
    for (uint32_t j = 0; j < A; ++j) { lc.merged_src.mod[j] = p.max_level + j; lc.merged_src.pos[j] = L + j; }
    lc.merged_src.mod[A] = L - 1; lc.merged_src.pos[A] = E;  // the extra source lives in slot E of the accumulator
    lc.last_lm.mod[0] = L - 1; lc.last_lm.pos[0] = 0;
    BConvTable rest;
    rest.src = src; rest.src.push_back(L - 1);
    for (uint32_t i = 0; i + 1 < L; ++i) rest.dst.push_back(i);
    const uint32_t nr = L - 1;
    rest.hat.assign((size_t)(A + 1) * nr, 0);
    std::vector<double> fold(3 * (size_t)A);
    std::vector<u64> fold_c(A);
    for (uint32_t j = 0; j < A; ++j) {
      for (uint32_t i = 0; i < nr; ++i) rest.hat[(size_t)j * nr + i] = h_mulmod(bt.hat[(size_t)j * L + i], pinv_i[i], p.mod[i]);
      const u64 ql = p.mod[L - 1], t = h_mulmod(bt.hat[(size_t)j * L + L - 1], pinv_i[L - 1], ql);
      const u64 neg = t ? ql - t : 0;  // minus: r = slot_E - v[L-1] * P^-1
      fold_c[j] = neg;
      fold[3 * j] = (double)(neg & 0xFFF); fold[3 * j + 1] = (double)((neg >> 12) & 0xFFF); fold[3 * j + 2] = (double)(neg >> 24);
    }
    for (uint32_t i = 0; i < nr; ++i) rest.hat[(size_t)A * nr + i] = 1;
    std::vector<uint32_t> rest_pos(nr);
    for (uint32_t i = 0; i < nr; ++i) rest_pos[i] = i;
    if ((rc = prepare_bconv(ctx, rest, rest_pos, lc.merged_rest, &fold_c, L - 1))) return rc;
    if ((rc = upload(ctx, fold, &lc.merged_fold))) return rc;
  }
  // ---- Rescale
  {
    std::vector<double2> ql(L > 1 ? L - 1 : 0);
    for (uint32_t l = 0; l + 1 < L; ++l) ql[l] = mk_cst(p.ql_inv(L, l), p.mod[l]);
    if ((rc = upload(ctx, ql, &lc.qlinv))) return rc;
  }
  auto ins = ctx->levels.emplace(L, lc);
  *out = &ins.first->second;
  return HML_OK;
}

int check_level(hml_ctx *ctx, uint32_t L, uint32_t min_level) {
  if (!ctx) return HML_ERR_INVALID;
  if (L < min_level || L > ctx->p.max_level) return fail(ctx, HML_ERR_INVALID, "currentLevel out of range");
  return HML_OK;
}

// ------------------------------------------------------------------------------------------------ primitives
static int ntt_api(hml_ctx *ctx, bool inverse, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs,
                   void *stream) {
  if (!ctx || !in || !out || !mod_idx) return HML_ERR_INVALID;
  const size_t N = ctx->p.N;
  for (uint32_t i = 0; i < n_limbs; ++i)
    if (mod_idx[i] >= ctx->p.n_mod()) return fail(ctx, HML_ERR_INVALID, "modulus index out of range");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ws_enter(ctx, (cudaStream_t)stream);  // the transform's queue counters are per ctx, like the workspace
  for (uint32_t off = 0; off < n_limbs; off += NTT_MAX_LIMBS) {
    const uint32_t n = std::min<uint32_t>(NTT_MAX_LIMBS, n_limbs - off);
    LimbMap lm;
    id_map(lm, mod_idx + off, n);
    NttLaunch l{};
    l.n_batch = 1;
    l.in = (const u64 *)in + off * N; l.out = (u64 *)out + off * N;
    l.in_limb_stride = l.out_limb_stride = N; l.n_limbs = n; l.n_polys = 1; l.post_scale = nullptr;
    run_ntt(ctx, inverse, lm, l, (cudaStream_t)stream);
  }
  return check_launch(ctx, inverse ? "intt" : "ntt");
}
extern "C" int hml_ntt(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n, void *s) {
  return ntt_api(ctx, false, in, out, mod_idx, n, s);
}
extern "C" int hml_intt(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n, void *s) {
  return ntt_api(ctx, true, in, out, mod_idx, n, s);
}

static int ntt_batch_api(hml_ctx *ctx, bool inverse, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs,
                         uint32_t n_batch, void *stream) {
  if (!ctx || !in || !out || !mod_idx) return HML_ERR_INVALID;
  if (n_limbs == 0 || n_batch == 0) return HML_OK;
  if (n_limbs > NTT_MAX_LIMBS) return fail(ctx, HML_ERR_UNSUPPORTED, "more than 128 limbs per batched transform");
  for (uint32_t i = 0; i < n_limbs; ++i)
    if (mod_idx[i] >= ctx->p.n_mod()) return fail(ctx, HML_ERR_INVALID, "modulus index out of range");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ws_enter(ctx, (cudaStream_t)stream);
  const size_t N = ctx->p.N;
  LimbMap lm;
  id_map(lm, mod_idx, n_limbs);
  // the launch's linear work index must stay below 2^31 tiles: chunk the batch
  const uint32_t per = std::max<uint32_t>(1, 16384 / n_limbs);
  for (uint32_t b0 = 0; b0 < n_batch; b0 += per) {
    NttLaunch l{};
    l.in = (const u64 *)in + (size_t)b0 * n_limbs * N; l.out = (u64 *)out + (size_t)b0 * n_limbs * N;
    l.in_limb_stride = l.out_limb_stride = N; l.n_limbs = n_limbs; l.n_polys = 1; l.post_scale = nullptr;
    l.n_batch = std::min(per, n_batch - b0); l.in_batch_stride = l.out_batch_stride = (long long)n_limbs * N;
    run_ntt(ctx, inverse, lm, l, (cudaStream_t)stream);
  }
  return check_launch(ctx, inverse ? "intt batch" : "ntt batch");
}
extern "C" int hml_ntt_batch(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n, uint32_t nb, void *s) {
  return ntt_batch_api(ctx, false, in, out, mod_idx, n, nb, s);
}
extern "C" int hml_intt_batch(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n, uint32_t nb, void *s) {
  return ntt_batch_api(ctx, true, in, out, mod_idx, n, nb, s);
}

extern "C" int hml_ewe(hml_ctx *ctx, const uint64_t *x1, const uint64_t *x2, const uint64_t *x3, const uint64_t *x4,
                       int subtract, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs, void *stream) {
  if (!ctx || !out || !mod_idx) return HML_ERR_INVALID;
  if ((x2 && !x1) || (x4 && !x3)) return fail(ctx, HML_ERR_INVALID, "a multiplier needs its multiplicand");
  const size_t N = ctx->p.N;
  for (uint32_t i = 0; i < n_limbs; ++i)
    if (mod_idx[i] >= ctx->p.n_mod()) return fail(ctx, HML_ERR_INVALID, "modulus index out of range");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (uint32_t off = 0; off < n_limbs; off += NTT_MAX_LIMBS) {
    const uint32_t n = std::min<uint32_t>(NTT_MAX_LIMBS, n_limbs - off);
    LimbMap lm;
    id_map(lm, mod_idx + off, n);
    auto sh = [&](const uint64_t *p) { return p ? (const u64 *)p + off * N : nullptr; };
    launch_ewe(ctx->mc, lm, (int)N, (int)n, sh(x1), sh(x2), sh(x3), sh(x4), subtract, (u64 *)out + off * N, (cudaStream_t)stream);
    prof_mark(ctx, HML_CLS_EWE, (cudaStream_t)stream);
    ctx->exec.kernel_launches++;
  }
  ctx->exec.ewe_limbs += n_limbs;
  return check_launch(ctx, "ewe");
}

extern "C" int hml_automorph(hml_ctx *ctx, const uint64_t *in, uint64_t *out, uint64_t g, uint32_t n_limbs, void *stream) {
  if (!ctx || !in || !out || in == out) return HML_ERR_INVALID;
  if (!(g & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  for (uint32_t off = 0; off < n_limbs; off += 32768) {
    const uint32_t n = std::min<uint32_t>(32768, n_limbs - off);
    launch_automorph(ctx->p.logN, n, (const u64 *)in + (size_t)off * ctx->p.N, (u64 *)out + (size_t)off * ctx->p.N, g, (cudaStream_t)stream);
    prof_mark(ctx, HML_CLS_AUTO, (cudaStream_t)stream);
    ctx->exec.kernel_launches++;
  }
  ctx->exec.automorph_limbs += n_limbs;
  return check_launch(ctx, "automorph");
}

extern "C" int hml_bconv_batch(hml_ctx *ctx, const uint64_t *in, const uint32_t *src_idx, uint32_t n_src, uint64_t *out,
                               const uint32_t *dst_idx, uint32_t n_dst, uint32_t n_batch, void *stream) {
  if (!ctx || !in || !out || !src_idx || !dst_idx || !n_src || !n_dst || !n_batch) return HML_ERR_INVALID;
  if (n_src > NTT_MAX_LIMBS || n_dst > NTT_MAX_LIMBS) return fail(ctx, HML_ERR_UNSUPPORTED, "more than 128 limbs in one conversion");
  for (uint32_t i = 0; i < n_src; ++i) if (src_idx[i] >= ctx->p.n_mod()) return fail(ctx, HML_ERR_INVALID, "modulus index out of range");
  for (uint32_t i = 0; i < n_dst; ++i) if (dst_idx[i] >= ctx->p.n_mod()) return fail(ctx, HML_ERR_INVALID, "modulus index out of range");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  std::vector<uint32_t> key(src_idx, src_idx + n_src);
  key.push_back(0xFFFFFFFFu);
  key.insert(key.end(), dst_idx, dst_idx + n_dst);
  auto it = ctx->bconv_cache.find(key);
  if (it == ctx->bconv_cache.end()) {
    BConvTable bt;
    make_bconv_table(ctx->p, std::vector<uint32_t>(src_idx, src_idx + n_src), std::vector<uint32_t>(dst_idx, dst_idx + n_dst), bt);
    std::vector<double2> s1(n_src);
    for (uint32_t i = 0; i < n_src; ++i) s1[i] = mk_cst(bt.hat_inv[i], ctx->p.mod[src_idx[i]]);
    DevBConv d;
    int rc;
    if ((rc = upload(ctx, s1, &d.step1))) return rc;
    std::vector<uint32_t> ident(n_dst);
    for (uint32_t t = 0; t < n_dst; ++t) ident[t] = t;
    if ((rc = prepare_bconv(ctx, bt, ident, d.host))) return rc;
    it = ctx->bconv_cache.emplace(key, d).first;
  }
  LimbMap slm;
  id_map(slm, src_idx, n_src);
  BConvArgs a{};
  a.in = (const u64 *)in; a.out = (u64 *)out; a.step1 = it->second.step1;
  a.N = ctx->p.N; a.n_batches = (int)n_batch;
  a.in_batch_stride = (long long)n_src * ctx->p.N; a.out_batch_stride = (long long)n_dst * ctx->p.N;
  run_bconv(ctx, it->second.host, slm, a, (cudaStream_t)stream);
  ctx->exec.ewe_limbs += (uint64_t)n_src * n_batch;  // step 1
  return check_launch(ctx, "bconv");
}

extern "C" int hml_bconv(hml_ctx *ctx, const uint64_t *in, const uint32_t *src_idx, uint32_t n_src, uint64_t *out,
                         const uint32_t *dst_idx, uint32_t n_dst, void *stream) {
  return hml_bconv_batch(ctx, in, src_idx, n_src, out, dst_idx, n_dst, 1, stream);
}

// ------------------------------------------------------------------------------------------------ key switch
static size_t ks_ws_words(const Params &p, uint32_t L) {
  const size_t N = p.N, E = L + p.alpha;
  return N * (L + (size_t)p.beta(L) * E + 2 * E + 2 * (size_t)L);
}


// K1..K4: ModUp (INTT + digit scaling, base conversion, NTT of the converted limbs).  Buffers: yb [nb][L] | ext [nb][beta][E].
// The fusion pays for ONE ciphertext per launch (measured at the north-star shape: ModUp transform + inner product 112 -> 95 us,
// hmult 245 -> 233 us, hrotate 249 -> 227 us): there the stand-alone inner product is latency-bound on the 150 MB key.  In a
// 32-ciphertext chunk the key is read once per chunk and k_inner streams at the HBM rate, while the row pass is bound by the
// FP64 pipe and the fused multiply-accumulates (+45 % FP64 work) land exactly there: 168 -> 178 us per hmult.
static bool ks_uses_hpip(const hml_ctx *ctx, uint32_t L, uint32_t nb) {
  return ctx->p.logN > NTT_SMALL_LOG && ctx->p.beta(L) >= 2 && nb == 1;
}

static int ks_modup(hml_ctx *ctx, LevelConsts *lc, uint32_t L, uint32_t nb, BatchPtr d, u64 *yb, u64 *ext, cudaStream_t s, const NttMac *mac = nullptr,
                    const KsAuto *au = nullptr, const KsTensor *ten = nullptr) {
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t A = p.alpha, E = L + A, beta = lc->beta;
  const bool two_pass = p.logN > NTT_SMALL_LOG;
  // K1 + K2 (reference :63-135): INTT of the input, digit scaling folded into the N^-1 multiply
  {
    NttLaunch l{};
    l.in = d.ptr; l.out = yb; l.in_limb_stride = l.out_limb_stride = N; l.n_limbs = L; l.n_polys = 1; l.post_scale = lc->modup_scale;
    l.n_batch = nb; l.in_batch_stride = d.stride; l.out_batch_stride = (long long)L * N;
    if (au) {  // hrotate: d = sigma_g(raw input), permuted while the row pass loads it; sigma_g(d) is kept for K5's own-digit term
      unsigned gi = 1;
      const unsigned g8 = (unsigned)(au->g & 255);
      for (int i = 0; i < 7; ++i) gi = gi * (2u - g8 * gi);  // Newton: g^-1 mod 256 (g odd)
      l.in_galois = galois_mod(au->g, N); l.in_ginv8 = gi & 255u;
      l.side_out = au->sigma_d; l.side_batch_stride = au->sigma_stride;
    }
    if (ten) {  // d = a1 * b1, formed on load (tallied with the tensor product in ks_inner)
      l.in = ten->a + ten->comp_stride; l.in_mul = ten->b + ten->comp_stride; l.in_batch_stride = ten->batch_stride;
    }
    run_ntt(ctx, true, lc->q_lm, l, s);
  }
  // K3 (reference :137-188): convert every digit to the limbs of the extended basis it does not own
  {
    BConvArgs a{};
    a.in = yb; a.out = ext; a.step1 = nullptr; a.N = N; a.n_batches = nb;
    a.in_batch_stride = (long long)L * N; a.out_batch_stride = (long long)beta * E * N;
    a.out_f64 = two_pass;  // hand-off to the forward NTT as doubles
    // the one-launch form only for small chunks: big ones amortise the per-launch set-up anyway and run 3 % faster digit by digit
    run_modup_bconv(ctx, lc->up, lc->up_src, nb <= 4 ? lc->up_jobs : nullptr, nullptr, a, (long long)A * N, (long long)E * N, s);
  }
  // K4 (reference :190-292): NTT of the converted limbs.  The digit's own limbs are the untouched input
  // (delta D3: the reference also counts an NTT for those).
  {
    NttLaunch l{};
    l.in = ext; l.out = ext; l.in_limb_stride = l.out_limb_stride = N; l.in_poly_stride = l.out_poly_stride = (long long)E * N;
    l.n_limbs = E; l.n_polys = beta;  // digit j skips the limbs it owns (LimbMap::skip)
    l.n_batch = nb; l.in_batch_stride = l.out_batch_stride = (long long)beta * E * N;
    l.in_f64 = l.out_f64 = two_pass;  // doubles in from the conversion, raw lazy doubles out to the inner product
    if (mac) {  // K5 rides in the row pass (HPIP analogue): the transformed digits are multiplied by the key and never stored
      l.mac = *mac;
      ctx->exec.ewe_limbs += 2ull * nb * E * beta;
    }
    run_ntt(ctx, false, lc->ext_lm, l, s);
  }
  return HML_OK;
}

// The evaluation key of a level-L key switch, decoded once from (evk, evk_q_limbs): q_limbs Q-limbs, then the alpha P-limbs,
// so extended limb e (the L Q-limbs, then the P-limbs) is key limb pos(e, L).
struct KeyDesc {
  const u64 *evk;
  uint32_t q_limbs;  // evk_q_limbs without HML_KEY_PACKED
  bool packed;       // HML_KEY_PACKED: the limb slots hold packed limbs (hml_key_pack)
  uint32_t pos(uint32_t e, uint32_t L) const { return e < L ? e : q_limbs + (e - L); }
};
static int key_desc(hml_ctx *ctx, uint32_t L, const u64 *evk, uint32_t evk_q_limbs, KeyDesc *k) {
  const Params &p = ctx->p;
  const uint32_t q = evk_q_limbs & ~HML_KEY_PACKED;
  if (q < L || q > p.max_level) return fail(ctx, HML_ERR_INVALID, "evk_q_limbs must be in [L, maxLevel]");
  if (p.beta(L) > 8) return fail(ctx, HML_ERR_UNSUPPORTED, "more than 8 key-switch digits (ceil(L/alpha) > 8)");
  *k = KeyDesc{evk, q, (evk_q_limbs & HML_KEY_PACKED) != 0};
  return HML_OK;
}

// K5..K7: inner product with the key, INTT (+ step-1 scaling) of the P-limbs of both accumulators.  acc [nb][2][AL], AL >= E.
// galois != 0: the digits are read through the automorphism X -> X^galois (hoisted rotation, see InnerArgs::galois).
static int ks_inner(hml_ctx *ctx, LevelConsts *lc, uint32_t L, uint32_t nb, BatchPtr d, const KeyDesc &key, const u64 *ext, u64 *acc,
                    uint32_t AL, u64 galois, cudaStream_t s, const MergedU *mu = nullptr, bool ip_done = false, const KsTensor *ten = nullptr) {
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t A = p.alpha, E = L + A, beta = lc->beta;
  const int logN = p.logN, npass = logN <= NTT_SMALL_LOG ? 1 : 2;
  // K5 (reference :294-414): inner product with the key (key words loaded once per batch) — unless the ModUp transform's row
  // pass has already done it (ks_front with HPIP)
  if (!ip_done) {
    LimbMap ip = lc->ext_lm;  // pos = limb index inside the key
    for (uint32_t e = 0; e < E; ++e) ip.pos[e] = (uint16_t)key.pos(e, L);
    InnerArgs a{};
    a.d = d.ptr; a.ext = ext; a.evk = key.evk; a.evk_packed = key.packed ? 1 : 0; a.acc = acc; a.N = N; a.n_ext = E; a.beta = beta;
    a.evk_limbs = key.q_limbs + A;
    a.n_batch = nb; a.d_batch_stride = d.stride; a.ext_batch_stride = (long long)beta * E * N; a.acc_batch_stride = 2ll * AL * N;
    a.acc_comp_stride = (long long)AL * N; a.ext_f64 = npass == 2;
    // Q-limb accumulators only feed element-wise epilogues: packed (5 B / coefficient) — but the HPIP path, which some other
    // call of this level may take, leaves words, and the consumers are told per call (ks_tail's acc_packed)
    a.acc_pack_limbs = npass == 2 ? (int)L : 0;
    a.galois = inner_galois(galois, N); a.logN = logN;
    a.u_limb = -1;
    if (mu && nb == 1) {  // hmult: u[L-1] = acc[L-1] * P^-1 + d[L-1] lands in slot E of each accumulator (host copy of the constant)
      a.u_limb = (int)L - 1; a.u_slot = (int)E; a.u_add = mu->add; a.u_add_comp_stride = mu->comp_stride; a.u_add_batch_stride = mu->batch_stride;
      a.u_cst = lc->pinv_last;
      ctx->exec.ewe_limbs += 4ull * nb;
    }
    if (!ten) {
      launch_inner_product(ctx->mc, ip, a, s);
      prof_mark(ctx, HML_CLS_EWE, s);
      ctx->exec.kernel_launches++;
    } else {
      // the Q-limbs form d0, d1, d2 (the tensor product, reference :592-739) and carry d0 * P, d1 * P; the P-limbs need none of
      // it and run in the lean kernel (78 registers, three CTAs per SM, instead of 128 and two), as a launch of their own
      InnerArgs aq = a;
      aq.ct_a = ten->a; aq.ct_b = ten->b; aq.ct_comp_stride = ten->comp_stride; aq.ct_batch_stride = ten->batch_stride;
      aq.tensor_pmod = lc->pmod;
      launch_inner_product(ctx->mc, ip, aq, s, (int)L);
      prof_mark(ctx, HML_CLS_EWE, s);
      ctx->exec.ewe_limbs += 3ull * nb * L; ctx->exec.kernel_launches++;
      LimbMap pl = ip;  // extended limbs L.. renumbered from 0; ext and acc start at limb L
      for (uint32_t j = 0; j < A; ++j) { pl.mod[j] = ip.mod[L + j]; pl.pos[j] = ip.pos[L + j]; pl.skip[j] = ip.skip[L + j]; }
      InnerArgs ap = a;
      ap.ext = ext + (size_t)L * N; ap.acc = acc + (size_t)L * N; ap.acc_pack_limbs = 0;
      launch_inner_product(ctx->mc, pl, ap, s, (int)A);
      prof_mark(ctx, HML_CLS_EWE, s);
      ctx->exec.kernel_launches++;
    }
    ctx->exec.ewe_limbs += 2ull * nb * E * beta;
    if (mu && nb > 1) {
      // batches keep the inner product's kernel lean: u[L-1] = acc[L-1] * P^-1 + d[L-1] -> slot E is two small element-wise
      // launches per chunk (one per component, every ciphertext of the chunk) instead of a side output.  With the tensor
      // product in the inner product (mu->add null) acc[L-1] already holds the d term.
      for (int c = 0; c < 2; ++c) {
        SubMulArgs u{};
        u.x = acc + ((size_t)c * AL + (L - 1)) * N; u.x_poly_stride = 2ll * AL * N;
        u.y = nullptr;
        u.z = mu->add ? mu->add + c * mu->comp_stride + (size_t)(L - 1) * N : nullptr; u.z_poly_stride = mu->batch_stride;
        u.out = acc + ((size_t)c * AL + E) * N; u.out_poly_stride = 2ll * AL * N;
        u.cst = lc->pinv + (L - 1); u.N = N; u.n_limbs = 1; u.n_polys = nb; u.x_packed = u.z_packed = 1;
        launch_sub_mul_add(ctx->mc, lc->last_lm, u, s);
        prof_mark(ctx, HML_CLS_EWE, s);
        ctx->exec.ewe_limbs += 2ull * nb; ctx->exec.kernel_launches++;
      }
    }
  }
  // K6 + K7 (reference :417-487): INTT of the P-limbs of both accumulators, in place, BConv step 1 folded in.  hmult adds
  // one limb to the same launch: slot E (modulus q_{L-1}) = u[L-1], the Rescale INTT (reference :766-805)
  {
    NttLaunch l{};
    l.in = acc; l.out = acc; l.in_limb_stride = l.out_limb_stride = N; l.in_poly_stride = l.out_poly_stride = (long long)AL * N;
    l.n_limbs = A + (mu ? 1 : 0); l.n_polys = 2 * nb; l.post_scale = mu ? lc->moddown_scale_u : lc->moddown_scale;  // acc is [nb][2][AL][N]
    l.n_batch = 1;
    run_ntt(ctx, true, mu ? lc->pu_lm : lc->p_lm, l, s);
  }
  return HML_OK;
}

// K1..K7.  Buffers: yb [nb][L] | ext [nb][beta][E] | acc [nb][2][AL] with AL >= E limbs per accumulator.
// Two-pass rings with at least two digits fuse the inner product into the ModUp transform (NttMac): the Q-limb accumulators are
// then 8-byte words (not packed limbs); ks_uses_hpip() tells the consumers.
static int ks_front(hml_ctx *ctx, LevelConsts *lc, uint32_t L, uint32_t nb, BatchPtr d, const KeyDesc &key, u64 *yb,
                    u64 *ext, u64 *acc, uint32_t AL, cudaStream_t s, const MergedU *mu = nullptr, const KsAuto *au = nullptr,
                    const KsTensor *ten = nullptr) {
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t A = p.alpha, E = L + A;
  const bool hpip = ks_uses_hpip(ctx, L, nb);
  const BatchPtr d_raw = d;
  if (au) d = {au->sigma_d, au->sigma_stride};  // what K5 reads (written by the ModUp INTT)
  NttMac mac{};
  if (hpip) {
    mac.evk = key.evk; mac.evk_packed = key.packed ? 1 : 0; mac.d = d.ptr; mac.acc = acc; mac.d_batch_stride = d.stride; mac.acc_batch_stride = 2ll * AL * N;
    mac.acc_comp_stride = (long long)AL * N; mac.evk_limbs = (int)(key.q_limbs + A);
    for (uint32_t e = 0; e < E; ++e) mac.key_pos[e] = (uint16_t)key.pos(e, L);
    mac.u_limb = -1;
    if (mu) {
      mac.u_limb = (int)L - 1; mac.u_slot = (int)E; mac.u_add = mu->add; mac.u_add_comp_stride = mu->comp_stride;
      mac.u_add_batch_stride = mu->batch_stride; mac.u_cst = lc->pinv_last;
      ctx->exec.ewe_limbs += 4ull * nb;
    }
  }
  int rc = ks_modup(ctx, lc, L, nb, d_raw, yb, ext, s, hpip ? &mac : nullptr, au, ten);
  if (rc) return rc;
  return ks_inner(ctx, lc, L, nb, d, key, ext, acc, AL, 0, s, mu, hpip, ten);
}

// The addends of a ModDown epilogue: component 0 reads z0, component 1 reads z1 (either may be null)
static void set_addends(NttFuse &f, const u64 *z0, const u64 *z1) {
  f.z = z0 ? z0 : z1;
  f.z_c_stride = z0 && z1 ? (long long)(z1 - z0) : 0;
  f.z_mask = (z0 ? 1u : 0u) | (z1 ? 2u : 0u);
}

// K8..K10 (+ the caller's addends): ModDown of nb accumulator pairs acc [nb][2][E] -> out_c[b] = (acc_c - NTT(BConv(acc_c; P -> Q))) * P^-1 (+ add_c[b]).
// out0 / out1 and add0 / add1 share one batch stride.
static int ks_tail(hml_ctx *ctx, LevelConsts *lc, uint32_t L, uint32_t nb, u64 *acc, u64 *vb, BatchOut out0, BatchOut out1, BatchPtr add0, BatchPtr add1,
                   cudaStream_t s, bool acc_packed, u64 add0_galois) {
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t A = p.alpha, E = L + A;
  const bool two_pass = p.logN > NTT_SMALL_LOG;
  // K8 (reference :489-519): P -> Q_L
  {
    BConvArgs a{};
    a.in = acc; a.out = vb; a.in_batch_stride = (long long)E * N; a.out_batch_stride = (long long)L * N;  // p_lm.pos = L + j
    a.step1 = nullptr; a.N = N; a.n_batches = 2 * nb; a.out_f64 = two_pass;
    run_bconv(ctx, lc->down, lc->p_lm, a, s);
  }
  if (add0_galois && (!add0.ptr || add1.ptr)) return fail(ctx, HML_ERR_INVALID, "automorphism on the addend needs the fused ModDown epilogue");
  // K9 (reference :521-546, emitted with opcode INTT — delta D1): forward NTT of the converted limbs, and
  // K10 (reference :548-590) (+ the caller's addend: HMULT add :967-1005 / HROTATE add :1339-1357)
  NttLaunch l{};
  l.in = vb; l.out = vb; l.in_limb_stride = l.out_limb_stride = N; l.in_poly_stride = l.out_poly_stride = (long long)L * N;
  l.n_limbs = L; l.n_polys = 2 * nb; l.n_batch = 1; l.in_f64 = two_pass;
  NttFuse &f = l.fuse;
  f.x = acc; f.x_c_stride = (long long)E * N; f.x_b_stride = 2ll * E * N; f.x_packed = acc_packed ? 1 : 0;
  set_addends(f, add0.ptr, add1.ptr);
  f.z_b_stride = add0.ptr ? add0.stride : add1.stride;
  f.dst = out0.ptr; f.dst_c_stride = (long long)(out1.ptr - out0.ptr); f.dst_b_stride = out0.stride;
  f.cst = lc->pinv; f.n_c = 2;
  f.z_galois = galois_mod(add0_galois, N);
  int rc = ntt_sub_mul(ctx, lc->q_lm, l, s);
  if (rc) return rc;
  ctx->exec.ewe_limbs += (uint64_t)nb * (2 * L + (add0.ptr ? L : 0) + (add1.ptr ? L : 0));
  return check_launch(ctx, "keyswitch");
}

// nb independent key switches sharing one key, one kernel launch per stage:
// d[b] [L][N] -> out_c[b] = KS_c(d[b]) (+ add_c[b]).  `ws` must hold nb * ks_ws_words().
static int ks_run(hml_ctx *ctx, uint32_t L, uint32_t nb, BatchPtr d, const u64 *evk, uint32_t evk_q_limbs, BatchOut out0,
                  BatchOut out1, BatchPtr add0, BatchPtr add1, u64 *ws, cudaStream_t s, const KsAuto *au = nullptr) {
  const Params &p = ctx->p;
  KeyDesc key;
  int rc = key_desc(ctx, L, evk, evk_q_limbs, &key);
  if (rc) return rc;
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const size_t N = p.N;
  const uint32_t A = p.alpha, E = L + A, beta = lc->beta;
  // workspace, every buffer batch-major: yb [nb][L] | ext [nb][beta][E] | acc [nb][2][E] | vb [nb][2][L]  (limbs of N words)
  u64 *yb = ws, *ext = yb + (size_t)nb * L * N, *acc = ext + (size_t)nb * beta * E * N, *vb = acc + (size_t)nb * 2 * E * N;
  if ((rc = ks_front(ctx, lc, L, nb, d, key, yb, ext, acc, E, s, nullptr, au))) return rc;
  return ks_tail(ctx, lc, L, nb, acc, vb, out0, out1, add0, add1, s, p.logN > NTT_SMALL_LOG && !ks_uses_hpip(ctx, L, nb), au ? au->g : 0);
}

extern "C" int hml_key_pack(hml_ctx *ctx, const uint64_t *words_dev, uint64_t n_limbs, uint64_t *packed_dev, void *stream) {
  if (!ctx) return HML_ERR_INVALID;
  if (!words_dev || !packed_dev) return fail(ctx, HML_ERR_INVALID, "null buffer");
  const size_t N = ctx->p.N;
  if (packed_dev < words_dev + n_limbs * N && words_dev < packed_dev + n_limbs * N) return fail(ctx, HML_ERR_INVALID, "hml_key_pack: buffers overlap");
  if (n_limbs == 0) return HML_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  launch_pack_limbs((int)N, (size_t)n_limbs, (const u64 *)words_dev, (u64 *)packed_dev, (cudaStream_t)stream);
  return check_launch(ctx, "key pack");
}

extern "C" int hml_keyswitch(hml_ctx *ctx, uint32_t L, const uint64_t *d, const uint64_t *evk, uint32_t evk_q_limbs,
                             uint64_t *out0, uint64_t *out1, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (!d || !evk || !out0 || !out1) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, ks_ws_words(ctx->p, L)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return ks_run(ctx, L, 1, {(const u64 *)d, 0}, (const u64 *)evk, evk_q_limbs, {(u64 *)out0, 0}, {(u64 *)out1, 0}, {nullptr, 0},
                {nullptr, 0}, ctx->ws, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------ limb-sharded key switch
// SURVEY.md 8e mode 2: one ciphertext, the E = L + alpha extended limbs partitioned over `world` GPUs.  Extended limb e
// is owned by rank e % world — the reference's own rule for mapping limbs to clusters (reference include/Driver.h:158,
// :178).  Every primitive except base conversion is limb-local; BConv needs all input limbs of a digit, so there is
// exactly one all-gather before each conversion (the reference's analogue is its inter-cluster NoC fetch,
// reference include/mem.h:612-621, src/mem.cpp:78-100):
//   begin:  INTT (+ digit scaling) of the owned Q-limbs, written straight into this rank's slot of gather buffer 1
//   [all-gather 1: world x ceil(L/world) limbs]
//   mid:    BConv digit -> owned extended limbs, NTT, inner product with the owned key slices, INTT (+ scaling) of
//           the owned P-limbs of both accumulators, copied into this rank's slot of gather buffer 2
//   [all-gather 2: world x 2 x ceil(alpha/world) limbs]
//   end:    BConv P -> owned Q-limbs, NTT, (acc - v) * P^-1 for the owned Q-limbs
// The collective itself is issued by the caller (NCCL all-gather on the same stream; homulator_b200/api.py uses
// torch.distributed) so the library stays free of a communicator dependency.
static int get_shard_plan(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, ShardPlan **out) {
  const uint64_t key = ((uint64_t)L << 32) | ((uint64_t)world << 16) | rank;
  auto it = ctx->shard_plans.find(key);
  if (it != ctx->shard_plans.end()) { *out = &it->second; return HML_OK; }
  const Params &p = ctx->p;
  const uint32_t A = p.alpha, E = L + A, beta = p.beta(L);
  ShardPlan sp;
  sp.L = L; sp.world = world; sp.rank = rank; sp.beta = beta;
  sp.gq = (L + world - 1) / world; sp.gp = (A + world - 1) / world;
  for (uint32_t e = 0; e < E; ++e)
    if (e % world == rank) { (e < L ? sp.own_q : sp.own_p).push_back(e < L ? e : e - L); }
  const uint32_t nq = sp.own_q.size(), np = sp.own_p.size(), ne = nq + np;
  auto gpos1 = [&](uint32_t i) { return (i % world) * sp.gq + i / world; };                    // Q-limb i in gather buffer 1
  auto gpos2 = [&](uint32_t j) { return ((L + j) % world) * 2 * sp.gp + ((L + j) / world - sp.first_p_slot((L + j) % world, L, world)); };
  clear_map(sp.q_lm); clear_map(sp.p_lm); clear_map(sp.e_lm);
  std::vector<double2> s1(nq), s2(np), pinv(nq);
  for (uint32_t k = 0; k < nq; ++k) {
    const uint32_t i = sp.own_q[k];
    sp.q_lm.mod[k] = i; sp.q_lm.pos[k] = k;
    sp.e_lm.mod[k] = i; sp.e_lm.pos[k] = k; sp.e_lm.skip[k] = (uint8_t)(i / A);
    s1[k] = mk_cst(p.modup_scale(L, i), p.mod[i]);
    pinv[k] = mk_cst(p.p_inv(i), p.mod[i]);
  }
  for (uint32_t k = 0; k < np; ++k) {
    const uint32_t j = sp.own_p[k], mi = p.max_level + j;
    sp.p_lm.mod[k] = mi; sp.p_lm.pos[k] = nq + k;
    sp.e_lm.mod[nq + k] = mi; sp.e_lm.pos[nq + k] = nq + k;
    s2[k] = mk_cst(p.moddown_scale(j), p.mod[mi]);
  }
  int rc;
  if ((rc = upload(ctx, s1, &sp.scale1))) return rc;
  if ((rc = upload(ctx, s2, &sp.scale2))) return rc;
  if ((rc = upload(ctx, pinv, &sp.pinv))) return rc;
  if (L >= 2) {
    std::vector<double2> ql;
    for (uint32_t k = 0; k < nq; ++k) {
      const uint32_t i = sp.own_q[k];
      if (i + 1 < L) ql.push_back(mk_cst(p.ql_inv(L, i), p.mod[i]));
    }
    if ((rc = upload(ctx, ql, &sp.qlinv_own))) return rc;
  }
  // ModUp conversions: digit j (all its limbs, read from gather buffer 1) -> owned extended limbs outside the digit
  for (uint32_t j = 0; j < beta; ++j) {
    const uint32_t lo = j * A, aj = p.digit_size(L, j);
    std::vector<uint32_t> src, dst, dst_pos;
    LimbMap slm; clear_map(slm);
    for (uint32_t i = 0; i < aj; ++i) { src.push_back(lo + i); slm.mod[i] = lo + i; slm.pos[i] = gpos1(lo + i); }
    for (uint32_t le = 0; le < ne; ++le) {
      const uint32_t e = le < nq ? sp.own_q[le] : L + sp.own_p[le - nq];
      if (e >= lo && e < lo + aj) continue;
      dst.push_back(p.ext_mod(L, e)); dst_pos.push_back(le);
    }
    sp.up.emplace_back();
    sp.up_src.push_back(slm);
    if (!dst.empty()) {
      BConvTable bt;
      make_bconv_table(p, src, dst, bt);
      if ((rc = prepare_bconv(ctx, bt, dst_pos, sp.up.back()))) return rc;
    }
  }
  {  // ModDown conversion: all P-limbs (read from gather buffer 2) -> owned Q-limbs
    std::vector<uint32_t> src, dst, dst_pos;
    clear_map(sp.down_src);
    for (uint32_t j = 0; j < A; ++j) { src.push_back(p.max_level + j); sp.down_src.mod[j] = p.max_level + j; sp.down_src.pos[j] = gpos2(j); }
    for (uint32_t k = 0; k < nq; ++k) { dst.push_back(sp.own_q[k]); dst_pos.push_back(k); }
    if (!dst.empty()) {
      BConvTable bt;
      make_bconv_table(p, src, dst, bt);
      if ((rc = prepare_bconv(ctx, bt, dst_pos, sp.down))) return rc;
    }
  }
  auto ins = ctx->shard_plans.emplace(key, sp);
  *out = &ins.first->second;
  return HML_OK;
}

static size_t shard_ws_words(const Params &p, const ShardPlan &sp) {
  const size_t ne = sp.own_q.size() + sp.own_p.size(), nq = sp.own_q.size();
  return (size_t)p.N * ((size_t)sp.beta * ne + 2 * ne + 2 * nq);
}

int shard_check(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (world == 0 || rank >= world || world > 64) return fail(ctx, HML_ERR_INVALID, "bad rank / world");
  return HML_OK;
}

extern "C" int hml_shard_layout(uint32_t L, uint32_t alpha, uint32_t rank, uint32_t world, hml_shard_info *out) {
  if (!out || world == 0 || rank >= world || L == 0 || alpha == 0 || L + alpha > HML_MAX_SHARD_LIMBS) return HML_ERR_INVALID;
  const uint32_t A = alpha, E = L + A;
  memset(out, 0, sizeof(*out));
  out->gather1_slots = (L + world - 1) / world;
  out->gather2_slots = (A + world - 1) / world;
  for (uint32_t e = 0; e < E; ++e) {
    out->owner[e] = e % world;
    if (e % world == rank) {
      if (e < L) out->own_q[out->n_own_q++] = e; else out->own_p[out->n_own_p++] = e - L;
    }
    // slot of limb e inside its owner's contribution to the gather buffer
    out->slot[e] = e < L ? e / world : (e / world - ShardPlan::first_p_slot(e % world, L, world));
  }
  return HML_OK;
}

extern "C" int hml_keyswitch_shard_begin(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *d_own,
                                         uint64_t *gather1, void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (!d_own || !gather1) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ShardPlan *sp;
  if ((rc = get_shard_plan(ctx, L, rank, world, &sp))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  const size_t N = ctx->p.N;
  const uint32_t nq = sp->own_q.size();
  if (nq) {
    NttLaunch l{};
    l.n_batch = 1;
    l.in = (const u64 *)d_own; l.out = (u64 *)gather1 + (size_t)rank * sp->gq * N;
    l.in_limb_stride = l.out_limb_stride = N; l.n_limbs = nq; l.n_polys = 1; l.post_scale = sp->scale1;
    run_ntt(ctx, true, sp->q_lm, l, (cudaStream_t)stream);
  }
  return check_launch(ctx, "keyswitch shard begin");
}

// forward NTT of the owned extended digits ext [beta][ne] in place; with hpip the inner product with evk_own rides in the row
// pass (NttMac) and the transformed digits are never stored
static void shard_ext_ntt(hml_ctx *ctx, ShardPlan *sp, u64 *ext, bool hpip, const u64 *d_own, const u64 *evk_own, u64 *acc, cudaStream_t s) {
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t ne = sp->own_q.size() + sp->own_p.size(), beta = sp->beta;
  NttLaunch l{};
  l.n_batch = 1;
  l.in = ext; l.out = ext; l.in_limb_stride = l.out_limb_stride = N; l.in_poly_stride = l.out_poly_stride = (long long)ne * N;
  l.n_limbs = ne; l.n_polys = beta;
  l.in_f64 = l.out_f64 = p.logN > NTT_SMALL_LOG;
  if (hpip) {
    NttMac &m = l.mac;
    m.evk = evk_own; m.d = d_own; m.acc = acc; m.d_batch_stride = 0; m.acc_batch_stride = 0; m.acc_comp_stride = (long long)ne * N;
    m.evk_limbs = (int)ne; m.u_limb = -1;
    for (uint32_t k = 0; k < ne; ++k) m.key_pos[k] = (uint16_t)k;
    ctx->exec.ewe_limbs += 2ull * ne * beta;
  }
  run_ntt(ctx, false, sp->e_lm, l, s);
}

// everything of the middle phase after the ModUp conversions: NTT of the extended digits, inner product with the owned key
// slices, INTT (+ scaling) of the owned P-limbs, copied into this rank's slot of gather buffer 2
static int shard_mid_tail(hml_ctx *ctx, ShardPlan *sp, uint32_t rank, const u64 *d_own, const u64 *evk_own, u64 *gather2, cudaStream_t s) {
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t nq = sp->own_q.size(), np = sp->own_p.size(), ne = nq + np, beta = sp->beta;
  u64 *ext = ctx->ws, *acc = ext + (size_t)beta * ne * N;
  // one ciphertext's slice per rank: the inner product rides in the ModUp transform's row pass (NttMac) whenever it can
  const bool hpip = ks_uses_hpip(ctx, sp->L, 1);
  shard_ext_ntt(ctx, sp, ext, hpip, d_own, evk_own, acc, s);
  if (!hpip) {
    InnerArgs a{};
    a.d = d_own; a.ext = ext; a.evk = evk_own; a.acc = acc; a.N = N; a.n_ext = ne; a.beta = beta;
    a.evk_limbs = ne; a.n_batch = 1; a.u_limb = -1; a.ext_f64 = p.logN > NTT_SMALL_LOG;
    launch_inner_product(ctx->mc, sp->e_lm, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.ewe_limbs += 2ull * ne * beta; ctx->exec.kernel_launches++;
  }
  if (np) {
    NttLaunch l{};
    l.n_batch = 1;
    // straight into this rank's contribution to gather buffer 2, [2][gp][N] at slot `rank`: limb k of p_lm sits at position
    // nq + k of an accumulator, so the output base is shifted back by nq limbs (never dereferenced below the slot)
    l.in = acc; l.in_limb_stride = N; l.in_poly_stride = (long long)ne * N;
    l.out = gather2 + (size_t)rank * 2 * sp->gp * N - (size_t)nq * N; l.out_limb_stride = N; l.out_poly_stride = (long long)sp->gp * N;
    l.n_limbs = np; l.n_polys = 2; l.post_scale = sp->scale2;
    run_ntt(ctx, true, sp->p_lm, l, s);
  }
  return check_launch(ctx, "keyswitch shard mid");
}

extern "C" int hml_keyswitch_shard_mid(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *d_own,
                                       const uint64_t *gather1, const uint64_t *evk_own, uint64_t *gather2, void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (!d_own || !gather1 || !evk_own || !gather2) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ShardPlan *sp;
  if ((rc = get_shard_plan(ctx, L, rank, world, &sp))) return rc;
  if ((rc = ensure_ws(ctx, shard_ws_words(ctx->p, *sp)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  const uint32_t ne = sp->own_q.size() + sp->own_p.size();
  cudaStream_t s = (cudaStream_t)stream;
  if (ne == 0) return HML_OK;
  BConvArgs a{};
  a.in = (const u64 *)gather1; a.out = ctx->ws; a.step1 = nullptr; a.N = ctx->p.N; a.n_batches = 1; a.out_f64 = ctx->p.logN > NTT_SMALL_LOG;
  run_modup_bconv(ctx, sp->up, sp->up_src, nullptr, nullptr, a, 0, (long long)ne * ctx->p.N, s);
  return shard_mid_tail(ctx, sp, rank, (const u64 *)d_own, (const u64 *)evk_own, (u64 *)gather2, s);
}

// last phase: BConv P -> owned Q-limbs (sources in `gather2`, or at src_off relative to it), NTT, (acc - v) * P^-1 (+ the
// caller's addends: HROTATE add, component 0 only; HMULT add, both; owned limbs [nq][N]).  The accumulator pair is r of the
// workspace [beta][ne] | acc [H][2][ne] | vb [2][nq] (r = 0, H = 1: the key switch's layout).  add0_galois != 0 reads add0
// through that automorphism (fused epilogue, two-pass rings only).
static int shard_end_run(hml_ctx *ctx, ShardPlan *sp, const u64 *gather2, const long long *src_off, u64 *out0_own, u64 *out1_own, cudaStream_t s,
                         const u64 *add0_own = nullptr, const u64 *add1_own = nullptr, uint32_t r = 0, uint32_t H = 1, u64 add0_galois = 0) {
  int rc;
  if ((rc = ensure_ws(ctx, shard_ws_words(ctx->p, *sp)))) return rc;
  ws_enter(ctx, s);
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t nq = sp->own_q.size(), np = sp->own_p.size(), ne = nq + np;
  const bool two_pass = p.logN > NTT_SMALL_LOG;
  if (nq == 0) return HML_OK;
  const u64 *acc0 = ctx->ws + (size_t)sp->beta * ne * N;
  u64 *vb = (u64 *)acc0 + 2 * (size_t)H * ne * N;
  if (add0_galois && (!add0_own || add1_own)) return fail(ctx, HML_ERR_INVALID, "automorphism on the addend needs the fused ModDown epilogue");
  {
    BConvArgs a{};
    a.in = gather2; a.out = vb; a.in_batch_stride = (long long)sp->gp * N; a.out_batch_stride = (long long)nq * N;
    a.step1 = nullptr; a.N = N; a.n_batches = 2; a.src_off = src_off; a.out_f64 = two_pass;
    run_bconv(ctx, sp->down, sp->down_src, a, s);
  }
  NttLaunch l{};
  l.n_batch = 1;
  l.in = vb; l.out = vb; l.in_limb_stride = l.out_limb_stride = N; l.in_poly_stride = l.out_poly_stride = (long long)nq * N;
  l.n_limbs = nq; l.n_polys = 2; l.in_f64 = two_pass;
  NttFuse &f = l.fuse;
  f.x = acc0 + 2 * (size_t)r * ne * N; f.x_c_stride = (long long)ne * N;
  set_addends(f, add0_own, add1_own);
  f.dst = out0_own; f.dst_c_stride = (long long)(out1_own - out0_own);
  f.cst = sp->pinv; f.n_c = 2;
  f.z_galois = galois_mod(add0_galois, N);
  if ((rc = ntt_sub_mul(ctx, sp->q_lm, l, s))) return rc;
  ctx->exec.ewe_limbs += 2 * nq;
  return check_launch(ctx, "keyswitch shard end");
}

extern "C" int hml_keyswitch_shard_end(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *gather2,
                                       uint64_t *out0_own, uint64_t *out1_own, void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (!gather2 || !out0_own || !out1_own) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ShardPlan *sp;
  if ((rc = get_shard_plan(ctx, L, rank, world, &sp))) return rc;
  return shard_end_run(ctx, sp, (const u64 *)gather2, nullptr, (u64 *)out0_own, (u64 *)out1_own, (cudaStream_t)stream);
}

// ---- peer-direct variant: no collective.  Every rank keeps its contribution in its OWN gather buffer; the base
// conversions of the other ranks read the source limbs straight out of the owners' memory over NVLink (per-source offsets,
// BConvArgs::src_off) while they compute: the all-gather is fused into the consumer's tile loop (cp.async ring of the tcgen05
// kernel, two tiles ahead) instead of being a separate NCCL step.  Ordering between GPUs: monotonically increasing epoch
// counters in a per-rank flag block ([0, world): "gather buffer 1 of rank r is ready", [world, 2 world): buffer 2), written
// into every peer by hml_shard_signal after the producing kernels, polled by hml_shard_wait before the consuming conversion.
// Write-after-read safety needs no extra flags: a rank passes wait(ready2, t) only after every peer has finished its ModUp
// reads of epoch t, and wait(ready1, t + 1) only after every peer has finished the ModDown reads of epoch t.
__global__ void k_shard_signal(unsigned long long *const *peer_flags, int slot, unsigned long long epoch, int world) {
  const int p = threadIdx.x;
  if (p >= world) return;
  __threadfence_system();
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(peer_flags[p] + slot), "l"(epoch) : "memory");
}
// Spin-waits poll with a wall-clock limit (globaltimer, default 20 s, HML_SHARD_TIMEOUT_MS): a peer that is merely slow
// (first-call planning, allocation, a debugger) must not be mistaken for a dead one, and a dead one must not kill the CUDA
// context: on time-out the kernel sets the status word (word 3 * world + 4 of the rank's flag block) and returns; the host
// turns it into HML_ERR_CUDA (hml_shard_status / the hml_shard ops).
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void spin_until(const unsigned long long *flag, unsigned long long epoch, unsigned long long *status,
                                           unsigned long long timeout_ns) {
  const unsigned long long t0 = globaltimer_ns();
  unsigned long long v;
  for (;;) {
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
    if (v >= epoch) return;
    if (globaltimer_ns() - t0 > timeout_ns) {
      atomicExch(status, 1ull);
      return;
    }
  }
}
static unsigned long long shard_timeout_ns() {
  static const unsigned long long v = [] {
    const char *e = getenv("HML_SHARD_TIMEOUT_MS");
    const long long ms = e ? atoll(e) : 20000;
    return (unsigned long long)(ms > 0 ? ms : 20000) * 1000000ull;
  }();
  return v;
}
__global__ void k_shard_wait(const unsigned long long *flags, int base, unsigned long long epoch, int world, unsigned long long timeout_ns) {
  const int r = threadIdx.x;
  if (r >= world) return;
  spin_until(flags + base + r, epoch, const_cast<unsigned long long *>(flags) + 3 * world + 4, timeout_ns);
}

// signal + wait in one launch (one rank per GPU; ranks emulated on ONE stream must use the two separate calls, because a
// rank's wait would otherwise sit in front of the signals it is waiting for)
// epoch == 0: the epoch is this rank's own counter for the exchange group (word 3 * world + base / world of its flag block),
// read and advanced here — no host-side state, so a captured CUDA graph of a whole op sequence can be replayed.
__global__ void k_shard_sync(unsigned long long *const *peer_flags, int slot, unsigned long long *flags, int base,
                             unsigned long long epoch, int world, unsigned long long timeout_ns) {
  __shared__ unsigned long long e_sh;
  const int r = threadIdx.x;
  unsigned long long *ctr = flags + 3 * world + base / world;
  if (r == 0) e_sh = epoch ? epoch : *ctr + 1;
  __syncthreads();
  const unsigned long long e = e_sh;
  if (r < world) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(peer_flags[r] + slot), "l"(e) : "memory");
    spin_until(flags + base + r, e, flags + 3 * world + 4, timeout_ns);
  }
  __syncthreads();
  if (r == 0 && !epoch) *ctr = e;
}
extern "C" int hml_shard_sync(hml_ctx *ctx, uint64_t *const *peer_flags_dev, uint32_t slot, uint64_t *flags, uint32_t base,
                              uint64_t epoch, uint32_t world, void *stream) {
  if (!ctx || !peer_flags_dev || !flags || world == 0 || world > 64) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  k_shard_sync<<<1, 64, 0, (cudaStream_t)stream>>>((unsigned long long *const *)peer_flags_dev, (int)slot, (unsigned long long *)flags,
                                                   (int)base, epoch, (int)world, shard_timeout_ns());
  ctx->exec.kernel_launches++;
  return check_launch(ctx, "shard sync");
}

extern "C" int hml_shard_signal(hml_ctx *ctx, uint64_t *const *peer_flags_dev, uint32_t slot, uint64_t epoch, uint32_t world, void *stream) {
  if (!ctx || !peer_flags_dev || world == 0 || world > 64) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  // a plain launch (no programmatic dependent launch): it starts after the producing kernels have completed and flushed
  k_shard_signal<<<1, 64, 0, (cudaStream_t)stream>>>((unsigned long long *const *)peer_flags_dev, (int)slot, epoch, (int)world);
  ctx->exec.kernel_launches++;
  return check_launch(ctx, "shard signal");
}
extern "C" int hml_shard_wait(hml_ctx *ctx, const uint64_t *flags, uint32_t base, uint64_t epoch, uint32_t world, void *stream) {
  if (!ctx || !flags || world == 0 || world > 64) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  k_shard_wait<<<1, 64, 0, (cudaStream_t)stream>>>((const unsigned long long *)flags, (int)base, epoch, (int)world, shard_timeout_ns());
  ctx->exec.kernel_launches++;
  return check_launch(ctx, "shard wait");
}

extern "C" int hml_shard_status(hml_ctx *ctx, const uint64_t *flags, uint32_t world, void *stream) {
  if (!ctx || !flags || world == 0 || world > 64) return HML_ERR_INVALID;
  HML_CU_TRY(ctx, cudaSetDevice(ctx->device));
  unsigned long long st = 0;
  HML_CU_TRY(ctx, cudaMemcpyAsync(&st, flags + 3 * world + 4, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  HML_CU_TRY(ctx, cudaStreamSynchronize((cudaStream_t)stream));
  if (st) return fail(ctx, HML_ERR_CUDA, "limb-sharded exchange timed out waiting for a peer (HML_SHARD_TIMEOUT_MS); results of this rank are invalid");
  return HML_OK;
}

extern "C" int hml_ipc_export(hml_ctx *ctx, const uint64_t *dev_ptr, unsigned char handle[64]) {
  if (!ctx || !dev_ptr || !handle) return HML_ERR_INVALID;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CU_TRY(ctx, cudaIpcGetMemHandle(&h, (void *)dev_ptr));
  memcpy(handle, &h, 64);
  return HML_OK;
}
extern "C" int hml_ipc_import(hml_ctx *ctx, const unsigned char handle[64], uint64_t **out) {
  if (!ctx || !handle || !out) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CU_TRY(ctx, cudaIpcOpenMemHandle((void **)out, h, cudaIpcMemLazyEnablePeerAccess));
  return HML_OK;
}
extern "C" int hml_ipc_close(hml_ctx *ctx, uint64_t *ptr) {
  if (!ctx || !ptr) return HML_ERR_INVALID;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  CU_TRY(ctx, cudaIpcCloseMemHandle(ptr));
  return HML_OK;
}

// (re)build the per-source offset tables for the given peer buffers
static int shard_peer_offsets(hml_ctx *ctx, ShardPlan *sp, const uint64_t *const *peers, bool second) {
  const Params &p = ctx->p;
  const uint32_t world = sp->world, rank = sp->rank, A = p.alpha, L = sp->L;
  std::vector<const void *> sig(peers, peers + world);
  std::vector<const void *> &cur = second ? sp->peers2_sig : sp->peers1_sig;
  if (cur == sig) return HML_OK;
  const long long N = p.N;
  auto rel = [&](uint32_t owner) { return (long long)(peers[owner] - peers[rank]); };  // words
  int rc;
  if (!second) {
    for (auto *o : sp->d_off1) cudaFree(o);
    sp->d_off1.clear();
    for (uint32_t j = 0; j < sp->beta; ++j) {
      const uint32_t lo = j * A, aj = p.digit_size(L, j);
      std::vector<long long> off(aj);
      for (uint32_t i = 0; i < aj; ++i) off[i] = rel((lo + i) % world) + (long long)sp->up_src[j].pos[i] * N;
      long long *d = nullptr;
      if ((rc = upload(ctx, off, &d))) return rc;
      sp->d_off1.push_back(d);
    }
    // the one-launch form of the ModUp conversions: every CTA serves one digit and reads its sources from the owners' buffers
    cudaFree(sp->up_jobs);
    if ((rc = upload_up_jobs(ctx, sp->up, 0, (long long)(sp->own_q.size() + sp->own_p.size()) * N, &sp->d_off1, &sp->up_jobs))) return rc;
  } else {
    cudaFree(sp->d_off2); sp->d_off2 = nullptr;
    std::vector<long long> off(A);
    for (uint32_t j = 0; j < A; ++j) off[j] = rel((L + j) % world) + (long long)sp->down_src.pos[j] * N;
    if ((rc = upload(ctx, off, &sp->d_off2))) return rc;
  }
  cur = sig;
  return HML_OK;
}

static int shard_p2p_check(hml_ctx *ctx, const HostBConv &hb) {
  if (hb.empty()) return HML_OK;
  if (!hb.im.img || ctx->p.N < 128 || !bconv_umma_enabled())
    return fail(ctx, HML_ERR_UNSUPPORTED, "peer-direct key switch needs the tcgen05 base conversion (N >= 128, <= 48 x 48 limbs)");
  return HML_OK;
}

// the ModUp conversions of the peer-direct middle phase: every digit (its limbs read from the owners' gather buffers 1, at the
// offsets built by shard_peer_offsets relative to this rank's own buffer g1_own) -> owned extended limbs, ext [beta][ne]
static void shard_modup_p2p(hml_ctx *ctx, ShardPlan *sp, const uint64_t *g1_own, u64 *ext, cudaStream_t s) {
  BConvArgs a{};
  a.in = (const u64 *)g1_own; a.out = ext; a.step1 = nullptr; a.N = ctx->p.N; a.n_batches = 1; a.out_f64 = ctx->p.logN > NTT_SMALL_LOG;
  run_modup_bconv(ctx, sp->up, sp->up_src, sp->up_jobs, &sp->d_off1, a, 0, (long long)(sp->own_q.size() + sp->own_p.size()) * ctx->p.N, s);
}

// the preamble of the internal sharded functions: rank / level checks, the context's device, the plan
static int shard_plan_on_device(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, ShardPlan **sp) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  HML_CU_TRY(ctx, cudaSetDevice(ctx->device));
  return get_shard_plan(ctx, L, rank, world, sp);
}

extern "C" int hml_keyswitch_shard_mid_p2p(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *d_own,
                                           const uint64_t *const *peers1, const uint64_t *evk_own, uint64_t *gather2_own, void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (!d_own || !peers1 || !evk_own || !gather2_own) return fail(ctx, HML_ERR_INVALID, "null buffer");
  for (uint32_t r = 0; r < world; ++r) if (!peers1[r]) return fail(ctx, HML_ERR_INVALID, "null peer buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ShardPlan *sp;
  if ((rc = get_shard_plan(ctx, L, rank, world, &sp))) return rc;
  for (auto &u : sp->up) if ((rc = shard_p2p_check(ctx, u))) return rc;
  if ((rc = shard_peer_offsets(ctx, sp, peers1, false))) return rc;
  if ((rc = ensure_ws(ctx, shard_ws_words(ctx->p, *sp)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  const uint32_t ne = sp->own_q.size() + sp->own_p.size();
  if (ne == 0) return HML_OK;
  shard_modup_p2p(ctx, sp, peers1[rank], ctx->ws, (cudaStream_t)stream);
  return shard_mid_tail(ctx, sp, rank, (const u64 *)d_own, (const u64 *)evk_own, (u64 *)gather2_own, (cudaStream_t)stream);
}

// the peer-direct ModDown of accumulator pair r (shard_end_run): its sources read from slot r (slot_words apart) of the owners'
// gather buffers 2
int shard_end_p2p(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers2, uint64_t *out0_own, uint64_t *out1_own,
                  const uint64_t *add0_own, const uint64_t *add1_own, cudaStream_t s, uint32_t r, uint32_t H, size_t slot_words, uint64_t add0_galois) {
  ShardPlan *sp;
  int rc = shard_plan_on_device(ctx, L, rank, world, &sp);
  if (rc) return rc;
  if ((rc = shard_p2p_check(ctx, sp->down))) return rc;
  if ((rc = shard_peer_offsets(ctx, sp, peers2, true))) return rc;
  return shard_end_run(ctx, sp, (const u64 *)peers2[rank] + (size_t)r * slot_words, sp->d_off2, (u64 *)out0_own, (u64 *)out1_own, s,
                       (const u64 *)add0_own, (const u64 *)add1_own, r, H, add0_galois);
}

extern "C" int hml_keyswitch_shard_end_p2p(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers2,
                                           uint64_t *out0_own, uint64_t *out1_own, void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (!peers2 || !out0_own || !out1_own) return fail(ctx, HML_ERR_INVALID, "null buffer");
  for (uint32_t r = 0; r < world; ++r) if (!peers2[r]) return fail(ctx, HML_ERR_INVALID, "null peer buffer");
  return shard_end_p2p(ctx, L, rank, world, peers2, out0_own, out1_own, nullptr, nullptr, (cudaStream_t)stream);
}

// ---- hoisted rotations of one limb-sharded ciphertext (shard.cu, hml_hrotate_hoisted_sharded).  One ModUp of c1 serves every
// rotation; a group of up to H rotations shares one inner-product launch, one P-limb INTT and one exchange.  Workspace:
//   ext [beta][ne] | acc [H][2][ne] | vb [2][nq]        (H = 1: the key switch's layout)
static size_t shard_hoist_ws_words(const Params &p, const ShardPlan &sp, uint32_t H) {
  const size_t ne = sp.own_q.size() + sp.own_p.size(), nq = sp.own_q.size();
  return (size_t)p.N * ((size_t)sp.beta * ne + 2 * (size_t)H * ne + 2 * nq);
}

// the ModUp of the hoisted ops: the conversions from the owners' gather buffers 1 and the forward NTT of the owned extended
// digits into ext [beta][ne], stored for the inner products (no fused inner product)
static int shard_hoist_modup(hml_ctx *ctx, ShardPlan *sp, const uint64_t *const *peers1, u64 *ext, cudaStream_t s) {
  int rc;
  for (auto &u : sp->up) if ((rc = shard_p2p_check(ctx, u))) return rc;
  if ((rc = shard_peer_offsets(ctx, sp, peers1, false))) return rc;
  shard_modup_p2p(ctx, sp, peers1[sp->rank], ext, s);
  shard_ext_ntt(ctx, sp, ext, false, nullptr, nullptr, nullptr, s);
  return HML_OK;
}

// phase 1 of a group of n <= H rotations.  peers1 != null (the op's first group): the ModUp conversions from the owners' gather
// buffers 1 and the forward NTT of the owned extended digits, stored for the later groups (no fused inner product).  Then ONE
// launch of the inner product for all n rotations: acc[r] = sum_j sigma_r(t_j) * keys[r][j]; the own-digit term reads c1_own
// through sigma_r as well.
int shard_hoist_inner(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t H, const uint64_t *const *peers1, const uint64_t *c1_own,
                      uint32_t n, const uint64_t *const *keys, const uint64_t *galois, cudaStream_t s) {
  ShardPlan *sp;
  int rc = shard_plan_on_device(ctx, L, rank, world, &sp);
  if (rc) return rc;
  if (n == 0 || n > H || H > IP_MAX_ROT) return fail(ctx, HML_ERR_INVALID, "hoisted group larger than the shard's rotation capacity");
  if ((rc = ensure_ws(ctx, shard_hoist_ws_words(ctx->p, *sp, H)))) return rc;
  ws_enter(ctx, s);
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t ne = sp->own_q.size() + sp->own_p.size(), beta = sp->beta;
  if (ne == 0) return HML_OK;
  u64 *ext = ctx->ws, *acc = ext + (size_t)beta * ne * N;
  if (peers1 && (rc = shard_hoist_modup(ctx, sp, peers1, ext, s))) return rc;
  InnerRotArgs a{};
  a.d = (const u64 *)c1_own; a.ext = ext; a.acc = acc; a.acc_rot_stride = 2ll * ne * N;
  a.N = (int)N; a.n_ext = (int)ne; a.beta = (int)beta; a.evk_limbs = (int)ne; a.logN = p.logN; a.ext_f64 = p.logN > NTT_SMALL_LOG;
  for (uint32_t r = 0; r < n; ++r) { a.evk[r] = (const u64 *)keys[r]; a.galois[r] = inner_galois(galois[r], N); }
  launch_inner_product_rot(ctx->mc, sp->e_lm, a, (int)n, s);
  prof_mark(ctx, HML_CLS_EWE, s);
  ctx->exec.ewe_limbs += 2ull * n * ne * beta; ctx->exec.kernel_launches++;
  return check_launch(ctx, "hoisted shard inner product");
}

// phase 1 of the sharded double-hoisted rotation sum (shard.cu, hml_hrotate_sum_hoisted_sharded) before its P-limb INTT: the
// ModUp of c1, then k_inner_rot_sum on the owned extended limbs, one launch per group of IP_MAX_ROT rotations (later groups
// add to the stored sums).  The kernel's limb index is the position in the owned layout (Q-limbs first), so L = nq and
// pt_q_limbs = nq make it read Q-limb rows and P-limb rows of the owned plaintext slices [nq + np][N] alike.  acc [2][ne]
// lands where shard_hoist_intt reads accumulator pair 0; z [nq][N] = sum_r pt_r * sigma_r(c0) on the owned Q-limbs.
int shard_rot_sum_inner(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers1, const uint64_t *ct_own,
                        uint32_t n_rot, const uint64_t *const *keys, const uint64_t *galois, const uint64_t *const *pts, uint64_t *z_own,
                        cudaStream_t s) {
  ShardPlan *sp;
  int rc = shard_plan_on_device(ctx, L, rank, world, &sp);
  if (rc) return rc;
  if ((rc = ensure_ws(ctx, shard_hoist_ws_words(ctx->p, *sp, 1)))) return rc;
  ws_enter(ctx, s);
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t nq = sp->own_q.size(), ne = nq + sp->own_p.size(), beta = sp->beta;
  if (ne == 0) return HML_OK;
  u64 *ext = ctx->ws, *acc = ext + (size_t)beta * ne * N;
  if ((rc = shard_hoist_modup(ctx, sp, peers1, ext, s))) return rc;
  InnerRotSumArgs a{};
  a.d = (const u64 *)ct_own + (size_t)nq * N; a.ext = ext; a.c0 = (const u64 *)ct_own; a.acc = acc; a.z = (u64 *)z_own;
  a.N = (int)N; a.n_ext = (int)ne; a.L = (int)nq; a.beta = (int)beta; a.evk_limbs = (int)ne; a.pt_q_limbs = (int)nq; a.logN = p.logN;
  a.ext_f64 = p.logN > NTT_SMALL_LOG; a.evk_packed = 0;
  for (uint32_t r0 = 0; r0 < n_rot; r0 += IP_MAX_ROT) {
    const uint32_t n = std::min<uint32_t>(IP_MAX_ROT, n_rot - r0);
    a.accumulate = r0 > 0; a.n_rot = (int)n;
    for (uint32_t k = 0; k < n; ++k) {
      a.evk[k] = (const u64 *)keys[r0 + k]; a.pt[k] = (const u64 *)pts[r0 + k]; a.galois[k] = inner_galois(galois[r0 + k], N);
    }
    launch_inner_product_rot_sum(ctx->mc, sp->e_lm, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.kernel_launches++;
    ctx->exec.ewe_limbs += (uint64_t)n * (2ull * ne * beta + 2ull * ne + nq);
    ctx->exec.automorph_limbs += (uint64_t)n * nq;  // sigma_r(c0), applied on load
  }
  return check_launch(ctx, "sharded rotation sum inner product");
}

// phase 0 of the sharded product sum (shard.cu, hml_hmult_sum_sharded): d0 | d1 | d2 [nq][N] words = the sums of the n tensor
// products a[k] (x) b[k] on the owned Q-limbs, k_tensor_sum once per group of IP_MAX_ROT terms
int shard_tensor_sum(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t n, const uint64_t *const *a_own,
                     const uint64_t *const *b_own, uint64_t *d0, uint64_t *d1, uint64_t *d2, cudaStream_t s) {
  ShardPlan *sp;
  int rc = shard_plan_on_device(ctx, L, rank, world, &sp);
  if (rc) return rc;
  ws_enter(ctx, s);
  const uint32_t nq = sp->own_q.size();
  if (nq == 0) return HML_OK;
  TensorSumArgs a{};
  a.d0 = (u64 *)d0; a.d1 = (u64 *)d1; a.d2 = (u64 *)d2;
  a.comp_stride = (long long)nq * ctx->p.N; a.in_stride = 0; a.out_stride = 0;
  a.N = (int)ctx->p.N; a.pack01 = 0; a.mod0 = (int)rank; a.mod_step = (int)world;  // the sharded ModDown adds d0 / d1 as words
  for (uint32_t k0 = 0; k0 < n; k0 += IP_MAX_ROT) {
    const uint32_t m = std::min<uint32_t>(IP_MAX_ROT, n - k0);
    a.accumulate = k0 > 0; a.n_pairs = (int)m;
    for (uint32_t k = 0; k < m; ++k) { a.a[k] = (const u64 *)a_own[k0 + k]; a.b[k] = (const u64 *)b_own[k0 + k]; }
    launch_tensor_sum(ctx->mc, (int)nq, 1, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.ewe_limbs += 3ull * m * nq; ctx->exec.kernel_launches++;
  }
  return check_launch(ctx, "sharded tensor product sum");
}

// the rest of phase 1: ONE inverse NTT (+ scaling) of the owned P-limbs of all 2n accumulators, rotation r into this rank's
// contribution to slot r of its gather buffer 2 (slot_words apart; slot 0 is the key switch's layout)
int shard_hoist_intt(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, uint32_t n, uint64_t *g2_own, size_t slot_words, cudaStream_t s) {
  ShardPlan *sp;
  int rc = shard_plan_on_device(ctx, L, rank, world, &sp);
  if (rc) return rc;
  ws_enter(ctx, s);
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t nq = sp->own_q.size(), np = sp->own_p.size(), ne = nq + np;
  if (np == 0) return HML_OK;
  NttLaunch l{};
  l.in = ctx->ws + (size_t)sp->beta * ne * N; l.in_limb_stride = N; l.in_poly_stride = (long long)ne * N; l.in_batch_stride = 2ll * ne * N;
  // as in shard_mid_tail: limb k of p_lm sits at position nq + k of an accumulator, so the output base is shifted back by nq limbs
  l.out = (u64 *)g2_own + (size_t)rank * 2 * sp->gp * N - (size_t)nq * N; l.out_limb_stride = N; l.out_poly_stride = (long long)sp->gp * N;
  l.out_batch_stride = (long long)slot_words;
  l.n_limbs = np; l.n_polys = 2; l.n_batch = (int)n; l.post_scale = sp->scale2;
  run_ntt(ctx, true, sp->p_lm, l, s);
  return check_launch(ctx, "hoisted shard P-limb INTT");
}

// everything a sharded op at level L needs that costs host time or synchronises the device (plans, conversion images, offset
// tables, workspace for up to max_rot hoisted rotations): done ahead of the first exchange so that no rank sits in a spin-wait
// while a peer is still preparing
int shard_prepare(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers1, const uint64_t *const *peers2,
                  uint32_t max_rot) {
  ShardPlan *sp;
  int rc = shard_plan_on_device(ctx, L, rank, world, &sp);
  if (rc) return rc;
  for (auto &u : sp->up) if ((rc = shard_p2p_check(ctx, u))) return rc;
  if ((rc = shard_p2p_check(ctx, sp->down))) return rc;
  if ((rc = shard_peer_offsets(ctx, sp, peers1, false))) return rc;
  if ((rc = shard_peer_offsets(ctx, sp, peers2, true))) return rc;
  const uint32_t nq = sp->own_q.size();
  return ensure_ws(ctx, std::max(shard_hoist_ws_words(ctx->p, *sp, max_rot), (size_t)2 * nq * ctx->p.N));
}

// ------------------------------------------------------------------------------------------------ rescale
static size_t rs_ws_words(const Params &p, uint32_t L, uint32_t n_polys) { return (size_t)p.N * n_polys * L; }

// in: n_polys polys of L limbs (uniform stride in_poly_stride) -> out: n_polys polys of L-1 limbs
static int rescale_run(hml_ctx *ctx, uint32_t L, const u64 *in, long long in_poly_stride, uint32_t n_polys, u64 *out,
                       long long out_poly_stride, u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  LevelConsts *lc;
  int rc = get_level(ctx, L, &lc);
  if (rc) return rc;
  const size_t N = p.N;
  u64 *rb = ws, *rh = ws + (size_t)n_polys * N;  // rb [n_polys][N], rh [n_polys][L-1][N]
  {  // INTT of the dropped limb (reference :766-805)
    LimbMap lm; clear_map(lm);
    lm.mod[0] = L - 1; lm.pos[0] = 0;
    NttLaunch l{};
    l.n_batch = 1;
    l.in = in + (size_t)(L - 1) * N; l.out = rb; l.in_limb_stride = l.out_limb_stride = N;
    l.in_poly_stride = in_poly_stride; l.out_poly_stride = N; l.n_limbs = 1; l.n_polys = n_polys;
    run_ntt(ctx, true, lm, l, s);
  }
  // NTT of that polynomial under each remaining modulus (reference :807-822 counts ONE; delta D2), then the sub + mul
  // (reference :825-911)
  NttLaunch l{};
  l.n_batch = 1;
  l.in = rb; l.out = rh; l.in_limb_stride = 0; l.out_limb_stride = N; l.in_poly_stride = N;
  l.out_poly_stride = (long long)(L - 1) * N; l.n_limbs = L - 1; l.n_polys = n_polys;
  NttFuse &f = l.fuse;
  f.x = in; f.x_c_stride = in_poly_stride; f.dst = out; f.dst_c_stride = out_poly_stride; f.cst = lc->qlinv; f.n_c = (int)n_polys;
  if ((rc = ntt_sub_mul(ctx, lc->q_lm, l, s))) return rc;
  ctx->exec.ewe_limbs += 2ull * n_polys * (L - 1);
  return check_launch(ctx, "rescale");
}

extern "C" int hml_rescale(hml_ctx *ctx, uint32_t L, const uint64_t *in, uint64_t *out, void *stream) {
  int rc = check_level(ctx, L, 2);
  if (rc) return rc;
  if (!in || !out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, rs_ws_words(ctx->p, L, 1)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return rescale_run(ctx, L, (const u64 *)in, 0, 1, (u64 *)out, 0, ctx->ws, (cudaStream_t)stream);
}

// Sharded rescale (reference Rescale, src/Operation.cpp:741-911, on limb-sharded polynomials): the rank that owns limb L-1
// turns it to coefficient form (begin); after one flag exchange every rank transforms that polynomial under its own
// remaining moduli — reading it from the owner's buffer, over NVLink when the owner is a peer — and applies sub + mul (end).
//   x_own   [2][nq][N]   the two polynomials, this rank's Q-limbs at level L (ascending limb index)
//   r_own   [2][N]       this rank's peer-visible buffer; written only by the owner of limb L-1
//   r_src   [2][N]       the OWNER's buffer (own allocation or peer mapping)
//   out_own [2][nq'][N]  nq' = owned limbs below L-1
extern "C" int hml_rescale_shard_begin(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *x_own, uint64_t *r_own,
                                       void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (L < 2) return fail(ctx, HML_ERR_INVALID, "rescale needs L >= 2");
  if (!x_own || !r_own) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((L - 1) % world != rank) return HML_OK;  // not the owner of the dropped limb
  ShardPlan *sp;
  if ((rc = get_shard_plan(ctx, L, rank, world, &sp))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  const size_t N = ctx->p.N;
  const uint32_t nq = sp->own_q.size();
  LimbMap lm; clear_map(lm);
  lm.mod[0] = L - 1; lm.pos[0] = nq - 1;  // the dropped limb is the last one this rank owns
  NttLaunch l{};
  l.n_batch = 1;
  l.in = (const u64 *)x_own; l.in_limb_stride = N; l.in_poly_stride = (long long)nq * N;
  l.out = (u64 *)r_own - (size_t)(nq - 1) * N; l.out_limb_stride = N; l.out_poly_stride = N;  // position nq-1 lands on r_own
  l.n_limbs = 1; l.n_polys = 2;
  run_ntt(ctx, true, lm, l, (cudaStream_t)stream);
  return check_launch(ctx, "rescale shard begin");
}

extern "C" int hml_rescale_shard_end(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *x_own, const uint64_t *r_src,
                                     uint64_t *out_own, void *stream) {
  int rc = shard_check(ctx, L, rank, world);
  if (rc) return rc;
  if (L < 2) return fail(ctx, HML_ERR_INVALID, "rescale needs L >= 2");
  if (!x_own || !r_src || !out_own) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  ShardPlan *sp;
  if ((rc = get_shard_plan(ctx, L, rank, world, &sp))) return rc;
  const Params &p = ctx->p;
  const size_t N = p.N;
  const uint32_t nq = sp->own_q.size();
  const uint32_t nk = nq - ((L - 1) % world == rank ? 1 : 0);  // owned limbs that survive
  if (nk == 0) return HML_OK;
  if ((rc = ensure_ws(ctx, std::max(shard_ws_words(p, *sp), (size_t)2 * nk * N)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  LimbMap lm; clear_map(lm);
  for (uint32_t k = 0; k < nk; ++k) { lm.mod[k] = sp->own_q[k]; lm.pos[k] = k; }
  NttLaunch l{};
  l.n_batch = 1;
  l.in = (const u64 *)r_src; l.in_limb_stride = 0; l.in_poly_stride = N;
  l.out = ctx->ws; l.out_limb_stride = N; l.out_poly_stride = (long long)nk * N; l.n_limbs = nk; l.n_polys = 2;  // ws: [2][nk][N]
  NttFuse &f = l.fuse;
  f.x = (const u64 *)x_own; f.x_c_stride = (long long)nq * N;
  f.dst = (u64 *)out_own; f.dst_c_stride = (long long)nk * N; f.cst = sp->qlinv_own; f.n_c = 2;
  if ((rc = ntt_sub_mul(ctx, lm, l, (cudaStream_t)stream))) return rc;
  ctx->exec.ewe_limbs += 4ull * nk;
  return check_launch(ctx, "rescale shard end");
}

// ------------------------------------------------------------------------------------------------ top-level ops
// Batched ops run HML_BATCH_CHUNK (default 64; 32 until the end of round 2: 1-2 % slower, burst and sustained) ciphertexts per kernel launch: per-CTA set-up (twiddle staging, conversion matrices,
// key words) is paid once per chunk instead of once per ciphertext and grids are large enough to hide launch tails.
static uint32_t batch_chunk() {
  static const uint32_t v = [] {
    const char *e = getenv("HML_BATCH_CHUNK");  // tuning knob
    const int n = e ? atoi(e) : 64;
    return (uint32_t)std::min(std::max(n, 1), 64);
  }();
  return v;
}
#define HML_BATCH_CHUNK batch_chunk()

size_t hmult_ws_words(const Params &p, uint32_t L, uint32_t nb) {
  return (size_t)nb * ((size_t)p.N * 5 * L + std::max(ks_ws_words(p, L), rs_ws_words(p, L, 2)));
}

// nb ciphertext pairs [nb][2][L][N] -> [nb][2][L-1][N]
//
// Two-pass rings merge ModDown with Rescale.  With u = d + acc_Q * P^-1 (evaluation form) and v = BConv(z; P -> Q)
// (coefficient form), the textbook sequence is  c = u - NTT(v) * P^-1,  r = INTT(c[L-1]),
// out[l] = (c[l] - NTT_l([r]_{q_l})) * q_{L-1}^-1.  Every step is exact arithmetic mod q_l and the NTT is linear, so
//   r      = INTT_{L-1}(u[L-1]) - v[L-1] * P^-1                      (no forward transform of limb L-1 at all)
//   out[l] = (u[l] - NTT_l(v_l * P^-1 + [r]_{q_l})) * q_{L-1}^-1      (ONE forward transform per output limb instead of two)
// yields bit-identical residues with 2(L-1) forward transforms instead of 2L + 2(L-1).  v_l * P^-1 + [r]_{q_l} comes
// straight out of the base conversion: P^-1 is folded into the matrix on the host, r is computed by the conversion kernel on
// its staged tile (a 15-term dot product per coefficient) and rides in the otherwise padded 16th source row with matrix
// entry 1 (exact: it only adds one term < 2^36 to the 16-term sums).
//
// Everything after the tensor product: ten == null reads d0 | d1 | d2 from the workspace (each [nb][L][N]; d0 / d1 packed limbs
// on two-pass rings), ten != null (two-pass rings only) forms the tensor product inside the key switch.
static int hmult_tail(hml_ctx *ctx, uint32_t L, uint32_t nb, const KsTensor *ten, const u64 *evk, uint32_t evk_q_limbs, u64 *ct_out,
                      u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  const size_t N = p.N, PL = N * L;
  // d0 | d1 | d2 each [nb][L][N], cb [nb][2][L][N], then the key-switch / rescale workspace
  u64 *d0 = ws, *d1 = d0 + nb * PL, *d2 = d1 + nb * PL;
  const int merged = p.logN > NTT_SMALL_LOG;
  const bool in_ks = ten != nullptr;
  if (!merged) {  // single-pass rings: the textbook sequence
    u64 *cb = d2 + nb * PL, *rest = cb + 2 * nb * PL;
    int rc = ks_run(ctx, L, nb, {d2, (long long)PL}, evk, evk_q_limbs, {cb, (long long)(2 * PL)}, {cb + PL, (long long)(2 * PL)}, {d0, (long long)PL},
                    {d1, (long long)PL}, rest, s);
    if (rc) return rc;
    return rescale_run(ctx, L, cb, (long long)PL, 2 * nb, ct_out, (long long)(L - 1) * N, rest, s);
  }
  KeyDesc key;
  int rc = key_desc(ctx, L, evk, evk_q_limbs, &key);
  if (rc) return rc;
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const uint32_t A = p.alpha, E = L + A, AL = E + 1, beta = lc->beta;
  // yb [nb][L] | ext [nb][beta][E] | acc [nb][2][E+1] | wb [nb][2][L-1]; yb is free again after ModUp: ul [nb][2][N] reuses it
  u64 *yb = d2 + nb * PL, *ext = yb + (size_t)nb * L * N, *acc = ext + (size_t)nb * beta * E * N, *wb = acc + (size_t)nb * 2 * AL * N;
  // u[L-1] = d_c[L-1] + acc_c[L-1] * P^-1 is produced by the inner product itself (slot E of each accumulator) and its INTT
  // (reference Rescale INTT :766-805) rides in the launch that transforms the P-limbs: no extra launches, no re-reads
  const MergedU mu{in_ks ? nullptr : d0, (long long)(d1 - d0), (long long)PL};
  if ((rc = ks_front(ctx, lc, L, nb, {d2, (long long)PL}, key, yb, ext, acc, AL, s, &mu, nullptr, ten))) return rc;
  {  // w_l = v_l * P^-1 + [r]_{q_l}, l < L-1, with r = slot_E - v[L-1] * P^-1 folded on the staged tile (reference K8 :489-519)
    BConvArgs a{};
    a.in = acc; a.in_batch_stride = (long long)AL * N; a.out = wb; a.out_batch_stride = (long long)(L - 1) * N;
    a.step1 = nullptr; a.N = N; a.n_batches = 2 * nb; a.fold = lc->merged_fold; a.fold_mod = (int)(L - 1); a.out_f64 = 1;
    run_bconv(ctx, lc->merged_rest, lc->merged_src, a, s);
  }
  {  // out[l] = ((acc[l] * P^-1 + d[l]) - NTT_l(w_l)) * q_{L-1}^-1  (K9, K10, HMULT add and Rescale in one transform); with the
     // tensor product in the key switch acc[l] * P^-1 already holds d[l]
    NttLaunch l{};
    l.in = wb; l.out = wb; l.in_limb_stride = l.out_limb_stride = N; l.in_poly_stride = l.out_poly_stride = (long long)(L - 1) * N;
    l.n_limbs = L - 1; l.n_polys = 2 * nb; l.n_batch = 1; l.in_f64 = 1;
    NttFuse &f = l.fuse;
    f.x = acc; f.x_c_stride = (long long)AL * N; f.x_b_stride = 2ll * AL * N;
    if (!in_ks) { f.z = d0; f.z_c_stride = (long long)(d1 - d0); f.z_b_stride = (long long)PL; f.z_mask = 3; }
    f.dst = ct_out; f.dst_c_stride = (long long)(L - 1) * N; f.dst_b_stride = 2ll * (L - 1) * N;
    f.cst = lc->pinv; f.cst2 = lc->qlinv; f.n_c = 2; f.x_packed = ks_uses_hpip(ctx, L, nb) ? 0 : 1; f.z_packed = 1;
    run_ntt(ctx, false, lc->q_lm, l, s);
    ctx->exec.ewe_limbs += 2ull * nb * 4 * (L - 1);  // (+ d: with the tensor product in the key switch, the inner product's fold)
  }
  return check_launch(ctx, "hmult");
}

int hmult_run(hml_ctx *ctx, uint32_t L, uint32_t nb, const u64 *ct_a, const u64 *ct_b, const u64 *evk, uint32_t evk_q_limbs,
                     u64 *ct_out, u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  const size_t N = p.N, PL = N * L;
  const int merged = p.logN > NTT_SMALL_LOG;  // d0 / d1 then only feed element-wise epilogues: stored packed
  // batches on two-pass rings form the tensor product (reference :592-739) inside the key switch (KsTensor): d2 on the ModUp
  // transform's load, d0 / d1 folded into the accumulators by the inner product, so neither is stored nor read back
  const KsTensor ten{ct_a, ct_b, (long long)PL, (long long)(2 * PL)};
  const bool in_ks = merged && nb > 1;
  if (!in_ks) {
    u64 *d0 = ws, *d1 = d0 + nb * PL, *d2 = d1 + nb * PL;
    launch_tensor3(ctx->mc, (int)N, (int)L, ct_a, ct_a + PL, ct_b, ct_b + PL, d0, d1, d2, (int)nb, (long long)(2 * PL), (long long)PL, s, merged);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.ewe_limbs += 3ull * nb * L; ctx->exec.kernel_launches++;
  }
  return hmult_tail(ctx, L, nb, in_ks ? &ten : nullptr, evk, evk_q_limbs, ct_out, ws, s);
}

// Lazy relinearisation: out[b] = Rescale(Relin(sum_k a_k[b] (x) b_k[b])) for the nb outputs of a chunk, with ONE key switch and
// ONE rescale per output.  The tensor products are summed over Q (k_tensor_sum, one launch per group of IP_MAX_ROT pairs, later
// groups adding to the stored sums) into hmult_tail's d0 | d1 | d2, which then runs unchanged on them.  n_terms = 1 is
// hmult_run bit for bit; for n_terms >= 2 the result is not the sum of the products' hmults bit for bit (the approximate ModUp
// conversion and the rescale's lift are not additive) and the oracle defines the op (tests/orc_hmult_sum.py).  Input pointers
// advance by `off` words (the chunk's first output).
static int hmult_sum_run(hml_ctx *ctx, uint32_t L, uint32_t nb, uint32_t n_terms, const uint64_t *const *cts_a, const uint64_t *const *cts_b,
                         size_t off, const u64 *evk, uint32_t evk_q_limbs, u64 *ct_out, u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  const size_t N = p.N, PL = N * L;
  TensorSumArgs a{};
  a.d0 = ws; a.d1 = a.d0 + nb * PL; a.d2 = a.d1 + nb * PL;
  a.comp_stride = (long long)PL; a.in_stride = (long long)(2 * PL); a.out_stride = (long long)PL;
  a.N = (int)N; a.pack01 = p.logN > NTT_SMALL_LOG; a.mod0 = 0; a.mod_step = 1;
  for (uint32_t k0 = 0; k0 < n_terms; k0 += IP_MAX_ROT) {
    const uint32_t n = std::min<uint32_t>(IP_MAX_ROT, n_terms - k0);
    a.accumulate = k0 > 0; a.n_pairs = (int)n;
    for (uint32_t k = 0; k < n; ++k) { a.a[k] = (const u64 *)cts_a[k0 + k] + off; a.b[k] = (const u64 *)cts_b[k0 + k] + off; }
    launch_tensor_sum(ctx->mc, (int)L, (int)nb, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.ewe_limbs += 3ull * n * nb * L; ctx->exec.kernel_launches++;
  }
  return hmult_tail(ctx, L, nb, nullptr, evk, evk_q_limbs, ct_out, ws, s);
}

extern "C" int hml_hmult(hml_ctx *ctx, uint32_t L, const uint64_t *ct_a, const uint64_t *ct_b, const uint64_t *evk,
                         uint32_t evk_q_limbs, uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 2);
  if (rc) return rc;
  if (!ct_a || !ct_b || !evk || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, hmult_ws_words(ctx->p, L, 1)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return hmult_run(ctx, L, 1, (const u64 *)ct_a, (const u64 *)ct_b, (const u64 *)evk, evk_q_limbs, (u64 *)ct_out, ctx->ws, (cudaStream_t)stream);
}

size_t hrot_ws_words(const Params &p, uint32_t L, uint32_t nb) { return (size_t)nb * ((size_t)p.N * 2 * L + ks_ws_words(p, L)); }

// nb ciphertexts [nb][2][L][N] -> [nb][2][L][N]
int hrot_run(hml_ctx *ctx, uint32_t L, uint32_t nb, const u64 *ct, const u64 *rk, uint32_t evk_q_limbs, u64 g, u64 *ct_out,
                    u64 *ws, cudaStream_t s) {
  const size_t N = ctx->p.N, PL = N * L;
  u64 *sb = ws, *rest = sb + 2 * nb * PL;  // sb [nb][2][L][N]
  const bool in_place = ct_out < ct + 2 * nb * PL && ct < ct_out + 2 * nb * PL;  // the epilogue would gather c0 rows it has overwritten
  if (!in_place && ctx->p.logN > NTT_SMALL_LOG && galois_mod(g, N) != 1) {
    // two-pass rings: no kernel for the automorphism (reference :1302-1319).  In evaluation order sigma_g maps every 256-slot
    // row onto one source row (ntt_core.cuh RowSigma), so the ModUp INTT permutes c1 while it loads it (and leaves sigma(c1)
    // in sb for the inner product's own-digit term) and the ModDown epilogue gathers sigma(c0) from the raw c0
    const KsAuto au{g, sb + PL, (long long)(2 * PL)};
    ctx->exec.automorph_limbs += 2ull * nb * L;
    return ks_run(ctx, L, nb, {ct + PL, (long long)(2 * PL)}, rk, evk_q_limbs, {ct_out, (long long)(2 * PL)}, {ct_out + PL, (long long)(2 * PL)},
                  {ct, (long long)(2 * PL)}, {nullptr, 0}, rest, s, &au);
  }
  launch_automorph(ctx->p.logN, 2 * L * nb, ct, sb, g, s);  // reference :1302-1319
  prof_mark(ctx, HML_CLS_AUTO, s);
  ctx->exec.automorph_limbs += 2ull * nb * L; ctx->exec.kernel_launches++;
  // reference :1326-1357 key-switches AUTOOutput(0) and adds AUTOOutput(1) (naming only, delta D4):
  // textbook = key-switch sigma(c1), add sigma(c0) to the first output
  return ks_run(ctx, L, nb, {sb + PL, (long long)(2 * PL)}, rk, evk_q_limbs, {ct_out, (long long)(2 * PL)}, {ct_out + PL, (long long)(2 * PL)}, {sb, (long long)(2 * PL)},
                {nullptr, 0}, rest, s);
}

extern "C" int hml_hrotate(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *rotkey, uint32_t evk_q_limbs,
                           uint64_t galois_elt, uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (!ct || !rotkey || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  if (!(galois_elt & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, hrot_ws_words(ctx->p, L, 1)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return hrot_run(ctx, L, 1, (const u64 *)ct, (const u64 *)rotkey, evk_q_limbs, galois_elt, (u64 *)ct_out, ctx->ws, (cudaStream_t)stream);
}

// Hoisted rotations (SURVEY.md 8f rank 3): n_rot rotations of ONE ciphertext share one ModUp.  With t_j = NTT(ModUp_j(INTT(c1)))
// the extended digits of c1 (K1..K4, computed once),
//   out_r = (sigma_r(c0) + ks0, ks1),   (ks0, ks1) = ModDown( sum_j sigma_r(t_j) * rk_r[j] )
// sigma_r is applied to the digits while the inner product loads them, so the rotated digits never exist in memory.  This is
// NOT bit-identical to hml_hrotate: the approximate base conversion is not equivariant under the automorphism
// (ModUp(sigma(c1)) and sigma(ModUp(c1)) differ by multiples of the digit's modulus product), both are valid key-switch
// inputs; the oracle defines this op separately (oracle/oracle.c orc_hrotate_hoisted).  Reference: the rotation it replaces is
// src/Operation.cpp:1271-1358 run n_rot times; the reference itself cannot chain or share work between ops (:636,:675,:714).
static int hrot_hoisted_run(hml_ctx *ctx, uint32_t L, const u64 *ct, uint32_t n_rot, const uint64_t *const *rotkeys, uint32_t evk_q_limbs,
                            const uint64_t *galois, uint64_t *const *outs, u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  KeyDesc key;  // key.evk: rotation r's key, set in the loop
  int rc = key_desc(ctx, L, nullptr, evk_q_limbs, &key);
  if (rc) return rc;
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const size_t N = p.N, PL = N * L;
  const uint32_t A = p.alpha, E = L + A, beta = lc->beta;
  u64 *sb = ws, *yb = sb + 2 * PL, *ext = yb + PL, *acc = ext + (size_t)beta * E * N, *vb = acc + 2 * (size_t)E * N;
  const BatchPtr c1{ct + PL, 0};
  if ((rc = ks_modup(ctx, lc, L, 1, c1, yb, ext, s, nullptr))) return rc;
  for (uint32_t r = 0; r < n_rot; ++r) {
    // sigma_r(c0), the addend of the ModDown epilogue: gathered by the epilogue itself on two-pass rings (hrot_run), else a kernel
    const bool gather = p.logN > NTT_SMALL_LOG && galois_mod(galois[r], N) != 1;
    if (!gather) {
      launch_automorph(p.logN, L, ct, sb, galois[r], s);
      prof_mark(ctx, HML_CLS_AUTO, s);
      ctx->exec.kernel_launches++;
    }
    ctx->exec.automorph_limbs += L;
    key.evk = (const u64 *)rotkeys[r];
    if ((rc = ks_inner(ctx, lc, L, 1, c1, key, ext, acc, E, galois[r], s, nullptr, false))) return rc;
    u64 *o = (u64 *)outs[r];
    if ((rc = ks_tail(ctx, lc, L, 1, acc, vb, {o, 0}, {o + PL, 0}, {gather ? ct : sb, 0}, {nullptr, 0}, s, p.logN > NTT_SMALL_LOG,
                      gather ? galois[r] : 0)))
      return rc;
  }
  return check_launch(ctx, "hrotate hoisted");
}

extern "C" int hml_hrotate_hoisted(hml_ctx *ctx, uint32_t L, const uint64_t *ct, uint32_t n_rot, const uint64_t *const *rotkeys,
                                   uint32_t evk_q_limbs, const uint64_t *galois_elts, uint64_t *const *ct_outs, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (n_rot == 0) return HML_OK;
  if (!ct || !rotkeys || !galois_elts || !ct_outs) return fail(ctx, HML_ERR_INVALID, "null buffer");
  for (uint32_t r = 0; r < n_rot; ++r) {
    if (!rotkeys[r] || !ct_outs[r] || ct_outs[r] == ct) return fail(ctx, HML_ERR_INVALID, "null key / output, or an output aliasing the input");
    if (!(galois_elts[r] & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  }
  if (n_rot == 0) return HML_OK;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, hrot_ws_words(ctx->p, L, 1)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return hrot_hoisted_run(ctx, L, (const u64 *)ct, n_rot, rotkeys, evk_q_limbs, galois_elts, ct_outs, ctx->ws, (cudaStream_t)stream);
}

// Double-hoisted rotation sum (Bossuat et al., Eurocrypt 2021):  out = sum_r pt_r * rotate_r(ct) with ONE ModUp and ONE ModDown.
// With t = ModUp(c1) (K1..K4, once), the inner products stay in the extended basis, are weighted by the plaintexts there and
// summed (k_inner_rot_sum, one launch per group of IP_MAX_ROT rotations, later groups adding to the stored sums):
//   acc_c = sum_r pt_r * sum_j sigma_r(t_j) * rk_r[j][c],   z = sum_r pt_r * sigma_r(c0)   (Q-limbs)
//   out   = (ModDown(acc_0) + z, ModDown(acc_1))            (the P-limb INTT of ks_inner, then ks_tail, once)
// Not bit-identical to sum_r pt_r * hml_hrotate_hoisted_r: ModDown of a sum differs from the sum of ModDowns by the
// approximate conversion's overflow terms; the oracle defines the op itself (tests/orc_rotsum.py).  n = 1 with pt = 1 on every
// limb of the extended basis is hml_hrotate_hoisted bit for bit.
static int hrot_sum_hoisted_run(hml_ctx *ctx, uint32_t L, const u64 *ct, uint32_t n_rot, const uint64_t *const *rotkeys, uint32_t evk_q_limbs,
                                const uint64_t *galois, const uint64_t *const *pts, uint32_t pt_q_limbs, u64 *ct_out, u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  KeyDesc key;  // one key per rotation: only the layout is shared
  int rc = key_desc(ctx, L, nullptr, evk_q_limbs, &key);
  if (rc) return rc;
  if (pt_q_limbs < L || pt_q_limbs > p.max_level) return fail(ctx, HML_ERR_INVALID, "pt_q_limbs must be in [L, maxLevel]");
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const size_t N = p.N, PL = N * L;
  const uint32_t A = p.alpha, E = L + A, beta = lc->beta;
  // the workspace of hrot_hoisted_run: zb [L] (of 2L) | yb [L] | ext [beta][E] | acc [2][E] | vb [2][L]
  u64 *zb = ws, *yb = zb + 2 * PL, *ext = yb + PL, *acc = ext + (size_t)beta * E * N, *vb = acc + 2 * (size_t)E * N;
  const BatchPtr c1{ct + PL, 0};
  if ((rc = ks_modup(ctx, lc, L, 1, c1, yb, ext, s, nullptr))) return rc;
  LimbMap ip = lc->ext_lm;  // pos = limb index inside the key
  for (uint32_t e = 0; e < E; ++e) ip.pos[e] = (uint16_t)key.pos(e, L);
  InnerRotSumArgs a{};
  a.d = c1.ptr; a.ext = ext; a.c0 = ct; a.acc = acc; a.z = zb;
  a.N = (int)N; a.n_ext = (int)E; a.L = (int)L; a.beta = (int)beta; a.evk_limbs = (int)(key.q_limbs + A); a.pt_q_limbs = (int)pt_q_limbs; a.logN = p.logN;
  a.ext_f64 = p.logN > NTT_SMALL_LOG; a.evk_packed = key.packed ? 1 : 0;
  for (uint32_t r0 = 0; r0 < n_rot; r0 += IP_MAX_ROT) {
    const uint32_t n = std::min<uint32_t>(IP_MAX_ROT, n_rot - r0);
    a.accumulate = r0 > 0; a.n_rot = (int)n;
    for (uint32_t k = 0; k < n; ++k) {
      a.evk[k] = (const u64 *)rotkeys[r0 + k]; a.pt[k] = (const u64 *)pts[r0 + k]; a.galois[k] = inner_galois(galois[r0 + k], N);
    }
    launch_inner_product_rot_sum(ctx->mc, ip, a, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.kernel_launches++;
    ctx->exec.ewe_limbs += (uint64_t)n * (2ull * E * beta + 2ull * E + L);
    ctx->exec.automorph_limbs += (uint64_t)n * L;  // sigma_r(c0), applied on load
  }
  if ((rc = ks_inner(ctx, lc, L, 1, c1, key, ext, acc, E, 0, s, nullptr, true))) return rc;
  if ((rc = ks_tail(ctx, lc, L, 1, acc, vb, {ct_out, 0}, {ct_out + PL, 0}, {zb, 0}, {nullptr, 0}, s, false, 0))) return rc;
  return check_launch(ctx, "hrotate sum hoisted");
}

extern "C" int hml_hrotate_sum_hoisted(hml_ctx *ctx, uint32_t L, const uint64_t *ct, uint32_t n_rot, const uint64_t *const *rotkeys,
                                       uint32_t evk_q_limbs, const uint64_t *galois_elts, const uint64_t *const *pts, uint32_t pt_q_limbs,
                                       uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (n_rot == 0) return fail(ctx, HML_ERR_INVALID, "n_rot must be at least 1");
  if (!ct || !rotkeys || !galois_elts || !pts || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  const size_t w = 2 * (size_t)ctx->p.N * L;
  if (ct_out < ct + w && ct < ct_out + w) return fail(ctx, HML_ERR_INVALID, "the output overlaps the input");
  for (uint32_t r = 0; r < n_rot; ++r) {
    if (!rotkeys[r] || !pts[r]) return fail(ctx, HML_ERR_INVALID, "null key or plaintext");
    if (!(galois_elts[r] & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  }
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, hrot_ws_words(ctx->p, L, 1)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return hrot_sum_hoisted_run(ctx, L, (const u64 *)ct, n_rot, rotkeys, evk_q_limbs, galois_elts, pts, pt_q_limbs, (u64 *)ct_out, ctx->ws,
                              (cudaStream_t)stream);
}

// Z [2][L] | yb [L] | ext [beta][E] | A [2][E] | vb [2][L] | acc_j [2][E] | z_j [2][L] | ct_j [2][L] | ext_j [beta][E]
static size_t bsgs_ws_words(const Params &p, uint32_t L) {
  const size_t N = p.N, E = L + p.alpha;
  return N * (9 * (size_t)L + 4 * E + 2 * (size_t)p.beta(L) * E);
}

// Double-hoisted baby-step / giant-step linear transform (Bossuat et al., Eurocrypt 2021):
//   out = sum_j rotate( sum_i pt_{j,i} * rotate(ct, b_i), G_j )
// with the ModUp of c1 shared by every baby step and ONE final ModDown.  IP_g(c) = sum_d sigma_g(ModUp(c)_d) * rk_g[d] (in Q*P):
//   inner sum j:  acc_j = sum_{b_i != 1} pt_{j,i} * IP_{b_i}(c1),  z0_j = sum_i pt_{j,i} * sigma_{b_i}(c0),  z1_j = sum_{b_i = 1} pt_{j,i} * c1
//   giant j != 1: ct_j = (ModDown(acc_j) + (z0_j, z1_j)), then A += IP_{G_j}(ct_j.c1) and Z0 += sigma_{G_j}(ct_j.c0)
//   giant j  = 1: A += acc_j, Z0 += z0_j, Z1 += z1_j
//   out   = ModDown(A) + (Z0, Z1)
// Identity elements (g = 1 mod 2N) pay no key switch.  ModUps: 1 + k, ModDowns: k + 1 (k = non-identity giant steps), whatever
// n1.  The oracle defines the op (tests/orc_bsgs.py).
static int hrot_bsgs_hoisted_run(hml_ctx *ctx, uint32_t L, const u64 *ct, uint32_t n1, const uint64_t *baby_galois,
                                 const uint64_t *const *baby_keys, uint32_t n2, const uint64_t *giant_galois, const uint64_t *const *giant_keys,
                                 uint32_t evk_q_limbs, const uint64_t *const *pts, uint32_t pt_q_limbs, u64 *ct_out, u64 *ws, cudaStream_t s) {
  const Params &p = ctx->p;
  KeyDesc key;  // one key per rotation: only the layout is shared
  int rc = key_desc(ctx, L, nullptr, evk_q_limbs, &key);
  if (rc) return rc;
  if (pt_q_limbs < L || pt_q_limbs > p.max_level) return fail(ctx, HML_ERR_INVALID, "pt_q_limbs must be in [L, maxLevel]");
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const size_t N = p.N, PL = N * L;
  const uint32_t A = p.alpha, E = L + A, beta = lc->beta;
  u64 *Z = ws, *yb = Z + 2 * PL, *ext = yb + PL, *acc = ext + (size_t)beta * E * N, *vb = acc + 2 * (size_t)E * N;
  u64 *acc_j = vb + 2 * PL, *z_j = acc_j + 2 * (size_t)E * N, *ct_j = z_j + 2 * PL, *ext_j = ct_j + 2 * PL;
  const BatchPtr c1{ct + PL, 0};
  if ((rc = ks_modup(ctx, lc, L, 1, c1, yb, ext, s, nullptr))) return rc;
  LimbMap ip = lc->ext_lm;  // pos = limb index inside the key
  for (uint32_t e = 0; e < E; ++e) ip.pos[e] = (uint16_t)key.pos(e, L);
  InnerBsgsArgs a{};
  a.d = c1.ptr; a.ext = ext; a.c0 = ct;
  a.N = (int)N; a.n_ext = (int)E; a.L = (int)L; a.beta = (int)beta; a.evk_limbs = (int)(key.q_limbs + A); a.pt_q_limbs = (int)pt_q_limbs; a.logN = p.logN;
  a.ext_f64 = p.logN > NTT_SMALL_LOG; a.evk_packed = key.packed ? 1 : 0;
  // the inner sum of giant step j into (out_acc, z0, z1), in launches of IP_MAX_ROT baby steps
  auto inner_sum = [&](uint32_t j, u64 *out_acc, u64 *z0, u64 *z1, bool accumulate) {
    a.acc = out_acc; a.z = z0; a.z1 = z1;
    for (uint32_t i0 = 0; i0 < n1; i0 += IP_MAX_ROT) {
      const uint32_t n = std::min<uint32_t>(IP_MAX_ROT, n1 - i0);
      a.accumulate = accumulate || i0 > 0; a.n_rot = (int)n;
      uint32_t n_id = 0;
      for (uint32_t k = 0; k < n; ++k) {
        const unsigned g = inner_galois(baby_galois[i0 + k], N);
        a.galois[k] = g; a.evk[k] = g ? (const u64 *)baby_keys[i0 + k] : nullptr; a.pt[k] = (const u64 *)pts[(size_t)j * n1 + i0 + k];
        n_id += g ? 0 : 1;
      }
      launch_inner_product_bsgs(ctx->mc, ip, a, false, s);
      prof_mark(ctx, HML_CLS_EWE, s);
      ctx->exec.kernel_launches++;
      ctx->exec.ewe_limbs += (uint64_t)(n - n_id) * (2ull * E * beta + 2ull * E + L) + 2ull * n_id * L;
      ctx->exec.automorph_limbs += (uint64_t)(n - n_id) * L;  // sigma(c0), applied on load
    }
  };
  bool have_acc = false;  // A / Z0 hold a sum (later launches add to it); Z1 is used only by identity giant steps
  for (uint32_t j = 0; j < n2; ++j)
    if (!inner_galois(giant_galois[j], N)) { inner_sum(j, acc, Z, Z + PL, have_acc); have_acc = true; }
  const bool z1_used = have_acc;
  for (uint32_t j = 0; j < n2; ++j) {
    const unsigned g = inner_galois(giant_galois[j], N);
    if (!g) continue;
    inner_sum(j, acc_j, z_j, z_j + PL, false);
    if ((rc = ks_inner(ctx, lc, L, 1, c1, key, ext, acc_j, E, 0, s, nullptr, true))) return rc;
    if ((rc = ks_tail(ctx, lc, L, 1, acc_j, vb, {ct_j, 0}, {ct_j + PL, 0}, {z_j, 0}, {z_j + PL, 0}, s, false, 0))) return rc;
    // the baby digits in ext serve every later giant step: ct_j's digits get their own buffer
    if ((rc = ks_modup(ctx, lc, L, 1, {ct_j + PL, 0}, yb, ext_j, s, nullptr))) return rc;
    InnerBsgsArgs ga = a;
    ga.d = ct_j + PL; ga.ext = ext_j; ga.c0 = ct_j; ga.acc = acc; ga.z = Z; ga.z1 = nullptr;
    ga.accumulate = have_acc; ga.n_rot = 1; ga.evk[0] = (const u64 *)giant_keys[j]; ga.pt[0] = nullptr; ga.galois[0] = g;
    launch_inner_product_bsgs(ctx->mc, ip, ga, true, s);
    prof_mark(ctx, HML_CLS_EWE, s);
    ctx->exec.kernel_launches++;
    ctx->exec.ewe_limbs += 2ull * E * beta + L;
    ctx->exec.automorph_limbs += L;
    have_acc = true;
  }
  if ((rc = ks_inner(ctx, lc, L, 1, c1, key, ext, acc, E, 0, s, nullptr, true))) return rc;
  if ((rc = ks_tail(ctx, lc, L, 1, acc, vb, {ct_out, 0}, {ct_out + PL, 0}, {Z, 0}, {z1_used ? Z + PL : nullptr, 0}, s, false, 0))) return rc;
  return check_launch(ctx, "hrotate bsgs hoisted");
}

extern "C" int hml_hrotate_bsgs_hoisted(hml_ctx *ctx, uint32_t L, const uint64_t *ct, uint32_t n1, const uint64_t *baby_galois,
                                        const uint64_t *const *baby_keys, uint32_t n2, const uint64_t *giant_galois,
                                        const uint64_t *const *giant_keys, uint32_t evk_q_limbs, const uint64_t *const *pts,
                                        uint32_t pt_q_limbs, uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (n1 == 0 || n2 == 0) return fail(ctx, HML_ERR_INVALID, "n1 and n2 must be at least 1");
  if (!ct || !baby_galois || !giant_galois || !pts || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  const size_t N = ctx->p.N, w = 2 * N * L;
  if (ct_out < ct + w && ct < ct_out + w) return fail(ctx, HML_ERR_INVALID, "the output overlaps the input");
  for (int giant = 0; giant < 2; ++giant) {
    const uint64_t *gs = giant ? giant_galois : baby_galois;
    const uint64_t *const *keys = giant ? giant_keys : baby_keys;
    for (uint32_t i = 0; i < (giant ? n2 : n1); ++i) {
      if (!(gs[i] & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
      if (inner_galois(gs[i], N) && !(keys && keys[i])) return fail(ctx, HML_ERR_INVALID, "null key for a non-identity galois element");
    }
  }
  for (size_t k = 0; k < (size_t)n1 * n2; ++k)
    if (!pts[k]) return fail(ctx, HML_ERR_INVALID, "null plaintext");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  if ((rc = ensure_ws(ctx, bsgs_ws_words(ctx->p, L)))) return rc;
  ws_enter(ctx, (cudaStream_t)stream);
  return hrot_bsgs_hoisted_run(ctx, L, (const u64 *)ct, n1, baby_galois, baby_keys, n2, giant_galois, giant_keys, evk_q_limbs, pts,
                               pt_q_limbs, (u64 *)ct_out, ctx->ws, (cudaStream_t)stream);
}

static int ew_ct_op(hml_ctx *ctx, uint32_t L, const uint64_t *a, const uint64_t *b, bool b_is_pt, bool mul, uint64_t *out, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (!a || !b || !out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const size_t N = ctx->p.N, PL = N * L;
  // both components in one launch; a plaintext operand is repeated (stride 0)
  const long long ct = (long long)PL, pt = b_is_pt ? 0 : (long long)PL;
  if (mul) {
    const long long cs[5] = {ct, pt, 0, 0, ct};
    launch_ewe(ctx->mc, lc->q_lm, (int)N, (int)L, (const u64 *)a, (const u64 *)b, nullptr, nullptr, 0, (u64 *)out, (cudaStream_t)stream, 2, cs);
    prof_mark(ctx, HML_CLS_EWE, (cudaStream_t)stream);
  } else {
    const long long cs[5] = {ct, 0, pt, 0, ct};
    launch_ewe(ctx->mc, lc->q_lm, (int)N, (int)L, (const u64 *)a, nullptr, (const u64 *)b, nullptr, 0, (u64 *)out, (cudaStream_t)stream, 2, cs);
    prof_mark(ctx, HML_CLS_EWE, (cudaStream_t)stream);
  }
  ctx->exec.ewe_limbs += 2ull * L; ctx->exec.kernel_launches++;
  return check_launch(ctx, "ewe op");
}
// out = ct * pt + ct_add: PMULT followed by HADD as ONE element-wise pass — the reference's MULT instruction computes
// x1 * x2 + x3 * x4 natively (InsGen::GenEWE, reference src/InsGen.cpp:77-125), the two ops just never meet in one trace there.
// Bit-identical to hml_pmult + hml_hadd (exact arithmetic mod q).  `out` may alias ct_add.
extern "C" int hml_pmult_add(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *pt, const uint64_t *ct_add, uint64_t *out, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (!ct || !pt || !ct_add || !out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  LevelConsts *lc;
  if ((rc = get_level(ctx, L, &lc))) return rc;
  const long long PL = (long long)ctx->p.N * L;
  const long long cs[5] = {PL, 0, PL, 0, PL};
  launch_ewe(ctx->mc, lc->q_lm, (int)ctx->p.N, (int)L, (const u64 *)ct, (const u64 *)pt, (const u64 *)ct_add, nullptr, 0, (u64 *)out, (cudaStream_t)stream, 2, cs);
  prof_mark(ctx, HML_CLS_EWE, (cudaStream_t)stream);
  ctx->exec.ewe_limbs += 4ull * L; ctx->exec.kernel_launches++;
  return check_launch(ctx, "pmult + hadd");
}
extern "C" int hml_hadd(hml_ctx *ctx, uint32_t L, const uint64_t *a, const uint64_t *b, uint64_t *out, void *s) {
  return ew_ct_op(ctx, L, a, b, false, false, out, s);
}
extern "C" int hml_pmult(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *pt, uint64_t *out, void *s) {
  return ew_ct_op(ctx, L, ct, pt, true, true, out, s);
}
extern "C" int hml_padd(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *pt, uint64_t *out, void *s) {
  return ew_ct_op(ctx, L, ct, pt, true, false, out, s);
}

// ------------------------------------------------------------------------------------------------ batched
// chunks of at most HML_BATCH_CHUNK ciphertexts, one after the other on the caller's stream, sharing one workspace
template <class RunChunk>
static int run_batch_chunks(hml_ctx *ctx, uint32_t n, size_t ws_per_ct, cudaStream_t user, RunChunk run) {
  const uint32_t chunk = std::min<uint32_t>(HML_BATCH_CHUNK, n);
  int rc = ensure_ws(ctx, (size_t)chunk * ws_per_ct);
  if (rc) return rc;
  ws_enter(ctx, user);
  for (uint32_t i = 0; i < n; i += chunk)
    if ((rc = run(i, std::min(chunk, n - i), ctx->ws, user))) break;
  return rc;
}

extern "C" int hml_hmult_batch(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct_a, const uint64_t *ct_b,
                               const uint64_t *evk, uint32_t evk_q_limbs, uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 2);
  if (rc) return rc;
  if (n == 0) return HML_OK;  // an empty batch is a no-op whatever the pointers are
  if (!ct_a || !ct_b || !evk || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t N = ctx->p.N, in_w = 2 * N * L, out_w = 2 * N * (L - 1);
  return run_batch_chunks(ctx, n, hmult_ws_words(ctx->p, L, 1), (cudaStream_t)stream, [&](uint32_t i, uint32_t nb, u64 *ws, cudaStream_t s) {
    return hmult_run(ctx, L, nb, (const u64 *)ct_a + i * in_w, (const u64 *)ct_b + i * in_w, (const u64 *)evk, evk_q_limbs,
                     (u64 *)ct_out + i * out_w, ws, s);
  });
}

extern "C" int hml_hmult_sum(hml_ctx *ctx, uint32_t L, uint32_t n_terms, const uint64_t *const *cts_a, const uint64_t *const *cts_b,
                             uint32_t n_out, const uint64_t *evk, uint32_t evk_q_limbs, uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 2);
  if (rc) return rc;
  if (n_out == 0) return HML_OK;  // an empty batch is a no-op whatever the pointers are, as for hml_hmult_batch
  if (n_terms == 0) return fail(ctx, HML_ERR_INVALID, "n_terms must be at least 1");
  if (!cts_a || !cts_b || !evk || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  const size_t N = ctx->p.N, in_w = 2 * N * L, out_w = 2 * N * (L - 1);
  const uint64_t *out_end = ct_out + n_out * out_w;
  for (uint32_t k = 0; k < n_terms; ++k) {
    if (!cts_a[k] || !cts_b[k]) return fail(ctx, HML_ERR_INVALID, "null ciphertext");
    for (const uint64_t *in : {cts_a[k], cts_b[k]})
      if (ct_out < in + n_out * in_w && in < out_end) return fail(ctx, HML_ERR_INVALID, "the output overlaps an input");
  }
  KeyDesc key;  // checked before anything is enqueued
  if ((rc = key_desc(ctx, L, (const u64 *)evk, evk_q_limbs, &key))) return rc;
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  return run_batch_chunks(ctx, n_out, hmult_ws_words(ctx->p, L, 1), (cudaStream_t)stream, [&](uint32_t i, uint32_t nb, u64 *ws, cudaStream_t s) {
    return hmult_sum_run(ctx, L, nb, n_terms, cts_a, cts_b, i * in_w, (const u64 *)evk, evk_q_limbs, (u64 *)ct_out + i * out_w, ws, s);
  });
}

extern "C" int hml_hrotate_batch(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct, const uint64_t *rotkey,
                                 uint32_t evk_q_limbs, uint64_t galois_elt, uint64_t *ct_out, void *stream) {
  int rc = check_level(ctx, L, 1);
  if (rc) return rc;
  if (n == 0) return HML_OK;
  if (!ct || !rotkey || !ct_out) return fail(ctx, HML_ERR_INVALID, "null buffer");
  if (!(galois_elt & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  CU_TRY(ctx, cudaSetDevice(ctx->device));
  const size_t w = 2 * (size_t)ctx->p.N * L;
  return run_batch_chunks(ctx, n, hrot_ws_words(ctx->p, L, 1), (cudaStream_t)stream, [&](uint32_t i, uint32_t nb, u64 *ws, cudaStream_t s) {
    return hrot_run(ctx, L, nb, (const u64 *)ct + i * w, (const u64 *)rotkey, evk_q_limbs, galois_elt, (u64 *)ct_out + i * w, ws, s);
  });
}

// ------------------------------------------------------------------------------------------------ counts
extern "C" int hml_trace_counts(const char *op, uint32_t N, uint32_t batch_size, uint32_t max_level, uint32_t L, uint32_t alpha,
                                uint32_t bconv_high, uint32_t bconv_width, hml_counts *out) {
  if (!op || !out) return HML_ERR_INVALID;
  TraceShape s{N, batch_size, max_level, L, alpha, bconv_high, bconv_width};
  std::vector<StageCount> st;
  std::string err;
  memset(out, 0, sizeof(*out));
  if (!trace_op(op, s, st, err)) {
    g_create_err = err;
    const std::string o(op);
    const bool known = o == "hmult" || o == "hrotate" || o == "hadd" || o == "pmult" || o == "padd";
    return known ? HML_ERR_INVALID : HML_ERR_OP;
  }
  const uint64_t bc = s.batch_count();
  out->n_stages = (uint32_t)std::min<size_t>(st.size(), HML_MAX_STAGES);
  for (size_t i = 0; i < st.size(); ++i) {
    const uint64_t ins = st[i].limb_ops * bc;
    if (st[i].opcode == "NTT") out->ntt += ins;
    else if (st[i].opcode == "INTT") out->intt += ins;
    else if (st[i].opcode == "MULT") out->mult += ins;
    else if (st[i].opcode == "BCONV_STEP2") out->bconv_step2 += ins;
    else if (st[i].opcode == "AUTO") out->automorph += ins;
    if (i < HML_MAX_STAGES) {
      snprintf(out->stages[i].label, sizeof(out->stages[i].label), "%s", st[i].label.c_str());
      snprintf(out->stages[i].opcode, sizeof(out->stages[i].opcode), "%s", st[i].opcode.c_str());
      out->stages[i].limb_ops = st[i].limb_ops;
      out->stages[i].instructions = ins;
    }
  }
  out->total = out->ntt + out->intt + out->mult + out->bconv_step2 + out->automorph;
  out->driver_total = out->total - out->bconv_step2 + (uint64_t)bconv_high * bconv_width * out->bconv_step2;
  return HML_OK;
}

extern "C" int hml_get_counts(const hml_ctx *ctx, const char *op, uint32_t L, hml_counts *out) {
  if (!ctx) return HML_ERR_INVALID;
  const Params &p = ctx->p;
  return hml_trace_counts(op, p.N, p.batch_size, p.max_level, L, p.alpha, p.bconv_high, p.bconv_width, out);
}

extern "C" int hml_buffer_plan(const hml_ctx *ctx, const char *op, uint32_t L, char *out, uint64_t cap) {
  if (!ctx || !op || !out || cap == 0) return HML_ERR_INVALID;
  const Params &p = ctx->p;
  if (L < 1 || L > p.max_level) return HML_ERR_INVALID;
  const std::string o(op);
  const uint32_t A = p.alpha, E = L + A, beta = p.beta(L), bs = std::max<uint32_t>(1, p.batch_size);
  const bool merged = o == "hmult" && p.logN > NTT_SMALL_LOG;
  std::string text;
  uint64_t limb = 0;  // running limb index inside the workspace
  auto add = [&](const std::string &name, uint64_t n_limbs) {
    char line[160];
    snprintf(line, sizeof(line), "Malloc %s from %llu to %llu\n", name.c_str(), (unsigned long long)(limb * bs),
             (unsigned long long)((limb + (n_limbs ? n_limbs - 1 : 0)) * bs));
    text += line;
    limb += n_limbs;
  };
  auto keyswitch = [&](uint32_t acc_limbs, bool with_vb) {
    add("ModUpINTTOut", L);  // K1 + K2 (digit scaling folded in)
    for (uint32_t j = 0; j < beta; ++j) add("BConvOut_(" + std::to_string(j) + ") = NTTOut_beta(" + std::to_string(j) + ")", E);
    for (int k = 0; k < 2; ++k) add("InnerProduceOut_Key" + std::to_string(k) + (acc_limbs > E ? " (+ Rescale INTT slot)" : ""), acc_limbs);
    if (with_vb) for (int k = 0; k < 2; ++k) add("ModdownBConvOut_Key" + std::to_string(k) + " = NTTOut_ModDown_Key" + std::to_string(k), L);
  };
  if (o == "hmult") {
    if (L < 2) return HML_ERR_INVALID;
    add("TensorD0Out", L); add("TensorD1Out", L); add("TensorD2Out", L);
    if (merged) {
      keyswitch(E + 1, false);
      for (int k = 0; k < 2; ++k) add("ModdownBConvOut_Key" + std::to_string(k) + " (merged with Rescale)", L - 1);
    } else {
      for (int k = 0; k < 2; ++k) add("HMULTHaddOutput" + std::to_string(k), L);
      keyswitch(E, true);
    }
  } else if (o == "hrotate") {
    add("AUTOOutput(0)", L); add("AUTOOutput(1)", L);
    keyswitch(E, true);
  } else if (o == "hadd" || o == "pmult" || o == "padd") {
    text = "(no intermediates: one element-wise pass per component)\n";
  } else {
    return HML_ERR_OP;
  }
  snprintf(out, (size_t)cap, "%s", text.c_str());
  return HML_OK;
}

extern "C" int hml_exec_counts_get(const hml_ctx *ctx, hml_exec_counts *out) {
  if (!ctx || !out) return HML_ERR_INVALID;
  *out = ctx->exec;
  return HML_OK;
}
extern "C" int hml_exec_counts_reset(hml_ctx *ctx) {
  if (!ctx) return HML_ERR_INVALID;
  memset(&ctx->exec, 0, sizeof(ctx->exec));
  return HML_OK;
}
