// Host-buffer entry points: "the call a user makes" when the ciphertexts live in host memory.
//
// hml_hmult_host / hml_hrotate_host take the reference's own layout, uint64_t words (reference include/Context.h:8).  The
// *_packed variants take the 5-byte format (a plane of N uint32 low words followed by a plane of N high bytes per limb, the
// compact form of the device's packed limbs, modarith.cuh): a residue has elementBitWidth <= 36 significant bits, so 3 of the 8
// bytes of every word carry nothing over PCIe.  Both run the same pipeline: chunks of up to HOST_CHUNK ciphertexts, three
// streams (copy-in, compute, copy-out) and two staging slots, so the H2D of chunk i+1 and the D2H of chunk i-1 overlap the
// kernels of chunk i, and every chunk runs through the BATCHED schedule (one launch per stage for the whole chunk).
#include <algorithm>
#include <cstring>

#include "launch.h"
#include "ops.h"

using namespace hml;

// Ciphertexts per pipeline step.  The path is PCIe-bound (73 MB in and 36 MB out per hmult in the uint64 layout against
// ~0.2 ms of kernels), so what a larger chunk buys in kernel efficiency is invisible while the pipeline's tail — the last
// chunk's kernels and copy-out, which nothing overlaps — grows with it.
constexpr uint32_t HOST_CHUNK = 2;

// packed [n_limbs][5N] <-> words [n_limbs][N]; two coefficients per thread.  The packed limbs of the device (modarith.cuh)
// with a 5N-byte slot stride: 5N is a multiple of 80, so every slot stays 8-byte aligned.
__global__ void __launch_bounds__(256) k_unpack(const unsigned char *__restrict__ in, u64 *__restrict__ out, size_t N) {
  pdl_wait();
  const size_t i2 = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (i2 >= N / 2) return;
  const u64 *limb = reinterpret_cast<const u64 *>(in + (size_t)blockIdx.y * 5 * N);
  reinterpret_cast<ulonglong2 *>(out + (size_t)blockIdx.y * N)[i2] = ld_packed2(limb, N, i2);
}
__global__ void __launch_bounds__(256) k_pack(const u64 *__restrict__ in, unsigned char *__restrict__ out, size_t N) {
  pdl_wait();
  const size_t i2 = (size_t)blockIdx.x * 256 + threadIdx.x;
  if (i2 >= N / 2) return;
  const ulonglong2 v = __ldg(reinterpret_cast<const ulonglong2 *>(in + (size_t)blockIdx.y * N) + i2);
  st_packed2(reinterpret_cast<u64 *>(out + (size_t)blockIdx.y * 5 * N), N, i2, v.x, v.y);
}

extern "C" uint64_t hml_packed_bytes(const hml_ctx *ctx, uint64_t n_limbs) { return ctx ? 5ull * ctx->p.N * n_limbs : 0; }

extern "C" int hml_pack_host(const hml_ctx *ctx, const uint64_t *words, uint64_t n_limbs, void *packed) {
  if (!ctx || !words || !packed) return HML_ERR_INVALID;
  const size_t N = ctx->p.N;
  for (uint64_t l = 0; l < n_limbs; ++l) {
    const uint64_t *w = words + l * N;
    unsigned char *limb = (unsigned char *)packed + l * 5 * N;
    uint32_t *lo = (uint32_t *)limb;
    unsigned char *hi = limb + 4 * N;
    for (size_t i = 0; i < N; ++i) { lo[i] = (uint32_t)w[i]; hi[i] = (unsigned char)(w[i] >> 32); }
  }
  return HML_OK;
}
extern "C" int hml_unpack_host(const hml_ctx *ctx, const void *packed, uint64_t n_limbs, uint64_t *words) {
  if (!ctx || !words || !packed) return HML_ERR_INVALID;
  const size_t N = ctx->p.N;
  for (uint64_t l = 0; l < n_limbs; ++l) {
    uint64_t *w = words + l * N;
    const unsigned char *limb = (const unsigned char *)packed + l * 5 * N;
    const uint32_t *lo = (const uint32_t *)limb;
    const unsigned char *hi = limb + 4 * N;
    for (size_t i = 0; i < N; ++i) w[i] = ((uint64_t)hi[i] << 32) | lo[i];
  }
  return HML_OK;
}

#define HP_TRY(call)                                                                                                     \
  do {                                                                                                                   \
    cudaError_t e_ = (call);                                                                                             \
    if (e_ != cudaSuccess && first_err == cudaSuccess) { first_err = e_; where = #call; }                                \
  } while (0)

static int host_pipeline(hml_ctx *ctx, bool is_mult, bool packed, uint32_t L, uint32_t n, const void *a_host, const void *b_host,
                         const uint64_t *key_dev, uint32_t evk_q_limbs, uint64_t g, void *out_host) {
  int rc = check_level(ctx, L, is_mult ? 2 : 1);
  if (rc) return rc;
  if (!a_host || (is_mult && !b_host) || !key_dev || !out_host) return fail(ctx, HML_ERR_INVALID, "null buffer");
  if (n == 0) return HML_OK;
  HML_CU_TRY(ctx, cudaSetDevice(ctx->device));
  const uint32_t chunk = std::min(n, HOST_CHUNK);
  if ((rc = ensure_ws(ctx, is_mult ? hmult_ws_words(ctx->p, L, chunk) : hrot_ws_words(ctx->p, L, chunk)))) return rc;
  const size_t N = ctx->p.N, in_l = 2 * (size_t)L, out_l = 2 * (size_t)(is_mult ? L - 1 : L);  // limbs per ciphertext
  const size_t in_w = in_l * N, out_w = out_l * N;                                            // words per ciphertext
  const size_t n_in = is_mult ? 2 : 1;
  // one staging slot: word buffers for the chunk's inputs and output (+ byte buffers for the packed transfers)
  const size_t slot_words = chunk * (n_in * in_w + out_w);
  const size_t slot_bytes_packed = packed ? chunk * 5 * N * (n_in * in_l + out_l) : 0;
  const size_t slot_total = slot_words + (slot_bytes_packed + 7) / 8;
  if (ctx->stage_words < 2 * slot_total) {
    HML_CU_TRY(ctx, cudaDeviceSynchronize());
    if (ctx->stage) HML_CU_TRY(ctx, cudaFree(ctx->stage));
    ctx->stage = nullptr; ctx->stage_words = 0;
    HML_CU_TRY(ctx, cudaMalloc((void **)&ctx->stage, 2 * slot_total * 8));
    ctx->stage_words = 2 * slot_total;
  }
  if (!ctx->s_in) {
    HML_CU_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    HML_CU_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_comp, cudaStreamNonBlocking));
    HML_CU_TRY(ctx, cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
  }
  cudaEvent_t ev_in[2], ev_comp[2], ev_out[2];
  for (int k = 0; k < 2; ++k) {
    HML_CU_TRY(ctx, cudaEventCreateWithFlags(&ev_in[k], cudaEventDisableTiming));
    HML_CU_TRY(ctx, cudaEventCreateWithFlags(&ev_comp[k], cudaEventDisableTiming));
    HML_CU_TRY(ctx, cudaEventCreateWithFlags(&ev_out[k], cudaEventDisableTiming));
  }
  cudaError_t first_err = cudaSuccess;
  const char *where = "";
  ws_enter(ctx, ctx->s_comp);  // the workspace may still be in use by an op queued earlier on a caller stream
  const size_t ct_in_bytes = packed ? 5 * N * in_l : in_w * 8, ct_out_bytes = packed ? 5 * N * out_l : out_w * 8;
  rc = HML_OK;
  uint32_t k = 0;
  for (uint32_t i = 0; i < n && rc == HML_OK && first_err == cudaSuccess; i += chunk, ++k) {
    const uint32_t nb = std::min(chunk, n - i);
    const int sl = k & 1;
    u64 *sa = ctx->stage + sl * slot_total, *sb = sa + chunk * in_w, *so = sa + chunk * n_in * in_w;
    unsigned char *pa = reinterpret_cast<unsigned char *>(sa + slot_words), *pb = pa + chunk * 5 * N * in_l, *po = pa + chunk * n_in * 5 * N * in_l;
    if (k >= 2) HP_TRY(cudaStreamWaitEvent(ctx->s_in, ev_comp[sl], 0));  // the slot's inputs are free once chunk k-2 has been computed
    HP_TRY(cudaMemcpyAsync(packed ? (void *)pa : (void *)sa, (const char *)a_host + (size_t)i * ct_in_bytes, nb * ct_in_bytes, cudaMemcpyHostToDevice, ctx->s_in));
    if (is_mult)
      HP_TRY(cudaMemcpyAsync(packed ? (void *)pb : (void *)sb, (const char *)b_host + (size_t)i * ct_in_bytes, nb * ct_in_bytes, cudaMemcpyHostToDevice, ctx->s_in));
    HP_TRY(cudaEventRecord(ev_in[sl], ctx->s_in));
    HP_TRY(cudaStreamWaitEvent(ctx->s_comp, ev_in[sl], 0));
    if (k >= 2) HP_TRY(cudaStreamWaitEvent(ctx->s_comp, ev_out[sl], 0));  // the slot's output is free once chunk k-2 has been copied out
    if (packed) {
      const dim3 grid((unsigned)((N / 2 + 255) / 256), (unsigned)(nb * in_l));
      launch_pdl(k_unpack, grid, dim3(256), 0, ctx->s_comp, (const unsigned char *)pa, sa, N);
      if (is_mult) launch_pdl(k_unpack, grid, dim3(256), 0, ctx->s_comp, (const unsigned char *)pb, sb, N);
      ctx->exec.kernel_launches += is_mult ? 2 : 1;
    }
    rc = is_mult ? hmult_run(ctx, L, nb, sa, sb, (const u64 *)key_dev, evk_q_limbs, so, ctx->ws, ctx->s_comp)
                 : hrot_run(ctx, L, nb, sa, (const u64 *)key_dev, evk_q_limbs, g, so, ctx->ws, ctx->s_comp);
    if (packed) {
      launch_pdl(k_pack, dim3((unsigned)((N / 2 + 255) / 256), (unsigned)(nb * out_l)), dim3(256), 0, ctx->s_comp, (const u64 *)so, po, N);
      ctx->exec.kernel_launches++;
    }
    HP_TRY(cudaEventRecord(ev_comp[sl], ctx->s_comp));
    HP_TRY(cudaStreamWaitEvent(ctx->s_out, ev_comp[sl], 0));
    HP_TRY(cudaMemcpyAsync((char *)out_host + (size_t)i * ct_out_bytes, packed ? (const void *)po : (const void *)so, nb * ct_out_bytes, cudaMemcpyDeviceToHost,
                           ctx->s_out));
    HP_TRY(cudaEventRecord(ev_out[sl], ctx->s_out));
  }
  HP_TRY(cudaStreamSynchronize(ctx->s_in));
  HP_TRY(cudaStreamSynchronize(ctx->s_comp));
  HP_TRY(cudaStreamSynchronize(ctx->s_out));
  for (int q = 0; q < 2; ++q) { cudaEventDestroy(ev_in[q]); cudaEventDestroy(ev_comp[q]); cudaEventDestroy(ev_out[q]); }
  ctx->have_last = false;  // everything has completed: nothing left to order against
  if (rc) return rc;
  if (first_err != cudaSuccess) return fail(ctx, HML_ERR_CUDA, std::string("host pipeline: ") + where + ": " + cudaGetErrorString(first_err));
  return HML_OK;
}

extern "C" int hml_hmult_host(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *a, const uint64_t *b, const uint64_t *evk_dev,
                              uint32_t evk_q_limbs, uint64_t *out) {
  if (!ctx) return HML_ERR_INVALID;
  return host_pipeline(ctx, true, false, L, n, a, b, evk_dev, evk_q_limbs, 0, out);
}
extern "C" int hml_hrotate_host(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct, const uint64_t *rk_dev,
                                uint32_t evk_q_limbs, uint64_t g, uint64_t *out) {
  if (!ctx) return HML_ERR_INVALID;
  if (!(g & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  return host_pipeline(ctx, false, false, L, n, ct, nullptr, rk_dev, evk_q_limbs, g, out);
}
extern "C" int hml_hmult_host_packed(hml_ctx *ctx, uint32_t L, uint32_t n, const void *a, const void *b, const uint64_t *evk_dev,
                                     uint32_t evk_q_limbs, void *out) {
  if (!ctx) return HML_ERR_INVALID;
  return host_pipeline(ctx, true, true, L, n, a, b, evk_dev, evk_q_limbs, 0, out);
}
extern "C" int hml_hrotate_host_packed(hml_ctx *ctx, uint32_t L, uint32_t n, const void *ct, const uint64_t *rk_dev, uint32_t evk_q_limbs,
                                       uint64_t g, void *out) {
  if (!ctx) return HML_ERR_INVALID;
  if (!(g & 1)) return fail(ctx, HML_ERR_INVALID, "galois element must be odd");
  return host_pipeline(ctx, false, true, L, n, ct, nullptr, rk_dev, evk_q_limbs, g, out);
}
