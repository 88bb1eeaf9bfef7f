// Base conversion on the 5th-generation tensor cores: tcgen05.mma kind::i8 (u8 x u8 -> s32), accumulators in TMEM.
//
// Reference instruction class: BCONV_STEP2, InsGen::GenBCONV reference src/InsGen.cpp:263-313 (simulated unit BCONVU,
// reference src/Components.cpp:268-362); call sites KeySwitch::ModUpBConvStep2 reference src/Operation.cpp:137-188 and
// KeySwitch::ModDownBConvStep2 :489-519.
//
//   out[t][m] = sum_i y_i[m] * H[i][t]   (mod q_t),      y_i < 2^36,  H[i][t] < q_t < 2^36
//
// is an integer matrix product [coefficients x sources] x [sources x targets].  Integer split: y_i = sum_a Y_ia 2^(8a)
// (five bytes), and for every byte position a the host precomputes H_a[i][t] = H[i][t] * 2^(8a) mod q_t and splits THAT
// into five bytes B_b.  Then
//   out[t] = sum_b 2^(8b) T_b[t],     T_b[t] = sum_{(i,a)} Y_ia * byte_b(H_a[i][t])
// so ONE u8 x u8 -> s32 GEMM with K = 5 * n_src and five s32 columns per target does all the multiply work, and the
// epilogue is a 5-term shift-add (exact: < 2^52 for <= 48 sources, because byte 4 of a 36-bit value has 4 bits) plus a
// single reduction mod q_t on the FP64 pipe.  SURVEY.md / BASELINE.json north_star: "tensor cores are used only if an
// integer-split BConv beats CUDA cores in ncu" — measured numbers in profiles/README.md.
//
// Kernel shape (persistent CTAs, no warp specialisation, one __syncthreads per tile).  Two variants (template NT):
//   NT=256  conversions with <= 16 sources: TWO CTAs per SM, one TMEM accumulator buffer (256 columns) each; a CTA runs
//           pack -> MMA -> epilogue strictly in turn and the co-resident CTA fills its barrier and MMA waits
//   NT=512  more sources (shared memory allows one CTA): two TMEM buffers, the MMA of tile n+1 runs while tile n is drained
//   tile    128 coefficients (UMMA M = 128: TMEM lane = coefficient) x all targets (UMMA N = NP <= 256 s32 columns: byte
//           levels 0 and 4 of target t in columns 2t, 2t + 1, levels 1..3 in columns (b + 1) * ND + t) x K = 80 bytes per
//           16 sources, padded to a multiple of 32
//   A       [K/16][128 rows][16 B] in shared memory = the canonical K-major no-swizzle UMMA layout (core matrix = 8 rows x
//           16 B contiguous; SBO = 128 B between 8-row groups, LBO = 2048 B between 16-byte K chunks).  K order: chunk
//           (i/16)*5 + a holds byte a of sources 16*(i/16) .. +15, so a thread that holds four consecutive sources of one
//           coefficient emits one 32-bit word per byte position (3 PRMT) and a warp's 32 words are conflict-free
//   B       the host-built image, same layout with NP rows, copied once per CTA
//   loads   cp.async (8 B) into a ring of per-thread staging slots, issued STAGES tiles ahead; with BConvArgs::src_off the
//           sources may live in ANOTHER GPU's memory (limb-sharded key switch: the all-gather is this ring, over NVLink)
//   epilog  tcgen05.ld of 4 targets x 5 levels per trip (the next trip's load in flight), shift-add on the integer pipe, one
//           FP64 reduction, predicated-asm store (256 B coalesced per warp and target); the targets are dealt evenly to the
//           warps of a TMEM lane quarter as contiguous ranges, 3 or 4 per trip
// The optional fold of hmult's merged ModDown + Rescale (context.cu) is one more (virtual) target: its remainder r is
// computed first by every warp for its rows and added to every real target's sum before the reduction.
#include <algorithm>
#include <cstring>
#include <vector>

#include "ewe.cuh"
#include "launch.h"

namespace hml {

// ------------------------------------------------------------------------------------------------ host: operand image
static inline u64 h_mulmod64(u64 a, u64 b, u64 q) { return (u64)((unsigned __int128)a * b % q); }

static inline int umma_k_index(int i, int a) { return ((i >> 4) * 5 + a) * 16 + (i & 15); }
// accumulator column of (byte level b, target t): levels 0 and 4 are interleaved (columns 2t, 2t + 1) so that one TMEM load
// hands the epilogue the register pair (low word, top bits) it assembles the 64-bit sum in; levels 1..3 follow, ND apart
static inline int umma_n_index(int b, int t, int ND) { return b == 0 ? 2 * t : b == 4 ? 2 * t + 1 : (b + 1) * ND + t; }

bool bconv_image_shape(int n_src, int n_dst, int fold, BConvImage &im) {
  im = BConvImage{};
  if (n_src < 1 || n_src > 48 || n_dst < 1) return false;
  const int ntv = n_dst + (fold ? 1 : 0);
  const int ND = (ntv + 7) & ~7;
  const int NP = (5 * ND + 15) & ~15;
  if (NP > 256) return false;
  im.n16 = (n_src + 15) >> 4;
  im.K = (im.n16 * 80 + 31) & ~31;
  im.NP = NP; im.ND = ND; im.fold = fold ? 1 : 0;
  return true;
}

// hat [n_src][n_dst] row-major; dst_q[t] modulus of target t.  With fold != null the LAST source is the folded remainder's
// seed (see BConvArgs::fold): its matrix entries for the real targets are ignored (the remainder is added in the
// epilogue), fold[i] (i < n_src - 1) are the constants of the virtual target, modulus fold_q.
bool bconv_image_build(const u64 *hat, int n_src, int n_dst, const u64 *dst_q, const u64 *fold, u64 fold_q,
                       std::vector<uint8_t> &img, BConvImage &im) {
  if (!bconv_image_shape(n_src, n_dst, fold != nullptr, im)) return false;
  img.assign((size_t)im.K * im.NP, 0);
  const int ntv = n_dst + im.fold;
  for (int t = 0; t < ntv; ++t) {
    const bool virt = t == n_dst;
    const u64 q = virt ? fold_q : dst_q[t];
    if (q >> 36) return false;
    for (int i = 0; i < n_src; ++i) {
      u64 h;
      if (virt) h = i + 1 < n_src ? fold[i] % q : 1;
      else h = (fold && i + 1 == n_src) ? 0 : hat[(size_t)i * n_dst + t] % q;
      for (int a = 0; a < 5; ++a) {
        const u64 ha = h_mulmod64(h, (1ull << (8 * a)) % q, q);
        const int k = umma_k_index(i, a);
        for (int b = 0; b < 5; ++b) {
          const int n = umma_n_index(b, t, im.ND);
          img[(size_t)(k >> 4) * im.NP * 16 + (size_t)n * 16 + (k & 15)] = (uint8_t)(ha >> (8 * b));
        }
      }
    }
  }
  return true;
}

// CPU model of the kernel's data path (A packing order, image addressing, epilogue arithmetic), used by the CPU tests to
// check the host-built image and the exactness argument without a GPU.  y [n_src][M] canonical, out [n_dst][M] canonical.
extern "C" int hml_dbg_bconv_umma_model(const uint64_t *hat, int n_src, int n_dst, const uint64_t *dst_q, const uint64_t *fold,
                                        uint64_t fold_q, const uint64_t *y, int M, uint64_t *out) {
  BConvImage im;
  std::vector<uint8_t> img;
  if (!bconv_image_build((const u64 *)hat, n_src, n_dst, (const u64 *)dst_q, (const u64 *)fold, fold_q, img, im)) return 1;
  std::vector<uint8_t> arow(im.K);
  std::vector<int32_t> T(im.NP);
  auto value = [&](int t) {  // exact integer sum_b 2^(8b) T_b[t] as the epilogue forms it
    u64 acc = ((u64)(0x43300000u + (uint32_t)T[umma_n_index(4, t, im.ND)]) << 32) | (uint32_t)T[umma_n_index(0, t, im.ND)];
    acc += (u64)(uint32_t)T[umma_n_index(1, t, im.ND)] << 8;
    acc += (u64)(uint32_t)T[umma_n_index(2, t, im.ND)] << 16;
    acc += (u64)(uint32_t)T[umma_n_index(3, t, im.ND)] << 24;
    double d;
    memcpy(&d, &acc, 8);
    return d - 4503599627370496.0;
  };
  auto reduce = [](double v, double q) {
    const double qinv = 1.0 / q;
    const double qh = __builtin_fma(v, qinv, 6755399441055744.0) - 6755399441055744.0;
    return __builtin_fma(-qh, q, v);
  };
  for (int m = 0; m < M; ++m) {
    std::fill(arow.begin(), arow.end(), 0);
    for (int i = 0; i < n_src; ++i)
      for (int a = 0; a < 5; ++a) arow[umma_k_index(i, a)] = (uint8_t)(y[(size_t)i * M + m] >> (8 * a));
    for (int n = 0; n < im.NP; ++n) {
      int64_t s = 0;
      for (int k = 0; k < im.K; ++k) s += (int64_t)arow[k] * img[(size_t)(k >> 4) * im.NP * 16 + (size_t)n * 16 + (k & 15)];
      if (s > 0x7FFFFFFFll) return 2;
      T[n] = (int32_t)s;
    }
    double rf = 0.0;
    if (im.fold) {
      rf = reduce(value(n_dst), (double)fold_q);
      if (rf < 0.0) rf += (double)fold_q;
    }
    for (int t = 0; t < n_dst; ++t) {
      const double v = value(t) + rf;
      if (!(v < 9007199254740992.0)) return 3;
      double r = reduce(v, (double)dst_q[t]);
      if (r < 0.0) r += (double)dst_q[t];
      out[(size_t)t * M + m] = (uint64_t)r;
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------ device helpers
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor, K-major, no swizzle (layout_type 0), descriptor version 1 (sm_100)
__device__ __forceinline__ uint64_t umma_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!ok && ++spins > (1u << 24)) __trap();  // a tensor-core launch that never completes must not hang the device
  } while (!ok);
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
  uint32_t v;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr));
  return v;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&f)[5]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(f[0]), "+r"(f[1]), "+r"(f[2]), "+r"(f[3]), "+r"(f[4]) : : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// sum_b 2^(8b) T_b as an exact double (< 2^52): the 64-bit integer is assembled directly inside the mantissa of 2^52
// The multipliers arrive as kernel parameters (LevelMul) the compiler cannot see through, otherwise ptxas expands the wide
// multiply-adds by 2^8 / 2^16 / 2^24 into nine shift / carry instructions; (t0, t4) come out of one TMEM load as an aligned
// register pair, so the 64-bit accumulator is formed in place.
struct LevelMul {
  uint32_t m8, m16, m24;  // 2^8, 2^16, 2^24, passed as kernel parameters
};
__device__ __forceinline__ double level_sum(const LevelMul &lm, uint32_t t0, uint32_t t1, uint32_t t2, uint32_t t3, uint32_t t4) {
  u64 acc;
  asm("{\n\t.reg .b32 h;\n\tadd.u32 h, %2, 0x43300000;\n\tmov.b64 %0, {%1, h};\n\t}" : "=l"(acc) : "r"(t0), "r"(t4));
  asm("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc) : "r"(t1), "r"(lm.m8));
  asm("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc) : "r"(t2), "r"(lm.m16));
  asm("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc) : "r"(t3), "r"(lm.m24));
  return __longlong_as_double((long long)acc) - 4503599627370496.0;
}

constexpr int UMMA_THREADS = 512;
constexpr int UMMA_TM = 128;

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}
// accumulators of four consecutive targets: e = (level 0, level 4) pairs, l[b - 1] = levels 1..3
struct Quad {
  uint32_t e[8];
  uint32_t l[3][4];
};
// the loaded registers are operands of the wait, so that no use of them can be scheduled above it
__device__ __forceinline__ void tmem_ld_wait(Quad &q) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(q.e[0]), "+r"(q.e[1]), "+r"(q.e[2]), "+r"(q.e[3]), "+r"(q.e[4]), "+r"(q.e[5]), "+r"(q.e[6]), "+r"(q.e[7]),
                 "+r"(q.l[0][0]), "+r"(q.l[0][1]), "+r"(q.l[0][2]), "+r"(q.l[0][3]), "+r"(q.l[1][0]), "+r"(q.l[1][1]), "+r"(q.l[1][2]),
                 "+r"(q.l[1][3]), "+r"(q.l[2][0]), "+r"(q.l[2][1]), "+r"(q.l[2][2]), "+r"(q.l[2][3])
               :
               : "memory");
}
// the store is an asm statement so that the reduction above it is computed unconditionally (four interleaved dependency
// chains per trip) instead of being sunk into a per-target branch
__device__ __forceinline__ void st_if(void *p, u64 bits, bool on) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %2, 0;\n\t@p st.global.b64 [%0], %1;\n\t}" ::"l"(p), "l"(bits), "r"((uint32_t)on) : "memory");
}

// tile -> (batch, 128-coefficient block) without a division per tile: the walk advances by gridDim.x tiles
struct TileWalk {
  int batch, m;
  __device__ __forceinline__ void init(int tile, int tpb) { batch = tile / tpb; m = tile - batch * tpb; }
  __device__ __forceinline__ void step(int by, int tpb) {
    m += by;
    while (m >= tpb) { m -= tpb; ++batch; }
  }
};

// N16 = 16-source slabs; W = targets reduced per epilogue trip (3 or 4, whichever wastes fewer masked slots); NT = threads:
//   NT = 512  one CTA per SM, two TMEM buffers (512 columns): the MMA of tile n+1 overlaps the epilogue of tile n
//   NT = 256  two CTAs per SM, one TMEM buffer each (256 columns): a CTA runs pack -> MMA -> epilogue strictly in turn and
//             the OTHER CTA of the SM fills its barrier / MMA waits (16-source conversions only: shared memory)
template <int N16, bool FOLD, bool F64, int W, int NT>
__global__ void __launch_bounds__(NT, NT == 512 ? 1 : 2)
k_bconv_umma(const ModConst *__restrict__ mc, LimbMap src_lm, LimbMap dst_lm, BConvArgs a, const uint8_t *__restrict__ img, int K, int NP,
             int ND, int tiles_per_batch, int n_tiles, LevelMul lmul, const BConvJob *__restrict__ jobs, int n_jobs) {
  extern __shared__ __align__(128) unsigned char smem[];
  // multi-conversion launch: this CTA serves job blockIdx.x % n_jobs; its view of the grid is the CTAs of that job
  int bx = blockIdx.x, gx = gridDim.x;
  const BConvJob *job = nullptr;
  if (n_jobs > 0) {
    const int jid = blockIdx.x % n_jobs;
    job = jobs + jid;
    bx = blockIdx.x / n_jobs; gx = ((int)gridDim.x - jid + n_jobs - 1) / n_jobs;
    img = job->img; K = job->K; NP = job->NP; ND = job->ND;
    a.n_src = job->n_src; a.n_dst = job->n_dst;
    a.in += job->in_off; a.out += job->out_off;
  }
  auto src_pos = [&](int i) -> long long { return job ? (long long)job->src_pos[i] : (long long)src_lm.pos[i]; };
  auto dst_mod = [&](int t) -> int { return job ? (int)job->dst_mod[t] : (int)dst_lm.mod[t]; };
  auto dst_pos = [&](int t) -> long long { return job ? (long long)job->dst_pos[t] : (long long)dst_lm.pos[t]; };
  // the shuffle tells the compiler that `warp` is warp-uniform: TMEM addresses and target indices then live in uniform registers
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  constexpr int NBUF = NT == 512 ? 2 : 1;    // TMEM accumulator buffers = A operand buffers
  constexpr int IPT = UMMA_THREADS / NT;     // (coefficient, source group) items per thread and slab
  constexpr int NSUB = NT / 128;             // epilogue warps per TMEM lane quarter
  const uint32_t a_bytes = (uint32_t)UMMA_TM * K;
  unsigned char *As = smem;                                  // NBUF buffers
  unsigned char *Bs = smem + NBUF * a_bytes;                 // NP * K
  double2 *tq = reinterpret_cast<double2 *>(Bs + (size_t)NP * K);   // [ND + 4] (q, 1/q) per target (a trip may run 3 past the last)
  long long *toff = reinterpret_cast<long long *>(tq + ND + 4);  // [ND + 4] byte offset of the target's limb in the output
  uint64_t *bars = reinterpret_cast<uint64_t *>(toff + ND + 4);  // two mbarriers
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2);
  // raw source words on their way from HBM: STAGES tiles of [N16 * 4][512 threads] words, every thread owns its slots
  constexpr int STAGES = N16 <= 2 ? 3 : 2;
  constexpr uint32_t stage_bytes = N16 * 4 * UMMA_THREADS * 8;
  unsigned char *St = reinterpret_cast<unsigned char *>(bars + 4);

  uint32_t tmem_base = 0, idesc = 0, bar0 = 0;  // set after the set-up below; the role lambdas capture them by reference

  // loader role: coefficient row lr (+ NT/4 for the thread's second item when NT = 256), source group g (sources
  // 16 s + 4 g .. + 3 of every 16-source slab s)
  const int g = tid & 3, lr = tid >> 2;
  long long soff[N16][4];  // word offset of each of the thread's sources inside a batch (may be negative: a peer's buffer)
  unsigned live[N16] = {};  // bit k: source 16 s + 4 g + k exists (the others are zero rows)
#pragma unroll
  for (int s = 0; s < N16; ++s)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = s * 16 + g * 4 + k;
      const long long *so = job && job->src_off ? job->src_off : a.src_off;
      soff[s][k] = i < a.n_src ? (so ? __ldg(so + i) : src_pos(i) * a.N) + lr : -1;
      live[s] |= (i < a.n_src ? 1u : 0u) << k;
      if (i >= a.n_src) {  // padding sources: their staging slots are never written by a copy, they stay zero
#pragma unroll
        for (int d = 0; d < STAGES; ++d)
#pragma unroll
          for (int h = 0; h < IPT; ++h) reinterpret_cast<u64 *>(St + (size_t)d * stage_bytes)[(s * 4 + k) * UMMA_THREADS + tid + h * NT] = 0;
      }
    }
  // epilogue role: TMEM lanes 32 (warp % 4) .. + 31 = coefficient rows; the targets are dealt evenly to the four warps of a
  // lane quarter as contiguous ranges, walked W targets per trip
  const int row = ((warp & 3) << 5) | lane, sub = warp >> 2;
  const uint32_t t_lane = (uint32_t)((warp & 3) << 5) << 16;
  const int cb = a.n_dst / NSUB, cr = a.n_dst % NSUB;
  const int t_first = sub * cb + min(sub, cr);
  const int t_end = t_first + cb + (sub < cr ? 1 : 0);

  auto load_tile = [&](const TileWalk &w, int stage, bool on) {  // asynchronous: global -> the thread's staging slots
    if (on) {
      const u64 *in = a.in + (size_t)w.batch * a.in_batch_stride + (size_t)w.m * UMMA_TM;
      const uint32_t dst = smem_addr(St + (size_t)stage * stage_bytes) + tid * 8;
#pragma unroll
      for (int s = 0; s < N16; ++s)
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if ((live[s] >> k) & 1u) {
#pragma unroll
            for (int h = 0; h < IPT; ++h)
              asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + ((s * 4 + k) * UMMA_THREADS + h * NT) * 8),
                           "l"(in + soff[s][k] + h * (NT / 4))
                           : "memory");
          }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");  // one group per tile slot, empty or not: the wait counts stay uniform
  };
  auto pack_tile = [&](int stage, unsigned char *Ab) {
    const u64 *src = reinterpret_cast<const u64 *>(St + (size_t)stage * stage_bytes) + tid;
#pragma unroll
    for (int h = 0; h < IPT; ++h)
#pragma unroll
      for (int s = 0; s < N16; ++s) {
        u64 y[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) y[k] = src[(s * 4 + k) * UMMA_THREADS + h * NT];
        if (a.step1) {  // uniform: per-source scaling inside the conversion (primitive entry point)
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int i = s * 16 + g * 4 + k;
            if (i < a.n_src) {
              const ModConst m = mc[src_lm.mod[i]];
              const double2 sc = a.step1[i];
              y[k] = f64_to_canonical(mulmod_const(u64_to_f64(y[k]), sc.x, sc.y, m.q), m.qi);
            }
          }
        }
        const uint32_t l0 = (uint32_t)y[0], l1 = (uint32_t)y[1], l2 = (uint32_t)y[2], l3 = (uint32_t)y[3];
        const uint32_t h0 = (uint32_t)(y[0] >> 32), h1 = (uint32_t)(y[1] >> 32), h2 = (uint32_t)(y[2] >> 32), h3 = (uint32_t)(y[3] >> 32);
        uint32_t *dst = reinterpret_cast<uint32_t *>(Ab + ((size_t)(s * 5) * UMMA_TM + lr + h * (NT / 4)) * 16 + 4 * g);
        dst[0 * UMMA_TM * 4] = __byte_perm(__byte_perm(l0, l1, 0x0040), __byte_perm(l2, l3, 0x0040), 0x5410);
        dst[1 * UMMA_TM * 4] = __byte_perm(__byte_perm(l0, l1, 0x0051), __byte_perm(l2, l3, 0x0051), 0x5410);
        dst[2 * UMMA_TM * 4] = __byte_perm(__byte_perm(l0, l1, 0x0062), __byte_perm(l2, l3, 0x0062), 0x5410);
        dst[3 * UMMA_TM * 4] = __byte_perm(__byte_perm(l0, l1, 0x0073), __byte_perm(l2, l3, 0x0073), 0x5410);
        dst[4 * UMMA_TM * 4] = __byte_perm(__byte_perm(h0, h1, 0x0040), __byte_perm(h2, h3, 0x0040), 0x5410);
      }
  };
  auto issue_mma = [&](int buf) {  // one thread
    const uint32_t a_addr = smem_addr(As + (size_t)buf * a_bytes), b_addr = smem_addr(Bs);
    const uint32_t a_lbo = UMMA_TM * 16, b_lbo = (uint32_t)NP * 16;
    for (int ks = 0; ks < (K >> 5); ++ks)
      umma_i8(tmem_base + (uint32_t)buf * 256u, umma_desc(a_addr + ks * 2 * a_lbo, a_lbo, 128), umma_desc(b_addr + ks * 2 * b_lbo, b_lbo, 128), idesc,
              ks > 0);
    umma_commit(bar0 + 8u * buf);
  };
  auto epilogue = [&](const TileWalk &w, int buf) {
    unsigned char *out = reinterpret_cast<unsigned char *>(a.out + (size_t)w.batch * a.out_batch_stride + (size_t)w.m * UMMA_TM + row);
    const uint32_t tb = tmem_base + t_lane + (uint32_t)buf * 256u;
    double rf = 0.0;
    if (FOLD) {
      uint32_t f[5];
      f[0] = tmem_ld1(tb + 2 * a.n_dst);
      f[4] = tmem_ld1(tb + 2 * a.n_dst + 1);
#pragma unroll
      for (int b = 1; b < 4; ++b) f[b] = tmem_ld1(tb + (b + 1) * ND + a.n_dst);
      tmem_ld_wait(f);
      const double2 c = tq[a.n_dst];
      rf = canonicalize(reduce_signed(level_sum(lmul, f[0], f[1], f[2], f[3], f[4]), c.x, c.y), c.x);
    }
    auto fetch = [&](int t, Quad &q) {
      tmem_ld8(tb + 2 * t, q.e);
#pragma unroll
      for (int b = 0; b < 3; ++b) tmem_ld4(tb + (b + 2) * ND + t, q.l[b]);
    };
    auto reduce4 = [&](int t, Quad &q) {
#pragma unroll
      for (int j = 0; j < W; ++j) {
        const double2 c = tq[t + j];
        unsigned char *o = out + toff[t + j];
        double s = level_sum(lmul, q.e[2 * j], q.l[0][j], q.l[1][j], q.l[2][j], q.e[2 * j + 1]);
        if (FOLD) s += rf;
        const double r = reduce_signed(s, c.x, c.y);
        st_if(o, F64 ? (u64)__double_as_longlong(r) : f64_to_canonical(r, (u64)c.x), t + j < t_end);
      }
    };
    Quad qa, qb;
    if (t_first < t_end) fetch(t_first, qa);
#pragma unroll 1
    for (int t = t_first; t < t_end; t += 2 * W) {  // the next trip's accumulators are on their way from TMEM while this one is reduced
      tmem_ld_wait(qa);
      const bool more = t + W < t_end;
      if (more) fetch(t + W, qb);
      reduce4(t, qa);
      if (!more) break;
      tmem_ld_wait(qb);
      if (t + 2 * W < t_end) fetch(t + 2 * W, qa);
      reduce4(t + W, qb);
    }
    tmem_ld_wait();
  };

  const int n_my = bx < n_tiles ? (n_tiles - 1 - bx) / gx + 1 : 0;
  const int stride = gx;
  // the matrix image (a constant table) starts its trip before the programmatic dependency is resolved: asynchronous 16-byte
  // copies, the OLDEST copy group of every thread, so every later wait_group covers it
  for (uint32_t e = tid; e < (uint32_t)NP * K / 16; e += NT)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr(Bs + (size_t)e * 16)), "l"(img + (size_t)e * 16) : "memory");
  asm volatile("cp.async.commit_group;" ::: "memory");
  pdl_wait();  // the sources are another kernel's output; the outputs may still be read by one
  if (n_my > 0) {
    TileWalk wl, we;  // the loader runs STAGES tiles ahead of the epilogue
    wl.init(bx, tiles_per_batch);
    we = wl;
#pragma unroll
    for (int d = 0; d < STAGES; ++d) {
      load_tile(wl, d, d < n_my);
      wl.step(stride, tiles_per_batch);
    }
    // ---- constant set-up, while the matrix image and the first tiles are on their way: per-target table, TMEM, barriers
    {  // K padding of the A operand (chunks past 5 per slab): written once, never touched by the packer
      const uint32_t used = (uint32_t)N16 * 5 * UMMA_TM * 16, pad = a_bytes - used;
      for (uint32_t e = tid; e < NBUF * pad / 16; e += NT) {
        const uint32_t b = e / (pad / 16), o = e - b * (pad / 16);
        reinterpret_cast<uint4 *>(As + (size_t)b * a_bytes + used)[o] = make_uint4(0, 0, 0, 0);
      }
    }
    const int ntv = a.n_dst + (FOLD ? 1 : 0);
    for (int t = tid; t < ND + 4; t += NT) {
      double2 c = make_double2(1.0, 1.0);
      if (t < ntv) {
        const ModConst m = mc[t < a.n_dst ? dst_mod(t) : a.fold_mod];
        c = make_double2(m.q, m.qinv);
      }
      tq[t] = c;
      toff[t] = t < a.n_dst ? dst_pos(t) * a.N * 8 : 0;
    }
    if (warp == 0) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(tmem_slot)), "n"(256 * NBUF) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 32) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&bars[0])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&bars[1])));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("cp.async.wait_group %0;" ::"n"(STAGES) : "memory");  // the image has landed (the tile groups may still fly)
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    tmem_base = *tmem_slot;
    idesc = 0x20u | ((uint32_t)(NP >> 3) << 17) | (8u << 24);   // D = s32, A = B = u8, K-major, N = NP, M = 128
    bar0 = smem_addr(&bars[0]);
    if (NBUF == 2) {
      asm volatile("cp.async.wait_group %0;" ::"n"(STAGES - 1) : "memory");
      pack_tile(0, As);
      fence_async_smem();
      tc_fence_before();
      __syncthreads();
      if (tid == 0) {
        tc_fence_after();
        issue_mma(0);
      }
      int st_next = STAGES > 1 ? 1 : 0, st_load = 0;  // stage of tile it + 1 / stage the next load refills (= the one tile `it` was in)
      for (int it = 0; it < n_my; ++it) {
        const int buf = it & 1;
        const bool next = it + 1 < n_my;
        if (next) {
          asm volatile("cp.async.wait_group %0;" ::"n"(STAGES - 2) : "memory");
          pack_tile(st_next, As + (size_t)(buf ^ 1) * a_bytes);
          fence_async_smem();
        }
        tc_fence_before();
        __syncthreads();
        if (next && tid == 0) {
          tc_fence_after();
          issue_mma(buf ^ 1);
        }
        load_tile(wl, st_load, it + STAGES < n_my);
        wl.step(stride, tiles_per_batch);
        st_next = st_next + 1 == STAGES ? 0 : st_next + 1;
        st_load = st_load + 1 == STAGES ? 0 : st_load + 1;
        mbar_wait(bar0 + 8u * buf, (uint32_t)(it >> 1) & 1u);
        tc_fence_after();
        epilogue(we, buf);
        we.step(stride, tiles_per_batch);
      }
    } else {  // one accumulator buffer: pack -> MMA -> epilogue in turn; the co-resident CTA fills the waits
      int st = 0;
      for (int it = 0; it < n_my; ++it) {
        asm volatile("cp.async.wait_group %0;" ::"n"(STAGES - 1) : "memory");
        pack_tile(st, As);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();  // also: every warp has drained the accumulators of tile it - 1
        if (tid == 0) {
          tc_fence_after();
          issue_mma(0);
        }
        load_tile(wl, st, it + STAGES < n_my);
        wl.step(stride, tiles_per_batch);
        st = st + 1 == STAGES ? 0 : st + 1;
        mbar_wait(bar0, (uint32_t)it & 1u);
        tc_fence_after();
        epilogue(we, 0);
        we.step(stride, tiles_per_batch);
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(256 * NBUF) : "memory");
  }
}

template <int N16, bool FOLD, bool F64, int W, int NT>
static void launch_umma_t(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const BConvImage &im, cudaStream_t s) {
  const int tiles_per_batch = a.N / UMMA_TM, n_tiles = tiles_per_batch * a.n_batches;
  constexpr int STAGES = N16 <= 2 ? 3 : 2;
  constexpr int NBUF = NT == 512 ? 2 : 1;
  const size_t need = (size_t)NBUF * UMMA_TM * im.K + (size_t)im.NP * im.K + (size_t)(im.ND + 4) * 24 + 32 + (size_t)STAGES * N16 * 4 * UMMA_THREADS * 8;
  // NT = 512: at least half of the SM's shared memory, so that exactly ONE CTA is resident per SM (a second one would only
  // sit in tcgen05.alloc until the first ends); NT = 256: two fit (<= 113 KB each), a third does not
  const size_t smem = NT == 512 ? std::max<size_t>(need, 116 * 1024) : std::max<size_t>(need, 80 * 1024);
  static PerDeviceOnce once;
  static int n_sm[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (once.first()) {
    cudaFuncSetAttribute(k_bconv_umma<N16, FOLD, F64, W, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, NT == 512 ? 227 * 1024 : 113 * 1024);
    cudaDeviceGetAttribute(&n_sm[dev & 63], cudaDevAttrMultiProcessorCount, dev);
  }
  const int grid = std::min(n_tiles, (NT == 512 ? 1 : 2) * std::max(1, n_sm[dev & 63]));
  launch_pdl(k_bconv_umma<N16, FOLD, F64, W, NT>, dim3(grid), dim3(NT), smem, s, mc, src_lm, dst_lm, a, im.img, im.K, im.NP, im.ND, tiles_per_batch, n_tiles,
             LevelMul{256u, 65536u, 16777216u}, (const BConvJob *)nullptr, 0);
}

// several conversions with <= 16 sources each in one launch (the ModUp digits of a key switch): two CTAs per SM as above
template <bool F64, int W>
static void launch_umma_multi_t(const ModConst *mc, const BConvJob *d_jobs, int n_jobs, const BConvArgs &a, int K, int NP, int ND, cudaStream_t s) {
  constexpr int N16 = 1, NT = 256, STAGES = 3;
  const int tiles_per_batch = a.N / UMMA_TM, n_tiles = tiles_per_batch * a.n_batches;  // per job
  const size_t need = (size_t)UMMA_TM * K + (size_t)NP * K + (size_t)(ND + 4) * 24 + 32 + (size_t)STAGES * N16 * 4 * UMMA_THREADS * 8;
  const size_t smem = std::max<size_t>(need, 80 * 1024);
  static PerDeviceOnce once;
  static int n_sm[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (once.first()) {
    cudaFuncSetAttribute(k_bconv_umma<N16, false, F64, W, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024);
    cudaDeviceGetAttribute(&n_sm[dev & 63], cudaDevAttrMultiProcessorCount, dev);
  }
  const int grid = std::max(n_jobs, std::min(n_tiles * n_jobs, 2 * std::max(1, n_sm[dev & 63])));
  launch_pdl(k_bconv_umma<N16, false, F64, W, NT>, dim3(grid), dim3(NT), smem, s, mc, LimbMap{}, LimbMap{}, a, (const uint8_t *)nullptr, K, NP, ND,
             tiles_per_batch, n_tiles, LevelMul{256u, 65536u, 16777216u}, d_jobs, n_jobs);
}

bool launch_bconv_umma_multi(const ModConst *mc, const BConvJob *d_jobs, const BConvImage *ims, const int *n_dst, int n_jobs, const BConvArgs &a,
                             cudaStream_t s) {
  if (n_jobs < 2 || n_jobs > 8 || !d_jobs || a.N < 128 || a.N % 128 != 0 || a.step1 || a.fold || a.src_off || !bconv_umma_enabled())
    return false;
  int K = 0, NP = 0, ND = 0, waste3 = 0, waste4 = 0;
  for (int j = 0; j < n_jobs; ++j) {
    if (!ims[j].img || ims[j].n16 != 1 || ims[j].fold) return false;
    K = std::max(K, ims[j].K); NP = std::max(NP, ims[j].NP); ND = std::max(ND, ims[j].ND);
    const int c = (n_dst[j] + 1) / 2;  // targets per epilogue warp
    waste3 += ((c + 2) / 3) * 3 - c; waste4 += ((c + 3) / 4) * 4 - c;
  }
  // the shared-memory carve-up of a CTA follows ITS job's (K, NP, ND); the launch reserves the largest
  if (waste3 <= waste4) a.out_f64 ? launch_umma_multi_t<true, 3>(mc, d_jobs, n_jobs, a, K, NP, ND, s) : launch_umma_multi_t<false, 3>(mc, d_jobs, n_jobs, a, K, NP, ND, s);
  else a.out_f64 ? launch_umma_multi_t<true, 4>(mc, d_jobs, n_jobs, a, K, NP, ND, s) : launch_umma_multi_t<false, 4>(mc, d_jobs, n_jobs, a, K, NP, ND, s);
  return true;
}

template <int N16, bool FOLD, bool F64>
static void launch_umma_w(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const BConvImage &im, cudaStream_t s) {
  // targets per epilogue warp; trips of 3 or 4, whichever leaves fewer masked slots
  if constexpr (N16 == 1) {
    const int c = (a.n_dst + 1) / 2;
    if (((c + 2) / 3) * 3 < ((c + 3) / 4) * 4) launch_umma_t<1, FOLD, F64, 3, 256>(mc, src_lm, dst_lm, a, im, s);
    else launch_umma_t<1, FOLD, F64, 4, 256>(mc, src_lm, dst_lm, a, im, s);
  } else {
    const int c = (a.n_dst + 3) / 4;
    if (((c + 2) / 3) * 3 < ((c + 3) / 4) * 4) launch_umma_t<N16, FOLD, F64, 3, 512>(mc, src_lm, dst_lm, a, im, s);
    else launch_umma_t<N16, FOLD, F64, 4, 512>(mc, src_lm, dst_lm, a, im, s);
  }
}

template <int N16>
static void launch_umma_n(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const BConvImage &im, cudaStream_t s) {
  if (im.fold) {
    if (a.out_f64) launch_umma_w<N16, true, true>(mc, src_lm, dst_lm, a, im, s);
    else launch_umma_w<N16, true, false>(mc, src_lm, dst_lm, a, im, s);
  } else {
    if (a.out_f64) launch_umma_w<N16, false, true>(mc, src_lm, dst_lm, a, im, s);
    else launch_umma_w<N16, false, false>(mc, src_lm, dst_lm, a, im, s);
  }
}

void launch_bconv_umma(const ModConst *mc, const LimbMap &src_lm, const LimbMap &dst_lm, const BConvArgs &a, const BConvImage &im, cudaStream_t s) {
  switch (im.n16) {
    case 1: launch_umma_n<1>(mc, src_lm, dst_lm, a, im, s); break;
    case 2: launch_umma_n<2>(mc, src_lm, dst_lm, a, im, s); break;
    default: launch_umma_n<3>(mc, src_lm, dst_lm, a, im, s); break;
  }
}

}  // namespace hml
