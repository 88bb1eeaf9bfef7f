// Device-side building blocks of the two-kernel transforms (ntt.cu): asynchronous copies, the 16-point butterfly network and
// the row pass's swizzled shared-memory addressing.
#pragma once
#include "ntt.cuh"
#include "launch.h"

namespace hml {

// ---- asynchronous copies global -> shared
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
// bulk copy (TMA engine, no tensor map), completion on an mbarrier
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
  // no PTX labels: the helper can be inlined any number of times into one kernel
  unsigned ok = 0;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}
// 16-byte per-thread asynchronous copy (LDGSTS), L2 only
__device__ __forceinline__ void cp_async16(unsigned smem_dst, const void *gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory"); }

// ------------------------------------------------------------------------------------------------
// The 16-point network.  Level T (0..3) pairs registers D = 8 >> T apart; the 2^T butterfly groups of the
// level use w[0 .. 2^T).  Four levels = four radix-2 stages on 16 register-resident points; with the
// registers holding points  base + stride * j  the levels are the stages of distance 8, 4, 2, 1 strides.
// ------------------------------------------------------------------------------------------------
template <int T>
__device__ __forceinline__ void ct_level(double (&a)[16], const double (&w)[8], double q, double qinv) {
  constexpr int D = 8 >> T;
#pragma unroll
  for (int g = 0; g < (1 << T); ++g)
#pragma unroll
    for (int o = 0; o < D; ++o) ct_butterfly(a[g * 2 * D + o], a[g * 2 * D + o + D], w[g], q, qinv);
}
template <int T>
__device__ __forceinline__ void gs_level(double (&a)[16], const double (&w)[8], double q, double qinv) {
  constexpr int D = 8 >> T;
#pragma unroll
  for (int g = 0; g < (1 << T); ++g)
#pragma unroll
    for (int o = 0; o < D; ++o) gs_butterfly(a[g * 2 * D + o], a[g * 2 * D + o + D], w[g], q, qinv);
}
// CNT contiguous twiddles from shared memory (16-byte aligned when CNT >= 2)
template <int CNT>
__device__ __forceinline__ void lds_run(double (&w)[8], const double *p) {
  if constexpr (CNT == 1) {
    w[0] = p[0];
  } else {
#pragma unroll
    for (int k = 0; k < CNT / 2; ++k) {
      const double2 v = reinterpret_cast<const double2 *>(p)[k];
      w[2 * k] = v.x; w[2 * k + 1] = v.y;
    }
  }
}

constexpr int ROW_TILE_BYTES = NTT_TILE * 8;
constexpr int ROW_SMEM_BYTES = 3 * ROW_TILE_BYTES;  // twiddle blob + two data stages

// Byte offsets inside a stage, each family = one per-thread base XOR a compile-time constant (+ a constant):
//   round A, point l + 16*j:                  (pa ^ ((j & 7) << 4)) + 128 * j
//   round B, chunk of points 16*l + 2m, 2m+1:  pb ^ (m << 4)
//   output chunk (line 2m + l/8, chunk l%8):  (pc ^ (((2*m) & 7) << 4)) + 256 * m
struct RowAddr {
  unsigned pa, pb, pc;
  __device__ __forceinline__ unsigned A(int j) const { return (pa ^ ((j & 7) << 4)) + 128 * j; }
  __device__ __forceinline__ unsigned B(int m) const { return pb ^ (m << 4); }
  __device__ __forceinline__ unsigned C(int m) const { return (pc ^ (((2 * m) & 7) << 4)) + 256 * m; }
};
__device__ __forceinline__ RowAddr row_addr(int lane, int warp) {
  RowAddr r;
  const int l = lane & 15, rr = 2 * warp + (lane >> 4);
  const unsigned base = rr * 2048;
  r.pa = base + ((l >> 1) << 4) + ((l & 1) << 3);
  r.pb = base + l * 128 + ((l & 7) << 4);
  r.pc = base + (l >> 3) * 128 + (((l & 7) ^ (l >> 3)) << 4);
  return r;
}

// the warp's two rows (4 KB) of item `src_tile` (pointer to the CTA's first row): 8 chunks per lane
__device__ __forceinline__ void row_issue(const u64 *src_tile, unsigned stage_smem, int lane, int warp) {
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int qd = lane + 32 * k, g = (qd >> 3) & 15, cpos = qd & 7;
    const unsigned dst = stage_smem + (2 * warp + (qd >> 7)) * 2048 + g * 128 + ((cpos ^ (g & 7)) << 4);
    cp_async16(dst, src_tile + (size_t)warp * 512 + 2 * qd);
  }
}

// ---- automorphism inside a row pass.  Slot k of a limb holds the evaluation at psi^(2 brev(k) + 1); sigma_g: out[k] = in[k'],
// brev(k') = g * brev(k) + (g - 1) / 2 (mod N) (k_automorph, ewe.cu).  With k = R * 256 + klo (R = row, h = logN - 8 bits) the
// natural index is j = brev8(klo) * 2^h + brev_h(R), so
//   low h bits of j'  = (g * brev_h(R) + (g - 1) / 2) mod 2^h   -> depend on the row only: ONE source row R' per row
//   high 8 bits of j' = (g * brev8(klo) + d) mod 256,  d = (g * brev_h(R) + (g - 1) / 2) >> h    -> a permutation inside the row
struct RowSigma {
  unsigned src_row, d;
};
__device__ __forceinline__ RowSigma row_sigma(unsigned R, unsigned g, int h) {
  const unsigned b = __brev(R) >> (32 - h), t = g * b + ((g - 1u) >> 1);
  RowSigma r;
  r.src_row = __brev(t & ((1u << h) - 1u)) >> (32 - h);
  r.d = t >> h;
  return r;
}
// source slot (inside the source row) of destination slot klo
__device__ __forceinline__ unsigned sigma_src(unsigned klo, unsigned g, unsigned d) {
  return __brev((g * (__brev(klo) >> 24) + d) & 255u) >> 24;
}
// destination slot of source slot kp (ginv8 = g^-1 mod 256)
__device__ __forceinline__ unsigned sigma_dst(unsigned kp, unsigned ginv8, unsigned d) {
  return __brev((ginv8 * ((__brev(kp) >> 24) - d)) & 255u) >> 24;
}
__device__ __forceinline__ void cp_async8(unsigned smem_dst, const void *gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
// row_issue through the automorphism: the warp's two rows of tile `tile` of the limb at `src_limb`; every instruction reads
// 256 contiguous bytes of the source row and scatters them to the slots the transform expects
__device__ __forceinline__ void row_issue_sigma(const u64 *src_limb, unsigned stage_smem, int lane, int warp, int tile, unsigned g,
                                                unsigned ginv8, int logN) {
#pragma unroll
  for (int r2 = 0; r2 < 2; ++r2) {
    const RowSigma rs = row_sigma((unsigned)(tile * 16 + 2 * warp + r2), g, logN - NTT_ROW_LOG);
    const u64 *src = src_limb + ((size_t)rs.src_row << NTT_ROW_LOG);
    const unsigned row0 = stage_smem + (2 * warp + r2) * 2048;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const unsigned kp = lane + 32 * i, klo = sigma_dst(kp, ginv8, rs.d), line = klo >> 4;
      cp_async8(row0 + line * 128 + ((((klo >> 1) & 7) ^ (line & 7)) << 4) + (klo & 1) * 8, src + kp);
    }
  }
}

}  // namespace hml
