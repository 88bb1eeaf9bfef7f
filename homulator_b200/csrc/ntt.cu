// See ntt.cuh for the algorithm.  sm_100a only.
#include "ntt_core.cuh"

#include <cstring>
#include <type_traits>

namespace hml {

// ================================================================================ column passes
// Tile = C adjacent columns x all R1 rows = 16 * NT points for a CTA of NT threads (NT = 256: 32 KB tiles, two CTAs per
// SM; NT = 128: 16 KB tiles, four CTAs per SM, i.e. four independent barrier domains);
// thread (c, u) = (tid % C, tid / C), U = R1 / 16 row groups.
//   round A: rows u + U*j   (shared-memory word tid + NT*j): stages 0..3
//   round B: rows 16*u + j  : stages 4..LOGR1-1 (the last LOGR1-4 levels of the network)
// Work item = (limb-poly-batch y, tile); a CTA walks items blockIdx.x, + gridDim.x, ... with the next item's tile, its R1
// twiddles and its modulus constants already in flight (two stages).
template <int LOGR1, int NT>
struct ColCfg {
  static constexpr int R1 = 1 << LOGR1, TILE = 16 * NT, C = TILE / R1, SKIP = 8 - LOGR1, TILES = (1 << NTT_ROW_LOG) / C;
  static constexpr int STAGE_BYTES = TILE * 8 + 2048 + 64;  // tile | R1 twiddles | ModConst (48 B) | post-scale (16 B)
  static constexpr int MIN_CTAS = NT == 256 ? 3 : 6;
  static_assert(C >= 2 && C * (R1 / 16) == NT, "thread map");
};

struct ColWork {
  const u64 *in;
  u64 *out;
  int mi, limb, tile;
};

// Position of a work item in the (batch, poly, limb, tile) lattice.  A CTA starts at item blockIdx.x and advances by
// gridDim.x items per step; both are decomposed once, so the per-tile cost is a few adds instead of divisions.
struct ColPos {
  int tile, limb, poly, batch;
};
__device__ __forceinline__ ColPos col_pos(int wi, int tiles, int n_limbs, int n_polys) {
  ColPos p;
  p.tile = wi % tiles; wi /= tiles;
  p.limb = wi % n_limbs; wi /= n_limbs;
  p.poly = wi % n_polys; p.batch = wi / n_polys;
  return p;
}
__device__ __forceinline__ void col_advance(ColPos &p, const ColPos &st, int tiles, int n_limbs, int n_polys) {
  p.tile += st.tile; int c = p.tile >= tiles; p.tile -= c ? tiles : 0;
  p.limb += st.limb + c; c = p.limb >= n_limbs; p.limb -= c ? n_limbs : 0;
  p.poly += st.poly + c; c = p.poly >= n_polys; p.poly -= c ? n_polys : 0;
  p.batch += st.batch + c;
}
// next item of this CTA that is not skipped (digit-owned limbs of ModUp); false when the CTA has run out of work
template <int LOGR1, int NT>
__device__ __forceinline__ bool col_next(ColPos &p, const ColPos &st, bool first, const LimbMap &lm, const NttLaunch &l, bool in_is_out,
                                         ColWork &w) {
  using K = ColCfg<LOGR1, NT>;
  if (!first) col_advance(p, st, K::TILES, l.n_limbs, l.n_polys);
  while (p.batch < l.n_batch && p.poly == lm.skip[p.limb]) col_advance(p, st, K::TILES, l.n_limbs, l.n_polys);
  if (p.batch >= l.n_batch) return false;
  const long long slot = lm.pos[p.limb];
  w.out = l.out + (long long)p.batch * l.out_batch_stride + (long long)p.poly * l.out_poly_stride + slot * l.out_limb_stride + p.tile * K::C;
  w.in = in_is_out ? w.out
                   : l.in + (long long)p.batch * l.in_batch_stride + (long long)p.poly * l.in_poly_stride + slot * l.in_limb_stride + p.tile * K::C;
  w.mi = lm.mod[p.limb];
  w.limb = p.limb;
  w.tile = p.tile;
  return true;
}

template <int LOGR1, int NT>
__device__ __forceinline__ void col_issue(const ColWork &w, const double *tw_table, const ModConst *mc, const double2 *post_scale, int logN,
                                          unsigned stage_smem) {
  using K = ColCfg<LOGR1, NT>;
  const int tid = threadIdx.x;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int qd = tid + NT * k, row = qd / (K::C / 2), cc = qd % (K::C / 2);
    cp_async16(stage_smem + qd * 16, w.in + (size_t)row * (1 << NTT_ROW_LOG) + 2 * cc);
  }
  // the R1 twiddles and the per-modulus constants ride along, so the transform never waits on a dependent global load
  for (int x = tid; x < K::R1 / 2 + 4; x += NT) {
    const int y = x - K::R1 / 2;
    if (y < 0) cp_async16(stage_smem + K::TILE * 8 + x * 16, tw_table + ((size_t)w.mi << logN) + 2 * x);
    else if (y < 3) cp_async16(stage_smem + K::TILE * 8 + 2048 + y * 16, reinterpret_cast<const char *>(mc + w.mi) + y * 16);
    else if (post_scale) cp_async16(stage_smem + K::TILE * 8 + 2048 + 48, post_scale + w.limb);
  }
}

// ---- dynamic tile queue.  Measured with ncu (profiles/r2/ncu_hmult_batch32_r2.txt): with a static split (item i, i + grid, ...)
// the three persistent CTAs of an SM do not finish together — the warp scheduler favours the older CTA, which runs out of
// tiles early and leaves its slot empty (achieved occupancy 4.5 of 6 warps per scheduler, FP64 pipe 60 % busy).  With a queue
// (one atomic counter per launch, popped by thread 0 one tile ahead of its use) every CTA works until the launch is drained.
// Items are enumerated without the skipped (digit-owned) polys: tile fastest, then the (limb, poly) pairs of a ciphertext —
// the n_skip leading limbs of the launch have n_polys - 1 members, the others n_polys — then the ciphertexts.
struct ColSlot {
  const u64 *in;
  u64 *out;
  int mi, limb, tile, valid;
};
struct ColQueue {
  unsigned *ctr;   // [0] next item, [1] CTAs done (the last one zeroes both: the counters are ready for the next launch)
  int n_skip, pairs;
};
template <int LOGR1, int NT>
__device__ __forceinline__ void col_decode(unsigned wi, int total, const ColQueue &qu, const LimbMap &lm, const NttLaunch &l, bool in_is_out,
                                           ColSlot &s) {
  using K = ColCfg<LOGR1, NT>;
  s.valid = wi < (unsigned)total;
  if (!s.valid) return;
  const int tile = wi % K::TILES, r = wi / K::TILES, batch = r / qu.pairs;
  int rr = r - batch * qu.pairs, limb, poly;
  const int own_members = qu.n_skip * (l.n_polys - 1);
  if (rr < own_members) {
    limb = rr / (l.n_polys - 1); poly = rr - limb * (l.n_polys - 1);
    poly += poly >= lm.skip[limb];
  } else {
    rr -= own_members;
    limb = qu.n_skip + rr / l.n_polys; poly = rr % l.n_polys;
  }
  const long long slot = lm.pos[limb];
  s.out = l.out + (long long)batch * l.out_batch_stride + (long long)poly * l.out_poly_stride + slot * l.out_limb_stride + tile * K::C;
  s.in = in_is_out ? s.out : l.in + (long long)batch * l.in_batch_stride + (long long)poly * l.in_poly_stride + slot * l.in_limb_stride + tile * K::C;
  s.mi = lm.mod[limb]; s.limb = limb; s.tile = tile;
}
__device__ __forceinline__ ColWork col_take(const ColSlot &s) {
  ColWork w;
  w.in = s.in; w.out = s.out; w.mi = s.mi; w.limb = s.limb; w.tile = s.tile;
  return w;
}
__device__ __forceinline__ void col_queue_exit(const ColQueue &qu) {
  if (threadIdx.x == 0 && atomicAdd(qu.ctr + 1, 1u) == gridDim.x - 1) { qu.ctr[0] = 0; qu.ctr[1] = 0; __threadfence(); }
}

template <int LOGR1, int NT, bool IN_F64, bool DYN>
__global__ void __launch_bounds__(NT, (ColCfg<LOGR1, NT>::MIN_CTAS)) ntt_fwd_cols(NttTables t, int logN, LimbMap lm, NttLaunch l, int total, ColQueue qu) {
  using K = ColCfg<LOGR1, NT>;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, c = tid % K::C, u = tid / K::C;
  const unsigned smem0 = smem_u32(smem);
  __shared__ ColSlot slot[2];
  ColWork cur, nxt;
  ColPos pos, step;
  unsigned pend = 0;
  bool have;
  if constexpr (DYN) {
    // the first items are static (CTA b takes items b and b + grid: no queue round trip before the first loads); the queue hands out the rest
    ColSlot first;
    col_decode<LOGR1, NT>(blockIdx.x, total, qu, lm, l, false, first);
    have = first.valid;
    cur = col_take(first);
    pdl_wait();
    pend = blockIdx.x + gridDim.x;  // the second item is static too: the first pop of every CTA (a burst on one address when the
                                    // launch starts) then has a whole tile's time to return
  } else {
    pos = col_pos(blockIdx.x < total ? blockIdx.x : 0, K::TILES, l.n_limbs, l.n_polys);
    step = col_pos(gridDim.x, K::TILES, l.n_limbs, l.n_polys);
    pdl_wait();
    have = blockIdx.x < total && col_next<LOGR1, NT>(pos, step, true, lm, l, false, cur);
  }
  if (have) col_issue<LOGR1, NT>(cur, t.fwd, t.mc, nullptr, logN, smem0);
  cp_async_commit();
  for (int it = 0; have; ++it) {
    bool have_next;
    if constexpr (DYN) {
      if (tid == 0) col_decode<LOGR1, NT>(pend, total, qu, lm, l, false, slot[(it + 1) & 1]);  // the item popped during the previous tile
    } else {
      have_next = col_next<LOGR1, NT>(pos, step, false, lm, l, false, nxt);
    }
    cp_async_wait<0>();
    __syncthreads();  // tile `it` has landed for every thread; everybody is done with the other stage
    if constexpr (DYN) { have_next = slot[(it + 1) & 1].valid; nxt = col_take(slot[(it + 1) & 1]); }
    if (have_next) col_issue<LOGR1, NT>(nxt, t.fwd, t.mc, nullptr, logN, smem0 + ((it + 1) & 1) * K::STAGE_BYTES);
    cp_async_commit();
    double *data = reinterpret_cast<double *>(smem + (it & 1) * K::STAGE_BYTES);
    const double *tw = data + K::TILE;
    const ModConst &mc = *reinterpret_cast<const ModConst *>(tw + 256);
    const double q = mc.q, qinv = mc.qinv;
    double a[16], w[8];
#pragma unroll
    for (int j = 0; j < 16; ++j) a[j] = IN_F64 ? data[tid + NT * j] : u64_to_f64(reinterpret_cast<const u64 *>(data)[tid + NT * j]);
    // A constant added to coefficient 0 appears unchanged in every evaluation slot: subtracting h = (q-1)/2 here makes
    // the row pass's centred reduction land in [-h, h] = [0, q-1] - h, so its canonicalisation is one add (no sign fix).
    if (cur.tile == 0 && tid == 0 && l.fuse.x == nullptr && !l.out_f64) a[0] -= (q - 1.0) * 0.5;
    lds_run<1>(w, tw + 1); ct_level<0>(a, w, q, qinv);
    lds_run<2>(w, tw + 2); ct_level<1>(a, w, q, qinv);
    lds_run<4>(w, tw + 4); ct_level<2>(a, w, q, qinv);
    lds_run<8>(w, tw + 8); ct_level<3>(a, w, q, qinv);
#pragma unroll
    for (int j = 0; j < 16; ++j) data[tid + NT * j] = a[j];
    __syncthreads();
    // pop the tile after the next one half a tile before its loads are issued: late enough that the CTAs the scheduler
    // favours get there first (they are the ones that will have time for it), early enough to hide the round trip
    if constexpr (DYN) { if (tid == 0 && have_next) pend = 2 * gridDim.x + atomicAdd(qu.ctr, 1u); }
#pragma unroll
    for (int j = 0; j < 16; ++j) a[j] = data[(16 * u + j) * K::C + c];
    if constexpr (K::SKIP <= 0) { lds_run<1>(w, tw + (1 << (LOGR1 - 4)) + u); ct_level<0>(a, w, q, qinv); }
    if constexpr (K::SKIP <= 1) { lds_run<2>(w, tw + (1 << (LOGR1 - 3)) + 2 * u); ct_level<1>(a, w, q, qinv); }
    if constexpr (K::SKIP <= 2) { lds_run<4>(w, tw + (1 << (LOGR1 - 2)) + 4 * u); ct_level<2>(a, w, q, qinv); }
    lds_run<8>(w, tw + (1 << (LOGR1 - 1)) + 8 * u); ct_level<3>(a, w, q, qinv);
    double *outd = reinterpret_cast<double *>(cur.out) + c;
#pragma unroll
    for (int j = 0; j < 16; ++j) outd[(size_t)(16 * u + j) << NTT_ROW_LOG] = a[j];
    have = have_next; cur = nxt;
  }
  if constexpr (DYN) col_queue_exit(qu);
}

// inverse, second pass: raw doubles in `out` -> canonical words, post-scale folded into the N^-1 multiply
template <int LOGR1, int NT, bool DYN>
__global__ void __launch_bounds__(NT, (ColCfg<LOGR1, NT>::MIN_CTAS)) ntt_inv_cols(NttTables t, int logN, LimbMap lm, NttLaunch l, int total, ColQueue qu) {
  using K = ColCfg<LOGR1, NT>;
  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x, c = tid % K::C, u = tid / K::C;
  const unsigned smem0 = smem_u32(smem);
  __shared__ ColSlot slot[2];
  ColWork cur, nxt;
  ColPos pos, step;
  unsigned pend = 0;
  bool have;
  if constexpr (DYN) {
    // the first items are static (CTA b takes items b and b + grid: no queue round trip before the first loads); the queue hands out the rest
    ColSlot first;
    col_decode<LOGR1, NT>(blockIdx.x, total, qu, lm, l, true, first);
    have = first.valid;
    cur = col_take(first);
    pdl_wait();
    pend = blockIdx.x + gridDim.x;  // the second item is static too: the first pop of every CTA (a burst on one address when the
                                    // launch starts) then has a whole tile's time to return
  } else {
    pos = col_pos(blockIdx.x < total ? blockIdx.x : 0, K::TILES, l.n_limbs, l.n_polys);
    step = col_pos(gridDim.x, K::TILES, l.n_limbs, l.n_polys);
    pdl_wait();
    have = blockIdx.x < total && col_next<LOGR1, NT>(pos, step, true, lm, l, true, cur);
  }
  if (have) col_issue<LOGR1, NT>(cur, t.inv, t.mc, l.post_scale, logN, smem0);
  cp_async_commit();
  for (int it = 0; have; ++it) {
    bool have_next;
    if constexpr (DYN) {
      if (tid == 0) col_decode<LOGR1, NT>(pend, total, qu, lm, l, true, slot[(it + 1) & 1]);  // the item popped during the previous tile
    } else {
      have_next = col_next<LOGR1, NT>(pos, step, false, lm, l, true, nxt);
    }
    cp_async_wait<0>();
    __syncthreads();  // tile `it` has landed for every thread; everybody is done with the other stage
    if constexpr (DYN) { have_next = slot[(it + 1) & 1].valid; nxt = col_take(slot[(it + 1) & 1]); }
    if (have_next) col_issue<LOGR1, NT>(nxt, t.inv, t.mc, l.post_scale, logN, smem0 + ((it + 1) & 1) * K::STAGE_BYTES);
    cp_async_commit();
    double *data = reinterpret_cast<double *>(smem + (it & 1) * K::STAGE_BYTES);
    const double *tw = data + K::TILE;
    const ModConst &mc = *reinterpret_cast<const ModConst *>(tw + 256);
    const double q = mc.q, qinv = mc.qinv;
    double a[16], w[8];
#pragma unroll
    for (int j = 0; j < 16; ++j) a[j] = data[(16 * u + j) * K::C + c];
    lds_run<8>(w, tw + (1 << (LOGR1 - 1)) + 8 * u); gs_level<3>(a, w, q, qinv);
    if constexpr (K::SKIP <= 2) { lds_run<4>(w, tw + (1 << (LOGR1 - 2)) + 4 * u); gs_level<2>(a, w, q, qinv); }
    if constexpr (K::SKIP <= 1) { lds_run<2>(w, tw + (1 << (LOGR1 - 3)) + 2 * u); gs_level<1>(a, w, q, qinv); }
    if constexpr (K::SKIP <= 0) { lds_run<1>(w, tw + (1 << (LOGR1 - 4)) + u); gs_level<0>(a, w, q, qinv); }
#pragma unroll
    for (int j = 0; j < 16; ++j) data[(16 * u + j) * K::C + c] = a[j];
    __syncthreads();
    if constexpr (DYN) { if (tid == 0 && have_next) pend = 2 * gridDim.x + atomicAdd(qu.ctr, 1u); }  // see ntt_fwd_cols
#pragma unroll
    for (int j = 0; j < 16; ++j) a[j] = data[tid + NT * j];
    lds_run<8>(w, tw + 8); gs_level<3>(a, w, q, qinv);
    lds_run<4>(w, tw + 4); gs_level<2>(a, w, q, qinv);
    lds_run<2>(w, tw + 2); gs_level<1>(a, w, q, qinv);
    // last level (one twiddle w1 for the whole limb) with the post-scale c folded in: (x + y) * c and (x - y) * (w1 * c)
    double2 sc;
    if (l.post_scale) sc = *reinterpret_cast<const double2 *>(tw + 256 + 6);
    else sc = make_double2(mc.ninv, mc.ninv_q);
    const double w1c = mulmod_var(tw[1], sc.x, q, qinv);
    const u64 qi = mc.qi;
    u64 *outp = cur.out + tid % K::C;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const double sum = __dadd_rn(a[j], a[j + 8]), dif = __dsub_rn(a[j], a[j + 8]);
      outp[(size_t)(u + (K::R1 / 16) * j) << NTT_ROW_LOG] = f64_to_canonical(mulmod_const(sum, sc.x, sc.y, q), qi);
      outp[(size_t)(u + (K::R1 / 16) * (j + 8)) << NTT_ROW_LOG] = f64_to_canonical(mulmod_var(dif, w1c, q, qinv), qi);
    }
    have = have_next; cur = nxt;
  }
  if constexpr (DYN) col_queue_exit(qu);
}

// ================================================================================ row passes
// A CTA owns 16 consecutive 256-point rows (32 KB contiguous) of one limb and walks the items (ciphertext, poly) that
// share the limb's modulus; warp w owns rows 2w, 2w+1 (one per half-warp), so the whole pipeline is warp-local:
// no block barrier after the twiddle blob has landed.  Thread (rr, l) = (2w + lane/16, lane%16):
//   round A: points l + 16*j   (stages t = 128 .. 16),   round B: points 16*l + j   (stages t = 8 .. 1)
// Shared-memory rows are stored with their 16-byte chunks XOR-swizzled inside each 128-byte line
// (chunk c of line g at position c ^ (g & 7)): round A's 8-byte accesses, round B's per-thread 128-byte runs and the
// coalesced 16-byte output reads are all conflict-free.
// Items (ciphertext b, poly p) of one limb, walked with stride zn (the item splits of the grid) in the linear order b * n_polys + p.
struct RowItem {
  int b, p;
};
struct RowItems {
  int n_polys, n_batch, skip, step;
  __device__ __forceinline__ bool valid(const RowItem &i) const { return i.b < n_batch; }
  __device__ __forceinline__ RowItem next(RowItem i) const {
    do {
      i.p += step;
      while (i.p >= n_polys) { i.p -= n_polys; ++i.b; }
    } while (i.b < n_batch && i.p == skip);
    return i;
  }
};

// MAC launches (NttMac): a CTA must own ALL members (digits) of a ciphertext's limb tile, so the grid splits the ciphertexts
// (b = zi, + zn, ...) and walks the digits innermost.
struct RowItemsB {
  int n_polys, n_batch, skip, step;
  __device__ __forceinline__ bool valid(const RowItem &i) const { return i.b < n_batch; }
  __device__ __forceinline__ int first_p() const { return skip == 0 ? 1 : 0; }
  __device__ __forceinline__ int last_p() const { return skip == n_polys - 1 ? n_polys - 2 : n_polys - 1; }
  __device__ __forceinline__ RowItem next(RowItem i) const {
    ++i.p;
    if (i.p == skip) ++i.p;
    if (i.p >= n_polys) { i.p = first_p(); i.b += step; }
    return i;
  }
};

// MODE 0: plain transform; 1: fused element-wise epilogue (NttFuse); 2: fused key-switch inner product (NttMac); 3: the same
// with a packed key; 4 (inverse only): the input multiplied by NttLaunch::in_mul on load; 5: MODE 1 with cst2 and without z
// (the batched hmult's epilogue, whose addend is already in x)
template <bool INV, int MODE>
__global__ void __launch_bounds__(NTT_THREADS, 2) ntt_rows(NttTables t, int logN, LimbMap lm, NttLaunch l) {
  constexpr bool FUSE = MODE == 1 || MODE == 5, MAC = MODE == 2 || MODE == 3, KPK = MODE == 3;  // MODE 3: MAC with packed key limbs (NttMac::evk_packed)
  constexpr bool NOZ = MODE == 5;
  constexpr bool MUL = INV && MODE == 4;
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) unsigned long long bar;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // grid = (tiles * item splits, limbs), split index fastest: the CTAs that share a (limb, tile) — hence its 32 KB twiddle blob —
  // are adjacent in launch order, so all but the first of them find the blob in L2 (row-pass reads 2217 -> 1990 MB per launch)
  // (MAC launches walk the limbs backwards: the P-limbs, whose CTAs have one more digit to transform, start first)
  const int limb = MAC ? (int)(gridDim.y - 1 - blockIdx.y) : (int)blockIdx.y;
  const int zn = gridDim.x >> (logN - NTT_ROW_LOG - 4), tile_i = blockIdx.x / zn, zi = blockIdx.x - tile_i * zn;
  const int mi = lm.mod[limb];
  const double *blob = reinterpret_cast<const double *>(smem);
  if (tid == 0) mbar_init(&bar, 1);
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(&bar, ROW_TILE_BYTES);
    bulk_g2s(smem, (INV ? t.inv_rows : t.fwd_rows) + ((size_t)mi << logN) + (size_t)tile_i * NTT_TILE, ROW_TILE_BYTES, &bar);
  }
  const ModConst mc = t.mc[mi];
  const double q = mc.q, qinv = mc.qinv;
  const double hb = 4503599627370496.0 + (q - 1.0) * 0.5;  // 2^52 + h
  const RowAddr ad = row_addr(lane, warp);
  const unsigned data0 = smem_u32(smem) + ROW_TILE_BYTES;
  const long long slot = lm.pos[limb];
  const size_t tile_off = (size_t)tile_i * NTT_TILE;
  // forward rows read the raw doubles pass 1 left in `out`; inverse rows read the canonical input words
  auto src_of = [&](const RowItem &i) -> const u64 * {
    return (INV ? l.in + (long long)i.b * l.in_batch_stride + (long long)i.p * l.in_poly_stride + slot * l.in_limb_stride
                : l.out + (long long)i.b * l.out_batch_stride + (long long)i.p * l.out_poly_stride + slot * l.out_limb_stride) + tile_off;
  };
  auto dst_of = [&](const RowItem &i) -> u64 * {
    return l.out + (long long)i.b * l.out_batch_stride + (long long)i.p * l.out_poly_stride + slot * l.out_limb_stride + tile_off;
  };
  using Items = typename std::conditional<MAC, RowItemsB, RowItems>::type;
  const Items items{l.n_polys, l.n_batch, lm.skip[limb], zn};
  RowItem cur;
  if constexpr (MAC) cur = RowItem{zi, items.first_p()};
  else cur = items.next(RowItem{0, zi - zn});
  RowItem nxt = items.valid(cur) ? items.next(cur) : cur;
  // the multiplier's share of item i (NttLaunch::in_mul), addressed like `in`
  auto mul_of = [&](const RowItem &i) -> const u64 * {
    return l.in_mul + (long long)i.b * l.in_batch_stride + (long long)i.p * l.in_poly_stride + slot * l.in_limb_stride + tile_off;
  };
  // inverse rows may load through an automorphism (NttLaunch::in_galois)
  auto issue = [&](const RowItem &i, unsigned stage) {
    if constexpr (INV && MODE == 0) {
      if (l.in_galois) { row_issue_sigma(src_of(i) - tile_off, stage, lane, warp, tile_i, l.in_galois, l.in_ginv8, logN); return; }
    }
    if constexpr (MUL) {  // the multiplier's 4 KB for this warp's rows start their trip to L2 with the tile (one line per lane)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(mul_of(i) + (size_t)warp * 512 + (size_t)lane * 16));
    }
    row_issue(src_of(i), stage, lane, warp);
  };
  pdl_wait();  // the twiddle blob (a constant table) is already in flight; the data is another kernel's output
  if (items.valid(cur)) issue(cur, data0);
  cp_async_commit();
  if (items.valid(nxt)) issue(nxt, data0 + ROW_TILE_BYTES);
  cp_async_commit();
  mbar_wait(&bar, 0);
  const int l16 = lane & 15, rr = 2 * warp + (lane >> 4);
  const double *tw_a = blob + rr * 16;
  for (int k = 0; items.valid(cur); ++k) {
    const RowItem nn = items.valid(nxt) ? items.next(nxt) : nxt;
    cp_async_wait<1>();
    __syncwarp();
    unsigned char *data = smem + ROW_TILE_BYTES + (k & 1) * ROW_TILE_BYTES;
    double a[16], w[8];
    if constexpr (FUSE) {
      // the epilogue's operands (this warp's two rows = 512 coefficients of x and z) start their trip to L2 now
      const NttFuse &f = l.fuse;
      const long long fb = cur.p / f.n_c, fc = cur.p % f.n_c;
      const size_t nn = (size_t)1 << logN, c0 = tile_off + (size_t)warp * 512;  // first coefficient of the warp's rows
      auto prefetch = [&](const u64 *slot, int packed) {
        const unsigned char *b = reinterpret_cast<const unsigned char *>(slot);
        const unsigned char *p = nullptr;
        if (!packed) p = b + c0 * 8 + lane * 128;                       // 4 KB of words
        else if (lane < 16) p = b + c0 * 4 + lane * 128;                 // 2 KB of low words
        else if (lane < 20) p = b + 4 * nn + c0 + (lane - 16) * 128;     // 512 high bytes
        if (p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
      };
      prefetch(f.x + fc * f.x_c_stride + fb * f.x_b_stride + (size_t)limb * nn, f.x_packed);
      if (f.z != nullptr && ((f.z_mask >> fc) & 1u)) {
        const u64 *zslot = f.z + fc * f.z_c_stride + fb * f.z_b_stride + (size_t)limb * nn;
        if (f.z_galois) {  // the two source rows of this warp's rows (2 KB each: one line per lane)
          const RowSigma rs = row_sigma((unsigned)(tile_i * 16 + 2 * warp + (lane >> 4)), f.z_galois, logN - NTT_ROW_LOG);
          asm volatile("prefetch.global.L2 [%0];" ::"l"(zslot + ((size_t)rs.src_row << NTT_ROW_LOG) + (lane & 15) * 16));
        } else {
          prefetch(zslot, f.z_packed);
        }
      }
    }
    if constexpr (MAC) {
      // the key words this warp's two rows will be multiplied with (2 x 4 KB, + the own digit's at the first member) start
      // their trip to L2 now; one 128-byte line per lane
      const NttMac &mq = l.mac;
      const size_t nn = (size_t)1 << logN, c0 = tile_off + (size_t)warp * 512 + (size_t)lane * 16;
      const size_t kl = mq.key_pos[limb];
      auto pf = [&](const u64 *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); };
      // a key limb's share of the warp's 512 coefficients: 4 KB of words, or 2 KB of low words + 512 high bytes when packed
      auto pf_key = [&](int j, int c) {
        const u64 *slot = mq.evk + (((size_t)j * 2 + c) * mq.evk_limbs + kl) * nn;
        if constexpr (!KPK) { pf(slot + c0); return; }
        const unsigned char *b = reinterpret_cast<const unsigned char *>(slot);
        const size_t w0 = tile_off + (size_t)warp * 512;
        if (lane < 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(b + w0 * 4 + lane * 128));
        else if (lane < 20) asm volatile("prefetch.global.L2 [%0];" ::"l"(b + 4 * nn + w0 + (lane - 16) * 128));
      };
      pf_key(cur.p, 0);
      pf_key(cur.p, 1);
      const int own = lm.skip[limb];
      if (cur.p == items.first_p() && own != 0xFF) {
        pf_key(own, 0);
        pf_key(own, 1);
        pf(mq.d + (size_t)cur.b * mq.d_batch_stride + (size_t)limb * nn + c0);
      }
    }
    if constexpr (!INV) {
#pragma unroll
      for (int j = 0; j < 16; ++j) a[j] = *reinterpret_cast<const double *>(data + ad.A(j));
      lds_run<1>(w, tw_a + 1); ct_level<0>(a, w, q, qinv);
      lds_run<2>(w, tw_a + 2); ct_level<1>(a, w, q, qinv);
      lds_run<4>(w, tw_a + 4); ct_level<2>(a, w, q, qinv);
      lds_run<8>(w, tw_a + 8); ct_level<3>(a, w, q, qinv);
#pragma unroll
      for (int j = 0; j < 16; ++j) *reinterpret_cast<double *>(data + ad.A(j)) = a[j];
      __syncwarp();
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const double2 v = *reinterpret_cast<const double2 *>(data + ad.B(m));
        a[2 * m] = v.x; a[2 * m + 1] = v.y;
      }
      w[0] = blob[256 + tid]; ct_level<0>(a, w, q, qinv);
      lds_run<2>(w, blob + 512 + 2 * tid); ct_level<1>(a, w, q, qinv);
      lds_run<2>(w, blob + 1024 + 2 * tid);
      { const double2 v = *reinterpret_cast<const double2 *>(blob + 1536 + 2 * tid); w[2] = v.x; w[3] = v.y; }
      ct_level<2>(a, w, q, qinv);
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const double2 v = *reinterpret_cast<const double2 *>(blob + 2048 + 512 * m + 2 * tid);
        w[2 * m] = v.x; w[2 * m + 1] = v.y;
      }
      ct_level<3>(a, w, q, qinv);
      if constexpr (MAC) {
        // key-switch inner product on the transform's output (HPIP analogue, see NttMac): the lazy sums go through the
        // swizzled tile so that every lane works on the 16-byte chunks it loads and stores (256 B per half-warp)
#pragma unroll
        for (int m = 0; m < 8; ++m) *reinterpret_cast<double2 *>(data + ad.B(m)) = make_double2(a[2 * m], a[2 * m + 1]);
        __syncwarp();
        const NttMac &mq = l.mac;
        const size_t nn = (size_t)1 << logN;
        const size_t ci = tile_off + (size_t)rr * 256 + (l16 >> 3) * 16 + (l16 & 7) * 2;
        const size_t kl = mq.key_pos[limb];
        const int own = lm.skip[limb];
        const bool first = cur.p == items.first_p(), last = cur.p == items.last_p();
        const u64 *k0 = mq.evk + (((size_t)cur.p * 2 + 0) * mq.evk_limbs + kl) * nn + ci;
        const u64 *k1 = mq.evk + (((size_t)cur.p * 2 + 1) * mq.evk_limbs + kl) * nn + ci;
        u64 *A0 = mq.acc + (size_t)cur.b * mq.acc_batch_stride + (size_t)limb * nn + ci, *A1 = A0 + mq.acc_comp_stride;
        const bool with_own = first && own != 0xFF;
        const u64 *o0 = mq.evk + (((size_t)(with_own ? own : 0) * 2 + 0) * mq.evk_limbs + kl) * nn + ci;
        const u64 *o1 = mq.evk + (((size_t)(with_own ? own : 0) * 2 + 1) * mq.evk_limbs + kl) * nn + ci;
        const u64 *dd = mq.d + (size_t)cur.b * mq.d_batch_stride + (size_t)limb * nn + ci;
        const bool with_u = last && limb == mq.u_limb;
#pragma unroll
        for (int h = 0; h < 2; ++h) {  // four chunks at a time: every load of the half is in flight before the first product
          ulonglong2 kv0[4], kv1[4];
          double2 old0[4], old1[4];
          if constexpr (KPK) {  // packed key limbs (NttMac::evk_packed): joined after all loads are out
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              kv0[m] = ld_packed2_raw(k0 - ci, nn, (ci >> 1) + 16 * (4 * h + m));
              kv1[m] = ld_packed2_raw(k1 - ci, nn, (ci >> 1) + 16 * (4 * h + m));
            }
          } else {
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              kv0[m] = __ldg(reinterpret_cast<const ulonglong2 *>(k0 + 32 * (4 * h + m)));
              kv1[m] = __ldg(reinterpret_cast<const ulonglong2 *>(k1 + 32 * (4 * h + m)));
            }
          }
          if (!first) {  // this thread wrote these slots itself while it processed the previous member: plain (coherent) loads
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              old0[m] = *reinterpret_cast<const double2 *>(A0 + 32 * (4 * h + m));
              old1[m] = *reinterpret_cast<const double2 *>(A1 + 32 * (4 * h + m));
            }
          } else if (with_own) {  // the digit that owns this limb contributes the untouched input
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              const ulonglong2 dv = __ldg(reinterpret_cast<const ulonglong2 *>(dd + 32 * (4 * h + m)));
              const ulonglong2 w0 = KPK ? packed2_join(ld_packed2_raw(o0 - ci, nn, (ci >> 1) + 16 * (4 * h + m))) : __ldg(reinterpret_cast<const ulonglong2 *>(o0 + 32 * (4 * h + m)));
              const ulonglong2 w1 = KPK ? packed2_join(ld_packed2_raw(o1 - ci, nn, (ci >> 1) + 16 * (4 * h + m))) : __ldg(reinterpret_cast<const ulonglong2 *>(o1 + 32 * (4 * h + m)));
              const double dx = u64_to_f64(dv.x), dy = u64_to_f64(dv.y);
              old0[m] = make_double2(mulmod_var(dx, u64_to_f64(w0.x), q, qinv), mulmod_var(dy, u64_to_f64(w0.y), q, qinv));
              old1[m] = make_double2(mulmod_var(dx, u64_to_f64(w1.x), q, qinv), mulmod_var(dy, u64_to_f64(w1.y), q, qinv));
            }
          } else {
#pragma unroll
            for (int m = 0; m < 4; ++m) old0[m] = old1[m] = make_double2(0.0, 0.0);
          }
          if constexpr (KPK) {
#pragma unroll
            for (int m = 0; m < 4; ++m) { kv0[m] = packed2_join(kv0[m]); kv1[m] = packed2_join(kv1[m]); }
          }
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int mm = 4 * h + m;
            const double2 y = *reinterpret_cast<const double2 *>(data + ad.C(mm));
            const double s00 = old0[m].x + mulmod_var(y.x, u64_to_f64(kv0[m].x), q, qinv);
            const double s01 = old0[m].y + mulmod_var(y.y, u64_to_f64(kv0[m].y), q, qinv);
            const double s10 = old1[m].x + mulmod_var(y.x, u64_to_f64(kv1[m].x), q, qinv);
            const double s11 = old1[m].y + mulmod_var(y.y, u64_to_f64(kv1[m].y), q, qinv);
            if (!last) {
              *reinterpret_cast<double2 *>(A0 + 32 * mm) = make_double2(s00, s01);
              *reinterpret_cast<double2 *>(A1 + 32 * mm) = make_double2(s10, s11);
            } else {
              const u64 r00 = f64_to_canonical(reduce_signed(s00, q, qinv), mc.qi), r01 = f64_to_canonical(reduce_signed(s01, q, qinv), mc.qi);
              const u64 r10 = f64_to_canonical(reduce_signed(s10, q, qinv), mc.qi), r11 = f64_to_canonical(reduce_signed(s11, q, qinv), mc.qi);
              *reinterpret_cast<ulonglong2 *>(A0 + 32 * mm) = make_ulonglong2(r00, r01);
              *reinterpret_cast<ulonglong2 *>(A1 + 32 * mm) = make_ulonglong2(r10, r11);
              if (with_u) {  // hmult: u = acc * P^-1 + d on the limb the rescale drops, into slot u_slot (see InnerArgs::u_limb)
                const u64 *ua = mq.u_add + (size_t)cur.b * mq.u_add_batch_stride + (size_t)limb * nn;
                const ulonglong2 d0v = ld_packed2(ua, nn, (ci >> 1) + 16 * mm), d1v = ld_packed2(ua + mq.u_add_comp_stride, nn, (ci >> 1) + 16 * mm);
                const double2 c = mq.u_cst;
                const long long so = ((long long)mq.u_slot - limb) * (long long)nn;
                auto fin = [&](u64 r, u64 dw) { return f64_to_canonical(reduce_signed(mulmod_const(u64_to_f64(r), c.x, c.y, q) + u64_to_f64(dw), q, qinv), mc.qi); };
                *reinterpret_cast<ulonglong2 *>(A0 + so + 32 * mm) = make_ulonglong2(fin(r00, d0v.x), fin(r01, d0v.y));
                *reinterpret_cast<ulonglong2 *>(A1 + so + 32 * mm) = make_ulonglong2(fin(r10, d1v.x), fin(r11, d1v.y));
              }
            }
          }
        }
      } else if constexpr (!FUSE) {
        // canonical words back through the swizzled tile so that the global stores are 16 bytes per lane, 256 B per half-warp
        if (l.out_f64) {  // uniform: the consumer takes the lazy sums as they are
#pragma unroll
          for (int m = 0; m < 8; ++m) *reinterpret_cast<double2 *>(data + ad.B(m)) = make_double2(a[2 * m], a[2 * m + 1]);
        } else {
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          // values are (true - h) mod q (bias planted by the column pass): centred remainder + h is canonical
          const u64 v0 = (u64)__double_as_longlong(reduce_signed(a[2 * m], q, qinv) + hb) & 0x000FFFFFFFFFFFFFull;
          const u64 v1 = (u64)__double_as_longlong(reduce_signed(a[2 * m + 1], q, qinv) + hb) & 0x000FFFFFFFFFFFFFull;
          *reinterpret_cast<ulonglong2 *>(data + ad.B(m)) = make_ulonglong2(v0, v1);
        }
        }
        __syncwarp();
        u64 *outp = dst_of(cur) + (size_t)rr * 256 + (l16 >> 3) * 16 + (l16 & 7) * 2;
#pragma unroll
        for (int m = 0; m < 8; ++m)
          *reinterpret_cast<ulonglong2 *>(outp + 32 * m) = *reinterpret_cast<const ulonglong2 *>(data + ad.C(m));
      } else {
        // fused epilogue: the raw lazy sums go through the swizzled tile, then every lane handles the 16-byte chunks it
        // will store, so x, z and dst are all accessed 256 B per half-warp
#pragma unroll
        for (int m = 0; m < 8; ++m) *reinterpret_cast<double2 *>(data + ad.B(m)) = make_double2(a[2 * m], a[2 * m + 1]);
        __syncwarp();
        const NttFuse &f = l.fuse;
        const long long fb = cur.p / f.n_c, fc = cur.p % f.n_c;  // n_batch == 1 for fused launches
        const size_t nn = (size_t)1 << logN;
        const size_t ci = tile_off + (size_t)rr * 256 + (l16 >> 3) * 16 + (l16 & 7) * 2;  // first coefficient of this lane's chunk m = 0
        const u64 *xs = f.x + fc * f.x_c_stride + fb * f.x_b_stride + (size_t)limb * nn;  // limb slots
        const bool has_z = f.z != nullptr && ((f.z_mask >> fc) & 1u);
        const u64 *zs = has_z ? f.z + fc * f.z_c_stride + fb * f.z_b_stride + (size_t)limb * nn : nullptr;
        u64 *dp = f.dst + fc * f.dst_c_stride + fb * f.dst_b_stride + (size_t)limb * nn + ci;
        const double2 cst = f.cst[limb];
        auto load_chunk = [&](const u64 *slot, int packed, int m) -> ulonglong2 {
          return packed ? ld_packed2(slot, nn, (ci >> 1) + 16 * m) : __ldg(reinterpret_cast<const ulonglong2 *>(slot + ci + 32 * m));
        };
        ulonglong2 xv[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) xv[m] = load_chunk(xs, f.x_packed, m);
        if (f.cst2 != nullptr) {  // ((x * c + z) - y) * c2: z is mandatory, except in MODE 5
          const double2 cst2 = f.cst2[limb];
          ulonglong2 zv[8];
#pragma unroll
          for (int m = 0; m < 8; ++m) zv[m] = NOZ ? make_ulonglong2(0, 0) : load_chunk(zs, f.z_packed, m);
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const double2 y = *reinterpret_cast<const double2 *>(data + ad.C(m));
            const double u0 = mulmod_const(u64_to_f64(xv[m].x), cst.x, cst.y, q) + u64_to_f64(zv[m].x) - y.x;
            const double u1 = mulmod_const(u64_to_f64(xv[m].y), cst.x, cst.y, q) + u64_to_f64(zv[m].y) - y.y;
            const u64 v0 = f64_to_canonical(mulmod_const(u0, cst2.x, cst2.y, q), mc.qi);
            const u64 v1 = f64_to_canonical(mulmod_const(u1, cst2.x, cst2.y, q), mc.qi);
            *reinterpret_cast<ulonglong2 *>(dp + 32 * m) = make_ulonglong2(v0, v1);
          }
        } else if (has_z) {
          ulonglong2 zv[8];
          if (f.z_galois) {  // sigma(z): this row's 256 slots come from ONE source row, permuted (RowSigma)
            const RowSigma rs = row_sigma((unsigned)(tile_i * 16 + rr), f.z_galois, logN - NTT_ROW_LOG);
            const u64 *zr = zs + ((size_t)rs.src_row << NTT_ROW_LOG);
            const unsigned k0 = (l16 >> 3) * 16 + (l16 & 7) * 2;
#pragma unroll
            for (int m = 0; m < 8; ++m)
              zv[m] = make_ulonglong2(__ldg(zr + sigma_src(k0 + 32 * m, f.z_galois, rs.d)), __ldg(zr + sigma_src(k0 + 32 * m + 1, f.z_galois, rs.d)));
          } else {
#pragma unroll
            for (int m = 0; m < 8; ++m) zv[m] = load_chunk(zs, f.z_packed, m);
          }
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const double2 y = *reinterpret_cast<const double2 *>(data + ad.C(m));
            // z - h rides on the integer -> double conversion: (2^52 | z) - (2^52 + h)
            const double z0 = __longlong_as_double((long long)(zv[m].x | 0x4330000000000000ull)) - hb;
            const double z1 = __longlong_as_double((long long)(zv[m].y | 0x4330000000000000ull)) - hb;
            const double r0 = mulmod_const(u64_to_f64(xv[m].x) - y.x, cst.x, cst.y, q) + z0;
            const double r1 = mulmod_const(u64_to_f64(xv[m].y) - y.y, cst.x, cst.y, q) + z1;
            const u64 v0 = (u64)__double_as_longlong(reduce_signed(r0, q, qinv) + hb) & 0x000FFFFFFFFFFFFFull;
            const u64 v1 = (u64)__double_as_longlong(reduce_signed(r1, q, qinv) + hb) & 0x000FFFFFFFFFFFFFull;
            *reinterpret_cast<ulonglong2 *>(dp + 32 * m) = make_ulonglong2(v0, v1);
          }
        } else {
#pragma unroll
          for (int m = 0; m < 8; ++m) {
            const double2 y = *reinterpret_cast<const double2 *>(data + ad.C(m));
            const u64 v0 = f64_to_canonical(mulmod_const(u64_to_f64(xv[m].x) - y.x, cst.x, cst.y, q), mc.qi);
            const u64 v1 = f64_to_canonical(mulmod_const(u64_to_f64(xv[m].y) - y.y, cst.x, cst.y, q), mc.qi);
            *reinterpret_cast<ulonglong2 *>(dp + 32 * m) = make_ulonglong2(v0, v1);
          }
        }
      }
    } else {
      if (l.side_out != nullptr) {  // the permuted input rows as they sit in the tile, 256 B per half-warp
        u64 *so = l.side_out + (long long)cur.b * l.side_batch_stride + slot * l.out_limb_stride + tile_off + (size_t)rr * 256 + (l16 >> 3) * 16 + (l16 & 7) * 2;
#pragma unroll
        for (int m = 0; m < 8; ++m) *reinterpret_cast<ulonglong2 *>(so + 32 * m) = *reinterpret_cast<const ulonglong2 *>(data + ad.C(m));
      }
      if constexpr (MUL) {
        // in * in_mul on the chunks this lane would store (coalesced loads, 256 B per half-warp); the centred products
        // (|v| <= 0.51 q) go back into the tile as doubles
        const u64 *mp = mul_of(cur) + (size_t)rr * 256 + (l16 >> 3) * 16 + (l16 & 7) * 2;
        ulonglong2 mv[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) mv[m] = __ldg(reinterpret_cast<const ulonglong2 *>(mp + 32 * m));
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(data + ad.C(m));
          *reinterpret_cast<double2 *>(data + ad.C(m)) = make_double2(mulmod_var(u64_to_f64(v.x), u64_to_f64(mv[m].x), q, qinv),
                                                                      mulmod_var(u64_to_f64(v.y), u64_to_f64(mv[m].y), q, qinv));
        }
        __syncwarp();
      }
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        if constexpr (MUL) {
          const double2 v = *reinterpret_cast<const double2 *>(data + ad.B(m));
          a[2 * m] = v.x; a[2 * m + 1] = v.y;
        } else {
          const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(data + ad.B(m));
          a[2 * m] = u64_to_f64(v.x); a[2 * m + 1] = u64_to_f64(v.y);
        }
      }
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const double2 v = *reinterpret_cast<const double2 *>(blob + 2048 + 512 * m + 2 * tid);
        w[2 * m] = v.x; w[2 * m + 1] = v.y;
      }
      gs_level<3>(a, w, q, qinv);
      lds_run<2>(w, blob + 1024 + 2 * tid);
      { const double2 v = *reinterpret_cast<const double2 *>(blob + 1536 + 2 * tid); w[2] = v.x; w[3] = v.y; }
      gs_level<2>(a, w, q, qinv);
      lds_run<2>(w, blob + 512 + 2 * tid); gs_level<1>(a, w, q, qinv);
      w[0] = blob[256 + tid]; gs_level<0>(a, w, q, qinv);
#pragma unroll
      for (int m = 0; m < 8; ++m) *reinterpret_cast<double2 *>(data + ad.B(m)) = make_double2(a[2 * m], a[2 * m + 1]);
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 16; ++j) a[j] = *reinterpret_cast<const double *>(data + ad.A(j));
      lds_run<8>(w, tw_a + 8); gs_level<3>(a, w, q, qinv);
      lds_run<4>(w, tw_a + 4); gs_level<2>(a, w, q, qinv);
      lds_run<2>(w, tw_a + 2); gs_level<1>(a, w, q, qinv);
      lds_run<1>(w, tw_a + 1); gs_level<0>(a, w, q, qinv);
      // the sums have grown to <= 2^8 q: bring them back to |v| <= q/2 before the column pass doubles them again
      double *outd = reinterpret_cast<double *>(dst_of(cur)) + (size_t)rr * 256 + l16;
#pragma unroll
      for (int j = 0; j < 16; ++j) outd[16 * j] = reduce_signed(a[j], q, qinv);
    }
    __syncwarp();  // every lane is done with this stage before it is refilled
    if (items.valid(nn)) issue(nn, data0 + (k & 1) * ROW_TILE_BYTES);
    cp_async_commit();
    cur = nxt; nxt = nn;
  }
  cp_async_wait<0>();
}

// ================================================================================ small N (<= 4096): one CTA per limb
__global__ void __launch_bounds__(256) ntt_small(NttTables t, int logN, LimbMap lm, NttLaunch l, int inverse) {
  extern __shared__ double sm[];
  pdl_wait();
  const int limb = blockIdx.y % l.n_limbs, poly = (blockIdx.y / l.n_limbs) % l.n_polys, batch = blockIdx.y / (l.n_limbs * l.n_polys);
  if (poly == lm.skip[limb]) return;
  const int mi = lm.mod[limb];
  const ModConst mc = t.mc[mi];
  const double q = mc.q, qinv = mc.qinv;
  const double *tw = (inverse ? t.inv : t.fwd) + ((size_t)mi << logN);
  const long long slot = lm.pos[limb];
  const u64 *in = l.in + (long long)batch * l.in_batch_stride + (long long)poly * l.in_poly_stride + slot * l.in_limb_stride;
  u64 *out = l.out + (long long)batch * l.out_batch_stride + (long long)poly * l.out_poly_stride + slot * l.out_limb_stride;
  const int N = 1 << logN, half = N >> 1;
  for (int i = threadIdx.x; i < N; i += blockDim.x) sm[i] = u64_to_f64(__ldg(&in[i]));
  __syncthreads();
  if (!inverse) {
    for (int s = 0; s < logN; ++s) {
      const int tt = N >> (s + 1);
      for (int b = threadIdx.x; b < half; b += blockDim.x) {
        const int grp = b / tt, j = b % tt, i0 = grp * 2 * tt + j;
        const double w = __ldg(&tw[(1 << s) + grp]);
        double x = sm[i0], y = sm[i0 + tt];
        ct_butterfly(x, y, w, q, qinv);
        sm[i0] = x; sm[i0 + tt] = y;
      }
      __syncthreads();
    }
    for (int i = threadIdx.x; i < N; i += blockDim.x) out[i] = f64_to_canonical(reduce_signed(sm[i], q, qinv), mc.qi);
  } else {
    for (int s = logN - 1; s >= 0; --s) {
      const int tt = N >> (s + 1);
      for (int b = threadIdx.x; b < half; b += blockDim.x) {
        const int grp = b / tt, j = b % tt, i0 = grp * 2 * tt + j;
        const double w = __ldg(&tw[(1 << s) + grp]);
        double x = sm[i0], y = sm[i0 + tt];
        gs_butterfly(x, y, w, q, qinv);
        if (((logN - s) & 3) == 0) { x = reduce_signed(x, q, qinv); }  // bound the doubling every 4 stages
        sm[i0] = x; sm[i0 + tt] = y;
      }
      __syncthreads();
    }
    double2 sc;
    if (l.post_scale) sc = l.post_scale[limb];
    else sc = make_double2(mc.ninv, mc.ninv_q);
    for (int i = threadIdx.x; i < N; i += blockDim.x) out[i] = f64_to_canonical(mulmod_const(sm[i], sc.x, sc.y, q), mc.qi);
  }
}

// ================================================================================ host side
void ntt_permute_row_twiddles(const double *nat, int logN, double *out) {
  const size_t N = (size_t)1 << logN, R1 = N >> NTT_ROW_LOG;
  memset(out, 0, N * sizeof(double));
  for (size_t r = 0; r < R1; ++r) {
    double *blob = out + (r / 16) * NTT_TILE;
    const size_t rr = r % 16, base = R1 + r;
    for (int s = 0; s < 4; ++s)
      for (size_t g = 0; g < ((size_t)1 << s); ++g) blob[rr * 16 + ((size_t)1 << s) + g] = nat[(base << s) + g];
    for (size_t l = 0; l < 16; ++l) {
      const size_t ts = rr * 16 + l;
      blob[256 + ts] = nat[(base << 4) + l];
      for (size_t x = 0; x < 2; ++x) blob[512 + ts * 2 + x] = nat[(base << 5) + 2 * l + x];
      for (size_t k = 0; k < 2; ++k)
        for (size_t x = 0; x < 2; ++x) blob[1024 + k * 512 + ts * 2 + x] = nat[(base << 6) + 4 * l + 2 * k + x];
      for (size_t k = 0; k < 4; ++k)
        for (size_t x = 0; x < 2; ++x) blob[2048 + k * 512 + ts * 2 + x] = nat[(base << 7) + 8 * l + 2 * k + x];
    }
  }
}

static int sm_count() {
  static int n = [] {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    return v;
  }();
  return n;
}

template <class KERNEL>
static void allow_smem(KERNEL k, int bytes) {
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

// items of a row CTA: short CTAs keep the tail of the launch small (a CTA is dispatched whenever a slot frees up, so the
// launch ends about one CTA-time after the ideal), long CTAs amortise the 32 KB twiddle blob
constexpr int ROW_ITEMS = 8;
static int row_split(int n_items, int ctas_xy) {
  int z = (n_items + ROW_ITEMS - 1) / ROW_ITEMS;
  while (z > 1 && (long long)ctas_xy * z > 64ll * sm_count()) --z;
  return z < 1 ? 1 : z;
}

template <int LOGR1, int NT>
static void launch_cols_t(bool inverse, const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s) {
  using K = ColCfg<LOGR1, NT>;
  const int resident = K::MIN_CTAS * sm_count();
  static PerDeviceOnce once;
  if (once.first()) {
    allow_smem(ntt_fwd_cols<LOGR1, NT, false, false>, 2 * K::STAGE_BYTES);
    allow_smem(ntt_fwd_cols<LOGR1, NT, true, false>, 2 * K::STAGE_BYTES);
    allow_smem(ntt_inv_cols<LOGR1, NT, false>, 2 * K::STAGE_BYTES);
    allow_smem(ntt_fwd_cols<LOGR1, NT, false, true>, 2 * K::STAGE_BYTES);
    allow_smem(ntt_fwd_cols<LOGR1, NT, true, true>, 2 * K::STAGE_BYTES);
    allow_smem(ntt_inv_cols<LOGR1, NT, true>, 2 * K::STAGE_BYTES);
  }
  // the queue enumerates the members of the launch without the skipped ones: the limbs that skip a poly must come first
  ColQueue qu{t.col_ctr, 0, 0};
  bool dyn = t.col_ctr != nullptr;
  for (int i = 0; i < l.n_limbs; ++i) {
    const bool sk = lm.skip[i] < l.n_polys;
    if (sk && i != qu.n_skip) dyn = false;
    qu.n_skip += sk;
  }
  qu.pairs = qu.n_skip * (l.n_polys - 1) + (l.n_limbs - qu.n_skip) * l.n_polys;
  if (qu.pairs <= 0) return;
  const long long total64 = (long long)qu.pairs * l.n_batch * K::TILES;
  // (with at most two tiles per CTA there is nothing to hand out)
  const long long min_tiles = 2;
  if (dyn && total64 > min_tiles * resident && total64 <= 0x3FFFFFFF) {
    const int total = (int)total64, grid = resident;
    if (inverse) launch_pdl(ntt_inv_cols<LOGR1, NT, true>, grid, NT, 2 * K::STAGE_BYTES, s, t, logN, lm, l, total, qu);
    else if (l.in_f64) launch_pdl(ntt_fwd_cols<LOGR1, NT, true, true>, grid, NT, 2 * K::STAGE_BYTES, s, t, logN, lm, l, total, qu);
    else launch_pdl(ntt_fwd_cols<LOGR1, NT, false, true>, grid, NT, 2 * K::STAGE_BYTES, s, t, logN, lm, l, total, qu);
    return;
  }
  const int total = l.n_limbs * l.n_polys * l.n_batch * K::TILES;
  const int grid = total < resident ? total : resident;
  if (inverse) launch_pdl(ntt_inv_cols<LOGR1, NT, false>, grid, NT, 2 * K::STAGE_BYTES, s, t, logN, lm, l, total, qu);
  else if (l.in_f64) launch_pdl(ntt_fwd_cols<LOGR1, NT, true, false>, grid, NT, 2 * K::STAGE_BYTES, s, t, logN, lm, l, total, qu);
  else launch_pdl(ntt_fwd_cols<LOGR1, NT, false, false>, grid, NT, 2 * K::STAGE_BYTES, s, t, logN, lm, l, total, qu);
}

static void launch_cols(bool inverse, const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s) {
  // one ciphertext's worth of limbs is only a few 32 KB tiles per resident CTA: 16 KB tiles (128 threads, six CTAs per SM) fill
  // the machine more evenly there (measured: 55.9 vs 60.1 us for the 115-limb ModUp launch); big batches prefer 32 KB tiles
  const long long tiles32 = (long long)l.n_limbs * l.n_polys * l.n_batch << (logN - 12);
  const bool big = tiles32 >= 6ll * 3 * sm_count();
  switch (logN - NTT_ROW_LOG) {
    case 5: big ? launch_cols_t<5, 256>(inverse, t, logN, lm, l, s) : launch_cols_t<5, 128>(inverse, t, logN, lm, l, s); break;
    case 6: big ? launch_cols_t<6, 256>(inverse, t, logN, lm, l, s) : launch_cols_t<6, 128>(inverse, t, logN, lm, l, s); break;
    case 7: big ? launch_cols_t<7, 256>(inverse, t, logN, lm, l, s) : launch_cols_t<7, 128>(inverse, t, logN, lm, l, s); break;
    case 8: big ? launch_cols_t<8, 256>(inverse, t, logN, lm, l, s) : launch_cols_t<8, 128>(inverse, t, logN, lm, l, s); break;
  }
}

static void launch_rows(bool inverse, const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s) {
  static PerDeviceOnce once;
  if (once.first()) {
    allow_smem(ntt_rows<false, 0>, ROW_SMEM_BYTES);
    allow_smem(ntt_rows<false, 1>, ROW_SMEM_BYTES);
    allow_smem(ntt_rows<false, 5>, ROW_SMEM_BYTES);
    allow_smem(ntt_rows<false, 2>, ROW_SMEM_BYTES);
    allow_smem(ntt_rows<false, 3>, ROW_SMEM_BYTES);
    allow_smem(ntt_rows<true, 0>, ROW_SMEM_BYTES);
    allow_smem(ntt_rows<true, 4>, ROW_SMEM_BYTES);
  }
  const int tiles = 1 << (logN - NTT_ROW_LOG - 4);
  if (!inverse && l.mac.evk) {  // the grid splits the ciphertexts; every CTA walks all digits of its (ciphertext, limb, tile)
    const int per = std::max(1, ROW_ITEMS / std::max(1, l.n_polys));
    int z = (l.n_batch + per - 1) / per;
    while (z > 1 && (long long)tiles * l.n_limbs * z > 64ll * sm_count()) --z;
    if (l.mac.evk_packed) launch_pdl(ntt_rows<false, 3>, dim3(tiles * std::max(1, z), l.n_limbs), NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
    else launch_pdl(ntt_rows<false, 2>, dim3(tiles * std::max(1, z), l.n_limbs), NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
    return;
  }
  const dim3 grid(tiles * row_split(l.n_polys * l.n_batch, tiles * l.n_limbs), l.n_limbs);
  if (inverse && l.in_mul) launch_pdl(ntt_rows<true, 4>, grid, NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
  else if (inverse) launch_pdl(ntt_rows<true, 0>, grid, NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
  else if (l.fuse.x && l.fuse.cst2 && !l.fuse.z) launch_pdl(ntt_rows<false, 5>, grid, NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
  else if (l.fuse.x) launch_pdl(ntt_rows<false, 1>, grid, NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
  else launch_pdl(ntt_rows<false, 0>, grid, NTT_THREADS, ROW_SMEM_BYTES, s, t, logN, lm, l);
}

void launch_ntt_forward(const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s) {
  if (logN <= NTT_SMALL_LOG) {
    launch_pdl(ntt_small, dim3(1, l.n_limbs * l.n_polys * l.n_batch), 256, sizeof(double) << logN, s, t, logN, lm, l, 0);
    return;
  }
  launch_cols(false, t, logN, lm, l, s);
  launch_rows(false, t, logN, lm, l, s);
}

void launch_ntt_inverse(const NttTables &t, int logN, const LimbMap &lm, const NttLaunch &l, cudaStream_t s) {
  if (logN <= NTT_SMALL_LOG) {
    launch_pdl(ntt_small, dim3(1, l.n_limbs * l.n_polys * l.n_batch), 256, sizeof(double) << logN, s, t, logN, lm, l, 1);
    return;
  }
  launch_rows(true, t, logN, lm, l, s);
  launch_cols(true, t, logN, lm, l, s);
}

}  // namespace hml
