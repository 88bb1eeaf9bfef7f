/*
 * homulator_b200 — C ABI of the B200-native RNS-CKKS primitive datapath.
 *
 * The reference (FHE-ACCELE/Homulator) has NO plugin / FFI interface: its boundary is the CLI
 * (reference bench_test/bench_micro24.cpp:5-52) wrapping five C++ op objects
 *     OP(std::string label, uint32_t maxLevel, uint32_t currentLevel, uint32_t alpha, Config*, Arch*)
 *     bool OP::simulate()                OP in {HMULT, HROTATE, HADD, PMULT, PADD}
 * (reference include/Operation.h:200-203, 229-232, 258-261, 287-290, 316-319), whose constructors
 * decompose the op into NTT / INTT / MULT(EWE) / BCONV_STEP2 / AUTO instruction streams
 * (reference src/Operation.cpp, src/InsGen.cpp) that the rest of the reference only *times*.
 * This ABI is the boundary a maintainer would bind in their place: the same ops, executed on real
 * data on the GPU, plus the per-op instruction counts of the reference's trace.
 *
 * Conventions
 *   - plain C, no exceptions cross the boundary: every call returns an hml_status; the message for the
 *     last failure is hml_last_error(ctx) (hml_last_create_error() when no ctx exists yet).
 *   - a ctx is bound to one CUDA device and is NOT thread-safe (the reference is single-threaded and
 *     not re-entrant either: globals at reference src/Instruction.cpp:3, src/Operation.cpp:7).
 *   - all polynomial buffers are DEVICE pointers to uint64_t (reference include/Context.h:8
 *     `DataType = uint64_t`), caller-owned, layout [.. ][limb][N].  Every residue of limb i must be CANONICAL,
 *     in [0, q_i) (not merely < 2^elementBitWidth): the kernels convert words to doubles and centre them assuming it, and
 *     a word in [q_i, 2^elementBitWidth) gives undefined results.  Every output residue is canonical too.
 *     A ciphertext is [2][L][N] (c0 limbs, then c1 limbs), in EVALUATION form:
 *         slot k of limb i holds a(psi_i^(2*bitrev(k)+1)) mod q_i      (bitrev over log2 N bits)
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls are asynchronous.  The ops of one ctx share
 *     one device workspace: calls may arrive on different streams (the library orders the workspace between them with an
 *     event, i.e. ops of ONE ctx never overlap each other), but every INPUT — including the key — must already be ordered
 *     before the call on the stream it is issued to.  The *_host entry points run on internal streams and return after
 *     completion; their device-resident key must be complete (synchronise its producer) before the call.
 *   - modulus indices: 0..maxLevel-1 are q_i, maxLevel..maxLevel+alpha-1 are p_j.  The moduli are all
 *     primes = 1 (mod 2N) in (2^(w-1), 2^w), w = elementBitWidth, scanned downward from 2^w.
 *   - evaluation / rotation key layout: [beta][2][evk_q_limbs + alpha][N], Q-limbs first then the alpha
 *     P-limbs; evk_q_limbs is L (the compact per-level layout the reference allocates,
 *     reference src/Operation.cpp:300-304 `IP_Key{c}_{j}` of Level+Alpha limbs) or maxLevel.
 *     A key may also be handed over PACKED (hml_key_pack: every limb slot keeps its 8N bytes but holds N 32-bit low words
 *     followed by N high bytes, 5 of every 8 bytes are read): OR HML_KEY_PACKED into the evk_q_limbs argument of the call.
 *     One ciphertext's key switch reads its 150 MB key once, so this is worth ~4 % of a single hmult / hrotate; the limb-sharded
 *     entry points take word keys only.
 *   - there is NO CPU fallback: every compute entry point fails with HML_ERR_CUDA when no device
 *     is usable.
 */
#ifndef HOMULATOR_B200_H
#define HOMULATOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hml_ctx hml_ctx;

typedef enum {
  HML_OK = 0,
  HML_ERR_INVALID = 1,     /* bad argument (level out of range, null pointer, ...) */
  HML_ERR_CONFIG = 2,      /* config file missing / key missing (reference: uncaught runtime_error, Config.h:14-20) */
  HML_ERR_CUDA = 3,        /* CUDA runtime failure, or no device */
  HML_ERR_UNSUPPORTED = 4, /* parameter outside what the kernels implement */
  HML_ERR_OP = 5           /* unknown operation name (reference: bench_micro24.cpp:49-51) */
} hml_status;

/* ------------------------------------------------------------------ context
 * Replaces `new Config(path)` + `new Arch(config)` (reference bench_micro24.cpp:16-27).  Reads N,
 * elementBitWidth, batchSize, bconv_num_high/width from the .cfg (format of reference src/Config.cpp:16-37);
 * every other key is accepted and ignored.  maxLevel and alpha are CLI arguments in the reference. */
int hml_ctx_create(const char *cfg_path, uint32_t max_level, uint32_t alpha, int device, hml_ctx **out);
int hml_ctx_create_params(uint32_t N, uint32_t element_bit_width, uint32_t batch_size, uint32_t max_level,
                          uint32_t alpha, int device, hml_ctx **out);
void hml_ctx_destroy(hml_ctx *ctx);
const char *hml_last_error(const hml_ctx *ctx);
const char *hml_last_create_error(void);

uint32_t hml_ring_degree(const hml_ctx *ctx);
uint32_t hml_n_moduli(const hml_ctx *ctx);
int hml_get_moduli(const hml_ctx *ctx, uint64_t *out, uint32_t cap); /* q_0.., then p_0.. */
int hml_get_roots(const hml_ctx *ctx, uint64_t *out, uint32_t cap);  /* psi per modulus */

/* device-memory helpers so a host without the CUDA runtime (cgo / JNI / ctypes) can drive the library */
int hml_dev_alloc(hml_ctx *ctx, uint64_t n_words, uint64_t **out);
int hml_dev_free(hml_ctx *ctx, uint64_t *ptr);
int hml_h2d(hml_ctx *ctx, uint64_t *dst_dev, const uint64_t *src_host, uint64_t n_words, void *stream);
int hml_d2h(hml_ctx *ctx, uint64_t *dst_host, const uint64_t *src_dev, uint64_t n_words, void *stream);
int hml_sync(hml_ctx *ctx, void *stream);
/* words [n_limbs][N] -> packed limbs [n_limbs][N-word slots] (device to device, out must not overlap in); for evaluation /
 * rotation keys: n_limbs = beta * 2 * (evk_q_limbs + alpha).  See HML_KEY_PACKED above. */
#define HML_KEY_PACKED 0x80000000u
int hml_key_pack(hml_ctx *ctx, const uint64_t *words_dev, uint64_t n_limbs, uint64_t *packed_dev, void *stream);

/* ------------------------------------------------------------------ primitives
 * One entry point per instruction class of the reference (reference include/Instruction.h:6-20; only
 * NTT, INTT, MULT, BCONV_STEP2, AUTO are ever generated).  Each call processes n_limbs whole limbs
 * (= n_limbs * N/batchSize reference instructions). mod_idx is a HOST array of n_limbs modulus indices. */

/* replaces InsGen::GenNTT(ntt=true/false)  (reference src/InsGen.cpp:17-44).  in == out allowed. */
int hml_ntt(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs, void *stream);
int hml_intt(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs, void *stream);
/* The same transforms for n_batch polynomials that share one limb list: in / out are [n_batch][n_limbs][N].  This is the
 * shape the batched ops launch (reference batchCount, src/InsGen.cpp:12): one kernel pair for the whole batch, the per-limb
 * twiddles staged once per CTA and reused by every polynomial.  n_limbs <= 128. */
int hml_ntt_batch(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs, uint32_t n_batch,
                  void *stream);
int hml_intt_batch(hml_ctx *ctx, const uint64_t *in, uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs, uint32_t n_batch,
                   void *stream);

/* replaces InsGen::GenEWE (reference src/InsGen.cpp:77-125): out = x1*x2 (+|-) x3*x4 mod m per limb.
 * NULL x2/x4: multiplier 1.  NULL x1/x3: that product is absent (the reference's "address 0",
 * src/mem.cpp:30).  Each operand is [n_limbs][N]. */
int hml_ewe(hml_ctx *ctx, const uint64_t *x1, const uint64_t *x2, const uint64_t *x3, const uint64_t *x4, int subtract,
            uint64_t *out, const uint32_t *mod_idx, uint32_t n_limbs, void *stream);

/* replaces InsGen::GenAUTO (reference src/InsGen.cpp:46-71): out[k] = in[k'],
 * 2*bitrev(k')+1 = galois_elt*(2*bitrev(k)+1) mod 2N, on n_limbs evaluation-form limbs. in != out. */
int hml_automorph(hml_ctx *ctx, const uint64_t *in, uint64_t *out, uint64_t galois_elt, uint32_t n_limbs, void *stream);

/* replaces BConv step 1 (a MULT in the reference, src/Operation.cpp:104-135, :447-487) + step 2
 * (InsGen::GenBCONV, src/InsGen.cpp:263-313): in [n_src][N] coefficient form over moduli src_idx,
 * out [n_dst][N]: out_m = sum_i [in_i * (D/s_i)^-1]_{s_i} * [D/s_i]_m mod m, no overflow correction. */
int hml_bconv(hml_ctx *ctx, const uint64_t *in, const uint32_t *src_idx, uint32_t n_src, uint64_t *out,
              const uint32_t *dst_idx, uint32_t n_dst, void *stream);
/* The same conversion for n_batch independent polynomials: in [n_batch][n_src][N], out [n_batch][n_dst][N], ONE launch (the
 * shape the batched ops use).  Conversions with <= 48 sources and <= 48 targets on rings with N >= 128 run on the 5th-gen
 * tensor cores (tcgen05.mma kind::i8, accumulators in TMEM; homulator_b200/csrc/bconv_umma.cu), the rest on the FP64
 * tensor-core path; HML_BCONV_UMMA=0 forces the latter. */
int hml_bconv_batch(hml_ctx *ctx, const uint64_t *in, const uint32_t *src_idx, uint32_t n_src, uint64_t *out,
                    const uint32_t *dst_idx, uint32_t n_dst, uint32_t n_batch, void *stream);

/* ------------------------------------------------------------------ sub-operations */
/* replaces KeySwitch::KeySwitch (reference src/Operation.cpp:9-54, stages :63-590).
 * d [L][N] -> out0,out1 [L][N]. */
int hml_keyswitch(hml_ctx *ctx, uint32_t L, const uint64_t *d, const uint64_t *evk, uint32_t evk_q_limbs,
                  uint64_t *out0, uint64_t *out1, void *stream);
/* replaces Rescale::Rescale (reference src/Operation.cpp:741-911): in [L][N] -> out [L-1][N]. */
int hml_rescale(hml_ctx *ctx, uint32_t L, const uint64_t *in, uint64_t *out, void *stream);

/* Limb-sharded key switch over `world` GPUs of one node (BASELINE.json configs[4], SURVEY.md 8e mode 2).
 * Extended limb e (Q-limbs 0..L-1, then P-limbs) is owned by rank e % world — the rule the reference uses to map
 * limbs to clusters (reference include/Driver.h:158,:178).  Every stage is limb-local except base conversion, so the
 * caller performs one all-gather before each conversion (NCCL, same stream), between the three calls below; this is
 * the GPU counterpart of the reference's inter-cluster NoC fetch (reference include/mem.h:612-621).
 *   d_own    [n_own_q][N]              the owned Q-limbs of the input, ascending limb index
 *   evk_own  [beta][2][n_own_e][N]     key slices for the owned extended limbs (owned Q-limbs, then owned P-limbs)
 *   gather1  [world][gather1_slots][N] begin() fills slot `rank`; the caller all-gathers it in place
 *   gather2  [world][2][gather2_slots][N] mid() fills slot `rank`; the caller all-gathers it in place
 *   out*_own [n_own_q][N]              the owned Q-limbs of the two outputs
 * hml_shard_layout reports ownership and slot numbers (pure host code). */
#define HML_MAX_SHARD_LIMBS 128
typedef struct {
  uint32_t gather1_slots, gather2_slots;   /* ceil(L/world), ceil(alpha/world) */
  uint32_t n_own_q, n_own_p;
  uint32_t own_q[HML_MAX_SHARD_LIMBS];     /* owned Q-limb indices */
  uint32_t own_p[HML_MAX_SHARD_LIMBS];     /* owned P-limb indices j (extended limb L + j) */
  uint32_t owner[HML_MAX_SHARD_LIMBS];     /* owner rank of every extended limb */
  uint32_t slot[HML_MAX_SHARD_LIMBS];      /* slot of extended limb e inside its owner's gather contribution */
} hml_shard_info;
int hml_shard_layout(uint32_t L, uint32_t alpha, uint32_t rank, uint32_t world, hml_shard_info *out);
int hml_keyswitch_shard_begin(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *d_own,
                              uint64_t *gather1, void *stream);
int hml_keyswitch_shard_mid(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *d_own,
                            const uint64_t *gather1, const uint64_t *evk_own, uint64_t *gather2, void *stream);
int hml_keyswitch_shard_end(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *gather2,
                            uint64_t *out0_own, uint64_t *out1_own, void *stream);

/* Peer-direct variant of the same three phases: NO collective.  Every rank keeps its contribution in its own gather
 * buffers; the base conversions of the other ranks read the source limbs straight out of the owners' memory over NVLink
 * while they compute (the all-gather is fused into the consumer kernel's tile loop, homulator_b200/csrc/bconv_umma.cu).
 *   peers1[r] / peers2[r]   rank r's gather buffer 1 / 2 as a pointer valid on THIS device: the rank's own allocation for
 *                           r == rank, a cudaIpcOpenMemHandle / peer-enabled mapping otherwise (HOST arrays of `world` pointers)
 *   flags                   per rank 3 * world zero-initialised words: [r] = epoch up to which rank r's buffer 1 is ready,
 *                           [world + r] = the same for buffer 2, [2 world + r] = the sharded rescale's exchange
 * Sequence per key switch (epoch = 1, 2, ... per call): shard_begin(own buffer 1) -> shard_signal(slot rank) ->
 * shard_wait(base 0) -> shard_mid_p2p -> shard_signal(slot world + rank) -> shard_wait(base world) -> shard_end_p2p.
 * hml_shard_signal writes `epoch` into flags[slot] of EVERY peer (peer_flags_dev = DEVICE array of `world` pointers);
 * hml_shard_wait spins on the device until flags[base + r] >= epoch for all r (traps after ~2 s).  hml_ipc_export / import
 * wrap cudaIpcGetMemHandle / cudaIpcOpenMemHandle for buffers obtained from hml_dev_alloc, so a host without the CUDA
 * runtime can exchange them between the per-GPU processes. */
int hml_keyswitch_shard_mid_p2p(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *d_own,
                                const uint64_t *const *peers1, const uint64_t *evk_own, uint64_t *gather2_own, void *stream);
int hml_keyswitch_shard_end_p2p(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *const *peers2,
                                uint64_t *out0_own, uint64_t *out1_own, void *stream);
int hml_shard_signal(hml_ctx *ctx, uint64_t *const *peer_flags_dev, uint32_t slot, uint64_t epoch, uint32_t world, void *stream);
int hml_shard_wait(hml_ctx *ctx, const uint64_t *flags, uint32_t base, uint64_t epoch, uint32_t world, void *stream);
/* signal followed by wait in ONE launch (one rank per GPU only: ranks emulated on a single stream need the separate calls).
 * epoch == 0: use and advance this rank's device-side counter of the exchange group (word 3 * world + base / world of its
 * flag block, which then needs 3 * world + 3 words) — no host state, so a captured CUDA graph of a whole op sequence replays. */
int hml_shard_sync(hml_ctx *ctx, uint64_t *const *peer_flags_dev, uint32_t slot, uint64_t *flags, uint32_t base,
                   uint64_t epoch, uint32_t world, void *stream);
/* Sharded rescale of a limb-sharded ciphertext (reference Rescale, src/Operation.cpp:741-911): x_own [2][nq][N] = the two
 * polynomials' owned Q-limbs at level L (ascending); the owner of limb L-1 writes its coefficient form to r_own [2][N]
 * (begin); after one flag exchange (third slot group of the flag block, base 2 * world) every rank reads r_src = the OWNER's
 * buffer (own or peer mapping) and produces out_own [2][nq'][N], nq' = owned limbs below L-1 (end). */
int hml_rescale_shard_begin(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *x_own, uint64_t *r_own, void *stream);
int hml_rescale_shard_end(hml_ctx *ctx, uint32_t L, uint32_t rank, uint32_t world, const uint64_t *x_own, const uint64_t *r_src,
                          uint64_t *out_own, void *stream);
/* hml_shard_wait / hml_shard_sync never trap: a wait that exceeds HML_SHARD_TIMEOUT_MS (default 20000) sets the status word
 * (word 3 * world + 4 of the rank's flag block, which therefore needs 3 * world + 8 words) and returns; hml_shard_status
 * synchronises `stream` and reports it as HML_ERR_CUDA. */
int hml_shard_status(hml_ctx *ctx, const uint64_t *flags, uint32_t world, void *stream);
int hml_ipc_export(hml_ctx *ctx, const uint64_t *dev_ptr, unsigned char handle[64]);
int hml_ipc_import(hml_ctx *ctx, const unsigned char handle[64], uint64_t **out);
int hml_ipc_close(hml_ctx *ctx, uint64_t *ptr);

/* ------------------------------------------------------------------ limb-sharded OPERATIONS (one call per op and rank)
 * An hml_shard is one rank's view of a limb-shard group: its peer-visible buffers (two gather buffers sized for levels up to
 * max_L, a rescale buffer, a flag block), the mappings of every peer's, and the scratch of the composite ops.  The whole op —
 * limb-local phases, the exchanges between them (one launch each: release this rank's epoch to every peer, acquire-spin on
 * theirs; epochs live in device memory, so a captured CUDA graph replays), the base conversions reading the peers' limbs
 * over NVLink — is composed inside the library (homulator_b200/csrc/shard.cu); this replaces the reference's limb -> cluster
 * mapping and NoC (reference include/Driver.h:155-246, include/mem.h:612-621).
 * Group set-up, (a) one process per GPU: hml_shard_create -> hml_shard_handles (4 cudaIpc handles) -> exchange them by any
 * means -> hml_shard_connect_ipc(all ranks' handles, [world][4][64] bytes); (b) one process driving several devices (one ctx
 * per device): hml_shard_create for every rank -> hml_shard_connect_local(group).  hml_shard_prepare(L) builds every table
 * and sizes the workspace for level L ahead of the first exchange (call it on all ranks before a barrier).
 * Sharded layouts: a polynomial = this rank's Q-limbs [nq][N] (limb i on rank i % world, ascending), a ciphertext [2][nq][N],
 * a key [beta][2][n_own_ext][N] (owned Q-limbs, then owned P-limbs); hmult / rescale outputs hold the owned limbs below L-1.
 * Every rank of the group must issue the same sequence of sharded calls. */
typedef struct hml_shard hml_shard;
int hml_shard_create(hml_ctx *ctx, uint32_t max_L, uint32_t rank, uint32_t world, hml_shard **out);
/* The same with room for max_rot (1..16) hoisted rotations per exchange (hml_hrotate_hoisted_sharded): gather buffer 2 holds
 * max_rot slots of the key switch's size, back to back (about 2 * alpha * N * 8 bytes per slot and rank), and
 * hml_shard_prepare sizes the workspace for max_rot rotations.  hml_shard_create is max_rot = 1.  Every rank of a group must
 * use the same max_rot (the slots are addressed at the same offsets in every rank's buffer): hml_shard_connect_local rejects
 * mixed values; IPC groups must agree on it before they exchange handles. */
int hml_shard_create_ex(hml_ctx *ctx, uint32_t max_L, uint32_t rank, uint32_t world, uint32_t max_rot, hml_shard **out);
int hml_shard_destroy(hml_shard *sh);
int hml_shard_handles(hml_shard *sh, unsigned char *out_4x64);
int hml_shard_connect_ipc(hml_shard *sh, const unsigned char *handles_world_4x64);
int hml_shard_connect_local(hml_shard *const *group, uint32_t world);
int hml_shard_prepare(hml_shard *sh, uint32_t L);
int hml_shard_check(hml_shard *sh, void *stream);   /* synchronises; HML_ERR_CUDA if an exchange of this rank timed out */
int hml_shard_own_limbs(const hml_shard *sh, uint32_t L, uint32_t *n_own_q, uint32_t *n_own_q_after_rescale);
/* KeySwitch / HROTATE / HMULT / Rescale on sharded operands (reference src/Operation.cpp:9-54, :1271-1358, :913-1023, :741-911) */
int hml_keyswitch_sharded(hml_shard *sh, uint32_t L, const uint64_t *d_own, const uint64_t *evk_own, uint64_t *out0_own,
                          uint64_t *out1_own, void *stream);
int hml_hrotate_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, const uint64_t *rotkey_own, uint64_t galois_elt,
                        uint64_t *out_own, void *stream);
int hml_hmult_sharded(hml_shard *sh, uint32_t L, const uint64_t *a_own, const uint64_t *b_own, const uint64_t *evk_own,
                      uint64_t *out_own, void *stream);
int hml_rescale_sharded(hml_shard *sh, uint32_t L, const uint64_t *x_own, uint64_t *out_own, void *stream);
/* HADD (kind 0, b = ciphertext), PMULT (1), PADD (2) (b = plaintext [nq][N]), PMULT + HADD in one pass (3: out = a * b + out)
 * on the owned limbs: no exchange */
int hml_ew_sharded(hml_shard *sh, uint32_t L, int kind, const uint64_t *a_own, const uint64_t *b_own, uint64_t *out_own, void *stream);
/* All ranks of a group driven by ONE host thread, phase by phase (the CLI's [cluster] argument; tests on a one-GPU box).
 * op_kind: 0 keyswitch (a = d_own, out0, out1), 1 hrotate (a = ct_own, out0), 2 hmult (a, b, out0), 3 rescale (a, out0); every
 * array is indexed by rank.  Ranks that share a device must share one stream: they are ordered by that stream and exchange
 * with separate signal / wait launches, so no kernel ever spins on a flag a not-yet-launched kernel has to write. */
int hml_group_op(hml_shard *const *group, uint32_t world, int op_kind, uint32_t L, const uint64_t *const *a, const uint64_t *const *b,
                 const uint64_t *const *key, uint64_t *const *out0, uint64_t *const *out1, uint64_t galois_elt, void *const *streams);
/* Hoisted rotations of ONE limb-sharded ciphertext (one call per rank, like hml_hrotate_sharded): ct_own [2][nq][N] ->
 * outs_own[r] [2][nq][N] = (sigma_r(c0) + ks0, ks1) on the owned limbs, bit-identical to the owned rows of hml_hrotate_hoisted.
 * One ModUp of c1 and its two exchanges serve all n_rot rotations; groups of up to max_rot rotations (hml_shard_create_ex)
 * share one inner-product launch, one P-limb INTT and one exchange.  rotkeys_own / galois_elts / outs_own are HOST arrays of
 * n_rot entries (owned key slices, word keys); a key may be null on a rank that owns no extended limb.  n_rot = 0 is a no-op;
 * no output may alias the input. */
int hml_hrotate_hoisted_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, uint32_t n_rot, const uint64_t *const *rotkeys_own,
                                const uint64_t *galois_elts, uint64_t *const *outs_own, void *stream);
/* The same for all ranks of a local group from one host thread (as hml_group_op): ct_own and streams are indexed by rank,
 * rotkeys_own and outs_own rank-major ([rank * n_rot + i]). */
int hml_group_hrotate_hoisted(hml_shard *const *group, uint32_t world, uint32_t L, const uint64_t *const *ct_own, uint32_t n_rot,
                              const uint64_t *const *rotkeys_own, const uint64_t *galois_elts, uint64_t *const *outs_own,
                              void *const *streams);
/* Double-hoisted rotation sum of ONE limb-sharded ciphertext (one call per rank): out_own [2][nq][N] =
 * sum_i pts_own[i] * rotate(ct_own, galois_elts[i]) on the owned limbs, bit-identical to the owned rows of
 * hml_hrotate_sum_hoisted (same formula: acc_c = sum_i pt_i * sum_j sigma_i(t_j) * rk_i[j][c] over the owned extended limbs,
 * z = sum_i pt_i * sigma_i(c0) over the owned Q-limbs, out = (z + ModDown(acc_0), ModDown(acc_1))).
 *   begin(c1) | X0 | ModUp + NTT of the owned digits, one inner-product launch per group of 16 rotations, P-limb INTT | X1 |
 *   one ModDown with addend z
 * Two exchanges per call whatever n_rot and max_rot; no slot of gather buffer 2 beyond the first is used.  ct_own, out_own
 * [2][nq][N], not overlapping.  rotkeys_own / galois_elts / pts_own are HOST arrays of n_rot entries: word key slices
 * [beta][2][n_own_ext][N] (no HML_KEY_PACKED) and plaintext slices [nq + np][N] holding the rank's owned rows of the extended
 * basis (owned Q-limbs, then owned P-limbs, as the key slices).  A rank that owns no extended limb may pass null keys and
 * plaintexts; a rank that owns only P-limbs needs both.  HML_ERR_INVALID (before anything is enqueued): n_rot = 0, a null
 * ct / output / galois array, a null key or plaintext on a rank that owns extended limbs, an even galois element, out_own
 * overlapping ct_own, L above the shard's maximum.  Executed counts per rank: the transforms and conversions of one
 * hml_hrotate_hoisted_sharded rotation whatever n_rot; one kernel launch per group of 16 rotations; per rotation
 * ewe_limbs += 2 * beta * ne + 2 * ne + nq and automorph_limbs += nq (ne = owned extended limbs).  After hml_shard_prepare(L) the
 * call neither allocates nor synchronises (it can be captured in a CUDA graph). */
int hml_hrotate_sum_hoisted_sharded(hml_shard *sh, uint32_t L, const uint64_t *ct_own, uint32_t n_rot, const uint64_t *const *rotkeys_own,
                                    const uint64_t *galois_elts, const uint64_t *const *pts_own, uint64_t *out_own, void *stream);
/* The same for all ranks of a local group from one host thread (as hml_group_op): ct_own, out_own and streams are indexed by
 * rank, rotkeys_own and pts_own rank-major ([rank * n_rot + i]). */
int hml_group_hrotate_sum_hoisted(hml_shard *const *group, uint32_t world, uint32_t L, const uint64_t *const *ct_own, uint32_t n_rot,
                                  const uint64_t *const *rotkeys_own, const uint64_t *galois_elts, const uint64_t *const *pts_own,
                                  uint64_t *const *out_own, void *const *streams);
/* Sum of ciphertext products on limb-sharded operands (one call per rank, one output): out_own [2][nk][N] =
 * Rescale(Relin(sum_i a_own[i] (x) b_own[i])) on the owned limbs below L-1 (nk from hml_shard_own_limbs), bit-identical to the
 * owned rows of hml_hmult_sum with n_out = 1; with n_terms = 1 it is hml_hmult_sharded.  The phases of hml_hmult_sharded,
 * whose tensor product becomes the sums D0 / D1 / D2 of the n_terms tensor products on the owned limbs (one launch per group of
 * 16 terms); the key switch, the exchanges and the rescale run once.  a_own / b_own are HOST arrays of n_terms device pointers
 * to [2][nq][N]; a_own[i] == b_own[i] is a square and reads its ciphertext once.  evk_own [beta][2][n_own_ext][N] (word key;
 * may be null on a rank that owns no extended limb).  HML_ERR_INVALID (before anything is enqueued): n_terms = 0, L < 2, L above
 * the shard's maximum, a null array, entry or output, a null key on a rank that owns extended limbs, out_own overlapping an
 * input.  Executed counts per rank: the transforms and conversions of hml_hmult_sharded whatever n_terms; ewe_limbs += 3 * nq
 * per term.  After hml_shard_prepare(L) the call neither allocates nor synchronises (it can be captured in a CUDA graph). */
int hml_hmult_sum_sharded(hml_shard *sh, uint32_t L, uint32_t n_terms, const uint64_t *const *a_own, const uint64_t *const *b_own,
                          const uint64_t *evk_own, uint64_t *out_own, void *stream);
/* The same for all ranks of a local group from one host thread: evk_own, out_own and streams are indexed by rank, a_own and
 * b_own rank-major ([rank * n_terms + i]). */
int hml_group_hmult_sum(hml_shard *const *group, uint32_t world, uint32_t L, uint32_t n_terms, const uint64_t *const *a_own,
                        const uint64_t *const *b_own, const uint64_t *const *evk_own, uint64_t *const *out_own, void *const *streams);

/* ------------------------------------------------------------------ operations (reference include/Operation.h) */
/* HMULT (reference src/Operation.cpp:913-1023): tensor + keyswitch(relinearise) + add + rescale x2.
 * ct_a, ct_b [2][L][N]; ct_out [2][L-1][N].  Requires L >= 2 (the reference segfaults at L=1). */
int hml_hmult(hml_ctx *ctx, uint32_t L, const uint64_t *ct_a, const uint64_t *ct_b, const uint64_t *evk,
              uint32_t evk_q_limbs, uint64_t *ct_out, void *stream);
/* HROTATE (reference src/Operation.cpp:1271-1358): automorphism of both polys + keyswitch + add.
 * The reference takes no rotation amount; galois_elt is the one addition (5^r mod 2N; r=1 -> 5).
 * ct [2][L][N] -> ct_out [2][L][N] = (sigma(c0) + ks0, ks1), ks = KeySwitch(sigma(c1)).  ct_out may be ct (in place).
 * The AUTO instruction class (reference InsGen::GenAUTO, src/InsGen.cpp:46-71) is executed inside the key switch's loads on
 * rings with N >= 8192 (in evaluation order the automorphism maps every 256-slot row onto one source row), by a kernel of its
 * own otherwise; the executed counts report the 2L limbs either way. */
int hml_hrotate(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *rotkey, uint32_t evk_q_limbs,
                uint64_t galois_elt, uint64_t *ct_out, void *stream);
/* Hoisted rotations (SURVEY.md 8f rank 3): n_rot rotations of ONE ciphertext share one ModUp of c1; the automorphism is
 * applied to the extended digits as the inner product loads them.  out_r = (sigma_r(c0) + ks0, ks1).  A different function
 * from hml_hrotate bit for bit (the approximate base conversion is not equivariant under the automorphism) and an equally
 * valid rotation; pinned by its own oracle definition (oracle/oracle.c orc_hrotate_hoisted).  rotkeys / galois_elts /
 * ct_outs are HOST arrays of n_rot entries; no output may alias the input. */
int hml_hrotate_hoisted(hml_ctx *ctx, uint32_t L, const uint64_t *ct, uint32_t n_rot, const uint64_t *const *rotkeys,
                        uint32_t evk_q_limbs, const uint64_t *galois_elts, uint64_t *const *ct_outs, void *stream);
/* Double-hoisted rotation sum (Bossuat et al., Eurocrypt 2021): ct_out = sum_i pts[i] * rotate(ct, galois_elts[i]) with ONE
 * ModUp of c1 and ONE ModDown.  With t = ModUp(c1) and E = (q_0..q_{L-1}, p_0..p_{alpha-1}):
 *   acc_c[m] = sum_i pt_i[m] * sum_j sigma_i(t_j)[m] * rotkeys[i][j][c][m]     (m in E, c = 0, 1)
 *   z[l]     = sum_i pt_i[l] * sigma_i(c0)[l]                                  (l < L)
 *   ct_out   = (z + ModDown(acc_0), ModDown(acc_1))
 * sigma_i is applied to every digit limb, as in hml_hrotate_hoisted; galois element 1 is the identity (with a key).  With
 * n_rot = 1 and pt = 1 on every limb of E the result is hml_hrotate_hoisted's bit for bit.  In general it is NOT
 * sum_i pt_i * hml_hrotate_hoisted_i bit for bit (ModDown of a sum differs from the sum of ModDowns through the approximate base
 * conversion) and an equally valid result, pinned by its own oracle definition (tests/orc_rotsum.py).
 * ct, ct_out [2][L][N], not overlapping.  rotkeys / galois_elts / pts are HOST arrays of n_rot entries; pts[i] is
 * [pt_q_limbs + alpha][N] in the key's convention (Q-limbs first, P-limb j at row pt_q_limbs + j), so a plaintext laid out for
 * a higher level serves every level from L up to pt_q_limbs.  evk_q_limbs and pt_q_limbs lie in [L, maxLevel] (keys may be
 * packed: HML_KEY_PACKED).  HML_ERR_INVALID: n_rot = 0, a null key / plaintext / output, an even galois element, overlapping
 * ct / ct_out, limbs out of range; HML_ERR_UNSUPPORTED: more than 8 digits.
 * Executed counts: per call the key switch's ModUp, the P-limb INTT of both accumulators and one ModDown (as hml_keyswitch),
 * and one kernel launch per group of 16 rotations; per rotation ewe_limbs += 2 * beta * E + 2 * E + L and
 * automorph_limbs += L (the automorphism rides on the loads).  No transform or conversion grows with n_rot. */
int hml_hrotate_sum_hoisted(hml_ctx *ctx, uint32_t L, const uint64_t *ct, uint32_t n_rot, const uint64_t *const *rotkeys,
                            uint32_t evk_q_limbs, const uint64_t *galois_elts, const uint64_t *const *pts, uint32_t pt_q_limbs,
                            uint64_t *ct_out, void *stream);
/* Double-hoisted baby-step / giant-step linear transform (Bossuat et al., Eurocrypt 2021), the form of CoeffToSlot /
 * SlotToCoeff and of any plaintext-matrix x encrypted-vector product:
 *   ct_out = sum_j rotate( sum_i pts[j * n1 + i] * rotate(ct, baby_galois[i]), giant_galois[j] )     i < n1, j < n2
 * with ONE ModUp of c1 for every baby step, one ModUp per non-identity giant step and ONE final ModDown.  With
 * IP_g(c) = sum_d sigma_g(ModUp(c)_d) * rk_g[d], a pair of accumulators over E = (q_0..q_{L-1}, p_0..p_{alpha-1}):
 *   1. per giant step j:  acc_j = sum_{b_i != 1} pt_{j,i} * IP_{b_i}(c1),  z0_j = sum_i pt_{j,i} * sigma_{b_i}(c0),
 *                         z1_j  = sum_{b_i = 1} pt_{j,i} * c1
 *   2. per G_j != 1:      ct_j  = (ModDown(acc_j, 0) + z0_j, ModDown(acc_j, 1) + z1_j)
 *   3. A  = sum_{G_j = 1} acc_j + sum_{G_j != 1} IP_{G_j}(ct_j.c1),   Z0 = sum_{G_j = 1} z0_j + sum_{G_j != 1} sigma_{G_j}(ct_j.c0),
 *      Z1 = sum_{G_j = 1} z1_j
 *   4. ct_out = (ModDown(A, 0) + Z0, ModDown(A, 1) + Z1)
 * Identity elements (g = 1 mod 2N) pay no key switch and their key entry may be NULL; every other element needs its rotation
 * key.  Keys follow hml_hrotate_sum_hoisted: one layout for all (evk_q_limbs, optionally | HML_KEY_PACKED).  pts[j * n1 + i]
 * (j-major) is [pt_q_limbs + alpha][N], P-limb m at row pt_q_limbs + m.  With n2 = 1, G_0 = 1 and no identity baby step the
 * result is hml_hrotate_sum_hoisted's bit for bit.  The oracle defines the op (tests/orc_bsgs.py).
 * ct, ct_out [2][L][N], not overlapping.  The key, galois and plaintext arrays are HOST arrays.  HML_ERR_INVALID: n1 = 0 or
 * n2 = 0, a null ct / ct_out / galois array / plaintext, a null key for a non-identity element, an even galois element,
 * overlapping ct / ct_out, evk_q_limbs or pt_q_limbs outside [L, maxLevel]; HML_ERR_UNSUPPORTED: more than 8 digits.
 * Executed counts: with k non-identity giant steps, the transforms and conversions of (k + 1) hml_hrotate_sum_hoisted calls
 * of one rotation, whatever n1; one kernel launch per group of 16 baby steps of every giant step and one per non-identity
 * giant step.  After the workspace exists the call neither allocates nor synchronises (it can be captured in a CUDA graph). */
int hml_hrotate_bsgs_hoisted(hml_ctx *ctx, uint32_t L, const uint64_t *ct, uint32_t n1, const uint64_t *baby_galois,
                             const uint64_t *const *baby_keys, uint32_t n2, const uint64_t *giant_galois, const uint64_t *const *giant_keys,
                             uint32_t evk_q_limbs, const uint64_t *const *pts, uint32_t pt_q_limbs, uint64_t *ct_out, void *stream);
/* HADD / PMULT / PADD (reference src/Operation.cpp:1114-1176, :1453-1523, :1618-1680).  pt is [L][N].
 * PADD adds the plaintext to BOTH components, as the reference's trace does (:1650-1672). */
int hml_hadd(hml_ctx *ctx, uint32_t L, const uint64_t *ct_a, const uint64_t *ct_b, uint64_t *ct_out, void *stream);
int hml_pmult(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *pt, uint64_t *ct_out, void *stream);
int hml_padd(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *pt, uint64_t *ct_out, void *stream);
/* ct_out = ct * pt + ct_add: PMULT followed by HADD as one element-wise pass (the reference's MULT instruction is natively
 * x1 * x2 + x3 * x4, src/InsGen.cpp:77-125); bit-identical to the two calls.  ct_out may alias ct_add.  hml_replay_* uses it
 * for "t = a * pt; d = d + t" pairs whose t is dead afterwards. */
int hml_pmult_add(hml_ctx *ctx, uint32_t L, const uint64_t *ct, const uint64_t *pt, const uint64_t *ct_add, uint64_t *ct_out, void *stream);

/* Batched, data-parallel over independent ciphertexts sharing one key (BASELINE.json configs[3]).
 * ct_a, ct_b [n][2][L][N]; ct_out [n][2][L-1][N] (hmult) / [n][2][L][N] (hrotate). */
int hml_hmult_batch(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct_a, const uint64_t *ct_b,
                    const uint64_t *evk, uint32_t evk_q_limbs, uint64_t *ct_out, void *stream);
/* out_k = Rescale(Relin(sum_i cts_a[i][k] (x) cts_b[i][k])), k < n_out: one key switch and one rescale per output.
 * Sums of ciphertext products (dot products, sums of squares, the inner sums of polynomial evaluation) with lazy
 * relinearisation: for each output k, over the Q-limbs l < L,
 *   D0 = sum_i a_i0 * b_i0,   D1 = sum_i (a_i0 * b_i1 + a_i1 * b_i0),   D2 = sum_i a_i1 * b_i1      (mod q_l)
 *   out_k = Rescale( D0 + KS0(D2), D1 + KS1(D2) )                                                    [2][L-1][N]
 * with the hybrid key switch and the rescale hml_hmult runs after its tensor product.  n_terms = 1 is hml_hmult (n_out = 1) and
 * hml_hmult_batch (n_out > 1) bit for bit.  For n_terms >= 2 it is NOT sum_i hml_hmult(a_i, b_i) bit for bit (the approximate
 * ModUp conversion of a sum differs from the sum of the conversions, and the rescale's lift is not additive) and an equally
 * valid result, decrypting to sum_i m_ai * m_bi / q_{L-1} within the noise; the oracle defines the op (tests/orc_hmult_sum.py).
 * cts_a / cts_b are HOST arrays of n_terms device pointers, each to [n_out][2][L][N]; a term with cts_a[i] == cts_b[i] is a
 * square and reads its ciphertext once.  ct_out [n_out][2][L-1][N] overlaps no input.  evk as in hml_hmult (evk_q_limbs in
 * [L, maxLevel], optionally | HML_KEY_PACKED).  n_out = 0 is a no-op.  HML_ERR_INVALID: L < 2, n_terms = 0, a null array,
 * entry, key or output, ct_out overlapping an input, evk_q_limbs out of range; HML_ERR_UNSUPPORTED: more than 8 digits.
 * Executed counts: the transforms and conversions of hml_hmult (n_out = 1) or hml_hmult_batch (n_out > 1) whatever n_terms;
 * ewe_limbs += 3L per term and output, and one kernel launch per group of 16 terms and chunk of outputs.  After the workspace
 * exists the call neither allocates nor synchronises (it can be captured in a CUDA graph). */
int hml_hmult_sum(hml_ctx *ctx, uint32_t L, uint32_t n_terms, const uint64_t *const *cts_a, const uint64_t *const *cts_b,
                  uint32_t n_out, const uint64_t *evk, uint32_t evk_q_limbs, uint64_t *ct_out, void *stream);
int hml_hrotate_batch(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct, const uint64_t *rotkey,
                      uint32_t evk_q_limbs, uint64_t galois_elt, uint64_t *ct_out, void *stream);

/* Host-buffer variants (the "call a user makes" with data in host memory): pinned or pageable HOST
 * pointers for the ciphertexts, key resident on the device.  Copies are pipelined against compute on
 * internal streams; the call returns when ct_out_host is complete. */
int hml_hmult_host(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct_a_host, const uint64_t *ct_b_host,
                   const uint64_t *evk_dev, uint32_t evk_q_limbs, uint64_t *ct_out_host);
int hml_hrotate_host(hml_ctx *ctx, uint32_t L, uint32_t n, const uint64_t *ct_host, const uint64_t *rotkey_dev,
                     uint32_t evk_q_limbs, uint64_t galois_elt, uint64_t *ct_out_host);
/* The same two calls with the ciphertexts PACKED in host memory: a residue has elementBitWidth <= 36 significant bits, so the
 * reference's uint64_t words (include/Context.h:8) carry three empty bytes each over PCIe.  Packed limb = N uint32 low words
 * followed by N high bytes (5N bytes; the compact form of the device's packed limbs); a packed ciphertext = its 2L limbs back
 * to back.  hml_pack_host / hml_unpack_host convert on the CPU (plain loops; for clients that keep words). */
uint64_t hml_packed_bytes(const hml_ctx *ctx, uint64_t n_limbs);
int hml_pack_host(const hml_ctx *ctx, const uint64_t *words, uint64_t n_limbs, void *packed);
int hml_unpack_host(const hml_ctx *ctx, const void *packed, uint64_t n_limbs, uint64_t *words);
int hml_hmult_host_packed(hml_ctx *ctx, uint32_t L, uint32_t n, const void *ct_a_packed, const void *ct_b_packed, const uint64_t *evk_dev,
                          uint32_t evk_q_limbs, void *ct_out_packed);
int hml_hrotate_host_packed(hml_ctx *ctx, uint32_t L, uint32_t n, const void *ct_packed, const uint64_t *rotkey_dev, uint32_t evk_q_limbs,
                            uint64_t galois_elt, void *ct_out_packed);
int hml_host_alloc_pinned(hml_ctx *ctx, uint64_t n_words, uint64_t **out);
int hml_host_free_pinned(hml_ctx *ctx, uint64_t *ptr);

/* ------------------------------------------------------------------ op-sequence replay (BASELINE.json configs[4])
 * The reference runs one operation per process and cannot chain them (reference src/Operation.cpp:636,675,714).  A trace is
 * a list of the CLI's five operations (reference bench_test/bench_micro24.cpp:29-48) over numbered ciphertext slots: slot 0 is
 * the bound input at level L, every other slot is allocated by the replay object; an hmult result sits one level lower and
 * later ops go on from there (the two sources of hadd / hmult must be at the same level; keys bound in a layout with
 * evk_q_limbs >= L serve every level, a plaintext's first limbs serve the lower ones).  In-place ops (dst == a) are allowed
 * except for hmult.
 *   HROTATE dst = rotate(a, 5^b)   (needs the key bound for rotation amount b)      PMULT / PADD dst = a (*|+) plaintext[b]
 *   HADD    dst = a + slot b                                                     HMULT dst = rescale(relin(a * slot b))
 * flags: HML_REPLAY_GRAPH — the whole sequence is captured once into a CUDA graph (after a warm-up run) and every run is one
 * graph launch; HML_REPLAY_HOIST — consecutive rotations of one source share a ModUp (hml_hrotate_hoisted, or
 * hml_hrotate_hoisted_sharded when sh != NULL); HML_REPLAY_HOIST_SUM — a run of at least two such rotations (same rule)
 * that is directly followed by a plaintext-weighted accumulation of all their outputs,
 *   PMULT y = d_k * pt,  then  { PMULT t = d_k * pt; HADD y = y + t (or t + y) }  once for every other output d_k,
 * becomes ONE hml_hrotate_sum_hoisted that writes y — when y is neither the source nor a rotation output and every d_k and t is
 * dead afterwards (its next access, if any, is a write).  The fused rotation outputs and t are then left unwritten, as the t of
 * a fused PMULT / HADD pair already is.  Anything else runs as without the flag (through HML_REPLAY_HOIST when that is set
 * too).  With HML_REPLAY_HOIST_SUM every plaintext is bound as [L + alpha][N] (P-limb j at row L + j, L = the replay's
 * level); PMULT and PADD read its first limbs as before.  Not available with sh != NULL (HML_ERR_UNSUPPORTED).
 * HML_REPLAY_HMULT_SUM — a chain of products summed right after they are formed,
 *   HMULT y = a_0 * b_0,  then  { HMULT t = a_k * b_k; HADD y = y + t (or t + y) }  for k = 1 .. n-1  (n >= 2),
 * becomes ONE hml_hmult_sum (n_out = 1) that writes y — when every product runs at the same level, y and every t are neither
 * sources of any product of the chain nor each other, and every t is dead afterwards (its next access, if any, is a write); t
 * is then left unwritten.  Anything else runs as without the flag.  Not available with sh != NULL (HML_ERR_UNSUPPORTED).
 * With sh != NULL the trace runs limb-sharded: every pointer is the rank's owned-limb slice (see the sharded layouts above). */
enum { HML_OP_HROTATE = 0, HML_OP_PMULT = 1, HML_OP_HADD = 2, HML_OP_PADD = 3, HML_OP_HMULT = 4 };
enum { HML_REPLAY_GRAPH = 1, HML_REPLAY_HOIST = 2, HML_REPLAY_HOIST_SUM = 4, HML_REPLAY_HMULT_SUM = 8 };
typedef struct { uint32_t kind, dst, a, b; } hml_trace_op;
typedef struct hml_replay hml_replay;
int hml_replay_create(hml_ctx *ctx, hml_shard *sh, uint32_t L, const hml_trace_op *ops, uint32_t n_ops, uint32_t flags,
                      hml_replay **out);
int hml_replay_bind(hml_replay *rp, const uint64_t *x, const uint64_t *const *plaintexts, uint32_t n_plaintexts,
                    const uint32_t *rot_amounts, const uint64_t *const *rot_keys, uint32_t n_rot_keys, const uint64_t *evk,
                    uint32_t evk_q_limbs);
int hml_replay_run(hml_replay *rp, void *stream);
int hml_replay_slot(hml_replay *rp, uint32_t slot, uint64_t **ptr, uint32_t *n_limbs);   /* n_limbs per polynomial (final content) */
int hml_replay_slot_level(hml_replay *rp, uint32_t slot, uint32_t *level);                /* level of the slot after the trace */
int hml_replay_destroy(hml_replay *rp);

/* ------------------------------------------------------------------ the count contract
 * Instruction counts of the reference's InsGen trace for one op (what `new OP(...)` generates,
 * reference src/Operation.cpp), computed by walking the same stage list.  One instruction = batchSize
 * coefficients of one limb (reference src/InsGen.cpp:9-13); limb_ops = instructions / (N/batchSize).
 * Pure host code: needs no device, so hml_trace_counts can be called without a ctx. */
#define HML_MAX_STAGES 48
typedef struct {
  char label[48];        /* stage label as embedded in the reference's Instruction::Name */
  char opcode[16];       /* NTT | INTT | MULT | BCONV_STEP2 | AUTO */
  uint64_t limb_ops;
  uint64_t instructions;
} hml_stage_count;
typedef struct {
  uint64_t ntt, intt, mult, bconv_step2, automorph;
  uint64_t total;        /* sum of the five */
  uint64_t driver_total; /* Driver::getTotalIns(): BCONV replicated bconv_num_high*bconv_num_width times (Driver.h:307-320) */
  uint32_t n_stages;
  hml_stage_count stages[HML_MAX_STAGES];
} hml_counts;
int hml_trace_counts(const char *op, uint32_t N, uint32_t batch_size, uint32_t max_level, uint32_t L,
                     uint32_t alpha, uint32_t bconv_high, uint32_t bconv_width, hml_counts *out);
int hml_get_counts(const hml_ctx *ctx, const char *op, uint32_t L, hml_counts *out);

/* Limb-ops the GPU schedule actually EXECUTED since the last reset, per kernel class, so the deltas
 * against the reference trace (SURVEY.md 3.5 D1-D3) are explicit rather than folded in. */
typedef struct {
  uint64_t ntt_limbs, intt_limbs, ewe_limbs, bconv_limb_macs, automorph_limbs;
  uint64_t kernel_launches;
} hml_exec_counts;
/* Buffer plan of one op at level L (reference AddrManage::MallocMem, include/Addr.h:29-48, which prints one
 * `Malloc <name> from A to B` line per intermediate): the device workspace this library carves up for the op, one line per
 * buffer with the reference's buffer names and address unit (limb stride = batchSize addresses; A and B are the base
 * addresses of the first and last limb).  Writes a NUL-terminated string of at most cap bytes; returns HML_OK. */
int hml_buffer_plan(const hml_ctx *ctx, const char *op, uint32_t L, char *out, uint64_t cap);

int hml_exec_counts_get(const hml_ctx *ctx, hml_exec_counts *out);
int hml_exec_counts_reset(hml_ctx *ctx);

/* Per-kernel-class device time of everything executed on `stream` between the two calls — the executed counterpart of the
 * reference's per-unit busy statistics (`NTT_(c)`, `BCONV_(c)`, `EWE_(c)`, `AUTO_(c)`; reference include/Staistics.h:6-40,
 * dumped at src/Operation.cpp:1100-1108).  While profiling, an event follows every launch group, so kernels do not overlap
 * (a measuring mode, not the fast path).  Classes: the reference's opcodes. */
enum { HML_CLS_NTT = 0, HML_CLS_INTT = 1, HML_CLS_BCONV = 2, HML_CLS_EWE = 3, HML_CLS_AUTO = 4, HML_CLS_COUNT = 5 };
typedef struct {
  double us[HML_CLS_COUNT];          /* device time per class */
  uint64_t launches[HML_CLS_COUNT];  /* launch groups per class */
  double total_us;
} hml_profile;
int hml_profile_begin(hml_ctx *ctx, void *stream);
int hml_profile_end(hml_ctx *ctx, hml_profile *out);

/* ------------------------------------------------------------------ the CLI as a library call
 * `Homulator.run <configfile> <operationName> <maxExecutionLevel> <currentLevel> <alpha> [cluster] [--flags]`
 * (reference bench_test/bench_micro24.cpp:5-52).  Runs the op on seeded synthetic data on `device`,
 * prints the config dump, timings, counts and one JSON line to stdout.  Returns the process exit code. */
int hml_cli_main(int argc, char **argv);

#ifdef __cplusplus
}
#endif
#endif
