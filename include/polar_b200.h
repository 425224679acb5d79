/* polar_b200.h -- C ABI of the B200 (sm_100a) polar-code hot path.
 *
 * Drop-in boundary for jaco267/polar-code-pytorch-sionna.  The reference has no FFI (it is pure
 * Python); the boundary it exposes is the nn.Module call surface of its encoder / decoders / link
 * model.  Each entry point below replaces the *body* of one of those Python methods; the Python
 * mirror under polar-code-pytorch-sionna_b200/{x_run_sn_polar,my_sn} keeps the reference signatures
 * and calls these through ctypes (x_run_sn_polar/d_kernels.py is the loader).  Reference file:line
 * cited per function are relative to the reference checkout.
 *
 * Conventions
 *  - Every pointer named d_* is a DEVICE pointer into caller-owned memory (e.g. a torch CUDA
 *    tensor's data_ptr()); h_* is a HOST pointer.  No torch types cross this boundary.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Device entry
 *    points only enqueue work: they never synchronise, never allocate and never read the environment, so they
 *    are safe under stream capture.  The one allocation the kernels need -- the SC stage scratch (one slot per SM,
 *    76 MB on a 148-SM part, csrc/polar_sc4.cu) -- is made by polar_init(device), which a caller runs once per
 *    device before decoding (the Python loader does it when it builds a code's device tables); an SC decode of
 *    n >= 1024 on a device that was not initialised returns POLAR_EINVAL with a message saying so.
 *  - Bit packing: bit (i % 32) of 32-bit word (i / 32) holds position i (LSB first); a row of n
 *    positions occupies POLAR_WORDS(n) = max(1, n/32) words.
 *  - Logits follow the reference decoder input: ln P(1)/P(0), fp32, row-major [B, n]
 *    (polar_sc.py:113-122).  Decisions are bit-exact with the reference on the same logits.
 *  - Return value: POLAR_OK (0) or a negative POLAR_E* code; polar_last_error() gives the text
 *    (thread local).  The Python mirror turns codes into the reference's exception types.
 */
#ifndef POLAR_B200_H_
#define POLAR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POLAR_OK 0
#define POLAR_EINVAL (-1)   /* bad n / L / k / B, or null pointer                     */
#define POLAR_EALIGN (-2)   /* pointer not aligned as documented                      */
#define POLAR_ENOMEM (-3)   /* workspace too small / shared memory does not fit       */
#define POLAR_ECUDA (-4)    /* CUDA runtime error (launch failed, no device ...)      */

#define POLAR_MAX_N 8192    /* SC decoder / encoder / front end                       */
#define POLAR_SCL_MAX_N 4096
#define POLAR_SCL_MAX_L 32
#define POLAR_WORDS(n) ((n) < 32 ? 1 : (n) / 32)

const char *polar_last_error(void);
/* One-time per-device set-up (may allocate and synchronise; idempotent, thread safe, restores the current device):
 * queries the device and allocates the SC stage scratch.  Required before polar_sc_decode_* of n >= 1024; the
 * host-buffer entry points call it themselves. */
int polar_init(int device);
/* Tuning / test options, by the name of the POLAR_* environment variable they shadow (an explicit override wins over
 * the environment; the environment is looked up once per option, never on the launch path).  Not needed by callers. */
int polar_set_option(const char *name, int value);
void polar_clear_options(void);
/* library / device info: writes "polar_b200 <version> sm_100a ..." */
const char *polar_version(void);
/* number of kernels this library has launched in the calling process (bench.py: gpu_launches) */
unsigned long long polar_launch_count(void);

/* ---- SC decoder --------------------------------------------------------------------------
 * Replaces SC_Dec._decode_batch + _polar_decode_sc_tf + _cn_op_tf/_vn_op_tf + the info_pos gather
 * (x_run_sn_polar/polar/polar_sc.py:33-133).  fp32 min-sum, f clipped to +-30, g unclipped.
 *  d_logit        [B, n] fp32, 16-byte aligned rows (n >= 4) -- NOT negated by the caller
 *  d_frozen_mask  [POLAR_WORDS(n)] bit set = frozen position (polar_sc.py:23-24)
 *  d_u_packed     [B, POLAR_WORDS(n)] all n decisions, frozen = 0 (msg_uhat[:,0,:]); may be NULL
 *  d_u_info_f32   [B, k] fp32 0./1. at ascending info_pos (the tensor SC_Dec.forward returns);
 *                 may be NULL.  d_info_pos [k] int32 (required iff d_u_info_f32 != NULL)
 *  n power of two, 2 <= n <= POLAR_MAX_N. */
int polar_sc_decode_f32(const float *d_logit, const uint32_t *d_frozen_mask, int n, int64_t B,
                        uint32_t *d_u_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                        void *stream);

/* Same call, exact-boxplus check-node update f = ln(1+e^(x+y)) - ln(e^x+e^y) (inputs clipped to +-30, fp32) instead
 * of min-sum: the arithmetic of the Sionna-style SC_Dec in my_sn/fec/polar/dec.py:13-157 (SURVEY 8f row N2).  Same
 * kernels compiled a second time (csrc/polar_bp_wrap.cu).  Parity with the CPU reference is statistical for this
 * mode: its exp/log come from the host libm and the boxplus difference cancels to rounding noise near ties. */
int polar_sc_decode_boxplus_f32(const float *d_logit, const uint32_t *d_frozen_mask, int n, int64_t B,
                                uint32_t *d_u_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                void *stream);

/* ---- SCL decoder -------------------------------------------------------------------------
 * Replaces SCL_Dec._decode_np_batch and everything under it (x_run_sn_polar/polar/polar_scl.py:49-209),
 * the argmin/gather of forward (:224-228) and, when crc_len > 0, the CRC-aided selection of
 * my_sn/fec/polar/dec.py:507-527 (+ my_sn/fec/crc.py:119-138).  fp64 LLR tree and path metrics,
 * pm += log(1+exp(-x)) evaluated literally; lazy copy-on-write of the tree through per-stage pointer tables.
 * Two mappings behind the one entry point: csrc/polar_scl3.cu (n in [64,4096], L in [2,32], 16-byte aligned rows:
 * two virtual top stages computed from the channel row, tree in shared memory) and csrc/polar_scl.cu (everything
 * else); they return identical bits (tests/test_gpu_parity.py::test_scl3_equals_scl2_lists_and_path_metrics).
 *  L power of two, 1 <= L <= 32; n power of two, 2 <= n <= POLAR_SCL_MAX_N
 *  d_best_packed  [B, POLAR_WORDS(n)] decisions of the selected path
 *  d_u_info_f32   [B, k] fp32 or NULL (as above)
 *  d_pm_sorted    [B, L] fp64 ascending path metrics (before any CRC penalty) or NULL
 *  d_list_packed  [B, L, POLAR_WORDS(n)] decisions of all L survivors, pm-ascending, or NULL
 *  d_crc_rows     [n] uint32: for info position i, the crc_len-bit syndrome contribution of that bit
 *                 (row of the reference's [k, crc_len] generator matrix, crc.py:54-74, MSB = parity
 *                 bit 0); 0 for frozen positions.  NULL / crc_len == 0: plain argmin.  With crc_len > 0, k must be
 *                 the number of information positions (it scales the penalty 30 k of dec.py:517-518) even when
 *                 d_u_info_f32 is NULL; k < 1 is rejected.
 *  d_workspace    polar_scl_workspace_bytes(n, L, B) bytes, 256-byte aligned. */
size_t polar_scl_workspace_bytes(int n, int L, int64_t B);
int polar_scl_decode(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                     uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                     double *d_pm_sorted, uint32_t *d_list_packed,
                     const uint32_t *d_crc_rows, int crc_len,
                     void *d_workspace, size_t workspace_bytes, void *stream);

/* Same calls with the exact boxplus check-node update in fp64 (my_sn/fec/polar/dec.py:331-340): the list decoder of the
 * Sionna-style SCL_Dec with leaf-level path-metric updates (its use_fast_scl=False arithmetic; SURVEY 8f row N2).
 * The workspace size is the same function of (n, L, B). */
size_t polar_scl_boxplus_workspace_bytes(int n, int L, int64_t B);
int polar_scl_decode_boxplus(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                             uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                             double *d_pm_sorted, uint32_t *d_list_packed,
                             const uint32_t *d_crc_rows, int crc_len,
                             void *d_workspace, size_t workspace_bytes, void *stream);
/* The same decoder with the reference's fast-SCL node shortcuts (use_fast_scl=True, my_sn/fec/polar/dec.py:269-306,
 * 354-376): a rate-0 node (all leaves frozen) or REP node (only the last leaf carries information) of up to 32 leaves is
 * not descended into -- its path-metric update is the sum of log(1+exp(-+llr)) over the node's own LLRs (for REP: one
 * sum per value of the information bit, then the usual sort / keep L).  Exact under the boxplus f (not under min-sum, so
 * there is no min-sum counterpart).  Same arguments and workspace. */
int polar_scl_decode_boxplus_pruned(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                                    uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                                    double *d_pm_sorted, uint32_t *d_list_packed,
                                    const uint32_t *d_crc_rows, int crc_len,
                                    void *d_workspace, size_t workspace_bytes, void *stream);

/* ---- hybrid SC -> SCL decoder (use_hybrid_sc=True of the Sionna-style SCL_Dec, my_sn/fec/polar/dec.py:437-470) --------
 * For each row b:  s = SC(x[b]) (all n decisions, frozen = 0);  out[b] = s if the CRC over s holds, else the CRC-aided
 * list decision of x[b] (L paths, selection as in polar_scl_decode).  An SC decision that passes the CRC by chance is kept,
 * so the result is not the full list decoder's.  Four operations enqueued on `stream`, no synchronisation, no allocation:
 *   1. the SC decoder of the chosen arithmetic over all B rows -> d_best_packed (the workspace when NULL) and d_u_info_f32
 *   2. a memset of the failing-row count (d_n_list_out when given, else the workspace)
 *   3. csrc/polar_scl_api.cu: syndrome of every SC row (XOR of d_crc_rows[i] over its set bits i), failing rows compacted
 *   4. the generic list kernel (csrc/polar_scl.cu scl2, in every arithmetic) over the failing rows only, overwriting
 *      their d_best_packed / d_u_info_f32 rows in place; its decisions equal polar_scl_decode*'s for the same row
 *  cn_mode         0: min-sum (polar_sc_decode_f32 + the min-sum list kernel), 1: exact boxplus (polar_sc_decode_boxplus_f32
 *                  + polar_scl_decode_boxplus's kernel), 2: boxplus with fast-SCL pruning (list stage as
 *                  polar_scl_decode_boxplus_pruned)
 *  d_logit etc.    as polar_sc_decode_f32 (16-byte aligned rows) and polar_scl_decode; n, L in the SCL range
 *  d_crc_rows      required, crc_len in 1..32, k in 1..n (the number of information positions)
 *  d_best_packed / d_u_info_f32   at least one of the two; there is no path-metric or list output
 *  d_n_list_out    device int32, or NULL: number of list-decoded rows (stream ordered)
 *  d_workspace     polar_scl_hybrid_workspace_bytes(n, L, B, cn_mode) bytes, 256-byte aligned (ENOMEM / EALIGN).  Layout:
 *                  packed SC rows [B, POLAR_WORDS(n)] uint32 | count int32 | failing rows [B] int32 | list-kernel
 *                  workspace for a persistent grid sized for B rows, each region 256-byte aligned.  The list workspace
 *                  dominates: at n = 1024, L = 8 it is about 1.3 GB once B fills the grid (B >= 4 x the resident warps,
 *                  18944 rows on a 148-SM B200); the other regions add 132 B per row.
 *  B == 0 returns POLAR_OK and launches nothing. */
size_t polar_scl_hybrid_workspace_bytes(int n, int L, int64_t B, int cn_mode);
int polar_scl_decode_hybrid(const float *d_logit, const uint32_t *d_frozen_mask, int n, int L, int64_t B,
                            uint32_t *d_best_packed, float *d_u_info_f32, const int32_t *d_info_pos, int k,
                            const uint32_t *d_crc_rows, int crc_len, int cn_mode, int32_t *d_n_list_out,
                            void *d_workspace, size_t workspace_bytes, void *stream);

/* ---- encoder-----------------------------------------------------------------------------
 * polar_encode_packed: x = u.G over GF(2) on bit-packed rows (XOR butterfly; the transform of
 * my_sn/fec/polar/enc.py:85-96 == (c @ G) % 2 of x_run_sn_polar/polar/enc.py:42).
 * polar_encode_f32: the whole PolarEncoder.forward (x_run enc.py:30-43 / my_sn enc.py:97-113):
 * scatter u[B,k] (fp32 0/1) to info positions, transform, write c[B,n] fp32 0/1.
 *  d_info_rank [n] int32: index into u for info positions, -1 for frozen. */
int polar_encode_packed(const uint32_t *d_u_full_packed, int n, int64_t B, uint32_t *d_c_packed,
                        void *stream);
int polar_encode_f32(const float *d_u, const int32_t *d_info_rank, int n, int k, int64_t B,
                     float *d_c, uint32_t *d_c_packed_or_null, void *stream);

/* ---- 5G rate matching / rate recovery (TS 38.212 5.4.1; SURVEY 8f row N3) -----------------------------------
 * polar_gather_cols_f32: out[b, e] = x[b, idx[e]] -- Polar5GEncoder.forward's combined sub-block interleaver +
 * circular buffer + channel interleaver (my_sn/fec/polar/enc.py:378-381; idx built on the host, enc.py:262-361).
 * polar_rate_recover_f32: out[b, j] = fill[j], replaced by x[b, src0[j]] when src0[j] >= 0, plus x[b, src1[j]] when
 * src1[j] >= 0 -- Polar5GDecoder.forward's channel de-interleaver, de-puncturing (fill 0), de-shortening (fill -100),
 * repetition combining and sub-block de-interleaver in one pass (my_sn/fec/polar/dec.py:600-634). */
int polar_gather_cols_f32(const float *d_x, const int32_t *d_idx, int n_in, int n_out, int64_t B, float *d_out,
                          void *stream);
int polar_rate_recover_f32(const float *d_x, const int32_t *d_src0, const int32_t *d_src1, const float *d_fill,
                           int n_in, int n_out, int64_t B, float *d_out, void *stream);
/* polar_nr5g_awgn_frontend: the 5G uplink link up to the decoder in one launch, per codeword: Bernoulli(1/2) payload ->
 * CRC attach -> channel allocation -> polar transform -> rate matching (the gather index above) -> QPSK/AWGN ->
 * closed-form demapper (as polar_awgn_frontend).  One warp per codeword.
 *  n               mother-code length, power of two in [32, 1024]; e: channel bits, 1 <= e <= POLAR_MAX_N
 *  d_payload_mask  [POLAR_WORDS(n)] bit set at the k payload positions (info_pos[:k])
 *  d_crc_rows      [n] at payload position info_pos[t]: the CRC generator word of payload bit t (MSB = parity bit 0,
 *                  i.e. bit crc_len-1-j is parity bit j; CRCEncoder(crc_degree, k)._rows); 0 elsewhere
 *  d_crc_pos       [crc_len] polar position of parity bit j (info_pos[k + j]); 1 <= crc_len <= 32
 *  d_rm_idx        [e] polar position sent at channel position i; entries must lie in [0, n) (not checked)
 *  d_u_packed_out  [B, POLAR_WORDS(n)] payload + CRC at their positions, frozen 0: what a correct decoder returns
 *  d_c_packed_out  [B, (e+31)/32] rate-matched codeword, LSB first, tail bits 0; may be NULL
 *  d_logit_out     [B, e] fp32, any 4-byte alignment
 * Random numbers: the payload is a pure function of (seed, offset + b); row b of the logits equals the first e columns
 * of polar_qpsk_awgn_llr(seed, offset + b, no, c) for that row's rate-matched codeword c zero-padded to a multiple of 4.
 * POLAR_EINVAL for bad n / e / crc_len, B < 0, no <= 0 or a null table / output pointer.  B == 0 launches nothing.
 * No allocation, no synchronisation. */
int polar_nr5g_awgn_frontend(uint64_t seed, uint64_t offset, float no, const uint32_t *d_payload_mask,
                             const uint32_t *d_crc_rows, const int32_t *d_crc_pos, int crc_len,
                             const int32_t *d_rm_idx, int n, int e, int64_t B, uint32_t *d_u_packed_out,
                             uint32_t *d_c_packed_out, float *d_logit_out, void *stream);

/* ---- BPSK/AWGN LLR front end -----------------------------------------------------------------
 * Replaces System_AWGN_model.forward up to the decoder call (z_sys_model/awgn_model.py:33-40):
 * BinarySource -> PolarEncoder -> Mapper (QPSK = BPSK per dimension, amplitude 1/sqrt2) -> AWGN
 * (variance no/2 per real dimension) -> Demapper (closed form logit = -2.sqrt2.y/no).
 * Random numbers: counter-based Philox4x32-10 keyed by (seed, codeword index + offset); the
 * stream is a pure function of (seed, offset, b, i), independent of launch geometry.
 *  d_u_packed_out [B, POLAR_WORDS(n)] transmitted u (info bits at info positions, frozen 0)
 *  d_c_packed_out [B, POLAR_WORDS(n)] transmitted codeword, or NULL
 *  d_logit_out    [B, n] fp32 */
int polar_awgn_frontend(uint64_t seed, uint64_t offset, float no, const uint32_t *d_frozen_mask,
                        int n, int64_t B, uint32_t *d_u_packed_out, uint32_t *d_c_packed_out,
                        float *d_logit_out, void *stream);
/* Channel + demapper only, for caller-supplied codewords (Mapper/AWGN/Demapper layers,
 * my_sn/trans/mapping.py:136-149,225-241, my_sn/trans/channel/awgn.py:19-29). */
int polar_qpsk_awgn_llr(uint64_t seed, uint64_t offset, float no, const float *d_c /*[B,n] 0/1*/,
                        int n, int64_t B, float *d_logit_out, void *stream);

/* Binary erasure channel with LLR output (my_sn/trans/channel/discrete_channel.py:79-107 with return_llrs=True, used by
 * z_sys_model/bec_model.py:19-27; SURVEY 8f row N4): logit = +llr_max (bit 1) / -llr_max (bit 0), set to 0 with
 * probability pe per position.  polar_bec_frontend = BinarySource -> PolarEncoder -> channel in one launch;
 * polar_bec_llr applies the channel to caller-supplied codewords (fp32 0/1, n a multiple of 4). */
int polar_bec_frontend(uint64_t seed, uint64_t offset, float pe, float llr_max, const uint32_t *d_frozen_mask,
                       int n, int64_t B, uint32_t *d_u_packed_out, uint32_t *d_c_packed_out, float *d_logit_out,
                       void *stream);
int polar_bec_llr(uint64_t seed, uint64_t offset, float pe, float llr_max, const float *d_c /*[B,n] 0/1*/,
                  int n, int64_t B, float *d_logit_out, void *stream);

/* ---- error counting ------------------------------------------------------------------------
 * count_errors / count_block_errors (my_sn/sim.py:7-18).  d_counters[0] += bit errors,
 * d_counters[1] += block errors (unsigned 64-bit, caller zeroes them). */
int polar_count_errors_packed(const uint32_t *d_a, const uint32_t *d_b, const uint32_t *d_mask_or_null,
                              int n, int64_t B, unsigned long long *d_counters, void *stream);
int polar_count_errors_f32(const float *d_b, const float *d_b_hat, int k, int64_t B,
                           unsigned long long *d_counters, void *stream);

/* ---- Monte-Carlo stop rules on the device ----------------------------------------------------------
 * Replaces the host logic of sim_ber (my_sn/sim.py:79-133): accumulate the counters of a group of 1..POLAR_MC_GROUP_MAX
 * queued iterations that may span SNR points and evaluate the target-bit-error / target-block-error / max-iteration
 * rules and the early stop (:128-133) in a one-thread kernel, so the host can keep iterations queued without reading
 * counters back (SURVEY 8f row N1).  The Monte-Carlo loop packs several iterations into one decoder launch so that a
 * small per-rank batch still fills the GPU.
 *  d_delta        uint64[n_items,4]: (bit errors, block errors, bits, blocks) of each iteration (all-reduced over ranks
 *                 when the batch is sharded); cleared by the call.
 *  h_item_point   HOST int32[n_items]: SNR-point index each iteration was simulated for (read during the call).
 *  d_state        int64[n_points,8]: one state row per SNR point: [0..3] running totals, [4] stop flag, [5] status
 *                 (1 max iter, 2 no errors (early stop), 3 bit target, 4 block target, sim.py:63-66), [6] iterations
 *                 counted, [7] reserved.  Once [4] is set, later iterations of that point are ignored.
 *  d_sweep8       int64[8]: [0] current point, [1] sweep ended, [2] iterations counted so far (= position in the random
 *                 number sequence), [3] groups seen, [4] iterations of this group that counted.
 *  expect_q       value of d_sweep8[2] the group was planned for; on a mismatch nothing counts.
 *  target_*       < 0: rule disabled.
 * Iteration j counts only if all earlier ones of the group did, the sweep has not ended and the loop is at point
 * h_item_point[j]; the first that does not ends the group. */
#define POLAR_MC_GROUP_MAX 32
int polar_mc_control_group(unsigned long long *d_delta, const int32_t *h_item_point, int n_items, long long *d_state,
                           int n_points, long long *d_sweep8, long long expect_q, long long target_bit_errs,
                           long long target_block_errs, long long max_mc_iter, int early_stop, void *stream);

/* ---- N4: ordered-statistics decoder (my_sn/fec/osd/dec.py:8-192, OSDecoder.forward :149-191) -------------------
 * One CTA per codeword: reliability sort, most-reliable basis by the reference's pivot method (:99-117), hard decisions
 * on the pivots re-encoded, every error pattern of weight 1..t in itertools.combinations order (:57-62) under the
 * LLR distance mean log(1 + exp(llr (1 - 2c))) (:64-79, fp32), first minimum within a weight, strictly smaller across
 * weights (:181-184).  Decisions equal the reference's except where two candidates are closer than fp32 rounding.
 *  d_gm_rows   generator matrix, bit-packed rows [k, (n+31)/32] in the ORIGINAL column order (dec.py:40-42)
 *  d_c_packed  [B, (n+31)/32] decided codeword bits (all n positions, like the reference) or NULL
 *  d_c_f32     [B, n] the same as fp32 0./1. (what OSDecoder.forward returns) or NULL (one of the two is required)
 *  d_dist      [B] distance of the decided codeword, or NULL
 *  2 <= n <= 1024, 1 <= k <= n, 0 <= t <= 6, C(k, t) < 2^31. */
int polar_osd_decode(const float *d_logit, const uint32_t *d_gm_rows, int n, int k, int t, int64_t B,
                     uint32_t *d_c_packed, float *d_c_f32, float *d_dist, void *stream);

/* Test hook: d_mismatch3[0..2] += how many of `count` pseudo-random arguments in [-30, 30] make the decoder's own
 * exp / log / log(1+exp(.)) sequences (csrc/polar_softplus.cuh) differ BITWISE from the CUDA math library's. */
int polar_scl3_math_selftest(uint64_t count, unsigned long long *d_mismatch3, void *stream);

/* ---- bit (un)packing helpers used by the Python mirror ---------------------------------------- */
int polar_pack_bits_f32(const float *d_x /*[B,n] 0/1*/, int n, int64_t B, uint32_t *d_packed, void *stream);
int polar_unpack_info_f32(const uint32_t *d_packed, const int32_t *d_pos /*[k]*/, int n, int k, int64_t B,
                          float *d_out /*[B,k]*/, void *stream);

/* ---- host-buffer entry points (end-to-end path: H2D + decode + D2H inside the call) -------------
 * Same semantics as the device entry points but with HOST buffers; the batch is cut into chunks
 * that are copied, decoded and copied back on two streams so PCIe transfers overlap the kernels.
 * h_logit should be page-locked for full overlap (pageable memory works, slower).  Synchronous. */
int polar_sc_decode_host(const float *h_logit, const uint32_t *h_frozen_mask, int n, int64_t B,
                         uint32_t *h_u_packed, int device);
int polar_scl_decode_host(const float *h_logit, const uint32_t *h_frozen_mask, int n, int L, int64_t B,
                          uint32_t *h_best_packed, double *h_pm_sorted_or_null,
                          const uint32_t *h_crc_rows_or_null, int crc_len, int device);
/* The same with the tensor the reference's forward() returns: h_u_info_f32 [B, k] fp32 0./1. at ascending h_info_pos
 * (polar_sc.py:127-133, polar_scl.py:224-234).  Either output may be NULL (not both).  This is what SC_Dec.forward /
 * SCL_Dec.forward call for a CPU tensor.  Pageable caller buffers are staged through page-locked memory by a few
 * host threads (POLAR_HOST_COPY_THREADS, default 4); page-locked ones are DMA'd directly. */
int polar_sc_decode_host_f32(const float *h_logit, const uint32_t *h_frozen_mask, int n, int64_t B,
                             uint32_t *h_u_packed_or_null, float *h_u_info_f32_or_null, const int32_t *h_info_pos, int k,
                             int device);
int polar_scl_decode_host_f32(const float *h_logit, const uint32_t *h_frozen_mask, int n, int L, int64_t B,
                              uint32_t *h_best_packed_or_null, float *h_u_info_f32_or_null, const int32_t *h_info_pos, int k,
                              double *h_pm_sorted_or_null, const uint32_t *h_crc_rows_or_null, int crc_len, int device);

#ifdef __cplusplus
}
#endif
#endif /* POLAR_B200_H_ */
