/*
 * typlonk_b200 -- C ABI of the B200-native PLONK proving backend.
 *
 * This is the drop-in boundary under fabrizio-m/TyPLONK's unchanged Rust API.  The
 * reference has no FFI of its own (it is 100% Rust on arkworks 0.3); each entry point
 * below replaces the body of the cited reference function, and a thin Rust shim
 * (INTEGRATION.md) forwards the reference's public functions to it.
 *
 * Conventions
 *  - every function returns an int status (TP_OK == 0); nothing throws across the ABI;
 *    the Rust shim turns a non-zero status into `panic!` where the reference panics.
 *  - Fr is 4 x u64, Fq is 6 x u64, little-endian limbs, MONTGOMERY form (R = 2^256 /
 *    2^384) -- byte-identical to ark_ff::Fp256 / Fp384 in memory, so buffers cross the
 *    boundary without conversion.
 *  - an affine G1 point is 97 bytes: x (48 B) | y (48 B) Montgomery limbs | 1 byte
 *    infinity flag (ark_ec GroupAffine {x, y, infinity}, packed; when the flag is 1,
 *    (x, y) = (0, 1) in Montgomery form like `GroupAffine::zero()`).
 *  - SRS G1 points cross as packed 96-byte (x | y) records; the all-zero record encodes
 *    the point at infinity.
 *  - pointers are HOST pointers unless the function name ends in `_dev`.
 *  - one in-flight call per tp_ctx (the reference is single-threaded).
 *  - there is no CPU fallback: without a CUDA device tp_ctx_create fails with
 *    TP_ERR_NO_DEVICE and nothing else can be called.
 */
#ifndef TYPLONK_B200_H
#define TYPLONK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tp_ctx tp_ctx;
typedef struct tp_srs tp_srs;
typedef struct tp_circuit tp_circuit;
typedef struct tp_trace tp_trace;
typedef struct tp_permutation_builder tp_permutation_builder;

enum {
  TP_OK = 0,
  TP_ERR_INVALID_ARG = 1,
  TP_ERR_CUDA = 2,
  TP_ERR_SRS_TOO_SHORT = 3,   /* assert!(srs.len() > polynomial.degree())   kzg/src/lib.rs:43 */
  TP_ERR_EMPTY_POLY = 4,      /* .expect("at least 1")                      kzg/src/lib.rs:58 */
  TP_ERR_ZERO_DENOMINATOR = 5,/* Fr division by zero panics                 permutation/src/proving.rs:21 */
  TP_ERR_GATE_UNSATISFIED = 6,/* vanishes() assert                          plonk/src/proof.rs:321,361,504-508 */
  TP_ERR_NO_DEVICE = 7,
  TP_ERR_COLLECTIVE = 8,
  TP_ERR_BUFFER_TOO_SMALL = 9,
  TP_ERR_INVALID_TAG = 10,       /* add_constrain(..) -> Err(()) .unwrap()   permutation/src/lib.rs:48-51, plonk/src/builder.rs:155-159 */
  TP_ERR_UNPLACED_VARIABLE = 11, /* assert!(inner.pending_eq.is_empty())     plonk/src/builder.rs:177 */
  TP_ERR_MALFORMED = 12,         /* a wire encoding that is not canonical / not on the curve */
  TP_ERR_INTERNAL = 13           /* a result the library's own invariants rule out (a defect of the library, not of the input) */
};

#define TP_G1_BYTES 97
#define TP_G2_BYTES 193 /* x.c0 | x.c1 | y.c0 | y.c1 (48 B Montgomery limbs each) | 1 byte infinity flag */
#define TP_PROOF_FIXED_BYTES 1472 /* 13 G1 x 96 + 7 Fr x 32 (uncompressed ark-serialize 0.3 layout) */

/* ---- context ------------------------------------------------------------------------ */

/* Binds to CUDA device `device`.  `stream` is a cudaStream_t to run on (e.g. the caller's
 * torch stream) or NULL to create a private one. */
int tp_ctx_create(int device, void* stream, tp_ctx** out);
int tp_ctx_destroy(tp_ctx* ctx);
const char* tp_last_error(tp_ctx* ctx);
int tp_sync(tp_ctx* ctx);

/* ---- multi-GPU (SURVEY.md 8(e)) ---------------------------------------------------------------------------
 * The prover is SPMD over `world` ranks, one GPU each; every rank ends up with the same proof bytes.  What is split:
 *  - every MSM (kzg/src/lib.rs:41-54) by BUCKET: all ranks extract the signed window digits of all scalars, rank r
 *    sorts / accumulates / reduces only the buckets b with b mod world == r (the window size stays the one planned for
 *    the whole length, so additions and bucket reduction both shrink 1/world).  The per-rank reduction outputs
 *    (a few KB) are all-gathered device-to-device and combined by one small kernel; the host reads back one buffer.
 *  - the quotient (plonk/src/proof.rs:292-375) by coset of the 4n domain, one device broadcast per coset;
 *  - tp_prove's witness upload: each rank copies 1/world of every column over PCIe, the slices travel over NVLink.
 * The communicator lives INSIDE the library (NCCL, loaded with dlopen("libnccl.so.2"); in a torch process that is the
 * copy torch already loaded): no host-language callback runs during a proof.
 *
 * (a) One process per GPU (torchrun, MPI): rank 0 calls tp_comm_unique_id, the host language hands the 128 bytes to
 *     every rank once (any channel), every rank calls tp_ctx_comm_init_rank on its own tp_ctx_create'd context BEFORE
 *     creating the SRS (the MSM plan depends on `world`).  All ranks then make the same calls with the same inputs. */
#define TP_COMM_ID_BYTES 128
int tp_comm_unique_id(uint8_t out[TP_COMM_ID_BYTES]);
int tp_ctx_comm_init_rank(tp_ctx* ctx, int rank, int world, const uint8_t id[TP_COMM_ID_BYTES]);
/* (b) One process, `ndev` GPUs -- the shape of the reference, where CompiledCircuit::prove (plonk/src/proof.rs:26-57)
 *     is one call on one thread.  The returned context is a front for ndev per-device contexts, each with its own
 *     stream and worker thread, joined by ncclCommInitAll.  tp_srs_* , tp_circuit_*, tp_commit, tp_open, tp_prove,
 *     tp_prove_inputs, tp_verify, tp_sync and the tp_prof_* / stat calls accept it unchanged and return one result
 *     (host-pointer arguments are read by every worker; `_dev` entry points are per device and are refused).
 *     A device may be listed more than once: those ranks then exchange through peer copies and a host barrier
 *     instead of NCCL -- slower, but it runs the complete sharded path on a single GPU (used by the tests). */
#define TP_MAX_GROUP 16
int tp_ctx_create_multi(const int* devices, int ndev, tp_ctx** out);
/* ranks behind `ctx` (1 for a plain context) and whether they exchange through NCCL */
int tp_ctx_group_size(const tp_ctx* ctx, int* ndev, int* uses_nccl);

/* Tunables of the MSM behind tp_commit / tp_open / tp_prove.  Results are identical for every
 * setting (the affine sum of a bucket is unique).
 *   "msm_affine_chains" (0/1, $TP_MSM_AFFINE): accumulate buckets in affine coordinates, 16 chunks of the
 *       bucket-sorted list per thread in lockstep with one shared inversion per step (5M + 1S per addition);
 *   "msm_affine_rounds" (0..8, $TP_MSM_AFF_ROUNDS): batch-affine pair-addition rounds run on the bucket-sorted
 *       points before the XYZZ accumulation (kept for comparison; see profiles/);
 *   "msm_reduce_l1" (0 = by size, 1 = never, 2 = whenever possible): whether the bucket reduction runs a level of
 *       16-bucket running sums before its row / column tree sums (big bucket sets: yes; small / sharded ones: no);
 *   "msm_pipeline" (0 = never [default], 1 = on sharded contexts, 2 = always; $TP_MSM_PIPELINE): run a batch of MSMs as
 *       sub-batches on three streams of the library's own, so that the sort and the latency-bound reduction tails of
 *       one sub-batch run under the accumulation of its neighbours; "msm_pipe_min_log" (default 15): only for inputs
 *       of at least 2^this points.  Measured slower than the one-stream order on 1 and on 8 B200s (the accumulation
 *       fills every SM's register file, a second kernel only gets slots as its blocks retire): kept as an experiment;
 *   "ntt_radix_log" (2 [default] or 3): butterfly stages a thread runs on the elements it holds in registers between
 *       two trips through shared memory -- 2: four elements per thread, 1024-element tiles, three blocks per SM;
 *       3: eight elements, 2048-element tiles, two blocks per SM (the round-1 shape);
 *   "msm_acc_staged" (0/1): the accumulation kernel fetches the next table point into shared memory with cp.async
 *       while the current addition runs;
 *   "msm_fq_lazy" (1 [default] or 0): the MSM's XYZZ addition laws keep Fq values in [0, 2q) -- products without
 *       their final conditional subtraction, sums and differences modulo 2q -- and normalise the reduction's outputs
 *       to [0, q) before they leave the device; 0: every value canonical after every operation;
 *   "quotient_all_cosets" (0/1): evaluate the quotient numerator on all four cosets of the 4n domain even when it is
 *       known to vanish on H (gates and copy constraints hold); by default that coset is skipped. */
int tp_ctx_set_option(tp_ctx* ctx, const char* name, long value);
/* Work counters since the last tp_prof_reset: "msm_entries" (bucket additions issued by the accumulation
 * kernels), "msm_calls"; and the plan of the last MSM: "msm_window_bits", "msm_windows", "msm_table_levels",
 * "msm_chunk"; "prove_batch_wave": the proofs per wave of the last tp_prove_batch.  Unknown names fail with
 * TP_ERR_INVALID_ARG. */
int tp_ctx_get_stat(tp_ctx* ctx, const char* name, double* out);

/* Per-phase device timers (CUDA events on the ctx stream).  Phase ids: TP_PHASE_*. */
enum {
  TP_PHASE_MSM_TOTAL = 0,
  TP_PHASE_MSM_SORT = 1,       /* digit extraction + counting sort */
  TP_PHASE_MSM_ACCUM = 2,      /* bucket accumulation kernel (dominant) */
  TP_PHASE_MSM_REDUCE = 3,     /* boundary merge + bucket reduction */
  TP_PHASE_NTT = 4,
  TP_PHASE_QUOTIENT = 5,       /* pointwise numerator + division by Z_H */
  TP_PHASE_PERM = 6,           /* grand product */
  TP_PHASE_SCAN = 7,           /* openings: Horner + division by (X - z) */
  TP_PHASE_COUNT = 8
};
int tp_prof_enable(tp_ctx* ctx, int on);
int tp_prof_reset(tp_ctx* ctx);
/* ms[TP_PHASE_COUNT], launches[TP_PHASE_COUNT]: accumulated since the last reset. */
int tp_prof_get(tp_ctx* ctx, double* ms, uint64_t* launches);
/* total number of kernels this library launched on ctx since creation */
int tp_launch_count(tp_ctx* ctx, uint64_t* out);

/* ---- SRS  (kzg/src/srs.rs) ------------------------------------------------------------ */

/* Srs::from_secret(s, gates) (srs.rs:30-34): gates + 3 powers [G, sG, s^2 G, ...] generated
 * on the device (fixed-base windowed multiplication + batched affine normalisation). */
int tp_srs_from_secret(tp_ctx* ctx, const uint64_t tau[4], size_t gates, tp_srs** out);
/* Adopt an existing Vec<G1Affine> (srs.rs:43-45 g1_ref), packed to 96 B / point. */
int tp_srs_upload(tp_ctx* ctx, const uint8_t* g1_xy, size_t len, tp_srs** out);
int tp_srs_len(const tp_srs* srs, size_t* len);
int tp_srs_g1_download(tp_ctx* ctx, const tp_srs* srs, size_t offset, size_t count, uint8_t* out_xy);
int tp_srs_destroy(tp_ctx* ctx, tp_srs* srs);
/* Srs::g2_ref / g2s_ref (srs.rs:46-51): (G2, tau G2).  tp_srs_from_secret derives them (Srs::g2, srs.rs:25-28);
 * an uploaded SRS has none until tp_srs_set_g2, and the verifier entry points fail with TP_ERR_INVALID_ARG
 * without them. */
int tp_srs_g2(const tp_srs* srs, uint8_t g2[TP_G2_BYTES], uint8_t g2s[TP_G2_BYTES]);
int tp_srs_set_g2(tp_srs* srs, const uint8_t g2[TP_G2_BYTES], const uint8_t g2s[TP_G2_BYTES]);

/* ---- SRS ceremony (additive API: a powers-of-tau setup that no single party's secret controls) ------------------ */

/* One ceremony contribution: *out = a new SRS with g1[i] = s^i * srs.g1[i], g2 unchanged, g2s = s * srs.g2s;
 * pubkey = [s]G2 (TP_G2_BYTES, ABI encoding as tp_srs_g2), which proves the link (tp_srs_update_check).
 * s: Montgomery limbs like tp_srs_from_secret's tau; s == 0 or s >= r -> TP_ERR_INVALID_ARG; an SRS without G2
 * points -> TP_ERR_INVALID_ARG.  srs is left untouched (destroy it once the link is checked).  Device groups: every
 * rank scales its own copy. */
int tp_srs_contribute(tp_ctx* ctx, const tp_srs* srs, const uint64_t s[4], tp_srs** out, uint8_t pubkey[TP_G2_BYTES]);
/* *ok = 1 iff the SRS is the powers of one secret: g1[0] = G, g2 = the G2 generator, every g1[i] in G1 and not
 * infinity, g2s in G2 and not infinity, and g1[i+1] = t g1[i] for all i where g2s = [t]G2 (a pairing check of a
 * combination with random weights rho^i, rho drawn inside the call from the operating system; a wrong SRS passes
 * with probability at most (len - 1) / (r - 1)).  len < 2, no G2 points -> TP_ERR_INVALID_ARG.  A bad point is
 * *ok = 0, not an error.  Device groups: one rho for every rank, the verdict is rank 0's. */
int tp_srs_verify(tp_ctx* ctx, const tp_srs* srs, int* ok);
/* One ceremony link, host only: *ok = 1 iff e(next_tau_g1, G2) == e(prev_tau_g1, pubkey), with both G1 points
 * on the curve, in G1, not infinity, and pubkey in G2, not infinity.  (tau_g1 = g1[1] of each SRS.) */
int tp_srs_update_check(const uint8_t prev_tau_g1[TP_G1_BYTES], const uint8_t next_tau_g1[TP_G1_BYTES],
                        const uint8_t pubkey[TP_G2_BYTES], int* ok);

/* ---- KZG  (kzg/src/lib.rs) ------------------------------------------------------------- */

/* KzgScheme::commit (lib.rs:37-54): sum_i coeffs[i] * srs[i].  len == 0 -> infinity.
 * len > srs length -> TP_ERR_SRS_TOO_SHORT. */
int tp_commit(tp_ctx* ctx, const tp_srs* srs, const uint64_t* coeffs, size_t len, uint8_t out[TP_G1_BYTES]);
int tp_commit_dev(tp_ctx* ctx, const tp_srs* srs, const void* coeffs_dev, size_t len, uint8_t out[TP_G1_BYTES]);
/* KzgScheme::open (lib.rs:55-64): y = p(z), W = commit((p - y) / (X - z)).
 * len == 0 -> TP_ERR_EMPTY_POLY. */
int tp_open(tp_ctx* ctx, const tp_srs* srs, const uint64_t* coeffs, size_t len, const uint64_t z[4],
            uint8_t w_out[TP_G1_BYTES], uint64_t y_out[4]);

/* KzgScheme::verify (lib.rs:66-81): *ok = [ e(W, g2s - z g2) == e(C - y G, g2) ], evaluated as the single product
 * e(W, g2s) e(-(z W + C - y G), g2) == 1 (the same predicate by bilinearity; one shared Miller loop, one final
 * exponentiation).  Host arithmetic only -- the pairing is O(1) work per proof and has no data-parallel part; no
 * device or context is involved.  Points off the curve give *ok = 0. */
int tp_kzg_verify(const uint8_t g2[TP_G2_BYTES], const uint8_t g2s[TP_G2_BYTES], const uint8_t commitment[TP_G1_BYTES],
                  const uint8_t w[TP_G1_BYTES], const uint64_t y[4], const uint64_t z[4], int* ok);
/* *ok = [ prod_i e(g1[i], g2[i]) == 1 ] for `count` pairs (97 B / 193 B records).  Host only. */
int tp_pairing_check(const uint8_t* g1, const uint8_t* g2, size_t count, int* ok);

/* ---- NTT  (ark-poly Evaluations::interpolate / evaluate_over_domain; call sites
 *      plonk/src/proof.rs:50,106,115,125,128,337,415; builder.rs:85; permutation/src/lib.rs:171,188) */

/* In place, natural order in and out, size 2^log_n (1 <= log_n <= 28).  inverse != 0 scales by
 * n^-1.  coset != NULL: forward evaluates on coset*H (input scaled by coset^i); inverse
 * interpolates from coset*H (output scaled by coset^-i). */
int tp_ntt(tp_ctx* ctx, uint64_t* data, unsigned log_n, int inverse, const uint64_t* coset);
int tp_ntt_dev(tp_ctx* ctx, void* data_dev, unsigned log_n, int inverse, const uint64_t* coset);

/* ---- permutation argument  (permutation/src/proving.rs:7-31) -------------------------- */

/* CompiledPermutation::prove: out[0] = 1, out[j+1] = out[j] * prod_i (v_ij + beta id_ij + gamma) /
 * (v_ij + beta sigma_ij + gamma); writes n + 1 values.  A zero denominator ->
 * TP_ERR_ZERO_DENOMINATOR. */
int tp_perm_prove(tp_ctx* ctx, const uint64_t* const values[3], const uint64_t* const id[3],
                  const uint64_t* const sigma[3], size_t n, const uint64_t beta[4], const uint64_t gamma[4],
                  uint64_t* out);

/* ---- circuit + prover  (plonk/src/lib.rs:18-35, plonk/src/proof.rs:96-194) ------------- */

/* Upload a CompiledCircuit: 5 selector polynomials in COEFFICIENT form (q_l q_r q_o q_m q_c,
 * each zero-padded to n), the permutation columns `cols` split into id[i][j] and sigma[i][j]
 * (evaluation form, n each), and the three coset representatives k_i (permutation/src/lib.rs:141-154).
 * Caches what the reference recomputes per proof (sigma coefficient forms, 4n-domain evaluations). */
int tp_circuit_load(tp_ctx* ctx, const tp_srs* srs, const uint64_t* const selectors[5],
                    const uint64_t* const id[3], const uint64_t* const sigma[3], const uint64_t cosets[3][4],
                    size_t n, tp_circuit** out);
/* Setup path (CircuitBuilder::compile numerics, plonk/src/builder.rs:70-88 + Permutation::compile,
 * permutation/src/lib.rs:101-128): selector EVALUATIONS (n each) and the flat permutation
 * `perm[3n]` (index = j + i*n) -> device sigma/id tables, selector interpolation, and the five
 * fixed commitments (5 x 97 B). */
int tp_circuit_compile(tp_ctx* ctx, const tp_srs* srs, const uint64_t* const selector_evals[5],
                       const uint64_t* perm, size_t n, tp_circuit** out, uint8_t fixed_commitments[5 * TP_G1_BYTES]);
int tp_circuit_destroy(tp_ctx* ctx, tp_circuit* c);
/* sigma commitments / evaluations the verifier recomputes per call (permutation/src/lib.rs:165-194). */
int tp_circuit_sigma_commitments(tp_ctx* ctx, tp_circuit* c, uint8_t out[3 * TP_G1_BYTES]);

/* prove() (proof.rs:96-194) from the three witness columns in EVALUATION form (n each, the
 * last three rows already hold the blinders, proof.rs:43-49) and the n-padded public inputs.
 * Writes TP_PROOF_FIXED_BYTES bytes: a.com a.W a.y | b.. | c.. | z.com z.W z.y zw.W zw.y |
 * evaluation_point | t0 t1 t2 | r.W r.y  (G1 = ark-serialize 0.3 uncompressed 96 B, Fr = 32 B LE
 * canonical).  The gate equation failing on any row -> TP_ERR_GATE_UNSATISFIED. */
int tp_prove(tp_ctx* ctx, tp_circuit* c, const uint64_t* const advice[3], const uint64_t* public_inputs,
             uint8_t* proof_out, size_t proof_cap);
int tp_prove_dev(tp_ctx* ctx, tp_circuit* c, const void* const advice_dev[3], const void* public_inputs_dev,
                 uint8_t* proof_out, size_t proof_cap);
/* The same from the public-input vector AS THE CALLER OF CompiledCircuit::prove PASSES IT (proof.rs:26-31: any
 * length <= n, e.g. `vec![0]`): the first n_public rows are uploaded, the rest are zero-filled on the device --
 * the `public_inputs.resize(self.rows, Fr::zero())` of proof.rs:52-53.  When every public input is zero (the only
 * vectors the reference can prove, SURVEY.md App. D.1) the prover skips that polynomial's transforms. */
int tp_prove_inputs(tp_ctx* ctx, tp_circuit* c, const uint64_t* const advice[3], const uint64_t* public_inputs,
                    size_t n_public, uint8_t* proof_out, size_t proof_cap);
/* Prove `count` witnesses of circuit c in one call: tp_prove_inputs for each, with the MSMs, NTTs and scans of
 * all proofs batched and one host round trip per stage for the whole batch.
 * advice: 3 * count host column pointers, advice[3k + i] = column i of proof k (n Montgomery Fr, blinders in place).
 * public_inputs[k] / n_public[k]: as tp_prove_inputs takes them (NULL allowed when n_public[k] == 0;
 *   public_inputs may be NULL when every n_public[k] is 0).
 * proofs_out: count x TP_PROOF_FIXED_BYTES; block k is byte-identical to what tp_prove_inputs writes for proof k.
 * status (count ints, may be NULL): status[k] = what tp_prove_inputs returns for proof k (TP_OK,
 *   TP_ERR_GATE_UNSATISFIED, TP_ERR_ZERO_DENOMINATOR); block k is zero-filled when it is not TP_OK and the call
 *   still returns TP_OK.  With status == NULL the call returns the lowest-index failure's code (index in
 *   tp_last_error); the other blocks are written as above.
 * count == 0 -> TP_OK.  count > 65536, null pointers, n_public[k] > n -> TP_ERR_INVALID_ARG;
 * proofs_cap < count * TP_PROOF_FIXED_BYTES -> TP_ERR_BUFFER_TOO_SMALL.
 * The proofs run in waves of W at a time (tp_ctx_get_stat "prove_batch_wave"): W is at most 64 and as many as fit
 * half of the free device memory, at least 1; each proof of a wave needs 44n + 1 Fr of device buffers, which the
 * circuit keeps (they only grow) until tp_circuit_destroy.  The circuit's own buffers -- what
 * tp_circuit_read_poly shows -- are left untouched.  Device groups: every rank runs the batch, the MSMs are sharded
 * by bucket, everything else is replicated. */
int tp_prove_batch(tp_ctx* ctx, tp_circuit* c, size_t count, const uint64_t* const* advice,
                   const uint64_t* const* public_inputs, const size_t* n_public,
                   uint8_t* proofs_out, size_t proofs_cap, int* status);

/* Inspection: an intermediate polynomial of the LAST proof made with `c`, read from the prover's device buffers
 * (Montgomery Fr): the quotient t as 3n coefficients (quotient_polynomial, proof.rs:292-375; slices t0 | t1 | t2), the
 * linearisation polynomial r (proof.rs:376-439; n coefficients), the grand product as its n + 1 evaluations
 * (CompiledPermutation::prove, permutation/src/proving.rs:7-31) and as coefficients, the witness polynomials.  With
 * out == NULL only *count is written.  Lets tests compare every stage with the reference's own function, not only
 * the final bytes. */
enum { TP_POLY_QUOTIENT = 0, TP_POLY_LINEARISATION = 1, TP_POLY_Z_EVALS = 2, TP_POLY_Z = 3, TP_POLY_A = 4, TP_POLY_B = 5, TP_POLY_C = 6 };
int tp_circuit_read_poly(tp_ctx* ctx, tp_circuit* c, int which, uint64_t* out, size_t cap_elems, size_t* count);

/* verify() (proof.rs:195-233, 441-503): `proof` is the TP_PROOF_FIXED_BYTES block tp_prove writes, `public_inputs`
 * the proof's public-input vector (n_public Montgomery Fr; resized to n like proof.rs:204-205).  The device
 * interpolates and evaluates the public-input polynomial, evaluates sigma_1..3 at the challenge point and (first call
 * only; cached in the circuit) computes the five selector and three sigma commitments with the MSM; the host
 * re-derives the challenges, checks the five openings, assembles the linearisation commitment and checks its
 * opening (12 pairings as 6 two-pair products).  *ok = 1 accept / 0 reject; a malformed encoding (coordinate >= q,
 * scalar >= r) is TP_ERR_INVALID_ARG. */
int tp_verify(tp_ctx* ctx, tp_circuit* c, const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs,
              size_t n_public, int* ok);
/* Verify `count` proofs of circuit c at once (proof.rs:195-233 for each, folded into one check).
 * proofs: count x TP_PROOF_FIXED_BYTES, contiguous (the block tp_prove writes).
 * public_inputs[k] / n_public[k]: proof k's public-input vector as tp_verify takes it (NULL allowed when n_public[k] == 0;
 * public_inputs itself may be NULL when every n_public[k] is 0).
 * *all_ok = 1 iff every proof is accepted.  each_ok (count ints, may be NULL): per-proof verdicts.
 * count == 0 -> *all_ok = 1.  count > 65536, null pointers, n_public[k] > n, unreduced public input
 * -> TP_ERR_INVALID_ARG.  A proof that tp_verify rejects or reports as malformed gets each_ok[k] = 0; the call still succeeds.
 * The six KZG equations of every proof are weighted by scalars drawn from a Blake2b-512 hash of the circuit's
 * commitments and of every proof with its public inputs (so the verdicts are a pure function of the inputs) and summed
 * into one two-pair pairing product over two MSMs; when that check fails and each_ok is given, the failing set is
 * halved and re-checked down to sets of 8 proofs, which get tp_verify's own host check.
 * Stricter than tp_verify: random linear combinations are only sound in the prime-order subgroup, so every proof
 * point is checked for [r]P = 0 and a proof with a point outside the subgroup is rejected (tp_verify checks only that
 * the points are on the curve).  For proofs whose points are all in the subgroup, each_ok[k] equals tp_verify's
 * verdict except with probability about 2^-250.  Device groups: as tp_verify (the MSMs are sharded by bucket). */
int tp_verify_batch(tp_ctx* ctx, tp_circuit* c, const uint8_t* proofs, size_t count,
                    const uint64_t* const* public_inputs, const size_t* n_public, int* all_ok, int* each_ok);
/* The host half of tp_verify with every circuit-dependent value supplied by the caller, for callers that compute
 * sigma_1(zeta), sigma_2(zeta) and PI(zeta) themselves: the eight commitments, the domain size n (power of two), the
 * coset representatives k_i, those three evaluations for THIS proof's challenge point, [1]G (srs[0]) and the two G2
 * points.  No device involved.  The proof does not carry sigma_1(zeta) and sigma_2(zeta) (verify() evaluates them
 * from the circuit, proof.rs:458-459): a verifier without the circuit uses a verification key (tp_vk_*) instead. */
typedef struct tp_verifier_inputs {
  uint8_t fixed_commitments[5][TP_G1_BYTES];
  uint8_t sigma_commitments[3][TP_G1_BYTES];
  uint8_t identity[TP_G1_BYTES];
  uint8_t g2[TP_G2_BYTES], g2s[TP_G2_BYTES];
  uint64_t cosets[3][4];
  uint64_t sigma_evals[2][4];
  uint64_t public_eval[4];
  uint64_t n;
} tp_verifier_inputs;
int tp_verify_prepared(const tp_verifier_inputs* in, const uint8_t* proof, size_t proof_len, int* ok);
/* ---- verification keys ----------------------------------------------------------------------------------------
 * A tp_vk holds exactly what verify() reads of a compiled circuit: n, the coset representatives k_i, the five selector
 * and three sigma commitments, identity = srs[0], the SRS's G2 and tau G2, and sigma_1, sigma_2 in coefficient form on
 * the device (n Fr each).  The proof does not carry sigma_1(zeta), sigma_2(zeta), so the key must hold both
 * polynomials: it is O(n), 64n bytes (64 MiB at 2^20, 1 GiB at 2^24); sigma_3 enters only through its commitment.
 * A key does not hold the prover's state (about 99n Fr of caches and per-proof buffers for a tp_circuit).
 * Made on a device group, a key holds one part per rank; serialisation reads rank 0's part. */
typedef struct tp_vk tp_vk;
/* Export from a compiled circuit: the commitments come from the circuit's cache (one MSM on first use, as
 * tp_verify), sigma_1 and sigma_2 are copied on the device.  The key owns its copies and outlives the circuit.
 * An SRS without G2 points -> TP_ERR_INVALID_ARG. */
int tp_vk_from_circuit(tp_ctx* ctx, tp_circuit* c, tp_vk** out);
int tp_vk_destroy(tp_ctx* ctx, tp_vk* vk);
/* Wire form, ark-serialize 0.3 uncompressed items: "TPVK" | u32 LE version = 1 | u64 n | 3 x Fr k |
 * 9 x G1 (q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 identity) | G2 g2 | G2 g2s | Vec<Fr> sigma_1 | Vec<Fr> sigma_2:
 * 1376 + 64n bytes.  The scalars are converted on the device.  Buffer too small -> TP_ERR_BUFFER_TOO_SMALL. */
int tp_vk_serialized_size(const tp_vk* vk, size_t* bytes);
int tp_vk_serialize(tp_ctx* ctx, const tp_vk* vk, uint8_t* out, size_t cap, size_t* written);
/* check 0: exact length, tag and version, n a power of two in [2, 2^28], both Vec lengths == n, every scalar < r,
 * every coordinate < q, valid flags (and both G2 points on the twist, which the pairings need); 1: + every point on
 * its curve; 2: + the nine G1 points in the prime-order subgroup and g2, g2s in G2.  A rejected record ->
 * TP_ERR_MALFORMED naming the field (or the sigma index) in tp_last_error.  Device groups: every rank decodes its own
 * part. */
int tp_vk_deserialize(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_vk** out);
/* tp_verify against a key: the same checks, the same code and the same verdict as tp_verify on the circuit the key
 * came from, malformed-input errors included.  PI(zeta) takes two n-Fr device buffers, allocated with the key on the
 * first non-zero public-input vector; all-zero public inputs need no device work.  A key made on another context ->
 * TP_ERR_INVALID_ARG. */
int tp_vk_verify(tp_ctx* ctx, tp_vk* vk, const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs,
                 size_t n_public, int* ok);
/* tp_verify_batch over proofs of several circuits: proof k (block k of `proofs`) is checked against keys[key_of[k]].
 * Keys may differ in n and in SRS.  sigma_1, sigma_2 of every key are evaluated at all of its proofs' points in one
 * launch; the proofs are grouped by their key's (g2, g2s) and every group g gets its own L_g, R_g, all in one batched
 * MSM (up to eight groups per MSM call), checked by one pairing product of 2G pairs.  The weights rho are drawn from
 * a Blake2b-512 hash of every key (n, k, the nine G1 points, g2, g2s) and of every proof with its key index and public
 * inputs.  Localisation, each_ok and the subgroup check as tp_verify_batch.
 * count == 0 -> *all_ok = 1.  count > 65536, n_keys not in [1, 4096], key_of[k] >= n_keys, null pointers,
 * n_public[k] > that key's n, an unreduced public input, a key made on another context -> TP_ERR_INVALID_ARG.
 * Device groups: every rank runs, the MSMs are sharded by bucket, the verdict is rank 0's. */
int tp_vk_verify_batch(tp_ctx* ctx, tp_vk* const* keys, size_t n_keys, const uint32_t* key_of, const uint8_t* proofs,
                       size_t count, const uint64_t* const* public_inputs, const size_t* n_public, int* all_ok,
                       int* each_ok);
/* ---- proof format v2 -------------------------------------------------------------------------------------------
 * The format above (v1) matches the reference's prove() and verify() byte for byte, and it is NOT SOUND: its
 * challenge zeta is drawn from [a], [b], [c], [z] alone, and the quotient commitments [t0], [t1], [t2] are made after
 * zeta is known and never hashed.  A prover who knows zeta can take t = Lin(zeta) / Z_H(zeta) as a constant, so that
 * r(zeta) = 0 for ANY witness, and tp_verify accepts.  v1 also has no working public inputs (no gate reads them; only
 * all-zero vectors prove).  v1 is kept for reference parity; new users should use v2 (DESIGN.md, "Proof format v2").
 *
 * v2: the first l inputs of a circuit are public (tp_trace_create_public puts them in public gates, rows 0..l-1,
 * q_l = 1, PI_i = -x_i); a Blake2b-512 transcript binds the key, the public values and every commitment before each
 * challenge; one batched KZG opening at zeta and one at zeta * omega; a 1056-byte block
 *   [a] [b] [c] [z] [t0] [t1] [t2] [W_zeta] [W_zeta_omega] | a(zeta) b(zeta) c(zeta) s1(zeta) s2(zeta) z(zeta omega)
 * and a constant-size key (1368 B).  Verification is host only: no context, no device. */
#define TP_PROOF_V2_FIXED_BYTES 1056 /* 9 G1 x 96 + 6 Fr x 32 */
#define TP_VK2_BYTES 1368
typedef struct tp_vk2 tp_vk2;
/* The key of circuit c with its first n_public rows public: n, l, the cosets, the five selector and three sigma
 * commitments (the circuit's cache: one MSM on first use), srs[0], g2 and g2s (prepared for the pairing).  Host
 * memory only; it outlives the circuit and the context.  An SRS without G2, n_public > n - 3, or rows 0..n_public-1
 * not all public gates (q_l = 1, other selectors 0) or row n_public one too -> TP_ERR_INVALID_ARG: the key's l must be
 * the number of public gates the circuit was traced with. */
int tp_vk2_from_circuit(tp_ctx* ctx, tp_circuit* c, size_t n_public, tp_vk2** out);
int tp_vk2_destroy(tp_vk2* vk);
/* "TPK2" | u32 LE version = 1 | u64 n | u64 l | 3 x Fr k | 9 x G1 (q_l q_r q_o q_m q_c sigma_1 sigma_2 sigma_3 srs[0])
 * | G2 g2 | G2 g2s, ark-serialize 0.3 uncompressed items: TP_VK2_BYTES.  cap < TP_VK2_BYTES -> TP_ERR_BUFFER_TOO_SMALL. */
int tp_vk2_serialize(const tp_vk2* vk, uint8_t* out, size_t cap);
/* check 0: exact length, tag, version, n a power of two in [4, 2^28], l <= n - 3, every scalar < r, every coordinate
 * < q, valid flags, both G2 points on the twist; 1: + the nine G1 points on the curve; 2: + in the prime-order
 * subgroup, g2 and g2s in G2.  A rejected field -> TP_ERR_MALFORMED; tp_vk2_last_error names it.  Host only. */
int tp_vk2_deserialize(const uint8_t* bytes, size_t len, int check, tp_vk2** out);
/* The reason of the last failed tp_vk2_deserialize / tp_proof_v2_decode of the calling thread. */
const char* tp_vk2_last_error(void);
/* Proves with c: advice = three host columns (n Montgomery Fr each, as tp_prove).  The public values are column a,
 * rows 0..l-1 (l = the key's); they are written to public_out (l x 4 limbs, may be NULL when l = 0).  A key whose n,
 * cosets, commitments or srs[0] are not c's -> TP_ERR_INVALID_ARG; proof_cap < TP_PROOF_V2_FIXED_BYTES ->
 * TP_ERR_BUFFER_TOO_SMALL; a gate that fails -> TP_ERR_GATE_UNSATISFIED.  A witness that breaks a copy constraint
 * gives a proof that tp_verify_v2 rejects; r(zeta) != 0 for a witness that meets its constraints (which the protocol
 * rules out) -> TP_ERR_INTERNAL.  Device groups: every rank proves, rank 0's bytes go out. */
int tp_prove_v2(tp_ctx* ctx, tp_circuit* c, const tp_vk2* vk, const uint64_t* const advice[3], uint8_t* proof_out,
                size_t proof_cap, uint64_t* public_out);
/* Host only.  *ok = 1 iff the TP_PROOF_V2_FIXED_BYTES block is canonical, its nine points are on the curve and in G1,
 * n_public equals the key's l, and the pairing check holds for these public values (Montgomery limbs).
 * proof_len != TP_PROOF_V2_FIXED_BYTES -> *ok = 0.  An unreduced public input -> TP_ERR_INVALID_ARG. */
int tp_verify_v2(const tp_vk2* vk, const uint8_t* proof, size_t proof_len, const uint64_t* public_inputs,
                 size_t n_public, int* ok);
/* Wire form: the block | u64 LE l | l x Fr (32 B canonical LE).  encode: cap < 1064 + 32 l -> TP_ERR_BUFFER_TOO_SMALL
 * (*written, if not NULL, gets the size either way).  decode: exact length, canonical scalars and coordinates, points
 * on the curve, else TP_ERR_MALFORMED; fixed_out and public_out may be NULL (ask for *n_public first; public_cap: the
 * values public_out holds).  Host only. */
int tp_proof_v2_encode(const uint8_t fixed[TP_PROOF_V2_FIXED_BYTES], const uint64_t* public_inputs, size_t n_public,
                       uint8_t* out, size_t cap, size_t* written);
int tp_proof_v2_decode(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_V2_FIXED_BYTES],
                       uint64_t* public_out, size_t public_cap, size_t* n_public);
/* The challenges verify() derives from a proof (proof.rs:235-244): alpha, beta, gamma, evaluation point. */
int tp_proof_challenges(const uint8_t* proof, size_t proof_len, uint64_t alpha[4], uint64_t beta[4], uint64_t gamma[4],
                        uint64_t point[4]);

/* ---- circuit tracing, copy constraints, witness generation (host; SURVEY.md 8 f3) --------
 * The reference records a circuit by running its closure over BuildVar, and computes a witness
 * by running it again over ComputeVar, under a Mutex and with a println! per gate.  Here the
 * host language records each `+` / `*` / `assert_eq` of the closure ONCE into a tp_trace (a
 * flat gate list); padding, selector columns, the copy-constraint permutation and every
 * witness are derived from it natively.  No device involved; feeds tp_circuit_compile and
 * tp_prove.  Variables are dense ids: the n_inputs inputs are 0..n_inputs-1 in order. */
enum { TP_GATE_MUL = 0, TP_GATE_ADD = 1, TP_GATE_DUMMY = 2, TP_GATE_PUBLIC = 3 }; /* plonk/src/builder.rs:30-36; PUBLIC: proof format v2 */

/* Context::default + BuildVar::input per input (plonk/src/builder.rs:371-377, 95-99). */
int tp_trace_create(size_t n_inputs, tp_trace** out);
/* tp_trace_create with the first n_public inputs public (proof format v2): public gate i (row i, i < n_public,
 * kind TP_GATE_PUBLIC, q_l = 1, all other selectors 0) places input i at (0, i); a later use of input i gets a copy
 * constraint like any already-placed operand.  The witness has a = x_i, b = c = 0 there.  tp_trace_gate(s) refuse the
 * kind.  n_public > n_inputs -> TP_ERR_INVALID_ARG. */
int tp_trace_create_public(size_t n_inputs, size_t n_public, tp_trace** out);
int tp_trace_destroy(tp_trace* t);
/* BuildVar::binary_operation (plonk/src/builder.rs:339-370): appends a gate row j, gives the
 * output a new id placed at (2, j), and places each operand at (0, j) / (1, j) -- an operand
 * that already sits in a cell gets a fresh id there plus a copy constraint old = fresh. */
int tp_trace_gate(tp_trace* t, int kind, uint64_t lhs, uint64_t rhs, uint64_t* out_var);
/* The same for `count` gates in one call (out_vars may be NULL). */
int tp_trace_gates(tp_trace* t, size_t count, const uint8_t* kinds, const uint64_t* lhs, const uint64_t* rhs,
                   uint64_t* out_vars);
/* Var::assert_eq on BuildVar -> Context::add_eq (plonk/src/builder.rs:427-433, 148-166): a copy
 * constraint when both variables are placed, otherwise parked until tp_trace_finish. */
int tp_trace_assert_eq(tp_trace* t, uint64_t a, uint64_t b);
/* Context::finish + CircuitBuilder::fill (plonk/src/builder.rs:167-186, 47-58): resolves the
 * parked equalities (one still unplaced -> TP_ERR_UNPLACED_VARIABLE), pads with Dummy gates to
 * rows = the first power of two >= gates + 3 (minimum 2).  Idempotent. */
int tp_trace_finish(tp_trace* t, size_t* rows, size_t* gates);
/* `rows` gate kinds (TP_GATE_*), Dummy padding included. */
int tp_trace_gate_kinds(const tp_trace* t, uint8_t* out);
/* Selector EVALUATIONS q_l | q_r | q_o | q_m | q_c, 5 x rows Montgomery Fr, contiguous
 * (Gate::to_row, plonk/src/builder.rs:73-84, 316-324) -- tp_circuit_compile's input. */
int tp_trace_selectors(const tp_trace* t, uint64_t* out);
/* PermutationBuilder::build(rows) (permutation/src/lib.rs:62-93) over the recorded copy
 * constraints: perm[3 * rows], index = j + i * rows.  Constraint classes are visited in
 * first-insertion order (the reference's HashMap order is random per process).  Consumes the
 * constraints (mem::take), so a second call returns the identity. */
int tp_trace_permutation(tp_trace* t, uint64_t* perm);
/* The witness half of CompiledCircuit::prove (plonk/src/proof.rs:33-49; ComputeVar,
 * plonk/src/builder.rs:380-397): replays the gates over `inputs` (n_inputs Montgomery Fr) and
 * writes the three advice columns in evaluation form (rows Fr each): left | right | value per
 * gate, zeros up to rows - 3, then blinders[3k..3k+3] for column k.  Like the reference's
 * ComputeVar::assert_eq, equalities are NOT checked here. */
int tp_trace_witness(const tp_trace* t, const uint64_t* inputs, size_t n_inputs, const uint64_t* blinders,
                     uint64_t* const advice[3]);

/* The permutation crate's builder on its own (permutation/src/lib.rs:28-93): with_rows,
 * add_row, add_constrain (a tag with i > 3 or j >= rows -> TP_ERR_INVALID_TAG), build. */
int tp_permutation_builder_create(size_t rows, tp_permutation_builder** out);
int tp_permutation_builder_destroy(tp_permutation_builder* b);
int tp_permutation_builder_add_row(tp_permutation_builder* b);
int tp_permutation_builder_add_constrain(tp_permutation_builder* b, size_t left_i, size_t left_j, size_t right_i,
                                         size_t right_j);
int tp_permutation_builder_build(tp_permutation_builder* b, size_t size, uint64_t* perm);
/* Permutation::compile (permutation/src/lib.rs:101-154) on its own: from the flat permutation (index = j + i n, n a
 * power of two) the device builds id[i][j] = k_i w^j and sigma[i][j] = k_i' w^j' for (i', j') = perm[i n + j], n
 * Montgomery Fr per column, and the coset representatives k_i (the first three k >= 1 with k^n != 1; may be NULL).
 * tp_circuit_compile does the same internally; this entry feeds tp_perm_prove / tp_circuit_load. */
int tp_permutation_compile(tp_ctx* ctx, const uint64_t* perm, size_t n, uint64_t* const id[3], uint64_t* const sigma[3],
                           uint64_t cosets[3][4]);

/* Fr conversions for host languages without a big-integer type (host only): Fr::from(i64) with negatives as
 * r - |v| (plonk/src/utils.rs:152-153); 32-byte LE canonical <-> Montgomery limbs (>= r -> TP_ERR_MALFORMED). */
int tp_fr_from_i64(int64_t v, uint64_t out[4]);
int tp_fr_from_canonical(const uint8_t in[32], uint64_t out[4]);
int tp_fr_to_canonical(const uint64_t in[4], uint8_t out[32]);

/* ---- wire formats (SURVEY.md 8 f4 / App. A.6) --------------------------------------------
 * The reference derives no (de)serialisation for Proof or Srs, so the framing is ours; every
 * item is encoded the way ark-serialize 0.3 writes that type uncompressed (the encoding the
 * reference's own transcript uses for G1, plonk/src/proof/challenges.rs:17-22): Fr = 32 B LE
 * canonical; G1 = x | y, 48 B LE canonical each, bit 6 of the last byte = infinity; G2 =
 * x.c0 | x.c1 | y.c0 | y.c1 likewise; Vec = u64 LE length + items. */
#define TP_WIRE_G1_BYTES 96
#define TP_WIRE_G2_BYTES 192
/* Proof (plonk/src/proof.rs:85-95) = the TP_PROOF_FIXED_BYTES block of tp_prove | Vec<Fr> of
 * the n-padded public inputs.  Host only.  `public_inputs` are Montgomery limbs. */
int tp_proof_encoded_size(size_t n_public, size_t* bytes);
int tp_proof_encode(const uint8_t* fixed, const uint64_t* public_inputs, size_t n_public, uint8_t* out, size_t cap,
                    size_t* written);
/* Checked decoding: exact length, every scalar < r, every coordinate < q, every point on the
 * curve (or flagged infinity), no compressed-form flag -> otherwise TP_ERR_MALFORMED.
 * `public_inputs_out` (Montgomery, capacity cap_public elements) and `fixed_out` may be NULL. */
int tp_proof_decode(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_FIXED_BYTES],
                    uint64_t* public_inputs_out, size_t cap_public, size_t* n_public);
/* The prime-order subgroup check ark-serialize's checked deserialisation adds on top of tp_proof_decode's "on the
 * curve": *ok = 1 iff [r]P = 0 for all 13 points of the fixed block (host only; a malformed point -> TP_ERR_MALFORMED). */
int tp_proof_points_in_subgroup(const uint8_t* fixed, size_t len, int* ok);
/* Srs (kzg/src/srs.rs:8-14) = Vec<G1> | G2 | tau G2.  The device converts the points out of /
 * into Montgomery form and validates them, one point per thread.  check: 0 = canonical
 * encoding only (ark `deserialize_unchecked`), 1 = + on the curve, 2 = + in the prime-order
 * subgroup ([r]P = 0; ark's checked deserialisation).  A rejected point -> TP_ERR_MALFORMED
 * with its index in tp_last_error. */
int tp_srs_serialized_size(const tp_srs* srs, size_t* bytes);
int tp_srs_serialize(tp_ctx* ctx, const tp_srs* srs, uint8_t* out, size_t cap, size_t* written);
int tp_srs_deserialize(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_srs** out);

/* Compressed encodings (ark-serialize 0.3 `serialize`, what CanonicalSerialize writes by default): a G1 point is its
 * canonical x, 48 B LE, with bit 7 of the last byte set iff y > -y (canonical integers) and bit 6 for infinity
 * (written as x = 0, sign bit clear; both bits set is invalid); a G2 point is x.c0 | x.c1 with the flags in the last
 * byte of x.c1, y > -y comparing c1 first, then c0.  Decoding recovers y = (x^3 + b)^((q+1)/4): an x without a root is
 * rejected at every check level.  A proof block is the same fields in the same order as the TP_PROOF_FIXED_BYTES
 * block: 13 x 48 + 7 x 32 bytes.  The Fiat-Shamir transcript still hashes uncompressed points, so challenges do not
 * depend on the wire form. */
#define TP_WIRE_G1_COMPRESSED_BYTES 48
#define TP_WIRE_G2_COMPRESSED_BYTES 96
#define TP_PROOF_COMPRESSED_FIXED_BYTES 848
/* TP_PROOF_FIXED_BYTES block -> compressed block (host only).  len != TP_PROOF_FIXED_BYTES, or anything
 * tp_proof_decode rejects in the block -> TP_ERR_MALFORMED; cap < TP_PROOF_COMPRESSED_FIXED_BYTES ->
 * TP_ERR_BUFFER_TOO_SMALL. */
int tp_proof_compress(const uint8_t* fixed, size_t len, uint8_t* out, size_t cap);
/* Compressed block -> TP_PROOF_FIXED_BYTES block (host only, checked: what tp_verify and tp_verify_prepared take).
 * len != TP_PROOF_COMPRESSED_FIXED_BYTES, a scalar >= r, x >= q, an x without a root or invalid flags ->
 * TP_ERR_MALFORMED; cap < TP_PROOF_FIXED_BYTES -> TP_ERR_BUFFER_TOO_SMALL.  fixed_out is untouched on failure. */
int tp_proof_decompress(const uint8_t* in, size_t len, uint8_t* fixed_out, size_t cap);
/* The Proof framing of tp_proof_encode / tp_proof_decode with the compressed block: block | Vec<Fr>.  Encoding takes
 * and decoding returns the uncompressed TP_PROOF_FIXED_BYTES block, so everything downstream is unchanged. */
int tp_proof_encoded_size_compressed(size_t n_public, size_t* bytes);
int tp_proof_encode_compressed(const uint8_t* fixed, const uint64_t* public_inputs, size_t n_public, uint8_t* out,
                               size_t cap, size_t* written);
int tp_proof_decode_compressed(const uint8_t* bytes, size_t len, uint8_t fixed_out[TP_PROOF_FIXED_BYTES],
                               uint64_t* public_inputs_out, size_t cap_public, size_t* n_public);
/* tp_proof_decompress for `count` contiguous compressed blocks at once, the square roots on the device (one point per
 * thread): fixed_out gets count x TP_PROOF_FIXED_BYTES, ready for tp_verify_batch.
 * status (count ints, may be NULL): status[k] = tp_proof_decompress's verdict on block k (TP_OK or TP_ERR_MALFORMED);
 *   a failed block is zero-filled and the call still returns TP_OK.  With status == NULL the call returns
 *   TP_ERR_MALFORMED for the lowest failing index (named in tp_last_error); the other blocks are written as above.
 * count == 0 -> TP_OK.  count > 65536, null pointers -> TP_ERR_INVALID_ARG; cap < count * TP_PROOF_FIXED_BYTES ->
 * TP_ERR_BUFFER_TOO_SMALL.  Device groups: rank 0 does the work. */
int tp_proofs_decompress(tp_ctx* ctx, const uint8_t* in, size_t count, uint8_t* fixed_out, size_t cap, int* status);
/* Srs with compressed points: u64 count | count x 48 B G1 | G2 | tau G2 (96 B each), half the size of the
 * uncompressed form.  check as tp_srs_deserialize: 0 and 1 recover y (on the curve by construction), 2 adds the
 * prime-order subgroup check; a rejected point -> TP_ERR_MALFORMED with the count and the first index in
 * tp_last_error.  Device groups: serialisation reads rank 0's copy, every rank decodes its own. */
int tp_srs_serialized_size_compressed(const tp_srs* srs, size_t* bytes);
int tp_srs_serialize_compressed(tp_ctx* ctx, const tp_srs* srs, uint8_t* out, size_t cap, size_t* written);
int tp_srs_deserialize_compressed(tp_ctx* ctx, const uint8_t* bytes, size_t len, int check, tp_srs** out);

/* ---- helpers ---------------------------------------------------------------------------- */
/* Measured dependent-free IMAD throughput of this device (instructions/s), for rooflines. */
int tp_measure_imad_peak(tp_ctx* ctx, double* imad_per_s, double* imad_wide_per_s);
/* Synthetic-input helper (SURVEY.md 8(d)): `count` x ark-ff 0.3 `Fr::rand` drawn from rand 0.8
 * `StdRng::seed_from_u64(seed)` (ChaCha12), written as Montgomery limbs -- the same stream the
 * reference's Fiat-Shamir uses (plonk/src/proof/challenges.rs:38-45).  Host only. */
int tp_fr_rand_stream(uint64_t seed, size_t count, uint64_t* out);
/* The raw output words of the library's `StdRng` (rand 0.8: ChaCha12; csrc/transcript.h), seeded either with a 32-byte
 * seed (`from_seed`, seed32 != NULL) or with `seed_from_u64(seed_u64)` (rand_core 0.6 PCG32 expansion).  Host only; lets
 * the generator behind the Fiat-Shamir challenges be checked against the rand crates' own value-stability constants. */
int tp_stdrng_words(const uint8_t* seed32, uint64_t seed_u64, size_t count, uint32_t* out);
/* "tp-build-stamp:<sha256 of the sources and flags this binary was compiled from>" (host only). */
const char* tp_build_stamp(void);
/* Self-test of the device field/curve arithmetic against host arithmetic; 0 failures expected. */
int tp_selftest(tp_ctx* ctx, int* failures);

#ifdef __cplusplus
}
#endif
#endif
