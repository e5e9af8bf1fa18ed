/* virgo_b200.h -- C ABI of the B200-native Virgo++ GKR sumcheck prover.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types. The C++ class
 * `prover` shipped in virgo-plus_b200/host/prover.{h,cpp} (same public API as the reference's
 * src/prover.h:12-42) forwards 1:1 to these entry points; INTEGRATION.md shows the binding.
 * Citations are into /root/reference.
 *
 * Conventions: every function returns 0 on success or a negative vp_status; vp_last_error()
 * returns a description of the last failure on the calling thread. There is NO CPU fallback: all
 * prover entry points fail with VP_ERR_CUDA when no sm_100 device / driver is usable.
 * A context is single-threaded (like the reference prover: one prover per process, SURVEY 8b).
 *
 * Limits (checked; violations return VP_ERR_CIRCUIT / VP_ERR_ARG / VP_ERR_CUDA with a message, never undefined behaviour):
 *   - 2 <= layers <= 120; layer_size * instances <= 2^31 per layer (table indices are 32 bit), hence at most 31 rounds
 *     per sumcheck phase (the whole-proof kernel takes the phase's <= 32 challenges through its parameters);
 *   - in-layer gate indices, lv and dadId entries fit 32 bits; every dadId entry must be < the source layer's size;
 *   - .pws files: variable ids dense and < 2^40 (main.cpp indexes a vector by id); malformed numbers reject the file;
 *   - sharded contexts: world in {1, 2, 4, 8}, one process per GPU of ONE node;
 *   - witness inputs are read like the reference reads them, as F((long long) x) (prover.cpp:30-36,
 *     fieldElement.cpp:24-27): 0 <= x < p as is, x < 0 as p + x; other values are reduced mod p (the reference keeps
 *     them non-canonical). The circuit-level setters (vp_circuit_set_inputs, .pws inputs) only accept 0 <= x < p;
 *   - challenges must be canonical (both components < p): vp_set_challenges / vp_prove / vp_round reject others.
 */
#ifndef VIRGO_B200_H
#define VIRGO_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* bit-identical to virgo::fieldElement {real, img} (lib/virgo/src/fieldElement.hpp:96-97) */
typedef struct { uint64_t re, im; } vp_F;

typedef struct vp_circuit vp_circuit; /* host-side layered circuit (+ instance count) */
typedef struct vp_ctx vp_ctx;         /* prover context: owns all device memory */

typedef enum {
    VP_OK = 0,
    VP_ERR_ARG = -1,      /* bad argument / call out of protocol order */
    VP_ERR_CIRCUIT = -2,  /* malformed circuit or .pws */
    VP_ERR_CUDA = -3,     /* CUDA / NCCL failure, or no usable device */
    VP_ERR_ASSERT = -4,   /* an is_assert gate evaluates to non-zero (prover.cpp:18-21, :211) */
    VP_ERR_NOMEM = -5
} vp_status;

const char* vp_last_error(void);
const char* vp_version(void);

/* ------------------------------------------------------------------ circuit (host side)
 * Replaces parse()+DAG_to_layered() (src/main.cpp:15-137,176-231) and layeredCircuit::subsetInit()
 * (src/circuit.cpp:43-80), including their observable quirks (SURVEY.md 9.2). */
int vp_circuit_load_pws(const char* path, vp_circuit** out);
int vp_circuit_load_pws_text(const char* text, size_t len, vp_circuit** out);
/* Synthetic random add/mul circuit, semantics of layeredCircuit::randomize (circuit.cpp:17-41). */
int vp_circuit_random(int n_layers, int log_size, uint64_t seed, vp_circuit** out);
/* Build from flat arrays (concatenated over layers 0..n-1, gate_off-style: layer i occupies
 * [sum_{j<i} layer_size[j], ...)). Layer-0 entries carry the input VALUE in u (like gate.u of an
 * Input gate, main.cpp:108-110). If dad_size == NULL the subsets and lv are derived with the
 * subsetInit rule; otherwise lv / dad_size[i*n+l] / dad_id (concatenated in (i,l) order) are taken
 * as given (what the reference's `layeredCircuit` holds after c.subsetInit()). c / is_assert may be
 * NULL. */
int vp_circuit_from_arrays(int n_layers, const uint64_t* layer_size, const uint8_t* ty, const int32_t* l,
                           const uint64_t* u, const uint64_t* v, const uint64_t* lv, const vp_F* c,
                           const uint8_t* is_assert, const uint64_t* dad_size, const uint64_t* dad_id,
                           vp_circuit** out);
/* K data-parallel instances of the same template (instance-major replication, SURVEY.md 9.3);
 * inputs are drawn like the reference draws them at parse time (main.cpp:188). */
int vp_circuit_replicate(const vp_circuit* c, uint64_t instances, vp_circuit** out);
/* Materialise the instances into one flat circuit (instances == 1), subsets re-derived. */
int vp_circuit_expand(const vp_circuit* c, vp_circuit** out);
void vp_circuit_free(vp_circuit* c);

int vp_circuit_num_layers(const vp_circuit* c);
uint64_t vp_circuit_instances(const vp_circuit* c);
uint64_t vp_circuit_layer_size(const vp_circuit* c, int layer);      /* of ONE instance */
int vp_circuit_bit_length(const vp_circuit* c, int layer);          /* of the replicated layer */
uint64_t vp_circuit_dad_size(const vp_circuit* c, int layer, int src); /* of ONE instance */
int vp_circuit_max_dad_bit_length(const vp_circuit* c, int layer);  /* -1: phase 2 skipped */
uint64_t vp_circuit_total_gates(const vp_circuit* c);               /* non-input gates, all instances */
uint64_t vp_circuit_num_inputs(const vp_circuit* c);                /* instances * layer_size(0) */
/* Export the gates of one template layer (arrays of layer_size entries; any pointer may be NULL). */
int vp_circuit_export_layer(const vp_circuit* c, int layer, uint8_t* ty, int32_t* l, uint32_t* u, uint32_t* v,
                            uint32_t* lv, vp_F* cst, uint8_t* is_assert);
int vp_circuit_export_dad(const vp_circuit* c, int layer, int src, uint32_t* dad_id /* dad_size entries */);
int vp_circuit_get_inputs(const vp_circuit* c, uint64_t* out /* num_inputs */);
int vp_circuit_set_inputs(vp_circuit* c, const uint64_t* in /* num_inputs, each < p */);

/* Challenges in the verifier's draw order (src/verifier.cpp:144-145,196,202,236,278-279) from glibc
 * random() after srand(seed) (fieldElement.cpp:106-124); seed 3396 reproduces F::init(). */
size_t vp_challenge_count(const vp_circuit* c);
int vp_draw_challenges(const vp_circuit* c, unsigned seed, vp_F* out /* vp_challenge_count */);
/* The same generator as a plain stream: the first n values of fieldElement::random() after srand(seed). */
int vp_draw_field(unsigned seed, size_t n, vp_F* out);
/* Prover messages: Vres; per layer top..1: bl(i-1) x (a,b,c), claim_u, [maxDad(i) x (a,b,c), claims_v[0..i)],
 * bl(i-1) x (a,b,c), claim_liu; finally the input-layer MLE. */
size_t vp_transcript_len(const vp_circuit* c);

/* Transcript containers. GKRProof byte stream = the layout of GKRProof::write (src/GKRProof.hpp:23-58; the struct is
 * dead code in the reference, SURVEY.md 9.4): members final_claims_u, final_claims, final_claims_v, polys_u, polys_v,
 * polys, outer vectors indexed by layer id; the reference's undefined poly_proof part is replaced by a trailer
 * {u64 2, Vres, input MLE}. out == NULL: only *len is set. Text dump: "TAG real img" lines (SURVEY.md 9.5). */
int vp_transcript_to_gkrproof(const vp_circuit* c, const vp_F* transcript, unsigned char* out, size_t cap, size_t* len);
int vp_gkrproof_to_transcript(const vp_circuit* c, const unsigned char* bytes, size_t len, vp_F* transcript);
int vp_transcript_text(const vp_circuit* c, const vp_F* transcript, const vp_F* challenges, char* out, size_t cap,
                       size_t* len);

/* ------------------------------------------------------------------ prover
 * One context = one `prover` object (src/prover.h:12-67) on one GPU. */
int vp_create(const vp_circuit* c, int device, vp_ctx** out);
/* Sharded context: this process is `rank` of `world` GPUs of one box; nccl_id is the 128-byte
 * ncclUniqueId shared by all ranks (vp_nccl_unique_id on rank 0, broadcast by the caller). */
int vp_nccl_unique_id(uint8_t out[128]);
int vp_create_sharded(const vp_circuit* c, int device, int rank, int world, const uint8_t nccl_id[128],
                      vp_ctx** out);
void vp_destroy(vp_ctx* ctx);
/* Host-only: how phase (1, 2 = phase 2, 3 = Liu) of `layer` is dealt out to `rank` of `world` GPUs.
 * out: 10 values per table {bits, live, sharded, m, row_lo, row_hi, local_len, present, n_blocks, reversed}:
 * the rank holds the live table entries [row_lo, row_hi). */
int vp_shard_describe(const vp_circuit* c, int world, int rank, int layer, int phase, uint32_t* out, size_t cap,
                      size_t* n_tables);
/* Host-only: index map of a rank holding the table entries [lo, hi): returns 1 and *local if idx belongs to it. */
/* Host-only (no device needed): the instances [lo[l], hi[l]) of layer l that `rank` of a `world`-GPU sharded context
   evaluates -- the hull of what its tables read from layer l and from every layer above it. lo, hi: n_layers entries. */
int vp_shard_eval_ranges(const vp_circuit* c, int world, int rank, uint32_t* lo, uint32_t* hi);
int vp_shard_map_index(uint32_t lo, uint32_t hi, uint32_t idx, uint32_t* local);

/* SHARDED CONTEXTS and the method-by-method API. Every entry point below except vp_get_values also works on a sharded
 * context, as a COLLECTIVE call: all ranks call it in the same order with the same arguments and all get the same
 * results (like the reference's single prover, whose messages every rank's verifier copy sees). A round of a sharded
 * phase folds the rank's own table rows and exchanges 48 bytes per rank (the partial round polynomial, partial add_term
 * included); after the local rounds the remaining <= 2^10 values per table are gathered once and the last rounds run
 * replicated (SURVEY 8(e); src/prover.cpp:436-455 per round). */
/* Upload the witness inputs (instances * layer_size(0) values < p); default: the circuit's own. */
int vp_set_inputs(vp_ctx* ctx, const uint64_t* inputs, size_t n);
/* prover::evaluate (prover.cpp:27-91) + the assert check of the constructor (:16-24). */
int vp_evaluate(vp_ctx* ctx);
/* Copy circuitValue[layer] to the host (layer 0 is what commit_private hands to the PC, :524-530). */
int vp_get_values(vp_ctx* ctx, int layer, vp_F* out, size_t n);

/* prover::Vres (prover.cpp:99-129): MLE of the output layer at r[0..n). */
int vp_vres(vp_ctx* ctx, const vp_F* r, int n, vp_F* out);
/* prover::sumcheckInitAll (:162-170) */
int vp_sumcheck_init_all(vp_ctx* ctx, const vp_F* r_last, int n);
/* prover::sumcheckInit (:177-184): step to the next layer (top -> 1). */
int vp_sumcheck_init(vp_ctx* ctx);
/* prover::sumcheckInitPhase1 (:189-280) / Phase2 (:282-367) / Liu (:369-420; sig has n entries,
 * n >= n_layers - layer + 1). */
int vp_init_phase1(vp_ctx* ctx, const vp_F* assert_random);
int vp_init_phase2(vp_ctx* ctx);
int vp_init_liu(vp_ctx* ctx, const vp_F* sig, int n);
/* prover::sumcheckUpdatePhase1 / Phase2 / LiuUpdate (:422-455): phase = 1, 2, 3. out_abc = the
 * round's quadratic_poly {a,b,c}. */
int vp_round(vp_ctx* ctx, int phase, const vp_F* previous_random, vp_F out_abc[3]);
/* prover::sumcheckFinalize1 (:494-501), Finalize2 (:504-516; claims has `layer` entries),
 * LiuFinalize (:518-521). */
int vp_finalize1(vp_ctx* ctx, const vp_F* previous_random, vp_F* claim);
int vp_finalize2(vp_ctx* ctx, const vp_F* previous_random, vp_F* claims, int n);
int vp_finalize_liu(vp_ctx* ctx, const vp_F* previous_random, vp_F* claim);
/* prover::inner_prod(circuitValue[0], pub, n) as used by commit_public (:532-546). */
int vp_inner_prod(vp_ctx* ctx, const vp_F* pub, size_t n, vp_F* out);
/* prover::inner_prod(a, b, n) for two HOST vectors (the public method, prover.h:40). */
int vp_dot_host(vp_ctx* ctx, const vp_F* a, const vp_F* b, size_t n, vp_F* out);
/* Input-layer MLE at r[0..n): <circuitValue[0], eq(r,.)> without materialising eq on the host. */
int vp_input_mle(vp_ctx* ctx, const vp_F* r, int n, vp_F* out);
/* prover::proofSize() in bytes (:451,:500,:512) and the accumulated device time inside prover
 * entry points in seconds (the analogue of proveTime(), :549-551). */
uint64_t vp_proof_size_bytes(const vp_ctx* ctx);
double vp_prove_seconds(const vp_ctx* ctx);

/* ------------------------------------------------------------------ whole proof, no per-round host sync
 * The reference verifier's challenges do not depend on prover messages (SURVEY.md 0), so the whole
 * stream can be handed over up front. vp_prove runs evaluate + every phase of every layer on the
 * device and returns the transcript (vp_transcript_len entries).
 * host_io != 0: `inputs`/`challenges`/`transcript` are HOST buffers (copied inside the call).
 * host_io == 0: inputs already uploaded with vp_set_inputs and challenges with vp_set_challenges;
 *               the transcript stays on the device until vp_get_transcript. */
int vp_set_challenges(vp_ctx* ctx, const vp_F* challenges, size_t n);
int vp_prove(vp_ctx* ctx, int host_io, const uint64_t* inputs, size_t n_inputs, const vp_F* challenges,
             size_t n_challenges, vp_F* transcript, size_t transcript_cap);
/* Sharded contexts: a rank only uploads the witness of the data-parallel instances [first, end) it evaluates (its own
 * K/world slice plus the few neighbours its tables read, vp_shard_eval_ranges). vp_prove_local is vp_prove(host_io=1)
 * for a caller that holds just that slice: local_inputs = (end - first) * layer_size(0) values, instance-major.
 * On an unsharded context the range is [0, instances) and the two calls are the same. */
int vp_input_range(const vp_ctx* ctx, uint64_t* first_instance, uint64_t* end_instance);
int vp_prove_local(vp_ctx* ctx, const uint64_t* local_inputs, size_t n_local, const vp_F* challenges, size_t n_challenges,
                   vp_F* transcript, size_t transcript_cap);
/* ------------------------------------------------------------------ polynomial commitment, commit phase (SURVEY 8(f) N1)
 * Replaces poly_commit_prover::commit_private_array (lib/virgo/src/poly_commit.h:41-124: per-slice inverse FFT + 32x
 * Reed-Solomon extension, RS_polynomial.cpp:26-220), fri::request_init_commit (fri.cpp:36-139: SHA3-256 leaf chains,
 * my_hhash.h:27-33) and merkle_tree_prover::create_tree (merkle_tree.cpp:7-51) as prover::commit_private uses them
 * (prover.cpp:524-530: circuitValue[0] padded to 2^bitLength, ONE zero mask element -- other masks return VP_ERR_ARG).
 * root = the 32-byte Merkle root (the __hhash_digest commit_private returns). The codeword array l_eval
 * [65 * slice_size], the leaf hashes [slice_size / 2 * 32 B] and the Merkle tree [slice_size * 32 B, array heap, node 1 =
 * root] stay on the device; vp_commit_export copies them out for the reference's CPU opening phase (any pointer may be
 * NULL). slice_size = 2^(bitLength(0) - 1). Needs bitLength(0) >= 6; unsharded contexts.
 * Not reproduced: with bitLength(0) == 8 the reference's 4-point inverse FFT returns uninitialised scratch memory
 * (RS_polynomial.cpp:100: `blk_size / packed_size * 2` iterations == 0); this library computes the transform. */
int vp_commit_private(vp_ctx* ctx, const vp_F* mask, size_t n_mask, uint8_t root[32]);
int vp_commit_export(vp_ctx* ctx, vp_F* l_eval, uint8_t* leaf_hash, uint8_t* tree);
uint64_t vp_commit_slice_size(const vp_ctx* ctx);
float vp_last_commit_ms(const vp_ctx* ctx);   /* device time of the last vp_commit_private */
/* prover::commit_public (prover.cpp:542-546) -> commit_public_array (poly_commit.h:126-349) after vp_commit_private: pub =
 * the public array (the verifier's eq table over r_liu, verifier.cpp:367-381; n <= 2^bitLength(0) canonical elements), mask
 * = the public mask (one zero: others return VP_ERR_ARG). Encodes pub like the private array, gets the 2n coefficients
 * of l*q per slice from its values on the 2n-th roots, extends the quotient h (l q = g + (x^n - 1) h) to all points, builds
 * the virtual oracle (g - const) n / x and all_sum[65], and commits to h_eval_arr (second Merkle tree): root_h.
 * vp_commit_public_export: h_eval_arr [65 * slice_size], virtual_oracle_witness [64 * slice_size] (interleaved like
 * fri::virtual_oracle_witness), leaf hashes and tree of the second commitment (any pointer may be NULL).
 * Not reproduced: bitLength(0) == 7 (the reference's 4-point inverse FFT, see above). */
int vp_commit_public(vp_ctx* ctx, const vp_F* pub, size_t n, const vp_F* mask, size_t n_mask, uint8_t root_h[32], vp_F all_sum[65]);
int vp_commit_public_export(vp_ctx* ctx, vp_F* h_eval, vp_F* vow, uint8_t* leaf_hash, uint8_t* tree);
/* The 64 codewords of commitment `which` (0: after vp_commit_private, 1: after vp_commit_public) in the layout of
 * fri::witness_rs_codeword_interleaved[which] (fri.cpp:69-96): out[(j << 7) | (slice << 1) | h] = codeword[slice][j + h *
 * slice_size / 2], 64 * slice_size elements; transposed on the device. Before the first vp_fri_commit_steps call. */
int vp_commit_export_interleaved(vp_ctx* ctx, int which, vp_F* out);
/* The same on a host array of n canonical field elements, zero-padded to 2^log_len (6 <= log_len <= 30). */
int vp_pc_commit(int device, const vp_F* array, size_t n, int log_len, uint8_t root[32], vp_F* l_eval, uint8_t* leaf_hash,
                 uint8_t* tree, float* device_ms);
int vp_pc_commit_public(int device, const vp_F* array, size_t n, const vp_F* pub, size_t n_pub, int log_len, uint8_t root_l[32],
                        uint8_t root_h[32], vp_F all_sum[65], vp_F* h_eval, vp_F* vow, float* device_ms);

/* FRI commit phase (fri::commit_phase_step, lib/virgo/src/fri.cpp:289-418, as poly_commit_prover::commit_phase drives it,
 * vpd_verifier.cpp:43-73) on the virtual oracle vp_commit_public left on the device. One step per fold challenge: every
 * slice's codeword f on the M-th roots becomes g(x^2) = (f(x) + f(-x))/2 + r (f(x) - f(-x))/(2x) on the M/2-th roots, the
 * M/4 leaves (one pair of opposite points of all 64 slices + the zero mask pair each) are hashed and the level's tree
 * built; roots[k] = the root after step k. vp_fri_steps(ctx) = bitLength(0) - 6 steps leave 32 points per slice (the
 * reference stops there). vp_fri_export_level: level lvl's codewords in the layout of fri::cpd.rs_codeword[lvl]
 * (64 * (slice_size >> (lvl+1)) elements) and its tree (array heap, (slice_size >> (lvl+1)) nodes of 32 bytes); any pointer
 * may be NULL. vp_fri_restart: back to step 0 on the same virtual oracle. Challenges must be canonical. */
int vp_fri_commit_steps(vp_ctx* ctx, const vp_F* randomness, int n_steps, uint8_t* roots /* n_steps * 32 */);
int vp_fri_steps(const vp_ctx* ctx);
int vp_fri_restart(vp_ctx* ctx);
int vp_fri_export_level(vp_ctx* ctx, int lvl, vp_F* rs_codeword, uint8_t* merkle);
/* Stand-alone: both commitments of host arrays (as vp_pc_commit_public), then n_steps <= log_len - 6 FRI steps.
 * codes / trees (may be NULL): the levels back to back. 7 <= log_len <= 30. */
int vp_pc_fri(int device, const vp_F* array, size_t n, const vp_F* pub, size_t n_pub, int log_len, const vp_F* randomness, int n_steps,
              uint8_t root_l[32], uint8_t root_h[32], uint8_t* roots, vp_F* codes, uint8_t* trees, float* device_ms);

/* ------------------------------------------------------------------ the commitment's inner GKR (SURVEY 8(f) N4)
 * fft_circuit_gkr::fft_gkr (lib/virgo/src/fft_circuit_GKR.cpp:833-849), which poly_commit_verifier::verify_poly_commitment
 * runs once per opening (vpd_verifier.cpp:92): prover and verifier of a layered GKR over a fixed circuit family -- the eq
 * table of a random point, lg_size inverse-FFT butterfly layers, a scaling, 64 x 2^lg_size products with the powers of 64
 * random points and their row sums -- walked from the outputs back to the eq table with 2 + 2 lg_size sumchecks. The
 * reference draws all randomness with fieldElement::random() and none of it depends on a prover message; here the caller
 * passes it as one array in the reference's draw order:
 *   r[lg] | x[64] | r_0[lg+10] | r_1[lg+10] | addition layer: r_u[lg+6], r_v[lg+6] | mult layer: r_u[lg], r_v[lg] |
 *   per butterfly layer (lg of them): r_u[lg], r_v[lg], alpha, beta          (vp_fft_gkr_rnd_count(lg) elements, canonical)
 * The prover side (circuit evaluation, all sumcheck tables and rounds) runs on the device without a host round trip; the
 * verifier's claim chain and closed-form wiring predicates run on the host afterwards.
 * Outputs: proof_size = the reference's `ps` (48 bytes per round + extension_gkr's count), ok = 1 if every verifier check
 * passed (the reference prints "Error, fft gkr failed" otherwise), verifier_seconds / prover_seconds = its `vt` / `pt`;
 * optional (NULL to skip): layers = E, F_{lg-1}..F_0, S (2^lg each), P (64 * 2^lg), O (64); polys = 3 elements per round in
 * protocol order (vp_fft_gkr_poly_count(lg) rounds); claims = the running claim a_0, after the addition / mult /
 * intermediate layer, after every butterfly layer, then the final alpha, beta (4 + lg + 2 elements). 1 <= lg_size <= 24. */
/* The two sumcheck objects of a size (lg_size and lg_size + 6 variables: device tables of 3 x 2 x 16 bytes per entry) are kept
 * per (device, lg_size) for the next call; vp_fft_gkr_release() frees them. Calls are serialised by an internal lock. */
void vp_fft_gkr_release(void);
size_t vp_fft_gkr_rnd_count(int lg_size);
size_t vp_fft_gkr_poly_count(int lg_size);
int vp_fft_gkr(int device, int lg_size, const vp_F* rnd, size_t n_rnd, vp_F* layers, vp_F* polys, size_t polys_cap, vp_F* claims,
               int* proof_size, int* ok, double* verifier_seconds, double* prover_seconds, float* device_ms);

/* ------------------------------------------------------------------ Fiat-Shamir mode (SURVEY 8(f) N4)
 * The reference ships a hash-based challenge source, transcriptCache (lib/virgo/src/transcriptCache.hpp:14-50: a byte
 * pool hashed with SHA3-256 per challenge, challenge = first two digest words mod p), but never calls it. This mode uses
 * exactly that class, fed with seed[32] and then every prover message (16 bytes {u64 real, u64 img} each) in emission
 * order; a round's challenge is drawn right after the round's polynomial was stored (order: host/fiat_shamir.h). Only the
 * one-round-per-launch path applies (a challenge depends on the previous message). vp_prove_fs uses the resident inputs
 * and returns the transcript and, optionally, the challenges it drew (usual layout, unused slots zero);
 * vp_fs_challenges recomputes them from a transcript alone; vp_verify_fs = vp_fs_challenges + vp_verify (fail_code 7:
 * a non-canonical transcript element). Not parity-bound to the reference (it has no such mode); pinned against the
 * oracle's restatement of transcriptCache.
 * The seed MUST be a digest of the statement (circuit, inputs, outputs): this mode absorbs nothing else, so with a seed
 * that does not commit to them a prover can fix a transcript first and pick inputs that pass the input-layer check
 * afterwards, and the verifier never learns the outputs. vp_prove_fs_bound / vp_verify_fs_bound below derive the seed
 * from the statement; vp_prove_fs(ctx, statement) is the same proof.
 * On an unsharded context the whole proof is queued on the device (the transcript cache is a device buffer, every
 * round's challenge is drawn inside the sumcheck phase kernel); sharded contexts draw on the host between rounds. */
int vp_prove_fs(vp_ctx* ctx, const uint8_t seed[32], vp_F* transcript, size_t transcript_cap, vp_F* challenges, size_t challenges_cap);
int vp_fs_challenges(const vp_circuit* c, const uint8_t seed[32], const vp_F* transcript, size_t n, vp_F* challenges, size_t cap);
int vp_verify_fs(vp_ctx* ctx, const uint8_t seed[32], const vp_F* transcript, size_t n, int* accept, int* fail_code, int* fail_layer);

/* ------------------------------------------------------------------ statement-bound Fiat-Shamir proofs
 * Every integer is little-endian; H = SHA3-256 (FIPS 202).
 * Vector root R(bytes): zero-pad bytes to 64 * 2^k bytes, 2^k the smallest power of two >= max(1, ceil(len / 64)); leaf j =
 *   H(64-byte block j); array-heap Merkle tree with node = H(left | right), leaves at nodes 2^k .. 2^(k+1) - 1, root = node 1
 *   (one leaf: the root is that leaf's hash).
 * Inputs root  = R over circuitValue[0] as the prover holds it (instances * layer_size(0) canonical elements, 16 bytes
 *   {re, im} each, after vp_set_inputs' reading rules). Outputs root = R over circuitValue[n-1] (instances * layer_size(n-1)).
 * Circuit digest = R(circuit_bytes), from what vp_circuit_export_layer / vp_circuit_export_dad return:
 *   "VPCIRC01" | u64 n_layers | u64 instances | u64 layer_size(i), i = 0..n-1 |
 *   for i = 1..n-1, every template gate, packed 34 bytes: u8 ty, u8 is_assert, i32 l, u32 u, u32 v, u32 lv, u64 c.re, u64 c.im |
 *   for i = 1..n-1, s = 0..i-1: u64 dad_size(i, s) | u32 dad_id[dad_size(i, s)].
 *   Layer 0 contributes its size only (its values are bound by the inputs root). A replicated circuit is hashed as its
 *   template + K: vp_circuit_expand of it is another circuit object with another digest.
 * Statement = H("VPSTMT01" | circuit digest | u64 n_inputs | inputs root | u64 n_outputs | outputs root | context[32]) (152
 *   bytes); context = 32 caller-chosen bytes (application tag, session id; may be zero).
 * vp_prove_fs_bound(ctx, context) is, by definition, vp_prove_fs(ctx, statement).
 * vp_statement_digest: the four digests of the context's resident inputs (the circuit is evaluated first if needed);
 *   circuit / inputs / outputs may be NULL. The circuit digest is computed once per context (on the device, from bytes
 *   serialised on the host) and kept.
 * vp_prove_fs_bound: the proof; transcript / challenges as vp_prove_fs; statement (may be NULL) = the seed it used.
 * vp_verify_fs_bound: the verifier's side, from its own circuit and resident inputs and the CLAIMED outputs (n_outputs =
 *   instances * layer_size(n-1) canonical elements, else VP_ERR_ARG): computes the statement, the challenges
 *   (vp_fs_challenges), checks Vres == MLE(outputs)(r_out) (fail_code 8), then vp_verify's checks. fail_code 7: a
 *   non-canonical transcript element.
 * vp_fs_round_stamps: %globaltimer stamps (ns) of block 0 in the last device Fiat-Shamir proof, 4 per sumcheck round in
 *   proof order {round start, own fold work done, polynomial reduced (after the grid barrier), challenge drawn};
 *   *n_rounds = the number of rounds; out may be NULL (cap >= 4 * rounds otherwise).
 * Sharded contexts: all of these return VP_ERR_ARG. */
int vp_statement_digest(vp_ctx* ctx, const uint8_t context[32], uint8_t circuit[32], uint8_t inputs[32], uint8_t outputs[32],
                        uint8_t statement[32]);
int vp_prove_fs_bound(vp_ctx* ctx, const uint8_t context[32], vp_F* transcript, size_t cap, vp_F* challenges, size_t ch_cap,
                      uint8_t statement[32]);
int vp_verify_fs_bound(vp_ctx* ctx, const uint8_t context[32], const vp_F* outputs, size_t n_outputs, const vp_F* transcript, size_t n,
                       int* accept, int* fail_code, int* fail_layer);
int vp_fs_round_stamps(vp_ctx* ctx, unsigned long long* out, size_t cap, size_t* n_rounds);

/* Aggregate statement-bound proofs: ONE Fiat-Shamir proof that binds B statements of one circuit, each with its own inputs,
 * outputs and 32-byte context. The context's circuit is replicate(template, N); for 1 <= B <= 65535 with B | N, K = N / B,
 * statement b covers instances [b K, (b + 1) K) of the resident inputs and of the output layer:
 *   statement_b = H("VPSTMT01" | circuit digest of template + K (the VPCIRC01 bytes with u64 instances = K) | u64 K * S_0 |
 *                   R(statement b's slice of circuitValue[0]) | u64 K * S_out | R(its slice of the output layer) | context_b),
 *   i.e. vp_statement_digest on a context of replicate(template, K) (the template itself when K = 1) holding inputs b, with
 *   context b: exactly the seed a single bound proof of statement b would use;
 *   aggregate = H("VPAGGR01" | u64 B | R(statement_0 | ... | statement_{B-1})) (48 bytes hashed; domain-separated from
 *   VPSTMT01, so the aggregate of one statement is not that statement's seed).
 * vp_prove_fs_aggregate(ctx, B, contexts) is, by definition, vp_prove_fs(ctx, aggregate): its rounds grow with log B, not
 * with B. contexts: B * 32 bytes; statements (may be NULL): B * 32 bytes, statement-major; aggregate (may be NULL in the
 * prover): 32 bytes.
 * vp_aggregate_digest: the statements and the aggregate of the resident inputs (evaluated first if needed).
 * vp_prove_fs_aggregate: on the context's own buffers, like vp_prove_fs_bound: the resident challenges are the proof's
 *   afterwards (a later vp_verify sees them); vp_last_prove_ms / vp_last_prove_launches describe the call; VP_ERR_ASSERT
 *   when an is_assert gate is non-zero.
 * vp_verify_fs_aggregate: vp_verify_fs_bound's order and codes with the aggregate as the seed, from the resident inputs and
 *   the CLAIMED outputs (n_outputs = N * layer_size(n-1) canonical elements): fail_code 7 a non-canonical transcript
 *   element, 8 Vres != MLE(outputs)(r_out), then vp_verify's checks.
 * VP_ERR_ARG: B = 0, B > 65535, B not dividing N, short buffers, wrong counts, non-canonical outputs, sharded contexts.
 * On the device, on the context's stream: the B inputs roots and the B outputs roots in one pc_vector_root pass each, the B
 * statements by one thread each (k_fs_statements), R over them, then one thread hashes the aggregate into the pool; no
 * launch per statement and no hashing of statement data on the host. The circuit digest of template + K is kept for the
 * last K. */
int vp_aggregate_digest(vp_ctx* ctx, size_t B, const uint8_t* contexts, uint8_t* statements, uint8_t aggregate[32]);
int vp_prove_fs_aggregate(vp_ctx* ctx, size_t B, const uint8_t* contexts, vp_F* transcript, size_t cap, vp_F* challenges, size_t ch_cap,
                          uint8_t* statements, uint8_t aggregate[32]);
int vp_verify_fs_aggregate(vp_ctx* ctx, size_t B, const uint8_t* contexts, const vp_F* outputs, size_t n_outputs, const vp_F* transcript,
                           size_t n, int* accept, int* fail_code, int* fail_layer);

/* B independent statement-bound proofs over this context's circuit (template + K, as the context was created), in one pass.
 * inputs: B * vp_circuit_num_inputs values, statement-major, read with vp_circuit_set_inputs' rules (0 <= x < p; others VP_ERR_ARG).
 * contexts: B * 32 bytes. transcripts: B * n_tr (cap >= that), statement-major; challenges (may be NULL): B * n_chal;
 * statements (may be NULL): B * 32 bytes.
 * Proof b is, bit for bit, vp_prove_fs_bound on this circuit with inputs b and context b.
 * The context's resident inputs, values, transcript and challenges are not changed.
 * VP_ERR_ASSERT: an is_assert gate is non-zero in some statement; vp_last_error names the first such b.
 * Sharded contexts: VP_ERR_ARG.
 * The statements share the circuit's wiring, plans and digest and one sequence of launches: every kernel of the proof runs
 * all B statements at once (statement b in blockIdx.z), so the launch count does not grow with B (the sumcheck phase
 * kernel, a cooperative launch, runs in chunks of statements when B exceeds the blocks that can be co-resident). The
 * per-statement buffers live in a slab kept on the context for the next call (grown when needed, freed by vp_destroy).
 * vp_last_prove_ms / vp_last_prove_launches describe the batch; vp_fs_round_stamps are statement 0's. */
int vp_prove_fs_bound_batch(vp_ctx* ctx, size_t B, const uint64_t* inputs, size_t n_inputs, const uint8_t* contexts,
                            vp_F* transcripts, size_t cap, vp_F* challenges, size_t ch_cap, uint8_t* statements);
/* The output layers of the last successful vp_prove_fs_bound_batch: B * (instances * layer_size(n-1)) elements, statement-major
 * (what a verifier passes to vp_verify_fs_bound(_batch) as the claimed outputs). Valid until the next batch call on the
 * context (vp_prove_fs_bound_batch or vp_verify_fs_bound_batch). VP_ERR_ARG: no batch has run, the last batch failed,
 * or cap is too small. */
int vp_last_batch_outputs(vp_ctx* ctx, vp_F* out, size_t cap);
/* B statement-bound proofs of this context's circuit checked in one pass. inputs / contexts as vp_prove_fs_bound_batch;
 * outputs: B * (instances * layer_size(n-1)) claimed outputs, statement-major; transcripts: B * n_tr, statement-major.
 * accept / fail_code / fail_layer: B entries each (fail_code / fail_layer may be NULL); challenges (may be NULL, ch_cap >=
 * B * n_chal): statement-major.
 * Verdict b is, exactly, (accept, fail_code, fail_layer) of vp_verify_fs_bound(context b, outputs b, transcript b) on a
 * context whose resident inputs are inputs b, and challenges b are what vp_fs_challenges derives from statement b and
 * transcript b. A non-canonical transcript element rejects that statement alone (code 7, layer 0; its challenges are
 * zero). VP_ERR_ARG: B not in [1, 65535], a count that does not match B, an input >= p or a non-canonical output
 * (vp_last_error names the statement), a sharded context.
 * The context's resident inputs, values, transcript and challenges are not changed (vp_verify_fs_bound, in contrast,
 * leaves the proof's challenges resident).
 * On the device: one upload, the roots and statements of all B statements (as in the batch prover), every challenge
 * replayed from the transcripts by one warp per statement (k_fs_replay), then the verifier's O(#gates) sums, the
 * outputs' MLE at r_out and the input MLE of every statement, one sequence of launches for all B (the launch count
 * does not grow with B); one read-back of the sums and the challenges, then the round checks on the host. Memory: the
 * batch prover's slab for B statements (vp_prove_fs_bound_batch), plus the verifier's sums per statement.
 * vp_last_prove_ms / vp_last_prove_launches describe the call. */
int vp_verify_fs_bound_batch(vp_ctx* ctx, size_t B, const uint64_t* inputs, size_t n_inputs, const uint8_t* contexts,
                             const vp_F* outputs, size_t n_outputs, const vp_F* transcripts, size_t n_tr,
                             int* accept, int* fail_code, int* fail_layer, vp_F* challenges, size_t ch_cap);
/* The two batch calls above on arrays in DEVICE memory, as one stage of a GPU pipeline: every array is device (or managed)
 * memory of the context's device, statement-major in the layout of its host counterpart: inputs B * num_inputs (u64),
 * contexts B * 32 bytes, transcripts B * n_tr, challenges B * n_chal, outputs B * (instances * layer_size(n-1)),
 * statements B * 32 bytes, status / accept / code / layer B int32 each. May be NULL: the prover's challenges, outputs and
 * statements; the verifier's code, layer and challenges. The library cannot see the arrays' sizes: the caller guarantees
 * them.
 * Ordering: the work is queued on the context's stream (vp_set_stream) after whatever was queued there before, and the call
 * returns once it is queued; the results are in the caller's arrays once the stream has passed the call.
 * Checked when called (VP_ERR_ARG): 1 <= B <= 65535, every non-NULL array device or managed memory of the context's device
 * (cudaPointerGetAttributes), vp_F arrays 16-byte aligned and the others 8-byte aligned, an unsharded context.
 * A failing statement never fails the call and changes no other statement's results; every failing statement is reported.
 * Prover: status[b] = 0 proved (transcript, challenges, outputs and statement b are bit for bit vp_prove_fs_bound_batch's,
 *   so vp_prove_fs_bound's, for inputs b and context b); 1 an input of statement b is not < p (its inputs are proved as
 *   zeros, the caller's array is not touched); 2 + l an is_assert gate of layer l is non-zero in statement b (the layer
 *   VP_ERR_ASSERT names). When status[b] != 0 all four of b's result rows are zero.
 * Verifier: (accept, code, layer)[b], checked in this order: code 9 an input or claimed output of statement b is not
 *   canonical (layer 0; the host-memory call fails with VP_ERR_ARG instead), 7 a non-canonical transcript element, 8 Vres
 *   is not the claimed outputs' MLE at r_out, then vp_verify's codes 1-6. Apart from code 9 the verdicts and the challenges
 *   are vp_verify_fs_bound_batch's; a statement with code 7 or 9 has zero challenges. The claim chain runs on the device,
 *   one thread per statement (vp_verify_fs_bound_batch keeps its host loop).
 * After one call of a kind with B statements (warm-up: the slab, the circuit digest and the per-context tables), a call of
 * the same kind with at most B statements allocates nothing and does not synchronise with the host. vp_last_prove_launches
 * describes the call; vp_last_prove_ms waits for the call's end when it is read. The context's resident inputs, values,
 * transcript and challenges are not changed; vp_last_batch_outputs has nothing after a device call (use the outputs
 * array). CUDA graph capture is not supported. */
int vp_prove_fs_bound_batch_dev(vp_ctx* ctx, size_t B, const uint64_t* d_inputs, const uint8_t* d_contexts,
                                vp_F* d_transcripts, vp_F* d_challenges, vp_F* d_outputs, uint8_t* d_statements,
                                int32_t* d_status);
int vp_verify_fs_bound_batch_dev(vp_ctx* ctx, size_t B, const uint64_t* d_inputs, const uint8_t* d_contexts,
                                 const vp_F* d_outputs, const vp_F* d_transcripts,
                                 int32_t* d_accept, int32_t* d_code, int32_t* d_layer, vp_F* d_challenges);

/* Self-test of the device-only arithmetic paths of csrc/field.cuh (inline-PTX carry chains, mul.wide / mad.wide):
   runs one routine on n caller-provided operand triples and returns the results, so that tests can feed edge values
   (0, 1, p-1, p, limb boundaries) and compare with big-integer arithmetic.  op: 0 weak fold a + c*(b-a); 1 the same for
   base-field a, b; 2 lazy dot product sum a_i*b_i -> out[0]; 3 {fp_reduce_ut_weak(a.re, a.im, b.re), fp_weak(b.im)};
   4 c + a*b (weak); 5 c + a*b.re (weak); 6 lazy sum (b_i - a_i)*c_i.re -> out[0]; 7 like 0 with the folded difference. */
int vp_selftest_field(int device, int op, const vp_F* a, const vp_F* b, const vp_F* c, vp_F* out, size_t n);

/* Verifier (SURVEY 8(f) N2): replaces verifier::verify's checks, src/verifier.cpp:134-337, on a finished transcript:
   the O(#gates) sums of predicatePhase1/2 (:63-113) and verifyLiu's gr (:311-323) run on the device, the round
   checks / getFinalValue (:115-132) / Liu check on the host. Uses the context's circuit, its resident inputs
   (vp_set_inputs or vp_prove with host_io) and challenge stream (vp_set_challenges / vp_prove). *accept = 1, or 0 with
   *fail_code = 1 phase-1 round, 2 phase-2 round, 3 layer final value, 4 Liu round, 5 Liu final, 6 input layer, and
   *fail_layer (either may be NULL). The polynomial-commitment opening (verifyPoly) is out of scope: the input-layer
   MLE is recomputed from the inputs. On a sharded context this is a COLLECTIVE call: every rank passes the same
   transcript, sums the gates of its own slice of the instances, the partial sums meet in one all-gather and every
   rank returns the same verdict. */
int vp_verify(vp_ctx* ctx, const vp_F* transcript, size_t n, int* accept, int* fail_code, int* fail_layer);
int vp_get_transcript(vp_ctx* ctx, vp_F* transcript, size_t cap);
/* Device-side time of the last vp_prove (CUDA events on the context's stream), milliseconds. */
float vp_last_prove_ms(const vp_ctx* ctx);
/* Number of kernel launches issued by the last vp_prove. */
uint64_t vp_last_prove_launches(const vp_ctx* ctx);
/* Run every kernel of the context on the caller's stream (cudaStream_t; NULL: back to an own stream). */
int vp_set_stream(vp_ctx* ctx, void* cuda_stream);
/* Per-kernel-class device timing (CUDA events around every launch while on). Classes, in order:
 * 0 round(fold) [K6], 1 round(first), 2 phase-1 init [K3], 3 phase-2 init [K4], 4 Liu init [K5],
 * 5 evaluate [K1], 6 other. bytes = algorithmic bytes of the launches (DESIGN.md). */
int vp_set_profiling(vp_ctx* ctx, int on);
/* Whole-proof mode runs phase 1, phase 2 and the Liu phases of vp_prove on up to three concurrent streams ("lanes",
   DESIGN.md). lanes = 1 runs them one after the other (used by bench.py's instrumented pass so that a launch's
   CUDA-event duration is its own), 2 = Liu phases on their own lane, 3 = one lane per phase kind, 6 = two sets of
   three lanes taking alternate layers (the default on unsharded contexts). Returns the setting in force. */
int vp_set_lanes(vp_ctx* ctx, int lanes);
int vp_get_profile(vp_ctx* ctx, double* ms, double* bytes, uint64_t* launches, int n_classes);
/* The context's CUDA stream (cudaStream_t) so callers can bracket it with their own events. */
void* vp_stream(vp_ctx* ctx);

/* ------------------------------------------------------------------ stand-alone sumcheck (config C2)
 * Three tables V, add, mult of 2^log_n entries (device-resident copies are made once); runs the
 * log_n rounds of sumcheckUpdateEach with challenges r[0..log_n) and returns 3*log_n + 3 values:
 * per round (a,b,c), then the three fully-folded table values. */
typedef struct vp_sumcheck vp_sumcheck;
int vp_sumcheck_create(int log_n, int device, vp_sumcheck** out);
int vp_sumcheck_load(vp_sumcheck* s, const vp_F* V, const vp_F* add, const vp_F* mult); /* host -> device */
int vp_sumcheck_fill_random(vp_sumcheck* s, uint64_t seed);  /* SplitMix64 per entry, on device */
int vp_sumcheck_export(vp_sumcheck* s, vp_F* V, vp_F* add, vp_F* mult);  /* device -> host (pristine copy) */
int vp_sumcheck_run(vp_sumcheck* s, const vp_F* r, vp_F* out /* 3*log_n+3 */, float* device_ms);
/* Same outputs, all rounds in one cooperative launch, two rounds per pass (the challenges are all known). */
int vp_sumcheck_run_fused(vp_sumcheck* s, const vp_F* r, vp_F* out, float* device_ms);
/* profiling aid: ns time stamps of block 0 at {pass start, work done, barrier passed, pass end} per pass of the last fused run */
int vp_sumcheck_pass_stamps(vp_sumcheck* s, unsigned long long* out, int n);
/* per-round device time of the last vp_sumcheck_run (log_n floats, ms) */
int vp_sumcheck_round_ms(vp_sumcheck* s, float* out);
void vp_sumcheck_destroy(vp_sumcheck* s);

#ifdef __cplusplus
}
#endif
#endif
