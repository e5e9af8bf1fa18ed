// Commit phase of Virgo's polynomial commitment on the device (SURVEY 8(f) N1): internal C++ interface between
// pc_commit.cu (kernels + driver) and engine.cu (the context-level C ABI entry points).
// Replaces, for the GKR prover's use of it (prover.cpp:524-530: one zero mask element):
//   poly_commit_prover::commit_private_array   lib/virgo/src/poly_commit.h:41-124
//   vpd_prover_init / fri::request_init_commit lib/virgo/src/vpd_prover.cpp:9-14, fri.cpp:36-139
//   merkle_tree_prover::create_tree            lib/virgo/src/merkle_tree.cpp:7-51
//   my_hhash (SHA3-256 of 64-byte blocks)      lib/virgo/src/my_hhash.h:27-33
//   poly_commit_prover::commit_public_array    lib/virgo/src/poly_commit.h:126-349
//   fri::commit_phase_step                     lib/virgo/src/fri.cpp:289-418
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "field.cuh"

namespace vp {

struct PcCommit;   // device buffers of one commitment (codeword array, leaf hashes, Merkle tree)

// log_len: the committed array has 2^log_len entries (>= 6: 64 slices). Throws std::runtime_error on CUDA failure.
PcCommit* pc_create(int device, int log_len);
void pc_destroy(PcCommit* p);
// d_array: n_valid field elements on the device (the rest of the 2^log_len entries are zero). Runs on `stream`,
// leaves the Merkle root in root[32] (host) after synchronising the stream. Returns the device time in ms.
float pc_commit(PcCommit* p, const F* d_array, size_t n_valid, cudaStream_t stream, uint8_t root[32]);
size_t pc_slice_size(const PcCommit* p);
// copies to the host (any pointer may be null): l_eval [65 * slice_size], leaf hashes [slice_size / 2 * 32 B],
// Merkle tree [slice_size * 32 B] as the array heap of merkle_tree.cpp (node 1 = root, node 0 unused = zero)
void pc_export(PcCommit* p, cudaStream_t stream, F* l_eval, uint8_t* leaf_hash, uint8_t* tree);
// commit_public_array (lib/virgo/src/poly_commit.h:126-349, zero masks) on the object pc_commit ran on: d_pub = the
// public array (n_valid elements on the device, zero-padded). Leaves the root of the second commitment (h) in root_h and
// all_sum[65] on the host. pc_export_public: h_eval_arr [65 N], virtual oracle [64 N], leaf hashes, tree of h.
float pc_commit_public(PcCommit* p, const F* d_pub, size_t n_valid, cudaStream_t stream, uint8_t root_h[32], F all_sum_host[65]);
void pc_export_public(PcCommit* p, cudaStream_t stream, F* h_eval, F* vow, uint8_t* leaf_hash, uint8_t* tree);
// FRI commit phase (fri::commit_phase_step, lib/virgo/src/fri.cpp:289-418, driven by poly_commit_prover::commit_phase,
// vpd_verifier.cpp:43-73) on the virtual oracle pc_commit_public left on the device: one step per fold challenge r;
// pc_fri_steps = log_len - 6 steps bring the 64 codewords down to 32 points each. pc_fri_steps_run returns the device time
// in ms and leaves every level's Merkle root in roots. pc_fri_export: level lvl's codewords (64 * (slice_size >> (lvl+1)) elements in
// the layout of fri::cpd.rs_codeword[lvl]) and tree (array heap of (slice_size >> (lvl+1)) nodes).
int pc_fri_steps(const PcCommit* p);
int pc_fri_steps_done(const PcCommit* p);
void pc_fri_restart(PcCommit* p);
float pc_fri_steps_run(PcCommit* p, const F* r, int n, cudaStream_t stream, uint8_t* roots);   // n steps, roots[n * 32]
void pc_fri_export(PcCommit* p, cudaStream_t stream, int lvl, F* code, uint8_t* tree);
// the codewords of commitment `which` (0: l_eval, 1: h_eval_arr) in the layout of fri::witness_rs_codeword_interleaved
// (fri.cpp:69-96): out[(j << 7) | (slice << 1) | h] = eval[slice][j + h * slice_size / 2], 64 * slice_size elements
void pc_export_interleaved(PcCommit* p, cudaStream_t stream, int which, F* out);
uint64_t pc_launches(const PcCommit* p);

// Merkle root R of a vector of n_words little-endian words on the device (the statement digest of the Fiat-Shamir mode,
// include/virgo_b200.h): the words zero-padded to 2^k 64-byte leaves (2^k the smallest power of two >= max(1, ceil(n_words /
// 8))), leaf j = SHA3-256(block j), an array-heap tree with node = SHA3-256(left | right), root = node 1 (with one leaf: that
// leaf's hash). d_scratch: pc_vector_root_scratch(n_words) bytes; the 32-byte root goes to d_root (device). Asynchronous on
// `st`; returns the number of kernel launches.
// n_vec > 1: the roots of n_vec vectors of n_words words each, lying end to end from d_words, in the same launches;
// d_scratch holds n_vec * pc_vector_root_scratch(n_words) bytes and root v goes to d_root + v * root_stride bytes.
size_t pc_vector_root_scratch(size_t n_words);
int pc_vector_root(const uint64_t* d_words, size_t n_words, uint64_t* d_scratch, uint8_t* d_root, cudaStream_t st, uint32_t n_vec = 1,
                   size_t root_stride = 0);

}  // namespace vp
