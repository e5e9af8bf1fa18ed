// Transcript containers (host side).
//  * GKRProof byte stream: the layout of GKRProof::write in the reference's (dead) src/GKRProof.hpp:23-58 --
//    for each member in the order final_claims_u, final_claims, final_claims_v, polys_u, polys_v, polys:
//    u64 count, then (nested vectors: per inner vector u64 len, then) the raw elements; F = 16 B {real, img}
//    little endian, quadratic_poly = 48 B {a, b, c}. Outer vectors are indexed by layer id (n_layers entries,
//    entry 0 empty). The reference's poly_proof part (a type that does not exist in its tree) is replaced by
//    a two-element trailer: u64 2, Vres, input-layer MLE.
//  * text dump: "TAG real img" per line in emission order (SURVEY.md 9.4/9.5): VRES; per round CH,PA,PB,PC;
//    CH,CLAIM_U; CLAIM_V x layer; CH,CLAIM_LIU; INPUT_MLE.
#pragma once
#include <string>
#include <vector>

#include "circuit_model.h"

namespace vp {

// Where each message of a proof sits in the flat transcript, and each challenge in the challenge array (the draw order of
// vp_draw_challenges). Layers run from n-1 down to 1; per layer the transcript holds phase 1's rounds, claim_u, phase 2's
// rounds and claims_v[0..i) (if the layer has a phase 2), then Liu's rounds and claim_liu; Vres comes first, the input-layer
// MLE last. A round is three elements {a, b, c}.
struct LayerLayout {
    int pb = 0;    // rounds of phase 1 and of Liu: the bit length of layer i-1
    int m = -1;    // rounds of phase 2; -1: the layer has no phase 2
    uint32_t ci_ru = 0, ci_assert = 0, ci_rv = 0, ci_sig = 0, ci_rliu = 0;
    uint32_t tr_p1 = 0, tr_claim_u = 0, tr_p2 = 0, tr_claims_v = 0, tr_liu = 0, tr_claim_liu = 0;
};
struct ProofLayout {
    int out_bits = 0;                 // challenges r_out: the bit length of the output layer
    uint32_t ci_out = 0, tr_vres = 0, tr_input = 0;
    size_t n_chal = 0, n_tr = 0;
    std::vector<LayerLayout> layer;   // by layer id; entry 0 is unused
    uint64_t proof_size = 0;          // bytes of a whole proof (the accounting of prover.cpp:451,500,512)
    size_t rounds = 0;                // sumcheck rounds of a whole proof
};
ProofLayout proof_layout(const Circuit& c);

std::vector<unsigned char> transcript_to_gkrproof(const Circuit& c, const F* transcript);
// returns "" on success; transcript must have vp_transcript_len entries
std::string gkrproof_to_transcript(const Circuit& c, const unsigned char* bytes, size_t len, F* transcript);
std::string transcript_text(const Circuit& c, const F* transcript, const F* challenges);
}  // namespace vp
