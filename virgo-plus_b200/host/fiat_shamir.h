// Fiat-Shamir challenge source (SURVEY 8(f) N4): the reference ships `transcriptCache`
// (/root/reference/lib/virgo/src/transcriptCache.hpp:14-50) -- a byte pool that is hashed with SHA3-256 whenever a
// challenge is requested -- but never calls it (its verifier draws glibc random() values that do not depend on the
// prover's messages, SURVEY 0). This is that class restated, plus the one thing the dead code leaves open: WHEN
// messages are stored and challenges drawn (fs_schedule below).
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <vector>

#include "../csrc/field.cuh"
#include "proof_io.h"

namespace vp {

void sha3_256(const unsigned char* msg, size_t len, unsigned char out[32]);   // FIPS 202 (XKCP's SHA3_256 in the reference)

class FsCache {   // transcriptCache.hpp:14-50
public:
    void store(const void* in, size_t n) { const unsigned char* p = (const unsigned char*)in; pool.insert(pool.end(), p, p + n); }
    void store(const F& x) { store(&x, sizeof x); }   // 16 bytes {u64 real, u64 img}, like store(const T&) on a fieldElement
    F random() {   // :40-46: hash the pool, the digest becomes the pool, first two words mod p
        unsigned char out[32];
        sha3_256(pool.data(), pool.size(), out);
        pool.assign(out, out + 32);
        uint64_t re, im;
        __builtin_memcpy(&re, out, 8);
        __builtin_memcpy(&im, out + 8, 8);
        return F{re % P, im % P};
    }
private:
    std::vector<unsigned char> pool;
};

// Order of stores and draws in Fiat-Shamir mode (a sound variant of the interactive order of verifier.cpp:134-337: a round's
// challenge is drawn AFTER the round's polynomial was stored; the reference's interactive verifier draws a phase's
// challenges before the phase because they are independent of the messages):
//   store(seed[32]);  r_out[0..bl(out)) = draws;  store(Vres);
//   per layer i = n-1..1:  assert_random = draw;
//      phase 1: per round j: store(a, b, c); r_u[j] = draw;                     then store(claim_u);
//      phase 2 (if any): per round j: store(a, b, c); r_v[j] = draw;            then store(claims_v[0..i));
//      sig[0..n) = draws;  Liu: per round j: store(a, b, c); r_liu[j] = draw;   then store(claim_liu).
// Nothing is drawn after layer 1's Liu rounds, so the schedule ends there: its claim_liu and the input MLE stay unstored.
// Challenge slots of the usual layout that are never used (r_u[j], r_liu[j] for j >= the phase's rounds) stay zero.
// fs_schedule is this order over a proof layout; the provers, the host verifier and the device replay all walk it.

// store transcript elements [tr_begin, tr_begin + n_store), then draw challenges [ci_begin, ci_begin + n_draw)
struct FsStep { uint32_t tr_begin, n_store, ci_begin, n_draw; };

// `count` consecutive steps: step k stores and draws the k-th block of the same size after `first`'s. A sumcheck phase is
// one entry of a step per round, {3 coefficients, 1 challenge}; between phases an entry is one step.
struct FsEntry {
    FsStep first;
    uint32_t count;
    int layer, phase;   // phase 0: between phases; 1, 2, 3: phase 1, phase 2 or Liu of `layer`
    FsStep step(uint32_t k) const { return FsStep{first.tr_begin + k * first.n_store, first.n_store, first.ci_begin + k * first.n_draw, first.n_draw}; }
};
std::vector<FsEntry> fs_schedule(const ProofLayout& layout);

// The challenges of a Fiat-Shamir transcript, recomputed from the messages alone (what a verifier does first), in the
// usual challenge layout (vp_draw_challenges order; unused slots zero).
void fs_challenges(const ProofLayout& layout, const std::vector<FsEntry>& schedule, const uint8_t seed[32], const F* tr, F* ch);

}  // namespace vp
