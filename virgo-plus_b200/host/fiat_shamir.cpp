// The Fiat-Shamir challenge source (see fiat_shamir.h): SHA3-256 (FIPS 202: Keccak-f[1600], rate 136, suffix 0x06) and
// the order of stores and draws.
#include "fiat_shamir.h"

#include <string.h>

namespace vp {

namespace {
const uint64_t RC[24] = {
    0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL, 0x000000000000808bULL,
    0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL, 0x000000000000008aULL, 0x0000000000000088ULL,
    0x0000000080008009ULL, 0x000000008000000aULL, 0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL,
    0x8000000000008003ULL, 0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,
    0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL};
inline uint64_t rol(uint64_t x, int n) { return (x << n) | (x >> (64 - n)); }
void keccak_f(uint64_t a[25]) {
    static const int rot[5][5] = {{0, 36, 3, 41, 18}, {1, 44, 10, 45, 2}, {62, 6, 43, 15, 61}, {28, 55, 25, 21, 56}, {27, 20, 39, 8, 14}};   // rot[x][y]
    for (int r = 0; r < 24; ++r) {
        uint64_t c[5], b[25];
        for (int x = 0; x < 5; ++x) c[x] = a[x] ^ a[x + 5] ^ a[x + 10] ^ a[x + 15] ^ a[x + 20];
        for (int x = 0; x < 5; ++x) {
            const uint64_t d = c[(x + 4) % 5] ^ rol(c[(x + 1) % 5], 1);
            for (int y = 0; y < 5; ++y) a[x + 5 * y] ^= d;
        }
        for (int x = 0; x < 5; ++x)
            for (int y = 0; y < 5; ++y) {   // rho + pi: B[y][2x+3y] = rot(A[x][y])
                const int nx = y, ny = (2 * x + 3 * y) % 5;
                b[nx + 5 * ny] = rot[x][y] ? rol(a[x + 5 * y], rot[x][y]) : a[x + 5 * y];
            }
        for (int y = 0; y < 5; ++y)
            for (int x = 0; x < 5; ++x) a[x + 5 * y] = b[x + 5 * y] ^ (~b[(x + 1) % 5 + 5 * y] & b[(x + 2) % 5 + 5 * y]);
        a[0] ^= RC[r];
    }
}
}  // namespace

void sha3_256(const unsigned char* msg, size_t len, unsigned char out[32]) {
    uint64_t st[25];
    memset(st, 0, sizeof st);
    const size_t rate = 136;
    while (len >= rate) {
        for (size_t i = 0; i < rate / 8; ++i) {
            uint64_t w;
            memcpy(&w, msg + 8 * i, 8);
            st[i] ^= w;
        }
        keccak_f(st);
        msg += rate;
        len -= rate;
    }
    unsigned char blk[136];
    memset(blk, 0, sizeof blk);
    memcpy(blk, msg, len);
    blk[len] ^= 0x06;
    blk[rate - 1] ^= 0x80;
    for (size_t i = 0; i < rate / 8; ++i) {
        uint64_t w;
        memcpy(&w, blk + 8 * i, 8);
        st[i] ^= w;
    }
    keccak_f(st);
    memcpy(out, st, 32);
}

std::vector<FsEntry> fs_schedule(const ProofLayout& P) {
    std::vector<FsEntry> s;
    auto run = [&](uint32_t tr, uint32_t n_store, uint32_t ci, uint32_t n_draw) { s.push_back(FsEntry{{tr, n_store, ci, n_draw}, 1, 0, 0}); };
    auto phase = [&](int i, int ph, uint32_t tr, uint32_t ci, int rounds) { s.push_back(FsEntry{{tr, 3, ci, 1}, (uint32_t)rounds, i, ph}); };
    const int n = (int)P.layer.size();
    run(0, 0, P.ci_out, (uint32_t)P.out_bits);
    uint32_t tr_prev = P.tr_vres;   // the message stored before the next layer's assert_random: Vres, then claim_liu
    for (int i = n - 1; i >= 1; --i) {
        const LayerLayout& X = P.layer[i];
        run(tr_prev, 1, X.ci_assert, 1);
        phase(i, 1, X.tr_p1, X.ci_ru, X.pb);
        if (X.m != -1) {
            run(X.tr_claim_u, 1, 0, 0);
            phase(i, 2, X.tr_p2, X.ci_rv, X.m);
            run(X.tr_claims_v, (uint32_t)i, X.ci_sig, (uint32_t)n);
        } else
            run(X.tr_claim_u, 1, X.ci_sig, (uint32_t)n);
        phase(i, 3, X.tr_liu, X.ci_rliu, X.pb);
        tr_prev = X.tr_claim_liu;
    }
    return s;
}

void fs_challenges(const ProofLayout& P, const std::vector<FsEntry>& schedule, const uint8_t seed[32], const F* tr, F* ch) {
    FsCache fs;
    fs.store(seed, 32);
    for (size_t k = 0; k < P.n_chal; ++k) ch[k] = F{0, 0};
    for (const FsEntry& e : schedule)
        for (uint32_t k = 0; k < e.count; ++k) {
            const FsStep st = e.step(k);
            for (uint32_t q = 0; q < st.n_store; ++q) fs.store(tr[st.tr_begin + q]);
            for (uint32_t q = 0; q < st.n_draw; ++q) ch[st.ci_begin + q] = fs.random();
        }
}

}  // namespace vp
