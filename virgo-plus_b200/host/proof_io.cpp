#include "proof_io.h"

#include <algorithm>
#include <cstdio>
#include <cstring>

namespace vp {

ProofLayout proof_layout(const Circuit& C) {
    const int n = C.n_layers(), mbl = C.max_bit_length();
    ProofLayout P;
    P.layer.resize(n);
    uint32_t ci = 0, ti = 0;
    P.out_bits = C.bit_length(n - 1);
    P.ci_out = ci;
    ci += (uint32_t)P.out_bits;
    P.tr_vres = ti++;
    for (int i = n - 1; i >= 1; --i) {
        LayerLayout& X = P.layer[i];
        const int pb = C.bit_length(i - 1), m = C.max_dad_bit_length(i);
        X.pb = pb;
        X.m = m;
        X.ci_ru = ci; ci += (uint32_t)mbl;
        X.ci_assert = ci++;
        X.ci_rv = ci; if (m != -1) ci += (uint32_t)m;
        X.ci_sig = ci; ci += (uint32_t)n;
        X.ci_rliu = ci; ci += (uint32_t)mbl;
        X.tr_p1 = ti; ti += 3u * (uint32_t)pb;
        X.tr_claim_u = ti++;
        X.tr_p2 = ti; if (m != -1) ti += 3u * (uint32_t)m;
        X.tr_claims_v = ti; if (m != -1) ti += (uint32_t)i;
        X.tr_liu = ti; ti += 3u * (uint32_t)pb;
        X.tr_claim_liu = ti++;
        const int rounds = 2 * pb + std::max(m, 0);
        P.rounds += (size_t)rounds;
        P.proof_size += (uint64_t)rounds * 3 * sizeof(F) + sizeof(F);
        if (m != -1) P.proof_size += (uint64_t)i * sizeof(F);
    }
    P.tr_input = ti++;
    P.n_chal = ci;
    P.n_tr = ti;
    return P;
}

namespace {
void put_u64(std::vector<unsigned char>& o, uint64_t v) {
    unsigned char b[8];
    memcpy(b, &v, 8);
    o.insert(o.end(), b, b + 8);
}
void put_f(std::vector<unsigned char>& o, const F* p, size_t n) {
    const unsigned char* b = reinterpret_cast<const unsigned char*>(p);
    o.insert(o.end(), b, b + n * sizeof(F));
}
}  // namespace

std::vector<unsigned char> transcript_to_gkrproof(const Circuit& C, const F* tr) {
    const ProofLayout P = proof_layout(C);
    const auto& s = P.layer;
    const int n = C.n_layers();
    std::vector<unsigned char> o;
    // final_claims_u [layer], final_claims (Liu) [layer]
    put_u64(o, (uint64_t)n);
    for (int i = 0; i < n; ++i) { F z{0, 0}; put_f(o, i ? tr + s[i].tr_claim_u : &z, 1); }
    put_u64(o, (uint64_t)n);
    for (int i = 0; i < n; ++i) { F z{0, 0}; put_f(o, i ? tr + s[i].tr_claim_liu : &z, 1); }
    // final_claims_v [layer][src]
    put_u64(o, (uint64_t)n);
    for (int i = 0; i < n; ++i) {
        const uint64_t len = (i && s[i].m != -1) ? (uint64_t)i : 0;
        put_u64(o, len);
        if (len) put_f(o, tr + s[i].tr_claims_v, len);
    }
    // polys_u, polys_v, polys [layer][round] of quadratic_poly {a,b,c}
    auto polys = [&](int which) {
        put_u64(o, (uint64_t)n);
        for (int i = 0; i < n; ++i) {
            uint64_t len = 0;
            size_t at = 0;
            if (i) {
                if (which == 0) { len = (uint64_t)s[i].pb; at = s[i].tr_p1; }
                if (which == 1) { len = s[i].m != -1 ? (uint64_t)s[i].m : 0; at = s[i].tr_p2; }
                if (which == 2) { len = (uint64_t)s[i].pb; at = s[i].tr_liu; }
            }
            put_u64(o, len);
            if (len) put_f(o, tr + at, 3 * len);
        }
    };
    polys(0);
    polys(1);
    polys(2);
    put_u64(o, 2);
    put_f(o, tr + P.tr_vres, 1);
    put_f(o, tr + P.tr_input, 1);
    return o;
}

std::string gkrproof_to_transcript(const Circuit& C, const unsigned char* b, size_t len, F* tr) {
    const ProofLayout P = proof_layout(C);
    const auto& s = P.layer;
    const int n = C.n_layers();
    size_t pos = 0;
    auto get_u64 = [&](uint64_t& v) { if (pos + 8 > len) return false; memcpy(&v, b + pos, 8); pos += 8; return true; };
    auto get_f = [&](F* dst, size_t cnt) { if (pos + cnt * sizeof(F) > len) return false; if (dst) memcpy(dst, b + pos, cnt * sizeof(F)); pos += cnt * sizeof(F); return true; };
    uint64_t cnt;
    for (int which = 0; which < 2; ++which) {   // final_claims_u, final_claims
        if (!get_u64(cnt) || cnt != (uint64_t)n) return "GKRProof: bad claim vector length";
        for (int i = 0; i < n; ++i)
            if (!get_f(i ? tr + (which == 0 ? s[i].tr_claim_u : s[i].tr_claim_liu) : nullptr, 1)) return "GKRProof: truncated";
    }
    if (!get_u64(cnt) || cnt != (uint64_t)n) return "GKRProof: bad final_claims_v length";
    for (int i = 0; i < n; ++i) {
        uint64_t l;
        if (!get_u64(l)) return "GKRProof: truncated";
        const uint64_t want = (i && s[i].m != -1) ? (uint64_t)i : 0;
        if (l != want) return "GKRProof: final_claims_v does not match the circuit";
        if (l && !get_f(tr + s[i].tr_claims_v, l)) return "GKRProof: truncated";
    }
    for (int which = 0; which < 3; ++which) {
        if (!get_u64(cnt) || cnt != (uint64_t)n) return "GKRProof: bad poly vector length";
        for (int i = 0; i < n; ++i) {
            uint64_t l;
            if (!get_u64(l)) return "GKRProof: truncated";
            uint64_t want = 0;
            size_t at = 0;
            if (i) {
                if (which == 0) { want = (uint64_t)s[i].pb; at = s[i].tr_p1; }
                if (which == 1) { want = s[i].m != -1 ? (uint64_t)s[i].m : 0; at = s[i].tr_p2; }
                if (which == 2) { want = (uint64_t)s[i].pb; at = s[i].tr_liu; }
            }
            if (l != want) return "GKRProof: round count does not match the circuit";
            if (l && !get_f(tr + at, 3 * l)) return "GKRProof: truncated";
        }
    }
    if (!get_u64(cnt) || cnt != 2 || !get_f(tr + P.tr_vres, 1) || !get_f(tr + P.tr_input, 1)) return "GKRProof: bad trailer";
    if (pos != len) return "GKRProof: trailing bytes";
    return "";
}

std::string transcript_text(const Circuit& C, const F* tr, const F* ch) {
    const ProofLayout P = proof_layout(C);
    std::string out;
    char buf[96];
    auto line = [&](const char* tag, const F& x) {
        snprintf(buf, sizeof buf, "%s %llu %llu\n", tag, x.re, x.im);
        out += buf;
    };
    const F zero{0, 0};
    line("VRES", tr[P.tr_vres]);
    auto rounds = [&](size_t at, int count, const F* r) {
        F prev = zero;
        for (int j = 0; j < count; ++j) {
            line("CH", prev);
            line("PA", tr[at + 3 * j]);
            line("PB", tr[at + 3 * j + 1]);
            line("PC", tr[at + 3 * j + 2]);
            prev = r[j];
        }
        return prev;
    };
    for (int i = C.n_layers() - 1; i >= 1; --i) {
        const LayerLayout& X = P.layer[i];
        F prev = rounds(X.tr_p1, X.pb, ch + X.ci_ru);
        line("CH", prev);
        line("CLAIM_U", tr[X.tr_claim_u]);
        if (X.m != -1) {
            rounds(X.tr_p2, X.m, ch + X.ci_rv);
            for (int l = 0; l < i; ++l) line("CLAIM_V", tr[X.tr_claims_v + l]);
        }
        prev = rounds(X.tr_liu, X.pb, ch + X.ci_rliu);
        line("CH", prev);
        line("CLAIM_LIU", tr[X.tr_claim_liu]);
    }
    line("INPUT_MLE", tr[P.tr_input]);
    return out;
}

}  // namespace vp
