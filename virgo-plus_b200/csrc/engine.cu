// Host engine of the B200 GKR prover: device memory, the static proof plan, kernel launches, and
// the C ABI declared in include/virgo_b200.h.
//
// Reference behaviour mirrored here (file:line into /root/reference):
//   prover::evaluate/Vres/init/sumcheckInit*/sumcheckUpdate*/sumcheckFinalize*   src/prover.cpp:27-521
//   call order and challenge order                                               src/verifier.cpp:134-337
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <functional>
#include <mutex>
#include <thread>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/virgo_b200.h"
#include "../host/circuit_model.h"
#include "../host/proof_io.h"
#include "../host/fiat_shamir.h"
#include "kernels.cuh"
#include "fs_device.cuh"
#include "pc_commit.h"

using namespace vp;

// ------------------------------------------------------------------ error plumbing
static thread_local std::string g_err;
static std::string vformat(const char* fmt, va_list ap) {
    char buf[512];
    vsnprintf(buf, sizeof buf, fmt, ap);
    return buf;
}
static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    g_err = vformat(fmt, ap);
    va_end(ap);
    return code;
}
// an argument check inside API_BEGIN / API_END: VP_ERR_ARG with this message
[[noreturn]] static void bad_arg(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    std::string msg = vformat(fmt, ap);
    va_end(ap);
    throw std::invalid_argument(msg);
}
struct CudaError {
    std::string msg;
};
#define CK(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess) {                                                                      \
            char b_[400];                                                                             \
            snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            throw CudaError{b_};                                                                      \
        }                                                                                             \
    } while (0)

struct vp_circuit {
    Circuit c;
};

// ------------------------------------------------------------------ device buffer helper
template <class T>
struct DBuf {
    T* p = nullptr;
    size_t n = 0;
    void alloc(size_t count) {
        release();
        n = count;
        if (count) CK(cudaMalloc(&p, count * sizeof(T)));
    }
    void upload(const std::vector<T>& h, cudaStream_t s = 0) {
        alloc(h.size());
        if (!h.empty()) CK(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, s));
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
    }
    ~DBuf() { release(); }
    DBuf() = default;
    DBuf(const DBuf&) = delete;
    DBuf& operator=(const DBuf&) = delete;
    DBuf(DBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DBuf& operator=(DBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
        return *this;
    }
};

static inline uint32_t align4(uint32_t x) { return (x + 3u) & ~3u; }
static inline uint32_t cdiv(uint32_t a, uint32_t b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------ sumcheck plan (static)
struct PlanTable {
    int bits;          // ceil_log2(padded size); empty tables use 0
    uint32_t live;     // live entries at level 0
    int claim_slot;    // claims[] slot (phase 2: source layer), or -1
    uint32_t off0;     // offset in buffer 0 (filled by the builder)
};
struct RoundPlan {
    uint32_t tab_begin, n_tabs, col_begin, n_cols;
    uint32_t work;     // total work items
    int in_buf;        // 0 / 1
    bool fold;
    double bytes;      // algorithmic bytes of this round: 48 B read per live entry (+ 48 B written per live output entry)
};
struct SumcheckPlan {
    int rounds = 0;
    std::vector<RoundPlan> r;
    uint32_t fin_begin = 0, n_fin = 0;
    uint32_t rdev_begin = 0;
    uint32_t max_work = 0;
    double bytes = 0;   // algorithmic bytes of all rounds
    int fin_buf = 0;
    uint32_t cap0 = 0, cap1 = 0;   // entries needed in buffer 0 / 1
    std::vector<PlanTable> tabs;
    std::vector<uint32_t> end_off, end_live;  // where each table's stored values are after the last round (fin_buf)
};

struct PlanArena {  // descriptor pools shared by all plans of a context
    std::vector<TabDesc> tabs;
    std::vector<ColDesc> cols;
    std::vector<FinDesc> fins;
    std::vector<RoundDev> rdev;
    std::vector<FoldOnlyDesc> fo;
    std::vector<MergeTab> mt;
    std::vector<PassTab> ptabs;
    std::vector<PassCol> pcols;
    std::vector<PassDev> pdev;
};

// ------------------------------------------------------------------ pass plan: two rounds per pass (k_phase_dfs)
struct PassPlan {
    int rounds = 0;
    uint32_t pass_begin = 0, n_passes = 0, fin_begin = 0, n_fin = 0;
    int fin_buf = 0;
    uint32_t cap0 = 0, cap1 = 0, max_work = 0;
    double bytes = 0;                          // bytes this plan really moves: 48 B per live entry read + 48 B per entry written
    double alg_bytes = 0;                      // SURVEY 8(d) model: 144 B per live table entry over the whole sumcheck
    std::vector<uint32_t> off0, end_off, end_live;
};
static PassPlan build_pass_plan(const std::vector<PlanTable>& tabs, int rounds, const std::vector<uint32_t>& fin_out,
                                PlanArena& A) {
    PassPlan P;
    P.rounds = rounds;
    const size_t nt = tabs.size();
    std::vector<uint32_t> off(nt), live(nt);
    std::vector<uint8_t> gone(nt, 0);
    uint32_t o = 0;
    for (size_t t = 0; t < nt; ++t) {
        off[t] = o;
        live[t] = tabs[t].live;
        o += align4(std::max<uint32_t>(tabs[t].live, 1));
    }
    P.off0 = off;
    P.cap0 = o;
    for (size_t t = 0; t < nt; ++t) P.alg_bytes += 144.0 * tabs[t].live;
    P.pass_begin = (uint32_t)A.pdev.size();
    int cur = 0;
    for (int j = 1; j <= rounds;) {
        const int nr = (j + 1 <= rounds) ? 2 : 1;
        PassDev R;
        memset(&R, 0, sizeof R);
        R.tab_begin = (uint32_t)A.ptabs.size();
        R.col_begin = (uint32_t)A.pcols.size();
        R.in_buf = (uint32_t)cur;
        R.n_rounds = (uint32_t)nr;
        uint32_t work = 0, oo = 0;
        for (size_t t = 0; t < nt; ++t) {
            if (gone[t]) continue;
            const int rem = tabs[t].bits - (j - 1);   // rounds this table still has at the pass's input level
            if (rem <= 0) {                           // already a single value: joins add_term in round j
                A.pcols.push_back(PassCol{off[t], std::min<uint32_t>(live[t], 1u), tabs[t].claim_slot, 0});
                gone[t] = 1;
                continue;
            }
            const bool two = nr == 2 && rem >= 2;
            const uint32_t nl = two ? cdiv(cdiv(live[t], 2), 2) : cdiv(live[t], 2);
            work += (cdiv(live[t], two ? 4 : 2) + 31u) & ~31u;   // a warp's 32-item sub-chunk never spans two tables
            A.ptabs.push_back(PassTab{off[t], live[t], oo, work, two ? 1u : 0u, 0});
            P.bytes += 48.0 * live[t] + 48.0 * nl;
            off[t] = oo;
            live[t] = nl;
            oo += align4(std::max<uint32_t>(nl, 1));
            if (!two && rem == 1 && nr == 2) {        // reached one value in round j: joins add_term in round j+1
                A.pcols.push_back(PassCol{off[t], std::min<uint32_t>(live[t], 1u), tabs[t].claim_slot, 1});
                gone[t] = 1;
            }
        }
        R.n_tabs = (uint32_t)A.ptabs.size() - R.tab_begin;
        R.n_cols = (uint32_t)A.pcols.size() - R.col_begin;
        R.work = work;
        P.max_work = std::max(P.max_work, work);
        if (cur == 0) P.cap1 = std::max(P.cap1, oo);
        else P.cap0 = std::max(P.cap0, oo);
        A.pdev.push_back(R);
        cur ^= 1;
        j += nr;
    }
    P.n_passes = (uint32_t)A.pdev.size() - P.pass_begin;
    P.fin_buf = cur;
    P.end_off = off;
    P.end_live = live;
    P.fin_begin = (uint32_t)A.fins.size();
    if (fin_out.empty()) return P;
    for (size_t t = 0; t < nt; ++t) {
        FinDesc f;
        f.out_idx = fin_out[t];
        f.in_off = off[t];
        if (!gone[t]) { f.from_claim = -1; f.n_vals = std::min<uint32_t>(live[t], 1u); }
        else { f.from_claim = tabs[t].claim_slot; f.n_vals = 0; }
        A.fins.push_back(f);
    }
    P.n_fin = (uint32_t)nt;
    return P;
}

// ------------------------------------------------------------------ a sumcheck phase, possibly sharded over G ranks
// world == 1 (or a small phase): `planB` is the whole phase. Sharded: tables are block-cyclic over the ranks
// (block = 2^m entries); `planA` = the m local rounds on this rank's blocks, then fold-only + all-gather +
// merge, then `planB` = the remaining c rounds on the gathered tables (run identically by every rank).
struct PhaseTabG {   // one table of the phase, global view
    int bits;        // ceil_log2 of the padded size (empty tables do not appear)
    uint32_t live;   // live entries
    int claim_slot;  // claims[] slot, or -1
    uint32_t fin_out;  // transcript index of its final claim
};
struct PhasePlan {
    bool sharded = false;
    int rounds = 0, m = 0;
    SumcheckPlan planA, planB;         // one round per launch/pass (interactive entry points use planB)
    PassPlan ppA, ppB;                 // two rounds per pass (vp_prove)
    std::vector<ShardMap> maps;        // per global table
    std::vector<uint32_t> tab_off;     // offset of the table's level-0 values in buffer 0 on this rank
    std::vector<uint32_t> local_len;   // padded local length (multiple of the block size when sharded)
    std::vector<uint32_t> row_lo, row_hi;  // live table entries [row_lo, row_hi) this rank holds (global indices)
    std::vector<uint8_t> present;
    uint32_t fo_begin = 0, n_fo = 0, mt_begin = 0, n_mt = 0;
    uint32_t foi_begin = 0;            // the same hand-over descriptors for the one-round-per-launch plans (a fold pending)
    uint32_t rec_len = 0, sc_base = 0, n_poly = 0, n_claims = 0;
    uint32_t cap0 = 0, cap1 = 0;
    double bytes_total() const { return ppA.bytes + ppB.bytes; }
};

static constexpr int CYC_BITS = 10;   // a sharded table is dealt out in 2^CYC_BITS blocks (the largest table of the phase)

// slice s of G of a table with nb blocks: blocks [slice_begin(s), slice_begin(s+1))
static inline uint32_t slice_begin(uint32_t nb, uint32_t G, uint32_t s) { return (uint32_t)((uint64_t)nb * s / G); }

static SumcheckPlan build_plan(std::vector<PlanTable> tabs, int rounds, const std::vector<uint32_t>& fin_out,
                               PlanArena& A);

// empty_fin_out: transcript slots of tables that never enter a plan (empty subsets): claim 0
static PhasePlan make_phase(const std::vector<PhaseTabG>& T, int rounds, const std::vector<uint32_t>& empty_fin_out, int world,
                            int rank, int n_claims, PlanArena& A, bool rev = false) {
    PhasePlan P;
    P.rounds = rounds;
    const size_t nt = T.size();
    P.maps.assign(nt, ShardMap{0, 0xffffffffu});
    P.row_lo.assign(nt, 0);
    P.row_hi.assign(nt, 0);
    for (size_t t = 0; t < nt; ++t) P.row_hi[t] = T[t].live;
    P.tab_off.assign(nt, 0);
    P.local_len.assign(nt, 0);
    P.present.assign(nt, 1);
    int logG = 0;
    while ((1 << logG) < world) ++logG;
    const int c = std::min(rounds, std::max(CYC_BITS, logG));
    const int m = rounds - c;
    P.sharded = world > 1 && m >= 2;
    auto add_empty_fins = [&](SumcheckPlan& pl) {
        for (uint32_t o : empty_fin_out) {
            A.fins.push_back(FinDesc{0, 0, -1, o});
            ++pl.n_fin;
        }
    };
    if (!P.sharded) {
        std::vector<PlanTable> tabs;
        std::vector<uint32_t> fo;
        for (const auto& t : T) {
            tabs.push_back(PlanTable{t.bits, t.live, t.claim_slot, 0});
            fo.push_back(t.fin_out);
        }
        if (tabs.empty()) {  // phase without any table (cannot happen for phase 1 / Liu)
            P.planB.rounds = rounds;
            P.planB.fin_begin = (uint32_t)A.fins.size();
            P.planB.rdev_begin = (uint32_t)A.rdev.size();
        } else P.planB = build_plan(tabs, rounds, fo, A);
        add_empty_fins(P.planB);
        // the same phase as a pass plan (level-0 offsets are identical: both pack the tables 4-aligned in order)
        P.ppB = build_pass_plan(tabs, rounds, fo, A);
        for (uint32_t o : empty_fin_out) {
            A.fins.push_back(FinDesc{0, 0, -1, o});
            ++P.ppB.n_fin;
        }
        for (size_t t = 0; t < nt; ++t) {
            P.tab_off[t] = P.planB.tabs[t].off0;
            P.local_len[t] = T[t].live;
        }
        P.cap0 = std::max(P.planB.cap0, P.ppB.cap0);
        P.cap1 = std::max(P.planB.cap1, P.ppB.cap1);
        return P;
    }
    P.m = m;
    const uint32_t G = (uint32_t)world;
    std::vector<PlanTable> tabsA, tabsB;
    std::vector<uint32_t> finB, idxA(nt, ~0u);
    std::vector<FinDesc> collapsed_fins;
    struct Dist { size_t t; uint32_t n_blocks, local_blocks, cnt; };
    std::vector<Dist> dist;
    const uint32_t slice = rev ? G - 1 - (uint32_t)rank : (uint32_t)rank;   // phase-2 tables run in reverse instance order
    for (size_t t = 0; t < nt; ++t) {
        const uint32_t nb = std::max<uint32_t>(1, (T[t].live + (1u << m) - 1) >> m);
        const uint32_t b0 = slice_begin(nb, G, slice), b1 = slice_begin(nb, G, slice + 1);
        const uint32_t lo = std::min<uint64_t>((uint64_t)b0 << m, T[t].live), hi = std::min<uint64_t>((uint64_t)b1 << m, T[t].live);
        P.row_lo[t] = lo;
        P.row_hi[t] = hi;
        if (T[t].bits >= m) {  // distributed: stays alive through the m local rounds
            P.maps[t] = ShardMap{b0 << m, (uint32_t)std::min<uint64_t>((uint64_t)b1 << m, 0xffffffffull)};
            idxA[t] = (uint32_t)tabsA.size();
            tabsA.push_back(PlanTable{99, hi - lo, -1, 0});
            P.local_len[t] = (b1 - b0) << m;
            dist.push_back(Dist{t, nb, b1 - b0, (nb + G - 1) / G});
            tabsB.push_back(PlanTable{T[t].bits - m, nb, T[t].claim_slot, 0});
            finB.push_back(T[t].fin_out);
        } else {               // a single block: lives (and collapses) entirely on the rank holding the last slice
            P.present[t] = b1 > b0;
            if (P.present[t]) {
                idxA[t] = (uint32_t)tabsA.size();
                tabsA.push_back(PlanTable{T[t].bits, T[t].live, T[t].claim_slot, 0});
                P.local_len[t] = T[t].live;
            } else {
                P.maps[t] = ShardMap{0, 0};
                P.row_lo[t] = P.row_hi[t] = 0;
            }
            collapsed_fins.push_back(FinDesc{0, 0, T[t].claim_slot, T[t].fin_out});
        }
    }
    if (tabsA.empty()) tabsA.push_back(PlanTable{99, 0, -1, 0});
    P.ppA = build_pass_plan(tabsA, m, {}, A);
    for (size_t t = 0; t < nt; ++t)
        if (idxA[t] != ~0u) P.tab_off[t] = P.ppA.off0[idxA[t]];
    P.ppB = build_pass_plan(tabsB, rounds - m, finB, A);
    for (const FinDesc& f : collapsed_fins) {
        A.fins.push_back(f);
        ++P.ppB.n_fin;
    }
    for (uint32_t o : empty_fin_out) {
        A.fins.push_back(FinDesc{0, 0, -1, o});
        ++P.ppB.n_fin;
    }
    // gather record: per distributed table three regions of cnt entries, then the scalars
    P.fo_begin = (uint32_t)A.fo.size();
    P.mt_begin = (uint32_t)A.mt.size();
    uint32_t base = 0;
    for (size_t q = 0; q < dist.size(); ++q) {
        const Dist& d = dist[q];
        const uint32_t ia = idxA[d.t];
        // after the m local rounds every local block is down to one value: copy them into the record (fold = 0)
        A.fo.push_back(FoldOnlyDesc{P.ppA.end_off[ia], P.ppA.end_live[ia], d.local_blocks, base, d.cnt, 0});
        MergeTab mt;
        memset(&mt, 0, sizeof mt);
        mt.rec_base = base;
        mt.cnt = d.cnt;
        mt.n_blocks = d.n_blocks;
        mt.out_off = P.ppB.off0[q];
        mt.rev = rev ? 1 : 0;
        for (uint32_t sl = 0; sl <= G; ++sl) mt.sb[sl] = slice_begin(d.n_blocks, G, sl);
        A.mt.push_back(mt);
        base += 3 * d.cnt;
    }
    P.n_fo = (uint32_t)dist.size();
    P.n_mt = (uint32_t)dist.size();
    // the method-by-method entry points (vp_round) run the same stages with one round per launch: stage A = planA on
    // the local tables (after m rounds every block holds TWO stored values with the fold by r_m pending), stage B =
    // planB on the gathered tables
    P.planA = build_plan(tabsA, m, {}, A);
    P.planB = build_plan(tabsB, rounds - m, finB, A);
    for (const FinDesc& f : collapsed_fins) {
        A.fins.push_back(f);
        ++P.planB.n_fin;
    }
    for (uint32_t o : empty_fin_out) {
        A.fins.push_back(FinDesc{0, 0, -1, o});
        ++P.planB.n_fin;
    }
    P.foi_begin = (uint32_t)A.fo.size();
    {
        uint32_t b2 = 0;
        for (size_t q = 0; q < dist.size(); ++q) {
            const Dist& d = dist[q];
            const uint32_t ia = idxA[d.t];
            A.fo.push_back(FoldOnlyDesc{P.planA.end_off[ia], P.planA.end_live[ia], d.local_blocks, b2, d.cnt, 1});
            b2 += 3 * d.cnt;
        }
    }
    P.sc_base = base;
    P.n_poly = 3u * (uint32_t)m;
    P.n_claims = (uint32_t)n_claims;
    P.rec_len = base + P.n_poly + 1 + P.n_claims;
    P.cap0 = std::max({P.ppA.cap0, P.ppB.cap0, P.planA.cap0, P.planB.cap0});
    P.cap1 = std::max({P.ppA.cap1, P.ppB.cap1, P.planA.cap1, P.planB.cap1});
    return P;
}

// tabs must be sorted by bits descending. fin_out[t] = transcript index of table t's final claim.
static SumcheckPlan build_plan(std::vector<PlanTable> tabs, int rounds, const std::vector<uint32_t>& fin_out,
                               PlanArena& A) {
    SumcheckPlan P;
    P.rounds = rounds;
    const size_t nt = tabs.size();
    std::vector<uint32_t> off(nt), live(nt);
    uint32_t o = 0;
    for (size_t t = 0; t < nt; ++t) {
        tabs[t].off0 = o;
        off[t] = o;
        live[t] = tabs[t].live;
        o += align4(std::max<uint32_t>(tabs[t].live, 1));
    }
    P.cap0 = o;
    P.tabs = tabs;
    int cur_buf = 0;
    P.rdev_begin = (uint32_t)A.rdev.size();
    for (int j = 1; j <= rounds; ++j) {
        RoundPlan R;
        R.fold = j >= 2;
        R.in_buf = cur_buf;
        R.tab_begin = (uint32_t)A.tabs.size();
        R.col_begin = (uint32_t)A.cols.size();
        uint32_t work = 0, oo = 0;
        R.bytes = 0;
        for (size_t t = 0; t < nt; ++t) {
            const int b = tabs[t].bits;
            if (b >= j) {
                TabDesc d;
                d.in_off = off[t];
                d.in_live = live[t];
                R.bytes += 48.0 * live[t] + (R.fold ? 48.0 * cdiv(live[t], 2) : 0.0);
                d.out_off = oo;
                work += R.fold ? cdiv(live[t], 4) : cdiv(live[t], 2);
                d.work_end = work;
                A.tabs.push_back(d);
                if (R.fold) {
                    off[t] = oo;
                    live[t] = cdiv(live[t], 2);
                    oo += align4(std::max<uint32_t>(live[t], 1));
                }
            } else if (b == j - 1) {
                ColDesc c;
                c.in_off = off[t];
                c.n_vals = std::min<uint32_t>(live[t], R.fold ? 2u : 1u);
                c.claim_slot = tabs[t].claim_slot;
                c.pad = 0;
                A.cols.push_back(c);
            }
        }
        R.n_tabs = (uint32_t)A.tabs.size() - R.tab_begin;
        R.n_cols = (uint32_t)A.cols.size() - R.col_begin;
        R.work = work;
        A.rdev.push_back(RoundDev{R.tab_begin, R.n_tabs, R.col_begin, R.n_cols, R.work, (uint32_t)R.in_buf});
        P.max_work = std::max(P.max_work, R.work);
        P.bytes += R.bytes;
        if (R.fold) {
            if (cur_buf == 0) P.cap1 = std::max(P.cap1, oo);
            else P.cap0 = std::max(P.cap0, oo);
            cur_buf ^= 1;
        }
        P.r.push_back(R);
    }
    P.fin_buf = cur_buf;
    P.end_off = off;
    P.end_live = live;
    P.fin_begin = (uint32_t)A.fins.size();
    if (fin_out.empty()) return P;  // stage A of a sharded phase: no final claims
    for (size_t t = 0; t < nt; ++t) {
        FinDesc f;
        f.out_idx = fin_out[t];
        f.in_off = off[t];
        if (tabs[t].bits >= rounds) {  // alive to the end (bits == rounds)
            f.from_claim = -1;
            f.n_vals = std::min<uint32_t>(live[t], rounds >= 1 ? 2u : 1u);
        } else {
            f.from_claim = tabs[t].claim_slot;
            f.n_vals = 0;
        }
        A.fins.push_back(f);
    }
    P.n_fin = (uint32_t)nt;
    return P;
}

// ------------------------------------------------------------------ which instances a rank evaluates, per layer
// direct[l] = instances whose layer-l values some table of this rank reads (phase 1 / Liu of layer l+1 read rows of
// layer l; a phase-2 table (i, l) gathers from layer l; Vres / the input MLE use the rank's own slice). A layer must be
// evaluated for the hull of direct[l'] over all l' >= l, because a gate reads from any lower layer. Small phase-2
// tables with few blocks can hand one rank a wide slice of a LOW layer; the layers above it stay narrow.
// ph(i, phase) returns the PhasePlan of layer i (phase 2 only asked for layers that have one); p2_src(i) the source
// layer of each of its phase-2 tables.
struct EvalRanges {
    std::vector<uint32_t> lo, hi;                 // per layer
    std::vector<uint32_t> p1_k0, p1_k1;           // per layer: instance range of the rank's phase-1 rows
    std::vector<uint32_t> p2_kk0, p2_kk1;         // per layer: reversed-instance range of its phase-2 rows
    uint32_t own_lo = 0, own_hi = 0;
};
template <class PlanOf, class SrcOf>
static EvalRanges compute_eval_ranges(const Circuit& C, uint32_t K, int world, int rank, PlanOf ph, SrcOf p2_src) {
    const int n = C.n_layers();
    EvalRanges R;
    R.own_lo = (uint32_t)((uint64_t)K * rank / world);
    R.own_hi = (uint32_t)((uint64_t)K * (rank + 1) / world);
    R.p1_k0.assign(n, 0); R.p1_k1.assign(n, 0); R.p2_kk0.assign(n, 0); R.p2_kk1.assign(n, 0);
    std::vector<uint32_t> dlo(n, K), dhi(n, 0);
    auto need = [&](int l, uint32_t a, uint32_t b) { if (b > a) { dlo[l] = std::min(dlo[l], a); dhi[l] = std::max(dhi[l], b); } };
    need(n - 1, R.own_lo, R.own_hi);   // Vres
    need(0, R.own_lo, R.own_hi);       // input MLE
    for (int i = 1; i < n; ++i) {
        const uint32_t S_pre = (uint32_t)C.layers[i - 1].size;
        auto fwd = [&](const PhasePlan& P, uint32_t& a, uint32_t& b) {   // table over layer i-1: idx = k*S_pre + u0
            a = K; b = 0;
            if (P.row_hi[0] > P.row_lo[0]) { a = P.row_lo[0] / S_pre; b = (P.row_hi[0] - 1) / S_pre + 1; }
        };
        uint32_t a, b;
        fwd(ph(i, 1), a, b);
        R.p1_k0[i] = std::min(a, K); R.p1_k1[i] = std::max(b, R.p1_k0[i]);
        need(i - 1, a, std::min(b, K));
        fwd(ph(i, 3), a, b);
        need(i - 1, a, std::min(b, K));
        uint32_t kk0 = K, kk1 = 0;
        if (C.max_dad_bit_length(i) != -1) {
            const PhasePlan& P2 = ph(i, 2);
            const std::vector<int>& src = p2_src(i);
            for (size_t t = 0; t < src.size(); ++t) {
                const uint32_t Dsz = (uint32_t)C.layers[i].dadSize[src[t]];
                if (P2.row_hi[t] <= P2.row_lo[t]) continue;
                const uint32_t kka = P2.row_lo[t] / Dsz, kkb = (P2.row_hi[t] - 1) / Dsz + 1;   // idx = kk*D + lv0, kk = K-1-k
                kk0 = std::min(kk0, kka);
                kk1 = std::max(kk1, kkb);
                need(src[t], K - std::min(kkb, K), K - kka);
            }
        }
        if (kk1 < kk0) kk0 = kk1 = 0;
        R.p2_kk0[i] = kk0; R.p2_kk1[i] = kk1;
    }
    R.lo.assign(n, K);
    R.hi.assign(n, 0);
    uint32_t lo = K, hi = 0;
    for (int l = n - 1; l >= 0; --l) {
        lo = std::min(lo, dlo[l]); hi = std::max(hi, dhi[l]);
        R.lo[l] = std::min(lo, hi); R.hi[l] = std::min(hi, K);
    }
    return R;
}
// the phase-2 tables of layer i: non-empty subsets, bits descending (stable by source layer)
static std::vector<int> phase2_order(const Circuit& C, int i) {
    std::vector<int> order;
    for (int l = 0; l < i; ++l)
        if (C.layers[i].dadSize[l] > 0) order.push_back(l);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return C.dad_bit_length(i, x) > C.dad_bit_length(i, y); });
    return order;
}

// ------------------------------------------------------------------ CSR rows -> work items
static constexpr uint32_t ROW_CHUNK = 8;
struct ItemPlan {
    std::vector<RowItem> items;
    std::vector<LongRow> longs;
    uint32_t n_slots = 0;
};
// off: R+1 absolute entry positions of the rows of one table
static void add_rows(ItemPlan& P, const std::vector<uint32_t>& off, uint32_t tab) {
    const uint32_t R = (uint32_t)off.size() - 1;
    for (uint32_t r = 0; r < R; ++r) {
        const uint32_t len = off[r + 1] - off[r];
        if (len <= ROW_CHUNK) {
            P.items.push_back(RowItem{r, off[r], len, tab});
            continue;
        }
        LongRow lr{r, P.n_slots, 0, tab};
        for (uint32_t e = off[r]; e < off[r + 1]; e += ROW_CHUNK) {
            const uint32_t cnt = std::min(ROW_CHUNK, off[r + 1] - e);
            P.items.push_back(RowItem{r, e, cnt | ((P.n_slots + 1) << 8), tab});
            ++P.n_slots;
        }
        lr.slot_end = P.n_slots;
        P.longs.push_back(lr);
    }
}

// Threads take consecutive items, and an item's loop runs (cnt & 0xff) times: order the items of every window of
// `window` consecutive items by length, so that the 32 items of a warp have (nearly) the same trip count. Fan-in is
// skewed (SHA256: mean 2-5), unsorted warps keep only 21-26 of 32 lanes busy. The window keeps a block's stores
// within a few KB of each other (row order inside a window does not matter: an item carries its row).
static void sort_items_by_length(std::vector<RowItem>& items) {
    const char* e = getenv("VP_ITEM_SORT_WINDOW");
    const size_t window = e ? (size_t)atoi(e) : 8192;
    if (window < 2) return;
    std::vector<RowItem> tmp(std::min(items.size(), window));
    for (size_t b = 0; b < items.size(); b += window) {   // stable counting sort by length (0..255), longest first
        const size_t end = std::min(items.size(), b + window);
        size_t start[257] = {0};
        for (size_t i = b; i < end; ++i) ++start[256 - (items[i].cnt_slot & 0xff)];   // bucket k+1 holds length 255-k
        for (int k = 0; k < 256; ++k) start[k + 1] += start[k];
        for (size_t i = b; i < end; ++i) tmp[start[255 - (items[i].cnt_slot & 0xff)]++] = items[i];
        std::copy(tmp.begin(), tmp.begin() + (end - b), items.begin() + b);
    }
}

// ------------------------------------------------------------------ per-layer device data
// a layer's device state; its transcript and challenge indices are the proof layout's (Engine::build copies them)
struct LayerDev : LayerLayout {
    uint32_t S = 0;
    DBuf<uint8_t> ty;
    DBuf<int16_t> l;
    DBuf<uint32_t> u, v;
    DBuf<F> c;
    GateArrays G{};
    // phase 1 CSR (keyed by u0 in layer i-1), cut into work items of <= ROW_CHUNK entries
    DBuf<uint32_t> p1_g0, p1_v0, p1_tyl;
    DBuf<RowItem> p1_items;
    DBuf<LongRow> p1_long;
    uint32_t p1_nslots = 0;
    uint32_t p1_k0 = 0, p1_k1 = 0;       // instance range of this rank's phase-1 rows
    uint32_t p2_kk0 = 0, p2_kk1 = 0;     // reversed-instance range of this rank's phase-2 rows
    // phase 2
    DBuf<uint32_t> p2_dad_all, p2_g0, p2_u0;
    DBuf<uint8_t> p2_ty;
    DBuf<P2Table> p2_tabs;
    DBuf<RowItem> p2_items;
    DBuf<LongRow> p2_long;
    uint32_t p2_nslots = 0;
    int p2_ntabs = 0;            // tables with a non-empty subset
    double p2_out_entries = 0, p2_gates = 0;
    DBuf<uint32_t> un_g0, un_u0;
    DBuf<uint8_t> un_ty;
    uint32_t n_unary = 0;
    // Liu (tables into layer pre = i-1 from all layers j >= i)
    DBuf<uint32_t> liu_off, liu_perm;
    DBuf<LiuEntry> liu_ent;
    std::vector<int> liu_j;      // source layers j of the eq tables, in eq_id order
    // plans
    PhasePlan ph1, ph2, ph3;
    // eq build descriptor slices (indices into Engine::eq_descs)
    uint32_t eqb_g = 0, eqb_u = 0, eqb_u1 = 0, eqb_g2 = 0, eqb_u2 = 0, eqb_liu = 0, n_eqb_liu = 0;
    DBuf<EqTab> liu_eqtabs, liu_eqtabs_b;   // in eq region set A / B
    uint32_t ci_g = 0;   // challenges of the point g of phase 1: r_out (top layer) or r_liu of the layer above
    // verifier sums (vp_verify): gates in bucket order, built on first use
    std::vector<P2Table> h_p2;       // host copy of the phase-2 table descriptors (dadId lists on the device)
    std::vector<int> p2_src;         // source layer of each phase-2 table
    DBuf<VfGate> vf_gates;
    DBuf<VfBucket> vf_buckets;
    DBuf<uint8_t> vf_assert;
    std::vector<uint32_t> vf_key;    // per bucket: 0 Copy, 1 Not, 2 Addc (+ bias), 3 Mulc, 4 + 7*l + binary type index
    DBuf<VfLiuSeg> vf_liu;
    uint32_t n_vf_liu = 0, eqb_v = 0, eqb_rl = 0, vf_out = 0;
    bool vf_ready = false;
};

// ------------------------------------------------------------------ NCCL, loaded at run time (torch's bundled
// libnccl.so.2 is already in the process when the caller imported torch; otherwise the system one)
typedef void* vp_ncclComm_t;
struct NcclApi {
    void* h = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(vp_ncclComm_t*, int, /* ncclUniqueId by value: 128 bytes */ struct NcclId, int) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, vp_ncclComm_t, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, vp_ncclComm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(vp_ncclComm_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
struct NcclId {
    char internal[128];
};
static NcclApi g_nccl;
static void nccl_load() {
    if (g_nccl.h) return;
    const char* cands[] = {getenv("VP_NCCL_LIB"), "libnccl.so.2", "/usr/lib/x86_64-linux-gnu/libnccl.so.2", "libnccl.so"};
    for (const char* c : cands) {
        if (!c) continue;
        g_nccl.h = dlopen(c, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.h) break;
    }
    if (!g_nccl.h) throw CudaError{std::string("cannot load libnccl.so.2 (set VP_NCCL_LIB): ") + dlerror()};
    auto sym = [&](const char* n) {
        void* p = dlsym(g_nccl.h, n);
        if (!p) throw CudaError{std::string("libnccl: missing symbol ") + n};
        return p;
    };
    g_nccl.GetUniqueId = (int (*)(void*))sym("ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(vp_ncclComm_t*, int, NcclId, int))sym("ncclCommInitRank");
    g_nccl.AllGather = (int (*)(const void*, void*, size_t, int, vp_ncclComm_t, cudaStream_t))sym("ncclAllGather");
    g_nccl.Broadcast = (int (*)(const void*, void*, size_t, int, int, vp_ncclComm_t, cudaStream_t))sym("ncclBroadcast");
    g_nccl.CommDestroy = (int (*)(vp_ncclComm_t))sym("ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
}
#define NCK(call)                                                                                        \
    do {                                                                                                 \
        int r_ = (call);                                                                                 \
        if (r_ != 0) {                                                                                   \
            char b_[300];                                                                                \
            snprintf(b_, sizeof b_, "%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?"); \
            throw CudaError{b_};                                                                         \
        }                                                                                                \
    } while (0)

static constexpr size_t DFS_DYN_SMEM = (size_t)(DFS_THREADS / 32) * DFS_WARP_SMEM_F * sizeof(F);
static void dfs_enable_smem() {   // opt in to the dynamic shared memory of the staging pipeline (all instantiations)
    const void* ks[] = {(const void*)k_phase_dfs<true, DFS_VREAL>, (const void*)k_phase_dfs<false, DFS_VREAL>,
                        (const void*)k_phase_dfs<true, DFS_PLAIN>, (const void*)k_phase_dfs<false, DFS_PLAIN>,
                        (const void*)k_phase_dfs<true, DFS_NEED_B>};
    for (const void* k : ks) CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DFS_DYN_SMEM));
}

// One-kernel NVLink exchange (k_xchg): per lane an exchange buffer that every rank of the box maps through CUDA IPC.
// Layout (entries of F): [0, 16) the ranks' flags (u32 each), then two parity buffers of world * slot_stride entries.
struct XchgLane {
    F* base = nullptr;                   // own allocation (cudaMalloc: IPC handles refer to whole allocations)
    F* peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    uint32_t seq = 0;                    // exchanges done on this lane (the ranks run the same sequence)
    DBuf<F> d_sc;                        // this rank's partial scalars of the phase in flight (zero between phases)
    DBuf<unsigned int> ticket;
};
struct StatementAssert { uint32_t stmt; unsigned int flag; };   // a batch's first statement with a failed assert gate
struct Engine {
    Circuit C;
    int device = 0;
    int world = 1, rank = 0;
    uint32_t k_lo = 0, k_hi = 0;     // instances [k_lo, k_hi) whose inputs this rank holds (all of them when world == 1)
    std::vector<uint32_t> ev_lo, ev_hi;   // per layer: the instances this rank evaluates
    uint32_t ko_lo = 0, ko_hi = 0;   // this rank's own slice of the instances (disjoint over the ranks): dot products, unary sums
    vp_ncclComm_t comm = nullptr;
    DBuf<F> d_send, d_recv;
    DBuf<FoldOnlyDesc> d_fo;
    DBuf<MergeTab> d_mt;
    DBuf<PassTab> d_ptabs;
    DBuf<PassCol> d_pcols;
    DBuf<PassDev> d_pdev;
    // second lane: the Liu phases only need the challenges, not the results of phase 1/2, so vp_prove runs them on
    // their own stream with their own table buffers; the latency-bound tail of one phase then overlaps the bulk
    // passes of an independent phase. swap_lane() exchanges the lane-specific members (host-side pointer swaps).
    struct LaneRes {
        cudaStream_t stream = nullptr;
        DBuf<F> bufV[2], bufM[2], bufA[2], d_scal, d_partials, d_send, d_recv, d_claims;
        DBuf<unsigned int> d_counter;
        DBuf<F> d_rowpart, d_hs;
        vp_ncclComm_t comm = nullptr;
        size_t eq_off = 0;               // this lane's eq region set inside d_eq (entries)
        cudaEvent_t ev_done = nullptr;
        XchgLane x;                      // NVLink exchange state of this lane (sharded contexts)
    } lane1, lane2, lane0b, lane1b, lane2b;
    XchgLane x;                          // ... and of the main lane
    // third lane: phase 2 of layer i only needs V_u from phase 1 of the same layer, and phase 1 of layer i-1 needs
    // nothing from phase 2 of layer i (the challenges are known): phase 1 / phase 2 / Liu each run on their own stream,
    // phase 2 one event behind phase 1. V_u is kept per layer (d_vu) instead of in one scalar.
    // Six lanes (unsharded contexts): phases of different layers are independent as well, so a second set of lanes
    // (lane0b / lane1b / lane2b, with its own eq region set) takes every other layer. This only pays for latency-bound
    // proofs (one SHA256_64: 14 phases of ~50 us per lane; a 65-layer circuit of 2^20-gate layers); a throughput-bound
    // proof (SHA256_64 x 1024) is indifferent to it.
    bool three_lanes = false, six_lanes = false, on_lane2 = false;
    DBuf<F> d_vu;
    uint32_t region_g_lane2 = 0, region_u_lane2 = 0;
    std::vector<cudaEvent_t> ev_p1v;   // per layer: phase 1 done (V_u written)
    F* vu_ptr(int layer) { return three_lanes ? d_vu.p + layer : scal(SC_VU); }
    size_t eq_off = 0;                 // the active lane's eq region set
    LaneRes* active = nullptr;         // the lane whose members are swapped in (null: the main lane)
    void swap_res(LaneRes& R) {
        std::swap(stream, R.stream);
        for (int b = 0; b < 2; ++b) { std::swap(bufV[b], R.bufV[b]); std::swap(bufM[b], R.bufM[b]); std::swap(bufA[b], R.bufA[b]); }
        std::swap(d_scal, R.d_scal);
        std::swap(d_partials, R.d_partials);
        std::swap(d_counter, R.d_counter);
        std::swap(d_claims, R.d_claims);
        std::swap(d_rowpart, R.d_rowpart);
        std::swap(d_hs, R.d_hs);
        std::swap(d_send, R.d_send);
        std::swap(d_recv, R.d_recv);
        std::swap(comm, R.comm);
        std::swap(eq_off, R.eq_off);
        std::swap(x, R.x);
    }
    bool two_lanes = false, on_lane1 = false;
    // role of the lane being entered: 0 = phase 1 (behaves like the main lane), 1 = Liu, 2 = phase 2
    void enter(LaneRes& R, int role) {
        if (active) throw CudaError{"lane switch while another lane is active"};
        swap_res(R);
        active = &R;
        on_lane1 = role == 1;
        on_lane2 = role == 2;
    }
    void leave() {
        if (!active) return;
        swap_res(*active);
        active = nullptr;
        on_lane1 = on_lane2 = false;
    }
    PcCommit* pc = nullptr;          // polynomial-commitment commit phase (SURVEY 8(f) N1), created on first use
    float last_commit_ms = 0;
    bool use_ipc = false;            // sharded: one-kernel NVLink exchange (k_xchg) instead of NCCL all-gathers
    uint32_t x_stride = 0;           // entries of one rank's slot in an exchange buffer
    std::vector<void*> ipc_opened;   // peer mappings to close
    DBuf<unsigned int> d_xerr;       // set by k_xchg when the ranks exchange records of different phases
    void setup_ipc_exchange(uint32_t max_rec);
    bool direct_v = false;   // whole-proof: phase 1 / Liu read V from circuitValue[i-1] instead of a copy
    cudaEvent_t ev_eval = nullptr;
    uint32_t region_u_lane1 = 0;
    int cap_dfs = 0;
    int n = 0;            // layers
    uint32_t K = 1;
    int max_bl = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int max_grid = 148 * 4;

    std::vector<LayerDev> L;
    std::vector<DBuf<F>> val;          // circuitValue[i]
    DBuf<F*> d_valptr;
    DBuf<uint32_t> d_sizes;
    DBuf<uint64_t> d_inputs;
    DBuf<F> bufV[2], bufM[2], bufA[2];
    DBuf<F> d_eq;
    DBuf<F> d_chal, d_tr, d_scal, d_claims, d_partials, d_pub, d_rowpart;
    DBuf<unsigned int> d_counter;      // [0] grid-sum ticket, [1] assert flag
    DBuf<TabDesc> d_tabs;
    DBuf<ColDesc> d_cols;
    DBuf<FinDesc> d_fins;
    DBuf<RoundDev> d_rdev;
    DBuf<EqBuild> d_eqb;
    std::vector<EqBuild> eq_descs;
    PlanArena arena;
    uint32_t eq_half_cap = 0;          // entries of one half table
    size_t eq_set_entries = 0;         // entries of one eq region set
    uint32_t eqb_out = 0, eqb_in = 0;
    ProofLayout lay;                 // where every message and challenge of a proof sits
    std::vector<FsEntry> fs_sched;   // the Fiat-Shamir order over lay

    // scalars in d_scal
    enum { SC_ADD_TERM = 0, SC_VU = 1, SC_UNARY = 2, SC_N = 4 };

    // protocol state (interactive API)
    int cur_layer = 0;     // sumcheckLayerId
    int round = 0;
    int phase = 0;
    bool have_equ = false;
    uint64_t proof_size = 0;
    double prove_seconds = 0;
    float last_ms = 0;
    uint64_t launches = 0, last_launches = 0;
    bool evaluated = false, inputs_loaded = false;
    bool own_stream = true;

    // optional per-kernel-class profiling (CUDA events around every launch of a class)
    enum { KC_ROUND_FOLD = 0, KC_ROUND_FIRST, KC_INIT1, KC_INIT2, KC_INIT_LIU, KC_EVAL, KC_OTHER, KC_N };
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;
    struct ProfRec { int kc; size_t e0, e1; double bytes; };
    std::vector<ProfRec> prof;
    size_t ev_used = 0;
    double prof_ms[KC_N] = {0}, prof_bytes[KC_N] = {0};
    uint64_t prof_launches[KC_N] = {0};

    size_t prof_begin(int kc) {
        if (!profiling) return (size_t)-1;
        while (ev_pool.size() < ev_used + 2) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            ev_pool.push_back(e);
        }
        CK(cudaEventRecord(ev_pool[ev_used], stream));
        prof.push_back(ProfRec{kc, ev_used, ev_used + 1, 0.0});
        ev_used += 2;
        return prof.size() - 1;
    }
    void prof_end(size_t h, double bytes) {
        if (h == (size_t)-1) return;
        CK(cudaEventRecord(ev_pool[prof[h].e1], stream));
        prof[h].bytes = bytes;
    }
    void prof_collect() {  // stream must be idle
        for (const ProfRec& r : prof) {
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, ev_pool[r.e0], ev_pool[r.e1]));
            prof_ms[r.kc] += ms;
            prof_bytes[r.kc] += r.bytes;
            ++prof_launches[r.kc];
        }
        prof.clear();
        ev_used = 0;
    }

    // Interactive fast path (vp_round, one GPU): 64 bytes of pinned host memory mapped into the device -- the round kernel
    // leaves {a, b, c} and a sequence number there (RoundArgs::host_poly / host_seq) and the host spins on the number.
    struct RoundSlot { F poly[3]; unsigned int seq; unsigned int pad[3]; };
    RoundSlot* h_round = nullptr;    // host address
    RoundSlot* d_round = nullptr;    // the same memory as the device sees it
    unsigned int round_seq = 0;
    const vp_F* fast_prev = nullptr; // set around do_round by vp_round: previous challenge by value
    bool fast_out = false;           // set around do_round by vp_round: also write the polynomial to h_round
    void round_slot_alloc() {
        if (h_round) return;
        void* h = nullptr;
        if (cudaHostAlloc(&h, sizeof(RoundSlot), cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return; }   // (falls back to the copy path)
        void* d = nullptr;
        if (cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) { cudaGetLastError(); cudaFreeHost(h); return; }
        memset(h, 0, sizeof(RoundSlot));
        h_round = static_cast<RoundSlot*>(h);
        d_round = static_cast<RoundSlot*>(d);
    }
    // waits for sequence number `want` in the slot; polls the stream now and then so that a failed launch cannot hang the host
    void round_slot_wait(unsigned int want) {
        volatile unsigned int* seq = &h_round->seq;
        for (unsigned long it = 1;; ++it) {
            if (*seq == want) break;
            if ((it & 0xfffu) == 0) {
                const cudaError_t q = cudaStreamQuery(stream);
                if (q == cudaErrorNotReady) continue;
                CK(q);
                if (*seq != want) throw CudaError{"vp_round: the round kernel finished without delivering its polynomial"};
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
    }

    ~Engine() {
        if (h_round) cudaFreeHost(h_round);
        for (auto e : ev_pool) cudaEventDestroy(e);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        leave();
        if (stream && own_stream) cudaStreamDestroy(stream);
        for (LaneRes* R : {&lane1, &lane2, &lane0b, &lane1b, &lane2b}) {
            if (R->stream) cudaStreamDestroy(R->stream);
            if (R->ev_done) cudaEventDestroy(R->ev_done);
        }
        for (auto e : ev_p1v) if (e) cudaEventDestroy(e);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        for (auto e : ev_chunk) if (e) cudaEventDestroy(e);
        if (ev_copy_go) cudaEventDestroy(ev_copy_go);
        if (ev_extra) cudaEventDestroy(ev_extra);
        if (ev_eval) cudaEventDestroy(ev_eval);
        if (pc) pc_destroy(pc);
        for (void* q : ipc_opened) cudaIpcCloseMemHandle(q);
        for (XchgLane* X : {&x, &lane1.x, &lane2.x, &lane0b.x, &lane1b.x, &lane2b.x})
            if (X->base) cudaFree(X->base);
        if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
        if (lane1.comm && g_nccl.CommDestroy) g_nccl.CommDestroy(lane1.comm);
        if (lane2.comm && g_nccl.CommDestroy) g_nccl.CommDestroy(lane2.comm);
    }

    // ---------------------------------------------------------------- helpers
    EqTab eqtab(uint32_t region, int nbits) const {
        const int fh = nbits >> 1;
        EqTab t;
        t.f = d_eq.p + eq_off + (size_t)region * 2 * eq_half_cap;
        t.s = t.f + eq_half_cap;
        t.fh = (uint32_t)fh;
        t.mask = (1u << fh) - 1u;
        return t;
    }
    // appends the two half-table builds of eq(r[ci .. ci+nbits)) * chal[scale] into `region`
    void add_eq_build(uint32_t region, uint32_t ci, int nbits, int scale_idx) {
        const int fh = nbits >> 1, sh = nbits - fh;
        EqBuild a{ci, (uint32_t)fh, scale_idx, (uint32_t)(region * 2 * eq_half_cap)};
        EqBuild b{ci + (uint32_t)fh, (uint32_t)sh, -1, (uint32_t)(region * 2 * eq_half_cap + eq_half_cap)};
        eq_descs.push_back(a);
        eq_descs.push_back(b);
    }
    int n_sm = 148;
    int cap_p1il = 0, cap_p2v2 = 0;
    int dfs_grid_override = 0;   // VP_DFS_GRID: development knob
    bool old_p2 = false;   // VP_OLD_P2 (development knob): every phase-2 init runs the five-products-per-gate k_init_phase2
    bool getenv_no_hs = false, layer_order_by_size = true;
    DBuf<F> d_hs;   // phase-2 init: products of the second-half eq factors, K * ng * nu entries (k_p2_hs)
    bool values_real = true;   // no gate constant has an imaginary part: every circuit value is in the base field
    int cap_round = 0, cap_round1 = 0, cap_eval = 0, cap_p1 = 0, cap_p2 = 0, cap_un = 0, cap_liu = 0, cap_dot = 0, cap_comb = 0;
    template <class Kern>
    int occ_cap(Kern k, int threads = 256, size_t dyn_smem = 0) {  // resident blocks on the whole chip
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, threads, dyn_smem));
        return n_sm * std::max(1, occ);
    }
    int grid_for(uint32_t work, int cap) const { return (int)std::max<uint32_t>(1, std::min<uint32_t>(cdiv(work, 256), (uint32_t)cap)); }
    F* scal(int i) { return d_scal.p + i; }

    void build(const Circuit& circ, int dev, int world_, int rank_, const uint8_t* nccl_id);
    void load_inputs(const uint64_t* host, size_t cnt, bool from_host);
    void load_inputs_chunked(const uint64_t* host, size_t cnt, bool local = false);
    static constexpr int IN_CHUNKS = 4;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_chunk[IN_CHUNKS] = {nullptr, nullptr, nullptr, nullptr}, ev_copy_go = nullptr;
    uint32_t chunk_lo[IN_CHUNKS] = {0}, chunk_hi[IN_CHUNKS] = {0};
    int pending_chunks = 0;
    // Sharded contexts: the inputs a rank needs beyond [core_lo, core_hi) -- the instances whose higher layers it
    // evaluates -- are only read as layer-0 values (the V gathers of phase-2 tables sourced from the input layer and a
    // block's worth of rows of layer 1's tables). With host buffers they are uploaded AFTER the core range on the copy
    // stream and turned into circuitValue[0] there; only the kernels that may read them wait for ev_extra.
    uint32_t core_lo = 0, core_hi = 0;
    cudaEvent_t ev_extra = nullptr;
    bool extras_pending = false;
    void evaluate();
    void run_eq(uint32_t first, uint32_t count);
    void run_dot_eq(const F* X, uint32_t S, EqTab eq, F* out, bool local_only = false);
    void do_vres();
    void do_input_mle();
    void do_init_phase1(int i);
    void do_init_phase2(int i);
    void do_round(const SumcheckPlan& P, int j, uint32_t ci_prev, uint32_t tr_out, const F* at_init, bool continues = false, F* poly_out = nullptr);
    void sharded_round(const PhasePlan& PP, int phase, int j, uint32_t ci, uint32_t tr, const F* at_init);
    void fold_only(const PhasePlan& P, uint32_t fo_begin, int fin_buf, uint32_t ci);
    MergeArgs merge_args(const PhasePlan& P, uint32_t sc_base, uint32_t n_poly, F* out_poly);
    void do_finalize(const SumcheckPlan& P, uint32_t ci_last, F* keep);
    void do_phase(const PhasePlan& P, uint32_t ci, uint32_t tr_rounds, F* keep, const F* at_init, bool has_a = true,
                  const F* v_first = nullptr);
    void do_init_liu(int i, bool write_a);
    void launch_dfs_kernel(const PassPlan& P, uint32_t ci, uint32_t round_base, const F* at_init, F* add_term_out, F* claims,
                           F* out_poly, F* keep, bool has_a, int first, const F* v_first = nullptr);
    void derive_b();
    // verifier (SURVEY 8(f) N2): O(#gates) sums on the device, protocol checks on the host
    void verify_prepare(int i);
    int verify(const F* tr, int* fail_code, int* fail_layer);
    // the device half of verify: out_total sums per statement (vf_layout), queued into out (partials: vf_max_b * VF_GX * 2)
    uint32_t vf_out_total = 0, vf_max_b = 1;
    void vf_layout();
    void verify_sums_async(F* out, F* partial);
    // the host half: the protocol driver on one transcript, its sums and its challenges
    int verify_check(const F* tr, const F* out, const F* chal, int* fail_code, int* fail_layer) const;
    DBuf<F> d_vf_partial, d_vf_out, d_vf_gather;
    static constexpr uint32_t VF_GX = 64;
    DBuf<ChainDesc> d_chains;
    DBuf<ChainSeg> d_chain_segs;
    DBuf<ChainTerm> d_chain_terms;
    int n_chains = 0;
    uint32_t tail_work = 512;
    void prove_all();
    void prove_fs(const uint8_t seed[32], F* tr_out, F* ch_out);
    const PhasePlan& fs_phase_init(int i, int phase, F*& keep, const F*& at_init);
    // Fiat-Shamir mode on the device (fs_device.cuh): the pool, the per-round stamps and the statement digest's buffers
    DBuf<uint64_t> d_fs_pool;
    DBuf<unsigned long long> d_fs_stamps;
    size_t fs_rounds = 0;                  // rounds of the last device FS proof (4 stamps each)
    DBuf<uint64_t> d_stmt;                 // {circuit, inputs, outputs, statement} digests, 4 words each
    uint64_t* stmt_circuit() const { return d_stmt.p; }
    uint64_t* stmt_inputs() const { return d_stmt.p + 4; }
    uint64_t* stmt_outputs() const { return d_stmt.p + 8; }
    uint64_t* stmt_statement() const { return d_stmt.p + 12; }
    DBuf<uint64_t> d_root_scratch;
    DBuf<F> d_fs_outputs;                  // vp_verify_fs_bound(_batch): the claimed outputs, statements end to end
    DBuf<FsStep> d_fs_steps;               // vp_verify_fs_bound_batch: the store / draw order of a transcript (k_fs_replay)
    void fs_replay_table();
    // vp_verify_fs_bound_batch_dev: the claim chain's per-layer table (k_verify_check), built once per context after vf_layout
    DBuf<VfLayerDesc> d_vf_desc;
    DBuf<uint32_t> d_vf_keys;
    VfCheckArgs vf_check_table();
    void load_batch_inputs(const uint64_t* src, size_t cnt);
    bool circuit_digest_ready = false;
    int cap_phase_fs = 0;
    void fs_alloc();
    void fs_begin();
    void statement_async(const uint8_t context[32], const F* d_outputs, const uint64_t* d_contexts = nullptr);
    void circuit_digest_async();
    void circuit_digest_async(uint64_t instances, uint64_t* out);
    // Aggregate proofs (vp_prove_fs_aggregate): the circuit digest of template + K for the last K asked for (0: none yet),
    // and the B statements' {inputs roots, outputs roots, contexts, statements}, 4 * B words each, then the statements'
    // root and the aggregate (4 words each)
    DBuf<uint64_t> d_digest_k;
    uint64_t digest_k = 0;
    DBuf<uint64_t> d_agg;
    const uint64_t* circuit_digest_k_async(uint64_t K);
    void aggregate_async(uint32_t B, const uint8_t* contexts, const F* d_outputs);
    const uint64_t* agg_statements(uint32_t B) const { return d_agg.p + 12 * (size_t)B; }
    const uint64_t* agg_digest(uint32_t B) const { return d_agg.p + 16 * (size_t)B + 4; }
    void seed_pool(const uint8_t seed[32]);
    void prove_fs_device(F* tr_out, F* ch_out);
    void launch_phase_kernel_fs(const SumcheckPlan& P, uint32_t ci, F* keep, const F* at_init, uint32_t tr_rounds, size_t stamp_round);
    // A batch of statements (vp_prove_fs_bound_batch): the Fiat-Shamir path runs n_stmt statements at once, statement b
    // in blockIdx.z == b with its working set sstride bytes after statement b - 1's (kernels.cuh, stmt_at). A single proof
    // is n_stmt = 1, sstride = 0 on the context's own buffers.
    uint32_t n_stmt = 1;
    size_t sstride = 0;
    dim3 sgrid(uint32_t x, uint32_t y = 1) const { return dim3(x, y, n_stmt); }
    int grid_b(uint32_t work, int cap) const { return grid_for(work, std::max(1, cap / (int)n_stmt)); }   // x-width of one statement
    void memset_stmts(void* p, size_t bytes) {   // zero `bytes` at p in every statement's working set
        if (n_stmt == 1) CK(cudaMemsetAsync(p, 0, bytes, stream));
        else CK(cudaMemset2DAsync(p, sstride, 0, bytes, n_stmt, stream));
    }
    // A batch whose arrays are in device memory (vp_*_fs_bound_batch_dev): statuses instead of errors, copies device to
    // device, and no host synchronisation once the buffers are warm.
    bool dev_io = false;
    bool ms_pending = false;   // last_ms is that of a device-memory batch still in flight (vp_last_prove_ms waits for ev1)
    void copy_stmts_out(void* dst, size_t dpitch, const void* src, size_t bytes) {   // statement b's bytes to dst + b * dpitch
        const cudaMemcpyKind k = dev_io ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
        if (n_stmt == 1) CK(cudaMemcpyAsync(dst, src, bytes, k, stream));
        else CK(cudaMemcpy2DAsync(dst, dpitch, src, sstride, bytes, n_stmt, k, stream));
    }
    // The batch's own buffers, kept for the next batch and grown when needed: per statement a copy of every buffer the
    // Fiat-Shamir path writes (one slab, `stride` bytes per statement), and the layer values, inputs and the descriptors that
    // point into them (phase-2 tables: src_val; Liu eq tables: the eq region) for n_stmt * K instances.
    struct FsSlab {
        uint32_t cap = 0;                  // statements it holds
        size_t stride = 0;
        DBuf<uint8_t> mem;
        size_t o_vf = 0, vf_entries = 0;   // vp_verify_fs_bound_batch: the verifier's sums and partial sums (0: none yet)
        std::vector<DBuf<F>> val;
        DBuf<F*> valptr;
        DBuf<uint64_t> inputs, contexts, root_scratch;
        DBuf<int32_t> status;              // device-memory batches: the statements' statuses (k_batch_screen)
        std::vector<DBuf<P2Table>> p2_tabs;
        std::vector<DBuf<EqTab>> liu_eqtabs;
        std::vector<std::pair<void*, size_t>> views;   // statement 0's buffers in the slab (the context's while swapped)
    } slab;
    const uint64_t* d_circuit_digest = nullptr;   // the context's circuit digest (d_stmt[0 .. 4), shared by a batch)
    uint32_t batch_outputs = 0;   // statements of the last successful vp_prove_fs_bound_batch, whose outputs are in slab.val[n-1]
    void slab_reserve(uint32_t B, size_t vf_entries = 0);
    void slab_swap();   // exchanges the context's buffers with the slab's (an involution)
    // f(buffer, entries) for every buffer of the Fiat-Shamir path that the slab holds per statement, in slab order
    template <class Fn> void fs_buffers(Fn f) {
        for (int b = 0; b < 2; ++b) { f(bufV[b], bufV[b].n); f(bufM[b], bufM[b].n); f(bufA[b], bufA[b].n); }
        f(d_chal, d_chal.n); f(d_tr, d_tr.n); f(d_scal, d_scal.n); f(d_claims, d_claims.n); f(d_partials, d_partials.n);
        f(d_counter, d_counter.n); f(d_rowpart, d_rowpart.n); f(d_eq, eq_set_entries); f(d_hs, d_hs.n); f(d_fs_pool, d_fs_pool.n);
        f(d_stmt, d_stmt.n);
    }
    void fs_absorb_draw(uint32_t tr_begin, uint32_t n_store, uint32_t ci_begin, uint32_t n_draw) {
        k_fs_absorb_draw<<<sgrid(1), 32, 0, stream>>>(d_fs_pool.p, d_tr.p, tr_begin, n_store, d_chal.p, ci_begin, n_draw, sstride);
        ++launches;
    }
    std::vector<F> h_chal;   // host copy of the challenges: the pass kernel gets their limbs through its parameters
    void set_chal(uint32_t idx, const vp_F* v, size_t cnt = 1) {
        // the limb arithmetic needs canonical challenges (split31 would silently drop the top bits of anything else)
        for (size_t i = 0; i < cnt; ++i)
            if (v[i].re >= P || v[i].im >= P) throw std::invalid_argument("challenge " + std::to_string(idx + i) + " is not canonical (components must be < p)");
        CK(cudaMemcpyAsync(d_chal.p + idx, v, cnt * sizeof(F), cudaMemcpyHostToDevice, stream));
        if (h_chal.size() < idx + cnt) h_chal.resize(idx + cnt, f_zero());
        memcpy(h_chal.data() + idx, v, cnt * sizeof(F));
    }
    // the host copy only (vp_round's fast path hands the value to the round kernel, which files it in d_chal)
    void set_chal_host(uint32_t idx, const vp_F* v) {
        if (v->re >= P || v->im >= P) throw std::invalid_argument("challenge " + std::to_string(idx) + " is not canonical (components must be < p)");
        if (h_chal.size() < (size_t)idx + 1) h_chal.resize((size_t)idx + 1, f_zero());
        memcpy(h_chal.data() + idx, v, sizeof(F));
    }
    void get_tr(uint32_t idx, vp_F* out, size_t cnt = 1) {
        CK(cudaMemcpyAsync(out, d_tr.p + idx, cnt * sizeof(F), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
    }
    void check_assert_flag() {
        unsigned int flag = 0, xerr = 0;
        CK(cudaMemcpyAsync(&flag, d_counter.p + 1, sizeof flag, cudaMemcpyDeviceToHost, stream));
        if (d_xerr.p) CK(cudaMemcpyAsync(&xerr, d_xerr.p, sizeof xerr, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        if (xerr) {
            CK(cudaMemsetAsync(d_xerr.p, 0, sizeof(unsigned int), stream));
            throw CudaError{"sharded exchange: the ranks are not walking the same sequence of phases (same vp_set_lanes / same calls on every rank?)"};
        }
        if (flag) throw flag;
    }
};

// ------------------------------------------------------------------ build: upload wiring, CSRs, plans
void Engine::build(const Circuit& circ, int dev, int world_, int rank_, const uint8_t* nccl_id) {
    const bool timing = getenv("VP_CREATE_TIMING") != nullptr;   // development aid: where vp_create spends its host time
    auto t_prev = std::chrono::steady_clock::now();
    double t_acc[8] = {0};
    auto lap = [&](int k) {
        const auto now = std::chrono::steady_clock::now();
        t_acc[k] += std::chrono::duration<double>(now - t_prev).count();
        t_prev = now;
    };
    C = circ;
    lap(0);
    device = dev;
    world = world_;
    rank = rank_;
    if (world < 1 || (world & (world - 1)) || world > 8 || rank < 0 || rank >= world)
        throw CudaError{"sharded context: world must be 1, 2, 4 or 8 and 0 <= rank < world"};
    n = C.n_layers();
    K = (uint32_t)C.instances;
    max_bl = C.max_bit_length();
    if (n < 2) throw CudaError{"circuit needs at least 2 layers"};
    if (n > 120) throw CudaError{"more than 120 layers are not supported"};
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(e)};
    CK(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    if (world_ == 1 && !getenv("VP_ROUND_COPY")) round_slot_alloc();   // VP_ROUND_COPY=1: the copy + synchronise path (A/B timing)
    CK(cudaEventCreate(&ev0));
    CK(cudaEventCreate(&ev1));
    n_sm = prop.multiProcessorCount;
    cap_round = occ_cap(k_round<true>);
    cap_round1 = occ_cap(k_round<false>);
    cap_eval = occ_cap(k_eval_layer);
    cap_p1 = occ_cap(k_init_phase1);
    cap_p1il = occ_cap(k_init_phase1_real);
    cap_p2 = occ_cap(k_init_phase2);
    cap_p2v2 = occ_cap(k_init_phase2_v2);
    cap_un = occ_cap(k_phase2_unary);
    cap_liu = occ_cap(k_init_liu);
    cap_dot = occ_cap(k_dot_eq);
    cap_comb = occ_cap(k_combine_phase2);
    cap_phase_fs = occ_cap(k_sumcheck_phase_fs);
    dfs_enable_smem();
    cap_dfs = std::min({occ_cap(k_phase_dfs<true, DFS_VREAL>, DFS_THREADS, DFS_DYN_SMEM), occ_cap(k_phase_dfs<false, DFS_VREAL>, DFS_THREADS, DFS_DYN_SMEM),
                        occ_cap(k_phase_dfs<true, DFS_PLAIN>, DFS_THREADS, DFS_DYN_SMEM), occ_cap(k_phase_dfs<false, DFS_PLAIN>, DFS_THREADS, DFS_DYN_SMEM)});
    if (getenv("VP_DFS_GRID")) dfs_grid_override = atoi(getenv("VP_DFS_GRID"));
    values_real = true;
    for (const Layer& T : C.layers)
        for (size_t g = 0; g < T.c.size() && g < T.ty.size(); ++g)
            if ((T.ty[g] == T_ADDC || T.ty[g] == T_MULC) && T.c[g].im != 0) values_real = false;
    old_p2 = getenv("VP_OLD_P2") != nullptr;
    layer_order_by_size = getenv("VP_LAYERS_TOP_DOWN") == nullptr;
    getenv_no_hs = getenv("VP_NO_HS") != nullptr;
    d_hs.alloc((size_t)K * 64);
    {
        int coop = 0;
        CK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        if (!coop) throw CudaError{"device does not support cooperative launches"};
    }
    max_grid = std::max({cap_round, cap_round1, cap_un, cap_dot, cap_phase_fs, cap_dfs});  // sizes the block-partials buffer

    lay = proof_layout(C);
    fs_sched = fs_schedule(lay);
    L.resize(n);
    for (int i = n - 1; i >= 1; --i) {
        static_cast<LayerLayout&>(L[i]) = lay.layer[i];
        L[i].ci_g = (i == n - 1) ? lay.ci_out : L[i + 1].ci_rliu;
    }
    {   // claim chains for k_derive_b (verifier.cpp:150-166, 281-284, 333)
        std::vector<ChainDesc> ch;
        std::vector<ChainSeg> sg;
        std::vector<ChainTerm> tm;
        for (int i = n - 1; i >= 1; --i) {
            const LayerDev& D = L[i];
            const int pb = C.bit_length(i - 1), m = D.m;
            ChainDesc c12{(int32_t)(i == n - 1 ? lay.tr_vres : L[i + 1].tr_claim_liu), 0, 0, (uint32_t)sg.size(), 0};
            sg.push_back(ChainSeg{D.tr_p1, (uint32_t)pb, D.ci_ru});
            if (m != -1) sg.push_back(ChainSeg{D.tr_p2, (uint32_t)m, D.ci_rv});
            c12.n_segs = (uint32_t)sg.size() - c12.seg_begin;
            ch.push_back(c12);
            ChainDesc c3{-1, (uint32_t)tm.size(), 0, (uint32_t)sg.size(), 1};
            tm.push_back(ChainTerm{D.ci_sig, D.tr_claim_u});
            for (int j = i; j < n; ++j)
                if (L[j].m != -1) tm.push_back(ChainTerm{D.ci_sig + (uint32_t)(j - (i - 1)), L[j].tr_claims_v + (uint32_t)(i - 1)});
            c3.n_terms = (uint32_t)tm.size() - c3.term_begin;
            sg.push_back(ChainSeg{D.tr_liu, (uint32_t)pb, D.ci_rliu});
            ch.push_back(c3);
        }
        n_chains = (int)ch.size();
        if (tm.empty()) tm.push_back(ChainTerm{0, 0});
        if (n_chains) { d_chains.upload(ch, stream); d_chain_segs.upload(sg, stream); d_chain_terms.upload(tm, stream); }
    }

    // eq scratch: region 0 = beta_g, 1 = beta_u, 2 = output/input MLE, 3.. = Liu tables
    eq_half_cap = 1u << ((max_bl + 1) >> 1);
    const uint32_t n_regions = 8 + (uint32_t)n;   // + beta_v and eq(r_liu) of the verifier sums
    region_u_lane1 = 3 + (uint32_t)n;   // lane 1's own copy of beta_u
    region_g_lane2 = 4 + (uint32_t)n;   // lane 2's own copies of beta_g and beta_u
    region_u_lane2 = 5 + (uint32_t)n;
    eq_set_entries = (size_t)n_regions * 2 * eq_half_cap;
    d_eq.alloc(2 * eq_set_entries);   // region set A (main, lane1, lane2) and set B (lane0b, lane1b, lane2b)

    // values
    val.resize(n);
    std::vector<F*> h_ptr(n);
    std::vector<uint32_t> h_sizes(n);
    for (int i = 0; i < n; ++i) {
        val[i].alloc((size_t)C.layer_size(i));
        h_ptr[i] = val[i].p;
        h_sizes[i] = (uint32_t)C.layers[i].size;
    }
    d_valptr.upload(h_ptr, stream);
    d_sizes.upload(h_sizes, stream);
    d_inputs.alloc(C.layer_size(0));

    uint32_t cap0 = 4, cap1 = 4, max_rec = 0;
    size_t max_partial = 2;
    eqb_out = (uint32_t)eq_descs.size();
    add_eq_build(2, lay.ci_out, C.bit_length(n - 1), -1);
    // The per-layer host work (gate arrays, the three CSRs cut into work items, their sorts) is independent between the
    // layers apart from the plan arena, the eq descriptor list and a few running maxima (all under `mu`): worker threads
    // take the layers from a counter, each with its own stream for the uploads. A 65 x 2^20 random circuit took 11 s here
    // on one core.
    std::mutex mu;
    auto build_layer = [&](int i, cudaStream_t st) {
        const Layer& T = C.layers[i];
        LayerDev& D = L[i];
        const uint32_t S = (uint32_t)T.size, S_pre = (uint32_t)C.layers[i - 1].size;
        D.S = S;
        // gate arrays
        {
            std::vector<uint8_t> ty(S);
            std::vector<int16_t> l(S);
            for (uint32_t g = 0; g < S; ++g) {
                ty[g] = (uint8_t)(T.ty[g] | ((!T.is_assert.empty() && T.is_assert[g]) ? TY_ASSERT_BIT : 0));
                l[g] = (int16_t)T.l[g];
            }
            D.ty.upload(ty, st);
            D.l.upload(l, st);
            D.u.upload(T.u, st);
            D.v.upload(T.v, st);
            // the kernels index the constant array for every Addc / Mulc gate: a layer whose constants are all zero
            // (from_arrays keeps no array then) still gets one
            bool needs_c = false;
            for (uint32_t g = 0; g < S; ++g) needs_c |= (T.ty[g] == T_ADDC || T.ty[g] == T_MULC);
            if (!T.c.empty()) D.c.upload(T.c, st);
            else if (needs_c) D.c.upload(std::vector<F>(S, f_zero()), st);
            D.G = GateArrays{D.ty.p, D.l.p, D.u.p, D.v.p, D.c.p};
            CK(cudaStreamSynchronize(st));  // host vectors go out of scope
        }
        const int pb = C.bit_length(i - 1);
        // plans for phase 1 and Liu: one table over layer i-1 (the plan arena and the running maxima are shared: locked)
        {
            std::lock_guard<std::mutex> lk(mu);
            D.ph1 = make_phase({PhaseTabG{pb, (uint32_t)C.layer_size(i - 1), -1, D.tr_claim_u}}, pb, {}, world, rank, n, arena);
            D.ph3 = make_phase({PhaseTabG{pb, (uint32_t)C.layer_size(i - 1), -1, D.tr_claim_liu}}, pb, {}, world, rank, n, arena);
            cap0 = std::max(cap0, std::max(D.ph1.cap0, D.ph3.cap0));
            cap1 = std::max(cap1, std::max(D.ph1.cap1, D.ph3.cap1));
            max_rec = std::max(max_rec, std::max(D.ph1.rec_len, D.ph3.rec_len));
        }
        // A circuit that is ONE instance has no instance ranges to deal out: a rank of a sharded context keeps only the
        // work items (and long rows) of the table rows it owns, so the init kernels are owner-computes here as well.
        const bool own_rows_only = world > 1 && K == 1;
        // phase-1 CSR by u0
        {
            std::vector<uint32_t> off(S_pre + 1, 0), g0(S), v0(S), tyl(S);
            for (uint32_t g = 0; g < S; ++g) ++off[T.u[g] + 1];
            for (uint32_t x = 0; x < S_pre; ++x) off[x + 1] += off[x];
            std::vector<uint32_t> pos(off.begin(), off.end() - 1);
            for (uint32_t g = 0; g < S; ++g) {
                uint32_t p = pos[T.u[g]]++;
                g0[p] = g;
                v0[p] = T.v[g];
                uint32_t as = (!T.is_assert.empty() && T.is_assert[g]) ? TY_ASSERT_BIT : 0;
                tyl[p] = (uint32_t)T.ty[g] | as | ((uint32_t)(T.l[g] + 1) << 8);
            }
            ItemPlan ip;
            add_rows(ip, off, 0);
            if (own_rows_only && D.ph1.sharded) {
                const ShardMap sm = D.ph1.maps[0];
                auto mine = [&](uint32_t row) { return row >= sm.lo && row < sm.hi; };
                ip.items.erase(std::remove_if(ip.items.begin(), ip.items.end(), [&](const RowItem& x) { return !mine(x.row); }), ip.items.end());
                ip.longs.erase(std::remove_if(ip.longs.begin(), ip.longs.end(), [&](const LongRow& x) { return !mine(x.row); }), ip.longs.end());
            }
            sort_items_by_length(ip.items);
            D.p1_items.upload(ip.items, st);
            D.p1_long.upload(ip.longs, st);
            D.p1_nslots = ip.n_slots;
            { std::lock_guard<std::mutex> lk(mu); max_partial = std::max<size_t>(max_partial, (size_t)ip.n_slots * K * 2); }
            D.p1_g0.upload(g0, st);
            D.p1_v0.upload(v0, st);
            D.p1_tyl.upload(tyl, st);
            CK(cudaStreamSynchronize(st));
        }
        {   // eq build descriptors of the layer: adjacent entries (one k_eq_build launch covers neighbours): locked as a group
        std::lock_guard<std::mutex> lk(mu);
        D.eqb_g = (uint32_t)eq_descs.size();
        add_eq_build(0, D.ci_g, C.bit_length(i), -1);
        D.eqb_u = (uint32_t)eq_descs.size();
        add_eq_build(1, D.ci_ru, pb, -1);
        D.eqb_g2 = (uint32_t)eq_descs.size();
        add_eq_build(4 + (uint32_t)n, D.ci_g, C.bit_length(i), -1);
        D.eqb_u2 = (uint32_t)eq_descs.size();
        add_eq_build(5 + (uint32_t)n, D.ci_ru, pb, -1);
        D.eqb_v = (uint32_t)eq_descs.size();
        add_eq_build(6 + (uint32_t)n, D.ci_rv, std::max(D.m, 0), -1);
        D.eqb_rl = (uint32_t)eq_descs.size();
        add_eq_build(7 + (uint32_t)n, D.ci_rliu, pb, -1);
        }
        // phase 2
        if (D.m != -1) {
            const int m = D.m;
            // table order: bits descending (stable by l); empty subsets get no table (their claim is 0)
            std::vector<int> order;
            for (int l = 0; l < i; ++l)
                if (T.dadSize[l] > 0) order.push_back(l);
            auto bits_of = [&](int l) { return C.dad_bit_length(i, l); };
            std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return bits_of(a) > bits_of(b); });
            std::vector<PhaseTabG> tabs;
            for (int l : order) tabs.push_back(PhaseTabG{bits_of(l), (uint32_t)C.dad_size(i, l), l, D.tr_claims_v + (uint32_t)l});
            std::vector<uint32_t> empties;
            for (int l = 0; l < i; ++l)
                if (T.dadSize[l] == 0) empties.push_back(D.tr_claims_v + (uint32_t)l);
            {
                std::lock_guard<std::mutex> lk(mu);
                D.ph2 = make_phase(tabs, m, empties, world, rank, n, arena, /*rev=*/true);
                cap0 = std::max(cap0, D.ph2.cap0);
                cap1 = std::max(cap1, D.ph2.cap1);
                max_rec = std::max(max_rec, D.ph2.rec_len);
            }
            // CSR per table over lv0
            std::vector<uint32_t> dad_all, g0, u0;
            std::vector<uint8_t> tyv;
            std::vector<P2Table> ptabs;
            ItemPlan ip;
            // the binary gates of the layer by source layer, in gate order (one pass; a circuit with operands from any
            // earlier layer has up to i tables here)
            std::vector<std::vector<uint32_t>> by_src(i);
            for (uint32_t g = 0; g < S; ++g)
                if (is_binary(T.ty[g])) by_src[T.l[g]].push_back(g);
            for (size_t t = 0; t < order.size(); ++t) {
                const int l = order[t];
                const uint32_t Dsz = (uint32_t)T.dadSize[l];
                std::vector<uint32_t> cnt(Dsz + 1, 0);
                for (uint32_t g : by_src[l]) ++cnt[T.lv[g] + 1];
                for (uint32_t x = 0; x < Dsz; ++x) cnt[x + 1] += cnt[x];
                const uint32_t base = (uint32_t)g0.size();
                g0.resize(base + cnt[Dsz]);
                u0.resize(base + cnt[Dsz]);
                tyv.resize(base + cnt[Dsz]);
                std::vector<uint32_t> pos(cnt.begin(), cnt.end() - 1);
                for (uint32_t g : by_src[l])
                    {
                        uint32_t p = base + pos[T.lv[g]]++;
                        g0[p] = g;
                        u0[p] = T.u[g];
                        tyv[p] = (uint8_t)(T.ty[g] | ((!T.is_assert.empty() && T.is_assert[g]) ? TY_ASSERT_BIT : 0));
                    }
                P2Table pt;
                memset(&pt, 0, sizeof pt);
                pt.D = Dsz;
                pt.src_S = (uint32_t)C.layers[l].size;
                pt.tab_off = D.ph2.tab_off[t];
                pt.owned = D.ph2.present[t];
                pt.sm = D.ph2.maps[t];
                pt.src_val = val[l].p;
                // stash the offset into the concatenated array; patched to a pointer after upload
                pt.dadId = (const uint32_t*)(uintptr_t)dad_all.size();
                std::vector<uint32_t> off(Dsz + 1);
                for (uint32_t x = 0; x <= Dsz; ++x) off[x] = base + cnt[x];
                for (uint32_t x = 0; x < Dsz; ++x) dad_all.push_back(T.dadId[l][x]);
                add_rows(ip, off, (uint32_t)ptabs.size());
                ptabs.push_back(pt);
            }
            if (own_rows_only && D.ph2.sharded) {
                auto mine = [&](uint32_t tab, uint32_t row) { return D.ph2.present[tab] && row >= D.ph2.maps[tab].lo && row < D.ph2.maps[tab].hi; };
                ip.items.erase(std::remove_if(ip.items.begin(), ip.items.end(), [&](const RowItem& x) { return !mine(x.tab, x.row); }), ip.items.end());
                ip.longs.erase(std::remove_if(ip.longs.begin(), ip.longs.end(), [&](const LongRow& x) { return !mine(x.tab, x.row); }), ip.longs.end());
            }
            sort_items_by_length(ip.items);
            D.p2_items.upload(ip.items, st);
            D.p2_long.upload(ip.longs, st);
            D.p2_nslots = ip.n_slots;
            { std::lock_guard<std::mutex> lk(mu); max_partial = std::max<size_t>(max_partial, (size_t)ip.n_slots * K * 2); }
            D.p2_dad_all.upload(dad_all, st);
            D.p2_g0.upload(g0, st);
            D.p2_u0.upload(u0, st);
            D.p2_ty.upload(tyv, st);
            for (auto& pt : ptabs) pt.dadId = D.p2_dad_all.p + (uintptr_t)pt.dadId;
            D.p2_tabs.upload(ptabs, st);
            D.h_p2 = ptabs;
            D.p2_src = order;
            D.p2_ntabs = (int)ptabs.size();
            D.p2_gates = (double)g0.size();
            D.p2_out_entries = 0;
            for (auto& pt : ptabs) D.p2_out_entries += (double)pt.D * K;
            // unary gates
            std::vector<uint32_t> ug, uu;
            std::vector<uint8_t> ut;
            for (uint32_t g = 0; g < S; ++g)
                if (!is_binary(T.ty[g])) {
                    ug.push_back(g);
                    uu.push_back(T.u[g]);
                    ut.push_back((uint8_t)(T.ty[g] | ((!T.is_assert.empty() && T.is_assert[g]) ? TY_ASSERT_BIT : 0)));
                }
            D.n_unary = (uint32_t)ug.size();
            D.un_g0.upload(ug, st);
            D.un_u0.upload(uu, st);
            D.un_ty.upload(ut, st);
            CK(cudaStreamSynchronize(st));
        }
        // Liu CSR: all (j >= i, slot0) with dadId_j[i-1][slot0] = u0
        {
            const int pre = i - 1;
            std::vector<uint32_t> off(S_pre + 1, 0);
            D.liu_j.clear();
            for (int j = i; j < n; ++j)
                if (C.layers[j].dadSize[pre] > 0) {
                    D.liu_j.push_back(j);
                    for (uint32_t x : C.layers[j].dadId[pre]) ++off[x + 1];
                }
            for (uint32_t x = 0; x < S_pre; ++x) off[x + 1] += off[x];
            std::vector<LiuEntry> ent(off[S_pre]);
            std::vector<uint32_t> pos(off.begin(), off.end() - 1);
            for (size_t q = 0; q < D.liu_j.size(); ++q) {
                const int j = D.liu_j[q];
                const auto& ids = C.layers[j].dadId[pre];
                for (uint32_t s0 = 0; s0 < ids.size(); ++s0) {
                    LiuEntry E{(uint32_t)q, s0, (uint32_t)ids.size()};
                    ent[pos[ids[s0]]++] = E;
                }
            }
            D.liu_off.upload(off, st);
            D.liu_ent.upload(ent, st);
            {   // same idea as sort_items_by_length: entries of a window ordered by their number of scattered terms
                const char* ev = getenv("VP_ITEM_SORT_WINDOW");
                const size_t window = ev ? (size_t)atoi(ev) : 8192;
                std::vector<uint32_t> perm(S_pre);
                for (uint32_t x = 0; x < S_pre; ++x) perm[x] = x;
                if (window >= 2) {   // stable counting sort by the number of scattered terms, most first
                    std::vector<uint32_t> tmp(std::min<size_t>(S_pre, window)), start;
                    for (size_t b = 0; b < S_pre; b += window) {
                        const size_t end = std::min<size_t>(S_pre, b + window);
                        uint32_t mx = 0;
                        for (size_t x = b; x < end; ++x) mx = std::max(mx, off[x + 1] - off[x]);
                        start.assign((size_t)mx + 2, 0);
                        for (size_t x = b; x < end; ++x) ++start[mx - (off[x + 1] - off[x]) + 1];
                        for (uint32_t k = 0; k <= mx; ++k) start[k + 1] += start[k];
                        for (size_t x = b; x < end; ++x) tmp[start[mx - (off[x + 1] - off[x])]++] = (uint32_t)x;
                        std::copy(tmp.begin(), tmp.begin() + (end - b), perm.begin() + b);
                    }
                }
                D.liu_perm.upload(perm, st);
            }
            // lane 1's copy of beta_u is only used by Liu: bake s[0] in. Its descriptors sit right before the Liu tables'
            // so that one k_eq_build launch covers both.
            std::unique_lock<std::mutex> lk_eq(mu);
            D.eqb_u1 = (uint32_t)eq_descs.size();
            add_eq_build(3 + (uint32_t)n, D.ci_ru, pb, (int)D.ci_sig);
            // eq tables: region 3+q = eq(r_v[j], dadBl_j[pre]) * sig[j - pre]
            D.eqb_liu = (uint32_t)eq_descs.size();
            std::vector<EqTab> tabs;
            for (size_t q = 0; q < D.liu_j.size(); ++q) {
                const int j = D.liu_j[q];
                const int b = C.dad_bit_length(j, pre);
                add_eq_build(3 + (uint32_t)q, L[j].ci_rv, b, (int)(D.ci_sig + (uint32_t)(j - pre)));
                tabs.push_back(eqtab(3 + (uint32_t)q, b));
            }
            D.n_eqb_liu = (uint32_t)eq_descs.size() - D.eqb_liu;
            lk_eq.unlock();
            D.liu_eqtabs.upload(tabs, st);
            for (EqTab& t : tabs) { t.f += eq_set_entries; t.s += eq_set_entries; }   // the same tables in eq region set B
            D.liu_eqtabs_b.upload(tabs, st);
            CK(cudaStreamSynchronize(st));
        }
        };
    {
        const char* ev = getenv("VP_CREATE_THREADS");
        const int want = ev ? atoi(ev) : (int)std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency()), 8u);
        const int n_thr = std::max(1, std::min(want, n - 1));
        std::atomic<int> next{1};
        std::string first_error;
        auto worker = [&](bool own_stream_) {
            cudaStream_t st = stream;
            try {
                CK(cudaSetDevice(dev));
                if (own_stream_) CK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                for (int i; (i = next.fetch_add(1)) < n;) build_layer(i, st);
                CK(cudaStreamSynchronize(st));
            } catch (const CudaError& e) {
                std::lock_guard<std::mutex> lk(mu);
                if (first_error.empty()) first_error = e.msg;
                next.store(n);
            } catch (const std::exception& e) {
                std::lock_guard<std::mutex> lk(mu);
                if (first_error.empty()) first_error = e.what();
                next.store(n);
            }
            if (own_stream_ && st != stream) cudaStreamDestroy(st);
        };
        std::vector<std::thread> pool;
        for (int t = 1; t < n_thr; ++t) pool.emplace_back(worker, true);
        worker(false);
        for (auto& t : pool) t.join();
        if (!first_error.empty()) throw CudaError{first_error};
    }
    lap(5);
    eqb_in = (uint32_t)eq_descs.size();
    add_eq_build(2, L[1].ci_rliu, C.bit_length(0), -1);

    // which instances does this rank touch? (tables are instance-major and every rank holds a contiguous run of each)
    {
        std::vector<std::vector<int>> srcs(n);
        for (int i = 1; i < n; ++i) srcs[i] = phase2_order(C, i);
        const EvalRanges R = compute_eval_ranges(
            C, K, world, rank, [&](int i, int phase) -> const PhasePlan& { return phase == 1 ? L[i].ph1 : phase == 2 ? L[i].ph2 : L[i].ph3; },
            [&](int i) -> const std::vector<int>& { return srcs[i]; });
        ko_lo = R.own_lo; ko_hi = R.own_hi;
        ev_lo = R.lo; ev_hi = R.hi;
        for (int i = 1; i < n; ++i) {
            L[i].p1_k0 = R.p1_k0[i]; L[i].p1_k1 = R.p1_k1[i];
            L[i].p2_kk0 = R.p2_kk0[i]; L[i].p2_kk1 = R.p2_kk1[i];
        }
        k_lo = ev_lo[0];   // the inputs this rank uploads
        k_hi = std::min(ev_hi[0], K);
        core_lo = n > 1 ? std::max(k_lo, std::min(ev_lo[1], k_hi)) : k_lo;   // instances whose layers >= 1 this rank evaluates
        core_hi = n > 1 ? std::min(k_hi, std::max(ev_hi[1], core_lo)) : k_hi;
        if (getenv("VP_NO_EXTRAS")) { core_lo = k_lo; core_hi = k_hi; }
    }

    for (int b = 0; b < 2; ++b) {
        const uint32_t cap = b == 0 ? cap0 : cap1;
        bufV[b].alloc(cap);
        bufM[b].alloc(cap);
        bufA[b].alloc(cap);
    }
    two_lanes = !getenv("VP_ONE_LANE");
    three_lanes = two_lanes && !getenv("VP_TWO_LANES");
    // sharded contexts exchange through NVLink-mapped buffers (k_xchg) unless VP_NCCL_EXCHANGE is set or the IPC set-up
    // fails on some rank; the second set of lanes needs no NCCL communicators then
    const bool want_ipc = world > 1 && !getenv("VP_NCCL_EXCHANGE");
    six_lanes = three_lanes && (world == 1 || want_ipc) && !getenv("VP_THREE_LANES");
    d_rowpart.alloc(max_partial);
    auto alloc_lane = [&](LaneRes& R, int role, size_t eqo) {   // role: 0 phase 1, 1 Liu, 2 phase 2
        uint32_t c0 = 4, c1 = 4;
        for (int i = 1; i < n; ++i) {
            const PhasePlan* P = role == 0 ? &L[i].ph1 : role == 1 ? &L[i].ph3 : (L[i].m != -1 ? &L[i].ph2 : nullptr);
            if (P) { c0 = std::max(c0, P->cap0); c1 = std::max(c1, P->cap1); }
        }
        for (int bb = 0; bb < 2; ++bb) {
            const uint32_t cap = bb == 0 ? c0 : c1;
            R.bufV[bb].alloc(cap);
            R.bufM[bb].alloc(cap);
            // the Liu add table is never stored in whole-proof mode (sharded: the hand-over kernels still address the region)
            R.bufA[bb].alloc(role == 1 && world == 1 ? 4 : cap);
        }
        R.d_scal.alloc(SC_N);
        R.d_claims.alloc((size_t)n + 1);
        R.d_partials.alloc((size_t)12 * (size_t)max_grid);
        R.d_counter.alloc(4 + 64);
        if (role != 1) R.d_rowpart.alloc(max_partial);
        if (role == 2) R.d_hs.alloc((size_t)K * 64);
        R.eq_off = eqo;
        CK(cudaMemsetAsync(R.d_claims.p, 0, ((size_t)n + 1) * sizeof(F), stream));
        CK(cudaMemsetAsync(R.d_scal.p, 0, SC_N * sizeof(F), stream));
        CK(cudaMemsetAsync(R.d_counter.p, 0, (4 + 64) * sizeof(unsigned int), stream));
        CK(cudaStreamCreateWithFlags(&R.stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&R.ev_done, cudaEventDisableTiming));
    };
    if (two_lanes) {
        alloc_lane(lane1, 1, 0);
        CK(cudaEventCreateWithFlags(&ev_eval, cudaEventDisableTiming));
    }
    if (three_lanes) {
        alloc_lane(lane2, 2, 0);
        d_vu.alloc((size_t)n + 1);
        CK(cudaMemsetAsync(d_vu.p, 0, ((size_t)n + 1) * sizeof(F), stream));
        ev_p1v.assign(n, nullptr);
        for (int i = 1; i < n; ++i) CK(cudaEventCreateWithFlags(&ev_p1v[i], cudaEventDisableTiming));
    }
    if (six_lanes) {
        alloc_lane(lane0b, 0, eq_set_entries);
        alloc_lane(lane1b, 1, eq_set_entries);
        alloc_lane(lane2b, 2, eq_set_entries);
    }
    if (world > 1) {
        d_send.alloc(std::max<uint32_t>(max_rec, 1));
        d_recv.alloc((size_t)std::max<uint32_t>(max_rec, 1) * world);
        d_fo.upload(arena.fo, stream);
        d_mt.upload(arena.mt, stream);
        nccl_load();
        NcclId id;
        memcpy(id.internal, nccl_id, 128);
        NCK(g_nccl.CommInitRank(&comm, world, id, rank));
        if (want_ipc) setup_ipc_exchange(std::max<uint32_t>(max_rec, 1));
        if (!use_ipc) six_lanes = false;
    }
    if (two_lanes && world > 1 && !use_ipc) {
        // lane 1 issues its own all-gathers concurrently with lane 0: it needs its own communicator. Rank 0 draws a
        // second unique id and broadcasts it over the first communicator.
        DBuf<unsigned char> d_id;
        d_id.alloc(128);
        NcclId id2;
        memset(&id2, 0, sizeof id2);
        if (rank == 0) NCK(g_nccl.GetUniqueId(&id2));
        CK(cudaMemcpyAsync(d_id.p, id2.internal, 128, cudaMemcpyHostToDevice, stream));
        NCK(g_nccl.Broadcast(d_id.p, d_id.p, 128, /*ncclUint8*/ 1, 0, comm, stream));
        CK(cudaMemcpyAsync(id2.internal, d_id.p, 128, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        NCK(g_nccl.CommInitRank(&lane1.comm, world, id2, rank));
        lane1.d_send.alloc(std::max<uint32_t>(max_rec, 1));
        lane1.d_recv.alloc((size_t)std::max<uint32_t>(max_rec, 1) * world);
        if (three_lanes) {   // and a third communicator for the phase-2 lane
            NcclId id3;
            memset(&id3, 0, sizeof id3);
            if (rank == 0) NCK(g_nccl.GetUniqueId(&id3));
            CK(cudaMemcpyAsync(d_id.p, id3.internal, 128, cudaMemcpyHostToDevice, stream));
            NCK(g_nccl.Broadcast(d_id.p, d_id.p, 128, /*ncclUint8*/ 1, 0, comm, stream));
            CK(cudaMemcpyAsync(id3.internal, d_id.p, 128, cudaMemcpyDeviceToHost, stream));
            CK(cudaStreamSynchronize(stream));
            NCK(g_nccl.CommInitRank(&lane2.comm, world, id3, rank));
            lane2.d_send.alloc(std::max<uint32_t>(max_rec, 1));
            lane2.d_recv.alloc((size_t)std::max<uint32_t>(max_rec, 1) * world);
        }
    }
    d_chal.alloc(lay.n_chal + 1);
    d_tr.alloc(lay.n_tr);
    d_scal.alloc(SC_N);
    d_claims.alloc((size_t)n + 1);
    d_partials.alloc((size_t)12 * (size_t)max_grid);
    d_counter.alloc(4 + 64);
    d_tabs.upload(arena.tabs, stream);
    d_cols.upload(arena.cols, stream);
    d_fins.upload(arena.fins, stream);
    d_rdev.upload(arena.rdev, stream);
    d_ptabs.upload(arena.ptabs, stream);
    d_pcols.upload(arena.pcols, stream);
    d_pdev.upload(arena.pdev, stream);
    d_eqb.upload(eq_descs, stream);
    CK(cudaMemsetAsync(d_chal.p, 0, (lay.n_chal + 1) * sizeof(F), stream));
    CK(cudaMemsetAsync(d_tr.p, 0, lay.n_tr * sizeof(F), stream));
    CK(cudaMemsetAsync(d_scal.p, 0, SC_N * sizeof(F), stream));
    CK(cudaMemsetAsync(d_claims.p, 0, ((size_t)n + 1) * sizeof(F), stream));
    CK(cudaMemsetAsync(d_counter.p, 0, (4 + 64) * sizeof(unsigned int), stream));
    CK(cudaStreamSynchronize(stream));
    load_inputs(C.inputs.data(), C.inputs.size(), true);
    CK(cudaStreamSynchronize(stream));
    lap(6);
    if (timing)
        fprintf(stderr, "vp_create: circuit copy %.2f s, per-layer CSRs / plans / uploads (worker threads) %.2f s, buffers / lanes / communicators %.2f s\n",
                t_acc[0], t_acc[5], t_acc[6]);
}

// Exchange buffers of every lane, mapped into every rank (CUDA IPC over the box's NVLink fabric). Collective: the
// handles travel through one NCCL all-gather on the main communicator, and the ranks agree on the outcome.
void Engine::setup_ipc_exchange(uint32_t max_rec) {
    std::vector<XchgLane*> X{&x};
    if (two_lanes) X.push_back(&lane1.x);
    if (three_lanes) X.push_back(&lane2.x);
    if (six_lanes) { X.push_back(&lane0b.x); X.push_back(&lane1b.x); X.push_back(&lane2b.x); }
    const size_t nl = X.size();
    x_stride = align4(max_rec + 1);   // + the record's tag
    const size_t entries = 16 + 2 * (size_t)world * x_stride;
    const size_t n_sc = 3 * 32 + 1 + (size_t)n + 8;
    bool ok = true;
    std::string why;
    std::vector<cudaIpcMemHandle_t> mine(nl);
    for (size_t i = 0; i < nl && ok; ++i) {
        if (cudaMalloc(&X[i]->base, entries * sizeof(F)) != cudaSuccess) { ok = false; why = "cudaMalloc"; X[i]->base = nullptr; break; }
        CK(cudaMemsetAsync(X[i]->base, 0, entries * sizeof(F), stream));
        X[i]->d_sc.alloc(n_sc);
        CK(cudaMemsetAsync(X[i]->d_sc.p, 0, n_sc * sizeof(F), stream));
        X[i]->ticket.alloc(4);
        CK(cudaMemsetAsync(X[i]->ticket.p, 0, 4 * sizeof(unsigned int), stream));
        X[i]->seq = 0;
        if (cudaIpcGetMemHandle(&mine[i], X[i]->base) != cudaSuccess) { ok = false; why = "cudaIpcGetMemHandle"; }
    }
    cudaGetLastError();
    CK(cudaStreamSynchronize(stream));
    // all-gather the handles (64 bytes each)
    const size_t hb = sizeof(cudaIpcMemHandle_t), per = nl * hb + 8;   // + this rank's "ok so far"
    DBuf<unsigned char> d_mine, d_all;
    d_mine.alloc(per);
    d_all.alloc(per * world);
    std::vector<unsigned char> h_mine(per, 0), h_all(per * world, 0);
    memcpy(h_mine.data(), mine.data(), nl * hb);
    h_mine[nl * hb] = ok ? 1 : 0;
    CK(cudaMemcpyAsync(d_mine.p, h_mine.data(), per, cudaMemcpyHostToDevice, stream));
    NCK(g_nccl.AllGather(d_mine.p, d_all.p, per, /*ncclUint8*/ 1, comm, stream));
    CK(cudaMemcpyAsync(h_all.data(), d_all.p, per * world, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    for (int q = 0; q < world; ++q) ok = ok && h_all[(size_t)q * per + nl * hb] == 1;
    if (ok)
        for (int q = 0; q < world && ok; ++q)
            for (size_t i = 0; i < nl && ok; ++i) {
                if (q == rank) { X[i]->peer[q] = X[i]->base; continue; }
                cudaIpcMemHandle_t h;
                memcpy(&h, h_all.data() + (size_t)q * per + i * hb, hb);
                void* ptr = nullptr;
                const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
                if (e != cudaSuccess) { ok = false; why = std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorString(e); cudaGetLastError(); break; }
                ipc_opened.push_back(ptr);
                X[i]->peer[q] = (F*)ptr;
            }
    // second agreement: did every rank map every peer?
    h_mine[0] = ok ? 1 : 0;
    CK(cudaMemcpyAsync(d_mine.p, h_mine.data(), 8, cudaMemcpyHostToDevice, stream));
    NCK(g_nccl.AllGather(d_mine.p, d_all.p, 8, /*ncclUint8*/ 1, comm, stream));
    CK(cudaMemcpyAsync(h_all.data(), d_all.p, (size_t)8 * world, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    for (int q = 0; q < world; ++q) ok = ok && h_all[(size_t)q * 8] == 1;
    use_ipc = ok;
    d_xerr.alloc(1);
    CK(cudaMemsetAsync(d_xerr.p, 0, sizeof(unsigned int), stream));
    if (!ok) {
        if (rank == 0 || !why.empty())
            fprintf(stderr, "virgo_b200[rank %d]: NVLink exchange unavailable (%s), using NCCL all-gathers\n", rank, why.empty() ? "a peer failed" : why.c_str());
        if (pc) pc_destroy(pc);
        for (void* q : ipc_opened) cudaIpcCloseMemHandle(q);
        ipc_opened.clear();
    }
}

// ------------------------------------------------------------------ steps
void Engine::load_inputs(const uint64_t* host, size_t cnt, bool from_host) {
    if (cnt != C.layer_size(0)) throw CudaError{"vp_set_inputs: wrong number of inputs"};
    pending_chunks = 0;
    if (from_host) {   // only the instances this rank evaluates
        const size_t S0 = C.layers[0].size, b = (size_t)k_lo * S0, e = (size_t)k_hi * S0;
        if (e > b) CK(cudaMemcpyAsync(d_inputs.p + b, host + b, (e - b) * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    }
    inputs_loaded = true;
    evaluated = false;
}

// vp_prove with host buffers: the upload is cut into IN_CHUNKS instance ranges on a copy stream, and evaluate() walks
// the same ranges, each behind its chunk's event, so that all but the first chunk's copy overlaps evaluation
// (the upload of 59 MB is 1.1 ms of the C3 end-to-end step; evaluate is 0.8 ms).
void Engine::load_inputs_chunked(const uint64_t* host, size_t cnt, bool local) {
    if (local) {   // `host` holds only the instances [k_lo, k_hi) this rank uploads (vp_input_range)
        if (cnt != (size_t)(k_hi - k_lo) * C.layers[0].size) throw CudaError{"vp_prove_local: wrong number of inputs for this rank's instance range"};
        host -= (size_t)k_lo * C.layers[0].size;
    } else if (cnt != C.layer_size(0)) throw CudaError{"vp_prove: wrong number of inputs"};
    if (!copy_stream) {
        CK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        for (auto& e : ev_chunk) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_copy_go, cudaEventDisableTiming));
    }
    if (!ev_extra) CK(cudaEventCreateWithFlags(&ev_extra, cudaEventDisableTiming));
    const uint32_t span = core_hi - core_lo;
    const int nc = span >= 64 ? IN_CHUNKS : 1;
    CK(cudaEventRecord(ev_copy_go, stream));              // after everything queued so far (the previous proof read d_inputs)
    CK(cudaStreamWaitEvent(copy_stream, ev_copy_go, 0));
    const size_t S0 = C.layers[0].size;
    for (int c = 0; c < nc; ++c) {
        chunk_lo[c] = core_lo + (uint32_t)((uint64_t)span * c / nc);
        chunk_hi[c] = core_lo + (uint32_t)((uint64_t)span * (c + 1) / nc);
        const size_t b = (size_t)chunk_lo[c] * S0, e = (size_t)chunk_hi[c] * S0;
        if (e > b) CK(cudaMemcpyAsync(d_inputs.p + b, host + b, (e - b) * sizeof(uint64_t), cudaMemcpyHostToDevice, copy_stream));
        CK(cudaEventRecord(ev_chunk[c], copy_stream));
    }
    // the extra layer-0 instances left and right of the core range: copy + convert on the copy stream, off the critical path
    extras_pending = false;
    const uint32_t ex[2][2] = {{k_lo, core_lo}, {core_hi, k_hi}};
    for (int q = 0; q < 2; ++q) {
        const size_t b = (size_t)ex[q][0] * S0, e = (size_t)ex[q][1] * S0;
        if (e <= b) continue;
        CK(cudaMemcpyAsync(d_inputs.p + b, host + b, (e - b) * sizeof(uint64_t), cudaMemcpyHostToDevice, copy_stream));
        k_load_inputs<<<cdiv((uint32_t)(e - b), 256), 256, 0, copy_stream>>>(d_inputs.p, val[0].p, (uint32_t)b, (uint32_t)e);
        ++launches;
        extras_pending = true;
    }
    if (extras_pending) CK(cudaEventRecord(ev_extra, copy_stream));
    pending_chunks = nc;
    inputs_loaded = true;
    evaluated = false;
}

// A batch of n_stmt statements (unsharded) is one replicated circuit of n_stmt * K instances here.
void Engine::evaluate() {
    const uint32_t S0 = (uint32_t)C.layers[0].size;
    memset_stmts(d_counter.p + 1, sizeof(unsigned int));
    const int nc = pending_chunks > 0 ? pending_chunks : 1;
    for (int c = 0; c < nc; ++c) {
        const uint32_t ca = pending_chunks > 0 ? chunk_lo[c] : k_lo, cb = pending_chunks > 0 ? chunk_hi[c] : k_hi * n_stmt;
        if (pending_chunks > 0) CK(cudaStreamWaitEvent(stream, ev_chunk[c], 0));
        if (cb > ca) {
            k_load_inputs<<<cdiv(std::max<uint32_t>((cb - ca) * S0, 1), 256), 256, 0, stream>>>(d_inputs.p, val[0].p, ca * S0, cb * S0);
            ++launches;
        }
        for (int i = 1; i < n; ++i) {
            const uint32_t a = std::max(ca, ev_lo[i]), b = std::min(cb, ev_hi[i] * n_stmt);
            if (b <= a) continue;
            const uint32_t gb = a * L[i].S, ge = b * L[i].S, tot = ge - gb;
            size_t h = prof_begin(KC_EVAL);
            k_eval_layer<<<grid_for(std::max<uint32_t>(tot, 1), cap_eval), 256, 0, stream>>>(L[i].G, L[i].S, K, i, d_valptr.p, d_sizes.p,
                                                                                            val[i].p, d_counter.p + 1, gb, ge, values_real ? 1 : 0,
                                                                                            sstride);
            prof_end(h, (double)tot * (16.0 + 32.0 + 11.0 / K));  // out + two operand gathers (+ amortised wiring)
            ++launches;
        }
    }
    pending_chunks = 0;
    CK(cudaGetLastError());
    evaluated = true;
}

void Engine::run_eq(uint32_t first, uint32_t count) {
    if (!count) return;
    k_eq_build<<<sgrid(count), 1024, 0, stream>>>(d_eqb.p + first, d_chal.p, d_eq.p + eq_off, sstride);
    ++launches;
}

// <X, eq(r,.)> over the replicated layer of template size S. Sharded: every rank sums its own instance slice, the
// partial sums meet in one 16-byte-per-rank all-gather.
void Engine::run_dot_eq(const F* X, uint32_t S, EqTab eq, F* out, bool local_only) {
    const uint32_t begin = ko_lo * S, end = ko_hi * S;
    F* dst = (world > 1 && !local_only) ? d_send.p : out;
    k_dot_eq<<<sgrid(grid_b(std::max<uint32_t>(end - begin, 1), cap_dot)), 256, 0, stream>>>(X, begin, end, eq, dst, d_partials.p,
                                                                                            d_counter.p, sstride);
    ++launches;
    if (world > 1 && !local_only) {
        NCK(g_nccl.AllGather(d_send.p, d_recv.p, 2, /*ncclUint64*/ 5, comm, stream));
        k_sum_ranks<<<1, 32, 0, stream>>>(d_recv.p, (uint32_t)world, 1, out);
        ++launches;
    }
}

void Engine::do_vres() {
    run_eq(eqb_out, 2);
    run_dot_eq(val[n - 1].p, (uint32_t)C.layers[n - 1].size, eqtab(2, C.bit_length(n - 1)), d_tr.p + lay.tr_vres);
}

void Engine::do_input_mle() {
    run_eq(eqb_in, 2);
    run_dot_eq(val[0].p, (uint32_t)C.layers[0].size, eqtab(2, C.bit_length(0)), d_tr.p + lay.tr_input);
}

void Engine::do_init_phase1(int i) {
    LayerDev& D = L[i];
    run_eq(D.eqb_g, 2);
    const uint32_t S_pre = L[i - 1].S ? L[i - 1].S : (uint32_t)C.layers[i - 1].size;
    const uint32_t tot = (uint32_t)C.layer_size(i - 1);
    CsrP1 csr{D.p1_g0.p, D.p1_v0.p, D.p1_tyl.p};
    const uint32_t k0 = D.ph1.sharded ? D.p1_k0 : 0, k1 = D.ph1.sharded ? D.p1_k1 : K;
    const uint64_t work = (uint64_t)D.p1_items.n * (k1 - k0);
    size_t h = prof_begin(KC_INIT1);
    if (values_real && K >= 8 && k1 - k0 >= 4 && n <= 64) {   // template-major: an item of the template x 4 instances per thread
        dim3 grid(cdiv(std::max<uint32_t>((uint32_t)D.p1_items.n, 1), 256), cdiv(k1 - k0, 4), n_stmt);
        k_init_phase1_real_tm<4><<<grid, 256, 0, stream>>>(
            D.p1_items.p, (uint32_t)D.p1_items.n, csr, S_pre, D.S, K, eqtab(0, C.bit_length(i)), d_chal.p + D.ci_assert,
            d_valptr.p, d_sizes.p, D.c.p, val[i - 1].p, bufV[0].p + D.ph1.tab_off[0], bufM[0].p + D.ph1.tab_off[0],
            bufA[0].p + D.ph1.tab_off[0], d_rowpart.p, D.p1_nslots, direct_v ? 0 : 1, (uint32_t)i, D.ph1.maps[0], k0, k1, sstride);
    } else if (values_real && work < 0xffffffffull && n <= 64)
        k_init_phase1_real<<<sgrid(grid_b((uint32_t)std::min<uint64_t>(work, 0xffffffffu), cap_p1il)), 256, 0, stream>>>(
            D.p1_items.p, (uint32_t)D.p1_items.n, csr, S_pre, D.S, K, eqtab(0, C.bit_length(i)), d_chal.p + D.ci_assert,
            d_valptr.p, d_sizes.p, D.c.p, val[i - 1].p, bufV[0].p + D.ph1.tab_off[0], bufM[0].p + D.ph1.tab_off[0],
            bufA[0].p + D.ph1.tab_off[0], d_rowpart.p, D.p1_nslots, D.ph1.maps[0], direct_v ? 0 : 1, k0, k1, (uint32_t)i, sstride);
    else
    k_init_phase1<<<sgrid(grid_b((uint32_t)std::min<uint64_t>(work, 0xffffffffu), cap_p1)), 256, 0, stream>>>(
        D.p1_items.p, (uint32_t)D.p1_items.n, csr, S_pre, D.S, K, eqtab(0, C.bit_length(i)), d_chal.p + D.ci_assert,
        d_valptr.p, d_sizes.p, D.c.p, val[i - 1].p, bufV[0].p + D.ph1.tab_off[0], bufM[0].p + D.ph1.tab_off[0],
        bufA[0].p + D.ph1.tab_off[0], d_rowpart.p, D.p1_nslots, D.ph1.maps[0], direct_v ? 0 : 1, k0, k1, sstride);
    if (D.p1_long.n && k1 > k0) {
        k_combine_phase1<<<sgrid(grid_b((uint32_t)(D.p1_long.n * (k1 - k0)), cap_comb)), 256, 0, stream>>>(
            D.p1_long.p, (uint32_t)D.p1_long.n, S_pre, K, val[i - 1].p, bufV[0].p + D.ph1.tab_off[0],
            bufM[0].p + D.ph1.tab_off[0], bufA[0].p + D.ph1.tab_off[0], d_rowpart.p, D.p1_nslots, D.ph1.maps[0], direct_v ? 0 : 1, k0, k1,
            sstride);
        ++launches;
    }
    // per output this rank holds: V read + 3 table writes; per gate it visits: one gathered operand
    const double rows1 = D.ph1.sharded ? (double)(D.ph1.row_hi[0] - D.ph1.row_lo[0]) : (double)tot;
    prof_end(h, rows1 * (direct_v ? 32.0 : 64.0) + (double)D.S * (k1 - k0) * 16.0);
    ++launches;
    have_equ = false;
}

void Engine::do_init_phase2(int i) {
    LayerDev& D = L[i];
    const uint32_t S_pre = (uint32_t)C.layers[i - 1].size;
    if (on_lane2) run_eq(D.eqb_g2, 4);   // beta_g and beta_u: adjacent descriptors, one launch
    else { run_eq(D.eqb_u, 2); have_equ = true; }
    const EqTab eqg = eqtab(on_lane2 ? region_g_lane2 : 0, C.bit_length(i)), equ = eqtab(on_lane2 ? region_u_lane2 : 1, C.bit_length(i - 1));
    const F* Vu = on_lane2 ? d_vu.p + i : scal(SC_VU);
    if (D.p2_ntabs > 0) {
        CsrP2 csr{D.p2_g0.p, D.p2_u0.p, D.p2_ty.p};
        const uint32_t kk0 = D.ph2.sharded ? D.p2_kk0 : 0, kk1 = D.ph2.sharded ? D.p2_kk1 : K;
        const uint64_t work = (uint64_t)D.p2_items.n * (kk1 - kk0);
        size_t h = prof_begin(KC_INIT2);
        if (work < 0xffffffffull && !old_p2) {
            // few distinct second-half eq factors per instance: tabulate their products (k_p2_hs), two products per gate
            HsTab H{nullptr, 0, 0};
            const uint32_t ng = (D.S >> eqg.fh) + 2, nu = (S_pre >> equ.fh) + 2;
            if (K >= 8 && (uint64_t)ng * nu <= 64 && (uint64_t)K * ng * nu <= d_hs.n && !getenv_no_hs) {
                H = HsTab{d_hs.p, ng, nu};
                k_p2_hs<<<sgrid(grid_b(K * ng * nu, cap_dot)), 256, 0, stream>>>(eqg, equ, D.S, S_pre, K, ng, nu, d_hs.p, sstride);
                ++launches;
            }
            k_init_phase2_v2<<<sgrid(grid_b((uint32_t)work, cap_p2v2)), 256, 0, stream>>>(
                D.p2_items.p, (uint32_t)D.p2_items.n, D.p2_tabs.p, csr, S_pre, D.S, K, eqg, equ, d_chal.p + D.ci_assert,
                Vu, bufV[0].p, bufM[0].p, bufA[0].p, d_rowpart.p, D.p2_nslots, kk0, kk1, H, sstride);
        }
        else
        k_init_phase2<<<sgrid(grid_b((uint32_t)std::min<uint64_t>(work, 0xffffffffu), cap_p2)), 256, 0, stream>>>(
            D.p2_items.p, (uint32_t)D.p2_items.n, D.p2_tabs.p, csr, S_pre, D.S, K, eqg, equ, d_chal.p + D.ci_assert,
            Vu, bufV[0].p, bufM[0].p, bufA[0].p, d_rowpart.p, D.p2_nslots, kk0, kk1, sstride);
        if (D.p2_long.n && kk1 > kk0) {
            k_combine_phase2<<<sgrid(grid_b((uint32_t)(D.p2_long.n * (kk1 - kk0)), cap_comb)), 256, 0, stream>>>(
                D.p2_long.p, (uint32_t)D.p2_long.n, D.p2_tabs.p, K, bufV[0].p, bufM[0].p, bufA[0].p, d_rowpart.p, D.p2_nslots, kk0,
                kk1, sstride);
            ++launches;
        }
        double rows2 = D.p2_out_entries;   // table entries this rank holds
        if (D.ph2.sharded) { rows2 = 0; for (size_t t = 0; t < D.ph2.row_hi.size(); ++t) rows2 += (double)(D.ph2.row_hi[t] - D.ph2.row_lo[t]); }
        prof_end(h, rows2 * 64.0 + (double)D.p2_gates * (kk1 - kk0) * 16.0);
        ++launches;
    }
    // unary gates: their sum starts the phase's add_term (see k_phase2_unary); each rank sums its instance slice
    const bool slice = D.ph2.sharded;  // a replicated phase needs the whole sum on every rank
    const uint32_t k0 = slice ? ko_lo : 0, k1 = slice ? ko_hi : K;
    if (D.n_unary > 0 && k1 > k0) {
        CsrUnary un{D.un_g0.p, D.un_u0.p, D.un_ty.p, D.n_unary};
        const uint64_t tot = (uint64_t)D.n_unary * (k1 - k0);
        k_phase2_unary<<<sgrid(grid_b((uint32_t)std::min<uint64_t>(tot, 0xffffffffu), cap_un)), 256, 0, stream>>>(
            un, S_pre, D.S, K, eqg, equ, d_chal.p + D.ci_assert, Vu, D.c.p, scal(SC_UNARY), d_partials.p,
            d_counter.p, k0, k1, sstride);
        ++launches;
    } else memset_stmts(scal(SC_UNARY), sizeof(F));
}

void Engine::do_init_liu(int i, bool write_a) {
    LayerDev& D = L[i];
    const uint32_t S_pre = (uint32_t)C.layers[i - 1].size;
    const uint32_t reg_u = on_lane1 ? region_u_lane1 : 1;
    if (on_lane1) run_eq(D.eqb_u1, 2 + D.n_eqb_liu);   // scaled beta_u + the Liu tables: adjacent descriptors, one launch
    else {
        if (!have_equ) run_eq(D.eqb_u, 2);
        have_equ = false;
        run_eq(D.eqb_liu, D.n_eqb_liu);
    }
    const uint32_t tot = (uint32_t)C.layer_size(i - 1);
    size_t h = prof_begin(KC_INIT_LIU);
    const uint32_t n_local = D.ph3.sharded ? D.ph3.local_len[0] : tot;
    // the instances this rank's rows of the table touch (all of them on an unsharded context)
    uint32_t lk0 = 0, lk1 = K;
    if (D.ph3.sharded) {
        lk0 = lk1 = 0;
        if (D.ph3.row_hi[0] > D.ph3.row_lo[0]) { lk0 = D.ph3.row_lo[0] / S_pre; lk1 = std::min(K, (D.ph3.row_hi[0] - 1) / S_pre + 1); }
    }
    if (K >= 8 && lk1 - lk0 >= 8) {   // template-major: one thread per template entry, a chunk of instances each
        const uint32_t k_chunk = 8;
        dim3 grid(cdiv(S_pre, 256), cdiv(lk1 - lk0, k_chunk), n_stmt);
        k_init_liu_tm<<<grid, 256, 0, stream>>>(D.liu_off.p, D.liu_perm.p, D.liu_ent.p, eq_off ? D.liu_eqtabs_b.p : D.liu_eqtabs.p, S_pre, K, k_chunk,
                                               eqtab(reg_u, C.bit_length(i - 1)), d_chal.p + D.ci_sig, val[i - 1].p, bufV[0].p + D.ph3.tab_off[0],
                                               bufM[0].p + D.ph3.tab_off[0], bufA[0].p + D.ph3.tab_off[0], write_a ? 1 : 0, on_lane1 ? 1 : 0, direct_v ? 0 : 1,
                                               D.ph3.maps[0], lk0, lk1, sstride);
    } else
    k_init_liu<<<sgrid(grid_b(std::max<uint32_t>(n_local, 1), cap_liu)), 256, 0, stream>>>(
        D.liu_off.p, world == 1 ? D.liu_perm.p : nullptr, D.liu_ent.p, eq_off ? D.liu_eqtabs_b.p : D.liu_eqtabs.p, S_pre, K, eqtab(reg_u, C.bit_length(i - 1)), d_chal.p + D.ci_sig, val[i - 1].p,
        bufV[0].p + D.ph3.tab_off[0], bufM[0].p + D.ph3.tab_off[0], bufA[0].p + D.ph3.tab_off[0], D.ph3.maps[0], n_local,
        write_a ? 1 : 0, on_lane1 ? 1 : 0, direct_v ? 0 : 1, sstride);
    prof_end(h, (double)n_local * ((write_a ? 64.0 : 48.0) - (direct_v ? 32.0 : 0.0)));
    ++launches;
}

// round j (1-based) of plan P; ci_prev = challenge index of the previous round's challenge (j >= 2)
// continues: round 1 of the PLAN is not round 1 of the phase (stage B of a sharded phase): add_term carries over and is
// scaled by (1 - previous challenge) although no fold is pending. poly_out: where the polynomial goes (default: transcript).
void Engine::do_round(const SumcheckPlan& P, int j, uint32_t ci_prev, uint32_t tr_out, const F* at_init, bool continues, F* poly_out) {
    const RoundPlan& R = P.r[j - 1];
    RoundArgs a{};
    if (fast_prev) {
        a.prev_by_value = 1;
        a.prev_val = F{fast_prev->re, fast_prev->im};
        a.prev_w = d_chal.p + ci_prev;
    }
    if (fast_out) {
        a.host_poly = d_round->poly;
        a.host_seq = &d_round->seq;
        a.seq = ++round_seq;
    }
    const int ib = R.in_buf, ob = ib ^ 1;
    a.inV = bufV[ib].p; a.inM = bufM[ib].p; a.inA = bufA[ib].p;
    a.outV = bufV[ob].p; a.outM = bufM[ob].p; a.outA = bufA[ob].p;
    a.tabs = d_tabs.p + R.tab_begin;
    a.cols = d_cols.p + R.col_begin;
    a.n_tabs = R.n_tabs;
    a.n_cols = R.n_cols;
    a.prev_r = d_chal.p + ci_prev;
    a.add_term = scal(SC_ADD_TERM);
    a.claims = d_claims.p;
    a.out_poly = poly_out ? poly_out : d_tr.p + tr_out;
    a.partials = d_partials.p;
    a.counter = d_counter.p;
    a.first_round = j == 1 && !continues;
    a.reset_add_term = j == 1 && !continues;
    a.at_init = at_init;
    const int grid = grid_for(R.work, R.fold ? cap_round : cap_round1);
    size_t h = prof_begin(R.fold ? KC_ROUND_FOLD : KC_ROUND_FIRST);
    if (R.fold) k_round<true><<<grid, 256, 0, stream>>>(a);
    else k_round<false><<<grid, 256, 0, stream>>>(a);
    prof_end(h, R.bytes);
    ++launches;
}

// Round j (1-based) of a SHARDED phase through the method-by-method API (collective: every rank makes the same call).
// Rounds 1..m fold this rank's table rows (planA): the partial round polynomials -- which carry the rank's partial
// add_term -- meet in one 48-byte-per-rank all-gather and are summed (SURVEY 8(e): the per-round exchange of an
// interactive sharded prover). Before round m + 1 the blocks' two stored values are folded with r_m and gathered
// together with the partial add_term and the locally collapsed claims (k_fold_only + all-gather + k_shard_merge); the
// remaining rounds run replicated on every rank (planB), so no further communication is needed.
void Engine::sharded_round(const PhasePlan& PP, int phase, int j, uint32_t ci, uint32_t tr, const F* at_init) {
    (void)phase;
    if (j == 1) CK(cudaMemsetAsync(d_claims.p, 0, ((size_t)n + 1) * sizeof(F), stream));   // partial claims are summed over the ranks
    if (j <= PP.m) {
        F* part = d_send.p;   // 3 F
        do_round(PP.planA, j, ci + (uint32_t)std::max(0, j - 2), 0, at_init, false, part);
        NCK(g_nccl.AllGather(part, d_recv.p, 6, /*ncclUint64*/ 5, comm, stream));
        k_sum_ranks_vec<<<1, 32, 0, stream>>>(d_recv.p, (uint32_t)world, 3, d_tr.p + tr);
        ++launches;
        return;
    }
    if (j == PP.m + 1) {
        F* rec = d_send.p;
        const uint32_t sc0 = PP.sc_base + PP.n_poly;   // record: table regions, (unused polynomials), add_term, claims
        CK(cudaMemsetAsync(rec, 0, (size_t)PP.rec_len * sizeof(F), stream));
        fold_only(PP, PP.foi_begin, PP.planA.fin_buf, ci);
        CK(cudaMemcpyAsync(rec + sc0, scal(SC_ADD_TERM), sizeof(F), cudaMemcpyDeviceToDevice, stream));
        CK(cudaMemcpyAsync(rec + sc0 + 1, d_claims.p, (size_t)PP.n_claims * sizeof(F), cudaMemcpyDeviceToDevice, stream));
        NCK(g_nccl.AllGather(rec, d_recv.p, (size_t)PP.rec_len * 2, /*ncclUint64*/ 5, comm, stream));
        // no polynomials in this record: scalar 0 is add_term, then the claims (out_poly is not written)
        k_shard_merge<<<8, 256, 0, stream>>>(merge_args(PP, sc0, 0, d_send.p));
        ++launches;
        do_round(PP.planB, 1, ci + (uint32_t)(PP.m - 1), tr, nullptr, /*continues=*/true);
        return;
    }
    do_round(PP.planB, j - PP.m, ci + (uint32_t)(j - 2), tr, nullptr);
}

void Engine::do_finalize(const SumcheckPlan& P, uint32_t ci_last, F* keep) {
    const int fb = P.fin_buf;
    k_finalize<<<cdiv(P.n_fin, 128), 128, 0, stream>>>(d_fins.p + P.fin_begin, (int)P.n_fin, bufV[fb].p,
                                                        d_chal.p + ci_last, P.rounds >= 1 ? 1 : 0, d_claims.p, d_tr.p,
                                                        keep);
    ++launches;
}

// One cooperative launch of k_phase_dfs (two rounds per pass) over `P`.
static const void* dfs_kernel_ptr(bool has_a, int first) {
    if (first == DFS_VREAL) return has_a ? (const void*)k_phase_dfs<true, DFS_VREAL> : (const void*)k_phase_dfs<false, DFS_VREAL>;
    if (first == DFS_NEED_B) return (const void*)k_phase_dfs<true, DFS_NEED_B>;
    return has_a ? (const void*)k_phase_dfs<true, DFS_PLAIN> : (const void*)k_phase_dfs<false, DFS_PLAIN>;
}
void Engine::launch_dfs_kernel(const PassPlan& P, uint32_t ci, uint32_t round_base, const F* at_init, F* add_term_out,
                               F* claims, F* out_poly, F* keep, bool has_a, int first, const F* v_first) {
    DfsArgs a;
    for (int b = 0; b < 2; ++b) { a.bufV[b] = bufV[b].p; a.bufM[b] = bufM[b].p; a.bufA[b] = bufA[b].p; }
    a.passes = d_pdev.p + P.pass_begin;
    a.tabs = d_ptabs.p;
    a.cols = d_pcols.p;
    a.fins = d_fins.p + P.fin_begin;
    a.n_passes = P.n_passes;
    a.n_fin = P.n_fin;
    a.fin_buf = (uint32_t)P.fin_buf;
    a.tail_work = tail_work;
    a.round_base = round_base;
    a.at_init = at_init;
    a.chal = d_chal.p + ci;
    a.add_term = add_term_out;
    a.claims = claims;
    a.out_poly = out_poly;
    a.transcript = d_tr.p;
    a.keep = keep;
    a.partials = d_partials.p;
    a.bar = d_counter.p + 2;
    a.chunk_ctr = d_counter.p + 4;
    a.v_first = v_first;
    a.claim0 = nullptr;
    a.dbg = nullptr;
    if (P.rounds > 32) throw CudaError{"a sumcheck phase with more than 32 rounds"};
    for (int jr = 0; jr < 32; ++jr) {
        const size_t ix = (size_t)ci + round_base + (size_t)jr;
        a.rk[jr] = make_constk(jr < P.rounds && ix < h_chal.size() ? h_chal[ix] : f_zero());
    }
    // two lanes: leave a few block slots free so that the other lane's (cooperative) phase kernel can start as soon as
    // this one is down to its small passes
    // three lanes: two of the three block slots of an SM, so that the other lanes' kernels (gather-latency bound inits,
    // another phase's passes) are co-resident with a compute-bound pass (measured: C3 13.3 -> 12.9 ms)
    // six lanes: 1.25 blocks per SM per pass kernel (of three slots) -- measured on C3: 444 blocks 11.33 ms, 296 10.95, 222 10.65,
    // 185 10.78, 148 10.75, 111 11.02, 74 11.7; the 65 x 2^20 random circuit prefers 148 (profiles/r2b_dfs_grid_sweep.txt)
    uint32_t cap = six_lanes ? (uint32_t)std::max(2, std::min(cap_dfs, 5 * n_sm / 4))
                 : three_lanes ? (uint32_t)std::max(2, 2 * cap_dfs / 3) : two_lanes ? (uint32_t)std::max(1, cap_dfs - 8) : (uint32_t)cap_dfs;
    if (dfs_grid_override) cap = std::max<uint32_t>(2, std::min<uint32_t>((uint32_t)dfs_grid_override, (uint32_t)cap_dfs));
    // block 0 coordinates, blocks 1.. work; a phase that fits one block runs on block 0 alone
    const int grid = P.max_work <= DFS_CHUNK ? 1 : (int)std::min<uint32_t>(cdiv(P.max_work, DFS_CHUNK) + 1, std::max<uint32_t>(cap, 2));
    void* args[] = {&a};
    size_t h = prof_begin(KC_ROUND_FOLD);
    CK(cudaLaunchCooperativeKernel(dfs_kernel_ptr(has_a, first), dim3(grid), dim3(DFS_THREADS), args, DFS_DYN_SMEM, stream));
    prof_end(h, P.alg_bytes);
    ++launches;
}

// The hand-over of a sharded phase over NCCL (sharded_round, do_phase), first step: k_fold_only writes the level-m value of
// every block of stage A's final buffer fin_buf into the record at d_send, folding a pending pair with r_m.
void Engine::fold_only(const PhasePlan& P, uint32_t fo_begin, int fin_buf, uint32_t ci) {
    if (!P.n_fo) return;
    const FoldOnlyDesc& f0 = arena.fo[fo_begin];
    dim3 grid(std::max<uint32_t>(1, std::min<uint32_t>(cdiv(f0.cnt, 128), 64)), P.n_fo);
    k_fold_only<<<grid, 128, 0, stream>>>(d_fo.p + fo_begin, (int)P.n_fo, bufV[fin_buf].p, bufM[fin_buf].p, bufA[fin_buf].p,
                                         d_chal.p + ci + (uint32_t)(P.m - 1), d_send.p);
    ++launches;
}

// The merge of the gathered records of a sharded phase (k_shard_merge, k_xchg): the stage-B tables, and the sums of the
// record's scalars from sc_base on -- n_poly polynomial coefficients to out_poly, add_term, the claims.
MergeArgs Engine::merge_args(const PhasePlan& P, uint32_t sc_base, uint32_t n_poly, F* out_poly) {
    MergeArgs ma;
    ma.recv = d_recv.p;
    ma.rec_len = P.rec_len;
    ma.G = (uint32_t)world;
    ma.tabs = d_mt.p + P.mt_begin;
    ma.n_tabs = P.n_mt;
    ma.sc_base = sc_base;
    ma.n_poly = n_poly;
    ma.n_claims = P.n_claims;
    ma.outV = bufV[0].p; ma.outM = bufM[0].p; ma.outA = bufA[0].p;
    ma.out_poly = out_poly;
    ma.add_term = scal(SC_ADD_TERM);
    ma.claims = d_claims.p;
    return ma;
}

// All rounds + the final claims of one sumcheck phase. Unsharded: one cooperative launch. Sharded: the m local
// rounds on this rank's blocks, fold-only, ONE all-gather of the per-rank records (collapsed blocks + partial
// round polynomials + partial add_term + claims), merge, then the remaining rounds replicated on every rank.
void Engine::do_phase(const PhasePlan& P, uint32_t ci, uint32_t tr_rounds, F* keep, const F* at_init, bool has_a,
                      const F* v_first) {
    const int first = values_real ? DFS_VREAL : DFS_PLAIN;
    if (!P.sharded) {
        launch_dfs_kernel(P.ppB, ci, 0, at_init, scal(SC_ADD_TERM), d_claims.p, d_tr.p + tr_rounds, keep, has_a, first, v_first);
        return;
    }
    // phase 1 / Liu (one table over layer i-1): the local rows [lo, hi) of V are read straight from circuitValue[i-1]
    const F* v_local = (v_first && P.maps.size() == 1 && P.tab_off[0] == 0) ? v_first + P.maps[0].lo : nullptr;
    if (v_first && !v_local) throw CudaError{"direct V: unexpected table layout"};
    const MergeArgs mg = merge_args(P, P.sc_base, P.n_poly, d_tr.p + tr_rounds);
    if (use_ipc) {
        // stage A leaves its partial scalars in the lane's scalar buffer (zero between phases); ONE kernel pushes the
        // record to every rank over NVLink, waits for theirs and merges
        F* sc = x.d_sc.p;
        launch_dfs_kernel(P.ppA, ci, 0, at_init, sc + P.n_poly, sc + P.n_poly + 1, sc, nullptr, has_a, first, v_local);
        XchgArgs a;
        memset(&a, 0, sizeof a);
        for (int q = 0; q < world; ++q) a.peer[q] = x.peer[q];
        a.world = (uint32_t)world;
        a.me = (uint32_t)rank;
        a.seq = ++x.seq;
        a.slot_stride = x_stride;
        a.buf_off[0] = 16;
        a.buf_off[1] = 16 + (uint32_t)world * x_stride;
        a.rec_len = P.rec_len;
        a.fo = d_fo.p + P.fo_begin;
        a.n_fo = P.n_fo;
        const int fb = P.ppA.fin_buf;
        a.V = bufV[fb].p; a.M = bufM[fb].p; a.A = bufA[fb].p;
        a.has_a = has_a ? 1 : 0;
        a.sc = sc;
        a.sc_base = P.sc_base;
        a.n_sc = P.n_poly + 1 + P.n_claims;
        a.ticket = x.ticket.p;
        a.tag = tr_rounds;
        a.err = d_xerr.p;
        a.mg = mg;
        const int grid = (int)std::max<uint32_t>(2, std::min<uint32_t>(cdiv(P.rec_len, 512), 32));
        k_xchg<<<grid, 256, 0, stream>>>(a);
        ++launches;
    } else {
        F* rec = d_send.p;
        F* sc = rec + P.sc_base;
        CK(cudaMemsetAsync(sc, 0, (size_t)(P.n_poly + 1 + P.n_claims) * sizeof(F), stream));
        // stage A: partial polynomials, add_term and claims go straight into the record's scalar region
        launch_dfs_kernel(P.ppA, ci, 0, at_init, sc + P.n_poly, sc + P.n_poly + 1, sc, nullptr, has_a, first, v_local);
        fold_only(P, P.fo_begin, P.ppA.fin_buf, ci);
        NCK(g_nccl.AllGather(rec, d_recv.p, (size_t)P.rec_len * 2, /*ncclUint64*/ 5, comm, stream));
        k_shard_merge<<<8, 256, 0, stream>>>(mg);
        ++launches;
    }
    // stage B: replicated; starts from the summed add_term
    launch_dfs_kernel(P.ppB, ci, (uint32_t)P.m, scal(SC_ADD_TERM), scal(SC_ADD_TERM), d_claims.p,
                      d_tr.p + tr_rounds + 3u * (uint32_t)P.m, keep, has_a, DFS_PLAIN);
}

// Fill in the b coefficient of every round polynomial from the claim chain (k_derive_b); the transcript is complete
// (and, on a sharded context, replicated) when this runs.
void Engine::derive_b() {
    if (!n_chains) return;
    k_derive_b<<<cdiv((uint32_t)n_chains, 4), 128, 0, stream>>>(d_chains.p, n_chains, d_chain_segs.p, d_chain_terms.p, d_chal.p,
                                                             d_tr.p, nullptr);
    ++launches;
}

// ------------------------------------------------------------------ verifier (SURVEY 8(f) N2)
static int vf_binary_index(int ty) {
    switch (ty) {
        case T_ADD: return 0; case T_SUB: return 1; case T_ANTISUB: return 2; case T_MUL: return 3;
        case T_NAAB: return 4; case T_ANTINAAB: return 5; case T_XOR: return 6; default: return -1;
    }
}
// gates of layer i in bucket order (one bucket per accumulator of verifier.cpp:63-113) + the Liu segments
void Engine::verify_prepare(int i) {
    LayerDev& D = L[i];
    if (D.vf_ready) return;
    const Layer& T = C.layers[i];
    const uint32_t S = (uint32_t)T.size;
    std::vector<std::pair<uint32_t, uint32_t>> keyed;   // (key, gate)
    for (uint32_t g = 0; g < S; ++g) {
        const int ty = T.ty[g], bi = vf_binary_index(ty);
        uint32_t key;
        if (bi >= 0) key = 4u + 7u * (uint32_t)T.l[g] + (uint32_t)bi;
        else if (ty == T_COPY) key = 0;
        else if (ty == T_NOT) key = 1;
        else if (ty == T_ADDC) key = 2;
        else if (ty == T_MULC) key = 3;
        else continue;
        keyed.push_back({key, g});
    }
    {   // stable counting sort by key (keys < 4 + 7 * layers): a comparison sort of 2^20 gates x 64 layers took seconds
        const uint32_t n_keys = 4u + 7u * (uint32_t)n;
        std::vector<uint32_t> start(n_keys + 1, 0);
        for (const auto& kg : keyed) ++start[kg.first + 1];
        for (uint32_t k = 0; k < n_keys; ++k) start[k + 1] += start[k];
        std::vector<std::pair<uint32_t, uint32_t>> sorted(keyed.size());
        for (const auto& kg : keyed) sorted[start[kg.first]++] = kg;
        keyed.swap(sorted);
    }
    std::vector<VfGate> gates(keyed.size());
    std::vector<VfBucket> buckets;
    D.vf_key.clear();
    for (size_t x = 0; x < keyed.size(); ++x) {
        const uint32_t key = keyed[x].first, g = keyed[x].second;
        const bool bin = key >= 4;
        gates[x] = VfGate{g, T.u[g], bin ? T.lv[g] : 0u, bin ? (uint32_t)T.l[g] : g};
        if (buckets.empty() || D.vf_key.back() != key) {
            const uint32_t kind = bin ? 3u : key == 2 ? 2u : key == 3 ? 1u : 0u;
            buckets.push_back(VfBucket{(uint32_t)x, 0, kind, bin ? (uint32_t)T.dadSize[(key - 4) / 7] : 0u});
            D.vf_key.push_back(key);
        }
        ++buckets.back().cnt;
    }
    if (!gates.empty()) { D.vf_gates.upload(gates, stream); D.vf_buckets.upload(buckets, stream); }
    if (!T.is_assert.empty()) D.vf_assert.upload(T.is_assert, stream);
    // Liu segments: layer pre itself, then every source layer j >= i with a non-empty subset in pre (same order as liu_j)
    std::vector<VfLiuSeg> segs;
    segs.push_back(VfLiuSeg{nullptr, (uint32_t)C.layers[i - 1].size, 0, 0});
    for (size_t q = 0; q < D.liu_j.size(); ++q) {
        const LayerDev& J = L[D.liu_j[q]];
        const uint32_t* ids = nullptr;
        uint32_t Dsz = 0;
        for (size_t t = 0; t < J.p2_src.size(); ++t)
            if (J.p2_src[t] == i - 1) { ids = J.h_p2[t].dadId; Dsz = J.h_p2[t].D; }
        if (!ids) throw CudaError{"verify: missing dad subset"};
        segs.push_back(VfLiuSeg{ids, Dsz, (uint32_t)q, 0});
    }
    D.vf_liu.upload(segs, stream);
    D.n_vf_liu = (uint32_t)segs.size();
    CK(cudaStreamSynchronize(stream));   // host vectors go out of scope
    D.vf_ready = true;
}

// Where each layer's sums go: L[i].vf_out; vf_out_total entries per statement, the last two being the input MLE and (a
// batch only) the claimed outputs' MLE at r_out.
void Engine::vf_layout() {
    uint32_t out_total = 0, max_b = 1;
    for (int i = 1; i < n; ++i) {
        verify_prepare(i);
        L[i].vf_out = out_total;
        out_total += 2u * ((uint32_t)L[i].vf_key.size() + L[i].n_vf_liu);
        max_b = std::max<uint32_t>(max_b, std::max<uint32_t>((uint32_t)L[i].vf_key.size(), L[i].n_vf_liu));
    }
    vf_out_total = out_total + 2;
    vf_max_b = max_b;
}

// All O(#gates) sums of every layer and the input MLE into out (vf_out_total entries), with the challenges in d_chal and
// circuitValue[0] loaded. A batch: every statement's sums at once, statement b's out and partial sstride bytes apart; the
// x-width of a bucket shrinks with the batch (as grid_b does) so that a large batch does not launch B x VF_GX blocks.
void Engine::verify_sums_async(F* out, F* partial) {
    const uint32_t gx = std::max<uint32_t>(1, VF_GX / n_stmt);
    for (int i = n - 1; i >= 1; --i) {
        LayerDev& D = L[i];
        const uint32_t S_pre = (uint32_t)C.layers[i - 1].size, nb = (uint32_t)D.vf_key.size();
        const int pb = C.bit_length(i - 1), m = D.m;
        run_eq(D.eqb_g, 2);
        run_eq(D.eqb_u, 2);
        if (m != -1) run_eq(D.eqb_v, 2);
        if (nb) {
            k_verify_sums<<<sgrid(gx, nb), 256, 0, stream>>>(D.vf_buckets.p, D.vf_gates.p, D.vf_assert.p, D.c.p, S_pre, D.S, K,
                                                           eqtab(0, C.bit_length(i)), eqtab(1, pb), eqtab(6 + (uint32_t)n, std::max(m, 0)),
                                                           d_chal.p + D.ci_assert, partial, ko_lo, ko_hi, sstride);
            k_verify_reduce<<<sgrid(nb), 64, 0, stream>>>(partial, gx, out + D.vf_out, sstride);
            launches += 2;
        }
        run_eq(D.eqb_u1, 2);                 // sig[0] * eq(r_u, .)
        run_eq(D.eqb_rl, 2);                 // eq(r_liu, .)
        run_eq(D.eqb_liu, D.n_eqb_liu);      // sig[j - pre] * eq(r_v[j], .)
        k_verify_gr<<<sgrid(gx, D.n_vf_liu), 256, 0, stream>>>(D.vf_liu.p, D.liu_eqtabs.p, eqtab(3 + (uint32_t)n, pb),
                                                              eqtab(7 + (uint32_t)n, pb), S_pre, K, partial, ko_lo, ko_hi, sstride);
        k_verify_reduce<<<sgrid(D.n_vf_liu), 64, 0, stream>>>(partial, gx, out + D.vf_out + 2 * nb, sstride);
        launches += 2;
    }
    run_eq(eqb_in, 2);
    run_dot_eq(val[0].p, (uint32_t)C.layers[0].size, eqtab(2, C.bit_length(0)), out + vf_out_total - 2, /*local_only=*/true);
}

// verifier::verify (verifier.cpp:134-337) on a host transcript; challenges = the stream set by vp_set_challenges /
// vp_prove. Returns 1 (accept) or 0 with the failing check: 1 phase-1 round, 2 phase-2 round, 3 final value of the
// layer, 4 Liu round, 5 Liu final, 6 input layer -- the codes of the CPU oracle's verifier (tests compare them).
int Engine::verify(const F* tr, int* fail_code, int* fail_layer) {
    // Sharded context: a collective call -- every rank passes the same transcript, sums the gates of its own slice of
    // the instances (ko_lo .. ko_hi), and the partial sums of all ranks meet in ONE all-gather before the host checks.
    if (!inputs_loaded) throw CudaError{"vp_verify: inputs not loaded"};
    if (h_chal.size() < lay.n_chal) throw CudaError{"vp_verify: challenges not set"};
    if (active) throw CudaError{"vp_verify: lanes not joined"};
    // ---- device: all O(#gates) sums, every layer, results in one buffer
    vf_layout();
    const uint32_t out_total = vf_out_total;
    if (d_vf_out.n < out_total) d_vf_out.alloc(out_total);
    if (d_vf_partial.n < (size_t)vf_max_b * VF_GX * 2) d_vf_partial.alloc((size_t)vf_max_b * VF_GX * 2);
    {   // circuitValue[0] from the resident inputs (the verifier does not evaluate the circuit)
        const uint32_t S0 = (uint32_t)C.layers[0].size, b0 = k_lo * S0, e0 = k_hi * S0;   // the inputs this rank holds
        k_load_inputs<<<cdiv(std::max<uint32_t>(e0 - b0, 1), 256), 256, 0, stream>>>(d_inputs.p, val[0].p, b0, e0);
        ++launches;
    }
    CK(cudaMemsetAsync(d_vf_out.p, 0, (size_t)out_total * sizeof(F), stream));
    verify_sums_async(d_vf_out.p, d_vf_partial.p);
    if (world > 1) {
        if (d_vf_gather.n < (size_t)out_total * world) d_vf_gather.alloc((size_t)out_total * world);
        NCK(g_nccl.AllGather(d_vf_out.p, d_vf_gather.p, (size_t)out_total * 2, /*ncclUint64*/ 5, comm, stream));
        k_sum_ranks_vec<<<cdiv(out_total, 256), 256, 0, stream>>>(d_vf_gather.p, (uint32_t)world, out_total, d_vf_out.p);
        ++launches;
    }
    std::vector<F> out(out_total);
    CK(cudaMemcpyAsync(out.data(), d_vf_out.p, (size_t)out_total * sizeof(F), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    return verify_check(tr, out.data(), h_chal.data(), fail_code, fail_layer);
}

int Engine::verify_check(const F* tr, const F* out, const F* chal, int* fail_code, int* fail_layer) const {
    const uint32_t out_total = vf_out_total;
    // the protocol driver (canonical host arithmetic of field.cuh)
    auto ev = [](const F* q, const F& x) { return f_mul_add(f_mul_add(q[0], x, q[1]), x, q[2]); };   // a x^2 + b x + c
    auto ok_sum = [&](const F* q, const F& claim) { return f_eq(f_add(q[2], f_add(f_add(q[0], q[1]), q[2])), claim); };
#define VP_FAIL(cd, ly) do { if (fail_code) *fail_code = (cd); if (fail_layer) *fail_layer = (ly); return 0; } while (0)
    if (fail_code) *fail_code = 0;
    if (fail_layer) *fail_layer = 0;
    std::vector<std::vector<F>> claims_v(n);
    F previousSum = tr[lay.tr_vres];
    for (int i = n - 1; i >= 1; --i) {
        const LayerDev& D = L[i];
        const int pb = D.pb, m = D.m;
        const F* r_u = chal + D.ci_ru;
        for (int j = 0; j < pb; ++j) {
            const F* q = tr + D.tr_p1 + 3 * j;
            if (!ok_sum(q, previousSum)) VP_FAIL(1, i);
            previousSum = ev(q, r_u[j]);
        }
        const F claim_u = tr[D.tr_claim_u];
        claims_v[i].assign(i, f_zero());
        F bv0 = f_one();
        if (m != -1) {
            const F* r_v = chal + D.ci_rv;
            for (int j = 0; j < m; ++j) {
                const F* q = tr + D.tr_p2 + 3 * j;
                if (!ok_sum(q, previousSum)) VP_FAIL(2, i);
                previousSum = ev(q, r_v[j]);
                bv0 = f_mul(bv0, f_sub(f_one(), r_v[j]));   // beta_v[0]
            }
            claims_v[i].assign(tr + D.tr_claims_v, tr + D.tr_claims_v + i);
        }
        // getFinalValue (verifier.cpp:115-132) from the bucket sums
        F cl[4] = {f_zero(), f_zero(), f_zero(), f_zero()}, bias = f_zero(), res = f_zero();
        const F* o = out + D.vf_out;
        const F one_m_cu = f_sub(f_one(), claim_u);
        for (size_t b = 0; b < D.vf_key.size(); ++b) {
            const uint32_t key = D.vf_key[b];
            if (key < 4) {
                cl[key] = o[2 * b];
                if (key == 2) bias = o[2 * b + 1];
            }
        }
        if (m != -1) { for (auto& x : cl) x = f_mul(x, bv0); bias = f_mul(bias, bv0); }
        res = f_mul(cl[1], one_m_cu);                                 // Not
        res = f_add(res, f_mul(cl[0], claim_u));                      // Copy
        res = f_add(f_add(res, f_mul(cl[2], claim_u)), bias);         // Addc
        res = f_add(res, f_mul(cl[3], claim_u));                      // Mulc
        if (m != -1)
            for (size_t b = 0; b < D.vf_key.size(); ++b) {
                const uint32_t key = D.vf_key[b];
                if (key < 4) continue;
                const int l = (int)((key - 4) / 7), bi = (int)((key - 4) % 7);
                const F cu = claim_u, cv = claims_v[i][l], uv = f_mul(cu, cv);
                F w;
                switch (bi) {
                    case 0: w = f_add(cu, cv); break;
                    case 1: w = f_sub(cu, cv); break;
                    case 2: w = f_sub(cv, cu); break;
                    case 3: w = uv; break;
                    case 4: w = f_sub(cv, uv); break;
                    case 5: w = f_sub(cu, uv); break;
                    default: w = f_sub(f_add(cu, cv), f_dbl(uv)); break;
                }
                res = f_add(res, f_mul(o[2 * b], w));
            }
        if (!f_eq(previousSum, res)) VP_FAIL(3, i);
        // verifyLiu
        const int pre = i - 1;
        const F* sig = chal + D.ci_sig;
        const F* r_liu = chal + D.ci_rliu;
        previousSum = f_mul(sig[0], claim_u);
        // verifier.cpp:281-284 tests `~dadBitLength`, which is also true for an EMPTY subset (dadBitLength == INT_MIN there,
        // circuit.cpp:73): the claim the prover sent for it (0 if honest) counts, so a non-zero one is caught here
        for (int j = i; j < n; ++j) previousSum = f_add(previousSum, f_mul(sig[j - pre], claims_v[j][pre]));
        for (int j = 0; j < pb; ++j) {
            const F* q = tr + D.tr_liu + 3 * j;
            if (!ok_sum(q, previousSum)) VP_FAIL(4, i);
            previousSum = ev(q, r_liu[j]);
        }
        const F vr = tr[D.tr_claim_liu];
        F gr = f_zero();
        for (uint32_t sg = 0; sg < D.n_vf_liu; ++sg) gr = f_add(gr, o[2 * (D.vf_key.size() + sg)]);
        if (!f_eq(f_mul(vr, gr), previousSum)) VP_FAIL(5, i);
        previousSum = vr;
    }
    const F acc = out[out_total - 2], claimed = tr[lay.tr_input];
    if (!f_eq(claimed, acc) || !f_eq(previousSum, claimed)) VP_FAIL(6, 0);
#undef VP_FAIL
    return 1;
}

// The whole proof in verifier.cpp:134-189 order, challenges already in d_chal.
void Engine::prove_all() {
    leave();   // (a previous call may have failed inside a lane)
    direct_v = true;   // phase 1 / Liu read V from circuitValue[i-1] (sharded: the rank's rows of it)
    const bool lane = two_lanes;
    const bool lane3 = lane && three_lanes;
    const bool lane6 = lane3 && six_lanes;
    evaluate();
    if (lane) {   // fork: the other lanes need the circuit values (and the uploaded challenges)
        CK(cudaEventRecord(ev_eval, stream));
        CK(cudaStreamWaitEvent(lane1.stream, ev_eval, 0));
        if (lane3) CK(cudaStreamWaitEvent(lane2.stream, ev_eval, 0));
        if (lane6)
            for (LaneRes* R : {&lane0b, &lane1b, &lane2b}) CK(cudaStreamWaitEvent(R->stream, ev_eval, 0));
    }
    const bool extras = extras_pending;
    extras_pending = false;
    if (extras) {   // phase 2 gathers V from any lower layer, also from the extra layer-0 instances: its lanes wait at once
        if (lane3) CK(cudaStreamWaitEvent(lane2.stream, ev_extra, 0));
        if (lane6) CK(cudaStreamWaitEvent(lane2b.stream, ev_extra, 0));
        if (!lane3) CK(cudaStreamWaitEvent(stream, ev_extra, 0));
    }
    do_vres();
    // Order of the layers. All phases of a proof are independent once the challenges are known (only phase 2 of a layer
    // waits for phase 1 of the same layer), so the two lane sets need not walk the layers top-down: the layers are sorted by
    // size, dealt out alternately, and set A walks its share from the largest down while set B walks its share from the
    // smallest up -- at any time one large, throughput-bound layer is in flight next to a small, latency-bound one that
    // hides under it (top-down, the eight small top layers of SHA256 ran against each other with the GPU mostly idle).
    std::vector<std::pair<int, bool>> seq;   // (layer, on the second lane set)
    if (lane6 && layer_order_by_size) {
        std::vector<int> by_size;
        for (int i = 1; i < n; ++i) by_size.push_back(i);
        std::stable_sort(by_size.begin(), by_size.end(), [&](int a, int b) {
            return (double)C.layer_size(a - 1) * 2 + L[a].p2_out_entries > (double)C.layer_size(b - 1) * 2 + L[b].p2_out_entries;
        });
        std::vector<int> sa, sb;
        for (size_t k = 0; k < by_size.size(); ++k) (k & 1 ? sb : sa).push_back(by_size[k]);
        std::reverse(sb.begin(), sb.end());
        // Sharded: layer 1 may have to wait for the extra input instances, so it goes last in its set -- on EVERY rank and in
        // every call, whether this rank has extras or not: the ranks must walk the same sequence of phases per lane (the
        // NVLink exchange pairs the k-th exchange of a lane on one rank with the k-th on the others). Deciding this per rank
        // paired records of different phases on 4 GPUs, where only some ranks have extras (caught by bench.py's parity check).
        if (world > 1)
            for (std::vector<int>* v : {&sa, &sb}) {
                auto it = std::find(v->begin(), v->end(), 1);
                if (it != v->end()) { v->erase(it); v->push_back(1); }
            }
        for (size_t k = 0; k < std::max(sa.size(), sb.size()); ++k) {
            if (k < sa.size()) seq.push_back({sa[k], false});
            if (k < sb.size()) seq.push_back({sb[k], true});
        }
    } else
        for (int i = n - 1; i >= 1; --i) seq.push_back({i, lane6 && ((n - 1 - i) & 1)});   // every other layer on the second set of lanes
    for (const auto& lo : seq) {
        const int i = lo.first;
        LayerDev& D = L[i];
        const int m = D.m;
        const bool odd = lo.second;
        if (extras && i == 1) {   // layer 1's own tables run over layer 0: a block's worth of rows may lie outside the core range
            CK(cudaStreamWaitEvent(stream, ev_extra, 0));
            if (lane) CK(cudaStreamWaitEvent(lane1.stream, ev_extra, 0));
            if (lane6) { CK(cudaStreamWaitEvent(lane0b.stream, ev_extra, 0)); CK(cudaStreamWaitEvent(lane1b.stream, ev_extra, 0)); }
        }
        // ---- phase 1
        if (odd) enter(lane0b, 0);
        do_init_phase1(i);
        do_phase(D.ph1, D.ci_ru, D.tr_p1, lane3 ? d_vu.p + i : scal(SC_VU), nullptr, true, val[i - 1].p);
        if (lane3 && m != -1) CK(cudaEventRecord(ev_p1v[i], stream));
        if (odd) leave();
        // ---- phase 2: on its own lane, behind this layer's phase 1
        if (m != -1 && lane3) {
            enter(odd ? lane2b : lane2, 2);
            CK(cudaStreamWaitEvent(stream, ev_p1v[i], 0));
            do_init_phase2(i);
            do_phase(D.ph2, D.ci_rv, D.tr_p2, nullptr, scal(SC_UNARY));
            leave();
        } else if (m != -1) {
            do_init_phase2(i);
            do_phase(D.ph2, D.ci_rv, D.tr_p2, nullptr, scal(SC_UNARY));
        }
        // ---- Liu
        if (lane) enter(odd ? lane1b : lane1, 1);
        do_init_liu(i, false);   // the Liu add table is zero: the pass kernel runs without it (has_a)
        do_phase(D.ph3, D.ci_rliu, D.tr_liu, nullptr, nullptr, /*has_a=*/false, val[i - 1].p);
        if (lane) leave();
    }
    if (lane) {   // join: the b coefficients, the input MLE and the transcript copy follow on the main lane
        std::vector<LaneRes*> used{&lane1};
        if (lane3) used.push_back(&lane2);
        if (lane6) { used.push_back(&lane0b); used.push_back(&lane1b); used.push_back(&lane2b); }
        for (LaneRes* R : used) {
            CK(cudaEventRecord(R->ev_done, R->stream));
            CK(cudaStreamWaitEvent(stream, R->ev_done, 0));
        }
    }
    derive_b();
    do_input_mle();
    direct_v = false;
    CK(cudaGetLastError());
}

// A sumcheck phase of the Fiat-Shamir schedule, the prover's side: its init kernels, its plan, and where its final value
// goes (keep) and its round-1 scalar comes from (at_init).
const PhasePlan& Engine::fs_phase_init(int i, int phase, F*& keep, const F*& at_init) {
    cur_layer = i;
    LayerDev& D = L[i];
    keep = nullptr;
    at_init = nullptr;
    if (phase == 1) {
        do_init_phase1(i);
        keep = scal(SC_VU);
        return D.ph1;
    }
    if (phase == 2) {
        do_init_phase2(i);
        at_init = scal(SC_UNARY);
        return D.ph2;
    }
    do_init_liu(i, true);
    return D.ph3;
}

// Fiat-Shamir mode (SURVEY 8(f) N4): the whole proof through the one-round-per-launch path, every challenge drawn from
// the transcript cache right after the message it has to depend on (fs_schedule). The two-rounds-per-pass kernel cannot
// be used here: it needs the challenges of a phase before the phase starts.
void Engine::prove_fs(const uint8_t seed[32], F* tr_out, F* ch_out) {
    leave();
    FsCache fs;
    fs.store(seed, 32);
    std::vector<F> ch(lay.n_chal, f_zero());
    auto step = [&](const FsStep& st) {   // the messages from the device into the cache, the challenges back to the device
        if (st.n_store) get_tr(st.tr_begin, reinterpret_cast<vp_F*>(tr_out + st.tr_begin), st.n_store);
        for (uint32_t k = 0; k < st.n_store; ++k) fs.store(tr_out[st.tr_begin + k]);
        for (uint32_t k = 0; k < st.n_draw; ++k) {
            const uint32_t idx = st.ci_begin + k;
            ch[idx] = fs.random();
            const vp_F v{ch[idx].re, ch[idx].im};
            set_chal(idx, &v);
        }
    };
    {   // unused challenge slots are zero on the device as well
        CK(cudaMemsetAsync(d_chal.p, 0, (lay.n_chal + 1) * sizeof(F), stream));
        h_chal.assign(lay.n_chal, f_zero());
    }
    evaluate();
    check_assert_flag();
    for (const FsEntry& e : fs_sched) {
        if (!e.phase) {
            if (e.first.n_store && e.first.tr_begin == lay.tr_vres) do_vres();   // at r_out, drawn by the steps before
            step(e.first);
            continue;
        }
        F* keep;
        const F* at_init;
        const PhasePlan& PP = fs_phase_init(e.layer, e.phase, keep, at_init);
        for (uint32_t k = 0; k < e.count; ++k) {
            const FsStep st = e.step(k);
            const int j = (int)k + 1;
            if (PP.sharded) sharded_round(PP, e.phase, j, e.first.ci_begin, st.tr_begin, at_init);
            else do_round(PP.planB, j, e.first.ci_begin + (uint32_t)std::max(0, j - 2), st.tr_begin, at_init);
            step(st);
        }
        do_finalize(PP.planB, e.first.ci_begin + (uint32_t)std::max(0, (int)e.count - 1), keep);
    }
    do_input_mle();
    get_tr(0, reinterpret_cast<vp_F*>(tr_out), lay.n_tr);   // with what no step stores: the last claim_liu, the input MLE
    if (ch_out) memcpy(ch_out, ch.data(), lay.n_chal * sizeof(F));
    proof_size = lay.proof_size;
}

// ---- Fiat-Shamir mode on the device (fs_device.cuh): the order of prove_fs, with the transcript cache in a device pool;
// the host only enqueues. One synchronisation for the assert flag after evaluate, one at the end for the copies.
void Engine::fs_alloc() {
    if (d_fs_pool.p) return;
    d_fs_pool.alloc(1 + 4 + 2 * ((size_t)n + 4));   // the longest run of stores between two draws: claim_u + claims_v
    d_fs_stamps.alloc(4 * std::max<size_t>(lay.rounds, 1));
    d_stmt.alloc(16);
    d_circuit_digest = d_stmt.p;
}
void Engine::fs_begin() {
    leave();
    fs_alloc();
    memset_stmts(d_chal.p, (lay.n_chal + 1) * sizeof(F));   // unused challenge slots are zero
    if (n_stmt == 1) h_chal.assign(lay.n_chal, f_zero());
    evaluate();
    if (dev_io) {   // every statement's assert flag becomes its status on the device
        k_batch_assert_status<<<cdiv(n_stmt, 128), 128, 0, stream>>>(d_counter.p + 1, sstride, n_stmt, slab.status.p);
        ++launches;
        return;
    }
    if (n_stmt == 1) {
        check_assert_flag();
        return;
    }
    // the first statement with a failed assert gate
    std::vector<unsigned int> flags(n_stmt);
    copy_stmts_out(flags.data(), sizeof(unsigned int), d_counter.p + 1, sizeof(unsigned int));
    CK(cudaStreamSynchronize(stream));
    for (uint32_t b = 0; b < n_stmt; ++b)
        if (flags[b]) throw StatementAssert{b, flags[b]};
}

// Batch slab: per statement a copy of every buffer of fs_buffers, in its order, then the verifier's region, each 256-byte
// aligned.
void Engine::slab_reserve(uint32_t B, size_t vf_entries) {
    if (slab.cap >= B && slab.vf_entries >= vf_entries) return;
    vf_entries = std::max(vf_entries, slab.vf_entries);
    B = std::max(B, slab.cap);
    batch_outputs = 0;   // (the values are reallocated)
    size_t off = 0, o_eq = 0;
    auto put = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    std::vector<std::pair<size_t, size_t>> at;   // (offset, entries) of each buffer
    fs_buffers([&](auto& d, size_t entries) {
        at.push_back({put(entries * sizeof *d.p), entries});
        if ((const void*)&d == (const void*)&d_eq) o_eq = at.back().first;
    });
    slab.o_vf = put(vf_entries * sizeof(F));
    slab.vf_entries = vf_entries;
    slab.cap = 0;
    slab.stride = off;
    slab.mem.alloc((size_t)B * off);
    CK(cudaMemsetAsync(slab.mem.p, 0, (size_t)B * off, stream));   // the grid-sum tickets start at zero
    slab.val.resize(n);
    std::vector<F*> h_ptr(n);
    for (int i = 0; i < n; ++i) {
        slab.val[i].alloc((size_t)B * C.layer_size(i));
        h_ptr[i] = slab.val[i].p;
    }
    slab.valptr.upload(h_ptr, stream);
    slab.inputs.alloc((size_t)B * C.layer_size(0));
    slab.contexts.alloc((size_t)4 * B);
    slab.status.alloc(B);
    // descriptors that point into the context's values / eq tables, rebased on the slab's
    slab.p2_tabs.resize(n);
    slab.liu_eqtabs.resize(n);
    const uintptr_t eq0 = reinterpret_cast<uintptr_t>(d_eq.p), eq1 = reinterpret_cast<uintptr_t>(slab.mem.p + o_eq);
    for (int i = 1; i < n; ++i) {
        std::vector<P2Table> t = L[i].h_p2;
        for (P2Table& x : t)
            for (int l = 0; l < n; ++l)
                if (x.src_val == val[l].p) { x.src_val = slab.val[l].p; break; }
        slab.p2_tabs[i].upload(t, stream);
        std::vector<EqTab> e(L[i].liu_eqtabs.n);
        if (!e.empty()) CK(cudaMemcpy(e.data(), L[i].liu_eqtabs.p, e.size() * sizeof(EqTab), cudaMemcpyDeviceToHost));
        for (EqTab& x : e) {
            x.f = reinterpret_cast<const F*>(reinterpret_cast<uintptr_t>(x.f) - eq0 + eq1);
            x.s = reinterpret_cast<const F*>(reinterpret_cast<uintptr_t>(x.s) - eq0 + eq1);
        }
        slab.liu_eqtabs[i].upload(e, stream);
    }
    slab.views.clear();   // statement 0's
    for (const auto& [o, entries] : at) slab.views.push_back({slab.mem.p + o, entries});
    CK(cudaStreamSynchronize(stream));   // (the host vectors go out of scope)
    slab.cap = B;
}

// Exchanges the buffers of the Fiat-Shamir path with the slab's: statement 0 of the slab takes the context's place. Called
// twice, it restores the context (FsBatchScope).
void Engine::slab_swap() {
    size_t k = 0;
    fs_buffers([&](auto& d, size_t) {
        using T = std::remove_reference_t<decltype(*d.p)>;
        std::pair<void*, size_t>& v = slab.views[k++];
        T* const p = d.p;
        const size_t c = d.n;
        d.p = static_cast<T*>(v.first);
        d.n = v.second;
        v = {p, c};
    });
    std::swap(val, slab.val);
    std::swap(d_valptr, slab.valptr);
    std::swap(d_inputs, slab.inputs);
    std::swap(d_root_scratch, slab.root_scratch);
    for (int i = 1; i < n; ++i) {
        std::swap(L[i].p2_tabs, slab.p2_tabs[i]);
        std::swap(L[i].liu_eqtabs, slab.liu_eqtabs[i]);
    }
}

// one cooperative launch of k_sumcheck_phase_fs over P (unsharded: the whole phase)
void Engine::launch_phase_kernel_fs(const SumcheckPlan& P, uint32_t ci, F* keep, const F* at_init, uint32_t tr_rounds, size_t stamp_round) {
    PhaseArgs a;
    for (int b = 0; b < 2; ++b) { a.bufV[b] = bufV[b].p; a.bufM[b] = bufM[b].p; a.bufA[b] = bufA[b].p; }
    a.rounds = d_rdev.p + P.rdev_begin;
    a.tabs = d_tabs.p;
    a.cols = d_cols.p;
    a.fins = d_fins.p + P.fin_begin;
    a.n_rounds = (uint32_t)P.rounds;
    a.n_fin = P.n_fin;
    a.fin_buf = (uint32_t)P.fin_buf;
    a.tail_work = tail_work;
    a.at_init = at_init;
    a.add_term = scal(SC_ADD_TERM);
    a.claims = d_claims.p;
    a.out_poly = d_tr.p + tr_rounds;
    a.transcript = d_tr.p;
    a.keep = keep;
    a.partials = d_partials.p;
    FsPhaseArgs f;
    f.pool = d_fs_pool.p;
    f.chal = d_chal.p + ci;
    f.stamps = d_fs_stamps.p + 4 * stamp_round;
    f.ss = sstride;
    // a row of gx blocks per statement; the cooperative grid holds at most cap_phase_fs blocks, so a batch larger than
    // that runs in chunks of statements (row z of a chunk starting at statement s0 is statement s0 + z)
    const uint32_t rows = std::min<uint32_t>(n_stmt, (uint32_t)cap_phase_fs);
    const int gx = P.max_work > tail_work ? grid_for(P.max_work, std::max(1, cap_phase_fs / (int)rows)) : 1;
    for (uint32_t s0 = 0; s0 < n_stmt; s0 += rows) {
        const uint32_t nz = std::min(rows, n_stmt - s0);
        PhaseArgs ac = a;
        FsPhaseArgs fc = f;
        if (s0) {
            const size_t d = s0 * sstride;
            auto sh = [d](auto* q) { return q ? reinterpret_cast<decltype(q)>(reinterpret_cast<uintptr_t>(q) + d) : q; };
            for (int b = 0; b < 2; ++b) { ac.bufV[b] = sh(a.bufV[b]); ac.bufM[b] = sh(a.bufM[b]); ac.bufA[b] = sh(a.bufA[b]); }
            ac.at_init = sh(a.at_init); ac.add_term = sh(a.add_term); ac.claims = sh(a.claims);
            ac.out_poly = sh(a.out_poly); ac.transcript = sh(a.transcript); ac.keep = sh(a.keep); ac.partials = sh(a.partials);
            fc.pool = sh(f.pool); fc.chal = sh(f.chal); fc.stamps = nullptr;
        }
        void* args[] = {&ac, &fc};
        size_t h = prof_begin(KC_ROUND_FOLD);
        CK(cudaLaunchCooperativeKernel((const void*)k_sumcheck_phase_fs, dim3(gx, 1, nz), dim3(256), args, 0, stream));
        prof_end(h, P.bytes * nz);
        ++launches;
    }
}

// The circuit digest R(circuit_bytes) (include/virgo_b200.h), serialised on the host once per context and hashed on the device.
void Engine::circuit_digest_async() {
    if (circuit_digest_ready) return;
    circuit_digest_async(C.instances, const_cast<uint64_t*>(d_circuit_digest));
    circuit_digest_ready = true;
}
// ... of template + K, kept for the last K
const uint64_t* Engine::circuit_digest_k_async(uint64_t K) {
    if (digest_k != K) {
        if (!d_digest_k.p) d_digest_k.alloc(4);
        digest_k = 0;
        circuit_digest_async(K, d_digest_k.p);
        digest_k = K;
    }
    return d_digest_k.p;
}
// R(circuit_bytes) with `instances` as the serialised instance count, to out (4 words, device)
void Engine::circuit_digest_async(uint64_t instances, uint64_t* out) {
    std::vector<uint8_t> b;
    auto put = [&](const void* q, size_t len) { const uint8_t* c = static_cast<const uint8_t*>(q); b.insert(b.end(), c, c + len); };
    auto u64 = [&](uint64_t x) { put(&x, 8); };
    size_t total = 8 + 16 + 8 * (size_t)n;
    for (int i = 1; i < n; ++i) {
        total += 34 * C.layers[i].size;
        for (int s = 0; s < i; ++s) total += 8 + 4 * C.layers[i].dadId[s].size();
    }
    b.reserve(total + 64);
    put("VPCIRC01", 8);
    u64((uint64_t)n);
    u64(instances);
    for (int i = 0; i < n; ++i) u64(C.layers[i].size);
    for (int i = 1; i < n; ++i) {
        const Layer& T = C.layers[i];
        for (uint64_t g = 0; g < T.size; ++g) {
            const uint8_t ty = T.ty[g], as = T.is_assert.empty() ? 0 : T.is_assert[g];
            const int32_t l = T.l[g];
            const uint32_t u = T.u[g], v = T.v[g], lv = T.lv[g];
            const F c = T.c.empty() ? f_zero() : T.c[g];
            put(&ty, 1); put(&as, 1); put(&l, 4); put(&u, 4); put(&v, 4); put(&lv, 4); put(&c.re, 8); put(&c.im, 8);
        }
    }
    for (int i = 1; i < n; ++i)
        for (int s = 0; s < i; ++s) {
            u64(C.layers[i].dadSize[s]);
            put(C.layers[i].dadId[s].data(), 4 * C.layers[i].dadId[s].size());
        }
    b.resize((b.size() + 63) / 64 * 64, 0);   // whole leaves (R pads with zeros anyway)
    DBuf<uint64_t> words, scratch;
    words.alloc(b.size() / 8);
    CK(cudaMemcpyAsync(words.p, b.data(), b.size(), cudaMemcpyHostToDevice, stream));
    scratch.alloc(pc_vector_root_scratch(words.n) / 8);
    launches += (uint64_t)pc_vector_root(words.p, words.n, scratch.p, reinterpret_cast<uint8_t*>(out), stream);
    CK(cudaStreamSynchronize(stream));   // (the host bytes and the scratch go out of scope)
}

// The B statements of an aggregate proof and the aggregate (include/virgo_b200.h), which seeds the pool. Statement b covers
// instances [b K, (b + 1) K) of circuitValue[0] and of the outputs (d_outputs, or circuitValue[n-1]); the values are
// instance-major, so its slices lie end to end and each kind of root is one pass of pc_vector_root over B vectors.
// contexts: B * 32 bytes on the host.
void Engine::aggregate_async(uint32_t B, const uint8_t* contexts, const F* d_outputs) {
    const uint64_t K = C.instances / B;
    const uint64_t* circuit = circuit_digest_k_async(K);
    const size_t n_in = K * C.layers[0].size, n_out = K * C.layers[n - 1].size;
    const size_t need = std::max({B * pc_vector_root_scratch(2 * n_in), B * pc_vector_root_scratch(2 * n_out),
                                  pc_vector_root_scratch(4 * (size_t)B)}) / 8;
    if (d_root_scratch.n < need) d_root_scratch.alloc(need);
    if (d_agg.n < 16 * (size_t)B + 8) d_agg.alloc(16 * (size_t)B + 8);
    uint64_t* const in_roots = d_agg.p;
    uint64_t* const out_roots = in_roots + 4 * (size_t)B;
    uint64_t* const ctxs = out_roots + 4 * (size_t)B;
    uint64_t* const stmts = ctxs + 4 * (size_t)B;
    uint64_t* const root = stmts + 4 * (size_t)B;
    CK(cudaMemcpyAsync(ctxs, contexts, 32 * (size_t)B, cudaMemcpyHostToDevice, stream));
    launches += (uint64_t)pc_vector_root(reinterpret_cast<const uint64_t*>(val[0].p), 2 * n_in, d_root_scratch.p,
                                         reinterpret_cast<uint8_t*>(in_roots), stream, B, 32);
    launches += (uint64_t)pc_vector_root(reinterpret_cast<const uint64_t*>(d_outputs ? d_outputs : val[n - 1].p), 2 * n_out,
                                         d_root_scratch.p, reinterpret_cast<uint8_t*>(out_roots), stream, B, 32);
    k_fs_statements<<<cdiv(B, 128), 128, 0, stream>>>(circuit, in_roots, out_roots, ctxs, (uint64_t)n_in, (uint64_t)n_out, B, stmts);
    ++launches;
    launches += (uint64_t)pc_vector_root(stmts, 4 * (size_t)B, d_root_scratch.p, reinterpret_cast<uint8_t*>(root), stream);
    k_fs_aggregate<<<1, 32, 0, stream>>>(root, (uint64_t)B, d_fs_pool.p, root + 4);
    ++launches;
}

// inputs root (circuitValue[0]), outputs root (d_outputs, or circuitValue[n-1]) and the statement, which seeds the pool.
// A batch: the roots of every statement's slice in one pass each, the contexts from d_contexts (4 words per statement).
void Engine::statement_async(const uint8_t context[32], const F* d_outputs, const uint64_t* d_contexts) {
    circuit_digest_async();
    const size_t n_in = C.layer_size(0), n_out = C.layer_size(n - 1);
    const size_t need = n_stmt * std::max(pc_vector_root_scratch(2 * n_in), pc_vector_root_scratch(2 * n_out)) / 8;
    if (d_root_scratch.n < need) d_root_scratch.alloc(need);
    launches += (uint64_t)pc_vector_root(reinterpret_cast<const uint64_t*>(val[0].p), 2 * n_in, d_root_scratch.p,
                                         reinterpret_cast<uint8_t*>(stmt_inputs()), stream, n_stmt, sstride);
    launches += (uint64_t)pc_vector_root(reinterpret_cast<const uint64_t*>(d_outputs ? d_outputs : val[n - 1].p), 2 * n_out, d_root_scratch.p,
                                         reinterpret_cast<uint8_t*>(stmt_outputs()), stream, n_stmt, sstride);
    FsContext cx;
    memset(cx.w, 0, 32);
    if (context) memcpy(cx.w, context, 32);
    k_fs_statement<<<sgrid(1), 32, 0, stream>>>(d_circuit_digest, d_stmt.p, (uint64_t)n_in, (uint64_t)n_out, cx, d_contexts, d_fs_pool.p,
                                                stmt_statement(), sstride);
    ++launches;
}

// the pool starts with a 32-byte seed from the host
void Engine::seed_pool(const uint8_t seed[32]) {
    uint64_t h[5] = {4, 0, 0, 0, 0};
    memcpy(h + 1, seed, 32);
    CK(cudaMemcpyAsync(d_fs_pool.p, h, sizeof h, cudaMemcpyHostToDevice, stream));
}

// The proof in the order of fs_schedule, on a pool seeded by seed_pool, statement_async or aggregate_async. The
// transcript and the challenges come back in one copy each.
void Engine::prove_fs_device(F* tr_out, F* ch_out) {
    size_t sr = 0;   // stamp slot of the next phase's first round
    for (const FsEntry& e : fs_sched) {
        if (!e.phase) {
            if (e.first.n_store && e.first.tr_begin == lay.tr_vres) do_vres();   // at r_out, drawn by the steps before
            fs_absorb_draw(e.first.tr_begin, e.first.n_store, e.first.ci_begin, e.first.n_draw);
            continue;
        }
        F* keep;
        const F* at_init;
        const PhasePlan& PP = fs_phase_init(e.layer, e.phase, keep, at_init);
        launch_phase_kernel_fs(PP.planB, e.first.ci_begin, keep, at_init, e.first.tr_begin, sr);   // stores and draws e.count rounds
        sr += e.count;
    }
    do_input_mle();
    fs_rounds = sr;
    proof_size = lay.proof_size;
    if (dev_io) {   // into the caller's device arrays; nothing waits for them
        copy_stmts_out(tr_out, lay.n_tr * sizeof(F), d_tr.p, lay.n_tr * sizeof(F));
        if (ch_out) copy_stmts_out(ch_out, lay.n_chal * sizeof(F), d_chal.p, lay.n_chal * sizeof(F));
        CK(cudaGetLastError());
        return;
    }
    std::vector<F> ch((size_t)n_stmt * lay.n_chal);   // statement-major, like the transcripts
    copy_stmts_out(tr_out, lay.n_tr * sizeof(F), d_tr.p, lay.n_tr * sizeof(F));
    copy_stmts_out(ch.data(), lay.n_chal * sizeof(F), d_chal.p, lay.n_chal * sizeof(F));
    CK(cudaStreamSynchronize(stream));
    CK(cudaGetLastError());
    if (n_stmt == 1) h_chal = ch;   // a later vp_verify / vp_prove on this context sees the challenges the proof used
    if (ch_out) memcpy(ch_out, ch.data(), ch.size() * sizeof(F));
}

// fs_schedule as k_fs_replay's steps, one per round of a phase, built once per context.
void Engine::fs_replay_table() {
    if (d_fs_steps.p) return;
    std::vector<FsStep> st;
    for (const FsEntry& e : fs_sched)
        for (uint32_t k = 0; k < e.count; ++k) st.push_back(e.step(k));
    d_fs_steps.upload(st, stream);
    CK(cudaStreamSynchronize(stream));   // (the host vector goes out of scope)
}

// verify_check's view of the proof layout and of the bucket keys for k_verify_check, built once per context (after
// vf_layout, which places every layer's sums).
VfCheckArgs Engine::vf_check_table() {
    if (!d_vf_desc.p) {
        std::vector<VfLayerDesc> t(n);
        std::vector<uint32_t> keys;
        for (int i = 1; i < n; ++i) {
            const LayerDev& D = L[i];
            t[i] = VfLayerDesc{D.pb, D.m, D.tr_p1, D.tr_claim_u, D.tr_p2, D.tr_claims_v, D.tr_liu, D.tr_claim_liu, D.ci_ru, D.ci_rv,
                               D.ci_sig, D.ci_rliu, D.vf_out, (uint32_t)keys.size(), (uint32_t)D.vf_key.size(), D.n_vf_liu};
            keys.insert(keys.end(), D.vf_key.begin(), D.vf_key.end());
        }
        d_vf_desc.upload(t, stream);
        d_vf_keys.upload(keys, stream);
        CK(cudaStreamSynchronize(stream));   // (the host vectors go out of scope)
    }
    return VfCheckArgs{d_vf_desc.p, d_vf_keys.p, n, lay.tr_vres, lay.tr_input, vf_out_total};
}

// A batch's inputs (cnt, statement-major) into d_inputs: from the host (checked before the call), or from the caller's
// device array through k_batch_screen (status 1 and zeros for a statement with an input >= p).
void Engine::load_batch_inputs(const uint64_t* src, size_t cnt) {
    if (!dev_io) {
        CK(cudaMemcpyAsync(d_inputs.p, src, cnt * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
        return;
    }
    k_batch_screen<<<sgrid(1), 256, 0, stream>>>(src, d_inputs.p, (uint32_t)(cnt / n_stmt), nullptr, nullptr, 0, nullptr, 0, sstride, 1,
                                                 slab.status.p);
    ++launches;
}

struct vp_ctx {
    Engine e;
};

// ------------------------------------------------------------------ C ABI: misc
extern "C" const char* vp_last_error(void) { return g_err.c_str(); }
extern "C" const char* vp_version(void) { return "virgo-plus_b200 0.1 (sm_100a)"; }

#define API_BEGIN try {
#define API_END                                                          \
    }                                                                    \
    catch (const CudaError& e) { return fail(VP_ERR_CUDA, "%s", e.msg.c_str()); } \
    catch (const std::bad_alloc&) { return fail(VP_ERR_NOMEM, "out of host memory"); } \
    catch (unsigned int flag) { return fail(VP_ERR_ASSERT, "assert gate violated in layer %u", flag - 1); } \
    catch (const StatementAssert& a) { return fail(VP_ERR_ASSERT, "statement %u: assert gate violated in layer %u", a.stmt, a.flag - 1); } \
    catch (const std::invalid_argument& e) { return fail(VP_ERR_ARG, "%s", e.what()); } \
    catch (const std::length_error& e) { return fail(VP_ERR_CIRCUIT, "%s", e.what()); } \
    catch (const std::runtime_error& e) { return fail(VP_ERR_CUDA, "%s", e.what()); } \
    catch (const std::exception& e) { return fail(VP_ERR_ARG, "%s", e.what()); }

// ------------------------------------------------------------------ C ABI: circuit
static int wrap_circuit(Circuit&& c, vp_circuit** out) {
    std::string err = c.validate();
    if (!err.empty()) return fail(VP_ERR_CIRCUIT, "%s", err.c_str());
    *out = new vp_circuit{std::move(c)};
    return VP_OK;
}
extern "C" int vp_circuit_load_pws(const char* path, vp_circuit** out) {
    if (!path || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Circuit c;
    std::string err = load_pws(path, c);
    if (!err.empty()) return fail(VP_ERR_CIRCUIT, "%s", err.c_str());
    return wrap_circuit(std::move(c), out);
    API_END
}
extern "C" int vp_circuit_load_pws_text(const char* text, size_t len, vp_circuit** out) {
    if (!text || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Circuit c;
    std::string err = load_pws_text(text, len, c);
    if (!err.empty()) return fail(VP_ERR_CIRCUIT, "%s", err.c_str());
    return wrap_circuit(std::move(c), out);
    API_END
}
extern "C" int vp_circuit_random(int n_layers, int log_size, uint64_t seed, vp_circuit** out) {
    if (!out || n_layers < 2 || n_layers > 120 || log_size < 0 || log_size > 30) return fail(VP_ERR_ARG, "bad argument");
    API_BEGIN
    return wrap_circuit(random_circuit(n_layers, log_size, seed), out);
    API_END
}
extern "C" int vp_circuit_from_arrays(int n_layers, const uint64_t* layer_size, const uint8_t* ty, const int32_t* l,
                                      const uint64_t* u, const uint64_t* v, const uint64_t* lv, const vp_F* cst,
                                      const uint8_t* is_assert, const uint64_t* dad_size, const uint64_t* dad_id,
                                      vp_circuit** out) {
    if (n_layers < 1 || !layer_size || !ty || !l || !u || !v || !out) return fail(VP_ERR_ARG, "null argument");
    if (dad_size && (!lv || !dad_id)) return fail(VP_ERR_ARG, "dad_size given without lv / dad_id");
    API_BEGIN
    Circuit c;
    c.layers.resize(n_layers);
    size_t off = 0, doff = 0;
    for (int i = 0; i < n_layers; ++i) {
        Layer& L = c.layers[i];
        L.size = layer_size[i];
        if (L.size == 0 || L.size > (1ULL << 31)) return fail(VP_ERR_CIRCUIT, "layer %d: size %llu out of range", i, (unsigned long long)L.size);
        L.ty.resize(L.size);
        L.l.resize(L.size);
        L.u.resize(L.size);
        L.v.resize(L.size);
        L.lv.assign(L.size, 0);
        bool any_c = false, any_a = false;
        for (uint64_t g = 0; g < L.size; ++g) {
            L.ty[g] = ty[off + g];
            L.l[g] = l[off + g];
            if (i == 0) {
                c.inputs.push_back(u[off + g]);
                L.u[g] = 0;
                L.l[g] = -1;
            } else {
                if (u[off + g] > 0xffffffffULL || v[off + g] > 0xffffffffULL)
                    return fail(VP_ERR_CIRCUIT, "layer %d gate %llu: index exceeds 32 bits", i, (unsigned long long)g);
                L.u[g] = (uint32_t)u[off + g];
            }
            L.v[g] = (uint32_t)v[off + g];
            if (lv) {
                if (lv[off + g] > 0xffffffffULL) return fail(VP_ERR_CIRCUIT, "layer %d gate %llu: lv exceeds 32 bits", i, (unsigned long long)g);
                L.lv[g] = (uint32_t)lv[off + g];
            }
            if (cst && (cst[off + g].re | cst[off + g].im)) any_c = true;
            if (is_assert && is_assert[off + g]) any_a = true;
        }
        if (any_c) {
            L.c.resize(L.size);
            for (uint64_t g = 0; g < L.size; ++g) L.c[g] = F{cst[off + g].re, cst[off + g].im};
        }
        if (any_a) L.is_assert.assign(is_assert + off, is_assert + off + L.size);
        if (dad_size) {
            L.dadSize.resize(i);
            L.dadId.resize(i);
            for (int s = 0; s < i; ++s) {
                L.dadSize[s] = dad_size[(size_t)i * n_layers + s];
                if (L.dadSize[s] > c.layers[s].size) return fail(VP_ERR_CIRCUIT, "layer %d: dad subset of layer %d is larger than that layer", i, s);
                L.dadId[s].resize(L.dadSize[s]);
                for (uint64_t x = 0; x < L.dadSize[s]; ++x) {
                    if (dad_id[doff + x] > 0xffffffffULL) return fail(VP_ERR_CIRCUIT, "layer %d: dad_id exceeds 32 bits", i);
                    L.dadId[s][x] = (uint32_t)dad_id[doff + x];
                }
                doff += L.dadSize[s];
            }
        }
        off += L.size;
    }
    if (!dad_size) c.subset_init();
    return wrap_circuit(std::move(c), out);
    API_END
}
extern "C" int vp_circuit_replicate(const vp_circuit* c, uint64_t instances, vp_circuit** out) {
    if (!c || !out || instances == 0) return fail(VP_ERR_ARG, "bad argument");
    if (c->c.instances != 1) return fail(VP_ERR_ARG, "circuit is already replicated");
    API_BEGIN
    return wrap_circuit(c->c.replicate(instances), out);
    API_END
}
extern "C" int vp_circuit_expand(const vp_circuit* c, vp_circuit** out) {
    if (!c || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    return wrap_circuit(c->c.expand(), out);
    API_END
}
extern "C" void vp_circuit_free(vp_circuit* c) { delete c; }
extern "C" int vp_circuit_num_layers(const vp_circuit* c) { return c ? c->c.n_layers() : 0; }
extern "C" uint64_t vp_circuit_instances(const vp_circuit* c) { return c ? c->c.instances : 0; }
extern "C" uint64_t vp_circuit_layer_size(const vp_circuit* c, int layer) {
    return (c && layer >= 0 && layer < c->c.n_layers()) ? c->c.layers[layer].size : 0;
}
extern "C" int vp_circuit_bit_length(const vp_circuit* c, int layer) {
    return (c && layer >= 0 && layer < c->c.n_layers()) ? c->c.bit_length(layer) : -1;
}
extern "C" uint64_t vp_circuit_dad_size(const vp_circuit* c, int layer, int src) {
    return (c && layer >= 0 && layer < c->c.n_layers() && src >= 0 && src < layer) ? c->c.layers[layer].dadSize[src] : 0;
}
extern "C" int vp_circuit_max_dad_bit_length(const vp_circuit* c, int layer) {
    return (c && layer >= 1 && layer < c->c.n_layers()) ? c->c.max_dad_bit_length(layer) : -1;
}
extern "C" uint64_t vp_circuit_total_gates(const vp_circuit* c) { return c ? c->c.total_gates() : 0; }
extern "C" uint64_t vp_circuit_num_inputs(const vp_circuit* c) { return c ? c->c.layer_size(0) : 0; }
extern "C" int vp_circuit_export_layer(const vp_circuit* c, int layer, uint8_t* ty, int32_t* l, uint32_t* u, uint32_t* v,
                                       uint32_t* lv, vp_F* cst, uint8_t* is_assert) {
    if (!c || layer < 0 || layer >= c->c.n_layers()) return fail(VP_ERR_ARG, "bad layer");
    const Layer& L = c->c.layers[layer];
    for (uint64_t g = 0; g < L.size; ++g) {
        if (ty) ty[g] = L.ty[g];
        if (l) l[g] = L.l[g];
        if (u) u[g] = L.u[g];
        if (v) v[g] = L.v[g];
        if (lv) lv[g] = L.lv[g];
        if (cst) cst[g] = L.c.empty() ? vp_F{0, 0} : vp_F{L.c[g].re, L.c[g].im};
        if (is_assert) is_assert[g] = L.is_assert.empty() ? 0 : L.is_assert[g];
    }
    return VP_OK;
}
extern "C" int vp_circuit_export_dad(const vp_circuit* c, int layer, int src, uint32_t* dad_id) {
    if (!c || layer < 1 || layer >= c->c.n_layers() || src < 0 || src >= layer || !dad_id) return fail(VP_ERR_ARG, "bad argument");
    const auto& ids = c->c.layers[layer].dadId[src];
    std::copy(ids.begin(), ids.end(), dad_id);
    return VP_OK;
}
extern "C" int vp_circuit_get_inputs(const vp_circuit* c, uint64_t* out) {
    if (!c || !out) return fail(VP_ERR_ARG, "null argument");
    std::copy(c->c.inputs.begin(), c->c.inputs.end(), out);
    return VP_OK;
}
extern "C" int vp_circuit_set_inputs(vp_circuit* c, const uint64_t* in) {
    if (!c || !in) return fail(VP_ERR_ARG, "null argument");
    for (size_t i = 0; i < c->c.inputs.size(); ++i) {
        if (in[i] >= P) return fail(VP_ERR_ARG, "input %zu is not < p", i);
        c->c.inputs[i] = in[i];
    }
    return VP_OK;
}
extern "C" size_t vp_challenge_count(const vp_circuit* c) { return c ? proof_layout(c->c).n_chal : 0; }
extern "C" int vp_draw_challenges(const vp_circuit* c, unsigned seed, vp_F* out) {
    if (!c || !out) return fail(VP_ERR_ARG, "null argument");
    ChallengeStream cs = draw_challenges(c->c, seed);
    size_t k = 0;
    auto put = [&](const std::vector<F>& v) { for (const F& x : v) out[k++] = vp_F{x.re, x.im}; };
    put(cs.r_out);
    for (int i = c->c.n_layers() - 1; i >= 1; --i) {
        const LayerChallenges& lc = cs.layer[i];
        put(lc.r_u);
        out[k++] = vp_F{lc.assert_random.re, lc.assert_random.im};
        put(lc.r_v);
        put(lc.sig);
        put(lc.r_liu);
    }
    return VP_OK;
}
// n values of fieldElement::random() (fieldElement.cpp:119-124, 362-367) after srand(seed), as a plain stream
extern "C" int vp_draw_field(unsigned seed, size_t n, vp_F* out) {
    if (!out && n) return fail(VP_ERR_ARG, "null argument");
    GlibcRandom rng(seed);
    for (size_t i = 0; i < n; ++i) {
        const F x = rng.field();
        out[i] = vp_F{x.re, x.im};
    }
    return VP_OK;
}
extern "C" size_t vp_transcript_len(const vp_circuit* c) { return c ? proof_layout(c->c).n_tr : 0; }

// ------------------------------------------------------------------ C ABI: transcript containers
extern "C" int vp_transcript_to_gkrproof(const vp_circuit* c, const vp_F* transcript, unsigned char* out, size_t cap, size_t* len) {
    if (!c || !transcript || !len) return fail(VP_ERR_ARG, "null argument");
    std::vector<unsigned char> b = transcript_to_gkrproof(c->c, reinterpret_cast<const F*>(transcript));
    *len = b.size();
    if (!out) return VP_OK;   // size query
    if (cap < b.size()) return fail(VP_ERR_ARG, "output buffer too small (%zu < %zu)", cap, b.size());
    memcpy(out, b.data(), b.size());
    return VP_OK;
}
extern "C" int vp_gkrproof_to_transcript(const vp_circuit* c, const unsigned char* bytes, size_t len, vp_F* transcript) {
    if (!c || !bytes || !transcript) return fail(VP_ERR_ARG, "null argument");
    std::string err = gkrproof_to_transcript(c->c, bytes, len, reinterpret_cast<F*>(transcript));
    if (!err.empty()) return fail(VP_ERR_ARG, "%s", err.c_str());
    return VP_OK;
}
extern "C" int vp_transcript_text(const vp_circuit* c, const vp_F* transcript, const vp_F* challenges, char* out, size_t cap,
                                  size_t* len) {
    if (!c || !transcript || !challenges || !len) return fail(VP_ERR_ARG, "null argument");
    std::string t = transcript_text(c->c, reinterpret_cast<const F*>(transcript), reinterpret_cast<const F*>(challenges));
    *len = t.size();
    if (!out) return VP_OK;
    if (cap < t.size()) return fail(VP_ERR_ARG, "output buffer too small");
    memcpy(out, t.data(), t.size());
    return VP_OK;
}

// ------------------------------------------------------------------ C ABI: prover
extern "C" int vp_create(const vp_circuit* c, int device, vp_ctx** out) {
    if (!c || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    std::unique_ptr<vp_ctx> ctx(new vp_ctx());
    ctx->e.build(c->c, device, 1, 0, nullptr);
    *out = ctx.release();
    return VP_OK;
    API_END
}
extern "C" int vp_nccl_unique_id(uint8_t out[128]) {
    if (!out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    nccl_load();
    NcclId id;
    memset(&id, 0, sizeof id);
    NCK(g_nccl.GetUniqueId(&id));
    memcpy(out, id.internal, 128);
    return VP_OK;
    API_END
}
extern "C" int vp_create_sharded(const vp_circuit* c, int device, int rank, int world, const uint8_t nccl_id[128],
                                 vp_ctx** out) {
    if (!c || !out || (world > 1 && !nccl_id)) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    std::unique_ptr<vp_ctx> ctx(new vp_ctx());
    ctx->e.build(c->c, device, world, rank, nccl_id);
    *out = ctx.release();
    return VP_OK;
    API_END
}
// Host-only view of how one phase is dealt out to the ranks (tests of the partition logic).
// out: per table 10 values {bits, live, sharded, m, row_lo, row_hi, local_len, present, n_blocks, reversed}.
extern "C" int vp_shard_describe(const vp_circuit* c, int world, int rank, int layer, int phase, uint32_t* out, size_t cap,
                                 size_t* n_tables) {
    if (!c || !out || !n_tables) return fail(VP_ERR_ARG, "null argument");
    const Circuit& C = c->c;
    if (layer < 1 || layer >= C.n_layers() || phase < 1 || phase > 3) return fail(VP_ERR_ARG, "bad layer / phase");
    if (world < 1 || (world & (world - 1)) || rank < 0 || rank >= world) return fail(VP_ERR_ARG, "bad world / rank");
    std::vector<PhaseTabG> T;
    int rounds;
    if (phase == 2) {
        rounds = C.max_dad_bit_length(layer);
        if (rounds == -1) { *n_tables = 0; return VP_OK; }
        std::vector<int> order;
        for (int l = 0; l < layer; ++l)
            if (C.layers[layer].dadSize[l] > 0) order.push_back(l);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return C.dad_bit_length(layer, a) > C.dad_bit_length(layer, b); });
        for (int l : order) T.push_back(PhaseTabG{C.dad_bit_length(layer, l), (uint32_t)C.dad_size(layer, l), l, 0});
    } else {
        rounds = C.bit_length(layer - 1);
        T.push_back(PhaseTabG{rounds, (uint32_t)C.layer_size(layer - 1), -1, 0});
    }
    PlanArena A;
    PhasePlan P = make_phase(T, rounds, {}, world, rank, C.n_layers(), A, phase == 2);
    if (cap < T.size() * 10) return fail(VP_ERR_ARG, "output buffer too small");
    for (size_t t = 0; t < T.size(); ++t) {
        uint32_t* o = out + t * 10;
        o[0] = (uint32_t)T[t].bits; o[1] = T[t].live; o[2] = P.sharded; o[3] = (uint32_t)P.m; o[4] = P.row_lo[t];
        o[5] = P.row_hi[t]; o[6] = P.local_len[t]; o[7] = P.present[t];
        o[8] = P.sharded ? std::max<uint32_t>(1, (T[t].live + (1u << P.m) - 1) >> P.m) : 1; o[9] = phase == 2;
    }
    *n_tables = T.size();
    return VP_OK;
}
// Host-only: the per-layer instance ranges a rank of a sharded context evaluates (same code as vp_create_sharded).
extern "C" int vp_shard_eval_ranges(const vp_circuit* c, int world, int rank, uint32_t* lo, uint32_t* hi) {
    if (!c || !lo || !hi) return fail(VP_ERR_ARG, "null argument");
    const Circuit& C = c->c;
    if (world < 1 || (world & (world - 1)) || rank < 0 || rank >= world) return fail(VP_ERR_ARG, "bad world / rank");
    try {
        const int n = C.n_layers();
        PlanArena A;
        std::vector<PhasePlan> p1(n), p2(n), p3(n);
        std::vector<std::vector<int>> srcs(n);
        for (int i = 1; i < n; ++i) {
            const int pb = C.bit_length(i - 1);
            p1[i] = make_phase({PhaseTabG{pb, (uint32_t)C.layer_size(i - 1), -1, 0}}, pb, {}, world, rank, n, A);
            p3[i] = make_phase({PhaseTabG{pb, (uint32_t)C.layer_size(i - 1), -1, 0}}, pb, {}, world, rank, n, A);
            srcs[i] = phase2_order(C, i);
            if (C.max_dad_bit_length(i) != -1) {
                std::vector<PhaseTabG> T;
                for (int l : srcs[i]) T.push_back(PhaseTabG{C.dad_bit_length(i, l), (uint32_t)C.dad_size(i, l), l, 0});
                p2[i] = make_phase(T, C.max_dad_bit_length(i), {}, world, rank, n, A, /*rev=*/true);
            }
        }
        const EvalRanges R = compute_eval_ranges(
            C, (uint32_t)C.instances, world, rank,
            [&](int i, int phase) -> const PhasePlan& { return phase == 1 ? p1[i] : phase == 2 ? p2[i] : p3[i]; },
            [&](int i) -> const std::vector<int>& { return srcs[i]; });
        for (int l = 0; l < n; ++l) { lo[l] = R.lo[l]; hi[l] = R.hi[l]; }
        return VP_OK;
    } catch (const CudaError& e) {
        return fail(VP_ERR_ARG, "%s", e.msg.c_str());
    }
}
extern "C" int vp_shard_map_index(uint32_t lo, uint32_t hi, uint32_t idx, uint32_t* local) {
    uint32_t loc = 0;
    const bool mine = shard_local(ShardMap{lo, hi}, idx, loc);
    if (local) *local = loc;
    if (mine && shard_global(ShardMap{lo, hi}, loc) != idx) return -100;
    return mine ? 1 : 0;
}
extern "C" void vp_destroy(vp_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->e.device);
    delete ctx;
}

struct ScopedTimer {
    Engine& e;
    std::chrono::steady_clock::time_point t0;
    explicit ScopedTimer(Engine& en) : e(en), t0(std::chrono::steady_clock::now()) { cudaSetDevice(e.device); }
    ~ScopedTimer() { e.prove_seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
};
// The device window of vp_last_prove_ms and vp_last_prove_launches around body(); read_back() queues the results to the
// host after it, and one synchronisation ends the call. A device-memory batch (e.dev_io) does not wait: its window covers
// the whole call, read_back() included, and vp_last_prove_ms waits for the window's end when it is read.
template <class Body, class ReadBack>
static void device_window(Engine& e, Body body, ReadBack read_back) {
    const uint64_t l0 = e.launches;
    e.ms_pending = false;
    CK(cudaEventRecord(e.ev0, e.stream));
    body();
    if (e.dev_io) read_back();
    CK(cudaEventRecord(e.ev1, e.stream));
    if (!e.dev_io) read_back();
    e.last_launches = e.launches - l0;
    if (e.dev_io) {
        e.ms_pending = true;
        return;
    }
    CK(cudaStreamSynchronize(e.stream));
    CK(cudaEventElapsedTime(&e.last_ms, e.ev0, e.ev1));
}

extern "C" int vp_set_inputs(vp_ctx* ctx, const uint64_t* inputs, size_t n) {
    if (!ctx || !inputs) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(ctx->e.device);
    ctx->e.load_inputs(inputs, n, true);
    CK(cudaStreamSynchronize(ctx->e.stream));
    return VP_OK;
    API_END
}
extern "C" int vp_evaluate(vp_ctx* ctx) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    e.evaluate();
    ctx->e.check_assert_flag();
    return VP_OK;
    API_END
}
extern "C" int vp_get_values(vp_ctx* ctx, int layer, vp_F* out, size_t n) {
    if (!ctx || !out || layer < 0 || layer >= ctx->e.n) return fail(VP_ERR_ARG, "bad argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (e.world > 1) return fail(VP_ERR_ARG, "vp_get_values: a rank of a sharded context only holds the values of its own instance range");
    if (n > e.C.layer_size(layer)) return fail(VP_ERR_ARG, "n exceeds the layer size");
    CK(cudaMemcpyAsync(out, e.val[layer].p, n * sizeof(F), cudaMemcpyDeviceToHost, e.stream));
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
extern "C" int vp_vres(vp_ctx* ctx, const vp_F* r, int n, vp_F* out) {
    if (!ctx || !r || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (!e.evaluated) return fail(VP_ERR_ARG, "vp_vres before vp_evaluate");
    if (n != e.C.bit_length(e.n - 1)) return fail(VP_ERR_ARG, "vp_vres: n must be the output layer's bit length");
    if (n) e.set_chal(e.lay.ci_out, r, (size_t)n);
    e.do_vres();
    e.get_tr(e.lay.tr_vres, out);
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_init_all(vp_ctx* ctx, const vp_F* r_last, int n) {
    if (!ctx || (!r_last && n)) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (n != e.C.bit_length(e.n - 1)) return fail(VP_ERR_ARG, "sumcheck_init_all: wrong n");
    if (n) e.set_chal(e.lay.ci_out, r_last, (size_t)n);
    e.cur_layer = e.n;
    e.phase = 0;
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_init(vp_ctx* ctx) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    Engine& e = ctx->e;
    if (e.cur_layer <= 1) return fail(VP_ERR_ARG, "sumcheck_init below layer 1");
    --e.cur_layer;
    e.phase = 0;
    return VP_OK;
}
extern "C" int vp_init_phase1(vp_ctx* ctx, const vp_F* assert_random) {
    if (!ctx || !assert_random) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (e.cur_layer < 1 || e.cur_layer >= e.n) return fail(VP_ERR_ARG, "init_phase1 outside a layer");
    e.set_chal(e.L[e.cur_layer].ci_assert, assert_random);
    e.do_init_phase1(e.cur_layer);
    e.phase = 1;
    e.round = 0;
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
extern "C" int vp_init_phase2(vp_ctx* ctx) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (e.cur_layer < 1 || e.cur_layer >= e.n) return fail(VP_ERR_ARG, "init_phase2 outside a layer");
    if (e.L[e.cur_layer].m == -1) return fail(VP_ERR_ARG, "layer %d has no phase 2", e.cur_layer);
    e.do_init_phase2(e.cur_layer);
    e.phase = 2;
    e.round = 0;
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
extern "C" int vp_init_liu(vp_ctx* ctx, const vp_F* sig, int n) {
    if (!ctx || !sig) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (e.cur_layer < 1 || e.cur_layer >= e.n) return fail(VP_ERR_ARG, "init_liu outside a layer");
    const int need = e.n - e.cur_layer + 1;
    if (n < need) return fail(VP_ERR_ARG, "init_liu: need %d sigma values, got %d", need, n);
    e.set_chal(e.L[e.cur_layer].ci_sig, sig, (size_t)std::min(n, e.n));
    e.do_init_liu(e.cur_layer, true);
    e.phase = 3;
    e.round = 0;
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
static uint32_t phase_ci(Engine& e, int phase) {
    LayerDev& D = e.L[e.cur_layer];
    return phase == 1 ? D.ci_ru : phase == 2 ? D.ci_rv : D.ci_rliu;
}
static const PhasePlan& phase_plan(Engine& e, int phase) {
    LayerDev& D = e.L[e.cur_layer];
    return phase == 1 ? D.ph1 : phase == 2 ? D.ph2 : D.ph3;
}
extern "C" int vp_round(vp_ctx* ctx, int phase, const vp_F* previous_random, vp_F out_abc[3]) {
    if (!ctx || !previous_random || !out_abc) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (phase < 1 || phase > 3 || phase != e.phase) return fail(VP_ERR_ARG, "vp_round: phase %d not initialised", phase);
    LayerDev& D = e.L[e.cur_layer];
    const PhasePlan& PP = phase_plan(e, phase);
    if (e.round >= PP.rounds) return fail(VP_ERR_ARG, "vp_round: all %d rounds already done", PP.rounds);
    const uint32_t ci = phase_ci(e, phase);
    const bool fast = !PP.sharded && e.h_round != nullptr;
    if (e.round >= 1) {   // r_arr.at(round-1) = prev (prover.cpp:441)
        if (fast) e.set_chal_host(ci + (uint32_t)(e.round - 1), previous_random);   // the kernel files it on the device
        else e.set_chal(ci + (uint32_t)(e.round - 1), previous_random);
    }
    ++e.round;
    const uint32_t tr = (phase == 1 ? D.tr_p1 : phase == 2 ? D.tr_p2 : D.tr_liu) + 3u * (uint32_t)(e.round - 1);
    const F* at_init = phase == 2 ? e.scal(Engine::SC_UNARY) : nullptr;
    if (PP.sharded) e.sharded_round(PP, phase, e.round, ci, tr, at_init);
    else if (fast) {
        struct Reset { Engine& e; ~Reset() { e.fast_prev = nullptr; e.fast_out = false; } } reset{e};
        e.fast_prev = e.round >= 2 ? previous_random : nullptr;
        e.fast_out = true;
        e.do_round(PP.planB, e.round, ci + (uint32_t)std::max(0, e.round - 2), tr, at_init);
        CK(cudaGetLastError());
        e.round_slot_wait(e.round_seq);
        memcpy(out_abc, e.h_round->poly, 3 * sizeof(F));
    } else e.do_round(PP.planB, e.round, ci + (uint32_t)std::max(0, e.round - 2), tr, at_init);
    if (!fast) e.get_tr(tr, out_abc, 3);
    e.proof_size += 3 * sizeof(F);
    return VP_OK;
    API_END
}
static int finalize_common(vp_ctx* ctx, int phase, const vp_F* prev, vp_F* out, int n_out) {
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (phase != e.phase) return fail(VP_ERR_ARG, "finalize: phase %d not initialised", phase);
    LayerDev& D = e.L[e.cur_layer];
    const PhasePlan& PP = phase_plan(e, phase);
    if (e.round != PP.rounds) return fail(VP_ERR_ARG, "finalize after %d of %d rounds", e.round, PP.rounds);
    const uint32_t ci = phase_ci(e, phase);
    if (e.round >= 1) e.set_chal(ci + (uint32_t)(e.round - 1), prev);
    // a sharded phase ends in its replicated stage B: every rank holds the same claims
    e.do_finalize(PP.planB, ci + (uint32_t)std::max(0, PP.rounds - 1), phase == 1 ? e.scal(Engine::SC_VU) : nullptr);
    const uint32_t tr = phase == 1 ? D.tr_claim_u : phase == 2 ? D.tr_claims_v : D.tr_claim_liu;
    e.get_tr(tr, out, (size_t)n_out);
    e.phase = 0;
    return VP_OK;
}
extern "C" int vp_finalize1(vp_ctx* ctx, const vp_F* previous_random, vp_F* claim) {
    if (!ctx || !previous_random || !claim) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    int rc = finalize_common(ctx, 1, previous_random, claim, 1);
    if (rc == VP_OK) ctx->e.proof_size += sizeof(F);
    return rc;
    API_END
}
extern "C" int vp_finalize2(vp_ctx* ctx, const vp_F* previous_random, vp_F* claims, int n) {
    if (!ctx || !previous_random || !claims) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    if (n != ctx->e.cur_layer) return fail(VP_ERR_ARG, "finalize2: claims must have %d entries", ctx->e.cur_layer);
    int rc = finalize_common(ctx, 2, previous_random, claims, n);
    // prover.cpp:512 adds 16 B for every l < layer (also empty subsets: ~INT_MIN != 0, SURVEY 9.2.7)
    if (rc == VP_OK) ctx->e.proof_size += (uint64_t)n * sizeof(F);
    return rc;
    API_END
}
extern "C" int vp_finalize_liu(vp_ctx* ctx, const vp_F* previous_random, vp_F* claim) {
    if (!ctx || !previous_random || !claim) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    return finalize_common(ctx, 3, previous_random, claim, 1);
    API_END
}
extern "C" int vp_inner_prod(vp_ctx* ctx, const vp_F* pub, size_t n, vp_F* out) {
    if (!ctx || !pub || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (n > e.C.layer_size(0)) return fail(VP_ERR_ARG, "inner_prod: n exceeds the input layer");
    if (e.d_pub.n < n) e.d_pub.alloc(n);
    CK(cudaMemcpyAsync(e.d_pub.p, pub, n * sizeof(F), cudaMemcpyHostToDevice, e.stream));
    if (e.world == 1) {
        k_dot<<<e.grid_for((uint32_t)n, e.cap_dot), 256, 0, e.stream>>>(e.val[0].p, e.d_pub.p, (uint32_t)n, e.d_tr.p + e.lay.tr_input,
                                                               e.d_partials.p, e.d_counter.p);
        ++e.launches;
    } else {   // every rank sums its own slice of the instances, one 16-byte-per-rank all-gather (collective call)
        const size_t S0 = e.C.layers[0].size, b = std::min(n, (size_t)e.ko_lo * S0), en = std::min(n, (size_t)e.ko_hi * S0);
        k_dot<<<e.grid_for((uint32_t)std::max<size_t>(en - b, 1), e.cap_dot), 256, 0, e.stream>>>(e.val[0].p + b, e.d_pub.p + b, (uint32_t)(en - b),
                                                                                              e.d_send.p, e.d_partials.p, e.d_counter.p);
        NCK(g_nccl.AllGather(e.d_send.p, e.d_recv.p, 2, /*ncclUint64*/ 5, e.comm, e.stream));
        k_sum_ranks<<<1, 32, 0, e.stream>>>(e.d_recv.p, (uint32_t)e.world, 1, e.d_tr.p + e.lay.tr_input);
        e.launches += 3;
    }
    e.get_tr(e.lay.tr_input, out);
    return VP_OK;
    API_END
}
extern "C" int vp_dot_host(vp_ctx* ctx, const vp_F* a, const vp_F* b, size_t n, vp_F* out) {
    if (!ctx || !a || !b || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (n > 0xffffffffULL) return fail(VP_ERR_ARG, "vp_dot_host: n too large");
    DBuf<F> da, db;
    da.alloc(std::max<size_t>(n, 1));
    db.alloc(std::max<size_t>(n, 1));
    CK(cudaMemcpyAsync(da.p, a, n * sizeof(F), cudaMemcpyHostToDevice, e.stream));
    CK(cudaMemcpyAsync(db.p, b, n * sizeof(F), cudaMemcpyHostToDevice, e.stream));
    k_dot<<<e.grid_for((uint32_t)n, e.cap_dot), 256, 0, e.stream>>>(da.p, db.p, (uint32_t)n, e.d_tr.p + e.lay.tr_input, e.d_partials.p,
                                                           e.d_counter.p);
    ++e.launches;
    e.get_tr(e.lay.tr_input, out);
    return VP_OK;
    API_END
}
extern "C" int vp_input_mle(vp_ctx* ctx, const vp_F* r, int n, vp_F* out) {
    if (!ctx || !out || (!r && n)) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (n != e.C.bit_length(0)) return fail(VP_ERR_ARG, "input_mle: n must be the input layer's bit length");
    if (n) e.set_chal(e.L[1].ci_rliu, r, (size_t)n);
    e.do_input_mle();
    e.get_tr(e.lay.tr_input, out);
    return VP_OK;
    API_END
}
extern "C" uint64_t vp_proof_size_bytes(const vp_ctx* ctx) { return ctx ? ctx->e.proof_size : 0; }
extern "C" double vp_prove_seconds(const vp_ctx* ctx) { return ctx ? ctx->e.prove_seconds : 0; }

extern "C" int vp_set_challenges(vp_ctx* ctx, const vp_F* challenges, size_t n) {
    if (!ctx || !challenges) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (n != e.lay.n_chal) return fail(VP_ERR_ARG, "expected %zu challenges, got %zu", e.lay.n_chal, n);
    e.set_chal(0, challenges, n);
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
static int prove_impl(vp_ctx* ctx, int host_io, bool local_inputs, const uint64_t* inputs, size_t n_inputs, const vp_F* challenges,
                      size_t n_challenges, vp_F* transcript, size_t transcript_cap) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    if (host_io) {
        if (!inputs || !challenges || !transcript) return fail(VP_ERR_ARG, "host_io needs inputs, challenges and transcript");
        if (n_challenges != e.lay.n_chal) return fail(VP_ERR_ARG, "expected %zu challenges, got %zu", e.lay.n_chal, n_challenges);
        if (transcript_cap < e.lay.n_tr) return fail(VP_ERR_ARG, "transcript buffer too small (%zu < %zu)", transcript_cap, e.lay.n_tr);
    }
    device_window(e, [&] {
        if (host_io) {
            e.set_chal(0, challenges, n_challenges);
            e.load_inputs_chunked(inputs, n_inputs, local_inputs);   // copies overlap evaluate chunk by chunk
        }
        e.prove_all();
        if (host_io) CK(cudaMemcpyAsync(transcript, e.d_tr.p, e.lay.n_tr * sizeof(F), cudaMemcpyDeviceToHost, e.stream));
    }, [&] { e.check_assert_flag(); });
    e.proof_size = e.lay.proof_size;
    return VP_OK;
    API_END
}
extern "C" int vp_prove(vp_ctx* ctx, int host_io, const uint64_t* inputs, size_t n_inputs, const vp_F* challenges,
                        size_t n_challenges, vp_F* transcript, size_t transcript_cap) {
    return prove_impl(ctx, host_io, false, inputs, n_inputs, challenges, n_challenges, transcript, transcript_cap);
}
extern "C" int vp_input_range(const vp_ctx* ctx, uint64_t* first_instance, uint64_t* end_instance) {
    if (!ctx || !first_instance || !end_instance) return fail(VP_ERR_ARG, "null argument");
    *first_instance = ctx->e.k_lo;
    *end_instance = ctx->e.k_hi;
    return VP_OK;
}
extern "C" int vp_prove_local(vp_ctx* ctx, const uint64_t* local_inputs, size_t n_local, const vp_F* challenges, size_t n_challenges,
                              vp_F* transcript, size_t transcript_cap) {
    return prove_impl(ctx, 1, true, local_inputs, n_local, challenges, n_challenges, transcript, transcript_cap);
}
// ------------------------------------------------------------------ C ABI: polynomial commitment, commit phase (N1)
static bool mask_all_zero(const vp_F* mask, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (mask[i].re | mask[i].im) return false;
    return true;
}
extern "C" int vp_commit_private(vp_ctx* ctx, const vp_F* mask, size_t n_mask, uint8_t root[32]) {
    if (!ctx || !root || (n_mask && !mask)) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (e.world > 1) return fail(VP_ERR_ARG, "vp_commit_private needs an unsharded context");
    if (!e.inputs_loaded) return fail(VP_ERR_ARG, "vp_commit_private: inputs not loaded");
    if (!mask_all_zero(mask, n_mask)) return fail(VP_ERR_ARG, "vp_commit_private: only the GKR prover's zero mask is supported (prover.cpp:524-530)");
    const int bl = e.C.bit_length(0);
    if (bl < 6) return fail(VP_ERR_ARG, "vp_commit_private: the input layer needs at least 2^6 padded entries (64 slices)");
    if (!e.pc) e.pc = pc_create(e.device, bl);
    if (!e.evaluated) {   // circuitValue[0] from the resident inputs (what prover::evaluate leaves in layer 0)
        const uint32_t tot0 = (uint32_t)e.C.layer_size(0);
        k_load_inputs<<<cdiv(std::max<uint32_t>(tot0, 1), 256), 256, 0, e.stream>>>(e.d_inputs.p, e.val[0].p, 0, tot0);
        ++e.launches;
    }
    e.last_commit_ms = pc_commit(e.pc, e.val[0].p, e.C.layer_size(0), e.stream, root);
    return VP_OK;
    API_END
}
extern "C" int vp_commit_export(vp_ctx* ctx, vp_F* l_eval, uint8_t* leaf_hash, uint8_t* tree) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    if (!e.pc) return fail(VP_ERR_ARG, "vp_commit_export before vp_commit_private");
    pc_export(e.pc, e.stream, reinterpret_cast<F*>(l_eval), leaf_hash, tree);
    return VP_OK;
    API_END
}
// prover::commit_public (prover.cpp:542-546) -> commit_public_array (poly_commit.h:126-349), zero masks
extern "C" int vp_commit_public(vp_ctx* ctx, const vp_F* pub, size_t n, const vp_F* mask, size_t n_mask, uint8_t root_h[32], vp_F all_sum[65]) {
    if (!ctx || !pub || !root_h || !all_sum || (n_mask && !mask)) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (!e.pc) return fail(VP_ERR_ARG, "vp_commit_public before vp_commit_private");
    if (!mask_all_zero(mask, n_mask)) return fail(VP_ERR_ARG, "vp_commit_public: only the zero public mask of verifier.cpp:376 is supported");
    if (n > ((size_t)1 << e.C.bit_length(0))) return fail(VP_ERR_ARG, "vp_commit_public: public array longer than the padded input layer");
    for (size_t i = 0; i < n; ++i)
        if (pub[i].re >= P || pub[i].im >= P) return fail(VP_ERR_ARG, "vp_commit_public: element %zu is not canonical", i);
    if (e.d_pub.n < n) e.d_pub.alloc(n);
    CK(cudaMemcpyAsync(e.d_pub.p, pub, n * sizeof(F), cudaMemcpyHostToDevice, e.stream));
    e.last_commit_ms = pc_commit_public(e.pc, e.d_pub.p, n, e.stream, root_h, reinterpret_cast<F*>(all_sum));
    return VP_OK;
    API_END
}
extern "C" int vp_commit_public_export(vp_ctx* ctx, vp_F* h_eval, vp_F* vow, uint8_t* leaf_hash, uint8_t* tree) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    if (!e.pc) return fail(VP_ERR_ARG, "vp_commit_public_export before vp_commit_public");
    pc_export_public(e.pc, e.stream, reinterpret_cast<F*>(h_eval), reinterpret_cast<F*>(vow), leaf_hash, tree);
    return VP_OK;
    API_END
}
extern "C" int vp_commit_export_interleaved(vp_ctx* ctx, int which, vp_F* out) {
    if (!ctx || !out || (which != 0 && which != 1)) return fail(VP_ERR_ARG, "bad argument");
    API_BEGIN
    Engine& e = ctx->e;
    if (!e.pc) return fail(VP_ERR_ARG, "vp_commit_export_interleaved before vp_commit_private");
    pc_export_interleaved(e.pc, e.stream, which, reinterpret_cast<F*>(out));
    return VP_OK;
    API_END
}
extern "C" uint64_t vp_commit_slice_size(const vp_ctx* ctx) { return (ctx && ctx->e.pc) ? pc_slice_size(ctx->e.pc) : 0; }
extern "C" float vp_last_commit_ms(const vp_ctx* ctx) { return ctx ? ctx->e.last_commit_ms : 0.f; }
// Stand-alone form on a host array (any field elements, e.g. test vectors): array[0..n) zero-padded to 2^log_len.
extern "C" int vp_pc_commit(int device, const vp_F* array, size_t n, int log_len, uint8_t root[32], vp_F* l_eval, uint8_t* leaf_hash,
                            uint8_t* tree, float* device_ms) {
    if (!array || !root) return fail(VP_ERR_ARG, "null argument");
    if (log_len < 6 || log_len > 30 || n > ((size_t)1 << log_len)) return fail(VP_ERR_ARG, "vp_pc_commit: log_len in [6, 30], n <= 2^log_len");
    API_BEGIN
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(ce)};
    for (size_t i = 0; i < n; ++i)
        if (array[i].re >= P || array[i].im >= P) return fail(VP_ERR_ARG, "vp_pc_commit: element %zu is not canonical", i);
    CK(cudaSetDevice(device));
    struct Guard { PcCommit* p = nullptr; ~Guard() { if (p) pc_destroy(p); } } g;
    g.p = pc_create(device, log_len);
    DBuf<F> d;
    d.alloc(std::max<size_t>(n, 1));
    CK(cudaMemcpy(d.p, array, n * sizeof(F), cudaMemcpyHostToDevice));
    const float ms = pc_commit(g.p, d.p, n, 0, root);
    if (device_ms) *device_ms = ms;
    pc_export(g.p, 0, reinterpret_cast<F*>(l_eval), leaf_hash, tree);
    return VP_OK;
    API_END
}
// Both phases on host arrays: commit_private_array on `array`, then commit_public_array with the public array `pub`.
extern "C" int vp_pc_commit_public(int device, const vp_F* array, size_t n, const vp_F* pub, size_t n_pub, int log_len, uint8_t root_l[32],
                                   uint8_t root_h[32], vp_F all_sum[65], vp_F* h_eval, vp_F* vow, float* device_ms) {
    if (!array || !pub || !root_l || !root_h || !all_sum) return fail(VP_ERR_ARG, "null argument");
    if (log_len < 6 || log_len > 30 || n > ((size_t)1 << log_len) || n_pub > ((size_t)1 << log_len)) return fail(VP_ERR_ARG, "vp_pc_commit_public: log_len in [6, 30], n <= 2^log_len");
    API_BEGIN
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(ce)};
    for (size_t i = 0; i < n; ++i)
        if (array[i].re >= P || array[i].im >= P) return fail(VP_ERR_ARG, "vp_pc_commit_public: array element %zu is not canonical", i);
    for (size_t i = 0; i < n_pub; ++i)
        if (pub[i].re >= P || pub[i].im >= P) return fail(VP_ERR_ARG, "vp_pc_commit_public: public element %zu is not canonical", i);
    CK(cudaSetDevice(device));
    struct Guard { PcCommit* p = nullptr; ~Guard() { if (p) pc_destroy(p); } } g;
    g.p = pc_create(device, log_len);
    DBuf<F> d, dq;
    d.alloc(std::max<size_t>(n, 1));
    dq.alloc(std::max<size_t>(n_pub, 1));
    CK(cudaMemcpy(d.p, array, n * sizeof(F), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dq.p, pub, n_pub * sizeof(F), cudaMemcpyHostToDevice));
    pc_commit(g.p, d.p, n, 0, root_l);
    const float ms = pc_commit_public(g.p, dq.p, n_pub, 0, root_h, reinterpret_cast<F*>(all_sum));
    if (device_ms) *device_ms = ms;
    pc_export_public(g.p, 0, reinterpret_cast<F*>(h_eval), reinterpret_cast<F*>(vow), nullptr, nullptr);
    return VP_OK;
    API_END
}
// fri::commit_phase_step (fri.cpp:289-418), n_steps of them from the context's current FRI level (0 right after
// vp_commit_public): fold every slice's codeword with randomness[k], hash the leaves, build the level's tree.
extern "C" int vp_fri_commit_steps(vp_ctx* ctx, const vp_F* randomness, int n_steps, uint8_t* roots) {
    if (!ctx || !randomness || !roots || n_steps < 0) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    if (!e.pc) return fail(VP_ERR_ARG, "vp_fri_commit_steps before vp_commit_public");
    if (pc_fri_steps_done(e.pc) + n_steps > pc_fri_steps(e.pc))
        return fail(VP_ERR_ARG, "vp_fri_commit_steps: %d steps asked, %d of %d already done", n_steps, pc_fri_steps_done(e.pc), pc_fri_steps(e.pc));
    for (int k = 0; k < n_steps; ++k)
        if (randomness[k].re >= P || randomness[k].im >= P) return fail(VP_ERR_ARG, "vp_fri_commit_steps: challenge %d is not canonical", k);
    e.last_commit_ms = pc_fri_steps_run(e.pc, reinterpret_cast<const F*>(randomness), n_steps, e.stream, roots);
    return VP_OK;
    API_END
}
extern "C" int vp_fri_steps(const vp_ctx* ctx) { return (ctx && ctx->e.pc) ? pc_fri_steps(ctx->e.pc) : 0; }
extern "C" int vp_fri_restart(vp_ctx* ctx) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    if (!ctx->e.pc) return fail(VP_ERR_ARG, "vp_fri_restart before vp_commit_public");
    pc_fri_restart(ctx->e.pc);
    return VP_OK;
    API_END
}
extern "C" int vp_fri_export_level(vp_ctx* ctx, int lvl, vp_F* rs_codeword, uint8_t* merkle) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    if (!e.pc) return fail(VP_ERR_ARG, "vp_fri_export_level before vp_fri_commit_steps");
    if (lvl < 0 || lvl >= pc_fri_steps_done(e.pc)) return fail(VP_ERR_ARG, "vp_fri_export_level: level %d not computed (%d done)", lvl, pc_fri_steps_done(e.pc));
    pc_fri_export(e.pc, e.stream, lvl, reinterpret_cast<F*>(rs_codeword), merkle);
    return VP_OK;
    API_END
}
// Stand-alone form: both commitments on host arrays, then the whole FRI commit phase with the given fold challenges.
// codes / trees (may be NULL): the levels back to back (level l: 64 * (slice_size >> (l+1)) elements, (slice_size >> (l+1)) * 32 bytes).
extern "C" int vp_pc_fri(int device, const vp_F* array, size_t n, const vp_F* pub, size_t n_pub, int log_len, const vp_F* randomness, int n_steps,
                         uint8_t root_l[32], uint8_t root_h[32], uint8_t* roots, vp_F* codes, uint8_t* trees, float* device_ms) {
    if (!array || !pub || !root_l || !root_h || !randomness || !roots) return fail(VP_ERR_ARG, "null argument");
    if (log_len < 7 || log_len > 30 || n > ((size_t)1 << log_len) || n_pub > ((size_t)1 << log_len)) return fail(VP_ERR_ARG, "vp_pc_fri: log_len in [7, 30], n <= 2^log_len");
    if (n_steps < 0 || n_steps > log_len - 6) return fail(VP_ERR_ARG, "vp_pc_fri: at most log_len - 6 steps");
    API_BEGIN
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(ce)};
    for (size_t i = 0; i < n; ++i)
        if (array[i].re >= P || array[i].im >= P) return fail(VP_ERR_ARG, "vp_pc_fri: array element %zu is not canonical", i);
    for (size_t i = 0; i < n_pub; ++i)
        if (pub[i].re >= P || pub[i].im >= P) return fail(VP_ERR_ARG, "vp_pc_fri: public element %zu is not canonical", i);
    for (int k = 0; k < n_steps; ++k)
        if (randomness[k].re >= P || randomness[k].im >= P) return fail(VP_ERR_ARG, "vp_pc_fri: challenge %d is not canonical", k);
    CK(cudaSetDevice(device));
    struct Guard { PcCommit* p = nullptr; ~Guard() { if (p) pc_destroy(p); } } g;
    g.p = pc_create(device, log_len);
    DBuf<F> d, dq;
    d.alloc(std::max<size_t>(n, 1));
    dq.alloc(std::max<size_t>(n_pub, 1));
    CK(cudaMemcpy(d.p, array, n * sizeof(F), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dq.p, pub, n_pub * sizeof(F), cudaMemcpyHostToDevice));
    F all_sum[65];
    pc_commit(g.p, d.p, n, 0, root_l);
    pc_commit_public(g.p, dq.p, n_pub, 0, root_h, all_sum);
    const float ms = pc_fri_steps_run(g.p, reinterpret_cast<const F*>(randomness), n_steps, 0, roots);
    if (device_ms) *device_ms = ms;
    const size_t N = pc_slice_size(g.p);
    size_t off = 0;
    for (int l = 0; l < n_steps; ++l) {
        const size_t m = N >> (l + 1);
        pc_fri_export(g.p, 0, l, codes ? reinterpret_cast<F*>(codes) + 64 * off : nullptr, trees ? trees + 32 * off : nullptr);
        off += m;
    }
    return VP_OK;
    API_END
}
// ------------------------------------------------------------------ C ABI: Fiat-Shamir mode (N4)
// Argument checks shared by the entry points below (VP_ERR_ARG through bad_arg).
static void check_unsharded(const Engine& e, const char* fn) {
    if (e.world != 1) bad_arg("%s: sharded contexts are not supported", fn);
}
static void check_inputs_loaded(const Engine& e, const char* fn) {
    if (!e.inputs_loaded) bad_arg("%s: inputs not loaded", fn);
}
// room for B transcripts and, when asked for, B challenge vectors
static void check_capacity(const Engine& e, size_t B, size_t tr_cap, const vp_F* challenges, size_t ch_cap) {
    if (tr_cap < B * e.lay.n_tr) bad_arg("transcript buffer too small (%zu < %zu)", tr_cap, B * e.lay.n_tr);
    if (challenges && ch_cap < B * e.lay.n_chal) bad_arg("challenge buffer too small (%zu < %zu)", ch_cap, B * e.lay.n_chal);
}
static void check_count(size_t B, const char* fn) {
    if (B == 0 || B > 65535) bad_arg("%s: statement count %zu is not in [1, 65535]", fn, B);
}
// the index of the first non-canonical element of x[0, n), or n
static size_t first_noncanonical(const vp_F* x, size_t n) {
    size_t i = 0;
    while (i < n && x[i].re < P && x[i].im < P) ++i;
    return i;
}
// B statements' inputs (outputs), `per` each, end to end: their count, and every value canonical
static void check_inputs(const uint64_t* x, size_t n, size_t B, size_t per) {
    if (n != B * per) bad_arg("expected %zu inputs (%zu statements of %zu), got %zu", B * per, B, per, n);
    for (size_t i = 0; i < n; ++i)
        if (x[i] >= P) bad_arg("input %zu of statement %zu is not < p", i % per, i / per);
}
static void check_outputs(const vp_F* x, size_t n, size_t B, size_t per) {
    if (n != B * per) bad_arg("expected %zu outputs (%zu statements of %zu), got %zu", B * per, B, per, n);
    const size_t i = first_noncanonical(x, n);
    if (i < n) bad_arg("output %zu of statement %zu is not canonical (components must be < p)", i % per, i / per);
}
static void aggregate_check(const Engine& e, size_t B, const char* fn) {
    check_unsharded(e, fn);
    check_count(B, fn);
    if (e.C.instances % B) bad_arg("%s: %zu statements do not divide the %llu instances", fn, B, (unsigned long long)e.C.instances);
}

// The device Fiat-Shamir prover of vp_prove_fs (unsharded), vp_prove_fs_bound, vp_prove_fs_bound_batch and
// vp_prove_fs_aggregate, in the window of vp_last_prove_ms: a batch's inputs (null: the resident ones), fs_begin, seed()
// (queues the pool's seed), the proof; read_back() queues the digests to the host after the window.
template <class Seed, class ReadBack>
static void prove_fs_window(Engine& e, const uint64_t* inputs, size_t n_inputs, Seed seed, vp_F* transcript, vp_F* challenges,
                            ReadBack read_back) {
    device_window(e, [&] {
        if (inputs) e.load_batch_inputs(inputs, n_inputs);
        e.fs_begin();
        seed();
        e.prove_fs_device(reinterpret_cast<F*>(transcript), reinterpret_cast<F*>(challenges));
    }, read_back);
}
extern "C" int vp_prove_fs(vp_ctx* ctx, const uint8_t seed[32], vp_F* transcript, size_t transcript_cap, vp_F* challenges, size_t challenges_cap) {
    if (!ctx || !seed || !transcript) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    check_capacity(e, 1, transcript_cap, challenges, challenges_cap);
    check_inputs_loaded(e, "vp_prove_fs");
    if (e.world == 1)   // the whole proof queued on the device; sharded contexts keep the host loop
        prove_fs_window(e, nullptr, 0, [&] { e.seed_pool(seed); }, transcript, challenges, [] {});
    else
        device_window(e, [&] { e.prove_fs(seed, reinterpret_cast<F*>(transcript), reinterpret_cast<F*>(challenges)); }, [] {});
    return VP_OK;
    API_END
}
extern "C" int vp_fs_challenges(const vp_circuit* c, const uint8_t seed[32], const vp_F* transcript, size_t n, vp_F* challenges, size_t cap) {
    if (!c || !seed || !transcript || !challenges) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    const ProofLayout lay = proof_layout(c->c);
    if (n != lay.n_tr) return fail(VP_ERR_ARG, "expected a transcript of %zu field elements, got %zu", lay.n_tr, n);
    if (cap < lay.n_chal) return fail(VP_ERR_ARG, "challenge buffer too small (%zu < %zu)", cap, lay.n_chal);
    const size_t i = first_noncanonical(transcript, n);
    if (i < n) return fail(VP_ERR_ARG, "transcript element %zu is not canonical", i);
    fs_challenges(lay, fs_schedule(lay), seed, reinterpret_cast<const F*>(transcript), reinterpret_cast<F*>(challenges));
    return VP_OK;
    API_END
}
static int fs_reject(int code, int* accept, int* fail_code, int* fail_layer) {
    *accept = 0;
    if (fail_code) *fail_code = code;
    if (fail_layer) *fail_layer = 0;
    return VP_OK;
}
// The single-transcript Fiat-Shamir verifier of vp_verify_fs, vp_verify_fs_bound and vp_verify_fs_aggregate: code 7 for a
// non-canonical transcript element; the seed, from the host or, with claimed outputs, read back from where queue_seed()
// queued it on the device; the challenges replayed on the host; with claimed outputs, code 8 unless Vres is their MLE at
// r_out; then vp_verify's checks. The challenges stay resident.
static int fs_verify(Engine& e, const uint8_t* seed, const vp_F* outputs, const std::function<const uint64_t*()>& queue_seed,
                     const vp_F* transcript, size_t n, int* accept, int* fail_code, int* fail_layer) {
    if (n != e.lay.n_tr) bad_arg("expected a transcript of %zu field elements, got %zu", e.lay.n_tr, n);
    if (first_noncanonical(transcript, n) < n) return fs_reject(7, accept, fail_code, fail_layer);
    uint64_t h[4];
    if (outputs) {
        // the verifier's circuitValue[0] from the resident inputs (it does not evaluate the circuit) and the claimed
        // outputs (the output layer) in d_fs_outputs, ahead of the seed's roots
        const size_t n_out = e.C.layer_size(e.n - 1);
        e.leave();
        e.fs_alloc();
        if (e.d_fs_outputs.n < n_out) e.d_fs_outputs.alloc(n_out);
        CK(cudaMemcpyAsync(e.d_fs_outputs.p, outputs, n_out * sizeof(F), cudaMemcpyHostToDevice, e.stream));
        const uint32_t S0 = (uint32_t)e.C.layers[0].size, b0 = e.k_lo * S0, e0 = e.k_hi * S0;
        k_load_inputs<<<cdiv(std::max<uint32_t>(e0 - b0, 1), 256), 256, 0, e.stream>>>(e.d_inputs.p, e.val[0].p, b0, e0);
        ++e.launches;
        CK(cudaMemcpyAsync(h, queue_seed(), sizeof h, cudaMemcpyDeviceToHost, e.stream));
        CK(cudaStreamSynchronize(e.stream));
        seed = reinterpret_cast<const uint8_t*>(h);
    }
    std::vector<F> ch(e.lay.n_chal);
    fs_challenges(e.lay, e.fs_sched, seed, reinterpret_cast<const F*>(transcript), ch.data());
    e.set_chal(0, reinterpret_cast<const vp_F*>(ch.data()), e.lay.n_chal);
    if (outputs) {
        e.run_eq(e.eqb_out, 2);
        if (e.d_vf_out.n < 1) e.d_vf_out.alloc(2);
        e.run_dot_eq(e.d_fs_outputs.p, (uint32_t)e.C.layers[e.n - 1].size, e.eqtab(2, e.C.bit_length(e.n - 1)), e.d_vf_out.p);
        F mle;
        CK(cudaMemcpyAsync(&mle, e.d_vf_out.p, sizeof mle, cudaMemcpyDeviceToHost, e.stream));
        CK(cudaStreamSynchronize(e.stream));
        if (!f_eq(mle, reinterpret_cast<const F*>(transcript)[e.lay.tr_vres])) return fs_reject(8, accept, fail_code, fail_layer);
    }
    *accept = e.verify(reinterpret_cast<const F*>(transcript), fail_code, fail_layer);
    return VP_OK;
}
extern "C" int vp_verify_fs(vp_ctx* ctx, const uint8_t seed[32], const vp_F* transcript, size_t n, int* accept, int* fail_code, int* fail_layer) {
    if (!ctx || !seed || !transcript || !accept) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    return fs_verify(e, seed, nullptr, nullptr, transcript, n, accept, fail_code, fail_layer);
    API_END
}
// ---- statement-bound Fiat-Shamir proofs (unsharded contexts)
// vp_statement_digest and vp_aggregate_digest: the context's values (evaluated if needed), then queue() queues the
// digests and their copies to the host; one synchronisation.
template <class Queue>
static void fs_digest(Engine& e, Queue queue) {
    e.leave();
    e.fs_alloc();
    if (!e.evaluated) e.evaluate();
    queue();
    CK(cudaStreamSynchronize(e.stream));
}
extern "C" int vp_statement_digest(vp_ctx* ctx, const uint8_t context[32], uint8_t circuit[32], uint8_t inputs[32], uint8_t outputs[32],
                                   uint8_t statement[32]) {
    if (!ctx || !context || !statement) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    check_unsharded(e, "vp_statement_digest");
    check_inputs_loaded(e, "vp_statement_digest");
    uint64_t h[4][4];   // d_stmt: circuit, inputs, outputs, statement
    fs_digest(e, [&] {
        e.statement_async(context, nullptr);
        CK(cudaMemcpyAsync(h, e.stmt_circuit(), sizeof h, cudaMemcpyDeviceToHost, e.stream));
    });
    uint8_t* const out[4] = {circuit, inputs, outputs, statement};
    for (int k = 0; k < 4; ++k)
        if (out[k]) memcpy(out[k], h[k], 32);
    return VP_OK;
    API_END
}
extern "C" int vp_prove_fs_bound(vp_ctx* ctx, const uint8_t context[32], vp_F* transcript, size_t cap, vp_F* challenges, size_t ch_cap,
                                 uint8_t statement[32]) {
    if (!ctx || !context || !transcript) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    check_unsharded(e, "vp_prove_fs_bound");
    check_capacity(e, 1, cap, challenges, ch_cap);
    check_inputs_loaded(e, "vp_prove_fs_bound");
    prove_fs_window(e, nullptr, 0, [&] { e.statement_async(context, nullptr); }, transcript, challenges,
                    [&] { if (statement) e.copy_stmts_out(statement, 32, e.stmt_statement(), 32); });
    return VP_OK;
    API_END
}
// A batch runs on the context's slab (Engine::FsSlab): the scope swaps the slab in and, on every exit, the context's own
// buffers and host state back, so that the context's inputs, values, transcript and challenges are untouched. dev: the
// batch's arrays are in device memory (Engine::dev_io).
struct FsBatchScope {
    Engine& e;
    std::vector<F> h_chal;
    bool evaluated;
    int pending_chunks;
    FsBatchScope(Engine& e_, uint32_t B, bool dev, size_t vf_entries = 0)
        : e(e_), h_chal(e_.h_chal), evaluated(e_.evaluated), pending_chunks(e_.pending_chunks) {
        e.slab_reserve(B, vf_entries);
        e.slab_swap();
        e.n_stmt = B;
        e.sstride = e.slab.stride;
        e.pending_chunks = 0;
        e.dev_io = dev;
    }
    ~FsBatchScope() {
        e.slab_swap();
        e.n_stmt = 1;
        e.sstride = 0;
        e.h_chal.swap(h_chal);
        e.evaluated = evaluated;
        e.pending_chunks = pending_chunks;
        e.dev_io = false;
    }
};
// Argument checks of the device-memory batches: every non-null array is device or managed memory of the context's device,
// aligned to `align` bytes (the library cannot see their sizes; the binding checks them from tensor shapes).
struct DevArray {
    const void* p;
    size_t align;
    const char* name;
};
static void check_device_arrays(const Engine& e, const char* fn, std::initializer_list<DevArray> arrays) {
    for (const DevArray& a : arrays) {
        if (!a.p) continue;
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, a.p) != cudaSuccess) {
            cudaGetLastError();
            bad_arg("%s: %s is not a CUDA pointer", fn, a.name);
        }
        if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != e.device)
            bad_arg("%s: %s is not device memory of device %d", fn, a.name, e.device);
        if (reinterpret_cast<uintptr_t>(a.p) % a.align) bad_arg("%s: %s is not %zu-byte aligned", fn, a.name, a.align);
    }
}
// The batch prover of vp_prove_fs_bound_batch (host arrays, checked by the caller; a failed assert gate throws) and
// vp_prove_fs_bound_batch_dev (device arrays: status[b] per statement, the rows of a failed statement zeroed, nothing
// waited for). outputs and status: device arrays only.
static void prove_batch(Engine& e, uint32_t B, bool dev, const uint64_t* inputs, const uint8_t* contexts, vp_F* transcripts,
                        vp_F* challenges, vp_F* outputs, uint8_t* statements, int32_t* status) {
    e.leave();
    e.fs_alloc();
    e.circuit_digest_async();
    e.batch_outputs = 0;
    FsBatchScope scope(e, B, dev);
    prove_fs_window(e, inputs, (size_t)B * e.C.layer_size(0), [&] {
        CK(cudaMemcpyAsync(e.slab.contexts.p, contexts, 32 * (size_t)B, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, e.stream));
        e.statement_async(nullptr, nullptr, e.slab.contexts.p);
    }, transcripts, challenges, [&] {
        if (statements) e.copy_stmts_out(statements, 32, e.stmt_statement(), 32);
        if (!dev) return;
        const size_t n_out = e.C.layer_size(e.n - 1);
        if (outputs) CK(cudaMemcpyAsync(outputs, e.val[e.n - 1].p, B * n_out * sizeof(F), cudaMemcpyDeviceToDevice, e.stream));
        k_batch_zero_failed<<<e.sgrid(1), 256, 0, e.stream>>>(e.slab.status.p, reinterpret_cast<F*>(transcripts), (uint32_t)e.lay.n_tr,
                                                             reinterpret_cast<F*>(challenges), (uint32_t)e.lay.n_chal,
                                                             reinterpret_cast<F*>(outputs), (uint32_t)n_out,
                                                             reinterpret_cast<uint64_t*>(statements), 4);
        ++e.launches;
        CK(cudaMemcpyAsync(status, e.slab.status.p, B * sizeof(int32_t), cudaMemcpyDeviceToDevice, e.stream));
        CK(cudaGetLastError());
    });
    if (!dev) e.batch_outputs = B;
}
extern "C" int vp_prove_fs_bound_batch(vp_ctx* ctx, size_t B, const uint64_t* inputs, size_t n_inputs, const uint8_t* contexts,
                                       vp_F* transcripts, size_t cap, vp_F* challenges, size_t ch_cap, uint8_t* statements) {
    if (!ctx || !inputs || !contexts || !transcripts) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    check_unsharded(e, "vp_prove_fs_bound_batch");
    check_count(B, "vp_prove_fs_bound_batch");
    check_capacity(e, B, cap, challenges, ch_cap);
    check_inputs(inputs, n_inputs, B, e.C.layer_size(0));
    prove_batch(e, (uint32_t)B, false, inputs, contexts, transcripts, challenges, nullptr, statements, nullptr);
    return VP_OK;
    API_END
}
extern "C" int vp_prove_fs_bound_batch_dev(vp_ctx* ctx, size_t B, const uint64_t* d_inputs, const uint8_t* d_contexts,
                                           vp_F* d_transcripts, vp_F* d_challenges, vp_F* d_outputs, uint8_t* d_statements,
                                           int32_t* d_status) {
    if (!ctx || !d_inputs || !d_contexts || !d_transcripts || !d_status) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    const char* fn = "vp_prove_fs_bound_batch_dev";
    check_unsharded(e, fn);
    check_count(B, fn);
    check_device_arrays(e, fn, {{d_inputs, 8, "inputs"}, {d_contexts, 8, "contexts"}, {d_transcripts, 16, "transcripts"},
                                {d_challenges, 16, "challenges"}, {d_outputs, 16, "outputs"}, {d_statements, 8, "statements"},
                                {d_status, 8, "status"}});
    prove_batch(e, (uint32_t)B, true, d_inputs, d_contexts, d_transcripts, d_challenges, d_outputs, d_statements, d_status);
    return VP_OK;
    API_END
}
// The batch's output layers are still in the slab (statement-major: instance-major over B * K instances).
extern "C" int vp_last_batch_outputs(vp_ctx* ctx, vp_F* out, size_t cap) {
    if (!ctx || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (!e.batch_outputs) return fail(VP_ERR_ARG, "vp_last_batch_outputs: no successful vp_prove_fs_bound_batch since the last batch call");
    const size_t cnt = (size_t)e.batch_outputs * e.C.layer_size(e.n - 1);
    if (cap < cnt) return fail(VP_ERR_ARG, "output buffer too small (%zu < %zu)", cap, cnt);
    CK(cudaMemcpyAsync(out, e.slab.val[e.n - 1].p, cnt * sizeof(F), cudaMemcpyDeviceToHost, e.stream));
    CK(cudaStreamSynchronize(e.stream));
    return VP_OK;
    API_END
}
// The batch verifier of vp_verify_fs_bound_batch (host arrays, checked by the caller, whose non-canonical transcripts come
// as zero rows) and vp_verify_fs_bound_batch_dev (device arrays, screened on the device: codes 9 and 7 in slab.status).
// Queues the upload, the roots and statements, the challenge replay and every sum of all B statements; read_back(sums)
// then queues what follows them (sums: statement 0's vf_out_total sums in the slab, sstride bytes per statement).
template <class ReadBack>
static void verify_batch(Engine& e, uint32_t B, bool dev, const uint64_t* inputs, const uint8_t* contexts, const vp_F* outputs,
                         const vp_F* transcripts, ReadBack read_back) {
    const size_t n_in = e.C.layer_size(0), n_out = e.C.layer_size(e.n - 1), n_outputs = (size_t)B * n_out;
    e.leave();
    e.fs_alloc();
    e.circuit_digest_async();
    e.fs_replay_table();
    e.vf_layout();
    if (dev) e.vf_check_table();   // (built once per context: k_verify_check's table)
    e.batch_outputs = 0;
    const uint32_t out_total = e.vf_out_total;
    if (e.d_fs_outputs.n < n_outputs) e.d_fs_outputs.alloc(n_outputs);
    FsBatchScope scope(e, B, dev, (size_t)out_total + (size_t)e.vf_max_b * Engine::VF_GX * 2);
    F* const d_out = reinterpret_cast<F*>(e.slab.mem.p + e.slab.o_vf);
    F* const d_part = d_out + out_total;
    const size_t tr_bytes = e.lay.n_tr * sizeof(F);
    device_window(e, [&] {
        if (dev) {
            CK(cudaMemcpy2DAsync(e.d_tr.p, e.sstride, transcripts, tr_bytes, tr_bytes, B, cudaMemcpyDeviceToDevice, e.stream));
            k_batch_screen<<<e.sgrid(1), 256, 0, e.stream>>>(inputs, e.d_inputs.p, (uint32_t)n_in, reinterpret_cast<const F*>(outputs),
                                                            e.d_fs_outputs.p, (uint32_t)n_out, e.d_tr.p, (uint32_t)e.lay.n_tr, e.sstride, 9,
                                                            e.slab.status.p);
            ++e.launches;
        } else {
            CK(cudaMemcpyAsync(e.d_inputs.p, inputs, B * n_in * sizeof(uint64_t), cudaMemcpyHostToDevice, e.stream));
            CK(cudaMemcpyAsync(e.d_fs_outputs.p, outputs, n_outputs * sizeof(F), cudaMemcpyHostToDevice, e.stream));
            CK(cudaMemcpy2DAsync(e.d_tr.p, e.sstride, transcripts, tr_bytes, tr_bytes, B, cudaMemcpyHostToDevice, e.stream));
        }
        CK(cudaMemcpyAsync(e.slab.contexts.p, contexts, 32 * (size_t)B, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, e.stream));
        e.memset_stmts(e.d_chal.p, (e.lay.n_chal + 1) * sizeof(F));   // unused challenge slots are zero
        e.memset_stmts(d_out, (size_t)out_total * sizeof(F));
        const uint32_t n0 = (uint32_t)(B * n_in);   // circuitValue[0] of every statement, instance-major over B * K
        k_load_inputs<<<cdiv(n0, 256), 256, 0, e.stream>>>(e.d_inputs.p, e.val[0].p, 0, n0);
        ++e.launches;
        e.statement_async(nullptr, e.d_fs_outputs.p, e.slab.contexts.p);
        k_fs_replay<<<e.sgrid(1), 32, 0, e.stream>>>(e.d_fs_steps.p, (uint32_t)e.d_fs_steps.n, e.d_fs_pool.p, e.d_tr.p, e.d_chal.p, e.sstride);
        ++e.launches;
        // the claim chain starts from Vres: the MLE of the claimed outputs at r_out, next to the input MLE
        e.run_eq(e.eqb_out, 2);
        e.run_dot_eq(e.d_fs_outputs.p, (uint32_t)e.C.layers[e.n - 1].size, e.eqtab(2, e.C.bit_length(e.n - 1)), d_out + out_total - 1);
        e.verify_sums_async(d_out, d_part);
    }, [&] { read_back(static_cast<const F*>(d_out)); });
}
extern "C" int vp_verify_fs_bound_batch(vp_ctx* ctx, size_t B, const uint64_t* inputs, size_t n_inputs, const uint8_t* contexts,
                                        const vp_F* outputs, size_t n_outputs, const vp_F* transcripts, size_t n_tr, int* accept,
                                        int* fail_code, int* fail_layer, vp_F* challenges, size_t ch_cap) {
    if (!ctx || !inputs || !contexts || !outputs || !transcripts || !accept) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    check_unsharded(e, "vp_verify_fs_bound_batch");
    check_count(B, "vp_verify_fs_bound_batch");
    const size_t n_in = e.C.layer_size(0), n_out = e.C.layer_size(e.n - 1);
    check_inputs(inputs, n_inputs, B, n_in);
    check_outputs(outputs, n_outputs, B, n_out);
    if (n_tr != B * e.lay.n_tr) return fail(VP_ERR_ARG, "expected %zu transcript elements (%zu statements of %zu), got %zu", B * e.lay.n_tr, B, e.lay.n_tr, n_tr);
    check_capacity(e, B, n_tr, challenges, ch_cap);
    // a statement with a non-canonical transcript element is rejected (code 7) on its own; its row goes up as zeros
    const F* tr = reinterpret_cast<const F*>(transcripts);
    std::vector<uint8_t> bad(B, 0);
    std::vector<F> clean;
    for (size_t b = 0; b < B; ++b) bad[b] = first_noncanonical(transcripts + b * e.lay.n_tr, e.lay.n_tr) < e.lay.n_tr;
    if (std::find(bad.begin(), bad.end(), 1) != bad.end()) {
        clean.assign(tr, tr + n_tr);
        for (size_t b = 0; b < B; ++b)
            if (bad[b]) std::fill(clean.begin() + b * e.lay.n_tr, clean.begin() + (b + 1) * e.lay.n_tr, f_zero());
        tr = clean.data();
    }
    std::vector<F> sums, ch((size_t)B * e.lay.n_chal);
    uint32_t out_total = 0;
    verify_batch(e, (uint32_t)B, false, inputs, contexts, outputs, reinterpret_cast<const vp_F*>(tr), [&](const F* d_out) {
        out_total = e.vf_out_total;
        sums.resize((size_t)B * out_total);
        e.copy_stmts_out(sums.data(), out_total * sizeof(F), d_out, out_total * sizeof(F));
        e.copy_stmts_out(ch.data(), e.lay.n_chal * sizeof(F), e.d_chal.p, e.lay.n_chal * sizeof(F));
        CK(cudaGetLastError());
    });
    // the host driver, one statement at a time, in vp_verify_fs_bound's order: code 7, code 8, then vp_verify's checks
    for (size_t b = 0; b < B; ++b) {
        int code = 0, layer = 0, ok = 0;
        const F* tb = tr + b * e.lay.n_tr;
        const F* sb = sums.data() + b * out_total;
        if (bad[b]) code = 7;
        else if (!f_eq(sb[out_total - 1], tb[e.lay.tr_vres])) code = 8;
        else ok = e.verify_check(tb, sb, ch.data() + b * e.lay.n_chal, &code, &layer);
        accept[b] = ok;
        if (fail_code) fail_code[b] = code;
        if (fail_layer) fail_layer[b] = layer;
        if (bad[b]) std::fill(ch.begin() + b * e.lay.n_chal, ch.begin() + (b + 1) * e.lay.n_chal, f_zero());
    }
    if (challenges) memcpy(challenges, ch.data(), ch.size() * sizeof(F));
    return VP_OK;
    API_END
}
extern "C" int vp_verify_fs_bound_batch_dev(vp_ctx* ctx, size_t B, const uint64_t* d_inputs, const uint8_t* d_contexts,
                                            const vp_F* d_outputs, const vp_F* d_transcripts, int32_t* d_accept, int32_t* d_code,
                                            int32_t* d_layer, vp_F* d_challenges) {
    if (!ctx || !d_inputs || !d_contexts || !d_outputs || !d_transcripts || !d_accept) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    const char* fn = "vp_verify_fs_bound_batch_dev";
    check_unsharded(e, fn);
    check_count(B, fn);
    check_device_arrays(e, fn, {{d_inputs, 8, "inputs"}, {d_contexts, 8, "contexts"}, {d_outputs, 16, "outputs"},
                                {d_transcripts, 16, "transcripts"}, {d_accept, 8, "accept"}, {d_code, 8, "code"}, {d_layer, 8, "layer"},
                                {d_challenges, 16, "challenges"}});
    verify_batch(e, (uint32_t)B, true, d_inputs, d_contexts, d_outputs, d_transcripts, [&](const F* d_out) {
        // the claim chain on the device, one thread per statement, then the challenges (zero for codes 7 and 9)
        k_verify_check<<<cdiv((uint32_t)B, 128), 128, 0, e.stream>>>(e.vf_check_table(), e.d_tr.p, e.d_chal.p, d_out, e.sstride,
                                                                    (uint32_t)B, e.slab.status.p, d_accept, d_code, d_layer);
        ++e.launches;
        if (d_challenges) {
            e.copy_stmts_out(d_challenges, e.lay.n_chal * sizeof(F), e.d_chal.p, e.lay.n_chal * sizeof(F));
            k_batch_zero_failed<<<e.sgrid(1), 256, 0, e.stream>>>(e.slab.status.p, reinterpret_cast<F*>(d_challenges), (uint32_t)e.lay.n_chal, nullptr, 0,
                                                                 nullptr, 0, nullptr, 0);
            ++e.launches;
        }
        CK(cudaGetLastError());
    });
    return VP_OK;
    API_END
}
extern "C" int vp_verify_fs_bound(vp_ctx* ctx, const uint8_t context[32], const vp_F* outputs, size_t n_outputs, const vp_F* transcript,
                                  size_t n, int* accept, int* fail_code, int* fail_layer) {
    if (!ctx || !context || !outputs || !transcript || !accept) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    check_unsharded(e, "vp_verify_fs_bound");
    check_inputs_loaded(e, "vp_verify_fs_bound");
    check_outputs(outputs, n_outputs, 1, e.C.layer_size(e.n - 1));
    return fs_verify(e, nullptr, outputs, [&] { e.statement_async(context, e.d_fs_outputs.p); return e.stmt_statement(); }, transcript, n,
                     accept, fail_code, fail_layer);
    API_END
}
// ---- aggregate proofs: one Fiat-Shamir proof of B statements (unsharded contexts)
// after aggregate_async: the statements (B * 32 bytes, may be null) and the aggregate (32 bytes, may be null) to the host
static void aggregate_read(Engine& e, uint32_t B, uint8_t* statements, uint8_t* aggregate) {
    if (statements) CK(cudaMemcpyAsync(statements, e.agg_statements(B), 32 * (size_t)B, cudaMemcpyDeviceToHost, e.stream));
    if (aggregate) CK(cudaMemcpyAsync(aggregate, e.agg_digest(B), 32, cudaMemcpyDeviceToHost, e.stream));
}
extern "C" int vp_aggregate_digest(vp_ctx* ctx, size_t B, const uint8_t* contexts, uint8_t* statements, uint8_t aggregate[32]) {
    if (!ctx || !contexts || !aggregate) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    aggregate_check(e, B, "vp_aggregate_digest");
    check_inputs_loaded(e, "vp_aggregate_digest");
    fs_digest(e, [&] {
        e.aggregate_async((uint32_t)B, contexts, nullptr);
        aggregate_read(e, (uint32_t)B, statements, aggregate);
    });
    return VP_OK;
    API_END
}
extern "C" int vp_prove_fs_aggregate(vp_ctx* ctx, size_t B, const uint8_t* contexts, vp_F* transcript, size_t cap, vp_F* challenges,
                                     size_t ch_cap, uint8_t* statements, uint8_t aggregate[32]) {
    if (!ctx || !contexts || !transcript) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    ScopedTimer t(e);
    aggregate_check(e, B, "vp_prove_fs_aggregate");
    check_capacity(e, 1, cap, challenges, ch_cap);
    check_inputs_loaded(e, "vp_prove_fs_aggregate");
    prove_fs_window(e, nullptr, 0, [&] { e.aggregate_async((uint32_t)B, contexts, nullptr); }, transcript, challenges,
                    [&] { aggregate_read(e, (uint32_t)B, statements, aggregate); });
    return VP_OK;
    API_END
}
extern "C" int vp_verify_fs_aggregate(vp_ctx* ctx, size_t B, const uint8_t* contexts, const vp_F* outputs, size_t n_outputs,
                                      const vp_F* transcript, size_t n, int* accept, int* fail_code, int* fail_layer) {
    if (!ctx || !contexts || !outputs || !transcript || !accept) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    aggregate_check(e, B, "vp_verify_fs_aggregate");
    check_inputs_loaded(e, "vp_verify_fs_aggregate");
    check_outputs(outputs, n_outputs, B, e.C.layer_size(e.n - 1) / B);
    return fs_verify(e, nullptr, outputs, [&] { e.aggregate_async((uint32_t)B, contexts, e.d_fs_outputs.p); return e.agg_digest((uint32_t)B); },
                     transcript, n, accept, fail_code, fail_layer);
    API_END
}
extern "C" int vp_fs_round_stamps(vp_ctx* ctx, unsigned long long* out, size_t cap, size_t* n_rounds) {
    if (!ctx || !n_rounds) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    *n_rounds = e.fs_rounds;
    if (out && e.fs_rounds) {
        if (cap < 4 * e.fs_rounds) return fail(VP_ERR_ARG, "stamp buffer too small (%zu < %zu)", cap, 4 * e.fs_rounds);
        CK(cudaMemcpy(out, e.d_fs_stamps.p, 4 * e.fs_rounds * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    }
    return VP_OK;
    API_END
}
extern "C" int vp_selftest_field(int device, int op, const vp_F* a, const vp_F* b, const vp_F* c, vp_F* out, size_t n) {
    if (!a || !b || !c || !out || n == 0 || n > (1u << 24) || op < 0 || op > 7) return fail(VP_ERR_ARG, "bad argument");
    API_BEGIN
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(e)};
    CK(cudaSetDevice(device));
    DBuf<F> da, db, dc, dout;
    da.alloc(n); db.alloc(n); dc.alloc(n); dout.alloc(n);
    CK(cudaMemcpy(da.p, a, n * sizeof(F), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(db.p, b, n * sizeof(F), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dc.p, c, n * sizeof(F), cudaMemcpyHostToDevice));
    CK(cudaMemset(dout.p, 0, n * sizeof(F)));
    k_selftest_field<<<cdiv((uint32_t)n, 128), 128>>>(op, da.p, db.p, dc.p, dout.p, (uint32_t)n);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout.p, n * sizeof(F), cudaMemcpyDeviceToHost));
    return VP_OK;
    API_END
}
extern "C" int vp_verify(vp_ctx* ctx, const vp_F* transcript, size_t n, int* accept, int* fail_code, int* fail_layer) {
    if (!ctx || !transcript || !accept) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (n != e.lay.n_tr) return fail(VP_ERR_ARG, "expected a transcript of %zu field elements, got %zu", e.lay.n_tr, n);
    *accept = e.verify(reinterpret_cast<const F*>(transcript), fail_code, fail_layer);
    return VP_OK;
    API_END
}
extern "C" int vp_get_transcript(vp_ctx* ctx, vp_F* transcript, size_t cap) {
    if (!ctx || !transcript) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    if (cap < e.lay.n_tr) return fail(VP_ERR_ARG, "transcript buffer too small");
    e.get_tr(0, transcript, e.lay.n_tr);
    return VP_OK;
    API_END
}
extern "C" int vp_set_stream(vp_ctx* ctx, void* cuda_stream) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    CK(cudaStreamSynchronize(e.stream));
    if (e.own_stream && e.stream) cudaStreamDestroy(e.stream);
    if (cuda_stream) {
        e.stream = (cudaStream_t)cuda_stream;
        e.own_stream = false;
    } else {
        CK(cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking));
        e.own_stream = true;
    }
    return VP_OK;
    API_END
}
extern "C" int vp_set_profiling(vp_ctx* ctx, int on) {
    if (!ctx) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    CK(cudaStreamSynchronize(e.stream));
    e.prof_collect();
    e.profiling = on != 0;
    if (on) {
        for (int k = 0; k < Engine::KC_N; ++k) { e.prof_ms[k] = 0; e.prof_bytes[k] = 0; e.prof_launches[k] = 0; }
    }
    return VP_OK;
    API_END
}
extern "C" int vp_set_lanes(vp_ctx* ctx, int lanes) {
    if (!ctx) return 0;
    Engine& e = ctx->e;
    const bool have2 = e.lane1.stream != nullptr, have3 = e.lane2.stream != nullptr, have6 = e.lane0b.stream != nullptr;
    e.two_lanes = lanes >= 2 && have2;
    e.three_lanes = lanes >= 3 && have2 && have3;
    e.six_lanes = lanes >= 6 && e.three_lanes && have6;
    return e.six_lanes ? 6 : e.three_lanes ? 3 : e.two_lanes ? 2 : 1;
}
extern "C" int vp_get_profile(vp_ctx* ctx, double* ms, double* bytes, uint64_t* launches, int n) {
    if (!ctx || !ms || !bytes || !launches) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    Engine& e = ctx->e;
    cudaSetDevice(e.device);
    CK(cudaStreamSynchronize(e.stream));
    e.prof_collect();
    for (int k = 0; k < n && k < Engine::KC_N; ++k) { ms[k] = e.prof_ms[k]; bytes[k] = e.prof_bytes[k]; launches[k] = e.prof_launches[k]; }
    return VP_OK;
    API_END
}
extern "C" float vp_last_prove_ms(const vp_ctx* ctx) {
    if (!ctx) return 0.f;
    Engine& e = const_cast<vp_ctx*>(ctx)->e;
    if (e.ms_pending) {   // a device-memory batch: wait for its window's end
        e.ms_pending = false;
        cudaSetDevice(e.device);
        if (cudaEventSynchronize(e.ev1) != cudaSuccess || cudaEventElapsedTime(&e.last_ms, e.ev0, e.ev1) != cudaSuccess) {
            cudaGetLastError();
            e.last_ms = 0.f;
        }
    }
    return e.last_ms;
}
extern "C" uint64_t vp_last_prove_launches(const vp_ctx* ctx) { return ctx ? ctx->e.last_launches : 0; }
extern "C" void* vp_stream(vp_ctx* ctx) { return ctx ? (void*)ctx->e.stream : nullptr; }

// ------------------------------------------------------------------ stand-alone sumcheck (config C2)
struct vp_sumcheck {
    int log_n = 0, device = 0;
    uint32_t N = 0;
    cudaStream_t stream = nullptr;
    DBuf<F> src[3];               // pristine V, add, mult
    DBuf<F> bufV[2], bufM[2], bufA[2];
    DBuf<F> d_r, d_out, d_scal, d_claims, d_partials;
    DBuf<unsigned int> d_counter;
    DBuf<TabDesc> d_tabs;
    DBuf<ColDesc> d_cols;
    DBuf<FinDesc> d_fins;
    PlanArena arena;
    SumcheckPlan plan;
    PassPlan pp;
    DBuf<PassTab> d_ptabs;
    DBuf<PassCol> d_pcols;
    DBuf<PassDev> d_pdev;
    DBuf<unsigned long long> d_dbg;
    DBuf<ChainDesc> d_chain;
    DBuf<ChainSeg> d_chain_seg;
    DBuf<ChainTerm> d_chain_term;
    int max_grid = 148 * 4, cap_fold = 148, cap_first = 148, cap_dfs = 148;
    std::vector<cudaEvent_t> ev;
    std::vector<float> round_ms;
    ~vp_sumcheck() {
        for (auto e : ev) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
};

static int sumcheck_create_impl(int log_n, int device, vp_sumcheck** out, bool with_src);
extern "C" int vp_sumcheck_create(int log_n, int device, vp_sumcheck** out) { return sumcheck_create_impl(log_n, device, out, true); }
// with_src = false: no pristine copies of the three tables (the caller fills buf[0] itself before every run)
static int sumcheck_create_impl(int log_n, int device, vp_sumcheck** out, bool with_src) {
    if (!out || log_n < 1 || log_n > 30) return fail(VP_ERR_ARG, "bad argument");
    API_BEGIN
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(e)};
    std::unique_ptr<vp_sumcheck> s(new vp_sumcheck());
    s->log_n = log_n;
    s->device = device;
    s->N = 1u << log_n;
    CK(cudaSetDevice(device));
    struct { int multiProcessorCount = 0; } prop;   // (cudaGetDeviceProperties takes milliseconds; one attribute is all that is needed)
    CK(cudaDeviceGetAttribute(&prop.multiProcessorCount, cudaDevAttrMultiProcessorCount, device));
    int occ = 0, occ1 = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_round<true>, 256, 0));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ1, k_round<false>, 256, 0));
    s->cap_fold = prop.multiProcessorCount * std::max(1, occ);
    s->cap_first = prop.multiProcessorCount * std::max(1, occ1);
    s->max_grid = std::max(s->cap_fold, s->cap_first);
    CK(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
    // out layout: per round (a,b,c) at 3*(j-1); finals: V, add, mult at 3*log_n + {0,1,2}. The plan
    // finalises one table (V); add/mult finals are folded by two more k_finalize launches.
    std::vector<PlanTable> t{{log_n, s->N, -1, 0}};
    s->plan = build_plan(t, log_n, {3u * (uint32_t)log_n}, s->arena);
    s->pp = build_pass_plan(t, log_n, {3u * (uint32_t)log_n}, s->arena);
    {
        int occd = 0;
        dfs_enable_smem();
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occd, k_phase_dfs<true, DFS_NEED_B>, DFS_THREADS, DFS_DYN_SMEM));
        s->cap_dfs = prop.multiProcessorCount * std::max(1, occd);
        s->max_grid = std::max(s->max_grid, s->cap_dfs);
    }
    if (with_src)
        for (int i = 0; i < 3; ++i) s->src[i].alloc(s->N);
    for (int b = 0; b < 2; ++b) {
        const uint32_t cap = std::max<uint32_t>(4, b == 0 ? std::max(s->plan.cap0, s->pp.cap0) : std::max(s->plan.cap1, s->pp.cap1));
        s->bufV[b].alloc(cap);
        s->bufM[b].alloc(cap);
        s->bufA[b].alloc(cap);
    }
    s->d_r.alloc((size_t)log_n + 1);
    s->d_out.alloc((size_t)3 * log_n + 3);
    s->d_scal.alloc(4);
    s->d_claims.alloc(4);
    s->d_partials.alloc((size_t)12 * s->max_grid);
    s->d_counter.alloc(4 + 64);
    s->d_dbg.alloc(256 + 2048);
    s->d_ptabs.upload(s->arena.ptabs, s->stream);
    s->d_pcols.upload(s->arena.pcols, s->stream);
    s->d_pdev.upload(s->arena.pdev, s->stream);
    s->d_chain.upload(std::vector<ChainDesc>{ChainDesc{-2, 0, 0, 0, 1}}, s->stream);
    s->d_chain_seg.upload(std::vector<ChainSeg>{ChainSeg{0, (uint32_t)log_n, 0}}, s->stream);
    s->d_chain_term.upload(std::vector<ChainTerm>{ChainTerm{0, 0}}, s->stream);
    // FinDesc for add and mult finals (same offsets as V's)
    FinDesc fv = s->arena.fins[s->plan.fin_begin];
    FinDesc fa = fv, fm = fv;
    fa.out_idx = 3u * (uint32_t)log_n + 1;
    fm.out_idx = 3u * (uint32_t)log_n + 2;
    s->arena.fins.push_back(fa);
    s->arena.fins.push_back(fm);
    s->d_tabs.upload(s->arena.tabs, s->stream);
    s->d_cols.upload(s->arena.cols, s->stream);
    s->d_fins.upload(s->arena.fins, s->stream);
    CK(cudaMemsetAsync(s->d_counter.p, 0, (4 + 64) * sizeof(unsigned int), s->stream));
    CK(cudaMemsetAsync(s->d_scal.p, 0, 4 * sizeof(F), s->stream));
    s->ev.resize((size_t)log_n + 2);
    for (auto& evx : s->ev) CK(cudaEventCreate(&evx));
    s->round_ms.assign((size_t)log_n, 0.f);
    CK(cudaStreamSynchronize(s->stream));
    *out = s.release();
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_load(vp_sumcheck* s, const vp_F* V, const vp_F* add, const vp_F* mult) {
    if (!s || !V || !add || !mult) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(s->device);
    const vp_F* h[3] = {V, add, mult};
    for (int i = 0; i < 3; ++i)
        CK(cudaMemcpyAsync(s->src[i].p, h[i], (size_t)s->N * sizeof(F), cudaMemcpyHostToDevice, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_fill_random(vp_sumcheck* s, uint64_t seed) {
    if (!s) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(s->device);
    for (int i = 0; i < 3; ++i)
        k_fill_random<<<cdiv(s->N, 256), 256, 0, s->stream>>>(s->src[i].p, s->N, seed * 3 + (uint64_t)i);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(s->stream));
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_export(vp_sumcheck* s, vp_F* V, vp_F* add, vp_F* mult) {
    if (!s || !V || !add || !mult) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(s->device);
    vp_F* h[3] = {V, add, mult};
    for (int i = 0; i < 3; ++i)
        CK(cudaMemcpyAsync(h[i], s->src[i].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToHost, s->stream));
    CK(cudaStreamSynchronize(s->stream));
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_run(vp_sumcheck* s, const vp_F* r, vp_F* out, float* device_ms) {
    if (!s || !r || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(s->device);
    cudaStream_t st = s->stream;
    const int n = s->log_n;
    CK(cudaMemcpyAsync(s->d_r.p, r, (size_t)n * sizeof(F), cudaMemcpyHostToDevice, st));
    // restore the working tables (untimed: the reference's tables also exist before round 1)
    CK(cudaMemcpyAsync(s->bufV[0].p, s->src[0].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(s->bufA[0].p, s->src[1].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(s->bufM[0].p, s->src[2].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToDevice, st));
    CK(cudaEventRecord(s->ev[0], st));
    for (int j = 1; j <= n; ++j) {
        const RoundPlan& R = s->plan.r[j - 1];
        RoundArgs a{};
        const int ib = R.in_buf, ob = ib ^ 1;
        a.inV = s->bufV[ib].p; a.inM = s->bufM[ib].p; a.inA = s->bufA[ib].p;
        a.outV = s->bufV[ob].p; a.outM = s->bufM[ob].p; a.outA = s->bufA[ob].p;
        a.tabs = s->d_tabs.p + R.tab_begin;
        a.cols = s->d_cols.p + R.col_begin;
        a.n_tabs = R.n_tabs;
        a.n_cols = R.n_cols;
        a.prev_r = s->d_r.p + std::max(0, j - 2);
        a.add_term = s->d_scal.p;
        a.claims = s->d_claims.p;
        a.out_poly = s->d_out.p + 3 * (j - 1);
        a.partials = s->d_partials.p;
        a.counter = s->d_counter.p;
        a.first_round = j == 1;
        a.reset_add_term = j == 1;
        const int grid = (int)std::max<uint32_t>(1, std::min<uint32_t>(cdiv(R.work, 256), (uint32_t)(R.fold ? s->cap_fold : s->cap_first)));
        if (R.fold) k_round<true><<<grid, 256, 0, st>>>(a);
        else k_round<false><<<grid, 256, 0, st>>>(a);
        CK(cudaEventRecord(s->ev[j], st));
    }
    const int fb = s->plan.fin_buf;
    const F* tabs3[3] = {s->bufV[fb].p, s->bufA[fb].p, s->bufM[fb].p};
    for (int k = 0; k < 3; ++k) {
        const uint32_t fi = k == 0 ? s->plan.fin_begin : (uint32_t)s->arena.fins.size() - 3 + (uint32_t)k;
        k_finalize<<<1, 32, 0, st>>>(s->d_fins.p + fi, 1, tabs3[k], s->d_r.p + (n - 1), 1, s->d_claims.p, s->d_out.p, nullptr);
    }
    CK(cudaEventRecord(s->ev[n + 1], st));
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, s->d_out.p, ((size_t)3 * n + 3) * sizeof(F), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float tot = 0;
    CK(cudaEventElapsedTime(&tot, s->ev[0], s->ev[n + 1]));
    for (int j = 1; j <= n; ++j) CK(cudaEventElapsedTime(&s->round_ms[j - 1], s->ev[j - 1], s->ev[j]));
    if (device_ms) *device_ms = tot;
    return VP_OK;
    API_END
}
// Same result as vp_sumcheck_run, all rounds in ONE cooperative launch with two rounds per pass (k_phase_dfs):
// possible because all challenges r[] are known up front.
// (the launches only: tables already in buf[0], challenges r[] on the host; results stay in s->d_out)
static void sumcheck_fused_async(vp_sumcheck* s, const vp_F* r) {
    cudaStream_t st = s->stream;
    const int n = s->log_n;
    CK(cudaMemcpyAsync(s->d_r.p, r, (size_t)n * sizeof(F), cudaMemcpyHostToDevice, st));
    DfsArgs a;
    for (int b = 0; b < 2; ++b) { a.bufV[b] = s->bufV[b].p; a.bufM[b] = s->bufM[b].p; a.bufA[b] = s->bufA[b].p; }
    a.passes = s->d_pdev.p + s->pp.pass_begin;
    a.tabs = s->d_ptabs.p;
    a.cols = s->d_pcols.p;
    a.fins = s->d_fins.p + s->pp.fin_begin;   // arena.fins is uploaded as a whole: indices are global
    a.n_passes = s->pp.n_passes;
    a.n_fin = s->pp.n_fin;
    a.fin_buf = (uint32_t)s->pp.fin_buf;
    a.tail_work = 512;
    a.round_base = 0;
    a.at_init = nullptr;
    a.chal = s->d_r.p;
    a.add_term = s->d_scal.p;
    a.claims = s->d_claims.p;
    a.out_poly = s->d_out.p;
    a.transcript = s->d_out.p;
    a.keep = nullptr;
    a.partials = s->d_partials.p;
    a.bar = s->d_counter.p + 2;
    a.chunk_ctr = s->d_counter.p + 4;
    a.v_first = nullptr;
    a.claim0 = s->d_scal.p + 1;
    for (int jr = 0; jr < 32; ++jr) a.rk[jr] = make_constk(jr < n ? F{r[jr].re, r[jr].im} : f_zero());
    a.dbg = s->d_dbg.p;
    CK(cudaMemsetAsync(s->d_dbg.p, 0, 256 * sizeof(unsigned long long), st));
    const int grid = s->pp.max_work <= DFS_CHUNK ? 1 : (int)std::min<uint32_t>(cdiv(s->pp.max_work, DFS_CHUNK) + 1, std::max<uint32_t>((uint32_t)s->cap_dfs, 2));
    void* args[] = {&a};
    CK(cudaLaunchCooperativeKernel((const void*)k_phase_dfs<true, DFS_NEED_B>, dim3(grid), dim3(DFS_THREADS), args, DFS_DYN_SMEM, st));
    // b of every round from the claim chain; round 1's claim p(0) + p(1) was summed by the kernel
    k_derive_b<<<1, 32, 0, st>>>(s->d_chain.p, 1, s->d_chain_seg.p, s->d_chain_term.p, s->d_r.p, s->d_out.p, s->d_scal.p + 1);
    // the fully folded add / mult values sit where V's does
    const FinDesc fv = s->arena.fins[s->pp.fin_begin];
    const F* fin_tabs[2] = {s->bufA[s->pp.fin_buf].p, s->bufM[s->pp.fin_buf].p};
    for (int k = 0; k < 2; ++k) k_strict_copy<<<1, 32, 0, st>>>(s->d_out.p + 3 * n + 1 + k, fin_tabs[k] + fv.in_off, 1);
}
extern "C" int vp_sumcheck_run_fused(vp_sumcheck* s, const vp_F* r, vp_F* out, float* device_ms) {
    if (!s || !r || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(s->device);
    cudaStream_t st = s->stream;
    const int n = s->log_n;
    CK(cudaMemcpyAsync(s->bufV[0].p, s->src[0].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(s->bufA[0].p, s->src[1].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(s->bufM[0].p, s->src[2].p, (size_t)s->N * sizeof(F), cudaMemcpyDeviceToDevice, st));
    CK(cudaEventRecord(s->ev[0], st));
    sumcheck_fused_async(s, r);
    CK(cudaEventRecord(s->ev[1], st));
    CK(cudaMemcpyAsync(out, s->d_out.p, ((size_t)3 * n + 3) * sizeof(F), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float tot = 0;
    CK(cudaEventElapsedTime(&tot, s->ev[0], s->ev[1]));
    if (device_ms) *device_ms = tot;
    return VP_OK;
    API_END
}
// profiling aid: %globaltimer stamps (ns) of block 0 at {pass start, work done, barrier passed, pass end} of the last fused run
extern "C" int vp_sumcheck_pass_stamps(vp_sumcheck* s, unsigned long long* out, int n) {
    if (!s || !out) return fail(VP_ERR_ARG, "null argument");
    API_BEGIN
    cudaSetDevice(s->device);
    CK(cudaMemcpy(out, s->d_dbg.p, (size_t)std::min(n, 256 + 2048) * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return VP_OK;
    API_END
}
extern "C" int vp_sumcheck_round_ms(vp_sumcheck* s, float* out) {
    if (!s || !out) return fail(VP_ERR_ARG, "null argument");
    std::copy(s->round_ms.begin(), s->round_ms.end(), out);
    return VP_OK;
}
extern "C" void vp_sumcheck_destroy(vp_sumcheck* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    delete s;
}

// ------------------------------------------------------------------ the polynomial commitment's inner GKR (SURVEY 8(f) N4)
#include "fft_gkr.cuh"
extern "C" size_t vp_fft_gkr_rnd_count(int lg_size) { return (lg_size < 1 || lg_size > 24) ? 0 : fg::rnd_count(lg_size); }
extern "C" size_t vp_fft_gkr_poly_count(int lg_size) { return (lg_size < 1 || lg_size > 24) ? 0 : fg::poly_count(lg_size); }
extern "C" void vp_fft_gkr_release(void) { fg::release_cache(); }
// fft_circuit_gkr::fft_gkr (lib/virgo/src/fft_circuit_GKR.cpp:833-849) with the randomness handed in
extern "C" int vp_fft_gkr(int device, int lg_size, const vp_F* rnd, size_t n_rnd, vp_F* layers, vp_F* polys, size_t polys_cap, vp_F* claims,
                          int* proof_size, int* ok, double* verifier_seconds, double* prover_seconds, float* device_ms) {
    if (!rnd || !proof_size || !ok) return fail(VP_ERR_ARG, "null argument");
    if (lg_size < 1 || lg_size > 24) return fail(VP_ERR_ARG, "vp_fft_gkr: lg_size must be in [1, 24]");
    if (n_rnd < fg::rnd_count(lg_size)) return fail(VP_ERR_ARG, "vp_fft_gkr: %zu random elements given, %zu needed", n_rnd, fg::rnd_count(lg_size));
    if (polys && polys_cap < fg::poly_count(lg_size)) return fail(VP_ERR_ARG, "vp_fft_gkr: polynomial buffer too small (%zu < %zu)", polys_cap, fg::poly_count(lg_size));
    for (size_t i = 0; i < fg::rnd_count(lg_size); ++i)
        if (rnd[i].re >= P || rnd[i].im >= P) return fail(VP_ERR_ARG, "vp_fft_gkr: random element %zu is not canonical", i);
    API_BEGIN
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        throw CudaError{std::string("no CUDA device available (there is no CPU fallback): ") + cudaGetErrorString(ce)};
    const fg::Result r = fg::run(device, lg_size, reinterpret_cast<const F*>(rnd), reinterpret_cast<F*>(layers), reinterpret_cast<F*>(polys),
                                 reinterpret_cast<F*>(claims));
    *proof_size = r.proof_size;
    *ok = r.ok;
    if (verifier_seconds) *verifier_seconds = r.verifier_seconds;
    if (prover_seconds) *prover_seconds = r.prover_seconds;
    if (device_ms) *device_ms = r.device_ms;
    return VP_OK;
    API_END
}
