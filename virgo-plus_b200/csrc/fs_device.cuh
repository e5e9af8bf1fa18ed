// Fiat-Shamir mode on the device (DESIGN.md section 7): the transcript cache of host/fiat_shamir.h (FsCache, the reference's
// transcriptCache) restated as a small device buffer, so that a whole Fiat-Shamir proof is queued on one stream without a
// host round trip per round.
//
// Pool layout (FS_POOL words): pool[0] = number of message words held, pool[1 ..] = the bytes of FsCache::pool as
// little-endian words. Everything FsCache stores is a whole number of words (the 32-byte seed / digest, 16-byte field
// elements), so the pool is a word array. Only one thread at a time touches it: the kernels below run in stream order and
// inside k_sumcheck_phase_fs only thread 0 of block 0 does.
// A batch of B statements (vp_prove_fs_bound_batch) gives every statement its own pool, transcript and challenges, `ss`
// bytes apart (kernels.cuh, stmt_at); statement b runs in blockIdx.z == b: one warp per statement in the kernels between
// phases, one row of blocks per statement in the phase kernel.
#pragma once
#include "../host/fiat_shamir.h"   // FsStep
#include "kernels.cuh"
#include "keccak.cuh"

namespace vp {

// store(x): 16 bytes {re, im}
VP_D void fs_store(uint64_t* pool, const F& x) {
    const uint64_t n = pool[0];
    pool[1 + n] = x.re;
    pool[2 + n] = x.im;
    pool[0] = n + 2;
}
// random(): hash the pool, the digest becomes the pool, the challenge is the first two digest words mod p
VP_D F fs_draw(uint64_t* pool) {
    uint64_t d[4];
    sha3_256_words(pool + 1, (uint32_t)pool[0], d);
#pragma unroll
    for (int k = 0; k < 4; ++k) pool[1 + k] = d[k];
    pool[0] = 4;
    return F{fp_mod(d[0]), fp_mod(d[1])};
}

// One warp, lane 0 hashes: store transcript[tr_begin .. + n_store), then draw chal[ci_begin .. + n_draw).
VP_D void fs_absorb_draw_warp(uint64_t* pool, const F* transcript, uint32_t tr_begin, uint32_t n_store, F* chal, uint32_t ci_begin,
                              uint32_t n_draw) {
    const uint64_t n0 = pool[0];
    __syncwarp();
    for (uint32_t k = threadIdx.x; k < n_store; k += 32) {
        const F x = transcript[tr_begin + k];
        pool[1 + n0 + 2 * k] = x.re;
        pool[2 + n0 + 2 * k] = x.im;
    }
    __syncwarp();
    if (threadIdx.x == 0) {
        pool[0] = n0 + 2ull * n_store;
        for (uint32_t k = 0; k < n_draw; ++k) st_f(chal + ci_begin + k, fs_draw(pool));
    }
    __syncwarp();   // (the next call's lanes read pool[0])
}

// Between phases (host/fiat_shamir.h: Vres / claim_u / claims_v / claim_liu, then r_out / assert_random / sig).
__global__ void k_fs_absorb_draw(uint64_t* pool, const F* __restrict__ transcript, uint32_t tr_begin, uint32_t n_store, F* chal,
                                 uint32_t ci_begin, uint32_t n_draw, size_t ss) {
    fs_absorb_draw_warp(stmt_at(pool, ss), stmt_at(transcript, ss), tr_begin, n_store, stmt_at(chal, ss), ci_begin, n_draw);
}

// The verifier's side (vp_verify_fs_bound_batch): every challenge of a transcript recomputed from its messages, in the
// store / draw order of host/fiat_shamir.h (fs_schedule). The order is a table of steps built once per context: one per
// sumcheck round (store the 3 coefficients, draw the round's challenge) and one per store / draw run between phases.
// One warp per statement (blockIdx.z), lane 0 hashes; the pool must hold the statement (k_fs_statement).
__global__ void k_fs_replay(const FsStep* __restrict__ steps, uint32_t n_steps, uint64_t* pool, const F* __restrict__ transcript, F* chal,
                            size_t ss) {
    pool = stmt_at(pool, ss); transcript = stmt_at(transcript, ss); chal = stmt_at(chal, ss);
    for (uint32_t s = 0; s < n_steps; ++s) {
        const FsStep st = steps[s];
        fs_absorb_draw_warp(pool, transcript, st.tr_begin, st.n_store, chal, st.ci_begin, st.n_draw);
    }
}

// The statement (include/virgo_b200.h): H("VPSTMT01" | circuit | u64 n_inputs | inputs root | u64 n_outputs | outputs root |
// context[32]), 152 bytes. circuit: its digest (4 words, shared by a batch); roots = {-, inputs, outputs} digests, 4 words
// each. The context is `ctx`, or ctxs[4b ..] for statement b when ctxs is not null. Seeds the pool with the statement and
// copies it to `out` (4 words).
struct FsContext { uint64_t w[4]; };
VP_D void fs_statement_digest(const uint64_t* circuit, const uint64_t* in_root, const uint64_t* out_root, uint64_t n_inputs,
                              uint64_t n_outputs, const uint64_t (&ctx)[4], uint64_t (&d)[4]) {
    uint64_t m[19];
    m[0] = 0x3130544d54535056ull;   // "VPSTMT01"
#pragma unroll
    for (int k = 0; k < 4; ++k) { m[1 + k] = circuit[k]; m[6 + k] = in_root[k]; m[11 + k] = out_root[k]; m[15 + k] = ctx[k]; }
    m[5] = n_inputs;
    m[10] = n_outputs;
    sha3_256_words(m, 19, d);
}
__global__ void k_fs_statement(const uint64_t* __restrict__ circuit, const uint64_t* __restrict__ roots, uint64_t n_inputs,
                               uint64_t n_outputs, FsContext ctx, const uint64_t* __restrict__ ctxs, uint64_t* pool, uint64_t* out,
                               size_t ss) {
    if (threadIdx.x != 0) return;
    roots = stmt_at(roots, ss); pool = stmt_at(pool, ss); out = stmt_at(out, ss);
    if (ctxs) {
#pragma unroll
        for (int k = 0; k < 4; ++k) ctx.w[k] = ctxs[4 * (size_t)blockIdx.z + k];
    }
    uint64_t d[4];
    fs_statement_digest(circuit, roots + 4, roots + 8, n_inputs, n_outputs, ctx.w, d);
#pragma unroll
    for (int k = 0; k < 4; ++k) { pool[1 + k] = d[k]; out[k] = d[k]; }
    pool[0] = 4;
}

// The statements of an aggregate proof (vp_prove_fs_aggregate), one thread per statement: statement b from in_roots[4b ..],
// out_roots[4b ..] and ctxs[4b ..] (the roots of its slices, its context) to out[4b ..]. The circuit digest is that of
// template + K, shared by all B.
__global__ void k_fs_statements(const uint64_t* __restrict__ circuit, const uint64_t* __restrict__ in_roots,
                                const uint64_t* __restrict__ out_roots, const uint64_t* __restrict__ ctxs, uint64_t n_inputs,
                                uint64_t n_outputs, uint32_t B, uint64_t* out) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    uint64_t c[4], d[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = ctxs[4 * (size_t)b + k];
    fs_statement_digest(circuit, in_roots + 4 * (size_t)b, out_roots + 4 * (size_t)b, n_inputs, n_outputs, c, d);
#pragma unroll
    for (int k = 0; k < 4; ++k) out[4 * (size_t)b + k] = d[k];
}

// The aggregate H("VPAGGR01" | u64 B | root), root = R over the B statements (48 bytes hashed). Seeds the pool with it, as
// k_fs_statement does with a statement, and copies it to `out` (4 words).
__global__ void k_fs_aggregate(const uint64_t* __restrict__ root, uint64_t B, uint64_t* pool, uint64_t* out) {
    if (threadIdx.x != 0) return;
    uint64_t m[6], d[4];
    m[0] = 0x3130524747415056ull;   // "VPAGGR01"
    m[1] = B;
#pragma unroll
    for (int k = 0; k < 4; ++k) m[2 + k] = root[k];
    sha3_256_words(m, 6, d);
#pragma unroll
    for (int k = 0; k < 4; ++k) { pool[1 + k] = d[k]; out[k] = d[k]; }
    pool[0] = 4;
}

// ------------------------------------------------------------------ K6f: a Fiat-Shamir sumcheck phase in ONE launch
// All rounds of one phase (phase 1, phase 2 or Liu of one layer; the plan is PhaseArgs, kernels.cuh), with the challenges
// drawn inside. A cooperative grid walks the rounds; blocks meet at a grid barrier once per round (the round's tables are
// written by all blocks and read by all blocks in the next round). After round j's barrier block 0 reduces the per-block
// partials, writes (a, b, c) to the transcript, stores them in the pool and draws the round's challenge into chal[j - 1];
// a second grid barrier then releases the other blocks into round j + 1's fold, which needs that challenge. Block 0 keeps
// add_term in a register. Once a round's work fits one block, block 0 runs the remaining rounds alone, storing and drawing
// the same way behind block barriers, and writes the final claims; storing them is the next k_fs_absorb_draw's job.
// stamps (4 per round, block 0, %globaltimer): round start, own fold work done, polynomial reduced (grid rounds: after the
// barrier), challenge drawn. The next round's start minus "drawn" is the release barrier.
// A batch runs a gridDim.x x B grid: row blockIdx.z is statement b, its block x == 0 reduces the row's partials and draws
// the statement's challenge, and one grid barrier serves all rows. Stamps are those of row 0.
struct FsPhaseArgs {
    uint64_t* pool;
    F* chal;                     // chal[j - 1]: the challenge drawn after round j
    unsigned long long* stamps;  // 4 * n_rounds, may be null
    size_t ss;                   // bytes between two statements' working sets (0: one statement)
};
VP_D void fs_stamp(unsigned long long* s, uint32_t j, int k) {
    if (!s) return;
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    s[4 * (j - 1) + k] = t;
}

// Round j of k_sumcheck_phase_fs on threads t, t + stride, ... (t == 0: thread 0 of block 0): fold the round's tables
// with the previous challenge and sum them into v. reduce(v, collapse) makes v the round's sums and calls collapse() on
// thread 0 of block 0 (the tables that collapse in this round join add_term); it returns true on that thread alone, which
// then writes the round polynomial, stores it in the pool and draws the round's challenge.
template <class Reduce>
VP_D void fs_round(const PhaseArgs& p, const RoundDev& R, uint32_t j, uint32_t t, uint32_t stride, size_t ss, uint32_t* s_wend,
                   uint64_t* pool, F* chal, F* claims, F& at, unsigned long long* stamps, Reduce reduce) {
    if (t == 0) fs_stamp(stamps, j, 0);
    __syncthreads();   // (tail rounds: also publishes the previous round's challenge to the block)
    for (uint32_t i = threadIdx.x; i < R.n_tabs; i += blockDim.x) s_wend[i] = p.tabs[R.tab_begin + i].work_end;
    __syncthreads();
    const uint32_t ib = R.in_buf, ob = ib ^ 1;
    const bool fold = j >= 2;
    const F prev = fold ? ld_f_cg(chal + j - 2) : f_zero();   // drawn by block 0 in this launch: bypass L1
    const FoldK rk = make_foldk(prev);
    F* const inV = stmt_at(p.bufV[ib], ss);
    F* const inM = stmt_at(p.bufM[ib], ss);
    F* const inA = stmt_at(p.bufA[ib], ss);
    RoundAcc acc;
    racc_init(acc);
    if (fold) round_work<true, false>(acc, p.tabs + R.tab_begin, R.n_tabs, s_wend, inV, inM, inA, stmt_at(p.bufV[ob], ss),
                                      stmt_at(p.bufM[ob], ss), stmt_at(p.bufA[ob], ss), rk, t, stride);
    else round_work<false, false>(acc, p.tabs + R.tab_begin, R.n_tabs, s_wend, inV, inM, inA, stmt_at(p.bufV[ob], ss),
                                  stmt_at(p.bufM[ob], ss), stmt_at(p.bufA[ob], ss), rk, t, stride);
    F v[3];
    racc_finish(acc, v);
    const auto collapse = [&] {
        at = collapse_update<false>(at, p.cols + R.col_begin, R.n_cols, inV, inM, inA, fold, /*scale=*/fold, prev, rk, claims);
    };
    if (!reduce(v, collapse)) return;
    const F o[3] = {v[0], f_sub(v[1], at), f_add(v[2], at)};
    F* out = stmt_at(p.out_poly, ss) + 3 * (j - 1);
    fs_stamp(stamps, j, 2);
    for (int k = 0; k < 3; ++k) { st_f(out + k, o[k]); fs_store(pool, o[k]); }
    st_f(chal + j - 1, fs_draw(pool));
    fs_stamp(stamps, j, 3);
}

__global__ void __launch_bounds__(256, 2) k_sumcheck_phase_fs(PhaseArgs p, FsPhaseArgs f) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ F smem[3 * 32];
    __shared__ uint32_t s_wend[128];
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gstride = gridDim.x * blockDim.x;
    const size_t ss = f.ss;
    uint64_t* const pool = stmt_at(f.pool, ss);
    F* const chal = stmt_at(f.chal, ss);
    F* const claims = stmt_at(p.claims, ss);
    unsigned long long* const stamps = blockIdx.z == 0 ? f.stamps : nullptr;
    const bool stamp = blockIdx.x == 0 && threadIdx.x == 0;
    F at = p.at_init ? *stmt_at(p.at_init, ss) : f_zero();  // add_term: meaningful in block 0 / thread 0 only
    uint32_t j = 1;
    // ---- grid rounds
    for (; j <= p.n_rounds; ++j) {
        const RoundDev R = p.rounds[j - 1];
        if (R.work <= p.tail_work) break;
        F* part = stmt_at(p.partials, ss) + (size_t)(j & 1) * gridDim.x * 3;
        fs_round(p, R, j, gtid, gstride, ss, s_wend, pool, chal, claims, at, stamps, [&](F (&v)[3], auto collapse) {
            block_sum<3>(v, smem);
            if (threadIdx.x == 0) {
                st_f(part + (size_t)blockIdx.x * 3 + 0, v[0]);
                st_f(part + (size_t)blockIdx.x * 3 + 1, v[1]);
                st_f(part + (size_t)blockIdx.x * 3 + 2, v[2]);
                // tables collapsing in this round are inputs of this round: read them before the barrier, the next
                // round may overwrite that buffer
                if (blockIdx.x == 0) collapse();
            }
            if (stamp) fs_stamp(stamps, j, 1);
            grid.sync();
            if (blockIdx.x != 0) return false;
            v[0] = v[1] = v[2] = f_zero();
            for (uint32_t b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
                v[0] = f_add(v[0], ld_one<false>(part + (size_t)b * 3 + 0));
                v[1] = f_add(v[1], ld_one<false>(part + (size_t)b * 3 + 1));
                v[2] = f_add(v[2], ld_one<false>(part + (size_t)b * 3 + 2));
            }
            block_sum<3>(v, smem);
            return threadIdx.x == 0;
        });
        grid.sync();   // release: round j + 1 folds with the challenge just drawn
    }
    if (blockIdx.x != 0) return;
    // ---- tail rounds: block 0 alone
    for (; j <= p.n_rounds; ++j) {
        const RoundDev R = p.rounds[j - 1];
        fs_round(p, R, j, threadIdx.x, blockDim.x, ss, s_wend, pool, chal, claims, at, stamps, [&](F (&v)[3], auto collapse) {
            if (stamp) fs_stamp(stamps, j, 1);
            block_sum<3>(v, smem);
            if (threadIdx.x != 0) return false;
            collapse();
            return true;
        });
    }
    __syncthreads();  // the last round's table writes, the claims of collapsed tables and the last challenge
    if (threadIdx.x == 0) st_f(stmt_at(p.add_term, ss), at);
    // ---- final claims (prover.cpp:494-521)
    const F* V = stmt_at(p.bufV[p.fin_buf], ss);
    F* const transcript = stmt_at(p.transcript, ss);
    for (uint32_t i = threadIdx.x; i < p.n_fin; i += blockDim.x) {
        const FinDesc fd = p.fins[i];
        F c;
        if (fd.from_claim >= 0) c = ld_one<false>(claims + fd.from_claim);
        else {
            const F v0 = fd.n_vals >= 1 ? ld_one<false>(V + fd.in_off) : f_zero();
            if (p.n_rounds >= 1) {
                const F v1 = fd.n_vals >= 2 ? ld_one<false>(V + fd.in_off + 1) : f_zero();
                c = f_fold(v0, v1, ld_f_cg(chal + p.n_rounds - 1));
            } else c = v0;
        }
        st_f(transcript + fd.out_idx, c);
        if (p.keep && i == 0) st_f(stmt_at(p.keep, ss), c);
    }
}

// ------------------------------------------------------------------ batches in device memory (vp_*_fs_bound_batch_dev)
// A statement that fails is reported in status[b] (one int32 per statement) and must not change any other statement's
// results, so nothing non-canonical it holds reaches the arithmetic.
VP_D bool f_canonical(const F& x) { return x.re < P && x.im < P; }

// One block per statement (blockIdx.z == b): statement b's inputs (and, in the verifier, its claimed outputs) from the
// caller's packed arrays into the batch's buffers -- as zeros when one of them is not canonical -- and its transcript,
// already in its working set (tr, ss bytes per statement; may be null), zeroed when one of its elements is not canonical.
// status[b] = io_code (prover 1, verifier 9) for an input or output, else 7 for a transcript element, else 0.
__global__ void k_batch_screen(const uint64_t* __restrict__ in_src, uint64_t* __restrict__ in_dst, uint32_t n_in,
                               const F* __restrict__ out_src, F* __restrict__ out_dst, uint32_t n_out, F* tr, uint32_t n_tr,
                               size_t ss, int32_t io_code, int32_t* __restrict__ status) {
    const size_t b = blockIdx.z;
    in_src += b * n_in;
    in_dst += b * n_in;
    if (out_src) { out_src += b * n_out; out_dst += b * n_out; }
    if (tr) tr = stmt_at(tr, ss);
    int bad_io = 0, bad_tr = 0;
    for (uint32_t i = threadIdx.x; i < n_in; i += blockDim.x) bad_io |= in_src[i] >= P;
    if (out_src)
        for (uint32_t i = threadIdx.x; i < n_out; i += blockDim.x) bad_io |= !f_canonical(ld_f(out_src + i));
    if (tr)
        for (uint32_t i = threadIdx.x; i < n_tr; i += blockDim.x) bad_tr |= !f_canonical(tr[i]);
    bad_io = __syncthreads_or(bad_io);
    bad_tr = __syncthreads_or(bad_tr);
    for (uint32_t i = threadIdx.x; i < n_in; i += blockDim.x) in_dst[i] = bad_io ? 0 : in_src[i];
    if (out_src)
        for (uint32_t i = threadIdx.x; i < n_out; i += blockDim.x) st_f(out_dst + i, bad_io ? f_zero() : ld_f(out_src + i));
    if (bad_tr)
        for (uint32_t i = threadIdx.x; i < n_tr; i += blockDim.x) st_f(tr + i, f_zero());
    if (threadIdx.x == 0) status[b] = bad_io ? io_code : bad_tr ? 7 : 0;
}

// The prover's assert flags (statement b's copy of d_counter[1], ss bytes apart: 1 + the layer of a non-zero is_assert
// gate, k_eval_layer) as statuses 2 + layer, one thread per statement; a status already set stays.
__global__ void k_batch_assert_status(const unsigned int* __restrict__ flag, size_t ss, uint32_t B, int32_t* __restrict__ status) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const unsigned int f = *reinterpret_cast<const unsigned int*>(reinterpret_cast<uintptr_t>(flag) + (size_t)b * ss);
    if (status[b] == 0 && f) status[b] = (int32_t)f + 1;
}

// One block per statement (blockIdx.z == b): when status[b] != 0, zero its row of each packed array (null: none).
__global__ void k_batch_zero_failed(const int32_t* __restrict__ status, F* a, uint32_t na, F* c, uint32_t nc, F* o, uint32_t no,
                                    uint64_t* w, uint32_t nw) {
    const size_t b = blockIdx.z;
    if (!status[b]) return;
    if (a) for (uint32_t i = threadIdx.x; i < na; i += blockDim.x) st_f(a + b * na + i, f_zero());
    if (c) for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) st_f(c + b * nc + i, f_zero());
    if (o) for (uint32_t i = threadIdx.x; i < no; i += blockDim.x) st_f(o + b * no + i, f_zero());
    if (w) for (uint32_t i = threadIdx.x; i < nw; i += blockDim.x) w[b * nw + i] = 0;
}

// The verifier's claim chain (Engine::verify_check, verifier.cpp:134-337) on the device. Per layer: its rounds, where its
// messages and challenges sit, where its sums sit among the statement's vf_out_total sums and its bucket keys (keys[key_begin
// .. + n_keys): 0 Copy, 1 Not, 2 Addc, 3 Mulc, 4 + 7 l + binary type index).
struct VfLayerDesc {
    int32_t pb, m;
    uint32_t tr_p1, tr_claim_u, tr_p2, tr_claims_v, tr_liu, tr_claim_liu;
    uint32_t ci_ru, ci_rv, ci_sig, ci_rliu;
    uint32_t vf_out, key_begin, n_keys, n_vf_liu;
};
struct VfCheckArgs {
    const VfLayerDesc* layers;   // by layer id; entry 0 is unused
    const uint32_t* keys;
    int32_t n;
    uint32_t tr_vres, tr_input, out_total;
};
// claims_v[j][l] of verify_check: layer j's claims on layers l < j, zero when layer j has no phase 2
VP_D F vf_claim_v(const VfCheckArgs& a, const F* tr, int j, int l) {
    const VfLayerDesc& J = a.layers[j];
    return J.m != -1 ? tr[J.tr_claims_v + l] : f_zero();
}
// 0 (accept) or verify_check's fail code, with its layer in *fail_layer; canonical field routines only (as k_verify_sums)
VP_D int vf_chain(const VfCheckArgs& a, const F* tr, const F* out, const F* chal, int* fail_layer) {
    auto ev = [](const F* q, const F& x) { return f_mul_add(f_mul_add(q[0], x, q[1]), x, q[2]); };   // a x^2 + b x + c
    auto ok_sum = [](const F* q, const F& claim) { return f_eq(f_add(q[2], f_add(f_add(q[0], q[1]), q[2])), claim); };
    *fail_layer = 0;
    F prev = tr[a.tr_vres];
    for (int i = a.n - 1; i >= 1; --i) {
        const VfLayerDesc D = a.layers[i];
        *fail_layer = i;
        for (int j = 0; j < D.pb; ++j) {
            const F* q = tr + D.tr_p1 + 3 * j;
            if (!ok_sum(q, prev)) return 1;
            prev = ev(q, chal[D.ci_ru + j]);
        }
        const F claim_u = tr[D.tr_claim_u];
        F bv0 = f_one();
        for (int j = 0; j < D.m; ++j) {   // (m == -1: no phase 2)
            const F* q = tr + D.tr_p2 + 3 * j;
            if (!ok_sum(q, prev)) return 2;
            const F r = chal[D.ci_rv + j];
            prev = ev(q, r);
            bv0 = f_mul(bv0, f_sub(f_one(), r));
        }
        // getFinalValue (verifier.cpp:115-132) from the bucket sums
        F cl[4] = {f_zero(), f_zero(), f_zero(), f_zero()}, bias = f_zero();
        const F* o = out + D.vf_out;
        for (uint32_t b = 0; b < D.n_keys; ++b) {
            const uint32_t key = a.keys[D.key_begin + b];
            if (key < 4) {
                cl[key] = o[2 * b];
                if (key == 2) bias = o[2 * b + 1];
            }
        }
        if (D.m != -1) {
            for (int k = 0; k < 4; ++k) cl[k] = f_mul(cl[k], bv0);
            bias = f_mul(bias, bv0);
        }
        F res = f_mul(cl[1], f_sub(f_one(), claim_u));
        res = f_add(res, f_mul(cl[0], claim_u));
        res = f_add(f_add(res, f_mul(cl[2], claim_u)), bias);
        res = f_add(res, f_mul(cl[3], claim_u));
        if (D.m != -1)
            for (uint32_t b = 0; b < D.n_keys; ++b) {
                const uint32_t key = a.keys[D.key_begin + b];
                if (key < 4) continue;
                const int l = (int)((key - 4) / 7), bi = (int)((key - 4) % 7);
                const F cu = claim_u, cv = tr[D.tr_claims_v + l], uv = f_mul(cu, cv);
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
        if (!f_eq(prev, res)) return 3;
        // verifyLiu (an EMPTY subset's claim counts as well, as in verify_check)
        const int pre = i - 1;
        const F* sig = chal + D.ci_sig;
        prev = f_mul(sig[0], claim_u);
        for (int j = i; j < a.n; ++j) prev = f_add(prev, f_mul(sig[j - pre], vf_claim_v(a, tr, j, pre)));
        for (int j = 0; j < D.pb; ++j) {
            const F* q = tr + D.tr_liu + 3 * j;
            if (!ok_sum(q, prev)) return 4;
            prev = ev(q, chal[D.ci_rliu + j]);
        }
        const F vr = tr[D.tr_claim_liu];
        F gr = f_zero();
        for (uint32_t sg = 0; sg < D.n_vf_liu; ++sg) gr = f_add(gr, o[2 * (D.n_keys + sg)]);
        if (!f_eq(f_mul(vr, gr), prev)) return 5;
        prev = vr;
    }
    *fail_layer = 0;
    const F acc = out[a.out_total - 2], claimed = tr[a.tr_input];
    if (!f_eq(claimed, acc) || !f_eq(prev, claimed)) return 6;
    return 0;
}
// One thread per statement: its verdict from its screening status (7 or 9), else code 8 when Vres is not the claimed
// outputs' MLE at r_out (the statement's last sum), else the claim chain. tr / chal / sums: statement 0's, ss bytes apart.
// code and layer may be null.
__global__ void k_verify_check(VfCheckArgs a, const F* __restrict__ tr, const F* __restrict__ chal, const F* __restrict__ sums,
                               size_t ss, uint32_t B, const int32_t* __restrict__ status, int32_t* accept, int32_t* code,
                               int32_t* layer) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const size_t d = (size_t)b * ss;
    tr = reinterpret_cast<const F*>(reinterpret_cast<uintptr_t>(tr) + d);
    chal = reinterpret_cast<const F*>(reinterpret_cast<uintptr_t>(chal) + d);
    sums = reinterpret_cast<const F*>(reinterpret_cast<uintptr_t>(sums) + d);
    int cd = status[b], ly = 0;
    if (!cd) {
        if (!f_eq(sums[a.out_total - 1], tr[a.tr_vres])) cd = 8;
        else cd = vf_chain(a, tr, sums, chal, &ly);
    }
    accept[b] = cd == 0;
    if (code) code[b] = cd;
    if (layer) layer[b] = ly;
}

}  // namespace vp
