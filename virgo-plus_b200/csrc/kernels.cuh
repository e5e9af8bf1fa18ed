// sm_100a kernels of the GKR sumcheck prover. One kernel per reference loop (SURVEY.md 2.1 K1-K9).
// All tables hold one F (16 B) per entry: the reference's linear_poly {a,b} (src/polynomial.h:35-46)
// is re-derived as a = T[2i+1]-T[2i], b = T[2i], so a table costs 16 B/entry instead of 32.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "field.cuh"

namespace vp {

// gate type codes: /root/reference/src/inputCircuit.hpp:14-16
enum : uint32_t { T_MUL = 0, T_ADD, T_SUB, T_ANTISUB, T_NAAB, T_ANTINAAB, T_INPUT, T_MULC, T_ADDC, T_XOR, T_NOT, T_COPY };
static constexpr uint32_t TY_ASSERT_BIT = 0x80;

// ------------------------------------------------------------------ loads / stores
VP_D F ld_f(const F* p) {
    ulonglong2 t = __ldg(reinterpret_cast<const ulonglong2*>(p));
    return F{t.x, t.y};
}
VP_D F ld_f_cg(const F* p) {  // bypass L1 (data written by other blocks of the same launch)
    ulonglong2 t = __ldcg(reinterpret_cast<const ulonglong2*>(p));
    return F{t.x, t.y};
}
VP_D void st_f(F* p, const F& v) { *reinterpret_cast<ulonglong2*>(p) = make_ulonglong2(v.re, v.im); }
// Two adjacent entries with one 256-bit access (sm_100: LDG.E.256 / STG.E.256); p must be 32-byte aligned.
// NC = read-only path (tables written by an EARLIER launch); !NC = coherent load (tables written earlier in
// the SAME launch by other blocks, ordered by a grid barrier).
template <bool NC>
VP_D void ld_pair(const F* p, F& a, F& b) {
    if (NC) asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a.re), "=l"(a.im), "=l"(b.re), "=l"(b.im) : "l"(p));
    else asm volatile("ld.global.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a.re), "=l"(a.im), "=l"(b.re), "=l"(b.im) : "l"(p) : "memory");
}
VP_D void st_pair(F* p, const F& a, const F& b) {
    asm volatile("st.global.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(a.re), "l"(a.im), "l"(b.re), "l"(b.im) : "memory");
}
template <bool NC>
VP_D F ld_one(const F* p) {
    if (NC) return ld_f(p);
    F r;
    asm volatile("ld.global.v2.u64 {%0,%1}, [%2];" : "=l"(r.re), "=l"(r.im) : "l"(p) : "memory");
    return r;
}

// eq(r, idx) = half_f[idx & mask] * half_s[idx >> fh]   (utils.cpp:41-42)
struct EqTab {
    const F* f;
    const F* s;
    uint32_t fh;
    uint32_t mask;
};
VP_D F eq_at(const EqTab& t, uint32_t idx) { return f_mul(ld_f(t.f + (idx & t.mask)), ld_f(t.s + (idx >> t.fh))); }

// ------------------------------------------------------------------ statements of a batch (vp_prove_fs_bound_batch)
// The Fiat-Shamir kernels run B independent statements of one circuit at once, statement b in blockIdx.z == b. Every
// per-statement buffer of statement b (tables, challenges, transcript, claims, scalars, eq tables, partial sums, pool)
// sits `ss` bytes after statement b - 1's: stmt_at shifts a statement-0 pointer to this block's statement. Layer values
// are instance-major over the B * K instances instead (statement b, instance k = global instance b * K + k). A single
// proof is the batch of one: blockIdx.z == 0, and every shift is zero.
template <class T>
VP_D T* stmt_at(T* p, size_t ss) { return reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(p) + (size_t)blockIdx.z * ss); }
VP_D EqTab stmt_at(EqTab t, size_t ss) { t.f = stmt_at(t.f, ss); t.s = stmt_at(t.s, ss); return t; }

// ------------------------------------------------------------------ sharding of a table over G GPUs
// A table is cut into blocks of 2^m consecutive entries and every rank holds a CONTIGUOUS run of blocks, i.e. the
// entries [lo, hi) (multiples of 2^m), stored from local index 0. Rounds 1..m of a sumcheck pair entries inside one
// block, so they need no communication. Contiguous runs keep the instances a rank touches contiguous as well
// (tables are instance-major), so a rank only evaluates its own slice of the data-parallel instances.
struct ShardMap {
    uint32_t lo, hi;
};
VP_HD bool shard_local(const ShardMap& s, uint32_t idx, uint32_t& local) {
    local = idx - s.lo;
    return idx >= s.lo && idx < s.hi;
}
VP_HD uint32_t shard_global(const ShardMap& s, uint32_t local) { return local + s.lo; }

// ------------------------------------------------------------------ reductions
VP_D F warp_sum(F x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        F y;
        y.re = __shfl_down_sync(0xffffffffu, x.re, off);
        y.im = __shfl_down_sync(0xffffffffu, x.im, off);
        x = f_add(x, y);
    }
    return x;
}

// Block-wide sum of NV field elements per thread; result valid in thread 0. smem: NV * 32 F.
template <int NV>
VP_D void block_sum(F (&v)[NV], F* smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
    __syncthreads();
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) smem[i * 32 + warp] = v[i];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            F x = lane < nwarp ? smem[i * 32 + lane] : f_zero();
            v[i] = warp_sum(x);
        }
    }
}

// Grid-wide: every block deposits NV partials; the last block to arrive sums them.
// Returns true in ALL threads of the last block; the total is valid in its thread 0.
template <int NV>
VP_D bool grid_sum(F (&v)[NV], F* smem, F* partials, unsigned int* counter) {
    __shared__ bool s_last;
    block_sum<NV>(v, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) st_f(partials + (size_t)blockIdx.x * NV + i, v[i]);
        __threadfence();
        unsigned int t = atomicAdd(counter, 1u);
        s_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return false;
    __threadfence();
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = f_zero();
    for (unsigned int b = threadIdx.x; b < gridDim.x; b += blockDim.x) {
#pragma unroll
        for (int i = 0; i < NV; ++i) v[i] = f_add(v[i], ld_f_cg(partials + (size_t)b * NV + i));
    }
    block_sum<NV>(v, smem);
    if (threadIdx.x == 0) *counter = 0;
    return true;
}

// ------------------------------------------------------------------ K2: eq half tables
// utils.cpp:8-27 initHalfTable. One block per half table.
struct EqBuild {
    uint32_t r_idx;      // index of the first challenge of this half in the challenge array
    uint32_t nbits;      // bits of this half
    int32_t scale_idx;   // challenge index of the `init` scalar, or -1 for F_ONE
    uint32_t out_off;    // offset (entries) into the eq scratch buffer
};

__global__ void __launch_bounds__(1024) k_eq_build(const EqBuild* __restrict__ descs, const F* __restrict__ chal,
                                                    F* __restrict__ eqbuf, size_t ss) {
    chal = stmt_at(chal, ss);
    eqbuf = stmt_at(eqbuf, ss);
    const EqBuild d = descs[blockIdx.x];
    F* T = eqbuf + d.out_off;
    if (threadIdx.x == 0) T[0] = d.scale_idx >= 0 ? chal[d.scale_idx] : f_one();
    __syncthreads();
    for (uint32_t i = 0; i < d.nbits; ++i) {
        const F r = chal[d.r_idx + i];
        const uint32_t n = 1u << i;
        for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
            F t0 = T[j];
            F tmp = f_mul(t0, r);
            T[j | n] = tmp;
            T[j] = f_sub(t0, tmp);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ K1: evaluate
// prover.cpp:30-36: layer 0 = F((long long) gate.u), i.e. x for 0 <= x, p + x for x < 0 (fieldElement.cpp:24-27).
// The reference keeps a non-negative x >= p as it is (a non-canonical element its arithmetic does not expect); here
// every input is reduced, so the limb arithmetic always sees canonical values.
__global__ void k_load_inputs(const uint64_t* __restrict__ in, F* __restrict__ val, uint32_t begin, uint32_t end) {
    uint32_t i = begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (i < end) {
        const u64 x = in[i];
        st_f(val + i, F{(long long)x < 0 ? fp_canon(fp_fold(x) + P - 8) : fp_canon(x), 0});   // 2^64 = 8 (mod p): x - 2^64 + p
    }
}

struct GateArrays {          // one template layer (one instance)
    const uint8_t* ty;       // low 7 bits gate type, bit 7 = is_assert
    const int16_t* l;
    const uint32_t* u;
    const uint32_t* v;
    const F* c;              // may be null
};

// prover.cpp:38-90. Thread per gate of the replicated layer: g = k*S + g0.
// vals[l] = device pointer of circuitValue[l]; sizes[l] = template size S_l. A batch of statements is evaluated as one
// replicated layer of B * K instances; a failed assert of instance k raises the flag of statement k / K (flags ss bytes apart).
__global__ void __launch_bounds__(256) k_eval_layer(GateArrays G, uint32_t S, uint32_t K, int layer,
                                                     F* const* __restrict__ vals, const uint32_t* __restrict__ sizes,
                                                     F* __restrict__ out, unsigned int* __restrict__ assert_fail,
                                                     uint32_t g_begin, uint32_t g_end, int real_only, size_t ss) {
    const uint32_t S_pre = sizes[layer - 1];
    const F* __restrict__ pre = vals[layer - 1];
    for (uint32_t g = g_begin + blockIdx.x * blockDim.x + threadIdx.x; g < g_end; g += gridDim.x * blockDim.x) {
        const uint32_t k = g / S, g0 = g - k * S;
        const uint32_t tyb = G.ty[g0], ty = tyb & 0x7f;
        const int l = G.l[g0];
        const F x = ld_f(pre + (size_t)k * S_pre + G.u[g0]);
        F y = f_zero();
        if (l >= 0) y = ld_f(vals[l] + (size_t)k * sizes[l] + G.v[g0]);
        F r;
        if (real_only) {   // base-field circuit (no complex constants): one 61-bit product instead of a complex one
            const u64 a = x.re, b = y.re;
            u64 o;
            switch (ty) {
                case T_ADD: o = fp_add(a, b); break;
                case T_SUB: o = fp_sub(a, b); break;
                case T_ANTISUB: o = fp_sub(b, a); break;
                case T_MUL: o = fp_mul(a, b); break;
                case T_NAAB: o = fp_sub(b, fp_mul(a, b)); break;
                case T_ANTINAAB: o = fp_sub(a, fp_mul(a, b)); break;
                case T_ADDC: o = fp_add(a, G.c[g0].re); break;
                case T_MULC: o = fp_mul(a, G.c[g0].re); break;
                case T_COPY: o = a; break;
                case T_NOT: o = fp_sub(1, a); break;
                case T_XOR: { const u64 ab = fp_mul(a, b); o = fp_sub(fp_add(a, b), fp_add(ab, ab)); break; }
                default: o = 0; break;
            }
            r = F{o, 0};
        } else
        switch (ty) {
            case T_ADD: r = f_add(x, y); break;
            case T_SUB: r = f_sub(x, y); break;
            case T_ANTISUB: r = f_sub(y, x); break;
            case T_MUL: r = f_mul(x, y); break;
            case T_NAAB: r = f_sub(y, f_mul(x, y)); break;
            case T_ANTINAAB: r = f_sub(x, f_mul(x, y)); break;
            case T_ADDC: r = f_add(x, G.c[g0]); break;
            case T_MULC: r = f_mul(x, G.c[g0]); break;
            case T_COPY: r = x; break;
            case T_NOT: r = f_sub(f_one(), x); break;
            case T_XOR: r = f_sub(f_add(x, y), f_dbl(f_mul(x, y))); break;
            default: r = f_zero(); break;
        }
        st_f(out + g, r);
        if ((tyb & TY_ASSERT_BIT) && !f_is_zero(r))
            atomicExch(reinterpret_cast<unsigned int*>(reinterpret_cast<uintptr_t>(assert_fail) + (size_t)(k / K) * ss), 1u + (unsigned)layer);
    }
}

// ------------------------------------------------------------------ K3 / K4: table init from the wiring
// Both inits are "owner computes by output index": the gates that add into one table entry form a CSR
// row (sorted on the host), so no atomics are needed. Fan-in is heavily skewed (SHA256: mean 2-5, max
// 624), so rows are cut into work items of at most C entries: a row that fits one item is written
// directly, longer rows deposit per-item partial sums that a small second kernel combines.
struct RowItem {
    uint32_t row;        // row of the template (phase 1: u0; phase 2: lv0 within table `tab`)
    uint32_t e_begin;    // first CSR entry
    uint32_t cnt_slot;   // low 8 bits: number of entries; high 24 bits: partial slot + 1 (0 = direct write)
    uint32_t tab;        // phase 2: table id
};
struct LongRow {
    uint32_t row, slot_begin, slot_end, tab;
};

// prover.cpp:214-273
struct CsrP1 {
    const uint32_t* g0;    // template gate id (for the eq lookup and the constant)
    const uint32_t* v0;    // template v
    const uint32_t* tyl;   // ty | assert<<7 | (l+1)<<8
};

VP_D void p1_gate(uint32_t tyl, const F& beta, const F& Vv, const F* cst, uint32_t g0, F& M, F& A) {
    switch (tyl & 0x7f) {
        case T_ADD:
            A = f_mul_add(Vv, beta, A);
            M = f_add(M, beta);
            break;
        case T_SUB:
            A = f_sub(A, f_mul(Vv, beta));
            M = f_add(M, beta);
            break;
        case T_ANTISUB:
            A = f_mul_add(Vv, beta, A);
            M = f_sub(M, beta);
            break;
        case T_MUL:
            M = f_mul_add(Vv, beta, M);
            break;
        case T_NAAB: {
            const F t = f_mul(Vv, beta);
            A = f_add(A, t);
            M = f_sub(M, t);
            break;
        }
        case T_ANTINAAB:
            M = f_add(M, f_sub(beta, f_mul(Vv, beta)));
            break;
        case T_ADDC:
            A = f_mul_add(cst[g0], beta, A);
            M = f_add(M, beta);
            break;
        case T_MULC:
            M = f_mul_add(cst[g0], beta, M);
            break;
        case T_COPY:
            M = f_add(M, beta);
            break;
        case T_NOT:
            A = f_add(A, beta);
            M = f_sub(M, beta);
            break;
        case T_XOR: {
            const F t = f_mul(Vv, beta);
            A = f_add(A, t);
            M = f_add(M, f_sub(beta, f_dbl(t)));
            break;
        }
        default: break;
    }
}

__global__ void __launch_bounds__(256)
k_init_phase1(const RowItem* __restrict__ items, uint32_t n_items, CsrP1 csr, uint32_t S_pre, uint32_t S_cur, uint32_t K,
              EqTab eqg, const F* __restrict__ assert_r, F* const* __restrict__ vals, const uint32_t* __restrict__ sizes,
              const F* __restrict__ cst, const F* __restrict__ Vpre, F* __restrict__ tV, F* __restrict__ tM,
              F* __restrict__ tA, F* __restrict__ partial, uint32_t n_slots, ShardMap sm, int write_v, uint32_t k_begin,
              uint32_t k_end, size_t ss) {
    const size_t kz = (size_t)blockIdx.z * K;   // this statement's first global instance
    eqg = stmt_at(eqg, ss); assert_r = stmt_at(assert_r, ss);
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss); partial = stmt_at(partial, ss);
    Vpre += kz * S_pre;
    const uint64_t total = (uint64_t)n_items * (k_end - k_begin);
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t kq = (uint32_t)(w / n_items), it = (uint32_t)(w - (uint64_t)kq * n_items), k = k_begin + kq;
        const RowItem I = items[it];
        uint32_t loc;
        if (!shard_local(sm, k * S_pre + I.row, loc)) continue;   // another rank owns this table entry
        F M = f_zero(), A = f_zero();
        const uint32_t e1 = I.e_begin + (I.cnt_slot & 0xff);
        for (uint32_t e = I.e_begin; e < e1; ++e) {
            const uint32_t g0 = csr.g0[e], tyl = csr.tyl[e];
            const int l = (int)(tyl >> 8) - 1;
            F beta = eq_at(eqg, k * S_cur + g0);
            if (tyl & TY_ASSERT_BIT) beta = f_mul(beta, *assert_r);
            F Vv = f_zero();
            if (l >= 0) Vv = ld_f(vals[l] + (kz + k) * sizes[l] + csr.v0[e]);
            p1_gate(tyl, beta, Vv, cst, g0, M, A);
        }
        const uint32_t slot = I.cnt_slot >> 8;
        if (slot == 0) {
            if (write_v) st_f(tV + loc, ld_f(Vpre + k * S_pre + I.row));
            st_f(tM + loc, M);
            st_f(tA + loc, A);
        } else {
            F* dst = partial + 2 * ((size_t)k * n_slots + (slot - 1));
            st_f(dst, M);
            st_f(dst + 1, A);
        }
    }
}

// ---- phase-1 init when every circuit value is in the base field (no complex gate constants: all .pws circuits)
// Every contribution is +-beta, +-P or a small combination with P = beta * (a real scalar: the gathered operand or the
// constant) -- prover.cpp:229-272 with Vv real -- so a gate costs one eq product (kept weakly canonical), ONE
// real-scalar product (two limb chains per component) and a few additions into lazily folded sums; the gate type
// only selects the additions (no divergent heavy code). The kernel is bound
// by the latency of its dependent loads (CSR entry -> layer pointer -> gathered operand), so registers are kept low
// (lazy 96-bit sums were slower here: fewer resident warps) and the layer pointers / sizes sit in shared memory.
// Tried and dropped: one instance per lane (uniform control flow, but every lookup / gather / store of a warp then
// touches 32 different sectors and the eq half tables fall out of L1: 2.2x slower on SHA256_64 x 1024).
VP_D F eq_at_acc_w(const EqTab& t, uint32_t idx, const F& acc);
VP_D F f_mul_w(const F& a, const F& b);
VP_D F f_mul_add_w(const F& a, const F& b, const F& acc);
VP_D F eq_at_weak(const EqTab& t, uint32_t idx) { return eq_at_acc_w(t, idx, f_zero()); }   // components in [0,p]
VP_D F eq_at_acc_w(const EqTab& t, uint32_t idx, const F& acc) {   // acc + eq(idx), acc components < 2^64: [0,p]
    const F a = ld_f(t.f + (idx & t.mask)), b = ld_f(t.s + (idx >> t.fh));
    const LOp m = make_lop(a.re, a.im);
    const ROpD v = make_ropd(b);
    const u64 u_re = mad32(m.nim1, v.im1d, mad32(m.re1, v.re1d, mad32(m.nim0, v.im0, mul32(m.re0, v.re0))));
    const u64 t_re = mad32(m.nim1, v.im0, mad32(m.nim0, v.im1, mad32(m.re1, v.re0, mul32(m.re0, v.re1))));
    const u64 u_im = mad32(m.im1, v.re1d, mad32(m.re1, v.im1d, mad32(m.im0, v.re0, mul32(m.re0, v.im0))));
    const u64 t_im = mad32(m.im1, v.re0, mad32(m.im0, v.re1, mad32(m.re1, v.im0, mul32(m.re0, v.im1))));
    return F{fp_reduce_ut_weak(u_re, t_re, acc.re), fp_reduce_ut_weak(u_im, t_im, acc.im)};
}
__global__ void __launch_bounds__(256, 4)
k_init_phase1_real(const RowItem* __restrict__ items, uint32_t n_items, CsrP1 csr, uint32_t S_pre, uint32_t S_cur, uint32_t K,
                   EqTab eqg, const F* __restrict__ assert_r, F* const* __restrict__ vals, const uint32_t* __restrict__ sizes,
                   const F* __restrict__ cst, const F* __restrict__ Vpre, F* __restrict__ tV, F* __restrict__ tM,
                   F* __restrict__ tA, F* __restrict__ partial, uint32_t n_slots, ShardMap sm, int write_v, uint32_t k_begin,
                   uint32_t k_end, uint32_t n_src, size_t ss) {
    const size_t kz = (size_t)blockIdx.z * K;   // this statement's first global instance
    eqg = stmt_at(eqg, ss); assert_r = stmt_at(assert_r, ss);
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss); partial = stmt_at(partial, ss);
    Vpre += kz * S_pre;
    __shared__ const u64* s_vals[64];
    __shared__ uint32_t s_sizes[64];
    for (uint32_t i = threadIdx.x; i < min(n_src, 64u); i += blockDim.x) {
        s_vals[i] = reinterpret_cast<const u64*>(vals[i] + kz * sizes[i]);
        s_sizes[i] = sizes[i];
    }
    __syncthreads();
    const uint32_t total = n_items * (k_end - k_begin);   // < 2^32 (host check)
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < total; w += gridDim.x * blockDim.x) {
        const uint32_t kq = w / n_items, it = w - kq * n_items, k = k_begin + kq;
        const RowItem I = items[it];
        uint32_t loc;
        if (!shard_local(sm, k * S_pre + I.row, loc)) continue;   // another rank owns this table entry
        F M = f_zero(), A = f_zero();
        const uint32_t e1 = I.e_begin + (I.cnt_slot & 0xff);
        // two-deep software pipeline: while entry e is computed, the gathered operand and the two eq half-table entries
        // of entry e+1 are in flight and the CSR words of entry e+2 are being read
        struct Ent { uint32_t g0, tyl, v0; };
        struct Dat { u64 Vv; ulonglong2 ha, hb; };
        auto rd_csr = [&](uint32_t e) { return Ent{csr.g0[e], csr.tyl[e], csr.v0[e]}; };
        auto rd_dat = [&](const Ent& E) {
            Dat d;
            const int l = (int)(E.tyl >> 8) - 1;
            const uint32_t lc = l >= 0 ? (uint32_t)l : 0u;
            const u64* vp_ = s_vals[lc] + 2 * ((size_t)k * s_sizes[lc] + E.v0);
            asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(d.Vv) : "l"(vp_));   // real part of circuitValue[l][k * S_l + v0]
            const uint32_t idx = k * S_cur + E.g0;
            asm volatile("ld.global.nc.v2.u64 {%0,%1}, [%2];" : "=l"(d.ha.x), "=l"(d.ha.y) : "l"(eqg.f + (idx & eqg.mask)));
            asm volatile("ld.global.nc.v2.u64 {%0,%1}, [%2];" : "=l"(d.hb.x), "=l"(d.hb.y) : "l"(eqg.s + (idx >> eqg.fh)));
            return d;
        };
        Ent cur{0, 0, 0};
        Dat dc{0, {0, 0}, {0, 0}};
        if (I.e_begin < e1) { cur = rd_csr(I.e_begin); dc = rd_dat(cur); }   // a row without gates reads nothing
        Ent nxt = I.e_begin + 1 < e1 ? rd_csr(I.e_begin + 1) : cur;
        Dat dn = dc;
        for (uint32_t e = I.e_begin; e < e1; ++e) {
            if (e + 1 < e1) dn = rd_dat(nxt);
            const Ent nn = e + 2 < e1 ? rd_csr(e + 2) : nxt;
            const int l = (int)(cur.tyl >> 8) - 1;
            const uint32_t ty = cur.tyl & 0x7f, is_as = cur.tyl & TY_ASSERT_BIT, g0c = cur.g0;
            const u64 Vv = l < 0 ? 0 : dc.Vv;
            F beta = f_mul_w(F{dc.ha.x, dc.ha.y}, F{dc.hb.x, dc.hb.y});
            if (is_as) beta = f_mul(beta, *assert_r);
            cur = nxt; nxt = nn; dc = dn;
            // one product P = beta * x per gate (x = the gathered operand or the constant), the rest are additions of
            // beta, P and their negations into lazily folded sums (components stay below 2^63)
            const u64 x = (ty == T_ADDC || ty == T_MULC) ? cst[g0c].re : Vv;
            F Pp = f_zero();
            if (ty != T_COPY && ty != T_NOT) Pp = f_mad_real_w(f_zero(), beta, x);
            const F nP = F{P - Pp.re, P - Pp.im}, nB = F{P - beta.re, P - beta.im};
            switch (ty) {   // prover.cpp:229-272
                case T_ADD: case T_ADDC: A.re += Pp.re; A.im += Pp.im; M.re += beta.re; M.im += beta.im; break;
                case T_SUB: A.re += nP.re; A.im += nP.im; M.re += beta.re; M.im += beta.im; break;
                case T_ANTISUB: A.re += Pp.re; A.im += Pp.im; M.re += nB.re; M.im += nB.im; break;
                case T_MUL: case T_MULC: M.re += Pp.re; M.im += Pp.im; break;
                case T_NAAB: A.re += Pp.re; A.im += Pp.im; M.re += nP.re; M.im += nP.im; break;
                case T_ANTINAAB: M.re += beta.re + nP.re; M.im += beta.im + nP.im; break;
                case T_COPY: M.re += beta.re; M.im += beta.im; break;
                case T_NOT: A.re += beta.re; A.im += beta.im; M.re += nB.re; M.im += nB.im; break;
                case T_XOR: A.re += Pp.re; A.im += Pp.im; M.re += beta.re + 2 * nP.re; M.im += beta.im + 2 * nP.im; break;
                default: break;
            }
            A.re = fp_fold(A.re); A.im = fp_fold(A.im); M.re = fp_fold(M.re); M.im = fp_fold(M.im);   // <= p + 7
        }
        const F Mr = F{fp_canon(M.re), fp_canon(M.im)}, Ar = F{fp_canon(A.re), fp_canon(A.im)};
        const uint32_t slot = I.cnt_slot >> 8;
        if (slot == 0) {
            if (write_v) st_f(tV + loc, ld_f(Vpre + k * S_pre + I.row));
            st_f(tM + loc, Mr);
            st_f(tA + loc, Ar);
        } else {
            F* dst = partial + 2 * ((size_t)k * n_slots + (slot - 1));
            st_f(dst, Mr);
            st_f(dst + 1, Ar);
        }
    }
}

// Template-major form of k_init_phase1_real for K >= KC instances: a thread owns one work item
// of the TEMPLATE and a chunk of KC consecutive instances. The CSR words of an entry (gate id, type, source layer,
// operand index, constant) are read and decoded once for the KC instances, whose loads (gathered operand + two eq
// half-table entries each) are all address-computable at once and whose product chains are independent: 3 KC loads in
// flight per entry instead of a dependent CSR -> pointer -> operand chain per (entry, instance). Lanes of a warp hold
// neighbouring items of the same instances, so gathers and stores coalesce as before.
template <int KC>
__global__ void __launch_bounds__(256, 2)
k_init_phase1_real_tm(const RowItem* __restrict__ items, uint32_t n_items, CsrP1 csr, uint32_t S_pre, uint32_t S_cur, uint32_t K,
                      EqTab eqg, const F* __restrict__ assert_r, F* const* __restrict__ vals, const uint32_t* __restrict__ sizes,
                      const F* __restrict__ cst, const F* __restrict__ Vpre, F* __restrict__ tV, F* __restrict__ tM,
                      F* __restrict__ tA, F* __restrict__ partial, uint32_t n_slots, int write_v, uint32_t n_src, ShardMap sm,
                      uint32_t k_begin, uint32_t k_end, size_t ss) {
    const size_t kz = (size_t)blockIdx.z * K;   // this statement's first global instance
    eqg = stmt_at(eqg, ss); assert_r = stmt_at(assert_r, ss);
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss); partial = stmt_at(partial, ss);
    Vpre += kz * S_pre;
    __shared__ const u64* s_vals[64];
    __shared__ uint32_t s_sizes[64];
    for (uint32_t i = threadIdx.x; i < min(n_src, 64u); i += blockDim.x) {
        s_vals[i] = reinterpret_cast<const u64*>(vals[i] + kz * sizes[i]);
        s_sizes[i] = sizes[i];
    }
    __syncthreads();
    const uint32_t it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= n_items) return;
    const uint32_t k0 = k_begin + blockIdx.y * KC, nk = min((uint32_t)KC, k_end - k0);   // sharded: the rank's instance range
    const RowItem I = items[it];
    u64 Mre[KC], Mim[KC], Are[KC], Aim[KC];
#pragma unroll
    for (int j = 0; j < KC; ++j) { Mre[j] = Mim[j] = Are[j] = Aim[j] = 0; }
    const uint32_t e1 = I.e_begin + (I.cnt_slot & 0xff);
    for (uint32_t e = I.e_begin; e < e1; ++e) {
        const uint32_t g0 = csr.g0[e], tyl = csr.tyl[e], v0 = csr.v0[e];
        const int l = (int)(tyl >> 8) - 1;
        const uint32_t ty = tyl & 0x7f, lc = l >= 0 ? (uint32_t)l : 0u;
        const bool is_as = (tyl & TY_ASSERT_BIT) != 0, has_v = l >= 0, is_const = ty == T_ADDC || ty == T_MULC;
        const u64* vb = s_vals[lc] + 2 * (size_t)v0;
        const size_t vstride = 2 * (size_t)s_sizes[lc];
        const u64 xc = is_const ? cst[g0].re : 0;
        ulonglong2 ha[KC], hb[KC];
        u64 Vv[KC];
#pragma unroll
        for (int j = 0; j < KC; ++j) {
            const uint32_t k = k0 + (j < (int)nk ? j : 0), idx = k * S_cur + g0;
            ha[j] = __ldg(reinterpret_cast<const ulonglong2*>(eqg.f + (idx & eqg.mask)));
            hb[j] = __ldg(reinterpret_cast<const ulonglong2*>(eqg.s + (idx >> eqg.fh)));
            Vv[j] = has_v ? __ldg(vb + (size_t)k * vstride) : 0;
        }
#pragma unroll
        for (int j = 0; j < KC; ++j) {
            F beta = f_mul_w(F{ha[j].x, ha[j].y}, F{hb[j].x, hb[j].y});
            if (is_as) beta = f_mul(beta, *assert_r);
            const u64 x = is_const ? xc : Vv[j];
            F Pp = f_zero();
            if (ty != T_COPY && ty != T_NOT) Pp = f_mad_real_w(f_zero(), beta, x);
            const F nP = F{P - Pp.re, P - Pp.im}, nB = F{P - beta.re, P - beta.im};
            u64 are = 0, aim = 0, mre = 0, mim = 0;
            switch (ty) {   // prover.cpp:229-272 (same table as k_init_phase1_real)
                case T_ADD: case T_ADDC: are = Pp.re; aim = Pp.im; mre = beta.re; mim = beta.im; break;
                case T_SUB: are = nP.re; aim = nP.im; mre = beta.re; mim = beta.im; break;
                case T_ANTISUB: are = Pp.re; aim = Pp.im; mre = nB.re; mim = nB.im; break;
                case T_MUL: case T_MULC: mre = Pp.re; mim = Pp.im; break;
                case T_NAAB: are = Pp.re; aim = Pp.im; mre = nP.re; mim = nP.im; break;
                case T_ANTINAAB: mre = beta.re + nP.re; mim = beta.im + nP.im; break;
                case T_COPY: mre = beta.re; mim = beta.im; break;
                case T_NOT: are = beta.re; aim = beta.im; mre = nB.re; mim = nB.im; break;
                case T_XOR: are = Pp.re; aim = Pp.im; mre = beta.re + 2 * nP.re; mim = beta.im + 2 * nP.im; break;
                default: break;
            }
            Are[j] = fp_fold(Are[j] + are); Aim[j] = fp_fold(Aim[j] + aim);
            Mre[j] = fp_fold(Mre[j] + mre); Mim[j] = fp_fold(Mim[j] + mim);   // <= p + 7
        }
    }
    const uint32_t slot = I.cnt_slot >> 8;
#pragma unroll
    for (int j = 0; j < KC; ++j) {
        if (j >= (int)nk) break;
        const uint32_t k = k0 + j;
        const F Mr = F{fp_canon(Mre[j]), fp_canon(Mim[j])}, Ar = F{fp_canon(Are[j]), fp_canon(Aim[j])};
        uint32_t loc;
        if (!shard_local(sm, k * S_pre + I.row, loc)) continue;   // (sharded) another rank owns this table entry
        if (slot == 0) {
            if (write_v) st_f(tV + loc, ld_f(Vpre + k * S_pre + I.row));
            st_f(tM + loc, Mr);
            st_f(tA + loc, Ar);
        } else {
            F* dst = partial + 2 * ((size_t)k * n_slots + (slot - 1));
            st_f(dst, Mr);
            st_f(dst + 1, Ar);
        }
    }
}

__global__ void __launch_bounds__(256)
k_combine_phase1(const LongRow* __restrict__ rows, uint32_t n_rows, uint32_t S_pre, uint32_t K, const F* __restrict__ Vpre,
                 F* __restrict__ tV, F* __restrict__ tM, F* __restrict__ tA, const F* __restrict__ partial, uint32_t n_slots,
                 ShardMap sm, int write_v, uint32_t k_begin, uint32_t k_end, size_t ss) {
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss); partial = stmt_at(partial, ss);
    Vpre += (size_t)blockIdx.z * K * S_pre;
    const uint64_t total = (uint64_t)n_rows * (k_end - k_begin);
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t kq = (uint32_t)(w / n_rows), j = (uint32_t)(w - (uint64_t)kq * n_rows), k = k_begin + kq;
        const LongRow R = rows[j];
        const uint32_t u = k * S_pre + R.row;
        uint32_t loc;
        if (!shard_local(sm, u, loc)) continue;
        F M = f_zero(), A = f_zero();
        for (uint32_t s = R.slot_begin; s < R.slot_end; ++s) {
            const F* src = partial + 2 * ((size_t)k * n_slots + s);
            M = f_add(M, ld_f_cg(src));
            A = f_add(A, ld_f_cg(src + 1));
        }
        if (write_v) st_f(tV + loc, ld_f(Vpre + u));
        st_f(tM + loc, M);
        st_f(tA + loc, A);
    }
}

// prover.cpp:291-361. Output index = (table, lv); lv = (K-1-k)*D + lv0 (SURVEY 9.2.6).
// Per gate t = beta_g[g]*beta_u[u]; contributions are linear in t:  mult += cM[ty]*t, add += cA[ty]*t
// with cM/cA built from V_u (see make_p2_coef).
struct P2Table {
    const uint32_t* dadId;   // [D] template v of each subset slot
    uint32_t D;              // subset size of one instance
    uint32_t src_S;          // template size of the source layer
    uint32_t tab_off;        // offset of this table in the output buffers (entries)
    uint32_t owned;          // 0: this rank holds no part of the table
    const F* src_val;        // circuitValue[l]
    ShardMap sm;             // which entries of the table this rank holds, and where
};
struct CsrP2 {
    const uint32_t* g0;
    const uint32_t* u0;
    const uint8_t* ty;
};

VP_D void make_p2_coef(const F& Vu, F* cM, F* cA) {
    // prover.cpp:319-357, mult / add coefficient of tmp for each binary gate type
    const F one = f_one(), z = f_zero();
    for (int t = 0; t < 12; ++t) { cM[t] = z; cA[t] = z; }
    cM[T_ADD] = one;                          cA[T_ADD] = Vu;
    cM[T_SUB] = f_neg(one);                   cA[T_SUB] = Vu;
    cM[T_ANTISUB] = one;                      cA[T_ANTISUB] = f_neg(Vu);
    cM[T_MUL] = Vu;
    cM[T_NAAB] = f_sub(one, Vu);
    cM[T_ANTINAAB] = f_neg(Vu);               cA[T_ANTINAAB] = Vu;
    cM[T_XOR] = f_sub(one, f_dbl(Vu));        cA[T_XOR] = Vu;
}

__global__ void __launch_bounds__(256)
k_init_phase2(const RowItem* __restrict__ items, uint32_t n_items, const P2Table* __restrict__ tabs, CsrP2 csr,
              uint32_t S_pre, uint32_t S_cur, uint32_t K, EqTab eqg, EqTab equ, const F* __restrict__ assert_r,
              const F* __restrict__ Vu_ptr, F* __restrict__ tV, F* __restrict__ tM, F* __restrict__ tA,
              F* __restrict__ partial, uint32_t n_slots, uint32_t kk_begin, uint32_t kk_end, size_t ss) {
    const size_t kz = (size_t)blockIdx.z * K;   // this statement's first global instance
    eqg = stmt_at(eqg, ss); equ = stmt_at(equ, ss); assert_r = stmt_at(assert_r, ss); Vu_ptr = stmt_at(Vu_ptr, ss);
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss); partial = stmt_at(partial, ss);
    __shared__ F s_cM[12], s_cA[12];
    if (threadIdx.x == 0) make_p2_coef(*Vu_ptr, s_cM, s_cA);
    __syncthreads();
    const uint64_t total = (uint64_t)n_items * (kk_end - kk_begin);
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t kq = (uint32_t)(w / n_items), it = (uint32_t)(w - (uint64_t)kq * n_items), kk = kk_begin + kq, k = K - 1 - kk;
        const RowItem I = items[it];
        const P2Table T = tabs[I.tab];
        uint32_t loc;
        if (!T.owned || !shard_local(T.sm, kk * T.D + I.row, loc)) continue;
        F M = f_zero(), A = f_zero();
        const uint32_t e1 = I.e_begin + (I.cnt_slot & 0xff);
        for (uint32_t e = I.e_begin; e < e1; ++e) {
            const uint32_t g0 = csr.g0[e], tyb = csr.ty[e], ty = tyb & 0x7f;
            F bg = eq_at(eqg, k * S_cur + g0);
            if (tyb & TY_ASSERT_BIT) bg = f_mul(bg, *assert_r);
            const F tmp = f_mul(bg, eq_at(equ, k * S_pre + csr.u0[e]));
            M = f_mul_add(tmp, s_cM[ty], M);
            if (ty != T_MUL && ty != T_NAAB) A = f_mul_add(tmp, s_cA[ty], A);
        }
        const uint32_t slot = I.cnt_slot >> 8;
        if (slot == 0) {
            const uint32_t o = T.tab_off + loc;
            st_f(tV + o, ld_f(T.src_val + (kz + k) * T.src_S + T.dadId[I.row]));
            st_f(tM + o, M);
            st_f(tA + o, A);
        } else {
            F* dst = partial + 2 * ((size_t)kk * n_slots + (slot - 1));
            st_f(dst, M);
            st_f(dst + 1, A);
        }
    }
}

// ---- phase-2 init, restructured: every coefficient of prover.cpp:319-357 is a0 + a1*V_u (mult) or b1*V_u (add)
// with small integers (a0,a1) in {(1,0),(-1,0),(0,1),(1,-1),(0,-1),(1,-2)} and b1 in {0,1,-1}: a row keeps three plain
// sums S0 = sum a0*t, S1 = sum a1*t, SA = sum b1*t of t = beta_g*beta_u and multiplies by V_u ONCE per row item:
//   mult = S0 + V_u*S1, add = V_u*SA.   Three products per gate (all weakly canonical) instead of five.
VP_D F f_add_w(const F& a, const F& b) { return F{fp_weak(a.re + b.re), fp_weak(a.im + b.im)}; }            // [0,p] x [0,p] -> [0,p]
VP_D F f_sub_w(const F& a, const F& b) { return F{fp_weak(a.re + P - b.re), fp_weak(a.im + P - b.im)}; }
VP_D F f_mul_add_w(const F& a, const F& b, const F& acc);
VP_D F f_mul_w(const F& a, const F& b) { return f_mul_add_w(a, b, f_zero()); }   // a components <= 2p, b in [0,p] -> [0,p]
VP_D F f_mul_add_w(const F& a, const F& b, const F& acc) {   // acc + a*b, acc components < 2^64 -> [0,p]
    const LOp m = make_lop(a.re, a.im);
    const ROpD v = make_ropd(b);
    const u64 u_re = mad32(m.nim1, v.im1d, mad32(m.re1, v.re1d, mad32(m.nim0, v.im0, mul32(m.re0, v.re0))));
    const u64 t_re = mad32(m.nim1, v.im0, mad32(m.nim0, v.im1, mad32(m.re1, v.re0, mul32(m.re0, v.re1))));
    const u64 u_im = mad32(m.im1, v.re1d, mad32(m.re1, v.im1d, mad32(m.im0, v.re0, mul32(m.re0, v.im0))));
    const u64 t_im = mad32(m.im1, v.re0, mad32(m.im0, v.re1, mad32(m.re1, v.im0, mul32(m.re0, v.im1))));
    return F{fp_reduce_ut_weak(u_re, t_re, acc.re), fp_reduce_ut_weak(u_im, t_im, acc.im)};
}
VP_D void p2_accumulate(uint32_t ty, const F& t, F& S0, F& S1, F& SA) {
    switch (ty) {
        case T_ADD: S0 = f_add_w(S0, t); SA = f_add_w(SA, t); break;                       // mult 1,        add  Vu
        case T_SUB: S0 = f_sub_w(S0, t); SA = f_add_w(SA, t); break;                       // mult -1,       add  Vu
        case T_ANTISUB: S0 = f_add_w(S0, t); SA = f_sub_w(SA, t); break;                   // mult 1,        add -Vu
        case T_MUL: S1 = f_add_w(S1, t); break;                                            // mult Vu
        case T_NAAB: S0 = f_add_w(S0, t); S1 = f_sub_w(S1, t); break;                      // mult 1 - Vu
        case T_ANTINAAB: S1 = f_sub_w(S1, t); SA = f_add_w(SA, t); break;                  // mult -Vu,      add  Vu
        case T_XOR: S0 = f_add_w(S0, t); S1 = f_sub_w(S1, f_add_w(t, t)); SA = f_add_w(SA, t); break;   // mult 1 - 2Vu, add Vu
        default: break;
    }
}
// Replicated circuits: eq(r, k*S + g0) = f[idx & mask] * s[idx >> fh], and within ONE instance idx >> fh only takes
// (S >> fh) + 2 consecutive values (SHA256_64 x 1024: at most 6). The product of the two second-half factors of a gate,
// s_g[ig] * s_u[iu], is therefore one of ng*nu values per instance: k_p2_hs tabulates them once per layer
// (HS[(k*ng + i)*nu + j]) and a gate needs two products (f_g*f_u, then * HS) instead of three.
struct HsTab {
    const F* hs;           // null: not used (too many distinct factors per instance, e.g. one huge instance)
    uint32_t ng, nu;
};
__global__ void k_p2_hs(EqTab eqg, EqTab equ, uint32_t S_cur, uint32_t S_pre, uint32_t K, uint32_t ng, uint32_t nu, F* __restrict__ hs,
                        size_t ss) {
    eqg = stmt_at(eqg, ss); equ = stmt_at(equ, ss); hs = stmt_at(hs, ss);
    const uint32_t ig_max = (K * S_cur - 1) >> eqg.fh, iu_max = (K * S_pre - 1) >> equ.fh;   // last second-half entries in use
    const uint32_t per = ng * nu, total = K * per;
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < total; w += gridDim.x * blockDim.x) {
        const uint32_t k = w / per, r = w - k * per, i = r / nu, j = r - i * nu;
        const uint32_t ig = ((k * S_cur) >> eqg.fh) + i, iu = ((k * S_pre) >> equ.fh) + j;
        // (i, j) combinations past the last entry in use belong to no gate: any value will do, but stay inside the tables
        st_f(hs + w, f_mul(ld_f(eqg.s + min(ig, ig_max)), ld_f(equ.s + min(iu, iu_max))));
    }
}
__global__ void __launch_bounds__(256, 4)
k_init_phase2_v2(const RowItem* __restrict__ items, uint32_t n_items, const P2Table* __restrict__ tabs, CsrP2 csr,
                 uint32_t S_pre, uint32_t S_cur, uint32_t K, EqTab eqg, EqTab equ, const F* __restrict__ assert_r,
                 const F* __restrict__ Vu_ptr, F* __restrict__ tV, F* __restrict__ tM, F* __restrict__ tA,
                 F* __restrict__ partial, uint32_t n_slots, uint32_t kk_begin, uint32_t kk_end, HsTab H, size_t ss) {
    // this statement's buffers are zo entries on: one offset instead of ten shifted pointers (those would spill here)
    const size_t zo = (size_t)blockIdx.z * (ss / sizeof(F));
    const F Vu = Vu_ptr[zo];
    const uint32_t total = n_items * (kk_end - kk_begin);   // < 2^32 (host check)
    for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < total; w += gridDim.x * blockDim.x) {
        const uint32_t kq = w / n_items, it = w - kq * n_items, kk = kk_begin + kq, k = K - 1 - kk;
        const RowItem I = items[it];
        const P2Table T = tabs[I.tab];
        uint32_t loc;
        if (!T.owned || !shard_local(T.sm, kk * T.D + I.row, loc)) continue;
        F S0 = f_zero(), S1 = f_zero(), SA = f_zero();
        const uint32_t e1 = I.e_begin + (I.cnt_slot & 0xff);
        for (uint32_t e = I.e_begin; e < e1; ++e) {
            const uint32_t g0 = csr.g0[e], tyb = csr.ty[e], u0 = csr.u0[e];
            F t;
            if (H.hs) {
                const uint32_t ig = k * S_cur + g0, iu = k * S_pre + u0;
                const uint32_t i = (ig >> eqg.fh) - ((k * S_cur) >> eqg.fh), j = (iu >> equ.fh) - ((k * S_pre) >> equ.fh);
                const F ff = f_mul_w(ld_f(eqg.f + zo + (ig & eqg.mask)), ld_f(equ.f + zo + (iu & equ.mask)));
                t = f_mul_w(ff, ld_f(H.hs + zo + (k * H.ng + i) * H.nu + j));
                if (tyb & TY_ASSERT_BIT) t = f_mul(t, assert_r[zo]);
            } else {
                const EqTab g{eqg.f + zo, eqg.s + zo, eqg.fh, eqg.mask}, u{equ.f + zo, equ.s + zo, equ.fh, equ.mask};
                F bg = eq_at_weak(g, k * S_cur + g0);
                if (tyb & TY_ASSERT_BIT) bg = f_mul(bg, assert_r[zo]);
                t = f_mul_w(bg, eq_at_weak(u, k * S_pre + u0));
            }
            p2_accumulate(tyb & 0x7f, t, S0, S1, SA);
        }
        const F M = f_strict(f_add_w(S0, f_mul_w(S1, Vu))), A = f_strict(f_mul_w(SA, Vu));
        const uint32_t slot = I.cnt_slot >> 8;
        if (slot == 0) {
            const uint32_t o = T.tab_off + loc;
            st_f(tV + zo + o, ld_f(T.src_val + ((size_t)blockIdx.z * K + k) * T.src_S + T.dadId[I.row]));
            st_f(tM + zo + o, M);
            st_f(tA + zo + o, A);
        } else {
            F* dst = partial + zo + 2 * ((size_t)kk * n_slots + (slot - 1));
            st_f(dst, M);
            st_f(dst + 1, A);
        }
    }
}

__global__ void __launch_bounds__(256)
k_combine_phase2(const LongRow* __restrict__ rows, uint32_t n_rows, const P2Table* __restrict__ tabs, uint32_t K,
                 F* __restrict__ tV, F* __restrict__ tM, F* __restrict__ tA, const F* __restrict__ partial, uint32_t n_slots,
                 uint32_t kk_begin, uint32_t kk_end, size_t ss) {
    const size_t kz = (size_t)blockIdx.z * K;   // this statement's first global instance
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss); partial = stmt_at(partial, ss);
    const uint64_t total = (uint64_t)n_rows * (kk_end - kk_begin);
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t kq = (uint32_t)(w / n_rows), j = (uint32_t)(w - (uint64_t)kq * n_rows), kk = kk_begin + kq, k = K - 1 - kk;
        const LongRow R = rows[j];
        const P2Table T = tabs[R.tab];
        uint32_t loc;
        if (!T.owned || !shard_local(T.sm, kk * T.D + R.row, loc)) continue;
        F M = f_zero(), A = f_zero();
        for (uint32_t s = R.slot_begin; s < R.slot_end; ++s) {
            const F* src = partial + 2 * ((size_t)kk * n_slots + s);
            M = f_add(M, ld_f_cg(src));
            A = f_add(A, ld_f_cg(src + 1));
        }
        const uint32_t o = T.tab_off + loc;
        st_f(tV + o, ld_f(T.src_val + (kz + k) * T.src_S + T.dadId[R.row]));
        st_f(tM + o, M);
        st_f(tA + o, A);
    }
}

// Unary gates of phase 2 (prover.cpp:342-353): all of them add into addVArray[i-1][0].
// U = sum_g beta_g[g]*beta_u[u] * coef(ty), coef = c+Vu | c*Vu | Vu | 1-Vu. The add table enters the
// round polynomials only linearly, and entry 0 is "low bit 0" in every round, so adding U to add[i-1][0]
// is the same as starting the phase with add_term = U (it is scaled by (1 - r) every round exactly like
// the folded table entry would be). The grid sums U over the instances [k_begin, k_end) into *dst; a
// sharded context gives every rank its own instance slice and the partial add_terms add up.
struct CsrUnary {
    const uint32_t* g0;
    const uint32_t* u0;
    const uint8_t* ty;
    uint32_t n;   // unary gates in one instance
};
__global__ void __launch_bounds__(256)
k_phase2_unary(CsrUnary un, uint32_t S_pre, uint32_t S_cur, uint32_t K, EqTab eqg, EqTab equ,
               const F* __restrict__ assert_r, const F* __restrict__ Vu_ptr, const F* __restrict__ cst,
               F* __restrict__ dst, F* partials, unsigned int* counter, uint32_t k_begin, uint32_t k_end, size_t ss) {
    __shared__ F smem[32];
    // this statement's eq tables are zo entries on; the outputs are shifted after the loop (fewer live registers)
    const size_t zo = (size_t)blockIdx.z * (ss / sizeof(F));
    const EqTab g{eqg.f + zo, eqg.s + zo, eqg.fh, eqg.mask}, u{equ.f + zo, equ.s + zo, equ.fh, equ.mask};
    const F Vu = Vu_ptr[zo];
    const uint64_t total = (uint64_t)un.n * (k_end - k_begin);
    F acc[1] = {f_zero()};
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k = k_begin + (uint32_t)(w / un.n), j = (uint32_t)(w % un.n);
        const uint32_t g0 = un.g0[j], tyb = un.ty[j], ty = tyb & 0x7f;
        F bg = eq_at(g, k * S_cur + g0);
        if (tyb & TY_ASSERT_BIT) bg = f_mul(bg, assert_r[zo]);
        const F tmp = f_mul(bg, eq_at(u, k * S_pre + un.u0[j]));
        F coef;
        switch (ty) {
            case T_ADDC: coef = f_add(cst[g0], Vu); break;
            case T_MULC: coef = f_mul(cst[g0], Vu); break;
            case T_COPY: coef = Vu; break;
            default: coef = f_sub(f_one(), Vu); break;  // T_NOT
        }
        acc[0] = f_add(acc[0], f_mul(tmp, coef));
    }
    if (grid_sum<1>(acc, smem, stmt_at(partials, ss), stmt_at(counter, ss)) && threadIdx.x == 0) st_f(stmt_at(dst, ss), acc[0]);
}

// ------------------------------------------------------------------ K5: Liu table init
// prover.cpp:389-414. mult[u] = s0*eq(r_u,u) + sum_{(j,slot): dadId_j[pre][slot]==u} eq_j(slot)
// where eq_j already carries the scale s[j-i+1] in its first half table.
struct LiuEntry {       // one (j, slot0) pair pointing at template u0
    uint32_t eq_id;     // index into the per-init EqTab array
    uint32_t slot0;
    uint32_t D;         // subset size of one instance (for the reversed instance order)
};
__global__ void __launch_bounds__(256)
k_init_liu(const uint32_t* __restrict__ off, const uint32_t* __restrict__ perm, const LiuEntry* __restrict__ ent, const EqTab* __restrict__ eqs,
           uint32_t S_pre, uint32_t K, EqTab equ, const F* __restrict__ s0_ptr, const F* __restrict__ Vpre,
           F* __restrict__ tV, F* __restrict__ tM, F* __restrict__ tA, ShardMap sm, uint32_t n_local, int write_a,
           int equ_scaled, int write_v, size_t ss) {
    equ = stmt_at(equ, ss); s0_ptr = stmt_at(s0_ptr, ss);
    tV = stmt_at(tV, ss); tM = stmt_at(tM, ss); tA = stmt_at(tA, ss);
    Vpre += (size_t)blockIdx.z * K * S_pre;
    const uint32_t n = S_pre * K;
    const F s0 = *s0_ptr;
    for (uint32_t loc0 = blockIdx.x * blockDim.x + threadIdx.x; loc0 < n_local; loc0 += gridDim.x * blockDim.x) {
        uint32_t loc = loc0;
        if (perm) {   // unsharded: visit the entries of an instance in length-sorted order (uniform trip counts per warp)
            const uint32_t kq = loc0 / S_pre;
            loc = kq * S_pre + perm[loc0 - kq * S_pre];
        }
        const uint32_t u = shard_global(sm, loc);
        if (u >= n) continue;
        const uint32_t k = u / S_pre, u0 = u - k * S_pre;
        F M = eq_at_weak(equ, u);                  // equ_scaled: its first half table already carries s[0]
        if (!equ_scaled) M = f_mul(M, s0);
        for (uint32_t e = off[u0]; e < off[u0 + 1]; ++e) {   // the running sum rides as the addend of each product's reduction
            const LiuEntry E = ent[e];
            M = eq_at_acc_w(stmt_at(eqs[E.eq_id], ss), (K - 1 - k) * E.D + E.slot0, M);
        }
        if (write_v) st_f(tV + loc, ld_f(Vpre + u));   // unsharded whole-proof mode reads V straight from circuitValue
        st_f(tM + loc, f_strict(M));
        if (write_a) st_f(tA + loc, f_zero());   // the Liu add table is identically zero: only the one-round-per-launch path reads it
    }
}

// Template-major form of K5: a thread owns ONE template entry u0 (visited in length-sorted order)
// and walks a chunk of the data-parallel instances, so everything that only depends on the template -- the CSR bounds,
// the scattered terms' (table, slot, subset size), the tables' descriptors -- is read once per thread instead of once
// per (entry, instance), the instance index needs no division, and two instances are in flight per iteration
// (independent reduction chains). Lanes of a warp still hold neighbouring entries of the same instance: the table
// stores and the eq lookups stay as coalesced as in k_init_liu.
__global__ void __launch_bounds__(256)
k_init_liu_tm(const uint32_t* __restrict__ off, const uint32_t* __restrict__ perm, const LiuEntry* __restrict__ ent, const EqTab* __restrict__ eqs,
              uint32_t S_pre, uint32_t K, uint32_t k_chunk, EqTab equ, const F* __restrict__ s0_ptr, const F* __restrict__ Vpre,
              F* __restrict__ tV, F* __restrict__ tM, F* __restrict__ tA, int write_a, int equ_scaled, int write_v, ShardMap sm,
              uint32_t k_begin, uint32_t k_end, size_t ss) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= S_pre) return;
    // this statement's buffers are zo entries on, its values vz: two offsets instead of six shifted pointers (registers)
    const size_t zo = (size_t)blockIdx.z * (ss / sizeof(F)), vz = (size_t)blockIdx.z * K * S_pre;
    const uint32_t u0 = perm ? perm[x] : x;
    const uint32_t eb = off[u0], n_terms = off[u0 + 1] - eb;
    const uint32_t k0 = k_begin + blockIdx.y * k_chunk, k1 = min(k_end, k0 + k_chunk);   // sharded: the instances the rank's rows touch
    const F s0 = s0_ptr[zo];
    // the first two scattered terms live in registers (most entries have at most two)
    LiuEntry E0{0, 0, 0}, E1{0, 0, 0};
    const EqTab eu{equ.f + zo, equ.s + zo, equ.fh, equ.mask};
    EqTab T0 = eu, T1 = eu;
    if (n_terms >= 1) { E0 = ent[eb]; T0 = stmt_at(eqs[E0.eq_id], ss); }
    if (n_terms >= 2) { E1 = ent[eb + 1]; T1 = stmt_at(eqs[E1.eq_id], ss); }
    for (uint32_t k = k0; k < k1; ++k) {
        const uint32_t u = k * S_pre + u0, kk = K - 1 - k;
        uint32_t loc;
        if (!shard_local(sm, u, loc)) continue;   // (sharded) a row of another rank
        F M = eq_at_weak(eu, u);
        if (!equ_scaled) M = f_mul(M, s0);
        if (n_terms >= 1) M = eq_at_acc_w(T0, kk * E0.D + E0.slot0, M);
        if (n_terms >= 2) M = eq_at_acc_w(T1, kk * E1.D + E1.slot0, M);
        for (uint32_t q = 2; q < n_terms; ++q) {
            const LiuEntry E = ent[eb + q];
            M = eq_at_acc_w(stmt_at(eqs[E.eq_id], ss), kk * E.D + E.slot0, M);
        }
        if (write_v) st_f(tV + zo + loc, ld_f(Vpre + vz + u));
        st_f(tM + zo + loc, f_strict(M));
        if (write_a) st_f(tA + zo + loc, f_zero());
    }
}

// ------------------------------------------------------------------ K6: fused fold + round polynomial
// prover.cpp:436-492 (sumcheckUpdate / sumcheckUpdateEach).
struct TabDesc {        // a table that is still >= one pair in this round
    uint32_t in_off;    // entries into the input buffers (multiple of 4)
    uint32_t in_live;   // live (possibly non-zero) stored entries; entries beyond are zero and never read
    uint32_t out_off;   // entries into the output buffers (FOLD rounds)
    uint32_t work_end;  // inclusive prefix of work items (pairs when !FOLD, quads when FOLD)
};
struct ColDesc {        // a table that collapses to a scalar in this round (total == 1, prover.cpp:462-467)
    uint32_t in_off;
    uint32_t n_vals;    // stored live values: 0, 1 or 2 (2 => fold with the previous challenge)
    int32_t claim_slot; // where to keep V for Finalize2, or -1
    uint32_t pad;
};
struct RoundArgs {
    const F *inV, *inM, *inA;
    F *outV, *outM, *outA;
    const TabDesc* tabs;
    const ColDesc* cols;
    uint32_t n_tabs, n_cols;
    const F* prev_r;          // previous challenge (ignored when !FOLD and no 2-value collapse)
    F* add_term;              // device scalar (prover.h:62)
    F* claims;                // V of collapsed tables
    F* out_poly;              // 3 F: a, b, c
    F* partials;
    unsigned int* counter;
    uint32_t first_round;     // 1: add_term is not scaled by (1 - prev) (prev == 0)
    uint32_t reset_add_term;  // 1: start from add_term = *at_init (or 0)
    const F* at_init;         // initial add_term of the phase (phase 2: the unary-gate sum), may be null
    // Interactive fast path (vp_round on one GPU): the previous challenge comes BY VALUE (prev_by_value != 0; the last
    // block also files it at prev_w for the kernels that read the challenge array later) and the round polynomial is also
    // written to host_poly -- pinned host memory mapped into the device -- followed by the sequence number host_seq the
    // host spins on: no copy call, no stream synchronisation per round.
    F prev_val;
    F* prev_w;
    uint32_t prev_by_value;
    F* host_poly;
    unsigned int* host_seq;
    unsigned int seq;
};

VP_D F ld_bound(const F* base, uint32_t idx, uint32_t live) { return idx < live ? ld_f(base + idx) : f_zero(); }

// Per-thread running sums of one round. With B = sum m1*v1, C = sum m0*v0, E = sum (m0+m1)*(v0+v1):
//   a = sum (m1-m0)(v1-v0)               = 2B + 2C - E
//   b = sum (m1-m0)v0 + (v1-v0)m0 + ...  = E - B - 3C + (sum a1 - sum a0)
//   c = sum m0*v0 + sum a0               = C + sum a0
// (three complex products per pair, no differences to canonicalise). B, C, E stay canonical: the
// running value rides as the `extra` term of each product's single reduction.
struct RoundAcc {
    F B, C, E;
    u64 s0re, s0im, s1re, s1im;  // lazy sums of the add table (folded every 4 pairs)
    int pending;
};
VP_D void racc_init(RoundAcc& s) {
    s.B = f_zero(); s.C = f_zero(); s.E = f_zero();
    s.s0re = s.s0im = s.s1re = s.s1im = 0;
    s.pending = 0;
}
VP_D void racc_pair(RoundAcc& s, const F& v0, const F& v1, const F& m0, const F& m1, const F& a0, const F& a1) {
    // running sums stay "loose" (<= p + 5, folded once): they only ride as the next product's addend
    s.C = f_mul_add_k_loose(make_lop(m0.re, m0.im), make_ropd(v0), s.C);
    s.B = f_mul_add_k_loose(make_lop(m1.re, m1.im), make_ropd(v1), s.B);
    s.E = f_mul_add_loose2(make_lop(m0.re + m1.re, m0.im + m1.im), make_rop(v0.re + v1.re, v0.im + v1.im), s.E);
    s.s0re += a0.re; s.s0im += a0.im; s.s1re += a1.re; s.s1im += a1.im;
    if (++s.pending == 4) {
        s.s0re = fp_fold(s.s0re); s.s0im = fp_fold(s.s0im); s.s1re = fp_fold(s.s1re); s.s1im = fp_fold(s.s1im);
        s.pending = 0;
    }
}
VP_D void racc_finish(const RoundAcc& s, F (&v)[3]) {
    const F sa0 = F{fp_canon(s.s0re), fp_canon(s.s0im)}, sa1 = F{fp_canon(s.s1re), fp_canon(s.s1im)};
    const F B = F{fp_red1(s.B.re), fp_red1(s.B.im)}, C = F{fp_red1(s.C.re), fp_red1(s.C.im)},
            E = F{fp_red1(s.E.re), fp_red1(s.E.im)};   // loose (<= p + 5) -> canonical
    const F twoBC = f_dbl(f_add(B, C));
    v[0] = f_sub(twoBC, E);
    v[1] = f_add(f_sub(f_sub(E, B), f_add(f_dbl(C), C)), f_sub(sa1, sa0));
    v[2] = f_add(C, sa0);
}

// Work of one round over the tables [tabs, tabs + n_tabs): each thread strides over pairs (!FOLD) or
// quads (FOLD) of the concatenated work range and leaves its sums in `acc`.
// s_wend: shared array of the tables' inclusive work prefixes (filled by the caller).
template <bool FOLD, bool NC>
VP_D void round_work(RoundAcc& acc, const TabDesc* __restrict__ tabs, uint32_t n_tabs, const uint32_t* s_wend,
                     const F* inV, const F* inM, const F* inA, F* outV, F* outM, F* outA, const FoldK& rk,
                     uint32_t first, uint32_t stride) {
    const uint32_t total = n_tabs ? s_wend[n_tabs - 1] : 0;
    uint32_t t = 0;
    TabDesc T = n_tabs ? tabs[0] : TabDesc{0, 0, 0, 0};
    uint32_t wbeg = 0;
    for (uint32_t w = first; w < total; w += stride) {
        if (w >= s_wend[t]) {
            do { ++t; } while (w >= s_wend[t]);
            T = tabs[t];
            wbeg = s_wend[t - 1];
        }
        const uint32_t q = w - wbeg;
        const F* V = inV + T.in_off;
        const F* M = inM + T.in_off;
        const F* A = inA + T.in_off;
        if (!FOLD) {
            const uint32_t i0 = 2 * q;
            F v0, v1, m0, m1, a0, a1;
            if (i0 + 1 < T.in_live) {
                ld_pair<NC>(V + i0, v0, v1);
                ld_pair<NC>(M + i0, m0, m1);
                ld_pair<NC>(A + i0, a0, a1);
            } else {
                v0 = ld_one<NC>(V + i0); m0 = ld_one<NC>(M + i0); a0 = ld_one<NC>(A + i0);
                v1 = m1 = a1 = f_zero();
            }
            racc_pair(acc, v0, v1, m0, m1, a0, a1);
        } else {
            const uint32_t i0 = 4 * q;
            F xv[4], xm[4], xa[4];
            if (i0 + 3 < T.in_live) {
                ld_pair<NC>(V + i0, xv[0], xv[1]); ld_pair<NC>(V + i0 + 2, xv[2], xv[3]);
                ld_pair<NC>(M + i0, xm[0], xm[1]); ld_pair<NC>(M + i0 + 2, xm[2], xm[3]);
                ld_pair<NC>(A + i0, xa[0], xa[1]); ld_pair<NC>(A + i0 + 2, xa[2], xa[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const bool in = i0 + j < T.in_live;
                    xv[j] = in ? ld_one<NC>(V + i0 + j) : f_zero();
                    xm[j] = in ? ld_one<NC>(M + i0 + j) : f_zero();
                    xa[j] = in ? ld_one<NC>(A + i0 + j) : f_zero();
                }
            }
            const F v0 = f_fold_k(xv[0], xv[1], rk), v1 = f_fold_k(xv[2], xv[3], rk);
            const F m0 = f_fold_k(xm[0], xm[1], rk), m1 = f_fold_k(xm[2], xm[3], rk);
            const F a0 = f_fold_k(xa[0], xa[1], rk), a1 = f_fold_k(xa[2], xa[3], rk);
            const uint32_t o = T.out_off + 2 * q;   // buffers are padded to 4 entries: the pair store is always in bounds
            st_pair(outV + o, v0, v1);
            st_pair(outM + o, m0, m1);
            st_pair(outA + o, a0, a1);
            racc_pair(acc, v0, v1, m0, m1, a0, a1);
        }
    }
}

// add_term bookkeeping of one round (prover.cpp:445,462-467): at' = at*(1 - prev) + sum over tables that
// collapse in this round of V*mult + add (their two stored values folded with prev when !first).
// fold_vals: the collapsing tables hold two stored values still to be folded with prev (false in the first
// round of a kernel's plan); scale: a previous challenge exists (false only in round 1 of the phase).
template <bool NC>
VP_D F collapse_update(F at, const ColDesc* __restrict__ cols, uint32_t n_cols, const F* inV, const F* inM, const F* inA,
                       bool fold_vals, bool scale, const F& prev, const FoldK& rk, F* claims) {
    const bool first = !fold_vals;
    if (scale) at = f_mul(at, f_sub(f_one(), prev));
    for (uint32_t i = 0; i < n_cols; ++i) {
        const ColDesc c = cols[i];
        F cv = f_zero(), cm = f_zero(), ca = f_zero();
        if (c.n_vals >= 1) {
            cv = ld_one<false>(inV + c.in_off); cm = ld_one<false>(inM + c.in_off); ca = ld_one<false>(inA + c.in_off);
            if (!first) {
                F v1 = f_zero(), m1 = f_zero(), a1 = f_zero();
                if (c.n_vals >= 2) {
                    v1 = ld_one<false>(inV + c.in_off + 1); m1 = ld_one<false>(inM + c.in_off + 1); a1 = ld_one<false>(inA + c.in_off + 1);
                }
                cv = f_fold_k(cv, v1, rk); cm = f_fold_k(cm, m1, rk); ca = f_fold_k(ca, a1, rk);
            }
        }
        at = f_add(at, f_mul_add(cv, cm, ca));
        if (c.claim_slot >= 0) st_f(claims + c.claim_slot, cv);
    }
    return at;
}

// One round per launch: the interactive path (the next challenge only arrives after this round's
// polynomial went back to the verifier).
template <bool FOLD>
__global__ void __launch_bounds__(256, 2) k_round(RoundArgs p) {
    __shared__ F smem[3 * 32];
    __shared__ uint32_t s_wend[128];
    for (uint32_t i = threadIdx.x; i < p.n_tabs; i += blockDim.x) s_wend[i] = p.tabs[i].work_end;
    __syncthreads();
    FoldK rk = make_foldk(f_zero());
    if (FOLD) rk = make_foldk(p.prev_by_value ? p.prev_val : *p.prev_r);
    RoundAcc acc;
    racc_init(acc);
    round_work<FOLD, true>(acc, p.tabs, p.n_tabs, s_wend, p.inV, p.inM, p.inA, p.outV, p.outM, p.outA, rk,
                           blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
    F v[3];
    racc_finish(acc, v);
    if (!grid_sum<3>(v, smem, p.partials, p.counter)) return;
    if (threadIdx.x != 0) return;
    F at = p.reset_add_term ? (p.at_init ? *p.at_init : f_zero()) : *p.add_term;
    const F prev = p.first_round ? f_zero() : (p.prev_by_value ? p.prev_val : *p.prev_r);
    if (p.prev_by_value) st_f(p.prev_w, p.prev_val);
    at = collapse_update<true>(at, p.cols, p.n_cols, p.inV, p.inM, p.inA, FOLD, !p.first_round, prev, rk, p.claims);
    st_f(p.add_term, at);
    const F b = f_sub(v[1], at), c = f_add(v[2], at);
    st_f(p.out_poly + 0, v[0]);
    st_f(p.out_poly + 1, b);
    st_f(p.out_poly + 2, c);
    if (p.host_poly) {
        st_f(p.host_poly + 0, v[0]);
        st_f(p.host_poly + 1, b);
        st_f(p.host_poly + 2, c);
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.host_seq), "r"(p.seq) : "memory");
    }
}

// ------------------------------------------------------------------ K7: finalize
// prover.cpp:494-521: claim = Vmult[.][0].eval(last challenge) for tables still alive, the kept
// collapse value otherwise.
struct FinDesc {
    uint32_t in_off;
    uint32_t n_vals;     // 0,1,2 stored live values of V; 2 => fold with last challenge
    int32_t from_claim;  // >= 0: table collapsed earlier, value is claims[from_claim]
    uint32_t out_idx;    // transcript index
};
__global__ void k_finalize(const FinDesc* __restrict__ d, int n, const F* __restrict__ V, const F* __restrict__ last_r,
                           int have_r, const F* __restrict__ claims, F* __restrict__ transcript, F* __restrict__ keep) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const FinDesc f = d[i];
    F c;
    if (f.from_claim >= 0) c = claims[f.from_claim];
    else {
        F v0 = f.n_vals >= 1 ? V[f.in_off] : f_zero();
        if (have_r) {
            F v1 = f.n_vals >= 2 ? V[f.in_off + 1] : f_zero();
            c = f_fold(v0, v1, *last_r);
        } else c = v0;
    }
    st_f(transcript + f.out_idx, c);
    if (keep && i == 0) st_f(keep, c);   // V_u for phase 2 (prover.cpp:497)
}

// ------------------------------------------------------------------ K6f: one sumcheck phase in ONE launch, one round per pass
// The plan of k_sumcheck_phase_fs (fs_device.cuh), which runs all rounds of one phase (phase 1, phase 2 or Liu of one
// layer) of a Fiat-Shamir proof and draws each round's challenge itself.
struct RoundDev {
    uint32_t tab_begin, n_tabs, col_begin, n_cols;
    uint32_t work;     // pairs (first round) or quads
    uint32_t in_buf;   // 0 / 1
};
struct PhaseArgs {
    F* bufV[2];
    F* bufM[2];
    F* bufA[2];
    const RoundDev* rounds;
    const TabDesc* tabs;
    const ColDesc* cols;
    const FinDesc* fins;
    uint32_t n_rounds, n_fin, fin_buf;
    uint32_t tail_work;        // rounds with work <= tail_work run on block 0 alone
    const F* at_init;          // initial add_term (phase 2: the unary-gate sum), may be null
    F* add_term;
    F* claims;
    F* out_poly;               // round j -> out_poly[3*(j-1) ..]
    F* transcript;             // FinDesc.out_idx indexes this
    F* keep;                   // V_u (phase 1) or null
    F* partials;               // 2 * gridDim.x * 3
};

// ------------------------------------------------------------------ K6d: two rounds per pass (whole-proof mode)
// With the challenges on the device a pass can run TWO rounds on data it holds in registers: a thread reads a
// quad x[4q..4q+3] of level-L values, accumulates round L+1's polynomial from the pairs (x0,x1),(x2,x3), folds them
// with r_{L+1}, accumulates round L+2's polynomial from the folded pair, folds with r_{L+2} and writes ONE value.
// HBM traffic per table triple drops from 192*N (one round per pass: 144*N, plus the challenge-less first read)
// to 48*N*(1 + 1/4 + ...) + 12*N*(...) = 80*N, which makes the kernel INT-pipe bound instead of HBM bound.
// Stored tables hold level-L values with nothing pending (the one-round kernel keeps a fold pending).
struct PassTab {
    uint32_t in_off, in_live, out_off;
    uint32_t work_end;   // inclusive prefix of work items: quads (two == 1) or pairs
    uint32_t two;        // 1: the table runs both rounds of the pass; 0: one round (pair -> one value)
    uint32_t pad;
};
struct PassCol {         // a table that is down to one value and joins add_term (prover.cpp:462-467)
    uint32_t off;        // where its single value sits
    uint32_t n_vals;     // 0: empty table
    int32_t claim_slot;
    uint32_t which;      // 0: collapses in the pass's first round (value in the IN buffer); 1: second round (OUT buffer)
};
struct PassDev {
    uint32_t tab_begin, n_tabs, col_begin, n_cols;
    uint32_t work, in_buf, n_rounds, pad;   // n_rounds: 1 or 2 rounds in this pass
};
struct DfsArgs {
    F* bufV[2];
    F* bufM[2];
    F* bufA[2];
    const PassDev* passes;
    const PassTab* tabs;
    const PassCol* cols;
    const FinDesc* fins;
    uint32_t n_passes, n_fin, fin_buf;
    uint32_t tail_work;        // unused (kept for layout); the tail is whatever fits one block
    uint32_t round_base;       // global rounds done before this kernel
    const F* at_init;
    const F* chal;             // chal[g-1] = challenge bound after global round g
    F* add_term;
    F* claims;
    F* out_poly;               // local round j (1-based) -> out_poly[3*(j-1)]
    F* transcript;
    F* keep;
    F* partials;               // 2 * gridDim.x * 6
    unsigned int* bar;         // grid-barrier counter, zero at launch (the kernel leaves it zero)
    unsigned int* chunk_ctr;   // one work counter per pass, zero at launch (the kernel leaves them zero)
    const F* v_first;          // if set: the first pass reads its V table from here (circuitValue[i-1], no copy made)
    ConstK rk[32];             // rk[j]: the challenge bound after local round j+1 of this launch, pre-split (host side)
    F* claim0;                 // DFS_NEED_B: where round 1's p(0) + p(1) goes (the claim the chain starts from)
    unsigned long long* dbg;   // optional: block 0 writes %globaltimer at 4 points of every pass (profiling aid)
};

// Per-thread running sums of one round of the pass kernel. The round polynomial a*x^2 + b*x + c is sent as
//   a = sum (m1-m0)(v1-v0),  c = sum m0*v0 + sum a0 (+ add_term),  b = claim - 2c - a
// where claim = p(0) + p(1) is the previous round's polynomial at its challenge (the honest prover's messages satisfy
// the verifier's check verifier.cpp:209,248,296 identically, so b need not be summed: k_derive_b fills it in from the
// claim chain once the claims it starts from are known). Two complex products per pair instead of the reference's
// four (polynomial.cpp:101-110); both sums are LAZY (96-bit partial sums of the limb products, reduced once per pass).
struct PassAcc {
    CAcc A, C;
    u64 s0re, s0im;   // sum of a0, folded once per work item
};
VP_D void pacc_init(PassAcc& s) {
    s.A = cacc_zero(); s.C = cacc_zero();
    s.s0re = s.s0im = 0;
}
VP_D void pacc_finish(const PassAcc& s, F& a, F& c) {
    a = cacc_reduce(s.A);
    c = f_add(cacc_reduce(s.C), F{fp_canon(s.s0re), fp_canon(s.s0im)});
}
VP_D void pacc_mad(CAcc& acc, const F& m, const F& v) { cacc_mad(acc, make_lop(m.re, m.im), make_ropd(v)); }
VP_D void pacc_mad_real(CAcc& acc, const F& m, u64 v) { cacc_mad_real(acc, m, v); }
typedef CAcc PassSum;
VP_D PassSum psum_zero() { return cacc_zero(); }
VP_D F psum_reduce(const PassSum& s) { return cacc_reduce(s); }
// Second round of a pass: the same two sums, but as weakly canonical running values that ride in the products'
// reductions (8 registers instead of 28: the pass kernel is register bound, and the second round is a third of the work)
struct PassAcc2 {
    F A, C;
    u64 s0re, s0im;
};
VP_D void pacc2_init(PassAcc2& s) { s.A = f_zero(); s.C = f_zero(); s.s0re = s.s0im = 0; }
VP_D void pacc2_finish(const PassAcc2& s, F& a, F& c) {
    a = f_strict(s.A);
    c = f_add(f_strict(s.C), F{fp_canon(s.s0re), fp_canon(s.s0im)});
}
VP_D void dfs_pair2(PassAcc2& s, bool has_a, const F& v0, const F& v1, const F& m0, const F& m1, const F& a0, const F& a1,
                    const ConstK& rk, F& ov, F& om, F& oa) {
    const F dm = f_diff2p(m0, m1), dv = f_diff_w(v0, v1);
    s.C = f_mul_add_w(m0, v0, s.C);
    s.A = f_mul_add_w(dm, dv, s.A);
    ov = f_fold_w(v0, dv, rk);
    om = f_fold_w(m0, dm, rk);
    if (has_a) {
        s.s0re += a0.re; s.s0im += a0.im;
        oa = f_fold_w(a0, f_diff2p(a0, a1), rk);
    }
}
// only the very first round of a stand-alone sumcheck has no claim to start from: it also sums p(1) = sum m1*v1 + a1
struct PassAccB {
    PassSum B;
    u64 s1re, s1im;
};
// One pair of one round: accumulate, fold the three tables with the round's challenge.
// VREAL: the V table is in the base field (circuit values, first pass of every GKR phase): half the limb products.
// Operands are weakly canonical ([0,p]); so are the folded values.
template <bool VREAL, bool HAS_A, bool NEED_B>
VP_D void dfs_pair(PassAcc& s, PassAccB* sb, const F& v0, const F& v1, const F& m0, const F& m1, const F& a0, const F& a1,
                   const ConstK& rk, F& ov, F& om, F& oa) {
    const F dm = f_diff2p(m0, m1);
    if (VREAL) {
        const u64 dv = fp_weak(v1.re + P - v0.re);
        pacc_mad_real(s.C, m0, v0.re);
        pacc_mad_real(s.A, dm, dv);
        if (NEED_B) pacc_mad_real(sb->B, m1, v1.re);
        ov = f_fold_w_real(v0.re, dv, rk);
    } else {
        const F dv = f_diff_w(v0, v1);
        pacc_mad(s.C, m0, v0);
        pacc_mad(s.A, dm, dv);
        if (NEED_B) pacc_mad(sb->B, m1, v1);
        ov = f_fold_w(v0, dv, rk);
    }
    om = f_fold_w(m0, dm, rk);
    if (HAS_A) {
        s.s0re += a0.re; s.s0im += a0.im;
        if (NEED_B) { sb->s1re += a1.re; sb->s1im += a1.im; }
        oa = f_fold_w(a0, f_diff2p(a0, a1), rk);
    }
}

// Work distribution and staging of the pass kernel.
//  * A pass's work items (quads, or pairs for a table in its last odd round) are numbered over the concatenated
//    tables; every table's share is padded to a multiple of 32, so a SUB-CHUNK of 32 consecutive items (one per lane)
//    lies in one table. Items past a table's live entries read zeros, add nothing and store nothing.
//  * Each WARP runs its own two-stage cp.async pipeline through shared memory: while it computes sub-chunk n from
//    stage n&1, the 16-byte pieces of sub-chunk n+1 are in flight into the other stage (zero-filled past the live
//    entries with src-size 0). No block barrier and no exposed load latency in the loop; no registers are tied up
//    by prefetched data. Pieces are copied with consecutive lanes on consecutive 16 bytes (coalesced) and land at
//    slot 4q + (j ^ ((q >> 1) & 3)) so that lane q's four 128-bit reads of its quad are bank-conflict free.
//  * Warps take chunks of DFS_WCHUNK = 128 items (4 sub-chunks) from an atomic counter, fetched one chunk ahead:
//    equal static shares finish up to 1.5x apart across SMs (measured), so the fast SMs take more.
#ifndef VP_DFS_MINB
#define VP_DFS_MINB 3
#endif
#ifndef VP_DFS_THREADS
#define VP_DFS_THREADS 128
#endif
static constexpr uint32_t DFS_WCHUNK = 128;   // items per warp chunk
static constexpr uint32_t DFS_CHUNK = (VP_DFS_THREADS / 32) * DFS_WCHUNK;    // items a block covers in one sweep (sizing of grids / worker counts)
#ifndef VP_DFS_SOLO
#define VP_DFS_SOLO 128
#endif
#ifndef VP_DFS_SOLO_THIN
#define VP_DFS_SOLO_THIN 1
#endif
static constexpr uint32_t DFS_SOLO = VP_DFS_SOLO;   // a pass of at most this many items runs on block 0 alone (no grid barrier)
static constexpr uint32_t DFS_STAGE_F = 3 * 128;              // F slots per stage: 3 tables x 32 quads
static constexpr uint32_t DFS_WARP_SMEM_F = 2 * DFS_STAGE_F;  // two stages per warp

VP_D void cp_async16(uint32_t smem_addr, const void* gptr, uint32_t src_size) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr), "l"(gptr), "r"(src_size) : "memory");
}
VP_D void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
VP_D void cp_async_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

template <bool HAS_A, bool VREAL, bool NEED_B>
VP_D void dfs_work(PassAcc& acc1, PassAcc2& acc2, PassAccB* accb, const PassTab* __restrict__ tabs, uint32_t n_tabs,
                   const uint32_t* s_wend, const F* inV, const F* inM, const F* inA, F* outV, F* outM, F* outA,
                   const ConstK& rk1, const ConstK& rk2, unsigned int* chunk_ctr, uint32_t stage_base /* this warp's smem */,
                   const F* stage_ptr /* the same, as a pointer */,
                   uint32_t static_base /* this warp's only chunk, or 0xffffffff: chunks from the atomic counter */,
                   uint32_t share /* items of the static chunk (multiple of 32, <= DFS_WCHUNK) */) {
    const uint32_t total = n_tabs ? s_wend[n_tabs - 1] : 0;   // multiple of 32
    const bool solo = static_base != 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    // ---- sub-chunk stream of this warp
    uint32_t c_cur, c_next = 0, sub = 0;
    if (solo) c_cur = static_base;
    else {
        uint32_t c0 = 0, c1 = 0;
        if (lane == 0) { c0 = atomicAdd(chunk_ctr, 1u); c1 = atomicAdd(chunk_ctr, 1u); }
        c_cur = __shfl_sync(0xffffffffu, c0, 0) * DFS_WCHUNK;
        c_next = __shfl_sync(0xffffffffu, c1, 0) * DFS_WCHUNK;
    }
    auto gen = [&]() -> uint32_t {   // base item of the next sub-chunk, or 0xffffffff
        if (solo && 32 * sub >= share) return 0xffffffffu;
        if (sub == DFS_WCHUNK / 32) {
            sub = 0;
            c_cur = c_next;
            uint32_t c = 0;
            if (lane == 0 && c_cur < total) c = atomicAdd(chunk_ctr, 1u);   // consumed 4 sub-chunks from now
            c_next = c_cur < total ? __shfl_sync(0xffffffffu, c, 0) * DFS_WCHUNK : 0xffffffffu;
        }
        const uint32_t b = c_cur + 32 * sub;
        ++sub;
        return (c_cur < total && b < total) ? b : 0xffffffffu;
    };
    // ---- issue the copies of one sub-chunk into a stage
    uint32_t t_is = 0;
    auto issue = [&](uint32_t b, uint32_t st) {
        while (b >= s_wend[t_is]) ++t_is;
        const PassTab T = tabs[t_is];
        const uint32_t q0 = b - (t_is ? s_wend[t_is - 1] : 0);
        const uint32_t sbase = stage_base + st * (DFS_STAGE_F * 16);
        const uint32_t per = T.two ? 4u : 2u;             // entries per item
        const uint32_t e0 = q0 * per;
        const F* V = inV + T.in_off;
        const F* M = inM + T.in_off;
        const F* A = inA + T.in_off;
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j) {
            if (j >= per) break;
            const uint32_t k = j * 32 + lane;             // piece of this table's 32-item region
            const uint32_t q = T.two ? (k >> 2) : (k >> 1), jj = T.two ? (k & 3) : (k & 1);
            const uint32_t slot = 4 * q + (jj ^ ((q >> 1) & 3));
            const uint32_t e = e0 + k;
            const bool in = e < T.in_live;
            const uint32_t sz = in ? 16u : 0u;
            const uint32_t eo = in ? e : 0u;
            cp_async16(sbase + slot * 16, V + eo, sz);
            cp_async16(sbase + (128 + slot) * 16, M + eo, sz);
            if (HAS_A) cp_async16(sbase + (256 + slot) * 16, A + eo, sz);
        }
    };
    uint32_t t_cp = 0;
    uint32_t b_cur = gen();
    if (b_cur != 0xffffffffu) issue(b_cur, 0);
    cp_async_commit();
    uint32_t st = 0;
    while (b_cur != 0xffffffffu) {
        const uint32_t b_next = gen();
        if (b_next != 0xffffffffu) issue(b_next, st ^ 1);
        cp_async_commit();
        cp_async_wait1();
        __syncwarp();
        // ---- this lane's item
        while (b_cur >= s_wend[t_cp]) ++t_cp;
        const PassTab T = tabs[t_cp];
        const uint32_t q = b_cur - (t_cp ? s_wend[t_cp - 1] : 0) + lane;
        // plain shared-memory loads (not volatile asm): the compiler places each next to its use, so only the pair
        // being worked on occupies registers; the stage is not refilled before the __syncwarp at the end of the iteration
        const F* sp = stage_ptr + st * DFS_STAGE_F + 4 * lane;
        const uint32_t sw = (lane >> 1) & 3;
        F xv[4], xm[4], xa[4];
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j) {
            xv[j] = sp[j ^ sw];
            xm[j] = sp[128 + (j ^ sw)];
            xa[j] = HAS_A ? sp[256 + (j ^ sw)] : f_zero();
        }
        if (T.two) {
            F v0, v1, m0, m1, a0 = f_zero(), a1 = f_zero(), ov, om, oa = f_zero();
            dfs_pair<VREAL, HAS_A, NEED_B>(acc1, accb, xv[0], xv[1], xm[0], xm[1], xa[0], xa[1], rk1, v0, m0, a0);
            dfs_pair<VREAL, HAS_A, NEED_B>(acc1, accb, xv[2], xv[3], xm[2], xm[3], xa[2], xa[3], rk1, v1, m1, a1);
            dfs_pair2(acc2, HAS_A, v0, v1, m0, m1, a0, a1, rk2, ov, om, oa);
            if (4 * q < T.in_live) {
                const uint32_t o = T.out_off + q;
                st_f(outV + o, ov);
                st_f(outM + o, om);
                if (HAS_A) st_f(outA + o, oa);
            }
            if (HAS_A) { acc2.s0re = fp_fold(acc2.s0re); acc2.s0im = fp_fold(acc2.s0im); }
        } else {
            // a pair item uses the first two slots of its lane's quad (xv[2..3] are stale shared memory, unused)
            F ov, om, oa = f_zero();
            dfs_pair<VREAL, HAS_A, NEED_B>(acc1, accb, xv[0], xv[1], xm[0], xm[1], xa[0], xa[1], rk1, ov, om, oa);
            if (2 * q < T.in_live) {
                const uint32_t o = T.out_off + q;
                st_f(outV + o, ov);
                st_f(outM + o, om);
                if (HAS_A) st_f(outA + o, oa);
            }
        }
        if (HAS_A) {
            acc1.s0re = fp_fold(acc1.s0re); acc1.s0im = fp_fold(acc1.s0im);
            if (NEED_B) { accb->s1re = fp_fold(accb->s1re); accb->s1im = fp_fold(accb->s1im); }
        }
        __syncwarp();   // every lane is done with this stage: the next iteration's copies may refill it
        b_cur = b_next;
        st ^= 1;
    }
}

// add_term after one more round: at*(1 - prev) (if a previous challenge exists) + tables collapsing now
VP_D F dfs_collapse(F at, const PassCol* __restrict__ cols, uint32_t n_cols, uint32_t which, const F* V, const F* M, const F* A,
                    bool scale, const F& prev, F* claims, bool has_a = true) {
    if (scale) at = f_mul(at, f_sub(f_one(), prev));
    for (uint32_t i = 0; i < n_cols; ++i) {
        const PassCol c = cols[i];
        if (c.which != which) continue;
        F cv = f_zero(), cm = f_zero(), ca = f_zero();
        if (c.n_vals) { cv = ld_one<false>(V + c.off); cm = ld_one<false>(M + c.off); if (has_a) ca = ld_one<false>(A + c.off); }
        at = f_add(at, f_mul_add(cv, cm, ca));
        if (c.claim_slot >= 0) st_f(claims + c.claim_slot, f_strict(cv));
    }
    return at;
}

// Grid barrier for the pass kernel. Only the blocks that still have work take part: the work of a phase only
// shrinks, so block b leaves the kernel for good after the last pass in which b * blockDim < work (it arrives,
// but does not wait). `target` is the cumulative number of arrivals up to and including this pass.
VP_D void pass_arrive(unsigned int* bar) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(bar, 1u);
    }
}
VP_D void pass_wait(unsigned int* bar, unsigned int target) {
    if (threadIdx.x == 0) {
        unsigned int v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
        } while (v < target);
        __threadfence();
    }
    __syncthreads();
}

static constexpr int DFS_THREADS = VP_DFS_THREADS;
// FIRST: what the very first pass of the launch looks like
enum : int { DFS_PLAIN = 0,    // like every other pass (stage B of a sharded phase, stand-alone tables with a known claim)
             DFS_VREAL = 1,    // V is in the base field (circuit values): every GKR phase
             DFS_NEED_B = 2 }; // stand-alone sumcheck: no claim to start from, round 1 also sums p(1) -> *claim0
// Roles. Block 0 is the COORDINATOR: in a pass that needs more than one block it takes no work; it keeps add_term,
// handles the tables that collapse to one value, sums the workers' partial round sums and writes the polynomials --
// all of that while the workers (blocks 1..) are already in the next pass, so none of it sits on the critical path.
// It takes part in the grid barrier only as a gate: it arrives for pass k+1 after it has finished its duties for
// pass k, which bounds its lag to one pass (the partial-sum buffers and the table buffers are double buffered).
// Once a pass fits one block (<= DFS_CHUNK items) block 0 does the remaining passes alone with block barriers only.
template <bool HAS_A, int FIRST>
__global__ void __launch_bounds__(VP_DFS_THREADS, VP_DFS_MINB) k_phase_dfs(DfsArgs p) {
    __shared__ F smem[6 * 32];
    __shared__ uint32_t s_wend[128];
    extern __shared__ __align__(16) unsigned char dfs_dyn_smem[];   // per warp: two stages x 3 tables x 32 quads
    const uint32_t stage_base = (uint32_t)__cvta_generic_to_shared(dfs_dyn_smem) + (threadIdx.x >> 5) * (DFS_WARP_SMEM_F * 16);
    const F* stage_ptr = reinterpret_cast<const F*>(dfs_dyn_smem) + (threadIdx.x >> 5) * DFS_WARP_SMEM_F;
    constexpr int NV = FIRST == DFS_NEED_B ? 5 : 4;   // a1, c1, a2, c2 and (stand-alone, first pass) p1(1) = sum m1*v1 + a1
    const bool coord = blockIdx.x == 0;
    const uint32_t n_workers = gridDim.x - 1;
    constexpr uint32_t WPB = DFS_THREADS / 32;
    // Which workers take part in which pass. A pass uses workers 1..active(work) (see below); `active` is NOT monotone in
    // the work (the share per warp is rounded to 32 items: 2100 items on 8 workers -> 6 of them, 2048 items -> all 8), so a
    // worker may idle in one pass and be needed again later. s_alive[ps] = the largest `active` of this and all later
    // passes: workers 1..s_alive[ps] arrive at pass ps's barrier (working or not), the others have left for good.
    __shared__ uint32_t s_alive[34], s_active[34], s_share[34];
    if (threadIdx.x < 34) {   // (one load per pass, in parallel: this sits in front of the first pass of every launch)
        const uint32_t q = threadIdx.x;
        uint32_t a = 0, sh = DFS_WCHUNK;
        if (q < p.n_passes) {
            const uint32_t work = p.passes[q].work;
            if (work > DFS_SOLO && n_workers != 0) {
                const uint32_t per_warp = (work + n_workers * WPB - 1) / (n_workers * WPB);
                sh = min(DFS_WCHUNK, (per_warp + 31u) & ~31u);
                a = min(n_workers, (work + sh * WPB - 1) / (sh * WPB));
            } else if (work <= DFS_CHUNK && VP_DFS_SOLO_THIN) {
                // block 0 alone: spread the items over its warps as thinly as possible as well (an item is a ~4.5 us
                // dependent chain: 128 items on one warp are four of them back to back, on four warps one)
                sh = min(DFS_WCHUNK, max(32u, ((work + WPB - 1) / WPB + 31u) & ~31u));
            }
        }
        s_alive[q] = a;
        s_active[q] = a;
        s_share[q] = sh;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t mx = 0;
        for (int q = 33; q >= 0; --q) { mx = max(mx, s_alive[q]); s_alive[q] = mx; }
    }
    __syncthreads();
    F at = p.at_init ? *p.at_init : f_zero();
    uint32_t j = 1;       // local round of the pass's first round (= 1 + 2 * ps: every pass but the last has two rounds)
    unsigned int target = 0;
    for (uint32_t ps = 0; ps < p.n_passes; ++ps) {
#define VP_DBG_T(k) do { if (p.dbg && blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); p.dbg[4 * ps + (k)] = t_; } } while (0)
        VP_DBG_T(0);
        const PassDev R = p.passes[ps];
        // How the pass is spread. Small passes are latency bound (one item is ~1250 dependent-ish instructions), so a
        // pass that one sweep of the workers can cover is spread as thinly as possible: every warp gets ONE share of
        // `share` items (a multiple of 32, at most DFS_WCHUNK), on as many workers as that takes. Larger passes hand out
        // DFS_WCHUNK-item chunks from an atomic counter.
        const bool solo = R.work <= DFS_SOLO || n_workers == 0;        // block 0 alone
        // share = roundup32(ceil(work / (workers * warps))) capped at DFS_WCHUNK, active = ceil(work / (share * warps))
        // worker blocks 1..active (tabulated per pass at the top of the kernel)
        const uint32_t share = s_share[ps], active = s_active[ps];
        const bool is_static = solo ? R.work <= DFS_CHUNK : (uint64_t)active * share * WPB >= R.work;
        const uint32_t alive = s_alive[ps];
        if (!coord && blockIdx.x > alive) return;                      // not needed in this or any later pass
        const bool idle = !coord && blockIdx.x > active;               // needed again later: only keeps the barrier count
        const uint32_t ib = R.in_buf, ob = ib ^ 1;
        const uint32_t g1 = p.round_base + j;                          // global round of the pass's first round
        const bool scale1 = g1 >= 2;
        const PassCol* cols = p.cols + R.col_begin;
        F* part = p.partials + (size_t)(ps & 1) * gridDim.x * 6;
        F v[NV];
        if ((!coord && !idle) || (coord && solo)) {
            __syncthreads();
            for (uint32_t i = threadIdx.x; i < R.n_tabs; i += blockDim.x) s_wend[i] = p.tabs[R.tab_begin + i].work_end;
            __syncthreads();
            // the challenges' limbs come pre-split through the kernel parameters
            const ConstK& rk1 = p.rk[2 * ps];
            const ConstK& rk2 = p.rk[2 * ps + 1];
            PassAcc acc1;
            PassAcc2 acc2;
            pacc_init(acc1);
            pacc2_init(acc2);
            PassAccB accb;
            accb.B = psum_zero(); accb.s1re = accb.s1im = 0;
            const F* inV = (ps == 0 && p.v_first) ? p.v_first : p.bufV[ib];
            // static shares when one sweep of the workers covers the pass, chunks from the atomic counter otherwise
            const uint32_t wb = solo ? 0 : blockIdx.x - 1;
            const uint32_t static_base = is_static ? (wb * WPB + (threadIdx.x >> 5)) * share : 0xffffffffu;
            if (FIRST == DFS_VREAL && ps == 0)
                dfs_work<HAS_A, true, false>(acc1, acc2, nullptr, p.tabs + R.tab_begin, R.n_tabs, s_wend, inV, p.bufM[ib], p.bufA[ib],
                                             p.bufV[ob], p.bufM[ob], p.bufA[ob], rk1, rk2, p.chunk_ctr + ps, stage_base, stage_ptr, static_base, share);
            else if (FIRST == DFS_NEED_B && ps == 0)
                dfs_work<HAS_A, false, true>(acc1, acc2, &accb, p.tabs + R.tab_begin, R.n_tabs, s_wend, inV, p.bufM[ib], p.bufA[ib],
                                             p.bufV[ob], p.bufM[ob], p.bufA[ob], rk1, rk2, p.chunk_ctr + ps, stage_base, stage_ptr, static_base, share);
            else
                dfs_work<HAS_A, false, false>(acc1, acc2, nullptr, p.tabs + R.tab_begin, R.n_tabs, s_wend, inV, p.bufM[ib], p.bufA[ib],
                                              p.bufV[ob], p.bufM[ob], p.bufA[ob], rk1, rk2, p.chunk_ctr + ps, stage_base, stage_ptr, static_base, share);
            pacc_finish(acc1, v[0], v[1]);
            pacc2_finish(acc2, v[2], v[3]);
            if (FIRST == DFS_NEED_B) v[NV - 1] = f_add(psum_reduce(accb.B), F{fp_canon(accb.s1re), fp_canon(accb.s1im)});
            if (p.dbg && ps == 0 && threadIdx.x == 0 && blockIdx.x < 1024) {   // per-block finish time + SM id of the first pass
                unsigned long long t_; unsigned int sm_;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
                asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_));
                p.dbg[256 + 2 * blockIdx.x] = t_;
                p.dbg[256 + 2 * blockIdx.x + 1] = sm_;
            }
            block_sum<NV>(v, smem);
        }
        VP_DBG_T(1);
        // tables that were already down to one value join add_term in the pass's first round; their value sits in the
        // IN buffer, which the next pass overwrites: read it before arriving
        if (coord && threadIdx.x == 0)
            at = dfs_collapse(at, cols, R.n_cols, 0, p.bufV[ib], p.bufM[ib], p.bufA[ib], scale1, scale1 ? p.chal[g1 - 2] : f_zero(),
                              p.claims, HAS_A);
        if (!solo) {
            if (!coord && !idle && threadIdx.x == 0) {
#pragma unroll
                for (int k = 0; k < NV; ++k) st_f(part + (size_t)blockIdx.x * 6 + k, v[k]);
            }
            pass_arrive(p.bar);
            target += alive + 1;                                        // workers 1..alive and the coordinator
            if (!coord && blockIdx.x > s_alive[ps + 1]) return;         // no later pass needs this worker: no need to wait
            pass_wait(p.bar, target);
            VP_DBG_T(2);
            if (coord) {
#pragma unroll
                for (int k = 0; k < NV; ++k) v[k] = f_zero();
                for (uint32_t b = 1 + threadIdx.x; b <= active; b += blockDim.x) {
#pragma unroll
                    for (int k = 0; k < NV; ++k) v[k] = f_add(v[k], ld_f_cg(part + (size_t)b * 6 + k));
                }
                block_sum<NV>(v, smem);
            }
        } else __syncthreads();   // this pass's outputs (a table reaching one value) are visible to thread 0
        if (coord && threadIdx.x == 0) {
            // the b slots stay zero here: k_derive_b fills them from the claim chain
            F* o = p.out_poly + 3 * (j - 1);
            const F c1 = f_add(v[1], at);
            st_f(o + 0, v[0]);
            st_f(o + 1, f_zero());
            st_f(o + 2, c1);
            if (FIRST == DFS_NEED_B && ps == 0 && p.claim0) st_f(p.claim0, f_add(c1, v[NV - 1]));   // p(0) + p(1)
            if (R.n_rounds == 2) {
                // tables that reached one value in this pass's first round join in its second round (OUT buffer)
                at = dfs_collapse(at, cols, R.n_cols, 1, p.bufV[ob], p.bufM[ob], p.bufA[ob], true, p.chal[g1 - 1], p.claims, HAS_A);
                st_f(o + 3, v[2]);
                st_f(o + 4, f_zero());
                st_f(o + 5, f_add(v[3], at));
            }
        }
        VP_DBG_T(3);
        j += R.n_rounds;
    }
    if (!coord) return;
    __syncthreads();
    if (threadIdx.x == 0) {
        st_f(p.add_term, at);
        *p.bar = 0;   // every other block has arrived for the last time: ready for the next launch
    }
    for (uint32_t i = threadIdx.x; i < p.n_passes; i += blockDim.x) p.chunk_ctr[i] = 0;
    // final claims: a table alive to the end is down to its level-R value (prover.cpp:494-521); the tables are
    // weakly canonical, what leaves the kernel is canonical
    const F* V = (p.n_passes == 0 && p.v_first) ? p.v_first : p.bufV[p.fin_buf];   // zero rounds: the value was never copied
    for (uint32_t i = threadIdx.x; i < p.n_fin; i += blockDim.x) {
        const FinDesc f = p.fins[i];
        F c;
        if (f.from_claim >= 0) c = ld_one<false>(p.claims + f.from_claim);
        else c = f.n_vals >= 1 ? ld_one<false>(V + f.in_off) : f_zero();
        c = f_strict(c);
        st_f(p.transcript + f.out_idx, c);
        if (p.keep && i == 0) st_f(p.keep, c);
    }
}

// ------------------------------------------------------------------ the b coefficients, from the claim chain
// k_phase_dfs leaves b = 0 in every round polynomial. The verifier's check p(0) + p(1) == claim (verifier.cpp:209,
// 248, 296) holds identically for the honest prover, so b = claim - 2c - a, with the claim chain
//   phase 1 of the top layer: Vres; phase 1 of layer i: the Liu claim of layer i+1 (verifier.cpp:333);
//   phase 2: continues phase 1's chain (verifier.cpp:157-158); Liu: sum_k sig_k * claim_k (verifier.cpp:281-284);
//   next claim = p(r) (verifier.cpp:215,254,302).
// All starting claims are fully folded V values, which do not depend on any b: the chains are independent, one thread each.
struct ChainSeg { uint32_t tr_off, n_rounds, ci; };   // polynomials at tr[tr_off + 3j], challenges chal[ci + j]
struct ChainTerm { uint32_t ci, tr; };                // claim0 += chal[ci] * tr[tr]
struct ChainDesc {
    int32_t claim_tr;            // >= 0: claim0 = tr[claim_tr]; -1: the weighted sum of the terms; -2: *claim_ext
    uint32_t term_begin, n_terms;
    uint32_t seg_begin, n_segs;
};
// One WARP per chain. Within a segment the claims obey claim_{k+1} = r_k*claim_k + d_k with
// d_k = a_k*(r_k^2 - r_k) + c_k*(1 - 2 r_k) (substitute b_k = claim_k - 2c_k - a_k into p_k(r_k)): the lanes compute
// (r_k, d_k) for 32 rounds at a time and a warp prefix scan over the affine maps (m,t)o(m',t') = (m*m', t*m' + t')
// yields every claim_k, hence every b_k, in 5 steps instead of 32 dependent ones.
__global__ void k_derive_b(const ChainDesc* __restrict__ chains, int n_chains, const ChainSeg* __restrict__ segs,
                           const ChainTerm* __restrict__ terms, const F* __restrict__ chal, F* tr, const F* claim_ext) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= n_chains) return;
    const ChainDesc c = chains[i];
    F claim = f_zero();
    if (c.claim_tr >= 0) claim = tr[c.claim_tr];
    else if (c.claim_tr == -2) claim = *claim_ext;
    else {
        for (uint32_t k = lane; k < c.n_terms; k += 32) {
            const ChainTerm t = terms[c.term_begin + k];
            claim = f_mul_add(chal[t.ci], tr[t.tr], claim);
        }
        claim = warp_sum(claim);
        claim.re = __shfl_sync(0xffffffffu, claim.re, 0);
        claim.im = __shfl_sync(0xffffffffu, claim.im, 0);
    }
    for (uint32_t s = 0; s < c.n_segs; ++s) {
        const ChainSeg g = segs[c.seg_begin + s];
        for (uint32_t base = 0; base < g.n_rounds; base += 32) {
            const uint32_t jr = base + lane;
            const bool live = jr < g.n_rounds;
            F* o = tr + g.tr_off + 3 * jr;
            F a = f_zero(), cc = f_zero(), m = f_one(), t = f_zero();   // identity map for idle lanes
            if (live) {
                a = o[0]; cc = o[2];
                const F r = chal[g.ci + jr];
                m = r;
                t = f_mul_add(a, f_sub(f_mul(r, r), r), f_mul(cc, f_sub(f_one(), f_dbl(r))));
            }
            // inclusive scan of the affine maps: after it, lane k holds the map claim_base -> claim_{base+k+1}
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                F pm, pt;
                pm.re = __shfl_up_sync(0xffffffffu, m.re, off); pm.im = __shfl_up_sync(0xffffffffu, m.im, off);
                pt.re = __shfl_up_sync(0xffffffffu, t.re, off); pt.im = __shfl_up_sync(0xffffffffu, t.im, off);
                if (lane >= off) { t = f_mul_add(pt, m, t); m = f_mul(pm, m); }   // (pm,pt) first, then (m,t)
            }
            const F after = f_mul_add(m, claim, t);   // claim_{base+lane+1}
            F before;                                  // claim_{base+lane}
            before.re = __shfl_up_sync(0xffffffffu, after.re, 1);
            before.im = __shfl_up_sync(0xffffffffu, after.im, 1);
            if (lane == 0) before = claim;
            if (live) st_f(o + 1, f_sub(f_sub(before, f_dbl(cc)), a));
            const uint32_t last = min(31u, g.n_rounds - base - 1);
            claim.re = __shfl_sync(0xffffffffu, after.re, last);
            claim.im = __shfl_sync(0xffffffffu, after.im, last);
        }
    }
}

__global__ void k_strict_copy(F* dst, const F* src, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) st_f(dst + i, f_strict(src[i]));
}

// ------------------------------------------------------------------ sharded phases: hand-over between the local
// rounds (stage A, tables block-cyclic over the ranks) and the replicated tail rounds (stage B)
// After the m local rounds every block of a distributed table is down to two stored values; fold them with
// r_m (no pairing: the partner block lives on another rank) and put the block's value into this rank's
// gather record at [base + {0,1,2}*cnt + local_block].
struct FoldOnlyDesc {
    uint32_t in_off;     // local table in the stage-A final buffer
    uint32_t in_live;    // live stored values (<= 2 * n_blocks)
    uint32_t n_blocks;   // local blocks (records written, zero-filled beyond the live ones)
    uint32_t out_base;   // offset (F) of this table's V region in the gather record
    uint32_t cnt;        // region length (max local blocks over ranks)
    uint32_t fold;       // 1: two values per block, fold with r; 0: one value per block (m == 0 never happens; m >= 1)
};
__global__ void k_fold_only(const FoldOnlyDesc* __restrict__ descs, int n_desc, const F* __restrict__ V, const F* __restrict__ M,
                            const F* __restrict__ A, const F* __restrict__ r_ptr, F* __restrict__ rec) {
    const FoldK rk = make_foldk(*r_ptr);
    for (int t = blockIdx.y; t < n_desc; t += gridDim.y) {
        const FoldOnlyDesc d = descs[t];
        for (uint32_t b = blockIdx.x * blockDim.x + threadIdx.x; b < d.cnt; b += gridDim.x * blockDim.x) {
            F v = f_zero(), m = f_zero(), a = f_zero();
            if (b < d.n_blocks && !d.fold) {          // the two-rounds-per-pass kernel leaves one value per block
                if (b < d.in_live) { v = V[d.in_off + b]; m = M[d.in_off + b]; a = A[d.in_off + b]; }
            } else if (b < d.n_blocks) {
                const uint32_t i0 = d.in_off + 2 * b, l0 = 2 * b;
                if (l0 < d.in_live) {
                    const F v0 = V[i0], m0 = M[i0], a0 = A[i0];
                    F v1 = f_zero(), m1 = f_zero(), a1 = f_zero();
                    if (l0 + 1 < d.in_live) { v1 = V[i0 + 1]; m1 = M[i0 + 1]; a1 = A[i0 + 1]; }
                    v = f_fold_k(v0, v1, rk); m = f_fold_k(m0, m1, rk); a = f_fold_k(a0, a1, rk);
                }
            }
            st_f(rec + d.out_base + b, v);
            st_f(rec + d.out_base + d.cnt + b, m);
            st_f(rec + d.out_base + 2 * d.cnt + b, a);
        }
    }
}

// After the all-gather of the per-rank records: build the stage-B tables (block beta of a table came from rank
// (beta mod G == first_r) as its local block beta / G) and add up the per-rank partial scalars (round
// polynomials of the local rounds, add_term, claims of tables that collapsed locally).
struct MergeTab {
    uint32_t rec_base;   // offset of the table's V region inside one rank's record
    uint32_t cnt;        // region length
    uint32_t n_blocks;   // live blocks of the whole table (= live entries of the stage-B table)
    uint32_t out_off;    // stage-B table offset in buffer 0
    uint32_t rev;        // 0: slice s belongs to rank s; 1: to rank G-1-s (phase-2 tables are in reverse instance order)
    uint32_t sb[9];      // slice s holds blocks [sb[s], sb[s+1])
};
struct MergeArgs {
    const F* recv;            // G records of rec_len F
    uint32_t rec_len, G;
    const MergeTab* tabs;
    uint32_t n_tabs;
    uint32_t sc_base;         // offset of the scalar region inside a record
    uint32_t n_poly;          // 3 * local rounds
    uint32_t n_claims;
    F *outV, *outM, *outA;    // stage-B buffers
    F* out_poly;              // transcript slots of rounds 1..m
    F* add_term;              // summed add_term
    F* claims;
};
__global__ void k_shard_merge(MergeArgs p) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    for (uint32_t t = 0; t < p.n_tabs; ++t) {
        const MergeTab T = p.tabs[t];
        for (uint32_t beta = tid; beta < T.n_blocks; beta += stride) {
            uint32_t sl = 0;
            while (sl + 1 < p.G && beta >= T.sb[sl + 1]) ++sl;
            const uint32_t owner = T.rev ? p.G - 1 - sl : sl, q = beta - T.sb[sl];
            const F* rec = p.recv + (size_t)owner * p.rec_len + T.rec_base;
            st_f(p.outV + T.out_off + beta, rec[q]);
            st_f(p.outM + T.out_off + beta, rec[T.cnt + q]);
            st_f(p.outA + T.out_off + beta, rec[2 * T.cnt + q]);
        }
    }
    const uint32_t n_sc = p.n_poly + 1 + p.n_claims;
    for (uint32_t i = tid; i < n_sc; i += stride) {
        F s = f_zero();
        for (uint32_t g = 0; g < p.G; ++g) s = f_add(s, p.recv[(size_t)g * p.rec_len + p.sc_base + i]);
        if (i < p.n_poly) st_f(p.out_poly + i, s);
        else if (i == p.n_poly) st_f(p.add_term, s);
        else st_f(p.claims + (i - p.n_poly - 1), s);
    }
}

// ------------------------------------------------------------------ the same hand-over in ONE kernel over NVLink
// (sharded contexts, default): every rank's exchange buffer is mapped into every other rank of the box (CUDA IPC). The
// kernel (a) stores this rank's record -- the level-m value of each of its blocks, its partial round polynomials, partial
// add_term and locally collapsed claims -- straight into slot `me` of EVERY rank's buffer (peer stores through
// NVSwitch, 16 bytes per thread, coalesced), (b) the last block to finish raises this rank's flag on every peer
// (release at system scope), (c) waits until all ranks' flags for this exchange are up and (d) builds the stage-B
// tables and sums the partial scalars from the local buffer -- what memset + k_fold_only + ncclAllGather +
// k_shard_merge did in four stream operations and one NCCL launch. Flags carry the exchange's sequence number
// (monotonic per lane, the ranks run the same sequence of phases), buffers are double buffered by its parity: a rank
// can be at most one exchange ahead of a peer that is still reading (it needs that peer's next flag to go further).
struct XchgArgs {
    F* peer[8];               // base of every rank's exchange buffer as mapped here (peer[me]: the local one)
    uint32_t world, me, seq;  // this exchange's sequence number (>= 1)
    uint32_t slot_stride;     // entries between two ranks' slots
    uint32_t buf_off[2];      // entry offsets of the two parity buffers inside an exchange buffer
    uint32_t rec_len;
    const FoldOnlyDesc* fo;   // this rank's distributed tables after the local rounds (one value per block)
    uint32_t n_fo;
    const F *V, *M, *A;       // stage-A final buffers
    uint32_t has_a;
    F* sc;                    // this rank's partial scalars (written by the stage-A kernel), zeroed again here
    uint32_t sc_base, n_sc;
    unsigned int* ticket;     // zero at launch, left zero
    uint32_t tag;             // identifies the phase (its transcript offset): every rank must be exchanging the same phase
    unsigned int* err;        // set to 1 if a peer's record carries another tag / sequence number
    MergeArgs mg;             // recv is not read: the kernel merges from the exchange buffer
};
VP_D void st_f_sys(F* p, const F& v) {   // peer memory: plain 128-bit store, ordered by the release below
    asm volatile("st.global.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(v.re), "l"(v.im) : "memory");
}
__global__ void __launch_bounds__(256) k_xchg(XchgArgs p) {
    __shared__ bool s_last;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    const uint32_t par = p.seq & 1u;
    const size_t slot = (size_t)p.buf_off[par] + (size_t)p.me * p.slot_stride;
    // ---- (a) push: one pass over the record, every element stored to all ranks
    for (uint32_t t = 0; t < p.n_fo; ++t) {
        const FoldOnlyDesc d = p.fo[t];
        for (uint32_t i = tid; i < 3 * d.cnt; i += stride) {
            const uint32_t which = i / d.cnt, b = i - which * d.cnt;
            F v = f_zero();
            if (b < d.in_live && b < d.n_blocks) {
                const F* src = which == 0 ? p.V : which == 1 ? p.M : p.A;
                if (which < 2 || p.has_a) v = f_strict(src[d.in_off + b]);
            }
            for (uint32_t q = 0; q < p.world; ++q) st_f_sys(p.peer[q] + slot + d.out_base + i, v);
        }
    }
    for (uint32_t i = tid; i < p.n_sc; i += stride) {
        const F v = p.sc[i];
        for (uint32_t q = 0; q < p.world; ++q) st_f_sys(p.peer[q] + slot + p.sc_base + i, v);
    }
    if (tid == 0)   // what this record belongs to (checked by every receiver)
        for (uint32_t q = 0; q < p.world; ++q) st_f_sys(p.peer[q] + slot + p.rec_len, F{p.tag, p.seq});
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last) {
        // ---- (b) every block's stores are done (each fenced before its ticket): raise the flags, clear the scalars
        __threadfence_system();
        if (threadIdx.x < p.world) {
            unsigned int* flag = reinterpret_cast<unsigned int*>(p.peer[threadIdx.x]) + p.me;
            asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(p.seq) : "memory");
        }
        for (uint32_t i = threadIdx.x; i < p.n_sc; i += blockDim.x) p.sc[i] = f_zero();
        if (threadIdx.x == 0) *p.ticket = 0;
    }
    // ---- (c) wait for every rank's record of this exchange
    if (threadIdx.x < p.world) {
        const unsigned int* flag = reinterpret_cast<const unsigned int*>(p.peer[p.me]) + threadIdx.x;
        unsigned int v;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        } while ((int)(v - p.seq) < 0);
        __threadfence_system();
    }
    __syncthreads();
    // ---- (d) merge from the local buffer (written by the peers: bypass L1)
    const F* recv = p.peer[p.me] + p.buf_off[par];
    if (tid < p.world) {   // the ranks must walk the same sequence of phases per lane: a record of another phase is an error
        const F t = ld_f_cg(recv + (size_t)tid * p.slot_stride + p.rec_len);
        if (t.re != p.tag || t.im != p.seq) atomicExch(p.err, 1u);
    }
    const MergeArgs& m = p.mg;
    for (uint32_t t = 0; t < m.n_tabs; ++t) {
        const MergeTab T = m.tabs[t];
        for (uint32_t beta = tid; beta < T.n_blocks; beta += stride) {
            uint32_t sl = 0;
            while (sl + 1 < m.G && beta >= T.sb[sl + 1]) ++sl;
            const uint32_t owner = T.rev ? m.G - 1 - sl : sl, q = beta - T.sb[sl];
            const F* rec = recv + (size_t)owner * p.slot_stride + T.rec_base;
            st_f(m.outV + T.out_off + beta, ld_f_cg(rec + q));
            st_f(m.outM + T.out_off + beta, ld_f_cg(rec + T.cnt + q));
            st_f(m.outA + T.out_off + beta, ld_f_cg(rec + 2 * T.cnt + q));
        }
    }
    const uint32_t n_sc = m.n_poly + 1 + m.n_claims;
    for (uint32_t i = tid; i < n_sc; i += stride) {
        F s = f_zero();
        for (uint32_t g = 0; g < m.G; ++g) s = f_add(s, ld_f_cg(recv + (size_t)g * p.slot_stride + m.sc_base + i));
        if (i < m.n_poly) st_f(m.out_poly + i, s);
        else if (i == m.n_poly) st_f(m.add_term, s);
        else st_f(m.claims + (i - m.n_poly - 1), s);
    }
}

// ------------------------------------------------------------------ K8 / K9: MLE evaluation = dot with eq
// prover.cpp:99-129 (Vres) and :532-540 (inner_prod against eq(r_liu,.), verifier.cpp:368-369).
__global__ void __launch_bounds__(256)
k_dot_eq(const F* __restrict__ X, uint32_t begin, uint32_t n, EqTab eq, F* __restrict__ out, F* partials, unsigned int* counter,
         size_t ss) {
    __shared__ F smem[32];
    X += (size_t)blockIdx.z * n;   // statement b's slice of the layer (a batch lays the statements' layers end to end)
    eq = stmt_at(eq, ss); out = stmt_at(out, ss); partials = stmt_at(partials, ss); counter = stmt_at(counter, ss);
    Acc acc = acc_zero();
    F run = f_zero();
    int pending = 0;
    for (uint32_t i = begin + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        acc_mad(acc, ld_f(X + i), eq_at(eq, i));
        if (++pending == 8) { run = f_add(run, acc_reduce(acc)); acc = acc_zero(); pending = 0; }
    }
    F v[1] = {f_add(run, acc_reduce(acc))};
    if (grid_sum<1>(v, smem, partials, counter) && threadIdx.x == 0) st_f(out, v[0]);
}
__global__ void __launch_bounds__(256)
k_dot(const F* __restrict__ X, const F* __restrict__ Y, uint32_t n, F* __restrict__ out, F* partials,
      unsigned int* counter) {
    __shared__ F smem[32];
    Acc acc = acc_zero();
    F run = f_zero();
    int pending = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        acc_mad(acc, ld_f(X + i), ld_f(Y + i));
        if (++pending == 8) { run = f_add(run, acc_reduce(acc)); acc = acc_zero(); pending = 0; }
    }
    F v[1] = {f_add(run, acc_reduce(acc))};
    if (grid_sum<1>(v, smem, partials, counter) && threadIdx.x == 0) st_f(out, v[0]);
}

// out[i] = sum over the G ranks of recv[g * n + i] (sharded vp_verify: partial sums of every rank)
__global__ void k_sum_ranks_vec(const F* __restrict__ recv, uint32_t G, uint32_t n, F* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    F s = f_zero();
    for (uint32_t g = 0; g < G; ++g) s = f_add(s, recv[(size_t)g * n + i]);
    st_f(out + i, s);
}
// sum of one field element per rank (sharded Vres / input MLE)
__global__ void k_sum_ranks(const F* __restrict__ recv, uint32_t G, uint32_t stride, F* __restrict__ out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        F s = f_zero();
        for (uint32_t g = 0; g < G; ++g) s = f_add(s, recv[(size_t)g * stride]);
        st_f(out, s);
    }
}

// ------------------------------------------------------------------ V1 / V2: the verifier's linear-time sums
// (SURVEY 8(f) N2) verifier.cpp:63-113 predicatePhase1/2 and the gr sum of verifyLiu :311-323. The protocol driver
// (round checks, getFinalValue, the Liu check) stays on the host; these kernels produce the O(#gates) quantities it
// needs. They are written against the circuit wiring directly (buckets of gates, plain dadId lists) and use only the
// canonical field routines: none of the prover's tables, CSRs or lazy/weak primitives are involved, so the
// verifier's accept is an independent check of the prover's messages.
// A batch (vp_verify_fs_bound_batch) runs statement b in blockIdx.z == b: its eq tables, challenges, partial sums and
// outputs sit `ss` bytes after statement b - 1's (stmt_at); gates, buckets and Liu segments are shared.
struct VfGate {          // one template gate in bucket order
    uint32_t g0, u0, lv0;
    uint32_t l_c;        // binary: source layer l; unary: index of the gate's constant (== g0)
};
struct VfBucket {
    uint32_t begin, cnt;     // gates [begin, begin + cnt) of the sorted array
    uint32_t kind;           // 0: sum t; 1: sum t*c; 2: sum t and, second output, sum t*c (Addc: coeff and bias); 3: binary, sum t*beta_v[lv]
    uint32_t D;              // binary: subset size of one instance (lv = (K-1-k)*D + lv0)
};
// partial[(bucket * gridDim.x + blockIdx.x) * 2 + {0,1}]
__global__ void __launch_bounds__(256)
k_verify_sums(const VfBucket* __restrict__ buckets, const VfGate* __restrict__ gates, const uint8_t* __restrict__ is_assert,
              const F* __restrict__ cst, uint32_t S_pre, uint32_t S_cur, uint32_t K, EqTab eqg, EqTab equ, EqTab eqv,
              const F* __restrict__ assert_r, F* __restrict__ partial, uint32_t k_begin, uint32_t k_end, size_t ss) {
    __shared__ F smem[2 * 32];
    eqg = stmt_at(eqg, ss); equ = stmt_at(equ, ss); eqv = stmt_at(eqv, ss); assert_r = stmt_at(assert_r, ss); partial = stmt_at(partial, ss);
    const VfBucket B = buckets[blockIdx.y];
    const uint64_t total = (uint64_t)B.cnt * (k_end - k_begin);   // sharded: this rank's slice of the instances
    F acc[2] = {f_zero(), f_zero()};
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t kq = (uint32_t)(w / B.cnt), j = (uint32_t)(w - (uint64_t)kq * B.cnt), k = k_begin + kq;
        const VfGate G = gates[B.begin + j];
        F bg = eq_at(eqg, k * S_cur + G.g0);
        if (is_assert && is_assert[G.g0]) bg = f_mul(bg, *assert_r);
        F t = f_mul(bg, eq_at(equ, k * S_pre + G.u0));
        if (B.kind == 3) t = f_mul(t, eq_at(eqv, (K - 1 - k) * B.D + G.lv0));
        if (B.kind == 1) t = f_mul(t, cst[G.l_c]);
        acc[0] = f_add(acc[0], t);
        if (B.kind == 2) acc[1] = f_add(acc[1], f_mul(t, cst[G.l_c]));
    }
    block_sum<2>(acc, smem);
    if (threadIdx.x == 0) {
        F* dst = partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 2;
        st_f(dst, acc[0]);
        st_f(dst + 1, acc[1]);
    }
}
// out[bucket * 2 + {0,1}] = sum over the gx partials of the bucket
__global__ void k_verify_reduce(const F* __restrict__ partial, uint32_t gx, F* __restrict__ out, size_t ss) {
    __shared__ F smem[2 * 32];
    partial = stmt_at(partial, ss); out = stmt_at(out, ss);
    F acc[2] = {f_zero(), f_zero()};
    for (uint32_t b = threadIdx.x; b < gx; b += blockDim.x) {
        acc[0] = f_add(acc[0], partial[((size_t)blockIdx.x * gx + b) * 2]);
        acc[1] = f_add(acc[1], partial[((size_t)blockIdx.x * gx + b) * 2 + 1]);
    }
    block_sum<2>(acc, smem);
    if (threadIdx.x == 0) { st_f(out + 2 * blockIdx.x, acc[0]); st_f(out + 2 * blockIdx.x + 1, acc[1]); }
}
// gr of verifyLiu: segment 0 = sum_u beta_g'[u]*beta_u'[u] over layer pre (beta_g' = sig[0]*eq(r_u,.), beta_u' = eq(r_liu,.));
// segment 1+q = sum_g eq_q[g] * beta_u'[dadId_q[g]] over the K-instance subset of source layer j_q (eq_q carries sig[j-pre]).
struct VfLiuSeg {
    const uint32_t* dadId;   // one instance, null for segment 0
    uint32_t D;              // subset size of one instance (segment 0: S_pre)
    uint32_t eq_id;          // index into eqs (segment 0: unused)
    uint32_t pad;
};
__global__ void __launch_bounds__(256)
k_verify_gr(const VfLiuSeg* __restrict__ segs, const EqTab* __restrict__ eqs, EqTab eq_g0, EqTab eq_rl, uint32_t S_pre, uint32_t K,
            F* __restrict__ partial, uint32_t k_begin, uint32_t k_end, size_t ss) {
    __shared__ F smem[2 * 32];
    eq_g0 = stmt_at(eq_g0, ss); eq_rl = stmt_at(eq_rl, ss); partial = stmt_at(partial, ss);
    const VfLiuSeg Sg = segs[blockIdx.y];
    // sharded: this rank's slice [k_begin, k_end) of the instances; a subset segment runs in reverse instance order
    const uint64_t w_lo = (uint64_t)Sg.D * (blockIdx.y == 0 ? k_begin : K - k_end), total = (uint64_t)Sg.D * (blockIdx.y == 0 ? k_end : K - k_begin);
    F acc[2] = {f_zero(), f_zero()};
    for (uint64_t w = w_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (uint64_t)gridDim.x * blockDim.x) {
        if (blockIdx.y == 0) acc[0] = f_add(acc[0], f_mul(eq_at(eq_g0, (uint32_t)w), eq_at(eq_rl, (uint32_t)w)));
        else {
            const uint32_t kk = (uint32_t)(w / Sg.D), g0 = (uint32_t)(w - (uint64_t)kk * Sg.D), k = K - 1 - kk;
            acc[0] = f_add(acc[0], f_mul(eq_at(stmt_at(eqs[Sg.eq_id], ss), (uint32_t)w), eq_at(eq_rl, k * S_pre + Sg.dadId[g0])));
        }
    }
    block_sum<2>(acc, smem);
    if (threadIdx.x == 0) {
        F* dst = partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 2;
        st_f(dst, acc[0]);
        st_f(dst + 1, acc[1]);
    }
}

// ------------------------------------------------------------------ self-test of the device-only arithmetic paths
// field.cuh compiles for host and device, but the carry-chain routines (fp_reduce_ut_weak, a96_add) and mul32/mad32
// take inline-PTX paths on the device that the host build (tests/native) cannot exercise. vp_selftest_field runs them
// on caller-provided operands so that tests can feed the edge values (0, 1, p-1, p, limb boundaries) that random
// transcripts practically never contain, and compare with big-integer arithmetic.
__global__ void k_selftest_field(int op, const F* __restrict__ a, const F* __restrict__ b, const F* __restrict__ c,
                                 F* __restrict__ out, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (op == 2 || op == 6) {   // lazy dot products over all n operands, one thread
        if (i != 0) return;
        CAcc s = cacc_zero();
        for (uint32_t j = 0; j < n; ++j) {
            if (op == 2) cacc_mad(s, make_lop(a[j].re, a[j].im), make_ropd(b[j]));
            else cacc_mad_real(s, f_diff2p(a[j], b[j]), c[j].re);
        }
        st_f(out, cacc_reduce(s));
        return;
    }
    if (i >= n) return;
    F r = f_zero();
    switch (op) {
        case 0: r = f_fold_w(a[i], f_diff2p(a[i], b[i]), make_constk(c[i])); break;
        case 1: r = f_fold_w_real(a[i].re, fp_weak(b[i].re + P - a[i].re), make_constk(c[i])); break;
        case 3: r = F{fp_reduce_ut_weak(a[i].re, a[i].im, b[i].re), fp_weak(b[i].im)}; break;
        case 4: r = f_mul_add_w(a[i], b[i], c[i]); break;
        case 5: r = f_mad_real_w(c[i], a[i], b[i].re); break;
        case 7: r = f_fold_w(a[i], f_diff_w(a[i], b[i]), make_constk(c[i])); break;
        default: break;
    }
    st_f(out + i, r);
}

// ------------------------------------------------------------------ misc
// SplitMix64-filled random table entries (limbs uniform in [0,p) by rejection), config C2.
__global__ void k_fill_random(F* __restrict__ T, uint32_t n, uint64_t seed) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t s = seed + 0x9E3779B97F4A7C15ULL * (2ULL * i + 1);
    uint64_t out[2];
    for (int k = 0; k < 2; ++k) {
        uint64_t z;
        do {
            s += 0x9E3779B97F4A7C15ULL;
            z = s;
            z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
            z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
            z = (z ^ (z >> 31)) >> 3;
        } while (z >= P);
        out[k] = z;
    }
    st_f(T + i, F{out[0], out[1]});
}

}  // namespace vp
