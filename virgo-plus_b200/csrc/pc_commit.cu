// Commit phase of Virgo's polynomial commitment on the device -- see pc_commit.h for what it replaces.
//
// What commit_private_array computes (poly_commit.h:41-124, constants.h: 2^6 slices, code rate 2^-5):
//   the array of 2^b values is cut into 64 slices of n = 2^(b-6) consecutive values; every slice is interpolated
//   (inverse FFT of size n) and re-evaluated on the 32x larger domain (FFT of size N = 32 n) -> l_eval[s][0..N);
//   a 65th slice holds the mask polynomial (the GKR prover passes a single zero: all zeros);
//   leaf i (i < N/2) = SHA3 chain over the 65 slices of  H( l_eval[s][i] | l_eval[s][i + N/2] | previous )  (fri.cpp:97-126);
//   an array-heap Merkle tree over the N/2 leaves with H(left | right) (merkle_tree.cpp:7-51); the root is the commitment.
//
// How it is laid out here:
//   * ONE table of the N powers of the N-th root of unity (k_pc_twiddles: product of the precomputed 2^b-th powers
//     over the set bits of the exponent); every other twiddle (n-th roots, inverse roots, coset shifts) is an index
//     into it.
//   * The size-N evaluation of a degree < n polynomial is 32 size-n transforms on the cosets of the n-th roots:
//     l_eval[s][32 k + c] = NTT_n( coef_i * w_N^(c i) )[k]   (1/32 of the butterflies of a zero-padded size-N FFT).
//   * inverse transform = decimation in frequency (natural in, bit-reversed out), forward = decimation in time
//     (bit-reversed in, natural out): no permutation pass. Up to 2^11 points of a transform are processed in shared
//     memory (11 stages per pass); longer transforms add one global pass per extra stage.
//   * SHA3-256 of a 64-byte block is one Keccak-f[1600] permutation (rate 136 bytes); one thread per leaf walks the
//     65-slice chain with coalesced 16-byte loads, one thread per tree node hashes a level.
// All arithmetic is the canonical F_{p^2} arithmetic of field.cuh: exact, hence bit-identical to the reference's
// packed-AVX FFT whatever the butterfly order.
#include "pc_commit.h"
#include "keccak.cuh"

#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

namespace vp {

#define PCK(call)                                                                                                  \
    do {                                                                                                           \
        cudaError_t e_ = (call);                                                                                   \
        if (e_ != cudaSuccess) throw std::runtime_error(std::string(#call) + " failed: " + cudaGetErrorString(e_)); \
    } while (0)

static constexpr int PC_LOG_SLICES = 6, PC_SLICES = 64, PC_LOG_RATE = 5, PC_COSETS = 32;
static constexpr int PC_SMEM_LOG = 11;   // points of one transform held in shared memory (32 KB)

VP_D F pc_ld(const F* p) {
    const ulonglong2 t = *reinterpret_cast<const ulonglong2*>(p);
    return F{t.x, t.y};
}
VP_D void pc_st(F* p, const F& v) { *reinterpret_cast<ulonglong2*>(p) = make_ulonglong2(v.re, v.im); }

struct PcPow {
    F sq[32];   // sq[b] = w_N^(2^b)
};
// tw[t] = w_N^t  (fieldElement::getRootOfUnity, fieldElement.cpp:237-249, gives w_N; L_group of fri.cpp:62-67 is this table)
__global__ void k_pc_twiddles(F* __restrict__ tw, uint32_t N, PcPow pw) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N) return;
    F r = f_one();
    for (uint32_t b = 0; (t >> b) != 0; ++b)
        if ((t >> b) & 1u) r = f_mul(r, pw.sq[b]);
    pc_st(tw + t, r);
}

// the committed array, zero-padded to 2^log_len
__global__ void k_pc_pad(const F* __restrict__ src, size_t n_valid, F* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        pc_st(dst + i, i < n_valid ? pc_ld(src + i) : f_zero());
}

// ---- inverse transform (RS_polynomial.cpp:155-220): DIF with the inverse n-th root, natural in, bit-reversed out.
// One global stage over `batch` transforms of size n stored back to back: stage s pairs p and p + half, half = n >> (s+1).
__global__ void k_pc_dif_stage(F* __restrict__ a, uint32_t log_n, uint32_t s, size_t total_pairs, const F* __restrict__ tw, uint32_t log_N,
                               uint32_t tw_shift /* log2(N / transform size): w_size = w_N^(2^tw_shift) */) {
    const uint32_t lh = log_n - s - 1, half = 1u << lh, N = 1u << log_N;
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < total_pairs; w += (size_t)gridDim.x * blockDim.x) {
        const size_t t = w >> (log_n - 1);                       // transform
        const uint32_t q = (uint32_t)(w & ((1u << (log_n - 1)) - 1));
        const uint32_t j = q & (half - 1), p = ((q >> lh) << (lh + 1)) | j;
        F* x = a + (t << log_n);
        const F u = pc_ld(x + p), v = pc_ld(x + p + half);
        const uint32_t e = j << s;                               // exponent of w_n^-1
        pc_st(x + p, f_add(u, v));
        pc_st(x + p + half, f_mul(f_sub(u, v), pc_ld(tw + ((N - (e << tw_shift)) & (N - 1)))));
    }
}
// The last min(log_n, 11) DIF stages of every transform in shared memory, then the scaling by 1/n (inv_n = n^(p-2)).
// One block per chunk of m = 2^log_m points (a chunk never straddles two transforms).
__global__ void __launch_bounds__(512) k_pc_intt_smem(F* __restrict__ a, uint32_t log_n, uint32_t log_m, const F* __restrict__ tw, uint32_t log_N,
                                                       F inv_n, uint32_t tw_shift) {
    extern __shared__ __align__(16) unsigned char pc_smem[];
    F* sh = reinterpret_cast<F*>(pc_smem);
    const uint32_t m = 1u << log_m, N = 1u << log_N;
    F* x = a + ((size_t)blockIdx.x << log_m);
    for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) sh[i] = pc_ld(x + i);
    __syncthreads();
    for (uint32_t s = log_n - log_m; s < log_n; ++s) {           // global stage index: half = n >> (s+1) < m
        const uint32_t lh = log_n - s - 1, half = 1u << lh;
        for (uint32_t q = threadIdx.x; q < m / 2; q += blockDim.x) {
            const uint32_t j = q & (half - 1), p = ((q >> lh) << (lh + 1)) | j;
            const F u = sh[p], v = sh[p + half];
            const uint32_t e = j << s;
            sh[p] = f_add(u, v);
            sh[p + half] = f_mul(f_sub(u, v), pc_ld(tw + ((N - (e << tw_shift)) & (N - 1))));
        }
        __syncthreads();
    }
    for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) pc_st(x + i, f_mul(sh[i], inv_n));
}

// ---- forward transform on coset c (RS_polynomial.cpp:26-153 evaluates the same polynomial on all N points):
// DIT, bit-reversed in (what the inverse transform left), natural out.
// First min(log_n, 11) stages in shared memory. coef: [64][n] bit-reversed coefficients. One block per
// (chunk, coset, slice). If direct != 0 (log_n <= 11) the result goes straight to l_eval[s][32 k + c], else to the work
// buffer work[(s * 32 + c) * n + p].
// Coefficient i of slice sl sits at coef[sl * slice_stride + i * in_stride + in_off] (private / public array: stride 1;
// the quotient h of commit_public: the odd positions of the bit-reversed 2n coefficients of l*q).
__global__ void __launch_bounds__(512) k_pc_ntt_smem(const F* __restrict__ coef, uint32_t log_n, uint32_t log_m, const F* __restrict__ tw,
                                                      uint32_t log_N, F* __restrict__ out, int direct, size_t slice_stride, uint32_t in_stride,
                                                      uint32_t in_off) {
    extern __shared__ __align__(16) unsigned char pc_smem[];
    F* sh = reinterpret_cast<F*>(pc_smem);
    const uint32_t m = 1u << log_m, n = 1u << log_n, N = 1u << log_N;
    const uint32_t chunk = blockIdx.x, c = blockIdx.y, sl = blockIdx.z, base = chunk << log_m;
    const F* x = coef + (size_t)sl * slice_stride + (size_t)base * in_stride + in_off;
    for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) {
        const uint32_t p = base + i, ci = log_n ? __brev(p) >> (32 - log_n) : 0u;   // coefficient index held at position p
        const F v = pc_ld(x + (size_t)i * in_stride);
        sh[i] = (c == 0 || log_n == 0) ? v : f_mul(v, pc_ld(tw + (((uint64_t)c * ci) & (N - 1))));   // coef_i * w_N^(c i)
    }
    __syncthreads();
    for (uint32_t s = 0; s < log_m; ++s) {
        const uint32_t half = 1u << s;
        for (uint32_t q = threadIdx.x; q < m / 2; q += blockDim.x) {
            const uint32_t j = q & (half - 1), p = ((q >> s) << (s + 1)) | j;
            const F u = sh[p], v = f_mul(sh[p + half], pc_ld(tw + ((size_t)j << (log_N - s - 1))));   // w_n^(j n / 2^(s+1))
            sh[p] = f_add(u, v);
            sh[p + half] = f_sub(u, v);
        }
        __syncthreads();
    }
    if (direct) {
        F* o = out + ((size_t)sl << log_N);
        for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) pc_st(o + (((size_t)(base + i)) << PC_LOG_RATE) + c, sh[i]);
    } else {
        F* o = out + ((((size_t)sl << PC_LOG_RATE) + c) << log_n) + base;
        for (uint32_t i = threadIdx.x; i < m; i += blockDim.x) pc_st(o + i, sh[i]);
    }
    (void)n;
}
// g <= 6 consecutive global DIT stages s0 .. s0+g-1 in ONE pass over the work buffer. Those stages only couple positions that
// differ in bits s0 .. s0+g-1, so position p = top << (s0+g) | mid << s0 | lo splits every transform into independent 2^g-point
// columns of stride 2^s0; a block takes 32 neighbouring columns (32 consecutive lo: 512-byte rows) into shared memory
// (2^g x 32 elements <= 32 KB), runs the g stages there and writes the tile back -- or, in the last group, to
// l_eval[slice][32 p + coset].
static constexpr int PC_DIT_GROUP = 6, PC_DIT_COLS_LOG = 5;
__global__ void __launch_bounds__(256) k_pc_dit_group(F* __restrict__ work, uint32_t log_n, uint32_t s0, uint32_t g, const F* __restrict__ tw,
                                                       uint32_t log_N, F* __restrict__ l_eval, int last) {
    __shared__ __align__(16) F sh[(1 << PC_DIT_GROUP) << PC_DIT_COLS_LOG];
    const uint32_t tiles_log = log_n - g - PC_DIT_COLS_LOG;                     // tiles per transform
    const size_t t = (size_t)blockIdx.x >> tiles_log;                          // transform = slice * 32 + coset
    const uint32_t tile = blockIdx.x & ((1u << tiles_log) - 1);
    const uint32_t lo_bits = s0 - PC_DIT_COLS_LOG;                              // tile = top << lo_bits | (lo >> 5)
    const uint32_t top = tile >> lo_bits, lo0 = (tile & ((1u << lo_bits) - 1)) << PC_DIT_COLS_LOG;
    const uint32_t base = (top << (s0 + g)) | lo0, cols = 1u << PC_DIT_COLS_LOG, count = cols << g;
    F* x = work + (t << log_n);
    for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) sh[i] = pc_ld(x + (base | ((i >> PC_DIT_COLS_LOG) << s0) | (i & (cols - 1))));
    __syncthreads();
    for (uint32_t k = 0; k < g; ++k) {
        const uint32_t s = s0 + k;
        for (uint32_t q = threadIdx.x; q < count / 2; q += blockDim.x) {
            const uint32_t w = q & (cols - 1), mq = q >> PC_DIT_COLS_LOG, jl = mq & ((1u << k) - 1), m0 = ((mq >> k) << (k + 1)) | jl;
            const uint32_t i0 = (m0 << PC_DIT_COLS_LOG) | w, i1 = i0 + (cols << k);
            const uint32_t j = (jl << s0) | lo0 | w;                            // p & (2^s - 1)
            const F u = sh[i0], v = f_mul(sh[i1], pc_ld(tw + ((size_t)j << (log_N - s - 1))));
            sh[i0] = f_add(u, v);
            sh[i1] = f_sub(u, v);
        }
        __syncthreads();
    }
    if (last) {
        F* o = l_eval + ((t >> PC_LOG_RATE) << log_N) + (t & (PC_COSETS - 1));
        for (uint32_t i = threadIdx.x; i < count; i += blockDim.x)
            pc_st(o + ((size_t)(base | ((i >> PC_DIT_COLS_LOG) << s0) | (i & (cols - 1))) << PC_LOG_RATE), sh[i]);
    } else {
        for (uint32_t i = threadIdx.x; i < count; i += blockDim.x) pc_st(x + (base | ((i >> PC_DIT_COLS_LOG) << s0) | (i & (cols - 1))), sh[i]);
    }
}

// ---- commit_public_array (poly_commit.h:126-349): products of the two codewords on the 2n-th roots, the quotient
// polynomial's oracle values
// lq[s][j] = l_eval[s][16 j] * q_eval[s][16 j], j < 2n  (the 2n evaluations of l*q that determine it: degree < 2n - 1)
__global__ void k_pc_lq(const F* __restrict__ l_eval, const F* __restrict__ q_eval, uint32_t log_n, uint32_t log_N, F* __restrict__ lq, size_t total) {
    const uint32_t step_log = log_N - log_n - 1;
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (size_t)gridDim.x * blockDim.x) {
        const size_t sl = w >> (log_n + 1), j = w & (((size_t)1 << (log_n + 1)) - 1);
        const size_t at = (sl << log_N) + (j << step_log);
        pc_st(lq + w, f_mul(pc_ld(l_eval + at), pc_ld(q_eval + at)));
    }
}
// lqc: bit-reversed coefficients of l*q per slice (2n each): coefficient 0 at position 0, coefficient n (= h_0) at position 1.
// all_sum[s] = n (lq_0 + h_0) (poly_commit.h:330); per point x = w_N^j:
//   vow[(j mod N/2) << 7 | s << 1 | (j >= N/2)] = (l q - (x^n - 1) h - (lq_0 + h_0)) * n * x^-1        (:303-323)
// A block produces 16 leaves of the virtual oracle (2048 elements, 32 KB contiguous): it reads, for every slice and both
// halves, 16 consecutive codeword positions (256-byte segments), and writes the tile through shared memory so that the
// interleaved output goes out in full lines.
static constexpr int PC_VOW_LEAVES_LOG = 4;
__global__ void __launch_bounds__(256) k_pc_vow(const F* __restrict__ l_eval, const F* __restrict__ q_eval, const F* __restrict__ h_eval,
                                                 const F* __restrict__ lqc, const F* __restrict__ tw, uint32_t log_n, uint32_t log_N,
                                                 F* __restrict__ vow, F* __restrict__ all_sum) {
    __shared__ __align__(16) F sh[(2 * PC_SLICES) << PC_VOW_LEAVES_LOG];
    const uint32_t N = 1u << log_N, n = 1u << log_n, half = N >> 1, leaves = 1u << PC_VOW_LEAVES_LOG;
    const uint32_t j0 = blockIdx.x << PC_VOW_LEAVES_LOG;
    const F n_fe{(u64)n, 0};
    for (uint32_t i = threadIdx.x; i < (2 * PC_SLICES) << PC_VOW_LEAVES_LOG; i += blockDim.x) {
        const uint32_t jj = i & (leaves - 1), hf = (i >> PC_VOW_LEAVES_LOG) & 1u, sl = i >> (PC_VOW_LEAVES_LOG + 1);
        const uint32_t j = j0 + jj + hf * half;
        const size_t w = ((size_t)sl << log_N) + j;
        const F* c = lqc + ((size_t)sl << (log_n + 1));
        const F c0 = f_add(pc_ld(c), pc_ld(c + 1));
        if (j == 0) pc_st(all_sum + sl, f_mul(c0, n_fe));
        const F x_n = pc_ld(tw + (((size_t)j << log_n) & (N - 1)));                    // (w_N^n)^j
        const F inv_x = f_mul(n_fe, pc_ld(tw + ((N - j) & (N - 1))));                    // n * w_N^-j
        const F lqv = f_mul(pc_ld(l_eval + w), pc_ld(q_eval + w));
        const F g = f_sub(lqv, f_mul(f_sub(x_n, f_one()), pc_ld(h_eval + w)));
        sh[(jj << (PC_LOG_SLICES + 1)) | (sl << 1) | hf] = f_mul(f_sub(g, c0), inv_x);
    }
    __syncthreads();
    F* o = vow + ((size_t)j0 << (PC_LOG_SLICES + 1));
    for (uint32_t i = threadIdx.x; i < (2 * PC_SLICES) << PC_VOW_LEAVES_LOG; i += blockDim.x) pc_st(o + i, sh[i]);
}

// fri.cpp:69-96: the 64 codewords of a commitment interleaved as pairs of opposite points, out[(j << 7) | (s << 1) | h] =
// eval[s][j + h N/2] -- what witness_rs_codeword_interleaved holds. Same tiling as k_pc_vow: 16 leaves (32 KB) per block.
__global__ void __launch_bounds__(256) k_pc_interleave(const F* __restrict__ eval, uint32_t log_N, F* __restrict__ out) {
    __shared__ __align__(16) F sh[(2 * PC_SLICES) << PC_VOW_LEAVES_LOG];
    const uint32_t half = 1u << (log_N - 1), leaves = 1u << PC_VOW_LEAVES_LOG, j0 = blockIdx.x << PC_VOW_LEAVES_LOG;
    for (uint32_t i = threadIdx.x; i < (2 * PC_SLICES) << PC_VOW_LEAVES_LOG; i += blockDim.x) {
        const uint32_t jj = i & (leaves - 1), hf = (i >> PC_VOW_LEAVES_LOG) & 1u, sl = i >> (PC_VOW_LEAVES_LOG + 1);
        sh[(jj << (PC_LOG_SLICES + 1)) | (sl << 1) | hf] = pc_ld(eval + ((size_t)sl << log_N) + j0 + jj + hf * half);
    }
    __syncthreads();
    F* o = out + ((size_t)j0 << (PC_LOG_SLICES + 1));
    for (uint32_t i = threadIdx.x; i < (2 * PC_SLICES) << PC_VOW_LEAVES_LOG; i += blockDim.x) pc_st(o + i, sh[i]);
}

// ---- SHA3-256 of a 64-byte block (my_hhash.h:27-33 -> XKCP SHA3_256; FIPS 202): one Keccak-f[1600] permutation (keccak.cuh)
VP_D void pc_sha3_64(const uint64_t (&msg)[8], uint64_t (&dig)[4]) { sha3_256_64(msg, dig); }

// fri.cpp:97-126: leaf i = chain over the slices; slice 64 (the mask) is all zero for the GKR prover's zero mask
__global__ void __launch_bounds__(128) k_pc_leaf_hash(const F* __restrict__ l_eval, uint32_t log_N, uint64_t* __restrict__ leaf, int mask_is_zero) {
    const uint32_t half = 1u << (log_N - 1);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= half) return;
    uint64_t h[4] = {0, 0, 0, 0};
    for (int s = 0; s <= PC_SLICES; ++s) {
        uint64_t msg[8];
        if (s == PC_SLICES && mask_is_zero) { msg[0] = msg[1] = msg[2] = msg[3] = 0; }
        else {
            const F x = pc_ld(l_eval + ((size_t)s << log_N) + i), y = pc_ld(l_eval + ((size_t)s << log_N) + i + half);
            msg[0] = x.re; msg[1] = x.im; msg[2] = y.re; msg[3] = y.im;
        }
        msg[4] = h[0]; msg[5] = h[1]; msg[6] = h[2]; msg[7] = h[3];
        pc_sha3_64(msg, h);
    }
    uint64_t* o = leaf + (size_t)i * 4;
    o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
}
// merkle_tree.cpp:39-50: one level of the array heap: node lvl + i = H(node 2(lvl + i) | node 2(lvl + i) + 1)
// (blockIdx.y: one of several trees, tree_stride words apart)
__global__ void __launch_bounds__(128) k_pc_merkle_level(uint64_t* __restrict__ tree, uint32_t lvl, size_t tree_stride) {
    tree += blockIdx.y * tree_stride;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= lvl) return;
    const uint64_t* c = tree + (size_t)(2 * (lvl + i)) * 4;
    uint64_t msg[8], h[4];
#pragma unroll
    for (int k = 0; k < 8; ++k) msg[k] = c[k];
    pc_sha3_64(msg, h);
    uint64_t* o = tree + (size_t)(lvl + i) * 4;
    o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
}
// the top of the tree (levels of <= 128 nodes) in one block
__global__ void __launch_bounds__(128) k_pc_merkle_top(uint64_t* __restrict__ tree, uint32_t first_lvl, size_t tree_stride) {
    tree += blockIdx.y * tree_stride;
    for (uint32_t lvl = first_lvl; lvl >= 1; lvl >>= 1) {
        const uint32_t i = threadIdx.x;
        if (i < lvl) {
            const uint64_t* c = tree + (size_t)(2 * (lvl + i)) * 4;
            uint64_t msg[8], h[4];
#pragma unroll
            for (int k = 0; k < 8; ++k) msg[k] = c[k];
            pc_sha3_64(msg, h);
            uint64_t* o = tree + (size_t)(lvl + i) * 4;
            o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
        }
        __syncthreads();
    }
}

// ---- FRI commit phase (fri.cpp:289-418). A level stores the 64 codewords of M points as pairs of opposite points:
// point k of slice j at (k mod M/2) << 7 | j << 1 | (k >= M/2), so that leaf i of the level's tree is 2 KB of consecutive
// memory. One thread folds the two pairs (i, i + M/2) and (i + M/4, i + 3M/4) of one slice into the pair (i, i + M/4) of
// the next level: g[i] = ((a + b) + r w_M^-i (a - b)) / 2 -- two 32-byte loads, one 32-byte store per thread, a warp covers
// 1 KB of each of the two source leaves.
__global__ void k_pc_fri_fold(const F* __restrict__ prev, uint32_t log_M, const F* __restrict__ tw, uint32_t log_N, F r_half, F inv2,
                              F* __restrict__ out, size_t total) {
    const uint32_t N = 1u << log_N, quarter = 1u << (log_M - 2), sh = log_N - log_M;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const uint32_t i = (uint32_t)(t >> PC_LOG_SLICES), j = (uint32_t)(t & (PC_SLICES - 1));
        F v[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t k = i + h * quarter;
            const F* src = prev + (((size_t)k << (PC_LOG_SLICES + 1)) | ((size_t)j << 1));
            const F a = pc_ld(src), b = pc_ld(src + 1);
            const F inv_mu = pc_ld(tw + ((N - (k << sh)) & (N - 1)));                  // w_M^-k
            v[h] = f_add(f_mul(inv2, f_add(a, b)), f_mul(f_mul(r_half, inv_mu), f_sub(a, b)));
        }
        F* dst = out + (((size_t)i << (PC_LOG_SLICES + 1)) | ((size_t)j << 1));
        pc_st(dst, v[0]);
        pc_st(dst + 1, v[1]);
    }
}
// fri.cpp:383-404: leaf i of a level = chain over the 64 pairs of the leaf, then the (zero) pair of the mask codeword
__global__ void __launch_bounds__(128) k_pc_fri_leaf_hash(const F* __restrict__ code, uint32_t n_leaves, uint64_t* __restrict__ leaf) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_leaves) return;
    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(code + ((size_t)i << (PC_LOG_SLICES + 1)));
    uint64_t h[4] = {0, 0, 0, 0};
    for (int s = 0; s <= PC_SLICES; ++s) {
        uint64_t msg[8];
        if (s == PC_SLICES) { msg[0] = msg[1] = msg[2] = msg[3] = 0; }
        else {
            const ulonglong2 x = src[2 * s], y = src[2 * s + 1];
            msg[0] = x.x; msg[1] = x.y; msg[2] = y.x; msg[3] = y.y;
        }
        msg[4] = h[0]; msg[5] = h[1]; msg[6] = h[2]; msg[7] = h[3];
        pc_sha3_64(msg, h);
    }
    uint64_t* o = leaf + (size_t)i * 4;
    o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
}
// The levels lie back to back and a leaf is 128 consecutive elements, so the leaves of ALL levels form one array: global leaf
// g of level l (local index g - goff(l), goff(l) = N/2 - (N >> (l+1))) starts at code + 128 g. Hashing the levels of several
// steps in one launch matters for small codewords, where a level's 65-permutation chains are latency-bound.
__global__ void __launch_bounds__(128) k_pc_fri_leaf_hash_all(const F* __restrict__ code, uint32_t g_begin, uint32_t g_end, uint32_t log_N,
                                                              uint64_t* __restrict__ tree) {
    const uint32_t g = g_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= g_end) return;
    const uint32_t half_N = 1u << (log_N - 1), d = half_N - g;                    // N >> (l+2) < d <= N >> (l+1)
    const uint32_t l = log_N - 1 - (32 - __clz(d - 1));                          // ceil(log2 d) = 32 - clz(d - 1)  (d >= 16)
    const uint32_t leaves = 1u << (log_N - l - 2), goff = half_N - (2u * leaves);
    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(code + ((size_t)g << (PC_LOG_SLICES + 1)));
    uint64_t h[4] = {0, 0, 0, 0};
    for (int s = 0; s <= PC_SLICES; ++s) {
        uint64_t msg[8];
        if (s == PC_SLICES) { msg[0] = msg[1] = msg[2] = msg[3] = 0; }
        else {
            const ulonglong2 x = src[2 * s], y = src[2 * s + 1];
            msg[0] = x.x; msg[1] = x.y; msg[2] = y.x; msg[3] = y.y;
        }
        msg[4] = h[0]; msg[5] = h[1]; msg[6] = h[2]; msg[7] = h[3];
        pc_sha3_64(msg, h);
    }
    uint64_t* o = tree + ((size_t)2 * goff + leaves + (g - goff)) * 4;            // level l's heap starts at node 2 goff(l)
    o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
}
// pass `hgt` of all levels' trees at once: blockIdx.y = level first + y; in level l the nodes [c, 2c), c = leaves_l >> hgt,
// are hashed from their children if c > 128 (the last <= 128-node part of every tree is k_pc_fri_tree_top_all's)
__global__ void __launch_bounds__(128) k_pc_fri_tree_pass_all(uint64_t* __restrict__ tree, uint32_t log_N, uint32_t first, uint32_t hgt) {
    const uint32_t l = first + blockIdx.y;
    const uint32_t leaves = 1u << (log_N - l - 2), c = leaves >> hgt, i = blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= 128 || i >= c) return;
    uint64_t* t = tree + ((size_t)(1u << log_N) - ((size_t)(1u << log_N) >> l)) * 4;
    const uint64_t* ch = t + (size_t)(2 * (c + i)) * 4;
    uint64_t msg[8], h[4];
#pragma unroll
    for (int k = 0; k < 8; ++k) msg[k] = ch[k];
    pc_sha3_64(msg, h);
    uint64_t* o = t + (size_t)(c + i) * 4;
    o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
}
// one block per level: node 0 zeroed, then the levels of <= 128 nodes
__global__ void __launch_bounds__(128) k_pc_fri_tree_top_all(uint64_t* __restrict__ tree, uint32_t log_N, uint32_t first) {
    const uint32_t l = first + blockIdx.x;
    const uint32_t leaves = 1u << (log_N - l - 2);
    uint64_t* t = tree + ((size_t)(1u << log_N) - ((size_t)(1u << log_N) >> l)) * 4;
    if (threadIdx.x < 4) t[threadIdx.x] = 0;
    for (uint32_t lvl = min(leaves / 2, 128u); lvl >= 1; lvl >>= 1) {
        const uint32_t i = threadIdx.x;
        if (i < lvl) {
            const uint64_t* c = t + (size_t)(2 * (lvl + i)) * 4;
            uint64_t msg[8], h[4];
#pragma unroll
            for (int k = 0; k < 8; ++k) msg[k] = c[k];
            pc_sha3_64(msg, h);
            uint64_t* o = t + (size_t)(lvl + i) * 4;
            o[0] = h[0]; o[1] = h[1]; o[2] = h[2]; o[3] = h[3];
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ driver
struct PcCommit {
    int device = 0, log_len = 0, log_n = 0, log_N = 0;
    size_t n = 0, N = 0;
    F *tw = nullptr, *coef = nullptr, *work = nullptr, *l_eval = nullptr;
    uint64_t* tree = nullptr;        // N/2 * 2 nodes of 32 bytes; leaves at [N/2, N)
    // commit_public (allocated on first use): the public array's codewords, l*q coefficients, h's codewords, the
    // virtual oracle, the second tree, all_sum
    F *q_eval = nullptr, *lqc = nullptr, *h_eval = nullptr, *vow = nullptr, *all_sum = nullptr;
    uint64_t* tree_h = nullptr;
    // FRI commit phase: the levels back to back (level l: 64 * (N >> (l+1)) elements, (N >> (l+1)) tree nodes)
    F* fri_code = nullptr;
    uint64_t* fri_tree = nullptr;
    int fri_step = -1;               // next step; -1: no virtual oracle yet
    F inv_2n;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool tw_ready = false;
    uint64_t launches = 0;
    F inv_n;
};

static F host_pow(F x, unsigned __int128 e) {
    F r = f_one();
    while (e) {
        if (e & 1) r = f_mul(r, x);
        x = f_mul(x, x);
        e >>= 1;
    }
    return r;
}

PcCommit* pc_create(int device, int log_len) {
    if (log_len < PC_LOG_SLICES || log_len > 30) throw std::runtime_error("polynomial commitment: log_len must be in [6, 30]");
    PcCommit* p = new PcCommit();
    try {
        p->device = device;
        p->log_len = log_len;
        p->log_n = log_len - PC_LOG_SLICES;
        p->log_N = p->log_n + PC_LOG_RATE;
        p->n = (size_t)1 << p->log_n;
        p->N = (size_t)1 << p->log_N;
        PCK(cudaSetDevice(device));
        PCK(cudaMalloc(&p->tw, p->N * sizeof(F)));
        PCK(cudaMalloc(&p->coef, (PC_SLICES * p->n) * sizeof(F)));
        if (p->log_n > PC_SMEM_LOG) PCK(cudaMalloc(&p->work, (size_t)PC_SLICES * PC_COSETS * p->n * sizeof(F)));
        PCK(cudaMalloc(&p->l_eval, (size_t)(PC_SLICES + 1) * p->N * sizeof(F)));
        PCK(cudaMalloc(&p->tree, p->N * 32));
        PCK(cudaEventCreate(&p->e0));
        PCK(cudaEventCreate(&p->e1));
        const F nn{(u64)p->n, 0};
        p->inv_n = host_pow(nn, (unsigned __int128)P - 2);   // RS_polynomial.cpp:211
        p->inv_2n = host_pow(F{(u64)(2 * p->n), 0}, (unsigned __int128)P - 2);
        PCK(cudaFuncSetAttribute(k_pc_intt_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(F) << PC_SMEM_LOG)));
        PCK(cudaFuncSetAttribute(k_pc_ntt_smem, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(F) << PC_SMEM_LOG)));
    } catch (...) {
        pc_destroy(p);
        throw;
    }
    return p;
}
void pc_destroy(PcCommit* p) {
    if (!p) return;
    cudaSetDevice(p->device);
    cudaFree(p->tw); cudaFree(p->coef); cudaFree(p->work); cudaFree(p->l_eval); cudaFree(p->tree);
    cudaFree(p->q_eval); cudaFree(p->lqc); cudaFree(p->h_eval); cudaFree(p->vow); cudaFree(p->all_sum); cudaFree(p->tree_h);
    cudaFree(p->fri_code); cudaFree(p->fri_tree);
    if (p->e0) cudaEventDestroy(p->e0);
    if (p->e1) cudaEventDestroy(p->e1);
    delete p;
}
size_t pc_slice_size(const PcCommit* p) { return p->N; }
uint64_t pc_launches(const PcCommit* p) { return p->launches; }

static inline unsigned pc_grid(size_t work, unsigned threads, unsigned cap = 148 * 16) {
    return (unsigned)std::max<size_t>(1, std::min<size_t>((work + threads - 1) / threads, cap));
}

// twiddles (once), then: zero-padded copy -> 64 inverse transforms -> 32 coset transforms per slice -> eval[0 .. 64 N)
static void pc_twiddles(PcCommit* p, cudaStream_t st) {
    if (p->tw_ready) return;   // w_N = the order-2^62 element of fieldElement.cpp:240-241 squared 62 - log_N times
    F w{2147483648ULL, 1033321771269002680ULL};
    for (int i = 0; i < 62 - p->log_N; ++i) w = f_mul(w, w);
    PcPow pw;
    for (int b = 0; b < 32; ++b) { pw.sq[b] = w; w = f_mul(w, w); }
    k_pc_twiddles<<<pc_grid(p->N, 256, 1u << 30), 256, 0, st>>>(p->tw, (uint32_t)p->N, pw);
    ++p->launches;
    p->tw_ready = true;
}
// forward transforms on the 32 cosets of every slice: coefficients (bit-reversed) at src[sl * slice_stride + i * in_stride + in_off]
static void pc_extend(PcCommit* p, const F* src, size_t slice_stride, uint32_t in_stride, uint32_t in_off, F* eval, cudaStream_t st) {
    const uint32_t log_n = (uint32_t)p->log_n, log_N = (uint32_t)p->log_N, log_m = std::min<uint32_t>(log_n, PC_SMEM_LOG);
    const unsigned threads = (unsigned)std::max<size_t>(32, std::min<size_t>(512, ((size_t)1 << log_m) / 2));
    const bool direct = log_n <= PC_SMEM_LOG;
    dim3 grid((unsigned)(1u << (log_n - log_m)), PC_COSETS, PC_SLICES);
    k_pc_ntt_smem<<<grid, threads, sizeof(F) << log_m, st>>>(src, log_n, log_m, p->tw, log_N, direct ? eval : p->work, direct ? 1 : 0, slice_stride,
                                                            in_stride, in_off);
    ++p->launches;
    if (!direct) {
        for (uint32_t s0 = log_m; s0 < log_n;) {                   // up to 6 stages per pass
            const uint32_t g = std::min<uint32_t>(PC_DIT_GROUP, log_n - s0);
            const size_t blocks = ((size_t)PC_SLICES * PC_COSETS) << (log_n - g - PC_DIT_COLS_LOG);
            k_pc_dit_group<<<(unsigned)blocks, 256, 0, st>>>(p->work, log_n, s0, g, p->tw, log_N, eval, s0 + g == log_n ? 1 : 0);
            ++p->launches;
            s0 += g;
        }
    }
}
// `count` inverse transforms of size 2^log_t stored back to back in buf (in place; natural in, bit-reversed out, scaled)
static void pc_inverse(PcCommit* p, F* buf, uint32_t log_t, size_t count, F inv, cudaStream_t st) {
    const uint32_t log_N = (uint32_t)p->log_N, log_m = std::min<uint32_t>(log_t, PC_SMEM_LOG), tw_shift = log_N - log_t;
    const size_t total = count << log_t;
    for (uint32_t s = 0; s + log_m < log_t; ++s) {
        k_pc_dif_stage<<<pc_grid(total / 2, 256), 256, 0, st>>>(buf, log_t, s, total / 2, p->tw, log_N, tw_shift);
        ++p->launches;
    }
    const unsigned threads = (unsigned)std::max<size_t>(32, std::min<size_t>(512, ((size_t)1 << log_m) / 2));
    k_pc_intt_smem<<<(unsigned)(total >> log_m), threads, sizeof(F) << log_m, st>>>(buf, log_t, log_m, p->tw, log_N, inv, tw_shift);
    ++p->launches;
}
static void pc_encode(PcCommit* p, const F* d_array, size_t n_valid, F* eval, cudaStream_t st) {
    const size_t total = (size_t)PC_SLICES << p->log_n;
    if (n_valid > total) throw std::runtime_error("polynomial commitment: array longer than 2^log_len");
    pc_twiddles(p, st);
    k_pc_pad<<<pc_grid(total, 256), 256, 0, st>>>(d_array, n_valid, p->coef, total);
    ++p->launches;
    pc_inverse(p, p->coef, (uint32_t)p->log_n, PC_SLICES, p->inv_n, st);
    pc_extend(p, p->coef, p->n, 1, 0, eval, st);
    PCK(cudaMemsetAsync(eval + ((size_t)PC_SLICES << p->log_N), 0, p->N * sizeof(F), st));   // the zero mask's codeword
}
// leaves + tree over eval[65][N] (mask slice zero) -> tree (array heap), root to the host
static void pc_tree_levels(PcCommit* p, uint64_t* tree, uint32_t n_leaves, cudaStream_t st);
static void pc_merkle(PcCommit* p, const F* eval, uint64_t* tree, cudaStream_t st) {
    const uint32_t half = (uint32_t)(p->N / 2);
    PCK(cudaMemsetAsync(tree, 0, 64, st));   // nodes 0 and 1 (node 1 is overwritten: there are always >= 16 leaves)
    k_pc_leaf_hash<<<(half + 127) / 128, 128, 0, st>>>(eval, (uint32_t)p->log_N, tree + (size_t)half * 4, 1);
    ++p->launches;
    pc_tree_levels(p, tree, half, st);
}
// the inner nodes of an array heap whose n_leaves (a power of two >= 2) leaves are in place (n_trees such heaps,
// tree_stride words apart, in the same launches)
static int pc_tree_levels_raw(uint64_t* tree, uint32_t n_leaves, cudaStream_t st, uint32_t n_trees = 1, size_t tree_stride = 0) {
    int launches = 0;
    uint32_t lvl = n_leaves / 2;
    for (; lvl > 128; lvl >>= 1) {
        k_pc_merkle_level<<<dim3((lvl + 127) / 128, n_trees), 128, 0, st>>>(tree, lvl, tree_stride);
        ++launches;
    }
    if (lvl >= 1) {
        k_pc_merkle_top<<<dim3(1, n_trees), 128, 0, st>>>(tree, lvl, tree_stride);
        ++launches;
    }
    return launches;
}
static void pc_tree_levels(PcCommit* p, uint64_t* tree, uint32_t n_leaves, cudaStream_t st) {
    p->launches += (uint64_t)pc_tree_levels_raw(tree, n_leaves, st);
}

// ---- Merkle root of a word vector (the statement digest, see pc_commit.h): leaf j = H(words [8j, 8j + 8)), zero past the
// end. One thread per leaf; a block of 128 leaves then climbs min(7, log2 leaves) levels in shared memory and leaves its
// subtree root at its place in the array heap, so that k_pc_merkle_level / k_pc_merkle_top only see the upper levels
// (a tree of 2^21 leaves: 8 launches instead of 16). The per-level hashes are the same ones either way.
__global__ void __launch_bounds__(128) k_pc_vec_leaves(const uint64_t* __restrict__ words, size_t n_words, uint32_t log_leaves,
                                                       uint32_t climb, uint64_t* __restrict__ tree, size_t tree_stride) {
    __shared__ uint64_t sh[128][4];
    words += blockIdx.y * n_words;   // vector blockIdx.y of a batch: the vectors lie end to end, each tree tree_stride words
    tree += blockIdx.y * tree_stride;
    const uint32_t t = threadIdx.x, width = 1u << climb;
    const size_t leaf = (size_t)blockIdx.x * width + t;
    if (t < width) {
        uint64_t msg[8], h[4];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const size_t w = leaf * 8 + (size_t)k;
            msg[k] = w < n_words ? words[w] : 0;
        }
        pc_sha3_64(msg, h);
#pragma unroll
        for (int k = 0; k < 4; ++k) sh[t][k] = h[k];
    }
    __syncthreads();
    for (uint32_t w = width / 2; w >= 1; w >>= 1) {
        uint64_t msg[8], h[4];
        if (t < w) {
#pragma unroll
            for (int k = 0; k < 4; ++k) { msg[k] = sh[2 * t][k]; msg[4 + k] = sh[2 * t + 1][k]; }
            pc_sha3_64(msg, h);
        }
        __syncthreads();
        if (t < w)
#pragma unroll
            for (int k = 0; k < 4; ++k) sh[t][k] = h[k];
        __syncthreads();
    }
    if (t < 4) tree[(((size_t)1 << (log_leaves - climb)) + blockIdx.x) * 4 + t] = sh[0][t];
}

static uint32_t pc_vector_log_leaves(size_t n_words) {
    uint32_t k = 0;
    while (((size_t)8 << k) < n_words) ++k;
    return k;
}
size_t pc_vector_root_scratch(size_t n_words) {   // nodes 0 .. 2^(k - climb + 1) - 1 of the heap: the leaf level itself is never stored
    const uint32_t k = pc_vector_log_leaves(n_words);
    return (size_t)64 << (k - std::min<uint32_t>(k, 7));
}
int pc_vector_root(const uint64_t* d_words, size_t n_words, uint64_t* d_scratch, uint8_t* d_root, cudaStream_t st, uint32_t n_vec,
                   size_t root_stride) {
    const uint32_t k = pc_vector_log_leaves(n_words), climb = std::min<uint32_t>(k, 7);
    if (k - climb > 31) throw std::runtime_error("vector root: more than 2^38 leaves");
    if (n_vec < 1 || n_vec > 65535) throw std::runtime_error("vector root: 1 to 65535 vectors per pass");
    const size_t blocks = (size_t)1 << (k - climb), tree_words = pc_vector_root_scratch(n_words) / 8;
    k_pc_vec_leaves<<<dim3((unsigned)blocks, n_vec), 128, 0, st>>>(d_words, n_words, k, climb, d_scratch, tree_words);
    int launches = 1 + pc_tree_levels_raw(d_scratch, (uint32_t)blocks, st, n_vec, tree_words);
    PCK(cudaGetLastError());
    if (n_vec == 1) PCK(cudaMemcpyAsync(d_root, d_scratch + 4, 32, cudaMemcpyDeviceToDevice, st));
    else PCK(cudaMemcpy2DAsync(d_root, root_stride, d_scratch + 4, tree_words * 8, 32, n_vec, cudaMemcpyDeviceToDevice, st));
    return launches;
}

float pc_commit(PcCommit* p, const F* d_array, size_t n_valid, cudaStream_t st, uint8_t root[32]) {
    PCK(cudaSetDevice(p->device));
    PCK(cudaEventRecord(p->e0, st));
    pc_encode(p, d_array, n_valid, p->l_eval, st);
    pc_merkle(p, p->l_eval, p->tree, st);
    PCK(cudaEventRecord(p->e1, st));
    PCK(cudaGetLastError());
    PCK(cudaMemcpyAsync(root, p->tree + 4, 32, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
    float ms = 0;
    PCK(cudaEventElapsedTime(&ms, p->e0, p->e1));
    return ms;
}

// commit_public_array (poly_commit.h:126-349) for zero masks, after pc_commit on the same object (needs l_eval):
// q_eval = the public array encoded like the private one; per slice the 2n coefficients of l*q from its values on the
// 2n-th roots; h = the upper n coefficients, extended to all N points; the virtual oracle and all_sum; the Merkle
// commitment of h_eval_arr (fri::request_init_commit(.., 1)).
float pc_commit_public(PcCommit* p, const F* d_pub, size_t n_valid, cudaStream_t st, uint8_t root_h[32], F all_sum_host[65]) {
    PCK(cudaSetDevice(p->device));
    const uint32_t log_n = (uint32_t)p->log_n, log_N = (uint32_t)p->log_N;
    if (!p->q_eval) {
        PCK(cudaMalloc(&p->q_eval, (size_t)(PC_SLICES + 1) * p->N * sizeof(F)));
        PCK(cudaMalloc(&p->h_eval, (size_t)(PC_SLICES + 1) * p->N * sizeof(F)));
        PCK(cudaMalloc(&p->vow, (size_t)PC_SLICES * p->N * sizeof(F)));
        PCK(cudaMalloc(&p->lqc, (size_t)PC_SLICES * 2 * p->n * sizeof(F)));
        PCK(cudaMalloc(&p->all_sum, (PC_SLICES + 1) * sizeof(F)));
        PCK(cudaMalloc(&p->tree_h, p->N * 32));
    }
    PCK(cudaEventRecord(p->e0, st));
    pc_encode(p, d_pub, n_valid, p->q_eval, st);
    const size_t n_lq = (size_t)PC_SLICES << (log_n + 1);
    k_pc_lq<<<pc_grid(n_lq, 256), 256, 0, st>>>(p->l_eval, p->q_eval, log_n, log_N, p->lqc, n_lq);
    ++p->launches;
    pc_inverse(p, p->lqc, log_n + 1, PC_SLICES, p->inv_2n, st);
    // h's coefficient j (natural) is coefficient n + j of l*q = position (bitrev(j) << 1) | 1 of the bit-reversed output
    pc_extend(p, p->lqc, 2 * p->n, 2, 1, p->h_eval, st);
    PCK(cudaMemsetAsync(p->h_eval + ((size_t)PC_SLICES << log_N), 0, p->N * sizeof(F), st));
    PCK(cudaMemsetAsync(p->all_sum, 0, (PC_SLICES + 1) * sizeof(F), st));
    k_pc_vow<<<(unsigned)((p->N / 2) >> PC_VOW_LEAVES_LOG), 256, 0, st>>>(p->l_eval, p->q_eval, p->h_eval, p->lqc, p->tw, log_n, log_N, p->vow, p->all_sum);
    ++p->launches;
    pc_merkle(p, p->h_eval, p->tree_h, st);
    p->fri_step = 0;
    PCK(cudaEventRecord(p->e1, st));
    PCK(cudaGetLastError());
    PCK(cudaMemcpyAsync(root_h, p->tree_h + 4, 32, cudaMemcpyDeviceToHost, st));
    if (all_sum_host) PCK(cudaMemcpyAsync(all_sum_host, p->all_sum, (PC_SLICES + 1) * sizeof(F), cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
    float ms = 0;
    PCK(cudaEventElapsedTime(&ms, p->e0, p->e1));
    return ms;
}
void pc_export_public(PcCommit* p, cudaStream_t st, F* h_eval, F* vow, uint8_t* leaf_hash, uint8_t* tree) {
    PCK(cudaSetDevice(p->device));
    if (!p->q_eval) throw std::runtime_error("polynomial commitment: export before commit_public");
    if (h_eval) PCK(cudaMemcpyAsync(h_eval, p->h_eval, (size_t)(PC_SLICES + 1) * p->N * sizeof(F), cudaMemcpyDeviceToHost, st));
    if (vow) PCK(cudaMemcpyAsync(vow, p->vow, (size_t)PC_SLICES * p->N * sizeof(F), cudaMemcpyDeviceToHost, st));
    if (leaf_hash) PCK(cudaMemcpyAsync(leaf_hash, p->tree_h + (p->N / 2) * 4, (p->N / 2) * 32, cudaMemcpyDeviceToHost, st));
    if (tree) PCK(cudaMemcpyAsync(tree, p->tree_h, p->N * 32, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
}

// ---- FRI commit phase
int pc_fri_steps(const PcCommit* p) { return p->log_n; }
int pc_fri_steps_done(const PcCommit* p) { return p->fri_step < 0 ? 0 : p->fri_step; }
static inline size_t pc_fri_offset(const PcCommit* p, int lvl) { return p->N - (p->N >> lvl); }   // sum of N >> (l+1), l < lvl
void pc_fri_restart(PcCommit* p) {
    if (p->fri_step < 0) throw std::runtime_error("polynomial commitment: FRI commit phase before commit_public");
    p->fri_step = 0;
}
// one fold (+ leaf hashes + tree if with_tree) on the stream; no synchronisation
static void pc_fri_step_async(PcCommit* p, F r, cudaStream_t st, bool with_tree) {
    if (p->fri_step < 0) throw std::runtime_error("polynomial commitment: FRI commit phase before commit_public");
    if (p->fri_step >= p->log_n) throw std::runtime_error("polynomial commitment: the FRI commit phase is finished (32 points per slice left)");
    if (!p->fri_code) {
        PCK(cudaMalloc(&p->fri_code, (size_t)PC_SLICES * p->N * sizeof(F)));
        PCK(cudaMalloc(&p->fri_tree, p->N * 32));
    }
    const int s = p->fri_step;
    const uint32_t log_M = (uint32_t)(p->log_N - s);
    const size_t quarter = ((size_t)1 << log_M) / 4;
    const F* prev = s == 0 ? p->vow : p->fri_code + PC_SLICES * pc_fri_offset(p, s - 1);
    F* out = p->fri_code + PC_SLICES * pc_fri_offset(p, s);
    uint64_t* tree = p->fri_tree + pc_fri_offset(p, s) * 4;
    const F inv2{(P + 1) / 2, 0};
    const size_t total = quarter << PC_LOG_SLICES;
    k_pc_fri_fold<<<pc_grid(total, 256), 256, 0, st>>>(prev, log_M, p->tw, (uint32_t)p->log_N, f_mul(r, inv2), inv2, out, total);
    ++p->launches;
    ++p->fri_step;
    if (!with_tree) return;
    PCK(cudaMemsetAsync(tree, 0, 64, st));
    k_pc_fri_leaf_hash<<<(unsigned)((quarter + 127) / 128), 128, 0, st>>>(out, (uint32_t)quarter, tree + quarter * 4);
    ++p->launches;
    pc_tree_levels(p, tree, (uint32_t)quarter, st);
}
// several steps whose challenges are all known: the folds one after the other (each needs only the previous level's
// codewords), then the leaf chains of ALL new levels in one launch and their trees side by side
static void pc_fri_steps_batched(PcCommit* p, const F* r, int n, cudaStream_t st) {
    const int first = p->fri_step;
    for (int k = 0; k < n; ++k) pc_fri_step_async(p, r[k], st, false);
    const uint32_t log_N = (uint32_t)p->log_N;
    const uint32_t g_begin = (uint32_t)(pc_fri_offset(p, first) / 2), g_end = (uint32_t)(pc_fri_offset(p, first + n) / 2);
    k_pc_fri_leaf_hash_all<<<(g_end - g_begin + 127) / 128, 128, 0, st>>>(p->fri_code, g_begin, g_end, log_N, p->fri_tree);
    ++p->launches;
    const uint32_t leaves0 = 1u << (log_N - first - 2);
    for (uint32_t hgt = 1; (leaves0 >> hgt) > 128; ++hgt) {
        dim3 grid(((leaves0 >> hgt) + 127) / 128, (unsigned)n);
        k_pc_fri_tree_pass_all<<<grid, 128, 0, st>>>(p->fri_tree, log_N, (uint32_t)first, hgt);
        ++p->launches;
    }
    k_pc_fri_tree_top_all<<<(unsigned)n, 128, 0, st>>>(p->fri_tree, log_N, (uint32_t)first);
    ++p->launches;
}
// n steps from the current one; roots: n * 32 bytes on the host
float pc_fri_steps_run(PcCommit* p, const F* r, int n, cudaStream_t st, uint8_t* roots) {
    PCK(cudaSetDevice(p->device));
    const int first = p->fri_step;
    PCK(cudaEventRecord(p->e0, st));
    if (n >= 2 && !getenv("VP_FRI_STEPWISE")) pc_fri_steps_batched(p, r, n, st);
    else for (int k = 0; k < n; ++k) pc_fri_step_async(p, r[k], st, true);
    PCK(cudaEventRecord(p->e1, st));
    PCK(cudaGetLastError());
    for (int k = 0; k < n; ++k)
        PCK(cudaMemcpyAsync(roots + (size_t)k * 32, p->fri_tree + pc_fri_offset(p, first + k) * 4 + 4, 32, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
    float ms = 0;
    PCK(cudaEventElapsedTime(&ms, p->e0, p->e1));
    return ms;
}
void pc_fri_export(PcCommit* p, cudaStream_t st, int lvl, F* code, uint8_t* tree) {
    PCK(cudaSetDevice(p->device));
    if (lvl < 0 || lvl >= p->fri_step) throw std::runtime_error("polynomial commitment: FRI level not computed");
    const size_t m = p->N >> (lvl + 1);
    if (code) PCK(cudaMemcpyAsync(code, p->fri_code + PC_SLICES * pc_fri_offset(p, lvl), PC_SLICES * m * sizeof(F), cudaMemcpyDeviceToHost, st));
    if (tree) PCK(cudaMemcpyAsync(tree, p->fri_tree + pc_fri_offset(p, lvl) * 4, m * 32, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
}

// which = 0: l_eval (after pc_commit), 1: h_eval_arr (after pc_commit_public) -> out[64 N] in the layout of
// fri::witness_rs_codeword_interleaved[which]. Staged in the FRI level buffer (free at both points of the protocol: the FRI
// steps come after the exports).
void pc_export_interleaved(PcCommit* p, cudaStream_t st, int which, F* out) {
    PCK(cudaSetDevice(p->device));
    if (which == 1 && !p->q_eval) throw std::runtime_error("polynomial commitment: export before commit_public");
    if (p->fri_step > 0) throw std::runtime_error("polynomial commitment: interleaved export after the FRI commit phase began");
    if (!p->fri_code) {
        PCK(cudaMalloc(&p->fri_code, (size_t)PC_SLICES * p->N * sizeof(F)));
        PCK(cudaMalloc(&p->fri_tree, p->N * 32));
    }
    k_pc_interleave<<<(unsigned)((p->N / 2) >> PC_VOW_LEAVES_LOG), 256, 0, st>>>(which ? p->h_eval : p->l_eval, (uint32_t)p->log_N, p->fri_code);
    ++p->launches;
    PCK(cudaGetLastError());
    PCK(cudaMemcpyAsync(out, p->fri_code, (size_t)PC_SLICES * p->N * sizeof(F), cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
}

void pc_export(PcCommit* p, cudaStream_t st, F* l_eval, uint8_t* leaf_hash, uint8_t* tree) {
    PCK(cudaSetDevice(p->device));
    if (l_eval) PCK(cudaMemcpyAsync(l_eval, p->l_eval, (size_t)(PC_SLICES + 1) * p->N * sizeof(F), cudaMemcpyDeviceToHost, st));
    if (leaf_hash) PCK(cudaMemcpyAsync(leaf_hash, p->tree + (p->N / 2) * 4, (p->N / 2) * 32, cudaMemcpyDeviceToHost, st));
    if (tree) PCK(cudaMemcpyAsync(tree, p->tree, p->N * 32, cudaMemcpyDeviceToHost, st));
    PCK(cudaStreamSynchronize(st));
}

}  // namespace vp
