// F_{p^2} = F_p[i]/(i^2+1), p = 2^61-1  --  Virgo's field, device + host.
//
// Replaces: /root/reference/lib/virgo/src/fieldElement.cpp:34-96 (operator+,*,-),
//           :336-360 (myMod, mymult); storage layout fieldElement.hpp:96-97
//           ({u64 real; u64 img;}, 16 bytes, always canonical: both limbs < p).
//
// Every function here returns CANONICAL values (< p) unless its name says otherwise. The
// arithmetic is exact, so any association order gives the same bits as the reference.
//
// Multiplication (the hot operation) is built for the sm_100a integer pipes:
//   * operands are split into two 31-bit limbs  x = x1*2^31 + x0;
//   * a complex product is two chains of four IMAD.WIDE.U32 per component (schoolbook, the
//     subtraction in re = ac - bd is folded in by multiplying with p - b instead of b), accumulated
//     in 64-bit registers with NO carry handling: four 31x31-bit products cannot overflow 64 bits;
//   * weights: 2^62 = 2 (mod p) is absorbed by pre-doubling one hi limb, so a component is just
//     u + 2^31 * t  with two 64-bit partials, reduced ONCE with the Mersenne identities
//     2^61 = 1: (u & p) + (u >> 61) + (t >> 30) + ((t mod 2^30) << 31).
// This moves the work to the FMA pipe (IMAD.WIDE) and leaves ~16 ALU-pipe instructions per
// reduced component; see DESIGN.md "Field arithmetic" for the instruction budget.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define VP_HD __host__ __device__ __forceinline__
#define VP_D __device__ __forceinline__
#else
#define VP_HD inline
#define VP_D inline
#endif

namespace vp {

typedef unsigned long long u64;
typedef unsigned int u32;

static constexpr u64 P = 2305843009213693951ULL;  // 2^61 - 1

struct alignas(16) F {
    u64 re, im;
};

// ---------------------------------------------------------------- base field F_p
VP_HD u64 fp_red1(u64 x) { return x >= P ? x - P : x; }          // x < 2p  ->  [0,p)
VP_HD u64 fp_fold(u64 x) { return (x & P) + (x >> 61); }         // any u64 -> [0, p + 7], same class
VP_HD u64 fp_canon(u64 x) { return fp_red1(fp_fold(x)); }        // any u64 < 2^64 - 2^61 -> [0,p)
VP_HD u64 fp_mod(u64 x) { return fp_red1(fp_fold(fp_fold(x))); }  // any u64 -> x % p (a Fiat-Shamir digest word)
VP_HD u64 fp_add(u64 a, u64 b) { return fp_red1(a + b); }
VP_HD u64 fp_sub(u64 a, u64 b) { return fp_red1(a + (P - b)); }
VP_HD u64 fp_neg(u64 a) { return a ? P - a : 0; }

// x = hi*2^31 + lo
struct Limbs {
    u32 lo, hi;
};
VP_HD Limbs split31(u64 x) {  // x < 2^63
    Limbs r;
    r.lo = (u32)x & 0x7FFFFFFFu;
    r.hi = (u32)(x >> 31);
    return r;
}
// 32x32 -> 64 multiply and multiply-accumulate. On the device these are spelled as PTX mul.wide / mad.wide:
// the C expression (u64)a * b + c makes nvcc 12.9 emit one junk "add 0 to the high word" (VIADD) per product.
VP_HD u64 mul32(u32 a, u32 b) {
#if defined(__CUDA_ARCH__)
    u64 d;
    asm("mul.wide.u32 %0, %1, %2;" : "=l"(d) : "r"(a), "r"(b));
    return d;
#else
    return (u64)a * (u64)b;
#endif
}
VP_HD u64 mad32(u32 a, u32 b, u64 c) {  // a*b + c  (IMAD.WIDE.U32 with a 64-bit addend)
#if defined(__CUDA_ARCH__)
    u64 d;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(d) : "r"(a), "r"(b), "l"(c));
    return d;
#else
    return (u64)a * (u64)b + c;
#endif
}

// value = u + 2^31*t + extra (mod p), canonical.  u, t < 2^64; extra < 2^62.
VP_HD u64 fp_reduce_ut(u64 u, u64 t, u64 extra) {
    u64 s = (u & P) + (u >> 61) + (t >> 30) + ((t & 0x3FFFFFFFULL) << 31) + extra;  // < 2^63 + 2^35
    return fp_canon(s);
}
// Same value, folded once only: result <= p + 4 (same residue class, not canonical). extra < 2^62.
VP_HD u64 fp_reduce_ut_loose(u64 u, u64 t, u64 extra) {
    u64 s = (u & P) + (u >> 61) + (t >> 30) + ((t & 0x3FFFFFFFULL) << 31) + extra;
    return fp_fold(s);
}
// value = u + 2^31*t + 2^62*w + extra (mod p), canonical.  u, t, w < 2^64; extra < 2^62.
VP_HD u64 fp_reduce_utw(u64 u, u64 t, u64 w, u64 extra) {
    // 2^62 * w = 2w: (w << 1) may drop bit 63 of w, worth 2^64 = 8 (mod p)
    u64 s = (u & P) + (u >> 61) + (t >> 30) + ((t & 0x3FFFFFFFULL) << 31) + extra;   // < 2^63 + 2^35
    u64 w2 = ((w << 1) & P) + ((w << 1) >> 61) + ((w >> 63) << 3);                   // < 2^61 + 16
    return fp_canon(s + w2);
}

VP_HD u64 fp_mul(u64 a, u64 b) {  // a, b < 2^62
    const Limbs x = split31(a), y = split31(b);
    const u64 u = mul32(x.lo, y.lo), t = mad32(x.hi, y.lo, mul32(x.lo, y.hi)), w = mul32(x.hi, y.hi);
    return fp_reduce_utw(u, t, w, 0);
}

// ---------------------------------------------------------------- extension field: basic ops
VP_HD F f_zero() { return F{0, 0}; }
VP_HD F f_one() { return F{1, 0}; }
VP_HD F f_make(u64 re, u64 im) { return F{re, im}; }
VP_HD bool f_is_zero(const F& a) { return (a.re | a.im) == 0; }
VP_HD bool f_eq(const F& a, const F& b) { return a.re == b.re && a.im == b.im; }
VP_HD F f_add(const F& a, const F& b) { return F{fp_add(a.re, b.re), fp_add(a.im, b.im)}; }
VP_HD F f_sub(const F& a, const F& b) { return F{fp_sub(a.re, b.re), fp_sub(a.im, b.im)}; }
VP_HD F f_neg(const F& a) { return F{fp_neg(a.re), fp_neg(a.im)}; }
VP_HD F f_dbl(const F& a) { return f_add(a, a); }

// ---------------------------------------------------------------- complex product by limb chains
// Left operand m (re, im < 2^62): limbs of re, im and of the negated im (2p - im).
struct LOp {
    u32 re0, re1, im0, im1, nim0, nim1;
};
// Right operand v (re, im < 2^62): limbs of re, im.
struct ROp {
    u32 re0, re1, im0, im1;
};
VP_HD LOp make_lop(u64 re, u64 im) {  // re, im <= 2p
    const Limbs a = split31(re), b = split31(im), c = split31(2 * P - im);
    return LOp{a.lo, a.hi, b.lo, b.hi, c.lo, c.hi};
}
VP_HD ROp make_rop(u64 re, u64 im) {
    const Limbs a = split31(re), b = split31(im);
    return ROp{a.lo, a.hi, b.lo, b.hi};
}

// Partials of m*v: component = u + 2^31 t + 2^62 w.
struct CPart {
    u64 u_re, t_re, w_re, u_im, t_im, w_im;
};
// Valid for m, v components <= 2p (hi limbs < 2^31): every chain is a sum of <= 4 products < 2^62.
VP_HD CPart cprod_parts(const LOp& m, const ROp& v) {
    CPart c;
    c.u_re = mad32(m.nim0, v.im0, mul32(m.re0, v.re0));
    c.t_re = mad32(m.nim1, v.im0, mad32(m.nim0, v.im1, mad32(m.re1, v.re0, mul32(m.re0, v.re1))));
    c.w_re = mad32(m.nim1, v.im1, mul32(m.re1, v.re1));
    c.u_im = mad32(m.im0, v.re0, mul32(m.re0, v.im0));
    c.t_im = mad32(m.im1, v.re0, mad32(m.im0, v.re1, mad32(m.re1, v.im0, mul32(m.re0, v.im1))));
    c.w_im = mad32(m.im1, v.re1, mul32(m.re1, v.im1));
    return c;
}
// m*v + acc for operands with components <= 2p; acc < 2^62. Canonical result.
VP_HD F f_mul_add_loose(const LOp& m, const ROp& v, const F& acc) {
    const CPart c = cprod_parts(m, v);
    return F{fp_reduce_utw(c.u_re, c.t_re, c.w_re, acc.re), fp_reduce_utw(c.u_im, c.t_im, c.w_im, acc.im)};
}
// Same with a result that is only folded once (<= p + 5, not canonical).
VP_HD u64 fp_reduce_utw_loose(u64 u, u64 t, u64 w, u64 extra) {
    u64 s = (u & P) + (u >> 61) + (t >> 30) + ((t & 0x3FFFFFFFULL) << 31) + extra;
    u64 w2 = ((w << 1) & P) + ((w << 1) >> 61) + ((w >> 63) << 3);
    return fp_fold(s + w2);
}
VP_HD F f_mul_add_loose2(const LOp& m, const ROp& v, const F& acc) {
    const CPart c = cprod_parts(m, v);
    return F{fp_reduce_utw_loose(c.u_re, c.t_re, c.w_re, acc.re), fp_reduce_utw_loose(c.u_im, c.t_im, c.w_im, acc.im)};
}

// Canonical operands (< 2^61: hi limbs < 2^30) let the 2^62-weight products ride in the u chain by
// pre-doubling the right operand's hi limbs: two partials per component instead of three.
struct ROpD {
    u32 re0, re1, re1d, im0, im1, im1d;
};
VP_HD ROpD make_ropd(const F& v) {  // v canonical
    const Limbs a = split31(v.re), b = split31(v.im);
    return ROpD{a.lo, a.hi, a.hi << 1, b.lo, b.hi, b.hi << 1};
}
// m components <= 2p, v canonical: u chains hold 2 x (< 2^62) + 2 x (2^31 * 2^31) < 2^64.
VP_HD F f_mul_add_k(const LOp& m, const ROpD& v, const F& acc) {
    const u64 u_re = mad32(m.nim1, v.im1d, mad32(m.re1, v.re1d, mad32(m.nim0, v.im0, mul32(m.re0, v.re0))));
    const u64 t_re = mad32(m.nim1, v.im0, mad32(m.nim0, v.im1, mad32(m.re1, v.re0, mul32(m.re0, v.re1))));
    const u64 u_im = mad32(m.im1, v.re1d, mad32(m.re1, v.im1d, mad32(m.im0, v.re0, mul32(m.re0, v.im0))));
    const u64 t_im = mad32(m.im1, v.re0, mad32(m.im0, v.re1, mad32(m.re1, v.im0, mul32(m.re0, v.im1))));
    return F{fp_reduce_ut(u_re, t_re, acc.re), fp_reduce_ut(u_im, t_im, acc.im)};
}
// Same, but the result is only folded once (<= p + 4, NOT canonical): for running sums that are fed back as `acc`.
VP_HD F f_mul_add_k_loose(const LOp& m, const ROpD& v, const F& acc) {
    const u64 u_re = mad32(m.nim1, v.im1d, mad32(m.re1, v.re1d, mad32(m.nim0, v.im0, mul32(m.re0, v.re0))));
    const u64 t_re = mad32(m.nim1, v.im0, mad32(m.nim0, v.im1, mad32(m.re1, v.re0, mul32(m.re0, v.re1))));
    const u64 u_im = mad32(m.im1, v.re1d, mad32(m.re1, v.im1d, mad32(m.im0, v.re0, mul32(m.re0, v.im0))));
    const u64 t_im = mad32(m.im1, v.re0, mad32(m.im0, v.re1, mad32(m.re1, v.im0, mul32(m.re0, v.im1))));
    return F{fp_reduce_ut_loose(u_re, t_re, acc.re), fp_reduce_ut_loose(u_im, t_im, acc.im)};
}

VP_HD F f_mul(const F& a, const F& b) {  // canonical operands
    return f_mul_add_k(make_lop(a.re, a.im), make_ropd(b), f_zero());
}
VP_HD F f_mul_add(const F& a, const F& b, const F& acc) { return f_mul_add_k(make_lop(a.re, a.im), make_ropd(b), acc); }
// a * b where b is in the base field (b.im == 0)
VP_HD F f_mul_base(const F& a, u64 b) { return F{fp_mul(a.re, b), fp_mul(a.im, b)}; }

// v0 + r*(v1 - v0): linear_poly{v1-v0, v0}.eval(r)   (reference src/polynomial.cpp:128-131)
// FoldK = the challenge r pre-split (built once per kernel).
typedef ROpD FoldK;
VP_HD FoldK make_foldk(const F& r) { return make_ropd(r); }
VP_HD F f_fold_k(const F& v0, const F& v1, const FoldK& k) {
    // d = v1 - v0 + p  in (0, 2p)
    return f_mul_add_k(make_lop(v1.re + P - v0.re, v1.im + P - v0.im), k, v0);
}
VP_HD F f_fold(const F& v0, const F& v1, const F& r) { return f_fold_k(v0, v1, make_foldk(r)); }

// ---------------------------------------------------------------- weakly canonical values, lazy product sums
// The whole-proof pass kernel (k_phase_dfs) keeps its tables WEAKLY canonical: components in [0, p], where p is an
// alias of 0. Every function above accepts such operands (their bounds only need "<= p") and +,-,* map [0,p] into
// [0,p]; only equality tests and values that leave the device (transcript, claims) need f_strict().
VP_HD u64 fp_weak(u64 s) {  // any u64 -> [0, p], same residue class
    s = (s & P) + (s >> 61);  // <= p + 7
    return (s & P) + (s >> 61);
}
VP_HD u64 fp_strict(u64 x) { return x == P ? 0 : x; }  // [0,p] -> [0,p)
VP_HD F f_strict(const F& a) { return F{fp_strict(a.re), fp_strict(a.im)}; }

// value = u + 2^31*t + e (mod p) in [0,p]; any u, t, e < 2^64. The 96-bit sum S = u + (t << 31) + e is built with
// carry chains (6 adds, 3 shifts), then S mod 2^61 + S >> 61 (< 2^61 + 2^35) and one more Mersenne fold.
VP_HD u64 fp_reduce_ut_weak(u64 u, u64 t, u64 e) {
#if defined(__CUDA_ARCH__)
    const u32 uL = (u32)u, uH = (u32)(u >> 32), tL = (u32)t, tH = (u32)(t >> 32), eL = (u32)e, eH = (u32)(e >> 32);
    const u32 a0 = tL << 31, a1 = (u32)(t >> 1), a2 = tH >> 1;
    u32 w0, w1, w2;
    asm("add.cc.u32 %0, %3, %4;\n\t"
        "addc.cc.u32 %1, %5, %6;\n\t"
        "addc.u32 %2, %7, 0;\n\t"
        "add.cc.u32 %0, %0, %8;\n\t"
        "addc.cc.u32 %1, %1, %9;\n\t"
        "addc.u32 %2, %2, 0;"
        : "=&r"(w0), "=&r"(w1), "=&r"(w2)
        : "r"(uL), "r"(a0), "r"(uH), "r"(a1), "r"(a2), "r"(eL), "r"(eH));
    const u64 lo = ((u64)(w1 & 0x1FFFFFFFu) << 32) | w0;
    const u64 hi = ((u64)w2 << 3) | (w1 >> 29);
    const u64 r = lo + hi;
    return (r & P) + (r >> 61);
#else
    const unsigned __int128 S = (unsigned __int128)u + ((unsigned __int128)t << 31) + e;
    const u64 r = ((u64)S & P) + (u64)(S >> 61);
    return (r & P) + (r >> 61);
#endif
}

// A constant right operand (a challenge), pre-split once per kernel: limbs of re, im and of -im, hi limbs also doubled.
struct ConstK {
    u32 re0, re1, re1d, im0, im1, im1d, nim0, nim1, nim1d;
};
VP_HD ConstK make_constk(const F& r) {  // r canonical
    const Limbs a = split31(r.re), b = split31(r.im), c = split31(r.im ? P - r.im : 0);
    return ConstK{a.lo, a.hi, a.hi << 1, b.lo, b.hi, b.hi << 1, c.lo, c.hi, c.hi << 1};
}
// v0 + k*d  for d with components <= 2p (hi limbs < 2^31), v0 in [0,p]: result in [0,p].
// Chains: every product is < 2^31 * 2^31, four per chain: no overflow.
VP_HD F f_fold_w(const F& v0, const F& d, const ConstK& k) {
    const Limbs a = split31(d.re), b = split31(d.im);
    const u64 u_re = mad32(b.hi, k.nim1d, mad32(a.hi, k.re1d, mad32(b.lo, k.nim0, mul32(a.lo, k.re0))));
    const u64 t_re = mad32(b.hi, k.nim0, mad32(b.lo, k.nim1, mad32(a.hi, k.re0, mul32(a.lo, k.re1))));
    const u64 u_im = mad32(b.hi, k.re1d, mad32(a.hi, k.im1d, mad32(b.lo, k.re0, mul32(a.lo, k.im0))));
    const u64 t_im = mad32(b.hi, k.re0, mad32(b.lo, k.re1, mad32(a.hi, k.im0, mul32(a.lo, k.im1))));
    return F{fp_reduce_ut_weak(u_re, t_re, v0.re), fp_reduce_ut_weak(u_im, t_im, v0.im)};
}
// Same for base-field data (v0.im == d.im == 0): v0 + k*d with v0, d real.
VP_HD F f_fold_w_real(u64 v0, u64 d, const ConstK& k) {
    const Limbs a = split31(d);
    const u64 u_re = mad32(a.hi, k.re1d, mul32(a.lo, k.re0));
    const u64 t_re = mad32(a.hi, k.re0, mul32(a.lo, k.re1));
    const u64 u_im = mad32(a.hi, k.im1d, mul32(a.lo, k.im0));
    const u64 t_im = mad32(a.hi, k.im0, mul32(a.lo, k.im1));
    return F{fp_reduce_ut_weak(u_re, t_re, v0), fp_reduce_ut_weak(u_im, t_im, 0)};
}
// x1 - x0 as a value in [0, 2p] (operands in [0,p]); and the same folded into [0,p]
VP_HD F f_diff2p(const F& x0, const F& x1) { return F{x1.re + P - x0.re, x1.im + P - x0.im}; }
VP_HD F f_diff_w(const F& x0, const F& x1) { return F{fp_weak(x1.re + P - x0.re), fp_weak(x1.im + P - x0.im)}; }

// 96-bit accumulator: sums up to 2^32 chain values (< 2^64 each) without any reduction.
struct A96 {
    u32 w0, w1, w2;
};
VP_HD void a96_add(A96& a, u64 x) {
#if defined(__CUDA_ARCH__)
    asm("add.cc.u32 %0, %0, %3;\n\t"
        "addc.cc.u32 %1, %1, %4;\n\t"
        "addc.u32 %2, %2, 0;"
        : "+r"(a.w0), "+r"(a.w1), "+r"(a.w2)
        : "r"((u32)x), "r"((u32)(x >> 32)));
#else
    unsigned __int128 s = ((unsigned __int128)a.w2 << 64) | ((u64)a.w1 << 32) | a.w0;
    s += x;
    a.w0 = (u32)s; a.w1 = (u32)(s >> 32); a.w2 = (u32)(s >> 64);
#endif
}
VP_HD u64 a96_mod(const A96& a) {  // -> < 2^61 + 2^35, same class
    const u64 lo = ((u64)(a.w1 & 0x1FFFFFFFu) << 32) | a.w0;
    const u64 hi = ((u64)a.w2 << 3) | (a.w1 >> 29);
    return lo + hi;
}
// Lazy sum of complex products: per component  value = U + 2^31 * T.
struct CAcc {
    A96 u_re, t_re, u_im, t_im;
};
VP_HD CAcc cacc_zero() { return CAcc{{0, 0, 0}, {0, 0, 0}, {0, 0, 0}, {0, 0, 0}}; }
// acc += m * v.  m: components <= 2p (LOp, with the limbs of 2p - im); v: components in [0,p] (ROpD).
VP_HD void cacc_mad(CAcc& s, const LOp& m, const ROpD& v) {
    a96_add(s.u_re, mad32(m.nim1, v.im1d, mad32(m.re1, v.re1d, mad32(m.nim0, v.im0, mul32(m.re0, v.re0)))));
    a96_add(s.t_re, mad32(m.nim1, v.im0, mad32(m.nim0, v.im1, mad32(m.re1, v.re0, mul32(m.re0, v.re1)))));
    a96_add(s.u_im, mad32(m.im1, v.re1d, mad32(m.re1, v.im1d, mad32(m.im0, v.re0, mul32(m.re0, v.im0)))));
    a96_add(s.t_im, mad32(m.im1, v.re0, mad32(m.im0, v.re1, mad32(m.re1, v.im0, mul32(m.re0, v.im1)))));
}
// acc += m * v for a base-field v in [0,p]; m components <= 2p.
VP_HD void cacc_mad_real(CAcc& s, const F& m, u64 v) {
    const Limbs a = split31(m.re), b = split31(m.im), c = split31(v);
    const u32 c1d = c.hi << 1;
    a96_add(s.u_re, mad32(a.hi, c1d, mul32(a.lo, c.lo)));
    a96_add(s.t_re, mad32(a.hi, c.lo, mul32(a.lo, c.hi)));
    a96_add(s.u_im, mad32(b.hi, c1d, mul32(b.lo, c.lo)));
    a96_add(s.t_im, mad32(b.hi, c.lo, mul32(b.lo, c.hi)));
}
// acc + m * v for a base-field v in [0,p]; m components <= 2p, acc components < 2^64: result in [0,p]
VP_HD F f_mad_real_w(const F& acc, const F& m, u64 v) {
    const Limbs a = split31(m.re), b = split31(m.im), c = split31(v);
    const u32 c1d = c.hi << 1;
    return F{fp_reduce_ut_weak(mad32(a.hi, c1d, mul32(a.lo, c.lo)), mad32(a.hi, c.lo, mul32(a.lo, c.hi)), acc.re),
             fp_reduce_ut_weak(mad32(b.hi, c1d, mul32(b.lo, c.lo)), mad32(b.hi, c.lo, mul32(b.lo, c.hi)), acc.im)};
}
VP_HD F cacc_reduce(const CAcc& s) {  // canonical
    return F{fp_reduce_ut(a96_mod(s.u_re), a96_mod(s.t_re), 0), fp_reduce_ut(a96_mod(s.u_im), a96_mod(s.t_im), 0)};
}

// ---------------------------------------------------------------- lazy sums of products
// Acc: unreduced 128-bit sums of the Karatsuba base products; kept for the dot-product kernels.
struct U128 {
    u64 lo, hi;
};
VP_HD U128 mul_wide(u64 a, u64 b) {
#if defined(__CUDA_ARCH__)
    U128 r;
    r.lo = a * b;
    r.hi = __umul64hi(a, b);
    return r;
#else
    unsigned __int128 t = (unsigned __int128)a * b;
    U128 r;
    r.lo = (u64)t;
    r.hi = (u64)(t >> 64);
    return r;
#endif
}
VP_HD U128 add128(U128 a, U128 b) {
    U128 r;
    r.lo = a.lo + b.lo;
    r.hi = a.hi + b.hi + (r.lo < a.lo ? 1ULL : 0ULL);
    return r;
}
// Reduce any 128-bit value to [0,p).  x = hi*2^64 + lo;  2^61 = 1, 2^64 = 8, 2^125 = 8 (mod p).
VP_HD u64 fp_reduce128(U128 x) {
    u64 h = (x.hi << 3) | (x.lo >> 61);                     // bits 61..124 of x
    u64 s = fp_fold(h) + (x.lo & P) + ((x.hi >> 61) << 3);  // < 2^62 + 64
    return fp_canon(s);
}
struct Acc {
    U128 ac, bd, x;  // sum a*c, sum b*d, sum (a+b)*(c+d); up to 8 products between reductions
};
VP_HD Acc acc_zero() { return Acc{{0, 0}, {0, 0}, {0, 0}}; }
VP_HD void acc_mad(Acc& s, const F& a, const F& b) {
    s.ac = add128(s.ac, mul_wide(a.re, b.re));
    s.bd = add128(s.bd, mul_wide(a.im, b.im));
    s.x = add128(s.x, mul_wide(a.re + a.im, b.re + b.im));
}
VP_HD F acc_reduce(const Acc& s) {
    u64 ac = fp_reduce128(s.ac), bd = fp_reduce128(s.bd), x = fp_reduce128(s.x);
    F r;
    r.re = fp_sub(ac, bd);
    r.im = fp_sub(fp_sub(x, ac), bd);
    return r;
}

}  // namespace vp
