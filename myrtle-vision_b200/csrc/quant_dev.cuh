// quant_dev.cuh — per-element fake-quantisation arithmetic shared by the standalone kernels
// and by the fused prologues/epilogues (GEMM, LayerNorm, GELU, attention).
//
// Bit-for-bit the algorithm of QPyTorch 0.3.0's float/fixed/block kernels that myrtle-vision
// invokes at src/myrtle_vision/utils/quantize.py:84 (formats built at :47-72); the algorithm
// is written down in SURVEY.md Appendix B and checked against oracle/quant_oracle.c.
#pragma once
#include <stdint.h>

namespace mv {

struct FloatFmt {
    int exp_bits;   // 0 => identity
    int man_bits;
};

__device__ __forceinline__ uint32_t round_bits_nearest(uint32_t t, int man_bits) {
    const uint32_t mask = (1u << (23 - man_bits)) - 1u;
    return (t + (1u << (22 - man_bits))) & ~mask;
}
__device__ __forceinline__ uint32_t round_bits_stochastic(uint32_t t, uint32_t r, int man_bits) {
    const uint32_t mask = (1u << (23 - man_bits)) - 1u;
    return (t + (r & mask)) & ~mask;
}

// float_quantize for one element.  kStochastic selects round_bitwise_stochastic with the
// element's 32 random bits `r`.
template <bool kStochastic>
__device__ __forceinline__ float float_quantize_elem(float a, uint32_t r, int exp_bits,
                                                     int man_bits) {
    const uint32_t target = __float_as_uint(a);
    const int target_exp = int((target << 1) >> 24) - 127;
    const int min_exp = -((1 << (exp_bits - 1)) - 2);
    if (target_exp < min_exp) {
        // below the lowest normal binade: shift up to it, round there, shift back
        const uint32_t shift_bits = (uint32_t(127 + min_exp) << 23) | (target & 0x80000000u);
        const float shift = __uint_as_float(shift_bits);
        const float val = __fadd_rn(a, shift);
        const uint32_t vb = __float_as_uint(val);
        const uint32_t qb =
            kStochastic ? round_bits_stochastic(vb, r, man_bits) : round_bits_nearest(vb, man_bits);
        return __fsub_rn(__uint_as_float(qb), shift);
    }
    uint32_t q = kStochastic ? round_bits_stochastic(target, r, man_bits)
                             : round_bits_nearest(target, man_bits);
    // clip_exponent: the top exponent code is not used for finite values -> saturate to +-max
    const int e = int((q << 1) >> 24);
    const int max_e = (1 << (exp_bits - 1)) - 1 + 127;
    if (q != 0u && e > max_e) {
        const uint32_t max_man = (0x007FFFFFu >> (23 - man_bits)) << (23 - man_bits);
        q = (target & 0x80000000u) | (uint32_t(max_e) << 23) | max_man;
    }
    return __uint_as_float(q);
}

__device__ __forceinline__ float fq_nearest(float a, FloatFmt f) {
    return f.exp_bits == 0 ? a : float_quantize_elem<false>(a, 0u, f.exp_bits, f.man_bits);
}

// Same result as float_quantize_elem<false>(a, 0, 5, 10), with a short path for the normal
// fp16 range (the subnormal / zero branch is rare for activations and falls back).
static __device__ __noinline__ float fq_generic_slow(float a, int exp_bits, int man_bits) {
    return float_quantize_elem<false>(a, 0u, exp_bits, man_bits);
}
__device__ __forceinline__ float fq_half_fast(float a) {
    const uint32_t t = __float_as_uint(a);
    if (((t >> 23) & 0xFFu) < 113u) {
        // below fp16's lowest normal binade (rare for activations): shift up to 2^-14, round there,
        // shift back — float_quantize_elem's subnormal branch for (5,10), inline so that a warp
        // with one such lane pays ~8 instructions instead of a call
        const float shift = __uint_as_float(0x38800000u | (t & 0x80000000u));
        const uint32_t vb = __float_as_uint(__fadd_rn(a, shift));
        return __fsub_rn(__uint_as_float((vb + 0x1000u) & 0xFFFFE000u), shift);
    }
    uint32_t q = (t + 0x1000u) & 0xFFFFE000u;
    if ((q & 0x7FFFFFFFu) > 0x477FE000u) q = (t & 0x80000000u) | 0x477FE000u;
    return __uint_as_float(q);
}
// quantiser selected once per kernel: 0 = identity, 1 = (5,10) fast path, 2 = generic
__device__ __forceinline__ int fq_mode(FloatFmt f) {
    return f.exp_bits == 0 ? 0 : ((f.exp_bits == 5 && f.man_bits == 10) ? 1 : 2);
}
__device__ __forceinline__ float fq_apply(float a, int mode, FloatFmt f) {
    if (mode == 1) return fq_half_fast(a);
    if (mode == 2) return fq_generic_slow(a, f.exp_bits, f.man_bits);
    return a;
}

// ---- (5,10) on four values at once: one range test for the group instead of one per value ----
// Out of line on purpose: inline, ptxas if-converts the rare branch into ~50 predicated instructions.
static __device__ __noinline__ float4 fq_half4_rare(float a, float b, float c, float d) {
    return make_float4(fq_half_fast(a), fq_half_fast(b), fq_half_fast(c), fq_half_fast(d));
}
__device__ __forceinline__ bool fq_half4_all_normal(float a, float b, float c, float d) {
    // all four at or above fp16's lowest normal binade (2^-14); zeros take the rare path
    return fminf(fminf(fabsf(a), fabsf(b)), fminf(fabsf(c), fabsf(d))) >= 6.103515625e-05f;
}
__device__ __forceinline__ bool fq_half4_none_saturates(float a, float b, float c, float d) {
    // |x| < 65520 rounds to at most 65504 (the half-ulp point of the top binade is 65520)
    return fmaxf(fmaxf(fabsf(a), fabsf(b)), fmaxf(fabsf(c), fabsf(d))) < 65520.0f;
}
// fp32 results (the value feeds more fp32 math): one range test for the group, then add-and-mask per value
__device__ __forceinline__ float4 fq_half4_f32(float4 v) {
    if (fq_half4_all_normal(v.x, v.y, v.z, v.w) && fq_half4_none_saturates(v.x, v.y, v.z, v.w)) {
        return make_float4(__uint_as_float((__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u),
                           __uint_as_float((__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u),
                           __uint_as_float((__float_as_uint(v.z) + 0x1000u) & 0xFFFFE000u),
                           __uint_as_float((__float_as_uint(v.w) + 0x1000u) & 0xFFFFE000u));
    }
    return fq_half4_rare(v.x, v.y, v.z, v.w);
}
// packed fp16 results (the value is stored as a tensor-core operand).  In the normal range
// float_quantize(5,10) nearest is "add half an fp16 ulp to the fp32 word, drop the low 13 bits, clip to
// +-65504": adding 0x1000 and converting with round-toward-zero does exactly that — RZ truncates the low
// bits and never rounds a finite value to infinity (satfinite also clips an infinite input) — at 1.5
// instructions per value.
__device__ __forceinline__ uint32_t cvt_rz_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rz.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint2 fq_half4_pack(float a, float b, float c, float d) {
    if (!fq_half4_all_normal(a, b, c, d)) {
        const float4 r = fq_half4_rare(a, b, c, d);           // exactly representable: any rounding mode
        return make_uint2(cvt_rz_f16x2(r.x, r.y), cvt_rz_f16x2(r.z, r.w));
    }
    return make_uint2(cvt_rz_f16x2(__uint_as_float(__float_as_uint(a) + 0x1000u), __uint_as_float(__float_as_uint(b) + 0x1000u)),
                      cvt_rz_f16x2(__uint_as_float(__float_as_uint(c) + 0x1000u), __uint_as_float(__float_as_uint(d) + 0x1000u)));
}

// fixed_point_quantize for one element: floor(a * 2^fl + r) * 2^-fl, then clamp.
// Nearest passes r = 0.5 (QPyTorch's CUDA kernel: ties toward +inf).
__device__ __forceinline__ float fixed_quantize_elem(float a, float r, float scale_up,
                                                     float scale_down, float t_min, float t_max,
                                                     bool clamp) {
    float v = floorf(__fadd_rn(__fmul_rn(a, scale_up), r));
    v = __fmul_rn(v, scale_down);
    if (clamp) v = fminf(fmaxf(v, t_min), t_max);
    return v;
}

// block_quantize for one element given the block's max |a|
template <bool kStochastic>
__device__ __forceinline__ float block_quantize_elem(float a, float max_entry, uint32_t r, int wl) {
    const uint32_t max_exp = ((__float_as_uint(max_entry) << 1) >> 24) << 23;
    const float base = __fmul_rn(6.0f, __uint_as_float(max_exp));
    const float t = __fadd_rn(a, base);
    const uint32_t tb = __float_as_uint(t);
    const uint32_t qb = kStochastic ? round_bits_stochastic(tb, r, wl) : round_bits_nearest(tb, wl);
    return __fsub_rn(__uint_as_float(qb), base);
}

// Philox4x32-10 counter RNG: element i consumes word (i & 3) of
// philox(key = seed, counter = {lo(i>>2), hi(i>>2), lo(offset), hi(offset)}).
__device__ __forceinline__ uint4 philox4x32_10(uint64_t seed, uint64_t ctr, uint64_t offset) {
    uint32_t c0 = uint32_t(ctr), c1 = uint32_t(ctr >> 32), c2 = uint32_t(offset),
             c3 = uint32_t(offset >> 32);
    uint32_t k0 = uint32_t(seed), k1 = uint32_t(seed >> 32);
#pragma unroll
    for (int i = 0; i < 10; i++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// "16-bit stream" of stochastic float_quantize for formats with man_bits >= 7: element i takes half-word (i & 7) of
// philox(seed, i >> 3, offset) — low half of word ((i & 7) >> 1) when i is even, high half when odd.
__device__ __forceinline__ uint32_t philox_half16(uint64_t seed, uint64_t i, uint64_t offset) {
    const uint4 w = philox4x32_10(seed, i >> 3, offset);
    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
    const uint32_t word = ws[(i & 7) >> 1];
    return (i & 1) ? (word >> 16) : (word & 0xFFFFu);
}

// ---- dropout mask (include/mv_b200.h "dropout mask"): keep(i) = bits16(seed, site, i) >= thr ----
struct DropDev {
    const uint64_t* seed;       // device pointer; NULL: off
    uint32_t thr;
    float scale;
    int site;
};
// keep bits of elements i .. i+3 (i % 4 == 0: one half of a Philox block) from that half's two words: bit j = element i+j
__device__ __forceinline__ uint32_t drop_bits4(uint2 h, uint32_t thr) {
    return uint32_t((h.x & 0xFFFFu) >= thr) | (uint32_t((h.x >> 16) >= thr) << 1) |
           (uint32_t((h.y & 0xFFFFu) >= thr) << 2) | (uint32_t((h.y >> 16) >= thr) << 3);
}
// the half of element i's Philox block that holds i .. i+3 (i % 4 == 0), computed by this lane alone
__device__ __forceinline__ uint32_t drop_keep4(uint64_t seed, const DropDev& d, uint64_t i) {
    const uint4 w = philox4x32_10(seed, i >> 3, uint64_t(uint32_t(d.site)));
    return drop_bits4((i & 4) ? make_uint2(w.z, w.w) : make_uint2(w.x, w.y), d.thr);
}
// One Philox call serves eight elements, i.e. two lanes that own four each.  Lanes 2k and 2k+1 each need their half of two
// blocks A and B (the even lane elements 0..3 of a block, the odd lane 4..7): the even lane computes A, the odd lane B
// (`ctr` = that block's counter), and each hands the other the half it needs — one call per lane instead of two.
// Returns the keep bits of this lane's half of A (bits 0..3) and of B (bits 4..7).
__device__ __forceinline__ uint32_t drop_keep4_pair(uint64_t seed, const DropDev& d, uint64_t ctr, bool odd) {
    const uint4 w = philox4x32_10(seed, ctr, uint64_t(uint32_t(d.site)));
    const uint2 mine = odd ? make_uint2(w.z, w.w) : make_uint2(w.x, w.y);
    const uint2 give = odd ? make_uint2(w.x, w.y) : make_uint2(w.z, w.w);
    const uint2 got = make_uint2(__shfl_xor_sync(0xffffffffu, give.x, 1), __shfl_xor_sync(0xffffffffu, give.y, 1));
    const uint32_t a = drop_bits4(odd ? got : mine, d.thr), b = drop_bits4(odd ? mine : got, d.thr);
    return a | (b << 4);
}
__device__ __forceinline__ float drop_mul(uint32_t bits, int j, float scale) { return ((bits >> j) & 1u) ? scale : 0.f; }

// ---- stochastic gradient rounding (include/mv_b200.h "gradient rounding stream"): element i of a site tensor is rounded
// with the bits mv_float_quantize(..., MV_ROUND_STOCHASTIC, seed, offset) gives element i ----
struct SrDev {
    const uint64_t* seed;       // device pointer; NULL: off
    uint64_t offset;            // site + (rank << 32)
};
__device__ __forceinline__ uint64_t sr_seed(const SrDev& s) { return __ldg(reinterpret_cast<const unsigned long long*>(s.seed)); }
// the four half-words of one half of a 16-bit-stream block, element order
__device__ __forceinline__ uint4 sr_halves(uint2 h) {
    return make_uint4(h.x & 0xFFFFu, h.x >> 16, h.y & 0xFFFFu, h.y >> 16);
}
// random bits of elements i .. i+3 (i % 4 == 0), computed by this lane alone: half (i & 4) of the 16-bit block i >> 3
// (s16, man_bits >= 7) or the whole 32-bit block i >> 2
__device__ __forceinline__ uint4 sr_bits4(uint64_t seed, uint64_t offset, uint64_t i, bool s16) {
    if (s16) {
        const uint4 w = philox4x32_10(seed, i >> 3, offset);
        return sr_halves((i & 4) ? make_uint2(w.z, w.w) : make_uint2(w.x, w.y));
    }
    return philox4x32_10(seed, i >> 2, offset);
}
// random bits of element i alone (word selects, not an indexed array: that would live in local memory)
__device__ __forceinline__ uint32_t sr_bits1(uint64_t seed, uint64_t offset, uint64_t i, bool s16) {
    const uint4 w = philox4x32_10(seed, s16 ? (i >> 3) : (i >> 2), offset);
    const uint64_t k = s16 ? ((i & 7) >> 1) : (i & 3);
    const uint32_t word = (k & 2) ? ((k & 1) ? w.w : w.z) : ((k & 1) ? w.y : w.x);
    return s16 ? ((i & 1) ? (word >> 16) : (word & 0xFFFFu)) : word;
}
// float_quantize_elem<true> with the normal range inline ("add the tail bits, clear the tail, clip to the largest finite
// value") and everything else (below the lowest normal binade, inf / NaN) out of line, so that the rare branch does not hold
// registers across an unrolled epilogue.  Same results.
static __device__ __noinline__ float fq_stoch_rare(float a, uint32_t r, int exp_bits, int man_bits) {
    return float_quantize_elem<true>(a, r, exp_bits, man_bits);
}
__device__ __forceinline__ float fq_stoch_elem(float a, uint32_t r, FloatFmt f) {
    const uint32_t t = __float_as_uint(a), mag = t & 0x7FFFFFFFu;
    const uint32_t mask = (1u << (23 - f.man_bits)) - 1u;
    const uint32_t lo_bits = uint32_t(127 - ((1 << (f.exp_bits - 1)) - 2)) << 23;
    const uint32_t hi_bits = (uint32_t((1 << (f.exp_bits - 1)) - 1 + 127) << 23) | (0x007FFFFFu & ~mask);
    if (mag < lo_bits || mag > hi_bits) return fq_stoch_rare(a, r, f.exp_bits, f.man_bits);
    const uint32_t q = (t + (r & mask)) & ~mask;
    return __uint_as_float((q & 0x7FFFFFFFu) > hi_bits ? ((t & 0x80000000u) | hi_bits) : q);
}

// 16-bit stream shared by a lane pair, as drop_keep4_pair: the even lane computes block `ctr` for its row A, the odd lane
// for its row B; returns this lane's half of A (.x) and of B (.y), each as the two words of four half-words
__device__ __forceinline__ uint4 sr_pair16(uint64_t seed, uint64_t offset, uint64_t ctr, bool odd) {
    const uint4 w = philox4x32_10(seed, ctr, offset);
    const uint2 mine = odd ? make_uint2(w.z, w.w) : make_uint2(w.x, w.y);
    const uint2 give = odd ? make_uint2(w.x, w.y) : make_uint2(w.z, w.w);
    const uint2 got = make_uint2(__shfl_xor_sync(0xffffffffu, give.x, 1), __shfl_xor_sync(0xffffffffu, give.y, 1));
    const uint2 a = odd ? got : mine, b = odd ? mine : got;
    return make_uint4(a.x, a.y, b.x, b.y);
}

__device__ __forceinline__ float bits_to_uniform(uint32_t b) {
    return float(b >> 8) * (1.0f / 16777216.0f);
}

}  // namespace mv
