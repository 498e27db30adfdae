// quant.cu — standalone fake-quantisation kernels (north-star kernel class (a)).
// HBM-bound bit manipulation on float words: 128-bit coalesced accesses, 4 independent
// vector loads in flight per thread, streaming cache policy, counter-based Philox RNG.
// Algorithmic traffic: 8 B/element (fp32 -> fp32), 6 B/element (fp32 -> fp16 container).
//
// Replaces QPyTorch 0.3.0 quant_cuda.{float,fixed_point,block}_quantize_* as invoked from
// src/myrtle_vision/utils/quantize.py:84 (reference), which moves >= 12 B/element
// (zeros_like memset + scalar load + scalar store).
#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {

extern int64_t g_launches;

constexpr int kQThreads = 256;
constexpr int kQUnroll = 4;

template <typename T> struct Vec4Store;
template <> struct Vec4Store<float> {
    static __device__ __forceinline__ void st(float* p, float4 v) {
        __stcs(reinterpret_cast<float4*>(p), v);
    }
};
template <> struct Vec4Store<__half> {
    static __device__ __forceinline__ void st(__half* p, float4 v) {
        __half2 lo = __floats2half2_rn(v.x, v.y), hi = __floats2half2_rn(v.z, v.w);
        uint2 u = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        __stcs(reinterpret_cast<uint2*>(p), u);
    }
};
// eight consecutive values: two 16-byte stores (fp32) or one (fp16 container)
template <typename T> struct Vec8Store;
template <> struct Vec8Store<float> {
    static __device__ __forceinline__ void st(float* p, float4 a, float4 b) {
        __stcs(reinterpret_cast<float4*>(p), a);
        __stcs(reinterpret_cast<float4*>(p) + 1, b);
    }
};
template <> struct Vec8Store<__half> {
    static __device__ __forceinline__ void st(__half* p, float4 a, float4 b) {
        const __half2 h0 = __floats2half2_rn(a.x, a.y), h1 = __floats2half2_rn(a.z, a.w);
        const __half2 h2 = __floats2half2_rn(b.x, b.y), h3 = __floats2half2_rn(b.z, b.w);
        __stcs(reinterpret_cast<uint4*>(p), make_uint4(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1),
                                                        *reinterpret_cast<const uint32_t*>(&h2), *reinterpret_cast<const uint32_t*>(&h3)));
    }
};
template <typename T> __device__ __forceinline__ T cvt_out(float v);
template <> __device__ __forceinline__ float cvt_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __half cvt_out<__half>(float v) { return __float2half_rn(v); }

struct FixedParams {
    float scale_up, scale_down, t_min, t_max;
    int clamp;
};

// float_quantize, stochastic, formats that drop at most 16 mantissa bits (man_bits >= 7): the rounding needs
// 23 - man_bits <= 16 random bits per element, so one Philox4x32-10 call (128 bits) serves EIGHT elements instead of
// four — element i takes half-word (i & 7) of philox(seed, i >> 3, offset) (include/mv_b200.h, "16-bit stream").  Ten
// Philox rounds per 4 elements were the bound of the stochastic kernel (0.65 - 0.74 of copy bandwidth); a thread now
// owns two adjacent 16-byte vectors (32 contiguous bytes) per Philox call.
// Four values with the random half-words (lo, hi) of two Philox words.  One range test for the group, voted over the
// warp (`valid`: lanes past the end vote yes): when every magnitude in the warp lies between the format's lowest normal and
// its largest finite value (unsigned compares of the magnitude bits, so NaN / inf fail it), float_quantize's stochastic
// rounding is "add the tail bits, clear the tail" — three instructions per value; otherwise every value takes the
// general path (subnormal shift, saturation), as before.  Same results.  Narrow-range tensors (randn: 4.8 -> 6.3 TB/s into
// the fp16 container) take the short path; with 15 % of the values below the normal range no warp does (a test per lane
// instead of the vote makes those warps run both paths, 5.7 -> 4.75 TB/s), and even the vote's range test costs them
// 15 %: a warp whose last vote failed tests again only every eighth iteration (try_short).
// float_quantize_elem<true> with both of its branches evaluated and selected (no divergence: on a wide-range tensor nearly
// every warp holds values below the lowest normal binade next to normal ones).  lo_bits / hi_bits / mask as below.
__device__ __forceinline__ float float_quantize_stoch_bf(float a, uint32_t r, uint32_t lo_bits, uint32_t hi_bits, uint32_t mask) {
    const uint32_t t = __float_as_uint(a), sign = t & 0x80000000u, rm = r & mask;
    uint32_t q = (t + rm) & ~mask;                                     // normal range: add the tail bits, clear the tail
    q = (q & 0x7FFFFFFFu) > hi_bits ? (sign | hi_bits) : q;            // clip_exponent: saturate to +-max
    const float shift = __uint_as_float(lo_bits | sign);               // below it: shift up to the lowest normal binade,
    const uint32_t vb = __float_as_uint(__fadd_rn(a, shift));          // round there, shift back
    const float sub = __fsub_rn(__uint_as_float((vb + rm) & ~mask), shift);
    return (t & 0x7FFFFFFFu) < lo_bits ? sub : __uint_as_float(q);
}
__device__ __forceinline__ float4 float_quantize_stoch4(float4 v, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3, int exp_bits, int man_bits,
                                                        uint32_t lo_bits, uint32_t hi_bits, uint32_t mask, bool valid,
                                                        bool try_short, bool& all_short) {
    const uint32_t tx = __float_as_uint(v.x), ty = __float_as_uint(v.y), tz = __float_as_uint(v.z), tw = __float_as_uint(v.w);
    bool take = false;
    if (try_short) {                                    // warp-uniform
        const uint32_t mx = tx & 0x7FFFFFFFu, my = ty & 0x7FFFFFFFu, mz = tz & 0x7FFFFFFFu, mw = tw & 0x7FFFFFFFu;
        const uint32_t mn = min(min(mx, my), min(mz, mw)), mxx = max(max(mx, my), max(mz, mw));
        take = __all_sync(0xffffffffu, !valid || (mn >= lo_bits && mxx <= hi_bits));
        all_short = all_short && take;
    }
    if (take) {
        return make_float4(__uint_as_float((tx + (r0 & mask)) & ~mask), __uint_as_float((ty + (r1 & mask)) & ~mask),
                           __uint_as_float((tz + (r2 & mask)) & ~mask), __uint_as_float((tw + (r3 & mask)) & ~mask));
    }
    return make_float4(float_quantize_stoch_bf(v.x, r0, lo_bits, hi_bits, mask), float_quantize_stoch_bf(v.y, r1, lo_bits, hi_bits, mask),
                       float_quantize_stoch_bf(v.z, r2, lo_bits, hi_bits, mask), float_quantize_stoch_bf(v.w, r3, lo_bits, hi_bits, mask));
}

// kStoch = false: nearest rounding on the same access pattern (a thread owns 32 contiguous input bytes, four such
// groups in flight): every tail word is half a step of the tail, no Philox (5.57 -> TB/s on randn against
// 16 bytes per thread and load in quant_vec_kernel)
// kDevSeed (every kernel of this file that has it): the seed is read from device memory, seed_dev, not the `seed` argument —
// a captured CUDA graph then rounds with whatever seed the step drew (mv_float_quantize_dev)
template <typename OutT, bool kStoch = true, bool kDevSeed = false>
__global__ void __launch_bounds__(kQThreads)
quant_vec16_kernel(const float* __restrict__ in, OutT* __restrict__ out, int64_t n, int exp_bits, int man_bits,
                   uint64_t seed, uint64_t offset, const uint64_t* __restrict__ seed_dev = nullptr) {
    if (kDevSeed) seed = __ldg(reinterpret_cast<const unsigned long long*>(seed_dev));
    const int64_t n8 = n >> 3;
    constexpr int kU = 4;                                   // 4 x 32 B in flight per thread
    const uint32_t mask = (1u << (23 - man_bits)) - 1u;
    const uint32_t lo_bits = uint32_t(127 - ((1 << (exp_bits - 1)) - 2)) << 23;                      // lowest normal
    const uint32_t hi_bits = (uint32_t((1 << (exp_bits - 1)) - 1 + 127) << 23) | (0x007FFFFFu & ~mask);  // largest finite
    const int64_t stride = int64_t(gridDim.x) * kQThreads * kU;
    // warp-uniform trip count (the lanes of a warp hold consecutive indices): the loop body votes over the whole warp
    bool last_short = true;                                 // did every group of this warp's previous iteration take the short path?
    int iter = 0;
    for (int64_t base = int64_t(blockIdx.x) * kQThreads * kU + threadIdx.x; base - (threadIdx.x & 31) < n8; base += stride, iter++) {
        const bool try_short = last_short || (iter & 7) == 0;
        bool all_short = try_short;
        float4 v[kU][2];
#pragma unroll
        for (int j = 0; j < kU; j++) {
            const int64_t i = base + int64_t(j) * kQThreads;
            v[j][0] = v[j][1] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n8) {
                v[j][0] = __ldcs(reinterpret_cast<const float4*>(in) + 2 * i);
                v[j][1] = __ldcs(reinterpret_cast<const float4*>(in) + 2 * i + 1);
            }
        }
#pragma unroll
        for (int j = 0; j < kU; j++) {
            const int64_t i = base + int64_t(j) * kQThreads;
            const bool valid = i < n8;                      // (the whole warp stays in the loop body: warp vote below)
            const uint32_t half_step = (mask + 1u) >> 1;
            uint4 r = make_uint4(0, 0, 0, 0);
            if (kStoch) r = philox4x32_10(seed, uint64_t(i), offset);
            const uint32_t w[4] = {r.x, r.y, r.z, r.w};
            float4 o[2];
#pragma unroll
            for (int h = 0; h < 2; h++)
                o[h] = kStoch ? float_quantize_stoch4(v[j][h], w[2 * h], w[2 * h] >> 16, w[2 * h + 1], w[2 * h + 1] >> 16, exp_bits, man_bits,
                                                      lo_bits, hi_bits, mask, valid, try_short, all_short)
                              : float_quantize_stoch4(v[j][h], half_step, half_step, half_step, half_step, exp_bits, man_bits,
                                                      lo_bits, hi_bits, mask, valid, try_short, all_short);
            if (valid) Vec8Store<OutT>::st(out + 8 * i, o[0], o[1]);
        }
        last_short = all_short;
    }
}
// scalar companion (tails, unaligned buffers): the same 16-bit stream
template <typename OutT, bool kDevSeed = false>
__global__ void quant_scalar16_kernel(const float* __restrict__ in, OutT* __restrict__ out, int64_t begin, int64_t n,
                                      int exp_bits, int man_bits, uint64_t seed, uint64_t offset,
                                      const uint64_t* __restrict__ seed_dev = nullptr) {
    if (kDevSeed) seed = __ldg(reinterpret_cast<const unsigned long long*>(seed_dev));
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = begin + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = cvt_out<OutT>(float_quantize_elem<true>(in[i], philox_half16(seed, uint64_t(i), offset), exp_bits, man_bits));
}

// MODE 0: float_quantize ; MODE 1: fixed_point_quantize
template <int MODE, bool STOCH, typename OutT, bool kDevSeed = false>
__global__ void __launch_bounds__(kQThreads)
quant_vec_kernel(const float* __restrict__ in, OutT* __restrict__ out, uint8_t* __restrict__ mask,
                 int64_t n, int exp_bits, int man_bits, FixedParams fp, uint64_t seed,
                 uint64_t offset, const uint64_t* __restrict__ seed_dev = nullptr) {
    if (kDevSeed) seed = __ldg(reinterpret_cast<const unsigned long long*>(seed_dev));
    const int64_t n4 = n >> 2;
    const int64_t stride = int64_t(gridDim.x) * kQThreads * kQUnroll;
    // MODE 0: the format's tail mask, half a step of it, its lowest normal and largest finite magnitudes
    const int mb = MODE == 0 ? man_bits : 10, eb = MODE == 0 ? exp_bits : 5;
    const uint32_t tail_mask = (1u << (23 - mb)) - 1u, half_step = (tail_mask + 1u) >> 1;
    const uint32_t lo_bits = uint32_t(127 - ((1 << (eb - 1)) - 2)) << 23;
    const uint32_t hi_bits = (uint32_t((1 << (eb - 1)) - 1 + 127) << 23) | (0x007FFFFFu & ~tail_mask);
    for (int64_t base = int64_t(blockIdx.x) * kQThreads * kQUnroll + threadIdx.x; base < n4;
         base += stride) {
        float4 v[kQUnroll];
#pragma unroll
        for (int j = 0; j < kQUnroll; j++) {
            const int64_t i = base + int64_t(j) * kQThreads;
            if (i < n4) v[j] = __ldcs(reinterpret_cast<const float4*>(in) + i);
        }
#pragma unroll
        for (int j = 0; j < kQUnroll; j++) {
            const int64_t i = base + int64_t(j) * kQThreads;
            if (i >= n4) continue;
            uint4 r = make_uint4(0, 0, 0, 0);
            if (STOCH) r = philox4x32_10(seed, uint64_t(i), offset);
            float4 o;
            if (MODE == 0) {
#ifdef MV_QUANT_BRANCHY
                o.x = float_quantize_elem<STOCH>(v[j].x, r.x, exp_bits, man_bits);
                o.y = float_quantize_elem<STOCH>(v[j].y, r.y, exp_bits, man_bits);
                o.z = float_quantize_elem<STOCH>(v[j].z, r.z, exp_bits, man_bits);
                o.w = float_quantize_elem<STOCH>(v[j].w, r.w, exp_bits, man_bits);
#else
                // both branches of float_quantize_elem evaluated and selected (float_quantize_stoch_bf); nearest rounding
                // adds half a step of the tail where stochastic rounding adds random tail bits
                o.x = float_quantize_stoch_bf(v[j].x, STOCH ? r.x : half_step, lo_bits, hi_bits, tail_mask);
                o.y = float_quantize_stoch_bf(v[j].y, STOCH ? r.y : half_step, lo_bits, hi_bits, tail_mask);
                o.z = float_quantize_stoch_bf(v[j].z, STOCH ? r.z : half_step, lo_bits, hi_bits, tail_mask);
                o.w = float_quantize_stoch_bf(v[j].w, STOCH ? r.w : half_step, lo_bits, hi_bits, tail_mask);
#endif
            } else {
                const bool cl = fp.clamp != 0 && mask == nullptr;
                float4 u;
                u.x = fixed_quantize_elem(v[j].x, STOCH ? bits_to_uniform(r.x) : 0.5f, fp.scale_up, fp.scale_down, fp.t_min, fp.t_max, cl);
                u.y = fixed_quantize_elem(v[j].y, STOCH ? bits_to_uniform(r.y) : 0.5f, fp.scale_up, fp.scale_down, fp.t_min, fp.t_max, cl);
                u.z = fixed_quantize_elem(v[j].z, STOCH ? bits_to_uniform(r.z) : 0.5f, fp.scale_up, fp.scale_down, fp.t_min, fp.t_max, cl);
                u.w = fixed_quantize_elem(v[j].w, STOCH ? bits_to_uniform(r.w) : 0.5f, fp.scale_up, fp.scale_down, fp.t_min, fp.t_max, cl);
                if (mask != nullptr) {
                    uchar4 m;
                    m.x = (u.x < fp.t_min || u.x > fp.t_max); m.y = (u.y < fp.t_min || u.y > fp.t_max);
                    m.z = (u.z < fp.t_min || u.z > fp.t_max); m.w = (u.w < fp.t_min || u.w > fp.t_max);
                    reinterpret_cast<uchar4*>(mask)[i] = m;
                    u.x = fminf(fmaxf(u.x, fp.t_min), fp.t_max); u.y = fminf(fmaxf(u.y, fp.t_min), fp.t_max);
                    u.z = fminf(fmaxf(u.z, fp.t_min), fp.t_max); u.w = fminf(fmaxf(u.w, fp.t_min), fp.t_max);
                }
                o = u;
            }
            Vec4Store<OutT>::st(out + 4 * i, o);
        }
    }
}

// scalar path: tails (n % 4) and unaligned buffers.  Element index i keeps its RNG word.
template <int MODE, bool STOCH, typename OutT, bool kDevSeed = false>
__global__ void quant_scalar_kernel(const float* __restrict__ in, OutT* __restrict__ out,
                                    uint8_t* __restrict__ mask, int64_t begin, int64_t n,
                                    int exp_bits, int man_bits, FixedParams fp, uint64_t seed,
                                    uint64_t offset, const uint64_t* __restrict__ seed_dev = nullptr) {
    if (kDevSeed) seed = __ldg(reinterpret_cast<const unsigned long long*>(seed_dev));
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = begin + int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        uint32_t r = 0;
        if (STOCH) {
            const uint4 w = philox4x32_10(seed, uint64_t(i >> 2), offset);
            const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
            r = ws[i & 3];
        }
        float o;
        if (MODE == 0) {
            o = float_quantize_elem<STOCH>(in[i], r, exp_bits, man_bits);
        } else {
            const bool cl = fp.clamp != 0 && mask == nullptr;
            o = fixed_quantize_elem(in[i], STOCH ? bits_to_uniform(r) : 0.5f, fp.scale_up,
                                    fp.scale_down, fp.t_min, fp.t_max, cl);
            if (mask != nullptr) {
                mask[i] = (o < fp.t_min || o > fp.t_max);
                o = fminf(fmaxf(o, fp.t_min), fp.t_max);
            }
        }
        out[i] = cvt_out<OutT>(o);
    }
}

static inline int grid_for(int64_t work_items, int per_block) {
    int64_t blocks = (work_items + per_block - 1) / per_block;
    const int64_t cap = int64_t(kNumSMs) * 8;   // resident CTAs of 256 threads per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return int(blocks);
}

template <typename OutT, bool kDevSeed = false>
static int launch_quant16(const float* in, OutT* out, int64_t n, int exp_bits, int man_bits, uint64_t seed,
                          uint64_t offset, cudaStream_t st, const uint64_t* seed_dev = nullptr) {
    if (n == 0) return 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(in) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
    int64_t done = 0;
    if (aligned && n >= 8) {
        const int64_t n8 = n >> 3;
        quant_vec16_kernel<OutT, true, kDevSeed><<<grid_for(n8, kQThreads * 4), kQThreads, 0, st>>>(in, out, n, exp_bits, man_bits, seed, offset,
                                                                                                  seed_dev);
        g_launches++;
        done = n8 << 3;
    }
    if (done < n) {
        quant_scalar16_kernel<OutT, kDevSeed><<<grid_for(n - done, 256), 256, 0, st>>>(in, out, done, n, exp_bits, man_bits, seed, offset,
                                                                                        seed_dev);
        g_launches++;
    }
    return check_cuda(cudaGetLastError(), "quant launch");
}

// float_quantize, nearest: eight values per thread (quant_vec16_kernel<OutT, false>), scalar tail
template <typename OutT>
static int launch_quant_nearest8(const float* in, OutT* out, int64_t n, int exp_bits, int man_bits, cudaStream_t st) {
    if (n == 0) return 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(in) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
    int64_t done = 0;
    if (aligned && n >= 8) {
        const int64_t n8 = n >> 3;
        quant_vec16_kernel<OutT, false><<<grid_for(n8, kQThreads * 4), kQThreads, 0, st>>>(in, out, n, exp_bits, man_bits, 0, 0);
        g_launches++;
        done = n8 << 3;
    }
    if (done < n) {
        quant_scalar_kernel<0, false, OutT><<<grid_for(n - done, 256), 256, 0, st>>>(in, out, nullptr, done, n, exp_bits, man_bits,
                                                                                    FixedParams{}, 0, 0);
        g_launches++;
    }
    return check_cuda(cudaGetLastError(), "quant launch");
}

template <int MODE, bool STOCH, typename OutT, bool kDevSeed = false>
static int launch_quant(const float* in, OutT* out, uint8_t* mask, int64_t n, int exp_bits,
                        int man_bits, FixedParams fp, uint64_t seed, uint64_t offset,
                        cudaStream_t st, const uint64_t* seed_dev = nullptr) {
    if (n == 0) return 0;
    const bool aligned = (reinterpret_cast<uintptr_t>(in) % 16 == 0) &&
                         (reinterpret_cast<uintptr_t>(out) % (4 * sizeof(OutT)) == 0) &&
                         (mask == nullptr || reinterpret_cast<uintptr_t>(mask) % 4 == 0);
    int64_t done = 0;
    if (aligned && n >= 4) {
        const int64_t n4 = n >> 2;
        quant_vec_kernel<MODE, STOCH, OutT, kDevSeed><<<grid_for(n4, kQThreads * kQUnroll), kQThreads, 0, st>>>(
            in, out, mask, n, exp_bits, man_bits, fp, seed, offset, seed_dev);
        g_launches++;
        done = n4 << 2;
    }
    if (done < n) {
        quant_scalar_kernel<MODE, STOCH, OutT, kDevSeed><<<grid_for(n - done, 256), 256, 0, st>>>(
            in, out, mask, done, n, exp_bits, man_bits, fp, seed, offset, seed_dev);
        g_launches++;
    }
    return check_cuda(cudaGetLastError(), "quant launch");
}

// ------------------------------------------------------------------ block quantize
__global__ void absmax_whole_kernel(const float* __restrict__ in, int64_t n, uint32_t* __restrict__ mx) {
    float m = 0.f;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        m = fmaxf(m, fabsf(in[i]));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ float sm[32];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.f;
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (threadIdx.x == 0) atomicMax(mx, __float_as_uint(m));   // non-negative floats order as uints
    }
}
// one block per (outer index u, dim index d) slab of `inner` contiguous elements
__global__ void absmax_dim_kernel(const float* __restrict__ in, int64_t dsize, int64_t inner,
                                  uint32_t* __restrict__ mx) {
    const int64_t slab = blockIdx.x;
    const int64_t d = slab % dsize;
    const float* p = in + slab * inner;
    float m = 0.f;
    for (int64_t i = threadIdx.x; i < inner; i += blockDim.x) m = fmaxf(m, fabsf(p[i]));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(mx + d, __float_as_uint(m));
}
// inner == 1 (dim is the last axis): threads across d (coalesced), loop over outer
__global__ void absmax_lastdim_kernel(const float* __restrict__ in, int64_t outer, int64_t dsize,
                                      uint32_t* __restrict__ mx) {
    const int64_t d = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (d >= dsize) return;
    float m = 0.f;
    for (int64_t u = blockIdx.y; u < outer; u += gridDim.y) m = fmaxf(m, fabsf(in[u * dsize + d]));
    atomicMax(mx + d, __float_as_uint(m));
}
// the same maxima with 16-byte loads (inner a multiple of 4, 16-byte aligned input): whole tensor (dsize = 1, one
// "slab" of n elements split over gridDim.x) or one (outer, d) slab per blockIdx.y
__global__ void __launch_bounds__(256)
absmax_vec_kernel(const float* __restrict__ in, int64_t dsize, int64_t inner4, int64_t nslabs, uint32_t* __restrict__ mx) {
    for (int64_t slab = blockIdx.y; slab < nslabs; slab += gridDim.y) {
        const float4* p = reinterpret_cast<const float4*>(in) + slab * inner4;
        float m = 0.f;
        const int64_t stride = int64_t(gridDim.x) * 256 * 4;
        for (int64_t j0 = int64_t(blockIdx.x) * 256 * 4 + threadIdx.x; j0 < inner4; j0 += stride) {
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int64_t j = j0 + u * 256;
                v[u] = j < inner4 ? __ldg(p + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; u++)
                m = fmaxf(m, fmaxf(fmaxf(fabsf(v[u].x), fabsf(v[u].y)), fmaxf(fabsf(v[u].z), fabsf(v[u].w))));
        }
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(mx + slab % dsize, __float_as_uint(m));
    }
}

// Random tail bits of block_quantize, as for float_quantize (include/mv_b200.h): wl >= 7 drops at most 16 bits and uses
// the 16-bit stream (eight elements per Philox call), wl < 7 the 32-bit stream.
template <bool STOCH>
__global__ void block_quant_kernel(const float* __restrict__ in, float* __restrict__ out,
                                   const float* __restrict__ mx, int64_t n, int64_t dsize,
                                   int64_t inner, int whole, int wl, uint64_t seed,
                                   uint64_t offset) {
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float m = whole ? mx[0] : mx[(i / inner) % dsize];
        uint32_t r = 0;
        if (STOCH) {
            if (wl >= 7) {
                r = philox_half16(seed, uint64_t(i), offset);
            } else {
                const uint4 w = philox4x32_10(seed, uint64_t(i >> 2), offset);
                const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
                r = ws[i & 3];
            }
        }
        out[i] = block_quantize_elem<STOCH>(in[i], m, r, wl);
    }
}

// Vectorised: a thread owns 8 consecutive elements (two 16-byte vectors) of one slab.  kLast: `dim` is the last axis
// (inner = 1, a "slab" = one outer row of dsize elements, the eight maxima are loaded as two vectors); otherwise the
// slab's maximum is looked up once per slab — no per-element divide.  Slabs (dsize * outer of them, or 1) on grid.y.
template <bool STOCH, bool kLast>
__global__ void __launch_bounds__(256)
block_quant_vec_kernel(const float* __restrict__ in, float* __restrict__ out, const float* __restrict__ mx,
                       int64_t dsize, int64_t len8, int64_t nslabs, int wl, uint64_t seed, uint64_t offset) {
    for (int64_t slab = blockIdx.y; slab < nslabs; slab += gridDim.y) {
        const float ms = kLast ? 0.f : mx[slab % dsize];
        const int64_t base8 = slab * len8;                           // index of the slab's first 8-element group
        const int64_t stride = int64_t(gridDim.x) * 256;
        for (int64_t j = int64_t(blockIdx.x) * 256 + threadIdx.x; j < len8; j += stride) {
            const int64_t g8 = base8 + j;
            const float4 a = __ldcs(reinterpret_cast<const float4*>(in) + 2 * g8);
            const float4 b = __ldcs(reinterpret_cast<const float4*>(in) + 2 * g8 + 1);
            float4 ma = make_float4(ms, ms, ms, ms), mb = ma;
            if (kLast) {
                ma = __ldg(reinterpret_cast<const float4*>(mx) + 2 * j);
                mb = __ldg(reinterpret_cast<const float4*>(mx) + 2 * j + 1);
            }
            uint32_t r[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            if (STOCH) {
                if (wl >= 7) {
                    const uint4 w = philox4x32_10(seed, uint64_t(g8), offset);
                    r[0] = w.x & 0xFFFFu; r[1] = w.x >> 16; r[2] = w.y & 0xFFFFu; r[3] = w.y >> 16;
                    r[4] = w.z & 0xFFFFu; r[5] = w.z >> 16; r[6] = w.w & 0xFFFFu; r[7] = w.w >> 16;
                } else {
                    const uint4 w0 = philox4x32_10(seed, uint64_t(2 * g8), offset);
                    const uint4 w1 = philox4x32_10(seed, uint64_t(2 * g8 + 1), offset);
                    r[0] = w0.x; r[1] = w0.y; r[2] = w0.z; r[3] = w0.w; r[4] = w1.x; r[5] = w1.y; r[6] = w1.z; r[7] = w1.w;
                }
            }
            float4 oa, ob;
            oa.x = block_quantize_elem<STOCH>(a.x, ma.x, r[0], wl); oa.y = block_quantize_elem<STOCH>(a.y, ma.y, r[1], wl);
            oa.z = block_quantize_elem<STOCH>(a.z, ma.z, r[2], wl); oa.w = block_quantize_elem<STOCH>(a.w, ma.w, r[3], wl);
            ob.x = block_quantize_elem<STOCH>(b.x, mb.x, r[4], wl); ob.y = block_quantize_elem<STOCH>(b.y, mb.y, r[5], wl);
            ob.z = block_quantize_elem<STOCH>(b.z, mb.z, r[6], wl); ob.w = block_quantize_elem<STOCH>(b.w, mb.w, r[7], wl);
            __stcs(reinterpret_cast<float4*>(out) + 2 * g8, oa);
            __stcs(reinterpret_cast<float4*>(out) + 2 * g8 + 1, ob);
        }
    }
}

__global__ void philox_dump_kernel(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset) {
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint4 w = philox4x32_10(seed, uint64_t(i >> 2), offset);
        const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
        out[i] = ws[i & 3];
    }
}

__global__ void philox_dump16_kernel(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset) {
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = philox_half16(seed, uint64_t(i), offset);
}

// --------------------------------------------------------- weight quant (+ transpose)
// 32x32 tiles through shared memory so both q(W) and q(W)^T are written coalesced.
template <typename OutT>
__global__ void quant_weight_kernel(const float* __restrict__ w, OutT* __restrict__ out,
                                    OutT* __restrict__ out_t, int rows, int cols, int exp_bits,
                                    int man_bits) {
    __shared__ float tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        float v = 0.f;
        if (r < rows && c < cols) {
            v = w[int64_t(r) * cols + c];
            if (exp_bits > 0) v = float_quantize_elem<false>(v, 0u, exp_bits, man_bits);
            out[int64_t(r) * cols + c] = cvt_out<OutT>(v);
        }
        tile[j][threadIdx.x] = v;
    }
    if (out_t == nullptr) return;
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < rows && c < cols) out_t[int64_t(c) * rows + r] = cvt_out<OutT>(tile[threadIdx.x][j]);
    }
}

}  // namespace mv

using namespace mv;

extern "C" int mv_float_quantize(const float* in, void* out, int out_dtype, int64_t n, int exp_bits,
                                 int man_bits, int rounding, uint64_t seed, uint64_t offset,
                                 void* stream) {
    MV_CHECK(n >= 0, "mv_float_quantize: negative n");
    MV_CHECK(exp_bits >= 1 && exp_bits <= 8, "mv_float_quantize: exp_bits %d not in [1,8]", exp_bits);
    MV_CHECK(man_bits >= 1 && man_bits <= 22, "mv_float_quantize: man_bits %d not in [1,22]", man_bits);
    MV_CHECK(n == 0 || (in && out), "mv_float_quantize: null buffer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FixedParams fp{};
    // stochastic rounding of a tail of at most 16 bits: the 16-bit stream (eight elements per Philox call)
    const bool s16 = rounding == MV_ROUND_STOCHASTIC && man_bits >= 7;
    if (out_dtype == MV_F32) {
        if (s16) return launch_quant16<float>(in, (float*)out, n, exp_bits, man_bits, seed, offset, st);
        return rounding == MV_ROUND_STOCHASTIC
                   ? launch_quant<0, true, float>(in, (float*)out, nullptr, n, exp_bits, man_bits, fp, seed, offset, st)
                   : launch_quant_nearest8<float>(in, (float*)out, n, exp_bits, man_bits, st);
    }
    MV_CHECK(out_dtype == MV_F16, "mv_float_quantize: unsupported out_dtype %d", out_dtype);
    MV_CHECK(exp_bits <= 5 && man_bits <= 10,
             "mv_float_quantize: (exp=%d, man=%d) is not exactly representable in an fp16 container",
             exp_bits, man_bits);
    if (s16) return launch_quant16<__half>(in, (__half*)out, n, exp_bits, man_bits, seed, offset, st);
    return rounding == MV_ROUND_STOCHASTIC
               ? launch_quant<0, true, __half>(in, (__half*)out, nullptr, n, exp_bits, man_bits, fp, seed, offset, st)
               : launch_quant_nearest8<__half>(in, (__half*)out, n, exp_bits, man_bits, st);
}

extern "C" int mv_float_quantize_dev(const float* in, void* out, int out_dtype, int64_t n, int exp_bits, int man_bits,
                                     const uint64_t* seed_dev, uint64_t offset, void* stream) {
    MV_CHECK(n >= 0, "mv_float_quantize_dev: negative n");
    MV_CHECK(exp_bits >= 1 && exp_bits <= 8, "mv_float_quantize_dev: exp_bits %d not in [1,8]", exp_bits);
    MV_CHECK(man_bits >= 1 && man_bits <= 22, "mv_float_quantize_dev: man_bits %d not in [1,22]", man_bits);
    MV_CHECK(n == 0 || (in && out && seed_dev), "mv_float_quantize_dev: null buffer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FixedParams fp{};
    const bool s16 = man_bits >= 7;             // the streams of mv_float_quantize, MV_ROUND_STOCHASTIC
    if (out_dtype == MV_F32) {
        if (s16) return launch_quant16<float, true>(in, (float*)out, n, exp_bits, man_bits, 0, offset, st, seed_dev);
        return launch_quant<0, true, float, true>(in, (float*)out, nullptr, n, exp_bits, man_bits, fp, 0, offset, st, seed_dev);
    }
    MV_CHECK(out_dtype == MV_F16, "mv_float_quantize_dev: unsupported out_dtype %d", out_dtype);
    MV_CHECK(exp_bits <= 5 && man_bits <= 10,
             "mv_float_quantize_dev: (exp=%d, man=%d) is not exactly representable in an fp16 container", exp_bits, man_bits);
    if (s16) return launch_quant16<__half, true>(in, (__half*)out, n, exp_bits, man_bits, 0, offset, st, seed_dev);
    return launch_quant<0, true, __half, true>(in, (__half*)out, nullptr, n, exp_bits, man_bits, fp, 0, offset, st, seed_dev);
}

extern "C" int mv_fixed_point_quantize(const float* in, float* out, uint8_t* mask, int64_t n, int wl,
                                       int fl, int clamp, int symmetric, int rounding,
                                       uint64_t seed, uint64_t offset, void* stream) {
    MV_CHECK(n >= 0, "mv_fixed_point_quantize: negative n");
    MV_CHECK(wl >= 1 && wl <= 32 && fl >= -100 && fl <= 100, "mv_fixed_point_quantize: bad wl/fl %d/%d", wl, fl);
    MV_CHECK(n == 0 || (in && out), "mv_fixed_point_quantize: null buffer");
    FixedParams fp;
    fp.scale_up = ldexpf(1.0f, fl);
    fp.scale_down = ldexpf(1.0f, -fl);
    fp.t_min = -ldexpf(1.0f, wl - fl - 1);
    fp.t_max = -fp.t_min - ldexpf(1.0f, -fl);
    if (symmetric) fp.t_min = fp.t_min + ldexpf(1.0f, -fl);
    fp.clamp = clamp;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return rounding == MV_ROUND_STOCHASTIC
               ? launch_quant<1, true, float>(in, out, mask, n, 0, 0, fp, seed, offset, st)
               : launch_quant<1, false, float>(in, out, mask, n, 0, 0, fp, seed, offset, st);
}

extern "C" int mv_block_quantize(const float* in, float* out, float* workspace, int64_t outer,
                                 int64_t dsize, int64_t inner, int whole_tensor, int wl,
                                 int rounding, uint64_t seed, uint64_t offset, void* stream) {
    const int64_t n = outer * dsize * inner;
    MV_CHECK(n >= 0 && wl >= 1 && wl <= 22, "mv_block_quantize: bad arguments");
    if (n == 0) return 0;
    MV_CHECK(in && out && workspace, "mv_block_quantize: null buffer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint32_t* mx = reinterpret_cast<uint32_t*>(workspace);
    const int64_t nblk = whole_tensor ? 1 : dsize;
    MV_CUDA(cudaMemsetAsync(mx, 0, sizeof(uint32_t) * nblk, st));
    // vector paths: 16-byte aligned buffers and slabs that are multiples of 8 elements
    const bool al16 = reinterpret_cast<uintptr_t>(in) % 16 == 0 && reinterpret_cast<uintptr_t>(out) % 16 == 0 &&
                      reinterpret_cast<uintptr_t>(workspace) % 16 == 0;
    const bool vec_whole = al16 && whole_tensor && n % 8 == 0;
    const bool vec_slab = al16 && !whole_tensor && inner > 1 && inner % 8 == 0;
    const bool vec_last = al16 && !whole_tensor && inner == 1 && dsize % 8 == 0;
    auto grid2 = [](int64_t len_items, int per_block, int64_t nslabs) {
        int64_t gx = (len_items + per_block - 1) / per_block;
        const int64_t gy = nslabs < 65535 ? nslabs : 65535;
        const int64_t cap = (int64_t(kNumSMs) * 16 + gy - 1) / gy;              // about 16 CTAs per SM in total
        if (gx > cap) gx = cap;
        if (gx < 1) gx = 1;
        return dim3((unsigned)gx, (unsigned)gy);
    };
    if (vec_whole) {
        absmax_vec_kernel<<<grid2(n / 4, 256 * 4, 1), 256, 0, st>>>(in, 1, n / 4, 1, mx);
    } else if (vec_slab) {
        absmax_vec_kernel<<<grid2(inner / 4, 256 * 4, outer * dsize), 256, 0, st>>>(in, dsize, inner / 4, outer * dsize, mx);
    } else if (whole_tensor) {
        absmax_whole_kernel<<<grid_for(n, 256 * 8), 256, 0, st>>>(in, n, mx);
    } else if (inner == 1) {
        dim3 grid((unsigned)((dsize + 255) / 256), (unsigned)(outer < 64 ? outer : 64));
        absmax_lastdim_kernel<<<grid, 256, 0, st>>>(in, outer, dsize, mx);
    } else {
        MV_CHECK(outer * dsize < (int64_t(1) << 31), "mv_block_quantize: too many slabs");
        absmax_dim_kernel<<<(unsigned)(outer * dsize), 128, 0, st>>>(in, dsize, inner, mx);
    }
    g_launches++;
    const bool stoch = rounding == MV_ROUND_STOCHASTIC;
    if (vec_whole || vec_slab || vec_last) {
        const int64_t nslabs = vec_whole ? 1 : (vec_slab ? outer * dsize : outer);
        const int64_t len8 = (vec_whole ? n : (vec_slab ? inner : dsize)) / 8;
        const int64_t ds = vec_whole ? 1 : dsize;
        const dim3 grid = grid2(len8, 256, nslabs);
        if (vec_last) {
            if (stoch) block_quant_vec_kernel<true, true><<<grid, 256, 0, st>>>(in, out, workspace, ds, len8, nslabs, wl, seed, offset);
            else block_quant_vec_kernel<false, true><<<grid, 256, 0, st>>>(in, out, workspace, ds, len8, nslabs, wl, seed, offset);
        } else {
            if (stoch) block_quant_vec_kernel<true, false><<<grid, 256, 0, st>>>(in, out, workspace, ds, len8, nslabs, wl, seed, offset);
            else block_quant_vec_kernel<false, false><<<grid, 256, 0, st>>>(in, out, workspace, ds, len8, nslabs, wl, seed, offset);
        }
        g_launches++;
        return check_cuda(cudaGetLastError(), "block quant launch");
    }
    if (rounding == MV_ROUND_STOCHASTIC)
        block_quant_kernel<true><<<grid_for(n, 256 * 4), 256, 0, st>>>(in, out, workspace, n, dsize, inner, whole_tensor, wl, seed, offset);
    else
        block_quant_kernel<false><<<grid_for(n, 256 * 4), 256, 0, st>>>(in, out, workspace, n, dsize, inner, whole_tensor, wl, seed, offset);
    g_launches++;
    return check_cuda(cudaGetLastError(), "block quant launch");
}

extern "C" int mv_philox_bits16(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, void* stream) {
    if (n <= 0) return 0;
    philox_dump16_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(out, n, seed, offset);
    g_launches++;
    return check_cuda(cudaGetLastError(), "philox dump launch");
}
extern "C" int mv_philox_bits(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, void* stream) {
    if (n <= 0) return 0;
    philox_dump_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(out, n, seed, offset);
    g_launches++;
    return check_cuda(cudaGetLastError(), "philox dump launch");
}

extern "C" int mv_quantize_weight(const float* w, void* out, void* out_t, int out_dtype, int rows,
                                  int cols, int exp_bits, int man_bits, void* stream) {
    MV_CHECK(rows > 0 && cols > 0 && w && out, "mv_quantize_weight: bad arguments");
    dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (out_dtype == MV_F16) {
        MV_CHECK(exp_bits >= 1 && exp_bits <= 5 && man_bits <= 10, "mv_quantize_weight: format does not fit fp16");
        quant_weight_kernel<__half><<<grid, block, 0, st>>>(w, (__half*)out, (__half*)out_t, rows, cols, exp_bits, man_bits);
    } else {
        MV_CHECK(out_dtype == MV_F32, "mv_quantize_weight: unsupported container");
        quant_weight_kernel<float><<<grid, block, 0, st>>>(w, (float*)out, (float*)out_t, rows, cols, exp_bits, man_bits);
    }
    g_launches++;
    return check_cuda(cudaGetLastError(), "quant weight launch");
}
