// norm.cu — warp-shuffle LayerNorm forward/backward fused with its fake-quantisers, plus the
// small memory-bound helpers of the step (north-star kernel class (c)).
//
// Forward (one warp per token row, row held in registers, 128-bit accesses):
//     y = q_post( LN( q_in(x) ; gamma, beta ) )      -> fp16 / fp32 container
// which is the reference's Sequential(QuantStub, LayerNorm) followed by the next Linear's
// QuantStub (src/myrtle_vision/models/vit.py:37-41, utils/quantize.py:215-220, Appendix A of
// SURVEY.md); q is idempotent so LN-output quant (FP16_16) and the next stub collapse.
// Backward (straight-through quantisers, utils/quantize.py:87-89):
//     dx = LN'(dy; q_in(x)) + dres,   dgamma += sum dy*xhat,   dbeta += sum dy,
//     dbias_prev += sum dx   (bias gradient of the Linear that produced the residual stream)
// HBM traffic per element: fwd 4 B read + 2 B write (fp16 container); bwd 12 B read + 6 B write.
#include <type_traits>

#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {

extern int64_t g_launches;

constexpr int kLnWarps = 8;
constexpr int kLnMaxVec = 8;     // float4 per lane: D <= 32*4*8 = 1024

__device__ __forceinline__ float sat16(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
// two fp32 -> packed fp16x2, round-to-nearest, clipped to +-65504 in the conversion itself
__device__ __forceinline__ uint32_t pack_h2_sat(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <int NV, typename OutT>
__global__ void __launch_bounds__(kLnWarps * 32, 4)
ln_fwd_kernel(const float* __restrict__ x, int64_t ld_x, const float* __restrict__ gamma,
              const float* __restrict__ beta, OutT* __restrict__ y, int64_t ld_y,
              float* __restrict__ mean_out, float* __restrict__ rstd_out, int rows, int D, float eps,
              FloatFmt q_in, FloatFmt q_post) {
    // Each warp owns two rows per iteration: both rows' loads are issued before either is
    // reduced, doubling the bytes in flight per warp.  gamma/beta stay in L1 (re-read per row)
    // instead of occupying 2*NV*4 registers.
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nvec = D >> 2;
    const int mi = fq_mode(q_in), mp = fq_mode(q_post);
    const float inv_d = 1.0f / float(D);
    const int wstride = gridDim.x * kLnWarps * 2;
    for (int row0 = (blockIdx.x * kLnWarps + warp) * 2; row0 < rows; row0 += wstride) {
        float4 v[2][NV];
        float s[2] = {0.f, 0.f};
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
            const int row = row0 + rr;
            const float4* xr = reinterpret_cast<const float4*>(x + int64_t(row) * ld_x);
#pragma unroll
            for (int i = 0; i < NV; i++) {
                const int c = lane + 32 * i;
                if (c < nvec && row < rows) v[rr][i] = __ldcs(xr + c);
                else v[rr][i] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
#pragma unroll
            for (int i = 0; i < NV; i++) {
                if (mi == 1) {
                    v[rr][i] = fq_half4_f32(v[rr][i]);          // one range test per four values
                } else {
                    v[rr][i].x = fq_apply(v[rr][i].x, mi, q_in); v[rr][i].y = fq_apply(v[rr][i].y, mi, q_in);
                    v[rr][i].z = fq_apply(v[rr][i].z, mi, q_in); v[rr][i].w = fq_apply(v[rr][i].w, mi, q_in);
                }
                s[rr] += (v[rr][i].x + v[rr][i].y) + (v[rr][i].z + v[rr][i].w);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s[0] += __shfl_xor_sync(0xffffffffu, s[0], o);
            s[1] += __shfl_xor_sync(0xffffffffu, s[1], o);
        }
        const float mean[2] = {s[0] * inv_d, s[1] * inv_d};
        float ss[2] = {0.f, 0.f};
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
#pragma unroll
            for (int i = 0; i < NV; i++) {
                const int c = lane + 32 * i;
                if (c < nvec) {
                    const float dx = v[rr][i].x - mean[rr], dy = v[rr][i].y - mean[rr];
                    const float dz = v[rr][i].z - mean[rr], dw = v[rr][i].w - mean[rr];
                    ss[rr] += (dx * dx + dy * dy) + (dz * dz + dw * dw);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            ss[0] += __shfl_xor_sync(0xffffffffu, ss[0], o);
            ss[1] += __shfl_xor_sync(0xffffffffu, ss[1], o);
        }
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
            const int row = row0 + rr;
            if (row >= rows) break;
            const float rstd = rsqrtf(ss[rr] * inv_d + eps);
            if (lane == 0 && mean_out != nullptr) { mean_out[row] = mean[rr]; rstd_out[row] = rstd; }
            OutT* yr = y + int64_t(row) * ld_y;
#pragma unroll
            for (int i = 0; i < NV; i++) {
                const int c = lane + 32 * i;
                if (c < nvec) {
                    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c);
                    const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + c);
                    float4 o;
                    o.x = fmaf((v[rr][i].x - mean[rr]) * rstd, g.x, b.x);
                    o.y = fmaf((v[rr][i].y - mean[rr]) * rstd, g.y, b.y);
                    o.z = fmaf((v[rr][i].z - mean[rr]) * rstd, g.z, b.z);
                    o.w = fmaf((v[rr][i].w - mean[rr]) * rstd, g.w, b.w);
                    if (mp == 1 && sizeof(OutT) == 2) {
                        // quantise + convert + pack in one step (cvt.rz on the half-ulp-biased word)
                        __stcs(reinterpret_cast<uint2*>(yr) + c, fq_half4_pack(o.x, o.y, o.z, o.w));
                        continue;
                    }
                    o.x = fq_apply(o.x, mp, q_post); o.y = fq_apply(o.y, mp, q_post);
                    o.z = fq_apply(o.z, mp, q_post); o.w = fq_apply(o.w, mp, q_post);
                    if (sizeof(OutT) == 4) {
                        __stcs(reinterpret_cast<float4*>(yr) + c, o);
                    } else {
                        __half2 lo = __floats2half2_rn(o.x, o.y), hi = __floats2half2_rn(o.z, o.w);
                        __stcs(reinterpret_cast<uint2*>(yr) + c, make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi)));
                    }
                }
            }
        }
    }
}

// dy: fp32 [rows, D] gradient w.r.t. the LN output; dres: fp32 [rows, D] gradient flowing
// along the residual connection (nullable); dx (fp32) and dx_lp (fp16, nullable) receive
// LN'(dy) + dres.  Column sums are accumulated per lane over the warp's rows, reduced across
// the CTA in shared memory and added to global memory with one atomic per column per CTA.
__device__ __forceinline__ float4 load_dy4(const float* p, int c) { return __ldcs(reinterpret_cast<const float4*>(p) + c); }
__device__ __forceinline__ float4 load_dy4(const __half* p, int c) {
    const uint2 u = __ldcs(reinterpret_cast<const uint2*>(p) + c);
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

template <int NV, typename DyT> struct LnBwdRow {
    float4 x[NV];
    float4 dres[NV];
    typename std::conditional<sizeof(DyT) == 2, uint2, float4>::type dy[NV];
};
__device__ __forceinline__ float4 unpack_dy(const float4& v) { return v; }
__device__ __forceinline__ float4 unpack_dy(const uint2& u) {
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
    const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    return make_float4(a.x, a.y, b.x, b.y);
}

// kGQ: the gradient quantiser of the LayerNorm's input stub (QPyTorch backward_number; q_grad) rounds the
// LayerNorm-input gradient before the residual gradient is added to it
// kDrop: dropout mask `drop` on dx_lp and dbias_prev (and on dx when mask_dx): the gradient of the dropped branch that the
// residual stream's producer receives.  A lane owns float4 c = lane + 32 i; with D % 8 == 0 lanes 2k / 2k+1 hold the two
// halves of one Philox block, so vectors i and i+1 take one call per lane (drop_keep4_pair).  Separate instantiations:
// the kernels without it keep their register allocation.
// kSR (with kGQ): the gradient quantiser rounds stochastically with the gradient rounding stream `sr` (element
// row * D + c of the site tensor; one Philox call per lane and float4).  Separate instantiations likewise.
template <int NV, typename DyT, bool kGQ = false, bool kDrop = false, bool kSR = false>
__global__ void __launch_bounds__(kLnWarps * 32, 2)
ln_bwd_kernel(const DyT* __restrict__ dy, int64_t ld_dy, const float* __restrict__ x, int64_t ld_x,
              const float* __restrict__ dres, int64_t ld_dres, const float* __restrict__ gamma,
              const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
              float* __restrict__ dx, int64_t ld_dx, __half* __restrict__ dx_lp, int64_t ld_lp,
              float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ dbias_prev,
              int rows, int D, FloatFmt q_in, int* __restrict__ ovf, FloatFmt q_grad = FloatFmt{0, 0},
              DropDev drop = DropDev{nullptr, 0u, 0.f, 0}, int mask_dx = 0, SrDev sr = SrDev{nullptr, 0ull}) {
    // Column sums (dgamma, dbeta, previous bias grad) are kept per warp in shared memory — each
    // lane owns its columns, so plain read-modify-write — which frees ~36 registers per thread for
    // occupancy; the next row's loads are issued before the current row is reduced.
    extern __shared__ float red[];      // [kLnWarps][3][D]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nvec = D >> 2;
    const int mi = fq_mode(q_in);
    const float inv_d = 1.0f / float(D);
    float4* acc = reinterpret_cast<float4*>(red + size_t(warp) * 3 * D);
    using dy_vec = typename std::conditional<sizeof(DyT) == 2, uint2, float4>::type;
#pragma unroll
    for (int i = 0; i < NV; i++) {
        const int c = lane + 32 * i;
        if (c < nvec) {
            acc[c] = make_float4(0, 0, 0, 0); acc[nvec + c] = make_float4(0, 0, 0, 0); acc[2 * nvec + c] = make_float4(0, 0, 0, 0);
        }
    }
    const int rstride = gridDim.x * kLnWarps;
    auto load_row = [&](int row, LnBwdRow<NV, DyT>& r) {
        const float4* xr = reinterpret_cast<const float4*>(x + int64_t(row) * ld_x);
        const dy_vec* dyr = reinterpret_cast<const dy_vec*>(dy + int64_t(row) * ld_dy);
        const float4* rr = reinterpret_cast<const float4*>(dres + int64_t(row) * ld_dres);
#pragma unroll
        for (int i = 0; i < NV; i++) {
            const int c = lane + 32 * i;
            if (c < nvec) {
                r.x[i] = __ldcs(xr + c);
                r.dy[i] = __ldcs(dyr + c);
                if (dres != nullptr) r.dres[i] = __ldcs(rr + c);
            }
        }
    };
    int row = blockIdx.x * kLnWarps + warp;
    const uint64_t seed = kDrop ? __ldg(reinterpret_cast<const unsigned long long*>(drop.seed)) : 0ull;
    const uint64_t sr_s = kSR ? sr_seed(sr) : 0ull;
    LnBwdRow<NV, DyT> cur;
    float amax = 0.f;                   // largest |dx| rounded into the fp16 operand copy (overflow sink)
    if (row < rows) load_row(row, cur);
    for (; row < rows; row += rstride) {
        LnBwdRow<NV, DyT> nxt;
        const int nrow = row + rstride;
        if (nrow < rows) load_row(nrow, nxt);
        const float mean = mean_in[row], rstd = rstd_in[row];
        const float nmr = -mean * rstd;
        float4 xh[NV], gy[NV];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < NV; i++) {
            const int c = lane + 32 * i;
            if (c < nvec) {
                const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + c);
                const float4 d = unpack_dy(cur.dy[i]);
                float4 xv = cur.x[i];
                if (mi == 1) {
                    xv = fq_half4_f32(xv);
                } else {
                    xv.x = fq_apply(xv.x, mi, q_in); xv.y = fq_apply(xv.y, mi, q_in);
                    xv.z = fq_apply(xv.z, mi, q_in); xv.w = fq_apply(xv.w, mi, q_in);
                }
                xv.x = fmaf(xv.x, rstd, nmr); xv.y = fmaf(xv.y, rstd, nmr);       // (x - mean) * rstd
                xv.z = fmaf(xv.z, rstd, nmr); xv.w = fmaf(xv.w, rstd, nmr);
                xh[i] = xv;
                float4 a = acc[c];
                a.x = fmaf(d.x, xv.x, a.x); a.y = fmaf(d.y, xv.y, a.y); a.z = fmaf(d.z, xv.z, a.z); a.w = fmaf(d.w, xv.w, a.w);
                acc[c] = a;
                float4 bsum = acc[nvec + c];
                bsum.x += d.x; bsum.y += d.y; bsum.z += d.z; bsum.w += d.w;
                acc[nvec + c] = bsum;
                gy[i] = make_float4(d.x * g.x, d.y * g.y, d.z * g.z, d.w * g.w);
                s1 += (gy[i].x + gy[i].y) + (gy[i].z + gy[i].w);
                s2 += (gy[i].x * xv.x + gy[i].y * xv.y) + (gy[i].z * xv.z + gy[i].w * xv.w);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        // dx = rstd * (gy - mean(gy) - xhat * mean(gy * xhat))  as two FMAs per value
        const float cb = -rstd * (s2 * inv_d), cc = -rstd * (s1 * inv_d);
        float* dxr = dx + int64_t(row) * ld_dx;
        uint32_t keep = 0;                  // bits 4 i .. 4 i + 3: the four columns of float4 i
        if (kDrop) {
            const bool odd = lane & 1;
            const uint64_t rbase = uint64_t(row) * uint64_t(D);
#pragma unroll
            for (int i = 0; i < NV; i += 2) {
                if (i + 1 < NV && (D & 7) == 0) {
                    const uint64_t e = rbase + 4ull * uint64_t(lane + 32 * (i + (odd ? 1 : 0)));
                    keep |= drop_keep4_pair(seed, drop, e >> 3, odd) << (4 * i);
                } else {
                    keep |= drop_keep4(seed, drop, rbase + 4ull * uint64_t(lane + 32 * i)) << (4 * i);
                    if (i + 1 < NV) keep |= drop_keep4(seed, drop, rbase + 4ull * uint64_t(lane + 32 * (i + 1))) << (4 * (i + 1));
                }
            }
        }
#pragma unroll
        for (int i = 0; i < NV; i++) {
            const int c = lane + 32 * i;
            if (c < nvec) {
                float4 o;
                o.x = fmaf(gy[i].x, rstd, fmaf(xh[i].x, cb, cc)); o.y = fmaf(gy[i].y, rstd, fmaf(xh[i].y, cb, cc));
                o.z = fmaf(gy[i].z, rstd, fmaf(xh[i].z, cb, cc)); o.w = fmaf(gy[i].w, rstd, fmaf(xh[i].w, cb, cc));
                if (kGQ && kSR) {
                    const uint4 r = sr_bits4(sr_s, sr.offset, uint64_t(row) * uint64_t(D) + 4ull * uint64_t(c), q_grad.man_bits >= 7);
                    o.x = float_quantize_elem<true>(o.x, r.x, q_grad.exp_bits, q_grad.man_bits);
                    o.y = float_quantize_elem<true>(o.y, r.y, q_grad.exp_bits, q_grad.man_bits);
                    o.z = float_quantize_elem<true>(o.z, r.z, q_grad.exp_bits, q_grad.man_bits);
                    o.w = float_quantize_elem<true>(o.w, r.w, q_grad.exp_bits, q_grad.man_bits);
                } else if (kGQ) {
                    o.x = fq_nearest(o.x, q_grad); o.y = fq_nearest(o.y, q_grad);
                    o.z = fq_nearest(o.z, q_grad); o.w = fq_nearest(o.w, q_grad);
                }
                if (dres != nullptr) {
                    const float4 r = cur.dres[i];
                    o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
                }
                float4 om = o;              // what the dropped branch receives
                if (kDrop) {
                    om.x *= drop_mul(keep, 4 * i, drop.scale); om.y *= drop_mul(keep, 4 * i + 1, drop.scale);
                    om.z *= drop_mul(keep, 4 * i + 2, drop.scale); om.w *= drop_mul(keep, 4 * i + 3, drop.scale);
                    if (mask_dx) o = om;
                }
                float4 ps = acc[2 * nvec + c];
                ps.x += om.x; ps.y += om.y; ps.z += om.z; ps.w += om.w;
                acc[2 * nvec + c] = ps;
                __stcs(reinterpret_cast<float4*>(dxr) + c, o);
                if (dx_lp != nullptr) {
                    amax = fmaxf(amax, fmaxf(fmaxf(fabsf(om.x), fabsf(om.y)), fmaxf(fabsf(om.z), fabsf(om.w))));
                    __stcs(reinterpret_cast<uint2*>(dx_lp + int64_t(row) * ld_lp) + c,
                           make_uint2(pack_h2_sat(om.x, om.y), pack_h2_sat(om.z, om.w)));
                }
            }
        }
        cur = nxt;
    }
    raise_overflow(ovf, amax);
    __syncthreads();
    // CTA-level column reduction over the warps, then one atomic per column per CTA
    for (int which = 0; which < 3; which++) {
        float* dst = which == 0 ? dgamma : (which == 1 ? dbeta : dbias_prev);
        if (dst == nullptr) continue;
        for (int c = threadIdx.x; c < D; c += blockDim.x) {
            float sacc = 0.f;
#pragma unroll
            for (int w = 0; w < kLnWarps; w++) sacc += red[(size_t(w) * 3 + which) * D + c];
            atomicAdd(dst + c, sacc);
        }
    }
}

// out[c] += sum_r in[r, c]   (bias gradients of to_qkv / net.0 from their fp16 dY)
// A warp reads 256 (fp16) or 128 (fp32) consecutive columns of a row with one 16-byte load per
// lane, four rows in flight; the 8 warps of a CTA stride over rows and are combined in shared
// memory before one atomicAdd per column.
template <typename T>
__global__ void __launch_bounds__(256)
colsum_kernel(const T* __restrict__ in, int64_t ld, int rows, int cols, float* __restrict__ out) {
    constexpr int VEC = 16 / sizeof(T);               // elements per 16-byte load
    __shared__ float sm[8][32 * VEC + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int c0 = (blockIdx.x * 32 + lane) * VEC;
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; j++) acc[j] = 0.f;
    if (c0 < cols) {
        const int rstride = gridDim.y * 8;
        int r = blockIdx.y * 8 + warp;
        for (; r + 3 * rstride < rows; r += 4 * rstride) {
            uint4 w[4];
#pragma unroll
            for (int u = 0; u < 4; u++)
                w[u] = __ldcs(reinterpret_cast<const uint4*>(in + int64_t(r + u * rstride) * ld + c0));
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (sizeof(T) == 2) {
                    const __half2* h = reinterpret_cast<const __half2*>(&w[u]);
#pragma unroll
                    for (int j = 0; j < 4; j++) { const float2 f = __half22float2(h[j]); acc[2 * j] += f.x; acc[2 * j + 1] += f.y; }
                } else {
                    const float* f = reinterpret_cast<const float*>(&w[u]);
#pragma unroll
                    for (int j = 0; j < VEC; j++) acc[j] += f[j];
                }
            }
        }
        for (; r < rows; r += rstride) {
            const uint4 w = __ldcs(reinterpret_cast<const uint4*>(in + int64_t(r) * ld + c0));
            if (sizeof(T) == 2) {
                const __half2* h = reinterpret_cast<const __half2*>(&w);
#pragma unroll
                for (int j = 0; j < 4; j++) { const float2 f = __half22float2(h[j]); acc[2 * j] += f.x; acc[2 * j + 1] += f.y; }
            } else {
                const float* f = reinterpret_cast<const float*>(&w);
#pragma unroll
                for (int j = 0; j < VEC; j++) acc[j] += f[j];
            }
        }
    }
#pragma unroll
    for (int j = 0; j < VEC; j++) sm[warp][lane * VEC + j] = acc[j];
    __syncthreads();
    for (int t = threadIdx.x; t < 32 * VEC; t += 256) {
        const int c = blockIdx.x * 32 * VEC + t;
        if (c < cols) {
            float sacc = 0.f;
#pragma unroll
            for (int w8 = 0; w8 < 8; w8++) sacc += sm[w8][t];
            atomicAdd(out + c, sacc);
        }
    }
}

// patchify + input quant:  img NCHW fp32 -> patches [B*gh*gw, p*p*C] with (ph, pw, c) minor
// order (src/myrtle_vision/models/vit.py:271-275), each value through q_in, fp16/fp32 container.
// kMix: image b is first mixed with image B - 1 - b as recs[b] says (mv_patchify_mix_q); recs is unused otherwise.
template <typename OutT, bool kMix>
__global__ void __launch_bounds__(256)
patchify_kernel(const float* __restrict__ img, OutT* __restrict__ out, int B, int C, int H, int W,
                int P, FloatFmt q_in, int cls_slot, const mv_mix_rec* __restrict__ recs) {
    // One CTA per (b, patch row gy).  Phase 1 reads the C x P image rows (W contiguous floats each,
    // 16-byte loads), quantises and scatters them into shared memory at their OUTPUT position
    // [gx][ph][pw][c] (the index arithmetic is per 16-byte load, not per element); phase 2 copies the
    // gw * pdim elements of this patch row — one contiguous span of `out` — with 16-byte vectors.
    extern __shared__ __align__(16) uint8_t patch_smem[];
    OutT* sm = reinterpret_cast<OutT*>(patch_smem);
    const int gw = W / P, gh = H / P;
    const int b = blockIdx.x / gh, gy = blockIdx.x % gh;
    const int pdim = P * P * C;
    const int PC = P * C;
    const int64_t rows_per_img = int64_t(gh) * gw + cls_slot;
    OutT* obase = out + (int64_t(b) * rows_per_img + (cls_slot != 0) + int64_t(gy) * gw) * pdim;
    if (cls_slot && gy == 0) {          // row b*N + 0 is the (zero) slot of the class token
        OutT* z = out + int64_t(b) * rows_per_img * pdim;
        for (int i = threadIdx.x; i < pdim; i += blockDim.x) z[i] = OutT(0.f);
        if (cls_slot == 2) {            // ... and row b*N + N-1 the (zero) slot of the distillation token
            z += (rows_per_img - 1) * pdim;
            for (int i = threadIdx.x; i < pdim; i += blockDim.x) z[i] = OutT(0.f);
        }
    }
    const int mode = fq_mode(q_in);
    const int w4 = W >> 2;              // W % 4 == 0 checked on the host
    [[maybe_unused]] mv_mix_rec rec;
    if constexpr (kMix) {               // the record, read once per CTA
        __shared__ mv_mix_rec sm_rec;
        if (threadIdx.x == 0) sm_rec = recs[b];
        __syncthreads();
        rec = sm_rec;
    }
    for (int i = threadIdx.x; i < C * P * w4; i += blockDim.x) {
        const int wv = i % w4, r = i / w4;                 // r = c * P + ph
        const int c = r / P, ph = r % P;
        float4 v = __ldcs(reinterpret_cast<const float4*>(img + ((int64_t(b) * C + c) * H + gy * P + ph) * W) + wv);
        if constexpr (kMix) {
            const int y = gy * P + ph, x = wv * 4;
            const float4* prow = reinterpret_cast<const float4*>(img + ((int64_t(B - 1 - b) * C + c) * H + y) * W) + wv;
            if (rec.cutmix) {                              // only the vectors that overlap the box read the partner
                if (y >= rec.y0 && y < rec.y1 && x + 4 > rec.x0 && x < rec.x1) {
                    const float4 p = __ldcs(prow);
                    if (x >= rec.x0 && x < rec.x1) v.x = p.x;
                    if (x + 1 >= rec.x0 && x + 1 < rec.x1) v.y = p.y;
                    if (x + 2 >= rec.x0 && x + 2 < rec.x1) v.z = p.z;
                    if (x + 3 >= rec.x0 && x + 3 < rec.x1) v.w = p.w;
                }
            } else if (rec.w_other != 0.f || rec.w_self != 1.f) {   // Mixup: two rounded products, one rounded add
                const float4 p = __ldcs(prow);
                v.x = __fadd_rn(__fmul_rn(rec.w_self, v.x), __fmul_rn(rec.w_other, p.x));
                v.y = __fadd_rn(__fmul_rn(rec.w_self, v.y), __fmul_rn(rec.w_other, p.y));
                v.z = __fadd_rn(__fmul_rn(rec.w_self, v.z), __fmul_rn(rec.w_other, p.z));
                v.w = __fadd_rn(__fmul_rn(rec.w_self, v.w), __fmul_rn(rec.w_other, p.w));
            }
        }
        if (mode == 1) v = fq_half4_f32(v);
        else { v.x = fq_apply(v.x, mode, q_in); v.y = fq_apply(v.y, mode, q_in); v.z = fq_apply(v.z, mode, q_in); v.w = fq_apply(v.w, mode, q_in); }
        const int w = wv * 4;
        if ((P & 3) == 0) {                                // the four pixels share a patch
            OutT* d = sm + (w / P) * pdim + ph * PC + (w % P) * C + c;
            d[0] = OutT(v.x); d[C] = OutT(v.y); d[2 * C] = OutT(v.z); d[3 * C] = OutT(v.w);
        } else {
            const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; j++) sm[((w + j) / P) * pdim + ph * PC + ((w + j) % P) * C + c] = OutT(e[j]);
        }
    }
    __syncthreads();
    const int total = gw * pdim;
    constexpr int kVec = 16 / int(sizeof(OutT));
    const bool vec_ok = (total % kVec) == 0 && (reinterpret_cast<uintptr_t>(obase) & 15) == 0;
    if (vec_ok) {
        for (int o = threadIdx.x; o < total / kVec; o += blockDim.x)
            reinterpret_cast<uint4*>(obase)[o] = reinterpret_cast<const uint4*>(sm)[o];
    } else {
        for (int o = threadIdx.x; o < total; o += blockDim.x) obase[o] = sm[o];
    }
}

// scatter-add of the patch gradient back to NCHW is never needed (images need no grad).

// cls rows: x[b, 0, :] = q_ff( q_ff(cls) + pos_q[0, :] )   (vit.py:283-310, FP16_16 quantises
// the cat and the add; other formats pass q_ff = identity)
__global__ void cls_row_kernel(const float* __restrict__ cls, const float* __restrict__ pos_q,
                               float* __restrict__ x, int B, int n_tokens, int D, FloatFmt q_ff) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * D) return;
    const int b = i / D, d = i % D;
    const float v = fq_nearest(fq_nearest(cls[d], q_ff) + pos_q[d], q_ff);
    x[(int64_t(b) * n_tokens) * D + d] = v;
}

// token row: x[b, row, :] = q_ff(tok) for every image (the distillation token: no positional embedding)
__global__ void token_row_kernel(const float* __restrict__ tok, float* __restrict__ x, int B, int n_tokens, int D,
                                 int row, FloatFmt q_ff) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * D) return;
    const int b = i / D, d = i % D;
    x[(int64_t(b) * n_tokens + row) * D + d] = fq_nearest(tok[d], q_ff);
}

// out32 = in * s and / or out16 = fp16(in * s), s = *scale_dev or its reciprocal (a power of two: exact).
// The loss-scale style gradient scale lives in device memory, so no host synchronisation.
__global__ void __launch_bounds__(256)
scale_kernel(const float* __restrict__ in, const float* __restrict__ scale_dev, int invert, float* __restrict__ out32,
             __half* __restrict__ out16, int64_t n4, int* __restrict__ ovf) {
    const float s = invert ? 1.0f / __ldg(scale_dev) : __ldg(scale_dev);
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    // overflow sink: a non-finite result anywhere (the final un-scale of the parameter gradients: GradScaler's
    // inf / NaN test, element by element like its isfinite), or a value that does not fit the fp16 copy.  One test per
    // element, !(|v| < limit), is true for NaN as well; fp32 only, the limit is +inf, so FLT_MAX passes.
    const float limit = out16 != nullptr ? kHalfOverflow : __int_as_float(0x7f800000);
    bool bad = false;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 v = __ldcs(reinterpret_cast<const float4*>(in) + i);
        v.x *= s; v.y *= s; v.z *= s; v.w *= s;
        bad |= !(fabsf(v.x) < limit) | !(fabsf(v.y) < limit) | !(fabsf(v.z) < limit) | !(fabsf(v.w) < limit);
        if (out32 != nullptr) reinterpret_cast<float4*>(out32)[i] = v;
        if (out16 != nullptr) {
            __half2 lo = __floats2half2_rn(sat16(v.x), sat16(v.y)), hi = __floats2half2_rn(sat16(v.z), sat16(v.w));
            reinterpret_cast<uint2*>(out16)[i] = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        }
    }
    if (bad && ovf != nullptr) *ovf = 1;
}

// GradScaler bookkeeping on the device (torch.cuda.amp.GradScaler.update: backoff on inf, growth after a run of good
// steps), for the power-of-two gradient operand scale.  state = {found_inf, scale_target, good_steps}.
__global__ void overflow_update_kernel(const int* __restrict__ flag, const float* __restrict__ shared_slot,
                                       float* __restrict__ state, float backoff, float growth, float interval,
                                       float min_target, float max_target) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    bool found = *flag != 0;
    if (shared_slot != nullptr) found |= !(*shared_slot == 0.0f);          // NaN counts
    float target = state[1], good = state[2];
    if (found) { target = fmaxf(target * backoff, min_target); good = 0.f; }
    else if (++good >= interval) { target = fminf(target * growth, max_target); good = 0.f; }
    // found_inf is sticky (gradient accumulation runs several backwards per optimizer step): whoever consumes it clears it
    state[0] = (found || state[0] != 0.0f) ? 1.0f : 0.0f; state[1] = target; state[2] = good;
}

template <int NV>
static int launch_ln_fwd(const float* x, int64_t ld_x, const float* gamma, const float* beta, void* y,
                         int64_t ld_y, int y_dtype, float* mean, float* rstd, int rows, int D,
                         float eps, FloatFmt q_in, FloatFmt q_post, cudaStream_t st) {
    int grid = (rows + 2 * kLnWarps - 1) / (2 * kLnWarps);
    const int cap = kNumSMs * 4;
    if (grid > cap) grid = cap;
    if (y_dtype == MV_F16)
        ln_fwd_kernel<NV, __half><<<grid, kLnWarps * 32, 0, st>>>(x, ld_x, gamma, beta, (__half*)y, ld_y, mean, rstd, rows, D, eps, q_in, q_post);
    else
        ln_fwd_kernel<NV, float><<<grid, kLnWarps * 32, 0, st>>>(x, ld_x, gamma, beta, (float*)y, ld_y, mean, rstd, rows, D, eps, q_in, q_post);
    g_launches++;
    return check_cuda(cudaGetLastError(), "ln fwd launch");
}

// Every ln_bwd_kernel instantiation may take the shared memory of the widest row (D = 128 * kLnMaxVec); the attribute is
// set on its first launch.
template <auto kKernel>
static decltype(kKernel) ln_bwd_ready() {
    static const cudaError_t once = cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                         kLnWarps * 3 * 128 * kLnMaxVec * 4);
    (void)once;
    return kKernel;
}

template <int NV>
static int launch_ln_bwd(const mv_layernorm_bwd_args& a, cudaStream_t st) {
    int grid = (a.rows + kLnWarps - 1) / kLnWarps;
    const int cap = kNumSMs * 2;
    if (grid > cap) grid = cap;
    const size_t smem = size_t(kLnWarps) * 3 * a.D * sizeof(float);
    const FloatFmt q_in{a.q_in_exp, a.q_in_man}, q_grad{a.q_grad_exp, a.q_grad_man};
    const DropDev drop{a.drop_seed, a.drop_thr, a.drop_scale, a.drop_site};
    const SrDev sr{a.round_seed, a.round_offset};
    auto launch = [&](auto kernel, auto* dy) {
        kernel<<<grid, kLnWarps * 32, smem, st>>>(dy, a.ld_dy, a.x, a.ld_x, a.dres, a.ld_dres, a.gamma, a.mean, a.rstd, a.dx,
                                                  a.ld_dx, (__half*)a.dx_f16, a.ld_lp, a.dgamma, a.dbeta, a.dbias_prev, a.rows,
                                                  a.D, q_in, g_overflow, q_grad, drop, a.mask_dx, sr);
    };
    // kGQ: gradient quantiser; kDrop: dropout; kSR: the quantiser rounds stochastically (a round_seed without a
    // gradient format has no effect).  Only the plain kernel also takes fp32 dy.
    const bool gq = a.q_grad_exp != 0, dp = a.drop_seed != nullptr, sr_on = gq && a.round_seed != nullptr;
    if (a.dy_dtype == MV_F32) {
        launch(ln_bwd_ready<ln_bwd_kernel<NV, float>>(), (const float*)a.dy);
    } else {
        const auto kernel = sr_on ? (dp ? ln_bwd_ready<ln_bwd_kernel<NV, __half, true, true, true>>()
                                        : ln_bwd_ready<ln_bwd_kernel<NV, __half, true, false, true>>())
                          : dp    ? (gq ? ln_bwd_ready<ln_bwd_kernel<NV, __half, true, true>>()
                                        : ln_bwd_ready<ln_bwd_kernel<NV, __half, false, true>>())
                          : gq    ? ln_bwd_ready<ln_bwd_kernel<NV, __half, true>>()
                                  : ln_bwd_ready<ln_bwd_kernel<NV, __half>>();
        launch(kernel, (const __half*)a.dy);
    }
    g_launches++;
    return check_cuda(cudaGetLastError(), "ln bwd launch");
}

// mv_dropout: out = in * keep * scale over [rows, cols] with row pitches.  A thread takes eight consecutive elements of
// the flat (pitch-free) index, i.e. one Philox block; with cols, both pitches and both bases multiples of eight elements /
// 16 bytes it moves them as 16-byte vectors, otherwise element by element.
__device__ __forceinline__ float ld_elem(const float* p) { return *p; }
__device__ __forceinline__ float ld_elem(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ void st_elem(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_elem(__half* p, float v) { *p = __float2half_rn(sat16(v)); }
__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
    const float4 a = __ldcs(reinterpret_cast<const float4*>(p)), b = __ldcs(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld8(const __half* p, float (&v)[8]) {
    const uint4 u = __ldcs(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
        v[2 * j] = f.x; v[2 * j + 1] = f.y;
    }
}
__device__ __forceinline__ void st8(float* p, const float (&v)[8]) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void st8(__half* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack_h2_sat(v[0], v[1]), pack_h2_sat(v[2], v[3]), pack_h2_sat(v[4], v[5]),
                                              pack_h2_sat(v[6], v[7]));
}
template <typename InT, typename OutT>
__global__ void __launch_bounds__(256)
dropout_kernel(const InT* in, int64_t ld_in, OutT* out, int64_t ld_out, int rows, int cols, DropDev d, int vec,
               int* __restrict__ ovf) {
    const uint64_t seed = __ldg(reinterpret_cast<const unsigned long long*>(d.seed));
    const uint64_t n = uint64_t(rows) * uint64_t(cols), blocks = (n + 7) >> 3;
    float amax = 0.f;
    for (uint64_t g = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; g < blocks; g += uint64_t(gridDim.x) * blockDim.x) {
        const uint4 w = philox4x32_10(seed, g, uint64_t(uint32_t(d.site)));
        const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
        float v[8];
        if (vec) {
            const uint64_t r = (g * 8) / uint64_t(cols), c = (g * 8) % uint64_t(cols);
            ld8(in + r * ld_in + c, v);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t h = (j & 1) ? (ws[j >> 1] >> 16) : (ws[j >> 1] & 0xFFFFu);
                v[j] *= h >= d.thr ? d.scale : 0.f;
                amax = fmaxf(amax, fabsf(v[j]));
            }
            st8(out + r * ld_out + c, v);
        } else {
            for (int j = 0; j < 8; j++) {
                const uint64_t i = g * 8 + j;
                if (i >= n) break;
                const uint64_t r = i / uint64_t(cols), c = i % uint64_t(cols);
                const uint32_t h = (j & 1) ? (ws[j >> 1] >> 16) : (ws[j >> 1] & 0xFFFFu);
                const float x = ld_elem(in + r * ld_in + c) * (h >= d.thr ? d.scale : 0.f);
                amax = fmaxf(amax, fabsf(x));
                st_elem(out + r * ld_out + c, x);
            }
        }
    }
    if (sizeof(OutT) == 2) raise_overflow(ovf, amax);
}

// fp16 / fp32 [rows, cols] (row pitch ld) -> fp32 copy and / or fp32 transpose [cols, rows], 32x32 tiles
// through shared memory so both directions are coalesced.  Feeds the kind::tf32 GEMMs of the 32-bit
// formats (TF32 / FP32): wgrad there takes K-major operands, i.e. dY^T and X^T.
template <typename InT>
__global__ void widen_transpose_kernel(const InT* __restrict__ in, int64_t ld, int rows, int cols,
                                       float* __restrict__ out, float* __restrict__ out_t, int64_t ld_t,
                                       float mul) {
    __shared__ float tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int r = r0 + j, c = c0 + threadIdx.x;
        float v = 0.f;
        if (r < rows && c < cols) {
            v = float(in[int64_t(r) * ld + c]) * mul;
            if (out != nullptr) out[int64_t(r) * cols + c] = v;
        }
        tile[j][threadIdx.x] = v;
    }
    if (out_t == nullptr) return;
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int c = c0 + j, r = r0 + threadIdx.x;
        if (r < rows && c < cols) out_t[int64_t(c) * ld_t + r] = tile[threadIdx.x][j];
    }
}

// 3xTF32 operand preparation (q_format FP32): x = hi + lo with hi = the tf32 the tensor core would see
// (low 13 mantissa bits cleared) and lo = x - hi (exact in fp32).  A GEMM over the K-concatenated
// operands A' = [hi | lo | hi], B' = [hi | hi | lo] accumulates hi*hi + lo*hi + hi*lo in fp32: the
// product error drops from 2^-11 to ~2^-21 relative, using the unchanged kind::tf32 kernel.
__global__ void split_tf32_kernel(const float* __restrict__ in, int64_t ld, int rows, int cols,
                                  float* __restrict__ out, int mode) {
    const int64_t n = int64_t(rows) * cols;
    for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
        const int r = int(i / cols), c = int(i % cols);
        const float x = in[int64_t(r) * ld + c];
        const float hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
        const float lo = x - hi;
        float* o = out + int64_t(r) * 3 * cols + c;
        o[0] = hi;
        o[cols] = mode == 0 ? lo : hi;
        o[2 * cols] = mode == 0 ? hi : lo;
    }
}

}  // namespace mv

using namespace mv;

extern "C" int mv_layernorm_q_fwd(const float* x, int64_t ld_x, const float* gamma, const float* beta,
                                  void* y, int64_t ld_y, int y_dtype, float* mean, float* rstd, int rows,
                                  int D, float eps, int q_in_exp, int q_in_man, int q_post_exp,
                                  int q_post_man, void* stream) {
    MV_CHECK(rows >= 0 && D > 0 && D % 4 == 0 && D <= 128 * kLnMaxVec, "mv_layernorm_q_fwd: D=%d unsupported (multiple of 4, <= %d)", D, 128 * kLnMaxVec);
    MV_CHECK(ld_x % 4 == 0 && ld_y % 4 == 0, "mv_layernorm_q_fwd: row pitches must be multiples of 4 elements");
    MV_CHECK(y_dtype == MV_F16 || y_dtype == MV_F32, "mv_layernorm_q_fwd: bad output container");
    if (rows == 0) return 0;
    const FloatFmt qi{q_in_exp, q_in_man}, qp{q_post_exp, q_post_man};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int nv = (D / 4 + 31) / 32;
    switch (nv) {
        case 1: return launch_ln_fwd<1>(x, ld_x, gamma, beta, y, ld_y, y_dtype, mean, rstd, rows, D, eps, qi, qp, st);
        case 2: return launch_ln_fwd<2>(x, ld_x, gamma, beta, y, ld_y, y_dtype, mean, rstd, rows, D, eps, qi, qp, st);
        case 3: return launch_ln_fwd<3>(x, ld_x, gamma, beta, y, ld_y, y_dtype, mean, rstd, rows, D, eps, qi, qp, st);
        case 4: return launch_ln_fwd<4>(x, ld_x, gamma, beta, y, ld_y, y_dtype, mean, rstd, rows, D, eps, qi, qp, st);
        case 5: case 6: return launch_ln_fwd<6>(x, ld_x, gamma, beta, y, ld_y, y_dtype, mean, rstd, rows, D, eps, qi, qp, st);
        default: return launch_ln_fwd<8>(x, ld_x, gamma, beta, y, ld_y, y_dtype, mean, rstd, rows, D, eps, qi, qp, st);
    }
}

extern "C" int mv_layernorm_q_bwd(const mv_layernorm_bwd_args* args, void* stream) {
    MV_CHECK(args != nullptr, "mv_layernorm_q_bwd: null args");
    const mv_layernorm_bwd_args& a = *args;
    MV_CHECK(a.rows >= 0 && a.D > 0 && a.D % 4 == 0 && a.D <= 128 * kLnMaxVec, "mv_layernorm_q_bwd: D=%d unsupported", a.D);
    MV_CHECK(a.dy_dtype == MV_F16 || a.dy_dtype == MV_F32, "mv_layernorm_q_bwd: dy must be fp16 or fp32");
    MV_CHECK(a.ld_dy % 4 == 0 && a.ld_x % 4 == 0 && a.ld_dx % 4 == 0 && a.ld_dres % 4 == 0 && a.ld_lp % 4 == 0,
             "mv_layernorm_q_bwd: row pitches must be multiples of 4");
    MV_CHECK(a.q_grad_exp == 0 || (a.q_grad_exp >= 2 && a.q_grad_exp <= 8 && a.q_grad_man >= 1 && a.q_grad_man <= 22),
             "mv_layernorm_q_bwd: unsupported gradient format (%d, %d)", a.q_grad_exp, a.q_grad_man);
    MV_CHECK(a.drop_seed == nullptr || a.drop_thr <= 65536u, "mv_layernorm_q_bwd: dropout threshold %u above 65536", a.drop_thr);
    MV_CHECK((a.q_grad_exp == 0 && a.drop_seed == nullptr) || a.dy_dtype == MV_F16,
             "mv_layernorm_q_bwd: the gradient quantiser and dropout take fp16 dy");
    if (a.rows == 0) return 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch ((a.D / 4 + 31) / 32) {
        case 1: return launch_ln_bwd<1>(a, st);
        case 2: return launch_ln_bwd<2>(a, st);
        case 3: return launch_ln_bwd<3>(a, st);
        case 4: return launch_ln_bwd<4>(a, st);
        case 5: case 6: return launch_ln_bwd<6>(a, st);
        default: return launch_ln_bwd<8>(a, st);
    }
}

extern "C" int mv_dropout(const void* in, int in_dtype, int64_t ld_in, void* out, int out_dtype, int64_t ld_out, int rows,
                          int cols, const uint64_t* seed_dev, int site, uint32_t thr, float scale, void* stream) {
    MV_CHECK(in && out && seed_dev, "mv_dropout: null pointer");
    MV_CHECK(rows >= 0 && cols > 0 && ld_in >= cols && ld_out >= cols, "mv_dropout: bad shape %d x %d (pitches %lld, %lld)", rows, cols,
             (long long)ld_in, (long long)ld_out);
    MV_CHECK((in_dtype == MV_F32 || in_dtype == MV_F16) && (out_dtype == MV_F32 || out_dtype == MV_F16), "mv_dropout: fp32 or fp16 only");
    MV_CHECK(thr <= 65536u, "mv_dropout: threshold %u above 65536", thr);
    MV_CHECK(in != out || (in_dtype == out_dtype && ld_in == ld_out), "mv_dropout: in place needs one dtype and one pitch");
    if (rows == 0) return 0;
    const DropDev d{seed_dev, thr, scale, site};
    const uint64_t blocks8 = (uint64_t(rows) * uint64_t(cols) + 7) / 8;
    const int vec = cols % 8 == 0 && ld_in % 8 == 0 && ld_out % 8 == 0 && reinterpret_cast<uintptr_t>(in) % 16 == 0 &&
                    reinterpret_cast<uintptr_t>(out) % 16 == 0;
    int64_t grid = int64_t((blocks8 + 255) / 256);
    if (grid > kNumSMs * 8) grid = kNumSMs * 8;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (in_dtype == MV_F32 && out_dtype == MV_F32)
        dropout_kernel<float, float><<<int(grid), 256, 0, st>>>((const float*)in, ld_in, (float*)out, ld_out, rows, cols, d, vec, g_overflow);
    else if (in_dtype == MV_F32)
        dropout_kernel<float, __half><<<int(grid), 256, 0, st>>>((const float*)in, ld_in, (__half*)out, ld_out, rows, cols, d, vec, g_overflow);
    else if (out_dtype == MV_F32)
        dropout_kernel<__half, float><<<int(grid), 256, 0, st>>>((const __half*)in, ld_in, (float*)out, ld_out, rows, cols, d, vec, g_overflow);
    else
        dropout_kernel<__half, __half><<<int(grid), 256, 0, st>>>((const __half*)in, ld_in, (__half*)out, ld_out, rows, cols, d, vec, g_overflow);
    g_launches++;
    return check_cuda(cudaGetLastError(), "dropout launch");
}

extern "C" int mv_colsum(const void* in, int in_dtype, int64_t ld, int rows, int cols, float* out, void* stream) {
    MV_CHECK(in_dtype == MV_F16 || in_dtype == MV_F32, "mv_colsum: dtype must be f16 or f32");
    const int vec = in_dtype == MV_F16 ? 8 : 4;
    MV_CHECK(rows >= 0 && cols > 0 && cols % vec == 0 && ld % vec == 0 && reinterpret_cast<uintptr_t>(in) % 16 == 0,
             "mv_colsum: cols/ld must be multiples of %d and the base 16-byte aligned", vec);
    if (rows == 0) return 0;
    const int gx = (cols + 32 * vec - 1) / (32 * vec);
    int gy = (kNumSMs * 4 + gx - 1) / gx;
    const int max_gy = (rows + 31) / 32;
    if (gy > max_gy) gy = max_gy;
    if (gy < 1) gy = 1;
    dim3 grid(gx, gy);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (in_dtype == MV_F16) colsum_kernel<__half><<<grid, 256, 0, st>>>((const __half*)in, ld, rows, cols, out);
    else colsum_kernel<float><<<grid, 256, 0, st>>>((const float*)in, ld, rows, cols, out);
    g_launches++;
    return check_cuda(cudaGetLastError(), "colsum launch");
}

template <bool kMix>
static int patchify_launch(const char* fn, const float* img, const mv_mix_rec* recs, void* out, int out_dtype, int B,
                           int C, int H, int W, int P, int q_exp, int q_man, int cls_slot, void* stream) {
    MV_CHECK(B > 0 && C > 0 && P > 0 && H % P == 0 && W % P == 0, "%s: image dims must be divisible by the patch size", fn);
    MV_CHECK(cls_slot >= 0 && cls_slot <= 2, "%s: cls_slot must be 0, 1 or 2", fn);
    const FloatFmt q{q_exp, q_man};
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MV_CHECK(W % 4 == 0 && (reinterpret_cast<uintptr_t>(img) & 15) == 0, "%s: image rows must be 16-byte aligned (W %% 4 == 0)", fn);
    const int grid = B * (H / P);
    const size_t smem = size_t(C) * P * W * (out_dtype == MV_F16 ? 2 : 4);
    MV_CHECK(smem <= 200 * 1024, "%s: C * P * W too large for the shared-memory staging buffer", fn);
    if (out_dtype == MV_F16) {
        MV_CUDA(cudaFuncSetAttribute(patchify_kernel<__half, kMix>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        patchify_kernel<__half, kMix><<<grid, 256, smem, st>>>(img, (__half*)out, B, C, H, W, P, q, cls_slot, recs);
    } else if (out_dtype == MV_F32) {
        MV_CUDA(cudaFuncSetAttribute(patchify_kernel<float, kMix>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        patchify_kernel<float, kMix><<<grid, 256, smem, st>>>(img, (float*)out, B, C, H, W, P, q, cls_slot, recs);
    } else MV_CHECK(false, "%s: bad container", fn);
    g_launches++;
    return check_cuda(cudaGetLastError(), "patchify launch");
}

extern "C" int mv_patchify_q(const float* img, void* out, int out_dtype, int B, int C, int H, int W, int P,
                             int q_exp, int q_man, int cls_slot, void* stream) {
    return patchify_launch<false>("mv_patchify_q", img, nullptr, out, out_dtype, B, C, H, W, P, q_exp, q_man, cls_slot,
                                  stream);
}

extern "C" int mv_patchify_mix_q(const float* img, const mv_mix_rec* recs_dev, void* out, int out_dtype, int B, int C,
                                 int H, int W, int P, int q_exp, int q_man, int cls_slot, void* stream) {
    MV_CHECK(recs_dev != nullptr, "mv_patchify_mix_q: null records");
    MV_CHECK(B > 0 && B % 2 == 0, "mv_patchify_mix_q: the batch must be even (got B=%d)", B);
    return patchify_launch<true>("mv_patchify_mix_q", img, recs_dev, out, out_dtype, B, C, H, W, P, q_exp, q_man,
                                 cls_slot, stream);
}

extern "C" int mv_cls_rows(const float* cls, const float* pos_q, float* x, int B, int n_tokens, int D,
                           int q_exp, int q_man, void* stream) {
    const FloatFmt q{q_exp, q_man};
    const int n = B * D;
    cls_row_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(cls, pos_q, x, B, n_tokens, D, q);
    g_launches++;
    return check_cuda(cudaGetLastError(), "cls rows launch");
}

extern "C" int mv_token_row(const float* tok, float* x, int B, int n_tokens, int D, int row, int q_exp, int q_man,
                            void* stream) {
    MV_CHECK(tok && x && B > 0 && D > 0 && row >= 0 && row < n_tokens, "mv_token_row: bad arguments");
    const FloatFmt q{q_exp, q_man};
    const int n = B * D;
    token_row_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(tok, x, B, n_tokens, D, row, q);
    g_launches++;
    return check_cuda(cudaGetLastError(), "token row launch");
}

extern "C" int mv_scale_f32(const float* in, const float* scale_dev, int invert, float* out_f32, void* out_f16, int64_t n,
                            void* stream) {
    MV_CHECK(in && scale_dev && (out_f32 || out_f16), "mv_scale_f32: null pointer");
    MV_CHECK(n % 4 == 0, "mv_scale_f32: n must be a multiple of 4");
    if (n == 0) return 0;
    const int64_t n4 = n / 4;
    int64_t blocks = (n4 + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    scale_kernel<<<int(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, scale_dev, invert, out_f32,
                                                                           reinterpret_cast<__half*>(out_f16), n4, g_overflow);
    g_launches++;
    return check_cuda(cudaGetLastError(), "scale launch");
}

extern "C" int mv_overflow_update(const int* flag_dev, const float* shared_slot_dev, float* state_dev, float backoff,
                                  float growth, int growth_interval, float min_target, float max_target, void* stream) {
    MV_CHECK(flag_dev && state_dev, "mv_overflow_update: null pointer");
    overflow_update_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(flag_dev, shared_slot_dev, state_dev, backoff, growth,
                                                                          float(growth_interval), min_target, max_target);
    g_launches++;
    return check_cuda(cudaGetLastError(), "overflow update launch");
}

extern "C" int mv_widen_transpose(const void* in, int in_dtype, int64_t ld, int rows, int cols, float* out,
                                  float* out_t, int64_t ld_t, float mul, void* stream) {
    MV_CHECK(in && rows > 0 && cols > 0 && (out || out_t) && (!out_t || ld_t >= rows), "mv_widen_transpose: bad arguments");
    MV_CHECK((rows + 31) / 32 <= 65535, "mv_widen_transpose: too many rows");
    dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (in_dtype == MV_F16) widen_transpose_kernel<__half><<<grid, block, 0, st>>>((const __half*)in, ld, rows, cols, out, out_t, ld_t, mul);
    else if (in_dtype == MV_F32) widen_transpose_kernel<float><<<grid, block, 0, st>>>((const float*)in, ld, rows, cols, out, out_t, ld_t, mul);
    else MV_CHECK(false, "mv_widen_transpose: bad dtype");
    g_launches++;
    return check_cuda(cudaGetLastError(), "widen transpose launch");
}

extern "C" int mv_split_tf32(const float* in, int64_t ld, int rows, int cols, float* out, int mode, void* stream) {
    MV_CHECK(in && out && rows > 0 && cols > 0 && (mode == 0 || mode == 1), "mv_split_tf32: bad arguments");
    const int64_t n = int64_t(rows) * cols;
    int64_t blocks = (n + 255) / 256;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    split_tf32_kernel<<<int(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, ld, rows, cols, out, mode);
    g_launches++;
    return check_cuda(cudaGetLastError(), "split tf32 launch");
}
