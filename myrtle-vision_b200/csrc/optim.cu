// optim.cu — multi-tensor AdamW fused with the next step's weight fake-quantisation.
//
// SURVEY.md §8(f).1: the step on the far side of backward (reference classification/train.py:274-277,
// timm AdamW).  One launch updates every parameter of the model; for the Linear weights the same thread
// that wrote the new fp32 weight also emits the tensor-core operands of the NEXT forward / backward —
// q(W) [out,in] and q(W)^T [in,out] in the fp16 (or fp32 for the 32-bit formats) container — so the
// per-step weight_fake_quant pass (torch.nn.qat.Linear re-quantises W every forward) never re-reads
// the weights from HBM.  HBM-bound: 28 B per parameter (p, g, m, v read; p, m, v written) + 4 B per
// Linear weight for the two fp16 operand copies.
//
// Work is cut into chunks of 1024 elements — a run of 1024 consecutive elements of a plain tensor,
// or one 32x32 tile of a weight matrix (so the transposed operand is written coalesced through
// shared memory).  Hyper-parameters that change between steps live in device memory: a captured
// CUDA graph replays the same launch with new values.
#include <type_traits>

#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {
extern int64_t g_launches;

template <typename T> __device__ __forceinline__ T opt_cvt(float v);
template <> __device__ __forceinline__ float opt_cvt<float>(float v) { return v; }
template <> __device__ __forceinline__ __half opt_cvt<__half>(float v) { return __float2half_rn(v); }

struct AdamHyper { float lr_mul, beta1, beta2, eps, bc1, bc2_rsqrt, inv_scale; bool skip; };

__device__ __forceinline__ float adamw_elem(float p, float g, float& m, float& v, float lr, float wd,
                                            const AdamHyper& h) {
    g *= h.inv_scale;
    m = h.beta1 * m + (1.f - h.beta1) * g;
    v = h.beta2 * v + (1.f - h.beta2) * g * g;
    const float denom = sqrtf(v) * h.bc2_rsqrt + h.eps;
    p *= 1.f - lr * wd;
    return p - (lr / h.bc1) * (m / denom);
}

// hyper (device): [0] beta1 [1] beta2 [2] eps [3] step (float, >= 1) [4] inv_scale (gradient un-scale)
// [5] found_inf (non-zero: skip the update, GradScaler semantics; operands are still emitted)
__global__ void __launch_bounds__(256)
adamw_kernel(const mv_adamw_tensor* __restrict__ tensors, int n_tensors, int total_chunks,
             const float* __restrict__ hyper) {
    __shared__ float tile[32][33];
    AdamHyper h;
    h.beta1 = hyper[0]; h.beta2 = hyper[1]; h.eps = hyper[2];
    const float step = hyper[3];
    h.bc1 = 1.f - powf(h.beta1, step);
    h.bc2_rsqrt = rsqrtf(1.f - powf(h.beta2, step));
    h.inv_scale = hyper[4];
    h.skip = hyper[5] != 0.f;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    for (int chunk = blockIdx.x; chunk < total_chunks; chunk += gridDim.x) {
        // owner tensor: last one whose chunk0 <= chunk
        int lo = 0, hi = n_tensors - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (tensors[mid].chunk0 <= chunk) lo = mid; else hi = mid - 1;
        }
        const mv_adamw_tensor t = tensors[lo];
        const int local = chunk - t.chunk0;
        if (t.wq == nullptr) {
            const int64_t base = int64_t(local) * 1024;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int64_t i = base + j * 256 + tid;
                if (i < t.n && !h.skip) {
                    float m = t.exp_avg[i], v = t.exp_avg_sq[i];
                    t.param[i] = adamw_elem(t.param[i], t.grad[i], m, v, t.lr, t.weight_decay, h);
                    t.exp_avg[i] = m; t.exp_avg_sq[i] = v;
                }
            }
        } else {
            const int tiles_x = (t.cols + 31) >> 5;
            const int r0 = (local / tiles_x) * 32, c0 = (local % tiles_x) * 32;
            __syncthreads();                                   // previous tile fully consumed
            for (int j = threadIdx.y; j < 32; j += blockDim.y) {
                const int r = r0 + j, c = c0 + threadIdx.x;
                float p = 0.f;
                if (r < t.rows && c < t.cols) {
                    const int64_t i = int64_t(r) * t.cols + c;
                    p = t.param[i];
                    if (!h.skip) {
                        float m = t.exp_avg[i], v = t.exp_avg_sq[i];
                        p = adamw_elem(p, t.grad[i], m, v, t.lr, t.weight_decay, h);
                        t.param[i] = p; t.exp_avg[i] = m; t.exp_avg_sq[i] = v;
                    }
                    if (t.q_exp > 0) p = float_quantize_elem<false>(p, 0u, t.q_exp, t.q_man);
                }
                tile[j][threadIdx.x] = p;
            }
            __syncthreads();
            // q(W) row-major and q(W)^T through the tile, both coalesced (inline: keeps `tile` in the shared space)
            auto emit = [&](auto* wq, auto* wq_t) {
                using OutT = typename std::remove_pointer<decltype(wq)>::type;
                for (int j = threadIdx.y; j < 32; j += blockDim.y) {
                    const int r = r0 + j, c = c0 + threadIdx.x;
                    if (r < t.rows && c < t.cols) wq[int64_t(r) * t.cols + c] = opt_cvt<OutT>(tile[j][threadIdx.x]);
                }
                if (wq_t == nullptr) return;
                for (int j = threadIdx.y; j < 32; j += blockDim.y) {
                    const int c = c0 + j, r = r0 + threadIdx.x;
                    if (r < t.rows && c < t.cols) wq_t[int64_t(c) * t.rows + r] = opt_cvt<OutT>(tile[threadIdx.x][j]);
                }
            };
            if (t.wq_dtype == MV_F16) emit(static_cast<__half*>(t.wq), static_cast<__half*>(t.wq_t));
            else emit(static_cast<float*>(t.wq), static_cast<float*>(t.wq_t));
        }
    }
}

// ---- low-precision optimizer (include/mv_b200.h "low-precision optimizer"): QPyTorch's OptimLP quantisers fused into the
// same pass.  One site's quantiser, resolved on the host; every switch is uniform over the grid.
struct LpSite {
    int kind;                     // MV_LPQ_*
    bool stoch, s16;              // stochastic; 16-bit stream (float, man >= 7)
    FloatFmt f;
    float scale_up, scale_down, t_min, t_max;
    bool clamp;
};
struct LpSpec {
    LpSite site[5];               // 0 grad, 1 exp_avg, 2 exp_avg_sq, 3 acc, 4 weight
    float grad_scaling;
    uint64_t seed;
};

__device__ __forceinline__ float lp_round(float x, uint32_t r, const LpSite& q) {
    if (q.kind == MV_LPQ_FLOAT)
        return q.stoch ? fq_stoch_elem(x, r, q.f) : float_quantize_elem<false>(x, 0u, q.f.exp_bits, q.f.man_bits);
    if (q.kind == MV_LPQ_FIXED)
        return fixed_quantize_elem(x, q.stoch ? bits_to_uniform(r) : 0.5f, q.scale_up, q.scale_down, q.t_min, q.t_max,
                                   q.clamp);
    return x;
}
__device__ __forceinline__ uint32_t lp_word(uint4 v, int j) { return j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w; }
__device__ __forceinline__ bool lp_s16(const LpSite& q) { return q.kind != MV_LPQ_NONE && q.stoch && q.s16; }
__device__ __forceinline__ bool lp_s32(const LpSite& q) { return q.kind != MV_LPQ_NONE && q.stoch && !q.s16; }

// Random bits of the four elements i0 .. i0+3 at every stochastic site (uniform control flow: every lane of the warp
// runs this, in or out of range).  vec: i0 % 4 == 0 and lanes 2k / 2k+1 hold the two halves of one 16-bit block (odd =
// i0 & 4).  Then a 32-bit site costs one Philox call per lane, and two 16-bit sites share one call per lane: the even lane
// computes the block at the first site, the odd lane at the second, and each hands the other the half it needs (eight
// elements per call).  Otherwise (Linear weights with cols % 8 != 0) each element computes its own block.
__device__ __forceinline__ uint4 lp_bits_one(const LpSpec& sp, int s, uint64_t off, int64_t i0, bool vec) {
    const LpSite& q = sp.site[s];
    if (!lp_s16(q) && !lp_s32(q)) return make_uint4(0, 0, 0, 0);
    if (vec) return sr_bits4(sp.seed, off | uint64_t(s), uint64_t(i0), q.s16);
    return make_uint4(sr_bits1(sp.seed, off | uint64_t(s), uint64_t(i0), q.s16),
                      sr_bits1(sp.seed, off | uint64_t(s), uint64_t(i0 + 1), q.s16),
                      sr_bits1(sp.seed, off | uint64_t(s), uint64_t(i0 + 2), q.s16),
                      sr_bits1(sp.seed, off | uint64_t(s), uint64_t(i0 + 3), q.s16));
}
__device__ __forceinline__ void lp_bits_pair(const LpSpec& sp, int a, uint64_t off, int64_t i0, bool vec, uint4& ra,
                                             uint4& rb) {
    if (vec && lp_s16(sp.site[a]) && lp_s16(sp.site[a + 1])) {
        const bool odd = (i0 & 4) != 0;
        const uint4 w = sr_pair16(sp.seed, off | uint64_t(odd ? a + 1 : a), uint64_t(i0) >> 3, odd);
        ra = sr_halves(make_uint2(w.x, w.y));
        rb = sr_halves(make_uint2(w.z, w.w));
        return;
    }
    ra = lp_bits_one(sp, a, off, i0, vec);
    rb = lp_bits_one(sp, a + 1, off, i0, vec);
}

// adamw_elem with each rounding spelled out as adamw_kernel's SASS performs it (fused multiply-adds for the moments, the decay
// factor and the final step).  Left to the compiler's contraction, the two kernels fuse different products (the surroundings
// differ) and the results differ in the last bit.
__device__ __forceinline__ float adamw_elem_rn(float p, float g, float& m, float& v, float lr, float wd,
                                               const AdamHyper& h) {
    m = __fmaf_rn(h.beta1, m, __fmul_rn(1.f - h.beta1, g));
    v = __fmaf_rn(h.beta2, v, __fmul_rn(g, __fmul_rn(1.f - h.beta2, g)));
    const float denom = __fmaf_rn(h.bc2_rsqrt, sqrtf(v), h.eps);
    return __fmaf_rn(-(lr / h.bc1), m / denom, __fmul_rn(__fmaf_rn(-lr, wd, 1.f), p));
}

// Steps 1-5 on the elements i0 .. i0+3 (the first nv valid); pv receives the final parameter values (the current ones
// when the step is skipped), for the operand tile.
__device__ __forceinline__ void lp_update4(const mv_adamw_tensor& t, const mv_adamw_lp_tensor& x, const LpSpec& sp,
                                           const AdamHyper& h, float inv_scale, uint64_t off, int64_t i0, int nv,
                                           bool vec, float pv[4]) {
    if (h.skip) {
#pragma unroll
        for (int j = 0; j < 4; j++) pv[j] = j < nv ? t.param[i0 + j] : 0.f;
        return;
    }
    uint4 r[5];
    lp_bits_pair(sp, 0, off, i0, vec, r[0], r[1]);
    lp_bits_pair(sp, 2, off, i0, vec, r[2], r[3]);
    r[4] = lp_bits_one(sp, 4, off, i0, vec);
#pragma unroll
    for (int j = 0; j < 4; j++) {
        pv[j] = 0.f;
        if (j >= nv) continue;
        const int64_t i = i0 + j;
        const float g = lp_round(__fmul_rn(__fmul_rn(t.grad[i], inv_scale), sp.grad_scaling), lp_word(r[0], j), sp.site[0]);
        if (x.grad_out != nullptr) x.grad_out[i] = g;
        float m = t.exp_avg[i], v = t.exp_avg_sq[i];
        float w = adamw_elem_rn(x.acc != nullptr ? x.acc[i] : t.param[i], g, m, v, t.lr, t.weight_decay, h);
        t.exp_avg[i] = lp_round(m, lp_word(r[1], j), sp.site[1]);
        t.exp_avg_sq[i] = lp_round(v, lp_word(r[2], j), sp.site[2]);
        w = lp_round(w, lp_word(r[3], j), sp.site[3]);
        if (x.acc != nullptr) x.acc[i] = w;
        pv[j] = lp_round(w, lp_word(r[4], j), sp.site[4]);
        t.param[i] = pv[j];
    }
}

// adamw_kernel's chunks and hyper-parameters; each thread owns four consecutive elements of a chunk (a 1024-element
// run, or one row quarter of a 32x32 weight tile) so that the random bits of a Philox block serve whole lanes.
__global__ void __launch_bounds__(256)
adamw_lp_kernel(const mv_adamw_tensor* __restrict__ tensors, const mv_adamw_lp_tensor* __restrict__ lp, int n_tensors,
                int total_chunks, const float* __restrict__ hyper, const LpSpec sp) {
    __shared__ float tile[32][33];
    AdamHyper h;
    h.beta1 = hyper[0]; h.beta2 = hyper[1]; h.eps = hyper[2];
    const float step = hyper[3];
    h.bc1 = 1.f - powf(h.beta1, step);
    h.bc2_rsqrt = rsqrtf(1.f - powf(h.beta2, step));
    const float inv_scale = hyper[4];
    h.skip = hyper[5] != 0.f;
    const uint64_t step_hi = uint64_t(step) << 32;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    for (int chunk = blockIdx.x; chunk < total_chunks; chunk += gridDim.x) {
        int lo = 0, hi = n_tensors - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (tensors[mid].chunk0 <= chunk) lo = mid; else hi = mid - 1;
        }
        const mv_adamw_tensor t = tensors[lo];
        const mv_adamw_lp_tensor x = lp[lo];
        const uint64_t off = step_hi | (uint64_t(x.index) << 3);
        const int local = chunk - t.chunk0;
        float pv[4];
        if (t.wq == nullptr) {
            const int64_t i0 = int64_t(local) * 1024 + 4 * tid;
            const int64_t left = t.n - i0;
            lp_update4(t, x, sp, h, inv_scale, off, i0, left < 0 ? 0 : (left > 4 ? 4 : int(left)), true, pv);
        } else {
            const int tiles_x = (t.cols + 31) >> 5;
            const int r0 = (local / tiles_x) * 32, c0 = (local % tiles_x) * 32;
            const int tr = tid >> 3, tc = 4 * (tid & 7);
            const int r = r0 + tr, c = c0 + tc;
            const int left = t.cols - c;
            const int nv = r < t.rows ? (left < 0 ? 0 : (left > 4 ? 4 : left)) : 0;
            __syncthreads();                                   // previous tile fully consumed
            lp_update4(t, x, sp, h, inv_scale, off, int64_t(r) * t.cols + c, nv, (t.cols & 7) == 0, pv);
#pragma unroll
            for (int j = 0; j < 4; j++)
                tile[tr][tc + j] = (j < nv && t.q_exp > 0) ? float_quantize_elem<false>(pv[j], 0u, t.q_exp, t.q_man) : pv[j];
            __syncthreads();
            auto emit = [&](auto* wq, auto* wq_t) {
                using OutT = typename std::remove_pointer<decltype(wq)>::type;
                for (int j = threadIdx.y; j < 32; j += blockDim.y) {
                    const int rr = r0 + j, cc = c0 + threadIdx.x;
                    if (rr < t.rows && cc < t.cols) wq[int64_t(rr) * t.cols + cc] = opt_cvt<OutT>(tile[j][threadIdx.x]);
                }
                if (wq_t == nullptr) return;
                for (int j = threadIdx.y; j < 32; j += blockDim.y) {
                    const int cc = c0 + j, rr = r0 + threadIdx.x;
                    if (rr < t.rows && cc < t.cols) wq_t[int64_t(cc) * t.rows + rr] = opt_cvt<OutT>(tile[threadIdx.x][j]);
                }
            };
            if (t.wq_dtype == MV_F16) emit(static_cast<__half*>(t.wq), static_cast<__half*>(t.wq_t));
            else emit(static_cast<float*>(t.wq), static_cast<float*>(t.wq_t));
        }
    }
}

}  // namespace mv

using namespace mv;

static int lp_site(const mv_lp_quant& q, const char* name, LpSite& s) {
    s = LpSite{};
    MV_CHECK(q.kind == MV_LPQ_NONE || q.kind == MV_LPQ_FLOAT || q.kind == MV_LPQ_FIXED,
             "mv_adamw_lp_step: %s: unknown quantiser kind %d", name, q.kind);
    MV_CHECK(q.rounding == MV_ROUND_NEAREST || q.rounding == MV_ROUND_STOCHASTIC,
             "mv_adamw_lp_step: %s: unknown rounding %d", name, q.rounding);
    s.kind = q.kind;
    s.stoch = q.rounding == MV_ROUND_STOCHASTIC;
    if (q.kind == MV_LPQ_FLOAT) {
        MV_CHECK(q.exp_bits >= 1 && q.exp_bits <= 8, "mv_adamw_lp_step: %s: exp_bits %d not in [1,8]", name, q.exp_bits);
        MV_CHECK(q.man_bits >= 1 && q.man_bits <= 22, "mv_adamw_lp_step: %s: man_bits %d not in [1,22]", name, q.man_bits);
        s.f = FloatFmt{q.exp_bits, q.man_bits};
        s.s16 = q.man_bits >= 7;
    } else if (q.kind == MV_LPQ_FIXED) {
        // the parameters of mv_fixed_point_quantize
        MV_CHECK(q.wl >= 1 && q.wl <= 32 && q.fl >= -100 && q.fl <= 100, "mv_adamw_lp_step: %s: bad wl/fl %d/%d", name,
                 q.wl, q.fl);
        s.scale_up = ldexpf(1.0f, q.fl);
        s.scale_down = ldexpf(1.0f, -q.fl);
        s.t_min = -ldexpf(1.0f, q.wl - q.fl - 1);
        s.t_max = -s.t_min - ldexpf(1.0f, -q.fl);
        if (q.symmetric) s.t_min = s.t_min + ldexpf(1.0f, -q.fl);
        s.clamp = q.clamp != 0;
    }
    return 0;
}

extern "C" int mv_adamw_lp_step(const mv_adamw_tensor* tensors_dev, const mv_adamw_lp_tensor* lp_dev, int n_tensors,
                                int total_chunks, const float* hyper_dev, const mv_optim_lp* spec, void* stream) {
    MV_CHECK(tensors_dev && lp_dev && hyper_dev && spec && n_tensors > 0 && total_chunks > 0,
             "mv_adamw_lp_step: bad arguments");
    LpSpec sp;
    const mv_lp_quant* q[5] = {&spec->grad, &spec->exp_avg, &spec->exp_avg_sq, &spec->acc, &spec->weight};
    const char* names[5] = {"grad", "exp_avg", "exp_avg_sq", "acc", "weight"};
    for (int s = 0; s < 5; s++)
        if (lp_site(*q[s], names[s], sp.site[s]) != 0) return 1;
    sp.grad_scaling = spec->grad_scaling;
    sp.seed = spec->seed;
    const int grid = total_chunks < kNumSMs * 8 ? total_chunks : kNumSMs * 8;
    adamw_lp_kernel<<<grid, dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(tensors_dev, lp_dev, n_tensors,
                                                                                   total_chunks, hyper_dev, sp);
    g_launches++;
    return check_cuda(cudaGetLastError(), "adamw_lp launch");
}

extern "C" int mv_adamw_step(const mv_adamw_tensor* tensors_dev, int n_tensors, int total_chunks,
                             const float* hyper_dev, void* stream) {
    MV_CHECK(tensors_dev && hyper_dev && n_tensors > 0 && total_chunks > 0, "mv_adamw_step: bad arguments");
    const int grid = total_chunks < kNumSMs * 8 ? total_chunks : kNumSMs * 8;
    adamw_kernel<<<grid, dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(tensors_dev, n_tensors,
                                                                                total_chunks, hyper_dev);
    g_launches++;
    return check_cuda(cudaGetLastError(), "adamw launch");
}
