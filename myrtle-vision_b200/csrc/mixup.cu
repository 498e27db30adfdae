// mixup.cu — Mixup / CutMix records drawn on the device, and the soft-target cross-entropy of the mixed batch
// (timm 0.5.4's Mixup, mixup_target and SoftTargetCrossEntropy; include/mv_b200.h "Mixup / CutMix", DESIGN.md
// section 7).  The pixels are mixed inside the patch gather (patchify_kernel<., true> in norm.cu).
//
// mix_draw_kernel: one thread per image.  A thread recomputes its unit's draw from the counter-based mix stream, so
// the images of one unit get identical records without any communication.
// mix_ce_rows_kernel: one CTA per row, as distill.cu: the maximum, then the exp sum with the maximum's exact terms kept
// apart (log Z = log1p(Z - 1)), then the gradient row with 1 - p formed without cancelling; the batch sum is distill.cu's
// fixed-order reduction, so the loss is deterministic.
#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {
extern int64_t g_launches;
int row_mean_launch(const float* row_loss, int B, float* loss, cudaStream_t st);      // distill.cu

constexpr int kGammaTries = 16;                 // Marsaglia-Tsang attempts per Gamma draw
constexpr uint32_t kGammaSpan = kGammaTries + 1;  // draw indices per Gamma draw: the boost uniform, then the attempts

__device__ __forceinline__ uint4 mix_bits(uint64_t seed, uint32_t unit, uint32_t draw, uint32_t rank) {
    // counter = {unit, draw, rank, tag}: philox4x32_10's counter words are {lo(ctr), hi(ctr), lo(offset), hi(offset)}
    return philox4x32_10(seed, (uint64_t(draw) << 32) | unit, (uint64_t(MV_MIX_TAG) << 32) | rank);
}

__device__ __forceinline__ double unit_open(uint32_t w) { return (double(w) + 0.5) * 0x1p-32; }     // (0, 1)

// Gamma(alpha) by Marsaglia-Tsang in fp64; alpha < 1 as Gamma(alpha + 1) U^(1 / alpha)
__device__ double gamma_draw(uint64_t seed, uint32_t unit, uint32_t rank, int g, double alpha) {
    const uint32_t base = 1 + kGammaSpan * uint32_t(g);
    double a = alpha, boost = 1.0;
    if (alpha < 1.0) {
        boost = pow(unit_open(mix_bits(seed, unit, base, rank).x), 1.0 / alpha);
        a = alpha + 1.0;
    }
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (int k = 0; k < kGammaTries; k++) {
        const uint4 w = mix_bits(seed, unit, base + 1 + uint32_t(k), rank);
        const double x = sqrt(-2.0 * log(unit_open(w.x))) * cospi(2.0 * unit_open(w.y));
        double v = 1.0 + c * x;
        if (v <= 0.0) continue;
        v = v * v * v;
        if (log(unit_open(w.z)) < 0.5 * x * x + d - d * v + d * log(v)) return d * v * boost;
    }
    return d * boost;           // 16 rejections in a row: below 1e-20 for every alpha
}

__global__ void __launch_bounds__(128)
mix_draw_kernel(const int64_t* __restrict__ seed_dev, int rank, int B, int H, int W, mv_mix_spec spec,
                mv_mix_rec* __restrict__ recs) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const uint32_t unit = spec.mode == MV_MIX_BATCH ? 0u : spec.mode == MV_MIX_PAIR ? uint32_t(min(b, B - 1 - b))
                                                                                    : uint32_t(b);
    const uint64_t seed = uint64_t(*seed_dev);
    const uint32_t rk = uint32_t(rank);
    const uint4 w0 = mix_bits(seed, unit, 0, rk);
    mv_mix_rec r{1.f, 1.f, 0.f, 0, 0, 0, 0, 0};
    if (unit_open(w0.x) < double(spec.prob)) {
        const bool cut = spec.mixup_alpha > 0.f && spec.cutmix_alpha > 0.f ? unit_open(w0.y) < double(spec.switch_prob)
                                                                           : spec.cutmix_alpha > 0.f;
        const double alpha = cut ? spec.cutmix_alpha : spec.mixup_alpha;
        const double x = gamma_draw(seed, unit, rk, 0, alpha), y = gamma_draw(seed, unit, rk, 1, alpha);
        const double lam = x + y > 0.0 ? x / (x + y) : 0.5;
        if (cut) {
            const double rat = sqrt(1.0 - lam);
            const int ch = int(H * rat), cw = int(W * rat);
            const int cy = min(int(unit_open(w0.z) * H), H - 1), cx = min(int(unit_open(w0.w) * W), W - 1);
            r.y0 = min(max(cy - ch / 2, 0), H); r.y1 = min(max(cy + ch / 2, 0), H);
            r.x0 = min(max(cx - cw / 2, 0), W); r.x1 = min(max(cx + cw / 2, 0), W);
            r.cutmix = 1;
            r.lam = float(1.0 - double(r.y1 - r.y0) * double(r.x1 - r.x0) / (double(H) * double(W)));
        } else {
            r.lam = r.w_self = float(lam);
            r.w_other = float(1.0 - lam);
        }
    }
    recs[b] = r;
}

constexpr int kMcThreads = 256;
constexpr int kMcWarps = kMcThreads / 32;

template <int K>
__device__ __forceinline__ void mc_block_sum(float (&v)[K], float (*sm)[K]) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < K; k++)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    __syncthreads();
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < K; k++) sm[warp][k] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; k++) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kMcWarps; w++) t += sm[w][k];
        v[k] = t;
    }
}

__global__ void __launch_bounds__(kMcThreads)
mix_ce_rows_kernel(const float* __restrict__ x, const int64_t* __restrict__ labels, const mv_mix_rec* __restrict__ recs,
                   int B, int C, float smoothing, float inv_b, float* __restrict__ row_loss, float* __restrict__ dx) {
    __shared__ float sm_max[kMcWarps];
    __shared__ float sm_sum[kMcWarps][3];
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t base = int64_t(b) * C;
    const float* xr = x + base;

    float m = -INFINITY;
    for (int c = threadIdx.x; c < C; c += kMcThreads) m = fmaxf(m, __ldg(xr + c));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) sm_max[warp] = m;
    __syncthreads();
    m = sm_max[0];
#pragma unroll
    for (int w = 1; w < kMcWarps; w++) m = fmaxf(m, sm_max[w]);

    // Z = n + r (n: the elements at the maximum, each e^0 = 1 exactly; r: the rest); S = sum_c (m - x_c) >= 0
    float acc[3] = {0.f, 0.f, 0.f};                  // r, n, S
    for (int c = threadIdx.x; c < C; c += kMcThreads) {
        const float xs = __ldg(xr + c) - m;
        if (xs == 0.f) acc[1] += 1.f; else acc[0] += expf(xs);
        acc[2] -= xs;
    }
    mc_block_sum<3>(acc, sm_sum);
    const float z1 = acc[0] + (acc[1] - 1.f), z = acc[1] + acc[0];
    const float lz = log1pf(z1);                     // lse - m

    const float lam = recs ? recs[b].lam : 1.f;
    const int64_t ya = labels[b], yb = recs ? labels[B - 1 - b] : ya;
    const bool valid = (!(lam > 0.f) || (ya >= 0 && ya < C)) && (!(lam < 1.f) || (yb >= 0 && yb < C));
    const int ia = ya >= 0 && ya < C ? int(ya) : 0, ib = yb >= 0 && yb < C ? int(yb) : 0;
    const float off = smoothing / float(C), on_off = 1.f - smoothing;
    const float la = lz + (m - __ldg(xr + ia)), lb = lz + (m - __ldg(xr + ib));
    const float loss = off * (float(C) * lz + acc[2]) + on_off * (lam * la + (1.f - lam) * lb);
    const float nan = __int_as_float(0x7fffffff);
    if (threadIdx.x == 0) row_loss[b] = valid ? loss : nan;

    // the gradient row (p - t) / B.  Where p or t is above 1/2 it is formed as (1 - t) - (1 - p), with
    // 1 - p = ((Z - 1) - (e^x - 1)) / Z and 1 - t = (1 - s)(1 - w) + (s - off), w = lam [c == ya] + (1 - lam) [c == yb].
    const float rz = 1.f / z, s_off = smoothing - off;
    for (int c = threadIdx.x; c < C; c += kMcThreads) {
        const float xs = __ldg(xr + c) - m;
        const float p = expf(xs) * rz;
        const bool a = c == ia, bb = c == ib;
        const float w = (a ? lam : 0.f) + (bb ? 1.f - lam : 0.f);
        const float t = off + on_off * w;
        float g;
        if (p > 0.5f || t > 0.5f) {
            const float one_w = a && bb ? 0.f : a ? 1.f - lam : bb ? lam : 1.f;
            g = (on_off * one_w + s_off) - (z1 - expm1f(xs)) * rz;
        } else {
            g = p - t;
        }
        dx[base + c] = valid ? g * inv_b : nan;
    }
}

}  // namespace mv

using namespace mv;

extern "C" int mv_mix_draw(const int64_t* seed_dev, int rank, int B, int H, int W, mv_mix_spec spec,
                           mv_mix_rec* recs_dev, void* stream) {
    MV_CHECK(seed_dev && recs_dev, "mv_mix_draw: null pointer");
    MV_CHECK(B > 0 && B % 2 == 0, "mv_mix_draw: the batch must be even (got B=%d)", B);
    MV_CHECK(H > 0 && W > 0 && rank >= 0, "mv_mix_draw: needs H, W > 0 and rank >= 0");
    MV_CHECK(spec.mode == MV_MIX_BATCH || spec.mode == MV_MIX_PAIR || spec.mode == MV_MIX_ELEM,
             "mv_mix_draw: unknown mode %d", spec.mode);
    MV_CHECK(spec.mixup_alpha >= 0.f && spec.cutmix_alpha >= 0.f && (spec.mixup_alpha > 0.f || spec.cutmix_alpha > 0.f),
             "mv_mix_draw: needs alphas >= 0, not both 0");
    MV_CHECK(spec.prob >= 0.f && spec.prob <= 1.f && spec.switch_prob >= 0.f && spec.switch_prob <= 1.f,
             "mv_mix_draw: prob and switch_prob must be in [0, 1]");
    mix_draw_kernel<<<(B + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(seed_dev, rank, B, H, W, spec,
                                                                                     recs_dev);
    g_launches++;
    return check_cuda(cudaGetLastError(), "mix draw launch");
}

extern "C" int mv_mix_ce_loss(const float* logits, const int64_t* labels, const mv_mix_rec* recs_dev, int B, int C,
                              float smoothing, float* loss, float* row_loss, float* dlogits, void* stream) {
    MV_CHECK(logits && labels && loss && row_loss && dlogits, "mv_mix_ce_loss: null pointer");
    MV_CHECK(B > 0 && C >= 2, "mv_mix_ce_loss: needs B >= 1 and C >= 2 (got B=%d, C=%d)", B, C);
    MV_CHECK(recs_dev == nullptr || B % 2 == 0, "mv_mix_ce_loss: mixed batches must be even (got B=%d)", B);
    MV_CHECK(smoothing >= 0.f && smoothing <= 1.f, "mv_mix_ce_loss: needs smoothing in [0, 1]");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    mix_ce_rows_kernel<<<B, kMcThreads, 0, st>>>(logits, labels, recs_dev, B, C, smoothing, 1.f / float(B), row_loss,
                                                 dlogits);
    g_launches++;
    if (check_cuda(cudaGetLastError(), "mix ce rows launch")) return 1;
    return row_mean_launch(row_loss, B, loss, st);
}
