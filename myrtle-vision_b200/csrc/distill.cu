// distill.cu — the distillation loss of DistillWrapper (models/distill.py), forward and backward in one pass.
//
// Replaces the ATen composite (cross_entropy + log_softmax + softmax + kl_div, or argmax + a second cross_entropy,
// their backwards and the weighted sum: about a dozen launches) with one CTA per row and a fixed-order batch sum.
// Per row: three maxima (s, d', t') and the teacher argmax, then the three exp sums and the KL numerator, then both
// gradient rows.  The row is re-read from L1 / L2 between phases: at C <= 1000 the three rows are 12 KB.
#include "common.cuh"
#include "../../include/mv_b200.h"

namespace mv {
extern int64_t g_launches;

constexpr int kDlThreads = 256;
constexpr int kDlWarps = kDlThreads / 32;

// torch.argmax: the largest value, the first index among equal ones, NaN above everything
__device__ __forceinline__ void argmax_merge(float& v, int& i, float v2, int i2) {
    const bool n1 = v != v, n2 = v2 != v2;
    bool take;
    if (n1 || n2) take = n2 && (!n1 || i2 < i);
    else take = v2 > v || (v2 == v && i2 < i);
    if (take) { v = v2; i = i2; }
}

template <int K>
__device__ __forceinline__ void block_sum(float (&v)[K], float (*sm)[K]) {
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
        for (int w = 0; w < kDlWarps; w++) t += sm[w][k];
        v[k] = t;
    }
}

__global__ void __launch_bounds__(kDlThreads)
distill_loss_rows_kernel(const float* __restrict__ s, const float* __restrict__ d, const float* __restrict__ t,
                         const int64_t* __restrict__ labels, int C, float T, float alpha, int hard, float inv_b,
                         float* __restrict__ row_loss, float* __restrict__ ds, float* __restrict__ dd) {
    __shared__ float sm_max[kDlWarps][3];
    __shared__ int sm_arg[kDlWarps];
    __shared__ float sm_arg_v[kDlWarps];
    __shared__ float sm_sum[kDlWarps][7];
    const int b = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t base = int64_t(b) * C;
    const float* sr = s + base;
    const float* dr = d + base;
    const float* tr = t + base;
    // soft: d' = d / T and t' = t / T (torch's division); hard: d' = d, and t only feeds the argmax
    const float Td = hard ? 1.f : T;

    // phase 1: maxima of s, d', t' and the argmax of t
    float ms = -INFINITY, md = -INFINITY, mt = -INFINITY, av = -INFINITY;
    int ai = 0x7fffffff;
    for (int c = threadIdx.x; c < C; c += kDlThreads) {
        const float tv = __ldg(tr + c);
        ms = fmaxf(ms, __ldg(sr + c));
        md = fmaxf(md, __ldg(dr + c) / Td);
        mt = fmaxf(mt, tv / T);
        argmax_merge(av, ai, tv, c);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ms = fmaxf(ms, __shfl_xor_sync(0xffffffffu, ms, o));
        md = fmaxf(md, __shfl_xor_sync(0xffffffffu, md, o));
        mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, o));
        argmax_merge(av, ai, __shfl_xor_sync(0xffffffffu, av, o), __shfl_xor_sync(0xffffffffu, ai, o));
    }
    if (lane == 0) { sm_max[warp][0] = ms; sm_max[warp][1] = md; sm_max[warp][2] = mt; sm_arg_v[warp] = av; sm_arg[warp] = ai; }
    __syncthreads();
    ms = sm_max[0][0]; md = sm_max[0][1]; mt = sm_max[0][2]; av = sm_arg_v[0]; ai = sm_arg[0];
#pragma unroll
    for (int w = 1; w < kDlWarps; w++) {
        ms = fmaxf(ms, sm_max[w][0]); md = fmaxf(md, sm_max[w][1]); mt = fmaxf(mt, sm_max[w][2]);
        argmax_merge(av, ai, sm_arg_v[w], sm_arg[w]);
    }

    // phase 2: the exp sums Z = n + r of s, d', t' (n: the elements at the maximum, each e^0 = 1 exactly; r: the rest)
    // and W = sum_c e^(t'-mt) ((t'-mt) - (d'-md)), so that KL = W / Zt - log Zt + log Zd.  Z - 1 = (n - 1) + r is
    // formed without rounding r against 1: log Z = log1p(Z - 1), and p - 1 of a dominant class does not cancel.
    float acc[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};        // rs, rd, rt, ns, nd, nt, W
    for (int c = threadIdx.x; c < C; c += kDlThreads) {
        const float xs = __ldg(sr + c) - ms, xd = __ldg(dr + c) / Td - md, xt = __ldg(tr + c) / T - mt;
        const float et = expf(xt);
        if (xs == 0.f) acc[3] += 1.f; else acc[0] += expf(xs);
        if (xd == 0.f) acc[4] += 1.f; else acc[1] += expf(xd);
        if (xt == 0.f) acc[5] += 1.f; else acc[2] += et;
        acc[6] += et * (xt - xd);
    }
    block_sum<7>(acc, sm_sum);
    const float zs1 = acc[0] + (acc[3] - 1.f), zd1 = acc[1] + (acc[4] - 1.f), zt1 = acc[2] + (acc[5] - 1.f);
    const float zs = acc[3] + acc[0], zd = acc[4] + acc[1], zt = acc[5] + acc[2];

    const int64_t y = labels[b];
    const bool valid = y >= 0 && y < C;
    const int yi = valid ? int(y) : 0;
    const float ce = log1pf(zs1) + (ms - __ldg(sr + yi));
    float dl;
    if (hard) dl = log1pf(zd1) + (md - __ldg(dr + ai));
    else dl = T * T * (acc[6] / zt - log1pf(zt1) + log1pf(zd1));
    const float nan = __int_as_float(0x7fffffff);
    if (threadIdx.x == 0) row_loss[b] = valid ? (1.f - alpha) * ce + alpha * dl : nan;

    // phase 3: the gradient rows, already divided by B.  A probability above 1/2 is used as 1 - (1 - p), with
    // 1 - p = ((Z - 1) - (e^x - 1)) / Z, so that p - 1 and the difference of two such probabilities keep their digits.
    const float gs = (1.f - alpha) * inv_b;
    const float gd = hard ? alpha * inv_b : alpha * T * inv_b;
    const float rzs = 1.f / zs, rzd = 1.f / zd, rzt = 1.f / zt;
    for (int c = threadIdx.x; c < C; c += kDlThreads) {
        const float xs = __ldg(sr + c) - ms, xd = __ldg(dr + c) / Td - md;
        const float ps = expf(xs) * rzs, pd = expf(xd) * rzd;
        const float qs = (zs1 - expm1f(xs)) * rzs, qd = (zd1 - expm1f(xd)) * rzd;     // 1 - ps, 1 - pd
        float gsv = c == yi ? -qs : ps;
        float gdv;
        if (hard) {
            gdv = c == ai ? -qd : pd;
        } else {
            const float xt = __ldg(tr + c) / T - mt;
            const float pt = expf(xt) * rzt;
            gdv = (pd > 0.5f || pt > 0.5f) ? (zt1 - expm1f(xt)) * rzt - qd : pd - pt;
        }
        ds[base + c] = valid ? gs * gsv : nan;
        dd[base + c] = valid ? gd * gdv : nan;
    }
}

// loss = sum_b row_loss[b] / B in a fixed order: per-thread strided sums, then the warp and CTA trees
__global__ void __launch_bounds__(kDlThreads)
distill_loss_sum_kernel(const float* __restrict__ row_loss, int B, float* __restrict__ loss) {
    __shared__ float sm[kDlWarps][1];
    float v[1] = {0.f};
    for (int i = threadIdx.x; i < B; i += kDlThreads) v[0] += row_loss[i];
    block_sum<1>(v, sm);
    if (threadIdx.x == 0) loss[0] = v[0] / float(B);
}

// loss[0] = mean of row_loss[0, B) with distill_loss_sum_kernel (also the batch sum of mixup.cu's loss)
int row_mean_launch(const float* row_loss, int B, float* loss, cudaStream_t st) {
    distill_loss_sum_kernel<<<1, kDlThreads, 0, st>>>(row_loss, B, loss);
    g_launches++;
    return check_cuda(cudaGetLastError(), "row mean launch");
}

}  // namespace mv

using namespace mv;

extern "C" int mv_distill_loss(const float* student, const float* distill, const float* teacher, const int64_t* labels,
                               int B, int C, float T, float alpha, int hard, float* loss, float* row_loss,
                               float* d_student, float* d_distill, void* stream) {
    MV_CHECK(student && distill && teacher && labels && loss && row_loss && d_student && d_distill,
             "mv_distill_loss: null pointer");
    MV_CHECK(B > 0 && C >= 2, "mv_distill_loss: needs B >= 1 and C >= 2 (got B=%d, C=%d)", B, C);
    MV_CHECK(T > 0.f && alpha >= 0.f && alpha <= 1.f, "mv_distill_loss: needs T > 0 and alpha in [0, 1]");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    distill_loss_rows_kernel<<<B, kDlThreads, 0, st>>>(student, distill, teacher, labels, C, T, alpha, hard ? 1 : 0,
                                                       1.f / float(B), row_loss, d_student, d_distill);
    distill_loss_sum_kernel<<<1, kDlThreads, 0, st>>>(row_loss, B, loss);
    g_launches += 2;
    return check_cuda(cudaGetLastError(), "distill loss launch");
}
