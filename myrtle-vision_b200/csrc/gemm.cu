// gemm.cu — persistent, warp-specialised tcgen05 GEMM with fused fake-quant epilogues
// (north-star kernel class (b)).  C[M,N] = A * B^T over K, fp32 accumulation in TMEM.
//
//   warp 0      TMA producer   (cp.async.bulk.tensor, 128B-swizzled tiles, 6-stage mbarrier ring)
//   warp 1      MMA issuer     (one elected lane issues tcgen05.mma; owns the TMEM allocation)
//   warps 2..5  epilogue       (tcgen05.ld 32 lanes x 32 columns; bias / quant / GELU / residual)
//
// TMEM holds two 128x128 fp32 accumulators so the epilogue of tile i overlaps the MMAs of
// tile i+1.  Operands are the *exact* fp16 containers of the fake-quantised tensors (or
// tf32-in-fp32 for the TF32 format), so products are exact and only the fp32 accumulation
// order differs from the reference's F.linear (torch.nn.qat.Linear.forward; SURVEY.md K3/K4).
// Both K-major and MN-major operands are supported through the UMMA shared-memory
// descriptors, which lets wgrad (dW = dY^T X) read dY and X in their natural layouts.
#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {

extern int64_t g_launches;

constexpr int BM = 128;
constexpr int kATileBytes = BM * 128;                 // A tile per stage: 128 rows x 128 B = 16 KB
constexpr int kEpiWarps = 16;                         // four warps per TMEM lane quadrant
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;
// single-CTA kernel: 128 x 128 tiles, 6-stage ring
constexpr int kGemmBN = 128;
constexpr int kGemmStages = 6;
constexpr int kGemmStageBytes = kATileBytes + kGemmBN * 128;
constexpr int kGemmSmem = kGemmStages * kGemmStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;

// Debug timeline (tools/trace_gemm.py, library built with MV_NVCC_FLAGS=-DMV_GEMM_TRACE): CTA 0 stamps
// clock64() at the hand-offs between the MMA issuer and two of its epilogue warps.  Record = {event, index, clock}.
static unsigned long long* g_gemm_trace = nullptr;
extern "C" int mv_debug_set_gemm_trace(void* dev_buf) { g_gemm_trace = static_cast<unsigned long long*>(dev_buf); return 0; }
#ifndef MV_GEMM_TRACE
#define GEMM_TRACE(cond, region, ev, idx) do { } while (0)
#else
#define GEMM_TRACE(cond, region, ev, idx)                                                      \
    do {                                                                                       \
        if (p.trace != nullptr && blockIdx.x == 0 && (cond)) {                                 \
            unsigned long long* t_ = p.trace + (region) * 3072 + 3 * (trace_n++ % 1024);       \
            t_[0] = (ev); t_[1] = (unsigned long long)(idx); t_[2] = clock64();                \
        }                                                                                      \
    } while (0)
#endif

struct GemmDev {
    unsigned long long* trace;
    int M, N, K;
    int m_tiles, n_tiles, splits, kb_total, kb_per_split;
    int a_major, b_major;
    uint32_t idesc;
    uint32_t idesc2;            // CTA-pair kernel, 384-wide tiles: the second (N = 128) MMA of every k step
    int transpose_out;          // CTA-pair kernel, accumulate: out[n, m] += acc[m, n]
    const float* bias;
    const float* residual; int ld_res;
    __half* aux; int ld_aux;
    void* out; int ld_out; int out_dtype;
    int epilogue;
    FloatFmt q_out, q_res;
    int accumulate;
    int rows_per_img;
    int variant;                // CTA-pair kernel: compile-time epilogue variant (0 = generic), see gemm2_host
    float* colsum;              // CTA-pair kernel: fp32 [N] += column sums of the stored values (fused bias gradient)
    int* ovf;                   // overflow sink (mv_set_overflow_flag) or NULL
    DropDev drop;               // dropout mask of the output (CTA-pair kernel, kDrop instantiations); seed NULL: off
    SrDev sr;                   // stochastic rounding of q_out (CTA-pair kernel, kSR instantiations); seed NULL: off
};

__device__ __forceinline__ float sat16(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }

// erf-GELU (nn.GELU default, models/vit.py:49) and its derivative, branch-free:
//   0.5*erfc(|x|/sqrt2) = t (b1 + t (b2 + t (b3 + t (b4 + t b5)))) exp(-x^2/2),  t = 1 / (1 + 0.2316419 |x|)
// (Abramowitz & Stegun 26.2.17 / 7.1.26).  The exponential is shared with the derivative's pdf term,
// so gelu and gelu' together cost 16 FP32 instructions + 2 MUFU.  Max abs error against the exact fp64
// GELU over [-12, 12]: 4.2e-7 (gelu), 3.0e-7 (gelu') — below half an fp16 ulp of the stored values.
__device__ __forceinline__ void gelu_both(float x, float& g, float& dg) {
    const float t = rcp_fast(fmaf(fabsf(x), 0.2316418882f, 1.0f));
    const float E = ex2_fast(x * x * -0.7213475204f);
    float poly = fmaf(t, 0.5307027145f, -0.7265760135f);
    poly = fmaf(poly, t, 0.7107068705f);
    poly = fmaf(poly, t, -0.142248368f);
    poly = fmaf(poly, t, 0.127414796f);
    const float half_erfc = poly * t * E;
    const float cdf = x >= 0.f ? 1.0f - half_erfc : half_erfc;
    g = x * cdf;
    dg = fmaf(x, 0.3989422804f * E, cdf);
}

// The same arithmetic on two values per instruction (fma/mul/add.f32x2 = FFMA2 / FMUL2 / FADD2 on sm_100a: the FP32 pipe
// does the same lane work, but the epilogue warps issue half as many instructions — the fc1 + GELU kernel is bound
// by issue slots, not by the FP32 pipe).  Operation order per lane is that of gelu_both: bit-identical results.
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t bc2(float c) { return pk2(c, c); }
__device__ __forceinline__ void gelu_both2(float x0, float x1, float& g0, float& g1, float& d0, float& d1) {
    const uint64_t X = pk2(x0, x1);
    float den0, den1, s0, s1;
    upk2(fma2(pk2(fabsf(x0), fabsf(x1)), bc2(0.2316418882f), bc2(1.0f)), den0, den1);
    upk2(mul2(mul2(X, X), bc2(-0.7213475204f)), s0, s1);
    const uint64_t T = pk2(rcp_fast(den0), rcp_fast(den1));
    const uint64_t E = pk2(ex2_fast(s0), ex2_fast(s1));
    uint64_t poly = fma2(T, bc2(0.5307027145f), bc2(-0.7265760135f));
    poly = fma2(poly, T, bc2(0.7107068705f));
    poly = fma2(poly, T, bc2(-0.142248368f));
    poly = fma2(poly, T, bc2(0.127414796f));
    const uint64_t H = mul2(mul2(poly, T), E);                       // 0.5 erfc(|x| / sqrt 2)
    float h0, h1, u0, u1;
    upk2(H, h0, h1);
    upk2(fma2(H, bc2(-1.0f), bc2(1.0f)), u0, u1);                    // 1 - h (the product is exact: same as 1.0f - h)
    const uint64_t C = pk2(x0 >= 0.f ? u0 : h0, x1 >= 0.f ? u1 : h1);
    upk2(mul2(X, C), g0, g1);
    upk2(fma2(X, mul2(E, bc2(0.3989422804f)), C), d0, d1);
}

// float_quantize(5,10) of four values at once: one range test for the group, then 2 integer
// instructions per value.  kSatLater: the caller converts with cvt.rn.satfinite.f16, which performs
// the clip to +-65504 (the rounded value is exactly representable in fp16 otherwise).
template <bool kSatLater>
__device__ __forceinline__ void fq_half4(float (&v)[4]) {
    const float mn = fminf(fminf(fabsf(v[0]), fabsf(v[1])), fminf(fabsf(v[2]), fabsf(v[3])));
    if (mn >= 6.103515625e-05f) {                       // all four at or above fp16's lowest normal binade
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t t = __float_as_uint(v[j]);
            uint32_t q = (t + 0x1000u) & 0xFFFFE000u;
            if (!kSatLater && (q & 0x7FFFFFFFu) > 0x477FE000u) q = (t & 0x80000000u) | 0x477FE000u;
            v[j] = __uint_as_float(q);
        }
    } else {
        // out of line on purpose: inline, ptxas if-converts this into ~50 predicated instructions per group
        const float4 r = fq_half4_rare(v[0], v[1], v[2], v[3]);
        v[0] = r.x; v[1] = r.y; v[2] = r.z; v[3] = r.w;
    }
}

__device__ __forceinline__ void store16(float* dst, const float (&v)[16]) {
#pragma unroll
    for (int j = 0; j < 4; j++)
        reinterpret_cast<float4*>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}
__device__ __forceinline__ void store16(__half* dst, const float (&v)[16]) {
#pragma unroll
    for (int j = 0; j < 2; j++) {
        __half2 h0 = __floats2half2_rn(v[8 * j + 0], v[8 * j + 1]), h1 = __floats2half2_rn(v[8 * j + 2], v[8 * j + 3]);
        __half2 h2 = __floats2half2_rn(v[8 * j + 4], v[8 * j + 5]), h3 = __floats2half2_rn(v[8 * j + 6], v[8 * j + 7]);
        reinterpret_cast<uint4*>(dst)[j] = make_uint4(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1),
                                                     *reinterpret_cast<uint32_t*>(&h2), *reinterpret_cast<uint32_t*>(&h3));
    }
}
// row-major store of 16 consecutive outputs; fp16 stores saturate (gradient operands)
__device__ __forceinline__ void store_out16(void* base, int dtype, int64_t row, int ld, int col,
                                            float (&v)[16], bool vec_ok, int nvalid) {
    if (dtype == MV_F32) {
        float* p = reinterpret_cast<float*>(base) + row * ld + col;
        if (vec_ok) store16(p, v);
        else for (int j = 0; j < 16; j++) if (j < nvalid) p[j] = v[j];
    } else {
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = sat16(v[j]);
        __half* p = reinterpret_cast<__half*>(base) + row * ld + col;
        if (vec_ok) store16(p, v);
        else for (int j = 0; j < 16; j++) if (j < nvalid) p[j] = __float2half_rn(v[j]);
    }
}

// Single-CTA kernel: tf32-in-fp32 operands (kind::tf32), 128 x 128 tiles.
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
            const GemmDev p) {
    constexpr int BN = kGemmBN;
    constexpr int kStages = kGemmStages;
    constexpr int kStageBytes = kGemmStageBytes;
    constexpr int kTileBytes = kATileBytes;
    constexpr int kEsz = 4;                    // operand element size
    constexpr int BK = 128 / kEsz;             // elements of K per stage (one 128-byte swizzle row)
    constexpr int UMMA_K = 32 / kEsz;          // K elements per tcgen05.mma
    constexpr int kMnChunk = 128 / kEsz;       // MN elements per 128-byte row (MN-major tiles)
    constexpr int kMnBoxBytes = BK * 128;      // one MN-major TMA box: BK k-rows of 128 bytes

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; offset arithmetic keeps the shared address space
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
        for (int s = 0; s < kStages; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; a++) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], kEpiWarps); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<2 * BN>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // work units: (tile, k split)
    const int unit0 = blockIdx.x, unit_stride = gridDim.x;
    const int total_units = p.m_tiles * p.n_tiles * p.splits;

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int u = unit0; u < total_units; u += unit_stride) {
                const int split = u % p.splits;
                const int tile = u / p.splits;
                const int m0 = (tile / p.n_tiles) * BM, n0 = (tile % p.n_tiles) * BN;
                const int kb0 = split * p.kb_per_split;
                const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * kStageBytes;
                    uint8_t* sb = sa + kTileBytes;
                    mbar_arrive_expect_tx(&full_bar[stage], kStageBytes);
                    if (p.a_major == 0) {
                        tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * BK, m0);
                    } else {
#pragma unroll
                        for (int c = 0; c < BM / kMnChunk; c++)
                            tma_load_2d(sa + c * kMnBoxBytes, &tmap_a, &full_bar[stage], m0 + c * kMnChunk, kb * BK);
                    }
                    if (p.b_major == 0) {
                        // two half-tiles of BN/2 rows
#pragma unroll
                        for (int c = 0; c < 2; c++)
                            tma_load_2d(sb + c * (BN / 2) * 128, &tmap_b, &full_bar[stage], kb * BK, n0 + c * (BN / 2));
                    } else {
#pragma unroll
                        for (int c = 0; c < BN / kMnChunk; c++)
                            tma_load_2d(sb + c * kMnBoxBytes, &tmap_b, &full_bar[stage], n0 + c * kMnChunk, kb * BK);
                    }
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ==================================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            // K-major: 8-row groups 1024 B apart, K advance = 32 B inside the swizzled row.
            // MN-major: 128-byte rows are k-slices; 8 k-rows per 1024 B group (SBO), next 64/32
            // MN elements one TMA box further (LBO); K advance = UMMA_K rows.
            const uint32_t a_lbo = p.a_major ? kMnBoxBytes : 16, b_lbo = p.b_major ? kMnBoxBytes : 16;
            const uint32_t a_kstep = p.a_major ? UMMA_K * 128 : 32, b_kstep = p.b_major ? UMMA_K * 128 : 32;
            for (int u = unit0; u < total_units; u += unit_stride) {
                const int split = u % p.splits;
                const int kb0 = split * p.kb_per_split;
                const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * kStageBytes);
                    const uint32_t sb = sa + kTileBytes;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adesc = make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024);
                        const uint64_t bdesc = make_smem_desc_sw128(sb + k * b_kstep, b_lbo, 1024);
                        const uint32_t accum = (kb > kb0 || k > 0) ? 1u : 0u;
                        umma_tf32(tmem_d, adesc, bdesc, p.idesc, accum);
                    }
                    umma_commit(&empty_bar[stage]);            // frees the smem slot when the MMAs retire
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full[acc]);                  // accumulator ready for the epilogue
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ================================ epilogue ====================================
        // 16 warps: warp e covers TMEM lane quadrant (warp & 3) and column group (e >> 2) of the tile.
        // Each epilogue warp is latency-bound (dependent math on one element set), so the step's
        // elementwise work is spread over 4 warps per scheduler.
        const int quad = warp & 3;
        const int cgrp = (warp - 2) >> 2;
        constexpr int kColsPerWarp = BN / (kEpiWarps / 4);
        const int mode_out = fq_mode(p.q_out), mode_res = fq_mode(p.q_res);
        int acc = 0; uint32_t acc_phase = 0;
        for (int u = unit0; u < total_units; u += unit_stride) {
            const int tile = u / p.splits;
            const int m0 = (tile / p.n_tiles) * BM, n0 = (tile % p.n_tiles) * BN;
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const int m = m0 + quad * 32 + lane;
            const bool row_ok = m < p.M;
            const int64_t rrow = p.rows_per_img > 0 ? (m % p.rows_per_img) : m;
#pragma unroll 1
            for (int c = 0; c < kColsPerWarp / 16; c++) {
                // 16 columns per iteration keeps the unrolled math small enough for the instruction cache
                const int col = cgrp * kColsPerWarp + c * 16;
                const int n = n0 + col;
                const int nvalid = min(16, p.N - n);
                const bool live = row_ok && nvalid > 0;
                // issue the epilogue's global loads before waiting on the accumulator so their
                // HBM latency overlaps the TMEM read
                const bool vec_res = live && p.residual != nullptr && nvalid == 16 && (p.ld_res & 3) == 0;
                const bool vec_aux = live && p.epilogue == MV_EPI_DGELU && nvalid == 16 && (p.ld_aux & 7) == 0;
                float4 res4[4];
                uint4 aux4[2];
                if (vec_res) {
                    const float4* rp4 = reinterpret_cast<const float4*>(p.residual + rrow * p.ld_res + n);
#pragma unroll
                    for (int j = 0; j < 4; j++) res4[j] = __ldcs(rp4 + j);
                }
                if (vec_aux) {
                    const uint4* ap4 = reinterpret_cast<const uint4*>(p.aux + int64_t(m) * p.ld_aux + n);
#pragma unroll
                    for (int j = 0; j < 2; j++) aux4[j] = __ldcs(ap4 + j);
                }
                uint32_t r[16];
                tmem_ld_32x16(tmem_base + (uint32_t(quad * 32) << 16) + acc * BN + col, r);
                tmem_ld_wait();
                if (!live) continue;
                float v[16];
#pragma unroll
                for (int j = 0; j < 16; j++) v[j] = __uint_as_float(r[j]);
                if (p.accumulate) {
                    float* o = reinterpret_cast<float*>(p.out) + int64_t(m) * p.ld_out + n;
#pragma unroll
                    for (int j = 0; j < 16; j++) if (j < nvalid) atomicAdd(o + j, v[j]);
                    continue;
                }
                const bool full = nvalid == 16;
                if (p.bias != nullptr) {
                    if (full) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n) + j);
                            v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
                        }
                    } else {
                        for (int j = 0; j < 16; j++) if (j < nvalid) v[j] += __ldg(p.bias + n + j);
                    }
                }
                if (mode_out) {
#pragma unroll
                    for (int j = 0; j < 16; j++) v[j] = fq_apply(v[j], mode_out, p.q_out);
                }
                if (p.epilogue == MV_EPI_GELU) {
                    // out = gelu(u); aux = gelu'(u) (all the backward needs)
                    float d[16];
#pragma unroll
                    for (int j = 0; j < 16; j++) gelu_both(v[j], v[j], d[j]);
                    __half* up = p.aux + int64_t(m) * p.ld_aux + n;
                    if (full && (p.ld_aux & 7) == 0) store16(up, d);
                    else for (int j = 0; j < 16; j++) if (j < nvalid) up[j] = __float2half_rn(d[j]);
                } else if (p.epilogue == MV_EPI_DGELU) {
                    const __half* up = p.aux + int64_t(m) * p.ld_aux + n;
                    if (vec_aux) {
#pragma unroll
                        for (int j = 0; j < 2; j++) {
                            const uint4 w = aux4[j];
                            const __half2* h = reinterpret_cast<const __half2*>(&w);
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const float2 f = __half22float2(h[q]);
                                v[8 * j + 2 * q] *= f.x;
                                v[8 * j + 2 * q + 1] *= f.y;
                            }
                        }
                    } else {
                        for (int j = 0; j < 16; j++) if (j < nvalid) v[j] *= __half2float(up[j]);
                    }
                }
                if (p.residual != nullptr) {
                    const float* rp = p.residual + rrow * p.ld_res + n;
                    if (vec_res) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const float4 b = res4[j];
                            v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
                        }
                    } else {
                        for (int j = 0; j < 16; j++) if (j < nvalid) v[j] += rp[j];
                    }
                }
                if (mode_res) {
#pragma unroll
                    for (int j = 0; j < 16; j++) v[j] = fq_apply(v[j], mode_res, p.q_res);
                }
                if (p.out_dtype == MV_F16 && !mode_out && !mode_res && p.epilogue != MV_EPI_GELU) {
                    float amax = 0.f;
#pragma unroll
                    for (int j = 0; j < 16; j++) if (j < nvalid) amax = fmaxf(amax, fabsf(v[j]));
                    raise_overflow(p.ovf, amax);
                }
                const int esz_o = p.out_dtype == MV_F32 ? 4 : 2;
                const bool vec_o = full && ((p.ld_out * esz_o) % 16 == 0);
                store_out16(p.out, p.out_dtype, m, p.ld_out, n, v, vec_o, nvalid);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<2 * BN>(tmem_base);
    }
}

// =====================================================================================
// CTA-pair kernel (cta_group::2): fp16 operands.
//
// A cluster of two CTAs (one TPC) owns a 256 x BN output tile.  Each CTA stages its own 128 rows
// of A and BN/2 rows of B (one third less L2->SM operand traffic per flop than two independent
// 128 x BN tiles, the bound of the K=384 GEMMs of ViT-Small); the leader CTA's elected lane issues
// tcgen05.mma.cta_group::2 (M=256) and each CTA ends up with its 128 x BN half of the accumulator
// in its own TMEM.  Barriers:
//   full[s]   (leader's)  1 arrive.expect_tx by the leader's producer + TMA bytes of both CTAs
//   empty[s]  (per CTA)   multicast tcgen05.commit from the leader: the stage is free in both CTAs
//   tmem_full[a] (per CTA) multicast commit: accumulator a is complete
//   tmem_empty[a] (leader's) 2 x kEpi2Warps arrivals: both CTAs' epilogues have drained accumulator a
//
// Epilogue: the TMEM layout (thread = row) would make every global access touch 32 different
// lines per warp instruction, which made the previous kernel LSU-bound.  Here each warp moves a
// 32 x 32 fp32 chunk TMEM -> registers -> padded shared memory and then works in a row-contiguous
// layout (8 lanes x 16 B per row, 4 rows per instruction): every bias / residual / aux load and
// every store covers whole 32-byte sectors of consecutive addresses.
// Epilogue warps per CTA, a launch-time choice between two instantiations.  18 warps (16 + producer + issuer)
// put five warps on one scheduler's 16 K registers, which caps every thread at 96 registers and makes the
// epilogues with residual / aux prefetch spill; 14 warps (12 + 2) allow 128.  The elementwise-heavy GELU /
// gelu' epilogues (N = 1536 outputs) are bound by issue slots and latency and run faster on 16 warps; every
// other epilogue runs faster on 12 spill-free ones (measured per shape).
constexpr int kStgPitch = 36;                                  // floats per staged row: 32 + 4 pad
constexpr int kStgBytesPerWarp = 32 * kStgPitch * 4;           // 4608
// AUX: the gelu' epilogue's second operand (aux, fp16 [M, N]) arrives by TMA, one 32 x 32 chunk per epilogue warp, requested
// by that warp a chunk ahead (kAuxChunkBytes each): loaded with LDG just before use, its latency was a quarter of all stall
// samples of that kernel (ncu, r2_gemm_dgelu), and fetching it earlier into registers spills.
// AUX = 2: the same for the fp32 residual of the x + Linear(...) epilogues (32 x 32 fp32 = 4 KB per chunk).
// AUX = 3: no extra buffer (fp16 outputs leave by TMA store from the warp's staging area, epi_chunk_tma16).
template <int AUX> struct AuxChunk { static constexpr int kBytes = AUX == 3 ? 0 : (AUX == 2 ? 32 * 128 : 32 * 64); };
template <int BN, int EW, int AUX = 0> struct Gemm2Cfg {
    static constexpr int kThreads = 64 + 32 * EW;
    static constexpr int kBHalfBytes = (BN / 2) * 128;
    static constexpr int kStageBytes = kATileBytes + kBHalfBytes;
    static constexpr int kStagingBytes = EW * kStgBytesPerWarp;
    static constexpr int kAuxBytes = AUX ? EW * AuxChunk<AUX>::kBytes : 0;
    static constexpr int kBarBytes = 512;
    static constexpr int kStages = (232448 - kStagingBytes - kAuxBytes - 1024 - kBarBytes) / kStageBytes;
    static constexpr int kSmem = kStages * kStageBytes + kStagingBytes + kAuxBytes + 1024 + kBarBytes;
    static constexpr int kTmemCols = 2 * BN <= 256 ? 256 : 512;
};

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d)
                 : "memory");
}
__device__ __forceinline__ uint2 pack4_f16_sat(const float (&v)[4]) {
    uint2 r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r.x) : "f"(v[1]), "f"(v[0]));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r.y) : "f"(v[3]), "f"(v[2]));
    return r;
}
// 4 consecutive outputs of one row; vec: 16-byte (fp32) / 8-byte (fp16) aligned and all 4 in range
__device__ __forceinline__ void store_out4(void* base, int dtype, int64_t row, int ld, int col,
                                           const float (&v)[4], bool vec, int nvalid) {
    if (dtype == MV_F32) {
        float* o = reinterpret_cast<float*>(base) + row * ld + col;
        if (vec) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        else for (int j = 0; j < 4; j++) if (j < nvalid) o[j] = v[j];
    } else {
        __half* o = reinterpret_cast<__half*>(base) + row * ld + col;
        if (vec) *reinterpret_cast<uint2*>(o) = pack4_f16_sat(v);
        else for (int j = 0; j < 4; j++) if (j < nvalid) o[j] = __float2half_rn(sat16(v[j]));
    }
}


// ---- epilogue of the CTA-pair kernel ----------------------------------------------------------
struct EpiWarp {
    unsigned long long* tr;     // debug timeline slot of this warp (MV_GEMM_TRACE), else unused
    float* stg;                 // this warp's 32 x kStgPitch fp32 staging tile
    uint32_t stg_s;             // ... as a shared-space address
    int lane, lr, lc;           // row-contiguous layout: row = 4*it + lr, columns lc .. lc+3 of the chunk
    int mode_out, mode_res;
};

// explicit shared-space accesses: through the EpiWarp struct the compiler loses the address space and emits
// generic LD / ST for the staging tile, which go down the global-memory path (long scoreboard)
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, float a, float b, float c, float d) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// accumulator chunk (32 TMEM lanes x 32 columns): thread = row -> padded shared memory; optionally
// release the accumulator buffer (arrive on the leader's tmem_empty barrier) right after the read
__device__ __forceinline__ void stage_chunk(const EpiWarp& w, uint32_t taddr, uint32_t release) {
    uint32_t r[32];
    tmem_ld_32x32(taddr, r);
    tmem_ld_wait();
    const uint32_t srow = w.stg_s + w.lane * (kStgPitch * 4);
#pragma unroll
    for (int j = 0; j < 8; j++)
        sts128(srow + 16 * j, __uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
               __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
    if (release != 0u) {
        tc_fence_before();
        __syncwarp();
        if (w.lane == 0) mbar_arrive_cluster(release);
    }
    __syncwarp();
}

// Fast path: the chunk lies inside [M, N], every pointer / pitch is vector-aligned (checked on the
// host, GemmDev::variant) and the epilogue's shape is a compile-time choice, so the unrolled row
// loop is a few instructions per 4 outputs.  kRes: 0 none, 1 residual[m, n], 2 residual[m % rows_per_img, n].
// kDrop: dropout after q_out (include/mv_b200.h "dropout mask"; the host guarantees N % 8 == 0, so the four columns of a
// lane are one half of a Philox block and lanes 2k / 2k+1 share the block: drop_keep4_pair, rows 2j / 2j+1).
// kSR: q_out rounds stochastically with the gradient rounding stream (p.sr; the host sets kQO = 0 and N % 8 == 0).  The
// 16-bit stream shares each Philox block between lanes 2k / 2k+1 as kDrop does (rows 2j / 2j+1, sr_pair16); the 32-bit
// stream takes one call per lane and row.
template <int kOut, int kEpi, int kRes, int kQO, int kQR, bool kAcc, bool kCS = false, bool kDrop = false, bool kSR = false>
__device__ __forceinline__ void epi_chunk(const GemmDev& p, const EpiWarp& w, uint32_t taddr, uint32_t release,
                                          int mrow0, int nc0, const uint2* aux_pre = nullptr, const float4* res_pre = nullptr) {
    const int n = nc0 + w.lc;
    const int m_first = mrow0 + w.lr;
    float4 res4[8];
    uint2 aux2[8];
    if (kRes != 0) {
#pragma unroll
        for (int it = 0; it < 8; it++) {
            const int m = m_first + it * 4;
            const int64_t rrow = kRes == 2 ? (m % p.rows_per_img) : m;
            res4[it] = res_pre != nullptr ? res_pre[it] : __ldcs(reinterpret_cast<const float4*>(p.residual + rrow * p.ld_res + n));
        }
    }
    if (kEpi == MV_EPI_DGELU) {
#pragma unroll
        for (int it = 0; it < 8; it++)
            aux2[it] = aux_pre != nullptr ? aux_pre[it]
                                          : __ldcs(reinterpret_cast<const uint2*>(p.aux + int64_t(m_first + it * 4) * p.ld_aux + n));
    }
    float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!kAcc && p.bias != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n));
    uint32_t keep = 0;                                 // bit 4 * it + j: row m_first + 4 * it, column n + j is kept
    if (kDrop) {
        const uint64_t seed = __ldg(reinterpret_cast<const unsigned long long*>(p.drop.seed));
        const bool odd = w.lane & 1;
#pragma unroll
        for (int it = 0; it < 8; it += 2) {
            const uint64_t i = uint64_t(m_first + (it + (odd ? 1 : 0)) * 4) * uint64_t(p.N) + uint64_t(n);
            keep |= drop_keep4_pair(seed, p.drop, i >> 3, odd) << (4 * it);
        }
    }
#ifdef MV_GEMM_TRACE
    if (w.tr != nullptr && w.lane == 0) { w.tr[0] = 20; w.tr[1] = nc0; w.tr[2] = clock64(); }
#endif
    stage_chunk(w, taddr, release);
#ifdef MV_GEMM_TRACE
    if (w.tr != nullptr && w.lane == 0) { w.tr[3] = 21; w.tr[4] = nc0; w.tr[5] = clock64(); }
#endif
    const uint32_t sp = w.stg_s + (w.lr * kStgPitch + w.lc) * 4;
    float cs[4] = {0.f, 0.f, 0.f, 0.f};
    // unquantised values rounded into an fp16 container (gradient operands; qkv of FP16_32): report saturation
    constexpr bool kOvf = kOut == MV_F16 && kQO == 0 && kQR == 0 && kEpi != MV_EPI_GELU && !kAcc;
    float amax = 0.f;
    uint64_t sr_s = 0;
    bool s16 = false;
    if (kSR) { sr_s = sr_seed(p.sr); s16 = p.q_out.man_bits >= 7; }
    uint2 sr_next = make_uint2(0u, 0u);                // 16-bit stream: the odd row's half, computed with the even row
#pragma unroll
    for (int it = 0; it < 8; it++) {
        const int m = m_first + it * 4;
        const float4 a4 = lds128(sp + it * 4 * kStgPitch * 4);
        float v[4] = {a4.x, a4.y, a4.z, a4.w};
        if (kAcc) {
            red_add_v4(reinterpret_cast<float*>(p.out) + int64_t(m) * p.ld_out + n, v[0], v[1], v[2], v[3]);
            continue;
        }
        if (kEpi == MV_EPI_GELU) {
            upk2(add2(pk2(v[0], v[1]), pk2(b4.x, b4.y)), v[0], v[1]);
            upk2(add2(pk2(v[2], v[3]), pk2(b4.z, b4.w)), v[2], v[3]);
        } else {
            v[0] += b4.x; v[1] += b4.y; v[2] += b4.z; v[3] += b4.w;
        }
        if (kQO == 1) fq_half4<false>(v);
        if (kSR) {
            uint4 r;
            if (s16) {
                if ((it & 1) == 0) {
                    const bool odd = w.lane & 1;
                    const uint64_t i = uint64_t(m_first + (it + (odd ? 1 : 0)) * 4) * uint64_t(p.N) + uint64_t(n);
                    const uint4 ab = sr_pair16(sr_s, p.sr.offset, i >> 3, odd);
                    r = sr_halves(make_uint2(ab.x, ab.y));
                    sr_next = make_uint2(ab.z, ab.w);
                } else {
                    r = sr_halves(sr_next);
                }
            } else {
                r = sr_bits4(sr_s, p.sr.offset, uint64_t(m) * uint64_t(p.N) + uint64_t(n), false);
            }
            const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int j = 0; j < 4; j++) {
                amax = fmaxf(amax, fabsf(v[j]));       // a value the format saturates beyond the fp16 range still raises the flag
                v[j] = fq_stoch_elem(v[j], rr[j], p.q_out);
            }
        }
        if (kEpi == MV_EPI_GELU) {
            float d[4];
            gelu_both2(v[0], v[1], v[0], v[1], d[0], d[1]);
            gelu_both2(v[2], v[3], v[2], v[3], d[2], d[3]);
            if (kDrop) {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const float s = drop_mul(keep, 4 * it + j, p.drop.scale);
                    v[j] *= s; d[j] *= s;
                }
            }
            *reinterpret_cast<uint2*>(p.aux + int64_t(m) * p.ld_aux + n) = pack4_f16_sat(d);
            if (kQR == 1 && kOut == MV_F16 && !kCS) {
                // fc2's input quantiser: add half an fp16 ulp, convert with RZ (fq_half4_pack) — 1.5 instructions per value
                *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out) + int64_t(m) * p.ld_out + n) =
                    fq_half4_pack(v[0], v[1], v[2], v[3]);
                continue;
            }
        } else if (kEpi == MV_EPI_DGELU) {
            const __half2* hh = reinterpret_cast<const __half2*>(&aux2[it]);
            const float2 f0 = __half22float2(hh[0]), f1 = __half22float2(hh[1]);
            v[0] *= f0.x; v[1] *= f0.y; v[2] *= f1.x; v[3] *= f1.y;
        }
        if (kDrop && kEpi != MV_EPI_GELU) {
#pragma unroll
            for (int j = 0; j < 4; j++) v[j] *= drop_mul(keep, 4 * it + j, p.drop.scale);
        }
        if (kRes != 0) { v[0] += res4[it].x; v[1] += res4[it].y; v[2] += res4[it].z; v[3] += res4[it].w; }
        if (kQR == 1) fq_half4<kOut == MV_F16>(v);
        if (kCS) { cs[0] += v[0]; cs[1] += v[1]; cs[2] += v[2]; cs[3] += v[3]; }
        if (kOvf) amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v[0]), fabsf(v[1])), fmaxf(fabsf(v[2]), fabsf(v[3]))));
        if (kOut == MV_F32)
            *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + int64_t(m) * p.ld_out + n) =
                make_float4(v[0], v[1], v[2], v[3]);
        else
            *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.out) + int64_t(m) * p.ld_out + n) = pack4_f16_sat(v);
    }
    if (kCS) {
        // this warp's 32 rows of columns n .. n+3: the 4 lanes that share the columns hold 8 rows each
#pragma unroll
        for (int j = 0; j < 4; j++) {
            cs[j] += __shfl_xor_sync(0xffffffffu, cs[j], 8);
            cs[j] += __shfl_xor_sync(0xffffffffu, cs[j], 16);
        }
        if (w.lr == 0) red_add_v4(p.colsum + n, cs[0], cs[1], cs[2], cs[3]);
    }
    if (kOvf) raise_overflow(p.ovf, amax);
#ifdef MV_GEMM_TRACE
    if (w.tr != nullptr && w.lane == 0) { w.tr[6] = 22; w.tr[7] = nc0; w.tr[8] = clock64(); }
#endif
    __syncwarp();                                      // staging is rewritten by the next chunk
}

// fp16 outputs with no second operand (qkv forward, the plain dgrads): the chunk never takes the fp32 staging round trip.
// Each thread keeps its accumulator row (thread = row, 32 columns), adds the bias, quantises, packs 64 bytes of fp16 into a
// [32 rows][64 B] tile (64-byte TMA swizzle: 16-byte chunk c of row r sits at c ^ ((r >> 1) & 3), conflict-free) and one
// TMA store per chunk writes it out — no LDS, no per-lane global stores.  Two tiles per warp inside its staging area: the
// store of chunk i - 2 must have been read before chunk i overwrites its tile (bulk-group wait by the issuing lane).
template <int kQO>
__device__ __forceinline__ void epi_chunk_tma16(const GemmDev& p, const EpiWarp& w, uint32_t taddr, uint32_t release,
                                                int mrow0, int nc0, const CUtensorMap* tmap_out, int which) {
    uint32_t r[32];
    tmem_ld_32x32(taddr, r);
    tmem_ld_wait();
    if (release != 0u) {
        tc_fence_before();
        __syncwarp();
        if (w.lane == 0) mbar_arrive_cluster(release);
    }
    float amax = 0.f;
    uint32_t h[16];
#pragma unroll
    for (int g4 = 0; g4 < 8; g4++) {
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + nc0) + g4);
        float v[4] = {__uint_as_float(r[4 * g4]) + b4.x, __uint_as_float(r[4 * g4 + 1]) + b4.y,
                      __uint_as_float(r[4 * g4 + 2]) + b4.z, __uint_as_float(r[4 * g4 + 3]) + b4.w};
        if (kQO == 1) fq_half4<true>(v);
        else amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v[0]), fabsf(v[1])), fmaxf(fabsf(v[2]), fabsf(v[3]))));
        const uint2 pk = pack4_f16_sat(v);
        h[2 * g4] = pk.x; h[2 * g4 + 1] = pk.y;
    }
    if (kQO == 0) raise_overflow(p.ovf, amax);
    if (w.lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the tile's previous store has been read
    __syncwarp();
    const uint32_t tile = w.stg_s + which * 2048;
    const uint32_t row = tile + w.lane * 64;
    const int sw = (w.lane >> 1) & 3;
#pragma unroll
    for (int c = 0; c < 4; c++)
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + ((c ^ sw) << 4)), "r"(h[4 * c]), "r"(h[4 * c + 1]),
                     "r"(h[4 * c + 2]), "r"(h[4 * c + 3]) : "memory");
    fence_proxy_async();
    __syncwarp();
    if (w.lane == 0) {
        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                         reinterpret_cast<uint64_t>(tmap_out)), "r"(tile), "r"(nc0), "r"(mrow0) : "memory");
        tma_store_commit();
    }
}

// Split-K accumulation into the TRANSPOSED output, out[n, m] += acc[m, n]: the staged 32 x 32 chunk is read
// column-wise (lane = column, conflict-free with the 36-float pitch), so every lane adds 4 consecutive m of one
// output row with one red.add.v4.  Lets a wgrad whose natural output is 384 tall and wide (fc2: [384, 1536]) run
// as its transpose on 256 x 384 tiles without padding rows.
__device__ __forceinline__ void epi_chunk_acc_t(const GemmDev& p, const EpiWarp& w, uint32_t taddr, uint32_t release,
                                                int mrow0, int nc0) {
    stage_chunk(w, taddr, release);
    float* o = reinterpret_cast<float*>(p.out) + int64_t(nc0 + w.lane) * p.ld_out + mrow0;
    const uint32_t sp = w.stg_s + w.lane * 4;
#pragma unroll
    for (int g = 0; g < 8; g++) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; j++)
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v[j]) : "r"(sp + (4 * g + j) * kStgPitch * 4));
        red_add_v4(o + 4 * g, v[0], v[1], v[2], v[3]);
    }
    __syncwarp();
}

// Generic path: tails in M / N, unaligned pitches.  Same arithmetic, rolled loops.
// kDrop: the dropout mask element by element (any N).  kSR: q_out rounds stochastically, element by element (any N).
template <bool kDrop = false, bool kSR = false>
__device__ __forceinline__ void epi_chunk_generic(const GemmDev& p, const EpiWarp& w, uint32_t taddr, uint32_t release,
                                               int mrow0, int nc0) {
    stage_chunk(w, taddr, release);
    const int n = nc0 + w.lc;
    const int nvalid = min(4, p.N - n);
    if (nvalid > 0) {
        const uint64_t sr_s = kSR ? sr_seed(p.sr) : 0ull;
        float cs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
        for (int it = 0; it < 8; it++) {
            const int row = it * 4 + w.lr;
            const int m = mrow0 + row;
            if (m >= p.M) break;
            const float4 a4 = *reinterpret_cast<const float4*>(w.stg + row * kStgPitch + w.lc);
            float v[4] = {a4.x, a4.y, a4.z, a4.w};
            if (p.accumulate) {
                float* o = reinterpret_cast<float*>(p.out) + (p.transpose_out ? int64_t(n) * p.ld_out + m : int64_t(m) * p.ld_out + n);
                const int64_t step = p.transpose_out ? p.ld_out : 1;
                for (int j = 0; j < 4; j++) if (j < nvalid) atomicAdd(o + j * step, v[j]);
                continue;
            }
            if (p.bias != nullptr) for (int j = 0; j < 4; j++) if (j < nvalid) v[j] += __ldg(p.bias + n + j);
            if (kSR) {
                for (int j = 0; j < 4; j++)
                    if (j < nvalid) {
                        if (p.out_dtype == MV_F16) raise_overflow(p.ovf, fabsf(v[j]));
                        const uint32_t r = sr_bits1(sr_s, p.sr.offset, uint64_t(m) * uint64_t(p.N) + uint64_t(n + j), p.q_out.man_bits >= 7);
                        v[j] = float_quantize_elem<true>(v[j], r, p.q_out.exp_bits, p.q_out.man_bits);
                    }
            } else if (w.mode_out) for (int j = 0; j < 4; j++) v[j] = fq_apply(v[j], w.mode_out, p.q_out);
            float dm[4] = {1.f, 1.f, 1.f, 1.f};
            if (kDrop) {
                const uint64_t seed = __ldg(reinterpret_cast<const unsigned long long*>(p.drop.seed));
                for (int j = 0; j < 4; j++)
                    if (j < nvalid)
                        dm[j] = philox_half16(seed, uint64_t(m) * uint64_t(p.N) + uint64_t(n + j), uint64_t(uint32_t(p.drop.site))) >= p.drop.thr
                                    ? p.drop.scale : 0.f;
            }
            if (p.epilogue == MV_EPI_GELU) {
                __half* up = p.aux + int64_t(m) * p.ld_aux + n;
                for (int j = 0; j < 4; j++) {
                    float d;
                    gelu_both(v[j], v[j], d);
                    if (kDrop) { v[j] *= dm[j]; d *= dm[j]; }
                    if (j < nvalid) up[j] = __float2half_rn(d);
                }
            } else if (p.epilogue == MV_EPI_DGELU) {
                const __half* up = p.aux + int64_t(m) * p.ld_aux + n;
                for (int j = 0; j < 4; j++) if (j < nvalid) v[j] *= __half2float(up[j]);
            }
            if (kDrop && p.epilogue != MV_EPI_GELU) for (int j = 0; j < 4; j++) v[j] *= dm[j];
            if (p.residual != nullptr) {
                const int64_t rrow = p.rows_per_img > 0 ? (m % p.rows_per_img) : m;
                const float* rp = p.residual + rrow * p.ld_res + n;
                for (int j = 0; j < 4; j++) if (j < nvalid) v[j] += rp[j];
            }
            if (w.mode_res) for (int j = 0; j < 4; j++) v[j] = fq_apply(v[j], w.mode_res, p.q_res);
            for (int j = 0; j < 4; j++) cs[j] += v[j];
            if (p.out_dtype == MV_F16 && (kSR || !w.mode_out) && !w.mode_res && p.epilogue != MV_EPI_GELU)
                for (int j = 0; j < 4; j++) if (j < nvalid) raise_overflow(p.ovf, fabsf(v[j]));
            store_out4(p.out, p.out_dtype, m, p.ld_out, n, v, false, nvalid);
        }
        if (p.colsum != nullptr && !p.accumulate)
            for (int j = 0; j < 4; j++) if (j < nvalid) atomicAdd(p.colsum + n + j, cs[j]);
    }
    __syncwarp();
}

// kDrop: the dropout instantiations (variants 3, 4, 5, 9 and the generic path with the mask).  Separate kernels so that
// the register allocation of the kernels without dropout — the maximum over every epilogue a kernel contains — stays as it is.
// kSR: the stochastic gradient-rounding instantiations (variants 1, 6, 11 with q_out rounded by the stream of p.sr, and
// the generic path with it), separate for the same reason.
template <int BN, int EW, int AUX = 0, bool kDrop = false, bool kSR = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(64 + 32 * EW, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
             const __grid_constant__ CUtensorMap tmap_aux, const __grid_constant__ GemmDev p) {
    using Cfg = Gemm2Cfg<BN, EW, AUX>;
    constexpr int kEpi2Warps = EW;
    constexpr int kStages = Cfg::kStages;
    constexpr int kStageBytes = Cfg::kStageBytes;
    constexpr int BK = 64, UMMA_K = 16;
    constexpr int kMnBoxBytes = BK * 128;      // one MN-major TMA box: 64 k-rows x 128 B (64 elements)
    constexpr int BNH = BN / 2;                // B rows staged by each CTA
    // BN = 384 (split-K wgrad with MN-major B, outputs 384 wide): two MMAs per k step, N = 256 into accumulator
    // columns [0, 256) and N = 128 into [256, 384) — a 256 x 128 tile needs 105 GB/s of operands per SM, more
    // than the L2 delivers (~72 GB/s per SM), a 256 x 384 tile 59 GB/s.  One accumulator buffer (384 of the 512
    // TMEM columns): the epilogue of these long-K units is a few per cent of their time.
    constexpr int kAccBufs = 2 * BN <= 512 ? 2 : 1;

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; offset arithmetic keeps the shared address space
    float* staging = reinterpret_cast<float*>(smem + kStages * kStageBytes);
    uint8_t* aux_buf = smem + kStages * kStageBytes + Cfg::kStagingBytes;            // [EW][32 rows][64 B] (AUX)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * kStageBytes + Cfg::kStagingBytes + Cfg::kAuxBytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full = empty_bar + kStages;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    uint64_t* aux_full = tmem_empty + 4;                                             // [EW] (AUX)

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int rank = int(cluster_ctarank());
    [[maybe_unused]] int trace_n = 0;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
        for (int s = 0; s < kStages; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; a++) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 2 * kEpi2Warps); }
        if (AUX) { tma_prefetch_desc(&tmap_aux); for (int e = 0; e < EW; e++) mbar_init(&aux_full[e], 1); }
        (void)aux_buf;
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc_cg2<Cfg::kTmemCols>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                        // both CTAs' barriers and TMEM exist before any cross-CTA signal
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // work units: (256 x BN tile, k split); both CTAs of a pair walk the same sequence
    const int unit0 = blockIdx.x >> 1, unit_stride = gridDim.x >> 1;
    const int total_units = p.m_tiles * p.n_tiles * p.splits;

    if (warp == 0) {
        // ================================ TMA producer (both CTAs) ================================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int u = unit0; u < total_units; u += unit_stride) {
                const int split = u % p.splits;
                const int tile = u / p.splits;
                const int m0 = (tile / p.n_tiles) * 256 + rank * 128;
                const int nbase = (tile % p.n_tiles) * BN;
                const int n0 = nbase + rank * BNH;
                const int kb0 = split * p.kb_per_split;
                const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * kStageBytes;
                    uint8_t* sb = sa + kATileBytes;
                    const uint32_t lead_full = mapa_shared(smem_u32(&full_bar[stage]), 0);
                    if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * kStageBytes);
                    if (p.a_major == 0) {
                        tma_load_2d_cg2(sa, &tmap_a, lead_full, kb * BK, m0);
                    } else {
#pragma unroll
                        for (int c = 0; c < 2; c++)
                            tma_load_2d_cg2(sa + c * kMnBoxBytes, &tmap_a, lead_full, m0 + c * 64, kb * BK);
                    }
                    if (p.b_major == 0) {
                        tma_load_2d_cg2(sb, &tmap_b, lead_full, kb * BK, n0);
                    } else {
#pragma unroll
                        for (int c = 0; c < BNH / 64; c++) {
                            // 384-wide tiles: this CTA's half of the N = 256 MMA (2 chunks), then of the N = 128 MMA
                            const int nc = BN == 384 ? (c < 2 ? nbase + rank * 128 + c * 64 : nbase + 256 + rank * 64)
                                                     : n0 + c * 64;
                            tma_load_2d_cg2(sb + c * kMnBoxBytes, &tmap_b, lead_full, nc, kb * BK);
                        }
                    }
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer (leader CTA only) ============================
        if (rank == 0 && lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            const uint32_t a_lbo = p.a_major ? kMnBoxBytes : 16, b_lbo = p.b_major ? kMnBoxBytes : 16;
            const uint32_t a_kstep = p.a_major ? UMMA_K * 128 : 32, b_kstep = p.b_major ? UMMA_K * 128 : 32;
            for (int u = unit0; u < total_units; u += unit_stride) {
                const int split = u % p.splits;
                const int kb0 = split * p.kb_per_split;
                const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
                GEMM_TRACE(true, 0, 1, u);                     // issuer: waits for a free accumulator
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                GEMM_TRACE(true, 0, 2, u);                     // accumulator free
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * BN;
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(&full_bar[stage], phase);
                    if (kb == kb0) GEMM_TRACE(true, 0, 3, u);  // first operand stage landed
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + stage * kStageBytes);
                    const uint32_t sb = sa + kATileBytes;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adesc = make_smem_desc_sw128(sa + k * a_kstep, a_lbo, 1024);
                        const uint64_t bdesc = make_smem_desc_sw128(sb + k * b_kstep, b_lbo, 1024);
                        umma_f16_cg2(tmem_d, adesc, bdesc, p.idesc, (kb > kb0 || k > 0) ? 1u : 0u);
                        if (BN == 384) {
                            const uint64_t bdesc2 = make_smem_desc_sw128(sb + 2 * kMnBoxBytes + k * b_kstep, b_lbo, 1024);
                            umma_f16_cg2(tmem_d + 256, adesc, bdesc2, p.idesc2, (kb > kb0 || k > 0) ? 1u : 0u);
                        }
                    }
                    umma_commit_cg2(&empty_bar[stage], 3);     // stage free in both CTAs when the MMAs retire
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
                umma_commit_cg2(&tmem_full[acc], 3);           // both CTAs' epilogues may read accumulator acc
                GEMM_TRACE(true, 0, 4, u);                     // all MMAs of the tile issued
                if (++acc == kAccBufs) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ================================ epilogue (both CTAs) ====================================
        const int quad = warp & 3;                             // TMEM lane quadrant this warp may read
        const int cg = (warp - 2) >> 2;                        // chunks cg, cg+4, ... of the tile's 32-column chunks
        EpiWarp w;
        w.stg = staging + (warp - 2) * (32 * kStgPitch);
        w.stg_s = smem_u32(w.stg);
        w.lane = lane; w.lr = lane >> 3; w.lc = (lane & 7) * 4;
        w.tr = nullptr;
        w.mode_out = fq_mode(p.q_out); w.mode_res = fq_mode(p.q_res);
        const uint32_t lead_empty0 = mapa_shared(smem_u32(&tmem_empty[0]), 0);
        int acc = 0; uint32_t acc_phase = 0;
        // The epilogue variant is chosen ONCE, outside the tile / chunk loops (a per-chunk switch costs an
        // indirect branch and an instruction-cache excursion on every chunk): `walk` is the loop nest, `chunk`
        // the compile-time epilogue of a chunk that lies inside [M, N].
        auto walk = [&](auto chunk) {
            for (int u = unit0; u < total_units; u += unit_stride) {
                const int tile = u / p.splits;
                const int mrow0 = (tile / p.n_tiles) * 256 + rank * 128 + quad * 32;
                const int n0 = (tile % p.n_tiles) * BN;
                GEMM_TRACE(lane == 0 && (warp == 2 || warp == 17), warp == 2 ? 1 : 2, 5, u);    // epilogue warp waits for the tile
                mbar_wait(&tmem_full[acc], acc_phase);
                GEMM_TRACE(lane == 0 && (warp == 2 || warp == 17), warp == 2 ? 1 : 2, 6, u);    // accumulator complete
                tc_fence_after();
#pragma unroll 1
                for (int c = cg; c < BN / 32; c += kEpi2Warps / 4) {
                    const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + acc * BN + c * 32;
                    // last TMEM read of this tile by this warp: hand the accumulator back to the MMA issuer
                    const uint32_t release = (c + kEpi2Warps / 4 >= BN / 32) ? lead_empty0 + acc * 8 : 0u;
                    const int nc0 = n0 + c * 32;
                    const bool fast = p.variant != 0 && mrow0 + 32 <= p.M && nc0 + 32 <= p.N;
#ifdef MV_GEMM_TRACE
                    if (p.trace != nullptr && blockIdx.x == 0 && warp == 2) { w.tr = p.trace + 3072 + 3 * (trace_n % 1021); trace_n += 3; }
#endif
                    if (fast) chunk(taddr, release, mrow0, nc0);
                    else {
                        if constexpr (AUX == 3) {          // the generic path stages through the area the TMA tiles live in
                            if (lane == 0) tma_store_wait_read();
                            __syncwarp();
                        }
                        epi_chunk_generic<kDrop, kSR>(p, w, taddr, release, mrow0, nc0);
                    }
                }
                GEMM_TRACE(lane == 0 && (warp == 2 || warp == 17), warp == 2 ? 1 : 2, 7, u);    // this warp's chunks done
                if (++acc == kAccBufs) { acc = 0; acc_phase ^= 1; }
            }
        };
        // AUX: the same walk with this warp's aux chunk requested one chunk ahead (TMA into its 2 KB buffer; the request
        // for the next chunk — of this tile or of the warp's next tile — goes out as soon as the current one is in registers)
        [[maybe_unused]] auto walk_aux = [&](auto chunk) {
            const int wi = warp - 2;
            constexpr int kAuxChunkBytes = AuxChunk<AUX>::kBytes;
            uint8_t* abuf = aux_buf + wi * kAuxChunkBytes;
            uint64_t* abar = &aux_full[wi];
            uint32_t aphase = 0;
            constexpr int kStep = kEpi2Warps / 4;
            auto request = [&](int u, int c) {
                const int tile = u / p.splits;
                const int mrow0 = (tile / p.n_tiles) * 256 + rank * 128 + quad * 32;
                const int nc0 = (tile % p.n_tiles) * BN + c * 32;
                if (lane == 0) {
                    mbar_arrive_expect_tx(abar, kAuxChunkBytes);
                    tma_load_2d(abuf, &tmap_aux, abar, nc0, mrow0);
                }
            };
            if (unit0 < total_units) request(unit0, cg);
            for (int u = unit0; u < total_units; u += unit_stride) {
                const int tile = u / p.splits;
                const int mrow0 = (tile / p.n_tiles) * 256 + rank * 128 + quad * 32;
                const int n0 = (tile % p.n_tiles) * BN;
                mbar_wait(&tmem_full[acc], acc_phase);
                tc_fence_after();
#pragma unroll 1
                for (int c = cg; c < BN / 32; c += kStep) {
                    const uint32_t taddr = tmem_base + (uint32_t(quad * 32) << 16) + acc * BN + c * 32;
                    const uint32_t release = (c + kStep >= BN / 32) ? lead_empty0 + acc * 8 : 0u;
                    const int nc0 = n0 + c * 32;
                    const bool fast = mrow0 + 32 <= p.M && nc0 + 32 <= p.N;
                    mbar_wait(abar, aphase);
                    aphase ^= 1;
                    uint2 aux2[8];
                    float4 res4[8];
#pragma unroll
                    for (int it = 0; it < 8; it++) {
                        if (AUX == 2) res4[it] = *reinterpret_cast<const float4*>(abuf + (it * 4 + w.lr) * 128 + (lane & 7) * 16);
                        else aux2[it] = *reinterpret_cast<const uint2*>(abuf + (it * 4 + w.lr) * 64 + (lane & 7) * 8);
                    }
                    // the buffer is about to be overwritten through the async proxy: without this fence single 64-byte rows of
                    // the NEXT chunk's box showed up in these (generic-proxy) reads, a few hundred values per launch
                    fence_proxy_async();
                    __syncwarp();
                    if (c + kStep < BN / 32) request(u, c + kStep);
                    else if (u + unit_stride < total_units) request(u + unit_stride, cg);
                    if (fast) chunk(taddr, release, mrow0, nc0, aux2, res4);
                    else epi_chunk_generic<kDrop, kSR>(p, w, taddr, release, mrow0, nc0);
                }
                if (++acc == kAccBufs) { acc = 0; acc_phase ^= 1; }
            }
        };
        if constexpr (kSR && AUX == 1) {
            if (p.variant == 11)
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2* aux2, const float4*) {
                    epi_chunk<MV_F16, MV_EPI_DGELU, 0, 0, 0, false, true, false, true>(p, w, taddr, release, mrow0, nc0, aux2);
                });
            else
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2* aux2, const float4*) {
                    epi_chunk<MV_F16, MV_EPI_DGELU, 0, 0, 0, false, false, false, true>(p, w, taddr, release, mrow0, nc0, aux2);
                });
        } else if constexpr (kSR) {
            if (p.variant == 1)
                walk([&](uint32_t taddr, uint32_t release, int mrow0, int nc0) {
                    epi_chunk<MV_F16, MV_EPI_NONE, 0, 0, 0, false, false, false, true>(p, w, taddr, release, mrow0, nc0);
                });
            else           // every chunk takes the generic path with stochastic rounding
                walk([&](uint32_t, uint32_t, int, int) {});
        } else if constexpr (kDrop && AUX == 2) {
            if (p.variant == 4)
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2*, const float4* res4) {
                    epi_chunk<MV_F32, MV_EPI_NONE, 1, 1, 1, false, false, true>(p, w, taddr, release, mrow0, nc0, nullptr, res4);
                });
            else
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2*, const float4* res4) {
                    epi_chunk<MV_F32, MV_EPI_NONE, 1, 0, 0, false, false, true>(p, w, taddr, release, mrow0, nc0, nullptr, res4);
                });
        } else if constexpr (kDrop) {
#define MV_EPI_DROP_CASE(id, ...)                                                                              \
    case id:                                                                                                   \
        walk([&](uint32_t taddr, uint32_t release, int mrow0, int nc0) {                                       \
            epi_chunk<__VA_ARGS__, false, true>(p, w, taddr, release, mrow0, nc0);                             \
        });                                                                                                    \
        break;
            switch (p.variant) {
                //                   out     epilogue      res qo qr acc
                MV_EPI_DROP_CASE(3, MV_F32, MV_EPI_NONE, 1, 0, 0, false)
                MV_EPI_DROP_CASE(4, MV_F32, MV_EPI_NONE, 1, 1, 1, false)
                MV_EPI_DROP_CASE(5, MV_F16, MV_EPI_GELU, 0, 0, 1, false)
                MV_EPI_DROP_CASE(9, MV_F16, MV_EPI_GELU, 0, 1, 1, false)
                default:   // every chunk takes the generic path with the mask
                    walk([&](uint32_t, uint32_t, int, int) {});
                    break;
            }
#undef MV_EPI_DROP_CASE
        } else if constexpr (AUX == 1) {
            if (p.variant == 11)
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2* aux2, const float4*) {
                    epi_chunk<MV_F16, MV_EPI_DGELU, 0, 0, 0, false, true>(p, w, taddr, release, mrow0, nc0, aux2);
                });
            else
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2* aux2, const float4*) {
                    epi_chunk<MV_F16, MV_EPI_DGELU, 0, 0, 0, false>(p, w, taddr, release, mrow0, nc0, aux2);
                });
        } else if constexpr (AUX == 3) {
            // fp16 outputs without a second operand: direct TMA-store epilogue (epi_chunk_tma16), tiles alternate per chunk
            int which = 0;
            if (p.variant == 2)
                walk([&](uint32_t taddr, uint32_t release, int mrow0, int nc0) {
                    epi_chunk_tma16<1>(p, w, taddr, release, mrow0, nc0, &tmap_aux, which); which ^= 1; });
            else
                walk([&](uint32_t taddr, uint32_t release, int mrow0, int nc0) {
                    epi_chunk_tma16<0>(p, w, taddr, release, mrow0, nc0, &tmap_aux, which); which ^= 1; });
            if (lane == 0) tma_store_wait_all();
        } else if constexpr (AUX == 2) {
            if (p.variant == 4)
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2*, const float4* res4) {
                    epi_chunk<MV_F32, MV_EPI_NONE, 1, 1, 1, false>(p, w, taddr, release, mrow0, nc0, nullptr, res4);
                });
            else
                walk_aux([&](uint32_t taddr, uint32_t release, int mrow0, int nc0, const uint2*, const float4* res4) {
                    epi_chunk<MV_F32, MV_EPI_NONE, 1, 0, 0, false>(p, w, taddr, release, mrow0, nc0, nullptr, res4);
                });
        } else {
#define MV_EPI_CASE(id, ...)                                                                                   \
    case id:                                                                                                   \
        walk([&](uint32_t taddr, uint32_t release, int mrow0, int nc0) {                                       \
            epi_chunk<__VA_ARGS__>(p, w, taddr, release, mrow0, nc0);                                          \
        });                                                                                                    \
        break;
        switch (p.variant) {
            //              out     epilogue      res qo qr acc
            MV_EPI_CASE(1, MV_F16, MV_EPI_NONE, 0, 0, 0, false)
            MV_EPI_CASE(2, MV_F16, MV_EPI_NONE, 0, 1, 0, false)
            MV_EPI_CASE(3, MV_F32, MV_EPI_NONE, 1, 0, 0, false)
            MV_EPI_CASE(4, MV_F32, MV_EPI_NONE, 1, 1, 1, false)
            MV_EPI_CASE(5, MV_F16, MV_EPI_GELU, 0, 0, 1, false)
            MV_EPI_CASE(6, MV_F16, MV_EPI_DGELU, 0, 0, 0, false)
            MV_EPI_CASE(7, MV_F32, MV_EPI_NONE, 2, 0, 0, false)
            MV_EPI_CASE(8, MV_F32, MV_EPI_NONE, 0, 0, 0, true)
            MV_EPI_CASE(9, MV_F16, MV_EPI_GELU, 0, 1, 1, false)
            MV_EPI_CASE(10, MV_F32, MV_EPI_NONE, 2, 1, 1, false)
            MV_EPI_CASE(11, MV_F16, MV_EPI_DGELU, 0, 0, 0, false, true)
            case 12:
                walk([&](uint32_t taddr, uint32_t release, int mrow0, int nc0) { epi_chunk_acc_t(p, w, taddr, release, mrow0, nc0); });
                break;
            default:       // variant 0: every chunk takes the generic path (`fast` is false)
                walk([&](uint32_t, uint32_t, int, int) {});
                break;
        }
#undef MV_EPI_CASE
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                        // the peer may still be signalling / reading this CTA
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_cg2<Cfg::kTmemCols>(tmem_base);
    }
}

template <int BN, int EW, int AUX = 0, bool kDrop = false, bool kSR = false>
static int launch_gemm2(const CUtensorMap& ta, const CUtensorMap& tb, const GemmDev& p, int grid, cudaStream_t st,
                        const CUtensorMap* taux = nullptr) {
    using Cfg = Gemm2Cfg<BN, EW, AUX>;
    static bool attr_done = false;
    if (!attr_done) {
        MV_CUDA(cudaFuncSetAttribute(gemm2_kernel<BN, EW, AUX, kDrop, kSR>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem));
        attr_done = true;
    }
    gemm2_kernel<BN, EW, AUX, kDrop, kSR><<<grid, Cfg::kThreads, Cfg::kSmem, st>>>(ta, tb, taux != nullptr ? *taux : ta, p);
    return 0;
}

}  // namespace mv

using namespace mv;

// CTA-pair path: fp16 operands, 256 x BN cluster tiles
static int gemm2_host(const mv_gemm_args* a, void* stream) {
    constexpr int BK = 64;
    // BN: least padding of N, ties to the wider tile; MN-major B is staged in 64-element chunks per CTA
    int BN = 128, best = -1;
    const int cands[3] = {256, 192, 128};
    for (int i = 0; i < 3; i++) {
        const int bn = cands[i];
        if (a->b_major == 1 && bn == 192) continue;
        if (a->tile_n != 0 && a->tile_n != bn) continue;
        const int padded = ((a->N + bn - 1) / bn) * bn;
        if (best < 0 || padded < best) { best = padded; BN = bn; }
    }
    // split-K wgrad into outputs whose width is a multiple of 384 but not of 256: 256 x 384 tiles (see gemm2_kernel).
    // Measured at 65792 tokens (tools/probe_gemm_wgrad.py): [1536,384] 88 -> 66 us (1178 TFLOP/s), [1152,384]
    // 81 -> 62 us, [384,384] 33 -> 28 us; widths that 256 also divides gain nothing ([384,1536] 83 -> 81 us) or lose
    // to the larger split count ([384,768] 45 -> 55 us) and keep the 256-wide tiles unless tile_n asks for 384.
    if (a->b_major == 1 && a->accumulate && a->N % 384 == 0 &&
        (a->tile_n == 384 || (a->tile_n == 0 && a->N % 256 != 0))) { BN = 384; best = a->N; }
    MV_CHECK(best >= 0, "mv_gemm: tile_n %d not available for this operand layout", a->tile_n);
    CUtensorMap ta, tb;
    if (a->a_major == 0) { if (make_tmap_2d(&ta, a->A, a->a_dtype, a->M, a->K, a->lda, BM, BK)) return 1; }
    else                 { if (make_tmap_2d(&ta, a->A, a->a_dtype, a->K, a->M, a->lda, BK, 64)) return 1; }
    if (a->b_major == 0) { if (make_tmap_2d(&tb, a->B, a->b_dtype, a->N, a->K, a->ldb, BN / 2, BK)) return 1; }
    else                 { if (make_tmap_2d(&tb, a->B, a->b_dtype, a->K, a->N, a->ldb, BK, 64)) return 1; }

    GemmDev p;
    p.trace = g_gemm_trace;
    p.M = a->M; p.N = a->N; p.K = a->K;
    p.m_tiles = (a->M + 255) / 256;
    p.n_tiles = (a->N + BN - 1) / BN;
    p.kb_total = (a->K + BK - 1) / BK;
    int splits = 1;
    if (a->accumulate) {
        // split K so that the work units fill whole rounds of the 74 clusters: the split count (at most two
        // rounds' worth) with the best units / (rounds * clusters); ties go to fewer splits (fewer red.adds)
        const int tiles = p.m_tiles * p.n_tiles, clusters = kNumSMs / 2;
        double best = -1.0;
        for (int sp = 1; sp <= p.kb_total && sp * tiles <= 2 * clusters; sp++) {
            const int units = sp * tiles;
            const double eff = double(units) / double(((units + clusters - 1) / clusters) * clusters);
            if (eff > best + 1e-9) { best = eff; splits = sp; }
        }
    }
    p.kb_per_split = (p.kb_total + splits - 1) / splits;
    p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
    p.a_major = a->a_major; p.b_major = a->b_major;
    p.idesc = make_idesc(0, 0, a->a_major, a->b_major, 256, BN == 384 ? 256 : BN);
    p.idesc2 = make_idesc(0, 0, a->a_major, a->b_major, 256, 128);
    p.bias = a->bias; p.residual = a->residual; p.ld_res = a->ld_res;
    p.aux = reinterpret_cast<__half*>(a->aux); p.ld_aux = a->ld_aux;
    p.out = a->out; p.ld_out = a->ld_out; p.out_dtype = a->out_dtype;
    p.epilogue = a->epilogue;
    p.q_out = FloatFmt{a->q_out_exp, a->q_out_man};
    p.q_res = FloatFmt{a->q_res_exp, a->q_res_man};
    p.accumulate = a->accumulate;
    p.transpose_out = a->transpose_out;
    p.rows_per_img = a->rows_per_img;
    p.colsum = a->accumulate ? nullptr : a->colsum;
    p.ovf = g_overflow;
    const bool drop = a->drop_seed != nullptr;
    MV_CHECK(!drop || (!a->accumulate && a->colsum == nullptr),
             "mv_gemm: dropout needs a plain output (no accumulate or colsum)");
    MV_CHECK(!drop || a->epilogue != MV_EPI_DGELU, "mv_gemm: the gelu' epilogue takes its mask from aux, not from drop_seed");
    p.drop = DropDev{a->drop_seed, a->drop_thr, a->drop_scale, a->drop_site};
    const bool srnd = a->round_seed != nullptr;
    p.sr = SrDev{a->round_seed, a->round_offset};
    // epilogue variant (epi_chunk<> instantiations in gemm2_kernel); anything else runs the generic path
    {
        auto al = [](const void* q, int bytes) { return (reinterpret_cast<uintptr_t>(q) & (bytes - 1)) == 0; };
        auto qkind = [](int e, int m) { return e == 0 ? 0 : ((e == 5 && m == 10) ? 1 : 2); };
        // stochastic rounding replaces q_out in the kSR kernels: the variant is chosen as for an output without q_out
        const int qo = srnd ? 0 : qkind(a->q_out_exp, a->q_out_man), qr = qkind(a->q_res_exp, a->q_res_man);
        const int res = a->residual == nullptr ? 0 : (a->rows_per_img > 0 ? 2 : 1);
        const int cs = a->colsum != nullptr ? 1 : 0;
        const bool ok = (a->ld_out & 3) == 0 && (a->bias == nullptr || al(a->bias, 16)) &&
                        (cs == 0 || al(a->colsum, 16)) &&
                        (res == 0 || ((a->ld_res & 3) == 0 && al(a->residual, 16))) &&
                        (a->aux == nullptr || ((a->ld_aux & 3) == 0 && al(a->aux, 8))) &&
                        al(a->out, a->out_dtype == MV_F32 ? 16 : 8);
        struct Row { int id, out, epi, res, qo, qr, cs; };
        static const Row table[] = {
            {1, MV_F16, MV_EPI_NONE, 0, 0, 0, 0}, {2, MV_F16, MV_EPI_NONE, 0, 1, 0, 0}, {3, MV_F32, MV_EPI_NONE, 1, 0, 0, 0},
            {4, MV_F32, MV_EPI_NONE, 1, 1, 1, 0}, {5, MV_F16, MV_EPI_GELU, 0, 0, 1, 0}, {6, MV_F16, MV_EPI_DGELU, 0, 0, 0, 0},
            {7, MV_F32, MV_EPI_NONE, 2, 0, 0, 0}, {9, MV_F16, MV_EPI_GELU, 0, 1, 1, 0}, {10, MV_F32, MV_EPI_NONE, 2, 1, 1, 0},
            {11, MV_F16, MV_EPI_DGELU, 0, 0, 0, 1}};
        int v = 0;
        if (ok && a->accumulate) v = a->transpose_out ? 12 : 8;
        else if (ok)
            for (const Row& r : table)
                if (r.out == a->out_dtype && r.epi == a->epilogue && r.res == res && r.qo == qo && r.qr == qr && r.cs == cs) v = r.id;
        // the dropout kernels have compile-time epilogues for the residual and GELU variants; a lane's four columns must be
        // half a Philox block (N % 8 == 0, epi_chunk), everything else takes the generic path with the mask
        if (drop && !((v == 3 || v == 4 || v == 5 || v == 9) && a->N % 8 == 0)) v = 0;
        // the kSR kernels have compile-time epilogues for the plain fp16 dgrad and the gelu' dgrad (its four columns per
        // lane are half a 16-bit-stream block only with N % 8 == 0); everything else takes the generic path
        if (srnd && !((v == 1 || v == 6 || v == 11) && a->N % 8 == 0)) v = 0;
        p.variant = v;
    }

    const int units = p.m_tiles * p.n_tiles * p.splits;
    const int grid = 2 * (units < kNumSMs / 2 ? units : kNumSMs / 2);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc;
    // 16 epilogue warps only where 12 would be unbalanced: BN = 256 is 8 chunks over 3 column groups (3 / 3 / 2)
    const bool heavy = (a->epilogue == MV_EPI_GELU || a->epilogue == MV_EPI_DGELU) && BN == 256;
    // gelu' epilogue on 256-wide tiles with a compile-time variant: its aux operand by TMA, a chunk ahead
    const bool aux_tma = heavy && BN == 256 && (p.variant == 6 || p.variant == 11) && (a->ld_aux & 7) == 0 &&
                         (reinterpret_cast<uintptr_t>(a->aux) & 15) == 0;
    // the kSR kernels have the gelu' epilogue only with its aux operand by TMA (AUX = 1); without it (tiles narrower than
    // 256: an mlp_dim that 256 does not divide, or a forced tile_n; an unaligned aux) every chunk takes the generic path
    if (srnd && (p.variant == 6 || p.variant == 11) && !aux_tma) p.variant = 0;
    // x + Linear(...) epilogues with a row-for-row fp32 residual on 192-wide tiles (proj at D = 384): likewise, where the
    // epilogue and not the operand stream bounds the tile (short K: 56.5 -> 46.6 us at K = 384; at K = 1536 the two
    // operand stages it costs lose more than the prefetch gains, 93.3 -> 96.5 us)
    const bool res_tma = !heavy && BN == 192 && a->K <= 768 && (p.variant == 3 || p.variant == 4) && (a->ld_res & 3) == 0 &&
                         (reinterpret_cast<uintptr_t>(a->residual) & 15) == 0;
    CUtensorMap taux;
    if (aux_tma && make_tmap_2d_plain(&taux, a->aux, MV_F16, a->M, a->N, a->ld_aux, 32, 32)) return 1;
    if (res_tma && make_tmap_2d_plain(&taux, a->residual, MV_F32, a->M, a->N, a->ld_res, 32, 32)) return 1;
    // plain fp16 outputs (variants 1, 2) on 192- / 128-wide tiles: TMA-store epilogue
    const bool out_tma = !srnd && !heavy && (BN == 192 || BN == 128) && (p.variant == 1 || p.variant == 2) && (a->ld_out & 7) == 0 &&
                         (reinterpret_cast<uintptr_t>(a->out) & 15) == 0;
    if (out_tma && make_tmap_2d_plain(&taux, a->out, MV_F16, a->M, a->N, a->ld_out, 32, 32, 1)) return 1;
    if (srnd) {
        if (aux_tma) rc = launch_gemm2<256, 16, 1, false, true>(ta, tb, p, grid, st, &taux);
        else if (BN == 256) rc = heavy ? launch_gemm2<256, 16, 0, false, true>(ta, tb, p, grid, st) : launch_gemm2<256, 12, 0, false, true>(ta, tb, p, grid, st);
        else if (BN == 192) rc = launch_gemm2<192, 12, 0, false, true>(ta, tb, p, grid, st);
        else rc = launch_gemm2<128, 12, 0, false, true>(ta, tb, p, grid, st);
    } else if (drop) {
        if (res_tma) rc = launch_gemm2<192, 12, 2, true>(ta, tb, p, grid, st, &taux);
        else if (BN == 256) rc = heavy ? launch_gemm2<256, 16, 0, true>(ta, tb, p, grid, st) : launch_gemm2<256, 12, 0, true>(ta, tb, p, grid, st);
        else if (BN == 192) rc = launch_gemm2<192, 12, 0, true>(ta, tb, p, grid, st);
        else rc = launch_gemm2<128, 12, 0, true>(ta, tb, p, grid, st);
    } else if (BN == 384) rc = launch_gemm2<384, 12>(ta, tb, p, grid, st);
    else if (out_tma) rc = BN == 192 ? launch_gemm2<192, 12, 3>(ta, tb, p, grid, st, &taux) : launch_gemm2<128, 12, 3>(ta, tb, p, grid, st, &taux);
    else if (aux_tma) rc = launch_gemm2<256, 16, 1>(ta, tb, p, grid, st, &taux);
    else if (res_tma) rc = launch_gemm2<192, 12, 2>(ta, tb, p, grid, st, &taux);
    else if (BN == 256) rc = heavy ? launch_gemm2<256, 16>(ta, tb, p, grid, st) : launch_gemm2<256, 12>(ta, tb, p, grid, st);
    else if (BN == 192) rc = launch_gemm2<192, 12>(ta, tb, p, grid, st);
    else rc = launch_gemm2<128, 12>(ta, tb, p, grid, st);
    if (rc) return rc;
    g_launches++;
    return check_cuda(cudaGetLastError(), "gemm2 launch");
}

extern "C" int mv_gemm(const mv_gemm_args* a, void* stream) {
    MV_CHECK(a != nullptr, "mv_gemm: null args");
    MV_CHECK(a->M > 0 && a->N > 0 && a->K > 0, "mv_gemm: bad shape %dx%dx%d", a->M, a->N, a->K);
    MV_CHECK(a->A && a->B && a->out, "mv_gemm: null operand");
    MV_CHECK((a->a_dtype == MV_F16 || a->a_dtype == MV_F32) && a->b_dtype == a->a_dtype,
             "mv_gemm: A and B must share one element type, MV_F16 or MV_F32 (got %d x %d)", a->a_dtype, a->b_dtype);
    MV_CHECK(a->out_dtype == MV_F16 || a->out_dtype == MV_F32, "mv_gemm: output type %d is neither MV_F16 nor MV_F32", a->out_dtype);
    const bool tf32 = a->a_dtype == MV_F32;
    if (a->accumulate) MV_CHECK(a->out_dtype == MV_F32, "mv_gemm: accumulate needs an fp32 output");
    MV_CHECK(!a->transpose_out || (a->accumulate && !tf32),
             "mv_gemm: transpose_out needs accumulate on the CTA-pair kernel (fp16 operands)");
    if (a->epilogue == MV_EPI_GELU || a->epilogue == MV_EPI_DGELU) MV_CHECK(a->aux != nullptr, "mv_gemm: GELU epilogues need aux");
    if (a->round_seed != nullptr) {
        MV_CHECK(!tf32, "mv_gemm: stochastic rounding is only fused into the CTA-pair kernel (fp16 operands)");
        MV_CHECK(a->q_out_exp >= 1 && a->q_out_exp <= 8 && a->q_out_man >= 1 && a->q_out_man <= 22,
                 "mv_gemm: q_out (%d, %d) is not a float format to round stochastically", a->q_out_exp, a->q_out_man);
        MV_CHECK(!a->accumulate && a->drop_seed == nullptr && a->residual == nullptr && a->epilogue != MV_EPI_GELU,
                 "mv_gemm: stochastic rounding needs a plain or gelu' output (no accumulate, dropout, residual or GELU)");
    }
    if (!tf32) return gemm2_host(a, stream);
    // tf32: the single-CTA kernel
    MV_CHECK(a->colsum == nullptr, "mv_gemm: colsum is only fused into the CTA-pair kernel (fp16 operands)");
    MV_CHECK(a->drop_seed == nullptr, "mv_gemm: dropout is only fused into the CTA-pair kernel (fp16 operands); "
                                      "apply mv_dropout to the output instead");
    constexpr int BK = 32;                     // tf32 elements per 128-byte row
    constexpr int BN = kGemmBN;
    static bool attr_done = false;
    if (!attr_done) {
        MV_CUDA(cudaFuncSetAttribute(gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGemmSmem));
        attr_done = true;
    }

    CUtensorMap ta, tb;
    // K-major operand [rows = M|N, cols = K]: box = 128 rows x 128 B of K.
    // MN-major operand stored [K, M|N]: box = BK k-rows x 128 B of M|N.
    if (a->a_major == 0) { if (make_tmap_2d(&ta, a->A, MV_F32, a->M, a->K, a->lda, BM, BK)) return 1; }
    else                 { if (make_tmap_2d(&ta, a->A, MV_F32, a->K, a->M, a->lda, BK, BK)) return 1; }
    if (a->b_major == 0) { if (make_tmap_2d(&tb, a->B, MV_F32, a->N, a->K, a->ldb, BN / 2, BK)) return 1; }
    else                 { if (make_tmap_2d(&tb, a->B, MV_F32, a->K, a->N, a->ldb, BK, BK)) return 1; }

    GemmDev p;
    p.trace = nullptr;
    p.M = a->M; p.N = a->N; p.K = a->K;
    p.m_tiles = (a->M + BM - 1) / BM;
    p.n_tiles = (a->N + BN - 1) / BN;
    p.kb_total = (a->K + BK - 1) / BK;
    int splits = 1;
    if (a->accumulate) {
        const int tiles = p.m_tiles * p.n_tiles;
        splits = kNumSMs / tiles;
        if (splits < 1) splits = 1;
        if (splits > p.kb_total) splits = p.kb_total;
    }
    p.kb_per_split = (p.kb_total + splits - 1) / splits;
    p.splits = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;
    p.a_major = a->a_major; p.b_major = a->b_major;
    p.idesc = make_idesc(2, 2, a->a_major, a->b_major, BM, BN);
    p.bias = a->bias; p.residual = a->residual; p.ld_res = a->ld_res;
    p.aux = reinterpret_cast<__half*>(a->aux); p.ld_aux = a->ld_aux;
    p.out = a->out; p.ld_out = a->ld_out; p.out_dtype = a->out_dtype;
    p.epilogue = a->epilogue;
    p.q_out = FloatFmt{a->q_out_exp, a->q_out_man};
    p.q_res = FloatFmt{a->q_res_exp, a->q_res_man};
    p.accumulate = a->accumulate;
    p.rows_per_img = a->rows_per_img;
    p.variant = 0; p.colsum = nullptr; p.idesc2 = 0; p.transpose_out = 0; p.ovf = g_overflow;
    p.drop = DropDev{nullptr, 0u, 0.f, 0};
    p.sr = SrDev{nullptr, 0ull};

    const int units = p.m_tiles * p.n_tiles * p.splits;
    const int grid = units < kNumSMs ? units : kNumSMs;
    gemm_kernel<<<grid, kGemmThreads, kGemmSmem, static_cast<cudaStream_t>(stream)>>>(ta, tb, p);
    g_launches++;
    return check_cuda(cudaGetLastError(), "gemm launch");
}
