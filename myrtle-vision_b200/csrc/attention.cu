// attention.cu — fused softmax attention forward/backward on tcgen05 (north-star kernel (b)).
//
// Replaces Attention.forward's  (q @ k^T) * scale -> softmax -> @ v -> transpose/reshape
// (src/myrtle_vision/models/vit.py:87-97) and its autograd backward.  Scores and
// probabilities live only in TMEM / shared memory: the reference's two [B,h,N,N] fp32
// tensors per layer never reach HBM.  Head dim is fixed at 64 (models/vit.py:178).
//
// Layout: qkv fp16 [B*N, 3*D] exactly as the to_qkv GEMM writes it (q | k | v, heads contiguous,
// 64 columns each), read through one 3-D TMA map {3D, N, B} so rows past N are zero-filled
// instead of running into the next image.  Output / gradients use the same token-major layout,
// which is what the next GEMM consumes ("transpose(1,2).reshape" is free).
//
//   warp 0     TMA producer           warp 1     tcgen05.mma issuer (+ TMEM alloc)
//   warps 2-5  one thread per query row (TMEM lane): softmax / dS math, epilogue
//
// Forward:  S = Q K^T (TMEM) -> online softmax in registers -> P (fp16) to swizzled smem ->
//           O_j = P V (TMEM) -> rescale-accumulate in registers -> q_out -> fp16 store.
//           Saves L = m + log2(l) (log2 domain) per row for the backward.
// Backward (CTA = 64-key block, attn_bwd64_kernel): dV += P^T dO, dK += dS^T Q (MN-major A operands) over the
//   query blocks; dQ_i += dS K_j by fp32 red.add into a scratch buffer that dq_convert_kernel rounds into dqkv.
//   P = exp2(S*c - L), dS = P * (dP - Delta) * scale, dP = dO V^T, Delta = rowsum(dO*O).
#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {

extern int64_t g_launches;

constexpr int kAttThreads = 192;
constexpr int kTile = 16384;          // 128 rows x 128 B
constexpr int kStgPitchF = 36;        // floats per staged fp32 row chunk (32 + 4 pad: conflict-free 16 B accesses)
constexpr uint32_t kIdescPV = make_idesc(0, 0, 0, 1, 128, 64);     // A K-major, B MN-major, N=64

__device__ __forceinline__ float sat16f(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
// {lo, hi} -> packed fp16x2 with saturation to +-65504 in one F2FP
__device__ __forceinline__ uint32_t pack_h2_sat(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
// write 32 consecutive fp16 columns [c32*32, c32*32+32) of row r into a [128 x 128-col] operand
// stored as two K-major SW128 sub-tiles of 64 columns (16 KB each)
__device__ __forceinline__ void store_p_chunk(uint8_t* tile_base, int r, int c32, const uint32_t (&w)[16]) {
    uint8_t* sub = tile_base + (c32 >> 1) * kTile + r * 128;
#pragma unroll
    for (int t = 0; t < 4; t++) {
        const int chunk = ((c32 & 1) * 4 + t) ^ (r & 7);
        *reinterpret_cast<uint4*>(sub + chunk * 16) = make_uint4(w[4 * t], w[4 * t + 1], w[4 * t + 2], w[4 * t + 3]);
    }
}

struct AttnFwdDev {
    int B, H, N, D;
    float scale_log2;
    void* out; int out_dtype; int ld_out;
    FloatFmt q_out;
    float* lse;
};

__global__ void __launch_bounds__(kAttThreads, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const AttnFwdDev p) {
    // 80 KB of shared memory and 256 TMEM columns per CTA: two CTAs share an SM, so one CTA's
    // softmax (CUDA cores) overlaps the other's MMAs and TMA loads.
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; offset arithmetic keeps the shared address space
    uint8_t* sQ = smem;
    uint8_t* sK = smem + kTile;
    uint8_t* sV = smem + 2 * kTile;
    uint8_t* sP = smem + 3 * kTile;              // 2 sub-tiles of 64 keys
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 5 * kTile);
    uint64_t* q_full = bars;
    uint64_t* k_full = bars + 1;
    uint64_t* k_empty = bars + 2;
    uint64_t* v_full = bars + 3;
    uint64_t* v_empty = bars + 4;
    uint64_t* s_full = bars + 5;
    uint64_t* p_full = bars + 6;
    uint64_t* o_full = bars + 7;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
    const int nblk = (p.N + 127) / 128;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_qkv);
        mbar_init(q_full, 1);
        mbar_init(k_full, 1); mbar_init(k_empty, 1); mbar_init(v_full, 1); mbar_init(v_empty, 1);
        mbar_init(s_full, 1); mbar_init(p_full, 4); mbar_init(o_full, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<256>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tS = tmem_base, tO = tmem_base + 128;

    if (warp == 0) {
        if (lane == 0) {
            mbar_arrive_expect_tx(q_full, kTile);
            tma_load_3d(sQ, &tmap_qkv, q_full, h * 64, q0, b);
            for (int j = 0; j < nblk; j++) {
                mbar_wait(k_empty, (j & 1) ^ 1);
                mbar_arrive_expect_tx(k_full, kTile);
                tma_load_3d(sK, &tmap_qkv, k_full, p.D + h * 64, j * 128, b);
                mbar_wait(v_empty, (j & 1) ^ 1);
                mbar_arrive_expect_tx(v_full, kTile);
                tma_load_3d(sV, &tmap_qkv, v_full, 2 * p.D + h * 64, j * 128, b);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t aQ = smem_u32(sQ), aP = smem_u32(sP), aK = smem_u32(sK), aV = smem_u32(sV);
            mbar_wait(q_full, 0);
            auto issue_s = [&](int j) {
                // the last key block only multiplies the keys that exist (rounded up to 16)
                const int nk16 = (min(128, p.N - j * 128) + 15) & ~15;
                mbar_wait(k_full, j & 1);
                tc_fence_after();
                const uint32_t idesc = make_idesc(0, 0, 0, 0, 128, nk16);
#pragma unroll
                for (int k = 0; k < 4; k++)
                    umma_f16(tS, make_smem_desc_sw128(aQ + k * 32, 16, 1024),
                             make_smem_desc_sw128(aK + k * 32, 16, 1024), idesc, k > 0);
                umma_commit(s_full);
                umma_commit(k_empty);
            };
            issue_s(0);
            for (int j = 0; j < nblk; j++) {
                const int ksteps = ((min(128, p.N - j * 128) + 15) & ~15) >> 4;
                mbar_wait(v_full, j & 1);
                mbar_wait(p_full, j & 1);
                tc_fence_after();
                for (int k = 0; k < ksteps; k++)
                    umma_f16(tO, make_smem_desc_sw128(aP + (k >> 2) * kTile + (k & 3) * 32, 16, 1024),
                             make_smem_desc_sw128(aV + k * 2048, 8192, 1024), kIdescPV, k > 0);
                umma_commit(o_full);
                umma_commit(v_empty);
                if (j + 1 < nblk) issue_s(j + 1);
            }
        }
    } else {
        const int quad = warp & 3;
        const int r = quad * 32 + lane;
        const int qrow = q0 + r;
        const uint32_t lane_off = uint32_t(quad * 32) << 16;
        if (q0 + quad * 32 >= p.N) {
            // none of this warp's 32 query rows exists: only keep the barrier protocol going
            for (int j = 0; j < nblk; j++) {
                mbar_wait(s_full, j & 1);
                __syncwarp();
                if (lane == 0) mbar_arrive(p_full);
                mbar_wait(o_full, j & 1);
            }
        } else {
            float m = -INFINITY, l = 0.f;
            float o[64];
#pragma unroll
            for (int i = 0; i < 64; i++) o[i] = 0.f;
            for (int j = 0; j < nblk; j++) {
                mbar_wait(s_full, j & 1);
                tc_fence_after();
                const int kbase = j * 128;
                const int nk16 = (min(128, p.N - kbase) + 15) & ~15;
                const int nchunk = (nk16 + 31) >> 5;
                // pass 1: row max of the scaled scores
                float mx = -INFINITY;
                const bool full_blk = kbase + 128 <= p.N;       // only the last block needs key masking
                if (full_blk) {
                    // 128 live keys: the next 32 columns are in flight while the current ones are reduced
                    uint32_t sa[32], sb[32];
                    float mx1 = -INFINITY;
                    tmem_ld_32x32(tS + lane_off, sa);
                    tmem_ld_wait();
#pragma unroll
                    for (int c = 0; c < 4; c += 2) {
                        tmem_ld_32x32(tS + lane_off + (c + 1) * 32, sb);
#pragma unroll
                        for (int t = 0; t < 16; t++) {
                            mx = fmaxf(mx, __uint_as_float(sa[2 * t])); mx1 = fmaxf(mx1, __uint_as_float(sa[2 * t + 1]));
                        }
                        tmem_ld_wait();
                        if (c + 2 < 4) tmem_ld_32x32(tS + lane_off + (c + 2) * 32, sa);
#pragma unroll
                        for (int t = 0; t < 16; t++) {
                            mx = fmaxf(mx, __uint_as_float(sb[2 * t])); mx1 = fmaxf(mx1, __uint_as_float(sb[2 * t + 1]));
                        }
                        tmem_ld_wait();
                    }
                    mx = fmaxf(mx, mx1);
                } else {
#pragma unroll 1
                    for (int c = 0; c < nchunk; c++) {
                        uint32_t s[32];
                        tmem_ld_32x32(tS + lane_off + c * 32, s);
                        tmem_ld_wait();
#pragma unroll
                        for (int t = 0; t < 32; t++)
                            if (kbase + c * 32 + t < p.N) mx = fmaxf(mx, __uint_as_float(s[t]));
                    }
                }
                const float m_new = fmaxf(m, mx * p.scale_log2);
                const float alpha = ex2_fast(m - m_new);         // m = -inf on the first block -> 0
                float psum = 0.f;
                // pass 2: P = exp2(s*c - m_new) -> fp16 -> swizzled smem (A operand of P.V)
#pragma unroll 1
                for (int c = 0; c < nchunk; c++) {
                    uint32_t s[32];
                    tmem_ld_32x32(tS + lane_off + c * 32, s);
                    tmem_ld_wait();
                    uint32_t w[16];
                    if (full_blk) {
#pragma unroll
                        for (int t = 0; t < 16; t++) {
                            const float p0 = ex2_fast(fmaf(__uint_as_float(s[2 * t]), p.scale_log2, -m_new));
                            const float p1 = ex2_fast(fmaf(__uint_as_float(s[2 * t + 1]), p.scale_log2, -m_new));
                            psum += p0 + p1;
                            w[t] = pack_h2(p0, p1);
                        }
                    } else {
#pragma unroll
                        for (int t = 0; t < 16; t++) {
                            const int k0 = kbase + c * 32 + 2 * t;
                            const float p0 = k0 < p.N ? ex2_fast(fmaf(__uint_as_float(s[2 * t]), p.scale_log2, -m_new)) : 0.f;
                            const float p1 = k0 + 1 < p.N ? ex2_fast(fmaf(__uint_as_float(s[2 * t + 1]), p.scale_log2, -m_new)) : 0.f;
                            psum += p0 + p1;
                            w[t] = pack_h2(p0, p1);
                        }
                    }
                    store_p_chunk(sP, r, c, w);
                }
                l = l * alpha + psum;
                m = m_new;
                fence_proxy_async();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(p_full);
                // O_j = P V_j ; accumulate with rescale
                mbar_wait(o_full, j & 1);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    uint32_t v[32];
                    tmem_ld_32x32(tO + lane_off + c * 32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int t = 0; t < 32; t++) o[c * 32 + t] = fmaf(o[c * 32 + t], alpha, __uint_as_float(v[t]));
                }
                tc_fence_before();
            }
            if (qrow < p.N) {
                const float inv = 1.0f / l;
                const int64_t grow = int64_t(b) * p.N + qrow;
                if (p.lse != nullptr) p.lse[(int64_t(b) * p.H + h) * p.N + qrow] = m + log2f(l);
                const int mode = fq_mode(p.q_out);
#pragma unroll
                for (int i = 0; i < 64; i++) o[i] = fq_apply(o[i] * inv, mode, p.q_out);
                if (p.out_dtype == MV_F16) {
                    __half* dst = reinterpret_cast<__half*>(p.out) + grow * p.ld_out + h * 64;
#pragma unroll
                    for (int i = 0; i < 8; i++)
                        reinterpret_cast<uint4*>(dst)[i] = make_uint4(pack_h2(sat16f(o[8 * i]), sat16f(o[8 * i + 1])), pack_h2(sat16f(o[8 * i + 2]), sat16f(o[8 * i + 3])),
                                                                      pack_h2(sat16f(o[8 * i + 4]), sat16f(o[8 * i + 5])), pack_h2(sat16f(o[8 * i + 6]), sat16f(o[8 * i + 7])));
                } else {
                    float* dst = reinterpret_cast<float*>(p.out) + grow * p.ld_out + h * 64;
#pragma unroll
                    for (int i = 0; i < 16; i++)
                        reinterpret_cast<float4*>(dst)[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<256>(tmem_base); }
}

// Delta[b,h,n] = sum_d dO[bn, h*64+d] * O[bn, h*64+d]
__global__ void attn_delta_kernel(const __half* __restrict__ dO, const __half* __restrict__ O,
                                  float* __restrict__ delta, int B, int H, int N, int D) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;     // (row, head)
    if (i >= int64_t(B) * N * H) return;
    const int64_t row = i / H; const int h = int(i % H);
    const uint4* a = reinterpret_cast<const uint4*>(dO + row * D + h * 64);
    const uint4* c = reinterpret_cast<const uint4*>(O + row * D + h * 64);
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < 8; t++) {
        const uint4 x = a[t], y = c[t];
        const __half2* xh = reinterpret_cast<const __half2*>(&x);
        const __half2* yh = reinterpret_cast<const __half2*>(&y);
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const float2 fx = __half22float2(xh[u]), fy = __half22float2(yh[u]);
            s += fx.x * fy.x + fx.y * fy.y;
        }
    }
    const int b = int(row / N), n = int(row % N);
    delta[(int64_t(b) * H + h) * N + n] = s;
}

struct AttnBwdDev {
    int B, H, N, D;
    float scale_log2, scale;
    const float* lse;
    const float* delta;
    __half* dqkv; int ld_dqkv;
    float* dq_accum;          // fp32 [B*N, D]: dQ += dS K by red.add
    int* ovf;                 // overflow sink (mv_set_overflow_flag) or NULL
};

// ---------------------------------------------------------------------------------------------
// Backward, 64-key blocks: 80 KB of shared memory and 256 TMEM columns per CTA so that two CTAs
// share an SM (one CTA's exp/dS math overlaps the other's MMAs and TMA loads).  CTA = (64 keys, head,
// image); loops over 128-row query blocks; dK, dV accumulate in TMEM (lanes 0-63), dQ_i = dS K_j is
// produced per iteration into the (dead) S columns and red.add-ed into an fp32 buffer.
constexpr uint32_t kIdescTT64 = make_idesc(0, 0, 1, 1, 128, 64);

__global__ void __launch_bounds__(kAttThreads, 2)
attn_bwd64_kernel(const __grid_constant__ CUtensorMap tmap_q128, const __grid_constant__ CUtensorMap tmap_kv64,
                  const __grid_constant__ CUtensorMap tmap_do, const AttnBwdDev p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; offset arithmetic keeps the shared address space
    // order matters: the MN-major M=128 A descriptors of P / dS step one tile (LBO) past their own
    // 64-key tile for the unused upper 64 rows; that neighbour must hold finite data (dS, then Q)
    uint8_t* sP = smem;                        // [128 q][64 keys] fp16
    uint8_t* sdS = smem + kTile;
    uint8_t* sQ = smem + 2 * kTile;            // ring: Q_i
    uint8_t* sdO = smem + 3 * kTile;           // ring: dO_i
    uint8_t* sK = smem + 4 * kTile;            // resident K_j  [64 keys][64 d] (8 KB)
    uint8_t* sV = smem + 4 * kTile + 8192;     // resident V_j
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 5 * kTile);
    float* sStg = reinterpret_cast<float*>(smem + 5 * kTile + 256);      // [4 math warps][32 rows][kStgPitchF]
    uint64_t* res_full = bars;
    uint64_t* ring_full = bars + 1;            // Q_i landed
    uint64_t* ring_empty = bars + 2;           // Q_i consumed (dK MMAs done)
    uint64_t* do_full = bars + 9;              // dO_i landed / consumed (dV MMAs done): its own pair of barriers, so that the
    uint64_t* do_empty = bars + 10;            // next dO is on its way while the dK MMAs still run
    uint64_t* sdp_full = bars + 3;
    uint64_t* pds_full = bars + 4;
    uint64_t* pds_empty = bars + 5;
    uint64_t* dq_full = bars + 6;
    uint64_t* dq_done = bars + 7;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int blk0 = blockIdx.x * 64, h = blockIdx.y, b = blockIdx.z;
    const int nblk = (p.N + 127) / 128;                      // query blocks
    const int nk16 = (min(64, p.N - blk0) + 15) & ~15;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_q128); tma_prefetch_desc(&tmap_kv64); tma_prefetch_desc(&tmap_do);
        mbar_init(res_full, 1); mbar_init(ring_full, 1); mbar_init(ring_empty, 1);
        mbar_init(do_full, 1); mbar_init(do_empty, 1);
        mbar_init(sdp_full, 1); mbar_init(pds_full, 4); mbar_init(pds_empty, 1);
        mbar_init(dq_full, 1); mbar_init(dq_done, 4);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<256>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tS = tmem_base, tdP = tmem_base + 64, tdV = tmem_base + 128, tdK = tmem_base + 192;
    const uint32_t tdQ = tS;                                   // S is dead once P / dS are in smem

    if (warp == 0) {
        if (lane == 0) {
            mbar_arrive_expect_tx(res_full, 16384);
            tma_load_3d(sK, &tmap_kv64, res_full, p.D + h * 64, blk0, b);
            tma_load_3d(sV, &tmap_kv64, res_full, 2 * p.D + h * 64, blk0, b);
            for (int it = 0; it < nblk; it++) {
                mbar_wait(do_empty, (it & 1) ^ 1);
                mbar_arrive_expect_tx(do_full, kTile);
                tma_load_3d(sdO, &tmap_do, do_full, h * 64, it * 128, b);
                mbar_wait(ring_empty, (it & 1) ^ 1);
                mbar_arrive_expect_tx(ring_full, kTile);
                tma_load_3d(sQ, &tmap_q128, ring_full, h * 64, it * 128, b);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t aP = smem_u32(sP), adS = smem_u32(sdS), aQ = smem_u32(sQ), aDO = smem_u32(sdO),
                           aK = smem_u32(sK), aV = smem_u32(sV);
            const uint32_t idesc_s = make_idesc(0, 0, 0, 0, 128, nk16);
            mbar_wait(res_full, 0);
            for (int it = 0; it < nblk; it++) {
                const int nq16 = (min(128, p.N - it * 128) + 15) & ~15;
                // dP first: dO arrives first, and its TMEM columns are not the ones the previous dQ tile is still read from
                mbar_wait(do_full, it & 1);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 4; k++)
                    umma_f16(tdP, make_smem_desc_sw128(aDO + k * 32, 16, 1024), make_smem_desc_sw128(aV + k * 32, 16, 1024), idesc_s, k > 0);
                mbar_wait(ring_full, it & 1);
                if (it > 0) mbar_wait(dq_done, (it - 1) & 1);        // dQ tile (aliasing S) has been read
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < 4; k++)
                    umma_f16(tS, make_smem_desc_sw128(aQ + k * 32, 16, 1024), make_smem_desc_sw128(aK + k * 32, 16, 1024), idesc_s, k > 0);
                umma_commit(sdp_full);
                mbar_wait(pds_full, it & 1);
                tc_fence_after();
                // dQ_i contribution of this key block = dS K_j — first, with its own commit: the math warps read it out
                // and red.add it while the dV / dK MMAs below run
                for (int k = 0; k < (nk16 >> 4); k++)
                    umma_f16(tdQ, make_smem_desc_sw128(adS + k * 32, 16, 1024),
                             make_smem_desc_sw128(aK + k * 2048, 8192, 1024), kIdescPV, k > 0);
                umma_commit(dq_full);
                // dV[keys, d] += P^T dO ; dK[keys, d] += dS^T Q   (M = 128: rows 64..127 are don't-care)
                for (int k = 0; k < (nq16 >> 4); k++)
                    umma_f16(tdV, make_smem_desc_sw128(aP + k * 2048, kTile, 1024),
                             make_smem_desc_sw128(aDO + k * 2048, 8192, 1024), kIdescTT64, (it > 0 || k > 0));
                umma_commit(do_empty);
                for (int k = 0; k < (nq16 >> 4); k++)
                    umma_f16(tdK, make_smem_desc_sw128(adS + k * 2048, kTile, 1024),
                             make_smem_desc_sw128(aQ + k * 2048, 8192, 1024), kIdescTT64, (it > 0 || k > 0));
                umma_commit(ring_empty);
                umma_commit(pds_empty);
            }
        }
    } else {
        const int quad = warp & 3;
        const int r = quad * 32 + lane;
        const uint32_t lane_off = uint32_t(quad * 32) << 16;
        for (int it = 0; it < nblk; it++) {
            const int qrow = it * 128 + r;
            const bool q_ok = qrow < p.N;
            const int nq16 = (min(128, p.N - it * 128) + 15) & ~15;
            const int nchunk = (quad * 32 < nq16) ? ((nk16 + 31) >> 5) : 0;
            float L = 0.f, dl = 0.f;
            if (q_ok) {
                const int64_t si = (int64_t(b) * p.H + h) * p.N + qrow;
                L = p.lse[si]; dl = p.delta[si];
            }
            mbar_wait(sdp_full, it & 1);
            tc_fence_after();
            mbar_wait(pds_empty, (it & 1) ^ 1);
#pragma unroll 1
            for (int c = 0; c < nchunk; c++) {
                uint32_t s[32], dp[32];
                tmem_ld_32x32(tS + lane_off + c * 32, s);
                tmem_ld_32x32(tdP + lane_off + c * 32, dp);
                tmem_ld_wait();
                uint32_t wp[16], wd[16];
#pragma unroll
                for (int t = 0; t < 16; t++) {
                    float pv[2], dv[2];
#pragma unroll
                    for (int u = 0; u < 2; u++) {
                        const bool ok = q_ok && (blk0 + c * 32 + 2 * t + u < p.N);
                        const float pe = ok ? ex2_fast(fmaf(__uint_as_float(s[2 * t + u]), p.scale_log2, -L)) : 0.f;
                        pv[u] = pe;
                        dv[u] = pe * (__uint_as_float(dp[2 * t + u]) - dl) * p.scale;
                    }
                    wp[t] = pack_h2(pv[0], pv[1]);
                    wd[t] = pack_h2_sat(dv[0], dv[1]);
                }
                store_p_chunk(sdS, r, c, wd);
                store_p_chunk(sP, r, c, wp);
            }
            fence_proxy_async();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(pds_full);
            // dQ contribution: TMEM -> fp32 red.add
            mbar_wait(dq_full, it & 1);
            tc_fence_after();
            if (nchunk > 0) {
                // One TMEM lane = one query row per thread: reduced straight from registers, every red.add of a
                // warp would touch 32 different lines.  The rows go through the warp's staging tile so that
                // eight lanes add one row's 128 contiguous bytes: 4 full lines per instruction.
                const int qrow0 = qrow - lane;                              // first row of this warp
                float* dst0 = p.dq_accum + (int64_t(b) * p.N + qrow0) * p.D + h * 64;
                float* stg = sStg + quad * (32 * kStgPitchF);
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    uint32_t v[32];
                    tmem_ld_32x32(tdQ + lane_off + c * 32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; i++)
                        *reinterpret_cast<float4*>(stg + lane * kStgPitchF + 4 * i) =
                            make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                        __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const int row = i * 4 + (lane >> 3), chunk = lane & 7;
                        const float4 w = *reinterpret_cast<const float4*>(stg + row * kStgPitchF + 4 * chunk);
                        if (qrow0 + row < p.N)
                            atomicAdd(reinterpret_cast<float4*>(dst0 + int64_t(row) * p.D + c * 32) + chunk, w);
                    }
                    __syncwarp();
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(dq_done);
        }
        mbar_wait(pds_empty, (nblk - 1) & 1);
        tc_fence_after();
        const int key = blk0 + r;
        if (quad < 2) {                        // TMEM lanes 0..63 hold this CTA's 64 keys
            for (int a = 0; a < 2; a++) {
                uint32_t v[32];
                const int col = (a == 0 ? 2 : 1) * p.D + h * 64;       // dV | dK
                __half* dst = p.dqkv + (int64_t(b) * p.N + key) * p.ld_dqkv + col;
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    tmem_ld_32x32((a == 0 ? tdV : tdK) + lane_off + c * 32, v);
                    tmem_ld_wait();
                    if (key < p.N) {
                        float amax = 0.f;
#pragma unroll
                        for (int i = 0; i < 32; i++) amax = fmaxf(amax, fabsf(__uint_as_float(v[i])));
                        raise_overflow(p.ovf, amax);
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            reinterpret_cast<uint4*>(dst + c * 32)[i] =
                                make_uint4(pack_h2(sat16f(__uint_as_float(v[8 * i])), sat16f(__uint_as_float(v[8 * i + 1]))),
                                           pack_h2(sat16f(__uint_as_float(v[8 * i + 2])), sat16f(__uint_as_float(v[8 * i + 3]))),
                                           pack_h2(sat16f(__uint_as_float(v[8 * i + 4])), sat16f(__uint_as_float(v[8 * i + 5]))),
                                           pack_h2(sat16f(__uint_as_float(v[8 * i + 6])), sat16f(__uint_as_float(v[8 * i + 7]))));
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<256>(tmem_base); }
}

constexpr int kAttnBwd64Smem = 5 * kTile + 1024 + 256 + 4 * 32 * kStgPitchF * 4;

// dq fp32 [rows, D] -> fp16 into the q columns of dqkv [rows, ld]
__global__ void __launch_bounds__(256)
dq_convert_kernel(const float* __restrict__ dq, __half* __restrict__ dqkv, int64_t rows, int D, int ld, int* __restrict__ ovf) {
    const int vec_per_row = D >> 2;
    const int64_t total = rows * vec_per_row;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int64_t row = i / vec_per_row;
        const int c = int(i % vec_per_row);
        const float4 v = __ldcs(reinterpret_cast<const float4*>(dq) + i);
        raise_overflow(ovf, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        reinterpret_cast<uint2*>(dqkv + row * ld)[c] =
            make_uint2(pack_h2(sat16f(v.x), sat16f(v.y)), pack_h2(sat16f(v.z), sat16f(v.w)));
    }
}

constexpr int kAttnFwdSmem = 5 * kTile + 1024 + 256;

}  // namespace mv

using namespace mv;

extern "C" int mv_attention_sn_supported(int N);
int mv_attention_fwd_sn(const void* qkv, void* out, int out_dtype, float* lse, int B, int H, int N,
                        float scale, int q_out_exp, int q_out_man, void* stream);
int mv_attention_bwd_sn(const void* qkv, const void* o, const void* d_o, const float* lse, float* delta,
                        void* dqkv, float* dbias, int B, int H, int N, float scale, void* stream);

extern "C" int mv_attention_fwd(const void* qkv, void* out, int out_dtype, float* lse, int B, int H, int N,
                                float scale, int q_out_exp, int q_out_man, void* stream) {
    MV_CHECK(B > 0 && H > 0 && N > 0 && qkv && out, "mv_attention_fwd: bad arguments");
    MV_CHECK(out_dtype == MV_F16 || out_dtype == MV_F32, "mv_attention_fwd: bad output container");
    if (mv_attention_sn_supported(N))
        return mv_attention_fwd_sn(qkv, out, out_dtype, lse, B, H, N, scale, q_out_exp, q_out_man, stream);
    const int D = H * 64;
    static bool attr_done = false;
    if (!attr_done) {
        MV_CUDA(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kAttnFwdSmem));
        attr_done = true;
    }
    CUtensorMap tm;
    if (make_tmap_3d(&tm, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 128, 1)) return 1;
    AttnFwdDev p;
    p.B = B; p.H = H; p.N = N; p.D = D;
    p.scale_log2 = scale * 1.4426950408889634f;
    p.out = out; p.out_dtype = out_dtype; p.ld_out = D;
    p.q_out = FloatFmt{q_out_exp, q_out_man};
    p.lse = lse;
    dim3 grid((N + 127) / 128, H, B);
    attn_fwd_kernel<<<grid, kAttThreads, kAttnFwdSmem, static_cast<cudaStream_t>(stream)>>>(tm, p);
    g_launches++;
    return check_cuda(cudaGetLastError(), "attention fwd launch");
}

extern "C" int mv_attention_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, float* delta,
                                float* dq_accum, void* dqkv, float* dbias, int B, int H, int N, float scale,
                                void* stream) {
    MV_CHECK(B > 0 && H > 0 && N > 0 && qkv && o && d_o && lse && delta && dqkv, "mv_attention_bwd: bad arguments");
    MV_CHECK((reinterpret_cast<uintptr_t>(dbias) & 15) == 0, "mv_attention_bwd: dbias must be 16-byte aligned");
    if (N <= 272)
        return mv_attention_bwd_sn(qkv, o, d_o, lse, delta, dqkv, dbias, B, H, N, scale, stream);
    MV_CHECK(dq_accum != nullptr, "mv_attention_bwd: N = %d > 272 needs dq_accum (fp32 [B*N, H*64] scratch)", N);
    const int D = H * 64;
    static bool attr_done = false;
    if (!attr_done) {
        MV_CUDA(cudaFuncSetAttribute(attn_bwd64_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kAttnBwd64Smem));
        attr_done = true;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUtensorMap tq, td;
    if (make_tmap_3d(&tq, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 128, 1)) return 1;
    if (make_tmap_3d(&td, d_o, MV_F16, D, N, B, D, uint64_t(N) * D, 64, 128, 1)) return 1;
    const int64_t nrh = int64_t(B) * N * H;
    attn_delta_kernel<<<unsigned((nrh + 255) / 256), 256, 0, st>>>((const __half*)d_o, (const __half*)o, delta, B, H, N, D);
    g_launches++;
    AttnBwdDev p;
    p.B = B; p.H = H; p.N = N; p.D = D;
    p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
    p.lse = lse; p.delta = delta;
    p.dqkv = reinterpret_cast<__half*>(dqkv); p.ld_dqkv = 3 * D;
    p.dq_accum = dq_accum;
    p.ovf = g_overflow;
    // dK, dV per key block and dQ accumulated across key blocks with fp32 red.add
    const int64_t n = int64_t(B) * N * D;
    MV_CUDA(cudaMemsetAsync(dq_accum, 0, sizeof(float) * n, st));
    CUtensorMap tk64;
    if (make_tmap_3d(&tk64, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 64, 1)) return 1;
    dim3 grid64((N + 63) / 64, H, B);
    attn_bwd64_kernel<<<grid64, kAttThreads, kAttnBwd64Smem, st>>>(tq, tk64, td, p);
    g_launches++;
    int64_t blocks = (n / 4 + 255) / 256;
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    dq_convert_kernel<<<int(blocks), 256, 0, st>>>(dq_accum, reinterpret_cast<__half*>(dqkv), int64_t(B) * N, D, 3 * D, g_overflow);
    g_launches++;
    if (check_cuda(cudaGetLastError(), "attention bwd launch")) return 1;
    // long sequences: the bias gradient is a separate pass over dqkv (the short-sequence kernel fuses it)
    if (dbias != nullptr) return mv_colsum(dqkv, MV_F16, 3 * D, B * N, 3 * D, dbias, stream);
    return 0;
}
