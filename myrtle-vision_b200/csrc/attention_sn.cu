// attention_sn.cu — softmax attention for SHORT sequences (N <= 272 keys, head dim 64): the ViT
// classification / segmentation shapes (256x256 images, patch 16 -> N = 257).
//
// Same operator as attention.cu (Attention.forward's (q @ k^T) * scale -> softmax -> @ v,
// src/myrtle_vision/models/vit.py:87-97, and its autograd backward), different schedule:
//   * one persistent CTA per SM walks (image, head) pairs; the pair's whole K and V (<= 272 x 64 fp16
//     each) are resident in shared memory and double-buffered across pairs, so the next pair's loads
//     overlap this pair's math;
//   * the full score row of a 128-query tile fits TMEM (<= 256 fp32 columns): plain two-pass softmax,
//     no online rescaling; P is written back over the consumed S columns as the fp16 TMEM A operand
//     of P.V (never touches shared memory) and O lands in the same 256-column region, so TWO query
//     tiles are in flight per SM — one group of 4 math warps (one thread per query row) each — and one
//     tile's MMAs run under the other's softmax;
//   * N = 257 = 2 x 128 + 1 = 16 x 16 + 1: neither the odd query row nor the odd key is padded up to a
//     tensor-core tile.  Tail query rows (N mod 128 <= kSnTailMax) are computed by SIMT warps from the
//     K / V already in shared memory, concurrently with the tiles; keys past the last multiple of 16
//     (<= kSnExtraMax) are folded in by the math threads (one 64-element dot product per row).
#include "common.cuh"
#include "quant_dev.cuh"
#include "../../include/mv_b200.h"

namespace mv {

extern int64_t g_launches;

constexpr int kSnMaxKeys = 272;                 // padded keys (multiple of 16) that fit the TMEM plan
constexpr int kSnTailMax = 2;                   // tail query rows (N mod 128) handled by the SIMT warp
constexpr int kSnKVBytes = kSnMaxKeys * 128;    // one K or V stage: 272 rows x 128 B
constexpr int kSnTile = 16384;                  // 128 rows x 128 B
constexpr int kSnStgPitch = 80;                 // bytes per staged row (64 B + pad: conflict-free 16 B stores)
constexpr int kSnExtraMax = 2;                  // keys beyond the last multiple of 16 folded in on the CUDA cores
constexpr int kSnMathWarps = 8;                 // two groups of four: one thread per query row
constexpr int kSnTailWarps = 2;
constexpr int kSnFwdThreads = 32 * (2 + kSnMathWarps + kSnTailWarps);   // producer, MMA, math, tail

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// warp-level MMA (m16n8k16, fp16 operands, fp32 accumulators) and its fragment loads: used where the problem is a few
// rows or columns wide (the odd keys of the backward), far below a tcgen05 tile
__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(smem_row)));
}
__device__ __forceinline__ void ldmatrix_x2_trans(uint32_t& r0, uint32_t& r1, const void* smem_row) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];"
                 : "=r"(r0), "=r"(r1) : "r"(smem_u32(smem_row)));
}
// non-blocking: has the phase with this parity completed?
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
__device__ __forceinline__ uint32_t pack_h2_rn(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_h2_satf(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}

// Debug timeline (tools/trace_attn_bwd.py): when a trace buffer is registered, CTA 0 stamps clock64() at
// the hand-offs between the MMA issuer and the math groups.  Record = {event, index, clock}.
static unsigned long long* g_sn_trace = nullptr;
extern "C" int mv_debug_set_attn_trace(void* dev_buf) { g_sn_trace = static_cast<unsigned long long*>(dev_buf); return 0; }
#ifndef MV_SN_TRACE
#define SN_TRACE(cond, region, ev, idx) do { } while (0)
#else
#define SN_TRACE(cond, region, ev, idx)                                                        \
    do {                                                                                       \
        if (p.trace != nullptr && blockIdx.x == 0 && (cond)) {                                 \
            unsigned long long* t_ = p.trace + (region) * 3072 + 3 * (trace_n++ % 1024);       \
            t_[0] = (ev); t_[1] = (unsigned long long)(idx); t_[2] = clock64();                \
        }                                                                                      \
    } while (0)
#endif

// Accumulator rows leave TMEM one row per thread; written like that, every 16-byte store instruction of a
// warp touches 32 different lines and the LSU serialises them (3000+ cycles per epilogue, measured with
// the clock64 timeline).  Each warp parks half a row per lane (32 fp16) in its private staging tile and
// writes it back with four lanes per row: 8 rows x 64 contiguous bytes per store instruction.
// v0 / v1: columns 0..31 / 32..63 of this lane's row (fp32 bits).  dst0: row 0 of the warp's 32 rows.
// kCS: also accumulate the column sums of the stored (fp16-rounded) rows — the fused bias gradient — into the
// lane's registers: in the write-back phase lane l always owns columns half * 32 + (l & 3) * 8 .. + 7, so
// acc[half][k] simply grows over every store of the kernel and is reduced over the 8 lanes that share a column
// chunk only when it is flushed (sn_flush_colsum).  (Reducing per store — shuffles plus global or shared
// atomics — was measured at +34 / +65 us per launch.)
__device__ __forceinline__ void sn_red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d)
                 : "memory");
}
template <bool kCS>
__device__ __forceinline__ void sn_store_rows(uint8_t* stg, const uint32_t (&v0)[32], const uint32_t (&v1)[32],
                                              __half* dst0, int64_t ld, int nvalid, int lane, float (&acc)[2][8],
                                              float& amax) {
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const uint32_t (&v)[32] = half == 0 ? v0 : v1;
#pragma unroll
        for (int i = 0; i < 32; i += 2)
            amax = fmaxf(amax, fmaxf(fabsf(__uint_as_float(v[i])), fabsf(__uint_as_float(v[i + 1]))));
#pragma unroll
        for (int i = 0; i < 4; i++)
            *reinterpret_cast<uint4*>(stg + lane * kSnStgPitch + i * 16) = make_uint4(
                pack_h2_satf(__uint_as_float(v[8 * i]), __uint_as_float(v[8 * i + 1])),
                pack_h2_satf(__uint_as_float(v[8 * i + 2]), __uint_as_float(v[8 * i + 3])),
                pack_h2_satf(__uint_as_float(v[8 * i + 4]), __uint_as_float(v[8 * i + 5])),
                pack_h2_satf(__uint_as_float(v[8 * i + 6]), __uint_as_float(v[8 * i + 7])));
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 4; it++) {
            const int row = it * 8 + (lane >> 2), chunk = lane & 3;
            const uint4 w = *reinterpret_cast<const uint4*>(stg + row * kSnStgPitch + chunk * 16);
            if (row < nvalid) {
                *reinterpret_cast<uint4*>(dst0 + row * ld + half * 32 + chunk * 8) = w;
                if (kCS) {
                    const __half2* hp = reinterpret_cast<const __half2*>(&w);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const float2 f = __half22float2(hp[k]);
                        acc[half][2 * k] += f.x; acc[half][2 * k + 1] += f.y;
                    }
                }
            }
        }
        __syncwarp();
    }
}
// dst: fp32 [64] in global memory, += the warp's accumulated column sums; the accumulators restart from zero
__device__ __forceinline__ void sn_flush_colsum(float (&acc)[2][8], float* dst, int lane) {
#pragma unroll
    for (int half = 0; half < 2; half++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            float c = acc[half][k];
            c += __shfl_xor_sync(0xffffffffu, c, 4);
            c += __shfl_xor_sync(0xffffffffu, c, 8);
            c += __shfl_xor_sync(0xffffffffu, c, 16);
            acc[half][k] = c;
        }
        if (lane < 4) {
            sn_red_add_v4(dst + half * 32 + lane * 8, acc[half][0], acc[half][1], acc[half][2], acc[half][3]);
            sn_red_add_v4(dst + half * 32 + lane * 8 + 4, acc[half][4], acc[half][5], acc[half][6], acc[half][7]);
        }
#pragma unroll
        for (int k = 0; k < 8; k++) acc[half][k] = 0.f;
    }
}

struct SnFwdDev {
    unsigned long long* trace;
    int B, H, N, D;
    int Nk;                     // keys multiplied on the tensor cores (multiple of 16, <= 256)
    int n_extra;                // keys [Nk, N) (at most kSnExtraMax) folded in by the math threads (SIMT)
    int Nld;                    // key rows to stage in shared memory: Nk + 16 if n_extra else Nk
    int n_tiles;                // 128-row tensor-core query tiles per (image, head)
    int n_tail;                 // query rows [128 * n_tiles, N) computed by the SIMT warps
    float scale_log2;
    const __half* qkv;          // for the tail warps' q row
    void* out; int out_dtype; int ld_out;
    FloatFmt q_out;
    float* lse;
};

// K / V loads of one (image, head): 128-row boxes, then 16-row boxes for the remainder
__device__ __forceinline__ void sn_load_kv(uint8_t* dst, const CUtensorMap* m128, const CUtensorMap* m16,
                                           uint64_t* bar, int col, int b, int rows) {
    int r = 0;
    for (; r + 128 <= rows; r += 128) tma_load_3d(dst + r * 128, m128, bar, col, r, b);
    for (; r < rows; r += 16) tma_load_3d(dst + r * 128, m16, bar, col, r, b);
}

// dot product of two 64-element fp16 rows held in 128-byte-swizzled tiles (row index selects the XOR)
// (rolled: it runs once per row and tile, and the forward kernel's code must stay inside the instruction cache)
__device__ __forceinline__ float sn_dot64(const uint8_t* tile_a, int ra, const uint8_t* tile_b, int rb) {
    float acc = 0.f;
#pragma unroll 2
    for (int c = 0; c < 8; c++) {
        const uint4 wa = *reinterpret_cast<const uint4*>(tile_a + ra * 128 + ((c ^ (ra & 7)) << 4));
        const uint4 wb = *reinterpret_cast<const uint4*>(tile_b + rb * 128 + ((c ^ (rb & 7)) << 4));
        const __half2* ha = reinterpret_cast<const __half2*>(&wa);
        const __half2* hb = reinterpret_cast<const __half2*>(&wb);
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const float2 fa = __half22float2(ha[u]), fb = __half22float2(hb[u]);
            acc = fmaf(fa.x, fb.x, acc);
            acc = fmaf(fa.y, fb.y, acc);
        }
    }
    return acc;
}

// ---- SIMT attention row (tail rows): one warp, K / V from the resident swizzled shared-memory tiles.
// lane l owns output dims 2l, 2l+1.  scratch: 64 floats (q) + kSnMaxKeys floats (p).
__device__ __forceinline__ void sn_tail_row_fwd(const SnFwdDev& p, const uint8_t* sK, const uint8_t* sV,
                                                float* scratch, int b, int h, int row, int lane) {
    float* sq = scratch;
    float* sp = scratch + 64;
    const __half* qrow = p.qkv + (int64_t(b) * p.N + row) * (3 * p.D) + h * 64;
    {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(qrow + 2 * lane));
        sq[2 * lane] = f.x; sq[2 * lane + 1] = f.y;
    }
    __syncwarp();
    // rolled loops, scores parked in the scratch row: this runs for one row per (image, head) on its own warps, and
    // unrolled over nine key groups it was a quarter of the kernel's 120 KB of code (no-instruction stalls: 17 %)
    constexpr int kMaxPerLane = (kSnMaxKeys + 31) / 32;
    float mx = -INFINITY;
#pragma unroll 1
    for (int i = 0; i < kMaxPerLane; i++) {
        const int j = lane + 32 * i;
        float acc = -INFINITY;
        if (j < p.N) {
            acc = 0.f;
            const uint8_t* krow = sK + j * 128;
#pragma unroll 2
            for (int c = 0; c < 8; c++) {
                const uint4 w = *reinterpret_cast<const uint4*>(krow + ((c ^ (j & 7)) << 4));
                const __half2* hh = reinterpret_cast<const __half2*>(&w);
                const float4 qa = *reinterpret_cast<const float4*>(sq + 8 * c);
                const float4 qb = *reinterpret_cast<const float4*>(sq + 8 * c + 4);
                const float2 k0 = __half22float2(hh[0]), k1 = __half22float2(hh[1]);
                const float2 k2 = __half22float2(hh[2]), k3 = __half22float2(hh[3]);
                acc = fmaf(qa.x, k0.x, acc); acc = fmaf(qa.y, k0.y, acc);
                acc = fmaf(qa.z, k1.x, acc); acc = fmaf(qa.w, k1.y, acc);
                acc = fmaf(qb.x, k2.x, acc); acc = fmaf(qb.y, k2.y, acc);
                acc = fmaf(qb.z, k3.x, acc); acc = fmaf(qb.w, k3.y, acc);
            }
        }
        if (j < p.Nld) sp[j] = acc;
        mx = fmaxf(mx, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float m = mx * p.scale_log2;
    float sum = 0.f;
#pragma unroll 1
    for (int i = 0; i < kMaxPerLane; i++) {
        const int j = lane + 32 * i;
        const float e = j < p.N ? ex2_fast(fmaf(sp[j], p.scale_log2, -m)) : 0.f;       // (this lane wrote sp[j] itself)
        sum += e;
        if (j < p.Nld) sp[j] = e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    __syncwarp();
    // o[2l], o[2l+1] = sum_j p_j V[j][2l..2l+1]; V row j: 16-byte chunk (l >> 2) sits at position (l >> 2) ^ (j & 7)
    float o0 = 0.f, o1 = 0.f;
    const int cl = lane >> 2, wi = (lane & 3) * 4;
#pragma unroll 1
    for (int j0 = 0; j0 < p.Nld; j0 += 8) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int j = j0 + u;
            const float pj = sp[j];
            const float2 v = __half22float2(*reinterpret_cast<const __half2*>(sV + j * 128 + ((cl ^ u) << 4) + wi));
            o0 = fmaf(pj, v.x, o0); o1 = fmaf(pj, v.y, o1);
        }
    }
    const float inv = 1.0f / sum;
    const int mode = fq_mode(p.q_out);
    o0 = fq_apply(o0 * inv, mode, p.q_out);
    o1 = fq_apply(o1 * inv, mode, p.q_out);
    const int64_t grow = int64_t(b) * p.N + row;
    if (p.out_dtype == MV_F16)
        *reinterpret_cast<uint32_t*>(reinterpret_cast<__half*>(p.out) + grow * p.ld_out + h * 64 + 2 * lane) = pack_h2_satf(o0, o1);
    else
        *reinterpret_cast<float2*>(reinterpret_cast<float*>(p.out) + grow * p.ld_out + h * 64 + 2 * lane) = make_float2(o0, o1);
    if (lane == 0 && p.lse != nullptr) p.lse[(int64_t(b) * p.H + h) * p.N + row] = m + log2f(sum);
    __syncwarp();
}

// One TMEM lane = one output row per thread: stored directly, each 16-byte store instruction of a warp
// touches 32 different lines and the LSU serialises them.  Each warp parks half a row per lane (32 fp16)
// in its private staging tile and writes it back with four lanes per row — 8 rows x 64 contiguous bytes
// per store instruction.  o: this lane's 64 output values; dst0: row 0 of the warp's 32 rows.
__device__ __forceinline__ void sn_store_rows_f(uint8_t* stg, const float (&o)[64], __half* dst0, int64_t ld,
                                                int nvalid, int lane) {
#pragma unroll
    for (int half = 0; half < 2; half++) {
#pragma unroll
        for (int i = 0; i < 4; i++)
            *reinterpret_cast<uint4*>(stg + lane * kSnStgPitch + i * 16) = make_uint4(
                pack_h2_satf(o[32 * half + 8 * i], o[32 * half + 8 * i + 1]),
                pack_h2_satf(o[32 * half + 8 * i + 2], o[32 * half + 8 * i + 3]),
                pack_h2_satf(o[32 * half + 8 * i + 4], o[32 * half + 8 * i + 5]),
                pack_h2_satf(o[32 * half + 8 * i + 6], o[32 * half + 8 * i + 7]));
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 4; it++) {
            const int row = it * 8 + (lane >> 2), chunk = lane & 3;
            const uint4 w = *reinterpret_cast<const uint4*>(stg + row * kSnStgPitch + chunk * 16);
            if (row < nvalid) *reinterpret_cast<uint4*>(dst0 + row * ld + half * 32 + chunk * 8) = w;
        }
        __syncwarp();
    }
}

// Same store, with the softmax normalisation and the (5,10) output quantiser folded into the packing:
// four values per range test, cvt.rz on the half-ulp-biased word (quant_dev.cuh: fq_half4_pack).
__device__ __forceinline__ void sn_store_rows_q16(uint8_t* stg, const float (&o)[64], float inv, __half* dst0,
                                                  int64_t ld, int nvalid, int lane) {
#pragma unroll
    for (int half = 0; half < 2; half++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const float* v = &o[32 * half + 8 * i];
            const uint2 lo = fq_half4_pack(v[0] * inv, v[1] * inv, v[2] * inv, v[3] * inv);
            const uint2 hi = fq_half4_pack(v[4] * inv, v[5] * inv, v[6] * inv, v[7] * inv);
            *reinterpret_cast<uint4*>(stg + lane * kSnStgPitch + i * 16) = make_uint4(lo.x, lo.y, hi.x, hi.y);
        }
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 4; it++) {
            const int row = it * 8 + (lane >> 2), chunk = lane & 3;
            const uint4 w = *reinterpret_cast<const uint4*>(stg + row * kSnStgPitch + chunk * 16);
            if (row < nvalid) *reinterpret_cast<uint4*>(dst0 + row * ld + half * 32 + chunk * 8) = w;
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kSnFwdThreads, 1)
attn_fwd_sn_kernel(const __grid_constant__ CUtensorMap tmap128, const __grid_constant__ CUtensorMap tmap16,
                   const __grid_constant__ SnFwdDev p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; offset arithmetic keeps the shared address space
    uint8_t* sK = smem;                                   // [2 stages][272 x 128 B]
    uint8_t* sV = smem + 2 * kSnKVBytes;
    uint8_t* sQ = smem + 4 * kSnKVBytes;                  // ring of 2 query tiles
    float* s_tail = reinterpret_cast<float*>(smem + 4 * kSnKVBytes + 2 * kSnTile);   // [2 warps][64 + kSnMaxKeys]
    uint8_t* sStg = reinterpret_cast<uint8_t*>(s_tail + kSnTailWarps * (64 + kSnMaxKeys));   // [8 math warps][32 rows][kSnStgPitch]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sStg + kSnMathWarps * 32 * kSnStgPitch);
    uint64_t* k_full = bars;            // [2]
    uint64_t* k_empty = bars + 2;       // [2]
    uint64_t* v_full = bars + 4;        // [2]
    uint64_t* v_empty = bars + 6;       // [2]
    uint64_t* q_full = bars + 8;        // [2]
    uint64_t* q_empty = bars + 10;      // [2]
    uint64_t* s_full = bars + 12;       // [2]  per math group
    uint64_t* p_full = bars + 14;       // [2]
    uint64_t* o_full = bars + 16;       // [2]
    uint64_t* o_empty = bars + 18;      // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    [[maybe_unused]] int trace_n = 0;
    const int n_bh = p.B * p.H;
    const int n_local = blockIdx.x < n_bh ? (n_bh - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;   // pairs of this CTA
    const int total_tiles = n_local * p.n_tiles;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap128); tma_prefetch_desc(&tmap16);
        for (int s = 0; s < 2; s++) {
            // a K / V stage is released by the MMA commit, the tail warp and the 4 math warps of every query tile
            mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 2 + 4 * p.n_tiles);
            mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 2 + 4 * p.n_tiles);
            mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 1 + 4);       // MMA commit + the tile's 4 math warps
            mbar_init(&s_full[s], 1); mbar_init(&p_full[s], 4); mbar_init(&o_full[s], 1); mbar_init(&o_empty[s], 4);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // TMEM, per math group (256 columns): S fp32 [0, Nk) -> P fp16 in place [0, Nk/2) -> O fp32 [128, 192)

    if (warp == 0) {
        // ================================ TMA producer ================================
        if (lane == 0) {
            int qi = 0;
            for (int n = 0; n < n_local; n++) {
                const int bh = blockIdx.x + n * gridDim.x;
                const int b = bh / p.H, h = bh % p.H, s = n & 1;
                const uint32_t ph = (n >> 1) & 1;
                mbar_wait_relaxed(&k_empty[s], ph ^ 1);
                mbar_arrive_expect_tx(&k_full[s], p.Nld * 128);
                sn_load_kv(sK + s * kSnKVBytes, &tmap128, &tmap16, &k_full[s], p.D + h * 64, b, p.Nld);
                for (int t = 0; t < p.n_tiles; t++, qi++) {
                    const int qs = qi & 1;
                    mbar_wait_relaxed(&q_empty[qs], ((qi >> 1) & 1) ^ 1);
                    mbar_arrive_expect_tx(&q_full[qs], kSnTile);
                    tma_load_3d(sQ + qs * kSnTile, &tmap128, &q_full[qs], h * 64, t * 128, b);
                    if (t == 0) {                                           // V is first needed after the first softmax
                        mbar_wait_relaxed(&v_empty[s], ph ^ 1);
                        mbar_arrive_expect_tx(&v_full[s], p.Nld * 128);
                        sn_load_kv(sV + s * kSnKVBytes, &tmap128, &tmap16, &v_full[s], 2 * p.D + h * 64, b, p.Nld);
                    }
                }
                if (p.n_tiles == 0) {
                    mbar_wait_relaxed(&v_empty[s], ph ^ 1);
                    mbar_arrive_expect_tx(&v_full[s], p.Nld * 128);
                    sn_load_kv(sV + s * kSnKVBytes, &tmap128, &tmap16, &v_full[s], 2 * p.D + h * 64, b, p.Nld);
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ================================
        if (lane == 0) {
            const uint32_t idesc_s = make_idesc(0, 0, 0, 0, 128, p.Nk);
            const uint32_t idesc_pv = make_idesc(0, 0, 0, 1, 128, 64);     // A (TMEM) K-major, B = V MN-major
            const int ksteps = p.Nk >> 4;
            // This lane sits between the two math groups on every tile: walk the schedule with counters (no
            // divisions) and build every descriptor as a base plus a small offset.
            const uint64_t dQ0 = make_smem_desc_sw128(smem_u32(sQ), 16, 1024);
            const uint64_t dK0 = make_smem_desc_sw128(smem_u32(sK), 16, 1024);
            const uint64_t dV0 = make_smem_desc_sw128(smem_u32(sV), 8192, 1024);
            constexpr uint64_t kQOff = kSnTile >> 4, kKVOff = kSnKVBytes >> 4;
            int gs = 0, ns = 0, ts = 0;                                      // S schedule: tile, pair, tile in pair
            auto issue_s = [&]() {
                const int g = gs, n = ns, t = ts, s = n & 1, grp = g & 1;
                const uint32_t tS = tmem_base + grp * 256;
                if (g >= 2) mbar_wait(&o_empty[grp], ((g - 2) >> 1) & 1);   // O(g-2) (inside this region) has been read
                if (t == 0) mbar_wait(&k_full[s], (n >> 1) & 1);
                mbar_wait(&q_full[g & 1], (g >> 1) & 1);
                tc_fence_after();
                const uint64_t dq = dQ0 + (g & 1) * kQOff, dk = dK0 + s * kKVOff;
#pragma unroll
                for (int k = 0; k < 4; k++) umma_f16(tS, dq + 2 * k, dk + 2 * k, idesc_s, k > 0);
                umma_commit(&s_full[grp]);
                SN_TRACE(true, 0, 1, g);                                    // S MMAs issued
                umma_commit(&q_empty[g & 1]);
                if (t == p.n_tiles - 1) umma_commit(&k_empty[s]);
                gs++;
                if (++ts == p.n_tiles) { ts = 0; ns++; }
            };
            if (p.n_tiles == 0) {
                for (int n = 0; n < n_local; n++) {
                    mbar_wait(&k_full[n & 1], (n >> 1) & 1); mbar_arrive(&k_empty[n & 1]);
                    mbar_wait(&v_full[n & 1], (n >> 1) & 1); mbar_arrive(&v_empty[n & 1]);
                }
            } else {
                if (total_tiles > 0) issue_s();
                if (total_tiles > 1) issue_s();
                int n = 0, t = 0;
                for (int g = 0; g < total_tiles; g++) {
                    const int s = n & 1, grp = g & 1;
                    const uint32_t tP = tmem_base + grp * 256, tO = tP + 128;
                    if (t == 0) mbar_wait(&v_full[s], (n >> 1) & 1);
                    SN_TRACE(true, 0, 2, g);
                    mbar_wait(&p_full[grp], (g >> 1) & 1);
                    SN_TRACE(true, 0, 3, g);                                // softmax of tile g done (seen by issuer)
                    tc_fence_after();
                    uint64_t dv = dV0 + s * kKVOff;
                    uint32_t ta = tP;
                    umma_f16_ts(tO, ta, dv, idesc_pv, 0u);
                    for (int k = 1; k < ksteps; k++) {
                        dv += 128; ta += 8;                                  // 16 keys further: 2048 B of V, 8 columns of P
                        umma_f16_ts(tO, ta, dv, idesc_pv, 1u);
                    }
                    umma_commit(&o_full[grp]);
                    SN_TRACE(true, 0, 4, g);                                // PV MMAs issued
                    if (t == p.n_tiles - 1) umma_commit(&v_empty[s]);
                    if (g + 2 < total_tiles) issue_s();
                    if (++t == p.n_tiles) { t = 0; n++; }
                }
            }
        }
    } else if (warp < 2 + kSnMathWarps) {
        // ================================ softmax / epilogue: two groups of 4 warps ================================
        // group = tile parity; one thread per query row (TMEM lane), all keys of the row
        const int quad = warp & 3;
        const int grp = (warp - 2) >> 2;
        const int rl = quad * 32 + lane;
        const uint32_t tS = tmem_base + grp * 256 + (uint32_t(quad * 32) << 16);
        const uint32_t tO = tS + 128;
        const int mode = fq_mode(p.q_out);
        for (int g = grp; g < total_tiles; g += 2) {
            const int n = g / p.n_tiles, t = g % p.n_tiles, s = n & 1;
            const int bh = blockIdx.x + n * gridDim.x;
            const int b = bh / p.H, h = bh % p.H;
            const int row = t * 128 + rl;
            const uint8_t* cK = sK + s * kSnKVBytes;
            const uint8_t* cV = sV + s * kSnKVBytes;
            // the loads themselves must be observed by this thread before it reads the tiles
            mbar_wait(&k_full[s], (n >> 1) & 1);
            mbar_wait(&q_full[g & 1], (g >> 1) & 1);
            // keys beyond the tensor-core part: s = q . k on the CUDA cores
            float sx[kSnExtraMax];
#pragma unroll
            for (int e = 0; e < kSnExtraMax; e++)
                sx[e] = e < p.n_extra ? sn_dot64(sQ + (g & 1) * kSnTile, rl, cK, p.Nk + e) : -INFINITY;
            __syncwarp();
            if (lane == 0) { mbar_arrive(&q_empty[g & 1]); mbar_arrive(&k_empty[s]); }
            SN_TRACE(quad == 0 && lane == 0, 1 + grp, 5, g);
            mbar_wait(&s_full[grp], (g >> 1) & 1);
            SN_TRACE(quad == 0 && lane == 0, 1 + grp, 6, g);                 // S ready
            tc_fence_after();
            // pass 1: row max
            float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
            for (int e = 0; e < kSnExtraMax; e++) mx0 = fmaxf(mx0, sx[e]);
            // whole 64-key steps inside [0, N): the next 32 columns are in flight while the current ones are reduced
            int k_pipe = 0;
            if (p.Nk >= 64 && p.Nk <= p.N) {
                const int kend = p.Nk & ~63;
                uint32_t va[32], vb[32];
                tmem_ld_32x32(tS, va);
                tmem_ld_wait();
#pragma unroll 1
                for (int k0 = 0; k0 < kend; k0 += 64) {
                    tmem_ld_32x32(tS + k0 + 32, vb);
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        mx0 = fmaxf(mx0, __uint_as_float(va[2 * i]));
                        mx1 = fmaxf(mx1, __uint_as_float(va[2 * i + 1]));
                    }
                    tmem_ld_wait();
                    if (k0 + 64 < kend) tmem_ld_32x32(tS + k0 + 64, va);
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        mx0 = fmaxf(mx0, __uint_as_float(vb[2 * i]));
                        mx1 = fmaxf(mx1, __uint_as_float(vb[2 * i + 1]));
                    }
                    tmem_ld_wait();
                }
                k_pipe = kend;
            }
#pragma unroll 1
            for (int k0 = k_pipe; k0 < p.Nk; k0 += 32) {
                if (k0 + 32 <= p.Nk) {
                    uint32_t v[32];
                    tmem_ld_32x32(tS + k0, v);
                    tmem_ld_wait();
                    if (k0 + 32 <= p.N) {
#pragma unroll
                        for (int i = 0; i < 16; i++) {
                            mx0 = fmaxf(mx0, __uint_as_float(v[2 * i]));
                            mx1 = fmaxf(mx1, __uint_as_float(v[2 * i + 1]));
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 32; i++) if (k0 + i < p.N) mx0 = fmaxf(mx0, __uint_as_float(v[i]));
                    }
                } else {
                    uint32_t v[16];
                    tmem_ld_32x16(tS + k0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; i++) if (k0 + i < p.N) mx0 = fmaxf(mx0, __uint_as_float(v[i]));
                }
            }
            const float m = fmaxf(mx0, mx1) * p.scale_log2;
            SN_TRACE(quad == 0 && lane == 0, 1 + grp, 12, g);                // max pass done
            // pass 2: P = exp2(s * c - m) -> fp16, written over the S columns already consumed
            float sum0 = 0.f, sum1 = 0.f;
#pragma unroll 1
            for (int k0 = 0; k0 < p.Nk; k0 += 32) {
                if (k0 + 32 <= p.Nk) {
                    uint32_t v[32], w[16];
                    tmem_ld_32x32(tS + k0, v);
                    tmem_ld_wait();
                    if (k0 + 32 <= p.N) {
#pragma unroll
                        for (int i = 0; i < 16; i++) {
                            const float p0 = ex2_fast(fmaf(__uint_as_float(v[2 * i]), p.scale_log2, -m));
                            const float p1 = ex2_fast(fmaf(__uint_as_float(v[2 * i + 1]), p.scale_log2, -m));
                            sum0 += p0; sum1 += p1;
                            w[i] = pack_h2_rn(p0, p1);
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; i++) {
                            const float p0 = k0 + 2 * i < p.N ? ex2_fast(fmaf(__uint_as_float(v[2 * i]), p.scale_log2, -m)) : 0.f;
                            const float p1 = k0 + 2 * i + 1 < p.N ? ex2_fast(fmaf(__uint_as_float(v[2 * i + 1]), p.scale_log2, -m)) : 0.f;
                            sum0 += p0; sum1 += p1;
                            w[i] = pack_h2_rn(p0, p1);
                        }
                    }
                    tmem_st_32x16(tS + (k0 >> 1), w);
                } else {
                    uint32_t v[16], w[8];
                    tmem_ld_32x16(tS + k0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const float p0 = k0 + 2 * i < p.N ? ex2_fast(fmaf(__uint_as_float(v[2 * i]), p.scale_log2, -m)) : 0.f;
                        const float p1 = k0 + 2 * i + 1 < p.N ? ex2_fast(fmaf(__uint_as_float(v[2 * i + 1]), p.scale_log2, -m)) : 0.f;
                        sum0 += p0; sum1 += p1;
                        w[i] = pack_h2_rn(p0, p1);
                    }
                    tmem_st_32x8(tS + (k0 >> 1), w);
                }
            }
            float px[kSnExtraMax];
#pragma unroll
            for (int e = 0; e < kSnExtraMax; e++) {
                px[e] = e < p.n_extra ? ex2_fast(fmaf(sx[e], p.scale_log2, -m)) : 0.f;
                sum0 += px[e];
            }
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&p_full[grp]);
            SN_TRACE(quad == 0 && lane == 0, 1 + grp, 7, g);                 // P written
            const float l = sum0 + sum1;
            // O = P V (+ the extra keys' p * v)
            mbar_wait(&v_full[s], (n >> 1) & 1);
            mbar_wait(&o_full[grp], (g >> 1) & 1);
            SN_TRACE(quad == 0 && lane == 0, 1 + grp, 9, g);                 // O ready
            tc_fence_after();
            float o[64];
            {
                uint32_t v0[32], v1[32];
                tmem_ld_32x32(tO, v0);
                tmem_ld_32x32(tO + 32, v1);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&o_empty[grp]);
#pragma unroll
                for (int i = 0; i < 32; i++) { o[i] = __uint_as_float(v0[i]); o[32 + i] = __uint_as_float(v1[i]); }
            }
            for (int e = 0; e < p.n_extra; e++) {
                const int j = p.Nk + e;
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    const uint4 wv = *reinterpret_cast<const uint4*>(cV + j * 128 + ((c ^ (j & 7)) << 4));
                    const __half2* hv = reinterpret_cast<const __half2*>(&wv);
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const float2 f = __half22float2(hv[u]);
                        o[8 * c + 2 * u] = fmaf(px[e], f.x, o[8 * c + 2 * u]);
                        o[8 * c + 2 * u + 1] = fmaf(px[e], f.y, o[8 * c + 2 * u + 1]);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&v_empty[s]);
            {
                const bool live = row < p.N;
                const float inv = live ? 1.0f / l : 0.f;
                const int64_t grow = int64_t(b) * p.N + row;
                const int row0 = row - lane;                                 // first row of this warp
                if (p.out_dtype == MV_F16 && mode == 1) {
                    __half* dst0 = reinterpret_cast<__half*>(p.out) + (int64_t(b) * p.N + row0) * p.ld_out + h * 64;
                    sn_store_rows_q16(sStg + (warp - 2) * 32 * kSnStgPitch, o, inv, dst0, p.ld_out, p.N - row0, lane);
                } else {
                    if (mode == 1) {
#pragma unroll
                        for (int i = 0; i < 16; i++) {                       // four at a time: one range test, rare path out of line
                            const float4 q4 = fq_half4_f32(make_float4(o[4 * i] * inv, o[4 * i + 1] * inv, o[4 * i + 2] * inv, o[4 * i + 3] * inv));
                            o[4 * i] = q4.x; o[4 * i + 1] = q4.y; o[4 * i + 2] = q4.z; o[4 * i + 3] = q4.w;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 64; i++) o[i] = fq_apply(o[i] * inv, mode, p.q_out);
                    }
                    if (p.out_dtype == MV_F16) {
                        __half* dst0 = reinterpret_cast<__half*>(p.out) + (int64_t(b) * p.N + row0) * p.ld_out + h * 64;
                        sn_store_rows_f(sStg + (warp - 2) * 32 * kSnStgPitch, o, dst0, p.ld_out, p.N - row0, lane);
                    } else if (live) {
                        float* dst = reinterpret_cast<float*>(p.out) + grow * p.ld_out + h * 64;
#pragma unroll
                        for (int i = 0; i < 16; i++)
                            reinterpret_cast<float4*>(dst)[i] = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
                    }
                }
                if (live && p.lse != nullptr) p.lse[(int64_t(b) * p.H + h) * p.N + row] = m + log2f(l);
                SN_TRACE(quad == 0 && lane == 0, 1 + grp, 16, g);            // output rows stored
            }
        }
    } else {
        // ================================ SIMT tail rows: the tail warps alternate (image, head) pairs ================================
        const int tw = warp - (2 + kSnMathWarps);
        for (int n = 0; n < n_local; n++) {
            const int s = n & 1;
            if ((n % kSnTailWarps) != tw) continue;
            const int bh = blockIdx.x + n * gridDim.x;
            const int b = bh / p.H, h = bh % p.H;
            const uint32_t ph = (n >> 1) & 1;
            mbar_wait_relaxed(&k_full[s], ph);
            mbar_wait_relaxed(&v_full[s], ph);
            for (int r = 0; r < p.n_tail; r++)
                sn_tail_row_fwd(p, sK + s * kSnKVBytes, sV + s * kSnKVBytes, s_tail + tw * (64 + kSnMaxKeys), b, h,
                                p.n_tiles * 128 + r, lane);
            __syncwarp();
            if (lane == 0) { mbar_arrive(&k_empty[s]); mbar_arrive(&v_empty[s]); }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<512>(tmem_base); }
}

constexpr int kSnFwdSmem = 4 * kSnKVBytes + 2 * kSnTile + kSnTailWarps * (64 + kSnMaxKeys) * 4 +
                           kSnMathWarps * 32 * kSnStgPitch + 256 + 1024;


// =====================================================================================
// Backward.  One persistent CTA per SM walks (image, head) pairs; Q and dO of the pair (<= 272 rows)
// are resident in shared memory, K_j / V_j stream through a 2-stage ring, one 128-key tile per pass.
// Everything is computed TRANSPOSED — keys on the TMEM lanes, query rows on the columns:
//   pre   S^T = K_j Q_c^T,  dP^T = V_j dO_c^T                     [128 keys x 64 rows] per block
//   math  P^T = exp2(S^T c - L_row),  dS^T = P^T (dP^T - Delta_row) scale      (one thread per key)
//   post  dV_j += P^T dO_c,  dK_j += dS^T Q_c      A = P^T / dS^T straight from TMEM (fp16, in place)
//         dQ_i += dS_i K_j   per pair of blocks     A = the two blocks' dS^T tiles in shared memory
//                                                   (MN-major: 64 query rows contiguous per key)
// so P never leaves TMEM, dV_j / dK_j / dQ_i accumulate in TMEM (no atomics, no dQ pass, deterministic)
// and the 512 TMEM columns hold two blocks in flight (one per math group of 4 warps) + 4 accumulators.
// Rows >= 256 (the 257th token) form a 16-wide tail block; their dQ has no TMEM accumulator and is
// reduced on the CUDA cores into shared memory.  Keys beyond N are zero rows (TMA fill) and fall out.
// 16 math warps: two per TMEM lane quadrant and block in flight (each takes 32 of the block's 64 columns), four per
// scheduler, so that one warp's TMEM read / exp / TMEM write chain hides under the others'.  576 threads: 112 registers.
// One more warp does nothing but the per-row statistics (L, Delta) of the NEXT pair — cold global reads, kept a whole
// pair ahead of the math warps.  Code that runs once per pass or pair (tail block, epilogues, statistics) is kept small
// on purpose: the kernel is far larger than the instruction caches, and a rarely executed, fully unrolled section costs
// more in instruction-fetch misses than in arithmetic (the 16-wide tail block took 5 000 cycles that way).
constexpr int kSnBwdMathWarps = 16, kSnBwdStatWarps = 2, kSnStatU = 4;   // 20 warps: 5 per scheduler, 96 registers
constexpr int kSnBwdMathThreads = 32 * kSnBwdMathWarps, kSnBwdStatThreads = 32 * kSnBwdStatWarps;
// One more warp owns the TMA stores: the math warps park dV_j / dK_j / dQ_i as fp16 in 128-byte-swizzled tiles (idle slots
// of the dS^T ring) and go on; written straight from the registers — one accumulator row per thread — every 16-byte
// store instruction of a warp touches 32 different lines and the LSU serialises them (4 000 cycles per pass epilogue,
// 17 000 of a pair's 43 000, clock64 timeline).
constexpr int kSnBwdThreads = 32 * (2 + kSnBwdMathWarps + kSnBwdStatWarps);
constexpr int kSnQBytes = kSnMaxKeys * 128;            // Q or dO of one pair: 272 rows x 128 B
constexpr int kSnOffQ = 4 * kSnTile;
constexpr int kSnOffDO = kSnOffQ + kSnQBytes;
constexpr int kSnOffDS = kSnOffDO + kSnQBytes;
// Odd keys (N = 256 + w, w <= kSnOddMax — the class token of the 256-patch configurations): instead of a third 128-key
// pass with w live keys (a quarter of the kernel's time for one key), keys 256 .. 256 + w - 1 are handled on the CUDA
// cores at the end of the pair's last pass, from the Q / dO rows resident in shared memory (odd_phase below).
constexpr int kSnOddMax = 4;
constexpr int kSnOffKo = kSnOffDS + 4 * kSnTile;       // K / V rows 256 .. 271 as the TMA leaves them (2 x 2 KB, 1024-aligned)
constexpr int kSnOffVec = kSnOffKo + 4096;             // L[272], Delta[272], dQ tail accumulators [16][64]
constexpr int kSnOffVec2 = kSnOffVec + (2 * kSnMaxKeys + 16 * 64) * 4;  // L / Delta of the next pair (double buffer)
// odd keys: k_u, v_u in fp32 [w][64] each; p[u][row], dS[u][row] (fp32, [w][272] each); dV_u / dK_u sums [w][2][64]
constexpr int kSnOffOdd = kSnOffVec2 + 2 * kSnMaxKeys * 4;
constexpr int kSnOddFloats = kSnOddMax * (2 * 64 + 2 * kSnMaxKeys + 2 * 64);
constexpr int kSnOffBar = kSnOffOdd + kSnOddFloats * 4;
constexpr int kSnBwdSmem = kSnOffBar + 256 + 1024;
static_assert(kSnBwdSmem <= 232448, "attention bwd (short sequences): shared memory over the 227 KB limit");

struct SnBwdDev {
    unsigned long long* trace;
    int B, H, N, D;
    int n_pass;                 // 128-key tiles
    int n_reg;                  // regular 64-row blocks per pass (2 per 128 query rows below 256)
    int tail_w;                 // width (multiple of 16) of the tail block of rows [256, 256 + tail_w); 0 if N <= 256
    int n_odd;                  // keys 256 .. 256 + n_odd - 1 handled by odd_phase instead of a third pass (0: none)
    float scale_log2, scale;
    const float* lse;
    const __half* o;            // forward output and its gradient, [B*N, D]: Delta = rowsum(dO * O) per head
    const __half* d_o;
    __half* dqkv; int ld_dqkv;
    float* dbias;               // NULL or fp32 [3 * D]: += column sums of dqkv (the to_qkv Linear's bias gradient)
    int* ovf;                   // overflow sink (mv_set_overflow_flag) or NULL: a dqkv value saturated its fp16 container
};

__global__ void __launch_bounds__(kSnBwdThreads, 1)
attn_bwd_sn_kernel(const __grid_constant__ CUtensorMap tm_qkv128, const __grid_constant__ CUtensorMap tm_qkv16,
                   const __grid_constant__ CUtensorMap tm_do128, const __grid_constant__ CUtensorMap tm_do16,
                   const __grid_constant__ CUtensorMap tm_dqkv128, const __grid_constant__ SnBwdDev p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned; offset arithmetic keeps the shared address space
    uint8_t* sK = smem;                                   // [2 stages][128 x 128 B]
    uint8_t* sV = smem + 2 * kSnTile;
    uint8_t* sQ = smem + kSnOffQ;                         // rows 0..271
    uint8_t* sdO = smem + kSnOffDO;
    uint8_t* sdS = smem + kSnOffDS;                       // ring of 4 dS^T tiles [128 keys][64 rows]
    float* sLD0 = reinterpret_cast<float*>(smem + kSnOffVec);     // L[272], Delta[272] of even pairs
    float* sLD1 = reinterpret_cast<float*>(smem + kSnOffVec2);    // ... of odd pairs
    float* sdQt = sLD0 + 2 * kSnMaxKeys;
    const uint8_t* sKo = smem + kSnOffKo;                          // K rows 256 .. 271 of the pair (128-byte swizzle)
    const uint8_t* sVo = sKo + 2048;
    float* kof = reinterpret_cast<float*>(smem + kSnOffOdd);       // [w][64] k_u as fp32
    float* vof = kof + kSnOddMax * 64;
    float* po = vof + kSnOddMax * 64;                              // [w][272] P[row, 256 + u]
    float* dso = po + kSnOddMax * kSnMaxKeys;                      // [w][272] dS[row, 256 + u]
    float* ored = dso + kSnOddMax * kSnMaxKeys;                    // [w][2][64] dV_u, dK_u
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kSnOffBar);
    uint64_t* kv_full = bars;           // [2]
    uint64_t* kv_empty = bars + 2;      // [2]
    uint64_t* qdo_full = bars + 4;
    uint64_t* qdo_empty = bars + 5;
    uint64_t* sdp_full = bars + 6;      // [2] per math group
    uint64_t* pds_full = bars + 8;      // [2]
    uint64_t* acc_full = bars + 10;
    uint64_t* acc_empty = bars + 11;
    uint64_t* dq_full = bars + 12;
    uint64_t* dq_empty = bars + 13;
    uint64_t* st_full = bars + 14;      // [2] statistics buffer (pair parity) written by the stats warps
    uint64_t* st_empty = bars + 16;     // [2] ... no longer read by the math warps
    // Staging tiles for the TMA stores = slots of the dS^T ring, idle at an epilogue.  "hi" (slots 2, 3 — the ones the
    // following blocks write last): dV_j / dK_j of every pass but a pair's last one, then the pair's dQ tiles, which stay
    // parked longer (column sums).  "lo" (slots 0, 1): dV_j / dK_j of the last pass.  hi events are numbered by the pass
    // counter pc, lo events by the pair counter n.
    uint64_t* sg_full = bars + 18;      // [2] lo / hi: all math warps have parked their slices
    uint64_t* sg_free = bars + 20;      // [2] lo / hi: the TMA engine has read the tiles
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 22);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    [[maybe_unused]] int trace_n = 0;
    const int n_bh = p.B * p.H;
    const int n_local = blockIdx.x < n_bh ? (n_bh - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int nblk = p.n_reg + (p.tail_w > 0 ? 1 : 0);           // blocks per pass

    const int nb_bh = p.n_pass * nblk;                            // blocks per (image, head)

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tm_qkv128); tma_prefetch_desc(&tm_qkv16);
        tma_prefetch_desc(&tm_do128); tma_prefetch_desc(&tm_do16); tma_prefetch_desc(&tm_dqkv128);
        for (int s = 0; s < 2; s++) { mbar_init(&sg_full[s], kSnBwdMathWarps); mbar_init(&sg_free[s], 1); }
        for (int s = 0; s < 2; s++) {
            mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1);
            mbar_init(&sdp_full[s], 1); mbar_init(&pds_full[s], kSnBwdMathWarps / 2);
        }
        mbar_init(qdo_full, 1); mbar_init(qdo_empty, p.n_odd > 0 ? 2 : 1);   // + the math warps' odd-key phase
        mbar_init(acc_full, 1); mbar_init(acc_empty, kSnBwdMathWarps);
        mbar_init(dq_full, 1); mbar_init(dq_empty, kSnBwdMathWarps);
        for (int s = 0; s < 2; s++) { mbar_init(&st_full[s], kSnBwdStatWarps); mbar_init(&st_empty[s], kSnBwdMathWarps); }
        fence_barrier_init();
    }
    // the dS^T tiles feed a K dimension: rows of keys that no thread writes must hold finite values
    for (int i = threadIdx.x; i < 4 * kSnTile / 16; i += kSnBwdThreads)
        reinterpret_cast<uint4*>(sdS)[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = threadIdx.x; i < 2 * kSnOddMax * kSnMaxKeys; i += kSnBwdThreads) po[i] = 0.f;     // P, dS of the odd keys: rows >= N stay zero
    fence_proxy_async();
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // TMEM columns: group g: S^T [g*128, +64) (P^T fp16 in place), dP^T [g*128+64, +64) (dS^T fp16 in place);
    // dV_j 256, dK_j 320, dQ_0 384, dQ_1 448
    const uint32_t tdV = tmem_base + 256, tdK = tmem_base + 320, tdQ = tmem_base + 384;

    if (warp == 0) {
        // ================================ TMA warp: loads and stores ================================
        // One warp serves two independent in-order queues without ever blocking on either (20 warps is what 96
        // registers per thread allow, and the per-row statistics need two of them):
        //   loads   per pair: K / V of pass 0, Q / dO (+ the odd K / V rows), K / V of the later passes — each as soon as
        //           its buffer is free;
        //   stores  per pair: dV_j / dK_j of every pass, then the dQ tiles — as soon as the 16 math warps have parked them
        //           (rows >= N of a box are clipped by the tensor map); the tiles are released once the TMA engine has
        //           read them.
        const int q_tiles = p.n_reg >> 1;
        int ln = 0, lk = 0;                       // load queue: pair, step (0: K/V of pass 0, 1: Q/dO, k >= 2: K/V of pass k - 1)
        int en = 0, ek = 0, cs_row = -1;          // store queue: pair, event (j < n_pass: pass j, n_pass: dQ), column-sum progress
        while (ln < n_local || en < n_local) {
            bool progress = false;
            if (ln < n_local) {
                const int bh = blockIdx.x + ln * gridDim.x;
                const int b = bh / p.H, h = bh % p.H;
                if (lk == 1) {
                    if (mbar_test(qdo_empty, (ln & 1) ^ 1)) {
                        if (lane == 0) {
                            mbar_arrive_expect_tx(qdo_full, 2 * (q_tiles * kSnTile + p.tail_w * 128) + (p.n_odd > 0 ? 4096 : 0));
                            if (p.n_odd > 0) {
                                tma_load_3d(const_cast<uint8_t*>(sKo), &tm_qkv16, qdo_full, p.D + h * 64, 256, b);
                                tma_load_3d(const_cast<uint8_t*>(sVo), &tm_qkv16, qdo_full, 2 * p.D + h * 64, 256, b);
                            }
                            for (int i = 0; i < q_tiles; i++) {
                                tma_load_3d(sQ + i * kSnTile, &tm_qkv128, qdo_full, h * 64, i * 128, b);
                                tma_load_3d(sdO + i * kSnTile, &tm_do128, qdo_full, h * 64, i * 128, b);
                            }
                            for (int r = 0; r < p.tail_w; r += 16) {
                                tma_load_3d(sQ + (256 + r) * 128, &tm_qkv16, qdo_full, h * 64, 256 + r, b);
                                tma_load_3d(sdO + (256 + r) * 128, &tm_do16, qdo_full, h * 64, 256 + r, b);
                            }
                        }
                        progress = true;
                        lk++;
                    }
                } else {
                    const int j = lk == 0 ? 0 : lk - 1;
                    const int pc = ln * p.n_pass + j, st = pc & 1;
                    if (mbar_test(&kv_empty[st], ((pc >> 1) & 1) ^ 1)) {
                        if (lane == 0) {
                            mbar_arrive_expect_tx(&kv_full[st], 2 * kSnTile);
                            tma_load_3d(sK + st * kSnTile, &tm_qkv128, &kv_full[st], p.D + h * 64, j * 128, b);
                            tma_load_3d(sV + st * kSnTile, &tm_qkv128, &kv_full[st], 2 * p.D + h * 64, j * 128, b);
                        }
                        progress = true;
                        lk++;
                    }
                }
                if (lk > p.n_pass) { lk = 0; ln++; }
            }
            if (en < n_local) {
                const int bh = blockIdx.x + en * gridDim.x;
                const int b = bh / p.H, h = bh % p.H;
                const int pc_last = en * p.n_pass + p.n_pass - 1;
                if (ek < p.n_pass) {
                    const bool last = ek == p.n_pass - 1;
                    if (last ? mbar_test(&sg_full[0], en & 1) : mbar_test(&sg_full[1], (en * p.n_pass + ek) & 1)) {
                        if (lane == 0) {
                            const uint8_t* src = sdS + (last ? 0 : 2 * kSnTile);
                            tma_store_3d(&tm_dqkv128, src, 2 * p.D + h * 64, ek * 128, b);
                            tma_store_3d(&tm_dqkv128, src + kSnTile, p.D + h * 64, ek * 128, b);
                            tma_store_commit();
                            tma_store_wait_read();
                            mbar_arrive(&sg_free[last ? 0 : 1]);
                        }
                        progress = true;
                        ek++;
                    }
                } else if (cs_row < 0) {
                    if (mbar_test(&sg_full[1], pc_last & 1)) {                 // the dQ tiles: the hi event of the last pass
                        if (lane == 0) {
                            for (int t = 0; t < q_tiles; t++) tma_store_3d(&tm_dqkv128, sdS + (2 + t) * kSnTile, h * 64, t * 128, b);
                            tma_store_commit();
                        }
                        progress = true;
                        cs_row = q_tiles * 128;
                    }
                } else {
                    if (cs_row >= q_tiles * 128) {
                        __syncwarp();
                        if (lane == 0) { tma_store_wait_read(); mbar_arrive(&sg_free[1]); }
                        cs_row = -1;
                        ek = 0;
                        en++;
                    }
                    progress = true;
                }
            }
            __syncwarp();
            if (!progress) __nanosleep(64);
        }
        if (lane == 0) tma_store_wait_all();
    } else if (warp == 1) {
        // ================================ MMA issuer ================================
        // the whole warp walks the schedule (uniform values live in uniform registers); one elected lane issues
        {
            const bool leader = elect_one();
            const uint32_t aK = smem_u32(sK), aV = smem_u32(sV), aQ = smem_u32(sQ), adO = smem_u32(sdO), adS = smem_u32(sdS);
            const uint32_t idesc_mn = make_idesc(0, 0, 0, 1, 128, 64);     // A K-major (TMEM), B MN-major, N = 64
            const uint32_t idesc_tt = make_idesc(0, 0, 1, 1, 128, 64);     // A MN-major, B MN-major, N = 64
            const uint32_t idesc_s64 = make_idesc(0, 0, 0, 0, 128, 64);
            const uint32_t idesc_stail = make_idesc(0, 0, 0, 0, 128, p.tail_w > 0 ? p.tail_w : 16);
            // This one lane is on the critical path of every block (the math groups wait for its MMAs and it
            // waits for theirs): the schedule is walked with counters instead of divisions and every
            // descriptor is a base built once plus a small offset.
            const uint64_t dK0 = make_smem_desc_sw128(aK, 16, 1024), dV0 = make_smem_desc_sw128(aV, 16, 1024);
            const uint64_t dQ0 = make_smem_desc_sw128(aQ, 16, 1024), dD0 = make_smem_desc_sw128(adO, 16, 1024);
            const uint64_t bD0 = make_smem_desc_sw128(adO, 8192, 1024), bQ0 = make_smem_desc_sw128(aQ, 8192, 1024);
            const uint64_t bK0 = make_smem_desc_sw128(aK, 8192, 1024), aS0 = make_smem_desc_sw128(adS, kSnTile, 1024);
            constexpr uint64_t kTileOff = kSnTile >> 4;            // one 16 KB tile further, in descriptor units
            int gb_pre = 0, gb_post = 0;                           // global block counters (parity = math group)
            int pc0 = 0;
            for (int n = 0; n < n_local; n++, pc0 += p.n_pass) {
                mbar_wait(qdo_full, n & 1);
                int j_pre = 0, c_pre = 0, j_post = 0, c_post = 0, rb_post = 0;     // rb: regular blocks before this one
                auto pre = [&]() {
                    const int gb = gb_pre, g = gb & 1, j = j_pre, c = c_pre;
                    const int pc = pc0 + j, st = pc & 1;
                    if (c == 0) mbar_wait(&kv_full[st], (pc >> 1) & 1);
                    tc_fence_after();
                    const bool regular = c < p.n_reg;
                    const uint64_t roff = uint64_t(regular ? 64 * c : 256) * 8;          // row0 * 128 B >> 4
                    const uint32_t idesc = regular ? idesc_s64 : idesc_stail;
                    const uint32_t tS = tmem_base + g * 128, tdP = tS + 64;
                    const uint64_t dk = dK0 + st * kTileOff, dv = dV0 + st * kTileOff;
                    const uint64_t dq = dQ0 + roff, dd = dD0 + roff;
                    if (leader) {
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            umma_f16(tS, dk + 2 * k, dq + 2 * k, idesc, k > 0);
                            umma_f16(tdP, dv + 2 * k, dd + 2 * k, idesc, k > 0);
                        }
                        umma_commit(&sdp_full[g]);
                        SN_TRACE(true, 0, 1, gb);                       // pre MMAs issued
                    }
                    gb_pre++;
                    if (++c_pre == nblk) { c_pre = 0; j_pre++; }
                    __syncwarp();
                };
                // post, first half: dV_j += P^T dO_c, dK_j += dS^T Q_c (A straight from TMEM)
                auto post_vk = [&]() {
                    const int gb = gb_post, g = gb & 1, j = j_post, c = c_post;
                    const int pc = pc0 + j;
                    const bool regular = c < p.n_reg;
                    const uint64_t roff = uint64_t(regular ? 64 * c : 256) * 8;
                    const uint32_t tS = tmem_base + g * 128, tdP = tS + 64;
                    const uint64_t bdo = bD0 + roff, bq = bQ0 + roff;                     // B = dO / Q rows, MN-major
                    mbar_wait(&pds_full[g], (gb >> 1) & 1);
                    SN_TRACE(leader, 0, 3, gb);                             // math of block gb done (seen by issuer)
                    if (c == 0 && pc > 0) mbar_wait(acc_empty, (pc - 1) & 1);       // dV / dK of the previous pass were read
                    tc_fence_after();
                    const uint32_t acc0 = c > 0 ? 1u : 0u;
                    if (leader) {
                        const int ksteps = regular ? 4 : (p.tail_w >> 4);
                        for (int k = 0; k < ksteps; k++) {
                            umma_f16_ts(tdV, tS + k * 8, bdo + 128 * k, idesc_mn, acc0 | uint32_t(k > 0));
                            umma_f16_ts(tdK, tdP + k * 8, bq + 128 * k, idesc_mn, acc0 | uint32_t(k > 0));
                        }
                    }
                    __syncwarp();
                };
                // post, second half — issued AFTER the S^T / dP^T MMAs of the group's next block, which the math warps are
                // waiting for and which do not depend on it: dQ_i += dS_i K_j for the block pair (c - 1, c), A = the pair's
                // dS^T tiles in shared memory (M = 2 x 64 rows, K = 128 keys); then the pass's / pair's commits
                auto post_dq = [&]() {
                    const int j = j_post, c = c_post;
                    const int pc = pc0 + j, st = pc & 1;
                    const bool regular = c < p.n_reg;
                    const bool with_dq = regular && (c & 1) != 0;
                    if (with_dq && c == 1 && j == 0 && n > 0) mbar_wait(dq_empty, (n - 1) & 1);  // dQ of the previous pair was read
                    if (leader) {
                        if (with_dq) {
                            const uint64_t ads = aS0 + uint64_t((rb_post - 1) & 3) * kTileOff;
                            const uint64_t bk = bK0 + st * kTileOff;
                            const uint32_t accq = j > 0 ? 1u : 0u;
                            const uint32_t tq = tdQ + (c >> 1) * 64;
#pragma unroll
                            for (int k = 0; k < 8; k++)
                                umma_f16(tq, ads + 128 * k, bk + 128 * k, idesc_tt, accq | uint32_t(k > 0));
                        }
                        SN_TRACE(true, 0, 4, gb_post);                          // post MMAs issued
                        if (c == nblk - 1) {
                            umma_commit(acc_full);
                            umma_commit(&kv_empty[st]);
                            if (j == p.n_pass - 1) { umma_commit(dq_full); umma_commit(qdo_empty); }
                        }
                    }
                    gb_post++;
                    if (regular) rb_post++;
                    if (++c_post == nblk) { c_post = 0; j_post++; }
                    __syncwarp();
                };
                pre();
                if (nb_bh > 1) pre();
                for (int lb = 0; lb < nb_bh; lb++) {
                    post_vk();
#ifdef SN_NO_REORDER
                    post_dq();
                    if (lb + 2 < nb_bh) pre();
#else
                    if (lb + 2 < nb_bh) pre();
                    post_dq();
#endif
                }
            }
        }
    } else if (warp >= 2 + kSnBwdMathWarps) {
        // ================================ statistics warps ================================
        // Per-row statistics of every pair (L from the forward, Delta = rowsum(dO * O)); rows >= N get L = +inf so that
        // their P is exactly 0.  Double-buffered by pair parity and written a whole pair ahead of the math warps, so the
        // cold global reads never sit on anybody's critical path.  Eight lanes share a row (one 16-byte chunk of the
        // head's 128 B each): a warp instruction reads four whole lines; eight row groups are in flight per thread.
        // cs_v: column sums of dO (this lane's chunk, every row it visits) — the v part of the fused bias gradient,
        //   sum_k dV[k, :] = sum_q (sum_k P[q, k]) dO[q, :] = the column sums of dO (rows of P sum to one).
        const int tid = threadIdx.x - 32 * (2 + kSnBwdMathWarps);
        const int sub = tid >> 3, ch = tid & 7;              // 4 rows per load instruction
        float cs_v[8];
#pragma unroll
        for (int k = 0; k < 8; k++) cs_v[k] = 0.f;
        for (int n = 0; n < n_local; n++) {
            const int bh = blockIdx.x + n * gridDim.x;
            const int b = bh / p.H, h = bh % p.H;
            float* dL = (n & 1) ? sLD1 : sLD0;
            if (n >= 2) mbar_wait_relaxed(&st_empty[n & 1], ((n >> 1) - 1) & 1);     // the math warps are done with pair n - 2
            const __half* pdo = p.d_o + int64_t(b) * p.N * p.D + h * 64;
            const __half* po = p.o + int64_t(b) * p.N * p.D + h * 64;
            const float* pl = p.lse + (int64_t(b) * p.H + h) * p.N;
#pragma unroll 1
            for (int base = 0; base < kSnMaxKeys; base += kSnStatU * (kSnBwdStatThreads >> 3)) {
                uint4 xa[kSnStatU], ya[kSnStatU];
                float Lr[kSnStatU];
#pragma unroll
                for (int u = 0; u < kSnStatU; u++) {
                    const int r = base + u * (kSnBwdStatThreads >> 3) + sub;
                    xa[u] = make_uint4(0u, 0u, 0u, 0u); ya[u] = xa[u]; Lr[u] = INFINITY;
                    if (r < p.N) {
                        // streamed once: keep them out of the small L1 (227 KB of it is shared memory)
                        xa[u] = __ldcs(reinterpret_cast<const uint4*>(pdo + int64_t(r) * p.D) + ch);
                        ya[u] = __ldcs(reinterpret_cast<const uint4*>(po + int64_t(r) * p.D) + ch);
                        if (ch == 0) Lr[u] = __ldcs(pl + r);
                    }
                }
#pragma unroll
                for (int u = 0; u < kSnStatU; u++) {
                    const int r = base + u * (kSnBwdStatThreads >> 3) + sub;
                    const __half2* xh = reinterpret_cast<const __half2*>(&xa[u]);
                    const __half2* yh = reinterpret_cast<const __half2*>(&ya[u]);
                    float dl = 0.f;
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const float2 fx = __half22float2(xh[q]), fy = __half22float2(yh[q]);
                        dl = fmaf(fx.x, fy.x, dl); dl = fmaf(fx.y, fy.y, dl);
                        cs_v[2 * q] += fx.x; cs_v[2 * q + 1] += fx.y;           // rows >= N contribute zeros
                    }
                    dl += __shfl_xor_sync(0xffffffffu, dl, 1);
                    dl += __shfl_xor_sync(0xffffffffu, dl, 2);
                    dl += __shfl_xor_sync(0xffffffffu, dl, 4);
                    if (ch == 0 && r < kSnMaxKeys) { dL[r] = Lr[u]; dL[kSnMaxKeys + r] = dl; }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&st_full[n & 1]);
        }
        if (p.dbias != nullptr && n_local > 0) {
            const int h = blockIdx.x % p.H;
#pragma unroll
            for (int k = 0; k < 8; k++) {                                   // lanes l, l ^ 8, l ^ 16, l ^ 24 share a chunk
                cs_v[k] += __shfl_xor_sync(0xffffffffu, cs_v[k], 8);
                cs_v[k] += __shfl_xor_sync(0xffffffffu, cs_v[k], 16);
            }
            if (lane < 8) {
                float* dv = p.dbias + 2 * p.D + h * 64 + lane * 8;
                sn_red_add_v4(dv, cs_v[0], cs_v[1], cs_v[2], cs_v[3]);
                sn_red_add_v4(dv + 4, cs_v[4], cs_v[5], cs_v[6], cs_v[7]);
            }
        }
    } else {
        // ================================ math: 16 warps, one thread per key ================================
        // group g = block parity (which of the two S^T / dP^T regions), half = which 32 of the block's 64 columns
        const int idx = warp - 2;
        const int quad = warp & 3;
        const int g = (idx >> 2) & 1, half = idx >> 3;
        const int slice = 2 * g + half;                      // 16-column slice of the accumulators this warp stores
        const int lr = quad * 32 + lane;                     // key row within the 128-key tile = TMEM lane
        const int mt = threadIdx.x - 64;                     // 0..511
        const uint32_t lane_off = uint32_t(quad * 32) << 16;
        const uint32_t tS = tmem_base + g * 128 + lane_off, tdP = tS + 64;
        int gb0 = 0, pc0 = 0;
        // Fused to_qkv bias gradient (p.dbias != NULL; the host then sizes the grid so that a CTA stays on one head
        // and the sums are flushed once, after the last pair):
        //   q: column sums of the parked dQ tiles (store warp) and, per thread, columns 2 * lane, 2 * lane + 1 of the dQ
        //      rows >= 256 (cs_t0 / cs_t1);
        //   k: nothing to add — sum_k dS[q, k] = sum_k P (dP - Delta_q) = 0, the key bias never reaches the softmax;
        //   v: the column sums of dO (statistics warps).
        float cs_t0 = 0.f, cs_t1 = 0.f;
        const bool do_cs = p.dbias != nullptr;
        float amax = 0.f;                                    // largest |dqkv| value stored (overflow sink)
        // Epilogues: this thread's accumulator row, its 16-column slice -> fp16 -> two 16-byte chunks of a 128-byte-swizzled
        // [128 rows][64 columns] staging tile (8 consecutive lanes cover the 8 chunk positions: conflict-free).
        auto park_slice = [&](const uint32_t (&v)[16], uint8_t* tile) {
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const float a = __uint_as_float(v[2 * i]), c = __uint_as_float(v[2 * i + 1]);
                amax = fmaxf(amax, fmaxf(fabsf(a), fabsf(c)));
                w[i] = pack_h2_satf(a, c);
            }
            uint8_t* row = tile + lr * 128;
            *reinterpret_cast<uint4*>(row + (((2 * slice) ^ (lr & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(row + (((2 * slice + 1) ^ (lr & 7)) << 4)) = make_uint4(w[4], w[5], w[6], w[7]);
        };
        // ---- odd keys (p.n_odd = w > 0): keys 256 .. 256 + w - 1 against every query row, by the math warps with warp-level
        // MMAs, from the Q / dO rows resident in shared memory.  Runs after the last block of the pair's last pass, while
        // its tcgen05 MMAs drain.  (The same sums as FMA loops on the CUDA cores cost 6 000 cycles per pair.)
        //   A  s = q_row . k_u, dP = dO_row . v_u -> P, dS (fp32, shared memory): a warp per 16 rows
        //   B  dV_u = sum_rows P dO_row, dK_u = sum_rows dS q_row: warp = (matrix, 8 columns)
        //   C  dV_u / dK_u rows to global memory;  D (pair epilogue): dQ_row += dS k_u before the rows are parked or, for
        //      rows >= 256, when their shared-memory accumulators are flushed
        auto odd_phase = [&](int n, int b, int h, const float* sL, const float* sDelta) {
            mbar_wait(qdo_full, n & 1);                  // the TMA writes of this pair's Q / dO / odd K, V rows, seen by this thread
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 25, n);
            {
                // A: [16 rows x 64] x [64 x 8 keys] per warp and matrix: a warp-level MMA per 16 dims.  The B fragments are
                // read straight from the TMA's K / V rows (row u of the 16-row box; rows >= N arrive as zeros).
                const int gq = lane >> 2, tq = lane & 3;
                for (int rt = idx; 16 * rt < p.N; rt += kSnBwdMathWarps) {
                    // (one accumulator per 16 dims: eight independent MMAs instead of two chains of four)
                    float cs4[4][4], cd4[4][4];
                    const int lrow = 16 * rt + (lane & 7) + ((lane >> 3) & 1) * 8;      // ldmatrix: this lane's row address
#pragma unroll
                    for (int kk = 0; kk < 4; kk++) {
                        float (&cs)[4] = cs4[kk];
                        float (&cd)[4] = cd4[kk];
#pragma unroll
                        for (int i = 0; i < 4; i++) { cs[i] = 0.f; cd[i] = 0.f; }
                        const int ch = 2 * kk + (lane >> 4);
                        uint32_t aq[4], ao[4];
                        ldmatrix_x4(aq, sQ + lrow * 128 + ((ch ^ (lrow & 7)) << 4));
                        ldmatrix_x4(ao, sdO + lrow * 128 + ((ch ^ (lrow & 7)) << 4));
                        const uint32_t off0 = gq * 128 + (((2 * kk) ^ gq) << 4) + 4 * tq;
                        const uint32_t off1 = gq * 128 + (((2 * kk + 1) ^ gq) << 4) + 4 * tq;
                        mma_16816(cs, aq, *reinterpret_cast<const uint32_t*>(sKo + off0), *reinterpret_cast<const uint32_t*>(sKo + off1));
                        mma_16816(cd, ao, *reinterpret_cast<const uint32_t*>(sVo + off0), *reinterpret_cast<const uint32_t*>(sVo + off1));
                    }
                    float cs[4], cd[4];
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        cs[i] = (cs4[0][i] + cs4[1][i]) + (cs4[2][i] + cs4[3][i]);
                        cd[i] = (cd4[0][i] + cd4[1][i]) + (cd4[2][i] + cd4[3][i]);
                    }
                    // this lane: rows 16 rt + gq and + 8, keys u = 2 tq and 2 tq + 1
#pragma unroll
                    for (int hr = 0; hr < 2; hr++) {
                        const int r = 16 * rt + gq + 8 * hr;
#pragma unroll
                        for (int e = 0; e < 2; e++) {
                            const int u = 2 * tq + e;
                            if (u < p.n_odd && r < p.N) {
                                const float pe = ex2_fast(fmaf(cs[2 * hr + e], p.scale_log2, -sL[r]));
                                po[u * kSnMaxKeys + r] = pe;
                                dso[u * kSnMaxKeys + r] = pe * (cd[2 * hr + e] - sDelta[r]) * p.scale;
                            }
                        }
                    }
                }
            }
            // k_u as fp32 for D (the rank-1 dQ updates of the pair epilogue), while the other warps finish A
            for (int i = mt; i < p.n_odd * 64; i += kSnBwdMathThreads) {
                const int u = i >> 6, d = i & 63;
                kof[u * 64 + d] = __half2float(*reinterpret_cast<const __half*>(sKo + u * 128 + (((d >> 3) ^ u) << 4) + (d & 7) * 2));
            }
            named_bar_sync(1, kSnBwdMathThreads);
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 26, n);
            {
                // B: [16 keys x 272 rows] x [272 x 8 columns] per warp = (matrix, 8-column chunk): one warp-level MMA per 16
                // rows.  A = P / dS of the odd keys (fp16 like the tensor-core passes; keys >= w and rows >= N are zeros),
                // B = the dO / Q rows through a transposing ldmatrix.
                const int m = idx >> 3, cc = idx & 7;                          // m = 0: dV_u (P, dO); 1: dK_u (dS, Q)
                const uint8_t* rows = m ? sQ : sdO;
                const float* wgt = (m ? dso : po) + (lane >> 2) * kSnMaxKeys;
                const bool has = (lane >> 2) < p.n_odd;
                const int tq = lane & 3;
                // 17 steps over the 272 resident rows (zeros beyond N), four independent accumulators
                float acc4[4][4];
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int i = 0; i < 4; i++) acc4[a][i] = 0.f;
#pragma unroll
                for (int ks = 0; ks < kSnMaxKeys / 16; ks++) {
                    float (&acc)[4] = acc4[ks & 3];
                    uint32_t af[4] = {0u, 0u, 0u, 0u};
                    if (has) {
                        const float2 w0 = *reinterpret_cast<const float2*>(wgt + 16 * ks + 2 * tq);
                        const float2 w1 = *reinterpret_cast<const float2*>(wgt + 16 * ks + 8 + 2 * tq);
                        af[0] = pack_h2_rn(w0.x, w0.y); af[2] = pack_h2_rn(w1.x, w1.y);
                    }
                    const int r = 16 * ks + (lane & 15);                        // ldmatrix.x2: lanes 0..15 give the row addresses
                    uint32_t b0, b1;
                    ldmatrix_x2_trans(b0, b1, rows + r * 128 + ((cc ^ (r & 7)) << 4));
                    mma_16816(acc, af, b0, b1);
                }
                if (has) {
                    float* dst = ored + (2 * (lane >> 2) + m) * 64 + cc * 8 + 2 * tq;
                    dst[0] = (acc4[0][0] + acc4[1][0]) + (acc4[2][0] + acc4[3][0]);
                    dst[1] = (acc4[0][1] + acc4[1][1]) + (acc4[2][1] + acc4[3][1]);
                }
            }
            named_bar_sync(1, kSnBwdMathThreads);
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 27, n);
            if (mt == 0) mbar_arrive(qdo_empty);         // Q, dO and the odd K / V rows are no longer read by the CUDA cores
            for (int i = mt; i < p.n_odd * 64; i += kSnBwdMathThreads) {
                const int u = i >> 6, m = (i >> 5) & 1, d2 = (i & 31) * 2;
                float* src = ored + (2 * u + m) * 64 + d2;
                const float a = src[0], c = src[1];
                amax = fmaxf(amax, fmaxf(fabsf(a), fabsf(c)));
                *reinterpret_cast<uint32_t*>(p.dqkv + (int64_t(b) * p.N + 256 + u) * p.ld_dqkv + (m == 0 ? 2 : 1) * p.D + h * 64 + d2) =
                    pack_h2_satf(a, c);
            }
        };
        // Staging events handed to the store warp (lo / hi tiles): has this warp seen the latest one released?  Checked
        // before anything is written to the dS^T ring or to a staging tile; a warp is never more than one event behind
        // (it waits for event k before it takes part in event k + 1).  The latest hi event is always number pc - 1
        // (pc: the current pass), the latest lo event number n - 1.
        bool pend_lo = false, pend_hi = false;
        for (int n = 0; n < n_local; n++, gb0 += nb_bh, pc0 += p.n_pass) {
            const int bh = blockIdx.x + n * gridDim.x;
            const int b = bh / p.H, h = bh % p.H;
            const float* sL = (n & 1) ? sLD1 : sLD0;
            const float* sDelta = sL + kSnMaxKeys;
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 19, n);                 // pair starts
            for (int i = mt; i < 16 * 64; i += kSnBwdMathThreads) sdQt[i] = 0.f;
            mbar_wait(&st_full[n & 1], (n >> 1) & 1);                                    // this pair's statistics are written
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 11, n);
            named_bar_sync(1, kSnBwdMathThreads);
            for (int j = 0; j < p.n_pass; j++) {
                const int pc = pc0 + j, st = pc & 1;
                const bool warp_live = j * 128 + quad * 32 < p.N;      // some key of this warp exists
                for (int c = 0; c < nblk; c++) {
                    const int gb = gb0 + j * nblk + c;
                    if ((gb & 1) != g) continue;
                    const bool regular = c < p.n_reg;
                    const int row0 = regular ? 64 * c : 256;
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 5, gb);         // math group starts waiting for S^T / dP^T
                    mbar_wait(&sdp_full[g], (gb >> 1) & 1);
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 6, gb);         // S^T / dP^T ready
                    tc_fence_after();
                    // only the pair of ring slots this block writes: the dQ tiles stay parked in slots 2, 3 for the column
                    // sums well into the next pair, whose first blocks write slots 0, 1
                    const bool slot_hi = (((j * p.n_reg + c) & 3) >> 1) != 0;
                    auto staging_released = [&]() {
                        if (!slot_hi && pend_lo) { mbar_wait(&sg_free[0], (n - 1) & 1); pend_lo = false; }
                        if (slot_hi && pend_hi) { mbar_wait(&sg_free[1], (pc - 1) & 1); pend_hi = false; }
                    };
                    if (warp_live) {
                        uint8_t* ds_row = sdS + ((j * p.n_reg + c) & 3) * kSnTile + lr * 128;
                        // 16 columns (query rows) of S^T / dP^T -> P^T / dS^T (fp16, in place in TMEM; dS^T also to
                        // shared memory for the dQ MMA).  de: optionally the fp32 dS values (tail block).
                        auto math16 = [&](const uint32_t (&sv)[16], const uint32_t (&dv)[16], int c0) {
                            uint32_t wp[8], wd[8];
#pragma unroll
                            for (int q4 = 0; q4 < 4; q4++) {
                                const float4 L4 = *reinterpret_cast<const float4*>(sL + row0 + c0 + 4 * q4);
                                const float4 D4 = *reinterpret_cast<const float4*>(sDelta + row0 + c0 + 4 * q4);
                                const float Ls[4] = {L4.x, L4.y, L4.z, L4.w}, Ds[4] = {D4.x, D4.y, D4.z, D4.w};
                                float pe[4], de[4];
#pragma unroll
                                for (int u = 0; u < 4; u++) {
                                    pe[u] = ex2_fast(fmaf(__uint_as_float(sv[4 * q4 + u]), p.scale_log2, -Ls[u]));
                                    de[u] = pe[u] * (__uint_as_float(dv[4 * q4 + u]) - Ds[u]) * p.scale;
                                }
                                wp[2 * q4] = pack_h2_rn(pe[0], pe[1]); wp[2 * q4 + 1] = pack_h2_rn(pe[2], pe[3]);
                                wd[2 * q4] = pack_h2_satf(de[0], de[1]); wd[2 * q4 + 1] = pack_h2_satf(de[2], de[3]);
                            }
                            tmem_st_32x8(tS + (c0 >> 1), wp);
                            tmem_st_32x8(tdP + (c0 >> 1), wd);
                            staging_released();                  // (first write into the dS^T ring after an epilogue)
#pragma unroll
                            for (int t = 0; t < 2; t++)
                                *reinterpret_cast<uint4*>(ds_row + ((((c0 >> 3) + t) ^ (lr & 7)) << 4)) =
                                    make_uint4(wd[4 * t], wd[4 * t + 1], wd[4 * t + 2], wd[4 * t + 3]);
                        };
                        if (regular) {
                            // Columns: half 0 takes fp32 chunks [0, 16) and [32, 48), half 1 takes [16, 32) and [48, 64).
                            // The fp16 results go back IN PLACE at columns c0 / 2 .. c0 / 2 + 7: the results of chunk
                            // [16, 32) land in the partner's first chunk [0, 16), those of chunk [32, 48) in the
                            // partner's first chunk [16, 32) — the two warps of a lane quadrant meet on a named barrier
                            // after their first loads, before anything is written back.  (Requesting the second chunk
                            // before the arithmetic of the first — 64 more live registers — spills at the 96 registers
                            // that 20 warps leave a thread, and the spills cost more than the exposed TMEM latency:
                            // 0.234 vs 0.213 ms.)
                            const int cb = 16 * half;
                            uint32_t sA[16], dA[16];
                            tmem_ld_32x16(tS + cb, sA); tmem_ld_32x16(tdP + cb, dA);
                            tmem_ld_wait();
                            named_bar_sync(3 + 4 * g + quad, 64);         // the partner has read its first chunk too
                            math16(sA, dA, cb);
                            tmem_ld_32x16(tS + cb + 32, sA); tmem_ld_32x16(tdP + cb + 32, dA);
                            tmem_ld_wait();                               // (the fp16 results only ever land in columns [0, 32))
                            math16(sA, dA, cb + 32);
                        } else if (half == 0) {
                            // 16-wide tail block: rows 256 .. 271 (tail_w == 16).  Same arithmetic through math16; the
                            // dQ of these rows has no TMEM accumulator: sum over this warp's 32 keys of
                            // dS[row, key] K[key, :] on the CUDA cores (lane l owns dims 2l, 2l+1), from the fp16 dS^T row
                            // this lane has just written to shared memory, accumulated in shared memory.
                            uint32_t sA[16], dA[16];
                            tmem_ld_32x16(tS, sA); tmem_ld_32x16(tdP, dA);
                            tmem_ld_wait();
                            math16(sA, dA, 0);
                            __syncwarp();
                            const int nrows = min(16, p.N - 256);
                            const int cl = lane >> 2, wi = (lane & 3) * 4;
                            const uint8_t* kt = sK + st * kSnTile;
                            const uint8_t* dsw = sdS + ((j * p.n_reg + c) & 3) * kSnTile + quad * 32 * 128;   // this warp's 32 key rows
#pragma unroll 1
                            for (int u = 0; u < nrows; u++) {
                                float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
                                for (int kk = 0; kk < 32; kk++) {
                                    const int kr = quad * 32 + kk;
                                    // dS^T[key kr][row u]: fp16 element u of the key's 128-byte row (16-byte chunk u >> 3)
                                    const float v = __half2float(*reinterpret_cast<const __half*>(
                                        dsw + kk * 128 + (((u >> 3) ^ (kr & 7)) << 4) + (u & 7) * 2));
                                    const float2 kf = __half22float2(*reinterpret_cast<const __half2*>(
                                        kt + kr * 128 + ((cl ^ (kr & 7)) << 4) + wi));
                                    a0 = fmaf(v, kf.x, a0); a1 = fmaf(v, kf.y, a1);
                                }
                                atomicAdd(&sdQt[u * 64 + 2 * lane], a0);
                                atomicAdd(&sdQt[u * 64 + 2 * lane + 1], a1);
                            }
                        }
                        tmem_st_wait();
                        fence_proxy_async();
                    }
                    staging_released();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&pds_full[g]);
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 7, gb);         // P^T / dS^T written
                }
                if (p.n_odd > 0 && j == p.n_pass - 1) {
                    odd_phase(n, b, h, sL, sDelta);
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 24, n);         // odd keys done
                }
                // ---- pass epilogue: every warp stores its 16-column slice of dV_j and of dK_j
                SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 8, pc);
                mbar_wait(acc_full, pc & 1);
                SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 9, pc);             // dV / dK of the pass complete
                tc_fence_after();
                {
                    uint32_t va[16], vb[16];
                    tmem_ld_32x16(tdV + lane_off + 16 * slice, va);
                    tmem_ld_32x16(tdK + lane_off + 16 * slice, vb);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty);
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 20, pc);        // accumulators in registers
                    const bool last = j == p.n_pass - 1;
                    if (last) { if (pend_lo) { mbar_wait(&sg_free[0], (n - 1) & 1); pend_lo = false; } }
                    else if (pend_hi) { mbar_wait(&sg_free[1], (pc - 1) & 1); pend_hi = false; }
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 21, pc);        // staging tiles free
                    uint8_t* tile = sdS + (last ? 0 : 2 * kSnTile);
                    park_slice(va, tile);
                    park_slice(vb, tile + kSnTile);
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sg_full[last ? 0 : 1]);
                    if (last) pend_lo = true; else pend_hi = true;
                    SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 22, pc);        // parked
                }
            }
            if (lane == 0) mbar_arrive(&st_empty[n & 1]);                                // this pair's statistics are consumed
            // ---- pair epilogue: dQ of query rows [128 t, 128 t + 128), every warp its 16-column slice
            const int pc_last = pc0 + p.n_pass - 1;
            mbar_wait(dq_full, n & 1);
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 10, n);
            tc_fence_after();
            {
                uint32_t va[16], vb[16];
                tmem_ld_32x16(tdQ + lane_off + 16 * slice, va);
                if (p.n_reg > 2) tmem_ld_32x16(tdQ + 64 + lane_off + 16 * slice, vb);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(dq_empty);
                for (int u = 0; u < p.n_odd; u++) {                   // dQ_row += dS[row, 256 + u] k_u
                    const float d0 = dso[u * kSnMaxKeys + lr], d1 = dso[u * kSnMaxKeys + 128 + lr];
                    const float* kk = kof + u * 64 + 16 * slice;
#pragma unroll
                    for (int i = 0; i < 16; i++) {
                        va[i] = __float_as_uint(fmaf(d0, kk[i], __uint_as_float(va[i])));
                        vb[i] = __float_as_uint(fmaf(d1, kk[i], __uint_as_float(vb[i])));
                    }
                }
                if (pend_hi) { mbar_wait(&sg_free[1], (pc_last - 1) & 1); pend_hi = false; }
                park_slice(va, sdS + 2 * kSnTile);
                if (p.n_reg > 2) park_slice(vb, sdS + 3 * kSnTile);
                if (do_cs) {
                    // q part of the fused to_qkv bias gradient: column sums of the parked tiles, 16 rows per warp, lane l
                    // owns columns 2l, 2l + 1 (rows >= N are exact zeros).  (One warp doing all 256 rows kept the tiles
                    // parked for 5 000 cycles and stalled the next pair's blocks that write these ring slots.)
                    named_bar_sync(2, kSnBwdMathThreads);
                    const uint8_t* tile = sdS + 2 * kSnTile;
                    if (16 * idx < (p.n_reg >> 1) * 128) {
#pragma unroll
                        for (int r = 16 * idx; r < 16 * idx + 16; r++) {
                            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(
                                tile + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + (lane & 3) * 4));
                            cs_t0 += f.x; cs_t1 += f.y;
                        }
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sg_full[1]);
                pend_hi = true;
            }
            // rows >= 256: dQ from the shared-memory accumulators
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 16, n);                 // dQ rows stored
            if (p.tail_w > 0) {
                named_bar_sync(1, kSnBwdMathThreads);
                for (int i = mt; i < (p.N - 256) * 32; i += kSnBwdMathThreads) {
                    const int r = i >> 5, l2 = i & 31;
                    for (int u = 0; u < p.n_odd; u++) {                 // the corner: odd keys against rows >= 256
                        const float de = dso[u * kSnMaxKeys + 256 + r];
                        sdQt[r * 64 + 2 * l2] = fmaf(de, kof[u * 64 + 2 * l2], sdQt[r * 64 + 2 * l2]);
                        sdQt[r * 64 + 2 * l2 + 1] = fmaf(de, kof[u * 64 + 2 * l2 + 1], sdQt[r * 64 + 2 * l2 + 1]);
                    }
                    amax = fmaxf(amax, fmaxf(fabsf(sdQt[r * 64 + 2 * l2]), fabsf(sdQt[r * 64 + 2 * l2 + 1])));
                    const uint32_t pk = pack_h2_satf(sdQt[r * 64 + 2 * l2], sdQt[r * 64 + 2 * l2 + 1]);
                    *reinterpret_cast<uint32_t*>(p.dqkv + (int64_t(b) * p.N + 256 + r) * p.ld_dqkv + h * 64 + 2 * l2) = pk;
                    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&pk));
                    cs_t0 += f.x; cs_t1 += f.y;                                 // l2 == lane for every i of this thread
                }
                named_bar_sync(1, kSnBwdMathThreads);
            }
            SN_TRACE(quad == 0 && lane == 0 && half == 0, 1 + g, 18, n);                 // pair finished
        }
        raise_overflow(p.ovf, amax);
        if (do_cs && n_local > 0) {
            const int h = blockIdx.x % p.H;
            // the 16 warps' sums meet in shared memory (the dQ tail accumulators are idle now), one global add per column
            named_bar_sync(1, kSnBwdMathThreads);
            if (idx == 0) { sdQt[2 * lane] = 0.f; sdQt[2 * lane + 1] = 0.f; }
            named_bar_sync(1, kSnBwdMathThreads);
            atomicAdd(&sdQt[2 * lane], cs_t0);
            atomicAdd(&sdQt[2 * lane + 1], cs_t1);
            named_bar_sync(1, kSnBwdMathThreads);
            if (idx == 0) {
                atomicAdd(p.dbias + h * 64 + 2 * lane, sdQt[2 * lane]);
                atomicAdd(p.dbias + h * 64 + 2 * lane + 1, sdQt[2 * lane + 1]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc<512>(tmem_base); }
}

}  // namespace mv

using namespace mv;

// dispatch rule shared with attention.cu
// keys on the tensor cores: a multiple of 16, at most 256 (two score tiles share the 512 TMEM columns);
// up to kSnExtraMax keys beyond that are folded in by the math threads
static void sn_key_split(int N, int* Nk, int* n_extra) {
    const int rem = N % 16;
    if (rem > 0 && rem <= kSnExtraMax && N > 16) { *Nk = N - rem; *n_extra = rem; }
    else { *Nk = (N + 15) & ~15; *n_extra = 0; }
}
extern "C" int mv_attention_sn_supported(int N) {
    int Nk, ne;
    sn_key_split(N, &Nk, &ne);
    return Nk <= 256 ? 1 : 0;
}

int mv_attention_fwd_sn(const void* qkv, void* out, int out_dtype, float* lse, int B, int H, int N,
                        float scale, int q_out_exp, int q_out_man, void* stream) {
    const int D = H * 64;
    static bool attr_done = false;
    if (!attr_done) {
        MV_CUDA(cudaFuncSetAttribute(attn_fwd_sn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSnFwdSmem));
        attr_done = true;
    }
    CUtensorMap t128, t16;
    if (make_tmap_3d(&t128, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 128, 1)) return 1;
    if (make_tmap_3d(&t16, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 16, 1)) return 1;
    SnFwdDev p;
    p.trace = g_sn_trace;
    p.B = B; p.H = H; p.N = N; p.D = D;
    sn_key_split(N, &p.Nk, &p.n_extra);
    p.Nld = p.Nk + (p.n_extra > 0 ? 16 : 0);
    const int tail = N % 128;
    if (tail > 0 && tail <= kSnTailMax) { p.n_tiles = N / 128; p.n_tail = tail; }
    else { p.n_tiles = (N + 127) / 128; p.n_tail = 0; }
    p.scale_log2 = scale * 1.4426950408889634f;
    p.qkv = reinterpret_cast<const __half*>(qkv);
    p.out = out; p.out_dtype = out_dtype; p.ld_out = D;
    p.q_out = FloatFmt{q_out_exp, q_out_man};
    p.lse = lse;
    const int n_bh = B * H;
    const int grid = n_bh < kNumSMs ? n_bh : kNumSMs;
    attn_fwd_sn_kernel<<<grid, kSnFwdThreads, kSnFwdSmem, static_cast<cudaStream_t>(stream)>>>(t128, t16, p);
    g_launches++;
    return check_cuda(cudaGetLastError(), "attention fwd (short-sequence) launch");
}

int mv_attention_bwd_sn(const void* qkv, const void* o, const void* d_o, const float* lse, float* delta,
                        void* dqkv, float* dbias, int B, int H, int N, float scale, void* stream) {
    const int D = H * 64;
    static bool attr_done = false;
    if (!attr_done) {
        MV_CUDA(cudaFuncSetAttribute(attn_bwd_sn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSnBwdSmem));
        attr_done = true;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUtensorMap q128, q16, d128, d16;
    if (make_tmap_3d(&q128, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 128, 1)) return 1;
    if (make_tmap_3d(&q16, qkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 16, 1)) return 1;
    if (make_tmap_3d(&d128, d_o, MV_F16, D, N, B, D, uint64_t(N) * D, 64, 128, 1)) return 1;
    if (make_tmap_3d(&d16, d_o, MV_F16, D, N, B, D, uint64_t(N) * D, 64, 16, 1)) return 1;
    CUtensorMap s128;                              // dqkv, stored by TMA from the staging tiles (rows >= N clipped)
    if (make_tmap_3d(&s128, dqkv, MV_F16, 3 * D, N, B, 3 * D, uint64_t(N) * 3 * D, 64, 128, 1)) return 1;
    (void)delta;                                   // Delta is computed inside the kernel
    SnBwdDev p;
    p.trace = g_sn_trace;
    p.B = B; p.H = H; p.N = N; p.D = D;
#ifdef SN_NO_ODD
    p.n_odd = 0;
#else
    p.n_odd = (N > 256 && N - 256 <= kSnOddMax) ? N - 256 : 0;
#endif
    p.n_pass = p.n_odd > 0 ? 2 : (N + 127) / 128;
    p.n_reg = 2 * (((N < 256 ? N : 256) + 127) / 128);
    p.tail_w = N > 256 ? ((N - 256 + 15) & ~15) : 0;
    p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
    p.lse = lse;
    p.o = reinterpret_cast<const __half*>(o); p.d_o = reinterpret_cast<const __half*>(d_o);
    p.dqkv = reinterpret_cast<__half*>(dqkv); p.ld_dqkv = 3 * D;
    const int n_bh = B * H;
    // Fused bias gradient: the kernel keeps per-head sums in registers, so a CTA must stay on one head — pair index =
    // blockIdx + n * grid with the grid a multiple of H (or one pair per CTA).  Same number of rounds as a full grid
    // whenever ceil(n_bh / grid) does not change (B = 256, H = 6: 11 rounds with 144 or 148 CTAs).
    const bool fuse = dbias != nullptr && H <= kNumSMs;
    const int grid = n_bh <= kNumSMs ? n_bh : (fuse ? (kNumSMs / H) * H : kNumSMs);
    p.dbias = fuse ? dbias : nullptr;
    p.ovf = g_overflow;
    attn_bwd_sn_kernel<<<grid, kSnBwdThreads, kSnBwdSmem, st>>>(q128, q16, d128, d16, s128, p);
    g_launches++;
    if (check_cuda(cudaGetLastError(), "attention bwd (short-sequence) launch")) return 1;
    if (dbias != nullptr && !fuse) return mv_colsum(dqkv, MV_F16, 3 * D, B * N, 3 * D, dbias, stream);
    return 0;
}
