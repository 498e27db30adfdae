// common.cuh — error plumbing and sm_100a PTX wrappers (mbarrier, TMA, tcgen05, TMEM).
// Hand-written for this repo; no CUTLASS/CuTe in the product path.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "quant_dev.cuh"

namespace mv {

void set_error(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

#define MV_CHECK(cond, ...)            \
    do {                               \
        if (!(cond)) {                 \
            mv::set_error(__VA_ARGS__); \
            return 1;                  \
        }                              \
    } while (0)

#define MV_CUDA(expr)                                   \
    do {                                                \
        if (mv::check_cuda((expr), #expr)) return 1;    \
    } while (0)

constexpr int kNumSMs = 148;

// Overflow sink (mv_set_overflow_flag): kernels that round gradient values into fp16 containers keep the largest
// |value| they convert and raise the flag when it would not fit (>= 65520 rounds past 65504: the container
// saturates; +-inf included.  NaNs are caught by the final un-scale pass, which tests every parameter gradient).
extern int* g_overflow;
constexpr float kHalfOverflow = 65520.0f;
__device__ __forceinline__ void raise_overflow(int* flag, float amax) {
    if (flag != nullptr && amax >= kHalfOverflow) *flag = 1;
}

// ------------------------------------------------------------------ misc
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// single-instruction MUFU forms (exp2f() / __fdividef() add range handling the fused epilogues do not need)
__device__ __forceinline__ float ex2_fast(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// -------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// same, for waits that are expected to be long (producers, side warps): back off between polls so the
// spinning lane does not take issue slots from the math warps of its scheduler
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred P1;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, P1;\n\t}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(200);
    }
}

// ------------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0,
                                            int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
        "{%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* tmap, uint64_t* bar, int c0,
                                            int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
        "{%3, %4, %5}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// TMA store (shared -> global, bulk async-group completion): rows / columns of the box that fall outside the
// tensor are not written.  The source tile must be visible to the async proxy (fence_proxy_async) first.
__device__ __forceinline__ void tma_store_3d(const void* tmap, const void* smem_src, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(tmap)),
                 "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the source tiles of every committed group have been read (shared memory reusable)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... and written (before the kernel ends)
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// --------------------------------------------------------------- clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// shared::cluster address of `local_addr` (a shared::cta address) in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
// arrive on an mbarrier that may live in the peer CTA (shared::cluster address).  Default
// (.release.cta) semantics on purpose: .release.cluster makes ptxas emit MEMBAR.ALL.GPU, which waits
// for every outstanding global store of the warp; the TMEM hand-off only needs the tcgen05 fence.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// CTA-pair TMA load: lands in this CTA's shared memory, completes bytes on an mbarrier that may be
// the peer's (the pair's leader waits for both halves of a stage on one barrier)
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const void* tmap, uint32_t bar_cluster_addr,
                                                int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
        "{%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}

// --------------------------------------------------------------- tcgen05, CTA pair (cta_group::2)
template <int kCols>
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* dst_smem) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(dst_smem)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
                 : "memory");
}
// D[tmem, both CTAs] (+)= A[256 x K: 128 rows per CTA] * B[N x K: N/2 rows per CTA]; issued by the leader
__device__ __forceinline__ void umma_f16_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                             uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the mbarrier at this offset in every CTA of cta_mask once the pair's MMAs have completed
__device__ __forceinline__ void umma_commit_cg2(uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"(cta_mask)
        : "memory");
}

// --------------------------------------------------------------- tcgen05
__device__ __forceinline__ void tc_fence_before() {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(dst_smem)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols)
                 : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc];  kind::f16 covers fp16/bf16 operands
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                         uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                          uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand from TMEM (used by attention: P stays on chip)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile(
        "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
            smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp gets lane (base + t)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
          "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
          "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
          "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
          "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]),
        "r"(r[15])
        : "memory");
}

// ------------------------------------------------- UMMA descriptors (sm_100)
// Shared-memory matrix descriptor, 128-byte swizzle, version 1:
//   [0,14) start>>4   [16,30) LBO>>4   [32,46) SBO>>4   [46,48) version=1   [61,64) layout=2 (SW128)
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes,
                                                         uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// Instruction descriptor for kind::f16 / kind::tf32, fp32 accumulate.
//   fmt: 0 = f16, 1 = bf16, 2 = tf32 ; major: 0 = K-major, 1 = MN-major
__host__ __device__ constexpr uint32_t make_idesc(int a_fmt, int b_fmt, int a_major, int b_major,
                                                  int m, int n) {
    return (1u << 4) | (uint32_t(a_fmt) << 7) | (uint32_t(b_fmt) << 10) |
           (uint32_t(a_major) << 15) | (uint32_t(b_major) << 16) | (uint32_t(n >> 3) << 17) |
           (uint32_t(m >> 4) << 24);
}

// ------------------------------------------------------- host: TMA maps
// dtype: MV_F32 (4 B) or MV_F16 (2 B).  2-D row-major tensor [rows, cols] with row pitch
// `ld` elements; box = [box_rows, box_cols]; 128-byte swizzle.
int make_tmap_2d(CUtensorMap* map, const void* ptr, int dtype, uint64_t rows, uint64_t cols,
                 uint64_t ld, uint32_t box_rows, uint32_t box_cols);
int make_tmap_2d_plain(CUtensorMap* map, const void* ptr, int dtype, uint64_t rows, uint64_t cols,
                       uint64_t ld, uint32_t box_rows, uint32_t box_cols, int swizzle64 = 0);  // same, no / 64-byte swizzle, any 16-byte inner extent
// 3-D: [d2, d1, d0] with d0 contiguous, strides in elements
int make_tmap_3d(CUtensorMap* map, const void* ptr, int dtype, uint64_t d0, uint64_t d1,
                 uint64_t d2, uint64_t stride1, uint64_t stride2, uint32_t box0, uint32_t box1,
                 uint32_t box2);

}  // namespace mv
