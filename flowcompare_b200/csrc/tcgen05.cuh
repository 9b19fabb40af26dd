// Shared PTX helpers for the tcgen05 kernels (gemm_tc.cu, attention_tc.cu): mbarriers with bounded waits, TMA
// tile loads, tcgen05.mma (TS form: A in tensor memory, B through a shared-memory descriptor), TMEM ld/st.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>

namespace {

// ----------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a pipeline bug must surface as a trapped kernel with a message, never as a hung GPU.
// (kept inline: an out-of-line report cost 3 % of the step -- the call ABI pins registers around every wait)
__device__ __forceinline__ void mbar_timeout(int tag, uint32_t parity) {
    printf("flowcompare_b200 tcgen05 kernel: mbarrier wait timed out (tag %d, block %d,%d thread %d, parity %u)\n", tag,
           blockIdx.x, blockIdx.y, threadIdx.x, parity);
    __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag = 0) {
    uint32_t done = 0;
    for (uint32_t spin = 0; spin < (1u << 22); ++spin) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (done) return;
    }
    mbar_timeout(tag, parity);
}
// non-blocking probe of a phase: lets an issuing warp check the NEXT stage before it blocks on the tensor queue
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return done != 0;
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, void* smem_dst, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// TMA store of a shared-memory tile (bulk async group): generic-proxy writes must be fenced (fence.proxy.async) before it
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool elect_one() {   // one lane of a converged warp
    uint32_t pred;
    asm volatile("{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\telect.sync rx|px, 0xffffffff;\n\tselp.u32 %0, 1, 0, px;\n\t}" : "=r"(pred));
    return pred != 0;
}
// D[tmem] (+)= A[tmem] * B[smem descriptor]   (A: 128 lanes x 8 columns of TF32, B: K-major tile)
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem descriptor]   (kind::f16: A = 128 lanes x 8 columns, each column two fp16 (k even in the low half); B: K-major fp16 tile, K = 16)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major operand tile, 64-byte rows (32 fp16), SWIZZLE_64B: 8-row groups are 512 B apart (SBO)
__device__ __forceinline__ uint64_t make_kmajor_sw64_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(512 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)4 << 61;                              // SWIZZLE_64B
    return d;
}
// two fp32 -> packed fp16x2 (first argument in the LOW half), round to nearest even, overflow -> inf (never silently clipped)
__device__ __forceinline__ uint32_t pack_f16x2(float lo_half, float hi_half) {
    uint32_t r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi_half), "f"(lo_half));
    return r;
}
__device__ __forceinline__ void unpack_f16x2(uint32_t v, float& lo_half, float& hi_half) {
    asm("{\n\t.reg .f16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(lo_half), "=f"(hi_half) : "r"(v));
}
// K-major operand tile, 128-byte rows, SWIZZLE_128B: 8-row groups are 1024 B apart (SBO), version 1 (Blackwell)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);        // start address  [0,14)
    d |= (uint64_t)1 << 16;                              // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset [32,46)
    d |= (uint64_t)1 << 46;                              // descriptor version
    d |= (uint64_t)2 << 61;                              // SWIZZLE_128B
    return d;
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"   // same asm statement: no use of r[] can be scheduled before the wait
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
// two 16-column loads (main and compensation accumulator of a chunk) in flight together, ONE wait: half the TMEM round trips
__device__ __forceinline__ void tmem_ld16x2(uint32_t taddr_a, uint32_t taddr_b, uint32_t (&a)[16], uint32_t (&b)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%32];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%33];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]),
          "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]),
          "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]), "=r"(b[8]),
          "=r"(b[9]), "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15])
        : "r"(taddr_a), "r"(taddr_b) : "memory");
}
// the same pair of loads split into issue and wait, so that a chunk's loads can be in flight while the previous chunk is
// processed: the wait names every destination register as in/out, which keeps the compiler from reading them early
__device__ __forceinline__ void tmem_ld16x2_issue(uint32_t taddr_a, uint32_t taddr_b, uint32_t (&a)[16], uint32_t (&b)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%32];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%33];"
        : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]),
          "=r"(a[9]), "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]),
          "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]), "=r"(b[8]),
          "=r"(b[9]), "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15])
        : "r"(taddr_a), "r"(taddr_b) : "memory");
}
__device__ __forceinline__ void tmem_ld16x2_wait(uint32_t (&a)[16], uint32_t (&b)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
        : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(a[8]),
          "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
          "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]), "+r"(b[8]),
          "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15])
        :: "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
          "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
          "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31]) : "memory");
}

// A in TMEM / accumulator layout: lane = tile row, one 32-bit column per element
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
        "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]),
          "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]),
          "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, void* smem_dst, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

typedef CUresult (*FcEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline FcEncodeTiledFn fc_get_encode_fn() {
    static FcEncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<FcEncodeTiledFn>(p);
    }
    return fn;
}

}  // namespace
