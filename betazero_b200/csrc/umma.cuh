// tcgen05 / TMEM / mbarrier / bulk-copy building blocks of the net's kernels (pair_net.cuh; the single-CTA helpers are
// those of profiles/experiments/mlp_onecta.cu): inline PTX for sm_100a.  Descriptor encodings follow the PTX ISA
// "tcgen05 shared memory descriptor" / "instruction descriptor" tables.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>

namespace bz {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// UMMA shared-memory matrix descriptor, K-major, SWIZZLE_128B: 8-row groups 1024 B apart (SBO), LBO = 1 (unused
// for swizzled K-major), version 1 (sm_100), layout type 2.  See cute/arch/mma_sm100_desc.hpp (CUTLASS).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// umma_desc as 32-bit halves (umma_bf16_pair_lohi): LBO = 1 in the low word beside the address; SBO, version and
// SWIZZLE_128B in the high word, the same for every operand
constexpr uint32_t kDescLo = 1u << 16, kDescHi32 = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);

// instruction descriptor for kind::f16: D = F32, A = B = BF16, both K-major, shape M x N
__device__ __forceinline__ uint32_t umma_idesc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, bool valid) {
    const int bytes = valid ? 16 : 0;  // src-size 0: zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(bytes) : "memory");
}

// mbarrier phase wait with a bounded spin: a descriptor bug must trap, not hang the GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
    }
    __trap();
}

// The same wait for warps that may wait for microseconds beside working warps (the one-launch search): try_wait with a
// suspend-time hint parks the thread in hardware instead of spinning through the issue slots of the SM sub-partition
// (a plain try_wait loop was 36 % of all instructions issued by search_fused_kernel).
__device__ __forceinline__ void mbar_wait_parked(uint32_t bar, uint32_t parity) {
    for (uint32_t spin = 0; spin < (1u << 22); ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity), "r"(20000u)
            : "memory");
        if (done) return;
    }
    __trap();
}

// Short waits beside working warps: poll, but yield the issue slot for kNapNs between polls (measured on the final
// one-launch kernel: 20 / 40 / 100 ns all +0.7 % from the start position, +0.3 % in the bench region, against a plain spin)
constexpr unsigned kNapNs = 32;
__device__ __forceinline__ void mbar_wait_nap(uint32_t bar, uint32_t parity) {
    for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
        __nanosleep(kNapNs);
    }
    __trap();
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&v);
}

// ---- CTA pairs (clusters of 2, tcgen05 cta_group::2): the net of pair_net.cuh ---------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// relaxed: the only cross-CTA state published through these barriers is the mbarrier initialisation (which has its own
// fence.mbarrier_init.release.cluster) and "my tcgen05.ld have completed" (tcgen05 fences); a releasing arrive costs ~1000 clk
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster.  Default semantics (release at
// CTA scope), the form CUTLASS's ClusterBarrier::arrive(cta_id) uses for its 2-SM pipelines: the data the leader's MMA
// will read sits in THIS CTA's shared memory and was made visible to the async proxy by its writers' fence.proxy.async
// before the CTA-local barrier.  A .release.cluster arrive was measured at 0.25 - 0.9 us per handshake (longest while
// bulk copies are in flight on the SM); this form at 0.06 - 0.12 us.
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(bar),
        "r"(rank)
        : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
    }
    __trap();
}
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n" : "=r"(pred));
    return pred;
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// the same load without the wait: the caller overlaps it with other work and then executes tmem_ld_wait()
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// (a0 + b0, a1 + b1), each sum rounded to fp32 (FADD2: one issue slot for two adds)
__device__ __forceinline__ float2 add2(uint32_t a0, uint32_t a1, float b0, float b1) {
    uint64_t a, b, r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(a0), "r"(a1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    float2 f;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(f.x), "=f"(f.y) : "l"(r));
    return f;
}
// bf16x2 {lo = relu(v.x), hi = relu(v.y)}, round to nearest even: max(x, 0) and the rounding commute
__device__ __forceinline__ uint32_t pack_relu_bf16(float2 v) {
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(v.y), "f"(v.x));
    return d;
}

// the same MMA with the descriptors as 32-bit halves: the low words (the only ones that change from MMA to MMA) stay
// 32-bit values the compiler can keep and advance in uniform registers
__device__ __forceinline__ void umma_bf16_pair_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                                    uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ uint4 bias_pack8(const uint32_t *acc, const float *bias) {
    const float4 b0 = *reinterpret_cast<const float4 *>(bias), b1 = *reinterpret_cast<const float4 *>(bias + 4);
    const float2 s0 = add2(acc[0], acc[1], b0.x, b0.y), s1 = add2(acc[2], acc[3], b0.z, b0.w);
    const float2 s2 = add2(acc[4], acc[5], b1.x, b1.y), s3 = add2(acc[6], acc[7], b1.z, b1.w);
    uint4 v;
    v.x = pack_bf16(s0.x, s0.y);
    v.y = pack_bf16(s1.x, s1.y);
    v.z = pack_bf16(s2.x, s2.y);
    v.w = pack_bf16(s3.x, s3.y);
    return v;
}

}  // namespace bz
