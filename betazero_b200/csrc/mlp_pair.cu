// The policy/value MLP on CTA PAIRS (pair_net.cuh): tcgen05.mma.cta_group::2, all weights resident in shared memory.
//
// Why pairs: at the self-play batch (4096 leaves) the net is a latency chain, not a throughput problem.  With one CTA
// per 128 leaves (profiles/experiments/mlp_onecta.cu) a hidden layer costs 16 MMAs x 128 clk (M = 128, N = 256 on one
// SM) plus the epilogue of 128 x 256 accumulators (bias, ReLU, bf16, swizzled st.shared: ~1 us), and the next layer's
// 128 KB of weights can only be fetched once the previous ones have been consumed (they do not fit beside the
// activations).
// Two CTAs of a cluster sharing one 128-leaf tile halve all three terms:
//   * the pair executes ONE M = 128, N = 256 MMA per K step (64 leaves per SM): 64 clk instead of 128;
//   * each SM converts only its own 64 x 256 accumulators;
//   * each SM holds HALF of every weight matrix (the B operand of a cta_group::2 MMA is split across the pair by
//     N), 180 KB for all four layers, so the whole net is fetched once, at kernel start, by four bulk copies
//     that do not wait for the tree kernel (programmatic dependent launch) -- no weight wait between layers.
// Activations stay private to the SM that owns the rows: no DSMEM traffic, only one remote mbarrier arrive per
// layer ("my half of the operands is ready") and the multicast tcgen05.commit that releases both epilogues.
//
// TMEM layout of a cta_group::2, M = 128 accumulator (PTX ISA "Data path layout organisation", 2x2 atom): in each
// CTA, row m (0..63) and column n live at lane m + 64 * (n / (N/2)), column n % (N/2).
#include "pair_net.cuh"

namespace bz {
namespace {

constexpr int kThreads = 512;    // 16 warps: 4 per TMEM lane quadrant x 4 groups of 32 accumulator columns
constexpr int kSmemTotal = kSmemA + kSmemW + kSmemBias + 128 + 1024;
constexpr int kTmemCols = 128;

#ifdef BZ_MLP_TRACE
__device__ long long g_pair_trace[64];
#define PAIR_TRACE(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_pair_trace[i] = clock64(); } while (0)
#define PAIR_TRACE2(i) do { if (blockIdx.x == 0 && (threadIdx.x == 0 || threadIdx.x == 480)) g_pair_trace[(i) + (threadIdx.x ? 16 : 0)] = clock64(); } while (0)
#else
#define PAIR_TRACE(i) do { } while (0)
#define PAIR_TRACE2(i) do { } while (0)
#endif

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) mlp_pair_kernel(const PairParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;  // identical in both CTAs: the MMA uses the leader's descriptors for both
    uint8_t *smem = smem_raw + (base - raw);
    const uint32_t sA = base, sW = base + kSmemA;
    const float *sBias = reinterpret_cast<const float *>(smem + kSmemA + kSmemW);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kSmemA + kSmemW + kSmemBias);
    // bars[0..3] weights of layer l landed (local); bars[4] accumulators complete (multicast commit);
    // bars[5] the peer CTA's operands are ready (used in the leader only: one remote arrival per layer);
    // bars[6] biases landed (local); bars[7] this CTA's operands are ready (one arrival per warp and layer)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 8);
    const uint32_t bar0 = smem_u32(bars);
    const uint32_t mma_bar = bar0 + 8u * 4, ready_bar = bar0 + 8u * 5, bias_bar = bar0 + 8u * 6, local_bar = bar0 + 8u * 7;

    PAIR_TRACE(0);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // provably warp-uniform
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int row0 = (int)(blockIdx.x >> 1) * kTileRows + (int)rank * kCtaRows;
    const int valid_rows = max(0, min(kCtaRows, p.B - row0));
    const uint8_t *img = p.wimg + (size_t)rank * kImgRank;

    // ---- prologue: nothing here depends on the previous kernel (it overlaps its tail under PDL) ----
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else if (threadIdx.x == 32) {
        for (int i = 0; i < 4; ++i) mbar_init(bar0 + 8u * i, 1);
        mbar_init(mma_bar, 1);
        mbar_init(ready_bar, 1);
        mbar_init(bias_bar, 1);
        mbar_init(local_bar, kThreads / 32);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // First in the queue: what layer 0 needs (this CTA's half of W1, the biases).  An SM ingests ~64 B/clk from
        // L2, so the order of the copies is the order in which the layers can start.
        load_layer(sW, img, 0, bar0);
        load_biases(sW + kSmemW, img, bias_bar);
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_arrive();  // both CTAs: barriers initialised, TMEM allocated; completes while the x copies are in flight

    // ---- the leaf planes are the previous kernel's output ----
    pdl_wait();
    pdl_launch_dependents();
    PAIR_TRACE(1);
    load_x_rows(sA, p.x, row0, p.B, threadIdx.x, kThreads);
    if (threadIdx.x == 32) {  // behind the x copies: this CTA's half of the other three layers, one bulk copy per layer
        for (int l = 1; l < 4; ++l) load_layer(sW + layer_off(l), img, l, bar0 + 8u * l);
    }
    PAIR_TRACE(25);
    cluster_wait();
    PAIR_TRACE(26);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    asm volatile("cp.async.wait_all;" ::: "memory");
    PAIR_TRACE(2);

    const int q = warp & 3, g = warp >> 2;
    const int r = (q & 1) * 32 + lane;                                // accumulator row of this thread
    const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);          // TMEM lanes of this warp

#pragma unroll 1
    for (int layer = 0; layer < 4; ++layer) {
        // this warp's part of the A operand (generic-proxy stores) -> visible to the tensor cores of the pair;
        // its accumulator reads of the previous layer are complete.  One arrival per warp on the leader's barrier.
        PAIR_TRACE2(31 + 4 * layer);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        PAIR_TRACE2(32 + 4 * layer);
        if (lane == 0) mbar_arrive(local_bar);
        if (warp == 0) {  // the whole warp, converged
            mbar_wait(local_bar, (uint32_t)(layer & 1));  // all 16 warps of this CTA
            mbar_wait(bar0 + 8u * layer, 0);              // this CTA's half of the layer's weights has landed
            PAIR_TRACE(3 + 5 * layer);
            if (rank != 0 && lane == 0) mbar_arrive_remote(ready_bar, 0);  // one remote arrival per layer (remote arrivals serialise)
            __syncwarp();
        }
        if (warp == 0 && rank == 0) {  // MMA issue: one elected lane per instruction, operands in uniform registers
            mbar_wait_cluster(ready_bar, (uint32_t)(layer & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            PAIR_TRACE(5 + 5 * layer);
            pair_issue_layer(elect_one(), tmem, sA, sW + layer_off(layer), layer, mma_bar);
            __syncwarp();
            PAIR_TRACE(6 + 5 * layer);
        }
        if (layer == 0) mbar_wait(bias_bar, 0);
        const float *bias = sBias + layer * kHidden;
        // this thread's 32 accumulator columns: logical columns (q / 2) * 128 + g * 32 ..; their biases are fetched
        // while the MMAs run
        const int c0 = (q >> 1) * (kHidden / 2) + g * 32;
        float4 bv[8];
        if (layer < 3) {
            const float4 *b4 = reinterpret_cast<const float4 *>(bias + c0);
#pragma unroll
            for (int j = 0; j < 8; ++j) bv[j] = b4[j];
        }
        mbar_wait(mma_bar, (uint32_t)(layer & 1));
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        PAIR_TRACE(7 + 5 * layer);
        if (layer < 3) {
            uint32_t acc[32];
            tmem_ld32(trow + (uint32_t)(g * 32), acc);
            PAIR_TRACE2(30 + 4 * layer);
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) st_shared_v4(a_chunk(sA, r, (c0 >> 3) + qq), hidden_chunk(acc + 8 * qq, bv + 2 * qq));
        } else {
            // head: N = 80 -> 40 TMEM columns per lane half; 72 output columns (65 logits, value, padding).
            // The cluster barrier that guards the TMEM release is signalled as soon as the accumulators are in
            // registers, so its latency hides behind the stores.
            const int chalf = (q >> 1) * (kHeadRows / 2);
            __nv_bfloat16 *orow = p.out + (size_t)(row0 + r) * kOutStride;
            if (g == 0) {
                uint32_t acc[32];
                tmem_ld32(trow, acc);
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                cluster_arrive();
                if (r < valid_rows) {
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq) {
                        const int c = chalf + qq * 8;  // < 72 for both halves
                        *reinterpret_cast<uint4 *>(orow + c) = bias_pack8(acc + qq * 8, bias + c);
                    }
                }
            } else if (g == 1 && q < 2) {  // columns 32..39 of the first half
                uint32_t acc[8];
                tmem_ld8(trow + 32u, acc);
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                cluster_arrive();
                if (r < valid_rows) *reinterpret_cast<uint4 *>(orow + 32) = bias_pack8(acc, bias + 32);
            } else {
                cluster_arrive();
            }
        }
    }
    PAIR_TRACE(23);
    cluster_wait();  // nobody frees TMEM (or exits) while the peer may still read its accumulators
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
    PAIR_TRACE(24);
}

}  // namespace
}  // namespace bz

using namespace bz;

#ifdef BZ_MLP_TRACE
extern "C" int bz_mlp_pair_debug_trace(long long *host_out) {
    return cuda_rc(cudaMemcpyFromSymbol(host_out, g_pair_trace, sizeof(long long) * 64));
}
#endif

extern "C" int64_t bz_mlp_pair_image_bytes(void) { return 2 * (int64_t)kImgRank; }

extern "C" int bz_mlp_forward_pair(const void *x_bf16, const void *weight_image_pair, void *out_bf16, int64_t n, bz_stream_t stream) {
    static bool configured[64] = {};
    return launch_pair_mlp(mlp_pair_kernel, kTileRows, kThreads, kSmemTotal, configured, x_bf16, weight_image_pair, out_bf16, n, stream);
}
