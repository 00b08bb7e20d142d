// The CTA-pair MLP of mlp_pair.cu with TWO 128-leaf tiles per pair, ping-ponged: for batches of 9 473 .. 18 944 leaves
// (the 16 384 leaves per iteration of the default 4-leaves search = 64 pairs = 128 CTAs, one wave).
//
// In mlp_pair.cu a hidden layer of one tile is 0.64 us of tcgen05.mma followed by 0.8 us in which the tensor cores
// idle (accumulator read-out, bias/ReLU/bf16, proxy fence, CTA barrier, remote handshake).  With two independent tiles
// per pair those 0.8 us are the other tile's MMAs: a dedicated control warp issues MMA(tile 0), MMA(tile 1), MMA(tile 0),
// ... as the tiles' operands become ready, the 16 epilogue warps convert tile 0 then tile 1 then tile 0 ..., each
// tile has its own accumulators (2 x 128 TMEM columns), its own activation buffer (2 x 32 KB) and its own barriers.
// A pair therefore finishes 256 leaves in about the time mlp_pair.cu needs for 128.
//
// Weights: with 64 KB of activations per CTA the whole net no longer fits beside them, so two 64 KB weight regions
// are recycled (each CTA still holds only its HALF of every matrix):
//   region B: layer 0's half (32 KB, fetched first)            -> after both tiles' layer-0 MMAs: layer 2's half (64 KB)
//   region A: layer 1's half (64 KB, fetched behind the input) -> after both tiles' layer-1 MMAs: the head's half (20 KB)
// so every layer's weights are requested a full layer before they are needed.
// Same weight image (bz_mlp_pair_image_bytes), numerics and results as bz_mlp_forward_pair.
#include "pair_net.cuh"

namespace bz {
namespace {

constexpr int kPairRows = 2 * kTileRows;  // leaves per CTA pair (two tiles)
constexpr int kEpiWarps = 16;    // epilogue: 4 warps per TMEM lane quadrant x 4 groups of 32 accumulator columns
constexpr int kThreads = (kEpiWarps + 2) * 32;  // + the control warp + the loader warp
constexpr int kRegion = 4 * kSlabW;               // 64 KB: one recycled weight region
constexpr int kSmemTotal = 2 * kSmemA + 2 * kRegion + kSmemBias + 256 + 1024;
constexpr int kTmemCols = 256;                    // 2 tiles x 128 columns

#ifdef BZ_MLP_TRACE
// debug timeline of CTA 0: slots written by lane 0 of the control warp (MMA side) or of epilogue warp 0
__device__ long long g_pair2_trace[96];
#define P2_TRACE(i) do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0) g_pair2_trace[i] = clock64(); } while (0)
#else
#define P2_TRACE(i) do { } while (0)
#endif

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1) mlp_pair2_kernel(const PairParams p) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;  // identical in both CTAs: the MMA uses the leader's descriptors for both
    uint8_t *smem = smem_raw + (base - raw);
    const uint32_t sA = base;                                   // tile t: sA + t * kSmemA
    const uint32_t sRegA = base + 2 * kSmemA, sRegB = sRegA + kRegion;
    const float *sBias = reinterpret_cast<const float *>(smem + 2 * kSmemA + 2 * kRegion);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + 2 * kSmemA + 2 * kRegion + kSmemBias);
    // bars[0..3] weights of layer l landed (local)          bars[4] biases landed (local)
    // bars[5 + t] accumulators of tile t complete (multicast commit)
    // bars[7 + t] this CTA's part of tile t's A operand is stored (one arrival per epilogue warp and layer)
    // bars[9 + t] (leader only) the peer's part of tile t's A operand is stored (one remote arrival per layer)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 11);
    const uint32_t bar0 = smem_u32(bars);
    const uint32_t bias_bar = bar0 + 8u * 4;
    auto mma_bar = [&](int t) { return bar0 + 8u * (uint32_t)(5 + t); };
    auto local_bar = [&](int t) { return bar0 + 8u * (uint32_t)(7 + t); };
    auto ready_bar = [&](int t) { return bar0 + 8u * (uint32_t)(9 + t); };

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // provably warp-uniform
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair_row0 = (int)(blockIdx.x >> 1) * kPairRows;
    const uint8_t *wsrc = p.wimg + (size_t)rank * kImgRank;
    const bool control = warp == kEpiWarps, loader = warp == kEpiWarps + 1;

    // ---- prologue: nothing here depends on the previous kernel (it overlaps its tail under PDL) ----
    if (control) {
        if (lane == 0) {
            for (int i = 0; i < 5; ++i) mbar_init(bar0 + 8u * i, 1);
            for (int t = 0; t < 2; ++t) {
                mbar_init(mma_bar(t), 1);
                mbar_init(local_bar(t), kEpiWarps);
                mbar_init(ready_bar(t), 1);
            }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    __syncthreads();  // barriers initialised before the loader warp arms them
    // All bulk copies come from the loader WARP: a releasing remote arrive (control warp) otherwise waits for the bulk
    // copies its own warp has in flight (+0.8 us per handshake, whichever lane issued them).
    if (loader && lane == 0) {
        load_layer(sRegB, wsrc, 0, bar0);  // layer 0's half -> region B, first in the queue
        load_biases(sRegA + 2 * kRegion, wsrc, bias_bar);  // the bias array behind the regions
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_arrive();  // both CTAs: barriers initialised, TMEM allocated; completes while the x copies are in flight

    // ---- the leaf planes are the previous kernel's output ----
    pdl_wait();
    pdl_launch_dependents();
    if (warp < kEpiWarps) {
        // both tiles' rows of this CTA: tile t, rank r -> rows pair_row0 + t * 128 + r * 64 ..
        for (int t = 0; t < 2; ++t)
            load_x_rows(sA + (uint32_t)t * kSmemA, p.x, pair_row0 + t * kTileRows + (int)rank * kCtaRows, p.B, threadIdx.x, kEpiWarps * 32);
    } else if (loader && lane == 0) {  // behind the x copies: layer 1's half -> region A
        load_layer(sRegA, wsrc, 1, bar0 + 8u);
    }
    cluster_wait();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    if (control) P2_TRACE(0);

    if (control) {
        // ================= control warp (converged; one elected lane per tcgen05 instruction) =================
        const uint32_t elected = elect_one();
#pragma unroll 1
        for (int layer = 0; layer < 4; ++layer) {
            const uint32_t sWl = (layer & 1) ? sRegA : sRegB;  // layers 0, 2 read region B; layers 1, 3 region A
            const uint32_t par = (uint32_t)(layer & 1);
#pragma unroll 1
            for (int t = 0; t < 2; ++t) {
                mbar_wait(local_bar(t), par);                       // this CTA's 16 epilogue warps have stored tile t's operand
                if (t == 0) mbar_wait(bar0 + 8u * layer, 0);        // this CTA's half of the layer's weights has landed
                P2_TRACE(1 + 8 * layer + 4 * t);
                if (rank != 0) {
                    if (lane == 0) mbar_arrive_remote(ready_bar(t), 0);
                    __syncwarp();
                } else {
                    mbar_wait_cluster(ready_bar(t), par);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    P2_TRACE(2 + 8 * layer + 4 * t);
                    pair_issue_layer(elected, tmem + (uint32_t)t * 128u, sA + (uint32_t)t * kSmemA, sWl, layer, mma_bar(t));
                    __syncwarp();
                    P2_TRACE(3 + 8 * layer + 4 * t);
                }
            }
        }
        cluster_arrive();
    } else if (loader) {
        // ================= loader warp: recycles the weight regions =================
        // the region a layer has read is free for the layer after next once BOTH tiles' MMAs of that layer are done
        for (int layer = 0; layer < 2; ++layer) {
            mbar_wait(mma_bar(0), (uint32_t)(layer & 1));
            mbar_wait(mma_bar(1), (uint32_t)(layer & 1));
            if (lane == 0) {
                if (layer == 0) load_layer(sRegB, wsrc, 2, bar0 + 16u);
                else load_layer(sRegA, wsrc, 3, bar0 + 24u);
            }
            __syncwarp();
        }
        cluster_arrive();
    } else {
        // ================= epilogue warps: tile 0, tile 1, tile 0, ... =================
        const int q = warp & 3, g = warp >> 2;
        const int r = (q & 1) * 32 + lane;                        // accumulator row of this thread inside the CTA's 64
        const uint32_t trow = tmem + ((uint32_t)(q * 32) << 16);  // TMEM lanes of this warp
        const int c0 = (q >> 1) * (kHidden / 2) + g * 32;         // hidden layers: this thread's 32 logical columns
        // layer-0 operands: both tiles' x
        asm volatile("cp.async.wait_all;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            mbar_arrive(local_bar(0));
            mbar_arrive(local_bar(1));
        }
        mbar_wait(bias_bar, 0);
#pragma unroll 1
        for (int layer = 0; layer < 4; ++layer) {
            const float *bias = sBias + layer * kHidden;
            const uint32_t par = (uint32_t)(layer & 1);
            float4 bv[8];
            if (layer < 3) {  // the biases of this thread's columns, shared by both tiles, fetched while the MMAs run
                const float4 *b4 = reinterpret_cast<const float4 *>(bias + c0);
#pragma unroll
                for (int j = 0; j < 8; ++j) bv[j] = b4[j];
            }
#pragma unroll 1
            for (int t = 0; t < 2; ++t) {
                mbar_wait(mma_bar(t), par);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (warp == 0) P2_TRACE(40 + 4 * layer + 2 * t);
                const uint32_t tcol = trow + (uint32_t)t * 128u;
                if (layer < 3) {
                    uint32_t acc[32];
                    tmem_ld32(tcol + (uint32_t)(g * 32), acc);
#pragma unroll
                    for (int qq = 0; qq < 4; ++qq)
                        st_shared_v4(a_chunk(sA + (uint32_t)t * kSmemA, r, (c0 >> 3) + qq), hidden_chunk(acc + 8 * qq, bv + 2 * qq));
                    // this warp's part of tile t's next operand -> visible to the tensor cores; its accumulator reads are done
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(local_bar(t));
                    if (warp == 0) P2_TRACE(41 + 4 * layer + 2 * t);
                } else {
                    // head: N = 80 -> 40 TMEM columns per lane half; 72 output columns (65 logits, value, padding)
                    const int chalf = (q >> 1) * (kHeadRows / 2);
                    const int row = pair_row0 + t * kTileRows + (int)rank * kCtaRows + r;
                    __nv_bfloat16 *orow = p.out + (size_t)row * kOutStride;
                    if (g == 0) {
                        uint32_t acc[32];
                        tmem_ld32(tcol, acc);
                        if (t == 1) {  // the last accumulator read of this thread: release the TMEM guard early
                            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                            cluster_arrive();
                        }
                        if (row < p.B) {
#pragma unroll
                            for (int qq = 0; qq < 4; ++qq) {
                                const int c = chalf + qq * 8;  // < 72 for both halves
                                *reinterpret_cast<uint4 *>(orow + c) = bias_pack8(acc + qq * 8, bias + c);
                            }
                        }
                    } else if (g == 1 && q < 2) {  // columns 32..39 of the first half
                        uint32_t acc[8];
                        tmem_ld8(tcol + 32u, acc);
                        if (t == 1) {
                            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                            cluster_arrive();
                        }
                        if (row < p.B) *reinterpret_cast<uint4 *>(orow + 32) = bias_pack8(acc, bias + 32);
                    } else if (t == 1) {
                        cluster_arrive();
                    }
                }
            }
        }
    }
    if (control) P2_TRACE(60);
    cluster_wait();  // nobody frees TMEM (or exits) while the peer may still read its accumulators
    if (control) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
}

}  // namespace
}  // namespace bz

using namespace bz;

#ifdef BZ_MLP_TRACE
extern "C" int bz_mlp_pair2_debug_trace(long long *host_out) {
    return cuda_rc(cudaMemcpyFromSymbol(host_out, g_pair2_trace, sizeof(long long) * 96));
}
#endif

extern "C" int bz_mlp_forward_pair2(const void *x_bf16, const void *weight_image_pair, void *out_bf16, int64_t n, bz_stream_t stream) {
    static bool configured[64] = {};
    return launch_pair_mlp(mlp_pair2_kernel, kPairRows, kThreads, kSmemTotal, configured, x_bf16, weight_image_pair, out_bf16, n, stream);
}
