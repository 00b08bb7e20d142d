// The bf16 policy/value net 128-256-256-256-(65+1) on a CTA pair (cluster of 2, tcgen05 cta_group::2), shared by the
// MLP kernels (mlp_pair.cu, mlp_pair2.cu) and the one-launch search (search_fused_kernel in mcts.cu): the layout of
// the weight image and of the operands in shared memory, the MMA issue of one layer, the hidden layers' epilogue
// arithmetic, the bulk copies of the weights and the host launcher of the MLP kernels.  Each kernel keeps its own
// schedule: which warp waits how, when the biases are read, where the operands live.
//
// A pair computes one M = 128 tile: each CTA holds 64 of its rows (the A operand) and half of every weight matrix (the
// B operand is split across the pair by N).  Numerics: bf16 operands, fp32 accumulate, fp32 bias, ReLU, bf16 round
// per layer; the head's 80 columns are 65 logits, the value and padding.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"
#include "umma.cuh"

namespace bz {

constexpr int kIn = 128;
constexpr int kHidden = 256;
constexpr int kHeadRows = 80;                     // 65 logits + value, padded to a legal UMMA N
constexpr int kOutStride = 72;                    // bf16 columns of an output row
constexpr int kTileRows = 128;                    // rows of the pair's tile == UMMA M
constexpr int kCtaRows = 64;                      // rows of the tile held by one CTA
constexpr int kSlabA = kCtaRows * 128;            // one 64-element K slab of A: 64 rows x 128 B
constexpr int kSmemA = 4 * kSlabA;                // 32 KB: the A operand of the widest layer (K = 256)

// ---- the weight image (net.pack_mlp_pair_image): per rank, its half of every layer's rows, layer after layer, each
// layer K / 64 slabs of N / 2 rows x 128 B in the shared-memory layout; then all biases as fp32 --------------------------
__host__ __device__ constexpr int layer_k(int l) { return l == 0 ? kIn : kHidden; }
__host__ __device__ constexpr int layer_n(int l) { return l == 3 ? kHeadRows : kHidden; }
__host__ __device__ constexpr int layer_slab(int l) { return layer_n(l) / 2 * 128; }  // this rank's N / 2 rows x 128 B
__host__ __device__ constexpr int layer_bytes(int l) { return layer_k(l) / 64 * layer_slab(l); }
constexpr int kSlabW = layer_slab(0), kSlabHead = layer_slab(3);
constexpr int kW0 = layer_bytes(0), kW1 = layer_bytes(1), kW2 = layer_bytes(2), kW3 = layer_bytes(3);
__host__ __device__ constexpr int layer_off(int l) { return l == 0 ? 0 : l == 1 ? kW0 : l == 2 ? kW0 + kW1 : kW0 + kW1 + kW2; }
constexpr int kSmemW = kW0 + kW1 + kW2 + kW3;     // 180 KB: one rank's half of every layer
constexpr int kNumBias = 3 * kHidden + kHeadRows;
constexpr int kSmemBias = kNumBias * 4;
constexpr int kImgRank = kSmemW + kSmemBias;      // one rank's row of the image: its weights, then all biases
static_assert(kImgRank == 187712, "the image of net.pack_mlp_pair_image is uint8 [2, 187712]");

// Shared address of the 16-byte chunk c (elements 8 c .. 8 c + 7) of row r of a K-major SWIZZLE_128B A operand: K / 64
// slabs of 64 rows x 128 B, chunk c % 8 of a row stored at chunk (c % 8) ^ (r % 8) of its 128-byte row
__device__ __forceinline__ uint32_t a_chunk(uint32_t sA, int r, int c) {
    return sA + (uint32_t)(c >> 3) * kSlabA + (uint32_t)r * 128u + (uint32_t)(((c & 7) ^ (r & 7)) << 4);
}

// The MMAs of one layer for the pair's tile (leader CTA, converged warp; A at sA, this layer's weights at sW), then the
// multicast commit that completes `bar` in both CTAs.  ONE elected-thread region, descriptors as 32-bit halves: the
// compiler keeps and advances them in uniform registers (an `if (elected)` around every MMA costs ~7 R2UR moves each).
__device__ __forceinline__ void pair_issue_layer(uint32_t elected, uint32_t tmem, uint32_t sA, uint32_t sW, int layer, uint32_t bar) {
    const uint32_t idesc = umma_idesc(kTileRows, layer_n(layer));
    // one K = 16 step is 32 bytes inside a 128-byte swizzle row, one 64-element slab kSlabA / layer_slab bytes: the
    // descriptors' address fields (units of 16 bytes, no carry out of their 14 bits) advance by constants
    uint32_t alo = kDescLo | ((sA >> 4) & 0x3FFFu);
    uint32_t blo = kDescLo | ((sW >> 4) & 0x3FFFu);
    const uint32_t bslab = (layer_slab(layer) - 96u) >> 4;
    const int nslab = layer_k(layer) / 64;
    if (elected) {
#pragma unroll 1
        for (int sl = 0; sl < nslab; ++sl) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                umma_bf16_pair_lohi(tmem, alo, blo, kDescHi32, idesc, (uint32_t)(sl | kk));
                alo += kk < 3 ? 2u : (uint32_t)((kSlabA - 96) >> 4);
                blo += kk < 3 ? 2u : bslab;
            }
        }
    }
    if (elected)
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                     "h"((uint16_t)3)
                     : "memory");
}

// Hidden layers' epilogue: 8 accumulators (consecutive columns) + their 8 biases, ReLU, bf16 -> one 16-byte chunk of the
// next layer's A operand
__device__ __forceinline__ uint4 hidden_chunk(const uint32_t *acc, const float4 *bias) {
    uint4 v;
    const float4 b0 = bias[0];
    v.x = pack_relu_bf16(add2(acc[0], acc[1], b0.x, b0.y));
    v.y = pack_relu_bf16(add2(acc[2], acc[3], b0.z, b0.w));
    const float4 b1 = bias[1];
    v.z = pack_relu_bf16(add2(acc[4], acc[5], b1.x, b1.y));
    v.w = pack_relu_bf16(add2(acc[6], acc[7], b1.z, b1.w));
    return v;
}

// this rank's half of layer l's weights (img: the rank's row of the image) -> dst, completing `bar`
__device__ __forceinline__ void load_layer(uint32_t dst, const uint8_t *img, int layer, uint32_t bar) {
    mbar_expect_tx(bar, layer_bytes(layer));
    bulk_load(dst, img + layer_off(layer), layer_bytes(layer), bar);
}
__device__ __forceinline__ void load_biases(uint32_t dst, const uint8_t *img, uint32_t bar) {
    mbar_expect_tx(bar, kSmemBias);
    bulk_load(dst, img + kSmemW, kSmemBias, bar);
}

// the CTA's 64 rows of x (rows row0 ..; rows at or past n are zero) -> a layer-0 A operand, cp.async by `nthreads` threads
__device__ __forceinline__ void load_x_rows(uint32_t sA, const __nv_bfloat16 *x, int row0, int n, int tid, int nthreads) {
    for (int i = tid; i < kCtaRows * (kIn / 8); i += nthreads) {
        const int r = i >> 4, c = i & 15;
        const bool ok = row0 + r < n;
        cp_async16(a_chunk(sA, r, c), x + (size_t)(ok ? row0 + r : 0) * kIn + c * 8, ok);
    }
}

// ---- the MLP kernels' launch: bz_mlp_forward_pair / bz_mlp_forward_pair2 ------------------------------------------------
struct PairParams {
    const __nv_bfloat16 *x;  // [B, 128]
    const uint8_t *wimg;     // [2 ranks][kImgRank]
    __nv_bfloat16 *out;      // [B, 72]
    int B;
};

// argument checks, the shared-memory opt-in (once per device), one launch of 2 CTAs per `pair_rows` rows under PDL
inline int launch_pair_mlp(void (*kernel)(PairParams), int pair_rows, int threads, int smem, bool (&configured)[64],
                           const void *x_bf16, const void *weight_image_pair, void *out_bf16, int64_t n, bz_stream_t stream) {
    if (n < 0 || (n && (!x_bf16 || !weight_image_pair || !out_bf16))) return BZ_ERR_ARG;
    if (!aligned16(x_bf16) || !aligned16(weight_image_pair) || !aligned16(out_bf16)) return BZ_ERR_UNALIGNED;
    if (n == 0) return BZ_OK;
    cudaError_t e = allow_dynamic_smem(kernel, smem, configured);
    if (e != cudaSuccess) return cuda_rc(e);
    const PairParams p = {(const __nv_bfloat16 *)x_bf16, (const uint8_t *)weight_image_pair, (__nv_bfloat16 *)out_bf16, (int)n};
    const unsigned pairs = (unsigned)((n + pair_rows - 1) / pair_rows);
    e = launch_kernel(kernel, dim3(2 * pairs), dim3(threads), (size_t)smem, as_stream(stream), pdl_enabled(), p);
    if (e != cudaSuccess) return cuda_rc(e);
    return launch_rc();
}

}  // namespace bz
