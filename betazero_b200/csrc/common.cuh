// Launch helpers shared by the .cu files of libbetazero_b200.so
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/betazero_b200.h"

namespace bz {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

inline int cuda_rc(cudaError_t e) { return e == cudaSuccess ? BZ_OK : -(1000 + (int)e); }

inline int launch_rc() { return cuda_rc(cudaGetLastError()); }

inline cudaStream_t as_stream(bz_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// grid for a grid-stride kernel over `items` work items: whole multiples of the SM count,
// enough CTAs to fill the machine (`ctas_per_sm` resident), never more than the work needs
inline int persistent_grid(int64_t items, int threads, int ctas_per_sm) {
    int64_t need = (items + threads - 1) / threads;
    int64_t full = (int64_t)kNumSMs * ctas_per_sm;
    if (need >= full) return (int)full;
    if (need <= 0) return 1;
    // round up to a multiple of the SM count when that does not overshoot the work by much
    int64_t r = ((need + kNumSMs - 1) / kNumSMs) * kNumSMs;
    return (int)(r <= need + kNumSMs / 2 ? r : need);
}

// Programmatic dependent launch (PDL): when enabled (bz_set_pdl), the tree step kernel and the fused MLP kernel
// are launched with cudaLaunchAttributeProgrammaticStreamSerialization, so the prologue of each (record / root
// loads; TMEM allocation + first weight tile) overlaps the tail of the other instead of waiting for a full drain.
// Both kernels execute griddepcontrol.wait before touching the other's output (a no-op without the attribute).
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl,
                                 Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// opt a kernel in to more than 48 KB of dynamic shared memory, once per device (the attribute is per device: a process that
// drives several GPUs must set it on each)
template <typename K>
inline cudaError_t allow_dynamic_smem(K kernel, int bytes, bool (&done)[64]) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    if (!done[dev]) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) return e;
        done[dev] = true;
    }
    return cudaSuccess;
}

// Debug build (-DBZ_BOUNDS_CHECK, profiles/sanitize.sh): every index the tree / self-play kernels form into a pool is
// checked against the pool's size before it is used; the first violation is recorded (code, block, thread) and counted,
// and bz_debug_checks() reports it.  compute-sanitizer is not available on the GPU pool this was developed on; these are
// the "bounds checks and asserts of your own".  Release builds compile the checks away.
#ifdef BZ_BOUNDS_CHECK
static __device__ int g_bz_check[4];  // [0] first failing check's code, [1] block, [2] thread, [3] number of violations (per .cu file)
#define BZ_CHECK(cond, code)                                              \
    do {                                                                  \
        if (!(cond)) {                                                    \
            if (atomicCAS(&g_bz_check[0], 0, (code)) == 0) {              \
                g_bz_check[1] = (int)blockIdx.x;                          \
                g_bz_check[2] = (int)threadIdx.x;                         \
            }                                                             \
            atomicAdd(&g_bz_check[3], 1);                                 \
        }                                                                 \
    } while (0)
#else
#define BZ_CHECK(cond, code) do { } while (0)
#endif

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- Philox4x32-10 (counter-based RNG; results depend only on (seed, game id, ply)) -------------
// self-play move sampling and match openings (selfplay.cu), the minimax players' random move (minimax.cu)
__host__ __device__ inline uint32_t philox_u32(uint64_t seed, uint64_t game_id, uint32_t ply) {
    uint32_t c0 = (uint32_t)game_id, c1 = (uint32_t)(game_id >> 32), c2 = ply, c3 = 0;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c1 = (uint32_t)p1;
        c3 = (uint32_t)p0;
        c0 = n0;
        c2 = n2;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c0;
}

// streaming (read-once / write-once) 128-bit global accesses that do not allocate in L1
__device__ __forceinline__ ulonglong2 ld_stream_u64x2(const uint64_t *p) {
    ulonglong2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];" : "=l"(r.x), "=l"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_u64x2(uint64_t *p, ulonglong2 v) {
    asm volatile("st.global.L1::no_allocate.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(v.x), "l"(v.y) : "memory");
}

}  // namespace bz
