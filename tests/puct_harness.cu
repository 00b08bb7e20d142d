// Test harness for the PUCT primitives of betazero_b200/csrc/puct.cuh (tests/test_gpu_puct_edges.py builds it with the
// library's nvcc flags on first use).  Sweep kernels enumerate a domain on the device and count what breaks a claim of
// the header; map kernels apply a primitive to host arrays for checks against numpy.  Every entry returns a cudaError_t.
#include <cstdint>
#include <cuda_runtime.h>

#include "../betazero_b200/csrc/puct.cuh"

namespace {

using bz::exp_nonpos;
using bz::fdiv_by_count;
using bz::order_key;

constexpr int kRecords = 8;  // mismatches kept for a test's message: 4 words each

struct Sink {
    unsigned long long *count;  // counters of the sweep
    unsigned *rec;              // [0] records taken, then kRecords x 4 words
};

__device__ void record(const Sink &s, unsigned kind, unsigned a, unsigned b, unsigned c) {
    const unsigned i = atomicAdd(&s.rec[0], 1u);
    if (i < kRecords) {
        s.rec[1 + 4 * i] = kind;
        s.rec[2 + 4 * i] = a;
        s.rec[3 + 4 * i] = b;
        s.rec[4 + 4 * i] = c;
    }
}

__device__ __forceinline__ unsigned mix(unsigned long long x) {  // splitmix64 finaliser
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return (unsigned)((x ^ (x >> 31)) >> 16);
}

__device__ __forceinline__ float from_parts(unsigned sign, int biased_exp, unsigned mant) {
    return __uint_as_float((sign << 31) | ((unsigned)biased_exp << 23) | (mant & 0x7FFFFFu));
}

__device__ __forceinline__ unsigned long long mulmod(unsigned long long a, unsigned long long b, unsigned long long m) {
    return (a * b) % m;  // a, b < m < 2^24
}

// numerator i (0..63) of divisor d: specials, denormals, random mantissas over the exponents of the range and beyond,
// and numerators whose quotient by d lies within 1/d of a unit in the last place of a rounding midpoint (or of a float)
__device__ float sweep_numerator(unsigned d, int i, unsigned seed, bool &near_mid) {
    const unsigned h = mix(((unsigned long long)d << 8 | (unsigned)i) ^ ((unsigned long long)seed << 40));
    const unsigned h2 = mix(h ^ 0x5bd1e995u);
    const unsigned sign = h2 >> 31;
    near_mid = false;
    if (i < 18) {
        constexpr unsigned kSpecial[15] = {
            0x00000000u, 0x80000000u,              // +-0
            0x0D800000u, 0x0D800001u, 0x0D7FFFFFu,  // 2^-100 and its neighbours (inside, outside)
            0x71800000u, 0x717FFFFFu, 0x71800001u,  // 2^100 and its neighbours (inside, outside)
            0x3F800000u, 0x7F7FFFFFu, 0x00800000u,  // 1, FLT_MAX, the smallest normal
            0x00000001u, 0x007FFFFFu,              // the smallest and the largest denormal
            0x7F800000u, 0x7FC00000u,              // inf, nan
        };
        if (i == 15) return (float)d;  // quotient 1, then just above 1, then a random in-range numerator
        if (i == 16) return __uint_as_float(__float_as_uint((float)d) + 1u);
        if (i == 17) return from_parts(sign, 27 + (int)(h % 200u), h2);
        const unsigned b = kSpecial[i];
        return __uint_as_float(i < 2 ? b : (b | ((d & 1u) << 31)));  // both signs over the divisors
    }
    if (i < 24) return __uint_as_float((sign << 31) | (h & 0x7FFFFFu) | 1u);  // denormals
    if (i < 44) return from_parts(sign, 27 + (int)(h % 200u), h2);          // 2^-100 <= |num| < 2^100
    if (i < 48) return from_parts(sign, 1 + (int)(h % 254u), h2);            // every normal exponent
    // near a midpoint: the odd part D of d, a 24-bit significand M and s with Q = M 2^s / D in [2^24, 2^25) (Q's last
    // bit is the half-ulp bit of the float quotient); M is moved so that M 2^s = r (mod D) with r = 1 or D - 1
    const unsigned D = d >> (__ffs(d) - 1);
    const int ex = -99 + (int)(h % 197u);  // the numerator's exponent
    if (D < 3) return from_parts(sign, 127 + ex, h2);
    unsigned long long M = 0x800000u | (h2 & 0x7FFFFFu);
    int s = 0;
    while ((M << s) < ((unsigned long long)D << 24)) ++s;
    const unsigned long long inv2 = (D + 1) / 2;
    unsigned long long inv = 1;  // 2^-s mod D
    for (int k = 0; k < s; ++k) inv = mulmod(inv, inv2, D);
    const unsigned long long r0 = (M << s) % D, r = (h & 1u) ? 1u : D - 1u;
    const unsigned long long delta = mulmod((r + D - r0) % D, inv, D);
    unsigned long long Mn = M + delta;
    if (Mn >= 0x1000000u) Mn = M + delta - D;
    if (Mn < 0x800000u || Mn >= 0x1000000u) return from_parts(sign, 127 + ex, h2);
    int s2 = 0;
    while ((Mn << s2) < ((unsigned long long)D << 24)) ++s2;
    const unsigned long long q = (Mn << s2) / D, rem = (Mn << s2) % D;
    near_mid = (q & 1u) && (rem == 1u || rem == D - 1u);  // 1/D ulp-of-the-last-bit from a midpoint
    return from_parts(sign, 127 + ex, (unsigned)Mn);
}

// counters: 0 cases, 1 in range (num != 0), 2 in range and != __fdiv_rn, 3 zero numerators, 4 zero numerators breaking
// the sign claim, 5 `bad` wrong, 6 outside the range (num != 0, inf, nan), 7 outside and != __fdiv_rn, 8 within 1/d of
// a midpoint (in range), 9 of those != __fdiv_rn, 10 outside, finite and != __fdiv_rn, 11 outside and finite
__global__ void fdiv_sweep_kernel(unsigned d_lo, unsigned d_hi, int per, unsigned seed, Sink s) {
    unsigned long long c[12] = {};
    const unsigned long long total = (unsigned long long)(d_hi - d_lo + 1) * per;
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < total;
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned d = d_lo + (unsigned)(k / per);
        const int i = (int)(k % per);
        bool near_mid;
        const float num = sweep_numerator(d, i, seed, near_mid);
        const float den = (float)d;
        bool bad = false;
        const float q = fdiv_by_count(num, den, bad);
        const float want = __fdiv_rn(num, den);
        const unsigned a = __float_as_uint(num) & 0x7FFFFFFFu;
        const bool inside = a >= 0x0D800000u && a <= 0x71800000u;
        ++c[0];
        if (bad != (a != 0u && !inside)) {
            ++c[5];
            record(s, 5, __float_as_uint(num), d, bad);
        }
        if (a == 0u) {
            ++c[3];
            // a zero whose sum with any u >= +0 is that sum (+0 + +0 = +0: a -0 would survive only against u = -0)
            if (q != 0.0f || __float_as_uint(__fadd_rn(q, 0.0f)) != 0u) {
                ++c[4];
                record(s, 4, __float_as_uint(num), d, __float_as_uint(q));
            }
        } else if (inside) {
            ++c[1];
            const bool ok = __float_as_uint(q) == __float_as_uint(want);
            if (!ok) {
                ++c[2];
                record(s, 2, __float_as_uint(num), d, __float_as_uint(q));
            }
            if (near_mid) {
                ++c[8];
                c[9] += !ok;
            }
        } else {
            const bool differs = __float_as_uint(q) != __float_as_uint(want) && !(q != q && want != want);
            ++c[6];
            c[7] += differs;
            if (a < 0x7F800000u) {
                ++c[11];
                c[10] += differs;
            }
        }
    }
    for (int j = 0; j < 12; ++j)
        if (c[j]) atomicAdd(&s.count[j], c[j]);
}

// order_key along the float order: every non-NaN pattern x and its successor; counters: 0 pairs, 1 not strictly
// increasing (-0 -> +0: not equal), 2 zero keys
__global__ void order_key_sweep_kernel(Sink s) {
    unsigned long long c[3] = {};
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k < (1ull << 32);
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned x = (unsigned)k;
        if ((x & 0x7FFFFFFFu) > 0x7F800000u) continue;  // NaN
        const unsigned kx = order_key(__uint_as_float(x));
        if (kx == 0u) {
            ++c[2];
            record(s, 2, x, kx, 0);
        }
        if (x == 0x7F800000u) continue;  // +inf: the last
        const unsigned y = x == 0x80000000u ? 0u : ((x >> 31) ? x - 1u : x + 1u);
        const unsigned ky = order_key(__uint_as_float(y));
        ++c[0];
        if (x == 0x80000000u ? ky != kx : ky <= kx) {
            ++c[1];
            record(s, 1, x, kx, ky);
        }
    }
    for (int j = 0; j < 3; ++j)
        if (c[j]) atomicAdd(&s.count[j], c[j]);
}

__device__ __forceinline__ void atomic_max_pos(double *p, double v) {  // v >= 0: the bit patterns order like the values
    atomicMax(reinterpret_cast<unsigned long long *>(p), (unsigned long long)__double_as_longlong(v));
}

// exp_nonpos over every float x <= 0 (and +0) against exp((double)x).  err2: ex2.approx's relative error bound; dc: the
// relative error of the rounded log2(e) constant.  counters: 0 cases, 1 over the bound, 2 denormal results, 3 zero
// although exp(x) is clearly above 2^-126, 4 nonzero although clearly below, 5 exp_nonpos(+-0) != 1, 6 results checked
// against the bound.  maxes: [0] relative error against exp(x), [1] ex2.approx's own relative error (against
// 2^fl(x log2 e)), [2] the largest ratio error / bound
__global__ void exp_sweep_kernel(double err2, double dc, Sink s, double *maxes) {
    unsigned long long c[7] = {};
    double m0 = 0, m1 = 0, m2 = 0;
    const double tiny = 0x1p-126;
    for (unsigned long long k = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; k <= 0x7F800001ull;
         k += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned x = k == 0x7F800001ull ? 0u : 0x80000000u | (unsigned)k;  // -0 .. -inf, then +0
        const float xf = __uint_as_float(x);
        const float y = exp_nonpos(xf);
        const double ref = exp((double)xf);
        ++c[0];
        const unsigned yb = __float_as_uint(y);
        if ((x & 0x7FFFFFFFu) == 0u && yb != 0x3F800000u) {
            ++c[5];
            record(s, 5, x, yb, 0);
        }
        if (yb != 0u && yb < 0x00800000u) {
            ++c[2];
            record(s, 2, x, yb, 0);
        }
        // |t - x log2 e| <= |x| log2 e (dc + 2^-24 + dc 2^-24): the rounded constant and the rounded product
        const double dt = fabs((double)xf) * 1.4426950408889634 * (dc + 0x1p-24 + dc * 0x1p-24);
        const double bound = (1.0 + err2) * exp2(dt) - 1.0;
        if (y == 0.0f) {
            if (ref * (1.0 - bound) >= tiny) {
                ++c[3];
                record(s, 3, x, yb, 0);
            }
            continue;
        }
        if (ref * (1.0 + bound) < tiny) {
            ++c[4];
            record(s, 4, x, yb, 0);
            continue;
        }
        ++c[6];
        const double rel = fabs((double)y - ref) / ref;
        const double t = (double)__fmul_rn(xf, 1.4426950408889634f);
        const double e2 = fabs((double)y - exp2(t)) / exp2(t);
        m0 = fmax(m0, rel);
        m1 = fmax(m1, e2);
        m2 = fmax(m2, rel / bound);
        if (rel > bound) {
            ++c[1];
            record(s, 1, x, yb, 0);
        }
    }
    for (int j = 0; j < 7; ++j)
        if (c[j]) atomicAdd(&s.count[j], c[j]);
    atomic_max_pos(&maxes[0], m0);
    atomic_max_pos(&maxes[1], m1);
    atomic_max_pos(&maxes[2], m2);
}

__global__ void fdiv_map_kernel(const float *num, const float *den, float *q, uint8_t *bad, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool b = false;
    q[i] = fdiv_by_count(num[i], den[i], b);
    bad[i] = b;
}

__global__ void score_map_kernel(const int *N, const float *W, const float *P, const float *sq, float c, float *straight,
                                 uint8_t *bad, float *exact, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool b = false;
    straight[i] = bz::puct_score_straight(N[i], W[i], P[i], sq[i], c, b);
    bad[i] = b;
    exact[i] = bz::puct_score(N[i], W[i], P[i], sq[i], c);
}

__global__ void sqrt_map_kernel(const int *n, float *small, float *full, int cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cnt) return;
    small[i] = bz::sqrt_of_small_count(n[i]);
    full[i] = bz::sqrt_of_count(n[i]);
}

constexpr int kCounters = 16;

// runs a sweep kernel with fresh counters and copies counters and records back
template <typename F>
int run_sweep(F launch, unsigned long long *count_out, unsigned *rec_out, double *maxes_out = nullptr) {
    unsigned long long *count = nullptr;
    unsigned *rec = nullptr;
    double *maxes = nullptr;
    cudaError_t e = cudaMalloc(&count, kCounters * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc(&rec, (1 + 4 * kRecords) * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMalloc(&maxes, 4 * sizeof(double));
    if (e == cudaSuccess) e = cudaMemset(count, 0, kCounters * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(rec, 0, (1 + 4 * kRecords) * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(maxes, 0, 4 * sizeof(double));
    if (e == cudaSuccess) {
        launch(Sink{count, rec}, maxes);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(count_out, count, kCounters * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(rec_out, rec, (1 + 4 * kRecords) * sizeof(unsigned), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && maxes_out) e = cudaMemcpy(maxes_out, maxes, 4 * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(count);
    cudaFree(rec);
    cudaFree(maxes);
    return (int)e;
}

// copies host arrays in, runs a map kernel over n items, copies the outputs back
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { cudaFree(p); }
};

constexpr int kGrid = 148 * 8, kBlock = 256;

}  // namespace

extern "C" {

int puct_fill_sqrt_table() {
    bz::sqrt_table_kernel<<<bz::kSqrtTab / 256, 256>>>();
    const cudaError_t e = cudaGetLastError();
    return (int)(e != cudaSuccess ? e : cudaDeviceSynchronize());
}

int puct_fdiv_sweep(unsigned d_lo, unsigned d_hi, int per, unsigned seed, unsigned long long *count, unsigned *rec) {
    if (d_lo < 1 || d_hi < d_lo || per < 1 || per > 64) return (int)cudaErrorInvalidValue;
    return run_sweep([&](Sink s, double *) { fdiv_sweep_kernel<<<kGrid, kBlock>>>(d_lo, d_hi, per, seed, s); }, count, rec);
}

int puct_order_key_sweep(unsigned long long *count, unsigned *rec) {
    return run_sweep([&](Sink s, double *) { order_key_sweep_kernel<<<kGrid, kBlock>>>(s); }, count, rec);
}

int puct_exp_sweep(double err2, double dc, unsigned long long *count, unsigned *rec, double *maxes) {
    return run_sweep([&](Sink s, double *m) { exp_sweep_kernel<<<kGrid, kBlock>>>(err2, dc, s, m); }, count, rec, maxes);
}

#define PUCT_TO_DEVICE(buf, host, bytes)                                                  \
    do {                                                                                  \
        cudaError_t e_ = cudaMalloc(&(buf).p, (bytes));                                   \
        if (e_ == cudaSuccess && (host)) e_ = cudaMemcpy((buf).p, (host), (bytes), cudaMemcpyHostToDevice); \
        if (e_ != cudaSuccess) return (int)e_;                                            \
    } while (0)

int puct_fdiv_map(const float *num, const float *den, float *q, uint8_t *bad, int n) {
    DevBuf a, b, c, d;
    PUCT_TO_DEVICE(a, num, n * sizeof(float));
    PUCT_TO_DEVICE(b, den, n * sizeof(float));
    PUCT_TO_DEVICE(c, (const float *)nullptr, n * sizeof(float));
    PUCT_TO_DEVICE(d, (const uint8_t *)nullptr, n);
    fdiv_map_kernel<<<(n + 255) / 256, 256>>>((const float *)a.p, (const float *)b.p, (float *)c.p, (uint8_t *)d.p, n);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(q, c.p, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(bad, d.p, n, cudaMemcpyDeviceToHost);
    return (int)e;
}

int puct_score_map(const int *N, const float *W, const float *P, const float *sq, float cp, float *straight, uint8_t *bad,
                   float *exact, int n) {
    DevBuf a, b, c, d, o1, o2, o3;
    PUCT_TO_DEVICE(a, N, n * sizeof(int));
    PUCT_TO_DEVICE(b, W, n * sizeof(float));
    PUCT_TO_DEVICE(c, P, n * sizeof(float));
    PUCT_TO_DEVICE(d, sq, n * sizeof(float));
    PUCT_TO_DEVICE(o1, (const float *)nullptr, n * sizeof(float));
    PUCT_TO_DEVICE(o2, (const uint8_t *)nullptr, n);
    PUCT_TO_DEVICE(o3, (const float *)nullptr, n * sizeof(float));
    score_map_kernel<<<(n + 255) / 256, 256>>>((const int *)a.p, (const float *)b.p, (const float *)c.p, (const float *)d.p, cp,
                                               (float *)o1.p, (uint8_t *)o2.p, (float *)o3.p, n);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(straight, o1.p, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(bad, o2.p, n, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(exact, o3.p, n * sizeof(float), cudaMemcpyDeviceToHost);
    return (int)e;
}

int puct_sqrt_map(const int *n, float *small, float *full, int cnt) {
    DevBuf a, b, c;
    PUCT_TO_DEVICE(a, n, cnt * sizeof(int));
    PUCT_TO_DEVICE(b, (const float *)nullptr, cnt * sizeof(float));
    PUCT_TO_DEVICE(c, (const float *)nullptr, cnt * sizeof(float));
    sqrt_map_kernel<<<(cnt + 255) / 256, 256>>>((const int *)a.p, (float *)b.p, (float *)c.p, cnt);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(small, b.p, cnt * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(full, c.p, cnt * sizeof(float), cudaMemcpyDeviceToHost);
    return (int)e;
}

}  // extern "C"
