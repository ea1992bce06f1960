// Probe kernels for tests/test_device_numerics.py: the hand-written numeric primitives of the step kernels, swept
// over their documented domains on the device and compared with the CUDA intrinsics they stand in for.  Built by the
// test with the library's own flags; the integer float32 -> float64 route is on, as in swarm_step_rotx.cu.
#define SWARM_ROT_INT_CVT 1
#include "swarm_rot_common.cuh"

#include <cuda_runtime.h>

struct ProbeResult {   // (outside the anonymous namespace: the exported probe_run takes it)
    unsigned long long checked, bad;
    unsigned long long first[8];   // the first failing inputs (in launch order, not sorted)
};

namespace {

__device__ void note(ProbeResult* r, bool ok, unsigned long long input) {
    if (ok) return;
    const unsigned long long k = atomicAdd(&r->bad, 1ull);
    if (k < 8) r->first[k] = input;
}

__device__ unsigned long long mix64(unsigned long long x) {   // splitmix64 finaliser: the sample generator
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

enum Test : int {
    kSqrt = 0,          // sqrt_rn_fast(s) == __fsqrt_rn(s)
    kNegSqrt2 = 1,      // neg_sqrt_rn_fast2(-s0, -s1) == (-sqrt(s0), -sqrt(s1)); s1 runs the range backwards
    kPosCvt = 2,        // f64_of_pos_f32<true>(a) == (double)a
    kNegCvt = 3,        // f64_of_neg_f32(a) == (double)a
    kPosTiny = 4,       // zero / denormal a: |f64_of_pos_f32<true>(a)| < 2^-125
    kNegTiny = 5,       // the same for f64_of_neg_f32
    kSumsq = 6,         // sumsq1d_fast by the integer route == by conversions, whenever that sum is >= 2^-28
    kMeanFixed = 7,     // mean_markstein == __ddiv_rn: sums are multiples of 2^-37 below 2^16 (param = n)
    kMeanWide = 8,      // ... positive doubles in [2^-40, 2^40]
    kMeanBoundary = 9,  // ... sums whose exact quotient lies within a few ulps of a rounding boundary
};

__device__ double mean_sum(int test, unsigned long long i, int n) {
    const unsigned long long h = mix64(i * 0x100000001B3ull + (unsigned long long)n);
    if (test == kMeanFixed) return (double)(h >> 11) * 0x1p-37;                 // < 2^53 * 2^-37 = 2^16
    if (test == kMeanWide) {
        const double m = 1.0 + (double)(h >> 12) * 0x1p-52;                      // [1, 2)
        return ldexp(m, (int)(mix64(h) % 80ull) - 40);                           // [2^-40, 2^40)
    }
    // boundary: q in [1, 2^10), the midpoint between q and its successor times n, nudged by -3..3 ulps of the sum
    const double q = ldexp(1.0 + (double)(h >> 12) * 0x1p-52, (int)(mix64(h) % 10ull));
    const double half_ulp = (__longlong_as_double(__double_as_longlong(q) + 1) - q) * 0.5;
    const double s = __fma_rn((double)n, q, (double)n * half_ulp);
    const long long nudge = (long long)(mix64(h + 1) % 7ull) - 3;
    return __longlong_as_double(__double_as_longlong(s) + nudge);
}

__global__ void probe_kernel(int test, unsigned long long lo, unsigned long long hi, int param, ProbeResult* r) {
    unsigned long long checked = 0;
    for (unsigned long long i = lo + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i <= hi;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned b = (unsigned)i;
        const float a = __uint_as_float(b);
        switch (test) {
            case kSqrt:
                note(r, __float_as_uint(swarm::sqrt_rn_fast(a)) == __float_as_uint(__fsqrt_rn(a)), i);
                ++checked;
                break;
            case kNegSqrt2: {
                const float a1 = __uint_as_float((unsigned)(hi - (i - lo)));
                float r0, r1;
                swarm::unpack2(swarm::neg_sqrt_rn_fast2(-a, -a1), r0, r1);
                note(r, __float_as_uint(r0) == __float_as_uint(-__fsqrt_rn(a)) &&
                            __float_as_uint(r1) == __float_as_uint(-__fsqrt_rn(a1)), i);
                ++checked;
                break;
            }
            case kPosCvt:
                note(r, __double_as_longlong(swarm::f64_of_pos_f32<true>(a)) == __double_as_longlong((double)a), i);
                ++checked;
                break;
            case kNegCvt:
                note(r, __double_as_longlong(swarm::f64_of_neg_f32(a)) == __double_as_longlong((double)a), i);
                ++checked;
                break;
            case kPosTiny:
                note(r, fabs(swarm::f64_of_pos_f32<true>(a)) < 0x1p-125, i);
                ++checked;
                break;
            case kNegTiny:
                note(r, fabs(swarm::f64_of_neg_f32(a)) < 0x1p-125, i);
                ++checked;
                break;
            case kSumsq: {
                // one component whose square is zero or denormal (|x| < 2^-63), the others spread over 2^-20 .. 2^4
                const unsigned long long h = mix64(i);
                const float x = __uint_as_float((unsigned)(h & 0x807FFFFFu) | ((unsigned)(27 + (h >> 23) % 37) << 23));
                const float y = __uint_as_float((unsigned)((h >> 32) & 0x807FFFFFu) | ((unsigned)(107 + (h >> 55) % 24) << 23));
                const unsigned long long g = mix64(h);
                const float z = (g & 1) ? x * __uint_as_float(0x3F000000u | (unsigned)((g >> 8) & 0x7FFFFF))
                                        : __uint_as_float((unsigned)((g >> 1) & 0x807FFFFFu) | ((unsigned)(100 + (g >> 40) % 31) << 23));
                const float px = __fmul_rn(x, x), py = __fmul_rn(y, y), pz = __fmul_rn(z, z);
                const float ref = __double2float_rn(__dadd_rn(__dadd_rn((double)px, (double)py), (double)pz));
                if (ref >= 0x1p-28f) {
                    const float fast = swarm::sumsq1d_fast(y, x, z);   // the tiny square in the middle as well
                    const float ref2 = __double2float_rn(__dadd_rn(__dadd_rn((double)py, (double)px), (double)pz));
                    note(r, __float_as_uint(fast) == __float_as_uint(ref2) &&
                                __float_as_uint(swarm::sumsq1d_fast(x, y, z)) == __float_as_uint(ref), i);
                    ++checked;
                }
                break;
            }
            default: {
                const double n = (double)param;
                const double s = mean_sum(test, i, param);
                const double want = __ddiv_rn(s, n);
                const double got = swarm::mean_markstein(s, n, __ddiv_rn(1.0, n));
                note(r, __double_as_longlong(got) == __double_as_longlong(want), i);
                ++checked;
            }
        }
    }
    atomicAdd(&r->checked, checked);
}

__global__ void mean_samples_kernel(int test, int n, int count, double* sums, double* quots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    sums[i] = mean_sum(test, (unsigned long long)i, n);
    quots[i] = __ddiv_rn(sums[i], (double)n);
}

}  // namespace

extern "C" {

// Runs one sweep over the inputs lo..hi (float32 bit patterns, or sample indices for the mean tests) and copies the
// result to *out.  Returns a cudaError_t.
int probe_run(int test, unsigned long long lo, unsigned long long hi, int param, ProbeResult* out) {
    ProbeResult* dev = nullptr;
    cudaError_t err = cudaMalloc(&dev, sizeof(ProbeResult));
    if (err != cudaSuccess) return (int)err;
    err = cudaMemset(dev, 0, sizeof(ProbeResult));
    if (err == cudaSuccess) {
        probe_kernel<<<148 * 16, 256>>>(test, lo, hi, param, dev);
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaMemcpy(out, dev, sizeof(ProbeResult), cudaMemcpyDeviceToHost);
    cudaFree(dev);
    return (int)err;
}

// The sums of sample indices 0..count-1 of a mean test and their __ddiv_rn quotients, for a host-side check.
int probe_mean_samples(int test, int n, int count, double* sums, double* quots) {
    double* dev = nullptr;
    cudaError_t err = cudaMalloc(&dev, 2 * sizeof(double) * (size_t)count);
    if (err != cudaSuccess) return (int)err;
    mean_samples_kernel<<<(count + 255) / 256, 256>>>(test, n, count, dev, dev + count);
    err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaMemcpy(sums, dev, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost);
    if (err == cudaSuccess) err = cudaMemcpy(quots, dev + count, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost);
    cudaFree(dev);
    return (int)err;
}

}  // extern "C"
