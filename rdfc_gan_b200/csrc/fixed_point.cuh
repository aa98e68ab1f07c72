// Deterministic scatters (the *_ex entry points with RDFC_DETERMINISTIC): 64-bit fixed-point accumulation.
//
// A scatter whose destinations receive contributions from many threads sums them as two's-complement integers
// (red.global.add.u64) instead of fp32 / fp64 atomics.  Integer addition is associative, so the result does not depend on the
// order in which the threads arrive.  Each contribution c is stored as round(c * 2^k); k comes from an upper bound on the sum
// of |contributions| at any one destination, bound = count * product of maxima, so that bound * 2^k < 2^62: no sum can overflow,
// and one integer step is 2^-62 of the bound or less.  The maxima are found on the device (no host synchronisation) and kept as
// the bit patterns of non-negative doubles, which order like unsigned integers with NaN above +Inf; a non-finite maximum makes
// the conversion write NaN, so a NaN or Inf input never turns into finite numbers.
#pragma once
#include "common.cuh"

namespace rdfc {
namespace {

__device__ __forceinline__ unsigned long long fx_bits(double v) { return (unsigned long long)__double_as_longlong(fabs(v)); }

// max over the warp, then one atomicMax per warp; every lane of the warp must call it
__device__ __forceinline__ void fx_warp_max(unsigned long long m, unsigned long long *am) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, m, s);
        m = o > m ? o : m;
    }
    if ((threadIdx.x & 31) == 0 && m) atomicMax(am, m);
}

__device__ __forceinline__ void fx_add(long long *p, long long v) {
    atomicAdd(reinterpret_cast<unsigned long long *>(p), (unsigned long long)v);
}

// the exponent k for bound = count * am[0] * ... * am[n-1]; ok = false when a maximum is not finite
struct FxExp { int k; bool ok; };
__device__ __forceinline__ FxExp fx_exponent(double count, const unsigned long long *am, int n) {
    int e, E;
    frexp(count, &E);                                   // count < 2^E
    bool zero = false, ok = true;
    for (int i = 0; i < n; ++i) {
        const unsigned long long b = am[i];
        if (b >= 0x7ff0000000000000ull) ok = false;
        else if (b == 0) zero = true;                   // every contribution is zero
        else { frexp(__longlong_as_double((long long)b), &e); E += e; }
    }
    return FxExp{zero ? 0 : 62 - E, ok};
}

template <typename T> struct Fx;

// fp32: 2^k applied as two exact power-of-two factors, each a normal float (|k| <= 252 covers every finite fp32 bound: a
// product of three fp32 maxima and a count < 2^31 stays below 2^420, and a larger k only meets contributions that are zero)
template <> struct Fx<float> {
    float up1, up2, dn1, dn2;
    bool ok;
    __device__ __forceinline__ Fx(double count, const unsigned long long *am, int n) {
        const FxExp x = fx_exponent(count, am, n);
        const int k = x.k > 252 ? 252 : (x.k < -252 ? -252 : x.k), k1 = k / 2, k2 = k - k1;
        up1 = __int_as_float((127 + k1) << 23); up2 = __int_as_float((127 + k2) << 23);
        dn1 = __int_as_float((127 - k1) << 23); dn2 = __int_as_float((127 - k2) << 23);
        ok = x.ok;
    }
    __device__ __forceinline__ long long to_fixed(float v) const { return __float2ll_rn(v * up1 * up2); }
    __device__ __forceinline__ float from_fixed(long long q) const { return ok ? __ll2float_rn(q) * dn1 * dn2 : __int_as_float(0x7fffffff); }
};

template <> struct Fx<double> {
    int k;
    bool ok;
    __device__ __forceinline__ Fx(double count, const unsigned long long *am, int n) {
        const FxExp x = fx_exponent(count, am, n);
        k = x.k; ok = x.ok;
    }
    __device__ __forceinline__ long long to_fixed(double v) const { return __double2ll_rn(ldexp(v, k)); }
    __device__ __forceinline__ double from_fixed(long long q) const { return ok ? ldexp((double)q, -k) : __longlong_as_double(0x7fffffffffffffffll); }
};

// am[0] = max |x| over n elements (am zero-initialised by the caller)
template <typename T>
__global__ void __launch_bounds__(256) fx_amax_kernel(const T *__restrict__ x, long long n, unsigned long long *__restrict__ am) {
    unsigned long long m = 0;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
        const unsigned long long b = fx_bits((double)x[i]);
        m = b > m ? b : m;
    }
    fx_warp_max(m, am);
}

// out[i] = acc[i] / 2^k with the scale the scatter used
template <typename T>
__global__ void __launch_bounds__(256) fx_convert_kernel(const long long *__restrict__ acc, T *__restrict__ out, long long n, double count,
                                                         const unsigned long long *__restrict__ am, int nam) {
    const Fx<T> fx(count, am, nam);
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256) out[i] = fx.from_fixed(acc[i]);
}

inline int fx_blocks(long long n) { return (int)min((long long)cdiv(n, 256), (long long)sm_count() * 8); }

template <typename T>
int fx_amax(const T *x, long long n, unsigned long long *am, cudaStream_t st) {
    if (n == 0) return 0;
    fx_amax_kernel<T><<<fx_blocks(n), 256, 0, st>>>(x, n, am);
    RDFC_CHECK_LAUNCH("fx_amax_kernel");
    return 0;
}

template <typename T>
int fx_convert(const long long *acc, T *out, long long n, double count, const unsigned long long *am, int nam, cudaStream_t st) {
    fx_convert_kernel<T><<<fx_blocks(n), 256, 0, st>>>(acc, out, n, count, am, nam);
    RDFC_CHECK_LAUNCH("fx_convert_kernel");
    return 0;
}

}  // namespace
}  // namespace rdfc
