// device_math_probe.cu - the device arithmetic of csrc/p2p_kernels.cuh, evaluated over whole input domains.
//
// Every kernel below calls the real __device__ functions of the projection kernels (the header is included, not
// copied), so a change to one of them changes what the tests in tests/test_gpu_device_math.py measure.  Built by that
// test module with the library's own nvcc flags (no fast-math, no flush-to-zero) and loaded with ctypes.  Every
// launcher takes device pointers and returns the cudaError_t of the launch (0 = success).
#include <cuda_runtime.h>
#include <stdint.h>

#include "p2p_kernels.cuh"

using namespace p2p;

namespace {

constexpr int kBlocks = 148 * 8, kBlockThreads = 256;

__device__ __forceinline__ void atomic_add_u64(unsigned long long *p, unsigned long long v) {
    if (v) atomicAdd(p, v);
}

__device__ __forceinline__ uint32_t mix32(uint32_t x) {  // lowbias32 (public domain integer hash)
    x ^= x >> 16;
    x *= 0x7feb352du;
    x ^= x >> 15;
    x *= 0x846ca68bu;
    x ^= x >> 16;
    return x;
}

// every bit pattern in [lo, hi): the fast sqrt against __fsqrt_rn.
// res[0] += mismatches, res[1] = min / res[2] = max mismatching pattern (res[1] must start at ~0).
__global__ void sqrt_kernel(uint32_t lo, uint32_t hi, unsigned long long *res) {
    unsigned long long bad = 0, bmin = ~0ull, bmax = 0;
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += step) {
        const float s = __uint_as_float((uint32_t)i);
        if (__float_as_uint(sqrt_rn_fast(s)) != __float_as_uint(__fsqrt_rn(s))) {
            ++bad;
            bmin = min(bmin, (unsigned long long)i);
            bmax = max(bmax, (unsigned long long)i);
        }
    }
    if (bad) {
        atomicAdd(&res[0], bad);
        atomicMin(&res[1], bmin);
        atomicMax(&res[2], bmax);
    }
}

// div_rn_with_rcp(a, d, rcp_refined(d)) against __fdiv_rn.  Divisor k = mantissa k of [m_lo, m_hi) with exponent
// e_lo + k % n_exp; n_num numerators per divisor, both signs: mantissas 1.0, all ones, d's own and the one below it,
// then seeded ones; exponents such that |a / d| lies in (2^-25, 1].  res[0] += mismatches, res[1..2] = (a, d) bits of
// one mismatch.
__global__ void div_kernel(uint32_t m_lo, uint32_t m_hi, int e_lo, int n_exp, int n_num, uint32_t seed,
                           unsigned long long *res) {
    unsigned long long bad = 0, wa = 0, wd = 0;
    const uint64_t total = (uint64_t)(m_hi - m_lo) * (uint64_t)n_num;
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += step) {
        const uint32_t m = m_lo + (uint32_t)(i / (uint64_t)n_num);
        const int k = (int)(i % (uint64_t)n_num);
        const int ed = e_lo + (int)(m % (uint32_t)n_exp);
        const uint32_t dbits = ((uint32_t)(ed + 127) << 23) | m;
        const float d = __uint_as_float(dbits);
        uint32_t ma;
        switch (k) {
            case 0: ma = 0u; break;
            case 1: ma = 0x7fffffu; break;
            case 2: ma = m; break;
            case 3: ma = (m == 0u) ? 0x7fffffu : m - 1u; break;
            default: ma = mix32(seed ^ mix32(m * 1024u + (uint32_t)k)) & 0x7fffffu;
        }
        int ea = ed - (int)(mix32(seed + 0x9e3779b9u * (uint32_t)k + m) % 25u);
        if (ea == ed && ma > m) --ea;
        if (k == 3 && m == 0u) ea = ed - 1;   // nextafter(d, 0) of a power of two
        const float r = rcp_refined(d);
#pragma unroll
        for (int sgn = 0; sgn < 2; ++sgn) {
            const float a = __uint_as_float(((uint32_t)sgn << 31) | ((uint32_t)(ea + 127) << 23) | ma);
            if (__float_as_uint(div_rn_with_rcp(a, d, r)) != __float_as_uint(__fdiv_rn(a, d))) {
                ++bad;
                wa = __float_as_uint(a);
                wd = dbits;
            }
        }
    }
    if (bad) {
        atomicAdd(&res[0], bad);
        res[1] = wa;
        res[2] = wd;
    }
}

// every float in [0, 32767): round_x32 and quantise against cvRound(f32(x * 32)).
// res[0] += round_x32 mismatches, res[1] += quantise mismatches (sx or sy).
__global__ void round_kernel(uint32_t hi, unsigned long long *res) {
    unsigned long long b0 = 0, b1 = 0;
    const uint64_t step = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += step) {
        const float x = __uint_as_float((uint32_t)i);
        const int want = __float2int_rn(__fmul_rn(x, 32.0f));
        b0 += round_x32(x) != want;
        const QCoord q = quantise(x, x, false);
        b1 += (q.sx != want) || (q.sy != want);
    }
    atomic_add_u64(&res[0], b0);
    atomic_add_u64(&res[1], b1);
}

// elementwise evaluation for the host comparisons.  a == nullptr: a[i] is the float with bit pattern base + i.
//   0 sqrt_rn_fast(a)   1 acos_svml(a)   2 atan2_svml(a, b)   3 atan2_svml_finish(atan2_svml_core(a, b), a, -b)
//   4 acos_fast(a)      5 atan2_fast(a, b)                    6 mirror_phi_fast(a)
__global__ void eval_kernel(int fn, const float *a, const float *b, uint32_t base, long long n, float *out) {
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const float x = a ? a[i] : __uint_as_float(base + (uint32_t)i);
        const float y = b ? b[i] : 0.0f;
        float r;
        switch (fn) {
            case 0: r = sqrt_rn_fast(x); break;
            case 1: r = acos_svml(x); break;
            case 2: r = atan2_svml(x, y); break;
            case 3: r = atan2_svml_finish(atan2_svml_core(x, y), x, -y); break;
            case 4: r = acos_fast(x); break;
            case 5: r = atan2_fast(x, y); break;
            default: r = mirror_phi_fast(x); break;
        }
        out[i] = r;
    }
}

// (y, x) pairs shaped like the operands the projection kernels pass to atan2: the y and x components of a unit ray
// (uniform direction on the sphere, then rounded to f32), both signs of x.  Pair i depends only on (seed, i).
__global__ void unit_pairs_kernel(uint32_t seed, uint64_t first, long long n, float *y, float *x) {
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const uint64_t k = first + (uint64_t)i;
        const uint32_t h1 = mix32(seed ^ mix32((uint32_t)k ^ mix32((uint32_t)(k >> 32) + 0x68e31da4u)));
        const uint32_t h2 = mix32(h1 ^ 0xb5297a4du);
        const double z = 2.0 * ((double)h1 * 0x1p-32) - 1.0;
        const double az = 6.283185307179586 * ((double)h2 * 0x1p-32);
        const double rho = sqrt(fmax(0.0, 1.0 - z * z));
        y[i] = (float)(rho * sin(az));
        x[i] = (float)(rho * cos(az));
    }
}

// accuracy of the minimax functions against the device's double functions.
//   fn 0: acos_fast(a) vs acos   1: atan2_fast(a, b) vs atan2   2: mirror_phi_fast(a) vs pi - a
// a == nullptr: a[i] is the float with bit pattern base + i.  Inputs whose double result is not finite are skipped.
// st[0] += finite results evaluated, st[1] += correctly rounded (among decided), st[2] += undecided: the double value
// lies within 4 double ulps of the midpoint between two floats, so its f32 rounding is not known for sure;
// st[3] = max |error| in ulps of the result's binade, as float bits; st[4] += results more than 1 ulp off;
// st[5] += NaN where the reference is finite.
__global__ void accuracy_kernel(int fn, const float *a, const float *b, uint32_t base, long long n,
                                unsigned long long *st) {
    unsigned long long cnt = 0, cr = 0, und = 0, far = 0, nan = 0;
    float worst = 0.0f;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const float x = a ? a[i] : __uint_as_float(base + (uint32_t)i);
        const float y = b ? b[i] : 0.0f;
        float got;
        double ref;
        if (fn == 0) {
            got = acos_fast(x);
            ref = acos((double)x);
        } else if (fn == 1) {
            got = atan2_fast(x, y);
            ref = atan2((double)x, (double)y);
        } else {
            got = mirror_phi_fast(x);
            ref = 3.141592653589793 - (double)x;   // error < 2^-51: far inside the undecided margin
        }
        if (!isfinite(ref)) continue;
        ++cnt;
        if (got != got) {
            ++nan;
            continue;
        }
        const float rn = __double2float_rn(ref);
        const double ar = fabs(ref);
        const int e = (ar < 0x1p-126) ? -126 : ilogb(ar);
        const double ulp = ldexp(1.0, e - 23);
        const float err = (float)(fabs((double)got - ref) / ulp);
        worst = fmaxf(worst, err);
        far += err > 1.0f;
        // the f32 neighbour on the other side of ref, and the rounding boundary between the two
        const float other = (ref > (double)rn) ? nextafterf(rn, INFINITY) : nextafterf(rn, -INFINITY);
        const double mid = 0.5 * ((double)rn + (double)other);
        const double dulp = ldexp(1.0, ((ar < 0x1p-1022) ? -1022 : ilogb(ar)) - 52);
        if (ref != (double)rn && fabs(ref - mid) <= 4.0 * dulp) {
            ++und;
        } else {
            cr += (__float_as_uint(got) == __float_as_uint(rn));
        }
    }
    atomic_add_u64(&st[0], cnt);
    atomic_add_u64(&st[1], cr);
    atomic_add_u64(&st[2], und);
    if (worst > 0.0f) atomicMax(&st[3], (unsigned long long)__float_as_uint(worst));
    atomic_add_u64(&st[4], far);
    atomic_add_u64(&st[5], nan);
}

}  // namespace

extern "C" {

int probe_sqrt(uint32_t lo, uint32_t hi, unsigned long long *res) {
    sqrt_kernel<<<kBlocks, kBlockThreads>>>(lo, hi, res);
    return (int)cudaGetLastError();
}

int probe_div(uint32_t m_lo, uint32_t m_hi, int e_lo, int n_exp, int n_num, uint32_t seed, unsigned long long *res) {
    div_kernel<<<kBlocks, kBlockThreads>>>(m_lo, m_hi, e_lo, n_exp, n_num, seed, res);
    return (int)cudaGetLastError();
}

int probe_round(uint32_t hi, unsigned long long *res) {
    round_kernel<<<kBlocks, kBlockThreads>>>(hi, res);
    return (int)cudaGetLastError();
}

int probe_eval(int fn, const float *a, const float *b, uint32_t base, long long n, float *out) {
    eval_kernel<<<kBlocks, kBlockThreads>>>(fn, a, b, base, n, out);
    return (int)cudaGetLastError();
}

int probe_unit_pairs(uint32_t seed, unsigned long long first, long long n, float *y, float *x) {
    unit_pairs_kernel<<<kBlocks, kBlockThreads>>>(seed, first, n, y, x);
    return (int)cudaGetLastError();
}

int probe_accuracy(int fn, const float *a, const float *b, uint32_t base, long long n, unsigned long long *st) {
    accuracy_kernel<<<kBlocks, kBlockThreads>>>(fn, a, b, base, n, st);
    return (int)cudaGetLastError();
}

}  // extern "C"
