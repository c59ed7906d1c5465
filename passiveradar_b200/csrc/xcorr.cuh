// xcorr.cuh -- long-lag cross-correlation and the zero-phase IIR decimator of find_channel_offset (reference
// passiveRadar/signal_utils.py:29-32 and :73-78, called once per run at main.py:54 / :83 with 10 000 001 lags).
//
// 1. Zero-phase SOS filter + decimation (scipy.signal.decimate(x, nd) = sosfiltfilt(cheby1 sections, x)[::nd]).
//    Float64 coefficients, state and intermediate.  sosfiltfilt runs the cascade forward over the odd extension
//    (27 samples each side for 4 sections) starting from zi * ext[0], then backward from zi * y[-1].  Both passes are
//    parallel over chunks of `chunk` samples, one thread per chunk: a thread starts `warm` samples before its chunk
//    with zero state and only writes its own chunk (the chunk that begins at the sequence start uses the exact
//    initial state instead).  The error of a warm-started output is the cascade's free response to the missing
//    state, which decays like rho^warm (rho = max |pole|); the host picks warm with rho^warm <= 1e-20 (1188 samples
//    at nd = 1, rho = 0.962), so the difference from a serial pass sits at float64 round-off
//    (tests/test_offset_host.py runs the same scheme in numpy against scipy's sosfiltfilt: <= 1e-12 relative).
//    The backward pass writes every nd-th sample as complex64: the operand of the transform stage.
//
// 2. Circular correlation of size P = L1 * L2 (L1, L2 in {1024, 2048, 4096}), four-step, built from fftcore.cuh's
//    per-group transforms.  n = L2 a + b, k = c + L1 d:
//        X[c + L1 d] = sum_b W_L2^{bd} W_P^{bc} sum_a x[L2 a + b] W_L1^{ac}
//    col_fwd_kernel   columns b (4 adjacent per thread, 32-byte sectors): natural -> permuted over a, times W_P^{bc};
//                     row rho = r T1 + t of Z holds frequency c = perm_freq(t, r)
//    row_fwd_kernel   each row: natural -> permuted over b (X spectrum stays in register layout r T2 + t)
//    row_prod_kernel  Y's row pass, S = X conj(Y) (+ S of earlier x segments); on the last segment the transposed
//                     factorisation starts right away: permuted -> natural over d, times W_P^{cb}
//    col_inv_kernel   columns: permuted -> natural over c; DFT(S)[m] = P sum_i x[i] conj(y[i + m]) in natural order
//                     m = L2 a + b (the DFT matrix is symmetric: no inverse transform, no reordering).  It writes the
//                     requested lag window (descending), and/or |xc| with a (max, first index) reduction.
//    W_P^e = W_P^{e mod 4096} W_P^{4096 (e div 4096)}: two 4096-entry tables built in float64.
#pragma once
#include <cuda_runtime.h>

#include "fftcore.cuh"

namespace prc {
namespace xc {

using fft::cmul;
using fft::cmulc;

// ------------------------------------------------------------------------------------------------ IIR decimator
constexpr int SOS_MAX = 8;
constexpr int SIG_C64 = 0, SIG_I8 = 1, SIG_I16 = 2, SIG_F64 = 3, SIG_C128 = 4;

struct IirParams {
    const void* in;
    int kind;                       // SIG_*
    long long n;                    // input samples
    int ns;                         // sections
    int pad;                        // odd-extension length
    long long ne;                   // n + 2 pad
    int chunk, warm;
    double c[SOS_MAX][5];           // b0 b1 b2 a1 a2 (a0 = 1)
    double zi[SOS_MAX][2];          // sosfilt_zi
    void* yf;                       // forward pass over the extension: double (real) / double2 (complex) [ne]
    float2* out;                    // decimated result, complex64 [nout]
    int nd;
    long long nout;
};

__device__ __forceinline__ double2 operator*(double a, double2 v) { return make_double2(a * v.x, a * v.y); }
__device__ __forceinline__ double2 operator+(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 operator-(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }

template <class T> __device__ __forceinline__ T vzero();
template <> __device__ __forceinline__ double vzero<double>() { return 0.0; }
template <> __device__ __forceinline__ double2 vzero<double2>() { return make_double2(0.0, 0.0); }

template <class T> __device__ __forceinline__ T from_real(double v);
template <> __device__ __forceinline__ double from_real<double>(double v) { return v; }
template <> __device__ __forceinline__ double2 from_real<double2>(double v) { return make_double2(v, 0.0); }

__device__ __forceinline__ float2 to_c64(double v) { return make_float2((float)v, 0.f); }
__device__ __forceinline__ float2 to_c64(double2 v) { return make_float2((float)v.x, (float)v.y); }

template <class T> __device__ __forceinline__ T load_sample(const IirParams& p, long long i);
template <> __device__ __forceinline__ double load_sample<double>(const IirParams& p, long long i) {
    switch (p.kind) {
        case SIG_I8: return (double)static_cast<const signed char*>(p.in)[i];
        case SIG_I16: return (double)static_cast<const short*>(p.in)[i];
        default: return static_cast<const double*>(p.in)[i];
    }
}
template <> __device__ __forceinline__ double2 load_sample<double2>(const IirParams& p, long long i) {
    if (p.kind == SIG_C64) {
        const float2 v = static_cast<const float2*>(p.in)[i];
        return make_double2(v.x, v.y);
    }
    return static_cast<const double2*>(p.in)[i];
}

// 2 e - x of the odd extension.  decimate hands integer arrays to sosfiltfilt as they are, so for int8 / int16 input
// the extension is computed in that integer type and wraps around (only the filter upcasts to float64)
template <class T> __device__ __forceinline__ T odd_point(const IirParams& p, long long ie, long long ix) {
    if (p.kind == SIG_I8) {
        const signed char* v = static_cast<const signed char*>(p.in);
        return from_real<T>((double)(signed char)(2 * (int)v[ie] - (int)v[ix]));
    }
    if (p.kind == SIG_I16) {
        const short* v = static_cast<const short*>(p.in);
        return from_real<T>((double)(short)(2 * (int)v[ie] - (int)v[ix]));
    }
    return 2.0 * load_sample<T>(p, ie) - load_sample<T>(p, ix);
}

// odd extension of sosfiltfilt (scipy.signal._arraytools.odd_ext)
template <class T> __device__ __forceinline__ T ext_sample(const IirParams& p, long long j) {
    if (j < p.pad) return odd_point<T>(p, 0, p.pad - j);
    const long long i = j - p.pad;
    if (i >= p.n) return odd_point<T>(p, p.n - 1, 2 * p.n - 2 - i);
    return load_sample<T>(p, i);
}

// one sample through the cascade, direct form II transposed (scipy's sosfilt)
template <class T> __device__ __forceinline__ T sos_step(T x, T (&z)[SOS_MAX][2], const IirParams& p) {
#pragma unroll
    for (int s = 0; s < SOS_MAX; ++s) {
        if (s < p.ns) {
            const T y = p.c[s][0] * x + z[s][0];
            z[s][0] = (p.c[s][1] * x - p.c[s][3] * y) + z[s][1];
            z[s][1] = p.c[s][2] * x - p.c[s][4] * y;
            x = y;
        }
    }
    return x;
}

template <class T> __device__ __forceinline__ void init_state(T (&z)[SOS_MAX][2], const IirParams& p, T x0) {
#pragma unroll
    for (int s = 0; s < SOS_MAX; ++s) {
        z[s][0] = p.zi[s][0] * x0;
        z[s][1] = p.zi[s][1] * x0;
    }
}

template <class T>
__global__ void __launch_bounds__(32) iir_fwd_kernel(const __grid_constant__ IirParams p) {
    const long long j0 = (long long)(blockIdx.x * blockDim.x + threadIdx.x) * p.chunk;
    if (j0 >= p.ne) return;
    const long long j1 = min(j0 + (long long)p.chunk, p.ne);
    long long j = j0 - p.warm;
    T z[SOS_MAX][2];
    if (j <= 0) {
        j = 0;
        init_state<T>(z, p, ext_sample<T>(p, 0));
    } else {
        init_state<T>(z, p, vzero<T>());
    }
    T* yf = static_cast<T*>(p.yf);
    for (; j < j0; ++j) sos_step<T>(ext_sample<T>(p, j), z, p);
    for (; j < j1; ++j) yf[j] = sos_step<T>(ext_sample<T>(p, j), z, p);
}

// backward pass over reversed yf; sample r of the reversed sequence is extension index ne-1-r, i.e. input index
// i = ne-1-pad-r; every i with i % nd == 0, 0 <= i < n becomes out[i / nd]
template <class T>
__global__ void __launch_bounds__(32) iir_bwd_kernel(const __grid_constant__ IirParams p) {
    const long long r0 = (long long)(blockIdx.x * blockDim.x + threadIdx.x) * p.chunk;
    if (r0 >= p.ne) return;
    const long long r1 = min(r0 + (long long)p.chunk, p.ne);
    const T* yf = static_cast<const T*>(p.yf);
    long long r = r0 - p.warm;
    T z[SOS_MAX][2];
    if (r <= 0) {
        r = 0;
        init_state<T>(z, p, yf[p.ne - 1]);
    } else {
        init_state<T>(z, p, vzero<T>());
    }
    for (; r < r0; ++r) sos_step<T>(yf[p.ne - 1 - r], z, p);
    long long i = p.ne - 1 - p.pad - r;
    int rem = (int)(((i % p.nd) + p.nd) % p.nd);
    for (; r < r1; ++r, --i) {
        const T v = sos_step<T>(yf[p.ne - 1 - r], z, p);
        if (rem == 0 && i >= 0 && i < p.n) p.out[i / p.nd] = to_c64(v);
        rem = rem == 0 ? p.nd - 1 : rem - 1;
    }
}

// ------------------------------------------------------------------------------------------------ four-step FFT
constexpr int NCOL = 4;             // adjacent columns per thread in the column passes: 4 x 8 B = one 32-byte sector

// W_P^e for 0 <= e < P: lo[e & 4095] * hi[e >> 12]
__device__ __forceinline__ float2 twiddle_p(const float2* __restrict__ lo, const float2* __restrict__ hi, long long e) {
    return cmul(lo[e & 4095], hi[e >> 12]);
}

// lo[j] = W_P^j (j < 4096), hi[j] = W_P^{4096 j} (j < P / 4096), evaluated in float64
__global__ void p_twiddle_kernel(float2* lo, float2* hi, long long P) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nhi = P / 4096;
    if (i < 4096) {
        double s, c;
        sincospi(-2.0 * (double)i / (double)P, &s, &c);
        lo[i] = make_float2((float)c, (float)s);
    } else if (i < 4096 + nhi) {
        const long long j = i - 4096;
        double s, c;
        sincospi(-2.0 * (double)(4096 * j) / (double)P, &s, &c);
        hi[j] = make_float2((float)c, (float)s);
    }
}

struct ColFwdParams {
    const float2* src;              // element i of the column-major input is src[off + i] when 0 <= off + i < nsrc, i < lim
    long long off, nsrc, lim;
    float2* Z;                      // [L1][L2], row r T1 + t <-> frequency perm_freq(t, r)
    int L2;
    const float2* tw;               // fftcore tables for L1
    const float2* plo;
    const float2* phi;
};

template <int R1>
__global__ void __launch_bounds__(16 * R1) col_fwd_kernel(const __grid_constant__ ColFwdParams p) {
    using G = fft::Geo<R1>;
    extern __shared__ __align__(16) float2 sm[];
    const int t = threadIdx.x;
    const fft::Smem<R1> S(sm);
    fft::stage_twiddles<R1>(sm, p.tw, t);
    const int b0 = blockIdx.x * NCOL;
    float2 a[NCOL][16];
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) {
        const long long i = (long long)(n1 * G::T + t) * p.L2 + b0;
#pragma unroll
        for (int g = 0; g < NCOL; ++g) {
            const long long q = p.off + i + g;
            a[g][n1] = (i + g < p.lim && q >= 0 && q < p.nsrc) ? p.src[q] : make_float2(0.f, 0.f);
        }
    }
    __syncthreads();
#pragma unroll 1
    for (int g = 0; g < NCOL; ++g) {
        float2 v[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = a[0][r];
        fft::fft_n2p<R1>(v, t, S);
        const long long b = b0 + g;
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const long long c = fft::perm_freq<R1>(t, r);
            p.Z[(long long)(r * G::T + t) * p.L2 + b] = cmul(v[r], twiddle_p(p.plo, p.phi, b * c));
        }
#pragma unroll
        for (int h = 0; h + 1 < NCOL; ++h)
#pragma unroll
            for (int r = 0; r < 16; ++r) a[h][r] = a[h + 1][r];
    }
}

struct RowParams {
    float2* Z;                      // [L1][L2]: column pass output, overwritten in place
    const float2* Xh;               // row_prod: X spectrum (register layout), or nullptr for row_fwd
    float2* S;                      // row_prod: accumulated spectrum of earlier segments
    int L2;
    int acc_in, last;               // row_prod: add S; finish (transposed row pass) instead of storing S
    const float2* tw;               // fftcore tables for L2
    const float2* plo;
    const float2* phi;
};

template <int R2>
__global__ void __launch_bounds__(16 * R2) row_fwd_kernel(const __grid_constant__ RowParams p) {
    using G = fft::Geo<R2>;
    extern __shared__ __align__(16) float2 sm[];
    const int t = threadIdx.x;
    const fft::Smem<R2> S(sm);
    fft::stage_twiddles<R2>(sm, p.tw, t);
    float2* row = p.Z + (long long)blockIdx.x * p.L2;
    float2 v[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) v[n1] = row[n1 * G::T + t];
    __syncthreads();
    fft::fft_n2p<R2>(v, t, S);
#pragma unroll
    for (int r = 0; r < 16; ++r) row[r * G::T + t] = v[r];
}

template <int R1, int R2>
__global__ void __launch_bounds__(16 * R2) row_prod_kernel(const __grid_constant__ RowParams p) {
    using G = fft::Geo<R2>;
    extern __shared__ __align__(16) float2 sm[];
    const int t = threadIdx.x;
    const fft::Smem<R2> S(sm);
    fft::stage_twiddles<R2>(sm, p.tw, t);
    const long long base = (long long)blockIdx.x * p.L2;
    float2* row = p.Z + base;
    float2 v[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) v[n1] = row[n1 * G::T + t];
    __syncthreads();
    fft::fft_n2p<R2>(v, t, S);
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        float2 s = cmulc(p.Xh[base + r * G::T + t], v[r]);          // X conj(Y)
        if (p.acc_in) s = fft::cadd(s, p.S[base + r * G::T + t]);
        v[r] = s;
    }
    if (!p.last) {
#pragma unroll
        for (int r = 0; r < 16; ++r) p.S[base + r * G::T + t] = v[r];
        return;
    }
    fft::fft_p2n<R2>(v, t, S);                                       // natural b = n1 T2 + t
    const int T1 = 16 * R1;
    const long long c = fft::perm_freq<R1>((int)blockIdx.x % T1, (int)blockIdx.x / T1);
#pragma unroll
    for (int n1 = 0; n1 < 16; ++n1) {
        const long long b = n1 * G::T + t;
        row[b] = cmul(v[n1], twiddle_p(p.plo, p.phi, b * c));
    }
}

struct ColInvParams {
    const float2* Z;                // row-pass output, rows in register layout of the column transform
    int L2;
    long long nt;                   // lags of this tile: natural m < nt is output j = j_hi - m
    long long j_hi;
    float scale;                    // 1 / P
    float2* out;                    // complex lags (xcorr) or nullptr
    float* absout;                  // |xc| or nullptr
    unsigned long long* best;       // (bits(|xc|) << 32 | ~j) max-reduction, or nullptr
    int real;                       // |Re| instead of |.| (real inputs: the imaginary part is round-off)
    const float2* tw;               // fftcore tables for L1
};

template <int R1>
__global__ void __launch_bounds__(16 * R1) col_inv_kernel(const __grid_constant__ ColInvParams p) {
    using G = fft::Geo<R1>;
    extern __shared__ __align__(16) float2 sm[];
    __shared__ unsigned long long red[16 * R1 / 32];
    const int t = threadIdx.x;
    const fft::Smem<R1> S(sm);
    fft::stage_twiddles<R1>(sm, p.tw, t);
    const int b0 = blockIdx.x * NCOL;
    float2 a[NCOL][16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const float2* src = p.Z + (long long)(r * G::T + t) * p.L2 + b0;
#pragma unroll
        for (int g = 0; g < NCOL; ++g) a[g][r] = src[g];
    }
    __syncthreads();
    unsigned long long mine = 0ull;
#pragma unroll 1
    for (int g = 0; g < NCOL; ++g) {
        float2 v[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = a[0][r];
        fft::fft_p2n<R1>(v, t, S);                                   // natural a = n1 T1 + t
        const long long b = b0 + g;
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const long long m = (long long)(n1 * G::T + t) * p.L2 + b;
            if (m < p.nt) {
                const long long j = p.j_hi - m;
                const float2 w = make_float2(v[n1].x * p.scale, v[n1].y * p.scale);
                if (p.out) p.out[j] = w;
                if (p.absout || p.best) {
                    const float av = p.real ? fabsf(w.x) : sqrtf(w.x * w.x + w.y * w.y);
                    if (p.absout) p.absout[j] = av;
                    const unsigned long long key =
                        ((unsigned long long)__float_as_uint(av) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)j);
                    mine = key > mine ? key : mine;
                }
            }
        }
#pragma unroll
        for (int h = 0; h + 1 < NCOL; ++h)
#pragma unroll
            for (int r = 0; r < 16; ++r) a[h][r] = a[h + 1][r];
    }
    if (!p.best) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, mine, o);
        mine = other > mine ? other : mine;
    }
    if ((t & 31) == 0) red[t >> 5] = mine;
    __syncthreads();
    if (t == 0) {
        for (int w = 1; w < G::T / 32; ++w) mine = red[w] > mine ? red[w] : mine;
        atomicMax(p.best, mine);
    }
}

// offset = (argmax - nl) * nd from the reduction key (first index on ties: the key keeps the smallest j)
__global__ void offset_kernel(const unsigned long long* best, long long nl, int nd, long long* offset) {
    const long long j = (long long)(0xFFFFFFFFu - (unsigned)(*best & 0xFFFFFFFFull));
    *offset = (j - nl) * (long long)nd;
}

}  // namespace xc
}  // namespace prc
