// Block-cooperative mixed-radix Stockham FFT over lines resident in shared memory.
//
// Every transform on the hot path (standalone fft2/ifft2 and the fused data-consistency kernels) runs
// through block_fft<>: `nlines` independent length-n complex lines live in shared memory (line l at
// base + l*ls), all threads of the CTA share the butterflies of one autosort stage, two buffers ping-pong
// between stages.  Radices 4, 2, 3, 5 are register butterflies; any other prime factor is handled by a
// generic O(p^2) shared-to-shared stage so every length works (the reference's tests use 3, 6, 10 ...).
// Twiddles come from an exact (double-precision generated) table exp(-2*pi*i*k/n) staged in shared memory.
#pragma once
#include "common.cuh"

namespace mrb {

constexpr int kMaxStages = 20;
constexpr int kMaxFftLen = 8192;

struct FftPlan {
    int n;
    int nstages;
    int ls;  // shared-memory line stride in float2 (n or n+1: keeps column-strip loads conflict free)
    int radix[kMaxStages];
    const float2* tw;  // device, [n]
};

// host: builds (and caches per device) the plan for length n. Returns MRB_* code.
int get_fft_plan(int n, FftPlan* plan);

__host__ __device__ inline size_t fft_smem_bytes(const FftPlan& p, int nlines) {
    return (size_t)(2 * (size_t)nlines * p.ls + p.n) * sizeof(float2);
}

// Stage twiddle table into shared memory (call once per CTA, then __syncthreads()).
__device__ __forceinline__ void load_twiddles(float2* tw_s, const FftPlan& p) {
    for (int i = threadIdx.x; i < p.n; i += blockDim.x) tw_s[i] = p.tw[i];
}

template <bool INV>
__device__ __forceinline__ float2 twd(const float2* tw_s, int idx) {
    float2 w = tw_s[idx];
    if (INV) w.y = -w.y;
    return w;
}

// multiply by -i (forward) / +i (inverse)
template <bool INV>
__device__ __forceinline__ float2 mul_mi(float2 a) {
    return INV ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x);
}

template <int R, bool INV>
__device__ __forceinline__ void butterfly(float2* v) {
    if (R == 2) {
        float2 a = v[0], b = v[1];
        v[0] = cadd(a, b);
        v[1] = csub(a, b);
    } else if (R == 4) {
        float2 t0 = cadd(v[0], v[2]), t1 = csub(v[0], v[2]);
        float2 t2 = cadd(v[1], v[3]), t3 = mul_mi<INV>(csub(v[1], v[3]));
        v[0] = cadd(t0, t2);
        v[1] = cadd(t1, t3);
        v[2] = csub(t0, t2);
        v[3] = csub(t1, t3);
    } else if (R == 3) {
        const float s = 0.86602540378443864676f;
        float2 t1 = cadd(v[1], v[2]);
        float2 t2 = make_float2(v[0].x - 0.5f * t1.x, v[0].y - 0.5f * t1.y);
        float2 t3 = mul_mi<INV>(cscale(csub(v[1], v[2]), s));
        v[0] = cadd(v[0], t1);
        v[1] = cadd(t2, t3);
        v[2] = csub(t2, t3);
    } else if (R == 5) {
        const float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
        const float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
        float2 p1 = cadd(v[1], v[4]), m1 = csub(v[1], v[4]);
        float2 p2 = cadd(v[2], v[3]), m2 = csub(v[2], v[3]);
        float2 a0 = v[0];
        float2 A = make_float2(a0.x + c1 * p1.x + c2 * p2.x, a0.y + c1 * p1.y + c2 * p2.y);
        float2 B = make_float2(a0.x + c2 * p1.x + c1 * p2.x, a0.y + c2 * p1.y + c1 * p2.y);
        float2 U = mul_mi<INV>(make_float2(s1 * m1.x + s2 * m2.x, s1 * m1.y + s2 * m2.y));
        float2 V = mul_mi<INV>(make_float2(s2 * m1.x - s1 * m2.x, s2 * m1.y - s1 * m2.y));
        v[0] = make_float2(a0.x + p1.x + p2.x, a0.y + p1.y + p2.y);
        v[1] = cadd(A, U);
        v[4] = csub(A, U);
        v[2] = cadd(B, V);
        v[3] = csub(B, V);
    }
}

template <int R, bool INV>
__device__ __forceinline__ void fft_stage(const float2* __restrict__ src, float2* __restrict__ dst, int nlines,
                                          int n, int ls, int Ns, const float2* __restrict__ tw_s) {
    const int nb = n / R;
    const int total = nlines * nb;
    const int twmul = n / (Ns * R);
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int line = t / nb;
        const int j = t - line * nb;
        const int k = j % Ns;
        const float2* s = src + (size_t)line * ls;
        float2* d = dst + (size_t)line * ls;
        float2 v[R];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = s[j + r * nb];
        if (Ns > 1) {
#pragma unroll
            for (int r = 1; r < R; ++r) v[r] = cmul(v[r], twd<INV>(tw_s, r * k * twmul));
        }
        butterfly<R, INV>(v);
        const int base = (j - k) * R + k;
#pragma unroll
        for (int r = 0; r < R; ++r) d[base + r * Ns] = v[r];
    }
}

// Any radix (used for prime factors other than 2, 3, 5): one thread per output element.
template <bool INV>
__device__ __forceinline__ void fft_stage_generic(const float2* __restrict__ src, float2* __restrict__ dst,
                                                  int nlines, int n, int ls, int Ns, int R,
                                                  const float2* __restrict__ tw_s) {
    const int nb = n / R;
    const int total = nlines * n;
    const int twmul = n / (Ns * R);
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int line = t / n;
        const int o = t - line * n;
        const int j = o / R;
        const int q = o - j * R;
        const int k = j % Ns;
        const float2* s = src + (size_t)line * ls;
        // fp64 running sum: a p-term fp32 sum rounds at every step (1.6e-6 rel-L2 at p = 8191, 1.2e-6 at 4093, against a
        // 2e-6 contract per transform); in fp64 only the fp32 twiddles and inputs round
        double ax = 0.0, ay = 0.0;
        // twiddle exponent e(r) = (r k twmul + ((r q) mod R) nb) mod n, advanced incrementally in 32-bit arithmetic (the
        // 64-bit modulo of the closed form cost more than the whole butterfly: 232 = 8 x 29 spent 7x the time of a
        // power-of-two length in this stage)
        const int step1 = (int)(((long long)k * twmul) % n);
        int e1 = 0, rq = 0;
        for (int r = 0; r < R; ++r) {
            int e = e1 + rq * nb;
            if (e >= n) e -= n;
            float2 w = twd<INV>(tw_s, e);
            float2 x = s[j + r * nb];
            ax += (double)x.x * w.x - (double)x.y * w.y;
            ay += (double)x.x * w.y + (double)x.y * w.x;
            e1 += step1;
            if (e1 >= n) e1 -= n;
            rq += q;
            if (rq >= R) rq -= R;
        }
        dst[(size_t)line * ls + (j - k) * R + k + q * Ns] = make_float2((float)ax, (float)ay);
    }
}

// ---- fixed-plan fast path (compile-time length and radices: 320 = 5*8*8, 640 = 10*8*8) --------------------------
// All index arithmetic folds to constants, radix-8/10 butterflies stay in registers, three shared-memory passes.
template <bool INV>
__device__ __forceinline__ void bf8(float2* v) {
    const float h = 0.70710678118654752440f;
    float2 e0 = cadd(v[0], v[4]), e1 = cadd(v[1], v[5]), e2 = cadd(v[2], v[6]), e3 = cadd(v[3], v[7]);
    float2 o0 = csub(v[0], v[4]), o1 = csub(v[1], v[5]), o2 = csub(v[2], v[6]), o3 = csub(v[3], v[7]);
    // o[n] *= w8^n ; w8 = exp(-+ 2 pi i / 8)
    o1 = INV ? make_float2(h * (o1.x - o1.y), h * (o1.x + o1.y)) : make_float2(h * (o1.x + o1.y), h * (o1.y - o1.x));
    o2 = mul_mi<INV>(o2);
    o3 = INV ? make_float2(-h * (o3.x + o3.y), h * (o3.x - o3.y)) : make_float2(h * (o3.y - o3.x), -h * (o3.x + o3.y));
    float2 e[4] = {e0, e1, e2, e3}, o[4] = {o0, o1, o2, o3};
    butterfly<4, INV>(e);
    butterfly<4, INV>(o);
    v[0] = e[0]; v[2] = e[1]; v[4] = e[2]; v[6] = e[3];
    v[1] = o[0]; v[3] = o[1]; v[5] = o[2]; v[7] = o[3];
}

template <bool INV>
__device__ __forceinline__ void bf10(float2* v) {
    float2 e[5] = {v[0], v[2], v[4], v[6], v[8]}, o[5] = {v[1], v[3], v[5], v[7], v[9]};
    butterfly<5, INV>(e);
    butterfly<5, INV>(o);
    // w10^k, k = 1..4 : exp(-+ 2 pi i k / 10)
    const float c1 = 0.80901699437494742410f, s1 = 0.58778525229247312917f;
    const float c2 = 0.30901699437494742410f, s2 = 0.95105651629515357212f;
    const float2 w1 = make_float2(c1, INV ? s1 : -s1), w2 = make_float2(c2, INV ? s2 : -s2);
    const float2 w3 = make_float2(-c2, INV ? s2 : -s2), w4 = make_float2(-c1, INV ? s1 : -s1);
    o[1] = cmul(o[1], w1); o[2] = cmul(o[2], w2); o[3] = cmul(o[3], w3); o[4] = cmul(o[4], w4);
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        v[k] = cadd(e[k], o[k]);
        v[k + 5] = csub(e[k], o[k]);
    }
}

template <int R, bool INV>
__device__ __forceinline__ void bf_fixed(float2* v) {
    if (R == 8) bf8<INV>(v);
    else if (R == 10) bf10<INV>(v);
    else butterfly<R, INV>(v);
}

template <int N, int R, int NS, bool INV>
__device__ __forceinline__ void fft_stage_fixed(const float2* __restrict__ src, float2* __restrict__ dst, int nlines,
                                                int ls, const float2* __restrict__ tw_s) {
    constexpr int NB = N / R;
    constexpr int TWMUL = N / (NS * R);
    const int total = nlines * NB;
    for (int t = threadIdx.x; t < total; t += blockDim.x) {
        const int line = t / NB;
        const int j = t - line * NB;
        const int k = (NS == 1) ? 0 : (j % NS);
        const float2* s = src + line * ls;
        float2* d = dst + line * ls;
        float2 v[R];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = s[j + r * NB];
        if (NS > 1) {
#pragma unroll
            for (int r = 1; r < R; ++r) v[r] = cmul(v[r], twd<INV>(tw_s, r * k * TWMUL));
        }
        bf_fixed<R, INV>(v);
        const int base = (j - k) * R + k;
#pragma unroll
        for (int r = 0; r < R; ++r) d[base + r * NS] = v[r];
    }
}

template <int N, int R1, int R2, int R3, bool INV>
__device__ __forceinline__ void block_fft_fixed3(float2* A, float2* B, int nlines, int ls, const float2* tw_s) {
    static_assert(R1 * R2 * R3 == N, "radices must multiply to N");
    __syncthreads();
    fft_stage_fixed<N, R1, 1, INV>(B, A, nlines, ls, tw_s);  // 3 stages: input in B, result in A
    __syncthreads();
    fft_stage_fixed<N, R2, R1, INV>(A, B, nlines, ls, tw_s);
    __syncthreads();
    fft_stage_fixed<N, R3, R1 * R2, INV>(B, A, nlines, ls, tw_s);
    __syncthreads();
}

// Which buffer the caller must fill so that the result of block_fft lands in A.
__device__ __forceinline__ float2* fft_start_buf(const FftPlan& p, float2* A, float2* B) {
    return (p.nstages & 1) ? B : A;
}

// All threads of the CTA must call this. Input in fft_start_buf(), output in A.  Ends with __syncthreads().
template <bool INV>
__device__ __forceinline__ void block_fft(float2* A, float2* B, int nlines, const FftPlan& p,
                                          const float2* tw_s) {
    if (p.n == 320) { block_fft_fixed3<320, 5, 8, 8, INV>(A, B, nlines, p.ls, tw_s); return; }
    if (p.n == 640) { block_fft_fixed3<640, 10, 8, 8, INV>(A, B, nlines, p.ls, tw_s); return; }
    float2* src = fft_start_buf(p, A, B);
    float2* dst = (src == A) ? B : A;
    int Ns = 1;
    __syncthreads();
    for (int s = 0; s < p.nstages; ++s) {
        const int R = p.radix[s];
        switch (R) {
            case 4: fft_stage<4, INV>(src, dst, nlines, p.n, p.ls, Ns, tw_s); break;
            case 2: fft_stage<2, INV>(src, dst, nlines, p.n, p.ls, Ns, tw_s); break;
            case 3: fft_stage<3, INV>(src, dst, nlines, p.n, p.ls, Ns, tw_s); break;
            case 5: fft_stage<5, INV>(src, dst, nlines, p.n, p.ls, Ns, tw_s); break;
            default: fft_stage_generic<INV>(src, dst, nlines, p.n, p.ls, Ns, R, tw_s); break;
        }
        Ns *= R;
        float2* t = src;
        src = dst;
        dst = t;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Register-resident building blocks of the 320-point transforms (320 = 16 x 20): used by the fused hybrid-space DC
// gradient (dc.cu, r320::row_dc320_kernel) and by the standalone 320-point line / column FFT (fft.cu).
// ---------------------------------------------------------------------------------------------------------------
namespace r320 {
template <bool INV>
__device__ __forceinline__ float2 mulw(float2 a, float wr, float wi) {  // a * (wr + i*wi), conjugated for the inverse
    return INV ? make_float2(a.x * wr + a.y * wi, a.y * wr - a.x * wi) : make_float2(a.x * wr - a.y * wi, a.x * wi + a.y * wr);
}

// Packed complex arithmetic: a complex value lives in one 64-bit register pair and the additions / real scalings of
// the butterflies are single add / sub / fma .f32x2 instructions (the kernel is instruction-issue bound); multiplications
// by +-i and by constant twiddles stay scalar (immediate-operand FMUL / FFMA on the two halves).
typedef unsigned long long cx;
__device__ __forceinline__ cx pk(float x, float y) {
    cx r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y));
    return r;
}
__device__ __forceinline__ cx pk(float2 a) { return pk(a.x, a.y); }
__device__ __forceinline__ float2 upk(cx a) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(a));
    return r;
}
__device__ __forceinline__ cx add2(cx a, cx b) {
    cx r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ cx sub2(cx a, cx b) {
    cx r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ cx mul2(cx a, cx b) {
    cx r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ cx fma2(cx a, cx b, cx c) {
    cx r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
template <bool INV>
__device__ __forceinline__ cx mulwp(cx a, float wr, float wi) { return pk(mulw<INV>(upk(a), wr, wi)); }
// t + (-i) d and t - (-i) d (forward; +i for the inverse)
template <bool INV>
__device__ __forceinline__ void rot_pm(cx t, cx d, cx& plus, cx& minus) {
    const float2 a = upk(t), e = upk(d);
    const cx p = pk(a.x + e.y, a.y - e.x), m = pk(a.x - e.y, a.y + e.x);
    plus = INV ? m : p;
    minus = INV ? p : m;
}
template <bool INV>
__device__ __forceinline__ void fft4p(cx* u) {
    const cx t0 = add2(u[0], u[2]), t1 = sub2(u[0], u[2]), t2 = add2(u[1], u[3]), d = sub2(u[1], u[3]);
    u[0] = add2(t0, t2);
    u[2] = sub2(t0, t2);
    rot_pm<INV>(t1, d, u[1], u[3]);
}
template <bool INV>
__device__ __forceinline__ void dft5p(cx* u) {
    constexpr float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
    constexpr float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
    const cx p1 = add2(u[1], u[4]), m1 = sub2(u[1], u[4]), p2 = add2(u[2], u[3]), m2 = sub2(u[2], u[3]), a0 = u[0];
    const cx A = fma2(p2, pk(c2, c2), fma2(p1, pk(c1, c1), a0));
    const cx B = fma2(p2, pk(c1, c1), fma2(p1, pk(c2, c2), a0));
    const cx U = fma2(m2, pk(s2, s2), mul2(m1, pk(s1, s1)));    // s1*m1 + s2*m2
    const cx V = fma2(m2, pk(-s1, -s1), mul2(m1, pk(s2, s2)));  // s2*m1 - s1*m2
    u[0] = add2(add2(a0, p1), p2);
    rot_pm<INV>(A, U, u[1], u[4]);
    rot_pm<INV>(B, V, u[2], u[3]);
}

// 16-point DFT in registers, natural order in and out (4 x 4 Cooley-Tukey: n = i + 4m, k = q + 4p)
template <bool INV>
__device__ __forceinline__ void dft16(cx* v) {
    constexpr float C1 = 0.92387953251128675613f, S1 = 0.38268343236508977173f, H = 0.70710678118654752440f;
    cx a[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        cx u[4] = {v[i], v[i + 4], v[i + 8], v[i + 12]};
        fft4p<INV>(u);
#pragma unroll
        for (int q = 0; q < 4; ++q) a[i][q] = u[q];
    }
    // twiddles w16^(i*q) = exp(-2*pi*i * i*q / 16)
    a[1][1] = mulwp<INV>(a[1][1], C1, -S1);
    a[1][2] = mulwp<INV>(a[1][2], H, -H);
    a[1][3] = mulwp<INV>(a[1][3], S1, -C1);
    a[2][1] = mulwp<INV>(a[2][1], H, -H);
    a[2][2] = pk(mul_mi<INV>(upk(a[2][2])));
    a[2][3] = mulwp<INV>(a[2][3], -H, -H);
    a[3][1] = mulwp<INV>(a[3][1], S1, -C1);
    a[3][2] = mulwp<INV>(a[3][2], -H, -H);
    a[3][3] = mulwp<INV>(a[3][3], -C1, S1);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        cx u[4] = {a[0][q], a[1][q], a[2][q], a[3][q]};
        fft4p<INV>(u);
#pragma unroll
        for (int p = 0; p < 4; ++p) v[q + 4 * p] = u[p];
    }
}

// 20-point DFT in registers, natural order in and out (4 x 5: n = 5*n1 + n2, k = k1 + 4*k2)
template <bool INV>
__device__ __forceinline__ void dft20(cx* v) {
    // w20^j = (cos(2*pi*j/20), -sin(2*pi*j/20)) for the exponents n2*k1 that occur
    constexpr float c1 = 0.95105651629515357212f, s1 = 0.30901699437494742410f;   // j = 1
    constexpr float c2 = 0.80901699437494742410f, s2 = 0.58778525229247312917f;   // j = 2
    constexpr float c3 = 0.58778525229247312917f, s3 = 0.80901699437494742410f;   // j = 3
    constexpr float c4 = 0.30901699437494742410f, s4 = 0.95105651629515357212f;   // j = 4
    cx a[5][4];
#pragma unroll
    for (int n2 = 0; n2 < 5; ++n2) {
        cx u[4] = {v[n2], v[n2 + 5], v[n2 + 10], v[n2 + 15]};
        fft4p<INV>(u);
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) a[n2][k1] = u[k1];
    }
    a[1][1] = mulwp<INV>(a[1][1], c1, -s1);    // j = 1
    a[1][2] = mulwp<INV>(a[1][2], c2, -s2);    // 2
    a[1][3] = mulwp<INV>(a[1][3], c3, -s3);    // 3
    a[2][1] = mulwp<INV>(a[2][1], c2, -s2);    // 2
    a[2][2] = mulwp<INV>(a[2][2], c4, -s4);    // 4
    a[2][3] = mulwp<INV>(a[2][3], -c4, -s4);   // 6: cos(108 deg) = -c4, sin = s4
    a[3][1] = mulwp<INV>(a[3][1], c3, -s3);    // 3
    a[3][2] = mulwp<INV>(a[3][2], -c4, -s4);   // 6
    a[3][3] = mulwp<INV>(a[3][3], -c1, -s1);   // 9: cos(162 deg) = -c1, sin = s1
    a[4][1] = mulwp<INV>(a[4][1], c4, -s4);    // 4
    a[4][2] = mulwp<INV>(a[4][2], -c2, -s2);   // 8: cos(144 deg) = -c2, sin = s2
    a[4][3] = mulwp<INV>(a[4][3], -c2, s2);    // 12: cos(216 deg) = -c2, sin = -s2
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) {
        cx u[5] = {a[0][k1], a[1][k1], a[2][k1], a[3][k1], a[4][k1]};
        dft5p<INV>(u);
#pragma unroll
        for (int k2 = 0; k2 < 5; ++k2) v[k1 + 4 * k2] = u[k2];
    }
}


// ---------------------------------------------------------------------------------------------------------------
// CTA-level 320-point transform with caller-supplied loads and stores (the body of fft.cu's fft320_kernel): 320 threads,
// up to 16 lines, shared memory = [16][16*22 + (COLS ? 1 : 4)] float2 exchange buffer + 320 float2 twiddles.
// ---------------------------------------------------------------------------------------------------------------
constexpr int CTA_N = 320, CTA_N1 = 16, CTA_N2 = 20, CTA_XS = 22, CTA_LINES = 16;

// One CTA of 320 threads transforms up to 16 lines: ld(l, j) -> element j of line l, st(l, k, X) <- bin k of line l.
// ROWS: thread (l = tid / 20, t = tid % 20); COLS: thread (t = tid / 16, l = tid % 16) -- see fft320_kernel.
template <bool INV, bool COLS, class Load, class Store>
__device__ __forceinline__ void fft320_cta(float2* xch, float2* tw1_s, const float2* __restrict__ tw, int nvalid, int in_sign,
                                           int out_sign, float scale, Load ld, Store st) {
    constexpr int CS = COLS ? CTA_N1 * CTA_XS + 1 : CTA_N1 * CTA_XS + 4;
    const int tid = threadIdx.x;
    const int l = COLS ? (tid & 15) : tid / CTA_N2, t = COLS ? (tid >> 4) : tid - (tid / CTA_N2) * CTA_N2;
    cx v[CTA_N1];
    if (l < nvalid) {
        float2 x[CTA_N1];
#pragma unroll
        for (int n1 = 0; n1 < CTA_N1; ++n1) x[n1] = ld(l, CTA_N2 * n1 + t);
        const float sg = (in_sign && (t & 1)) ? -1.f : 1.f;
#pragma unroll
        for (int n1 = 0; n1 < CTA_N1; ++n1) v[n1] = pk(x[n1].x * sg, x[n1].y * sg);
    }
    {
        const int a = tid / CTA_N2, b = tid - a * CTA_N2;
        tw1_s[tid] = __ldg(&tw[a * b]);  // tid = 20*k1 + t
    }
    __syncthreads();
    float2* xl = xch + (size_t)l * CS;
    if (l < nvalid) {
        dft16<INV>(v);
        xl[t] = upk(v[0]);
#pragma unroll
        for (int k1 = 1; k1 < CTA_N1; ++k1) {
            const float2 w = tw1_s[k1 * CTA_N2 + t];
            xl[k1 * CTA_XS + t] = mulw<INV>(upk(v[k1]), w.x, w.y);
        }
    }
    __syncthreads();
    if (tid < CTA_LINES * CTA_N1) {
        const int l2 = COLS ? (tid & 15) : (tid >> 4), k1 = COLS ? (tid >> 4) : (tid & 15);
        if (l2 < nvalid) {
            cx u[CTA_N2];
            const float2* row = xch + (size_t)l2 * CS + k1 * CTA_XS;
            if (COLS) {
#pragma unroll
                for (int i = 0; i < CTA_N2; ++i) u[i] = pk(row[i]);
            } else {
                const float4* row4 = reinterpret_cast<const float4*>(row);
#pragma unroll
                for (int i = 0; i < CTA_N2 / 2; ++i) {
                    const float4 q = row4[i];
                    u[2 * i] = pk(q.x, q.y);
                    u[2 * i + 1] = pk(q.z, q.w);
                }
            }
            dft20<INV>(u);
            const float sc = (out_sign && (k1 & 1)) ? -scale : scale;
#pragma unroll
            for (int k2 = 0; k2 < CTA_N2; ++k2) {
                const float2 r = upk(u[k2]);
                st(l2, k1 + CTA_N1 * k2, make_float2(r.x * sc, r.y * sc));
            }
        }
    }
}

// 640-point COLUMN transform of 8 adjacent columns per CTA: radix-2 decimation in time over two 320-point transforms (the
// even and the odd samples of a column are two of the 16 lines of fft320_cta), combined through shared memory:
// X[k] = E[k] + w640^k O[k], X[k + 320] = E[k] - w640^k O[k].  Centring: a half-length rotation of the input is the sign
// (-1)^k on the output (k and k + 320 have the same parity); a half-length rotation of the output is the modulation
// (-1)^n of the input, i.e. a minus sign on the odd-sample lines.  ld(col, n) -> sample n < 640 of column col < 8,
// st(col, k, X) <- bin k < 640.  buf: [16][321] float2.
template <bool INV, class Load, class Store>
__device__ __forceinline__ void fft640_cols_cta(float2* xch, float2* tw1_s, float2* buf, const float2* __restrict__ tw320,
                                                const float2* __restrict__ tw640, int ncols, int in_mod, int out_sign,
                                                float scale, Load ld, Store st) {
    auto ld2 = [&](int l, int j) {
        const int e = l >> 3, cl = l & 7;
        float2 v = make_float2(0.f, 0.f);
        if (cl < ncols) v = ld(cl, 2 * j + e);
        if (in_mod && e) v = make_float2(-v.x, -v.y);
        return v;
    };
    auto st2 = [&](int l, int k, float2 v) { buf[(size_t)l * (CTA_N + 1) + k] = v; };
    fft320_cta<INV, true>(xch, tw1_s, tw320, CTA_LINES, 0, 0, 1.f, ld2, st2);
    __syncthreads();
    for (int idx = threadIdx.x; idx < 8 * CTA_N; idx += blockDim.x) {
        const int cl = idx & 7, k = idx >> 3;
        if (cl >= ncols) continue;
        const float2 E = buf[(size_t)cl * (CTA_N + 1) + k], O = buf[(size_t)(8 + cl) * (CTA_N + 1) + k];
        const float2 w = __ldg(&tw640[k]);
        const float2 T = mulw<INV>(O, w.x, w.y);
        const float sc = (out_sign && (k & 1)) ? -scale : scale;
        st(cl, k, make_float2((E.x + T.x) * sc, (E.y + T.y) * sc));
        st(cl, k + CTA_N, make_float2((E.x - T.x) * sc, (E.y - T.y) * sc));
    }
}

}  // namespace r320

}  // namespace mrb
