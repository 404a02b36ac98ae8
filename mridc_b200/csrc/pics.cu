// l1-wavelet SENSE reconstruction (libmridc_b200_pics.so, C-ABI in include/mridc_b200_pics.h).
// Contract and kernels: DESIGN.md section 4.8.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "../../include/mridc_b200_pics.h"

namespace mrb {
namespace pics {

static thread_local char g_err[512] = "";

static void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define MRBP_REQUIRE(cond, code, ...)         \
    do {                                      \
        if (!(cond)) {                        \
            mrb::pics::set_error(__VA_ARGS__); \
            return (code);                    \
        }                                     \
    } while (0)

#define MRBP_LAUNCHED()                                                                                           \
    do {                                                                                                          \
        cudaError_t _e = cudaPeekAtLastError();                                                                   \
        if (_e != cudaSuccess) {                                                                                  \
            (void)cudaGetLastError();                                                                             \
            mrb::pics::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e));       \
            return MRBP_ECUDA;                                                                                    \
        }                                                                                                         \
    } while (0)

// db4 (pywt, extremal phase) low-pass analysis taps rounded to fp32; high-pass g[j] = (-1)^j h[7 - j]
#define DB4_H0 0.2303778133088964
#define DB4_H1 0.7148465705529154
#define DB4_H2 0.6308807679298587
#define DB4_H3 -0.0279837694168599
#define DB4_H4 -0.1870348117190931
#define DB4_H5 0.0308413818355607
#define DB4_H6 0.0328830116668852
#define DB4_H7 -0.0105974017850690
__constant__ float c_lo[8] = {(float)DB4_H0, (float)DB4_H1, (float)DB4_H2, (float)DB4_H3,
                              (float)DB4_H4, (float)DB4_H5, (float)DB4_H6, (float)DB4_H7};
__constant__ float c_hi[8] = {(float)DB4_H7, -(float)DB4_H6, (float)DB4_H5, -(float)DB4_H4,
                              (float)DB4_H3, -(float)DB4_H2, (float)DB4_H1, -(float)DB4_H0};

constexpr int T = 16;          // coarse coefficients per tile side (a synthesis tile: 2T x 2T samples)
constexpr int NI = 2 * T + 6;  // samples per side an analysis tile reads (8 taps)
constexpr int NU = T + 3;      // coarse coefficients per side a synthesis tile reads
constexpr int THREADS = 256;

__device__ __forceinline__ void fma2(float f, float2 v, float2& acc) {
    acc.x = fmaf(f, v.x, acc.x);
    acc.y = fmaf(f, v.y, acc.y);
}

// c * max(0, 1 - t / |c|); NaN propagates
__device__ __forceinline__ float2 soft(float2 c, float t) {
    const float a = sqrtf(fmaf(c.x, c.x, c.y * c.y));
    if (a <= t) return make_float2(0.f, 0.f);
    const float s = (a - t) / a;
    return make_float2(c.x * s, c.y * s);
}

// i mod n; one wrap in either direction is the common case (bands at least as long as a tile's reach)
__device__ __forceinline__ int wrap(int i, int n) {
    if (i >= n) i -= n;
    if (i < 0) i += n;
    return (i >= 0 && i < n) ? i : ((i % n) + n) % n;
}

struct AnaParams {
    const float2* src;    // band to transform, row stride src_stride, slice stride src_ss (FROM_GRADIENT: z)
    long long src_ss;
    int src_stride;
    const float* grad;    // FROM_GRADIENT: [B, 4, H, W], channels 2-3
    const float* alpha;   // [B]
    float lamda;
    float2* coef;         // detail bands, [B, H, W] Mallat layout
    float2* ll;           // coarse band destination, row stride ll_stride, slice stride ll_ss
    long long ll_ss;
    int ll_stride;
    int H, W, h, w;       // image and band size (both even)
    int last;             // SHRINK: the coarse band is thresholded too
};

// One level of the 2-D analysis: a CTA produces T x T coefficients of each of the four bands.  The input tile (with its
// 6-sample halo, periodic) is filtered along W into low / high halves in shared memory, then along H.
// FROM_GRADIENT: the band is z - alpha * grad, formed as the tile is loaded (level 1 of a FISTA step).
// SHRINK: every detail coefficient, and on the last level the coarse band, leaves soft-thresholded by alpha * lamda.
template <bool FROM_GRADIENT, bool SHRINK>
__global__ void __launch_bounds__(THREADS) analysis_kernel(AnaParams p) {
    __shared__ float2 in[NI][NI + 1];
    __shared__ float2 lo[NI][T + 1], hi[NI][T + 1];
    const int b = blockIdx.z, ky0 = blockIdx.y * T, kx0 = blockIdx.x * T;
    const int h = p.h, w = p.w, h2 = h / 2, w2 = w / 2;
    const long long HW = (long long)p.H * p.W;
    const float2* src = p.src + b * p.src_ss;
    float a = 0.f;
    const float* gre = nullptr;
    if (FROM_GRADIENT) {
        a = p.alpha[b];
        gre = p.grad + ((long long)b * 4 + 2) * HW;
    }
    for (int t = threadIdx.x; t < NI * NI; t += THREADS) {
        const int r = t / NI, c = t % NI;
        const int yy = wrap(2 * ky0 + r, h), xx = wrap(2 * kx0 + c, w);
        const long long o = (long long)yy * p.src_stride + xx;
        float2 v = src[o];
        if (FROM_GRADIENT) {
            v.x = fmaf(-a, gre[o], v.x);
            v.y = fmaf(-a, gre[o + HW], v.y);
        }
        in[r][c] = v;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < NI * T; t += THREADS) {
        const int r = t % NI, k = t / NI;
        float2 sl = make_float2(0.f, 0.f), sh = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float2 v = in[r][2 * k + j];
            fma2(c_lo[j], v, sl);
            fma2(c_hi[j], v, sh);
        }
        lo[r][k] = sl;
        hi[r][k] = sh;
    }
    __syncthreads();
    const int ky = threadIdx.x / T, kx = threadIdx.x % T;
    float2 ll = make_float2(0.f, 0.f), lh = ll, hl = ll, hh = ll;
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        const float2 L = lo[2 * ky + m][kx], Hv = hi[2 * ky + m][kx];
        fma2(c_lo[m], L, ll);
        fma2(c_hi[m], L, hl);
        fma2(c_lo[m], Hv, lh);
        fma2(c_hi[m], Hv, hh);
    }
    const int oy = ky0 + ky, ox = kx0 + kx;
    if (oy >= h2 || ox >= w2) return;
    if (SHRINK) {
        const float tau = p.alpha[b] * p.lamda;
        lh = soft(lh, tau);
        hl = soft(hl, tau);
        hh = soft(hh, tau);
        if (p.last) ll = soft(ll, tau);
    }
    float2* coef = p.coef + b * HW;
    coef[(long long)oy * p.W + w2 + ox] = lh;
    coef[(long long)(h2 + oy) * p.W + ox] = hl;
    coef[(long long)(h2 + oy) * p.W + w2 + ox] = hh;
    p.ll[b * p.ll_ss + (long long)oy * p.ll_stride + ox] = ll;
}

struct SynParams {
    const float2* ll;     // coarse band, row stride ll_stride, slice stride ll_ss
    long long ll_ss;
    int ll_stride;
    const float2* coef;   // detail bands, [B, H, W] Mallat layout
    float2* out;          // band destination, row stride out_stride, slice stride out_ss (FISTA: x)
    long long out_ss;
    int out_stride;
    float2* z;            // FISTA: z <- x_{k+1} + beta (x_{k+1} - x_k)
    float beta;
    int H, W, h, w;       // image and output band size (both even)
};

// One level of the 2-D synthesis (the transpose of analysis_kernel): a CTA produces 2T x 2T samples from the
// (T + 3) x (T + 3) coefficients of each band that reach them, first along H, then along W.
// FISTA: the output is x_{k+1}; x_k is read in place and z_{k+1} written beside it.
template <bool FISTA>
__global__ void __launch_bounds__(THREADS) synthesis_kernel(SynParams p) {
    __shared__ float2 cb[4][NU][NU + 1];  // LL, LH, HL, HH
    __shared__ float2 lx[2 * T][NU + 1], hx[2 * T][NU + 1];
    const int b = blockIdx.z, i0 = blockIdx.y * 2 * T, j0 = blockIdx.x * 2 * T;
    const int h = p.h, w = p.w, h2 = h / 2, w2 = w / 2;
    const long long HW = (long long)p.H * p.W;
    const float2* llb = p.ll + b * p.ll_ss;
    const float2* coef = p.coef + b * HW;
    for (int t = threadIdx.x; t < 4 * NU * NU; t += THREADS) {
        const int band = t / (NU * NU), u = (t / NU) % NU, v = t % NU;
        const int r = wrap(i0 / 2 - 3 + u, h2), c = wrap(j0 / 2 - 3 + v, w2);
        float2 val;
        if (band == 0)
            val = llb[(long long)r * p.ll_stride + c];
        else
            val = coef[(long long)(band >= 2 ? h2 + r : r) * p.W + (band & 1 ? w2 + c : c)];
        cb[band][u][v] = val;
    }
    __syncthreads();
    // sample i of a line takes coefficient k through tap i - 2k: the taps of i's parity, k = i/2 + 3 - q (tile coords)
    for (int t = threadIdx.x; t < 2 * T * NU; t += THREADS) {
        const int pi = t / NU, v = t % NU, par = pi & 1, u0 = (pi >> 1) + 3;
        float2 sl = make_float2(0.f, 0.f), sh = make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float fl = par ? c_lo[2 * q + 1] : c_lo[2 * q], fh = par ? c_hi[2 * q + 1] : c_hi[2 * q];
            fma2(fl, cb[0][u0 - q][v], sl);
            fma2(fh, cb[2][u0 - q][v], sl);
            fma2(fl, cb[1][u0 - q][v], sh);
            fma2(fh, cb[3][u0 - q][v], sh);
        }
        lx[pi][v] = sl;
        hx[pi][v] = sh;
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 4 * T * T; t += THREADS) {
        const int pi = t / (2 * T), qj = t % (2 * T), par = qj & 1, v0 = (qj >> 1) + 3;
        float2 s = make_float2(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float fl = par ? c_lo[2 * q + 1] : c_lo[2 * q], fh = par ? c_hi[2 * q + 1] : c_hi[2 * q];
            fma2(fl, lx[pi][v0 - q], s);
            fma2(fh, hx[pi][v0 - q], s);
        }
        const int oi = i0 + pi, oj = j0 + qj;
        if (oi >= h || oj >= w) continue;
        const long long o = b * p.out_ss + (long long)oi * p.out_stride + oj;
        if (FISTA) {
            const float2 xo = p.out[o];
            p.out[o] = s;
            p.z[o] = make_float2(fmaf(p.beta, s.x - xo.x, s.x), fmaf(p.beta, s.y - xo.y, s.y));
        } else {
            p.out[o] = s;
        }
    }
}

// alpha[b] = 1 / (max_r sum_c |S_bc(r)|^2 * max |M_b|): one CTA per slice; the coil sum runs in coil order, and a max
// does not depend on the order it is taken in.
__global__ void __launch_bounds__(1024) step_size_kernel(const float2* __restrict__ S, const void* __restrict__ mask,
                                                         int mask_dtype, int mask_b, int mask_h, int C, int HW, int W,
                                                         float* __restrict__ alpha) {
    __shared__ float red[2][32];
    const int b = blockIdx.x;
    const float2* s = S + (long long)b * C * HW;
    float smax = 0.f, mmax = 0.f;
    for (int r = threadIdx.x; r < HW; r += blockDim.x) {
        float acc = 0.f;
        for (int c = 0; c < C; ++c) {
            const float2 v = s[(long long)c * HW + r];
            acc = fmaf(v.x, v.x, fmaf(v.y, v.y, acc));
        }
        smax = fmaxf(smax, acc);
    }
    const long long nm = (long long)mask_h * W, m0 = (mask_b == 1 ? 0 : b) * nm;
    for (long long i = threadIdx.x; i < nm; i += blockDim.x) {
        const float v = mask_dtype == 0 ? (float)((const unsigned char*)mask)[m0 + i]
                                        : fabsf(((const float*)mask)[m0 + i]);
        mmax = fmaxf(mmax, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o /= 2) {
        smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, o));
        mmax = fmaxf(mmax, __shfl_xor_sync(0xffffffffu, mmax, o));
    }
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32, nw = blockDim.x / 32;
    if (lane == 0) {
        red[0][warp] = smax;
        red[1][warp] = mmax;
    }
    __syncthreads();
    if (warp) return;
    smax = lane < nw ? red[0][lane] : 0.f;
    mmax = lane < nw ? red[1][lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o /= 2) {
        smax = fmaxf(smax, __shfl_xor_sync(0xffffffffu, smax, o));
        mmax = fmaxf(mmax, __shfl_xor_sync(0xffffffffu, mmax, o));
    }
    if (lane == 0) {
        const float prod = smax * mmax;
        alpha[b] = prod > 0.f ? 1.f / prod : 0.f;
    }
}

}  // namespace pics
}  // namespace mrb

using namespace mrb::pics;

extern "C" const char* mrbp_last_error(void) { return g_err; }
extern "C" int mrbp_version(void) { return 100; }

extern "C" int mrbp_levels(int H, int W) {
    MRBP_REQUIRE(H >= 1 && W >= 1, MRBP_EINVAL, "mrbp_levels: bad size H=%d W=%d", H, W);
    const int m = H < W ? H : W;
    int L = 0;
    while (7LL * (2LL << L) <= m && (H % (2 << L)) == 0 && (W % (2 << L)) == 0) ++L;
    return L;
}

extern "C" size_t mrbp_workspace_bytes(int B, int H, int W) {
    if (B < 1 || H < 1 || W < 1) return 0;
    return (size_t)12 * B * H * W;
}

static int check_geometry(const char* who, int B, int H, int W, int levels, size_t ws_bytes) {
    MRBP_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRBP_EINVAL, "%s: bad shape B=%d H=%d W=%d", who, B, H, W);
    MRBP_REQUIRE(levels >= 1 && levels <= 16 && H % (1 << levels) == 0 && W % (1 << levels) == 0, MRBP_EINVAL,
                 "%s: %d levels do not divide %d x %d", who, levels, H, W);
    MRBP_REQUIRE(B <= 65535, MRBP_EUNSUPPORTED, "%s: batch %d > 65535", who, B);
    MRBP_REQUIRE((long long)H * W <= (1LL << 30), MRBP_EUNSUPPORTED, "%s: H*W = %lld too large", who, (long long)H * W);
    MRBP_REQUIRE(ws_bytes >= mrbp_workspace_bytes(B, H, W), MRBP_EINVAL, "%s: workspace %zu bytes < %zu", who,
                 ws_bytes, mrbp_workspace_bytes(B, H, W));
    return MRBP_OK;
}

static dim3 grid_of(int h, int w, int B) { return dim3((w / 2 + T - 1) / T, (h / 2 + T - 1) / T, B); }

// the coarse band of level l (l >= 1) lives in one of two half-size planes of the workspace, by parity
static float2* coarse_plane(void* ws, int B, int H, int W, int l) {
    float2* base = (float2*)ws + (size_t)B * H * W;
    return (l & 1) ? base : base + (size_t)B * (H / 2) * (W / 2);
}

// Levels 1..levels of the analysis.  FROM_GRADIENT (FISTA): level 1 reads z and grad; SHRINK on every level.
template <bool FROM_GRADIENT, bool SHRINK>
static void analyse(const float2* src, const float* grad, const float* alpha, float lamda, float2* coef, void* ws,
                    int B, int H, int W, int levels, cudaStream_t st) {
    for (int l = 1; l <= levels; ++l) {
        const int h = H >> (l - 1), w = W >> (l - 1);
        AnaParams p;
        if (l == 1) {
            p.src = src;
            p.src_ss = (long long)H * W;
            p.src_stride = W;
        } else {
            p.src = coarse_plane(ws, B, H, W, l - 1);
            p.src_ss = (long long)h * w;
            p.src_stride = w;
        }
        p.grad = grad;
        p.alpha = alpha;
        p.lamda = lamda;
        p.coef = coef;
        p.last = l == levels;
        if (p.last) {
            p.ll = coef;
            p.ll_ss = (long long)H * W;
            p.ll_stride = W;
        } else {
            p.ll = coarse_plane(ws, B, H, W, l);
            p.ll_ss = (long long)(h / 2) * (w / 2);
            p.ll_stride = w / 2;
        }
        p.H = H, p.W = W, p.h = h, p.w = w;
        if constexpr (FROM_GRADIENT) {
            if (l == 1) {
                analysis_kernel<true, SHRINK><<<grid_of(h, w, B), THREADS, 0, st>>>(p);
                continue;
            }
        }
        analysis_kernel<false, SHRINK><<<grid_of(h, w, B), THREADS, 0, st>>>(p);
    }
}

// Levels levels..1 of the synthesis.  FISTA: level 1 writes x (reading x_k) and z.
template <bool FISTA>
static void synthesise(const float2* coef, float2* out, float2* z, float beta, void* ws, int B, int H, int W,
                       int levels, cudaStream_t st) {
    for (int l = levels; l >= 1; --l) {
        const int h = H >> (l - 1), w = W >> (l - 1);
        SynParams p;
        if (l == levels) {
            p.ll = coef;
            p.ll_ss = (long long)H * W;
            p.ll_stride = W;
        } else {
            p.ll = coarse_plane(ws, B, H, W, l);
            p.ll_ss = (long long)(h / 2) * (w / 2);
            p.ll_stride = w / 2;
        }
        p.coef = coef;
        if (l == 1) {
            p.out = out;
            p.out_ss = (long long)H * W;
            p.out_stride = W;
        } else {
            p.out = coarse_plane(ws, B, H, W, l - 1);
            p.out_ss = (long long)h * w;
            p.out_stride = w;
        }
        p.z = z;
        p.beta = beta;
        p.H = H, p.W = W, p.h = h, p.w = w;
        if constexpr (FISTA) {
            if (l == 1) {
                synthesis_kernel<true><<<grid_of(h, w, B), THREADS, 0, st>>>(p);
                continue;
            }
        }
        synthesis_kernel<false><<<grid_of(h, w, B), THREADS, 0, st>>>(p);
    }
}

extern "C" int mrbp_step_size(const void* S, const void* mask, int mask_dtype, int mask_b, int mask_h, int B, int C,
                              int H, int W, void* alpha, void* stream) {
    MRBP_REQUIRE(S && mask && alpha, MRBP_EINVAL, "mrbp_step_size: null pointer");
    MRBP_REQUIRE(B >= 1 && C >= 1 && H >= 1 && W >= 1, MRBP_EINVAL, "mrbp_step_size: bad shape B=%d C=%d H=%d W=%d", B,
                 C, H, W);
    MRBP_REQUIRE(mask_dtype == 0 || mask_dtype == 1, MRBP_EINVAL, "mrbp_step_size: mask_dtype %d", mask_dtype);
    MRBP_REQUIRE((mask_b == 1 || mask_b == B) && (mask_h == 1 || mask_h == H), MRBP_EINVAL,
                 "mrbp_step_size: mask [%d, %d, W] does not broadcast to [%d, %d, W]", mask_b, mask_h, B, H);
    MRBP_REQUIRE(B <= (1 << 30) && (long long)H * W <= (1LL << 30), MRBP_EUNSUPPORTED, "mrbp_step_size: shape too large");
    step_size_kernel<<<B, 1024, 0, (cudaStream_t)stream>>>((const float2*)S, mask, mask_dtype, mask_b, mask_h, C, H * W,
                                                           W, (float*)alpha);
    MRBP_LAUNCHED();
    return MRBP_OK;
}

extern "C" int mrbp_dwt(const void* in, void* out, int inverse, int B, int H, int W, int levels, void* ws,
                        size_t ws_bytes, void* stream) {
    MRBP_REQUIRE(in && out && ws, MRBP_EINVAL, "mrbp_dwt: null pointer");
    MRBP_REQUIRE(in != out, MRBP_EINVAL, "mrbp_dwt: in and out must be distinct buffers");
    int rc = check_geometry("mrbp_dwt", B, H, W, levels, ws_bytes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (inverse)
        synthesise<false>((const float2*)in, (float2*)out, nullptr, 0.f, ws, B, H, W, levels, st);
    else
        analyse<false, false>((const float2*)in, nullptr, nullptr, 0.f, (float2*)out, ws, B, H, W, levels, st);
    MRBP_LAUNCHED();
    return MRBP_OK;
}

extern "C" int mrbp_fista_step(void* z, const void* grad, const void* alpha, float lamda, float beta, void* x, int B,
                               int H, int W, int levels, void* ws, size_t ws_bytes, void* stream) {
    MRBP_REQUIRE(z && grad && alpha && x && ws, MRBP_EINVAL, "mrbp_fista_step: null pointer");
    MRBP_REQUIRE(lamda >= 0.f, MRBP_EINVAL, "mrbp_fista_step: lamda %g < 0", (double)lamda);
    int rc = check_geometry("mrbp_fista_step", B, H, W, levels, ws_bytes);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    float2* coef = (float2*)ws;
    analyse<true, true>((const float2*)z, (const float*)grad, (const float*)alpha, lamda, coef, ws, B, H, W, levels, st);
    synthesise<true>(coef, (float2*)x, (float2*)z, beta, ws, B, H, W, levels, st);
    MRBP_LAUNCHED();
    return MRBP_OK;
}
