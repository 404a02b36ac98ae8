// ESPIRiT coil-sensitivity estimation (libmridc_b200_espirit.so, C-ABI in include/mridc_b200_espirit.h).
// Semantics: sigpy EspiritCalib, one map set; the conventions are derived in DESIGN.md section 4.7.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "../../include/mridc_b200_espirit.h"

namespace mrb {
namespace espirit {

static thread_local char g_err[512] = "";

static void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define MRBE_REQUIRE(cond, code, ...)     \
    do {                                  \
        if (!(cond)) {                    \
            mrb::espirit::set_error(__VA_ARGS__); \
            return (code);                \
        }                                 \
    } while (0)

#define MRBE_CUDA(expr)                                                                          \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            mrb::espirit::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return MRBE_ECUDA;                                                                   \
        }                                                                                        \
    } while (0)

#define MRBE_LAUNCHED()                                                                              \
    do {                                                                                             \
        cudaError_t _e = cudaPeekAtLastError();                                                      \
        if (_e != cudaSuccess) {                                                                     \
            (void)cudaGetLastError();                                                                \
            mrb::espirit::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return MRBE_ECUDA;                                                                       \
        }                                                                                            \
    } while (0)

__device__ __forceinline__ int pair_index(int c, int d, int C) { return c * C - c * (c - 1) / 2 + (d - c); }

// ---- calibration Gram matrix ---------------------------------------------------------------------
// One CTA per coil pair c <= d and slice.  The two coils' ACS blocks (complex64, exact in fp64) sit in shared memory;
// thread e owns entries (c,p,q) x (d,p',q') with e = pq * kw^2 + p'q' and sums its n*n window products in fp64 in
// row-major window order.  The (d,c) block is written as the conjugate transpose of the same sums; on the diagonal
// block only pq <= p'q' is computed, so each element has exactly one writer and the matrix is exactly Hermitian
// (with a real diagonal).
__global__ void __launch_bounds__(256) calib_gram_kernel(const float2* __restrict__ y, double2* __restrict__ gram,
                                                         int C, int H, int W, int cw, int kw, int centered) {
    extern __shared__ float2 acs[];  // [2][cw][cw]
    const int b = blockIdx.y;
    int c = 0, rest = blockIdx.x;
    while (rest >= C - c) {
        rest -= C - c;
        ++c;
    }
    const int d = c + rest;
    const int y0 = H / 2 - cw / 2, x0 = W / 2 - cw / 2;
    // centred row r lives at storage row r when centered, else at (r - H/2) mod H (fftshift by index rotation)
    const int ry = centered ? 0 : H - H / 2, rx = centered ? 0 : W - W / 2;
    const int cw2 = cw * cw;
    for (int t = threadIdx.x; t < 2 * cw2; t += blockDim.x) {
        const int which = t / cw2, i = (t % cw2) / cw, j = t % cw;
        const int coil = which ? d : c;
        const int row = (y0 + i + ry) % H, col = (x0 + j + rx) % W;
        acs[t] = y[(((long long)b * C + coil) * H + row) * W + col];
    }
    __syncthreads();
    const float2* a = acs;
    const float2* e2 = acs + cw2;
    const int n = cw - kw + 1, k2 = kw * kw, N = C * k2;
    double2* out = gram + (long long)b * N * N;
    for (int e = threadIdx.x; e < k2 * k2; e += blockDim.x) {
        const int u = e / k2, v = e % k2;
        if (c == d && u > v) continue;
        const int p = u / kw, q = u % kw, pp = v / kw, qq = v % kw;
        double sr = 0.0, si = 0.0;
        for (int i = 0; i < n; ++i) {
            const float2* ar = a + (i + p) * cw + q;
            const float2* br = e2 + (i + pp) * cw + qq;
            for (int j = 0; j < n; ++j) {
                const double xr = ar[j].x, xi = ar[j].y, zr = br[j].x, zi = br[j].y;
                // conj(x) * z
                sr = fma(xr, zr, fma(xi, zi, sr));
                si = fma(xr, zi, fma(-xi, zr, si));
            }
        }
        const long long rowi = (long long)c * k2 + u, coli = (long long)d * k2 + v;
        if (rowi == coli) {  // sum of |x|^2: real (the fma chain leaves product rounding residue in si)
            out[rowi * N + coli] = make_double2(sr, 0.0);
            continue;
        }
        out[rowi * N + coli] = make_double2(sr, si);
        out[coli * N + rowi] = make_double2(sr, -si);
    }
}

// ---- kernel-subspace taps ------------------------------------------------------------------------
// One thread per (position, coil pair, slice) of the zero-padded tap grid.  The lags that land on the position
// (one for 2kw-1 <= H, W) are summed in a fixed order: lag, then overlap (p, q), then eigenvector.
__global__ void __launch_bounds__(256) kernel_taps_kernel(const double2* __restrict__ vecs, const int* __restrict__ rank,
                                                          float2* __restrict__ taps, int C, int H, int W, int kw,
                                                          int centered) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= H * W) return;
    const int pr = blockIdx.y, b = blockIdx.z, P = C * (C + 1) / 2;
    int c = 0, rest = pr;
    while (rest >= C - c) {
        rest -= C - c;
        ++c;
    }
    const int d = c + rest;
    const int ty = pix / W, tx = pix % W;
    const int k2 = kw * kw, N = C * k2;
    // smallest lag >= -(kw-1) congruent to the position's lag modulo the grid
    const int by = centered ? ty - H / 2 : ty, bx = centered ? tx - W / 2 : tx;
    const int dy0 = ((by + kw - 1) % H + H) % H - (kw - 1), dx0 = ((bx + kw - 1) % W + W) % W - (kw - 1);
    const int K = min(max(rank[b], 0), N);
    const double2* V = vecs + (long long)b * N * N;
    double sr = 0.0, si = 0.0;
    for (int dy = dy0; dy <= kw - 1; dy += H) {
        for (int dx = dx0; dx <= kw - 1; dx += W) {
            const int p_lo = max(0, dy), p_hi = min(kw, kw + dy), q_lo = max(0, dx), q_hi = min(kw, kw + dx);
            for (int p = p_lo; p < p_hi; ++p) {
                for (int q = q_lo; q < q_hi; ++q) {
                    const int ic = c * k2 + p * kw + q, id = d * k2 + (p - dy) * kw + (q - dx);
                    for (int i = N - K; i < N; ++i) {
                        const double2 x = V[(long long)i * N + ic], z = V[(long long)i * N + id];
                        sr = fma(x.x, z.x, fma(x.y, z.y, sr));
                        si = fma(x.x, z.y, fma(-x.y, z.x, si));
                    }
                }
            }
        }
    }
    const double s = 1.0 / k2;
    taps[((long long)b * P + pr) * H * W + pix] = make_float2((float)(sr * s), (float)(si * s));
}

// ---- per-pixel power method ----------------------------------------------------------------------
// CM lanes per pixel (CM = 16 for C <= 16: two pixels per warp; CM = 32 otherwise).  Lane c holds row c of G(r) in
// registers; the iterate is exchanged through shared memory (one float4 broadcast read per two coils).  The norm is
// an xor-butterfly over the pixel's lanes: every lane ends with the same bits (fp addition commutes).
template <int CM>
__global__ void __launch_bounds__(256) power_maps_kernel(const float2* __restrict__ g, float2* __restrict__ maps,
                                                         float* __restrict__ lam_out, int C, int HW, int max_iter,
                                                         float crop) {
    constexpr int PPW = 32 / CM, STRIDE = CM + 2;  // pixels per warp; group stride keeps float4 alignment, no conflicts
    __shared__ __align__(16) float2 xs[8][PPW * STRIDE];
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32, grp = lane / CM, cc = lane % CM;
    const int b = blockIdx.y, P = C * (C + 1) / 2;
    const int pix = (blockIdx.x * 8 + warp) * PPW + grp;
    const bool valid = pix < HW;
    const bool active = valid && cc < C;
    const float2* gb = g + (long long)b * P * HW;
    float2 row[CM];
#pragma unroll
    for (int dd = 0; dd < CM; ++dd) {
        float2 v = make_float2(0.f, 0.f);
        if (active && dd < C) {
            if (cc <= dd) {
                v = gb[(long long)pair_index(cc, dd, C) * HW + pix];
            } else {
                v = gb[(long long)pair_index(dd, cc, C) * HW + pix];
                v.y = -v.y;
            }
        }
        row[dd] = v;
    }
    float2 x = make_float2(active ? 1.f : 0.f, 0.f);
    float lam = 0.f;
    float2* xw = &xs[warp][grp * STRIDE];
    for (int it = 0; it < max_iter; ++it) {
        xw[cc] = x;
        __syncwarp();
        float yr = 0.f, yi = 0.f;
#pragma unroll
        for (int dd = 0; dd < CM; dd += 2) {
            const float4 x2 = *reinterpret_cast<const float4*>(&xw[dd]);
            yr = fmaf(row[dd].x, x2.x, yr);
            yr = fmaf(-row[dd].y, x2.y, yr);
            yi = fmaf(row[dd].x, x2.y, yi);
            yi = fmaf(row[dd].y, x2.x, yi);
            yr = fmaf(row[dd + 1].x, x2.z, yr);
            yr = fmaf(-row[dd + 1].y, x2.w, yr);
            yi = fmaf(row[dd + 1].x, x2.w, yi);
            yi = fmaf(row[dd + 1].y, x2.z, yi);
        }
        __syncwarp();
        float n2 = yr * yr + yi * yi;
#pragma unroll
        for (int o = CM / 2; o > 0; o /= 2) n2 += __shfl_xor_sync(0xffffffffu, n2, o);
        lam = sqrtf(n2);
        if (lam > 0.f) {
            x = make_float2(__fdiv_rn(yr, lam), __fdiv_rn(yi, lam));
        } else {
            x = make_float2(0.f, 0.f);
            lam = 0.f;
        }
    }
    // phase of coil 0
    const float2 x0 = make_float2(__shfl_sync(0xffffffffu, x.x, grp * CM), __shfl_sync(0xffffffffu, x.y, grp * CM));
    const float a0 = sqrtf(x0.x * x0.x + x0.y * x0.y);
    if (a0 > 0.f) {
        const float pr = __fdiv_rn(x0.x, a0), pi = __fdiv_rn(-x0.y, a0);  // conj(x_0) / |x_0|
        x = make_float2(x.x * pr - x.y * pi, x.x * pi + x.y * pr);
    }
    if (!(lam > crop)) x = make_float2(0.f, 0.f);
    if (active) maps[((long long)b * C + cc) * HW + pix] = x;
    if (valid && cc == 0) lam_out[(long long)b * HW + pix] = lam;
}

}  // namespace espirit
}  // namespace mrb

using namespace mrb::espirit;

extern "C" const char* mrbe_last_error(void) { return g_err; }
extern "C" int mrbe_version(void) { return 100; }

static int check_geometry(const char* who, int B, int C, int H, int W) {
    MRBE_REQUIRE(B >= 1 && C >= 1 && H >= 1 && W >= 1, MRBE_EINVAL, "%s: bad shape B=%d C=%d H=%d W=%d", who, B, C, H, W);
    MRBE_REQUIRE(C <= MRBE_MAX_COILS, MRBE_EUNSUPPORTED, "%s: %d coils > %d", who, C, MRBE_MAX_COILS);
    MRBE_REQUIRE((long long)H * W <= (1LL << 30), MRBE_EUNSUPPORTED, "%s: H*W = %lld too large", who, (long long)H * W);
    MRBE_REQUIRE(B <= 65535, MRBE_EUNSUPPORTED, "%s: batch %d > 65535", who, B);
    return MRBE_OK;
}

static int check_kw(const char* who, int C, int H, int W, int kw) {
    MRBE_REQUIRE(kw >= 1 && kw <= H && kw <= W, MRBE_EINVAL, "%s: kernel width %d outside [1, min(H, W)]", who, kw);
    MRBE_REQUIRE(C * kw * kw <= MRBE_MAX_CALIB_COLS, MRBE_EUNSUPPORTED, "%s: C*kw*kw = %d > %d", who, C * kw * kw,
                 MRBE_MAX_CALIB_COLS);
    return MRBE_OK;
}

extern "C" int mrbe_calib_gram(const void* y, void* gram, int B, int C, int H, int W, int cw, int kw, int centered,
                               void* stream) {
    MRBE_REQUIRE(y && gram, MRBE_EINVAL, "mrbe_calib_gram: null pointer");
    int rc = check_geometry("mrbe_calib_gram", B, C, H, W);
    if (rc) return rc;
    if ((rc = check_kw("mrbe_calib_gram", C, H, W, kw))) return rc;
    MRBE_REQUIRE(cw >= kw && cw <= H && cw <= W, MRBE_EINVAL, "mrbe_calib_gram: calibration width %d outside [kw=%d, "
                 "min(H, W)]", cw, kw);
    MRBE_REQUIRE(cw <= MRBE_MAX_CALIB_WIDTH, MRBE_EUNSUPPORTED, "mrbe_calib_gram: calibration width %d > %d", cw,
                 MRBE_MAX_CALIB_WIDTH);
    const size_t smem = 2 * (size_t)cw * cw * sizeof(float2);
    if (smem > 48 * 1024)
        MRBE_CUDA(cudaFuncSetAttribute(calib_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(C * (C + 1) / 2, B);
    calib_gram_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>((const float2*)y, (double2*)gram, C, H, W, cw, kw,
                                                                 centered ? 1 : 0);
    MRBE_LAUNCHED();
    return MRBE_OK;
}

extern "C" int mrbe_kernel_taps(const void* vecs, const int* rank, void* taps, int B, int C, int H, int W, int kw,
                                int centered, void* stream) {
    MRBE_REQUIRE(vecs && rank && taps, MRBE_EINVAL, "mrbe_kernel_taps: null pointer");
    int rc = check_geometry("mrbe_kernel_taps", B, C, H, W);
    if (rc) return rc;
    if ((rc = check_kw("mrbe_kernel_taps", C, H, W, kw))) return rc;
    dim3 grid((H * W + 255) / 256, C * (C + 1) / 2, B);
    kernel_taps_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const double2*)vecs, rank, (float2*)taps, C, H, W, kw,
                                                               centered ? 1 : 0);
    MRBE_LAUNCHED();
    return MRBE_OK;
}

extern "C" int mrbe_power_maps(const void* g, void* maps, void* lambda, int B, int C, int H, int W, int max_iter,
                               float crop, void* stream) {
    MRBE_REQUIRE(g && maps && lambda, MRBE_EINVAL, "mrbe_power_maps: null pointer");
    int rc = check_geometry("mrbe_power_maps", B, C, H, W);
    if (rc) return rc;
    MRBE_REQUIRE(max_iter >= 1, MRBE_EINVAL, "mrbe_power_maps: max_iter %d < 1", max_iter);
    const int HW = H * W;
    if (C <= 16) {
        dim3 grid((HW + 15) / 16, B);  // 8 warps x 2 pixels
        power_maps_kernel<16><<<grid, 256, 0, (cudaStream_t)stream>>>((const float2*)g, (float2*)maps, (float*)lambda,
                                                                      C, HW, max_iter, crop);
    } else {
        dim3 grid((HW + 7) / 8, B);
        power_maps_kernel<32><<<grid, 256, 0, (cudaStream_t)stream>>>((const float2*)g, (float2*)maps, (float*)lambda,
                                                                      C, HW, max_iter, crop);
    }
    MRBE_LAUNCHED();
    return MRBE_OK;
}
