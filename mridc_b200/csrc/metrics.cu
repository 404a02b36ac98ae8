// On-device evaluation of a reconstruction (SURVEY 8f rank 3): what BaseMRIReconstructionModel.test_step does on the host
// after a blocking .cpu() (mridc/collections/reconstruction/models/base.py:415-436) --
//   output = |pred| / max|pred|, target = |target| / max|target|, then MSE / NMSE / PSNR / SSIM
//   (mridc/collections/common/metrics/reconstruction_metrics.py:11-41; PSNR / SSIM arithmetic = scikit-image's
//   peak_signal_noise_ratio and structural_similarity with win_size 7, uniform filter, sample covariance, K1 .01, K2 .03,
//   3-pixel border crop, float64).
// Reductions accumulate in fp64 (skimage converts to float64; numpy's float32 pairwise sums agree to ~1e-7 relative).
#include "common.cuh"

namespace mrb {

// ordered-int encoding so that atomicMax / atomicMin on ints order floats (any sign)
__device__ __forceinline__ int f2ord(float f) {
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

__device__ __forceinline__ float magnitude(const float* x, long long i, int is_complex) {
    if (!is_complex) return fabsf(x[i]);
    const float2 v = reinterpret_cast<const float2*>(x)[i];
    return hypotf(v.x, v.y);  // torch.abs(complex64)
}

// stats[0] = max |x| as an ordered int (zeroed by the host wrapper)
__global__ void abs_max_kernel(const float* __restrict__ x, long long n, int is_complex, int* __restrict__ stats) {
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, magnitude(x, i, is_complex));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(stats, f2ord(m));
}

// out = |x| / max (a true division, like `output / output.max()`, base.py:416-420)
__global__ void abs_normalize_kernel(const float* __restrict__ x, long long n, int is_complex, const int* __restrict__ stats,
                                     float* __restrict__ out) {
    const float mx = ord2f(stats[0]);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = __fdiv_rn(magnitude(x, i, is_complex), mx);
}

// unsigned order key of a float: fkey(a) < fkey(b) iff a < b for non-NaN a, b, and key 0 lies below every such key (it is
// the key of the all-ones NaN pattern), so a ZEROED word is a valid start for atomicMax.  A minimum is kept as the maximum
// of ~fkey (whose zero start stands for +inf).  Zero starts let the caller initialise the workspace with one memset.
__device__ __forceinline__ unsigned fkey(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

// sums[0] = sum (gt - pred)^2, sums[1] = sum gt^2 (fp64); ext[0..3] = fkey(max gt), ~fkey(min gt), fkey(max pred),
// ~fkey(min pred); sums and ext zeroed by the host wrapper
__global__ void metric_sums_kernel(const float* __restrict__ gt, const float* __restrict__ pred, long long n,
                                   double* __restrict__ sums, unsigned* __restrict__ ext) {
    double se = 0.0, sg = 0.0;
    float gmax = -INFINITY, gmin = INFINITY, pmax = -INFINITY, pmin = INFINITY;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float g = gt[i], p = pred[i];
        const double d = (double)g - (double)p;
        se += d * d;
        sg += (double)g * (double)g;
        gmax = fmaxf(gmax, g); gmin = fminf(gmin, g);
        pmax = fmaxf(pmax, p); pmin = fminf(pmin, p);
    }
    for (int o = 16; o > 0; o >>= 1) {
        se += __shfl_xor_sync(0xffffffffu, se, o);
        sg += __shfl_xor_sync(0xffffffffu, sg, o);
        gmax = fmaxf(gmax, __shfl_xor_sync(0xffffffffu, gmax, o)); gmin = fminf(gmin, __shfl_xor_sync(0xffffffffu, gmin, o));
        pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o)); pmin = fminf(pmin, __shfl_xor_sync(0xffffffffu, pmin, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&sums[0], se);
        atomicAdd(&sums[1], sg);
        atomicMax(&ext[0], fkey(gmax)); atomicMax(&ext[1], ~fkey(gmin));
        atomicMax(&ext[2], fkey(pmax)); atomicMax(&ext[3], ~fkey(pmin));
    }
}

constexpr int SSIM_WIN = 7, SSIM_TX = 32, SSIM_TY = 8;

// One thread per VALID window position (the 3-pixel border skimage crops is never evaluated): 7x7 sums of x, y, xx, yy,
// xy in fp64 from a shared-memory tile -> S; per-slice sum in out[b].  data_range: device pointer (double).
__global__ void ssim_sum_kernel(const float* __restrict__ gt, const float* __restrict__ pred, int H, int W,
                                const double* __restrict__ data_range, double* __restrict__ out) {
    __shared__ float tx[SSIM_TY + SSIM_WIN - 1][SSIM_TX + SSIM_WIN - 1];
    __shared__ float ty[SSIM_TY + SSIM_WIN - 1][SSIM_TX + SSIM_WIN - 1];
    const int b = blockIdx.z;
    const int x0 = blockIdx.x * SSIM_TX, y0 = blockIdx.y * SSIM_TY;  // top-left corner of the windows of this tile
    const float* g = gt + (long long)b * H * W;
    const float* p = pred + (long long)b * H * W;
    for (int i = threadIdx.y * SSIM_TX + threadIdx.x; i < (SSIM_TY + SSIM_WIN - 1) * (SSIM_TX + SSIM_WIN - 1);
         i += SSIM_TX * SSIM_TY) {
        const int r = i / (SSIM_TX + SSIM_WIN - 1), c = i - r * (SSIM_TX + SSIM_WIN - 1);
        const int yy = y0 + r, xx = x0 + c;
        const bool ok = yy < H && xx < W;
        tx[r][c] = ok ? g[(long long)yy * W + xx] : 0.f;
        ty[r][c] = ok ? p[(long long)yy * W + xx] : 0.f;
    }
    __syncthreads();
    const int wx = x0 + threadIdx.x, wy = y0 + threadIdx.y;
    double s = 0.0;
    if (wx + SSIM_WIN <= W && wy + SSIM_WIN <= H) {
        double sx = 0, sy = 0, sxx = 0, syy = 0, sxy = 0;
#pragma unroll
        for (int r = 0; r < SSIM_WIN; ++r)
#pragma unroll
            for (int c = 0; c < SSIM_WIN; ++c) {
                const double a = tx[threadIdx.y + r][threadIdx.x + c], q = ty[threadIdx.y + r][threadIdx.x + c];
                sx += a; sy += q; sxx += a * a; syy += q * q; sxy += a * q;
            }
        const double NP = SSIM_WIN * SSIM_WIN, cov = NP / (NP - 1.0);
        const double ux = sx / NP, uy = sy / NP;
        const double vx = cov * (sxx / NP - ux * ux), vy = cov * (syy / NP - uy * uy), vxy = cov * (sxy / NP - ux * uy);
        const double R = *data_range, C1 = (0.01 * R) * (0.01 * R), C2 = (0.03 * R) * (0.03 * R);
        s = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) atomicAdd(&out[b], s);
}

// Everything test_step derives from the sums, on the device (no host round trip between the reductions):
// res[0] = mse, [1] = nmse, [2] = psnr, [3] = NaN when SSIM is skipped (ssim_finish_kernel writes it otherwise),
// [4] = data range used.  maxval_mode 0: max(gt) (reconstruction_metrics.py:23,35), 1: max(pred) - min(pred)
// (base.py:431,434), 2: `maxval`.  Host values arrive as kernel arguments, which a captured CUDA graph holds by value.
__global__ void metrics_finish_kernel(const double* __restrict__ sums, const unsigned* __restrict__ ext, double n, int maxval_mode,
                                      double maxval, int want_ssim, double* __restrict__ res) {
    const double mse = sums[0] / n;
    double R = maxval;
    if (maxval_mode == 0) R = (double)key2f(ext[0]);
    if (maxval_mode == 1) R = (double)(key2f(ext[2]) - key2f(~ext[3]));  // float32 subtraction, like numpy on float32
    res[0] = mse;
    res[1] = sums[0] / sums[1];
    res[2] = 10.0 * log10(R * R / mse);
    if (!want_ssim) res[3] = __longlong_as_double(0x7ff8000000000000LL);
    res[4] = R;
}
__global__ void ssim_finish_kernel(const double* __restrict__ per_slice, int B, double windows, double* __restrict__ res) {
    double s = 0.0;
    for (int b = 0; b < B; ++b) s += per_slice[b] / windows;  // mean over the cropped map, then over slices (:37-41)
    res[3] = s / B;
}

static inline unsigned mgrid(long long n) {
    long long b = (n + 255) / 256;
    const long long cap = (long long)device_sm_count() * 8;
    return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace mrb

using namespace mrb;

extern "C" size_t mrb_metrics_workspace_bytes(int B) { return (size_t)(8 + 8 + (B > 0 ? B : 0)) * sizeof(double); }

extern "C" int mrb_abs_max_normalize(const void* x, long long n, int is_complex, void* out, void* ws, void* stream) {
    MRB_REQUIRE(x && out && ws && n > 0, MRB_EINVAL, "mrb_abs_max_normalize: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    MRB_CUDA(cudaMemsetAsync(ws, 0, sizeof(int), st));  // ordered-int encoding of +0.0f: magnitudes are >= 0
    abs_max_kernel<<<mgrid(n), 256, 0, st>>>((const float*)x, n, is_complex, (int*)ws);
    MRB_LAUNCHED();
    abs_normalize_kernel<<<mgrid(n), 256, 0, st>>>((const float*)x, n, is_complex, (const int*)ws, (float*)out);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_recon_metrics(const void* gt, const void* pred, int B, int H, int W, int maxval_mode, double maxval,
                                 void* res, void* ws, void* stream) {
    MRB_REQUIRE(gt && pred && res && ws, MRB_EINVAL, "mrb_recon_metrics: null pointer");
    const bool want_ssim = (maxval_mode & 4) == 0;  // + 4: MSE / NMSE / PSNR only (any image size, res[3] = NaN)
    maxval_mode &= 3;
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_recon_metrics: bad shape");
    MRB_REQUIRE(!want_ssim || (H >= SSIM_WIN && W >= SSIM_WIN), MRB_EINVAL,
                "mrb_recon_metrics: win_size exceeds image extent (need H, W >= 7; got %d x %d)", H, W);
    MRB_REQUIRE(maxval_mode >= 0 && maxval_mode <= 2, MRB_EINVAL, "mrb_recon_metrics: maxval_mode must be 0, 1 or 2 (+ 4)");
    cudaStream_t st = (cudaStream_t)stream;
    // workspace: doubles [0,1] sums | unsigned at double slot 2..3: ext[4] | doubles [8 .. 8+B) per-slice SSIM sums; every
    // start value is zero (see fkey), so one memset initialises it
    double* wsd = (double*)ws;
    double* resd = (double*)res;
    MRB_CUDA(cudaMemsetAsync(wsd, 0, sizeof(double) * (8 + (size_t)B), st));
    const long long n = (long long)B * H * W;
    metric_sums_kernel<<<mgrid(n), 256, 0, st>>>((const float*)gt, (const float*)pred, n, wsd, (unsigned*)(wsd + 2));
    MRB_LAUNCHED();
    metrics_finish_kernel<<<1, 1, 0, st>>>(wsd, (const unsigned*)(wsd + 2), (double)n, maxval_mode, maxval, want_ssim ? 1 : 0,
                                           resd);
    MRB_LAUNCHED();
    if (!want_ssim) return MRB_OK;
    const int vw = W - SSIM_WIN + 1, vh = H - SSIM_WIN + 1;
    dim3 grid((vw + SSIM_TX - 1) / SSIM_TX, (vh + SSIM_TY - 1) / SSIM_TY, B);
    ssim_sum_kernel<<<grid, dim3(SSIM_TX, SSIM_TY), 0, st>>>((const float*)gt, (const float*)pred, H, W, resd + 4, wsd + 8);
    MRB_LAUNCHED();
    ssim_finish_kernel<<<1, 1, 0, st>>>(wsd + 8, B, (double)vw * (double)vh, resd);
    MRB_LAUNCHED();
    return MRB_OK;
}
