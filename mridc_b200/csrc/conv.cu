// fp32 CUDA-core convolution + recurrent-cell kernels (NCHW).
//
// Reference behaviour:
//   ConvNonlinear           mridc/collections/reconstruction/models/rim/conv_layers.py:36-123
//   ConvGRU/MGU/IndRNN      mridc/collections/reconstruction/models/rim/rnn_cells.py:93-127, :230-261, :367-391
//   U-Net 3x3 / 1x1 convs   mridc/collections/reconstruction/models/unet_base/unet_block.py:185, :250-259
//
// conv2d: implicit GEMM on CUDA cores.  CTA = 4x32 output pixels x (8*TN) output channels, 128 threads, each
// thread an 8-pixel x TN-channel register tile; input halo patch and weight slab of CK input channels staged in
// shared memory per K step; the (k-1)*dil+8 wide input window of a row is loaded once and slid across the taps.
// This is the exact-fp32 path (U-Net, generic shapes); see conv_tc.cu for the tensor-core RIM path.
#include <stdlib.h>

#include "common.cuh"

namespace mrb {

constexpr int TH = 4, TW = 32;  // pixel tile
constexpr int CONV_THREADS = 128;

struct ConvParams {
    const float* x;
    const float* w;
    const float* bias;
    float* out;
    const float* add;
    const float* add_scale;
    const float* residual;
    long long x_bs, out_bs;
    int N, Cin, Cout, H, W, k, dil, pad, pad_mode, act, nhwc_res;
    float slope;
    int CK, PH, PW, PWs, tiles_x;
};

__device__ __forceinline__ float act_fn(float v, int act, float slope) {
    if (act == MRB_ACT_RELU) return v > 0.f ? v : 0.f;
    if (act == MRB_ACT_LEAKY) return v > 0.f ? v : v * slope;
    return v;
}

template <int TN, int K, int DIL>
__global__ void __launch_bounds__(CONV_THREADS) conv2d_kernel(ConvParams P) {
    constexpr int BN = 8 * TN;
    extern __shared__ float4 smem4[];
    float* patch = (float*)smem4;                               // [CK][PH][PWs] (+ slack)
    float* ws = patch + (size_t)P.CK * P.PH * P.PWs + 16;       // [CK*k*k][BN]
    ws = (float*)(((uintptr_t)ws + 15) & ~(uintptr_t)15);
    const int tid = threadIdx.x;
    const int cg = tid % 8, pg = tid / 8;
    const int prow = pg / 4, pcol0 = (pg % 4) * 8;
    const int ty = blockIdx.x / P.tiles_x, tx = blockIdx.x - ty * P.tiles_x;
    const int y0 = ty * TH, x0 = tx * TW;
    const int co0 = blockIdx.y * BN;
    const int n = blockIdx.z;
    const int k = (K > 0) ? K : P.k;
    const int dil = (K > 0) ? DIL : P.dil;
    const int kk = k * k;
    const long long HW = (long long)P.H * P.W;
    const float* xin = P.x + (long long)n * P.x_bs;

    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    for (int ci0 = 0; ci0 < P.Cin; ci0 += P.CK) {
        const int nci = min(P.CK, P.Cin - ci0);
        __syncthreads();
        // ---- stage input patch (halo handled here: zero or replicate/clamp) ----
        const int pelems = nci * P.PH * P.PW;
        for (int t = tid; t < pelems; t += CONV_THREADS) {
            int px = t % P.PW;
            int r = t / P.PW;
            int py = r % P.PH;
            int ci = r / P.PH;
            int gy = y0 - P.pad + py, gx = x0 - P.pad + px;
            float v = 0.f;
            if (P.pad_mode == MRB_PAD_REPLICATE) {
                gy = min(max(gy, 0), P.H - 1);
                gx = min(max(gx, 0), P.W - 1);
                v = xin[(long long)(ci0 + ci) * HW + (long long)gy * P.W + gx];
            } else if (gy >= 0 && gy < P.H && gx >= 0 && gx < P.W) {
                v = xin[(long long)(ci0 + ci) * HW + (long long)gy * P.W + gx];
            }
            patch[((size_t)ci * P.PH + py) * P.PWs + px] = v;
        }
        // ---- stage weights: ws[(ci*kk + tap)][co] = w[co0+co][ci0+ci][tap] ----
        const int welems = nci * kk * BN;
        for (int t = tid; t < welems; t += CONV_THREADS) {
            int co = t % BN;
            int r = t / BN;  // ci*kk + tap
            float v = 0.f;
            if (co0 + co < P.Cout) v = P.w[((long long)(co0 + co) * P.Cin + ci0) * kk + r];
            ws[(size_t)r * BN + co] = v;
        }
        __syncthreads();
        // ---- compute ----
        for (int ci = 0; ci < nci; ++ci) {
            for (int ky = 0; ky < k; ++ky) {
                const float* prow_p = patch + ((size_t)ci * P.PH + prow + ky * dil) * P.PWs + pcol0;
                const float* wrow = ws + (size_t)(ci * kk + ky * k) * BN + cg * TN;
                if (K > 0) {
                    constexpr int WIN = 8 + (K - 1) * DIL;
                    constexpr int WIN4 = (WIN + 3) / 4;
                    float win[WIN4 * 4];
#pragma unroll
                    for (int q = 0; q < WIN4; ++q) {
                        float4 v4 = *reinterpret_cast<const float4*>(prow_p + 4 * q);
                        win[4 * q] = v4.x; win[4 * q + 1] = v4.y; win[4 * q + 2] = v4.z; win[4 * q + 3] = v4.w;
                    }
#pragma unroll
                    for (int kx = 0; kx < K; ++kx) {
                        float wv[TN];
#pragma unroll
                        for (int j = 0; j < TN; ++j) wv[j] = wrow[kx * BN + j];
#pragma unroll
                        for (int i = 0; i < 8; ++i)
#pragma unroll
                            for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(win[i + kx * DIL], wv[j], acc[i][j]);
                    }
                } else {
                    for (int kx = 0; kx < k; ++kx) {
                        float wv[TN];
#pragma unroll
                        for (int j = 0; j < TN; ++j) wv[j] = wrow[kx * BN + j];
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float xv = prow_p[i + kx * dil];
#pragma unroll
                            for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(xv, wv[j], acc[i][j]);
                        }
                    }
                }
            }
        }
    }
    // ---- epilogue ----
    const int oy = y0 + prow;
    if (oy >= P.H) return;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
        const int co = co0 + cg * TN + j;
        if (co >= P.Cout) continue;
        const float b = P.bias ? P.bias[co] : 0.f;
        const float as = (P.add && P.add_scale) ? P.add_scale[co] : 1.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int ox = x0 + pcol0 + i;
            if (ox >= P.W) continue;
            float v = acc[i][j] + b;
            const long long pix = (long long)oy * P.W + ox;
            if (P.add) v += as * P.add[((long long)n * P.Cout + co) * HW + pix];
            v = act_fn(v, P.act, P.slope);
            if (P.nhwc_res) {
                const long long o = ((long long)n * HW + pix) * P.Cout + co;
                P.out[o] = P.residual[o] + v;
            } else {
                P.out[(long long)n * P.out_bs + (long long)co * HW + pix] = v;
            }
        }
    }
}

template <int TN>
static int launch_conv_tn(const ConvParams& P, dim3 grid, size_t smem, cudaStream_t st) {
#define MRB_CONV_CASE(KK, DD)                                                                                   \
    {                                                                                                           \
        auto kern = conv2d_kernel<TN, KK, DD>;                                                                  \
        MRB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));           \
        kern<<<grid, CONV_THREADS, smem, st>>>(P);                                                              \
    }
    if (P.k == 5 && P.dil == 1) MRB_CONV_CASE(5, 1)
    else if (P.k == 3 && P.dil == 2) MRB_CONV_CASE(3, 2)
    else if (P.k == 3 && P.dil == 1) MRB_CONV_CASE(3, 1)
    else if (P.k == 1) MRB_CONV_CASE(1, 1)
    else MRB_CONV_CASE(0, 0)
#undef MRB_CONV_CASE
    MRB_LAUNCHED();
    return MRB_OK;
}

// ---- fused ConvGRU cell, kernel size 1 --------------------------------------------------------------
// CTA = 64 pixels x 64 hidden channels, 256 threads, thread tile 4 px x 4 ch x {r,z,ih_n,hh_n}.
constexpr int GRU_PX = 64, GRU_CH = 64, GRU_KC = 16, GRU_THREADS = 256;

struct GruParams {
    const float* x;
    const float* h;
    const float* w_ih;
    const float* b_ih;
    const float* w_hh;
    float* h_out;
    int N, Cx, Ch;
    long long HW;
};

__device__ __forceinline__ float sigmoidf_acc(float v) { return 1.f / (1.f + expf(-v)); }

__global__ void __launch_bounds__(GRU_THREADS) gru_cell_1x1_kernel(GruParams P) {
    __shared__ __align__(16) float xs[GRU_KC][GRU_PX];
    __shared__ __align__(16) float wsm[GRU_KC][3][GRU_CH];
    const int tid = threadIdx.x;
    const int cg = tid % 16, pg = tid / 16;
    const long long p0 = (long long)blockIdx.x * GRU_PX;
    const int ch0 = blockIdx.y * GRU_CH;
    const int n = blockIdx.z;
    float ar[4][4], az[4][4], ai[4][4], ah[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) ar[i][j] = az[i][j] = ai[i][j] = ah[i][j] = 0.f;

    for (int src = 0; src < 2; ++src) {
        const float* in = src == 0 ? P.x : P.h;
        const float* w = src == 0 ? P.w_ih : P.w_hh;
        const int Cin = src == 0 ? P.Cx : P.Ch;
        const float* inb = in + (long long)n * Cin * P.HW;
        for (int k0 = 0; k0 < Cin; k0 += GRU_KC) {
            const int nk = min(GRU_KC, Cin - k0);
            __syncthreads();
            for (int t = tid; t < GRU_KC * GRU_PX; t += GRU_THREADS) {
                int p = t % GRU_PX, kk = t / GRU_PX;
                float v = 0.f;
                if (kk < nk && p0 + p < P.HW) v = inb[(long long)(k0 + kk) * P.HW + p0 + p];
                xs[kk][p] = v;
            }
            for (int t = tid; t < GRU_KC * 3 * GRU_CH; t += GRU_THREADS) {
                int c = t % GRU_CH;
                int r = t / GRU_CH;
                int g = r % 3, kk = r / 3;
                float v = 0.f;
                if (kk < nk && ch0 + c < P.Ch) v = w[((long long)g * P.Ch + ch0 + c) * Cin + k0 + kk];
                wsm[kk][g][c] = v;
            }
            __syncthreads();
#pragma unroll 4
            for (int kk = 0; kk < GRU_KC; ++kk) {
                float4 xv4 = *reinterpret_cast<const float4*>(&xs[kk][pg * 4]);
                float4 wr4 = *reinterpret_cast<const float4*>(&wsm[kk][0][cg * 4]);
                float4 wz4 = *reinterpret_cast<const float4*>(&wsm[kk][1][cg * 4]);
                float4 wn4 = *reinterpret_cast<const float4*>(&wsm[kk][2][cg * 4]);
                const float xv[4] = {xv4.x, xv4.y, xv4.z, xv4.w};
                const float wr[4] = {wr4.x, wr4.y, wr4.z, wr4.w};
                const float wz[4] = {wz4.x, wz4.y, wz4.z, wz4.w};
                const float wn[4] = {wn4.x, wn4.y, wn4.z, wn4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        ar[i][j] = fmaf(xv[i], wr[j], ar[i][j]);
                        az[i][j] = fmaf(xv[i], wz[j], az[i][j]);
                        if (src == 0) ai[i][j] = fmaf(xv[i], wn[j], ai[i][j]);
                        else ah[i][j] = fmaf(xv[i], wn[j], ah[i][j]);
                    }
            }
        }
    }
    // gates (rnn_cells.py:121-125)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int ch = ch0 + cg * 4 + j;
        if (ch >= P.Ch) continue;
        const float br = P.b_ih ? P.b_ih[ch] : 0.f;
        const float bz = P.b_ih ? P.b_ih[P.Ch + ch] : 0.f;
        const float bn = P.b_ih ? P.b_ih[2 * P.Ch + ch] : 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const long long p = p0 + pg * 4 + i;
            if (p >= P.HW) continue;
            const long long o = ((long long)n * P.Ch + ch) * P.HW + p;
            const float hp = P.h[o];
            const float r = sigmoidf_acc((ar[i][j] + br));
            const float z = sigmoidf_acc((az[i][j] + bz));
            const float nn = tanhf((ai[i][j] + bn) + r * ah[i][j]);
            P.h_out[o] = nn * (1.f - z) + z * hp;
        }
    }
}

__global__ void gru_gates_kernel(const float* __restrict__ ih, const float* __restrict__ hh,
                                 const float* __restrict__ h, float* __restrict__ h_out, int N, int Ch, long long HW) {
    const long long total = (long long)N * Ch * HW;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        long long p = t % HW;
        long long r0 = t / HW;
        int c = (int)(r0 % Ch);
        long long n = r0 / Ch;
        long long g = (n * 3 * Ch + c) * HW + p, gs = (long long)Ch * HW;
        float r = sigmoidf_acc(ih[g] + hh[g]);
        float z = sigmoidf_acc(ih[g + gs] + hh[g + gs]);
        float nn = tanhf(ih[g + 2 * gs] + r * hh[g + 2 * gs]);
        h_out[t] = nn * (1.f - z) + z * h[t];
    }
}

__global__ void mgu_gates_kernel(const float* __restrict__ ih, const float* __restrict__ hh,
                                 const float* __restrict__ h, float* __restrict__ h_out, int N, int Ch, long long HW) {
    const long long total = (long long)N * Ch * HW;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        long long p = t % HW;
        long long r0 = t / HW;
        int c = (int)(r0 % Ch);
        long long n = r0 / Ch;
        long long g = (n * 2 * Ch + c) * HW + p, gs = (long long)Ch * HW;
        float f = sigmoidf_acc(ih[g] + hh[g]);
        float cc = tanhf(ih[g + gs] + f * hh[g + gs]);
        h_out[t] = cc + f * (h[t] - cc);  // rnn_cells.py:261
    }
}

// Final RIM conv (k = 3, dilation 1) on a BH source: 64 -> 2 channels, replicate padding (the BH border), fused eta update.
// CTA = 32 x 16 output pixels, 128 threads, each thread FOUR vertically adjacent pixels x both outputs.
//   * the 18 x 34 halo patch travels in chunks of F_CH channels through a cp.async.cg double buffer (pixel stride padded
//     by 4 floats: conflict-free LDS.128), so the global latency of chunk c+1 hides behind the arithmetic of chunk c;
//   * the three kernel rows reuse the six patch rows a thread holds in registers (2x fewer shared-memory reads than
//     one pixel per thread);
//   * arithmetic is packed fp32x2 (fma.rn.f32x2): a pair = two input channels of one output, summed at the end.
constexpr int F_TX = 32, F_PW = F_TX + 2;
__device__ __forceinline__ void ffma2(float2& acc, float a0, float a1, float b0, float b1) {
    unsigned long long a, b, c;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(acc.x), "f"(acc.y));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.x), "=f"(acc.y) : "l"(c));
}
template <int ROWS, int F_CH>
__global__ void __launch_bounds__(128) conv_c2_k3_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                         const float* __restrict__ bias, const float* __restrict__ eta,
                                                         float* __restrict__ out, int B, int H, int W, int cin) {
    constexpr int F_TY = 4 * ROWS, F_PH = F_TY + 2, F_PS = F_CH + 4, NQ = F_CH / 4;
    extern __shared__ float4 c2smem[];
    float4* wq = c2smem;                                                   // [tap][cin/4][out] -> 4 input channels
    float* patch = reinterpret_cast<float*>(wq + (size_t)9 * (cin / 4) * 2);  // [2][F_PH*F_PW][F_PS]
    for (int t = threadIdx.x; t < 9 * (cin / 4) * 2; t += blockDim.x) {
        const int o = t & 1, cq = (t >> 1) % (cin / 4), tap = (t >> 1) / (cin / 4);
        const float* wp = w + ((long long)o * cin + cq * 4) * 9 + tap;
        wq[t] = make_float4(wp[0], wp[9], wp[18], wp[27]);
    }
    const int tiles_x = (W + F_TX - 1) / F_TX;
    const int ty = blockIdx.x / tiles_x, tx = blockIdx.x - ty * tiles_x;
    const int x0 = tx * F_TX, y0 = ty * F_TY;
    const int b = blockIdx.y;
    const int lx = threadIdx.x & 31, yg = threadIdx.x >> 5;  // pixels (lx, ROWS*yg + i), i = 0..ROWS-1
    // BH source (conv_tc2.cu): [B][H+4][W+4][64 hi bf16 | 64 lo bf16] with a valid replicate border: taps are plain offsets;
    // a staged position holds [F_CH hi | F_CH lo] bf16 (F_CH/2 + F_CH/2 words) and the fp32 value is rebuilt as hi + lo
    const int Hp = H + 4, Wp = W + 4;
    const float* xb = x + (long long)b * Hp * Wp * 64;
    const uint32_t patch_u32 = (uint32_t)__cvta_generic_to_shared(patch);
    // staging list of this thread: float4 t = tid + 128*i of the [F_PH*F_PW pixels][2 quads] chunk; the clamped source
    // offsets are the same for every chunk (computed once), the shared-memory offset is linear in i
    constexpr int kStage = (F_PH * F_PW * NQ + 127) / 128;
    int goff[kStage];
#pragma unroll
    for (int i = 0; i < kStage; ++i) {
        const int t = threadIdx.x + 128 * i;
        const int q = t % NQ, pp = t / NQ;
        const int py = pp / F_PW, px = pp - py * F_PW;
        // quads 0 .. NQ/2-1: the chunk's hi bf16 (16 B each), NQ/2 .. NQ-1: its lo bf16 (128 B further)
        const int gy = min(max(y0 + 1 + py, 0), Hp - 1), gx = min(max(x0 + 1 + px, 0), Wp - 1);
        goff[i] = t < F_PH * F_PW * NQ ? (gy * Wp + gx) * 64 + (q < NQ / 2 ? q * 4 : 32 + (q - NQ / 2) * 4) : -1;
    }
    const uint32_t soff0 = (uint32_t)(((threadIdx.x / NQ) * F_PS + (threadIdx.x % NQ) * 4) * 4);
    auto stage = [&](int chunk, int buf) {
        const uint32_t dst = patch_u32 + (uint32_t)(buf * F_PH * F_PW * F_PS * 4) + soff0;
        const float* g = xb + chunk * (F_CH / 2);  // F_CH bf16 = F_CH/2 words per chunk and half
#pragma unroll
        for (int i = 0; i < kStage; ++i)
            if (goff[i] >= 0)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)((128 / NQ) * F_PS * 4 * i)), "l"(g + goff[i])
                             : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    float2 acc[ROWS][2];
#pragma unroll
    for (int i = 0; i < ROWS; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
    const int nchunks = cin / F_CH;
    stage(0, 0);
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) {
            stage(c + 1, (c + 1) & 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();  // chunk c visible to every thread (and the weights, first time round)
        const float* pb = patch + (size_t)(c & 1) * F_PH * F_PW * F_PS;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                float4 xr[ROWS + 2];
#pragma unroll
                for (int r = 0; r < ROWS + 2; ++r) {
                    const float* pp = pb + (size_t)((ROWS * yg + r) * F_PW + lx + dx) * F_PS;
                    const uint2 hw = *reinterpret_cast<const uint2*>(pp + q * 2);
                    const uint2 lw = *reinterpret_cast<const uint2*>(pp + F_CH / 2 + q * 2);
                    xr[r] = make_float4(__uint_as_float(hw.x << 16) + __uint_as_float(lw.x << 16),
                                        __uint_as_float(hw.x & 0xffff0000u) + __uint_as_float(lw.x & 0xffff0000u),
                                        __uint_as_float(hw.y << 16) + __uint_as_float(lw.y << 16),
                                        __uint_as_float(hw.y & 0xffff0000u) + __uint_as_float(lw.y & 0xffff0000u));
                }
#pragma unroll
                for (int dy = 0; dy < 3; ++dy) {
                    const float4* wp = wq + (size_t)((dy * 3 + dx) * (cin / 4) + c * NQ + q) * 2;
                    const float4 w0 = wp[0], w1 = wp[1];
#pragma unroll
                    for (int i = 0; i < ROWS; ++i) {
                        const float4 v = xr[i + dy];
                        ffma2(acc[i][0], v.x, v.y, w0.x, w0.y);
                        ffma2(acc[i][0], v.z, v.w, w0.z, w0.w);
                        ffma2(acc[i][1], v.x, v.y, w1.x, w1.y);
                        ffma2(acc[i][1], v.z, v.w, w1.z, w1.w);
                    }
                }
            }
        }
        __syncthreads();  // everyone done with buffer c&1 before chunk c+2 overwrites it
    }
    const float b0 = bias ? bias[0] : 0.f, b1 = bias ? bias[1] : 0.f;
#pragma unroll
    for (int i = 0; i < ROWS; ++i) {
        const int oy = y0 + ROWS * yg + i, ox = x0 + lx;
        if (oy < H && ox < W) {
            const long long p = ((long long)b * H + oy) * W + ox;
            const float2 e = reinterpret_cast<const float2*>(eta)[p];
            reinterpret_cast<float2*>(out)[p] =
                make_float2(e.x + ((acc[i][0].x + acc[i][0].y) + b0), e.y + ((acc[i][1].x + acc[i][1].y) + b1));
        }
    }
}

template <int ROWS, int F_CH>
static int launch_c2_k3(const float* x, const float* w, const float* bias, const float* eta, float* out, int B, int H, int W,
                        int cin, cudaStream_t st) {
    constexpr int F_TY = 4 * ROWS, F_PH = F_TY + 2, F_PS = F_CH + 4;
    const size_t smem3 = (size_t)9 * (cin / 4) * 2 * sizeof(float4) + (size_t)2 * F_PH * F_PW * F_PS * sizeof(float);
    MRB_REQUIRE(smem3 <= 200 * 1024 && (long long)H * W * cin < 2147483647LL, MRB_EUNSUPPORTED,
                "mrb_conv_c2_bh_residual: image or channel count too large");
    MRB_REQUIRE((long long)(H + 4) * (W + 4) * 64 < 2147483647LL && cin == 64, MRB_EUNSUPPORTED,
                "mrb_conv_c2_bh_residual: needs 64 channels and < 2^31 words per image");
    static bool attr_set = false;
    if (!attr_set) {
        MRB_CUDA(cudaFuncSetAttribute(conv_c2_k3_kernel<ROWS, F_CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_set = true;
    }
    dim3 grid3((unsigned)(ceil_div(W, F_TX) * ceil_div(H, F_TY)), (unsigned)B);
    conv_c2_k3_kernel<ROWS, F_CH><<<grid3, 128, smem3, st>>>(x, w, bias, eta, out, B, H, W, cin);
    MRB_LAUNCHED();
    return MRB_OK;
}

}  // namespace mrb

using namespace mrb;

// The final conv on a BH source (64 channels, k = 3, dilation 1; the border of x must be valid: mrb_bh_fix_border).
// 4 rows per thread, 16-channel chunks (98 KB, two CTAs per SM).
extern "C" int mrb_conv_c2_bh_residual(const void* x_bh, const void* w, const void* bias, const void* eta, void* out, int B,
                                       int H, int W, void* stream) {
    MRB_REQUIRE(x_bh && w && eta && out, MRB_EINVAL, "mrb_conv_c2_bh_residual: null pointer");
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1 && B <= 65535, MRB_EINVAL, "mrb_conv_c2_bh_residual: bad shape");
    return launch_c2_k3<4, 16>((const float*)x_bh, (const float*)w, (const float*)bias, (const float*)eta, (float*)out, B, H,
                                     W, 64, (cudaStream_t)stream);
}

extern "C" int mrb_conv2d(const void* x, long long x_bstride, const void* w, const void* bias, void* out,
                          long long out_bstride, int N, int Cin, int Cout, int H, int W, int k, int dil, int pad_mode,
                          int act, float slope, const void* add, const void* add_scale, const void* residual,
                          int out_nhwc_residual, void* stream) {
    MRB_REQUIRE(x && w && out, MRB_EINVAL, "mrb_conv2d: null pointer");
    MRB_REQUIRE(N >= 1 && Cin >= 1 && Cout >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_conv2d: bad shape");
    MRB_REQUIRE(k >= 1 && (k % 2) == 1 && dil >= 1, MRB_EINVAL, "mrb_conv2d: kernel must be odd (got %d), dil >= 1", k);
    MRB_REQUIRE(pad_mode == MRB_PAD_ZERO || pad_mode == MRB_PAD_REPLICATE, MRB_EINVAL, "mrb_conv2d: bad pad mode");
    MRB_REQUIRE(act >= 0 && act <= 2, MRB_EINVAL, "mrb_conv2d: bad activation");
    MRB_REQUIRE(!out_nhwc_residual || residual, MRB_EINVAL, "mrb_conv2d: residual required");
    MRB_REQUIRE(N <= 65535, MRB_EUNSUPPORTED, "mrb_conv2d: N > 65535");
    ConvParams P;
    P.x = (const float*)x; P.w = (const float*)w; P.bias = (const float*)bias; P.out = (float*)out;
    P.add = (const float*)add; P.add_scale = (const float*)add_scale; P.residual = (const float*)residual;
    P.x_bs = x_bstride; P.out_bs = out_bstride;
    P.N = N; P.Cin = Cin; P.Cout = Cout; P.H = H; P.W = W; P.k = k; P.dil = dil;
    P.pad = dil * (k - 1) / 2; P.pad_mode = pad_mode; P.act = act; P.nhwc_res = out_nhwc_residual; P.slope = slope;
    P.PH = TH + 2 * P.pad;
    P.PW = TW + 2 * P.pad;
    P.PWs = ((P.PW + 3) / 4) * 4 + 4;
    P.tiles_x = ceil_div(W, TW);
    const int TN = Cout > 32 ? 8 : (Cout > 16 ? 4 : (Cout > 8 ? 2 : 1));
    const int BN = 8 * TN;
    int CK = 8;
    auto smem_for = [&](int ck) {
        return (size_t)((size_t)ck * P.PH * P.PWs + 16 + 8 + (size_t)ck * k * k * BN) * sizeof(float);
    };
    while (CK > 1 && (CK > Cin || smem_for(CK) > 64 * 1024)) CK /= 2;
    MRB_REQUIRE(smem_for(CK) <= 96 * 1024, MRB_EUNSUPPORTED, "mrb_conv2d: k=%d dil=%d needs too much shared memory", k, dil);
    P.CK = CK;
    dim3 grid((unsigned)(P.tiles_x * ceil_div(H, TH)), (unsigned)ceil_div(Cout, BN), (unsigned)N);
    cudaStream_t st = (cudaStream_t)stream;
    switch (TN) {
        case 8: return launch_conv_tn<8>(P, grid, smem_for(CK), st);
        case 4: return launch_conv_tn<4>(P, grid, smem_for(CK), st);
        case 2: return launch_conv_tn<2>(P, grid, smem_for(CK), st);
        default: return launch_conv_tn<1>(P, grid, smem_for(CK), st);
    }
}

extern "C" int mrb_gru_cell_1x1(const void* x, const void* h, const void* w_ih, const void* b_ih, const void* w_hh,
                                void* h_out, int N, int Cx, int Ch, long long HW, void* stream) {
    MRB_REQUIRE(x && h && w_ih && w_hh && h_out, MRB_EINVAL, "mrb_gru_cell_1x1: null pointer");
    MRB_REQUIRE(h_out != h, MRB_EINVAL, "mrb_gru_cell_1x1: h_out must not alias h");
    MRB_REQUIRE(N >= 1 && Cx >= 1 && Ch >= 1 && HW >= 1 && N <= 65535, MRB_EINVAL, "mrb_gru_cell_1x1: bad shape");
    GruParams P{(const float*)x, (const float*)h, (const float*)w_ih, (const float*)b_ih, (const float*)w_hh,
                (float*)h_out, N, Cx, Ch, HW};
    dim3 grid((unsigned)ceil_div(HW, GRU_PX), (unsigned)ceil_div(Ch, GRU_CH), (unsigned)N);
    gru_cell_1x1_kernel<<<grid, GRU_THREADS, 0, (cudaStream_t)stream>>>(P);
    MRB_LAUNCHED();
    return MRB_OK;
}

static unsigned pw_grid(long long total) {
    long long b = (total + 255) / 256, cap = (long long)device_sm_count() * 16;
    return (unsigned)(b > cap ? cap : (b < 1 ? 1 : b));
}

extern "C" int mrb_gru_gates(const void* ih, const void* hh, const void* h, void* h_out, int N, int Ch, long long HW,
                             void* stream) {
    MRB_REQUIRE(ih && hh && h && h_out && N >= 1 && Ch >= 1 && HW >= 1, MRB_EINVAL, "mrb_gru_gates: bad argument");
    gru_gates_kernel<<<pw_grid((long long)N * Ch * HW), 256, 0, (cudaStream_t)stream>>>(
        (const float*)ih, (const float*)hh, (const float*)h, (float*)h_out, N, Ch, HW);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_mgu_gates(const void* ih, const void* hh, const void* h, void* h_out, int N, int Ch, long long HW,
                             void* stream) {
    MRB_REQUIRE(ih && hh && h && h_out && N >= 1 && Ch >= 1 && HW >= 1, MRB_EINVAL, "mrb_mgu_gates: bad argument");
    mgu_gates_kernel<<<pw_grid((long long)N * Ch * HW), 256, 0, (cudaStream_t)stream>>>(
        (const float*)ih, (const float*)hh, (const float*)h, (float*)h_out, N, Ch, HW);
    MRB_LAUNCHED();
    return MRB_OK;
}
