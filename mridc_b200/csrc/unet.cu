// U-Net regulariser support kernels (NCHW fp32): instance norm + LeakyReLU, 2x2 average pool, 2x2 stride-2
// transposed convolution, pad/crop, and the NormUnet group-norm prologue / epilogue.
// Reference behaviour: mridc/collections/reconstruction/models/unet_base/unet_block.py:11-308.
// Statistics are accumulated in fp64 (sum, sum of squares) so the fp32 result is independent of the
// reduction order to well below fp32 round-off (E2EVN's fp32 noise floor is only ~4x under the tolerance).
#include <cooperative_groups.h>

#include <algorithm>

#include "common.cuh"

namespace mrb {
namespace cg = cooperative_groups;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// stats[2*plane + {0,1}] = (sum, sumsq) of one plane (planes are x + n*bs + c*HW).  A cluster of PS_CLUSTER CTAs owns a
// plane: element i is summed by thread i mod (PS_CLUSTER * PS_THREADS), four loads in flight per thread, and the CTA
// partials are combined through distributed shared memory in rank order.  The order of every addition is fixed by HW
// alone, so the statistics are the same bits run to run and whatever the number of planes in the launch (the atomics of a
// plane-count-dependent grid were neither).  The price: a launch of few planes reads them with 8 CTAs each.
constexpr int PS_CLUSTER = 8, PS_THREADS = 1024, PS_UNROLL = 4;
__global__ void __launch_bounds__(PS_THREADS) plane_stats_kernel(const float* __restrict__ x, long long bs, int C,
                                                                 long long HW, double* __restrict__ stats) {
    cg::cluster_group cluster = cg::this_cluster();
    const int cs = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int plane = blockIdx.x / cs;
    const int n = plane / C, c = plane - n * C;
    const float* p = x + (long long)n * bs + (long long)c * HW;
    double s = 0.0, ss = 0.0;
    const long long T = (long long)cs * PS_THREADS;
    for (long long i = (long long)rank * PS_THREADS + threadIdx.x; i < HW; i += PS_UNROLL * T) {
        float v[PS_UNROLL];
#pragma unroll
        for (int u = 0; u < PS_UNROLL; ++u) v[u] = i + u * T < HW ? __ldg(p + i + u * T) : 0.f;
#pragma unroll
        for (int u = 0; u < PS_UNROLL; ++u) {
            const double d = (double)v[u];
            s += d;
            ss += d * d;
        }
    }
    __shared__ double sh[2][32];
    __shared__ double part[2];
    s = warp_sum(s);
    ss = warp_sum(ss);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { sh[0][wid] = s; sh[1][wid] = ss; }
    __syncthreads();
    if (wid == 0) {
        const int nw = blockDim.x >> 5;
        s = lane < nw ? sh[0][lane] : 0.0;
        ss = lane < nw ? sh[1][lane] : 0.0;
        s = warp_sum(s);
        ss = warp_sum(ss);
        if (lane == 0) { part[0] = s; part[1] = ss; }
    }
    cluster.sync();  // every CTA's partial sums are published
    if (rank == 0 && threadIdx.x == 0) {
        double ts = 0.0, tss = 0.0;
        for (int r = 0; r < cs; ++r) {
            const double* rp = cluster.map_shared_rank(part, r);
            ts += rp[0];
            tss += rp[1];
        }
        stats[2 * plane] = ts;
        stats[2 * plane + 1] = tss;
    }
    cluster.sync();  // remote reads done before any CTA of the cluster may exit
}

__global__ void instnorm_apply_kernel(const float* __restrict__ x, long long xbs, float* __restrict__ out,
                                      long long obs, int C, long long HW, const double* __restrict__ stats, float eps,
                                      float slope) {
    const int plane = blockIdx.y;
    const int n = plane / C, c = plane - n * C;
    const double mean = stats[2 * plane] / (double)HW;
    double var = stats[2 * plane + 1] / (double)HW - mean * mean;  // biased variance (InstanceNorm2d)
    if (var < 0.0) var = 0.0;
    const float m = (float)mean;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float* p = x + (long long)n * xbs + (long long)c * HW;
    float* o = out + (long long)n * obs + (long long)c * HW;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < HW; i += (long long)gridDim.x * blockDim.x) {
        float v = (p[i] - m) * rstd;
        o[i] = v > 0.f ? v : v * slope;
    }
}

// InstanceNorm2d + LeakyReLU in ONE pass over global memory: a thread-block cluster owns one (n, c) plane, every CTA keeps
// its share of the plane in shared memory while it accumulates the fp64 sums, the per-CTA sums are exchanged through
// distributed shared memory (fixed rank order: the statistics do not depend on scheduling), and the normalised values are
// written from shared memory.  1 read + 1 write per element instead of the 2 reads + 1 write and two launches (statistics,
// apply) of the two-kernel form.  In-place use (out == x) is safe: an element is read before its own CTA writes it.
constexpr int IN_THREADS = 512;
__global__ void __launch_bounds__(IN_THREADS) instnorm_cluster_kernel(const float* __restrict__ x, long long xbs, float* out,
                                                                      long long obs, int C, int HW, int chunk, float eps,
                                                                      float slope) {
    extern __shared__ __align__(16) float in_buf[];
    __shared__ double part[2];
    __shared__ double sh[2][IN_THREADS / 32];
    cg::cluster_group cluster = cg::this_cluster();
    const int cs = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int plane = blockIdx.x / cs;
    const int n = plane / C, c = plane - n * C;
    const float* p = x + (long long)n * xbs + (long long)c * HW;
    float* o = out + (long long)n * obs + (long long)c * HW;
    const int beg = rank * chunk, end = min(HW, beg + chunk);  // chunk is a multiple of 4
    const int cnt = max(0, end - beg);
    const bool vec = ((reinterpret_cast<uintptr_t>(p + beg) | reinterpret_cast<uintptr_t>(o + beg)) & 15) == 0 && (cnt & 3) == 0;
    double s = 0.0, ss = 0.0;
    if (vec) {
        const float4* p4 = reinterpret_cast<const float4*>(p + beg);
        for (int i = threadIdx.x; i < cnt / 4; i += IN_THREADS) {
            const float4 v = __ldg(p4 + i);
            reinterpret_cast<float4*>(in_buf)[i] = v;
            s += ((double)v.x + (double)v.y) + ((double)v.z + (double)v.w);
            ss += ((double)v.x * v.x + (double)v.y * v.y) + ((double)v.z * v.z + (double)v.w * v.w);
        }
    } else {
        for (int i = threadIdx.x; i < cnt; i += IN_THREADS) {
            const float v = p[beg + i];
            in_buf[i] = v;
            s += (double)v;
            ss += (double)v * v;
        }
    }
    s = warp_sum(s);
    ss = warp_sum(ss);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { sh[0][wid] = s; sh[1][wid] = ss; }
    __syncthreads();
    if (wid == 0) {
        s = lane < IN_THREADS / 32 ? sh[0][lane] : 0.0;
        ss = lane < IN_THREADS / 32 ? sh[1][lane] : 0.0;
        s = warp_sum(s);
        ss = warp_sum(ss);
        if (lane == 0) { part[0] = s; part[1] = ss; }
    }
    cluster.sync();  // every CTA's partial sums are published
    double ts = 0.0, tss = 0.0;
    for (int r = 0; r < cs; ++r) {
        const double* rp = cluster.map_shared_rank(part, r);
        ts += rp[0];
        tss += rp[1];
    }
    cluster.sync();  // remote reads done before any CTA of the cluster may exit
    const double mean = ts / (double)HW;
    double var = tss / (double)HW - mean * mean;  // biased variance (InstanceNorm2d)
    if (var < 0.0) var = 0.0;
    const float m = (float)mean;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    if (vec) {
        float4* o4 = reinterpret_cast<float4*>(o + beg);
        for (int i = threadIdx.x; i < cnt / 4; i += IN_THREADS) {
            float4 v = reinterpret_cast<const float4*>(in_buf)[i];
            v.x = (v.x - m) * rstd; v.y = (v.y - m) * rstd; v.z = (v.z - m) * rstd; v.w = (v.w - m) * rstd;
            v.x = v.x > 0.f ? v.x : v.x * slope; v.y = v.y > 0.f ? v.y : v.y * slope;
            v.z = v.z > 0.f ? v.z : v.z * slope; v.w = v.w > 0.f ? v.w : v.w * slope;
            o4[i] = v;
        }
    } else {
        for (int i = threadIdx.x; i < cnt; i += IN_THREADS) {
            const float v = (in_buf[i] - m) * rstd;
            o[beg + i] = v > 0.f ? v : v * slope;
        }
    }
}

// 1x1 convolution with bias (the last layer of the U-Net, unet_block.py:185: Conv2d(ch, out_chans, kernel_size=1)): one
// thread = four consecutive pixels x up to four output channels; every input plane is read once with 16-byte loads.
__global__ void conv1x1_kernel(const float* __restrict__ x, long long xbs, const float* __restrict__ w,
                               const float* __restrict__ bias, float* __restrict__ out, long long obs, int Cin, int Cout,
                               long long HW4) {
    const int n = blockIdx.z, co0 = blockIdx.y * 4;
    const int nco = min(4, Cout - co0);
    const float4* p = reinterpret_cast<const float4*>(x + (long long)n * xbs);
    float4* o = reinterpret_cast<float4*>(out + (long long)n * obs);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < HW4; i += (long long)gridDim.x * blockDim.x) {
        float4 acc[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float b = (bias && j < nco) ? bias[co0 + j] : 0.f;
            acc[j] = make_float4(b, b, b, b);
        }
        for (int c = 0; c < Cin; ++c) {
            const float4 v = __ldg(p + (long long)c * HW4 + i);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (j < nco) {
                    const float wv = __ldg(w + (long long)(co0 + j) * Cin + c);
                    acc[j].x = fmaf(v.x, wv, acc[j].x); acc[j].y = fmaf(v.y, wv, acc[j].y);
                    acc[j].z = fmaf(v.z, wv, acc[j].z); acc[j].w = fmaf(v.w, wv, acc[j].w);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (j < nco) o[(long long)(co0 + j) * HW4 + i] = acc[j];
    }
}

__global__ void avgpool2_kernel(const float* __restrict__ x, long long xbs, float* __restrict__ out, long long obs,
                                int C, int H, int W) {
    const int Ho = H / 2, Wo = W / 2;
    const int plane = blockIdx.y;
    const int n = plane / C, c = plane - n * C;
    const float* p = x + (long long)n * xbs + (long long)c * H * W;
    float* o = out + (long long)n * obs + (long long)c * Ho * Wo;
    const long long total = (long long)Ho * Wo;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int yo = (int)(i / Wo), xo = (int)(i - (long long)yo * Wo);
        const float* q = p + (long long)(2 * yo) * W + 2 * xo;
        o[i] = (q[0] + q[1] + q[W] + q[W + 1]) * 0.25f;
    }
}

// out[n,co,2y+dy,2x+dx] = sum_ci x[n,ci,y,x] * w[ci,co,dy,dx]; thread = one input pixel x 8 output channels.
constexpr int TC_CO = 8;
__global__ void conv_transpose2x2_kernel(const float* __restrict__ x, long long xbs, const float* __restrict__ w,
                                         float* __restrict__ out, long long obs, int Cin, int Cout, int H, int W) {
    extern __shared__ float wsh[];  // [Cin][TC_CO][4]
    const int co0 = blockIdx.y * TC_CO;
    const int n = blockIdx.z;
    for (int t = threadIdx.x; t < Cin * TC_CO * 4; t += blockDim.x) {
        int q = t % 4, r = t / 4;
        int co = r % TC_CO, ci = r / TC_CO;
        wsh[t] = (co0 + co < Cout) ? w[((long long)ci * Cout + co0 + co) * 4 + q] : 0.f;
    }
    __syncthreads();
    const long long HW = (long long)H * W;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= HW) return;
    const int y = (int)(i / W), xx = (int)(i - (long long)y * W);
    float acc[TC_CO][4];
#pragma unroll
    for (int a = 0; a < TC_CO; ++a)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[a][q] = 0.f;
    const float* p = x + (long long)n * xbs + i;
    for (int ci = 0; ci < Cin; ++ci) {
        const float v = p[(long long)ci * HW];
        const float4* wr = reinterpret_cast<const float4*>(wsh + (size_t)ci * TC_CO * 4);
#pragma unroll
        for (int a = 0; a < TC_CO; ++a) {
            float4 w4 = wr[a];
            acc[a][0] = fmaf(v, w4.x, acc[a][0]);
            acc[a][1] = fmaf(v, w4.y, acc[a][1]);
            acc[a][2] = fmaf(v, w4.z, acc[a][2]);
            acc[a][3] = fmaf(v, w4.w, acc[a][3]);
        }
    }
    const int Wo = 2 * W;
#pragma unroll
    for (int a = 0; a < TC_CO; ++a) {
        if (co0 + a >= Cout) break;
        float* o = out + (long long)n * obs + (long long)(co0 + a) * 4 * HW + (long long)(2 * y) * Wo + 2 * xx;
        *reinterpret_cast<float2*>(o) = make_float2(acc[a][0], acc[a][1]);
        *reinterpret_cast<float2*>(o + Wo) = make_float2(acc[a][2], acc[a][3]);
    }
}

__global__ void pad2d_kernel(const float* __restrict__ x, long long xbs, float* __restrict__ out, long long obs, int C,
                             int Hin, int Win, int Hout, int Wout, int off_y, int off_x, int mode) {
    const int plane = blockIdx.y;
    const int n = plane / C, c = plane - n * C;
    const float* p = x + (long long)n * xbs + (long long)c * Hin * Win;
    float* o = out + (long long)n * obs + (long long)c * Hout * Wout;
    const long long total = (long long)Hout * Wout;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        int yo = (int)(i / Wout), xo = (int)(i - (long long)yo * Wout);
        int yi = yo - off_y, xi = xo - off_x;
        float v = 0.f;
        if (mode == 1) {
            yi = min(max(yi, 0), Hin - 1);
            xi = min(max(xi, 0), Win - 1);
            v = p[(long long)yi * Win + xi];
        } else if (mode == 2) {
            if (yi < 0) yi = -yi;
            if (yi >= Hin) yi = 2 * (Hin - 1) - yi;
            if (xi < 0) xi = -xi;
            if (xi >= Win) xi = 2 * (Win - 1) - xi;
            v = p[(long long)yi * Win + xi];
        } else if (yi >= 0 && yi < Hin && xi >= 0 && xi < Win) {
            v = p[(long long)yi * Win + xi];
        }
        o[i] = v;
    }
}

// stats over the re (g=0) / im (g=1) parts of x [B, C*HW, 2] -> stats[(b*2+g)*2 + {0,1}]
__global__ void normunet_stats_kernel(const float2* __restrict__ x, long long per_b, double* __restrict__ stats) {
    const int b = blockIdx.y;
    const float2* p = x + (long long)b * per_b;
    double s0 = 0, q0 = 0, s1 = 0, q1 = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_b; i += (long long)gridDim.x * blockDim.x) {
        float2 v = p[i];
        s0 += v.x; q0 += (double)v.x * v.x;
        s1 += v.y; q1 += (double)v.y * v.y;
    }
    __shared__ double sh[4][32];
    s0 = warp_sum(s0); q0 = warp_sum(q0); s1 = warp_sum(s1); q1 = warp_sum(q1);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { sh[0][wid] = s0; sh[1][wid] = q0; sh[2][wid] = s1; sh[3][wid] = q1; }
    __syncthreads();
    if (wid == 0) {
        const int nw = blockDim.x >> 5;
        s0 = lane < nw ? sh[0][lane] : 0.0; q0 = lane < nw ? sh[1][lane] : 0.0;
        s1 = lane < nw ? sh[2][lane] : 0.0; q1 = lane < nw ? sh[3][lane] : 0.0;
        s0 = warp_sum(s0); q0 = warp_sum(q0); s1 = warp_sum(s1); q1 = warp_sum(q1);
        if (lane == 0) {
            atomicAdd(&stats[(b * 2 + 0) * 2 + 0], s0);
            atomicAdd(&stats[(b * 2 + 0) * 2 + 1], q0);
            atomicAdd(&stats[(b * 2 + 1) * 2 + 0], s1);
            atomicAdd(&stats[(b * 2 + 1) * 2 + 1], q1);
        }
    }
}

__global__ void normunet_finalize_kernel(const double* __restrict__ stats, float* __restrict__ mean_std, int B2,
                                         long long cnt) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B2) return;
    double mean = stats[2 * i] / (double)cnt;
    double var = (stats[2 * i + 1] - (double)cnt * mean * mean) / (double)(cnt - 1);  // unbiased (torch.std)
    if (var < 0.0) var = 0.0;
    mean_std[2 * i] = (float)mean;
    mean_std[2 * i + 1] = (float)sqrt(var);
}

// x [B,C,HW,2] -> out [B,2C,HW] : out[b, g*C + c, p] = (x[b,c,p,g] - mean[b,g]) / std[b,g]
__global__ void normunet_in_kernel(const float2* __restrict__ x, float* __restrict__ out,
                                   const float* __restrict__ mean_std, int C, long long HW, int normalize) {
    const int b = blockIdx.y;
    float m0 = 0.f, s0 = 1.f, m1 = 0.f, s1 = 1.f;
    if (normalize) {
        m0 = mean_std[(b * 2) * 2]; s0 = mean_std[(b * 2) * 2 + 1];
        m1 = mean_std[(b * 2 + 1) * 2]; s1 = mean_std[(b * 2 + 1) * 2 + 1];
    }
    const long long per_b = (long long)C * HW;
    const float2* p = x + (long long)b * per_b;
    float* o = out + (long long)b * 2 * per_b;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_b; i += (long long)gridDim.x * blockDim.x) {
        float2 v = p[i];
        if (normalize) {
            o[i] = (v.x - m0) / s0;
            o[per_b + i] = (v.y - m1) / s1;
        } else {
            o[i] = v.x;
            o[per_b + i] = v.y;
        }
    }
}

__global__ void normunet_out_kernel(const float* __restrict__ x, const float* __restrict__ mean_std,
                                    float2* __restrict__ out, int C, long long HW, int normalize) {
    const int b = blockIdx.y;
    float m0 = 0.f, s0 = 1.f, m1 = 0.f, s1 = 1.f;
    if (normalize) {
        m0 = mean_std[(b * 2) * 2]; s0 = mean_std[(b * 2) * 2 + 1];
        m1 = mean_std[(b * 2 + 1) * 2]; s1 = mean_std[(b * 2 + 1) * 2 + 1];
    }
    const long long per_b = (long long)C * HW;
    const float* p = x + (long long)b * 2 * per_b;
    float2* o = out + (long long)b * per_b;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_b; i += (long long)gridDim.x * blockDim.x) {
        float re = p[i], im = p[per_b + i];
        if (normalize) { re = re * s0 + m0; im = im * s1 + m1; }
        o[i] = make_float2(re, im);
    }
}

static unsigned split_grid(long long per_plane, int planes) {
    long long b = (per_plane + 255) / 256;
    long long cap = ((long long)device_sm_count() * 8 + planes - 1) / planes;
    if (cap < 1) cap = 1;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

}  // namespace mrb

using namespace mrb;

extern "C" int mrb_instnorm_lrelu(const void* x, long long x_bstride, void* out, long long out_bstride, int N, int C,
                                  long long HW, float eps, float slope, void* stats, void* stream) {
    MRB_REQUIRE(x && out && stats, MRB_EINVAL, "mrb_instnorm_lrelu: null pointer");
    MRB_REQUIRE(N >= 1 && C >= 1 && HW >= 1 && (long long)N * C <= 65535, MRB_EINVAL, "mrb_instnorm_lrelu: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    const int planes = N * C;
    if (HW < 2147483647LL / 4 && !getenv("MRIDC_B200_INSTNORM_2PASS")) {
        // single-pass cluster form: 2 .. 8 CTAs per plane, each holding <= 64 KB of it in shared memory (one CTA for
        // planes up to 64 KB; planes above 8 x 200 KB take the two-kernel form below)
        int cs = 1;
        while (cs < 8 && (HW * 4 + cs - 1) / cs > 65536) cs *= 2;
        const int chunk = (int)((((HW + cs - 1) / cs) + 3) & ~3LL);
        const size_t smem = (size_t)chunk * 4;
        if (smem <= 200 * 1024 && (long long)planes * cs < 2147483647LL) {
            static bool attr_set = false;
            if (!attr_set) {
                MRB_CUDA(cudaFuncSetAttribute(instnorm_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
                attr_set = true;
            }
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(planes * cs));
            cfg.blockDim = dim3(IN_THREADS);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = (unsigned)cs;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            MRB_CUDA(cudaLaunchKernelEx(&cfg, instnorm_cluster_kernel, (const float*)x, x_bstride, (float*)out, out_bstride, C,
                                        (int)HW, chunk, eps, slope));
            MRB_LAUNCHED();
            return MRB_OK;
        }
    }
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(planes * PS_CLUSTER));
        cfg.blockDim = dim3(PS_THREADS);
        cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)PS_CLUSTER;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        MRB_CUDA(cudaLaunchKernelEx(&cfg, plane_stats_kernel, (const float*)x, x_bstride, C, HW, (double*)stats));
        MRB_LAUNCHED();
    }
    dim3 grid(split_grid(HW, planes), planes);
    instnorm_apply_kernel<<<grid, 256, 0, st>>>((const float*)x, x_bstride, (float*)out, out_bstride, C, HW,
                                                (const double*)stats, eps, slope);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_conv1x1(const void* x, long long x_bstride, const void* w, const void* bias, void* out,
                           long long out_bstride, int N, int Cin, int Cout, long long HW, void* stream) {
    MRB_REQUIRE(x && w && out, MRB_EINVAL, "mrb_conv1x1: null pointer");
    MRB_REQUIRE(N >= 1 && N <= 65535 && Cin >= 1 && Cout >= 1 && Cout <= 4 * 65535 && HW >= 1, MRB_EINVAL, "mrb_conv1x1: bad shape");
    MRB_REQUIRE((HW & 3) == 0 && (x_bstride & 3) == 0 && (out_bstride & 3) == 0 &&
                    ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
                MRB_EUNSUPPORTED, "mrb_conv1x1: planes must be 16-byte aligned (H*W and the batch strides multiples of 4)");
    const long long HW4 = HW / 4;
    const unsigned gx = (unsigned)std::min<long long>((HW4 + 255) / 256, (long long)device_sm_count() * 8);
    conv1x1_kernel<<<dim3(gx, (unsigned)((Cout + 3) / 4), (unsigned)N), 256, 0, (cudaStream_t)stream>>>(
        (const float*)x, x_bstride, (const float*)w, (const float*)bias, (float*)out, out_bstride, Cin, Cout, HW4);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_avgpool2(const void* x, long long x_bstride, void* out, long long out_bstride, int N, int C, int H,
                            int W, void* stream) {
    MRB_REQUIRE(x && out, MRB_EINVAL, "mrb_avgpool2: null pointer");
    MRB_REQUIRE(N >= 1 && C >= 1 && H >= 2 && W >= 2 && (long long)N * C <= 65535, MRB_EINVAL, "mrb_avgpool2: bad shape");
    const int planes = N * C;
    dim3 grid(split_grid((long long)(H / 2) * (W / 2), planes), planes);
    avgpool2_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)x, x_bstride, (float*)out, out_bstride, C, H, W);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_conv_transpose2x2(const void* x, long long x_bstride, const void* w, void* out,
                                     long long out_bstride, int N, int Cin, int Cout, int H, int W, void* stream) {
    MRB_REQUIRE(x && w && out, MRB_EINVAL, "mrb_conv_transpose2x2: null pointer");
    MRB_REQUIRE(N >= 1 && Cin >= 1 && Cout >= 1 && H >= 1 && W >= 1 && N <= 65535, MRB_EINVAL,
                "mrb_conv_transpose2x2: bad shape");
    size_t smem = (size_t)Cin * TC_CO * 4 * sizeof(float);
    MRB_REQUIRE(smem <= 96 * 1024, MRB_EUNSUPPORTED, "mrb_conv_transpose2x2: Cin=%d too large", Cin);
    MRB_CUDA(cudaFuncSetAttribute(conv_transpose2x2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    dim3 grid((unsigned)ceil_div((long long)H * W, 128), (unsigned)ceil_div(Cout, TC_CO), (unsigned)N);
    conv_transpose2x2_kernel<<<grid, 128, smem, (cudaStream_t)stream>>>((const float*)x, x_bstride, (const float*)w,
                                                                        (float*)out, out_bstride, Cin, Cout, H, W);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_pad2d(const void* x, long long x_bstride, void* out, long long out_bstride, int N, int C, int Hin,
                         int Win, int Hout, int Wout, int off_y, int off_x, int mode, void* stream) {
    MRB_REQUIRE(x && out, MRB_EINVAL, "mrb_pad2d: null pointer");
    MRB_REQUIRE(N >= 1 && C >= 1 && Hin >= 1 && Win >= 1 && Hout >= 1 && Wout >= 1 && (long long)N * C <= 65535,
                MRB_EINVAL, "mrb_pad2d: bad shape");
    MRB_REQUIRE(mode >= 0 && mode <= 2, MRB_EINVAL, "mrb_pad2d: bad mode");
    const int planes = N * C;
    dim3 grid(split_grid((long long)Hout * Wout, planes), planes);
    pad2d_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)x, x_bstride, (float*)out, out_bstride, C, Hin,
                                                         Win, Hout, Wout, off_y, off_x, mode);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_normunet_in(const void* x, void* out, void* mean_std, int B, int C, long long HW, int normalize,
                               void* stats, void* stream) {
    MRB_REQUIRE(x && out, MRB_EINVAL, "mrb_normunet_in: null pointer");
    MRB_REQUIRE(B >= 1 && C >= 1 && HW >= 1 && B <= 65535, MRB_EINVAL, "mrb_normunet_in: bad shape");
    cudaStream_t st = (cudaStream_t)stream;
    const long long per_b = (long long)C * HW;
    dim3 grid(split_grid(per_b, B), B);
    if (normalize) {
        MRB_REQUIRE(mean_std && stats, MRB_EINVAL, "mrb_normunet_in: mean_std/stats required");
        MRB_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 4 * B, st));
        normunet_stats_kernel<<<grid, 256, 0, st>>>((const float2*)x, per_b, (double*)stats);
        MRB_LAUNCHED();
        normunet_finalize_kernel<<<ceil_div(2 * B, 64), 64, 0, st>>>((const double*)stats, (float*)mean_std, 2 * B, per_b);
        MRB_LAUNCHED();
    }
    normunet_in_kernel<<<grid, 256, 0, st>>>((const float2*)x, (float*)out, (const float*)mean_std, C, HW, normalize);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_normunet_out(const void* x, const void* mean_std, void* out, int B, int C, long long HW,
                                int normalize, void* stream) {
    MRB_REQUIRE(x && out && (!normalize || mean_std), MRB_EINVAL, "mrb_normunet_out: null pointer");
    MRB_REQUIRE(B >= 1 && C >= 1 && HW >= 1 && B <= 65535, MRB_EINVAL, "mrb_normunet_out: bad shape");
    const long long per_b = (long long)C * HW;
    dim3 grid(split_grid(per_b, B), B);
    normunet_out_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)x, (const float*)mean_std, (float2*)out,
                                                                C, HW, normalize);
    MRB_LAUNCHED();
    return MRB_OK;
}
