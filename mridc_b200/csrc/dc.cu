// Fused data-consistency operator (SENSE expand -> 2-D FFT -> mask/residual -> inverse FFT -> conj-coil reduce).
//
// Reference behaviour:
//   RIM gradient     mridc/collections/reconstruction/models/rim/rim_utils.py:11-67
//   sens_reduce      mridc/collections/reconstruction/models/varnet/vn_block.py:71-87
//   sens_expand+DC   mridc/collections/reconstruction/models/varnet/vn_block.py:51-69, :109-119
//
// Three passes, intermediates T1/T2 ([B,C,H,W] complex64, caller workspace) stay L2-resident on B200:
//   K1 expand_rowfft      CTA = (b, row h): all coils of the row in smem; p = S*eta, forward FFT along W.
//   K2 col_dc / col_softdc CTA = (b, c, strip of 16 k_w): FFT along H, k-space epilogue, (inverse FFT along H).
//   K3 rowifft_reduce     CTA = (b, row h): inverse FFT along W for all coils in smem, sum_c conj(S)*.
// Centering is folded into index rotations on the loads/stores (valid for odd lengths too); the k-space in
// the middle is never physically shifted.
#include <stdlib.h>

#include "fft.cuh"

namespace mrb {

int fft1d_launch(const float2* in, float2* out, long long outer, int n, long long inner, int inverse, int in_rot,
                 int out_rot, float scale, cudaStream_t st);
float norm_scale(int norm, int inverse, double npts);

// Streamed operands (sensitivity maps, the T1/T2 intermediates): read through L2 only.  The L1 path costs issue slots
// on B200 without any reuse to win (same finding as the tensor-core loaders' cp.async.cg).
#ifndef MRB_DC_LDG
#define LDSTREAM(p) __ldcg(p)
#else
#define LDSTREAM(p) __ldg(p)
#endif
__device__ __forceinline__ int rot_add(int j, int rot, int n) {
    int s = j + rot;
    return s >= n ? s - n : s;
}

// Index arithmetic in these kernels is division-free (profiling showed the `t / W` style decompositions costing
// more instructions than the butterflies): row kernels walk coils in the outer loop and columns across threads
// (blockDim >= W when W <= 1024), column kernels split the thread index with shifts (strip width is a power of two).

// Mask-aware pruning.  With a 1-D mask (one value per k_w column, the fastMRI case) every unsampled k-space column has
// a zero residual, so only the sampled columns need the H-direction transforms and only they need to travel between
// the passes.  Each CTA rebuilds the ascending list of active un-centred k_w indices (cols_s, count returned) from
// the mask row with a ballot scan (W elements; cheaper than a separate launch plus a host-visible count).
// For 2-D masks every column is treated as active (dense path through the same code).
__device__ __forceinline__ int build_active_cols(const MaskDesc& mask, int b, int W, int rw, bool prune,
                                                 unsigned short* cols_s, int* scratch) {
    // scratch: [33] ints (warp totals + grand total)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int base = 0;
    for (int k0 = 0; k0 < W; k0 += blockDim.x) {
        const int kw = k0 + threadIdx.x;
        bool f = false;
        if (kw < W) f = prune ? (mask_value(mask, b, 0, rot_add(kw, rw, W)) != 0.f) : true;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        const int prefix = __popc(bal & ((1u << lane) - 1u));
        if (lane == 0) scratch[wid] = __popc(bal);
        __syncthreads();
        int woff = 0, tot = 0;
        for (int w = 0; w < nw; ++w) {
            const int cnt = scratch[w];
            if (w < wid) woff += cnt;
            tot += cnt;
        }
        if (f) cols_s[base + woff + prefix] = (unsigned short)kw;
        base += tot;
        __syncthreads();
    }
    return base;
}

// K1: T1[b,c,h,kw] = FFT_W( S[b,c,h,(j+rw)%W] * img[b,h,(j+rw)%W] )   (un-normalised, un-centred along W)
// COMPACT: only the active columns are stored, packed at the front of each T1 row (T1c[b,c,h,j] = X[cols[j]]).
template <bool COMPACT>
__global__ void expand_rowfft_kernel(const float2* __restrict__ img, const float2* __restrict__ S,
                                     float2* __restrict__ T1, int C, int H, int W, int cc, FftPlan p, int rw,
                                     MaskDesc mask, int prune) {
    extern __shared__ float2 smem[];
    float2* A = smem;
    float2* Bf = A + (size_t)cc * p.ls;
    float2* tw_s = Bf + (size_t)cc * p.ls;
    unsigned short* cols_s = reinterpret_cast<unsigned short*>(tw_s + p.n);
    __shared__ int scan_scratch[33];
    load_twiddles(tw_s, p);
    const int h = blockIdx.x, b = blockIdx.y;
    int ns = W;
    if (COMPACT) ns = build_active_cols(mask, b, W, rw, prune != 0, cols_s, scan_scratch);
    const float2* irow = img + ((long long)b * H + h) * W;
    const long long cstride = (long long)H * W;
    const float2* Srow = S + ((long long)b * C * H + h) * W;
    float2* Trow = T1 + ((long long)b * C * H + h) * W;
    float2* St = fft_start_buf(p, A, Bf);
    for (int c0 = 0; c0 < C; c0 += cc) {
        const int nc = min(cc, C - c0);
        if (c0 > 0) __syncthreads();
        for (int j = threadIdx.x; j < W; j += blockDim.x) {
            const int src = rot_add(j, rw, W);
            const float2 e = __ldg(&irow[src]);
            const float2* sp = Srow + (long long)c0 * cstride + src;
            float2* dp = St + j;
            int c = 0;
            for (; c + 4 <= nc; c += 4) {  // 4 independent loads in flight
                const float2 s0 = LDSTREAM(sp + (long long)(c + 0) * cstride), s1 = LDSTREAM(sp + (long long)(c + 1) * cstride);
                const float2 s2 = LDSTREAM(sp + (long long)(c + 2) * cstride), s3 = LDSTREAM(sp + (long long)(c + 3) * cstride);
                // rim_utils.py:47-48: re = e_re*s_re - e_im*s_im ; im = e_re*s_im + e_im*s_re
                dp[(size_t)(c + 0) * p.ls] = make_float2(e.x * s0.x - e.y * s0.y, e.x * s0.y + e.y * s0.x);
                dp[(size_t)(c + 1) * p.ls] = make_float2(e.x * s1.x - e.y * s1.y, e.x * s1.y + e.y * s1.x);
                dp[(size_t)(c + 2) * p.ls] = make_float2(e.x * s2.x - e.y * s2.y, e.x * s2.y + e.y * s2.x);
                dp[(size_t)(c + 3) * p.ls] = make_float2(e.x * s3.x - e.y * s3.y, e.x * s3.y + e.y * s3.x);
            }
            for (; c < nc; ++c) {
                const float2 s0 = LDSTREAM(sp + (long long)c * cstride);
                dp[(size_t)c * p.ls] = make_float2(e.x * s0.x - e.y * s0.y, e.x * s0.y + e.y * s0.x);
            }
        }
        block_fft<false>(A, Bf, nc, p, tw_s);
        for (int k = threadIdx.x; k < ns; k += blockDim.x) {
            float2* tp = Trow + (long long)c0 * cstride + k;
            const float2* ap = A + (COMPACT ? (int)cols_s[k] : k);
            for (int c = 0; c < nc; ++c) tp[(long long)c * cstride] = ap[(size_t)c * p.ls];
        }
    }
}

// column-strip helpers: strip of ti = 1 << tsh lines (k_w positions), thread -> (i = tid & (ti-1), row start tid >> tsh)
// K2 (RIM): per (b,c,strip): P = fscale * FFT_H(T1 rotated); r = mask*(P - y); T2 = IFFT_H(r) stored with the
// output rotation along H.  T1's k_w axis is un-centred: centred storage column = (k_w + rw) % W.
// T1 / T2 hold compact rows: column j of the strip is the j-th active k_w (cols_s[j]); strips past the active count exit.
__global__ void col_dc_kernel(const float2* __restrict__ T1, const float2* __restrict__ y, float2* __restrict__ T2,
                              MaskDesc mask, int C, int H, int W, int tsh, FftPlan p, int rh, int rw, float fscale,
                              int prune) {
    extern __shared__ float2 smem[];
    const int ti = 1 << tsh;
    float2* A = smem;
    float2* Bf = A + (size_t)ti * p.ls;
    float2* tw_s = Bf + (size_t)ti * p.ls;
    unsigned short* cols_s = reinterpret_cast<unsigned short*>(tw_s + p.n);
    __shared__ int scan_scratch[33];
    const int c = blockIdx.y, b = blockIdx.z;
    const int ns = build_active_cols(mask, b, W, rw, prune != 0, cols_s, scan_scratch);
    const int k0 = blockIdx.x * ti;
    if (k0 >= ns) return;  // uniform per CTA
    load_twiddles(tw_s, p);
    const int nl = min(ti, ns - k0);
    const long long plane = ((long long)b * C + c) * H * W;
    float2* St = fft_start_buf(p, A, Bf);
    const int i = threadIdx.x & (ti - 1), j0 = threadIdx.x >> tsh, jstep = blockDim.x >> tsh;
    const bool act = i < nl;
    const float2* tcol = T1 + plane + k0 + i;
    if (act) {
        int j = j0;
        for (; j + 3 * jstep < H; j += 4 * jstep) {
            const float2 v0 = LDSTREAM(tcol + (long long)rot_add(j, rh, H) * W), v1 = LDSTREAM(tcol + (long long)rot_add(j + jstep, rh, H) * W);
            const float2 v2 = LDSTREAM(tcol + (long long)rot_add(j + 2 * jstep, rh, H) * W);
            const float2 v3 = LDSTREAM(tcol + (long long)rot_add(j + 3 * jstep, rh, H) * W);
            float2* d = St + (size_t)i * p.ls + j;
            d[0] = v0; d[jstep] = v1; d[2 * jstep] = v2; d[3 * jstep] = v3;
        }
        for (; j < H; j += jstep) St[(size_t)i * p.ls + j] = LDSTREAM(tcol + (long long)rot_add(j, rh, H) * W);
    }
    block_fft<false>(A, Bf, nl, p, tw_s);
    // k-space epilogue: result of the forward FFT is in A; write the residual where the inverse wants its input.
    if (act) {
        const int mw = rot_add((int)cols_s[k0 + i], rw, W);
        for (int kh = j0; kh < H; kh += jstep) {
            const int mh = rot_add(kh, rh, H);
            const float m = mask_value(mask, b, mh, mw);
            const float2 P = cscale(A[(size_t)i * p.ls + kh], fscale);
            float2 r = make_float2(0.f, 0.f);
            if (m != 0.f) {  // unsampled entries contribute exactly 0 whatever y holds: skip the read
                const float2 yv = __ldg(&y[plane + (long long)mh * W + mw]);
                r = make_float2(m * (P.x - yv.x), m * (P.y - yv.y));  // rim_utils.py:54: mask * (pred - masked_kspace)
            }
            // in-place update (St == A) is safe: each (i,kh) is read and written by the same thread
            St[(size_t)i * p.ls + kh] = r;
        }
    }
    block_fft<true>(A, Bf, nl, p, tw_s);
    if (act) {
        float2* ocol = T2 + plane + k0 + i;
        for (int d = j0; d < H; d += jstep) {  // d = storage row (image coordinates), n = logical output index
            int n = d - rh;
            if (n < 0) n += H;
            ocol[(long long)d * W] = A[(size_t)i * p.ls + n];
        }
    }
}

// K2' (VarNet): out[b,c,mh,mw] = no_dc ? E : base - (mask!=0 ? pred - y : 0)*dcw - E,  E = fscale*FFT_H(T1 rot.)
__global__ void col_softdc_kernel(const float2* __restrict__ T1, const float2* __restrict__ base,
                                  const float2* __restrict__ pred,
                                  const float2* __restrict__ y, float2* __restrict__ out, MaskDesc mask, int C, int H,
                                  int W, int tsh, FftPlan p, int rh, int rw, float fscale, const float* __restrict__ dcw_p,
                                  int no_dc) {
    extern __shared__ float2 smem[];
    const int ti = 1 << tsh;
    float2* A = smem;
    float2* Bf = A + (size_t)ti * p.ls;
    float2* tw_s = Bf + (size_t)ti * p.ls;
    load_twiddles(tw_s, p);
    const int k0 = blockIdx.x * ti;
    const int nl = min(ti, W - k0);
    const int c = blockIdx.y, b = blockIdx.z;
    const long long plane = ((long long)b * C + c) * H * W;
    const float dcw = no_dc ? 0.f : *dcw_p;
    float2* St = fft_start_buf(p, A, Bf);
    const int i = threadIdx.x & (ti - 1), j0 = threadIdx.x >> tsh, jstep = blockDim.x >> tsh;
    const bool act = i < nl;
    if (act) {
        const float2* tcol = T1 + plane + k0 + i;
        for (int j = j0; j < H; j += jstep) St[(size_t)i * p.ls + j] = tcol[(long long)rot_add(j, rh, H) * W];
    }
    block_fft<false>(A, Bf, nl, p, tw_s);
    if (act) {
        const int mw = rot_add(k0 + i, rw, W);
        for (int kh = j0; kh < H; kh += jstep) {
            const int mh = rot_add(kh, rh, H);
            const float2 E = cscale(A[(size_t)i * p.ls + kh], fscale);
            const long long o = plane + (long long)mh * W + mw;
            if (no_dc) {
                out[o] = E;
            } else {
                const float2 bv = base[o];
                float2 sd = make_float2(0.f, 0.f);
                if (mask_value(mask, b, mh, mw) != 0.f) {  // vn_block.py:110 torch.where(mask.bool(), pred - ref, 0)
                    const float2 pv = pred[o], yv = y[o];
                    sd = make_float2(pv.x - yv.x, pv.y - yv.y);
                }
                // vn_block.py:110,117: (pred - soft_dc*dc_weight) - eta
                out[o] = make_float2((bv.x - sd.x * dcw) - E.x, (bv.y - sd.y * dcw) - E.y);
            }
        }
    }
}

// K3: acc[b,h,w] = sum_c conj(S[b,c,h,w]) * IFFT_W(T2[b,c,h,:])  ; w = (n + rw) % W.
// OUT_MODE 0: out [B,H,W] complex = acc*scale.   OUT_MODE 1 (RIM): out [B,4,H,W] = (eta_re, eta_im, acc*scale).
// OUT_MODE 2 (RIM, channels-last for the tensor-core regulariser): out [B,H,W,4].
// COMPACT: T2 rows hold only the active columns (packed); they are scattered into zero-filled lines.
template <int OUT_MODE, bool COMPACT>
__global__ void rowifft_reduce_kernel(const float2* __restrict__ T2, const float2* __restrict__ S,
                                      const float2* __restrict__ eta, float* __restrict__ out, int C, int H, int W,
                                      int cc, FftPlan p, int in_rw, int rw, float scale, MaskDesc mask, int prune) {
    extern __shared__ float2 smem[];
    float2* A = smem;
    float2* Bf = A + (size_t)cc * p.ls;
    float2* tw_s = Bf + (size_t)cc * p.ls;
    unsigned short* cols_s = reinterpret_cast<unsigned short*>(tw_s + p.n);
    __shared__ int scan_scratch[33];
    load_twiddles(tw_s, p);
    const int h = blockIdx.x, b = blockIdx.y;
    int ns = W;
    if (COMPACT) ns = build_active_cols(mask, b, W, rw, prune != 0, cols_s, scan_scratch);
    const long long cstride = (long long)H * W;
    const float2* Trow = T2 + ((long long)b * C * H + h) * W;
    const float2* Srow = S + ((long long)b * C * H + h) * W;
    float2* St = fft_start_buf(p, A, Bf);
    // each thread owns output columns d = threadIdx.x + i*blockDim.x (registers hold the running coil sum)
    constexpr int kMaxOwn = 4;
    float2 acc[kMaxOwn];
#pragma unroll
    for (int i = 0; i < kMaxOwn; ++i) acc[i] = make_float2(0.f, 0.f);
    for (int c0 = 0; c0 < C; c0 += cc) {
        const int nc = min(cc, C - c0);
        if (c0 > 0) __syncthreads();
        if (COMPACT && ns < W) {
            for (int j = threadIdx.x; j < W; j += blockDim.x)
                for (int c = 0; c < nc; ++c) St[(size_t)c * p.ls + j] = make_float2(0.f, 0.f);
            __syncthreads();
        }
        for (int j = threadIdx.x; j < ns; j += blockDim.x) {
            const float2* tp = Trow + (long long)c0 * cstride + (COMPACT ? j : rot_add(j, in_rw, W));
            float2* dp = St + (COMPACT ? (int)cols_s[j] : j);
            int c = 0;
            for (; c + 4 <= nc; c += 4) {
                const float2 v0 = LDSTREAM(tp + (long long)(c + 0) * cstride), v1 = LDSTREAM(tp + (long long)(c + 1) * cstride);
                const float2 v2 = LDSTREAM(tp + (long long)(c + 2) * cstride), v3 = LDSTREAM(tp + (long long)(c + 3) * cstride);
                dp[(size_t)(c + 0) * p.ls] = v0; dp[(size_t)(c + 1) * p.ls] = v1;
                dp[(size_t)(c + 2) * p.ls] = v2; dp[(size_t)(c + 3) * p.ls] = v3;
            }
            for (; c < nc; ++c) dp[(size_t)c * p.ls] = LDSTREAM(tp + (long long)c * cstride);
        }
        block_fft<true>(A, Bf, nc, p, tw_s);
#pragma unroll
        for (int i = 0; i < kMaxOwn; ++i) {
            const int d = threadIdx.x + i * blockDim.x;  // storage column
            if (d < W) {
                int n = d - rw;
                if (n < 0) n += W;
                float2 a = acc[i];
                const float2* sp = Srow + (long long)c0 * cstride + d;
                const float2* ap = A + n;
                int c = 0;
                for (; c + 4 <= nc; c += 4) {
                    const float2 s0 = LDSTREAM(sp + (long long)(c + 0) * cstride), s1 = LDSTREAM(sp + (long long)(c + 1) * cstride);
                    const float2 s2 = LDSTREAM(sp + (long long)(c + 2) * cstride), s3 = LDSTREAM(sp + (long long)(c + 3) * cstride);
                    const float2 v0 = ap[(size_t)(c + 0) * p.ls], v1 = ap[(size_t)(c + 1) * p.ls];
                    const float2 v2 = ap[(size_t)(c + 2) * p.ls], v3 = ap[(size_t)(c + 3) * p.ls];
                    // rim_utils.py:61-62: re += v_re*s_re + v_im*s_im ; im += v_im*s_re - v_re*s_im  (coil order kept)
                    a.x += v0.x * s0.x + v0.y * s0.y; a.y += v0.y * s0.x - v0.x * s0.y;
                    a.x += v1.x * s1.x + v1.y * s1.y; a.y += v1.y * s1.x - v1.x * s1.y;
                    a.x += v2.x * s2.x + v2.y * s2.y; a.y += v2.y * s2.x - v2.x * s2.y;
                    a.x += v3.x * s3.x + v3.y * s3.y; a.y += v3.y * s3.x - v3.x * s3.y;
                }
                for (; c < nc; ++c) {
                    const float2 s0 = LDSTREAM(sp + (long long)c * cstride);
                    const float2 v0 = ap[(size_t)c * p.ls];
                    a.x += v0.x * s0.x + v0.y * s0.y; a.y += v0.y * s0.x - v0.x * s0.y;
                }
                acc[i] = a;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < kMaxOwn; ++i) {
        const int d = threadIdx.x + i * blockDim.x;
        if (d < W) {
            if (OUT_MODE == 0) {
                ((float2*)out)[((long long)b * H + h) * W + d] = cscale(acc[i], scale);
            } else if (OUT_MODE == 2) {
                float2 e = eta[((long long)b * H + h) * W + d];
                reinterpret_cast<float4*>(out)[((long long)b * H + h) * W + d] =
                    make_float4(e.x, e.y, acc[i].x * scale, acc[i].y * scale);
            } else {
                const long long HW = (long long)H * W;
                float2 e = eta[((long long)b * H + h) * W + d];
                float* o = out + (long long)b * 4 * HW + (long long)h * W + d;
                o[0] = e.x;
                o[HW] = e.y;
                o[2 * HW] = acc[i].x * scale;
                o[3 * HW] = acc[i].y * scale;
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------------
// Hybrid-space form of the RIM gradient for 1-D (column) masks.
//
// With a mask that does not depend on k_h, the H-direction transforms of fft2 and ifft2 (rim_utils.py:50-58) cancel:
//     ifft2( M(k_w) * (fft2(x) - y) ) = bs*H * V_W[ M * (fs * U_W x - yh) ],      yh = (1/H) * V_H y
// (U/V unnormalised centred forward/inverse DFTs along one axis, fs/bs the normalisation factors of the 2-D pair).
// yh depends only on the measured k-space, which is constant over the whole unrolled network: it is prepared once
// per slice batch (mrb_dc_hybrid_prepare, sampled columns only, packed) and every gradient evaluation becomes ONE
// kernel of row transforms: no column pass, no T1/T2 intermediates, and S is read from HBM once instead of twice.
// ---------------------------------------------------------------------------------------------------------------

// yh[b,c,h,j] = tmp[b,c,h,(cols[j] + rw) % W]: pack the sampled columns of the H-transformed k-space
__global__ void compact_hybrid_kernel(const float2* __restrict__ tmp, float2* __restrict__ yh, MaskDesc mask, int C, int H,
                                      int W, int rw, int rows_per_cta) {
    extern __shared__ float2 smem[];
    unsigned short* cols_s = reinterpret_cast<unsigned short*>(smem);
    __shared__ int scan_scratch[33];
    const int c = blockIdx.y, b = blockIdx.z;
    const int ns = build_active_cols(mask, b, W, rw, true, cols_s, scan_scratch);
    const long long plane = ((long long)b * C + c) * H * W;
    const int h0 = blockIdx.x * rows_per_cta, h1 = min(H, h0 + rows_per_cta);
    for (int h = h0; h < h1; ++h)
        for (int j = threadIdx.x; j < ns; j += blockDim.x)
            yh[plane + (long long)h * W + j] = LDSTREAM(tmp + plane + (long long)h * W + rot_add((int)cols_s[j], rw, W));
}

#ifndef MRB_ROWDC_REGS
#define MRB_ROWDC_REGS 64  // 3 CTAs of 320 threads per SM
#endif
// One CTA per (b, image row h), all coils in shared memory (chunks of cc):
//   p = S*eta -> forward FFT along W -> r = m*(fs*P - yh) on the sampled columns, 0 elsewhere -> inverse FFT along W
//   -> acc += conj(S) * .   Thread t owns storage column t in both the load and the reduce step, so its S values stay
//   in registers (KEEP_S: blockDim >= W and cc <= 8); out modes as in rowifft_reduce_kernel.
template <int OUT_MODE, bool KEEP_S>
__global__ void __maxnreg__(MRB_ROWDC_REGS) row_dc_kernel(const float2* __restrict__ eta, const float2* __restrict__ S, const float2* __restrict__ yh,
                              float* __restrict__ out, int C, int H, int W, int cc, FftPlan p, int rw, float fscale,
                              float oscale, MaskDesc mask) {
    extern __shared__ float2 smem[];
    float2* A = smem;
    float2* Bf = A + (size_t)cc * p.ls;
    float2* tw_s = Bf + (size_t)cc * p.ls;
    unsigned short* cols_s = reinterpret_cast<unsigned short*>(tw_s + p.n);
    unsigned short* pos_s = cols_s + W;  // un-centred k_w -> index in the packed column list, 0xffff = not sampled
    __shared__ int scan_scratch[33];
    load_twiddles(tw_s, p);
    const int h = blockIdx.x, b = blockIdx.y;
    for (int k = threadIdx.x; k < W; k += blockDim.x) pos_s[k] = 0xffff;
    const int ns = build_active_cols(mask, b, W, rw, true, cols_s, scan_scratch);  // ends with a barrier
    for (int j = threadIdx.x; j < ns; j += blockDim.x) pos_s[cols_s[j]] = (unsigned short)j;
    const long long cstride = (long long)H * W;
    const long long rowoff = ((long long)b * C * H + h) * W;
    const float2* Srow = S + rowoff;
    const float2* Yrow = yh + rowoff;
    const float2* erow = eta + ((long long)b * H + h) * W;
    float2* St = fft_start_buf(p, A, Bf);
    constexpr int kMaxOwn = 4, kKeep = 8;
    float2 acc[kMaxOwn];
#pragma unroll
    for (int i = 0; i < kMaxOwn; ++i) acc[i] = make_float2(0.f, 0.f);
    for (int c0 = 0; c0 < C; c0 += cc) {
        const int nc = min(cc, C - c0);
        __syncthreads();  // pos_s ready (first chunk) / previous chunk's reduce done with the buffers
        float2 sreg[kKeep];
        // ---- expand: storage column d -> FFT input index j = d - rw ----
        for (int d = threadIdx.x; d < W; d += blockDim.x) {
            int j = d - rw;
            if (j < 0) j += W;
            const float2 e = __ldg(&erow[d]);
            const float2* sp = Srow + (long long)c0 * cstride + d;
            float2* dp = St + j;
            if (KEEP_S) {
#pragma unroll
                for (int c = 0; c < kKeep; ++c)
                    if (c < nc) sreg[c] = LDSTREAM(sp + (long long)c * cstride);
#pragma unroll
                for (int c = 0; c < kKeep; ++c)
                    if (c < nc)  // rim_utils.py:47-48
                        dp[(size_t)c * p.ls] = make_float2(e.x * sreg[c].x - e.y * sreg[c].y, e.x * sreg[c].y + e.y * sreg[c].x);
            } else {
                for (int c = 0; c < nc; ++c) {
                    const float2 s0 = LDSTREAM(sp + (long long)c * cstride);
                    dp[(size_t)c * p.ls] = make_float2(e.x * s0.x - e.y * s0.y, e.x * s0.y + e.y * s0.x);
                }
            }
        }
        block_fft<false>(A, Bf, nc, p, tw_s);
        // ---- k-space residual (in place when St == A; every (c,k) is read and written by the same thread) ----
        for (int k = threadIdx.x; k < W; k += blockDim.x) {
            const int j = pos_s[k];
            if (j == 0xffff) {
                for (int c = 0; c < nc; ++c) St[(size_t)c * p.ls + k] = make_float2(0.f, 0.f);
            } else {
                const float m = mask_value(mask, b, 0, rot_add(k, rw, W));
                const float2* yp = Yrow + (long long)c0 * cstride + j;
                for (int c = 0; c < nc; ++c) {
                    const float2 P = cscale(A[(size_t)c * p.ls + k], fscale);
                    const float2 yv = LDSTREAM(yp + (long long)c * cstride);
                    St[(size_t)c * p.ls + k] = make_float2(m * (P.x - yv.x), m * (P.y - yv.y));  // rim_utils.py:54
                }
            }
        }
        block_fft<true>(A, Bf, nc, p, tw_s);
        // ---- reduce: acc[d] += conj(S[c][d]) * A[c][d - rw]  (coil order kept, rim_utils.py:61-62) ----
#pragma unroll
        for (int i = 0; i < kMaxOwn; ++i) {
            const int d = threadIdx.x + i * blockDim.x;
            if (d < W) {
                int n = d - rw;
                if (n < 0) n += W;
                float2 a = acc[i];
                const float2* ap = A + n;
                if (KEEP_S) {
#pragma unroll
                    for (int c = 0; c < kKeep; ++c)
                        if (c < nc) {
                            const float2 v0 = ap[(size_t)c * p.ls], s0 = sreg[c];
                            a.x += v0.x * s0.x + v0.y * s0.y; a.y += v0.y * s0.x - v0.x * s0.y;
                        }
                } else {
                    const float2* sp = Srow + (long long)c0 * cstride + d;
                    for (int c = 0; c < nc; ++c) {
                        const float2 s0 = LDSTREAM(sp + (long long)c * cstride);
                        const float2 v0 = ap[(size_t)c * p.ls];
                        a.x += v0.x * s0.x + v0.y * s0.y; a.y += v0.y * s0.x - v0.x * s0.y;
                    }
                }
                acc[i] = a;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < kMaxOwn; ++i) {
        const int d = threadIdx.x + i * blockDim.x;
        if (d < W) {
            const float2 e = erow[d];
            if (OUT_MODE == 2) {
                reinterpret_cast<float4*>(out)[((long long)b * H + h) * W + d] =
                    make_float4(e.x, e.y, acc[i].x * oscale, acc[i].y * oscale);
            } else {
                const long long HW = (long long)H * W;
                float* o = out + (long long)b * 4 * HW + (long long)h * W + d;
                o[0] = e.x;
                o[HW] = e.y;
                o[2 * HW] = acc[i].x * oscale;
                o[3 * HW] = acc[i].y * oscale;
            }
        }
    }
}


// ---------------------------------------------------------------------------------------------------------------
// W = 320 fast path of the hybrid-space gradient (both fastMRI geometries have 320 columns): register-resident
// two-pass transforms, 320 = 16 x 20.
//
// Thread (c = tid / 20, t = tid % 20) of a 320-thread CTA (one image row, up to 16 coils):
//   pass 1 (t = n2):  loads S[c][20*n1 + t] * eta for n1 < 16 straight into registers, 16-point DFT over n1,
//                     twiddle w320^(t*k1), one shared-memory exchange (xch[c][k1][n2]);
//   pass 2 (t = k1 < 16): 20-point DFT over n2 -> X[k1 + 16*k2]; k-space residual against the (cp.async-prefetched)
//                     hybrid k-space row; inverse 20-point DFT over k2 of the SAME registers, twiddle, second exchange;
//   pass 3 (t = n2):  inverse 16-point DFT over k1 -> x[20*n1 + t], the ownership of pass 1, so conj(S) is still in
//                     registers; the coil sum goes through shared memory in coil order (rim_utils.py:61-62).
// Two exchanges per forward + inverse pair instead of six Stockham passes (3.5x fewer shared-memory wavefronts, all
// conflict free: k1 rows are 22 float2 apart, coils 356) and no per-stage index arithmetic.
// ---------------------------------------------------------------------------------------------------------------
namespace r320 {
constexpr int N = 320, N1 = 16, N2 = 20, XS = 22, CS = N1 * XS + 4, THREADS = 320, MAXC = 16, RS = N + 4;
#ifndef MRB_DC_PF_DIST
#define MRB_DC_PF_DIST 444
#endif
constexpr int PF_DIST = MRB_DC_PF_DIST;  // ~1.5 rounds of 2 CTAs x 148 SMs

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
                 : "memory");
}

__device__ __forceinline__ uint32_t bf16x2_rn(float e0, float e1) {  // (e0 -> low half, e1 -> high half), round to nearest even
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(e1), "f"(e0));
    return r;
}

inline size_t smem_bytes(int C) {
    return (size_t)MAXC * CS * sizeof(float2) + (size_t)C * RS * sizeof(float2) + 3 * (size_t)N * sizeof(float2) +
           (size_t)N * sizeof(float) + (size_t)N * sizeof(unsigned short) + 16;
}

template <int OUT_MODE>
__global__ void __launch_bounds__(THREADS, 2) row_dc320_kernel(const float2* __restrict__ eta, const float2* __restrict__ S,
                                                               const float2* __restrict__ yh, float* __restrict__ out, int C,
                                                               int H, const float2* __restrict__ tw, int rw, float fscale,
                                                               float oscale, MaskDesc mask) {
    extern __shared__ float2 smem[];
    float2* xch = smem;                              // [MAXC][CS] exchange buffer of the two transposes
    float2* yh_s = xch + MAXC * CS;                   // [C][ns2] packed hybrid k-space rows; later the coil-sum buffer [C][RS]
    float2* tw1_s = yh_s + (size_t)C * RS;            // [k1][t]  w320^(t*k1): pass-1 twiddles, lanes read consecutive t
    float2* tw2_s = tw1_s + N;                        // [n2][k1] w320^(n2*k1): pass-2 twiddles, lanes read consecutive k1
    float2* eta_s = tw2_s + N;                        // [N] the eta row (storage order)
    float* mval_s = reinterpret_cast<float*>(eta_s + N);                      // [N] mask value by un-centred k
    unsigned short* pos_s = reinterpret_cast<unsigned short*>(mval_s + N);    // [N] un-centred k -> packed index
    __shared__ int scan_s[THREADS / 32];
    __shared__ __align__(8) unsigned long long yh_bar;  // transaction barrier of the hybrid k-space bulk copies
    const int tid = threadIdx.x;
    const int h = blockIdx.x, b = blockIdx.y;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(&yh_bar)), "r"(C));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const int c = tid / N2, t = tid - c * N2;
    const bool active = c < C;
    const long long cstride = (long long)H * N;
    const long long rowoff = ((long long)b * C * H + h) * N;
    const float2* erow = eta + ((long long)b * H + h) * N;

    // Centring (rw = W/2) costs no index rotation here: a circular shift of the transform input by N/2 multiplies its
    // output by (-1)^k, and the same holds for the inverse, so the row is transformed in STORAGE order and only the
    // measured term changes sign on odd k:  (-1)^k m (fs (-1)^k X_s[k] - yh[k]) = m (fs X_s[k] - (-1)^k yh[k]).
    // k = k1 + 16*k2 has the parity of k1: one sign per thread.
    // ---- pass 1 loads first: their latency overlaps the table set-up ----
    float2 sreg[N1];
    if (active) {
        const float2* sp = S + rowoff + (long long)c * cstride + t;
#pragma unroll
        for (int n1 = 0; n1 < N1; ++n1) sreg[n1] = LDSTREAM(sp + N2 * n1);
    }
    {
        // L2 prefetch for the CTA that will run PF_DIST rows later (rows are scheduled in block-index order): its S row
        // (C x 2560 B = 20*C lines of 128 B) and the head of its hybrid k-space row then come from L2 instead of HBM.
        long long rid = (long long)b * H + h + PF_DIST;
        if (rid < (long long)gridDim.y * H) {
            const long long pb = rid / H, ph = rid - pb * H;
            const long long proff = (pb * C * H + ph) * N;
            if (tid < 20 * C) {
                const int pc = tid / 20, pl = tid - pc * 20;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(S + proff + (long long)pc * cstride + pl * 16));
                if (pl < 7) asm volatile("prefetch.global.L2 [%0];" ::"l"(yh + proff + (long long)pc * cstride + pl * 16));
            }
        }
    }
    tw1_s[tid] = __ldg(&tw[c * t]);                  // tid = 20*c + t  -> (k1 = c, t)
    tw2_s[tid] = __ldg(&tw[(tid >> 4) * (tid & 15)]);  // tid = 16*n2 + k1
    eta_s[tid] = __ldg(&erow[tid]);
    // Thread k owns un-centred k-space column k: its mask value, and (ballot scan) its slot in the packed row.
    const float mk = mask_value(mask, b, 0, rot_add(tid, rw, N));
    mval_s[tid] = mk;
    int ns;
    {
        const int lane = tid & 31, wid = tid >> 5;
        const unsigned bal = __ballot_sync(0xffffffffu, mk != 0.f);
        if (lane == 0) scan_s[wid] = __popc(bal);
        __syncthreads();
        int woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) {
            const int cnt = scan_s[w];
            woff += w < wid ? cnt : 0;
            tot += cnt;
        }
        ns = tot;
        // unsampled k: any valid slot (its mask value is 0, so the residual vanishes)
        pos_s[tid] = mk != 0.f ? (unsigned short)(woff + __popc(bal & ((1u << lane) - 1u))) : (unsigned short)0;
    }
    const int ns2 = max(2, (ns + 1) & ~1);
    // TMA staging of the packed hybrid k-space rows: one bulk copy per coil (ns2 x 8 bytes, a multiple of 16) issued by the
    // coil's first thread after its own arrive.expect_tx on a barrier of C arrivals (initialised before the scan's
    // __syncthreads); the flight time overlaps pass 1
    {
        const unsigned bar = (unsigned)__cvta_generic_to_shared(&yh_bar);
        if (active && t == 0) {
            const float2* ysrc = yh + rowoff + (long long)c * cstride;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((unsigned)(ns2 * 8)) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             (unsigned)__cvta_generic_to_shared(yh_s + (size_t)c * ns2)),
                         "l"(ysrc), "r"((unsigned)(ns2 * 8)), "r"(bar)
                         : "memory");
        }
    }
    float2* xc = xch + (size_t)c * CS;
    if (active) {
        cx v[N1];
#pragma unroll
        for (int n1 = 0; n1 < N1; ++n1) {
            const float2 e = eta_s[N2 * n1 + t], s0 = sreg[n1];
            v[n1] = pk(e.x * s0.x - e.y * s0.y, e.x * s0.y + e.y * s0.x);  // rim_utils.py:47-48
        }
        dft16<false>(v);
        xc[t] = upk(v[0]);
#pragma unroll
        for (int k1 = 1; k1 < N1; ++k1) {
            const float2 w = tw1_s[k1 * N2 + t];
            xc[k1 * XS + t] = mulw<false>(upk(v[k1]), w.x, w.y);
        }
    }
    {
        const unsigned bar = (unsigned)__cvta_generic_to_shared(&yh_bar);
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "YH_WAIT:\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n\t"
            "@p bra YH_DONE;\n\t"
            "bra YH_WAIT;\n\t"
            "YH_DONE:\n\t"
            "}\n" ::"r"(bar)
            : "memory");
    }
    __syncthreads();
    // ---- pass 2: forward 20-point DFT, residual, inverse 20-point DFT.  Only 16 lines per coil: the threads are re-dealt as
    // (coil = tid / 16, k1 = tid % 16) so that the 16*C busy lanes fill whole warps (7.5 instead of 10 at C = 15) ----
    const int c2 = tid >> 4, kk = tid & (N1 - 1);
    if (c2 < C) {
        cx v[N2];
        float4* row = reinterpret_cast<float4*>(xch + (size_t)c2 * CS + kk * XS);
#pragma unroll
        for (int i = 0; i < N2 / 2; ++i) {
            const float4 q = row[i];
            v[2 * i] = pk(q.x, q.y);
            v[2 * i + 1] = pk(q.z, q.w);
        }
        dft20<false>(v);
        const float2* yc = yh_s + (size_t)c2 * ns2;
        const float ysgn = (rw != 0 && (kk & 1)) ? -1.f : 1.f;
#pragma unroll
        for (int k2 = 0; k2 < N2; ++k2) {
            const int k = kk + N1 * k2;
            const float m = mval_s[k];  // 0 on unsampled columns: the residual vanishes there
            const float2 yv = yc[pos_s[k]], X = upk(v[k2]);
            v[k2] = pk(m * (X.x * fscale - ysgn * yv.x), m * (X.y * fscale - ysgn * yv.y));  // rim_utils.py:54
        }
        dft20<true>(v);
        float2 o[N2];
        o[0] = upk(v[0]);
#pragma unroll
        for (int n2 = 1; n2 < N2; ++n2) {
            const float2 w = tw2_s[n2 * N1 + kk];
            o[n2] = mulw<true>(upk(v[n2]), w.x, w.y);
        }
#pragma unroll
        for (int i = 0; i < N2 / 2; ++i) row[i] = make_float4(o[2 * i].x, o[2 * i].y, o[2 * i + 1].x, o[2 * i + 1].y);
    }
    __syncthreads();
    // ---- pass 3: inverse 16-point DFT over k1 (thread t = n2), conj(S), coil sum ----
    cx v[N1];
    if (active) {
#pragma unroll
        for (int k1 = 0; k1 < N1; ++k1) v[k1] = pk(xc[k1 * XS + t]);
        dft16<true>(v);
        // the coil-sum buffer aliases the hybrid k-space rows, which nobody reads after pass 2
        float2* rc = yh_s + (size_t)c * RS + t;
#pragma unroll
        for (int n1 = 0; n1 < N1; ++n1) {
            const float2 s0 = sreg[n1], x = upk(v[n1]);
            rc[N2 * n1] = make_float2(x.x * s0.x + x.y * s0.y, x.y * s0.x - x.x * s0.y);  // x * conj(S)
        }
    }
    __syncthreads();
    {
        float2 acc = make_float2(0.f, 0.f);
        for (int cc = 0; cc < C; ++cc) {
            const float2 r = yh_s[(size_t)cc * RS + tid];
            acc.x += r.x;
            acc.y += r.y;
        }
        const int d = tid;
        const float2 e = eta_s[d];
        if (OUT_MODE == 3) {
            // G8 (conv_tc2.cu): [eta.re, eta.im, g.re, g.im] as 4 bf16 hi + 4 bf16 lo = 16 bytes at padded position
            // (h + 2, d + 2) of a [B][H+4][W+4] grid behind 2 (W+4) + 2 guard positions; edge threads / edge rows also write
            // the replicate border (ReplicationPad2d(2) of the 5x5 conv)
            const float gx = acc.x * oscale, gy = acc.y * oscale;
            const uint32_t h01 = bf16x2_rn(e.x, e.y), h23 = bf16x2_rn(gx, gy);
            const uint32_t l01 = bf16x2_rn(e.x - __uint_as_float(h01 << 16), e.y - __uint_as_float(h01 & 0xffff0000u));
            const uint32_t l23 = bf16x2_rn(gx - __uint_as_float(h23 << 16), gy - __uint_as_float(h23 & 0xffff0000u));
            const uint4 v = make_uint4(h01, h23, l01, l23);
            constexpr int Wp = N + 4;
            const int Hp = H + 4;
            uint4* base = reinterpret_cast<uint4*>(out) + (2 * Wp + 2) + ((long long)b * Hp + h + 2) * Wp;
            const int r0 = h == 0 ? -2 : 0, r1 = h == H - 1 ? 2 : 0;
            for (int r = r0; r <= r1; ++r) {
                uint4* row = base + (long long)r * Wp;
                row[d + 2] = v;
                if (d == 0) row[0] = row[1] = v;
                if (d == N - 1) row[N + 2] = row[N + 3] = v;
            }
        } else if (OUT_MODE == 2) {
            reinterpret_cast<float4*>(out)[((long long)b * H + h) * N + d] = make_float4(e.x, e.y, acc.x * oscale, acc.y * oscale);
        } else {
            const long long HW = (long long)H * N;
            float* o = out + (long long)b * 4 * HW + (long long)h * N + d;
            o[0] = e.x;
            o[HW] = e.y;
            o[2 * HW] = acc.x * oscale;
            o[3 * HW] = acc.y * oscale;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// 320-point forms of the VarNet-side operators (vn_block.py:51-87,109-119): the same register-resident 16 x 20 transform as
// fft.cu's fft320_kernel (16 lines per CTA, one shared-memory transpose) with the surrounding arithmetic in its loads and
// stores.  Centring is the pair of thread-constant signs of that kernel, so every tensor stays in STORAGE order:
//   expand_row320:  T1[b,c,h,:]  = FFT_W(S[b,c,h,:] * img[b,h,:])            lines = the C <= 16 coils of one image row
//   col_softdc320:  out[b,c,:,w] = base - where(mask, pred - y, 0) dcw - fs FFT_H(T1[b,c,:,w])   lines = 16 columns
//   reduce_row320:  out[b,h,:]   = scale * sum_c conj(S[b,c,h,:]) IFFT_W(T2[b,c,h,:])            lines = the coils
// ---------------------------------------------------------------------------------------------------------------
constexpr int VLINES = CTA_LINES, VXS = CTA_XS;

inline size_t v320_smem(bool cols, bool reduce) {  // reduce: + the [16][N + 4] coil-sum / residual buffer
    return (size_t)(VLINES * (N1 * VXS + (cols ? 1 : 4)) + N + (reduce ? MAXC * (N + 4) : 0)) * sizeof(float2);
}

// K1 (VarNet expand, W = 320): grid (H, B)
__global__ void __launch_bounds__(THREADS, 3) expand_row320_kernel(const float2* __restrict__ img, const float2* __restrict__ S,
                                                                   float2* __restrict__ T1, int C, int H,
                                                                   const float2* __restrict__ tw, int rw) {
    extern __shared__ float2 smem[];
    float2* xch = smem;
    float2* tw1_s = xch + VLINES * (N1 * VXS + 4);
    const int h = blockIdx.x, b = blockIdx.y;
    const float2* irow = img + ((long long)b * H + h) * N;
    const long long cstride = (long long)H * N, rowoff = ((long long)b * C * H + h) * N;
    auto ld = [&](int c, int j) {
        const float2 e = __ldg(&irow[j]), s0 = LDSTREAM(S + rowoff + (long long)c * cstride + j);
        return make_float2(e.x * s0.x - e.y * s0.y, e.x * s0.y + e.y * s0.x);  // vn_block.py:66 complex_mul(x, sens)
    };
    auto st = [&](int c, int k, float2 v) { T1[rowoff + (long long)c * cstride + k] = v; };
    fft320_cta<false, false>(xch, tw1_s, tw, C, rw != 0, rw != 0, 1.f, ld, st);
}

// K2' (VarNet soft DC, H = 320): grid (W / 16 rounded up, C, B); the column transform of 16 adjacent k_w
__global__ void __launch_bounds__(THREADS, 3) col_softdc320_kernel(const float2* __restrict__ T1, const float2* __restrict__ base,
                                                                   const float2* __restrict__ pred, const float2* __restrict__ y,
                                                                   float2* __restrict__ out, MaskDesc mask, int C, int W,
                                                                   const float2* __restrict__ tw, int rh, float fscale,
                                                                   const float* __restrict__ dcw_p, int no_dc) {
    extern __shared__ float2 smem[];
    float2* xch = smem;
    float2* tw1_s = xch + VLINES * (N1 * VXS + 1);
    const int w0 = blockIdx.x * VLINES, c = blockIdx.y, b = blockIdx.z;
    const long long plane = ((long long)b * C + c) * N * W;
    const float dcw = no_dc ? 0.f : *dcw_p;
    auto ld = [&](int l, int j) { return T1[plane + (long long)j * W + w0 + l]; };
    auto st = [&](int l, int kh, float2 E) {
        const long long o = plane + (long long)kh * W + w0 + l;
        if (no_dc) {
            out[o] = E;
        } else {
            const float2 bv = base[o];
            float2 sd = make_float2(0.f, 0.f);
            if (mask_value(mask, b, kh, w0 + l) != 0.f) {  // vn_block.py:110 torch.where(mask.bool(), pred - ref, 0)
                const float2 pv = pred[o], yv = y[o];
                sd = make_float2(pv.x - yv.x, pv.y - yv.y);
            }
            out[o] = make_float2((bv.x - sd.x * dcw) - E.x, (bv.y - sd.y * dcw) - E.y);  // :110,117
        }
    };
    fft320_cta<false, true>(xch, tw1_s, tw, min(VLINES, W - w0), rh != 0, rh != 0, fscale, ld, st);
}

// K2' at H = 640 (brain geometry): 8 adjacent k_w columns per CTA on the 640-point column transform (fft640_cols_cta);
// grid (W / 8 rounded up, C, B)
__global__ void __launch_bounds__(THREADS, 2) col_softdc640_kernel(const float2* __restrict__ T1, const float2* __restrict__ base,
                                                                   const float2* __restrict__ pred, const float2* __restrict__ y,
                                                                   float2* __restrict__ out, MaskDesc mask, int C, int W,
                                                                   const float2* __restrict__ tw320,
                                                                   const float2* __restrict__ tw640, int rh, float fscale,
                                                                   const float* __restrict__ dcw_p, int no_dc) {
    extern __shared__ float2 smem[];
    float2* xch = smem;
    float2* tw1_s = xch + VLINES * (N1 * VXS + 1);
    float2* buf = tw1_s + N;
    const int w0 = blockIdx.x * 8, c = blockIdx.y, b = blockIdx.z;
    const long long plane = ((long long)b * C + c) * (2 * N) * W;
    const float dcw = no_dc ? 0.f : *dcw_p;
    auto ld = [&](int cl, int j) { return T1[plane + (long long)j * W + w0 + cl]; };
    auto st = [&](int cl, int kh, float2 E) {
        const long long o = plane + (long long)kh * W + w0 + cl;
        if (no_dc) {
            out[o] = E;
        } else {
            const float2 bv = base[o];
            float2 sd = make_float2(0.f, 0.f);
            if (mask_value(mask, b, kh, w0 + cl) != 0.f) {
                const float2 pv = pred[o], yv = y[o];
                sd = make_float2(pv.x - yv.x, pv.y - yv.y);
            }
            out[o] = make_float2((bv.x - sd.x * dcw) - E.x, (bv.y - sd.y * dcw) - E.y);
        }
    };
    fft640_cols_cta<false>(xch, tw1_s, buf, tw320, tw640, min(8, W - w0), rh != 0, rh != 0, fscale, ld, st);
}

// K3 (W = 320): grid (H, B).  OUT_MODE 0 (VarNet reduce): out [B, H, W] complex = acc * scale; 1 (RIM gradient): out
// [B, 4, H, W] = (eta_re, eta_im, acc * scale); 2: the same channels-last [B, H, W, 4]
template <int OUT_MODE>
__global__ void __launch_bounds__(THREADS, 2) reduce_row320_kernel(const float2* __restrict__ T2, const float2* __restrict__ S,
                                                                   const float2* __restrict__ eta, float* __restrict__ out,
                                                                   int C, int H, const float2* __restrict__ tw, int rw,
                                                                   float scale) {
    extern __shared__ float2 smem[];
    float2* xch = smem;
    float2* tw1_s = xch + VLINES * (N1 * VXS + 4);
    float2* red = tw1_s + N;  // [C][N + 4] conj(S) * IFFT_W(T2) per coil
    const int h = blockIdx.x, b = blockIdx.y;
    const long long cstride = (long long)H * N, rowoff = ((long long)b * C * H + h) * N;
    auto ld = [&](int c, int j) { return LDSTREAM(T2 + rowoff + (long long)c * cstride + j); };
    auto st = [&](int c, int n, float2 x) {
        const float2 s0 = LDSTREAM(S + rowoff + (long long)c * cstride + n);
        red[(size_t)c * (N + 4) + n] = make_float2(x.x * s0.x + x.y * s0.y, x.y * s0.x - x.x * s0.y);  // x * conj(S)
    };
    fft320_cta<true, false>(xch, tw1_s, tw, C, rw != 0, rw != 0, 1.f, ld, st);
    __syncthreads();
    float2 acc = make_float2(0.f, 0.f);
    for (int c = 0; c < C; ++c) {
        const float2 r = red[(size_t)c * (N + 4) + threadIdx.x];
        acc.x += r.x;
        acc.y += r.y;
    }
    const int d = threadIdx.x;
    if (OUT_MODE == 0) {
        reinterpret_cast<float2*>(out)[((long long)b * H + h) * N + d] = make_float2(acc.x * scale, acc.y * scale);
    } else {
        const float2 e = eta[((long long)b * H + h) * N + d];  // rim_utils.py:67: channels 0-1 are eta itself
        if (OUT_MODE == 2) {
            reinterpret_cast<float4*>(out)[((long long)b * H + h) * N + d] = make_float4(e.x, e.y, acc.x * scale, acc.y * scale);
        } else {
            const long long HW = (long long)H * N;
            float* o = out + (long long)b * 4 * HW + (long long)h * N + d;
            o[0] = e.x;
            o[HW] = e.y;
            o[2 * HW] = acc.x * scale;
            o[3 * HW] = acc.y * scale;
        }
    }
}

// K2 (RIM gradient, H = 320, any mask): per 16 adjacent columns of one (b, c) plane  P = fs FFT_H(T1),
// r = mask * (P - y) (rim_utils.py:54), T2 = IFFT_H(r); the residual crosses from the bin-owning threads of the first
// transform to the sample-owning threads of the second through shared memory.  grid (W / 16 rounded up, C, B)
__global__ void __launch_bounds__(THREADS, 2) col_dc320_kernel(const float2* __restrict__ T1, const float2* __restrict__ y,
                                                               float2* __restrict__ T2, MaskDesc mask, int C, int W,
                                                               const float2* __restrict__ tw, int rh, float fscale) {
    extern __shared__ float2 smem[];
    float2* xch = smem;
    float2* tw1_s = xch + VLINES * (N1 * VXS + 1);
    float2* res = tw1_s + N;  // [16][N + 1]
    const int w0 = blockIdx.x * VLINES, c = blockIdx.y, b = blockIdx.z;
    const long long plane = ((long long)b * C + c) * N * W;
    const int nv = min(VLINES, W - w0);
    auto ld = [&](int l, int j) { return LDSTREAM(T1 + plane + (long long)j * W + w0 + l); };
    auto st = [&](int l, int kh, float2 P) {
        const float m = mask_value(mask, b, kh, w0 + l);
        float2 r = make_float2(0.f, 0.f);
        if (m != 0.f) {  // unsampled entries contribute exactly 0 whatever y holds: skip the read
            const float2 yv = __ldg(&y[plane + (long long)kh * W + w0 + l]);
            r = make_float2(m * (P.x - yv.x), m * (P.y - yv.y));
        }
        res[(size_t)l * (N + 1) + kh] = r;
    };
    fft320_cta<false, true>(xch, tw1_s, tw, nv, rh != 0, rh != 0, fscale, ld, st);
    __syncthreads();
    auto ld2 = [&](int l, int j) { return res[(size_t)l * (N + 1) + j]; };
    auto st2 = [&](int l, int d, float2 v) { T2[plane + (long long)d * W + w0 + l] = v; };
    fft320_cta<true, true>(xch, tw1_s, tw, nv, rh != 0, rh != 0, 1.f, ld2, st2);
}
}  // namespace r320

struct DcGeom {
    FftPlan pw, ph;
    int cc;       // coils per smem chunk in the row kernels
    int ti;       // k_w strip width in the column kernels (power of two)
    int tsh;      // log2(ti)
    int threads_row;
    size_t smem_row, smem_col;
};

static int dc_geometry(int C, int H, int W, DcGeom* g) {
    int rc = get_fft_plan(W, &g->pw);
    if (rc) return rc;
    rc = get_fft_plan(H, &g->ph);
    if (rc) return rc;
    const size_t max_smem = device_max_smem_optin();
    // shared-memory budget per CTA: small enough for ~5 resident CTAs per SM (the kernels are latency bound:
    // more resident warps beat bigger tiles); MRB_DC_SMEM_KB overrides for experiments
    static int budget_kb = [] {
        const char* e = getenv("MRB_DC_SMEM_KB");
        int v = e ? atoi(e) : 44;
        return v < 8 ? 8 : v;
    }();
    const size_t row_budget = max_smem < (size_t)budget_kb * 1024 ? max_smem : (size_t)budget_kb * 1024;
    int cc = C;
    MRB_REQUIRE(W <= 65535 && H <= 65535, MRB_EUNSUPPORTED, "H and W must be <= 65535");
    while (cc > 1 && fft_smem_bytes(g->pw, cc) > row_budget) cc = (cc + 1) / 2;
    MRB_REQUIRE(fft_smem_bytes(g->pw, cc) <= max_smem, MRB_EUNSUPPORTED, "W=%d does not fit shared memory", W);
    g->cc = cc;
    g->smem_row = fft_smem_bytes(g->pw, cc) + (size_t)W * sizeof(unsigned short) + 16;
    int ti = 16;
    while (ti > 1 && fft_smem_bytes(g->ph, ti) > row_budget) ti /= 2;
    MRB_REQUIRE(fft_smem_bytes(g->ph, ti) <= max_smem, MRB_EUNSUPPORTED, "H=%d does not fit shared memory", H);
    g->ti = ti;
    g->tsh = 0;
    while ((1 << g->tsh) < ti) ++g->tsh;
    g->smem_col = fft_smem_bytes(g->ph, ti) + (size_t)W * sizeof(unsigned short) + 16;
    // row kernels: one thread per column when W <= 1024, else up to 4 columns per thread
    int tr = ((W + 31) / 32) * 32;
    if (tr > 1024) tr = 1024;
    if (tr < 128) tr = 128;
    MRB_REQUIRE(tr * 4 >= W, MRB_EUNSUPPORTED, "W=%d too large for the row-reduce kernel", W);
    g->threads_row = tr;
    return MRB_OK;
}

static int make_mask(const void* mask, int dtype, int mask_b, int mask_h, int B, int H, int W, MaskDesc* m) {
    MRB_REQUIRE(mask != nullptr, MRB_EINVAL, "mask is null");
    MRB_REQUIRE(dtype == MRB_MASK_U8 || dtype == MRB_MASK_F32, MRB_EINVAL, "bad mask dtype %d", dtype);
    MRB_REQUIRE(mask_b == 1 || mask_b == B, MRB_EINVAL, "mask batch %d must be 1 or %d", mask_b, B);
    MRB_REQUIRE(mask_h == 1 || mask_h == H, MRB_EINVAL, "mask height %d must be 1 or %d", mask_h, H);
    m->ptr = mask;
    m->dtype = dtype;
    m->hstride = mask_h == 1 ? 0 : W;
    m->bstride = mask_b == 1 ? 0 : mask_h * W;
    return MRB_OK;
}

static int check_dims(int B, int C, int H, int W, int norm, const char* who) {
    MRB_REQUIRE(B >= 1 && C >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "%s: bad shape B=%d C=%d H=%d W=%d", who, B, C, H, W);
    MRB_REQUIRE(B <= 65535 && C <= 65535, MRB_EUNSUPPORTED, "%s: B and C must be <= 65535", who);
    MRB_REQUIRE(norm >= 0 && norm <= 2, MRB_EINVAL, "%s: bad norm %d", who, norm);
    return MRB_OK;
}

template <typename K>
static int set_smem(K kernel) {
    // static shared memory (scan scratch) counts against the same limit
    MRB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)device_max_smem_optin() - 1024));
    return MRB_OK;
}

}  // namespace mrb

using namespace mrb;

extern "C" size_t mrb_dc_workspace_bytes(int B, int C, int H, int W) {
    return (size_t)2 * (size_t)B * C * H * W * sizeof(float2);
}

extern "C" int mrb_dc_rim_grad(const void* eta, const void* y, const void* S, const void* mask, int mask_dtype,
                               int mask_b, int mask_h, float inv_sigma2, void* out, int out_nhwc, int B, int C, int H,
                               int W, int centered, int norm, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_dims(B, C, H, W, norm, "mrb_dc_rim_grad");
    if (rc) return rc;
    MRB_REQUIRE(eta && y && S && out && ws, MRB_EINVAL, "mrb_dc_rim_grad: null pointer");
    MRB_REQUIRE(ws_bytes >= mrb_dc_workspace_bytes(B, C, H, W), MRB_EINVAL, "mrb_dc_rim_grad: workspace too small");
    MaskDesc m;
    rc = make_mask(mask, mask_dtype, mask_b, mask_h, B, H, W, &m);
    if (rc) return rc;
    DcGeom g;
    rc = dc_geometry(C, H, W, &g);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    float2* T1 = (float2*)ws;
    float2* T2 = T1 + (size_t)B * C * H * W;
    const int rh = centered ? H / 2 : 0, rw = centered ? W / 2 : 0;
    const double npts = (double)H * W;
    const float fs = norm_scale(norm, 0, npts), bs = norm_scale(norm, 1, npts);
    if ((rc = set_smem(expand_rowfft_kernel<true>))) return rc;
    if ((rc = set_smem(col_dc_kernel))) return rc;
    if ((rc = set_smem(rowifft_reduce_kernel<1, true>))) return rc;
    if ((rc = set_smem(rowifft_reduce_kernel<2, true>))) return rc;
    const int prune = (mask_h == 1) ? 1 : 0;  // 1-D masks: only sampled k_w columns are transformed along H
    if (!prune && W == r320::N && H == r320::N && C <= r320::MAXC && !getenv("MRIDC_B200_DC_STOCKHAM")) {
        // 2-D masks at 320 x 320: the three passes on the register-resident 320-point transform, every tensor in storage order
        const size_t sm_r = r320::v320_smem(false, false), sm_c = r320::v320_smem(true, true), sm_o = r320::v320_smem(false, true);
        MRB_CUDA(cudaFuncSetAttribute(r320::expand_row320_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_r));
        MRB_CUDA(cudaFuncSetAttribute(r320::col_dc320_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_c));
        r320::expand_row320_kernel<<<dim3(H, B), r320::THREADS, sm_r, st>>>((const float2*)eta, (const float2*)S, T1, C, H,
                                                                            g.pw.tw, rw);
        MRB_LAUNCHED();
        r320::col_dc320_kernel<<<dim3(ceil_div(W, r320::VLINES), C, B), r320::THREADS, sm_c, st>>>(
            T1, (const float2*)y, T2, m, C, W, g.ph.tw, rh, fs);
        MRB_LAUNCHED();
        if (out_nhwc) {
            MRB_CUDA(cudaFuncSetAttribute(r320::reduce_row320_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_o));
            r320::reduce_row320_kernel<2><<<dim3(H, B), r320::THREADS, sm_o, st>>>(T2, (const float2*)S, (const float2*)eta,
                                                                                   (float*)out, C, H, g.pw.tw, rw, bs * inv_sigma2);
        } else {
            MRB_CUDA(cudaFuncSetAttribute(r320::reduce_row320_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_o));
            r320::reduce_row320_kernel<1><<<dim3(H, B), r320::THREADS, sm_o, st>>>(T2, (const float2*)S, (const float2*)eta,
                                                                                   (float*)out, C, H, g.pw.tw, rw, bs * inv_sigma2);
        }
        MRB_LAUNCHED();
        return MRB_OK;
    }
    expand_rowfft_kernel<true><<<dim3(H, B), g.threads_row, g.smem_row, st>>>((const float2*)eta, (const float2*)S, T1,
                                                                              C, H, W, g.cc, g.pw, rw, m, prune);
    MRB_LAUNCHED();
    col_dc_kernel<<<dim3(ceil_div(W, g.ti), C, B), 256, g.smem_col, st>>>(T1, (const float2*)y, T2, m, C, H, W, g.tsh,
                                                                          g.ph, rh, rw, fs, prune);
    MRB_LAUNCHED();
    if (out_nhwc)
        rowifft_reduce_kernel<2, true><<<dim3(H, B), g.threads_row, g.smem_row, st>>>(
            T2, (const float2*)S, (const float2*)eta, (float*)out, C, H, W, g.cc, g.pw, 0, rw, bs * inv_sigma2, m, prune);
    else
        rowifft_reduce_kernel<1, true><<<dim3(H, B), g.threads_row, g.smem_row, st>>>(
            T2, (const float2*)S, (const float2*)eta, (float*)out, C, H, W, g.cc, g.pw, 0, rw, bs * inv_sigma2, m, prune);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_dc_hybrid_prepare(const void* y, const void* mask, int mask_dtype, int mask_b, void* yh, int B, int C,
                                     int H, int W, int centered, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_dims(B, C, H, W, 0, "mrb_dc_hybrid_prepare");
    if (rc) return rc;
    MRB_REQUIRE(y && yh && ws, MRB_EINVAL, "mrb_dc_hybrid_prepare: null pointer");
    MRB_REQUIRE(ws_bytes >= mrb_dc_workspace_bytes(B, C, H, W) / 2, MRB_EINVAL, "mrb_dc_hybrid_prepare: workspace too small");
    MRB_REQUIRE(W <= 65535, MRB_EUNSUPPORTED, "mrb_dc_hybrid_prepare: W must be <= 65535");
    MaskDesc m;
    rc = make_mask(mask, mask_dtype, mask_b, 1, B, H, W, &m);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int rh = centered ? H / 2 : 0, rw = centered ? W / 2 : 0;
    // (1/H) * centred inverse DFT along H of the whole k-space (once per slice batch), then pack the sampled columns
    rc = fft1d_launch((const float2*)y, (float2*)ws, (long long)B * C, H, W, 1, rh, rh, 1.0f / (float)H, st);
    if (rc) return rc;
    const int rows_per_cta = 16;
    compact_hybrid_kernel<<<dim3(ceil_div(H, rows_per_cta), C, B), 256, (size_t)W * sizeof(unsigned short) + 16, st>>>(
        (const float2*)ws, (float2*)yh, m, C, H, W, rw, rows_per_cta);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_dc_rim_grad_hybrid(const void* eta, const void* yh, const void* S, const void* mask, int mask_dtype,
                                      int mask_b, float inv_sigma2, void* out, int out_nhwc, int B, int C, int H, int W,
                                      int centered, int norm, void* stream) {
    int rc = check_dims(B, C, H, W, norm, "mrb_dc_rim_grad_hybrid");
    if (rc) return rc;
    MRB_REQUIRE(eta && yh && S && out, MRB_EINVAL, "mrb_dc_rim_grad_hybrid: null pointer");
    MaskDesc m;
    rc = make_mask(mask, mask_dtype, mask_b, 1, B, H, W, &m);
    if (rc) return rc;
    DcGeom g;
    rc = dc_geometry(C, H, W, &g);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int rw = centered ? W / 2 : 0;
    const double npts = (double)H * W;
    const float fs = norm_scale(norm, 0, npts);
    const float os = norm_scale(norm, 1, npts) * (float)H * inv_sigma2;
    const size_t smem = g.smem_row + (size_t)W * sizeof(unsigned short);
    if (W == r320::N && C <= r320::MAXC && !getenv("MRIDC_B200_DC_STOCKHAM")) {
        // register-resident two-pass row transforms (both fastMRI geometries have 320 columns)
        const size_t sm = r320::smem_bytes(C);
        if (out_nhwc == 2) {
            if ((rc = set_smem(r320::row_dc320_kernel<3>))) return rc;
            r320::row_dc320_kernel<3><<<dim3(H, B), r320::THREADS, sm, st>>>((const float2*)eta, (const float2*)S,
                                                                             (const float2*)yh, (float*)out, C, H, g.pw.tw, rw,
                                                                             fs, os, m);
        } else if (out_nhwc) {
            if ((rc = set_smem(r320::row_dc320_kernel<2>))) return rc;
            r320::row_dc320_kernel<2><<<dim3(H, B), r320::THREADS, sm, st>>>((const float2*)eta, (const float2*)S,
                                                                             (const float2*)yh, (float*)out, C, H, g.pw.tw, rw,
                                                                             fs, os, m);
        } else {
            if ((rc = set_smem(r320::row_dc320_kernel<1>))) return rc;
            r320::row_dc320_kernel<1><<<dim3(H, B), r320::THREADS, sm, st>>>((const float2*)eta, (const float2*)S,
                                                                             (const float2*)yh, (float*)out, C, H, g.pw.tw, rw,
                                                                             fs, os, m);
        }
        MRB_LAUNCHED();
        return MRB_OK;
    }
    MRB_REQUIRE(out_nhwc != 2, MRB_EUNSUPPORTED, "mrb_dc_rim_grad_hybrid: the G8 output needs W == 320 and C <= 16");
    const bool keep = g.threads_row >= W && g.cc <= 8;
#define MRB_ROW_DC(MODE, KEEP)                                                                                        \
    do {                                                                                                              \
        if ((rc = set_smem(row_dc_kernel<MODE, KEEP>))) return rc;                                                    \
        row_dc_kernel<MODE, KEEP><<<dim3(H, B), g.threads_row, smem, st>>>((const float2*)eta, (const float2*)S,      \
                                                                           (const float2*)yh, (float*)out, C, H, W,    \
                                                                           g.cc, g.pw, rw, fs, os, m);                 \
    } while (0)
    if (out_nhwc) {
        if (keep) MRB_ROW_DC(2, true); else MRB_ROW_DC(2, false);
    } else {
        if (keep) MRB_ROW_DC(1, true); else MRB_ROW_DC(1, false);
    }
#undef MRB_ROW_DC
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_sens_reduce(const void* x, const void* S, void* out, int B, int C, int H, int W, int centered,
                               int norm, void* ws, size_t ws_bytes, void* stream) {
    int rc = check_dims(B, C, H, W, norm, "mrb_sens_reduce");
    if (rc) return rc;
    MRB_REQUIRE(x && S && out && ws, MRB_EINVAL, "mrb_sens_reduce: null pointer");
    MRB_REQUIRE(ws_bytes >= mrb_dc_workspace_bytes(B, C, H, W) / 2, MRB_EINVAL, "mrb_sens_reduce: workspace too small");
    DcGeom g;
    rc = dc_geometry(C, H, W, &g);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    float2* T2 = (float2*)ws;
    const int rh = centered ? H / 2 : 0, rw = centered ? W / 2 : 0;
    const float bs = norm_scale(norm, 1, (double)H * W);
    // inverse FFT along H (strided lines), rotations applied on both sides; W axis untouched (still centred)
    rc = fft1d_launch((const float2*)x, T2, (long long)B * C, H, W, 1, rh, rh, 1.0f, st);
    if (rc) return rc;
    if (W == r320::N && C <= r320::MAXC && !getenv("MRIDC_B200_DC_STOCKHAM")) {
        // register-resident row transform + conj(S) + coil sum (both fastMRI geometries have 320 columns)
        const size_t sm = r320::v320_smem(false, true);
        MRB_CUDA(cudaFuncSetAttribute(r320::reduce_row320_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        r320::reduce_row320_kernel<0><<<dim3(H, B), r320::THREADS, sm, st>>>(T2, (const float2*)S, nullptr, (float*)out, C, H,
                                                                             g.pw.tw, rw, bs);
        MRB_LAUNCHED();
        return MRB_OK;
    }
    if ((rc = set_smem(rowifft_reduce_kernel<0, false>))) return rc;
    MaskDesc nomask;
    memset(&nomask, 0, sizeof(nomask));
    rowifft_reduce_kernel<0, false><<<dim3(H, B), g.threads_row, g.smem_row, st>>>(
        T2, (const float2*)S, nullptr, (float*)out, C, H, W, g.cc, g.pw, rw, rw, bs, nomask, 0);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_sens_expand_softdc(const void* img, const void* S, const void* base, const void* pred,
                                      const void* y,
                                      const void* mask, int mask_dtype, int mask_b, int mask_h,
                                      const void* dc_weight, int no_dc, void* out, int B, int C, int H, int W, int centered, int norm,
                                      void* ws, size_t ws_bytes, void* stream) {
    int rc = check_dims(B, C, H, W, norm, "mrb_sens_expand_softdc");
    if (rc) return rc;
    MRB_REQUIRE(img && S && out && ws, MRB_EINVAL, "mrb_sens_expand_softdc: null pointer");
    MRB_REQUIRE(ws_bytes >= mrb_dc_workspace_bytes(B, C, H, W) / 2, MRB_EINVAL,
                "mrb_sens_expand_softdc: workspace too small");
    MaskDesc m;
    memset(&m, 0, sizeof(m));
    if (!no_dc) {
        MRB_REQUIRE(base && pred && y && dc_weight, MRB_EINVAL,
                    "mrb_sens_expand_softdc: base/pred/y/dc_weight required unless no_dc");
        rc = make_mask(mask, mask_dtype, mask_b, mask_h, B, H, W, &m);
        if (rc) return rc;
    }
    DcGeom g;
    rc = dc_geometry(C, H, W, &g);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    float2* T1 = (float2*)ws;
    const int rh = centered ? H / 2 : 0, rw = centered ? W / 2 : 0;
    const float fs = norm_scale(norm, 0, (double)H * W);
    const bool fast = !getenv("MRIDC_B200_DC_STOCKHAM");
    // T1's k_w axis: storage (centred) order after the 320-point row kernel, un-centred after the Stockham one
    const bool row320 = fast && W == r320::N && C <= r320::MAXC;
    if (row320) {
        const size_t sm = r320::v320_smem(false, false);
        MRB_CUDA(cudaFuncSetAttribute(r320::expand_row320_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        r320::expand_row320_kernel<<<dim3(H, B), r320::THREADS, sm, st>>>((const float2*)img, (const float2*)S, T1, C, H,
                                                                          g.pw.tw, rw);
    } else {
        if ((rc = set_smem(expand_rowfft_kernel<false>))) return rc;
        expand_rowfft_kernel<false><<<dim3(H, B), g.threads_row, g.smem_row, st>>>((const float2*)img, (const float2*)S, T1,
                                                                                   C, H, W, g.cc, g.pw, rw, m, 0);
    }
    MRB_LAUNCHED();
    if (fast && H == r320::N && row320) {
        const size_t sm = r320::v320_smem(true, false);
        MRB_CUDA(cudaFuncSetAttribute(r320::col_softdc320_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        r320::col_softdc320_kernel<<<dim3(ceil_div(W, r320::VLINES), C, B), r320::THREADS, sm, st>>>(
            T1, (const float2*)base, (const float2*)pred, (const float2*)y, (float2*)out, m, C, W, g.ph.tw, rh, fs,
            (const float*)dc_weight, no_dc);
    } else if (fast && H == 2 * r320::N && row320) {
        const size_t sm = r320::v320_smem(true, true);
        MRB_CUDA(cudaFuncSetAttribute(r320::col_softdc640_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        r320::col_softdc640_kernel<<<dim3(ceil_div(W, 8), C, B), r320::THREADS, sm, st>>>(
            T1, (const float2*)base, (const float2*)pred, (const float2*)y, (float2*)out, m, C, W, g.pw.tw, g.ph.tw, rh, fs,
            (const float*)dc_weight, no_dc);
    } else {
        if ((rc = set_smem(col_softdc_kernel))) return rc;
        // after the 320-point row kernel the columns already sit at their storage position: no W rotation left
        col_softdc_kernel<<<dim3(ceil_div(W, g.ti), C, B), 256, g.smem_col, st>>>(
            T1, (const float2*)base, (const float2*)pred, (const float2*)y, (float2*)out, m, C, H, W, g.tsh, g.ph, rh,
            row320 ? 0 : rw, fs, (const float*)dc_weight, no_dc);
    }
    MRB_LAUNCHED();
    return MRB_OK;
}
