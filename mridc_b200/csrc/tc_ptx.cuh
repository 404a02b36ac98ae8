// PTX wrappers shared by the tcgen05 / TMEM kernels (conv_tc.cu: the BH k x k conv; conv_tc2.cu: the other BH kernels).
#pragma once
#include "common.cuh"

namespace mrb {
namespace tc {

// ---- PTX wrappers ----------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// polling wait with back-off: waiting warps must not steal issue slots from the single MMA-issuing thread
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// long waits (loaders on a free stage, epilogue on a finished tile): try_wait with a suspend-time hint parks the warp in
// hardware until the phase completes (or the hint expires) instead of spinning through issue slots
__device__ __forceinline__ void mbar_wait_sleep(uint64_t* bar, uint32_t parity, unsigned ns) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity), "r"(ns)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// The MMA-issuing warps run warp-uniform code and elect one lane per tcgen05 instruction (elect.sync picks the same
// lane for the same full mask): with every operand provably uniform the MMAs issue straight from uniform registers.
// Issued from a single-lane branch instead, each MMA costs a 12-instruction R2UR "waterfall" (~45 cycles measured).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
        "}\n" ::"r"(smem_u32(bar))
        : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (bf16 operands), M = 128, K = 16
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T: A = 128 lanes x 8 columns (16 packed bf16) starting at a_tmem
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Stacked-B segment (2 MMAs per k-step instead of 3), A and B from shared memory: the packed weight chunk holds the hi
// rows immediately followed by the lo rows, so ONE descriptor with N = 2n multiplies a_hi by [b_hi ; b_lo] -> columns
// [d, d+n) = a_hi*b_hi and [d+n, d+2n) = a_hi*b_lo; the second MMA adds a_lo*b_hi (N = n) onto the cross-term columns
// [d+n, d+2n).  Four k-steps of K = 16 advance every SWIZZLE_128B K-major descriptor by 32 bytes.
__device__ __forceinline__ void umma_segment_ss_stacked(uint32_t d, uint32_t dsm, uint64_t a_hi, uint64_t a_lo, uint64_t dbh,
                                                        uint32_t idesc2n, uint32_t idescn, uint32_t acc0) {
    asm volatile(
        "{\n\t"
        ".reg .pred pa, pt, pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        ".reg .b64 ah1, ah2, ah3, al1, al2, al3, bh1, bh2, bh3;\n\t"
        "setp.ne.b32 pa, %7, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "add.u64 ah1, %2, 2;\n\t add.u64 ah2, %2, 4;\n\t add.u64 ah3, %2, 6;\n\t"
        "add.u64 al1, %3, 2;\n\t add.u64 al2, %3, 4;\n\t add.u64 al3, %3, 6;\n\t"
        "add.u64 bh1, %4, 2;\n\t add.u64 bh2, %4, 4;\n\t add.u64 bh3, %4, 6;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], %2, %4, %5, pa;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%1], %3, %4, %6, pt;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], ah1, bh1, %5, pt;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%1], al1, bh1, %6, pt;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], ah2, bh2, %5, pt;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%1], al2, bh2, %6, pt;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], ah3, bh3, %5, pt;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%1], al3, bh3, %6, pt;\n\t"
        "}\n" ::"r"(d),
        "r"(dsm), "l"(a_hi), "l"(a_lo), "l"(dbh), "r"(idesc2n), "r"(idescn), "r"(acc0)
        : "memory");
}
// lane-0 broadcast: tells the compiler that a value is warp-uniform (see umma_commit)
__device__ __forceinline__ uint32_t uni(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }
__device__ __forceinline__ uint64_t uni64(uint64_t v) { return ((uint64_t)uni((uint32_t)(v >> 32)) << 32) | uni((uint32_t)v); }
// four 8-column loads with a single wait (GRU epilogue: hh_n, r, z, ih_n blocks)
__device__ __forceinline__ void tmem_ld8x4(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, float* v0, float* v1, float* v2,
                                           float* v3) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%32];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%8,%9,%10,%11,%12,%13,%14,%15}, [%33];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%16,%17,%18,%19,%20,%21,%22,%23}, [%34];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%24,%25,%26,%27,%28,%29,%30,%31}, [%35];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3)
        : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        v0[i] = __uint_as_float(r[i]);
        v1[i] = __uint_as_float(r[8 + i]);
        v2[i] = __uint_as_float(r[16 + i]);
        v3[i] = __uint_as_float(r[24 + i]);
    }
}
__device__ __forceinline__ void tmem_ld_wait() {}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (rows of 128 bytes, 8-row groups 1024 bytes apart).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);  // start address
    d |= (uint64_t)1 << 16;                  // leading byte offset (ignored for swizzled K-major), 16 B
    d |= (uint64_t)(1024 >> 4) << 32;        // stride byte offset: 1024 B between 8-row groups
    d |= (uint64_t)1 << 46;                  // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                  // SWIZZLE_128B
    return d;
}
// The same matrix `rows` 128-byte rows further on, for a descriptor of a 1024-byte aligned SWIZZLE_128B tile: only the
// start address moves (rows * 128 B).  The tensor core takes the swizzle phase of a row from the address bits, as TMA
// writes it, so a start inside the 8-row pattern needs no matrix base offset (bits 49-51 stay 0).
__device__ __forceinline__ uint64_t desc_rows(uint64_t d, uint32_t rows) { return d + (uint64_t)(rows * (128 >> 4)); }
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
    // c_format F32 (1) @4, a_format BF16 (1) @7, b_format BF16 (1) @10, K-major A and B, N>>3 @17, M>>4 @24
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// fp32 pair -> packed bf16 hi pair + packed bf16 lo pair (element 0 in the low half, as tcgen05 reads packed A rows).
// hi = rn_bf16(x); lo = rn_bf16(x - hi): the subtraction is exact in fp32 and |x - hi - lo| <= 2^-18 |x|.
// Five instructions per pair (cvt.pack, shl, and, packed sub, cvt.pack): the loaders are instruction-issue bound.
__device__ __forceinline__ uint32_t pack_bf16x2(float e0, float e1) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(e1), "f"(e0));  // first source -> upper half
    return r;
}
__device__ __forceinline__ void sub2(float x0, float x1, float y0, float y1, float& r0, float& r1);
__device__ __forceinline__ void split_bf16x2(float e0, float e1, uint32_t& hi, uint32_t& lo) {
    hi = pack_bf16x2(e0, e1);
    float l0, l1;
    sub2(e0, e1, __uint_as_float(hi << 16), __uint_as_float(hi & 0xffff0000u), l0, l1);
    lo = pack_bf16x2(l0, l1);
}
__host__ __device__ inline uint16_t bf16_rn_bits(float v) {  // host/pack-kernel side rounding (RNE), NaN/Inf pass through
    uint32_t u;
    memcpy(&u, &v, 4);
    if ((u & 0x7f800000u) == 0x7f800000u) return (uint16_t)(u >> 16);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
__device__ __forceinline__ void sts128(uint32_t saddr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// 16-byte global -> shared async copy (src_bytes 0 = zero fill); bypass_l1: .cg (streamed once) vs .ca (re-read by taps)
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g, uint32_t src_bytes, bool bypass_l1) {
    if (bypass_l1)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(src_bytes) : "memory");
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(saddr), "l"(g), "r"(src_bytes) : "memory");
}
// explicit shared-space 128-bit load (a generic pointer would compile to LD.E)
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
    return v;
}
// gate non-linearities on the SFU: one ex2.approx and one rcp.approx each (~2 ulp, |error| ~1e-7 on outputs in
// [-1, 1]); the raw PTX forms skip the range fix-ups of __expf / __fdividef (saturation is already exact: ex2 -> 0 or
// +inf, rcp(inf) = 0)
__device__ __forceinline__ float ex2_approx(float v) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
__device__ __forceinline__ float rcp_approx(float v) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}
constexpr float kLog2e = 1.4426950408889634f;
// sigmoid(a + b) with bs = -log2(e) * b folded on the host side of the epilogue (bias table)
__device__ __forceinline__ float sigmoid_fused(float a, float bs) { return rcp_approx(1.f + ex2_approx(fmaf(a, -kLog2e, bs))); }
__device__ __forceinline__ float tanh_acc(float v) { return fmaf(-2.f, rcp_approx(1.f + ex2_approx(v * (2.f * kLog2e))), 1.f); }

// (x0, x1) - (y0, y1) as one packed fp32x2 instruction (same IEEE result as two scalar subtractions)
__device__ __forceinline__ void sub2(float x0, float x1, float y0, float y1, float& r0, float& r1) {
    unsigned long long x, y, r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(x0), "f"(x1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(y) : "f"(y0), "f"(y1));
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(x), "l"(y));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r0), "=f"(r1) : "l"(r));
}

// ---- packed fp32x2 arithmetic (sm_100: one issue slot per PAIR of IEEE-RN operations; results are bit-identical to the
// scalar instructions).  A pair lives in one 64-bit register.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float a, float b) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void up2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2p(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// two 64-bit pairs from 16 bytes of shared memory
__device__ __forceinline__ void lds128p(uint32_t saddr, f32x2& a, f32x2& b) {
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(saddr) : "memory");
}

// byte offset of 16-byte chunk c (0..7) of row r inside a [rows x 128 B] SWIZZLE_128B tile
__device__ __forceinline__ uint32_t swz(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }


// ---- helpers shared with the BH (split-bf16) activation format --------------------------------------------------
__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }          // element 2i of a bf16 pair
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }  // element 2i + 1
__device__ __forceinline__ uint4 lds128u(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128u(uint32_t saddr, uint4 v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// 2-D TMA box load global -> shared memory, completing the box's bytes on the mbarrier's transaction count; m = address
// of a CUtensorMap.  Box rows outside the tensor (negative coordinates too) are zero-filled.
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* m, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(m), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
// contiguous bulk copy global -> shared memory, completing the mbarrier's transaction count
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 2-D TMA box store shared memory -> global (bulk async group of the issuing thread); m = address of a CUtensorMap
__device__ __forceinline__ void tma_store_2d(const void* m, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(m), "r"(src), "r"(c0), "r"(c1)
                 : "memory");
}

// weight packer (conv_tc.cu): [rows x 128 B] SWIZZLE_128B chunks of 64 bf16 K elements, hi rows then lo rows
struct PackDesc {
    const float* w;       // conv: [Cout][Cin][k][k]; GRU: w_ih [3Ch][Cx] then w_hh via w2
    const float* w2;
    int mode;             // 0 conv taps (chunk = tap), 1 GRU (chunk 0 = hh, 1 = ih)
    int cout, cin, ksz;   // conv geometry
    int nhalf;            // output channels per split part
    int rows;             // rows per chunk
    int n_chunks;
    int n_split;
};
int pack_launch(const PackDesc& D, void* dst, cudaStream_t st);
}  // namespace tc
namespace tc2 {
// TMA descriptor of a BH tensor seen as [Q positions][128 bf16] with boxes of 64 columns x box_rows positions (conv_tc2.cu);
// the descriptor is written to *m, which must be a CUtensorMap
int make_bh_tmap(void* m, const void* base, long long Q, int box_rows);
}  // namespace tc2
namespace tc {

}  // namespace tc
}  // namespace mrb
