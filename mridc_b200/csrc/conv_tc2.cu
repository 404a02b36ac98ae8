// ConvGRU cell on split-bf16 activations: TMA -> shared memory -> tcgen05.mma (A and B from shared memory) -> TMEM ->
// gate epilogue, one persistent CTA per SM.  Second-generation engine of the RIM regulariser (the first one, conv_tc.cu,
// keeps A in tensor memory and converts fp32 activations in loader warps; it still runs the convolutions).
//
// Reference behaviour: ConvGRUCell with kernel_size 1 (rim/rnn_cells.py:93-127) inside RIMBlock's time loop
// (rim/rim_block.py:217-249).
//
// Activation format "BH" (shared by every kernel of the time step): channels-last, 64 channels per pixel stored as
// 64 bf16 "hi" values followed by 64 bf16 "lo" values (x ~= hi + lo, |x - hi - lo| <= 2^-18 |x|; 256 bytes per pixel,
// the same as fp32), every image surrounded by a replicate-padded border of PAD = 2 pixels:
//     [B][H + 4][W + 4][hi 64 | lo 64]
// * the producer's epilogue does the hi/lo split once, where the fp32 value sits in a register; consumers feed the
//   tensor core without touching the data: one 2-D TMA box per operand tile lands in the UMMA K-major SWIZZLE_128B layout;
// * the replicate border turns ConvNonlinear's ReplicationPad2d (conv_layers.py:72-76) into plain address offsets: spatial
//   kernels (3x3 dil 2, final 3x3) never clamp; producers of tensors that are read spatially write the border copies;
// * pointwise kernels (this one) run over all (H+4)(W+4) positions of the flat [Q][128] matrix (2.5 % extra rows) with
//   no position logic at all; what they leave at border positions is not a replicate copy, so a producer whose output is
//   read spatially is followed by mrb_bh_fix_border (edge pixels -> border, ~1 % of the tensor).
//
// Work item = 128 consecutive positions x all 64 hidden channels (N = 192 gate rows per MMA: 96 tensor-pipe cycles, so
// the issuing thread's ~50-cycle latency is hidden; the channel-split kernel of the first engine issued N = 96).
//   TMA lane      four 16 KB boxes per tile: h_hi, h_lo through a two-tile ring (held until the epilogue has taken its
//                 h_prev values), x_hi, x_lo through a one-tile ring (released by the MMAs); mbarrier transaction counts;
//   MMA lane      25 tcgen05.mma.kind::f16 per tile (a_hi*b_hi, a_hi*b_lo, a_lo*b_hi for h and x; the r and z gates of
//                 both parts accumulate in shared columns), two 256-column accumulator buffers: the gate epilogue of
//                 tile t overlaps the MMAs of tile t+1;
//   16 epilogue warps (4 per TMEM lane quadrant, 16 channels each): h_prev straight from the TMA-landed operand slots
//                 (no second global read), batched tcgen05.ld, gates on the SFU, hi/lo split into an output tile in the
//                 TMA box layout;
//   TMA store lane  the two box stores of each tile.  No global load or store
//                 instruction is executed by any warp: a first version that fetched h_prev with cp.async and stored with
//                 st.global (16 lines per instruction) was bound by L1 wavefronts, not by HBM.
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "tc_ptx.cuh"

namespace mrb {
namespace tc2 {
using namespace mrb::tc;

constexpr int PADB = 2;            // replicate border of the BH layout
constexpr int PX_BYTES = 256;      // 64 hi + 64 lo bf16
constexpr int TILE = 128;
constexpr int EPI_W = 16;          // epilogue warps
constexpr int THREADS2 = (EPI_W + 3) * 32;  // + TMA load lane, MMA issuer, TMA store lane
constexpr int NSLOT = 8;           // 16 KB boxes: h ring 4 (two tiles x (h_hi, h_lo)), x ring 2 (x_hi, x_lo), output tile 2
constexpr int SLOT_BYTES = TILE * 128;
constexpr int W_CHUNK = 192 * 128; // hi (or lo) rows of one weight chunk

// ---- TMA ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}
// A BH tensor as the 2-D matrix [Q positions][128 bf16]; box = 64 columns (the hi or the lo half of a pixel, 128 B) x
// box_rows positions, written to shared memory in the SWIZZLE_128B pattern the UMMA descriptors expect.  Positions
// outside [0, Q) are zero-filled.
int make_bh_tmap(void* mp, const void* base, long long Q, int box_rows) {
    CUtensorMap* m = reinterpret_cast<CUtensorMap*>(mp);
    EncodeTiledFn fn = encode_fn();
    MRB_REQUIRE(fn != nullptr, MRB_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
    cuuint64_t dims[2] = {128, (cuuint64_t)Q};
    cuuint64_t strides[1] = {PX_BYTES};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MRB_REQUIRE(r == CUDA_SUCCESS, MRB_ECUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return MRB_OK;
}
#ifdef MRB_TC_PROF
__device__ int g_skip_mma = 0;
#endif
// D[tmem] (+)= A[smem] * B[smem]^T issued by one elected lane of a converged warp
__device__ __forceinline__ void umma_ss(uint32_t d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
#ifdef MRB_TC_PROF
    if (g_skip_mma) return;
#endif
    asm volatile(
        "{\n\t"
        ".reg .pred p, pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

#ifdef MRB_TC_PROF
#define T2P(...) __VA_ARGS__
#define T2_DBG(P, f) (((P).debug & (f)) != 0)
#else
#define T2P(...)
#define T2_DBG(P, f) false
#endif

struct Gru2Params {
    const void* wpack;   // chunk 0 = W_hh rows [n ; r ; z], chunk 1 = W_ih rows [r ; z ; n]; each [hi 192 x 128 B | lo]
    const float* bias;   // b_ih [192] (r, z, n) or null
    long long Q;         // B * (H+4) * (W+4) positions
    int n_tiles;
#ifdef MRB_TC_PROF
    int debug;                 // 1 skip MMAs, 2 skip TMA loads, 4 skip gate math, 8 skip global stores, 16 skip h_prev fetch
    unsigned long long* prof;  // [grid][16]
#endif
};

__global__ void __launch_bounds__(THREADS2, 1)
gru2_kernel(const __grid_constant__ CUtensorMap tm_h, const __grid_constant__ CUtensorMap tm_x,
            const __grid_constant__ CUtensorMap tm_o, const Gru2Params P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* w_s = smem;                                  // [2 chunks][hi | lo][192 x 128 B]
    uint8_t* ring = w_s + 4 * W_CHUNK;                    // [4] h boxes: tile parity p -> h_hi = 2p, h_lo = 2p + 1
    uint8_t* xring = ring + 4 * SLOT_BYTES;               // [2] x_hi, x_lo of the tile whose MMAs run next
    uint8_t* out_s = xring + 2 * SLOT_BYTES;              // [2] output tile: hi box | lo box
    float* bias_s = (float*)(out_s + 2 * SLOT_BYTES);     // [192]: r, z pre-scaled by -log2(e)
    uint64_t* hfull = (uint64_t*)(bias_s + 192);          // [4]
    uint64_t* hempty = hfull + 4;                         // [4] MMA commit + one arrival per epilogue warp (h_prev readers)
    uint64_t* xfull = hempty + 4;                         // [2]
    uint64_t* xempty = xfull + 2;                         // [2] MMA commit
    uint64_t* acc_full = xempty + 2;                      // [2]
    uint64_t* acc_empty = acc_full + 2;                   // [2]
    uint64_t* out_ready = acc_empty + 2;                  // [1] every epilogue warp has written its part of the output tile
    uint64_t* out_free = out_ready + 1;                   // [2] the TMA stores of tile it have read the output tile: [it & 1]
    uint32_t* tmem_slot = (uint32_t*)(out_free + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) {
            mbar_init(&hfull[i], 1);
            mbar_init(&hempty[i], 1 + EPI_W);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&xfull[i], 1);
            mbar_init(&xempty[i], 1);
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], EPI_W);
        }
        mbar_init(out_ready, EPI_W);
        mbar_init(&out_free[0], 1);
        mbar_init(&out_free[1], 1);
        fence_barrier_init();
    }
    for (int i = threadIdx.x; i < 192; i += THREADS2) {
        const float b = P.bias ? P.bias[i] : 0.f;
        bias_s[i] = i < 128 ? -kLog2e * b : b;
    }
    if (warp == EPI_W + 1) tmem_alloc(tmem_slot, 512);
    {
        const float4* g = reinterpret_cast<const float4*>(P.wpack);
        const uint32_t s = smem_u32(w_s);
        for (int i = threadIdx.x; i < 4 * W_CHUNK / 16; i += THREADS2) {
            const float4 v = __ldg(g + i);
            sts128(s + 16u * (uint32_t)i, v);
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == EPI_W) {
        // ============================== TMA PRODUCER ==============================
        // order: h(0) | x(0), h(1) | x(1), h(2) | ...: the h boxes run one tile ahead (their slots are free as soon as the
        // epilogue of two tiles ago has taken its h_prev values), the x boxes follow the MMAs of the previous tile
        if (lane == 0) {
            T2P(long long t_pw = 0, t_p0 = clock64(), c0;)
            auto load = [&](uint64_t* fullb, uint64_t* emptyb, uint32_t parity, uint8_t* dst, const CUtensorMap* tm, int c0e, int q0) {
                T2P(c0 = clock64();)
                mbar_wait_sleep(emptyb, parity ^ 1, 64);
                T2P(t_pw += clock64() - c0;)
                if (T2_DBG(P, 2)) {
                    mbar_arrive(fullb);
                } else {
                    mbar_expect_tx(fullb, SLOT_BYTES);
                    tma_load_2d(smem_u32(dst), tm, c0e, q0, smem_u32(fullb));
                }
            };
            int it = 0;
            uint32_t xph = 0;
            const int first = blockIdx.x;
            if (first < P.n_tiles) {
                load(&hfull[0], &hempty[0], 0, ring, &tm_h, 0, first * TILE);
                load(&hfull[1], &hempty[1], 0, ring + SLOT_BYTES, &tm_h, 64, first * TILE);
            }
            for (int tile = first; tile < P.n_tiles; tile += gridDim.x, ++it) {
                load(&xfull[0], &xempty[0], xph, xring, &tm_x, 0, tile * TILE);
                load(&xfull[1], &xempty[1], xph, xring + SLOT_BYTES, &tm_x, 64, tile * TILE);
                xph ^= 1;
                const int nt = tile + gridDim.x;
                if (nt < P.n_tiles) {
                    const int p = (it + 1) & 1;
                    const uint32_t hph = (uint32_t)((it + 1) >> 1) & 1u;
                    load(&hfull[2 * p], &hempty[2 * p], hph, ring + (2 * p) * SLOT_BYTES, &tm_h, 0, nt * TILE);
                    load(&hfull[2 * p + 1], &hempty[2 * p + 1], hph, ring + (2 * p + 1) * SLOT_BYTES, &tm_h, 64, nt * TILE);
                }
            }
            T2P(if (P.prof) { P.prof[blockIdx.x * 16 + 0] = clock64() - t_p0; P.prof[blockIdx.x * 16 + 1] = t_pw; })
        }
    } else if (warp == EPI_W + 1) {
        // ============================== MMA ISSUER (whole warp, one elected lane per instruction) ==============================
        const uint32_t tmem_u = uni(tmem_base);
        const uint32_t ws = smem_u32(w_s), rs = smem_u32(ring);
        const uint64_t wh_hi = make_desc(ws), wh_lo = make_desc(ws + W_CHUNK);
        const uint64_t wx_hi = make_desc(ws + 2 * W_CHUNK), wx_lo = make_desc(ws + 3 * W_CHUNK);
        const uint64_t wx_hi_n = make_desc(ws + 2 * W_CHUNK + 128 * 128);  // rows 128..191 of W_ih (the n gate)
        constexpr uint32_t id192 = make_idesc(TILE, 192), id128 = make_idesc(TILE, 128), id64 = make_idesc(TILE, 64);
        const uint32_t xs = smem_u32(xring);
        int buf = 0, it = 0;
        uint32_t acc_ph = 0, xph = 0;
        T2P(long long t_m0 = clock64(), t_wacc = 0, t_wfull = 0, c0;)
#ifdef MRB_TC_PROF
#define WAIT_FULL(bar, par) do { c0 = clock64(); mbar_wait(bar, par); t_wfull += clock64() - c0; } while (0)
#else
#define WAIT_FULL(bar, par) mbar_wait(bar, par)
#endif
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int p = it & 1;
            const uint32_t hph = (uint32_t)(it >> 1) & 1u;
            T2P(c0 = clock64();)
            mbar_wait(&acc_empty[buf], acc_ph ^ 1);
            T2P(t_wacc += clock64() - c0;)
            tc_fence_after();
            // accumulator columns: [0,64) hh_n | [64,128) r | [128,192) z | [192,256) ih_n
            const uint32_t d = tmem_u + (uint32_t)(buf * 256);
            // h_hi x (Whh_hi, Whh_lo): the first MMA overwrites columns [0,192)
            WAIT_FULL(&hfull[2 * p], hph);
            tc_fence_after();
            uint64_t a = make_desc(rs + (uint32_t)((2 * p) * SLOT_BYTES));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                umma_ss(d, a + 2 * k, wh_hi + 2 * k, id192, k > 0);
                umma_ss(d, a + 2 * k, wh_lo + 2 * k, id192, 1);
            }
            umma_commit(&hempty[2 * p]);
            // h_lo x Whh_hi
            WAIT_FULL(&hfull[2 * p + 1], hph);
            tc_fence_after();
            a = make_desc(rs + (uint32_t)((2 * p + 1) * SLOT_BYTES));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_ss(d, a + 2 * k, wh_hi + 2 * k, id192, 1);
            umma_commit(&hempty[2 * p + 1]);
            // x_hi x (Wih_hi, Wih_lo): r, z accumulate onto the h part, the ih_n columns start here
            WAIT_FULL(&xfull[0], xph);
            tc_fence_after();
            a = make_desc(xs);
            umma_ss(d + 64, a, wx_hi, id128, 1);
            umma_ss(d + 192, a, wx_hi_n, id64, 0);
            umma_ss(d + 64, a, wx_lo, id192, 1);
#pragma unroll
            for (int k = 1; k < 4; ++k) {
                umma_ss(d + 64, a + 2 * k, wx_hi + 2 * k, id192, 1);
                umma_ss(d + 64, a + 2 * k, wx_lo + 2 * k, id192, 1);
            }
            umma_commit(&xempty[0]);
            // x_lo x Wih_hi
            WAIT_FULL(&xfull[1], xph);
            tc_fence_after();
            a = make_desc(xs + SLOT_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_ss(d + 64, a + 2 * k, wx_hi + 2 * k, id192, 1);
            umma_commit(&xempty[1]);
            xph ^= 1;
            umma_commit(&acc_full[buf]);
            if (++buf == 2) { buf = 0; acc_ph ^= 1; }
        }
        T2P(if (P.prof && lane == 0) { P.prof[blockIdx.x * 16 + 2] = clock64() - t_m0; P.prof[blockIdx.x * 16 + 3] = t_wacc; P.prof[blockIdx.x * 16 + 4] = t_wfull; })
    } else if (warp == EPI_W + 2) {
        // ============================== TMA STORE LANE ==============================
        // waits until the 16 epilogue warps have written a tile's output boxes, stores them and frees the output tile as
        // soon as the stores have read it
        if (lane == 0) {
            uint32_t oph = 0;
            int it = 0;
            const uint32_t out_u32 = smem_u32(out_s);
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
                mbar_wait_sleep(out_ready, oph, 64);
                if (!T2_DBG(P, 8)) {
                    tma_store_2d(&tm_o, out_u32, 0, tile * TILE);
                    tma_store_2d(&tm_o, out_u32 + SLOT_BYTES, 64, tile * TILE);
                }
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                mbar_arrive(&out_free[it & 1]);
                oph ^= 1;
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before the CTA exits
        }
    } else {
        // ============================== EPILOGUE ==============================
        const int quad = warp & 3;   // TMEM lane quadrant
        const int cg = warp >> 2;    // channels 16*cg .. 16*cg + 15
        const int m = quad * 32 + lane;  // tile row = TMEM lane of this thread
        const uint32_t bias_u32 = smem_u32(bias_s);
        const uint32_t ring_u32 = smem_u32(ring), out_u32 = smem_u32(out_s);
        T2P(long long t_e0 = clock64(), t_ew = 0, t_eld = 0, t_emath = 0, t_est = 0, c0;)
        int it = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int p = it & 1, buf = it & 1;
            const uint32_t hph = (uint32_t)(it >> 1) & 1u, acc_ph = (uint32_t)(it >> 1) & 1u;
            // this thread's two 16-byte chunks (8 channels each) of row m inside a [128 x 128 B] SWIZZLE_128B box
            const uint32_t ch0 = swz(m, 2 * cg), ch1 = swz(m, 2 * cg + 1);
            // ---- h_prev of this thread's row and channels from the landed h_hi / h_lo boxes, which are released on
            // behalf of this warp after its last read.  (An arrival can never be counted for an earlier phase of the
            // same box: the data this warp has just waited for was loaded after that earlier phase had completed.)
            float hp[16];
            {
                uint4 hh[2], hl[2];
                mbar_wait_sleep(&hfull[2 * p], hph, 32);
                hh[0] = lds128u(ring_u32 + (uint32_t)((2 * p) * SLOT_BYTES) + ch0);
                hh[1] = lds128u(ring_u32 + (uint32_t)((2 * p) * SLOT_BYTES) + ch1);
                mbar_wait_sleep(&hfull[2 * p + 1], hph, 32);
                hl[0] = lds128u(ring_u32 + (uint32_t)((2 * p + 1) * SLOT_BYTES) + ch0);
                hl[1] = lds128u(ring_u32 + (uint32_t)((2 * p + 1) * SLOT_BYTES) + ch1);
                fence_proxy_async();  // the loads complete before the TMA may refill the boxes (see ind2_kernel)
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&hempty[2 * p]);
                    mbar_arrive(&hempty[2 * p + 1]);
                }
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const uint32_t hw[4] = {hh[j].x, hh[j].y, hh[j].z, hh[j].w}, lw[4] = {hl[j].x, hl[j].y, hl[j].z, hl[j].w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        up2(add2(pk2(bf_lo(hw[i]), bf_hi(hw[i])), pk2(bf_lo(lw[i]), bf_hi(lw[i]))), hp[8 * j + 2 * i],
                            hp[8 * j + 2 * i + 1]);
                }
            }
            T2P(c0 = clock64();)
            mbar_wait_sleep(&acc_full[buf], acc_ph, 64);
            T2P(t_ew += clock64() - c0;)
            tc_fence_after();
            const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 256 + cg * 16);
            float o[16];
#pragma unroll
            for (int jb = 0; jb < 2; ++jb) {
                float hn[8], ar[8], az[8], xn[8];
                T2P(c0 = clock64();)
                tmem_ld8x4(t0 + jb * 8, t0 + 64 + jb * 8, t0 + 128 + jb * 8, t0 + 192 + jb * 8, hn, ar, az, xn);
                T2P(t_eld += clock64() - c0; c0 = clock64();)
                if (jb == 1) {  // all of this warp's accumulator columns are in registers
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[buf]);
                }
                if (T2_DBG(P, 4)) {
#pragma unroll
                    for (int q = 0; q < 8; ++q) o[jb * 8 + q] = hn[q] + ar[q] + az[q] + xn[q] + hp[jb * 8 + q];
                } else
#pragma unroll
                for (int q4 = 0; q4 < 8; q4 += 4) {
                    const int c = cg * 16 + jb * 8 + q4;
                    f32x2 br[2], bz[2], bn[2];
                    lds128p(bias_u32 + 4u * (uint32_t)c, br[0], br[1]);
                    lds128p(bias_u32 + 4u * (uint32_t)(64 + c), bz[0], bz[1]);
                    lds128p(bias_u32 + 4u * (uint32_t)(128 + c), bn[0], bn[1]);
                    const f32x2 one2 = pk2(1.f, 1.f), nl2 = pk2(-kLog2e, -kLog2e), tl2 = pk2(2.f * kLog2e, 2.f * kLog2e);
                    const f32x2 m2 = pk2(-2.f, -2.f);
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int q = q4 + 2 * u;
                        // rnn_cells.py:121-125 (ih + hh of the r and z gates were summed by the tensor core) on PAIRS of
                        // channels: the fp32x2 forms are the same IEEE operations in half the issue slots (22 -> 14
                        // instructions per output; the 5 SFU operations stay -- Newton reciprocals on the FMA pipe
                        // measured slower, DESIGN 4.3).  r = 1/(1+ea), z = 1/(1+eb) share ONE
                        // reciprocal: 1/((1+ea)(1+eb)); the exponents are clamped so that the product stays finite (a
                        // gate below 2^-60 is zero to fp32 in everything it multiplies)
                        float a0, a1, b0, b1;
                        up2(fma2(pk2(ar[q], ar[q + 1]), nl2, br[u]), a0, a1);
                        up2(fma2(pk2(az[q], az[q + 1]), nl2, bz[u]), b0, b1);
                        const f32x2 xa = pk2(ex2_approx(fminf(a0, 60.f)), ex2_approx(fminf(a1, 60.f)));
                        const f32x2 ea = add2(one2, xa);
                        const f32x2 eb = add2(one2, pk2(ex2_approx(fminf(b0, 60.f)), ex2_approx(fminf(b1, 60.f))));
                        float p0, p1;
                        up2(mul2(ea, eb), p0, p1);
                        const f32x2 ip = pk2(rcp_approx(p0), rcp_approx(p1));
                        const f32x2 r = mul2(eb, ip), z = mul2(ea, ip);
                        // n = tanh(ih_n + b_n + r * hh_n) = 1 - 2 / (1 + 2^(2 log2(e) v))
                        float v0, v1;
                        up2(mul2(fma2(r, pk2(hn[q], hn[q + 1]), add2(pk2(xn[q], xn[q + 1]), bn[u])), tl2), v0, v1);
                        float d0, d1;
                        up2(add2(one2, pk2(ex2_approx(v0), ex2_approx(v1))), d0, d1);
                        const f32x2 n = fma2(m2, pk2(rcp_approx(d0), rcp_approx(d1)), one2);
                        // h' = z h + n (1 - z)
                        up2(fma2(z, pk2(hp[jb * 8 + q], hp[jb * 8 + q + 1]), mul2(n, sub2p(one2, z))), o[jb * 8 + q],
                            o[jb * 8 + q + 1]);
                    }
                }
                T2P(t_emath += clock64() - c0;)
            }
            T2P(c0 = clock64();)
            // ---- hi/lo split into the output tile (rows = positions, same box layout as the inputs) + TMA stores
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) split_bf16x2(o[2 * i], o[2 * i + 1], hi[i], lo[i]);
            // the stores of the previous tile have read the output tile.  The store lane signals tile j on
            // out_free[j & 1]; a parity wait only tells neighbouring phases apart, and on that barrier the phase before the
            // awaited one (tile it - 3) is known to be complete: this warp waited for it before it wrote tile it - 2
            if (it >= 1) mbar_wait_sleep(&out_free[(it - 1) & 1], (uint32_t)((it - 1) >> 1) & 1u, 32);
            sts128u(out_u32 + ch0, make_uint4(hi[0], hi[1], hi[2], hi[3]));
            sts128u(out_u32 + ch1, make_uint4(hi[4], hi[5], hi[6], hi[7]));
            sts128u(out_u32 + SLOT_BYTES + ch0, make_uint4(lo[0], lo[1], lo[2], lo[3]));
            sts128u(out_u32 + SLOT_BYTES + ch1, make_uint4(lo[4], lo[5], lo[6], lo[7]));
            fence_proxy_async();  // generic-proxy writes -> visible to the TMA (async proxy)
            __syncwarp();
            if (lane == 0) mbar_arrive(out_ready);
            T2P(t_est += clock64() - c0;)
        }
        T2P(if (P.prof && threadIdx.x == 0) { unsigned long long* o = P.prof + blockIdx.x * 16; o[5] = clock64() - t_e0; o[6] = t_ew; o[7] = t_eld; o[8] = t_emath; o[9] = t_est; })
    }
    tc_fence_before();
    __syncthreads();
    if (warp == EPI_W + 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// edge pixels -> replicate border of a BH tensor (one thread per (border position, 16-byte piece))
__global__ void bh_fix_border_kernel(uint8_t* __restrict__ bh, int B, int H, int W) {
    const int Hp = H + 2 * PADB, Wp = W + 2 * PADB;
    const int nb = Hp * Wp - H * W;  // border positions per image
    const long long total = (long long)B * nb * 16;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int piece = (int)(t & 15);
        const long long r = t >> 4;
        const int i = (int)(r % nb), b = (int)(r / nb);
        int yp, xp;
        if (i < 2 * PADB * Wp) {  // top and bottom bands
            const int row = i / Wp;
            yp = row < PADB ? row : H + row;  // rows 0,1 and H+2,H+3
            xp = i - row * Wp;
        } else {  // left and right bands of the interior rows
            const int j = i - 2 * PADB * Wp;
            const int row = j / (2 * PADB), c = j - row * 2 * PADB;
            yp = PADB + row;
            xp = c < PADB ? c : W + c;
        }
        const int ys = min(max(yp, PADB), H + PADB - 1), xs = min(max(xp, PADB), W + PADB - 1);
        const uint4 v = *reinterpret_cast<const uint4*>(bh + (((long long)b * Hp + ys) * Wp + xs) * PX_BYTES + piece * 16);
        *reinterpret_cast<uint4*>(bh + (((long long)b * Hp + yp) * Wp + xp) * PX_BYTES + piece * 16) = v;
    }
}

// ---- layout converters -------------------------------------------------------------------------------
// fp32 channels-last [B,H,W,64] -> BH (hi/lo split, replicate border)
__global__ void bh_from_nhwc_kernel(const float* __restrict__ x, uint8_t* __restrict__ bh, int B, int H, int W) {
    const int Hp = H + 2 * PADB, Wp = W + 2 * PADB;
    const long long total = (long long)B * Hp * Wp * 8;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(t & 7);
        const long long q = t >> 3;
        const int xp = (int)(q % Wp);
        const long long r = q / Wp;
        const int yp = (int)(r % Hp), b = (int)(r / Hp);
        const int xx = min(max(xp - PADB, 0), W - 1), yy = min(max(yp - PADB, 0), H - 1);
        const float4* s = reinterpret_cast<const float4*>(x + (((long long)b * H + yy) * W + xx) * 64 + g * 8);
        const float4 a = __ldg(s), c = __ldg(s + 1);
        uint32_t hi[4], lo[4];
        split_bf16x2(a.x, a.y, hi[0], lo[0]);
        split_bf16x2(a.z, a.w, hi[1], lo[1]);
        split_bf16x2(c.x, c.y, hi[2], lo[2]);
        split_bf16x2(c.z, c.w, hi[3], lo[3]);
        uint8_t* d = bh + q * PX_BYTES + g * 16;
        *reinterpret_cast<uint4*>(d) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(d + 128) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}
// BH -> fp32 channels-last [B,H,W,64] (interior only; x = hi + lo)
__global__ void bh_to_nhwc_kernel(const uint8_t* __restrict__ bh, float* __restrict__ x, int B, int H, int W) {
    const int Hp = H + 2 * PADB, Wp = W + 2 * PADB;
    const long long total = (long long)B * H * W * 8;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int g = (int)(t & 7);
        const long long p = t >> 3;
        const int xx = (int)(p % W);
        const long long r = p / W;
        const int yy = (int)(r % H), b = (int)(r / H);
        const uint8_t* s = bh + (((long long)b * Hp + yy + PADB) * Wp + xx + PADB) * PX_BYTES + g * 16;
        const uint4 h = *reinterpret_cast<const uint4*>(s), l = *reinterpret_cast<const uint4*>(s + 128);
        float4* d = reinterpret_cast<float4*>(x + p * 64 + g * 8);
        d[0] = make_float4(bf_lo(h.x) + bf_lo(l.x), bf_hi(h.x) + bf_hi(l.x), bf_lo(h.y) + bf_lo(l.y), bf_hi(h.y) + bf_hi(l.y));
        d[1] = make_float4(bf_lo(h.z) + bf_lo(l.z), bf_hi(h.z) + bf_hi(l.z), bf_lo(h.w) + bf_lo(l.w), bf_hi(h.w) + bf_hi(l.w));
    }
}

// ---- IndRNN cell on BH activations ------------------------------------------------------------------------------------
// IndRNNCell with kernel size 1 (rnn_cells.py:264-391, the cell base_cirim_run.yaml ships): h' = ReLU(W_ih x + b + hh * h),
// hh one recurrent weight per channel.  Same skeleton as gru2_kernel with a third of the tensor work: the x boxes feed
// 8 MMAs per tile (x_hi x [w_hi ; w_lo], N = 128: main | cross columns; x_lo x w_hi, N = 64 onto the cross columns), the h
// boxes are only read by the epilogue (h_prev from the TMA-landed slots), four accumulator buffers, double-buffered output
// tile.  Pointwise over all (H+4)(W+4) positions; HBM-bound like the ConvGRU (768 B per position).
struct Ind2Params {
    const void* wpack;   // mrb_tc_pack_conv(ih.weight, 64, 64, 1): [hi 64 x 128 B | lo 64 x 128 B], SWIZZLE_128B
    const float* bias;   // b_ih [64] or null
    const float* hh;     // [64]
    long long Q;
    int n_tiles;
};

__global__ void __launch_bounds__(THREADS2, 1)
ind2_kernel(const __grid_constant__ CUtensorMap tm_h, const __grid_constant__ CUtensorMap tm_x,
            const __grid_constant__ CUtensorMap tm_o, const Ind2Params P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* w_s = smem;                                  // [hi 64 rows | lo 64 rows] x 128 B
    uint8_t* hring = w_s + SLOT_BYTES;                    // [2 tiles][h_hi | h_lo]
    uint8_t* xring = hring + 4 * SLOT_BYTES;              // [2 tiles][x_hi | x_lo]
    uint8_t* out_s = xring + 4 * SLOT_BYTES;              // [2 buffers][hi box | lo box]
    float* bias_s = (float*)(out_s + 4 * SLOT_BYTES);     // [64] bias | [64] hh
    uint64_t* hfull = (uint64_t*)(bias_s + 128);          // [2]
    uint64_t* hempty = hfull + 2;                         // [2] one arrival per epilogue warp
    uint64_t* xfull = hempty + 2;                         // [2]
    uint64_t* xempty = xfull + 2;                         // [2] MMA commit
    uint64_t* acc_full = xempty + 2;                      // [4]
    uint64_t* acc_empty = acc_full + 4;                   // [4]
    uint64_t* out_ready = acc_empty + 4;                  // [2]
    uint64_t* out_free = out_ready + 2;                   // [2]
    uint32_t* tmem_slot = (uint32_t*)(out_free + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&hfull[i], 1);
            mbar_init(&hempty[i], EPI_W);
            mbar_init(&xfull[i], 1);
            mbar_init(&xempty[i], 1);
            mbar_init(&out_ready[i], EPI_W);
            mbar_init(&out_free[i], 1);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], EPI_W);
        }
        fence_barrier_init();
    }
    if (threadIdx.x < 64) {
        bias_s[threadIdx.x] = P.bias ? P.bias[threadIdx.x] : 0.f;
        bias_s[64 + threadIdx.x] = P.hh[threadIdx.x];
    }
    if (warp == EPI_W + 1) tmem_alloc(tmem_slot, 512);
    {
        const float4* g = reinterpret_cast<const float4*>(P.wpack);
        const uint32_t sa = smem_u32(w_s);
        for (int i = threadIdx.x; i < SLOT_BYTES / 16; i += THREADS2) sts128(sa + 16u * (uint32_t)i, __ldg(g + i));
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == EPI_W) {
        // ============================== TMA PRODUCER ==============================
        if (lane == 0) {
            int it = 0;
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
                const int p = it & 1;
                const uint32_t ph = (uint32_t)(it >> 1) & 1u;
                mbar_wait_sleep(&xempty[p], ph ^ 1, 64);
                mbar_expect_tx(&xfull[p], 2 * SLOT_BYTES);
                tma_load_2d(smem_u32(xring + (2 * p) * SLOT_BYTES), &tm_x, 0, tile * TILE, smem_u32(&xfull[p]));
                tma_load_2d(smem_u32(xring + (2 * p + 1) * SLOT_BYTES), &tm_x, 64, tile * TILE, smem_u32(&xfull[p]));
                mbar_wait_sleep(&hempty[p], ph ^ 1, 64);
                mbar_expect_tx(&hfull[p], 2 * SLOT_BYTES);
                tma_load_2d(smem_u32(hring + (2 * p) * SLOT_BYTES), &tm_h, 0, tile * TILE, smem_u32(&hfull[p]));
                tma_load_2d(smem_u32(hring + (2 * p + 1) * SLOT_BYTES), &tm_h, 64, tile * TILE, smem_u32(&hfull[p]));
            }
        }
    } else if (warp == EPI_W + 1) {
        // ============================== MMA ISSUER ==============================
        const uint32_t tmem_u = uni(tmem_base);
        const uint64_t w_stack = make_desc(smem_u32(w_s));  // N = 128: [w_hi ; w_lo]; N = 64: w_hi
        constexpr uint32_t id128 = make_idesc(TILE, 128), id64 = make_idesc(TILE, 64);
        const uint32_t xs = smem_u32(xring);
        int it = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int p = it & 1, buf = it & 3;
            mbar_wait(&acc_empty[buf], ((uint32_t)(it >> 2) & 1u) ^ 1u);
            mbar_wait(&xfull[p], (uint32_t)(it >> 1) & 1u);
            tc_fence_after();
            const uint32_t d = tmem_u + (uint32_t)(buf * 128);
            const uint64_t a_hi = make_desc(xs + (uint32_t)((2 * p) * SLOT_BYTES));
            const uint64_t a_lo = make_desc(xs + (uint32_t)((2 * p + 1) * SLOT_BYTES));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_ss(d, a_hi + 2 * k, w_stack + 2 * k, id128, k > 0);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_ss(d + 64, a_lo + 2 * k, w_stack + 2 * k, id64, 1);
            umma_commit(&xempty[p]);
            umma_commit(&acc_full[buf]);
        }
    } else if (warp == EPI_W + 2) {
        // ============================== TMA STORE LANE ==============================
        if (lane == 0) {
            int it = 0;
            const uint32_t out_u32 = smem_u32(out_s);
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
                const int ob = it & 1;
                mbar_wait_sleep(&out_ready[ob], (uint32_t)(it >> 1) & 1u, 64);
                tma_store_2d(&tm_o, out_u32 + (uint32_t)(ob * 2 * SLOT_BYTES), 0, tile * TILE);
                tma_store_2d(&tm_o, out_u32 + (uint32_t)(ob * 2 * SLOT_BYTES + SLOT_BYTES), 64, tile * TILE);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                mbar_arrive(&out_free[ob]);
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
    } else {
        // ============================== EPILOGUE ==============================
        const int quad = warp & 3, cg = warp >> 2;
        const int m = quad * 32 + lane;
        const uint32_t ch0 = swz(m, 2 * cg), ch1 = swz(m, 2 * cg + 1);
        const uint32_t hring_u32 = smem_u32(hring), out_u32 = smem_u32(out_s);
        float bs[16], hw[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            bs[i] = bias_s[cg * 16 + i];
            hw[i] = bias_s[64 + cg * 16 + i];
        }
        int it = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int p = it & 1, buf = it & 3;
            float hp[16];
            {
                mbar_wait_sleep(&hfull[p], (uint32_t)(it >> 1) & 1u, 32);
                const uint32_t hb = hring_u32 + (uint32_t)((2 * p) * SLOT_BYTES);
                const uint4 h0 = lds128u(hb + ch0), h1 = lds128u(hb + ch1);
                const uint4 l0 = lds128u(hb + SLOT_BYTES + ch0), l1 = lds128u(hb + SLOT_BYTES + ch1);
                // generic-proxy reads -> async-proxy (TMA) overwrite of the same boxes: the proxy fence makes the loads
                // complete before the release; without it the refill of the slot overtook the last loads of a late warp
                // (second 16-byte chunk of a few rows, about once per 800 tiles)
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&hempty[p]);
                const uint32_t hw_[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
                const uint32_t lw_[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    hp[2 * i] = bf_lo(hw_[i]) + bf_lo(lw_[i]);
                    hp[2 * i + 1] = bf_hi(hw_[i]) + bf_hi(lw_[i]);
                }
            }
            mbar_wait_sleep(&acc_full[buf], (uint32_t)(it >> 2) & 1u, 64);
            tc_fence_after();
            const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 128 + cg * 16);
            float m0[8], m1[8], c0[8], c1[8];
            tmem_ld8x4(t0, t0 + 8, t0 + 64, t0 + 72, m0, m1, c0, c1);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
            float o[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                // rnn_cells.py:391: ReLU(ih(x) + hh * h)
                o[i] = fmaxf(fmaf(hw[i], hp[i], (m0[i] + c0[i]) + bs[i]), 0.f);
                o[8 + i] = fmaxf(fmaf(hw[8 + i], hp[8 + i], (m1[i] + c1[i]) + bs[8 + i]), 0.f);
            }
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) split_bf16x2(o[2 * i], o[2 * i + 1], hi[i], lo[i]);
            const int ob = it & 1;
            mbar_wait_sleep(&out_free[ob], ((uint32_t)(it >> 1) & 1u) ^ 1u, 32);
            const uint32_t ou = out_u32 + (uint32_t)(ob * 2 * SLOT_BYTES);
            sts128u(ou + ch0, make_uint4(hi[0], hi[1], hi[2], hi[3]));
            sts128u(ou + ch1, make_uint4(hi[4], hi[5], hi[6], hi[7]));
            sts128u(ou + SLOT_BYTES + ch0, make_uint4(lo[0], lo[1], lo[2], lo[3]));
            sts128u(ou + SLOT_BYTES + ch1, make_uint4(lo[4], lo[5], lo[6], lo[7]));
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&out_ready[ob]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == EPI_W + 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}
static size_t ind2_smem() { return 1024 + 13 * SLOT_BYTES + 128 * 4 + 24 * 8 + 16; }

// ---- final RIM conv (64 -> 2, 3x3) as a tap GEMM + in-SM gather ------------------------------------------------------
// out[y][x][o] = eta + bias[o] + sum_{tap, c} w[o][c][tap] * h[clamp(y + dy)][clamp(x + dx)][c]   (rim_block.py:239-248,
// conv_layers.py:72-123 with ReplicationPad2d(1)).
// The channel contraction does not depend on where a tap is read from, so it runs ONCE per position on the tensor core:
//   T[pos][tap*2 + o] = sum_c h[pos][c] * w[o][c][tap]          (M = 128 positions, N = 18 padded to 32, K = 64)
// and the spatial part is nine fp32 additions per output, out = sum_tap T[pos + tap][tap], done by the epilogue warps
// through shared memory.  The CUDA-core kernel this replaces (conv_c2_k3_kernel<.., BH>) was FP32-pipe / latency bound at
// ~4x the HBM time of reading h once.
//   patch        16 x 16 positions (two M = 128 tiles) -> 14 x 14 outputs; one 3-D TMA box per operand half (hi / lo) lands
//                in the UMMA SWIZZLE_128B layout, three patches in flight; overlapping halo positions are L2 hits
//   MMA lane     per tile 4 k-steps x { h_hi x [w_hi ; w_lo] (N = 64: columns 0..31 hi*hi, 32..63 hi*lo), h_lo x w_hi (N = 32,
//                onto the cross-term columns) }; main and cross terms are added in RN fp32 by the epilogue
//   8 epilogue warps  T of their position -> shared memory, barrier, gather with the tap coordinates clamped to the image
//                (the replicate padding: the BH border of the source is never used, so no border fix-up is needed), + eta
constexpr int F2_PATCH = 16, F2_OUT = 14;
constexpr int F2_STAGES = 3;
constexpr int F2_STAGE_BYTES = 2 * 2 * SLOT_BYTES;  // hi box (2 tiles) | lo box (2 tiles)
constexpr int F2_EPI_W = 8;
constexpr int F2_THREADS = (F2_EPI_W + 2) * 32;
constexpr int F2_TS = 18;                            // floats per position in the T exchange tile

struct Fin2Params {
    const float* w;     // [2][64][3][3]
    const float* bias;  // [2] or null
    const float* eta;   // [B][H][W][2]
    float* out;         // [B][H][W][2]
    int B, H, W;
    int py, px;         // patches per image column / row
    int n_patches;
};

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, int c0, int c1, int c2, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
                 "l"(m), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
                 : "memory");
}
// 18 main + 18 cross-term columns of this thread's TMEM lane (columns [0,24) and [32,56) of the tile's accumulator)
__device__ __forceinline__ void tmem_ld_fin2(uint32_t a, float* v) {
    uint32_t r[48];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%48];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%8,%9,%10,%11,%12,%13,%14,%15}, [%49];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%16,%17,%18,%19,%20,%21,%22,%23}, [%50];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%24,%25,%26,%27,%28,%29,%30,%31}, [%51];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%32,%33,%34,%35,%36,%37,%38,%39}, [%52];\n\t"
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%40,%41,%42,%43,%44,%45,%46,%47}, [%53];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]),
          "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]),
          "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47])
        : "r"(a), "r"(a + 8), "r"(a + 16), "r"(a + 32), "r"(a + 40), "r"(a + 48)
        : "memory");
#pragma unroll
    for (int i = 0; i < F2_TS; ++i) v[i] = __uint_as_float(r[i]) + __uint_as_float(r[24 + i]);
}

__global__ void __launch_bounds__(F2_THREADS, 1)
fin2_kernel(const __grid_constant__ CUtensorMap tm_h, const Fin2Params P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* stage_s = smem;                                      // [F2_STAGES][hi 32 KB | lo 32 KB]
    uint8_t* w_s = stage_s + F2_STAGES * F2_STAGE_BYTES;          // [w_hi 32 rows x 128 B | w_lo 32 rows x 128 B]
    float* ts = (float*)(w_s + 2 * 32 * 128);                     // [256 positions][18]
    uint64_t* full = (uint64_t*)(ts + 256 * F2_TS);               // [F2_STAGES]
    uint64_t* empty = full + F2_STAGES;                           // [F2_STAGES] MMA commit
    uint64_t* acc_full = empty + F2_STAGES;                       // [2]
    uint64_t* acc_empty = acc_full + 2;                           // [2] one arrival per epilogue warp
    uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < F2_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], F2_EPI_W);
        }
        fence_barrier_init();
    }
    // weights: row n = tap*2 + o (18 used of 32), K = 64 input channels, split into bf16 hi / lo, SWIZZLE_128B rows
    for (int i = threadIdx.x; i < 32 * 64; i += F2_THREADS) {
        const int n = i >> 6, k = i & 63;
        const float v = n < 18 ? P.w[((n & 1) * 64 + k) * 9 + (n >> 1)] : 0.f;
        const uint16_t hb = bf16_rn_bits(v);
        const float hf = __uint_as_float((uint32_t)hb << 16);
        const uint16_t lb = bf16_rn_bits(v - hf);
        const uint32_t off = swz(n, k >> 3) + (uint32_t)((k & 7) * 2);
        *reinterpret_cast<uint16_t*>(w_s + off) = hb;
        *reinterpret_cast<uint16_t*>(w_s + 32 * 128 + off) = lb;
    }
    if (warp == F2_EPI_W + 1) tmem_alloc(tmem_slot, 256);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int Hp = P.H + 2 * PADB;
    const int per_img = P.py * P.px;

    if (warp == F2_EPI_W) {
        // ============================== TMA PRODUCER ==============================
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int t = blockIdx.x; t < P.n_patches; t += gridDim.x) {
                const int b = t / per_img, r = t - b * per_img;
                const int pi = r / P.px, pj = r - pi * P.px;
                // patch origin in padded coordinates: outputs (14 pi .. +13) sit at padded rows 14 pi + 2 ..; one halo row above
                const int y0 = b * Hp + F2_OUT * pi + PADB - 1, x0 = F2_OUT * pj + PADB - 1;
                mbar_wait_sleep(&empty[s], ph ^ 1, 64);
                mbar_expect_tx(&full[s], F2_STAGE_BYTES);
                const uint32_t dst = smem_u32(stage_s + s * F2_STAGE_BYTES);
                tma_load_3d(dst, &tm_h, 0, x0, y0, smem_u32(&full[s]));
                tma_load_3d(dst + 2 * SLOT_BYTES, &tm_h, 64, x0, y0, smem_u32(&full[s]));
                if (++s == F2_STAGES) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp == F2_EPI_W + 1) {
        // ============================== MMA ISSUER ==============================
        const uint32_t tmem_u = uni(tmem_base);
        const uint64_t w_stack = make_desc(smem_u32(w_s));
        constexpr uint32_t id64 = make_idesc(TILE, 64), id32 = make_idesc(TILE, 32);
        int s = 0, buf = 0;
        uint32_t ph = 0, acc_ph = 0;
        for (int t = blockIdx.x; t < P.n_patches; t += gridDim.x) {
            mbar_wait(&acc_empty[buf], acc_ph ^ 1);
            mbar_wait(&full[s], ph);
            tc_fence_after();
            const uint32_t sb = smem_u32(stage_s + s * F2_STAGE_BYTES);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const uint32_t d = tmem_u + (uint32_t)(buf * 128 + j * 64);
                const uint64_t a_hi = make_desc(sb + (uint32_t)(j * SLOT_BYTES));
                const uint64_t a_lo = make_desc(sb + (uint32_t)((2 + j) * SLOT_BYTES));
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    umma_ss(d, a_hi + 2 * k, w_stack + 2 * k, id64, k > 0);
                    umma_ss(d + 32, a_lo + 2 * k, w_stack + 2 * k, id32, 1);
                }
            }
            umma_commit(&empty[s]);
            umma_commit(&acc_full[buf]);
            if (++s == F2_STAGES) { s = 0; ph ^= 1; }
            if (++buf == 2) { buf = 0; acc_ph ^= 1; }
        }
    } else {
        // ============================== EPILOGUE ==============================
        const int quad = warp & 3, j = warp >> 2;
        const int m = quad * 32 + lane;          // TMEM lane = row of M-tile j
        const int pos = j * TILE + m;            // position inside the patch: row pos / 16, column pos % 16
        const int r = pos >> 4, c = pos & 15;
        const float b0 = P.bias ? P.bias[0] : 0.f, b1 = P.bias ? P.bias[1] : 0.f;
        const uint32_t ts_u32 = smem_u32(ts);
        int buf = 0;
        uint32_t acc_ph = 0;
        for (int t = blockIdx.x; t < P.n_patches; t += gridDim.x) {
            const int b = t / per_img, rr = t - b * per_img;
            const int pi = rr / P.px, pj = rr - pi * P.px;
            const int y = F2_OUT * pi + r - 1, x = F2_OUT * pj + c - 1;  // output pixel of this thread
            const bool valid = r >= 1 && r <= F2_OUT && c >= 1 && c <= F2_OUT && y < P.H && x < P.W;
            const long long p = ((long long)b * P.H + y) * P.W + x;
            float2 e = make_float2(0.f, 0.f);
            if (valid) e = __ldg(reinterpret_cast<const float2*>(P.eta) + p);
            mbar_wait_sleep(&acc_full[buf], acc_ph, 64);
            tc_fence_after();
            float v[F2_TS];
            tmem_ld_fin2(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 128 + j * 64), v);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
            asm volatile("bar.sync 1, %0;" ::"n"(F2_EPI_W * 32) : "memory");  // the previous patch has been gathered
#pragma unroll
            for (int i = 0; i < F2_TS / 2; ++i)
                asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(ts_u32 + (uint32_t)((pos * F2_TS + 2 * i) * 4)), "f"(v[2 * i]),
                             "f"(v[2 * i + 1])
                             : "memory");
            asm volatile("bar.sync 1, %0;" ::"n"(F2_EPI_W * 32) : "memory");
            if (valid) {
                // replicate padding = clamp the tap's image coordinates; a clamped tap is this thread's own row / column
                const int rm = y > 0 ? r - 1 : r, rp = y < P.H - 1 ? r + 1 : r;
                const int cm = x > 0 ? c - 1 : c, cp = x < P.W - 1 ? c + 1 : c;
                const int rows[3] = {rm, r, rp}, cols[3] = {cm, c, cp};
                float s0 = 0.f, s1 = 0.f;
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) {
                        float t0, t1;
                        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];"
                                     : "=f"(t0), "=f"(t1)
                                     : "r"(ts_u32 + (uint32_t)(((rows[dy] * F2_PATCH + cols[dx]) * F2_TS + 2 * (dy * 3 + dx)) * 4))
                                     : "memory");
                        s0 += t0;
                        s1 += t1;
                    }
                reinterpret_cast<float2*>(P.out)[p] = make_float2(e.x + (s0 + b0), e.y + (s1 + b1));
            }
            if (++buf == 2) { buf = 0; acc_ph ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == F2_EPI_W + 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256);
    }
}
static size_t fin2_smem() { return 1024 + F2_STAGES * F2_STAGE_BYTES + 2 * 32 * 128 + 256 * F2_TS * 4 + 16 * 8 + 16; }

// A BH tensor as the 3-D array [B*(H+4) rows][W+4 columns][128 bf16]; box = 64 channels (hi or lo half) x 16 columns x 16 rows
static int make_bh_tmap3(void* mp, const void* base, int B, int H, int W) {
    CUtensorMap* m = reinterpret_cast<CUtensorMap*>(mp);
    EncodeTiledFn fn = encode_fn();
    MRB_REQUIRE(fn != nullptr, MRB_ECUDA, "cuTensorMapEncodeTiled is not available from the driver");
    const cuuint64_t Wp = (cuuint64_t)(W + 2 * PADB), rows = (cuuint64_t)B * (cuuint64_t)(H + 2 * PADB);
    cuuint64_t dims[3] = {128, Wp, rows};
    cuuint64_t strides[2] = {PX_BYTES, Wp * PX_BYTES};
    cuuint32_t box[3] = {64, F2_PATCH, F2_PATCH};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MRB_REQUIRE(r == CUDA_SUCCESS, MRB_ECUDA, "cuTensorMapEncodeTiled (3-D) failed (%d)", (int)r);
    return MRB_OK;
}

// ---- first RIM conv (4 -> 64, 5x5) fed by bulk copies ---------------------------------------------------------------
// ConvNonlinear(4 -> 64, k = 5, ReplicationPad2d(2), ReLU) on the RIM input [eta.re, eta.im, grad.re, grad.im]
// (rim_block.py:233-238, conv_layers.py:72-123).
// Input format "G8": the 4 channels of a position as 4 bf16 hi + 4 bf16 lo = 16 bytes, positions in the padded BH geometry
// [B][H+4][W+4] (replicate border written by the producer), with zeroed guard positions before and after the tensor.  In
// the UMMA no-swizzle K-major layout a core matrix is 8 rows x 16 bytes stored contiguously, i.e. 8 consecutive positions of
// a G8 row ARE a core matrix: the A operand of tap (dy, dx) for 128 consecutive (flat) positions is the contiguous G8 range
// starting dy rows up / dx positions left.  Per tile the loader therefore issues five 1-D bulk copies (one per tap row,
// 136 positions = 2176 B) and every tap of that row is the same shared-memory segment at a 16-byte offset: an MMA with
// K = 16 takes two neighbouring taps (leading-dimension byte offset 16).  No im2col, no conversion, 10.6 KB of loads per
// 128 outputs.  K per position: 8 = [hi | lo]; weights B1 = [w_hi | w_hi] (main term (a_hi + a_lo) w_hi) stacked on
// B2 = [w_lo | 0] (cross term a_hi w_lo) -> one N = 128 MMA per tap pair, 15 per tile; the epilogue adds main + cross in RN
// fp32, bias, ReLU, splits into the BH box layout, and a store lane issues the two TMA stores.
// Pointwise in the flat padded position space like gru2_kernel: border positions of the output are written but are not
// replicate copies (the ConvGRU that follows is pointwise).
constexpr int C5_SEG_POS = 136;                      // 128 + 4 taps + pad tap, rounded to whole core matrices
constexpr int C5_SEG_BYTES = C5_SEG_POS * 16;
constexpr int C5_STAGE_BYTES = 5 * C5_SEG_BYTES;
constexpr int C5_STAGES = 4;
constexpr int C5_B_CHUNK = 128 * 16;                 // [128 rows][8 bf16] of one tap
constexpr int C5_B_BYTES = 15 * 2 * C5_B_CHUNK;      // (tap row, tap pair) x 2 taps
constexpr int C5_THREADS = (EPI_W + 3) * 32;

struct Conv5Params {
    const uint8_t* g8;   // first guard position
    const float* w;      // [64][4][5][5]
    const float* bias;   // [64] or null
    long long Q;         // B * (H+4) * (W+4)
    long long guard_lo;  // positions before position 0
    int Wp;
    int n_tiles;
    int relu;
};

__device__ __forceinline__ uint64_t make_desc_ns(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;  // byte distance between the two 16-byte K chunks of an MMA
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;  // byte distance between 8-row core matrices
    d |= (uint64_t)1 << 46;                      // descriptor version (Blackwell); layout type 0 = no swizzle
    return d;
}

__global__ void __launch_bounds__(C5_THREADS, 1)
conv5g_kernel(const __grid_constant__ CUtensorMap tm_o, const Conv5Params P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* out_s = smem;                                         // [2 buffers][hi box | lo box], SWIZZLE_128B
    uint8_t* w_s = out_s + 4 * SLOT_BYTES;                         // [15 pairs][2 taps][128 rows][16 B]
    uint8_t* a_s = w_s + C5_B_BYTES;                               // [C5_STAGES][5 tap rows][136 positions][16 B]
    float* bias_s = (float*)(a_s + C5_STAGES * C5_STAGE_BYTES);    // [64]
    uint64_t* full = (uint64_t*)(bias_s + 64);                     // [C5_STAGES]
    uint64_t* empty = full + C5_STAGES;                            // [C5_STAGES] MMA commit
    uint64_t* acc_full = empty + C5_STAGES;                        // [4]
    uint64_t* acc_empty = acc_full + 4;                            // [4] one arrival per epilogue warp
    uint64_t* out_ready = acc_empty + 4;                           // [2] one arrival per epilogue warp
    uint64_t* out_free = out_ready + 2;                            // [2] the TMA stores have read the buffer
    uint32_t* tmem_slot = (uint32_t*)(out_free + 2);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < C5_STAGES; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], 1);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], EPI_W);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&out_ready[i], EPI_W);
            mbar_init(&out_free[i], 1);
        }
        fence_barrier_init();
    }
    if (threadIdx.x < 64) bias_s[threadIdx.x] = P.bias ? P.bias[threadIdx.x] : 0.f;
    // weights: chunk (tap row dy, pair p, kc) = tap (dy, dx = 2p + kc) (dx = 5: zero pad tap); row n < 64: [w_hi | w_hi] of
    // output channel n, row 64 + n: [w_lo | 0]
    for (int i = threadIdx.x; i < 30 * 128; i += C5_THREADS) {
        const int chunk = i >> 7, n = i & 127;
        const int dy = chunk / 6, dx = chunk - dy * 6;
        uint32_t hi01 = 0, hi23 = 0, lo01 = 0, lo23 = 0;
        if (dx < 5) {
            const float* wp = P.w + ((long long)(n & 63) * 4) * 25 + dy * 5 + dx;
            split_bf16x2(wp[0], wp[25], hi01, lo01);
            split_bf16x2(wp[50], wp[75], hi23, lo23);
        }
        const uint4 v = n < 64 ? make_uint4(hi01, hi23, hi01, hi23) : make_uint4(lo01, lo23, 0u, 0u);
        *reinterpret_cast<uint4*>(w_s + (size_t)chunk * C5_B_CHUNK + n * 16) = v;
    }
    if (warp == EPI_W + 1) tmem_alloc(tmem_slot, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == EPI_W) {
        // ============================== BULK-COPY PRODUCER ==============================
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
                mbar_wait_sleep(&empty[s], ph ^ 1, 64);
                mbar_expect_tx(&full[s], C5_STAGE_BYTES);
                const uint32_t dst = smem_u32(a_s + s * C5_STAGE_BYTES);
                // tap row dy reads positions q0 + (dy - 2) Wp - 2 ... (+ 135)
                const uint8_t* src = P.g8 + (P.guard_lo + (long long)tile * TILE - 2LL * P.Wp - 2) * 16;
#pragma unroll
                for (int dy = 0; dy < 5; ++dy)
                    bulk_load_1d(dst + dy * C5_SEG_BYTES, src + (long long)dy * P.Wp * 16, C5_SEG_BYTES, smem_u32(&full[s]));
                if (++s == C5_STAGES) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp == EPI_W + 1) {
        // ============================== MMA ISSUER ==============================
        const uint32_t tmem_u = uni(tmem_base);
        const uint64_t bdesc0 = make_desc_ns(smem_u32(w_s), C5_B_CHUNK, 128);
        const uint64_t adesc0 = make_desc_ns(smem_u32(a_s), 16, 128);
        constexpr uint32_t id128 = make_idesc(TILE, 128);
        int s = 0, buf = 0;
        uint32_t ph = 0, acc_ph = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
            mbar_wait(&acc_empty[buf], acc_ph ^ 1);
            mbar_wait(&full[s], ph);
            tc_fence_after();
            const uint32_t d = tmem_u + (uint32_t)(buf * 128);
            const uint64_t a_st = adesc0 + (uint64_t)((s * C5_STAGE_BYTES) >> 4);
#pragma unroll
            for (int dy = 0; dy < 5; ++dy)
#pragma unroll
                for (int p = 0; p < 3; ++p)
                    umma_ss(d, a_st + (uint64_t)((dy * C5_SEG_BYTES + 2 * p * 16) >> 4),
                            bdesc0 + (uint64_t)(((dy * 3 + p) * 2 * C5_B_CHUNK) >> 4), id128, (dy | p) != 0);
            umma_commit(&empty[s]);
            umma_commit(&acc_full[buf]);
            if (++s == C5_STAGES) { s = 0; ph ^= 1; }
            if (++buf == 4) { buf = 0; acc_ph ^= 1; }
        }
    } else if (warp == EPI_W + 2) {
        // ============================== TMA STORE LANE ==============================
        if (lane == 0) {
            int it = 0;
            const uint32_t out_u32 = smem_u32(out_s);
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
                const int ob = it & 1;
                mbar_wait_sleep(&out_ready[ob], (uint32_t)(it >> 1) & 1u, 64);
                tma_store_2d(&tm_o, out_u32 + (uint32_t)(ob * 2 * SLOT_BYTES), 0, tile * TILE);
                tma_store_2d(&tm_o, out_u32 + (uint32_t)(ob * 2 * SLOT_BYTES + SLOT_BYTES), 64, tile * TILE);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                mbar_arrive(&out_free[ob]);
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
    } else {
        // ============================== EPILOGUE ==============================
        const int quad = warp & 3, cg = warp >> 2;
        const int m = quad * 32 + lane;
        const uint32_t ch0 = swz(m, 2 * cg), ch1 = swz(m, 2 * cg + 1);
        const uint32_t out_u32 = smem_u32(out_s);
        float bs[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) bs[i] = bias_s[cg * 16 + i];
        int buf = 0, it = 0;
        uint32_t acc_ph = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            mbar_wait_sleep(&acc_full[buf], acc_ph, 64);
            tc_fence_after();
            const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 128 + cg * 16);
            float m0[8], m1[8], c0[8], c1[8];
            tmem_ld8x4(t0, t0 + 8, t0 + 64, t0 + 72, m0, m1, c0, c1);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
            float o[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                o[i] = (m0[i] + c0[i]) + bs[i];
                o[8 + i] = (m1[i] + c1[i]) + bs[8 + i];
            }
            if (P.relu) {
#pragma unroll
                for (int i = 0; i < 16; ++i) o[i] = fmaxf(o[i], 0.f);
            }
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) split_bf16x2(o[2 * i], o[2 * i + 1], hi[i], lo[i]);
            const int ob = it & 1;
            mbar_wait_sleep(&out_free[ob], ((uint32_t)(it >> 1) & 1u) ^ 1u, 32);
            const uint32_t ou = out_u32 + (uint32_t)(ob * 2 * SLOT_BYTES);
            sts128u(ou + ch0, make_uint4(hi[0], hi[1], hi[2], hi[3]));
            sts128u(ou + ch1, make_uint4(hi[4], hi[5], hi[6], hi[7]));
            sts128u(ou + SLOT_BYTES + ch0, make_uint4(lo[0], lo[1], lo[2], lo[3]));
            sts128u(ou + SLOT_BYTES + ch1, make_uint4(lo[4], lo[5], lo[6], lo[7]));
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&out_ready[ob]);
            if (++buf == 4) { buf = 0; acc_ph ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == EPI_W + 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}
static size_t conv5g_smem() { return 1024 + 4 * SLOT_BYTES + C5_B_BYTES + C5_STAGES * C5_STAGE_BYTES + 64 * 4 + 24 * 8 + 16; }

// guard positions of a G8 tensor (zeroed by the allocation): tap rows reach 2 rows + 2 positions before a tile, and the last
// tile's segments 2 rows + 136 positions past the end
__host__ __device__ inline long long g8_guard_lo(int W) { return 2LL * (W + 2 * PADB) + 2; }
__host__ __device__ inline long long g8_guard_hi(int W) { return 2LL * (W + 2 * PADB) + C5_SEG_POS + TILE; }

// fp32 channels-last [B,H,W,4] -> G8 (hi/lo split, replicate border)
__global__ void g8_from_nhwc4_kernel(const float4* __restrict__ x, uint4* __restrict__ g8, int B, int H, int W) {
    const int Hp = H + 2 * PADB, Wp = W + 2 * PADB;
    const long long total = (long long)B * Hp * Wp;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
        const int xp = (int)(q % Wp);
        const long long r = q / Wp;
        const int yp = (int)(r % Hp), b = (int)(r / Hp);
        const int xx = min(max(xp - PADB, 0), W - 1), yy = min(max(yp - PADB, 0), H - 1);
        const float4 v = __ldg(x + ((long long)b * H + yy) * W + xx);
        uint32_t h01, l01, h23, l23;
        split_bf16x2(v.x, v.y, h01, l01);
        split_bf16x2(v.z, v.w, h23, l23);
        g8[q] = make_uint4(h01, h23, l01, l23);
    }
}

// ---- U-Net 3x3 convolution (unet_block.py:250-259: Conv2d(k = 3, padding = 1, bias = False)) on the tensor core ---------
// NCHW fp32 in (batch stride in floats: concat buffers are read in place), NCHW fp32 out, Cin <= 64, up to 64 output
// channels per launch.  Implicit GEMM over the flat positions of the [H][W + 1] grid of one image (one dummy column per row:
// it is the zero padding to the right of a row AND to the left of the next one, so a horizontal tap is a plain +-1 offset):
//   loaders (two groups of 5 warps, one A stage each)  thread = staged position; per kernel row dy and group of 8 input
//       channels: 8 coalesced plane loads, hi/lo split, two 16-byte stores -> the UMMA no-swizzle K-major layout
//       [dy][chunk = 8 channels, hi chunks then lo chunks][position][16 B]; the three horizontal taps of a row are the
//       same segment at a 16-byte offset (as in conv5g_kernel);
//   MMA lane   per tap and pair of chunks (K = 16 channels): a_hi x [w_hi ; w_lo] (N = 2 Coutp: main | cross columns) and
//       a_lo x w_hi (N = Coutp, the first rows of the same weight block); weights are split and laid out at kernel start.
//       Operands are FP16 halves (kind::f16 with F16 formats): the E2EVN metric gate (SSIM / PSNR to 4 decimals) does not
//       survive the 2^-17 of a bf16 split, the 2^-22 of the fp16 split is at the level of the fp32 kernels;
//   4 epilogue warps   main + cross in RN fp32, coalesced NCHW stores (lane = position = consecutive x).
// fp32 pair -> packed fp16 hi pair + packed fp16 lo pair (x ~= hi + lo to ~2^-22: fp16 carries 11 significant bits, so
// the two halves keep 22 of fp32's 24; the bf16 split of the RIM kernels keeps 16).  Valid for O(1) operands -- here the
// instance-normalised activations and the weights of the U-Net; values below 2^-14 lose relative (not absolute) accuracy.
__device__ __forceinline__ void split_f16x2(float e0, float e1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(e0, e1);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(e0 - hf.x, e1 - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    // as make_idesc, with F16 (format 0) A and B operands
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
constexpr float U3_WSCALE = 256.f;           // power of two applied to the weights before the fp16 split
constexpr int U3_ROWS = 136;                 // staged positions per segment: 128 + 2 halo, whole core matrices
constexpr int U3_SEG = U3_ROWS * 16;
constexpr int U3_LOAD_W = 5;                 // warps per loader group
constexpr int U3_LOAD_G = 3;                 // loader groups: every tile is split three ways (one kernel row per group)
constexpr int U3_THREADS = (4 + U3_LOAD_G * U3_LOAD_W + 1) * 32;

struct UConvParams {
    const float* x;     // [N][Cin][H][W], batch stride xbs floats
    const void* wpack;  // this launch's packed weights (uconv3_pack_kernel)
    float* out;         // [N][Cout_total][H][W], batch stride obs floats
    long long xbs, obs;
    int N, Cin, H, W;
    int co_begin, co_count;  // output channels of this launch
    int cg, cgp;             // channel groups of 8 (real, padded to even)
    int coutp;               // co_count padded to 16
    int stages;              // 1 .. 4 A stages
    int nbuf;                // accumulator buffers of 6 coutp TMEM columns: 4 (coutp 16) or 2 (coutp 32)
    int tiles_per_img, n_tiles;
#ifdef MRB_TC_PROF
    int debug;               // role switches (tools build): 1 no global loads, 2 no MMAs, 4 no stores, 8 no split / staging stores
    unsigned long long* prof;  // [grid][16] cycle counters
#endif
};

template <int PAIRS>  // pairs of 8-channel groups: cgp = 2 * PAIRS (compile-time: the loader and issue loops unroll)
__global__ void __launch_bounds__(U3_THREADS, 1) uconv3_kernel(const UConvParams P) {
    constexpr int CGP = 2 * PAIRS;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int stage_bytes = 3 * 2 * CGP * U3_SEG;
    const int bchunk = 2 * P.coutp * 16;                       // one weight chunk: [main rows | cross rows][16 B]
    uint8_t* a_s = smem;                                       // [stages][dy][2 cgp chunks][U3_ROWS][16 B]
    uint8_t* w_s = a_s + (size_t)P.stages * stage_bytes;       // [tap][cgp][2 coutp rows][16 B]
    uint64_t* full = (uint64_t*)(w_s + (size_t)9 * CGP * bchunk);  // [4]
    uint64_t* empty = full + 4;                                // [4]
    uint64_t* acc_full = empty + 4;                            // [4]
    uint64_t* acc_empty = acc_full + 4;                        // [4]
    uint32_t* tmem_slot = (uint32_t*)(acc_empty + 4);

    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    T2P(const long long t_k0 = clock64();)
    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) {
            mbar_init(&full[i], U3_LOAD_G * U3_LOAD_W);
            mbar_init(&empty[i], 1);
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], 4);
        }
        fence_barrier_init();
    }
    // zero the A stages once (padding chunks and rows that no loader writes must be finite), then the weights
    for (int i = threadIdx.x; i < P.stages * stage_bytes / 16; i += U3_THREADS)
        reinterpret_cast<uint4*>(a_s)[i] = make_uint4(0u, 0u, 0u, 0u);
    {   // weights: packed once per parameter version by uconv3_pack_kernel, [tap][group][main rows | cross rows][16 B]
        const uint4* g = reinterpret_cast<const uint4*>(P.wpack);
        for (int i = threadIdx.x; i < 9 * CGP * 2 * P.coutp; i += U3_THREADS) reinterpret_cast<uint4*>(w_s)[i] = __ldg(g + i);
    }
    if (warp == 4 + U3_LOAD_G * U3_LOAD_W) tmem_alloc(tmem_slot, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    T2P(if (P.prof && threadIdx.x == 0) P.prof[blockIdx.x * 16 + 15] = clock64() - t_k0;)
    const int Wq = P.W + 1;
    const long long HW = (long long)P.H * P.W;
    const int npos = P.H * Wq;

    if (warp >= 4 && warp < 4 + U3_LOAD_G * U3_LOAD_W) {
        // ============================== LOADERS ==============================
        const int grp = (warp - 4) / U3_LOAD_W;
        const int r = (warp - 4 - grp * U3_LOAD_W) * 32 + lane;  // staged position (row of every segment)
        // Tile number `it` of this CTA lives in A stage it % stages.  The three loader groups split EVERY tile: group g stages
        // kernel row dy = g (all channel groups), so a tile costs each thread one global round trip per 32 channels and a third
        // of the conversion work, and a single-stage configuration (56 input channels) still has 15 warps loading.
        // The loads of the next tile are issued before the current one is converted (register ping-pong) when a step is at
        // most 16 channels; wider steps do not fit the register budget twice.
        const int dy = grp;
        const bool active = r < TILE + 2;
        constexpr int NG = CGP < 4 ? CGP : 4;   // channel groups per step
        constexpr int NB = CGP > 4 ? 2 : 1;     // steps per tile and group
        const int hw32 = (int)HW;
        T2P(long long t_l0 = clock64(), t_lw = 0, t_lld = 0, c0;)
        auto issue = [&](int it, int g0, float* v) {
            const int tile = blockIdx.x + it * gridDim.x;
            const int n = tile / P.tiles_per_img, p0 = (tile - n * P.tiles_per_img) * TILE;
            const int q = p0 - 1 + r + (dy - 1) * Wq;
            const int yq = q >= 0 ? q / Wq : 0, xq = q - yq * Wq;
            const bool ok = active && q >= 0 && q < npos && xq < P.W && !T2_DBG(P, 1);
            const float* src = P.x + (long long)n * P.xbs + (ok ? yq * P.W + xq : 0) + 8 * g0 * hw32;
            const int cleft = P.Cin - 8 * g0;
#pragma unroll
            for (int e = 0; e < 8 * NG; ++e) v[e] = (ok && e < cleft) ? __ldg(src + e * hw32) : 0.f;
        };
        auto convert = [&](int it, int g0, const float* v) {
            const int s = it % P.stages;
            uint8_t* st = a_s + (size_t)s * stage_bytes + r * 16 + (size_t)(dy * 2 * CGP + g0) * U3_SEG;
#pragma unroll
            for (int gg = 0; gg < NG; ++gg) {
                if (active && g0 + gg < P.cg && !T2_DBG(P, 8)) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) split_f16x2(v[8 * gg + 2 * e], v[8 * gg + 2 * e + 1], hi[e], lo[e]);
                    uint8_t* d = st + (size_t)gg * U3_SEG;
                    *reinterpret_cast<uint4*>(d) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(d + (size_t)CGP * U3_SEG) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
            }
        };
        auto acquire = [&](int it) {
            T2P(c0 = clock64();)
            mbar_wait_sleep(&empty[it % P.stages], ((uint32_t)(it / P.stages) & 1u) ^ 1u, 40);
            T2P(t_lw += clock64() - c0;)
        };
        auto publish = [&](int it) {
            fence_proxy_async();  // generic-proxy stores -> visible to the tensor core's operand reads
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[it % P.stages]);
        };
        const int my_tiles = (int)blockIdx.x < P.n_tiles ? (P.n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
        if (NB == 1 && NG <= 2) {
            float va[8 * NG], vb[8 * NG];
            if (my_tiles > 0) issue(0, 0, va);
            for (int it = 0; it < my_tiles; it += 2) {
                if (it + 1 < my_tiles) issue(it + 1, 0, vb);
                acquire(it);
                convert(it, 0, va);
                publish(it);
                if (it + 2 < my_tiles) issue(it + 2, 0, va);
                if (it + 1 < my_tiles) {
                    acquire(it + 1);
                    convert(it + 1, 0, vb);
                    publish(it + 1);
                }
            }
        } else {
            for (int it = 0; it < my_tiles; ++it) {
                float v[8 * NG];
                issue(it, 0, v);
                acquire(it);
                convert(it, 0, v);
                if (NB == 2) {
                    issue(it, 4, v);
                    convert(it, 4, v);
                }
                publish(it);
            }
        }
        T2P(t_lld = clock64() - t_l0 - t_lw;)
        T2P(if (P.prof && lane == 0 && (warp - 4) % U3_LOAD_W == 0) { unsigned long long* o = P.prof + blockIdx.x * 16 + 4 * (grp < 2 ? grp : 0); if (grp < 2) { o[0] = clock64() - t_l0; o[1] = t_lw; o[2] = t_lld; } })
    } else if (warp == 4 + U3_LOAD_G * U3_LOAD_W) {
        // ============================== MMA ISSUER ==============================
        const uint32_t tmem_u = uni(tmem_base);
        const uint64_t adesc0 = make_desc_ns(smem_u32(a_s), U3_SEG, 128);
        const uint64_t bdesc0 = make_desc_ns(smem_u32(w_s), (uint32_t)bchunk, 128);
        const uint32_t id2 = make_idesc_f16(TILE, 2 * P.coutp), id1 = make_idesc_f16(TILE, P.coutp);
        int it = 0;
        T2P(long long t_m0 = clock64(), t_mwa = 0, t_mwf = 0, c0;)
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int s = it % P.stages;
            const uint32_t ph = (uint32_t)(it / P.stages) & 1u;
            const int buf = it % P.nbuf;
            const uint32_t acc_ph = (uint32_t)(it / P.nbuf) & 1u;
            T2P(c0 = clock64();)
            mbar_wait(&acc_empty[buf], acc_ph ^ 1);
            T2P(t_mwa += clock64() - c0; c0 = clock64();)
            mbar_wait(&full[s], ph);
            T2P(t_mwf += clock64() - c0;)
            tc_fence_after();
            // accumulator buffer = three groups (one per kernel row) of [main coutp | cross coutp] columns: the tensor core's
            // fp32 accumulation truncates, so the error of a chain grows with its length -- the long hi*hi chain is cut into
            // three (3 * PAIRS accumulations each), the small cross terms (hi*lo, lo*hi) go to their own columns, and the
            // epilogue adds the six partial sums in RN fp32
            const uint32_t d0 = tmem_u + (uint32_t)(buf * 6 * P.coutp);
            const uint64_t a_s0 = adesc0 + (uint64_t)((s * stage_bytes) >> 4);
            const uint32_t bc16 = (uint32_t)(bchunk >> 4);
            if (!T2_DBG(P, 2)) {
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                    const int dy = t / 3, dx = t - dy * 3;
                    const uint64_t a_t = a_s0 + (uint64_t)((dy * 2 * CGP * U3_SEG + dx * 16) >> 4);
                    const uint32_t d = d0 + (uint32_t)(dy * 2 * P.coutp);
#pragma unroll
                    for (int j = 0; j < PAIRS; ++j) {
                        const uint64_t bj = bdesc0 + (uint64_t)((t * CGP + 2 * j) * bc16);
                        umma_ss(d, a_t + (uint64_t)((2 * j * U3_SEG) >> 4), bj, id2, (dx | j) != 0);
                        const uint64_t a_lo = a_t + (uint64_t)(((CGP + 2 * j) * U3_SEG) >> 4);
                        umma_ss(d + P.coutp, a_lo, bj, id1, 1);                                   // a_lo * w_hi
                        umma_ss(d + P.coutp, a_lo, bj + (uint64_t)((P.coutp * 16) >> 4), id1, 1);  // a_lo * w_lo: the issue lane
                        // has slack, so the fourth product is kept and the sum is exact to the 2^-22 of the operand split
                    }
                }
            }
            umma_commit(&empty[s]);
            umma_commit(&acc_full[buf]);
        }
        T2P(if (P.prof && lane == 0) { unsigned long long* o = P.prof + blockIdx.x * 16 + 8; o[0] = clock64() - t_m0; o[1] = t_mwa; o[2] = t_mwf; })
    } else if (warp < 4) {
        // ============================== EPILOGUE ==============================
        const int m = warp * 32 + lane;
        int it = 0;
        T2P(long long t_e0 = clock64(), t_ew = 0, c0;)
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int n = tile / P.tiles_per_img, p = (tile - n * P.tiles_per_img) * TILE + m;
            const int y = p / Wq, x = p - y * Wq;
            const bool ok = p < npos && x < P.W;
            float* o = P.out + (long long)n * P.obs + (long long)P.co_begin * HW + (long long)y * P.W + x;
            const int buf = it % P.nbuf;
            T2P(c0 = clock64();)
            mbar_wait_sleep(&acc_full[buf], (uint32_t)(it / P.nbuf) & 1u, 64);
            T2P(t_ew += clock64() - c0;)
            tc_fence_after();
            const uint32_t t0 = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * 6 * P.coutp);
            for (int c8 = 0; c8 < P.coutp; c8 += 8) {  // 8 channels per step: main + cross columns of the three row groups
                float m0[8], x0[8], m1[8], x1[8], m2[8], x2[8], dum[8];
                const uint32_t g0 = t0 + c8, g1 = g0 + 2 * P.coutp, g2 = g1 + 2 * P.coutp;
                tmem_ld8x4(g0, g0 + P.coutp, g1, g1 + P.coutp, m0, x0, m1, x1);
                tmem_ld8x4(g2, g2 + P.coutp, g2, g2 + P.coutp, m2, x2, dum, dum);
                if (ok && !T2_DBG(P, 4)) {
#pragma unroll
                    for (int e = 0; e < 8; ++e)
                        if (c8 + e < P.co_count)
                            o[(long long)(c8 + e) * HW] =
                                (((m0[e] + m1[e]) + m2[e]) + ((x0[e] + x1[e]) + x2[e])) * (1.f / U3_WSCALE);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
        T2P(if (P.prof && threadIdx.x == 0) { unsigned long long* o = P.prof + blockIdx.x * 16 + 12; o[0] = clock64() - t_e0; o[1] = t_ew; })
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4 + U3_LOAD_G * U3_LOAD_W) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// weights [Cout][Cin][3][3] fp32 -> the kernel's shared-memory image of one launch (output channels co_begin .. +co_count):
// [tap][group of 8 input channels][rows: coutp x w_hi | coutp x w_lo][8 fp16]
__global__ void uconv3_pack_kernel(const float* __restrict__ w, uint4* __restrict__ dst, int Cin, int cgp, int co_begin,
                                   int co_count, int coutp) {
    const int total = 9 * cgp * 2 * coutp;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int n = i % (2 * coutp), kc = i / (2 * coutp);
        const int g = kc % cgp, t = kc / cgp;
        const int co = n < coutp ? n : n - coutp;
        uint32_t hw[4] = {0u, 0u, 0u, 0u}, lw[4] = {0u, 0u, 0u, 0u};
        if (co < co_count) {
            const float* wp = w + ((long long)(co_begin + co) * Cin) * 9 + t;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int c0 = 8 * g + 2 * e, c1 = c0 + 1;
                const float v0 = c0 < Cin ? wp[(long long)c0 * 9] : 0.f, v1 = c1 < Cin ? wp[(long long)c1 * 9] : 0.f;
                // weights of a 3x3 conv are O(1/sqrt(9 Cin)): times 2^8 (exact) their lo halves leave fp16's subnormal range;
                // the epilogue multiplies the sums by 2^-8
                split_f16x2(v0 * U3_WSCALE, v1 * U3_WSCALE, hw[e], lw[e]);
            }
        }
        dst[i] = n < coutp ? make_uint4(hw[0], hw[1], hw[2], hw[3]) : make_uint4(lw[0], lw[1], lw[2], lw[3]);
    }
}
// launches of one convolution: output channels per launch and the byte offset of each launch's packed weights
struct UConvPlan {
    int cg, cgp, per_pass, n_pass;
};
static UConvPlan uconv3_plan(int Cin, int Cout) {
    UConvPlan pl;
    pl.cg = (Cin + 7) / 8;
    pl.cgp = pl.cg <= 2 ? 2 : pl.cg <= 4 ? 4 : 8;
    pl.per_pass = 32;  // <= 32 output channels per launch: three accumulator groups x [main | cross] x 2 buffers of TMEM
    pl.n_pass = (Cout + pl.per_pass - 1) / pl.per_pass;
    return pl;
}
static size_t uconv3_pass_bytes(const UConvPlan& pl, int co_count) {
    return (size_t)9 * pl.cgp * 2 * ((co_count + 15) & ~15) * 16;
}

#ifdef MRB_TC_PROF
int g_debug2 = 0;
unsigned long long* g_prof2 = nullptr;
#endif
static size_t gru2_smem() { return 1024 + 4 * W_CHUNK + NSLOT * SLOT_BYTES + 192 * 4 + 20 * 8 + 16; }

}  // namespace tc2
}  // namespace mrb

using namespace mrb;

extern "C" size_t mrb_bh_bytes(int B, int H, int W) {
    return (size_t)B * (size_t)(H + 2 * tc2::PADB) * (size_t)(W + 2 * tc2::PADB) * tc2::PX_BYTES;
}

extern "C" int mrb_bh_from_nhwc(const void* x, void* bh, int B, int H, int W, void* stream) {
    MRB_REQUIRE(x && bh && B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_bh_from_nhwc: bad argument");
    const long long total = (long long)B * (H + 2 * tc2::PADB) * (W + 2 * tc2::PADB) * 8;
    const int grid = (int)std::min<long long>((total + 255) / 256, 148 * 16);
    tc2::bh_from_nhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)x, (uint8_t*)bh, B, H, W);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_bh_to_nhwc(const void* bh, void* x, int B, int H, int W, void* stream) {
    MRB_REQUIRE(x && bh && B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_bh_to_nhwc: bad argument");
    const long long total = (long long)B * H * W * 8;
    const int grid = (int)std::min<long long>((total + 255) / 256, 148 * 16);
    tc2::bh_to_nhwc_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)bh, (float*)x, B, H, W);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" int mrb_bh_fix_border(void* bh, int B, int H, int W, void* stream) {
    MRB_REQUIRE(bh && B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_bh_fix_border: bad argument");
    const long long nb = (long long)(H + 2 * tc2::PADB) * (W + 2 * tc2::PADB) - (long long)H * W;
    const long long total = (long long)B * nb * 16;
    const int grid = (int)std::min<long long>((total + 255) / 256, 148 * 8);
    tc2::bh_fix_border_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((uint8_t*)bh, B, H, W);
    MRB_LAUNCHED();
    return MRB_OK;
}

extern "C" size_t mrb_tc2_gru_packed_bytes(void) { return (size_t)4 * tc2::W_CHUNK; }

extern "C" int mrb_tc2_pack_gru(const void* w_ih, const void* w_hh, void* dst, int ch, int cx, void* stream) {
    MRB_REQUIRE(w_ih && w_hh && dst, MRB_EINVAL, "mrb_tc2_pack_gru: null pointer");
    MRB_REQUIRE(ch == 64 && cx == 64, MRB_EUNSUPPORTED, "mrb_tc2_pack_gru: 64 input and hidden channels only");
    tc::PackDesc D{(const float*)w_ih, (const float*)w_hh, 1, ch, cx, 1, ch, 3 * ch, 2, 1};  // no channel split: 192 rows per chunk
    return tc::pack_launch(D, dst, (cudaStream_t)stream);
}

extern "C" int mrb_tc2_gru(const void* x_bh, const void* h_bh, const void* wpack, const void* b_ih, void* out_bh, int B, int H,
                           int W, void* stream) {
    MRB_REQUIRE(x_bh && h_bh && wpack && out_bh, MRB_EINVAL, "mrb_tc2_gru: null pointer");
    MRB_REQUIRE(out_bh != h_bh && out_bh != x_bh, MRB_EINVAL, "mrb_tc2_gru: the output must not alias an input");
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_tc2_gru: bad shape");
    tc2::Gru2Params P;
    P.wpack = wpack; P.bias = (const float*)b_ih;
    P.Q = (long long)B * (H + 2 * tc2::PADB) * (W + 2 * tc2::PADB);
    MRB_REQUIRE(P.Q < 2147483647LL - tc2::TILE, MRB_EUNSUPPORTED, "mrb_tc2_gru: too many pixels");
    P.n_tiles = (int)((P.Q + tc2::TILE - 1) / tc2::TILE);
#ifdef MRB_TC_PROF
    P.debug = tc2::g_debug2; P.prof = tc2::g_prof2;
    { int skip = (tc2::g_debug2 & 1) ? 1 : 0; cudaMemcpyToSymbol(tc2::g_skip_mma, &skip, sizeof(int)); }
#endif
    CUtensorMap tm_h, tm_x, tm_o;
    int rc = tc2::make_bh_tmap(&tm_h, h_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    rc = tc2::make_bh_tmap(&tm_x, x_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    rc = tc2::make_bh_tmap(&tm_o, out_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    static bool attr_set = false;
    const size_t smem = device_max_smem_optin();  // the full opt-in size: same carve-out as the other tensor-core kernels
    if (!attr_set) {
        MRB_REQUIRE(tc2::gru2_smem() <= smem, MRB_EUNSUPPORTED, "mrb_tc2_gru: shared memory");
        MRB_CUDA(cudaFuncSetAttribute(tc2::gru2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = device_sm_count();
    if (grid > P.n_tiles) grid = P.n_tiles;
    tc2::gru2_kernel<<<grid, tc2::THREADS2, smem, (cudaStream_t)stream>>>(tm_h, tm_x, tm_o, P);
    MRB_LAUNCHED();
    return MRB_OK;
}

/* G8: the RIM conv input [eta.re, eta.im, grad.re, grad.im] as 4 hi + 4 lo bf16 per position of the padded BH geometry,
 * with guard positions before and after; the buffer must be ZERO-INITIALISED once by the caller (the guards are only read) */
extern "C" size_t mrb_g8_bytes(int B, int H, int W) {
    const long long Q = (long long)B * (H + 2 * tc2::PADB) * (W + 2 * tc2::PADB);
    return (size_t)(Q + tc2::g8_guard_lo(W) + tc2::g8_guard_hi(W)) * 16;
}

extern "C" int mrb_g8_from_nhwc4(const void* x, void* g8, int B, int H, int W, void* stream) {
    MRB_REQUIRE(x && g8 && B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_g8_from_nhwc4: bad argument");
    const long long total = (long long)B * (H + 2 * tc2::PADB) * (W + 2 * tc2::PADB);
    const int grid = (int)std::min<long long>((total + 255) / 256, 148 * 16);
    tc2::g8_from_nhwc4_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float4*)x, (uint4*)g8 + tc2::g8_guard_lo(W), B, H, W);
    MRB_LAUNCHED();
    return MRB_OK;
}

/* ConvNonlinear 5x5, 4 -> 64 (conv_layers.py:36-123) from a G8 input to a BH output; w [64,4,5,5] fp32 (split on the fly),
 * bias [64] or null.  Every position of out_bh is written; its border is not a replicate copy. */
extern "C" int mrb_tc2_conv5x5x4(const void* g8, const void* w, const void* bias, void* out_bh, int B, int H, int W, int relu,
                                 void* stream) {
    MRB_REQUIRE(g8 && w && out_bh, MRB_EINVAL, "mrb_tc2_conv5x5x4: null pointer");
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_tc2_conv5x5x4: bad shape");
    tc2::Conv5Params P;
    P.g8 = (const uint8_t*)g8; P.w = (const float*)w; P.bias = (const float*)bias;
    P.Wp = W + 2 * tc2::PADB;
    P.Q = (long long)B * (H + 2 * tc2::PADB) * P.Wp;
    P.guard_lo = tc2::g8_guard_lo(W);
    MRB_REQUIRE(P.Q < 2147483647LL - tc2::TILE, MRB_EUNSUPPORTED, "mrb_tc2_conv5x5x4: too many pixels");
    P.n_tiles = (int)((P.Q + tc2::TILE - 1) / tc2::TILE);
    P.relu = relu;
    CUtensorMap tm_o;
    int rc = tc2::make_bh_tmap(&tm_o, out_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    static bool attr_set = false;
    const size_t smem = device_max_smem_optin();
    if (!attr_set) {
        MRB_REQUIRE(tc2::conv5g_smem() <= smem, MRB_EUNSUPPORTED, "mrb_tc2_conv5x5x4: shared memory");
        MRB_CUDA(cudaFuncSetAttribute(tc2::conv5g_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = device_sm_count();
    if (grid > P.n_tiles) grid = P.n_tiles;
    tc2::conv5g_kernel<<<grid, tc2::C5_THREADS, smem, (cudaStream_t)stream>>>(tm_o, P);
    MRB_LAUNCHED();
    return MRB_OK;
}

/* U-Net 3x3 conv (zero padding, no bias; unet_block.py:250-259) on the tensor core, NCHW fp32 in / out with batch strides in
 * floats (concat buffers are read and written in place).  Cin <= 64, any Cout (launches of up to 32 output channels).  Error-compensated fp16-split products (x = hi + lo to 2^-22; operands must be O(1): instance-normalised
 * activations).  wpack = mrb_tc2_unet_pack of the layer's weight. */
extern "C" size_t mrb_tc2_unet_packed_bytes(int Cin, int Cout) {
    if (Cin < 1 || Cin > 64 || Cout < 1) return 0;
    const tc2::UConvPlan pl = tc2::uconv3_plan(Cin, Cout);
    size_t tot = 0;
    for (int p = 0; p < pl.n_pass; ++p) tot += tc2::uconv3_pass_bytes(pl, std::min(pl.per_pass, Cout - p * pl.per_pass));
    return tot;
}

extern "C" int mrb_tc2_unet_pack(const void* w, void* dst, int Cin, int Cout, void* stream) {
    MRB_REQUIRE(w && dst, MRB_EINVAL, "mrb_tc2_unet_pack: null pointer");
    MRB_REQUIRE(Cin >= 1 && Cin <= 64 && Cout >= 1, MRB_EUNSUPPORTED, "mrb_tc2_unet_pack: 1 <= Cin <= 64 (got %d)", Cin);
    const tc2::UConvPlan pl = tc2::uconv3_plan(Cin, Cout);
    size_t off = 0;
    for (int p = 0; p < pl.n_pass; ++p) {
        const int cnt = std::min(pl.per_pass, Cout - p * pl.per_pass), coutp = (cnt + 15) & ~15;
        const int total = 9 * pl.cgp * 2 * coutp;
        tc2::uconv3_pack_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
            (const float*)w, (uint4*)((uint8_t*)dst + off), Cin, pl.cgp, p * pl.per_pass, cnt, coutp);
        MRB_LAUNCHED();
        off += tc2::uconv3_pass_bytes(pl, cnt);
    }
    return MRB_OK;
}

extern "C" int mrb_tc2_unet_conv3x3(const void* x, long long x_bstride, const void* wpack, void* out, long long out_bstride,
                                    int N, int Cin, int Cout, int H, int W, void* stream) {
    MRB_REQUIRE(x && wpack && out, MRB_EINVAL, "mrb_tc2_unet_conv3x3: null pointer");
    MRB_REQUIRE(N >= 1 && Cin >= 1 && Cout >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_tc2_unet_conv3x3: bad shape");
    MRB_REQUIRE(Cin <= 64, MRB_EUNSUPPORTED, "mrb_tc2_unet_conv3x3: at most 64 input channels (got %d)", Cin);
    MRB_REQUIRE((long long)H * W * 64 < 2147483647LL, MRB_EUNSUPPORTED, "mrb_tc2_unet_conv3x3: image too large");
    const tc2::UConvPlan pl = tc2::uconv3_plan(Cin, Cout);
    tc2::UConvParams P;
    P.x = (const float*)x; P.out = (float*)out;
    P.xbs = x_bstride; P.obs = out_bstride;
    P.N = N; P.Cin = Cin; P.H = H; P.W = W;
    P.cg = pl.cg;
    P.cgp = pl.cgp;
    const long long npos = (long long)H * (W + 1);
    P.tiles_per_img = (int)((npos + tc2::TILE - 1) / tc2::TILE);
    MRB_REQUIRE((long long)N * P.tiles_per_img < 2147483647LL && npos < 2147483647LL - 1024, MRB_EUNSUPPORTED,
                "mrb_tc2_unet_conv3x3: too many pixels");
    P.n_tiles = N * P.tiles_per_img;
    const size_t smem_max = device_max_smem_optin();
    static bool attr_set = false;
    if (!attr_set) {
        MRB_CUDA(cudaFuncSetAttribute(tc2::uconv3_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        MRB_CUDA(cudaFuncSetAttribute(tc2::uconv3_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        MRB_CUDA(cudaFuncSetAttribute(tc2::uconv3_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
        attr_set = true;
    }
#ifdef MRB_TC_PROF
    P.debug = tc2::g_debug2; P.prof = tc2::g_prof2;
#endif
    size_t off = 0;
    for (int p = 0; p < pl.n_pass; ++p) {
        P.co_begin = p * pl.per_pass;
        P.co_count = std::min(pl.per_pass, Cout - P.co_begin);
        P.coutp = (P.co_count + 15) & ~15;
        P.nbuf = P.coutp <= 16 ? 4 : 2;
        P.wpack = (const uint8_t*)wpack + off;
        off += tc2::uconv3_pass_bytes(pl, P.co_count);
        const size_t stage = (size_t)3 * 2 * P.cgp * tc2::U3_SEG, wb = (size_t)9 * P.cgp * 2 * P.coutp * 16;
        MRB_REQUIRE(1024 + stage + wb + 512 <= smem_max, MRB_EUNSUPPORTED, "mrb_tc2_unet_conv3x3: shared memory");
        P.stages = (int)std::min<size_t>(4, (smem_max - 1024 - wb - 512) / stage);
        int grid = device_sm_count();
        if (grid > P.n_tiles) grid = P.n_tiles;
        if (pl.cgp == 2) tc2::uconv3_kernel<1><<<grid, tc2::U3_THREADS, smem_max, (cudaStream_t)stream>>>(P);
        else if (pl.cgp == 4) tc2::uconv3_kernel<2><<<grid, tc2::U3_THREADS, smem_max, (cudaStream_t)stream>>>(P);
        else tc2::uconv3_kernel<4><<<grid, tc2::U3_THREADS, smem_max, (cudaStream_t)stream>>>(P);
        MRB_LAUNCHED();
    }
    return MRB_OK;
}

/* IndRNNCell, kernel size 1, 64 -> 64 (rnn_cells.py:264-391) on BH tensors: out = ReLU(W_ih x + b_ih + hh * h); wpack =
 * mrb_tc_pack_conv(ih.weight, 64, 64, 1); hh [64]; out must not alias x or h; pointwise over all positions like mrb_tc2_gru */
extern "C" int mrb_tc2_indrnn(const void* x_bh, const void* h_bh, const void* wpack, const void* b_ih, const void* hh,
                              void* out_bh, int B, int H, int W, void* stream) {
    MRB_REQUIRE(x_bh && h_bh && wpack && hh && out_bh, MRB_EINVAL, "mrb_tc2_indrnn: null pointer");
    MRB_REQUIRE(out_bh != h_bh && out_bh != x_bh, MRB_EINVAL, "mrb_tc2_indrnn: the output must not alias an input");
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_tc2_indrnn: bad shape");
    tc2::Ind2Params P;
    P.wpack = wpack; P.bias = (const float*)b_ih; P.hh = (const float*)hh;
    P.Q = (long long)B * (H + 2 * tc2::PADB) * (W + 2 * tc2::PADB);
    MRB_REQUIRE(P.Q < 2147483647LL - tc2::TILE, MRB_EUNSUPPORTED, "mrb_tc2_indrnn: too many pixels");
    P.n_tiles = (int)((P.Q + tc2::TILE - 1) / tc2::TILE);
    CUtensorMap tm_h, tm_x, tm_o;
    int rc = tc2::make_bh_tmap(&tm_h, h_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    rc = tc2::make_bh_tmap(&tm_x, x_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    rc = tc2::make_bh_tmap(&tm_o, out_bh, P.Q, tc2::TILE);
    if (rc) return rc;
    static bool attr_set = false;
    const size_t smem = device_max_smem_optin();
    if (!attr_set) {
        MRB_REQUIRE(tc2::ind2_smem() <= smem, MRB_EUNSUPPORTED, "mrb_tc2_indrnn: shared memory");
        MRB_CUDA(cudaFuncSetAttribute(tc2::ind2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = device_sm_count();
    if (grid > P.n_tiles) grid = P.n_tiles;
    tc2::ind2_kernel<<<grid, tc2::THREADS2, smem, (cudaStream_t)stream>>>(tm_h, tm_x, tm_o, P);
    MRB_LAUNCHED();
    return MRB_OK;
}

/* final RIM conv on the tensor core (fin2_kernel): same contract as mrb_conv_c2_bh_residual except that the BH border of
 * x_bh is never read (the replicate padding is applied to the tap coordinates) */
extern "C" int mrb_tc2_final_conv(const void* x_bh, const void* w, const void* bias, const void* eta, void* out, int B, int H,
                                  int W, void* stream) {
    MRB_REQUIRE(x_bh && w && eta && out, MRB_EINVAL, "mrb_tc2_final_conv: null pointer");
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "mrb_tc2_final_conv: bad shape");
    MRB_REQUIRE((long long)B * (H + 2 * tc2::PADB) < 2147483647LL, MRB_EUNSUPPORTED, "mrb_tc2_final_conv: too many rows");
    tc2::Fin2Params P;
    P.w = (const float*)w; P.bias = (const float*)bias; P.eta = (const float*)eta; P.out = (float*)out;
    P.B = B; P.H = H; P.W = W;
    P.py = (H + tc2::F2_OUT - 1) / tc2::F2_OUT;
    P.px = (W + tc2::F2_OUT - 1) / tc2::F2_OUT;
    const long long np = (long long)B * P.py * P.px;
    MRB_REQUIRE(np < 2147483647LL, MRB_EUNSUPPORTED, "mrb_tc2_final_conv: too many patches");
    P.n_patches = (int)np;
    CUtensorMap tm_h;
    int rc = tc2::make_bh_tmap3(&tm_h, x_bh, B, H, W);
    if (rc) return rc;
    static bool attr_set = false;
    const size_t smem = device_max_smem_optin();
    if (!attr_set) {
        MRB_REQUIRE(tc2::fin2_smem() <= smem, MRB_EUNSUPPORTED, "mrb_tc2_final_conv: shared memory");
        MRB_CUDA(cudaFuncSetAttribute(tc2::fin2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = device_sm_count();
    if (grid > P.n_patches) grid = P.n_patches;
    tc2::fin2_kernel<<<grid, tc2::F2_THREADS, smem, (cudaStream_t)stream>>>(tm_h, P);
    MRB_LAUNCHED();
    return MRB_OK;
}

#ifdef MRB_TC_PROF
extern "C" void mrb_tc2_set_debug(int flags) { tc2::g_debug2 = flags; }
extern "C" void mrb_tc2_set_prof(void* buf) { tc2::g_prof2 = (unsigned long long*)buf; }
#endif
