// Tensor-core (tcgen05 / TMEM) implicit-GEMM k x k convolution of the RIM regulariser on BH activations.
//
// Reference behaviour: ConvNonlinear (rim/conv_layers.py:36-123, replicate padding) with 64 input and 64 output channels,
// as used for the second convolution of RIMBlock's time loop (rim/rim_block.py:217-249).  Input and output are BH tensors
// (conv_tc2.cu: [B][H+4][W+4][64 hi bf16 | 64 lo bf16], replicate border of the input valid), so the replicate padding
// is the tensor's own border and a tap is a plain offset into the flat positions.
//
// Numerics: the reference is fp32 and the end-to-end tolerance (rel-L2 1e-4) rules out plain TF32 / BF16 operands
// (SURVEY section 7: 9.3e-4 / 9.9e-3).  Every product is therefore evaluated as an error-compensated split sum
//     a*b ~= a_hi*b_hi + a_hi*b_lo + a_lo*b_hi,    x_hi = rn_bf16(x), x_lo = rn_bf16(x - x_hi)
// on tcgen05.mma.kind::f16 (bf16 operands, fp32 accumulation in TMEM).  hi + lo carries 16-17 significant bits
// (|x - hi - lo| <= 2^-18 |x|), the dropped a_lo*b_lo term is <= 2^-18 relative: ~3e-6 rms per operator, 2.5e-5
// end to end over the 40 time steps of CIRIM 5x8 (measured with a CPU emulation of this arithmetic against the fp32
// oracle; the budget is 1e-4).
//
// Structure: one persistent CTA per SM, A and B operands from shared memory, TMEM holds accumulators only.
//   Work item = one or two consecutive 128-position tiles of the flat [B(H+4)(W+4)] grid (a pair may straddle two
//   slices), all 64 output channels.  Unit = (item, kernel row ky): for each tile of the item one 2-D TMA box per half
//   (hi, lo) of 136 positions x 128 B in SWIZZLE_128B (17 x 1024 B), starting `pad` positions before the tile's first
//   position of that kernel row.  Tap (ky, kx) of a tile is the same box read kx*dil rows further on: only the A
//   descriptor's start moves, by kx*dil*128 B (desc_rows).  Box rows outside the tensor are zero-filled by TMA; they only
//   feed border outputs.
//   TMA producer (1 lane)  per unit: the item's A boxes, then the unit's k weight chunks ([b_hi; b_lo], 16 KB, one bulk
//                 copy each, packed by mrb_tc_pack_conv);
//   MMA issuer (1 warp, elected lane)  per tap: the 8 MMAs of tile 0 then the 8 of tile 1 from the same weight chunk
//                 (each streamed chunk feeds both tiles), in the order of umma_segment_ss_stacked: taps row-major, k-steps
//                 0..3, a_hi x [b_hi; b_lo] (N = 128) into [main | cross] then a_lo x b_hi (N = 64) into cross.  A tile's
//                 accumulation order does not depend on whether it runs in a pair, so every output is bit-identical
//                 whatever the batch or the grid;
//   epilogue warps (8)  tcgen05.ld the accumulator (one position per thread, 2 warps per lane quadrant), RN add of main +
//                 cross, bias, optional ReLU, split into hi / lo bf16 and stage the tile in the TMA box layout;
//   TMA store lane  the two box stores of each tile.
//
// Rings (each mbarrier parity wait must be within one phase of the barrier: a ring is deeper than the distance its
// producer can run ahead of its slowest consumer, since the parity cannot tell phase it from phase it - 2):
//   A units     2 slots (4 boxes = 68 KB each).  One producer and one consumer walk the same unit sequence; the producer
//               refills a slot after the issuer's commit of the unit two before (a_empty), the issuer waits a_full: the
//               producer is 0..2 units ahead, never 3.
//   weights     3 slots of 16 KB, same protocol per tap (b_full / b_empty).  The producer's order A(u), W(u, 0..k-1),
//               A(u+1) cannot deadlock: the A(u+2) wait needs only unit u's MMAs, whose chunks were issued before A(u+1).
//   accumulators 4 TMEM buffers of 128 columns [main 64 | cross 64] (all 512 columns); tile s of the CTA uses buffer
//               s % 4.  The issuer waits acc_empty (8 epilogue arrivals) of tile s - 4 before the first MMA of tile s,
//               an item takes at most 2 buffers, and every epilogue warp walks the tiles in order.
//   output tile 1 slot (hi box | lo box).  An epilogue warp writes tile s after out_free of tile s - 1 (store lane) and
//               cannot pass tile s + 1 before all 8 warps have arrived on out_ready for tile s.
// Nothing reads a TMA-landed slot through the generic proxy (the MMAs release A and B slots with tcgen05.commit), so no
// proxy fence is needed there; the epilogue's generic writes of the output tile are fenced before out_ready.
//
// Shared memory: 2 x 68 KB A + 3 x 16 KB weights + 32 KB output tile + barriers and bias = 216.5 KB (+ 1 KB alignment).
//
// Work dealing: all CTAs take pairs for as many rounds as every CTA completes, then the rem < 2 * grid remaining tiles
// are dealt so that no CTA runs a pair while another idles: rem - grid CTAs take a pair, the others one tile each.
#include <cuda.h>

#include "tc_ptx.cuh"

namespace mrb {
namespace tc {

constexpr int TILE_M = 128;
constexpr int COUT = 64;                      // output channels (all of them in one CTA)
constexpr int KCH = 64;                       // channels per K chunk (one 128-byte row of bf16 in the B operand)
constexpr int EPI_WARPS = 8;                  // 2 warps per TMEM lane quadrant (each takes half of the channels)
constexpr int PRODUCER_WARP = EPI_WARPS, MMA_WARP = EPI_WARPS + 1, STORE_WARP = EPI_WARPS + 2;
constexpr int THREADS = (EPI_WARPS + 3) * 32;
constexpr int MAX_SEGS = 25;
constexpr int W_CHUNK_BYTES = COUT * 128;     // hi (or lo) rows of one weight chunk
constexpr int B_STAGES = 3;                   // streamed-weights ring
constexpr int A_UNITS = 2;                    // A ring: (item, kernel row) units
constexpr int A_BOX_ROWS = 136;               // 128 + 2 * pad, rounded up to whole 8-row swizzle atoms
constexpr int A_BOX_BYTES = A_BOX_ROWS * 128; // 17 x 1024: every box stays 1024-aligned
constexpr int A_UNIT_BYTES = 4 * A_BOX_BYTES; // [tile 0 hi | tile 0 lo | tile 1 hi | tile 1 lo]
constexpr int ACC_BUFS = 4;
constexpr int ACC_COLS = 2 * COUT;            // [main | cross]
constexpr int BH_PAD = 2;                     // replicate border of the BH activation layout (conv_tc2.cu)
constexpr int OUT_BOX_BYTES = TILE_M * 128;   // one [128 positions x 64 bf16] TMA box
constexpr int BAR_BYTES = 256;
constexpr size_t SMEM_BYTES = 1024 + (size_t)A_UNITS * A_UNIT_BYTES + (size_t)B_STAGES * 2 * W_CHUNK_BYTES +
                              2 * OUT_BOX_BYTES + BAR_BYTES + COUT * sizeof(float);

// Profiling hooks (per-role cycle counters, role switches) exist only in the tools build (-DMRB_TC_PROF,
// tools/libmridc_b200_tools.so); the product kernel carries none of them.
#ifdef MRB_TC_PROF
#define TCP(...) __VA_ARGS__
#define TC_DBG(P, flag) (((P).debug & (flag)) != 0)
#else
#define TCP(...)
#define TC_DBG(P, flag) false
#endif

struct Params {
    const void* wpack;       // packed bf16 weights: [tap][hi|lo][64 rows x 128 B swizzled]
    const float* bias;       // [64] (may be null)
    int n_tiles;             // 128-position tiles over the B (H+4)(W+4) flat positions
    int pitch;               // W + 4
    int ksz, dil;            // conv geometry
    int relu;
#ifdef MRB_TC_PROF
    unsigned long long* prof; // optional [gridDim.x][16] cycle counters (tools/tc_roles.py)
    int debug;                // role switches: 1 skip MMAs, 2 skip TMA / bulk loads, 4 skip epilogue math
#endif
};

// The items of this CTA (see the header): item i covers tiles [t0, t0 + count); count 0 past the last one.
struct Deal {
    int rounds, base, n2, n_tiles;
    __device__ explicit Deal(int nt) : n_tiles(nt) {
        rounds = nt / (2 * (int)gridDim.x);
        base = 2 * (int)gridDim.x * rounds;
        n2 = max(0, nt - base - (int)gridDim.x);
    }
    __device__ int item(int i, int& t0) const {
        const int c = blockIdx.x;
        if (i < rounds) { t0 = 2 * (c + (int)gridDim.x * i); return 2; }
        if (i > rounds) return 0;
        if (c < n2) { t0 = base + 2 * c; return 2; }
        t0 = base + n2 + c;  // base + 2 n2 + (c - n2)
        return t0 < n_tiles ? 1 : 0;
    }
};

__global__ void __launch_bounds__(THREADS, 1)
tc_kernel(const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out, const Params P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* a_s = smem;                                             // [A_UNITS][A_UNIT_BYTES]
    uint8_t* w_s = a_s + (size_t)A_UNITS * A_UNIT_BYTES;             // [B_STAGES][hi rows | lo rows]
    uint8_t* out_s = w_s + (size_t)B_STAGES * 2 * W_CHUNK_BYTES;     // [hi box | lo box] output tile
    uint64_t* a_full = (uint64_t*)(out_s + 2 * OUT_BOX_BYTES);       // [A_UNITS]
    uint64_t* a_empty = a_full + A_UNITS;                            // [A_UNITS] tcgen05.commit of the unit's MMAs
    uint64_t* b_full = a_empty + A_UNITS;                            // [B_STAGES]
    uint64_t* b_empty = b_full + B_STAGES;                           // [B_STAGES] tcgen05.commit of the tap's MMAs
    uint64_t* acc_full = b_empty + B_STAGES;                         // [ACC_BUFS]
    uint64_t* acc_empty = acc_full + ACC_BUFS;                       // [ACC_BUFS] one arrival per epilogue warp
    uint64_t* out_ready = acc_empty + ACC_BUFS;                      // every epilogue warp has written its part of the tile
    uint64_t* out_free = out_ready + 1;                              // the TMA stores of the previous tile have read out_s
    uint32_t* tmem_slot = (uint32_t*)(out_free + 1);
    float* bias_s = (float*)(out_s + 2 * OUT_BOX_BYTES + BAR_BYTES); // [COUT] (16-byte aligned): bias staged once per CTA

    // warp index through a shuffle: provably warp-uniform for the compiler (role branches and the MMA issuer's operands
    // then live in uniform registers)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const Deal deal(P.n_tiles);

    if (threadIdx.x == 0) {
        for (int i = 0; i < A_UNITS; ++i) {
            mbar_init(&a_full[i], 1);   // the producer's arrive.expect_tx; the TMA boxes complete the transaction bytes
            mbar_init(&a_empty[i], 1);
        }
        for (int i = 0; i < B_STAGES; ++i) {
            mbar_init(&b_full[i], 1);
            mbar_init(&b_empty[i], 1);
        }
        for (int i = 0; i < ACC_BUFS; ++i) {
            mbar_init(&acc_full[i], 1);
            mbar_init(&acc_empty[i], EPI_WARPS);
        }
        mbar_init(out_ready, EPI_WARPS);
        mbar_init(out_free, 1);
        fence_barrier_init();
    }
    for (int i = threadIdx.x; i < COUT; i += THREADS) bias_s[i] = P.bias ? P.bias[i] : 0.f;
    if (warp == MMA_WARP) tmem_alloc(tmem_slot, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int k = P.ksz, dil = P.dil, pad = dil * (k - 1) / 2;

    if (warp == PRODUCER_WARP) {
        // ============================== TMA PRODUCER ==============================
        if (lane == 0) {
            TCP(long long t_start = clock64(), t_wa = 0, t_wb = 0, c0;)
            const bool ld_on = !TC_DBG(P, 2);
            const uint8_t* wpack = reinterpret_cast<const uint8_t*>(P.wpack);
            int u = 0, bs = 0;
            uint32_t uph = 0, bph = 0;
            int t0;
            for (int i = 0, cnt; (cnt = deal.item(i, t0)) > 0; ++i) {
                for (int ky = 0; ky < k; ++ky) {
                    TCP(c0 = clock64();)
                    mbar_wait_sleep(&a_empty[u], uph ^ 1, 64);
                    TCP(t_wa += clock64() - c0;)
                    // first position of the box: kernel row ky of the tile's first position, pad positions to the left
                    const int q_off = (ky * dil - pad) * P.pitch - pad;
                    const uint32_t dst = smem_u32(a_s + (size_t)u * A_UNIT_BYTES), bar = smem_u32(&a_full[u]);
                    if (ld_on) {
                        mbar_expect_tx(&a_full[u], (uint32_t)(cnt * 2 * A_BOX_BYTES));
                        for (int j = 0; j < cnt; ++j) {
                            const int q0 = (t0 + j) * TILE_M + q_off;
                            tma_load_2d(dst + (uint32_t)(2 * j * A_BOX_BYTES), &tm_in, 0, q0, bar);
                            tma_load_2d(dst + (uint32_t)((2 * j + 1) * A_BOX_BYTES), &tm_in, 64, q0, bar);
                        }
                    } else {
                        mbar_arrive(&a_full[u]);
                    }
                    if (++u == A_UNITS) { u = 0; uph ^= 1; }
                    for (int kx = 0; kx < k; ++kx) {
                        TCP(c0 = clock64();)
                        mbar_wait_sleep(&b_empty[bs], bph ^ 1, 64);
                        TCP(t_wb += clock64() - c0;)
                        if (ld_on) {
                            mbar_expect_tx(&b_full[bs], (uint32_t)(2 * W_CHUNK_BYTES));
                            bulk_load_1d(smem_u32(w_s + (size_t)bs * 2 * W_CHUNK_BYTES),
                                         wpack + (size_t)(ky * k + kx) * 2 * W_CHUNK_BYTES, (uint32_t)(2 * W_CHUNK_BYTES),
                                         smem_u32(&b_full[bs]));
                        } else {
                            mbar_arrive(&b_full[bs]);
                        }
                        if (++bs == B_STAGES) { bs = 0; bph ^= 1; }
                    }
                }
            }
#ifdef MRB_TC_PROF
            if (P.prof) {
                unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
                o[0] = clock64() - t_start; o[1] = t_wa; o[2] = t_wb;
            }
#endif
        }
    } else if (warp == MMA_WARP) {
        // ============================== MMA ISSUER ==============================
        // Whole warp, warp-uniform control flow, one elected lane per tcgen05 instruction (see umma_commit).
        TCP(const bool prof = P.prof != nullptr;)
        TCP(long long t_start = clock64(), t_wa = 0, t_wb = 0, t_wacc = 0, t_mma = 0, t_commit = 0, c0 = 0;)
        const uint32_t tmem_u = uni(tmem_base);
        // loop-invariant operands: only the unit slot, the tap row and the weight slot move
        const uint64_t adesc0 = make_desc(smem_u32(a_s)), bdesc0 = make_desc(smem_u32(w_s));
        constexpr uint32_t idesc_n = make_idesc(TILE_M, COUT), idesc_2n = make_idesc(TILE_M, 2 * COUT);
        constexpr uint32_t BOX16 = A_BOX_BYTES >> 4;  // descriptor units
        int u = 0, bs = 0, seq = 0;  // seq: tiles of this CTA so far (accumulator buffer seq % 4)
        uint32_t uph = 0, bph = 0;
        int t0;
        for (int i = 0, cnt; (cnt = deal.item(i, t0)) > 0; ++i) {
            TCP(if (prof) c0 = clock64();)
            for (int j = 0; j < cnt; ++j) mbar_wait(&acc_empty[(seq + j) & 3], (((uint32_t)(seq + j) >> 2) & 1u) ^ 1u);
            TCP(if (prof) t_wacc += clock64() - c0;)
            tc_fence_after();
            const uint32_t d0 = tmem_u + (uint32_t)((seq & 3) * ACC_COLS), d1 = tmem_u + (uint32_t)(((seq + 1) & 3) * ACC_COLS);
            for (int ky = 0; ky < k; ++ky) {
                const uint64_t au = adesc0 + (uint64_t)((u * A_UNIT_BYTES) >> 4);
                TCP(if (prof) c0 = clock64();)
                mbar_wait(&a_full[u], uph);
                TCP(if (prof) t_wa += clock64() - c0;)
                for (int kx = 0; kx < k; ++kx) {
                    const uint64_t a = desc_rows(au, (uint32_t)(kx * dil));
                    const uint64_t b = bdesc0 + (uint64_t)((bs * 2 * W_CHUNK_BYTES) >> 4);
                    const uint32_t acc = (ky | kx) != 0;  // the first MMA of a tile overwrites [main | cross]
                    TCP(if (prof) c0 = clock64();)
                    mbar_wait(&b_full[bs], bph);
                    TCP(if (prof) { t_wb += clock64() - c0; c0 = clock64(); })
                    tc_fence_after();
                    if (!TC_DBG(P, 1)) {
                        umma_segment_ss_stacked(d0, d0 + COUT, a, a + BOX16, b, idesc_2n, idesc_n, acc);
                        if (cnt == 2) umma_segment_ss_stacked(d1, d1 + COUT, a + 2 * BOX16, a + 3 * BOX16, b, idesc_2n, idesc_n, acc);
                    }
                    TCP(if (prof) { t_mma += clock64() - c0; c0 = clock64(); })
                    umma_commit(&b_empty[bs]);  // the chunk is reusable once both tiles' MMAs have read it
                    TCP(if (prof) t_commit += clock64() - c0;)
                    if (++bs == B_STAGES) { bs = 0; bph ^= 1u; }
                }
                umma_commit(&a_empty[u]);
                if (++u == A_UNITS) { u = 0; uph ^= 1u; }
            }
            for (int j = 0; j < cnt; ++j) umma_commit(&acc_full[(seq + j) & 3]);
            seq += cnt;
        }
#ifdef MRB_TC_PROF
        if (prof && lane == 0) {
            unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
            o[4] = clock64() - t_start; o[5] = t_wa; o[6] = t_wacc; o[7] = t_mma; o[10] = t_commit; o[11] = t_wb;
        }
#endif
    } else if (warp == STORE_WARP) {
        // ============================== TMA STORE LANE ==============================
        if (lane == 0) {
            TCP(long long t_start = clock64(), t_w = 0, c0;)
            const uint32_t out_u32 = smem_u32(out_s);
            uint32_t oph = 0;
            int t0;
            for (int i = 0, cnt; (cnt = deal.item(i, t0)) > 0; ++i) {
                for (int j = 0; j < cnt; ++j) {
                    TCP(c0 = clock64();)
                    mbar_wait_sleep(out_ready, oph, 64);
                    TCP(t_w += clock64() - c0;)
                    tma_store_2d(&tm_out, out_u32, 0, (t0 + j) * TILE_M);
                    tma_store_2d(&tm_out, out_u32 + OUT_BOX_BYTES, 64, (t0 + j) * TILE_M);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                    mbar_arrive(out_free);
                    oph ^= 1;
                }
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before the CTA exits
#ifdef MRB_TC_PROF
            if (P.prof) {
                unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
                o[12] = clock64() - t_start; o[13] = t_w;
            }
#endif
        }
    } else {
        // ============================== EPILOGUE ==============================
        const int quad = warp & 3;             // TMEM lane quadrant this warp may access
        const int chalf = warp >> 2;           // which half of the channels the warp handles
        const int m = quad * 32 + lane;        // TMEM lane = position row of the tile
        const int j_lo = chalf * (COUT / 2);
        const uint32_t bias_u32 = smem_u32(bias_s);
        const uint32_t out_u32 = smem_u32(out_s);
        uint32_t oph = 0;
        // 8 consecutive channels (chunk c8 = channel / 8) of this thread's position -> hi / lo bf16 in the output tile
        auto emit8 = [&](int c8, const float* v) {
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) split_bf16x2(v[2 * i], v[2 * i + 1], hi[i], lo[i]);
            sts128u(out_u32 + swz(m, c8), make_uint4(hi[0], hi[1], hi[2], hi[3]));
            sts128u(out_u32 + OUT_BOX_BYTES + swz(m, c8), make_uint4(lo[0], lo[1], lo[2], lo[3]));
        };
        TCP(long long e_start = clock64(), e_wait = 0;)
        int n_mine = 0, t0;
        for (int i = 0, cnt; (cnt = deal.item(i, t0)) > 0; ++i) n_mine += cnt;
        for (int seq = 0; seq < n_mine; ++seq) {
            const int buf = seq & 3;
            const uint32_t acc_phase = ((uint32_t)seq >> 2) & 1u;
            const uint32_t t0m = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * ACC_COLS);
            bool released = false;
            TCP(long long c0 = clock64();)
            mbar_wait_sleep(&acc_full[buf], acc_phase, 64);
            TCP(e_wait += clock64() - c0;)
            tc_fence_after();
            if (!TC_DBG(P, 4)) {
                // accumulator [main | cross]: all 32 channels of this thread with two batched loads, the buffer goes back
                // to the MMA issuer before any arithmetic
                float o[32];
#pragma unroll
                for (int jb = 0; jb < 2; ++jb) {
                    const int j = j_lo + jb * 16;
                    float a[8], a2[8], b1[8], b2[8];
                    tmem_ld8x4(t0m + j, t0m + 64 + j, t0m + j + 8, t0m + 64 + j + 8, a, a2, b1, b2);
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        o[jb * 16 + q] = a[q] + a2[q];
                        o[jb * 16 + 8 + q] = b1[q] + b2[q];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);
                released = true;
                mbar_wait_sleep(out_free, oph ^ 1, 32);  // the previous tile's stores have read the output tile
#pragma unroll
                for (int jb = 0; jb < 4; ++jb) {
                    const float4 b0 = lds128(bias_u32 + 4u * (uint32_t)(j_lo + jb * 8));
                    const float4 b1 = lds128(bias_u32 + 4u * (uint32_t)(j_lo + jb * 8 + 4));
                    float v[8] = {o[jb * 8 + 0] + b0.x, o[jb * 8 + 1] + b0.y, o[jb * 8 + 2] + b0.z, o[jb * 8 + 3] + b0.w,
                                  o[jb * 8 + 4] + b1.x, o[jb * 8 + 5] + b1.y, o[jb * 8 + 6] + b1.z, o[jb * 8 + 7] + b1.w};
                    if (P.relu) {
#pragma unroll
                        for (int q = 0; q < 8; ++q) v[q] = fmaxf(v[q], 0.f);
                    }
                    emit8(j_lo / 8 + jb, v);
                }
            }
            if (!released) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[buf]);
                mbar_wait_sleep(out_free, oph ^ 1, 32);
            }
            // the tile's [128 positions x (64 hi | 64 lo)] boxes are complete once all eight epilogue warps have
            // arrived; the TMA store lane takes it from there
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(out_ready);
            oph ^= 1;
        }
#ifdef MRB_TC_PROF
        if (P.prof && threadIdx.x == 0) {
            unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
            o[8] = clock64() - e_start; o[9] = e_wait;
        }
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ---- weight packing ----------------------------------------------------------------------------------
// dst chunk layout: [rows x 128 B] SWIZZLE_128B (64 bf16 K elements per row), hi rows then lo rows.  Source value for
// (half, chunk, row n, col k) is given by a small descriptor evaluated on the device.
__global__ void pack_weights_kernel(PackDesc D, uint16_t* dst) {
    const int total = D.n_split * D.n_chunks * D.rows * KCH;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
        int k = t % KCH;
        int r = (t / KCH) % D.rows;
        int ch = (t / (KCH * D.rows)) % D.n_chunks;
        int half = t / (KCH * D.rows * D.n_chunks);
        float v = 0.f;
        if (D.mode == 0) {
            const int tap = ch;
            const int co = half * D.nhalf + r, ci = k;
            if (co < D.cout && ci < D.cin) v = D.w[((long long)co * D.cin + ci) * D.ksz * D.ksz + tap];
        } else {
            // chunk 0: w_hh with rows [n ; r ; z] of this half (accumulator columns [0, 3*nhalf));
            // chunk 1: w_ih with rows [r ; z ; n] (columns [nhalf, 4*nhalf)): the r and z columns are shared
            const int Ch = D.cout;
            const int blk = r / D.nhalf, j = r % D.nhalf;
            const bool is_hh = ch == 0;
            const int g = is_hh ? ((blk + 2) % 3) : blk;  // hh order n,r,z -> gate index 2,0,1
            const int row = g * Ch + half * D.nhalf + j;
            const float* w = is_hh ? D.w2 : D.w;
            v = w[(long long)row * D.cin + k];
        }
        const uint16_t hi = bf16_rn_bits(v);
        const float hif = __uint_as_float((uint32_t)hi << 16);
        const uint16_t lo = bf16_rn_bits(v - hif);
        const size_t chunk_elems = (size_t)D.rows * KCH;
        uint16_t* base = dst + ((size_t)half * D.n_chunks + ch) * 2 * chunk_elems;
        const uint32_t off = (uint32_t)(r * 128 + (((k >> 3) ^ (r & 7)) << 4) + (k & 7) * 2);
        base[off / 2] = hi;
        base[chunk_elems + off / 2] = lo;
    }
}

int pack_launch(const PackDesc& D, void* dst, cudaStream_t st) {
    pack_weights_kernel<<<64, 256, 0, st>>>(D, (uint16_t*)dst);
    MRB_LAUNCHED();
    return MRB_OK;
}

#ifdef MRB_TC_PROF
static int g_debug = 0;
static unsigned long long* g_prof = nullptr;
#endif

static int launch(Params& P, const void* src, void* out, long long n_pos, cudaStream_t st) {
#ifdef MRB_TC_PROF
    P.debug = g_debug;
    P.prof = g_prof;
#endif
    const size_t max_smem = device_max_smem_optin();
    MRB_REQUIRE(SMEM_BYTES <= max_smem, MRB_EUNSUPPORTED, "tensor-core conv: %zu bytes of shared memory needed, %zu available",
                SMEM_BYTES, max_smem);
    // every TMA coordinate (a box starts up to pad rows and pad positions before its tile) must fit an int
    MRB_REQUIRE(n_pos + (long long)BH_PAD * (P.pitch + 1) + 2 * TILE_M < 2147483647LL, MRB_EUNSUPPORTED,
                "tensor-core conv: too many pixels");
    MRB_REQUIRE(P.ksz * P.ksz <= MAX_SEGS && P.dil * (P.ksz - 1) / 2 <= BH_PAD, MRB_EUNSUPPORTED,
                "tensor-core conv: bad geometry");
    CUtensorMap tm_in, tm_out;
    memset(&tm_in, 0, sizeof(tm_in));
    memset(&tm_out, 0, sizeof(tm_out));
    int rc = tc2::make_bh_tmap(&tm_in, src, n_pos, A_BOX_ROWS);
    if (rc) return rc;
    rc = tc2::make_bh_tmap(&tm_out, out, n_pos, TILE_M);
    if (rc) return rc;
    static bool attr_set = false;  // per-process, not per launch (the attribute calls are not free)
    if (!attr_set) {
        MRB_CUDA(cudaFuncSetAttribute(tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_smem));
        attr_set = true;
    }
    int grid = device_sm_count();
    if (grid > P.n_tiles) grid = P.n_tiles;
    // Every launch asks for the full opt-in shared memory (one CTA per SM anyway): all tensor-core kernels of the time
    // step then run with the same shared-memory carve-out.  Alternating this kernel between a ~195 KB and a ~227 KB
    // configuration (two different carve-outs) produced sporadic "Warp Illegal Instruction" traps in the weight streamer
    // and hangs on the B200; same-size sequences never failed.
    tc_kernel<<<grid, THREADS, max_smem, st>>>(tm_in, tm_out, P);
    MRB_LAUNCHED();
    return MRB_OK;
}

}  // namespace tc
}  // namespace mrb

using namespace mrb;

#ifdef MRB_TC_PROF
extern "C" void mrb_tc_set_debug(int flags) { tc::g_debug = flags; }
extern "C" void mrb_tc_set_prof(void* buf) { tc::g_prof = (unsigned long long*)buf; }
#endif

extern "C" size_t mrb_tc_packed_floats(int kind, int cout, int cin, int k) {
    // kind 0: conv k x k (cin == 64); no other kind is packed here (0 is returned).
    // Size of the packed bf16 hi/lo image, in 4-byte units (one chunk = 2 x rows x 128 B = 2 * rows * 32 floats).
    (void)cin;
    if (kind == 0) return (size_t)(k * k) * 2 * cout * 32;
    return 0;
}

extern "C" int mrb_tc_pack_conv(const void* w, void* dst, int cout, int cin, int k, void* stream) {
    MRB_REQUIRE(w && dst, MRB_EINVAL, "mrb_tc_pack_conv: null pointer");
    MRB_REQUIRE(cin == 64 && (cout % 32) == 0 && cout >= 32 && cout <= 128 && (k % 2) == 1 && k * k <= tc::MAX_SEGS,
                MRB_EUNSUPPORTED, "mrb_tc_pack_conv: need cin == 64, cout multiple of 32, k*k <= %d", tc::MAX_SEGS);
    tc::PackDesc D{(const float*)w, nullptr, 0, cout, cin, k, cout, cout, k * k, 1};
    tc::pack_weights_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(D, (uint16_t*)dst);
    MRB_LAUNCHED();
    return MRB_OK;
}

// ConvNonlinear k x k (dilated, replicate padding), 64 -> 64 channels, bias + optional ReLU, on BH tensors (conv_tc2.cu):
// x_bh with a valid replicate border (mrb_bh_fix_border), out_bh written at all (H+4)(W+4) positions (interior = the conv
// output; its border is not a replicate copy).
extern "C" int mrb_tc_conv_bh(const void* x_bh, const void* wpack, const void* bias, void* out_bh, int B, int H, int W, int cout,
                              int k, int dil, int relu, void* stream) {
    MRB_REQUIRE(x_bh && wpack && out_bh, MRB_EINVAL, "mrb_tc_conv_bh: null pointer");
    MRB_REQUIRE(cout == 64, MRB_EUNSUPPORTED, "mrb_tc_conv_bh: 64 output channels only");
    MRB_REQUIRE((k % 2) == 1 && k * k <= tc::MAX_SEGS && dil >= 1, MRB_EUNSUPPORTED, "mrb_tc_conv_bh: unsupported geometry");
    MRB_REQUIRE(dil * (k - 1) / 2 <= tc::BH_PAD, MRB_EUNSUPPORTED, "mrb_tc_conv_bh: the receptive field exceeds the BH border");
    MRB_REQUIRE(B >= 1 && H >= 1 && W >= 1, MRB_EINVAL, "tensor-core conv: bad shape");
    const long long n_pos = (long long)B * (H + 2 * tc::BH_PAD) * (W + 2 * tc::BH_PAD);
    long long nt = (n_pos + tc::TILE_M - 1) / tc::TILE_M;
    MRB_REQUIRE(nt <= 2147483647LL, MRB_EUNSUPPORTED, "tensor-core conv: too many pixels");
    tc::Params P;
    memset(&P, 0, sizeof(P));
    P.n_tiles = (int)nt;
    P.pitch = W + 2 * tc::BH_PAD;
    // One segment per tap (64 input channels = one 128-byte bf16 row of B), stacked MMAs of N = 128 and 64 (half the MMA
    // instructions of a channel split).  The k*k weight chunks (2*64*128 B each: hi rows | lo rows) are streamed from L2
    // through a small ring -- resident they would leave no room for the A boxes; each streamed chunk feeds two tiles.
    P.wpack = wpack; P.bias = (const float*)bias;
    P.relu = relu;
    P.ksz = k; P.dil = dil;
    return tc::launch(P, x_bh, out_bh, n_pos, (cudaStream_t)stream);
}
