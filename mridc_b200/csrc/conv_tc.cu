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
// oracle; the budget is 1e-4).  Round 1 used 3xTF32 (22 bits, 2.6e-6 end to end): same three MMAs per product but
// at half the tensor-pipe rate and twice the instruction count (K = 8 instead of 16 per MMA) -- the kernels were
// bound by exactly those two.
//
// Structure: one persistent CTA per SM.  Work item = one 128-position tile, all 64 output channels.  Segment = one tap
// (64 input channels = one K chunk of 64 bf16).
//   * B operand = the weights of one tap (hi rows | lo rows, pre-packed in the UMMA K-major SWIZZLE_128B layout by
//     mrb_tc_pack_conv), streamed from L2 through a small ring of shared-memory slots by the weight-streaming lane.
//   * A operand = activations, held in TENSOR MEMORY (tcgen05.mma with A from TMEM): a ring of TMEM stages of
//     64 columns (32 hi + 32 lo columns of packed bf16 pairs = one 64-channel K chunk for the 128 positions/lanes).
//     Shared memory therefore carries no activation traffic for the MMAs.
//   loader warps (2 groups x 4, alternating (tile, kernel row) units): cp.async gather of the warp's 32 positions plus
//                     the halo of one kernel row into a swizzled staging tile (current + next in flight); tap kx of that
//                     row is staging row lane + kx*dil, copied to the TMEM stage with tcgen05.st (thread = position = TMEM
//                     lane);
//   MMA warp (1 lane) 4 k-steps (K = 16) x 2 stacked tcgen05.mma.kind::f16 per segment (A from TMEM, B descriptor in smem)
//                     and tcgen05.commit of the stage back to the loaders / of the accumulator to the epilogue;
//   epilogue warps (8) tcgen05.ld the accumulator (one position per thread, 2 warps per lane quadrant), apply bias and
//                     optional ReLU, split into hi / lo bf16 and stage the tile in the TMA box layout;
//   TMA store lane    the two box stores of each tile.
#include <cuda.h>

#include "tc_ptx.cuh"

namespace mrb {
namespace tc {

constexpr int TILE_M = 128;
constexpr int COUT = 64;                      // output channels (all of them in one CTA)
constexpr int KC = 32;                        // TMEM columns of one K chunk half (hi or lo): 64 bf16 channels, packed in pairs
constexpr int KCH = 64;                       // channels per K chunk (one 128-byte row of bf16 in the B operand)
constexpr int A_STAGE_COLS = 2 * KC;          // hi + lo
constexpr int EPI_WARPS = 8;                  // 2 warps per TMEM lane quadrant (each takes half of the channels)
constexpr int LOAD_GROUPS = 2, LOAD_WARPS = 4 * LOAD_GROUPS;  // loader groups alternate (tile, kernel row) units
constexpr int MMA_WARPS = 2;                  // MMA issuer + TMA store lane
constexpr int THREADS = (EPI_WARPS + LOAD_WARPS + MMA_WARPS + 1) * 32;  // + weight-streaming warp
constexpr int B_STAGES = 6;                   // max depth of the streamed-weights ring (Params::b_stages)
constexpr int MAX_SEGS = 25;
constexpr int MAX_STAGES = 6;
constexpr int W_CHUNK_BYTES = COUT * 128;     // hi (or lo) rows of one weight chunk

constexpr int BH_PAD = 2;                     // replicate border of the BH activation layout (conv_tc2.cu)
constexpr int BH_PX_BYTES = 256;              // 64 hi + 64 lo bf16 per position
constexpr int OUT_BOX_BYTES = TILE_M * 128;   // one [128 positions x 64 bf16] TMA box
constexpr int HALO_ROWS = 32 + 2 * BH_PAD;    // staging rows of one loader unit at most: 32 positions + pad on each side
constexpr int BIAS_FLOATS = COUT;

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
    const uint8_t* src;      // BH input (replicate border valid)
    const void* wpack;       // packed bf16 weights: [tap][hi|lo][64 rows x 128 B swizzled]
    const float* bias;       // [64] (may be null)
    int B, H, W;             // image size
    long long P;             // flat positions of the BH layout, B (H+4)(W+4): the tiles run over them
    int n_tiles;
    int nseg;                // segments (taps) per tile; the global segment stream s = item * nseg + sgi is dealt to
                             // the TMEM stages and the weight ring
    int acc_cols;            // TMEM columns of one accumulator buffer: [hi*hi chain | cross-term chain]
    int acc_bufs;            // accumulator buffers
    int tmem_cols;           // allocation: 512
    int relu;
    int b_stages;            // depth of the streamed-weights ring (<= B_STAGES)
    int tb_depth;            // cp.async staging tiles per loader warp
    int tb_half;             // bytes of one staging half (32 + 2*pad rows x 128 B)
    int tb_bytes;            // bytes of one staging tile (2 halves)
    int ksz, dil;            // conv geometry
    int stages;              // A stages in TMEM (columns acc_bufs*acc_cols + 64*s)
#ifdef MRB_TC_PROF
    unsigned long long* prof; // optional [gridDim.x][16] cycle counters (tools/tc_roles.py)
    int debug;                // role switches: 1 skip MMAs, 2 skip global loads, 4 skip epilogue math, 8 skip tcgen05.st
#endif
};

__global__ void __launch_bounds__(THREADS, 1) tc_kernel(const __grid_constant__ CUtensorMap tm_out, const Params P) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // layout: [output tile][streamed-weights ring][loader staging tiles][barriers][bias]
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* out_s = smem;                                            // [hi box | lo box] output tile (1024-aligned)
    uint8_t* bst_s = smem + 2 * OUT_BOX_BYTES;                        // [b_stages][2*W_CHUNK_BYTES]
    uint8_t* tb_s = bst_s + (size_t)P.b_stages * 2 * W_CHUNK_BYTES;   // [LOAD_WARPS][depth][tb_bytes]
    uint64_t* bars = (uint64_t*)(tb_s + (size_t)LOAD_WARPS * P.tb_depth * P.tb_bytes);
    uint64_t* full = bars;                          // [MAX_STAGES]
    uint64_t* empty = bars + MAX_STAGES;            // [MAX_STAGES]
    uint64_t* acc_full = bars + 2 * MAX_STAGES;     // [2]
    uint64_t* acc_empty = acc_full + 2;             // [2]
    uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);
    uint64_t* b_full = acc_empty + 4;               // [B_STAGES]
    uint64_t* b_empty = b_full + B_STAGES;          // [B_STAGES]
    uint64_t* out_free = acc_empty + 3;             // [1] the TMA stores of the previous tile have read out_s
    uint64_t* out_ready = b_empty + B_STAGES;       // [1] every epilogue warp has written its part of the output tile
    float* bias_s = (float*)(out_ready + 2);        // [BIAS_FLOATS] (16-byte aligned): bias staged once per CTA

    // warp index through a shuffle: provably warp-uniform for the compiler (role branches and the MMA issuer's operands
    // then live in uniform registers)
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    const int first_tile = blockIdx.x;
    const int tile_stride = gridDim.x;

    if (threadIdx.x == 0) {
        for (int s = 0; s < P.stages; ++s) {
            mbar_init(&full[s], 4);    // one loader group fills a stage: one arrival per warp (lane 0, after __syncwarp)
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&acc_full[b], 1);
            mbar_init(&acc_empty[b], EPI_WARPS);  // one arrival per epilogue warp
        }
        for (int b = 0; b < B_STAGES; ++b) {
            mbar_init(&b_full[b], 1);   // the producer's arrive.expect_tx; the bulk copy completes the transaction bytes
            mbar_init(&b_empty[b], 1);  // tcgen05.commit of the MMAs that read the slot
        }
        mbar_init(out_free, 1);
        mbar_init(out_ready, EPI_WARPS);
        fence_barrier_init();
    }
    for (int i = threadIdx.x; i < COUT; i += THREADS) bias_s[i] = P.bias ? P.bias[i] : 0.f;
    if (warp == EPI_WARPS + LOAD_WARPS) tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t a_col0 = (uint32_t)(P.acc_bufs * P.acc_cols);  // first TMEM column of the A ring
    int n_items = 0;
    for (int t = first_tile; t < P.n_tiles; t += tile_stride) ++n_items;
    if (warp >= EPI_WARPS && warp < EPI_WARPS + LOAD_WARPS) {
        // ============================== LOADERS ==============================
        // The global segment stream s = item * nseg + sgi is dealt to the two loader groups in (tile, kernel row) units
        // of k segments; segment s goes to TMEM stage s % stages.
        const int lw = warp - EPI_WARPS;
        const int grp = lw >> 2;                     // loader group
        const int quad = lw & 3;                     // == warp % 4: the TMEM lane quadrant this warp may write
        const int c16 = lane & 7;                    // 16-byte chunk within a 128-byte half row (coalesced view)
        const int rl0 = lane >> 3;                   // rows rl0 + 4*i of the staging tile (coalesced view)
        const uint32_t tb_u32 = smem_u32(tb_s + (size_t)lw * P.tb_depth * P.tb_bytes);  // tb_depth staging tiles of this warp
        const uint32_t HB = (uint32_t)P.tb_half;     // the lo half of a staging row lives HB bytes after the hi half
        const bool ld_on = !TC_DBG(P, 2);
        TCP(long long t_start = clock64(), t_wait = 0, t_st = 0, t_issue = 0, t_stw = 0, c0;)

        int stage = 0;
        uint32_t phase = 0;
        auto stage_set = [&](long long s) { stage = (int)(s % P.stages); phase = (uint32_t)(s / P.stages) & 1u; };
        auto stage_adv = [&](int n) {
            stage += n;
            while (stage >= P.stages) { stage -= P.stages; phase ^= 1u; }
        };
        // staging row `row` of tile tb (64 hi bf16 in half 0, 64 lo bf16 in half 1) -> TMEM stage (thread = position =
        // TMEM lane quad*32 + lane): columns [0,32) = hi pairs, [32,64) = lo pairs -- a straight copy
        auto store_stage = [&](uint32_t tb, int row, int stg) {
            const uint32_t ta = tmem_base + ((uint32_t)(quad * 32) << 16) + a_col0 + (uint32_t)(stg * A_STAGE_COLS);
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                uint32_t v[32];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const float4 a = lds128(tb + hf * HB + swz(row, c));
                    v[4 * c] = __float_as_uint(a.x); v[4 * c + 1] = __float_as_uint(a.y);
                    v[4 * c + 2] = __float_as_uint(a.z); v[4 * c + 3] = __float_as_uint(a.w);
                }
                if (!TC_DBG(P, 8)) {
                    tmem_st16(ta + hf * KC, v);
                    tmem_st16(ta + hf * KC + 16, v + 16);
                }
            }
        };
        // wait for the stage, copy one staging row per lane, hand the stage to the issuer
        auto fill_stage = [&](uint32_t tb, int row) {
            TCP(c0 = clock64();)
            mbar_wait_sleep(&empty[stage], phase ^ 1, 40);
            TCP(t_wait += clock64() - c0;)
            tc_fence_after();
            TCP(c0 = clock64();)
            store_stage(tb, row, stage);
            TCP(const long long c2 = clock64();)
            tmem_st_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[stage]);
            TCP(t_st += clock64() - c0; t_stw += clock64() - c2;)
        };

        // unit = (tile, kernel row ky): the warp's 32 positions plus pad on each side of flat row offset
        // (ky*dil - pad) * pitch; tap kx reads staging row lane + kx*dil.  Positions outside the tensor are zero-filled
        // (they only feed border positions, whose results are not used).
        const int k = P.ksz, dil = P.dil, pad = dil * (k - 1) / 2;
        const long long pitch = P.W + 2 * BH_PAD;
        const int n_units = n_items * k;
        const int nrows = 32 + 2 * pad;
        auto issue_halo = [&](int tile, int ky, int slot) {
            const long long q0 = (long long)tile * TILE_M + quad * 32 - pad + (long long)(ky * dil - pad) * pitch;
            const uint32_t sbase = tb_u32 + (uint32_t)(slot * P.tb_bytes);
#pragma unroll
            for (int i = 0; i < HALO_ROWS / 4; ++i) {
                const int sr = rl0 + 4 * i;
                if (sr >= nrows) break;  // the staging tile has exactly nrows rows (a zero-fill would land in the lo half)
                const long long q = q0 + sr;
                const bool ok = q >= 0 && q < P.P;
                const uint8_t* g = P.src + q * BH_PX_BYTES + c16 * 16;
                const uint32_t nb = (ok && ld_on) ? 16u : 0u;
                cp_async16(sbase + swz(sr, c16), ok ? (const void*)g : (const void*)P.src, nb, true);
                cp_async16(sbase + HB + swz(sr, c16), ok ? (const void*)(g + 128) : (const void*)P.src, nb, true);
            }
        };
        int pf_u = grp, pf_tile = first_tile, pf_ky = grp, pf_slot = 0;
        while (pf_ky >= k) { pf_ky -= k; pf_tile += tile_stride; }
        auto prefetch_unit = [&]() {
            if (pf_u < n_units) issue_halo(pf_tile, pf_ky, pf_slot);
            asm volatile("cp.async.commit_group;" ::: "memory");
            pf_u += LOAD_GROUPS;
            pf_ky += LOAD_GROUPS;
            while (pf_ky >= k) { pf_ky -= k; pf_tile += tile_stride; }
            pf_slot ^= 1;
        };
        prefetch_unit();
        int slot = 0;
        stage_set((long long)grp * k);
        for (int u = grp; u < n_units; u += LOAD_GROUPS) {
            TCP(c0 = clock64();)
            prefetch_unit();
            TCP(t_issue += clock64() - c0;)
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            __syncwarp();
            const uint32_t tb = tb_u32 + (uint32_t)(slot * P.tb_bytes);
            for (int kx = 0; kx < k; ++kx) {
                fill_stage(tb, lane + kx * dil);
                stage_adv(1);
            }
            __syncwarp();  // every lane has read its rows before the slot is refilled
            stage_adv(k * (LOAD_GROUPS - 1));  // the other group's unit
            slot ^= 1;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
#ifdef MRB_TC_PROF
        if (P.prof && lane == 0 && lw == 0) {
            unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
            o[0] = clock64() - t_start; o[1] = t_wait; o[2] = t_st; o[3] = t_issue; o[13] = t_stw;
        }
#endif
    } else if (warp == EPI_WARPS + LOAD_WARPS) {
        // ============================== MMA ISSUER ==============================
        // Segments are issued in order into one accumulator buffer per tile, so a position's result is bit-identical run
        // to run and whatever the batch it is part of.  Whole warp, warp-uniform control flow (see umma_commit).
        TCP(const bool prof = P.prof != nullptr;)
        int stage = 0;
        uint32_t phase = 0;
        int bs = 0;
        uint32_t bphase = 0;
        TCP(long long t_start = clock64(), t_wfull = 0, t_wacc = 0, t_mma = 0, t_commit = 0, t_wb = 0, t_prep = 0, c0 = 0, c1 = 0;)
        int buf = 0;
        uint32_t acc_phase = 0;
        const uint32_t tmem_u = uni(tmem_base);
        const uint32_t bst_u32 = smem_u32(bst_s);
        // loop-invariant operands: every segment has N = 64 and the same accumulator columns; only the weight slot moves
        const uint64_t desc0 = make_desc(bst_u32);
        constexpr uint32_t idesc_n = make_idesc(TILE_M, COUT), idesc_2n = make_idesc(TILE_M, 2 * COUT);
        for (int tile = first_tile; tile < P.n_tiles; tile += tile_stride) {
            TCP(if (prof) c0 = clock64();)
            mbar_wait(&acc_empty[buf], acc_phase ^ 1);
            TCP(if (prof) t_wacc += clock64() - c0;)
            tc_fence_after();
            const uint32_t d = tmem_u + (uint32_t)(buf * P.acc_cols);
            for (int sgi = 0; sgi < P.nseg; ++sgi) {
                TCP(if (prof) c1 = clock64();)
                // every MMA operand is derived from kernel parameters and uniform loop state (no shared-memory table, no
                // shuffles): it stays in uniform registers, and it is ready before the waits return
                const uint64_t dbh = desc0 + (uint64_t)((bs * 2 * W_CHUNK_BYTES) >> 4);
                const uint32_t a_hi = tmem_u + a_col0 + (uint32_t)(stage * A_STAGE_COLS);
                TCP(if (prof) c0 = clock64();)
                mbar_wait(&b_full[bs], bphase);
                TCP(if (prof) t_wb += clock64() - c0;)
                TCP(if (prof) c0 = clock64();)
                mbar_wait(&full[stage], phase);
                TCP(if (prof) t_wfull += clock64() - c0;)
                tc_fence_after();
                TCP(if (prof) { c0 = clock64(); t_prep += c0 - c1; })
                if (!TC_DBG(P, 1)) {
                    // the N = 2n MMA of k-step 0 of the first segment overwrites [main | cross]; everything after it
                    // accumulates (MMAs of one thread execute in order)
                    umma_segment_ts_stacked(d, d + (uint32_t)COUT, a_hi, a_hi + KC, dbh, idesc_2n, idesc_n, sgi == 0 ? 0u : 1u);
                }
                TCP(if (prof) { t_mma += clock64() - c0; c0 = clock64(); })
                umma_commit(&empty[stage]);  // stage reusable once these MMAs have read it
                umma_commit(&b_empty[bs]);
                if (++bs == P.b_stages) { bs = 0; bphase ^= 1u; }
                TCP(if (prof) t_commit += clock64() - c0;)
                if (++stage == P.stages) { stage = 0; phase ^= 1u; }
            }
            umma_commit(&acc_full[buf]);
            if (++buf == P.acc_bufs) { buf = 0; acc_phase ^= 1u; }
        }
#ifdef MRB_TC_PROF
        if (prof && lane == 0) {
            unsigned long long* o = P.prof + (size_t)blockIdx.x * 16;
            o[4] = clock64() - t_start; o[5] = t_wfull; o[6] = t_wacc; o[7] = t_mma; o[10] = t_commit; o[11] = t_wb; o[12] = t_prep;
        }
#endif
    } else if (warp == EPI_WARPS + LOAD_WARPS + 1) {
        // ============================== TMA STORE LANE ==============================
        if (lane == 0) {
            const uint32_t out_u32 = smem_u32(out_s);
            uint32_t oph = 0;
            for (int tile = first_tile; tile < P.n_tiles; tile += tile_stride) {
                mbar_wait_sleep(out_ready, oph, 64);
                tma_store_2d(&tm_out, out_u32, 0, tile * TILE_M);
                tma_store_2d(&tm_out, out_u32 + OUT_BOX_BYTES, 64, tile * TILE_M);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                mbar_arrive(out_free);
                oph ^= 1;
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before the CTA exits
        }
    } else if (warp == EPI_WARPS + LOAD_WARPS + MMA_WARPS) {
        // ============================== WEIGHT STREAMER ==============================
        // one lane, one bulk copy (cp.async.bulk, 2*W_CHUNK_BYTES contiguous bytes: hi rows | lo rows) per segment
        if (lane == 0) {
            int bs = 0;
            uint32_t bphase = 0;
            const uint32_t bytes = (uint32_t)(2 * W_CHUNK_BYTES);
            for (int it = 0; it < n_items; ++it) {
                for (int sgi = 0; sgi < P.nseg; ++sgi) {
                    mbar_wait_sleep(&b_empty[bs], bphase ^ 1, 64);
                    const uint8_t* gsrc = reinterpret_cast<const uint8_t*>(P.wpack) + (size_t)sgi * bytes;
                    const uint32_t bar = smem_u32(&b_full[bs]);
                    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
                    asm volatile(
                        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                            smem_u32(bst_s + (size_t)bs * bytes)),
                        "l"(gsrc), "r"(bytes), "r"(bar)
                        : "memory");
                    if (++bs == P.b_stages) { bs = 0; bphase ^= 1; }
                }
            }
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
        int buf = 0;
        uint32_t acc_phase = 0;
        for (int tile = first_tile; tile < P.n_tiles; tile += tile_stride) {
            const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * P.acc_cols);
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
                    tmem_ld8x4(t0 + j, t0 + 64 + j, t0 + j + 8, t0 + 64 + j + 8, a, a2, b1, b2);
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
            }
            // the tile's [128 positions x (64 hi | 64 lo)] boxes are complete once all eight epilogue warps have
            // arrived; the TMA store lane takes it from there
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(out_ready);
            oph ^= 1;
            if (++buf == P.acc_bufs) { buf = 0; acc_phase ^= 1u; }
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
    if (warp == EPI_WARPS + LOAD_WARPS) {
        tc_fence_after();
        tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
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

static size_t smem_needed(const Params& P) {
    return 1024 + (size_t)2 * OUT_BOX_BYTES + (size_t)P.b_stages * 2 * W_CHUNK_BYTES +
           (size_t)LOAD_WARPS * P.tb_depth * P.tb_bytes + 256 + 2 * B_STAGES * 8 + BIAS_FLOATS * sizeof(float);
}

#ifdef MRB_TC_PROF
static int g_debug = 0;
static unsigned long long* g_prof = nullptr;
#endif

static int launch(Params& P, void* out, cudaStream_t st) {
#ifdef MRB_TC_PROF
    P.debug = g_debug;
    P.prof = g_prof;
#endif
    const size_t max_smem = device_max_smem_optin();
    P.tmem_cols = 512;
    P.stages = (512 - P.acc_bufs * P.acc_cols) / A_STAGE_COLS;
    if (P.stages > MAX_STAGES) P.stages = MAX_STAGES;
    MRB_REQUIRE(P.stages >= 2, MRB_EUNSUPPORTED, "tensor-core conv: accumulator leaves no room for the TMEM A ring");
    MRB_REQUIRE(P.P < 2147483647LL, MRB_EUNSUPPORTED, "tensor-core conv: too many pixels");
    MRB_REQUIRE(P.nseg >= 1 && P.nseg <= MAX_SEGS, MRB_EUNSUPPORTED, "tensor-core conv: bad segment count");
    CUtensorMap tm_out;
    memset(&tm_out, 0, sizeof(tm_out));
    int rc = tc2::make_bh_tmap(&tm_out, out, P.P, TILE_M);
    if (rc) return rc;
    // 32 + 2*pad flat positions per unit
    P.tb_half = (32 + P.dil * (P.ksz - 1)) * 128;
    P.tb_bytes = 2 * P.tb_half;
    P.tb_depth = 2;  // one staging tile feeds k segments: current + next is enough
    P.b_stages = B_STAGES;
    while (P.b_stages > 2 && smem_needed(P) > max_smem) --P.b_stages;
    MRB_REQUIRE(smem_needed(P) <= max_smem, MRB_EUNSUPPORTED, "tensor-core conv: staging does not fit shared memory");
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
    tc_kernel<<<grid, THREADS, max_smem, st>>>(tm_out, P);
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
    tc::Params P;
    memset(&P, 0, sizeof(P));
    P.B = B; P.H = H; P.W = W;
    P.P = (long long)B * (H + 2 * tc::BH_PAD) * (W + 2 * tc::BH_PAD);
    long long nt = (P.P + tc::TILE_M - 1) / tc::TILE_M;
    MRB_REQUIRE(nt <= 2147483647LL, MRB_EUNSUPPORTED, "tensor-core conv: too many pixels");
    P.n_tiles = (int)nt;
    P.src = (const uint8_t*)x_bh;
    P.wpack = wpack; P.bias = (const float*)bias;
    // One segment per tap (64 input channels = one 128-byte bf16 row of B), stacked MMAs of N = 128 and 64 (half the MMA
    // instructions of a channel split).  The k*k weight chunks (2*64*128 B each: hi rows | lo rows) are streamed from L2
    // through a small ring -- resident they would leave no room for the halo staging tiles.
    P.nseg = k * k;
    // One accumulator group per buffer (hi*hi chain | cross-term chain, summed in the epilogue), two buffers.  Measured
    // and removed: two MMA issuers on alternating segments with plain st.global from the epilogue -- 443 vs 371 us at
    // B = 16: the thread-per-position stores (32 cache lines per instruction) compete with the loaders' cp.async for L1
    // wavefronts.
    P.acc_cols = 2 * cout;
    P.acc_bufs = 2;
    P.relu = relu;
    P.ksz = k; P.dil = dil;
    return tc::launch(P, out_bh, (cudaStream_t)stream);
}
