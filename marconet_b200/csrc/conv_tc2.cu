// conv_tc2.cu -- tcgen05 / TMEM / TMA operand-split implicit-GEMM convolution for sm_100a: the tensor-core path of mn_conv2d_nhwc.
//
// Numerics: the reference computes every conv in fp32 and the parity budget (1e-3 end to end, bit-exact argmax) rules out
// single-pass fp16/bf16/tf32 operands (SURVEY.md section 0.7).  This kernel keeps fp32 activations in HBM and gets fp32-grade
// products out of the fp16 tensor pipe by operand splitting:
//     x = xh + xl,  w = wh + wl        (xh, xl, wh, wl fp16; |x - xh - xl| <= 2^-22 |x|)
//     x*w ~= xh*wh + (xh*wl + xl*wh)   (three kind::f16 MMAs per k-step into two fp32 TMEM accumulators: D takes xh*wh, Dc the
//                                       two cross terms; the epilogue adds D + Dc once, in fp32)
// The tensor core truncates every add into an fp32 accumulator; with the cross terms (2^-11 of the result) kept apart, only K/16
// instead of 3K/16 truncations hit the full-magnitude sum (DESIGN.md section 3.1).
// The weights are split once by mn_conv_pack_weights_tc (end of this file), the activations on the fly by the split warps.
//
// Loading the 128-pixel activation tile once per tap, with every CTA streaming its own copy of the weights, would move 64 KB from
// L2 to shared memory per 768 MMA cycles per SM and leave the kernel L2-bandwidth bound.  The design removes that traffic:
//   * HALO TILE.  Loop order is (64-channel block) outer, (tap) inner.  One TMA box per channel block brings the
//     (TH+2) x (TW+2) halo of the 128-pixel output tile (zero-filled outside the image = conv padding); the 9 taps are
//     9 shifted *reads* of that tile by the split warps (row r of tap (ky,kx) is halo row r0 + ky*(TW+2) + kx).
//     Activation traffic drops from 9 x 32 KB to ~1.4-1.6 x 32 KB per channel block.
//   * WEIGHT MULTICAST.  CTAs of a cluster (2 consecutive pixel tiles, same output-channel tile) each load 1/CS of
//     every weight tile and TMA-multicast it to all; the stage is released by tcgen05.commit multicast to every CTA.
//   * PERSISTENT tiles: one CTA per SM loops over work items; producers run ahead into the next tile while the split
//     warps drain TMEM (through a shared-memory staging buffer -> fully coalesced global stores).
//   * SPLIT ONCE.  fp32->fp16 pair conversion (F2FP) runs on the quarter-rate XU pipe; converting every tap's tile costs
//     ~1000 XU cycles per 768-cycle MMA block (measured: XU 53 % busy, tensor pipe 12 %).  Four dedicated warps now split
//     each halo tile ONCE per channel block, in place in shared memory (hi plane over box 0, lo plane over box 1, same
//     XOR swizzle), and the four TMEM-feeding warps only copy shifted rows smem -> TMEM per tap (no ALU work).
//   * OVERLAPPED EPILOGUE.  The split warps (which cover the four TMEM lane quarters) also own the epilogue: after splitting
//     the first two halo tiles of tile i+1 they drain tile i's accumulators (second half parked in registers so the
//     MMA warp is released after ~1k cycles), stage through shared memory and store with fully coalesced float4 rows,
//     while the feed + MMA warps are already working on tile i+1.
// Warp roles: 0 = weight (B) TMA producer, 1 = TMEM allocator + MMA issuer, 2..5 = TMEM feed,
//             6 = halo TMA producer, 7..10 = split (fp32 halo -> hi/lo fp16 halo), 11..14 = epilogue (round 2: its own warps).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include "conv_common.cuh"
#include "mn_common.cuh"
#include "tc_ptx.cuh"

namespace {
using namespace tcptx;

constexpr int KB = 64;
constexpr int NUM_THREADS2 = 480;               // 15 warps: see the role list in the header comment
constexpr int A_STAGES = 4;
constexpr int MAX_BSTAGES = 4;
constexpr int STG_COLS = 64;
constexpr int STG_PITCH = STG_COLS + 4;
constexpr int STG_BYTES = 128 * STG_PITCH * 4;
constexpr int TMEM_COLS2 = 512;
constexpr int SMEM_LIMIT = 232448;          // 227 KB

template <int A> struct ActTag { static constexpr int value = A; };

struct Tc2Geom {
    int TW, TH, TN, HWd, HHt, halo_rows, box_bytes, halo_stage_bytes;
    int tiles_w, tiles_h, tiles_n, m_tiles, m_groups, n_tiles;
    int cblocks, taps, KW, ph, pw;
    int ksplit, cbps;   // split-K over channel blocks for layers with too few tiles: work = (tile, k-slice), cbps channel blocks each
    int bstages, cs, cg;
    long long* trace;   // developer timeline (tools/trace_tc2.py): CTA 0 records (event, clock64) pairs; NULL in production
    int hstages;        // depth of the halo ring (2, or 3 when shared memory allows: layers with <= 2 channel blocks per tile
                        // otherwise stall every tile on the TMA latency of the next tile's second halo)
    int epi_cb;         // the split warps run the epilogue of tile i after splitting this channel block of tile i+1
    const float* wscale;
    int prec;
};

// CG = 2: the two CTAs of a cluster form ONE tcgen05 CTA pair (cta_group::2): a single MMA covers M = 256 pixels (128 per CTA,
// each CTA's A operand in its own TMEM) x NT channels, and each CTA keeps only ITS HALF of every weight tile in shared memory
// (NT/2 rows; no multicast).  Why: with cta_group::1 the tensor core reads B (4 KB per 64-cycle MMA = 64 B/clk) from the same
// shared-memory port that the TMEM-feed warps read the halo through (32 KB per k-block = 42 B/clk) and the split warps work
// in -- ~120 of the port's 128 B/clk, which is what held the kernel at ~73 % of the tensor pipe although the MMA stream alone
// issues at 95-100 % (tools/mma_probe2.cu).  The pair halves the B reads per SM.  Only the leader CTA (cluster rank 0) issues MMAs;
// its barriers collect the peer's TMA bytes (BF), feed-warp arrivals (CD) and epilogue arrivals (ACCE) through DSMEM, and its
// tcgen05.commit multicasts the stage-release / accumulator-full signals to both CTAs.
template <int NT, bool GN, int CG>
__global__ void __launch_bounds__(NUM_THREADS2, 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBhi,
                const __grid_constant__ CUtensorMap tmBlo, const ConvGeom g, const Tc2Geom t) {
    constexpr int B_HALF = (NT / CG) * 128;       // bytes of one (hi or lo) weight tile held by this CTA
    constexpr int B_STAGE = 2 * B_HALF;
    // TMEM: accumulator stage a: D [a*2NT, +NT), Dc [a*2NT+NT, +NT); A stage s at ACC_ST*2NT + 64s (hi) / +32 (lo).
    // NT = 64 leaves room for TWO accumulator stages: the MMAs of tile i+1 start while the epilogue still drains tile i (the drain
    // bubble is ~1k cycles against a 3.5k-cycle tile for the 64->64 layers at 128x2048).  NT = 128 fills TMEM with one.
    constexpr int ACC_ST = (NT == 64) ? 2 : 1;
    constexpr int A_COL0 = ACC_ST * 2 * NT;
    static_assert(A_COL0 + A_STAGES * 64 <= TMEM_COLS2, "TMEM budget");

    extern __shared__ uint8_t smem_raw[];
    // keep the pointer in the shared address space (offset arithmetic on the array) so loads compile to LDS, not generic LD
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t smem_base = smem_u32(smem);
    const int HS = t.hstages;
    const uint32_t off_b = HS * t.halo_stage_bytes;
    const uint32_t off_stg = off_b + t.bstages * B_STAGE;
    const uint32_t off_rowm = off_stg + STG_BYTES;
    const uint32_t off_bars = off_rowm + 1024;
    float* stg = reinterpret_cast<float*>(smem + off_stg);
    int* rowm = reinterpret_cast<int*>(smem + off_rowm);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + off_bars);
    // barrier indices
    constexpr int MAX_HS = 3;
    constexpr int I_HF = 0, I_HE = MAX_HS, I_BF = 2 * MAX_HS, I_BE = I_BF + MAX_BSTAGES, I_CD = I_BE + MAX_BSTAGES, I_AE = I_CD + A_STAGES,
                  I_ACCF = I_AE + A_STAGES, I_ACCE = I_ACCF + 2, I_SD = I_ACCE + 2, N_BARS = I_SD + MAX_HS;
    auto bar = [&](int i) { return smem_u32(bars + i); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + N_BARS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cs = t.cs;
    const uint32_t crank = cs > 1 ? cluster_ctarank() : 0u;
    const uint16_t cmask = (uint16_t)((1u << cs) - 1u);
    const int cluster_id = blockIdx.x / cs, num_clusters = gridDim.x / cs;
    const int total_work = t.m_groups * t.n_tiles * t.ksplit;
    const int BS = t.bstages;
    // work item -> (k-slice, channel tile, pixel-tile group); identical in every warp role
    auto work_ks = [&](int work) { return work % t.ksplit; };
    auto work_nt = [&](int work) { return (work / t.ksplit) % t.n_tiles; };
    auto work_mg = [&](int work) { return work / (t.ksplit * t.n_tiles); };

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmBlo) : "memory");
        for (int s = 0; s < MAX_HS; ++s) { mbar_init(bar(I_HF + s), 1); mbar_init(bar(I_HE + s), 128); mbar_init(bar(I_SD + s), 128); }
        for (int s = 0; s < MAX_BSTAGES; ++s) { mbar_init(bar(I_BF + s), 1); mbar_init(bar(I_BE + s), CG == 2 ? 1 : cs); }
        // CG = 2: one elected arrival per feed / epilogue warp of BOTH CTAs lands on the leader's barrier (4 local + 4 remote)
        for (int s = 0; s < A_STAGES; ++s) { mbar_init(bar(I_CD + s), CG == 2 ? 8 : 128); mbar_init(bar(I_AE + s), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(bar(I_ACCF + a), 1); mbar_init(bar(I_ACCE + a), CG == 2 ? 8 : 128); }
        fence_barrier_init();
    }
    if (warp == 1) { if (CG == 2) tmem_alloc_cg2(smem_u32(tmem_slot), TMEM_COLS2); else tmem_alloc(smem_u32(tmem_slot), TMEM_COLS2); }
    tc_fence_before();
    __syncthreads();
    if (cs > 1) cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) may overlap the
    // tail of the previous kernel in the stream; from here on we read its results, so wait for it to complete and flush.
    // Let our own dependents start their prologue as soon as SMs free up.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    // timeline instrumentation (off unless mn_debug_tc2_trace installed a buffer): event e of role-lane `who` at clock64()
    long long* const trace = (t.trace && blockIdx.x == 0) ? t.trace : nullptr;
    // Fixed slots, plain stores (an atomic slot counter stalls the marking warp for an L2 round trip per event and distorts the
    // timeline): tile iteration `it` of this CTA owns 64 int64s; events 1..15 at [it*64 + ev], per-k-block events ev >= 16 at
    // [it*64 + ev] (the caller adds the k-block index, < 24).
    auto mark = [&](int ev, int idx) {
        if (trace) {
            const int it = (idx - cluster_id) / num_clusters;
            if (it < 64 && ev < 64) trace[1 + it * 64 + ev] = clock64();
        }
    };
    auto tile_origin = [&](int work, int& n0, int& oy0, int& ox0) {
        int m_tile = work_mg(work) * cs + (int)crank;
        if (m_tile >= t.m_tiles) { n0 = g.N + 1024; oy0 = 0; ox0 = 0; return; }   // padding CTA of a cluster: everything out of bounds
        const int tw_i = m_tile % t.tiles_w; m_tile /= t.tiles_w;
        const int th_i = m_tile % t.tiles_h; m_tile /= t.tiles_h;
        n0 = m_tile * t.TN; oy0 = th_i * t.TH; ox0 = tw_i * t.TW;
    };

    if (warp == 0) {
        // =========================== weight (B) producer (whole warp converged, one elected lane issues) ===========================
        uint32_t s = 0, ph = 0;
        const int rows = NT / cs;
        const uint32_t dst0 = smem_base + off_b + (CG == 2 ? 0u : crank * rows * 128);
        for (int work = cluster_id; work < total_work; work += num_clusters) {
            const int row0 = work_nt(work) * NT + (int)crank * rows;
            const int cb0 = work_ks(work) * t.cbps;
            for (int cb = cb0; cb < cb0 + t.cbps; ++cb) {
                for (int tap = 0; tap < t.taps; ++tap) {
                    mbar_wait(bar(I_BE + s), ph ^ 1);
                    if (elect_one_sync()) {
                        const uint32_t dst = dst0 + s * B_STAGE;
                        if (CG == 2) {
                            // this CTA's half of the tile into its own smem; bytes of BOTH halves are counted on the LEADER's barrier
                            if (crank == 0) mbar_expect_tx(bar(I_BF + s), 2 * B_STAGE);
                            const uint32_t lbar = mapa_u32(bar(I_BF + s), 0);
                            tma_load_3d_cg2(&tmBhi, lbar, dst, cb * KB, row0, tap);
                            tma_load_3d_cg2(&tmBlo, lbar, dst + B_HALF, cb * KB, row0, tap);
                        } else if (cs > 1) {
                            mbar_expect_tx(bar(I_BF + s), B_STAGE);
                            tma_load_3d_mc(&tmBhi, bar(I_BF + s), dst, cb * KB, row0, tap, cmask);
                            tma_load_3d_mc(&tmBlo, bar(I_BF + s), dst + B_HALF, cb * KB, row0, tap, cmask);
                        } else {
                            mbar_expect_tx(bar(I_BF + s), B_STAGE);
                            tma_load_3d(&tmBhi, bar(I_BF + s), dst, cb * KB, row0, tap);
                            tma_load_3d(&tmBlo, bar(I_BF + s), dst + B_HALF, cb * KB, row0, tap);
                        }
                    }
                    __syncwarp();
                    if (++s == (uint32_t)BS) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == 6) {
        // =========================== halo (A) producer ===========================
        uint32_t hs = 0, ph = 0;
        for (int work = cluster_id; work < total_work; work += num_clusters) {
            int n0, oy0, ox0;
            tile_origin(work, n0, oy0, ox0);
            const int cb0 = work_ks(work) * t.cbps;
            for (int cb = cb0; cb < cb0 + t.cbps; ++cb) {
                mbar_wait(bar(I_HE + hs), ph ^ 1);
                if (elect_one_sync()) {
                    mark(1, work);                       // halo stage free -> TMA issue
                    mbar_expect_tx(bar(I_HF + hs), 2u * t.halo_rows * 128u);
                    const uint32_t dst = smem_base + hs * t.halo_stage_bytes;
                    tma_load_4d(&tmA, bar(I_HF + hs), dst, cb * KB, ox0 - t.pw, oy0 - t.ph, n0);
                    tma_load_4d(&tmA, bar(I_HF + hs), dst + t.box_bytes, cb * KB + 32, ox0 - t.pw, oy0 - t.ph, n0);
                }
                __syncwarp();
                if (++hs == (uint32_t)HS) { hs = 0; ph ^= 1; }
            }
        }
    } else if (warp >= 7) {
        // =========================== split warps: fp32 halo -> (hi, lo) 16-bit halo, in place ===========================
        const int sidx = (warp - 7) * 32 + lane;
        const bool bf = t.prec == MN_PREC_BF16X3_TC;
        const uint32_t mask = bf ? 0xFFFF0000u : 0xFFFFE000u;
        // ---- epilogue of one finished tile (these warps cover the four TMEM lane quarters: warp & 3) ----
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const float wscale = (t.wscale ? *t.wscale : 1.f) / g.x_scale;      // x_scale is a power of two: exact
        const float xs = g.x_scale;
        float amax = 0.f;                                                   // max |x * x_scale| this thread has split (range guard)
        // The tensor core truncates (toward zero) every time it adds into the fp32 accumulator: measured mean shrink of the
        // main accumulator = 1.56e-8 per accumulation step, sign-symmetric, independent of K (tools/probe_tc_bias.py).  Undo the
        // expected shrink of D (K/16 steps); Dc is 2^-11 of the result and needs nothing.
        const float dfix = 1.f + 1.5e-8f * (float)(t.taps * t.cbps * (KB / 16));
        const int tn = r / (t.TH * t.TW);
        const int rem = r - tn * (t.TH * t.TW);
        const int th = rem / t.TW, tw = rem - th * t.TW;
        uint32_t ecnt = 0;
        auto epilogue = [&](int work) {
            const int nt_i = work_nt(work);
            const int ks = work_ks(work);
            int n0, oy0, ox0;
            if (r == 0) mark(13, work);                    // epilogue loop top
            tile_origin(work, n0, oy0, ox0);
            {
                const int n = n0 + tn, oy = oy0 + th, ox = ox0 + tw;
                const bool ok = tn < t.TN && n < g.N && oy < g.OH && ox < g.OW;
                rowm[r] = ok ? (n * g.OH + oy) * g.OW + ox : -1;
                rowm[128 + r] = ok ? (n | ((g.valid_w && ox >= g.valid_w[n]) ? (1 << 30) : 0)) : 0;
            }
            const uint32_t acc_st = ACC_ST == 2 ? (ecnt & 1) : 0u, acc_ph = ACC_ST == 2 ? ((ecnt >> 1) & 1) : (ecnt & 1);
            const uint32_t acc_addr = lane_addr + acc_st * 2 * NT;
            mbar_wait(bar(I_ACCF + acc_st), acc_ph);
            if (r == 0) mark(8, work);                     // accumulators complete -> drain starts
            ++ecnt;
            tc_fence_after();
            constexpr int HALVES = NT / STG_COLS;
            float keep[(HALVES > 1) ? STG_COLS : 1];           // second half parked in registers so TMEM is released early
            auto drain = [&](int half, bool to_regs) {
#pragma unroll
                for (int chunk = 0; chunk < STG_COLS / 16; ++chunk) {
                    uint32_t acc[16];
                    tc_ld16(acc_addr + half * STG_COLS + chunk * 16, acc);
                    if (t.prec != MN_PREC_F16X1_TC) {
                        uint32_t cor[16];
                        tc_ld16(acc_addr + NT + half * STG_COLS + chunk * 16, cor);
                        tc_wait_ld();
#pragma unroll
                        for (int i = 0; i < 16; ++i) acc[i] = __float_as_uint(fmaf(__uint_as_float(acc[i]), dfix, __uint_as_float(cor[i])) * wscale);
                    } else {
                        tc_wait_ld();
#pragma unroll
                        for (int i = 0; i < 16; ++i) acc[i] = __float_as_uint(__uint_as_float(acc[i]) * wscale);
                    }
                    if (to_regs) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) keep[(HALVES > 1) ? chunk * 16 + i : 0] = __uint_as_float(acc[i]);
                    } else {
                        float4* dst = reinterpret_cast<float4*>(stg + r * STG_PITCH + chunk * 16);
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            dst[i] = make_float4(__uint_as_float(acc[4 * i]), __uint_as_float(acc[4 * i + 1]), __uint_as_float(acc[4 * i + 2]),
                                                 __uint_as_float(acc[4 * i + 3]));
                    }
                }
            };
            drain(0, false);
            if (HALVES > 1) drain(1, true);
            tc_fence_before();
            if (r == 0) mark(9, work);                           // drain done
            if (CG == 2) {                                       // one arrival per warp, on the LEADER's barrier (it issues the pair's MMAs)
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(mapa_u32(bar(I_ACCE + acc_st), 0));
            } else {
                mbar_arrive(bar(I_ACCE + acc_st));               // accumulators fully read: the MMA warp may start the next tile
            }
#pragma unroll 1
            for (int half = 0; half < HALVES; ++half) {
                if (half == 1) {
                    float4* dst = reinterpret_cast<float4*>(stg + r * STG_PITCH);
#pragma unroll
                    for (int i = 0; i < STG_COLS / 4; ++i)
                        dst[i] = make_float4(keep[(HALVES > 1) ? 4 * i : 0], keep[(HALVES > 1) ? 4 * i + 1 : 0], keep[(HALVES > 1) ? 4 * i + 2 : 0],
                                             keep[(HALVES > 1) ? 4 * i + 3 : 0]);
                }
                named_bar_sync(1, 128);
                if (r == 0) mark(11, work);                      // staging complete (all four warps drained)
                {
                    const int col = (lane & 15) * 4;
                    const int o = nt_i * NT + half * STG_COLS + col;
                    if (t.ksplit > 1) {
                        // raw partial sum of this k-slice; conv_splitk_reduce_kernel adds the slices and runs the epilogue
#pragma unroll 4
                        for (int i = 0; i < 16; ++i) {
                            const int row = q * 32 + i * 2 + (lane >> 4);
                            const int m = rowm[row];
                            if (m >= 0)
                                *reinterpret_cast<float4*>(g.ws + ((size_t)ks * g.M + m) * g.Cout + o) =
                                    *reinterpret_cast<const float4*>(stg + row * STG_PITCH + col);
                        }
                    } else {
                        const float4 bias4 = g.bias ? ldg4(g.bias + o) : make_float4(0.f, 0.f, 0.f, 0.f);
                        // one sample per tile (every layer except the 4x4 .. 8x8 maps): its per-sample scale vectors are loaded once
                        const bool one_n = t.TN == 1;
                        float4 os4 = make_float4(1.f, 1.f, 1.f, 1.f), y2s4 = os4;
                        float* y2base = g.y2;
                        if (one_n && n0 < g.N) {
                            if (g.out_scale) os4 = ldg4(g.out_scale + (size_t)n0 * g.os_stride + o);
                            if (g.y2 && g.y2_scale) y2s4 = ldg4(g.y2_scale + (size_t)n0 * g.y2s_stride + o);
                            // per-sample (possibly peer-GPU) destination of the second output, rebased so that row index m addresses it
                            if (g.y2_ptrs) y2base = g.y2_ptrs[n0] - (size_t)n0 * g.OH * g.OW * g.y2_cs;
                        }
                        float gs = 0.f, gq = 0.f;       // GroupNorm statistics of this thread's 16 rows x 4 channels (one group)
                        // One sample per tile and the tile inside the tensor (the plan guarantees H % TH == 0, W % TW == 0): every row is
                        // valid and its pixel index is arithmetic -- no rowm look-ups, no per-row branch, so the unrolled iterations overlap
                        // (the branchy loop serialised three dependent shared-memory loads per row: ~9k cycles per 64-column half,
                        // the limiter of the 64-wide tiles, tools/trace_tc2.py).
                        const bool dense_tile = one_n && n0 < g.N;
                        const int tws = __ffs(t.TW) - 1;
                        const int m00 = (n0 * g.OH + oy0) * g.OW + ox0;
                        const int vwn = (dense_tile && g.valid_w) ? g.valid_w[n0] : 0x7fffffff;
                        auto rows_dense = [&](auto tag) {
                            constexpr int ACT = decltype(tag)::value;
#pragma unroll 8
                            for (int i = 0; i < 16; ++i) {
                                const int row = q * 32 + i * 2 + (lane >> 4);
                                const int th = row >> tws, tw = row & (t.TW - 1);
                                const int m = m00 + th * g.OW + tw;
                                const float4 u = *reinterpret_cast<const float4*>(stg + row * STG_PITCH + col);
                                const float4 w4 = conv_epilogue_row4<ACT>(g, m, n0, ox0 + tw >= vwn, o, u, bias4, true, os4, true, y2s4, y2base);
                                if (g.gn_stats_out) {
                                    gs += (w4.x + w4.y) + (w4.z + w4.w);
                                    gq = fmaf(w4.x, w4.x, fmaf(w4.y, w4.y, fmaf(w4.z, w4.z, fmaf(w4.w, w4.w, gq))));
                                }
                            }
                        };
                        auto rows = [&](auto tag) {
                            constexpr int ACT = decltype(tag)::value;
                            if (dense_tile) { rows_dense(tag); return; }
                            if (one_n) return;                       // padding CTA of a cluster: nothing to store
#pragma unroll 4
                            for (int i = 0; i < 16; ++i) {
                                const int row = q * 32 + i * 2 + (lane >> 4);
                                const int m = rowm[row];
                                if (m >= 0) {
                                    const int nn = rowm[128 + row];
                                    const float4 u = *reinterpret_cast<const float4*>(stg + row * STG_PITCH + col);
                                    const float4 w4 = conv_epilogue_row4<ACT>(g, m, nn & 0x3FFFFFFF, (nn >> 30) != 0, o, u, bias4, one_n, os4, one_n, y2s4, y2base);
                                    if (g.gn_stats_out) {
                                        gs += (w4.x + w4.y) + (w4.z + w4.w);
                                        gq = fmaf(w4.x, w4.x, fmaf(w4.y, w4.y, fmaf(w4.z, w4.z, fmaf(w4.w, w4.w, gq))));
                                    }
                                }
                            }
                        };
                        switch (g.act) {
                            case MN_ACT_NONE: rows(ActTag<MN_ACT_NONE>{}); break;
                            case MN_ACT_RELU: rows(ActTag<MN_ACT_RELU>{}); break;
                            case MN_ACT_LRELU02: rows(ActTag<MN_ACT_LRELU02>{}); break;
                            default: rows(ActTag<-1>{}); break;
                        }
                        if (r == 0) mark(12, work);              // rows stored (this warp)
                        if (g.gn_stats_out) {
                            // lanes 0-7 / 8-15 (and 16-23 / 24-31, the odd rows) hold the two 32-channel groups of this 64-column half
#pragma unroll
                            for (int sh = 1; sh <= 4; sh <<= 1) { gs += __shfl_xor_sync(0xffffffffu, gs, sh); gq += __shfl_xor_sync(0xffffffffu, gq, sh); }
                            gs += __shfl_xor_sync(0xffffffffu, gs, 16); gq += __shfl_xor_sync(0xffffffffu, gq, 16);
                            if ((lane & 23) == 0 && n0 < g.N) {        // lanes 0 and 8
                                double* dst = g.gn_stats_out + ((size_t)n0 * (g.Cout >> 5) + (o >> 5)) * 2;
                                atomicAdd(dst, (double)gs);
                                atomicAdd(dst + 1, (double)gq);
                            }
                        }
                    }
                }
                named_bar_sync(1, 128);
            }
            if (r == 0) mark(10, work);                          // tile stored
        };
        // The epilogue of tile i runs after the first two halo tiles of tile i+1 have been split, so the feed/MMA warps have
        // ~2 x taps k-blocks of work queued while these warps drain TMEM and store tile i.
        if (warp >= 11) {
            // ======================= dedicated epilogue warps (11..14: warp & 3 = 3,0,1,2 -> the four TMEM lane quarters) =======================
            // Round 2: the four split warps used to run the epilogue as well and were the co-bottleneck of every tile with a short K
            // loop (ncu source page: 27 % of all stall samples in the row-store loop on 128->128 @128x128 against 5 % in the split);
            // 122 registers per thread at 480 threads, no spills.
            for (int work = cluster_id; work < total_work; work += num_clusters) epilogue(work);
        } else {
        uint32_t hs = 0, hph = 0;
        constexpr bool gn = GN;       // fused GroupNorm(+swish) input transform: separate instantiation, zero cost when off
        const int G = g.Cin >> 5;
        const int qs = sidx & 3, rs0 = sidx >> 2;            // 16-channel slice of the block, first halo row of this lane
        const int rows_up = (t.halo_rows + 31) & ~31;        // whole warps run every trip (__syncwarp inside)
        for (int work = cluster_id; work < total_work; work += num_clusters) {
            int hn0 = 0, hoy0 = 0, hox0 = 0, gvw = 0x7fffffff;
            if (gn) {
                tile_origin(work, hn0, hoy0, hox0);
                if (g.valid_w && hn0 < g.N) gvw = g.valid_w[hn0];
            }
            const int cb0 = work_ks(work) * t.cbps;
            for (int cbi = 0; cbi < t.cbps; ++cbi) {
                const int cb = cb0 + cbi;
                // Fused GroupNorm instantiation -- four lanes per halo row: lane slice qs owns fp32 chunks 2qs, 2qs+1 of both 128-byte boxes = channels [8qs, 8qs+8) and
                // [32+8qs, 32+8qs+8) of the block, i.e. exactly the 16-byte fp16 chunks qs and 4+qs of the hi and of the lo plane.
                // (Round 2, first version: one lane per row -- 180 rows on 128 lanes = two passes, the second 40 % full -- and, for the
                // fused GroupNorm, per-row global loads of mean / rstd and 48 table reads per row from shared memory, on the port that
                // bounds the kernel.)  The GroupNorm constants of the lane's 16 channels live in registers, loaded before the wait on
                // the halo so that their latency overlaps the TMA.
                float gm0 = 0.f, gm1 = 0.f, ga[16], gb[16];
                if (gn) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) { ga[e] = 0.f; gb[e] = 0.f; }
                    if (hn0 < g.N) {
                        const float2 mr0 = g.gn_mr[(size_t)hn0 * G + cb * 2], mr1 = g.gn_mr[(size_t)hn0 * G + cb * 2 + 1];
                        gm0 = mr0.x; gm1 = mr1.x;
#pragma unroll
                        for (int hlf = 0; hlf < 2; ++hlf)
#pragma unroll
                            for (int f = 0; f < 2; ++f) {
                                const int c0 = cb * KB + hlf * 32 + qs * 8 + f * 4;
                                const float4 gg = ldg4(g.gn_gamma + c0), be = ldg4(g.gn_beta + c0);
                                const float rs = hlf ? mr1.y : mr0.y;
                                ga[hlf * 8 + f * 4 + 0] = rs * gg.x; ga[hlf * 8 + f * 4 + 1] = rs * gg.y;
                                ga[hlf * 8 + f * 4 + 2] = rs * gg.z; ga[hlf * 8 + f * 4 + 3] = rs * gg.w;
                                gb[hlf * 8 + f * 4 + 0] = be.x; gb[hlf * 8 + f * 4 + 1] = be.y; gb[hlf * 8 + f * 4 + 2] = be.z; gb[hlf * 8 + f * 4 + 3] = be.w;
                            }
                    }
                }
                mbar_wait(bar(I_HF + hs), hph);
                if (sidx == 0) mark(2, work);            // halo landed -> split starts
                uint8_t* halo = smem + hs * t.halo_stage_bytes;
                if constexpr (!GN) {
                    // Plain split: ONE lane per halo row (two passes over <= 208 rows, the second partly idle).  Same-box A/B (driver
                    // arguments, tools/gpu_run32.sh): the four-lanes-per-row form below spends ~35 % more issue slots on the same work (per-trip
                    // overhead on 16 instead of 64 channels; no idle warps) and costs the feed warps 0.11 ms per line; without a transform to
                    // hide there is nothing to gain from it.
                    for (int rho = sidx; rho < t.halo_rows; rho += 128) {
                        uint8_t* row0 = halo + rho * 128;
                        uint8_t* row1 = row0 + t.box_bytes;
                        const int sw = rho & 7;
                        uint32_t hi[32], lo[32];
#pragma unroll
                        for (int box = 0; box < 2; ++box) {
                            const uint8_t* bsrc = box ? row1 : row0;
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                float4 v = *reinterpret_cast<const float4*>(bsrc + ((j ^ sw) << 4));
                                v.x *= xs; v.y *= xs; v.z *= xs; v.w *= xs;
                                amax = fmaxf(fmaxf(amax, fabsf(v.x)), fmaxf(fabsf(v.y), fmaxf(fabsf(v.z), fabsf(v.w))));   // 4 FMNMX (|.| is a free modifier)
                                const float h0 = __uint_as_float(__float_as_uint(v.x) & mask), h1 = __uint_as_float(__float_as_uint(v.y) & mask);
                                const float h2 = __uint_as_float(__float_as_uint(v.z) & mask), h3 = __uint_as_float(__float_as_uint(v.w) & mask);
                                const int c = box * 16 + j * 2;
                                if (bf) {
                                    hi[c] = pack_bf16(h0, h1); hi[c + 1] = pack_bf16(h2, h3);
                                    lo[c] = pack_bf16(v.x - h0, v.y - h1); lo[c + 1] = pack_bf16(v.z - h2, v.w - h3);
                                } else {
                                    hi[c] = pack_f16(h0, h1); hi[c + 1] = pack_f16(h2, h3);
                                    lo[c] = pack_f16(v.x - h0, v.y - h1); lo[c + 1] = pack_f16(v.z - h2, v.w - h3);
                                }
                            }
                        }
                        // all 256 B of this row are in registers now: overwrite it (row0 <- hi plane, row1 <- lo plane)
#pragma unroll
                        for (int jj = 0; jj < 8; ++jj) {
                            *reinterpret_cast<uint4*>(row0 + ((jj ^ sw) << 4)) = make_uint4(hi[4 * jj], hi[4 * jj + 1], hi[4 * jj + 2], hi[4 * jj + 3]);
                            *reinterpret_cast<uint4*>(row1 + ((jj ^ sw) << 4)) = make_uint4(lo[4 * jj], lo[4 * jj + 1], lo[4 * jj + 2], lo[4 * jj + 3]);
                        }
                    }
                } else
                for (int rho = rs0; rho < rows_up; rho += 32) {
                    const bool live = rho < t.halo_rows;
                    uint8_t* row0 = halo + rho * 128;
                    uint8_t* row1 = row0 + t.box_bytes;
                    const int sw = rho & 7;
                    const uint32_t o0 = (uint32_t)((2 * qs) ^ sw) << 4, o1 = (uint32_t)((2 * qs + 1) ^ sw) << 4;
                    float4 v[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (live) {
                        v[0] = *reinterpret_cast<const float4*>(row0 + o0); v[1] = *reinterpret_cast<const float4*>(row0 + o1);
                        v[2] = *reinterpret_cast<const float4*>(row1 + o0); v[3] = *reinterpret_cast<const float4*>(row1 + o1);
                    }
                    // fused GroupNorm(+swish): which pixel is this halo row, is it inside the image / the valid window?
                    bool inside = true;
                    if (gn) {
                        const int hy = rho / t.HWd, hx = rho - hy * t.HWd;          // one sample per tile (plan: TN == 1)
                        const int y = hoy0 - t.ph + hy, x = hox0 - t.pw + hx;
                        inside = hn0 < g.N && (unsigned)y < (unsigned)g.H && (unsigned)x < (unsigned)g.W && x < gvw;
                    }
                    uint32_t hw[8], lw[8];          // hi / lo words: [0..3] = chunk qs, [4..7] = chunk 4+qs
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float tt[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
                        if (gn) {
                            const float mean = (k >> 1) ? gm1 : gm0;
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                float u = fmaf(tt[e] - mean, ga[k * 4 + e], gb[k * 4 + e]);
                                if (g.gn_swish) u = __fdividef(u, 1.f + __expf(-u));     // ex2.approx + rcp.approx: ~2e-7 relative on the sigmoid
                                tt[e] = inside ? u : 0.f;
                            }
                        }
#pragma unroll
                        for (int e = 0; e < 4; ++e) tt[e] *= xs;
                        amax = fmaxf(fmaxf(amax, fabsf(tt[0])), fmaxf(fabsf(tt[1]), fmaxf(fabsf(tt[2]), fabsf(tt[3]))));   // 4 FMNMX (|.| is a free modifier)
                        const float h0 = __uint_as_float(__float_as_uint(tt[0]) & mask), h1 = __uint_as_float(__float_as_uint(tt[1]) & mask);
                        const float h2 = __uint_as_float(__float_as_uint(tt[2]) & mask), h3 = __uint_as_float(__float_as_uint(tt[3]) & mask);
                        if (bf) {
                            hw[2 * k] = pack_bf16(h0, h1); hw[2 * k + 1] = pack_bf16(h2, h3);
                            lw[2 * k] = pack_bf16(tt[0] - h0, tt[1] - h1); lw[2 * k + 1] = pack_bf16(tt[2] - h2, tt[3] - h3);
                        } else {
                            hw[2 * k] = pack_f16(h0, h1); hw[2 * k + 1] = pack_f16(h2, h3);
                            lw[2 * k] = pack_f16(tt[0] - h0, tt[1] - h1); lw[2 * k + 1] = pack_f16(tt[2] - h2, tt[3] - h3);
                        }
                    }
                    // the four lanes of a row (same warp) have read all 256 bytes of it: overwrite in place (row0 <- hi plane, row1 <- lo plane).
                    // Odd rows store their upper chunk first: the two rows of a quarter-warp then hit disjoint banks.
                    __syncwarp();
                    if (live) {
                        const uint32_t ca = (uint32_t)(qs ^ sw) << 4, cb2 = (uint32_t)((4 + qs) ^ sw) << 4;
                        const uint4 ha = make_uint4(hw[0], hw[1], hw[2], hw[3]), hb = make_uint4(hw[4], hw[5], hw[6], hw[7]);
                        const uint4 la = make_uint4(lw[0], lw[1], lw[2], lw[3]), lb = make_uint4(lw[4], lw[5], lw[6], lw[7]);
                        // selects, not a branch: a divergent warp would issue every store twice with half the lanes (2x the wavefronts
                        // -- measured: +10 % LSU shared wavefronts on the roofline layer)
                        const bool odd = (rho & 1) != 0;
                        const uint32_t c1 = odd ? cb2 : ca, c2 = odd ? ca : cb2;
                        const uint4 h1 = odd ? hb : ha, h2 = odd ? ha : hb, l1 = odd ? lb : la, l2 = odd ? la : lb;
                        *reinterpret_cast<uint4*>(row0 + c1) = h1; *reinterpret_cast<uint4*>(row1 + c1) = l1;
                        *reinterpret_cast<uint4*>(row0 + c2) = h2; *reinterpret_cast<uint4*>(row1 + c2) = l2;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // these generic writes precede the next TMA refill
                if (sidx == 0) mark(3, work);            // split done
                mbar_arrive(bar(I_SD + hs));
                if (++hs == (uint32_t)HS) { hs = 0; hph ^= 1; }
            }
        }
        conv_range_report(g, __float_as_uint(amax), t.prec == MN_PREC_F16X3_TC || t.prec == MN_PREC_F16X1_TC);
        }
    } else if (warp == 1) {
      if (CG == 1 || crank == 0) {
        // =========================== MMA issuer (whole warp converged, one elected lane issues) ===========================
        const uint32_t fmt = (t.prec == MN_PREC_BF16X3_TC) ? 1u : 0u;
        const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(NT >> 3) << 17) | ((uint32_t)((128 * CG) >> 4) << 24);
        const bool three = t.prec != MN_PREC_F16X1_TC;
        const int num_kb = t.cbps * t.taps;
        const uint64_t desc_hi0 = make_b_desc(smem_base + off_b);           // stage 0, hi plane, k-step 0
        uint32_t as = 0, aph = 0, bs = 0, bph = 0, tcnt = 0;
        for (int work = cluster_id; work < total_work; work += num_clusters, ++tcnt) {
            const uint32_t acc_st = ACC_ST == 2 ? (tcnt & 1) : 0u, acc_ph = ACC_ST == 2 ? ((tcnt >> 1) & 1) : (tcnt & 1);
            const uint32_t d_addr = tmem_base + acc_st * 2 * NT;
            mbar_wait(bar(I_ACCE + acc_st), acc_ph ^ 1);   // epilogue has drained this accumulator stage
            if (lane == 0) mark(6, work);                  // accumulator free -> MMAs of this tile may start
            tc_fence_after();
            for (int kb = 0; kb < num_kb; ++kb) {
                mbar_wait(bar(I_CD + as), aph);
                mbar_wait(bar(I_BF + bs), bph);
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint64_t dh0 = desc_hi0 + (uint64_t)((bs * B_STAGE) >> 4);   // start-address field is in 16-byte units
                    const uint64_t dl0 = dh0 + (uint64_t)(B_HALF >> 4);
                    const uint32_t a_hi = tmem_base + A_COL0 + as * 64;
#pragma unroll
                    for (int j = 0; j < KB / 16; ++j) {
                        if (CG == 2) {
                            tc_mma_ts_cg2(d_addr, a_hi + j * 8, dh0 + 2 * j, idesc, (kb | j) != 0);
                            if (three) {
                                tc_mma_ts_cg2(d_addr + NT, a_hi + j * 8, dl0 + 2 * j, idesc, (kb | j) != 0);
                                tc_mma_ts_cg2(d_addr + NT, a_hi + 32 + j * 8, dh0 + 2 * j, idesc, 1);
                            }
                        } else {
                            tc_mma_ts(d_addr, a_hi + j * 8, dh0 + 2 * j, idesc, (kb | j) != 0);
                            if (three) {
                                tc_mma_ts(d_addr + NT, a_hi + j * 8, dl0 + 2 * j, idesc, (kb | j) != 0);
                                tc_mma_ts(d_addr + NT, a_hi + 32 + j * 8, dh0 + 2 * j, idesc, 1);
                            }
                        }
                    }
                    if (CG == 2) {
                        tc_commit_mc_cg2(bar(I_AE + as), cmask);
                        tc_commit_mc_cg2(bar(I_BE + bs), cmask);
                    } else {
                        tc_commit(bar(I_AE + as));
                        if (cs > 1) tc_commit_mc(bar(I_BE + bs), cmask);
                        else tc_commit(bar(I_BE + bs));
                    }
                }
                __syncwarp();
                if (++as == A_STAGES) { as = 0; aph ^= 1; }
                if (++bs == (uint32_t)BS) { bs = 0; bph ^= 1; }
            }
            if (elect_one_sync()) { mark(7, work); if (CG == 2) tc_commit_mc_cg2(bar(I_ACCF + acc_st), cmask); else tc_commit(bar(I_ACCF + acc_st)); }   // last MMA of the tile issued
            __syncwarp();
        }
      }
    } else {
        // =========================== TMEM feed: shifted rows of the split halo -> A operand ===========================
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const int tn = r / (t.TH * t.TW);
        const int rem = r - tn * (t.TH * t.TW);
        const int th = rem / t.TW, tw = rem - th * t.TW;
        const int rho0 = tn < t.TN ? (tn * t.HHt + th) * t.HWd + tw : 0;   // halo row of tap (0,0); unused MMA rows read row 0
        uint32_t hs = 0, hph = 0, as = 0, aph = 0;
        for (int work = cluster_id; work < total_work; work += num_clusters) {
            for (int cb = 0; cb < t.cbps; ++cb) {
                mbar_wait(bar(I_SD + hs), hph);
                if (r == 0) mark(4, work);               // split halo visible -> feed of this channel block starts
                const uint8_t* halo = smem + hs * t.halo_stage_bytes;
                // Software-pipelined: the shared-memory reads of tap t+1 are issued right after the TMEM stores of tap t, so
                // their latency hides behind tcgen05.wait::st + the arrive (the register WAR hazard is the scoreboard's job).
                uint32_t hi[32], lo[32];
                auto load_tap = [&](int rho) {
                    const uint8_t* hsrc = halo + rho * 128;
                    const uint8_t* lsrc = hsrc + t.box_bytes;
                    const int sw = rho & 7;
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                        const uint4 a = *reinterpret_cast<const uint4*>(hsrc + ((jj ^ sw) << 4));
                        const uint4 b = *reinterpret_cast<const uint4*>(lsrc + ((jj ^ sw) << 4));
                        hi[4 * jj] = a.x; hi[4 * jj + 1] = a.y; hi[4 * jj + 2] = a.z; hi[4 * jj + 3] = a.w;
                        lo[4 * jj] = b.x; lo[4 * jj + 1] = b.y; lo[4 * jj + 2] = b.z; lo[4 * jj + 3] = b.w;
                    }
                };
                int ky = 0, kx = 0;
                load_tap(rho0);
                for (int tap = 0; tap < t.taps; ++tap) {
                    mbar_wait(bar(I_AE + as), aph ^ 1);
                    if (r == 0 && cb * t.taps + tap < 24) mark(16 + cb * t.taps + tap, work);          // A stage free
                    tc_fence_after();
                    const uint32_t a_dst = lane_addr + A_COL0 + as * 64;
#pragma unroll
                    for (int c = 0; c < 4; ++c) tc_st8(a_dst + c * 8, hi + c * 8);
#pragma unroll
                    for (int c = 0; c < 4; ++c) tc_st8(a_dst + 32 + c * 8, lo + c * 8);
                    if (tap + 1 < t.taps) {
                        if (++kx == t.KW) { kx = 0; ++ky; }
                        load_tap(rho0 + ky * t.HWd + kx);
                    }
                    tc_wait_st();
                    if (r == 0 && cb * t.taps + tap < 24) mark(40 + cb * t.taps + tap, work);          // TMEM stores of this tap complete
                    tc_fence_before();
                    if (CG == 2) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive_cluster(mapa_u32(bar(I_CD + as), 0));
                    } else {
                        mbar_arrive(bar(I_CD + as));
                    }
                    if (++as == A_STAGES) { as = 0; aph ^= 1; }
                }
                if (r == 0) mark(5, work);               // all taps of this channel block fed
                mbar_arrive(bar(I_HE + hs));         // all taps of this channel block have been read
                if (++hs == (uint32_t)HS) { hs = 0; hph ^= 1; }
            }

        }
    }
    tc_fence_before();
    __syncthreads();
    if (cs > 1) cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        if (CG == 2) tmem_dealloc_cg2(tmem_base, TMEM_COLS2); else tmem_dealloc(tmem_base, TMEM_COLS2);
    }
}

// ------------------------------------------------------------------------------------ weight packing
__global__ void absmax_kernel(const float* __restrict__ w, int64_t n, float* __restrict__ out) {
    float m = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(w[i]));
    m = mn_warp_max(m);
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<int*>(out), __float_as_int(m));   // m >= 0: int order == float order
}

// w: [taps*Cin][Cout] fp32 (the SIMT layout) -> hi/lo 16-bit [taps][Cout][Cin] scaled by 2^S; scale[0] = absmax in,
// scale[1] = 2^-S out.
__global__ void pack_tc_kernel(const float* __restrict__ w, int taps, int Cin, int Cout, int bf, uint16_t* __restrict__ hi,
                               uint16_t* __restrict__ lo, float* __restrict__ scale) {
    const float amax = scale[0];
    int e = 0;
    if (amax > 0.f) { frexpf(amax, &e); }                 // amax = f * 2^e, f in [0.5,1)
    const int S = bf ? 0 : (14 - e);                      // |w| * 2^S < 2^14
    const float up = ldexpf(1.f, S);
    if (blockIdx.x == 0 && threadIdx.x == 0) scale[1] = ldexpf(1.f, -S);
    const int64_t total = (int64_t)taps * Cin * Cout;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % Cin);
        const int64_t rest = i / Cin;
        const int o = (int)(rest % Cout);
        const int tap = (int)(rest / Cout);
        const float v = w[((size_t)tap * Cin + c) * Cout + o] * up;
        if (bf) {
            const __nv_bfloat16 h = __float2bfloat16_rn(v);
            const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
            hi[i] = *reinterpret_cast<const uint16_t*>(&h); lo[i] = *reinterpret_cast<const uint16_t*>(&l);
        } else {
            const __half h = __float2half_rn(v);
            const __half l = __float2half_rn(v - __half2float(h));
            hi[i] = *reinterpret_cast<const uint16_t*>(&h); lo[i] = *reinterpret_cast<const uint16_t*>(&l);
        }
    }
}

// ------------------------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode2() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

long long* g_tc2_trace = nullptr;      // mn_debug_tc2_trace

struct Tc2Plan { bool ok; const char* why; int NT; int smem; Tc2Geom t; };

bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

Tc2Plan plan_tc2(const ConvGeom& g) {
    Tc2Plan p{};
    auto fail = [&](const char* w) { p.ok = false; p.why = w; return p; };
    if (g.sh != 1 || g.sw != 1) return fail("stride != 1");
    const bool k3 = g.KH == 3 && g.KW == 3 && g.ph == 1 && g.pw == 1, k1 = g.KH == 1 && g.KW == 1 && g.ph == 0 && g.pw == 0;
    if (!k3 && !k1) return fail("only 3x3/pad1 and 1x1/pad0");
    if (g.Cin % KB != 0) return fail("Cin % 64 != 0");
    if (g.Cout % 64 != 0) return fail("Cout % 64 != 0");
    if (g.x_cs % 4 != 0 || (reinterpret_cast<uintptr_t>(g.x) & 15)) return fail("x alignment");
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if ((g.y && (g.y_cs % 4 || !al16(g.y))) || (g.y2 && (g.y2_cs % 4 || !al16(g.y2))) || (g.residual && (g.res_cs % 4 || !al16(g.residual))) ||
        (g.out_scale && (g.os_stride % 4 || !al16(g.out_scale))) || (g.y2_scale && (g.y2s_stride % 4 || !al16(g.y2_scale))) ||
        (g.bias && !al16(g.bias)))
        return fail("epilogue operands must be 16-byte aligned with channel strides that are multiples of 4");
    Tc2Geom& t = p.t;
    t.TH = g.H < 8 ? g.H : 8;
    if (!is_pow2(t.TH) || g.H % t.TH) return fail("H must be a multiple of 8 (or a power of two below 8)");
    const int maxw = 128 / t.TH;
    t.TW = g.W < maxw ? g.W : maxw;
    if (!is_pow2(t.TW) || g.W % t.TW) return fail("W must be a multiple of 128/TH (or a power of two below it)");
    t.TN = 128 / (t.TH * t.TW);
    t.ph = g.ph; t.pw = g.pw; t.KW = g.KW;
    t.HHt = t.TH + 2 * g.ph; t.HWd = t.TW + 2 * g.pw;
    // tiny images (4x4): 8 whole images per tile would need a 288-row halo; use fewer images per tile and leave the upper
    // TMEM lanes of the 128-row MMA unused (their rows map outside the tensor and are masked in the epilogue).
    while (t.TN > 1 && t.TN * t.HHt * t.HWd > 208) t.TN >>= 1;
    t.halo_rows = t.TN * t.HHt * t.HWd;
    if (t.halo_rows > 208) return fail("halo tile too large for shared memory");
    if ((g.y2_ptrs || g.gn_stats_out) && t.TN != 1)
        return fail("per-sample output pointers / epilogue GroupNorm statistics need samples of at least one whole pixel tile (OH*OW >= 128)");
    if (g.gn_mr && t.TN != 1) return fail("fused GroupNorm input transform needs samples of at least one whole pixel tile (H*W >= 128)");
    if (t.HWd > 256 || t.HHt > 256 || t.TN > 256) return fail("TMA box dim");
    t.box_bytes = (t.halo_rows * 128 + 1023) & ~1023;
    t.halo_stage_bytes = 2 * t.box_bytes;
    t.tiles_w = g.W / t.TW; t.tiles_h = g.H / t.TH; t.tiles_n = (g.N + t.TN - 1) / t.TN;
    t.m_tiles = t.tiles_w * t.tiles_h * t.tiles_n;
    t.cblocks = g.Cin / KB; t.taps = g.KH * g.KW;
    // 128-wide channel tiles unless that leaves most SMs idle (small-M layers at batch 1: ResNet 8x512 maps, 8x8 / 16x16
    // generator layers): then 64-wide tiles double the number of work items.
    static int nt_items = -1;       // developer knob: CTAs a 128-wide tiling must keep busy (MN_TC_NT_ITEMS, default 120)
    if (nt_items < 0) { const char* e = getenv("MN_TC_NT_ITEMS"); nt_items = e ? atoi(e) : 120; }
    p.NT = (g.Cout % 128 == 0 && (int64_t)((t.m_tiles + 1) / 2) * (g.Cout / 128) * 2 >= nt_items) ? 128 : 64;
    t.n_tiles = g.Cout / p.NT;
    static int force_cs = -1;
    if (force_cs < 0) { const char* e = getenv("MN_TC_CLUSTER"); force_cs = e ? atoi(e) : 0; }
    t.cs = force_cs > 0 ? force_cs : (t.m_tiles >= 2 ? 2 : 1);
    if (t.cs != 1 && t.cs != 2 && t.cs != 4) t.cs = 1;
    if ((p.NT / t.cs) % 8 != 0) t.cs = 1;
    t.m_groups = (t.m_tiles + t.cs - 1) / t.cs;
    // split-K: few tiles but a deep K loop (4x4 / 8x8 generator layers, ResNet stages at batch 1) -> spread the channel blocks of
    // a tile over several CTAs; partial sums go to the caller's workspace and conv_splitk_reduce_kernel finishes the job.
    t.ksplit = 1;
    {
        const int items = t.m_groups * t.n_tiles, slots = mn_num_sms() / t.cs;
        while (t.ksplit * 2 * items <= slots && t.cblocks % (t.ksplit * 2) == 0 && t.cblocks / (t.ksplit * 2) >= 1 && t.ksplit < 8) t.ksplit *= 2;
        while (t.ksplit > 1 && (int64_t)t.ksplit * g.M * g.Cout * 4 > g.ws_bytes) t.ksplit >>= 1;
        if (t.ksplit > 1 && (!g.ws || g.gn_mr || (g.Cout & 3) || g.y2_ptrs || g.gn_stats_out)) t.ksplit = 1;
    }
    t.cbps = t.cblocks / t.ksplit;
    // cta_group::2 pairs (see the kernel): default whenever the cluster has 2 CTAs; MN_TC_CG=1 forces the cta_group::1 + multicast path
    static int force_cg = -1;
    if (force_cg < 0) { const char* e = getenv("MN_TC_CG"); force_cg = e ? atoi(e) : 0; }
    t.cg = (t.cs == 2 && force_cg != 1) ? 2 : 1;
    // halo ring depth: a third stage when it still leaves >= 3 weight stages (cta_group::2 halves the weight stage) and the tile's
    // K loop is short (<= 4 channel blocks): then the whole next tile's halos are in flight while this tile computes.
    static int force_hs = -1, force_epi = -2;
    if (force_hs < 0) { const char* e = getenv("MN_TC_HALO_STAGES"); force_hs = e ? atoi(e) : 0; }
    if (force_epi < -1) { const char* e = getenv("MN_TC_EPI_CB"); force_epi = e ? atoi(e) : -1; }
    const int b_stage_bytes = 2 * (p.NT / t.cg) * 128;
    const int other = STG_BYTES + 1024 + 256 + 1024;
    t.hstages = 2;
    {
        const bool fits3 = 3 * t.halo_stage_bytes + other + 3 * b_stage_bytes <= SMEM_LIMIT;
        if (force_hs == 3 ? fits3 : (force_hs == 0 && fits3 && t.cbps <= 4 && t.cbps >= 2)) t.hstages = 3;
    }
    const int fixed = t.hstages * t.halo_stage_bytes + other;
    int bs = (SMEM_LIMIT - fixed) / b_stage_bytes;
    if (bs > MAX_BSTAGES) bs = MAX_BSTAGES;
    if (bs < 2) return fail("not enough shared memory for 2 weight stages");
    // epilogue of tile i after splitting channel block `epi_cb` of tile i+1 (its halos must fit the ring beside the running tile's)
    t.epi_cb = t.cbps > 1 ? 1 : 0;
    if (force_epi >= 0 && force_epi < t.cbps && force_epi < t.hstages) t.epi_cb = force_epi;
    t.bstages = bs;
    p.smem = fixed + bs * b_stage_bytes;
    p.ok = true;
    return p;
}

template <int NT, bool GN, int CG>
int launch_tc2(const CUtensorMap& ma, const CUtensorMap& mbh, const CUtensorMap& mbl, const ConvGeom& g, const Tc2Plan& p, cudaStream_t st) {
    static unsigned long long smem_done = 0;
    MN_CUDA_CHECK(mn_ensure_dyn_smem(conv_tc2_kernel<NT, GN, CG>, SMEM_LIMIT, &smem_done));
    const Tc2Geom& t = p.t;
    const int total_work = t.m_groups * t.n_tiles * t.ksplit;
    int sms = mn_num_sms();
    if (mn_max_ctas() > 0 && mn_max_ctas() < sms) sms = mn_max_ctas();
    int clusters = sms / t.cs;
    if (clusters < 1) clusters = 1;
    if (clusters > total_work) clusters = total_work;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(clusters * t.cs, 1, 1);
    cfg.blockDim = dim3(NUM_THREADS2, 1, 1);
    cfg.dynamicSmemBytes = p.smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = t.cs; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    static int pdl = -1;
    if (pdl < 0) { const char* e = getenv("MN_TC_PDL"); pdl = (e && e[0] == '0') ? 0 : 1; }
    cfg.attrs = attr; cfg.numAttrs = (pdl && mn_pdl_enabled()) ? 2 : 1;
    MN_CUDA_CHECK(cudaLaunchKernelEx(&cfg, conv_tc2_kernel<NT, GN, CG>, ma, mbh, mbl, g, t));
    return MN_OK;
}

}  // namespace

// Developer hook (tools/trace_tc2.py): zeroed device buffer of 1 + 64*64 int64 -- while installed, CTA 0 of every conv_tc2 launch
// writes clock64() of event e of its tile iteration `it` to [1 + it*64 + e].  NULL uninstalls.  Not part of the product API.
extern "C" int mn_debug_tc2_trace(long long* device_buffer) { g_tc2_trace = device_buffer; return 0; }

int mn_conv_tc2_supported(const ConvGeom& g, const char** why) {
    Tc2Plan p = plan_tc2(g);
    if (why) *why = p.ok ? "" : p.why;
    return p.ok ? 1 : 0;
}

int mn_conv_tc2_launch(const ConvGeom& g, const void* w_hi, const void* w_lo, const float* w_scale, int prec, cudaStream_t st) {
    Tc2Plan p = plan_tc2(g);
    if (!p.ok) { mn_set_error("mn_conv2d_nhwc: tensor-core path does not support this shape (%s)", p.why); return MN_ERR_UNSUPPORTED; }
    if (!w_hi || !w_lo || !w_scale) { mn_set_error("mn_conv2d_nhwc: tensor-core precision needs packed w_tc_hi/w_tc_lo/w_tc_scale"); return MN_ERR_INVALID; }
    PFN_encodeTiled enc = get_encode2();
    if (!enc) { mn_set_error("cuTensorMapEncodeTiled not available from the driver"); return MN_ERR_CUDA; }
    CUtensorMap ma, mbh, mbl;
    Tc2Geom& t = p.t;
    {
        cuuint64_t dims[4] = {(cuuint64_t)g.Cin, (cuuint64_t)g.W, (cuuint64_t)g.H, (cuuint64_t)g.N};
        cuuint64_t strides[3] = {(cuuint64_t)g.x_cs * 4, (cuuint64_t)g.W * g.x_cs * 4, (cuuint64_t)g.H * g.W * g.x_cs * 4};
        cuuint32_t box[4] = {32, (cuuint32_t)t.HWd, (cuuint32_t)t.HHt, (cuuint32_t)t.TN};
        cuuint32_t es[4] = {1, 1, 1, 1};
        CUresult r = enc(&ma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(g.x), dims, strides, box, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { mn_set_error("cuTensorMapEncodeTiled(A halo) failed: %d", (int)r); return MN_ERR_CUDA; }
    }
    const CUtensorMapDataType dt = (prec == MN_PREC_BF16X3_TC) ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
    for (int which = 0; which < 2; ++which) {
        cuuint64_t dims[3] = {(cuuint64_t)g.Cin, (cuuint64_t)g.Cout, (cuuint64_t)(g.KH * g.KW)};
        cuuint64_t strides[2] = {(cuuint64_t)g.Cin * 2, (cuuint64_t)g.Cin * g.Cout * 2};
        cuuint32_t box[3] = {64, (cuuint32_t)(p.NT / t.cs), 1};
        cuuint32_t es[3] = {1, 1, 1};
        CUresult r = enc(which ? &mbl : &mbh, dt, 3, const_cast<void*>(which ? w_lo : w_hi), dims, strides, box, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { mn_set_error("cuTensorMapEncodeTiled(B) failed: %d", (int)r); return MN_ERR_CUDA; }
    }
    t.wscale = w_scale + 1;
    t.prec = prec;
    t.trace = g_tc2_trace;
    int rc;
    if (t.cg == 2) {
        if (g.gn_mr) rc = p.NT == 128 ? launch_tc2<128, true, 2>(ma, mbh, mbl, g, p, st) : launch_tc2<64, true, 2>(ma, mbh, mbl, g, p, st);
        else rc = p.NT == 128 ? launch_tc2<128, false, 2>(ma, mbh, mbl, g, p, st) : launch_tc2<64, false, 2>(ma, mbh, mbl, g, p, st);
    } else {
        if (g.gn_mr) rc = p.NT == 128 ? launch_tc2<128, true, 1>(ma, mbh, mbl, g, p, st) : launch_tc2<64, true, 1>(ma, mbh, mbl, g, p, st);
        else rc = p.NT == 128 ? launch_tc2<128, false, 1>(ma, mbh, mbl, g, p, st) : launch_tc2<64, false, 1>(ma, mbh, mbl, g, p, st);
    }
    if (rc != MN_OK || t.ksplit == 1) return rc;
    ConvGeom gr = g;
    gr.splits = t.ksplit;
    return mn_conv_splitk_reduce_launch(gr, st);
}

extern "C" int mn_conv_pack_weights_tc(const float* w, int taps, int Cin, int Cout, int precision, void* hi, void* lo,
                                       float* scale2, void* stream) {
    MN_REQUIRE(w && hi && lo && scale2 && taps > 0 && Cin > 0 && Cout > 0, "mn_conv_pack_weights_tc: bad args");
    MN_REQUIRE(precision == MN_PREC_F16X3_TC || precision == MN_PREC_BF16X3_TC || precision == MN_PREC_F16X1_TC,
               "mn_conv_pack_weights_tc: precision must be a tensor-core mode");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t total = (int64_t)taps * Cin * Cout;
    MN_CUDA_CHECK(cudaMemsetAsync(scale2, 0, 2 * sizeof(float), st));
    const int blocks = (int)(mn_cdiv64(total, 256) < 1184 ? mn_cdiv64(total, 256) : 1184);
    absmax_kernel<<<blocks, 256, 0, st>>>(w, total, scale2);
    MN_LAUNCH_CHECK();
    pack_tc_kernel<<<blocks, 256, 0, st>>>(w, taps, Cin, Cout, precision == MN_PREC_BF16X3_TC ? 1 : 0,
                                           reinterpret_cast<uint16_t*>(hi), reinterpret_cast<uint16_t*>(lo), scale2);
    MN_LAUNCH_CHECK();
    return MN_OK;
}
