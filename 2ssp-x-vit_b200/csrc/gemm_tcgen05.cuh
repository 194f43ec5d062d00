// Persistent, warp-specialised bf16 GEMM for sm_100a:   C[M,N] = A[M,K] * W[N,K]^T  (+ fused epilogue)
//
//   * operands: bf16, K-contiguous (activations [M,K] and nn.Linear weights [N,K] as they are),
//     staged by TMA (SWIZZLE_128B) into a STAGES-deep shared-memory ring;
//   * math: tcgen05.mma cta_group::1, 128 x BN x 16 per instruction, fp32 accumulators in TMEM,
//     double-buffered (2 x BN columns) so the epilogue of tile i overlaps the MMAs of tile i+1;
//   * CTAS = 2: the same kernel on CTA pairs (cluster of 2, tcgen05 cta_group::2): a pair owns a 256 x BN tile, each
//     CTA loads its 128 rows of A and HALF of the W tile (32 KB instead of 48 KB per 64-deep K slab: the operand
//     stream from L2 is what bounds the single-CTA form, profiles/gemm_operand_traffic_r1.txt), the leader's MMA
//     thread issues 256 x BN x 16 instructions that read both halves, and every CTA keeps the accumulator rows and
//     the whole epilogue of its own 128 rows;
//   * roles: warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, warps 4.. = epilogue
//     (each epilogue warp owns the 32 TMEM lanes of its quadrant and, with 8 warps, one half of the columns);
//   * epilogues (template MODE):
//       EPI_BF16            out bf16 = acc + bias                                  (QKV projection)
//       EPI_BF16_GELU       out bf16 = gelu(acc + bias)                            (fc1, no scoring)
//       EPI_BF16_GELU_SCORE same + per-(32-row sub-tile, image segment, neuron) sum of squares of the
//                           stored activations -> `partials` (2SSP Stage-1 score, reference
//                           src/vit_pruning.py:151-152: vector_norm over tokens, then sum over images)
//       EPI_BF16_GELU_SCORE_PRE  same but the squares are taken before GELU (timm hook point,
//                           src/vit_pruning.py:135)
//       EPI_F32             out fp32 (=|+=) acc + bias; "+=" is a TMA reduce-add into the fp32 residual
//                           stream, so the residual is never loaded by the SMs   (proj, fc2, patch-embed, head)
//       EPI_F32_SCALED      out fp32 (=|+=) col_scale[c] * (acc + bias[c])   (proj / fc2 of LayerScale blocks: timm
//                           LayerScale.forward multiplies the branch output by gamma before the residual add)
//       EPI_BF16_QGELU, EPI_BF16_QGELU_SCORE_PRE   EPI_BF16_GELU / EPI_BF16_GELU_SCORE_PRE with QuickGELU,
//                           x * sigmoid(1.702 x), in place of erf GELU (fc1 of the OpenAI CLIP image towers)
//     Output tiles leave through a 4 KB per-warp staging slot and TMA stores (clipped at the tensor edge).
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace tssp {

enum GemmMode : int {
    EPI_BF16 = 0,
    EPI_BF16_GELU = 1,
    EPI_BF16_GELU_SCORE = 2,
    EPI_BF16_GELU_SCORE_PRE = 3,
    EPI_F32 = 4,
    EPI_BF16_ROWNORM = 5,  // EPI_BF16 + per-(row, 64-column chunk) sum of squares (|q|^2, |k|^2 per head for attention)
    EPI_F32_SCALED = 6,    // EPI_F32 with a per-column scale applied after the bias (LayerScale)
    EPI_BF16_QGELU = 7,    // EPI_BF16_GELU with QuickGELU
    EPI_BF16_QGELU_SCORE_PRE = 8,  // EPI_BF16_GELU_SCORE_PRE with QuickGELU (the squares are taken before the activation)
};

// epilogues that write Stage-1 score partials (32-row sub-tile, image segment, neuron)
__host__ __device__ constexpr bool gemm_mode_scores(int mode) {
    return mode == EPI_BF16_GELU_SCORE || mode == EPI_BF16_GELU_SCORE_PRE || mode == EPI_BF16_QGELU_SCORE_PRE;
}

struct GemmParams {
    int M;                  // valid rows of A / C (rows >= M are never scored; stores clip at the tensor map)
    int N;                  // columns of C = rows of W (multiple of 8)
    int K;                  // reduction length (multiple of 8)
    const float* bias;      // [N] or nullptr
    float* partials;        // SCORE modes: [ceil(M/32)][2][ldp] fp32 sum of squares
    int ldp;                // row pitch of partials (>= N)
    int tokens_per_image;   // T (>= 32): rows of one image are contiguous in A
    int reduce_add;         // EPI_F32: 1 => C += tile, 0 => C = tile
    float* rownorm;         // EPI_BF16_ROWNORM: [M][ld_rownorm] fp32, entry (row, c) = sum of squares of columns [64c, 64c+64)
    int ld_rownorm;
    int rownorm_chunks;     // only chunks c < rownorm_chunks are written (Q and K heads, not V)
    int reverse;            // 1 => walk the tile sequence from the last tile to the first (same tiles, same results):
                            //      a consumer that starts where its producer stopped finds those rows still in L2
    long long* trace;       // diagnostics (tssp_debug_gemm_trace): clock64() stamps of CTA 0, or nullptr
    const float* col_scale; // EPI_F32_SCALED: [N] per-column factor (kept last: the other instances read the fields above
                            //      at the same parameter offsets as before it existed)
};

// Trace layout: 16 int64 per tile, first GEMM_TRACE_TILES tiles of CTA 0. Slots 0-1: MMA thread (accumulator buffer
// granted, last MMA of the tile committed); 2-3: TMA thread (first / last K slab of the tile requested); 4-11: epilogue
// warp 0 (tile's accumulator ready, first TMEM half arrived, slot free, both halves staged, store issued, score pass
// done, partials written, buffer handed back); 12-15: the same warp's second chunk (halves staged ... handed back).
constexpr int GEMM_TRACE_TILES = 24;
#define GEMM_TRACE(cond, tile_it, slot_)                                                                  \
    do {                                                                                                  \
        if (p.trace != nullptr && blockIdx.x == 0 && (cond) && (tile_it) < GEMM_TRACE_TILES)              \
            p.trace[(tile_it) * 16 + (slot_)] = clock64();                                                \
    } while (0)

template <int MODE, int BN_, int STAGES_, int EPI_WARPS_, int CTAS_ = 1>
struct GemmCfg {
    static constexpr int CTAS = CTAS_;  // CTAs cooperating on one MMA (1, or 2 = CTA pair)
    static constexpr int BM = 128;      // rows per CTA
    static constexpr int BN = BN_;
    static constexpr int BK = 64;  // 128 B of bf16 = one SWIZZLE_128B row
    static constexpr int STAGES = STAGES_;
    static constexpr int EPI_WARPS = EPI_WARPS_;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_ROWS = BN / CTAS;  // rows of the W tile this CTA loads
    static constexpr int B_BYTES = B_ROWS * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int SLOT_BYTES = 4096;  // 32 rows x 128 B
    static constexpr int BAR_BYTES = 256;
    static constexpr int SMEM_BYTES = 1024 + STAGES * STAGE_BYTES + EPI_WARPS * SLOT_BYTES + BAR_BYTES;
    static constexpr int THREADS = 128 + 32 * EPI_WARPS;
    static constexpr int TMEM_COLS = 2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512));  // allocations are powers of two
    static constexpr bool OUT_BF16 = (MODE != EPI_F32 && MODE != EPI_F32_SCALED);
    static constexpr int CHUNK_COLS = OUT_BF16 ? 64 : 32;  // columns per 128-byte staging row
    static constexpr int CHUNKS = BN / CHUNK_COLS;
    static constexpr int COL_GROUPS = EPI_WARPS / 4;        // column halves handled by different warps
    static constexpr int CHUNKS_PER_WARP = CHUNKS / COL_GROUPS;
    static_assert(CTAS == 1 || CTAS == 2, "one CTA or a CTA pair");
    static_assert(EPI_WARPS == 4 || EPI_WARPS == 8, "whole warpgroups: every group covers the 4 TMEM lane quadrants");
    // More epilogue warps were measured and do not pay for the fused fc1 (profiles/gemm_trace_r2.txt, profiles/epilogue_probe_r2.txt):
    // its epilogue is bound by instruction issue -- ~13 issue cycles per element, a packed FFMA2 / FADD2 costs two -- which a
    // sub-partition's warps share, plus ~0.8 k clk of barrier round trips per tile that only a third accumulator buffer could
    // hide (TMEM holds two 256-column fp32 buffers). Sixteen warps on 256-column tiles (96 registers): 7.36 -> 7.82 k clk per
    // tile. Twelve warps on 192-column tiles (128 registers, one chunk per warp): 5.80 k clk per 192 columns = 7.74 k per 256,
    // 5 % slower at ViT-B (K = 768) and 6 % faster at ViT-S (K = 384). A setmaxnreg hand-over for 16 warps is refused by ptxas.
    // The two warpgroups on ALTERNATE tiles (each all 256 columns of its own tile and accumulator buffer, so that the two warps
    // of a sub-partition sit at different points of their tiles and fill each other's barrier / TMEM-load / store latencies):
    // bit-identical and slower -- fc1 + GELU + score 72.8 -> 81.1 us at K = 384, 187 -> 209 us at K = 768, 301 -> 323 us at
    // K = 1024 (profiles/epilogue_alt_tiles_r2.txt): a group holds its buffer for a whole drain, the MMA issuer waits for it.
    static_assert(BN % 16 == 0 && BN >= 64 && BN <= 256 && BN % CHUNK_COLS == 0, "BN: a UMMA N (multiple of 16, <= 256) made of whole staging chunks");
    static_assert((BN / CTAS) % 8 == 0, "each CTA loads whole 8-row swizzle atoms of W");
    static_assert(CHUNKS % COL_GROUPS == 0, "chunks must split evenly over the column groups");
    static_assert(SMEM_BYTES <= 232448, "shared memory budget (227 KB) exceeded");
};

// gelu(x) = x Phi(x) = max(x, 0) - |x| q(|x|),  q(a) = Phi(-a) = 0.5 erfc(a / sqrt 2)   (no cancellation on either side),
// with q(a) = 2^P(a), P a **degree-5** polynomial fit of log2 q (Lawson-weighted least squares on a <= 5; max |error| 2.4e-4
// in log2 q). Its leading coefficient is NEGATIVE, so beyond the fitted interval P keeps falling and 2^P underflows to 0 by
// itself: no clamp of |x| (round 1: degree 6 and min(|x|, 6.5)). Against the erf form: |gelu error| <= 2.3e-5 absolute (at
// x = 1.1, i.e. 2.3e-5 relative there), <= 1.1e-4 relative for x > 0 and <= 1.6e-4 relative for -5 <= x < 0 -- a twelfth of a
// bf16 half-ulp; below -5 both are < 1.5e-6 in magnitude.
// Pipes: the five Horner steps and the final multiply-add are packed FFMA2 (FMA pipe), 2^P is one MUFU.EX2, max(x, 0) one
// FMNMX on the ALU pipe. The epilogue is bound by instruction ISSUE, ~13 cycles per element with a packed operation
// costing two (tools/epi_probe.cu, profiles/epilogue_probe_r2.txt): a form that also replaced the FMNMX by packed adds on
// half arguments (y = x/2, max(x,0) = y + |y|) had fewer instructions and was 5 % slower.
__device__ __forceinline__ void gelu_erf_x2(float& x0, float& x1) {
    using namespace ptx;
    const float a0 = fabsf(x0), a1 = fabsf(x1);
    const uint64_t a = pack_f32x2(a0, a1);
    uint64_t pl = fma_f32x2(a, pack_f32x2(-2.69913406e-04f, -2.69913406e-04f), pack_f32x2(5.29729575e-03f, 5.29729575e-03f));
    pl = fma_f32x2(pl, a, pack_f32x2(-4.63191196e-02f, -4.63191196e-02f));
    pl = fma_f32x2(pl, a, pack_f32x2(-4.66907829e-01f, -4.66907829e-01f));
    pl = fma_f32x2(pl, a, pack_f32x2(-1.147788644f, -1.147788644f));
    pl = fma_f32x2(pl, a, pack_f32x2(-1.00022835788f, -1.00022835788f));
    float p0, p1;
    unpack_f32x2(pl, p0, p1);
    const uint64_t q = pack_f32x2(ex2_approx(p0), ex2_approx(p1));
    const uint64_t r = fma_f32x2(pack_f32x2(-a0, -a1), q, pack_f32x2(fmaxf(x0, 0.0f), fmaxf(x1, 0.0f)));
    unpack_f32x2(r, x0, x1);
}

// quickgelu(x) = x * sigmoid(1.702 x) = x / (1 + 2^(-1.702 log2(e) x)): one MUFU.EX2 and one MUFU.RCP per element, plus
// an FMUL and an FADD with immediate operands and the final FMUL. (The same with packed FMUL2 / FADD2 needs the constants in
// register pairs: in the 168-register epilogue it spilled 12 bytes more than this form, in both modes.) Both approximations are within a few fp32 ulps, so the result is
// within a fraction of a bf16 ulp of the exact value for |x| <= 50 (below about -51, 1 + 2^y exceeds 2^126 and the
// reciprocal flushes to zero: the result is -0 instead of a value under 1e-36). The one-MUFU form
// 0.5 x (1 + tanh.approx(0.851 x)) is not used: tanh.approx has about 2^-11 relative error and 1 + tanh cancels for
// negative x (4 % off at x = -3).
__device__ __forceinline__ void quick_gelu_x2(float& x0, float& x1) {
    using namespace ptx;
    constexpr float K = -2.45546696f;  // -1.702 * log2(e)
    x0 = x0 * rcp_approx(1.0f + ex2_approx(K * x0));
    x1 = x1 * rcp_approx(1.0f + ex2_approx(K * x1));
}

__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }

template <int MODE, int BN, int STAGES, int EPI_WARPS, int CTAS = 1>
__global__ void __launch_bounds__(GemmCfg<MODE, BN, STAGES, EPI_WARPS, CTAS>::THREADS, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ CUtensorMap tmap_c, const GemmParams p) {
    using Cfg = GemmCfg<MODE, BN, STAGES, EPI_WARPS, CTAS>;
    using namespace ptx;
    extern __shared__ uint8_t smem_raw[];

    const uint32_t warp_idx = threadIdx.x >> 5;
    const uint32_t lane = threadIdx.x & 31;

    const uint32_t raw_addr = smem_u32(smem_raw);
    const uint32_t base = (raw_addr + 1023u) & ~1023u;  // SWIZZLE_128B tiles need 1024-byte alignment
    const uint32_t slot_base = base + STAGES * Cfg::STAGE_BYTES;
    const uint32_t bar_base = slot_base + EPI_WARPS * Cfg::SLOT_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * STAGES + 2 + a); };
    const uint32_t tmem_slot_addr = bar_base + 8u * (2 * STAGES + 4);
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot_addr - raw_addr));

    // A tile is (CTAS * 128) x BN; a pair walks the same tile sequence, CTA `cta_rank` owning 128-row block
    // m_blk = CTAS * (tile / num_n_blks) + cta_rank of it.
    const uint32_t cta_rank = CTAS == 2 ? cluster_ctarank() : 0u;
    const int tile_first = CTAS == 2 ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
    const int tile_step = CTAS == 2 ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
    const int num_m_blks = (p.M + Cfg::BM * CTAS - 1) / (Cfg::BM * CTAS);
    const int num_n_blks = (p.N + BN - 1) / BN;
    const int num_tiles = num_m_blks * num_n_blks;
    const int num_kb = (p.K + Cfg::BK - 1) / Cfg::BK;

    if (warp_idx == 0 && lane == 0) {
        prefetch_tensormap(&tmap_a);
        prefetch_tensormap(&tmap_b);
        prefetch_tensormap(&tmap_c);
    }
    if (warp_idx == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull_bar(a), 1);
            mbar_init(tempty_bar(a), EPI_WARPS * CTAS);  // the leader's copy collects the epilogue warps of both CTAs
        }
        fence_mbar_init();
    }
    if (warp_idx == 2) {
        if constexpr (CTAS == 2) {
            tmem_alloc_pair(tmem_slot_addr, Cfg::TMEM_COLS);
            tmem_relinquish_pair();
        } else {
            tmem_alloc(tmem_slot_addr, Cfg::TMEM_COLS);
            tmem_relinquish();
        }
    }
    tc_fence_before();
    if constexpr (CTAS == 2) cluster_sync();  // the peer's barriers must be initialised before anything signals them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    // the prologue above may have overlapped the previous kernel's tail; from here on its output is read / overwritten
    griddep_launch_dependents();
    griddep_wait();

    if (warp_idx == 0) {
        // ===================== TMA producer =====================
        if (elect_one_sync()) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = tile_first; tile < num_tiles; tile += tile_step) {
                const int t = p.reverse ? num_tiles - 1 - tile : tile;
                const int m_blk = (t / num_n_blks) * CTAS + static_cast<int>(cta_rank);
                const int n_blk = t % num_n_blks;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1u);
                    if (kb == 0) GEMM_TRACE(true, (tile - tile_first) / tile_step, 2);
                    if (kb == num_kb - 1) GEMM_TRACE(true, (tile - tile_first) / tile_step, 3);
                    const uint32_t sa = base + stage * Cfg::STAGE_BYTES;
                    const uint32_t sb = sa + Cfg::A_BYTES;
                    if constexpr (CTAS == 2) {
                        // both halves are counted on the leader's barrier; the leader announces the total
                        if (cta_rank == 0) mbar_expect_tx(full_bar(stage), 2 * Cfg::STAGE_BYTES);
                        tma_load_2d_pair(sa, &tmap_a, full_bar(stage), kb * Cfg::BK, m_blk * Cfg::BM);
                        tma_load_2d_pair(sb, &tmap_b, full_bar(stage), kb * Cfg::BK, n_blk * BN + static_cast<int>(cta_rank) * Cfg::B_ROWS);
                    } else {
                        mbar_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
                        tma_load_2d(sa, &tmap_a, full_bar(stage), kb * Cfg::BK, m_blk * Cfg::BM);
                        tma_load_2d(sb, &tmap_b, full_bar(stage), kb * Cfg::BK, n_blk * BN);
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp_idx == 1) {
        // ===================== MMA issuer (single thread) =====================
        if (cta_rank == 0 && elect_one_sync()) {  // of a pair only the leader issues MMAs (for both CTAs)
            constexpr uint32_t idesc = umma_idesc_bf16_f32(Cfg::BM * CTAS, BN);
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int tile = tile_first; tile < num_tiles; tile += tile_step, ++it) {
                const int as = it & 1;
                const uint32_t aphase = (it >> 1) & 1;
                mbar_wait(tempty_bar(as), aphase ^ 1u);  // epilogue has drained this accumulator buffer
                tc_fence_after();
                GEMM_TRACE(true, it, 0);
                const uint32_t d_tmem = tmem_base + as * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t sa = base + stage * Cfg::STAGE_BYTES;
                    const uint32_t sb = sa + Cfg::A_BYTES;
#pragma unroll
                    for (int k = 0; k < Cfg::BK / 16; ++k) {
                        const uint64_t adesc = umma_desc_k_sw128(sa + k * 32);
                        const uint64_t bdesc = umma_desc_k_sw128(sb + k * 32);
                        if constexpr (CTAS == 2) umma_bf16_ss_pair(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                        else umma_bf16_ss(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    // smem slot is free once these MMAs retire (in both CTAs of a pair)
                    if constexpr (CTAS == 2) umma_commit_pair(empty_bar(stage), 3u);
                    else umma_commit(empty_bar(stage));
                    if (++stage == STAGES) { stage = 0; phase ^= 1u; }
                }
                // accumulator complete -> epilogue (of both CTAs)
                if constexpr (CTAS == 2) umma_commit_pair(tfull_bar(as), 3u);
                else umma_commit(tfull_bar(as));
                GEMM_TRACE(true, it, 1);
            }
        }
    } else if (warp_idx >= 4) {
        // ===================== epilogue warps =====================
        const uint32_t e = warp_idx - 4;
        const uint32_t quad = warp_idx & 3;           // TMEM lane quadrant this warp may access
        const uint32_t col_group = e >> 2;            // which share of the columns (8-warp configs)
        const uint32_t slot = slot_base + e * Cfg::SLOT_BYTES;
        const uint32_t my_row = slot + lane * 128;
        const uint32_t sw = lane & 7;
        int it = 0;
        for (int tile = tile_first; tile < num_tiles; tile += tile_step, ++it) {
            const int t = p.reverse ? num_tiles - 1 - tile : tile;
            const int m_blk = (t / num_n_blks) * CTAS + static_cast<int>(cta_rank);
            const int n_blk = t % num_n_blks;
            const int as = it & 1;
            const uint32_t aphase = (it >> 1) & 1;
            mbar_wait(tfull_bar(as), aphase);
            tc_fence_after();
            GEMM_TRACE(e == 0 && lane == 0, it, 4);
            const uint32_t t_row = tmem_base + ((quad * 32u) << 16) + as * BN;
            const int row0 = m_blk * Cfg::BM + quad * 32;

            // The accumulator buffer goes back to the MMA issuer as soon as this warp's LAST TMEM load of the tile has landed
            // -- bias / GELU / staging / store / score pass of that chunk work on registers and shared memory. The next-but-one
            // tile's MMAs then start ~3 k clk earlier and are never what the epilogue waits for (the fused fc1 is bound by its
            // epilogue's own busy time: period 7.35 k -> 6.8 k clk per tile, profiles/gemm_trace_r2.txt).
            bool handed_back = false;
            auto hand_back = [&]() {
                tc_fence_before();
                __syncwarp();
                if (elect_one_sync()) {
                    if constexpr (CTAS == 2) mbar_arrive_cluster(tempty_bar(as), 0u);
                    else mbar_arrive(tempty_bar(as));
                }
                handed_back = true;
            };
            // image segmentation of this warp's 32 rows (SCORE modes)
            int seg_split = 0, seg_end = 0;
            if constexpr (gemm_mode_scores(MODE)) {
                const int valid = min(32, max(0, p.M - row0));
                const int img0 = row0 / p.tokens_per_image;
                seg_end = valid;
                seg_split = min(valid, (img0 + 1) * p.tokens_per_image - row0);
            }

            if constexpr (!Cfg::OUT_BF16) {
                // fp32 epilogue: 32-column chunks, the TMEM load of chunk c+1 in flight while chunk c is staged and stored
                uint32_t buf0[32], buf1[32];
                const int chunk_base = col_group * Cfg::CHUNKS_PER_WARP;
                tmem_ld_32x32b_x32_nowait(t_row + chunk_base * 32, buf0);
#pragma unroll
                for (int cc = 0; cc < Cfg::CHUNKS_PER_WARP; ++cc) {
                    uint32_t(&r)[32] = (cc & 1) ? buf1 : buf0;
                    uint32_t(&nx)[32] = (cc & 1) ? buf0 : buf1;
                    const int tile_col = (chunk_base + cc) * 32;
                    const int gcol0 = n_blk * BN + tile_col;
                    tmem_ld_fence(r);
                    if (cc + 1 < Cfg::CHUNKS_PER_WARP) tmem_ld_32x32b_x32_nowait(t_row + tile_col + 32, nx);
                    if (gcol0 < p.N && row0 < p.M) {  // warp-uniform
                        if constexpr (MODE == EPI_F32_SCALED) {
                            // gamma * (acc + bias) in fp32, then the residual add: timm's order of operations
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const int gc = gcol0 + j;
                                if (gc < p.N) {
                                    const float4 b4 = p.bias != nullptr ? __ldg(reinterpret_cast<const float4*>(p.bias + gc))
                                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                                    const float4 g4 = __ldg(reinterpret_cast<const float4*>(p.col_scale + gc));
                                    r[j + 0] = __float_as_uint(__fmul_rn(g4.x, __fadd_rn(__uint_as_float(r[j + 0]), b4.x)));
                                    r[j + 1] = __float_as_uint(__fmul_rn(g4.y, __fadd_rn(__uint_as_float(r[j + 1]), b4.y)));
                                    r[j + 2] = __float_as_uint(__fmul_rn(g4.z, __fadd_rn(__uint_as_float(r[j + 2]), b4.z)));
                                    r[j + 3] = __float_as_uint(__fmul_rn(g4.w, __fadd_rn(__uint_as_float(r[j + 3]), b4.w)));
                                }
                            }
                        } else if (p.bias != nullptr) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const int gc = gcol0 + j;
                                if (gc < p.N) {
                                    const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + gc));
                                    r[j + 0] = __float_as_uint(__uint_as_float(r[j + 0]) + b4.x);
                                    r[j + 1] = __float_as_uint(__uint_as_float(r[j + 1]) + b4.y);
                                    r[j + 2] = __float_as_uint(__uint_as_float(r[j + 2]) + b4.z);
                                    r[j + 3] = __float_as_uint(__uint_as_float(r[j + 3]) + b4.w);
                                }
                            }
                        }
                        if (elect_one_sync()) tma_store_wait_read<0>();
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            st_shared_v4(my_row + ((j ^ sw) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (elect_one_sync()) {
                            if (p.reduce_add) tma_reduce_add_2d(&tmap_c, slot, gcol0, row0);
                            else tma_store_2d(&tmap_c, slot, gcol0, row0);
                            tma_store_commit();
                        }
                    }
                }
            }
#pragma unroll 1
            for (int cc = 0; Cfg::OUT_BF16 && cc < Cfg::CHUNKS_PER_WARP; ++cc) {
                const int chunk = col_group * Cfg::CHUNKS_PER_WARP + cc;
                const int tile_col = chunk * Cfg::CHUNK_COLS;
                const int gcol0 = n_blk * BN + tile_col;
                if (gcol0 >= p.N || row0 >= p.M) break;  // warp-uniform: nothing of this chunk is inside C

                if constexpr (Cfg::OUT_BF16) {
                    constexpr bool GELU = (MODE == EPI_BF16_GELU || MODE == EPI_BF16_GELU_SCORE || MODE == EPI_BF16_GELU_SCORE_PRE);
                    constexpr bool QGELU = (MODE == EPI_BF16_QGELU || MODE == EPI_BF16_QGELU_SCORE_PRE);
                    constexpr bool PRE = (MODE == EPI_BF16_GELU_SCORE_PRE || MODE == EPI_BF16_QGELU_SCORE_PRE);
                    // non-PRE modes stage each half as soon as it is packed, so only 16 packed words are ever live;
                    // the PRE mode (rare path) keeps the whole chunk twice: pre-activation values and activations
                    uint32_t packed[PRE ? 32 : 16];
                    uint32_t packed_pre[PRE ? 32 : 1];
                    float rn0 = 0.f, rn1 = 0.f;
                    // both 32-column halves of the chunk are requested up front: the second TMEM load is in flight
                    // while the first half goes through bias / GELU. (Requesting the NEXT chunk's halves before this
                    // chunk's fence / store / score pass was measured slower: 7.36 -> 7.91 k clk per tile, the two live
                    // buffers cost the math phase more than the hidden TMEM latency returns.)
                    uint32_t ra[32], rb[32];
                    tmem_ld_32x32b_x32_nowait(t_row + tile_col, ra);
                    tmem_ld_32x32b_x32_nowait(t_row + tile_col + 32, rb);
                    // the previous TMA store must have finished reading the slot before a half is staged into it
                    if (elect_one_sync()) tma_store_wait_read<0>();
                    __syncwarp();
                    GEMM_TRACE(e == 0 && lane == 0 && cc == 0, it, 6);
                    // Interior chunks (all 64 columns inside C, bias present: every chunk of the ViT widths except the tail
                    // of a pruned fc1) read the bias with plain loads; the guarded form costs seven instructions per
                    // four elements in predicates, zeroing and address descriptors. Both branches are warp-uniform.
                    auto halves = [&](auto interior_tag) {
                    constexpr bool INTERIOR = decltype(interior_tag)::value;
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        uint32_t(&r)[32] = hh ? rb : ra;
                        const int po = PRE ? hh * 16 : 0;
                        tmem_ld_fence(r);
                        if (hh == 0) GEMM_TRACE(e == 0 && lane == 0 && cc == 0, it, 5);
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const int gc = gcol0 + hh * 32 + j;
                            float4 b4;
                            if constexpr (INTERIOR) {
                                b4 = __ldg(reinterpret_cast<const float4*>(p.bias + gc));
                            } else {
                                b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (p.bias != nullptr && gc < p.N) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + gc));
                            }
                            float v0, v1, v2, v3;
                            const uint64_t a01 = pack_f32x2(__uint_as_float(r[j + 0]), __uint_as_float(r[j + 1]));
                            const uint64_t a23 = pack_f32x2(__uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                            unpack_f32x2(add_f32x2(a01, pack_f32x2(b4.x, b4.y)), v0, v1);
                            unpack_f32x2(add_f32x2(a23, pack_f32x2(b4.z, b4.w)), v2, v3);
                            if constexpr (PRE) {  // timm hook point: before the GELU
                                packed_pre[hh * 16 + j / 2] = pack_bf16x2(v0, v1);
                                packed_pre[hh * 16 + j / 2 + 1] = pack_bf16x2(v2, v3);
                            }
                            if constexpr (MODE == EPI_BF16_ROWNORM) {
                                rn0 = fmaf(v0, v0, fmaf(v2, v2, rn0));
                                rn1 = fmaf(v1, v1, fmaf(v3, v3, rn1));
                            }
                            if constexpr (GELU) {
                                gelu_erf_x2(v0, v1);
                                gelu_erf_x2(v2, v3);
                            }
                            if constexpr (QGELU) {
                                quick_gelu_x2(v0, v1);
                                quick_gelu_x2(v2, v3);
                            }
                            packed[po + j / 2] = pack_bf16x2(v0, v1);
                            packed[po + j / 2 + 1] = pack_bf16x2(v2, v3);
                        }
                        if constexpr (!PRE) {
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                st_shared_v4(my_row + (((hh * 4 + j) ^ sw) << 4), packed[4 * j], packed[4 * j + 1], packed[4 * j + 2],
                                             packed[4 * j + 3]);
                        }
                    }
                    };
                    if (p.bias != nullptr && gcol0 + Cfg::CHUNK_COLS <= p.N) halves(std::true_type{});
                    else halves(std::false_type{});
                    // both halves of this chunk are in registers: if it is the warp's last chunk inside C, TMEM is done with
                    if (cc + 1 == Cfg::CHUNKS_PER_WARP || gcol0 + Cfg::CHUNK_COLS >= p.N) hand_back();
                    if constexpr (MODE == EPI_BF16_ROWNORM) {
                        const int row = row0 + static_cast<int>(lane);
                        const int c64 = gcol0 >> 6;
                        if (row < p.M && c64 < p.rownorm_chunks) p.rownorm[static_cast<size_t>(row) * p.ld_rownorm + c64] = rn0 + rn1;
                    }

                    // (lo, hi) column pair of this lane as packed fp32 accumulators: one FFMA2 per staged word
                    uint64_t acc0 = 0ull, acc1 = 0ull;
                    auto score_pass = [&]() {
                        // lane l owns columns (2l, 2l+1) of the chunk: one 32-bit word per staged row
                        const uint32_t word = slot + (lane & 3) * 4;
                        const uint32_t c16 = lane >> 2;
                        if (seg_split == 32) {
                            // common case (5 of 6 sub-tiles at T=197): all 32 rows belong to one image
                            // (four independent accumulator chains instead of this one were measured: no faster)
#pragma unroll
                            for (int r = 0; r < 32; ++r) {
                                const uint32_t w = ld_shared_u32(word + r * 128 + ((c16 ^ (r & 7)) << 4));
                                const uint64_t v = pack_f32x2(bf16_lo(w), bf16_hi(w));
                                acc0 = fma_f32x2(v, v, acc0);
                            }
                            return;
                        }
#pragma unroll 4
                        for (int r = 0; r < seg_split; ++r) {
                            const uint32_t w = ld_shared_u32(word + r * 128 + ((c16 ^ (r & 7)) << 4));
                            const uint64_t v = pack_f32x2(bf16_lo(w), bf16_hi(w));
                            acc0 = fma_f32x2(v, v, acc0);
                        }
#pragma unroll 4
                        for (int r = seg_split; r < seg_end; ++r) {
                            const uint32_t w = ld_shared_u32(word + r * 128 + ((c16 ^ (r & 7)) << 4));
                            const uint64_t v = pack_f32x2(bf16_lo(w), bf16_hi(w));
                            acc1 = fma_f32x2(v, v, acc1);
                        }
                    };

                    if constexpr (PRE) {
                        // timm hook point: the slot first carries the pre-activation values (score pass), then the
                        // activations for the store
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            st_shared_v4(my_row + ((j ^ sw) << 4), packed_pre[4 * j], packed_pre[4 * j + 1],
                                         packed_pre[4 * j + 2], packed_pre[4 * j + 3]);
                        __syncwarp();
                        score_pass();
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            st_shared_v4(my_row + ((j ^ sw) << 4), packed[4 * j], packed[4 * j + 1], packed[4 * j + 2],
                                         packed[4 * j + 3]);
                    }
                    GEMM_TRACE(e == 0 && lane == 0, it, cc == 0 ? 7 : 12);
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (elect_one_sync()) {
                        tma_store_2d(&tmap_c, slot, gcol0, row0);
                        tma_store_commit();
                    }
                    GEMM_TRACE(e == 0 && lane == 0, it, cc == 0 ? 8 : 13);
                    // (running the score pass BEFORE the fence + TMA store, so that its shared-memory reads do not meet the TMA unit's,
                    // was measured: no faster)
                    if constexpr (MODE == EPI_BF16_GELU_SCORE) score_pass();
                    GEMM_TRACE(e == 0 && lane == 0, it, cc == 0 ? 9 : 14);
                    if constexpr (gemm_mode_scores(MODE)) {
                        const int gc = gcol0 + 2 * lane;
                        if (gc < p.N && row0 < p.M) {
                            const size_t sub = static_cast<size_t>(row0 >> 5);
                            float* dst = p.partials + (sub * 2) * p.ldp + gc;
                            float2 s0, s1;
                            unpack_f32x2(acc0, s0.x, s0.y);
                            unpack_f32x2(acc1, s1.x, s1.y);
                            *reinterpret_cast<float2*>(dst) = s0;
                            *reinterpret_cast<float2*>(dst + p.ldp) = s1;
                        }
                    }
                    GEMM_TRACE(e == 0 && lane == 0, it, cc == 0 ? 10 : 15);
                }
            }
            // accumulator buffer drained: hand it back to the MMA issuer (the bf16 epilogues have done so already, right
            // after their last TMEM load)
            if (!handed_back) hand_back();
            GEMM_TRACE(e == 0 && lane == 0, it, 11);
        }
        if (elect_one_sync()) tma_store_wait_all<0>();
    }

    tc_fence_before();
    if constexpr (CTAS == 2) cluster_sync();  // nobody leaves while the peer may still signal or read this CTA
    else __syncthreads();
    if (warp_idx == 2) {
        tc_fence_after();
        if constexpr (CTAS == 2) tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
        else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

}  // namespace tssp
