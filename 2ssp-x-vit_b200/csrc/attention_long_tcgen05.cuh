// Multi-head self-attention for long ViT sequences (208 < T <= 1025, head_dim 64) on tcgen05 / TMEM, keys in tiles.
//
// The short-sequence kernel (attention_tcgen05.cuh) keeps a whole padded key row of S in TMEM and K / V of a head whole
// in shared memory; neither fits past 208 keys. This one streams K and V in tiles of 128 keys through a ring of stages
// and accumulates O in TMEM across key tiles. DESIGN.md section 3 has the layout and the budgets.
//
// Work unit = (image, head, group of up to 4 query tiles of 128 rows). All query tiles of a group share every K / V tile
// of the head, so K / V cross L2 -> shared memory once per group instead of once per query tile (T = 577: 2 groups for 5
// query tiles; T = 1025: 3 groups for 9). One persistent CTA per SM walks units blockIdx.x, + gridDim.x, ...
//
// Roles (384 threads): warp 0 producer (per-row softmax shifts of the unit, then TMA of Q and the K / V tiles), warp 1
// MMA issuer, warps 4-7 and 8-11 two softmax / output warpgroups (thread = query row = TMEM lane). The items of a unit
// (key tile j, query tile m: S = Q_m K_j^T, softmax, O_m += P V_j) alternate between two S buffers in TMEM, buffer b is
// served by warpgroup b, so the MMAs of the next item run under the exponentials of this one.
//
// Softmax shift: single pass with the Cauchy-Schwarz bound s_ij <= |q_i| max_j |k_j| (max over all T keys of the head),
// one shift per row that is valid for every key tile: the P of each tile is added into O without the running-max
// rescale of FlashAttention; only the row sum accumulates. A unit in which some row's bound exceeds ATC_BOUND_LOG2 runs
// an extra first sweep over its key tiles that computes S and the true row maxima only, then the normal sweep with that
// shift (the S MMAs are issued twice; no O rescale exists anywhere).
//
// TMEM (512 columns): S / P buffer 0 [0,128), buffer 1 [128,256) (P bf16 written in place over the first 64 columns),
// O of query tile m of the group [256 + 64 m, 320 + 64 m).
#pragma once
#include "attention_tcgen05.cuh"

namespace tssp {

struct AttnLongParams {
    int n_img, T, heads, D;
    int MT;             // query tiles computed per (image, head): ceil(T / 128), or 1 for the first tile only
    int n_groups;       // query-tile groups per (image, head), each <= ATL_MAX_G tiles
    int NKT;            // key tiles: ceil(T / 128)
    float scale_log2e;  // log2(e) / sqrt(head_dim)
    const float* norms;  // optional [n*T][ld_norms]: |q|^2 per head in columns [0, heads), |k|^2 in [heads, 2 heads)
    int ld_norms;
    const __nv_bfloat16* qkv;  // [n*T][3 D]: the norms are taken from here when `norms` is null
    int reverse;        // 1 => units are visited from the last to the first
};

constexpr int ATL_THREADS = 384;
constexpr int ATL_MAX_G = 4;           // query tiles per unit: 4 O accumulators of 64 columns next to two 128-column S buffers
constexpr int ATL_KT = 128;            // keys per tile
constexpr int ATL_STAGES = 3;          // K / V ring depth
constexpr int ATL_TILE_BYTES = 128 * 128;  // 128 rows x 64 bf16
constexpr int ATL_Q_BYTES = ATL_MAX_G * ATL_TILE_BYTES;
constexpr int ATL_STAGE_BYTES = 2 * ATL_TILE_BYTES;  // K tile, V tile
constexpr int ATL_OUT_SLOT_BYTES = 4096;             // 32 rows x 128 B per softmax warp
constexpr int ATL_ROWS = ATL_MAX_G * 128;            // query rows of a unit
// per-unit shared state, after the tiles: shifts (2 unit slots), row sums (2 unit parities x 2 warpgroups), row maxima
// (2 warpgroups), exact-route flags, barriers, TMEM address
constexpr int ATL_OFF_Q = 0;
constexpr int ATL_OFF_KV = ATL_OFF_Q + ATL_Q_BYTES;
constexpr int ATL_OFF_OUT = ATL_OFF_KV + ATL_STAGES * ATL_STAGE_BYTES;
constexpr int ATL_OFF_BOUND = ATL_OFF_OUT + 8 * ATL_OUT_SLOT_BYTES;
constexpr int ATL_OFF_SUM = ATL_OFF_BOUND + 2 * ATL_ROWS * 4;
constexpr int ATL_OFF_MAX = ATL_OFF_SUM + 2 * 2 * ATL_ROWS * 4;
constexpr int ATL_OFF_FLAG = ATL_OFF_MAX + 2 * ATL_ROWS * 4;
constexpr int ATL_OFF_BAR = ATL_OFF_FLAG + 16;
constexpr int ATL_SMEM_BYTES = 1024 + ATL_OFF_BAR + 256;
constexpr int ATL_S_COLS = 128;
constexpr int ATL_O_COL = 256;
constexpr int ATL_MAX_T = 1025;  // 9 query tiles = 3 groups of 3
static_assert(ATL_SMEM_BYTES <= 232448, "long attention shared memory budget exceeded");

enum {
    ALB_FULL_Q = 0, ALB_EMPTY_Q,
    ALB_FULL_KV, ALB_EMPTY_KV = ALB_FULL_KV + ATL_STAGES,
    ALB_INFO_FULL = ALB_EMPTY_KV + ATL_STAGES, ALB_INFO_EMPTY = ALB_INFO_FULL + 2,
    ALB_S_FULL = ALB_INFO_EMPTY + 2, ALB_P_FULL = ALB_S_FULL + 2,
    ALB_O_FULL = ALB_P_FULL + 2, ALB_O_FREE,
    ALB_COUNT
};
static_assert(ALB_COUNT * 8 + 4 <= 256, "barrier area");

// (image, head, group) of unit u, and the group's first query tile and tile count (the MT tiles split as evenly as possible)
struct AtlUnit { int img, head, m0, G; };
__device__ __forceinline__ AtlUnit atl_unit(const AttnLongParams& p, int u) {
    AtlUnit r;
    const int g = u % p.n_groups;
    const int rest = u / p.n_groups;
    r.head = rest % p.heads;
    r.img = rest / p.heads;
    const int base = p.MT / p.n_groups, rem = p.MT % p.n_groups;
    r.G = base + (g < rem ? 1 : 0);
    r.m0 = g * base + (g < rem ? g : rem);
    return r;
}

// squared L2 norm of 64 bf16 values in global memory (the stand-alone path: no norms from the QKV epilogue)
__device__ __forceinline__ float atl_row_norm2_global(const __nv_bfloat16* row) {
    const uint4* v = reinterpret_cast<const uint4*>(row);
    float n0 = 0.f, n1 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const uint4 w4 = __ldg(v + j);
        const uint32_t w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float lo = __uint_as_float(w[k] << 16), hi = __uint_as_float(w[k] & 0xFFFF0000u);
            n0 = fmaf(lo, lo, n0);
            n1 = fmaf(hi, hi, n1);
        }
    }
    return n0 + n1;
}

// |x|^2 of token r of image img, head `head`, for q (which = 0) or k (which = 1)
__device__ __forceinline__ float atl_norm2(const AttnLongParams& p, int img, int r, int head, int which) {
    const size_t row = static_cast<size_t>(img) * p.T + r;
    if (p.norms != nullptr) return __ldg(p.norms + row * p.ld_norms + which * p.heads + head);
    return atl_row_norm2_global(p.qkv + row * (3 * static_cast<size_t>(p.D)) + static_cast<size_t>(which) * p.D + head * 64);
}

// one 32-column chunk of a score row: p = 2^(s*scale - shift) packed to bf16 pairs, masked beyond `valid` columns when
// MASKED; the (even, odd) column sums accumulate in sum2 (same packed arithmetic as the short kernel)
template <bool MASKED>
__device__ __forceinline__ void atl_chunk_exp(const uint32_t (&r)[32], uint32_t (&pk)[16], int col0, int valid, uint64_t scale2,
                                              uint64_t nshift2, uint64_t& sum2) {
    using namespace ptx;
#pragma unroll
    for (int j = 0; j < 32; j += 2) {
        const uint64_t t = fma_f32x2(pack_f32x2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), scale2, nshift2);
        float a, b;
        unpack_f32x2(t, a, b);
        a = ex2_approx(a);
        b = ex2_approx(b);
        if (MASKED) {
            if (col0 + j >= valid) a = 0.f;
            if (col0 + j + 1 >= valid) b = 0.f;
        }
        sum2 = add_f32x2(sum2, pack_f32x2(a, b));
        pk[j >> 1] = pack_bf16x2(a, b);
    }
}

// exponentials of one 128-column S tile of this warp's rows, P written back as bf16 over its first 64 columns; returns
// the row's sum. The TMEM load of chunk c+1 is in flight while chunk c is processed.
template <bool MASKED>
__device__ __forceinline__ float atl_tile_exp(uint32_t region, int valid, float scale_log2e, float shift) {
    using namespace ptx;
    uint32_t a[32], b[32], pk[16];
    uint64_t sum2 = pack_f32x2(0.f, 0.f);
    const uint64_t scale2 = pack_f32x2(scale_log2e, scale_log2e), nshift2 = pack_f32x2(-shift, -shift);
    tmem_ld_32x32b_x32_nowait(region, a);
#pragma unroll
    for (int c = 0; c < 4; c += 2) {
        tmem_ld_fence(a);
        tmem_ld_32x32b_x32_nowait(region + (c + 1) * 32, b);
        atl_chunk_exp<MASKED>(a, pk, c * 32, valid, scale2, nshift2, sum2);
        tmem_st_32x32b_x16(region + c * 16, pk);  // P chunk c overwrites S columns [16c, 16c+16): already consumed
        tmem_ld_fence(b);
        if (c + 2 < 4) tmem_ld_32x32b_x32_nowait(region + (c + 2) * 32, a);
        atl_chunk_exp<MASKED>(b, pk, (c + 1) * 32, valid, scale2, nshift2, sum2);
        tmem_st_32x32b_x16(region + (c + 1) * 16, pk);
    }
    float e0, e1;
    unpack_f32x2(sum2, e0, e1);
    tmem_st_wait();
    return e0 + e1;
}

// maximum of one 128-column S tile of this warp's rows over the first `valid` columns
__device__ __forceinline__ float atl_tile_max(uint32_t region, int valid, float mx) {
    using namespace ptx;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(region + c * 32, r);
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (c * 32 + j < valid) mx = fmaxf(mx, __uint_as_float(r[j]));
    }
    return mx;
}

__global__ void __launch_bounds__(ATL_THREADS, 1)
attention_long_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_ctx,
                              const AttnLongParams p) {
    using namespace ptx;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t warp_idx = threadIdx.x >> 5;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t raw_addr = smem_u32(smem_raw);
    const uint32_t base = (raw_addr + 1023u) & ~1023u;
    uint8_t* const base_ptr = smem_raw + (base - raw_addr);
    const uint32_t sq = base + ATL_OFF_Q;
    const uint32_t skv = base + ATL_OFF_KV;
    const uint32_t out_base = base + ATL_OFF_OUT;
    float* const s_bound = reinterpret_cast<float*>(base_ptr + ATL_OFF_BOUND);  // [2 slots][ATL_ROWS]
    float* const s_sum = reinterpret_cast<float*>(base_ptr + ATL_OFF_SUM);      // [2 parities][2 warpgroups][ATL_ROWS]
    float* const s_max = reinterpret_cast<float*>(base_ptr + ATL_OFF_MAX);      // [2 warpgroups][ATL_ROWS]
    volatile int* const s_flag = reinterpret_cast<volatile int*>(base_ptr + ATL_OFF_FLAG);  // [2 slots]
    const uint32_t bar_base = base + ATL_OFF_BAR;
    auto bar = [&](int which) { return bar_base + 8u * which; };
    const uint32_t tmem_slot_addr = bar_base + 8u * ALB_COUNT;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + ATL_OFF_BAR + 8 * ALB_COUNT);

    const int num_units = p.n_img * p.heads * p.n_groups;

    if (warp_idx == 0 && lane == 0) {
        prefetch_tensormap(&tmap_qkv);
        prefetch_tensormap(&tmap_ctx);
    }
    if (warp_idx == 1 && lane == 0) {
        mbar_init(bar(ALB_FULL_Q), 1);
        mbar_init(bar(ALB_EMPTY_Q), 1);
        for (int s = 0; s < ATL_STAGES; ++s) {
            mbar_init(bar(ALB_FULL_KV + s), 1);
            mbar_init(bar(ALB_EMPTY_KV + s), 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar(ALB_INFO_FULL + i), 32);     // every producer lane, after its shift writes
            mbar_init(bar(ALB_INFO_EMPTY + i), 1 + 8); // the MMA issuer and the 8 softmax warps
            mbar_init(bar(ALB_S_FULL + i), 1);
            mbar_init(bar(ALB_P_FULL + i), 4);
        }
        mbar_init(bar(ALB_O_FULL), 1);
        mbar_init(bar(ALB_O_FREE), 8);
        fence_mbar_init();
    }
    if (warp_idx == 2) {
        tmem_alloc(tmem_slot_addr, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    griddep_launch_dependents();  // the next kernel's prologue may overlap this kernel's tail ...
    griddep_wait();               // ... as this one's did: qkv / norms are valid from here on

    const int unit0 = blockIdx.x, unit_step = gridDim.x;
    auto unit_at = [&](int unit) { return atl_unit(p, p.reverse ? num_units - 1 - unit : unit); };

    // warps 0-3 keep 96 registers per thread (at 72 the producer's unit loop spilled), the two softmax warpgroups grow to
    // 200: 96 * 128 + 200 * 256 = 63488 <= the 168 * 384 allocated at launch
    if (warp_idx < 4) setmaxnreg_dec<96>();  // one instruction for the whole warpgroup
    if (warp_idx == 0) {
        // ===================== producer: per-row shifts, then Q and the K / V ring =====================
        uint32_t it = 0, ring = 0;
        for (int unit = unit0; unit < num_units; unit += unit_step, ++it) {
            const AtlUnit un = unit_at(unit);
            const int slot = it & 1;
            // max over all T keys of |k|^2 of this head
            float kmax2 = 0.f;
            if (p.norms != nullptr) {
#pragma unroll 4
                for (int r = lane; r < p.T; r += 32) kmax2 = fmaxf(kmax2, atl_norm2(p, un.img, r, un.head, 1));
            } else {
#pragma unroll 1
                for (int r = lane; r < p.T; r += 32) kmax2 = fmaxf(kmax2, atl_norm2(p, un.img, r, un.head, 1));
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) kmax2 = fmaxf(kmax2, __shfl_xor_sync(0xffffffffu, kmax2, o));
            mbar_wait(bar(ALB_INFO_EMPTY + slot), ((it >> 1) & 1) ^ 1u);
            bool exact = false;
#pragma unroll 1
            for (int i = lane; i < un.G * 128; i += 32) {
                const int r = un.m0 * 128 + i;
                const float qn = r < p.T ? atl_norm2(p, un.img, r, un.head, 0) : 0.f;
                // 1.0001: the norms may have been taken before the bf16 rounding of q and k
                const float bound = sqrtf(qn * kmax2) * p.scale_log2e * 1.0001f;
                s_bound[slot * ATL_ROWS + i] = bound;
                exact |= bound > ATC_BOUND_LOG2;
            }
            exact = __any_sync(0xffffffffu, exact);
            if (lane == 0) s_flag[slot] = exact ? 1 : 0;
            __syncwarp();
            mbar_arrive(bar(ALB_INFO_FULL + slot));  // release: the shifts and the flag above are visible to the waiters

            const int npass = exact ? 2 : 1;
            for (int t = 0; t < npass * p.NKT; ++t, ++ring) {
                const int j = t % p.NKT;
                const int stage = ring % ATL_STAGES;
                mbar_wait(bar(ALB_EMPTY_KV + stage), ((ring / ATL_STAGES) & 1) ^ 1u);
                __syncwarp();
                if (elect_one_sync()) {
                    const uint32_t dst = skv + stage * ATL_STAGE_BYTES;
                    mbar_expect_tx(bar(ALB_FULL_KV + stage), ATL_STAGE_BYTES);
                    tma_load_3d(dst, &tmap_qkv, bar(ALB_FULL_KV + stage), p.D + un.head * 64, j * ATL_KT, un.img);
                    tma_load_3d(dst + ATL_TILE_BYTES, &tmap_qkv, bar(ALB_FULL_KV + stage), 2 * p.D + un.head * 64, j * ATL_KT, un.img);
                }
                __syncwarp();
                if (t == 0) {  // Q after the first K / V tile: that tile's load overlaps the previous unit's last S MMAs
                    mbar_wait(bar(ALB_EMPTY_Q), (it & 1) ^ 1u);
                    __syncwarp();
                    if (elect_one_sync()) {
                        mbar_expect_tx(bar(ALB_FULL_Q), un.G * ATL_TILE_BYTES);
                        for (int m = 0; m < un.G; ++m)
                            tma_load_3d(sq + m * ATL_TILE_BYTES, &tmap_qkv, bar(ALB_FULL_Q), un.head * 64, (un.m0 + m) * 128, un.img);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp_idx == 1) {
        // ===================== MMA issuer =====================
        if (elect_one_sync()) {
            const uint32_t idesc_s = umma_idesc_bf16_f32(128, ATL_KT);
            const uint32_t idesc_o = umma_idesc_bf16_f32(128, 64) | (1u << 16);  // B (= V) is MN-major
            uint32_t it = 0, ring = 0, item = 0;
            uint32_t p_phase = 0;  // bit b: parity of the next P_FULL completion of S buffer b
            for (int unit = unit0; unit < num_units; unit += unit_step, ++it) {
                const AtlUnit un = unit_at(unit);
                const int slot = it & 1;
                mbar_wait(bar(ALB_INFO_FULL + slot), (it >> 1) & 1);
                const bool exact = s_flag[slot] != 0;
                mbar_arrive(bar(ALB_INFO_EMPTY + slot));
                const int npass = exact ? 2 : 1;
                const int per_pass = p.NKT * un.G;
                const int total = npass * per_pass;
                mbar_wait(bar(ALB_FULL_Q), it & 1);
                tc_fence_after();
                // S of item i (key tile j = (i / G) % NKT, query tile m = i % G) into S buffer (item + i) & 1
                auto issue_s = [&](int i) {
                    const int t = i / un.G, m = i % un.G;
                    const uint32_t r = ring + t;
                    const uint32_t stage = r % ATL_STAGES;
                    if (m == 0) {
                        mbar_wait(bar(ALB_FULL_KV + stage), (r / ATL_STAGES) & 1);
                        tc_fence_after();
                    }
                    const uint32_t b = (item + i) & 1;
                    const uint64_t qdesc0 = umma_desc_k_sw128(sq + m * ATL_TILE_BYTES);
                    const uint64_t kdesc0 = umma_desc_k_sw128(skv + stage * ATL_STAGE_BYTES);
#pragma unroll
                    for (int k = 0; k < 4; ++k)  // +32 B per 16-element K step: +2 in the descriptor's address field
                        umma_bf16_ss(tmem_base + b * ATL_S_COLS, qdesc0 + 2 * k, kdesc0 + 2 * k, idesc_s, k != 0);
                    umma_commit(bar(ALB_S_FULL + b));
                    if (i == total - 1) umma_commit(bar(ALB_EMPTY_Q));  // Q may be refilled for the next unit
                };
                issue_s(0);
                for (int i = 0; i < total; ++i) {
                    // S of the next item goes into the other buffer, whose previous item's PV has already been issued
                    // (tcgen05 MMAs of one thread execute in issue order)
                    if (i + 1 < total) issue_s(i + 1);
                    const uint32_t b = (item + i) & 1;
                    mbar_wait(bar(ALB_P_FULL + b), (p_phase >> b) & 1u);  // P written (or, first sweep, the row maxima taken)
                    p_phase ^= 1u << b;
                    tc_fence_after();
                    const int t = i / un.G, m = i % un.G;
                    const uint32_t stage = (ring + t) % ATL_STAGES;
                    if (t >= (npass - 1) * p.NKT) {  // the normal sweep: O_m += P V_j
                        const int j = t - (npass - 1) * p.NKT;
                        if (j == 0 && m == 0) {
                            mbar_wait(bar(ALB_O_FREE), (it & 1) ^ 1u);  // the previous unit's O has been read out
                            tc_fence_after();
                        }
                        const uint64_t vdesc0 = umma_desc_mn_sw128(skv + stage * ATL_STAGE_BYTES + ATL_TILE_BYTES, ATL_TILE_BYTES);
#pragma unroll
                        for (int kk = 0; kk < ATL_KT / 16; ++kk)  // 16 keys = two 1024-byte groups of V rows: +128 in the address field
                            umma_bf16_ts(tmem_base + ATL_O_COL + m * 64, tmem_base + b * ATL_S_COLS + kk * 8, vdesc0 + 128 * kk, idesc_o,
                                         (j != 0 || kk != 0) ? 1u : 0u);
                    }
                    if (m == un.G - 1) umma_commit(bar(ALB_EMPTY_KV + stage));  // every item of this K / V tile is issued
                }
                umma_commit(bar(ALB_O_FULL));
                ring += npass * p.NKT;
                item += total;
            }
        }
    } else if (warp_idx >= 4) {
        // ===================== softmax + output warpgroups (thread = query row) =====================
        setmaxnreg_inc<200>();
        const int wg = (warp_idx - 4) >> 2;  // serves S buffer wg
        const uint32_t quad = warp_idx & 3;
        const int row = quad * 32 + lane;    // row of a 128-row tile
        const uint32_t lane_off = (quad * 32u) << 16;
        const uint32_t region = tmem_base + wg * ATL_S_COLS + lane_off;
        const uint32_t out_slot = out_base + (warp_idx - 4) * ATL_OUT_SLOT_BYTES;
        const uint32_t out_row = out_slot + lane * 128;
        const uint32_t sw = lane & 7;
        uint32_t it = 0, item = 0, uses = 0;
        for (int unit = unit0; unit < num_units; unit += unit_step, ++it) {
            const AtlUnit un = unit_at(unit);
            const int slot = it & 1;
            mbar_wait(bar(ALB_INFO_FULL + slot), (it >> 1) & 1);
            const bool exact = s_flag[slot] != 0;
            const float* bound = s_bound + slot * ATL_ROWS;
            float* my_sum = s_sum + (slot * 2 + wg) * ATL_ROWS;
            float* my_max = s_max + wg * ATL_ROWS;
            for (int m = 0; m < un.G; ++m) {
                my_sum[m * 128 + row] = 0.f;
                my_max[m * 128 + row] = -INFINITY;
            }
            const int npass = exact ? 2 : 1;
            const int per_pass = p.NKT * un.G;
            const int total = npass * per_pass;
#pragma unroll 1
            for (int i = 0; i < total; ++i) {
                if (((item + i) & 1) == static_cast<uint32_t>(wg)) {
                    const int t = i / un.G, m = i % un.G;
                    const bool max_sweep = t < (npass - 1) * p.NKT;
                    const int j = max_sweep ? t : t - (npass - 1) * p.NKT;
                    const int valid = p.T - j * ATL_KT;  // real keys in this tile (> 0); >= 128 means no masking
                    mbar_wait(bar(ALB_S_FULL + wg), uses & 1);
                    ++uses;
                    tc_fence_after();
                    const int idx = m * 128 + row;
                    if (max_sweep) {
                        my_max[idx] = atl_tile_max(region, valid, my_max[idx]);
                    } else {
                        float shift;
                        if (exact) shift = fmaxf(s_max[idx], s_max[ATL_ROWS + idx]) * p.scale_log2e;
                        else shift = bound[idx];
                        const float sum = valid >= ATL_KT ? atl_tile_exp<false>(region, valid, p.scale_log2e, shift)
                                                          : atl_tile_exp<true>(region, valid, p.scale_log2e, shift);
                        my_sum[idx] += sum;
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (elect_one_sync()) mbar_arrive(bar(ALB_P_FULL + wg));
                }
                // end of the first sweep: the row maxima of both warpgroups are complete
                if (exact && i == per_pass - 1) asm volatile("bar.sync 1, 256;" ::: "memory");
            }
            // both warpgroups' row sums are in shared memory; the shifts are no longer needed
            asm volatile("bar.sync 1, 256;" ::: "memory");
            __syncwarp();
            if (elect_one_sync()) mbar_arrive(bar(ALB_INFO_EMPTY + slot));
            mbar_wait(bar(ALB_O_FULL), it & 1);
            tc_fence_after();
            const float* sum0 = s_sum + (slot * 2 + 0) * ATL_ROWS;
            const float* sum1 = s_sum + (slot * 2 + 1) * ATL_ROWS;
#pragma unroll 1
            for (int m = wg; m < un.G; m += 2) {  // warpgroup wg writes out query tiles wg, wg + 2
                uint32_t o0[32], o1[32];
                const uint32_t ocol = tmem_base + lane_off + ATL_O_COL + m * 64;
                tmem_ld_32x32b_x32_nowait(ocol, o0);
                tmem_ld_32x32b_x32_nowait(ocol + 32, o1);
                tmem_ld_fence(o0);
                tmem_ld_fence(o1);
                const int row0 = (un.m0 + m) * 128 + static_cast<int>(quad) * 32;
                if (row0 < p.T) {  // warp-uniform; rows >= T inside the tile are clipped by the TMA store
                    const float inv = 1.0f / (sum0[m * 128 + row] + sum1[m * 128 + row]);
                    if (elect_one_sync()) tma_store_wait_read<0>();
                    __syncwarp();
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        st_shared_v4(out_row + ((q ^ sw) << 4),
                                     pack_bf16x2(__uint_as_float(o0[8 * q + 0]) * inv, __uint_as_float(o0[8 * q + 1]) * inv),
                                     pack_bf16x2(__uint_as_float(o0[8 * q + 2]) * inv, __uint_as_float(o0[8 * q + 3]) * inv),
                                     pack_bf16x2(__uint_as_float(o0[8 * q + 4]) * inv, __uint_as_float(o0[8 * q + 5]) * inv),
                                     pack_bf16x2(__uint_as_float(o0[8 * q + 6]) * inv, __uint_as_float(o0[8 * q + 7]) * inv));
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        st_shared_v4(out_row + (((4 + q) ^ sw) << 4),
                                     pack_bf16x2(__uint_as_float(o1[8 * q + 0]) * inv, __uint_as_float(o1[8 * q + 1]) * inv),
                                     pack_bf16x2(__uint_as_float(o1[8 * q + 2]) * inv, __uint_as_float(o1[8 * q + 3]) * inv),
                                     pack_bf16x2(__uint_as_float(o1[8 * q + 4]) * inv, __uint_as_float(o1[8 * q + 5]) * inv),
                                     pack_bf16x2(__uint_as_float(o1[8 * q + 6]) * inv, __uint_as_float(o1[8 * q + 7]) * inv));
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (elect_one_sync()) {
                        tma_store_3d(&tmap_ctx, out_slot, un.head * 64, row0, un.img);
                        tma_store_commit();
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (elect_one_sync()) mbar_arrive(bar(ALB_O_FREE));
            item += total;
        }
        if (elect_one_sync()) tma_store_wait_all<0>();
    }

    tc_fence_before();
    __syncthreads();
    if (warp_idx == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

}  // namespace tssp
