// Non-GEMM kernels of the 2SSP ViT hot path (sm_100a): HBM-bound row kernels, the Stage-1 score finisher and the
// top-1 counter (attention lives in attention_tcgen05.cuh, the Stage-1 neuron gather in gather.cuh).
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace tssp {

// ------------------------------------------------------------------------------------------------
// fp32 [rows, cols] (pitch ld_in) -> bf16 [rows_pad, cols_pad] (pitch ld_out), zero padded.
// Used once per weight matrix when a model is loaded (nn.Linear weights are already [N, K] K-major).
// ------------------------------------------------------------------------------------------------
// `scale` multiplies every element before the rounding (1 for every matrix except the averaged two-head classifier, which
// packs both heads at 0.5: a power of two, so bf16(0.5 w) == 0.5 bf16(w) barring subnormals).
__global__ void cast_pad_bf16_kernel(const float* __restrict__ in, int rows, int cols, int ld_in,
                                     __nv_bfloat16* __restrict__ out, int rows_pad, int cols_pad, int ld_out, float scale) {
    const long long total = static_cast<long long>(rows_pad) * cols_pad;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int r = static_cast<int>(i / cols_pad);
        const int c = static_cast<int>(i % cols_pad);
        const float v = (r < rows && c < cols) ? in[static_cast<size_t>(r) * ld_in + c] * scale : 0.0f;
        out[static_cast<size_t>(r) * ld_out + c] = __float2bfloat16_rn(v);
    }
}

// ------------------------------------------------------------------------------------------------
// Patch extraction for the patch-embedding GEMM (HF ViTPatchEmbeddings: Conv2d(C, D, P, stride P) ==
// GEMM over non-overlapping patches). pixels fp32 [n, C, H, W] -> A bf16 [n*T, C*P*P] where rows
// img*T + r, r < prefix, are the (all-zero) slots of the prefix tokens (CLS, then a DeiT distillation token or timm
// register tokens) and row
// img*T + prefix + (py*G + px) holds patch (py, px) flattened as (c, ky, kx) -- the order of
// Conv2d.weight.view(D, -1). Each thread converts 8 consecutive kx.
// ------------------------------------------------------------------------------------------------
__global__ void im2col_patches_kernel(const float* __restrict__ pixels, __nv_bfloat16* __restrict__ out, int n_img,
                                      int C, int H, int W, int P, int T, int prefix) {
    const int G = W / P;
    const int Kp = C * P * P;
    const int k8_per_row = Kp / 8;
    const long long total = static_cast<long long>(n_img) * T * k8_per_row;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int k8 = static_cast<int>(i % k8_per_row);
        const long long row = i / k8_per_row;
        const int t = static_cast<int>(row % T);
        const int img = static_cast<int>(row / T);
        uint4 packed = make_uint4(0u, 0u, 0u, 0u);
        if (t >= prefix) {
            const int patch = t - prefix;
            const int py = patch / G, px = patch % G;
            const int k = k8 * 8;
            const int c = k / (P * P);
            const int ky = (k / P) % P;
            const int kx = k % P;
            const float* src = pixels + ((static_cast<size_t>(img) * C + c) * H + (py * P + ky)) * W + px * P + kx;
            const float4 a = __ldg(reinterpret_cast<const float4*>(src));
            const float4 b = __ldg(reinterpret_cast<const float4*>(src + 4));
            __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y);
            __nv_bfloat162 p1 = __floats2bfloat162_rn(a.z, a.w);
            __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y);
            __nv_bfloat162 p3 = __floats2bfloat162_rn(b.z, b.w);
            packed.x = *reinterpret_cast<uint32_t*>(&p0);
            packed.y = *reinterpret_cast<uint32_t*>(&p1);
            packed.z = *reinterpret_cast<uint32_t*>(&p2);
            packed.w = *reinterpret_cast<uint32_t*>(&p3);
        }
        *reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * Kp + k8 * 8) = packed;
    }
}

// The same for patches whose width is not a multiple of 8 (P = 14: DINOv2): rows of `ld` = round_up(C*P*P, 8) elements,
// the columns past C*P*P written as zeros (the patch weight is padded the same way, so they add nothing to the GEMM).
// A patch row of 14 floats starts only 8-byte aligned, so each thread converts its 8 columns as four pairs: with P even a
// pair never straddles two patch rows and is one 64-bit load; with P odd the pair is two scalar loads.
__global__ void im2col_patches_padded_kernel(const float* __restrict__ pixels, __nv_bfloat16* __restrict__ out, int n_img,
                                             int C, int H, int W, int P, int T, int prefix, int ld) {
    const int G = W / P;
    const int PP = P * P;
    const int K = C * PP;
    const int k8_per_row = ld / 8;
    const long long total = static_cast<long long>(n_img) * T * k8_per_row;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int k8 = static_cast<int>(i % k8_per_row);
        const long long row = i / k8_per_row;
        const int t = static_cast<int>(row % T);
        const int img = static_cast<int>(row / T);
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (t >= prefix) {
            const int patch = t - prefix;
            const int py = patch / G, px = patch % G;
            const float* base = pixels + static_cast<size_t>(img) * C * H * W + static_cast<size_t>(py * P) * W + px * P;
            auto at = [&](int k) {
                const int c = k / PP, r = k - c * PP, ky = r / P, kx = r - ky * P;
                return base + (static_cast<size_t>(c) * H + ky) * W + kx;
            };
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = k8 * 8 + 2 * q;
                float v0 = 0.0f, v1 = 0.0f;
                if ((P & 1) == 0) {
                    if (k < K) {  // K even: k + 1 < K as well
                        const float2 f = __ldg(reinterpret_cast<const float2*>(at(k)));
                        v0 = f.x;
                        v1 = f.y;
                    }
                } else {
                    if (k < K) v0 = __ldg(at(k));
                    if (k + 1 < K) v1 = __ldg(at(k + 1));
                }
                __nv_bfloat162 p2 = __floats2bfloat162_rn(v0, v1);
                w[q] = *reinterpret_cast<uint32_t*>(&p2);
            }
        }
        *reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * ld + k8 * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// uint8 pixels [n, C, H, W] (C <= 4) normalised on the way in: x = (float(u) * rescale - mean[c]) / std[c], each step one
// IEEE fp32 operation (no FMA contraction, correctly rounded division), so the bf16 written is the one the fp32 kernels
// above write for the fp32 image (u.float() * rescale - mean) / std computed by torch.
struct PixelNorm {
    float rescale;
    float mean[4];
    float std[4];
};

__device__ __forceinline__ float normalize_u8(uint32_t u, float rescale, float mean, float std) {
    return __fdiv_rn(__fsub_rn(__fmul_rn(static_cast<float>(u), rescale), mean), std);
}

// v[c] with constant indices only: a runtime index into a kernel parameter would copy the struct to local memory.
__device__ __forceinline__ float pick4(const float (&v)[4], int c) { return c == 0 ? v[0] : c == 1 ? v[1] : c == 2 ? v[2] : v[3]; }

// The bf16 a pixel becomes depends only on (channel, byte): every block first fills a table of those C * 256 values in
// shared memory, then looks pixels up. One correctly rounded division per pixel made the kernel issue-bound, slower than
// the fp32 kernel it replaces. Every thread of the block reaches the barrier (the kernels do not return early).
__device__ __forceinline__ void fill_u8_table(uint16_t (&lut)[4][256], const PixelNorm& norm, int C) {
    for (int j = threadIdx.x; j < C * 256; j += blockDim.x) {
        const int c = j >> 8;
        const float x = normalize_u8(static_cast<uint32_t>(j & 255), norm.rescale, pick4(norm.mean, c), pick4(norm.std, c));
        lut[c][j & 255] = __bfloat16_as_ushort(__float2bfloat16_rn(x));
    }
    __syncthreads();
}

// Two table entries as one bf16x2 word, the first in the low half (as __floats2bfloat162_rn packs them).
__device__ __forceinline__ uint32_t pack2(uint16_t lo, uint16_t hi) { return static_cast<uint32_t>(lo) | (static_cast<uint32_t>(hi) << 16); }

// im2col_patches_kernel for uint8 pixels (P a multiple of 8): each thread's 8 columns are one 8-byte load.
__global__ void im2col_patches_u8_kernel(const uint8_t* __restrict__ pixels, __nv_bfloat16* __restrict__ out, int n_img,
                                         int C, int H, int W, int P, int T, int prefix, const PixelNorm norm) {
    __shared__ uint16_t lut[4][256];
    fill_u8_table(lut, norm, C);
    const int G = W / P;
    const int Kp = C * P * P;
    const int k8_per_row = Kp / 8;
    const long long total = static_cast<long long>(n_img) * T * k8_per_row;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int k8 = static_cast<int>(i % k8_per_row);
        const long long row = i / k8_per_row;
        const int t = static_cast<int>(row % T);
        const int img = static_cast<int>(row / T);
        uint4 packed = make_uint4(0u, 0u, 0u, 0u);
        if (t >= prefix) {
            const int patch = t - prefix;
            const int py = patch / G, px = patch % G;
            const int k = k8 * 8;
            const int c = k / (P * P);
            const int ky = (k / P) % P;
            const int kx = k % P;
            const uint8_t* src = pixels + ((static_cast<size_t>(img) * C + c) * H + (py * P + ky)) * W + px * P + kx;
            const uint2 raw = __ldg(reinterpret_cast<const uint2*>(src));
            const uint16_t* tc = lut[c];
            packed.x = pack2(tc[raw.x & 0xffu], tc[(raw.x >> 8) & 0xffu]);
            packed.y = pack2(tc[(raw.x >> 16) & 0xffu], tc[raw.x >> 24]);
            packed.z = pack2(tc[raw.y & 0xffu], tc[(raw.y >> 8) & 0xffu]);
            packed.w = pack2(tc[(raw.y >> 16) & 0xffu], tc[raw.y >> 24]);
        }
        *reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * Kp + k8 * 8) = packed;
    }
}

// im2col_patches_padded_kernel for uint8 pixels: with P even a column pair is one 2-byte load inside one channel (C*P*P
// and P*P are even), with P odd two byte loads, each looked up in its own channel's table.
__global__ void im2col_patches_padded_u8_kernel(const uint8_t* __restrict__ pixels, __nv_bfloat16* __restrict__ out, int n_img,
                                                int C, int H, int W, int P, int T, int prefix, int ld, const PixelNorm norm) {
    __shared__ uint16_t lut[4][256];
    fill_u8_table(lut, norm, C);
    const int G = W / P;
    const int PP = P * P;
    const int K = C * PP;
    const int k8_per_row = ld / 8;
    const long long total = static_cast<long long>(n_img) * T * k8_per_row;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int k8 = static_cast<int>(i % k8_per_row);
        const long long row = i / k8_per_row;
        const int t = static_cast<int>(row % T);
        const int img = static_cast<int>(row / T);
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (t >= prefix) {
            const int patch = t - prefix;
            const int py = patch / G, px = patch % G;
            const uint8_t* base = pixels + static_cast<size_t>(img) * C * H * W + static_cast<size_t>(py * P) * W + px * P;
            auto at = [&](int k, int& c) {
                c = k / PP;
                const int r = k - c * PP, ky = r / P, kx = r - ky * P;
                return base + (static_cast<size_t>(c) * H + ky) * W + kx;
            };
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int k = k8 * 8 + 2 * q;
                uint16_t v0 = 0, v1 = 0;  // bf16 +0
                int c0 = 0, c1 = 0;
                if ((P & 1) == 0) {
                    if (k < K) {  // K even: k + 1 < K as well
                        const uint32_t pair = __ldg(reinterpret_cast<const unsigned short*>(at(k, c0)));
                        v0 = lut[c0][pair & 0xffu];
                        v1 = lut[c0][pair >> 8];
                    }
                } else {
                    if (k < K) {
                        const uint8_t* p0 = at(k, c0);
                        v0 = lut[c0][__ldg(p0)];
                    }
                    if (k + 1 < K) {
                        const uint8_t* p1 = at(k + 1, c1);
                        v1 = lut[c1][__ldg(p1)];
                    }
                }
                w[q] = pack2(v0, v1);
            }
        }
        *reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * ld + k8 * 8) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// x[img*T + t, :] = table[t, :]   (table = position embeddings with the CLS token / conv bias folded in)
__global__ void broadcast_rows_kernel(const float* __restrict__ table, float* __restrict__ x, int n_img, int T, int D) {
    const int d4 = D / 4;
    const long long total = static_cast<long long>(n_img) * T * d4;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(i % d4);
        const long long row = i / d4;
        const int t = static_cast<int>(row % T);
        reinterpret_cast<float4*>(x)[i] = __ldg(reinterpret_cast<const float4*>(table) + static_cast<size_t>(t) * d4 + c);
    }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm over the last dim, fp32 in (row pitch in_stride elements) -> bf16 out (pitch D) or fp32 out (any pitch);
// D % 128 == 0, D <= 1024, or D = 192.
// ------------------------------------------------------------------------------------------------
// Persistent LayerNorm: a fixed grid (a multiple of the SM count) walks the rows, one warp per row, and every warp has the
// NEXT row's loads in flight while it reduces / normalises / stores the current one. A row is NSLAB slabs of 128 * VPL
// elements; a lane owns 4 * VPL consecutive elements of each slab:
//   VPL = 2 (D % 256 == 0: ViT-B 768, ViT-L 1024): two 128-bit loads and ONE 128-bit bf16 store per slab (full sectors);
//   VPL = 1 (odd multiples of 128: ViT-S 384): one 128-bit load and one 64-bit store per slab.
// gamma / beta stay in registers (re-reading them from L1 at D = 1024 to save 64 registers was measured slower -- the
// launcher gives that width three CTAs of 128 threads per SM instead).
// OutT = float: the same rows in fp32 (the pre-norm of CLIP towers, written back into the residual stream). Statistics and
// arithmetic are the same, so bf16(fp32 output) is the bf16 output bit for bit; out may equal x (a warp has loaded a whole
// row before it stores any of it, and no other warp touches that row).
template <int NSLAB, int VPL, typename OutT>
__device__ __forceinline__ void layernorm_slab_rows(const float* x, long long in_stride, const float* __restrict__ gamma,
                                                    const float* __restrict__ beta, OutT* out, long long out_stride, int rows,
                                                    float eps, int reverse, int stream_in) {
    constexpr int D = NSLAB * 128 * VPL;
    // stream_in: x is loaded with an L2 evict-first policy, so the normalised rows this kernel writes (what the next
    // GEMM starts on) are what stays in L2, not the residual rows it has finished with
    const uint64_t in_policy = ptx::l2_policy_evict_first();
    auto ldx = [&](const float4* p) { return stream_in ? ptx::ld_global_v4_hint(p, in_policy) : *p; };
    if (reverse) {  // walk the rows from the last to the first: re-base the pointers on the last row, negative pitch
        x += static_cast<size_t>(rows - 1) * in_stride;
        out += static_cast<size_t>(rows - 1) * out_stride;
    }
    const long long xs = reverse ? -in_stride : in_stride;
    const long long os = reverse ? -out_stride : out_stride;
    ptx::griddep_launch_dependents();
    ptx::griddep_wait();
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * (blockDim.x >> 5);
    const float4* g4 = reinterpret_cast<const float4*>(gamma);
    const float4* b4 = reinterpret_cast<const float4*>(beta);
    float4 gm[NSLAB][VPL], bt[NSLAB][VPL];
#pragma unroll
    for (int i = 0; i < NSLAB; ++i)
#pragma unroll
        for (int h = 0; h < VPL; ++h) {
            gm[i][h] = __ldg(g4 + (i * 32 + lane) * VPL + h);
            bt[i][h] = __ldg(b4 + (i * 32 + lane) * VPL + h);
        }
    float4 nxt[NSLAB][VPL];
    int row = warp_global;
    if (row < rows) {
        const float4* src = reinterpret_cast<const float4*>(x + row * xs);
#pragma unroll
        for (int i = 0; i < NSLAB; ++i)
#pragma unroll
            for (int h = 0; h < VPL; ++h) nxt[i][h] = ldx(src + (i * 32 + lane) * VPL + h);
    }
    for (; row < rows; row += warp_stride) {
        float4 v[NSLAB][VPL];
#pragma unroll
        for (int i = 0; i < NSLAB; ++i)
#pragma unroll
            for (int h = 0; h < VPL; ++h) v[i][h] = nxt[i][h];
        const int next_row = row + warp_stride;
        if (next_row < rows) {
            const float4* src = reinterpret_cast<const float4*>(x + next_row * xs);
#pragma unroll
            for (int i = 0; i < NSLAB; ++i)
#pragma unroll
                for (int h = 0; h < VPL; ++h) nxt[i][h] = ldx(src + (i * 32 + lane) * VPL + h);
        }
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) {
            float part = (v[i][0].x + v[i][0].y) + (v[i][0].z + v[i][0].w);
            if constexpr (VPL == 2) part += (v[i][1].x + v[i][1].y) + (v[i][1].z + v[i][1].w);
            sum += part;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const float mean = sum * (1.0f / D);
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < NSLAB; ++i)
#pragma unroll
            for (int h = 0; h < VPL; ++h) {
                const float a = v[i][h].x - mean, b = v[i][h].y - mean, c = v[i][h].z - mean, d = v[i][h].w - mean;
                sq += (a * a + b * b) + (c * c + d * d);
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        const float rstd = 1.0f / sqrtf(sq * (1.0f / D) + eps);
        OutT* dst = out + row * os;
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) {
            uint32_t pk[2 * VPL];
#pragma unroll
            for (int h = 0; h < VPL; ++h) {
                const float4 g = gm[i][h];
                const float4 bb = bt[i][h];
                // the same expressions in both forms, so that both contract to the same FFMAs
                if constexpr (sizeof(OutT) == 4) {
                    reinterpret_cast<float4*>(dst)[(i * 32 + lane) * VPL + h] =
                        make_float4((v[i][h].x - mean) * rstd * g.x + bb.x, (v[i][h].y - mean) * rstd * g.y + bb.y,
                                    (v[i][h].z - mean) * rstd * g.z + bb.z, (v[i][h].w - mean) * rstd * g.w + bb.w);
                } else {
                    __nv_bfloat162 lo = __floats2bfloat162_rn((v[i][h].x - mean) * rstd * g.x + bb.x, (v[i][h].y - mean) * rstd * g.y + bb.y);
                    __nv_bfloat162 hi = __floats2bfloat162_rn((v[i][h].z - mean) * rstd * g.z + bb.z, (v[i][h].w - mean) * rstd * g.w + bb.w);
                    pk[2 * h] = *reinterpret_cast<uint32_t*>(&lo);
                    pk[2 * h + 1] = *reinterpret_cast<uint32_t*>(&hi);
                }
            }
            if constexpr (sizeof(OutT) == 2) {
                if constexpr (VPL == 2) reinterpret_cast<uint4*>(dst)[i * 32 + lane] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                else reinterpret_cast<uint2*>(dst)[i * 32 + lane] = make_uint2(pk[0], pk[1]);
            }
        }
    }
}

template <int NSLAB, int VPL>
__global__ void __launch_bounds__(256) layernorm_bf16_slab_kernel(const float* __restrict__ x, long long in_stride,
                                                                  const float* __restrict__ gamma,
                                                                  const float* __restrict__ beta,
                                                                  __nv_bfloat16* __restrict__ out, int rows, float eps,
                                                                  int reverse, int stream_in) {
    layernorm_slab_rows<NSLAB, VPL>(x, in_stride, gamma, beta, out, NSLAB * 128 * VPL, rows, eps, reverse, stream_in);
}
template <int NSLAB, int VPL>
__global__ void __launch_bounds__(256) layernorm_f32_slab_kernel(const float* x, long long in_stride, const float* __restrict__ gamma,
                                                                 const float* __restrict__ beta, float* out, long long out_stride,
                                                                 int rows, float eps, int reverse, int stream_in) {
    layernorm_slab_rows<NSLAB, VPL>(x, in_stride, gamma, beta, out, out_stride, rows, eps, reverse, stream_in);
}

// The same persistent walk for widths that are a multiple of 64 but not of 128 (D = 192: DeiT-Ti, ViT-Ti): a row is
// NSLAB slabs of 64 elements, a lane owns two consecutive elements of each slab -- one 64-bit load and one bf16x2 (32-bit)
// store per slab, so a warp still reads and writes whole 256-byte / 128-byte rows of a slab.
template <int NSLAB, typename OutT>
__device__ __forceinline__ void layernorm_slab64_rows(const float* x, long long in_stride, const float* __restrict__ gamma,
                                                      const float* __restrict__ beta, OutT* out, long long out_stride, int rows,
                                                      float eps, int reverse, int stream_in) {
    constexpr int D = NSLAB * 64;
    const uint64_t in_policy = ptx::l2_policy_evict_first();
    auto ldx = [&](const float2* p) { return stream_in ? ptx::ld_global_v2_hint(p, in_policy) : *p; };
    if (reverse) {
        x += static_cast<size_t>(rows - 1) * in_stride;
        out += static_cast<size_t>(rows - 1) * out_stride;
    }
    const long long xs = reverse ? -in_stride : in_stride;
    const long long os = reverse ? -out_stride : out_stride;
    ptx::griddep_launch_dependents();
    ptx::griddep_wait();
    const int lane = threadIdx.x & 31;
    const int warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int warp_stride = gridDim.x * (blockDim.x >> 5);
    const float2* g2 = reinterpret_cast<const float2*>(gamma);
    const float2* b2 = reinterpret_cast<const float2*>(beta);
    float2 gm[NSLAB], bt[NSLAB];
#pragma unroll
    for (int i = 0; i < NSLAB; ++i) {
        gm[i] = __ldg(g2 + i * 32 + lane);
        bt[i] = __ldg(b2 + i * 32 + lane);
    }
    float2 nxt[NSLAB];
    int row = warp_global;
    if (row < rows) {
        const float2* src = reinterpret_cast<const float2*>(x + row * xs);
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) nxt[i] = ldx(src + i * 32 + lane);
    }
    for (; row < rows; row += warp_stride) {
        float2 v[NSLAB];
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) v[i] = nxt[i];
        const int next_row = row + warp_stride;
        if (next_row < rows) {
            const float2* src = reinterpret_cast<const float2*>(x + next_row * xs);
#pragma unroll
            for (int i = 0; i < NSLAB; ++i) nxt[i] = ldx(src + i * 32 + lane);
        }
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) sum += v[i].x + v[i].y;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const float mean = sum * (1.0f / D);
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) {
            const float a = v[i].x - mean, b = v[i].y - mean;
            sq += a * a + b * b;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        const float rstd = 1.0f / sqrtf(sq * (1.0f / D) + eps);
        OutT* dst = out + row * os;
#pragma unroll
        for (int i = 0; i < NSLAB; ++i) {
            if constexpr (sizeof(OutT) == 4) {
                reinterpret_cast<float2*>(dst)[i * 32 + lane] =
                    make_float2((v[i].x - mean) * rstd * gm[i].x + bt[i].x, (v[i].y - mean) * rstd * gm[i].y + bt[i].y);
            } else {
                __nv_bfloat162 pk = __floats2bfloat162_rn((v[i].x - mean) * rstd * gm[i].x + bt[i].x, (v[i].y - mean) * rstd * gm[i].y + bt[i].y);
                reinterpret_cast<__nv_bfloat162*>(dst)[i * 32 + lane] = pk;
            }
        }
    }
}

template <int NSLAB>
__global__ void __launch_bounds__(256) layernorm_bf16_slab64_kernel(const float* __restrict__ x, long long in_stride,
                                                                    const float* __restrict__ gamma,
                                                                    const float* __restrict__ beta,
                                                                    __nv_bfloat16* __restrict__ out, int rows, float eps,
                                                                    int reverse, int stream_in) {
    layernorm_slab64_rows<NSLAB>(x, in_stride, gamma, beta, out, NSLAB * 64, rows, eps, reverse, stream_in);
}
template <int NSLAB>
__global__ void __launch_bounds__(256) layernorm_f32_slab64_kernel(const float* x, long long in_stride, const float* __restrict__ gamma,
                                                                   const float* __restrict__ beta, float* out, long long out_stride,
                                                                   int rows, float eps, int reverse, int stream_in) {
    layernorm_slab64_rows<NSLAB>(x, in_stride, gamma, beta, out, out_stride, rows, eps, reverse, stream_in);
}

constexpr int ATT_HD = 64;  // head dimension of every supported ViT (attention_tcgen05.cuh)

// ------------------------------------------------------------------------------------------------
// Stage-1 score finisher. `partials` [ceil(M/32)][2][ldp] holds, per 32-row sub-tile and image segment,
// the sum of squared activations per neuron (written by the fc1 GEMM epilogue). Kernel A turns them into
// per-(image, neuron) L2 norms over tokens; kernel B adds the image norms, in image order, to the
// running per-neuron score (src/vit_pruning.py:151-152: vector_norm(dim=1) then sum(dim=0)).
// Both are fixed-order sums: results do not depend on scheduling.
// ------------------------------------------------------------------------------------------------
// all blocks of one batch in one launch: grid (ceil(Fmax/128), n_img, n_blocks)
struct ScoreBlocks {
    int F[64];         // neurons of block b
    int ldp[64];       // row pitch of block b's partial buffer
    int norm_off[64];  // column offset of block b in the norms / scores vectors
};

// Four neurons per thread (one 128-bit load per sub-tile row, all of an image's <= 8 sub-tiles requested before the
// first add), partial rows added in sub-tile order as before: same bits, more bytes in flight.
__global__ void __launch_bounds__(128) score_norms_all_kernel(const float* __restrict__ partials, size_t block_stride, const ScoreBlocks sb,
                                                              float* __restrict__ norms, int ldn, int n_img, int T) {
    const int b = blockIdx.z;
    const int col = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int img = blockIdx.y;
    const int F = sb.F[b];
    if (col >= F || img >= n_img) return;
    const float* base = partials + block_stride * b;
    const int ldp = sb.ldp[b];  // a multiple of 8 >= F: the 128-bit loads stay inside the row and aligned
    const int r_begin = img * T, r_end = r_begin + T;
    const int s_begin = r_begin >> 5, s_end = (r_end - 1) >> 5;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s0 = s_begin; s0 <= s_end; s0 += 8) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int s = s0 + u;
            if (s <= s_end) {
                const int seg = ((s << 5) / T == img) ? 0 : 1;
                v[u] = *reinterpret_cast<const float4*>(base + (static_cast<size_t>(s) * 2 + seg) * ldp + col);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
            if (s0 + u <= s_end) {
                acc.x += v[u].x;
                acc.y += v[u].y;
                acc.z += v[u].z;
                acc.w += v[u].w;
            }
    }
    float* dst = norms + static_cast<size_t>(img) * ldn + sb.norm_off[b] + col;
    dst[0] = sqrtf(acc.x);
    if (col + 1 < F) dst[1] = sqrtf(acc.y);
    if (col + 2 < F) dst[2] = sqrtf(acc.z);
    if (col + 3 < F) dst[3] = sqrtf(acc.w);
}

// scores[col] += sum over the batch's images IN IMAGE ORDER (one chain of adds per neuron, as before); sixteen loads
// are requested ahead of the adds that consume them.
__global__ void __launch_bounds__(128) score_accumulate_kernel(const float* __restrict__ norms, int ldn, int n_img, int F,
                                                               float* __restrict__ scores) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= F) return;
    float acc = scores[col];
    const float* src = norms + col;
    int img = 0;
    for (; img + 16 <= n_img; img += 16) {
        float v[16];
#pragma unroll
        for (int u = 0; u < 16; ++u) v[u] = src[static_cast<size_t>(img + u) * ldn];
#pragma unroll
        for (int u = 0; u < 16; ++u) acc += v[u];
    }
    for (; img < n_img; ++img) acc += src[static_cast<size_t>(img) * ldn];
    scores[col] = acc;
}

// ------------------------------------------------------------------------------------------------
// top-1 counter (src/vit_pruning.py:370-371): argmax over classes (first maximum wins), compare with the
// label, count matches with an integer atomic. One warp per image.
// ------------------------------------------------------------------------------------------------
__global__ void argmax_count_kernel(const float* __restrict__ logits, int ld, int n, int C,
                                    const long long* __restrict__ labels, int* __restrict__ preds,
                                    unsigned long long* __restrict__ correct) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= n) return;
    const float* row = logits + static_cast<size_t>(warp) * ld;
    float best = -INFINITY;
    int best_i = 0x7fffffff;
    for (int c = lane; c < C; c += 32) {
        const float v = row[c];
        if (v > best || (v == best && c < best_i)) { best = v; best_i = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
        if (ov > best || (ov == best && oi < best_i)) { best = ov; best_i = oi; }
    }
    if (lane == 0) {
        if (preds != nullptr) preds[warp] = best_i;
        if (labels != nullptr && correct != nullptr && static_cast<long long>(best_i) == labels[warp]) atomicAdd(correct, 1ULL);
    }
}

}  // namespace tssp
