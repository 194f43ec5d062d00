// Engine + C ABI (include/tssp.h) of the B200-native 2SSP ViT hot path.
// Owns the packed weights, the activation workspace and the launch sequences; every compute step is one of
// the hand-written sm_100a kernels in gemm_tcgen05.cuh / kernels.cuh. No library GEMM, no CPU fallback.
#include <charconv>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/tssp.h"
#include "gemm_tcgen05.cuh"
#include "kernels.cuh"
#include "attention_tcgen05.cuh"
#include "attention_long_tcgen05.cuh"
#include "mask_builders.cuh"
#include "gather.cuh"

namespace tssp {

// ------------------------------------------------------------------------------------------------ errors
static thread_local std::string g_last_error;
static unsigned long long g_launches = 0;

// Every entry point of the C ABI takes this lock: ctypes.CDLL releases the Python GIL around a call, so the
// process-wide caches below (tensor maps, device block pool, per-device kernel attributes, profiler records) would
// otherwise be reachable from two threads at once. One process drives one GPU on this path (torch.distributed, one
// rank per GPU), so the lock is never contended in the intended use; it makes the library safe, not parallel.
static std::recursive_mutex g_lib_mutex;
#define TSSP_ENTRY() std::lock_guard<std::recursive_mutex> _tssp_lock(tssp::g_lib_mutex)

// Per-chain launch state (serpentine direction, dependent-launch choice). An engine owns one; the kernel-level
// tssp_op_* entry points use a library-wide default. Entry points make theirs current for the calling thread.
struct LaunchCtx {
    int chain_dir = 0;     // next kernel of the chain walks last-to-first when 1 (see chain_dir())
    bool pdl_auto = false; // programmatic dependent launch unless TSSP_PDL forces it (set from the hidden size)
};
static LaunchCtx g_default_ctx;
static thread_local LaunchCtx* t_ctx = &g_default_ctx;
struct CtxScope {
    LaunchCtx* prev;
    explicit CtxScope(LaunchCtx* c) : prev(t_ctx) { t_ctx = c; }
    ~CtxScope() { t_ctx = prev; }
};

static int fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return 1;
}

#define TSSP_CUDA(expr)                                                                                   \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define TSSP_TRY(expr)               \
    do {                             \
        int _rc = (expr);            \
        if (_rc != 0) return _rc;    \
    } while (0)
#define TSSP_LAUNCH_CHECK(name)                                                                      \
    do {                                                                                             \
        ++g_launches;                                                                                \
        cudaError_t _e = cudaGetLastError();                                                         \
        if (_e != cudaSuccess) return fail("launch of %s failed: %s", name, cudaGetErrorString(_e)); \
    } while (0)

// ------------------------------------------------------------------------------------------------ profiler
// Optional per-kernel-class timing with CUDA events recorded on the launching stream (bench.py's roofline):
// tssp_profile_begin() arms it, every instrumented launch is bracketed by an event pair, tssp_profile_end()
// synchronises and returns the summed device time and launch count per class.
enum KernelClass { KC_FC1 = 0, KC_QKV, KC_PROJ, KC_FC2, KC_PATCH, KC_HEAD, KC_ATTN, KC_LN, KC_SCORE, KC_MISC, KC_COUNT };
struct ProfRec { int cls; cudaEvent_t start, stop; };
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof_recs;
static std::vector<cudaEvent_t> g_prof_pool;

static cudaEvent_t prof_event() {
    if (!g_prof_pool.empty()) {
        cudaEvent_t e = g_prof_pool.back();
        g_prof_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct ProfScope {
    bool active;
    cudaStream_t stream;
    ProfRec rec;
    ProfScope(int cls, cudaStream_t s) : active(g_prof_on), stream(s) {
        if (active) {
            rec.cls = cls;
            rec.start = prof_event();
            rec.stop = prof_event();
            cudaEventRecord(rec.start, stream);
        }
    }
    ~ProfScope() {
        if (active) {
            cudaEventRecord(rec.stop, stream);
            g_prof_recs.push_back(rec);
        }
    }
};
#define TSSP_PROF(cls, stream, expr)   \
    do {                               \
        ProfScope _ps(cls, stream);    \
        TSSP_TRY(expr);                \
    } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }
constexpr int TSSP_MAX_PREFIX = 1 + TSSP_MAX_REGISTER_TOKENS;  // CLS + register tokens (or CLS + distillation token)

// ------------------------------------------------------------------------------------------------ TMA maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

static int load_encode_fn() {
    if (g_encode != nullptr) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    TSSP_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (fn == nullptr || qres != cudaDriverEntryPointSuccess) return fail("cuTensorMapEncodeTiled not available from the driver");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

// 2-D row-major tensor [outer, inner] with `pitch_bytes` between rows, boxes of [box_outer, box_inner],
// SWIZZLE_128B (box_inner * elem_bytes must be 128).
static int make_tmap(CUtensorMap* out, const void* ptr, bool is_f32, uint64_t inner, uint64_t outer, uint64_t pitch_bytes,
                     uint32_t box_inner, uint32_t box_outer) {
    TSSP_TRY(load_encode_fn());
    if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0) return fail("tensor map: base pointer not 16-byte aligned");
    if ((pitch_bytes & 15u) != 0) return fail("tensor map: row pitch %llu not a multiple of 16 bytes", (unsigned long long)pitch_bytes);
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(out, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                          const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d (inner=%llu outer=%llu pitch=%llu box=%ux%u)",
                                       (int)r, (unsigned long long)inner, (unsigned long long)outer,
                                       (unsigned long long)pitch_bytes, box_inner, box_outer);
    return 0;
}

// ------------------------------------------------------------------------------------------------ GEMM launch
constexpr int GEMM_BN = 256;
constexpr int GEMM_STAGES = 4;
constexpr int GEMM_EPI_WARPS = 8;

struct TmapKey {
    const void* ptr; int is_f32; uint64_t inner, outer, pitch; uint32_t bi, bo;
    bool operator<(const TmapKey& o) const {
        return std::tie(ptr, is_f32, inner, outer, pitch, bi, bo) < std::tie(o.ptr, o.is_f32, o.inner, o.outer, o.pitch, o.bi, o.bo);
    }
};
static std::map<TmapKey, CUtensorMap> g_tmap_cache;  // guarded by g_lib_mutex; bounded (see get_tmap)
constexpr size_t TMAP_CACHE_MAX = 4096;  // the tssp_op_* entry points see arbitrary caller pointers: start over when full

static int get_tmap(const CUtensorMap** out, const void* ptr, bool is_f32, uint64_t inner, uint64_t outer, uint64_t pitch,
                    uint32_t bi, uint32_t bo) {
    TmapKey key{ptr, is_f32 ? 1 : 0, inner, outer, pitch, bi, bo};
    auto it = g_tmap_cache.find(key);
    if (it == g_tmap_cache.end()) {
        if (g_tmap_cache.size() >= TMAP_CACHE_MAX) g_tmap_cache.clear();  // maps are passed to kernels by value: safe
        CUtensorMap m;
        TSSP_TRY(make_tmap(&m, ptr, is_f32, inner, outer, pitch, bi, bo));
        it = g_tmap_cache.emplace(key, m).first;
    }
    *out = &it->second;
    return 0;
}

// Device attributes and kernel opt-ins are per device (and per context): a second engine on another GPU of the same
// process needs its own. Both are keyed by the current device.
static std::map<int, int> g_num_sms;
static int num_sms() {
    int dev = 0;
    cudaGetDevice(&dev);
    auto it = g_num_sms.find(dev);
    if (it == g_num_sms.end()) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        it = g_num_sms.emplace(dev, n > 0 ? n : 148).first;
    }
    return it->second;
}
static std::map<std::pair<int, const void*>, int> g_smem_optin;  // (device, kernel) -> configured dynamic shared memory
template <typename K>
static int ensure_smem(K kern, int bytes) {
    int dev = 0;
    cudaGetDevice(&dev);
    const auto key = std::make_pair(dev, reinterpret_cast<const void*>(kern));
    auto it = g_smem_optin.find(key);
    if (it != g_smem_optin.end() && it->second >= bytes) return 0;
    TSSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    g_smem_optin[key] = bytes;
    return 0;
}
struct DeviceScope {  // entry points that must run on an engine's device leave the caller's current device as it was
    int prev = -1;
    explicit DeviceScope(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev); else prev = -1;
    }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
};

// Launch with programmatic stream serialization: the kernel may be scheduled while the previous kernel of the stream
// is draining, and blocks in griddepcontrol.wait before touching its data. Used for the per-block kernels (GEMMs,
// LayerNorm, attention), 99 % of the launches of a sweep. Measured (profiles/pdl_ab_r1.txt): +4.6 % images/s for
// ViT-S, whose kernels are launch-latency bound, but -1.5 % for ViT-B, where the GPU sits at its power cap and the
// filled gaps only lower the clock. TSSP_PDL=1 / 0 forces it; the default enables it for hidden sizes below 768.
static bool pdl_enabled() {
    static const int forced = [] {
        const char* e = getenv("TSSP_PDL");
        return e == nullptr ? -1 : (strcmp(e, "0") != 0 ? 1 : 0);
    }();
    return forced < 0 ? t_ctx->pdl_auto : forced == 1;
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_ex(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, unsigned cluster_x,
                             Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    unsigned n = 0;
    if (pdl_enabled()) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster_x > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = cluster_x;
        attr[n].val.clusterDim.y = 1;
        attr[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = attr;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    return launch_ex(kern, grid, block, smem, stream, 1u, static_cast<Args&&>(args)...);
}

// CTA-pair form (CTAS = 2, gemm_tcgen05.cuh): 256-row tiles over num_sms / 2 clusters. It streams a third less operand
// data per FLOP (the single-CTA form is bound by that stream: profiles/gemm_operand_traffic_r1.txt) but quantises into
// twice-as-coarse waves, so it is used when its wave count, discounted by the measured per-tile gain, is lower.
// TSSP_GEMM_CTAS=1 / 2 forces either form.
constexpr int GEMM_PAIR_STAGES = 6;
static long long* g_gemm_trace = nullptr;  // device buffer set by tssp_debug_gemm_trace (diagnostics only)
static unsigned long long g_launch_epoch = 0;  // bumped when a process-wide launch setting changes: captured chains are stale then
static int g_gemm_form = -1;  // 0 automatic, 1 single CTA, 2 CTA pair; -1: take TSSP_GEMM_CTAS on first use
static bool gemm_use_pair(int M, int N, int bn = GEMM_BN) {
    if (g_gemm_form < 0) {
        const char* e = getenv("TSSP_GEMM_CTAS");
        g_gemm_form = (e != nullptr && (atoi(e) == 1 || atoi(e) == 2)) ? atoi(e) : 0;
    }
    if (g_gemm_form == 1) return false;
    if (g_gemm_form == 2) return true;
    const int n_blks = ceil_div(N, bn);
    const int waves1 = ceil_div(ceil_div(M, 128) * n_blks, num_sms());
    const int waves2 = ceil_div(ceil_div(M, 256) * n_blks, num_sms() / 2);
    return waves2 * 90 < waves1 * 100;
}

// Serpentine traversal (TSSP_SERPENTINE=0 disables): the kernels of the forward chain (LayerNorm, GEMMs, attention)
// take turns walking their rows / tiles / units first-to-last and last-to-first, so each one starts on the rows its
// producer wrote last -- the part of a 77-310 MB activation that is still in the 126 MB L2. Same work, same bits.
static int chain_dir() {
    static const bool serpentine = [] { const char* e = getenv("TSSP_SERPENTINE"); return !(e != nullptr && strcmp(e, "0") == 0); }();
    if (!serpentine) return 0;
    const int d = t_ctx->chain_dir;
    t_ctx->chain_dir ^= 1;
    return d;
}

// L2 policy hint: the LayerNorm before the FFN loads the residual rows evict-first, so that the normalised rows it
// WRITES (what fc1 starts on) are what survives in L2: LayerNorm 3 % faster, nothing else slower. The same hint on the
// LayerNorm before attention was neutral, on attention's qkv loads it cost proj 8 %, on the A operand of proj / fc2 it
// cost 12 % / 7 % (an A tile is re-read by the column tiles of its row block): profiles/l2_hints_ab_r1.txt. Those
// three were removed with their switches.
template <int MODE, int CTAS, int BN = GEMM_BN>
static int launch_gemm_mode(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmParams& p,
                            cudaStream_t stream) {
    constexpr int STAGES = CTAS == 2 ? GEMM_PAIR_STAGES : GEMM_STAGES;
    using Cfg = GemmCfg<MODE, BN, STAGES, GEMM_EPI_WARPS, CTAS>;
    auto kern = gemm_bf16_tn_kernel<MODE, BN, STAGES, GEMM_EPI_WARPS, CTAS>;
    TSSP_TRY(ensure_smem(kern, Cfg::SMEM_BYTES));
    const int tiles = ceil_div(p.M, Cfg::BM * CTAS) * ceil_div(p.N, BN);
    const int slots = num_sms() / CTAS;
    const int grid = (tiles < slots ? tiles : slots) * CTAS;
    TSSP_CUDA(launch_ex(kern, dim3(grid), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, stream, static_cast<unsigned>(CTAS), ta, tb, tc, p));
    TSSP_LAUNCH_CHECK("gemm_bf16_tn_kernel");
    return 0;
}

// C[M,N] (ldc) = A[M,K] (lda) * W[N,K]^T (ldw) with epilogue `mode` (GemmMode)
static int gemm(int mode, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                const float* bias, float* partials, int ldp, int T, int reduce_add, cudaStream_t stream,
                float* rownorm = nullptr, int ld_rownorm = 0, int rownorm_chunks = 0, const float* col_scale = nullptr) {
    if (M <= 0 || N <= 0 || K <= 0) return fail("gemm: empty problem M=%d N=%d K=%d", M, N, K);
    if ((N & 7) || (K & 7)) return fail("gemm: N=%d and K=%d must be multiples of 8", N, K);
    const bool f32_out = (mode == EPI_F32 || mode == EPI_F32_SCALED);
    if (mode == EPI_F32_SCALED && col_scale == nullptr) return fail("gemm: scaled fp32 epilogue needs a column scale");
    const bool score = gemm_mode_scores(mode);
    if (score && (partials == nullptr || T < 32 || ldp < N)) return fail("gemm: score epilogue needs partials, ldp >= N and T >= 32 (T=%d)", T);
    // the epilogue stores each lane's two partials as one float2 and the finisher reads them as float4
    if (score && (ldp & 3)) return fail("gemm: score partial row pitch %d must be a multiple of 4", ldp);
    const CUtensorMap *ta, *tb, *tc;
    TSSP_TRY(get_tmap(&ta, A, false, K, M, static_cast<uint64_t>(lda) * 2, 64, 128));
    // fp32-output GEMMs with a short reduction whose last 256-column tile would be at most half full (N = 384, K = 384: the
    // ViT-S proj; N = 128) run 128-column tiles instead: no padded MMA work (ViT-S proj 42 -> 38 us). With a long K the
    // narrower tile loses more to its 50 % higher operand traffic per MAC than it saves (ViT-S fc2, K = 1536: 71 -> 77 us),
    // so those keep 256 columns.
    // Widths that are whole multiples of 192 but not of 256 (N = 384: ViT-S proj / fc2 / patch-embed) run 192-column tiles:
    // two full tiles instead of one and a half, at any K.
    int bn = GEMM_BN;
    if (f32_out && N % GEMM_BN != 0) {
        if (N % 192 == 0) bn = 192;
        else if (K <= 512 && N % GEMM_BN <= GEMM_BN / 2) bn = GEMM_BN / 2;
    }
    const bool pair = gemm_use_pair(M, N, bn);
    TSSP_TRY(get_tmap(&tb, W, false, K, N, static_cast<uint64_t>(ldw) * 2, 64, pair ? bn / 2 : bn));
    if (f32_out) TSSP_TRY(get_tmap(&tc, C, true, N, M, static_cast<uint64_t>(ldc) * 4, 32, 32));
    else TSSP_TRY(get_tmap(&tc, C, false, N, M, static_cast<uint64_t>(ldc) * 2, 64, 32));
    GemmParams p;
    p.M = M; p.N = N; p.K = K; p.bias = bias; p.partials = partials; p.ldp = ldp; p.tokens_per_image = T;
    p.reduce_add = reduce_add;
    p.reverse = chain_dir();
    p.trace = g_gemm_trace;
    p.rownorm = rownorm; p.ld_rownorm = ld_rownorm; p.rownorm_chunks = rownorm_chunks;
    p.col_scale = col_scale;
    if (mode == EPI_BF16_ROWNORM && rownorm == nullptr) return fail("gemm: row-norm epilogue needs an output buffer");
#define TSSP_GEMM_CASE(m) \
    case m: return pair ? launch_gemm_mode<m, 2>(*ta, *tb, *tc, p, stream) : launch_gemm_mode<m, 1>(*ta, *tb, *tc, p, stream);
#define TSSP_GEMM_F32_BN(m, bn_)                                                                                   \
    if (bn == bn_)                                                                                                 \
        return pair ? launch_gemm_mode<m, 2, bn_>(*ta, *tb, *tc, p, stream) : launch_gemm_mode<m, 1, bn_>(*ta, *tb, *tc, p, stream);
    if (mode == EPI_F32_SCALED) {  // the fp32 tile widths of EPI_F32 (see above), with the LayerScale factor
        TSSP_GEMM_F32_BN(EPI_F32_SCALED, GEMM_BN / 2)
        TSSP_GEMM_F32_BN(EPI_F32_SCALED, 192)
        TSSP_GEMM_F32_BN(EPI_F32_SCALED, GEMM_BN)
    }
#undef TSSP_GEMM_F32_BN
    if (bn == GEMM_BN / 2)  // EPI_F32 only (see above)
        return pair ? launch_gemm_mode<EPI_F32, 2, GEMM_BN / 2>(*ta, *tb, *tc, p, stream) : launch_gemm_mode<EPI_F32, 1, GEMM_BN / 2>(*ta, *tb, *tc, p, stream);
    if (bn == 192)
        return pair ? launch_gemm_mode<EPI_F32, 2, 192>(*ta, *tb, *tc, p, stream) : launch_gemm_mode<EPI_F32, 1, 192>(*ta, *tb, *tc, p, stream);
    switch (mode) {
        TSSP_GEMM_CASE(EPI_BF16)
        TSSP_GEMM_CASE(EPI_BF16_GELU)
        TSSP_GEMM_CASE(EPI_BF16_GELU_SCORE)
        TSSP_GEMM_CASE(EPI_BF16_GELU_SCORE_PRE)
        TSSP_GEMM_CASE(EPI_F32)
        TSSP_GEMM_CASE(EPI_BF16_ROWNORM)
        TSSP_GEMM_CASE(EPI_BF16_QGELU)
        TSSP_GEMM_CASE(EPI_BF16_QGELU_SCORE_PRE)
#undef TSSP_GEMM_CASE
        default: return fail("gemm: unknown epilogue mode %d", mode);
    }
}

// ------------------------------------------------------------------------------------------------ small launchers
static inline int grid_for(long long work, int threads) {
    long long g = (work + threads - 1) / threads;
    const long long cap = static_cast<long long>(num_sms()) * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return static_cast<int>(g);
}

static int op_cast(const float* in, int rows, int cols, int ld_in, void* out, int rows_pad, int cols_pad, int ld_out, cudaStream_t s,
                   float scale = 1.0f) {
    const long long total = static_cast<long long>(rows_pad) * cols_pad;
    if (total == 0) return 0;
    cast_pad_bf16_kernel<<<grid_for(total, 256), 256, 0, s>>>(in, rows, cols, ld_in, static_cast<__nv_bfloat16*>(out), rows_pad, cols_pad, ld_out,
                                                              scale);
    TSSP_LAUNCH_CHECK("cast_pad_bf16_kernel");
    return 0;
}

// prefix: zero rows ahead of every image's patches (1: CLS; 2: CLS and the DeiT distillation token; 1 + R: CLS and R
// register tokens). Rows are patch_width(C, P) = round_up(C*P*P, 8) elements, zero padded past C*P*P.
static int patch_width(int C, int P) { return round_up(C * P * P, 8); }
// The pixel format of an im2col input (tssp_pixel_input_t): refused unless its normalisation can be applied to C channels.
static int check_pixel_input(const tssp_pixel_input_t& in, int C, const char* where) {
    if (in.format != TSSP_PIXELS_F32 && in.format != TSSP_PIXELS_U8)
        return fail("%s: format=%d must be %d (fp32) or %d (uint8)", where, in.format, TSSP_PIXELS_F32, TSSP_PIXELS_U8);
    if (in.format == TSSP_PIXELS_F32) return 0;
    if (C < 1 || C > TSSP_MAX_PIXEL_CHANNELS)
        return fail("%s: uint8 pixels need 1 to %d channels, got C=%d", where, TSSP_MAX_PIXEL_CHANNELS, C);
    if (!std::isfinite(in.rescale)) return fail("%s: rescale=%g is not finite", where, in.rescale);
    for (int c = 0; c < C; ++c) {
        if (!std::isfinite(in.mean[c])) return fail("%s: mean[%d]=%g is not finite", where, c, in.mean[c]);
        if (!std::isfinite(in.std[c]) || !(in.std[c] > 0.0f)) return fail("%s: std[%d]=%g must be finite and > 0", where, c, in.std[c]);
    }
    return 0;
}

// in == nullptr or TSSP_PIXELS_F32: fp32 pixels. TSSP_PIXELS_U8: uint8 pixels, normalised per channel on the way in
// (kernels.cuh: the fp32 kernels' bits for the normalised image).
static int op_im2col(const void* pixels, void* out, int n, int C, int H, int W, int P, int prefix, const tssp_pixel_input_t* in,
                     cudaStream_t s) {
    if (P < 1 || H % P || W % P || H != W) return fail("im2col: H=%d W=%d P=%d unsupported (square images, P dividing them)", H, W, P);
    if (prefix < 1 || prefix > TSSP_MAX_PREFIX) return fail("im2col: prefix=%d must be in [1,%d]", prefix, TSSP_MAX_PREFIX);
    if (in != nullptr) TSSP_TRY(check_pixel_input(*in, C, "im2col"));
    const bool u8 = in != nullptr && in->format == TSSP_PIXELS_U8;
    const int T = (H / P) * (W / P) + prefix;
    const int ld = patch_width(C, P);
    const long long total = static_cast<long long>(n) * T * (ld / 8);
    __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out);
    if (!u8) {
        const float* px = static_cast<const float*>(pixels);
        if ((P & 7) == 0) {
            im2col_patches_kernel<<<grid_for(total, 256), 256, 0, s>>>(px, o, n, C, H, W, P, T, prefix);
            TSSP_LAUNCH_CHECK("im2col_patches_kernel");
        } else {
            im2col_patches_padded_kernel<<<grid_for(total, 256), 256, 0, s>>>(px, o, n, C, H, W, P, T, prefix, ld);
            TSSP_LAUNCH_CHECK("im2col_patches_padded_kernel");
        }
        return 0;
    }
    const uintptr_t align = (P & 7) == 0 ? 8 : ((P & 1) == 0 ? 2 : 1);  // the 8-byte / 2-byte loads of the two kernels
    if (reinterpret_cast<uintptr_t>(pixels) % align != 0)
        return fail("im2col (uint8 pixels): pointer %p is not %d-byte aligned, as the loads at P=%d need", pixels, static_cast<int>(align), P);
    PixelNorm pn;
    pn.rescale = in->rescale;
    for (int c = 0; c < 4; ++c) {
        pn.mean[c] = c < C ? in->mean[c] : 0.0f;
        pn.std[c] = c < C ? in->std[c] : 1.0f;
    }
    const uint8_t* px = static_cast<const uint8_t*>(pixels);
    if ((P & 7) == 0) {
        im2col_patches_u8_kernel<<<grid_for(total, 256), 256, 0, s>>>(px, o, n, C, H, W, P, T, prefix, pn);
        TSSP_LAUNCH_CHECK("im2col_patches_u8_kernel");
    } else {
        im2col_patches_padded_u8_kernel<<<grid_for(total, 256), 256, 0, s>>>(px, o, n, C, H, W, P, T, prefix, ld, pn);
        TSSP_LAUNCH_CHECK("im2col_patches_padded_u8_kernel");
    }
    return 0;
}

// out: bf16 rows of pitch D, or (f32_out) fp32 rows of pitch out_stride; an fp32 out may be x itself
static int op_layernorm_any(const float* x, long long in_stride, const float* g, const float* b, void* out, bool f32_out,
                            long long out_stride, int rows, int D, float eps, cudaStream_t s, bool stream_in) {
    if (((D & 127) && D != 192) || D > 1024) return fail("layernorm: D=%d must be 192 or a multiple of 128 <= 1024", D);
    if (in_stride & 3) return fail("layernorm: row pitch %lld must be a multiple of 4 elements", in_stride);
    if (f32_out && ((out_stride & 3) || out_stride < D))
        return fail("layernorm: output row pitch %lld must be a multiple of 4 elements and >= D=%d", out_stride, D);
    if (rows <= 0) return 0;
    // persistent: resident CTAs per SM. Narrow rows need more warps for the same bytes in flight; at D = 1024 the kernel
    // holds 150 registers (row, prefetched row, gamma, beta), so 12 warps fit as three CTAs of 128 threads but only 8
    // as one CTA of 256 (re-reading gamma / beta instead of holding them was measured slower: 0.60 against 0.75 of peak).
    // D = 192 (64-element slabs, six values a lane) takes the D <= 512 setting.
    const int threads = D > 768 ? 128 : 256;
    const int per_sm = D <= 512 ? 4 : (D > 768 ? 3 : 2);
    const int ctas = ceil_div(rows, threads / 32);
    const int grid = ctas < per_sm * num_sms() ? ctas : per_sm * num_sms();
    __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out);
    float* of = static_cast<float*>(out);
    const int rev = chain_dir();
    const int hint = stream_in ? 1 : 0;
#define TSSP_LN_LAUNCH(kbf16, kf32)                                                                                                 \
    TSSP_CUDA(f32_out ? launch_pdl(kf32, dim3(grid), dim3(threads), 0, s, x, in_stride, g, b, of, out_stride, rows, eps, rev, hint) \
                      : launch_pdl(kbf16, dim3(grid), dim3(threads), 0, s, x, in_stride, g, b, o, rows, eps, rev, hint))
#define TSSP_LN_CASE(d, NS, VPL) \
    case d: TSSP_LN_LAUNCH((layernorm_bf16_slab_kernel<NS, VPL>), (layernorm_f32_slab_kernel<NS, VPL>)); break;
    switch (D) {
        case 192: TSSP_LN_LAUNCH(layernorm_bf16_slab64_kernel<3>, layernorm_f32_slab64_kernel<3>); break;
        TSSP_LN_CASE(128, 1, 1)
        TSSP_LN_CASE(256, 1, 2)
        TSSP_LN_CASE(384, 3, 1)
        TSSP_LN_CASE(512, 2, 2)
        TSSP_LN_CASE(640, 5, 1)
        TSSP_LN_CASE(768, 3, 2)
        TSSP_LN_CASE(896, 7, 1)
        TSSP_LN_CASE(1024, 4, 2)
        default: return fail("layernorm: D=%d has no kernel instance", D);
    }
#undef TSSP_LN_CASE
#undef TSSP_LN_LAUNCH
    TSSP_LAUNCH_CHECK(f32_out ? "layernorm_f32_slab_kernel" : "layernorm_bf16_slab_kernel");
    return 0;
}

static int op_layernorm(const float* x, long long in_stride, const float* g, const float* b, void* out, int rows, int D, float eps, cudaStream_t s,
                        bool stream_in = false) {
    return op_layernorm_any(x, in_stride, g, b, out, false, D, rows, D, eps, s, stream_in);
}
static int op_layernorm_f32(const float* x, long long in_stride, const float* g, const float* b, float* out, long long out_stride, int rows,
                            int D, float eps, cudaStream_t s) {
    return op_layernorm_any(x, in_stride, g, b, out, true, out_stride, rows, D, eps, s, false);
}

// 3-D tensor map over a token-major bf16 activation viewed as [n_img][T][width] (width = 3D for the fused qkv, D for
// ctx): boxes of [1][box_rows][64 columns], SWIZZLE_128B; rows >= T of an image are out of bounds: they load as zeros
// and are not stored.
static int make_tmap_qkv(CUtensorMap* out, const void* qkv, int n_img, int T, int width, uint32_t box_rows) {
    TSSP_TRY(load_encode_fn());
    if ((reinterpret_cast<uintptr_t>(qkv) & 15u) != 0) return fail("attention: qkv pointer not 16-byte aligned");
    cuuint64_t dims[3] = {static_cast<cuuint64_t>(width), static_cast<cuuint64_t>(T), static_cast<cuuint64_t>(n_img)};
    cuuint64_t strides[2] = {static_cast<cuuint64_t>(width) * 2, static_cast<cuuint64_t>(T) * width * 2};
    cuuint32_t box[3] = {64, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(qkv), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled (qkv, 3-D) failed with CUresult %d", (int)r);
    return 0;
}

struct QkvMapKey {
    const void* ptr; int n, T, D; uint32_t rows;
    bool operator<(const QkvMapKey& o) const { return std::tie(ptr, n, T, D, rows) < std::tie(o.ptr, o.n, o.T, o.D, o.rows); }
};
static std::map<QkvMapKey, CUtensorMap> g_qkv_maps;

static int get_tmap_qkv(const CUtensorMap** out, const void* qkv, int n, int T, int D, uint32_t rows) {
    QkvMapKey key{qkv, n, T, D, rows};
    auto it = g_qkv_maps.find(key);
    if (it == g_qkv_maps.end()) {
        if (g_qkv_maps.size() >= TMAP_CACHE_MAX) g_qkv_maps.clear();
        CUtensorMap m;
        TSSP_TRY(make_tmap_qkv(&m, qkv, n, T, D, rows));
        it = g_qkv_maps.emplace(key, m).first;
    }
    *out = &it->second;
    return 0;
}

// softmax(Q K^T / sqrt(64)) V per (image, head): attention_tcgen05.cuh up to 208 padded keys, attention_long_tcgen05.cuh
// (keys in tiles of 128) beyond
static long long* g_attn_trace = nullptr;  // device buffer set by tssp_debug_attention_trace (diagnostics only)

static int op_attention_long(const void* qkv, void* ctx, int n, int T, int heads, int D, cudaStream_t s, const float* qk_norms,
                             int ld_norms, bool first_tile_only) {
    const CUtensorMap *tqkv, *tctx;
    TSSP_TRY(get_tmap_qkv(&tqkv, qkv, n, T, 3 * D, 128));
    TSSP_TRY(get_tmap_qkv(&tctx, ctx, n, T, D, 32));
    TSSP_TRY(ensure_smem(attention_long_tcgen05_kernel, ATL_SMEM_BYTES));
    AttnLongParams p;
    p.n_img = n; p.T = T; p.heads = heads; p.D = D;
    p.MT = first_tile_only ? 1 : ceil_div(T, 128);
    p.n_groups = ceil_div(p.MT, ATL_MAX_G);
    p.NKT = ceil_div(T, ATL_KT);
    p.scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(ATT_HD));
    p.norms = qk_norms; p.ld_norms = ld_norms;
    p.qkv = static_cast<const __nv_bfloat16*>(qkv);
    p.reverse = chain_dir();
    const long long units = static_cast<long long>(n) * heads * p.n_groups;
    const int grid = units < num_sms() ? static_cast<int>(units) : num_sms();
    TSSP_CUDA(launch_pdl(attention_long_tcgen05_kernel, dim3(grid), dim3(ATL_THREADS), ATL_SMEM_BYTES, s, *tqkv, *tctx, p));
    TSSP_LAUNCH_CHECK("attention_long_tcgen05_kernel");
    return 0;
}

// first_tile_only: only the first 128 query rows of every (image, head) are computed (the rest of ctx is left alone) --
// for the last block of a classifier forward, where the CLS row (row 0) is all that is read afterwards
static int op_attention(const void* qkv, void* ctx, int n, int T, int heads, int D, cudaStream_t s,
                        const float* qk_norms = nullptr, int ld_norms = 0, bool first_tile_only = false) {
    if (D != heads * ATT_HD) return fail("attention: head_dim must be 64 (D=%d heads=%d)", D, heads);
    const int Tp = round_up(T, 16);
    if (T < 16 || T > ATL_MAX_T) return fail("attention: T=%d outside the supported [16, %d] tokens", T, ATL_MAX_T);
    if (Tp > ATC_KV_ROWS) return op_attention_long(qkv, ctx, n, T, heads, D, s, qk_norms, ld_norms, first_tile_only);
    const float scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(ATT_HD));
    const CUtensorMap *tq, *tkv;
    const CUtensorMap* tctx;
    TSSP_TRY(get_tmap_qkv(&tq, qkv, n, T, 3 * D, 128));
    TSSP_TRY(get_tmap_qkv(&tkv, qkv, n, T, 3 * D, static_cast<uint32_t>(Tp)));
    TSSP_TRY(get_tmap_qkv(&tctx, ctx, n, T, D, 32));
    TSSP_TRY(ensure_smem(attention_tcgen05_kernel, ATC_SMEM_BYTES));
    AttnParams p;
    p.n_img = n; p.T = T; p.heads = heads; p.D = D; p.KP = Tp; p.MT = first_tile_only ? 1 : ceil_div(T, 128); p.scale_log2e = scale_log2e;
    p.trace = g_attn_trace;
    p.reverse = chain_dir();
    p.norms = qk_norms; p.ld_norms = ld_norms;
    const int units = n * heads;
    const int grid = units < num_sms() ? units : num_sms();
    TSSP_CUDA(launch_pdl(attention_tcgen05_kernel, dim3(grid), dim3(ATC_THREADS), ATC_SMEM_BYTES, s, *tq, *tkv, *tctx, p));
    TSSP_LAUNCH_CHECK("attention_tcgen05_kernel");
    return 0;
}

// one block's partials -> per-image norms (+ optional accumulation): the kernel-level entry point of the parity tests;
// the engine finishes all blocks of a batch in one launch (finish_scores)
static int op_score_finish(const float* partials, int ldp, float* norms, int ldn, int n, int T, int F, float* scores, cudaStream_t s) {
    if (ldp & 3) return fail("score_finish: partial row pitch %d must be a multiple of 4", ldp);
    ScoreBlocks sb;
    memset(&sb, 0, sizeof(sb));
    sb.F[0] = F; sb.ldp[0] = ldp; sb.norm_off[0] = 0;
    score_norms_all_kernel<<<dim3(ceil_div(F, 512), n, 1), 128, 0, s>>>(partials, 0, sb, norms, ldn, n, T);
    TSSP_LAUNCH_CHECK("score_norms_all_kernel");
    if (scores != nullptr) {
        score_accumulate_kernel<<<ceil_div(F, 128), 128, 0, s>>>(norms, ldn, n, F, scores);
        TSSP_LAUNCH_CHECK("score_accumulate_kernel");
    }
    return 0;
}

static int op_argmax(const float* logits, int ld, int n, int C, const long long* labels, int* preds, unsigned long long* correct, cudaStream_t s) {
    if (n <= 0) return 0;
    argmax_count_kernel<<<ceil_div(n * 32, 256), 256, 0, s>>>(logits, ld, n, C, labels, preds, correct);
    TSSP_LAUNCH_CHECK("argmax_count_kernel");
    return 0;
}

// ------------------------------------------------------------------------------------------------ engine
struct BlockWeights {
    const float *ln1_w, *ln1_b, *ln2_w, *ln2_b;  // fp32 (arena)
    __nv_bfloat16 *qkv_w, *proj_w, *fc1_w, *fc2_w;
    float *qkv_b, *proj_b, *fc1_b, *fc2_b;
    float *ls1, *ls2; // LayerScale gammas of the attention / MLP branch [D] (cfg.layer_scale), else nullptr
    int F, Fp;        // current width and its padding to a multiple of 8
    int F_cap;        // allocated (padded) width
    int score_off;    // column offset of this block in the concatenated score / norm vectors
};

}  // namespace tssp

// One captured launch sequence (see run_graphed): replayed with cudaGraphLaunch on the caller's stream.
struct GraphKey {
    int kind, n, flags;
    unsigned long long mask;   // per-block bits (skipped / candidate blocks)
    const void *p0, *p1;       // caller-owned pointers baked into the captured kernels (labels, counters), or nullptr
    bool operator<(const GraphKey& o) const {
        return std::tie(kind, n, flags, mask, p0, p1) < std::tie(o.kind, o.n, o.flags, o.mask, o.p0, o.p1);
    }
};
struct GraphEntry {
    cudaGraphExec_t exec;
    unsigned long long launches;  // kernels inside (tssp_launch_count grows by this on every replay)
};

struct tssp_engine {
    tssp_config_t cfg;
    int device;
    int T, M_cap, Kp, G;
    int prefix;     // tokens ahead of the patches: 1 (CLS) + cfg.dist_token + cfg.register_tokens
    int head_rows;  // rows the classifier may read: 2 with a distillation token (CLS, distillation), else 1 (CLS)
    bool dist_head; // a distillation head is loaded: logits = (cls_head(row 0) + dist_head(row 1)) / 2
    int sumF;  // sum of current F over blocks (score vector length)
    int ldn;   // pitch of the per-image norm buffer = sum of F_cap
    bool weights_loaded;
    tssp::LaunchCtx launch;  // serpentine direction / dependent-launch choice of this engine's chains
    std::vector<void*> allocs;
    std::vector<size_t> alloc_bytes;
    std::vector<tssp::BlockWeights> blk;
    // global weights
    __nv_bfloat16 *patch_w, *head0_w, *head_w, *head_dist_w;  // with a distillation head both heads are packed at 0.5 scale
    float *posmod, *final_ln_w, *final_ln_b, *head_b, *head_dist_b;
    float *norm_pre_w, *norm_pre_b;  // cfg.pre_norm: LayerNorm over every token before block 0, else nullptr
    int Cp, Hhp;  // padded classes / head hidden
    // workspace
    float* pixels[2];          // double-buffered staging of host pixel batches (fp32-sized: a uint8 batch fits too)
    tssp_pixel_input_t pix;    // format of the pixels the batch entry points are handed (tssp_set_pixel_input)
    long long* labels[2];      // ... and of their labels (same slot, same copy stream)
    long long* labels_dev;     // device-resident labels are copied here on the caller's stream: captured chains then only
                               // ever reference engine-owned label buffers (a fresh tensor per batch would force a re-capture)
    cudaStream_t copy_stream;
    cudaEvent_t ev_copied[2], ev_consumed[2], ev_labels_done[2];
    cudaEvent_t ev_part[3];  // the leading parts of a split first batch have landed (tssp_s1_batch)
    bool s1_fresh;         // no batch since tssp_s1_reset: nothing is running that a host copy could hide behind
    int next_slot, staged_slot;
    int host_slot;         // slot of the host batch staged by the running entry point (-1: none); see finish_host_batch
    __nv_bfloat16 *patchA, *xn, *qkv, *ctx, *h, *head_hidden;
    __nv_bfloat16* cls_norm;   // final LayerNorm of the head rows: [head_rows][max_images][D] (CLS rows, then distillation rows)
    float *x, *partials, *norms, *scores, *logits;
    float* qk_norms;  // [M_cap][2*heads]: |q|^2 and |k|^2 per (token, head), written by the QKV GEMM epilogue
    size_t partials_stride;  // floats between two blocks' partial buffers
    std::vector<float*> x_cache;
    int* preds;
    unsigned long long* counts;  // [B + 1]
    int32_t attn_present[TSSP_MAX_BLOCKS];
    // captured launch sequences
    cudaStream_t capture_stream;
    std::map<GraphKey, GraphEntry> graphs;
    unsigned long long graph_epoch;  // g_launch_epoch the cached graphs were captured under
};

namespace tssp {

// Device-block pool: the buffers of a destroyed engine are kept (per device, by exact size) and handed to the next
// engine that asks for the same sizes -- the pruning flow builds an engine per model copy / per mutated signature, and
// cudaMalloc of its 3-4 GB costs 30 ms alone and 200 ms when several ranks of a node allocate at once. Nothing in the
// engine relies on fresh memory being zero (every buffer is written before it is read; the GPU tests run on recycled
// blocks throughout). TSSP_POOL_MB caps the pooled bytes per process (default 16384; 0 disables); tssp_trim_pool()
// returns everything to the driver (torch's allocator cannot see or reclaim parked blocks: the Python layer calls it
// from release_engine(trim=True) and on a torch out-of-memory error).
struct PoolKey {
    int device;
    size_t bytes;
    bool operator<(const PoolKey& o) const { return std::tie(device, bytes) < std::tie(o.device, o.bytes); }
};
static std::multimap<PoolKey, void*> g_pool;  // guarded by g_lib_mutex
static size_t g_pool_bytes = 0;
static size_t pool_cap_bytes() {
    static const size_t cap = [] { const char* e = getenv("TSSP_POOL_MB"); return (e != nullptr ? static_cast<size_t>(atoll(e)) : 16384u) << 20; }();
    return cap;
}
static void pool_release(int device, void* p, size_t bytes) {
    // TSSP_POOL_POISON=1 (tests): parked blocks are filled with 0xFF bytes (NaN patterns), so an engine that read a
    // buffer before writing it would show
    static const bool poison = [] { const char* e = getenv("TSSP_POOL_POISON"); return e != nullptr && strcmp(e, "1") == 0; }();
    if (poison) cudaMemset(p, 0xFF, bytes);
    if (g_pool_bytes + bytes > pool_cap_bytes()) {
        cudaFree(p);
        return;
    }
    g_pool.insert({PoolKey{device, bytes}, p});
    g_pool_bytes += bytes;
}
static void pool_trim() {
    int prev = 0;
    cudaGetDevice(&prev);
    for (auto& kv : g_pool) {
        cudaSetDevice(kv.first.device);
        cudaFree(kv.second);
    }
    cudaSetDevice(prev);
    g_pool.clear();
    g_pool_bytes = 0;
}

template <typename Tp>
static int dev_alloc(tssp_engine* e, Tp** out, size_t count) {
    void* p = nullptr;
    size_t bytes = count * sizeof(Tp);
    if (bytes == 0) bytes = 256;
    auto it = g_pool.find(PoolKey{e->device, bytes});
    if (it != g_pool.end()) {
        p = it->second;
        g_pool.erase(it);
        g_pool_bytes -= bytes;
    } else {
        cudaError_t err = cudaMalloc(&p, bytes);
        if (err != cudaSuccess && !g_pool.empty()) {  // out of memory with blocks parked in the pool: give them back and retry
            cudaGetLastError();
            pool_trim();
            err = cudaMalloc(&p, bytes);
        }
        if (err != cudaSuccess) return fail("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(err));
    }
    e->allocs.push_back(p);
    e->alloc_bytes.push_back(bytes);
    *out = static_cast<Tp*>(p);
    return 0;
}

static int validate(const tssp_config_t& c) {
    if (c.dist_token != 0 && c.dist_token != 1) return fail("config: dist_token=%d must be 0 or 1", c.dist_token);
    if (c.register_tokens < 0 || c.register_tokens > TSSP_MAX_REGISTER_TOKENS)
        return fail("config: register_tokens=%d must be in [0,%d]", c.register_tokens, TSSP_MAX_REGISTER_TOKENS);
    if (c.dist_token && c.register_tokens > 0) return fail("config: a distillation token and register tokens cannot be combined");
    if (c.pos_patches_only != 0 && c.pos_patches_only != 1) return fail("config: pos_patches_only=%d must be 0 or 1", c.pos_patches_only);
    if (c.layer_scale != 0 && c.layer_scale != 1) return fail("config: layer_scale=%d must be 0 or 1", c.layer_scale);
    if (c.pre_norm != 0 && c.pre_norm != 1) return fail("config: pre_norm=%d must be 0 or 1", c.pre_norm);
    if (c.ffn_act != TSSP_FFN_GELU && c.ffn_act != TSSP_FFN_QUICK_GELU)
        return fail("config: ffn_act=%d must be %d (erf GELU) or %d (QuickGELU)", c.ffn_act, TSSP_FFN_GELU, TSSP_FFN_QUICK_GELU);
    if (c.ffn_act == TSSP_FFN_QUICK_GELU && c.score_point != 1)
        return fail("config: QuickGELU is scored before the activation only (score_point=1, got %d)", c.score_point);
    const int prefix = 1 + c.dist_token + c.register_tokens;
    if (c.n_blocks < 1 || c.n_blocks > TSSP_MAX_BLOCKS) return fail("config: n_blocks=%d out of range", c.n_blocks);
    if ((c.hidden % 128 && c.hidden != 192) || c.hidden > 1024 || c.hidden < 128)
        return fail("config: hidden=%d must be 192 or a multiple of 128 in [128,1024]", c.hidden);
    if (c.heads * 64 != c.hidden) return fail("config: head_dim must be 64 (hidden=%d heads=%d)", c.hidden, c.heads);
    if (c.patch_size < 1 || c.image_size % c.patch_size) return fail("config: image %d / patch %d unsupported", c.image_size, c.patch_size);
    const int G = c.image_size / c.patch_size, T = G * G + prefix;
    if (T < 32 || T > ATL_MAX_T) return fail("config: tokens per image T=%d must be in [32,%d]", T, ATL_MAX_T);
    if (c.channels < 1) return fail("config: channels=%d", c.channels);
    if (c.max_images < 1) return fail("config: max_images=%d", c.max_images);
    for (int b = 0; b < c.n_blocks; ++b)
        if (c.ffn_dims[b] < 1) return fail("config: ffn_dims[%d]=%d", b, c.ffn_dims[b]);
    return 0;
}

static int engine_create(const tssp_config_t* cfg, int device, tssp_engine** out) {
    TSSP_TRY(validate(*cfg));
    const int prefix = 1 + cfg->dist_token + cfg->register_tokens;
    int n_dev = 0;
    TSSP_CUDA(cudaGetDeviceCount(&n_dev));
    if (device < 0 || device >= n_dev) return fail("device %d out of range (%d visible)", device, n_dev);
    DeviceScope on_device(device);  // the caller's current device is restored on return
    int cc_major = 0, cc_minor = 0;
    TSSP_CUDA(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
    TSSP_CUDA(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, device));
    if (cc_major != 10) return fail("device %d is sm_%d%d; this library contains sm_100a code only", device, cc_major, cc_minor);
    tssp_engine* e = new tssp_engine();
    e->cfg = *cfg;
    e->device = device;
    e->weights_loaded = false;
    const int D = cfg->hidden, B = cfg->n_blocks;
    e->G = cfg->image_size / cfg->patch_size;
    e->prefix = prefix;
    e->head_rows = 1 + cfg->dist_token;
    e->dist_head = false;
    e->T = e->G * e->G + prefix;
    e->M_cap = cfg->max_images * e->T;
    e->Kp = patch_width(cfg->channels, cfg->patch_size);
    e->Cp = round_up(cfg->n_classes > 0 ? cfg->n_classes : 8, 8);
    e->Hhp = cfg->head_hidden > 0 ? round_up(cfg->head_hidden, 8) : 0;
    memcpy(e->attn_present, cfg->attn_present, sizeof(e->attn_present));
    int rc = 0;
    auto A = [&](auto** p, size_t n) { if (rc == 0) rc = dev_alloc(e, p, n); };
    // weights
    A(&e->patch_w, static_cast<size_t>(D) * e->Kp);
    A(&e->posmod, static_cast<size_t>(e->T) * D);
    A(&e->final_ln_w, D); A(&e->final_ln_b, D);
    A(&e->head0_w, static_cast<size_t>(e->Hhp) * D);
    A(&e->head_w, static_cast<size_t>(e->Cp) * (e->Hhp > 0 ? e->Hhp : D));
    A(&e->head_b, e->Cp);
    e->head_dist_w = nullptr;
    e->head_dist_b = nullptr;
    e->norm_pre_w = nullptr;
    e->norm_pre_b = nullptr;
    if (cfg->pre_norm) {
        A(&e->norm_pre_w, D);
        A(&e->norm_pre_b, D);
    }
    if (cfg->dist_token && cfg->n_classes > 0) {
        A(&e->head_dist_w, static_cast<size_t>(e->Cp) * D);
        A(&e->head_dist_b, e->Cp);
    }
    e->blk.resize(B);
    int Fp_max = 0, off = 0;
    for (int b = 0; b < B; ++b) {
        BlockWeights& w = e->blk[b];
        w.F = cfg->ffn_dims[b]; w.Fp = round_up(w.F, 8); w.F_cap = w.Fp; w.score_off = off;
        off += w.F_cap;
        if (w.Fp > Fp_max) Fp_max = w.Fp;
        float *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr, *ln2b = nullptr;  // A() leaves them alone once an allocation has failed
        A(&ln1w, D); A(&ln1b, D); A(&ln2w, D); A(&ln2b, D);
        w.ln1_w = ln1w; w.ln1_b = ln1b; w.ln2_w = ln2w; w.ln2_b = ln2b;
        A(&w.qkv_w, static_cast<size_t>(3) * D * D); A(&w.qkv_b, 3 * D);
        A(&w.proj_w, static_cast<size_t>(D) * D); A(&w.proj_b, D);
        A(&w.fc1_w, static_cast<size_t>(w.F_cap) * D); A(&w.fc1_b, w.F_cap);
        A(&w.fc2_w, static_cast<size_t>(D) * w.F_cap); A(&w.fc2_b, D);
        w.ls1 = w.ls2 = nullptr;
        if (cfg->layer_scale) { A(&w.ls1, D); A(&w.ls2, D); }
    }
    e->ldn = off;
    e->sumF = 0;
    for (int b = 0; b < B; ++b) e->sumF += e->blk[b].F;
    // workspace
    const size_t M = e->M_cap;
    for (int i = 0; i < 2; ++i) {
        A(&e->pixels[i], static_cast<size_t>(cfg->max_images) * cfg->channels * cfg->image_size * cfg->image_size);
        A(&e->labels[i], cfg->max_images);
    }
    A(&e->labels_dev, cfg->max_images);
    A(&e->patchA, M * e->Kp);
    A(&e->x, M * D);
    A(&e->xn, M * D);
    A(&e->qkv, M * 3 * D);
    A(&e->ctx, M * D);
    A(&e->qk_norms, M * 2 * cfg->heads);
    A(&e->h, M * Fp_max);
    e->partials_stride = static_cast<size_t>(ceil_div(e->M_cap, 32)) * 2 * Fp_max;
    A(&e->partials, e->partials_stride * B);
    A(&e->norms, static_cast<size_t>(cfg->max_images) * e->ldn);
    A(&e->scores, e->ldn);
    A(&e->cls_norm, static_cast<size_t>(e->head_rows) * cfg->max_images * D);
    A(&e->head_hidden, static_cast<size_t>(cfg->max_images) * (e->Hhp > 0 ? e->Hhp : 8));
    A(&e->logits, static_cast<size_t>(cfg->max_images) * e->Cp);
    A(&e->preds, cfg->max_images);
    A(&e->counts, B + 1);
    if (cfg->cache_blocks) {
        e->x_cache.resize(B, nullptr);
        for (int b = 0; b < B; ++b) A(&e->x_cache[b], M * D);
    }
    if (rc != 0) {
        for (size_t i = 0; i < e->allocs.size(); ++i) pool_release(e->device, e->allocs[i], e->alloc_bytes[i]);
        delete e;
        return rc;
    }
    e->next_slot = 0;
    e->pix = tssp_pixel_input_t{TSSP_PIXELS_F32, 1.0f, {0.0f, 0.0f, 0.0f, 0.0f}, {1.0f, 1.0f, 1.0f, 1.0f}};
    e->staged_slot = -1;
    e->host_slot = -1;
    e->s1_fresh = false;
    e->launch.pdl_auto = cfg->hidden < 768;
    e->graph_epoch = g_launch_epoch;
    cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&e->capture_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&e->ev_copied[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->ev_consumed[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->ev_labels_done[i], cudaEventDisableTiming);
    }
    for (int k = 0; k < 3; ++k) cudaEventCreateWithFlags(&e->ev_part[k], cudaEventDisableTiming);
    cudaMemset(e->scores, 0, sizeof(float) * e->ldn);
    cudaMemset(e->norms, 0, sizeof(float) * static_cast<size_t>(cfg->max_images) * e->ldn);
    cudaMemset(e->counts, 0, sizeof(unsigned long long) * (B + 1));
    *out = e;
    return 0;
}

// posmod[0] = cls + pos[0]; posmod[t < prefix] = tokens[t - 1] + pos[t] (the distillation token or the register tokens);
// posmod[t >= prefix] = pos[t] + conv_bias (so the patch GEMM needs no bias and the prefix rows, whose im2col rows are
// zero, receive exactly token + pos: HF ViTEmbeddings.forward / DeiTEmbeddings.forward, timm _pos_embed). With a
// class-free position table (pos_patches_only = 1, timm no_embed_class) pos has G^2 rows: the prefix rows are the
// bare tokens and patch row t takes pos[t - prefix].
__global__ void build_posmod_kernel(const float* __restrict__ pos, const float* __restrict__ cls, const float* __restrict__ tokens,
                                    const float* __restrict__ conv_b, float* __restrict__ out, int T, int D, int prefix,
                                    int pos_covers_prefix) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T * D) return;
    const int t = i / D, d = i % D;
    if (pos_covers_prefix) {
        out[i] = pos[i] + (t < prefix ? (t == 0 ? cls[d] : tokens[(t - 1) * D + d]) : (conv_b != nullptr ? conv_b[d] : 0.0f));
    } else {
        out[i] = t < prefix ? (t == 0 ? cls[d] : tokens[(t - 1) * D + d])
                            : pos[(t - prefix) * D + d] + (conv_b != nullptr ? conv_b[d] : 0.0f);
    }
}

__global__ void copy_pad_f32_kernel(const float* __restrict__ in, int n, float* __restrict__ out, int n_pad, float scale) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_pad) out[i] = (in != nullptr && i < n) ? in[i] * scale : 0.0f;
}

// out[0, n_pad) = in[0, n), zero padded
static int copy_vec(const float* in, int n, float* out, int n_pad, cudaStream_t s, float scale = 1.0f) {
    copy_pad_f32_kernel<<<ceil_div(n_pad, 256), 256, 0, s>>>(in, n, out, n_pad, scale);
    TSSP_LAUNCH_CHECK("copy_pad_f32_kernel");
    return 0;
}

static int pack_ffn(tssp_engine* e, int b, int F, const float* fc1_w, const float* fc1_b, const float* fc2_w, cudaStream_t s) {
    BlockWeights& w = e->blk[b];
    const int D = e->cfg.hidden;
    const int Fp = round_up(F, 8);
    if (Fp > w.F_cap) return fail("block %d: FFN width %d exceeds the allocated %d", b, F, w.F_cap);
    w.F = F; w.Fp = Fp;
    TSSP_TRY(op_cast(fc1_w, F, D, D, w.fc1_w, Fp, D, D, s));
    TSSP_TRY(copy_vec(fc1_b, F, w.fc1_b, Fp, s));
    TSSP_TRY(op_cast(fc2_w, D, F, F, w.fc2_w, D, Fp, Fp, s));
    return 0;
}

static int engine_load(tssp_engine* e, const float* const* t, int n_entries, cudaStream_t s) {
    const tssp_config_t& c = e->cfg;
    const int D = c.hidden, B = c.n_blocks;
    const int n_expected = TSSP_W_GLOBAL_COUNT + B * TSSP_BW_COUNT;
    if (n_entries != n_expected)
        return fail("load_weights: expected %d pointers (TSSP_W_GLOBAL_COUNT + %d blocks * TSSP_BW_COUNT), got %d", n_expected, B, n_entries);
    auto need = [&](int idx, const char* name) -> int { return t[idx] == nullptr ? fail("load_weights: %s is NULL", name) : 0; };
    TSSP_TRY(need(TSSP_W_PATCH_W, "patch_w")); TSSP_TRY(need(TSSP_W_CLS, "cls_token")); TSSP_TRY(need(TSSP_W_POS, "pos_embed"));
    TSSP_TRY(need(TSSP_W_FINAL_LN_W, "final_ln_w")); TSSP_TRY(need(TSSP_W_FINAL_LN_B, "final_ln_b"));
    // the slots of an option the config leaves off must be NULL: a table built for another config is refused
    auto unused = [&](int idx, const char* slot, const char* field) -> int {
        return t[idx] != nullptr ? fail("load_weights: %s is set, but the config has %s=0", slot, field) : 0;
    };
    if (!c.dist_token) {
        TSSP_TRY(unused(TSSP_W_DIST_TOKEN, "TSSP_W_DIST_TOKEN", "dist_token"));
        TSSP_TRY(unused(TSSP_W_HEAD_DIST_W, "TSSP_W_HEAD_DIST_W", "dist_token"));
        TSSP_TRY(unused(TSSP_W_HEAD_DIST_B, "TSSP_W_HEAD_DIST_B", "dist_token"));
    }
    if (c.register_tokens == 0) TSSP_TRY(unused(TSSP_W_REG_TOKENS, "TSSP_W_REG_TOKENS", "register_tokens"));
    if (!c.pre_norm) {
        TSSP_TRY(unused(TSSP_W_NORM_PRE_W, "TSSP_W_NORM_PRE_W", "pre_norm"));
        TSSP_TRY(unused(TSSP_W_NORM_PRE_B, "TSSP_W_NORM_PRE_B", "pre_norm"));
    }
    for (int b = 0; b < B; ++b) {
        const float* const* w = t + TSSP_W_GLOBAL_COUNT + b * TSSP_BW_COUNT;
        if (!c.layer_scale && (w[TSSP_BW_LS1] != nullptr || w[TSSP_BW_LS2] != nullptr))
            return fail("load_weights: block %d TSSP_BW_LS%d is set, but the config has layer_scale=0", b, w[TSSP_BW_LS1] != nullptr ? 1 : 2);
        if (c.layer_scale && w[TSSP_BW_LS2] == nullptr) return fail("load_weights: block %d LS2 gamma is NULL", b);
        if (c.layer_scale && c.attn_present[b] && w[TSSP_BW_LS1] == nullptr) return fail("load_weights: block %d LS1 gamma is NULL", b);
    }
    if (c.register_tokens > 0 && t[TSSP_W_REG_TOKENS] == nullptr) return fail("load_weights: register tokens are NULL");
    if (c.pre_norm && (t[TSSP_W_NORM_PRE_W] == nullptr || t[TSSP_W_NORM_PRE_B] == nullptr))
        return fail("load_weights: norm_pre weight or bias is NULL");
    const bool dist_head = c.dist_token && t[TSSP_W_HEAD_DIST_W] != nullptr;
    if (c.dist_token) {
        if (t[TSSP_W_DIST_TOKEN] == nullptr) return fail("load_weights: distillation token is NULL");
        if (dist_head && c.n_classes <= 0) return fail("load_weights: a distillation head needs n_classes > 0");
        if (dist_head && c.head_hidden > 0) return fail("load_weights: a distillation head cannot be combined with a Sequential head");
    }
    const int K = c.channels * c.patch_size * c.patch_size;  // Kp = K rounded up to 8: zero columns past K
    TSSP_TRY(op_cast(t[TSSP_W_PATCH_W], D, K, K, e->patch_w, D, e->Kp, e->Kp, s));
    build_posmod_kernel<<<ceil_div(e->T * D, 256), 256, 0, s>>>(t[TSSP_W_POS], t[TSSP_W_CLS],
                                                               t[c.dist_token ? TSSP_W_DIST_TOKEN : TSSP_W_REG_TOKENS], t[TSSP_W_PATCH_B],
                                                               e->posmod, e->T, D, e->prefix, !c.pos_patches_only);
    TSSP_LAUNCH_CHECK("build_posmod_kernel");
    TSSP_TRY(copy_vec(t[TSSP_W_FINAL_LN_W], D, e->final_ln_w, D, s));
    TSSP_TRY(copy_vec(t[TSSP_W_FINAL_LN_B], D, e->final_ln_b, D, s));
    if (c.pre_norm) {
        TSSP_TRY(copy_vec(t[TSSP_W_NORM_PRE_W], D, e->norm_pre_w, D, s));
        TSSP_TRY(copy_vec(t[TSSP_W_NORM_PRE_B], D, e->norm_pre_b, D, s));
    }
    if (c.n_classes > 0 && dist_head) {
        // (cls_head(x0) + dist_head(x1)) / 2 as two GEMMs into the same logits (run_head): both heads at half scale
        TSSP_TRY(need(TSSP_W_HEAD_W, "head_w"));
        TSSP_TRY(op_cast(t[TSSP_W_HEAD_W], c.n_classes, D, D, e->head_w, e->Cp, D, D, s, 0.5f));
        TSSP_TRY(copy_vec(t[TSSP_W_HEAD_B], c.n_classes, e->head_b, e->Cp, s, 0.5f));
        TSSP_TRY(op_cast(t[TSSP_W_HEAD_DIST_W], c.n_classes, D, D, e->head_dist_w, e->Cp, D, D, s, 0.5f));
        TSSP_TRY(copy_vec(t[TSSP_W_HEAD_DIST_B], c.n_classes, e->head_dist_b, e->Cp, s, 0.5f));
    } else if (c.n_classes > 0) {
        TSSP_TRY(need(TSSP_W_HEAD_W, "head_w"));
        if (c.head_hidden > 0) {
            TSSP_TRY(need(TSSP_W_HEAD0_W, "head0_w"));
            TSSP_TRY(op_cast(t[TSSP_W_HEAD0_W], c.head_hidden, D, D, e->head0_w, e->Hhp, D, D, s));
            TSSP_TRY(op_cast(t[TSSP_W_HEAD_W], c.n_classes, c.head_hidden, c.head_hidden, e->head_w, e->Cp, e->Hhp, e->Hhp, s));
        } else {
            TSSP_TRY(op_cast(t[TSSP_W_HEAD_W], c.n_classes, D, D, e->head_w, e->Cp, D, D, s));
        }
        TSSP_TRY(copy_vec(t[TSSP_W_HEAD_B], c.n_classes, e->head_b, e->Cp, s));
    }
    for (int b = 0; b < B; ++b) {
        const float* const* w = t + TSSP_W_GLOBAL_COUNT + b * TSSP_BW_COUNT;
        BlockWeights& bw = e->blk[b];
        static const int required[] = {TSSP_BW_LN2_W, TSSP_BW_LN2_B, TSSP_BW_FC1_W, TSSP_BW_FC2_W};
        for (int idx : required) if (w[idx] == nullptr) return fail("load_weights: block %d entry %d is NULL", b, idx);
        TSSP_TRY(copy_vec(w[TSSP_BW_LN2_W], D, const_cast<float*>(bw.ln2_w), D, s));
        TSSP_TRY(copy_vec(w[TSSP_BW_LN2_B], D, const_cast<float*>(bw.ln2_b), D, s));
        if (e->attn_present[b]) {
            static const int req_attn[] = {TSSP_BW_LN1_W, TSSP_BW_LN1_B, TSSP_BW_Q_W, TSSP_BW_K_W, TSSP_BW_V_W, TSSP_BW_PROJ_W};
            for (int idx : req_attn) if (w[idx] == nullptr) return fail("load_weights: block %d attention entry %d is NULL", b, idx);
            TSSP_TRY(copy_vec(w[TSSP_BW_LN1_W], D, const_cast<float*>(bw.ln1_w), D, s));
            TSSP_TRY(copy_vec(w[TSSP_BW_LN1_B], D, const_cast<float*>(bw.ln1_b), D, s));
            TSSP_TRY(op_cast(w[TSSP_BW_Q_W], D, D, D, bw.qkv_w, D, D, D, s));
            TSSP_TRY(op_cast(w[TSSP_BW_K_W], D, D, D, bw.qkv_w + static_cast<size_t>(D) * D, D, D, D, s));
            TSSP_TRY(op_cast(w[TSSP_BW_V_W], D, D, D, bw.qkv_w + static_cast<size_t>(2) * D * D, D, D, D, s));
            TSSP_TRY(copy_vec(w[TSSP_BW_Q_B], D, bw.qkv_b, D, s));
            TSSP_TRY(copy_vec(w[TSSP_BW_K_B], D, bw.qkv_b + D, D, s));
            TSSP_TRY(copy_vec(w[TSSP_BW_V_B], D, bw.qkv_b + 2 * D, D, s));
            TSSP_TRY(op_cast(w[TSSP_BW_PROJ_W], D, D, D, bw.proj_w, D, D, D, s));
            TSSP_TRY(copy_vec(w[TSSP_BW_PROJ_B], D, bw.proj_b, D, s));
        }
        TSSP_TRY(pack_ffn(e, b, bw.F, w[TSSP_BW_FC1_W], w[TSSP_BW_FC1_B], w[TSSP_BW_FC2_W], s));
        TSSP_TRY(copy_vec(w[TSSP_BW_FC2_B], D, bw.fc2_b, D, s));
        if (c.layer_scale) {
            TSSP_TRY(copy_vec(w[TSSP_BW_LS1], D, bw.ls1, D, s));  // NULL (no attention) -> zeros, never read
            TSSP_TRY(copy_vec(w[TSSP_BW_LS2], D, bw.ls2, D, s));
        }
    }
    e->dist_head = dist_head;
    e->weights_loaded = true;
    return 0;
}

// ---- host batches ----------------------------------------------------------------------------------
// Host pixels (and labels) are staged through two device slots on the engine's copy stream, so that the transfer of
// batch k+1 runs under the kernels of batch k. LIFETIME RULE of the C ABI: a host buffer belongs to the caller again as
// soon as the entry point returns -- every entry point that staged host data ends with finish_host_batch(), which
// blocks the HOST until the copies out of the caller's buffers have completed (the kernels enqueued behind them keep
// the GPU busy meanwhile). A DataLoader(pin_memory=True) batch that is dropped or overwritten right after the call is
// therefore safe; torch's pinned-memory allocator knows nothing about the engine's private copy stream.
// `bounds` (optional): up to three ascending image counts 0 < b0 < b1 < b2 < n; the pixels are copied as n_bounds + 1
// consecutive parts, ev_part[i] fires when the images below bounds[i] have landed, and only the FIRST part is waited
// for on `s` here -- the caller waits for the others as it reaches them.
static size_t pixel_bytes(const tssp_engine* e) { return e->pix.format == TSSP_PIXELS_U8 ? 1 : sizeof(float); }

static int stage_batch(tssp_engine* e, const void* pixels, const int64_t* labels, int n, int on_host, const void** dev_pixels,
                       const long long** dev_labels, cudaStream_t s, const int* bounds = nullptr, int n_bounds = 0, int* slot_out = nullptr) {
    if (n < 1 || n > e->cfg.max_images) return fail("batch of %d images outside [1, max_images=%d]", n, e->cfg.max_images);
    if (!e->weights_loaded) return fail("weights have not been loaded");
    if (pixels == nullptr) return fail("pixels is NULL");
    if (dev_labels != nullptr && labels == nullptr) return fail("labels is NULL");
    e->host_slot = -1;
    if (!on_host) {
        e->staged_slot = -1;
        *dev_pixels = pixels;
        if (dev_labels != nullptr) {  // stream-ordered behind the previous batch's last argmax kernel, which read this buffer
            TSSP_CUDA(cudaMemcpyAsync(e->labels_dev, labels, sizeof(int64_t) * n, cudaMemcpyDeviceToDevice, s));
            *dev_labels = e->labels_dev;
        }
        return 0;
    }
    const size_t bytes = static_cast<size_t>(n) * e->cfg.channels * e->cfg.image_size * e->cfg.image_size * pixel_bytes(e);
    const int slot = e->next_slot;
    e->next_slot ^= 1;
    e->host_slot = slot;  // from here on the caller's buffers are in use until finish_host_batch()
    TSSP_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_consumed[slot], 0));
    if (dev_labels != nullptr) {
        TSSP_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_labels_done[slot], 0));
        TSSP_CUDA(cudaMemcpyAsync(e->labels[slot], labels, sizeof(int64_t) * n, cudaMemcpyHostToDevice, e->copy_stream));
        *dev_labels = e->labels[slot];
    }
    if (bounds != nullptr && n_bounds > 0) {
        const size_t img_bytes = bytes / n;
        size_t done = 0;
        for (int i = 0; i <= n_bounds; ++i) {
            const size_t upto = (i < n_bounds ? static_cast<size_t>(bounds[i]) : static_cast<size_t>(n)) * img_bytes;
            TSSP_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(e->pixels[slot]) + done, reinterpret_cast<const char*>(pixels) + done,
                                      upto - done, cudaMemcpyHostToDevice, e->copy_stream));
            TSSP_CUDA(cudaEventRecord(i < n_bounds ? e->ev_part[i] : e->ev_copied[slot], e->copy_stream));
            done = upto;
        }
        TSSP_CUDA(cudaStreamWaitEvent(s, e->ev_part[0], 0));
    } else {
        TSSP_CUDA(cudaMemcpyAsync(e->pixels[slot], pixels, bytes, cudaMemcpyHostToDevice, e->copy_stream));
        TSSP_CUDA(cudaEventRecord(e->ev_copied[slot], e->copy_stream));
        TSSP_CUDA(cudaStreamWaitEvent(s, e->ev_copied[slot], 0));
    }
    if (slot_out != nullptr) *slot_out = slot;
    e->staged_slot = slot;
    *dev_pixels = e->pixels[slot];
    return 0;
}

// End of an entry point that may have staged a host batch: marks the slot's label buffer as read (`labels_used`) and
// waits, on the host, for the copies out of the caller's buffers. `rc` is the entry point's status so far: the wait
// happens on the error path as well (the copy may already be in flight).
static int finish_host_batch(tssp_engine* e, cudaStream_t s, bool labels_used, int rc) {
    const int slot = e->host_slot;
    if (slot < 0) return rc;
    e->host_slot = -1;
    if (labels_used && rc == 0) {
        const cudaError_t er = cudaEventRecord(e->ev_labels_done[slot], s);
        if (er != cudaSuccess) rc = fail("cudaEventRecord failed: %s", cudaGetErrorString(er));
    }
    const cudaError_t err = cudaEventSynchronize(e->ev_copied[slot]);
    if (err != cudaSuccess && rc == 0) rc = fail("host-to-device copy of the batch failed: %s", cudaGetErrorString(err));
    return rc;
}

// ---- captured launch sequences -----------------------------------------------------------------------
// The per-batch chains are 90 (Stage-1 sweep) to 700 (Stage-2 search) launches of 10-200 us kernels. Issued one by one
// they leave a few microseconds between kernels and put the host on the critical path whenever a batch is short (the
// 128-image shards of an 8-GPU run, ViT-S); so every chain is captured once per (kind, batch size, flags, block masks,
// baked-in caller pointers) into a CUDA graph -- on the engine's own capture stream, the caller's stream may be the
// legacy default stream -- and replayed with one cudaGraphLaunch on the caller's stream. The kernels, their order and
// arguments are exactly those of the eager path (serpentine directions and dependent-launch edges included), so the
// bits are the same (tested). Profiling runs (tssp_profile_begin) and TSSP_GRAPHS=0 / tssp_set_graphs(0) stay eager.
enum GraphKind { GK_S1 = 1, GK_FORWARD = 2, GK_EVAL = 3, GK_S2 = 4 };
constexpr size_t GRAPH_CACHE_MAX = 48;
static int g_graphs = -1;  // -1: take TSSP_GRAPHS on first use
static unsigned long long g_graph_captures = 0;  // chains captured since load (tssp_graph_capture_count: tests)
static bool graphs_enabled() {
    if (g_graphs < 0) {
        const char* e = getenv("TSSP_GRAPHS");
        g_graphs = (e != nullptr && strcmp(e, "0") == 0) ? 0 : 1;
    }
    return g_graphs == 1 && !g_prof_on;
}

static void drop_graphs(tssp_engine* e) {
    for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second.exec);
    e->graphs.clear();
}

template <typename F>
static int run_graphed(tssp_engine* e, const GraphKey& key, cudaStream_t s, F&& body) {
    if (!graphs_enabled()) return body(s);
    if (e->graph_epoch != g_launch_epoch) {  // tile form / trace buffer changed since the capture
        drop_graphs(e);
        e->graph_epoch = g_launch_epoch;
    }
    auto it = e->graphs.find(key);
    if (it == e->graphs.end()) {
        if (e->graphs.size() >= GRAPH_CACHE_MAX) drop_graphs(e);
        const unsigned long long before = g_launches;
        TSSP_CUDA(cudaStreamBeginCapture(e->capture_stream, cudaStreamCaptureModeRelaxed));
        const int rc = body(e->capture_stream);
        cudaGraph_t graph = nullptr;
        const cudaError_t err = cudaStreamEndCapture(e->capture_stream, &graph);
        GraphEntry entry;
        entry.launches = g_launches - before;
        g_launches = before;  // nothing has run yet: replays do the counting
        if (rc != 0) {
            if (graph != nullptr) cudaGraphDestroy(graph);
            cudaGetLastError();
            return rc;
        }
        if (err != cudaSuccess || graph == nullptr) return fail("stream capture failed: %s", cudaGetErrorString(err));
        const cudaError_t ierr = cudaGraphInstantiate(&entry.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ierr != cudaSuccess) return fail("cudaGraphInstantiate failed: %s", cudaGetErrorString(ierr));
        it = e->graphs.emplace(key, entry).first;
        ++g_graph_captures;
    }
    TSSP_CUDA(cudaGraphLaunch(it->second.exec, s));
    g_launches += it->second.launches;
    return 0;
}

static unsigned long long block_mask(const int32_t* flags, int B) {
    unsigned long long m = 0;
    if (flags != nullptr)
        for (int b = 0; b < B; ++b)
            if (flags[b] != 0) m |= 1ull << b;
    return m;
}

// ---- launch sequences ----------------------------------------------------------------------------
// patch extraction (HF ViTPatchEmbeddings as a GEMM over non-overlapping patches): the one kernel that reads the
// caller's / the staged pixels, kept outside the captured chains so that those do not depend on where a batch lives
static int run_im2col(tssp_engine* e, const void* dev_pixels, int n, cudaStream_t s) {
    const tssp_config_t& c = e->cfg;
    TSSP_PROF(KC_MISC, s, op_im2col(dev_pixels, e->patchA, n, c.channels, c.image_size, c.image_size, c.patch_size, e->prefix, &e->pix, s));
    if (e->staged_slot >= 0) {  // the host-staged pixel buffer may be refilled once im2col has read it
        TSSP_CUDA(cudaEventRecord(e->ev_consumed[e->staged_slot], s));
        e->staged_slot = -1;
    }
    return 0;
}

// embeddings: x = [cls | patches W^T + b] + pos      (HF ViTEmbeddings / ViTPatchEmbeddings); with a pre-norm (timm
// pre_norm=True: CLIP towers) x = norm_pre(x), in place, before block 0 (and so before the Stage-2 snapshot of block 0)
static int run_embed(tssp_engine* e, int n, cudaStream_t s) {
    e->launch.chain_dir = 0;  // every batch starts its chain in the same direction
    const tssp_config_t& c = e->cfg;
    const int M = n * e->T, D = c.hidden;
    {
        ProfScope ps(KC_MISC, s);
        broadcast_rows_kernel<<<grid_for(static_cast<long long>(M) * D / 4, 256), 256, 0, s>>>(e->posmod, e->x, n, e->T, D);
        TSSP_LAUNCH_CHECK("broadcast_rows_kernel");
    }
    TSSP_PROF(KC_PATCH, s, gemm(EPI_F32, e->patchA, e->Kp, e->patch_w, e->Kp, e->x, D, M, D, e->Kp, nullptr, nullptr, 0, e->T, 1, s));
    if (c.pre_norm) TSSP_PROF(KC_LN, s, op_layernorm_f32(e->x, D, e->norm_pre_w, e->norm_pre_b, e->x, D, M, D, c.ln_eps, s));
    return 0;
}

enum Fc1Mode { FC1_PLAIN = 0, FC1_SCORE = 1 };

// one encoder block on the fp32 residual stream e->x   (HF ViTLayer.forward; timm Block.forward)
//
// cls_only (the LAST block of a forward that only feeds the classifier): the logits depend on the CLS row of the last
// block alone, and after the attention -- which needs every token's K and V -- all of a block's work is row-wise. So the
// output projection, the LayerNorm before the FFN, fc1 and fc2 run on the n CLS rows in place (tensor maps over x / ctx with
// a row pitch of T rows) instead of on n * T rows; the other rows of x are left as they are, nobody reads them. One block
// forward of the 13 per Stage-2 candidate sweep and of every evaluation loses two thirds of its work.
// With a distillation head the classifier also reads row 1 (DeiT's distillation token): the row-wise part then runs a second
// time on the n rows 1, at base offset D with the same pitch. (Attention's first query tile already covers both rows.)
static int run_block(tssp_engine* e, int b, int n, bool skip_attn, Fc1Mode fc1_mode, bool run_fc2, cudaStream_t s, bool cls_only = false) {
    const tssp_config_t& c = e->cfg;
    const int M = n * e->T, D = c.hidden;
    BlockWeights& w = e->blk[b];
    cls_only = cls_only && fc1_mode == FC1_PLAIN && run_fc2;
    const int rows = cls_only ? n : M;              // rows the row-wise part of the block works on
    const int pitch = cls_only ? e->T * D : D;      // their distance in x / ctx
    const bool attn = e->attn_present[b] && !skip_attn;
    const bool qgelu = e->cfg.ffn_act == TSSP_FFN_QUICK_GELU;
    const int fc1_plain = qgelu ? EPI_BF16_QGELU : EPI_BF16_GELU;
    // proj / fc2 add their branch into the residual stream, scaled by the block's LayerScale gamma when the model has one
    auto residual_gemm = [&](const void* A, int lda, const __nv_bfloat16* W, int ldw, float* xr, int rows_, int K, const float* bias,
                             const float* gamma) {
        return gemm(gamma != nullptr ? EPI_F32_SCALED : EPI_F32, A, lda, W, ldw, xr, pitch, rows_, D, K, bias, nullptr, 0, e->T, 1, s,
                    nullptr, 0, 0, gamma);
    };
    if (attn) {
        TSSP_PROF(KC_LN, s, op_layernorm(e->x, D, w.ln1_w, w.ln1_b, e->xn, M, D, c.ln_eps, s));
        TSSP_PROF(KC_QKV, s, gemm(EPI_BF16_ROWNORM, e->xn, D, w.qkv_w, D, e->qkv, 3 * D, M, 3 * D, D, w.qkv_b, nullptr, 0, e->T, 0, s,
                                  e->qk_norms, 2 * c.heads, 2 * c.heads));
        TSSP_PROF(KC_ATTN, s, op_attention(e->qkv, e->ctx, n, e->T, c.heads, D, s, e->qk_norms, 2 * c.heads, /*first_tile_only=*/cls_only));
    }
    if (cls_only && e->dist_head) {
        for (int r = 0; r < 2; ++r) {
            float* xr = e->x + static_cast<size_t>(r) * D;
            if (attn) TSSP_PROF(KC_PROJ, s, residual_gemm(e->ctx + static_cast<size_t>(r) * D, pitch, w.proj_w, D, xr, n, D, w.proj_b, w.ls1));
            TSSP_PROF(KC_LN, s, op_layernorm(xr, pitch, w.ln2_w, w.ln2_b, e->xn, n, D, c.ln_eps, s));
            TSSP_PROF(KC_FC1, s, gemm(fc1_plain, e->xn, D, w.fc1_w, D, e->h, w.Fp, n, w.Fp, D, w.fc1_b, nullptr, 0, e->T, 0, s));
            TSSP_PROF(KC_FC2, s, residual_gemm(e->h, w.Fp, w.fc2_w, w.Fp, xr, n, w.Fp, w.fc2_b, w.ls2));
        }
        return 0;
    }
    if (attn) TSSP_PROF(KC_PROJ, s, residual_gemm(e->ctx, pitch, w.proj_w, D, e->x, rows, D, w.proj_b, w.ls1));
    TSSP_PROF(KC_LN, s, op_layernorm(e->x, pitch, w.ln2_w, w.ln2_b, e->xn, rows, D, c.ln_eps, s, /*stream_in=*/!cls_only));
    if (fc1_mode == FC1_SCORE) {
        // QuickGELU engines score before the activation only (validate)
        const int mode = c.score_point == 1 ? (qgelu ? EPI_BF16_QGELU_SCORE_PRE : EPI_BF16_GELU_SCORE_PRE) : EPI_BF16_GELU_SCORE;
        // per-block partial sums of squares; the square roots and the image sums are taken once per batch
        // for all blocks together (finish_scores)
        TSSP_PROF(KC_FC1, s, gemm(mode, e->xn, D, w.fc1_w, D, e->h, w.Fp, M, w.Fp, D, w.fc1_b,
                                  e->partials + static_cast<size_t>(b) * e->partials_stride, w.Fp, e->T, 0, s));
    } else {
        TSSP_PROF(KC_FC1, s, gemm(fc1_plain, e->xn, D, w.fc1_w, D, e->h, w.Fp, rows, w.Fp, D, w.fc1_b, nullptr, 0, e->T, 0, s));
    }
    if (run_fc2) TSSP_PROF(KC_FC2, s, residual_gemm(e->h, w.Fp, w.fc2_w, w.Fp, e->x, rows, w.Fp, w.fc2_b, w.ls2));
    return 0;
}

// final LayerNorm on the CLS rows + classification head -> e->logits [n, Cp]. With a distillation head (DeiT
// ForImageClassificationWithTeacher, timm's distilled models in eval) the rows 1 are normalised too, and
// logits = (cls_head(row 0) + dist_head(row 1)) / 2: the CLS GEMM stores half its result, the distillation GEMM adds half of
// its own (both heads are packed at 0.5 scale, exact in bf16 and fp32), one fp32 rounding of the sum as in the module.
static int run_head(tssp_engine* e, int n, cudaStream_t s) {
    const tssp_config_t& c = e->cfg;
    const int D = c.hidden;
    if (c.n_classes <= 0) return fail("model has no classification head: logits unavailable");
    TSSP_PROF(KC_LN, s, op_layernorm(e->x, static_cast<long long>(e->T) * D, e->final_ln_w, e->final_ln_b, e->cls_norm, n, D, c.ln_eps, s));
    if (e->dist_head) {
        __nv_bfloat16* dist_norm = e->cls_norm + static_cast<size_t>(n) * D;
        TSSP_PROF(KC_LN, s, op_layernorm(e->x + D, static_cast<long long>(e->T) * D, e->final_ln_w, e->final_ln_b, dist_norm, n, D, c.ln_eps, s));
        TSSP_PROF(KC_HEAD, s, gemm(EPI_F32, e->cls_norm, D, e->head_w, D, e->logits, e->Cp, n, e->Cp, D, e->head_b, nullptr, 0, e->T, 0, s));
        TSSP_PROF(KC_HEAD, s, gemm(EPI_F32, dist_norm, D, e->head_dist_w, D, e->logits, e->Cp, n, e->Cp, D, e->head_dist_b, nullptr, 0, e->T, 1, s));
        return 0;
    }
    if (c.head_hidden > 0) {
        TSSP_PROF(KC_HEAD, s, gemm(EPI_BF16_GELU, e->cls_norm, D, e->head0_w, D, e->head_hidden, e->Hhp, n, e->Hhp, D, nullptr, nullptr, 0, e->T, 0, s));
        TSSP_PROF(KC_HEAD, s, gemm(EPI_F32, e->head_hidden, e->Hhp, e->head_w, e->Hhp, e->logits, e->Cp, n, e->Cp, e->Hhp, e->head_b, nullptr, 0, e->T, 0, s));
    } else {
        TSSP_PROF(KC_HEAD, s, gemm(EPI_F32, e->cls_norm, D, e->head_w, D, e->logits, e->Cp, n, e->Cp, D, e->head_b, nullptr, 0, e->T, 0, s));
    }
    return 0;
}

// embeddings (from the patch matrix), all blocks, head
static int run_forward(tssp_engine* e, int n, const int32_t* skip, bool cache, cudaStream_t s, Fc1Mode fc1_mode = FC1_PLAIN) {
    const int B = e->cfg.n_blocks;
    const size_t xbytes = static_cast<size_t>(n) * e->T * e->cfg.hidden * sizeof(float);
    TSSP_TRY(run_embed(e, n, s));
    for (int b = 0; b < B; ++b) {
        if (cache) TSSP_CUDA(cudaMemcpyAsync(e->x_cache[b], e->x, xbytes, cudaMemcpyDeviceToDevice, s));
        TSSP_TRY(run_block(e, b, n, skip != nullptr && skip[b] != 0, fc1_mode, true, s, /*cls_only=*/b + 1 == B));
    }
    return run_head(e, n, s);
}

// Stage-1 finisher for one batch, all blocks at once: per-(image, neuron) norms from the sub-tile partials, then
// scores[j] += sum over this batch's images in image order (src/vit_pruning.py:151-157).
static int finish_scores(tssp_engine* e, int n, cudaStream_t s) {
    const int B = e->cfg.n_blocks;
    ScoreBlocks sb;
    int Fmax = 0;
    for (int b = 0; b < B; ++b) {
        sb.F[b] = e->blk[b].F;
        sb.ldp[b] = e->blk[b].Fp;
        sb.norm_off[b] = e->blk[b].score_off;
        if (sb.F[b] > Fmax) Fmax = sb.F[b];
    }
    {
        ProfScope ps(KC_SCORE, s);
        score_norms_all_kernel<<<dim3(ceil_div(Fmax, 512), n, B), 128, 0, s>>>(e->partials, e->partials_stride, sb, e->norms, e->ldn, n, e->T);
        TSSP_LAUNCH_CHECK("score_norms_all_kernel");
    }
    {
        ProfScope ps(KC_SCORE, s);
        score_accumulate_kernel<<<ceil_div(e->ldn, 128), 128, 0, s>>>(e->norms, e->ldn, n, e->ldn, e->scores);
        TSSP_LAUNCH_CHECK("score_accumulate_kernel");
    }
    return 0;
}

// compact copy of the batch's per-image norms into the caller's [n][sum F] buffer (GPU-count-invariant reductions)
static int copy_img_norms(tssp_engine* e, int n, float* img_norms, cudaStream_t s) {
    int dst_off = 0;
    for (int b = 0; b < e->cfg.n_blocks; ++b) {
        TSSP_CUDA(cudaMemcpy2DAsync(img_norms + dst_off, sizeof(float) * e->sumF, e->norms + e->blk[b].score_off, sizeof(float) * e->ldn,
                                    sizeof(float) * e->blk[b].F, n, cudaMemcpyDeviceToDevice, s));
        dst_off += e->blk[b].F;
    }
    return 0;
}

}  // namespace tssp

// =================================================================================================== C ABI
using namespace tssp;

// every engine entry point: library lock, the engine's launch context, the engine's device
#define TSSP_ENGINE_ENTRY(h, name)                                      \
    TSSP_ENTRY();                                                       \
    if ((h) == nullptr) return fail(name ": NULL handle");              \
    CtxScope _ctx(&(h)->launch);                                           \
    DeviceScope _dev((h)->device)

extern "C" {

int tssp_abi_version(void) { return TSSP_ABI_VERSION; }
const char* tssp_last_error(void) { return g_last_error.c_str(); }
int tssp_set_gemm_form(int ctas) {
    TSSP_ENTRY();
    if (ctas < 0 || ctas > 2) return fail("tssp_set_gemm_form: %d is not 0 (automatic), 1 (single CTA) or 2 (CTA pair)", ctas);
    g_gemm_form = ctas;
    ++g_launch_epoch;
    return 0;
}
int tssp_set_graphs(int on) {
    TSSP_ENTRY();
    if (on != 0 && on != 1) return fail("tssp_set_graphs: %d is not 0 (eager launches) or 1 (captured chains)", on);
    g_graphs = on;
    return 0;
}

unsigned long long tssp_launch_count(void) {
    TSSP_ENTRY();
    return g_launches;
}
unsigned long long tssp_graph_capture_count(void) {
    TSSP_ENTRY();
    return g_graph_captures;
}

int tssp_profile_begin(void) {
    TSSP_ENTRY();
    for (const ProfRec& r : g_prof_recs) { g_prof_pool.push_back(r.start); g_prof_pool.push_back(r.stop); }
    g_prof_recs.clear();
    g_prof_on = true;
    return 0;
}

int tssp_profile_end(double* ms_per_class, unsigned long long* launches_per_class, int n_classes) {
    TSSP_ENTRY();
    g_prof_on = false;
    if (ms_per_class == nullptr || launches_per_class == nullptr || n_classes < KC_COUNT) return fail("tssp_profile_end: need room for %d classes", (int)KC_COUNT);
    TSSP_CUDA(cudaDeviceSynchronize());
    for (int i = 0; i < n_classes; ++i) { ms_per_class[i] = 0.0; launches_per_class[i] = 0; }
    for (const ProfRec& r : g_prof_recs) {
        float ms = 0.f;
        TSSP_CUDA(cudaEventElapsedTime(&ms, r.start, r.stop));
        ms_per_class[r.cls] += ms;
        launches_per_class[r.cls] += 1;
        g_prof_pool.push_back(r.start);
        g_prof_pool.push_back(r.stop);
    }
    g_prof_recs.clear();
    return 0;
}

int tssp_create(const tssp_config_t* cfg, int device, tssp_handle_t* out) {
    TSSP_ENTRY();
    if (cfg == nullptr || out == nullptr) return fail("tssp_create: NULL argument");
    return engine_create(cfg, device, out);
}

int tssp_destroy(tssp_handle_t h) {
    TSSP_ENTRY();
    if (h == nullptr) return 0;
    DeviceScope on_device(h->device);
    cudaDeviceSynchronize();
    drop_graphs(h);
    for (size_t i = 0; i < h->allocs.size(); ++i) pool_release(h->device, h->allocs[i], h->alloc_bytes[i]);
    cudaStreamDestroy(h->copy_stream);
    cudaStreamDestroy(h->capture_stream);
    for (int i = 0; i < 2; ++i) {
        cudaEventDestroy(h->ev_copied[i]);
        cudaEventDestroy(h->ev_consumed[i]);
        cudaEventDestroy(h->ev_labels_done[i]);
    }
    for (int k = 0; k < 3; ++k) cudaEventDestroy(h->ev_part[k]);
    delete h;
    return 0;
}

int tssp_trim_pool(void) {
    TSSP_ENTRY();
    pool_trim();  // parked blocks belong to destroyed engines, and tssp_destroy synchronised their device
    return 0;
}

int tssp_load_weights(tssp_handle_t h, const float* const* table, int n_entries, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_load_weights");
    if (table == nullptr) return fail("tssp_load_weights: NULL argument");
    drop_graphs(h);
    return engine_load(h, table, n_entries, static_cast<cudaStream_t>(stream));
}

int tssp_update_ffn(tssp_handle_t h, int block, int new_F, const float* fc1_w, const float* fc1_b, const float* fc2_w, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_update_ffn");
    if (fc1_w == nullptr || fc2_w == nullptr) return fail("tssp_update_ffn: NULL argument");
    if (block < 0 || block >= h->cfg.n_blocks) return fail("tssp_update_ffn: block %d out of range", block);
    if (new_F < 1) return fail("tssp_update_ffn: new_F=%d", new_F);
    drop_graphs(h);  // captured GEMMs carry the old width
    TSSP_TRY(pack_ffn(h, block, new_F, fc1_w, fc1_b, fc2_w, static_cast<cudaStream_t>(stream)));
    h->sumF = 0;
    for (int b = 0; b < h->cfg.n_blocks; ++b) h->sumF += h->blk[b].F;
    return 0;
}

int tssp_set_attention(tssp_handle_t h, const int32_t* present) {
    TSSP_ENGINE_ENTRY(h, "tssp_set_attention");
    if (present == nullptr) return fail("tssp_set_attention: NULL argument");
    for (int b = 0; b < h->cfg.n_blocks; ++b)
        if (present[b] && !h->cfg.attn_present[b]) return fail("tssp_set_attention: block %d has no attention weights loaded", b);
    drop_graphs(h);
    for (int b = 0; b < h->cfg.n_blocks; ++b) h->attn_present[b] = present[b] ? 1 : 0;
    return 0;
}

int tssp_set_pixel_input(tssp_handle_t h, const tssp_pixel_input_t* input) {
    TSSP_ENGINE_ENTRY(h, "tssp_set_pixel_input");
    if (input == nullptr) return fail("tssp_set_pixel_input: NULL argument");
    TSSP_TRY(check_pixel_input(*input, h->cfg.channels, "tssp_set_pixel_input"));
    h->pix = *input;
    return 0;
}

int tssp_s1_reset(tssp_handle_t h, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_s1_reset");
    TSSP_CUDA(cudaMemsetAsync(h->scores, 0, sizeof(float) * h->ldn, static_cast<cudaStream_t>(stream)));
    h->s1_fresh = true;
    return 0;
}

// Stage-1 forward of n device-resident images: patch extraction, then ONE captured chain (embeddings, the blocks up
// to the last fc1, score finisher)
static int s1_sweep(tssp_engine* h, const void* px, int n, float* img_norms, cudaStream_t s) {
    TSSP_TRY(run_im2col(h, px, n, s));
    const GraphKey key{GK_S1, n, h->cfg.score_point, 0ull, nullptr, nullptr};
    TSSP_TRY(run_graphed(h, key, s, [&](cudaStream_t gs) -> int {
        TSSP_TRY(run_embed(h, n, gs));
        const int B = h->cfg.n_blocks;
        // everything after the last block's fc1 (its fc2, the final LayerNorm, the head) cannot influence a score
        for (int b = 0; b < B; ++b) TSSP_TRY(run_block(h, b, n, false, FC1_SCORE, b + 1 < B, gs));
        return finish_scores(h, n, gs);
    }));
    if (img_norms != nullptr) TSSP_TRY(copy_img_norms(h, n, img_norms, s));
    return 0;
}

// The first host batch after a reset has no running kernels to hide its copy behind. It is copied in two parts (a
// quarter of the images, then the rest) and swept as two sub-batches, so that the kernels of the leading images run under
// the transfer of the rest. Every part is a multiple of 32 / gcd(T, 32) images, so n_part * T is a multiple of 32 rows:
// every image keeps its position inside the 32-row score sub-tiles, the per-image partial sums and the image order of
// the accumulation are those of the unsplit batch -- same bits (tested). A finer split (n/8, n/8, n/4, n/2) was measured
// 1.4 ms per sweep SLOWER: 32- and 64-image sub-batches fill the GEMM waves too badly to repay the earlier start
// (profiles/e2e_phases_r1.txt), so it was removed. Round 2, host-to-device at 55 GB/s: a single 128-image batch (the 8-GPU
// per-rank step) takes 6.45 ms end to end split and 6.86 ms unsplit; four batches of 256 are indifferent (41.82 / 41.83 ms).
// Re-measured with the chains captured, 4 ranks copying at once (profiles/e2e_scaling_probe_r2.txt): quarter split 11.4 / 6.2 ms
// per call at 256 / 128 images per rank, unsplit 12.4 / 6.8, (n/8, n/4, n/2) 12.1 / 7.6, equal quarters 12.4 / 7.5, thirds 12.0 / 6.8.
static int s1_split_bounds(const tssp_engine* h, int n, int* bounds) {
    if (n < 128) return 0;
    int g = h->T, r = 32;
    while (r) { const int t = g % r; g = r; r = t; }  // gcd(T, 32)
    const int k = 32 / g;
    int b = n / 4;
    if (b < 32) b = 32;
    b = (b + k - 1) / k * k;
    if (b >= n) return 0;
    bounds[0] = b;
    return 1;
}

static int s1_batch(tssp_engine* h, const float* pixels, int n, int pixels_on_host, float* img_norms, cudaStream_t s) {
    const void* px = nullptr;
    const bool fresh = h->s1_fresh;
    h->s1_fresh = false;
    int bounds[3];
    const int nb = (fresh && pixels_on_host) ? s1_split_bounds(h, n, bounds) : 0;
    if (nb > 0) {
        int slot = -1;
        TSSP_TRY(stage_batch(h, pixels, nullptr, n, 1, &px, nullptr, s, bounds, nb, &slot));
        const size_t img_bytes = static_cast<size_t>(h->cfg.channels) * h->cfg.image_size * h->cfg.image_size * pixel_bytes(h);
        int begin = 0;
        for (int i = 0; i <= nb; ++i) {
            const int end = i < nb ? bounds[i] : n;
            if (i > 0) TSSP_CUDA(cudaStreamWaitEvent(s, i < nb ? h->ev_part[i] : h->ev_copied[slot], 0));
            h->staged_slot = (i == nb) ? slot : -1;  // the staging buffer is released by the last sub-batch
            TSSP_TRY(s1_sweep(h, static_cast<const char*>(px) + img_bytes * begin, end - begin,
                              img_norms != nullptr ? img_norms + static_cast<size_t>(begin) * h->sumF : nullptr, s));
            begin = end;
        }
        return 0;
    }
    TSSP_TRY(stage_batch(h, pixels, nullptr, n, pixels_on_host, &px, nullptr, s));
    return s1_sweep(h, px, n, img_norms, s);
}

int tssp_s1_batch(tssp_handle_t h, const float* pixels, int n, int pixels_on_host, float* img_norms, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_s1_batch");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return finish_host_batch(h, s, false, s1_batch(h, pixels, n, pixels_on_host, img_norms, s));
}

int tssp_s1_scores(tssp_handle_t h, float* scores, int out_on_host, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_s1_scores");
    if (scores == nullptr) return fail("tssp_s1_scores: NULL argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const cudaMemcpyKind kind = out_on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    if (h->sumF == h->ldn) {  // no block is narrower than its allocation (unpruned widths, multiples of 8): one copy
        TSSP_CUDA(cudaMemcpyAsync(scores, h->scores, sizeof(float) * h->ldn, kind, s));
    } else {
        int dst = 0;
        for (int b = 0; b < h->cfg.n_blocks; ++b) {
            const BlockWeights& w = h->blk[b];
            TSSP_CUDA(cudaMemcpyAsync(scores + dst, h->scores + w.score_off, sizeof(float) * w.F, kind, s));
            dst += w.F;
        }
    }
    if (out_on_host) TSSP_CUDA(cudaStreamSynchronize(s));
    return 0;
}

static int forward_logits(tssp_engine* h, const float* pixels, int n, int pixels_on_host, const int32_t* skip_attn,
                          float* logits, int out_on_host, cudaStream_t s) {
    const void* px = nullptr;
    TSSP_TRY(stage_batch(h, pixels, nullptr, n, pixels_on_host, &px, nullptr, s));
    TSSP_TRY(run_im2col(h, px, n, s));
    const GraphKey key{GK_FORWARD, n, 0, block_mask(skip_attn, h->cfg.n_blocks), nullptr, nullptr};
    TSSP_TRY(run_graphed(h, key, s, [&](cudaStream_t gs) -> int { return run_forward(h, n, skip_attn, false, gs); }));
    const int C = h->cfg.n_classes;
    TSSP_CUDA(cudaMemcpy2DAsync(logits, sizeof(float) * C, h->logits, sizeof(float) * h->Cp, sizeof(float) * C, n,
                                out_on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s));
    if (out_on_host) TSSP_CUDA(cudaStreamSynchronize(s));
    return 0;
}

int tssp_forward_logits(tssp_handle_t h, const float* pixels, int n, int pixels_on_host, const int32_t* skip_attn,
                        float* logits, int out_on_host, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_forward_logits");
    if (h->cfg.n_classes <= 0) return fail("tssp_forward_logits: model has no classification head: logits unavailable");
    if (logits == nullptr) return fail("tssp_forward_logits: NULL argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return finish_host_batch(h, s, false, forward_logits(h, pixels, n, pixels_on_host, skip_attn, logits, out_on_host, s));
}

static int eval_batch(tssp_engine* h, const float* pixels, const int64_t* labels, int n, int on_host, const int32_t* skip_attn,
                      unsigned long long* correct_dev, cudaStream_t s) {
    const void* px = nullptr;
    const long long* lb = nullptr;
    TSSP_TRY(stage_batch(h, pixels, labels, n, on_host, &px, &lb, s));
    TSSP_TRY(run_im2col(h, px, n, s));
    const GraphKey key{GK_EVAL, n, 0, block_mask(skip_attn, h->cfg.n_blocks), lb, correct_dev};
    return run_graphed(h, key, s, [&](cudaStream_t gs) -> int {
        TSSP_TRY(run_forward(h, n, skip_attn, false, gs));
        return op_argmax(h->logits, h->Cp, n, h->cfg.n_classes, lb, h->preds, correct_dev, gs);
    });
}

int tssp_eval_batch(tssp_handle_t h, const float* pixels, const int64_t* labels, int n, int on_host,
                    const int32_t* skip_attn, unsigned long long* correct_dev, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_eval_batch");
    if (correct_dev == nullptr) return fail("tssp_eval_batch: NULL argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return finish_host_batch(h, s, true, eval_batch(h, pixels, labels, n, on_host, skip_attn, correct_dev, s));
}

int tssp_s2_reset(tssp_handle_t h, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_s2_reset");
    TSSP_CUDA(cudaMemsetAsync(h->counts, 0, sizeof(unsigned long long) * (h->cfg.n_blocks + 1), static_cast<cudaStream_t>(stream)));
    return 0;
}

static int s2_batch(tssp_engine* h, const float* pixels, const int64_t* labels, int n, int on_host, const int32_t* cand_mask,
                    int run_baseline, cudaStream_t s) {
    if (!h->cfg.cache_blocks) return fail("tssp_s2_batch: engine was created without cache_blocks");
    const int B = h->cfg.n_blocks;
    const void* px = nullptr;
    const long long* lb = nullptr;
    TSSP_TRY(stage_batch(h, pixels, labels, n, on_host, &px, &lb, s));
    TSSP_TRY(run_im2col(h, px, n, s));
    const int C = h->cfg.n_classes;
    const size_t xbytes = static_cast<size_t>(n) * h->T * h->cfg.hidden * sizeof(float);
    // baseline pass: caches the activations entering every block; with TSSP_S2_WITH_SCORES its fc1 launches use the
    // scoring epilogue and the Stage-1 sums of this batch are accumulated as tssp_s1_batch would (the two passes of
    // Auto2SSPInterface.fit() over the same images become one)
    const bool scored = (run_baseline & TSSP_S2_WITH_SCORES) != 0;
    if (scored) h->s1_fresh = false;
    const unsigned long long cands = cand_mask != nullptr ? block_mask(cand_mask, B) : ~0ull;
    const GraphKey key{GK_S2, n, (run_baseline & 3) | (h->cfg.score_point << 2), cands, lb, nullptr};
    // the baseline and all candidates of the batch are ONE captured chain (about 700 launches for 12 blocks)
    return run_graphed(h, key, s, [&](cudaStream_t gs) -> int {
        TSSP_TRY(run_forward(h, n, nullptr, true, gs, scored ? FC1_SCORE : FC1_PLAIN));
        if (scored) TSSP_TRY(finish_scores(h, n, gs));
        if (run_baseline & TSSP_S2_COUNT_BASELINE) TSSP_TRY(op_argmax(h->logits, h->Cp, n, C, lb, h->preds, h->counts, gs));
        // candidate i: restart from the cached input of block i, drop its attention, recompute blocks i..B-1
        for (int i = 0; i < B; ++i) {
            if (((cands >> i) & 1ull) == 0) continue;
            TSSP_CUDA(cudaMemcpyAsync(h->x, h->x_cache[i], xbytes, cudaMemcpyDeviceToDevice, gs));
            for (int b = i; b < B; ++b) TSSP_TRY(run_block(h, b, n, b == i, FC1_PLAIN, true, gs, /*cls_only=*/b + 1 == B));
            TSSP_TRY(run_head(h, n, gs));
            TSSP_TRY(op_argmax(h->logits, h->Cp, n, C, lb, h->preds, h->counts + 1 + i, gs));
        }
        return 0;
    });
}

int tssp_s2_batch(tssp_handle_t h, const float* pixels, const int64_t* labels, int n, int on_host,
                  const int32_t* cand_mask, int run_baseline, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_s2_batch");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    return finish_host_batch(h, s, true, s2_batch(h, pixels, labels, n, on_host, cand_mask, run_baseline, s));
}

int tssp_s2_counts(tssp_handle_t h, int64_t* counts_host, void* stream) {
    TSSP_ENGINE_ENTRY(h, "tssp_s2_counts");
    if (counts_host == nullptr) return fail("tssp_s2_counts: NULL argument");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    TSSP_CUDA(cudaMemcpyAsync(counts_host, h->counts, sizeof(int64_t) * (h->cfg.n_blocks + 1), cudaMemcpyDeviceToHost, s));
    TSSP_CUDA(cudaStreamSynchronize(s));
    return 0;
}

// all blocks in chunks of GB_MAX_BLOCKS, one launch each (csrc/gather.cuh)
static int gather_batch(int n_blocks, const float* const* fc1_w, const float* const* fc1_b, const float* const* fc2_w,
                        const int* F, int D, const int64_t* const* keep, const int* k, float* const* fc1_w_out,
                        float* const* fc1_b_out, float* const* fc2_w_out, cudaStream_t s) {
    if (D < 4 || (D & 3)) return fail("tssp_ffn_gather: D=%d must be a positive multiple of 4", D);
    for (int b0 = 0; b0 < n_blocks; b0 += GB_MAX_BLOCKS) {
        const int nb = n_blocks - b0 < GB_MAX_BLOCKS ? n_blocks - b0 : GB_MAX_BLOCKS;
        GatherBatch g;
        memset(&g, 0, sizeof(g));
        int max_F = 0, max_k = 0, a_items = 0;
        for (int i = 0; i < nb; ++i) {
            const int b = b0 + i;
            if (fc1_w[b] == nullptr || fc2_w[b] == nullptr || keep[b] == nullptr || fc1_w_out[b] == nullptr || fc2_w_out[b] == nullptr)
                return fail("tssp_ffn_gather: NULL argument (block %d)", b);
            if (k[b] < 1 || k[b] > F[b]) return fail("tssp_ffn_gather: block %d: k=%d F=%d D=%d", b, k[b], F[b], D);
            if ((reinterpret_cast<size_t>(fc1_w[b]) | reinterpret_cast<size_t>(fc1_w_out[b])) & 15)
                return fail("tssp_ffn_gather: block %d: fc1 weights must be 16-byte aligned", b);
            g.w1[i] = fc1_w[b]; g.w2[i] = fc2_w[b]; g.keep[i] = reinterpret_cast<const long long*>(keep[b]);
            g.b1[i] = fc1_b != nullptr ? fc1_b[b] : nullptr;
            g.w1o[i] = fc1_w_out[b]; g.w2o[i] = fc2_w_out[b];
            g.b1o[i] = fc1_b_out != nullptr ? fc1_b_out[b] : nullptr;
            g.F[i] = F[b]; g.k[i] = k[b];
            a_items += ceil_div(k[b], GB_ROWS_PER_ITEM) + 1;
            g.a_end[i] = a_items;
            if (F[b] > max_F) max_F = F[b];
            if (k[b] > max_k) max_k = k[b];
        }
        g.n_blocks = nb; g.D = D;
        int rows_b = (32 * 1024) / (max_F * 4);  // about 32 KB per staging buffer
        rows_b = rows_b < 1 ? 1 : (rows_b > 8 ? 8 : rows_b);
        g.rows_b = rows_b;
        g.stage_f = round_up(rows_b * max_F, 4);
        g.keep_cap = max_k;
        const size_t smem = 128 + static_cast<size_t>(round_up(max_k * 4, 128)) + 2 * static_cast<size_t>(g.stage_f) * 4;
        if (smem > 227 * 1024) return fail("tssp_ffn_gather: F=%d too wide for the shared-memory row stage", max_F);
        TSSP_TRY(ensure_smem(ffn_gather_batch_kernel, static_cast<int>(smem)));
        int per_sm = 0;
        TSSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ffn_gather_batch_kernel, GB_THREADS, smem));
        if (per_sm < 1) per_sm = 1;
        const int b_items = nb * ceil_div(D, rows_b);
        const int most = a_items > b_items ? a_items : b_items;
        const int cap = num_sms() * per_sm;  // persistent: every CTA resident, a whole number of CTAs per SM
        ffn_gather_batch_kernel<<<most < cap ? most : cap, GB_THREADS, smem, s>>>(g);
        TSSP_LAUNCH_CHECK("ffn_gather_batch_kernel");
    }
    return 0;
}

int tssp_ffn_gather(const float* fc1_w, const float* fc1_b, const float* fc2_w, int F, int D, const int64_t* keep,
                    int k, float* fc1_w_out, float* fc1_b_out, float* fc2_w_out, void* stream) {
    TSSP_ENTRY();
    if (fc1_w == nullptr || fc2_w == nullptr || keep == nullptr || fc1_w_out == nullptr || fc2_w_out == nullptr)
        return fail("tssp_ffn_gather: NULL argument");
    const bool bias = fc1_b != nullptr && fc1_b_out != nullptr;
    return gather_batch(1, &fc1_w, bias ? &fc1_b : nullptr, &fc2_w, &F, D, &keep, &k, &fc1_w_out, bias ? &fc1_b_out : nullptr,
                        &fc2_w_out, static_cast<cudaStream_t>(stream));
}

int tssp_ffn_gather_batch(int n_blocks, const float* const* fc1_w, const float* const* fc1_b, const float* const* fc2_w,
                          const int32_t* F, int D, const int64_t* const* keep, const int32_t* k, float* const* fc1_w_out,
                          float* const* fc1_b_out, float* const* fc2_w_out, void* stream) {
    TSSP_ENTRY();
    if (n_blocks < 1 || fc1_w == nullptr || fc2_w == nullptr || F == nullptr || keep == nullptr || k == nullptr ||
        fc1_w_out == nullptr || fc2_w_out == nullptr)
        return fail("tssp_ffn_gather_batch: NULL argument or n_blocks=%d", n_blocks);
    return gather_batch(n_blocks, fc1_w, fc1_b, fc2_w, F, D, keep, k, fc1_w_out, fc1_b_out, fc2_w_out, static_cast<cudaStream_t>(stream));
}

int tssp_op_gemm(int mode, const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K,
                 const float* bias, float* partials, int ldp, int tokens_per_image, int reduce_add, void* stream) {
    TSSP_ENTRY();
    if (A == nullptr || W == nullptr || C == nullptr) return fail("tssp_op_gemm: NULL argument");
    return gemm(mode, A, lda, W, ldw, C, ldc, M, N, K, bias, partials, ldp, tokens_per_image, reduce_add, static_cast<cudaStream_t>(stream));
}
int tssp_op_gemm_scaled(const void* A, int lda, const void* W, int ldw, float* C, int ldc, int M, int N, int K, const float* bias,
                        const float* col_scale, int reduce_add, void* stream) {
    TSSP_ENTRY();
    if (A == nullptr || W == nullptr || C == nullptr || col_scale == nullptr) return fail("tssp_op_gemm_scaled: NULL argument");
    return gemm(EPI_F32_SCALED, A, lda, W, ldw, C, ldc, M, N, K, bias, nullptr, 0, 0, reduce_add, static_cast<cudaStream_t>(stream),
                nullptr, 0, 0, col_scale);
}
int tssp_op_gemm_rownorm(const void* A, int lda, const void* W, int ldw, void* C, int ldc, int M, int N, int K, const float* bias,
                         float* rownorm, int ld_rownorm, int rownorm_chunks, void* stream) {
    TSSP_ENTRY();
    if (A == nullptr || W == nullptr || C == nullptr || rownorm == nullptr) return fail("tssp_op_gemm_rownorm: NULL argument");
    if (rownorm_chunks < 0 || rownorm_chunks > ld_rownorm || rownorm_chunks * 64 > N)
        return fail("tssp_op_gemm_rownorm: %d chunks of 64 columns with ld_rownorm=%d and N=%d", rownorm_chunks, ld_rownorm, N);
    return gemm(EPI_BF16_ROWNORM, A, lda, W, ldw, C, ldc, M, N, K, bias, nullptr, 0, 0, 0, static_cast<cudaStream_t>(stream), rownorm,
                ld_rownorm, rownorm_chunks);
}
int tssp_op_score_finish(const float* partials, int ldp, float* norms, int ldn, int n_img, int T, int F, float* scores, void* stream) {
    TSSP_ENTRY();
    if (partials == nullptr || norms == nullptr) return fail("tssp_op_score_finish: NULL argument");
    return op_score_finish(partials, ldp, norms, ldn, n_img, T, F, scores, static_cast<cudaStream_t>(stream));
}
int tssp_op_layernorm(const float* x, int64_t in_stride, const float* gamma, const float* beta, void* out_bf16, int rows, int D, float eps, void* stream) {
    TSSP_ENTRY();
    if (x == nullptr || gamma == nullptr || beta == nullptr || out_bf16 == nullptr) return fail("tssp_op_layernorm: NULL argument");
    return op_layernorm(x, in_stride, gamma, beta, out_bf16, rows, D, eps, static_cast<cudaStream_t>(stream));
}
int tssp_op_layernorm_f32(const float* x, int64_t in_stride, const float* gamma, const float* beta, float* out_f32, int64_t out_stride,
                          int rows, int D, float eps, void* stream) {
    TSSP_ENTRY();
    if (x == nullptr || gamma == nullptr || beta == nullptr || out_f32 == nullptr) return fail("tssp_op_layernorm_f32: NULL argument");
    return op_layernorm_f32(x, in_stride, gamma, beta, out_f32, out_stride, rows, D, eps, static_cast<cudaStream_t>(stream));
}
int tssp_op_attention(const void* qkv_bf16, void* ctx_bf16, int n_img, int T, int heads, int D, const float* qk_norms,
                      int ld_norms, int first_tile_only, void* stream) {
    TSSP_ENTRY();
    if (qkv_bf16 == nullptr || ctx_bf16 == nullptr) return fail("tssp_op_attention: NULL argument");
    if (qk_norms != nullptr && ld_norms < 2 * heads)
        return fail("tssp_op_attention: ld_norms=%d is less than 2*heads=%d (|q|^2 and |k|^2 columns of every head)", ld_norms, 2 * heads);
    return op_attention(qkv_bf16, ctx_bf16, n_img, T, heads, D, static_cast<cudaStream_t>(stream), qk_norms, ld_norms,
                        first_tile_only != 0);
}
int tssp_debug_gemm_trace(long long* device_buf) {
    TSSP_ENTRY();
    g_gemm_trace = device_buf;  // >= 24 * 16 int64; nullptr disables
    ++g_launch_epoch;
    return 0;
}
int tssp_debug_attention_trace(long long* device_buf) {
    TSSP_ENTRY();
    g_attn_trace = device_buf;  // >= 256 int64; nullptr disables
    ++g_launch_epoch;
    return 0;
}
int tssp_op_im2col(const void* pixels, void* out_bf16, int n_img, int C, int H, int W, int P, int prefix_tokens,
                   const tssp_pixel_input_t* input, void* stream) {
    TSSP_ENTRY();
    if (pixels == nullptr || out_bf16 == nullptr) return fail("tssp_op_im2col: NULL argument");
    return op_im2col(pixels, out_bf16, n_img, C, H, W, P, prefix_tokens, input, static_cast<cudaStream_t>(stream));
}
int tssp_op_cast_bf16(const float* in, int rows, int cols, int ld_in, void* out_bf16, int rows_pad, int cols_pad, int ld_out, void* stream) {
    TSSP_ENTRY();
    if (in == nullptr || out_bf16 == nullptr) return fail("tssp_op_cast_bf16: NULL argument");
    return op_cast(in, rows, cols, ld_in, out_bf16, rows_pad, cols_pad, ld_out, static_cast<cudaStream_t>(stream));
}
int tssp_op_argmax_count(const float* logits, int ld, int n, int C, const int64_t* labels, int32_t* preds, unsigned long long* correct_dev, void* stream) {
    TSSP_ENTRY();
    if (logits == nullptr) return fail("tssp_op_argmax_count: NULL argument");
    return op_argmax(logits, ld, n, C, reinterpret_cast<const long long*>(labels), preds, correct_dev, static_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------- score file text (host only)
// repr(float(v)) of CPython for a finite double: the shortest digit string that round-trips (std::to_chars gives exactly
// that), laid out by CPython's rule (pystrtod.c, format code 'r'): scientific iff the decimal exponent is < -4 or >= 16,
// exponent with at least two digits, ".0" appended to integral fixed values. json.dumps writes NaN / Infinity / -Infinity.
static char* py_float_repr(char* out, double v) {
    if (std::isnan(v)) { memcpy(out, "NaN", 3); return out + 3; }
    if (std::isinf(v)) {
        if (v < 0) *out++ = '-';
        memcpy(out, "Infinity", 8);
        return out + 8;
    }
    char buf[40];
    const auto res = std::to_chars(buf, buf + sizeof(buf), v, std::chars_format::scientific);
    const char* p = buf;
    if (*p == '-') { *out++ = '-'; ++p; }
    char digits[24];
    int nd = 0;
    for (; p < res.ptr && *p != 'e'; ++p)
        if (*p != '.') digits[nd++] = *p;
    int e = 0;
    if (p < res.ptr) {  // "e+XX" / "e-XX"
        ++p;
        const bool neg = (*p == '-');
        ++p;
        for (; p < res.ptr; ++p) e = e * 10 + (*p - '0');
        if (neg) e = -e;
    }
    if (e < -4 || e >= 16) {
        *out++ = digits[0];
        if (nd > 1) {
            *out++ = '.';
            memcpy(out, digits + 1, nd - 1);
            out += nd - 1;
        }
        *out++ = 'e';
        *out++ = e < 0 ? '-' : '+';
        int a = e < 0 ? -e : e;
        char eb[8];
        int ne = 0;
        do { eb[ne++] = static_cast<char>('0' + a % 10); a /= 10; } while (a > 0);
        if (ne < 2) eb[ne++] = '0';
        while (ne > 0) *out++ = eb[--ne];
        return out;
    }
    if (e >= 0) {
        const int int_digits = e + 1;
        for (int i = 0; i < int_digits; ++i) *out++ = i < nd ? digits[i] : '0';
        *out++ = '.';
        if (nd > int_digits) {
            memcpy(out, digits + int_digits, nd - int_digits);
            out += nd - int_digits;
        } else {
            *out++ = '0';
        }
        return out;
    }
    *out++ = '0';
    *out++ = '.';
    for (int i = 0; i < -e - 1; ++i) *out++ = '0';
    memcpy(out, digits, nd);
    return out + nd;
}

static char* put_uint(char* out, unsigned v) {
    char b[12];
    int n = 0;
    do { b[n++] = static_cast<char>('0' + v % 10); v /= 10; } while (v > 0);
    while (n > 0) *out++ = b[--n];
    return out;
}

extern "C" long long tssp_format_ffn_scores(const float* scores, const int32_t* widths, int n_blocks, char* out, long long cap) {
    TSSP_ENTRY();
    if (widths == nullptr || n_blocks < 0 || (scores == nullptr && n_blocks > 0)) { fail("tssp_format_ffn_scores: NULL argument"); return -1; }
    long long total = 0;
    for (int b = 0; b < n_blocks; ++b) {
        if (widths[b] < 0) { fail("tssp_format_ffn_scores: negative width"); return -1; }
        total += widths[b];
    }
    const long long need = 64 * total + 64;   // "    \"bb:jjjjj\": " (<= 22) + repr (<= 25) + ",\n"
    if (out == nullptr || cap < need) return need;
    char* p = out;
    if (total == 0) {
        static const char empty[] = "{\n  \"ffn\": {}\n}";
        memcpy(p, empty, sizeof(empty) - 1);
        return static_cast<long long>(sizeof(empty) - 1);
    }
    static const char head[] = "{\n  \"ffn\": {\n";
    memcpy(p, head, sizeof(head) - 1);
    p += sizeof(head) - 1;
    const float* v = scores;
    bool first = true;
    for (int b = 0; b < n_blocks; ++b) {
        for (int j = 0; j < widths[b]; ++j, ++v) {
            if (!first) { *p++ = ','; *p++ = '\n'; }
            first = false;
            memcpy(p, "    \"", 5);
            p += 5;
            p = put_uint(p, static_cast<unsigned>(b));
            *p++ = ':';
            p = put_uint(p, static_cast<unsigned>(j));
            *p++ = '"'; *p++ = ':'; *p++ = ' ';
            p = py_float_repr(p, static_cast<double>(*v));   // float(v) of the reference: the exact double of the fp32 score
        }
    }
    static const char tail[] = "\n  }\n}";
    memcpy(p, tail, sizeof(tail) - 1);
    p += sizeof(tail) - 1;
    return static_cast<long long>(p - out);
}

// ---------------------------------------------------------------- mask builders (manual-experiments scripts)
static int mask_args_ok(const char* fn, const void* a, const void* b, int n_files, int n_blocks, int ld, int max_width) {
    if (a == nullptr || b == nullptr) return fail("%s: NULL argument", fn);
    if (n_files <= 0 || n_blocks <= 0 || ld <= 0) return fail("%s: n_files=%d n_blocks=%d ld=%d must be positive", fn, n_files, n_blocks, ld);
    if (max_width <= 0 || max_width > ld) return fail("%s: max_width=%d must be in [1, ld=%d]", fn, max_width, ld);
    if (max_width > 6000) return fail("%s: max_width=%d exceeds the 6000-entry shared-memory row", fn, max_width);
    return 0;
}

int tssp_op_stable_rank_f64(const double* values, int rows, int cols, int ld, int32_t* ranks, void* stream) {
    TSSP_ENTRY();
    TSSP_TRY(mask_args_ok("tssp_op_stable_rank_f64", values, ranks, 1, rows, ld, cols));
    stable_rank_f64_kernel<<<dim3(ceil_div(cols, MB_THREADS), rows), MB_THREADS, cols * sizeof(double), static_cast<cudaStream_t>(stream)>>>(
        values, cols, ld, nullptr, 1, ranks);
    TSSP_LAUNCH_CHECK("stable_rank_f64_kernel");
    return 0;
}

int tssp_mask_consensus_prepare(const double* scores, int n_files, int n_blocks, const int32_t* widths, int max_width, int ld,
                                int32_t* ranks_ws, int32_t* rmax, double* sums, void* stream) {
    TSSP_ENTRY();
    TSSP_TRY(mask_args_ok("tssp_mask_consensus_prepare", scores, widths, n_files, n_blocks, ld, max_width));
    if (ranks_ws == nullptr || rmax == nullptr || sums == nullptr) return fail("tssp_mask_consensus_prepare: NULL output");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    stable_rank_f64_kernel<<<dim3(ceil_div(max_width, MB_THREADS), n_files * n_blocks), MB_THREADS, max_width * sizeof(double), s>>>(
        scores, max_width, ld, widths, n_blocks, ranks_ws);
    TSSP_LAUNCH_CHECK("stable_rank_f64_kernel");
    consensus_reduce_kernel<<<dim3(ceil_div(max_width, MB_THREADS), n_blocks), MB_THREADS, 0, s>>>(ranks_ws, scores, n_files, n_blocks, ld, widths, rmax, sums);
    TSSP_LAUNCH_CHECK("consensus_reduce_kernel");
    return 0;
}

int tssp_mask_count_less(const int32_t* rmax, int n_blocks, const int32_t* widths, int ld, const int32_t* k, int32_t* counts, void* stream) {
    TSSP_ENTRY();
    if (rmax == nullptr || widths == nullptr || k == nullptr || counts == nullptr) return fail("tssp_mask_count_less: NULL argument");
    if (n_blocks <= 0) return fail("tssp_mask_count_less: n_blocks=%d", n_blocks);
    count_less_i32_kernel<<<n_blocks, MB_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(rmax, ld, widths, k, counts);
    TSSP_LAUNCH_CHECK("count_less_i32_kernel");
    return 0;
}

int tssp_mask_consensus_select(const int32_t* rmax, const double* sums, int n_files, int n_blocks, const int32_t* widths,
                               int max_width, int ld, const int32_t* k, int k_common, uint8_t* mask, void* stream) {
    TSSP_ENTRY();
    TSSP_TRY(mask_args_ok("tssp_mask_consensus_select", rmax, sums, n_files, n_blocks, ld, max_width));
    if (widths == nullptr || k == nullptr || mask == nullptr) return fail("tssp_mask_consensus_select: NULL argument");
    consensus_select_kernel<<<n_blocks, MB_THREADS, max_width * sizeof(double), static_cast<cudaStream_t>(stream)>>>(
        rmax, sums, n_files, ld, widths, k, k_common, mask);
    TSSP_LAUNCH_CHECK("consensus_select_kernel");
    return 0;
}

int tssp_mask_summation(const double* scores, int n_files, int n_blocks, const int32_t* widths, int max_width, int ld,
                        int k_common, double* sums, int32_t* ranks_ws, uint8_t* mask, void* stream) {
    TSSP_ENTRY();
    TSSP_TRY(mask_args_ok("tssp_mask_summation", scores, widths, n_files, n_blocks, ld, max_width));
    if (sums == nullptr || ranks_ws == nullptr || mask == nullptr) return fail("tssp_mask_summation: NULL output");
    if (k_common < 0) return fail("tssp_mask_summation: k_common=%d", k_common);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const dim3 grid(ceil_div(max_width, MB_THREADS), n_blocks);
    consensus_reduce_kernel<<<grid, MB_THREADS, 0, s>>>(nullptr, scores, n_files, n_blocks, ld, widths, nullptr, sums);
    TSSP_LAUNCH_CHECK("consensus_reduce_kernel");
    stable_rank_f64_kernel<<<grid, MB_THREADS, max_width * sizeof(double), s>>>(sums, max_width, ld, widths, n_blocks, ranks_ws);
    TSSP_LAUNCH_CHECK("stable_rank_f64_kernel");
    rank_threshold_mask_kernel<<<grid, MB_THREADS, 0, s>>>(ranks_ws, ld, widths, k_common, mask);
    TSSP_LAUNCH_CHECK("rank_threshold_mask_kernel");
    return 0;
}

int tssp_op_minmax_normalize_f64(const double* values, long long n, double* minmax, double* out, void* stream) {
    TSSP_ENTRY();
    if (values == nullptr || minmax == nullptr || out == nullptr) return fail("tssp_op_minmax_normalize_f64: NULL argument");
    if (n <= 0) return fail("tssp_op_minmax_normalize_f64: n=%lld", n);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    minmax_f64_kernel<<<1, 1024, 0, s>>>(values, n, minmax);
    TSSP_LAUNCH_CHECK("minmax_f64_kernel");
    minmax_normalize_f64_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(values, n, minmax, out);
    TSSP_LAUNCH_CHECK("minmax_normalize_f64_kernel");
    return 0;
}

}  // extern "C"
