// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM).
// Everything here is device-only and header-only; no CUTLASS/CuTe dependency.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace tssp {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() {
    uint32_t l;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
    return l;
}

// One lane of the (fully active) warp. Unlike `lane == 0`, the compiler KNOWS that exactly one thread runs the guarded
// region, so values that feed uniform-register operands (UTCHMMA / UTMALDG descriptors, barrier addresses) move there
// with a plain R2UR instead of an ELECT + R2UR.BROADCAST + BRA.U.ANY waterfall loop per instruction: the MMA issue loop
// of the GEMM shrank from 21 to 9 instructions per tcgen05.mma (it could not keep the tensor pipe fed next to busy
// epilogue warps: tools/gemm_trace.py, profiles/gemm_trace_r2.txt).
__device__ __forceinline__ bool elect_one_sync() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// try_wait suspends the thread in hardware until the phase completes or the time hint (ns) expires, so a waiting
// role warp does not burn issue slots of the sub-partition it shares with an epilogue warp.
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(1000000u)
        : "memory");
    return ok != 0;
}
// Bounded spin: a protocol bug traps (-> launch failure the host reports) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (!mbar_try_wait(bar, parity)) {
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > 10000000000ull) __trap();  // 10 s: a protocol bug, not a slow kernel
    }
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tensormap(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tile load global -> shared, completion signalled on an mbarrier (bytes).
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* tmap, uint32_t bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
// The same load with an L2 cache policy (evict-first for operands that are streamed once: they should not push the
// tensors the NEXT kernel starts on out of L2).
__device__ __forceinline__ void tma_load_2d_hint(uint32_t smem_dst, const void* tmap, uint32_t bar, int32_t c0, int32_t c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
// 2-D tile store shared -> global (bulk async group).
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 :
                 : "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1)
                 : "memory");
}
// Same store with an L2 evict-first policy: for outputs that are far larger than L2 and are streamed once by their
// consumer (the fc1 activation h), so they do not push the residual stream and the next operands out of L2.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void tma_store_2d_hint(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1, uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;"
                 :
                 : "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1), "l"(policy)
                 : "memory");
}
// 2-D tile reduce-add shared -> global: element-wise global += tile, done by the TMA unit at L2.
__device__ __forceinline__ void tma_reduce_add_2d(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
                 :
                 : "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the smem source of all but N most recent groups has been read
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// make generic-proxy smem writes visible to the async proxy (TMA store source)
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------- packed fp32 pairs (sm_100 FFMA2 / FADD2)
// One instruction, two IEEE fp32 operations (same rounding as the scalar forms): it occupies the FMA pipe for two
// cycles but a single issue slot, which is what the GEMM epilogues are short of (tools/ffma2_probe.cu).
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// ---------------------------------------------------------------- CTA pair (cluster of 2, tcgen05 cta_group::2)
// Both CTAs of a pair run the same code with the same shared-memory layout; in the shared::cluster window bit 24 of an
// address selects the odd CTA, so `addr & PEER_BIT_MASK` names the even (leader) CTA's copy of a local object.
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same offset in CTA `cta` of the cluster (works for the own CTA too). Default (CTA-scope)
// release: the barriers signalled this way hand over TMEM buffers, which the tcgen05 fences order; a cluster-scope
// release costs a membar per arrival (12 % of the epilogue's stall samples when it was tried).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_local, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(bar_local), "r"(cta)
        : "memory");
}
// TMA load issued by either CTA of a pair: data lands in the issuer's shared memory, the bytes are counted on the
// LEADER's barrier (the one thread that issues the pair's MMAs waits there for both halves).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t smem_dst, const void* tmap, uint32_t bar_local, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_local & PEER_BIT_MASK), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_hint(uint32_t smem_dst, const void* tmap, uint32_t bar_local, int32_t c0, int32_t c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_local & PEER_BIT_MASK), "r"(c0), "r"(c1), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_result_addr, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B over the pair: 256 x N x 16, rows 0-127 of A and D in the leader, 128-255 in the
// peer, each CTA holding its own half of B's N rows. Issued by one thread of the LEADER only.
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive (once all MMAs issued so far have retired) on the barrier at this offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_pair(uint32_t bar_local, uint32_t cta_mask) {
    asm volatile(
        "{\n\t.reg .b16 lo, hi;\n\t"
        "mov.b32 {lo, hi}, %1;\n\t"
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], lo;\n\t}" ::"r"(bar_local), "r"(cta_mask)
        : "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start while its predecessor in the
// stream is still draining: its CTAs take the SMs the predecessor's CTAs leave and run their prologue (barrier init,
// TMEM allocation, descriptor prefetch). griddep_wait() blocks until the predecessor has completed and its writes
// are visible; nothing that touches activations may precede it. Both are no-ops for an ordinary launch.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- register file hand-over between warpgroups
// Executed by every warp of one warpgroup (4 consecutive warps). The register file is allocated per thread at launch
// (launch-bounds count for all 12 warps); producer / issuer warpgroups give most of theirs back and the math
// warpgroups take them, so the compiler can keep TMEM prefetch buffers live next to the working set.
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 operands, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread t = TMEM lane base+t).
// The load and its wait::ld sit in ONE asm statement so the compiler cannot schedule a use of the
// destination registers between them (the registers are undefined until the wait retires).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Split form for software pipelining: issue the load, do other work, then tmem_ld_fence(r) before touching r.
// The fence lists r as read-write operands so no use of r can be scheduled above it.
__device__ __forceinline__ void tmem_ld_32x32b_x32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_fence(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                   "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                   "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
}

// 16-column variant of the split form: fills r[0..15] of a 32-register buffer (fence it with tmem_ld_fence as usual)
__device__ __forceinline__ void tmem_ld_32x32b_x16_nowait(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

// registers -> TMEM: this warp's 32 lanes x 16 (or 8) consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        :
        : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :
                 : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem desc]: A (bf16, K-major, two elements per 32-bit column) read from tensor memory.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// 3-D tile load global -> shared (coordinates innermost first)
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const void* tmap, uint32_t bar, int32_t c0, int32_t c1, int32_t c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

__device__ __forceinline__ void tma_load_3d_hint(uint32_t smem_dst, const void* tmap, uint32_t bar, int32_t c0, int32_t c1, int32_t c2, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        :
        : "r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
        : "memory");
}
// 128-bit global load that bypasses L1 and carries an L2 cache policy
__device__ __forceinline__ float4 ld_global_v4_hint(const float4* p, uint64_t policy) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p), "l"(policy));
    return v;
}
__device__ __forceinline__ float2 ld_global_v2_hint(const float2* p, uint64_t policy) {
    float2 v;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v2.f32 {%0, %1}, [%2], %3;" : "=f"(v.x), "=f"(v.y) : "l"(p), "l"(policy));
    return v;
}

// 3-D tile store shared -> global (bulk async group); elements outside the tensor are not written
__device__ __forceinline__ void tma_store_3d(const void* tmap, uint32_t smem_src, int32_t c0, int32_t c1, int32_t c2) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                 :
                 : "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}

// Shared-memory descriptor for an MN-major bf16 operand (rows = K index, 64 MN elements = 128 B contiguous per row,
// written by TMA with SWIZZLE_128B): 8-row (K) groups are 1024 B apart (SBO); LBO = distance to the next 64-wide MN panel.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Shared-memory matrix descriptor for a K-major bf16 operand tile written by TMA with SWIZZLE_128B:
// rows are 128 B (64 bf16) apart, 8-row groups are 1024 B apart (SBO), LBO unused for swizzled K-major.
// Field layout follows the sm_100 UMMA descriptor (start>>4 [0,14), LBO>>4 [16,30), SBO>>4 [32,46),
// version=1 [46,48), layout type [61,64) with SWIZZLE_128B = 2).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;              // LBO (ignored for SW128 K-major), canonical value 1
    d |= static_cast<uint64_t>(1024 >> 4) << 32;      // SBO = 1024 B
    d |= static_cast<uint64_t>(1) << 46;              // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;              // SWIZZLE_128B
    return d;
}

// Instruction descriptor for kind::f16, A=B=bf16 (K-major both), D=fp32, shape M x N (K=16 implied).
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(int M, int N) {
    return (1u << 4)                               // c_format = F32
           | (1u << 7)                             // a_format = BF16
           | (1u << 10)                            // b_format = BF16
           | (static_cast<uint32_t>(N >> 3) << 17) // n_dim
           | (static_cast<uint32_t>(M >> 4) << 24);// m_dim
}

// ---------------------------------------------------------------- misc
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t ld_shared_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}

}  // namespace ptx
}  // namespace tssp
