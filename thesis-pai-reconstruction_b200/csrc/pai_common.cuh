// Shared device helpers for the sm_100a kernels: mbarrier, TMA, tcgen05 / TMEM wrappers
// (inline PTX), error plumbing for the C-ABI.  Nothing here is reference-derived; the
// reference (cristianpjensen/thesis-pai-reconstruction) ships no native code.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace pai {

// ---- host-side error channel (see pai_last_error in include/pai_b200.h)
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
#define PAI_CUDA_OK(expr)                                                   \
    do {                                                                    \
        cudaError_t _e = (expr);                                            \
        if (_e != cudaSuccess) return ::pai::cuda_fail(_e, #expr);          \
    } while (0)
#define PAI_REQUIRE(cond, ...)                                              \
    do {                                                                    \
        if (!(cond)) {                                                      \
            ::pai::set_error(__VA_ARGS__);                                  \
            return -2;                                                      \
        }                                                                   \
    } while (0)

// Per-device one-time set-up (cudaFuncSetAttribute opt-ins, constant uploads): the library may serve several GPUs of
// one process from several threads, so "done" is a bit per device ordinal, set after the (idempotent) set-up ran.
struct DeviceOnce {
    unsigned long long mask = 0;
    bool need(int dev) const { return ((__atomic_load_n(&mask, __ATOMIC_ACQUIRE) >> (dev & 63)) & 1ull) == 0; }
    void mark(int dev) { __atomic_fetch_or(&mask, 1ull << (dev & 63), __ATOMIC_RELEASE); }
};
// Current device ordinal and its SM count (cached per device); negative on a CUDA error (pai_last_error is set).
int current_device();
int sm_count(int dev);
// SMs the persistent (one CTA per SM) kernels may occupy: sm_count minus the reservation of pai_reserve_sms()
int persistent_ctas(int dev);

// ---- programmatic dependent launch (PDL).  The training step is ~200 dependent launches replayed as one CUDA graph; a
// kernel launched with `programmaticStreamSerializationAllowed` may be SCHEDULED as soon as every CTA of the previous
// kernel has executed griddepcontrol.launch_dependents (done at kernel entry), so its launch latency, CTA scheduling and
// prologue (barrier init, TMEM allocation, tensor-map prefetch) overlap the previous kernel's tail; its own
// griddepcontrol.wait then blocks until the previous grid has COMPLETED and its memory is visible.  Rule kept by every
// launch site: a kernel is launched through launch_pdl only if it executes pdl_wait() before its first dependent memory
// access (kernels with the two instructions launched the ordinary way see them as no-ops).  OPT-IN (PAI_PDL=1): on the
// graph-replayed training step it measured 0.5-1 % slower than plain serialisation (7.74 against 7.69 ms, A/B on one box) --
// the graph's kernel-to-kernel gaps are already ~1 us and early-resident CTAs compete with the running kernel's tail.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled();
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     int cluster_x, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (cluster_x > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = (unsigned)cluster_x, attr[na].val.clusterDim.y = 1, attr[na].val.clusterDim.z = 1;
        ++na;
    }
    if (pdl_enabled()) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = attr, cfg.numAttrs = (unsigned)na;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Encodes a bf16 tiled tensor map (rank <= 5, SWIZZLE_128B, zero OOB fill) through the driver
// entry point fetched at run time, so the library loads on a box without libcuda.
int encode_tmap_bf16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box);

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// One lane of a converged warp; the compiler then issues the single-thread uniform-datapath instructions (UTCHMMA,
// UTMALDG, UTCBAR) directly instead of wrapping each in an elect-and-retry loop.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n"
        ".reg .pred P;\n"
        "elect.sync _|P, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, P;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug traps (kernel error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
            printf("pai: mbarrier wait timed out (block %d,%d,%d thread %d)\n", blockIdx.x, blockIdx.y,
                   blockIdx.z, threadIdx.x);
            __trap();
        }
    }
}

// ---- TMA (cp.async.bulk.tensor), completes on an mbarrier with complete_tx::bytes
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, "
        "%7}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
// L2 prefetch of a 5-D box (no shared-memory destination, no barrier)
__device__ __forceinline__ void tma_prefetch_5d(const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4) {
    asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global.tile [%0, {%1, %2, %3, %4, %5}];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
                 : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
// TMA store of a 4-D box from shared memory (elements outside the map's extents are not written), tracked by the
// issuing thread's bulk async-groups: commit after the store, then wait_group_read before that thread (and, after a
// warp sync, its warp) writes the source buffer again, and wait_group before the CTA exits.  The shared-memory writes
// the store reads must be fenced to the async proxy first (fence_proxy_async_smem in every writing thread).
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// every committed bulk store of this thread has finished READING its shared-memory source
__device__ __forceinline__ void bulk_wait_group_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// every committed bulk store of this thread has completed (its global writes are performed)
__device__ __forceinline__ void bulk_wait_group0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> fp32, one CTA.
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Same with the accumulate flag fixed to 1 (no predicate set-up on the issuing thread).
__device__ __forceinline__ void umma_bf16_acc(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.eq.b32 p, 0, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc)
        : "memory");
}
// Arrives on `bar` once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives TMEM lane (base_lane + i).
__device__ __forceinline__ void tmem_ld_16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA pairs (cta_group::2): two CTAs of a 2-CTA cluster on the two SMs of one TPC run ONE M = 256 MMA; each CTA
// stages its own 128 A rows and HALF of the B tile, the even-ranked ("leader") CTA issues the MMAs and owns the `full`
// barriers that both CTAs' TMA loads complete on.  A shared-memory address of the executing CTA with bit 24 cleared is
// the same offset in the leader CTA (the convention CUTLASS ships as Sm100MmaPeerBitMask).
static constexpr uint32_t kPairLeaderMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint64_t* leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(leader_bar) & kPairLeaderMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(void* dst, const CUtensorMap* map, uint64_t* leader_bar, int c0, int c1,
                                                 int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
        "%5, %6, %7}], [%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(leader_bar) & kPairLeaderMask), "r"(c0), "r"(c1), "r"(c2),
        "r"(c3), "r"(c4)
        : "memory");
}
// arrive (count 1) on the LEADER CTA's copy of `bar`, from either CTA of the pair
// Relaxed arrivals for the accumulator hand-off: the TMEM reads being released are ordered by tcgen05.wait::ld +
// tcgen05.fence::before_thread_sync, so the arrival need not wait for the epilogue's outstanding global stores and
// reductions the way the default .release form does (measured: +10 .. +50 us per layer with the release form).
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader_relaxed(uint64_t* bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPairLeaderMask)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPairLeaderMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {  // one warp of EACH CTA
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {    // one warp of EACH CTA
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[256 rows: 128 per CTA] * B[N columns: N/2 rows per CTA]; issued by the leader CTA only
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_acc_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.eq.b32 p, 0, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc)
        : "memory");
}
// arrives on the barrier at `bar`'s offset in BOTH CTAs once every previously issued pair MMA has completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
}

// ---- lean forms for the MMA-issuing warp (igemm fprop).  Measured with -DPAI_PROFILE_ROLES: the issuing thread spent
// ~290 cycles per pipeline stage outside the MMAs (64-bit descriptor arithmetic, generic->shared conversions, register ->
// uniform-register moves), more than the 256 cycles of tensor work of an N = 128 stage.  Here barriers are addressed by
// their 32-bit shared address and descriptors by their LOW word only: the high word of every K-major SWIZZLE_128B
// descriptor is the constant kDescHiSw128 (SBO 1024 B, version 1, SWIZZLE_128B), and stepping K by 16 elements or moving
// to another tile never carries out of the 14-bit address field of the low word.
static constexpr uint32_t kDescHiSw128 = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t umma_desc_lo_kmajor(uint32_t saddr) { return ((saddr & 0x3FFFF) >> 4) | (1u << 16); }

__device__ __forceinline__ bool mbar_try_wait_u32(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait_u32(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait_u32(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("pai: mbarrier wait timed out (block %d,%d,%d thread %d)\n", blockIdx.x, blockIdx.y, blockIdx.z,
                   threadIdx.x);
            __trap();
        }
    }
}
// KSTEPS MMAs over one 64-wide K block (16 elements = 2 descriptor units per step); `accumulate` applies to the first.
template <bool PAIR, int KSTEPS>
__device__ __forceinline__ void umma_kblock_lo(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                                               uint32_t accumulate) {
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) {
        if (PAIR)
            asm volatile(
                "{\n"
                ".reg .pred p;\n"
                ".reg .b64 da, db;\n"
                "setp.ne.b32 p, %4, 0;\n"
                "mov.b64 da, {%1, %5};\n"
                "mov.b64 db, {%2, %5};\n"
                "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n"
                "}\n" ::"r"(tmem_d),
                "r"(a_lo + 2 * k), "r"(b_lo + 2 * k), "r"(idesc), "r"(k == 0 ? accumulate : 1u), "r"(kDescHiSw128)
                : "memory");
        else
            asm volatile(
                "{\n"
                ".reg .pred p;\n"
                ".reg .b64 da, db;\n"
                "setp.ne.b32 p, %4, 0;\n"
                "mov.b64 da, {%1, %5};\n"
                "mov.b64 db, {%2, %5};\n"
                "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n"
                "}\n" ::"r"(tmem_d),
                "r"(a_lo + 2 * k), "r"(b_lo + 2 * k), "r"(idesc), "r"(k == 0 ? accumulate : 1u), "r"(kDescHiSw128)
                : "memory");
    }
}
template <bool PAIR>
__device__ __forceinline__ void umma_commit_u32(uint32_t bar) {
    if (PAIR)
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
            "h"((uint16_t)3)
            : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// Shared-memory matrix descriptors for SWIZZLE_128B tiles whose rows are 128 B (64 bf16) wide and
// whose 8-row groups are 1024 B apart (exactly what a TMA box with a 64-element inner dimension
// writes).  K-major: rows are M/N, the 128 B row holds 64 K-values.  MN-major: rows are K, the
// 128 B row holds 64 M/N values and `mn_block_bytes` is the distance to the next 64-wide block.
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t saddr, uint32_t mn_block_bytes) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)((mn_block_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// Instruction descriptor, kind::f16: bf16 A/B, fp32 accumulate, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif  // __CUDACC__

}  // namespace pai
