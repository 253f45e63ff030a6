// svb_common.cuh -- shared host/device helpers for libspine_b200 (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/spine_b200.h"

namespace svb {

// ----------------------------------------------------------------------------- host: errors
std::string& last_error_ref();
int set_error(int code, const char* fmt, ...);

#define SVB_CUDA_OK(expr)                                                                          \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return svb::set_error(SVB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                    \
                                  cudaGetErrorString(_e), __FILE__, __LINE__);                     \
    } while (0)

#define SVB_REQUIRE(cond, code, ...)                                                               \
    do {                                                                                           \
        if (!(cond)) return svb::set_error((code), __VA_ARGS__);                                   \
    } while (0)

// every kernel launch of the library is counted (bench.py reports it as gpu_launches); a CUDA graph replay adds its kernel nodes
void count_launch(long long n = 1);
#define SVB_LAUNCHED()                          \
    do {                                        \
        svb::count_launch();                    \
        SVB_CUDA_OK(cudaGetLastError());        \
    } while (0)

int check_device_sm100();
int num_sms();

template <typename T>
static inline T ceil_div(T a, T b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ----------------------------------------------------------------------------- device: small utils
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// float32 -> uint8 exactly as NumPy's astype(uint8) behaves on x86-64: truncate to int32
// (out-of-range / NaN -> 0x80000000) and keep the low byte.
__device__ __forceinline__ uint32_t cast_f32_u8(float v) {
    if (!(v >= -2147483648.0f && v < 2147483648.0f)) return 0u;
    return static_cast<uint32_t>(__float2int_rz(v)) & 0xFFu;
}

// (x - mn) / rng * 255 in fp32 with no contraction / reciprocal (io/__init__.py:28-29)
__device__ __forceinline__ uint32_t normalize_px(float x, float mn, float rng) {
    float v = x;
    if (rng > 0.0f) v = __fmul_rn(__fdiv_rn(__fsub_rn(x, mn), rng), 255.0f);
    return cast_f32_u8(v);
}

// order-preserving float <-> uint key (for atomicMin / atomicMax on floats of any sign)
__device__ __forceinline__ uint32_t float_key(float f) {
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

template <typename T> struct Cvt;
template <> struct Cvt<__nv_bfloat16> {
    static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
    static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
    static __device__ __forceinline__ uint32_t pack2(float a, float b) {
        __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&p);
    }
    static __device__ __forceinline__ float2 unpack2(uint32_t u) {
        return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xFFFF0000u));
    }
};
template <> struct Cvt<__half> {
    static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
    static __device__ __forceinline__ __half from_f(float v) {
        return __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f));
    }
    static __device__ __forceinline__ uint32_t pack2(float a, float b) {
        // one F2FP.SATFINITE.F16.F32.PACK_AB: round to nearest even, out-of-range values saturate at +-65504
        uint32_t r;
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
        return r;
    }
    static __device__ __forceinline__ float2 unpack2(uint32_t u) {
        __half2 p = *reinterpret_cast<__half2*>(&u);
        return __half22float2(p);
    }
};

// ----------------------------------------------------------------------------- device: PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
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
// Relaxed arrive: no fence in front.  The default (.release) compiles to MEMBAR.ALL.CTA in front of SYNCS.ARRIVE, which
// waits for every outstanding memory operation of the thread (measured: ~18 % of the GEMM epilogue warps' samples sat in
// MEMBAR / ERRBAR).  Safe wherever the barrier only returns a buffer whose contents the warp has already READ into
// registers: a TMEM accumulator after tcgen05.wait::ld, a shared-memory stage whose ld.shared results have been consumed.
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must trap, not hang the GPU box (see the gpurun strike rule).
__device__ __forceinline__ uint64_t global_timer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity) {
    uint32_t done = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, 0x989680;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    return done != 0;
}
static __device__ __noinline__ void mbar_wait_slow(uint32_t addr, uint32_t parity) {
    const uint64_t t0 = global_timer_ns();
    while (!mbar_try_wait(addr, parity)) {
        if (global_timer_ns() - t0 > 4000000000ull) {  // 4 s: no healthy wait is this long
            printf("svb: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n", blockIdx.x,
                   threadIdx.x, addr, parity);
            __trap();
        }
    }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    if (mbar_try_wait(addr, parity)) return;
    mbar_wait_slow(addr, parity);
}

__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// TMA tiled loads (global -> shared), completion on an mbarrier
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// TMA tiled store (shared -> global), bulk-group completion
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {  // at most N groups still reading shared memory
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- programmatic dependent launch (PDL): a kernel launched with programmaticStreamSerialization may start while its
// predecessor in the stream is still running; it must call pdl_wait() before its first access to memory the predecessor
// reads or writes (the wait returns once the predecessor grid has completed and its writes are visible).
// pdl_launch_dependents() lets the successor's CTAs be scheduled as soon as every CTA of this grid has issued it.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---- thread-block cluster / CTA-pair helpers (cta_group::2)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// distributed shared memory: plain loads / stores at a shared::cluster address (see mapa_shared)
__device__ __forceinline__ float ld_cluster_f32(uint32_t cluster_addr) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr) : "memory");
    return v;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t cluster_addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(cluster_addr), "f"(v) : "memory");
}
// same hand-over to the pair leader's barrier without the MEMBAR.ALL.GPU + ERRBAR a cluster-scope release costs
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// CTA-pair TMA load: the data lands in THIS CTA's shared memory, the bytes are counted on the
// mbarrier at shared::cluster address `bar_cluster` (the pair leader's "full" barrier).
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1)
        : "memory");
}

__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ---- packed fp32 pairs (FFMA2 / FMUL2 / FADD2 on sm_100): half the issue slots of scalar FP32
__device__ __forceinline__ uint64_t pk2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// tcgen05 / TMEM
template <int CG = 1>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    if (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG = 1>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// CG == 1: arrive on this CTA's mbarrier when all prior MMAs retire.  CG == 2: the same offset in BOTH CTAs of the pair.
template <int CG = 1>
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    if (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
    } else {
        const uint16_t mask = 3;
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                         smem_u32(bar)),
                     "h"(mask)
                     : "memory");
    }
}
// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (bf16 or fp16 operands, fp32 accumulate).
// CG == 2: issued by the pair leader only; A = 256 rows (128 per CTA), B = N rows (N/2 per CTA).
template <int CG = 1>
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                           uint32_t accumulate) {
    if (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
            : "memory");
    }
}
// The same two instructions issued by the lane whose `lead` flag is set, with NO branch around them: the MMA warp runs
// warp-uniform code (every lane waits on the barriers and computes the descriptors), so the descriptors stay in uniform
// registers instead of going through an ELECT / R2UR.BROADCAST / BRA.U.ANY sequence per instruction.
template <int CG = 1>
__device__ __forceinline__ void tc_mma_f16_if(uint32_t lead, uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                              uint32_t accumulate) {
    if (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
            "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(lead)
            : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %4, 0;\n\tsetp.ne.b32 q, %5, 0;\n\t"
            "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
            "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(lead)
            : "memory");
    }
}
template <int CG = 1>
__device__ __forceinline__ void tc_commit_if(uint32_t lead, uint64_t* bar) {
    if (CG == 1) {
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %1, 0;\n\t"
                     "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" ::"r"(smem_u32(bar)), "r"(lead)
                     : "memory");
    } else {
        const uint16_t mask = 3;
        asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
                     "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}\n" ::"r"(
                         smem_u32(bar)),
                     "h"(mask), "r"(lead)
                     : "memory");
    }
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets lane (base+i), columns c..c+31
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled shared-memory operand descriptor (sm_100 UMMA):
// rows of 128 B (64 x 16-bit), 8-row swizzle atoms 1024 B apart (SBO), LBO unused (=1), version 1.
__device__ __forceinline__ uint64_t make_sw128_kmajor_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFFu);
    d |= static_cast<uint64_t>(1) << 16;   // leading byte offset (ignored for swizzled K-major)
    d |= static_cast<uint64_t>(64) << 32;  // stride byte offset: 1024 B >> 4
    d |= static_cast<uint64_t>(1) << 46;   // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;   // SWIZZLE_128B
    return d;
}

// ----------------------------------------------------------------------------- host: TMA descriptors
int encode_tmap(CUtensorMap* map, CUtensorMapDataType dt, uint32_t rank, const void* base, const uint64_t* dims,
                const uint64_t* strides_bytes /*rank-1*/, const uint32_t* box, CUtensorMapSwizzle swz);

}  // namespace svb
