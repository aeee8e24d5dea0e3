// tc_common.cuh — sm_100a PTX wrappers (mbarrier, TMA, tcgen05), the fp64 exp / log-sum-exp helpers and the
// tensor-map / CTA-pair launch plumbing shared by the tensor-core --LD kernels (ld_mma.cu: shared windows;
// ld_vmma.cu: per-target windows).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#include <algorithm>
#include <utility>

#include "engine.h"

namespace ibdgem {

// ---------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// non-blocking probe: lets the issue loop overlap the latency of several barrier tests
__device__ __forceinline__ bool mbar_test(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return done != 0;
}
// wait used by the many epilogue warps: backs off so the spinning does not steal issue slots
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    for (;;) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) break;
        __nanosleep(64);
    }
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// 32 consecutive accumulator columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, int (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand slab (rows of 128 bytes, 8-row groups 1024 bytes apart):
// the tcgen05 shared-memory matrix descriptor.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);  // start address, bits [0,14)
    d |= (uint64_t)1 << 16;                   // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;         // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                   // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                   // SWIZZLE_128B
    return d;
}

// exp(x) for x <= 0 in fp64: Cody-Waite reduction, degree-12 Taylor polynomial on |r| <= ln2/2
// (truncation 2e-16), exponent rebuilt by integer add.  Used only on screened elements.
__device__ __forceinline__ double exp_nonpos(double x) {
    if (!(x > -700.0)) return 0.0;
    const double t = fma(x, 1.4426950408889634074, 6755399441055744.0);  // round(x log2 e) in the low word
    const int n = __double2loint(t);
    const double nr = t - 6755399441055744.0;
    double r = fma(nr, -6.93147180369123816490e-01, x);
    r = fma(nr, -1.90821492927058770002e-10, r);
    double p = 2.08767569878680989792e-09;  // 1/12!
    p = fma(p, r, 2.50521083854417187751e-08);
    p = fma(p, r, 2.75573192239858906526e-07);
    p = fma(p, r, 2.75573192239858906526e-06);
    p = fma(p, r, 2.48015873015873015873e-05);
    p = fma(p, r, 1.98412698412698412698e-04);
    p = fma(p, r, 1.38888888888888888889e-03);
    p = fma(p, r, 8.33333333333333333333e-03);
    p = fma(p, r, 4.16666666666666666667e-02);
    p = fma(p, r, 1.66666666666666666667e-01);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    return __hiloint2double(__double2hiint(p) + n * 1048576, __double2loint(p));
}

// exp(x) for x <= 0 with relative error below 3e-10: same reduction as exp_nonpos, degree-8 Taylor
// polynomial evaluated by Estrin's scheme (dependency depth 5 instead of 12).  Used for the screened
// candidates of the GEMM epilogue only: every such term is at most the row maximum, so the row's
// log-sum-exp moves by less than 3e-10.
__device__ __forceinline__ double exp_nonpos_fast(double x) {
    if (!(x > -700.0)) return 0.0;
    const double t = fma(x, 1.4426950408889634074, 6755399441055744.0);
    const int n = __double2loint(t);
    const double nr = t - 6755399441055744.0;
    double r = fma(nr, -6.93147180369123816490e-01, x);
    r = fma(nr, -1.90821492927058770002e-10, r);
    const double r2 = r * r, r4 = r2 * r2;
    const double p01 = fma(r, 1.0, 1.0);
    const double p23 = fma(r, 1.66666666666666666667e-01, 0.5);
    const double p45 = fma(r, 8.33333333333333333333e-03, 4.16666666666666666667e-02);
    const double p67 = fma(r, 1.98412698412698412698e-04, 1.38888888888888888889e-03);
    const double lo = fma(r2, p23, p01);
    const double hi = fma(r2, p67, p45);
    const double p = fma(r4, fma(r4, 2.48015873015873015873e-05, hi), lo);
    return __hiloint2double(__double2hiint(p) + n * 1048576, __double2loint(p));
}

// running log-sum-exp (max m, scaled sum s) += e^x
__device__ __forceinline__ void lse_add(double &m, double &s, double x) {
    const bool up = x > m;
    const double e = exp_nonpos(up ? m - x : x - m);  // one exp whichever way the maximum moves
    s = up ? fma(s, e, 1.0) : s + e;
    m = up ? x : m;
}

// the same with the short-chain exp, for the screened candidates of the GEMM epilogue.  Two tiers: a term more than
// 12 nats below the running maximum is at most 6e-6 of the sum, so its exponential is taken in fp32 (ex2.approx,
// relative error ~2e-7: 1e-12 of the sum per term, 1e-8 for ten thousand of them — the window tolerance is 1e-6);
// rows without a dominant column send most of their survivors through this tier.
__device__ __forceinline__ void lse_add_fast(double &m, double &s, double x) {
    const double d = x - m;
    if (d < -12.0) {
        s += (double)__expf((float)d);
        return;
    }
    const bool up = d > 0.0;
    const double e = exp_nonpos_fast(up ? -d : d);
    s = up ? fma(s, e, 1.0) : s + e;
    m = up ? x : m;
}

// v[j] for a per-lane j in 0..31: binary select tree (registers cannot be indexed dynamically)
template <int N>
__device__ __forceinline__ int pick_tree(const int *v, int j) {
    if constexpr (N == 1) {
        return v[0];
    } else {
        const int lo = pick_tree<N / 2>(v, j), hi = pick_tree<N / 2>(v + N / 2, j);
        return (j & (N / 2)) ? hi : lo;
    }
}
__device__ __forceinline__ int pick32(const int (&v)[32], int j) { return pick_tree<32>(v, j); }

// 4 bits -> 4 bytes of 0 / 1 (bit i to byte i)
__device__ __forceinline__ uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }
__device__ __forceinline__ unsigned warp_sum(unsigned v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// CTA-pair (tcgen05 cta_group::2) helpers and the dynamic unit ring shared by the persistent kernels
namespace tcx {
// Units are handed out dynamically (an atomic counter) by CTA 0's producer lane and travel to every role
// of both CTAs of a pair through a ring in shared memory: no "empty" barriers are needed as long as no
// role runs more than URING - 1 units ahead of another.
constexpr int URING = 8;
constexpr uint32_t PEER_MASK = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address -> CTA 0 of the pair

// executed by both CTAs of the pair; the bytes are counted on CTA 0's barrier
__device__ __forceinline__ void tma_load_3d_cg(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(smem_u32(bar) & PEER_MASK), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap *map, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
constexpr int PF_TILES = 2;
// arrives on the barrier at this offset in BOTH CTAs once the pair's MMAs retire
__device__ __forceinline__ void tc_commit_cg(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, int8 x int8 -> int32, over the pair's 256 rows
__device__ __forceinline__ void umma_i8_cg(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on CTA 0's copy of a barrier (CTA 0 itself: a plain local arrive)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_MASK) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// wait with cluster-scope acquire: the ring entry may have been written by the peer CTA
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    for (;;) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
        if (done) break;
    }
}
// unit number of iteration `it` for any role of either CTA (-1: no more units)
__device__ __forceinline__ int unit_of(const int *uring, uint64_t *ufull, int it) {
    mbar_wait_cluster(ufull + (it % URING), (uint32_t)((it / URING) & 1));
    return *reinterpret_cast<const volatile int *>(uring + (it % URING));
}
// scheduler (producer lane of CTA 0): publish unit u for iteration `it` in both CTAs of the pair
__device__ __forceinline__ void unit_publish(int *uring, uint64_t *ufull, int it, int u) {
    const int i = it % URING;
    *reinterpret_cast<volatile int *>(uring + i) = u;
    asm volatile("mbarrier.arrive.release.cluster.shared::cta.b64 _, [%0];" ::"r"(smem_u32(ufull + i)) : "memory");
    uint32_t rdata, rbar;
    asm volatile("mapa.shared::cluster.u32 %0, %1, 1;" : "=r"(rdata) : "r"(smem_u32(uring + i)));
    asm volatile("mapa.shared::cluster.u32 %0, %1, 1;" : "=r"(rbar) : "r"(smem_u32(ufull + i)));
    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(rdata), "r"(u) : "memory");
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(rbar) : "memory");
}

}  // namespace tcx

// ---------------------------------------------------------------------------------------------
// host side of the persistent CTA-pair GEMMs

// Screening distance in nats.  An element more than D below its row maximum contributes at most e^-D of the row's
// sum, so dropping every such element of a row with `ncols` columns changes the row's log-sum-exp by less than
// ncols * e^-D.  D = ln(ncols) + ln(1e7) keeps that below 1e-7 (the window tolerance is 1e-6).
constexpr double SCREEN_NATS = 32.0;
inline double screen_nats(int ncols) { return std::min(SCREEN_NATS, log((double)std::max(ncols, 2)) + 16.2); }

// TMA map of a 3-D uint8 array (dims[0] bytes contiguous; strides of dims 1 and 2 in bytes): 128-byte swizzle,
// zero fill outside
inline int encode_u8_3d(CUtensorMap *m, void *base, const cuuint64_t (&dims)[3], const cuuint64_t (&strides)[2],
                        const cuuint32_t (&box)[3]) {
    typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                      const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static const EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return (EncodeTiledFn) nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    if (!fn) {
        set_error("[::] ERROR: cuTensorMapEncodeTiled is not available from the CUDA driver.");
        return 1;
    }
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("[::] ERROR: cuTensorMapEncodeTiled failed (%d) for a %llu x %llu x %llu operand.", (int)r, (unsigned long long)dims[0],
                  (unsigned long long)dims[1], (unsigned long long)dims[2]);
        return 1;
    }
    return 0;
}

// Persistent launch of a CTA-pair kernel: clusters of 2 x 1 x 1, one pair per two SMs and at most one per unit.
template <class... Exp, class... Act>
inline int launch_pairs(void (*kernel)(Exp...), int threads, int smem_bytes, int n_units, int sm_count, cudaStream_t st, Act &&...args) {
    // function attributes are per device (the command-line front-end drives one engine per GPU from threads of one
    // process); setting it is cheap enough to do on every launch
    IBD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    const int groups = std::max(1, std::min(n_units, sm_count / 2));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(groups * 2));
    cfg.blockDim = dim3((unsigned)threads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    IBD_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<Act>(args)...));
    return 0;
}

}  // namespace ibdgem
