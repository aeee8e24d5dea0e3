// ld_vmma.cu — tensor-core --LD window scoring (L1 + L2, src/ibdgem.c:673-753) with PER-TARGET windows:
// -v (the reference's recommended flag: hom-ref sites of the compared sample are skipped,
// src/ibdgem.c:584-587) and -D (per-target thinned counts, :627-628).
//
// Algebra.  For target t the kept set is Sigma_t = { s : kept, informative, v_t(s) } with v_t = a0 | a1 under -v
// (1 otherwise); its windows are runs of W members, so they differ from target to target.  With the
// depth-linear class table (DESIGN.md 2: l1 - l0 = alpha n_ref + beta n_alt, l2 - 2 l1 + l0 = kappa n) a window
// (t, w) and a background haplotype k give, for the target's haplotype a_i,
//     ln prod_{s in Sigma_tw} P_s[a_i + k] = C0_tw + R_tw[a_i] + Y_tw[k] + kappa M_tw[a_i, k]
//     M_tw[a_i, k] = sum n_s a_i,s k_s                 -- a_i = 1 implies v = 1: no mask needed, only the range
//     Y_tw[k]      = alpha sum v_s nref_s k_s + beta sum v_s nalt_s k_s   -- TWO more integer contractions
// and for a background individual b = (r0, r1), with h = r0 & r1,
//     ln prod P_s[r0 + r1] = C0_tw + Y_tw[r0] + Y_tw[r1] + kappa (sum v nref h + sum v nalt h).
// So every (target, window) is FOUR int8 rows (n a0, n a1, v nref, v nalt) against THREE 0/1 columns per background
// individual (r0, r1, h): one exact integer GEMM whose K axis is the shared axis of informative sites, restricted
// row by row to the window's range of that axis.  Windows of different targets overlap arbitrarily, so rows are
// (target, window) pairs sorted by their start on the K axis and cut into tiles of 64 (32 per CTA of a pair);
// a tile's K range is the hull of its rows' ranges (~15 % more than a single row's at C3 with -v).
//
// The K range of a tile (~3,800 sites at C3 -v: 1,000 variable sites spread over 3.3x as many informative
// ones) does not fit shared memory, so unlike ld_mma.cu BOTH operands stream: a stage holds one 128-site
// k-block of the tile's rows (16 KB) and of the column tile (120 rows = 15 KB per CTA), accumulators
// (128 lanes x 240 columns, two slots) stay in TMEM across the whole K range, and the fused epilogue
// (fp32 screen against the row's running maximum, fp64 log-sum-exp of the survivors) runs once per
// (row tile, column tile).  Lanes 4j .. 4j+3 of a CTA hold the four rows of one (target, window): the
// epilogue exchanges them with warp shuffles.
//
// Kernels: v_slots, ld_transpose (shared with ld_mma.cu) — cached per prepared panel; v_wmap / v_tw (rank-space
// window map and per-window scalars for -v), v_tw_site (site-space variant for -D), v_sort_*, v_expand_a,
// v_expand_b, ld_vmma (per call).
#include <cuda.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "engine.h"
#include "site_math.cuh"
#include "tc_common.cuh"

namespace ibdgem {

struct VCache {
    bool valid = false;
    bool transposed = false;
    int64_t K = 0;        // informative kept sites (the K axis)
    int nblk = 0;         // blocks of 1,024 slots
    int nKB = 0;          // 128-slot k-blocks that hold at least one site
    int H = 0, N = 0;
    int32_t *d_slotsite = nullptr;  // [nblk * 1024] panel line of each slot, -1 = padding
    uint8_t *d_nk = nullptr;        // [nblk * 1024] depth of the slot (original counts)
    uint8_t *d_nr = nullptr;        // [nblk * 1024] REF-matching bases
    double *d_l0 = nullptr;         // [nblk * 1024] ln P(D | 00) of the slot's class
    uint32_t *d_tbits = nullptr;    // [nblk][H][32] haplotype-major bits over the K axis
    size_t b_slot = 0, b_n = 0, b_l0 = 0, b_tbits = 0;
    // the column operand depends on the background only: it is expanded on a side stream while the engine stream builds
    // the per-target window maps and the row tiles
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

namespace vmma {
using namespace tcx;
constexpr int BM = 128, KBYTES = 128, UK = 32;
constexpr int TW_CTA = 32;                 // (target, window) pairs per CTA: 4 accumulator lanes each
constexpr int TW_TILE = 2 * TW_CTA;        // per CTA pair
constexpr int IND_HALF = 40;               // background individuals per CTA half of a column tile
constexpr int BROWS = 3 * IND_HALF;        // rows of a B slab per CTA: r0 | r1 | h of its 40 individuals
constexpr int TILE_N = 2 * BROWS;          // 240 accumulator columns
constexpr int TILE_IND = 2 * IND_HALF;     // 80 individuals per column tile
constexpr int A_SLAB = BM * KBYTES;        // 16 KB
constexpr int B_SLAB = BROWS * KBYTES;     // 15 KB
constexpr int NSTAGE = 6;
constexpr int NACC = 2;
constexpr int ACC_STRIDE = 256;            // TMEM columns between the two accumulator slots
constexpr int EPI_WARP0 = 4;
constexpr int NSETS = 4;                   // epilogue warp sets of 4 warps (one per TMEM lane quarter); every set works on every
                                           // tile and owns a quarter of its individuals
constexpr int SET_IND = TILE_IND / NSETS;  // 20 individuals per set and tile, in chunks of 4
constexpr int THREADS = 128 + NSETS * 128;
constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + NSTAGE * A_SLAB;
constexpr int OFF_MERGE = OFF_B + NSTAGE * B_SLAB;           // NSETS x 128 double2
constexpr int OFF_SMAX = OFF_MERGE + NSETS * BM * 16;         // 2 x 128 int32: the rows' running maxima, shared by the sets
constexpr int OFF_BAR = OFF_SMAX + 2 * BM * 4;
constexpr int NBAR = 2 * NSTAGE + 2 * NACC + URING;
constexpr int OFF_TMEM = OFF_BAR + NBAR * 8;
constexpr int OFF_URING = OFF_TMEM + 16;
constexpr int SMEM_BYTES = OFF_URING + URING * 4 + 1024;
constexpr uint32_t IDESC = (2u << 4) /* D = s32 */ | (0u << 7) /* A = u8 */ | (0u << 10) /* B = u8 */ |
                           ((uint32_t)(TILE_N >> 3) << 17) | ((uint32_t)((BM * 2) >> 4) << 24);
static_assert(SMEM_BYTES <= 232448, "over the 227 KB shared memory limit");
static_assert(B_SLAB % 1024 == 0, "swizzled slabs are 1,024-byte aligned");

struct Params {
    int n_units;                 // row tiles of this batch
    int unit0;                   // first row tile of the batch (index into the tile tables)
    int NT, nKB;                 // column tiles, k-blocks of the K axis
    int n_tw;                    // (target, window) pairs in total
    int outW;
    float alpha_f, beta_f, kappa_f, screen_f;
    double alpha, beta, kappa;
    const int32_t *tile_kb0;     // [tiles] first k-block of the tile's hull
    const int32_t *tile_nkb;     // [tiles] k-blocks of the hull
    const int64_t *tile_slab;    // [tiles] first A slab of the tile within the batch buffer (rank 0; rank 1 follows)
    const int32_t *order;        // [tiles * 64] (target, window) ids in tile order, -1 = padding
    const int32_t *tw_t, *tw_w;  // [n_tw]
    const int32_t *tw_own;       // [n_tw] column individual to leave out (index into the unique background list) or -1
    const double *tw_C0, *tw_R0, *tw_R1;
    const double *lnc;           // [NT * 80] ln(multiplicity) of each column individual, -inf = padding
    const double *lognb;         // [T] ln n_refpanel or NaN
    double *wll;                 // [T][outW][3]
    double *wll_host;            // the caller's page-locked table (device alias) or nullptr: finished scores go there too
    int *unit_counter;
};

// order-preserving float <-> int map, so that atomicMax on ints is a max on floats
__device__ __forceinline__ int f2ord(float f) {
    const int i = __float_as_int(f);
    return i ^ ((i >> 31) & 0x7fffffff);
}
__device__ __forceinline__ float ord2f(int i) { return __int_as_float(i ^ ((i >> 31) & 0x7fffffff)); }
constexpr int ORD_NEG_INF = (int)0x807fffff;  // f2ord(-inf)

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, int (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}

__global__ void __launch_bounds__(THREADS, 1)
ld_vmma_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapB, const Params p) {
    constexpr int CG = 2;
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
    uint64_t *s_full = bars, *s_empty = bars + NSTAGE;
    uint64_t *acc_full = s_empty + NSTAGE, *acc_empty = acc_full + NACC;
    uint64_t *ufull = acc_empty + NACC;
    int *uring = reinterpret_cast<int *>(smem + OFF_URING);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_TMEM);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapB) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < NSTAGE; i++) { mbar_init(s_full + i, 1); mbar_init(s_empty + i, 1); }
        for (int i = 0; i < NACC; i++) { mbar_init(acc_full + i, 1); mbar_init(acc_empty + i, 4 * NSETS * CG); }
        for (int i = 0; i < URING; i++) mbar_init(ufull + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 3)
        for (int i = lane; i < 2 * BM; i += 32) reinterpret_cast<int *>(smem + OFF_SMAX)[i] = ORD_NEG_INF;
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer: both CTAs load their own rows of the tile and their own half of the column tile =====
        if (lane == 0) {
            int st = 0;
            uint32_t ph = 0;
            int u_next = -1, pending = -1;
            if (rank == 0) {
                const int v = atomicAdd(p.unit_counter, 1);
                u_next = v < p.n_units ? v : -1;
                unit_publish(uring, ufull, 0, u_next);
                pending = atomicAdd(p.unit_counter, 1);
            }
            for (int it = 0;; it++) {
                int u;
                if (rank == 0) {
                    u = u_next;
                } else {
                    u = unit_of(uring, ufull, it);
                }
                if (u < 0) break;
                const int tile = p.unit0 + u;
                const int kb0 = __ldg(p.tile_kb0 + tile), nkb = __ldg(p.tile_nkb + tile);
                const int slabA = (int)(__ldg(p.tile_slab + tile) + (int64_t)rank * nkb);
                for (int n = 0; n < p.NT; n++) {
                    const int slabB = (n * 2 + (int)rank) * p.nKB + kb0;
                    for (int kr = 0; kr < nkb; kr++) {
                        mbar_wait(s_empty + st, ph ^ 1u);
                        if (rank == 0) mbar_expect_tx(s_full + st, (uint32_t)(CG * (A_SLAB + B_SLAB)));
                        tma_load_3d_cg(smem + OFF_A + st * A_SLAB, &tmapA, s_full + st, 0, 0, slabA + kr);
                        tma_load_3d_cg(smem + OFF_B + st * B_SLAB, &tmapB, s_full + st, 0, 0, slabB + kr);
                        if (++st == NSTAGE) { st = 0; ph ^= 1u; }
                    }
                }
                if (rank == 0) {
                    u_next = pending < p.n_units ? pending : -1;
                    unit_publish(uring, ufull, it + 1, u_next);
                    if (u_next >= 0) pending = atomicAdd(p.unit_counter, 1);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (CTA 0 of the pair) =====
        if (rank == 0) {
            int st = 0;
            uint32_t ph = 0;
            uint32_t g = 0;
            const uint64_t adesc0 = umma_desc_sw128(smem_u32(smem + OFF_A));
            const uint64_t bdesc0 = umma_desc_sw128(smem_u32(smem + OFF_B));
            for (int it = 0;; it++) {
                const int u = unit_of(uring, ufull, it);
                if (u < 0) break;
                const int nkb = __ldg(p.tile_nkb + p.unit0 + u);
                for (int n = 0; n < p.NT; n++, g++) {
                    const uint32_t acc = g % NACC, use = g / NACC;
                    mbar_wait(acc_empty + acc, (use & 1u) ^ 1u);
                    const uint32_t d_tmem = tmem_base + acc * ACC_STRIDE;
                    for (int kr = 0; kr < nkb; kr++) {
                        mbar_wait(s_full + st, ph);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint64_t ad = adesc0 + (uint64_t)((st * A_SLAB) >> 4);
                            const uint64_t bd = bdesc0 + (uint64_t)((st * B_SLAB) >> 4);
#pragma unroll
                            for (int k = 0; k < KBYTES / UK; k++)
                                umma_i8_cg(d_tmem, ad + (uint64_t)(k * (UK >> 4)), bd + (uint64_t)(k * (UK >> 4)), IDESC,
                                           (uint32_t)((kr | k) != 0));
                            tc_commit_cg(s_empty + st);
                            if (kr + 1 == nkb) tc_commit_cg(acc_full + acc);
                        }
                        __syncwarp();
                        if (++st == NSTAGE) { st = 0; ph ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 2) {
        // ===== merge warp: joins the two sets' partial (max, sum) of every row, adds the row terms, writes
        // LIBD1 (rows a0, a1 of the quad) and LIBD0 (row v nref of the quad); lane j owns (target, window) j =====
        const double2 *mb = reinterpret_cast<const double2 *>(smem + OFF_MERGE);
        asm volatile("bar.arrive 2, %0;" ::"n"(NSETS * 128 + 32) : "memory");
        for (int it = 0;; it++) {
            const int u = unit_of(uring, ufull, it);
            if (u < 0) break;
            const int tile = p.unit0 + u;
            const int tw = __ldg(p.order + ((size_t)tile * 2 + rank) * TW_CTA + lane);
            double c0 = 0, r0 = 0, r1 = 0, lnb = 0;
            int t = 0, w = 0;
            if (tw >= 0) {
                c0 = __ldg(p.tw_C0 + tw); r0 = __ldg(p.tw_R0 + tw); r1 = __ldg(p.tw_R1 + tw);
                t = __ldg(p.tw_t + tw); w = __ldg(p.tw_w + tw);
                lnb = __ldg(p.lognb + t);
            }
            asm volatile("bar.sync 1, %0;" ::"n"(NSETS * 128 + 32) : "memory");
            double L[3];
#pragma unroll
            for (int c = 0; c < 3; c++) {
                double2 o[NSETS];
#pragma unroll
                for (int q = 0; q < NSETS; q++) o[q] = mb[q * BM + lane * 4 + c];
                double M = o[0].x;
#pragma unroll
                for (int q = 1; q < NSETS; q++) M = fmax(M, o[q].x);
                double S = 0.0;
#pragma unroll
                for (int q = 0; q < NSETS; q++) S = fma(o[q].y, exp_nonpos(o[q].x - M), S);
                L[c] = (S > 0.0) ? M + log(S) : -INFINITY;
            }
            asm volatile("bar.arrive 2, %0;" ::"n"(NSETS * 128 + 32) : "memory");
            if (tw >= 0) {
                const double x0 = r0 + L[0], x1 = r1 + L[1];
                const double mm = fmax(x0, x1);
                double l1 = mm == -INFINITY ? -INFINITY : mm + log(exp_nonpos(x0 - mm) + exp_nonpos(x1 - mm));
                l1 = (c0 + l1) - (lnb + 1.3862943611198906);  // ln(4 n_refpanel)
                double l0 = (c0 + L[2]) - lnb;
                if (!(lnb == lnb)) l0 = l1 = __longlong_as_double(0x7ff8000000000000LL);  // n_refpanel = 0: 0/0
                const size_t oi = ((size_t)t * p.outW + w) * 3;
                p.wll[oi] = l0;
                p.wll[oi + 1] = l1;
                if (p.wll_host) {  // posted writes over PCIe, under the remaining tiles
                    p.wll_host[oi] = l0;
                    p.wll_host[oi + 1] = l1;
                }
            }
        }
    } else if (warp >= EPI_WARP0) {
        // ===== epilogue.  Every set works on every tile: set q owns individuals [20 q, 20 q + 20) of the tile, in
        // chunks of 4.  Lane = one accumulator row; quad = one (target, window): row 0/1 = n a_i (-> M), row 2 = v nref,
        // row 3 = v nalt (-> Y, and the hom columns of the chain).  A chunk is handled in two steps so that the hot
        // path is straight-line code the compiler can interleave: first all shuffles and the fp32 screen values of the
        // chunk's 8 elements, then — rarely — the fp64 terms of the elements that passed. =====
        const int ew = warp - EPI_WARP0, set = ew >> 2, quarter = warp & 3;
        const int rloc = quarter * 32 + lane;
        const int c = lane & 3, qb = lane & ~3;
        double2 *merge = reinterpret_cast<double2 *>(smem + OFF_MERGE);
        uint32_t g0 = 0;
        for (int it = 0;; it++, g0 += (uint32_t)p.NT) {
            const int u = unit_of(uring, ufull, it);
            if (u < 0) break;
            const int tile = p.unit0 + u;
            const int tw = __ldg(p.order + ((size_t)tile * 2 + rank) * TW_CTA + (rloc >> 2));
            const int own = tw >= 0 ? __ldg(p.tw_own + tw) : -1;
            double m = -INFINITY, s = 0.0;  // rows 0, 1: the row's sum over background haplotypes; row 2: the chain over individuals
            float fmx = -INFINITY;
            // The sets see disjoint columns.  They share the row's running maximum through shared memory (monotone,
            // so a stale read only lets more elements through the screen).
            int *smax = reinterpret_cast<int *>(smem + OFF_SMAX) + (it & 1) * BM + rloc;
            for (int n = 0; n < p.NT; n++) {
                const uint32_t g = g0 + (uint32_t)n;
                const int slot = (int)(g & 1u);
                mbar_wait_relaxed(acc_full + slot, (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + slot * ACC_STRIDE + ((uint32_t)(quarter * 32) << 16);
                const double *lncn = p.lnc + (size_t)n * TILE_IND;
                fmx = fmaxf(fmx, ord2f(*reinterpret_cast<volatile int *>(smax)));
                // the screen is relative to the running row maximum, which starts at -inf: the first tile of a unit is
                // read twice, once for its maximum alone (shared by the sets)
                for (int pass = (n == 0 ? 0 : 1); pass < 2; pass++) {
                    if (pass == 1 && n == 0) {
                        atomicMax(smax, f2ord(fmx));
                        asm volatile("bar.sync 3, %0;" ::"n"(NSETS * 128) : "memory");
                        fmx = fmaxf(fmx, ord2f(*reinterpret_cast<volatile int *>(smax)));
                    }
#pragma unroll 1
                    for (int ch = 0; ch < SET_IND / 4; ch++) {
                        const int ci = set * SET_IND + ch * 4;          // first individual of the chunk within the tile
                        const int hf = ci / IND_HALF, i0 = ci % IND_HALF;
                        int v0[4], v1[4], vh[4];
                        __syncwarp();
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(v0[0]), "=r"(v0[1]), "=r"(v0[2]), "=r"(v0[3]) : "r"(taddr + hf * BROWS + i0) : "memory");
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(v1[0]), "=r"(v1[1]), "=r"(v1[2]), "=r"(v1[3]) : "r"(taddr + hf * BROWS + IND_HALF + i0) : "memory");
                        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(vh[0]), "=r"(vh[1]), "=r"(vh[2]), "=r"(vh[3]) : "r"(taddr + hf * BROWS + 2 * IND_HALF + i0) : "memory");
                        double lc[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) lc[i] = __ldg(lncn + ci + i);
                        tmem_ld_wait();
                        int vr0[4], va0[4], vr1[4], va1[4], vah[4];
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            vr0[i] = __shfl_sync(0xffffffffu, v0[i], qb | 2);
                            va0[i] = __shfl_sync(0xffffffffu, v0[i], qb | 3);
                            vr1[i] = __shfl_sync(0xffffffffu, v1[i], qb | 2);
                            va1[i] = __shfl_sync(0xffffffffu, v1[i], qb | 3);
                            vah[i] = __shfl_sync(0xffffffffu, vh[i], qb | 3);
                        }
                        float t0[4], t1[4];
                        float cmx = -INFINITY;
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const float lcf = (n * TILE_IND + ci + i == own) ? -INFINITY : (float)lc[i];
                            const float y0 = fmaf(p.alpha_f, (float)vr0[i], p.beta_f * (float)va0[i]);
                            const float y1 = fmaf(p.alpha_f, (float)vr1[i], p.beta_f * (float)va1[i]);
                            // rows 0, 1: the two pairings of the row's haplotype with the individual's; row 2: the chain
                            // P[r0 + r1] of the individual; row 3 only supplies counts
                            const float a = c < 2 ? fmaf(p.kappa_f, (float)v0[i], y0) : fmaf(p.kappa_f, (float)(vh[i] + vah[i]), y0 + y1);
                            const float b = fmaf(p.kappa_f, (float)v1[i], y1);
                            t0[i] = c < 3 ? a + lcf : -INFINITY;
                            t1[i] = c < 2 ? b + lcf : -INFINITY;
                            cmx = fmaxf(cmx, fmaxf(t0[i], t1[i]));
                        }
                        fmx = fmaxf(fmx, cmx);
                        if (pass == 0) continue;
                        const float thr = fmx - p.screen_f;
                        uint32_t mask = 0;
#pragma unroll
                        for (int i = 0; i < 4; i++) mask |= (t0[i] > thr ? 1u << (2 * i) : 0u) | (t1[i] > thr ? 2u << (2 * i) : 0u);
                        if (mask) {  // rare: the fp64 terms of the survivors
#pragma unroll
                            for (int i = 0; i < 4; i++) {
                                if (mask & (1u << (2 * i))) {
                                    double x;
                                    if (c < 2)
                                        x = fma(p.kappa, (double)v0[i], fma(p.alpha, (double)vr0[i], p.beta * (double)va0[i])) + lc[i];
                                    else
                                        x = fma(p.kappa, (double)(vh[i] + vah[i]),
                                                fma(p.alpha, (double)(vr0[i] + vr1[i]), p.beta * (double)(va0[i] + va1[i]))) + lc[i];
                                    lse_add_fast(m, s, x);
                                }
                                if (mask & (2u << (2 * i))) {
                                    const double x = fma(p.kappa, (double)v1[i], fma(p.alpha, (double)vr1[i], p.beta * (double)va1[i])) + lc[i];
                                    lse_add_fast(m, s, x);
                                }
                            }
                        }
                    }
                }
                atomicMax(smax, f2ord(fmx));
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(acc_empty + slot);
            }
            if (set == 0) reinterpret_cast<int *>(smem + OFF_SMAX)[((it + 1) & 1) * BM + rloc] = ORD_NEG_INF;  // next unit's slot (idle since unit it - 1)
            asm volatile("bar.sync 2, %0;" ::"n"(NSETS * 128 + 32) : "memory");  // previous unit's partials consumed
            merge[set * BM + rloc] = make_double2(m, s);
            asm volatile("bar.arrive 1, %0;" ::"n"(NSETS * 128 + 32) : "memory");
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}
}  // namespace vmma

// ---------------------------------------------------------------------------------------------
// target-independent: slots of the K axis
__global__ void __launch_bounds__(256)
v_slots_kernel(int64_t S, const uint8_t *__restrict__ status, const uint32_t *__restrict__ rank, const uint8_t *__restrict__ nref,
               const uint8_t *__restrict__ nalt, const double *__restrict__ lnP, int C, int32_t *__restrict__ slotsite,
               uint8_t *__restrict__ nk, uint8_t *__restrict__ nr, double *__restrict__ l0) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= S || status[s] != 1) return;
    const uint32_t j = rank[s];
    const int a = nref[s], b = nalt[s];
    slotsite[j] = (int32_t)s;
    nk[j] = (uint8_t)(a + b);
    nr[j] = (uint8_t)a;
    l0[j] = lnP[(size_t)(a * C + b) * 3];
}

// -v window map in rank space: one warp per target walks the words v = x0 | x1 of the target's two haplotype
// rows (32 slots per word, 32 words per pass) and records the slot of the first and last member of every
// window (W2, src/ibdgem.c:559-578, 723-730).
constexpr int WMAP_WARPS = 8;
__global__ void __launch_bounds__(WMAP_WARPS * 32)
v_wmap_kernel(int T, const int32_t *__restrict__ targets, const uint32_t *__restrict__ tbits, int H, int nblk, int W, int mapW,
              int32_t *__restrict__ ks, int32_t *__restrict__ ke, int32_t *__restrict__ nwin, int64_t *__restrict__ ktot) {
    // one CTA per target; warp k takes the k-th contiguous share of the 1,024-slot blocks: a first pass counts its
    // members, a prefix over the warps gives its starting rank, a second pass records the window boundaries
    __shared__ int64_t wcnt[WMAP_WARPS];
    __shared__ int wlast[WMAP_WARPS];
    const int t = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (t >= T) return;
    const int ind = __ldg(targets + t);
    const int per = (nblk + WMAP_WARPS - 1) / WMAP_WARPS;
    const int b_lo = min(nblk, wid * per), b_hi = min(nblk, b_lo + per);
    const uint32_t *r0 = tbits + (size_t)(2 * ind) * 32 + lane, *r1 = r0 + 32;
    int64_t cnt = 0;
    for (int b = b_lo; b < b_hi; b++) cnt += __popc(__ldg(r0 + (size_t)b * H * 32) | __ldg(r1 + (size_t)b * H * 32));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) wcnt[wid] = cnt;
    __syncthreads();
    int64_t running = 0;
    for (int k = 0; k < wid; k++) running += wcnt[k];
    int last = -1;
    for (int b = b_lo; b < b_hi; b++) {
        const uint32_t m = __ldg(r0 + (size_t)b * H * 32) | __ldg(r1 + (size_t)b * H * 32);
        const int pc = __popc(m);
        int incl = pc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        const int64_t excl = running + incl - pc;
        if (pc) {
            const int slot0 = (b * 32 + lane) * 32;
            for (int64_t r = (excl + W - 1) / W * W; r < excl + pc; r += W) {  // members that open a window
                const int64_t wi = r / W;
                if (wi < mapW) ks[(size_t)t * mapW + wi] = slot0 + (int)__fns(m, 0, (int)(r - excl) + 1);
            }
            for (int64_t r = excl + ((W - 1 - excl % W) + W) % W; r < excl + pc; r += W) {  // members that close one
                const int64_t wi = r / W;
                if (wi < mapW) ke[(size_t)t * mapW + wi] = slot0 + (int)__fns(m, 0, (int)(r - excl) + 1);
            }
            last = slot0 + 31 - __clz(m);
        }
        running += __shfl_sync(0xffffffffu, incl, 31);
    }
    last = __reduce_max_sync(0xffffffffu, last);
    if (lane == 0) wlast[wid] = last;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t total = 0;
        int lastall = -1;
        for (int k = 0; k < WMAP_WARPS; k++) {
            total += wcnt[k];
            lastall = max(lastall, wlast[k]);
        }
        const int64_t nw = (total + W - 1) / W;
        if (total % W != 0 && nw - 1 < mapW) ke[(size_t)t * mapW + nw - 1] = lastall;  // the partial last window (src/ibdgem.c:575-578)
        nwin[t] = (int32_t)nw;
        ktot[t] = total;
    }
}

// exclusive prefix of the window counts -> first (target, window) id of every target, and the total
__global__ void __launch_bounds__(1024) v_twbase_kernel(int T, const int32_t *__restrict__ nwin, int32_t *__restrict__ twbase) {
    __shared__ int ws[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int t0 = 0; t0 < T; t0 += 1024) {
        const int t = t0 + threadIdx.x;
        const int v = t < T ? nwin[t] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if ((threadIdx.x & 31) >= o) x += y;
        }
        if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
        __syncthreads();
        int off = 0;
        for (int k = 0; k < (int)(threadIdx.x >> 5); k++) off += ws[k];
        const int excl = carry + off + x - v;
        if (t < T) twbase[t] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) twbase[T] = carry;
}

// Per (target, window) scalars in rank space (-v, shared counts): one warp per pair.
//   C0 = sum l0 over the members, R[a_i] = alpha sum a_i nref + beta sum a_i nalt, LIBD2 = C0 + R0 + R1 + kappa sum n a0 a1
// plus the window bookkeeping (W2).  Members of the window = set bits of v = x0 | x1 in [ks, ke].
__global__ void __launch_bounds__(256)
v_tw_kernel(int T, int mapW, int outW, const int32_t *__restrict__ targets, const int32_t *__restrict__ nwin, const int32_t *__restrict__ twbase,
            const int32_t *__restrict__ ks, const int32_t *__restrict__ ke, const uint32_t *__restrict__ tbits, int H,
            const uint8_t *__restrict__ nr, const uint8_t *__restrict__ nk, const double *__restrict__ l0, const int32_t *__restrict__ slotsite,
            const uint64_t *__restrict__ pos, double alpha, double beta, double kappa, int32_t *__restrict__ tw_t, int32_t *__restrict__ tw_w,
            int32_t *__restrict__ tw_ks, int32_t *__restrict__ tw_ke, double *__restrict__ tw_C0, double *__restrict__ tw_R0,
            double *__restrict__ tw_R1, double *__restrict__ wll, int32_t *__restrict__ wn, uint64_t *__restrict__ ws, uint64_t *__restrict__ we,
            int32_t *__restrict__ nwout, const int32_t *__restrict__ ownT, int32_t *__restrict__ tw_own) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (gw >= (int64_t)T * mapW) return;
    const int t = (int)(gw / mapW), w = (int)(gw % mapW);
    const int nw = nwin[t];
    if (w == 0 && lane == 0) nwout[t] = nw;
    if (w >= nw || w >= outW) return;
    const int ind = __ldg(targets + t);
    const int k0 = ks[(size_t)t * mapW + w], k1 = ke[(size_t)t * mapW + w];
    unsigned A0 = 0, N0 = 0, A1 = 0, N1 = 0, M = 0, cnt = 0;
    double c0 = 0.0;
    for (int j = (k0 >> 5) + lane; j <= (k1 >> 5); j += 32) {
        const size_t base = ((size_t)(j >> 5) * H) * 32 + (j & 31);
        uint32_t x0 = __ldg(tbits + base + (size_t)(2 * ind) * 32), x1 = __ldg(tbits + base + (size_t)(2 * ind + 1) * 32);
        uint32_t rm = 0xffffffffu;  // slots of this word inside [k0, k1]
        if (j == (k0 >> 5)) rm &= 0xffffffffu << (k0 & 31);
        if (j == (k1 >> 5)) rm &= 0xffffffffu >> (31 - (k1 & 31));
        x0 &= rm;
        x1 &= rm;
        const uint4 *cr = reinterpret_cast<const uint4 *>(nr + (size_t)j * 32);
        const uint4 *cn = reinterpret_cast<const uint4 *>(nk + (size_t)j * 32);
        const uint4 r0 = __ldg(cr), r1 = __ldg(cr + 1), n0 = __ldg(cn), n1 = __ldg(cn + 1);
        const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
        const uint32_t nn[8] = {n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, n1.z, n1.w};
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const uint32_t e0 = spread4((x0 >> (4 * k)) & 15u), e1 = spread4((x1 >> (4 * k)) & 15u);
            A0 = __dp4a(e0, rr[k], A0);
            N0 = __dp4a(e0, nn[k], N0);
            A1 = __dp4a(e1, rr[k], A1);
            N1 = __dp4a(e1, nn[k], N1);
            M = __dp4a(e0 & e1, nn[k], M);
        }
        uint32_t v = x0 | x1;
        cnt += __popc(v);
        // walk over the ~10 set bits, four at a time so that four loads are in flight before the first add needs its
        // value (one bit at a time was a chain of L1 latencies; 32 predicated loads per word measured slower still)
        const double *lw = l0 + (size_t)j * 32;
        while (v) {
            const int b0 = __ffs((int)v) - 1;
            v &= v - 1u;
            const int b1 = __ffs((int)v) - 1;  // -1 when v is empty
            v &= v - 1u;                       // (0 & anything stays 0)
            const int b2 = __ffs((int)v) - 1;
            v &= v - 1u;
            const int b3 = __ffs((int)v) - 1;
            v &= v - 1u;
            const double q0 = __ldg(lw + b0);
            const double q1 = b1 >= 0 ? __ldg(lw + b1) : 0.0;
            const double q2 = b2 >= 0 ? __ldg(lw + b2) : 0.0;
            const double q3 = b3 >= 0 ? __ldg(lw + b3) : 0.0;
            c0 += (q0 + q1) + (q2 + q3);
        }
    }
    A0 = warp_sum(A0); N0 = warp_sum(N0); A1 = warp_sum(A1); N1 = warp_sum(N1); M = warp_sum(M); cnt = warp_sum(cnt);
    c0 = warp_sum(c0);
    if (lane == 0) {
        const int tw = twbase[t] + w;
        const double R0 = fma(alpha, (double)A0, beta * (double)(N0 - A0));
        const double R1 = fma(alpha, (double)A1, beta * (double)(N1 - A1));
        tw_t[tw] = t; tw_w[tw] = w; tw_ks[tw] = k0; tw_ke[tw] = k1; tw_own[tw] = ownT[t];
        tw_C0[tw] = c0; tw_R0[tw] = R0; tw_R1[tw] = R1;
        const int64_t o = (int64_t)t * outW + w;
        wll[o * 3 + 2] = ((c0 + R0) + R1) + kappa * (double)M;
        wn[o] = (int32_t)cnt;
        ws[o] = pos[slotsite[k0]];
        we[o] = pos[slotsite[k1]];
    }
}

// The same per (target, window) scalars in SITE space, for per-target counts (-D, with or without -v): the window
// map comes from the scan kernels of engine.cu (first / last panel line of every window).
__global__ void __launch_bounds__(256)
v_tw_site_kernel(SiteView v, int T, int mapW, int outW, const int32_t *__restrict__ targets, const int32_t *__restrict__ nwin,
                 const int32_t *__restrict__ twbase, const int64_t *__restrict__ wfirst, const int64_t *__restrict__ wlast,
                 const uint32_t *__restrict__ rank, const double *__restrict__ lnP, int C, const uint64_t *__restrict__ pos, double alpha,
                 double beta, double kappa, int32_t *__restrict__ tw_t, int32_t *__restrict__ tw_w, int32_t *__restrict__ tw_ks,
                 int32_t *__restrict__ tw_ke, double *__restrict__ tw_C0, double *__restrict__ tw_R0, double *__restrict__ tw_R1,
                 double *__restrict__ wll, int32_t *__restrict__ wn, uint64_t *__restrict__ ws, uint64_t *__restrict__ we,
                 int32_t *__restrict__ nwout, const int32_t *__restrict__ ownT, int32_t *__restrict__ tw_own) {
    const int lane = threadIdx.x & 31;
    const int64_t gw = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (gw >= (int64_t)T * mapW) return;
    const int t = (int)(gw / mapW), w = (int)(gw % mapW);
    const int nw = nwin[t];
    if (w == 0 && lane == 0) nwout[t] = nw;
    if (w >= nw || w >= outW) return;
    const int ind = __ldg(targets + t);
    const int64_t s0 = wfirst[(size_t)t * mapW + w], s1 = wlast[(size_t)t * mapW + w];
    unsigned A0 = 0, B0 = 0, A1 = 0, B1 = 0, M = 0, cnt = 0;
    double c0 = 0.0;
    for (int64_t s = s0 + lane; s <= s1; s += 32) {
        int r, a, g;
        if (site_eval(v, t, ind, s, r, a, g) != 1) continue;
        const uint32_t pr = hap_pair(v.bits + s * v.Wh, ind);
        const unsigned a0 = pr & 1u, a1 = pr >> 1;
        cnt++;
        A0 += a0 * r; B0 += a0 * a; A1 += a1 * r; B1 += a1 * a; M += (a0 & a1) * (r + a);
        c0 += __ldg(lnP + (size_t)(r * C + a) * 3);
    }
    A0 = warp_sum(A0); B0 = warp_sum(B0); A1 = warp_sum(A1); B1 = warp_sum(B1); M = warp_sum(M); cnt = warp_sum(cnt);
    c0 = warp_sum(c0);
    if (lane == 0) {
        const int tw = twbase[t] + w;
        const double R0 = fma(alpha, (double)A0, beta * (double)B0), R1 = fma(alpha, (double)A1, beta * (double)B1);
        tw_t[tw] = t; tw_w[tw] = w; tw_ks[tw] = (int32_t)rank[s0]; tw_ke[tw] = (int32_t)rank[s1]; tw_own[tw] = ownT[t];
        tw_C0[tw] = c0; tw_R0[tw] = R0; tw_R1[tw] = R1;
        const int64_t o = (int64_t)t * outW + w;
        wll[o * 3 + 2] = ((c0 + R0) + R1) + kappa * (double)M;
        wn[o] = (int32_t)cnt;
        ws[o] = pos[s0];
        we[o] = pos[s1];
    }
}

// ---------------------------------------------------------------------------------------------
// (target, window) pairs sorted by the k-block of their first member (counting sort), then cut into tiles of 64
__global__ void __launch_bounds__(256) v_sort_hist_kernel(int n_tw, const int32_t *__restrict__ tw_ks, int32_t *__restrict__ hist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_tw) atomicAdd(hist + (tw_ks[i] >> 7), 1);
}
__global__ void __launch_bounds__(1024) v_sort_scan_kernel(int nb, int32_t *__restrict__ hist /* in: counts, out: exclusive offsets */) {
    __shared__ int ws[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int b0 = 0; b0 < nb; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        const int v = i < nb ? hist[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if ((threadIdx.x & 31) >= o) x += y;
        }
        if ((threadIdx.x & 31) == 31) ws[threadIdx.x >> 5] = x;
        __syncthreads();
        int off = 0;
        for (int k = 0; k < (int)(threadIdx.x >> 5); k++) off += ws[k];
        const int excl = carry + off + x - v;
        if (i < nb) hist[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256)
v_sort_scatter_kernel(int n_tw, const int32_t *__restrict__ tw_ks, int32_t *__restrict__ cursor, int32_t *__restrict__ order) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_tw) order[atomicAdd(cursor + (tw_ks[i] >> 7), 1)] = i;
}
// hull of every tile on the K axis, in k-blocks; pads the order list of the last tile with -1
__global__ void __launch_bounds__(64)
v_tiles_kernel(int n_tw, int n_tiles, int32_t *__restrict__ order, const int32_t *__restrict__ tw_ks, const int32_t *__restrict__ tw_ke,
               int32_t *__restrict__ tile_kb0, int32_t *__restrict__ tile_nkb) {
    const int tile = blockIdx.x;
    const int i = tile * vmma::TW_TILE + threadIdx.x;
    int lo = 0x7fffffff, hi = -1;
    if (i < n_tw) {
        const int tw = order[i];
        lo = tw_ks[tw] >> 7;
        hi = tw_ke[tw] >> 7;
    } else {
        order[i] = -1;
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    __shared__ int slo[2], shi[2];
    if ((threadIdx.x & 31) == 0) { slo[threadIdx.x >> 5] = lo; shi[threadIdx.x >> 5] = hi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        lo = min(slo[0], slo[1]);
        hi = max(shi[0], shi[1]);
        tile_kb0[tile] = lo;
        tile_nkb[tile] = hi - lo + 1;
    }
}

// A slabs: block = (k-block of the tile's hull, tile half); thread = (pair j of the CTA, 32-slot word of the k-block).
// Rows 4j .. 4j+3 of the slab: n a0, n a1, v nref, v nalt, zero outside the window's own range [ks, ke].
__global__ void __launch_bounds__(128)
v_expand_a_kernel(int unit0, const int32_t *__restrict__ tile_kb0, const int32_t *__restrict__ tile_nkb, const int64_t *__restrict__ tile_slab,
                  const int32_t *__restrict__ order, const int32_t *__restrict__ tw_t, const int32_t *__restrict__ tw_ks,
                  const int32_t *__restrict__ tw_ke, const int32_t *__restrict__ targets, const uint32_t *__restrict__ tbits, int H,
                  const uint8_t *__restrict__ nr, const uint8_t *__restrict__ nk, const int32_t *__restrict__ slotsite,
                  const uint8_t *__restrict__ tgt_counts, int64_t S, int vflag, unsigned char *__restrict__ out) {
    const int tile = unit0 + blockIdx.y / 2, rank = blockIdx.y & 1;
    const int kr = blockIdx.x;
    if (kr >= tile_nkb[tile]) return;
    const int kb = tile_kb0[tile] + kr;
    const int j = threadIdx.x >> 2, part = threadIdx.x & 3;
    const int tw = order[((size_t)tile * 2 + rank) * vmma::TW_CTA + j];
    uint32_t e[4][8];
#pragma unroll
    for (int c = 0; c < 4; c++)
#pragma unroll
        for (int k = 0; k < 8; k++) e[c][k] = 0u;
    if (tw >= 0) {
        const int t = tw_t[tw];
        const int ind = targets[t];
        const int word = kb * 4 + part;          // 32-slot word of the K axis
        const int slot0 = word * 32;
        const int k0 = tw_ks[tw], k1 = tw_ke[tw];
        uint32_t rm = 0u;
        if (slot0 + 31 >= k0 && slot0 <= k1) {
            rm = 0xffffffffu;
            if (k0 > slot0) rm &= 0xffffffffu << (k0 - slot0);
            if (k1 < slot0 + 31) rm &= 0xffffffffu >> (31 - (k1 - slot0));
        }
        if (rm) {
            const size_t base = ((size_t)(word >> 5) * H) * 32 + (word & 31);
            const uint32_t x0 = __ldg(tbits + base + (size_t)(2 * ind) * 32) & rm, x1 = __ldg(tbits + base + (size_t)(2 * ind + 1) * 32) & rm;
            const uint32_t vm = vflag ? (x0 | x1) : rm;
            uint32_t rr[8], nn[8];
            if (tgt_counts) {  // -D: this target's own thinned counts, gathered through the slot -> panel line map
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    uint32_t r4 = 0, n4 = 0;
#pragma unroll
                    for (int b = 0; b < 4; b++) {
                        const int32_t s = __ldg(slotsite + slot0 + k * 4 + b);
                        if (s >= 0) {
                            const uint8_t *cc = tgt_counts + ((size_t)t * S + s) * 2;
                            const uint32_t r = cc[0], a = cc[1];
                            r4 |= r << (8 * b);
                            n4 |= (r + a) << (8 * b);
                        }
                    }
                    rr[k] = r4;
                    nn[k] = n4;
                }
            } else {
                const uint4 *cr = reinterpret_cast<const uint4 *>(nr + (size_t)slot0);
                const uint4 *cn = reinterpret_cast<const uint4 *>(nk + (size_t)slot0);
                const uint4 r0 = __ldg(cr), r1 = __ldg(cr + 1), n0 = __ldg(cn), n1 = __ldg(cn + 1);
                rr[0] = r0.x; rr[1] = r0.y; rr[2] = r0.z; rr[3] = r0.w; rr[4] = r1.x; rr[5] = r1.y; rr[6] = r1.z; rr[7] = r1.w;
                nn[0] = n0.x; nn[1] = n0.y; nn[2] = n0.z; nn[3] = n0.w; nn[4] = n1.x; nn[5] = n1.y; nn[6] = n1.z; nn[7] = n1.w;
            }
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const uint32_t m0 = spread4((x0 >> (4 * k)) & 15u) * 0xFFu, m1 = spread4((x1 >> (4 * k)) & 15u) * 0xFFu;
                const uint32_t mv = spread4((vm >> (4 * k)) & 15u) * 0xFFu;
                e[0][k] = m0 & nn[k];
                e[1][k] = m1 & nn[k];
                e[2][k] = mv & rr[k];
                e[3][k] = mv & (nn[k] - rr[k]);  // bytewise: n >= nref in every byte, no borrow crosses a byte
            }
        }
    }
    const size_t slab = (size_t)tile_slab[tile] + (size_t)rank * tile_nkb[tile] + kr;
    unsigned char *base = out + slab * vmma::A_SLAB + (size_t)(4 * j) * 128 + part * 32;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        uint4 *o = reinterpret_cast<uint4 *>(base + c * 128);
        __stcs(o, make_uint4(e[c][0], e[c][1], e[c][2], e[c][3]));
        __stcs(o + 1, make_uint4(e[c][4], e[c][5], e[c][6], e[c][7]));
    }
}

// B slabs: block = (1,024-slot block = 8 k-blocks, column tile half); thread = (individual of the half, 32-slot word
// of the k-block).  Rows i, 40 + i, 80 + i of the slab: r0, r1, r0 & r1 of individual i as 0/1 bytes.  All 16 loads of a
// thread are issued before its first store.
__global__ void __launch_bounds__(160)
v_expand_b_kernel(int nKB, int nU, const int32_t *__restrict__ bgU, const uint32_t *__restrict__ tbits, int H, unsigned char *__restrict__ out) {
    const int blk = blockIdx.x, half = blockIdx.y;  // half = n * 2 + rank
    const int i = threadIdx.x >> 2, part = threadIdx.x & 3;
    const int u = half * vmma::IND_HALF + i;
    uint32_t x0[8], x1[8];
#pragma unroll
    for (int j = 0; j < 8; j++) x0[j] = x1[j] = 0;
    if (u < nU) {
        const int ind = __ldg(bgU + u);
        const uint32_t *r0 = tbits + ((size_t)blk * H + (size_t)(2 * ind)) * 32 + part;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            x0[j] = __ldg(r0 + 4 * j);
            x1[j] = __ldg(r0 + 32 + 4 * j);
        }
    }
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int kb = blk * 8 + j;
        if (kb >= nKB) break;
        const uint32_t xs[3] = {x0[j], x1[j], x0[j] & x1[j]};
        unsigned char *slab = out + ((size_t)half * nKB + kb) * vmma::B_SLAB;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            uint32_t e[8];
#pragma unroll
            for (int k = 0; k < 8; k++) e[k] = spread4((xs[c] >> (4 * k)) & 15u);
            uint4 *o = reinterpret_cast<uint4 *>(slab + (size_t)(c * vmma::IND_HALF + i) * 128 + part * 32);
            __stcs(o, make_uint4(e[0], e[1], e[2], e[3]));
            __stcs(o + 1, make_uint4(e[4], e[5], e[6], e[7]));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// `nslabs` slabs of `rows` rows of 128 bytes, box = one slab
static int make_slab_map(CUtensorMap *m, void *base, int rows, int64_t nslabs) {
    return encode_u8_3d(m, base, {128, (cuuint64_t)rows, (cuuint64_t)nslabs}, {128, (cuuint64_t)rows * 128}, {128, (cuuint32_t)rows, 1});
}

constexpr size_t V_A_BUDGET = (size_t)8 << 30;    // bytes of A slabs per batch of row tiles
constexpr size_t V_B_LIMIT = (size_t)64 << 30;    // the B operand covers the whole K axis: beyond this the general path runs

void ld_vtensor_release(ibdgem_engine *e) {
    VCache *c = e->vc;
    if (!c) return;
    dev_free(e, c->d_slotsite, c->b_slot);
    dev_free(e, c->d_nk, c->b_n);
    dev_free(e, c->d_nr, c->b_n);
    dev_free(e, c->d_l0, c->b_l0);
    dev_free(e, c->d_tbits, c->b_tbits);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_join) cudaEventDestroy(c->ev_join);
    delete c;
    e->vc = nullptr;
}
void ld_vtensor_invalidate(ibdgem_engine *e) {
    if (e->vc) e->vc->valid = false;
}

bool ld_vtensor_eligible(ibdgem_engine *e, int32_t n_targets, int32_t nU) {
    if (!e->depth_linear || !(e->kappa < -1e-3)) return false;
    if (e->K_shared <= 0 || n_targets <= 0 || nU <= 0) return false;
    // the screen runs in fp32: |Y + kappa M| <= W * max_cov * (|alpha| + |beta| + |kappa|) must leave its ulp well under a nat
    const double mag = (double)e->prm.window_size * e->prm.max_cov * (fabs(e->alpha) + fabs(e->beta) + fabs(e->kappa));
    if (mag > 4.0e6) return false;
    const int64_t nKB = (e->K_shared + 127) / 128;
    const int NT = (e->N + vmma::TILE_IND - 1) / vmma::TILE_IND;
    if ((size_t)NT * 2 * (size_t)nKB * vmma::B_SLAB > V_B_LIMIT) return false;
    if ((int64_t)e->prm.max_cov * e->K_shared >= ((int64_t)1 << 31)) return false;  // int32 accumulators
    return true;
}

static int v_build_cache(ibdgem_engine *e) {
    if (e->vc && e->vc->valid) return 0;
    const int nblk = (int)((e->K_shared + 1023) / 1024);
    if (e->vc && (e->vc->nblk != nblk || e->vc->N != e->N)) ld_vtensor_release(e);
    VCache *c = e->vc;
    if (!c) {
        c = new VCache();
        e->vc = c;
        c->nblk = nblk;
        c->N = e->N;
        c->H = 2 * e->N;
        const size_t slots = (size_t)nblk * 1024;
        c->b_slot = slots * 4; c->b_n = slots; c->b_l0 = slots * 8; c->b_tbits = (size_t)nblk * c->H * 32 * 4;
        if (dev_alloc(e, (void **)&c->d_slotsite, c->b_slot) || dev_alloc(e, (void **)&c->d_nk, c->b_n) ||
            dev_alloc(e, (void **)&c->d_nr, c->b_n) || dev_alloc(e, (void **)&c->d_l0, c->b_l0) ||
            dev_alloc(e, (void **)&c->d_tbits, c->b_tbits))
            return 1;
    }
    c->K = e->K_shared;
    c->nKB = (int)((c->K + 127) / 128);
    IBD_CUDA(cudaMemsetAsync(c->d_slotsite, 0xFF, c->b_slot, e->stream));
    IBD_CUDA(cudaMemsetAsync(c->d_nk, 0, c->b_n, e->stream));
    IBD_CUDA(cudaMemsetAsync(c->d_nr, 0, c->b_n, e->stream));
    IBD_CUDA(cudaMemsetAsync(c->d_l0, 0, c->b_l0, e->stream));
    {
        LaunchScope ls(e, K_V_SLOTS);
        v_slots_kernel<<<(unsigned)((e->S + 255) / 256), 256, 0, e->stream>>>(e->S, e->d_status, e->d_rank, e->d_nref, e->d_nalt, e->d_lnP,
                                                                            e->C, c->d_slotsite, c->d_nk, c->d_nr, c->d_l0);
    }
    IBD_CUDA(cudaGetLastError());
    // haplotype-major bits over the K axis: the transposition kernel of the shared-window path with 1,024-slot "windows"
    if (ld_transpose_launch(e, 0, nblk, c->d_slotsite, 1024, 32, c->H, c->d_tbits)) return 1;
    c->valid = true;
    return 0;
}

// Fills every window output of the call (d_wll [T][outW][3], d_wn, d_ws, d_we [T][outW], d_nwout [T]).
int ld_vtensor_score(ibdgem_engine *e, ScoreCall &sc) {
    using namespace vmma;
    if (ensure_table(e, e->S)) return 1;  // waits for the whole panel
    if (v_build_cache(e)) return 1;
    VCache *c = e->vc;
    const SiteView &v = sc.v;
    const int T = sc.T, outW = sc.outW;
    const int32_t *d_targets = sc.d_targets;
    const uint8_t *d_tgt_counts = v.tgt_counts;
    double *d_wll = sc.d_wll;
    const int W = e->prm.window_size;
    const int mapW = map_windows(e);

    LdBackground &bg = sc.bg;
    const int nU = (int)bg.bgU.size();
    const int NT = (nU + TILE_IND - 1) / TILE_IND;
    bg.lnc.resize((size_t)NT * TILE_IND, -INFINITY);  // padding columns of the last tile

    // ---- background operand over the whole K axis, on the side stream ----------------------------
    const int nKB = c->nKB;
    double *d_lnc, *d_lognb;
    int32_t *d_bgU, *d_ownT;
    if (scratch(e, SC_V_MISC, (size_t)NT * TILE_IND * 8 + (size_t)T * 8 + (size_t)nU * 4 + (size_t)T * 4 + 64, (void **)&d_lnc)) return 1;
    d_lognb = d_lnc + (size_t)NT * TILE_IND;
    d_bgU = reinterpret_cast<int32_t *>(d_lognb + T);
    d_ownT = d_bgU + nU;
    IBD_CUDA(cudaMemcpyAsync(d_lnc, bg.lnc.data(), bg.lnc.size() * 8, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(d_lognb, bg.lognb.data(), (size_t)T * 8, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(d_bgU, bg.bgU.data(), (size_t)nU * 4, cudaMemcpyHostToDevice, e->stream));
    IBD_CUDA(cudaMemcpyAsync(d_ownT, bg.own.data(), (size_t)T * 4, cudaMemcpyHostToDevice, e->stream));
    unsigned char *d_B;
    const size_t b_bytes = (size_t)NT * 2 * nKB * B_SLAB;
    if (scratch(e, SC_MMA_BG, b_bytes, (void **)&d_B)) return 1;
    if (!c->side) {
        IBD_CUDA(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
        IBD_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        IBD_CUDA(cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    }
    IBD_CUDA(cudaEventRecord(c->ev_fork, e->stream));
    IBD_CUDA(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
    {
        LaunchScope ls(e, K_V_EXPAND_B, c->side);
        v_expand_b_kernel<<<dim3((unsigned)((nKB + 7) / 8), (unsigned)(NT * 2)), 160, 0, c->side>>>(nKB, nU, d_bgU, c->d_tbits, c->H, d_B);
    }
    IBD_CUDA(cudaEventRecord(c->ev_join, c->side));
    // every way out of this function rejoins the side stream: the scratch it writes belongs to the engine stream's next call
    struct Join {
        ibdgem_engine *e;
        VCache *c;
        ~Join() { cudaStreamWaitEvent(e->stream, c->ev_join, 0); }
    } join{e, c};
    IBD_CUDA(cudaGetLastError());
    CUtensorMap mapB;
    if (make_slab_map(&mapB, d_B, BROWS, (int64_t)NT * 2 * nKB)) return 1;

    // ---- per-target window map -> (target, window) records -------------------------------------
    int32_t *d_ks, *d_ke, *d_nwin, *d_twbase;
    int64_t *d_ktot;
    if (scratch(e, SC_V_KS, (size_t)T * mapW * 4, (void **)&d_ks) || scratch(e, SC_V_KE, (size_t)T * mapW * 4, (void **)&d_ke) ||
        scratch(e, SC_NWIN, (size_t)T * 4, (void **)&d_nwin) || scratch(e, SC_KTOT, (size_t)T * 8, (void **)&d_ktot) ||
        scratch(e, SC_V_TWBASE, (size_t)(T + 1) * 4, (void **)&d_twbase))
        return 1;
    int64_t *d_wf = nullptr, *d_wl = nullptr;
    if (d_tgt_counts) {
        if (scratch(e, SC_WFIRST, (size_t)T * mapW * 8, (void **)&d_wf) || scratch(e, SC_WLAST, (size_t)T * mapW * 8, (void **)&d_wl)) return 1;
        if (build_window_map(e, v, d_targets, T, mapW, d_wf, d_wl, d_nwin, d_ktot, nullptr)) return 1;
    } else {
        LaunchScope ls(e, K_V_WMAP);
        v_wmap_kernel<<<(unsigned)T, WMAP_WARPS * 32, 0, e->stream>>>(T, d_targets, c->d_tbits, c->H, c->nblk, W, mapW, d_ks, d_ke, d_nwin, d_ktot);
    }
    {
        LaunchScope ls(e, K_V_SORT);
        v_twbase_kernel<<<1, 1024, 0, e->stream>>>(T, d_nwin, d_twbase);
    }
    IBD_CUDA(cudaGetLastError());
    std::vector<int32_t> h_twbase((size_t)T + 1);
    IBD_CUDA(cudaMemcpyAsync(h_twbase.data(), d_twbase, (size_t)(T + 1) * 4, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    const int n_tw = h_twbase[(size_t)T];
    for (int t = 0; t < T; t++)
        if (h_twbase[(size_t)t + 1] - h_twbase[(size_t)t] > outW) {
            set_error("[::] ERROR: target %d has %d windows but max_windows = %d.", t, h_twbase[(size_t)t + 1] - h_twbase[(size_t)t], outW);
            return 1;
        }
    if (n_tw == 0) {  // no target has a single kept site: nothing to score (n_windows = 0 everywhere)
        IBD_CUDA(cudaMemsetAsync(sc.d_nwout, 0, (size_t)T * 4, e->stream));
        return 0;
    }
    const int n_tiles = (n_tw + TW_TILE - 1) / TW_TILE;

    int32_t *d_tw_t, *d_tw_w, *d_tw_ks, *d_tw_ke, *d_tw_own, *d_order, *d_hist, *d_tile_kb0, *d_tile_nkb;
    double *d_tw_C0, *d_tw_R0, *d_tw_R1;
    int64_t *d_tile_slab;
    const size_t twn = (size_t)n_tiles * TW_TILE;
    if (scratch(e, SC_V_TWI, twn * 4 * 5, (void **)&d_tw_t) || scratch(e, SC_V_TWD, twn * 8 * 3, (void **)&d_tw_C0) ||
        scratch(e, SC_V_ORDER, twn * 4, (void **)&d_order) || scratch(e, SC_V_HIST, (size_t)(nKB + 2) * 4 * 2, (void **)&d_hist) ||
        scratch(e, SC_V_TILES, (size_t)n_tiles * (4 + 4 + 8), (void **)&d_tile_slab))
        return 1;
    d_tw_w = d_tw_t + twn; d_tw_ks = d_tw_w + twn; d_tw_ke = d_tw_ks + twn; d_tw_own = d_tw_ke + twn;
    d_tw_R0 = d_tw_C0 + twn; d_tw_R1 = d_tw_R0 + twn;
    d_tile_kb0 = reinterpret_cast<int32_t *>(d_tile_slab + n_tiles); d_tile_nkb = d_tile_kb0 + n_tiles;
    int32_t *d_cursor = d_hist + (nKB + 2);
    {
        LaunchScope ls(e, K_V_TW);
        const int64_t warps = (int64_t)T * mapW;
        if (d_tgt_counts)
            v_tw_site_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, e->stream>>>(
                v, T, mapW, outW, d_targets, d_nwin, d_twbase, d_wf, d_wl, e->d_rank, e->d_lnP, e->C, e->d_pos, e->alpha, e->beta, e->kappa,
                d_tw_t, d_tw_w, d_tw_ks, d_tw_ke, d_tw_C0, d_tw_R0, d_tw_R1, d_wll, sc.d_wn, sc.d_ws, sc.d_we, sc.d_nwout, d_ownT, d_tw_own);
        else
            v_tw_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, e->stream>>>(
                T, mapW, outW, d_targets, d_nwin, d_twbase, d_ks, d_ke, c->d_tbits, c->H, c->d_nr, c->d_nk, c->d_l0, c->d_slotsite, e->d_pos,
                e->alpha, e->beta, e->kappa, d_tw_t, d_tw_w, d_tw_ks, d_tw_ke, d_tw_C0, d_tw_R0, d_tw_R1, d_wll, sc.d_wn, sc.d_ws, sc.d_we, sc.d_nwout, d_ownT,
                d_tw_own);
    }
    // The bookkeeping arrays and LIBD2 are final here: they leave for the host now, under the rest of the preparation
    // and the GEMM (score_common copies the bookkeeping on the copy stream once ev_book has fired).  With a page-locked
    // host table the whole device table goes out once — LIBD2 in place, NaN everywhere else — and the GEMM's merge warps
    // then store LIBD0 / LIBD1 of every finished (target, window) into it themselves; the GEMM waits for that copy.
    IBD_CUDA(cudaEventRecord(e->ev_book, e->stream));
    sc.bookkeeping_ready = true;
    double *h_wll_mapped = host_table_alias(sc);
    cudaEvent_t ev_table = nullptr;  // the copy of the whole table is done
    if (h_wll_mapped) {
        cudaEvent_t ev_ready;
        if (range_event(e, 0, &ev_ready) || range_event(e, 1, &ev_table)) return 1;
        IBD_CUDA(cudaEventRecord(ev_ready, e->stream));
        IBD_CUDA(cudaStreamWaitEvent(e->d2h_stream, ev_ready, 0));
        sc.streamed = true;
        IBD_CUDA(cudaMemcpyAsync(sc.w_loglik, d_wll, (size_t)T * outW * 24, cudaMemcpyDeviceToHost, e->d2h_stream));
        IBD_CUDA(cudaEventRecord(ev_table, e->d2h_stream));
    }
    {
        LaunchScope ls(e, K_V_SORT);
        IBD_CUDA(cudaMemsetAsync(d_hist, 0, (size_t)(nKB + 2) * 4, e->stream));
        v_sort_hist_kernel<<<(n_tw + 255) / 256, 256, 0, e->stream>>>(n_tw, d_tw_ks, d_hist);
        v_sort_scan_kernel<<<1, 1024, 0, e->stream>>>(nKB + 1, d_hist);
        IBD_CUDA(cudaMemcpyAsync(d_cursor, d_hist, (size_t)(nKB + 2) * 4, cudaMemcpyDeviceToDevice, e->stream));
        v_sort_scatter_kernel<<<(n_tw + 255) / 256, 256, 0, e->stream>>>(n_tw, d_tw_ks, d_cursor, d_order);
        v_tiles_kernel<<<n_tiles, 64, 0, e->stream>>>(n_tw, n_tiles, d_order, d_tw_ks, d_tw_ke, d_tile_kb0, d_tile_nkb);
    }
    IBD_CUDA(cudaGetLastError());
    std::vector<int32_t> h_nkb((size_t)n_tiles);
    IBD_CUDA(cudaMemcpyAsync(h_nkb.data(), d_tile_nkb, (size_t)n_tiles * 4, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));

    // ---- row tiles in batches under the A budget ---------------------------------------------------
    static const int budget_mb = env_int("IBDGEM_V_BUDGET_MB", 0);  // (tests exercise the row-tile batching with it)
    const size_t a_budget = budget_mb > 0 ? (size_t)budget_mb << 20 : V_A_BUDGET;
    std::vector<int64_t> h_slab((size_t)n_tiles);
    int *d_unit;
    if (scratch(e, SC_MMA_UNIT, 64, (void **)&d_unit)) return 1;
    int u0 = 0;
    // slab offsets restart at every batch; all batches' offsets go up in one copy
    std::vector<std::pair<int, int>> batches;
    std::vector<int64_t> batch_slabs;
    while (u0 < n_tiles) {
        int u1 = u0;
        int64_t slabs = 0;
        while (u1 < n_tiles && (u1 == u0 || (size_t)(slabs + 2 * (int64_t)h_nkb[(size_t)u1]) * A_SLAB <= a_budget)) {
            h_slab[(size_t)u1] = slabs;
            slabs += 2 * (int64_t)h_nkb[(size_t)u1];
            u1++;
        }
        batches.push_back({u0, u1});
        batch_slabs.push_back(slabs);
        u0 = u1;
    }
    IBD_CUDA(cudaMemcpyAsync(d_tile_slab, h_slab.data(), (size_t)n_tiles * 8, cudaMemcpyHostToDevice, e->stream));
    int64_t max_slabs = 0;
    for (auto s : batch_slabs) max_slabs = std::max(max_slabs, s);
    unsigned char *d_A;
    if (scratch(e, SC_MMA_TGT, (size_t)max_slabs * A_SLAB, (void **)&d_A)) return 1;
    for (size_t bi = 0; bi < batches.size(); bi++) {
        const int b0 = batches[bi].first, b1 = batches[bi].second;
        int max_nkb = 1;
        for (int u = b0; u < b1; u++) max_nkb = std::max(max_nkb, h_nkb[(size_t)u]);
        {
            LaunchScope ls(e, K_V_EXPAND_A);
            for (int y0 = 0; y0 < (b1 - b0) * 2; y0 += 65534) {  // tile halves ride on gridDim.y
                const int ny = std::min(65534, (b1 - b0) * 2 - y0);
                v_expand_a_kernel<<<dim3((unsigned)max_nkb, (unsigned)ny), 128, 0, e->stream>>>(
                    b0 + y0 / 2, d_tile_kb0, d_tile_nkb, d_tile_slab, d_order, d_tw_t, d_tw_ks, d_tw_ke, d_targets, c->d_tbits, c->H, c->d_nr,
                    c->d_nk, c->d_slotsite, d_tgt_counts, e->S, v.vflag, d_A);
            }
        }
        IBD_CUDA(cudaGetLastError());
        CUtensorMap mapA;
        if (make_slab_map(&mapA, d_A, BM, batch_slabs[bi])) return 1;
        Params p;
        p.n_units = b1 - b0;
        p.unit0 = b0;
        p.NT = NT; p.nKB = nKB; p.n_tw = n_tw; p.outW = outW;
        p.alpha = e->alpha; p.beta = e->beta; p.kappa = e->kappa;
        p.alpha_f = (float)e->alpha; p.beta_f = (float)e->beta; p.kappa_f = (float)e->kappa;
        p.screen_f = (float)(screen_nats(2 * nU) + 2.0);
        p.tile_kb0 = d_tile_kb0; p.tile_nkb = d_tile_nkb; p.tile_slab = d_tile_slab; p.order = d_order;
        p.tw_t = d_tw_t; p.tw_w = d_tw_w; p.tw_own = d_tw_own; p.tw_C0 = d_tw_C0; p.tw_R0 = d_tw_R0; p.tw_R1 = d_tw_R1;
        p.lnc = d_lnc; p.lognb = d_lognb; p.wll = d_wll;
        p.wll_host = h_wll_mapped;
        IBD_CUDA(cudaMemsetAsync(d_unit, 0, 8, e->stream));
        p.unit_counter = d_unit;
        if (bi == 0) {
            IBD_CUDA(cudaStreamWaitEvent(e->stream, c->ev_join, 0));
            if (h_wll_mapped) IBD_CUDA(cudaStreamWaitEvent(e->stream, ev_table, 0));
        }
        {
            LaunchScope ls(e, K_LD_VMMA);
            if (launch_pairs(ld_vmma_kernel, THREADS, SMEM_BYTES, p.n_units, e->sm_count, e->stream, mapA, mapB, p)) return 1;
        }
        IBD_CUDA(cudaGetLastError());
    }
    return 0;
}

}  // namespace ibdgem
