// ld_mma.cu — tensor-core --LD window scoring (L1 + L2, src/ibdgem.c:673-753) for the common case
// of shared windows (no -v, no -D) and a depth-linear class table.
//
// Algebra (DESIGN.md "tensor path").  With l_g(s) = ln P_s(D|G=g), d1 = l1 - l0 and
// l2 - 2 l1 + l0 = n_s * kappa (kappa = ln 4 eps (1-eps), n_s = pileup depth), two haplotypes x, y
// over a window w give
//     ln prod_s P_s[x_s + y_s] = C0_w + R_w[x] + R_w[y] + kappa * M_w[x, y],
//     C0 = sum l0,   R[x] = sum x_s d1_s,   M[x, y] = sum n_s x_s y_s   (an INTEGER).
// So the 4 pseudo-diploid pairings of every target x background pair (the loop the reference
// spends 78 % of its time in) are one exact int8 GEMM per window, [2T x W] . [W x 2B] -> int32,
// on the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM), and
//     LIBD1_w(t) = C0 + LSE_i ( R[a_i] + LSE_{k not own(t)} ( R'[k] + kappa M[a_i, k] ) ) - ln 4 nB
// is evaluated in the epilogue straight out of TMEM in fp64.  Because M is an integer, the
// epilogue first screens every element with an integer key (round(R'[k]/|kappa|) - M); only
// elements within D = ln(2N) + 16 nats of the running row maximum reach the fp64 exp — the dropped
// mass is below 1e-7 relative.  LIBD0 (the chain over background individuals) and LIBD2 are
// target-independent per individual: Q_w[b] = C0 + R[r0] + R[r1] + kappa M[r0, r1].
//
// d1 is linear in the counts (d1 = n_ref * alpha + n_alt * beta), so R and the M of an individual's own
// two haplotypes are integer dot products of 0/1 bytes with count bytes: the expansion kernels take them
// with dp4a from the bytes they write.
//
// Kernels in this file: ld_compact, ld_c0, ld_transpose (cached per prepared panel); ld_stage,
// ld_expand_bg, ld_expand_tgt, ld_windows, ld_mma, ld_ibd0 (per call).
#include <cuda.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "engine.h"
#include "tc_common.cuh"

namespace ibdgem {

// ---------------------------------------------------------------------------------------------
// cached, target-independent operands
struct LdCache {
    bool valid = false;       // per-site operands (slots, depths, C0) are current
    int tw_upto = 0;          // windows [0, tw_upto) have their transposed bits
    int32_t nW = 0;
    int64_t K = 0;
    int W = 0, Wpad = 0, WP32 = 0, KB = 0;
    int H = 0, N = 0;
    int32_t *d_infsite = nullptr;  // [nW][Wpad] site index of each window slot, -1 = padding
    uint8_t *d_nk = nullptr;       // [nW][Wpad] pileup depth n_s of the slot
    uint8_t *d_nr = nullptr;       // [nW][Wpad] REF-matching bases n_ref of the slot (n_alt = n_s - n_ref)
    double *d_l0 = nullptr;        // [nW][Wpad] l0
    double *d_C0 = nullptr;        // [nW]
    uint32_t *d_tbits = nullptr;   // [nW][H][WP32] haplotype-major window-padded bits
    size_t b_infsite = 0, b_nk = 0, b_nr = 0, b_l0 = 0, b_C0 = 0, b_tbits = 0;
};

constexpr int KEY_PAD = -(1 << 30);   // key of padding / excluded columns
constexpr int KEY_INIT = -(1 << 29);  // initial running maximum
constexpr int MAX_GRID_Y = 65535;  // windows ride on gridDim.y of the transposition and expansion kernels
constexpr size_t LD_OPERAND_BUDGET = (size_t)12 << 30;  // bytes of expanded int8 operands per window batch

// ---------------------------------------------------------------------------------------------
// cached-operand kernels

// one thread per panel line: informative kept sites go to their window slot
__global__ void __launch_bounds__(256)
ld_compact_kernel(int64_t S, const uint8_t *__restrict__ status, const uint32_t *__restrict__ rank,
                  const uint8_t *__restrict__ nref, const uint8_t *__restrict__ nalt,
                  const double *__restrict__ lnP, int C, int W, int Wpad, int32_t *__restrict__ infsite,
                  uint8_t *__restrict__ nk, uint8_t *__restrict__ nr, double *__restrict__ l0) {
    const int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= S || status[s] != 1) return;
    const uint32_t r = rank[s];
    const int64_t slot = (int64_t)(r / (uint32_t)W) * Wpad + (r % (uint32_t)W);
    const int a = nref[s], b = nalt[s];
    infsite[slot] = (int32_t)s;
    nk[slot] = (uint8_t)(a + b);
    nr[slot] = (uint8_t)a;
    l0[slot] = lnP[(size_t)(a * C + b) * 3];
}

// C0_w = sum of l0 over the window, fixed-order tree so the value is reproducible
__global__ void __launch_bounds__(256) ld_c0_kernel(const double *__restrict__ l0, int Wpad, double *__restrict__ C0) {
    __shared__ double sh[256];
    const double *p = l0 + (size_t)blockIdx.x * Wpad;
    double a = 0;
    for (int k = threadIdx.x; k < Wpad; k += 256) a += p[k];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) C0[blockIdx.x] = sh[0];
}

// 32 x 32 bit transpose across a warp: lane i holds row i on entry, column i on exit.  Five
// butterfly exchanges of half-blocks, each one shuffle + one funnel rotate + one bitwise select:
// a lane in the lower half keeps its bits under m and takes the partner's bits under m moved up
// by j (a left rotate puts them there), a lane in the upper half the mirror image.
__device__ __forceinline__ uint32_t transpose32(uint32_t x, int lane) {
#pragma unroll
    for (int k = 0; k < 5; k++) {
        const int j = 16 >> k;
        const uint32_t m = k == 0 ? 0x0000FFFFu : k == 1 ? 0x00FF00FFu : k == 2 ? 0x0F0F0F0Fu : k == 3 ? 0x33333333u : 0x55555555u;
        const bool hi = (lane & j) != 0;
        const uint32_t keep = hi ? ~m : m;
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, j);
        const uint32_t t = __funnelshift_l(y, y, hi ? 32 - j : j);
        x = (x & keep) | (t & ~keep);
    }
    return x;
}

// K_LD_TRANSPOSE: site-major panel bits -> [window][haplotype][32-site words].  Block = (8 word
// columns = 256 haplotypes, one window); warp g transposes the 32 x 32 bit blocks of window slots
// 32g .. 32g+31 in registers; the tile goes through shared memory so the stores are whole rows.
__global__ void __launch_bounds__(1024)
ld_transpose_kernel(int w_off, const uint32_t *__restrict__ bits, int64_t Wh, int H, const int32_t *__restrict__ infsite,
                    int Wpad, int WP32, uint32_t *__restrict__ tbits) {
    __shared__ uint32_t tile[256 * 33];
    // the word-column group is the fastest grid dimension: the blocks that share a window's panel rows
    // run together, so every 32-byte piece of a row is fetched from HBM once
    const int w = w_off + blockIdx.y, j0 = blockIdx.x * 8;
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    if (g < WP32) {
        const int32_t s = infsite[(size_t)w * Wpad + g * 32 + lane];
        const uint32_t *row = bits + (size_t)(s < 0 ? 0 : s) * Wh;
        uint32_t word[8];
        if ((Wh & 3) == 0) {
            // rows are 16-byte aligned: two 16-byte loads per lane (a lane reads its own row, so every
            // load instruction costs 32 L1 wavefronts whatever its width)
            uint4 lo = make_uint4(0u, 0u, 0u, 0u), hi = lo;
            if (s >= 0 && j0 < Wh) lo = __ldg(reinterpret_cast<const uint4 *>(row + j0));
            if (s >= 0 && j0 + 4 < Wh) hi = __ldg(reinterpret_cast<const uint4 *>(row + j0 + 4));
            word[0] = lo.x; word[1] = lo.y; word[2] = lo.z; word[3] = lo.w;
            word[4] = hi.x; word[5] = hi.y; word[6] = hi.z; word[7] = hi.w;
        } else {
#pragma unroll
            for (int jj = 0; jj < 8; jj++) word[jj] = (s >= 0 && j0 + jj < Wh) ? __ldg(row + j0 + jj) : 0u;
        }
#pragma unroll
        for (int jj = 0; jj < 8; jj++) tile[(jj * 32 + lane) * 33 + g] = transpose32(word[jj], lane);
    }
    __syncthreads();
    if (lane < WP32)  // a warp stores one haplotype row of the tile per pass
        for (int hl = g; hl < 256; hl += 32) {
            const int hap = j0 * 32 + hl;
            if (hap < H) tbits[((size_t)w * H + hap) * WP32 + lane] = tile[hl * 33 + lane];
        }
}

// ---------------------------------------------------------------------------------------------
// per-call kernels

// One 32-site word of a haplotype as 0/1 bytes (eight 32-bit lanes of four sites).
__device__ __forceinline__ void spread32(uint32_t x, uint32_t (&e)[8]) {
#pragma unroll
    for (int k = 0; k < 8; k++) e[k] = spread4((x >> (4 * k)) & 15u);
}
// K_LD_STAGE: words from pinned (mapped) host memory to the device
__global__ void __launch_bounds__(256) ld_stage_kernel(uint32_t *__restrict__ dst, const uint32_t *__restrict__ src, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i];
}

// K_LD_EXPAND_BG: one warp per (window, background individual), lane = 32-site word.  Writes the
// individual's two haplotype columns of the GEMM's background operand (0/1 bytes, K-major) and, from
// the same bytes, the integers of the window's marginals by dp4a against the slot counts:
//   A = sum x n_ref, N = sum x n  ->  R[x] = alpha A + beta (N - A)   (l1 - l0 is linear in the counts)
//   M = sum n r0 r1               ->  Q[b] = C0 + R[r0] + R[r1] + kappa M   (the chain of src/ibdgem.c:715)
// and from them the column tables of the call: R'[k] = R[k] + ln(multiplicity), the screening key
// round(R'/|kappa|), Q'[b] = Q[b] + ln(multiplicity).  Individuals nU .. npadU-1 are the padding columns.
__global__ void __launch_bounds__(256)
ld_expand_bg_kernel(int w0, int nU, int npadU, int ncols, int ncolpad, int H, int Wpad, int WP32,
                    const int32_t *__restrict__ bgU, const double *__restrict__ lnc, const uint32_t *__restrict__ tbits,
                    const uint8_t *__restrict__ nr, const uint8_t *__restrict__ nk, const double *__restrict__ C0,
                    double alpha, double beta, double kappa, double inv_abs_kappa, unsigned char *__restrict__ out,
                    int32_t *__restrict__ akey, double *__restrict__ Rp, double *__restrict__ Qp, double *__restrict__ Fp) {
    const int lane = threadIdx.x & 31;
    const int u = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int wl = blockIdx.y, w = w0 + wl;
    if (u >= npadU) return;
    if (u >= nU) {  // padding columns never pass the screen
        if (lane < 2 && 2 * u + lane < ncolpad) {
            akey[(size_t)w * ncolpad + 2 * u + lane] = KEY_PAD;
            Rp[(size_t)w * ncolpad + 2 * u + lane] = -INFINITY;
            Fp[(size_t)w * ncolpad + 2 * u + lane] = 0.0;
        }
        return;
    }
    const int ind = __ldg(bgU + u);
    unsigned A0 = 0, N0 = 0, A1 = 0, N1 = 0, M = 0;
    if (lane < WP32) {
        const uint32_t x0 = __ldg(tbits + ((size_t)w * H + 2 * ind) * WP32 + lane);
        const uint32_t x1 = __ldg(tbits + ((size_t)w * H + 2 * ind + 1) * WP32 + lane);
        const uint4 *cr = reinterpret_cast<const uint4 *>(nr + (size_t)w * Wpad + lane * 32);
        const uint4 *cn = reinterpret_cast<const uint4 *>(nk + (size_t)w * Wpad + lane * 32);
        const uint4 r0 = __ldg(cr), r1 = __ldg(cr + 1), n0 = __ldg(cn), n1 = __ldg(cn + 1);
        const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
        const uint32_t nn[8] = {n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, n1.z, n1.w};
        uint32_t e0[8], e1[8];
        spread32(x0, e0);
        spread32(x1, e1);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            A0 = __dp4a(e0[k], rr[k], A0);
            N0 = __dp4a(e0[k], nn[k], N0);
            A1 = __dp4a(e1[k], rr[k], A1);
            N1 = __dp4a(e1[k], nn[k], N1);
            M = __dp4a(e0[k] & e1[k], nn[k], M);
        }
        uint4 *o0 = reinterpret_cast<uint4 *>(out + ((size_t)wl * ncols + 2 * u) * Wpad) + lane * 2;
        uint4 *o1 = reinterpret_cast<uint4 *>(out + ((size_t)wl * ncols + 2 * u + 1) * Wpad) + lane * 2;
        __stcs(o0, make_uint4(e0[0], e0[1], e0[2], e0[3]));
        __stcs(o0 + 1, make_uint4(e0[4], e0[5], e0[6], e0[7]));
        __stcs(o1, make_uint4(e1[0], e1[1], e1[2], e1[3]));
        __stcs(o1 + 1, make_uint4(e1[4], e1[5], e1[6], e1[7]));
    }
    A0 = warp_sum(A0); N0 = warp_sum(N0); A1 = warp_sum(A1); N1 = warp_sum(N1); M = warp_sum(M);
    if (lane == 0) {
        const double R0 = fma(alpha, (double)A0, beta * (double)(N0 - A0));  // N - A = sum x n_alt >= 0
        const double R1 = fma(alpha, (double)A1, beta * (double)(N1 - A1));
        const double lc = lnc[u];
        const double p0 = R0 + lc, p1 = R1 + lc;
        Rp[(size_t)w * ncolpad + 2 * u] = p0;
        Rp[(size_t)w * ncolpad + 2 * u + 1] = p1;
        const double k0 = rint(p0 * inv_abs_kappa), k1 = rint(p1 * inv_abs_kappa);
        akey[(size_t)w * ncolpad + 2 * u] = (int32_t)k0;
        akey[(size_t)w * ncolpad + 2 * u + 1] = (int32_t)k1;
        // exp(R' - key |kappa|), the argument within |kappa| / 2 of zero (-inf -> 0 for a column of multiplicity 0)
        Fp[(size_t)w * ncolpad + 2 * u] = p0 == -INFINITY ? 0.0 : exp(fma(k0, kappa, p0));
        Fp[(size_t)w * ncolpad + 2 * u + 1] = p1 == -INFINITY ? 0.0 : exp(fma(k1, kappa, p1));
        Qp[(size_t)w * nU + u] = (((C0[w] + R0) + R1) + kappa * (double)M) + lc;
    }
}

// K_LD_EXPAND_TGT: one warp per (window, target).  Writes the target's two haplotype rows of the
// GEMM's target operand (n_s x_s bytes, K-major; skipped when out == nullptr), R of both rows for the
// merge step, and LIBD2_w(t) = Q_w[t] (the non-LD product of src/ibdgem.c:667, 752 in log space).
__global__ void __launch_bounds__(256)
ld_expand_tgt_kernel(int w0, int T, int H, int Wpad, int WP32, int outW, const int32_t *__restrict__ targets,
                     const uint32_t *__restrict__ tbits, const uint8_t *__restrict__ nr, const uint8_t *__restrict__ nk,
                     const double *__restrict__ C0, double alpha, double beta, double kappa,
                     unsigned char *__restrict__ out, double *__restrict__ Rt, double *__restrict__ wll) {
    const int lane = threadIdx.x & 31;
    const int t = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int wl = blockIdx.y, w = w0 + wl;
    if (t >= T) return;
    const int ind = __ldg(targets + t);
    unsigned A0 = 0, N0 = 0, A1 = 0, N1 = 0, M = 0;
    if (lane < WP32) {
        const uint32_t x0 = __ldg(tbits + ((size_t)w * H + 2 * ind) * WP32 + lane);
        const uint32_t x1 = __ldg(tbits + ((size_t)w * H + 2 * ind + 1) * WP32 + lane);
        const uint4 *cr = reinterpret_cast<const uint4 *>(nr + (size_t)w * Wpad + lane * 32);
        const uint4 *cn = reinterpret_cast<const uint4 *>(nk + (size_t)w * Wpad + lane * 32);
        const uint4 r0 = __ldg(cr), r1 = __ldg(cr + 1), n0 = __ldg(cn), n1 = __ldg(cn + 1);
        const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
        const uint32_t nn[8] = {n0.x, n0.y, n0.z, n0.w, n1.x, n1.y, n1.z, n1.w};
        uint32_t e0[8], e1[8];
        spread32(x0, e0);
        spread32(x1, e1);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            A0 = __dp4a(e0[k], rr[k], A0);
            N0 = __dp4a(e0[k], nn[k], N0);
            A1 = __dp4a(e1[k], rr[k], A1);
            N1 = __dp4a(e1[k], nn[k], N1);
            M = __dp4a(e0[k] & e1[k], nn[k], M);
        }
        if (out) {
#pragma unroll
            for (int k = 0; k < 8; k++) {  // n_s where the allele is 1
                e0[k] = (e0[k] * 0xFFu) & nn[k];
                e1[k] = (e1[k] * 0xFFu) & nn[k];
            }
            uint4 *o0 = reinterpret_cast<uint4 *>(out + ((size_t)wl * 2 * T + 2 * t) * Wpad) + lane * 2;
            uint4 *o1 = reinterpret_cast<uint4 *>(out + ((size_t)wl * 2 * T + 2 * t + 1) * Wpad) + lane * 2;
            __stcs(o0, make_uint4(e0[0], e0[1], e0[2], e0[3]));
            __stcs(o0 + 1, make_uint4(e0[4], e0[5], e0[6], e0[7]));
            __stcs(o1, make_uint4(e1[0], e1[1], e1[2], e1[3]));
            __stcs(o1 + 1, make_uint4(e1[4], e1[5], e1[6], e1[7]));
        }
    }
    A0 = warp_sum(A0); N0 = warp_sum(N0); A1 = warp_sum(A1); N1 = warp_sum(N1); M = warp_sum(M);
    if (lane == 0) {
        const double R0 = fma(alpha, (double)A0, beta * (double)(N0 - A0));  // N - A = sum x n_alt >= 0
        const double R1 = fma(alpha, (double)A1, beta * (double)(N1 - A1));
        Rt[((size_t)w * T + t) * 2] = R0;
        Rt[((size_t)w * T + t) * 2 + 1] = R1;
        wll[((size_t)t * outW + w) * 3 + 2] = ((C0[w] + R0) + R1) + kappa * (double)M;
    }
}

// Columns [w_lo, w_lo + ncols) of the score table [T][outW][3] stored straight into the caller's page-locked host
// buffer (same layout) over PCIe: a strided copy of T short rows costs the copy engine one descriptor per row
// (10,000 rows of 3 KB at C5 over 8 GPUs: 2.4 ms for 30 MB); coalesced stores from a kernel run at link speed.
__global__ void __launch_bounds__(256)
ld_store_cols_kernel(const double *__restrict__ src, double *__restrict__ dst, int T, int outW, int w_lo, int ncols) {
    const int64_t per = (int64_t)ncols * 3;
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * per) return;
    const int64_t t = i / per, c = i % per;
    const int64_t o = (t * outW + w_lo) * 3 + c;
    dst[o] = src[o];
}

// the same columns packed WINDOW-major into a compact table [ncols][T][3] (window shards with a compact host table:
// any sub-range of the shard's windows is then one contiguous block)
__global__ void __launch_bounds__(256)
ld_pack_cols_kernel(const double *__restrict__ src, double *__restrict__ dst, int T, int outW, int w_lo, int ncols) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * ncols * 3) return;
    const int64_t c = i % 3, t = (i / 3) % T, w = i / ((int64_t)3 * T);
    dst[i] = src[(t * outW + w_lo + w) * 3 + c];
}

// window bookkeeping (W2) for every (target, window)
__global__ void __launch_bounds__(256)
ld_windows_kernel(int w_lo, int w_hi, int T, int nW, int outW, int W, int64_t K, const int64_t *__restrict__ wfirst,
                  const int64_t *__restrict__ wlast, const uint64_t *__restrict__ pos, int32_t *__restrict__ wn,
                  uint64_t *__restrict__ ws, uint64_t *__restrict__ we, int32_t *__restrict__ nwout) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int span = w_hi - w_lo;
    if (j >= (int64_t)T * span) return;
    const int t = (int)(j / span), w = w_lo + (int)(j % span);
    const int64_t i = (int64_t)t * outW + w;
    if (w == w_lo) nwout[t] = nW;
    if (w >= nW) return;
    const int64_t left = K - (int64_t)w * W;
    wn[i] = (int32_t)(left < W ? left : W);
    ws[i] = pos[wfirst[w]];
    we[i] = pos[wlast[w]];
}

// LIBD0: log-mean-exp of Q'_w over the background without the target's own entry.  One block per
// window; 64 chunk partials so that re-summing without a dominating own entry scans one chunk only.
constexpr int IBD0_CHUNKS = 64;
__global__ void __launch_bounds__(256, 4)  // latency-bound: several windows per SM, not one
ld_ibd0_kernel(int w_off, int T, int nU, int outW, const double *__restrict__ Qp, const int32_t *__restrict__ ownU,
               const double *__restrict__ lognb, double *__restrict__ wll, int stage) {
    extern __shared__ double qs[];
    __shared__ double cm[IBD0_CHUNKS], cs[IBD0_CHUNKS];
    __shared__ double tot_m, tot_s;
    const int w = w_off + blockIdx.x;
    const double *q = Qp + (size_t)w * nU;
    if (stage) {
        for (int u = threadIdx.x; u < nU; u += blockDim.x) qs[u] = __ldg(q + u);
        __syncthreads();
        q = qs;
    }
    const int clen = (nU + IBD0_CHUNKS - 1) / IBD0_CHUNKS;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int c = wid; c < IBD0_CHUNKS; c += 8) {
        const int u0 = c * clen, u1 = min(nU, u0 + clen);
        double m = -INFINITY;
        for (int u = u0 + lane; u < u1; u += 32) m = fmax(m, q[u]);
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        double s = 0;
        if (m > -INFINITY)
            for (int u = u0 + lane; u < u1; u += 32) s += exp_nonpos(q[u] - m);
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) { cm[c] = m; cs[c] = s; }
    }
    __syncthreads();
    if (wid == 0) {  // combine the chunk partials across the lanes of one warp
        double m = fmax(cm[lane], cm[lane + 32]);
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        double s = 0;
        if (cs[lane] > 0) s += cs[lane] * exp_nonpos(cm[lane] - m);
        if (cs[lane + 32] > 0) s += cs[lane + 32] * exp_nonpos(cm[lane + 32] - m);
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) { tot_m = m; tot_s = s; }
    }
    __syncthreads();
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const double lnb = lognb[t];
        double r;
        if (!(lnb == lnb)) {
            r = nan;  // n_refpanel = 0: 0/0 in the reference
        } else {
            const int own = ownU[t];
            double x = 0;
            if (own >= 0 && q[own] >= tot_m - 60.0) x = exp_nonpos(q[own] - tot_m);
            if (x + x <= tot_s) {
                // own term at most half of the mass: tot_s - x loses at most one bit.  A dominating own
                // term (the target is the pileup's source) would cancel, so it is left out by re-summing.
                r = tot_m + log(tot_s - x) - lnb;
            } else {
                const int oc = own / clen;
                double m = -INFINITY;
                for (int c = 0; c < IBD0_CHUNKS; c++)
                    if (c != oc) m = fmax(m, cm[c]);
                const int u0 = oc * clen, u1 = min(nU, u0 + clen);
                for (int u = u0; u < u1; u++)
                    if (u != own) m = fmax(m, q[u]);
                double s = 0;
                for (int c = 0; c < IBD0_CHUNKS; c++)
                    if (c != oc && cs[c] > 0) s += cs[c] * exp_nonpos(cm[c] - m);
                for (int u = u0; u < u1; u++)
                    if (u != own) s += exp_nonpos(q[u] - m);
                r = m + log(s) - lnb;
            }
        }
        wll[((size_t)t * outW + w) * 3 + 0] = r;
    }
}

// ---------------------------------------------------------------------------------------------
// K_LD_MMA: persistent, warp-specialised window GEMM with the fused log-sum-exp epilogue.
//   unit = (window w, block of 128 target haplotypes); the unit's A tile (128 rows x Wpad bytes)
//   stays resident in shared memory while the background tiles (128 columns x 128 bytes per
//   stage) stream through a TMA ring; accumulators (128 x 128 int32) rotate through 4 TMEM
//   slots; two sets of 4 epilogue warps alternate tiles, each thread owning one target
//   haplotype row, so the reduction over background columns needs no cross-thread traffic.
namespace mma {
using namespace tcx;
constexpr int BM = 128, BN = 128, KBYTES = 128, UK = 32;
constexpr int MAXKB = 8;              // Wpad <= 1024
constexpr int A_SLAB = BM * KBYTES;   // 16 KB
constexpr int B_SLAB = BN * KBYTES;   // 16 KB
constexpr int EPI_WARP0 = 4;
constexpr int NSETS = 4;              // epilogue warp sets of 4 warps (one warp per TMEM lane quarter)
constexpr int ETAB_N = 512;           // entries of the exp(|kappa| d) table in shared memory
// Units are handed out dynamically (an atomic counter): CTA pairs differ by ~15 % in speed (the two
// dies), and pairs that pick up neighbouring units — the row blocks of one window — stream the same
// background tiles at the same time, which is what lets L2 serve them.  The number travels to every
// role of both CTAs through a ring in shared memory.  No "empty" barriers: the producer is at most one
// unit ahead of the MMA issuer (operand rings), which is at most two tiles ahead of the epilogue
// (accumulator slots), which is at most one unit ahead of the merge warps (bar 2) — 3 < URING.

// CTA pairs (tcgen05 cta_group::2) on 256 x 256 tiles: each CTA keeps its own 128 target rows resident and streams
// HALF of every background tile, which halves the shared-memory traffic per MMA — the resource ncu showed saturated
// with single-CTA 128 x 128 tiles.
constexpr int CG = 2;                           // CTAs per MMA
constexpr int NSTAGE = 5;                       // background stages
constexpr int TILE_N = BN * CG;                 // accumulator tile columns
constexpr int NACC = 512 / TILE_N;              // TMEM accumulator slots
constexpr int SETCOLS = TILE_N / NSETS;         // accumulator columns per epilogue set
constexpr int THREADS = 128 + NSETS * 128;
constexpr int OFF_A = 0;
constexpr int OFF_B = OFF_A + MAXKB * A_SLAB;
constexpr int OFF_KEYS = OFF_B + NSTAGE * B_SLAB;             // per epilogue warp: 128 int32
constexpr int OFF_MERGE = OFF_KEYS + NSETS * 4 * SETCOLS * 4;  // NSETS x 128 x double2: the sets' (max, sum) per row
constexpr int OFF_KMAX = OFF_MERGE + NSETS * BM * 16;          // 2 x 128 int32, shared by the sets
constexpr int OFF_BAR = OFF_KMAX + 2 * BM * 4;
constexpr int NBAR = 2 * MAXKB + 2 * NSTAGE + 2 * NACC + URING;
constexpr int OFF_TMEM = OFF_BAR + NBAR * 8;
constexpr int OFF_URING = OFF_TMEM + 16;                      // URING unit numbers handed out by the scheduler
constexpr int OFF_ETAB = OFF_URING + URING * 4;               // ETAB_N doubles: exp(|kappa| d) over the screen's reach
constexpr int SMEM_BYTES = OFF_ETAB + ETAB_N * 8 + 1024;      // + alignment slack
constexpr uint32_t IDESC = (2u << 4) /* D = s32 */ | (0u << 7) /* A = u8 */ | (0u << 10) /* B = u8 */ |
                           ((uint32_t)(TILE_N >> 3) << 17) | ((uint32_t)((BM * CG) >> 4) << 24);
static_assert(SMEM_BYTES <= 232448, "over the 227 KB shared memory limit");
static_assert(SETCOLS % 32 == 0 && SETCOLS <= BN, "epilogue sets split the tile into 32-column chunks");

struct Params {
    int w0;                  // first window of this batch (operands hold windows w0 .. w0 + nW - 1)
    int nW, MB, NT, KB;      // windows, row blocks (of 128 * CG) per window, column tiles (of 128 * CG), 128-byte k blocks
    int n_units;
    int nrows, ncolpad;      // 2T, padded column count of the key tables
    int H, outW;
    int delta;               // screening distance in key units
    double kappa;
    const int32_t *akey;     // [nW][ncolpad]
    const double *Rp;        // [nW][ncolpad]
    const double *Fp;        // [nW][ncolpad] exp(R' - key |kappa|): the part of a term the integer key does not carry
    int tab_n, dpos;         // table mode (tab_n > 0): entries delta + dpos + 1 of exp(|kappa| (i - delta)); a row's
                             // reference key may trail its running maximum by up to dpos
    const double *Rt;        // [nW][nrows] R_w of each target row
    const int32_t *row_own;  // [nrows] first excluded column of the row, or -1
    const double *C0;        // [nW]
    const double *lognb4;    // [T] ln(4 n_refpanel) or NaN
    double *wll;             // [T][outW][3]
    double *wll_host;        // the same table in the caller's page-locked host memory (device alias), or nullptr
    int *unit_counter;       // next unit to hand out (zeroed before the launch)
};

__global__ void __launch_bounds__(THREADS, 1)
ld_mma_kernel(const __grid_constant__ CUtensorMap tmapA, const __grid_constant__ CUtensorMap tmapB, const Params p) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + OFF_BAR);
    // the resident target tile has one (full, empty) pair per 128-byte k-block: the next unit's
    // k-block is fetched as soon as the last tile of this unit has consumed it
    uint64_t *a_full = bars, *a_empty = bars + MAXKB;
    uint64_t *b_full = bars + 2 * MAXKB, *b_empty = b_full + NSTAGE;
    uint64_t *acc_full = b_empty + NSTAGE, *acc_empty = acc_full + NACC;
    uint64_t *ufull = acc_empty + NACC;
    int *uring = reinterpret_cast<int *>(smem + OFF_URING);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + OFF_TMEM);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t rank;  // CTA rank in the pair; rank 0 issues the MMAs
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmapB) : "memory");
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < MAXKB; i++) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 1); }
        for (int i = 0; i < URING; i++) mbar_init(ufull + i, 1);
        for (int i = 0; i < NSTAGE; i++) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 1); }
        for (int i = 0; i < NACC; i++) { mbar_init(acc_full + i, 1); mbar_init(acc_empty + i, 4 * NSETS * CG); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 3)
        for (int i = lane; i < 2 * BM; i += 32) reinterpret_cast<int *>(smem + OFF_KMAX)[i] = KEY_INIT;
    for (int i = threadIdx.x; i < p.tab_n; i += THREADS)
        reinterpret_cast<double *>(smem + OFF_ETAB)[i] = exp(-p.kappa * (double)(i - p.delta));
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // peer barriers are initialised before anyone signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < EPI_WARP0) {
    if (warp == 0) {
        // ===== TMA producer (both CTAs of a pair: own A rows, own half of every background tile) =====
        if (lane == 0) {
            int st = 0;
            uint32_t ph = 0;
            int u_next = -1;
            auto fetch_unit = [&]() {
                const int v = atomicAdd(p.unit_counter, 1);
                return v < p.n_units ? v : -1;
            };
            // scheduler: CTA 0 of the pair draws the unit numbers for every role of both CTAs.  The atomic
            // for the unit after next is issued at the START of a unit and its result is first touched
            // when the unit's loads are all out — a global round trip in front of a unit's first load
            // showed up as a ~7,000-cycle bubble per unit in the device trace.
            int pending = -1;
            if (rank == 0) {
                u_next = fetch_unit();
                unit_publish(uring, ufull, 0, u_next);
                pending = atomicAdd(p.unit_counter, 1);
            }
            for (int it = 0;; it++) {
                int u;
                if (rank == 0) {
                    u = u_next;
                    if (u < 0) break;
                } else {
                    u = unit_of(uring, ufull, it);
                    if (u < 0) break;
                }
                const int w = u / p.MB, mb = u % p.MB;
                auto load_a = [&](int kb) {
                    mbar_wait(a_empty + kb, (uint32_t)((it & 1) ^ 1));
                    if (rank == 0) mbar_expect_tx(a_full + kb, (uint32_t)(CG * A_SLAB));
                    tma_load_3d_cg(smem + OFF_A + kb * A_SLAB, &tmapA, a_full + kb, kb * KBYTES, (mb * CG + (int)rank) * BM, w);
                };
                for (int n = 0; n < p.NT; n++)
                    for (int kb = 0; kb < p.KB; kb++) {
                        // the unit's target k-blocks are interleaved with its first background tile, in
                        // the order the MMA issuer needs them
                        if (n == 0) load_a(kb);
                        if (n + PF_TILES < p.NT)  // pull the same k-block of a later tile into L2
                            tma_prefetch_3d(&tmapB, kb * KBYTES, ((n + PF_TILES) * CG + (int)rank) * BN, w);
                        mbar_wait(b_empty + st, ph ^ 1u);
                        if (rank == 0) mbar_expect_tx(b_full + st, (uint32_t)(CG * B_SLAB));
                        tma_load_3d_cg(smem + OFF_B + st * B_SLAB, &tmapB, b_full + st, kb * KBYTES,
                                           (n * CG + (int)rank) * BN, w);
                        if (++st == NSTAGE) { st = 0; ph ^= 1u; }
                    }
                if (rank == 0) {
                    u_next = pending < p.n_units ? pending : -1;
                    unit_publish(uring, ufull, it + 1, u_next);
                    if (u_next >= 0) pending = atomicAdd(p.unit_counter, 1);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (CTA 0 of the pair): the whole warp walks the loop convergently so every
        // operand stays in uniform registers; one elected lane issues the tcgen05 instructions =====
        if (rank == 0) {
            int st = 0;
            uint32_t ph = 0;
            int it = 0;
            uint32_t g = 0;  // accumulator tile counter
            const uint64_t adesc0 = umma_desc_sw128(smem_u32(smem + OFF_A));
            const uint64_t bdesc0 = umma_desc_sw128(smem_u32(smem + OFF_B));
            for (;; it++) {
                const int u_cur = unit_of(uring, ufull, it);
                if (u_cur < 0) break;
                for (int n = 0; n < p.NT; n++, g++) {
                    const bool first = n == 0, last = n == p.NT - 1;
                    const uint32_t acc = g % NACC, use = g / NACC;
                    mbar_wait(acc_empty + acc, (use & 1u) ^ 1u);
                    const uint32_t d_tmem = tmem_base + acc * TILE_N;
                    // two k-blocks per trip: both barrier probes are in flight together
                    for (int kb = 0; kb < p.KB; kb += 2) {
                        const bool two = kb + 1 < p.KB;
                        int st2 = st + 1;
                        uint32_t ph2 = ph;
                        if (st2 == NSTAGE) { st2 = 0; ph2 ^= 1u; }
                        const bool r1 = mbar_test(b_full + st, ph);
                        const bool r2 = two ? mbar_test(b_full + st2, ph2) : true;
                        if (!r1) mbar_wait(b_full + st, ph);
                        if (!r2) mbar_wait(b_full + st2, ph2);
                        if (first) {  // the unit's target k-blocks arrive one by one
                            mbar_wait(a_full + kb, (uint32_t)(it & 1));
                            if (two) mbar_wait(a_full + kb + 1, (uint32_t)(it & 1));
                        }
                        tc_fence_after();
                        if (elect_one()) {
                            const uint64_t ad = adesc0 + (uint64_t)((kb * A_SLAB) >> 4);
                            const uint64_t bd = bdesc0 + (uint64_t)((st * B_SLAB) >> 4);
#pragma unroll
                            for (int k = 0; k < KBYTES / UK; k++)
                                umma_i8_cg(d_tmem, ad + (uint64_t)(k * (UK >> 4)), bd + (uint64_t)(k * (UK >> 4)), IDESC,
                                           (uint32_t)((kb | k) != 0));
                            tc_commit_cg(b_empty + st);
                            if (last) tc_commit_cg(a_empty + kb);
                            if (two) {
                                const uint64_t ad2 = ad + (uint64_t)(A_SLAB >> 4);
                                const uint64_t bd2 = bdesc0 + (uint64_t)((st2 * B_SLAB) >> 4);
#pragma unroll
                                for (int k = 0; k < KBYTES / UK; k++)
                                    umma_i8_cg(d_tmem, ad2 + (uint64_t)(k * (UK >> 4)), bd2 + (uint64_t)(k * (UK >> 4)), IDESC, 1u);
                                tc_commit_cg(b_empty + st2);
                                if (last) tc_commit_cg(a_empty + kb + 1);
                            }
                            if (kb + 2 >= p.KB) tc_commit_cg(acc_full + acc);
                        }
                        __syncwarp();
                        if (two) { st = st2; ph = ph2; }
                        if (++st == NSTAGE) { st = 0; ph ^= 1u; }
                    }
                }
            }
        }
    } else {
        // ===== merge warps (2, 3): at the end of every unit the four epilogue sets leave their partial
        // (max, scaled sum) per row in shared memory and move on; these two warps join them, add the
        // rows' own terms and write LIBD1.  One thread per target (both haplotype rows), so the fp64
        // exp / log chains (~8k cycles per unit) are off the accumulator hand-back path. =====
        const double2 *mb_buf = reinterpret_cast<const double2 *>(smem + OFF_MERGE);
        const int r0 = (warp - 2) * 64 + lane * 2;  // first of the target's two rows within the CTA's 128
        asm volatile("bar.arrive 2, %0;" ::"n"(NSETS * 128 + 64) : "memory");  // buffer free for unit 0
        for (int it = 0;; it++) {
            const int u = unit_of(uring, ufull, it);
            if (u < 0) break;
            const int w = p.w0 + u / p.MB, mb = u % p.MB;
            const int row = (mb * CG + (int)rank) * BM + r0;
            const bool ok = row < p.nrows;  // nrows is even: both rows or neither
            double rw0 = 0.0, rw1 = 0.0, lnb = 0.0;
            if (ok) {
                rw0 = __ldg(p.Rt + (size_t)w * p.nrows + row);
                rw1 = __ldg(p.Rt + (size_t)w * p.nrows + row + 1);
                lnb = __ldg(p.lognb4 + (row >> 1));
            }
            const double c0w = __ldg(p.C0 + w);
            asm volatile("bar.sync 1, %0;" ::"n"(NSETS * 128 + 64) : "memory");  // the sets' partials are in place
            double A[2], S[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                double2 o[NSETS];
#pragma unroll
                for (int q = 0; q < NSETS; q++) o[q] = mb_buf[q * BM + r0 + h];
                double M2 = o[0].x;
#pragma unroll
                for (int q = 1; q < NSETS; q++) M2 = fmax(M2, o[q].x);
                double S2 = 0.0;
#pragma unroll
                for (int q = 0; q < NSETS; q++) S2 = fma(o[q].y, exp_nonpos(o[q].x - M2), S2);
                S[h] = S2;
                A[h] = (S2 > 0.0) ? M2 + (h ? rw1 : rw0) : -INFINITY;
            }
            asm volatile("bar.arrive 2, %0;" ::"n"(NSETS * 128 + 64) : "memory");  // partials consumed
            // a row is A + ln S; the two haplotypes of the target are joined under one logarithm
            const double mm = fmax(A[0], A[1]);
            double r = mm + log(fma(S[0], exp_nonpos(A[0] - mm), S[1] * exp_nonpos(A[1] - mm)));
            if (mm == -INFINITY) r = -INFINITY;
            r = (c0w + r) - lnb;
            if (!(lnb == lnb)) r = __longlong_as_double(0x7ff8000000000000LL);  // n_refpanel = 0: 0/0 in the reference
            if (ok) {
                double *o = p.wll + ((size_t)(row >> 1) * p.outW + w) * 3;
                o[1] = r;
                if (p.wll_host) {
                    // LIBD0 (ld_ibd0) and LIBD2 (ld_expand_tgt) of this cell were written before the launch: the finished
                    // triple goes straight to the caller's page-locked buffer over PCIe, so no result copy is left
                    // when the GEMM ends (24 MB at C3: 0.44 ms of tail)
                    double *h = p.wll_host + ((size_t)(row >> 1) * p.outW + w) * 3;
                    const double l0 = o[0], l2 = o[2];
                    h[0] = l0;
                    h[1] = r;
                    h[2] = l2;
                }
            }
        }
    }
    } else {
        // ===== epilogue: TMEM -> integer screen -> fp64 log-sum-exp =====
        // every set works on every tile: set q owns columns [q * SETCOLS, (q + 1) * SETCOLS) of the
        // accumulator, so all four epilogue warps of a scheduler drain the slot together and the
        // slot is handed back to the MMA issuer in half the time; each thread owns one target row
        const int ew = warp - EPI_WARP0, set = ew >> 2, quarter = warp & 3;
        const int rloc = quarter * 32 + lane;
        int *skeys = reinterpret_cast<int *>(smem + OFF_KEYS) + ew * SETCOLS;
        double2 *merge = reinterpret_cast<double2 *>(smem + OFF_MERGE);
        int *skmax_all = reinterpret_cast<int *>(smem + OFF_KMAX);
        uint32_t g0 = 0;  // tile counter at the start of the unit
        int it = 0;
        for (;; it++, g0 += (uint32_t)p.NT) {
            const int u = unit_of(uring, ufull, it);
            if (u < 0) break;
            const int w = p.w0 + u / p.MB, mb = u % p.MB;
            const int row = (mb * CG + (int)rank) * BM + rloc;
            const bool row_ok = row < p.nrows;
            const int own0 = row_ok ? p.row_own[row] : -1;
            const int32_t *akw = p.akey + (size_t)w * p.ncolpad;
            // Table mode.  A term is exp(kappa M + R') = exp(|kappa| (key - M)) * F with F = exp(R' - key |kappa|): relative
            // to a per-row reference key the first factor is a table entry and the term one fp64 FMA — no exp on the
            // candidate path, which is what rows with many near-maximal columns (a pileup whose source is not in the
            // background) spend their time on.  The row's partial is (|kappa| vref, s).
            const bool tab = p.tab_n > 0;
            const double *etab = reinterpret_cast<const double *>(smem + OFF_ETAB);
            const double *rpw = (tab ? p.Fp : p.Rp) + (size_t)w * p.ncolpad;
            int vref = KEY_INIT;
            int kmax = row_ok ? KEY_INIT : (1 << 30);  // padding rows never reach the fp64 path
            // the sets see disjoint columns: they share the row's running maximum key through shared
            // memory (monotone, so a stale read only lets more elements through the screen)
            int *skmax = skmax_all + (it & 1) * BM + rloc;
            double m = -INFINITY, s = 0.0;
            // screening keys and R'[k] of the NEXT tile are fetched while the current one is processed,
            // so no global-load latency sits between acc_full and the hand-back of the slot
            constexpr int NCH = SETCOLS / 32;
            int4 kv_next = make_int4(0, 0, 0, 0);
            double rp_next[NCH];
            auto fetch = [&](int n) {
                const int col = n * TILE_N + set * SETCOLS;
                if (lane < SETCOLS / 4) kv_next = __ldg(reinterpret_cast<const int4 *>(akw + col) + lane);
#pragma unroll
                for (int c = 0; c < NCH; c++) rp_next[c] = __ldg(rpw + col + c * 32 + lane);
            };
            fetch(0);
            for (int n = 0; n < p.NT; n++) {
                const uint32_t g = g0 + (uint32_t)n;
                const int slot = (int)(g % NACC);
                const uint32_t use = g / NACC;
                const int col0 = n * TILE_N + set * SETCOLS;  // first column this warp handles
                double rp_cur[NCH];  // lane l holds R' of column col0 + 32 c + l
#pragma unroll
                for (int c = 0; c < NCH; c++) rp_cur[c] = rp_next[c];
                __syncwarp();
                if (lane < SETCOLS / 4) reinterpret_cast<int4 *>(skeys)[lane] = kv_next;
                __syncwarp();
                if (n + 1 < p.NT) fetch(n + 1);
                // does any row of this warp exclude a column of this tile?
                const bool own_here = own0 >= col0 && own0 < col0 + SETCOLS;
                const bool any_own = __any_sync(0xffffffffu, own_here);
                kmax = max(kmax, *skmax);
                mbar_wait_relaxed(acc_full + slot, use & 1u);
                tc_fence_after();
                const uint32_t taddr = tmem_base + slot * TILE_N + set * SETCOLS + ((uint32_t)(quarter * 32) << 16);
                // chunk c of this warp's columns: v[j] = key[j] - M[row, j], returns the chunk maximum
                auto load_chunk = [&](int c, int (&v)[32]) -> int {
                    __syncwarp();
                    tmem_ld32(taddr + c * 32, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const int4 a4 = *reinterpret_cast<const int4 *>(skeys + c * 32 + j);
                        v[j] = a4.x - v[j];
                        v[j + 1] = a4.y - v[j + 1];
                        v[j + 2] = a4.z - v[j + 2];
                        v[j + 3] = a4.w - v[j + 3];
                    }
                    if (any_own) {
                        const int jo = own0 - (col0 + c * 32);  // own columns jo, jo+1 (jo even)
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if ((j & ~1) == jo) v[j] = KEY_PAD;
                    }
                    // 3-input max, four independent chains
                    int c0 = __vimax3_s32(v[0], v[1], v[2]), c1 = __vimax3_s32(v[8], v[9], v[10]);
                    int c2 = __vimax3_s32(v[16], v[17], v[18]), c3 = __vimax3_s32(v[24], v[25], v[26]);
                    c0 = __vimax3_s32(c0, v[3], v[4]); c1 = __vimax3_s32(c1, v[11], v[12]);
                    c2 = __vimax3_s32(c2, v[19], v[20]); c3 = __vimax3_s32(c3, v[27], v[28]);
                    c0 = __vimax3_s32(c0, v[5], v[6]); c1 = __vimax3_s32(c1, v[13], v[14]);
                    c2 = __vimax3_s32(c2, v[21], v[22]); c3 = __vimax3_s32(c3, v[29], v[30]);
                    c0 = __vimax3_s32(c0, v[7], c1); c2 = __vimax3_s32(c2, v[15], c3);
                    return __vimax3_s32(c0, c2, max(v[23], v[31]));
                };
                if (n == 0) {
                    // The screen is relative to the RUNNING row maximum, which starts at -inf: without
                    // help the first tile of a unit sends nearly every element down the fp64 path
                    // (measured: ~40k cycles per unit, 1/3 of the kernel).  So the first tile is read
                    // twice: once for the maximum over all its 256 columns (shared by the four sets
                    // through skmax), then screened against that.
                    int tm = KEY_PAD;
#pragma unroll
                    for (int c = 0; c < NCH; c++) {
                        int v[32];
                        tm = max(tm, load_chunk(c, v));
                    }
                    if (tm > kmax) {
                        kmax = tm;
                        if (row_ok) atomicMax(skmax, tm);
                    }
                    asm volatile("bar.sync 3, %0;" ::"n"(NSETS * 128) : "memory");
                    kmax = max(kmax, *skmax);
                }
#pragma unroll
                for (int c = 0; c < NCH; c++) {
                    int v[32];
                    const int cm = load_chunk(c, v);
                    if (cm > kmax) {
                        kmax = cm;
                        if (row_ok) atomicMax(skmax, cm);
                    }
                    const int thr = kmax - p.delta;
                    if (tab && row_ok && cm > vref + p.dpos) {
                        // rare: the row's first chunk, or a maximum far above the reference: move the reference
                        s *= exp(p.kappa * (double)(kmax - vref));  // (kmax >= cm here; 0 stays 0)
                        vref = kmax;
                    }
                    // an element passes the screen only if the chunk maximum does: the per-element
                    // mask is built only when some row of the warp has a candidate in this chunk
                    uint32_t mask = 0;
                    if (__any_sync(0xffffffffu, cm > thr)) {
#pragma unroll
                        for (int j = 0; j < 32; j++)
                            if (v[j] > thr) mask |= 1u << j;
                    }
                    // Candidates are rare and scattered over rows and columns, so each lane walks ITS
                    // OWN candidate columns: trip count = the largest number of candidates any row of
                    // the warp has in this chunk (usually 1), one convergent exp per trip.  v[j] for
                    // the lane's own j is a 31-select tree over the registers.
                    uint32_t mk = mask;
                    const int trips = __reduce_max_sync(0xffffffffu, (unsigned)__popc(mk));
                    for (int q = 0; q < trips; q++) {
                        const bool act = mk != 0u;
                        const int j = act ? __ffs((int)mk) - 1 : 0;
                        mk &= mk - 1u;
                        const int vj = pick32(v, j);
                        const double rp = __shfl_sync(0xffffffffu, rp_cur[c], j);
                        if (tab) {
                            if (act) s = fma(etab[vj - vref + p.delta], rp, s);  // thr < vj <= vref + dpos
                        } else {
                            const int M = skeys[c * 32 + j] - vj;  // v = key - M
                            if (act) lse_add_fast(m, s, fma(p.kappa, (double)M, rp));
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_leader(acc_empty + slot);
            }
            // hand the partial (max, sum) of this set's columns to the merge warps and move on
            if (set == 0) skmax_all[((it + 1) & 1) * BM + rloc] = KEY_INIT;  // next unit's slot (idle since unit it - 1)
            asm volatile("bar.sync 2, %0;" ::"n"(NSETS * 128 + 64) : "memory");  // previous unit's partials consumed
            merge[set * BM + rloc] = tab ? make_double2(-p.kappa * (double)vref, s) : make_double2(m, s);
            asm volatile("bar.arrive 1, %0;" ::"n"(NSETS * 128 + 64) : "memory");
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's shared memory and barriers stay alive until both are done
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}
}  // namespace mma

// ---------------------------------------------------------------------------------------------
// host side

// [windows][rows][Wpad] bytes, box = 128 bytes x 128 rows
static int make_operand_map(CUtensorMap *m, void *base, int Wpad, int rows, int nW) {
    return encode_u8_3d(m, base, {(cuuint64_t)Wpad, (cuuint64_t)rows, (cuuint64_t)nW}, {(cuuint64_t)Wpad, (cuuint64_t)Wpad * rows},
                        {(cuuint32_t)mma::KBYTES, (cuuint32_t)mma::BM, 1});
}

bool ld_tensor_eligible(ibdgem_engine *e, int32_t n_targets, int32_t n_bg, const uint8_t *tgt_counts) {
    if (tgt_counts || e->prm.variable_sites_only) return false;
    if (!e->depth_linear || !(e->kappa < -1e-3)) return false;
    if (e->nW_shared <= 0 || e->K_shared <= 0) return false;
    const int Wpad = (e->prm.window_size + 127) / 128 * 128;
    if (Wpad > mma::MAXKB * mma::KBYTES) return false;
    if ((int64_t)e->prm.max_cov * Wpad >= (1 << 24)) return false;
    if (n_targets <= 0 || n_bg <= 0) return false;
    if (ceil(SCREEN_NATS / -e->kappa) > 1e6) return false;
    return true;
}

void ld_tensor_release(ibdgem_engine *e) {
    LdCache *c = e->ld;
    if (!c) return;
    dev_free(e, c->d_infsite, c->b_infsite);
    dev_free(e, c->d_nk, c->b_nk);
    dev_free(e, c->d_nr, c->b_nr);
    dev_free(e, c->d_l0, c->b_l0);
    dev_free(e, c->d_C0, c->b_C0);
    dev_free(e, c->d_tbits, c->b_tbits);
    delete c;
    e->ld = nullptr;
}

// New inputs: the cached operands are stale, but the buffers are kept — a re-upload of the same
// shape (every end-to-end step) then rebuilds in place without cudaFree / cudaMalloc.
void ld_tensor_invalidate(ibdgem_engine *e) {
    if (e->ld) e->ld->valid = false;
}

static int build_cache(ibdgem_engine *e) {
    if (e->ld && e->ld->valid) return 0;
    const int Wpad = (e->prm.window_size + 127) / 128 * 128;
    if (e->ld && (e->ld->nW != e->nW_shared || e->ld->N != e->N || e->ld->Wpad != Wpad)) ld_tensor_release(e);
    LdCache *c = e->ld;
    if (!c) {
        c = new LdCache();
        e->ld = c;
        c->nW = e->nW_shared;
        c->W = e->prm.window_size;
        c->Wpad = Wpad;
        c->WP32 = c->Wpad / 32;
        c->KB = c->Wpad / 128;
        c->N = e->N;
        c->H = 2 * e->N;
        const size_t slots = (size_t)c->nW * c->Wpad;
        c->b_infsite = slots * 4; c->b_nk = slots; c->b_nr = slots; c->b_l0 = slots * 8; c->b_C0 = (size_t)c->nW * 8;
        c->b_tbits = (size_t)c->nW * c->H * c->WP32 * 4;
        if (dev_alloc(e, (void **)&c->d_infsite, c->b_infsite) || dev_alloc(e, (void **)&c->d_nk, c->b_nk) ||
            dev_alloc(e, (void **)&c->d_nr, c->b_nr) || dev_alloc(e, (void **)&c->d_l0, c->b_l0) ||
            dev_alloc(e, (void **)&c->d_C0, c->b_C0) || dev_alloc(e, (void **)&c->d_tbits, c->b_tbits))
            return 1;
    }
    c->K = e->K_shared;
    IBD_CUDA(cudaMemsetAsync(c->d_infsite, 0xFF, c->b_infsite, e->stream));
    IBD_CUDA(cudaMemsetAsync(c->d_nk, 0, c->b_nk, e->stream));
    IBD_CUDA(cudaMemsetAsync(c->d_nr, 0, c->b_nr, e->stream));
    IBD_CUDA(cudaMemsetAsync(c->d_l0, 0, c->b_l0, e->stream));
    {
        LaunchScope ls(e, K_LD_COMPACT);
        ld_compact_kernel<<<(unsigned)((e->S + 255) / 256), 256, 0, e->stream>>>(
            e->S, e->d_status, e->d_rank, e->d_nref, e->d_nalt, e->d_lnP, e->C, c->W, c->Wpad, c->d_infsite, c->d_nk,
            c->d_nr, c->d_l0);
    }
    {
        LaunchScope ls(e, K_LD_C0);
        ld_c0_kernel<<<c->nW, 256, 0, e->stream>>>(c->d_l0, c->Wpad, c->d_C0);
    }
    IBD_CUDA(cudaGetLastError());
    c->valid = true;
    c->tw_upto = 0;
    return 0;
}

int ld_transpose_launch(ibdgem_engine *e, int w_begin, int w_end, const int32_t *infsite, int Wpad, int WP32, int H, uint32_t *tbits) {
    LaunchScope ls(e, K_LD_TRANSPOSE);
    const int words = (H + 31) / 32;
    for (int w0 = w_begin; w0 < w_end; w0 += MAX_GRID_Y)  // windows ride on gridDim.y
        ld_transpose_kernel<<<dim3((words + 7) / 8, std::min(MAX_GRID_Y, w_end - w0)), 1024, 0, e->stream>>>(
            w0, e->d_bits, e->Wh, H, infsite, Wpad, WP32, tbits);
    IBD_CUDA(cudaGetLastError());
    return 0;
}

void ld_background(int32_t N, int32_t T, const int32_t *h_targets, int32_t n_bg, const int32_t *h_bg, int32_t pu_idx, LdBackground *out) {
    // (ordinals were range-checked by the caller; plain arrays — this runs on the host between two stretches of device work)
    std::vector<int32_t> mult((size_t)N, 0), where((size_t)N, -1);
    int64_t total_bg = 0;
    for (int n = 0; n < n_bg; n++)
        if (h_bg[n] != pu_idx) { mult[h_bg[n]]++; total_bg++; }
    out->bgU.clear();
    out->lnc.clear();
    for (int32_t b = 0; b < N; b++)
        if (mult[b]) {
            where[b] = (int32_t)out->bgU.size();
            out->bgU.push_back(b);
            out->lnc.push_back(mult[b] == 1 ? 0.0 : log((double)mult[b]));
        }
    out->own.resize((size_t)T);
    out->nb.resize((size_t)T);
    out->lognb.resize((size_t)T);
    for (int t = 0; t < T; t++) {
        const int own = where[h_targets[t]];
        const int64_t nb = total_bg - (own >= 0 ? mult[h_targets[t]] : 0);
        out->own[t] = own;
        out->nb[t] = (int32_t)nb;
        out->lognb[t] = nb > 0 ? log((double)nb) : (double)NAN;
    }
}

double *host_table_alias(const ScoreCall &c) {
    if (!c.w_loglik) return nullptr;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, c.w_loglik) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
        return static_cast<double *>(attr.devicePointer);
    cudaGetLastError();
    return nullptr;
}

int range_event(ibdgem_engine *e, size_t k, cudaEvent_t *ev) {
    while (e->range_ev.size() <= k) {
        cudaEvent_t x;
        IBD_CUDA(cudaEventCreateWithFlags(&x, cudaEventDisableTiming));
        e->range_ev.push_back(x);
    }
    *ev = e->range_ev[k];
    return 0;
}

// Transposed bits of windows [tw_upto, w_hi).  The caller has made the engine stream
// wait for the panel rows of those windows (wait_panel_upto / ensure_table).
static int cache_windows(ibdgem_engine *e, int w_hi) {
    LdCache *c = e->ld;
    if (e->shard_count > 1 && c->tw_upto == 0) {  // a window shard never looks at the windows before its own
        int32_t wb = 0;
        window_shard_bounds(e, &wb, nullptr, nullptr, nullptr);
        c->tw_upto = wb;
    }
    if (c->tw_upto >= w_hi) return 0;
    if (ld_transpose_launch(e, c->tw_upto, w_hi, c->d_infsite, c->Wpad, c->WP32, c->H, c->d_tbits)) return 1;
    c->tw_upto = w_hi;
    return 0;
}

int ld_tensor_prepare(ibdgem_engine *e) {
    if (build_cache(e) || ensure_table(e, e->S)) return 1;
    return cache_windows(e, e->ld->nW);
}

// Fills every window output of the call: d_wll [T][outW][3], d_wn, d_ws, d_we [T][outW], d_nwout [T].
int ld_tensor_score(ibdgem_engine *e, ScoreCall &sc) {
    if (build_cache(e)) return 1;
    LdCache *c = e->ld;
    // duplicate background entries are a ln(multiplicity) weight on one individual (sc.bg)
    const LdBackground &bg = sc.bg;
    const int T = sc.T, outW = sc.outW;
    const int32_t *d_targets = sc.d_targets;
    double *d_wll = sc.d_wll;
    const int nU = (int)bg.bgU.size();
    std::vector<int32_t> row_own(2 * (size_t)T);
    std::vector<double> lognb4(T);
    for (int t = 0; t < T; t++) {
        lognb4[t] = bg.nb[t] > 0 ? log(4.0 * (double)bg.nb[t]) : (double)NAN;
        row_own[2 * t] = row_own[2 * t + 1] = bg.own[t] >= 0 ? 2 * bg.own[t] : -1;
    }
    const int nW = c->nW;
    // Window ranges: one per panel chunk still in flight (a range is the windows whose last site has
    // arrived), so the scoring of early windows overlaps the rest of the upload; a single range when
    // the panel is already resident.
    std::vector<int> range_end;
    const bool in_flight = e->chunks_waited < (int)e->chunk_end.size() && e->chunk_end.size() > 1 &&
                           cudaEventQuery(e->chunk_ev[e->chunk_end.size() - 1]) == cudaErrorNotReady;
    if (in_flight && c->tw_upto == 0) {  // (by_chunk below)
        int w = 0;
        for (size_t k = 0; k < e->chunk_end.size(); k++) {
            while (w < nW && e->h_wlast[(size_t)w] < e->chunk_end[k]) w++;
            range_end.push_back(k + 1 == e->chunk_end.size() ? nW : w);
        }
    } else {
        // Panel resident: one range.  (Splitting off a tail range, so that the first range's columns travel to the host
        // while the tail is scored, was measured at C3 to buy nothing: a second round of launches costs what the
        // hidden 0.4 ms copy saves.)
        range_end.push_back(nW);
    }
    bool by_chunk = in_flight && c->tw_upto == 0;
    // a window shard scores its own windows only, as one range, and waits for (and tabulates) its own rows only
    int32_t shard_wb = 0, shard_we = nW;
    int64_t shard_se = e->S;
    const bool sharded = e->shard_count > 1;
    if (sharded) {
        window_shard_bounds(e, &shard_wb, &shard_we, nullptr, &shard_se);
        range_end.clear();
        // three sub-ranges when results go to the host and the shard is large: the copy of a sub-range's columns runs
        // under the next sub-range's GEMM, so only the last one's is left at the end
        const int span = shard_we - shard_wb;
        static const int parts_env = env_int("IBDGEM_SHARD_PARTS", 3);
        // ... as long as every sub-range still keeps the persistent GEMM busy for >= 8 rounds of units (IBDGEM_SHARD_PARTS < 0
        // forces |value| parts, for tests)
        const int64_t units = (int64_t)span * ((2 * T + 255) / 256);
        int parts = 1;
        if (parts_env < 0) parts = std::min(span, -parts_env);
        else if (sc.w_loglik && parts_env > 1 && (size_t)T * span * 24 >= ((size_t)20 << 20))
            // (a sub-range costs ~0.1 ms in launches and GEMM ramps: measured a loss below ~20 MB of shard table — C3 over
            // 2 and 4 GPUs — and a gain above — C5 over 8)
            parts = (int)std::max<int64_t>(1, std::min<int64_t>(parts_env, units / (8 * std::max(1, e->sm_count / 2))));
        // sub-ranges shrink (parts : parts - 1 : ... : 1): what is left after the last GEMM is the copy of the smallest one
        const int64_t wsum = (int64_t)parts * (parts + 1) / 2;
        int64_t acc = 0;
        for (int k = 0; k < parts; k++) {
            acc += parts - k;
            range_end.push_back(shard_wb + (int)((int64_t)span * acc / wsum));
        }
        by_chunk = false;
    }
    auto range_sites = [&](size_t k) { return by_chunk ? e->chunk_end[k] : shard_se; };
    const int nrows = 2 * T;
    if (nU == 0) {  // every background member excluded: LIBD0 = LIBD1 = 0/0 (d_wll is NaN-filled)
        double *d_Rt;
        if (ensure_table(e, e->S) || cache_windows(e, nW) || scratch(e, SC_MMA_ROWLSE, (size_t)nW * nrows * 8, (void **)&d_Rt))
            return 1;
        {
            LaunchScope ls(e, K_LD_WINDOWS);
            const int64_t n = (int64_t)T * nW;
            ld_windows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(
                0, nW, T, nW, outW, c->W, c->K, e->d_wfirst, e->d_wlast, e->d_pos, sc.d_wn, sc.d_ws, sc.d_we, sc.d_nwout);
        }
        {
            LaunchScope ls(e, K_LD_EXPAND_TGT);
            for (int w0 = 0; w0 < nW; w0 += MAX_GRID_Y)
                ld_expand_tgt_kernel<<<dim3((unsigned)((T + 7) / 8), (unsigned)std::min(MAX_GRID_Y, nW - w0)), 256, 0, e->stream>>>(
                    w0, T, c->H, c->Wpad, c->WP32, outW, d_targets, c->d_tbits, c->d_nr, c->d_nk, c->d_C0, e->alpha, e->beta,
                    e->kappa, nullptr, d_Rt, d_wll);
        }
        IBD_CUDA(cudaGetLastError());
        return 0;
    }
    const int ncols = 2 * nU;
    const int NT = (ncols + mma::TILE_N - 1) / mma::TILE_N;
    const int ncolpad = NT * mma::TILE_N;
    const int MB = (nrows + mma::BM * mma::CG - 1) / (mma::BM * mma::CG);

    const size_t per_window = (size_t)(ncols + nrows) * c->Wpad;
    // IBDGEM_LD_BUDGET_MB: operand budget override (tests exercise the window batching with it)
    static const int budget_mb = env_int("IBDGEM_LD_BUDGET_MB", 0);
    const size_t budget = budget_mb > 0 ? (size_t)budget_mb << 20 : LD_OPERAND_BUDGET;
    const int nWb = (int)std::max<size_t>(1, std::min<size_t>({(size_t)nW, budget / per_window, (size_t)MAX_GRID_Y}));
    int32_t *d_bgU, *d_ownU, *d_rowown, *d_akey;
    double *d_lnc, *d_lognb, *d_lognb4, *d_Rp, *d_Qp, *d_Rt, *d_Fp;
    unsigned char *d_A, *d_B;
    const size_t misc_i = (size_t)nU + T + 2 * (size_t)T;
    const size_t misc_d = (size_t)nU + 2 * (size_t)T;
    if (scratch(e, SC_MMA_MISC, misc_i * 4 + misc_d * 8 + 64, (void **)&d_lnc) ||
        scratch(e, SC_MMA_BGIDX, (size_t)nW * ncolpad * 4, (void **)&d_akey) ||
        scratch(e, SC_MMA_ROWLSE, (2 * (size_t)nW * ncolpad + (size_t)nW * nU + (size_t)nW * nrows) * 8, (void **)&d_Rp) ||
        scratch(e, SC_MMA_TGT, (size_t)nWb * nrows * c->Wpad, (void **)&d_A) ||
        scratch(e, SC_MMA_BG, (size_t)nWb * ncols * c->Wpad, (void **)&d_B))
        return 1;
    d_lognb = d_lnc + nU;
    d_lognb4 = d_lognb + T;
    d_bgU = reinterpret_cast<int32_t *>(d_lognb4 + T);
    d_ownU = d_bgU + nU;
    d_rowown = d_ownU + T;
    d_Fp = d_Rp + (size_t)nW * ncolpad;
    d_Qp = d_Fp + (size_t)nW * ncolpad;
    d_Rt = d_Qp + (size_t)nW * nU;
    {
        // the call's small tables go up in one piece from pinned memory, laid out like SC_MMA_MISC
        void *h_misc;
        if (pinned_stage(e, misc_d * 8 + misc_i * 4, &h_misc)) return 1;
        double *hd = static_cast<double *>(h_misc);
        memcpy(hd, bg.lnc.data(), (size_t)nU * 8);
        memcpy(hd + nU, bg.lognb.data(), (size_t)T * 8);
        memcpy(hd + nU + T, lognb4.data(), (size_t)T * 8);
        int32_t *hi = reinterpret_cast<int32_t *>(hd + misc_d);
        memcpy(hi, bg.bgU.data(), (size_t)nU * 4);
        memcpy(hi + nU, bg.own.data(), (size_t)T * 4);
        memcpy(hi + nU + T, row_own.data(), (size_t)T * 8);
        // Not a cudaMemcpyAsync: a DMA copy would queue on the host-to-device copy engine behind the panel
        // chunks still in flight and hold the scoring of the first windows back until the whole panel is up.
        LaunchScope ls(e, K_LD_STAGE);
        const int n = (int)((misc_d * 8 + misc_i * 4) / 4);
        ld_stage_kernel<<<(n + 255) / 256, 256, 0, e->stream>>>(reinterpret_cast<uint32_t *>(d_lnc),
                                                               static_cast<const uint32_t *>(h_misc), n);
    }

    const bool stream_out = (range_end.size() > 1 || sharded) && sc.w_loglik != nullptr;
    // the optional device destination (the root's gather buffer, possibly peer memory over NVLink) is
    // filled range by range too
    const bool stream_dev = sc.w_loglik_device != nullptr;
    // page-locked host destination: its device alias, for stores from a kernel
    double *h_wll_mapped = host_table_alias(sc);
    // direct mode: the GEMM's merge warps store finished score triples into the page-locked host table themselves
    // (not while panel chunks are still arriving: measured at C3 end to end, the 24-byte posted writes of every range
    // compete with the upload on the link — 13.3 ms against 12.6 with the per-range store kernel)
    // (nor for window shards: eight ranks scattering 24-byte writes over a 10,000-row host table — one 4 KB page per
    // write — slowed the GEMM by 15 % at C5 over 8 GPUs; there the shard's columns leave by one store kernel at the end)
    const bool direct = h_wll_mapped != nullptr && !by_chunk && !sharded;
    if (stream_out || stream_dev || direct) {
        if (side_streams(e)) return 1;
        sc.streamed = stream_out || direct;
        sc.dev_streamed = stream_dev;
    }
    auto launch_ibd0 = [&](int wa, int wb_) -> int {
        LaunchScope ls(e, K_LD_IBD0);
        // the window's Q' row is staged in shared memory when it fits (one bulk, coalesced load instead
        // of latency-bound passes over global memory)
        const size_t q_smem = (size_t)nU * 8 <= 160 * 1024 ? (size_t)nU * 8 : 0;
        IBD_CUDA(cudaFuncSetAttribute(ld_ibd0_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        ld_ibd0_kernel<<<wb_ - wa, 256, q_smem, e->stream>>>(wa, T, nU, outW, d_Qp, d_ownU, d_lognb, d_wll, q_smem ? 1 : 0);
        return 0;
    };
    // columns [w, w + n) of d_wll to the same columns of dst [T][outW][3] on d2h_stream; many short rows go by coalesced
    // stores from a kernel (ld_store_cols_kernel) where dst has a device address dst_dev (local, peer or mapped host
    // memory), not by T DMA descriptors
    auto export_cols = [&](double *dst, double *dst_dev, int w, int n) -> int {
        if (dst_dev && T >= 256) {
            const int64_t cnt = (int64_t)T * n * 3;
            ld_store_cols_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, e->d2h_stream>>>(d_wll, dst_dev, T, outW, w, n);
            e->k_launches[K_LD_WINDOWS]++;
        } else {
            IBD_CUDA(cudaMemcpy2DAsync(dst + (size_t)w * 3, (size_t)outW * 24, d_wll + (size_t)w * 3, (size_t)outW * 24, (size_t)n * 24,
                                       (size_t)T, cudaMemcpyDefault, e->d2h_stream));
        }
        return 0;
    };
    // d2h_stream waits for the engine stream's work so far (range event k)
    auto d2h_after = [&](size_t k) -> int {
        cudaEvent_t ev;
        if (range_event(e, k, &ev)) return 1;
        IBD_CUDA(cudaEventRecord(ev, e->stream));
        IBD_CUDA(cudaStreamWaitEvent(e->d2h_stream, ev, 0));
        return 0;
    };
    int w_lo = shard_wb;
    for (size_t rk = 0; rk < range_end.size(); rk++) {
    const int w_hi = range_end[rk];
    if (ensure_table(e, range_sites(rk))) return 1;  // waits for the chunk, evaluates its per-site table
    if (w_hi == w_lo && !(sharded && rk == 0)) continue;
    if (w_hi > w_lo && cache_windows(e, w_hi)) return 1;
    if (!sharded || rk == 0) {
        // (a window shard still reports the bookkeeping of ALL windows: it is the same on every rank; once, with its first sub-range)
        LaunchScope ls(e, K_LD_WINDOWS);
        const int b_lo = sharded ? 0 : w_lo, b_hi = sharded ? nW : w_hi;
        const int64_t n = (int64_t)T * (b_hi - b_lo);
        ld_windows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(
            b_lo, b_hi, T, nW, outW, c->W, c->K, e->d_wfirst, e->d_wlast, e->d_pos, sc.d_wn, sc.d_ws, sc.d_we, sc.d_nwout);
    }
    // START / END / NUM_SITES of every window are final: their copy to the host can overlap the GEMM (score_common).
    // Recorded ONCE: the copy waits for the event's latest record, so a record per sub-range of a shard held the
    // bookkeeping copy back until the last sub-range (200 MB at C5: it then outlasted the last GEMM on the root rank).
    if (!sc.bookkeeping_ready && (sharded ? rk == 0 : w_hi == nW)) {
        IBD_CUDA(cudaEventRecord(e->ev_book, e->stream));
        sc.bookkeeping_ready = true;
    }
    IBD_CUDA(cudaGetLastError());
    if (w_hi == w_lo) continue;  // (an empty shard: bookkeeping only)
    // windows are processed in batches so the expanded int8 operands stay within a fixed budget
    for (int w0 = w_lo; w0 < w_hi; w0 += nWb) {
        const int nw = std::min(nWb, w_hi - w0);
        {
            LaunchScope ls(e, K_LD_EXPAND_BG);
            const int npadU = ncolpad / 2;
            ld_expand_bg_kernel<<<dim3((unsigned)((npadU + 7) / 8), (unsigned)nw), 256, 0, e->stream>>>(
                w0, nU, npadU, ncols, ncolpad, c->H, c->Wpad, c->WP32, d_bgU, d_lnc, c->d_tbits, c->d_nr, c->d_nk, c->d_C0,
                e->alpha, e->beta, e->kappa, 1.0 / -e->kappa, d_B, d_akey, d_Rp, d_Qp, d_Fp);
        }
        {
            LaunchScope ls(e, K_LD_EXPAND_TGT);
            ld_expand_tgt_kernel<<<dim3((unsigned)((T + 7) / 8), (unsigned)nw), 256, 0, e->stream>>>(
                w0, T, c->H, c->Wpad, c->WP32, outW, d_targets, c->d_tbits, c->d_nr, c->d_nk, c->d_C0, e->alpha, e->beta,
                e->kappa, d_A, d_Rt, d_wll);
        }
        IBD_CUDA(cudaGetLastError());
        CUtensorMap mapA, mapB;
        if (make_operand_map(&mapA, d_A, c->Wpad, nrows, nw)) return 1;
        if (make_operand_map(&mapB, d_B, c->Wpad, ncols, nw)) return 1;
        mma::Params p;
        p.w0 = w0;
        p.nW = nw; p.MB = MB; p.NT = NT; p.KB = c->KB;
        p.n_units = nw * MB;
        p.nrows = nrows; p.ncolpad = ncolpad;
        p.H = c->H; p.outW = outW;
        p.delta = (int)ceil(screen_nats(ncols) / -e->kappa) + 2;
        p.kappa = e->kappa;
        p.akey = d_akey; p.Rp = d_Rp; p.Rt = d_Rt;
        p.Fp = d_Fp;
        {
            // table mode when the screen's reach plus the head-room above a row's reference key fits the shared-memory
            // table and exp(|kappa| dpos) stays far from overflow
            const int dpos = (int)std::min(256.0, floor(600.0 / -e->kappa));
            const int tab_n = p.delta + dpos + 1;
            const bool tab = dpos >= 8 && tab_n <= mma::ETAB_N;
            p.tab_n = tab ? tab_n : 0;
            p.dpos = dpos;
        }
        p.row_own = d_rowown;
        p.C0 = c->d_C0; p.lognb4 = d_lognb4; p.wll = d_wll;
        p.wll_host = direct ? h_wll_mapped : nullptr;
        if (direct && launch_ibd0(w0, w0 + nw)) return 1;  // LIBD0 must be in the table before the GEMM's merge warps read it
        {
            int *d_unit;
            if (scratch(e, SC_MMA_UNIT, 64, (void **)&d_unit)) return 1;
            IBD_CUDA(cudaMemsetAsync(d_unit, 0, 4, e->stream));
            p.unit_counter = d_unit;
        }
        {
            LaunchScope ls(e, K_LD_MMA);
            if (launch_pairs(mma::ld_mma_kernel, mma::THREADS, mma::SMEM_BYTES, p.n_units, e->sm_count, e->stream, mapA, mapB, p)) return 1;
        }
        IBD_CUDA(cudaGetLastError());
    }
    if (!direct && launch_ibd0(w_lo, w_hi)) return 1;
    if (stream_out || stream_dev) {
        // the range's columns of d_wll [T][outW][3] are final: they leave on their own stream
        if (d2h_after(rk)) return 1;
        if (stream_dev && export_cols(sc.w_loglik_device, sc.w_loglik_device, w_lo, w_hi - w_lo)) return 1;
        if (stream_out && sharded && e->shard_compact) {
            // compact host table of a window shard: pack on the device, one contiguous copy
            double *d_pack;
            const int64_t n = (int64_t)T * (w_hi - w_lo) * 3, off = (int64_t)T * (w_lo - shard_wb) * 3;
            if (scratch(e, SC_WLL_PACK, (size_t)T * (shard_we - shard_wb) * 24, (void **)&d_pack)) return 1;
            ld_pack_cols_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->d2h_stream>>>(d_wll, d_pack + off, T, outW, w_lo, w_hi - w_lo);
            e->k_launches[K_LD_WINDOWS]++;
            IBD_CUDA(cudaMemcpyAsync(sc.w_loglik + off, d_pack + off, (size_t)n * 8, cudaMemcpyDeviceToHost, e->d2h_stream));
        } else if (stream_out && !direct) {
            if (export_cols(sc.w_loglik, h_wll_mapped, w_lo, w_hi - w_lo)) return 1;
        }
    }
    w_lo = w_hi;
    }  // window ranges
    if ((stream_out || direct) && outW > nW && !sharded) {  // the unused columns nW .. outW-1 (NaN since the fill at the start of the call)
        if (d2h_after(range_end.size()) || export_cols(sc.w_loglik, h_wll_mapped, nW, outW - nW)) return 1;
    }
    IBD_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace ibdgem
