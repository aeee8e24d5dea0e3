// posterior.cu — batched hiddengem posterior: per-bin IBD-state probabilities by forward-backward over the same path
// weights the Viterbi pass (hidden.cu) maximises,
//   W(x) = prod_i nrm[i][x_i] * prod_{i>0} pen(x_{i-1}, x_i),   gamma[i][s] = sum_{x : x_i = s} W(x) / sum_x W(x),
// with pen = 1 on the diagonal and p01 / p02 / p12 off it (symmetric), and no prior on bin 0.  The penalties are the
// reference's weights, not transition probabilities; the posterior is the marginal of those weights, so the Viterbi
// path is its mode.
//
// Scaled forward-backward in fp64 linear space.  Only the direction of a row of alpha or beta matters, so every row is
// rescaled by the power of two that brings its sum into [1, 2): an exact multiplication, no division on the solver's
// critical path, and the row's sum cannot under- or overflow however long the table.  The entries inside a row can:
// a state more than 700 nats behind in one bin gets emission 0, and an entry below 2^-1074 of its row is flushed.
// That is harmless while every penalty keeps all states within reach of each other (linear_penalties below); with a
// zero penalty, or penalties spread wider than 2^400, the only paths between two states can run through such
// entries.  Those calls run the same two kernels in natural-log arithmetic (LG = true: log-sum-exp mixing, rows
// shifted to maximum 0), which has no range limit; they cost more fp64 work on the solver lane.
//
// Two kernels on the chunked block of hg_block.cuh (shared with viterbi_fused_kernel): a block takes 32 tables, worker
// warps stage 16-bin chunks with coalesced loads and compute the emissions in shared memory, ONE solver warp
// (lane = table) walks the chunk, chunks are double buffered.
//   forward   walks the chunks in order and stores only alpha of each chunk's last bin (a checkpoint, 24 B per table
//             per 16 bins);
//   backward  walks the chunks in reverse; per chunk the solver recomputes alpha from the previous chunk's checkpoint
//             (the same operations, hence the same doubles), then walks beta down the chunk; the workers form
//             gamma = alpha * beta / sum, write it and accumulate the expected occupancy.
// Bytes per bin: 24 read by each pass, 24 written once, plus the checkpoints (3 B): ~75 B, against ~120 B for a
// design that stores alpha of every bin and reads it back.
//   moments   (hiddengem_posterior_moments_*) the backward kernel with MOM = true: the solver lane also carries the
//             moment recursion down the table (moment_step) and sums each table's covariance terms in bin order
//             (moment_acc).  The sums stay on the solver lane: staging its per-bin state in shared memory for the
//             workers would add 32-74 KB per block and drop residency from three blocks per SM to two or one, and at
//             C4 the 313 blocks then need two waves.  The posteriors are optional there.
//
// Emissions (nrm; any positive per-bin factor cancels in gamma, so only the direction is needed):
//   is_log = 0  l_s / ((l0 + l1) + l2) as hiddengem normalises summary-file likelihoods, with the division replaced
//               by the exact power-of-two scaling that brings the total into [1, 2);
//   is_log = 1  exp(L_s - max_k L_k).
// A bin whose normalised row is undefined (text: a total that is not a positive finite number, e.g. all three 0 or a
// NaN; log: a NaN score, or a row maximum that is not finite) carries no information and gets the uniform emission (1, 1, 1).  A table whose total weight is
// 0 as a real number (possible only with zero penalties, so decided in log arithmetic, where it is exact) has NaN
// posteriors and NaN expected counts.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "engine.h"
#include "hg_block.cuh"
#include "tc_common.cuh"

namespace ibdgem {

constexpr int PB_FWD_SMEM = 2 * HG_TABLES * HG_ROW * 8 + HG_HEAD_SMEM;
constexpr int PB_BWD_SMEM = 4 * HG_TABLES * HG_ROW * 8 + HG_HEAD_SMEM + HG_TABLES * 4;
static_assert(HG_TABLES * HG_BINS * 3 <= HG_TABLES * HG_ROW, "expected-count partials fit in one staging buffer");

// 2^-floor(log2 s) for s >= 0: multiplying by it is exact and brings s into [1, 2) (0 stays 0)
__device__ __forceinline__ double pow2_recip(double s) {
    const int ex = min(max((__double2hiint(s) >> 20) & 0x7ff, 1), 2045);
    return __hiloint2double((2046 - ex) << 20, 0);
}

// 1 / s for a positive normal s: hardware estimate and two Newton steps on s scaled into [1, 2) (no slow-path call)
__device__ __forceinline__ double recip(double s) {
    const double k = pow2_recip(s), m = s * k;
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(m));
    y = fma(y, fma(-m, y, 1.0), y);
    y = fma(y, fma(-m, y, 1.0), y);
    return y * k;
}

// log(exp(x) + exp(y) + exp(z)) for x, y, z < +inf; -inf when all three are -inf.  Terms more than 700 below the
// largest are dropped (relative weight < 1e-304).
__device__ __forceinline__ double lse3(double x, double y, double z) {
    const double m = fmax(x, fmax(y, z)), ms = m > -INFINITY ? m : 0.0;
    return ms + log(exp_nonpos(x - ms) + exp_nonpos(y - ms) + exp_nonpos(z - ms));
}

// shift a row of log weights so its maximum is 0 (a row of -inf stays -inf)
__device__ __forceinline__ void shift_max0(double &u0, double &u1, double &u2) {
    const double m = fmax(u0, fmax(u1, u2)), ms = m > -INFINITY ? m : 0.0;
    u0 -= ms;
    u1 -= ms;
    u2 -= ms;
}

// Emission row of one bin, in place: linear (LG = false) or natural log (LG = true, no range limit).
template <bool LG>
__device__ __forceinline__ void emission(double *L, int is_log) {
    double e0, e1, e2;
    bool bad;
    if (is_log) {
        const double m = fmax(L[0], fmax(L[1], L[2]));
        bad = isnan(L[0]) || isnan(L[1]) || isnan(L[2]) || !isfinite(m);
        if (LG) {
            e0 = L[0] - m;
            e1 = L[1] - m;
            e2 = L[2] - m;
        } else {
            e0 = exp_nonpos(L[0] - m);
            e1 = exp_nonpos(L[1] - m);
            e2 = exp_nonpos(L[2] - m);
        }
    } else {  // l_s / tot up to a power of two (exact, and no division); in log space log l_s - log tot, which
              // keeps a ratio l_s / tot below the double range
        const double tot = __dadd_rn(__dadd_rn(L[0], L[1]), L[2]);
        bad = !(tot > 0) || !isfinite(tot);
        if (LG) {
            const double lt = log(tot);
            e0 = log(L[0]) - lt;
            e1 = log(L[1]) - lt;
            e2 = log(L[2]) - lt;
        } else {
            const double sc = pow2_recip(tot);
            e0 = L[0] * sc;
            e1 = L[1] * sc;
            e2 = L[2] * sc;
        }
    }
    const double one = LG ? 0.0 : 1.0;
    L[0] = bad ? one : e0;
    L[1] = bad ? one : e1;
    L[2] = bad ? one : e2;
}

// one forward step: alpha[i] from alpha[i - 1] (or nothing, on bin 0) and the emission of bin i; LG: every value a
// natural log, p01 / p02 / p12 the logs of the penalties
template <bool LG>
__device__ __forceinline__ void fwd_step(double &a0, double &a1, double &a2, double e0, double e1, double e2, bool first, bool live,
                                         double p01, double p02, double p12) {
    if (LG) {
        double u0 = e0 + (first ? 0.0 : lse3(a0, a1 + p01, a2 + p02));
        double u1 = e1 + (first ? 0.0 : lse3(a0 + p01, a1, a2 + p12));
        double u2 = e2 + (first ? 0.0 : lse3(a0 + p02, a1 + p12, a2));
        shift_max0(u0, u1, u2);
        a0 = live ? u0 : a0;
        a1 = live ? u1 : a1;
        a2 = live ? u2 : a2;
        return;
    }
    const double t0 = first ? 1.0 : fma(a2, p02, fma(a1, p01, a0));
    const double t1 = first ? 1.0 : fma(a2, p12, fma(a0, p01, a1));
    const double t2 = first ? 1.0 : fma(a1, p12, fma(a0, p02, a2));
    const double u0 = e0 * t0, u1 = e1 * t1, u2 = e2 * t2;
    const double sc = pow2_recip(u0 + u1 + u2);
    a0 = live ? u0 * sc : a0;
    a1 = live ? u1 * sc : a1;
    a2 = live ? u2 * sc : a2;
}

// one backward step: beta[i - 1] = sum_k pen(s, k) nrm[i][k] beta[i][k], rescaled (LG: in logs)
template <bool LG>
__device__ __forceinline__ void bwd_step(double &b0, double &b1, double &b2, double e0, double e1, double e2, bool live, double p01,
                                         double p02, double p12) {
    if (LG) {
        const double v0 = e0 + b0, v1 = e1 + b1, v2 = e2 + b2;
        double t0 = lse3(v0, v1 + p01, v2 + p02);
        double t1 = lse3(v0 + p01, v1, v2 + p12);
        double t2 = lse3(v0 + p02, v1 + p12, v2);
        shift_max0(t0, t1, t2);
        b0 = live ? t0 : b0;
        b1 = live ? t1 : b1;
        b2 = live ? t2 : b2;
        return;
    }
    const double v0 = e0 * b0, v1 = e1 * b1, v2 = e2 * b2;
    const double t0 = fma(v2, p02, fma(v1, p01, v0));
    const double t1 = fma(v2, p12, fma(v0, p01, v1));
    const double t2 = fma(v1, p12, fma(v0, p02, v2));
    const double sc = pow2_recip(t0 + t1 + t2);
    b0 = live ? t0 * sc : b0;
    b1 = live ? t1 * sc : b1;
    b2 = live ? t2 * sc : b2;
}

// gamma of one bin from alpha and beta (NaN for a table of total weight 0)
template <bool LG>
__device__ __forceinline__ void gamma(const double *A, const double *B, bool dead, double &y0, double &y1, double &y2) {
    double g0, g1, g2;
    if (LG) {  // a live table has a finite maximum in every bin
        g0 = A[0] + B[0];
        g1 = A[1] + B[1];
        g2 = A[2] + B[2];
        shift_max0(g0, g1, g2);
        g0 = exp_nonpos(g0);
        g1 = exp_nonpos(g1);
        g2 = exp_nonpos(g2);
    } else {
        g0 = A[0] * B[0];
        g1 = A[1] * B[1];
        g2 = A[2] * B[2];
    }
    const double inv = dead ? __longlong_as_double(0x7ff8000000000000LL) : recip(g0 + g1 + g2);
    y0 = g0 * inv;
    y1 = g1 * inv;
    y2 = g2 * inv;
}

// Moments (the MOM variant of the backward pass).  Conditioned on x_{i-1} = k the rest of the path is Markov with
// P(x_i = l | k) = pen(k, l) nrm[i][l] beta[i][l] / t_k, t_k = sum_l pen(k, l) nrm[i][l] beta[i][l] (the sum bwd_step
// forms).  With h_i^t[k] = E[#{j > i : x_j = t} | x_i = k],
//     h_{i-1}^t[k] = sum_l P(l | k) (delta_lt + h_i^t[l]),   h_{n-1} = 0,
//     Cov(N_s, N_t) = sum_i gamma_i(s) (delta_st - gamma_i(t)) + gamma_i(s) (h_i^t[s] - H_i^t) + gamma_i(t) (h_i^s[t] - H_i^s),
// H_i^t = sum_k gamma_i(k) h_i^t[k].  Every term is invariant to adding one constant per t to h_i^t[0..2], so the
// solver carries u^t[k] = h^t[k] minus h^t of the state with the largest t_k (a live state): bounded by the
// correlation length, where h grows with n and its differences would lose a digit per factor 10 of table length.
// u^2 is -u^0 - u^1 up to such a constant (sum_t h^t[k] = n - 1 - i for every k), so only t = 0, 1 are carried.
// A state with t_k = 0 (or below the normal range) has gamma 0 there and no weight in the next step: its m is set to 0.
template <bool LG>
__device__ __forceinline__ void moment_step(double (&u)[2][3], double e0, double e1, double e2, double b0, double b1, double b2,
                                            double p01, double p02, double p12) {
    double m[2][3], t0, t1, t2;
    if (LG) {  // P(l | k) = exp(lp(k, l) + v_l - t_k), 0 where t_k = -inf
        const double v0 = e0 + b0, v1 = e1 + b1, v2 = e2 + b2;
        t0 = lse3(v0, v1 + p01, v2 + p02);
        t1 = lse3(v0 + p01, v1, v2 + p12);
        t2 = lse3(v0 + p02, v1 + p12, v2);
        const double x[3][3] = {{v0, v1 + p01, v2 + p02}, {v0 + p01, v1, v2 + p12}, {v0 + p02, v1 + p12, v2}};
        const double tk[3] = {t0, t1, t2};
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const bool ok = tk[k] > -INFINITY;
            const double q0 = ok ? exp_nonpos(x[k][0] - tk[k]) : 0.0, q1 = ok ? exp_nonpos(x[k][1] - tk[k]) : 0.0,
                         q2 = ok ? exp_nonpos(x[k][2] - tk[k]) : 0.0;
#pragma unroll
            for (int t = 0; t < 2; t++) m[t][k] = fma(q0, u[t][0], fma(q1, u[t][1], fma(q2, u[t][2], t == 0 ? q0 : q1)));
        }
    } else {  // m^t[k] = (sum_l pen(k, l) v_l (delta_lt + u^t[l])) / t_k
        const double v0 = e0 * b0, v1 = e1 * b1, v2 = e2 * b2;
        t0 = fma(v2, p02, fma(v1, p01, v0));
        t1 = fma(v2, p12, fma(v0, p01, v1));
        t2 = fma(v1, p12, fma(v0, p02, v2));
        const double r0 = t0 >= 0x1p-1022 ? recip(t0) : 0.0, r1 = t1 >= 0x1p-1022 ? recip(t1) : 0.0,
                     r2 = t2 >= 0x1p-1022 ? recip(t2) : 0.0;
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const double w0 = v0 * (u[t][0] + (t == 0)), w1 = v1 * (u[t][1] + (t == 1)), w2 = v2 * u[t][2];
            m[t][0] = r0 * fma(w2, p02, fma(w1, p01, w0));
            m[t][1] = r1 * fma(w2, p12, fma(w0, p01, w1));
            m[t][2] = r2 * fma(w1, p12, fma(w0, p02, w2));
        }
    }
    const int r = (t1 > t0) ? (t2 > t1 ? 2 : 1) : (t2 > t0 ? 2 : 0);  // a live state (largest t_k)
#pragma unroll
    for (int t = 0; t < 2; t++) {
        const double ref = r == 0 ? m[t][0] : r == 1 ? m[t][1] : m[t][2];
        u[t][0] = m[t][0] - ref;
        u[t][1] = m[t][1] - ref;
        u[t][2] = m[t][2] - ref;
    }
}

// one bin's cross terms (gamma y of the bin, u of the bin) into the upper triangle C = {00, 01, 02, 11, 12, 22}
__device__ __forceinline__ void moment_acc(double (&C)[6], const double (&u)[2][3], double y0, double y1, double y2) {
    const double y[3] = {y0, y1, y2};
    double d[3][3];  // d[t][s] = gamma(s) (u^t[s] - U^t)
#pragma unroll
    for (int t = 0; t < 3; t++) {
        const double a0 = t < 2 ? u[t][0] : -u[0][0] - u[1][0], a1 = t < 2 ? u[t][1] : -u[0][1] - u[1][1],
                     a2 = t < 2 ? u[t][2] : -u[0][2] - u[1][2];
        const double U = fma(y2, a2, fma(y1, a1, y0 * a0));
        d[t][0] = y0 * (a0 - U);
        d[t][1] = y1 * (a1 - U);
        d[t][2] = y2 * (a2 - U);
    }
    int k = 0;
#pragma unroll
    for (int s = 0; s < 3; s++)
#pragma unroll
        for (int t = s; t < 3; t++, k++) C[k] += fma(y[s], (s == t ? 1.0 : 0.0) - y[t], d[t][s] + d[s][t]);
}

// Workers: emissions of chunk c in place, once every worker has stored its part
template <bool LG>
__device__ __forceinline__ void emit(const ChunkLoader &ld, int c, double (*buf)[HG_ROW], int is_log) {
    sync_workers();
    const int64_t i0 = (int64_t)c * HG_BINS;
#pragma unroll 1  // unrolled, the two bins need more registers than three blocks per SM leave
    for (int k = 0; k < HG_NBIN; k++) {
        const int idx = k * HG_WORKERS + ld.w;
        const int t = idx / HG_BINS, i = idx % HG_BINS;
        if (i0 + i < ld.s_len[t]) emission<LG>(&buf[t][i * 3], is_log);
    }
    __threadfence_block();
}

// Forward pass: alpha of each chunk's last bin -> ckpt[chunk][n_tables][3]; 0 in expected[t][0] exactly when the
// table's total weight is 0 (a positive value otherwise).
template <bool LG>
__global__ void __launch_bounds__(HG_THREADS, 3)
posterior_fwd_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const double *__restrict__ lik,
                     int is_log, double p01, double p02, double p12, double *__restrict__ ckpt, double *__restrict__ expected) {
    extern __shared__ double pb_smem[];
    double (*em)[HG_TABLES][HG_ROW] = reinterpret_cast<double (*)[HG_TABLES][HG_ROW]>(pb_smem);
    int64_t *s_start = reinterpret_cast<int64_t *>(pb_smem + 2 * HG_TABLES * HG_ROW), *s_len = s_start + HG_TABLES;
    const int tb0 = blockIdx.x * HG_TABLES;
    const int nchunk = block_tables(n_tables, start, len, s_start, s_len);
    if (threadIdx.x >= 32) {
        const ChunkLoader ld{s_start, s_len, (int)threadIdx.x - 32};
        double pre[HG_NLD];
        if (nchunk > 0) ld.fetch(lik, 0, pre);
        for (int c = 0; c <= nchunk; c++) {
            if (c < nchunk) {
                const int b = c & 1;
                if (c >= 2) sync_solved(b);  // the solver is done with chunk c - 2 in this buffer
                ld.store(pre, em[b]);
                if (c + 1 < nchunk) ld.fetch(lik, c + 1, pre);  // in flight under this chunk's work
                emit<LG>(ld, c, em[b], is_log);
                arrive_ready(b);
            } else {
                for (int k = max(0, nchunk - 2); k < nchunk; k++) sync_solved(k & 1);  // every arrival is consumed
            }
        }
    } else {
        const int lane = threadIdx.x;
        const int64_t n = s_len[lane];
        const int tb = tb0 + lane;
        const double one = LG ? 0.0 : 1.0;
        double a0 = one, a1 = one, a2 = one;
        for (int c = 0; c < nchunk; c++) {
            const int b = c & 1;
            sync_ready(b);
            const int64_t i0 = (int64_t)c * HG_BINS;
            const double *nr = &em[b][lane][0];
#pragma unroll 4
            for (int q = 0; q < HG_BINS; q++)
                fwd_step<LG>(a0, a1, a2, nr[q * 3], nr[q * 3 + 1], nr[q * 3 + 2], i0 + q == 0, i0 + q < n, p01, p02, p12);
            if (tb < n_tables) {
                double *o = ckpt + ((size_t)c * n_tables + tb) * 3;
                o[0] = a0; o[1] = a1; o[2] = a2;
            }
            __threadfence_block();
            arrive_solved(b);
        }
        if (tb < n_tables) expected[(size_t)tb * 3] = LG ? (fmax(a0, fmax(a1, a2)) > -INFINITY ? 1.0 : 0.0) : a0 + a1 + a2;
    }
}

// Backward pass: gamma -> posterior (the caller's layout), expected occupancy -> expected[t][3].  MOM: the solver
// also carries the moment recursion (moment_step) and sums each table's cross terms in bin order, from the last bin
// down, into cov[t][3][3]; posterior may then be null (nothing per bin is written).  The workers' gamma, posterior and
// expected are those of the plain pass, bit for bit.
template <bool LG, bool MOM = false>
__global__ void __launch_bounds__(HG_THREADS, 3)
posterior_bwd_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const double *__restrict__ lik,
                     int is_log, double p01, double p02, double p12, const double *__restrict__ ckpt, double *__restrict__ posterior,
                     double *__restrict__ expected, double *__restrict__ cov = nullptr) {
    extern __shared__ double pb_smem[];
    double (*em)[HG_TABLES][HG_ROW] = reinterpret_cast<double (*)[HG_TABLES][HG_ROW]>(pb_smem);  // emissions, then beta
    double (*al)[HG_TABLES][HG_ROW] = reinterpret_cast<double (*)[HG_TABLES][HG_ROW]>(pb_smem + 2 * HG_TABLES * HG_ROW);
    int64_t *s_start = reinterpret_cast<int64_t *>(pb_smem + 4 * HG_TABLES * HG_ROW), *s_len = s_start + HG_TABLES;
    int *s_dead = reinterpret_cast<int *>(s_len + HG_TABLES);
    const int tb0 = blockIdx.x * HG_TABLES;
    if (threadIdx.x < HG_TABLES) {
        const int tb = tb0 + threadIdx.x;
        s_dead[threadIdx.x] = tb < n_tables && len[tb] > 0 && !(expected[(size_t)tb * 3] > 0);  // total weight 0
    }
    const int nchunk = block_tables(n_tables, start, len, s_start, s_len);
    const int w = (int)threadIdx.x - 32;
    double E[HG_NBIN][3] = {};  // a worker's share of the expected counts: the same (table, bin slot) every chunk
    double mu[2][3] = {}, mc[6] = {};  // MOM, solver lane: u of the bin below, the table's cross-term sums
    if (threadIdx.x >= 32) {
        const ChunkLoader ld{s_start, s_len, w};
        double pre[HG_NLD];
        if (nchunk > 0) ld.fetch(lik, nchunk - 1, pre);
        for (int r = 0; r <= nchunk; r++) {  // r-th chunk from the end
            if (r < nchunk) {
                const int c = nchunk - 1 - r, b = r & 1;
                ld.store(pre, em[b]);
                if (c >= 1) ld.fetch(lik, c - 1, pre);  // in flight under this chunk's work
                emit<LG>(ld, c, em[b], is_log);
                arrive_ready(b);
            }
            if (r >= 1) {  // gamma of the chunk the solver has just finished
                const int c = nchunk - r, pb = (r - 1) & 1;
                sync_solved(pb);
                const int64_t i0 = (int64_t)c * HG_BINS;
#pragma unroll
                for (int k = 0; k < HG_NBIN; k++) {
                    const int idx = k * HG_WORKERS + w;
                    const int t = idx / HG_BINS, i = idx % HG_BINS;
                    if (i0 + i < s_len[t]) {
                        double y0, y1, y2;
                        gamma<LG>(&al[pb][t][i * 3], &em[pb][t][i * 3], s_dead[t], y0, y1, y2);
                        if (!MOM || posterior) {
                            double *o = posterior + (s_start[t] + i0 + i) * 3;
                            __stcs(o, y0);
                            __stcs(o + 1, y1);
                            __stcs(o + 2, y2);
                        }
                        E[k][0] += y0;
                        E[k][1] += y1;
                        E[k][2] += y2;
                    }
                }
                sync_workers();  // buffer pb is free for the next chunk
            }
        }
    } else {
        const int lane = threadIdx.x;
        const int64_t n = s_len[lane];
        const int tb = tb0 + lane;
        const double one = LG ? 0.0 : 1.0;
        double b0 = one, b1 = one, b2 = one;
        for (int r = 0; r < nchunk; r++) {
            const int c = nchunk - 1 - r, b = r & 1;
            double a0 = one, a1 = one, a2 = one;  // alpha entering the chunk: the previous chunk's checkpoint
            if (c >= 1 && tb < n_tables) {
                const double *ck = ckpt + ((size_t)(c - 1) * n_tables + tb) * 3;
                a0 = ck[0]; a1 = ck[1]; a2 = ck[2];
            }
            sync_ready(b);
            const int64_t i0 = (int64_t)c * HG_BINS;
            double *nr = &em[b][lane][0], *ao = &al[b][lane][0];
#pragma unroll 4
            for (int q = 0; q < HG_BINS; q++) {
                fwd_step<LG>(a0, a1, a2, nr[q * 3], nr[q * 3 + 1], nr[q * 3 + 2], i0 + q == 0, i0 + q < n, p01, p02, p12);
                ao[q * 3] = a0; ao[q * 3 + 1] = a1; ao[q * 3 + 2] = a2;
            }
            // beta down the chunk: the slot of bin i trades its emission for beta[i], then beta[i - 1]
            if (!MOM) {
#pragma unroll 4
                for (int q = HG_BINS - 1; q >= 0; q--) {
                    const double e0 = nr[q * 3], e1 = nr[q * 3 + 1], e2 = nr[q * 3 + 2];
                    nr[q * 3] = b0; nr[q * 3 + 1] = b1; nr[q * 3 + 2] = b2;
                    bwd_step<LG>(b0, b1, b2, e0, e1, e2, i0 + q < n, p01, p02, p12);
                }
            } else {
                const bool dead = s_dead[lane];
#pragma unroll 1
                for (int q = HG_BINS - 1; q >= 0; q--) {
                    const double e0 = nr[q * 3], e1 = nr[q * 3 + 1], e2 = nr[q * 3 + 2];
                    nr[q * 3] = b0; nr[q * 3 + 1] = b1; nr[q * 3 + 2] = b2;
                    if (i0 + q < n) {  // the bin's cross terms with u of bin i, then u of bin i - 1
                        double y0, y1, y2;
                        gamma<LG>(&ao[q * 3], &nr[q * 3], dead, y0, y1, y2);
                        moment_acc(mc, mu, y0, y1, y2);
                        moment_step<LG>(mu, e0, e1, e2, b0, b1, b2, p01, p02, p12);
                    }
                    bwd_step<LG>(b0, b1, b2, e0, e1, e2, i0 + q < n, p01, p02, p12);
                }
            }
            __threadfence_block();
            arrive_solved(b);
        }
    }
    __syncthreads();
    // expected[t] = the 16 bin slots' partial sums of table t, added in a fixed order (reproducible)
    double *part = &em[0][0][0];  // [HG_TABLES][HG_BINS][3]
    if (threadIdx.x >= 32) {
#pragma unroll
        for (int k = 0; k < HG_NBIN; k++) {
            const int idx = k * HG_WORKERS + w;
            const int t = idx / HG_BINS, i = idx % HG_BINS;
#pragma unroll
            for (int s = 0; s < 3; s++) part[(t * HG_BINS + i) * 3 + s] = E[k][s];
        }
    }
    __syncthreads();
    if (threadIdx.x < HG_TABLES) {
        const int tb = tb0 + threadIdx.x;
        if (tb < n_tables) {
            double x[3] = {0, 0, 0};
            for (int i = 0; i < HG_BINS; i++)
                for (int s = 0; s < 3; s++) x[s] += part[(threadIdx.x * HG_BINS + i) * 3 + s];
            const double nan = __longlong_as_double(0x7ff8000000000000LL);
            for (int s = 0; s < 3; s++) expected[(size_t)tb * 3 + s] = s_dead[threadIdx.x] ? nan : x[s];
            if (MOM) {  // this thread is the table's solver lane: its own sums
                double *o = cov + (size_t)tb * 9;
                const int ix[9] = {0, 1, 2, 1, 3, 4, 2, 4, 5};
#pragma unroll
                for (int k = 0; k < 9; k++) o[k] = s_dead[threadIdx.x] ? nan : mc[ix[k]];
            }
        }
    }
}

}  // namespace ibdgem

using namespace ibdgem;

bool ibdgem::bad_penalties(const char *fn, double p01, double p02, double p12) {
    const bool ok = std::isfinite(p01) && std::isfinite(p02) && std::isfinite(p12) && p01 >= 0 && p02 >= 0 && p12 >= 0;
    if (!ok) set_error("[::] ERROR in %s(): penalties must be finite and >= 0 (p01 = %g, p02 = %g, p12 = %g).", fn, p01, p02, p12);
    return !ok;
}

namespace {

// The linear-space kernels are exact to far below 1e-9 when every entry of the penalty matrix (1 on the diagonal) is
// within a factor r = max(1, p) / min(1, p) <= 2^400 of every other.  Mixing keeps each alpha / beta entry above
// 1/r of its row's share, so an entry flushed below 2^-1074 of its row, or an emission clipped below e^-700, moves
// the next row by at most a relative 3 * 2^-1073 * r, or 3 * e^-700 * r^2 = 3 * 2^-210; such perturbations do not
// grow along the table.  Rows stay within [2^-460, 2^403] before rescaling.  Zero penalties, and spreads above
// 2^400, go to the same kernels in natural-log arithmetic, which has no range limit.
bool linear_penalties(double p01, double p02, double p12) {
    const double lo = std::min({1.0, p01, p02, p12}), hi = std::max({1.0, p01, p02, p12});
    return lo > 0 && hi / lo <= 0x1p400;
}

}  // namespace

// One batch of tables, everything in device memory (start / len per table); kernels only, no host synchronisation.
int ibdgem::posterior_on_device(ibdgem_engine *e, int n_tables, int64_t maxbins, const int64_t *d_start, const int64_t *d_len, const double *d_lik,
                        int is_log, double p01, double p02, double p12, double *d_post, double *d_expected, double *d_cov) {
    const int64_t nck = (maxbins + HG_BINS - 1) / HG_BINS;
    if (nck == 0) {  // only empty tables: no bins, expected occupancy 0 (and covariance 0)
        IBD_CUDA(cudaMemsetAsync(d_expected, 0, (size_t)n_tables * 24, e->stream));
        if (d_cov) IBD_CUDA(cudaMemsetAsync(d_cov, 0, (size_t)n_tables * 72, e->stream));
        return 0;
    }
    double *d_ckpt;
    if (scratch(e, SC_HG_CKPT, (size_t)nck * n_tables * 24, (void **)&d_ckpt)) return 1;
    const unsigned grid = (unsigned)((n_tables + HG_TABLES - 1) / HG_TABLES);
    if (linear_penalties(p01, p02, p12)) {
        {
            LaunchScope ls(e, K_POSTERIOR_FWD);
            posterior_fwd_kernel<false><<<grid, HG_THREADS, PB_FWD_SMEM, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, p01, p02, p12,
                                                                                      d_ckpt, d_expected);
        }
        if (d_cov) {
            LaunchScope ls(e, K_POSTERIOR_BWD_MOMENTS);
            IBD_CUDA(cudaFuncSetAttribute(posterior_bwd_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PB_BWD_SMEM));
            posterior_bwd_kernel<false, true><<<grid, HG_THREADS, PB_BWD_SMEM, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, p01, p02,
                                                                                            p12, d_ckpt, d_post, d_expected, d_cov);
        } else {
            LaunchScope ls(e, K_POSTERIOR_BWD);
            IBD_CUDA(cudaFuncSetAttribute(posterior_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PB_BWD_SMEM));
            posterior_bwd_kernel<false><<<grid, HG_THREADS, PB_BWD_SMEM, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, p01, p02, p12,
                                                                                      d_ckpt, d_post, d_expected);
        }
    } else {
        const double l01 = log(p01), l02 = log(p02), l12 = log(p12);  // log(0) = -inf: a forbidden transition
        {
            LaunchScope ls(e, K_POSTERIOR_FWD);
            e->k_launches[K_POSTERIOR_FWD_LOG]++;
            posterior_fwd_kernel<true><<<grid, HG_THREADS, PB_FWD_SMEM, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, l01, l02, l12,
                                                                                     d_ckpt, d_expected);
        }
        if (d_cov) {
            LaunchScope ls(e, K_POSTERIOR_BWD_MOMENTS);
            e->k_launches[K_POSTERIOR_BWD_LOG]++;
            IBD_CUDA(cudaFuncSetAttribute(posterior_bwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PB_BWD_SMEM));
            posterior_bwd_kernel<true, true><<<grid, HG_THREADS, PB_BWD_SMEM, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, l01, l02,
                                                                                           l12, d_ckpt, d_post, d_expected, d_cov);
        } else {
            LaunchScope ls(e, K_POSTERIOR_BWD);
            e->k_launches[K_POSTERIOR_BWD_LOG]++;
            IBD_CUDA(cudaFuncSetAttribute(posterior_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PB_BWD_SMEM));
            posterior_bwd_kernel<true><<<grid, HG_THREADS, PB_BWD_SMEM, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, l01, l02, l12,
                                                                                     d_ckpt, d_post, d_expected);
        }
    }
    IBD_CUDA(cudaGetLastError());
    return 0;
}

// Host buffers in, host buffers out: the likelihoods go up, both passes run, posteriors and expected counts come down.
extern "C" int hiddengem_posterior_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik, int32_t is_log,
                                         double p01, double p02, double p12, double *posterior, double *expected) {
    if (!e || n_tables <= 0 || !bin_offsets || !expected) {
        set_error("[::] ERROR in hiddengem_posterior_batch(): bad arguments.");
        return 1;
    }
    if (bad_penalties("hiddengem_posterior_batch", p01, p02, p12)) return 1;
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_posterior_batch", n_tables, bin_offsets, 0, &h_sl, &maxbins, &total)) return 1;
    const int64_t nb = total > 0 ? bin_offsets[n_tables] : 0;  // bins of lik / posterior
    if (nb > 0 && (!lik || !posterior)) {
        set_error("[::] ERROR in hiddengem_posterior_batch(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    double *d_lik = nullptr, *d_post = nullptr, *d_expected;
    int64_t *d_start;
    if (scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start) || scratch(e, SC_HG_COUNTS, (size_t)n_tables * 24, (void **)&d_expected))
        return 1;
    if (nb > 0 && (scratch(e, SC_HG_LIK, (size_t)nb * 24, (void **)&d_lik) || scratch(e, SC_HG_SCORE, (size_t)nb * 24, (void **)&d_post)))
        return 1;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    if (nb > 0) IBD_CUDA(cudaMemcpyAsync(d_lik, lik, (size_t)nb * 24, cudaMemcpyHostToDevice, e->stream));
    if (posterior_on_device(e, n_tables, maxbins, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_post, d_expected)) return 1;
    if (nb > 0) IBD_CUDA(cudaMemcpyAsync(posterior, d_post, (size_t)nb * 24, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaMemcpyAsync(expected, d_expected, (size_t)n_tables * 24, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    settle_timers(e);
    return 0;
}

// Device buffers in, device buffers out; bin_offsets is a HOST array.  table_stride > 0: table t starts at bin
// t * table_stride (ibdgem_scores.w_loglik_device with table_stride = max_windows), and its posteriors are written at
// the same positions.
extern "C" int hiddengem_posterior_batch_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                                const double *d_lik, int32_t is_log, double p01, double p02, double p12, double *d_posterior,
                                                double *d_expected) {
    if (!e || n_tables <= 0 || !bin_offsets || !d_lik || !d_posterior || !d_expected || table_stride < 0) {
        set_error("[::] ERROR in hiddengem_posterior_batch_device(): bad arguments.");
        return 1;
    }
    if (bad_penalties("hiddengem_posterior_batch_device", p01, p02, p12)) return 1;
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_posterior_batch_device", n_tables, bin_offsets, table_stride, &h_sl, &maxbins, &total)) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    int64_t *d_start;
    if (scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start)) return 1;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    if (posterior_on_device(e, n_tables, maxbins, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_posterior, d_expected)) return 1;
    IBD_CUDA(cudaStreamSynchronize(e->stream));  // h_sl is read by the copy above
    settle_timers(e);
    return 0;
}

// Posterior moments: the posterior pass with the moment variant of the backward kernel.  Host buffers in, host
// buffers out; without posterior (null) only the 96 B of expected + cov per table come back.
extern "C" int hiddengem_posterior_moments_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik,
                                                 int32_t is_log, double p01, double p02, double p12, double *posterior, double *expected,
                                                 double *cov) {
    if (!e || n_tables <= 0 || !bin_offsets || !expected || !cov) {
        set_error("[::] ERROR in hiddengem_posterior_moments_batch(): bad arguments.");
        return 1;
    }
    if (bad_penalties("hiddengem_posterior_moments_batch", p01, p02, p12)) return 1;
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_posterior_moments_batch", n_tables, bin_offsets, 0, &h_sl, &maxbins, &total)) return 1;
    const int64_t nb = total > 0 ? bin_offsets[n_tables] : 0;  // bins of lik / posterior
    if (nb > 0 && !lik) {
        set_error("[::] ERROR in hiddengem_posterior_moments_batch(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    double *d_lik = nullptr, *d_post = nullptr, *d_out;
    int64_t *d_start;
    if (scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start) || scratch(e, SC_HG_COUNTS, (size_t)n_tables * 96, (void **)&d_out))
        return 1;
    if (nb > 0 && scratch(e, SC_HG_LIK, (size_t)nb * 24, (void **)&d_lik)) return 1;
    if (nb > 0 && posterior && scratch(e, SC_HG_SCORE, (size_t)nb * 24, (void **)&d_post)) return 1;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    if (nb > 0) IBD_CUDA(cudaMemcpyAsync(d_lik, lik, (size_t)nb * 24, cudaMemcpyHostToDevice, e->stream));
    double *d_cov = d_out + (size_t)n_tables * 3;
    if (posterior_on_device(e, n_tables, maxbins, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_post, d_out, d_cov)) return 1;
    if (d_post) IBD_CUDA(cudaMemcpyAsync(posterior, d_post, (size_t)nb * 24, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaMemcpyAsync(expected, d_out, (size_t)n_tables * 24, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaMemcpyAsync(cov, d_cov, (size_t)n_tables * 72, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    settle_timers(e);
    return 0;
}

// Device buffers in, device buffers out (d_posterior may be null); bin_offsets is a HOST array, table_stride as for
// hiddengem_posterior_batch_device.
extern "C" int hiddengem_posterior_moments_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                                  const double *d_lik, int32_t is_log, double p01, double p02, double p12, double *d_posterior,
                                                  double *d_expected, double *d_cov) {
    if (!e || n_tables <= 0 || !bin_offsets || !d_lik || !d_expected || !d_cov || table_stride < 0) {
        set_error("[::] ERROR in hiddengem_posterior_moments_device(): bad arguments.");
        return 1;
    }
    if (bad_penalties("hiddengem_posterior_moments_device", p01, p02, p12)) return 1;
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_posterior_moments_device", n_tables, bin_offsets, table_stride, &h_sl, &maxbins, &total)) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    int64_t *d_start;
    if (scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start)) return 1;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    if (posterior_on_device(e, n_tables, maxbins, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_posterior, d_expected, d_cov))
        return 1;
    IBD_CUDA(cudaStreamSynchronize(e->stream));  // h_sl is read by the copy above
    settle_timers(e);
    return 0;
}
