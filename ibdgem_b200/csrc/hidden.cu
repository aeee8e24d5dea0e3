// hidden.cu — batched hiddengem: three-state Viterbi over per-window likelihoods (H1-H3,
// src/hiddengem.c:51-147, 246-283), one summary table per thread, in fp64 log space.
//
// The reference keeps running PRODUCTS of normalised likelihoods in x87 long double
// (src/hiddengem.c:43, 110-141); here the same recurrence runs on log values, so
//   score[s][i] = max_k ( (score[k][i-1] + ln nrm[s][i]) + ln pen(k,s) )
// with the reference's strict-'>' argmax (lowest index wins ties, NaN never wins,
// src/hiddengem.c:91-99).  Zeros become -inf and NaN rows (0/0, src/hiddengem.c:74-76)
// propagate exactly as they do through the products.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <thread>
#include <vector>

#include "engine.h"
#include "hg_block.cuh"
#include "tc_common.cuh"

namespace ibdgem {

constexpr uint8_t FROM_SELF = 0 | (1 << 2) | (2 << 4);  // back-pointers of bin 0: every state from itself

__device__ __forceinline__ int argmax3(const double *c) {
    int b = 0;
    double v = c[0];
    if (c[1] > v) { b = 1; v = c[1]; }
    if (c[2] > v) { b = 2; }
    return b;
}
__device__ __forceinline__ double pick3(const double *c, int k) { return k == 0 ? c[0] : (k == 1 ? c[1] : c[2]); }

// c[s][k] = (prev_k + ln nrm_s) + ln pen(k, s), the candidates of state s; the diagonal has no penalty factor
__device__ __forceinline__ void candidates(const double *p, const double *n, double lp01, double lp02, double lp12, double (&c)[3][3]) {
    c[0][0] = p[0] + n[0], c[0][1] = (p[1] + n[0]) + lp01, c[0][2] = (p[2] + n[0]) + lp02;
    c[1][0] = (p[0] + n[1]) + lp01, c[1][1] = p[1] + n[1], c[1][2] = (p[2] + n[1]) + lp12;
    c[2][0] = (p[0] + n[2]) + lp02, c[2][1] = (p[1] + n[2]) + lp12, c[2][2] = p[2] + n[2];
}

// ln nrm = ln of the normalised likelihoods of one bin.  FAST_EXP: exp_nonpos (arguments are <= 0, degree-12
// polynomial, error ~1 ulp, half the instructions of exp()) for the batched kernel; viterbi_kernel keeps libm exp.
template <bool FAST_EXP>
__device__ __forceinline__ void ln_nrm(const double *L, int is_log, double *n) {
    if (is_log) {  // ln nrm = ll - logsumexp(ll)
        const double m = fmax(L[0], fmax(L[1], L[2]));
        if (m == -INFINITY) {
            n[0] = n[1] = n[2] = __longlong_as_double(0x7ff8000000000000LL);  // 0/0 in the reference
        } else {
            const double z = FAST_EXP ? m + log(exp_nonpos(L[0] - m) + exp_nonpos(L[1] - m) + exp_nonpos(L[2] - m))
                                      : m + log(exp(L[0] - m) + exp(L[1] - m) + exp(L[2] - m));
            n[0] = L[0] - z; n[1] = L[1] - z; n[2] = L[2] - z;
        }
    } else {  // src/hiddengem.c:74-76: l_s / (l0 + l1 + l2) in fp64, then the log
        const double tot = __dadd_rn(__dadd_rn(L[0], L[1]), L[2]);
        n[0] = log(__ddiv_rn(L[0], tot));
        n[1] = log(__ddiv_rn(L[1], tot));
        n[2] = log(__ddiv_rn(L[2], tot));
    }
}

// Near-tie guard.  The reference multiplies x87 long doubles (src/hiddengem.c:110-141); sums of fp64 logs carry a
// rounding error of up to ~i * 2^-53 * |score| after i bins, so an arg-max whose winner leads the runner-up by less
// than that could come out differently.  Such tables (and, on the text path, tables whose scores leave the range
// of a normal long double, where the reference's products lose bits and then vanish) are flagged and re-evaluated
// on the host in long double.  NaN / -inf candidates never flag: their comparisons are exact in both worlds.
constexpr double LN_LDBL_MIN = -11355.137111933024;  // ln(3.3621e-4932)
__device__ __forceinline__ double tie_scale(int64_t i) { return (double)(int)(i + 1) * 4.440892098500626e-16; }  // 4 (i + 1) 2^-53
__device__ __forceinline__ bool near_tie(const double *c, int best, double scale) {
    const double w = pick3(c, best);
    const double r = best == 0 ? fmax(c[1], c[2]) : (best == 1 ? fmax(c[0], c[2]) : fmax(c[0], c[1]));
    return (w - r) < fma(scale, fabs(w), 1e-12);  // false for NaN and for inf - inf
}
// a finite score below the smallest normal long double: the reference's product is a denormal (or zero) there
__device__ __forceinline__ bool below_ldbl(const double *s) {
    return (s[0] < LN_LDBL_MIN && s[0] > -INFINITY) || (s[1] < LN_LDBL_MIN && s[1] > -INFINITY) || (s[2] < LN_LDBL_MIN && s[2] > -INFINITY);
}

// One table per thread, for small or ragged batches.
__global__ void __launch_bounds__(128)
viterbi_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const double *__restrict__ lik, int is_log,
               double lp01, double lp02, double lp12, uint8_t *__restrict__ state,
               double *__restrict__ score, long long *__restrict__ counts, uint8_t *__restrict__ flag) {
    const int tb = blockIdx.x * blockDim.x + threadIdx.x;
    if (tb >= n_tables) return;
    const int64_t b0 = start[tb];
    const int64_t n = len[tb];
    if (n <= 0) {
        counts[tb * 3 + 0] = counts[tb * 3 + 1] = counts[tb * 3 + 2] = 0;
        flag[tb] = 0;
        return;
    }
    double s[3] = {0, 0, 0};
    bool tie = false;
    for (int64_t i = 0; i < n; i++) {
        double nv[3];
        ln_nrm<false>(lik + (b0 + i) * 3, is_log, nv);
        uint8_t from;
        if (i == 0) {  // src/hiddengem.c:112-118
            s[0] = nv[0]; s[1] = nv[1]; s[2] = nv[2];
            from = FROM_SELF;
        } else {
            double c[3][3];
            candidates(s, nv, lp01, lp02, lp12, c);
            const int k0 = argmax3(c[0]), k1 = argmax3(c[1]), k2 = argmax3(c[2]);
            const double ts = tie_scale(i);
            tie |= near_tie(c[0], k0, ts) | near_tie(c[1], k1, ts) | near_tie(c[2], k2, ts);
            s[0] = pick3(c[0], k0);
            s[1] = pick3(c[1], k1);
            s[2] = pick3(c[2], k2);
            from = (uint8_t)(k0 | (k1 << 2) | (k2 << 4));
        }
        if (!is_log) tie |= below_ldbl(s);
        state[b0 + i] = from;
        double *o = score + (b0 + i) * 3;
        o[0] = s[0]; o[1] = s[1]; o[2] = s[2];
    }
    int cur = argmax3(s);  // src/hiddengem.c:246-249
    tie |= near_tie(s, cur, tie_scale(n));
    long long c[3] = {0, 0, 0};
    for (int64_t i = n - 1; i >= 0; i--) {  // src/hiddengem.c:252-257
        const uint8_t from = state[b0 + i];
        state[b0 + i] = (uint8_t)cur;
        c[cur]++;
        cur = (from >> (2 * cur)) & 3;
    }
    counts[tb * 3 + 0] = c[0];
    counts[tb * 3 + 1] = c[1];
    counts[tb * 3 + 2] = c[2];
    flag[tb] = tie ? 1 : 0;
}

// ---------------------------------------------------------------------------------------------
// Batched pipeline for many tables (C4: 10,000 tables x 10,000 bins), three kernels: the fused forward pass, the
// back-trace, and the states back to the caller's layout.
//
// Fused forward pass: one read of the likelihoods, one write of the scores, on the chunked block of hg_block.cuh.
// The workers turn each chunk's likelihoods into ln nrm in shared memory — that is where the fp64 exp / log work is,
// and it is parallel over bins; the solver walks the recursion.  The arithmetic is that of viterbi_kernel, operation
// for operation.  Back-pointers leave bin-major (coalesced over tables) for viterbi_back_kernel; scores leave in the
// caller's table-major layout.
constexpr int VF_SMEM = 4 * HG_TABLES * HG_ROW * 8 + HG_HEAD_SMEM + 2 * HG_TABLES * 3 * 8 + HG_TABLES * 4 + 2 * HG_BINS * HG_TABLES;

// The solver's walk over one chunk (lane = table, nq = bins of the table in the chunk, <= 0: none).  A single warp
// walks the bins, so its time is (instructions per bin) x (issue latency): the step is branch-free.  FIRST: chunk 0,
// whose bin 0 takes s = ln nrm and the identity back-pointers, as in viterbi_kernel.
template <bool FIRST>
__device__ __forceinline__ void solve_chunk(const double *nr, double *so, uint8_t (*frm)[HG_TABLES], int lane, int nq, double lp01,
                                            double lp02, double lp12, double (&s)[3]) {
    if (FIRST) {
        s[0] = nr[0]; s[1] = nr[1]; s[2] = nr[2];
        so[0] = s[0]; so[1] = s[1]; so[2] = s[2];
        frm[0][lane] = FROM_SELF;
    }
#pragma unroll 4
    for (int q = FIRST ? 1 : 0; q < HG_BINS; q++) {
        double c[3][3];
        candidates(s, nr + q * 3, lp01, lp02, lp12, c);
        // strict '>' arg-max: lowest index wins, NaN never wins
        const bool ga = c[0][1] > c[0][0], gb = c[1][1] > c[1][0], gc = c[2][1] > c[2][0];
        const double ma = ga ? c[0][1] : c[0][0], mb = gb ? c[1][1] : c[1][0], mc = gc ? c[2][1] : c[2][0];
        const bool ha = c[0][2] > ma, hb = c[1][2] > mb, hc = c[2][2] > mc;
        const bool live = q < nq;
        s[0] = live ? (ha ? c[0][2] : ma) : s[0];
        s[1] = live ? (hb ? c[1][2] : mb) : s[1];
        s[2] = live ? (hc ? c[2][2] : mc) : s[2];
        so[q * 3] = s[0];
        so[q * 3 + 1] = s[1];
        so[q * 3 + 2] = s[2];
        frm[q][lane] = (uint8_t)((ha ? 2 : (int)ga) | ((hb ? 2 : (int)gb) << 2) | ((hc ? 2 : (int)gc) << 4));
    }
}

__global__ void __launch_bounds__(HG_THREADS, 3)
viterbi_fused_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const double *__restrict__ lik,
                     int is_log, double lp01, double lp02, double lp12, double *__restrict__ score,
                     uint8_t *__restrict__ fromT /*[maxbins][n_tables]*/, double *__restrict__ last /*[n_tables][3]*/,
                     uint8_t *__restrict__ flag) {
    extern __shared__ double vf_smem[];
    double (*nrm)[HG_TABLES][HG_ROW] = reinterpret_cast<double (*)[HG_TABLES][HG_ROW]>(vf_smem);
    double (*sco)[HG_TABLES][HG_ROW] = reinterpret_cast<double (*)[HG_TABLES][HG_ROW]>(vf_smem + 2 * HG_TABLES * HG_ROW);
    int64_t *s_start = reinterpret_cast<int64_t *>(vf_smem + 4 * HG_TABLES * HG_ROW), *s_len = s_start + HG_TABLES;
    double (*prevlast)[HG_TABLES][3] = reinterpret_cast<double (*)[HG_TABLES][3]>(s_len + HG_TABLES);  // last bin's scores of a chunk
    int *tieflag = reinterpret_cast<int *>(&prevlast[2][0][0]);
    uint8_t (*frm)[HG_BINS][HG_TABLES] = reinterpret_cast<uint8_t (*)[HG_BINS][HG_TABLES]>(tieflag + HG_TABLES);
    const int tb0 = blockIdx.x * HG_TABLES;
    if (threadIdx.x < HG_TABLES) tieflag[threadIdx.x] = 0;
    const int nchunk = block_tables(n_tables, start, len, s_start, s_len);
    if (threadIdx.x >= 32) {
        // ===== workers =====
        const int w = threadIdx.x - 32;
        const ChunkLoader ld{s_start, s_len, w};
        // raw likelihoods of the NEXT chunk are fetched before this chunk's exp / log work starts, so DRAM latency
        // hides under it
        double pre[HG_NLD];
        if (nchunk > 0) ld.fetch(lik, 0, pre);
        for (int c = 0; c <= nchunk; c++) {
            const int b = c & 1;
            if (c < nchunk) {
                const int64_t i0 = (int64_t)c * HG_BINS;
                ld.store(pre, nrm[b]);
                if (c + 1 < nchunk) ld.fetch(lik, c + 1, pre);
                sync_workers();
                // ln nrm in place: 512 bins, 2 per worker
#pragma unroll
                for (int k = 0; k < HG_NBIN; k++) {
                    const int idx = k * HG_WORKERS + w;
                    const int t = idx / HG_BINS, i = idx % HG_BINS;
                    if (i0 + i < s_len[t]) {
                        const double v[3] = {nrm[b][t][i * 3], nrm[b][t][i * 3 + 1], nrm[b][t][i * 3 + 2]};
                        ln_nrm<true>(v, is_log, &nrm[b][t][i * 3]);
                    }
                }
                __threadfence_block();
                arrive_ready(b);
            }
            if (c >= 1) {  // drain the chunk the solver has just finished
                const int pb = (c - 1) & 1;
                sync_solved(pb);
                const int64_t i0 = (int64_t)(c - 1) * HG_BINS;
                // Near-tie and long-double-range tests, moved off the solver's critical path: with the scores of bin
                // i - 1 and ln nrm of bin i both still in shared memory, every bin's nine candidates can be rebuilt
                // independently (the same expressions, hence the same doubles) — 512 bins over 256 workers.
#pragma unroll
                for (int k = 0; k < HG_NBIN; k++) {
                    const int idx = k * HG_WORKERS + w;
                    const int t = idx / HG_BINS, i = idx % HG_BINS;
                    const int64_t gi = i0 + i;
                    if (gi < s_len[t]) {
                        const double *cur = &sco[pb][t][i * 3];
                        bool tie = !is_log && below_ldbl(cur);
                        if (gi > 0) {
                            const double *pv = i > 0 ? &sco[pb][t][(i - 1) * 3] : &prevlast[pb ^ 1][t][0];
                            const double p[3] = {pv[0], pv[1], pv[2]};
                            const double nv[3] = {nrm[pb][t][i * 3], nrm[pb][t][i * 3 + 1], nrm[pb][t][i * 3 + 2]};
                            const double ts = tie_scale(gi);
                            double cd[3][3];
                            candidates(p, nv, lp01, lp02, lp12, cd);
                            tie |= near_tie(cd[0], argmax3(cd[0]), ts) | near_tie(cd[1], argmax3(cd[1]), ts) |
                                   near_tie(cd[2], argmax3(cd[2]), ts);
                        }
                        if (tie) tieflag[t] = 1;
                        if (i == HG_BINS - 1) { prevlast[pb][t][0] = cur[0]; prevlast[pb][t][1] = cur[1]; prevlast[pb][t][2] = cur[2]; }
                    }
                }
                ld.write(c - 1, sco[pb], score);
#pragma unroll
                for (int k = 0; k < HG_NBIN; k++) {
                    const int idx = k * HG_WORKERS + w;
                    const int i = idx / HG_TABLES, t = idx % HG_TABLES;
                    if (tb0 + t < n_tables && i0 + i < s_len[t]) fromT[(size_t)(i0 + i) * n_tables + tb0 + t] = frm[pb][i][t];
                }
                sync_workers();  // buffer pb is free for chunk c + 1
            }
        }
    } else {
        // ===== solver: lane = table =====
        const int lane = threadIdx.x;
        const int64_t n = s_len[lane];
        double s[3] = {0, 0, 0};
        for (int c = 0; c < nchunk; c++) {
            const int b = c & 1;
            sync_ready(b);
            const int nq = (int)min((int64_t)HG_BINS, n - (int64_t)c * HG_BINS);
            if (c == 0) solve_chunk<true>(&nrm[b][lane][0], &sco[b][lane][0], frm[b], lane, nq, lp01, lp02, lp12, s);
            else solve_chunk<false>(&nrm[b][lane][0], &sco[b][lane][0], frm[b], lane, nq, lp01, lp02, lp12, s);
            __threadfence_block();
            arrive_solved(b);
        }
        const int tb = tb0 + lane;
        if (tb < n_tables) {
            last[(size_t)tb * 3 + 0] = s[0];
            last[(size_t)tb * 3 + 1] = s[1];
            last[(size_t)tb * 3 + 2] = s[2];
        }
    }
    __syncthreads();  // the workers' last drain has set the tie flags
    if (threadIdx.x < HG_TABLES) {
        const int tb = tb0 + threadIdx.x;
        if (tb < n_tables) {
            const int64_t n = s_len[threadIdx.x];
            bool tie = tieflag[threadIdx.x] != 0;
            if (n > 0) {
                const double l[3] = {last[(size_t)tb * 3], last[(size_t)tb * 3 + 1], last[(size_t)tb * 3 + 2]};
                tie |= near_tie(l, argmax3(l), tie_scale(n));
            }
            flag[tb] = tie ? 1 : 0;
        }
    }
}

// back-trace, thread = table; the state overwrites the back-pointer byte in place
__global__ void __launch_bounds__(64)
viterbi_back_kernel(int n_tables, const int64_t *__restrict__ len, uint8_t *__restrict__ fromT, const double *__restrict__ last,
                    long long *__restrict__ counts) {
    const int tb = blockIdx.x * blockDim.x + threadIdx.x;
    if (tb >= n_tables) return;
    const int64_t n = len[tb];
    const size_t nT = (size_t)n_tables;
    long long c0 = 0, c1 = 0, c2 = 0;
    if (n > 0) {
        int cur = argmax3(last + (size_t)tb * 3);
        constexpr int BU = 32;
        for (int64_t ib = n; ib > 0; ib -= BU) {
            uint8_t f[BU];
#pragma unroll
            for (int u = 0; u < BU; u++)
                if (ib - 1 - u >= 0) f[u] = fromT[(size_t)(ib - 1 - u) * nT + tb];
#pragma unroll
            for (int u = 0; u < BU; u++) {
                const int64_t i = ib - 1 - u;
                if (i < 0) break;
                fromT[(size_t)i * nT + tb] = (uint8_t)cur;
                c0 += cur == 0; c1 += cur == 1; c2 += cur == 2;
                cur = (f[u] >> (2 * cur)) & 3;
            }
        }
    }
    counts[tb * 3 + 0] = c0;
    counts[tb * 3 + 1] = c1;
    counts[tb * 3 + 2] = c2;
}

// states of the back-trace (bin-major) -> the caller's table-major layout
__global__ void __launch_bounds__(1024)
viterbi_state_out_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const uint8_t *__restrict__ stateT,
                         uint8_t *__restrict__ state) {
    __shared__ uint8_t st[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int t_in = blockIdx.x * 32 + tx;
    const int64_t i_in = (int64_t)blockIdx.y * 32 + ty;
    if (t_in < n_tables && i_in < len[t_in]) st[ty][tx] = stateT[(size_t)i_in * n_tables + t_in];
    __syncthreads();
    const int t_out = blockIdx.x * 32 + ty;
    const int64_t i_out = (int64_t)blockIdx.y * 32 + tx;
    if (t_out < n_tables && i_out < len[t_out]) state[start[t_out] + i_out] = st[tx][ty];
}

}  // namespace ibdgem

using namespace ibdgem;

// ---------------------------------------------------------------------------------------------
// host side
namespace {

// The reference's own recurrence for one table, in x87 long double (src/hiddengem.c:74-76, 108-147, 246-257): the
// arbiter for tables the device flagged (near-tie at an arg-max, or scores outside the normal long double range).
// is_log = 1 (the engine's natural-log window scores) runs the same recurrence on long double logarithms.
void viterbi_long_double(const double *lik, int64_t n, int is_log, double p01, double p02, double p12, uint8_t *state,
                         double *score_log, int64_t counts[3]) {
    counts[0] = counts[1] = counts[2] = 0;
    if (n <= 0) return;
    std::vector<uint8_t> from((size_t)n);
    long double s[3] = {0, 0, 0};
    const long double pen[3][3] = {{1.0L, (long double)p01, (long double)p02},
                                   {(long double)p01, 1.0L, (long double)p12},
                                   {(long double)p02, (long double)p12, 1.0L}};
    long double lpen[3][3];
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) lpen[a][b] = a == b ? 0.0L : logl(pen[a][b]);
    for (int64_t i = 0; i < n; i++) {
        const double *L = lik + i * 3;
        long double nrm[3];
        if (is_log) {
            const long double m = fmaxl(L[0], fmaxl(L[1], L[2]));
            if (m == -INFINITY) {
                nrm[0] = nrm[1] = nrm[2] = NAN;
            } else {
                const long double z = m + logl(expl(L[0] - m) + expl(L[1] - m) + expl(L[2] - m));
                for (int k = 0; k < 3; k++) nrm[k] = (long double)L[k] - z;
            }
        } else {
            volatile double tot = L[0] + L[1];
            tot = tot + L[2];
            for (int k = 0; k < 3; k++) {
                volatile double q = L[k] / tot;  // fp64 quotient, as the reference stores it
                nrm[k] = q;
            }
        }
        if (i == 0) {
            for (int k = 0; k < 3; k++) s[k] = nrm[k];
            from[0] = (uint8_t)(0 | (1 << 2) | (2 << 4));
        } else {
            long double ns[3];
            uint8_t f = 0;
            for (int j = 0; j < 3; j++) {
                long double c[3];
                for (int k = 0; k < 3; k++) {
                    if (is_log)
                        c[k] = k == j ? s[k] + nrm[j] : (s[k] + nrm[j]) + lpen[k][j];
                    else
                        c[k] = k == j ? s[k] * nrm[j] : s[k] * nrm[j] * pen[k][j];
                }
                int best = 0;
                for (int k = 0; k < 3; k++)
                    if (c[k] > c[best]) best = k;  // find_max_idx: strict >, lowest index wins, NaN never wins
                ns[j] = c[best];
                f |= (uint8_t)(best << (2 * j));
            }
            for (int k = 0; k < 3; k++) s[k] = ns[k];
            from[(size_t)i] = f;
        }
        for (int k = 0; k < 3; k++) score_log[i * 3 + k] = is_log ? (double)s[k] : (double)logl(s[k]);
    }
    int cur = 0;
    for (int k = 0; k < 3; k++)
        if (s[k] > s[cur]) cur = k;
    for (int64_t i = n - 1; i >= 0; i--) {
        state[i] = (uint8_t)cur;
        counts[cur]++;
        cur = (from[(size_t)i] >> (2 * cur)) & 3;
    }
}

}  // namespace

// One batch of tables, everything in device memory.  start / len describe where each table's bins sit in lik /
// state / score; counts and flag are per table.  Kernels only (no host synchronisation).
int ibdgem::viterbi_on_device(ibdgem_engine *e, int n_tables, int64_t maxbins, int64_t total_bins, const int64_t *d_start, const int64_t *d_len,
                      const double *d_lik, int is_log, double p01, double p02, double p12, uint8_t *d_state, double *d_score,
                      long long *d_counts, uint8_t *d_flag) {
    const bool batched = n_tables >= 64 && (double)maxbins * n_tables <= 2.0 * (double)total_bins;
    if (batched) {
        double *d_last;
        uint8_t *d_fromT;
        if (scratch(e, SC_HG_FROMT, (size_t)maxbins * n_tables, (void **)&d_fromT) || scratch(e, SC_HG_LAST, (size_t)n_tables * 24, (void **)&d_last))
            return 1;
        {
            LaunchScope ls(e, K_VITERBI);
            IBD_CUDA(cudaFuncSetAttribute(viterbi_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, VF_SMEM));
            viterbi_fused_kernel<<<(n_tables + HG_TABLES - 1) / HG_TABLES, HG_THREADS, VF_SMEM, e->stream>>>(
                n_tables, d_start, d_len, d_lik, is_log, log(p01), log(p02), log(p12), d_score, d_fromT, d_last, d_flag);
        }
        {
            LaunchScope ls(e, K_VITERBI_BACK);
            viterbi_back_kernel<<<(n_tables + 63) / 64, 64, 0, e->stream>>>(n_tables, d_len, d_fromT, d_last, d_counts);
        }
        {
            LaunchScope ls(e, K_VITERBI_OUT);
            const dim3 tiles((unsigned)((n_tables + 31) / 32), (unsigned)((maxbins + 31) / 32));
            viterbi_state_out_kernel<<<tiles, 1024, 0, e->stream>>>(n_tables, d_start, d_len, d_fromT, d_state);
        }
    } else {
        LaunchScope ls(e, K_VITERBI);
        viterbi_kernel<<<(n_tables + 127) / 128, 128, 0, e->stream>>>(n_tables, d_start, d_len, d_lik, is_log, log(p01), log(p02), log(p12),
                                                                     d_state, d_score, d_counts, d_flag);
    }
    IBD_CUDA(cudaGetLastError());
    return 0;
}

// Flagged tables: the reference's long double recurrence decides (tables are independent: a few host threads).
void ibdgem::viterbi_redo_flagged(const std::vector<int> &flagged, const int64_t *bin_offsets, const double *lik, int is_log, double p01,
                                  double p02, double p12,
                                  const std::function<void(size_t, int, const uint8_t *, const double *, const int64_t *)> &sink) {
    auto redo = [&](size_t k0, size_t step) {
        std::vector<uint8_t> st_tmp;
        std::vector<double> sc_tmp;
        for (size_t k = k0; k < flagged.size(); k += step) {
            const int t = flagged[k];
            const int64_t b0 = bin_offsets[t], n = bin_offsets[t + 1] - b0;
            int64_t c[3];
            st_tmp.resize((size_t)n);
            sc_tmp.resize((size_t)n * 3);
            viterbi_long_double(lik + b0 * 3, n, is_log, p01, p02, p12, st_tmp.data(), sc_tmp.data(), c);
            sink(k, t, st_tmp.data(), sc_tmp.data(), c);
        }
    };
    const size_t nthr = std::max<size_t>(1, std::min<size_t>({flagged.size(), (size_t)16, (size_t)std::thread::hardware_concurrency()}));
    if (nthr <= 1) {
        redo(0, 1);
    } else {
        std::vector<std::thread> pool;
        for (size_t k = 0; k < nthr; k++) pool.emplace_back(redo, k, nthr);
        for (auto &th : pool) th.join();
    }
}

// Host start / length of every table (stride > 0: table t starts at bin t * table_stride); 1 (error set) on a negative
// length or one past the stride.
int ibdgem::table_layout(const char *fn, int n_tables, const int64_t *bin_offsets, int64_t table_stride, std::vector<int64_t> *sl,
                         int64_t *maxbins, int64_t *total) {
    sl->assign((size_t)n_tables * 2, 0);
    *maxbins = *total = 0;
    for (int t = 0; t < n_tables; t++) {
        const int64_t n = bin_offsets[t + 1] - bin_offsets[t];
        if (n < 0 || (table_stride > 0 && n > table_stride)) {
            set_error("[::] ERROR in %s(): table %d has %lld bins (stride %lld).", fn, t, (long long)n, (long long)table_stride);
            return 1;
        }
        (*sl)[(size_t)t] = table_stride > 0 ? (int64_t)t * table_stride : bin_offsets[t];
        (*sl)[(size_t)n_tables + t] = n;
        *maxbins = std::max(*maxbins, n);
        *total += n;
    }
    return 0;
}

// Host buffers in, host buffers out.  The tables go through in batches: while batch b is scored, batch b + 1 is on its
// way up and the results of batch b - 1 on their way down (three streams; page-locked buffers make the copies
// asynchronous, pageable ones are simply staged by the driver).
extern "C" int hiddengem_viterbi_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets,
                                       const double *lik, int32_t is_log, double p01, double p02,
                                       double p12, uint8_t *state, double *score_log,
                                       int64_t *state_counts) {
    if (!e || n_tables <= 0 || !bin_offsets || !lik) {
        set_error("[::] ERROR in hiddengem_viterbi_batch(): bad arguments.");
        return 1;
    }
    std::vector<int64_t> h_sl;
    int64_t maxbins_all, total;
    if (table_layout("hiddengem_viterbi_batch", n_tables, bin_offsets, 0, &h_sl, &maxbins_all, &total)) return 1;
    IBD_CUDA(cudaSetDevice(e->device));
    const int64_t nb = bin_offsets[n_tables];
    if (nb <= 0) {
        set_error("[::] ERROR parsing likelihood data; make sure input is valid.");
        return 1;
    }
    double *d_lik, *d_score;
    int64_t *d_start;
    uint8_t *d_state, *d_flag;
    long long *d_counts;
    if (scratch(e, SC_HG_LIK, (size_t)nb * 24, (void **)&d_lik) || scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start) ||
        scratch(e, SC_HG_STATE, (size_t)nb + (size_t)n_tables, (void **)&d_state) || scratch(e, SC_HG_SCORE, (size_t)nb * 24, (void **)&d_score) ||
        scratch(e, SC_HG_COUNTS, (size_t)n_tables * 24, (void **)&d_counts))
        return 1;
    d_flag = d_state + nb;
    int64_t *d_len = d_start + n_tables;
    if (!e->copy_stream) {
        IBD_CUDA(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        IBD_CUDA(cudaEventCreateWithFlags(&e->ev_order, cudaEventDisableTiming));
    }
    if (!e->d2h_stream) IBD_CUDA(cudaStreamCreateWithFlags(&e->d2h_stream, cudaStreamNonBlocking));
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    // earlier work on the engine stream may still use the scratch buffers: the side streams start after it
    IBD_CUDA(cudaEventRecord(e->ev_order, e->stream));
    IBD_CUDA(cudaStreamWaitEvent(e->copy_stream, e->ev_order, 0));
    IBD_CUDA(cudaStreamWaitEvent(e->d2h_stream, e->ev_order, 0));
    // Batches of whole tables, at least 64 so the batched kernels apply.  A batch's kernels take the time of one block
    // (the recursion is sequential in bins) however few tables it holds, so batches are few: about six per call —
    // copy-bound with ~1/6 of the upload exposed at the front and ~1/6 of the download at the back — and never below
    // ~192 MB of likelihoods.
    const int64_t target_bins = std::max<int64_t>((int64_t)8 << 20, nb / 6);
    std::vector<int> cuts{0};
    for (int t = 0; t < n_tables;) {
        int t1 = t;
        while (t1 < n_tables && (t1 - t < 64 || bin_offsets[t1] - bin_offsets[t] < target_bins)) t1++;
        if (n_tables - t1 < 64) t1 = n_tables;  // no runt batch at the end
        cuts.push_back(t1);
        t = t1;
    }
    const size_t nbatch = cuts.size() - 1;
    std::vector<cudaEvent_t> ev_up(nbatch), ev_done(nbatch);
    for (size_t b = 0; b < nbatch; b++) {
        IBD_CUDA(cudaEventCreateWithFlags(&ev_up[b], cudaEventDisableTiming));
        IBD_CUDA(cudaEventCreateWithFlags(&ev_done[b], cudaEventDisableTiming));
    }
    int rc = 0;
    for (size_t b = 0; b < nbatch && !rc; b++) {
        const int t0 = cuts[b], t1 = cuts[b + 1];
        const int64_t b0 = bin_offsets[t0], b1 = bin_offsets[t1];
        IBD_CUDA(cudaMemcpyAsync(d_lik + b0 * 3, lik + b0 * 3, (size_t)(b1 - b0) * 24, cudaMemcpyHostToDevice, e->copy_stream));
        IBD_CUDA(cudaEventRecord(ev_up[b], e->copy_stream));
    }
    for (size_t b = 0; b < nbatch && !rc; b++) {
        const int t0 = cuts[b], t1 = cuts[b + 1];
        const int64_t b0 = bin_offsets[t0], b1 = bin_offsets[t1];
        int64_t maxbins = 0;
        for (int t = t0; t < t1; t++) maxbins = std::max<int64_t>(maxbins, bin_offsets[t + 1] - bin_offsets[t]);
        IBD_CUDA(cudaStreamWaitEvent(e->stream, ev_up[b], 0));
        rc = viterbi_on_device(e, t1 - t0, maxbins, b1 - b0, d_start + t0, d_len + t0, d_lik, is_log, p01, p02, p12, d_state, d_score,
                               d_counts + (size_t)t0 * 3, d_flag + t0);
        if (rc) break;
        IBD_CUDA(cudaEventRecord(ev_done[b], e->stream));
        IBD_CUDA(cudaStreamWaitEvent(e->d2h_stream, ev_done[b], 0));
        if (state) IBD_CUDA(cudaMemcpyAsync(state + b0, d_state + b0, (size_t)(b1 - b0), cudaMemcpyDeviceToHost, e->d2h_stream));
        if (score_log) IBD_CUDA(cudaMemcpyAsync(score_log + b0 * 3, d_score + b0 * 3, (size_t)(b1 - b0) * 24, cudaMemcpyDeviceToHost, e->d2h_stream));
    }
    std::vector<uint8_t> h_flag((size_t)n_tables, 0);
    std::vector<long long> h_counts((size_t)n_tables * 3);
    if (!rc) {
        IBD_CUDA(cudaMemcpyAsync(h_counts.data(), d_counts, (size_t)n_tables * 24, cudaMemcpyDeviceToHost, e->stream));
        IBD_CUDA(cudaMemcpyAsync(h_flag.data(), d_flag, (size_t)n_tables, cudaMemcpyDeviceToHost, e->stream));
    }
    cudaStreamSynchronize(e->copy_stream);
    cudaStreamSynchronize(e->stream);
    cudaStreamSynchronize(e->d2h_stream);
    for (size_t b = 0; b < nbatch; b++) {
        cudaEventDestroy(ev_up[b]);
        cudaEventDestroy(ev_done[b]);
    }
    if (rc) return 1;
    IBD_CUDA(cudaGetLastError());
    settle_timers(e);
    std::vector<int> flagged;
    for (int t = 0; t < n_tables; t++) {
        if (state_counts) {
            state_counts[(size_t)t * 3] = h_counts[(size_t)t * 3];
            state_counts[(size_t)t * 3 + 1] = h_counts[(size_t)t * 3 + 1];
            state_counts[(size_t)t * 3 + 2] = h_counts[(size_t)t * 3 + 2];
        }
        if (h_flag[(size_t)t]) flagged.push_back(t);
    }
    e->hg_flagged = (int64_t)flagged.size();
    viterbi_redo_flagged(flagged, bin_offsets, lik, is_log, p01, p02, p12,
                         [&](size_t, int t, const uint8_t *st, const double *sc, const int64_t *c) {
                             const int64_t b0 = bin_offsets[t], n = bin_offsets[t + 1] - b0;
                             if (state) memcpy(state + b0, st, (size_t)n);
                             if (score_log) memcpy(score_log + b0 * 3, sc, (size_t)n * 24);
                             if (state_counts) {
                                 state_counts[(size_t)t * 3] = c[0];
                                 state_counts[(size_t)t * 3 + 1] = c[1];
                                 state_counts[(size_t)t * 3 + 2] = c[2];
                             }
                         });
    return 0;
}

// Device buffers in, device buffers out: the hiddengem front-end for scores that never left the GPU (SURVEY.md 8f-3).
//   table_stride = 0: tables are packed, table t holds bins [bin_offsets[t], bin_offsets[t+1]) of d_lik / d_state / d_score;
//   table_stride > 0: table t starts at bin t * table_stride (the layout of ibdgem_scores.w_loglik_device with
//                     table_stride = max_windows) and has bin_offsets[t+1] - bin_offsets[t] bins.
// bin_offsets is a HOST array.  Flagged tables (near-ties) are re-evaluated on the host in long double and patched
// back into the device buffers.
extern "C" int hiddengem_viterbi_batch_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                              const double *d_lik, int32_t is_log, double p01, double p02, double p12,
                                              uint8_t *d_state, double *d_score_log, int64_t *d_state_counts) {
    if (!e || n_tables <= 0 || !bin_offsets || !d_lik || !d_state || !d_score_log || !d_state_counts || table_stride < 0) {
        set_error("[::] ERROR in hiddengem_viterbi_batch_device(): bad arguments.");
        return 1;
    }
    IBD_CUDA(cudaSetDevice(e->device));
    std::vector<int64_t> h_sl;
    int64_t maxbins, total;
    if (table_layout("hiddengem_viterbi_batch_device", n_tables, bin_offsets, table_stride, &h_sl, &maxbins, &total)) return 1;
    if (total <= 0) {
        set_error("[::] ERROR parsing likelihood data; make sure input is valid.");
        return 1;
    }
    int64_t *d_start;
    uint8_t *d_flag;
    if (scratch(e, SC_HG_OFF, (size_t)n_tables * 16, (void **)&d_start) || scratch(e, SC_HG_STATE, (size_t)n_tables, (void **)&d_flag)) return 1;
    IBD_CUDA(cudaMemcpyAsync(d_start, h_sl.data(), h_sl.size() * 8, cudaMemcpyHostToDevice, e->stream));
    static_assert(sizeof(long long) == sizeof(int64_t), "state counts are 64-bit");
    if (viterbi_on_device(e, n_tables, maxbins, total, d_start, d_start + n_tables, d_lik, is_log, p01, p02, p12, d_state, d_score_log,
                          reinterpret_cast<long long *>(d_state_counts), d_flag))
        return 1;
    std::vector<uint8_t> h_flag((size_t)n_tables);
    IBD_CUDA(cudaMemcpyAsync(h_flag.data(), d_flag, (size_t)n_tables, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    settle_timers(e);
    e->hg_flagged = 0;
    for (int t = 0; t < n_tables; t++) {
        if (!h_flag[(size_t)t]) continue;
        const int64_t b0 = h_sl[(size_t)t], n = h_sl[(size_t)n_tables + t];
        std::vector<double> l((size_t)n * 3), sc((size_t)n * 3);
        std::vector<uint8_t> st((size_t)n);
        int64_t c[3];
        IBD_CUDA(cudaMemcpy(l.data(), d_lik + b0 * 3, (size_t)n * 24, cudaMemcpyDeviceToHost));
        viterbi_long_double(l.data(), n, is_log, p01, p02, p12, st.data(), sc.data(), c);
        IBD_CUDA(cudaMemcpy(d_state + b0, st.data(), (size_t)n, cudaMemcpyHostToDevice));
        IBD_CUDA(cudaMemcpy(d_score_log + b0 * 3, sc.data(), (size_t)n * 24, cudaMemcpyHostToDevice));
        IBD_CUDA(cudaMemcpy(d_state_counts + (size_t)t * 3, c, 24, cudaMemcpyHostToDevice));
        e->hg_flagged++;
    }
    return 0;
}

// Tables of the last hiddengem call that were re-evaluated on the host in long double (near-tie guard).
extern "C" int64_t hiddengem_last_flagged(ibdgem_engine *e) { return e ? e->hg_flagged : -1; }
