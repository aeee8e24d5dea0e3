// tract_lengths.cu — hiddengem posterior tract-length spectrum: for each table, state s and threshold X, the posterior
// expected number of maximal runs of s whose length reaches X,
//     E[R_s(X)] = sum_i d_i(s) * prod_{m=i+1}^{J} c_m(s) * gamma_J(s),      J = J(i, X), the first bin J >= i whose run
// [i, J] is X long (end[J] - start[i] + 1 with coordinates, J - i + 1 in bins); a start bin without such a J adds 0.
// Conditioned on x_J = s the past is a backward Markov chain with kernel alpha * pen normalised, so the term is
// P(x_{i-1} != s, x_i = ... = x_J = s | data): each run of length >= X is counted once, at its first bin.
//
// The backward pass of posterior.cu in mode BWD_RUNS writes gamma, d and ln c of every bin (runs[bin][9]); then
// tract_lengths_kernel, one warp per table:
//   phase A  strides of 32 bins (lane = bin): the in-stride inclusive prefix of ln c per bin (pf), and per stride its
//            total (st) and, within its 1,024-bin block, the inclusive prefix (sp) and suffix (ss) of stride totals,
//            and per block its total (bt).  The coordinates are checked here (start <= end, both non-decreasing).
//   phase B  strides of 32 start bins (lane = i): per threshold, J (bins: i + X - 1; coordinates: binary search over
//            END from the previous threshold's J), then the window sum of ln c over (i, J] from pieces that lie
//            inside the window only: the rest of i's stride (a warp suffix scan), whole strides or the block-suffix,
//            whole blocks and block-prefix of stride totals, and pf of J's stride; within one stride, the terms
//            themselves.  Every ln c <= 0, so no piece cancels: the sum is exact to a few ulps of its own size,
//            where prefix sums over the whole table would subtract numbers of 1e6-1e7 nats.
// Each lane adds its terms in stride order, the lanes' sums meet in a fixed tree: the same table gives the same bits
// in any batch or layout.
#include <math.h>

#include <algorithm>
#include <vector>

#include "engine.h"

namespace ibdgem {

constexpr int TL_WARPS = 4;  // tables (warps) per block
constexpr int TL_MAXK = 16;  // thresholds per call
constexpr unsigned TL_FULL = 0xffffffffu;

struct TlThresholds {
    unsigned long long x[TL_MAXK];
    int k;
};

// Hierarchy of one call: pf [bins][3] in the layout of the likelihoods; st / sp / ss [stride slots][3] and bt
// [block slots][3], table t's stride (block) q at slot (start_t >> 5) + t + q ((start_t >> 10) + t + q): no two
// tables share a slot in a packed or strided layout.
struct TlSums {
    double *pf, *st, *sp, *ss, *bt;
};

__device__ __forceinline__ double tl_scan_up(double v, int lane) {  // inclusive prefix over the lanes
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double u = __shfl_up_sync(TL_FULL, v, d);
        if (lane >= d) v = u + v;
    }
    return v;
}

__device__ __forceinline__ double tl_scan_down(double v, int lane) {  // inclusive suffix over the lanes
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double u = __shfl_down_sync(TL_FULL, v, d);
        if (lane + d < 32) v = v + u;
    }
    return v;
}

// spectrum[t][k][s]; expected[t][0] NaN marks a table of total weight 0 (the backward pass writes it so).  bstart /
// bend null: lengths in bins.  *bad = 1 when a table's coordinates are not monotone.
__global__ void __launch_bounds__(TL_WARPS * 32)
tract_lengths_kernel(int n_tables, const int64_t *__restrict__ start, const int64_t *__restrict__ len, const double *__restrict__ runs,
                     const double *__restrict__ expected, const uint64_t *__restrict__ bstart, const uint64_t *__restrict__ bend,
                     TlThresholds th, TlSums h, double *__restrict__ spectrum, int *__restrict__ bad) {
    __shared__ double acc[TL_WARPS][TL_MAXK * 3][32];  // each lane's running sums, [k * 3 + s]
    const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int t = blockIdx.x * TL_WARPS + wp;
    if (t >= n_tables) return;  // whole warps
    const int64_t b0 = start[t], n = len[t];
    const double *R = runs + b0 * 9;
    const uint64_t *BS = bstart ? bstart + b0 : nullptr, *BE = bend ? bend + b0 : nullptr;
    double *PF = h.pf + b0 * 3, *ST = h.st + ((b0 >> 5) + t) * 3, *SP = h.sp + ((b0 >> 5) + t) * 3, *SS = h.ss + ((b0 >> 5) + t) * 3,
           *BT = h.bt + ((b0 >> 10) + t) * 3;
    // phase A
    bool wrong = false;
    double blk[3] = {0, 0, 0};  // lane q: the total of stride q of the current block
    for (int64_t i0 = 0; i0 < n; i0 += 32) {
        const int64_t i = i0 + lane;
        const bool live = i < n;
        const int q = (int)((i0 >> 5) & 31);
        if (BS && live) wrong |= BS[i] > BE[i] || (i > 0 && (BS[i - 1] > BS[i] || BE[i - 1] > BE[i]));
#pragma unroll
        for (int s = 0; s < 3; s++) {
            const double p = tl_scan_up(live ? R[i * 9 + 6 + s] : 0.0, lane);
            if (live) PF[i * 3 + s] = p;
            const double tot = __shfl_sync(TL_FULL, p, 31);
            if (lane == q) blk[s] = tot;
        }
        if (q == 31 || i0 + 32 >= n) {  // the block is complete: lanes 0..q hold its strides
            const int64_t sq = (i0 >> 5) - q + lane;
#pragma unroll
            for (int s = 0; s < 3; s++) {
                const double p = tl_scan_up(blk[s], lane), u = tl_scan_down(blk[s], lane);
                if (lane <= q) {
                    ST[sq * 3 + s] = blk[s];
                    SP[sq * 3 + s] = p;
                    SS[sq * 3 + s] = u;
                }
                const double tot = __shfl_sync(TL_FULL, p, 31);
                if (lane == 0) BT[(i0 >> 10) * 3 + s] = tot;
                blk[s] = 0.0;
            }
        }
    }
    if (__any_sync(TL_FULL, wrong) && lane == 0) *bad = 1;
    __syncwarp();  // phase A's stores are visible to the whole warp
    double *out = spectrum + (size_t)t * th.k * 3;
    if (n > 0 && isnan(expected[(size_t)t * 3])) {  // total weight 0
        for (int j = lane; j < th.k * 3; j += 32) out[j] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    double *a = &acc[wp][0][lane];
    for (int j = 0; j < th.k * 3; j++) a[j * 32] = 0.0;
    // phase B
    for (int64_t i0 = 0; i0 < n; i0 += 32) {
        const int64_t i = i0 + lane;
        const bool live = i < n;
        const int64_t si = i0 >> 5;
        double d[3], sx[3];  // d_i, and the sum of ln c over the rest of i's stride (i + 1 .. the stride's end)
#pragma unroll
        for (int s = 0; s < 3; s++) {
            d[s] = live ? R[i * 9 + 3 + s] : 0.0;
            const double u = __shfl_down_sync(TL_FULL, tl_scan_down(live ? R[i * 9 + 6 + s] : 0.0, lane), 1);
            sx[s] = lane < 31 ? u : 0.0;
        }
        if (!live) continue;  // only the last stride; no shuffles below
        const uint64_t si0 = BS ? BS[i] : 0;
        int64_t lo = i;  // J of the previous threshold: J is non-decreasing in X
        for (int k = 0; k < th.k; k++) {
            const unsigned long long X = th.x[k];
            int64_t J;
            if (!BS) {
                J = X - 1 < (unsigned long long)(n - i) ? i + (int64_t)(X - 1) : n;
            } else {  // first J in [lo, n) with end[J] - start[i] + 1 >= X (end[J] >= end[i] >= start[i]): a galloping
                      // bracket from lo, as J is mostly near, then bisection
                int64_t hi = lo;
                for (int64_t step = 1; hi < n && BE[hi] - si0 < X - 1; step <<= 1) {
                    lo = hi + 1;
                    hi = min(n, hi + step);
                }
                while (lo < hi) {
                    const int64_t mid = lo + (hi - lo) / 2;
                    if (BE[mid] - si0 >= X - 1) hi = mid;
                    else lo = mid + 1;
                }
                J = lo;
            }
            if (J >= n) break;  // no longer threshold is reached either
            lo = J;
            const int64_t sj = J >> 5;
            double w[3];
            if (sj == si) {
#pragma unroll
                for (int s = 0; s < 3; s++) w[s] = 0.0;
                for (int64_t m = i + 1; m <= J; m++) {
#pragma unroll
                    for (int s = 0; s < 3; s++) w[s] += R[m * 9 + 6 + s];
                }
            } else {
                double mid[3] = {0, 0, 0};  // strides si + 1 .. sj - 1
                const int64_t qa = si + 1, qb = sj - 1;
                if (qa <= qb && (qa >> 5) == (qb >> 5)) {
                    for (int64_t q = qa; q <= qb; q++) {
#pragma unroll
                        for (int s = 0; s < 3; s++) mid[s] += ST[q * 3 + s];
                    }
                } else if (qa <= qb) {
#pragma unroll
                    for (int s = 0; s < 3; s++) mid[s] = SS[qa * 3 + s];
                    for (int64_t bq = (qa >> 5) + 1; bq < (qb >> 5); bq++) {
#pragma unroll
                        for (int s = 0; s < 3; s++) mid[s] += BT[bq * 3 + s];
                    }
#pragma unroll
                    for (int s = 0; s < 3; s++) mid[s] += SP[qb * 3 + s];
                }
#pragma unroll
                for (int s = 0; s < 3; s++) w[s] = (sx[s] + mid[s]) + PF[J * 3 + s];
            }
#pragma unroll
            for (int s = 0; s < 3; s++) a[(k * 3 + s) * 32] += R[J * 9 + s] * d[s] * exp(w[s]);
        }
    }
    __syncwarp();
    for (int j = 0; j < th.k * 3; j++) {  // the lanes' sums in a fixed tree
        double v = a[j * 32];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(TL_FULL, v, o);
        if (lane == 0) out[j] = v;
    }
}

}  // namespace ibdgem

using namespace ibdgem;

namespace {

// The body of both entries.  lik, bstart / bend and spectrum are host buffers (packed) or, with on_device, device
// buffers in the layout of table_stride; thresholds is a host array.
int tract_lengths_call(ibdgem_engine *e, const char *fn, int n_tables, const int64_t *bin_offsets, int64_t table_stride, const double *lik,
                       bool on_device, int is_log, double p01, double p02, double p12, const uint64_t *bstart, const uint64_t *bend,
                       int n_thresholds, const uint64_t *thresholds, double *spectrum) {
    if (bad_penalties(fn, p01, p02, p12)) return 1;
    if (!bstart != !bend) {
        set_error("[::] ERROR in %s(): give both bin_start and bin_end, or neither (lengths in bins).", fn);
        return 1;
    }
    bool ok = thresholds && n_thresholds >= 1 && n_thresholds <= TL_MAXK;
    for (int k = 0; ok && k < n_thresholds; k++) ok = thresholds[k] >= 1 && (k == 0 || thresholds[k] > thresholds[k - 1]);
    if (!ok) {
        set_error("[::] ERROR in %s(): thresholds must be 1 to %d values >= 1, strictly increasing.", fn, TL_MAXK);
        return 1;
    }
    HgCall c;
    if (hg_begin(e, fn, n_tables, bin_offsets, table_stride, false, &c)) return 1;
    if (c.total > 0 && !lik) {
        set_error("[::] ERROR in %s(): bad arguments.", fn);
        return 1;
    }
    int64_t extent = 0;  // bins of the layout
    for (int t = 0; t < n_tables; t++) extent = std::max(extent, c.start(t) + c.len(t));
    const size_t nsp = (size_t)n_tables * n_thresholds * 3;
    // SC_HG_COUNTS: expected [n_tables][3], the flag, and the host entry's spectrum
    double *d_expected, *d_spec = spectrum;
    if (scratch(e, SC_HG_COUNTS, (size_t)n_tables * 24 + 8 + (on_device ? 0 : nsp * 8), (void **)&d_expected)) return 1;
    int *d_bad = reinterpret_cast<int *>(d_expected + (size_t)n_tables * 3);
    if (!on_device) d_spec = d_expected + (size_t)n_tables * 3 + 1;
    IBD_CUDA(cudaMemsetAsync(d_bad, 0, 8, e->stream));
    if (c.maxbins == 0) {  // only empty tables
        IBD_CUDA(cudaMemsetAsync(d_spec, 0, nsp * 8, e->stream));
    } else {
        const double *d_lik = lik;
        const uint64_t *d_bs = bstart, *d_be = bend;
        if (!on_device) {  // packed: extent = the call's bins
            double *d_up;
            if (scratch(e, SC_HG_LIK, (size_t)extent * 24, (void **)&d_up)) return 1;
            IBD_CUDA(cudaMemcpyAsync(d_up, lik, (size_t)extent * 24, cudaMemcpyHostToDevice, e->stream));
            d_lik = d_up;
            if (bstart) {
                uint64_t *d_co;
                if (scratch(e, SC_HG_COORD, (size_t)extent * 16, (void **)&d_co)) return 1;
                IBD_CUDA(cudaMemcpyAsync(d_co, bstart, (size_t)extent * 8, cudaMemcpyHostToDevice, e->stream));
                IBD_CUDA(cudaMemcpyAsync(d_co + extent, bend, (size_t)extent * 8, cudaMemcpyHostToDevice, e->stream));
                d_bs = d_co;
                d_be = d_co + extent;
            }
        }
        const size_t nst = (size_t)(extent >> 5) + n_tables + 1, nbk = (size_t)(extent >> 10) + n_tables + 1;
        double *d_runs, *d_sums;
        if (scratch(e, SC_HG_RUNS, (size_t)extent * 72, (void **)&d_runs) ||
            scratch(e, SC_HG_RUNSUM, ((size_t)extent + 3 * nst + nbk) * 24, (void **)&d_sums))
            return 1;
        const TlSums hs{d_sums, d_sums + (size_t)extent * 3, d_sums + ((size_t)extent + nst) * 3, d_sums + ((size_t)extent + 2 * nst) * 3,
                        d_sums + ((size_t)extent + 3 * nst) * 3};
        if (posterior_on_device(e, n_tables, c.maxbins, c.d_start, c.d_len, d_lik, is_log, p01, p02, p12, nullptr, d_expected, nullptr,
                                nullptr, nullptr, d_runs))
            return 1;
        TlThresholds th{};
        th.k = n_thresholds;
        for (int k = 0; k < n_thresholds; k++) th.x[k] = thresholds[k];
        {
            LaunchScope ls(e, K_TRACT_LENGTHS);
            tract_lengths_kernel<<<(unsigned)((n_tables + TL_WARPS - 1) / TL_WARPS), TL_WARPS * 32, 0, e->stream>>>(
                n_tables, c.d_start, c.d_len, d_runs, d_expected, d_bs, d_be, th, hs, d_spec, d_bad);
        }
        IBD_CUDA(cudaGetLastError());
    }
    int h_bad = 0;
    IBD_CUDA(cudaMemcpyAsync(&h_bad, d_bad, 4, cudaMemcpyDeviceToHost, e->stream));
    if (!on_device) IBD_CUDA(cudaMemcpyAsync(spectrum, d_spec, nsp * 8, cudaMemcpyDeviceToHost, e->stream));
    IBD_CUDA(cudaStreamSynchronize(e->stream));
    settle_timers(e);
    if (h_bad) {
        set_error("[::] ERROR in %s(): bin coordinates are not sorted within a table (need start <= end, both non-decreasing).", fn);
        return 1;
    }
    return 0;
}

}  // namespace

// Host buffers in, host buffers out: the likelihoods (and coordinates) go up once, only the spectrum comes back.
extern "C" int hiddengem_tract_lengths_batch(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, const double *lik,
                                             int32_t is_log, double p01, double p02, double p12, const uint64_t *bin_start,
                                             const uint64_t *bin_end, int32_t n_thresholds, const uint64_t *thresholds, double *spectrum) {
    if (!e || n_tables <= 0 || !bin_offsets || !spectrum) {
        set_error("[::] ERROR in hiddengem_tract_lengths_batch(): bad arguments.");
        return 1;
    }
    return tract_lengths_call(e, "hiddengem_tract_lengths_batch", n_tables, bin_offsets, 0, lik, false, is_log, p01, p02, p12, bin_start,
                              bin_end, n_thresholds, thresholds, spectrum);
}

// Device buffers in, device buffers out; bin_offsets and thresholds are HOST arrays, table_stride as for
// hiddengem_posterior_batch_device (the coordinates in the same layout).
extern "C" int hiddengem_tract_lengths_device(ibdgem_engine *e, int32_t n_tables, const int64_t *bin_offsets, int64_t table_stride,
                                              const double *d_lik, int32_t is_log, double p01, double p02, double p12,
                                              const uint64_t *d_bin_start, const uint64_t *d_bin_end, int32_t n_thresholds,
                                              const uint64_t *thresholds, double *d_spectrum) {
    if (!e || n_tables <= 0 || !bin_offsets || !d_lik || !d_spectrum || table_stride < 0) {
        set_error("[::] ERROR in hiddengem_tract_lengths_device(): bad arguments.");
        return 1;
    }
    return tract_lengths_call(e, "hiddengem_tract_lengths_device", n_tables, bin_offsets, table_stride, d_lik, true, is_log, p01, p02, p12,
                              d_bin_start, d_bin_end, n_thresholds, thresholds, d_spectrum);
}
