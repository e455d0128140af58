// Batch statistics of a solved batch (hpf_batch_stats): per row r of the R = nH + 2n rows
// (V_m of order harmonics[h] at bus i = row h*n + i, THD_F of bus i = row nH + i, THD_R = row nH + n + i)
// the mean, population std, min, max, number above a limit and K exact nearest-rank quantiles over the
// included scenarios (status == HPF_ST_CONVERGED, or all of them without a status array).
//
// One thread-block CLUSTER per row (grid = CS x R CTAs, cluster = CS along x); its CS CTAs split the row into CS contiguous segments and combine
// their partial results through distributed shared memory, in rank order:
//   pass 1  count, sum, min / max (as order-preserving keys), exceed, status counts (row 0)
//   pass 2  sum of squared deviations from the combined mean (two-pass std)
//   pass 3+ MSD radix select of all K quantiles at once, 8 bits per pass: every pass builds one
//           256-bin histogram per distinct prefix of the active quantiles (shared memory, integer
//           atomics), the cluster adds them up and every quantile descends into the bin holding its
//           rank.  The select starts below the bits min and max share, and a quantile whose bin holds
//           ONE element takes that element's key (stored next to the bin count) without descending
//           further, so a row of distinct values needs about log256(B) passes.
// Determinism: every floating-point sum runs in a fixed order - each thread over its strided elements,
// a fixed shuffle tree per warp, warp 0 over the warps, then the cluster's CTAs in rank order - so the
// bits depend on (B, CS, block size) only.  Quantiles and counts are exact integers / order statistics.
#pragma once
#include <cooperative_groups.h>
#include <cstdint>

#define HPF_STATS_THREADS 256
#define HPF_STATS_WARPS (HPF_STATS_THREADS / 32)
#define HPF_STATS_BINS 256
#define HPF_STATS_UNROLL 8

struct StatsArgs {
    int B, R, nH, K;
    const double* V_m;      // [nH, B]: rows 0 .. nH-1
    const double* thd;      // [2n, B]: rows nH .. R-1
    const int* status;      // [B] or null (every scenario included)
    const double* limits;   // [R] or null
    int* counts;            // [4]
    double* stats;          // [5 + K, R]
    double q[HPF_STATS_MAX_Q];
};

// dynamic shared memory of stats_kernel: a double-buffered histogram and key slot per bin and quantile
static inline size_t stats_smem_bytes(int K) {
    return (size_t)2 * K * HPF_STATS_BINS * (sizeof(int) + sizeof(unsigned long long));
}

// Order-preserving 64-bit key of a double: the sign bit of a non-negative value is set, every bit of a
// negative one flipped (-0 sorts just below +0, NaNs by their sign bit beyond the infinities).
__device__ __forceinline__ unsigned long long stats_key(double x) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double stats_value(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

struct StatsPart {          // one CTA's share of a row
    double sum, ss;
    unsigned long long kmin, kmax;
    int n, exceed;
    int st[4];
};

// fixed-order block reductions (warp shuffle tree, then warp 0 over the warp results)
template <class T, class Op>
__device__ __forceinline__ T stats_block_reduce(T v, T* red, Op op) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_down_sync(0xffffffffu, v, o));
    __syncthreads();                           // red[] may still be read by the previous reduction
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        v = lane < HPF_STATS_WARPS ? red[lane] : red[0];
#pragma unroll
        for (int o = HPF_STATS_WARPS / 2; o > 0; o >>= 1) {
            const T w = __shfl_down_sync(0xffffffffu, v, o);
            if (lane + o < HPF_STATS_WARPS) v = op(v, w);
        }
    }
    return v;                                  // valid in thread 0
}

__global__ void __launch_bounds__(HPF_STATS_THREADS) stats_kernel(const StatsArgs a) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int cs = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int row = blockIdx.x / cs, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t B = (size_t)a.B;
    const double* x = row < a.nH ? a.V_m + (size_t)row * B : a.thd + (size_t)(row - a.nH) * B;
    const size_t lo = B * rank / cs, hi = B * (rank + 1) / cs;
    const int* status = a.status;
    const double lim = a.limits ? a.limits[row] : __longlong_as_double(0x7ff0000000000000ll);
    const int K = a.K;

    extern __shared__ __align__(16) unsigned char stats_smem[];
    int* hist = reinterpret_cast<int*>(stats_smem);                                  // [2][K][256]
    unsigned long long* hkey = reinterpret_cast<unsigned long long*>(hist + 2 * K * HPF_STATS_BINS);
    __shared__ StatsPart part;
    __shared__ double red_d[HPF_STATS_WARPS];
    __shared__ int red_i[HPF_STATS_WARPS];
    __shared__ unsigned long long red_k[HPF_STATS_WARPS];
    // row totals, identical in every CTA of the cluster
    __shared__ double t_mean;
    __shared__ int t_n;
    __shared__ unsigned long long t_kmin, t_kmax;
    // radix-select state per quantile: prefix above the current digit, rank inside it, done flag, key
    __shared__ unsigned long long q_pre[HPF_STATS_MAX_Q], q_key[HPF_STATS_MAX_Q], u_pre[HPF_STATS_MAX_Q];
    __shared__ long long q_rank[HPF_STATS_MAX_Q];
    __shared__ int q_act[HPF_STATS_MAX_Q], q_u[HPF_STATS_MAX_Q], n_u;

    const int rounds = (int)((hi - lo + HPF_STATS_THREADS * HPF_STATS_UNROLL - 1) / (HPF_STATS_THREADS * HPF_STATS_UNROLL));

    // ---- pass 1: count, sum, min / max keys, exceed, status counts ------------------------------
    double s = 0.0;
    int n = 0, ex = 0, sc[4] = {0, 0, 0, 0};
    unsigned long long kmin = ~0ull, kmax = 0ull;
    for (int it = 0; it < rounds; ++it) {
        double v[HPF_STATS_UNROLL];
        bool in[HPF_STATS_UNROLL];
#pragma unroll
        for (int j = 0; j < HPF_STATS_UNROLL; ++j) {
            const size_t b = lo + ((size_t)it * HPF_STATS_UNROLL + j) * HPF_STATS_THREADS + tid;
            in[j] = b < hi;
            v[j] = in[j] ? __ldg(x + b) : 0.0;
            if (in[j] && status) {
                const int st = __ldg(status + b);
#pragma unroll
                for (int i = 0; i < 4; ++i) sc[i] += st == i;
                in[j] = st == 0;
            }
        }
#pragma unroll
        for (int j = 0; j < HPF_STATS_UNROLL; ++j) {
            if (!in[j]) continue;
            const unsigned long long k = stats_key(v[j]);
            s += v[j];
            ++n;
            ex += v[j] > lim;
            kmin = k < kmin ? k : kmin;
            kmax = k > kmax ? k : kmax;
        }
    }
    auto add_d = [](double p, double q) { return p + q; };
    auto add_i = [](int p, int q) { return p + q; };
    s = stats_block_reduce(s, red_d, add_d);
    if (tid == 0) part.sum = s;
    n = stats_block_reduce(n, red_i, add_i);
    if (tid == 0) part.n = n;
    ex = stats_block_reduce(ex, red_i, add_i);
    if (tid == 0) part.exceed = ex;
    kmin = stats_block_reduce(kmin, red_k, [](unsigned long long p, unsigned long long q) { return q < p ? q : p; });
    if (tid == 0) part.kmin = kmin;
    kmax = stats_block_reduce(kmax, red_k, [](unsigned long long p, unsigned long long q) { return q > p ? q : p; });
    if (tid == 0) part.kmax = kmax;
    if (row == 0)                              // the status counts come from the first row's cluster
        for (int i = 0; i < 4; ++i) {
            const int c = status ? stats_block_reduce(sc[i], red_i, add_i) : (i == 0 ? (int)(hi - lo) : 0);
            if (tid == 0) part.st[i] = c;
        }
    cluster.sync();
    if (tid == 0) {
        double sum = 0.0;
        int nn = 0, ee = 0, tc[4] = {0, 0, 0, 0};
        unsigned long long mn = ~0ull, mx = 0ull;
        for (int r = 0; r < cs; ++r) {
            const StatsPart* p = cluster.map_shared_rank(&part, r);
            sum = r ? sum + p->sum : p->sum;
            nn += p->n;
            ee += p->exceed;
            mn = p->kmin < mn ? p->kmin : mn;
            mx = p->kmax > mx ? p->kmax : mx;
            if (row == 0)
                for (int i = 0; i < 4; ++i) tc[i] += p->st[i];
        }
        t_n = nn;
        t_mean = sum / nn;
        t_kmin = mn;
        t_kmax = mx;
        if (rank == 0) {
            const double nan = __longlong_as_double(0x7ff8000000000000ll);
            a.stats[row] = nn ? t_mean : nan;
            a.stats[2 * a.R + row] = nn ? stats_value(mn) : nan;
            a.stats[3 * a.R + row] = nn ? stats_value(mx) : nan;
            a.stats[4 * a.R + row] = (double)ee;
            if (row == 0)
                for (int i = 0; i < 4; ++i) a.counts[i] = tc[i];
        }
    }
    __syncthreads();
    const int nv = t_n;
    const double mean = t_mean;

    // ---- pass 2: squared deviations ----------------------------------------------------------------
    double ss = 0.0;
    if (nv) {
        for (int it = 0; it < rounds; ++it) {
            double v[HPF_STATS_UNROLL];
            bool in[HPF_STATS_UNROLL];
#pragma unroll
            for (int j = 0; j < HPF_STATS_UNROLL; ++j) {
                const size_t b = lo + ((size_t)it * HPF_STATS_UNROLL + j) * HPF_STATS_THREADS + tid;
                in[j] = b < hi && (!status || __ldg(status + b) == 0);
                v[j] = in[j] ? __ldg(x + b) : 0.0;
            }
#pragma unroll
            for (int j = 0; j < HPF_STATS_UNROLL; ++j) {
                if (!in[j]) continue;
                const double d = v[j] - mean;
                ss += d * d;
            }
        }
    }
    ss = stats_block_reduce(ss, red_d, add_d);
    if (tid == 0) part.ss = ss;
    cluster.sync();
    if (tid == 0 && rank == 0) {
        double t = 0.0;
        for (int r = 0; r < cs; ++r) {
            const double v = cluster.map_shared_rank(&part, r)->ss;
            t = r ? t + v : v;
        }
        a.stats[a.R + row] = nv ? sqrt(t / nv) : __longlong_as_double(0x7ff8000000000000ll);
    }

    // ---- pass 3+: radix select of the K quantiles ---------------------------------------------------
    if (K == 0) { cluster.sync(); return; }
    if (nv == 0) {
        if (rank == 0 && tid < K) a.stats[(size_t)(5 + tid) * a.R + row] = __longlong_as_double(0x7ff8000000000000ll);
        cluster.sync();
        return;
    }
    const unsigned long long kmn = t_kmin, kmx = t_kmax;
    // first digit: the highest 8-bit digit in which min and max differ (everything above is common)
    int shift = kmn == kmx ? 0 : ((63 - __clzll((long long)(kmn ^ kmx))) / 8) * 8;
    if (tid < K) {
        long long r = (long long)ceil(a.q[tid] * (double)nv);
        r = r < 1 ? 1 : r;
        q_rank[tid] = r;
        q_act[tid] = !(kmn == kmx || r == 1 || r == nv);
        q_key[tid] = (r == nv && kmn != kmx) ? kmx : kmn;
        q_pre[tid] = shift + 8 >= 64 ? 0ull : kmn >> (shift + 8);
    }
    __syncthreads();
    for (int buf = 0;; buf ^= 1, shift -= 8) {
        if (tid == 0) {                            // distinct prefixes of the active quantiles
            int nu = 0;
            for (int k = 0; k < K; ++k) {
                if (!q_act[k]) continue;
                int u = 0;
                while (u < nu && u_pre[u] != q_pre[k]) ++u;
                if (u == nu) u_pre[nu++] = q_pre[k];
                q_u[k] = u;
            }
            n_u = nu;
        }
        __syncthreads();
        const int nu = n_u;
        if (nu == 0) break;                        // the same decision in every CTA of the cluster
        int* hb = hist + buf * K * HPF_STATS_BINS;
        unsigned long long* kb = hkey + (size_t)buf * K * HPF_STATS_BINS;
        for (int i = tid; i < nu * HPF_STATS_BINS; i += HPF_STATS_THREADS) hb[i] = 0;
        __syncthreads();
        for (int it = 0; it < rounds; ++it) {
            double v[HPF_STATS_UNROLL];
            bool in[HPF_STATS_UNROLL];
#pragma unroll
            for (int j = 0; j < HPF_STATS_UNROLL; ++j) {
                const size_t b = lo + ((size_t)it * HPF_STATS_UNROLL + j) * HPF_STATS_THREADS + tid;
                in[j] = b < hi && (!status || __ldg(status + b) == 0);
                v[j] = in[j] ? __ldg(x + b) : 0.0;
            }
#pragma unroll
            for (int j = 0; j < HPF_STATS_UNROLL; ++j) {
                const unsigned long long k = stats_key(v[j]);
                const unsigned long long top = shift + 8 >= 64 ? 0ull : k >> (shift + 8);
                int idx = -1;
                if (in[j])
                    for (int u = 0; u < nu; ++u)
                        if (u_pre[u] == top) { idx = u * HPF_STATS_BINS + (int)((k >> shift) & 0xff); break; }
                // values of a row crowd into few bins: one atomic per group of equal bins in the warp
                const unsigned peers = __match_any_sync(0xffffffffu, idx);
                if (idx >= 0 && lane == __ffs(peers) - 1) {
                    atomicAdd(&hb[idx], __popc(peers));
                    kb[idx] = k;                   // read only when the bin holds one element
                }
            }
        }
        cluster.sync();
        // one warp per quantile: add the cluster's histograms of its prefix, find the bin of its rank
        for (int k = warp; k < K; k += HPF_STATS_WARPS) {
            if (!q_act[k]) continue;
            const int base = q_u[k] * HPF_STATS_BINS + lane * 8;
            int c[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                int t = 0;
                for (int r = 0; r < cs; ++r) t += cluster.map_shared_rank(hb, r)[base + j];
                c[j] = t;
                tot += t;
            }
            int incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int w = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += w;
            }
            const long long rk = q_rank[k];
            long long below = incl - tot;
            if (rk > below && rk <= incl) {          // exactly one lane
                int j = -1, cj = 0;
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    if (j >= 0) continue;
                    if (rk <= below + c[t]) { j = t; cj = c[t]; }
                    else below += c[t];
                }
                const int bin = lane * 8 + j;
                const unsigned long long pre = (q_pre[k] << 8) | (unsigned long long)bin;
                if (cj == 1) {
                    for (int r = 0; r < cs; ++r)
                        if (cluster.map_shared_rank(hb, r)[base + j] == 1) q_key[k] = cluster.map_shared_rank(kb, r)[base + j];
                    q_act[k] = 0;
                } else if (shift == 0) {
                    q_key[k] = pre;
                    q_act[k] = 0;
                } else {
                    q_pre[k] = pre;
                    q_rank[k] = rk - below;
                }
            }
        }
        __syncthreads();
    }
    if (rank == 0 && tid < K) a.stats[(size_t)(5 + tid) * a.R + row] = stats_value(q_key[tid]);
    cluster.sync();                                // keep this CTA's shared memory alive for the cluster
}
