// Lock-step batched harmonic Newton-Raphson for the LARGE networks (BASELINE configs 4, 5: 200-bus
// feeder, 1000-bus meshed network), structured step (hpf_structured.cuh), batches of hundreds to
// thousands of scenarios.
//
// harm_cta_kernel (hpf_kernels.cu) gives every scenario ONE persistent CTA: its border system (order
// 238 / 1198) is factorised by that CTA alone and the operator G (nZ x m complex, 119 MB for the
// 1000-bus network) is streamed once per scenario and iteration.  Here all scenarios of a wave take
// their Newton iteration TOGETHER, so that every phase is a throughput kernel over the whole batch:
//
//   round r:  ls_mismatch   CTA per active scenario: apply the pending update, phasors, mismatch
//                           (HG:313-390), convergence decision (HG:536), results of finished scenarios
//             ls_compact    next list of active slots (stable order)
//             ls_pack_vf  + zgemm   U0 = G[0:q,:] V_F            (tensor cores, hpf_zgemm.cuh)
//             ls_border     border systems [ldb x (nx+1)] of all active scenarios (HG:451-467 reduced)
//             batched LU    per 32-column panel: ls_panel (CTA per matrix: register sub-panels with
//                           partial pivoting) -> ls_swap_trsm (interchanges + U12) -> ls_update
//                           (A22 -= L21 U12 on the FP64 tensor cores, 128 x 128 tiles of ALL matrices)
//             ls_backsub    x_F
//             ls_uf + zgemm G (V_F + u_F) for all active scenarios: ONE complex GEMM [nZ x m][m x S]
//
// The number of active scenarios lives in device memory (nact[]); the host enqueues max_h + 1 rounds
// without synchronising (kernels of a round with no active scenario exit at once), so hpf_solve stays
// asynchronous and capturable.  Same Newton step as every other strategy (dx = J^-1 f); the sums of
// the two G products are formed by the tensor-core GEMM (different summation order: results agree to
// round-off, iteration counts are compared with the oracle in tests/test_gpu_parity.py).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

#define LS_NB 32                   // panel width
#define LS_PERM_INTS 100           // per slot: srcTop[32] | cnt | mvSrc[32] | mvDst[32]
#define LS_PANEL_FIXED_BYTES 29696   // orig 8192 | tmp 4096 | Ubuf 8192 | cand 8192 | keys, lists 1024
#define LS_UT 128                  // update tile (rows and columns)

struct LsArgs {
    int B, b0, nwave, S, flags;
    const double *P, *Q;
    const double2 *I_N, *wN;
    double thresh_h;
    int max_h;
    double *V_m, *V_a;
    double2* I_inj;
    int *n_iter_h, *status;
    double *err_h, *hist_h;
    double* state;  size_t state_stride;      // per-slot scenario state (carve() layout)
    double* M;      size_t mat_stride;        // per-slot border system, column-major
    int ldb;
    double2 *X, *GX, *U0;                     // [m x S], [nZ x S], [q x S] (row-major, ld = S)
    int *act, *nact, *flag, *itc, *stat, *info, *perm;
};

__global__ void ls_init_kernel(const LsArgs a) {
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < a.S; t += gridDim.x * blockDim.x) {
        a.act[t] = t;
        a.itc[t] = 0;
        a.info[t] = 0;
        a.flag[t] = 0;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { a.nact[0] = a.nwave; a.nact[1] = 0; }
}

// ---------------------------------------------------------------------------------------
// round start: pending update, mismatch, decision, results
__global__ void __launch_bounds__(256)
ls_mismatch_kernel(const DevNet net, const StructNet sn, const LsArgs a, const int cur, const int first) {
    __shared__ double red[72];
    const int tid = threadIdx.x;
    const int n = net.n, m = net.m, c = net.c, H = net.H, q = net.q, nH = net.nH;
    const int nZ = sn.nZ, nx = sn.nx, nth = m - 1;
    const size_t B = (size_t)a.B, S = (size_t)a.S;
    const int nin = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    for (int ai = blockIdx.x; ai < nin; ai += gridDim.x) {
        __syncthreads();
        const int slot = act[ai];
        const int b = a.b0 + slot;
        ScnSmem s = carve(a.state + (size_t)slot * a.state_stride, net, false);
        s.red = red;
        s.flag = reinterpret_cast<int*>(red + 66);
        double* rhs = s.rinv;
        if (first) {
            for (int t = tid; t < n; t += blockDim.x) {
                s.P[t] = a.P[t * B + b];
                s.Q[t] = a.Q[t * B + b];
            }
            for (int t = tid; t < q * H; t += blockDim.x) s.IN[t] = a.I_N[t * B + b];
            for (int t = tid; t < nH; t += blockDim.x) {
                if (t < n) {
                    s.Vm[t] = a.V_m[t * B + b];
                    s.Va[t] = a.V_a[t * B + b];
                } else {
                    s.Vm[t] = 0.1;                             // flat start of the harmonics (HG:183)
                    s.Va[t] = 0.0;
                }
            }
            if (tid == 0) a.stat[slot] = a.status[b];
        } else {
            // x_new = x + delta of the step solved in the previous round (HG:476-485):
            // u_Z = -V_Z - G (V_F + u_F) - w_N, polar conversion; F rows from x_F
            const double* xF = a.M + (size_t)slot * a.mat_stride + (size_t)nx * a.ldb;
            for (int z = tid; z < nZ; z += blockDim.x) {
                const int sz = z + m;
                const double2 w = a.wN[(size_t)z * B + b];
                const double2 g = a.GX[(size_t)z * S + ai];
                const double2 acc = make_double2(s.Vre[sz] + w.x + g.x, s.Vim[sz] + w.y + g.y);
                const double2 wv = cmul(make_double2(s.Ere[sz], -s.Eim[sz]), cneg(acc));
                const double vm = s.Vm[sz];
                s.Va[sz] += wv.y / vm;
                s.Vm[sz] = vm + wv.x;
            }
            for (int i = 1 + tid; i < m; i += blockDim.x) {
                s.Va[i] += xF[i - 1];
                if (i >= c) s.Vm[i] += xF[nth + i - c];
            }
            if (tid == 0 && a.info[slot]) {
                if (a.stat[slot] == HPF_ST_CONVERGED) a.stat[slot] = HPF_ST_SINGULAR;
                a.info[slot] = 0;
            }
        }
        const int it = a.itc[slot];                            // (read before the barriers below: thread 0 updates it)
        __syncthreads();
        const double err = cta_harmonic_mismatch(net, s, rhs);
        if (a.hist_h && tid == 0) a.hist_h[(size_t)it * B + b] = err;
        const bool cont = (err > a.thresh_h) && (it < a.max_h);
        if (cont) {
            if (tid == 0) { a.flag[ai] = 1; a.itc[slot] = it + 1; }
            continue;
        }
        int status = a.stat[slot];
        if (it >= a.max_h && status == HPF_ST_CONVERGED) status = HPF_ST_MAXITER;
        if (!(err < CUDART_INF)) status = HPF_ST_NONFINITE;
        for (int t = tid; t < nH; t += blockDim.x) {
            double vm = s.Vm[t], va = s.Va[t];
            if (!(a.flags & HPF_SOLVE_RAW)) {
                if (vm < 0.0) va += CUDART_PI;
                va = mod_twopi(va);
                if (vm < 0.0) vm = -vm;
            }
            a.V_m[t * B + b] = vm;
            a.V_a[t * B + b] = va;
        }
        if (a.I_inj)
            for (int t = tid; t < q * H; t += blockDim.x) a.I_inj[t * B + b] = s.Iinj[t];
        if (tid == 0) {
            a.n_iter_h[b] = it;
            a.err_h[b] = err;
            a.status[b] = status;
            a.flag[ai] = 0;
        }
    }
}

// stable compaction of the continuing slots into the other list (one CTA)
__global__ void __launch_bounds__(1024) ls_compact_kernel(const LsArgs a, const int cur) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nin = a.nact[cur];
    const int* in = a.act + (size_t)cur * a.S;
    int* out = a.act + (size_t)(cur ^ 1) * a.S;
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int t0 = 0; t0 < nin; t0 += 1024) {
        const int t = t0 + tid;
        const int f = (t < nin) ? (a.flag[t] != 0) : 0;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        const int pre = __popc(bal & ((1u << lane) - 1u));
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int off = base_s;
        for (int w = 0; w < warp; ++w) off += wsum[w];
        if (f) out[off + pre] = in[t];
        __syncthreads();
        if (tid == 0) { int tot = 0; for (int w = 0; w < 32; ++w) tot += wsum[w]; base_s += tot; }
        __syncthreads();
    }
    if (tid == 0) a.nact[cur ^ 1] = base_s;
}

// X[i][a] = V_i of the linear buses at the fundamental (operand of U0 = G[0:q,:] V_F)
__global__ void ls_pack_vf_kernel(const DevNet net, const LsArgs a, const int cur) {
    const int nact = a.nact[cur], m = net.m;
    const int* act = a.act + (size_t)cur * a.S;
    const long long tot = (long long)nact * m;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < tot; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / nact), ai = (int)(t - (long long)i * nact);
        const ScnSmem s = carve(a.state + (size_t)act[ai] * a.state_stride, net, false);
        a.X[(size_t)i * a.S + ai] = make_double2(s.Vre[i], s.Vim[i]);
    }
}

// X[i][a] = V_i + u_F,i with u_F = (j V_i) dtheta_i + E_i dV_m,i from the border solution
__global__ void ls_uf_kernel(const DevNet net, const StructNet sn, const LsArgs a, const int cur) {
    const int nact = a.nact[cur], m = net.m, c = net.c, nth = m - 1;
    const int* act = a.act + (size_t)cur * a.S;
    const long long tot = (long long)nact * m;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < tot; t += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(t / nact), ai = (int)(t - (long long)i * nact);
        const int slot = act[ai];
        const ScnSmem s = carve(a.state + (size_t)slot * a.state_stride, net, false);
        const double* xF = a.M + (size_t)slot * a.mat_stride + (size_t)sn.nx * a.ldb;
        const double dth = (i >= 1) ? xF[i - 1] : 0.0;
        const double dvm = (i >= c) ? xF[nth + i - c] : 0.0;
        const double2 vi = make_double2(s.Vre[i], s.Vim[i]);
        a.X[(size_t)i * a.S + ai] = make_double2(vi.x + (-vi.y * dth + s.Ere[i] * dvm),
                                                 vi.y + (vi.x * dth + s.Eim[i] * dvm));
    }
}

// ---------------------------------------------------------------------------------------
// border systems: 32 x 32 tiles of (power row i, column), lanes over the columns while the entries
// are formed (Y1 and G rows are read contiguously), transposed through shared memory so that the
// column-major matrix is written with lanes over the rows
#define LS_NBC 256                 // (row, nonlinear neighbour) pairs of a 32-row tile kept in shared memory
__global__ void __launch_bounds__(256)
ls_border_kernel(const DevNet net, const StructNet sn, const LsArgs a, const int cur) {
    __shared__ double tre[32][33], tim[32][33];
    __shared__ double nbc[7][LS_NBC];          // per pair: dS_i/dtheta_b (2), dS_i/dV_m,b (2), conj(E_b) (2), 1/V_m,b
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = net.n, m = net.m, c = net.c, nH = net.nH;
    const int nx = sn.nx, nth = m - 1, ldb = a.ldb;
    const size_t B = (size_t)a.B, S = (size_t)a.S;
    const int nact = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    const int ntr = (nth + 31) / 32, ntc = (nx + 1 + 31) / 32;
    const long long items = (long long)nact * ntr * ntc;
    for (long long w = blockIdx.x; w < items; w += gridDim.x) {
        const int ai = (int)(w / (ntr * ntc));
        const int rem = (int)(w - (long long)ai * ntr * ntc);
        const int tc = rem / ntr, tr = rem - tc * ntr;
        const int slot = act[ai], b = a.b0 + slot;
        const ScnSmem s = carve(a.state + (size_t)slot * a.state_stride, net, false);
        const double* rhs = s.rinv;
        double* Mb = a.M + (size_t)slot * a.mat_stride;
        const int col = tc * 32 + lane;
        const bool is_rhs = (col == nx), is_v = (col >= nth);
        const int j = is_rhs ? 0 : (is_v ? c + (col - nth) : col + 1);
        double2 vj = make_double2(0.0, 0.0), ej = vj;
        if (col < nx) {
            vj = make_double2(s.Vre[j], s.Vim[j]);
            ej = make_double2(s.Ere[j], s.Eim[j]);
        }
        // the column-independent factors of the eliminated nonlinear neighbours, once per tile
        const int i0 = 1 + tr * 32, iend = (i0 + 32 < m) ? i0 + 32 : m;
        const int e0 = sn.nbr_ptr[i0], e1 = sn.nbr_ptr[iend];
        const bool pre = e1 - e0 <= LS_NBC;
        if (pre) {
            for (int ri = warp; ri < 32; ri += 8) {
                const int i = i0 + ri;
                if (i >= m) break;
                const double2 vi = make_double2(s.Vre[i], s.Vim[i]);
                const double2 jvi = cmulj(vi);
                for (int en = sn.nbr_ptr[i] + lane; en < sn.nbr_ptr[i + 1]; en += 32) {
                    const int bk = m + sn.nbr_idx[en];
                    const double2 y = ldg2(net.Y + (size_t)i * n + bk);
                    const double2 vb = make_double2(s.Vre[bk], s.Vim[bk]);
                    const double2 eb = make_double2(s.Ere[bk], s.Eim[bk]);
                    const double2 ak = cmul(jvi, cconj(cneg(cmul(y, vb))));
                    const double2 vk = cmul(vi, cconj(cmul(y, eb)));
                    const int t = en - e0;
                    nbc[0][t] = ak.x; nbc[1][t] = ak.y; nbc[2][t] = vk.x; nbc[3][t] = vk.y;
                    nbc[4][t] = eb.x; nbc[5][t] = -eb.y; nbc[6][t] = 1.0 / s.Vm[bk];
                }
            }
            __syncthreads();
        }
#pragma unroll 1
        for (int ri = warp; ri < 32; ri += 8) {
            const int i = i0 + ri;
            double2 e = make_double2(0.0, 0.0);
            if (i < m && col <= nx) {
                const double2 vi = make_double2(s.Vre[i], s.Vim[i]);
                const double2 jvi = cmulj(vi);
                if (is_rhs) {
                    // f_S of bus i: Re at row i-1, Im at row (nH-1) + (i-1) - (c-1) of the mismatch
                    e = make_double2(-rhs[i - 1], (i >= c) ? -rhs[(nH - 1) + (i - 1) - (c - 1)] : 0.0);
                } else {
                    const double2 y = ldg2(net.Y + (size_t)i * n + j);
                    if (is_v) {
                        e = cmul(vi, cconj(cmul(y, ej)));
                        if (i == j) e = cadd(cmul(make_double2(s.Ere[i], s.Eim[i]), cconj(s.I1[i])), e);
                    } else {
                        const double2 yv = cmul(y, vj);
                        e = cmul(jvi, cconj((i == j) ? csub(s.I1[i], yv) : cneg(yv)));
                    }
                }
                const double2 tj = is_v ? ej : cmulj(vj);
                for (int en = sn.nbr_ptr[i]; en < sn.nbr_ptr[i + 1]; ++en) {   // nonlinear neighbours of bus i
                    const int k = sn.nbr_idx[en], bk = m + k;
                    double2 ak, vk, ceb;
                    double rvb;
                    if (pre) {
                        const int t = en - e0;
                        ak = make_double2(nbc[0][t], nbc[1][t]);
                        vk = make_double2(nbc[2][t], nbc[3][t]);
                        ceb = make_double2(nbc[4][t], nbc[5][t]);
                        rvb = nbc[6][t];
                    } else {
                        const double2 y = ldg2(net.Y + (size_t)i * n + bk);
                        const double2 vb = make_double2(s.Vre[bk], s.Vim[bk]);
                        const double2 eb = make_double2(s.Ere[bk], s.Eim[bk]);
                        ak = cmul(jvi, cconj(cneg(cmul(y, vb))));
                        vk = cmul(vi, cconj(cmul(y, eb)));
                        ceb = cconj(eb);
                        rvb = 1.0 / s.Vm[bk];
                    }
                    double2 uu;
                    if (is_rhs) {                       // u0 of the fundamental nonlinear row k (closed form)
                        const double2 wk = a.wN[(size_t)k * B + b];
                        const double2 g = a.U0[(size_t)k * S + ai];
                        uu = make_double2(-(s.Vre[bk] + wk.x + g.x), -(s.Vim[bk] + wk.y + g.y));
                    } else {
                        uu = cmul(ldg2(sn.G + (size_t)k * m + j), tj);
                    }
                    const double2 ce = cmul(ceb, uu);
                    const double dth = ce.y * rvb, dvm = ce.x;
                    e.x -= ak.x * dth + vk.x * dvm;
                    e.y -= ak.y * dth + vk.y * dvm;
                }
            }
            tre[ri][lane] = e.x;
            tim[ri][lane] = e.y;
        }
        __syncthreads();
        {
            const int i = i0 + lane;
            for (int cl = warp; cl < 32; cl += 8) {
                const int cc = tc * 32 + cl;
                if (i < m && cc <= nx) {
                    Mb[(i - 1) + (size_t)cc * ldb] = tre[lane][cl];
                    if (i >= c) Mb[(nth + i - c) + (size_t)cc * ldb] = tim[lane][cl];
                }
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------
// Batched LU, step 1: the 32-column panel at k0 of every active matrix, one CTA per matrix.
// The panel is staged in shared memory when it fits (else worked on in place, L2) and factorised
// in sub-panels of W columns held in REGISTERS: thread t owns the rows t, t + T, .. (R of them) of
// the sub-panel for its W elimination steps - rows do not move, every register row carries the
// position it would have after the classic interchanges and is scattered there afterwards; argmax
// with warp REDUX on the bit patterns (ties -> lowest position = idamax), one block barrier per step.  After a sub-panel the
// moved rows of the panel's other columns are exchanged, the columns to its right take the
// W x W unit-lower solve and the rank-W update.  W = 32, R = 1 when every row has a thread (no
// in-panel update at all); W = 8, R <= 4 for up to 4 T rows.  The net permutation of the panel is
// left in perm[slot] as lists (see ls_swap_trsm_kernel).  Panels are taken in PAIRS (launch_ls_lu): the
// first panel is applied to the second panel's 32 columns only, the rest of the trailing matrix takes
// both panels in one rank-64 tensor-core pass (half the HBM passes over the matrices).
template <int R, int W>
__global__ void __launch_bounds__(512, 1)
ls_panel_kernel(const LsArgs a, const int cur, const int N, const int k0, const int staged, const int left) {
    extern __shared__ __align__(16) unsigned char ls_sm[];
    int* orig = reinterpret_cast<int*>(ls_sm);                          // [rows <= 2048] original row now at a position
    double* tmp = reinterpret_cast<double*>(ls_sm + 2048 * 4);          // [16][32]
    double* Ubuf = tmp + 16 * 32;                                       // [W <= 32][32]
    double* cand = Ubuf + 32 * 32;                                      // [2][16][W <= 32] candidate pivot row of every warp
    unsigned* rkey = reinterpret_cast<unsigned*>(cand + 2 * 16 * 32);   // [2][16][2]
    int* redi = reinterpret_cast<int*>(rkey + 64);                      // [2][16]
    int* mvs = redi + 32;                                               // [16] moved rows: source
    int* mvd = mvs + 16;                                                // [16] destination
    int* mcnt = mvd + 16;                                               // [2]
    double* stage = reinterpret_cast<double*>(ls_sm + LS_PANEL_FIXED_BYTES);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, T = blockDim.x, nw = T >> 5;
    const int rows = N - k0, nb = min(LS_NB, rows), ld = a.ldb;
    const int nact = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    for (int ai = blockIdx.x; ai < nact; ai += gridDim.x) {
        const int slot = act[ai];
        double* A = a.M + (size_t)slot * a.mat_stride;
        __syncthreads();
        for (int t = tid; t < rows; t += T) orig[t] = t;
        if (tid == 0) mcnt[1] = 0;
        double* PB = staged ? stage : A + (size_t)k0 * ld + k0;
        const size_t ps = staged ? (size_t)rows : (size_t)ld;
        if (staged) {
            for (int t = tid; t < rows * nb; t += T) {
                const int jj = t / rows, i = t - jj * rows;
                stage[t] = A[(size_t)(k0 + jj) * ld + k0 + i];
            }
        }
        __syncthreads();
        int bad = 0;
        for (int o = 0; o < nb; o += W) {
            const int w = min(W, nb - o);
            const int rows_s = rows - o;
            double v[R][W];
            int pos[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int i = tid + r * T;
                pos[r] = (i < rows_s) ? i : -1;
#pragma unroll
                for (int jj = 0; jj < W; ++jj)
                    v[r][jj] = (pos[r] >= 0 && jj < w) ? PB[(size_t)(o + jj) * ps + o + i] : 0.0;
            }
            if (tid == 0) mcnt[0] = 0;
#pragma unroll
            for (int j = 0; j < W; ++j) {
                if (j < w) {
                    // thread-local best row, then warp, then CTA (every warp reduces the partials redundantly)
                    unsigned hi = 0u, lo = 0u, pp = 0x7fffffffu;
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (pos[r] >= j) {
                            double av = fabs(v[r][j]);
                            if (av != av) av = CUDART_INF;               // a NaN candidate must surface as a bad pivot
                            const unsigned h2 = (unsigned)__double2hiint(av), l2 = (unsigned)__double2loint(av);
                            if (pp == 0x7fffffffu || h2 > hi || (h2 == hi && (l2 > lo || (l2 == lo && (unsigned)pos[r] < pp)))) {
                                hi = h2; lo = l2; pp = (unsigned)pos[r];
                            }
                        }
                    }
                    unsigned mhi = __reduce_max_sync(0xffffffffu, hi);
                    unsigned mlo = __reduce_max_sync(0xffffffffu, (hi == mhi) ? lo : 0u);
                    unsigned p = __reduce_min_sync(0xffffffffu, (hi == mhi && lo == mlo) ? pp : 0x7fffffffu);
                    if constexpr (W <= 8) {
                    // ONE barrier per elimination step: every warp publishes its candidate (key, position
                    // and the row itself); after the barrier every warp picks the winner redundantly and
                    // reads the pivot row from the winning warp's slot (slots alternate with the parity
                    // of the step: a warp is at most one step ahead of the slowest one)
                    const int sb = (j & 1) * 16;
                    if (lane == 0) { rkey[2 * (sb + warp)] = mhi; rkey[2 * (sb + warp) + 1] = mlo; redi[sb + warp] = (int)p; }
                    {
                        double* cw = cand + (sb + warp) * W;
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            if (pos[r] >= 0 && (unsigned)pos[r] == p) {
#pragma unroll
                                for (int jj = j; jj < W; ++jj) cw[jj] = v[r][jj];
                            }
                        }
                    }
                    __syncthreads();
                    unsigned ww;
                    {
                        const unsigned h2 = (lane < nw) ? rkey[2 * (sb + lane)] : 0u;
                        const unsigned l2 = (lane < nw) ? rkey[2 * (sb + lane) + 1] : 0u;
                        const unsigned p2 = (lane < nw) ? (unsigned)redi[sb + lane] : 0x7fffffffu;
                        mhi = __reduce_max_sync(0xffffffffu, h2);
                        mlo = __reduce_max_sync(0xffffffffu, (h2 == mhi) ? l2 : 0u);
                        p = __reduce_min_sync(0xffffffffu, (h2 == mhi && l2 == mlo && p2 != 0x7fffffffu) ? p2 : 0x7fffffffu);
                        ww = __reduce_min_sync(0xffffffffu, (h2 == mhi && l2 == mlo && p2 == p && p2 != 0x7fffffffu) ? (unsigned)lane : 0x7fffffffu);
                    }
                    const double best = __hiloint2double((int)mhi, (int)mlo);
                    if ((!(best > 0.0) || !(best < CUDART_INF)) && bad == 0) bad = k0 + o + j + 1;
                    const int pi = (p == 0x7fffffffu) ? j : (int)p;
                    const double* prow = cand + (sb + (ww == 0x7fffffffu ? 0u : ww)) * W;
                    if (tid == 0 && pi != j) { const int x = orig[o + j]; orig[o + j] = orig[o + pi]; orig[o + pi] = x; }
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (pos[r] == pi) pos[r] = j;
                        else if (pos[r] == j) pos[r] = pi;
                    }
                    const double rp = 1.0 / prow[j];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (pos[r] > j) {
                            const double l = v[r][j] * rp;
                            v[r][j] = l;
#pragma unroll
                            for (int jj = j + 1; jj < W; ++jj) v[r][jj] = fma(-l, prow[jj], v[r][jj]);
                        }
                    }
                    } else {
                        // (32-column register panel: publishing every warp's candidate row would cost the owner
                        // lanes up to 32 stores per step - two barriers, the winner alone publishes its row)
                        double* prow_s = cand;
                    if (lane == 0) { rkey[2 * warp] = mhi; rkey[2 * warp + 1] = mlo; redi[warp] = (int)p; }
                    __syncthreads();
                    {
                        const unsigned h2 = (lane < nw) ? rkey[2 * lane] : 0u;
                        const unsigned l2 = (lane < nw) ? rkey[2 * lane + 1] : 0u;
                        const unsigned p2 = (lane < nw) ? (unsigned)redi[lane] : 0x7fffffffu;
                        mhi = __reduce_max_sync(0xffffffffu, h2);
                        mlo = __reduce_max_sync(0xffffffffu, (h2 == mhi) ? l2 : 0u);
                        p = __reduce_min_sync(0xffffffffu, (h2 == mhi && l2 == mlo && p2 != 0x7fffffffu) ? p2 : 0x7fffffffu);
                    }
                    const double best = __hiloint2double((int)mhi, (int)mlo);
                    if ((!(best > 0.0) || !(best < CUDART_INF)) && bad == 0) bad = k0 + o + j + 1;
                    const int pi = (p == 0x7fffffffu) ? j : (int)p;
                    if (tid == 0 && pi != j) { const int x = orig[o + j]; orig[o + j] = orig[o + pi]; orig[o + pi] = x; }
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (pos[r] == pi) pos[r] = j;
                        else if (pos[r] == j) pos[r] = pi;
                        if (pos[r] == j) {
#pragma unroll
                            for (int jj = j; jj < W; ++jj) prow_s[jj] = v[r][jj];
                        }
                    }
                    __syncthreads();
                    const double rp = 1.0 / prow_s[j];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (pos[r] > j) {
                            const double l = v[r][j] * rp;
                            v[r][j] = l;
#pragma unroll
                            for (int jj = j + 1; jj < W; ++jj) v[r][jj] = fma(-l, prow_s[jj], v[r][jj]);
                        }
                    }
                    }
                }
            }
            // factored sub-panel back at the rows' final positions; moved rows of the other columns
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (pos[r] >= 0) {
#pragma unroll
                    for (int jj = 0; jj < W; ++jj)
                        if (jj < w) PB[(size_t)(o + jj) * ps + o + pos[r]] = v[r][jj];
                    if (W < LS_NB && pos[r] != tid + r * T) {   // (compile-time false for W = 32)
                        const int e = atomicAdd(mcnt, 1);
                        mvs[e] = o + tid + r * T;
                        mvd[e] = o + pos[r];
                    }
                }
            }
            if constexpr (W < LS_NB) {
                __syncthreads();
                const int cnt = mcnt[0];
                const int e = tid >> 5, jc = tid & 31;
                const bool other = e < cnt && jc < nb && (jc < o || jc >= o + w);
                if (other) tmp[e * 32 + jc] = PB[(size_t)jc * ps + mvs[e]];
                __syncthreads();
                if (other) PB[(size_t)jc * ps + mvd[e]] = tmp[e * 32 + jc];
                __syncthreads();
                // columns to the right inside the panel: unit-lower solve with the sub-panel's L11 ...
                const int nright = nb - (o + w);
                if (tid >= nright && tid < 32) {
#pragma unroll
                    for (int k = 0; k < W; ++k) Ubuf[k * 32 + tid] = 0.0;
                }
                if (tid < nright) {
                    const int jc2 = o + w + tid;
                    double u[W];
#pragma unroll
                    for (int k = 0; k < W; ++k) u[k] = (k < w) ? PB[(size_t)jc2 * ps + o + k] : 0.0;
#pragma unroll
                    for (int k = 1; k < W; ++k) {
                        if (k < w) {
                            double acc = u[k];
#pragma unroll
                            for (int s2 = 0; s2 < k; ++s2) acc = fma(-PB[(size_t)(o + s2) * ps + o + k], u[s2], acc);
                            u[k] = acc;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < W; ++k) {
                        if (k < w) PB[(size_t)jc2 * ps + o + k] = u[k];
                        Ubuf[k * 32 + tid] = u[k];
                    }
                }
                __syncthreads();
                // ... and the rank-w update of the rows below (multipliers in registers; 8 columns at a
                // time with all loads issued before the first FMA: in place in global memory every
                // dependent load -> FMA -> store round trip costs an L2 latency)
                for (int t0 = 0; t0 < nright; t0 += 8) {
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (pos[r] >= w) {
                            double* dst = PB + (size_t)(o + w + t0) * ps + o + pos[r];
                            double cb[8];
#pragma unroll
                            for (int u = 0; u < 8; ++u) cb[u] = (t0 + u < nright) ? dst[(size_t)u * ps] : 0.0;
#pragma unroll
                            for (int k = 0; k < W; ++k) {
                                const double l = -v[r][k];
#pragma unroll
                                for (int u = 0; u < 8; u += 2) {
                                    const double2 uu = *reinterpret_cast<const double2*>(Ubuf + k * 32 + t0 + u);
                                    cb[u] = fma(l, uu.x, cb[u]);
                                    cb[u + 1] = fma(l, uu.y, cb[u + 1]);
                                }
                            }
#pragma unroll
                            for (int u = 0; u < 8; ++u)
                                if (t0 + u < nright) dst[(size_t)u * ps] = cb[u];
                        }
                    }
                }
            }
            __syncthreads();
        }
        if (staged) {
            for (int t = tid; t < rows * nb; t += T) {
                const int jj = t / rows, i = t - jj * rows;
                A[(size_t)(k0 + jj) * ld + k0 + i] = stage[t];
            }
        }
        // net permutation of the panel: rows that end in the top block come from anywhere, rows that
        // end below it always come from the top block
        int* pg = a.perm + (size_t)slot * LS_PERM_INTS;
        for (int t = tid; t < rows; t += T) {
            const int src = orig[t];
            if (t < nb) pg[t] = src;
            else if (src != t) {
                const int e = atomicAdd(mcnt + 1, 1);
                pg[33 + e] = src;
                pg[65 + e] = t;
            }
        }
        __syncthreads();
        if (tid == 0) {
            pg[32] = mcnt[1];
            if (bad && a.info[slot] == 0) a.info[slot] = bad;
        }
        // second panel of a pair: its interchanges also move the rows of the first panel's L21 (the
        // `left` columns before k0), which the deferred rank-64 update reads
        if (tid < left) {
            double* col = A + (size_t)(k0 - left + tid) * ld + k0;
            double vt[LS_NB];
#pragma unroll
            for (int t = 0; t < LS_NB; ++t) vt[t] = (t < nb) ? col[pg[t]] : 0.0;
            const int cnt = mcnt[1];
            for (int e = 0; e < cnt; ++e) col[pg[65 + e]] = col[pg[33 + e]];
#pragma unroll
            for (int t = 0; t < LS_NB; ++t)
                if (t < nb) col[t] = vt[t];
        }
    }
}

// step 2: the panel's interchanges and U12 = L11^-1 A12 for every column to the right (incl. the
// right-hand side, column N): one thread per column, 32 values in registers; L11 (and, for the second
// panel of a pair, the first panel's multipliers of this panel's pivot rows) broadcast from shared
// memory two at a time (LDS.128).  Every CTA takes a contiguous range of (matrix, 128-column chunk) items.
#define LS_ST 128
__global__ void __launch_bounds__(LS_ST, 4)
ls_swap_trsm_kernel(const LsArgs a, const int cur, const int N, const int k0, const int pair) {
    __shared__ __align__(16) double L11[LS_NB][LS_NB + 2];
    __shared__ __align__(16) double Ltop[LS_NB][LS_NB + 2];
    __shared__ int pl[LS_PERM_INTS];
    const int tid = threadIdx.x;
    const int nb = min(LS_NB, N - k0), cr = k0 + nb, ld = a.ldb;
    const int nact = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    const int nchunk = (N + 1 - cr + LS_ST - 1) / LS_ST;
    const long long items = (long long)nact * nchunk;
    const long long per = (items + gridDim.x - 1) / gridDim.x;
    const long long w0 = (long long)blockIdx.x * per, w1 = (w0 + per < items) ? w0 + per : items;
    int last = -1;
    for (long long w = w0; w < w1; ++w) {
        const int ai = (int)(w / nchunk), ch = (int)(w - (long long)ai * nchunk);
        const int slot = act[ai];
        double* A = a.M + (size_t)slot * a.mat_stride;
        if (ai != last) {
            __syncthreads();
            for (int t = tid; t < LS_NB * LS_NB; t += LS_ST) {
                const int cc = t / LS_NB, r = t - cc * LS_NB;
                L11[r][cc] = (r < nb && cc < nb) ? A[(size_t)(k0 + cc) * ld + k0 + r] : 0.0;
                if (pair) Ltop[r][cc] = A[(size_t)(k0 - LS_NB + cc) * ld + k0 + r];
            }
            if (tid < LS_PERM_INTS) pl[tid] = a.perm[(size_t)slot * LS_PERM_INTS + tid];
            __syncthreads();
            last = ai;
        }
        const int cc = cr + ch * LS_ST + tid;
        if (cc > N) continue;
        double* col = A + (size_t)cc * ld + k0;
        double v[LS_NB];
#pragma unroll
        for (int t = 0; t < LS_NB; ++t) v[t] = (t < nb) ? col[pl[t]] : 0.0;
        const int cnt = pl[32];
        for (int e = 0; e < cnt; ++e) col[pl[65 + e]] = col[pl[33 + e]];
        if (pair) {
            // the first panel's contribution to the 32 pivot rows of this panel (deferred update)
            const double2* u1 = reinterpret_cast<const double2*>(col - LS_NB);
#pragma unroll 4
            for (int k = 0; k < LS_NB; k += 2) {
                const double2 u = u1[k >> 1];
#pragma unroll
                for (int t = 0; t < LS_NB; ++t) {
                    const double2 l = *reinterpret_cast<const double2*>(&Ltop[t][k]);
                    v[t] = fma(-l.x, u.x, v[t]);
                    v[t] = fma(-l.y, u.y, v[t]);
                }
            }
        }
#pragma unroll
        for (int t = 1; t < LS_NB; ++t) {
            double acc = v[t];
#pragma unroll
            for (int s2 = 0; s2 + 1 < t; s2 += 2) {
                const double2 l = *reinterpret_cast<const double2*>(&L11[t][s2]);
                acc = fma(-l.x, v[s2], acc);
                acc = fma(-l.y, v[s2 + 1], acc);
            }
            if (t & 1) acc = fma(-L11[t][t - 1], v[t - 1], acc);
            v[t] = acc;
        }
#pragma unroll
        for (int t = 0; t < LS_NB; ++t)
            if (t < nb) col[t] = v[t];
    }
}

// step 3: C -= L U on the FP64 tensor cores for rows >= rlo, columns clo .. chi of every active matrix,
// L = columns kb .. kb+K-1, U = rows kb .. kb+K-1 (K = 32: one panel; K = 64: a pair of panels).  Work
// item = one 128 x TC tile of one matrix; every CTA takes a CONTIGUOUS range of items (column tiles
// fastest) so that the L slice of a row tile is staged once for all its column tiles.  Same fragment
// mapping as lub_update_big (hpf_lu_blocked.cuh): the product is formed transposed so that the C
// fragment is a 16-byte access of the column-major matrix.
template <int K, int TR, int TC, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB)
ls_update_kernel(const LsArgs a, const int cur, const int N, const int kb, const int rlo, const int clo, const int chi) {
    extern __shared__ __align__(16) double ls_us[];
    constexpr int SU = K + 4, SL = TR + 4, NSR = TR / 32, NSUB = NSR * (TC / 32), NWARP = NT / 32;
    double* Ls = ls_us;                           // [K][SL]  Ls[k][r] = L[r0 + r][kb + k] (negated when the fragment is loaded)
    double* Us = Ls + K * SL;                 // [TC][SU]     Us[c][k] = U[kb + k][c0 + c]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ld = a.ldb;
    const int nact = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    const int ntr = (N - rlo + TR - 1) / TR, ntc = (chi + 1 - clo + TC - 1) / TC;
    // A strip = one row tile of one matrix, swept over its column tiles (the L slice is staged once per
    // strip); CTA b takes the strips b, b + grid, ..: neighbouring CTAs sweep neighbouring row tiles of
    // the SAME matrix at the same time, so the U slice of a column tile is fetched from HBM once and
    // served to the other row tiles by L2 (contiguous item ranges per CTA re-read it from HBM for every
    // row tile: ncu 8.2 GB read against 3.9 GB written by the first update of 512 systems of order 1038)
    const long long strips = (long long)nact * ntr;
    const int fr = lane >> 2, fk = lane & 3;
    for (long long sidx = blockIdx.x; sidx < strips; sidx += gridDim.x)
    for (int tc = 0; tc < ntc; ++tc) {
        const int ai = (int)(sidx / ntr), tr = (int)(sidx - (long long)ai * ntr);
        double* A = a.M + (size_t)act[ai] * a.mat_stride;
        const int r0 = rlo + tr * TR, c0 = clo + tc * TC;
        __syncthreads();                                          // previous item's slices consumed
        if (tc == 0) {                                            // (asynchronous like the U slice; r0 is even)
            for (int t = tid; t < K * (TR >> 1); t += NT) {
                const int k = t / (TR >> 1), r = (t - k * (TR >> 1)) << 1;
                const int nbytes = (r0 + r + 1 < N) ? 16 : ((r0 + r < N) ? 8 : 0);
                lub_cp_async16(Ls + k * SL + r, nbytes ? A + (size_t)(kb + k) * ld + r0 + r : A, nbytes);
            }
        }
        for (int t = tid; t < TC * (K >> 1); t += NT) {
            const int cc = t / (K >> 1), k = (t - cc * (K >> 1)) << 1;
            const bool in = c0 + cc <= chi;
            lub_cp_async16(Us + cc * SU + k, in ? A + (size_t)(c0 + cc) * ld + kb + k : A, in ? 16 : 0);
        }
        lub_cp_async_commit();
        // the C fragment of the warp's first sub-tile is requested BEFORE the wait for the slices: its
        // HBM latency overlaps their staging
        double acc[4][4][2];
        auto load_c = [&](const int st) {
            const int sc = st / NSR, sr = st - sc * NSR;
            const int cb = c0 + sc * 32, rbb = r0 + sr * 32;
#pragma unroll
            for (int ic = 0; ic < 4; ++ic)
#pragma unroll
                for (int ir = 0; ir < 4; ++ir) {
                    const int cc = cb + 8 * ic + fr, r = rbb + 8 * ir + 2 * fk;
                    if (cc <= chi && r + 1 < N) {
                        const double2 v2 = *reinterpret_cast<const double2*>(A + (size_t)cc * ld + r);
                        acc[ic][ir][0] = v2.x; acc[ic][ir][1] = v2.y;
                    } else {
                        acc[ic][ir][0] = (cc <= chi && r < N) ? A[(size_t)cc * ld + r] : 0.0;
                        acc[ic][ir][1] = 0.0;
                    }
                }
        };
        load_c(warp);
        lub_cp_async_wait();
        __syncthreads();
        for (int st = warp; st < NSUB; st += NWARP) {
            const int sc = st / NSR, sr = st - sc * NSR;
            const int cb = c0 + sc * 32, rbb = r0 + sr * 32;
            if (cb > chi || rbb >= N) continue;
            if (st != warp) load_c(st);
            const double* us = Us + (sc * 32 + fr) * SU + fk;
            const double* ls = Ls + fk * SL + sr * 32 + fr;
#pragma unroll 2
            for (int kk = 0; kk < K; kk += 4) {
                double af[4], bf[4];
#pragma unroll
                for (int ic = 0; ic < 4; ++ic) af[ic] = us[(8 * ic) * SU + kk];
#pragma unroll
                for (int ir = 0; ir < 4; ++ir) {                 // -L: sign flip on the high word (integer pipe)
                    const double l = ls[kk * SL + 8 * ir];
                    bf[ir] = __hiloint2double(__double2hiint(l) ^ (int)0x80000000, __double2loint(l));
                }
#pragma unroll
                for (int ic = 0; ic < 4; ++ic)
#pragma unroll
                    for (int ir = 0; ir < 4; ++ir) dmma884(acc[ic][ir][0], acc[ic][ir][1], af[ic], bf[ir]);
            }
#pragma unroll
            for (int ic = 0; ic < 4; ++ic)
#pragma unroll
                for (int ir = 0; ir < 4; ++ir) {
                    const int cc = cb + 8 * ic + fr, r = rbb + 8 * ir + 2 * fk;
                    if (cc <= chi && r + 1 < N) {
                        *reinterpret_cast<double2*>(A + (size_t)cc * ld + r) = make_double2(acc[ic][ir][0], acc[ic][ir][1]);
                    } else if (cc <= chi && r < N) {
                        A[(size_t)cc * ld + r] = acc[ic][ir][0];
                    }
                }
        }
    }
}

// step 4: blocked back substitution U x = y (y = column N), one CTA per matrix
__global__ void __launch_bounds__(256)
ls_backsub_kernel(const LsArgs a, const int cur, const int N) {
    __shared__ double U11[LS_NB][LS_NB + 1];
    __shared__ double xs[LS_NB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, ld = a.ldb;
    const int nact = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    for (int ai = blockIdx.x; ai < nact; ai += gridDim.x) {
        double* A = a.M + (size_t)act[ai] * a.mat_stride;
        double* y = A + (size_t)N * ld;
        for (int kb = ((N - 1) / LS_NB) * LS_NB; kb >= 0; kb -= LS_NB) {
            const int nb = min(LS_NB, N - kb);
            __syncthreads();
            for (int t = tid; t < nb * nb; t += 256) {
                const int cc = t / nb, r = t - cc * nb;
                U11[r][cc] = A[(size_t)(kb + cc) * ld + kb + r];
            }
            __syncthreads();
            if (warp == 0) {
                double v = (lane < nb) ? y[kb + lane] : 0.0;
                for (int j = nb - 1; j >= 0; --j) {
                    const double d = U11[j][j];
                    const double xj = __shfl_sync(0xffffffffu, v, j) / d;
                    if (lane == j) v = xj;
                    else if (lane < j) v = fma(-U11[lane][j], xj, v);
                }
                if (lane < nb) { y[kb + lane] = v; xs[lane] = v; }
            }
            __syncthreads();
            for (int i = tid; i < kb; i += 256) {
                double acc = y[i];
                for (int j = 0; j < nb; ++j) acc = fma(-A[(size_t)(kb + j) * ld + i], xs[j], acc);
                y[i] = acc;
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------
// Fundamental Newton-Raphson (HG:244-275) in lock step: `nf` is the one-harmonic view of the network
// (H = 1, N = Nf); the dense Jacobians [ldb x (Nf+1)] of all active scenarios go through the batched LU.
__global__ void __launch_bounds__(256)
ls_fund_mismatch_kernel(const DevNet nf, const LsArgs a, const int cur, const int first) {
    __shared__ double red[72];
    const int tid = threadIdx.x, n = nf.n, c = nf.c, Nf = nf.N;
    const size_t B = (size_t)a.B;
    const int nin = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    for (int ai = blockIdx.x; ai < nin; ai += gridDim.x) {
        __syncthreads();
        const int slot = act[ai];
        const int b = a.b0 + slot;
        ScnSmem s = carve(a.state + (size_t)slot * a.state_stride, nf, false);
        s.red = red;
        s.flag = reinterpret_cast<int*>(red + 66);
        double* rhs = s.rinv;
        if (first) {
            for (int t = tid; t < n; t += blockDim.x) {
                s.P[t] = a.P[t * B + b];
                s.Q[t] = a.Q[t * B + b];
                s.Vm[t] = 1.0;                                 // flat start (HG:174-184)
                s.Va[t] = 0.0;
            }
            if (tid == 0) a.stat[slot] = HPF_ST_CONVERGED;
        } else {
            const double* dx = a.M + (size_t)slot * a.mat_stride + (size_t)Nf * a.ldb;
            for (int t = tid; t < Nf; t += blockDim.x) {       // HG:226-235
                const double d = dx[t];
                if (t < n - 1) s.Va[t + 1] -= d;
                else s.Vm[c + (t - (n - 1))] -= d;
            }
            if (tid == 0 && a.info[slot]) { a.stat[slot] = HPF_ST_SINGULAR; a.info[slot] = 0; }
        }
        const int it = a.itc[slot];
        __syncthreads();
        const double err = cta_fund_mismatch(nf, s, rhs);
        if (a.hist_h && tid == 0) a.hist_h[(size_t)it * B + b] = err;
        const bool cont = (err > a.thresh_h) && (it < a.max_h);
        if (cont) {
            if (tid == 0) { a.flag[ai] = 1; a.itc[slot] = it + 1; }
            continue;
        }
        int status = a.stat[slot];
        if (it >= a.max_h) status = HPF_ST_MAXITER;
        if (err != err) status = HPF_ST_NONFINITE;
        for (int t = tid; t < n; t += blockDim.x) {
            a.V_m[t * B + b] = s.Vm[t];
            a.V_a[t * B + b] = s.Va[t];
        }
        if (tid == 0) {
            a.n_iter_h[b] = it;
            if (a.status) a.status[b] = status;
            a.flag[ai] = 0;
        }
    }
}

__global__ void __launch_bounds__(256)
ls_fund_jac_kernel(const DevNet nf, const LsArgs a, const int cur) {
    const int Nf = nf.N, ld = a.ldb;
    const int nact = a.nact[cur];
    const int* act = a.act + (size_t)cur * a.S;
    for (int ai = blockIdx.x; ai < nact; ai += gridDim.x) {
        const int slot = act[ai];
        const ScnSmem s = carve(a.state + (size_t)slot * a.state_stride, nf, false);
        double* A = a.M + (size_t)slot * a.mat_stride;
        __syncthreads();
        {
            double2* A2 = reinterpret_cast<double2*>(A);
            const size_t cnt2 = (size_t)ld * Nf / 2;             // (ld is a multiple of 8)
            for (size_t t = threadIdx.x; t < cnt2; t += blockDim.x) A2[t] = make_double2(0.0, 0.0);
        }
        __syncthreads();
        cta_fund_jacobian(nf, s, A, 1, ld);
        for (int t = threadIdx.x; t < Nf; t += blockDim.x) A[(size_t)Nf * ld + t] = s.rinv[t];
    }
}

// ---------------------------------------------------------------------------------------
// kernel 4 standalone (hpf_lu_solve) through the batched LU: row-major Jacobians [B, stride] into the
// column-major slots (32 x 32 tiles transposed through shared memory), right-hand side as column N
__global__ void __launch_bounds__(256)
ls_lu_load_kernel(const LsArgs a, const int N, const double* __restrict__ J, const size_t stride,
                  const double* __restrict__ f) {
    __shared__ double t[32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nt = (N + 31) / 32;
    const long long items = (long long)a.nwave * nt * nt;
    for (long long w = blockIdx.x; w < items; w += gridDim.x) {
        const int slot = (int)(w / (nt * nt));
        const int rem = (int)(w - (long long)slot * nt * nt);
        const int tr = rem / nt, tc = rem - tr * nt;
        const double* Jb = J + (size_t)(a.b0 + slot) * stride;
        double* A = a.M + (size_t)slot * a.mat_stride;
        __syncthreads();
        for (int ri = warp; ri < 32; ri += 8) {
            const int r = tr * 32 + ri, c = tc * 32 + lane;
            t[ri][lane] = (r < N && c < N) ? Jb[(size_t)r * N + c] : 0.0;
        }
        __syncthreads();
        for (int ci = warp; ci < 32; ci += 8) {
            const int r = tr * 32 + lane, c = tc * 32 + ci;
            if (r < N && c < N) A[(size_t)c * a.ldb + r] = t[lane][ci];
        }
        if (tc == 0 && tr == 0)
            for (int r = threadIdx.x; r < N; r += 256) A[(size_t)N * a.ldb + r] = f[(size_t)r * a.B + a.b0 + slot];
    }
}

__global__ void ls_lu_store_kernel(const LsArgs a, const int N, double* __restrict__ dx, int* __restrict__ info) {
    const long long tot = (long long)a.nwave * N;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < tot; t += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(t / a.nwave), slot = (int)(t - (long long)r * a.nwave);
        dx[(size_t)r * a.B + a.b0 + slot] = a.M[(size_t)slot * a.mat_stride + (size_t)N * a.ldb + r];
        if (r == 0) info[a.b0 + slot] = a.info[slot];
    }
}
