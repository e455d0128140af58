// sm_100a kernels of the harmonic power-flow solve path + their C ABI (include/hpf_b200.h).
//
//   kernel 1  ybus_kernel            Y(h) assembly                      HG:132-171
//   kernel 2  mismatch_tile_kernel   fused power/current mismatch       HG:313-390
//   kernel 3  jacobian_kernel        dense FP64 Jacobian -> HBM (TMA)   HG:401-473
//   kernel 4  lu_solve_kernel        batched smem LU + solves           HG:476-479
//   fused     solve_kernel           pf() + hpf() Newton loops          HG:244-275,511-560
//   after     stats_kernel           batch statistics (hpf_stats.cuh)
//
// HG = "Harmonic Power Flow/hcne_generalized.py" of the reference.  No reference code is
// used; the arithmetic is restated from the formulas (see hpf_device.cuh).
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <limits>
#include <memory>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "../../include/hpf_b200.h"
#include "hpf_device.cuh"
#include "hpf_lu_panel.cuh"
#include "hpf_structured.cuh"
#include "hpf_lu_blocked.cuh"
#include "hpf_ne_extract.cuh"
#include "hpf_zgemm.cuh"

#define HPF_THREADS 256
#define HPF_TILE 32          // scenarios per CTA in the tile kernels

// =======================================================================================
// kernel 1: Y(h).  One thread per (harmonic, bus row).  Sequential semantics of HG:147-170
// are kept per row: later lines overwrite earlier ones, the diagonal is minus the
// sequential row sum, bus shunt only for h != 1, pi-shunts matched with the off-by-one
// index (1-based ID compared with the 0-based row).
// Optional transformer branches (tau != nullptr), the model of the reference's
// "Fundamental Power Flow/pi_trafo_pf_test.py" (FPF:117-145): tap ratio tau and phase shift phi
// (degrees) per branch, Y[f,t] = y / (tau e^{-j phi}), Y[t,f] = y / (tau e^{+j phi}); the
// pi-shunt of a branch whose toID matches divides the accumulated diagonal by tau^2 (FPF:137-145,
// same index quirk as HG:163-168, `elif` so a from-match wins).
__device__ __forceinline__ double2 cdiv_smith(double2 a, double2 b) {      // numpy's complex division
    if (fabs(b.x) >= fabs(b.y)) {
        if (b.x == 0.0 && b.y == 0.0) return make_double2(a.x / fabs(b.x), a.y / fabs(b.y));
        const double rat = b.y / b.x, scl = 1.0 / __dadd_rn(b.x, __dmul_rn(b.y, rat));
        return make_double2(__dadd_rn(a.x, __dmul_rn(a.y, rat)) * scl, __dadd_rn(a.y, -__dmul_rn(a.x, rat)) * scl);
    }
    const double rat = b.x / b.y, scl = 1.0 / __dadd_rn(b.y, __dmul_rn(b.x, rat));
    return make_double2(__dadd_rn(__dmul_rn(a.x, rat), a.y) * scl, __dadd_rn(__dmul_rn(a.y, rat), -a.x) * scl);
}

__global__ void ybus_kernel(int n, int H, int L, const int* __restrict__ harmonics,
                            const int* __restrict__ from_id, const int* __restrict__ to_id,
                            const double* __restrict__ R, const double* __restrict__ X,
                            const double* __restrict__ G, const double* __restrict__ Bsh,
                            const double* __restrict__ X_sh, const double* __restrict__ tau,
                            const double* __restrict__ phase_deg, const int yflags, double2* __restrict__ Y) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * H) return;
    const int hi = idx / n, k = idx - hi * n;
    const double h = (double)harmonics[hi];
    double2* row = Y + ((size_t)hi * n + k) * n;
    for (int j = 0; j < n; ++j) row[j] = make_double2(0.0, 0.0);
    for (int l = 0; l < L; ++l) {
        const int f = from_id[l] - 1, t = to_id[l] - 1;
        if (f != k && t != k) continue;
        // -1 / (R + j X h): Smith's algorithm like numpy's complex division
        const double br = R[l], bi = X[l] * h;
        double2 y;
        if (fabs(br) >= fabs(bi)) {
            if (br == 0.0 && bi == 0.0) {
                y = make_double2(1.0 / fabs(br), 0.0 / fabs(bi));
            } else {
                const double rat = bi / br, scl = 1.0 / __dadd_rn(br, __dmul_rn(bi, rat));
                y = make_double2(scl, -rat * scl);
            }
        } else {
            const double rat = br / bi, scl = 1.0 / __dadd_rn(bi, __dmul_rn(br, rat));
            y = make_double2(rat * scl, -scl);
        }
        y = make_double2(-y.x, -y.y);
        if (tau) {
            // (tau * exp(-+ j phi)), phi = phase_shift / 180 * pi   (FPF:118-124)
            const double phi = phase_deg[l] / 180.0 * CUDART_PI;
            double sn, cs;
            sincos(phi, &sn, &cs);
            const double2 dft = make_double2(tau[l] * cs, tau[l] * -sn);
            const double2 dtf = make_double2(tau[l] * cs, tau[l] * sn);
            const double2 yft = cdiv_smith(y, dft), ytf = cdiv_smith(y, dtf);
            if (yflags & HPF_Y_SUM_PARALLEL) {
                if (f == k) row[t] = cadd(row[t], yft);
                if (t == k) row[f] = cadd(row[f], ytf);
            } else {
                if (f == k) row[t] = yft;
                if (t == k) row[f] = ytf;                    // (a self-loop keeps the later assignment)
            }
        } else if (yflags & HPF_Y_SUM_PARALLEL) {
            if (f == k) row[t] = cadd(row[t], y);
            if (t == k) row[f] = cadd(row[f], y);
        } else {
            if (f == k) row[t] = y;
            if (t == k) row[f] = y;
        }
    }
    double2 s = make_double2(0.0, 0.0);
    for (int j = 0; j < n; ++j) s = cadd(s, row[j]);
    double2 d = make_double2(-s.x, -s.y);
    if (X_sh[k] != 0.0 && harmonics[hi] != 1) {
        // 1 / (j X_sh h) = -j / (X_sh h)
        d.y += -1.0 / (X_sh[k] * h);
    }
    const int ko = (yflags & HPF_Y_FIX_SHUNT_INDEX) ? k + 1 : k;   // reference: 1-based ID compared with 0-based row
    for (int l = 0; l < L; ++l) {
        if (from_id[l] == ko || (!tau && to_id[l] == ko)) {
            d.x += G[l] / 2.0;
            d.y += (h * Bsh[l]) / 2.0;
        } else if (tau && to_id[l] == ko) {                  // FPF:142-145
            const double t2 = tau[l] * tau[l];
            d.x = (d.x + G[l] / 2.0) / t2;
            d.y = (d.y + (h * Bsh[l]) / 2.0) / t2;
        }
    }
    row[k] = d;
}

// =======================================================================================
// Shared-memory carve-up of one scenario (fused and per-CTA kernels).
struct ScnSmem {
    double* A;                                 // ld * (N + 1), column-major, odd ld
    double* lup;                               // work area of the panel LU (hpf_lu_panel.cuh), with the matrix only
    double *Vm, *Va, *Vre, *Vim, *Ere, *Eim;   // nH each
    double2 *I1, *Iinj, *IN;                   // n, q*H, q*H
    double *P, *Q;                             // n each
    double* rinv;                              // N
    double* red;                               // 64
    int* flag;                                 // 8 ints
};

__host__ __device__ inline int odd_ld(int N) { return N | 1; }

__host__ __device__ inline size_t scn_smem_bytes(int n, int H, int q, int N, bool with_matrix) {
    const size_t nH = (size_t)n * H;
    size_t d = 0;
    if (with_matrix) d += (size_t)odd_ld(N) * (N + 1) + lup_extra_doubles(N);
    d += 6 * nH + 2 * n + 4 * (size_t)q * H + 2 * n + N + 64 + 4;
    return d * sizeof(double) + 16;
}

__device__ __forceinline__ ScnSmem carve(double* base, const DevNet& net, bool with_matrix) {
    ScnSmem s;
    double* p = base;
    const int nH = net.nH, qH = net.q * net.H;
    s.A = p;
    s.lup = nullptr;
    if (with_matrix) {
        p += (size_t)odd_ld(net.N) * (net.N + 1);
        if ((reinterpret_cast<uintptr_t>(p) & 15) != 0) p += 1;
        s.lup = p;
        p += lup_extra_doubles(net.N);
    }
    if ((reinterpret_cast<uintptr_t>(p) & 15) != 0) p += 1;   // double2 alignment
    s.I1 = reinterpret_cast<double2*>(p);   p += 2 * net.n;
    s.Iinj = reinterpret_cast<double2*>(p); p += 2 * qH;
    s.IN = reinterpret_cast<double2*>(p);   p += 2 * qH;
    s.Vm = p;  p += nH;
    s.Va = p;  p += nH;
    s.Vre = p; p += nH;
    s.Vim = p; p += nH;
    s.Ere = p; p += nH;
    s.Eim = p; p += nH;
    s.P = p;   p += net.n;
    s.Q = p;   p += net.n;
    s.rinv = p; p += net.N;
    s.red = p; p += 64;
    s.flag = reinterpret_cast<int*>(p);
    return s;
}

// ---- per-CTA phases (VS = 1) -----------------------------------------------------------
__device__ __forceinline__ void cta_phasors(const ScnSmem& s, int lo, int hi, bool abs_norm) {
    for (int t = lo + threadIdx.x; t < hi; t += blockDim.x)
        phasor_one<1>(t, 0, s.Vm, s.Va, s.Vre, s.Vim, s.Ere, s.Eim, abs_norm);
    __syncthreads();
}

// I1 = Y1 V1 and (harmonic stage) the Norton injections.
__device__ __forceinline__ void cta_currents(const DevNet& net, const ScnSmem& s, bool with_norton) {
    const int qH = with_norton ? net.q * net.H : 0;
    for (int t = threadIdx.x; t < net.n + qH; t += blockDim.x) {
        if (t < net.n) {
            s.I1[t] = ydotv<1>(net, 0, t, 0, s.Vre, s.Vim);
        } else {
            const int u = t - net.n, k = u / net.H, h = u - k * net.H;
            s.Iinj[u] = norton_injection<1>(net, k, h, 0, s.Vre, s.Vim, s.IN[u]);
        }
    }
    __syncthreads();
}

// Harmonic mismatch into rhs[] (N doubles); returns ||f||_inf (NaN-propagating) to all threads.
__device__ __forceinline__ double cta_harmonic_mismatch(const DevNet& net, const ScnSmem& s, double* rhs) {
    cta_phasors(s, 0, net.nH, false);
    cta_currents(net, s, true);
    double mx = 0.0;
    for (int e = threadIdx.x; e < net.nH - 1; e += blockDim.x) {
        const double2 f = harmonic_mismatch_entry<1>(net, e, 0, s.Vre, s.Vim, s.I1, s.Iinj, s.P, s.Q);
        rhs[h_row_re(net, e)] = f.x;
        double a = fabs(f.x);
        if (e >= net.c - 1) {
            rhs[h_row_im(net, e)] = f.y;
            const double b = fabs(f.y);
            a = (b != b || b > a) ? b : a;
        }
        mx = (a != a || a > mx) ? a : mx;
    }
    return block_max_nan(mx, s.red);
}

// Fundamental mismatch (HG:195-202) into rhs[] (Nf doubles).
__device__ __forceinline__ double cta_fund_mismatch(const DevNet& net, const ScnSmem& s, double* rhs) {
    cta_phasors(s, 0, net.n, true);
    cta_currents(net, s, false);
    const int n = net.n, c = net.c;
    double mx = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double2 v = make_double2(s.Vre[i], s.Vim[i]);
        const double2 sl = cmul(v, cconj(s.I1[i]));
        const double fr = sl.x + s.P[i], fi = sl.y + s.Q[i];
        double a = 0.0;
        if (i >= 1) { rhs[i - 1] = fr; a = fabs(fr); }
        if (i >= c) {
            rhs[(n - 1) + i - c] = fi;
            const double b = fabs(fi);
            a = (b != b || b > a) ? b : a;
        }
        mx = (a != a || a > mx) ? a : mx;
    }
    return block_max_nan(mx, s.red);
}

// Zero `cnt` doubles at A (cnt even or odd; A 8-byte aligned).
__device__ __forceinline__ void cta_zero(double* A, size_t cnt) {
    for (size_t t = threadIdx.x; t < cnt; t += blockDim.x) A[t] = 0.0;
}

// Harmonic Jacobian into a dense matrix addressed A[row*rs + col*cs] (pre-zeroed).
__device__ __forceinline__ void cta_harmonic_jacobian(const DevNet& net, const ScnSmem& s, double* A,
                                                      size_t rs, size_t cs) {
    const int slots = net.n + (net.coupled ? net.H : 0);
    const int items = (net.nH - 1) * slots;
    auto put = [=](int row, int col, double v) { A[row * rs + col * cs] = v; };
    for (int t = threadIdx.x; t < items; t += blockDim.x) {
        const int e = t / slots, slot = t - e * slots;
        harmonic_jacobian_item(net, e, slot, s.Vre, s.Vim, s.Ere, s.Eim, s.I1, put);
    }
}

__device__ __forceinline__ void cta_fund_jacobian(const DevNet& net, const ScnSmem& s, double* A,
                                                  size_t rs, size_t cs) {
    const int n = net.n;
    auto put = [=](int row, int col, double v) { A[row * rs + col * cs] = v; };
    if (net.ell_col) {                                   // (every non-zero of Y1 and the diagonal is listed)
        for (int t = threadIdx.x; t < n * net.ell_w; t += blockDim.x) {
            const int i = t / net.ell_w, j = net.ell_col[t];
            if (j >= 0) fund_jacobian_item(net, i, j, s.Vre, s.Vim, s.Ere, s.Eim, s.I1, put);
        }
        return;
    }
    for (int t = threadIdx.x; t < n * n; t += blockDim.x) {
        const int i = t / n, j = t - i * n;
        fund_jacobian_item(net, i, j, s.Vre, s.Vim, s.Ere, s.Eim, s.I1, put);
    }
}

// =======================================================================================
// Fused solve kernel: persistent CTAs pull scenarios from a global work counter
// (iteration counts differ between scenarios, 8..34+, so static striding would idle SMs).
// mode 0: fundamental + harmonic (hpf);  mode 1: fundamental only (pf).
struct SolveArgs {
    int B, mode, flags;
    const double *P, *Q;
    const double2* I_N;
    double thresh_f, thresh_h;
    int max_f, max_h;
    double *V_m, *V_a;
    double2* I_inj;
    int *n_iter_f, *n_iter_h, *status;
    double *err_h, *err_f, *hist_f, *hist_h;
    int* work_counter;
    double* workspace;     // GMEM variant: gridDim.x * ld * (N + 1) doubles
    int lub_doubles;       // GMEM variant: shared-memory work area of the blocked LU (doubles)
    int lu_classic;        // shared-memory LU: 1 = rank-1 updates (lu_solve_smem), 0 = panel-blocked (default)
};

#define HPF_THREADS_GMEM 512
// GMEM kernels: the matrix lives in a per-CTA global workspace with leading dimension
// lub_ld(N); the blocked LU's staging buffers follow the scenario state in shared memory.
__host__ __device__ inline size_t scn_smem_doubles_aligned(int n, int H, int q, int N) {
    return (scn_smem_bytes(n, H, q, N, false) + 15) / 16 * 2;
}
__host__ __device__ inline size_t gmem_kernel_smem_bytes(int n, int H, int q, int N) {     // minimum
    return (scn_smem_doubles_aligned(n, H, q, N) + LUB_SMEM_DOUBLES) * sizeof(double) + 16;
}
// blocked-LU work area (doubles) for an N-row system next to the scenario state, within `optin`
static inline size_t gmem_kernel_lub_doubles(int n, int H, int q, int N, size_t optin) {
    const size_t state = scn_smem_doubles_aligned(n, H, q, N) * sizeof(double) + 16;
    return lub_smem_doubles_for(N, optin > state ? optin - state : 0);
}
// LU: 0 = shared-memory LU (matrix in smem), 1 = blocked LU (matrix in the global workspace or
// behind the work area), 2 = blocked LU for systems whose panels do not fit the staging buffer
template <int LU>
__global__ void __launch_bounds__(LU ? HPF_THREADS_GMEM : HPF_THREADS, LU ? 1 : 2)
solve_kernel(const DevNet net, const SolveArgs a) {
    constexpr bool GMEM = LU != 0;
    extern __shared__ __align__(16) double smem[];
    ScnSmem s = carve(smem, net, !GMEM);
    const int tid = threadIdx.x;
    const int n = net.n, c = net.c, nH = net.nH, N = net.N, Nf = net.Nf, H = net.H, q = net.q;
    const int ld = GMEM ? lub_ld(N) : odd_ld(N);
    double* lub = smem + scn_smem_doubles_aligned(n, H, q, N);      // GMEM only
    // (blocked LU: the matrix sits in the per-CTA global workspace, or - small systems, when it
    // fits - in shared memory behind the LU work area)
    if (GMEM) s.A = a.workspace ? a.workspace + (size_t)blockIdx.x * ld * (N + 1) : lub + a.lub_doubles;
    const size_t B = (size_t)a.B;

    for (;;) {
        __syncthreads();
        if (tid == 0) s.flag[1] = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int b = s.flag[1];
        if (b >= a.B) break;

        // ---- load scenario, flat start (HG:174-184) ----
        for (int t = tid; t < n; t += blockDim.x) {
            s.P[t] = a.P[t * B + b];
            s.Q[t] = a.Q[t * B + b];
        }
        if (a.mode == 0)
            for (int t = tid; t < q * H; t += blockDim.x) s.IN[t] = a.I_N[t * B + b];
        for (int t = tid; t < nH; t += blockDim.x) {
            s.Vm[t] = (t < n) ? 1.0 : 0.1;
            s.Va[t] = 0.0;
        }
        __syncthreads();

        int status = HPF_ST_CONVERGED;
        // ---- fundamental Newton-Raphson (HG:244-275) ----
        double* rhs_f = s.A + (size_t)Nf * ld;
        double err = cta_fund_mismatch(net, s, rhs_f);
        int it_f = 0;
        if (a.hist_f && tid == 0) a.hist_f[b] = err;
        while (err > a.thresh_f && it_f < a.max_f) {
            cta_zero(s.A, (size_t)ld * Nf);
            __syncthreads();
            cta_fund_jacobian(net, s, s.A, 1, ld);
            const int info = GMEM ? lu_solve_blocked_t<LU == 2>(s.A, Nf, ld, lub, a.lub_doubles, s.flag)
                                  : (a.lu_classic ? lu_solve_smem(s.A, Nf, ld, s.rinv, s.flag)
                                                  : lu_solve_smem_panel(s.A, Nf, ld, s.rinv, s.flag, s.lup));
            if (info) status = HPF_ST_SINGULAR;
            for (int t = tid; t < Nf; t += blockDim.x) {       // HG:226-235
                const double dx = rhs_f[t];
                if (t < n - 1) s.Va[t + 1] -= dx;
                else s.Vm[c + (t - (n - 1))] -= dx;
            }
            __syncthreads();
            err = cta_fund_mismatch(net, s, rhs_f);
            ++it_f;
            if (a.hist_f && tid == 0) a.hist_f[(size_t)it_f * B + b] = err;
        }
        if (a.hist_f)
            for (int t = it_f + 1 + tid; t <= a.max_f; t += blockDim.x) a.hist_f[(size_t)t * B + b] = CUDART_NAN;
        if (it_f >= a.max_f) status = HPF_ST_MAXITER;
        if (err != err) status = HPF_ST_NONFINITE;
        if (tid == 0) {
            a.n_iter_f[b] = it_f;
            if (a.err_f) a.err_f[b] = err;
        }

        if (a.mode == 1) {
            for (int t = tid; t < nH; t += blockDim.x) {
                a.V_m[t * B + b] = s.Vm[t];
                a.V_a[t * B + b] = s.Va[t];
            }
            if (tid == 0 && a.status) a.status[b] = status;
            continue;
        }

        // ---- harmonic Newton-Raphson (HG:531-542) ----
        double* rhs = s.A + (size_t)N * ld;
        double err_h = cta_harmonic_mismatch(net, s, rhs);
        int it_h = 0;
        if (a.hist_h && tid == 0) a.hist_h[b] = err_h;
        while (err_h > a.thresh_h && it_h < a.max_h) {
            cta_zero(s.A, (size_t)ld * N);
            __syncthreads();
            cta_harmonic_jacobian(net, s, s.A, 1, ld);
            const int info = GMEM ? lu_solve_blocked_t<LU == 2>(s.A, N, ld, lub, a.lub_doubles, s.flag)
                                  : (a.lu_classic ? lu_solve_smem(s.A, N, ld, s.rinv, s.flag)
                                                  : lu_solve_smem_panel(s.A, N, ld, s.rinv, s.flag, s.lup));
            if (info && status == HPF_ST_CONVERGED) status = HPF_ST_SINGULAR;
            for (int t = tid; t < N; t += blockDim.x) {        // HG:476-485
                const double dx = rhs[t];
                if (t < nH - 1) s.Va[t + 1] -= dx;
                else s.Vm[c + (t - (nH - 1))] -= dx;
            }
            __syncthreads();
            err_h = cta_harmonic_mismatch(net, s, rhs);
            ++it_h;
            if (a.hist_h && tid == 0) a.hist_h[(size_t)it_h * B + b] = err_h;
        }
        if (a.hist_h)
            for (int t = it_h + 1 + tid; t <= a.max_h; t += blockDim.x) a.hist_h[(size_t)t * B + b] = CUDART_NAN;
        if (it_h >= a.max_h && status == HPF_ST_CONVERGED) status = HPF_ST_MAXITER;
        if (err_h != err_h) status = HPF_ST_NONFINITE;

        // ---- post-processing (HG:547-549) and result write-out ----
        for (int t = tid; t < nH; t += blockDim.x) {
            double vm = s.Vm[t], va = s.Va[t], r = va;
            if (!(a.flags & HPF_SOLVE_RAW)) {
                if (vm < 0.0) va += CUDART_PI;
                const double twopi = 2.0 * CUDART_PI;
                r = fmod(va, twopi);                 // numpy's % : result takes the divisor's sign
                if (r != 0.0) { if (r < 0.0) r += twopi; } else r = 0.0;
                if (vm < 0.0) vm = -vm;
            }
            if (!(vm == vm) || !(r == r) || fabs(vm) == CUDART_INF) status = HPF_ST_NONFINITE;
            a.V_m[t * B + b] = vm;
            a.V_a[t * B + b] = r;
        }
        if (a.I_inj)
            for (int t = tid; t < q * H; t += blockDim.x) a.I_inj[t * B + b] = s.Iinj[t];
        // status may differ between threads only through the non-finite check above
        const int st_any = __syncthreads_or(status == HPF_ST_NONFINITE);
        if (tid == 0) {
            a.n_iter_h[b] = it_h;
            a.err_h[b] = err_h;
            a.status[b] = st_any ? HPF_ST_NONFINITE : status;
        }
    }
}

// =======================================================================================
// kernel 2 (standalone): 32 scenarios per CTA, lane = scenario, warps stride over rows.
// HBM traffic is batch-innermost and fully coalesced: every global access of a warp is one
// contiguous 256-byte (double) or 512-byte (double2) segment.
struct MismatchArgs {
    int B;
    const double *V_m, *V_a, *P, *Q;
    const double2* I_N;
    double *f, *err;
    double2* I_inj;
};

__host__ __device__ inline size_t tile_smem_bytes(int n, int H, int q, int m, int yn_elems) {
    const size_t nH = (size_t)n * H;
    // constants Y, Y_N (c128); I_N [qH][32] c128; V (re, im) [nH][32]; P, Q [m][32]; red [8][32]
    return (2 * ((size_t)H * n * n + yn_elems) + (2 * (size_t)q * H + 2 * nH + 2 * m + 8) * HPF_TILE) *
               sizeof(double) + 16;
}

__device__ __forceinline__ void cp_async8(void* sdst, const void* gsrc) {
    const uint32_t sa = (uint32_t)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async16(void* sdst, const void* gsrc) {
    const uint32_t sa = (uint32_t)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
}

// The whole input tile (V_m, V_a, P, Q, I_N of 32 scenarios) is requested with asynchronous
// copies (LDGSTS) before anything is computed, so every byte of the tile is in flight at once.
// ncu shows the kernel is bound by INSTRUCTION ISSUE, not by HBM (52 FP64 sincos + ~400
// complex MACs per 1.9 KB of traffic), so the instruction count is what matters: network
// constants live in shared memory and the shape-specialised instances (class D, see
// hpf_structured.cuh) fold all index arithmetic into immediates.
template <class D>
__global__ void __launch_bounds__(HPF_THREADS, 4)
mismatch_tile_kernel(const DevNet net, const MismatchArgs a, const int yn_elems) {
    extern __shared__ __align__(16) double smem[];
    constexpr int NW = HPF_THREADS / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = D::n ? D::n : net.n, m = D::n ? D::m : net.m, c = D::n ? D::c : net.c;
    const int H = D::n ? D::H : net.H, q = D::n ? D::q : net.q, nH = n * H;
    constexpr int SR = D::n ? (D::n * D::H + NW - 1) / NW : 0;
    constexpr int HR = D::n ? (D::q * D::H + NW - 1) / NW : 0;
    constexpr int LR = D::n ? (D::m * D::H + NW - 1) / NW : 0;
    const size_t B = (size_t)a.B;
    double2* sY = reinterpret_cast<double2*>(smem);
    double2* sYN = sY + (size_t)H * n * n;
    double2* IN = sYN + yn_elems;
    double* Vre = reinterpret_cast<double*>(IN + (size_t)q * H * HPF_TILE);   // raw V_m, then Re V
    double* Vim = Vre + (size_t)nH * HPF_TILE;                                  // raw V_a, then Im V
    double* Pl = Vim + (size_t)nH * HPF_TILE;
    double* Ql = Pl + (size_t)m * HPF_TILE;
    double* red = Ql + (size_t)m * HPF_TILE;
    for (int t = threadIdx.x; t < H * n * n; t += HPF_THREADS) sY[t] = net.Y[t];
    for (int t = threadIdx.x; t < yn_elems; t += HPF_THREADS) sYN[t] = net.YN[t];
#define TA(X, i) X[(i) * HPF_TILE + lane]

    for (size_t tile = blockIdx.x; tile * HPF_TILE < B; tile += gridDim.x) {
        const size_t b = tile * HPF_TILE + lane;
        const bool ok = b < B;
        const size_t bb = ok ? b : B - 1;            // clamp: compute, do not store
        __syncthreads();
        // phase L: request the tile
        for (int t = warp; t < nH; t += NW) {
            cp_async8(&TA(Vre, t), a.V_m + t * B + bb);
            cp_async8(&TA(Vim, t), a.V_a + t * B + bb);
        }
        for (int t = 1 + warp; t < m; t += NW) {
            cp_async8(&TA(Pl, t), a.P + t * B + bb);
            cp_async8(&TA(Ql, t), a.Q + t * B + bb);
        }
        for (int u = warp; u < q * H; u += NW) cp_async16(&TA(IN, u), a.I_N + u * B + bb);
        cp_async_wait_all();
        __syncthreads();
        // phase A: phasors in place, V = V_m e^{j theta}
        row_loop<SR>(warp, nH, NW, [&](int t) {
            const double vm = TA(Vre, t);
            double sn, cs;
            sincos(TA(Vim, t), &sn, &cs);
            TA(Vre, t) = vm * cs;
            TA(Vim, t) = vm * sn;
        });
        __syncthreads();
        // phase B: rows of the mismatch (HG:360-388)
        double mx = 0.0;
        auto emit = [&](int s, double2 f) {          // s = stacked index of the row, entry e = s - 1
            const int e = s - 1;
            double v1 = fabs(f.x);
            if (ok) __stcs(a.f + (size_t)e * B + b, f.x);
            if (e >= c - 1) {
                if (ok) __stcs(a.f + (size_t)((nH - 1) + e - (c - 1)) * B + b, f.y);
                const double v2 = fabs(f.y);
                v1 = (v2 != v2 || v2 > v1) ? v2 : v1;
            }
            mx = (v1 != v1 || v1 > mx) ? v1 : mx;
        };
        // nonlinear buses: (Y_h V_h)_i + I_N - sum_p Y_N[h][p] V_p,i   (HG:313-323,335-354)
        row_loop<HR>(warp, q * H, NW, [&](int u) {
            const int k = u / H, h = u - k * H, i = m + k, s = h * n + i;
            const int dev = net.dev_of_nl[k];
            double2 acc;
            if (net.coupled) {
                const double2* row = sYN + ((size_t)dev * H + h) * H;
                acc = make_double2(0.0, 0.0);
                for (int pp = 0; pp < H; ++pp) {
                    const int t2 = pp * n + i;
                    acc = cfma(acc, row[pp], make_double2(TA(Vre, t2), TA(Vim, t2)));
                }
            } else {
                acc = cmul(sYN[(size_t)dev * H + h], make_double2(TA(Vre, s), TA(Vim, s)));
            }
            const double2 inj = csub(TA(IN, u), acc);
            if (a.I_inj && ok) a.I_inj[u * B + b] = inj;
            const double2* Yrow = sY + ((size_t)h * n + i) * n;
            double2 f = make_double2(0.0, 0.0);
            for (int j = 0; j < n; ++j) {
                const int t2 = h * n + j;
                f = cfma(f, Yrow[j], make_double2(TA(Vre, t2), TA(Vim, t2)));
            }
            emit(s, cadd(f, inj));
        });
        // linear buses: current balance at h >= 1 (index), power balance at the fundamental
        row_loop<LR>(warp, m * H, NW, [&](int t) {
            const int h = t / m, i = t - h * m, s = h * n + i;
            if (s == 0) return;                                  // slack: no row
            const double2* Yrow = sY + ((size_t)h * n + i) * n;
            double2 f = make_double2(0.0, 0.0);
            for (int j = 0; j < n; ++j) {
                const int t2 = h * n + j;
                f = cfma(f, Yrow[j], make_double2(TA(Vre, t2), TA(Vim, t2)));
            }
            if (h == 0) {                                        // dS = (P + jQ) + V conj(Y1 V)  (HG:372-380)
                const double2 v = make_double2(TA(Vre, i), TA(Vim, i));
                const double2 sl = cmul(v, cconj(f));
                f = make_double2(TA(Pl, i) + sl.x, TA(Ql, i) + sl.y);
            }
            emit(s, f);
        });
        TA(red, warp) = mx;
        __syncthreads();
        if (warp == 0) {
            double r = 0.0;
            bool bad = false;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                const double v = TA(red, w);
                bad |= (v != v);
                r = fmax(r, v);
            }
            if (ok) a.err[b] = bad ? CUDART_NAN : r;
        }
    }
#undef TA
}

#include "hpf_lane.cuh"
#include "hpf_harmonic_warp.cuh"

// Fallback for networks whose 32-scenario tile does not fit in shared memory (e.g. net1 with
// 26 harmonics): one scenario per CTA, same arithmetic (VS = 1), strided HBM access.
__global__ void __launch_bounds__(HPF_THREADS)
mismatch_cta_kernel(const DevNet net, const MismatchArgs a) {
    extern __shared__ __align__(16) double smem[];
    const ScnSmem s = carve(smem, net, false);
    double* rhs = s.rinv;                        // N doubles, unused otherwise in this kernel
    const int nH = net.nH, qH = net.q * net.H;
    const size_t B = (size_t)a.B;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        __syncthreads();
        for (int t = threadIdx.x; t < nH; t += blockDim.x) {
            s.Vm[t] = a.V_m[t * B + b];
            s.Va[t] = a.V_a[t * B + b];
        }
        for (int t = threadIdx.x; t < net.n; t += blockDim.x) {
            s.P[t] = a.P[t * B + b];
            s.Q[t] = a.Q[t * B + b];
        }
        for (int t = threadIdx.x; t < qH; t += blockDim.x) s.IN[t] = a.I_N[t * B + b];
        __syncthreads();
        const double err = cta_harmonic_mismatch(net, s, rhs);
        for (int t = threadIdx.x; t < net.N; t += blockDim.x) a.f[t * B + b] = rhs[t];
        if (a.I_inj)
            for (int t = threadIdx.x; t < qH; t += blockDim.x) a.I_inj[t * B + b] = s.Iinj[t];
        if (threadIdx.x == 0) a.err[b] = err;
    }
}

// =======================================================================================
// kernel 3 (standalone): one scenario per CTA iteration; the N x N matrix is assembled
// row-major in shared memory and leaves the SM as ONE bulk asynchronous copy
// (cp.async.bulk shared -> global, the TMA engine), so the store stream is full 128-byte
// lines without occupying LSU issue slots.
__device__ __forceinline__ void bulk_store_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    const uint32_t sa = (uint32_t)__cvta_generic_to_shared(ssrc);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n"
                 :: "l"(gdst), "r"(sa), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
}
__device__ __forceinline__ void bulk_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}

struct JacobianArgs {
    int B;
    const double *V_m, *V_a;
    double* J;
    long long stride;     // doubles between scenarios (even, >= N*N)
};

__host__ __device__ inline size_t jac_smem_bytes(int n, int H, int q, int N, long long stride) {
    return (size_t)stride * sizeof(double) + scn_smem_bytes(n, H, q, N, false) + 16;
}

#define HPF_JAC_THREADS 512
__global__ void __launch_bounds__(HPF_JAC_THREADS)
jacobian_kernel(const DevNet net, const JacobianArgs a) {
    extern __shared__ __align__(16) double smem[];
    double* Jt = smem;                                   // stride doubles, 16-byte aligned
    const ScnSmem s = carve(smem + a.stride, net, false);
    const int nH = net.nH, N = net.N;
    const size_t B = (size_t)a.B;
    // The sparsity pattern of J is fixed by the network (positions where Y(h) or Y_N are
    // zero never change), so the tile is zero-filled ONCE; every scenario overwrites the
    // same non-zero positions.
    cta_zero(Jt, (size_t)a.stride);
    // software pipeline: the state of the NEXT scenario is fetched into registers while the
    // current matrix is assembled (nH <= 2 * blockDim.x entries per thread pair)
    double pvm = 0.0, pva = 0.0;
    const bool own = (int)threadIdx.x < nH;
    if (own && (int)blockIdx.x < a.B) {
        pvm = __ldcs(a.V_m + threadIdx.x * B + blockIdx.x);
        pva = __ldcs(a.V_a + threadIdx.x * B + blockIdx.x);
    }
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        if (own) { s.Vm[threadIdx.x] = pvm; s.Va[threadIdx.x] = pva; }
        for (int t = threadIdx.x + blockDim.x; t < nH; t += blockDim.x) {   // (large networks)
            s.Vm[t] = __ldcs(a.V_m + t * B + b);
            s.Va[t] = __ldcs(a.V_a + t * B + b);
        }
        const int bn = b + gridDim.x;
        if (own && bn < a.B) {
            pvm = __ldcs(a.V_m + threadIdx.x * B + bn);
            pva = __ldcs(a.V_a + threadIdx.x * B + bn);
        }
        __syncthreads();
        cta_phasors(s, 0, nH, false);                    // (contains a barrier)
        cta_currents(net, s, false);                     // overlaps the previous bulk store
        if (threadIdx.x == 0) bulk_store_wait_read();   // previous matrix has left smem
        __syncthreads();
        cta_harmonic_jacobian(net, s, Jt, (size_t)N, 1);
        fence_proxy_async_smem();                        // generic-proxy writes -> async proxy
        __syncthreads();
        if (threadIdx.x == 0)
            bulk_store_s2g(a.J + (size_t)b * a.stride, Jt, (uint32_t)(a.stride * sizeof(double)));
    }
    if (threadIdx.x == 0) bulk_store_wait_read();
}

// Fallback when the N x N matrix does not fit in shared memory: zero-fill and scatter
// straight into global memory (the CTA's own L2-resident lines).
__global__ void __launch_bounds__(HPF_THREADS)
jacobian_gmem_kernel(const DevNet net, const JacobianArgs a) {
    extern __shared__ __align__(16) double smem[];
    const ScnSmem s = carve(smem, net, false);
    const int nH = net.nH, N = net.N;
    const size_t B = (size_t)a.B;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        __syncthreads();
        for (int t = threadIdx.x; t < nH; t += blockDim.x) {
            s.Vm[t] = a.V_m[t * B + b];
            s.Va[t] = a.V_a[t * B + b];
        }
        double* Jb = a.J + (size_t)b * a.stride;
        cta_zero(Jb, (size_t)a.stride);
        __syncthreads();
        cta_phasors(s, 0, nH, false);
        cta_currents(net, s, false);
        cta_harmonic_jacobian(net, s, Jb, (size_t)N, 1);
    }
}

// =======================================================================================
// kernel 4 (standalone): J [B, stride] row-major from HBM -> padded column-major smem,
// LU + solves, dx [N, B].
struct LuArgs {
    int B;
    const double *J, *f;
    double* dx;
    int* info;
    long long stride;
    double* workspace;
    int lub_doubles;
    int lu_classic;
};

template <int LU>
__global__ void __launch_bounds__(LU ? HPF_THREADS_GMEM : HPF_THREADS, LU ? 1 : 2)
lu_solve_kernel(const DevNet net, const LuArgs a) {
    constexpr bool GMEM = LU != 0;
    extern __shared__ __align__(16) double smem[];
    ScnSmem s = carve(smem, net, !GMEM);
    const int N = net.N, ld = GMEM ? lub_ld(N) : odd_ld(N);
    double* lub = smem + scn_smem_doubles_aligned(net.n, net.H, net.q, N);   // GMEM only
    if (GMEM) s.A = a.workspace ? a.workspace + (size_t)blockIdx.x * ld * (N + 1) : lub + a.lub_doubles;
    const size_t B = (size_t)a.B;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        __syncthreads();
        const double* Jb = a.J + (size_t)b * a.stride;
        for (int t = threadIdx.x; t < N * N; t += blockDim.x) {
            const int r = t / N, cidx = t - r * N;
            s.A[r + (size_t)cidx * ld] = Jb[t];
        }
        double* rhs = s.A + (size_t)N * ld;
        for (int t = threadIdx.x; t < N; t += blockDim.x) rhs[t] = a.f[t * B + b];
        const int info = GMEM ? lu_solve_blocked_t<LU == 2>(s.A, N, ld, lub, a.lub_doubles, s.flag)
                              : (a.lu_classic ? lu_solve_smem(s.A, N, ld, s.rinv, s.flag)
                                              : lu_solve_smem_panel(s.A, N, ld, s.rinv, s.flag, s.lup));
        for (int t = threadIdx.x; t < N; t += blockDim.x) a.dx[t * B + b] = rhs[t];
        if (threadIdx.x == 0) a.info[b] = info;
    }
}

// =======================================================================================
// Structured Newton step for networks whose 32-scenario tile does not fit in shared memory
// (e.g. net1: 20 buses x 26 harmonics): one scenario per CTA, threads over the rows, same
// closed-form step as harm_tile_kernel (hpf_structured.cuh); Y(h), G and W_NL stay in
// global memory (L2), the border system is solved by the block LU (lu_solve_smem).
// For the 200- / 1000-bus configurations not even one scenario fits: the state then lives in a
// per-CTA global-memory slab (gstate; L2 resident or streamed) and the border system
// (2m-1-c up to 1199 unknowns) goes through the blocked tensor-core LU; shared memory keeps
// only the reduction scratch and the LU staging buffers.
__host__ __device__ inline size_t harm_cta_state_doubles(int n, int H, int m, int c, int q, int N, bool gmem) {
    const size_t nH = (size_t)n * H, nZ = nH - m, nx = (size_t)(m - 1) + (m - c);
    const size_t ldb = gmem ? (size_t)lub_ld((int)nx) : (size_t)odd_ld((int)nx);
    return (scn_smem_bytes(n, H, q, N, false) + 15) / 16 * 2 + 2 * nZ + 2 * q + 2 * m + ldb * (nx + 1) + nx + 16;
}
__host__ __device__ inline size_t harm_cta_smem_bytes(int n, int H, int m, int c, int q, int N) {
    return harm_cta_state_doubles(n, H, m, c, q, N, false) * sizeof(double);
}
static inline size_t harm_cta_gmem_lub_doubles(int nx, size_t optin) {
    return lub_smem_doubles_for(nx, optin - 80 * sizeof(double));
}

template <int THREADS, bool BIGLU>
__global__ void __launch_bounds__(THREADS)
harm_cta_kernel(const DevNet net, const StructNet sn, const HarmTileArgs a) {
    extern __shared__ __align__(16) double smem[];
    const bool gst = a.gstate != nullptr;
    double* base = gst ? a.gstate + (size_t)blockIdx.x * a.gstate_stride : smem;
    ScnSmem s = carve(base, net, false);
    double* lub = smem + 80;                                  // gstate only: LU staging
    if (gst) {                                                // barriers / reductions need real smem
        s.red = smem;
        s.flag = reinterpret_cast<int*>(smem + 66);
    }
    const int tid = threadIdx.x;
    const int n = net.n, m = net.m, c = net.c, H = net.H, q = net.q, nH = net.nH, N = net.N;
    const int nZ = sn.nZ, nx = sn.nx, nth = m - 1, ldb = gst ? lub_ld(nx) : odd_ld(nx);
    const size_t B = (size_t)a.B;
    double* rhs = s.rinv;                                     // f, N doubles
    double* wbase = base + (scn_smem_bytes(n, H, q, N, false) + 15) / 16 * 2;
    double2* W = reinterpret_cast<double2*>(wbase);
    double2* U0 = W + nZ;
    double2* UF = U0 + q;
    double* Mb = reinterpret_cast<double*>(UF + m);           // ldb x (nx + 1), column-major
    if ((reinterpret_cast<uintptr_t>(Mb) & 63) != 0) Mb += (64 - (reinterpret_cast<uintptr_t>(Mb) & 63)) / 8;
    double* brinv = Mb + (size_t)ldb * (nx + 1);

    int step_b = (int)blockIdx.x;                             // step mode: static striding
    for (;;) {
        __syncthreads();
        if (tid == 0) s.flag[1] = a.step_only ? step_b : atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int b = s.flag[1];
        if (b >= a.B) break;
        step_b += (int)gridDim.x;
        for (int t = tid; t < n; t += blockDim.x) {
            s.P[t] = a.P[t * B + b];
            s.Q[t] = a.Q[t * B + b];
        }
        for (int t = tid; t < q * H; t += blockDim.x) s.IN[t] = a.I_N[t * B + b];
        for (int t = tid; t < nZ; t += blockDim.x) W[t] = a.wN[t * B + b];
        for (int t = tid; t < nH; t += blockDim.x) {
            if (a.step_only || t < n) {
                s.Vm[t] = a.V_m[t * B + b];
                s.Va[t] = a.V_a[t * B + b];
            } else {
                s.Vm[t] = 0.1;                                 // flat start of the harmonics (HG:183)
                s.Va[t] = 0.0;
            }
        }
        __syncthreads();
        int status = a.step_only ? 0 : a.status[b];
        int it = 0;
        double err;
        for (;;) {
            err = cta_harmonic_mismatch(net, s, rhs);          // phasors, I1, Iinj, f
            if (a.hist_h && !a.step_only && tid == 0) a.hist_h[(size_t)it * B + b] = err;
            if (!a.step_only && !((err > a.thresh_h) && (it < a.max_h))) break;
            // u0 of the fundamental nonlinear rows (closed form)
            for (int k = tid; k < q; k += blockDim.x) {
                const int sk = m + k;
                double2 acc = make_double2(s.Vre[sk] + W[k].x, s.Vim[sk] + W[k].y);
#pragma unroll 8
                for (int i = 0; i < m; ++i)
                    acc = cfma(acc, ldg2(sn.GT + (size_t)i * nZ + k), make_double2(s.Vre[i], s.Vim[i]));
                U0[k] = cneg(acc);
            }
            __syncthreads();
            // border system: one thread per (power row i, column), entries accumulated in registers
            for (int t = tid; t < nth * (nx + 1); t += blockDim.x) {
                const int i = 1 + t / (nx + 1), col = t - (i - 1) * (nx + 1);
                const double2 vi = make_double2(s.Vre[i], s.Vim[i]);
                const double2 ei = make_double2(s.Ere[i], s.Eim[i]);
                const double2 i1 = s.I1[i];
                const double2 jvi = cmulj(vi);
                const bool is_rhs = (col == nx), is_v = (col >= nth);
                const int j = is_rhs ? 0 : (is_v ? c + (col - nth) : col + 1);
                double2 e, vj = make_double2(0.0, 0.0), ej = vj;
                if (is_rhs) {
                    // f_S of bus i sits in rhs[]: Re at row i-1, Im at row (nH-1) + (i-1) - (c-1)
                    e = make_double2(-rhs[i - 1], (i >= c) ? -rhs[(nH - 1) + (i - 1) - (c - 1)] : 0.0);
                } else {
                    const double2 y = ldg2(net.Y + (size_t)i * n + j);
                    vj = make_double2(s.Vre[j], s.Vim[j]);
                    ej = make_double2(s.Ere[j], s.Eim[j]);
                    if (is_v) {
                        e = cmul(vi, cconj(cmul(y, ej)));
                        if (i == j) e = cadd(cmul(ei, cconj(i1)), e);
                    } else {
                        const double2 yv = cmul(y, vj);
                        e = cmul(jvi, cconj((i == j) ? csub(i1, yv) : cneg(yv)));
                    }
                }
                for (int en = sn.nbr_ptr[i]; en < sn.nbr_ptr[i + 1]; ++en) {   // nonlinear neighbours of bus i
                    const int k = sn.nbr_idx[en], bk = m + k;
                    const double2 y = ldg2(net.Y + (size_t)i * n + bk);
                    const double2 vb = make_double2(s.Vre[bk], s.Vim[bk]);
                    const double2 eb = make_double2(s.Ere[bk], s.Eim[bk]);
                    const double2 ak = cmul(jvi, cconj(cneg(cmul(y, vb))));
                    const double2 vk = cmul(vi, cconj(cmul(y, eb)));
                    const double2 uu = is_rhs ? U0[k] : cmul(ldg2(sn.G + (size_t)k * m + j), is_v ? ej : cmulj(vj));
                    const double2 ce = cmul(cconj(eb), uu);
                    const double dth = ce.y / s.Vm[bk], dvm = ce.x;
                    e.x -= ak.x * dth + vk.x * dvm;
                    e.y -= ak.y * dth + vk.y * dvm;
                }
                Mb[(i - 1) + (size_t)col * ldb] = e.x;
                if (i >= c) Mb[(nth + i - c) + (size_t)col * ldb] = e.y;
            }
            int info = 0;
            if (nx > 0) {                                                   // (both start with a barrier)
                if (gst) { __syncthreads(); info = lu_solve_blocked_t<BIGLU>(Mb, nx, ldb, lub, a.lub_doubles, s.flag); }
                else info = lu_solve_smem(Mb, nx, ldb, brinv, s.flag);
            } else {
                __syncthreads();
            }
            if (info && status == HPF_ST_CONVERGED) status = HPF_ST_SINGULAR;
            const double* xF = Mb + (size_t)nx * ldb;
            // V_F + u_F (the LU staging area is free again: keep it in shared memory)
            double2* UFs = gst ? reinterpret_cast<double2*>(lub) : UF;
            for (int i = tid; i < m; i += blockDim.x) {
                const double dth = (i >= 1) ? xF[i - 1] : 0.0;
                const double dvm = (i >= c) ? xF[nth + i - c] : 0.0;
                const double2 vi = make_double2(s.Vre[i], s.Vim[i]);
                const double2 uf = make_double2(-vi.y * dth + s.Ere[i] * dvm, vi.x * dth + s.Eim[i] * dvm);
                UFs[i] = make_double2(vi.x + uf.x, vi.y + uf.y);
            }
            __syncthreads();
            // u_Z = -V_Z - G (V_F + u_F) - w_N, polar conversion, update (Vre/Vim/E are this
            // round's phasors and are not touched here, so rows can be updated in any order)
            for (int z = tid; z < nZ; z += blockDim.x) {
                const int sz = z + m;
                double2 acc = make_double2(s.Vre[sz] + W[z].x, s.Vim[sz] + W[z].y);
                const double2* gcol = sn.GT + z;
#pragma unroll 8
                for (int i = 0; i < m; ++i) acc = cfma(acc, ldg2(gcol + (size_t)i * nZ), UFs[i]);
                const double2 wv = cmul(make_double2(s.Ere[sz], -s.Eim[sz]), cneg(acc));
                const double vm = s.Vm[sz];
                const double dth = wv.y / vm, dvm = wv.x;
                if (a.step_only) {
                    a.dx_out[(size_t)(sz - 1) * B + b] = -dth;
                    a.dx_out[(size_t)((nH - 1) + sz - c) * B + b] = -dvm;
                } else {
                    s.Va[sz] += dth;
                    s.Vm[sz] = vm + dvm;
                }
            }
            for (int i = 1 + tid; i < m; i += blockDim.x) {
                const double dth = xF[i - 1];
                const double dvm = (i >= c) ? xF[nth + i - c] : 0.0;
                if (a.step_only) {
                    a.dx_out[(size_t)(i - 1) * B + b] = -dth;
                    if (i >= c) a.dx_out[(size_t)((nH - 1) + i - c) * B + b] = -dvm;
                } else {
                    s.Va[i] += dth;
                    if (i >= c) s.Vm[i] += dvm;
                }
            }
            __syncthreads();
            if (a.step_only) break;
            ++it;
        }
        if (a.step_only) continue;
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
        }
    }
    (void)N;
}

#include "hpf_lockstep.cuh"

// flat start of the harmonic rows (HG:183): |V| = 0.1, angle 0
__global__ void flat_start_fill_kernel(double* __restrict__ Vm, double* __restrict__ Va, size_t cnt) {
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < cnt; t += (size_t)gridDim.x * blockDim.x) {
        Vm[t] = 0.1;
        Va[t] = 0.0;
    }
}

// =======================================================================================
// THD (HG:563-572): one thread per (bus, scenario); sums run sequentially over the
// harmonics like Python's sum(); coalesced across the batch.
__global__ void thd_kernel(int n, int H, const int* __restrict__ harmonics, int B,
                           const double* __restrict__ V_m, double* __restrict__ thd) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nB = (size_t)n * B;
    if (idx >= nB) return;
    double sh = 0.0, sa = 0.0;
    for (int h = 0; h < H; ++h) {
        const double v = V_m[(size_t)h * nB + idx];
        const double v2 = v * v;
        if (harmonics[h] >= 3) sh = sh + v2;
        sa = sa + v2;
    }
    const double r = sqrt(sh);
    thd[idx] = r / V_m[idx];
    thd[nB + idx] = r / sqrt(sa);
}

// =======================================================================================
// Per-bus current spectra I = Y(h) V (post-processing next to get_THD; the quantity the
// reference logs in the I_log.json layout): one thread per (harmonic, bus, scenario), coalesced
// over the batch, through the sparsity pattern of Y(h) when the handle has one.
__global__ void bus_currents_kernel(const DevNet net, int B, const double* __restrict__ V_m,
                                    const double* __restrict__ V_a, double2* __restrict__ I_bus) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)net.nH * B;
    if (idx >= total) return;
    const int s = (int)(idx / B), h = s / net.n, i = s - h * net.n;
    const size_t b = idx - (size_t)s * B;
    const double2* Yrow = net.Y + ((size_t)h * net.n + i) * net.n;
    double2 acc = make_double2(0.0, 0.0);
    auto term = [&](int j) {
        const double2 y = ldg2(Yrow + j);
        if (y.x == 0.0 && y.y == 0.0) return;
        const size_t t = (size_t)(h * net.n + j) * B + b;
        double sn, cs;
        sincos(V_a[t], &sn, &cs);
        const double vm = V_m[t];
        acc = cfma(acc, y, make_double2(vm * cs, vm * sn));
    };
    if (net.ell_col) {
        const int* cols = net.ell_col + (size_t)i * net.ell_w;
        for (int e = 0; e < net.ell_w; ++e) {
            const int j = cols[e];
            if (j < 0) break;
            term(j);
        }
    } else {
        for (int j = 0; j < net.n; ++j) term(j);
    }
    I_bus[idx] = acc;
}

#include "hpf_stats.cuh"

// =======================================================================================
// Host side: handle + C ABI
#define HPF_HOST_MAX_CHUNKS 16          // chunks of one hpf_solve_host call (work-counter slots, event pairs)
#define HPF_HOST_RAMP 4096, 8192, 12288, 16384   // default chunk plan (sizes in scenarios; the last one repeats)
#define HPF_HOST_RAMP_MIN_B 8192        // smaller batches go in one chunk
#define HPF_HOST_STREAMS_DEFAULT 2
#define HPF_LS_AUTO_MIN_B 128           // large networks: batches of at least this many scenarios take the lock-step path
#define HPF_LS_MAX_ORDER 2048           // largest system of the lock-step LU (panel kernel: at most 4 rows per thread of 512)
#define HPF_HW_SERVICE_EPOCH 3          // service interval of finished lanes in the one-warp-per-harmonic kernel (profiles/r2_small_batch_ab.txt)

// Owners of CUDA resources: device memory, streams and events are released when they are reset or
// replaced, and when the handle is deleted.  AsyncPtr frees in stream order, on the stream it holds.
struct CudaFree { void operator()(void* p) const { cudaFree(p); } };
struct AsyncFree { cudaStream_t st = nullptr; void operator()(void* p) const { cudaFreeAsync(p, st); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
template <class T> using DevPtr = std::unique_ptr<T, CudaFree>;
template <class T> using AsyncPtr = std::unique_ptr<T, AsyncFree>;
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;

// A grow-only scratch buffer and its size in bytes (see grow)
template <class T>
struct Scratch {
    DevPtr<T> p;
    size_t bytes = 0;
    T* get() const { return p.get(); }
};

// Operators of the structured strategy (ensure_struct): built, and dropped, together
struct StructBufs {
    DevPtr<double2> Ainv, Gz, GzT, WNL;
    DevPtr<int> nbr_ptr, nbr_idx;
};

struct hpf_handle {
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0;
    int n = 0, m = 0, c = 0, H = 0, q = 0, L = 0, n_dev = 0, coupled = 0;
    bool have_net = false, have_dev = false, have_Y = false;
    DevPtr<int> d_harm, d_from, d_to, d_devof;
    DevPtr<double> d_R, d_X, d_G, d_B, d_Xsh;
    DevPtr<double> d_tau, d_phase;                           // optional transformer data (hpf_set_transformers)
    int y_flags = 0;                                         // HPF_Y_* (hpf_set_y_options)
    DevPtr<double2> d_Y, d_YN;
    DevPtr<int> d_counter;
    Scratch<double> d_work;
    Scratch<double> d_io;         // staging buffers of hpf_solve_host
    Stream st_io[6];              // copy-in, compute, copy-out, compute 2..4
    Event ev_io[3 * HPF_HOST_MAX_CHUNKS];   // per chunk: inputs copied, solved, V_m kept (hpf_solve_host_stats)
    Scratch<double> d_stats;      // hpf_batch_stats: THD rows; hpf_solve_host_stats: whole-batch V_m, THD rows, limits, results
    // structured strategy: 0 = not set up yet, 1 = ready, -1 = not available for this network
    int struct_state = 0;
    StructBufs d_struct;
    Scratch<double2> d_wN;
    DevPtr<int> d_ell_col;        // sparsity pattern of Y(h) for the larger networks (see DevNet)
    int ell_w = 0;
    Scratch<double> d_gstate;     // variant 3: per-CTA scenario state slabs
    int no_specialise = 0;        // $HPF_NO_SPECIALISE=1: always use the runtime-dimension kernels
    int shape = 0;                // shape-specialised instances of the network (see with_shape), 0 = none
    int fund_shape = 0;           // the same for fund_tile_kernel, matched on (n, c) only: it reads no other dimension
    int mismatch_tile = 0;        // $HPF_MISMATCH_TILE=1: standalone mismatch through the tile kernel
    int gj_single_max = 768;      // $HPF_GJ_SINGLE_MAX: largest order inverted by the one-CTA Gauss-Jordan kernel (tests: 0 forces the multi-CTA paths)
    int gj_unblocked = 0;         // $HPF_GJ_UNBLOCKED=1: multi-CTA Gauss-Jordan with one rank-1 update of the whole matrix per pivot (round-1 kernel) instead of the blocked one
    int setup_gj = 0;             // $HPF_SETUP=gj: variant 3 set-up by Gauss-Jordan inversion of the whole A_ZZ (round-1 path) instead of the Woodbury form
    int wn_kernel = 0;            // $HPF_WN_KERNEL=fma|dmma: generic w_N = W_NL I_N product on the CUDA-core pipe (wn_tile_kernel) or on the FP64 tensor cores (zgemm_dmma_kernel); 0 = default
    int lu_classic = 0;           // $HPF_LU_CLASSIC=1: shared-memory LU with rank-1 updates (lu_solve_smem) instead of the panel LU
    int force_variant = 0;        // $HPF_STRUCT_VARIANT=2|3: force a per-CTA variant of the harmonic stage
    // lock-step batched harmonic stage of the large networks (hpf_lockstep.cuh)
    int lockstep = -1;            // $HPF_LOCKSTEP=0|1: never / always; default (-1): batches of at least HPF_LS_AUTO_MIN_B scenarios
    size_t ls_budget = 0;         // $HPF_LOCKSTEP_GB: device memory the lock-step work areas may take (0 = 40 % of the free memory, at most 64 GB)
    Scratch<char> d_ls;           // one allocation: state slabs | border systems | X | GX | U0 | ints
    int last_path = 0;            // hpf_last_solve_path
    // host mirror of the network constants for kernels that take them as parameters
    // (constant bank): fetched lazily from the device tables, see host_consts()
    std::vector<double2> hY, hYN, hWNL, hG;
    std::vector<char> hw_consts;  // HwConsts<D, coupled> of the one-warp-per-harmonic kernel (empty: not built)
    int harm_tile_only = 0;       // $HPF_HARM_KERNEL=tile: 32-scenario tile kernel instead (A/B measurements)
    int max_ctas = 0;             // $HPF_MAX_CTAS: cap on the grid of the persistent kernels (tests: forces queue refills on small batches)
    std::vector<int> hdev;
    bool host_consts_valid = false;
    double pivot_min = 0.0, pivot_max = 0.0;
    int profiling = 0;
    Event ev[3];
    int ev_valid = 0;             // 0 none, 1 structured (3 events), 2 dense (ev[1], ev[2])
    long long launches = 0;
    Event ev_last;                // recorded after the last kernel sequence of this handle
    cudaStream_t last_stream = nullptr;
    bool last_valid = false;
    std::string err;
};

static thread_local std::string g_create_err;

static int fail(hpf_t* h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_create_err = msg;
    return code;
}
#define CK(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess)                                                           \
            return fail(h, HPF_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

// Makes the handle's device current for the duration of an entry point and restores the caller's
// current device on exit: a process may hold handles on several GPUs, and torch reads the
// current device with cudaGetDevice.
struct DeviceGuard {
    int prev = -1;
    cudaError_t err;
    explicit DeviceGuard(int dev) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ENTER_DEVICE(h) DeviceGuard dg_((h)->device); CK(dg_.err)

// One kernel sequence in flight per handle.  The work-queue counter, the w_N scratch, the LU
// workspaces and Y(h) itself live in the handle, so a call that arrives on a DIFFERENT stream than
// the previous one is ordered after it (event wait on the device, the host does not block);
// calls on the same stream are ordered by the stream.  A stream that is being CAPTURED into a
// CUDA graph is left alone (an event recorded inside a capture cannot be waited on from outside
// it, and the other way round): the owner of the graph orders its replays against other work.
static bool stream_capturing(cudaStream_t st) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
    return cs != cudaStreamCaptureStatusNone;
}
static int order_after_previous(hpf_t* h, cudaStream_t st) {
    if (h->last_valid && st != h->last_stream && !stream_capturing(st)) CK(cudaStreamWaitEvent(st, h->ev_last.get(), 0));
    return HPF_OK;
}
static int mark_last(hpf_t* h, cudaStream_t st) {
    if (stream_capturing(st)) return HPF_OK;
    CK(cudaEventRecord(h->ev_last.get(), st));
    h->last_stream = st;
    h->last_valid = true;
    return HPF_OK;
}

// Runs one entry point's launches ordered after the handle's previous kernel sequence and
// records the event the next one will wait on.
template <class F>
static int ordered(hpf_t* h, void* stream, F body) {
    if (!h) return body();
    ENTER_DEVICE(h);
    int rc = order_after_previous(h, (cudaStream_t)stream);
    if (rc) return rc;
    rc = body();
    if (rc) return rc;
    return mark_last(h, (cudaStream_t)stream);
}

static DevNet devnet(const hpf_t* h) {
    DevNet d;
    d.n = h->n; d.m = h->m; d.c = h->c; d.H = h->H; d.q = h->q;
    d.nH = h->n * h->H;
    d.N = 2 * d.nH - 1 - h->c;
    d.Nf = 2 * h->n - 1 - h->c;
    d.coupled = h->coupled;
    d.Y = h->d_Y.get(); d.YN = h->d_YN.get(); d.dev_of_nl = h->d_devof.get();
    d.ell_col = h->d_ell_col.get(); d.ell_w = h->ell_w;
    return d;
}

// Reports a failed allocation of `bytes` for `who` (entry point and buffer).  A failed allocation
// leaves its error as the runtime's last error, which is consumed here: the next launch check
// would otherwise report it as its own.
static int alloc_failed(hpf_t* h, cudaError_t e, const char* who, size_t bytes) {
    cudaGetLastError();
    return fail(h, e == cudaErrorMemoryAllocation ? HPF_E_NOMEM : HPF_E_CUDA,
                std::string(who) + ": allocation of " + std::to_string(bytes) + " B: " + cudaGetErrorString(e));
}

// Frees what p holds, then allocates `bytes` into it
template <class T>
static int dev_alloc(hpf_t* h, DevPtr<T>& p, size_t bytes, const char* who) {
    p.reset();
    void* raw = nullptr;
    const cudaError_t e = cudaMalloc(&raw, bytes);
    if (e != cudaSuccess) return alloc_failed(h, e, who, bytes);
    p.reset(static_cast<T*>(raw));
    return HPF_OK;
}

template <class T>
static int upload(hpf_t* h, DevPtr<T>& dst, const T* src, size_t count, const char* who) {
    const int rc = dev_alloc(h, dst, (count ? count : 1) * sizeof(T), who);
    if (rc) return rc;
    if (src && count) CK(cudaMemcpy(dst.get(), src, count * sizeof(T), cudaMemcpyHostToDevice));
    return HPF_OK;
}

// Grow-only scratch: reallocated only for a request larger than any before it.  Work in flight may
// still read the old buffer, so the device is synchronised before it is freed; after
// hpf_prepare(B_max), solves of up to B_max scenarios return at the first line.
template <class T>
static int grow(hpf_t* h, Scratch<T>& buf, size_t bytes, const char* who) {
    if (bytes <= buf.bytes) return HPF_OK;
    if (buf.p) CK(cudaDeviceSynchronize());
    const int rc = dev_alloc(h, buf.p, bytes, who);
    buf.bytes = rc ? 0 : bytes;
    return rc;
}

// Y(h) or the device tables changed: the structured operators and the host mirrors are rebuilt
// when next needed.  `pattern`: Y(h) itself changed, so its sparsity pattern goes as well.
static void invalidate_derived(hpf_t* h, bool pattern) {
    h->struct_state = 0;
    h->host_consts_valid = false;
    if (pattern) { h->d_ell_col.reset(); h->ell_w = 0; }
}

static cudaError_t create_event(Event& ev, unsigned flags) {
    cudaEvent_t raw = nullptr;
    const cudaError_t e = cudaEventCreateWithFlags(&raw, flags);
    if (e == cudaSuccess) ev.reset(raw);
    return e;
}

static int ready(hpf_t* h, const char* who, bool need_dev) {
    if (!h) return HPF_E_INVALID;
    if (!h->have_net || !h->have_Y)
        return fail(h, HPF_E_INVALID, std::string(who) + ": call hpf_set_network and hpf_build_Y first");
    if (need_dev && h->q > 0 && !h->have_dev)
        return fail(h, HPF_E_INVALID, std::string(who) + ": call hpf_set_devices first");
    return HPF_OK;
}

// Does the dense system fit the shared-memory LU (matrix + state in smem, N <= 32*MAXCHUNK)?
static bool fits_smem_lu(const hpf_t* h, const DevNet& net) {
    return net.N <= 32 * HPF_LU_MAXCHUNK &&
           scn_smem_bytes(net.n, net.H, net.q, net.N, true) <= (size_t)h->smem_optin;
}

// ---- kernel launches --------------------------------------------------------------------
// A kernel takes up to 48 KB of dynamic shared memory by default; beyond that it must be allowed per kernel.
template <class K>
static cudaError_t allow_smem(K kernel, size_t smem) {
    if (smem <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

// CTAs of `kernel` the device holds at once with `threads` threads and `smem` B of dynamic shared
// memory -> *ctas.  `who`: the entry point named in the error messages.
template <class K>
static int resident_ctas(hpf_t* h, K kernel, int threads, size_t smem, const char* who, long long* ctas) {
    if (smem > (size_t)h->smem_optin)
        return fail(h, HPF_E_UNSUPPORTED,
                    std::string(who) + ": system too large for the shared-memory path (needs " +
                        std::to_string(smem) + " B of shared memory per CTA, device offers " +
                        std::to_string(h->smem_optin) + ")");
    CK(allow_smem(kernel, smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem));
    if (occ < 1) return fail(h, HPF_E_UNSUPPORTED, std::string(who) + ": kernel does not fit on an SM");
    *ctas = (long long)occ * h->sm_count;
    return HPF_OK;
}

// Grid of a kernel whose CTAs loop over `items` work items: the resident CTAs, at most one per item and
// at least one; a work-queue kernel (`queue`) also at most $HPF_MAX_CTAS.
static unsigned fill_grid(const hpf_t* h, long long ctas, long long items, bool queue) {
    long long g = ctas < items ? ctas : items;
    if (queue && h->max_ctas && g > h->max_ctas) g = h->max_ctas;
    return (unsigned)(g < 1 ? 1 : g);
}

// Grid, block, dynamic shared memory and stream of one launch; cluster > 0: thread-block clusters of
// that many CTAs along x
struct LaunchCfg {
    dim3 grid, block;
    size_t smem;
    cudaStream_t st;
    int cluster = 0;
};

// The one place that launches a kernel.  The launch counts 1 (hpf_launch_count) and is checked at once;
// its error is consumed so that it does not stay behind as the runtime's last error.
template <class... P, class... A>
static int launch(hpf_t* h, void (*kernel)(P...), const LaunchCfg& c, A&&... args) {
    CK(allow_smem(kernel, c.smem));
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = (unsigned)c.cluster; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = c.grid; cfg.blockDim = c.block; cfg.dynamicSmemBytes = c.smem; cfg.stream = c.st;
    cfg.attrs = &attr; cfg.numAttrs = c.cluster > 0 ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(h, HPF_E_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e));
    }
    h->launches++;
    return HPF_OK;
}

// Shape-specialised instances exist for the BASELINE configurations' 4-bus networks: shape 1 is
// config 3 (net3, 13 harmonics), shape 2 config 2 (net2 with two nonlinear buses, 10 harmonics).
// with_shape(s, f) calls f(Dims<...>{}) of shape s = 1..HPF_SHAPES; with_dims also takes s = 0 and
// then calls f(DynDims{}), the runtime-dimension instance.
#define HPF_SHAPES 2
template <class F>
static auto with_shape(int shape, F&& f) {
    return shape == 1 ? f(Dims<4, 3, 2, 13, 1>{}) : f(Dims<4, 2, 1, 10, 2>{});
}
template <class F>
static auto with_dims(int shape, F&& f) {
    return shape ? with_shape(shape, f) : f(DynDims{});
}

// LU of the per-scenario kernels (solve_kernel, lu_solve_kernel, harm_cta_kernel): kind 0 = matrix
// in shared memory; 1 = matrix in a per-CTA global workspace, scenario state + blocked-LU staging
// (lubd doubles) in shared memory; 2 = the same with oversized panels.  with_lu_kind calls
// f(std::integral_constant<int, kind>{}).
struct LuPlan {
    int kind;
    size_t lubd, smem;
};
static LuPlan lu_plan(const hpf_t* h, const DevNet& net) {
    if (fits_smem_lu(h, net)) return {0, 0, scn_smem_bytes(net.n, net.H, net.q, net.N, true)};
    const size_t lubd = gmem_kernel_lub_doubles(net.n, net.H, net.q, net.N, (size_t)h->smem_optin);
    const size_t smem = (scn_smem_doubles_aligned(net.n, net.H, net.q, net.N) + lubd) * sizeof(double) + 16;
    return {lub_needs_big(net.N, lubd) ? 2 : 1, lubd, smem};
}
template <class F>
static auto with_lu_kind(int kind, F&& f) {
    return kind == 0 ? f(std::integral_constant<int, 0>{})
                     : kind == 1 ? f(std::integral_constant<int, 1>{}) : f(std::integral_constant<int, 2>{});
}

// Flat start (HG:183) of the harmonic rows h = 2..H of a batch whose fundamental stage ran on the
// one-harmonic view.
static int flat_start_harmonics(hpf_t* h, int n, int H, int B, double* V_m, double* V_a, cudaStream_t st) {
    const size_t cnt = (size_t)(H - 1) * n * B;
    return launch(h, flat_start_fill_kernel, {(unsigned)((cnt + 255) / 256 < 65535 * 8 ? (cnt + 255) / 256 : 65535 * 8), 256, 0, st},
                  V_m + (size_t)n * B, V_a + (size_t)n * B, cnt);
}

// ---- solve requests -------------------------------------------------------------------
// Outputs of a batch solve ([rows, B] layout): the device buffers of hpf_solve, the host arrays of
// hpf_solve_host, or the device copies that hpf_solve_host_keep leaves behind.
struct BatchOut {
    double *V_m = nullptr, *V_a = nullptr;
    double2* I_inj = nullptr;
    int *n_iter_f = nullptr, *n_iter_h = nullptr, *status = nullptr;
    double* err_h = nullptr;
};

// One solve request as it travels through the host solve path: built once by the entry point,
// then read by every stage and kernel argument block.
struct SolveReq {
    int B = 0, flags = 0;
    const double *P = nullptr, *Q = nullptr;
    const double2* I_N = nullptr;
    double thresh_f = 0.0, thresh_h = 0.0;
    int max_f = 0, max_h = 0;
    BatchOut out;
    double *err_f = nullptr, *hist_f = nullptr, *hist_h = nullptr;
    // hpf_solve_host runs consecutive chunks on several compute streams (the tail of chunk k overlaps
    // the start of chunk k+1), so each chunk in flight has its own work counter and w_N scratch
    int slot = 0;                 // work-counter slot: the chunk index of a dual-stream hpf_solve_host, else 0
    size_t wN_off = 0;            // offset of this solve's w_N scratch inside h->d_wN
};

// Argument checks of a solve request at entry point `who`, in this order: handle ready, B < 0, NULL
// buffers.  I_N is needed only with nonlinear buses; the fundamental-only solve (mode 1) needs no
// device tables and has no harmonic outputs.  A request with B == 0 passes: it has nothing to do.
// Mode 2 is the statistics host solve: a whole solve whose per-scenario outputs are all optional.
static int check_request(hpf_t* h, const SolveReq& r, int mode, const char* who) {
    int rc = ready(h, who, mode != 1);
    if (rc) return rc;
    if (r.B < 0) return fail(h, HPF_E_INVALID, std::string(who) + ": B < 0");
    if (r.B == 0) return HPF_OK;
    const BatchOut& o = r.out;
    const bool outs = mode == 2 || (o.V_m && o.V_a && o.n_iter_f && (mode == 1 || (o.n_iter_h && o.err_h && o.status)));
    if (!r.P || !r.Q || !outs || (mode != 1 && h->q > 0 && !r.I_N))
        return fail(h, HPF_E_INVALID, std::string(who) + ": NULL buffer");
    return HPF_OK;
}

// The fundamental stage of a request on its own: the harmonic stage's inputs, limits and outputs
// cleared, as hpf_fund_solve passes them.
static SolveReq fund_stage(SolveReq r) {
    r.flags = 0; r.I_N = nullptr; r.thresh_h = 0.0; r.max_h = 0; r.hist_h = nullptr;
    r.out.I_inj = nullptr; r.out.n_iter_h = nullptr; r.out.err_h = nullptr;
    return r;
}

static SolveArgs solve_args(const hpf_t* h, const SolveReq& r, int mode, const LuPlan& lu, double* workspace) {
    SolveArgs a;
    a.B = r.B; a.mode = mode; a.flags = r.flags; a.P = r.P; a.Q = r.Q; a.I_N = r.I_N;
    a.hist_f = r.hist_f; a.hist_h = r.hist_h;
    a.thresh_f = r.thresh_f; a.thresh_h = r.thresh_h; a.max_f = r.max_f; a.max_h = r.max_h;
    a.V_m = r.out.V_m; a.V_a = r.out.V_a; a.I_inj = r.out.I_inj;
    a.n_iter_f = r.out.n_iter_f; a.n_iter_h = r.out.n_iter_h; a.status = r.out.status; a.err_h = r.out.err_h;
    a.err_f = r.err_f;
    a.work_counter = h->d_counter.get() + r.slot;
    a.workspace = workspace;
    a.lub_doubles = (int)lu.lubd;
    a.lu_classic = h->lu_classic;
    return a;
}

// Per-scenario solve kernel over a checked request with B > 0: mode 0 the whole solve (dense path),
// mode 1 the fundamental stage only.
static int solve_common(hpf_t* h, int mode, const SolveReq& r, cudaStream_t st) {
    const char* who = mode ? "hpf_fund_solve" : "hpf_solve";
    DevNet net = devnet(h);
    if (mode == 1) net.N = net.Nf;      // fundamental only: size the matrix for Nf
    const int H_full = net.H;
    if (mode == 1 && !fits_smem_lu(h, net)) {
        // large network: the fundamental stage only needs the h = 1 block of the state, so the
        // kernel sees a one-harmonic view (its per-scenario arrays are sized by nH) and the
        // flat start of the harmonic rows is written by a fill kernel
        net.H = 1; net.nH = net.n;
    }
    const LuPlan lu = lu_plan(h, net);
    const auto kernel = with_lu_kind(lu.kind, [](auto k) { return solve_kernel<decltype(k)::value>; });
    const int threads = lu.kind ? HPF_THREADS_GMEM : HPF_THREADS;
    long long ctas = 0;
    int rc = resident_ctas(h, kernel, threads, lu.smem, who, &ctas);
    if (rc) return rc;
    CK(cudaMemsetAsync(h->d_counter.get() + r.slot, 0, sizeof(int), st));
    const unsigned grid = fill_grid(h, ctas, r.B, true);
    double* workspace = nullptr;
    if (lu.kind) {
        rc = grow(h, h->d_work, (size_t)grid * lub_ld(net.N) * (net.N + 1) * sizeof(double),
                  mode ? "hpf_fund_solve: LU workspace" : "hpf_solve: LU workspace");
        if (rc) return rc;
        workspace = h->d_work.get();
    }
    if (h->profiling) { CK(cudaEventRecord(h->ev[1].get(), st)); }
    rc = launch(h, kernel, {grid, threads, lu.smem, st}, net, solve_args(h, r, mode, lu, workspace));
    if (!rc && net.H != H_full) rc = flat_start_harmonics(h, net.n, H_full, r.B, r.out.V_m, r.out.V_a, st);
    if (rc) return rc;
    if (h->profiling) { CK(cudaEventRecord(h->ev[2].get(), st)); h->ev_valid = 2; }
    return HPF_OK;
}

// ---- structured strategy: setup (once per network) and launches -----------------------
static StructNet structnet(const hpf_t* h) {
    StructNet s;
    s.nZ = h->n * h->H - h->m;
    s.nx = (h->m - 1) + (h->m - h->c);
    s.Ainv = h->d_struct.Ainv.get();
    s.G = h->d_struct.Gz.get();
    s.GT = h->d_struct.GzT.get();
    s.nbr_ptr = h->d_struct.nbr_ptr.get();
    s.nbr_idx = h->d_struct.nbr_idx.get();
    s.WNL = h->d_struct.WNL.get();
    s.yn_elems = h->n_dev * (h->coupled ? h->H * h->H : h->H);
    return s;
}

static int host_consts(hpf_t* h);
static int launch_zgemm(hpf_t* h, int M, int N, int K, const double2* A, size_t lda, const double2* B, size_t ldb,
                        double2* C, size_t ldc, cudaStream_t st, bool subtract = false, const int* n_dev = nullptr);

// In-place complex Gauss-Jordan inverse with partial pivoting of one matrix of order nn (row-major):
// one CTA for nn <= gj_single_max (768), else four small launches per pivot over the whole GPU.  info[0] = 0
// or k + 1 (zero pivot), pr[0..1] = min / max pivot modulus.  ipiv: nn ints, tmp: 2 nn + 1 double2 (only
// read for nn > gj_single_max).
static int gj_invert(hpf_t* h, double2* A, int nn, int* ipiv, int* info, double* pr, double2* tmp, cudaStream_t st,
                     double2* FR = nullptr) {
    if (nn <= h->gj_single_max) return launch(h, cinv_gj_kernel, {1, 1024, 0, st}, nn, A, ipiv, info, pr);
    const unsigned g1 = (nn + 255) / 256;
    int rc;
    if (FR && !h->gj_unblocked) {
        // blocked: panels of GJB_NB pivots, the rest of the matrix updated by one tensor-core GEMM per panel
        double2 *rowk = tmp, *pinv = tmp + 2 * (size_t)nn;
        double2 *F = FR, *R = FR + (size_t)nn * GJB_NB, *pinv_all = R + (size_t)GJB_NB * nn;
        for (int j0 = 0; j0 < nn; j0 += GJB_NB) {
            const int nb = nn - j0 < GJB_NB ? nn - j0 : GJB_NB, j1 = j0 + nb;
            int ge = (nn + 3) / 4;
            if (ge > h->sm_count * 8) ge = h->sm_count * 8;
            for (int k = j0; k < j1; ++k) {
                if ((rc = launch(h, gjb_pivot_row_kernel, {1, 1024, 0, st}, nn, k, j0, j1, A, ipiv, info, pr, pinv, rowk, F,
                                 pinv_all))) return rc;
                if ((rc = launch(h, gjb_col_elim_kernel, {(unsigned)ge, dim3(GJB_NB, 4), 0, st}, nn, k, j0, j1, A, rowk, pinv,
                                 F))) return rc;
            }
            if ((rc = launch(h, gjb_rows_kernel, {g1, 256, 0, st}, nn, j0, nb, A, ipiv, F, pinv_all, R))) return rc;
            if ((rc = launch_zgemm(h, nn, nn, nb, F, (size_t)GJB_NB, R, (size_t)nn, A, (size_t)nn, st, true))) return rc;
        }
    } else {
        double2 *rowk = tmp, *colk = tmp + nn, *pinv = tmp + 2 * (size_t)nn;
        unsigned gy = (h->sm_count * 8 + g1 - 1) / g1;
        if (gy > (unsigned)nn) gy = nn;
        for (int k = 0; k < nn; ++k) {
            if ((rc = launch(h, gjm_pivot_kernel, {1, 1024, 0, st}, nn, k, A, ipiv, info, pr, pinv))) return rc;
            if ((rc = launch(h, gjm_row_kernel, {g1, 256, 0, st}, nn, k, A, ipiv, pinv, rowk))) return rc;
            if ((rc = launch(h, gjm_col_kernel, {g1, 256, 0, st}, nn, k, A, colk))) return rc;
            if ((rc = launch(h, gjm_elim_kernel, {dim3(g1, gy), 256, 0, st}, nn, k, A, rowk, colk))) return rc;
        }
    }
    return launch(h, gjm_unpermute_kernel, {g1, 256, 0, st}, nn, A, ipiv);
}

template <class T>
static int alloc_async(hpf_t* h, AsyncPtr<T>& p, size_t count, cudaStream_t st, const char* who) {
    void* raw = nullptr;
    const cudaError_t e = cudaMallocAsync(&raw, count * sizeof(T), st);
    if (e != cudaSuccess) return alloc_failed(h, e, who, count * sizeof(T));
    p = AsyncPtr<T>(static_cast<T*>(raw), AsyncFree{st});
    return HPF_OK;
}

// Structured set-up of the large networks through the block structure of A_ZZ (Woodbury identity,
// see hpf_structured.cuh): fills the operators W_NL, G, G^T; *info_out = 0 or a zero-pivot indicator,
// prh = min / max pivot modulus over all inversions.
static int setup_woodbury(hpf_t* h, const DevNet& net, cudaStream_t st, int* info_out, double* prh) {
    const int n = net.n, m = net.m, q = net.q, H = net.H, qH = q * H, nZ = net.nH - m;
    const size_t nblk = (size_t)q * q + (size_t)(H - 1) * n * n;
    const int nmax = n > qH ? n : qH;
    double2 *const WNL = h->d_struct.WNL.get(), *const Gz = h->d_struct.Gz.get(), *const GzT = h->d_struct.GzT.get();
    const bool timing = getenv("HPF_SETUP_TIMING") != nullptr;       // phase times on stderr (synchronises)
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto tprev = now();
    auto tick = [&](const char* what) {
        if (!timing) return;
        cudaStreamSynchronize(st);
        const auto t = now();
        fprintf(stderr, "[hpf setup] %-34s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t - tprev).count());
        tprev = t;
    };
    // stream-ordered temporaries: a plain cudaFree of these ~1.7 GB costs 160 ms
    AsyncPtr<double2> Dinv, Mx, T, U, tmp, FR;
    AsyncPtr<int> ipiv, info;
    AsyncPtr<double> pr;
    const char* who = "structured set-up: Woodbury temporaries";
    int rc = alloc_async(h, Dinv, nblk + 1, st, who);
    if (!rc) rc = alloc_async(h, Mx, (size_t)qH * qH + 1, st, who);
    if (!rc) rc = alloc_async(h, T, (size_t)q * m + 1, st, who);
    if (!rc) rc = alloc_async(h, U, (size_t)qH * m + 1, st, who);
    if (!rc) rc = alloc_async(h, tmp, (size_t)2 * nmax + 1, st, who);
    if (!rc) rc = alloc_async(h, FR, (size_t)2 * nmax * GJB_NB + GJB_NB + 1, st, who);      // F, R, 1 / pivots
    if (!rc) rc = alloc_async(h, ipiv, (size_t)nmax + 2, st, who);
    if (!rc) rc = alloc_async(h, info, (size_t)H + 1, st, who);
    if (!rc) rc = alloc_async(h, pr, (size_t)2 * (H + 1), st, who);
    if (rc) return rc;
    tick("allocations");
    const unsigned g8 = h->sm_count * 8;
    rc = launch(h, wb_blocks_kernel, {g8, 256, 0, st}, net, Dinv.get());
    for (int hh = 0; hh < H && !rc; ++hh) {
        double2* blk = hh == 0 ? Dinv.get() : Dinv.get() + (size_t)q * q + (size_t)(hh - 1) * n * n;
        rc = gj_invert(h, blk, hh == 0 ? q : n, ipiv.get(), info.get() + hh, pr.get() + 2 * hh, tmp.get(), st, FR.get());
    }
    tick("block inversions D_h");
    if (!rc) rc = launch(h, wb_capacitance_kernel, {g8, 256, 0, st}, net, Dinv.get(), Mx.get());
    if (!rc) rc = gj_invert(h, Mx.get(), qH, ipiv.get(), info.get() + H, pr.get() + 2 * H, tmp.get(), st, FR.get());
    tick("capacitance matrix M: build + invert");
    // W_NL = (D^-1 E) M^-1, one GEMM per harmonic block: rows of block h x the rows (k, h) of M^-1
    for (int hh = 0; hh < H && !rc; ++hh) {
        const double2* blk = hh == 0 ? Dinv.get() : Dinv.get() + (size_t)q * q + (size_t)(hh - 1) * n * n;
        const int rows = hh == 0 ? q : n;
        const double2* Ablk = hh == 0 ? blk : blk + m;               // columns of the nonlinear buses
        const size_t z0 = hh == 0 ? 0 : (size_t)hh * n - m;
        rc = launch_zgemm(h, rows, qH, q, Ablk, (size_t)rows, Mx.get() + (size_t)hh * qH, (size_t)H * qH,
                          WNL + z0 * qH, (size_t)qH, st);
    }
    // T = D_0^-1 Y_0[nl, lin];  U = YN E^T D^-1 A_ZF;  G = W_NL U + [T; 0]
    if (!rc) rc = launch_zgemm(h, q, m, q, Dinv.get(), (size_t)q, net.Y + (size_t)m * n, (size_t)n, T.get(), (size_t)m, st);
    if (!rc) rc = launch(h, wb_coupling_rhs_kernel, {(unsigned)h->sm_count * 4, 256, 0, st}, net, T.get(), U.get());
    if (!rc) rc = launch_zgemm(h, nZ, m, qH, WNL, (size_t)qH, U.get(), (size_t)m, Gz, (size_t)m, st);
    if (!rc) rc = launch(h, wb_finish_G_kernel, {g8, 256, 0, st}, nZ, m, q, T.get(), Gz, GzT);
    tick("W_NL, G (tensor-core GEMMs)");
    if (rc) return rc;
    std::vector<int> hinfo((size_t)H + 1);
    std::vector<double> hpr((size_t)2 * (H + 1));
    CK(cudaMemcpyAsync(hinfo.data(), info.get(), hinfo.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hpr.data(), pr.get(), hpr.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    tick("read-back");
    *info_out = 0;
    prh[0] = 1.0e308; prh[1] = 0.0;
    for (int t = 0; t <= H; ++t) {
        if (hinfo[(size_t)t] != 0 && *info_out == 0) *info_out = hinfo[(size_t)t];
        prh[0] = hpr[(size_t)2 * t] < prh[0] ? hpr[(size_t)2 * t] : prh[0];
        prh[1] = hpr[(size_t)2 * t + 1] > prh[1] ? hpr[(size_t)2 * t + 1] : prh[1];
    }
    return HPF_OK;
}

// Constants of the one-warp-per-harmonic kernel (hpf_harmonic_warp.cuh) for a shape-specialised
// network, from the host mirrors of Y(h), Y_N and G: kept in the handle, passed BY VALUE at launch.
template <class D>
static void build_hw_consts(hpf_t* h) {
    constexpr int n = D::n, m = D::m, H = D::H, q = D::q;
    auto fill = [&](auto* C) {
        for (int t = 0; t < H * n * n; ++t) C->Y[t] = h->hY[(size_t)t];
        const int per = h->coupled ? H * H : H;
        for (int k = 0; k < q; ++k)
            for (int t = 0; t < per; ++t) C->YNk[k * per + t] = h->hYN[(size_t)h->hdev[(size_t)k] * per + t];
        for (size_t t = 0; t < h->hG.size(); ++t) C->G[t] = h->hG[t];
        // Yeff_ij = Y1_ij - sum_k Y1_{i,m+k} G[k][j]   (row z = k of G: fundamental, nonlinear bus k)
        for (int i = 0; i < m; ++i)
            for (int j = 0; j < m; ++j) {
                double2 v = h->hY[(size_t)i * n + j];
                for (int k = 0; k < q; ++k) {
                    const double2 y = h->hY[(size_t)i * n + m + k], g = h->hG[(size_t)k * m + j];
                    v.x -= y.x * g.x - y.y * g.y;
                    v.y -= y.x * g.y + y.y * g.x;
                }
                C->Yeff[i * m + j] = v;
            }
    };
    if (h->coupled) {
        h->hw_consts.assign(sizeof(HwConsts<D, true>), 0);
        fill(reinterpret_cast<HwConsts<D, true>*>(h->hw_consts.data()));
    } else {
        h->hw_consts.assign(sizeof(HwConsts<D, false>), 0);
        fill(reinterpret_cast<HwConsts<D, false>*>(h->hw_consts.data()));
    }
}

// Structured set-up, once per network.  Variants of the harmonic stage:
//   1  32-scenario tile kernels (state of 32 scenarios in shared memory: the 4-bus networks)
//   2  one scenario per CTA, state in shared memory (net1: 20 buses x 26 harmonics)
//   3  one scenario per CTA, state in a global-memory slab, blocked tensor-core LU for the
//      border system (200- / 1000-bus configurations)
static int ensure_struct(hpf_t* h, cudaStream_t st) {
    if (h->struct_state != 0) return HPF_OK;
    h->struct_state = -1;
    // allocation inside the set-up: out of device memory is not an error of the solve - the structured
    // buffers are released, the reason is left in hpf_last_error() and hpf_solve uses the dense strategy
#define SK(ptr, bytes)                                                                                \
    do {                                                                                              \
        const int rc_ = dev_alloc(h, ptr, (bytes), "structured set-up: " #ptr);                        \
        if (rc_ == HPF_E_NOMEM) {                                                                     \
            h->d_struct = {};                                                                         \
            h->err = "structured set-up skipped (out of device memory for " #ptr "): dense strategy"; \
            return HPF_OK;                                                                            \
        }                                                                                             \
        if (rc_) return rc_;                                                                          \
    } while (0)
    const DevNet net = devnet(h);
    const int nZ = net.nH - net.m;
    if (nZ < 1) return HPF_OK;
    int variant = 1;
    if (harm_tile_smem_bytes(net.n, net.H, net.m, net.c, net.q, 8,
                             h->n_dev * (h->coupled ? h->H * h->H : h->H)) > (size_t)h->smem_optin ||
        fund_tile_doubles_per_warp(net.n, net.Nf) * sizeof(double) > (size_t)h->smem_optin)
        variant = 2;
    if (variant == 2) {
        const int nx = (net.m - 1) + (net.m - net.c);
        if (harm_cta_smem_bytes(net.n, net.H, net.m, net.c, net.q, net.N) > (size_t)h->smem_optin ||
            nx > 32 * HPF_LU_MAXCHUNK || net.Nf > 32 * HPF_LU_MAXCHUNK ||
            scn_smem_bytes(net.n, net.H, net.q, net.Nf, true) > (size_t)h->smem_optin)
            variant = 3;
    }
    if (h->force_variant >= 2 && h->force_variant > variant) variant = h->force_variant;   // (tests)
    if (variant == 3) {                                 // fundamental stage: one-harmonic view, see solve_common
        DevNet nf = net;
        nf.N = nf.Nf; nf.H = 1; nf.nH = nf.n;
        if (!fits_smem_lu(h, nf) && gmem_kernel_smem_bytes(nf.n, 1, nf.q, nf.N) > (size_t)h->smem_optin)
            return HPF_OK;                              // (n beyond ~2000 buses)
    }
    StructBufs& sb = h->d_struct;
    sb = {};
    const int qH = net.q * net.H;
    // nonlinear neighbours of the linear buses (structure of Y1), from the host mirror of Y
    {
        int rc = host_consts(h);
        if (rc) return rc;
        std::vector<int> ptr((size_t)net.m + 1, 0), idx;
        for (int i = 0; i < net.m; ++i) {
            for (int k = 0; k < net.q; ++k) {
                const double2 y = h->hY[(size_t)i * net.n + net.m + k];
                if (y.x != 0.0 || y.y != 0.0) idx.push_back(k);
            }
            ptr[(size_t)i + 1] = (int)idx.size();
        }
        rc = upload(h, sb.nbr_ptr, ptr.data(), ptr.size(), "structured set-up: neighbour lists");
        if (!rc) rc = upload(h, sb.nbr_idx, idx.data(), idx.size(), "structured set-up: neighbour lists");
        if (rc) return rc;
        // sparsity pattern of Y(h), union over the harmonics (diagonal always listed)
        h->d_ell_col.reset(); h->ell_w = 0;
        if (net.n >= 16) {
            const int n = net.n;
            std::vector<std::vector<int>> cols((size_t)n);
            int w = 0;
            for (int i = 0; i < n; ++i) {
                for (int j = 0; j < n; ++j) {
                    bool nz = (i == j);
                    for (int hh = 0; hh < net.H && !nz; ++hh) {
                        const double2 y = h->hY[((size_t)hh * n + i) * n + j];
                        nz = (y.x != 0.0 || y.y != 0.0);
                    }
                    if (nz) cols[(size_t)i].push_back(j);
                }
                if ((int)cols[(size_t)i].size() > w) w = (int)cols[(size_t)i].size();
            }
            if (w * 2 <= n) {                            // sparse enough to pay off
                std::vector<int> ell((size_t)n * w, -1);
                for (int i = 0; i < n; ++i)
                    for (size_t e = 0; e < cols[(size_t)i].size(); ++e) ell[(size_t)i * w + e] = cols[(size_t)i][e];
                rc = upload(h, h->d_ell_col, ell.data(), ell.size(), "structured set-up: sparsity pattern of Y(h)");
                if (rc) return rc;
                h->ell_w = w;
            }
        }
    }
    SK(sb.WNL, ((size_t)nZ * qH + 1) * sizeof(double2));
    SK(sb.Gz, (size_t)nZ * net.m * sizeof(double2));
    SK(sb.GzT, (size_t)nZ * net.m * sizeof(double2));
    if (variant == 3 && qH > 0 && !h->setup_gj) {
        // large networks: the operator inverse through its block structure (Woodbury) - no nZ x nZ inverse
        int winfo = -1;
        double wpr[2] = {0.0, 0.0};
        int rcw = setup_woodbury(h, net, st, &winfo, wpr);
        if (rcw) return rcw;
        h->hWNL.clear(); h->hG.clear(); h->hw_consts.clear();
        h->pivot_min = wpr[0]; h->pivot_max = wpr[1];
        if (winfo == 0 && wpr[0] > 0.0 && wpr[1] / wpr[0] < 1e12) h->struct_state = variant;
        return HPF_OK;
    }
    DevPtr<double2> AZF, tmp;         // temporaries of the set-up
    DevPtr<int> ipiv;
    DevPtr<double> pr;
    SK(sb.Ainv, (size_t)nZ * nZ * sizeof(double2));
    SK(AZF, (size_t)nZ * net.m * sizeof(double2));
    SK(ipiv, (size_t)(nZ + 2) * sizeof(int));
    SK(pr, 2 * sizeof(double));
    int rc = launch(h, struct_assemble_kernel, {(unsigned)h->sm_count * 8, 256, 0, st}, net, sb.Ainv.get(), AZF.get());
    if (rc) return rc;
    if (nZ > h->gj_single_max) SK(tmp, ((size_t)2 * nZ + 1) * sizeof(double2));
    rc = gj_invert(h, sb.Ainv.get(), nZ, ipiv.get(), ipiv.get() + nZ, pr.get(), tmp.get(), st);
    if (!rc)
        rc = launch(h, struct_G_kernel, {(unsigned)(((size_t)nZ * net.m + 127) / 128), 128, 0, st}, nZ, net.m,
                    net.q < nZ ? net.q : nZ, sb.Ainv.get(), AZF.get(), sb.Gz.get(), sb.GzT.get());
    if (!rc && qH > 0)
        rc = launch(h, struct_WNL_kernel, {(unsigned)(((size_t)nZ * qH + 127) / 128), 128, 0, st}, net, nZ, sb.Ainv.get(),
                    sb.WNL.get());
    if (rc) return rc;
    int info = -1;
    double prh[2] = {0.0, 0.0};
    cudaError_t e = cudaMemcpyAsync(&info, ipiv.get() + nZ, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(prh, pr.get(), sizeof(prh), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    h->hWNL.clear();
    h->hG.clear();
    h->hw_consts.clear();
    if (variant == 1 && e == cudaSuccess && qH > 0 && (size_t)nZ * qH <= 1024) {   // small operators: host mirror
        h->hWNL.resize((size_t)nZ * qH);
        e = cudaMemcpy(h->hWNL.data(), sb.WNL.get(), h->hWNL.size() * sizeof(double2), cudaMemcpyDeviceToHost);
        h->hG.resize((size_t)nZ * net.m);
        if (e == cudaSuccess)
            e = cudaMemcpy(h->hG.data(), sb.Gz.get(), h->hG.size() * sizeof(double2), cudaMemcpyDeviceToHost);
    }
    if (variant == 3) sb.Ainv.reset();                                   // (GBs for the 1000-bus network)
    if (e != cudaSuccess) return fail(h, HPF_E_CUDA, std::string("structured setup: ") + cudaGetErrorString(e));
    h->pivot_min = prh[0]; h->pivot_max = prh[1];
    // usable when the inversion met no zero pivot and the pivots span < 1e12 (well conditioned)
    if (info == 0 && prh[0] > 0.0 && prh[1] / prh[0] < 1e12) h->struct_state = variant;
    if (h->struct_state == 1 && !h->hG.empty() && h->shape)
        with_shape(h->shape, [&](auto d) { build_hw_consts<decltype(d)>(h); return 0; });
    return HPF_OK;
#undef SK
}

// C [M x N] = A [M x K] B [K x N] (complex, row-major) on the FP64 tensor cores (hpf_zgemm.cuh)
static int launch_zgemm(hpf_t* h, int M, int N, int K, const double2* A, size_t lda, const double2* B, size_t ldb,
                        double2* C, size_t ldc, cudaStream_t st, bool subtract, const int* n_dev) {
    if (M <= 0 || N <= 0) return HPF_OK;
    const dim3 grid((unsigned)((N + ZG_BN - 1) / ZG_BN), (unsigned)((M + ZG_BM - 1) / ZG_BM));
    return launch(h, subtract ? zgemm_dmma_kernel<true> : zgemm_dmma_kernel<false>, {grid, 256, ZG_SMEM_BYTES, st},
                  M, N, K, A, lda, B, ldb, C, ldc, n_dev);
}

// The generic Norton contraction w_N = W_NL I_N runs on the tensor cores for batches of at least one
// full 64-scenario column tile (measured A/B: profiles/r2_wn_dmma_ab.txt: 5-10x the CUDA-core kernel);
// smaller batches - a single scenario would waste 63 / 64 of every DMMA - keep the CUDA-core kernel.
// The choice depends on nothing but B >= 64, and neither kernel's arithmetic depends on the position
// of a scenario in the batch: results are bit-identical for every split of a batch into parts of at
// least 64 scenarios (e.g. over GPUs).  $HPF_WN_KERNEL=fma|dmma forces either.
static bool wn_use_dmma(const hpf_t* h, int nZ, int qH, int B) {
    if (h->wn_kernel) return h->wn_kernel == 2;
    return B >= ZG_BN && nZ >= ZG_BM && qH >= 64;
}

// w_N of a batch into the scratch at offset `off` of h->d_wN; *wN <- where it was written
static int launch_wn(hpf_t* h, const DevNet& net, const StructNet& sn, int B, const double2* I_N, size_t off,
                     const double2** wN, cudaStream_t st) {
    int rc = grow(h, h->d_wN, (off + (size_t)sn.nZ * B) * sizeof(double2), "hpf_solve: w_N scratch");
    if (rc) return rc;
    WnArgs wa;
    wa.B = B; wa.I_N = I_N; wa.wN = h->d_wN.get() + off;
    *wN = wa.wN;
    const int qH = net.q * net.H;
    if (qH == 0) { CK(cudaMemsetAsync(wa.wN, 0, (size_t)sn.nZ * B * sizeof(double2), st)); return HPF_OK; }
    if (h->shape && h->struct_state == 1 && !h->hWNL.empty()) {
        return with_shape(h->shape, [&](auto d) {
            using D = decltype(d);
            static_assert(sizeof(WnConsts<D>) + sizeof(WnArgs) <= 32000, "kernel parameter space");
            WnConsts<D> C;
            memcpy(C.W, h->hWNL.data(), sizeof(C.W));
            return launch(h, wn_lane_kernel<D>, {(unsigned)((B + 127) / 128), 128, 0, st}, C, wa);
        });
    }
    if (wn_use_dmma(h, sn.nZ, qH, B))
        return launch_zgemm(h, sn.nZ, B, qH, sn.WNL, (size_t)qH, I_N, (size_t)B, wa.wN, (size_t)B, st);
    const size_t smem = (size_t)(qH < HPF_WN_UCH ? qH : HPF_WN_UCH) * HPF_T * sizeof(double2) + 16;
    long long ctas = 0;
    rc = resident_ctas(h, wn_tile_kernel, 256, smem, "hpf_solve", &ctas);
    if (rc) return rc;
    const unsigned grid = fill_grid(h, ctas, ((long long)B + HPF_T - 1) / HPF_T, false);
    // few tiles (large networks, small batches): spread the row groups over grid.y as well
    const long long groups = (sn.nZ + 8 * HPF_WN_RPW - 1) / (8 * HPF_WN_RPW);
    long long gy = (ctas + grid - 1) / grid;
    if (gy > groups) gy = groups;
    if (gy < 1) gy = 1;
    return launch(h, wn_tile_kernel, {dim3(grid, (unsigned)gy), 256, smem, st}, net, sn, sn.WNL, wa);
}

template <int NW, int MINB, class D>
static int launch_harm_t(hpf_t* h, const DevNet& net, const StructNet& sn, const HarmTileArgs& ha,
                         bool persistent, cudaStream_t st) {
    const size_t smem = harm_tile_smem_bytes(net.n, net.H, net.m, net.c, net.q, NW, sn.yn_elems);
    long long ctas = 0;
    const int rc = resident_ctas(h, harm_tile_kernel<NW, MINB, D>, NW * 32, smem, "hpf_solve", &ctas);
    if (rc) return rc;
    const long long tiles = ((long long)ha.B + HPF_T - 1) / HPF_T;
    const unsigned grid = persistent ? fill_grid(h, ctas, tiles, true) : (unsigned)tiles;
    return launch(h, harm_tile_kernel<NW, MINB, D>, {grid, NW * 32, smem, st}, net, sn, ha);
}

template <class D>
static int launch_harm_hw(hpf_t* h, const HarmTileArgs& ha, cudaStream_t st) {
    constexpr size_t smem = harm_hw_smem_bytes<D>();
    constexpr int threads = D::H * 32;
    auto go = [&](auto kernel, const auto* C) -> int {
        static_assert(sizeof(*C) + sizeof(HarmTileArgs) <= 32000, "kernel parameter space");
        long long ctas = 0;
        const int rc = resident_ctas(h, kernel, threads, smem, "hpf_solve", &ctas);
        if (rc) return rc;
        const long long tiles = ((long long)ha.B + HPF_T - 1) / HPF_T;
        return launch(h, kernel, {fill_grid(h, ctas, tiles, true), threads, smem, st}, *C, ha);
    };
    if (h->coupled) return go(harm_hw_kernel<D, true>, reinterpret_cast<const HwConsts<D, true>*>(h->hw_consts.data()));
    return go(harm_hw_kernel<D, false>, reinterpret_cast<const HwConsts<D, false>*>(h->hw_consts.data()));
}

static int launch_harm(hpf_t* h, const DevNet& net, const StructNet& sn, const HarmTileArgs& ha,
                       bool persistent, cudaStream_t st) {
    if (h->struct_state >= 2) {
        const bool gst = h->struct_state == 3;
        const size_t lubd = gst ? harm_cta_gmem_lub_doubles(sn.nx, (size_t)h->smem_optin) : 0;
        // threads per CTA: every phase of this kernel is barrier- / latency-bound, and a border system whose
        // panels fit one row per thread of 8 warps runs faster with 8 warps than with 16 (measured, 200-bus
        // feeder, nx = 238: 217 -> 183 ms per 2,048 scenarios; 1000-bus network, nx = 1198: 2.40 -> 2.78 s
        // the other way round) - profiles/r2_gmem_ctas_ab.txt
        const int gthreads = sn.nx <= 256 ? 256 : HPF_THREADS_GMEM;
        const size_t smem = gst ? (lubd + 80) * sizeof(double)
                                : harm_cta_smem_bytes(net.n, net.H, net.m, net.c, net.q, net.N);
        // global-state variant: every phase waits on L2 / HBM, so it runs with twice the warps
        const int kind = !gst ? 0 : lub_needs_big(sn.nx, lubd) ? 2 : 1;
        const auto kernel = with_lu_kind(kind, [](auto k) {
            return harm_cta_kernel<decltype(k)::value ? HPF_THREADS_GMEM : HPF_THREADS, decltype(k)::value == 2>;
        });
        const int threads = gst ? gthreads : HPF_THREADS;
        long long ctas = 0;
        int rc = resident_ctas(h, kernel, threads, smem, "hpf_solve", &ctas);
        if (rc) return rc;
        const unsigned grid = persistent || gst ? fill_grid(h, ctas, ha.B, persistent) : (unsigned)ha.B;
        HarmTileArgs ha2 = ha;
        ha2.gstate = nullptr; ha2.gstate_stride = 0; ha2.lub_doubles = (int)lubd;
        if (gst) {
            const size_t stride = (harm_cta_state_doubles(net.n, net.H, net.m, net.c, net.q, net.N, true) + 15) / 8 * 8;
            const size_t need = stride * (size_t)grid;
            rc = grow(h, h->d_gstate, need * sizeof(double), "hpf_solve: scenario state slabs");
            if (rc) return rc;
            ha2.gstate = h->d_gstate.get(); ha2.gstate_stride = stride;
        }
        return launch(h, kernel, {grid, threads, smem, st}, net, sn, ha2);
    }
    if (h->shape && !h->hw_consts.empty() && !h->harm_tile_only && !ha.step_only && persistent)
        return with_shape(h->shape, [&](auto d) { return launch_harm_hw<decltype(d)>(h, ha, st); });
    if (h->shape)
        return with_shape(h->shape, [&](auto d) { return launch_harm_t<8, 2, decltype(d)>(h, net, sn, ha, persistent, st); });
    const bool two = 2 * harm_tile_smem_bytes(net.n, net.H, net.m, net.c, net.q, 8, sn.yn_elems) + 2048 <=
                     (size_t)h->smem_optin + 1024;
    if (two) return launch_harm_t<8, 2, DynDims>(h, net, sn, ha, persistent, st);
    return launch_harm_t<8, 1, DynDims>(h, net, sn, ha, persistent, st);
}

// $HPF_LS_TIMING=1: per-phase device times of the lock-step rounds on stderr (diagnostics: records an
// event after every launch group and synchronises at the end of the call)
struct LsTimer {
    bool on = false;
    cudaStream_t st = nullptr;
    std::vector<cudaEvent_t> ev;
    std::vector<int> tag;
    void mark(int t) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        ev.push_back(e);
        tag.push_back(t);
    }
    void report(const char* what) {
        if (!on) return;
        static const char* names[] = {"start", "mismatch+compact", "pack+zgemm U0", "border assembly", "LU panel",
                                      "LU swap+trsm", "LU update", "LU backsub", "uf+zgemm G X", "load/store"};
        cudaStreamSynchronize(st);
        double acc[10] = {0};
        for (size_t i = 1; i < ev.size(); ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            acc[tag[i]] += ms;
        }
        double tot = 0;
        for (int t = 1; t < 10; ++t) tot += acc[t];
        fprintf(stderr, "[hpf lock-step timing] %s: total %.1f ms", what, tot);
        for (int t = 1; t < 10; ++t) if (acc[t] > 0) fprintf(stderr, " | %s %.1f", names[t], acc[t]);
        fprintf(stderr, "\n");
        for (auto e : ev) cudaEventDestroy(e);
        ev.clear(); tag.clear();
    }
};
static LsTimer g_ls_timer;

// ---- lock-step batched harmonic stage (hpf_lockstep.cuh) ---------------------------------
// Whether a batch of B systems of the given order goes through the lock-step LU ($HPF_LOCKSTEP)
static bool use_lockstep(const hpf_t* h, int order, int B) {
    if (h->lockstep == 0 || order < 1 || order > HPF_LS_MAX_ORDER) return false;
    return h->lockstep == 1 || B >= HPF_LS_AUTO_MIN_B;
}

// Doubles per lock-step slot for its matrix [lub_ld(N) x (N+1)], padded to a multiple of 16
static size_t ls_mat_stride(int N) { return ((size_t)lub_ld(N) * (N + 1) + 15) / 16 * 16; }

// Integer block of the lock-step work area, behind the slots' floating-point arrays
static void ls_carve_ints(LsArgs& la, char* p, int S) {
    int* ip = reinterpret_cast<int*>(p);
    la.act = ip;  ip += 2 * (size_t)S;
    la.flag = ip; ip += S;
    la.itc = ip;  ip += S;
    la.stat = ip; ip += S;
    la.info = ip; ip += S;
    la.nact = ip; ip += 2;
    la.perm = ip;
}

// Batched LU with partial pivoting + solve of the systems [ld x (N+1)] of all active slots
// (ls_panel -> ls_swap_trsm -> ls_update per 32-column panel, ls_backsub).
static int launch_ls_lu(hpf_t* h, const LsArgs& la, int cur, int N, int nwave, cudaStream_t st) {
    const size_t cap = (size_t)h->smem_optin;
    // every kernel of the LU takes (la, cur, N, ...) and runs one CTA per item, at most the resident CTAs
    auto go = [&](auto kernel, int threads, size_t smem, long long items, auto... args) -> int {
        long long ctas = 0;
        const int rc = resident_ctas(h, kernel, threads, smem, "hpf_solve", &ctas);
        if (rc) return rc;
        return launch(h, kernel, {fill_grid(h, ctas, items, false), (unsigned)threads, smem, st}, la, cur, N, args...);
    };
    auto panel = [&](int k0, int left) -> int {
        const int rows = N - k0, nb = rows < LS_NB ? rows : LS_NB;
        // all-register when every row has a thread, else sub-panels of 8 columns; staged in shared memory when it fits
        const size_t want = LS_PANEL_FIXED_BYTES + (size_t)rows * nb * sizeof(double);
        const int staged = want <= cap ? 1 : 0;
        const size_t psm = staged ? want : (size_t)LS_PANEL_FIXED_BYTES;
        const int rc = rows <= 512 ? go(ls_panel_kernel<1, 32>, rows <= 128 ? 128 : rows <= 256 ? 256 : 512, psm, nwave, k0, staged, left)
                     : rows <= 1024 ? go(ls_panel_kernel<2, 8>, 512, psm, nwave, k0, staged, left)
                                    : go(ls_panel_kernel<4, 8>, 512, psm, nwave, k0, staged, left);
        if (rc) return rc;
        g_ls_timer.mark(4);
        return HPF_OK;
    };
    auto swap_trsm = [&](int k0, int pair) -> int {
        const int nb = (N - k0) < LS_NB ? (N - k0) : LS_NB, cr = k0 + nb;
        const int nchunk = (N + 1 - cr + LS_ST - 1) / LS_ST;
        const int rc = go(ls_swap_trsm_kernel, LS_ST, 0, (long long)nwave * nchunk, k0, pair);
        if (rc) return rc;
        g_ls_timer.mark(5);
        return HPF_OK;
    };
    auto update = [&](int K, int kb, int rlo, int clo, int chi) -> int {
        if (rlo >= N || clo > chi) return HPF_OK;
        auto tiles = [&](auto kernel, int TR, int TC, int NT) -> int {
            const size_t usm = ((size_t)K * (TR + 4) + (size_t)TC * (K + 4)) * sizeof(double);
            const long long ntr = (N - rlo + TR - 1) / TR;          // (strips: row tiles of the matrices)
            return go(kernel, NT, usm, (long long)nwave * ntr, kb, rlo, clo, chi);
        };
        const int rc = K == 64 ? tiles(ls_update_kernel<64, 64, 64, 128, 3>, 64, 64, 128)
                               : tiles(ls_update_kernel<32, 128, 128, 256, 2>, 128, 128, 256);
        if (rc) return rc;
        g_ls_timer.mark(6);
        return HPF_OK;
    };
    int rc;
    for (int k0 = 0; k0 < N;) {
        const int rows = N - k0, nb = rows < LS_NB ? rows : LS_NB, cr = k0 + nb;
        const bool pair = nb == LS_NB && N - cr >= LS_NB;
        if ((rc = panel(k0, 0))) return rc;
        if ((rc = swap_trsm(k0, 0))) return rc;
        if (!pair) {
            if ((rc = update(32, k0, cr, cr, N))) return rc;
            k0 = cr;
            continue;
        }
        // pair of panels: the first one is applied to the second one's 32 columns only; after the second
        // one is factored (its interchanges also move the first one's L21) and its pivot rows have taken
        // the first one's contribution (ls_swap_trsm, pair), the rest takes both in ONE rank-64 pass
        const int k1 = cr, c2 = k1 + LS_NB;
        if ((rc = update(32, k0, k1, k1, c2 - 1))) return rc;
        if ((rc = panel(k1, LS_NB))) return rc;
        if ((rc = swap_trsm(k1, 1))) return rc;
        if ((rc = update(64, k0, c2, c2, N))) return rc;
        k0 = c2;
    }
    if ((rc = go(ls_backsub_kernel, 256, 0, nwave))) return rc;
    g_ls_timer.mark(7);
    return HPF_OK;
}

// Grow-only work area of the lock-step kernels: room for min(B, budget / per_slot) slots; -> slots
static int ensure_ls(hpf_t* h, size_t per_slot, int B, int* slots, const char* who) {
    size_t have = h->d_ls.bytes > 4096 ? (h->d_ls.bytes - 4096) / per_slot : 0;
    if (have < (size_t)B) {
        size_t budget = h->ls_budget;
        if (!budget) {
            size_t fr = 0, tot = 0;
            CK(cudaMemGetInfo(&fr, &tot));
            budget = (size_t)(0.4 * (double)(fr + h->d_ls.bytes));
            if (budget > ((size_t)64 << 30)) budget = (size_t)64 << 30;
        }
        size_t want = budget / per_slot;
        if (want > (size_t)B) want = (size_t)B;
        if (want < 1) want = 1;
        if (want > have) {
            const int rc = grow(h, h->d_ls, per_slot * want + 4096, who);
            if (rc) return rc;
            have = want;
        }
    }
    *slots = (int)(have < (size_t)B ? have : (size_t)B);
    return HPF_OK;
}

// hpf_lu_solve for systems beyond shared memory through the batched LU (all matrices panel by panel)
static int lu_solve_batched(hpf_t* h, int N, int B, const double* J, size_t stride, const double* f, double* dx,
                            int* info, cudaStream_t st) {
    const size_t mat_stride = ls_mat_stride(N);
    const size_t per_slot = mat_stride * sizeof(double) + (size_t)(LS_PERM_INTS + 8) * sizeof(int);
    int S = 0;
    int rc = ensure_ls(h, per_slot, B, &S, "hpf_lu_solve: lock-step work areas");
    if (rc) return rc;
    LsArgs la;
    memset(&la, 0, sizeof(la));
    la.B = B; la.S = S; la.ldb = lub_ld(N); la.mat_stride = mat_stride;
    char* p = h->d_ls.get();
    la.M = reinterpret_cast<double*>(p); p += mat_stride * sizeof(double) * (size_t)S;
    ls_carve_ints(la, p, S);
    const long long nt = (N + 31) / 32;
    for (int b0 = 0; b0 < B; b0 += S) {
        la.b0 = b0;
        la.nwave = (B - b0 < S) ? B - b0 : S;
        const long long items = (long long)la.nwave * nt * nt, tot = (long long)la.nwave * N;
        if ((rc = launch(h, ls_init_kernel, {(unsigned)(S + 255) / 256, 256, 0, st}, la))) return rc;
        if ((rc = launch(h, ls_lu_load_kernel, {(unsigned)std::min<long long>(items, (long long)h->sm_count * 8), 256, 0, st},
                         la, N, J, stride, f))) return rc;
        if ((rc = launch_ls_lu(h, la, 0, N, la.nwave, st))) return rc;
        if ((rc = launch(h, ls_lu_store_kernel, {(unsigned)std::min<long long>((tot + 255) / 256, (long long)h->sm_count * 8),
                                                 256, 0, st}, la, N, dx, info))) return rc;
    }
    return HPF_OK;
}

// LsArgs of a request's harmonic stage (wN: its w_N), or of its fundamental stage (fund); the
// caller carves the work area and sets the wave.
static LsArgs ls_args(const SolveReq& r, bool fund, const double2* wN) {
    LsArgs la;
    memset(&la, 0, sizeof(la));
    la.B = r.B; la.P = r.P; la.Q = r.Q; la.V_m = r.out.V_m; la.V_a = r.out.V_a; la.status = r.out.status;
    if (fund) {
        // the lock-step rounds read the limits of the stage they run and write its iteration counts and
        // error history through the _h fields: the fundamental stage puts its _f values there
        la.thresh_h = r.thresh_f; la.max_h = r.max_f; la.n_iter_h = r.out.n_iter_f; la.hist_h = r.hist_f;
    } else {
        la.flags = r.flags; la.I_N = r.I_N; la.wN = wN; la.thresh_h = r.thresh_h; la.max_h = r.max_h;
        la.I_inj = r.out.I_inj; la.n_iter_h = r.out.n_iter_h; la.err_h = r.out.err_h; la.hist_h = r.hist_h;
    }
    return la;
}

// fundamental stage of the large networks in lock step (dense Jacobians of order Nf through the batched LU)
static int launch_lockstep_fund(hpf_t* h, const SolveReq& r, cudaStream_t st) {
    const int B = r.B, max_f = r.max_f;
    DevNet nf = devnet(h);
    const int H_full = nf.H, Nf = nf.Nf;
    nf.N = Nf; nf.H = 1; nf.nH = nf.n;
    const size_t mat_stride = ls_mat_stride(Nf);
    const size_t state_stride = (scn_smem_doubles_aligned(nf.n, 1, nf.q, Nf) + 15) / 16 * 16;
    const size_t per_slot = (mat_stride + state_stride) * sizeof(double) + (size_t)(LS_PERM_INTS + 8) * sizeof(int);
    int S = 0;
    int rc = ensure_ls(h, per_slot, B, &S, "hpf_solve: lock-step work areas");
    if (rc) return rc;
    LsArgs la = ls_args(r, true, nullptr);
    la.S = S; la.ldb = lub_ld(Nf); la.mat_stride = mat_stride; la.state_stride = state_stride;
    {
        char* p = h->d_ls.get();
        la.M = reinterpret_cast<double*>(p);      p += mat_stride * sizeof(double) * (size_t)S;
        la.state = reinterpret_cast<double*>(p);  p += state_stride * sizeof(double) * (size_t)S;
        ls_carve_ints(la, p, S);
    }
    long long c_mis = 0, c_jac = 0;
    if ((rc = resident_ctas(h, ls_fund_mismatch_kernel, 256, 0, "hpf_solve", &c_mis))) return rc;
    if ((rc = resident_ctas(h, ls_fund_jac_kernel, 256, 0, "hpf_solve", &c_jac))) return rc;
    const unsigned g_mis = fill_grid(h, c_mis, S, false), g_jac = fill_grid(h, c_jac, S, false);
    g_ls_timer.on = getenv("HPF_LS_TIMING") != nullptr && !stream_capturing(st);
    g_ls_timer.st = st;
    for (int b0 = 0; b0 < B; b0 += S) {
        la.b0 = b0;
        la.nwave = (B - b0 < S) ? B - b0 : S;
        if ((rc = launch(h, ls_init_kernel, {(unsigned)(S + 255) / 256, 256, 0, st}, la))) return rc;
        g_ls_timer.mark(0);
        for (int it = 0; it <= max_f; ++it) {
            const int cur = it & 1, nxt = cur ^ 1;
            if ((rc = launch(h, ls_fund_mismatch_kernel, {g_mis, 256, 0, st}, nf, la, cur, it == 0))) return rc;
            if ((rc = launch(h, ls_compact_kernel, {1, 1024, 0, st}, la, cur))) return rc;
            g_ls_timer.mark(1);
            if (it == max_f) break;
            if ((rc = launch(h, ls_fund_jac_kernel, {g_jac, 256, 0, st}, nf, la, nxt))) return rc;
            g_ls_timer.mark(3);
            if ((rc = launch_ls_lu(h, la, nxt, Nf, la.nwave, st))) return rc;
        }
    }
    if (H_full > 1 && (rc = flat_start_harmonics(h, nf.n, H_full, B, r.out.V_m, r.out.V_a, st))) return rc;
    g_ls_timer.report("fundamental stage");
    g_ls_timer.on = false;
    return HPF_OK;
}

static int launch_lockstep(hpf_t* h, const DevNet& net, const StructNet& sn, const SolveReq& r, const double2* wN,
                           cudaStream_t st) {
    const int nx = sn.nx, nZ = sn.nZ, m = net.m, q = net.q;
    const size_t mat_stride = ls_mat_stride(nx);
    const size_t state_stride = (scn_smem_doubles_aligned(net.n, net.H, net.q, net.N) + 15) / 16 * 16;
    const size_t per_slot = (mat_stride + state_stride) * sizeof(double) + ((size_t)m + nZ + q) * sizeof(double2) +
                            (size_t)(LS_PERM_INTS + 8) * sizeof(int);
    // slots: the whole batch when it fits the memory budget, else waves
    int S = 0;
    int rc = ensure_ls(h, per_slot, r.B, &S, "hpf_solve: lock-step work areas");
    if (rc) return rc;
    LsArgs la = ls_args(r, false, wN);
    la.S = S;
    {
        char* p = h->d_ls.get();
        la.M = reinterpret_cast<double*>(p);      p += mat_stride * sizeof(double) * (size_t)S;
        la.state = reinterpret_cast<double*>(p);  p += state_stride * sizeof(double) * (size_t)S;
        la.X = reinterpret_cast<double2*>(p);     p += (size_t)m * S * sizeof(double2);
        la.GX = reinterpret_cast<double2*>(p);    p += (size_t)nZ * S * sizeof(double2);
        la.U0 = reinterpret_cast<double2*>(p);    p += (size_t)q * S * sizeof(double2);
        ls_carve_ints(la, p, S);
    }
    la.mat_stride = mat_stride; la.state_stride = state_stride; la.ldb = lub_ld(nx);
    long long c_mis = 0, c_bor = 0;
    if ((rc = resident_ctas(h, ls_mismatch_kernel, 256, 0, "hpf_solve", &c_mis))) return rc;
    if ((rc = resident_ctas(h, ls_border_kernel, 256, 0, "hpf_solve", &c_bor))) return rc;
    const long long btiles = (long long)((m - 1 + 31) / 32) * ((nx + 1 + 31) / 32);
    const unsigned g_mis = fill_grid(h, c_mis, S, false), g_bor = fill_grid(h, c_bor, (long long)S * btiles, false);
    const unsigned g_el = (unsigned)std::min<long long>(((long long)S * m + 255) / 256, (long long)h->sm_count * 8);
    g_ls_timer.on = getenv("HPF_LS_TIMING") != nullptr && !stream_capturing(st);
    g_ls_timer.st = st;
    for (int b0 = 0; b0 < r.B; b0 += S) {
        la.b0 = b0;
        la.nwave = (r.B - b0 < S) ? r.B - b0 : S;
        if ((rc = launch(h, ls_init_kernel, {(unsigned)(S + 255) / 256, 256, 0, st}, la))) return rc;
        g_ls_timer.mark(0);
        for (int it = 0; it <= r.max_h; ++it) {
            const int cur = it & 1, nxt = cur ^ 1;
            if ((rc = launch(h, ls_mismatch_kernel, {g_mis, 256, 0, st}, net, sn, la, cur, it == 0))) return rc;
            if ((rc = launch(h, ls_compact_kernel, {1, 1024, 0, st}, la, cur))) return rc;
            g_ls_timer.mark(1);
            if (it == r.max_h) break;
            if ((rc = launch(h, ls_pack_vf_kernel, {g_el, 256, 0, st}, net, la, nxt))) return rc;
            if (q > 0 && (rc = launch_zgemm(h, q, la.nwave, m, sn.G, (size_t)m, la.X, (size_t)S, la.U0, (size_t)S, st, false,
                                            la.nact + nxt))) return rc;
            g_ls_timer.mark(2);
            if ((rc = launch(h, ls_border_kernel, {g_bor, 256, 0, st}, net, sn, la, nxt))) return rc;
            g_ls_timer.mark(3);
            if ((rc = launch_ls_lu(h, la, nxt, nx, la.nwave, st))) return rc;
            if ((rc = launch(h, ls_uf_kernel, {g_el, 256, 0, st}, net, sn, la, nxt))) return rc;
            if ((rc = launch_zgemm(h, nZ, la.nwave, m, sn.G, (size_t)m, la.X, (size_t)S, la.GX, (size_t)S, st, false,
                                   la.nact + nxt))) return rc;
            g_ls_timer.mark(8);
        }
    }
    g_ls_timer.report("harmonic stage");
    g_ls_timer.on = false;
    return HPF_OK;
}

static FundTileArgs fund_tile_args(const SolveReq& r) {
    FundTileArgs fa;
    fa.B = r.B; fa.P = r.P; fa.Q = r.Q; fa.thresh_f = r.thresh_f; fa.max_f = r.max_f;
    fa.V_m = r.out.V_m; fa.V_a = r.out.V_a; fa.n_iter_f = r.out.n_iter_f; fa.status = r.out.status; fa.hist_f = r.hist_f;
    return fa;
}

// HarmTileArgs of a request's harmonic stage (wN: its w_N).  With dx_out, one Newton step of the
// iterate in r.out instead (hpf_newton_step): the update goes to dx_out, and there is no work queue
// and no lane servicing.
static HarmTileArgs harm_args(const hpf_t* h, const SolveReq& r, const double2* wN, double* dx_out = nullptr) {
    const bool step = dx_out != nullptr;
    HarmTileArgs ha;
    ha.B = r.B; ha.flags = r.flags; ha.step_only = step ? 1 : 0; ha.P = r.P; ha.Q = r.Q; ha.I_N = r.I_N; ha.wN = wN;
    ha.thresh_h = r.thresh_h; ha.max_h = r.max_h; ha.V_m = r.out.V_m; ha.V_a = r.out.V_a; ha.I_inj = r.out.I_inj;
    ha.n_iter_h = r.out.n_iter_h; ha.status = r.out.status; ha.err_h = r.out.err_h; ha.hist_h = r.hist_h;
    ha.work_counter = step ? nullptr : h->d_counter.get() + r.slot;
    ha.dx_out = dx_out; ha.gstate = nullptr; ha.gstate_stride = 0; ha.lub_doubles = 0;
    ha.epoch = step ? 1 : HPF_HW_SERVICE_EPOCH;
    return ha;
}

static int solve_structured(hpf_t* h, const SolveReq& r, cudaStream_t st) {
    const DevNet net = devnet(h);
    const StructNet sn = structnet(h);
    const int B = r.B;
    int* const counter = h->d_counter.get() + r.slot;
    // error histories: the unused tail is NaN (all-ones bytes are a quiet NaN)
    if (r.hist_f) CK(cudaMemsetAsync(r.hist_f, 0xff, (size_t)(r.max_f + 1) * B * sizeof(double), st));
    if (r.hist_h) CK(cudaMemsetAsync(r.hist_h, 0xff, (size_t)(r.max_h + 1) * B * sizeof(double), st));
    CK(cudaMemsetAsync(counter, 0, sizeof(int), st));
    if (h->profiling) { CK(cudaEventRecord(h->ev[0].get(), st)); }
    // fundamental stage: one lane per scenario (variant 1) or the per-CTA kernel (variant 2)
    if (h->struct_state >= 2) {
        int rc = h->struct_state == 3 && use_lockstep(h, net.Nf, B) ? launch_lockstep_fund(h, r, st)
                                                                     : solve_common(h, 1, fund_stage(r), st);
        if (rc) return rc;
        CK(cudaMemsetAsync(counter, 0, sizeof(int), st));     // solve_common used the counter
    } else {
        const size_t per_warp = fund_tile_doubles_per_warp(net.n, net.Nf) * sizeof(double);
        int warps = 4;
        while (warps > 1 && per_warp * warps > (size_t)h->smem_optin / 2) warps >>= 1;
        const size_t smem = per_warp * warps;
        const FundTileArgs fa = fund_tile_args(r);
        const long long tiles = ((long long)B + HPF_T - 1) / HPF_T;
        const int rcf = with_dims(h->fund_shape, [&](auto d) {
            const auto kernel = fund_tile_kernel<decltype(d)>;
            long long ctas = 0;
            const int rc = resident_ctas(h, kernel, warps * 32, smem, "hpf_solve", &ctas);
            if (rc) return rc;
            return launch(h, kernel, {fill_grid(h, ctas, (tiles + warps - 1) / warps, false), (unsigned)warps * 32, smem, st},
                          net, fa);
        });
        if (rcf) return rcf;
    }
    if (h->profiling) { CK(cudaEventRecord(h->ev[1].get(), st)); }
    // per-scenario constant w_N = A_ZZ^-1 I_N,Z, then the harmonic stage
    {
        const double2* wN = nullptr;
        int rc = launch_wn(h, net, sn, B, r.I_N, r.wN_off, &wN, st);
        if (rc) return rc;
        const bool ls = h->struct_state == 3 && use_lockstep(h, sn.nx, B);
        rc = ls ? launch_lockstep(h, net, sn, r, wN, st) : launch_harm(h, net, sn, harm_args(h, r, wN), true, st);
        if (rc) return rc;
        h->last_path = ls ? 4 : (h->struct_state >= 2 ? h->struct_state : 1);
    }
    if (h->profiling) { CK(cudaEventRecord(h->ev[2].get(), st)); h->ev_valid = 1; }
    return HPF_OK;
}

// Host mirror of Y(h), Y_N and the device map (a few KB).  Y(h) is produced on the device
// (ybus_kernel), so the FIRST call after a network change waits for the stream that built it.
static int host_consts(hpf_t* h) {
    if (h->host_consts_valid) return HPF_OK;
    CK(cudaDeviceSynchronize());
    const size_t ny = (size_t)h->H * h->n * h->n;
    const size_t nyn = (size_t)h->n_dev * (h->coupled ? (size_t)h->H * h->H : (size_t)h->H);
    h->hY.resize(ny);
    h->hYN.resize(nyn);
    h->hdev.resize((size_t)h->q);
    CK(cudaMemcpy(h->hY.data(), h->d_Y.get(), ny * sizeof(double2), cudaMemcpyDeviceToHost));
    if (nyn && h->have_dev) CK(cudaMemcpy(h->hYN.data(), h->d_YN.get(), nyn * sizeof(double2), cudaMemcpyDeviceToHost));
    if (h->q && h->have_dev) CK(cudaMemcpy(h->hdev.data(), h->d_devof.get(), (size_t)h->q * sizeof(int), cudaMemcpyDeviceToHost));
    h->host_consts_valid = true;
    return HPF_OK;
}

template <class D>
static int launch_mismatch_lane(hpf_t* h, const MismatchArgs& a, cudaStream_t st) {
    int rc = host_consts(h);
    if (rc) return rc;
    static_assert(sizeof(LaneConsts<D>) + sizeof(MismatchArgs) <= 32000, "kernel parameter space");
    LaneConsts<D> C;
    memset(&C, 0, sizeof(C));
    for (int t = 0; t < D::H * D::n * D::n; ++t) C.Y[t] = h->hY[t];
    const int per = h->coupled ? D::H * D::H : D::H;
    for (int k = 0; k < D::q; ++k)
        for (int t = 0; t < per; ++t) C.YNk[k * per + t] = h->hYN[(size_t)h->hdev[k] * per + t];
    const int threads = HPF_LANE_THREADS;
    const unsigned grid = (unsigned)(((long long)a.B + threads - 1) / threads);
    return launch(h, h->coupled ? mismatch_lane_kernel<D, true> : mismatch_lane_kernel<D, false>, {grid, threads, 0, st}, C, a);
}

extern "C" {

int hpf_abi_version(void) { return HPF_ABI_VERSION; }

const char* hpf_last_error(const hpf_t* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int hpf_create(hpf_t** out, int device) {
    hpf_t* h = nullptr;
    if (!out) return fail(nullptr, HPF_E_INVALID, "hpf_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, HPF_E_CUDA, std::string("hpf_create: no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(nullptr, HPF_E_INVALID, "hpf_create: bad device ordinal");
    h = new (std::nothrow) hpf_handle();
    if (!h) return fail(nullptr, HPF_E_NOMEM, "hpf_create: out of host memory");
    h->device = device;
    cudaDeviceProp prop;
    DeviceGuard dg_(device);
    e = dg_.err;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        delete h;
        return fail(nullptr, HPF_E_CUDA, std::string("hpf_create: ") + cudaGetErrorString(e));
    }
    if (prop.major < 10) {
        delete h;
        return fail(nullptr, HPF_E_UNSUPPORTED, "hpf_create: this library is built for sm_100a (B200) only");
    }
    if (const char* ev = getenv("HPF_NO_SPECIALISE")) h->no_specialise = atoi(ev) ? 1 : 0;
    if (const char* ev = getenv("HPF_MISMATCH_TILE")) h->mismatch_tile = atoi(ev) ? 1 : 0;
    if (const char* ev = getenv("HPF_STRUCT_VARIANT")) h->force_variant = atoi(ev);
    if (const char* ev = getenv("HPF_LOCKSTEP")) h->lockstep = atoi(ev) ? 1 : 0;
    if (const char* ev = getenv("HPF_LOCKSTEP_GB")) h->ls_budget = (size_t)(atof(ev) > 0 ? atof(ev) * 1073741824.0 : 0);
    if (const char* ev = getenv("HPF_LU_CLASSIC")) h->lu_classic = atoi(ev) ? 1 : 0;
    if (const char* ev = getenv("HPF_GJ_SINGLE_MAX")) h->gj_single_max = atoi(ev);
    if (const char* ev = getenv("HPF_GJ_UNBLOCKED")) h->gj_unblocked = atoi(ev) ? 1 : 0;
    if (const char* ev = getenv("HPF_SETUP")) h->setup_gj = (strcmp(ev, "gj") == 0) ? 1 : 0;
    if (const char* ev = getenv("HPF_WN_KERNEL")) h->wn_kernel = (strcmp(ev, "dmma") == 0) ? 2 : (strcmp(ev, "fma") == 0) ? 1 : 0;
    if (const char* ev = getenv("HPF_HARM_KERNEL")) h->harm_tile_only = (strcmp(ev, "tile") == 0) ? 1 : 0;
    if (const char* ev = getenv("HPF_MAX_CTAS")) h->max_ctas = atoi(ev) > 0 ? atoi(ev) : 0;
    h->sm_count = prop.multiProcessorCount;
    h->smem_optin = (int)prop.sharedMemPerBlockOptin;
    int rc = dev_alloc(nullptr, h->d_counter, HPF_HOST_MAX_CHUNKS * sizeof(int), "hpf_create: work counters");
    if (!rc && (e = create_event(h->ev_last, cudaEventDisableTiming)) != cudaSuccess)
        rc = fail(nullptr, HPF_E_CUDA, std::string("hpf_create: ") + cudaGetErrorString(e));
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return HPF_OK;
}

int hpf_destroy(hpf_t* h) {
    if (!h) return HPF_OK;
    DeviceGuard dg_(h->device);
    cudaDeviceSynchronize();
    delete h;                     // the members release their memory, streams and events on the handle's device
    return HPF_OK;
}

int hpf_set_network(hpf_t* h, int n, int m, int c, int H, const int* harmonics, int L,
                    const int* from_id, const int* to_id, const double* R, const double* X,
                    const double* G, const double* B, const double* X_sh) {
    if (!h) return HPF_E_INVALID;
    if (n < 1 || H < 1 || m < 1 || m > n || c < 1 || c > m || L < 0 || !harmonics || !X_sh ||
        (L > 0 && (!from_id || !to_id || !R || !X || !G || !B)))
        return fail(h, HPF_E_INVALID, "hpf_set_network: invalid dimensions or NULL pointer "
                                      "(need 1 <= c <= m <= n, H >= 1)");
    if (harmonics[0] != 1) return fail(h, HPF_E_INVALID, "hpf_set_network: harmonics[0] must be 1");
    for (int l = 0; l < L; ++l)
        if (from_id[l] < 1 || from_id[l] > n || to_id[l] < 1 || to_id[l] > n)
            return fail(h, HPF_E_INVALID, "hpf_set_network: line endpoint outside 1..n");
    ENTER_DEVICE(h);
    // the previous network goes first: after a failed upload the handle has no network
    h->have_net = h->have_Y = h->have_dev = false;
    invalidate_derived(h, true);
    h->d_tau.reset(); h->d_phase.reset();
    int rc = upload(h, h->d_harm, harmonics, (size_t)H, "hpf_set_network: harmonics");
    if (!rc) rc = upload(h, h->d_from, from_id, (size_t)L, "hpf_set_network: from_id");
    if (!rc) rc = upload(h, h->d_to, to_id, (size_t)L, "hpf_set_network: to_id");
    if (!rc) rc = upload(h, h->d_R, R, (size_t)L, "hpf_set_network: R");
    if (!rc) rc = upload(h, h->d_X, X, (size_t)L, "hpf_set_network: X");
    if (!rc) rc = upload(h, h->d_G, G, (size_t)L, "hpf_set_network: G");
    if (!rc) rc = upload(h, h->d_B, B, (size_t)L, "hpf_set_network: B");
    if (!rc) rc = upload(h, h->d_Xsh, X_sh, (size_t)n, "hpf_set_network: X_sh");
    if (!rc) rc = upload(h, h->d_Y, (const double2*)nullptr, (size_t)H * n * n, "hpf_set_network: Y(h)");
    if (rc) return rc;
    h->n = n; h->m = m; h->c = c; h->H = H; h->q = n - m; h->L = L;
    h->shape = h->fund_shape = 0;
    for (int s = 1; s <= HPF_SHAPES && !h->no_specialise; ++s)
        with_shape(s, [&](auto d) {
            using D = decltype(d);
            if (n == D::n && m == D::m && c == D::c && H == D::H && n - m == D::q) h->shape = s;
            if (n == D::n && c == D::c && !h->fund_shape) h->fund_shape = s;
            return 0;
        });
    h->have_net = true;
    return HPF_OK;
}

int hpf_set_devices(hpf_t* h, int n_dev, int coupled, const double* Y_N, const int* dev_of_nl_bus) {
    if (!h) return HPF_E_INVALID;
    if (!h->have_net) return fail(h, HPF_E_INVALID, "hpf_set_devices: call hpf_set_network first");
    if (h->q > 0 && (n_dev < 1 || !Y_N || !dev_of_nl_bus))
        return fail(h, HPF_E_INVALID, "hpf_set_devices: nonlinear buses present but no device tables");
    for (int k = 0; k < h->q; ++k)
        if (dev_of_nl_bus[k] < 0 || dev_of_nl_bus[k] >= n_dev)
            return fail(h, HPF_E_INVALID, "hpf_set_devices: dev_of_nl_bus entry outside 0..n_dev-1");
    ENTER_DEVICE(h);
    h->have_dev = false;                                     // after a failed upload: no devices
    invalidate_derived(h, false);
    const size_t per = coupled ? (size_t)h->H * h->H : (size_t)h->H;
    int rc = upload(h, h->d_YN, (const double2*)Y_N, per * (size_t)(n_dev > 0 ? n_dev : 0), "hpf_set_devices: Y_N");
    if (!rc) rc = upload(h, h->d_devof, dev_of_nl_bus, (size_t)h->q, "hpf_set_devices: dev_of_nl_bus");
    if (rc) return rc;
    h->n_dev = n_dev;
    h->coupled = coupled ? 1 : 0;
    h->have_dev = true;
    return HPF_OK;
}

int hpf_set_transformers(hpf_t* h, const double* tau, const double* phase_shift_deg) {
    if (!h) return HPF_E_INVALID;
    if (!h->have_net) return fail(h, HPF_E_INVALID, "hpf_set_transformers: call hpf_set_network first");
    if ((tau == nullptr) != (phase_shift_deg == nullptr))
        return fail(h, HPF_E_INVALID, "hpf_set_transformers: give both arrays or neither");
    for (int l = 0; tau && l < h->L; ++l)
        if (!(tau[l] != 0.0)) return fail(h, HPF_E_INVALID, "hpf_set_transformers: tau must be non-zero");
    ENTER_DEVICE(h);
    h->have_Y = false;                                       // Y(h) must be rebuilt
    invalidate_derived(h, false);
    h->d_tau.reset(); h->d_phase.reset();
    if (tau) {
        int rc = upload(h, h->d_tau, tau, (size_t)h->L, "hpf_set_transformers: tau");
        if (!rc) rc = upload(h, h->d_phase, phase_shift_deg, (size_t)h->L, "hpf_set_transformers: phase_shift_deg");
        if (rc) { h->d_tau.reset(); return rc; }             // Y(h) reads both or neither
    }
    return HPF_OK;
}

int hpf_set_y_options(hpf_t* h, int flags) {
    if (!h) return HPF_E_INVALID;
    if (flags & ~(HPF_Y_FIX_SHUNT_INDEX | HPF_Y_SUM_PARALLEL))
        return fail(h, HPF_E_INVALID, "hpf_set_y_options: unknown flag");
    h->y_flags = flags;
    h->have_Y = false;                                       // Y(h) must be rebuilt
    invalidate_derived(h, false);
    return HPF_OK;
}

static int build_Y_impl(hpf_t* h, double* Y_out, void* stream) {
    if (!h) return HPF_E_INVALID;
    if (!h->have_net) return fail(h, HPF_E_INVALID, "hpf_build_Y: call hpf_set_network first");
    ENTER_DEVICE(h);
    cudaStream_t st = (cudaStream_t)stream;
    const int total = h->n * h->H;
    const int rc = launch(h, ybus_kernel, {(unsigned)(total + 127) / 128, 128, 0, st}, h->n, h->H, h->L, h->d_harm.get(),
                          h->d_from.get(), h->d_to.get(), h->d_R.get(), h->d_X.get(), h->d_G.get(), h->d_B.get(),
                          h->d_Xsh.get(), h->d_tau.get(), h->d_phase.get(), h->y_flags, h->d_Y.get());
    if (rc) return rc;
    if (Y_out)
        CK(cudaMemcpyAsync(Y_out, h->d_Y.get(), (size_t)h->H * h->n * h->n * sizeof(double2),
                           cudaMemcpyDeviceToDevice, st));
    h->have_Y = true;
    invalidate_derived(h, true);
    return HPF_OK;
}

int hpf_build_Y(hpf_t* h, double* Y_out, void* stream) {
    return ordered(h, stream, [&] { return build_Y_impl(h, Y_out, stream); });
}

// The copy runs on the legacy stream, which does not wait for non-blocking streams: without the
// wait on ev_last, a solve still in flight on such a stream could read the new Y(h) partway through.
int hpf_set_Y(hpf_t* h, const double* Y) {
    if (!h) return HPF_E_INVALID;
    if (!h->have_net) return fail(h, HPF_E_INVALID, "hpf_set_Y: call hpf_set_network first");
    if (!Y) return fail(h, HPF_E_INVALID, "hpf_set_Y: Y is NULL");
    ENTER_DEVICE(h);
    if (h->last_valid) CK(cudaEventSynchronize(h->ev_last.get()));
    CK(cudaMemcpy(h->d_Y.get(), Y, (size_t)h->H * h->n * h->n * sizeof(double2), cudaMemcpyHostToDevice));
    h->have_Y = true;
    invalidate_derived(h, true);
    return HPF_OK;
}

int hpf_thd(hpf_t* h, int B, const double* V_m, double* thd, void* stream) {
    if (!h) return HPF_E_INVALID;
    if (!h->have_net) return fail(h, HPF_E_INVALID, "hpf_thd: call hpf_set_network first");
    if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_thd: B < 0");
    if (!V_m || !thd) return fail(h, HPF_E_INVALID, "hpf_thd: NULL buffer");
    ENTER_DEVICE(h);
    const size_t total = (size_t)h->n * B;
    return launch(h, thd_kernel, {(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream}, h->n, h->H, h->d_harm.get(),
                  B, V_m, thd);
}

int hpf_bus_currents(hpf_t* h, int B, const double* V_m, const double* V_a, double* I_bus, void* stream) {
    int rc = ready(h, "hpf_bus_currents", false);
    if (rc) return rc;
    if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_bus_currents: B < 0");
    if (!V_m || !V_a || !I_bus) return fail(h, HPF_E_INVALID, "hpf_bus_currents: NULL buffer");
    ENTER_DEVICE(h);
    const DevNet net = devnet(h);
    const size_t total = (size_t)net.nH * B;
    return launch(h, bus_currents_kernel, {(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream}, net, B, V_m, V_a,
                  (double2*)I_bus);
}

int hpf_set_profiling(hpf_t* h, int enabled) {
    if (!h) return HPF_E_INVALID;
    ENTER_DEVICE(h);
    if (enabled)
        for (int i = 0; i < 3; ++i)
            if (!h->ev[i]) CK(create_event(h->ev[i], cudaEventDefault));
    h->profiling = enabled ? 1 : 0;
    h->ev_valid = 0;
    return HPF_OK;
}

int hpf_last_kernel_ms(hpf_t* h, double* ms) {
    if (!h || !ms) return HPF_E_INVALID;
    if (!h->profiling || !h->ev_valid) return fail(h, HPF_E_INVALID, "hpf_last_kernel_ms: no profiled solve");
    CK(cudaEventSynchronize(h->ev[2].get()));
    float a = 0.f, b = 0.f;
    if (h->ev_valid == 1) CK(cudaEventElapsedTime(&a, h->ev[0].get(), h->ev[1].get()));
    CK(cudaEventElapsedTime(&b, h->ev[1].get(), h->ev[2].get()));
    ms[0] = a; ms[1] = b;
    return HPF_OK;
}

int hpf_dim_N(const hpf_t* h) { return (h && h->have_net) ? 2 * h->n * h->H - 1 - h->c : 0; }
int hpf_dim_Nf(const hpf_t* h) { return (h && h->have_net) ? 2 * h->n - 1 - h->c : 0; }
long long hpf_launch_count(const hpf_t* h) { return h ? h->launches : 0; }
int hpf_last_solve_path(const hpf_t* h) { return h ? h->last_path : 0; }

long long hpf_jacobian_stride(const hpf_t* h) {
    if (!h || !h->have_net) return 0;
    const long long N = hpf_dim_N(h);
    return (N * N + 1) & ~1LL;
}

} // extern "C"

// hpf_solve proper, for a checked request with B > 0 on the handle's device; hpf_solve_host calls it
// per chunk with the chunk's scratch slot.
static int solve_dispatch(hpf_t* h, const SolveReq& r, cudaStream_t st) {
    // default strategy: structured Newton step; dense LU when forced or when the network does
    // not admit the structured set-up
    if (!(r.flags & HPF_SOLVE_DENSE)) {
        int rc = ensure_struct(h, st);
        if (rc) return rc;
        if (h->struct_state >= 1) return solve_structured(h, r, st);
    }
    const int rc = solve_common(h, 0, r, st);
    if (rc == HPF_OK) h->last_path = 5;
    return rc;
}

extern "C" {

int hpf_solve(hpf_t* h, int B, const double* P, const double* Q, const double* I_N, double thresh_f,
              int max_iter_f, double thresh_h, int max_iter_h, int flags, double* V_m, double* V_a,
              double* I_inj, int* n_iter_f, int* n_iter_h, double* err_h, int* status,
              double* err_hist_f, double* err_hist_h, void* stream) {
    SolveReq r;
    r.B = B; r.flags = flags; r.P = P; r.Q = Q; r.I_N = (const double2*)I_N;
    r.thresh_f = thresh_f; r.max_f = max_iter_f; r.thresh_h = thresh_h; r.max_h = max_iter_h;
    r.out.V_m = V_m; r.out.V_a = V_a; r.out.I_inj = (double2*)I_inj;
    r.out.n_iter_f = n_iter_f; r.out.n_iter_h = n_iter_h; r.out.err_h = err_h; r.out.status = status;
    r.hist_f = err_hist_f; r.hist_h = err_hist_h;
    return ordered(h, stream, [&] {
        const int rc = check_request(h, r, 0, "hpf_solve");
        if (rc || B == 0) return rc;
        return solve_dispatch(h, r, (cudaStream_t)stream);
    });
}

int hpf_prepare(hpf_t* h, int B_max, void* stream) {
    int rc = ready(h, "hpf_prepare", true);
    if (rc) return rc;
    if (B_max <= 0) return fail(h, HPF_E_INVALID, "hpf_prepare: B_max <= 0");
    ENTER_DEVICE(h);
    cudaStream_t st = (cudaStream_t)stream;
    // a zero-iteration solve of B_max all-zero scenarios (thresholds above every mismatch) walks exactly
    // the allocation paths of hpf_solve: structured set-up, w_N scratch, LU workspaces, state slabs
    const size_t B = (size_t)B_max, n = h->n, H = h->H, q = h->q;
    const size_t nd = 2 * n * B + 2 * q * H * B + 2 * n * H * B + 2 * q * H * B + B + 2 * B + 8;
    DevPtr<double> buf;
    rc = dev_alloc(h, buf, nd * sizeof(double), "hpf_prepare: scenario buffers");
    if (rc) return rc;
    const cudaError_t e = cudaMemsetAsync(buf.get(), 0, nd * sizeof(double), st);
    double *P = buf.get(), *Q = P + n * B, *IN = Q + n * B, *Vm = IN + 2 * q * H * B, *Va = Vm + n * H * B,
           *Inj = Va + n * H * B, *err = Inj + 2 * q * H * B;
    int* iw = reinterpret_cast<int*>(err + B);
    SolveReq r;
    r.B = B_max; r.P = P; r.Q = Q; r.I_N = q ? (const double2*)IN : nullptr;
    r.thresh_f = 1e300; r.max_f = 1; r.thresh_h = 1e300; r.max_h = 1;
    r.out.V_m = Vm; r.out.V_a = Va; r.out.I_inj = q ? (double2*)Inj : nullptr;
    r.out.n_iter_f = iw; r.out.n_iter_h = iw + B; r.out.err_h = err; r.out.status = iw + 2 * B;
    if (e == cudaSuccess) rc = ordered(h, stream, [&] { return solve_dispatch(h, r, st); });
    const cudaError_t e2 = cudaStreamSynchronize(st);
    if (rc) return rc;
    if (e != cudaSuccess || e2 != cudaSuccess)
        return fail(h, HPF_E_CUDA, std::string("hpf_prepare: ") + cudaGetErrorString(e != cudaSuccess ? e : e2));
    return HPF_OK;
}

int hpf_struct_info(hpf_t* h, int* available, int* nZ, double* pivot_min, double* pivot_max) {
    int rc = ready(h, "hpf_struct_info", true);
    if (rc) return rc;
    ENTER_DEVICE(h);
    rc = ensure_struct(h, nullptr);
    if (rc) return rc;
    if (available) *available = h->struct_state >= 1 ? h->struct_state : 0;
    if (nZ) *nZ = h->n * h->H - h->m;
    if (pivot_min) *pivot_min = h->pivot_min;
    if (pivot_max) *pivot_max = h->pivot_max;
    return HPF_OK;
}

static int newton_step_impl(hpf_t* h, int B, const double* V_m, const double* V_a, const double* P,
                            const double* Q, const double* I_N, double* dx, void* stream) {
    int rc = ready(h, "hpf_newton_step", true);
    if (rc) return rc;
    if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_newton_step: B < 0");
    if (!V_m || !V_a || !P || !Q || !dx || (h->q > 0 && !I_N))
        return fail(h, HPF_E_INVALID, "hpf_newton_step: NULL buffer");
    ENTER_DEVICE(h);
    rc = ensure_struct(h, (cudaStream_t)stream);
    if (rc) return rc;
    if (h->struct_state < 1)
        return fail(h, HPF_E_UNSUPPORTED, "hpf_newton_step: structured strategy not available for this network");
    const DevNet net = devnet(h);
    const StructNet sn = structnet(h);
    SolveReq r;
    r.B = B; r.P = P; r.Q = Q; r.I_N = (const double2*)I_N; r.max_h = 1;
    r.out.V_m = const_cast<double*>(V_m); r.out.V_a = const_cast<double*>(V_a);
    const double2* wN = nullptr;
    rc = launch_wn(h, net, sn, B, r.I_N, 0, &wN, (cudaStream_t)stream);
    if (rc) return rc;
    return launch_harm(h, net, sn, harm_args(h, r, wN, dx), false, (cudaStream_t)stream);
}

int hpf_newton_step(hpf_t* h, int B, const double* V_m, const double* V_a, const double* P,
                    const double* Q, const double* I_N, double* dx, void* stream) {
    return ordered(h, stream, [&] { return newton_step_impl(h, B, V_m, V_a, P, Q, I_N, dx, stream); });
}

int hpf_norton_wn(hpf_t* h, int B, const double* I_N, double* wN, void* stream) {
    return ordered(h, stream, [&] {
        int rc = ready(h, "hpf_norton_wn", true);
        if (rc) return rc;
        if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_norton_wn: B < 0");
        if (!wN || (h->q > 0 && !I_N)) return fail(h, HPF_E_INVALID, "hpf_norton_wn: NULL buffer");
        ENTER_DEVICE(h);
        rc = ensure_struct(h, (cudaStream_t)stream);
        if (rc) return rc;
        if (h->struct_state < 1)
            return fail(h, HPF_E_UNSUPPORTED, "hpf_norton_wn: structured strategy not available for this network");
        const DevNet net = devnet(h);
        const StructNet sn = structnet(h);
        const double2* w = nullptr;
        rc = launch_wn(h, net, sn, B, (const double2*)I_N, 0, &w, (cudaStream_t)stream);
        if (rc) return rc;
        CK(cudaMemcpyAsync(wN, w, (size_t)sn.nZ * B * sizeof(double2), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        return HPF_OK;
    });
}

int hpf_ne_extract(hpf_t* h, int D, int N, const double* Vf, const double* Vh, const double* I_f,
                   const double* I_h, double* Y_N_c, double* I_N_c, double* Y_N_uc, double* I_N_uc,
                   int* info, void* stream) {
    if (!h) return HPF_E_INVALID;
    if (D <= 0) return D == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_ne_extract: D < 0");
    if (N < 2) return fail(h, HPF_E_INVALID, "hpf_ne_extract: at least 2 frequencies needed");
    if (!Vf || !Vh || !I_f || !I_h || !Y_N_c || !I_N_c || !Y_N_uc || !I_N_uc || !info)
        return fail(h, HPF_E_INVALID, "hpf_ne_extract: NULL buffer");
    ENTER_DEVICE(h);
    const size_t smem = ne_extract_smem_bytes(N);
    long long ctas = 0;
    const int rc = resident_ctas(h, ne_extract_kernel, 256, smem, "hpf_ne_extract", &ctas);
    if (rc) return rc;
    NeExtractArgs a;
    a.D = D; a.N = N;
    a.Vf = (const double2*)Vf; a.Vh = (const double2*)Vh; a.I_f = (const double2*)I_f; a.I_h = (const double2*)I_h;
    a.Y_N_c = (double2*)Y_N_c; a.I_N_c = (double2*)I_N_c; a.Y_N_uc = (double2*)Y_N_uc; a.I_N_uc = (double2*)I_N_uc;
    a.info = info;
    return launch(h, ne_extract_kernel, {fill_grid(h, ctas, D, false), 256, smem, (cudaStream_t)stream}, a);
}

int hpf_fund_solve(hpf_t* h, int B, const double* P, const double* Q, double thresh_f, int max_iter_f,
                   double* V_m, double* V_a, int* n_iter_f, double* err_f, double* err_hist_f,
                   void* stream) {
    SolveReq r;
    r.B = B; r.P = P; r.Q = Q; r.thresh_f = thresh_f; r.max_f = max_iter_f;
    r.out.V_m = V_m; r.out.V_a = V_a; r.out.n_iter_f = n_iter_f; r.err_f = err_f; r.hist_f = err_hist_f;
    return ordered(h, stream, [&] {
        const int rc = check_request(h, r, 1, "hpf_fund_solve");
        if (rc || B == 0) return rc;
        return solve_common(h, 1, r, (cudaStream_t)stream);
    });
}

} // extern "C"

// ---- batch statistics -------------------------------------------------------------------
// Argument checks shared by hpf_batch_stats and hpf_solve_host_stats (h != NULL).
static int check_stats_args(hpf_t* h, int B, int K, const double* quantiles, const int* counts,
                            const double* stats, const char* who) {
    const std::string w(who);
    if (!h->have_net) return fail(h, HPF_E_INVALID, w + ": call hpf_set_network first");
    if (B < 0) return fail(h, HPF_E_INVALID, w + ": B < 0");
    if (K < 0 || K > HPF_STATS_MAX_Q)
        return fail(h, HPF_E_INVALID, w + ": K = " + std::to_string(K) + " outside [0, HPF_STATS_MAX_Q]");
    if ((K > 0 && !quantiles) || !counts || !stats) return fail(h, HPF_E_INVALID, w + ": NULL buffer");
    for (int k = 0; k < K; ++k)
        if (!(quantiles[k] >= 0.0 && quantiles[k] <= 1.0))
            return fail(h, HPF_E_INVALID, w + ": quantile " + std::to_string(k) + " is NaN or outside [0, 1]");
    return HPF_OK;
}

// CTAs per row (the cluster size of stats_kernel): about four CTAs per SM over all rows, at most 8 (the
// portable cluster size), at least 2,048 scenarios per CTA.  The reduction order follows from it, so it
// depends on (R, B) and the device only.
static int stats_cluster(const hpf_t* h, int R, int B) {
    int cs = (4 * h->sm_count + R - 1) / R;
    if (cs > 8) cs = 8;
    const int by_b = (B + 2047) / 2048;
    if (cs > by_b) cs = by_b;
    return cs < 1 ? 1 : cs;
}

// THD rows of V_m into `thd` ([2, n, B] scratch, thd_kernel as in hpf_thd), then one cluster of
// stats_kernel per row.  Checked arguments; all pointers device memory except `quantiles`.
static int launch_batch_stats(hpf_t* h, int B, const double* V_m, const int* status, int K, const double* quantiles,
                              const double* limits, int* counts, double* stats, double* thd, cudaStream_t st) {
    const int n = h->n, nH = n * h->H, R = nH + 2 * n;
    if (B > 0) {
        const size_t total = (size_t)n * B;
        const int rc = launch(h, thd_kernel, {(unsigned)((total + 255) / 256), 256, 0, st}, n, h->H, h->d_harm.get(), B, V_m, thd);
        if (rc) return rc;
    }
    StatsArgs a;
    a.B = B; a.R = R; a.nH = nH; a.K = K;
    a.V_m = V_m; a.thd = thd; a.status = status; a.limits = limits; a.counts = counts; a.stats = stats;
    for (int k = 0; k < HPF_STATS_MAX_Q; ++k) a.q[k] = k < K ? quantiles[k] : 0.0;
    const int cs = stats_cluster(h, R, B);
    return launch(h, stats_kernel, {(unsigned)(cs * R), HPF_STATS_THREADS, stats_smem_bytes(K), st, cs}, a);
}

extern "C" {

int hpf_batch_stats(hpf_t* h, int B, const double* V_m, const int* status, int K, const double* quantiles,
                    const double* limits, int* status_counts, double* stats, void* stream) {
    if (!h) return HPF_E_INVALID;
    int rc = check_stats_args(h, B, K, quantiles, status_counts, stats, "hpf_batch_stats");
    if (rc) return rc;
    if (B > 0 && !V_m) return fail(h, HPF_E_INVALID, "hpf_batch_stats: NULL V_m");
    return ordered(h, stream, [&] {
        const int r = grow(h, h->d_stats, (size_t)2 * h->n * B * sizeof(double), "hpf_batch_stats: THD rows");
        if (r) return r;
        return launch_batch_stats(h, B, V_m, status, K, quantiles, limits, status_counts, stats, h->d_stats.get(),
                                  (cudaStream_t)stream);
    });
}

} // extern "C"

// Chunk plan of hpf_solve_host: boundaries cb[0..nchunk] (multiples of 32 scenarios except the end) and
// the number of compute streams the chunks rotate over.  $HPF_HOST_PLAN = comma-separated chunk sizes
// (the last size repeats until the batch is covered; at most HPF_HOST_MAX_CHUNKS chunks, the last one
// takes the rest), else HPF_HOST_RAMP for batches of at least HPF_HOST_RAMP_MIN_B, else one chunk;
// $HPF_HOST_STREAMS = 1..4 compute streams.
static int host_chunk_plan(size_t Bs, size_t* cb, int* streams) {
    static const size_t ramp_default[] = {HPF_HOST_RAMP};
    size_t sizes[HPF_HOST_MAX_CHUNKS];
    int ns = 0;
    if (const char* ev = getenv("HPF_HOST_PLAN")) {
        for (const char* p = ev; *p && ns < HPF_HOST_MAX_CHUNKS;) {
            char* end = nullptr;
            const long v = strtol(p, &end, 10);
            if (end == p) break;
            if (v > 0) sizes[ns++] = (size_t)v;
            p = (*end == ',') ? end + 1 : end;
            if (*end != ',') break;
        }
    }
    if (ns == 0 && Bs >= HPF_HOST_RAMP_MIN_B)
        for (size_t i = 0; i < sizeof(ramp_default) / sizeof(ramp_default[0]); ++i) sizes[ns++] = ramp_default[i];
    if (ns == 0) { sizes[0] = Bs; ns = 1; }
    int k = 0;
    size_t b = 0;
    cb[0] = 0;
    while (b < Bs) {
        size_t sz = (sizes[k < ns ? k : ns - 1] + 31) / 32 * 32;
        if (k == HPF_HOST_MAX_CHUNKS - 1 || b + sz > Bs) sz = Bs - b;
        b += sz;
        cb[++k] = b;
    }
    int st = HPF_HOST_STREAMS_DEFAULT;
    if (const char* ev = getenv("HPF_HOST_STREAMS")) { const int v = atoi(ev); if (v >= 1 && v <= 4) st = v; }
    *streams = st;
    return k;
}

// What hpf_solve_host_stats asks of the host solve path: statistics instead of phasors (host buffers).
struct StatsOut {
    int K = 0;
    const double *quantiles = nullptr, *limits = nullptr;
    int* counts = nullptr;
    double* stats = nullptr;
};

// hpf_solve_host: `hr` holds host arrays; keep, when given, receives device copies of the results.
// With `so` (hpf_solve_host_stats) no phasor goes back: each chunk's V_m is kept in a whole-batch device
// array, and after the last chunk the copy-out stream reduces it with the whole-batch status array
// (launch_batch_stats) and copies back the statistics and the flag arrays that hr asks for.
static int solve_host_impl(hpf_t* h, const SolveReq& hr, const BatchOut* keep, const StatsOut* so = nullptr) {
    int rc = check_request(h, hr, so ? 2 : 0, so ? "hpf_solve_host_stats" : "hpf_solve_host");
    if (rc || hr.B == 0) return rc;
    ENTER_DEVICE(h);
    // Pipelined in chunks of scenarios: while chunk k is being solved, chunk k+1 is copied in and
    // the results of chunk k-1 are copied out (PCIe is full duplex); consecutive chunks rotate over
    // the compute streams so that the long-iteration tail of one chunk overlaps the start of the
    // next.  The copy-out of the results is the floor of the call (1.24 ms for 65,536 net3 scenarios;
    // 1 chunk 2.30 ms, 8 equal chunks on two compute streams 1.65 ms, the growing plan 1.61 ms:
    // profiles/r2_e2e_chunk_plans.txt), so the plan starts with a SMALL chunk - the copy-out stream
    // gets its first results after one short solve - and grows the chunks while the copy engine is
    // busy: fewer, larger copies and solves later on (host_chunk_plan).
    // The host arrays are batch-innermost [rows, B]; a chunk is a column block, moved with 2-D
    // copies into compact [rows, Bc] device arrays (pinned host memory makes them asynchronous).
    const size_t n = h->n, H = h->H, q = h->q, Bs = (size_t)hr.B;
    size_t cb[HPF_HOST_MAX_CHUNKS + 1];
    int ncs = 2;
    const int nchunk = host_chunk_plan(Bs, cb, &ncs);
    // per scenario and chunk (compact): P, Q [n] | I_N [2qH] | V_m, V_a [nH] | I_inj [2qH]; chunk k lives
    // at per_scn * cb[k] (chunk starts are multiples of 32 scenarios).  err_h and the three flag arrays
    // are one row per scenario: they sit behind the chunks as whole-batch arrays [Bp] and go back with
    // ONE copy each after the last chunk (a copy costs ~3 us of the copy-out stream whatever its size).
    const size_t per_scn = 2 * n + 2 * q * H + 2 * n * H + 2 * q * H;
    const size_t Bp = (Bs + 3) / 4 * 4;
    const size_t nd = per_scn * Bs + Bp + 3 * (Bp / 2);
    rc = grow(h, h->d_io, nd * sizeof(double), "hpf_solve_host: staging buffers");
    if (rc) return rc;
    // statistics: whole-batch V_m [H, n, B] | THD rows [2, n, B] | limits [R] | stats [5 + K, R] | counts
    const size_t R = n * H + 2 * n;
    if (so) {
        rc = grow(h, h->d_stats, ((H + 2) * n * Bs + R + (5 + so->K) * R + 2) * sizeof(double),
                  "hpf_solve_host_stats: statistics scratch");
        if (rc) return rc;
    }
    double *const dVfull = h->d_stats.get(), *const dThd = dVfull + H * n * Bs, *const dLim = dThd + 2 * n * Bs,
           *const dStats = dLim + R;
    int* const dCounts = so ? reinterpret_cast<int*>(dStats + (5 + so->K) * R) : nullptr;
    BatchOut keep_vm;                    // the statistics keep V_m only: the flag arrays already sit in d_io
    keep_vm.V_m = dVfull;
    if (so) keep = &keep_vm;
    if (!h->st_io[0]) {
        // all or nothing: the handle takes the streams and events only when every one of them exists
        Stream st[6];
        Event ev[3 * HPF_HOST_MAX_CHUNKS];
        for (auto& s : st) {
            cudaStream_t raw = nullptr;
            CK(cudaStreamCreateWithFlags(&raw, cudaStreamNonBlocking));
            s.reset(raw);
        }
        for (auto& e : ev) CK(create_event(e, cudaEventDisableTiming));
        for (int i = 0; i < 6; ++i) h->st_io[i] = std::move(st[i]);
        for (int i = 0; i < 3 * HPF_HOST_MAX_CHUNKS; ++i) h->ev_io[i] = std::move(ev[i]);
    }
    cudaStream_t s_in = h->st_io[0].get(), s_out = h->st_io[2].get();
    const int cmp_stream[4] = {1, 3, 4, 5};
    // ordered after the handle's previous kernel sequence like every other entry point (the copy-in
    // overwrites the staging buffers, the solves share the handle's scratch)
    if (h->last_valid)
        for (auto& s : h->st_io) CK(cudaStreamWaitEvent(s.get(), h->ev_last.get(), 0));
    // several compute streams only where concurrent solves share no scratch (tile variant)
    rc = ensure_struct(h, h->st_io[1].get());
    if (rc) return rc;
    const bool dual = (h->struct_state == 1) && nchunk > 1 && ncs > 1;
    const size_t wN_rows = (size_t)(h->n * h->H - h->m);
    if (dual) {
        // reserve the w_N scratch of all chunks up front (no reallocation while chunks are in flight)
        rc = grow(h, h->d_wN, wN_rows * Bs * sizeof(double2), "hpf_solve_host: w_N scratch");
        if (rc) return rc;
    }
    auto cp2d = [&](void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows,
                    cudaMemcpyKind kind, cudaStream_t st) {
        return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, rows, kind, st);
    };
    rc = HPF_OK;
    cudaError_t e = cudaSuccess;
    double* const dErr_all = h->d_io.get() + per_scn * Bs;
    int* const di_all = reinterpret_cast<int*>(dErr_all + Bp);
    // $HPF_HOST_TIMELINE: per-chunk completion times of copy-in, solve and copy-out on stderr
    const bool tl = getenv("HPF_HOST_TIMELINE") != nullptr;
    Event tle[3 * HPF_HOST_MAX_CHUNKS + 1];
    if (tl) {
        for (auto& ev : tle) create_event(ev, cudaEventDefault);
        cudaEventRecord(tle[3 * HPF_HOST_MAX_CHUNKS].get(), s_in);
    }
    const BatchOut& ho = hr.out;
    for (int k = 0; k < nchunk && !rc; ++k) {
        const size_t b0 = cb[k], Bc = cb[k + 1] - cb[k];
        double* d = h->d_io.get() + per_scn * b0;
        double *dP = d, *dQ = dP + n * Bc, *dI = dQ + n * Bc, *dVm = dI + 2 * q * H * Bc, *dVa = dVm + n * H * Bc,
               *dInj = dVa + n * H * Bc, *dErr = dErr_all + b0;
        int *di_f = di_all + b0, *di_h = di_all + Bp + b0, *di_s = di_all + 2 * Bp + b0;
        const size_t w8 = Bc * sizeof(double), w16 = Bc * 2 * sizeof(double);
        const size_t p8 = Bs * sizeof(double), p16 = Bs * 2 * sizeof(double);
        e = cp2d(dP, w8, hr.P + b0, p8, w8, n, cudaMemcpyHostToDevice, s_in);
        if (e == cudaSuccess) e = cp2d(dQ, w8, hr.Q + b0, p8, w8, n, cudaMemcpyHostToDevice, s_in);
        if (e == cudaSuccess && q)
            e = cp2d(dI, w16, hr.I_N + b0, p16, w16, q * H, cudaMemcpyHostToDevice, s_in);
        cudaStream_t s_cmp = h->st_io[dual ? cmp_stream[k % ncs] : 1].get();
        if (e == cudaSuccess) e = cudaEventRecord(h->ev_io[k].get(), s_in);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s_cmp, h->ev_io[k].get(), 0);
        if (e != cudaSuccess) break;
        if (tl) cudaEventRecord(tle[3 * k].get(), s_in);
        SolveReq c = hr;          // the same thresholds and limits on the chunk's device buffers
        c.B = (int)Bc; c.P = dP; c.Q = dQ; c.I_N = (const double2*)dI;
        c.out.V_m = dVm; c.out.V_a = dVa; c.out.I_inj = ho.I_inj ? (double2*)dInj : nullptr;
        c.out.n_iter_f = di_f; c.out.n_iter_h = di_h; c.out.err_h = dErr; c.out.status = di_s;
        c.slot = dual ? k : 0;
        c.wN_off = dual ? wN_rows * b0 : 0;
        rc = solve_dispatch(h, c, s_cmp);
        if (rc) break;
        e = cudaEventRecord(h->ev_io[HPF_HOST_MAX_CHUNKS + k].get(), s_cmp);
        if (tl) cudaEventRecord(tle[3 * k + 1].get(), s_cmp);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(s_out, h->ev_io[HPF_HOST_MAX_CHUNKS + k].get(), 0);
        if (e == cudaSuccess && !so) e = cp2d(ho.V_m + b0, p8, dVm, w8, w8, n * H, cudaMemcpyDeviceToHost, s_out);
        if (e == cudaSuccess && !so) e = cp2d(ho.V_a + b0, p8, dVa, w8, w8, n * H, cudaMemcpyDeviceToHost, s_out);
        if (e == cudaSuccess && ho.I_inj && q)
            e = cp2d(ho.I_inj + b0, p16, dInj, w16, w16, q * H, cudaMemcpyDeviceToHost, s_out);
        if (e == cudaSuccess && k == nchunk - 1) {       // s_out has waited for every chunk by now
            // (the statistics host solve copies back only the flag arrays it is given)
            if (ho.err_h) e = cudaMemcpyAsync(ho.err_h, dErr_all, Bs * sizeof(double), cudaMemcpyDeviceToHost, s_out);
            if (e == cudaSuccess && ho.n_iter_f) e = cudaMemcpyAsync(ho.n_iter_f, di_all, Bs * sizeof(int), cudaMemcpyDeviceToHost, s_out);
            if (e == cudaSuccess && ho.n_iter_h) e = cudaMemcpyAsync(ho.n_iter_h, di_all + Bp, Bs * sizeof(int), cudaMemcpyDeviceToHost, s_out);
            if (e == cudaSuccess && ho.status) e = cudaMemcpyAsync(ho.status, di_all + 2 * Bp, Bs * sizeof(int), cudaMemcpyDeviceToHost, s_out);
        }
        if (tl) cudaEventRecord(tle[3 * k + 2].get(), s_out);
        if (e == cudaSuccess && keep) {
            // also leave the results on the device in the full [rows, B] layout (device-to-device
            // 2-D copies on the compute stream, ~20 us for the whole batch)
            e = cp2d(keep->V_m + b0, p8, dVm, w8, w8, n * H, cudaMemcpyDeviceToDevice, s_cmp);
            if (e == cudaSuccess && keep->V_a) e = cp2d(keep->V_a + b0, p8, dVa, w8, w8, n * H, cudaMemcpyDeviceToDevice, s_cmp);
            if (e == cudaSuccess && keep->I_inj && ho.I_inj && q)
                e = cp2d(keep->I_inj + b0, p16, dInj, w16, w16, q * H, cudaMemcpyDeviceToDevice, s_cmp);
            if (e == cudaSuccess && keep->err_h) e = cudaMemcpyAsync(keep->err_h + b0, dErr, Bc * sizeof(double), cudaMemcpyDeviceToDevice, s_cmp);
            if (e == cudaSuccess && keep->n_iter_f) e = cudaMemcpyAsync(keep->n_iter_f + b0, di_f, Bc * sizeof(int), cudaMemcpyDeviceToDevice, s_cmp);
            if (e == cudaSuccess && keep->n_iter_h) e = cudaMemcpyAsync(keep->n_iter_h + b0, di_h, Bc * sizeof(int), cudaMemcpyDeviceToDevice, s_cmp);
            if (e == cudaSuccess && keep->status) e = cudaMemcpyAsync(keep->status + b0, di_s, Bc * sizeof(int), cudaMemcpyDeviceToDevice, s_cmp);
        }
        if (e == cudaSuccess && so) {
            // the keep copies run on the compute stream AFTER the chunk's "solved" event: the statistics
            // wait for an event recorded behind them
            e = cudaEventRecord(h->ev_io[2 * HPF_HOST_MAX_CHUNKS + k].get(), s_cmp);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(s_out, h->ev_io[2 * HPF_HOST_MAX_CHUNKS + k].get(), 0);
        }
        if (e != cudaSuccess) break;
    }
    if (!rc && e == cudaSuccess && so) {
        // s_out has waited for every chunk's V_m copy: reduce the whole batch, copy back the results
        if (so->limits) e = cudaMemcpyAsync(dLim, so->limits, R * sizeof(double), cudaMemcpyHostToDevice, s_out);
        if (e == cudaSuccess)
            rc = launch_batch_stats(h, hr.B, dVfull, di_all + 2 * Bp, so->K, so->quantiles, so->limits ? dLim : nullptr,
                                    dCounts, dStats, dThd, s_out);
        if (!rc && e == cudaSuccess)
            e = cudaMemcpyAsync(so->stats, dStats, (5 + so->K) * R * sizeof(double), cudaMemcpyDeviceToHost, s_out);
        if (!rc && e == cudaSuccess) e = cudaMemcpyAsync(so->counts, dCounts, 4 * sizeof(int), cudaMemcpyDeviceToHost, s_out);
    }
    if (!rc && e != cudaSuccess)
        rc = fail(h, HPF_E_CUDA, std::string(so ? "hpf_solve_host_stats: " : "hpf_solve_host: ") + cudaGetErrorString(e));
    for (auto& s : h->st_io) {
        const cudaError_t e2 = cudaStreamSynchronize(s.get());
        if (!rc && e2 != cudaSuccess) rc = fail(h, HPF_E_CUDA, std::string("hpf_solve_host: ") + cudaGetErrorString(e2));
    }
    if (tl) {
        for (int k = 0; k < nchunk && !rc; ++k) {
            float t[3] = {0.f, 0.f, 0.f};
            for (int i = 0; i < 3; ++i) cudaEventElapsedTime(&t[i], tle[3 * HPF_HOST_MAX_CHUNKS].get(), tle[3 * k + i].get());
            fprintf(stderr, "hpf_solve_host chunk %2d [%6zu..%6zu): copy-in done %.3f ms, solve done %.3f ms, copy-out done %.3f ms\n",
                    k, cb[k], cb[k + 1], t[0], t[1], t[2]);
        }
    }
    if (!rc) h->last_valid = false;        // everything this handle issued has completed
    return rc;
}

extern "C" {

int hpf_solve_host(hpf_t* h, int B, const double* P, const double* Q, const double* I_N, double thresh_f,
                   int max_iter_f, double thresh_h, int max_iter_h, double* V_m, double* V_a,
                   double* I_inj, int* n_iter_f, int* n_iter_h, double* err_h, int* status) {
    SolveReq r;
    r.B = B; r.P = P; r.Q = Q; r.I_N = (const double2*)I_N;
    r.thresh_f = thresh_f; r.max_f = max_iter_f; r.thresh_h = thresh_h; r.max_h = max_iter_h;
    r.out.V_m = V_m; r.out.V_a = V_a; r.out.I_inj = (double2*)I_inj;
    r.out.n_iter_f = n_iter_f; r.out.n_iter_h = n_iter_h; r.out.err_h = err_h; r.out.status = status;
    return solve_host_impl(h, r, nullptr);
}

int hpf_solve_host_keep(hpf_t* h, int B, const double* P, const double* Q, const double* I_N, double thresh_f,
                        int max_iter_f, double thresh_h, int max_iter_h, double* V_m, double* V_a,
                        double* I_inj, int* n_iter_f, int* n_iter_h, double* err_h, int* status,
                        double* dV_m, double* dV_a, double* dI_inj, int* dn_iter_f, int* dn_iter_h,
                        double* derr_h, int* dstatus) {
    if (!dV_m || !dV_a || !dn_iter_f || !dn_iter_h || !derr_h || !dstatus)
        return fail(h, HPF_E_INVALID, "hpf_solve_host_keep: NULL device buffer");
    SolveReq r;
    r.B = B; r.P = P; r.Q = Q; r.I_N = (const double2*)I_N;
    r.thresh_f = thresh_f; r.max_f = max_iter_f; r.thresh_h = thresh_h; r.max_h = max_iter_h;
    r.out.V_m = V_m; r.out.V_a = V_a; r.out.I_inj = (double2*)I_inj;
    r.out.n_iter_f = n_iter_f; r.out.n_iter_h = n_iter_h; r.out.err_h = err_h; r.out.status = status;
    BatchOut k;
    k.V_m = dV_m; k.V_a = dV_a; k.I_inj = (double2*)dI_inj; k.err_h = derr_h;
    k.n_iter_f = dn_iter_f; k.n_iter_h = dn_iter_h; k.status = dstatus;
    return solve_host_impl(h, r, &k);
}

int hpf_solve_host_stats(hpf_t* h, int B, const double* P, const double* Q, const double* I_N, double thresh_f,
                         int max_iter_f, double thresh_h, int max_iter_h, int K, const double* quantiles,
                         const double* limits, int* status_counts, double* stats, int* n_iter_f, int* n_iter_h,
                         double* err_h, int* status) {
    if (!h) return HPF_E_INVALID;
    int rc = check_stats_args(h, B, K, quantiles, status_counts, stats, "hpf_solve_host_stats");
    if (rc) return rc;
    SolveReq r;
    r.B = B; r.P = P; r.Q = Q; r.I_N = (const double2*)I_N;
    r.thresh_f = thresh_f; r.max_f = max_iter_f; r.thresh_h = thresh_h; r.max_h = max_iter_h;
    r.out.n_iter_f = n_iter_f; r.out.n_iter_h = n_iter_h; r.out.err_h = err_h; r.out.status = status;
    StatsOut so;
    so.K = K; so.quantiles = quantiles; so.limits = limits; so.counts = status_counts; so.stats = stats;
    rc = solve_host_impl(h, r, nullptr, &so);
    if (rc || B > 0) return rc;
    // an empty batch: no scenario included
    const size_t R = (size_t)h->n * h->H + 2 * h->n;
    for (int i = 0; i < 4; ++i) status_counts[i] = 0;
    for (size_t p = 0; p < (size_t)(5 + K); ++p)
        for (size_t i = 0; i < R; ++i) stats[p * R + i] = p == 4 ? 0.0 : std::numeric_limits<double>::quiet_NaN();
    return HPF_OK;
}

static int mismatch_impl(hpf_t* h, int B, const double* V_m, const double* V_a, const double* P, const double* Q,
                 const double* I_N, double* f, double* err, double* I_inj, void* stream) {
    int rc = ready(h, "hpf_mismatch", true);
    if (rc) return rc;
    if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_mismatch: B < 0");
    if (!V_m || !V_a || !P || !Q || !f || !err || (h->q > 0 && !I_N))
        return fail(h, HPF_E_INVALID, "hpf_mismatch: NULL buffer");
    ENTER_DEVICE(h);
    const DevNet net = devnet(h);
    MismatchArgs a;
    a.B = B; a.V_m = V_m; a.V_a = V_a; a.P = P; a.Q = Q; a.I_N = (const double2*)I_N;
    a.f = f; a.err = err; a.I_inj = (double2*)I_inj;
    const int yn_elems = h->n_dev * (h->coupled ? h->H * h->H : h->H);
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = tile_smem_bytes(net.n, net.H, net.q, net.m, yn_elems);
    if (h->shape && !h->mismatch_tile)
        return with_shape(h->shape, [&](auto d) { return launch_mismatch_lane<decltype(d)>(h, a, st); });
    if (smem <= (size_t)h->smem_optin) {
        // one CTA per 32-scenario tile: the hardware scheduler balances the tail (a persistent
        // grid of occ*SMs CTAs quantises 2048 tiles into 4 rounds of 592, 13 % idle)
        const unsigned tiles = (unsigned)(((long long)B + HPF_TILE - 1) / HPF_TILE);
        return with_dims(h->shape, [&](auto d) {
            return launch(h, mismatch_tile_kernel<decltype(d)>, {tiles, HPF_THREADS, smem, st}, net, a, yn_elems);
        });
    }
    const size_t csmem = scn_smem_bytes(net.n, net.H, net.q, net.N, false);
    long long ctas = 0;
    rc = resident_ctas(h, mismatch_cta_kernel, HPF_THREADS, csmem, "hpf_mismatch", &ctas);
    if (rc) return rc;
    return launch(h, mismatch_cta_kernel, {fill_grid(h, ctas, B, false), HPF_THREADS, csmem, st}, net, a);
}

int hpf_mismatch(hpf_t* h, int B, const double* V_m, const double* V_a, const double* P, const double* Q,
                 const double* I_N, double* f, double* err, double* I_inj, void* stream) {
    return ordered(h, stream, [&] { return mismatch_impl(h, B, V_m, V_a, P, Q, I_N, f, err, I_inj, stream); });
}

static int jacobian_impl(hpf_t* h, int B, const double* V_m, const double* V_a, double* J, void* stream) {
    int rc = ready(h, "hpf_jacobian", true);
    if (rc) return rc;
    if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_jacobian: B < 0");
    if (!V_m || !V_a || !J) return fail(h, HPF_E_INVALID, "hpf_jacobian: NULL buffer");
    if ((reinterpret_cast<uintptr_t>(J) & 15) != 0)
        return fail(h, HPF_E_INVALID, "hpf_jacobian: J must be 16-byte aligned");
    ENTER_DEVICE(h);
    const DevNet net = devnet(h);
    JacobianArgs a;
    a.B = B; a.V_m = V_m; a.V_a = V_a; a.J = J; a.stride = hpf_jacobian_stride(h);
    const size_t smem = jac_smem_bytes(net.n, net.H, net.q, net.N, a.stride);
    const bool in_smem = smem <= (size_t)h->smem_optin;
    const auto kernel = in_smem ? jacobian_kernel : jacobian_gmem_kernel;
    const int threads = in_smem ? HPF_JAC_THREADS : HPF_THREADS;
    const size_t ksmem = in_smem ? smem : scn_smem_bytes(net.n, net.H, net.q, net.N, false);
    long long ctas = 0;
    rc = resident_ctas(h, kernel, threads, ksmem, "hpf_jacobian", &ctas);
    if (rc) return rc;
    return launch(h, kernel, {fill_grid(h, ctas, B, false), (unsigned)threads, ksmem, (cudaStream_t)stream}, net, a);
}

int hpf_jacobian(hpf_t* h, int B, const double* V_m, const double* V_a, double* J, void* stream) {
    return ordered(h, stream, [&] { return jacobian_impl(h, B, V_m, V_a, J, stream); });
}

static int lu_solve_impl(hpf_t* h, int B, const double* J, const double* f, double* dx, int* info, void* stream) {
    int rc = ready(h, "hpf_lu_solve", false);
    if (rc) return rc;
    if (B <= 0) return B == 0 ? HPF_OK : fail(h, HPF_E_INVALID, "hpf_lu_solve: B < 0");
    if (!J || !f || !dx || !info) return fail(h, HPF_E_INVALID, "hpf_lu_solve: NULL buffer");
    ENTER_DEVICE(h);
    const DevNet net = devnet(h);
    LuArgs a;
    a.B = B; a.J = J; a.f = f; a.dx = dx; a.info = info; a.stride = hpf_jacobian_stride(h);
    const LuPlan lu = lu_plan(h, net);
    a.lub_doubles = (int)lu.lubd;
    a.lu_classic = h->lu_classic;
    const auto kernel = with_lu_kind(lu.kind, [](auto k) { return lu_solve_kernel<decltype(k)::value>; });
    const int threads = lu.kind ? HPF_THREADS_GMEM : HPF_THREADS;
    long long ctas = 0;
    rc = resident_ctas(h, kernel, threads, lu.smem, "hpf_lu_solve", &ctas);
    if (rc) return rc;
    if (lu.kind && use_lockstep(h, net.N, B))
        return lu_solve_batched(h, net.N, B, J, a.stride, f, dx, info, (cudaStream_t)stream);
    const unsigned grid = fill_grid(h, ctas, B, false);
    a.workspace = nullptr;
    if (lu.kind) {
        rc = grow(h, h->d_work, (size_t)grid * lub_ld(net.N) * (net.N + 1) * sizeof(double), "hpf_lu_solve: LU workspace");
        if (rc) return rc;
        a.workspace = h->d_work.get();
    }
    return launch(h, kernel, {grid, (unsigned)threads, lu.smem, (cudaStream_t)stream}, net, a);
}

int hpf_lu_solve(hpf_t* h, int B, const double* J, const double* f, double* dx, int* info, void* stream) {
    return ordered(h, stream, [&] { return lu_solve_impl(h, B, J, f, dx, info, stream); });
}

}  // extern "C"
