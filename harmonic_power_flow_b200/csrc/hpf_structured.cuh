// Structured Newton step ("strategy 1") - same Newton-Raphson iteration as HG:536-542, the
// linear solve of HG:476-479 done by exact block elimination instead of a dense LU of J.
//
// Why it is the same step.  The current-balance rows of the harmonic mismatch (HG:326-357)
// are LINEAR in the complex voltages:  f_I = A V + I_N  with the constant complex operator
//     A = blockdiag_h Y(h)  -  scatter(Y_N)            (rows/cols: stacked index s = h n + i).
// Their Jacobian rows (HG:403-446) are therefore  A T,  T = dV/d(theta, V_m) the 2x2-block
// diagonal polar map  dV = E (dV_m + j V_m dtheta),  E = e^{j theta}.  Only the fundamental
// power rows of the linear buses (HG:451-467) depend on the state.  Partition the stacked
// indices into  F = {h = 1, linear buses}  (power rows, polar unknowns x_F) and
// Z = everything else (current rows, full complex unknowns u_Z).  J dx = -f becomes
//     A_ZZ u_Z + A_ZF T_F x_F = -f_I        =>  u_Z = u0 - G T_F x_F,
//     u0 = -A_ZZ^{-1} f_I,   G = A_ZZ^{-1} A_ZF      (A_ZZ^{-1}, G: once per network)
//     J_SF x_F + J_SZ1 T_Z1^{-1} u_Z1 = -f_S        =>  a (2m-1-c)-sized real system for x_F
// followed by the exact polar conversion  dtheta = Im(conj(E) u)/V_m,  dV_m = Re(conj(E) u).
// cond(A_ZZ) ~ 1e3..1e5 on the reference networks while cond(J) reaches 2e7..4e9 (the polar
// scaling), so this step is at least as accurate as an LU of J; round-off differs, exactly
// as it does between SuperLU and LAPACK (SURVEY 7.3).
//
// Kernels: struct_assemble / cinv_gj / struct_G (setup, once per network), fund_tile_kernel
// (fundamental NR, one lane per scenario) and harm_tile_kernel (harmonic NR, 32 scenarios
// per CTA with lane = scenario; lanes are refilled from a global queue as soon as their
// scenario finishes because iteration counts differ, 8..34+).
#pragma once
#include <cstdint>
#include "hpf_device.cuh"

#define HPF_T 32            // scenarios per tile (= lanes)

struct StructNet {
    int nZ, nx;
    const double2* Ainv;   // [nZ][nZ] row-major
    const double2* G;      // [nZ][m]
    const double2* GT;     // [m][nZ]   transposed copy (coalesced over rows in the per-CTA kernel)
    const double2* WNL;    // [nZ][qH]  columns of Ainv that multiply the Norton currents
    int yn_elems;          // complex entries of the Y_N table
    // nonlinear neighbours of the linear buses at the fundamental (CSR over i = 0..m-1):
    // k = nbr_idx[e] for nbr_ptr[i] <= e < nbr_ptr[i+1]  <=>  Y1[i][m+k] != 0
    const int* nbr_ptr;
    const int* nbr_idx;
};

// ---------------------------------------------------------------------------------------
// setup 1: A_ZZ and A_ZF from Y(h) and Y_N
__global__ void struct_assemble_kernel(const DevNet net, double2* __restrict__ AZZ,
                                       double2* __restrict__ AZF) {
    const int n = net.n, m = net.m, H = net.H, nZ = net.nH - m;
    const size_t total = (size_t)nZ * (nZ + m);
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(t / (nZ + m)), cc = (int)(t - (size_t)r * (nZ + m));
        const int s = r + m, h = s / n, i = s - h * n;
        const int sc = (cc < nZ) ? cc + m : cc - nZ;      // column stacked index (Z first, then F)
        const int hc = sc / n, jc = sc - hc * n;
        double2 v = make_double2(0.0, 0.0);
        if (hc == h) v = net.Y[((size_t)h * n + i) * n + jc];
        if (i >= m && jc == i) {
            const int dev = net.dev_of_nl[i - m];
            if (net.coupled) v = csub(v, net.YN[((size_t)dev * H + h) * H + hc]);
            else if (hc == h) v = csub(v, net.YN[(size_t)dev * H + h]);
        }
        if (cc < nZ) AZZ[(size_t)r * nZ + cc] = v;
        else AZF[(size_t)r * m + (cc - nZ)] = v;
    }
}

__device__ __forceinline__ double2 crecip(double2 a) {
    // 1 / a, scaled (Smith) to avoid overflow
    if (fabs(a.x) >= fabs(a.y)) {
        const double r = a.y / a.x, d = 1.0 / (a.x + a.y * r);
        return make_double2(d, -r * d);
    }
    const double r = a.x / a.y, d = 1.0 / (a.y + a.x * r);
    return make_double2(r * d, -d);
}

// setup 2: in-place Gauss-Jordan inverse with partial (row) pivoting, complex, one CTA,
// matrix in global memory (L2 resident).  info[0] = 0 or k+1 (zero pivot);
// info[1..2] = min / max pivot modulus as doubles (a cheap conditioning indicator).
__global__ void __launch_bounds__(1024)
cinv_gj_kernel(int n, double2* __restrict__ A, int* __restrict__ ipiv, int* __restrict__ info,
               double* __restrict__ pivrange) {
    __shared__ double redv[33];
    __shared__ int redi[33];
    __shared__ double2 spiv;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    double pmin = CUDART_INF, pmax = 0.0;
    if (tid == 0) info[0] = 0;
    for (int k = 0; k < n; ++k) {
        __syncthreads();
        double best = -1.0;
        int bi = k;
        for (int i = k + tid; i < n; i += blockDim.x) {
            const double2 a = A[(size_t)i * n + k];
            const double v = hypot(a.x, a.y);
            if (v > best) { best = v; bi = i; }
        }
        for (int o = 16; o; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) { redv[warp] = best; redi[warp] = bi; }
        __syncthreads();
        if (warp == 0) {
            best = (lane < nw) ? redv[lane] : -1.0;
            bi = (lane < nw) ? redi[lane] : 0x7fffffff;
            for (int o = 16; o; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, best, o);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
                if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
            }
            if (lane == 0) {
                redv[32] = best; redi[32] = bi;
                ipiv[k] = bi;
                if (!(best > 0.0) || !(best < CUDART_INF)) { if (info[0] == 0) info[0] = k + 1; }
            }
        }
        __syncthreads();
        const int p = redi[32];
        pmin = fmin(pmin, redv[32]); pmax = fmax(pmax, redv[32]);
        if (p != k)
            for (int j = tid; j < n; j += blockDim.x) {
                const double2 t = A[(size_t)k * n + j];
                A[(size_t)k * n + j] = A[(size_t)p * n + j];
                A[(size_t)p * n + j] = t;
            }
        __syncthreads();
        if (tid == 0) spiv = crecip(A[(size_t)k * n + k]);
        __syncthreads();
        const double2 pinv = spiv;
        for (int j = tid; j < n; j += blockDim.x) {
            const double2 a = (j == k) ? make_double2(1.0, 0.0) : A[(size_t)k * n + j];
            A[(size_t)k * n + j] = cmul(a, pinv);
        }
        __syncthreads();
        // eliminate column k from every other row; element (i, j): a_ij -= a_ik * a_kj,
        // with a_ik first replaced by 0 (its inverse-column value becomes -a_ik * a_kk).
        // Pass 1 caches the multipliers (column k) in place of nothing: read them on the fly,
        // but column k itself must be updated LAST (it is the multiplier source).
        for (size_t t = tid; t < (size_t)n * (n - 1); t += blockDim.x) {
            const int i = (int)(t / (n - 1));
            int j = (int)(t - (size_t)i * (n - 1));
            if (j >= k) ++j;                      // skip column k in this pass
            if (i == k) continue;
            const double2 f = A[(size_t)i * n + k];
            const double2 akj = A[(size_t)k * n + j];
            A[(size_t)i * n + j] = csub(A[(size_t)i * n + j], cmul(f, akj));
        }
        __syncthreads();
        const double2 akk = A[(size_t)k * n + k];
        __syncthreads();
        for (int i = tid; i < n; i += blockDim.x) {
            if (i == k) continue;
            const double2 f = A[(size_t)i * n + k];
            A[(size_t)i * n + k] = cneg(cmul(f, akk));
        }
    }
    __syncthreads();
    for (int k = n - 1; k >= 0; --k) {            // undo the row interchanges on the columns
        const int p = ipiv[k];
        if (p != k)
            for (int i = tid; i < n; i += blockDim.x) {
                const double2 t = A[(size_t)i * n + k];
                A[(size_t)i * n + k] = A[(size_t)i * n + p];
                A[(size_t)i * n + p] = t;
            }
        __syncthreads();
    }
    if (tid == 0) { pivrange[0] = pmin; pivrange[1] = pmax; }
}

// setup 2b: the same Gauss-Jordan inversion spread over the whole GPU for large operators
// (nZ in the thousands: 200- / 1000-bus networks), four small launches per pivot step:
//   gjm_pivot   (1 CTA)      pivot row p of column k, 1 / pivot, bookkeeping
//   gjm_row     (columns)    interchange rows k <-> p, scale the pivot row, keep a copy of it
//   gjm_col     (rows)       copy of column k (the multipliers), taken after the interchange
//   gjm_elim    (elements)   a_ij -= a_ik a_kj (j != k),  a_ik = -a_ik a_kk
// and gjm_unpermute (rows) to undo the interchanges on the columns at the end.
__global__ void __launch_bounds__(1024)
gjm_pivot_kernel(int n, int k, const double2* __restrict__ A, int* __restrict__ ipiv, int* __restrict__ info,
                 double* __restrict__ pivrange, double2* __restrict__ pinv_out) {
    __shared__ double redv[33];
    __shared__ int redi[33];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    double best = -1.0;
    int bi = k;
    for (int i = k + tid; i < n; i += blockDim.x) {
        const double2 a = A[(size_t)i * n + k];
        const double v = hypot(a.x, a.y);
        if (v > best) { best = v; bi = i; }
    }
    for (int o = 16; o; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if (lane == 0) { redv[warp] = best; redi[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        best = (lane < nw) ? redv[lane] : -1.0;
        bi = (lane < nw) ? redi[lane] : 0x7fffffff;
        for (int o = 16; o; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) {
            ipiv[k] = bi;
            if (k == 0) { info[0] = 0; pivrange[0] = CUDART_INF; pivrange[1] = 0.0; }
            if (!(best > 0.0) || !(best < CUDART_INF)) { if (info[0] == 0) info[0] = k + 1; }
            pivrange[0] = fmin(pivrange[0], best);
            pivrange[1] = fmax(pivrange[1], best);
            pinv_out[0] = crecip(A[(size_t)bi * n + k]);
        }
    }
}

__global__ void gjm_row_kernel(int n, int k, double2* __restrict__ A, const int* __restrict__ ipiv,
                               const double2* __restrict__ pinv_in, double2* __restrict__ rowk) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int p = ipiv[k];
    const double2 pinv = pinv_in[0];
    const double2 tk = A[(size_t)k * n + j], tp = A[(size_t)p * n + j];
    const double2 a = (j == k) ? make_double2(1.0, 0.0) : tp;
    const double2 v = cmul(a, pinv);
    A[(size_t)k * n + j] = v;
    if (p != k) A[(size_t)p * n + j] = tk;
    rowk[j] = v;
}

__global__ void gjm_col_kernel(int n, int k, const double2* __restrict__ A, double2* __restrict__ colk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    colk[i] = (i == k) ? make_double2(0.0, 0.0) : A[(size_t)i * n + k];
}

__global__ void gjm_elim_kernel(int n, int k, double2* __restrict__ A, const double2* __restrict__ rowk,
                                const double2* __restrict__ colk) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const double2 r = rowk[j];
    for (int i = blockIdx.y; i < n; i += gridDim.y) {
        if (i == k) continue;
        const double2 f = colk[i];
        double2* a = A + (size_t)i * n + j;
        *a = (j == k) ? cneg(cmul(f, r)) : csub(*a, cmul(f, r));
    }
}

// ---- blocked variant (panels of GJB_NB pivots): the pivot steps of a panel touch only the panel's
// columns [j0, j1) (gjb_pivot_row_kernel, gjb_col_elim_kernel); every other column receives the panel's GJB_NB rank-1
// updates at once, A -= F R, as one complex GEMM on the tensor cores (hpf_zgemm.cuh).  With column k
// of the pivot step reset to e_k, a Gauss-Jordan step IS a rank-1 update A -= f r^T over all rows when
// f_k = a_kk - 1 (a_kk the pivot), f_i = a_ik otherwise, r = (row k) / a_kk:
//   F [n x NB]  f of every step of the panel (rows interchanged along with the matrix rows),
//   R [NB x n]  the scaled pivot rows on the other columns: R_t = (a_{k_t,:} - sum_{s<t} F[k_t][s] R_s) / a_kk.
#define GJB_NB 64

// The two kernels of a blocked pivot step (the set-up is bound by the NUMBER of launches - ~6 us each,
// 12,400 pivots for the 1000-bus configuration - so pivot search + pivot row are one launch, multiplier
// column + elimination of the panel's columns the other).
__global__ void __launch_bounds__(1024)
gjb_pivot_row_kernel(int n, int k, int j0, int j1, double2* __restrict__ A, int* __restrict__ ipiv,
                     int* __restrict__ info, double* __restrict__ pivrange, double2* __restrict__ pinv_out,
                     double2* __restrict__ rowk, double2* __restrict__ F, double2* __restrict__ pinv_all) {
    __shared__ double redv[33];
    __shared__ int redi[33];
    __shared__ double2 spinv;
    __shared__ int sp;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
    double best = -1.0;
    int bi = k;
    for (int i = k + tid; i < n; i += blockDim.x) {
        const double2 a = A[(size_t)i * n + k];
        const double v = hypot(a.x, a.y);
        if (v > best) { best = v; bi = i; }
    }
    for (int o = 16; o; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if (lane == 0) { redv[warp] = best; redi[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        best = (lane < nw) ? redv[lane] : -1.0;
        bi = (lane < nw) ? redi[lane] : 0x7fffffff;
        for (int o = 16; o; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        }
        if (lane == 0) {
            ipiv[k] = bi;
            if (k == 0) { info[0] = 0; pivrange[0] = CUDART_INF; pivrange[1] = 0.0; }
            if (!(best > 0.0) || !(best < CUDART_INF)) { if (info[0] == 0) info[0] = k + 1; }
            pivrange[0] = fmin(pivrange[0], best);
            pivrange[1] = fmax(pivrange[1], best);
            const double2 pi = crecip(A[(size_t)bi * n + k]);
            pinv_out[0] = pi;
            spinv = pi;
            sp = bi;
        }
    }
    __syncthreads();
    // pivot row of step t = k - j0 on the panel's columns; earlier columns of F follow the interchange
    const int j = j0 + tid;
    if (j < j1) {
        const int p = sp, t = k - j0;
        const double2 pinv = spinv;
        const double2 tk = A[(size_t)k * n + j], tp = A[(size_t)p * n + j];
        const double2 a = (j == k) ? make_double2(1.0, 0.0) : tp;
        const double2 v = cmul(a, pinv);
        A[(size_t)k * n + j] = v;
        if (p != k) A[(size_t)p * n + j] = tk;
        rowk[tid] = v;
        if (tid < t && p != k) {
            const double2 fk = F[(size_t)k * GJB_NB + tid], fp = F[(size_t)p * GJB_NB + tid];
            F[(size_t)k * GJB_NB + tid] = fp;
            F[(size_t)p * GJB_NB + tid] = fk;
        }
        if (j == k) pinv_all[t] = pinv;
    }
}

// blockDim = (GJB_NB, 4): thread (x, y) = column j0 + x of one of the block's 4 rows per pass
__global__ void __launch_bounds__(GJB_NB * 4)
gjb_col_elim_kernel(int n, int k, int j0, int j1, double2* __restrict__ A, const double2* __restrict__ rowk,
                    const double2* __restrict__ pinv_in, double2* __restrict__ F) {
    const int j = j0 + threadIdx.x;
    const bool jok = j < j1;
    const double2 r = jok ? rowk[threadIdx.x] : make_double2(0.0, 0.0);
    const int rows_per_pass = gridDim.x * blockDim.y;
    for (int base = 0; base < n; base += rows_per_pass) {            // (uniform trip count: barrier inside)
        const int i = base + blockIdx.x * blockDim.y + threadIdx.y;
        const bool iok = i < n;
        const double2 f = iok ? A[(size_t)i * n + k] : make_double2(0.0, 0.0);     // multiplier, read by the whole row
        __syncthreads();                                             // ... before thread j == k overwrites it
        if (iok && jok) {
            if (i != k) {
                double2* a = A + (size_t)i * n + j;
                *a = (j == k) ? cneg(cmul(f, r)) : csub(*a, cmul(f, r));
            }
            if (j == k) {
                double2 fr = f;
                if (i == k) {                                        // a_kk - 1 (row k holds 1 / a_kk at column k)
                    const double2 piv = crecip(pinv_in[0]);
                    fr = make_double2(piv.x - 1.0, piv.y);
                }
                F[(size_t)i * GJB_NB + (k - j0)] = fr;
            }
        }
    }
}

// the other columns: the panel's interchanges, then R (forward substitution over the pivot rows);
// R = 0 on the panel's own columns so that the GEMM leaves them alone
__global__ void gjb_rows_kernel(int n, int j0, int nb, double2* __restrict__ A, const int* __restrict__ ipiv,
                                const double2* __restrict__ F, const double2* __restrict__ pinv_all,
                                double2* __restrict__ R) {
    __shared__ double2 sF[GJB_NB * GJB_NB / 2 + GJB_NB];     // strictly lower triangle of F on the pivot rows
    __shared__ double2 sP[GJB_NB];
    __shared__ int sPiv[GJB_NB];
    for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) {
        const int t = e / nb, s2 = e % nb;
        if (s2 < t) sF[t * (t - 1) / 2 + s2] = F[(size_t)(j0 + t) * GJB_NB + s2];
    }
    for (int t = threadIdx.x; t < nb; t += blockDim.x) { sP[t] = pinv_all[t]; sPiv[t] = ipiv[j0 + t]; }
    __syncthreads();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (j >= j0 && j < j0 + nb) {
        for (int t = 0; t < nb; ++t) R[(size_t)t * n + j] = make_double2(0.0, 0.0);
        return;
    }
    for (int t = 0; t < nb; ++t) {                           // the interchanges, in order
        const int k = j0 + t, p = sPiv[t];
        if (p != k) {
            const double2 a = A[(size_t)k * n + j], b = A[(size_t)p * n + j];
            A[(size_t)k * n + j] = b;
            A[(size_t)p * n + j] = a;
        }
    }
    for (int t = 0; t < nb; ++t) {
        double2 x = A[(size_t)(j0 + t) * n + j];
        for (int s2 = 0; s2 < t; ++s2) x = csub(x, cmul(sF[t * (t - 1) / 2 + s2], R[(size_t)s2 * n + j]));
        R[(size_t)t * n + j] = cmul(x, sP[t]);
    }
}

__global__ void gjm_unpermute_kernel(int n, double2* __restrict__ A, const int* __restrict__ ipiv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double2* row = A + (size_t)i * n;
    for (int k = n - 1; k >= 0; --k) {
        const int p = ipiv[k];
        if (p != k) {
            const double2 t = row[k];
            row[k] = row[p];
            row[p] = t;
        }
    }
}

// setup 3: G = Ainv * A_ZF
// (A_ZF is zero outside its first q rows - only the fundamental rows of the nonlinear buses
// see the fundamental voltages of the linear buses - so the sum stops at kmax = q.)
__global__ void struct_G_kernel(int nZ, int m, int kmax, const double2* __restrict__ Ainv,
                                const double2* __restrict__ AZF, double2* __restrict__ G,
                                double2* __restrict__ GT) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)nZ * m) return;
    const int r = (int)(t / m), j = (int)(t - (size_t)r * m);
    double2 acc = make_double2(0.0, 0.0);
    for (int k = 0; k < kmax; ++k) acc = cadd(acc, cmul(Ainv[(size_t)r * nZ + k], AZF[(size_t)k * m + j]));
    G[t] = acc;
    GT[(size_t)j * nZ + r] = acc;
}

// ---------------------------------------------------------------------------------------
// setup for large networks (variant 3): the operator inverse through its STRUCTURE instead of a
// Gauss-Jordan inversion of the whole A_ZZ (order nZ = 12,400 for the 1000-bus configuration:
// 8 nZ^3 = 1.5e13 flop and one HBM pass over 2.5 GB per pivot - 13 s).  With
//     A_ZZ = D - E YN E^T,   D = blockdiag(Y_0[nl, nl], Y_1, ..., Y_{H-1}),
//     E = the nZ x qH selection of the (harmonic, nonlinear bus) rows,  YN = the Norton admittances
//     (block diagonal per bus, HG:313-323),
// the Woodbury identity gives, with S = E^T D^-1 E (block diagonal per harmonic) and the
// qH x qH "capacitance" matrix M = I - YN S:
//     W_NL = A_ZZ^-1 E    = (D^-1 E) M^-1
//     G    = A_ZZ^-1 A_ZF = D^-1 A_ZF + W_NL (YN E^T D^-1 A_ZF),
// i.e. H block inversions of order <= n, ONE inversion of order qH and three families of complex
// GEMMs on the FP64 tensor cores (hpf_zgemm.cuh): ~1.7e12 flop instead of 1.5e13.
// Column index u = k H + h of W_NL / M  <->  nonlinear bus m + k at harmonic h.

// block h of D into its slot of Dinv (to be inverted in place): block 0 = Y_0[nl, nl] (q x q), else Y_h
__global__ void wb_blocks_kernel(const DevNet net, double2* __restrict__ Dinv) {
    const int n = net.n, m = net.m, q = net.q, H = net.H;
    const size_t total = (size_t)q * q + (size_t)(H - 1) * n * n;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        double2 v;
        int h, i, j;
        if (t < (size_t)q * q) {
            h = 0; i = m + (int)(t / q); j = m + (int)(t % q);
        } else {
            const size_t r = t - (size_t)q * q;
            h = 1 + (int)(r / ((size_t)n * n));
            const size_t e = r % ((size_t)n * n);
            i = (int)(e / n); j = (int)(e % n);
        }
        v = net.Y[((size_t)h * n + i) * n + j];
        // uncoupled Norton equivalents sit on the diagonal of their own harmonic block
        if (!net.coupled && i >= m && i == j) v = csub(v, net.YN[(size_t)net.dev_of_nl[i - m] * H + h]);
        Dinv[t] = v;
    }
}

__device__ __forceinline__ const double2* wb_block(const double2* Dinv, int h, int n, int q) {
    return h == 0 ? Dinv : Dinv + (size_t)q * q + (size_t)(h - 1) * n * n;
}

// M = I - YN S :  M[(k,h)][(k',p)] = delta - YN_k[h][p] * (D_p^-1)[nl k][nl k']   (coupled; uncoupled: M = I)
__global__ void wb_capacitance_kernel(const DevNet net, const double2* __restrict__ Dinv, double2* __restrict__ Mx) {
    const int n = net.n, m = net.m, q = net.q, H = net.H, qH = q * H;
    const size_t total = (size_t)qH * qH;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int u = (int)(t / qH), v = (int)(t % qH);
        const int k = u / H, h = u % H, k2 = v / H, p = v % H;
        double2 val = make_double2(u == v ? 1.0 : 0.0, 0.0);
        if (net.coupled) {
            const double2 yn = net.YN[((size_t)net.dev_of_nl[k] * H + h) * H + p];
            const double2* Dp = wb_block(Dinv, p, n, q);
            const double2 sp = (p == 0) ? Dp[(size_t)k * q + k2] : Dp[(size_t)(m + k) * n + m + k2];
            val = csub(val, cmul(yn, sp));
        }
        Mx[t] = val;
    }
}

// U [qH x m] = YN E^T D^-1 A_ZF :  U[(k,h)][j] = YN_k[h][0] T[k][j],  T = D_0^-1 Y_0[nl, lin]
__global__ void wb_coupling_rhs_kernel(const DevNet net, const double2* __restrict__ T, double2* __restrict__ U) {
    const int m = net.m, q = net.q, H = net.H;
    const size_t total = (size_t)q * H * m;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int u = (int)(t / m), j = (int)(t % m), k = u / H, h = u % H;
        double2 v = make_double2(0.0, 0.0);
        if (net.coupled) v = cmul(net.YN[((size_t)net.dev_of_nl[k] * H + h) * H + 0], T[(size_t)k * m + j]);
        U[t] = v;
    }
}

// G += [T; 0] (the D^-1 A_ZF term lives in the first q rows) and GT = G^T
__global__ void wb_finish_G_kernel(int nZ, int m, int q, const double2* __restrict__ T, double2* __restrict__ G,
                                   double2* __restrict__ GT) {
    const size_t total = (size_t)nZ * m;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(t / m), j = (int)(t % m);
        double2 g = G[t];
        if (r < q) g = cadd(g, T[(size_t)r * m + j]);
        G[t] = g;
        GT[(size_t)j * nZ + r] = g;
    }
}

// ---------------------------------------------------------------------------------------
// Per-lane dense solve of a small augmented real system M [nx][nx+1] stored with stride
// HPF_T (element (r, c) of lane l at M[(r*(nx+1)+c)*HPF_T + l] -> bank = lane, conflict
// free).  Gaussian elimination with partial pivoting, each lane pivots on its own data.
// The solution overwrites column nx.  Returns nonzero for a zero / non-finite pivot.
__device__ __forceinline__ int lane_gauss_solve(double* M, const int nx, const int lane) {
    const int w = nx + 1;
    int bad = 0;
#define MM(r, c) M[((r) * w + (c)) * HPF_T + lane]
    for (int k = 0; k < nx; ++k) {
        int p = k;
        double best = fabs(MM(k, k));
        for (int i = k + 1; i < nx; ++i) {
            const double v = fabs(MM(i, k));
            if (v > best) { best = v; p = i; }
        }
        if (!(best > 0.0) || !(best < CUDART_INF)) bad = 1;
        if (p != k)
            for (int c = k; c <= nx; ++c) {
                const double t = MM(k, c);
                MM(k, c) = MM(p, c);
                MM(p, c) = t;
            }
        const double r = 1.0 / MM(k, k);
        for (int i = k + 1; i < nx; ++i) {
            const double l = MM(i, k) * r;
            for (int c = k + 1; c <= nx; ++c) MM(i, c) -= l * MM(k, c);
        }
    }
    for (int k = nx - 1; k >= 0; --k) {
        double s = MM(k, nx);
        for (int c = k + 1; c < nx; ++c) s -= MM(k, c) * MM(c, nx);
        MM(k, nx) = s / MM(k, k);
    }
#undef MM
    return bad;
}

// Shape specialisation: when the network dimensions are compile-time constants every loop
// bound and every shared-memory offset folds into immediates (about a third of the generic
// kernel's instructions are integer address arithmetic).  Dims<0,...> = runtime dimensions.
template <int N_, int M_, int C_, int H_, int Q_>
struct Dims {
    static constexpr int n = N_, m = M_, c = C_, H = H_, q = Q_;
};
typedef Dims<0, 0, 0, 0, 0> DynDims;

// ---------------------------------------------------------------------------------------
// Small per-lane dense solve in REGISTERS (NX known at compile time): loads the augmented
// system from the strided smem array, Gaussian elimination with partial pivoting (per lane),
// leaves the solution in x[].  Returns nonzero for a zero / non-finite pivot.
template <int NX>
__device__ __forceinline__ int lane_gauss_solve_reg(const double* M, const int lane, double* x) {
    double A[NX][NX + 1];
#pragma unroll
    for (int r = 0; r < NX; ++r)
#pragma unroll
        for (int cc = 0; cc <= NX; ++cc) A[r][cc] = M[(r * (NX + 1) + cc) * HPF_T + lane];
    int bad = 0;
#pragma unroll
    for (int k = 0; k < NX; ++k) {
        // partial pivoting without dynamic register indexing: bubble the largest row up
#pragma unroll
        for (int i = k + 1; i < NX; ++i) {
            const bool sw = fabs(A[i][k]) > fabs(A[k][k]);
#pragma unroll
            for (int cc = k; cc <= NX; ++cc) {
                const double t0 = A[k][cc], t1 = A[i][cc];
                A[k][cc] = sw ? t1 : t0;
                A[i][cc] = sw ? t0 : t1;
            }
        }
        const double pv = fabs(A[k][k]);
        if (!(pv > 0.0) || !(pv < CUDART_INF)) bad = 1;
        const double r = 1.0 / A[k][k];
#pragma unroll
        for (int i = k + 1; i < NX; ++i) {
            const double l = A[i][k] * r;
#pragma unroll
            for (int cc = k + 1; cc <= NX; ++cc) A[i][cc] -= l * A[k][cc];
        }
    }
#pragma unroll
    for (int k = NX - 1; k >= 0; --k) {
        double sv = A[k][NX];
#pragma unroll
        for (int cc = k + 1; cc < NX; ++cc) sv -= A[k][cc] * x[cc];
        x[k] = sv / A[k][k];
    }
    return bad;
}

// ---------------------------------------------------------------------------------------
// Fundamental Newton-Raphson (HG:244-275), one lane per scenario, warps independent.
// Writes the fundamental solution into rows 0..n-1 of V_m / V_a [H, n, B] (the harmonic
// kernel picks it up there), n_iter_f and a preliminary status.
struct FundTileArgs {
    int B;
    const double *P, *Q;
    double thresh_f;
    int max_f;
    double *V_m, *V_a;
    int *n_iter_f, *status;
    double* hist_f;          // [max_f + 1, B] mismatch norm before each step and after the last one, or NULL
};

__host__ __device__ inline size_t fund_tile_doubles_per_warp(int n, int Nf) {
    // Vm, Va, Vre, Vim, Ere, Eim [n]; I1 [n] complex; P, Q [n]; M [Nf][Nf+1]
    return (size_t)(6 * n + 2 * n + 2 * n + Nf * (Nf + 1)) * HPF_T;
}

// (D: compile-time dimensions for the BASELINE 4-bus shapes - loops unroll, indices fold, the
// (2n-1-c)-sized system is solved in registers; same arithmetic as the runtime-dimension instance)
template <class D>
__global__ void __launch_bounds__(128)
fund_tile_kernel(const DevNet net, const FundTileArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const int n = D::n ? D::n : net.n, c = D::n ? D::c : net.c, Nf = D::n ? 2 * D::n - 1 - D::c : net.Nf;
    constexpr int NFC = D::n ? 2 * D::n - 1 - D::c : 1;
    const size_t B = (size_t)a.B;
    double* base = smem + (size_t)warp * fund_tile_doubles_per_warp(n, Nf);
    double* Vm = base;            double* Va = Vm + n * HPF_T;
    double* Vre = Va + n * HPF_T; double* Vim = Vre + n * HPF_T;
    double* Ere = Vim + n * HPF_T; double* Eim = Ere + n * HPF_T;
    double2* I1 = reinterpret_cast<double2*>(Eim + n * HPF_T);
    double* Pl = reinterpret_cast<double*>(I1 + n * HPF_T);
    double* Ql = Pl + n * HPF_T;
    double* M = Ql + n * HPF_T;
    const int w = Nf + 1;
    for (size_t tile = (size_t)blockIdx.x * nwarp + warp; tile * HPF_T < B; tile += (size_t)gridDim.x * nwarp) {
        const size_t b = tile * HPF_T + lane;
        const bool ok = b < B;
        const size_t bb = ok ? b : B - 1;
        for (int i = 0; i < n; ++i) {
            Pl[i * HPF_T + lane] = a.P[i * B + bb];
            Ql[i * HPF_T + lane] = a.Q[i * B + bb];
            Vm[i * HPF_T + lane] = 1.0;
            Va[i * HPF_T + lane] = 0.0;
        }
        int it = 0, status = HPF_ST_CONVERGED;
        bool running = true;
        double err = 0.0;
        for (;;) {
            // mismatch (HG:195-202)
            for (int i = 0; i < n; ++i)
                phasor_one<HPF_T>(i, lane, Vm, Va, Vre, Vim, Ere, Eim, true);
            for (int i = 0; i < n; ++i) I1[i * HPF_T + lane] = ydotv<HPF_T>(net, 0, i, lane, Vre, Vim);
            double mx = 0.0;
            for (int i = 0; i < n; ++i) {
                const double2 v = make_double2(Vre[i * HPF_T + lane], Vim[i * HPF_T + lane]);
                const double2 sl = cmul(v, cconj(I1[i * HPF_T + lane]));
                const double fr = sl.x + Pl[i * HPF_T + lane], fi = sl.y + Ql[i * HPF_T + lane];
                if (i >= 1) {
                    M[((i - 1) * w + Nf) * HPF_T + lane] = fr;
                    const double x = fabs(fr);
                    mx = (x != x || x > mx) ? x : mx;
                }
                if (i >= c) {
                    M[(((n - 1) + i - c) * w + Nf) * HPF_T + lane] = fi;
                    const double x = fabs(fi);
                    mx = (x != x || x > mx) ? x : mx;
                }
            }
            if (running) {
                err = mx;
                if (a.hist_f && ok) a.hist_f[(size_t)it * B + b] = err;
                running = (err > a.thresh_f) && (it < a.max_f);
            }
            if (!__any_sync(0xffffffffu, running)) break;
            // Jacobian (HG:205-223) into M[:, 0..Nf-1]
            for (int r = 0; r < Nf; ++r)
                for (int cc = 0; cc < Nf; ++cc) M[(r * w + cc) * HPF_T + lane] = 0.0;
            // per-lane arrays are strided: address element i of array X as X[i*HPF_T + lane]
            for (int i = 0; i < n; ++i)
                for (int j = 0; j < n; ++j) {
                    const double2 y = ldg2(net.Y + (size_t)i * n + j);
                    if (i != j && y.x == 0.0 && y.y == 0.0) continue;
                    const double2 vi = make_double2(Vre[i * HPF_T + lane], Vim[i * HPF_T + lane]);
                    const double2 ei = make_double2(Ere[i * HPF_T + lane], Eim[i * HPF_T + lane]);
                    const double2 vj = make_double2(Vre[j * HPF_T + lane], Vim[j * HPF_T + lane]);
                    const double2 ej = make_double2(Ere[j * HPF_T + lane], Eim[j * HPF_T + lane]);
                    const double2 i1 = I1[i * HPF_T + lane];
                    const double2 yv = cmul(y, vj);
                    const double2 d = (i == j) ? csub(i1, yv) : cneg(yv);
                    const double2 dA = cmul(cmulj(vi), cconj(d));
                    double2 dV = cmul(vi, cconj(cmul(y, ej)));
                    if (i == j) dV = cadd(cmul(ei, cconj(i1)), dV);
                    const int rr = i - 1, ri = (n - 1) + i - c, ca = j - 1, cv = (n - 1) + j - c;
                    if (i >= 1) {
                        if (j >= 1) M[(rr * w + ca) * HPF_T + lane] = dA.x;
                        if (j >= c) M[(rr * w + cv) * HPF_T + lane] = dV.x;
                    }
                    if (i >= c) {
                        if (j >= 1) M[(ri * w + ca) * HPF_T + lane] = dA.y;
                        if (j >= c) M[(ri * w + cv) * HPF_T + lane] = dV.y;
                    }
                }
            int bad;
            if constexpr (D::n != 0) {
                double xs[NFC];
                bad = lane_gauss_solve_reg<NFC>(M, lane, xs);
#pragma unroll
                for (int t = 0; t < NFC; ++t) M[(t * w + Nf) * HPF_T + lane] = xs[t];
            } else {
                bad = lane_gauss_solve(M, Nf, lane);
            }
            if (running) {
                if (bad) status = HPF_ST_SINGULAR;
                for (int t = 0; t < Nf; ++t) {          // x -= dx  (HG:226-235)
                    const double dx = M[(t * w + Nf) * HPF_T + lane];
                    if (t < n - 1) Va[(t + 1) * HPF_T + lane] -= dx;
                    else Vm[(c + t - (n - 1)) * HPF_T + lane] -= dx;
                }
                ++it;
            }
        }
        if (it >= a.max_f) status = HPF_ST_MAXITER;
        if (err != err) status = HPF_ST_NONFINITE;
        if (ok) {
            for (int i = 0; i < n; ++i) {
                a.V_m[i * B + b] = Vm[i * HPF_T + lane];
                a.V_a[i * B + b] = Va[i * HPF_T + lane];
            }
            a.n_iter_f[b] = it;
            a.status[b] = status;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// setup 4: W_NL = columns of Ainv that multiply Norton currents: W_NL[z][u] = Ainv[z][z(u)],
// u = k*H + h  <->  stacked s = h*n + m + k.
__global__ void struct_WNL_kernel(const DevNet net, int nZ, const double2* __restrict__ Ainv,
                                  double2* __restrict__ WNL) {
    const int qH = net.q * net.H;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)nZ * qH) return;
    const int z = (int)(t / qH), u = (int)(t - (size_t)z * qH), k = u / net.H, h = u - k * net.H;
    const int zc = h * net.n + net.m + k - net.m;
    WNL[t] = Ainv[(size_t)z * nZ + zc];
}

// Per-scenario constant of the harmonic stage:  w_N = A_ZZ^{-1} I_N,Z  (I_N enters the
// current balance additively, HG:351-354).  One lane per scenario, rows over warps,
// fully coalesced: wN [nZ, B] complex.
struct WnArgs {
    int B;
    const double2* I_N;   // [qH, B]
    double2* wN;          // [nZ, B]
};

#define HPF_WN_UCH 64      // Norton currents staged per chunk
#define HPF_WN_RPW 4       // rows accumulated per warp at a time

__global__ void __launch_bounds__(256)
wn_tile_kernel(const DevNet net, const StructNet sn, const double2* __restrict__ WNL, const WnArgs a) {
    extern __shared__ __align__(16) double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
    const int qH = net.q * net.H, nZ = sn.nZ;
    const size_t B = (size_t)a.B;
    double2* IN = reinterpret_cast<double2*>(smem);          // [min(qH, UCH)][32]
    const int uch = qH < HPF_WN_UCH ? qH : HPF_WN_UCH;
    for (size_t tile = blockIdx.x; tile * HPF_T < B; tile += gridDim.x) {
        const size_t b = tile * HPF_T + lane;
        const bool ok = b < B;
        const size_t bb = ok ? b : B - 1;
        // row groups of NW * RPW rows; the chunk loop is inside so that the accumulators stay in
        // registers (the staged currents are re-read from L2 once per row group)
        for (int z0 = blockIdx.y * NW * HPF_WN_RPW; z0 < nZ; z0 += gridDim.y * NW * HPF_WN_RPW) {
            double2 acc[HPF_WN_RPW];
#pragma unroll
            for (int r = 0; r < HPF_WN_RPW; ++r) acc[r] = make_double2(0.0, 0.0);
            for (int u0 = 0; u0 < qH; u0 += uch) {
                const int nu = min(uch, qH - u0);
                __syncthreads();
                for (int u = warp; u < nu; u += NW) IN[u * HPF_T + lane] = a.I_N[(size_t)(u0 + u) * B + bb];
                __syncthreads();
#pragma unroll
                for (int r = 0; r < HPF_WN_RPW; ++r) {
                    const int z = z0 + r * NW + warp;
                    if (z < nZ) {
                        const double2* row = WNL + (size_t)z * qH + u0;
                        double2 s2 = acc[r];
                        for (int u = 0; u < nu; ++u) s2 = cadd(s2, cmul(ldg2(row + u), IN[u * HPF_T + lane]));
                        acc[r] = s2;
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < HPF_WN_RPW; ++r) {
                const int z = z0 + r * NW + warp;
                if (z < nZ && ok) a.wN[(size_t)z * B + b] = acc[r];
            }
        }
    }
}

__device__ __forceinline__ void cp_async_f64(double* sdst, const double* gsrc) {
    const uint32_t sa = (uint32_t)__cvta_generic_to_shared(sdst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" :: "r"(sa), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N) : "memory"); }

// Out-of-line transcendental helpers: one copy each keeps the Newton loop inside the
// instruction cache (the inlined versions made the kernel 150 KB of SASS).
__device__ __noinline__ double2 sincos_ol(double x) {
    double sn_, cs_;
    sincos(x, &sn_, &cs_);
    return make_double2(cs_, sn_);
}
// numpy's float remainder a % (2 pi): fmod, then the divisor's sign (HG:548)
__device__ __noinline__ double mod_twopi(double va) {
    const double twopi = 2.0 * CUDART_PI;
    double r = fmod(va, twopi);
    if (r != 0.0) { if (r < 0.0) r += twopi; } else r = 0.0;
    return r;
}

// ---------------------------------------------------------------------------------------
// Harmonic Newton-Raphson, structured step, 32 scenarios per CTA (lane = scenario).
//
// Because f_I = A_ZZ V_Z + A_ZF V_F + I_N,Z is linear in V, the product -A_ZZ^{-1} f_I of the
// step has the closed form   u0 = -V_Z - G V_F - w_N   (w_N per scenario, see above): no
// matrix-vector product with A_ZZ^{-1} is left inside the Newton loop.
//
// Warp roles: the LAST warp is the "border warp": it owns the fundamental rows of the linear
// buses (F: state, power mismatch, the (2m-1-c)-sized border system, lane bookkeeping and
// refill); the other NW-1 warps own the Z rows.  One round:
//   A  load refilled lanes; F rows: apply the pending update; unit phasors E = e^{j theta}  | barrier
//   B  Z warps: current-mismatch rows (HG:326-357) incl. the Norton contraction
//      border warp: power mismatch (HG:372-380) and the border system -> u_F               | barrier
//   C  decisions (every warp, same result); results of finished lanes; Z warps:
//      u_Z = -V_Z - G (V_F + u_F) - w_N, polar conversion, state update;
//      border warp: status words, iteration counters, refill from the global queue          | barrier
struct HarmTileArgs {
    int B, flags, step_only;
    const double *P, *Q;
    const double2* I_N;
    const double2* wN;       // [nZ, B]
    double thresh_h;
    int max_h;
    double *V_m, *V_a;       // in: rows 0..n-1 hold the fundamental solution; out: results
    double2* I_inj;
    int *n_iter_h, *status;  // status in: fundamental-stage status
    double* err_h;
    int* work_counter;
    double* dx_out;          // step_only: [N, B] the Newton update dx (x_new = x - dx)
    double* gstate;          // per-CTA kernel, large networks: scenario state in global memory
    size_t gstate_stride;    //   doubles per CTA (0: state in shared memory)
    int lub_doubles;         //   shared-memory work area of the blocked LU (doubles)
    double* hist_h;          // [max_h + 1, B] mismatch norm before each step and after the last one, or NULL
    int epoch;               // harm_hw_kernel: finished lanes are serviced every `epoch` rounds (>= 1)
};


__host__ __device__ inline size_t harm_tile_const_doubles(int n, int H, int m, int yn_elems) {
    const size_t nH = (size_t)n * H, nZ = nH - m;
    return 2 * ((size_t)H * n * n + yn_elems + nZ * m);
}

__host__ __device__ inline size_t harm_tile_smem_bytes(int n, int H, int m, int c, int q, int nwarps,
                                                       int yn_elems) {
    const size_t nH = (size_t)n * H, nZ = nH - m, nx = (size_t)(m - 1) + (m - c);
    // per lane: Vm, Va, Ere, Eim [nH]; w_N [2 nZ]; I_N, I_inj [2 qH each]; FS, I1, PQ, UF [2 m each];
    // M [nx (nx+1)]; DXF [nx]; red [nwarps]
    const size_t d = 4 * nH + 2 * nZ + 4 * (size_t)q * H + 8 * m + nx * (nx + 1) + nx + nwarps;
    return (d * HPF_T + harm_tile_const_doubles(n, H, m, yn_elems)) * sizeof(double) +
           8 * HPF_T * sizeof(int) + 64;
}

// Row loop of one warp: rows start, start+stride, ... < end.  With a compile-time row count
// the loop is fully unrolled so the (independent) rows' dependency chains interleave: the
// kernel is latency-bound, each row being a chain of dependent FP64 operations.
template <int NR, class F>
__device__ __forceinline__ void row_loop(int start, int end, int stride, F f) {
    if constexpr (NR > 0) {
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int s = start + r * stride;
            if (s < end) f(s);
        }
    } else {
        for (int s = start; s < end; s += stride) f(s);
    }
}

template <int NW, int MINB, class D>
__global__ void __launch_bounds__(NW * 32, MINB)
harm_tile_kernel(const DevNet net, const StructNet sn, const HarmTileArgs a) {
    extern __shared__ __align__(16) double smem[];
    constexpr int CW = NW - 1;                     // Z ("compute") warps
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool border = (warp == NW - 1);
    const int n = D::n ? D::n : net.n, m = D::n ? D::m : net.m, c = D::n ? D::c : net.c;
    const int H = D::n ? D::H : net.H, q = D::n ? D::q : net.q, nH = n * H;
    const int nZ = nH - m, nx = (m - 1) + (m - c), nth = m - 1;
    // compile-time row counts per Z warp (0 = runtime loops)
    constexpr int ZR = D::n ? (D::n * D::H - D::m + CW - 1) / CW : 0;
    constexpr int HR = D::n ? (D::q * D::H + CW - 1) / CW : 0;
    constexpr int LR = D::n ? (D::m * (D::H - 1) + CW - 1) / CW : 0;
    const size_t B = (size_t)a.B;
#define AT(X, i) X[(i) * HPF_T + lane]
#define ATV(i) V2[(i) * HPF_T + lane]
    // ---- shared memory: network constants, then per-lane arrays ----
    double2* sY = reinterpret_cast<double2*>(smem);
    double2* sYN = sY + (size_t)H * n * n;
    double2* sG = sYN + sn.yn_elems;
    double* p = reinterpret_cast<double*>(sG + (size_t)nZ * m);
    double* Vm = p;  p += nH * HPF_T;
    double* Va = p;  p += nH * HPF_T;
    double2* V2 = reinterpret_cast<double2*>(p); p += 2 * nH * HPF_T;   // phasors (re, im) interleaved: one LDS.128 per operand
    double* Wre = p; p += nZ * HPF_T;      // w_N (index z = s - m), constant per scenario
    double* Wim = p; p += nZ * HPF_T;
    double* INre = p; p += q * H * HPF_T;  // I_N of the lane's scenario
    double* INim = p; p += q * H * HPF_T;
    double* IJre = p; p += q * H * HPF_T;  // Norton injections (result I_inj)
    double* IJim = p; p += q * H * HPF_T;
    double* FSre = p; p += m * HPF_T;      // power mismatch of buses s < m
    double* FSim = p; p += m * HPF_T;
    double* I1re = p; p += m * HPF_T;      // (Y1 V1)_i, i < m
    double* I1im = p; p += m * HPF_T;
    double* Pl = p;  p += m * HPF_T;
    double* Ql = p;  p += m * HPF_T;
    double* UFre = p; p += m * HPF_T;
    double* UFim = p; p += m * HPF_T;
    double* M = p;   p += nx * (nx + 1) * HPF_T;
    double* DXF = p; p += nx * HPF_T;
    double* red = p; p += NW * HPF_T;
    int* scen2 = reinterpret_cast<int*>(p);        // [2][32] double-buffered scenario index
    int* itc = scen2 + 2 * HPF_T;
    int* stat = itc + HPF_T;
    int* fnew = stat + HPF_T;

    for (int t = threadIdx.x; t < H * n * n; t += NW * 32) sY[t] = net.Y[t];
    for (int t = threadIdx.x; t < sn.yn_elems; t += NW * 32) sYN[t] = net.YN[t];
    for (int t = threadIdx.x; t < nZ * m; t += NW * 32) sG[t] = sn.G[t];

    // ---- initial fill ----
    if (border) {
        int idx;
        if (a.step_only) {
            idx = blockIdx.x * HPF_T + lane;
        } else {
            int base = 0;
            if (lane == 0) base = atomicAdd(a.work_counter, HPF_T);
            base = __shfl_sync(0xffffffffu, base, 0);
            idx = base + lane;
        }
        scen2[lane] = ((size_t)idx < B) ? idx : -1;
        itc[lane] = 0;
        fnew[lane] = 1;
        stat[lane] = 0;
    }
    __syncthreads();
    int cur = 0;
    bool pendF = false;                            // border warp: F-row update of the last step pending

    for (;;) {
        const int* scen = scen2 + cur * HPF_T;
        const int sc = scen[lane];
        const int itv = itc[lane];          // read before barrier A; the border warp updates it in C
        // ================= A: load refilled lanes, unit phasors =================
        {
            const bool isnew = fnew[lane] != 0;
            if (border) {
                // F rows (s < m): state, P, Q, status; pending update; sincos
                if (isnew) {
                    for (int s = 0; s < m; ++s) {
                        AT(Vm, s) = (sc >= 0) ? __ldcs(a.V_m + (size_t)s * B + sc) : 1.0;
                        AT(Va, s) = (sc >= 0) ? __ldcs(a.V_a + (size_t)s * B + sc) : 0.0;
                        AT(Pl, s) = (sc >= 0) ? __ldcs(a.P + (size_t)s * B + sc) : 0.0;
                        AT(Ql, s) = (sc >= 0) ? __ldcs(a.Q + (size_t)s * B + sc) : 0.0;
                    }
                    stat[lane] = (sc >= 0 && !a.step_only) ? a.status[sc] : 0;
                } else if (pendF) {
                    for (int i = 1; i < m; ++i) {                 // x_new = x + delta (HG:476-485)
                        AT(Va, i) += AT(DXF, i - 1);
                        if (i >= c) AT(Vm, i) += AT(DXF, nth + (i - c));
                    }
                }
                for (int s = 0; s < m; ++s) {
                    const double2 e = sincos_ol(AT(Va, s));
                    const double vm = AT(Vm, s);
                    ATV(s) = make_double2(vm * e.x, vm * e.y);                        // V = V_m e^{j theta} (HG:403)
                    
                }
            } else {
                if (isnew) {
                    for (int s = m + warp; s < nH; s += CW) {
                        if (sc >= 0 && (a.step_only || s < n)) {
                            AT(Vm, s) = __ldcs(a.V_m + (size_t)s * B + sc);
                            AT(Va, s) = __ldcs(a.V_a + (size_t)s * B + sc);
                        } else {
                            AT(Vm, s) = (sc >= 0) ? 0.1 : 1.0;     // flat start of the harmonics (HG:183)
                            AT(Va, s) = 0.0;
                        }
                    }
                    // I_N and w_N of a refilled lane are not needed before phases B / C: fetch them
                    // with asynchronous global->shared copies (LDGSTS) that complete behind the
                    // sincos work instead of stalling the whole tile on DRAM latency every round.
                    // group 0: I_N rows and the w_N rows the border system reads (z < q); group 1: rest
                    if (sc >= 0) {
                        for (int u = warp; u < q * H; u += CW) {
                            const double* src = reinterpret_cast<const double*>(a.I_N + (size_t)u * B + sc);
                            cp_async_f64(&AT(INre, u), src);
                            cp_async_f64(&AT(INim, u), src + 1);
                        }
                        for (int z = warp; z < q; z += CW) {
                            const double* src = reinterpret_cast<const double*>(a.wN + (size_t)z * B + sc);
                            cp_async_f64(&AT(Wre, z), src);
                            cp_async_f64(&AT(Wim, z), src + 1);
                        }
                    } else {
                        for (int u = warp; u < q * H; u += CW) { AT(INre, u) = 0.0; AT(INim, u) = 0.0; }
                        for (int z = warp; z < nZ; z += CW) { AT(Wre, z) = 0.0; AT(Wim, z) = 0.0; }
                    }
                }
                cp_async_commit();
                if (isnew && sc >= 0) {
                    for (int z = warp; z < nZ; z += CW) {
                        if (z < q) continue;
                        const double* src = reinterpret_cast<const double*>(a.wN + (size_t)z * B + sc);
                        cp_async_f64(&AT(Wre, z), src);
                        cp_async_f64(&AT(Wim, z), src + 1);
                    }
                }
                cp_async_commit();
                if constexpr (D::n != 0) {
                    // all sin/cos of the warp's rows as ONE branch-free group (hpf_device.cuh): the
                    // dependency chains of the rows interleave, half the instructions of the library
                    // routine, no per-row branch
                    double ang[ZR], sn_[ZR], cs_[ZR];
#pragma unroll
                    for (int r = 0; r < ZR; ++r) {
                        const int s = m + warp + r * CW;
                        ang[r] = (s < nH) ? AT(Va, s) : 0.0;
                    }
                    sincos_group<ZR>(ang, sn_, cs_);
#pragma unroll
                    for (int r = 0; r < ZR; ++r) {
                        const int s = m + warp + r * CW;
                        if (s < nH) {
                            const double vm = AT(Vm, s);
                            ATV(s) = make_double2(vm * cs_[r], vm * sn_[r]);
                            
                        }
                    }
                } else {
                    for (int s = m + warp; s < nH; s += CW) {
                        const double2 e = sincos_ol(AT(Va, s));
                        const double vm = AT(Vm, s);
                        ATV(s) = make_double2(vm * e.x, vm * e.y);
                        
                    }
                }
                cp_async_wait<1>();                 // group 0 (I_N, first w_N rows) has landed
            }
        }
        __syncthreads();
        // ================= B: mismatch rows (HG:360-388); border system =================
        {
            double mx = 0.0;
            if (!border) {
                // heavy rows first: nonlinear buses, (Y_h V_h)_i + I_N - sum_p Y_N[h][p] V_p,i
                row_loop<HR>(warp, q * H, CW, [&](int u) {
                    const int k = u / H, h = u - k * H, i = m + k, s = h * n + i;
                    const int dev = net.dev_of_nl[k];
                    double2 acc;
                    if (net.coupled) {
                        const double2* row = sYN + ((size_t)dev * H + h) * H;
                        acc = make_double2(0.0, 0.0);
                        for (int pp = 0; pp < H; ++pp) {
                            const int t2 = pp * n + i;
                            acc = cfma(acc, row[pp], ATV(t2));
                        }
                    } else {
                        acc = cmul(sYN[(size_t)dev * H + h], ATV(s));
                    }
                    const double2 inj = make_double2(AT(INre, u) - acc.x, AT(INim, u) - acc.y);
                    AT(IJre, u) = inj.x; AT(IJim, u) = inj.y;
                    const double2* Yrow = sY + ((size_t)h * n + i) * n;
                    double2 f = make_double2(0.0, 0.0);
                    for (int j = 0; j < n; ++j) {
                        const int t2 = h * n + j;
                        f = cfma(f, Yrow[j], ATV(t2));
                    }
                    f = cadd(f, inj);
                    const double v1 = fabs(f.x), v2 = fabs(f.y);      // s >= m >= c: both parts are rows
                    const double v = (v2 != v2 || v2 > v1) ? v2 : v1;
                    mx = (v != v || v > mx) ? v : mx;
                });
                // light rows: linear buses at the harmonics h >= 1 (index)
                const int nlin = m * (H - 1);
                row_loop<LR>(warp, nlin, CW, [&](int t) {
                    const int h = 1 + t / m, i = t - (h - 1) * m;
                    const double2* Yrow = sY + ((size_t)h * n + i) * n;
                    double2 f = make_double2(0.0, 0.0);
                    for (int j = 0; j < n; ++j) {
                        const int t2 = h * n + j;
                        f = cfma(f, Yrow[j], ATV(t2));
                    }
                    const double v1 = fabs(f.x), v2 = fabs(f.y);
                    const double v = (v2 != v2 || v2 > v1) ? v2 : v1;
                    mx = (v != v || v > mx) ? v : mx;
                });
            } else {
                // ---- border warp: power mismatch of the linear buses (HG:372-380) ----
                for (int i = 0; i < m; ++i) {
                    const double2* Yrow = sY + (size_t)i * n;
                    double2 f = make_double2(0.0, 0.0);
                    for (int j = 0; j < n; ++j) f = cfma(f, Yrow[j], ATV(j));
                    AT(I1re, i) = f.x; AT(I1im, i) = f.y;
                    if (i == 0) continue;                            // slack: no row
                    const double2 v = ATV(i);
                    const double2 sl = cmul(v, make_double2(f.x, -f.y));
                    const double2 fs = make_double2(AT(Pl, i) + sl.x, AT(Ql, i) + sl.y);
                    AT(FSre, i) = fs.x; AT(FSim, i) = fs.y;
                    double v1 = fabs(fs.x);
                    if (i >= c) {
                        const double v2 = fabs(fs.y);
                        v1 = (v2 != v2 || v2 > v1) ? v2 : v1;
                    }
                    mx = (v1 != v1 || v1 > mx) ? v1 : mx;
                }
                // ---- border system for x_F: every entry is accumulated in registers ----
                const int w = nx + 1;
                for (int i = 1; i < m; ++i) {
                    const double rvi = 1.0 / AT(Vm, i);
                    const double2 vi = ATV(i);
                    const double2 ei = make_double2(vi.x * rvi, vi.y * rvi);         // V / V_m (HG:455)
                    const double2 i1 = make_double2(AT(I1re, i), AT(I1im, i));
                    const double2 jvi = cmulj(vi);
                    const int rr = i - 1, ri = nth + (i - c);
                    const bool has_im = (i >= c);
                    for (int col = 0; col <= nx; ++col) {
                        double2 e;
                        const bool is_rhs = (col == nx);
                        const bool is_v = (col >= nth);
                        const int j = is_rhs ? 0 : (is_v ? c + (col - nth) : col + 1);
                        double2 vj = make_double2(0.0, 0.0), ej = vj;
                        if (is_rhs) {
                            e = make_double2(-AT(FSre, i), -AT(FSim, i));
                        } else {
                            const double2 y = sY[(size_t)i * n + j];
                            const double rvj = 1.0 / AT(Vm, j);
                            vj = ATV(j);
                            ej = make_double2(vj.x * rvj, vj.y * rvj);
                            if (is_v) {                               // dS_i/dV_m,j  (HG:458-459)
                                e = cmul(vi, cconj(cmul(y, ej)));
                                if (i == j) e = cadd(cmul(ei, cconj(i1)), e);
                            } else {                                  // dS_i/dtheta_j (HG:457)
                                const double2 yv = cmul(y, vj);
                                e = cmul(jvi, cconj((i == j) ? csub(i1, yv) : cneg(yv)));
                            }
                        }
                        // fundamental nonlinear buses, eliminated through u_Z1 = u0 - G T_F x_F
                        for (int k = 0; k < q; ++k) {
                            const int bk = m + k;
                            const double2 y = sY[(size_t)i * n + bk];
                            if (y.x == 0.0 && y.y == 0.0) continue;
                            const double vmb = AT(Vm, bk), rvb = 1.0 / vmb;
                            const double2 vb = ATV(bk);
                            const double2 eb = make_double2(vb.x * rvb, vb.y * rvb);
                            const double2 ak = cmul(jvi, cconj(cneg(cmul(y, vb))));    // dS_i/dtheta_b
                            const double2 vk = cmul(vi, cconj(cmul(y, eb)));           // dS_i/dV_m,b
                            double2 uu;
                            if (is_rhs) {            // u0 of row z = k (closed form)
                                uu = make_double2(vb.x + AT(Wre, k), vb.y + AT(Wim, k));
                                for (int i2 = 0; i2 < m; ++i2)
                                    uu = cfma(uu, sG[(size_t)k * m + i2], ATV(i2));
                                uu = cneg(uu);
                            } else {                 // column of G T_F: G (j V_j) or G E_j
                                uu = cmul(sG[(size_t)k * m + j], is_v ? ej : cmulj(vj));
                            }
                            const double2 ce = cmul(cconj(eb), uu);
                            const double dth = ce.y * rvb, dvm = ce.x;
                            e.x -= ak.x * dth + vk.x * dvm;
                            e.y -= ak.y * dth + vk.y * dvm;
                        }
                        AT(M, rr * w + col) = e.x;
                        if (has_im) AT(M, ri * w + col) = e.y;
                    }
                }
                int badp = 0;
                double xs[4] = {0.0, 0.0, 0.0, 0.0};
                switch (nx) {
                    case 0: break;
                    case 1: badp = lane_gauss_solve_reg<1>(M, lane, xs); break;
                    case 2: badp = lane_gauss_solve_reg<2>(M, lane, xs); break;
                    case 3: badp = lane_gauss_solve_reg<3>(M, lane, xs); break;
                    case 4: badp = lane_gauss_solve_reg<4>(M, lane, xs); break;
                    default: badp = lane_gauss_solve(M, nx, lane); break;
                }
                if (nx <= 4) { for (int t = 0; t < nx; ++t) AT(DXF, t) = xs[t]; }
                else { for (int t = 0; t < nx; ++t) AT(DXF, t) = AT(M, t * w + nx); }
                if (badp) stat[lane] |= 0x200;
                AT(UFre, 0) = 0.0; AT(UFim, 0) = 0.0;
                for (int i = 1; i < m; ++i) {
                    const double dth = AT(DXF, i - 1);
                    const double dvm = (i >= c) ? AT(DXF, nth + i - c) : 0.0;
                    const double rvi = 1.0 / AT(Vm, i);
                    const double2 vi = ATV(i);
                    AT(UFre, i) = -vi.y * dth + (vi.x * rvi) * dvm;      // u_F = (j V_i) dtheta + E_i dV_m
                    AT(UFim, i) = vi.x * dth + (vi.y * rvi) * dvm;
                }
            }
            AT(red, warp) = mx;
            if (!border) cp_async_wait<0>();        // remaining w_N rows (used in phase C by this thread)
        }
        __syncthreads();
        // ================= C: decisions, finished lanes, update, refill =================
        double err = 0.0;
        {
            bool bad = false;
#pragma unroll
            for (int w2 = 0; w2 < NW; ++w2) {
                const double v = AT(red, w2);
                bad |= (v != v);
                err = fmax(err, v);
            }
            if (bad) err = CUDART_NAN;
        }
        const bool active = sc >= 0;
        const bool cont = active && (err > a.thresh_h) && (itv < a.max_h);
        const bool step = a.step_only ? active : cont;
        const bool done = active && !cont && !a.step_only;
        if (__ballot_sync(0xffffffffu, active) == 0u) break;          // uniform over the CTA
        const unsigned donemask = __ballot_sync(0xffffffffu, done);
        if (donemask) {
            // post-processing (HG:547-549) + write-out: finished lanes are few (about 2 of 32
            // per round), so each one is written by ONE warp with its 32 lanes over the rows
            unsigned dm = donemask;
            int jd = 0;
            while (dm) {
                const int l = __ffs(dm) - 1;
                dm &= dm - 1;
                if ((jd++ % NW) != warp) continue;
                const int scl = scen[l];
                for (int s = lane; s < nH; s += 32) {
                    double vm = Vm[s * HPF_T + l], va = Va[s * HPF_T + l];
                    if (!(a.flags & HPF_SOLVE_RAW)) {
                        if (vm < 0.0) va += CUDART_PI;
                        va = mod_twopi(va);
                        if (vm < 0.0) vm = -vm;
                    }
                    a.V_m[(size_t)s * B + scl] = vm;
                    a.V_a[(size_t)s * B + scl] = va;
                }
                if (a.I_inj)
                    for (int u = lane; u < q * H; u += 32)
                        a.I_inj[(size_t)u * B + scl] = make_double2(IJre[u * HPF_T + l], IJim[u * HPF_T + l]);
            }
        }
        if (!border) {
            // u_z = -V_z - sum_i G[z][i] (V_i + u_F,i) - w_N,z ; polar conversion; update
            row_loop<ZR>(warp, nZ, CW, [&](int z) {
                const int s = z + m;
                const double2 vs = ATV(s);
                double2 acc = make_double2(vs.x + AT(Wre, z), vs.y + AT(Wim, z));
                for (int i = 0; i < m; ++i) {
                    const double2 vf = ATV(i);
                    const double2 tot = make_double2(vf.x + AT(UFre, i), vf.y + AT(UFim, i));
                    acc = cfma(acc, sG[(size_t)z * m + i], tot);
                }
                // conj(E) u with E = V / V_m:  dV_m = Re(conj(V) u) / V_m,  dtheta = Im(conj(V) u) / V_m^2
                const double2 cv = cmul(make_double2(vs.x, -vs.y), cneg(acc));
                const double vm = AT(Vm, s), rv = 1.0 / vm;
                const double dvm = cv.x * rv, dth = (cv.y * rv) * rv;
                if (a.step_only) {
                    if (sc >= 0) {
                        a.dx_out[(size_t)(s - 1) * B + sc] = -dth;
                        a.dx_out[(size_t)((nH - 1) + s - c) * B + sc] = -dvm;
                    }
                } else if (step) {
                    AT(Va, s) += dth;
                    AT(Vm, s) = vm + dvm;
                }
            });
        } else {
            if (a.step_only) {
                if (sc >= 0)
                    for (int i = 1; i < m; ++i) {
                        a.dx_out[(size_t)(i - 1) * B + sc] = -AT(DXF, i - 1);
                        if (i >= c) a.dx_out[(size_t)((nH - 1) + i - c) * B + sc] = -AT(DXF, nth + i - c);
                    }
            } else {
                // status words, iteration counters, refill (only this warp touches itc/stat/fnew)
                int* scen_next = scen2 + (cur ^ 1) * HPF_T;
                int nsc = sc;
                if (done) {
                    int st = stat[lane] & 0xff;
                    if ((stat[lane] & 0x200) && st == HPF_ST_CONVERGED) st = HPF_ST_SINGULAR;
                    if (itv >= a.max_h && st == HPF_ST_CONVERGED) st = HPF_ST_MAXITER;
                    if (!(err < CUDART_INF)) st = HPF_ST_NONFINITE;     // NaN or Inf mismatch
                    a.n_iter_h[sc] = itv;
                    a.err_h[sc] = err;
                    a.status[sc] = st;
                }
                if (a.hist_h && active) a.hist_h[(size_t)itv * B + sc] = err;
                if (step) itc[lane] = itv + 1;
                fnew[lane] = 0;
                pendF = step;
                if (donemask) {
                    int base = 0;
                    if (lane == 0) base = atomicAdd(a.work_counter, __popc(donemask));
                    base = __shfl_sync(0xffffffffu, base, 0);
                    if (done) {
                        const int idx = base + __popc(donemask & ((1u << lane) - 1u));
                        nsc = ((size_t)idx < B) ? idx : -1;
                        itc[lane] = 0;
                        fnew[lane] = 1;
                        stat[lane] = 0;
                    }
                }
                scen_next[lane] = nsc;
            }
        }
        if (a.step_only) break;
        __syncthreads();
        cur ^= 1;
    }
#undef AT
#undef ATV
}
