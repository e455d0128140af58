/*
 * hpf_b200.h - C ABI of the B200-native batched harmonic power-flow solve path.
 *
 * Drop-in boundary for the solve path of the reference's
 *   "Harmonic Power Flow/hcne_generalized.py"  (HG below, cited as HG:line).
 * The reference has no FFI/plugin interface (it is a flat Python script), so the
 * boundary is the function-level API of HG; each entry point below names the HG
 * function(s) it replaces.  The Python host layer (harmonic_power_flow_b200/)
 * binds these symbols with ctypes and mirrors the HG function names.
 *
 * Conventions
 *  - Plain C: pointers and sizes only, no C++/torch types.  Return 0 on success,
 *    a negative HPF_E_* code on failure; hpf_last_error() gives the text.
 *    Nothing throws across the ABI.  Per-scenario NUMERICAL outcomes are
 *    reported in status[B] (HPF_ST_*), never in the return code.
 *  - "host" pointers are read during the call and copied.  "device" pointers are
 *    caller-owned CUDA device memory on the handle's device; the handle owns only
 *    the network, Norton-equivalent tables, Y(h) and small scratch.
 *  - Every kernel entry point enqueues its work on `stream` (a cudaStream_t passed
 *    as void*, NULL = legacy default stream) and returns without waiting for it.
 *    LAZY SET-UP does synchronise, once: the first hpf_solve / hpf_newton_step /
 *    hpf_norton_wn / hpf_struct_info after a network, device-table or Y(h) change
 *    builds the structured-step operators (device allocations, a stream
 *    synchronisation and a small read-back); the first use of the one-thread-per-
 *    scenario mismatch kernel mirrors Y(h) to the host; a batch larger than any
 *    before it grows the handle's scratch (device synchronisation + reallocation).
 *    hpf_prepare() does all of that up front, after which solves of up to B_max
 *    scenarios neither allocate nor synchronise (and may be captured into a CUDA
 *    graph).  hpf_destroy() and the *_host calls synchronise by design.
 *  - One kernel sequence in flight per handle: the work queue, the w_N scratch and
 *    the LU workspaces live in the handle, so a call arriving on a different stream
 *    than the previous one is ordered after it on the device (event wait; the host
 *    does not block).  A stream under CUDA-graph capture is left alone.
 *  - All arithmetic is IEEE FP64.  Complex values are interleaved (re, im)
 *    doubles (numpy/torch complex128).
 *  - Batch arrays are BATCH-INNERMOST: element (i, b) of an [n, B] array is at
 *    i*B + b, so a warp touching consecutive scenarios issues one coalesced
 *    128-bit-vectorisable request.
 *  - Symbols (HG:11-17,122-127): n buses; m = 0-based index of the first
 *    nonlinear bus; q = n - m; c = 1 + number of PV buses; H harmonic orders
 *    including the fundamental; stacked index s = h*n + i (harmonic-major);
 *    N = 2nH - 1 - c unknowns of the harmonic Newton system,
 *    Nf = 2n - 1 - c of the fundamental one.  Bus order: slack, PV.., PQ..,
 *    nonlinear.. (HG:83).
 *  - Not thread-safe per handle; use one handle per GPU / per host thread.
 */
#ifndef HPF_B200_H
#define HPF_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hpf_handle hpf_t;

/* return codes */
#define HPF_OK              0
#define HPF_E_INVALID      -1   /* bad argument / call order                      */
#define HPF_E_CUDA         -2   /* CUDA runtime error (text in hpf_last_error)    */
#define HPF_E_UNSUPPORTED  -3   /* dimensions exceed what the kernels support     */
#define HPF_E_NOMEM        -4   /* out of device memory: the text names the call and the buffer; other CUDA errors stay HPF_E_CUDA */

/* per-scenario status word (status[B]) */
#define HPF_ST_CONVERGED    0
#define HPF_ST_MAXITER      1   /* n_iter == max_iter in either stage (HG:273,558) */
#define HPF_ST_SINGULAR     2   /* zero pivot met in a Newton step                 */
#define HPF_ST_NONFINITE    3   /* NaN/Inf in the mismatch or the state            */

/* ABI version of this header: bumped on any signature change. */
#define HPF_ABI_VERSION 12
int hpf_abi_version(void);

/* Lifetime.  `device` is the CUDA ordinal the handle is bound to. */
int hpf_create(hpf_t** out, int device);
int hpf_destroy(hpf_t* h);
/* Text of the last error on this handle (h == NULL: last create failure). */
const char* hpf_last_error(const hpf_t* h);

/*
 * Network in per-unit, exactly what init_network() yields (HG:45-128):
 * harmonics[H] orders with harmonics[0] == 1 (HG:584); lines with the CSV's
 * 1-BASED fromID/toID and R, X, G, B (HG:57-60); X_sh[n] (HG:92).  Host pointers.
 */
int hpf_set_network(hpf_t* h, int n, int m, int c, int H, const int* harmonics,
                    int L, const int* from_id, const int* to_id,
                    const double* R, const double* X, const double* G, const double* B,
                    const double* X_sh);

/*
 * Norton-equivalent admittances, what import_Norton_Equivalents() yields
 * (HG:278-310) minus I_N (which is per scenario): n_dev device types,
 * Y_N complex [n_dev, H, H] row-major (row = harmonic of the current, column =
 * harmonic of the voltage, HG:304) when coupled, else [n_dev, H] (HG:308);
 * dev_of_nl_bus[q] maps nonlinear bus m+k to its device type.  Host pointers.
 */
int hpf_set_devices(hpf_t* h, int n_dev, int coupled, const double* Y_N,
                    const int* dev_of_nl_bus);

/*
 * Optional transformer branches for the next hpf_build_Y (SURVEY 8(f) next-3): tap ratio tau[L]
 * and phase shift phase_shift_deg[L] per line, the branch model of the reference's
 * "Fundamental Power Flow/pi_trafo_pf_test.py":117-145 (off-diagonals divided by
 * tau e^{-+j phi}; the pi-shunt of a to-side match divides the accumulated diagonal by tau^2).
 * Host pointers, copied; both NULL restores plain lines (HG:132-171).  hpf_set_network clears them.
 */
int hpf_set_transformers(hpf_t* h, const double* tau, const double* phase_shift_deg);

/*
 * Opt-in corrections of two quirks of build_admittance_matrices (default 0 = reference behaviour,
 * which every parity test uses): HPF_Y_FIX_SHUNT_INDEX puts the pi-line shunt (G + jhB)/2 on
 * the buses the line actually connects (HG:163-168 compares the 1-based ID with the 0-based
 * row, so it lands one bus too low); HPF_Y_SUM_PARALLEL adds parallel branches instead of
 * letting the later one overwrite (HG:150-155).  Takes effect at the next hpf_build_Y.
 */
#define HPF_Y_FIX_SHUNT_INDEX 1
#define HPF_Y_SUM_PARALLEL    2
int hpf_set_y_options(hpf_t* h, int flags);

/*
 * Kernel 1 - per-harmonic bus admittance assembly.  Replaces
 * build_admittance_matrices() (HG:132-171), including its quirks (assignment of
 * parallel lines, shunt only for h != 1, pi-shunt index off-by-one).
 * Result is kept in the handle; if Y_out != NULL it is also written there
 * (device, complex [H, n, n]).
 */
int hpf_build_Y(hpf_t* h, double* Y_out, void* stream);

/*
 * Use a caller-supplied admittance table instead of building it: Y complex [H, n, n]
 * (host).  This is what pf(Y, buses) of the reference takes (HG:244,255).  The host waits
 * for the handle's previous kernel sequence before it copies, so a solve still in flight on
 * any stream finishes on the table it was issued with.
 */
int hpf_set_Y(hpf_t* h, const double* Y);

/*
 * Optional: run every lazy set-up NOW for batches of up to B_max scenarios - the structured-step
 * operators of the network, the handle's scratch (w_N, LU workspaces, scenario state slabs) - by
 * solving B_max all-zero scenarios with zero iterations.  Synchronises `stream`.  Afterwards
 * hpf_solve / hpf_mismatch / ... with B <= B_max neither allocate nor synchronise.
 */
int hpf_prepare(hpf_t* h, int B_max, void* stream);

/* hpf_solve flags */
#define HPF_SOLVE_RAW   1 /* skip the post-processing of HG:547-549: return the raw iterate */
#define HPF_SOLVE_DENSE 2 /* force the dense-LU Newton step (default: structured step when the
                             network admits it, see hpf_struct_info) */

/*
 * Whole solve for B scenarios: pf() (HG:244-275) followed by the harmonic
 * Newton-Raphson and post-processing of hpf() (HG:511-560), one fused
 * persistent kernel (mismatch, Jacobian, shared-memory LU, state update).
 *   in : P, Q [n, B] p.u.;  I_N complex [q, H, B] p.u.
 *   out: V_m, V_a [H, n, B] post-processed like HG:547-549 (|V|, angle in [0, 2pi))
 *        unless HPF_SOLVE_RAW;
 *        I_inj complex [q, H, B] = I_N - Y_N V at the solution (HG:313-323), may be NULL;
 *        n_iter_f, n_iter_h, status int32 [B]; err_h [B] final inf-norm mismatch;
 *        err_hist_f [max_iter_f + 1, B], err_hist_h [max_iter_h + 1, B] (may be NULL):
 *        the mismatch norm before each Newton step and after the last one (the
 *        reference's err_t / err_h_t dicts, HG:258,264,533,541); unused tail = NaN.
 * Loops are exactly `while err > thresh and n_iter < max_iter` (HG:259,536).
 */
int hpf_solve(hpf_t* h, int B, const double* P, const double* Q, const double* I_N,
              double thresh_f, int max_iter_f, double thresh_h, int max_iter_h, int flags,
              double* V_m, double* V_a, double* I_inj,
              int* n_iter_f, int* n_iter_h, double* err_h, int* status,
              double* err_hist_f, double* err_hist_h, void* stream);

/*
 * Same with HOST buffers (pageable or pinned): copies in, solves, copies out,
 * synchronises.  This is the call a reference-side binding would make.  Batches of
 * 8,192 scenarios and more are pipelined in growing chunks (4,096 / 8,192 / 12,288 /
 * 16,384 ... scenarios) over a copy-in, two compute and a copy-out stream; results do
 * not depend on the chunking (bit-identical to hpf_solve).
 */
int hpf_solve_host(hpf_t* h, int B, const double* P, const double* Q, const double* I_N,
                   double thresh_f, int max_iter_f, double thresh_h, int max_iter_h,
                   double* V_m, double* V_a, double* I_inj,
                   int* n_iter_f, int* n_iter_h, double* err_h, int* status);

/*
 * hpf_solve_host that ALSO leaves the results on the device (d* pointers: device memory, same
 * [rows, B] layouts) - for a caller that returns the results to its host AND feeds them to a
 * device-side consumer, e.g. the final NCCL gather of a multi-GPU run.  dI_inj may be NULL.
 */
int hpf_solve_host_keep(hpf_t* h, int B, const double* P, const double* Q, const double* I_N,
                        double thresh_f, int max_iter_f, double thresh_h, int max_iter_h,
                        double* V_m, double* V_a, double* I_inj,
                        int* n_iter_f, int* n_iter_h, double* err_h, int* status,
                        double* dV_m, double* dV_a, double* dI_inj, int* dn_iter_f, int* dn_iter_h,
                        double* derr_h, int* dstatus);

/*
 * Fundamental stage only: pf() (HG:244-275).  V_m, V_a [H, n, B] receive the flat
 * start (HG:174-184) with the h = 1 block replaced by the fundamental solution
 * (no post-processing, like HG:233-241).
 */
int hpf_fund_solve(hpf_t* h, int B, const double* P, const double* Q,
                   double thresh_f, int max_iter_f,
                   double* V_m, double* V_a, int* n_iter_f, double* err_f,
                   double* err_hist_f, void* stream);

/*
 * Kernel 2 - fused power/current mismatch, harmonic_mismatch() (HG:360-390) with
 * current_balance() (HG:326-357) and the Norton contraction I = I_N - Y_N V of
 * current_injections() (HG:313-323).
 *   in : V_m, V_a [H, n, B] (un-normalised iterate); P, Q [n, B]; I_N [q, H, B]
 *   out: f [N, B] (row order of HG:388), err [B] = ||f||_inf; I_inj [q,H,B] or NULL
 */
int hpf_mismatch(hpf_t* h, int B, const double* V_m, const double* V_a,
                 const double* P, const double* Q, const double* I_N,
                 double* f, double* err, double* I_inj, void* stream);

/*
 * Kernel 3 - harmonic Jacobian, build_harmonic_jacobian() (HG:401-473), dense FP64.
 *   out: J [B, hpf_jacobian_stride()] ; scenario b holds the N x N matrix
 *        row-major (same element order as the reference's J.toarray()) followed
 *        by padding up to the stride (a multiple of 2 doubles so that every
 *        matrix is 16-byte aligned for the bulk-copy engine).
 */
int hpf_jacobian(hpf_t* h, int B, const double* V_m, const double* V_a,
                 double* J, void* stream);
/* doubles between consecutive scenarios' matrices in hpf_jacobian/hpf_lu_solve */
long long hpf_jacobian_stride(const hpf_t* h);

/*
 * Kernel 4 - batched dense LU (partial pivoting, warp-shuffle pivot search) and
 * triangular solves in shared memory: dx = J^{-1} f, the linear algebra of
 * update_harmonic_state_vec() (HG:476-479).
 *   in : J [B, stride] as written by hpf_jacobian (not modified); f [N, B]
 *   out: dx [N, B]; info int32 [B] (0 ok, k+1 = zero pivot at step k)
 */
int hpf_lu_solve(hpf_t* h, int B, const double* J, const double* f,
                 double* dx, int* info, void* stream);

/*
 * Structured Newton step (the default strategy of hpf_solve when available): the
 * current-balance rows of J are A T with a CONSTANT complex operator
 * A = blockdiag Y(h) - scatter(Y_N) and the polar map T, so the step of HG:476-479 is
 * evaluated by block elimination with A_ZZ^{-1} (inverted once per network on the GPU)
 * plus a (2m-1-c)-sized dense system per scenario; mathematically the same dx = J^{-1} f.
 * hpf_struct_info: available = 1 if the strategy is set up for this network (0: falls back
 * to the dense LU: system too large for the tile kernel or A_ZZ singular); nZ = order of
 * A_ZZ; pivot_min/max = extreme pivot moduli of its Gauss-Jordan inversion.
 * hpf_newton_step: ONE step for given iterates, dx [N, B] with x_new = x - dx in the
 * reference's ordering [theta(1..nH-1), V_m(c..nH-1)] - comparable with hpf_lu_solve(J, f).
 */
int hpf_struct_info(hpf_t* h, int* available, int* nZ, double* pivot_min, double* pivot_max);
int hpf_newton_step(hpf_t* h, int B, const double* V_m, const double* V_a,
                    const double* P, const double* Q, const double* I_N,
                    double* dx, void* stream);

/*
 * The Norton contraction of the structured step for a whole batch: w_N = A_ZZ^{-1} I_N,Z = W_NL I_N,
 * complex [nZ, B] (nZ from hpf_struct_info; row z = stacked index s - m).  I_N enters the current
 * balance additively (current_injections / current_balance, HG:313-323,351-354), so this product is
 * the per-scenario constant of the harmonic Newton loop.  One complex GEMM [nZ x qH] [qH x B]: on the
 * FP64 tensor cores (DMMA) when it fills the machine, else on the CUDA-core FP64 pipe
 * ($HPF_WN_KERNEL=fma|dmma forces either; both kernels are kept for the A/B of the north star).
 *   in : I_N complex [q, H, B];  out: wN complex [nZ, B]
 */
int hpf_norton_wn(hpf_t* h, int B, const double* I_N, double* wN, void* stream);

/*
 * Post-processing after the path - get_THD() (HG:563-572): for every bus and scenario
 * THD_F = sqrt(sum_{order>=3} V_m^2) / V_m(order 1), THD_R = same / sqrt(sum_all V_m^2).
 *   in : V_m [H, n, B];  out: thd [2, n, B]  (plane 0 = THD_F, plane 1 = THD_R)
 */
int hpf_thd(hpf_t* h, int B, const double* V_m, double* thd, void* stream);

/*
 * Batch statistics of a solved batch, on the device: for a network of n buses and H orders the
 * R = n*H + 2n rows are  row h*n + i = V_m of order harmonics[h] at bus i (the V_m layout),
 * row n*H + i = THD_F of bus i, row n*H + n + i = THD_R of bus i (THD exactly as hpf_thd writes it).
 * A scenario is included when status[b] == HPF_ST_CONVERGED; status == NULL includes all of them;
 * n_valid = number included.
 *   in : V_m [H, n, B] (device), status [B] (device) or NULL, limits [R] (device) or NULL,
 *        quantiles [K] (host), 0 <= K <= HPF_STATS_MAX_Q, each in [0, 1]
 *   out: status_counts int[4] (device): scenarios per HPF_ST_* value ({B, 0, 0, 0} without status);
 *        stats [5 + K, R] doubles (device), one plane per statistic:
 *          0 mean, 1 population std (ddof 0, two passes: mean, then squared deviations), 2 min, 3 max,
 *          4 exceed = included scenarios with x > limits[r] (0 without limits or for limit +inf),
 *          5 + k = quantile p_k: the included value of rank max(1, ceil(p_k * n_valid)) in ascending
 *          order (nearest rank, numpy's method="inverted_cdf"; p = 0 gives min, p = 1 max) - an exact
 *          order statistic, no interpolation.
 *        Values are ordered by their bit patterns (-0 below +0).  n_valid == 0 (or B == 0): planes 0-3
 *        and the quantiles are NaN, exceed 0.
 * The same inputs give the same bits on every call and stream (no floating-point atomics; sums run in
 * an order fixed by B and the launch shape).  Uses the handle's scratch (THD rows), so it goes through
 * the handle's ordering like hpf_solve; the first call with a larger B than before grows that scratch
 * (device synchronisation + reallocation) like the other grow-only buffers.
 */
#define HPF_STATS_MAX_Q 16
int hpf_batch_stats(hpf_t* h, int B, const double* V_m, const int* status,
                    int K, const double* quantiles, const double* limits,
                    int* status_counts, double* stats, void* stream);

/*
 * hpf_solve_host that returns the statistics of hpf_batch_stats instead of the per-scenario phasors:
 * copies the inputs in (chunk-pipelined like hpf_solve_host), solves, reduces on the device and copies
 * back only status_counts int[4] and stats [5 + K, R] - a few KB instead of V_m, V_a and I_inj.  Every
 * buffer here is HOST memory, limits [R] (or NULL) included; quantiles and limits mean what they mean
 * in hpf_batch_stats.  n_iter_f, n_iter_h, err_h,
 * status [B] may each be NULL (then not copied back).  Bit-identical to hpf_batch_stats over the V_m and
 * status that hpf_solve_host_keep leaves on the device for the same inputs and chunk plan - and so, where
 * the chunked solve equals hpf_solve (the 4-bus paths), to hpf_solve followed by hpf_batch_stats.
 * Synchronises.
 */
int hpf_solve_host_stats(hpf_t* h, int B, const double* P, const double* Q, const double* I_N,
                         double thresh_f, int max_iter_f, double thresh_h, int max_iter_h,
                         int K, const double* quantiles, const double* limits,
                         int* status_counts, double* stats,
                         int* n_iter_f, int* n_iter_h, double* err_h, int* status);

/*
 * Post-processing after the path: per-bus current spectra I[h][i] = sum_j Y(h)[i][j] V[h][j] (what
 * the reference logs in the I_log.json layout: harmonic x bus, real and imaginary part).
 *   in : V_m, V_a [H, n, B];  out: I_bus complex [H, n, B]
 */
int hpf_bus_currents(hpf_t* h, int B, const double* V_m, const double* V_a, double* I_bus, void* stream);

/*
 * Before the path - Norton-equivalent extraction from simulated measurements, the arithmetic of
 * the reference's "Circuit Simulation/NE_from_sim.py" (NE): uncoupled two-point equivalents
 * (NE:86-118) and the coupled equivalent (NE:141-173: one (N+1) x (N+1) complex system with N
 * right-hand sides per device), for D devices / operating points at once.  Needs no network
 * (hpf_create only).  All pointers device memory, complex128 interleaved, K = N - 1 supply
 * harmonics, frequency index 0 = fundamental:
 *   in : Vf [D, 2]        fundamental supply phasor of the two fundamental-only measurements
 *        Vh [D, 2, K]     harmonic supply phasor, magnitude set 1 / 2, per supply frequency
 *        I_f [D, 2, N]    injected-current spectra of the fundamental-only measurements
 *        I_h [D, 2, K, N] spectra with the harmonic source at frequency k+1, magnitude set 1 / 2
 *   out: Y_N_c [D, N, N] (row = harmonic of the current, column = harmonic of the voltage),
 *        I_N_c [D, N], Y_N_uc [D, N], I_N_uc [D, N]; info int32 [D] (0, or k+1: zero pivot)
 */
int hpf_ne_extract(hpf_t* h, int D, int N, const double* Vf, const double* Vh, const double* I_f,
                   const double* I_h, double* Y_N_c, double* I_N_c, double* Y_N_uc, double* I_N_uc,
                   int* info, void* stream);

/*
 * Per-kernel device timing of hpf_solve (for roofline accounting): when enabled, CUDA events
 * are recorded on the launch stream around each kernel of a solve.  hpf_last_kernel_ms
 * waits for the last solve and returns ms[0] = fundamental-stage kernel, ms[1] = harmonic
 * kernel (structured strategy) or ms[0] = 0, ms[1] = fused kernel (dense strategy).
 */
int hpf_set_profiling(hpf_t* h, int enabled);
int hpf_last_kernel_ms(hpf_t* h, double* ms /* [2] */);

/* Dimensions derived by hpf_set_network (0 before it). */
int hpf_dim_N(const hpf_t* h);
int hpf_dim_Nf(const hpf_t* h);

/*
 * Number of kernel launches this handle has issued since creation (each CUDA
 * kernel launch of this library counts 1).  Used by bench.py for gpu_launches.
 */
long long hpf_launch_count(const hpf_t* h);

/*
 * Which kernels the last hpf_solve / hpf_solve_host of this handle ran for the harmonic
 * stage (HG:531-542; diagnostics for tests and bench.py): 0 none yet, 1 lane-per-scenario
 * tile / one-warp-per-harmonic kernels (small networks), 2 one CTA per scenario, state in
 * shared memory, 3 one CTA per scenario, state in global memory (large networks, small
 * batches), 4 lock-step batched rounds (large networks: batched tensor-core LU of the
 * border systems, G products as complex GEMMs), 5 dense Jacobian + LU (HPF_SOLVE_DENSE
 * or structured set-up not available).
 */
int hpf_last_solve_path(const hpf_t* h);

#ifdef __cplusplus
}
#endif
#endif /* HPF_B200_H */
