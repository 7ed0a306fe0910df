/* ustfwi.h -- C ABI of libustfwi.so: B200 (sm_100a) frequency-domain Helmholtz
 * forward/adjoint solves for ring-array FWI plus the adjoint-state gradient.
 *
 * This is the drop-in boundary for the ONE hot path of Alighieri1231/WaveformInversionUST
 * (paths below are relative to the reference repo):
 *   - Final_python/solve_helmholtz.py:21-101   solve_helmholtz(x,y,vel,src,f,a0,L_PML,adjoint)
 *   - Final_python/solve_helmholtz.py:85-93    the jax.pure_callback -> scipy spsolve seam
 *   - Final_python/fwi_loss_function.py:29-103 fwi_loss_function(...) (extended to (loss, grad))
 *   - Final_python/nonlinearcg.py:213-265      forward, source estimate, residual, adjoint, gradient
 *   - Final_python/nonlinearcg.py:268-301      NCG direction, perturbation solve, step (ust_ncg_*)
 *
 * Conventions
 *   - plain C, no exceptions cross the boundary; every call returns 0 on success, non-zero on
 *     failure, and ust_last_error() returns a thread-local message.
 *   - "dev" pointers are CUDA device pointers owned by the caller; "host" pointers are host memory.
 *   - complex numbers are interleaved (re, im); real type is float for UST_C64, double for UST_C128.
 *   - unknown ordering is the reference's: row-major node index y*Nx + x (solve_helmholtz.py:166-167);
 *     a multi-RHS array is (Ny*Nx, nrhs) row-major, source index fastest (solve_helmholtz.py:78,101).
 *   - all device work is enqueued on the cudaStream_t handed in (passed as void*); no device-wide
 *     synchronisation happens inside unless the function name ends in _host or _get_.
 *   - the plan owns factor storage and workspaces; nothing is allocated on the hot path (the _host entry points
 *     allocate their staging buffers on first use).
 *   - the _host entry points return 2 when a block inversion met a zero / non-finite pivot (the analogue of SciPy's
 *     MatrixRankWarning); device entry points record it in the flag read by ust_get_status.
 */
#ifndef USTFWI_H
#define USTFWI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ust_plan ust_plan;

enum { UST_C64 = 0, UST_C128 = 1 };
enum { UST_STENCIL_PYTHON = 0, UST_STENCIL_MATLAB = 1 }; /* SURVEY.md Appendix A.3 */
enum { UST_ENGINE_AUTO = 0, UST_ENGINE_SIMT = 1, /* 2: first tcgen05 engine of round 1, removed (missed the 1e-5 bar) */ UST_ENGINE_TC2 = 3,
       UST_ENGINE_TC2H = 4 /* ust_test_cgemm only: the 128 x 64-tile form of TC2 that the Gauss-Jordan kernels use */ };
/* SIMT: CUDA-core tile engine, FP32 FMA / FP64 mma.sync (the only engine for complex128).
 * TC2: tcgen05 fed by TMA from operands split once in HBM, leading products drained to FP32 registers (complex64;
 *      what AUTO selects). */

typedef struct ust_plan_desc {
    int nx, ny;       /* grid size (x.size, y.size of solve_helmholtz.py:27) */
    int dtype;        /* UST_C64 | UST_C128 */
    int max_freq;     /* frequencies factorised and swept concurrently on this GPU */
    int max_nrhs;     /* largest number of right-hand-side columns per solve */
    int device;       /* CUDA device ordinal */
    int stencil;      /* UST_STENCIL_* */
    int engine;       /* UST_ENGINE_* : block-GEMM engine for factor/sweeps */
    int fwi_buffers;  /* non-zero: also allocate wavefield buffers for ust_fwi_* (2 x max_freq x N x max_nrhs) */
} ust_plan_desc;

/* Library / error reporting. */
const char* ust_last_error(void);
const char* ust_version(void);

/* Plan lifetime.  Replaces nothing in the reference (it has no persistent state: the matrix is
 * rebuilt and refactorised on every solve_helmholtz call, nonlinearcg.py:213,263,279). */
int ust_plan_create(const ust_plan_desc* desc, ust_plan** out);
int ust_plan_destroy(ust_plan* plan);
size_t ust_plan_device_bytes(const ust_plan* plan);

/* Frequencies of one ust_factor / ust_fwi_* call are processed as `ngroups` independent launch chains on separate
 * streams inside the plan (default 2; 1 = a single chain; results are bit-identical).  No reference counterpart:
 * the reference handles one frequency at a time (fwi_script.py:24). */
int ust_plan_set_groups(ust_plan* plan, int ngroups);

/* Grid + PML: x (nx doubles), y (ny doubles) host arrays, a0, L_PML as in
 * solve_helmholtz.py:22-60 (h = mean(diff(x)), g = mean(diff(y))/h, half-grid PML profiles). */
int ust_plan_set_grid(ust_plan* plan, const double* x_host, const double* y_host, double a0, double L_pml);

/* Acquisition: one-hot source node of each transmitter (fwi_script.py:72-74), receiver node of every
 * ring element (row-major y*Nx+x; the reference's column-major ind_matlab, fwi_script.py:68, is
 * converted by the host layer) and the kept receivers per transmitter (mask_indices,
 * fwi_script.py:79-85, shape nt x nm). */
int ust_plan_set_acquisition(ust_plan* plan, int nt, const int32_t* src_lin_host, int nelem,
                             const int32_t* rx_lin_host, int nm, const int32_t* mask_idx_host);

/* Assemble the 9-point mixed-grid PML operator for nfreq frequencies from one sound-speed map and
 * factorise it (two-sided block-tridiagonal elimination, explicit block inverses).
 *   replaces: stencil_opt_params + assemble_Helmholtz (solve_helmholtz.py:104-290) and the LU half of
 *   SuperLU gssv behind scipy_solve (solve_helmholtz.py:15-18).
 * vel_dev: (ny, nx) real.  freqs_host: nfreq doubles.  bde_host: nfreq*3 doubles (b,d,e) or NULL to
 * compute them on the device from min/max(vel) like solve_helmholtz.py:62. */
int ust_factor(ust_plan* plan, const void* vel_dev, int nfreq, const double* freqs_host,
               const double* bde_host, void* stream);

/* Same for a lossy medium: complex slowness sigma = 1/vel - i kappa per node, wavenumber k = 2 pi f sigma, so the amplitude
 * attenuation is 2 pi f kappa Np/m (linear in frequency, no dispersion; alpha0 [dB/(cm MHz)] = 5.458e5 * kappa [s/m]).
 * kappa_dev: (ny, nx) real, >= 0 for a decaying wave; required (NULL is an error, not the lossless operator).  The stencil
 * weights come from min/max(vel) as in ust_factor.  ust_solve then solves the lossy operator. */
int ust_factor_lossy(ust_plan* plan, const void* vel_dev, const void* kappa_dev, int nfreq, const double* freqs_host,
                     const double* bde_host, void* stream);

/* In-place multi-RHS solve on the current factors of frequency slot ifreq:
 *   rhs_inout_dev (ny*nx, nrhs) complex, row-major; adjoint!=0 solves conj(H)^T u = rhs
 *   (solve_helmholtz.py:66-73) on the same factors.
 *   replaces: the triangular-solve half of gssv + the pure_callback round trip (solve_helmholtz.py:85-93). */
int ust_solve(ust_plan* plan, int ifreq, void* rhs_inout_dev, int nrhs, int adjoint, void* stream);

/* Convenience for host callers (the reference-facing solve_helmholtz): vel/src/out are HOST buffers;
 * copies, assembly, factorisation (skipped when refactor==0 and the plan already holds factors for
 * this vel/f) and the solve all happen inside.  src_host/out_host: (ny*nx, nrhs) complex. */
int ust_solve_helmholtz_host(ust_plan* plan, const void* vel_host, const void* src_host, void* out_host,
                             int nrhs, double f, const double* bde_host, int adjoint, int refactor);

/* Fused (loss, grad) of fwi_loss_function.py:29-103 + nonlinearcg.py:243-265 summed over nfreq
 * frequencies: factor, all-source forward sweeps (one-hot sources), source-strength estimate, residual,
 * loss, adjoint sweeps on the same factors, gradient w.r.t. slowness.
 *   slow_dev   (ny, nx) real slowness (params of fwi_loss_function.py:49)
 *   rec_dev    (nfreq, nt, nelem) complex observed data REC_DATA per frequency
 *   loss_dev   one double (sum over frequencies of 0.5*sum|rec_sim-rec_obs|^2)
 *   grad_dev   (ny, nx) real, overwritten */
int ust_fwi_loss_grad(ust_plan* plan, const void* slow_dev, const void* rec_dev, int nfreq,
                      const double* freqs_host, const double* bde_host, double* loss_dev, void* grad_dev,
                      void* stream);

/* Same, HOST buffers in and out (pinned staging inside): the reference-facing call that bench.py's
 * "e2e" times. */
int ust_fwi_loss_grad_host(ust_plan* plan, const void* slow_host, const void* rec_host, int nfreq,
                           const double* freqs_host, const double* bde_host, double* loss_host,
                           void* grad_host);

/* Joint (loss, grad) for a lossy medium (the complex slowness of ust_factor_lossy): the evaluation of ust_fwi_loss_grad with
 * the sigma^2 assembly, and the gradients with respect to both maps, alpha held fixed as in ust_fwi_loss_grad.  With
 * z_f = sum_t conj(alpha_t u_t) lambda_t, A = sum_f -2 w_f^2 Re z_f and B = sum_f -2 w_f^2 Im z_f per node:
 *   grad_s = s A - kappa B,   grad_kappa = -s B - kappa A      (kappa = 0: grad_s is ust_fwi_loss_grad's gradient, bit for bit)
 *   slow_dev, kappa_dev (ny, nx) real; kappa_dev is required.  grad_s_dev, grad_kappa_dev (ny, nx) real, overwritten.
 * After it, ust_ncg_linesearch and ust_fwi_gn_hvp refuse (their virtual source assumes a real slowness) until the next
 * ust_fwi_loss_grad; their lossy twins ust_ncg_linesearch_lossy and ust_fwi_gn_hvp_lossy run on its state instead. */
int ust_fwi_loss_grad_lossy(ust_plan* plan, const void* slow_dev, const void* kappa_dev, const void* rec_dev, int nfreq,
                            const double* freqs_host, const double* bde_host, double* loss_dev, void* grad_s_dev,
                            void* grad_kappa_dev, void* stream);

/* Same, HOST buffers in and out (the twin of ust_fwi_loss_grad_host). */
int ust_fwi_loss_grad_lossy_host(ust_plan* plan, const void* slow_host, const void* kappa_host, const void* rec_host, int nfreq,
                                 const double* freqs_host, const double* bde_host, double* loss_host, void* grad_s_host,
                                 void* grad_kappa_host);

/* NCG caller support (nonlinearcg.py:268-301), valid after ust_fwi_loss_grad on the same plan:
 * perturbation solve with RHS -VIRT*sd on the existing factors, gather at the receivers and return
 * the two line-search scalars  num = Re<dREC, REC_DATA-REC_SIM>, den = Re<dREC,dREC>
 * (compute_step_size, nonlinearcg.py:22-32) summed over frequencies.  out2_dev: two doubles.
 * Fails if ust_factor, ust_factor_lossy or ust_solve_helmholtz_host replaced the factors after that ust_fwi_loss_grad, and
 * after a lossy evaluation (ust_fwi_loss_grad_lossy); ust_ncg_linesearch_lossy is the line search of the lossy model. */
int ust_ncg_linesearch(ust_plan* plan, const void* sd_dev, double* out2_dev, void* stream);

/* Gauss-Newton Hessian-vector product of the joint objective on the factors, forward fields and source estimates of the last
 * ust_fwi_loss_grad on this plan (no assembly, no factorisation): hv = Re(J^H J v) with J the linearisation of
 * nonlinearcg.py:258,279 (alpha fixed).  v_dev, hv_dev: (ny, nx) real.  jv2_dev: one double, sum |J v|^2 (= <v, hv>).
 * jv_dev: (nfreq, nt, nm) complex J v at the kept receivers (mask order), or NULL.  Overwrites the adjoint wavefield.
 * J is the linearisation the gradient uses (virtual source 2 w^2 s alpha u without the stencil's mass weights and the PML
 * factor), not the exact derivative of the discrete forward map; the gradient equals Re(J^H (alpha P u - rec_obs)).
 * Fails if ust_factor, ust_factor_lossy or ust_solve_helmholtz_host replaced the factors after that ust_fwi_loss_grad, and
 * after a lossy evaluation (ust_fwi_loss_grad_lossy); ust_fwi_gn_hvp_lossy is the product of the lossy model. */
int ust_fwi_gn_hvp(ust_plan* plan, const void* v_dev, void* hv_dev, double* jv2_dev, void* jv_dev, void* stream);

/* Lossy twins of ust_ncg_linesearch and ust_fwi_gn_hvp for the joint (s, kappa) problem, valid only on the state of the last
 * ust_fwi_loss_grad_lossy: they fail before any evaluation, after a lossless evaluation, and after any factorisation
 * (ust_factor, ust_factor_lossy, ust_solve_helmholtz_host) or ust_plan_set_acquisition since that evaluation.  With the complex
 * slowness sigma = s - i kappa and alpha held fixed, the linearisation of a joint direction [v_s; v_kappa] is
 *   J [v_s; v_kappa] = P H^-1( -2 w^2 sigma alpha u (v_s - i v_kappa) )
 * and J^H r = [s A - kappa B, -s B - kappa A], the two gradients of ust_fwi_loss_grad_lossy formed from the adjoint field of r.
 * The kappa part of the direction (sd_kappa_dev, v_kappa_dev) is required.  At kappa = 0 and a zero kappa direction, out2 and
 * hv_s / jv2 / jv equal those of the lossless entry points on the same slowness, bit for bit.
 *   ust_ncg_linesearch_lossy: out2_dev = {num = Re<J sd, REC_DATA - REC_SIM>, den = |J sd|^2} (= -<sd, grad> and |J sd|^2).
 *   ust_fwi_gn_hvp_lossy:     hv_s_dev, hv_kappa_dev (ny, nx) real = Re(J^H J v); jv2_dev = sum |J v|^2 (= <v, hv>);
 *                             jv_dev (nfreq, nt, nm) complex J v at the kept receivers, or NULL. */
int ust_ncg_linesearch_lossy(ust_plan* plan, const void* sd_s_dev, const void* sd_kappa_dev, double* out2_dev, void* stream);
int ust_fwi_gn_hvp_lossy(ust_plan* plan, const void* v_s_dev, const void* v_kappa_dev, void* hv_s_dev, void* hv_kappa_dev,
                         double* jv2_dev, void* jv_dev /* (nfreq, nt, nm) complex or NULL */, void* stream);

/* Introspection for parity tests and callers that want the intermediate fields (device pointers into
 * plan-owned buffers, valid until the next ust_fwi_* call on the plan). */
int ust_get_bde(ust_plan* plan, double* bde_host /* max_freq*3 */);
int ust_get_planes(ust_plan* plan, int ifreq, void* planes_out_dev /* 9*ny*nx complex, order c,l,r,d,u,dl,dr,ul,ur */, void* stream);
int ust_get_src_est(ust_plan* plan, int ifreq, void* src_est_out_host /* nt complex */);
void* ust_get_wavefield(ust_plan* plan, int ifreq);  /* forward field, UNSCALED by src_est */
/* Size-independent check of the factor + sweep chain after ust_fwi_loss_grad: out2[0] = || H u_t - e_src(t) ||_2 over the
 * interior nodes for transmitter t of frequency slot ifreq (H from the coefficient planes = the rows assemble_Helmholtz
 * builds, solve_helmholtz.py:242-260), out2[1] = the 2-norm of the row sums |H||u| (the scale rounding errors live on:
 * out2[0] / out2[1] is ~1e-7 in complex64, ~1e-16 in complex128 for a correct solve).  Synchronises. */
int ust_residual_onehot(ust_plan* plan, int ifreq, int t, double* out2_host);
void* ust_get_adjoint_wavefield(ust_plan* plan, int ifreq);
int ust_get_status(ust_plan* plan, int* status_host); /* 0 ok; 1 = zero/NaN pivot met in a block inversion */

/* Engine unit-test hook: Cout = (Cin ? Cin with columns [mask_lo,mask_hi) read as zero : 0) + sgn*op(A)*B on
 * complex64 device arrays (row-major; ta!=0: op(A) = conj(A)^T with A stored K x M), with the block-GEMM
 * engine `engine` (UST_ENGINE_SIMT | UST_ENGINE_TC2 | UST_ENGINE_TC2H).  Rows [skip_lo,skip_hi) of Cout are left untouched (TC2, TC2H). */
int ust_test_cgemm(int engine, int ta, int M, int N, int K, const void* A_dev, int lda, const void* B_dev, int ldb,
                   const void* Cin_dev, int ldcin, void* Cout_dev, int ldc, float sgn, int mask_lo, int mask_hi,
                   int skip_lo, int skip_hi, void* stream);

/* Optional per-kernel-class device timing: while enabled every launch of the classes below is bracketed
 * by CUDA events on the launching stream; ust_get_profile synchronises, returns the accumulated
 * milliseconds and launch counts per class (arrays of 16) and clears the record.  Classes:
 * 0 assemble, 1 schur, 2 gj_panel, 3 gj_update, 4 tri_apply, 5 sweep_gemm, 6 receiver, 7 gradient, 8 t_split (unused: the block inverses leave the Gauss-Jordan epilogue as operand planes),
 * 9 gj_pivot (separate pivot launches: FMA engine, or look-ahead disabled), 10 gj_rowpanel (9-10 are the parts of 2),
 * 11 gj_k0 (TMA-fed engine: planes of block row / column 0 + inversion of pivot block 0, one launch per block row). */
int ust_profile(ust_plan* plan, int enable);
int ust_get_profile(ust_plan* plan, double* ms_out16, long long* count_out16);

/* Counters: number of kernel launches issued by this library on this thread since the last reset. */
/* Time-domain synthesis of frequency-domain wavefields (replaces the IDTFT of Lecture19_Fwi/TimeDomainSimulation.m:48-56,
 * `WVFIELD_T = pagemtimes(exp(1i*2*pi*f.*time')*df, resp_freq .* WVFIELD_F)`; an inverse discrete-time Fourier transform on
 * an arbitrary time axis, not an inverse FFT):
 *     out[t][p] = sum_k exp(i 2 pi freqs[k] time[t]) * df * resp[k] * U[k][p],   t < nt, p < npix.
 * U_dev: [nf][npix] complex (frequency-major stack of wavefields, any pixel order), out_dev: [nt][npix] complex, both of
 * `dtype` (UST_C64 | UST_C128) on the current device; freqs / resp / time are host arrays.  Enqueued on `stream`; the
 * weight matrix goes through a per-device buffer owned by the library that is grown on demand and reused (the one
 * exception to "the plan owns every workspace": this call has no plan). */
int ust_idtft(int dtype, const void* U_dev, int nf, long long npix, const double* freqs, const double* resp, double df,
              const double* time, int nt, void* out_dev, void* stream);

/* n float64 device values -> n (hi, lo) float32 pairs with hi + lo = value to ~1e-14 relative.  For callers whose runtime cannot
 * hold float64 (the reference runs JAX with x64 disabled, SURVEY.md A.1): the XLA FFI shim returns the loss this way. */
int ust_pack_f64_as_f32x2(const double* in_dev, float* out_dev, int n, void* stream);

long long ust_launch_count(void);
void ust_launch_count_reset(void);

#ifdef __cplusplus
}
#endif
#endif /* USTFWI_H */
