/* gpemu.h -- C ABI of libgpemu.so: the B200-native GP-emulator prediction engine.
 *
 * Drop-in boundary for the prediction hot path of UCL/gp_emulator.  Every entry point states the
 * reference interface it replaces (paths relative to the reference checkout).  Plain C: pointers and
 * sizes only; no CPython, numpy or torch types.  All matrices are ROW-MAJOR (C order), exactly as
 * numpy hands them over -- the reference's host-side transposes to column-major
 * (gp_emulator/gpu/_gpu_predict.cpp:129-132) do not exist here.
 *
 * Error convention: every function returns GPE_OK (0) or a negative gpe_status; the message of the
 * last failure on the calling thread is available from gpe_last_error().  Nothing here calls
 * exit() (the reference does: gp_emulator/gpu/gpu_predict.h:131-154, kernel_cdist.cu:28-32).
 *
 * Threading: different handles are independent.  Host-pointer calls on the same handle are serialised
 * inside the library (they share the handle's staging buffers); device-pointer calls are asynchronous on
 * the given stream and may be issued from several threads.  Creation / destruction of a handle must not
 * race with its use.
 */
#ifndef GPEMU_H_
#define GPEMU_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPE_VERSION 100

typedef enum gpe_status {
    GPE_OK = 0,
    GPE_ERR_INVALID = -1,      /* bad argument (shape, null pointer, unsupported size) */
    GPE_ERR_CUDA = -2,         /* a CUDA runtime call failed; see gpe_last_error() */
    GPE_ERR_NO_DEVICE = -3,    /* no usable sm_100 device */
    GPE_ERR_UNSUPPORTED = -4   /* valid request this build cannot serve (e.g. M > GPE_MAX_TRAIN) */
} gpe_status;

/* flags for the predict entry points */
#define GPE_WANT_MU     0x01u
#define GPE_WANT_VAR    0x02u  /* needs invQ at model creation */
#define GPE_WANT_DERIV  0x04u
#define GPE_WANT_HESS   0x08u
#define GPE_WANT_FWD    0x10u  /* banks with a basis: back-projected output fwd (N, W) */
#define GPE_WANT_DERIV_FULL 0x20u /* banks with a basis: back-projected Jacobian deriv_full (N, D, W) */
#define GPE_HOST_PTRS   0x100u /* testing/outputs are host pointers: the library streams them */
#define GPE_F32_FAST_TF32 0x200u /* gpe_predict_f32 only: one TF32 pass for the variance instead of the 3xTF32 split */
#define GPE_F32_FORCE_3X  0x400u /* gpe_predict_f32 only: 3xTF32 split also for M > 256 (default there: one pass) */

#define GPE_MAX_TRAIN 16384    /* largest M with a variance path: fused kernel to 1024, K*-scratch + column passes above
                                  (a bound on the packed invQ image, 2 GB at 16384; mean / gradient / Hessian have no limit) */
#define GPE_MAX_INPUTS 256     /* largest D; up to 32 the per-D compiled kernels run, above that generic ones (FP64 only) */

typedef struct gpe_model gpe_model;  /* one trained GP resident on one device */
typedef struct gpe_bank gpe_bank;    /* E GPs sharing training inputs (MultivariateEmulator / per-band bank) */

const char* gpe_last_error(void);
int gpe_version(void);
int gpe_device_count(void);

/* Upload one trained GP.
 * Replaces the per-call model upload of gpuPredict::init_gpu (gp_emulator/gpu/predict.cu:11-34) and the
 * model flattening in GaussianProcess.gpu_predict (gp_emulator/GaussianProcess.py:289-292); the model
 * stays resident behind the handle instead of being re-sent for every 2e5-point block.
 *   inputs  (M, D)  training inputs          == self.inputs
 *   expX    (D+1)   exp(theta)[0..D]         == np.exp(self.theta): D inverse squared length scales, then
 *                                               the signal variance (theta[D+1], the noise, is unused by predict)
 *   invQt   (M)     == self.invQt
 *   invQ    (M, M)  == self.invQ, may be NULL if variance is never requested
 * All host pointers, float64. */
int gpe_model_create(int device, int M, int D, const double* inputs, const double* expX,
                     const double* invQt, const double* invQ, gpe_model** out);
int gpe_model_destroy(gpe_model* m);

/* Same, with options.  GPE_OPT_SYMMETRIC_VARIANCE: evaluate the quadratic form of the variance
 * (`np.sum(a * np.dot(self.invQ, a), axis=0)`, gp_emulator/GaussianProcess.py:240) as k^T T k with T the
 * upper-triangular fold of invQ (T_ij = invQ_ij + invQ_ji for i < j, invQ_jj on the diagonal, 0 below).  The
 * identity is exact for ANY invQ, symmetric or not; only the rounding differs (by ~1e-16 of sum |terms|), and the
 * tensor-core work is halved.  Off by default: the default path evaluates the dense formula as numpy does.
 * gpe_model_create() honours the environment variable GPE_SYMMETRIC_VARIANCE=1 as the same opt-in. */
#define GPE_OPT_SYMMETRIC_VARIANCE 0x1u
int gpe_model_create_ex(int device, int M, int D, const double* inputs, const double* expX,
                        const double* invQt, const double* invQ, unsigned options, gpe_model** out);

/* Predict N test points: the whole of GaussianProcess.cpu_predict / gpu_predict
 * (gp_emulator/GaussianProcess.py:211-251, :273-323) and gpuPredict::predict
 * (gp_emulator/gpu/predict.cu:168-176) in one fused pass.
 *   testing (N, D) row-major; mu (N); var (N); deriv (N, D) row-major -- NOT the (D, N) layout the
 *   legacy extension returned (GaussianProcess.py:321).  hess (N, D, D) as GaussianProcess.hessian
 *   (GaussianProcess.py:345-366).  Output pointers whose GPE_WANT_* bit is clear may be NULL.
 *   Without GPE_HOST_PTRS all pointers are device pointers on the model's device and the call is
 *   asynchronous on `stream` (a cudaStream_t, NULL = legacy default stream).  Any N >= 0 is accepted
 *   (the reference exits for N < 1000, kernel_cdist.cu:28-32, and for N*M > 6.7e7, kernel_matrixExp.cu:29-33). */
int gpe_predict(gpe_model* m, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                double* hess, unsigned flags, void* stream);

/* Diagnostic: name and tile plan of the kernel(s) a mean + variance + gradient call of N points runs on this model,
 * written to buf (NUL-terminated, at most len bytes); returns the length.  bench.py reports it beside the roofline. */
int gpe_model_plan(gpe_model* m, int64_t N, char* buf, int len);

/* Single-precision variant on the 5th-generation tensor cores (tcgen05.mma.kind::tf32, accumulators in TMEM):
 * what the reference's FP32 build of gpuPredict computes (`real` = float, gp_emulator/gpu/gpu_predict.h:20-34;
 * Python side precision=np.float32, gp_emulator/GaussianProcess.py:289-316).  Same handle, float32 I/O
 * (testing (N, D), mu (N), var (N), deriv (N, D)), M <= 1024, no Hessian.  K*, mean and gradient are FP32.
 * Variance contraction: by default a 3xTF32 split (hi.hi + lo.hi + hi.lo, FP32 accumulation) that meets the
 * reference's own FP32 pass criterion of 1e-5 (tests/benchmark.py:56); with GPE_F32_FAST_TF32 a single TF32 pass
 * (relative error ~1e-4 of max|var|, bound 2^-11), about 1.7x faster at M = 250.  For M > 256 the single pass is
 * the default (the FP32 accumulation of 1000-term sums costs ~1e-5 by itself, so the split buys little for 3.6x the
 * time); GPE_F32_FORCE_3X selects the split there too. */
int gpe_predict_f32(gpe_model* m, const float* testing, int64_t N, float* mu, float* var, float* deriv,
                    unsigned flags, void* stream);

/* Binary-compatible stand-in for the legacy native entry point
 *   _gpu_predict.predict_wrap(expX, inputs, invQt, invQ, testing, result, error, deriv,
 *                             Npredict, Ntrain, Ninputs, theta_size)
 * (gp_emulator/gpu/_gpu_predict.cpp:115-159; call site gp_emulator/GaussianProcess.py:313-316):
 * same argument order and meaning, host float64 arrays flattened row-major, outputs written in place,
 * and -- for compatibility with the caller's reshape at GaussianProcess.py:321 -- deriv is written as
 * (Ninputs, Npredict).  Uses device 0 and a cached model keyed on the argument contents. */
int gpe_predict_wrap(const double* expX, const double* inputs, const double* invQt, const double* invQ,
                     const double* testing, double* result, double* error, double* deriv,
                     int Npredict, int Ntrain, int Ninputs, int theta_size);

/* One call, several devices: the GP is uploaded to every listed device and a host-resident batch is cut into chunks
 * that the devices' pipelines -- one host thread each inside the library -- pull from one shared cursor, so a GPU
 * behind a slower PCIe path takes fewer chunks instead of holding the call back (test points are independent:
 * gp_emulator/GaussianProcess.py:228-249; the reference has no multi-device code, doc/report.md:48,95 lists it as
 * future work).  Results are bit-identical to the single-device call.  This is what the drop-in classes run on with
 * `device="all"`: the reference API has no notion of ranks (gp_emulator/GaussianProcess.py:327), so the fan-out lives
 * below it. */
typedef struct gpe_multi gpe_multi;
int gpe_multi_create(int n_devices, const int* devices, int M, int D, const double* inputs, const double* expX,
                     const double* invQt, const double* invQ, unsigned options, gpe_multi** out);
/* host pointers */
int gpe_multi_predict(gpe_multi* mm, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                      double* hess, unsigned flags);
/* device pointers: arrays of n_devices entries, testing[g] (N[g], D) etc. resident on device g of the handle;
 * asynchronous on streams[g] (streams == NULL: the legacy default stream of each device).  N[g] may be 0. */
int gpe_multi_predict_device(gpe_multi* mm, const double* const* testing, const int64_t* N, double* const* mu,
                             double* const* var, double* const* deriv, double* const* hess, unsigned flags,
                             void* const* streams);
int gpe_multi_destroy(gpe_multi* mm);

/* Bank of E GPs that share the training inputs (M, D) and the test points, each with its own
 * hyper-parameters: the per-PC emulators of MultivariateEmulator (gp_emulator/multivariate_gp.py:176-188)
 * and the per-band banks of tests/test_perband_emulator.py:22-37.
 *   expX (E, D+1); invQt (E, M); invQ (E, M, M) or NULL;
 *   basis (E, W) or NULL: MultivariateEmulator.basis_functions for the PCA back-projection. */
int gpe_bank_create(int device, int E, int M, int D, const double* inputs, const double* expX,
                    const double* invQt, const double* invQ, const double* basis, int W, gpe_bank** out);
int gpe_bank_destroy(gpe_bank* b);

/* Bank prediction on shared test points.  Outputs are point-major:
 *   mu (N, E), var (N, E), deriv (N, E, D), hess (N, E, D, D).
 * Replaces the Python loop over emulators in MultivariateEmulator.predict
 * (gp_emulator/multivariate_gp.py:214-218) and over bands in tests/test_perband_emulator.py:39-47. */
int gpe_bank_predict(gpe_bank* b, const double* testing, int64_t N, double* mu, double* var,
                     double* deriv, double* hess, unsigned flags, void* stream);

/* Same, plus the back-projected outputs in the same call: fwd (N, W) with GPE_WANT_FWD, deriv_full (N, D, W) with
 * GPE_WANT_DERIV_FULL (gp_emulator/multivariate_gp.py:216,218).  With GPE_HOST_PTRS every array is a host array and
 * the library streams chunks through its pinned pipeline -- the chunk walk of GaussianProcess.gpu_predict
 * (gp_emulator/GaussianProcess.py:297-321) below the C ABI, for banks; the PC means / gradients a projection consumes
 * stay on the device unless they are requested too.  With device pointers a projection needs GPE_WANT_MU (and
 * GPE_WANT_DERIV for the Jacobian) as well.  Banks of more than 32 emulators project in slices of 32. */
int gpe_bank_predict_ex(gpe_bank* b, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                        double* hess, double* fwd, double* deriv_full, unsigned flags, void* stream);

/* Least-squares cost of the bank's means against observations and its input gradient, reduced over the E emulators
 * on the fly so the (N, E) means and (N, E, D) gradients never leave the device (they exist for one chunk at a time):
 *   cost_n = 1/2 sum_e w_e (mu_ne - obs_ne)^2        grad_nd = sum_e w_e (mu_ne - obs_ne) deriv_ned
 * What a caller of a per-band bank builds in numpy from E separate predicts (the loop of
 * gp_emulator/tests/test_perband_emulator.py:39-47 followed by the comparison with the observed bands); the reference
 * has no such function -- it is the "outputs consumed on the fly" item of SURVEY.md 8f-3.
 *   obs (N, E) with obs_ld >= E, or one (E) vector shared by every point with obs_ld = 0; weights (E) or NULL (all 1);
 *   cost (N) or NULL; grad (N, D) or NULL.  Device pointers, asynchronous on `stream`. */
int gpe_bank_cost(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                  const double* weights, double* cost, double* grad, void* stream);
/* The same reduction for host arrays (obs_ld = E or 0), streamed in chunks; synchronous. */
int gpe_bank_cost_host(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                       const double* weights, double* cost, double* grad);
/* gpe_bank_cost / gpe_bank_cost_host plus the exact input Hessian of the cost, hess (N, D, D) or NULL, laid out as
 * GaussianProcess.hessian:
 *   hess_n = sum_e w_e (mu_ne - obs_ne) H_ne + sum_e w_e deriv_ne deriv_ne^T      H_ne: the bank's per-emulator Hessians
 * (the hess of gpe_bank_predict).  Any non-empty subset of cost, grad and hess may be requested; cost and grad are bit
 * for bit those of the same call without hess.  hess_n equals its transpose bit for bit.  At obs = the bank's own mu the
 * first sum is exactly 0 and hess_n is the (positive semi-definite) Gauss-Newton term; elsewhere it may be indefinite.
 * Non-finite values propagate as in the formula evaluated in numpy: a NaN observation gives a NaN Hessian even where its
 * weight is 0.  Results do not depend on chunking, pointer placement or the device count. */
int gpe_bank_cost_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                     const double* weights, double* cost, double* grad, double* hess, void* stream);
int gpe_bank_cost_host_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                          const double* weights, double* cost, double* grad, double* hess);

/* Least-squares cost of the bank's back-projected spectra against observed spectra and its input gradient, per point:
 *   cost_n = 1/2 sum_w l_w (fwd_nw - obs_nw)^2          fwd = mu . basis           (gp_emulator/multivariate_gp.py:216)
 *   grad_nd =    sum_w l_w (fwd_nw - obs_nw) deriv_full_ndw    deriv_full_ndw = sum_e deriv_ned basis_ew   (:218)
 * fwd and deriv are the bank's own PC means and gradients: the values gpe_bank_predict_ex returns with GPE_WANT_FWD and
 * GPE_WANT_DERIV_FULL.  The residual is formed per wavelength, in one fused kernel, so neither fwd (N, W) nor
 * deriv_full (N, D, W) is ever written to memory.  An observation equal to the library's own fwd gives exactly 0.
 *   obs (N, W) with obs_ld >= W, or one (W) spectrum shared by every point with obs_ld = 0; weights (W) or NULL (all 1);
 *   cost (N) or NULL; grad (N, D) or NULL (not both).  The bank needs a basis, and at most 96 emulators.
 * Non-finite values propagate as in the formula above evaluated in numpy (no masking): a NaN observation gives a NaN
 * cost and gradient even where its weight is 0. Results do not depend on chunking, pointer placement or the device count.
 * Device pointers, asynchronous on `stream`; N = 0 launches nothing. */
int gpe_bank_forward_cost(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                          const double* weights, double* cost, double* grad, void* stream);
/* The same for host arrays (obs_ld = W or 0), streamed in chunks; synchronous. */
int gpe_bank_forward_cost_host(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                               const double* weights, double* cost, double* grad);
/* gpe_bank_forward_cost / gpe_bank_forward_cost_host plus the exact input Hessian of the cost, hess (N, D, D) or NULL,
 * laid out as GaussianProcess.hessian:
 *   hess_n = sum_e s_ne H_ne + deriv_n^T C deriv_n      s_ne = sum_w l_w (fwd_nw - obs_nw) basis_ew,
 *                                                       C = basis . diag(l) . basis^T (E, E), deriv_n (E, D)
 * which is sum_w l_w deriv_full_nw deriv_full_nw^T + sum_w l_w (fwd_nw - obs_nw) d2 fwd_nw / dx2 without forming either
 * per wavelength.  Any non-empty subset of cost, grad and hess may be requested; cost and grad are bit for bit those of
 * the same call without hess.  hess_n equals its transpose bit for bit.  At obs = the bank's own fwd s is exactly 0 and
 * hess_n is the (positive semi-definite) Gauss-Newton term.  A NaN observation gives a NaN Hessian even where its weight
 * is 0, as the formula evaluated in numpy does.  Same limits as gpe_bank_forward_cost (basis, at most 96 emulators). */
int gpe_bank_forward_cost_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                             const double* weights, double* cost, double* grad, double* hess, void* stream);
int gpe_bank_forward_cost_host_ex(gpe_bank* b, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                                  const double* weights, double* cost, double* grad, double* hess);

/* Banks on several devices, host arrays, one call: the bank counterpart of gpe_multi_create / gpe_multi_predict
 * (same handle type; destroy with gpe_multi_destroy).  Arguments as gpe_bank_create / gpe_bank_predict_ex /
 * gpe_bank_cost_host / gpe_bank_forward_cost_host. */
int gpe_multi_bank_create(int n_devices, const int* devices, int E, int M, int D, const double* inputs,
                          const double* expX, const double* invQt, const double* invQ, const double* basis, int W,
                          gpe_multi** out);
int gpe_multi_bank_predict(gpe_multi* mm, const double* testing, int64_t N, double* mu, double* var, double* deriv,
                           double* hess, double* fwd, double* deriv_full, unsigned flags);
int gpe_multi_bank_cost(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                        const double* weights, double* cost, double* grad);
int gpe_multi_bank_forward_cost(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                                const double* weights, double* cost, double* grad);
/* ... with the Hessian hess (N, D, D) or NULL, as gpe_bank_cost_host_ex / gpe_bank_forward_cost_host_ex. */
int gpe_multi_bank_cost_ex(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                           const double* weights, double* cost, double* grad, double* hess);
int gpe_multi_bank_forward_cost_ex(gpe_multi* mm, const double* testing, int64_t N, const double* obs, int64_t obs_ld,
                                   const double* weights, double* cost, double* grad, double* hess);

/* Inversion: per point, the x in the box lower <= x <= upper that minimises
 *   f(x) = cost(x) + 1/2 (x - m)^T P (x - m)
 * where cost is the band cost of gpe_bank_cost_ex (default) or, with GPE_SOLVE_SPECTRA, the spectrum cost of
 * gpe_bank_forward_cost_ex, and the Gaussian prior (mean m, precision P) is optional.  g = grad + P (x - m) and
 * H = hess + P.  Levenberg-Marquardt on the exact Hessian, every point independently:
 *   1. x = clip(x0, lower, upper); evaluate f, g, H there; lambda = lambda0, nu = 2.
 *   2. Free set F: every d except those with x_d = lower_d, g_d > 0 or x_d = upper_d, g_d < 0.  Solve
 *      (H_FF + lambda diag(s_F)) delta_F = -g_F by Cholesky, s_d = max(|H_dd|, 1e-12 max_{k in F} |H_kk|); while the
 *      factorisation fails (H may be indefinite away from the optimum): lambda *= nu, nu *= 2.
 *   3. x_t = clip(x + delta), delta' = x_t - x, pred = -(g^T delta' + 1/2 delta'^T H delta').
 *   4. Evaluate f_t, g_t, H_t at x_t; rho = (f - f_t) / pred.  f_t < f and rho > 0: accept x_t,
 *      lambda *= max(1/3, 1 - (2 rho - 1)^3), nu = 2.  Otherwise lambda *= nu, nu *= 2.
 * The point stops with (tests in this order after each evaluation: f at x0, ftol, gtol, lambda, xtol, max_iter)
 *   GPE_SOLVE_NONFINITE  f is not finite at clip(x0): returned there, with what was evaluated there;
 *   GPE_SOLVE_CONVERGED  an accepted step changed f by at most ftol |f|, or max_F |g_F| <= gtol, or the proposed
 *                        max |delta'| <= xtol (max |x| + xtol);
 *   GPE_SOLVE_STALLED    lambda passed 1e20 (failed factorisations and rejected steps both raise it) before a step
 *                        could be formed;
 *   GPE_SOLVE_MAX_ITER   max_iter evaluations after the first were used.
 * Outputs at the returned x (prior included): x (N, D); cost (N), grad (N, D), hess (N, D, D) or NULL; cov (N, D, D) =
 * inv(H) without damping, symmetric bit for bit, NaN where H is not positive definite, or NULL; info (N, 2) =
 * (status, evaluations after the first).
 * Arguments: x0 (N, D); obs and weights as the cost call (obs (N, K) with obs_ld >= K, or (K) with obs_ld = 0; K = E, or
 * W with GPE_SOLVE_SPECTRA; weights (K) or NULL); opts NULL takes the defaults below.  lower / upper (D) or NULL (no
 * bound; entries may be -inf / +inf); prior_mean (N, D) rows prior_ld >= D apart, one (D) row with prior_ld = 0, or NULL
 * (0); prior_prec (D, D), symmetric, or NULL (no prior; a prior_mean then is an error).
 * Every array follows the call's placement: device pointers on the bank's device, or host pointers with GPE_HOST_PTRS
 * (host obs_ld = K or 0, host prior_ld = D or 0).  The call is SYNCHRONOUS even with device pointers: it reads the number
 * of points still active once per iteration.  Iterations stay on the device and converged points are not evaluated again.
 * Results do not depend on chunking, pointer placement, the device count or the order of the points.
 * D <= 32; the spectrum cost takes banks of up to 96 emulators (GPE_ERR_UNSUPPORTED beyond). */
#define GPE_SOLVE_SPECTRA 0x1000u   /* spectrum cost (needs a basis); default: band cost */
#define GPE_SOLVE_MAX_D 32
#define GPE_SOLVE_CONVERGED 0
#define GPE_SOLVE_MAX_ITER 1
#define GPE_SOLVE_STALLED 2
#define GPE_SOLVE_NONFINITE 3
#define GPE_SOLVE_DEFAULT_MAX_ITER 50
typedef struct gpe_solve_opts {
    int max_iter;          /* >= 0 (default 50) */
    double ftol, xtol, gtol;   /* >= 0 (defaults 1e-10, 1e-10, 0) */
    double lambda0;        /* > 0 (default 1e-3) */
    const double* lower;
    const double* upper;
    const double* prior_mean;
    int64_t prior_ld;
    const double* prior_prec;
} gpe_solve_opts;
int gpe_bank_solve(gpe_bank* b, const double* x0, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                   const gpe_solve_opts* opts, double* x, double* cost, double* grad, double* hess, double* cov,
                   int32_t* info, unsigned flags, void* stream);
/* The same on every device of a bank handle; host arrays (GPE_HOST_PTRS is implied). */
int gpe_multi_bank_solve(gpe_multi* mm, const double* x0, int64_t N, const double* obs, int64_t obs_ld, const double* weights,
                         const gpe_solve_opts* opts, double* x, double* cost, double* grad, double* hess, double* cov,
                         int32_t* info, unsigned flags);

/* PCA back-projection of bank means: fwd (N, W) = mu (N, E) @ basis (E, W)
 * (the accumulation `fwd += pred_mu * basis_functions[i]`, gp_emulator/multivariate_gp.py:216, batched
 * over N points), and optionally deriv_full (N, D, W) = sum_e deriv[n, e, d] * basis[e, w] (:218).
 * Device pointers; mu/deriv as produced by gpe_bank_predict. */
int gpe_bank_project(gpe_bank* b, const double* mu, const double* deriv, int64_t N, double* fwd,
                     double* deriv_full, void* stream);

/* MultivariateEmulator.predict for host callers in ONE call (gp_emulator/multivariate_gp.py:195-222): test points
 * (N, D) on the host -> fwd (N, W) and, if deriv_full is not NULL, deriv_full (N, D, W) on the host; the per-PC
 * means / gradients never leave the device.  Built for the reference's usage pattern -- one point, or a few, per
 * call inside an optimisation loop: one H2D copy, three launches, one D2H copy and one synchronisation per chunk. */
int gpe_bank_forward(gpe_bank* b, const double* testing, int64_t N, double* fwd, double* deriv_full);

/* FP64 pipe peaks of the device, measured live (roofline denominators the driver's
 * MEASURED_PEAKS.json does not hold).  out9: DFMA TFLOP/s, DMMA TFLOP/s, mixed total, mixed DFMA part,
 * mixed DMMA part, gpe exp Gexp/s, CUDA exp Gexp/s, SM MHz under FP64 load, SM count. */
int gpe_measure_fp64_peaks(int device, double* out9);

/* ---- batched training objective (SURVEY.md 8f-1: the caller on the input side of the prediction path) -------------
 * Evaluates, for B (theta, target vector) problems at once, what the reference computes one theta at a time inside its
 * optimiser loop: GaussianProcess.loglikelihood (gp_emulator/GaussianProcess.py:78-95, i.e. _set_params ->
 * _prepare_likelihood :52-75) and GaussianProcess.partial_devs (:97-125).  All problems share the training inputs
 * (MultivariateEmulator.train_emulators fits every principal component on the same y_train,
 * gp_emulator/multivariate_gp.py:176-186).  Host pointers; synchronous.
 *   inputs   (M, D)      training inputs            == self.inputs
 *   targets  (T, M)      T target vectors           == self.targets of each GP
 *   target_index (B)     which target vector problem b fits (NULL: all use row 0)
 *   thetas   (B, D + 2)  hyper-parameters (log inverse squared length scales, log signal variance, log noise)
 *   loglik   (B)         the reference's cost: 1/2 log|Q| + 1/2 t' invQ t + M/2 log(2 pi)
 *   grad     (B, D + 2)  its gradient, as partial_devs returns it
 *   status   (B)         0, or 1 where Q is not positive definite / not finite (the reference's LinAlgError from
 *                        np.linalg.cholesky, :73-75): loglik and grad of that problem are NaN
 */
#define GPE_TRAIN_MAX_M 1024
#define GPE_TRAIN_MAX_D 32    /* the batched training kernel keeps exp(theta) for D + 2 <= 40 hyper-parameters on chip */
typedef struct gpe_trainer gpe_trainer;
int gpe_trainer_create(int device, int M, int D, int T, const double* inputs, const double* targets, gpe_trainer** out);
int gpe_trainer_eval(gpe_trainer* t, int B, const int* target_index, const double* thetas, double* loglik, double* grad,
                     int* status);
int gpe_trainer_destroy(gpe_trainer* t);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches claim). */
int64_t gpe_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GPEMU_H_ */
