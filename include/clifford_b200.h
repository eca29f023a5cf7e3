/* clifford_b200 -- C ABI of the B200-native latent hot path (sm_100a).
 *
 * This is the drop-in boundary: every entry point takes raw DEVICE pointers (fp32 unless noted),
 * explicit sizes / strides, a Philox (seed, offset) pair or pointers to pre-drawn base variates, and
 * a cudaStream_t passed as void*.  Nothing allocates, nothing synchronises, every call returns an
 * int status (0 = ok; see cvb_status below; text via cvb_last_error_string()).
 *
 * The reference (momalekabid/clifford-vae) has no FFI of its own: its boundary is a set of Python
 * symbols (SURVEY.md section 8(b)).  Each function below names the reference code it replaces; the
 * Python classes/functions with the reference's names live in clifford-vae_b200/{dists,utils,
 * hyperspherical_vae} and call these through ctypes (see INTEGRATION.md).
 *
 * Row conventions: "rows" are flattened leading dims (sample_shape x batch).  Parameters that are
 * shared across sample_shape are indexed with row % loc_rows.  A concentration tensor is addressed
 * as kappa[(row % loc_rows) * kappa_row_stride + k * kappa_el_stride]; kappa_el_stride == 0 means one
 * concentration per row (what every reference driver uses: mnist/mlp_vae.py:70,93, cnn/models.py:228).
 */
#ifndef CLIFFORD_B200_H_
#define CLIFFORD_B200_H_

#if defined(__GNUC__)
#define CVB_API __attribute__((visibility("default")))
#else
#define CVB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

enum cvb_status { CVB_OK = 0, CVB_BAD_ARGUMENT = 1, CVB_UNSUPPORTED = 2, CVB_CUDA_ERROR = 3 };

/* bind modes (cvb_vsa_bind) */
enum cvb_bind_mode {
  CVB_BIND_MUL = 0,          /* irfft(A * B)            utils/vsa.py:43-46  bind                          */
  CVB_BIND_MUL_CONJ = 1,     /* irfft(A * conj B)       utils/vsa.py:56-64  unbind "inv"/"*"; bind bwd    */
  CVB_BIND_DIV = 2,          /* irfft(A / (B + 1e-12))  utils/vsa.py:65-70  unbind "dagger"/"deconv"      */
  CVB_BIND_DIV_CONJ = 3,     /* irfft(A / conj(B+1e-12))  adjoint of DIV wrt its first operand            */
  CVB_BIND_NEG_MUL_CONJ = 4  /* -irfft(A * conj B)        adjoint of DIV wrt its second operand           */
};

CVB_API int cvb_version(void);
CVB_API const char* cvb_last_error_string(void);
/* Build the per-device twiddle table on the CURRENT device.  Call once per device before any other
 * entry point (and outside CUDA-graph capture); idempotent. */
CVB_API int cvb_init(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches claim). */
CVB_API long long cvb_launch_count(void);

/* ---- Clifford-torus power-spherical distribution: dists/clifford.py:281-327 ------------------- */

/* CliffordPowerSphericalDistribution.rsample (dists/clifford.py:295-308) fused with entropy()/KL
 * (:318-327, :241-242).  loc (loc_rows, d).  Base draws: pass tprime and gnoise (rows, d) to inject
 * t' ~ Beta(1/2 + kappa + 1e-7, 1/2) and g ~ N(0,1) (parity mode), or both NULL to draw on the device
 * with Philox4x32-10 keyed by (seed, offset).  Outputs: z (rows, 2d); optional tp_signed (rows, d):
 * the draws saved for cvb_clifford_ps_rsample_backward in RNG mode -- OPAQUE to the caller: copysign(t', sign), or, on
 * rows sampled through the inverse-CDF table (one concentration <= 32 per row, power-of-two d >= 512), the signed table
 * coordinate of the draw; element 0 of every row is left unwritten.  With one concentration per row and a power-of-two
 * d in [512, 8192], saving tp_signed in RNG mode needs z 8-byte aligned (else CVB_UNSUPPORTED): the saved format
 * depends on the kernel, and the kernel on z's alignment; optional entropy / kl / dentropy (rows)
 * (dentropy = d entropy / d kappa), written only when kappa_el_stride == 0 (otherwise call
 * cvb_ps_entropy_kl). */
CVB_API int cvb_clifford_ps_rsample(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                            long long loc_rows, const float* tprime, const float* gnoise,
                            unsigned long long seed, unsigned long long offset, float* z, float* tp_signed,
                            float* entropy, float* kl, float* dentropy, long long rows, int d, void* stream);

/* Backward of the above (autograd through ifft / exp / atan2 / _Dirichlet_backward in the reference).
 * Give either (tprime, gnoise) [injected draws: ATen's piecewise implicit Beta gradient, like the reference] or the
 * tp_signed buffer the forward wrote for the SAME (loc, kappa, rows, d) [table-sampled rows: the pathwise derivative of the
 * table map itself, i.e. the same implicit reparameterisation gradient evaluated to 2.5e-5 instead of ATen's
 * approximation of it].  With tp_signed, one concentration per row and a power-of-two d in [512, 8192], grad_z must be
 * 8-byte aligned (else CVB_UNSUPPORTED), like the forward's z.  dloc (rows, d); dkappa (rows) when kappa_el_stride == 0,
 * else (rows, d). */
CVB_API int cvb_clifford_ps_rsample_backward(const float* grad_z, const float* loc, const float* kappa,
                                     long long kappa_row_stride, int kappa_el_stride, long long loc_rows,
                                     const float* tprime, const float* gnoise, const float* tp_signed, float* dloc,
                                     float* dkappa, long long rows, int d, void* stream);

/* cvb_clifford_ps_rsample fused with a bind of every sample: bound[r] = bind(z[r], b[r % b_rows]) (utils/vsa.py:43-46 applied
 * to the fresh sample).  The sample's spectrum is known in closed form (the unit phasors), so the bind costs one forward
 * FFT of b and one inverse FFT instead of three transforms, and z is never read back from HBM.  One concentration per
 * row (kappa (loc_rows)); d a power of two in [16, 8192]; z may be NULL when only the bound vectors are wanted. */
CVB_API int cvb_clifford_ps_rsample_bind(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                         const float* gnoise, unsigned long long seed, unsigned long long offset,
                                         const float* b, long long b_rows, float* z, float* bound, float* entropy,
                                         float* kl, float* dentropy, long long rows, int d, void* stream);

/* cvb_clifford_ps_rsample that also returns log q(z) of every drawn sample -- the pair the IWAE estimator evaluates
 * (mnist/mlp_vae.py:161,181: q_z.rsample([S]) then q_z.log_prob(z)).  The sampled phase offsets are known, so
 * log_prob[r] = d log C(kappa) + kappa (log1p(clamp(cos loc_0)) + sum_{k>=1} log1p(clamp(t_k))) needs no FFT -> angle
 * pass over z (dists/clifford.py:310-316 evaluated on the sampler's own t).  One concentration per row (kappa
 * (loc_rows)); d a power of two in [16, 8192]; forward only.  log_prob (rows) is overwritten. */
CVB_API int cvb_clifford_ps_rsample_log_prob(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                             const float* gnoise, unsigned long long seed, unsigned long long offset,
                                             float* z, float* log_prob, float* entropy, float* kl, long long rows, int d,
                                             void* stream);

/* CliffordPowerSphericalDistribution.log_prob (dists/clifford.py:310-316, :198-202).  value (rows, 2d)
 * -> log_prob (rows).  Optional derivative outputs: dlp_dloc (rows, d) and dlp_dkappa ((rows) or (rows, d)) (give both
 * or neither), and dlp_dF (rows, d) complex = d log_prob / d (Re, Im) of the value's Fourier bin k. */
CVB_API int cvb_clifford_ps_log_prob(const float* value, const float* loc, const float* kappa, long long kappa_row_stride,
                             int kappa_el_stride, long long loc_rows, float* log_prob, float* dlp_dloc,
                             float* dlp_dkappa, float* dlp_dF, long long rows, int d, void* stream);
/* Adjoint of value (rows, 2d) -> first d bins of its real FFT: grad_value = Re sum_k H_k e^{+2 pi i jk/(2d)} for
 * H (rows, d) complex (the autograd of fft(value)[..., :d] in dists/clifford.py:311). */
CVB_API int cvb_clifford_spectrum_adjoint(const float* h_complex, float* grad_value, long long rows, int d, void* stream);

/* Power-spherical entropy / KL-to-uniform and dH/dkappa without sampling.
 * torus != 0: dists/clifford.py:318-327 -- sum over circles k >= 1 of the dim-2 entropy, kl = -H + (d-1) ln 2pi.
 * torus == 0: dists/clifford.py:204-212, :335-337 -- one (2*half_dm1+1)-dim PowerSpherical per row
 *             (el_stride ignored), kl = -H + prior_entropy.
 * dentropy: (rows) when kappa_el_stride == 0 or torus == 0, else (rows, d). */
CVB_API int cvb_ps_entropy_kl(const float* kappa, long long kappa_row_stride, int kappa_el_stride, long long rows, int d,
                      double half_dm1, int torus, double prior_entropy, float* entropy, float* kl, float* dentropy,
                      void* stream);

/* CliffordTorusDistribution.rsample (dists/clifford.py:261-275; scripts/sample_viz.py:55-64 restates it): phases
 * theta = loc + VonMises(0, kappa) drawn on the device with Best & Fisher's rejection (the algorithm behind
 * torch.distributions.VonMises.sample, which the reference calls at :262), then the same Hermitian spectrum -> C2R
 * inverse FFT.  kappa addressed like cvb_clifford_ps_rsample's.  Forward only; cvb_clifford_vm_rsample_kl draws the
 * same z and saves what its backward needs.  (The reference's own method stops at its Hermitian-symmetry assert, :274;
 * this entry point is the working version of what it computes.) */
CVB_API int cvb_clifford_vm_rsample(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                                    long long loc_rows, unsigned long long seed, unsigned long long offset, float* z,
                                    long long rows, int d, void* stream);
/* cvb_clifford_vm_rsample with a reparameterised backward: bitwise the same z for the same (seed, offset).  phi
 * (rows, d) optional: the drawn offsets theta_k - loc_k, saved for cvb_clifford_vm_rsample_backward (opaque; element 0
 * unwritten).  entropy / kl / dentropy (rows) optional, only with kappa_el_stride == 0: the row values that
 * cvb_clifford_vm_entropy gives, and kl = (d-1) ln 2 pi - entropy (the KL to CliffordTorusUniform), from the same launch. */
CVB_API int cvb_clifford_vm_rsample_kl(const float* loc, const float* kappa, long long kappa_row_stride, int kappa_el_stride,
                                       long long loc_rows, unsigned long long seed, unsigned long long offset, float* z,
                                       float* phi, float* entropy, float* kl, float* dentropy, long long rows, int d,
                                       void* stream);
/* Backward of cvb_clifford_vm_rsample_kl, the implicit reparameterisation gradient of the von Mises draws: phi from the
 * forward of the SAME (loc, kappa, rows, d).  dL/dtheta_k = -(1/d) Im(e^{i theta_k} conj(G_k)), G = rfft(grad_z);
 * dloc (rows, d) = dL/dtheta (circle 0: 0); dkappa = dL/dtheta_k * d phi_k / d kappa_k, (rows) row sums when
 * kappa_el_stride == 0, else (rows, d). */
CVB_API int cvb_clifford_vm_rsample_backward(const float* grad_z, const float* loc, const float* kappa,
                                             long long kappa_row_stride, int kappa_el_stride, long long loc_rows,
                                             const float* phi, float* dloc, float* dkappa, long long rows, int d,
                                             void* stream);
/* CliffordTorusDistribution.log_prob: value (rows, 2d), a_k = angle(rfft(value)_k) ->
 * log_prob (rows) = sum_{k=1}^{d-1} kappa_k cos(a_k - loc_k) - ln(2 pi I0(kappa_k)) (the circles of the entropy and of
 * the uniform prior).  Optional derivative outputs as cvb_clifford_ps_log_prob's (give dlp_dloc and dlp_dkappa both or
 * neither; dlp_dF (rows, d) complex); circle 0 gets zeros. */
CVB_API int cvb_clifford_vm_log_prob(const float* value, const float* loc, const float* kappa, long long kappa_row_stride,
                                     int kappa_el_stride, long long loc_rows, float* log_prob, float* dlp_dloc,
                                     float* dlp_dkappa, float* dlp_dF, long long rows, int d, void* stream);

/* CliffordTorusUniform.rsample (dists/clifford.py:228-236) and the shared "phases -> real vector with
 * unit-magnitude spectrum" map.  phases (rows, d) are multiplied by phase_scale (2*pi for uniform u);
 * phases == NULL draws u on the device.  z (rows, 2d). */
CVB_API int cvb_clifford_phases_to_vector(const float* phases, float phase_scale, unsigned long long seed,
                                  unsigned long long offset, float* z, long long rows, int d, void* stream);

/* ---- VSA / HRR ops: utils/vsa.py:9-96 ----------------------------------------------------------- */

/* bind / unbind family: out[r] = irfft(op(rfft a[r % a_rows], rfft b[r % b_rows])), rows of length d. */
CVB_API int cvb_vsa_bind(const float* a, const float* b, float* out, long long rows, long long a_rows, long long b_rows, int d,
                 int mode, void* stream);
/* Fused binding-depth chain (scripts/binding_depth_heatmap.py:25-35): vecs (trials, m_plus_1, d); per trial bind
 * vecs[:,0] with vecs[:,1..m] in order, unbind ("inv") in reverse order, out[trial] = cos(recovered, vecs[:,0]).
 * Evaluated in the frequency domain (X0 * prod |Y_j|^2, Parseval): 4 d (m+1) bytes read per trial.  d: power of
 * two in [32, 16384]. */
CVB_API int cvb_vsa_depth_chain_cosine(const float* vecs, float* out, long long trials, int m_plus_1, int d, void* stream);
/* invert (utils/vsa.py:49-53) */
CVB_API int cvb_vsa_invert(const float* a, float* out, long long rows, int d, void* stream);
/* permute_vector / unpermute_vector (utils/vsa.py:82-90); perm is int64 (d). */
CVB_API int cvb_vsa_permute(const float* v, const long long* perm, float* out, long long rows, int d, int inverse, void* stream);
/* bundle (utils/vsa.py:75-79): out (d) = scale * sum_k v[k]; workspace >= cvb_vsa_bundle_workspace_bytes. */
CVB_API long long cvb_vsa_bundle_workspace_bytes(long long k, int d);
CVB_API int cvb_vsa_bundle(const float* v, float* out, long long k, int d, float scale, void* workspace, void* stream);
/* similarity (utils/vsa.py:93-96): cosine, norms clamped at 1e-8; rows broadcast by modulo. */
CVB_API int cvb_vsa_cosine(const float* a, const float* b, float* out, long long rows, long long a_rows, long long b_rows, int d,
                   void* stream);
CVB_API int cvb_vsa_cosine_backward(const float* a, const float* b, const float* grad_out, float* da, float* db, long long rows,
                            long long a_rows, long long b_rows, int d, void* stream);
/* normalize_vectors (utils/vsa.py:39-40) */
CVB_API int cvb_vsa_normalize(const float* x, float* out, long long rows, int d, void* stream);
CVB_API int cvb_vsa_normalize_backward(const float* x, const float* grad_out, float* dx, long long rows, int d, void* stream);
/* hrr_init (utils/vsa.py:9-12): N(0, 1/d) ; unitary_init (utils/vsa.py:15-36) */
CVB_API int cvb_vsa_hrr_init(float* out, long long n, int d, unsigned long long seed, unsigned long long offset, void* stream);
CVB_API int cvb_vsa_unitary_init(float* out, long long n, int d, float eps, unsigned long long seed, unsigned long long offset,
                         void* stream);

/* ---- D-dimensional PowerSpherical: dists/clifford.py:85-212, :335-337 -------------------------- */

/* PowerSpherical.rsample (dists/clifford.py:152-185).  loc (loc_rows, D) unit rows, kappa (loc_rows).
 * Inject tprime (rows) ~ Beta((D-1)/2 + kappa + 1e-7, (D-1)/2) and gnoise (rows, D-1) ~ N(0,1), or both
 * NULL for device RNG (Philox (seed, offset)).  z (rows, D).  save (rows, 2) optional: (t', 0) for the
 * backward in RNG mode. */
CVB_API int cvb_powerspherical_rsample(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                       const float* gnoise, unsigned long long seed, unsigned long long offset,
                                       float* z, float* save, long long rows, int D, void* stream);
/* Backward: grad_z (rows, D) -> dloc (rows, D), dkappa (rows).  Injected mode: pass the same tprime /
 * gnoise; RNG mode: pass save from the forward and the same (seed, offset) -- the tangent normals are
 * replayed from the counter-based generator instead of being stored. */
/* The same sampler fused with entropy() / KL to HypersphericalUniform (dists/clifford.py:204-212, :335-337): ONE launch
 * for the latent terms of a training step (BASELINE config 2).  entropy / kl / dentropy: (loc_rows), each may be NULL. */
CVB_API int cvb_powerspherical_rsample_kl(const float* loc, const float* kappa, long long loc_rows, const float* tprime,
                                          const float* gnoise, unsigned long long seed, unsigned long long offset,
                                          float* z, float* save, float* entropy, float* kl, float* dentropy,
                                          long long rows, int D, void* stream);
CVB_API int cvb_powerspherical_rsample_backward(const float* grad_z, const float* loc, const float* kappa,
                                                long long loc_rows, const float* tprime, const float* gnoise,
                                                const float* save, unsigned long long seed, unsigned long long offset,
                                                float* dloc, float* dkappa, long long rows, int D, void* stream);
/* PowerSpherical.log_prob (dists/clifford.py:198-202).  Optional backward helpers: coef (rows) with
 * d lp/d loc = coef * value and d lp/d value = coef * loc, and dlp_dkappa (rows). */
CVB_API int cvb_powerspherical_log_prob(const float* value, const float* loc, const float* kappa, long long loc_rows,
                                        float* log_prob, float* coef, float* dlp_dkappa, long long rows, int D,
                                        void* stream);
/* PowerSpherical.log_normalizer (dists/clifford.py:187-196) and d/dkappa (optional), elementwise. */
CVB_API int cvb_ps_log_normalizer(const float* kappa, long long rows, double half_dm1, float* log_norm,
                                  float* dlog_norm, void* stream);
/* HypersphericalUniform.rsample (dists/clifford.py:100-107): gnoise (rows, D) or NULL -> z = g/(||g||+eps). */
CVB_API int cvb_sphere_uniform_rsample(const float* gnoise, unsigned long long seed, unsigned long long offset,
                                       float* z, long long rows, int D, float norm_eps, void* stream);

/* ---- von Mises-Fisher: vmf/hyperspherical_vae/distributions/von_mises_fisher.py:11-217 ---------- */

/* VonMisesFisher.rsample (:50-181).  kappa (loc_rows).  Injected mode: e_rounds / u_rounds
 * (n_rounds, rows) fp64 rejection proposals (e ~ Beta((m-1)/2,(m-1)/2), u ~ U(1e-20, 1-1e-20)); each row
 * takes its first accepted round; for D == 3 u_rounds row 0 is the closed-form uniform (:73-88); gnoise
 * (rows, D) normals whose column 0 is discarded (:59-65).  All NULL: device rejection loop.
 * z (rows, D); save (rows, 2) = (w, dw/dkappa) for the backward. */
CVB_API int cvb_vmf_rsample(const float* loc, const float* kappa, long long loc_rows, const double* e_rounds,
                            const double* u_rounds, int n_rounds, const float* gnoise, unsigned long long seed,
                            unsigned long long offset, float* z, float* save, long long rows, int D, void* stream);
/* cvb_vmf_rsample fused with entropy / KL to the uniform prior / log-normaliser and their kappa-derivatives
 * (von_mises_fisher.py:183-217): one launch; the five row outputs are (loc_rows) and optional. */
CVB_API int cvb_vmf_rsample_kl(const float* loc, const float* kappa, long long loc_rows, const double* e_rounds,
                               const double* u_rounds, int n_rounds, const float* gnoise, unsigned long long seed,
                               unsigned long long offset, float* z, float* save, float* entropy, float* kl,
                               float* dentropy, float* log_norm, float* dlog_norm, long long rows, int D, void* stream);
CVB_API int cvb_vmf_rsample_backward(const float* grad_z, const float* loc, const float* kappa, long long loc_rows,
                                     const float* gnoise, const float* save, unsigned long long seed,
                                     unsigned long long offset, float* dloc, float* dkappa, long long rows, int D,
                                     void* stream);
/* entropy (:183-191), log-normaliser (:200-212; device log I_v replaces scipy.special.ive on the host,
 * ops/ive.py:9-34) and their kappa-derivatives; all (rows), any pointer may be NULL. */
CVB_API int cvb_vmf_entropy_lognorm(const float* kappa, long long rows, int D, float* entropy, float* log_norm,
                                    float* dentropy, float* dlog_norm, void* stream);

/* CliffordTorusDistribution.entropy (dists/clifford.py:21-31 `_von_mises_entropy`, :277-278): sum over circles k >= 1 of
 * ln 2 pi + ln(i0e(kappa) + 1e-7) + kappa - kappa (i1e(kappa) + 1e-7) / (i0e(kappa) + 1e-7).  kappa addressed like
 * cvb_clifford_ps_rsample's.  entropy (rows); dentropy optional: (rows) when kappa_el_stride == 0, else (rows, d). */
CVB_API int cvb_clifford_vm_entropy(const float* kappa, long long kappa_row_stride, int kappa_el_stride, long long rows,
                                    int d, float* entropy, float* dentropy, void* stream);
/* VonMisesFisher.log_prob (von_mises_fisher.py:193-212): log_prob (rows) = kappa <loc, value> - log_norm, with log_norm
 * (loc_rows) from cvb_vmf_rsample_kl / cvb_vmf_entropy_lognorm; dot (rows) = <loc, value>, optional (for the backward). */
CVB_API int cvb_vmf_log_prob(const float* value, const float* loc, const float* kappa, const float* log_norm,
                             long long loc_rows, float* log_prob, float* dot, long long rows, int D, void* stream);
/* Backward of the row log-densities lp = f(<loc, value>) (PowerSpherical.log_prob, VonMisesFisher.log_prob): with
 * w (rows) = upstream * d lp / d <loc, value>:  dvalue (rows, D) = w loc,  dloc (loc_rows, D) = sum over the samples
 * sharing a parameter row of w value.  Either output may be NULL. */
CVB_API int cvb_sphere_logprob_backward(const float* w, const float* value, const float* loc, long long loc_rows,
                                        float* dvalue, float* dloc, long long rows, int D, void* stream);

/* ---- Concentration head folded into the samplers (SURVEY section 8(f)2) ------------------------------------------
 * Every reference model computes the concentration as  kappa = clamp(softplus(fc_scale(h)) + floor, max=kmax)
 * (mnist/mlp_vae.py:69-71 floor 0.8 | 0.03, max 10; cnn/models.py:96,99 floor 0.5 | concentration_floor) right before
 * it builds the distribution.  The *_head entry points take the RAW output of that linear layer, raw_scale (loc_rows),
 * one value per row, and evaluate softplus + floor + clamp inside the sampling kernel; the backward entry points and
 * every kappa-derivative output (dentropy_draw, dlog_norm_draw, draw_scale) carry the chain factor
 * d kappa / d raw = sigmoid(raw) * [softplus(raw) + floor <= kmax], i.e. they are derivatives with respect to raw_scale.
 * All other arguments are those of the entry point without the suffix. */
CVB_API int cvb_clifford_ps_rsample_head(const float* loc, const float* raw_scale, long long loc_rows, float floor, float kmax,
                                         const float* tprime, const float* gnoise, unsigned long long seed,
                                         unsigned long long offset, float* z, float* tp_signed, float* entropy, float* kl,
                                         float* dentropy_draw, long long rows, int d, void* stream);
CVB_API int cvb_clifford_ps_rsample_backward_head(const float* grad_z, const float* loc, const float* raw_scale,
                                                  long long loc_rows, float floor, float kmax, const float* tprime,
                                                  const float* gnoise, const float* tp_signed, float* dloc,
                                                  float* draw_scale, long long rows, int d, void* stream);
CVB_API int cvb_powerspherical_rsample_kl_head(const float* loc, const float* raw_scale, long long loc_rows, float floor,
                                               float kmax, const float* tprime, const float* gnoise,
                                               unsigned long long seed, unsigned long long offset, float* z, float* save,
                                               float* entropy, float* kl, float* dentropy_draw, long long rows, int D,
                                               void* stream);
CVB_API int cvb_powerspherical_rsample_backward_head(const float* grad_z, const float* loc, const float* raw_scale,
                                                     long long loc_rows, float floor, float kmax, const float* tprime,
                                                     const float* gnoise, const float* save, unsigned long long seed,
                                                     unsigned long long offset, float* dloc, float* draw_scale,
                                                     long long rows, int D, void* stream);
CVB_API int cvb_vmf_rsample_kl_head(const float* loc, const float* raw_scale, long long loc_rows, float floor, float kmax,
                                    const double* e_rounds, const double* u_rounds, int n_rounds, const float* gnoise,
                                    unsigned long long seed, unsigned long long offset, float* z, float* save,
                                    float* entropy, float* kl, float* dentropy_draw, float* log_norm,
                                    float* dlog_norm_draw, long long rows, int D, void* stream);
CVB_API int cvb_vmf_rsample_backward_head(const float* grad_z, const float* loc, const float* raw_scale, long long loc_rows,
                                          float floor, float kmax, const float* gnoise, const float* save,
                                          unsigned long long seed, unsigned long long offset, float* dloc,
                                          float* draw_scale, long long rows, int D, void* stream);

/* ---- CUDA-graph capture of the samplers.  (seed, offset) are kernel arguments chosen on the host, so a captured graph
 * would replay the same draws.  Register a device-resident 64-bit counter for the current device (NULL clears it): every
 * sampling kernel launched afterwards mixes it into its Philox offset.  The library only READS it; the caller bumps it
 * on the stream after each sampling launch (inside the capture), so every replay draws a fresh stream. */
CVB_API int cvb_set_rng_device_counter(const unsigned long long* counter);
/* The same registration in self-bumping mode: every launch that draws from the device generator adds 1 to *counter itself
 * when its last CTA retires, so a captured graph needs no counter-increment kernel between sampling launches.  Launches in
 * this mode must be serialised on one stream.  A backward launch that replays draws (cvb_powerspherical_rsample_backward,
 * cvb_vmf_rsample_backward) must read the value its forward read: snapshot the counter before the forward and register
 * the snapshot with cvb_set_rng_device_counter around the backward.  NULL leaves the mode. */
CVB_API int cvb_set_rng_device_counter_autobump(unsigned long long* counter);

/* ---- host-only: the inverse-CDF table behind the device sampler of dists/clifford.py:124-134's Beta(1/2 + kappa, 1/2)
 * draw for row-scalar concentrations <= *kappa_max (csrc/icdf_table.cuh).  Layout: [n_kappa][n_nodes][2] floats =
 * (H, dH/ds / (n_nodes - 1)) with concentration node i at kappa_i = expm1(log1p(kappa_max) * i / (n_kappa - 1)) and
 * s-node j at s = j / (n_nodes - 1); |psi| = H(s), s = v^(1 / (2 kappa + 1)), t' = cos^2(psi).  out may be NULL to
 * query the sizes only.  Needs no GPU (the CPU test checks it against SciPy's betaincinv). */
CVB_API int cvb_ps_halfangle_icdf_table(float* out, long long capacity_floats, int* n_kappa, int* n_nodes,
                                        float* kappa_max);

/* ---- test hook: raw Philox4x32-10 words, out[4*i .. 4*i+3] = philox(counter = (i, 0, 0, offset)) --- */
CVB_API int cvb_philox_fill(unsigned int* out, long long n_vec4, unsigned long long seed, unsigned long long offset,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLIFFORD_B200_H_ */
